// pymodule.cpp — pybind11 module `openfdcm_b200._openfdcm_cuda`: the reference's Python surface
// (reference modules/python/src/matching.cpp:62-308, core.cpp:39-50) over the CUDA types.
//
// Same class / function names and argument meaning as the reference's `openfdcm` module, with Dt3CudaParameters /
// build_cuda_featuremap / Dt3Cuda in place of the Dt3Cpu trio, the type-erased FeatureMap / SearchStrategy /
// OptimizeStrategy / MatchStrategy / PenaltyStrategy with the same implicit conversions, plus the fused search_topk.
// The reference binds Eigen types through pybind11/eigen.h; Eigen is not a dependency here, so line arrays come in as
// numpy (4, N) arrays of any dtype / layout (py::array_t<float, forcecast>, the same f64 -> f32 conversion the Eigen caster
// performs) and 2x3 transforms go out as numpy (2, 3) float32 arrays.
// Everything computes through the C ABI of libfdcm_b200.so; there is no CPU fallback.
#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include <sstream>

#include "openfdcm_b200/strategies.hpp"

namespace py = pybind11;
using namespace pybind11::literals;
using namespace openfdcm::cuda;
using LinesIn = py::array_t<float, py::array::forcecast>;

static LineArray to_lines(const LinesIn& a) {
    if (a.size() == 0) return {};
    if (a.ndim() == 1 && a.shape(0) == 4) {
        auto u = a.unchecked<1>();
        return LineArray{u(0), u(1), u(2), u(3)};
    }
    if (a.ndim() != 2 || a.shape(0) != 4) throw py::value_error("expected a (4, N) line array");
    auto u = a.unchecked<2>();
    const py::ssize_t n = a.shape(1);
    LineArray out((size_t)n * 4);
    for (py::ssize_t i = 0; i < n; ++i)
        for (int r = 0; r < 4; ++r) out[(size_t)i * 4 + (size_t)r] = u(r, i);
    return out;
}
static std::vector<LineArray> to_templates(const std::vector<LinesIn>& v) {
    std::vector<LineArray> out;
    out.reserve(v.size());
    for (const auto& a : v) out.push_back(to_lines(a));
    return out;
}
static py::array_t<float> mat23_out(const Mat23& t) {
    py::array_t<float> a({2, 3});
    auto u = a.mutable_unchecked<2>();
    for (int r = 0; r < 2; ++r)
        for (int c = 0; c < 3; ++c) u(r, c) = t[(size_t)(r * 3 + c)];
    return a;
}
static Mat23 mat23_in(const py::array_t<float, py::array::forcecast>& a) {
    if (a.ndim() != 2 || a.shape(0) != 2 || a.shape(1) != 3) throw py::value_error("expected a (2, 3) transform");
    auto u = a.unchecked<2>();
    Mat23 t{};
    for (int r = 0; r < 2; ++r)
        for (int c = 0; c < 3; ++c) t[(size_t)(r * 3 + c)] = u(r, c);
    return t;
}

struct PyDt3CudaParameters {   // PyDt3CpuParameters (matching.cpp:51-60) + device
    size_t depth;
    float dt3Coeff, padding;
    Distance distance;
    int device;
};
struct PyThreadPool { unsigned n; };   // BS::thread_pool stand-in: accepted and ignored (the device is the pool)

PYBIND11_MODULE(_openfdcm_cuda, m) {
    m.doc() = "B200-native OpenFDCM hot paths: pybind11 mirror of the reference's `openfdcm` module over CUDA types";

    py::enum_<Distance>(m, "distance")   // core.cpp:45-49
        .value("L2", Distance::L2)
        .value("L2_SQUARED", Distance::L2_SQUARED)
        .value("L1", Distance::L1);

    // ---- feature maps -------------------------------------------------------------------------
    py::class_<Dt3Cuda>(m, "Dt3Cuda")
        .def("get_scene_translation", [](const Dt3Cuda& a) {
            const Point2 t = a.getSceneTranslation();
            py::array_t<float> out(2);
            out.mutable_at(0) = t.x;
            out.mutable_at(1) = t.y;
            return out;
        })
        .def("get_feature_size", [](const Dt3Cuda& a) {
            const Size s = a.getFeatureSize();
            py::array_t<uint64_t> out(2);
            out.mutable_at(0) = s.x;
            out.mutable_at(1) = s.y;
            return out;
        })
        .def("angles", [](const Dt3Cuda& a) { return py::array_t<float>(py::cast(a.angles())); })
        .def("plane", [](const Dt3Cuda& a, int i) {
            const auto inf = a.info();
            py::array_t<float> out({inf.height, inf.width});
            check(fdcm_dt3_download_plane(a.handle(), i, out.mutable_data()));
            return out;
        }, "i"_a)
        .def("get_dt3_map", [](const Dt3Cuda& a) {   // {angle: H x W image} like Dt3Cpu::getDt3Map (downloads the whole map)
            py::dict d;
            const auto inf = a.info();
            const auto keys = a.angles();
            for (int i = 0; i < inf.depth; ++i) {
                py::array_t<float> out({inf.height, inf.width});
                check(fdcm_dt3_download_plane(a.handle(), i, out.mutable_data()));
                d[py::float_(keys[(size_t)i])] = out;
            }
            return d;
        })
        .def_property_readonly("depth", [](const Dt3Cuda& a) { return a.info().depth; })
        .def_property_readonly("width", [](const Dt3Cuda& a) { return a.info().width; })
        .def_property_readonly("height", [](const Dt3Cuda& a) { return a.info().height; })
        .def_property_readonly("device", [](const Dt3Cuda& a) { return a.info().device; })
        .def("__repr__", [](const Dt3Cuda& a) {
            const Point2 t = a.getSceneTranslation();
            const Size s = a.getFeatureSize();
            return "<Dt3Cuda: scene translation=(" + std::to_string(t.x) + ", " + std::to_string(t.y) + "), feature size=(" +
                   std::to_string(s.x) + ", " + std::to_string(s.y) + ")>";
        });

    py::class_<FeatureMap>(m, "FeatureMap").def(py::init<const Dt3Cuda&>()).def("__repr__", [](const FeatureMap&) { return "<FeatureMap>"; });
    py::implicitly_convertible<Dt3Cuda, FeatureMap>();

    py::class_<PyThreadPool>(m, "ThreadPool")
        .def(py::init([]() { return PyThreadPool{0}; }))
        .def(py::init([](unsigned n) { return PyThreadPool{n}; }), "num_threads"_a)
        .def("get_thread_count", [](const PyThreadPool& p) { return p.n; })
        .def("__repr__", [](const PyThreadPool& p) { return "<ThreadPool: threads=" + std::to_string(p.n) + " (ignored by the CUDA strategies)>"; });

    py::class_<PyDt3CudaParameters>(m, "Dt3CudaParameters")
        .def(py::init([](size_t depth, float coeff, float padding, Distance d, int device) { return PyDt3CudaParameters{depth, coeff, padding, d, device}; }),
             "depth"_a = 30, "dt3Coeff"_a = 5.f, "padding"_a = 2.2f, "distance"_a = Distance::L2, "device"_a = 0)
        .def_readwrite("depth", &PyDt3CudaParameters::depth)
        .def_readwrite("dt3_coeff", &PyDt3CudaParameters::dt3Coeff)
        .def_readwrite("padding", &PyDt3CudaParameters::padding)
        .def_readwrite("distance", &PyDt3CudaParameters::distance)
        .def_readwrite("device", &PyDt3CudaParameters::device)
        .def("__repr__", [](const PyDt3CudaParameters& p) {
            return "<Dt3CudaParameters: depth=" + std::to_string(p.depth) + ", dt3_coeff=" + std::to_string(p.dt3Coeff) +
                   ", padding=" + std::to_string(p.padding) + ">";
        });

    m.def("build_cuda_featuremap",
          [](const LinesIn& scene, const PyDt3CudaParameters& p, const py::object& /*pool*/) {
              return buildCudaFeaturemap(to_lines(scene), Dt3CudaParameters{p.depth, p.dt3Coeff, p.padding, p.distance, p.device});
          },
          "scene"_a, "params"_a = PyDt3CudaParameters{30, 5.f, 2.2f, Distance::L2, 0}, "pool"_a = py::none(),
          "Builds the Dt3Cuda featuremap given a scene and parameters (the thread pool argument of build_cpu_featuremap is accepted and ignored).");

    // ---- optimize strategies ------------------------------------------------------------------
    py::class_<OptimizeStrategy>(m, "OptimizeStrategy")
        .def(py::init<const DefaultOptimize&>())
        .def(py::init<const BatchOptimize&>())
        .def("__repr__", [](const OptimizeStrategy&) { return "<OptimizeStrategy>"; });
    py::class_<DefaultOptimize>(m, "DefaultOptimize")
        .def(py::init([](const py::object&) { return DefaultOptimize{}; }), "pool"_a = py::none())
        .def(py::init([](unsigned) { return DefaultOptimize{}; }), "num_threads"_a)
        .def("__repr__", [](const DefaultOptimize&) { return "<DefaultOptimize>"; });
    py::class_<BatchOptimize>(m, "BatchOptimize")
        .def(py::init([](size_t b, const py::object&) {
                 if (b < 1) throw py::value_error("batch_size must be >= 1");
                 return BatchOptimize{b};
             }), "batch_size"_a, "pool"_a = py::none())
        .def(py::init([](size_t b, unsigned) {
                 if (b < 1) throw py::value_error("batch_size must be >= 1");
                 return BatchOptimize{b};
             }), "batch_size"_a, "num_threads"_a)
        .def("get_batch_size", &BatchOptimize::getBatchSize)
        .def("__repr__", [](const BatchOptimize&) { return "<BatchOptimize>"; });
    py::implicitly_convertible<DefaultOptimize, OptimizeStrategy>();
    py::implicitly_convertible<BatchOptimize, OptimizeStrategy>();

    // ---- penalty strategies -------------------------------------------------------------------
    py::class_<PenaltyStrategy>(m, "PenaltyStrategy")
        .def(py::init<const DefaultPenalty&>())
        .def(py::init<const ExponentialPenalty&>())
        .def("__repr__", [](const PenaltyStrategy&) { return "<PenaltyStrategy>"; });
    py::class_<DefaultPenalty>(m, "DefaultPenalty").def(py::init<>()).def("__repr__", [](const DefaultPenalty&) { return "<DefaultPenalty>"; });
    py::class_<ExponentialPenalty>(m, "ExponentialPenalty")
        .def(py::init([](float tau) { return ExponentialPenalty{tau}; }), "tau"_a)
        .def("get_tau", &ExponentialPenalty::getTau)
        .def("__repr__", [](const ExponentialPenalty& a) { return "<ExponentialPenalty: tau=" + std::to_string(a.getTau()) + ">"; });
    py::implicitly_convertible<DefaultPenalty, PenaltyStrategy>();
    py::implicitly_convertible<ExponentialPenalty, PenaltyStrategy>();

    // ---- search strategies --------------------------------------------------------------------
    py::class_<SearchStrategy>(m, "SearchStrategy")
        .def(py::init<const DefaultSearch&>())
        .def(py::init<const ConcentricRangeStrategy&>())
        .def("__repr__", [](const SearchStrategy&) { return "<SearchStrategy>"; });
    py::class_<DefaultSearch>(m, "DefaultSearch")
        .def(py::init([](size_t t, size_t s) { return DefaultSearch{t, s}; }), "max_tmpl_lines"_a, "max_scene_lines"_a)
        .def("get_max_tmpl_lines", &DefaultSearch::getMaxTmplLines)
        .def("get_max_scene_lines", &DefaultSearch::getMaxSceneLines)
        .def("__repr__", [](const DefaultSearch& a) {
            return "<DefaultSearch: max tmpl lines=" + std::to_string(a.getMaxTmplLines()) + ", max scene lines=" + std::to_string(a.getMaxSceneLines()) + ">";
        });
    py::class_<ConcentricRangeStrategy>(m, "ConcentricRangeStrategy")
        .def(py::init([](size_t t, size_t s, const py::array_t<float, py::array::forcecast>& c, float lo, float hi) {
                 if (c.size() != 2) throw py::value_error("center_position must have two components");
                 py::array_t<float, py::array::c_style | py::array::forcecast> cc(c);
                 return ConcentricRangeStrategy{t, s, Point2{cc.data()[0], cc.data()[1]}, lo, hi};
             }), "max_tmpl_lines"_a, "max_scene_lines"_a, "center_position"_a, "low_boundary"_a, "high_boundary"_a)
        .def("get_max_tmpl_lines", &ConcentricRangeStrategy::getMaxTmplLines)
        .def("get_max_scene_lines", &ConcentricRangeStrategy::getMaxSceneLines)
        .def("get_center_position", [](const ConcentricRangeStrategy& a) {
            py::array_t<float> out(2);
            out.mutable_at(0) = a.center_position.x;
            out.mutable_at(1) = a.center_position.y;
            return out;
        })
        .def("get_low_radius_boundary", &ConcentricRangeStrategy::getLowBoundary)
        .def("get_high_radius_boundary", &ConcentricRangeStrategy::getHighBoundary);
    py::implicitly_convertible<DefaultSearch, SearchStrategy>();
    py::implicitly_convertible<ConcentricRangeStrategy, SearchStrategy>();

    // ---- match strategies ---------------------------------------------------------------------
    py::class_<MatchStrategy>(m, "MatchStrategy").def(py::init<const DefaultMatch&>()).def("__repr__", [](const MatchStrategy&) { return "<MatchStrategy>"; });
    py::class_<DefaultMatch>(m, "DefaultMatch").def(py::init<>()).def("__repr__", [](const DefaultMatch&) { return "<DefaultMatch>"; });
    py::implicitly_convertible<DefaultMatch, MatchStrategy>();
    m.attr("CudaMatch") = m.attr("DefaultMatch");   // the matcher whose search() fuses enumerate / optimise / match on the device

    py::class_<Match>(m, "Match")
        .def(py::init([](int idx, float score, const py::array_t<float, py::array::forcecast>& t) { return Match{idx, score, mat23_in(t)}; }))
        .def_readwrite("tmpl_idx", &Match::tmplIdx)
        .def_readwrite("score", &Match::score)
        .def_property("transform", [](const Match& a) { return mat23_out(a.transform); },
                      [](Match& a, const py::array_t<float, py::array::forcecast>& t) { a.transform = mat23_in(t); })
        .def("__repr__", [](const Match& a) {
            std::ostringstream oss;
            oss << "<Match tmplIdx=" << a.tmplIdx << ", score=" << a.score << ", transform=\n"
                << a.transform[0] << " " << a.transform[1] << " " << a.transform[2] << "\n"
                << a.transform[3] << " " << a.transform[4] << " " << a.transform[5] << ">";
            return oss.str();
        });

    m.def("search",
          [](const MatchStrategy& matcher, const SearchStrategy& searcher, const OptimizeStrategy& optimizer, const FeatureMap& featuremap,
             const std::vector<LinesIn>& templates, const LinesIn& scene) {
              const auto t = to_templates(templates);
              const auto s = to_lines(scene);
              py::gil_scoped_release release;
              return search(matcher, searcher, optimizer, featuremap, t, s);
          },
          "matcher"_a, "searcher"_a, "optimizer"_a, "featuremap"_a, "templates"_a, "scene"_a,
          "Search for optimal matches between the templates and the scene");

    py::class_<DistinctMatches>(m, "DistinctMatches")
        .def(py::init([](int max_per_template, float radius, float max_angle, bool across_templates) {
                 return DistinctMatches{max_per_template, radius, max_angle, across_templates};
             }), "max_per_template"_a = 0, "radius"_a = 0.f, "max_angle"_a = 3.14159265358979323846f, "across_templates"_a = false)
        .def_readwrite("max_per_template", &DistinctMatches::maxPerTemplate)
        .def_readwrite("radius", &DistinctMatches::radius)
        .def_readwrite("max_angle", &DistinctMatches::maxAngle)
        .def_readwrite("across_templates", &DistinctMatches::acrossTemplates)
        .def("__repr__", [](const DistinctMatches& a) {
            return "<DistinctMatches: max_per_template=" + std::to_string(a.maxPerTemplate) + ", radius=" + std::to_string(a.radius) +
                   ", max_angle=" + std::to_string(a.maxAngle) + ", across_templates=" + (a.acrossTemplates ? "True" : "False") + ">";
        });

    py::class_<PoseRefinement>(m, "PoseRefinement")
        .def(py::init([](int levels, int rot_steps, float rot_step, int trans_steps, float trans_step) {
                 return PoseRefinement{levels, rot_steps, rot_step, trans_steps, trans_step};
             }), "levels"_a = 3, "rot_steps"_a = 4, "rot_step"_a = 0.01f, "trans_steps"_a = 4, "trans_step"_a = 1.f)
        .def_readwrite("levels", &PoseRefinement::levels)
        .def_readwrite("rot_steps", &PoseRefinement::rotSteps)
        .def_readwrite("rot_step", &PoseRefinement::rotStep)
        .def_readwrite("trans_steps", &PoseRefinement::transSteps)
        .def_readwrite("trans_step", &PoseRefinement::transStep)
        .def("__repr__", [](const PoseRefinement& a) {
            return "<PoseRefinement: levels=" + std::to_string(a.levels) + ", rot_steps=" + std::to_string(a.rotSteps) + ", rot_step=" +
                   std::to_string(a.rotStep) + ", trans_steps=" + std::to_string(a.transSteps) + ", trans_step=" + std::to_string(a.transStep) + ">";
        });

    m.def("search_topk",
          [](const Dt3Cuda& featuremap, const std::vector<LinesIn>& templates, const LinesIn& scene, const DefaultSearch& searcher,
             const BatchOptimize& optimizer, const ExponentialPenalty& penalty, int k, const std::optional<DistinctMatches>& select,
             const std::optional<PoseRefinement>& refine) {
              const auto t = to_templates(templates);
              const auto s = to_lines(scene);
              py::gil_scoped_release release;
              if (refine && select) return searchTopK(searcher, optimizer, penalty, featuremap, t, s, k, *select, *refine);
              if (refine) return searchTopK(searcher, optimizer, penalty, featuremap, t, s, k, *refine);
              if (select) return searchTopK(searcher, optimizer, penalty, featuremap, t, s, k, *select);
              return searchTopK(searcher, optimizer, penalty, featuremap, t, s, k);
          },
          "featuremap"_a, "templates"_a, "scene"_a, "searcher"_a, "optimizer"_a, "penalty"_a, "k"_a = 10, py::kw_only(), "select"_a = py::none(),
          "refine"_a = py::none(),
          "Fused search -> penalize -> top-k on the device (ascending score); select: DistinctMatches for the distinct top-k; "
          "refine: PoseRefinement of the selected matches (not re-sorted; it minimises the score, which was measured to increase the "
          "error against known poses)");

    m.def("refine_matches",
          [](const Dt3Cuda& featuremap, const std::vector<LinesIn>& templates, const std::vector<Match>& matches, const PoseRefinement& refine,
             const std::optional<ExponentialPenalty>& penalty) {
              const auto t = to_templates(templates);
              py::gil_scoped_release release;
              if (penalty) return refineMatches(featuremap, t, matches, refine, *penalty);
              return refineMatches(featuremap, t, matches, refine);
          },
          "featuremap"_a, "templates"_a, "matches"_a, "refine"_a, "penalty"_a = py::none(),
          "Pose refinement of every match (entry i refines matches[i]) to the lowest evaluate score of its grid, not to a more "
          "accurate pose; with a penalty, scores are penalised like search_topk");

    py::class_<DenseSearch>(m, "DenseSearch")
        .def(py::init([](int rotations, float rot_start, std::optional<float> rot_step, int stride, int cell,
                         std::optional<std::array<float, 4>> roi) {
                 DenseSearch d;
                 d.rotations = rotations;
                 d.rotStart = rot_start;
                 d.rotStep = rot_step ? *rot_step : (rotations > 0 ? (float)(2.0 * 3.14159265358979323846 / rotations) : 0.f);
                 d.stride = stride;
                 d.cell = cell;
                 d.hasRoi = roi.has_value();
                 if (roi) d.roi = *roi;
                 return d;
             }), "rotations"_a = 72, "rot_start"_a = 0.f, "rot_step"_a = py::none(), "stride"_a = 2, "cell"_a = 8, "roi"_a = py::none())
        .def_readwrite("rotations", &DenseSearch::rotations)
        .def_readwrite("rot_start", &DenseSearch::rotStart)
        .def_readwrite("rot_step", &DenseSearch::rotStep)
        .def_readwrite("stride", &DenseSearch::stride)
        .def_readwrite("cell", &DenseSearch::cell)
        .def("__repr__", [](const DenseSearch& a) {
            return "<DenseSearch: rotations=" + std::to_string(a.rotations) + ", rot_start=" + std::to_string(a.rotStart) + ", rot_step=" +
                   std::to_string(a.rotStep) + ", stride=" + std::to_string(a.stride) + ", cell=" + std::to_string(a.cell) + ">";
        });

    m.def("search_dense",
          [](const Dt3Cuda& featuremap, const std::vector<LinesIn>& templates, const DenseSearch& dense, const ExponentialPenalty& penalty, int k,
             const std::optional<DistinctMatches>& select, const std::optional<PoseRefinement>& refine) {
              const auto t = to_templates(templates);
              py::gil_scoped_release release;
              return searchDense(featuremap, t, dense, penalty, k, select ? &*select : nullptr, refine ? &*refine : nullptr);
          },
          "featuremap"_a, "templates"_a, "dense"_a, "penalty"_a, "k"_a = 10, py::kw_only(), "select"_a = py::none(), "refine"_a = py::none(),
          "Dense pose-grid search on the device: the best pose of every (template, rotation, cell), then the top-k (ascending score) "
          "or with select the distinct top-k, then with refine the pose refinement of those");

    m.def("penalize",
          [](const PenaltyStrategy& penalty, const std::vector<Match>& matches, const std::vector<float>& templatelengths) {
              return penalize(penalty, matches, templatelengths);
          },
          "penalty"_a, "matches"_a, "templatelengths"_a, "Apply a given score penalty on a vector of matches");
    m.def("get_template_lengths", [](const std::vector<LinesIn>& templates) { return getTemplateLengths(to_templates(templates)); }, "templates"_a,
          "Get the lengths of templates represented by line arrays");
    m.def("sort_matches", [](std::vector<Match> matches) {
        sortMatches(matches);
        return matches;
    }, "matches"_a, "Sort the matches by score, with the best score (lowest) first.");

    // ---- FeatureMap / SearchStrategy / OptimizeStrategy concept entry points --------------------
    m.def("get_feature_size", [](const FeatureMap& fm) {
        const Size s = getFeatureSize(fm);
        py::array_t<uint64_t> out(2);
        out.mutable_at(0) = s.x;
        out.mutable_at(1) = s.y;
        return out;
    }, "featuremap"_a);
    m.def("minmax_translation", [](const FeatureMap& fm, const LinesIn& tmpl, const py::array_t<float, py::array::c_style | py::array::forcecast>& v) {
        if (v.size() != 2) throw py::value_error("align_vec must have two components");
        const auto r = minmaxTranslation(fm, to_lines(tmpl), Point2{v.data()[0], v.data()[1]});
        py::array_t<float> out(2);
        out.mutable_at(0) = r[0];
        out.mutable_at(1) = r[1];
        return out;
    }, "featuremap"_a, "tmpl"_a, "align_vec"_a);
    m.def("evaluate", [](const FeatureMap& fm, const std::vector<LinesIn>& templates,
                         const std::vector<py::array_t<float, py::array::c_style | py::array::forcecast>>& translations) {
        std::vector<std::vector<Point2>> tr(translations.size());
        for (size_t i = 0; i < translations.size(); ++i) {
            const auto& a = translations[i];
            if (a.size() % 2) throw py::value_error("translations must be (K, 2) arrays");
            for (py::ssize_t k = 0; k < a.size() / 2; ++k) tr[i].push_back(Point2{a.data()[2 * k], a.data()[2 * k + 1]});
        }
        return evaluate(fm, to_templates(templates), tr);
    }, "featuremap"_a, "templates"_a, "translations"_a);
    m.def("establish_search_strategy", [](const SearchStrategy& s, const LinesIn& tmpl, const LinesIn& scene) {
        const auto pairs = establishSearchStrategy(s, to_lines(tmpl), to_lines(scene));
        py::array_t<int64_t> out({(py::ssize_t)pairs.size(), (py::ssize_t)2});
        auto u = out.mutable_unchecked<2>();
        for (size_t i = 0; i < pairs.size(); ++i) {
            u((py::ssize_t)i, 0) = (int64_t)pairs[i].tmplLineIdx;
            u((py::ssize_t)i, 1) = (int64_t)pairs[i].sceneLineIdx;
        }
        return out;
    }, "searcher"_a, "tmpl"_a, "scene"_a);
    m.def("optimize", [](const OptimizeStrategy& o, const std::vector<LinesIn>& templates,
                         const std::vector<py::array_t<float, py::array::c_style | py::array::forcecast>>& alignments, const FeatureMap& fm) {
        std::vector<Point2> al;
        for (const auto& a : alignments) {
            if (a.size() != 2) throw py::value_error("alignments must be 2-vectors");
            al.push_back(Point2{a.data()[0], a.data()[1]});
        }
        const auto res = optimize(o, to_templates(templates), al, fm);
        py::list out;
        for (const auto& r : res) {
            if (!r) { out.append(py::none()); continue; }
            py::array_t<float> t(2);
            t.mutable_at(0) = r->translation.x;
            t.mutable_at(1) = r->translation.y;
            out.append(py::make_tuple(r->score, t));
        }
        return out;
    }, "optimizer"_a, "templates"_a, "alignments"_a, "featuremap"_a);

    py::register_exception<CudaError>(m, "CudaError", PyExc_RuntimeError);
}
