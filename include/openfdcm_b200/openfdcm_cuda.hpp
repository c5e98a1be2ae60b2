// openfdcm_cuda.hpp — C++ host mirror of the reference's strategy interfaces for the CUDA hot paths.
//
// Header-only C++17 on top of the C ABI (include/fdcm_b200.h).  It mirrors, name for name, the free-function
// "concept" API that openfdcm::matching dispatches on (reference modules/matching/include/openfdcm/matching/):
//   FeatureMap concept  (featuremap.h:27-52)      getFeatureSize / minmaxTranslation / evaluate  on Dt3Cuda
//   SearchStrategy      (searchstrategy.h:68-70)  establishSearchStrategy(DefaultSearch, tmpl, scene)
//   OptimizeStrategy    (optimizestrategy.h:62-64) optimize(BatchOptimize|DefaultOptimize, templates, alignments, Dt3Cuda)
//   MatchStrategy       (matchstrategy.h:78-81)   search(DefaultMatch, DefaultSearch, BatchOptimize, Dt3Cuda, templates, scene)
//   PenaltyStrategy     (penaltystrategy.h)       penalize(DefaultPenalty|ExponentialPenalty, matches, templatelengths)
// Eigen is not required: a LineArray is a std::vector<float> of packed [x1,y1,x2,y2] records, i.e. exactly the
// column-major memory of the reference's Eigen::Matrix<float,4,-1> (core/math.h:66); INTEGRATION.md shows the
// two-line adapters that plug these functions into the reference's type-erased FeatureMap / strategies.
#pragma once
#include <algorithm>
#include <array>
#include <cstdint>
#include <memory>
#include <optional>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "../fdcm_b200.h"

namespace openfdcm::cuda {

using LineArray = std::vector<float>;            // 4*N floats, records x1,y1,x2,y2
struct Point2 { float x, y; };
struct Size { size_t x, y; };                     // (width, height) like core::Size
using Mat23 = std::array<float, 6>;               // row-major r00 r01 tx r10 r11 ty

enum class Distance { L2 = 0, L2_SQUARED = 1, L1 = 2 };   // core/imgproc.h:148

struct CudaError : std::runtime_error {
    fdcm_status status;
    CudaError(fdcm_status st, const char* msg) : std::runtime_error(std::string("libfdcm_b200: ") + msg), status(st) {}
};
inline void check(fdcm_status st) {
    if (st == FDCM_ERR_OUT_OF_RANGE) throw std::out_of_range(fdcm_last_error());   // like the reference's penalize
    if (st != FDCM_OK) throw CudaError(st, fdcm_last_error());
}

// Dt3CpuParameters (featuremaps/dt3cpu.h:34-42) + distance (python/src/matching.cpp:51-60)
struct Dt3CudaParameters {
    size_t depth{30};
    float dt3Coeff{5.f}, padding{2.2f};
    Distance distance{Distance::L2};
    int device{0};
};

// Device-resident feature map; copies share one ref-counted handle (O(1), unlike FeatureMap::clone()).
class Dt3Cuda {
    std::shared_ptr<fdcm_dt3> h_;

public:
    Dt3Cuda() = default;
    explicit Dt3Cuda(fdcm_dt3* h) : h_(h, [](fdcm_dt3* p) { fdcm_dt3_release(p); }) {}
    fdcm_dt3* handle() const { return h_.get(); }
    fdcm_dt3_info info() const {
        fdcm_dt3_info i{};
        check(fdcm_dt3_get_info(h_.get(), &i));
        return i;
    }
    Point2 getSceneTranslation() const { auto i = info(); return {i.scene_translation[0], i.scene_translation[1]}; }
    Size getFeatureSize() const { auto i = info(); return {(size_t)i.width, (size_t)i.height}; }
    std::vector<float> angles() const {
        std::vector<float> k((size_t)info().depth);
        if (!k.empty()) check(fdcm_dt3_angles(h_.get(), k.data()));
        return k;
    }
    // one plane of getDt3Map() as a dense row-major height x width image
    std::vector<float> plane(int i) const {
        auto inf = info();
        std::vector<float> p((size_t)inf.width * inf.height);
        check(fdcm_dt3_download_plane(h_.get(), i, p.data()));
        return p;
    }
};

// buildCpuFeaturemap<D>(scene, params, pool) (dt3cpu.h:174-234)
inline Dt3Cuda buildCudaFeaturemap(const LineArray& scene, const Dt3CudaParameters& params = {}) {
    fdcm_dt3_params p{(int32_t)params.depth, params.dt3Coeff, params.padding, (int32_t)params.distance};
    fdcm_dt3* h = nullptr;
    check(fdcm_dt3_build(scene.data(), (int32_t)(scene.size() / 4), &p, params.device, 0, &h));
    return Dt3Cuda(h);
}

// ---- FeatureMap concept ------------------------------------------------------------------------
inline Size getFeatureSize(const Dt3Cuda& fm) noexcept {
    fdcm_dt3_info i{};
    return fdcm_dt3_get_info(fm.handle(), &i) == FDCM_OK ? Size{(size_t)i.width, (size_t)i.height} : Size{0, 0};
}

inline std::array<float, 2> minmaxTranslation(const Dt3Cuda& fm, const LineArray& tmpl, const Point2& align_vec) {
    const float v[2] = {align_vec.x, align_vec.y};
    std::array<float, 2> out{};
    check(fdcm_dt3_minmax_translation(fm.handle(), tmpl.data(), (int32_t)(tmpl.size() / 4), v, out.data()));
    return out;
}

namespace detail {
inline void pack(const std::vector<LineArray>& templates, std::vector<float>& flat, std::vector<int32_t>& off) {
    off.assign(templates.size() + 1, 0);
    for (size_t i = 0; i < templates.size(); ++i) off[i + 1] = off[i] + (int32_t)(templates[i].size() / 4);
    flat.clear();
    flat.reserve((size_t)off.back() * 4);
    for (const auto& t : templates) flat.insert(flat.end(), t.begin(), t.begin() + (t.size() / 4) * 4);
}
}   // namespace detail

inline std::vector<std::vector<float>> evaluate(const Dt3Cuda& fm, const std::vector<LineArray>& templates,
                                                const std::vector<std::vector<Point2>>& translations) {
    std::vector<float> flat, tr;
    std::vector<int32_t> off, troff(translations.size() + 1, 0);
    detail::pack(templates, flat, off);
    for (size_t i = 0; i < translations.size(); ++i) {
        troff[i + 1] = troff[i] + (int32_t)translations[i].size();
        for (const auto& p : translations[i]) { tr.push_back(p.x); tr.push_back(p.y); }
    }
    std::vector<float> scores((size_t)troff.back());
    check(fdcm_dt3_evaluate(fm.handle(), flat.data(), off.data(), (int32_t)templates.size(), tr.data(), troff.data(), scores.data()));
    std::vector<std::vector<float>> out(templates.size());
    for (size_t i = 0; i < templates.size(); ++i) out[i].assign(scores.begin() + troff[i], scores.begin() + troff[i + 1]);
    return out;
}

// ---- SearchStrategy concept --------------------------------------------------------------------
struct DefaultSearch {   // searchstrategies/defaultsearch.h:53-66
    size_t max_tmpl_lines, max_scene_lines;
    size_t getMaxTmplLines() const noexcept { return max_tmpl_lines; }
    size_t getMaxSceneLines() const noexcept { return max_scene_lines; }
};
struct SearchCombination { size_t tmplLineIdx, sceneLineIdx; };   // searchstrategy.h:32-45

inline std::vector<SearchCombination> establishSearchStrategy(const DefaultSearch& s, const LineArray& tmpl, const LineArray& scene) {
    const int32_t cap = (int32_t)(s.max_tmpl_lines * s.max_scene_lines) + 1;
    std::vector<int32_t> pairs((size_t)cap * 2);
    int32_t n = 0;
    check(fdcm_default_search(tmpl.data(), (int32_t)(tmpl.size() / 4), scene.data(), (int32_t)(scene.size() / 4),
                              (int32_t)s.max_tmpl_lines, (int32_t)s.max_scene_lines, pairs.data(), cap, &n));
    std::vector<SearchCombination> out((size_t)n);
    for (int32_t i = 0; i < n; ++i) out[(size_t)i] = {(size_t)pairs[2 * i], (size_t)pairs[2 * i + 1]};
    return out;
}

// ---- OptimizeStrategy concept -------------------------------------------------------------------
struct OptimalTranslation { float score; Point2 translation; };   // optimizestrategy.h:34-38
struct BatchOptimize { size_t batchSize; size_t getBatchSize() const noexcept { return batchSize; } };   // batchoptimize.h:8-23
struct DefaultOptimize {};                                                                             // defaultoptimize.h

namespace detail {
inline std::vector<std::optional<OptimalTranslation>> optimize(int batch, const std::vector<LineArray>& templates,
                                                               const std::vector<Point2>& alignments, const Dt3Cuda& fm) {
    if (templates.size() != alignments.size()) throw std::invalid_argument("templates.size() != alignments.size()");
    std::vector<float> flat, al;
    std::vector<int32_t> off;
    pack(templates, flat, off);
    for (const auto& a : alignments) { al.push_back(a.x); al.push_back(a.y); }
    const size_t n = templates.size();
    std::vector<uint8_t> has(n);
    std::vector<float> sc(n), tr(2 * n);
    check(fdcm_optimize(fm.handle(), flat.data(), off.data(), (int32_t)n, al.data(), batch, has.data(), sc.data(), tr.data()));
    std::vector<std::optional<OptimalTranslation>> out(n);
    for (size_t i = 0; i < n; ++i)
        if (has[i]) out[i] = OptimalTranslation{sc[i], {tr[2 * i], tr[2 * i + 1]}};
    return out;
}
}   // namespace detail

inline auto optimize(const BatchOptimize& o, const std::vector<LineArray>& templates, const std::vector<Point2>& alignments,
                     const Dt3Cuda& fm) { return detail::optimize((int)o.batchSize, templates, alignments, fm); }
inline auto optimize(const DefaultOptimize&, const std::vector<LineArray>& templates, const std::vector<Point2>& alignments,
                     const Dt3Cuda& fm) { return detail::optimize(0, templates, alignments, fm); }

// ---- MatchStrategy concept ----------------------------------------------------------------------
struct Match { int tmplIdx; float score; Mat23 transform; };   // matchstrategy.h:35-44
struct DefaultMatch {};
inline bool operator<(const Match& a, const Match& b) noexcept { return a.score < b.score; }

struct DefaultPenalty {};
struct ExponentialPenalty { float tau; float getTau() const noexcept { return tau; } };

namespace detail {
inline std::vector<Match> search_raw(const fdcm_search_params& p, const Dt3Cuda& fm, const std::vector<LineArray>& templates,
                                     const LineArray& scene) {
    std::vector<float> flat;
    std::vector<int32_t> off;
    pack(templates, flat, off);
    const int top_k = p.top_k;
    int64_t cap = top_k > 0 ? top_k : 0;
    if (top_k <= 0)
        for (const auto& t : templates) cap += 2 * (int64_t)std::min<size_t>(t.size() / 4, (size_t)p.max_tmpl_lines) * (int64_t)p.max_scene_lines;
    std::vector<fdcm_match> rec((size_t)std::max<int64_t>(cap, 1));
    int64_t n = 0;
    check(fdcm_search_host(fm.handle(), flat.data(), off.data(), (int32_t)templates.size(), scene.data(), (int32_t)(scene.size() / 4),
                           &p, rec.data(), (int64_t)rec.size(), &n));
    std::vector<Match> out((size_t)n);
    for (int64_t i = 0; i < n; ++i) {
        out[(size_t)i].tmplIdx = rec[(size_t)i].tmpl_idx;
        out[(size_t)i].score = rec[(size_t)i].score;
        for (int k = 0; k < 6; ++k) out[(size_t)i].transform[(size_t)k] = rec[(size_t)i].transform[k];
    }
    return out;
}
inline std::vector<Match> search(int batch, const DefaultSearch& s, const Dt3Cuda& fm, const std::vector<LineArray>& templates,
                                 const LineArray& scene, int penalty_kind, float tau, int top_k) {
    const fdcm_search_params p{(int32_t)s.max_tmpl_lines, (int32_t)s.max_scene_lines, batch, penalty_kind, tau, top_k, 0, 0, 0.f, 0.f, 0.f, 0.f};
    return search_raw(p, fm, templates, scene);
}
template <class Concentric>   // ConcentricRangeStrategy (strategies.hpp)
inline std::vector<Match> search_concentric(int batch, const Concentric& s, const Dt3Cuda& fm, const std::vector<LineArray>& templates,
                                            const LineArray& scene) {
    const fdcm_search_params p{(int32_t)s.max_tmpl_lines, (int32_t)s.max_scene_lines, batch, FDCM_PENALTY_NONE, 0.f, 0, 0, 1,
                               s.center_position.x, s.center_position.y, s.low_boundary, s.high_boundary};
    return search_raw(p, fm, templates, scene);
}
}   // namespace detail

// search(matcher, searcher, optimizer, featuremap, templates, originalScene) (defaultmatch.cpp:32-89):
// every match in hypothesis order, nullopt hypotheses dropped.
inline std::vector<Match> search(const DefaultMatch&, const DefaultSearch& s, const BatchOptimize& o, const Dt3Cuda& fm,
                                 const std::vector<LineArray>& templates, const LineArray& scene) {
    return detail::search((int)o.batchSize, s, fm, templates, scene, FDCM_PENALTY_NONE, 0.f, 0);
}
inline std::vector<Match> search(const DefaultMatch&, const DefaultSearch& s, const DefaultOptimize&, const Dt3Cuda& fm,
                                 const std::vector<LineArray>& templates, const LineArray& scene) {
    return detail::search(0, s, fm, templates, scene, FDCM_PENALTY_NONE, 0.f, 0);
}
// fused search -> penalize -> top-k on the device (ascending score)
inline std::vector<Match> searchTopK(const DefaultSearch& s, const BatchOptimize& o, const ExponentialPenalty& pen, const Dt3Cuda& fm,
                                     const std::vector<LineArray>& templates, const LineArray& scene, int k) {
    return detail::search((int)o.batchSize, s, fm, templates, scene, FDCM_PENALTY_EXPONENTIAL, pen.tau, k);
}

// distinct top-K (beyond the reference; rules of fdcm_search_select): at most maxPerTemplate matches of one template
// (0: no cap), and with radius > 0 no two matches whose template anchors lie within radius pixels at a rotation
// difference within maxAngle (>= pi: any), counted within one template unless acrossTemplates
struct DistinctMatches {
    int maxPerTemplate{0};
    float radius{0.f};
    float maxAngle{3.14159265358979323846f};
    bool acrossTemplates{false};
};
inline std::vector<Match> searchTopK(const DefaultSearch& s, const BatchOptimize& o, const ExponentialPenalty& pen, const Dt3Cuda& fm,
                                     const std::vector<LineArray>& templates, const LineArray& scene, int k, const DistinctMatches& select) {
    std::vector<float> flat;
    std::vector<int32_t> off;
    detail::pack(templates, flat, off);
    fdcm_templates* ts = nullptr;
    check(fdcm_templates_create(flat.data(), off.data(), (int32_t)templates.size(), fm.info().device, &ts));
    const std::unique_ptr<fdcm_templates, fdcm_status (*)(fdcm_templates*)> owner(ts, fdcm_templates_release);
    const fdcm_search_params p{(int32_t)s.max_tmpl_lines, (int32_t)s.max_scene_lines, (int32_t)o.batchSize, FDCM_PENALTY_EXPONENTIAL,
                               pen.tau, k, 0, 0, 0.f, 0.f, 0.f, 0.f};
    const fdcm_select_params q{select.maxPerTemplate, select.radius, select.maxAngle, select.acrossTemplates ? 1 : 0};
    std::vector<fdcm_match> rec((size_t)std::max(k, 1));
    int64_t n = 0;
    check(fdcm_search_select(fm.handle(), ts, scene.data(), (int32_t)(scene.size() / 4), &p, &q, rec.data(), (int64_t)rec.size(), &n));
    std::vector<Match> out((size_t)n);
    for (int64_t i = 0; i < n; ++i) {
        out[(size_t)i].tmplIdx = rec[(size_t)i].tmpl_idx;
        out[(size_t)i].score = rec[(size_t)i].score;
        for (int c = 0; c < 6; ++c) out[(size_t)i].transform[(size_t)c] = rec[(size_t)i].transform[c];
    }
    return out;
}

// pose refinement (beyond the reference; rules of fdcm_refine_matches): coarse-to-fine rotations about the template anchor
// and 2-D translations around each match, keeping the pose of lowest score over all template lines.  It minimises the
// evaluate score only, which was measured to increase the error against known poses (see fdcm_b200.h).
struct PoseRefinement {
    int levels{3};
    int rotSteps{4};
    float rotStep{0.01f};
    int transSteps{4};
    float transStep{1.f};
};
namespace detail {
inline fdcm_refine_params refine_params(const PoseRefinement& r) {
    return fdcm_refine_params{r.levels, r.rotSteps, r.rotStep, r.transSteps, r.transStep};
}
inline std::vector<Match> to_matches(const std::vector<fdcm_match>& rec, int64_t n) {
    std::vector<Match> out((size_t)n);
    for (int64_t i = 0; i < n; ++i) {
        out[(size_t)i].tmplIdx = rec[(size_t)i].tmpl_idx;
        out[(size_t)i].score = rec[(size_t)i].score;
        for (int c = 0; c < 6; ++c) out[(size_t)i].transform[(size_t)c] = rec[(size_t)i].transform[c];
    }
    return out;
}
inline std::vector<Match> search_refine(const DefaultSearch& s, const BatchOptimize& o, const ExponentialPenalty& pen, const Dt3Cuda& fm,
                                        const std::vector<LineArray>& templates, const LineArray& scene, int k, const DistinctMatches* select,
                                        const PoseRefinement& refine) {
    std::vector<float> flat;
    std::vector<int32_t> off;
    pack(templates, flat, off);
    fdcm_templates* ts = nullptr;
    check(fdcm_templates_create(flat.data(), off.data(), (int32_t)templates.size(), fm.info().device, &ts));
    const std::unique_ptr<fdcm_templates, fdcm_status (*)(fdcm_templates*)> owner(ts, fdcm_templates_release);
    const fdcm_search_params p{(int32_t)s.max_tmpl_lines, (int32_t)s.max_scene_lines, (int32_t)o.batchSize, FDCM_PENALTY_EXPONENTIAL,
                               pen.tau, k, 0, 0, 0.f, 0.f, 0.f, 0.f};
    fdcm_select_params q{};
    if (select) q = fdcm_select_params{select->maxPerTemplate, select->radius, select->maxAngle, select->acrossTemplates ? 1 : 0};
    const fdcm_refine_params r = refine_params(refine);
    std::vector<fdcm_match> rec((size_t)std::max(k, 1));
    int64_t n = 0;
    check(fdcm_search_refine(fm.handle(), ts, scene.data(), (int32_t)(scene.size() / 4), &p, select ? &q : nullptr, &r, rec.data(),
                             (int64_t)rec.size(), &n));
    return to_matches(rec, n);
}
inline std::vector<Match> refine_matches(const Dt3Cuda& fm, const std::vector<LineArray>& templates, const std::vector<Match>& matches,
                                         const PoseRefinement& refine, int penalty_kind, float tau) {
    std::vector<float> flat;
    std::vector<int32_t> off;
    pack(templates, flat, off);
    fdcm_templates* ts = nullptr;
    check(fdcm_templates_create(flat.data(), off.data(), (int32_t)templates.size(), fm.info().device, &ts));
    const std::unique_ptr<fdcm_templates, fdcm_status (*)(fdcm_templates*)> owner(ts, fdcm_templates_release);
    std::vector<fdcm_match> rec(matches.size());
    for (size_t i = 0; i < matches.size(); ++i) {
        rec[i].tmpl_idx = matches[i].tmplIdx;
        rec[i].score = matches[i].score;
        for (int c = 0; c < 6; ++c) rec[i].transform[c] = matches[i].transform[(size_t)c];
    }
    const fdcm_refine_params r = refine_params(refine);
    check(fdcm_refine_matches(fm.handle(), ts, 0, penalty_kind, tau, &r, rec.data(), (int64_t)rec.size(), rec.data()));
    return to_matches(rec, (int64_t)rec.size());
}
}   // namespace detail
// fused search -> top-k (or distinct top-k) -> pose refinement on the device; not re-sorted (sortMatches re-ranks)
inline std::vector<Match> searchTopK(const DefaultSearch& s, const BatchOptimize& o, const ExponentialPenalty& pen, const Dt3Cuda& fm,
                                     const std::vector<LineArray>& templates, const LineArray& scene, int k, const PoseRefinement& refine) {
    return detail::search_refine(s, o, pen, fm, templates, scene, k, nullptr, refine);
}
inline std::vector<Match> searchTopK(const DefaultSearch& s, const BatchOptimize& o, const ExponentialPenalty& pen, const Dt3Cuda& fm,
                                     const std::vector<LineArray>& templates, const LineArray& scene, int k, const DistinctMatches& select,
                                     const PoseRefinement& refine) {
    return detail::search_refine(s, o, pen, fm, templates, scene, k, &select, refine);
}
// refinement of any match list (tmplIdx indexes `templates`); without a penalty the scores are raw
inline std::vector<Match> refineMatches(const Dt3Cuda& fm, const std::vector<LineArray>& templates, const std::vector<Match>& matches,
                                        const PoseRefinement& refine) {
    return detail::refine_matches(fm, templates, matches, refine, FDCM_PENALTY_NONE, 0.f);
}
inline std::vector<Match> refineMatches(const Dt3Cuda& fm, const std::vector<LineArray>& templates, const std::vector<Match>& matches,
                                        const PoseRefinement& refine, const ExponentialPenalty& pen) {
    return detail::refine_matches(fm, templates, matches, refine, FDCM_PENALTY_EXPONENTIAL, pen.tau);
}

// dense pose-grid search (beyond the reference; rules of fdcm_search_dense): every template at `rotations` rotations
// rotStart + r * rotStep about its anchor (rotStep < 0: 2 pi / rotations) and at every stride-th map pixel (or of the
// region roi = {x0, y0, x1, y1} in scene coordinates when hasRoi); each cell of cell x cell grid points keeps its best pose
struct DenseSearch {
    int rotations{72};
    float rotStart{0.f};
    float rotStep{-1.f};
    int stride{2};
    int cell{8};
    bool hasRoi{false};
    std::array<float, 4> roi{{0.f, 0.f, 0.f, 0.f}};
};
// scale grid of the dense search (rules of fdcm_search_dense_scales): scales start * ratio^k, k = 0..scales-1.  The cost
// grows linearly with the number of scales; without a penalty the raw score favours small scales.
struct ScaleGrid {
    int scales{1};
    float start{1.f};
    float ratio{1.f};
};
namespace detail {
inline std::vector<Match> search_dense(const Dt3Cuda& fm, const std::vector<LineArray>& templates, const DenseSearch& dense, int penalty_kind,
                                       float tau, int k, const DistinctMatches* select, const PoseRefinement* refine,
                                       const fdcm_coverage_params* cov = nullptr, const ScaleGrid* scales = nullptr) {
    std::vector<float> flat;
    std::vector<int32_t> off;
    pack(templates, flat, off);
    fdcm_templates* ts = nullptr;
    check(fdcm_templates_create(flat.data(), off.data(), (int32_t)templates.size(), fm.info().device, &ts));
    const std::unique_ptr<fdcm_templates, fdcm_status (*)(fdcm_templates*)> owner(ts, fdcm_templates_release);
    const float step = dense.rotStep >= 0.f || dense.rotations < 1 ? dense.rotStep : (float)(2.0 * 3.14159265358979323846 / dense.rotations);
    const fdcm_dense_params d{dense.rotations, dense.rotStart, step, dense.stride, dense.cell, dense.hasRoi ? 1 : 0,
                              {dense.roi[0], dense.roi[1], dense.roi[2], dense.roi[3]}};
    fdcm_select_params q{};
    if (select) q = fdcm_select_params{select->maxPerTemplate, select->radius, select->maxAngle, select->acrossTemplates ? 1 : 0};
    fdcm_refine_params r{};
    if (refine) r = refine_params(*refine);
    std::vector<fdcm_match> rec((size_t)std::max(k, 1));
    int64_t n = 0;
    if (scales) {
        const fdcm_scale_grid g{scales->scales, scales->start, scales->ratio};
        check(fdcm_search_dense_scales(fm.handle(), ts, &d, &g, penalty_kind, tau, k, 0, select ? &q : nullptr, refine ? &r : nullptr, cov,
                                       rec.data(), (int64_t)rec.size(), &n));
    } else if (cov)
        check(fdcm_search_dense_verify(fm.handle(), ts, &d, penalty_kind, tau, k, 0, select ? &q : nullptr, refine ? &r : nullptr, cov,
                                       rec.data(), (int64_t)rec.size(), &n));
    else
        check(fdcm_search_dense(fm.handle(), ts, &d, penalty_kind, tau, k, 0, select ? &q : nullptr, refine ? &r : nullptr, rec.data(),
                                (int64_t)rec.size(), &n));
    return to_matches(rec, n);
}
}   // namespace detail
// dense search -> top-k (or distinct top-k) [-> pose refinement] on the device, penalised like searchTopK
inline std::vector<Match> searchDense(const Dt3Cuda& fm, const std::vector<LineArray>& templates, const DenseSearch& dense,
                                      const ExponentialPenalty& pen, int k) {
    return detail::search_dense(fm, templates, dense, FDCM_PENALTY_EXPONENTIAL, pen.tau, k, nullptr, nullptr);
}
inline std::vector<Match> searchDense(const Dt3Cuda& fm, const std::vector<LineArray>& templates, const DenseSearch& dense,
                                      const ExponentialPenalty& pen, int k, const DistinctMatches& select) {
    return detail::search_dense(fm, templates, dense, FDCM_PENALTY_EXPONENTIAL, pen.tau, k, &select, nullptr);
}
inline std::vector<Match> searchDense(const Dt3Cuda& fm, const std::vector<LineArray>& templates, const DenseSearch& dense,
                                      const ExponentialPenalty& pen, int k, const DistinctMatches* select, const PoseRefinement* refine) {
    return detail::search_dense(fm, templates, dense, FDCM_PENALTY_EXPONENTIAL, pen.tau, k, select, refine);
}

// match verification (beyond the reference; rules of fdcm_match_coverage): the fraction of a posed template's raster
// samples with a scene edge pixel within `radius` pixels on an orientation plane within `binTolerance` planes.  A support
// measure for a pose in [0, 1] (NaN outside the map), not a probability; the defaults are a starting point, not tuned.
// minCoverage > 0 filters the records of searchTopK / searchDense before their selection.
struct EdgeCoverage {
    int radius{2};
    int binTolerance{1};
    float minCoverage{0.f};
};
namespace detail {
inline fdcm_coverage_params coverage_params(const EdgeCoverage& c) { return fdcm_coverage_params{c.radius, c.binTolerance, c.minCoverage}; }
inline std::vector<Match> search_verify(const DefaultSearch& s, const BatchOptimize& o, const ExponentialPenalty& pen, const Dt3Cuda& fm,
                                        const std::vector<LineArray>& templates, const LineArray& scene, int k, const DistinctMatches* select,
                                        const PoseRefinement* refine, const EdgeCoverage& verify) {
    std::vector<float> flat;
    std::vector<int32_t> off;
    pack(templates, flat, off);
    fdcm_templates* ts = nullptr;
    check(fdcm_templates_create(flat.data(), off.data(), (int32_t)templates.size(), fm.info().device, &ts));
    const std::unique_ptr<fdcm_templates, fdcm_status (*)(fdcm_templates*)> owner(ts, fdcm_templates_release);
    const fdcm_search_params p{(int32_t)s.max_tmpl_lines, (int32_t)s.max_scene_lines, (int32_t)o.batchSize, FDCM_PENALTY_EXPONENTIAL,
                               pen.tau, k, 0, 0, 0.f, 0.f, 0.f, 0.f};
    fdcm_select_params q{};
    if (select) q = fdcm_select_params{select->maxPerTemplate, select->radius, select->maxAngle, select->acrossTemplates ? 1 : 0};
    fdcm_refine_params r{};
    if (refine) r = refine_params(*refine);
    const fdcm_coverage_params c = coverage_params(verify);
    std::vector<fdcm_match> rec((size_t)std::max(k, 1));
    int64_t n = 0;
    check(fdcm_search_verify(fm.handle(), ts, scene.data(), (int32_t)(scene.size() / 4), &p, select ? &q : nullptr, refine ? &r : nullptr,
                             &c, rec.data(), (int64_t)rec.size(), &n));
    return to_matches(rec, n);
}
}   // namespace detail
// coverage of every match (tmplIdx indexes `templates`), entry i for matches[i]
inline std::vector<float> matchCoverage(const Dt3Cuda& fm, const std::vector<LineArray>& templates, const std::vector<Match>& matches,
                                        const EdgeCoverage& coverage = EdgeCoverage{}) {
    std::vector<float> flat;
    std::vector<int32_t> off;
    detail::pack(templates, flat, off);
    fdcm_templates* ts = nullptr;
    check(fdcm_templates_create(flat.data(), off.data(), (int32_t)templates.size(), fm.info().device, &ts));
    const std::unique_ptr<fdcm_templates, fdcm_status (*)(fdcm_templates*)> owner(ts, fdcm_templates_release);
    std::vector<fdcm_match> rec(matches.size());
    for (size_t i = 0; i < matches.size(); ++i) {
        rec[i].tmpl_idx = matches[i].tmplIdx;
        rec[i].score = matches[i].score;
        for (int c = 0; c < 6; ++c) rec[i].transform[c] = matches[i].transform[(size_t)c];
    }
    const fdcm_coverage_params c = detail::coverage_params(coverage);
    std::vector<float> out(matches.size());
    check(fdcm_match_coverage(fm.handle(), ts, 0, &c, rec.data(), (int64_t)rec.size(), out.data()));
    return out;
}
// fused search -> coverage filter -> top-k (or distinct top-k) [-> pose refinement] on the device
inline std::vector<Match> searchTopK(const DefaultSearch& s, const BatchOptimize& o, const ExponentialPenalty& pen, const Dt3Cuda& fm,
                                     const std::vector<LineArray>& templates, const LineArray& scene, int k, const EdgeCoverage& verify) {
    return detail::search_verify(s, o, pen, fm, templates, scene, k, nullptr, nullptr, verify);
}
inline std::vector<Match> searchTopK(const DefaultSearch& s, const BatchOptimize& o, const ExponentialPenalty& pen, const Dt3Cuda& fm,
                                     const std::vector<LineArray>& templates, const LineArray& scene, int k, const DistinctMatches* select,
                                     const PoseRefinement* refine, const EdgeCoverage& verify) {
    return detail::search_verify(s, o, pen, fm, templates, scene, k, select, refine, verify);
}
// dense search -> coverage filter -> top-k (or distinct top-k) [-> pose refinement] on the device
inline std::vector<Match> searchDense(const Dt3Cuda& fm, const std::vector<LineArray>& templates, const DenseSearch& dense,
                                      const ExponentialPenalty& pen, int k, const DistinctMatches* select, const PoseRefinement* refine,
                                      const EdgeCoverage& verify) {
    const fdcm_coverage_params c = detail::coverage_params(verify);
    return detail::search_dense(fm, templates, dense, FDCM_PENALTY_EXPONENTIAL, pen.tau, k, select, refine, &c);
}
// dense search over a scale grid [-> coverage filter] -> top-k (or distinct top-k) [-> pose refinement] on the device
inline std::vector<Match> searchDense(const Dt3Cuda& fm, const std::vector<LineArray>& templates, const DenseSearch& dense,
                                      const ScaleGrid& scales, const ExponentialPenalty& pen, int k, const DistinctMatches* select = nullptr,
                                      const PoseRefinement* refine = nullptr) {
    return detail::search_dense(fm, templates, dense, FDCM_PENALTY_EXPONENTIAL, pen.tau, k, select, refine, nullptr, &scales);
}
inline std::vector<Match> searchDense(const Dt3Cuda& fm, const std::vector<LineArray>& templates, const DenseSearch& dense,
                                      const ScaleGrid& scales, const ExponentialPenalty& pen, int k, const DistinctMatches* select,
                                      const PoseRefinement* refine, const EdgeCoverage& verify) {
    const fdcm_coverage_params c = detail::coverage_params(verify);
    return detail::search_dense(fm, templates, dense, FDCM_PENALTY_EXPONENTIAL, pen.tau, k, select, refine, &c, &scales);
}

// line-alignment search over a scale grid (rules of fdcm_search_scales): the search of every template scaled by every
// s_k, each match expressed in its original template (tmplIdx), with the scale in the rotation part of its transform
namespace detail {
inline std::vector<Match> search_scales(const DefaultSearch& s, int batch, int penalty_kind, float tau, const Dt3Cuda& fm,
                                        const std::vector<LineArray>& templates, const LineArray& scene, int k, const ScaleGrid& scales,
                                        const DistinctMatches* select, const PoseRefinement* refine, const EdgeCoverage* verify) {
    std::vector<float> flat;
    std::vector<int32_t> off;
    pack(templates, flat, off);
    fdcm_templates* ts = nullptr;
    check(fdcm_templates_create(flat.data(), off.data(), (int32_t)templates.size(), fm.info().device, &ts));
    const std::unique_ptr<fdcm_templates, fdcm_status (*)(fdcm_templates*)> owner(ts, fdcm_templates_release);
    const fdcm_search_params p{(int32_t)s.max_tmpl_lines, (int32_t)s.max_scene_lines, batch, penalty_kind, tau, k, 0, 0, 0.f, 0.f, 0.f, 0.f};
    const fdcm_scale_grid g{scales.scales, scales.start, scales.ratio};
    fdcm_select_params q{};
    if (select) q = fdcm_select_params{select->maxPerTemplate, select->radius, select->maxAngle, select->acrossTemplates ? 1 : 0};
    fdcm_refine_params r{};
    if (refine) r = refine_params(*refine);
    fdcm_coverage_params c{};
    if (verify) c = coverage_params(*verify);
    int64_t cap = k > 0 ? k : 0;   // k == 0: every hypothesis of every copy may match
    if (k <= 0)
        for (const auto& t : templates)
            cap += 2 * (int64_t)std::max(scales.scales, 0) * (int64_t)std::min<size_t>(t.size() / 4, (size_t)s.max_tmpl_lines) *
                   (int64_t)s.max_scene_lines;
    std::vector<fdcm_match> rec((size_t)std::max<int64_t>(cap, 1));
    int64_t n = 0;
    check(fdcm_search_scales(fm.handle(), ts, scene.data(), (int32_t)(scene.size() / 4), &p, &g, select ? &q : nullptr, refine ? &r : nullptr,
                             verify ? &c : nullptr, rec.data(), (int64_t)rec.size(), &n));
    return to_matches(rec, n);
}
}   // namespace detail
// every match of the scaled copies in hypothesis order, nullopt hypotheses dropped
inline std::vector<Match> search(const DefaultMatch&, const DefaultSearch& s, const BatchOptimize& o, const Dt3Cuda& fm,
                                 const std::vector<LineArray>& templates, const LineArray& scene, const ScaleGrid& scales) {
    return detail::search_scales(s, (int)o.batchSize, FDCM_PENALTY_NONE, 0.f, fm, templates, scene, 0, scales, nullptr, nullptr, nullptr);
}
// fused search over a scale grid [-> coverage filter] -> top-k (or distinct top-k) [-> pose refinement] on the device
inline std::vector<Match> searchTopK(const DefaultSearch& s, const BatchOptimize& o, const ExponentialPenalty& pen, const Dt3Cuda& fm,
                                     const std::vector<LineArray>& templates, const LineArray& scene, int k, const ScaleGrid& scales,
                                     const DistinctMatches* select = nullptr, const PoseRefinement* refine = nullptr,
                                     const EdgeCoverage* verify = nullptr) {
    return detail::search_scales(s, (int)o.batchSize, FDCM_PENALTY_EXPONENTIAL, pen.tau, fm, templates, scene, k, scales, select, refine, verify);
}

// pose fit (beyond the reference; rules of fdcm_fit_matches): per match, up to `iterations` Gauss-Newton steps of oriented
// point-to-line least squares of the template's samples against the build scene's line segments (nearest scene line within
// maxDistance pixels on an orientation plane within binTolerance planes).  It needs scene lines near the pose, uses no
// robust loss beyond that gate and does not re-rank; the defaults are a starting point, not tuned.  scaleRange {lo, hi}: the
// scaled fit (fdcm_fit_matches_scaled), which also fits the scale within [lo, hi]; empty: the rigid fit.
struct PoseFit {
    int iterations{10};
    float maxDistance{3.f};
    float sampleStep{2.f};
    int binTolerance{1};
    float tolerance{1e-3f};
    int minInliers{6};
    std::optional<std::pair<float, float>> scaleRange{};
};
struct FitStats {
    int nSamples;
    int nInliers;     // correspondences at the returned pose
    int iterations;   // accepted updates
    float rms;        // root mean square residual of those correspondences (NaN without any)
};
namespace detail {
inline std::vector<Match> fit_matches(const Dt3Cuda& fm, const std::vector<LineArray>& templates, const std::vector<Match>& matches,
                                      const PoseFit& fit, int penalty_kind, float tau, std::vector<FitStats>* stats) {
    std::vector<float> flat;
    std::vector<int32_t> off;
    pack(templates, flat, off);
    fdcm_templates* ts = nullptr;
    check(fdcm_templates_create(flat.data(), off.data(), (int32_t)templates.size(), fm.info().device, &ts));
    const std::unique_ptr<fdcm_templates, fdcm_status (*)(fdcm_templates*)> owner(ts, fdcm_templates_release);
    std::vector<fdcm_match> rec(matches.size());
    for (size_t i = 0; i < matches.size(); ++i) {
        rec[i].tmpl_idx = matches[i].tmplIdx;
        rec[i].score = matches[i].score;
        for (int c = 0; c < 6; ++c) rec[i].transform[c] = matches[i].transform[(size_t)c];
    }
    const fdcm_fit_params p{fit.iterations, fit.maxDistance, fit.sampleStep, fit.binTolerance, fit.tolerance, fit.minInliers};
    std::vector<fdcm_match> out(matches.size());
    std::vector<fdcm_fit_stats> st(stats ? matches.size() : 0);
    if (fit.scaleRange) {
        const fdcm_fit_scale sc{fit.scaleRange->first, fit.scaleRange->second};
        check(fdcm_fit_matches_scaled(fm.handle(), ts, 0, penalty_kind, tau, &p, &sc, rec.data(), (int64_t)rec.size(), out.data(),
                                      stats ? st.data() : nullptr));
    } else {
        check(fdcm_fit_matches(fm.handle(), ts, 0, penalty_kind, tau, &p, rec.data(), (int64_t)rec.size(), out.data(), stats ? st.data() : nullptr));
    }
    if (stats) {
        stats->resize(matches.size());
        for (size_t i = 0; i < st.size(); ++i) (*stats)[i] = FitStats{st[i].n_samples, st[i].n_inliers, st[i].iterations, st[i].rms};
    }
    return to_matches(out, (int64_t)out.size());
}
}   // namespace detail
// fit of every match (tmplIdx indexes `templates`), entry i for matches[i], raw evaluate<Dt3Cpu> score at the fitted pose;
// stats (optional): one FitStats per match
inline std::vector<Match> fitMatches(const Dt3Cuda& fm, const std::vector<LineArray>& templates, const std::vector<Match>& matches,
                                     const PoseFit& fit = PoseFit{}, std::vector<FitStats>* stats = nullptr) {
    return detail::fit_matches(fm, templates, matches, fit, FDCM_PENALTY_NONE, 0.f, stats);
}
// the same, scored with the search's exponential penalty
inline std::vector<Match> fitMatches(const Dt3Cuda& fm, const std::vector<LineArray>& templates, const std::vector<Match>& matches,
                                     const ExponentialPenalty& pen, const PoseFit& fit = PoseFit{}, std::vector<FitStats>* stats = nullptr) {
    return detail::fit_matches(fm, templates, matches, fit, FDCM_PENALTY_EXPONENTIAL, pen.tau, stats);
}

// ---- PenaltyStrategy concept, template lengths, sort ----------------------------------------------
inline std::vector<float> getTemplateLengths(const std::vector<LineArray>& templates) {   // core/math.h:319-324
    std::vector<float> flat, len(templates.size());
    std::vector<int32_t> off;
    detail::pack(templates, flat, off);
    check(fdcm_template_lengths(flat.data(), off.data(), (int32_t)templates.size(), len.data()));
    return len;
}

namespace detail {
inline std::vector<Match> penalize(int kind, float tau, const std::vector<Match>& matches, const std::vector<float>& lengths) {
    std::vector<fdcm_match> rec(matches.size());
    for (size_t i = 0; i < matches.size(); ++i) {
        rec[i].tmpl_idx = matches[i].tmplIdx;
        rec[i].score = matches[i].score;
        for (int k = 0; k < 6; ++k) rec[i].transform[k] = matches[i].transform[(size_t)k];
    }
    check(fdcm_penalize(kind, tau, rec.data(), (int64_t)rec.size(), lengths.data(), (int64_t)lengths.size()));
    std::vector<Match> out = matches;
    for (size_t i = 0; i < out.size(); ++i) out[i].score = rec[i].score;
    return out;
}
}   // namespace detail
inline std::vector<Match> penalize(const DefaultPenalty&, const std::vector<Match>& m, const std::vector<float>& lengths) {
    return detail::penalize(FDCM_PENALTY_DEFAULT, 0.f, m, lengths);
}
inline std::vector<Match> penalize(const ExponentialPenalty& p, const std::vector<Match>& m, const std::vector<float>& lengths) {
    return detail::penalize(FDCM_PENALTY_EXPONENTIAL, p.tau, m, lengths);
}

inline void sortMatches(std::vector<Match>& matches) {   // matchstrategy.h:48-50
    std::vector<fdcm_match> rec(matches.size());
    for (size_t i = 0; i < matches.size(); ++i) {
        rec[i].tmpl_idx = matches[i].tmplIdx;
        rec[i].score = matches[i].score;
        for (int k = 0; k < 6; ++k) rec[i].transform[k] = matches[i].transform[(size_t)k];
    }
    check(fdcm_sort_matches(rec.data(), (int64_t)rec.size()));
    for (size_t i = 0; i < matches.size(); ++i) {
        matches[i].tmplIdx = rec[i].tmpl_idx;
        matches[i].score = rec[i].score;
        for (int k = 0; k < 6; ++k) matches[i].transform[(size_t)k] = rec[i].transform[k];
    }
}

}   // namespace openfdcm::cuda
