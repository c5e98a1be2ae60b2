"""Pose fit (fdcm_fit_matches, PoseFit): the properties of the float64 model of tests/models/fit.py, and the host hook
fdcm_fit_samples against it.  tests/test_gpu_fit.py compares the device against this model byte for byte.  No kernel is
launched here."""
import ctypes as C
import math

import numpy as np
import pytest

import openfdcm_b200 as fdcm
from openfdcm_b200 import _lib
from tests.helpers import anchor_of, house, offset_pose, one_match, pose, pose_errors, posed, scene_of
from tests.models.fit import fit_model, fit_one, line_samples
from tests.models.refine import valid_poses
from tests.util import F32


# ---- the tests -------------------------------------------------------------------------------------------------------
def test_struct_layouts_match_the_header():
    assert C.sizeof(_lib.FitParams) == 24
    assert [f[0] for f in _lib.FitParams._fields_] == ["iterations", "max_distance", "sample_step", "bin_tolerance", "tolerance",
                                                      "min_inliers"]
    assert _lib.FIT_STATS_DTYPE.itemsize == 16 and _lib.FIT_STATS_DTYPE.names == ("n_samples", "n_inliers", "iterations", "rms")
    f = fdcm.PoseFit()
    assert (f.iterations, f.max_distance, f.sample_step, f.bin_tolerance, f.tolerance, f.min_inliers) == (10, 3.0, 2.0, 1, 1e-3, 6)


def hook_samples(lines, step):
    rec = np.ascontiguousarray(np.asarray(lines, F32).reshape(-1, 4))
    n = C.c_int64(0)
    _lib.lib().fdcm_fit_samples(_lib.ptr(rec), rec.shape[0], step, None, 0, C.byref(n))
    out = np.zeros((max(n.value, 1), 2), np.float64)
    _lib.check(_lib.lib().fdcm_fit_samples(_lib.ptr(rec), rec.shape[0], step, _lib.ptr(out), n.value, C.byref(n)))
    return out[: n.value]


def test_fit_samples_hook_equals_the_model():
    rng = np.random.default_rng(5)
    lines = np.concatenate([
        np.array([[0, 0, 10, 0],            # len 10, step 2: n = 6 (an exact multiple)
                  [3, 3, 3, 3],             # zero length: no samples
                  [1, 1, 1, 9],             # len 8, step 2: n = 5
                  [0.5, 0.25, 7.3, 9.1],
                  [-4, 2, -4.0000005, 2]], F32),
        rng.uniform(-300, 300, (40, 4)).astype(F32)])
    for step in (0.5, 1.0, 2.0, 3.7, 1e30):
        want = [np.stack(line_samples(l, step), axis=1) for l in lines]
        got = hook_samples(lines, step)
        want = np.concatenate(want)
        assert got.shape == want.shape and got.tobytes() == want.tobytes()
    assert len(line_samples([0, 0, 10, 0], 2.0)[0]) == 6 and len(line_samples([3, 3, 3, 3], 2.0)[0]) == 0
    assert len(line_samples([0, 0, 10, 0], 1e30)[0]) == 2
    s = hook_samples([[0, 0, 10, 0]], 2.0)
    assert s[:, 0].tolist() == [0.0, 2.0, 4.0, 6.0, 8.0, 10.0] and (s[:, 1] == 0).all()
    n = C.c_int64(0)
    assert _lib.lib().fdcm_fit_samples(_lib.ptr(lines), len(lines), 2.0, None, 0, C.byref(n)) == _lib.FDCM_ERR_CAPACITY
    assert _lib.lib().fdcm_fit_samples(_lib.ptr(lines), len(lines), 0.25, None, 0, C.byref(n)) == _lib.FDCM_ERR_INVALID


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_model_recovers_the_exact_pose_of_noise_free_lines(seed):
    rng = np.random.default_rng(seed)
    tmpl = house()
    a = anchor_of(tmpl)
    truth = pose(rng.uniform(-math.pi, math.pi), rng.uniform(150, 250), rng.uniform(150, 250))
    sc = scene_of(posed(tmpl, truth))
    ang = rng.choice([-1, 1]) * 0.03
    d = rng.normal(size=2)
    d = 2.0 * d / np.hypot(*d)
    start = offset_pose(truth, a, ang, d[0], d[1])
    out, st = fit_model(sc, [tmpl], [a], one_match(start), fdcm.PoseFit())
    e_a, e_r, _ = pose_errors(out[0]["transform"], truth, a)
    assert e_a < 0.01 and e_r < 1e-4, (e_a, e_r, st)
    assert st[0]["n_inliers"] == st[0]["n_samples"] and st[0]["iterations"] >= 2 and st[0]["rms"] < 0.01


def test_model_recovers_the_pose_on_cut_scene_lines():
    """Every scene line cut into 2-3 pieces with gaps: the samples over a gap have no correspondence (or one at a piece's
    end), the rest still determine the pose."""
    rng = np.random.default_rng(11)
    tmpl = house()
    a = anchor_of(tmpl)
    truth = pose(0.7, 200.0, 190.0)
    full = posed(tmpl, truth).T.astype(np.float64)
    pieces = []
    for x1, y1, x2, y2 in full:
        k = int(rng.integers(2, 4))
        cuts = np.sort(rng.uniform(0.15, 0.85, k - 1))
        edges = [0.0] + [v for c in cuts for v in (c - 0.04, c + 0.04)] + [1.0]
        for u0, u1 in zip(edges[::2], edges[1::2]):
            pieces.append((x1 + (x2 - x1) * u0, y1 + (y2 - y1) * u0, x1 + (x2 - x1) * u1, y1 + (y2 - y1) * u1))
    sc = scene_of(np.asarray(pieces, F32).T)
    start = offset_pose(truth, a, -0.03, 1.2, -1.6)
    out, st = fit_model(sc, [tmpl], [a], one_match(start), fdcm.PoseFit(iterations=20))
    e_a, e_r, _ = pose_errors(out[0]["transform"], truth, a)
    assert e_a < 0.01 and e_r < 1e-4, (e_a, e_r, st)
    assert st[0]["n_inliers"] >= st[0]["n_samples"] // 2


def test_model_does_not_slide_a_template_of_parallel_lines():
    """Parallel lines leave the translation along them unobserved: g has no component there and the damping keeps the
    step out of that direction."""
    th = 0.4
    u = np.array([math.cos(th), math.sin(th)])
    tmpl = np.array([[0, 0, 80, 0], [0, 15, 80, 15], [0, 40, 80, 40]], F32).T.copy()
    a = anchor_of(tmpl)
    truth = pose(th, 180.0, 170.0)
    sc = scene_of(posed(tmpl, truth))
    for dth, perp in ((0.0, 1.5), (0.02, -1.0)):
        n = np.array([-u[1], u[0]])
        start = offset_pose(truth, a, dth, *(perp * n + 3.0 * u))   # 3 px along the lines, `perp` across
        out, st = fit_model(sc, [tmpl], [a], one_match(start), fdcm.PoseFit())
        _, e_r, off = pose_errors(out[0]["transform"], truth, a)
        assert abs(float(off @ n)) < 0.01 and e_r < 1e-4 and st[0]["iterations"] >= 1
        # the float64 pose state, before the float32 rounding of the output (1.5e-5 px at these coordinates)
        m0, m1, m3, m4, ex, ey = fit_one(sc, tmpl, a, start, fdcm.PoseFit())[2]
        ax, ay = float(a[0]), float(a[1])
        moved = np.array([(m0 * ax + m1 * ay) + ex, (m3 * ax + m4 * ay) + ey])
        T0 = start.astype(np.float64)
        start_anchor = np.array([(T0[0] * ax + T0[1] * ay) + T0[2], (T0[3] * ax + T0[4] * ay) + T0[5]])
        # started parallel, the step has no component along the lines; started 0.02 rad off, the first steps are normal to
        # the posed lines, which are not yet parallel to the scene's
        assert abs(float((moved - start_anchor) @ u)) < (1e-6 if dth == 0.0 else 2.0 * math.sin(abs(dth))), moved - start_anchor


def test_model_edge_cases():
    tmpl = house()
    a = anchor_of(tmpl)
    truth = pose(0.3, 200.0, 200.0)
    sc = scene_of(posed(tmpl, truth))
    fit = fdcm.PoseFit()
    # invalid inputs come back unchanged with score NaN and stats {0, 0, 0, NaN}
    bad = np.concatenate([one_match(truth.astype(F32)), one_match([np.nan, 0, 200, 0, 1, 200]), one_match([1, 0, 1e5, 0, 1, 0]),
                          one_match(truth.astype(F32), t=1)])
    out, st = fit_model(sc, [tmpl, np.zeros((4, 0), F32)], [a, (0.0, 0.0)], bad, fit)
    assert np.array_equal(out[1:]["transform"].view(np.uint32), bad[1:]["transform"].view(np.uint32))
    assert np.isnan(out[1:]["score"]).all() and st[1:]["n_samples"].tolist() == [0, 0, 0] and np.isnan(st[1:]["rms"]).all()
    # no scene line within max_distance: no update, the input transform itself
    far = offset_pose(truth, a, 0.0, 100.0, 0.0)
    out, st = fit_model(sc, [tmpl], [a], one_match(far), fit)
    assert out[0]["transform"].tobytes() == far.tobytes() and st[0]["iterations"] == 0 and st[0]["n_inliers"] < 6
    # a pose at the map border whose update would leave the map stops at the last valid pose
    edge = scene_of(posed(tmpl, pose(0.0, -1.0, 100.0)), W=400, H=400)   # the instance sticks out of the map by 1 px
    start = np.array([1, 0, 0.0, 0, 1, 100.0], F32)
    out, st = fit_model(edge, [tmpl], [a], one_match(start), fit)
    assert valid_poses(out["transform"], tmpl, edge.shift, edge.W, edge.H)[0] and out[0]["transform"][2] >= 0.0


@pytest.mark.parametrize("bad", [dict(iterations=0), dict(iterations=101), dict(max_distance=0.0), dict(max_distance=16.5),
                                 dict(max_distance=math.nan), dict(sample_step=0.4), dict(sample_step=math.inf),
                                 dict(bin_tolerance=-1), dict(bin_tolerance=33), dict(tolerance=-1e-3), dict(tolerance=math.nan),
                                 dict(min_inliers=2)])
def test_fit_matches_rejects_bad_parameters_before_any_device_work(bad):
    f = fdcm.PoseFit(**bad)
    st = _lib.lib().fdcm_fit_matches(None, None, 0, 0, 0.0, C.byref(f._params()), None, 0, None, None)
    assert st == _lib.FDCM_ERR_INVALID
    msg = _lib.lib().fdcm_last_error().decode()
    assert "pose fit" in msg, msg


def test_cpp_fit_matches_builds(tmp_path):
    """fitMatches of include/openfdcm_b200/openfdcm_cuda.hpp compiles and links."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "fit.cpp"
    src.write_text(r'''
#include "openfdcm_b200/openfdcm_cuda.hpp"
#include <cstdio>
int main() {
    using namespace openfdcm::cuda;
    try {
        const LineArray scene{0.f, 0.f, 50.f, 0.f, 50.f, 0.f, 50.f, 40.f};
        const std::vector<LineArray> templates{LineArray{0.f, 0.f, 20.f, 0.f}};
        const Dt3Cuda fm = buildCudaFeaturemap(scene, Dt3CudaParameters{});
        const auto a = searchTopK(DefaultSearch{4, 4}, BatchOptimize{10}, ExponentialPenalty{1.5f}, fm, templates, scene, 5);
        const PoseFit fit{};
        const std::vector<Match> b = fitMatches(fm, templates, a, fit);
        std::vector<FitStats> stats;
        const std::vector<Match> c = fitMatches(fm, templates, a, PoseFit{5, 2.f, 1.f, 1, 1e-3f, 6}, &stats);
        std::printf("%zu %zu %zu %zu\n", a.size(), b.size(), c.size(), stats.size());
    } catch (const std::exception& e) {
        std::printf("%s\n", e.what());
        return 1;
    }
    return 0;
}
''')
    exe = tmp_path / "fit"
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Werror", "-I" + os.path.join(root, "include"), str(src),
                           "-L" + os.path.join(root, "openfdcm_b200"), "-lfdcm_b200", "-Wl,-rpath," + os.path.join(root, "openfdcm_b200"),
                           "-o", str(exe)])
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode in (0, 1) and r.stdout
