"""Scale as a pose dimension (fdcm_search_dense_scales, ScaleGrid; fdcm_fit_matches_scaled, PoseFit(scale_range=...)): the
scale grid of the dense model (tests/models/dense.py) and the scaled fit of the float64 model (tests/models/fit.py), the
host hook fdcm_dense_scaled_poses against the model bit for bit, and parameter rejection.  The rules are in
include/fdcm_b200.h; tests/test_gpu_scale.py compares the device against these models.  No kernel is launched here."""
import ctypes as C
import math

import numpy as np
import pytest

import openfdcm_b200 as fdcm
from openfdcm_b200 import _lib
from openfdcm_b200._lib import MATCH_DTYPE
from tests.helpers import anchor_of, dense_poses_hook, house, one_match, pose_errors, posed, scale_error, scene_of, spose
from tests.models.dense import grid, poses, rot_table, scale_values
from tests.models.fit import fit_model, fit_one, sigma_of
from tests.models.select import select_model
from tests.util import F32


def offset_similarity(truth, anchor, dth, ds, dx, dy):
    """truth rotated by dth and scaled by (1 + ds) about its posed anchor, then moved by (dx, dy)."""
    T = np.asarray(truth, np.float64).reshape(2, 3)
    a = T @ np.array([float(anchor[0]), float(anchor[1]), 1.0])
    R = (1.0 + ds) * np.array([[math.cos(dth), -math.sin(dth)], [math.sin(dth), math.cos(dth)]])
    M = R @ T[:, :2]
    e = R @ (T[:, 2] - a) + a + np.array([dx, dy])
    return np.array([M[0, 0], M[0, 1], e[0], M[1, 0], M[1, 1], e[1]], F32)


# ---- the tests -------------------------------------------------------------------------------------------------------
def test_struct_layouts_match_the_header():
    assert C.sizeof(_lib.ScaleGridParams) == 12
    assert [(f, getattr(_lib.ScaleGridParams, f).offset) for f, _ in _lib.ScaleGridParams._fields_] == [
        ("scales", 0), ("scale_start", 4), ("scale_ratio", 8)]
    assert C.sizeof(_lib.FitScaleParams) == 8
    assert [(f, getattr(_lib.FitScaleParams, f).offset) for f, _ in _lib.FitScaleParams._fields_] == [("min_scale", 0), ("max_scale", 4)]
    # the existing structs keep their layouts
    assert C.sizeof(_lib.DenseParams) == 40 and C.sizeof(_lib.FitParams) == 24
    g = fdcm.ScaleGrid()
    assert (g.scales, g.start, g.ratio) == (1, 1.0, 1.0)
    assert fdcm.PoseFit().scale_range is None and fdcm.PoseFit(scale_range=(0.5, 2)).scale_range == (0.5, 2.0)
    assert _lib.lib().fdcm_abi_version() == 3


GRIDS = [fdcm.ScaleGrid(1, 1.0, 1.0), fdcm.ScaleGrid(3, 0.85, (1.15 / 0.85) ** 0.5),
         fdcm.ScaleGrid(5, 0.8, (1.25 / 0.8) ** 0.25), fdcm.ScaleGrid(4, 2.5, 0.5), fdcm.ScaleGrid(2, 1.0, 1.1)]


@pytest.mark.parametrize("g", GRIDS, ids=str)
def test_scaled_poses_hook_equals_the_model(g):
    rng = np.random.default_rng(3)
    for d, shift, W, H in ((fdcm.DenseSearch(7, rot_start=0.1, stride=3, cell=4), (12.5, -3.25), 120, 90),
                           (fdcm.DenseSearch(1, rot_start=0.0, stride=1, cell=2), (0.0, 0.0), 40, 30),
                           (fdcm.DenseSearch(12, stride=5, cell=1, roi=(-10.0, 5.5, 60.0, 70.0)), (20.0, 10.0), 100, 100)):
        anchor = rng.uniform(-30, 30, 2).astype(F32)
        for k in range(g.scales):
            for r in range(d.rotations):
                st, got, n, wh = dense_poses_hook(d, anchor, shift, W, H, r, g=g, k=k)
                assert st == 0, _lib.lib().fdcm_last_error()
                want = poses(d, anchor, shift, W, H, r, g, k)
                assert got.tobytes() == want.tobytes(), (g, d, k, r)
                assert wh == grid(d, shift, W, H)[2:]


def test_scale_one_equals_the_unscaled_grid():
    """With s_k == 1.0f the table is rule 1's (c_r, s_r) bit for bit, so the poses are fdcm_dense_poses's."""
    d = fdcm.DenseSearch(24, rot_start=0.3, stride=2, cell=3)
    for g in (fdcm.ScaleGrid(), fdcm.ScaleGrid(1, 1.0, 7.0), fdcm.ScaleGrid(3, 1.0, 1.5)):
        A, B = rot_table(d, g)
        for r in range(d.rotations):
            th = float(F32(0.3)) + r * float(F32(d.rot_step))
            assert A[0, r] == F32(math.cos(th)) and B[0, r] == F32(math.sin(th))
            st0, p0, _, _ = dense_poses_hook(d, (3.5, -2.0), (7.0, 4.0), 64, 48, r)
            st1, p1, _, _ = dense_poses_hook(d, (3.5, -2.0), (7.0, 4.0), 64, 48, r, g=g, k=0)
            assert st0 == st1 == 0 and p0.tobytes() == p1.tobytes()
    # the identity slice uses the end points as given, like the unscaled theta = 0 slice
    d1 = fdcm.DenseSearch(1, rot_start=0.0)
    A, B = rot_table(d1, fdcm.ScaleGrid())
    assert A[0, 0] == F32(1) and B[0, 0] == F32(0)


def test_scale_values_are_host_double_pow():
    g = fdcm.ScaleGrid(6, 0.7, 1.13)
    want = [F32(float(F32(0.7)) * math.pow(float(F32(1.13)), k)) for k in range(6)]
    assert scale_values(g).tolist() == [float(v) for v in want]
    A, B = rot_table(fdcm.DenseSearch(1, rot_start=0.0), g)
    assert A[:, 0].tobytes() == scale_values(g).tobytes() and (B == 0).all()


def test_scaled_select_model_reduces_to_the_walk_at_scale_one():
    rng = np.random.default_rng(9)
    n = 200
    rec = np.zeros(n, MATCH_DTYPE)
    rec["tmpl_idx"] = rng.integers(0, 4, n)
    rec["score"] = rng.uniform(0, 10, n).astype(F32)
    th = rng.uniform(-0.5, 0.5, n)
    rec["transform"] = np.stack([np.cos(th), -np.sin(th), rng.uniform(0, 30, n), np.sin(th), np.cos(th), rng.uniform(0, 30, n)], 1)
    anchors = rng.uniform(-5, 5, (4, 2)).astype(F32)
    ones = np.ones(n, F32)
    for kw in (dict(radius=8.0, max_angle=0.2), dict(radius=8.0, max_angle=0.2, across_templates=True), dict(max_per_template=3)):
        assert select_model(rec, anchors, 20, rs=ones, **kw).tolist() == select_model(rec, anchors, 20, **kw).tolist()
    # at scale 1.2 the rotation column has length 1.2: the threshold scales with the two scales, so the test stays an angle test
    r2 = rec.copy()
    r2["transform"][:, [0, 1, 3, 4]] *= F32(1.2)
    s12 = np.full(n, F32(1.2))
    kw = dict(radius=8.0, max_angle=0.2)
    assert len(select_model(r2, anchors, 20, rs=s12, **kw)) == len(select_model(rec, anchors, 20, **kw))


BAD_GRIDS = [fdcm.ScaleGrid(0), fdcm.ScaleGrid(65), fdcm.ScaleGrid(2, 0.0, 1.0), fdcm.ScaleGrid(2, -1.0, 1.0), fdcm.ScaleGrid(2, math.nan, 1.0),
             fdcm.ScaleGrid(2, math.inf, 1.0), fdcm.ScaleGrid(2, 1.0, 0.0), fdcm.ScaleGrid(2, 1.0, -2.0), fdcm.ScaleGrid(2, 1.0, math.nan),
             fdcm.ScaleGrid(64, 1.0, 1e10),    # s_k overflows float32
             fdcm.ScaleGrid(64, 1.0, 1e-10)]   # s_k underflows to 0


@pytest.mark.parametrize("g", BAD_GRIDS, ids=str)
def test_bad_scale_grids_are_rejected_before_any_device_work(g):
    d = fdcm.DenseSearch(4)
    st, _, _, _ = dense_poses_hook(d, (0.0, 0.0), (0.0, 0.0), 10, 10, 0, capacity=0, g=g)
    assert st == _lib.FDCM_ERR_INVALID
    assert "scale" in _lib.lib().fdcm_last_error().decode()
    n = C.c_int64(7)
    st = _lib.lib().fdcm_search_dense_scales(None, None, C.byref(d._params()), C.byref(g._params()), 0, 0.0, 10, 0, None, None, None, None,
                                             0, C.byref(n))
    assert st == _lib.FDCM_ERR_INVALID


def test_scaled_hook_rejects_bad_arguments():
    d, g = fdcm.DenseSearch(4), fdcm.ScaleGrid(3, 0.9, 1.1)
    for k, r in ((-1, 0), (3, 0), (0, -1), (0, 4)):
        assert dense_poses_hook(d, (0.0, 0.0), (0.0, 0.0), 10, 10, r, capacity=100, g=g, k=k)[0] == _lib.FDCM_ERR_INVALID
    assert dense_poses_hook(fdcm.DenseSearch(0), (0.0, 0.0), (0.0, 0.0), 10, 10, 0, capacity=100, g=g)[0] == _lib.FDCM_ERR_INVALID
    st, _, n, _ = dense_poses_hook(d, (0.0, 0.0), (0.0, 0.0), 10, 10, 0, capacity=3, g=g)
    assert st == _lib.FDCM_ERR_CAPACITY and n == 25   # (stride 2: 5 x 5 points)
    n = C.c_int64(7)
    assert _lib.lib().fdcm_search_dense_scales(None, None, C.byref(d._params()), None, 0, 0.0, 10, 0, None, None, None, None, 0,
                                               C.byref(n)) == _lib.FDCM_ERR_INVALID


@pytest.mark.parametrize("rng_", [(0.0, 1.0), (-1.0, 1.0), (1.2, 1.1), (math.nan, 1.0), (1.0, math.inf), (0.5, math.nan)])
def test_fit_matches_scaled_rejects_bad_scale_ranges(rng_):
    f = fdcm.PoseFit(scale_range=rng_)
    sc = _lib.FitScaleParams(*f.scale_range)
    st = _lib.lib().fdcm_fit_matches_scaled(None, None, 0, 0, 0.0, C.byref(f._params()), C.byref(sc), None, 0, None, None)
    assert st == _lib.FDCM_ERR_INVALID and "scale" in _lib.lib().fdcm_last_error().decode()
    # and the fit parameters are checked as for the rigid fit
    bad = fdcm.PoseFit(iterations=0, scale_range=(0.5, 2.0))
    sc = _lib.FitScaleParams(0.5, 2.0)
    assert _lib.lib().fdcm_fit_matches_scaled(None, None, 0, 0, 0.0, C.byref(bad._params()), C.byref(sc), None, 0, None, None) == 1
    assert _lib.lib().fdcm_fit_matches_scaled(None, None, 0, 0, 0.0, C.byref(fdcm.PoseFit()._params()), None, None, 0, None, None) == 1


FIT = fdcm.PoseFit(iterations=20, scale_range=(0.5, 2.0))


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_model_recovers_a_scaled_instance(seed):
    """A noise-free instance at s = 1.07, started at s = 1.0 about 1 px and 0.02 rad off."""
    rng = np.random.default_rng(seed)
    tmpl = house()
    a = anchor_of(tmpl)
    truth = spose(rng.uniform(-math.pi, math.pi), 1.07, rng.uniform(150, 250), rng.uniform(150, 250))
    sc = scene_of(posed(tmpl, truth))
    d = rng.normal(size=2)
    d = d / np.hypot(*d)
    start = offset_similarity(truth, a, rng.choice([-1, 1]) * 0.02, 1.0 / 1.07 - 1.0, d[0], d[1])
    assert abs(sigma_of((start[0], start[1], start[3], start[4])) - 1.0) < 1e-6
    out, st = fit_model(sc, [tmpl], [a], one_match(start), FIT)
    e_a, e_r, _ = pose_errors(out[0]["transform"], truth, a)
    assert e_a < 1e-4 and scale_error(out[0]["transform"], truth) < 1e-6 and e_r < 1e-6, (e_a, e_r, st)
    assert st[0]["n_inliers"] == st[0]["n_samples"] and st[0]["iterations"] >= 2 and st[0]["rms"] < 1e-4


def test_model_rigid_fit_keeps_the_scale():
    """The rigid fit on the same start keeps s = 1: it cannot reach the instance at 1.07."""
    tmpl = house()
    a = anchor_of(tmpl)
    truth = spose(0.4, 1.07, 200.0, 190.0)
    sc = scene_of(posed(tmpl, truth))
    start = offset_similarity(truth, a, 0.02, 1.0 / 1.07 - 1.0, 0.6, -0.8)
    rigid, _ = fit_model(sc, [tmpl], [a], one_match(start), fdcm.PoseFit(iterations=20))
    assert abs(math.sqrt(float(rigid[0]["transform"][0]) ** 2 + float(rigid[0]["transform"][3]) ** 2) - 1.0) < 1e-6
    assert scale_error(rigid[0]["transform"], truth) > 0.05


def test_model_stops_at_max_scale():
    """The truth at s = 1.2 lies beyond max_scale = 1.1: no accepted pose has a scale above the bound."""
    tmpl = house()
    a = anchor_of(tmpl)
    truth = spose(0.3, 1.2, 200.0, 200.0)
    sc = scene_of(posed(tmpl, truth))
    start = offset_similarity(truth, a, 0.0, 1.0 / 1.2 - 1.0, 0.5, 0.5)
    fit = fdcm.PoseFit(iterations=20, scale_range=(0.9, 1.1))
    out, st = fit_model(sc, [tmpl], [a], one_match(start), fit)
    P = fit_one(sc, tmpl, a, start, fit)[2]
    assert sigma_of(P) <= float(F32(1.1)) and sigma_of(P) > 1.0
    assert st[0]["iterations"] < 20
    # the next step would have left the range: an unbounded fit goes past 1.1
    free = fit_one(sc, tmpl, a, start, fdcm.PoseFit(iterations=20, scale_range=(0.5, 2.0)))[2]
    assert abs(sigma_of(free) - 1.2) < 1e-6


def test_model_does_not_drift_a_template_of_parallel_lines():
    """Parallel lines leave the translation along them unobserved; their spacing fixes the scale.  The fit recovers the
    scale and the normal offset and does not slide along the lines."""
    th = 0.4
    u = np.array([math.cos(th), math.sin(th)])
    n = np.array([-u[1], u[0]])
    tmpl = np.array([[0, 0, 80, 0], [0, 15, 80, 15], [0, 40, 80, 40]], F32).T.copy()
    a = anchor_of(tmpl)
    for s_true in (1.0, 1.05):
        truth = spose(th, s_true, 180.0, 170.0)
        sc = scene_of(posed(tmpl, truth))
        start = offset_similarity(truth, a, 0.0, 1.0 / s_true - 1.0, *(1.0 * n + 3.0 * u))
        out, st = fit_model(sc, [tmpl], [a], one_match(start), FIT)
        _, e_r, off = pose_errors(out[0]["transform"], truth, a)
        assert abs(float(off @ n)) < 0.01 and e_r < 1e-4 and scale_error(out[0]["transform"], truth) < 1e-4, (off, e_r, st)
        m0, m1, m3, m4, ex, ey = fit_one(sc, tmpl, a, start, FIT)[2]
        ax, ay = float(a[0]), float(a[1])
        moved = np.array([(m0 * ax + m1 * ay) + ex, (m3 * ax + m4 * ay) + ey])
        T0 = start.astype(np.float64)
        start_anchor = np.array([(T0[0] * ax + T0[1] * ay) + T0[2], (T0[3] * ax + T0[4] * ay) + T0[5]])
        assert abs(float((moved - start_anchor) @ u)) < 1e-6, moved - start_anchor


def test_model_edge_cases():
    tmpl = house()
    a = anchor_of(tmpl)
    truth = spose(0.3, 1.1, 200.0, 200.0)
    sc = scene_of(posed(tmpl, truth))
    bad = np.concatenate([one_match([np.nan, 0, 200, 0, 1, 200]), one_match([1, 0, 1e5, 0, 1, 0]), one_match(truth.astype(F32), t=1)])
    out, st = fit_model(sc, [tmpl, np.zeros((4, 0), F32)], [a, (0.0, 0.0)], bad, FIT)
    assert np.array_equal(out["transform"].view(np.uint32), bad["transform"].view(np.uint32))
    assert np.isnan(out["score"]).all() and st["n_samples"].tolist() == [0, 0, 0]
    far = offset_similarity(truth, a, 0.0, 0.0, 100.0, 0.0)
    out, st = fit_model(sc, [tmpl], [a], one_match(far), FIT)
    assert out[0]["transform"].tobytes() == far.tobytes() and st[0]["iterations"] == 0


def test_cpp_scale_mirror_builds(tmp_path):
    """ScaleGrid, the searchDense overloads that take it and PoseFit::scaleRange of include/openfdcm_b200/openfdcm_cuda.hpp
    compile and link; the existing aggregate initialisation of PoseFit still compiles."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "scale.cpp"
    src.write_text(r'''
#include "openfdcm_b200/openfdcm_cuda.hpp"
#include <cstdio>
int main() {
    using namespace openfdcm::cuda;
    try {
        const LineArray scene{0.f, 0.f, 50.f, 0.f, 50.f, 0.f, 50.f, 40.f};
        const std::vector<LineArray> templates{LineArray{0.f, 0.f, 20.f, 0.f}};
        const Dt3Cuda fm = buildCudaFeaturemap(scene, Dt3CudaParameters{});
        const DistinctMatches one{1, 0.f, 3.14159274f, false};
        const auto a = searchDense(fm, templates, DenseSearch{}, ScaleGrid{3, 0.9f, 1.1f}, ExponentialPenalty{1.5f}, 5);
        const auto b = searchDense(fm, templates, DenseSearch{}, ScaleGrid{}, ExponentialPenalty{1.5f}, 5, &one, nullptr, EdgeCoverage{});
        PoseFit fit{5, 2.f, 1.f, 1, 1e-3f, 6};
        fit.scaleRange = std::make_pair(0.8f, 1.25f);
        std::vector<FitStats> stats;
        const std::vector<Match> c = fitMatches(fm, templates, a, fit, &stats);
        std::printf("%zu %zu %zu %zu\n", a.size(), b.size(), c.size(), stats.size());
    } catch (const std::exception& e) {
        std::printf("%s\n", e.what());
        return 1;
    }
    return 0;
}
''')
    exe = tmp_path / "scale"
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Werror", "-I" + os.path.join(root, "include"), str(src),
                           "-L" + os.path.join(root, "openfdcm_b200"), "-lfdcm_b200", "-Wl,-rpath," + os.path.join(root, "openfdcm_b200"),
                           "-o", str(exe)])
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode in (0, 1) and r.stdout
