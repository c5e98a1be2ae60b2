"""Pose fit on the device (fdcm_fit_matches, fit_matches, search_topk / search_dense with fit=): byte-equal to the float64
model of tests/models/fit.py, and the model's recovery properties on the device."""
import math
import threading

import numpy as np
import pytest

import openfdcm_b200 as fdcm
from openfdcm_b200 import _lib
from tests.helpers import device_scores, fit_candidates, house, load_object, offset_pose, pose, pose_errors, posed, synthetic
from tests.models.fit import SceneLines, fit_model
from tests.models.refine import rotated, valid_poses
from tests.util import F32, synth_scene, synth_templates

pytestmark = pytest.mark.gpu

S, O, P = fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), fdcm.ExponentialPenalty(1.5)


def model(fm, scene, tmpls, matches, fit, penalty=None, tmpl_idx_base=0):
    sc = SceneLines.of(scene, fm.get_scene_translation(), fm.scene_bins(), fm.depth, fm.width, fm.height)
    scores = device_scores(fm)
    out, stats = fit_model(sc, tmpls, fdcm.get_template_anchors(tmpls), matches, fit,
                           lambda tmpl, F: scores([(tmpl, F.reshape(1, 6))])[0], tmpl_idx_base)
    if penalty is not None:
        out["tmpl_idx"] -= tmpl_idx_base
        out = fdcm.penalize(penalty, out, fdcm.get_template_lengths(tmpls))
        out["tmpl_idx"] += tmpl_idx_base
    return out, stats


def check_fit(fm, scene, tmpls, matches, fit, penalty=None, tmpl_idx_base=0):
    got, gst = fdcm.fit_matches(fm, tmpls, matches, fit, penalty, tmpl_idx_base, return_stats=True)
    want, wst = model(fm, scene, tmpls, matches, fit, penalty, tmpl_idx_base)
    assert got.dtype == fdcm.MATCH_DTYPE and got.shape == (len(matches),)
    bad = np.flatnonzero([a.tobytes() != b.tobytes() for a, b in zip(got, want)])
    assert len(bad) == 0, (bad[:5], got[bad[:2]], want[bad[:2]])
    assert gst.tobytes() == wst.tobytes(), np.flatnonzero([a.tobytes() != b.tobytes() for a, b in zip(gst, wst)])[:10]
    return got, gst


@pytest.mark.parametrize("dist", [fdcm.distance.L2, fdcm.distance.L2_SQUARED, fdcm.distance.L1])
def test_synthetic_scenes_against_the_model(dist):
    tmpls, scene = synthetic(n_tmpl=10, seed=500)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5, dist))
    m = fit_candidates(fm, tmpls, scene, 30)
    got, st = check_fit(fm, scene, tmpls, m, fdcm.PoseFit(), P)
    assert np.isnan(got[-3:]["score"]).all() and (st["iterations"][:-3] > 0).any()
    check_fit(fm, scene, tmpls, m[::3], fdcm.PoseFit(iterations=3, max_distance=6.0, sample_step=0.75, bin_tolerance=0, min_inliers=3))


def test_odd_depth_and_tmpl_idx_base():
    tmpls, scene = synthetic(n_tmpl=6, seed=510)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(7, 5.0, 1.5))
    m = fit_candidates(fm, tmpls, scene, 20)
    m["tmpl_idx"] += 100
    check_fit(fm, scene, tmpls, m, fdcm.PoseFit(bin_tolerance=2), tmpl_idx_base=100)


def test_literal_path_map():
    tmpls = synth_templates(4, 12, 2000, seed=520)
    scene = synth_scene(3000, 3000, 120, seed=521)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.05))
    assert fm.width > 2897
    check_fit(fm, scene, tmpls, fit_candidates(fm, tmpls, scene, 12), fdcm.PoseFit(max_distance=16.0))


@pytest.mark.parametrize("obj", ["obj_01", "obj_02", "obj_03", "obj_04"])
def test_real_assets(obj):
    tmpls, scenes = load_object(obj)
    fm = fdcm.build_cuda_featuremap(scenes[0], fdcm.Dt3CudaParameters(30, 5.0, 2.2))
    check_fit(fm, scenes[0], tmpls, fit_candidates(fm, tmpls, scenes[0], 10, seed=1), fdcm.PoseFit(), P)


# ---- the model's properties on the device ----------------------------------------------------------------------------
def instance_map(tmpl, truth, extra=()):
    scene = np.concatenate([posed(tmpl, truth)] + list(extra), axis=1)
    return scene, fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))


def test_recovers_the_exact_pose_of_noise_free_lines():
    tmpl = house()
    a = fdcm.get_template_anchors([tmpl])[0]
    rng = np.random.default_rng(530)
    for q in range(4):
        truth = pose(rng.uniform(-math.pi, math.pi), rng.uniform(100, 300), rng.uniform(100, 300))
        scene, fm = instance_map(tmpl, truth, [synth_scene(400, 400, 30, seed=531 + q)])
        d = rng.normal(size=2)
        d = 2.0 * d / np.hypot(*d)
        start = offset_pose(truth, a, 0.03 if q % 2 else -0.03, d[0], d[1])
        m = np.zeros(1, fdcm.MATCH_DTYPE)
        m["transform"] = start
        got, st = check_fit(fm, scene, [tmpl], m, fdcm.PoseFit())
        e_a, e_r, _ = pose_errors(got[0]["transform"], truth, a)
        assert e_a < 0.01 and e_r < 1e-4, (e_a, e_r, st)


def test_cut_lines_and_parallel_lines():
    tmpl = house()
    a = fdcm.get_template_anchors([tmpl])[0]
    truth = pose(-1.1, 200.0, 210.0)
    full = posed(tmpl, truth).T.astype(np.float64)
    pieces = []
    for x1, y1, x2, y2 in full:   # three pieces, gaps of 6 % of the length
        for u0, u1 in ((0.0, 0.3), (0.36, 0.62), (0.68, 1.0)):
            pieces.append((x1 + (x2 - x1) * u0, y1 + (y2 - y1) * u0, x1 + (x2 - x1) * u1, y1 + (y2 - y1) * u1))
    scene = np.asarray(pieces, F32).T.copy()
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    m = np.zeros(1, fdcm.MATCH_DTYPE)
    m["transform"] = offset_pose(truth, a, 0.03, -1.5, 1.3)
    got, _ = check_fit(fm, scene, [tmpl], m, fdcm.PoseFit(iterations=20))
    e_a, e_r, _ = pose_errors(got[0]["transform"], truth, a)
    assert e_a < 0.01 and e_r < 1e-4
    # parallel lines started parallel: the fit moves the pose across them only
    th = 0.4
    u, n = np.array([math.cos(th), math.sin(th)]), np.array([-math.sin(th), math.cos(th)])
    par = np.array([[0, 0, 80, 0], [0, 15, 80, 15], [0, 40, 80, 40]], F32).T.copy()
    pa = fdcm.get_template_anchors([par])[0]
    truth = pose(th, 180.0, 170.0)
    scene, fm = instance_map(par, truth)
    start = offset_pose(truth, pa, 0.0, *(1.5 * n + 3.0 * u))
    m["transform"] = start
    got, _ = check_fit(fm, scene, [par], m, fdcm.PoseFit())
    _, _, off = pose_errors(got[0]["transform"], truth, pa)
    _, _, off0 = pose_errors(start, truth, pa)
    assert abs(float(off @ n)) < 0.01 and abs(float((off - off0) @ u)) < 1e-4   # (float32 output: 1.5e-5 px at x ~ 200)


# ---- edge cases ------------------------------------------------------------------------------------------------------
def test_edge_cases():
    tmpls, scene = synthetic(n_tmpl=4, seed=540)
    tmpls = tmpls + [np.zeros((4, 0), F32)]
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    tset = fdcm.TemplateSet(tmpls)
    fit = fdcm.PoseFit()
    assert fdcm.fit_matches(fm, tset, np.zeros(0, fdcm.MATCH_DTYPE)).shape == (0,)
    base = fdcm.search_topk(fm, tset, None, S, O, None, k=2)
    recs = np.zeros(4, fdcm.MATCH_DTYPE)
    recs[:2] = base
    recs[2] = (4, 1.0, np.array([1, 0, 50, 0, 1, 50], F32))                     # empty template
    recs[3] = base[0]
    recs[3]["transform"][1] = np.nan                                            # NaN transform
    got, st = check_fit(fm, scene, tmpls, recs, fit)
    assert got[2:]["transform"].tobytes() == recs[2:]["transform"].tobytes() and np.isnan(got[2:]["score"]).all()
    assert st[2:]["n_samples"].tolist() == [0, 0] and np.isnan(st[2:]["rms"]).all()
    # at the map border: an update that would leave the map is rejected, the pose before it kept
    W = fm.width
    t = int(base[0]["tmpl_idx"])
    T = np.asarray(base[0]["transform"], F32).copy()
    R = rotated(T[None], tmpls[t])[0]
    T[2] = F32(W - 1) - fm.get_scene_translation()[0] - F32(max(R[:, 0].max(), R[:, 2].max())) - F32(0.25)   # 0.25 px from the edge
    edge = np.zeros(1, fdcm.MATCH_DTYPE)
    edge[0] = (t, 0.0, T)
    g, _ = check_fit(fm, scene, tmpls, edge, fit)
    assert valid_poses(g["transform"], tmpls[t], fm.get_scene_translation(), fm.width, fm.height).all()
    # an empty map: every input comes back with score NaN
    empty = fdcm.build_cuda_featuremap(np.zeros((4, 0), F32), fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    g, st = fdcm.fit_matches(empty, tset, recs, fit, return_stats=True)
    assert g["transform"].tobytes() == recs["transform"].tobytes() and np.isnan(g["score"]).all() and (st["iterations"] == 0).all()
    # out-of-range template indices
    with pytest.raises(IndexError):
        fdcm.fit_matches(fm, tset, recs, fit, tmpl_idx_base=len(tmpls))   # every index below the base
    bad = recs.copy()
    bad["tmpl_idx"][0] = 5
    with pytest.raises(IndexError):
        fdcm.fit_matches(fm, tset, bad, fit)
    with pytest.raises(fdcm.FdcmError, match="max_distance"):
        fdcm.fit_matches(fm, tset, recs, fdcm.PoseFit(max_distance=17.0))
    # two identical calls are byte-identical
    m = fit_candidates(fm, tmpls[:4], scene, 20)
    a1, s1 = fdcm.fit_matches(fm, tset, m, fit, P, return_stats=True)
    a2, s2 = fdcm.fit_matches(fm, tset, m, fit, P, return_stats=True)
    assert a1.tobytes() == a2.tobytes() and s1.tobytes() == s2.tobytes()


def test_composed_searches_equal_fit_matches():
    tmpls, scene = synthetic(n_tmpl=12, seed=550)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    tset = fdcm.TemplateSet(tmpls)
    fit = fdcm.PoseFit(iterations=5)
    sel, ref, ver = fdcm.DistinctMatches(max_per_template=1), fdcm.PoseRefinement(levels=1), fdcm.EdgeCoverage(2, 1, 0.3)
    for kw in (dict(), dict(select=sel), dict(select=sel, refine=ref), dict(select=sel, refine=ref, verify=ver)):
        plain = fdcm.search_topk(fm, tset, scene, S, O, P, k=8, **kw)
        assert len(plain) > 0
        got = fdcm.search_topk(fm, tmpls, scene, S, O, P, k=8, fit=fit, **kw)
        assert got.tobytes() == fdcm.fit_matches(fm, tset, plain, fit, P).tobytes()
        dense = fdcm.DenseSearch(rotations=8, stride=6, cell=4)
        plain = fdcm.search_dense(fm, tset, dense, P, k=6, **kw)
        got = fdcm.search_dense(fm, tmpls, dense, P, k=6, fit=fit, **kw)
        assert got.tobytes() == fdcm.fit_matches(fm, tset, plain, fit, P).tobytes()


# ---- the cached scene-line grid --------------------------------------------------------------------------------------
def test_grid_follows_rebuilds():
    tmpls, scene = synthetic(n_tmpl=6, seed=560)
    _, scene2 = synthetic(n_tmpl=6, seed=561)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    fit = fdcm.PoseFit()
    m = fit_candidates(fm, tmpls, scene, 12)
    first, _ = check_fit(fm, scene, tmpls, m, fit)
    fm.rebuild(scene2)
    second, _ = check_fit(fm, scene2, tmpls, m, fit)
    assert first.tobytes() != second.tobytes()
    fm.rebuild(scene)
    assert fdcm.fit_matches(fm, tmpls, m, fit).tobytes() == first.tobytes()


def test_async_rebuild_then_stream_switch():
    import torch
    tmpls, scene = synthetic(n_tmpl=6, seed=570)
    _, scene2 = synthetic(n_tmpl=6, seed=571)
    fm = fdcm.build_cuda_featuremap(scene2, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    ref = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    fit = fdcm.PoseFit()
    m = fit_candidates(ref, tmpls, scene, 12)
    want = fdcm.fit_matches(ref, tmpls, m, fit)
    fdcm.fit_matches(fm, tmpls, m, fit)   # a cached grid of the old scene
    fm.rebuild(scene, wait=False)
    side = torch.cuda.Stream()
    fdcm.set_stream(0, side.cuda_stream)
    try:
        got = fdcm.fit_matches(fm, tmpls, m, fit)
    finally:
        fdcm.set_stream(0, None)
    assert got.tobytes() == want.tobytes()


def test_two_threads_with_different_max_distance_on_one_map():
    tmpls, scene = synthetic(n_tmpl=6, seed=580)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    tset = fdcm.TemplateSet(tmpls)
    m = fit_candidates(fm, tmpls, scene, 12)
    fits = [fdcm.PoseFit(max_distance=1.5), fdcm.PoseFit(max_distance=8.0)]
    want = [model(fm, scene, tmpls, m, f)[0] for f in fits]
    errors = []

    def run(i):
        try:
            for _ in range(5):
                if fdcm.fit_matches(fm, tset, m, fits[i]).tobytes() != want[i].tobytes():
                    errors.append(i)
        except Exception as e:   # noqa: BLE001 (reported below)
            errors.append(repr(e))

    th = [threading.Thread(target=run, args=(i,)) for i in (0, 1)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errors


def _broadcast_rank(rank, uid, scene, other, tmpls, m, out):
    from openfdcm_b200 import distributed as fd
    comm = fd.Communicator(uid, rank, 2, rank)
    fm = fdcm.build_cuda_featuremap(other if rank else scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5, device=rank))
    fdcm.fit_matches(fm, fdcm.TemplateSet(tmpls, device=rank), m)   # rank 1: a grid of its own old scene
    comm.rebuild_broadcast(fm, scene, root=0)
    out[rank] = fdcm.fit_matches(fm, fdcm.TemplateSet(tmpls, device=rank), m).tobytes()


def test_broadcast_map_on_a_non_root_rank():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two devices")
    from openfdcm_b200 import distributed as fd
    tmpls, scene = synthetic(n_tmpl=6, seed=590)
    _, other = synthetic(n_tmpl=6, seed=591)
    ref = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    m = fit_candidates(ref, tmpls, scene, 12)
    want = model(ref, scene, tmpls, m, fdcm.PoseFit())[0]
    uid = fd.Communicator.unique_id()
    out = {}
    th = [threading.Thread(target=_broadcast_rank, args=(r, uid, scene, other, tmpls, m, out)) for r in (0, 1)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert out.get(0) == want.tobytes() and out.get(1) == want.tobytes()


# ---- pybind, profile names -------------------------------------------------------------------------------------------
def test_pybind_and_profile_names():
    from openfdcm_b200 import _openfdcm_cuda as pyfdcm
    tmpls, scene = synthetic(n_tmpl=6, seed=600)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    pfm = pyfdcm.build_cuda_featuremap(scene, pyfdcm.Dt3CudaParameters(30, 5.0, 1.5))
    m = fdcm.search_topk(fm, tmpls, scene, S, O, P, k=6)
    got = pyfdcm.search_topk(pfm, tmpls, scene, pyfdcm.DefaultSearch(4, 4), pyfdcm.BatchOptimize(10), pyfdcm.ExponentialPenalty(1.5), 6)
    pf = pyfdcm.PoseFit(iterations=4, max_distance=2.5)
    assert "PoseFit" in repr(pf)
    fitted = pyfdcm.fit_matches(pfm, tmpls, got, pf, pyfdcm.ExponentialPenalty(1.5))
    want = fdcm.fit_matches(fm, tmpls, m, fdcm.PoseFit(iterations=4, max_distance=2.5), P)
    assert [g.tmpl_idx for g in fitted] == want["tmpl_idx"].tolist()
    assert np.array_equal(np.array([g.score for g in fitted], F32), want["score"])
    fdcm.profile(True, reset=True)
    try:
        n0 = fdcm.kernel_launch_count()
        fdcm.fit_matches(fm, tmpls, m, fdcm.PoseFit(max_distance=4.0))   # a new distance: the grid is built again
        n1 = fdcm.kernel_launch_count()
        fdcm.fit_matches(fm, tmpls, m, fdcm.PoseFit(max_distance=4.0))   # cached: no second grid
        n2 = fdcm.kernel_launch_count()
        rep = fdcm.profile_report()
    finally:
        fdcm.profile(False, reset=True)
    # a profile entry counts scopes: one grid build (count + fill kernels) and two evaluations
    assert rep["fit_grid"]["launches"] == 1 and rep["fit_eval"]["launches"] == 2
    assert n1 - n0 == 3 and n2 - n1 == 1
    assert _lib.FIT_STATS_DTYPE.itemsize == 16
