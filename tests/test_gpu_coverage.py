"""Match verification on the device (fdcm_match_coverage, search_topk / search_dense with verify=): byte-equal to the numpy
model of tests/models/coverage.py, which reads the map's own edge masks (Dt3Cuda.mask)."""
import ctypes as C
import threading

import numpy as np
import pytest

import openfdcm_b200 as fdcm
from openfdcm_b200 import _lib
from tests.helpers import load_object, masks, synthetic
from tests.models.coverage import Dilated, coverage_model, filter_model
from tests.models.dense import output_model
from tests.util import F32, synth_scene, synth_templates

pytestmark = pytest.mark.gpu

S, O, P = fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), fdcm.ExponentialPenalty(1.5)


def model(fm, tmpls, matches, cov, tmpl_idx_base=0):
    return coverage_model(Dilated(masks(fm), cov.radius, cov.bin_tolerance), fm.get_scene_translation(), tmpls, matches, tmpl_idx_base)


def candidates(fm, tmpls, scene, n=300, seed=0):
    """Search matches (valid poses), the same matches moved by up to 3 px and 0.05 rad, and poses off the map."""
    rec = fdcm.search_all(fm, tmpls, scene, S, O, P)
    rng = np.random.default_rng(seed)
    rec = rec[rng.choice(len(rec), min(n, len(rec)), replace=False)] if len(rec) else rec
    moved = rec.copy()
    a = rng.uniform(-0.05, 0.05, len(rec)).astype(F32)
    c, s = np.cos(a).astype(F32), np.sin(a).astype(F32)
    T = moved["transform"].copy()
    moved["transform"][:, 0] = c * T[:, 0] - s * T[:, 3]
    moved["transform"][:, 1] = c * T[:, 1] - s * T[:, 4]
    moved["transform"][:, 3] = s * T[:, 0] + c * T[:, 3]
    moved["transform"][:, 4] = s * T[:, 1] + c * T[:, 4]
    moved["transform"][:, 2] += rng.uniform(-3, 3, len(rec)).astype(F32)
    moved["transform"][:, 5] += rng.uniform(-3, 3, len(rec)).astype(F32)
    off = rec[: min(5, len(rec))].copy()
    off["transform"][:, 2] += F32(1e5)
    return np.concatenate([rec, moved, off])


def check_coverage(fm, tmpls, matches, cov, tmpl_idx_base=0):
    got = fdcm.match_coverage(fm, tmpls, matches, cov, tmpl_idx_base=tmpl_idx_base)
    want = model(fm, tmpls, matches, cov, tmpl_idx_base)
    assert got.dtype == np.float32 and got.shape == (len(matches),)
    assert got.tobytes() == want.tobytes(), f"{np.flatnonzero(got.view(np.uint32) != want.view(np.uint32))[:10]}"
    return got


@pytest.mark.parametrize("dist", [fdcm.distance.L2, fdcm.distance.L1])
def test_synthetic_scenes_against_the_model(dist):
    tmpls, scene = synthetic(n_tmpl=12, seed=300)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5, dist))
    m = candidates(fm, tmpls, scene, 150)
    for r in (0, 1, 2, 16):
        for tol in (0, 1, fm.depth // 2):
            got = check_coverage(fm, tmpls, m, fdcm.EdgeCoverage(r, tol))
    assert np.isnan(got[-5:]).all() and np.nanmax(got) <= 1.0 and np.nanmin(got) >= 0.0


def test_tmpl_idx_base_and_odd_depth():
    tmpls, scene = synthetic(n_tmpl=6, seed=310)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(7, 5.0, 1.5))
    m = candidates(fm, tmpls, scene, 60)
    m["tmpl_idx"] += 100
    check_coverage(fm, tmpls, m, fdcm.EdgeCoverage(2, 3), tmpl_idx_base=100)


def test_literal_path_map():
    """A map of side > 2897 (the literal distance-transform path): words past the first few thousand columns."""
    tmpls = synth_templates(4, 12, 2000, seed=320)
    scene = synth_scene(3000, 3000, 120, seed=321)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.05))
    assert fm.width > 2897
    check_coverage(fm, tmpls, candidates(fm, tmpls, scene, 60), fdcm.EdgeCoverage(3, 1))


@pytest.mark.parametrize("obj", ["obj_01", "obj_02", "obj_03", "obj_04"])
def test_real_assets(obj):
    tmpls, scenes = load_object(obj)
    fm = fdcm.build_cuda_featuremap(scenes[0], fdcm.Dt3CudaParameters(30, 5.0, 2.2))
    m = candidates(fm, tmpls, scenes[0], 80, seed=1)
    check_coverage(fm, tmpls, m, fdcm.EdgeCoverage())
    check_coverage(fm, tmpls, m, fdcm.EdgeCoverage(5, 2))


def test_empty_inputs():
    tmpls, scene = synthetic(n_tmpl=3, seed=330)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    assert fdcm.match_coverage(fm, tmpls, np.zeros(0, _lib.MATCH_DTYPE)).shape == (0,)
    m = np.zeros(2, _lib.MATCH_DTYPE)
    m["transform"] = [1, 0, 0, 0, 1, 0]
    got = fdcm.match_coverage(fm, [np.zeros((4, 0), F32), tmpls[0]], m)   # empty template
    assert np.isnan(got[0])
    empty = fdcm.build_cuda_featuremap(np.zeros((4, 0), F32), fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    assert np.isnan(fdcm.match_coverage(empty, tmpls, m)).all()


# ---- the fused filter ------------------------------------------------------------------------------------------------
def filtered(fm, tmpls, rec, cov):
    return filter_model(model(fm, tmpls, rec, cov), cov.min_coverage)


@pytest.mark.parametrize("min_cov", [0.3, 0.6, 0.9])
def test_search_topk_filter(min_cov):
    tmpls, scene = synthetic(n_tmpl=20, seed=340)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    cov = fdcm.EdgeCoverage(2, 1, min_cov)
    rec = fdcm.search_all(fm, tmpls, scene, S, O, P)
    keep = filtered(fm, tmpls, rec, cov)
    assert 0 < keep.sum() < len(rec)
    anchors = fdcm.get_template_anchors(tmpls)
    for k in (1, 10, 100):
        got = fdcm.search_topk(fm, tmpls, scene, S, O, P, k=k, verify=cov)
        assert got.tobytes() == output_model(rec, keep, k).tobytes()
    sel = fdcm.DistinctMatches(max_per_template=2, radius=10.0)
    got = fdcm.search_topk(fm, tmpls, scene, S, O, P, k=15, select=sel, verify=cov)
    want = output_model(rec, keep, 15, anchors, sel)
    assert got.tobytes() == want.tobytes()
    ref = fdcm.PoseRefinement(levels=2)
    got = fdcm.search_topk(fm, tmpls, scene, S, O, P, k=15, select=sel, refine=ref, verify=cov)
    assert got.tobytes() == fdcm.refine_matches(fm, tmpls, want, ref, P).tobytes()


def test_search_dense_filter():
    tmpls, scene = synthetic(n_tmpl=4, seed=350, w=200, h=160, n_scene=40)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.3))
    dense = fdcm.DenseSearch(rotations=6, stride=4, cell=6)
    k = 100000   # covers every record
    every = fdcm.search_dense(fm, tmpls, dense, P, k=k)
    assert 0 < len(every) < k
    for min_cov in (0.2, 0.5):
        cov = fdcm.EdgeCoverage(1, 1, min_cov)
        keep = filtered(fm, tmpls, every, cov)
        assert 0 < keep.sum() < len(every)
        got = fdcm.search_dense(fm, tmpls, dense, P, k=k, verify=cov)
        assert got.tobytes() == every[keep].tobytes()
        got = fdcm.search_dense(fm, tmpls, dense, P, k=7, verify=cov)
        assert got.tobytes() == every[keep][:7].tobytes()
    sel = fdcm.DistinctMatches(max_per_template=3, radius=8.0)
    want = output_model(every, keep, 9, fdcm.get_template_anchors(tmpls), sel)
    assert fdcm.search_dense(fm, tmpls, dense, P, k=9, select=sel, verify=cov).tobytes() == want.tobytes()
    ref = fdcm.PoseRefinement(levels=1)
    got = fdcm.search_dense(fm, tmpls, dense, P, k=9, select=sel, refine=ref, verify=cov)
    assert got.tobytes() == fdcm.refine_matches(fm, tmpls, want, ref, P).tobytes()


def test_min_coverage_zero_is_the_call_without_verify():
    tmpls, scene = synthetic(n_tmpl=10, seed=360)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    dense = fdcm.DenseSearch(rotations=8, stride=6, cell=4)
    sel, ref = fdcm.DistinctMatches(max_per_template=1), fdcm.PoseRefinement(levels=1)
    for kw in (dict(), dict(select=sel), dict(select=sel, refine=ref)):
        calls = [lambda v: fdcm.search_topk(fm, tmpls, scene, S, O, P, k=12, **kw, **v),
                 lambda v: fdcm.search_dense(fm, tmpls, dense, P, k=12, **kw, **v)]
        for call in calls:
            n0 = fdcm.kernel_launch_count()
            a = call({})
            n1 = fdcm.kernel_launch_count()
            b = call(dict(verify=fdcm.EdgeCoverage(3, 2, 0.0)))
            n2 = fdcm.kernel_launch_count()
            assert a.tobytes() == b.tobytes() and n1 - n0 == n2 - n1


def test_verify_keeps_the_last_search_state():
    tmpls, scene = synthetic(n_tmpl=8, seed=370)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    fdcm.search_topk(fm, tmpls, scene, S, O, P, k=5)
    stats, hyp = fm.last_search_stats(), fm.last_hypotheses()
    m = fdcm.search_topk(fm, tmpls, scene, S, O, P, k=5)
    fdcm.match_coverage(fm, tmpls, m)
    fdcm.search_dense(fm, tmpls, fdcm.DenseSearch(rotations=4, stride=8), P, k=5, verify=fdcm.EdgeCoverage(min_coverage=0.5))
    assert fm.last_search_stats() == stats and np.array_equal(fm.last_hypotheses(), hyp)


# ---- cache and ordering ----------------------------------------------------------------------------------------------
def test_coverage_follows_rebuilds():
    tmpls, scene = synthetic(n_tmpl=8, seed=380)
    _, scene2 = synthetic(n_tmpl=8, seed=381)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    cov = fdcm.EdgeCoverage(2, 1)
    m = candidates(fm, tmpls, scene, 60)
    first = check_coverage(fm, tmpls, m, cov)
    fm.rebuild(scene2)
    second = check_coverage(fm, tmpls, m, cov)
    assert first.tobytes() != second.tobytes()
    fm.rebuild(scene)
    assert check_coverage(fm, tmpls, m, cov).tobytes() == first.tobytes()
    fm.rerun()
    assert fdcm.match_coverage(fm, tmpls, m, cov).tobytes() == first.tobytes()


def test_async_rebuild_then_stream_switch():
    import torch
    tmpls, scene = synthetic(n_tmpl=8, seed=390)
    _, scene2 = synthetic(n_tmpl=8, seed=391)
    fm = fdcm.build_cuda_featuremap(scene2, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    ref = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    cov = fdcm.EdgeCoverage(2, 1)
    m = candidates(ref, tmpls, scene, 60)
    want = fdcm.match_coverage(ref, tmpls, m, cov)
    fdcm.match_coverage(fm, tmpls, m, cov)   # a cached dilation of the old scene
    fm.rebuild(scene, wait=False)
    side = torch.cuda.Stream()
    fdcm.set_stream(0, side.cuda_stream)
    try:
        got = fdcm.match_coverage(fm, tmpls, m, cov)
    finally:
        fdcm.set_stream(0, None)
    assert got.tobytes() == want.tobytes()


def test_two_threads_with_different_parameters_on_one_map():
    tmpls, scene = synthetic(n_tmpl=8, seed=400)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    tset = fdcm.TemplateSet(tmpls)
    m = candidates(fm, tmpls, scene, 60)
    covs = [fdcm.EdgeCoverage(1, 0), fdcm.EdgeCoverage(4, 2)]
    want = [model(fm, tmpls, m, c) for c in covs]
    errors = []

    def run(i):
        try:
            for _ in range(6):
                if fdcm.match_coverage(fm, tset, m, covs[i]).tobytes() != want[i].tobytes():
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
    fdcm.match_coverage(fm, fdcm.TemplateSet(tmpls, device=rank), m)   # rank 1: a dilation of its own old scene
    comm.rebuild_broadcast(fm, scene, root=0)
    out[rank] = fdcm.match_coverage(fm, fdcm.TemplateSet(tmpls, device=rank), m).tobytes()


def test_broadcast_map_on_a_non_root_rank():
    """A non-root rank receives the planes of the broadcast but not the edge mask: coverage rasterises it first."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two devices")
    from openfdcm_b200 import distributed as fd
    tmpls, scene = synthetic(n_tmpl=6, seed=410)
    _, other = synthetic(n_tmpl=6, seed=411)
    ref = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    m = candidates(ref, tmpls, scene, 40)
    want = model(ref, tmpls, m, fdcm.EdgeCoverage())
    uid = fd.Communicator.unique_id()
    out = {}
    th = [threading.Thread(target=_broadcast_rank, args=(r, uid, scene, other, tmpls, m, out)) for r in (0, 1)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert out.get(0) == want.tobytes() and out.get(1) == want.tobytes()


# ---- validation, pybind, profile names -------------------------------------------------------------------------------
def test_validation_through_ctypes():
    tmpls, scene = synthetic(n_tmpl=3, seed=420)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    m = fdcm.search_topk(fm, tmpls, scene, S, O, P, k=3)
    for bad, msg in ((dict(radius=17), "0..16"), (dict(bin_tolerance=33), "0..32"), (dict(min_coverage=1.5), "[0, 1]")):
        with pytest.raises(fdcm.FdcmError, match=msg.replace("[", r"\[").replace("]", r"\]")):
            fdcm.match_coverage(fm, tmpls, m, fdcm.EdgeCoverage(**bad))
        with pytest.raises(fdcm.FdcmError):
            fdcm.search_topk(fm, tmpls, scene, S, O, P, k=3, verify=fdcm.EdgeCoverage(**bad))
        with pytest.raises(fdcm.FdcmError):
            fdcm.search_dense(fm, tmpls, fdcm.DenseSearch(rotations=2, stride=9), P, k=3, verify=fdcm.EdgeCoverage(**bad))
    bad = m.copy()
    bad["tmpl_idx"][0] = 3
    with pytest.raises(IndexError):
        fdcm.match_coverage(fm, tmpls, bad)
    with pytest.raises(IndexError):
        fdcm.match_coverage(fm, tmpls, m, tmpl_idx_base=100)
    with pytest.raises(fdcm.FdcmError, match="top_k"):
        fdcm.search_topk(fm, tmpls, scene, S, O, P, k=0, verify=fdcm.EdgeCoverage(min_coverage=0.5))
    p, n = _lib.CoverageParams(2, 1, 0.5), C.c_int64(0)
    st = _lib.lib().fdcm_search_verify(fm._h, fdcm.TemplateSet(tmpls)._h, None, _lib.FDCM_SCENE_RESIDENT, None, None, None, C.byref(p),
                                       None, 0, C.byref(n))
    assert st == _lib.FDCM_ERR_INVALID


def test_pybind():
    from openfdcm_b200 import _openfdcm_cuda as pyfdcm
    tmpls, scene = synthetic(n_tmpl=6, seed=430)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    pfm = pyfdcm.build_cuda_featuremap(scene, pyfdcm.Dt3CudaParameters(30, 5.0, 1.5))
    cov = fdcm.EdgeCoverage(2, 1, 0.4)
    pcov = pyfdcm.EdgeCoverage(radius=2, bin_tolerance=1, min_coverage=0.4)
    want = fdcm.search_topk(fm, tmpls, scene, S, O, P, k=8, verify=cov)
    got = pyfdcm.search_topk(pfm, tmpls, scene, pyfdcm.DefaultSearch(4, 4), pyfdcm.BatchOptimize(10), pyfdcm.ExponentialPenalty(1.5),
                             8, verify=pcov)
    assert [g.tmpl_idx for g in got] == want["tmpl_idx"].tolist()
    assert np.array_equal(np.array([g.score for g in got], F32), want["score"])
    c = pyfdcm.match_coverage(pfm, tmpls, got, pcov)
    assert np.array_equal(np.asarray(c, F32), fdcm.match_coverage(fm, tmpls, want, cov))
    dense = fdcm.DenseSearch(rotations=4, stride=8)
    want = fdcm.search_dense(fm, tmpls, dense, P, k=5, verify=cov)
    got = pyfdcm.search_dense(pfm, tmpls, pyfdcm.DenseSearch(rotations=4, stride=8), pyfdcm.ExponentialPenalty(1.5), 5, verify=pcov)
    assert [g.tmpl_idx for g in got] == want["tmpl_idx"].tolist()
    assert "EdgeCoverage" in repr(pcov)


def test_profile_names():
    tmpls, scene = synthetic(n_tmpl=6, seed=440)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    m = fdcm.search_topk(fm, tmpls, scene, S, O, P, k=5)
    fdcm.profile(True, reset=True)
    try:
        fdcm.match_coverage(fm, tmpls, m, fdcm.EdgeCoverage(3, 1))
        fdcm.match_coverage(fm, tmpls, m, fdcm.EdgeCoverage(3, 1))   # cached: no second dilation
        fdcm.search_topk(fm, tmpls, scene, S, O, P, k=5, verify=fdcm.EdgeCoverage(3, 1, 0.5))
        rep = fdcm.profile_report()
    finally:
        fdcm.profile(False, reset=True)
    assert rep["coverage_dilate"]["launches"] == 1 and rep["coverage_eval"]["launches"] == 3
    assert "coverage_raster" not in rep
