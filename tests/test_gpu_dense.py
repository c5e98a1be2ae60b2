"""Dense pose-grid search on the device (search_dense, DenseSearch): byte for byte against the numpy model of
tests/models/dense.py, whose pose scores come from the device evaluate (itself bit-exact with the oracle) or, in one
case, from the oracle directly."""
import ctypes as C
import itertools
import math

import numpy as np
import pytest

import openfdcm_b200 as fdcm
from openfdcm_b200 import _lib
from oracle import fdcm_oracle as orc
from tests.helpers import evaluate_fn, load_object, synthetic
from tests.models.dense import dense_records, output_model, penalised, rotate_template
from tests.util import F32, synth_scene

pytestmark = pytest.mark.gpu
PEN = fdcm.ExponentialPenalty(1.5)
OPT = fdcm.BatchOptimize(10)


def model_records(fm, tmpls, anchors, d, score_fn=None, tmpl_idx_base=0):
    return dense_records(tmpls, anchors, d, fm.get_scene_translation(), fm.width, fm.height, score_fn or evaluate_fn(fm), tmpl_idx_base)


def outputs(n_valid):
    """(k, select) of every output path; k = every valid record where that is at most 1000 (the plain top-K takes O(k n))"""
    yield 1, None
    yield 10, None
    if 1 <= n_valid <= 1000:
        yield n_valid, None
    yield 10, fdcm.DistinctMatches(max_per_template=1)
    yield 10, fdcm.DistinctMatches(radius=6.0, max_angle=0.3, across_templates=True)


def check_all(fm, tset, tmpls, anchors, d, what, tmpl_idx_base=0):
    rec, valid, _ = model_records(fm, tmpls, anchors, d, tmpl_idx_base=tmpl_idx_base)
    for pen in (None, PEN):
        prec = penalised(rec, valid, fdcm.get_template_lengths(tmpls), pen)
        for k, sel in outputs(int(valid.sum())):
            got = fdcm.search_dense(fm, tset, d, pen, k, tmpl_idx_base, select=sel)
            want = output_model(prec, valid, k, anchors, sel, tmpl_idx_base)
            assert got.tobytes() == want.tobytes(), f"{what} {d} {pen} k={k} {sel}: got {got[:3]} want {want[:3]}"
    return rec, valid


def small():
    tmpls, scene = synthetic(n_tmpl=4, n_lines=8, seed=60, w=200, h=150, n_scene=60)
    return tmpls, scene, fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))


def test_synthetic_bit_exact():
    tmpls, scene, fm = small()
    tset, anchors = fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls)
    roi = (20.0, 10.5, 150.25, 120.0)
    for rot, stride, cell, region in itertools.product((1, 7, 36), (1, 3), (1, 4, 1000), (None, roi)):
        if rot == 36 and stride == 1:
            stride = 2   # (keeps the model near 10^6 poses)
        d = fdcm.DenseSearch(rot, rot_start=0.0 if rot == 1 else 0.1, stride=stride, cell=cell, roi=region)
        rec, valid = check_all(fm, tset, tmpls, anchors, d, "synthetic")
        assert valid.any()


def test_record_index_base_and_partial_penalty():
    tmpls, scene, fm = small()
    tset, anchors = fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls)
    check_all(fm, tset, tmpls, anchors, fdcm.DenseSearch(5, rot_start=-0.4, rot_step=0.2, stride=5, cell=3), "base 50", tmpl_idx_base=50)


@pytest.mark.parametrize("obj", ["obj_01", "obj_02", "obj_03", "obj_04"])
def test_real_assets_bit_exact(obj):
    tmpls, scenes = load_object(obj)
    tmpls = tmpls[:3]
    tset, anchors = fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls)
    fm = fdcm.build_cuda_featuremap(scenes[0], fdcm.Dt3CudaParameters(30, 5.0, 1.0))
    d = fdcm.DenseSearch(12, stride=8, cell=4)
    rec, valid, _ = model_records(fm, tmpls, anchors, d)
    for k, sel in ((10, None), (10, fdcm.DistinctMatches(max_per_template=1))):
        want = output_model(penalised(rec, valid, fdcm.get_template_lengths(tmpls), PEN), valid, k, anchors, sel)
        assert fdcm.search_dense(fm, tset, d, PEN, k, select=sel).tobytes() == want.tobytes(), f"{obj} {sel}"


def test_oracle_closure():
    tmpls, scene = synthetic(n_tmpl=3, n_lines=8, seed=70, w=200, h=150, n_scene=60)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    om = orc.Dt3Cpu(scene, 30, 5.0, 1.5)
    assert (om.W, om.H) == (fm.width, fm.height)
    top = fdcm.search_dense(fm, tmpls, fdcm.DenseSearch(9, rot_start=0.05, stride=3, cell=5), None, 12)
    assert len(top) == 12
    for m in top:
        T = np.asarray(m["transform"], F32).reshape(6)
        Rt = rotate_template(tmpls[int(m["tmpl_idx"])], T[0], T[3])
        want = om.evaluate(np.ascontiguousarray(Rt.T), T[[2, 5]].reshape(1, 2))[0]
        assert F32(want).tobytes() == F32(m["score"]).tobytes()


def test_theta_zero_slice_is_evaluate_of_the_template():
    tmpls, scene, fm = small()
    # a vertical line at x = -0 with a negative y (the identity rule keeps its orientation bin)
    tmpls = tmpls + [np.array([[-0.0, 5.0], [-6.0, -3.0], [-0.0, 12.0], [7.0, -3.0]], F32)]
    d = fdcm.DenseSearch(1, rot_start=0.0, stride=2, cell=3)
    # every valid record, ascending score (the selection's sort instead of the O(k n) plain top-K)
    got = fdcm.search_dense(fm, tmpls, d, None, 100000, select=fdcm.DistinctMatches(max_per_template=100000))
    assert len(got) > 100 and set(got["tmpl_idx"].tolist()) == set(range(len(tmpls)))
    for t in range(len(tmpls)):
        g = got[got["tmpl_idx"] == t]
        ev = fdcm.evaluate(fm, [tmpls[t]], [g["transform"][:, [2, 5]]])[0]
        assert ev.tobytes() == g["score"].tobytes(), t
        assert (g["transform"][:, 0] == 1).all() and (g["transform"][:, 3] == 0).all()


def test_refinement_equals_refine_matches():
    tmpls, scene, fm = small()
    tset = fdcm.TemplateSet(tmpls)
    d = fdcm.DenseSearch(12, stride=3, cell=4)
    for r in (fdcm.PoseRefinement(), fdcm.PoseRefinement(2, 1, 0.03, 3, 0.5)):
        for sel in (None, fdcm.DistinctMatches(max_per_template=1)):
            for k in (1, 10):
                base = fdcm.search_dense(fm, tset, d, PEN, k, select=sel)
                fused = fdcm.search_dense(fm, tset, d, PEN, k, select=sel, refine=r)
                assert fused.tobytes() == fdcm.refine_matches(fm, tset, base, r, penalty=PEN).tobytes(), f"{r} {sel} k={k}"


def test_edge_cases():
    tmpls, scene, fm = small()
    d = fdcm.DenseSearch(6, stride=3, cell=4)
    assert len(fdcm.search_dense(fm, [], d)) == 0
    empty_fm = fdcm.build_cuda_featuremap(np.zeros((4, 0), F32), fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    assert len(fdcm.search_dense(empty_fm, tmpls, d)) == 0
    # an empty template inside a set: no records of its own
    with_empty = tmpls[:2] + [np.zeros((4, 0), F32)] + tmpls[2:]
    check_all(fm, fdcm.TemplateSet(with_empty), with_empty, fdcm.get_template_anchors(with_empty), d, "empty template")
    # a template larger than the map: no valid pose
    huge = np.array([[0.0], [0.0], [5000.0], [0.0]], F32)
    assert len(fdcm.search_dense(fm, [huge], d, PEN, 10)) == 0
    # a region outside the map: no grid point
    assert len(fdcm.search_dense(fm, tmpls, fdcm.DenseSearch(6, roi=(1e5, 1e5, 2e5, 2e5)))) == 0
    # top_k larger than the number of valid records
    d = fdcm.DenseSearch(6, stride=3, cell=1000)
    rec, valid, _ = model_records(fm, tmpls, fdcm.get_template_anchors(tmpls), d)
    got = fdcm.search_dense(fm, tmpls, d, None, int(valid.sum()) + 1000)
    assert len(got) == int(valid.sum()) and got.tobytes() == output_model(rec, valid, len(got)).tobytes()


def long_template(n, seed, half=50.0, seg=2.0):
    rng = np.random.default_rng(seed)
    c = rng.uniform(-half, half, (2, n))
    ang = rng.uniform(0, math.pi, n)
    d = np.stack([np.cos(ang), np.sin(ang)]) * seg
    return np.ascontiguousarray(np.concatenate([c - d, c + d]), F32)


def search_limit():
    import torch
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    L = optin // 17
    while 16 * (L + 1) + ((L + 1 + 15) & ~15) <= optin:
        L += 1
    while 16 * L + ((L + 15) & ~15) > optin:
        L -= 1
    return L


def test_long_templates():
    """A template of more than 3418 lines and one at the search's line limit (16 L + round_up(L, 16) bytes of opt-in
    shared memory) run; one line more is rejected like the search rejects it."""
    L = search_limit()
    lines = long_template(L + 1, 8)
    scene = synth_scene(640, 480, 150, seed=9)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    d = fdcm.DenseSearch(2, rot_step=0.3, stride=4, cell=3, roi=(300.0, 200.0, 340.0, 240.0))
    for tmpls in ([long_template(4000, 5), long_template(30, 6)], [np.ascontiguousarray(lines[:, :L])]):
        tset, anchors = fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls)
        rec, valid, _ = model_records(fm, tmpls, anchors, d)
        assert valid.any()
        for k, sel in ((5, None), (5, fdcm.DistinctMatches(max_per_template=1))):
            assert fdcm.search_dense(fm, tset, d, PEN, k, select=sel).tobytes() == \
                output_model(penalised(rec, valid, fdcm.get_template_lengths(tmpls), PEN), valid, k, anchors, sel).tobytes()
    with pytest.raises(fdcm.FdcmError) as e:
        fdcm.search_dense(fm, [lines], d)
    assert e.value.status == _lib.FDCM_ERR_INVALID and "lines per template" in str(e.value)


def test_last_search_state_is_kept():
    tmpls, scene, fm = small()
    tset = fdcm.TemplateSet(tmpls)
    s = fdcm.DefaultSearch(4, 4)
    allm = fdcm.search_all(fm, tset, None, s, OPT, PEN)
    hyp, stats = fm.last_hypotheses(), fm.last_search_stats()
    top = fdcm.search_topk(fm, tset, None, s, OPT, PEN, k=10, select=fdcm.DistinctMatches(max_per_template=1))
    hyp2, stats2 = fm.last_hypotheses(), fm.last_search_stats()
    for sel in (None, fdcm.DistinctMatches(max_per_template=1), fdcm.DistinctMatches(radius=5, across_templates=True)):
        fdcm.search_dense(fm, tset, fdcm.DenseSearch(8, stride=2, cell=4), PEN, 10, select=sel, refine=fdcm.PoseRefinement())
        assert fm.last_hypotheses().tobytes() == hyp2.tobytes() and fm.last_search_stats() == stats2
    assert hyp.tobytes() == hyp2.tobytes() and stats == stats2
    assert fdcm.search_all(fm, tset, None, s, OPT, PEN).tobytes() == allm.tobytes()
    assert fdcm.search_topk(fm, tset, None, s, OPT, PEN, k=10, select=fdcm.DistinctMatches(max_per_template=1)).tobytes() == top.tobytes()


BAD = [dict(rotations=0), dict(rotations=4097), dict(stride=0), dict(cell=0), dict(rot_start=math.nan), dict(rot_step=math.inf),
       dict(roi=(0.0, 0.0, math.nan, 5.0)), dict(roi=(6.0, 0.0, 5.0, 5.0)), dict(roi=(0.0, 6.0, 5.0, 5.0))]


def test_invalid_parameters():
    tmpls, scene, fm = small()
    tset = fdcm.TemplateSet(tmpls)
    lib = _lib.lib()
    out, n = np.zeros(64, fdcm.MATCH_DTYPE), C.c_int64(0)

    def call(d=fdcm.DenseSearch(4), pen=0, k=10, sel=None, ref=None, dense_ptr=True):
        return lib.fdcm_search_dense(fm._h, tset._h, C.byref(d._params()) if dense_ptr else None, pen, 1.5, k, 0,
                                     None if sel is None else C.byref(sel._params()), None if ref is None else C.byref(ref._params()),
                                     _lib.ptr(out), 64, C.byref(n))

    for bad in BAD:
        assert call(fdcm.DenseSearch(**{**dict(rotations=4, rot_step=0.1), **bad})) == _lib.FDCM_ERR_INVALID, bad
        assert b"dense search" in lib.fdcm_last_error()
    assert call(dense_ptr=False) == _lib.FDCM_ERR_INVALID
    assert call(pen=3) == _lib.FDCM_ERR_INVALID
    assert call(k=0) == _lib.FDCM_ERR_INVALID and b"top_k" in lib.fdcm_last_error()
    assert call(sel=fdcm.DistinctMatches(max_per_template=-1)) == _lib.FDCM_ERR_INVALID
    assert call(k=1025, sel=fdcm.DistinctMatches(radius=5, across_templates=True)) == _lib.FDCM_ERR_INVALID
    assert call(ref=fdcm.PoseRefinement(levels=0)) == _lib.FDCM_ERR_INVALID
    assert call(ref=fdcm.PoseRefinement(rot_steps=16)) == _lib.FDCM_ERR_INVALID
    # 2^31 records or more: 8 templates x 4096 rotations x every pixel of the map in its own cell
    big = fdcm.TemplateSet(tmpls * 2)
    assert 8 * 4096 * fm.width * fm.height >= 2 ** 31
    assert lib.fdcm_search_dense(fm._h, big._h, C.byref(fdcm.DenseSearch(4096, stride=1, cell=1)._params()), 0, 0.0, 10, 0, None, None,
                                 _lib.ptr(out), 64, C.byref(n)) == _lib.FDCM_ERR_INVALID and b"2^31" in lib.fdcm_last_error()
    # the bounds themselves are accepted
    assert call(fdcm.DenseSearch(1, rot_step=0.0, stride=10**6, cell=10**6)) == _lib.FDCM_OK
    assert call(fdcm.DenseSearch(4096, stride=40, cell=1000)) == _lib.FDCM_OK
    # capacity: n_out holds the required count
    assert lib.fdcm_search_dense(fm._h, tset._h, C.byref(fdcm.DenseSearch(4)._params()), 0, 0.0, 10, 0, None, None, _lib.ptr(out), 3,
                                 C.byref(n)) == _lib.FDCM_ERR_CAPACITY and n.value == 10


def test_pybind_and_profile_names():
    from openfdcm_b200 import _openfdcm_cuda as pyfdcm
    tmpls, scene, fm = small()
    pfm = pyfdcm.build_cuda_featuremap(scene, pyfdcm.Dt3CudaParameters(30, 5.0, 1.5))
    d = fdcm.DenseSearch(12, stride=3, cell=4, roi=(10.0, 10.0, 180.0, 140.0))
    pd = pyfdcm.DenseSearch(rotations=12, stride=3, cell=4, roi=(10.0, 10.0, 180.0, 140.0))
    assert pd.rot_step == F32(d.rot_step)
    r, pr = fdcm.PoseRefinement(2, 2, 0.02, 3, 1.0), pyfdcm.PoseRefinement(levels=2, rot_steps=2, rot_step=0.02, trans_steps=3, trans_step=1.0)
    for sel, psel in ((None, None), (fdcm.DistinctMatches(max_per_template=1), pyfdcm.DistinctMatches(max_per_template=1))):
        for ref, pref in ((None, None), (r, pr)):
            want = fdcm.search_dense(fm, tmpls, d, PEN, 10, select=sel, refine=ref)
            got = pyfdcm.search_dense(pfm, tmpls, pd, pyfdcm.ExponentialPenalty(1.5), 10, select=psel, refine=pref)
            assert [m.tmpl_idx for m in got] == want["tmpl_idx"].tolist()
            assert [m.score for m in got] == want["score"].tolist()
            assert np.array([m.transform for m in got], F32).tobytes() == want["transform"].tobytes()
    fdcm.profile(True, reset=True)
    fdcm.search_dense(fm, tmpls, d, PEN, 10, select=fdcm.DistinctMatches(max_per_template=1))
    rep = fdcm.profile_report()
    fdcm.profile(False)
    assert {"dense_eval", "dense_finish", "select_sort"} <= set(rep)
