"""Pose refinement on the device (refine_matches, search_topk(refine=...)): byte for byte against the numpy model of
tests/models/refine.py, whose pose scores come from the device evaluate (itself bit-exact with the oracle) or, in one
case, from the oracle directly.

No test asserts that refinement brings planted instances closer to their known poses: it does not.  The evaluate<Dt3Cpu>
score is not lowest at the true pose at sub-pixel and 0.01 rad scales, so the walk moves even a noise-free instance started
at its exact pose away from it; scripts/bench_refine.py measures the errors instead."""
import ctypes as C
import itertools
import math

import numpy as np
import pytest

import openfdcm_b200 as fdcm
from openfdcm_b200 import _lib
from oracle import fdcm_oracle as orc
from tests.helpers import device_scores, load_object, refine_reference, synthetic
from tests.models.refine import refine_model, rotated
from tests.util import F32, synth_scene, synth_templates

pytestmark = pytest.mark.gpu
PEN = fdcm.ExponentialPenalty(1.5)
OPT = fdcm.BatchOptimize(10)
STEPS = ((0.01, 1.0), (0.04, 0.5))


def settings():
    for levels, n_r, n_t, (rs, ts) in itertools.product((1, 3), (0, 2, 4), (0, 1, 4, 15), STEPS):
        yield fdcm.PoseRefinement(levels, n_r, rs, n_t, ts)


def centre_scores(fm, tmpls, matches):
    """evaluate of the rotation-only template at (c2, c5) of every match."""
    work = [(tmpls[int(m["tmpl_idx"])], np.asarray(m["transform"], F32).reshape(1, 6)) for m in matches]
    return device_scores(fm)(work) if work else np.zeros(0, F32)


def check_settings(fm, tset, tmpls, anchors, base, what, cases=None):
    lengths = tset.lengths()
    centre = centre_scores(fm, tmpls, base)
    for r in cases or settings():
        want = refine_reference(fm, tmpls, anchors, base, r)
        got = fdcm.refine_matches(fm, tset, base, r)
        assert got.tobytes() == want.tobytes(), f"{what} {r}: got {got} want {want}"
        gotp = fdcm.refine_matches(fm, tset, base, r, penalty=PEN)
        assert gotp.tobytes() == fdcm.penalize(PEN, want, lengths).tobytes(), f"{what} {r} penalised"
        # the centre is a candidate: refinement never scores worse than the match it starts from
        ok = ~np.isnan(centre)
        assert (got["score"][ok] <= centre[ok]).all(), f"{what} {r}"


def test_synthetic_bit_exact_and_invariants():
    tmpls, scene = synthetic()
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    tset, anchors = fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls)
    base = fdcm.search_topk(fm, tset, None, fdcm.DefaultSearch(4, 4), OPT, PEN, k=4)
    assert len(base) == 4
    check_settings(fm, tset, tmpls, anchors, base, "synthetic")
    # levels 1 without steps: the input transform, scored as evaluate of the rotated template at (c2, c5)
    got = fdcm.refine_matches(fm, tset, base, fdcm.PoseRefinement(1, 0, 0.01, 0, 1.0))
    assert got["transform"].tobytes() == base["transform"].tobytes()
    assert got["score"].tobytes() == centre_scores(fm, tmpls, base).tobytes()


@pytest.mark.parametrize("obj", ["obj_01", "obj_02", "obj_03", "obj_04"])
def test_real_assets_bit_exact(obj):
    tmpls, scenes = load_object(obj)
    tset, anchors = fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls)
    s = fdcm.DefaultSearch(4, 10)
    for i in (0, 1):
        fm = fdcm.build_cuda_featuremap(scenes[i], fdcm.Dt3CudaParameters(30, 5.0, 1.0))
        base = fdcm.search_topk(fm, tset, None, s, OPT, PEN, k=2, select=fdcm.DistinctMatches(max_per_template=1))
        check_settings(fm, tset, tmpls, anchors, base, f"{obj} scene {i}")


def test_oracle_closure():
    tmpls, scene = synthetic(n_tmpl=6, n_lines=12, seed=40, n_scene=80)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    om = orc.Dt3Cpu(scene, 30, 5.0, 1.5)
    tset, anchors = fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls)
    base = fdcm.search_topk(fm, tset, None, fdcm.DefaultSearch(4, 4), OPT, None, k=3)

    def oracle_scores(work):
        out = []
        for tmpl, poses in work:
            for P, R in zip(poses, rotated(poses, tmpl)):
                out.append(om.evaluate(np.ascontiguousarray(R.T), P[[2, 5]].reshape(1, 2))[0])
        return np.array(out, F32)

    for r in (fdcm.PoseRefinement(2, 1, 0.02, 1, 1.0), fdcm.PoseRefinement(1, 0, 0.0, 2, 0.5)):
        want = refine_model(base, tmpls, anchors, r, om.shift, om.W, om.H, oracle_scores)
        assert fdcm.refine_matches(fm, tset, base, r).tobytes() == want.tobytes()


def test_fused_equals_standalone():
    tmpls, scene = synthetic(seed=7)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    tset = fdcm.TemplateSet(tmpls)
    s = fdcm.DefaultSearch(4, 4)
    plain10 = fdcm.search_topk(fm, tset, None, s, OPT, PEN, k=10)
    for r in (fdcm.PoseRefinement(), fdcm.PoseRefinement(2, 1, 0.03, 15, 0.25)):
        for sel in (None, fdcm.DistinctMatches(max_per_template=1)):
            for k in (1, 10, len(tmpls)):
                base = fdcm.search_topk(fm, tset, None, s, OPT, PEN, k=k, select=sel)
                fused = fdcm.search_topk(fm, tset, None, s, OPT, PEN, k=k, select=sel, refine=r)
                assert fused.tobytes() == fdcm.refine_matches(fm, tset, base, r, penalty=PEN).tobytes(), f"{r} {sel} k={k}"
    # a search without refinement after refined ones is unchanged
    assert fdcm.search_topk(fm, tset, None, s, OPT, PEN, k=10).tobytes() == plain10.tobytes()


def test_edge_cases():
    tmpls, scene = synthetic(n_tmpl=5, seed=90)
    empty = np.zeros((4, 0), F32)
    tmpls = tmpls + [empty]
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    tset, anchors = fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls)
    r = fdcm.PoseRefinement(2, 2, 0.02, 4, 1.0)
    assert fdcm.refine_matches(fm, tset, np.zeros(0, fdcm.MATCH_DTYPE), r).shape == (0,)
    base = fdcm.search_topk(fm, tset, None, fdcm.DefaultSearch(4, 4), OPT, None, k=3)
    recs = np.zeros(5, fdcm.MATCH_DTYPE)
    recs[:3] = base
    # an empty template: every pose scores 0, the centre is kept
    recs[3] = (5, 0.0, np.array([0.6, -0.8, 300.0, 0.8, 0.6, 200.0], F32).reshape(6))
    # a match at the border of the map: part of the grid lies outside
    W = fm.width
    T = np.asarray(base[0]["transform"], F32).reshape(6).copy()
    R = rotated(T[None], tmpls[int(base[0]["tmpl_idx"])])[0]
    T[2] = F32(W - 1) - fm.get_scene_translation()[0] - F32(max(R[:, 0].max(), R[:, 2].max())) - F32(1.5)
    recs[4] = (base[0]["tmpl_idx"], 0.0, T.reshape(6))
    got = fdcm.refine_matches(fm, tset, recs, r)
    assert got.tobytes() == refine_reference(fm, tmpls, anchors, recs, r).tobytes()
    assert got[3]["score"] == 0.0 and got[3]["transform"].tobytes() == recs[3]["transform"].tobytes()
    # a NaN transform: no valid pose, score NaN, transform unchanged
    bad = recs[:1].copy()
    bad["transform"].reshape(-1)[1] = np.nan
    g = fdcm.refine_matches(fm, tset, bad, r)
    assert math.isnan(g[0]["score"]) and g["transform"].tobytes() == bad["transform"].tobytes()
    # tmpl_idx_base, and indices outside the set
    shifted = recs.copy()
    shifted["tmpl_idx"] += 100
    g = fdcm.refine_matches(fm, tset, shifted, r, tmpl_idx_base=100)
    assert g["tmpl_idx"].tolist() == shifted["tmpl_idx"].tolist()
    assert g["score"].tobytes() == got["score"].tobytes() and g["transform"].tobytes() == got["transform"].tobytes()
    with pytest.raises(IndexError):
        fdcm.refine_matches(fm, tset, shifted, r)
    with pytest.raises(IndexError):
        fdcm.refine_matches(fm, tset, recs, r, tmpl_idx_base=len(tmpls))


def test_template_longer_than_3418_lines():
    rng = np.random.default_rng(5)
    n = 4000
    c = rng.uniform(-60, 60, (2, n))
    ang = rng.uniform(0, math.pi, n)
    d = np.stack([np.cos(ang), np.sin(ang)]) * 3.0
    big = np.ascontiguousarray(np.concatenate([c - d, c + d]), F32)
    tmpls = [big, synth_templates(1, 20, 640, seed=6)[0]]
    scene = synth_scene(640, 480, 150, seed=7)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    tset, anchors = fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls)
    recs = np.zeros(2, fdcm.MATCH_DTYPE)
    for q in range(2):
        recs[q] = (q, 0.0, np.array([math.cos(0.3), -math.sin(0.3), 320.0, math.sin(0.3), math.cos(0.3), 240.0], F32))
    for r in (fdcm.PoseRefinement(2, 1, 0.02, 2, 1.0), fdcm.PoseRefinement(1, 0, 0.0, 1, 1.0)):
        assert fdcm.refine_matches(fm, tset, recs, r).tobytes() == refine_reference(fm, tmpls, anchors, recs, r).tobytes()
    base = fdcm.search_topk(fm, tset, None, fdcm.DefaultSearch(2, 4), OPT, PEN, k=2)
    r = fdcm.PoseRefinement(1, 1, 0.02, 1, 1.0)
    assert fdcm.search_topk(fm, tset, None, fdcm.DefaultSearch(2, 4), OPT, PEN, k=2, refine=r).tobytes() == \
        fdcm.refine_matches(fm, tset, base, r, penalty=PEN).tobytes()


def test_template_at_the_search_limit():
    """The longest template the search accepts (16 L + round_up(L, 16) bytes of opt-in shared memory) refines; one line
    more is rejected like the search rejects it."""
    import torch
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    L = optin // 17
    while 16 * (L + 1) + ((L + 1 + 15) & ~15) <= optin:
        L += 1
    while 16 * L + ((L + 15) & ~15) > optin:
        L -= 1
    rng = np.random.default_rng(8)
    c = rng.uniform(-50, 50, (2, L + 1))
    ang = rng.uniform(0, math.pi, L + 1)
    d = np.stack([np.cos(ang), np.sin(ang)]) * 2.0
    lines = np.ascontiguousarray(np.concatenate([c - d, c + d]), F32)
    scene = synth_scene(640, 480, 150, seed=9)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    tmpls = [np.ascontiguousarray(lines[:, :L])]
    tset, anchors = fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls)
    recs = np.zeros(1, fdcm.MATCH_DTYPE)
    recs[0] = (0, 0.0, np.array([math.cos(0.2), -math.sin(0.2), 320.0, math.sin(0.2), math.cos(0.2), 240.0], F32))
    r = fdcm.PoseRefinement(1, 1, 0.02, 1, 1.0)
    assert fdcm.refine_matches(fm, tset, recs, r).tobytes() == refine_reference(fm, tmpls, anchors, recs, r).tobytes()
    base = fdcm.search_topk(fm, tset, None, fdcm.DefaultSearch(1, 2), OPT, PEN, k=1)
    assert fdcm.search_topk(fm, tset, None, fdcm.DefaultSearch(1, 2), OPT, PEN, k=1, refine=r).tobytes() == \
        fdcm.refine_matches(fm, tset, base, r, penalty=PEN).tobytes()
    with pytest.raises(fdcm.FdcmError) as e:
        fdcm.refine_matches(fm, [lines], recs, r)
    assert e.value.status == _lib.FDCM_ERR_INVALID


BAD = [dict(levels=0), dict(rot_steps=-1), dict(rot_steps=16), dict(trans_steps=-1), dict(trans_steps=16), dict(rot_step=-0.1),
       dict(rot_step=math.nan), dict(rot_step=math.inf), dict(trans_step=-1.0), dict(trans_step=math.inf)]


def test_invalid_parameters():
    tmpls, scene = synthetic(n_tmpl=4, seed=11)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    tset = fdcm.TemplateSet(tmpls)
    s = fdcm.DefaultSearch(4, 4)
    base = fdcm.search_topk(fm, tset, None, s, OPT, PEN, k=2)
    for bad in BAD:
        r = fdcm.PoseRefinement(**bad)
        for call in (lambda: fdcm.refine_matches(fm, tset, base, r), lambda: fdcm.search_topk(fm, tset, None, s, OPT, PEN, k=2, refine=r)):
            with pytest.raises(fdcm.FdcmError) as e:
                call()
            assert e.value.status == _lib.FDCM_ERR_INVALID, bad
    out = np.zeros(2, fdcm.MATCH_DTYPE)
    assert _lib.lib().fdcm_refine_matches(fm._h, tset._h, 0, 0, 0.0, None, _lib.ptr(base), 2, _lib.ptr(out)) == _lib.FDCM_ERR_INVALID
    n = C.c_int64(0)
    p = _lib.SearchParams(4, 4, 10, 0, 0.0, 2, 0, 0, 0.0, 0.0, 0.0, 0.0)
    assert _lib.lib().fdcm_search_refine(fm._h, tset._h, None, _lib.FDCM_SCENE_RESIDENT, C.byref(p), None, None, _lib.ptr(out), 2,
                                         C.byref(n)) == _lib.FDCM_ERR_INVALID
    p.top_k = 0
    assert _lib.lib().fdcm_search_refine(fm._h, tset._h, None, _lib.FDCM_SCENE_RESIDENT, C.byref(p), None,
                                         C.byref(fdcm.PoseRefinement()._params()), _lib.ptr(out), 2, C.byref(n)) == _lib.FDCM_ERR_INVALID
    # a template longer than the search accepts
    longest = np.ascontiguousarray(np.tile(np.array([[0.0], [0.0], [5.0], [1.0]], F32), (1, 14000)))
    with pytest.raises(fdcm.FdcmError) as e:
        fdcm.refine_matches(fm, [longest], np.zeros(1, fdcm.MATCH_DTYPE), fdcm.PoseRefinement())
    assert e.value.status == _lib.FDCM_ERR_INVALID


def test_pybind_and_profile_names():
    from openfdcm_b200 import _openfdcm_cuda as pyfdcm
    tmpls, scene = synthetic(n_tmpl=12, seed=500)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    pfm = pyfdcm.build_cuda_featuremap(scene, pyfdcm.Dt3CudaParameters(30, 5.0, 1.5))
    r = fdcm.PoseRefinement(2, 2, 0.02, 3, 1.0)
    pr = pyfdcm.PoseRefinement(levels=2, rot_steps=2, rot_step=0.02, trans_steps=3, trans_step=1.0)
    for sel, psel in ((None, None), (fdcm.DistinctMatches(max_per_template=1), pyfdcm.DistinctMatches(max_per_template=1))):
        want = fdcm.search_topk(fm, tmpls, scene, fdcm.DefaultSearch(4, 4), OPT, PEN, k=10, select=sel, refine=r)
        got = pyfdcm.search_topk(pfm, tmpls, scene, pyfdcm.DefaultSearch(4, 4), pyfdcm.BatchOptimize(10), pyfdcm.ExponentialPenalty(1.5), 10,
                                 select=psel, refine=pr)
        assert [m.tmpl_idx for m in got] == want["tmpl_idx"].tolist()
        assert [m.score for m in got] == want["score"].tolist()
        assert np.array([m.transform for m in got], F32).tobytes() == want["transform"].tobytes()
    base = fdcm.search_topk(fm, tmpls, scene, fdcm.DefaultSearch(4, 4), OPT, PEN, k=5)
    want = fdcm.refine_matches(fm, tmpls, base, r, penalty=PEN)
    pm = [pyfdcm.Match(int(m["tmpl_idx"]), float(m["score"]), m["transform"].reshape(2, 3)) for m in base]
    got = pyfdcm.refine_matches(pfm, tmpls, pm, pr, penalty=pyfdcm.ExponentialPenalty(1.5))
    assert [m.score for m in got] == want["score"].tolist()
    assert np.array([m.transform for m in got], F32).tobytes() == want["transform"].tobytes()
    with pytest.raises(IndexError):
        pyfdcm.refine_matches(pfm, tmpls, [pyfdcm.Match(len(tmpls), 0.0, np.eye(2, 3))], pr)
    fdcm.profile(True, reset=True)
    fdcm.search_topk(fm, tmpls, scene, fdcm.DefaultSearch(4, 4), OPT, PEN, k=10, refine=r)
    rep = fdcm.profile_report()
    fdcm.profile(False)
    assert {"refine_init", "refine_eval", "refine_advance"} <= set(rep)
