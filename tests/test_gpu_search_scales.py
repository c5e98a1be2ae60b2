"""Scale in the line-alignment search on the device (fdcm_search_scales; search_topk / search_all with scales=ScaleGrid):
the CPU oracle's search of the scaled copies, mapped by rule 4 in numpy, byte for byte (records, hypothesis list, counters),
the top-K, the distinct selection (tests/models/select.py with the records' scales), refinement, the coverage filter and
the fit against their standalone calls, byte-identity with the unscaled entry points at one scale, edge cases, the
per-map cache of the copies, two threads, and planted scaled instances.  The rules are in include/fdcm_b200.h."""
import ctypes as C
import math
import threading

import numpy as np
import pytest

import openfdcm_b200 as fdcm
from openfdcm_b200 import _lib
from oracle import fdcm_oracle as orc
from tests.helpers import DIST, house, load_object, optimizer, oracle_penalized, posed, scale_error, spose, synthetic, topk_ref
from tests.models.dense import scale_values
from tests.models.select import select_model
from tests.util import F32, synth_scene, synth_templates

pytestmark = pytest.mark.gpu
PEN = fdcm.ExponentialPenalty(1.5)
S3 = fdcm.ScaleGrid(3, 0.85, 1.0 / 0.85)            # 0.85, 1.0, 1.1765
S5 = fdcm.ScaleGrid(5, 0.8, (1.25 / 0.8) ** 0.25)    # 0.8 .. 1.25


def copies(tmpls, g):
    """Rule 2: copy v = t * S + k is template t with every coordinate multiplied by s_k (one fp32 multiply)."""
    return [(s * np.asarray(t, F32)).astype(F32) for t in tmpls for s in scale_values(g)]


def remap(rec, g, base=0):
    """Rule 4 on oracle records of the copies (tmpl_idx = v): the records of the original templates and their scales."""
    sk = scale_values(g)
    S = len(sk)
    v = rec["tmpl_idx"].astype(np.int64)
    out = rec.copy()
    out["tmpl_idx"] = (v // S + base).astype(np.int32)
    rs = sk[v % S]
    for c in (0, 1, 3, 4):
        out["transform"][:, c] = rs * rec["transform"][:, c]
    return out, rs


def oracle_list(c, tmpls, scene, g, max_t, max_s, batch, penalty=None, base=0, concentric=None):
    """The oracle's search of the copies, penalised with the copies' lengths, mapped by rule 4; the hypothesis list and
    the counters of the copy search."""
    cp = copies(tmpls, g)
    orc.stats_reset()
    raw, hyp = c.search(cp, scene, max_t, max_s, batch=batch, want_hyp=True, concentric=concentric)
    counters = orc.stats_get()
    rec, rs = remap(oracle_penalized(raw, cp, penalty), g, base)
    hyp = hyp.copy()
    hyp[:, 0] += base
    return rec, rs, hyp, counters


def searcher(max_t, max_s, concentric=None):
    return fdcm.DefaultSearch(max_t, max_s) if concentric is None else fdcm.ConcentricRangeStrategy(max_t, max_s, *concentric)


def check_list(fm, c, tset, tmpls, scene, g, max_t=4, max_s=4, batch=10, penalty=None, base=0, concentric=None):
    """search_all(scales=g) against the oracle: every record, the hypothesis list and the counters."""
    got = fdcm.search_all(fm, tset, scene, searcher(max_t, max_s, concentric), optimizer(batch), penalty, base, scales=g)
    st = fm.last_search_stats()
    conc = None if concentric is None else (concentric[0][0], concentric[0][1], concentric[1], concentric[2])
    want, rs, hyp, (evals, lookups) = oracle_list(c, tmpls, scene, g, max_t, max_s, batch, penalty, base, conc)
    assert np.array_equal(fm.last_hypotheses(), hyp), "hypothesis list"
    assert (st["n_hypotheses"], st["n_valid"]) == (len(hyp), len(want))
    assert (st["n_evaluations"], st["n_lookups"]) == (evals, lookups), "counters"
    assert got.tobytes() == want.tobytes(), f"{g} batch {batch} {penalty} base {base}"
    return want, rs


def select_ref(rec, rs, anchors, k, sel, base=0):
    pos = select_model(rec, anchors, k, sel.max_per_template, sel.radius, sel.max_angle, sel.across_templates, base, rs)
    return rec[pos]


def small(dist="L2", seed=80, n_tmpl=5, n_lines=8):
    tmpls, scene = synthetic(n_tmpl=n_tmpl, n_lines=n_lines, seed=seed, w=240, h=180, n_scene=70)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5, DIST[dist][0]))
    return tmpls, scene, fm, orc.Dt3Cpu(scene, 30, 5.0, 1.5, DIST[dist][1])


# ---- the full list against the oracle ---------------------------------------------------------------------------------
@pytest.mark.parametrize("dist", ["L2", "L2_SQUARED", "L1"])
@pytest.mark.parametrize("batch", [0, 10])
def test_full_list_against_the_oracle(dist, batch):
    tmpls, scene, fm, c = small(dist)
    tset = fdcm.TemplateSet(tmpls)
    for g in (fdcm.ScaleGrid(), S3, S5):
        for pen in (None, fdcm.DefaultPenalty(), PEN):
            check_list(fm, c, tset, tmpls, scene, g, batch=batch, penalty=pen)


def test_concentric_range_and_tmpl_idx_base():
    tmpls, scene, fm, c = small(seed=81)
    tset = fdcm.TemplateSet(tmpls)
    conc = ((120.0, 90.0), 20.0, 90.0)
    for g in (S3, fdcm.ScaleGrid(2, 1.3, 0.7)):
        check_list(fm, c, tset, tmpls, scene, g, 3, 5, 10, PEN, base=40, concentric=conc)
        check_list(fm, c, tset, tmpls, scene, g, 4, 4, 0, fdcm.DefaultPenalty(), base=7)


# ---- top-K, selection, refinement, coverage and fit ---------------------------------------------------------------------
def test_topk_and_ties():
    tmpls, scene, fm, c = small(seed=82)
    tset = fdcm.TemplateSet(tmpls)
    for pen in (None, PEN):
        want, _ = check_list(fm, c, tset, tmpls, scene, S5, penalty=pen, base=3)
        for k in (1, 10, 97, len(want) + 5):
            got = fdcm.search_topk(fm, tset, scene, fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), pen, k, 3, scales=S5)
            w = topk_ref(want, k)   # (want carries the base already)
            assert got.tobytes() == w.tobytes(), (pen, k)


SELECTS = [fdcm.DistinctMatches(max_per_template=1), fdcm.DistinctMatches(max_per_template=2),
           fdcm.DistinctMatches(radius=8.0), fdcm.DistinctMatches(radius=8.0, max_angle=0.3),
           fdcm.DistinctMatches(max_per_template=2, radius=10.0, max_angle=0.2),
           fdcm.DistinctMatches(radius=8.0, max_angle=0.3, across_templates=True),
           fdcm.DistinctMatches(max_per_template=1, radius=15.0, across_templates=True)]


@pytest.mark.parametrize("sel", SELECTS, ids=str)
def test_selection_against_the_model(sel):
    tmpls, scene, fm, c = small(seed=83)
    tset = fdcm.TemplateSet(tmpls)
    anchors = fdcm.get_template_anchors(tmpls)
    for base in (0, 11):
        want, rs = check_list(fm, c, tset, tmpls, scene, S5, penalty=PEN, base=base)
        for k in (5, 40):
            got = fdcm.search_topk(fm, tset, scene, fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), PEN, k, base, select=sel, scales=S5)
            w = select_ref(want, rs, anchors, k, sel, base)
            assert got.tobytes() == w.tobytes(), (sel, base, k)
    if sel.max_per_template == 1 and not sel.across_templates:
        assert len(np.unique(got["tmpl_idx"])) == len(got), "max_per_template counts a template over all its scales"


def test_refinement_coverage_and_fit_compose():
    tmpls, scene, fm, c = small(seed=84)
    tset = fdcm.TemplateSet(tmpls)
    anchors = fdcm.get_template_anchors(tmpls)
    ds, bo = fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10)
    r = fdcm.PoseRefinement(2, 2, 0.02, 2, 1.0)
    sel = fdcm.DistinctMatches(max_per_template=2, radius=6.0)
    full, rs = check_list(fm, c, tset, tmpls, scene, S3, penalty=PEN, base=5)
    for s in (None, sel):
        plain = fdcm.search_topk(fm, tset, scene, ds, bo, PEN, 12, 5, select=s, scales=S3)
        fused = fdcm.search_topk(fm, tset, scene, ds, bo, PEN, 12, 5, select=s, refine=r, scales=S3)
        assert fused.tobytes() == fdcm.refine_matches(fm, tset, plain, r, PEN, 5).tobytes(), ("refine", s)
        for fit in (fdcm.PoseFit(), fdcm.PoseFit(scale_range=(0.7, 1.4))):
            fitted = fdcm.search_topk(fm, tset, scene, ds, bo, PEN, 12, 5, select=s, fit=fit, scales=S3)
            assert fitted.tobytes() == fdcm.fit_matches(fm, tset, plain, fit, PEN, 5).tobytes(), ("fit", s, fit)
    # the coverage filter runs on the remapped records (it poses the original template), before the top-K or the selection
    cov = fdcm.EdgeCoverage(radius=2, bin_tolerance=1, min_coverage=0.4)
    cv = fdcm.match_coverage(fm, tset, full, cov, 5)
    keep = cv >= F32(0.4)
    assert 0 < keep.sum() < len(full), "the filter must drop some records and keep others"
    kept, krs = full[keep], rs[keep]
    for s in (None, sel):
        got = fdcm.search_topk(fm, tset, scene, ds, bo, PEN, 12, 5, select=s, verify=cov, scales=S3)
        if s is None:
            w = topk_ref(kept, 12)
        else:
            w = select_ref(kept, krs, anchors, 12, s, 5)
        assert got.tobytes() == w.tobytes(), ("coverage", s)
    # min_coverage == 0: no filter
    assert fdcm.search_topk(fm, tset, scene, ds, bo, PEN, 12, 5, verify=fdcm.EdgeCoverage(), scales=S3).tobytes() == \
        fdcm.search_topk(fm, tset, scene, ds, bo, PEN, 12, 5, scales=S3).tobytes()


# ---- one scale is the unscaled search ---------------------------------------------------------------------------------
def unit_scale_matches(fm, tmpls, scene, what):
    tset = fdcm.TemplateSet(tmpls)
    one = fdcm.ScaleGrid(1, 1.0, 1.7)
    ds, bo = fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10)
    a = fdcm.search_all(fm, tset, scene, ds, bo, PEN, 9)
    h, st = fm.last_hypotheses(), fm.last_search_stats()
    b = fdcm.search_all(fm, tset, scene, ds, bo, PEN, 9, scales=one)
    assert a.tobytes() == b.tobytes() and np.array_equal(h, fm.last_hypotheses()) and st == fm.last_search_stats(), what
    cov = fdcm.EdgeCoverage(min_coverage=0.3)
    r = fdcm.PoseRefinement(1, 2, 0.02, 2, 1.0)
    for kw in (dict(), dict(select=fdcm.DistinctMatches(max_per_template=1, radius=5.0, max_angle=0.4)), dict(refine=r),
               dict(select=fdcm.DistinctMatches(radius=9.0, across_templates=True), refine=r), dict(verify=cov),
               dict(select=fdcm.DistinctMatches(max_per_template=2), refine=r, verify=cov)):
        a = fdcm.search_topk(fm, tset, scene, ds, bo, PEN, 25, 9, **kw)
        h, st = fm.last_hypotheses(), fm.last_search_stats()
        b = fdcm.search_topk(fm, tset, scene, ds, bo, PEN, 25, 9, scales=one, **kw)
        assert a.tobytes() == b.tobytes(), (what, kw)
        assert np.array_equal(h, fm.last_hypotheses()) and st == fm.last_search_stats(), (what, kw)


def test_one_scale_is_byte_identical_synthetic():
    tmpls, scene, fm, _ = small(seed=85)
    unit_scale_matches(fm, tmpls, scene, "synthetic")


@pytest.mark.parametrize("obj", ["obj_01", "obj_02", "obj_03", "obj_04"])
def test_one_scale_is_byte_identical_real_assets(obj):
    tmpls, scenes = load_object(obj)
    fm = fdcm.build_cuda_featuremap(scenes[0], fdcm.Dt3CudaParameters(30, 5.0, 1.0))
    unit_scale_matches(fm, tmpls[:40], scenes[0], obj)


# ---- edge cases ---------------------------------------------------------------------------------------------------------
def test_edge_cases():
    tmpls, scene, fm, c = small(seed=86)
    assert len(fdcm.search_topk(fm, [], scene, fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), PEN, 5, scales=S3)) == 0
    n = C.c_int64(-1)
    empty = fdcm.TemplateSet([np.zeros((4, 0), F32)])
    p = _lib.SearchParams(4, 4, 10, 2, 1.5, 5, 0, 0, 0.0, 0.0, 0.0, 0.0)
    out = np.zeros(5, _lib.MATCH_DTYPE)
    assert _lib.lib().fdcm_search_scales(fm._h, empty._h, _lib.ptr(_lib_records(scene)), scene.shape[1], C.byref(p), C.byref(S3._params()),
                                         None, None, None, _lib.ptr(out), 5, C.byref(n)) == 0 and n.value == 0
    # empty and zero-length template lines, a scale whose copies leave the map, and 64 scales
    odd = [np.zeros((4, 0), F32), np.array([[30.0, 30.0], [40.0, 5.0], [30.0, 60.0], [40.0, 5.0]], F32)] + tmpls[:3]
    tset = fdcm.TemplateSet(odd)
    check_list(fm, c, tset, odd, scene, fdcm.ScaleGrid(3, 0.5, 4.0), penalty=PEN)   # 0.5, 2, 8
    check_list(fm, c, fdcm.TemplateSet(tmpls[:2]), tmpls[:2], scene, fdcm.ScaleGrid(64, 0.7, 1.01), penalty=fdcm.DefaultPenalty())


def _lib_records(scene):
    return np.ascontiguousarray(np.asarray(scene, F32).reshape(4, -1).T)


def test_selection_limit_counts_the_copies():
    # 2 * 40 lines * 2000 scene lines = 160000 hypotheses per copy: 210 templates are below 2^31 at one scale, above at 64
    tmpls = synth_templates(210, 40, 1920, seed=87)
    scene = synth_scene(1920, 1080, 2100, seed=88)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    per_copy = 2 * 40 * 2000
    assert 210 * per_copy < 2 ** 31 <= 210 * 64 * per_copy
    with pytest.raises(fdcm.FdcmError, match="2\\^31"):
        fdcm.search_topk(fm, tmpls, scene, fdcm.DefaultSearch(40, 2000), fdcm.BatchOptimize(10), PEN, 10,
                         select=fdcm.DistinctMatches(max_per_template=1), scales=fdcm.ScaleGrid(64, 0.9, 1.001))


# ---- the per-map cache of the copies ------------------------------------------------------------------------------------
def test_cache_follows_the_grid_the_penalty_and_the_template_load():
    tmpls, scene, fm, c = small(seed=89)
    tset = fdcm.TemplateSet(tmpls)
    ds, bo = fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10)
    want = {}
    for g in (S3, S5):
        for pen in (PEN, fdcm.DefaultPenalty()):
            want[(g.scales, type(pen).__name__)], _ = remap(oracle_penalized(c.search(copies(tmpls, g), scene, 4, 4, batch=10), copies(tmpls, g),
                                                                             pen), g)
    flat, off = fdcm._pack(tmpls[:2])
    s = _lib_records(scene)
    for rnd in range(2):
        for g in (S3, S5, S3):
            for pen in (PEN, fdcm.DefaultPenalty()):
                got = fdcm.search_all(fm, tset, scene, ds, bo, pen, scales=g)
                assert got.tobytes() == want[(g.scales, type(pen).__name__)].tobytes(), (rnd, g, pen)
            # fdcm_search_host reloads the map's own template set in between
            p = _lib.SearchParams(4, 4, 10, 2, 1.5, 5, 0, 0, 0.0, 0.0, 0.0, 0.0)
            out, n = np.zeros(5, _lib.MATCH_DTYPE), C.c_int64(0)
            _lib.check(_lib.lib().fdcm_search_host(fm._h, _lib.ptr(flat), _lib.ptr(off), 2, _lib.ptr(s), s.shape[0], C.byref(p), _lib.ptr(out), 5,
                                                   C.byref(n)))
    # a new template set (a new load) with the same grid
    other = tmpls[1:] + tmpls[:1]
    cp = copies(other, S3)
    w, _ = remap(oracle_penalized(c.search(cp, scene, 4, 4, batch=10), cp, PEN), S3)
    assert fdcm.search_all(fm, fdcm.TemplateSet(other), scene, ds, bo, PEN, scales=S3).tobytes() == w.tobytes()


def test_two_threads_share_a_set_with_different_grids():
    tmpls, scene = synthetic(n_tmpl=30, n_lines=12, seed=90, w=400, h=300, n_scene=150)
    tset = fdcm.TemplateSet(tmpls)
    maps = [fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5)) for _ in range(2)]
    grids = (S3, S5)
    ds, bo = fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10)
    sel = fdcm.DistinctMatches(max_per_template=1)

    def run(i):
        return [fdcm.search_topk(maps[i], tset, scene, ds, bo, PEN, 50, select=sel, scales=grids[i]).tobytes() for _ in range(6)]

    serial = [run(0)[0], run(1)[0]]
    got, errs = [None, None], []

    def worker(i):
        try:
            got[i] = run(i)
        except Exception as e:   # pragma: no cover
            errs.append(e)

    th = [threading.Thread(target=worker, args=(i,)) for i in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errs, errs
    for i in range(2):
        assert all(x == serial[i] for x in got[i]), i
    assert serial[0] != serial[1]


# ---- planted instances --------------------------------------------------------------------------------------------------
def test_planted_scaled_instances_are_found_and_fitted():
    """Noise-free instances at s = 0.85, 1.0 and 1.15 (the grid has 0.85, 1.0 and 1.1765): each template is found once, at
    its instance, and the scaled fit brings it to within 0.01 px and 1e-4 relative scale."""
    rng = np.random.default_rng(91)
    pts = [(0, 0), (100, 0), (100, 30), (40, 70), (0, 50)]   # an outline of pairwise distinct side lengths, unlike a triangle's
    other = np.array([(*pts[i], *pts[(i + 1) % 5]) for i in range(5)] + [(15, 10, 70, 25)], F32).T.copy()
    tmpls = [house(), other]
    anchors = fdcm.get_template_anchors(tmpls)
    fit = fdcm.PoseFit(iterations=30, max_distance=6.0, scale_range=(0.7, 1.4))
    sel = fdcm.DistinctMatches(max_per_template=1)
    for s_true in (0.85, 1.0, 1.15):
        truths = [spose(rng.uniform(-math.pi, math.pi), s_true, 110 + 200 * i, rng.uniform(110, 190)) for i in range(2)]
        scene = np.concatenate([posed(tmpls[i], truths[i]) for i in range(2)], axis=1)
        fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
        got = fdcm.search_topk(fm, tmpls, scene, fdcm.DefaultSearch(4, 12), fdcm.BatchOptimize(10), fdcm.DefaultPenalty(), 2, select=sel,
                               scales=S3, fit=fit)
        assert sorted(got["tmpl_idx"].tolist()) == [0, 1], s_true
        for m in got:
            t = int(m["tmpl_idx"])
            a = np.array([anchors[t][0], anchors[t][1], 1.0])
            e_a = float(np.hypot(*(m["transform"].astype(np.float64).reshape(2, 3) @ a - truths[t].reshape(2, 3) @ a)))
            assert e_a < 0.01 and scale_error(m["transform"], truths[t]) < 1e-4, (s_true, t, e_a, scale_error(m["transform"], truths[t]))


def test_pybind_and_profile_names():
    from openfdcm_b200 import _openfdcm_cuda as pyfdcm
    tmpls, scene, fm, _ = small(seed=92)
    pfm = pyfdcm.build_cuda_featuremap(scene, pyfdcm.Dt3CudaParameters(30, 5.0, 1.5))
    sel = fdcm.DistinctMatches(max_per_template=1)
    want = fdcm.search_topk(fm, tmpls, scene, fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), PEN, 8, select=sel, scales=S3)
    got = pyfdcm.search_topk(pfm, tmpls, scene, pyfdcm.DefaultSearch(4, 4), pyfdcm.BatchOptimize(10), pyfdcm.ExponentialPenalty(1.5), 8,
                             select=pyfdcm.DistinctMatches(max_per_template=1), scales=pyfdcm.ScaleGrid(3, 0.85, 1.0 / 0.85))
    assert [m.tmpl_idx for m in got] == want["tmpl_idx"].tolist()
    assert np.array_equal(np.array([m.score for m in got], F32), want["score"])
    fdcm.profile(True, reset=True)
    try:
        fdcm.search_topk(fm, tmpls, scene, fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), PEN, 8, scales=S3)
        rep = fdcm.profile_report()
    finally:
        fdcm.profile(False, reset=True)
    assert rep["search"]["launches"] == 1 and rep["search_scale_remap"]["launches"] == 1
