"""Scale as a pose dimension on the device: fdcm_search_dense_scales against the numpy model of tests/models/dense.py
(scores through fdcm_dt3_evaluate, as tests/test_gpu_dense.py does), byte-identity with the unscaled search at one scale,
composition with refinement, the coverage filter and the fit, fdcm_fit_matches_scaled against the float64 model, recovery of
planted scaled instances, edge cases and the interfaces."""
import math

import numpy as np
import pytest

import openfdcm_b200 as fdcm
from openfdcm_b200 import _lib
from tests.helpers import device_scores, evaluate_fn, fit_candidates, house, load_object, posed, scale_error, spose, synthetic
from tests.models.dense import dense_records, output_model, penalised, scale_values
from tests.models.fit import SceneLines, fit_model
from tests.util import F32, synth_scene, synth_templates

pytestmark = pytest.mark.gpu
PEN = fdcm.ExponentialPenalty(1.5)


def model(fm, tmpls, d, g, tmpl_idx_base=0):
    return dense_records(tmpls, fdcm.get_template_anchors(tmpls), d, fm.get_scene_translation(), fm.width, fm.height, evaluate_fn(fm),
                         tmpl_idx_base, g)


def check_dense(fm, tset, tmpls, d, g, what, pens=(None, PEN), tmpl_idx_base=0):
    rec, valid, rs = model(fm, tmpls, d, g, tmpl_idx_base)
    anchors = fdcm.get_template_anchors(tmpls)
    lengths = fdcm.get_template_lengths(tmpls)
    n_valid = int(valid.sum())
    for pen in pens:
        prec = penalised(rec, valid, lengths, pen, g)
        for k, sel in ((1, None), (10, None), (min(max(n_valid, 1), 500), None), (10, fdcm.DistinctMatches(max_per_template=1)),
                       (10, fdcm.DistinctMatches(radius=6.0, max_angle=0.3)),
                       (10, fdcm.DistinctMatches(radius=6.0, max_angle=0.3, across_templates=True))):
            got = fdcm.search_dense(fm, tset, d, pen, k, tmpl_idx_base, select=sel, scales=g)
            want = output_model(prec, valid, k, anchors, sel, tmpl_idx_base, rs)
            assert got.tobytes() == want.tobytes(), f"{what} {g} {pen} k={k} {sel}: got {got[:3]} want {want[:3]}"
    return rec, valid


def small(dist=fdcm.distance.L2, seed=60):
    tmpls, scene = synthetic(n_tmpl=4, n_lines=8, seed=seed, w=200, h=150, n_scene=60)
    return tmpls, scene, fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5, dist))


# ---- the scaled dense records, bit for bit ---------------------------------------------------------------------------
@pytest.mark.parametrize("dist", [fdcm.distance.L2, fdcm.distance.L2_SQUARED, fdcm.distance.L1])
def test_synthetic_bit_exact(dist):
    tmpls, scene, fm = small(dist)
    tset = fdcm.TemplateSet(tmpls)
    for d, g in ((fdcm.DenseSearch(7, rot_start=0.1, stride=3, cell=4), fdcm.ScaleGrid(3, 0.85, 1.0 / 0.85)),
                 (fdcm.DenseSearch(1, rot_start=0.0, stride=2, cell=5, roi=(20.0, 10.5, 150.25, 120.0)), fdcm.ScaleGrid(4, 1.3, 0.8))):
        rec, valid = check_dense(fm, tset, tmpls, d, g, f"synthetic {dist}")
        assert valid.any()


def test_tmpl_idx_base_and_default_penalty():
    tmpls, scene, fm = small(seed=61)
    check_dense(fm, fdcm.TemplateSet(tmpls), tmpls, fdcm.DenseSearch(5, rot_start=-0.4, rot_step=0.2, stride=5, cell=3),
                fdcm.ScaleGrid(2, 0.9, 1.2), "base 50", pens=(fdcm.DefaultPenalty(),), tmpl_idx_base=50)


@pytest.mark.parametrize("obj", ["obj_01", "obj_02", "obj_03", "obj_04"])
def test_real_assets_bit_exact(obj):
    tmpls, scenes = load_object(obj)
    tmpls = tmpls[:3]
    tset = fdcm.TemplateSet(tmpls)
    fm = fdcm.build_cuda_featuremap(scenes[0], fdcm.Dt3CudaParameters(30, 5.0, 1.0))
    d, g = fdcm.DenseSearch(12, stride=8, cell=4), fdcm.ScaleGrid(3, 0.9, 1.1)
    rec, valid, rs = model(fm, tmpls, d, g)
    anchors, lengths = fdcm.get_template_anchors(tmpls), fdcm.get_template_lengths(tmpls)
    for pen in (PEN, fdcm.DefaultPenalty()):
        prec = penalised(rec, valid, lengths, pen, g)
        for sel in (None, fdcm.DistinctMatches(max_per_template=1), fdcm.DistinctMatches(radius=20.0, max_angle=0.2, across_templates=True)):
            want = output_model(prec, valid, 10, anchors, sel, rs=rs)
            got = fdcm.search_dense(fm, tset, d, pen, 10, select=sel, scales=g)
            assert got.tobytes() == want.tobytes(), f"{obj} {pen} {sel}"


# ---- one scale is the unscaled search --------------------------------------------------------------------------------
def test_one_scale_is_byte_identical_to_the_unscaled_search():
    tmpls, scene, fm = small(seed=62)
    tset = fdcm.TemplateSet(tmpls)
    d = fdcm.DenseSearch(12, stride=3, cell=4)
    cov = fdcm.EdgeCoverage(radius=2, min_coverage=0.3)
    for g in (fdcm.ScaleGrid(), fdcm.ScaleGrid(1, 1.0, 3.0)):
        for pen in (None, PEN, fdcm.DefaultPenalty()):
            for sel in (None, fdcm.DistinctMatches(max_per_template=1), fdcm.DistinctMatches(radius=6.0, max_angle=0.3, across_templates=True)):
                for ref in (None, fdcm.PoseRefinement(2, 1, 0.03, 2, 0.5)):
                    for ver in (None, cov):
                        kw = dict(select=sel, refine=ref, verify=ver)
                        a = fdcm.search_dense(fm, tset, d, pen, 10, **kw)
                        b = fdcm.search_dense(fm, tset, d, pen, 10, scales=g, **kw)
                        assert a.tobytes() == b.tobytes(), (g, pen, sel, ref, ver)


# ---- composition -----------------------------------------------------------------------------------------------------
def test_composed_refine_fit_and_coverage():
    tmpls, scene, fm = small(seed=63)
    tset = fdcm.TemplateSet(tmpls)
    d, g = fdcm.DenseSearch(12, stride=3, cell=4), fdcm.ScaleGrid(3, 0.9, 1.1)
    sel = fdcm.DistinctMatches(max_per_template=2)
    for pen in (None, PEN):
        base = fdcm.search_dense(fm, tset, d, pen, 10, select=sel, scales=g)
        assert len(base) == 8   # 4 templates, at most 2 each over all scales
        for r in (fdcm.PoseRefinement(), fdcm.PoseRefinement(2, 1, 0.03, 3, 0.5)):
            fused = fdcm.search_dense(fm, tset, d, pen, 10, select=sel, refine=r, scales=g)
            want = fdcm.refine_matches(fm, tset, base, r, penalty=pen)
            assert fused.tobytes() == want.tobytes(), r
            # refinement rotates the pose: each record keeps its scale
            s0 = np.hypot(base["transform"][:, 0], base["transform"][:, 3])
            s1 = np.hypot(fused["transform"][:, 0], fused["transform"][:, 3])
            assert np.allclose(s0, s1, rtol=1e-5)
        for fit in (fdcm.PoseFit(), fdcm.PoseFit(scale_range=(0.8, 1.25))):
            fused = fdcm.search_dense(fm, tset, d, pen, 10, select=sel, scales=g, fit=fit)
            assert fused.tobytes() == fdcm.fit_matches(fm, tset, base, fit, pen).tobytes(), fit
    # the coverage filter equals match_coverage applied to the records before the selection
    cov = fdcm.EdgeCoverage(radius=2, min_coverage=0.4)
    rec, valid, rs = model(fm, tmpls, d, g)
    c = fdcm.match_coverage(fm, tset, rec[valid], cov)
    keep = valid.copy()
    keep[np.flatnonzero(valid)] = c >= F32(0.4)
    prec = penalised(rec, keep, fdcm.get_template_lengths(tmpls), PEN, g)
    for s in (None, sel):
        got = fdcm.search_dense(fm, tset, d, PEN, 10, select=s, verify=cov, scales=g)
        assert got.tobytes() == output_model(prec, keep, 10, fdcm.get_template_anchors(tmpls), s, rs=rs).tobytes(), s


# ---- the scaled fit, bit for bit -------------------------------------------------------------------------------------
def check_fit(fm, scene, tmpls, matches, fit, penalty=None):
    got, gst = fdcm.fit_matches(fm, tmpls, matches, fit, penalty, return_stats=True)
    sc = SceneLines.of(scene, fm.get_scene_translation(), fm.scene_bins(), fm.depth, fm.width, fm.height)
    scores = device_scores(fm)
    want, wst = fit_model(sc, tmpls, fdcm.get_template_anchors(tmpls), matches, fit,
                          lambda tmpl, F: scores([(tmpl, F.reshape(1, 6))])[0])
    if penalty is not None:
        want = fdcm.penalize(penalty, want, fdcm.get_template_lengths(tmpls))
    bad = np.flatnonzero([a.tobytes() != b.tobytes() for a, b in zip(got, want)])
    assert len(bad) == 0, (bad[:5], got[bad[:2]], want[bad[:2]])
    assert gst.tobytes() == wst.tobytes(), np.flatnonzero([a.tobytes() != b.tobytes() for a, b in zip(gst, wst)])[:10]
    return got, gst


def scaled_candidates(fm, tmpls, scene, n, seed):
    """fit_candidates() of the rigid fit tests, some of them scaled by up to 6 % about their origin."""
    m = fit_candidates(fm, tmpls, scene, n, seed)
    rng = np.random.default_rng(seed)
    f = rng.uniform(0.94, 1.06, len(m)).astype(F32)
    f[::3] = F32(1)
    m["transform"][:, [0, 1, 3, 4]] *= f[:, None]
    return m


@pytest.mark.parametrize("dist", [fdcm.distance.L2, fdcm.distance.L2_SQUARED, fdcm.distance.L1])
def test_scaled_fit_synthetic_against_the_model(dist):
    tmpls, scene = synthetic(n_tmpl=10, seed=700)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5, dist))
    m = scaled_candidates(fm, tmpls, scene, 30, 1)
    got, st = check_fit(fm, scene, tmpls, m, fdcm.PoseFit(scale_range=(0.8, 1.25)), PEN)
    assert np.isnan(got[-3:]["score"]).all() and (st["iterations"][:-3] > 0).any()
    check_fit(fm, scene, tmpls, m[::3], fdcm.PoseFit(iterations=3, max_distance=6.0, sample_step=0.75, bin_tolerance=0, min_inliers=3,
                                                     scale_range=(0.97, 1.03)))


def test_scaled_fit_real_assets():
    for obj in ("obj_01", "obj_02", "obj_03", "obj_04"):
        tmpls, scenes = load_object(obj)
        fm = fdcm.build_cuda_featuremap(scenes[0], fdcm.Dt3CudaParameters(30, 5.0, 2.2))
        check_fit(fm, scenes[0], tmpls, scaled_candidates(fm, tmpls, scenes[0], 10, 2), fdcm.PoseFit(scale_range=(0.8, 1.25)), PEN)


def test_scaled_fit_literal_path_map():
    tmpls = synth_templates(4, 12, 2000, seed=720)
    scene = synth_scene(3000, 3000, 120, seed=721)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.05))
    assert fm.width > 2897
    check_fit(fm, scene, tmpls, scaled_candidates(fm, tmpls, scene, 12, 3), fdcm.PoseFit(max_distance=16.0, scale_range=(0.5, 2.0)))


# ---- recovery of planted scaled instances ----------------------------------------------------------------------------
def test_dense_scales_then_scaled_fit_recovers_noise_free_instances():
    """Clean scenes (the instance only): dense at 3 scales, distinct selection, then the scaled fit."""
    tmpl = house()
    a = fdcm.get_template_anchors([tmpl])[0]
    rng = np.random.default_rng(740)
    g = fdcm.ScaleGrid(3, 0.85, 1.0 / 0.85)   # 0.85, 1.0, 1.1765
    d = fdcm.DenseSearch(72, stride=2, cell=8)
    fit = fdcm.PoseFit(iterations=30, max_distance=6.0, scale_range=(0.7, 1.4))
    for s_true in (0.85, 1.0, 1.15):
        truth = spose(rng.uniform(-math.pi, math.pi), s_true, rng.uniform(120, 280), rng.uniform(120, 280))
        scene = posed(tmpl, truth)
        fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
        got = fdcm.search_dense(fm, [tmpl], d, fdcm.DefaultPenalty(), 1, select=fdcm.DistinctMatches(max_per_template=1), scales=g, fit=fit)
        assert len(got) == 1
        T = got[0]["transform"].astype(np.float64).reshape(2, 3)
        e_a = float(np.hypot(*(T @ np.array([a[0], a[1], 1.0]) - truth.reshape(2, 3) @ np.array([a[0], a[1], 1.0]))))
        assert e_a < 0.01 and scale_error(got[0]["transform"], truth) < 1e-4, (s_true, e_a, scale_error(got[0]["transform"], truth))


# ---- edge cases and interfaces ---------------------------------------------------------------------------------------
def test_edge_cases():
    tmpls, scene, fm = small(seed=64)
    d, g = fdcm.DenseSearch(6, stride=3, cell=4), fdcm.ScaleGrid(2, 0.9, 1.2)
    assert len(fdcm.search_dense(fm, [], d, scales=g)) == 0
    empty_fm = fdcm.build_cuda_featuremap(np.zeros((4, 0), F32), fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    assert len(fdcm.search_dense(empty_fm, tmpls, d, scales=g)) == 0
    assert len(fdcm.search_dense(fm, tmpls, fdcm.DenseSearch(6, roi=(1e5, 1e5, 2e5, 2e5)), scales=g)) == 0
    with_empty = tmpls[:2] + [np.zeros((4, 0), F32)] + tmpls[2:]
    check_dense(fm, fdcm.TemplateSet(with_empty), with_empty, d, g, "empty template", pens=(PEN,))
    # the fit of an empty map: every input invalid
    m = fdcm.search_dense(fm, tmpls, d, None, 3, scales=g)
    out, st = fdcm.fit_matches(empty_fm, tmpls, m, fdcm.PoseFit(scale_range=(0.5, 2.0)), return_stats=True)
    assert np.isnan(out["score"]).all() and (st["n_samples"] == 0).all()


def test_record_limit_counts_the_scales():
    tmpls, scene, fm = small(seed=65)
    # one template: 4096 rotations x (cells of a 1-px stride, 1-px cell grid) is below 2^31 at one scale, above at 64
    d = fdcm.DenseSearch(4096, stride=1, cell=1)
    per_scale = 4096 * fm.width * fm.height
    assert per_scale < 2 ** 31 and per_scale * 64 >= 2 ** 31
    with pytest.raises(fdcm.FdcmError, match="2\\^31"):
        fdcm.search_dense(fm, tmpls[:1], d, None, 10, scales=fdcm.ScaleGrid(64, 0.9, 1.001))


def test_invalid_parameters():
    tmpls, scene, fm = small(seed=66)
    d = fdcm.DenseSearch(6)
    for g in (fdcm.ScaleGrid(0), fdcm.ScaleGrid(65), fdcm.ScaleGrid(2, 0.0), fdcm.ScaleGrid(2, 1.0, math.nan), fdcm.ScaleGrid(64, 1.0, 1e10)):
        with pytest.raises(fdcm.FdcmError, match="scale"):
            fdcm.search_dense(fm, tmpls, d, scales=g)
    for bad in (dict(select=fdcm.DistinctMatches(max_per_template=-1)), dict(refine=fdcm.PoseRefinement(levels=0)),
                dict(verify=fdcm.EdgeCoverage(radius=99))):
        with pytest.raises(fdcm.FdcmError):
            fdcm.search_dense(fm, tmpls, d, scales=fdcm.ScaleGrid(2, 0.9, 1.1), **bad)
    with pytest.raises(fdcm.FdcmError):
        fdcm.search_dense(fm, tmpls, fdcm.DenseSearch(0), scales=fdcm.ScaleGrid())
    m = fdcm.search_dense(fm, tmpls, d, None, 3)
    for r in ((0.0, 1.0), (1.2, 1.1), (math.nan, 1.0)):
        with pytest.raises(fdcm.FdcmError, match="scale"):
            fdcm.fit_matches(fm, tmpls, m, fdcm.PoseFit(scale_range=r))
    bad = m.copy()
    bad["tmpl_idx"] = 99
    with pytest.raises(IndexError):
        fdcm.fit_matches(fm, tmpls, bad, fdcm.PoseFit(scale_range=(0.5, 2.0)))


def test_denominator_cache_across_scale_grids():
    """One map searched at S = 1, then at S = 4, then S = 1 again with the same penalty: each call reads its own
    denominators (a cache of T entries is never read as one of T x S)."""
    tmpls, scene, fm = small(seed=67)
    tset = fdcm.TemplateSet(tmpls)
    d = fdcm.DenseSearch(6, stride=4, cell=4)
    g4 = fdcm.ScaleGrid(4, 0.8, 1.15)
    want1 = fdcm.search_dense(fm, tset, d, PEN, 20)
    rec, valid, rs = model(fm, tmpls, d, g4)
    want4 = output_model(penalised(rec, valid, fdcm.get_template_lengths(tmpls), PEN, g4), valid, 20)
    for _ in range(2):
        assert fdcm.search_dense(fm, tset, d, PEN, 20, scales=fdcm.ScaleGrid()).tobytes() == want1.tobytes()
        assert fdcm.search_dense(fm, tset, d, PEN, 20, scales=g4).tobytes() == want4.tobytes()
        assert fdcm.search_dense(fm, tset, d, PEN, 20).tobytes() == want1.tobytes()
        # refinement after a scaled search uses the per-template denominators
        r = fdcm.PoseRefinement(1, 1, 0.02, 1, 1.0)
        fused = fdcm.search_dense(fm, tset, d, PEN, 5, refine=r, scales=g4)
        assert fused.tobytes() == fdcm.refine_matches(fm, tset, want4[:5], r, penalty=PEN).tobytes()


def test_pybind_and_profile_names():
    from openfdcm_b200 import _openfdcm_cuda as pyfdcm
    tmpls, scene, fm = small(seed=68)
    pfm = pyfdcm.build_cuda_featuremap(scene, pyfdcm.Dt3CudaParameters(30, 5.0, 1.5))
    g = pyfdcm.ScaleGrid(3, 0.9, 1.1)
    assert "ScaleGrid" in repr(g) and (g.scales, g.start) == (3, pytest.approx(0.9))
    d = fdcm.DenseSearch(12, stride=3, cell=4)
    pd = pyfdcm.DenseSearch(12, stride=3, cell=4)
    want = fdcm.search_dense(fm, tmpls, d, PEN, 8, select=fdcm.DistinctMatches(max_per_template=1), scales=fdcm.ScaleGrid(3, 0.9, 1.1))
    got = pyfdcm.search_dense(pfm, tmpls, pd, pyfdcm.ExponentialPenalty(1.5), 8, select=pyfdcm.DistinctMatches(max_per_template=1), scales=g)
    assert [m.tmpl_idx for m in got] == want["tmpl_idx"].tolist()
    assert np.array_equal(np.array([m.score for m in got], F32), want["score"])
    pf = pyfdcm.PoseFit(iterations=4, scale_range=(0.8, 1.25))
    assert pf.scale_range == pytest.approx((0.8, 1.25)) and pyfdcm.PoseFit().scale_range is None
    fitted = pyfdcm.fit_matches(pfm, tmpls, got, pf, pyfdcm.ExponentialPenalty(1.5))
    wfit = fdcm.fit_matches(fm, tmpls, want, fdcm.PoseFit(iterations=4, scale_range=(0.8, 1.25)), PEN)
    assert np.array_equal(np.array([m.score for m in fitted], F32), wfit["score"])
    fdcm.profile(True, reset=True)
    try:
        fdcm.search_dense(fm, tmpls, d, PEN, 8, scales=fdcm.ScaleGrid(3, 0.9, 1.1))
        fdcm.fit_matches(fm, tmpls, want, fdcm.PoseFit(scale_range=(0.8, 1.25)))
        fdcm.fit_matches(fm, tmpls, want, fdcm.PoseFit())
        rep = fdcm.profile_report()
    finally:
        fdcm.profile(False, reset=True)
    assert rep["dense_eval"]["launches"] == 1 and rep["dense_finish"]["launches"] == 1
    assert rep["fit_eval_scaled"]["launches"] == 1 and rep["fit_eval"]["launches"] == 1
    assert scale_values(fdcm.ScaleGrid(3, 0.9, 1.1)).dtype == F32 and _lib.ScaleGridParams is not None
