"""The DT3 build at the edges of the map geometry, bit-exact against the CPU oracle: maps of side 1 to 165 (the 32-float
pitch, one 32-row band, images smaller than the integral's TMA boxes and 128-chain strips), degenerate scene extents,
the exact / literal boundary at side 2897 / 2898, scenes far from the origin whose shifted end points leave the map (the
raster kernel's clipping), and rebuilds of one handle across sizes.

The build picks its kernels from the geometry (run_build_kernels); every case asserts, from profile_report() names of a
separate profiled build, the path it is meant to reach, and the last test asserts that the module reached all of them.
"""
import math

import numpy as np
import pytest

import openfdcm_b200 as fdcm
from oracle import fdcm_oracle as orc
from tests.helpers import (BOUNDARY, DIST, FAR, TINY, assert_matches, check_full_search, far_scene, host_geometry, map_templates,
                           oracle_penalized, pinned_scene, refine_reference, shifted_scene, topk_ref)
from tests.models.select import select_model
from tests.util import F32, plant_instances, synth_templates

pytestmark = pytest.mark.gpu
PEN = fdcm.ExponentialPenalty(1.5)
OPT = fdcm.BatchOptimize(10)

# ---- build paths ----------------------------------------------------------------------------------------------------
PATHS = ("band_split", "band_fused", "band_unfused", "literal", "l1_fused", "l1_unfused")
REACHED = set()


def path_of(names):
    """The DT path of one build from its profile_report() names."""
    found = []
    if {"dt_row_envelope_far", "dt_fill_propagate_far"} <= names:
        found.append("band_split")
    if "dt_fill_propagate" in names and not any(n.endswith("_far") for n in names):
        found.append("band_fused")
    if "dt_row_fill" in names:
        found.append("band_unfused")
    if {"dt_col_literal", "dt_row_literal"} <= names:
        found.append("literal")
    if "dt_l1_propagate" in names:
        found.append("l1_fused")
    if "dt_row_l1_band" in names:
        found.append("l1_unfused")
    assert len(found) == 1, f"one DT path per build, got {found} from {sorted(names)}"
    return found[0]


def build_path(scene, params, stage=0):
    """Build-kernel names of a separate, profiled build of `scene`."""
    fdcm.profile(True, reset=True)
    try:
        fdcm.build_cuda_featuremap(scene, params, stage=stage)
    finally:
        fdcm.profile(False)
    return set(fdcm.profile_report())


# ---- generators ---------------------------------------------------------------------------------------------------
def leaves_map(scene, padding):
    """Whether some shifted fp32 end point lies outside [0, W-1], so that the raster kernel has to clip."""
    shift, side = host_geometry(scene, padding)
    ts = shifted_scene(scene, shift)
    return bool(((ts < 0) | (ts > F32(side - 1))).any())


def check_generators():
    """The CPU-side properties the cases rely on (no GPU needed): pinned_scene gives maps of exactly `side`, and at every
    offset the padding-1.0 far scenes have a shifted fp32 end point outside the map, with host_geometry equal to the
    oracle's scene shift."""
    for side in TINY + BOUNDARY:
        c = orc.Dt3Cpu(pinned_scene(side, 12, side), 1, 5.0, 1.0)
        assert (c.W, c.H) == (side, side), f"pinned_scene({side}) gives a map of {c.W}"
    for offset in FAR:
        for source in ("small", "synthetic"):
            scene, _ = far_scene(offset, source)
            for padding in (1.0, 1.5):
                shift, side = host_geometry(scene, padding)
                oshift, osize = orc.scene_shift(scene, padding)
                assert shift.tobytes() == oshift.tobytes() and osize.tolist() == [side, side], (offset, source, padding)
            assert leaves_map(scene, 1.0), f"the {source} scene at offset {offset} stays inside the map"


def test_generators():
    check_generators()


# ---- checks ---------------------------------------------------------------------------------------------------------
def expected_path(scene, padding, dist, depth, stage):
    """The DT path run_build_kernels takes: L1 fused at depth 30 unless stage 1; L2 / L2^2 literal beyond side 2897,
    else fused at depth 30 unless stage 1, split when the 32-row bands that hold the scene's rows (rows floor(min y) - 1
    to ceil(max y) + 1 of the shifted scene) are not all of them."""
    shift, side = host_geometry(scene, padding)
    fused = depth == 30 and stage != 1
    if dist == "L1":
        return "l1_fused" if fused else "l1_unfused"
    if 2.0 * (side - 1) ** 2 >= 2 ** 24:
        return "literal"
    if not fused:
        return "band_unfused"
    ys = shifted_scene(scene, shift)[[1, 3]].astype(np.float64)
    row_lo = min(max(math.floor(ys.min()) - 1, 0), side - 1)
    row_hi = min(max(math.ceil(ys.max()) + 1, 0), side - 1)
    return "band_split" if (row_lo >> 5) > 0 or ((row_hi >> 5) + 1) * 32 < side else "band_fused"


def assert_plane(got, want, what):
    if np.array_equal(got, want):
        return
    if got.shape != want.shape:
        pytest.fail(f"{what}: shape {got.shape} != {want.shape}")
    bad = np.argwhere(~((got == want) | (np.isnan(got) & np.isnan(want))))
    y, x = bad[0]
    rel = np.abs(got.astype(np.float64) - want) / np.maximum(np.abs(want.astype(np.float64)), 1e-30)
    pytest.fail(f"{what}: {len(bad)} pixels differ, first at (x={x}, y={y}): {got[y, x]!r} != {want[y, x]!r}, "
                f"max relative difference {np.nanmax(rel):.3g}")


def check_map(g, c, scene, stage=0, planes=None, what=""):
    """Size, translation, angle keys, planes, scene bins (closest_orientation of the shifted scene) and, at stage 1, the
    edge masks."""
    assert (g.width, g.height, g.depth) == (c.W, c.H, c.depth), what
    assert g.get_scene_translation().tobytes() == c.shift.tobytes(), f"{what}: {g.get_scene_translation()} != {c.shift}"
    assert g.angles().tobytes() == c.keys.tobytes(), what
    for d in range(c.depth) if planes is None else planes:
        want = c.plane(d)
        assert_plane(g.plane(d), want, f"{what} plane {d}")
        if stage == 1:
            assert np.array_equal(g.mask(d), (want == 0).astype(np.uint8)), f"{what}: edge mask of plane {d}"
    ts = shifted_scene(scene, c.shift)
    bins = np.array([orc.closest_orientation(c.keys, ts[:, i]) for i in range(ts.shape[1])], np.int32)
    assert np.array_equal(g.scene_bins(), bins), f"{what}: scene bins"


def check_search(g, c, tmpls, scene, max_t, max_s, batches=(10,), what=""):
    """search_all (hypotheses, counters, every match) for each batch size, and the penalised top-10 of BatchOptimize(10)."""
    for batch in batches:
        raw, _ = check_full_search(g, c, tmpls, scene, max_t, max_s, batch)
        if batch == 10:
            raw10 = raw
    top = fdcm.search_topk(g, tmpls, scene, fdcm.DefaultSearch(max_t, max_s), OPT, PEN, k=10)
    assert_matches(top, topk_ref(oracle_penalized(raw10, tmpls, PEN), 10), f"{what} top-10")
    return raw10


ALIGNS = [[1, 0], [0, 1], [-1, 0], [0, -1], [1, 1], [0.3, -1], [-1, 0.45]]


def check_minmax_and_optimize(g, c, tmpls, what=""):
    """minmax_translation and optimize() of the templates placed at the map centre, for axis-aligned and oblique
    alignment vectors."""
    centre = (np.full(2, (c.W - 1) / 2, F32) - c.shift).astype(F32)
    placed = [(t.T.reshape(-1, 2) + centre).reshape(-1, 4).T.astype(F32) for t in tmpls]
    cases = [(t, np.array(v, F32)) for t in placed for v in ALIGNS]
    for i, (t, v) in enumerate(cases):
        assert np.array_equal(fdcm.minmax_translation(g, t, v), c.minmax_translation(t, v), equal_nan=True), f"{what} case {i}"
    for batch in (10, 0):
        got = fdcm.optimize(fdcm.BatchOptimize(batch) if batch else fdcm.DefaultOptimize(), [t for t, _ in cases], [v for _, v in cases], g)
        for i, ((t, v), r) in enumerate(zip(cases, got)):
            has, score, tr = c.optimize_one(t, v, batch)
            assert (r is not None) == has, f"{what} batch {batch} case {i}"
            if has:
                assert r[0] == score and np.array_equal(r[1], tr), f"{what} batch {batch} case {i}: {r} != {(score, tr)}"


def build_both(scene, depth, padding, dist, stage=0):
    gd, od = DIST[dist]
    params = fdcm.Dt3CudaParameters(depth, 5.0, padding, gd)
    want = expected_path(scene, padding, dist, depth, stage)
    got = path_of(build_path(scene, params, stage))
    assert got == want, f"expected the {want} path, the build ran {got}"
    REACHED.add(got)
    return fdcm.build_cuda_featuremap(scene, params, stage=stage), orc.Dt3Cpu(scene, depth, 5.0, padding, od, stage=stage)


# ---- 1. tiny maps ---------------------------------------------------------------------------------------------------
TINY_CASES = [(dist, depth, stage) for depth in (30, 7) for dist, stage in (("L2", 0), ("L2", 1), ("L2", 2), ("L2_SQUARED", 0), ("L1", 0))]


@pytest.mark.parametrize("dist,depth,stage", TINY_CASES, ids=[f"{d}-depth{n}-stage{s}" for d, n, s in TINY_CASES])
@pytest.mark.parametrize("side", TINY)
def test_tiny_maps(side, dist, depth, stage):
    scene = pinned_scene(side, 12, seed=side)
    g, c = build_both(scene, depth, 1.0, dist, stage)
    what = f"side {side} {dist} depth {depth} stage {stage}"
    assert c.W == side and g.info.exact_dt_path == 1
    check_map(g, c, scene, stage, what=what)
    if stage != 0:
        return
    tmpls = map_templates(side, seed=side + 1)
    raw = check_search(g, c, tmpls, scene, 3, 4, batches=(10, 0), what=what)
    assert not (raw["tmpl_idx"] == len(tmpls) - 1).any(), "a template larger than the map has no valid pose"
    check_minmax_and_optimize(g, c, tmpls, what)


# ---- 2. degenerate extents ------------------------------------------------------------------------------------------
def degenerate_scene(kind):
    """(scene, padding).  row: every line on one row, whose band is the only one the scene covers; column: every line
    on one column at padding 1, every row covered and an envelope window a few columns wide; point: four copies of one
    point (map side 1); corners: two short lines in opposite corners, the bands in between hold no edge; border: the
    borders of a tall extent at padding 1, edges in the first and last map row and every row covered."""
    rng = np.random.default_rng(17)
    if kind in ("row", "column"):
        a = rng.uniform(0, 400, (2, 8))
        b = np.full((2, 8), 123.25)
        if kind == "row":
            return np.ascontiguousarray(np.stack([a[0], b[0], a[1], b[1]]), F32), 1.3
        return np.ascontiguousarray(np.stack([b[0], a[0], b[1], a[1]]), F32), 1.0
    if kind == "point":
        return np.tile(np.array([[57.3], [-12.6], [57.3], [-12.6]], F32), (1, 4)), 1.3
    if kind == "corners":
        return np.array([[0, 0, 5, 3], [394, 396, 399, 399]], F32).T.copy(), 1.0
    return np.array([[0, 0, 0, 499], [99, 0, 99, 499], [0, 0, 99, 0], [0, 499, 99, 499], [50, 10, 50, 480]], F32).T.copy(), 1.0


DEGENERATE = ["row", "column", "point", "corners", "border"]


@pytest.mark.parametrize("dist", list(DIST))
@pytest.mark.parametrize("depth", [30, 7])
@pytest.mark.parametrize("kind", DEGENERATE)
def test_degenerate_extents(kind, depth, dist):
    scene, padding = degenerate_scene(kind)
    if depth == 30 and dist != "L1":   # the intended paths of the geometries, independent of expected_path
        want = {"row": "band_split", "column": "band_fused", "point": "band_fused", "corners": "band_fused", "border": "band_fused"}
        assert expected_path(scene, padding, dist, depth, 0) == want[kind]
    g, c = build_both(scene, depth, padding, dist)
    what = f"{kind} {dist} depth {depth}"
    check_map(g, c, scene, what=what)
    check_search(g, c, map_templates(c.W, seed=c.W), scene, 3, 4, what=what)


# ---- 3. the exact / literal boundary --------------------------------------------------------------------------------
BOUNDARY_CASES = [(s, d) for d in ("L2", "L2_SQUARED") for s in BOUNDARY] + [(2897, "L1"), (2898, "L1")]


@pytest.mark.parametrize("side,dist", BOUNDARY_CASES, ids=[f"{s}-{d}" for s, d in BOUNDARY_CASES])
def test_exact_literal_boundary(side, dist):
    """2*(side-1)^2 < 2^24 up to side 2897: the integer-exact band path there, the literal replay from 2898 on."""
    tmpls = synth_templates(20, 10, side, seed=side)
    scene = plant_instances(pinned_scene(side, 40, seed=side), tmpls, side, side, seed=side + 1)
    g, c = build_both(scene, 30, 1.0, dist)
    assert c.W == side and g.info.exact_dt_path == (1 if side <= 2897 else 0)
    what = f"side {side} {dist}"
    check_map(g, c, scene, what=what)
    raw = check_search(g, c, tmpls, scene, 4, 4, what=what)
    assert len(raw) > 0


# ---- 4. scenes far from the origin ----------------------------------------------------------------------------------
def in_map_translations(c, tmpl, n, seed):
    """Translations (scene coordinates) that keep every end point of `tmpl` at least 2 px inside the map: evaluate_kernel
    clamps lookups outside the map and the oracle does not, so those are left out.  None if the template does not fit."""
    pts = np.asarray(tmpl, F32).T.reshape(-1, 2).astype(np.float64)
    lo = 2.0 - c.shift.astype(np.float64) - pts.min(axis=0)
    hi = np.array([c.W - 3.0, c.H - 3.0]) - c.shift.astype(np.float64) - pts.max(axis=0)
    if (lo > hi).any():
        return None
    rng = np.random.default_rng(seed)
    t = [lo, hi, [lo[0], hi[1]], [hi[0], lo[1]]] + list(rng.uniform(lo, hi, (n, 2)))
    return np.array(t, F32)


FAR_CASES = [(o, s) for o in FAR for s in ("small", "synthetic")]


@pytest.mark.parametrize("dist", list(DIST))
@pytest.mark.parametrize("padding", [1.0, 1.5])
@pytest.mark.parametrize("offset,source", FAR_CASES, ids=[f"{o:g}-{s}" for o, s in FAR_CASES])
def test_far_from_origin(offset, source, padding, dist):
    scene, tmpls = far_scene(offset, source)
    if padding == 1.0:
        assert leaves_map(scene, padding), "the case must exercise the raster kernel's clipping"
    g, c = build_both(scene, 30, padding, dist)
    what = f"offset {offset:g} {source} padding {padding} {dist}"
    check_map(g, c, scene, what=what)
    raw = check_search(g, c, tmpls, scene, 3, 4, what=what)
    assert len(raw) > 0
    # evaluate at translations that keep the templates inside the map
    placed, trans = [], []
    for i, t in enumerate(tmpls):
        tr = in_map_translations(c, t, 12, seed=i)
        if tr is not None:
            placed.append(t)
            trans.append(tr)
    assert placed, "no template fits the map"
    for t, tr, s in zip(placed, trans, fdcm.evaluate(g, placed, trans)):
        assert s.tobytes() == c.evaluate(t, tr).tobytes(), f"{what}: evaluate"
    # distinct top-K and pose refinement against their models
    tset, anchors = fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls)
    s = fdcm.DefaultSearch(3, 4)
    allm = fdcm.search_all(g, tset, scene, s, OPT, PEN)
    sel = fdcm.search_topk(g, tset, scene, s, OPT, PEN, k=10, select=fdcm.DistinctMatches(max_per_template=1, radius=10))
    assert sel.tobytes() == allm[select_model(allm, anchors, 10, 1, 10.0)].tobytes(), f"{what}: distinct top-10"
    base = sel[:4]
    for r in (fdcm.PoseRefinement(), fdcm.PoseRefinement(2, 2, 0.02, 4, 0.5)):
        got = fdcm.refine_matches(g, tset, base, r)
        assert got.tobytes() == refine_reference(g, tmpls, anchors, base, r).tobytes(), f"{what}: {r}"


# ---- 5. rebuilds across sizes on one handle -------------------------------------------------------------------------
def check_step(g, c, scene, tset, tmpls, what):
    planes = range(c.depth) if c.W < 2000 else (0, 7, 14, 22, 29)
    check_map(g, c, scene, planes=planes, what=what)
    top = fdcm.search_topk(g, tset, None, fdcm.DefaultSearch(4, 4), OPT, PEN, k=10)
    assert_matches(top, topk_ref(oracle_penalized(c.search(tmpls, scene, 4, 4, batch=10), tmpls, PEN), 10), f"{what}: top-10")


@pytest.mark.parametrize("dist", list(DIST))
def test_rebuilds_across_sizes(dist):
    """One handle rebuilt 33 -> 2898 -> 300 -> 2897 -> 1 -> empty -> far offset -> 5 -> 2897: grow-only buffers, the
    integral plan and TMA descriptors cached on the geometry, the band / literal workspaces of each path.  Then a
    SceneBatch over tiny, far-offset and 2897-side scenes (its two maps swap sizes)."""
    gd, od = DIST[dist]
    params = fdcm.Dt3CudaParameters(30, 5.0, 1.0, gd)
    far, _ = far_scene(1e5, "small")
    big = pinned_scene(2897, 40, seed=4)
    steps = [pinned_scene(33, 12, 1), pinned_scene(2898, 40, 2), pinned_scene(300, 30, 3), big, pinned_scene(1, 1, 5),
             np.zeros((4, 0), F32), far, pinned_scene(5, 6, 6), big]
    tmpls = synth_templates(12, 8, 300, seed=9)
    tset = fdcm.TemplateSet(tmpls)
    oracles = {}

    def oracle(scene):
        key = scene.tobytes()
        if key not in oracles:
            oracles[key] = orc.Dt3Cpu(scene, 30, 5.0, 1.0, od)
        return oracles[key]

    g = fdcm.build_cuda_featuremap(steps[0], params)
    for i, scene in enumerate(steps):
        if i:
            g.rebuild(scene, wait=i % 2 == 0)
        what = f"{dist} step {i} ({scene.shape[1]} lines)"
        if scene.shape[1] == 0:
            assert g.get_feature_size().tolist() == [0, 0] and g.depth == 0, what
            assert len(fdcm.search_topk(g, tset, None, fdcm.DefaultSearch(4, 4), OPT, PEN, k=10)) == 0, what
            continue
        c = oracle(scene)
        check_step(g, c, scene, tset, tmpls, what)
        if i == 2:
            g.rerun()
            check_step(g, c, scene, tset, tmpls, what + " after rerun")

    synth, _ = far_scene(1e5, "synthetic")
    mix = [steps[7], far, big, steps[0], synth, steps[4], big]
    got = fdcm.SceneBatch(params).search_topk(mix, tset, fdcm.DefaultSearch(4, 4), OPT, PEN, k=10)
    assert len(got) == len(mix)
    for i, scene in enumerate(mix):
        want = topk_ref(oracle_penalized(oracle(scene).search(tmpls, scene, 4, 4, batch=10), tmpls, PEN), 10)
        assert_matches(got[i], want, f"{dist} SceneBatch scene {i}")


# ---- coverage of the build paths ------------------------------------------------------------------------------------
def test_every_build_path_reached():
    """Runs after the cases above (file order): together they must have run every DT path of the build."""
    if not REACHED:
        pytest.skip("no build case of this module ran")
    assert set(PATHS) - REACHED == set(), f"paths never reached: {sorted(set(PATHS) - REACHED)}"
