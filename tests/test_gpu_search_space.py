"""The fused search across the parameters its control flow branches on: BatchOptimize batch size (warp score-cache
span, first window, ballot vs sequential batch path, first-minimum tie rule, partial last batch, empty ranges),
template size (shared-memory staging: 48 KB default, per-block opt-in limit, fewer warps per block), top-k shape
(one or many level-1 blocks, the 592-block clamp, k around n_valid, ties across level-1 chunks), the fused penalty
and its per-TemplateSet denominator cache, and the map depth / propagation coefficient.

Every comparison is bit-exact against the CPU oracle: matches, hypothesis lists and, where the full list is returned,
the evaluation / lookup counters, so that the kernel is shown to score exactly the reference's candidate set.
"""
import numpy as np
import pytest

import openfdcm_b200 as fdcm
from oracle import fdcm_oracle as orc
from tests.helpers import assert_matches, check_full_search, optimizer, oracle_penalized, topk_ref
from tests.util import F32, plant_instances, synth_scene, synth_templates

pytestmark = pytest.mark.gpu

# 0 = DefaultOptimize.  Around 8, 16 and 32: the span / first-window branches of search_warp_kernel; >= 33: a batch never
# fits the 32-lane score cache; 1000 and 100000: the first batch of each direction runs to the map edge.
BATCHES = [0, 1, 2, 4, 7, 8, 9, 15, 16, 17, 31, 32, 33, 48, 64, 1000, 100000]
PENALTIES = [None, fdcm.DefaultPenalty(), fdcm.ExponentialPenalty(0.5), fdcm.ExponentialPenalty(1.5), fdcm.ExponentialPenalty(3.0)]
PENALTY_IDS = ["none", "default", "exp0.5", "exp1.5", "exp3"]


# ---- workloads ------------------------------------------------------------------------------------------------------
def plateau_workload():
    """Long horizontal, vertical and 45-degree lines across the whole 640x480 extent (map 960x960) and templates cut from
    them: walks slide along the lines over plateaus of equal scores and run hundreds of candidates to the map edge.
    DefaultSearch(4, 6) gives 60 hypotheses (identity processing order)."""
    scene = np.array([[0, 100, 639, 100], [0, 300, 639, 300], [200, 0, 200, 479], [0, 0, 479, 479], [0, 0, 1, 0],
                      [638, 479, 639, 479]], F32).T.copy()
    tmpls = [np.array([[-20, 0, 20, 0]], F32).T.copy(),
             np.array([[-20, 0, 20, 0], [-20, 5, 20, 5]], F32).T.copy(),
             np.array([[0, -15, 0, 15], [-10, -10, 10, 10]], F32).T.copy()]
    return scene, tmpls


def random_workload(seed=4100, n_tmpl=128, n_lines=16):
    """Random scene with planted instances; DefaultSearch(4, 4) gives 128 * 32 = 4096 hypotheses, the smallest count
    that takes the spatially ordered processing path."""
    scene = synth_scene(640, 480, 300, seed=seed)
    tmpls = synth_templates(n_tmpl, n_lines, 640, seed=seed + 1)
    return plant_instances(scene, tmpls, 640, 480, seed=seed + 2), tmpls


def tie_templates(n_base, seed):
    """n_base two-line templates followed by byte-identical copies of them: template i and i + n_base score the same on
    every hypothesis and have the same length, so every score of the first half is tied with one in the second half,
    which lies H / 2 hypotheses later (in another level-1 top-k chunk once there are several)."""
    base = synth_templates(n_base, 2, 640, seed=seed)
    return base + [t.copy() for t in base]


@pytest.fixture(scope="module")
def plateau():
    scene, tmpls = plateau_workload()
    return (fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5)), orc.Dt3Cpu(scene, 30, 5.0, 1.5), scene,
            tmpls)


@pytest.fixture(scope="module")
def random_wl():
    scene, tmpls = random_workload()
    return (fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5)), orc.Dt3Cpu(scene, 30, 5.0, 1.5), scene,
            fdcm.TemplateSet(tmpls), tmpls)


# ---- batch size ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("batch", BATCHES)
def test_batch_sweep_plateau(batch, plateau):
    g, c, scene, tmpls = plateau
    _, hyp = check_full_search(g, c, tmpls, scene, 4, 6, batch)
    assert len(hyp) == 60


@pytest.mark.parametrize("batch", BATCHES)
def test_batch_sweep_spatial_order(batch, random_wl):
    g, c, scene, tset, tmpls = random_wl
    _, hyp = check_full_search(g, c, tmpls, scene, 4, 4, batch, tset=tset)
    assert len(hyp) == 4096


def optimize_workload():
    """Scene: pairs of parallel lines 4 px apart (horizontal, vertical, 45 degrees) across the extent.  A template
    segment parallel to a pair and 26 px from it, walked towards it, meets two exact zero scores 4 multipliers apart: a
    batch holding both must return the first one in its evaluation order (upwards: lowest multiplier; downwards:
    highest).  Returns (scene, templates, alignment vectors); the templates that need the map geometry (whole-map
    bounding box, one border) are added by the caller."""
    scene = np.array([[0, 200, 639, 200], [0, 204, 639, 204],          # horizontal pair
                      [300, 0, 300, 479], [304, 0, 304, 479],          # vertical pair
                      [0, 0, 479, 479], [4, 0, 483, 479],              # 45-degree pair
                      [0, 0, 1, 0], [638, 479, 639, 479]], F32).T.copy()
    horiz = np.array([[100, 230, 160, 230]], F32).T.copy()
    horiz2 = np.array([[420, 174, 470, 174], [420, 170, 470, 170]], F32).T.copy()   # above the pair: walks downwards
    vert = np.array([[330, 50, 330, 110]], F32).T.copy()
    vert2 = np.array([[274, 300, 274, 360]], F32).T.copy()                          # left of the pair
    diag = np.array([[150, 124, 190, 164]], F32).T.copy()                           # 26 px right of the 45-degree pair
    cases = []
    for t in (horiz, horiz2):
        cases += [(t, v) for v in ([0, 1], [0, -1], [1, 1], [-1, -1], [1, -1], [1, 0])]
    for t in (vert, vert2):
        cases += [(t, v) for v in ([1, 0], [-1, 0], [1, 1], [-1, 1], [0, 1])]
    cases += [(diag, v) for v in ([1, 0], [-1, 0], [0, 1], [0, -1], [0.3, -1], [-1, 0.45])]
    return scene, cases


@pytest.fixture(scope="module")
def optimize_wl():
    scene, cases = optimize_workload()
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    c = orc.Dt3Cpu(scene, 30, 5.0, 1.5)
    # map corners in scene coordinates: map pixel (x, y) holds scene point (x, y) - shift
    x0, y0 = (np.zeros(2, F32) - c.shift).astype(F32)
    x1, y1 = (np.array([c.W - 1, c.H - 1], F32) - c.shift).astype(F32)
    full = np.array([[x0, y0, x1, y1], [x0, y1, x1, y0]], F32).T.copy()            # bounding box = the whole map
    left = np.array([[x0, 150, x0 + 40, 150], [x0 + 10, 140, x0 + 10, 175]], F32).T.copy()   # touches the left border
    top = np.array([[250, y0, 290, y0 + 30]], F32).T.copy()                                # touches the top border
    for v in ([1, 0], [0, 1], [1, 1], [-1, 0]):
        lo, hi = c.minmax_translation(full, v)
        assert int(lo) == 0 and int(hi) == 0, "the whole-map template must have an empty multiplier range"
    cases = cases + [(full, v) for v in ([1, 0], [0, 1], [1, 1], [-1, 0])]
    cases += [(left, v) for v in ([1, 0], [-1, 0], [1, 1], [0, -1])]
    cases += [(top, v) for v in ([0, 1], [0, -1], [1, 1])]
    lo, hi = c.minmax_translation(left, [1, 0])
    assert int(lo) == 0 and int(hi) > 0, "the border template must have one empty direction"
    return g, c, cases


@pytest.mark.parametrize("batch", BATCHES)
def test_optimize_entry_point_batch_sweep(batch, optimize_wl):
    g, c, cases = optimize_wl
    got = fdcm.optimize(optimizer(batch), [t for t, _ in cases], [np.array(v, F32) for _, v in cases], g)
    for i, ((t, v), r) in enumerate(zip(cases, got)):
        has, score, tr = c.optimize_one(t, np.array(v, F32), batch)
        assert (r is not None) == has, f"case {i} (align {v})"
        if has:
            assert r[0] == score and np.array_equal(r[1], tr), f"case {i} (align {v}): {r} != {(score, tr)}"


# ---- template size ------------------------------------------------------------------------------------------------
# 4 warps x (16 L + round16(L)) bytes of dynamic shared memory per block: 722 lines = 48 KB exactly, 3418 = 227 KB exactly
# (the B200's per-block opt-in limit); 3419 and 4000 need fewer warps per block.
SIZES = [1, 2, 3, 4, 5, 7, 8, 9, 15, 16, 17, 31, 32, 33, 63, 64, 65, 722, 723, 1500, 3418, 3419, 4000]


@pytest.fixture(scope="module")
def size_wl():
    scene = synth_scene(640, 480, 300, seed=4200)
    small = synth_templates(6, 12, 640, seed=4201)
    scene = plant_instances(scene, small, 640, 480, seed=4202)
    big = {L: synth_templates(1, L, 640, seed=L)[0] for L in SIZES}
    return (fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5)), orc.Dt3Cpu(scene, 30, 5.0, 1.5), scene,
            big)


@pytest.mark.parametrize("longest", [65, 722, 723, 3418, 3419, 4000])
def test_template_sizes(longest, size_wl):
    """Every size up to `longest` in one template set (the longest sets the shared-memory footprint), through the search
    with BatchOptimize(10) and DefaultOptimize and through optimize()."""
    g, c, scene, big = size_wl
    tmpls = [big[L] for L in SIZES if L <= longest]
    for batch in (10, 0):
        check_full_search(g, c, tmpls, scene, 4, 4, batch)
        rng = np.random.default_rng(longest + batch)
        placed = [(t.T.reshape(-1, 2) + np.array([320, 240], F32)).reshape(-1, 4).T.astype(F32) for t in tmpls]
        aligns = [rng.standard_normal(2).astype(F32) for _ in placed]
        got = fdcm.optimize(optimizer(batch), placed, aligns, g)
        for i, (t, a, r) in enumerate(zip(placed, aligns, got)):
            has, score, tr = c.optimize_one(t, a, batch)
            assert (r is not None) == has, f"template of {t.shape[1]} lines"
            if has:
                assert r[0] == score and np.array_equal(r[1], tr), f"template of {t.shape[1]} lines"


def test_ordinary_templates_next_to_a_long_one(size_wl):
    """200 ordinary templates and one of 4000 lines (6432 hypotheses, spatially ordered path): the long template changes
    the launch shape of the whole set, the ordinary ones must still be found as the reference finds them."""
    g, c, scene, big = size_wl
    tmpls = synth_templates(200, 20, 640, seed=4203)
    tmpls.insert(117, big[4000])
    raw, _ = check_full_search(g, c, tmpls, scene, 4, 4, 10)
    assert (raw["tmpl_idx"] != 117).sum() > 0


def _one_warp_line_limit():
    """Longest template one warp of the search kernel can stage: 16 L + round16(L) bytes within the device's per-block
    opt-in shared memory."""
    import torch
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    fits = lambda L: 16 * L + (L + 15) // 16 * 16 <= optin
    L = optin // 17
    while fits(L + 1):
        L += 1
    while not fits(L):
        L -= 1
    return L


def test_template_over_the_shared_memory_limit_is_rejected(size_wl):
    g, c, scene, big = size_wl
    limit = _one_warp_line_limit()
    too_long = synth_templates(1, limit + 1, 640, seed=4204)[0]
    ordinary = synth_templates(10, 20, 640, seed=4205)
    tset = fdcm.TemplateSet(ordinary + [too_long])
    for call in (lambda: fdcm.search_all(g, tset, scene, fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10)),
                 lambda: fdcm.search_topk(g, tset, None, fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), k=10),
                 lambda: fdcm.optimize(fdcm.BatchOptimize(10), [too_long], [np.array([1, 0], F32)], g),
                 lambda: fdcm.SceneBatch(fdcm.Dt3CudaParameters(30, 5.0, 1.5)).search_topk([scene], tset, fdcm.DefaultSearch(4, 4),
                                                                                          fdcm.BatchOptimize(10), k=10)):
        with pytest.raises(fdcm.FdcmError) as e:
            call()
        assert e.value.status == fdcm._lib.FDCM_ERR_INVALID and str(limit) in str(e.value), str(e.value)
    # the map, the template upload path and the search workspace are still usable
    check_full_search(g, c, ordinary, scene, 4, 4, 10)
    check_full_search(g, c, ordinary + [big[4000]], scene, 4, 4, 10)


# ---- top-k --------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def topk_wl():
    scene = synth_scene(640, 480, 300, seed=3)
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    c = orc.Dt3Cpu(scene, 30, 5.0, 1.5)
    sets = {}
    # (templates, max scene lines): 60 * 32 = 1920 hypotheses (one level-1 block), 156 * 32 = 4992 (three blocks),
    # 19000 * 64 = 1 216 000 (more than 592 * 2048: the block count is clamped and every block scans a longer chunk)
    for name, n_base, max_s in (("one_block", 30, 8), ("three_blocks", 78, 8), ("clamped", 9500, 16)):
        tmpls = tie_templates(n_base, seed=n_base)
        raw = c.search(tmpls, scene, 2, max_s, batch=10)
        sets[name] = (fdcm.TemplateSet(tmpls), tmpls, max_s, raw)
    return g, c, scene, sets


def _check_topk(g, tset, tmpls, scene, max_s, raw, penalty, ks, base):
    pen = oracle_penalized(raw, tmpls, penalty)
    for k in ks:
        got = fdcm.search_topk(g, tset, scene, fdcm.DefaultSearch(2, max_s), fdcm.BatchOptimize(10), penalty, k=k, tmpl_idx_base=base)
        assert_matches(got, topk_ref(pen, k, base), f"k={k}")


@pytest.mark.parametrize("penalty", PENALTIES, ids=PENALTY_IDS)
@pytest.mark.parametrize("size", ["one_block", "three_blocks"])
def test_topk_shapes(size, penalty, topk_wl):
    g, c, scene, sets = topk_wl
    tset, tmpls, max_s, raw = sets[size]
    H = len(tmpls) * 2 * max_s * 2
    n_valid = len(raw)
    pen = oracle_penalized(raw, tmpls, penalty)
    assert len(np.unique(pen["score"])) <= n_valid // 2, "the workload must be full of exact ties"
    ks = [1, 2, 31, 32, 33, 1023, 1024, 1025, n_valid - 1, n_valid, n_valid + 1, H + 7]
    _check_topk(g, tset, tmpls, scene, max_s, raw, penalty, ks, base=1000)
    assert g.last_search_stats()["n_hypotheses"] == H


@pytest.mark.parametrize("penalty", PENALTIES, ids=PENALTY_IDS)
def test_topk_clamped_block_count(penalty, topk_wl):
    """k up to 1025 on 1.2 M hypotheses.  (k near n_valid is not run here: the single-block level-2 merge is O(k * 592 * k)
    and its workspace 592 * k records, which is not what the top-k path is for.)"""
    g, c, scene, sets = topk_wl
    tset, tmpls, max_s, raw = sets["clamped"]
    _check_topk(g, tset, tmpls, scene, max_s, raw, penalty, [1, 2, 31, 32, 33, 1023, 1024, 1025], base=7)
    assert g.last_search_stats()["n_hypotheses"] == 1216000 > 592 * 2048


def test_penalty_switches_on_one_template_set(random_wl):
    """The denominators are cached per TemplateSet on (kind, tau): every switch must take effect, in both directions."""
    g, c, scene, tset, tmpls = random_wl
    raw = c.search(tmpls, scene, 4, 4, batch=10)
    for penalty in (None, fdcm.ExponentialPenalty(1.5), fdcm.DefaultPenalty(), fdcm.ExponentialPenalty(1.5), fdcm.ExponentialPenalty(2.0),
                    None, fdcm.DefaultPenalty()):
        what = "none" if penalty is None else f"{type(penalty).__name__}({penalty.tau})"
        got = fdcm.search_all(g, tset, scene, fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), penalty)
        assert_matches(got, oracle_penalized(raw, tmpls, penalty), what)
        top = fdcm.search_topk(g, tset, scene, fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), penalty, k=10)
        assert_matches(top, topk_ref(oracle_penalized(raw, tmpls, penalty), 10), what)


# ---- depth and propagation coefficient ------------------------------------------------------------------------------
@pytest.mark.parametrize("coeff", [0.0, 50.0])
@pytest.mark.parametrize("depth", [2, 33, 64])
def test_depth_and_coeff_through_search(depth, coeff):
    scene = synth_scene(320, 240, 80, seed=4300 + depth)
    tmpls = synth_templates(20, 15, 320, seed=4301)
    scene = plant_instances(scene, tmpls, 320, 240, seed=4302)
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(depth, coeff, 1.5))
    c = orc.Dt3Cpu(scene, depth, coeff, 1.5)
    assert g.depth == c.depth == depth
    for d in range(depth):
        assert np.array_equal(g.plane(d), c.plane(d)), f"plane {d}"
    raw, _ = check_full_search(g, c, tmpls, scene, 4, 4, 10)
    top = fdcm.search_topk(g, tmpls, scene, fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), fdcm.ExponentialPenalty(1.5), k=10)
    assert_matches(top, topk_ref(oracle_penalized(raw, tmpls, fdcm.ExponentialPenalty(1.5)), 10))
