"""GPU parity tests: the CUDA path (through the C ABI of libfdcm_b200.so) against the CPU oracle on the
same seeded inputs, stage by stage (SURVEY.md §4.4).  Bars (BASELINE.json north_star): edge masks,
orientation bins and hypothesis sets bit-exact; DT3 values within 1e-5 relative; scores within 1e-4
relative; identical top-10.  In practice every stage is bit-exact and the tests assert that first,
falling back to the stated tolerance only in the message.
"""
import numpy as np
import pytest

import openfdcm_b200 as fdcm
from oracle import fdcm_oracle as orc
from tests.util import F32, load_kats, plant_instances, synth_scene, synth_templates

pytestmark = pytest.mark.gpu
DIST = {"L2": (fdcm.distance.L2, orc.L2), "L2_SQUARED": (fdcm.distance.L2_SQUARED, orc.L2_SQUARED),
        "L1": (fdcm.distance.L1, orc.L1)}
KATS = load_kats()


def _assert_planes(gpu_map, cpu_map, what, rtol=1e-5):
    assert (gpu_map.width, gpu_map.height, gpu_map.depth) == (cpu_map.W, cpu_map.H, cpu_map.depth)
    assert np.array_equal(gpu_map.angles(), cpu_map.keys)
    for d in range(cpu_map.depth):
        g, c = gpu_map.plane(d), cpu_map.plane(d)
        if not np.array_equal(g, c):
            bad = ~np.isclose(g, c, rtol=rtol, atol=0)
            assert not bad.any(), f"{what}: plane {d}: {bad.sum()} values beyond rtol={rtol}, max abs diff {np.abs(g - c).max()}"
            pytest.fail(f"{what}: plane {d} within tolerance but not bit-exact ({(g != c).sum()} values differ)")


@pytest.mark.parametrize("dist", ["L2", "L2_SQUARED", "L1"])
@pytest.mark.parametrize("stage", [1, 2, 0], ids=["dt", "propagated", "integral"])
def test_build_stages_small(dist, stage):
    scene = synth_scene(320, 240, 60, seed=11)
    gd, od = DIST[dist]
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5, gd), stage=stage)
    c = orc.Dt3Cpu(scene, 30, 5.0, 1.5, od, stage=stage)
    assert g.info.exact_dt_path == 1
    assert np.allclose(g.get_scene_translation(), c.shift, rtol=0, atol=0)
    _assert_planes(g, c, f"{dist} stage {stage}")


@pytest.mark.parametrize("geom", [(320, 240, 1.5), (333, 517, 1.0), (1201, 130, 1.2)], ids=lambda g: f"{g[0]}x{g[1]}")
def test_line_integral_geometries(geom):
    """lineIntegral against the oracle on map sides that are / are not multiples of 4 and 32: strips that leave the image
    on either side, tile ranges clipped to the image."""
    w, h, pad = geom
    scene = synth_scene(w, h, 80, seed=w + h)
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, pad, fdcm.distance.L2))
    c = orc.Dt3Cpu(scene, 30, 5.0, pad, orc.L2)
    _assert_planes(g, c, f"integral {w}x{h}")


def test_fast_sqrt_is_exact():
    """The fused fill's rsqrt + Newton square root equals the IEEE sqrtf on every input it can see: all integers
    0 .. 2^24 (squared distances of the exact regime) and FLT_MAX (planes without edges)."""
    import ctypes as C
    from openfdcm_b200._lib import check, lib
    bad, first = C.c_int64(-1), C.c_uint32(0)
    check(lib().fdcm_debug_sqrt_check(0, C.byref(bad), C.byref(first)))
    assert bad.value == 0, f"{bad.value} mismatches, first at input {first.value}"


def test_edge_masks_and_bins_bit_exact():
    scene = synth_scene(640, 480, 300, seed=1000)
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5, fdcm.distance.L2_SQUARED), stage=1)
    c = orc.Dt3Cpu(scene, 30, 5.0, 1.5, orc.L2_SQUARED, stage=1)
    shifted = (scene.T.reshape(-1, 2) + c.shift).reshape(-1, 4).T.astype(F32)
    bins = np.array([orc.closest_orientation(c.keys, shifted[:, i]) for i in range(shifted.shape[1])])
    assert np.array_equal(g.scene_bins(), bins)
    for d in range(c.depth):
        assert np.array_equal(g.mask(d), (c.plane(d) == 0).astype(np.uint8)), f"edge mask of plane {d}"


@pytest.mark.parametrize("depth", [1, 4, 7, 30, 64])   # 64: the largest depth, fills the propagation tables exactly
def test_other_depths(depth):
    scene = synth_scene(200, 150, 40, seed=5)
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(depth, 3.0, 2.2, fdcm.distance.L2))
    c = orc.Dt3Cpu(scene, depth, 3.0, 2.2, orc.L2)
    _assert_planes(g, c, f"depth {depth}")


@pytest.mark.parametrize("dist", ["L2", "L1"])
def test_general_path_large_side(dist):
    """side > 2897: float(q^2) is inexact, the literal (non integer-exact) DT path must be taken."""
    scene = synth_scene(2000, 1500, 120, seed=21)
    gd, od = DIST[dist]
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(3, 5.0, 1.5, gd))
    c = orc.Dt3Cpu(scene, 3, 5.0, 1.5, od)
    assert g.width == 3000 and g.info.exact_dt_path == 0
    _assert_planes(g, c, f"general path {dist}")


@pytest.mark.parametrize("case", KATS["dt3_golden_rows"], ids=lambda c: c["cite"])
def test_reference_golden_rows_on_gpu(case):
    scene = np.array(case["scene"], F32)
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(case["depth"], case["coeff"], case["padding"]))
    f = g.plane(int(g.classify(scene)[0]))
    assert np.allclose(f[int(f.shape[0] / 2)], np.array(case["middle_row"], F32), rtol=0, atol=1e-5)


def test_empty_scene():
    g = fdcm.build_cuda_featuremap(np.zeros((4, 0), F32), fdcm.Dt3CudaParameters())
    assert g.get_feature_size().tolist() == [0, 0] and g.depth == 0
    assert fdcm.search(fdcm.DefaultMatch(), fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), g,
                       [synth_templates(1, 5, 100, 1)[0]], np.zeros((4, 0), F32)) == []


def test_classify_matches_host_atanf():
    rng = np.random.default_rng(3)
    scene = synth_scene(100, 100, 10, seed=2)
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    n = 20000
    ang = rng.uniform(-np.pi, np.pi, n)
    ln = rng.uniform(0.5, 200, n)
    p1 = rng.uniform(-500, 500, (2, n))
    lines = np.vstack([p1, p1 + ln * np.vstack([np.cos(ang), np.sin(ang)])]).astype(F32)
    lines[:, :200] = np.round(lines[:, :200])          # axis-aligned / degenerate slopes
    lines[2, 200:230] = lines[0, 200:230]              # vertical: dx == 0
    lines[2:, 230:240] = lines[:2, 230:240]            # null lines: 0/0
    keys = g.angles()
    want = np.array([orc.closest_orientation(keys, lines[:, i]) for i in range(n)])
    assert np.array_equal(g.classify(lines), want)


def _workload(seed, width=640, height=480, n_scene=300, n_tmpl=20, n_lines=30):
    scene = synth_scene(width, height, n_scene, seed=seed)
    tmpls = synth_templates(n_tmpl, n_lines, width, seed=seed + 1)
    scene = plant_instances(scene, tmpls, width, height, seed=seed + 2)
    return scene, tmpls


def test_evaluate_and_minmax():
    scene, tmpls = _workload(31, n_tmpl=6)
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    c = orc.Dt3Cpu(scene, 30, 5.0, 1.5)
    rng = np.random.default_rng(9)
    placed, trans = [], []
    for t in tmpls:
        placed.append((t.T.reshape(-1, 2) + np.array([320, 240], F32)).reshape(-1, 4).T.astype(F32))
        trans.append(rng.uniform(-40, 40, (17, 2)).astype(F32))
    got = fdcm.evaluate(g, placed, trans)
    for t, tr, s in zip(placed, trans, got):
        assert np.array_equal(s, c.evaluate(t, tr))
        for v in ([1, 0], [0.3, -1], [-1, 0.5], [0, 0], [0, 1]):
            a, b = fdcm.minmax_translation(g, t, v), c.minmax_translation(t, v)
            assert np.array_equal(a, b, equal_nan=True)


@pytest.mark.parametrize("batch", [10, 1, 0], ids=["BatchOptimize(10)", "BatchOptimize(1)", "DefaultOptimize"])
def test_search_full_list_config1(batch):
    """BASELINE config 1 (README example shape): every match compared, in hypothesis order."""
    scene, tmpls = _workload(1000)
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    c = orc.Dt3Cpu(scene, 30, 5.0, 1.5)
    opt = fdcm.BatchOptimize(batch) if batch else fdcm.DefaultOptimize()
    got = fdcm.search_all(g, tmpls, scene, fdcm.DefaultSearch(4, 4), opt)
    orc.stats_reset()
    want, hyp = c.search(tmpls, scene, 4, 4, batch=batch, want_hyp=True)
    evals, lookups = orc.stats_get()
    assert np.array_equal(g.last_hypotheses(), hyp), "hypothesis set must be bit-exact"
    st = g.last_search_stats()
    assert st["n_hypotheses"] == len(hyp) == 20 * 4 * 4 * 2
    assert (st["n_evaluations"], st["n_lookups"]) == (evals, lookups)
    assert len(got) == len(want) == st["n_valid"]
    assert np.array_equal(got["tmpl_idx"], want["tmpl_idx"])
    assert np.allclose(got["score"], want["score"], rtol=1e-4, atol=0)
    assert np.array_equal(got["transform"], want["transform"])
    assert np.array_equal(got["score"], want["score"]), "scores within 1e-4 but not bit-exact"


@pytest.mark.parametrize("max_t", [1, 2, 3, 4, 6, 9])
def test_host_template_order_with_tied_lengths(max_t):
    """fdcm_search_host only orders the max_tmpl_lines longest lines of a template (selection scan) and falls back to the
    reference's std::sort when the leading lengths tie: templates full of equal-length lines (rectangles, repeated
    segments, integer coordinates) must give the oracle's hypothesis list and matches for every max_tmpl_lines."""
    rng = np.random.default_rng(77)
    scene = synth_scene(640, 480, 200, seed=5)
    tmpls = []
    for k in range(40):
        w, h = int(rng.integers(10, 60)), int(rng.integers(10, 60))
        rect = np.array([[0, 0, w, 0], [w, 0, w, h], [w, h, 0, h], [0, h, 0, 0]], F32).T            # two pairs of equal lengths
        extra = rng.integers(-40, 40, (4, int(rng.integers(0, 12)))).astype(F32)                    # integer end points: more ties
        dup = rect[:, : int(rng.integers(0, 3))] + np.array([[3], [7], [3], [7]], F32)              # shifted copies: exact duplicates of lengths
        t = np.concatenate([rect, extra, dup], axis=1)
        tmpls.append(np.ascontiguousarray(t[:, rng.permutation(t.shape[1])], F32))
    tmpls += synth_templates(10, 20, 640, seed=9)                                                   # and ordinary ones (selection path)
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    c = orc.Dt3Cpu(scene, 30, 5.0, 1.5)
    import ctypes as C
    from openfdcm_b200 import _lib
    flat, off = fdcm._pack(tmpls)
    sc = fdcm._records(scene)
    p = _lib.SearchParams(max_t, 3, 10, 0, 0.0, 0, 0, 0, 0.0, 0.0, 0.0, 0.0)
    out = np.zeros(2 * len(tmpls) * max_t * 3, fdcm.MATCH_DTYPE)
    n = C.c_int64(0)
    fdcm.check(_lib.lib().fdcm_search_host(g._h, fdcm.ptr(flat), fdcm.ptr(off), len(tmpls), fdcm.ptr(sc), sc.shape[0], C.byref(p),
                                           fdcm.ptr(out), out.shape[0], C.byref(n)))
    got = out[: n.value]
    want, hyp = c.search(tmpls, scene, max_t, 3, batch=10, want_hyp=True)
    assert np.array_equal(g.last_hypotheses(), hyp), "hypothesis set must be bit-exact"
    assert np.array_equal(got["tmpl_idx"], want["tmpl_idx"])
    assert np.array_equal(got["score"], want["score"], equal_nan=True)
    assert np.array_equal(got["transform"], want["transform"], equal_nan=True)


@pytest.mark.parametrize("dist", ["L2", "L2_SQUARED", "L1"])
def test_search_top10(dist):
    scene, tmpls = _workload(77, n_tmpl=40, n_lines=25)
    gd, od = DIST[dist]
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5, gd))
    c = orc.Dt3Cpu(scene, 30, 5.0, 1.5, od)
    got = fdcm.search_topk(g, tmpls, scene, fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), fdcm.ExponentialPenalty(1.5), k=10)
    raw = c.search(tmpls, scene, 4, 4, batch=10)
    pen = orc.penalize(1, 1.5, raw, orc.template_lengths(tmpls))
    order = np.lexsort((np.arange(len(pen)), pen["score"]))[:10]   # ascending score, ties by hypothesis order
    want = pen[order]
    assert len(got) == 10
    assert np.array_equal(got["tmpl_idx"], want["tmpl_idx"])
    assert np.array_equal(got["transform"], want["transform"])
    assert np.allclose(got["score"], want["score"], rtol=1e-4, atol=0)
    assert np.array_equal(got["score"], want["score"])


def test_reference_api_roundtrip():
    """The reference README flow with the CUDA types (README.md:46-82)."""
    scene, tmpls = _workload(5, n_tmpl=8)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(depth=30, dt3Coeff=5.0, padding=1.5), fdcm.ThreadPool(4))
    matches = fdcm.search(fdcm.DefaultMatch(), fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10, fdcm.ThreadPool(4)), fm, tmpls, scene)
    pen = fdcm.penalize(fdcm.ExponentialPenalty(tau=1.5), matches, fdcm.get_template_lengths(tmpls))
    srt = fdcm.sort_matches(pen)
    assert len(srt) == len(matches) > 0
    assert all(srt[i].score <= srt[i + 1].score for i in range(len(srt) - 1))
    c = orc.Dt3Cpu(scene, 30, 5.0, 1.5)
    raw = c.search(tmpls, scene, 4, 4, batch=10)
    want = orc.sort_matches(orc.penalize(1, 1.5, raw, orc.template_lengths(tmpls)))
    assert np.array_equal(np.array([m.score for m in srt], F32), want["score"])
    assert np.allclose(fdcm.get_template_lengths(tmpls), orc.template_lengths(tmpls), rtol=0, atol=0)
    with pytest.raises(IndexError):
        fdcm.penalize(fdcm.DefaultPenalty(), matches, [])


def test_search_edge_cases():
    scene, tmpls = _workload(8, n_tmpl=3)
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    c = orc.Dt3Cpu(scene, 30, 5.0, 1.5)
    s, o = fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10)
    assert fdcm.search(fdcm.DefaultMatch(), s, o, g, [], scene) == []
    assert fdcm.search(fdcm.DefaultMatch(), s, o, g, [np.zeros((4, 0), F32)], scene) == []
    # ragged: an empty template between real ones, a 2-line template (fewer lines than max_tmpl_lines),
    # a template far outside the map (all hypotheses nullopt) and a degenerate (zero-length) line
    ragged = [tmpls[0], np.zeros((4, 0), F32), tmpls[1][:, :2], (tmpls[2] * 50).astype(F32),
              np.array([[1, 5], [1, 5], [1, 9], [1, 5]], F32)]
    got = fdcm.search_all(g, ragged, scene, fdcm.DefaultSearch(4, 6), o)
    want, hyp = c.search(ragged, scene, 4, 6, batch=10, want_hyp=True)
    assert np.array_equal(g.last_hypotheses(), hyp)
    assert np.array_equal(got["tmpl_idx"], want["tmpl_idx"])
    assert np.array_equal(got["score"], want["score"], equal_nan=True)
    assert np.array_equal(got["transform"], want["transform"], equal_nan=True)
    # more scene slots than scene lines
    tiny_scene = scene[:, :3]
    g2 = fdcm.build_cuda_featuremap(tiny_scene, fdcm.Dt3CudaParameters(30, 5.0, 2.2))
    c2 = orc.Dt3Cpu(tiny_scene, 30, 5.0, 2.2)
    got = fdcm.search_all(g2, tmpls, tiny_scene, fdcm.DefaultSearch(4, 10), o)
    want = c2.search(tmpls, tiny_scene, 4, 10, batch=10)
    assert np.array_equal(got["score"], want["score"]) and np.array_equal(got["transform"], want["transform"])


def _dt_rows(g, literal):
    import ctypes as C
    from openfdcm_b200 import _lib
    g = np.ascontiguousarray(g, np.uint16)
    out = np.zeros(g.shape, np.float32)
    _lib.check(_lib.lib().fdcm_debug_dt_rows(_lib.ptr(g), g.shape[0], g.shape[1], int(literal), 0, _lib.ptr(out)))
    return out


@pytest.mark.parametrize("n", [1, 2, 31, 32, 33, 64, 100, 1024, 2048, 2880, 2897])
def test_row_pass_exact_kernel_vs_literal_oracle(n):
    """The exact-regime warp kernel (leftmost-argmin owners + in-place chain) against the literal
    imgproc.h:91-130 restatement on adversarial rows: many ties, plateaus, steep ramps, sparse columns."""
    rng = np.random.default_rng(n)
    rows = []
    big = 0xFFFF
    rows.append(np.zeros(n))                                   # all edges
    rows.append(np.full(n, big))                               # no edge at all
    rows.append(np.where(np.arange(n) == n // 2, 0, big))      # a single finite column
    rows.append(np.arange(n) % 7)                              # periodic ties
    rows.append(np.abs(np.arange(n) - n // 3))                 # 45-degree ramp: three-way ties everywhere
    rows.append(np.minimum(np.arange(n) * 3, 2000))            # steep ramp (deep aliasing chains)
    rows.append(np.minimum((np.arange(n)[::-1]) // 2, 2500))   # shallow ramp from the right
    # finite columns on one side of the split of the two-stack envelope only, and a dense block around it
    rows.append(np.where(np.arange(n) < max(1, n // 4), rng.integers(0, 60, n), big))
    rows.append(np.where(np.arange(n) >= n - max(1, n // 4), rng.integers(0, 60, n), big))
    rows.append(np.where(np.abs(np.arange(n) - n // 2) < 40, rng.integers(0, 9, n), big))
    rows.append(np.where(np.arange(n) % 2 == 0, 700 - np.arange(n) % 700, big))      # long pops across the split
    for k in range(40):
        r = rng.integers(0, [3, 10, 50, 400, 2800][k % 5], n)
        if k % 3 == 0:
            r = np.where(rng.random(n) < 0.7, big, r)           # sparse finite columns
        if k % 4 == 1:
            r = np.repeat(r[:: 8], 8)[:n] if n >= 8 else r      # plateaus
        rows.append(r)
    g = np.stack([np.asarray(r).astype(np.int64)[:n] for r in rows]).astype(np.uint16)
    lit = _dt_rows(g, literal=1)
    band = _dt_rows(g, literal=2)   # lane-per-row band kernel (the product path), g given explicitly
    fmax = np.finfo(np.float32).max
    for i in range(g.shape[0]):
        f = np.where(g[i] == big, fmax, g[i].astype(np.float64) ** 2).astype(F32)
        want = orc.dt_pass_l2_1d(f)
        assert np.array_equal(lit[i], want), f"literal kernel row {i}"
        assert np.array_equal(band[i], want), f"band kernel row {i}: first diff at {np.flatnonzero(band[i] != want)[:5]}"


@pytest.mark.parametrize("batch", [10, 0], ids=["BatchOptimize(10)", "DefaultOptimize"])
@pytest.mark.parametrize("case", KATS["batch_optimize"], ids=lambda c: c["cite"][:30])
def test_reference_optimize_kats_on_gpu(case, batch):
    """batchoptimize.test.cpp:35-117 / defaultoptimize.test.cpp through the CUDA OptimizeStrategy entry point."""
    tmpl = np.array(case["tmpl"], F32)
    if case["pre_transform"] is not None:
        tmpl = orc.transform(tmpl, case["pre_transform"])
    fm = fdcm.build_cuda_featuremap(np.array(case["scene"], F32), fdcm.Dt3CudaParameters(case["depth"], case["coeff"], case["padding"]))
    opt = fdcm.BatchOptimize(batch) if batch else fdcm.DefaultOptimize()
    res = fdcm.optimize(opt, [tmpl], [case["align_vec"]], fm)[0]
    assert (res is not None) == case["has_value"]
    if res is None:
        return
    score, tr = res
    assert np.allclose(tr, case["translation"], rtol=0, atol=1e-5)
    if "score_exact" in case:
        assert score == case["score_exact"]
    else:
        assert abs(score - case["score_rel"]) <= 1.2e-5 * abs(case["score_rel"])


def test_optimize_entry_point_matches_oracle():
    scene, tmpls = _workload(91, n_tmpl=12, n_lines=27)
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    c = orc.Dt3Cpu(scene, 30, 5.0, 1.5)
    rng = np.random.default_rng(4)
    placed = [(t.T.reshape(-1, 2) + rng.uniform([200, 150], [440, 330]).astype(F32)).reshape(-1, 4).T.astype(F32) for t in tmpls]
    placed.append((tmpls[0] * 100).astype(F32))                      # out of the map -> nullopt
    aligns = [rng.standard_normal(2).astype(F32) for _ in placed]
    aligns[3] = np.zeros(2, F32)                                     # null alignment vector -> nullopt
    aligns[4] = np.array([0, 1], F32)
    aligns[5] = np.array([-1, 0], F32)
    for batch in (10, 3, 0):
        opt = fdcm.BatchOptimize(batch) if batch else fdcm.DefaultOptimize()
        got = fdcm.optimize(opt, placed, aligns, g)
        for t, a, r in zip(placed, aligns, got):
            has, score, tr = c.optimize_one(t, a, batch)
            assert (r is not None) == has
            if has:
                assert r[0] == score and np.array_equal(r[1], tr)


def test_cpp_host_mirror_pipeline():
    """examples/cpp_pipeline.cpp: README flow through include/openfdcm_b200/openfdcm_cuda.hpp."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "examples", "cpp_pipeline")
    if not os.path.exists(exe):
        subprocess.check_call(["g++", "-std=c++17", "-I" + os.path.join(root, "include"), os.path.join(root, "examples", "cpp_pipeline.cpp"),
                               "-L" + os.path.join(root, "openfdcm_b200"), "-lfdcm_b200", "-Wl,-rpath,$ORIGIN/../openfdcm_b200", "-o", exe])
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "matches; best" in r.stdout


def test_search_spatially_ordered_path():
    """>= 4096 hypotheses: the kernel walks the hypotheses in the spatial order of their scene lines; the match list
    must still come back in hypothesis order, bit-identical to the oracle."""
    scene, tmpls = _workload(123, n_tmpl=150, n_lines=20)
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    c = orc.Dt3Cpu(scene, 30, 5.0, 1.5)
    got = fdcm.search_all(g, tmpls, scene, fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), fdcm.ExponentialPenalty(1.5))
    raw, hyp = c.search(tmpls, scene, 4, 4, batch=10, want_hyp=True)
    want = orc.penalize(1, 1.5, raw, orc.template_lengths(tmpls))
    assert len(hyp) == 150 * 32 and np.array_equal(g.last_hypotheses(), hyp)
    assert np.array_equal(got["tmpl_idx"], want["tmpl_idx"])
    assert np.array_equal(got["score"], want["score"]) and np.array_equal(got["transform"], want["transform"])
    top = fdcm.search_topk(g, tmpls, scene, fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), fdcm.ExponentialPenalty(1.5), k=10)
    assert np.array_equal(top, want[np.lexsort((np.arange(len(want)), want["score"]))[:10]])


def test_config4_shape_wide_search_4k_scene():
    """BASELINE config 4 shape (scaled in template count only): 4K scene, 5000 lines, 60-line templates,
    DefaultSearch(16,16), BatchOptimize(20).  Side 5760 > 2897 -> literal DT path; 3.98 GB map."""
    scene = synth_scene(3840, 2160, 5000, seed=4000)
    tmpls = synth_templates(6, 60, 3840, seed=4001)
    scene = plant_instances(scene, tmpls, 3840, 2160, seed=4002)
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    assert g.width == 5760 and g.info.exact_dt_path == 0
    c = orc.Dt3Cpu(scene, 30, 5.0, 1.5)
    for d in (0, 4, 11, 15, 22, 29):
        assert np.array_equal(g.plane(d), c.plane(d)), f"plane {d}"
    got = fdcm.search_all(g, tmpls, scene, fdcm.DefaultSearch(16, 16), fdcm.BatchOptimize(20))
    want, hyp = c.search(tmpls, scene, 16, 16, batch=20, want_hyp=True)
    assert len(hyp) == 6 * 16 * 16 * 2 and np.array_equal(g.last_hypotheses(), hyp)
    assert np.array_equal(got["tmpl_idx"], want["tmpl_idx"])
    assert np.array_equal(got["score"], want["score"]) and np.array_equal(got["transform"], want["transform"])


def test_config5_shape_multiview_batch():
    """BASELINE config 5 shape (scaled): several scenes, one resident template set, per-scene rebuild of the same map
    object + top-10; scene sharding helper assigns scenes to ranks."""
    from openfdcm_b200 import distributed as fd
    tmpls = synth_templates(30, 40, 640, seed=5100)
    tset = fdcm.TemplateSet(tmpls)
    scenes = [plant_instances(synth_scene(640, 480, 200, seed=5000 + s), tmpls, 640, 480, seed=5200 + s) for s in range(4)]
    assert sorted(fd.shard_scenes(4, 0, 2) + fd.shard_scenes(4, 1, 2)) == [0, 1, 2, 3]
    fm = fdcm.build_cuda_featuremap(scenes[0], fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    for s, scene in enumerate(scenes):
        if s:
            fm.rebuild(scene, wait=(s % 2 == 0))   # odd scenes: asynchronous rebuild, the search is stream-ordered after it
        top = fdcm.search_topk(fm, tset, None, fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), fdcm.ExponentialPenalty(1.5), k=10)
        c = orc.Dt3Cpu(scene, 30, 5.0, 1.5)
        pen = orc.penalize(1, 1.5, c.search(tmpls, scene, 4, 4, batch=10), orc.template_lengths(tmpls))
        assert np.array_equal(top, pen[np.lexsort((np.arange(len(pen)), pen["score"]))[:10]]), f"scene {s}"


def test_concentric_range_search_on_gpu():
    """ConcentricRangeStrategy (concentricrange.cpp:29-60) through the fused CUDA search, incl. the resident-scene path
    switching between filters and the empty-filter case."""
    scene, tmpls = _workload(61, n_tmpl=10, n_lines=22)
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    c = orc.Dt3Cpu(scene, 30, 5.0, 1.5)
    opt = fdcm.BatchOptimize(10)
    for lo_r, hi_r in ((0.0, 150.0), (100.0, 260.0), (5000.0, 6000.0), (0.0, 150.0)):
        s = fdcm.ConcentricRangeStrategy(4, 5, (320, 240), lo_r, hi_r)
        for sc in (scene, None):
            got = fdcm.search_all(g, tmpls, sc, s, opt)
            want, hyp = c.search(tmpls, scene, 4, 5, batch=10, want_hyp=True, concentric=[320, 240, lo_r, hi_r])
            assert np.array_equal(g.last_hypotheses().reshape(-1, 4), hyp.reshape(-1, 4))
            assert np.array_equal(got["score"], want["score"]) and np.array_equal(got["transform"], want["transform"])
    got = fdcm.search_all(g, tmpls, None, fdcm.DefaultSearch(4, 5), opt)      # back to the unfiltered ordering
    assert np.array_equal(got["score"], c.search(tmpls, scene, 4, 5, batch=10)["score"])


def test_real_asset_regression():
    """Real detected lines (reference notebooks/assets/obj_01: one 557-line scene, 24 templates) with the parameters of
    notebooks/pose_extimation_example.ipynb: DefaultSearch(4,10), BatchOptimize(10), depth 30, coeff 5, padding 1.0, L2."""
    import glob
    import os
    real = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "real_assets", "obj_01")
    scene = fdcm.read(os.path.join(real, "scene_0", "camera_0.scene"))
    tmpls = [fdcm.read(os.path.join(real, "templates", f"template_{i}.tmpl")) for i in range(24)]
    assert len(tmpls) == 24
    for padding in (1.0, 2.2):
        g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, padding))
        c = orc.Dt3Cpu(scene, 30, 5.0, padding)
        for d in (0, 9, 15, 27):
            assert np.array_equal(g.plane(d), c.plane(d))
        got = fdcm.search_all(g, tmpls, scene, fdcm.DefaultSearch(4, 10), fdcm.BatchOptimize(10))
        want, hyp = c.search(tmpls, scene, 4, 10, batch=10, want_hyp=True)
        assert np.array_equal(g.last_hypotheses(), hyp)
        assert len(got) == len(want)
        assert np.array_equal(got["score"], want["score"]) and np.array_equal(got["transform"], want["transform"])
        top = fdcm.search_topk(g, tmpls, scene, fdcm.DefaultSearch(4, 10), fdcm.BatchOptimize(10), fdcm.ExponentialPenalty(1.5), k=10)
        pen = orc.penalize(1, 1.5, want, orc.template_lengths(tmpls))
        assert np.array_equal(top, pen[np.lexsort((np.arange(len(pen)), pen["score"]))[:10]])


def _special_scene(kind, w, h, rng):
    """Geometries that stress the band kernels: a single line, lines on the borders of the extent (edges in the first /
    last map row at padding 1), a dense corner cluster plus one far line, all lines in one orientation bin."""
    if kind == 0:
        return np.array([[w * 0.2], [h * 0.3], [w * 0.7], [h * 0.35]], F32)
    if kind == 1:
        ls = [[0, 0, w - 1, 0], [0, h - 1, w - 1, h - 1], [0, 0, 0, h - 1], [w - 1, 0, w - 1, h - 1], [w / 2, 0, w / 2, h - 1],
              [0, h / 2, w - 1, h / 2]]
        return np.array(ls, F32).T.copy()
    if kind == 2:
        s = synth_scene(max(w // 4, 80), max(h // 4, 60), 40, seed=int(rng.integers(1 << 30)), min_len=4.0)
        return np.ascontiguousarray(np.concatenate([s, np.array([[w - 30], [h - 20], [w - 5], [h - 3]], F32)], axis=1), F32)
    if kind == 3:
        n = 25
        cx, cy = rng.uniform(0, w - 1, n), rng.uniform(0, h - 1, n)
        ln, th = rng.uniform(10, 0.3 * w, n), 0.3 + rng.uniform(-0.02, 0.02, n)
        l = np.stack([cx - ln * np.cos(th) / 2, cy - ln * np.sin(th) / 2, cx + ln * np.cos(th) / 2, cy + ln * np.sin(th) / 2])
        l[[0, 2]] = np.clip(l[[0, 2]], 0, w - 1)
        l[[1, 3]] = np.clip(l[[1, 3]], 0, h - 1)
        return np.ascontiguousarray(l, F32)
    return synth_scene(w, h, int(rng.integers(3, 200)), seed=int(rng.integers(1 << 30)), max_len_frac=float(rng.uniform(0.3, 0.6)),
                       min_len=4.0)


@pytest.mark.parametrize("case", range(12))
def test_randomised_scenes_bit_exact(case):
    """Random sizes / paddings / special geometries, all three distances: full maps and full match lists bit-exact against
    the oracle (scripts/fuzz_parity.py runs a longer sweep of the same kind)."""
    rng = np.random.default_rng(1000 + case)
    w, h = int(rng.integers(40, 700)), int(rng.integers(40, 500))
    pad = float(rng.choice([1.0, 1.2, 1.5, 2.2]))
    name = ["L2", "L2_SQUARED", "L1"][case % 3]
    gd, od = DIST[name]
    scene = _special_scene(case % 6, w, h, rng)
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, pad, gd))
    c = orc.Dt3Cpu(scene, 30, 5.0, pad, od)
    assert (g.width, g.height) == (c.W, c.H)
    for d in range(30):
        assert np.array_equal(g.plane(d), c.plane(d)), f"plane {d} of case {case} ({name}, {w}x{h}, padding {pad})"
    tm = synth_templates(6, 12, max(w, 100), seed=case)
    got = fdcm.search_all(g, tm, scene, fdcm.DefaultSearch(3, 4), fdcm.BatchOptimize(10))
    want = c.search(tm, scene, 3, 4, batch=10)
    assert np.array_equal(got["tmpl_idx"], want["tmpl_idx"])
    assert np.array_equal(got["score"], want["score"], equal_nan=True)
    assert np.array_equal(got["transform"], want["transform"], equal_nan=True)


def test_empty_search_scene_yields_no_matches():
    """defaultmatch.cpp:40: an empty originalScene gives no matches — it must NOT fall back to the resident build scene
    (that is what n_scene == FDCM_SCENE_RESIDENT / scene=None asks for explicitly)."""
    scene, tmpls = _workload(8, n_tmpl=3)
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    s, o = fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10)
    assert fdcm.search(fdcm.DefaultMatch(), s, o, g, tmpls, np.zeros((4, 0), F32)) == []
    assert len(fdcm.search_all(g, tmpls, np.zeros((4, 0), F32), s, o)) == 0
    assert len(fdcm.search_all(g, tmpls, None, s, o)) == len(fdcm.search_all(g, tmpls, scene, s, o)) > 0


def test_failed_rebuild_leaves_an_empty_map():
    """A rebuild that is rejected (feature size out of range) must not leave a handle mixing the old map with the new
    scene: the map becomes the empty map and a search on it returns nothing."""
    scene, tmpls = _workload(8, n_tmpl=3)
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    huge = (scene * 100.0).astype(F32)           # side ~ 96000 > the supported maximum
    with pytest.raises(fdcm.FdcmError):
        g.rebuild(huge)
    g._refresh()
    assert g.get_feature_size().tolist() == [0, 0] and g.depth == 0
    assert len(fdcm.search_all(g, tmpls, None, fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10))) == 0
    g.rebuild(scene)                              # and the handle is still usable
    c = orc.Dt3Cpu(scene, 30, 5.0, 1.5)
    assert np.array_equal(g.plane(3), c.plane(3))


def test_two_devices_in_one_process():
    """The opt-in shared-memory attributes are per device: maps built on two devices from one process."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two devices")
    scene, tmpls = _workload(8, n_tmpl=3)
    c = orc.Dt3Cpu(scene, 30, 5.0, 1.5)
    want = c.search(tmpls, scene, 4, 4, batch=10)
    for dev in (0, 1, 0):
        g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5, device=dev))
        assert np.array_equal(g.plane(11), c.plane(11))
        got = fdcm.search_all(g, fdcm.TemplateSet(tmpls, device=dev), scene, fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10))
        assert np.array_equal(got["score"], want["score"])


def test_comm_world1_device_merge():
    """fdcm_comm_* with a single rank: the NCCL all-gather + merge kernel path returns the plain top-k."""
    from openfdcm_b200 import distributed as fd
    scene, tmpls = _workload(77, n_tmpl=40, n_lines=25)
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    comm = fd.Communicator(fd.Communicator.unique_id(), 0, 1, 0)
    assert comm.shard(40) == (0, 40)
    s, o, p = fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), fdcm.ExponentialPenalty(1.5)
    want = fdcm.search_topk(g, tmpls, scene, s, o, p, k=10)
    got = comm.search_topk(g, fdcm.TemplateSet(tmpls), scene, s, o, p, 10, 0)
    assert np.array_equal(got, want)
    # fewer matches than k, and an empty shard
    assert np.array_equal(comm.search_topk(g, fdcm.TemplateSet(tmpls[:1]), None, s, o, p, 50, 0), fdcm.search_topk(g, tmpls[:1], None, s, o, p, k=50))
    assert len(comm.search_topk(g, fdcm.TemplateSet([]), None, s, o, p, 10, 0)) == 0
    c = orc.Dt3Cpu(scene, 30, 5.0, 1.5)
    comm.rebuild_broadcast(g, scene, root=0)
    assert np.array_equal(g.plane(7), c.plane(7))


def test_cpp_type_erased_strategies():
    """tests/cpp/test_type_erasure.cpp: FeatureMap / SearchStrategy / OptimizeStrategy / MatchStrategy / PenaltyStrategy
    (Concept / Model + clone, featuremap.h:57-124, matchstrategy.h:83-140) over the CUDA types; fused path == generic
    composition == clones."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "tests", "cpp", "test_type_erasure")
    if not os.path.exists(exe):
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(root, "include"), exe + ".cpp", "-L" + os.path.join(root, "openfdcm_b200"),
                               "-lfdcm_b200", "-Wl,-rpath,$ORIGIN/../../openfdcm_b200", "-o", exe])
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "fused == generic == cloned" in r.stdout


def test_scene_batch_pipelined_builds():
    """fdcm_search_scenes: double-buffered maps, build(s+1) on a second stream under search(s); every scene's top-10 equals
    the oracle's, including an empty scene in the middle and scenes of different map sizes."""
    tmpls = synth_templates(30, 40, 640, seed=5100)
    tset = fdcm.TemplateSet(tmpls)
    scenes = [plant_instances(synth_scene(640, 480, 200, seed=5000 + s), tmpls, 640, 480, seed=5200 + s) for s in range(5)]
    scenes.insert(2, np.zeros((4, 0), F32))
    scenes.append(plant_instances(synth_scene(400, 300, 90, seed=5900), tmpls, 400, 300, seed=5901))
    batch = fdcm.SceneBatch(fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    s_, o_, p_ = fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), fdcm.ExponentialPenalty(1.5)
    for rep in range(2):          # the second pass reuses the two maps
        got = batch.search_topk(scenes, tset, s_, o_, p_, k=10)
        assert len(got) == len(scenes)
        for i, scene in enumerate(scenes):
            if scene.shape[1] == 0:
                assert len(got[i]) == 0
                continue
            c = orc.Dt3Cpu(scene, 30, 5.0, 1.5)
            pen = orc.penalize(1, 1.5, c.search(tmpls, scene, 4, 4, batch=10), orc.template_lengths(tmpls))
            assert np.array_equal(got[i], pen[np.lexsort((np.arange(len(pen)), pen["score"]))[:10]]), f"scene {i} (pass {rep})"
