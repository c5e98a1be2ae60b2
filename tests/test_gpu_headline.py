"""Parity AT THE HEADLINE SIZES (VERDICT r01 item J1): the CUDA path against the CPU oracle on the very workloads
bench.py times — config 2 (2880 x 2880 x 30 map of the padded 1080p scene, all three distances, every plane,
plus the stage-1 / stage-2 intermediates of L2) and config 3 (5000 templates x 40 lines, 160 000 hypotheses:
hypothesis list, full match list, top-10).  Reference pipeline being matched:
matching/featuremaps/dt3cpu.h:174-234 and matching/src/matchstrategies/defaultmatch.cpp:32-89.

Everything is asserted bit-exact (np.array_equal); the north-star tolerances (1e-5 DT3, 1e-4 scores) are only
quoted in the failure message.
"""
import os
import sys

import numpy as np
import pytest

import openfdcm_b200 as fdcm
from oracle import fdcm_oracle as orc
from tests.helpers import DIST
from tests.util import synth_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import bench  # noqa: E402  (the workload generator of the headline benchmark)

pytestmark = pytest.mark.gpu


def _compare_all_planes(g, c, what):
    assert (g.width, g.height, g.depth) == (c.W, c.H, c.depth) == (2880, 2880, 30)
    assert np.array_equal(g.angles(), c.keys)
    assert np.array_equal(g.get_scene_translation(), c.shift)
    for d in range(c.depth):
        a, b = g.plane(d), c.plane(d)
        if not np.array_equal(a, b):
            diff = a != b
            rel = np.abs(a[diff] - b[diff]) / np.maximum(np.abs(b[diff]), 1e-30)
            pytest.fail(f"{what}: plane {d}: {int(diff.sum())} of {a.size} values differ from the oracle "
                        f"(max rel {rel.max():.3g}; north-star tolerance 1e-5), first at {np.argwhere(diff)[:3].tolist()}")


@pytest.mark.parametrize("dist", ["L2", "L2_SQUARED", "L1"])
def test_config2_full_map_bit_exact(dist):
    """BASELINE config 2: synthetic 1920x1080 scene, 2000 lines, depth 30, padding 1.5 — all 30 planes of the
    2880x2880 map equal to orc.Dt3Cpu, for every distance type (band path for L2 / L2^2, record path for L1)."""
    scene = synth_scene(1920, 1080, 2000, seed=2000)
    gd, od = DIST[dist]
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5, gd))
    assert g.info.exact_dt_path == 1
    c = orc.Dt3Cpu(scene, 30, 5.0, 1.5, od)
    _compare_all_planes(g, c, f"config 2 {dist}")


@pytest.mark.parametrize("stage", [1, 2], ids=["dt", "propagated"])
def test_config2_l2_intermediates_bit_exact(stage):
    """The distance transforms (imgproc.h:169-194) and the propagated planes (dt3cpu.cpp:77-107) of config 2, L2."""
    scene = synth_scene(1920, 1080, 2000, seed=2000)
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5, fdcm.distance.L2), stage=stage)
    c = orc.Dt3Cpu(scene, 30, 5.0, 1.5, orc.L2, stage=stage)
    _compare_all_planes(g, c, f"config 2 L2 stage {stage}")


def test_config2_rerun_is_idempotent():
    """The bench times fdcm_dt3_rerun: re-running the build kernels on the resident scene must reproduce the map."""
    scene = synth_scene(1920, 1080, 2000, seed=2000)
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    before = [g.plane(d) for d in (0, 7, 15, 22, 29)]
    g.rerun()
    g.rerun()
    for d, b in zip((0, 7, 15, 22, 29), before):
        assert np.array_equal(g.plane(d), b)


@pytest.fixture(scope="module")
def config3():
    scene, tmpls = bench.make_workload(0)
    g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(bench.DEPTH, bench.COEFF, bench.PADDING, fdcm.distance.L2))
    c = orc.Dt3Cpu(scene, bench.DEPTH, bench.COEFF, bench.PADDING, orc.L2)
    raw, hyp = c.search(tmpls, scene, bench.MAX_T, bench.MAX_S, batch=bench.BATCH, want_hyp=True)
    pen = orc.penalize(1, bench.TAU, raw, orc.template_lengths(tmpls))
    return scene, tmpls, g, c, raw, hyp, pen


def test_config3_map_of_the_bench_scene(config3):
    _, _, g, c, _, _, _ = config3
    _compare_all_planes(g, c, "config 3 map")


def test_config3_full_match_list_bit_exact(config3):
    """bench.make_workload(0): hypothesis list, all 160 000 match records (penalised) in hypothesis order."""
    scene, tmpls, g, c, raw, hyp, pen = config3
    got = fdcm.search_all(g, tmpls, scene, fdcm.DefaultSearch(bench.MAX_T, bench.MAX_S), fdcm.BatchOptimize(bench.BATCH),
                          fdcm.ExponentialPenalty(bench.TAU))
    assert len(hyp) == bench.N_TMPL * bench.MAX_T * bench.MAX_S * 2 == 160000
    assert np.array_equal(g.last_hypotheses(), hyp), "hypothesis list must be bit-exact"
    assert len(got) == len(pen)
    assert np.array_equal(got["tmpl_idx"], pen["tmpl_idx"])
    assert np.array_equal(got["transform"], pen["transform"])
    assert np.allclose(got["score"], pen["score"], rtol=1e-4, atol=0)
    assert np.array_equal(got["score"], pen["score"]), "scores within 1e-4 but not bit-exact"


def test_config3_top10_bit_exact(config3):
    """The benched call: resident template set, resident scene, fused penalty + top-10."""
    scene, tmpls, g, c, raw, hyp, pen = config3
    want = pen[np.lexsort((np.arange(len(pen)), pen["score"]))[:bench.TOP_K]]
    tset = fdcm.TemplateSet(tmpls)
    for sc in (scene, None):
        top = fdcm.search_topk(g, tset, sc, fdcm.DefaultSearch(bench.MAX_T, bench.MAX_S), fdcm.BatchOptimize(bench.BATCH),
                               fdcm.ExponentialPenalty(bench.TAU), bench.TOP_K)
        assert np.array_equal(top, want)
    # template sharding keeps global indices: two shards merged == the single list
    half = bench.N_TMPL // 2
    parts = []
    for r, (lo, hi) in enumerate(((0, half), (half, bench.N_TMPL))):
        parts.append(fdcm.search_topk(g, tmpls[lo:hi], None, fdcm.DefaultSearch(bench.MAX_T, bench.MAX_S),
                                      fdcm.BatchOptimize(bench.BATCH), fdcm.ExponentialPenalty(bench.TAU), bench.TOP_K, lo))
    both = np.concatenate(parts)
    merged = both[np.lexsort((np.arange(len(both)), both["score"]))[:bench.TOP_K]]
    assert np.array_equal(merged["tmpl_idx"], want["tmpl_idx"]) and np.array_equal(merged["score"], want["score"])
