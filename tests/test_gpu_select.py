"""Distinct top-K on the device (fdcm_search_select, DistinctMatches): bit-exact against the numpy model of
tests/test_select_host.py applied to search_all(..., penalty), which is itself bit-exact with the oracle."""
import glob
import math
import os
import socket

import numpy as np
import pytest

import openfdcm_b200 as fdcm
from openfdcm_b200._lib import FDCM_ERR_INVALID
from tests.test_select_host import select_model
from tests.util import F32, plant_instances, synth_scene, synth_templates

pytestmark = pytest.mark.gpu
ASSETS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "real_assets")
PEN = fdcm.ExponentialPenalty(1.5)
OPT = fdcm.BatchOptimize(10)


def settings(n_tmpl):
    for cap in (0, 1, 2):
        for radius, angle in ((0.0, math.pi), (5.0, math.pi), (5.0, 0.2), (20.0, math.pi), (20.0, 0.2)):
            for across in (False, True):
                for k in (1, 10, n_tmpl):
                    yield cap, radius, angle, across, k


def check(fm, tset, anchors, scene, searcher, cases, what=""):
    """search_topk(select=...) == the model over search_all(..., penalty) for every (cap, radius, angle, across, k)."""
    allm = fdcm.search_all(fm, tset, scene, searcher, OPT, PEN)
    for cap, radius, angle, across, k in cases:
        sel = fdcm.DistinctMatches(cap, radius, angle, across)
        got = fdcm.search_topk(fm, tset, scene, searcher, OPT, PEN, k=k, select=sel)
        want = allm[select_model(allm, anchors, k, cap, radius, angle, across)]
        assert got.tobytes() == want.tobytes(), f"{what} {sel} k={k}: got {got['tmpl_idx']} want {want['tmpl_idx']}"
    return allm


def synthetic(n_tmpl=24, n_lines=20, seed=0, w=640, h=480, n_scene=200):
    tmpls = synth_templates(n_tmpl, n_lines, w, seed=seed + 1)
    scene = plant_instances(synth_scene(w, h, n_scene, seed=seed + 2), tmpls, w, h, seed=seed + 3, count=6)
    return tmpls, scene


def test_synthetic_scene_bit_exact():
    tmpls, scene = synthetic()
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    check(fm, fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls), scene, fdcm.DefaultSearch(4, 4), settings(len(tmpls)), "synthetic")


def load_object(obj):
    tm = sorted(glob.glob(os.path.join(ASSETS, obj, "templates", "*.tmpl")), key=lambda p: int(os.path.basename(p)[9:-5]))
    scenes = sorted(glob.glob(os.path.join(ASSETS, obj, "scene_*", "camera_0.scene")), key=lambda p: int(os.path.basename(os.path.dirname(p))[6:]))
    return [fdcm.read(p) for p in tm], [fdcm.read(p) for p in scenes]


@pytest.mark.parametrize("obj", ["obj_01", "obj_02", "obj_03", "obj_04"])
def test_real_assets_bit_exact(obj):
    """The notebook's parameters (DefaultSearch(4, 10), BatchOptimize(10), ExponentialPenalty(1.5), depth 30, padding 1)."""
    tmpls, scenes = load_object(obj)
    tset, anchors = fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls)
    s = fdcm.DefaultSearch(4, 10)
    for i in (0, 1):
        fm = fdcm.build_cuda_featuremap(scenes[i], fdcm.Dt3CudaParameters(30, 5.0, 1.0))
        allm = check(fm, tset, anchors, None, s, settings(len(tmpls)), f"{obj} scene {i}")
        # one best match per view: 10 distinct templates whenever 10 templates match
        top = fdcm.search_topk(fm, tset, None, s, OPT, PEN, k=10, select=fdcm.DistinctMatches(max_per_template=1))
        assert len(set(top["tmpl_idx"].tolist())) == len(top) == min(10, len(set(allm["tmpl_idx"].tolist())))
        # across templates, no two results with anchors within 10 px at a rotation difference within max_angle
        top = fdcm.search_topk(fm, tset, None, s, OPT, PEN, k=10, select=fdcm.DistinctMatches(radius=10, max_angle=0.26, across_templates=True))
        T = top["transform"].reshape(-1, 6)
        a = anchors[top["tmpl_idx"]]
        p = np.stack([T[:, 0] * a[:, 0] + T[:, 1] * a[:, 1] + T[:, 2], T[:, 3] * a[:, 0] + T[:, 4] * a[:, 1] + T[:, 5]], 1)
        for x in range(len(top)):
            for y in range(x):
                close = np.hypot(*(p[x] - p[y])) < 9.99
                same_rot = T[x, 0] * T[y, 0] + T[x, 3] * T[y, 3] > math.cos(0.26) + 1e-6
                assert not (close and same_rot), f"{obj} scene {i}: results {y} and {x}"


def test_no_op_selection_is_plain_top_k():
    tmpls, scene = synthetic(seed=40)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    tset = fdcm.TemplateSet(tmpls)
    for k in (1, 10, 500):
        for sel in (fdcm.DistinctMatches(), fdcm.DistinctMatches(across_templates=True, max_angle=0.1)):
            plain = fdcm.search_topk(fm, tset, scene, fdcm.DefaultSearch(4, 4), OPT, PEN, k=k)
            assert fdcm.search_topk(fm, tset, scene, fdcm.DefaultSearch(4, 4), OPT, PEN, k=k, select=sel).tobytes() == plain.tobytes()


@pytest.mark.parametrize("max_t,max_s,n_lines", [(4, 4, 20), (4, 10, 20), (16, 16, 24), (64, 40, 70)])
def test_segment_lengths(max_t, max_s, n_lines):
    """32, 80, 512 and 5120 hypotheses per template: one chunk of the per-template walk up to 160 chunks."""
    tmpls, scene = synthetic(n_tmpl=6, n_lines=n_lines, seed=100 + max_t, n_scene=300)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    searcher = fdcm.DefaultSearch(max_t, max_s)
    cases = [(cap, r, ang, across, k) for cap in (0, 1, 2) for r, ang in ((0.0, math.pi), (5.0, math.pi), (20.0, 0.2))
             for across in (False, True) for k in (1, 10, 300)]
    allm = check(fm, fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls), scene, searcher, cases, f"DefaultSearch({max_t},{max_s})")
    assert fm.last_search_stats()["n_hypotheses"] == 2 * 6 * max_t * max_s and len(allm) > 0


def test_edge_cases():
    tmpls, scene = synthetic(n_tmpl=10, seed=200)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    s = fdcm.DefaultSearch(4, 4)
    sel = fdcm.DistinctMatches(max_per_template=1, radius=5)
    # an empty scene: no matches
    assert len(fdcm.search_topk(fm, tmpls, np.zeros((4, 0), F32), s, OPT, PEN, k=10, select=sel)) == 0
    # a set with an empty template (no hypotheses of its own)
    with_empty = tmpls[:4] + [np.zeros((4, 0), F32)] + tmpls[4:]
    cases = [(1, 5.0, math.pi, False, 10), (0, 20.0, 0.2, True, 10), (2, 0.0, math.pi, False, 11)]
    check(fm, fdcm.TemplateSet(with_empty), fdcm.get_template_anchors(with_empty), scene, s, cases, "empty template")
    # k larger than the number of survivors: fewer records
    allm = fdcm.search_all(fm, tmpls, scene, s, OPT, PEN)
    got = fdcm.search_topk(fm, tmpls, scene, s, OPT, PEN, k=100, select=fdcm.DistinctMatches(max_per_template=1))
    assert len(got) == len(set(allm["tmpl_idx"].tolist())) < 100
    assert got.tobytes() == allm[select_model(allm, fdcm.get_template_anchors(tmpls), 100, 1)].tobytes()
    # ConcentricRange: only the scene lines in a ring take part, the selection applies to what remains
    ring = fdcm.ConcentricRangeStrategy(4, 4, [320, 240], 30, 220)
    check(fm, fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls), scene, ring,
          [(1, 0.0, math.pi, False, 10), (0, 20.0, 0.2, False, 10), (2, 20.0, math.pi, True, 5)], "concentric")


def test_scene_batch_equals_per_scene():
    tmpls = synth_templates(30, 30, 640, seed=300)
    tset = fdcm.TemplateSet(tmpls)
    scenes = [plant_instances(synth_scene(640, 480, 200, seed=310 + i), tmpls, 640, 480, seed=320 + i) for i in range(4)]
    params = fdcm.Dt3CudaParameters(30, 5.0, 1.5)
    batch = fdcm.SceneBatch(params)
    s = fdcm.DefaultSearch(4, 4)
    for sel in (fdcm.DistinctMatches(max_per_template=1), fdcm.DistinctMatches(2, 10.0, 0.26), fdcm.DistinctMatches(radius=10, across_templates=True)):
        got = batch.search_topk(scenes, tset, s, OPT, PEN, k=10, select=sel)
        for i, scene in enumerate(scenes):
            fm = fdcm.build_cuda_featuremap(scene, params)
            assert got[i].tobytes() == fdcm.search_topk(fm, tset, None, s, OPT, PEN, k=10, select=sel).tobytes(), f"{sel} scene {i}"


def test_invalid_parameters():
    tmpls, scene = synthetic(n_tmpl=4, seed=400)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    tset = fdcm.TemplateSet(tmpls)
    s = fdcm.DefaultSearch(4, 4)
    bad = [(0, fdcm.DistinctMatches(max_per_template=1)), (10, fdcm.DistinctMatches(max_per_template=-1)),
           (10, fdcm.DistinctMatches(radius=-1.0)), (10, fdcm.DistinctMatches(radius=math.inf)), (10, fdcm.DistinctMatches(radius=math.nan)),
           (10, fdcm.DistinctMatches(radius=5, max_angle=-0.1)), (10, fdcm.DistinctMatches(radius=5, max_angle=math.nan)),
           (1025, fdcm.DistinctMatches(radius=5, across_templates=True))]
    for k, sel in bad:
        with pytest.raises(fdcm.FdcmError) as e:
            fdcm.search_topk(fm, tset, scene, s, OPT, PEN, k=k, select=sel)
        assert e.value.status == FDCM_ERR_INVALID, sel
    with pytest.raises(fdcm.FdcmError) as e:
        fdcm.SceneBatch(fdcm.Dt3CudaParameters(30, 5.0, 1.5)).search_topk([scene], tset, s, OPT, PEN, k=10,
                                                                          select=fdcm.DistinctMatches(max_per_template=-1))
    assert e.value.status == FDCM_ERR_INVALID
    # the bound itself is accepted
    assert len(fdcm.search_topk(fm, tset, scene, s, OPT, PEN, k=1024, select=fdcm.DistinctMatches(radius=5, across_templates=True))) > 0
    from openfdcm_b200 import distributed as fd
    comm = fd.Communicator(fd.Communicator.unique_id(), 0, 1, 0)
    with pytest.raises(fdcm.FdcmError) as e:
        comm.search_topk(fm, tset, scene, s, OPT, PEN, 10, 0, select=fdcm.DistinctMatches(radius=5, across_templates=True))
    assert e.value.status == FDCM_ERR_INVALID
    sel = fdcm.DistinctMatches(max_per_template=1, radius=5)
    assert comm.search_topk(fm, tset, scene, s, OPT, PEN, 10, 0, select=sel).tobytes() == \
        fdcm.search_topk(fm, tset, scene, s, OPT, PEN, k=10, select=sel).tobytes()


def test_pybind_and_profile_names():
    from openfdcm_b200 import _openfdcm_cuda as pyfdcm
    tmpls, scene = synthetic(n_tmpl=12, seed=500)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    pfm = pyfdcm.build_cuda_featuremap(scene, pyfdcm.Dt3CudaParameters(30, 5.0, 1.5))
    want = fdcm.search_topk(fm, tmpls, scene, fdcm.DefaultSearch(4, 4), OPT, PEN, k=10, select=fdcm.DistinctMatches(1, 10.0, 0.3))
    got = pyfdcm.search_topk(pfm, tmpls, scene, pyfdcm.DefaultSearch(4, 4), pyfdcm.BatchOptimize(10), pyfdcm.ExponentialPenalty(1.5), 10,
                             select=pyfdcm.DistinctMatches(max_per_template=1, radius=10.0, max_angle=0.3))
    assert [m.tmpl_idx for m in got] == want["tmpl_idx"].tolist()
    assert [m.score for m in got] == want["score"].tolist()
    fdcm.profile(True, reset=True)
    fdcm.search_topk(fm, tmpls, scene, fdcm.DefaultSearch(4, 4), OPT, PEN, k=10, select=fdcm.DistinctMatches(1))
    fdcm.search_topk(fm, tmpls, scene, fdcm.DefaultSearch(4, 4), OPT, PEN, k=10, select=fdcm.DistinctMatches(radius=5, across_templates=True))
    rep = fdcm.profile_report()
    fdcm.profile(False)
    assert {"select_sort", "select_greedy", "select_topk", "select_walk"} <= set(rep)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _two_rank_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)   # ships the NCCL id; the search exchange is NCCL
    try:
        from openfdcm_b200 import distributed as fd
        tmpls, scene = synthetic(n_tmpl=40, seed=600)
        fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5, device=rank))
        comm = fd.Communicator.from_torch(rank)
        b, e = comm.shard(len(tmpls))
        sel = fdcm.DistinctMatches(max_per_template=1)
        got = comm.search_topk(fm, fdcm.TemplateSet(tmpls[b:e], device=rank), None, fdcm.DefaultSearch(4, 4), OPT, PEN, 10, b, select=sel)
        want = fdcm.search_topk(fm, fdcm.TemplateSet(tmpls, device=rank), None, fdcm.DefaultSearch(4, 4), OPT, PEN, k=10, select=sel)
        q.put((rank, got.tobytes() == want.tobytes() and len(got) == 10))
    finally:
        dist.destroy_process_group()


def test_two_ranks_equal_single_gpu():
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two devices")
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_two_rank_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=600) for _ in range(world)]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert sorted(res) == [(0, True), (1, True)]
