#!/usr/bin/env python
"""bench.py — headline benchmark (BASELINE.json): template matches/sec on the pose-estimation sweep
(config 3: 5000 templates x 40 lines vs one 1080p scene, DefaultSearch(4,4), BatchOptimize(10),
depth 30, coeff 5, padding 1.5, L2, ExponentialPenalty(1.5), top-10), plus the DT3 build ms of the
same padded 1080p scene (config 2) for L2 / L2_SQUARED / L1.

A step = one pass of the hot path over one batch: build the scene's DT3 map + search this rank's
template shard + top-10 (+ the device-side all-gather / merge of the ranks' top-10 when N > 1,
fdcm_comm_search_topk).  `value` is WEAK scaling: every rank searches its own 5000 templates of a
global set of N x 5000 (template sharding by tmpl_idx, each rank builds the map itself; the only
collective is the 320-byte top-K all-gather).  `strong_scaling` reports the same step with the 5000
templates of config 3 split over the N ranks (the replicated 1.5 ms build is its Amdahl term).

  value : templates/s with scene lines + templates already resident in HBM (kernels + top-K readback)
  e2e   : the same through the host-buffer C-ABI calls (pinned host lines in, matches out; H2D/D2H timed)
  roofline / build_roofline : dominant kernel and the whole build against the measured HBM peak
  parity : the benched top-10 equals the CPU oracle's (checked outside the timed region)
  config4 / config5 : templates/s of the wide 4K search, scenes/s of the multi-scene batch
  --impl reference : the CPU oracle (port of the reference, all host threads), whole job per step.
  --dump-outputs DIR : after the timed steps, the outputs of the last step as DIR/<name>.npy (see dump_outputs).

Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "template_matches_per_sec"
UNIT = "templates/s"
N_TMPL, N_TMPL_LINES, TOP_K = 5000, 40, 10
SCENE_W, SCENE_H, N_SCENE = 1920, 1080, 2000
DEPTH, COEFF, PADDING, TAU = 30, 5.0, 1.5, 1.5
MAX_T, MAX_S, BATCH = 4, 4, 10
L2_PEAK_GBS = 6300.0 * 1.965   # LTS cap of the microarchitecture notes (~6300 B/clk) x max SM clock: a reference figure, not measured here
CONFIG = {
    "workload": "config3 pose sweep: 5000 templates x 40 lines per GPU vs one 1920x1080 scene (2000 lines + planted "
                "instances), DefaultSearch(4,4), BatchOptimize(10), depth 30, coeff 5, padding 1.5, L2, "
                "ExponentialPenalty(1.5), top-10; step = DT3 build (2880x2880x30) + search + top-K",
    "sharding": "templates by tmpl_idx (weak: 5000 per GPU, global set of N x 5000); every rank builds the scene map itself; "
                "top-K merged on the device (NCCL all-gather of k x 32 B + merge kernel)",
    "l2_policy": "inputs larger than L2: the 995 MB map is rebuilt every step",
}


def make_workload(rank):
    from tests.util import plant_instances, synth_scene, synth_templates
    base = synth_templates(N_TMPL, N_TMPL_LINES, SCENE_W, seed=3001)               # rank 0's shard plants the instances
    scene = plant_instances(synth_scene(SCENE_W, SCENE_H, N_SCENE, seed=3000), base, SCENE_W, SCENE_H, seed=3002)
    tmpls = base if rank == 0 else synth_templates(N_TMPL, N_TMPL_LINES, SCENE_W, seed=3001 + 17 * rank)
    return scene, tmpls


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self._stop_evt = index, [], set(), None, threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for nm, v in zip(names, out[2:]):
                    if v.strip().lower() == "active":
                        self.reasons.add(nm)
            except Exception:
                pass
            self._stop_evt.wait(0.05)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=10)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def load_traffic():
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f)
    except Exception:
        return {}


MAP_SAMPLE_PER_PLANE = 1 << 17   # 30 planes x 128 Ki values x 4 B = 15.7 MB of the 995 MB map


def dump_outputs(out_dir, fm, top):
    """What a caller of the timed step receives from it: the top-10 matches and the DT3 map they were searched in.
    The map is too large to store whole, so a fixed, seeded sample of positions of every plane stands for it."""
    os.makedirs(out_dir, exist_ok=True)
    idx = np.random.default_rng(0).integers(0, fm.height * fm.width, (fm.depth, MAP_SAMPLE_PER_PLANE))
    arrays = {"top10_tmpl_idx": top["tmpl_idx"].astype(np.float64), "top10_score": top["score"],
              "top10_transform": top["transform"].reshape(-1, 2, 3),
              "dt3_map_sample": np.stack([fm.plane(d).reshape(-1)[idx[d]] for d in range(fm.depth)])}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def oracle_job(scene, tmpls, nthreads=0):
    """The CPU oracle (port of the reference, ThreadPool decomposition) on the WHOLE job: one full map build + the
    search / penalize / sort of every template.  Returns timings and the penalised match list."""
    from oracle import fdcm_oracle as orc
    cores = nthreads or orc.hardware_concurrency()
    t0 = time.perf_counter()
    fm = orc.Dt3Cpu(scene, DEPTH, COEFF, PADDING, orc.L2, nthreads=cores)
    t_build = time.perf_counter() - t0
    t0 = time.perf_counter()
    raw = fm.search(tmpls, scene, MAX_T, MAX_S, batch=BATCH, nthreads=cores)
    pen = orc.penalize(1, TAU, raw, orc.template_lengths(tmpls))
    srt = orc.sort_matches(pen)
    t_search = time.perf_counter() - t0
    del srt
    return {"cores": cores, "build_s": t_build, "search_s": t_search, "pen": pen}


def oracle_top(pen, k):
    return pen[np.lexsort((np.arange(len(pen)), pen["score"]))[:k]]


def cpu_baseline(scene, tmpls):
    j = oracle_job(scene, tmpls)
    t = j["build_s"] + j["search_s"]
    return {"value": len(tmpls) / t, "unit": UNIT, "cores": j["cores"], "kind": "port",
            "sample": f"the whole job once: 1 full DT3 build ({j['build_s']:.2f} s) + search/penalize/sort of all {len(tmpls)} templates "
                      f"({j['search_s']:.3f} s), no extrapolation",
            "build_s": j["build_s"], "search_s": j["search_s"]}, j["pen"]


def run_reference(args, rank):
    if rank != 0:
        return
    scene, tmpls = make_workload(0)
    vals, last = [], None
    for i in range(args.warmup + args.steps):
        last, _ = cpu_baseline(scene, tmpls)
        if i >= args.warmup:
            vals.append(last["value"])
    value = float(np.mean(vals))
    last["value"] = value
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * N_TMPL / value, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": CONFIG, "cpu_baseline": last,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), file=_JSON_OUT, flush=True)


_JSON_OUT = sys.stdout


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the config-4 / config-5 / strong-scaling legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the top-10 and a seeded sample of the DT3 map of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 timed path")
    # stdout carries exactly one JSON line: libraries that print to fd 1 (NCCL's version banner) are sent to stderr
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import ctypes as C

    import torch
    import torch.distributed as dist
    import openfdcm_b200 as fdcm
    from openfdcm_b200 import distributed as fd
    from tests.util import plant_instances, synth_scene, synth_templates

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    comm = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        comm = fd.Communicator.from_torch(local_rank)     # also bounds this rank's host pool to cores / world
    # a real (non-default) stream shared by torch and the library: the CUDA events of timed() are recorded on the stream the
    # kernels are launched on (torch's default stream has the null handle, which the library reads as "use your own stream")
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    fdcm.set_stream(local_rank, stream.cuda_stream)
    L = fdcm.lib()

    scene, tmpls = make_workload(rank)
    searcher, optimizer, penalty = fdcm.DefaultSearch(MAX_T, MAX_S), fdcm.BatchOptimize(BATCH), fdcm.ExponentialPenalty(TAU)
    params = fdcm.Dt3CudaParameters(DEPTH, COEFF, PADDING, fdcm.distance.L2, device=local_rank)
    base = rank * N_TMPL

    # pinned host copies of the inputs for the end-to-end arm
    flat, off = fdcm._pack(tmpls)
    h_lines = torch.from_numpy(flat).pin_memory()
    h_off = torch.from_numpy(off).pin_memory()
    h_scene = torch.from_numpy(fdcm._records(scene)).pin_memory()
    h2d = h_lines.numel() * 4 + h_off.numel() * 4 + h_scene.numel() * 4
    d2h = TOP_K * 32

    fm = fdcm.build_cuda_featuremap(scene, params)
    tset = fdcm.TemplateSet(tmpls, device=local_rank)

    def search_resident(ts, idx_base):
        if comm is not None:
            return comm.search_topk(fm, ts, None, searcher, optimizer, penalty, TOP_K, idx_base)
        return fdcm.search_topk(fm, ts, None, searcher, optimizer, penalty, TOP_K, idx_base)

    def step_resident():
        fm.rerun(wait=False)   # queued; the search below is stream-ordered after it and ends with the only host sync of the step
        return search_resident(tset, base)

    def step_e2e():
        fdcm.check(L.fdcm_dt3_rebuild_async(fm._h, h_scene.data_ptr(), h_scene.shape[0]))   # host prep of the search overlaps the build
        out = np.zeros(TOP_K, fdcm.MATCH_DTYPE)
        n = C.c_int64(0)
        p = fdcm._lib.SearchParams(MAX_T, MAX_S, BATCH, penalty.kind, penalty.tau, TOP_K, base, 0, 0.0, 0.0, 0.0, 0.0)
        if comm is None:
            fdcm.check(L.fdcm_search_host(fm._h, h_lines.data_ptr(), h_off.data_ptr(), N_TMPL, None, fdcm._lib.FDCM_SCENE_RESIDENT,
                                          C.byref(p), fdcm.ptr(out), TOP_K, C.byref(n)))
        else:   # host templates of this rank's shard in, the merged global top-10 out
            fdcm.check(L.fdcm_comm_search_host_topk(comm._h, fm._h, h_lines.data_ptr(), h_off.data_ptr(), N_TMPL, None,
                                                    fdcm._lib.FDCM_SCENE_RESIDENT, C.byref(p), fdcm.ptr(out), TOP_K, C.byref(n)))
        return out[: n.value]

    def timed(fn, steps, warmup, profile=False):
        for _ in range(warmup):
            fn()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        if profile:
            fdcm.profile(True, reset=True)
        launches0 = fdcm.kernel_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        res = None
        for _ in range(steps):
            res = fn()
        e1.record(stream)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        launches = fdcm.kernel_launch_count() - launches0
        prof = fdcm.profile_report() if profile else None
        if profile:
            fdcm.profile(False)
        return float(ms.item()), res, launches, prof

    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_res, top_res, launches, prof = timed(step_resident, args.steps, args.warmup, profile=True)
    stats = fm.last_search_stats()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, fm, top_res)
    ms_e2e, top_e2e, _, _ = timed(step_e2e, args.steps, args.warmup)
    clocks = sampler.stop()

    # ---- strong scaling: the 5000 templates of config 3 split over the ranks (same step otherwise) ----
    strong = None
    if not args.no_extras:
        base_set = tmpls if rank == 0 else synth_templates(N_TMPL, N_TMPL_LINES, SCENE_W, seed=3001)
        sb, se = fd.shard_range(N_TMPL, rank, world)
        strong_set = fdcm.TemplateSet(base_set[sb:se], device=local_rank)

        def step_strong():
            fm.rerun(wait=False)
            return search_resident(strong_set, sb)

        ms_strong, top_strong, _, _ = timed(step_strong, max(5, args.steps // 2), 3)
        ms_strong /= max(5, args.steps // 2)
        strong = {"value": N_TMPL / (ms_strong / 1e3), "unit": UNIT, "ms_per_step": ms_strong, "templates_total": N_TMPL,
                  "templates_per_gpu": se - sb, "top10": [[int(r["tmpl_idx"]), float(r["score"])] for r in top_strong]}
        del strong_set

    # ---- DT3 build ms (config 2 metric) per distance, kernels only, same 1080p scene ----
    build_ms, build_kernels = {}, {}
    for name, d in (("L2", fdcm.distance.L2), ("L2_SQUARED", fdcm.distance.L2_SQUARED), ("L1", fdcm.distance.L1)):
        m2 = fm if name == "L2" else fdcm.build_cuda_featuremap(
            scene, fdcm.Dt3CudaParameters(DEPTH, COEFF, PADDING, d, device=local_rank))
        # ten builds queued back to back on the stream, one host sync at the end: device time of a build, no per-build host round trip
        t, _, _, pr = timed(lambda: m2.rerun(wait=False), 10, 3, profile=(name == "L2"))
        build_ms[name] = t / 10
        if pr:
            build_kernels = pr
        if m2 is not fm:
            del m2

    # ---- config 5: multi-scene batch, scenes sharded over the ranks (s % world), 1000 templates, pipelined builds ----
    config5 = None
    if not args.no_extras:
        n_sc = 16 * world                                        # 16 scenes per GPU per batch (config 5: 64 scenes on 8 GPUs -> 8 each)
        t5 = synth_templates(1000, N_TMPL_LINES, SCENE_W, seed=5100)
        mine = fd.shard_scenes(n_sc, rank, world)
        sc5 = [plant_instances(synth_scene(SCENE_W, SCENE_H, N_SCENE, seed=5000 + s), t5, SCENE_W, SCENE_H, seed=5200 + s) for s in mine]
        set5 = fdcm.TemplateSet(t5, device=local_rank)
        batch = fdcm.SceneBatch(params)
        ms5, res5, _, _ = timed(lambda: batch.search_topk(sc5, set5, searcher, optimizer, penalty, TOP_K), 2, 1)
        ms5 /= 2
        fm_seq = fdcm.build_cuda_featuremap(sc5[0], params)

        def sequential():
            out = []
            for s in sc5:
                fm_seq.rebuild(s)
                out.append(fdcm.search_topk(fm_seq, set5, None, searcher, optimizer, penalty, TOP_K))
            return out

        ms5s, res5s, _, _ = timed(sequential, 2, 1)
        ms5s /= 2
        config5 = {"scenes_per_s": n_sc / (ms5 / 1e3), "templates_per_s": n_sc * 1000 / (ms5 / 1e3), "ms_per_batch": ms5, "scenes": n_sc,
                   "scenes_per_gpu": len(mine), "templates": 1000, "sequential_ms_per_batch": ms5s,
                   "pipelined_equals_sequential": bool(all(np.array_equal(a, b) for a, b in zip(res5, res5s))),
                   "note": "host scenes in, top-10 per scene out; build of scene s+1 on a second stream under the search of scene s"}
        del batch, set5, fm_seq

    # ---- config 4: wide combinatorial search on the 4K scene (rank 0 only: single-GPU number) ----
    config4 = None
    if not args.no_extras and rank == 0:
        t4 = synth_templates(2000, 60, 3840, seed=4001)
        sc4 = plant_instances(synth_scene(3840, 2160, 5000, seed=4000), t4, 3840, 2160, seed=4002)
        fm4 = fdcm.build_cuda_featuremap(sc4, fdcm.Dt3CudaParameters(DEPTH, COEFF, PADDING, fdcm.distance.L2, device=local_rank))
        set4 = fdcm.TemplateSet(t4, device=local_rank)
        s4, o4 = fdcm.DefaultSearch(16, 16), fdcm.BatchOptimize(20)
        torch.cuda.synchronize()
        reps = 3
        fm4.rerun()
        t0 = time.perf_counter()
        for _ in range(reps):
            fm4.rerun()
        tb4 = (time.perf_counter() - t0) / reps * 1e3
        fdcm.search_topk(fm4, set4, None, s4, o4, penalty, TOP_K)
        t0 = time.perf_counter()
        for _ in range(reps):
            top4 = fdcm.search_topk(fm4, set4, None, s4, o4, penalty, TOP_K)
        ts4 = (time.perf_counter() - t0) / reps * 1e3
        st4 = fm4.last_search_stats()
        config4 = {"templates_per_s": 2000 / ((tb4 + ts4) / 1e3), "build_ms": tb4, "search_ms": ts4, "map_side": fm4.width,
                   "hypotheses": st4["n_hypotheses"], "lookups_per_s": st4["n_lookups"] / (ts4 / 1e3),
                   "exact_dt_path": int(fm4.info.exact_dt_path), "top1": [int(top4[0]["tmpl_idx"]), float(top4[0]["score"])],
                   "note": "side 5760 > 2897: the distance transform runs the literal float kernels (parity-tested, not tuned)"}
        del fm4, set4

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    ms_step = ms_res / args.steps
    value = world * N_TMPL / (ms_step / 1e3)
    e2e_value = world * N_TMPL / (ms_e2e / args.steps / 1e3)
    same_arms = top_res is not None and len(top_res) == TOP_K and np.array_equal(top_res, top_e2e)

    # ---- parity: the benched top-10 against the CPU oracle on the same (global) template set, outside the timed region ----
    cpu, parity = None, None
    if not args.no_cpu_baseline:
        all_t = list(tmpls)
        for r in range(1, world):
            all_t += synth_templates(N_TMPL, N_TMPL_LINES, SCENE_W, seed=3001 + 17 * r)
        if world == 1:
            cpu, pen = cpu_baseline(scene, all_t)
        else:
            pen = oracle_job(scene, all_t)["pen"]
        want = oracle_top(pen, TOP_K)
        parity = bool(np.array_equal(top_res, want) and same_arms)
        if strong is not None:
            want_s = want if world == 1 else oracle_top(oracle_job(scene, list(tmpls))["pen"], TOP_K)
            got_s = np.array([(a, b) for a, b in strong["top10"]], dtype=[("i", "<i4"), ("s", "<f4")])
            strong["parity"] = bool(np.array_equal(got_s["i"], want_s["tmpl_idx"]) and np.array_equal(got_s["s"], want_s["score"]))

    # ---- rooflines ----
    peak, peak_kind = measured_peak()
    traffic = load_traffic()
    n_px_bytes = float(DEPTH) * fm.width * fm.height * 4
    # search: compulsory bytes = 4 B per map lookup + 32 B per emitted match (the 32 B/lookup sector model of SURVEY 8(d)
    # over-counts 5x because neighbouring candidate translations share sectors: it is kept as `sector_model_gbs` only)
    algo = {"search": 4.0 * stats["n_lookups"] + 32.0 * stats["n_valid"]}
    kernels = {}
    for name, v in prof.items():
        avg_ms = v["total_ms"] / max(1, v["launches"])
        by = algo.get(name, v["bytes_per_launch"])
        tr = traffic.get(name, {}) if isinstance(traffic.get(name), dict) else {}
        kernels[name] = {"avg_ms": avg_ms, "launches": v["launches"], "algorithmic_bytes": by,
                         "achieved_gbs": (by / (avg_ms * 1e-3) / 1e9) if avg_ms > 0 else None,
                         "dram_bytes": tr.get("dram_bytes"), "l2_bytes": tr.get("l2_bytes")}
    dom = max(kernels, key=lambda k: kernels[k]["avg_ms"] * kernels[k]["launches"])
    kd = kernels[dom]
    roofline = {"kernel": dom, "bound": "hbm", "achieved": kd["achieved_gbs"], "peak": peak, "peak_kind": peak_kind, "unit": "GB/s",
                "frac": (kd["achieved_gbs"] or 0.0) / peak, "traffic": kd["dram_bytes"],
                "share_of_step": kd["avg_ms"] * kd["launches"] / ms_res,
                "dram_gbs": (kd["dram_bytes"] / (kd["avg_ms"] * 1e-3) / 1e9) if kd["dram_bytes"] and kd["avg_ms"] > 0 else None,
                "dram_frac": (kd["dram_bytes"] / (kd["avg_ms"] * 1e-3) / 1e9 / peak) if kd["dram_bytes"] and kd["avg_ms"] > 0 else None,
                "l2_gbs": (kd["l2_bytes"] / (kd["avg_ms"] * 1e-3) / 1e9) if kd["l2_bytes"] and kd["avg_ms"] > 0 else None,
                "l2_frac": (kd["l2_bytes"] / (kd["avg_ms"] * 1e-3) / 1e9 / L2_PEAK_GBS) if kd["l2_bytes"] and kd["avg_ms"] > 0 else None,
                "note": "achieved = algorithmic bytes / live kernel time (CUDA events inside the timed region); traffic / l2_bytes = "
                        "DRAM and L2 bytes per launch of the ncu --set full capture in profiles/ (traffic.json)"}
    if dom == "search":
        roofline["sector_model_gbs"] = 32.0 * stats["n_lookups"] / (kd["avg_ms"] * 1e-3) / 1e9
        roofline["sector_efficiency"] = 4.0 / 32.0
    bk = {}
    for name, v in build_kernels.items():
        avg_ms = v["total_ms"] / max(1, v["launches"])
        tr = traffic.get(name, {}) if isinstance(traffic.get(name), dict) else {}
        bk[name] = {"avg_ms": avg_ms, "algorithmic_bytes": v["bytes_per_launch"], "dram_bytes": tr.get("dram_bytes"),
                    "dram_frac": (tr["dram_bytes"] / (avg_ms * 1e-3) / 1e9 / peak) if tr.get("dram_bytes") and avg_ms > 0 else None}
    build_dram = sum(v["dram_bytes"] for v in bk.values() if v["dram_bytes"])
    build_roofline = {"bound": "hbm", "algorithmic_bytes_5N": 5 * n_px_bytes, "ms_L2": build_ms["L2"],
                      "achieved": 5 * n_px_bytes / (build_ms["L2"] * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                      "frac": 5 * n_px_bytes / (build_ms["L2"] * 1e-3) / 1e9 / peak,
                      "traffic": build_dram or None,
                      "dram_frac": (build_dram / (build_ms["L2"] * 1e-3) / 1e9 / peak) if build_dram else None,
                      "kernels": bk,
                      "note": "SURVEY 8(d) model: 5 N bytes, N = depth x H x W x 4 B; the fused fill + propagate keeps the distance "
                              "transform planes out of HBM, so the real DRAM traffic (traffic) is about 3 N"}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": CONFIG,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches, "clocks": clocks, "parity": parity, "resident_equals_e2e": bool(same_arms),
            "roofline": roofline, "kernels": kernels,
            "dt3_build_ms": build_ms, "build_roofline": build_roofline,
            "strong_scaling": strong, "config4": config4, "config5": config5,
            "search_stats": stats, "lookups_per_s": stats["n_lookups"] / (kernels["search"]["avg_ms"] * 1e-3),
            "top10": [[int(r["tmpl_idx"]), float(r["score"])] for r in top_res]}
    if cpu is not None:
        line["cpu_baseline"] = cpu
        search_ms = sum(kernels[k]["avg_ms"] for k in ("search_order", "search", "topk") if k in kernels)
        line["vs_cpu"] = {"build_ratio": cpu["build_s"] * 1e3 / build_ms["L2"], "search_ratio": cpu["search_s"] * 1e3 / search_ms,
                          "step_ratio": (cpu["build_s"] + cpu["search_s"]) * 1e3 / ms_step,
                          "note": "CPU oracle on the box's host cores (cores above) vs device kernel times; the build ratio is "
                                  "dominated by the reference's single-threaded propagateOrientation"}
    print(json.dumps(line), file=_JSON_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
