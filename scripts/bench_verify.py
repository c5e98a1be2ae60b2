"""Cost and separation of the match verification (EdgeCoverage, match_coverage, verify=), one JSON line:
python scripts/bench_verify.py [reps]

Cost (every timed call ends in a device synchronisation: 3 warm-ups, then the median of `reps` calls):
- dilation: the config-2 map (the 1920 x 1080 scene of bench.py, padding 1.5: 2880^2 x 30 planes, a 31 MB edge mask),
  coverage_dilate kernel time from profile_report(), the cache defeated by alternating radius 2 and 3;
- match_coverage of k = 10 and k = 5000 matches of that map at the defaults (dilation cached);
- config 3 (bench.py: 5000 templates x 40 lines, DefaultSearch(4, 4), BatchOptimize(10), ExponentialPenalty(1.5),
  160 000 records), search_topk k = 10 without and with verify=EdgeCoverage(min_coverage=0.5);
- real assets (the first scene of each object, every template, padding 1.0), search_dense at the default DenseSearch() with
  DistinctMatches(max_per_template=1), k = 10, without and with verify=EdgeCoverage(min_coverage=0.5); the record count
  per scene is computed from the shapes (templates x rotations x cells), not measured.

Separation: the planted-noise workload of scripts/bench_dense.py (200 templates x 30 lines, 40 planted in a 1280 x 720
scene with +-0.5 px end-point noise), with the planted lines intact and cut.  For the k = 200, max_per_template = 1 results
of search_topk (DefaultSearch(4, 10)) and search_dense (defaults): the coverage quantiles of the matches within 10 px (anchor)
and 0.2 rad of a planted pose ("true") and of all others ("other"), and, for search_topk, the found / false
counts with verify=EdgeCoverage(min_coverage=m) for m in {0, 0.3, 0.5, 0.7, 0.9} (the filtered search_dense is not run on
this workload: its map holds about 2 x 10^8 dense records).  The verified real-asset dense call is timed once after one
warm-up."""
import glob
import json
import math
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import openfdcm_b200 as fdcm  # noqa: E402
from scripts.bench_dense import cut  # noqa: E402
from scripts.bench_select import gpu_info, median_ms  # noqa: E402
from tests.util import apply_transform, plant_instances, synth_scene, synth_templates  # noqa: E402

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 5
PEN = fdcm.ExponentialPenalty(1.5)
SEL = fdcm.DistinctMatches(max_per_template=1)
COV = fdcm.EdgeCoverage()
FILTER = fdcm.EdgeCoverage(min_coverage=0.5)
LEVELS = (0.0, 0.3, 0.5, 0.7, 0.9)


def config3():
    tmpls = synth_templates(5000, 40, 1920, seed=3001)
    scene = plant_instances(synth_scene(1920, 1080, 2000, seed=3000), tmpls, 1920, 1080, seed=3002)
    return scene, tmpls


def cost(reps):
    scene, tmpls = config3()
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    ts = fdcm.TemplateSet(tmpls)
    args = (fm, ts, scene, fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), PEN)
    out = {"map": [fm.width, fm.height, fm.depth], "mask_mb": round(fm.depth * fm.height * (-(-fm.width // 32) * 4) / 1e6, 1)}
    m5000 = fdcm.search_topk(*args, k=5000)
    one = m5000[:1]
    fdcm.match_coverage(fm, ts, one, fdcm.EdgeCoverage(3))
    fdcm.profile(True, reset=True)
    for i in range(2 * reps):
        fdcm.match_coverage(fm, ts, one, fdcm.EdgeCoverage(2 + i % 2))
    rep = fdcm.profile_report()
    fdcm.profile(False, reset=True)
    out["dilate_ms"] = round(rep["coverage_dilate"]["total_ms"] / rep["coverage_dilate"]["launches"], 4)
    for k in (10, 5000):
        out[f"match_coverage_k{k}_ms"] = round(median_ms(lambda: fdcm.match_coverage(fm, ts, m5000[:k], COV), reps), 3)
    out["config3_records"] = 5000 * 2 * 4 * 4
    out["config3_search_topk_ms"] = round(median_ms(lambda: fdcm.search_topk(*args, k=10), reps), 3)
    out["config3_search_topk_verify_ms"] = round(median_ms(lambda: fdcm.search_topk(*args, k=10, verify=FILTER), reps), 3)
    fdcm.profile(True, reset=True)
    fdcm.search_topk(*args, k=10, verify=FILTER)
    rep = fdcm.profile_report()
    fdcm.profile(False, reset=True)
    out["config3_kernels_ms"] = {k: round(v["total_ms"], 4) for k, v in rep.items()}
    return out


def dense_records(fm, n_tmpl, d):
    W, H = fm.width, fm.height
    nx, ny = (W - 1) // d.stride + 1, (H - 1) // d.stride + 1
    cell = min(d.cell, max(nx, ny))
    return n_tmpl * d.rotations * (-(-nx // cell)) * (-(-ny // cell))


def real_assets(reps):
    assets = os.path.join(ROOT, "tests", "golden", "real_assets")
    d = fdcm.DenseSearch()
    out = {}
    for obj in ("obj_01", "obj_02", "obj_03", "obj_04"):
        tm = sorted(glob.glob(os.path.join(assets, obj, "templates", "*.tmpl")), key=lambda q: int(os.path.basename(q)[9:-5]))
        sc = sorted(glob.glob(os.path.join(assets, obj, "scene_*", "camera_0.scene")), key=lambda q: int(os.path.basename(os.path.dirname(q))[6:]))
        tmpls = [fdcm.read(q) for q in tm]
        ts = fdcm.TemplateSet(tmpls)
        fm = fdcm.build_cuda_featuremap(fdcm.read(sc[0]), fdcm.Dt3CudaParameters(30, 5.0, 1.0))
        plain = median_ms(lambda: fdcm.search_dense(fm, ts, d, PEN, 10, select=SEL), reps)
        fdcm.search_dense(fm, ts, d, PEN, 10, select=SEL, verify=FILTER)   # (one warm-up: a verified call scores every record)
        t0 = time.perf_counter()
        fdcm.search_dense(fm, ts, d, PEN, 10, select=SEL, verify=FILTER)
        ver = (time.perf_counter() - t0) * 1e3
        out[obj] = {"templates": len(tmpls), "records": dense_records(fm, len(tmpls), d), "search_dense_ms": round(plain, 3),
                    "search_dense_verify_ms": round(ver, 3)}
    return out


def planted(cut_lines):
    w, h = 1280, 720
    tmpls = synth_templates(200, 30, w, seed=71)
    rng = np.random.default_rng(72)
    crng = np.random.default_rng(74)
    truth, extra = {}, []
    for q in range(40):
        th = rng.uniform(-math.pi, math.pi)
        T = np.array([[math.cos(th), -math.sin(th), rng.uniform(0.15 * w, 0.85 * w)],
                      [math.sin(th), math.cos(th), rng.uniform(0.15 * h, 0.85 * h)]])
        truth[q] = T
        inst = apply_transform(tmpls[q], T) + rng.uniform(-0.5, 0.5, (4, tmpls[q].shape[1])).astype(np.float32)
        extra.append(cut(inst, crng) if cut_lines else inst)
    scene = np.ascontiguousarray(np.concatenate([synth_scene(w, h, 300, seed=73)] + extra, axis=1), np.float32)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    ts, anchors = fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls)
    k = len(tmpls)

    def is_true(m):
        t = int(m["tmpl_idx"])
        if t not in truth:
            return False
        T = np.asarray(m["transform"], np.float64).reshape(2, 3)
        a = np.append(anchors[t].astype(np.float64), 1.0)
        rot = abs(math.remainder(math.atan2(T[1, 0], T[0, 0]) - math.atan2(truth[t][1, 0], truth[t][0, 0]), 2 * math.pi))
        return float(np.hypot(*(T @ a - truth[t] @ a))) < 10 and rot < 0.2

    def quantiles(v):
        v = v[~np.isnan(v)]
        return [round(float(x), 3) for x in np.quantile(v, [0.0, 0.1, 0.5, 0.9, 1.0])] if len(v) else []

    out = {"planted": len(truth)}
    calls = {"search_topk": lambda cov: fdcm.search_topk(fm, ts, None, fdcm.DefaultSearch(4, 10), fdcm.BatchOptimize(10), PEN, k=k,
                                                          select=SEL, verify=cov),
             "search_dense": lambda cov: fdcm.search_dense(fm, ts, fdcm.DenseSearch(), PEN, k, select=SEL, verify=cov)}
    for name, call in calls.items():
        base = call(None)
        flags = np.array([is_true(m) for m in base], bool)
        c = fdcm.match_coverage(fm, ts, base, COV)
        res = {"coverage_true_q0_10_50_90_100": quantiles(c[flags]), "coverage_other_q0_10_50_90_100": quantiles(c[~flags]),
               "n_true": int(flags.sum()), "n_other": int((~flags).sum())}
        if name == "search_dense":   # about 2 x 10^8 records on this map: the filtered dense calls are not run
            out[name] = res
            continue
        for lv in LEVELS:
            got = call(fdcm.EdgeCoverage(min_coverage=lv))
            f = [is_true(m) for m in got]
            res[f"min_{lv}"] = {"found": int(sum(f)), "false": int(len(f) - sum(f))}
        out[name] = res
    return out


def main():
    res = {"gpu": gpu_info(), "reps": REPS, "coverage": repr(COV), "filter": repr(FILTER), "cost": cost(REPS),
           "real_assets_dense": real_assets(REPS), "planted": {"intact_lines": planted(False), "cut_lines": planted(True)}}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
