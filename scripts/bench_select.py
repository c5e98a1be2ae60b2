"""Cost of the distinct top-K (search_topk(select=DistinctMatches(...))) against the plain top-10, one JSON line:
python scripts/bench_select.py [reps]

Workloads: config 3 (5000 templates x 40 lines vs one 1080p scene, padding 1.5, DefaultSearch(4,4), BatchOptimize(10),
ExponentialPenalty(1.5); the map is built once, every timed call is the search -> penalty -> selection on the resident
scene) and the 40 real-asset scenes (the notebook's parameters: DefaultSearch(4,10), padding 1.0).  Every timed call
ends in a device synchronisation (the call downloads its result): 3 warm-ups, then the median of `reps` calls.  Also
reported: the per-kernel split of profile_report() in a separate profiled pass, the distinct templates of every top-10
of the real assets, and the GPU name / power limit of this run."""
import glob
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import openfdcm_b200 as fdcm  # noqa: E402
from tests.util import plant_instances, synth_scene, synth_templates  # noqa: E402

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 30
DM = fdcm.DistinctMatches
VARIANTS = {   # name -> (k, select)
    "plain_k10": (10, None),
    "k10_cap1": (10, DM(max_per_template=1)),
    "k5000_cap1": (5000, DM(max_per_template=1)),
    "k10_cap2_r10_a0.26": (10, DM(max_per_template=2, radius=10.0, max_angle=0.26)),
    "k10_across_r10": (10, DM(radius=10.0, across_templates=True)),
    "k100_across_r10": (100, DM(radius=10.0, across_templates=True)),
}


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                               text=True, timeout=30).stdout.strip()
    except Exception as e:   # the number is still reported, without its power limit
        limit = f"unavailable ({e})"
    return {"name": name, "power_limit": limit}


def median_ms(fn, reps):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def kernel_split(fn, reps):
    fdcm.profile(True, reset=True)
    for _ in range(reps):
        fn()
    rep = fdcm.profile_report()
    fdcm.profile(False)
    return {k: round(v["total_ms"] / max(1, v["launches"]), 4) for k, v in rep.items()}


def config3(reps):
    tmpls = synth_templates(5000, 40, 1920, seed=3001)
    scene = plant_instances(synth_scene(1920, 1080, 2000, seed=3000), tmpls, 1920, 1080, seed=3002)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    ts = fdcm.TemplateSet(tmpls)
    args = (fm, ts, None, fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), fdcm.ExponentialPenalty(1.5))
    out = {}
    for name, (k, sel) in VARIANTS.items():
        call = lambda: fdcm.search_topk(*args, k=k, select=sel)  # noqa: E731
        top = call()
        out[name] = {"ms": round(median_ms(call, reps), 4), "kernels_ms": kernel_split(call, 10), "n": int(len(top)),
                     "distinct_templates_top10": len(set(top["tmpl_idx"][:10].tolist()))}
    base = out["plain_k10"]["ms"]
    for name in VARIANTS:
        out[name]["extra_ms_vs_plain"] = round(out[name]["ms"] - base, 4)
    return out


def real_assets(reps):
    assets = os.path.join(ROOT, "tests", "golden", "real_assets")
    s, o, p = fdcm.DefaultSearch(4, 10), fdcm.BatchOptimize(10), fdcm.ExponentialPenalty(1.5)
    times = {name: [] for name in VARIANTS if VARIANTS[name][0] <= 100}
    distinct = {"plain_k10": {}, "k10_cap1": {}}
    for obj in ("obj_01", "obj_02", "obj_03", "obj_04"):
        tm = sorted(glob.glob(os.path.join(assets, obj, "templates", "*.tmpl")), key=lambda q: int(os.path.basename(q)[9:-5]))
        sc = sorted(glob.glob(os.path.join(assets, obj, "scene_*", "camera_0.scene")), key=lambda q: int(os.path.basename(os.path.dirname(q))[6:]))
        ts = fdcm.TemplateSet([fdcm.read(q) for q in tm])
        for name in distinct:
            distinct[name][obj] = []
        for path in sc:
            fm = fdcm.build_cuda_featuremap(fdcm.read(path), fdcm.Dt3CudaParameters(30, 5.0, 1.0))
            for name in times:
                k, sel = VARIANTS[name]
                call = lambda: fdcm.search_topk(fm, ts, None, s, o, p, k=k, select=sel)  # noqa: E731
                times[name].append(median_ms(call, reps))
                if name in distinct:
                    distinct[name][obj].append(len(set(call()["tmpl_idx"].tolist())))
    return {"ms_median_over_scenes": {n: round(float(np.median(v)), 4) for n, v in times.items()},
            "distinct_templates_top10": distinct}


def main():
    res = {"gpu": gpu_info(), "reps": REPS, "config3": config3(REPS), "real_assets": real_assets(REPS)}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
