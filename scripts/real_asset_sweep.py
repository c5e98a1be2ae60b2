"""End-to-end time per scene on the reference's real assets with the notebook's parameters
(notebooks/pose_extimation_example.ipynb:216-244: DefaultSearch(4,10), BatchOptimize(10), depth 30, coeff 5, padding 1.0,
L2, ExponentialPenalty(1.5); "Should run at 22 FPS on an i7-14700"): host lines in -> build + search + penalize + sorted
top-10 out, per scene, for the 40 scenes; next to the CPU oracle timed on this box's host cores on the same scenes.
usage: python scripts/real_asset_sweep.py out.json"""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import openfdcm_b200 as fdcm
from oracle import fdcm_oracle as orc
from tests.helpers import load_object

out = {"parameters": "DefaultSearch(4,10), BatchOptimize(10), depth 30, coeff 5, padding 1.0, L2, ExponentialPenalty(1.5), top-10",
       "reference_claim": "22 FPS (45 ms / scene) on an i7-14700, notebooks/pose_extimation_example.ipynb:244", "objects": {}}
s_, o_, p_ = fdcm.DefaultSearch(4, 10), fdcm.BatchOptimize(10), fdcm.ExponentialPenalty(1.5)
params = fdcm.Dt3CudaParameters(30, 5.0, 1.0, fdcm.distance.L2)
gpu_all, cpu_all, batch_all = [], [], []
for obj in ("obj_01", "obj_02", "obj_03", "obj_04"):
    tmpls, scenes = load_object(obj)
    tset = fdcm.TemplateSet(tmpls)
    fm = fdcm.build_cuda_featuremap(scenes[0], params)
    for rep in range(3):                       # per-scene calls: rebuild (host lines in) + fused search / penalty / top-10
        ts = []
        for sc in scenes:
            t0 = time.perf_counter()
            fm.rebuild(sc, wait=False)
            top = fdcm.search_topk(fm, tset, None, s_, o_, p_, 10)
            ts.append((time.perf_counter() - t0) * 1e3)
    batch = fdcm.SceneBatch(params)
    batch.search_topk(scenes, tset, s_, o_, p_, 10)
    t0 = time.perf_counter()
    batch.search_topk(scenes, tset, s_, o_, p_, 10)
    tb = (time.perf_counter() - t0) * 1e3 / len(scenes)
    tc = []
    for sc in scenes[:3]:                      # CPU oracle, all host threads, the notebook's four calls
        t0 = time.perf_counter()
        c = orc.Dt3Cpu(sc, 30, 5.0, 1.0)
        pen = orc.sort_matches(orc.penalize(1, 1.5, c.search(tmpls, sc, 4, 10, batch=10), orc.template_lengths(tmpls)))
        tc.append((time.perf_counter() - t0) * 1e3)
    out["objects"][obj] = {"templates": len(tmpls), "scenes": len(scenes), "gpu_ms_per_scene": float(np.mean(ts)),
                           "gpu_batch_ms_per_scene": tb, "cpu_oracle_ms_per_scene": float(np.mean(tc)), "map_side": fm.width}
    gpu_all += ts
    cpu_all += tc
    batch_all.append(tb)
out["gpu_ms_per_scene"] = float(np.mean(gpu_all))
out["gpu_fps"] = 1e3 / out["gpu_ms_per_scene"]
out["gpu_batch_ms_per_scene"] = float(np.mean(batch_all))
out["cpu_oracle_ms_per_scene"] = float(np.mean(cpu_all))
out["cpu_cores"] = orc.hardware_concurrency()
json.dump(out, open(sys.argv[1] if len(sys.argv) > 1 else "gpurun_out/real_assets.json", "w"), indent=1)
print(json.dumps(out))
