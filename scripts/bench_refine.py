"""Cost and effect of the pose refinement (search_topk(refine=PoseRefinement())), one JSON line:
python scripts/bench_refine.py [reps]

Workloads: config 3 (5000 templates x 40 lines vs one 1080p scene, padding 1.5, DefaultSearch(4,4), BatchOptimize(10),
ExponentialPenalty(1.5); the map is built once, every timed call is the search -> penalty -> selection -> refinement on the
resident scene): the plain top-10 and one match per template at k = 5000, each with and without the default refinement
(k = 10 is the latency-bound case, k = 5000 the throughput case).  The 40 real-asset scenes (the notebook's parameters:
DefaultSearch(4,10), padding 1.0): the median over scenes of k = 10, max_per_template = 1 with and without refinement.
Every timed call ends in a device synchronisation (the call downloads its result): 3 warm-ups, then the median of `reps`
calls.  Also reported: the per-kernel split of profile_report() in a separate profiled pass, the anchor and rotation
errors before and after refinement of instances planted with +-0.5 px end-point noise, the errors after refinement started at
the exact pose of noise-free planted instances, and the GPU name / power limit."""
import json
import math
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import openfdcm_b200 as fdcm  # noqa: E402
from scripts.bench_select import gpu_info, kernel_split, median_ms  # noqa: E402
from tests.util import apply_transform, plant_instances, synth_scene, synth_templates  # noqa: E402

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 30
R = fdcm.PoseRefinement()
VARIANTS = {   # name -> (k, select, refine)
    "plain_k10": (10, None, None),
    "plain_k10_refine": (10, None, R),
    "k5000_cap1": (5000, fdcm.DistinctMatches(max_per_template=1), None),
    "k5000_cap1_refine": (5000, fdcm.DistinctMatches(max_per_template=1), R),
}


def config3(reps):
    tmpls = synth_templates(5000, 40, 1920, seed=3001)
    scene = plant_instances(synth_scene(1920, 1080, 2000, seed=3000), tmpls, 1920, 1080, seed=3002)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    ts = fdcm.TemplateSet(tmpls)
    args = (fm, ts, None, fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), fdcm.ExponentialPenalty(1.5))
    out = {}
    for name, (k, sel, ref) in VARIANTS.items():
        call = lambda: fdcm.search_topk(*args, k=k, select=sel, refine=ref)  # noqa: E731
        top = call()
        out[name] = {"ms": round(median_ms(call, reps), 4), "kernels_ms": kernel_split(call, 10), "n": int(len(top))}
    for name in ("plain_k10", "k5000_cap1"):
        out[name + "_refine"]["extra_ms"] = round(out[name + "_refine"]["ms"] - out[name]["ms"], 4)
    return out


def real_assets(reps):
    import glob
    assets = os.path.join(ROOT, "tests", "golden", "real_assets")
    s, o, p = fdcm.DefaultSearch(4, 10), fdcm.BatchOptimize(10), fdcm.ExponentialPenalty(1.5)
    sel = fdcm.DistinctMatches(max_per_template=1)
    times = {"k10_cap1": [], "k10_cap1_refine": []}
    for obj in ("obj_01", "obj_02", "obj_03", "obj_04"):
        tm = sorted(glob.glob(os.path.join(assets, obj, "templates", "*.tmpl")), key=lambda q: int(os.path.basename(q)[9:-5]))
        sc = sorted(glob.glob(os.path.join(assets, obj, "scene_*", "camera_0.scene")), key=lambda q: int(os.path.basename(os.path.dirname(q))[6:]))
        ts = fdcm.TemplateSet([fdcm.read(q) for q in tm])
        for path in sc:
            fm = fdcm.build_cuda_featuremap(fdcm.read(path), fdcm.Dt3CudaParameters(30, 5.0, 1.0))
            for name, ref in (("k10_cap1", None), ("k10_cap1_refine", R)):
                times[name].append(median_ms(lambda: fdcm.search_topk(fm, ts, None, s, o, p, k=10, select=sel, refine=ref), reps))
    med = {n: round(float(np.median(v)), 4) for n, v in times.items()}
    return {"n_scenes": len(times["k10_cap1"]), "ms_median_over_scenes": med,
            "extra_ms": round(med["k10_cap1_refine"] - med["k10_cap1"], 4)}


def planted_noise_instances():
    """200 templates, the first 40 planted at random poses with +-0.5 px end-point noise among 300 clutter lines:
    (templates, {template: planted 2x3 pose}, scene)."""
    w, h = 1280, 720
    tmpls = synth_templates(200, 30, w, seed=71)
    rng = np.random.default_rng(72)
    truth, extra = {}, []
    for q in range(40):
        th = rng.uniform(-math.pi, math.pi)
        T = np.array([[math.cos(th), -math.sin(th), rng.uniform(0.15 * w, 0.85 * w)],
                      [math.sin(th), math.cos(th), rng.uniform(0.15 * h, 0.85 * h)]])
        truth[q] = T
        extra.append(apply_transform(tmpls[q], T) + rng.uniform(-0.5, 0.5, (4, tmpls[q].shape[1])).astype(np.float32))
    scene = np.ascontiguousarray(np.concatenate([synth_scene(w, h, 300, seed=73)] + extra, axis=1), np.float32)
    return tmpls, truth, scene


def planted_noise():
    """Mean anchor (px) and rotation (rad) errors of the found planted instances, before and after refinement."""
    tmpls, truth, scene = planted_noise_instances()
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    ts, anchors = fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls)
    args = (fm, ts, None, fdcm.DefaultSearch(4, 10), fdcm.BatchOptimize(10), fdcm.ExponentialPenalty(1.5))
    base = fdcm.search_topk(*args, k=len(tmpls), select=fdcm.DistinctMatches(max_per_template=1))
    ref = fdcm.search_topk(*args, k=len(tmpls), select=fdcm.DistinctMatches(max_per_template=1), refine=R)

    def errors(m):
        t = int(m["tmpl_idx"])
        T = np.asarray(m["transform"], np.float64).reshape(2, 3)
        a = np.append(anchors[t].astype(np.float64), 1.0)
        rot = math.atan2(T[1, 0], T[0, 0]) - math.atan2(truth[t][1, 0], truth[t][0, 0])
        return float(np.hypot(*(T @ a - truth[t] @ a))), abs(math.remainder(rot, 2 * math.pi))

    def offset(m):   # signed anchor offset from the planted pose
        t = int(m["tmpl_idx"])
        a = np.append(anchors[t].astype(np.float64), 1.0)
        return np.asarray(m["transform"], np.float64).reshape(2, 3) @ a - truth[t] @ a

    before, after, off0, off1 = [], [], [], []
    for m0, m1 in zip(base, ref):
        if int(m0["tmpl_idx"]) in truth and errors(m0)[0] < 10 and errors(m0)[1] < 0.2:
            before.append(errors(m0))
            after.append(errors(m1))
            off0.append(offset(m0))
            off1.append(offset(m1))
    b = np.mean(before, axis=0) if before else [math.nan, math.nan]
    a = np.mean(after, axis=0) if after else [math.nan, math.nan]
    return {"planted": len(truth), "found": len(before), "anchor_px_before": round(float(b[0]), 4), "anchor_px_after": round(float(a[0]), 4),
            "rotation_rad_before": round(float(b[1]), 5), "rotation_rad_after": round(float(a[1]), 5),
            "mean_anchor_offset_px_before": np.round(np.mean(off0, axis=0), 4).tolist() if off0 else None,
            "mean_anchor_offset_px_after": np.round(np.mean(off1, axis=0), 4).tolist() if off1 else None}


def noise_free_instances():
    """40 templates planted noise-free among 100 clutter lines: (templates, the planted poses as records, scene)."""
    w, h = 1280, 720
    tmpls = synth_templates(40, 30, w, seed=81)
    rng = np.random.default_rng(82)
    recs, extra = np.zeros(len(tmpls), fdcm.MATCH_DTYPE), []
    for q in range(len(tmpls)):
        th = rng.uniform(-math.pi, math.pi)
        T = np.array([[math.cos(th), -math.sin(th), rng.uniform(0.15 * w, 0.85 * w)],
                      [math.sin(th), math.cos(th), rng.uniform(0.15 * h, 0.85 * h)]])
        recs[q] = (q, 0.0, T.reshape(6).astype(np.float32))
        extra.append(apply_transform(tmpls[q], recs[q]["transform"].reshape(2, 3)))
    scene = np.ascontiguousarray(np.concatenate([synth_scene(w, h, 100, seed=83)] + extra, axis=1), np.float32)
    return tmpls, recs, scene


def start_at_truth():
    """Noise-free planted instances, refinement started at the exact planted pose: mean anchor (px) and rotation (rad)
    errors after refinement (0 before), and the scores at the start and after."""
    tmpls, recs, scene = noise_free_instances()
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    ts, anchors = fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls)
    start = fdcm.refine_matches(fm, ts, recs, fdcm.PoseRefinement(1, 0, 0.0, 0, 0.0))
    out = {"instances": len(tmpls), "mean_score_at_truth": round(float(np.nanmean(start["score"])), 3)}
    for name, r in (("default", R), ("one_level_1px_0.01rad", fdcm.PoseRefinement(1, 1, 0.01, 1, 1.0))):
        ref = fdcm.refine_matches(fm, ts, recs, r)
        da, dr = [], []
        for m0, m1 in zip(recs, ref):
            a = np.append(anchors[int(m0["tmpl_idx"])].astype(np.float64), 1.0)
            T0 = m0["transform"].astype(np.float64).reshape(2, 3)
            T1 = m1["transform"].astype(np.float64).reshape(2, 3)
            da.append(float(np.hypot(*(T1 @ a - T0 @ a))))
            dr.append(abs(math.remainder(math.atan2(T1[1, 0], T1[0, 0]) - math.atan2(T0[1, 0], T0[0, 0]), 2 * math.pi)))
        out[name] = {"anchor_px_after": round(float(np.mean(da)), 4), "rotation_rad_after": round(float(np.mean(dr)), 5),
                     "mean_score_after": round(float(np.nanmean(ref["score"])), 3)}
    return out


def main():
    res = {"gpu": gpu_info(), "reps": REPS, "refine": repr(R), "config3": config3(REPS), "real_assets": real_assets(REPS),
           "planted_noise": planted_noise(), "start_at_truth": start_at_truth()}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
