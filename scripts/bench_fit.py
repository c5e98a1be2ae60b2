"""Cost and effect of the pose fit (search_topk(fit=PoseFit()), fit_matches), one JSON line:
python scripts/bench_fit.py [reps]

Workloads: config 3 (5000 templates x 40 lines vs one 1080p scene, padding 1.5, DefaultSearch(4,4), BatchOptimize(10),
ExponentialPenalty(1.5); the map is built once): the plain top-10 and one match per template at k = 5000, each with and
without the default fit, as bench_refine.py times refinement (k = 10 is the latency-bound case, k = 5000 the throughput
case).  The scene-line grid is built once per map write: it is timed on its own (profile_report "fit_grid" after a rerun),
and the timed composed calls reuse it.  The composed Python call is the search, then fit_matches on its output: the
standalone fit on the k records is timed too, and its time minus the fit_eval kernel is the host round trip (the records'
upload and download, the launch, the synchronisation).  The 40 real-asset scenes: the median over scenes of k = 10,
max_per_template = 1 with and without the fit.  Every timed call ends in a device synchronisation: 3 warm-ups, then the
median of `reps` calls.  Accuracy: mean anchor (px) and rotation (rad) errors on bench_refine.py's planted-noise instances
for the search alone, search + fit and search + refinement + fit, and on its noise-free instances started 2 px / 0.03 rad
off.  Also the GPU name / power limit."""
import json
import math
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import openfdcm_b200 as fdcm  # noqa: E402
from scripts.bench_refine import noise_free_instances, planted_noise_instances  # noqa: E402
from scripts.bench_select import gpu_info, kernel_split, median_ms  # noqa: E402
from tests.util import plant_instances, synth_scene, synth_templates  # noqa: E402

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 30
FIT = fdcm.PoseFit()
CAP1 = fdcm.DistinctMatches(max_per_template=1)


def config3(reps):
    tmpls = synth_templates(5000, 40, 1920, seed=3001)
    scene = plant_instances(synth_scene(1920, 1080, 2000, seed=3000), tmpls, 1920, 1080, seed=3002)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    ts = fdcm.TemplateSet(tmpls)
    pen = fdcm.ExponentialPenalty(1.5)
    args = (fm, ts, None, fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), pen)
    out = {}
    for name, (k, sel) in {"plain_k10": (10, None), "k5000_cap1": (5000, CAP1)}.items():
        plain = lambda: fdcm.search_topk(*args, k=k, select=sel)  # noqa: E731
        fitted = lambda: fdcm.search_topk(*args, k=k, select=sel, fit=FIT)  # noqa: E731
        top = plain()
        standalone = lambda: fdcm.fit_matches(fm, ts, top, FIT, pen)  # noqa: E731
        _, stats = fdcm.fit_matches(fm, ts, top, FIT, pen, return_stats=True)
        split = kernel_split(standalone, 10)
        r = {"n": int(len(top)), "ms": round(median_ms(plain, reps), 4), "fit_ms": round(median_ms(fitted, reps), 4),
             "kernels_ms_with_fit": kernel_split(fitted, 10), "fit_matches_ms": round(median_ms(standalone, reps), 4),
             "fit_eval_kernel_ms": split.get("fit_eval"),
             "mean_iterations": round(float(np.mean(stats["iterations"])), 3),
             "mean_inlier_share": round(float(np.mean(stats["n_inliers"] / np.maximum(stats["n_samples"], 1))), 4)}
        r["extra_ms"] = round(r["fit_ms"] - r["ms"], 4)
        r["host_round_trip_ms"] = round(r["fit_matches_ms"] - (r["fit_eval_kernel_ms"] or 0.0), 4)
        out[name] = r
    # the grid, once per map write: a rerun bumps the write, the next fit rebuilds it
    fdcm.profile(True, reset=True)
    for _ in range(10):
        fm.rerun()
        fdcm.fit_matches(fm, ts, top[:1], FIT)
    rep = fdcm.profile_report()
    fdcm.profile(False)
    out["grid_build_ms"] = round(rep["fit_grid"]["total_ms"] / 10, 4)
    return out


def real_assets(reps):
    import glob
    assets = os.path.join(ROOT, "tests", "golden", "real_assets")
    s, o, p = fdcm.DefaultSearch(4, 10), fdcm.BatchOptimize(10), fdcm.ExponentialPenalty(1.5)
    times = {"k10_cap1": [], "k10_cap1_fit": []}
    for obj in ("obj_01", "obj_02", "obj_03", "obj_04"):
        tm = sorted(glob.glob(os.path.join(assets, obj, "templates", "*.tmpl")), key=lambda q: int(os.path.basename(q)[9:-5]))
        sc = sorted(glob.glob(os.path.join(assets, obj, "scene_*", "camera_0.scene")), key=lambda q: int(os.path.basename(os.path.dirname(q))[6:]))
        ts = fdcm.TemplateSet([fdcm.read(q) for q in tm])
        for path in sc:
            fm = fdcm.build_cuda_featuremap(fdcm.read(path), fdcm.Dt3CudaParameters(30, 5.0, 1.0))
            for name, fit in (("k10_cap1", None), ("k10_cap1_fit", FIT)):
                times[name].append(median_ms(lambda: fdcm.search_topk(fm, ts, None, s, o, p, k=10, select=CAP1, fit=fit), reps))
    med = {n: round(float(np.median(v)), 4) for n, v in times.items()}
    return {"n_scenes": len(times["k10_cap1"]), "ms_median_over_scenes": med, "extra_ms": round(med["k10_cap1_fit"] - med["k10_cap1"], 4)}


def errors(m, truth, anchors):
    t = int(m["tmpl_idx"])
    T = np.asarray(m["transform"], np.float64).reshape(2, 3)
    a = np.append(anchors[t].astype(np.float64), 1.0)
    rot = math.atan2(T[1, 0], T[0, 0]) - math.atan2(truth[t][1, 0], truth[t][0, 0])
    return float(np.hypot(*(T @ a - truth[t] @ a))), abs(math.remainder(rot, 2 * math.pi))


def planted_noise():
    """Mean anchor (px) and rotation (rad) errors of the found planted instances (found: the search's match within 10 px
    and 0.2 rad), for the search alone, with the fit, and with refinement then the fit."""
    tmpls, truth, scene = planted_noise_instances()
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    ts, anchors = fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls)
    args = (fm, ts, None, fdcm.DefaultSearch(4, 10), fdcm.BatchOptimize(10), fdcm.ExponentialPenalty(1.5))
    k = len(tmpls)
    base = fdcm.search_topk(*args, k=k, select=CAP1)
    fit = fdcm.search_topk(*args, k=k, select=CAP1, fit=FIT)
    ref_fit = fdcm.search_topk(*args, k=k, select=CAP1, refine=fdcm.PoseRefinement(), fit=FIT)
    rows = {"search": [], "search_fit": [], "search_refine_fit": []}
    for m0, m1, m2 in zip(base, fit, ref_fit):
        if int(m0["tmpl_idx"]) in truth and errors(m0, truth, anchors)[0] < 10 and errors(m0, truth, anchors)[1] < 0.2:
            for name, m in (("search", m0), ("search_fit", m1), ("search_refine_fit", m2)):
                rows[name].append(errors(m, truth, anchors))
    out = {"planted": len(truth), "found": len(rows["search"])}
    for name, v in rows.items():
        e = np.mean(v, axis=0) if v else [math.nan, math.nan]
        out[name] = {"anchor_px": round(float(e[0]), 4), "rotation_rad": round(float(e[1]), 5)}
    return out


def noise_free_start_off():
    """Noise-free planted instances, the fit started 2 px / 0.03 rad off the planted pose: mean and max errors after."""
    tmpls, recs, scene = noise_free_instances()
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    ts, anchors = fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls)
    rng = np.random.default_rng(91)
    truth = {int(r["tmpl_idx"]): r["transform"].astype(np.float64).reshape(2, 3) for r in recs}
    start = recs.copy()
    for i, r in enumerate(recs):
        T = truth[int(r["tmpl_idx"])]
        a = T @ np.append(anchors[int(r["tmpl_idx"])].astype(np.float64), 1.0)
        th = 0.03 * rng.choice([-1.0, 1.0])
        d = rng.normal(size=2)
        d = 2.0 * d / np.hypot(*d)
        R = np.array([[math.cos(th), -math.sin(th)], [math.sin(th), math.cos(th)]])
        M, e = R @ T[:, :2], R @ (T[:, 2] - a) + a + d
        start[i]["transform"] = np.array([M[0, 0], M[0, 1], e[0], M[1, 0], M[1, 1], e[1]], np.float32)
    got = fdcm.fit_matches(fm, ts, start, FIT)
    e0 = np.array([errors(m, truth, anchors) for m in start])
    e1 = np.array([errors(m, truth, anchors) for m in got])
    return {"instances": len(recs), "anchor_px_start": round(float(e0[:, 0].mean()), 4), "rotation_rad_start": round(float(e0[:, 1].mean()), 5),
            "anchor_px_mean": round(float(e1[:, 0].mean()), 5), "anchor_px_max": round(float(e1[:, 0].max()), 5),
            "rotation_rad_mean": round(float(e1[:, 1].mean()), 6), "rotation_rad_max": round(float(e1[:, 1].max()), 6)}


def main():
    res = {"gpu": gpu_info(), "reps": REPS, "fit": repr(FIT), "config3": config3(REPS), "real_assets": real_assets(REPS),
           "planted_noise": planted_noise(), "noise_free_start_off": noise_free_start_off()}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
