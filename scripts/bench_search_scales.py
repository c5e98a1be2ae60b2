"""Cost and effect of scale in the line-alignment search (search_topk(scales=ScaleGrid), fdcm_search_scales), one JSON line:
python scripts/bench_search_scales.py [reps]

Workloads:
- Config 3 (5000 templates x 40 lines vs one 1080p scene, padding 1.5, DefaultSearch(4, 4), BatchOptimize(10),
  ExponentialPenalty(1.5); the map is built once): the plain top-10 and one match per template at k = 5000, without a grid
  and at S = 1, 3 and 5 (geometric grids over [0.8, 1.25]).  Per setting the median call time, the search, ordering and
  remap kernel times from the library's profile (a separate pass), the hypothesis count, and the first call on a freshly
  loaded template set (host preparation and upload of the copies) against a call that finds them cached.
- Accuracy: the planted scaled instances of scripts/bench_scale.py (40 templates at scales in [0.8, 1.25], +-0.5 px noise,
  300 clutter lines): the native search_topk(scales=S5, select=DistinctMatches(max_per_template=1)), with and without
  PoseFit(scale_range=(0.7, 1.4)), against bench_scale.py's row (c), the search of 5 scaled copies of every template whose
  best copy per template is mapped back by hand.  Also whether the native records before the fit equal row (c)'s mapped
  records byte for byte.
Every timed call ends in a device synchronisation: 3 warm-ups, then the median of `reps` calls.  Also the GPU name / power
limit, read in the same run."""
import json
import math
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import openfdcm_b200 as fdcm  # noqa: E402
from scripts.bench_scale import FIT_S, HI, LO, PEN, S5, SEL, planted_scaled_instances, scales_of  # noqa: E402
from scripts.bench_select import gpu_info, median_ms  # noqa: E402
from tests.util import plant_instances, synth_scene, synth_templates  # noqa: E402

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 10
GRIDS = {"none": None, "S1": fdcm.ScaleGrid(), "S3": fdcm.ScaleGrid(3, LO, (HI / LO) ** 0.5), "S5": S5}
KERNELS = ("search", "search_order", "search_scale_remap")


def kernel_ms(fn, reps):
    fdcm.profile(True, reset=True)
    for _ in range(reps):
        fn()
    rep = fdcm.profile_report()
    fdcm.profile(False, reset=True)
    return {k: round(rep[k]["total_ms"] / rep[k]["launches"], 4) for k in KERNELS if k in rep}


def config3(reps):
    tmpls = synth_templates(5000, 40, 1920, seed=3001)
    scene = plant_instances(synth_scene(1920, 1080, 2000, seed=3000), tmpls, 1920, 1080, seed=3002)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    ts = fdcm.TemplateSet(tmpls)
    ds, bo = fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10)
    out = {}
    for gname, g in GRIDS.items():
        for name, (k, sel) in {"k10": (10, None), "k5000_cap1": (5000, SEL)}.items():
            call = lambda t=ts: fdcm.search_topk(fm, t, None, ds, bo, PEN, k, select=sel, scales=g)  # noqa: E731
            r = {"ms": round(median_ms(call, reps), 4)}
            r["hypotheses"] = fm.last_search_stats()["n_hypotheses"]
            r["kernels_ms"] = kernel_ms(call, reps)
            if g is not None and name == "k10":
                # a new load of the same templates: its first scaled call prepares the copies, the second finds them cached
                first, cached = [], []
                for _ in range(3):
                    fresh = fdcm.TemplateSet(tmpls)
                    fdcm.search_topk(fm, fresh, None, ds, bo, PEN, k, scales=None)   # (the set's upload and denominators)
                    t0 = time.perf_counter()
                    call(fresh)
                    first.append((time.perf_counter() - t0) * 1e3)
                    t0 = time.perf_counter()
                    call(fresh)
                    cached.append((time.perf_counter() - t0) * 1e3)
                r["first_call_ms"] = round(float(np.median(first)), 4)
                r["cached_call_ms"] = round(float(np.median(cached)), 4)
            out[f"{gname}_{name}"] = r
    return out


def accuracy():
    tmpls, truth, scene = planted_scaled_instances()
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    ts, anchors = fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls)
    sk = scales_of(S5)

    def summary(matches):
        errs = []
        for m in matches:
            t = int(m["tmpl_idx"])
            T = np.asarray(m["transform"], np.float64).reshape(2, 3)
            a = np.append(anchors[t].astype(np.float64), 1.0)
            ea = float(np.hypot(*(T @ a - truth[t] @ a)))
            er = abs(math.remainder(math.atan2(T[1, 0], T[0, 0]) - math.atan2(truth[t][1, 0], truth[t][0, 0]), 2 * math.pi))
            es = abs(math.sqrt(abs(np.linalg.det(T[:, :2]))) / math.sqrt(np.linalg.det(truth[t][:, :2])) - 1.0)
            if ea < 10 and er < 0.2 and es < 0.1:
                errs.append((ea, er, es))
        m = np.mean(errs, axis=0) if errs else [math.nan] * 3
        return {"n": len(matches), "found": len(errs), "anchor_px": round(float(m[0]), 4), "rotation_rad": round(float(m[1]), 5),
                "rel_scale": round(float(m[2]), 5)}

    res = {"planted": len(truth)}
    ds, bo = fdcm.DefaultSearch(4, 10), fdcm.BatchOptimize(10)
    # row (c) of bench_scale.py: copies, the best copy per template, its pose and index mapped back by hand
    copies = [(np.asarray(t, np.float32) * np.float32(s)).astype(np.float32) for t in tmpls for s in sk]
    cs = fdcm.TemplateSet(copies)
    c = fdcm.search_topk(fm, cs, None, ds, bo, PEN, k=len(copies), select=SEL)
    _, first = np.unique(c["tmpl_idx"] // 5, return_index=True)
    c = c[np.sort(first)]
    c_fit = fdcm.fit_matches(fm, cs, c, FIT_S, PEN)
    for arr in (c, c_fit):
        for m in arr:
            s = np.float32(sk[int(m["tmpl_idx"]) % 5])
            m["transform"][[0, 1, 3, 4]] *= s
            m["tmpl_idx"] //= 5
    res["c_copies"] = summary(c)
    res["c_copies_scaled_fit"] = summary(c_fit)
    native = fdcm.search_topk(fm, ts, None, ds, bo, PEN, k=len(tmpls), select=SEL, scales=S5)
    res["native"] = summary(native)
    res["native_equals_mapped_copies"] = bool(native.tobytes() == c.tobytes())
    res["native_scaled_fit"] = summary(fdcm.search_topk(fm, ts, None, ds, bo, PEN, k=len(tmpls), select=SEL, scales=S5, fit=FIT_S))
    return res


def main():
    res = {"gpu": gpu_info(), "reps": REPS, "config3": config3(REPS), "accuracy": accuracy()}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
