"""Cost and recall of the dense pose-grid search (search_dense), one JSON line:
python scripts/bench_dense.py [reps]

Real assets (the 40 scenes of tests/golden/real_assets, every template of the object, padding 1.0, ExponentialPenalty(1.5)):
the median over scenes of the per-scene time of search_dense at the default DenseSearch() with
DistinctMatches(max_per_template=1), k = 10, with and without the default PoseRefinement().  Every timed call ends in a
device synchronisation (the call downloads its result): 3 warm-ups, then the median of `reps` calls.  Also reported: the
per-kernel split of profile_report() in a separate profiled pass (one call per scene), and map gathers per second of
dense_eval, with the gather count computed from the shapes below (2 L gathers per valid pose).

Recall: the planted-noise workload of scripts/bench_refine.py (200 templates x 30 lines, 40 of them planted in a 1280 x 720
scene with +-0.5 px end-point noise), once with the planted lines intact and once with every planted line cut into 2-3
pieces with gaps.  Found: instances with a match of their template within 10 px (anchor) and 0.2 rad of the planted pose,
among the k = 200, max_per_template = 1 results of search_topk with DefaultSearch(4, 10) and of search_dense at the
defaults, each without and with refinement.

Config 3 (5000 templates over a 2880^2 map, about 6 x 10^13 gathers at the defaults) is not a dense workload and is not run."""
import glob
import json
import math
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import openfdcm_b200 as fdcm  # noqa: E402
from scripts.bench_select import gpu_info, median_ms  # noqa: E402
from tests.util import apply_transform, synth_scene, synth_templates  # noqa: E402

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 5
D = fdcm.DenseSearch()
R = fdcm.PoseRefinement()
SEL = fdcm.DistinctMatches(max_per_template=1)
PEN = fdcm.ExponentialPenalty(1.5)


def dense_gathers(fm, tmpls, anchors, d):
    """Map gathers of one search_dense: 2 L per valid pose, the valid poses counted per (template, rotation) from the
    rotated template's bounding box (rules 2-4 of include/fdcm_b200.h in float32)."""
    W, H = fm.width, fm.height
    sx, sy = (np.float32(v) for v in fm.get_scene_translation())
    th = d.rot_start + np.arange(d.rotations) * np.float64(np.float32(d.rot_step))
    c, s = np.cos(th).astype(np.float32), np.sin(th).astype(np.float32)
    gx = np.arange(0, W, d.stride).astype(np.float32)
    gy = np.arange(0, H, d.stride).astype(np.float32)
    total = 0
    for t, tm in enumerate(tmpls):
        tm = np.asarray(tm, np.float32).reshape(4, -1)
        L = tm.shape[1]
        if L == 0:
            continue
        xs, ys = np.concatenate([tm[0], tm[2]]), np.concatenate([tm[1], tm[3]])
        rx = c[:, None] * xs[None, :] - s[:, None] * ys[None, :]
        ry = s[:, None] * xs[None, :] + c[:, None] * ys[None, :]
        ax, ay = anchors[t]
        ox = sx + ((gx[None, :] - sx) - (c * ax - s * ay)[:, None])
        oy = sy + ((gy[None, :] - sy) - (s * ax + c * ay)[:, None])
        nu = ((rx.min(1)[:, None] + ox >= 0) & (rx.max(1)[:, None] + ox <= W - 1)).sum(1)
        nv = ((ry.min(1)[:, None] + oy >= 0) & (ry.max(1)[:, None] + oy <= H - 1)).sum(1)
        total += int((nu.astype(np.int64) * nv).sum()) * 2 * L
    return total


def real_assets(reps):
    assets = os.path.join(ROOT, "tests", "golden", "real_assets")
    times = {"dense_k10_cap1": [], "dense_k10_cap1_refine": []}
    gathers, eval_ms, split = 0, 0.0, {}
    n_tmpl = {}
    for obj in ("obj_01", "obj_02", "obj_03", "obj_04"):
        tm = sorted(glob.glob(os.path.join(assets, obj, "templates", "*.tmpl")), key=lambda q: int(os.path.basename(q)[9:-5]))
        sc = sorted(glob.glob(os.path.join(assets, obj, "scene_*", "camera_0.scene")), key=lambda q: int(os.path.basename(os.path.dirname(q))[6:]))
        tmpls = [fdcm.read(q) for q in tm]
        n_tmpl[obj] = len(tmpls)
        ts, anchors = fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls)
        for path in sc:
            fm = fdcm.build_cuda_featuremap(fdcm.read(path), fdcm.Dt3CudaParameters(30, 5.0, 1.0))
            for name, ref in (("dense_k10_cap1", None), ("dense_k10_cap1_refine", R)):
                times[name].append(median_ms(lambda: fdcm.search_dense(fm, ts, D, PEN, 10, select=SEL, refine=ref), reps))
            fdcm.profile(True, reset=True)
            fdcm.search_dense(fm, ts, D, PEN, 10, select=SEL)
            rep = fdcm.profile_report()
            fdcm.profile(False)
            for k, v in rep.items():
                split.setdefault(k, []).append(v["total_ms"])
            eval_ms += rep["dense_eval"]["total_ms"]
            gathers += dense_gathers(fm, tmpls, anchors, D)
    med = {n: round(float(np.median(v)), 3) for n, v in times.items()}
    return {"n_scenes": len(times["dense_k10_cap1"]), "templates": n_tmpl, "dense": repr(D), "refine": repr(R),
            "ms_median_over_scenes": med, "refine_extra_ms": round(med["dense_k10_cap1_refine"] - med["dense_k10_cap1"], 3),
            "kernels_ms_median_over_scenes": {k: round(float(np.median(v)), 4) for k, v in split.items()},
            "gathers_per_scene_mean": int(gathers / max(1, len(times["dense_k10_cap1"]))),
            "dense_eval_gathers_per_s": float(f"{gathers / (eval_ms * 1e-3):.4g}") if eval_ms > 0 else None}


def cut(lines, rng):
    """Every line cut into 2-3 pieces with gaps of 8 % of its length between them."""
    out = []
    for x1, y1, x2, y2 in np.asarray(lines, np.float64).T:
        n = int(rng.integers(2, 4))
        cuts = np.sort(rng.uniform(0.2, 0.8, n - 1))
        ends = np.concatenate([[0.0], cuts, [1.0]])
        for a, b in zip(ends[:-1], ends[1:]):
            a2, b2 = (a + 0.04 if a > 0 else a), (b - 0.04 if b < 1 else b)
            if b2 > a2:
                out.append([x1 + a2 * (x2 - x1), y1 + a2 * (y2 - y1), x1 + b2 * (x2 - x1), y1 + b2 * (y2 - y1)])
    return np.ascontiguousarray(np.array(out, np.float32).T)


def recall(cut_lines):
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
    args = (fm, ts, None, fdcm.DefaultSearch(4, 10), fdcm.BatchOptimize(10), PEN)

    def found(matches):
        n = 0
        for m in matches:
            t = int(m["tmpl_idx"])
            if t not in truth:
                continue
            T = np.asarray(m["transform"], np.float64).reshape(2, 3)
            a = np.append(anchors[t].astype(np.float64), 1.0)
            rot = abs(math.remainder(math.atan2(T[1, 0], T[0, 0]) - math.atan2(truth[t][1, 0], truth[t][0, 0]), 2 * math.pi))
            n += float(np.hypot(*(T @ a - truth[t] @ a))) < 10 and rot < 0.2
        return n

    out = {"planted": len(truth), "scene_lines": int(scene.shape[1]), "map": [fm.width, fm.height]}
    for name, call in (("search_topk", lambda ref: fdcm.search_topk(*args, k=k, select=SEL, refine=ref)),
                       ("search_dense", lambda ref: fdcm.search_dense(fm, ts, D, PEN, k, select=SEL, refine=ref))):
        for suffix, ref in (("", None), ("_refine", R)):
            out[name + suffix] = found(call(ref))
    out["search_dense_ms"] = round(median_ms(lambda: fdcm.search_dense(fm, ts, D, PEN, k, select=SEL), 3), 2)
    return out


def main():
    res = {"gpu": gpu_info(), "reps": REPS, "real_assets": real_assets(REPS),
           "recall": {"intact_lines": recall(False), "cut_lines": recall(True)}}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
