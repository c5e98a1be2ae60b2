"""Cost and effect of scale as a pose dimension (search_dense(scales=ScaleGrid), PoseFit(scale_range=...)), one JSON line:
python scripts/bench_scale.py [reps]

Workloads:
- Scaled dense search: real assets (the first 2 scenes of each of the 4 objects, every template of the object, padding 1.0,
  ExponentialPenalty(1.5)), search_dense at the DenseSearch defaults with DistinctMatches(max_per_template=1), k = 10, at
  S = 1 (ScaleGrid()) and S = 5 (0.8 .. 1.25).  Median time per scene and the dense_eval gathers per second (2 L gathers
  per valid pose, counted by the model's bounding-box rule for every scale).
- Scaled fit: config 3 (5000 templates x 40 lines vs one 1080p scene), fit_matches rigid vs scaled on the search's top-10 and
  on one match per template at k = 5000.
- Accuracy: 40 templates planted at scales drawn from [0.8, 1.25] with +-0.5 px end-point noise among 300 clutter lines;
  found counts (anchor within 10 px, rotation within 0.2 rad, scale within 10 %), mean anchor / rotation / relative scale
  errors of (a) dense at one scale + the rigid fit, (b) dense at 5 scales with DefaultPenalty + the scaled fit, (c)
  search_topk over 5 scaled copies of every template (the best-scoring copy of each template) + the scaled fit.
Every timed call ends in a device synchronisation: 3 warm-ups, then the median of `reps` calls.  Also the GPU name / power
limit, read in the same run."""
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
from tests.util import apply_transform, plant_instances, synth_scene, synth_templates  # noqa: E402

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 10
D = fdcm.DenseSearch()
SEL = fdcm.DistinctMatches(max_per_template=1)
PEN = fdcm.ExponentialPenalty(1.5)
LO, HI = 0.8, 1.25
S5 = fdcm.ScaleGrid(5, LO, (HI / LO) ** 0.25)
FIT = fdcm.PoseFit()
FIT_S = fdcm.PoseFit(scale_range=(0.7, 1.4))


def scales_of(g):
    return [float(np.float32(float(np.float32(g.start)) * math.pow(float(np.float32(g.ratio)), k))) for k in range(g.scales)]


def dense_gathers(fm, tmpls, anchors, d, g):
    """Map gathers of one scaled search_dense: 2 L per valid pose, from the posed template's bounding box."""
    W, H = fm.width, fm.height
    sx, sy = (np.float32(v) for v in fm.get_scene_translation())
    th = d.rot_start + np.arange(d.rotations) * np.float64(np.float32(d.rot_step))
    gx = np.arange(0, W, d.stride).astype(np.float32)
    gy = np.arange(0, H, d.stride).astype(np.float32)
    total = 0
    for sk in scales_of(g):
        a_, b_ = (sk * np.cos(th)).astype(np.float32), (sk * np.sin(th)).astype(np.float32)
        for t, tm in enumerate(tmpls):
            tm = np.asarray(tm, np.float32).reshape(4, -1)
            if tm.shape[1] == 0:
                continue
            xs, ys = np.concatenate([tm[0], tm[2]]), np.concatenate([tm[1], tm[3]])
            rx = a_[:, None] * xs[None, :] - b_[:, None] * ys[None, :]
            ry = b_[:, None] * xs[None, :] + a_[:, None] * ys[None, :]
            ax, ay = anchors[t]
            ox = sx + ((gx[None, :] - sx) - (a_ * ax - b_ * ay)[:, None])
            oy = sy + ((gy[None, :] - sy) - (b_ * ax + a_ * ay)[:, None])
            nu = ((rx.min(1)[:, None] + ox >= 0) & (rx.max(1)[:, None] + ox <= W - 1)).sum(1)
            nv = ((ry.min(1)[:, None] + oy >= 0) & (ry.max(1)[:, None] + oy <= H - 1)).sum(1)
            total += int((nu.astype(np.int64) * nv).sum()) * 2 * tm.shape[1]
    return total


def real_assets(reps):
    assets = os.path.join(ROOT, "tests", "golden", "real_assets")
    out = {}
    for name, g in (("S1", fdcm.ScaleGrid()), ("S5", S5)):
        times, gathers, eval_ms = [], 0, 0.0
        for obj in ("obj_01", "obj_02", "obj_03", "obj_04"):
            tm = sorted(glob.glob(os.path.join(assets, obj, "templates", "*.tmpl")), key=lambda q: int(os.path.basename(q)[9:-5]))
            sc = sorted(glob.glob(os.path.join(assets, obj, "scene_*", "camera_0.scene")),
                        key=lambda q: int(os.path.basename(os.path.dirname(q))[6:]))[:2]
            tmpls = [fdcm.read(q) for q in tm]
            ts, anchors = fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls)
            for path in sc:
                fm = fdcm.build_cuda_featuremap(fdcm.read(path), fdcm.Dt3CudaParameters(30, 5.0, 1.0))
                times.append(median_ms(lambda: fdcm.search_dense(fm, ts, D, PEN, 10, select=SEL, scales=g), reps))
                fdcm.profile(True, reset=True)
                fdcm.search_dense(fm, ts, D, PEN, 10, select=SEL, scales=g)
                eval_ms += fdcm.profile_report()["dense_eval"]["total_ms"]
                fdcm.profile(False)
                gathers += dense_gathers(fm, tmpls, anchors, D, g)
        out[name] = {"scales": scales_of(g), "n_scenes": len(times), "ms_median_over_scenes": round(float(np.median(times)), 3),
                     "dense_eval_gathers_per_s": float(f"{gathers / (eval_ms * 1e-3):.4g}") if eval_ms > 0 else None}
    out["ratio_S5_over_S1"] = round(out["S5"]["ms_median_over_scenes"] / out["S1"]["ms_median_over_scenes"], 3)
    return out


def config3(reps):
    tmpls = synth_templates(5000, 40, 1920, seed=3001)
    scene = plant_instances(synth_scene(1920, 1080, 2000, seed=3000), tmpls, 1920, 1080, seed=3002)
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    ts = fdcm.TemplateSet(tmpls)
    args = (fm, ts, None, fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), PEN)
    out = {}
    for name, (k, sel) in {"k10": (10, None), "k5000_cap1": (5000, SEL)}.items():
        top = fdcm.search_topk(*args, k=k, select=sel)
        rigid = median_ms(lambda: fdcm.fit_matches(fm, ts, top, FIT, PEN), reps)
        scaled = median_ms(lambda: fdcm.fit_matches(fm, ts, top, FIT_S, PEN), reps)
        fdcm.profile(True, reset=True)
        fdcm.fit_matches(fm, ts, top, FIT, PEN)
        fdcm.fit_matches(fm, ts, top, FIT_S, PEN)
        rep = fdcm.profile_report()
        fdcm.profile(False)
        out[name] = {"n": int(len(top)), "rigid_ms": round(rigid, 4), "scaled_ms": round(scaled, 4),
                     "fit_eval_kernel_ms": round(rep["fit_eval"]["total_ms"], 4),
                     "fit_eval_scaled_kernel_ms": round(rep["fit_eval_scaled"]["total_ms"], 4)}
    return out


def planted_scaled_instances():
    """40 templates planted at scales in [0.8, 1.25] with +-0.5 px end-point noise among 300 clutter lines."""
    w, h = 1280, 720
    tmpls = synth_templates(40, 30, w, seed=91)
    rng = np.random.default_rng(92)
    truth, extra = {}, []
    for q in range(40):
        th, s = rng.uniform(-math.pi, math.pi), rng.uniform(LO, HI)
        T = np.array([[s * math.cos(th), -s * math.sin(th), rng.uniform(0.15 * w, 0.85 * w)],
                      [s * math.sin(th), s * math.cos(th), rng.uniform(0.15 * h, 0.85 * h)]])
        truth[q] = T
        extra.append(apply_transform(tmpls[q], T) + rng.uniform(-0.5, 0.5, (4, tmpls[q].shape[1])).astype(np.float32))
    scene = np.ascontiguousarray(np.concatenate([synth_scene(w, h, 300, seed=93)] + extra, axis=1), np.float32)
    return tmpls, truth, scene


def accuracy():
    tmpls, truth, scene = planted_scaled_instances()
    fm = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(30, 5.0, 1.5))
    ts, anchors = fdcm.TemplateSet(tmpls), fdcm.get_template_anchors(tmpls)
    d = fdcm.DenseSearch(72, stride=4, cell=8)
    k = len(tmpls)
    res = {"dense": repr(d), "planted": len(truth)}

    def summary(matches, tmpl_of=lambda t: t):
        errs = []
        for m in matches:
            t = tmpl_of(int(m["tmpl_idx"]))
            T = np.asarray(m["transform"], np.float64).reshape(2, 3)
            a = np.append(anchors[t].astype(np.float64), 1.0)
            ea = float(np.hypot(*(T @ a - truth[t] @ a)))
            er = abs(math.remainder(math.atan2(T[1, 0], T[0, 0]) - math.atan2(truth[t][1, 0], truth[t][0, 0]), 2 * math.pi))
            es = abs(math.sqrt(abs(np.linalg.det(T[:, :2]))) / math.sqrt(np.linalg.det(truth[t][:, :2])) - 1.0)
            if ea < 10 and er < 0.2 and es < 0.1:
                errs.append((ea, er, es))
        m = np.mean(errs, axis=0) if errs else [math.nan] * 3
        return {"found": len(errs), "anchor_px": round(float(m[0]), 4), "rotation_rad": round(float(m[1]), 5),
                "rel_scale": round(float(m[2]), 5)}

    a = fdcm.search_dense(fm, ts, d, PEN, k, select=SEL)
    res["a_dense_S1"] = summary(a)
    res["a_dense_S1_rigid_fit"] = summary(fdcm.fit_matches(fm, ts, a, FIT, PEN))
    b = fdcm.search_dense(fm, ts, d, fdcm.DefaultPenalty(), k, select=SEL, scales=S5)
    res["b_dense_S5"] = summary(b)
    res["b_dense_S5_scaled_fit"] = summary(fdcm.fit_matches(fm, ts, b, FIT_S, fdcm.DefaultPenalty()))
    # (c) scaled copies: copy j of template t is template t * 5 + j
    copies = [(np.asarray(t, np.float32) * np.float32(s)).astype(np.float32) for t in tmpls for s in scales_of(S5)]
    cs = fdcm.TemplateSet(copies)
    c = fdcm.search_topk(fm, cs, None, fdcm.DefaultSearch(4, 10), fdcm.BatchOptimize(10), PEN, k=len(copies), select=SEL)
    # one match per template, as DistinctMatches(max_per_template=1) gives the scaled search: the best-scoring copy
    _, first = np.unique(c["tmpl_idx"] // 5, return_index=True)
    c = c[np.sort(first)]
    c_fit = fdcm.fit_matches(fm, cs, c, FIT_S, PEN)
    # express the copies' poses in the original template's frame: T (s I) and the anchor scales with the copy
    for arr in (c, c_fit):
        for m in arr:
            s = np.float32(scales_of(S5)[int(m["tmpl_idx"]) % 5])
            m["transform"][[0, 1, 3, 4]] *= s
    res["c_copies_topk"] = summary(c, lambda t: t // 5)
    res["c_copies_topk_scaled_fit"] = summary(c_fit, lambda t: t // 5)
    return res


def main():
    res = {"gpu": gpu_info(), "reps": REPS, "real_assets_dense": real_assets(REPS), "config3_fit": config3(REPS), "accuracy": accuracy()}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
