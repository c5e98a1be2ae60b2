"""Helpers of more than one test module: the real assets and the synthetic workload of the device tests, the score
functions the models take from the device evaluate, the models' inputs taken from the CPU oracle instead (scores, edge
masks, scene bins), the parity hook of the dense poses, the oracle references of the search, the poses and scenes of the
fit tests, and the map-geometry generators (tiny maps, the exact / literal boundary, scenes far from the origin)."""
import ctypes as C
import glob
import math
import os

import numpy as np

import openfdcm_b200 as fdcm
from openfdcm_b200 import _lib
from oracle import fdcm_oracle as orc
from tests.models.coverage import table_bins
from tests.models.dense import grid
from tests.models.fit import SceneLines
from tests.models.refine import refine_model, rotated
from tests.util import F32, plant_instances, synth_scene, synth_templates

ASSETS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "real_assets")
DIST = {"L2": (fdcm.distance.L2, orc.L2), "L2_SQUARED": (fdcm.distance.L2_SQUARED, orc.L2_SQUARED), "L1": (fdcm.distance.L1, orc.L1)}


# ---- workloads -------------------------------------------------------------------------------------------------------
def load_object(obj):
    """The templates and the scenes of one object of the real assets, in index order."""
    tm = sorted(glob.glob(os.path.join(ASSETS, obj, "templates", "*.tmpl")), key=lambda p: int(os.path.basename(p)[9:-5]))
    scenes = sorted(glob.glob(os.path.join(ASSETS, obj, "scene_*", "camera_0.scene")), key=lambda p: int(os.path.basename(os.path.dirname(p))[6:]))
    return [fdcm.read(p) for p in tm], [fdcm.read(p) for p in scenes]


def synthetic(n_tmpl=24, n_lines=20, seed=0, w=640, h=480, n_scene=200):
    tmpls = synth_templates(n_tmpl, n_lines, w, seed=seed + 1)
    scene = plant_instances(synth_scene(w, h, n_scene, seed=seed + 2), tmpls, w, h, seed=seed + 3, count=6)
    return tmpls, scene


def masks(fm):
    """The edge masks of every plane of a map, (D, H, W)."""
    return np.stack([fm.mask(q) for q in range(fm.depth)]) if fm.depth else np.zeros((0, 0, 0), np.uint8)


def fit_candidates(fm, tmpls, scene, n=40, seed=0):
    """Distinct search matches, the same matches moved by up to 2 px and 0.03 rad, and poses off the map."""
    rec = fdcm.search_topk(fm, tmpls, scene, fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), fdcm.ExponentialPenalty(1.5), k=n,
                           select=fdcm.DistinctMatches(max_per_template=2))
    rng = np.random.default_rng(seed)
    moved = rec.copy()
    a = rng.uniform(-0.03, 0.03, len(rec)).astype(F32)
    c, s = np.cos(a).astype(F32), np.sin(a).astype(F32)
    T = moved["transform"].copy()
    moved["transform"][:, 0] = c * T[:, 0] - s * T[:, 3]
    moved["transform"][:, 1] = c * T[:, 1] - s * T[:, 4]
    moved["transform"][:, 3] = s * T[:, 0] + c * T[:, 3]
    moved["transform"][:, 4] = s * T[:, 1] + c * T[:, 4]
    moved["transform"][:, 2] += rng.uniform(-2, 2, len(rec)).astype(F32)
    moved["transform"][:, 5] += rng.uniform(-2, 2, len(rec)).astype(F32)
    off = rec[: min(3, len(rec))].copy()
    off["transform"][:, 2] += F32(1e5)
    return np.concatenate([rec, moved, off])


# ---- the device evaluate as the models' score functions --------------------------------------------------------------
def evaluate_fn(fm):
    """score_fn of the dense model: fdcm_dt3_evaluate of the rotated template at every translation."""
    def score(Rt, tr):
        flat = np.ascontiguousarray(Rt, F32).reshape(-1, 4)
        off = np.array([0, len(flat)], np.int32)
        trn = np.ascontiguousarray(tr, F32)
        troff = np.array([0, len(trn)], np.int32)
        out = np.zeros(len(trn), F32)
        _lib.check(_lib.lib().fdcm_dt3_evaluate(fm._h, _lib.ptr(flat), _lib.ptr(off), 1, _lib.ptr(trn), _lib.ptr(troff), _lib.ptr(out)))
        return out
    return score


def device_scores(fm):
    """score_fn of the refinement model: fdcm_dt3_evaluate of every rotated template at (P2, P5)."""
    def score(work):
        recs, tr = [], []
        for tmpl, poses in work:
            R = rotated(poses, tmpl)
            recs += list(R)
            tr.append(poses[:, [2, 5]])
        off = np.zeros(len(recs) + 1, np.int32)
        off[1:] = np.cumsum([r.shape[0] for r in recs])
        flat = np.ascontiguousarray(np.concatenate(recs) if off[-1] else np.zeros((1, 4), F32), F32)
        trn = np.ascontiguousarray(np.concatenate(tr), F32)
        troff = np.arange(len(recs) + 1, dtype=np.int32)
        out = np.zeros(len(recs), F32)
        _lib.check(_lib.lib().fdcm_dt3_evaluate(fm._h, _lib.ptr(flat), _lib.ptr(off), len(recs), _lib.ptr(trn), _lib.ptr(troff),
                                                _lib.ptr(out)))
        return out
    return score


# ---- the CPU oracle as the models' inputs ----------------------------------------------------------------------------
def oracle_scores(c):
    """score_fn of the dense model from an oracle map c (orc.Dt3Cpu): evaluate of the rotated template at every
    translation."""
    def score(Rt, tr):
        return c.evaluate(np.ascontiguousarray(np.asarray(Rt, F32).reshape(-1, 4).T), np.asarray(tr, F32).reshape(-1, 2))
    return score


def oracle_pose_score(c):
    """score_fn of the fit model from an oracle map c: evaluate of the template posed by F at (F2, F5)."""
    def score(tmpl, F):
        F = np.asarray(F, F32).reshape(6)
        return c.evaluate(np.ascontiguousarray(rotated(F[None], tmpl)[0].T), F[[2, 5]].reshape(1, 2))[0]
    return score


def oracle_masks(c):
    """The edge masks (D, H, W) of a stage-1 oracle map c: its zero pixels."""
    return np.stack([c.plane(d) == 0 for d in range(c.depth)]).astype(np.uint8) if c.depth else np.zeros((0, 0, 0), np.uint8)


def oracle_bins(c, scene):
    """The scene bins of an oracle map c: closest_orientation of every shifted scene line."""
    ts = shifted_scene(scene, c.shift)
    return np.array([orc.closest_orientation(c.keys, ts[:, i]) for i in range(ts.shape[1])], np.int32)


def refine_reference(fm, tmpls, anchors, matches, r, score_fn=None, tmpl_idx_base=0):
    """The refinement model on a map, scored by the device evaluate unless score_fn is given."""
    return refine_model(matches, tmpls, anchors, r, fm.get_scene_translation(), fm.width, fm.height, score_fn or device_scores(fm),
                        tmpl_idx_base)


# ---- the parity hook of the dense poses ------------------------------------------------------------------------------
def dense_poses_hook(d, anchor, shift, W, H, r, capacity=None, g=None, k=0):
    """fdcm_dense_poses, or fdcm_dense_scaled_poses of scale k with a scale grid g -> (status, transforms (n, 6), n,
    (nx, ny))."""
    lx, ly, nx, ny = grid(d, shift, W, H) if d.rotations >= 1 and d.stride >= 1 else (0, 0, 0, 0)
    cap = nx * ny if capacity is None else capacity
    out = np.zeros((max(cap, 1), 6), F32)
    n, wh = C.c_int64(-1), np.zeros(2, np.int32)
    a, sh = np.ascontiguousarray(anchor, F32), np.ascontiguousarray(shift, F32)
    if g is None:
        st = _lib.lib().fdcm_dense_poses(C.byref(d._params()), _lib.ptr(a), _lib.ptr(sh), W, H, r, _lib.ptr(out), cap, C.byref(n),
                                         _lib.ptr(wh))
    else:
        st = _lib.lib().fdcm_dense_scaled_poses(C.byref(d._params()), C.byref(g._params()), _lib.ptr(a), _lib.ptr(sh), W, H, k, r,
                                                _lib.ptr(out), cap, C.byref(n), _lib.ptr(wh))
    return st, out[: max(n.value, 0)], n.value, tuple(wh.tolist())


# ---- the search against the oracle -----------------------------------------------------------------------------------
def optimizer(batch):
    """BatchOptimize(batch), or DefaultOptimize for batch 0."""
    return fdcm.BatchOptimize(batch) if batch else fdcm.DefaultOptimize()


def oracle_penalized(raw, tmpls, penalty):
    """penalize() of the oracle: DefaultPenalty divides by the template length, ExponentialPenalty by length ** tau."""
    if penalty is None:
        return raw
    kind = 0 if isinstance(penalty, fdcm.DefaultPenalty) else 1
    return orc.penalize(kind, penalty.tau, raw, orc.template_lengths(tmpls))


def topk_ref(pen, k, base=0):
    """Ascending score (NaN ranks as +inf), ties by hypothesis order, template indices offset by base."""
    key = np.where(np.isnan(pen["score"]), np.inf, pen["score"])
    want = pen[np.lexsort((np.arange(len(pen)), key))[:k]].copy()
    want["tmpl_idx"] += base
    return want


def assert_matches(got, want, what=""):
    assert len(got) == len(want), what
    assert np.array_equal(got["tmpl_idx"], want["tmpl_idx"]), what
    assert np.array_equal(got["score"], want["score"], equal_nan=True), what
    assert np.array_equal(got["transform"], want["transform"], equal_nan=True), what


def check_full_search(g, c, tmpls, scene, max_t, max_s, batch, penalty=None, tset=None):
    """search_all against the oracle: hypothesis list, counters and every match in hypothesis order."""
    got = fdcm.search_all(g, tset or tmpls, scene, fdcm.DefaultSearch(max_t, max_s), optimizer(batch), penalty)
    st = g.last_search_stats()
    orc.stats_reset()
    raw, hyp = c.search(tmpls, scene, max_t, max_s, batch=batch, want_hyp=True)
    evals, lookups = orc.stats_get()
    assert np.array_equal(g.last_hypotheses(), hyp), "hypothesis list"
    assert st["n_hypotheses"] == len(hyp)
    assert (st["n_evaluations"], st["n_lookups"]) == (evals, lookups), "the kernel scored another candidate set"
    assert st["n_valid"] == len(raw)
    assert_matches(got, oracle_penalized(raw, tmpls, penalty), f"batch {batch}")
    return raw, hyp


# ---- poses and scenes of the fit tests -------------------------------------------------------------------------------
def pose(th, tx, ty):
    return np.array([math.cos(th), -math.sin(th), tx, math.sin(th), math.cos(th), ty], np.float64)


def spose(th, s, tx, ty):
    """A similarity transform: rotation th, scale s, translation (tx, ty)."""
    return np.array([s * math.cos(th), -s * math.sin(th), tx, s * math.sin(th), s * math.cos(th), ty], np.float64)


def posed(tmpl, T):
    t = np.asarray(tmpl, np.float64).reshape(4, -1)
    T = np.asarray(T, np.float64)
    return np.stack([T[0] * t[0] + T[1] * t[1] + T[2], T[3] * t[0] + T[4] * t[1] + T[5],
                     T[0] * t[2] + T[1] * t[3] + T[2], T[3] * t[2] + T[4] * t[3] + T[5]]).astype(F32)


def scene_of(lines, D=30, W=400, H=400):
    """A map-like context with zero translation: the lines are in map coordinates already."""
    rec = np.ascontiguousarray(np.asarray(lines, F32).reshape(4, -1).T)
    return SceneLines.of(lines, (0.0, 0.0), table_bins(D, rec), D, W, H)


def pose_errors(T, truth, anchor):
    a = np.array([float(anchor[0]), float(anchor[1]), 1.0])
    T = np.asarray(T, np.float64).reshape(2, 3)
    truth = np.asarray(truth, np.float64).reshape(2, 3)
    rot = math.atan2(T[1, 0], T[0, 0]) - math.atan2(truth[1, 0], truth[0, 0])
    return float(np.hypot(*(T @ a - truth @ a))), abs(math.remainder(rot, 2 * math.pi)), (T @ a - truth @ a)


def scale_error(T, truth):
    T, truth = np.asarray(T, np.float64).reshape(6), np.asarray(truth, np.float64).reshape(6)
    return abs(math.sqrt(T[0] * T[4] - T[1] * T[3]) / math.sqrt(truth[0] * truth[4] - truth[1] * truth[3]) - 1.0)


def house():
    """A closed outline with lines in several directions: every pose parameter is observable."""
    pts = [(0, 0), (60, 0), (60, 40), (30, 65), (0, 40)]
    lines = [(*pts[i], *pts[(i + 1) % len(pts)]) for i in range(len(pts))] + [(10, 10, 25, 30), (45, 8, 52, 30)]
    return np.asarray(lines, F32).T.copy()


def anchor_of(tmpl):
    return fdcm.get_template_anchors([tmpl])[0]


def offset_pose(truth, anchor, dth, dx, dy):
    """truth rotated by dth about its posed anchor, then moved by (dx, dy)."""
    T = np.asarray(truth, np.float64).reshape(2, 3)
    a = T @ np.array([float(anchor[0]), float(anchor[1]), 1.0])
    R = np.array([[math.cos(dth), -math.sin(dth)], [math.sin(dth), math.cos(dth)]])
    M = R @ T[:, :2]
    e = R @ (T[:, 2] - a) + a + np.array([dx, dy])
    return np.array([M[0, 0], M[0, 1], e[0], M[1, 0], M[1, 1], e[1]], F32)


def one_match(T, t=0):
    m = np.zeros(1, _lib.MATCH_DTYPE)
    m["tmpl_idx"], m["transform"] = t, T
    return m


# ---- the map geometry: tiny maps, the exact / literal boundary, scenes far from the origin -------------------------
def pinned_scene(side, n, seed):
    """n random lines in [0, side-1]^2 with lengths 0..side (a third of them on integer coordinates) plus two 1-px lines
    at the corners that pin the extent: at padding 1 the map side is exactly `side`.  Side 1: one point line."""
    if side == 1:
        return np.zeros((4, 1), F32)
    rng = np.random.default_rng(seed)
    p1 = rng.uniform(0, side - 1, (2, n))
    ang = rng.uniform(0, 2 * math.pi, n)
    ln = rng.uniform(0, side, n)
    p2 = np.clip(p1 + ln * np.stack([np.cos(ang), np.sin(ang)]), 0, side - 1)
    lines = np.concatenate([p1, p2])
    lines[:, : n // 3] = np.round(lines[:, : n // 3])
    pins = np.array([[0, 0, 1, 0], [side - 2, side - 1, side - 1, side - 1]], np.float64).T
    return np.ascontiguousarray(np.concatenate([lines, pins], axis=1), F32)


def map_templates(side, seed, n=6):
    """Templates scaled to a map of `side` px: lines of 1..side px about the origin, one template holding a zero-length
    line, one larger than the map (every hypothesis of it is nullopt)."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        k = int(rng.integers(1, 6))
        c = rng.uniform(-side / 4, side / 4, (2, k))
        ang = rng.uniform(0, math.pi, k)
        ln = rng.uniform(1, side, k) if side > 1 else np.ones(k)
        d = 0.5 * ln * np.stack([np.cos(ang), np.sin(ang)])
        out.append(np.ascontiguousarray(np.concatenate([c - d, c + d]), F32))
    out[1] = np.ascontiguousarray(np.concatenate([out[1], np.array([[0.5], [0.25], [0.5], [0.25]], F32)], axis=1), F32)
    big = 2.0 * side + 5.0
    out.append(np.array([[-big / 2, 0, big / 2, 0], [0, -big / 3, 0, big / 3]], F32).T.copy())
    return out


def shifted_scene(scene, shift):
    """The scene in map coordinates, as the host computes it: scene + shift in fp32 (core/math.h:352-354)."""
    return (np.asarray(scene, F32).T.reshape(-1, 2) + np.asarray(shift, F32)).reshape(-1, 4).T.astype(F32)


def host_geometry(scene, padding):
    """scene_centered_translation (host_math.hpp) in fp32: shift = req/2 - (mx+mn)/2, side = ceil(req + 1)."""
    pts = np.asarray(scene, F32).T.reshape(-1, 2)
    mn, mx = pts.min(axis=0), pts.max(axis=0)
    d = (mx - mn).astype(F32)
    req = F32(max(F32(1), F32(padding))) * F32(max(d[0], d[1]))
    shift = (req / F32(2) - (mx + mn) / F32(2)).astype(F32)
    return shift, int(math.ceil(float(req + F32(1))))


# offsets with fractional parts; per offset: the seed of a 3-line scene and (seed, scale) of a synthetic scene whose
# shifted end points leave the map at padding 1.0 (chosen on the CPU, asserted by check_generators)
FAR = {1e3: (1234.56, -987.31), 3e4: (-29999.37, 30123.71), 1e5: (-99999.63, 50000.21)}
FAR_SMALL_SEED = {1e3: 8, 3e4: 0, 1e5: 14}
FAR_SYNTH = {1e3: (104, 1.1), 3e4: (100, 1.2), 1e5: (100, 0.9)}


def far_small_scene(offset, seed):
    """3 random lines within an extent of 50..900 px, moved to the offset."""
    rng = np.random.default_rng(seed)
    ext = rng.uniform(50, 900)
    lines = rng.uniform(0, ext, (4, 3)) + np.array(FAR[offset] * 2, np.float64).reshape(4, 1)
    tmpls = synth_templates(6, 5, max(ext, 100.0), seed=seed + 1, max_len=max(8.0, ext / 4))
    return np.ascontiguousarray(lines, F32), tmpls


def far_synthetic_scene(offset, seed, scale):
    """The 640x480 synthetic scene with planted templates, without its corner lines, scaled and moved to the offset."""
    tmpls = synth_templates(10, 12, 640, seed=seed + 1)
    scene = plant_instances(synth_scene(640, 480, 120, seed=seed)[:, :-2], tmpls, 640, 480, seed=seed + 2)
    scene = scene.astype(np.float64) * scale + np.array(FAR[offset] * 2, np.float64).reshape(4, 1)
    return np.ascontiguousarray(scene, F32), [np.ascontiguousarray(t * F32(scale), F32) for t in tmpls]


def far_scene(offset, source):
    if source == "small":
        return far_small_scene(offset, FAR_SMALL_SEED[offset])
    seed, scale = FAR_SYNTH[offset]
    return far_synthetic_scene(offset, seed, scale)


TINY = [1, 2, 3, 5, 8, 31, 32, 33, 64, 65, 129, 160, 161, 164, 165]
BOUNDARY = [2896, 2897, 2898]
