"""Pose fit (fdcm_fit_matches, PoseFit): the float64 model of the rules in include/fdcm_b200.h and its properties.
tests/test_gpu_fit.py compares the device against this model byte for byte.  No kernel is launched here.

The sums of rule 4 are formed lane by lane in the stated order (np.add.accumulate is sequential); np.sum, np.dot and @
would sum pairwise or with fused multiply-adds and change the bits."""
import ctypes as C
import math
from dataclasses import dataclass

import numpy as np
import pytest

import openfdcm_b200 as fdcm
from openfdcm_b200 import _lib
from tests.test_coverage_host import table_bins
from tests.test_refine_host import valid_poses
from tests.util import F32


# ---- the model -------------------------------------------------------------------------------------------------------
@dataclass
class SceneLines:
    """What the fit reads of a map: its scene lines in map coordinates (float32, as the build stores them), their bins,
    the depth, the scene translation and the map size."""
    lines: np.ndarray      # (J, 4) float32
    bins: np.ndarray       # (J,) int
    D: int
    shift: tuple
    W: int
    H: int

    @classmethod
    def of(cls, scene, shift, bins, D, W, H):
        r = np.ascontiguousarray(np.asarray(scene, F32).reshape(4, -1).T)
        sh = np.asarray(shift, F32)
        lines = np.stack([r[:, 0] + sh[0], r[:, 1] + sh[1], r[:, 2] + sh[0], r[:, 3] + sh[1]], axis=1).astype(F32)
        return cls(lines, np.asarray(bins, np.int64), int(D), (F32(sh[0]), F32(sh[1])), int(W), int(H))


def line_samples(line, step):
    """Rule 2 for one (x1, y1, x2, y2) line: (sx, sy) float64 arrays."""
    x1, y1, x2, y2 = (F32(v) for v in line)
    dx, dy = x2 - x1, y2 - y1
    with np.errstate(all="ignore"):
        ln = np.sqrt(F32(dx * dx + dy * dy))
        if not ln > 0:
            return np.zeros(0), np.zeros(0)
        n = max(2, int(math.ceil(F32(ln / F32(step)))) + 1)
    f = np.arange(n, dtype=np.float64) / float(n - 1)
    return float(x1) + (float(x2) - float(x1)) * f, float(y1) + (float(y2) - float(y1)) * f


def fit_round(P, shift):
    """Rule 1: the float32 rounding F of a pose (m0, m1, m3, m4, ex, ey)."""
    m0, m1, m3, m4, ex, ey = P
    return np.array([F32(m0), F32(m1), F32(ex - float(shift[0])), F32(m3), F32(m4), F32(ey - float(shift[1]))], F32)


def butterfly(lanes):
    """v = v + v[lane ^ o] for o = 16, 8, 4, 2, 1; lane 0's values."""
    v = [list(x) for x in lanes]
    for o in (16, 8, 4, 2, 1):
        v = [[a + b for a, b in zip(v[l], v[l ^ o])] for l in range(32)]
    return v[0]


def correspondences(sc, recs, samples, P, F, anchor, fit):
    """Rules 3 and 4 at pose P (float rounding F): the ten sums after the butterfly, the inlier count and rho^2."""
    m0, m1, m3, m4, ex, ey = P
    ax, ay = float(anchor[0]), float(anchor[1])
    cx, cy = (m0 * ax + m1 * ay) + ex, (m3 * ax + m4 * ay) + ey
    with np.errstate(all="ignore"):
        R = (np.stack([F[0] * recs[:, 0] + F[1] * recs[:, 1], F[3] * recs[:, 0] + F[4] * recs[:, 1],
                       F[0] * recs[:, 2] + F[1] * recs[:, 3], F[3] * recs[:, 2] + F[4] * recs[:, 3]], axis=1).astype(F32))
    bins = table_bins(sc.D, R) if len(recs) else np.zeros(0, np.int64)
    A = sc.lines.astype(np.float64)
    Ax, Ay, dx, dy = A[:, 0], A[:, 1], A[:, 2] - A[:, 0], A[:, 3] - A[:, 1]
    l2 = dx * dx + dy * dy
    md = float(F32(fit.max_distance))
    md2 = md * md
    seqs = [[[] for _ in range(10)] for _ in range(32)]
    n_in, rho2 = 0, 0.0
    for q, (sx, sy) in enumerate(samples):
        if len(sx) == 0:
            continue
        rx, ry = sx - ax, sy - ay
        rho2 = max(rho2, float(np.max(rx * rx + ry * ry)))
        db = np.abs(sc.bins - int(bins[q]))
        cand = np.flatnonzero((np.minimum(db, sc.D - db) <= fit.bin_tolerance) & (l2 > 0))
        if len(cand) == 0:
            continue
        px, py = (m0 * sx + m1 * sy) + ex, (m3 * sx + m4 * sy) + ey
        cAx, cAy, cdx, cdy, cl2 = Ax[cand], Ay[cand], dx[cand], dy[cand], l2[cand]
        u = ((px[:, None] - cAx) * cdx + (py[:, None] - cAy) * cdy) / cl2
        u = np.where(u < 0.0, 0.0, np.where(u > 1.0, 1.0, u))
        ex_, ey_ = px[:, None] - (cAx + u * cdx), py[:, None] - (cAy + u * cdy)
        d2 = ex_ * ex_ + ey_ * ey_
        d2 = np.where(d2 <= md2, d2, np.inf)
        k = np.argmin(d2, axis=1)                    # the first least d2: the least j among equal distances
        hit = np.isfinite(d2[np.arange(len(sx)), k])
        i = np.flatnonzero(hit)
        j = cand[k[i]]
        qx, qy = px[i], py[i]
        l = np.sqrt(dx[j] * dx[j] + dy[j] * dy[j])
        nx, ny = -dy[j] / l, dx[j] / l
        r = nx * (qx - Ax[j]) + ny * (qy - Ay[j])
        jt = ny * (qx - cx) - nx * (qy - cy)
        terms = (nx * nx, nx * ny, nx * jt, ny * ny, ny * jt, jt * jt, nx * r, ny * r, jt * r, r * r)
        lane = i % 32
        for ln in range(32):
            sel = lane == ln
            for s, tv in enumerate(terms):
                seqs[ln][s].append(tv[sel])
        n_in += len(i)
    lanes = [[float(np.add.accumulate(np.concatenate([[0.0]] + seqs[ln][s]))[-1]) for s in range(10)] for ln in range(32)]
    return butterfly(lanes), n_in, rho2, (cx, cy)


def solve(a):
    """Rule 4: the damped Cholesky solve, or None."""
    lam = 1e-9 * ((a[0] + a[3]) + a[5])
    b00, b11, b22 = a[0] + lam, a[3] + lam, a[5] + lam
    if not b00 > 0.0:
        return None
    l00 = math.sqrt(b00)
    l10, l20 = a[1] / l00, a[2] / l00
    r1 = b11 - l10 * l10
    if not r1 > 0.0:
        return None
    l11 = math.sqrt(r1)
    l21 = (a[4] - l20 * l10) / l11
    r2 = (b22 - l20 * l20) - l21 * l21
    if not r2 > 0.0:
        return None
    l22 = math.sqrt(r2)
    y0 = -a[6] / l00
    y1 = (-a[7] - l10 * y0) / l11
    y2 = ((-a[8] - l20 * y0) - l21 * y1) / l22
    dt = y2 / l22
    dy = (y1 - l21 * dt) / l11
    dx = ((y0 - l10 * dy) - l20 * dt) / l00
    return dx, dy, dt


def update(P, c, d):
    """Rule 5: the half-angle rotation about c, then the translation."""
    m0, m1, m3, m4, ex, ey = P
    cx, cy = c
    tau = d[2] * 0.5
    k = 1.0 + tau * tau
    cr, sr = (1.0 - tau * tau) / k, (2.0 * tau) / k
    ux, uy = ex - cx, ey - cy
    return (cr * m0 - sr * m3, cr * m1 - sr * m4, sr * m0 + cr * m3, sr * m1 + cr * m4,
            ((cr * ux - sr * uy) + cx) + d[0], ((sr * ux + cr * uy) + cy) + d[1])


def fit_one(sc, tmpl, anchor, T, fit):
    """Rules 1-6 for one match: (float32 transform, stats tuple, final float64 pose), or None for an invalid input."""
    t = np.asarray(tmpl, F32).reshape(4, -1)
    T = np.asarray(T, F32).reshape(6)
    if t.shape[1] == 0 or sc.D == 0 or not valid_poses(T[None], t, sc.shift, sc.W, sc.H)[0]:
        return None
    recs = np.ascontiguousarray(t.T)
    samples = [line_samples(l, fit.sample_step) for l in recs]
    n_samples = sum(len(s[0]) for s in samples)
    P = (float(T[0]), float(T[1]), float(T[3]), float(T[4]), float(T[2]) + float(sc.shift[0]), float(T[5]) + float(sc.shift[1]))
    F = T.copy()
    iters, at_pose = 0, False
    tol = float(F32(fit.tolerance))
    for _ in range(fit.iterations):
        acc, n_in, rho2, c = correspondences(sc, recs, samples, P, F, anchor, fit)
        at_pose = True
        if n_in < fit.min_inliers:
            break
        d = solve(acc)
        if d is None:
            break
        N = update(P, c, d)
        FN = fit_round(N, sc.shift)
        if not valid_poses(FN[None], t, sc.shift, sc.W, sc.H)[0]:
            break
        P, F, iters, at_pose = N, FN, iters + 1, False
        if max(abs(d[0]), abs(d[1]), abs(d[2]) * math.sqrt(rho2)) <= tol:
            break
    if not at_pose:
        acc, n_in, rho2, c = correspondences(sc, recs, samples, P, F, anchor, fit)
    rms = F32(math.sqrt(acc[9] / n_in)) if n_in > 0 else F32(np.nan)
    return F, (n_samples, n_in, iters, rms), P


def fit_model(sc, tmpls, anchors, matches, fit, score_fn=None, tmpl_idx_base=0):
    """Every match: (MATCH_DTYPE records, FIT_STATS_DTYPE stats).  score_fn(tmpl, F) -> raw float32 score (None: NaN)."""
    out = np.array(matches, _lib.MATCH_DTYPE, copy=True).reshape(-1)
    stats = np.zeros(len(out), _lib.FIT_STATS_DTYPE)
    for i, m in enumerate(out):
        ti = int(m["tmpl_idx"]) - tmpl_idx_base
        r = fit_one(sc, tmpls[ti], anchors[ti], m["transform"], fit)
        if r is None:
            out[i]["score"] = np.nan
            stats[i] = (0, 0, 0, np.nan)
            continue
        out[i]["transform"] = r[0]
        out[i]["score"] = score_fn(tmpls[ti], r[0]) if score_fn else np.nan
        stats[i] = r[1]
    return out, stats


# ---- helpers of the property tests -----------------------------------------------------------------------------------
def pose(th, tx, ty):
    return np.array([math.cos(th), -math.sin(th), tx, math.sin(th), math.cos(th), ty], np.float64)


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


# ---- the tests -------------------------------------------------------------------------------------------------------
def test_struct_layouts_match_the_header():
    assert C.sizeof(_lib.FitParams) == 24
    assert [f[0] for f in _lib.FitParams._fields_] == ["iterations", "max_distance", "sample_step", "bin_tolerance", "tolerance",
                                                      "min_inliers"]
    assert _lib.FIT_STATS_DTYPE.itemsize == 16 and _lib.FIT_STATS_DTYPE.names == ("n_samples", "n_inliers", "iterations", "rms")
    f = fdcm.PoseFit()
    assert (f.iterations, f.max_distance, f.sample_step, f.bin_tolerance, f.tolerance, f.min_inliers) == (10, 3.0, 2.0, 1, 1e-3, 6)


def hook_samples(lines, step):
    rec = np.ascontiguousarray(np.asarray(lines, F32).reshape(-1, 4))
    n = C.c_int64(0)
    _lib.lib().fdcm_fit_samples(_lib.ptr(rec), rec.shape[0], step, None, 0, C.byref(n))
    out = np.zeros((max(n.value, 1), 2), np.float64)
    _lib.check(_lib.lib().fdcm_fit_samples(_lib.ptr(rec), rec.shape[0], step, _lib.ptr(out), n.value, C.byref(n)))
    return out[: n.value]


def test_fit_samples_hook_equals_the_model():
    rng = np.random.default_rng(5)
    lines = np.concatenate([
        np.array([[0, 0, 10, 0],            # len 10, step 2: n = 6 (an exact multiple)
                  [3, 3, 3, 3],             # zero length: no samples
                  [1, 1, 1, 9],             # len 8, step 2: n = 5
                  [0.5, 0.25, 7.3, 9.1],
                  [-4, 2, -4.0000005, 2]], F32),
        rng.uniform(-300, 300, (40, 4)).astype(F32)])
    for step in (0.5, 1.0, 2.0, 3.7, 1e30):
        want = [np.stack(line_samples(l, step), axis=1) for l in lines]
        got = hook_samples(lines, step)
        want = np.concatenate(want)
        assert got.shape == want.shape and got.tobytes() == want.tobytes()
    assert len(line_samples([0, 0, 10, 0], 2.0)[0]) == 6 and len(line_samples([3, 3, 3, 3], 2.0)[0]) == 0
    assert len(line_samples([0, 0, 10, 0], 1e30)[0]) == 2
    s = hook_samples([[0, 0, 10, 0]], 2.0)
    assert s[:, 0].tolist() == [0.0, 2.0, 4.0, 6.0, 8.0, 10.0] and (s[:, 1] == 0).all()
    n = C.c_int64(0)
    assert _lib.lib().fdcm_fit_samples(_lib.ptr(lines), len(lines), 2.0, None, 0, C.byref(n)) == _lib.FDCM_ERR_CAPACITY
    assert _lib.lib().fdcm_fit_samples(_lib.ptr(lines), len(lines), 0.25, None, 0, C.byref(n)) == _lib.FDCM_ERR_INVALID


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_model_recovers_the_exact_pose_of_noise_free_lines(seed):
    rng = np.random.default_rng(seed)
    tmpl = house()
    a = anchor_of(tmpl)
    truth = pose(rng.uniform(-math.pi, math.pi), rng.uniform(150, 250), rng.uniform(150, 250))
    sc = scene_of(posed(tmpl, truth))
    ang = rng.choice([-1, 1]) * 0.03
    d = rng.normal(size=2)
    d = 2.0 * d / np.hypot(*d)
    start = offset_pose(truth, a, ang, d[0], d[1])
    out, st = fit_model(sc, [tmpl], [a], one_match(start), fdcm.PoseFit())
    e_a, e_r, _ = pose_errors(out[0]["transform"], truth, a)
    assert e_a < 0.01 and e_r < 1e-4, (e_a, e_r, st)
    assert st[0]["n_inliers"] == st[0]["n_samples"] and st[0]["iterations"] >= 2 and st[0]["rms"] < 0.01


def test_model_recovers_the_pose_on_cut_scene_lines():
    """Every scene line cut into 2-3 pieces with gaps: the samples over a gap have no correspondence (or one at a piece's
    end), the rest still determine the pose."""
    rng = np.random.default_rng(11)
    tmpl = house()
    a = anchor_of(tmpl)
    truth = pose(0.7, 200.0, 190.0)
    full = posed(tmpl, truth).T.astype(np.float64)
    pieces = []
    for x1, y1, x2, y2 in full:
        k = int(rng.integers(2, 4))
        cuts = np.sort(rng.uniform(0.15, 0.85, k - 1))
        edges = [0.0] + [v for c in cuts for v in (c - 0.04, c + 0.04)] + [1.0]
        for u0, u1 in zip(edges[::2], edges[1::2]):
            pieces.append((x1 + (x2 - x1) * u0, y1 + (y2 - y1) * u0, x1 + (x2 - x1) * u1, y1 + (y2 - y1) * u1))
    sc = scene_of(np.asarray(pieces, F32).T)
    start = offset_pose(truth, a, -0.03, 1.2, -1.6)
    out, st = fit_model(sc, [tmpl], [a], one_match(start), fdcm.PoseFit(iterations=20))
    e_a, e_r, _ = pose_errors(out[0]["transform"], truth, a)
    assert e_a < 0.01 and e_r < 1e-4, (e_a, e_r, st)
    assert st[0]["n_inliers"] >= st[0]["n_samples"] // 2


def test_model_does_not_slide_a_template_of_parallel_lines():
    """Parallel lines leave the translation along them unobserved: g has no component there and the damping keeps the
    step out of that direction."""
    th = 0.4
    u = np.array([math.cos(th), math.sin(th)])
    tmpl = np.array([[0, 0, 80, 0], [0, 15, 80, 15], [0, 40, 80, 40]], F32).T.copy()
    a = anchor_of(tmpl)
    truth = pose(th, 180.0, 170.0)
    sc = scene_of(posed(tmpl, truth))
    for dth, perp in ((0.0, 1.5), (0.02, -1.0)):
        n = np.array([-u[1], u[0]])
        start = offset_pose(truth, a, dth, *(perp * n + 3.0 * u))   # 3 px along the lines, `perp` across
        out, st = fit_model(sc, [tmpl], [a], one_match(start), fdcm.PoseFit())
        _, e_r, off = pose_errors(out[0]["transform"], truth, a)
        assert abs(float(off @ n)) < 0.01 and e_r < 1e-4 and st[0]["iterations"] >= 1
        # the float64 pose state, before the float32 rounding of the output (1.5e-5 px at these coordinates)
        m0, m1, m3, m4, ex, ey = fit_one(sc, tmpl, a, start, fdcm.PoseFit())[2]
        ax, ay = float(a[0]), float(a[1])
        moved = np.array([(m0 * ax + m1 * ay) + ex, (m3 * ax + m4 * ay) + ey])
        T0 = start.astype(np.float64)
        start_anchor = np.array([(T0[0] * ax + T0[1] * ay) + T0[2], (T0[3] * ax + T0[4] * ay) + T0[5]])
        # started parallel, the step has no component along the lines; started 0.02 rad off, the first steps are normal to
        # the posed lines, which are not yet parallel to the scene's
        assert abs(float((moved - start_anchor) @ u)) < (1e-6 if dth == 0.0 else 2.0 * math.sin(abs(dth))), moved - start_anchor


def test_model_edge_cases():
    tmpl = house()
    a = anchor_of(tmpl)
    truth = pose(0.3, 200.0, 200.0)
    sc = scene_of(posed(tmpl, truth))
    fit = fdcm.PoseFit()
    # invalid inputs come back unchanged with score NaN and stats {0, 0, 0, NaN}
    bad = np.concatenate([one_match(truth.astype(F32)), one_match([np.nan, 0, 200, 0, 1, 200]), one_match([1, 0, 1e5, 0, 1, 0]),
                          one_match(truth.astype(F32), t=1)])
    out, st = fit_model(sc, [tmpl, np.zeros((4, 0), F32)], [a, (0.0, 0.0)], bad, fit)
    assert np.array_equal(out[1:]["transform"].view(np.uint32), bad[1:]["transform"].view(np.uint32))
    assert np.isnan(out[1:]["score"]).all() and st[1:]["n_samples"].tolist() == [0, 0, 0] and np.isnan(st[1:]["rms"]).all()
    # no scene line within max_distance: no update, the input transform itself
    far = offset_pose(truth, a, 0.0, 100.0, 0.0)
    out, st = fit_model(sc, [tmpl], [a], one_match(far), fit)
    assert out[0]["transform"].tobytes() == far.tobytes() and st[0]["iterations"] == 0 and st[0]["n_inliers"] < 6
    # a pose at the map border whose update would leave the map stops at the last valid pose
    edge = scene_of(posed(tmpl, pose(0.0, -1.0, 100.0)), W=400, H=400)   # the instance sticks out of the map by 1 px
    start = np.array([1, 0, 0.0, 0, 1, 100.0], F32)
    out, st = fit_model(edge, [tmpl], [a], one_match(start), fit)
    assert valid_poses(out["transform"], tmpl, edge.shift, edge.W, edge.H)[0] and out[0]["transform"][2] >= 0.0


@pytest.mark.parametrize("bad", [dict(iterations=0), dict(iterations=101), dict(max_distance=0.0), dict(max_distance=16.5),
                                 dict(max_distance=math.nan), dict(sample_step=0.4), dict(sample_step=math.inf),
                                 dict(bin_tolerance=-1), dict(bin_tolerance=33), dict(tolerance=-1e-3), dict(tolerance=math.nan),
                                 dict(min_inliers=2)])
def test_fit_matches_rejects_bad_parameters_before_any_device_work(bad):
    f = fdcm.PoseFit(**bad)
    st = _lib.lib().fdcm_fit_matches(None, None, 0, 0, 0.0, C.byref(f._params()), None, 0, None, None)
    assert st == _lib.FDCM_ERR_INVALID
    msg = _lib.lib().fdcm_last_error().decode()
    assert "pose fit" in msg, msg


def test_cpp_fit_matches_builds(tmp_path):
    """fitMatches of include/openfdcm_b200/openfdcm_cuda.hpp compiles and links."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "fit.cpp"
    src.write_text(r'''
#include "openfdcm_b200/openfdcm_cuda.hpp"
#include <cstdio>
int main() {
    using namespace openfdcm::cuda;
    try {
        const LineArray scene{0.f, 0.f, 50.f, 0.f, 50.f, 0.f, 50.f, 40.f};
        const std::vector<LineArray> templates{LineArray{0.f, 0.f, 20.f, 0.f}};
        const Dt3Cuda fm = buildCudaFeaturemap(scene, Dt3CudaParameters{});
        const auto a = searchTopK(DefaultSearch{4, 4}, BatchOptimize{10}, ExponentialPenalty{1.5f}, fm, templates, scene, 5);
        const PoseFit fit{};
        const std::vector<Match> b = fitMatches(fm, templates, a, fit);
        std::vector<FitStats> stats;
        const std::vector<Match> c = fitMatches(fm, templates, a, PoseFit{5, 2.f, 1.f, 1, 1e-3f, 6}, &stats);
        std::printf("%zu %zu %zu %zu\n", a.size(), b.size(), c.size(), stats.size());
    } catch (const std::exception& e) {
        std::printf("%s\n", e.what());
        return 1;
    }
    return 0;
}
''')
    exe = tmp_path / "fit"
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Werror", "-I" + os.path.join(root, "include"), str(src),
                           "-L" + os.path.join(root, "openfdcm_b200"), "-lfdcm_b200", "-Wl,-rpath," + os.path.join(root, "openfdcm_b200"),
                           "-o", str(exe)])
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode in (0, 1) and r.stdout
