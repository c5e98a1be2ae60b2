"""Pose fit (fdcm_fit_matches, PoseFit; fdcm_fit_matches_scaled, PoseFit(scale_range=...)): the float64 model of the rules
in include/fdcm_b200.h.  Like fit_eval_kernel<kScaled>, one model serves both fits: with fit.scale_range set it forms
five more sums, solves for the scale as well (rules 4' and 5') and keeps the scale inside the range.

The sums of rule 4 are formed lane by lane in the stated order (np.add.accumulate is sequential); np.sum, np.dot and @
would sum pairwise or with fused multiply-adds and change the bits."""
import math
from dataclasses import dataclass

import numpy as np

from openfdcm_b200 import _lib
from tests.models.coverage import table_bins
from tests.models.refine import valid_poses
from tests.util import F32


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


def sigma_of(P):
    """The scale sqrt(m0 m4 - m1 m3) of a pose (m0, m1, m3, m4, ...)."""
    m0, m1, m3, m4 = P[0], P[1], P[2], P[3]
    with np.errstate(all="ignore"):
        return float(np.sqrt(np.float64(m0 * m4 - m1 * m3)))


def correspondences(sc, recs, samples, P, F, anchor, fit):
    """Rules 3 and 4 (4') at pose P (float rounding F): the ten (fifteen) sums after the butterfly, the inlier count, rho^2
    and the centre."""
    scaled = fit.scale_range is not None
    n_sums = 15 if scaled else 10
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
    seqs = [[[] for _ in range(n_sums)] for _ in range(32)]
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
        if scaled:
            js = nx * (qx - cx) + ny * (qy - cy)
            terms = (nx * nx, nx * ny, nx * jt, nx * js, ny * ny, ny * jt, ny * js, jt * jt, jt * js, js * js,
                     nx * r, ny * r, jt * r, js * r, r * r)
        else:
            terms = (nx * nx, nx * ny, nx * jt, ny * ny, ny * jt, jt * jt, nx * r, ny * r, jt * r, r * r)
        lane = i % 32
        for ln in range(32):
            sel = lane == ln
            for s, tv in enumerate(terms):
                seqs[ln][s].append(tv[sel])
        n_in += len(i)
    lanes = [[float(np.add.accumulate(np.concatenate([[0.0]] + seqs[ln][s]))[-1]) for s in range(n_sums)] for ln in range(32)]
    return butterfly(lanes), n_in, rho2, (cx, cy)


def solve3(a):
    """Rule 4: the damped 3x3 Cholesky solve -> (dx, dy, dth), or None."""
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


def solve4(a):
    """Rule 4': the damped 4x4 Cholesky solve in the header's order -> (dx, dy, dth, ds), or None."""
    lam = 1e-9 * (((a[0] + a[4]) + a[7]) + a[9])
    b00, b11, b22, b33 = a[0] + lam, a[4] + lam, a[7] + lam, a[9] + lam
    if not b00 > 0.0:
        return None
    l00 = math.sqrt(b00)
    l10, l20, l30 = a[1] / l00, a[2] / l00, a[3] / l00
    r1 = b11 - l10 * l10
    if not r1 > 0.0:
        return None
    l11 = math.sqrt(r1)
    l21, l31 = (a[5] - l20 * l10) / l11, (a[6] - l30 * l10) / l11
    r2 = (b22 - l20 * l20) - l21 * l21
    if not r2 > 0.0:
        return None
    l22 = math.sqrt(r2)
    l32 = ((a[8] - l30 * l20) - l31 * l21) / l22
    r3 = ((b33 - l30 * l30) - l31 * l31) - l32 * l32
    if not r3 > 0.0:
        return None
    l33 = math.sqrt(r3)
    y0 = -a[10] / l00
    y1 = (-a[11] - l10 * y0) / l11
    y2 = ((-a[12] - l20 * y0) - l21 * y1) / l22
    y3 = (((-a[13] - l30 * y0) - l31 * y1) - l32 * y2) / l33
    ds = y3 / l33
    dt = (y2 - l32 * ds) / l22
    dy = ((y1 - l21 * dt) - l31 * ds) / l11
    dx = (((y0 - l10 * dy) - l20 * dt) - l30 * ds) / l00
    return dx, dy, dt, ds


def update(P, c, d):
    """Rule 5 (5'): the half-angle rotation (and, with a fourth component ds, the scale step) about c, then the
    translation."""
    m0, m1, m3, m4, ex, ey = P
    cx, cy = c
    tau = d[2] * 0.5
    k = 1.0 + tau * tau
    cr, sr = (1.0 - tau * tau) / k, (2.0 * tau) / k
    if len(d) == 4:
        f = 1.0 + d[3]
        cr, sr = f * cr, f * sr
    ux, uy = ex - cx, ey - cy
    return (cr * m0 - sr * m3, cr * m1 - sr * m4, sr * m0 + cr * m3, sr * m1 + cr * m4,
            ((cr * ux - sr * uy) + cx) + d[0], ((sr * ux + cr * uy) + cy) + d[1])


def fit_one(sc, tmpl, anchor, T, fit):
    """Rules 1-6 (with 4' and 5' when fit.scale_range is set) for one match: (float32 transform, stats tuple, final float64
    pose), or None for an invalid input."""
    scaled = fit.scale_range is not None
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
        d = solve4(acc) if scaled else solve3(acc)
        if d is None:
            break
        N = update(P, c, d)
        if scaled:
            sig_n = sigma_of(N)
            if not (sig_n >= float(F32(fit.scale_range[0])) and sig_n <= float(F32(fit.scale_range[1]))):
                break
            sigma = sigma_of(P)
        FN = fit_round(N, sc.shift)
        if not valid_poses(FN[None], t, sc.shift, sc.W, sc.H)[0]:
            break
        P, F, iters, at_pose = N, FN, iters + 1, False
        if scaled:
            rho = math.sqrt(rho2)
            ad0, ad1, adt, ads = abs(d[0]), abs(d[1]), (abs(d[2]) * sigma) * rho, (abs(d[3]) * sigma) * rho
            s01 = ad0 if ad0 > ad1 else ad1
            sts = adt if adt > ads else ads
            done = (s01 if s01 > sts else sts) <= tol
        else:
            done = max(abs(d[0]), abs(d[1]), abs(d[2]) * math.sqrt(rho2)) <= tol
        if done:
            break
    if not at_pose:
        acc, n_in, rho2, c = correspondences(sc, recs, samples, P, F, anchor, fit)
    rms = F32(math.sqrt(acc[-1] / n_in)) if n_in > 0 else F32(np.nan)
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
