"""Scale as a pose dimension (fdcm_search_dense_scales, ScaleGrid; fdcm_fit_matches_scaled, PoseFit(scale_range=...)): the
numpy model of the scaled dense grid and the float64 model of the scaled fit, the host hook fdcm_dense_scaled_poses against
the model bit for bit, and parameter rejection.  The rules are in include/fdcm_b200.h; tests/test_gpu_scale.py compares the
device against these models.  No kernel is launched here."""
import ctypes as C
import math

import numpy as np
import pytest

import openfdcm_b200 as fdcm
from openfdcm_b200 import _lib
from openfdcm_b200._lib import MATCH_DTYPE
from tests.test_coverage_host import table_bins
from tests.test_dense_host import grid, grid_valid, hook, rot_table, rotate_template
from tests.test_fit_host import (anchor_of, butterfly, fit_round, house, line_samples, one_match, pose_errors, posed,
                                 scene_of)
from tests.test_refine_host import valid_poses
from tests.test_select_host import PI_F32
from tests.util import F32


# ---- the model of the scaled dense grid ------------------------------------------------------------------------------
def scale_values(g):
    """Rule 1: s_k = (float)((double)scale_start * pow((double)scale_ratio, k)) of the float32 parameters."""
    st, ra = float(F32(g.start)), float(F32(g.ratio))
    return np.array([F32(st * math.pow(ra, k)) for k in range(g.scales)], F32)


def scaled_table(d, g):
    """Rule 1: (a, b) of every (k, r), arrays of shape (S, R)."""
    th = [float(F32(d.rot_start)) + r * float(F32(d.rot_step)) for r in range(d.rotations)]
    s = scale_values(g).astype(np.float64)
    a = np.array([[F32(sk * math.cos(x)) for x in th] for sk in s], F32)
    b = np.array([[F32(sk * math.sin(x)) for x in th] for sk in s], F32)
    return a, b


def scaled_poses(d, g, anchor, shift, W, H, k, r):
    """Dense rule 3 with (a_kr, b_kr): the (ny * nx, 6) transforms of scale k and rotation r in grid order."""
    lx, ly, nx, ny = grid(d, shift, W, H)
    A, B = scaled_table(d, g)
    a, b = A[k, r], B[k, r]
    ax, ay, sx, sy = F32(anchor[0]), F32(anchor[1]), F32(shift[0]), F32(shift[1])
    gx = (lx + np.arange(nx, dtype=np.int64) * d.stride).astype(F32)
    gy = (ly + np.arange(ny, dtype=np.int64) * d.stride).astype(F32)
    P = np.empty((ny, nx, 6), F32)
    with np.errstate(all="ignore"):
        P[..., 0], P[..., 1], P[..., 3], P[..., 4] = a, -b, b, a
        P[..., 2] = ((gx - sx) - (a * ax - b * ay))[None, :]
        P[..., 5] = ((gy - sy) - (b * ax + a * ay))[:, None]
    return P.reshape(-1, 6)


def scaled_records(tmpls, anchors, d, g, shift, W, H, score_fn, tmpl_idx_base=0):
    """Rules 1-2: every record h = ((((t S + k) R + r) cells_y + cv) cells_x + cu) with its valid flag, raw score and grid
    scale.  score_fn(Rt (L, 4), translations (n, 2)) -> float32 scores."""
    lx, ly, nx, ny = grid(d, shift, W, H)
    cx, cy = -(-nx // d.cell), -(-ny // d.cell)
    S, R = g.scales, d.rotations
    n = len(tmpls) * S * R * cx * cy
    rec, valid, rs = np.zeros(n, MATCH_DTYPE), np.zeros(n, bool), np.zeros(n, F32)
    if n == 0:
        return rec, valid, rs
    A, B = scaled_table(d, g)
    sv = scale_values(g)
    cell_of = ((np.arange(ny) // d.cell)[:, None] * cx + (np.arange(nx) // d.cell)[None, :]).reshape(-1)
    for t, tmpl in enumerate(tmpls):
        if np.asarray(tmpl).reshape(4, -1).shape[1] == 0:
            continue
        for k in range(S):
            for r in range(R):
                P = scaled_poses(d, g, anchors[t], shift, W, H, k, r)
                Rt = rotate_template(tmpl, A[k, r], B[k, r])
                gi = np.flatnonzero(grid_valid(Rt, P, shift, W, H, nx, ny))
                if not len(gi):
                    continue
                sc = np.asarray(score_fn(Rt, P[gi][:, [2, 5]]), F32)
                key = np.where(np.isnan(sc), np.inf, sc.astype(np.float64))
                cells = cell_of[gi]
                order = np.lexsort((gi, key, cells))
                first = order[np.r_[True, cells[order][1:] != cells[order][:-1]]]
                h = ((t * S + k) * R + r) * cx * cy + cells[first]
                rec["tmpl_idx"][h] = t + tmpl_idx_base
                rec["score"][h] = sc[first]
                rec["transform"][h] = P[gi[first]]
                valid[h] = True
                rs[h] = sv[k]
    return rec, valid, rs


def scaled_penalised(rec, valid, g, lengths, penalty, d, tmpl_idx_base=0):
    """Rule 3: the score of a record of (t, k) divided by the penalty denominator of len_t * s_k (fp32 product)."""
    if penalty is None:
        return rec
    sv = scale_values(g)
    per_k = len(rec) // (len(lengths) * g.scales) if len(lengths) else 0
    h = np.flatnonzero(valid)
    tk = h // per_k                                     # t * S + k
    scaled_len = (np.asarray(lengths, F32)[:, None] * sv[None, :]).astype(F32).reshape(-1)
    p = rec[h].copy()
    p["tmpl_idx"] = tk
    p = fdcm.penalize(penalty, p, scaled_len)
    p["tmpl_idx"] = rec[h]["tmpl_idx"]
    out = rec.copy()
    out[h] = p
    return out


def scaled_select_model(rec, rs, anchors, k, max_per_template=0, radius=0.0, max_angle=math.pi, across_templates=False, tmpl_idx_base=0):
    """Rule 4: fdcm_search_select's walk with the angle test Ta0*Tb0 + Ta3*Tb3 >= cos_thr * (s_a * s_b); positions in
    acceptance order."""
    n = len(rec)
    score = rec["score"].astype(F32)
    score = np.where(np.isnan(score), F32(np.inf), score)
    order = np.lexsort((np.arange(n), score))
    tmpl = rec["tmpl_idx"].astype(np.int64) - tmpl_idx_base
    T = rec["transform"].astype(F32).reshape(n, 6)
    a = np.asarray(anchors, F32).reshape(-1, 2)[tmpl] if n else np.zeros((0, 2), F32)
    px = (T[:, 0] * a[:, 0] + T[:, 1] * a[:, 1]) + T[:, 2]
    py = (T[:, 3] * a[:, 0] + T[:, 4] * a[:, 1]) + T[:, 5]
    radius_on = F32(radius) > 0
    r2 = F32(radius) * F32(radius)
    any_angle = F32(max_angle) >= PI_F32
    cos_thr = F32(math.cos(float(F32(max_angle))))
    acc, count = [], {}
    for b in order:
        if len(acc) == k:
            break
        tb = int(tmpl[b])
        if max_per_template and count.get(tb, 0) >= max_per_template:
            continue
        if radius_on and acc:
            A = np.asarray(acc)
            if not across_templates:
                A = A[tmpl[A] == tb]
            if len(A):
                dx, dy = px[A] - px[b], py[A] - py[b]
                near = (dx * dx + dy * dy) <= r2
                if not any_angle:
                    near &= (T[A, 0] * T[b, 0] + T[A, 3] * T[b, 3]) >= cos_thr * (rs[A] * rs[b])
                if near.any():
                    continue
        acc.append(b)
        count[tb] = count.get(tb, 0) + 1
    return np.asarray(acc, np.int64)


def scaled_output_model(rec, valid, rs, k, anchors=None, select=None, tmpl_idx_base=0):
    """Dense rule 6 on the scaled records: the top k in (score, h) order, or the scaled walk."""
    sub, srs = rec[valid], rs[valid]
    if select is None:
        s = sub["score"].astype(F32)
        s = np.where(np.isnan(s), F32(np.inf), s)
        return sub[np.lexsort((np.arange(len(sub)), s))[:k]]
    return sub[scaled_select_model(sub, srs, anchors, k, select.max_per_template, select.radius, select.max_angle, select.across_templates,
                                   tmpl_idx_base)]


def scaled_hook(d, g, anchor, shift, W, H, k, r, capacity=None):
    """fdcm_dense_scaled_poses -> (status, transforms (n, 6), n, (nx, ny))."""
    lx, ly, nx, ny = grid(d, shift, W, H)
    cap = nx * ny if capacity is None else capacity
    out = np.zeros((max(cap, 1), 6), F32)
    n, wh = C.c_int64(-1), np.zeros(2, np.int32)
    a, sh = np.ascontiguousarray(anchor, F32), np.ascontiguousarray(shift, F32)
    st = _lib.lib().fdcm_dense_scaled_poses(C.byref(d._params()), C.byref(g._params()), _lib.ptr(a), _lib.ptr(sh), W, H, k, r, _lib.ptr(out),
                                            cap, C.byref(n), _lib.ptr(wh))
    return st, out[: max(n.value, 0)], n.value, tuple(wh.tolist())


# ---- the float64 model of the scaled fit -----------------------------------------------------------------------------
def sigma_of(P):
    m0, m1, m3, m4 = P[0], P[1], P[2], P[3]
    with np.errstate(all="ignore"):
        return float(np.sqrt(np.float64(m0 * m4 - m1 * m3)))


def correspondences_scaled(sc, recs, samples, P, F, anchor, fit):
    """Rules 3 and 4' at pose P: the fifteen sums after the butterfly, the inlier count, rho^2 and the centre."""
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
    seqs = [[[] for _ in range(15)] for _ in range(32)]
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
        k = np.argmin(d2, axis=1)
        i = np.flatnonzero(np.isfinite(d2[np.arange(len(sx)), k]))
        j = cand[k[i]]
        qx, qy = px[i], py[i]
        l = np.sqrt(dx[j] * dx[j] + dy[j] * dy[j])
        nx, ny = -dy[j] / l, dx[j] / l
        r = nx * (qx - Ax[j]) + ny * (qy - Ay[j])
        jt = ny * (qx - cx) - nx * (qy - cy)
        js = nx * (qx - cx) + ny * (qy - cy)
        terms = (nx * nx, nx * ny, nx * jt, nx * js, ny * ny, ny * jt, ny * js, jt * jt, jt * js, js * js,
                 nx * r, ny * r, jt * r, js * r, r * r)
        lane = i % 32
        for ln in range(32):
            sel = lane == ln
            for s, tv in enumerate(terms):
                seqs[ln][s].append(tv[sel])
        n_in += len(i)
    lanes = [[float(np.add.accumulate(np.concatenate([[0.0]] + seqs[ln][s]))[-1]) for s in range(15)] for ln in range(32)]
    return butterfly(lanes), n_in, rho2, (cx, cy)


def solve_scaled(a):
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


def update_scaled(P, c, d):
    """Rule 5': the half-angle rotation and the scale step about c, then the translation."""
    m0, m1, m3, m4, ex, ey = P
    cx, cy = c
    tau = d[2] * 0.5
    k = 1.0 + tau * tau
    cr, sr = (1.0 - tau * tau) / k, (2.0 * tau) / k
    f = 1.0 + d[3]
    cr, sr = f * cr, f * sr
    ux, uy = ex - cx, ey - cy
    return (cr * m0 - sr * m3, cr * m1 - sr * m4, sr * m0 + cr * m3, sr * m1 + cr * m4,
            ((cr * ux - sr * uy) + cx) + d[0], ((sr * ux + cr * uy) + cy) + d[1])


def fit_one_scaled(sc, tmpl, anchor, T, fit):
    """Rules 1-6 with 4' and 5' for one match: (float32 transform, stats tuple, final float64 pose), or None."""
    lo, hi = float(F32(fit.scale_range[0])), float(F32(fit.scale_range[1]))
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
        acc, n_in, rho2, c = correspondences_scaled(sc, recs, samples, P, F, anchor, fit)
        at_pose = True
        if n_in < fit.min_inliers:
            break
        d = solve_scaled(acc)
        if d is None:
            break
        N = update_scaled(P, c, d)
        sig_n = sigma_of(N)
        if not (sig_n >= lo and sig_n <= hi):
            break
        sigma = sigma_of(P)
        FN = fit_round(N, sc.shift)
        if not valid_poses(FN[None], t, sc.shift, sc.W, sc.H)[0]:
            break
        P, F, iters, at_pose = N, FN, iters + 1, False
        rho = math.sqrt(rho2)
        ad0, ad1, adt, ads = abs(d[0]), abs(d[1]), (abs(d[2]) * sigma) * rho, (abs(d[3]) * sigma) * rho
        s01 = ad0 if ad0 > ad1 else ad1
        sts = adt if adt > ads else ads
        if (s01 if s01 > sts else sts) <= tol:
            break
    if not at_pose:
        acc, n_in, rho2, c = correspondences_scaled(sc, recs, samples, P, F, anchor, fit)
    rms = F32(math.sqrt(acc[14] / n_in)) if n_in > 0 else F32(np.nan)
    return F, (n_samples, n_in, iters, rms), P


def fit_model_scaled(sc, tmpls, anchors, matches, fit, score_fn=None, tmpl_idx_base=0):
    """Every match: (MATCH_DTYPE records, FIT_STATS_DTYPE stats).  score_fn(tmpl, F) -> raw float32 score."""
    out = np.array(matches, MATCH_DTYPE, copy=True).reshape(-1)
    stats = np.zeros(len(out), _lib.FIT_STATS_DTYPE)
    for i, m in enumerate(out):
        ti = int(m["tmpl_idx"]) - tmpl_idx_base
        r = fit_one_scaled(sc, tmpls[ti], anchors[ti], m["transform"], fit)
        if r is None:
            out[i]["score"] = np.nan
            stats[i] = (0, 0, 0, np.nan)
            continue
        out[i]["transform"] = r[0]
        out[i]["score"] = score_fn(tmpls[ti], r[0]) if score_fn else np.nan
        stats[i] = r[1]
    return out, stats


def spose(th, s, tx, ty):
    """A similarity transform: rotation th, scale s, translation (tx, ty)."""
    return np.array([s * math.cos(th), -s * math.sin(th), tx, s * math.sin(th), s * math.cos(th), ty], np.float64)


def scale_error(T, truth):
    T, truth = np.asarray(T, np.float64).reshape(6), np.asarray(truth, np.float64).reshape(6)
    return abs(math.sqrt(T[0] * T[4] - T[1] * T[3]) / math.sqrt(truth[0] * truth[4] - truth[1] * truth[3]) - 1.0)


def offset_similarity(truth, anchor, dth, ds, dx, dy):
    """truth rotated by dth and scaled by (1 + ds) about its posed anchor, then moved by (dx, dy)."""
    T = np.asarray(truth, np.float64).reshape(2, 3)
    a = T @ np.array([float(anchor[0]), float(anchor[1]), 1.0])
    R = (1.0 + ds) * np.array([[math.cos(dth), -math.sin(dth)], [math.sin(dth), math.cos(dth)]])
    M = R @ T[:, :2]
    e = R @ (T[:, 2] - a) + a + np.array([dx, dy])
    return np.array([M[0, 0], M[0, 1], e[0], M[1, 0], M[1, 1], e[1]], F32)


# ---- the tests -------------------------------------------------------------------------------------------------------
def test_struct_layouts_match_the_header():
    assert C.sizeof(_lib.ScaleGridParams) == 12
    assert [(f, getattr(_lib.ScaleGridParams, f).offset) for f, _ in _lib.ScaleGridParams._fields_] == [
        ("scales", 0), ("scale_start", 4), ("scale_ratio", 8)]
    assert C.sizeof(_lib.FitScaleParams) == 8
    assert [(f, getattr(_lib.FitScaleParams, f).offset) for f, _ in _lib.FitScaleParams._fields_] == [("min_scale", 0), ("max_scale", 4)]
    # the existing structs keep their layouts
    assert C.sizeof(_lib.DenseParams) == 40 and C.sizeof(_lib.FitParams) == 24
    g = fdcm.ScaleGrid()
    assert (g.scales, g.start, g.ratio) == (1, 1.0, 1.0)
    assert fdcm.PoseFit().scale_range is None and fdcm.PoseFit(scale_range=(0.5, 2)).scale_range == (0.5, 2.0)
    assert _lib.lib().fdcm_abi_version() == 3


GRIDS = [fdcm.ScaleGrid(1, 1.0, 1.0), fdcm.ScaleGrid(3, 0.85, (1.15 / 0.85) ** 0.5),
         fdcm.ScaleGrid(5, 0.8, (1.25 / 0.8) ** 0.25), fdcm.ScaleGrid(4, 2.5, 0.5), fdcm.ScaleGrid(2, 1.0, 1.1)]


@pytest.mark.parametrize("g", GRIDS, ids=str)
def test_scaled_poses_hook_equals_the_model(g):
    rng = np.random.default_rng(3)
    for d, shift, W, H in ((fdcm.DenseSearch(7, rot_start=0.1, stride=3, cell=4), (12.5, -3.25), 120, 90),
                           (fdcm.DenseSearch(1, rot_start=0.0, stride=1, cell=2), (0.0, 0.0), 40, 30),
                           (fdcm.DenseSearch(12, stride=5, cell=1, roi=(-10.0, 5.5, 60.0, 70.0)), (20.0, 10.0), 100, 100)):
        anchor = rng.uniform(-30, 30, 2).astype(F32)
        for k in range(g.scales):
            for r in range(d.rotations):
                st, got, n, wh = scaled_hook(d, g, anchor, shift, W, H, k, r)
                assert st == 0, _lib.lib().fdcm_last_error()
                want = scaled_poses(d, g, anchor, shift, W, H, k, r)
                assert got.tobytes() == want.tobytes(), (g, d, k, r)
                assert wh == grid(d, shift, W, H)[2:]


def test_scale_one_equals_the_unscaled_grid():
    """With s_k == 1.0f the table is (c_r, s_r) bit for bit, so the poses are fdcm_dense_poses's."""
    d = fdcm.DenseSearch(24, rot_start=0.3, stride=2, cell=3)
    c, s = rot_table(d)
    for g in (fdcm.ScaleGrid(), fdcm.ScaleGrid(1, 1.0, 7.0), fdcm.ScaleGrid(3, 1.0, 1.5)):
        A, B = scaled_table(d, g)
        assert A[0].tobytes() == c.tobytes() and B[0].tobytes() == s.tobytes()
        for r in range(d.rotations):
            st0, p0, _, _ = hook(d, (3.5, -2.0), (7.0, 4.0), 64, 48, r)
            st1, p1, _, _ = scaled_hook(d, g, (3.5, -2.0), (7.0, 4.0), 64, 48, 0, r)
            assert st0 == st1 == 0 and p0.tobytes() == p1.tobytes()
    # the identity slice uses the end points as given, like the unscaled theta = 0 slice
    d1 = fdcm.DenseSearch(1, rot_start=0.0)
    A, B = scaled_table(d1, fdcm.ScaleGrid())
    assert A[0, 0] == F32(1) and B[0, 0] == F32(0)


def test_scale_values_are_host_double_pow():
    g = fdcm.ScaleGrid(6, 0.7, 1.13)
    want = [F32(float(F32(0.7)) * math.pow(float(F32(1.13)), k)) for k in range(6)]
    assert scale_values(g).tolist() == [float(v) for v in want]
    A, B = scaled_table(fdcm.DenseSearch(1, rot_start=0.0), g)
    assert A[:, 0].tobytes() == scale_values(g).tobytes() and (B == 0).all()


def test_scaled_select_model_reduces_to_the_walk_at_scale_one():
    from tests.test_select_host import select_model
    rng = np.random.default_rng(9)
    n = 200
    rec = np.zeros(n, MATCH_DTYPE)
    rec["tmpl_idx"] = rng.integers(0, 4, n)
    rec["score"] = rng.uniform(0, 10, n).astype(F32)
    th = rng.uniform(-0.5, 0.5, n)
    rec["transform"] = np.stack([np.cos(th), -np.sin(th), rng.uniform(0, 30, n), np.sin(th), np.cos(th), rng.uniform(0, 30, n)], 1)
    anchors = rng.uniform(-5, 5, (4, 2)).astype(F32)
    ones = np.ones(n, F32)
    for kw in (dict(radius=8.0, max_angle=0.2), dict(radius=8.0, max_angle=0.2, across_templates=True), dict(max_per_template=3)):
        assert scaled_select_model(rec, ones, anchors, 20, **kw).tolist() == select_model(rec, anchors, 20, **kw).tolist()
    # at scale 1.2 the rotation column has length 1.2: the threshold scales with the two scales, so the test stays an angle test
    r2 = rec.copy()
    r2["transform"][:, [0, 1, 3, 4]] *= F32(1.2)
    s12 = np.full(n, F32(1.2))
    kw = dict(radius=8.0, max_angle=0.2)
    assert len(scaled_select_model(r2, s12, anchors, 20, **kw)) == len(select_model(rec, anchors, 20, **kw))


BAD_GRIDS = [fdcm.ScaleGrid(0), fdcm.ScaleGrid(65), fdcm.ScaleGrid(2, 0.0, 1.0), fdcm.ScaleGrid(2, -1.0, 1.0), fdcm.ScaleGrid(2, math.nan, 1.0),
             fdcm.ScaleGrid(2, math.inf, 1.0), fdcm.ScaleGrid(2, 1.0, 0.0), fdcm.ScaleGrid(2, 1.0, -2.0), fdcm.ScaleGrid(2, 1.0, math.nan),
             fdcm.ScaleGrid(64, 1.0, 1e10),    # s_k overflows float32
             fdcm.ScaleGrid(64, 1.0, 1e-10)]   # s_k underflows to 0


@pytest.mark.parametrize("g", BAD_GRIDS, ids=str)
def test_bad_scale_grids_are_rejected_before_any_device_work(g):
    d = fdcm.DenseSearch(4)
    st, _, _, _ = scaled_hook(d, g, (0.0, 0.0), (0.0, 0.0), 10, 10, 0, 0, capacity=0)
    assert st == _lib.FDCM_ERR_INVALID
    assert "scale" in _lib.lib().fdcm_last_error().decode()
    n = C.c_int64(7)
    st = _lib.lib().fdcm_search_dense_scales(None, None, C.byref(d._params()), C.byref(g._params()), 0, 0.0, 10, 0, None, None, None, None,
                                             0, C.byref(n))
    assert st == _lib.FDCM_ERR_INVALID


def test_scaled_hook_rejects_bad_arguments():
    d, g = fdcm.DenseSearch(4), fdcm.ScaleGrid(3, 0.9, 1.1)
    for k, r in ((-1, 0), (3, 0), (0, -1), (0, 4)):
        assert scaled_hook(d, g, (0.0, 0.0), (0.0, 0.0), 10, 10, k, r, capacity=100)[0] == _lib.FDCM_ERR_INVALID
    assert scaled_hook(fdcm.DenseSearch(0), g, (0.0, 0.0), (0.0, 0.0), 10, 10, 0, 0, capacity=100)[0] == _lib.FDCM_ERR_INVALID
    st, _, n, _ = scaled_hook(d, g, (0.0, 0.0), (0.0, 0.0), 10, 10, 0, 0, capacity=3)
    assert st == _lib.FDCM_ERR_CAPACITY and n == 25   # (stride 2: 5 x 5 points)
    n = C.c_int64(7)
    assert _lib.lib().fdcm_search_dense_scales(None, None, C.byref(d._params()), None, 0, 0.0, 10, 0, None, None, None, None, 0,
                                               C.byref(n)) == _lib.FDCM_ERR_INVALID


@pytest.mark.parametrize("rng_", [(0.0, 1.0), (-1.0, 1.0), (1.2, 1.1), (math.nan, 1.0), (1.0, math.inf), (0.5, math.nan)])
def test_fit_matches_scaled_rejects_bad_scale_ranges(rng_):
    f = fdcm.PoseFit(scale_range=rng_)
    sc = _lib.FitScaleParams(*f.scale_range)
    st = _lib.lib().fdcm_fit_matches_scaled(None, None, 0, 0, 0.0, C.byref(f._params()), C.byref(sc), None, 0, None, None)
    assert st == _lib.FDCM_ERR_INVALID and "scale" in _lib.lib().fdcm_last_error().decode()
    # and the fit parameters are checked as for the rigid fit
    bad = fdcm.PoseFit(iterations=0, scale_range=(0.5, 2.0))
    sc = _lib.FitScaleParams(0.5, 2.0)
    assert _lib.lib().fdcm_fit_matches_scaled(None, None, 0, 0, 0.0, C.byref(bad._params()), C.byref(sc), None, 0, None, None) == 1
    assert _lib.lib().fdcm_fit_matches_scaled(None, None, 0, 0, 0.0, C.byref(fdcm.PoseFit()._params()), None, None, 0, None, None) == 1


FIT = fdcm.PoseFit(iterations=20, scale_range=(0.5, 2.0))


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_model_recovers_a_scaled_instance(seed):
    """A noise-free instance at s = 1.07, started at s = 1.0 about 1 px and 0.02 rad off."""
    rng = np.random.default_rng(seed)
    tmpl = house()
    a = anchor_of(tmpl)
    truth = spose(rng.uniform(-math.pi, math.pi), 1.07, rng.uniform(150, 250), rng.uniform(150, 250))
    sc = scene_of(posed(tmpl, truth))
    d = rng.normal(size=2)
    d = d / np.hypot(*d)
    start = offset_similarity(truth, a, rng.choice([-1, 1]) * 0.02, 1.0 / 1.07 - 1.0, d[0], d[1])
    assert abs(sigma_of((start[0], start[1], start[3], start[4])) - 1.0) < 1e-6
    out, st = fit_model_scaled(sc, [tmpl], [a], one_match(start), FIT)
    e_a, e_r, _ = pose_errors(out[0]["transform"], truth, a)
    assert e_a < 1e-4 and scale_error(out[0]["transform"], truth) < 1e-6 and e_r < 1e-6, (e_a, e_r, st)
    assert st[0]["n_inliers"] == st[0]["n_samples"] and st[0]["iterations"] >= 2 and st[0]["rms"] < 1e-4


def test_model_rigid_fit_keeps_the_scale():
    """The rigid fit on the same start keeps s = 1: it cannot reach the instance at 1.07."""
    from tests.test_fit_host import fit_model
    tmpl = house()
    a = anchor_of(tmpl)
    truth = spose(0.4, 1.07, 200.0, 190.0)
    sc = scene_of(posed(tmpl, truth))
    start = offset_similarity(truth, a, 0.02, 1.0 / 1.07 - 1.0, 0.6, -0.8)
    rigid, _ = fit_model(sc, [tmpl], [a], one_match(start), fdcm.PoseFit(iterations=20))
    assert abs(math.sqrt(float(rigid[0]["transform"][0]) ** 2 + float(rigid[0]["transform"][3]) ** 2) - 1.0) < 1e-6
    assert scale_error(rigid[0]["transform"], truth) > 0.05


def test_model_stops_at_max_scale():
    """The truth at s = 1.2 lies beyond max_scale = 1.1: no accepted pose has a scale above the bound."""
    tmpl = house()
    a = anchor_of(tmpl)
    truth = spose(0.3, 1.2, 200.0, 200.0)
    sc = scene_of(posed(tmpl, truth))
    start = offset_similarity(truth, a, 0.0, 1.0 / 1.2 - 1.0, 0.5, 0.5)
    fit = fdcm.PoseFit(iterations=20, scale_range=(0.9, 1.1))
    out, st = fit_model_scaled(sc, [tmpl], [a], one_match(start), fit)
    P = fit_one_scaled(sc, tmpl, a, start, fit)[2]
    assert sigma_of(P) <= float(F32(1.1)) and sigma_of(P) > 1.0
    assert st[0]["iterations"] < 20
    # the next step would have left the range: an unbounded fit goes past 1.1
    free = fit_one_scaled(sc, tmpl, a, start, fdcm.PoseFit(iterations=20, scale_range=(0.5, 2.0)))[2]
    assert abs(sigma_of(free) - 1.2) < 1e-6


def test_model_does_not_drift_a_template_of_parallel_lines():
    """Parallel lines leave the translation along them unobserved; their spacing fixes the scale.  The fit recovers the
    scale and the normal offset and does not slide along the lines."""
    th = 0.4
    u = np.array([math.cos(th), math.sin(th)])
    n = np.array([-u[1], u[0]])
    tmpl = np.array([[0, 0, 80, 0], [0, 15, 80, 15], [0, 40, 80, 40]], F32).T.copy()
    a = anchor_of(tmpl)
    for s_true in (1.0, 1.05):
        truth = spose(th, s_true, 180.0, 170.0)
        sc = scene_of(posed(tmpl, truth))
        start = offset_similarity(truth, a, 0.0, 1.0 / s_true - 1.0, *(1.0 * n + 3.0 * u))
        out, st = fit_model_scaled(sc, [tmpl], [a], one_match(start), FIT)
        _, e_r, off = pose_errors(out[0]["transform"], truth, a)
        assert abs(float(off @ n)) < 0.01 and e_r < 1e-4 and scale_error(out[0]["transform"], truth) < 1e-4, (off, e_r, st)
        m0, m1, m3, m4, ex, ey = fit_one_scaled(sc, tmpl, a, start, FIT)[2]
        ax, ay = float(a[0]), float(a[1])
        moved = np.array([(m0 * ax + m1 * ay) + ex, (m3 * ax + m4 * ay) + ey])
        T0 = start.astype(np.float64)
        start_anchor = np.array([(T0[0] * ax + T0[1] * ay) + T0[2], (T0[3] * ax + T0[4] * ay) + T0[5]])
        assert abs(float((moved - start_anchor) @ u)) < 1e-6, moved - start_anchor


def test_model_edge_cases():
    tmpl = house()
    a = anchor_of(tmpl)
    truth = spose(0.3, 1.1, 200.0, 200.0)
    sc = scene_of(posed(tmpl, truth))
    bad = np.concatenate([one_match([np.nan, 0, 200, 0, 1, 200]), one_match([1, 0, 1e5, 0, 1, 0]), one_match(truth.astype(F32), t=1)])
    out, st = fit_model_scaled(sc, [tmpl, np.zeros((4, 0), F32)], [a, (0.0, 0.0)], bad, FIT)
    assert np.array_equal(out["transform"].view(np.uint32), bad["transform"].view(np.uint32))
    assert np.isnan(out["score"]).all() and st["n_samples"].tolist() == [0, 0, 0]
    far = offset_similarity(truth, a, 0.0, 0.0, 100.0, 0.0)
    out, st = fit_model_scaled(sc, [tmpl], [a], one_match(far), FIT)
    assert out[0]["transform"].tobytes() == far.tobytes() and st[0]["iterations"] == 0


def test_cpp_scale_mirror_builds(tmp_path):
    """ScaleGrid, the searchDense overloads that take it and PoseFit::scaleRange of include/openfdcm_b200/openfdcm_cuda.hpp
    compile and link; the existing aggregate initialisation of PoseFit still compiles."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "scale.cpp"
    src.write_text(r'''
#include "openfdcm_b200/openfdcm_cuda.hpp"
#include <cstdio>
int main() {
    using namespace openfdcm::cuda;
    try {
        const LineArray scene{0.f, 0.f, 50.f, 0.f, 50.f, 0.f, 50.f, 40.f};
        const std::vector<LineArray> templates{LineArray{0.f, 0.f, 20.f, 0.f}};
        const Dt3Cuda fm = buildCudaFeaturemap(scene, Dt3CudaParameters{});
        const DistinctMatches one{1, 0.f, 3.14159274f, false};
        const auto a = searchDense(fm, templates, DenseSearch{}, ScaleGrid{3, 0.9f, 1.1f}, ExponentialPenalty{1.5f}, 5);
        const auto b = searchDense(fm, templates, DenseSearch{}, ScaleGrid{}, ExponentialPenalty{1.5f}, 5, &one, nullptr, EdgeCoverage{});
        PoseFit fit{5, 2.f, 1.f, 1, 1e-3f, 6};
        fit.scaleRange = std::make_pair(0.8f, 1.25f);
        std::vector<FitStats> stats;
        const std::vector<Match> c = fitMatches(fm, templates, a, fit, &stats);
        std::printf("%zu %zu %zu %zu\n", a.size(), b.size(), c.size(), stats.size());
    } catch (const std::exception& e) {
        std::printf("%s\n", e.what());
        return 1;
    }
    return 0;
}
''')
    exe = tmp_path / "scale"
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Werror", "-I" + os.path.join(root, "include"), str(src),
                           "-L" + os.path.join(root, "openfdcm_b200"), "-lfdcm_b200", "-Wl,-rpath," + os.path.join(root, "openfdcm_b200"),
                           "-o", str(exe)])
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode in (0, 1) and r.stdout
