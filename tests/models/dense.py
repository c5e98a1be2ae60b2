"""Dense pose-grid search (fdcm_search_dense, DenseSearch; fdcm_search_dense_scales, ScaleGrid): the numpy model of its
rotation and scale table, grid, poses, cells, records, penalty and output.  The rules are in include/fdcm_b200.h.  Every
function takes the scale grid as an optional argument: without one there is one scale, s = 1.0, and the model is that of
the unscaled search."""
import math

import numpy as np

import openfdcm_b200 as fdcm
from openfdcm_b200._lib import MATCH_DTYPE
from tests.models.refine import rotated
from tests.models.select import select_model
from tests.util import F32


def scale_values(g=None):
    """Scaled rule 1: s_k = (float)((double)scale_start * pow((double)scale_ratio, k)) of the float32 parameters; the one
    scale 1.0 without a grid."""
    if g is None:
        return np.ones(1, F32)
    st, ra = float(F32(g.start)), float(F32(g.ratio))
    return np.array([F32(st * math.pow(ra, k)) for k in range(g.scales)], F32)


def rot_table(d, g=None):
    """Rule 1: (a, b) of every (k, r), arrays of shape (S, R): a = (float)(s_k * cos th_r), b = (float)(s_k * sin th_r) with
    th_r = (double)rot_start + r * (double)rot_step, host C library.  At s = 1 these are c_r, s_r."""
    th = [float(F32(d.rot_start)) + r * float(F32(d.rot_step)) for r in range(d.rotations)]
    s = scale_values(g).astype(np.float64)
    a = np.array([[F32(sk * math.cos(x)) for x in th] for sk in s], F32)
    b = np.array([[F32(sk * math.sin(x)) for x in th] for sk in s], F32)
    return a, b


def grid(d, shift, W, H):
    """Rule 2: (lo_x, lo_y, nx, ny); nx = ny = 0 when the range is empty."""
    lo, hi = [0.0, 0.0], [W - 1.0, H - 1.0]
    if d.roi is not None:
        for a in range(2):
            lo[a] = max(lo[a], math.ceil(float(F32(d.roi[a])) + float(F32(shift[a]))))
            hi[a] = min(hi[a], math.floor(float(F32(d.roi[a + 2])) + float(F32(shift[a]))))
    if lo[0] > hi[0] or lo[1] > hi[1]:
        return 0, 0, 0, 0
    lx, ly = int(lo[0]), int(lo[1])
    return lx, ly, (int(hi[0]) - lx) // d.stride + 1, (int(hi[1]) - ly) // d.stride + 1


def poses(d, anchor, shift, W, H, r, g=None, k=0):
    """Rule 3: the (ny * nx, 6) transforms of scale k and rotation r in grid order (row-major: v, then u)."""
    lx, ly, nx, ny = grid(d, shift, W, H)
    A, B = rot_table(d, g)
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


def rotate_template(tmpl, c, s):
    """(L, 4) rotated end points of a (4, L) template; the end points as given when c == 1 and s == 0 (rule 3)."""
    t = np.asarray(tmpl, F32).reshape(4, -1)
    if c == F32(1) and s == F32(0):
        return np.ascontiguousarray(t.T)
    return rotated(np.array([[c, -s, 0, s, c, 0]], F32), t)[0]


def grid_valid(Rt, P, shift, W, H, nx, ny):
    """Rule 4's validity of every grid pose, every end point checked: the x test depends on u only, the y test on v only."""
    P = P.reshape(ny, nx, 6)
    with np.errstate(all="ignore"):
        ox = F32(shift[0]) + P[0, :, 2]
        oy = F32(shift[1]) + P[:, 0, 5]
        xs = np.concatenate([Rt[:, 0], Rt[:, 2]])[None, :] + ox[:, None]
        ys = np.concatenate([Rt[:, 1], Rt[:, 3]])[None, :] + oy[:, None]
        vx = ((xs >= 0) & (xs <= F32(W - 1))).all(axis=1)
        vy = ((ys >= 0) & (ys <= F32(H - 1))).all(axis=1)
    ok = vy[:, None] & vx[None, :] & ~np.isnan(Rt).any() & ~np.isnan(P).any(axis=2)
    return ok.reshape(-1)


def dense_records(tmpls, anchors, d, shift, W, H, score_fn, tmpl_idx_base=0, g=None):
    """Rule 5: every record h = ((((t S + k) R + r) cells_y + cv) cells_x + cu) in record order with its valid flag, raw
    score and grid scale: (rec, valid, rs).  score_fn(Rt (L, 4), translations (n, 2)) -> float32 scores of the rotated
    template at those translations; only valid poses are scored."""
    lx, ly, nx, ny = grid(d, shift, W, H)
    cx, cy = -(-nx // d.cell), -(-ny // d.cell)
    sv = scale_values(g)
    S, R = len(sv), d.rotations
    n = len(tmpls) * S * R * cx * cy
    rec, valid, rs = np.zeros(n, MATCH_DTYPE), np.zeros(n, bool), np.zeros(n, F32)
    if n == 0:
        return rec, valid, rs
    A, B = rot_table(d, g)
    cell_of = ((np.arange(ny) // d.cell)[:, None] * cx + (np.arange(nx) // d.cell)[None, :]).reshape(-1)
    for t, tmpl in enumerate(tmpls):
        if np.asarray(tmpl).reshape(4, -1).shape[1] == 0:
            continue   # an empty template has no records
        for k in range(S):
            for r in range(R):
                P = poses(d, anchors[t], shift, W, H, r, g, k)
                Rt = rotate_template(tmpl, A[k, r], B[k, r])
                gi = np.flatnonzero(grid_valid(Rt, P, shift, W, H, nx, ny))
                if not len(gi):
                    continue
                sc = np.asarray(score_fn(Rt, P[gi][:, [2, 5]]), F32)
                key = np.where(np.isnan(sc), np.inf, sc.astype(np.float64))
                cells = cell_of[gi]
                order = np.lexsort((gi, key, cells))   # by cell, then raw score (NaN as +inf), then grid index
                first = order[np.r_[True, cells[order][1:] != cells[order][:-1]]]
                h = ((t * S + k) * R + r) * cx * cy + cells[first]
                rec["tmpl_idx"][h] = t + tmpl_idx_base
                rec["score"][h] = sc[first]
                rec["transform"][h] = P[gi[first]]
                valid[h] = True
                rs[h] = sv[k]
    return rec, valid, rs


def penalised(rec, valid, lengths, penalty, g=None):
    """The penalty of the valid records of dense_records: the score of a record of (t, k) divided by the penalty
    denominator of len_t * s_k (fp32 product)."""
    if penalty is None:
        return rec
    sv = scale_values(g)
    per_k = len(rec) // (len(lengths) * len(sv)) if len(lengths) else 0
    h = np.flatnonzero(valid)
    tk = h // per_k                                     # t * S + k
    lens = (np.asarray(lengths, F32)[:, None] * sv[None, :]).astype(F32).reshape(-1)
    p = rec[h].copy()
    p["tmpl_idx"] = tk
    p = fdcm.penalize(penalty, p, lens)
    p["tmpl_idx"] = rec[h]["tmpl_idx"]
    out = rec.copy()
    out[h] = p
    return out


def output_model(rec, valid, k, anchors=None, select=None, tmpl_idx_base=0, rs=None):
    """Rule 6 on (penalised) records: the top k in (score, h) order, or the distinct walk of fdcm_search_select (with the
    records' grid scales rs of a scaled search)."""
    sub = rec[valid]
    if select is None:
        s = sub["score"].astype(F32)
        s = np.where(np.isnan(s), F32(np.inf), s)
        return sub[np.lexsort((np.arange(len(sub)), s))[:k]]
    return sub[select_model(sub, anchors, k, select.max_per_template, select.radius, select.max_angle, select.across_templates,
                            tmpl_idx_base, None if rs is None else rs[valid])]
