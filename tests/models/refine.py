"""Pose refinement (fdcm_refine_matches, PoseRefinement): the numpy model of the pose grid, of pose validity and of the
walk.  The rules are in include/fdcm_b200.h."""
import math

import numpy as np

from tests.util import F32


def level_table(n_r, rot_step, trans_step, level):
    """ci, si (index i + n_r) and h of one level: host double cos / sin, fp32 step halving."""
    step = float(F32(rot_step)) / 2.0 ** level
    ci = np.array([F32(math.cos(i * step)) for i in range(-n_r, n_r + 1)], F32)
    si = np.array([F32(math.sin(i * step)) for i in range(-n_r, n_r + 1)], F32)
    return ci, si, F32(F32(trans_step) * F32(2.0 ** -level))


def grid_poses(c, anchor, n_r, n_t, rot_step, trans_step, level):
    """The (2 n_r + 1)(2 n_t + 1)^2 candidate transforms of one level in (i, k, j) order, float32 (G, 6)."""
    c = np.asarray(c, F32).reshape(6)
    ax, ay = F32(anchor[0]), F32(anchor[1])
    ci, si, h = level_table(n_r, rot_step, trans_step, level)
    NT = 2 * n_t + 1
    steps = np.arange(-n_t, n_t + 1).astype(F32) * h
    out = np.empty((2 * n_r + 1, NT, NT, 6), F32)
    with np.errstate(all="ignore"):
        px = (c[0] * ax + c[1] * ay) + c[2]
        py = (c[3] * ax + c[4] * ay) + c[5]
        ux, uy = c[2] - px, c[5] - py
        for ir, i in enumerate(range(-n_r, n_r + 1)):
            if i == 0:
                r0, r1, r3, r4, bx, by = c[0], c[1], c[3], c[4], c[2], c[5]
            else:
                a, b = ci[ir], si[ir]
                r0, r1, r3, r4 = a * c[0] - b * c[3], a * c[1] - b * c[4], b * c[0] + a * c[3], b * c[1] + a * c[4]
                bx, by = (a * ux - b * uy) + px, (b * ux + a * uy) + py
            out[ir, :, :, 0], out[ir, :, :, 1], out[ir, :, :, 3], out[ir, :, :, 4] = r0, r1, r3, r4
            out[ir, :, :, 2] = (bx + steps)[None, :]
            out[ir, :, :, 5] = (by + steps)[:, None]
    out[n_r, n_t, n_t] = c
    return out.reshape(-1, 6)


def centre_index(n_r, n_t):
    NT = 2 * n_t + 1
    return (n_r * NT + n_t) * NT + n_t


def rotated(poses, tmpl):
    """(G, L, 4) end points (P0 x + P1 y, P3 x + P4 y) of a (4, L) template under every pose."""
    t = np.asarray(tmpl, F32).reshape(4, -1)
    P = np.asarray(poses, F32).reshape(-1, 6)
    with np.errstate(all="ignore"):
        r0, r1, r3, r4 = (P[:, q, None] for q in (0, 1, 3, 4))
        return np.stack([r0 * t[0] + r1 * t[1], r3 * t[0] + r4 * t[1], r0 * t[2] + r1 * t[3], r3 * t[2] + r4 * t[3]], axis=2)


def valid_poses(poses, tmpl, shift, W, H):
    """Validity of every pose: no NaN in P or in a rotated end point, every end point inside [0, W-1] x [0, H-1]."""
    P = np.asarray(poses, F32).reshape(-1, 6)
    R = rotated(P, tmpl)
    with np.errstate(all="ignore"):
        ox = (F32(shift[0]) + P[:, 2])[:, None]
        oy = (F32(shift[1]) + P[:, 5])[:, None]
        xs = np.concatenate([R[:, :, 0] + ox, R[:, :, 2] + ox], axis=1)
        ys = np.concatenate([R[:, :, 1] + oy, R[:, :, 3] + oy], axis=1)
        ok = (xs >= 0) & (xs <= F32(W - 1)) & (ys >= 0) & (ys <= F32(H - 1))
    return ~np.isnan(P).any(axis=1) & ~np.isnan(R).any(axis=(1, 2)) & ok.all(axis=1)


def walk_order(n_r, n_t):
    """Grid indices by ascending i*i + k*k + j*j (the centre first), equal distances in (i, k, j) order."""
    ijk = [(i, k, j) for i in range(-n_r, n_r + 1) for k in range(-n_t, n_t + 1) for j in range(-n_t, n_t + 1)]
    return sorted(range(len(ijk)), key=lambda g: (sum(v * v for v in ijk[g]), g))


def walk(poses, valid, scores, n_r, n_t):
    """Index of the level's best pose (walk order; NaN as +inf, strict), or None."""
    best, best_key = None, None
    for g in walk_order(n_r, n_t):
        if not valid[g]:
            continue
        key = math.inf if math.isnan(scores[g]) else float(scores[g])
        if best is None or key < best_key:
            best, best_key = g, key
    return best


def refine_model(matches, tmpls, anchors, refine, shift, W, H, score_fn, tmpl_idx_base=0):
    """Raw refined records (no penalty).  score_fn(list of (tmpl (4, L), poses (G, 6))) -> the float32 scores of all
    poses, concatenated; only valid poses are scored.  All matches of a level are scored in one call."""
    out = np.array(matches, copy=True)
    cur = [np.asarray(m["transform"], F32).reshape(6).copy() for m in matches]
    raw = [F32(np.nan)] * len(matches)
    for level in range(refine.levels):
        grids, valids, work = [], [], []
        for q, m in enumerate(matches):
            t = int(m["tmpl_idx"]) - tmpl_idx_base
            g = grid_poses(cur[q], anchors[t], refine.rot_steps, refine.trans_steps, refine.rot_step, refine.trans_step, level)
            v = valid_poses(g, tmpls[t], shift, W, H)
            grids.append(g)
            valids.append(v)
            work.append((tmpls[t], g[v]))
        flat = score_fn(work) if work else np.zeros(0, F32)
        pos = 0
        for q in range(len(matches)):
            s = np.full(len(grids[q]), np.nan, F32)
            nv = int(valids[q].sum())
            s[valids[q]] = flat[pos:pos + nv]
            pos += nv
            b = walk(grids[q], valids[q], s, refine.rot_steps, refine.trans_steps)
            if b is not None:
                cur[q] = grids[q][b].copy()
                raw[q] = s[b]
    for q in range(len(matches)):
        out[q]["transform"] = cur[q].reshape(out[q]["transform"].shape)
        out[q]["score"] = raw[q]
    return out
