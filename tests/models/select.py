"""Distinct top-K (fdcm_search_select, DistinctMatches): the numpy model of its greedy walk.  The rules are in
include/fdcm_b200.h."""
import math

import numpy as np

from tests.util import F32

PI_F32 = F32(3.14159274)


def select_model(rec, anchors, k, max_per_template=0, radius=0.0, max_angle=math.pi, across_templates=False, tmpl_idx_base=0, rs=None):
    """The greedy walk of include/fdcm_b200.h over `rec`, the valid matches in hypothesis order (position = order of h).
    rs: the grid scale of every record (scaled dense search); the angle test is then Ta0*Tb0 + Ta3*Tb3 >= cos_thr * (s_a * s_b).
    Returns the positions of the accepted matches in acceptance order."""
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
    acc = np.zeros(min(k, n), np.int64)
    n_acc = 0
    count = {}
    for b in order:
        if n_acc == k:
            break
        tb = int(tmpl[b])
        if max_per_template and count.get(tb, 0) >= max_per_template:
            continue
        if radius_on and n_acc:
            A = acc[:n_acc]
            if not across_templates:
                A = A[tmpl[A] == tb]
            if len(A):
                dx, dy = px[A] - px[b], py[A] - py[b]
                near = (dx * dx + dy * dy) <= r2
                if not any_angle:
                    near &= (T[A, 0] * T[b, 0] + T[A, 3] * T[b, 3]) >= (cos_thr if rs is None else cos_thr * (rs[A] * rs[b]))
                if near.any():
                    continue
        acc[n_acc] = b
        n_acc += 1
        count[tb] = count.get(tb, 0) + 1
    return acc[:n_acc]


def per_template_model(rec, anchors, k, max_per_template=0, radius=0.0, max_angle=math.pi):
    """The within-template walk as the device runs it: every template on its own, then the first k survivors in global
    (score, h) order."""
    surv = []
    for t in np.unique(rec["tmpl_idx"]):
        sub = np.flatnonzero(rec["tmpl_idx"] == t)
        surv.extend(sub[select_model(rec[sub], anchors, k, max_per_template, radius, max_angle)].tolist())
    surv = np.array(sorted(surv), np.int64)
    s = rec["score"][surv].astype(F32)
    s = np.where(np.isnan(s), F32(np.inf), s)
    return surv[np.lexsort((surv, s))][:k]
