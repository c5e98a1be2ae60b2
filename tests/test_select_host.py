"""Distinct top-K (fdcm_search_select): the numpy model of its greedy walk, pinned by hand-built known answers, and the
host-side pieces of the C ABI (struct layout, template anchors).  The GPU tests (test_gpu_select.py) compare the device
against this model.  No kernel is launched here."""
import ctypes as C
import math

import numpy as np

import openfdcm_b200 as fdcm
from openfdcm_b200 import _lib
from openfdcm_b200._lib import MATCH_DTYPE
from tests.util import F32, synth_templates

PI_F32 = F32(3.14159274)


def select_model(rec, anchors, k, max_per_template=0, radius=0.0, max_angle=math.pi, across_templates=False, tmpl_idx_base=0):
    """The greedy walk of include/fdcm_b200.h over `rec`, the valid matches in hypothesis order (position = order of h).
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
                    near &= (T[A, 0] * T[b, 0] + T[A, 3] * T[b, 3]) >= cos_thr
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


def matches(rows):
    """rows of (tmpl, score, angle, tx, ty) -> MATCH_DTYPE records with transform [c -s tx s c ty]."""
    rec = np.zeros(len(rows), MATCH_DTYPE)
    for i, (t, s, ang, tx, ty) in enumerate(rows):
        c, sn = F32(math.cos(ang)), F32(math.sin(ang))
        rec[i] = (t, s, [c, -sn, tx, sn, c, ty])
    return rec


ZERO_ANCHORS = np.zeros((4, 2), F32)   # anchor (0, 0): a match's anchor is its translation


def test_select_params_layout():
    assert C.sizeof(_lib.SelectParams) == 16


def _numpy_anchor(t):
    t = np.asarray(t, F32).reshape(4, -1)
    if t.shape[1] == 0:
        return np.zeros(2, F32)
    xs, ys = np.concatenate([t[0], t[2]]), np.concatenate([t[1], t[3]])
    return np.array([(xs.min() + xs.max()) * F32(0.5), (ys.min() + ys.max()) * F32(0.5)], F32)


def test_template_anchors_match_numpy_bbox_centre():
    rng = np.random.default_rng(11)
    tmpls = synth_templates(20, 17, 640, seed=12)                                    # centred on the origin: negative coordinates
    tmpls += [rng.uniform(-1e4, 1e4, (4, n)).astype(F32) for n in (1, 2, 3, 40)]      # one-line templates, wide ranges
    tmpls.append(np.array([[5.5], [-7.25], [5.5], [-7.25]], F32))                     # a zero-length line
    tmpls.insert(3, np.zeros((4, 0), F32))                                            # an empty template
    tmpls.append((rng.uniform(0, 1, (4, 9)) * F32(1 / 3)).astype(F32))                # non-representable halves
    got = fdcm.get_template_anchors(tmpls)
    assert got.dtype == F32 and got.shape == (len(tmpls), 2)
    want = np.stack([_numpy_anchor(t) for t in tmpls])
    assert got.tobytes() == want.tobytes()
    assert got[3].tolist() == [0.0, 0.0]
    assert fdcm.get_template_anchors([]).shape == (0, 2)


def test_model_cap():
    rec = matches([(0, 1, 0, 0, 0), (0, 2, 0, 100, 0), (1, 3, 0, 200, 0), (0, 4, 0, 300, 0)])
    assert select_model(rec, ZERO_ANCHORS, 10, max_per_template=1).tolist() == [0, 2]
    assert select_model(rec, ZERO_ANCHORS, 10, max_per_template=2).tolist() == [0, 1, 2]
    assert select_model(rec, ZERO_ANCHORS, 10).tolist() == [0, 1, 2, 3]


def test_model_radius_boundary_suppresses():
    rec = matches([(0, 1, 0, 0, 0), (0, 2, 0, 3, 4), (0, 3, 0, 0, 10.5)])   # d^2 to the first: 25 = 5^2 and 110.25 = 10.5^2
    assert select_model(rec, ZERO_ANCHORS, 10, radius=5).tolist() == [0, 2]
    assert select_model(rec, ZERO_ANCHORS, 10, radius=4.99).tolist() == [0, 1, 2]
    assert select_model(rec, ZERO_ANCHORS, 10, radius=10.5).tolist() == [0]


def test_model_anchor_follows_the_transform():
    anchors = np.array([[10, 0], [0, 0]], F32)
    rec = matches([(0, 1, 0, 0, 0), (0, 2, math.pi / 2, 0, 0)])   # template anchor (10, 0) lands at (10, 0) and (0, 10)
    assert select_model(rec, anchors, 10, radius=14).tolist() == [0, 1]
    assert select_model(rec, anchors, 10, radius=14.2).tolist() == [0]


def test_model_angle_threshold():
    rec = matches([(0, 1, 0, 0, 0), (0, 2, 0.3, 1, 0)])
    assert select_model(rec, ZERO_ANCHORS, 10, radius=5, max_angle=0.2).tolist() == [0, 1]
    assert select_model(rec, ZERO_ANCHORS, 10, radius=5, max_angle=0.4).tolist() == [0]
    assert select_model(rec, ZERO_ANCHORS, 10, radius=5).tolist() == [0]
    rev = matches([(0, 1, 0, 0, 0), (0, 2, math.pi, 0, 0)])                 # the reversed hypothesis: rotated by pi
    assert select_model(rev, ZERO_ANCHORS, 10, radius=5, max_angle=3.0).tolist() == [0, 1]
    assert select_model(rev, ZERO_ANCHORS, 10, radius=5, max_angle=math.pi).tolist() == [0]
    assert select_model(rev, ZERO_ANCHORS, 10, radius=5, max_angle=100.0).tolist() == [0]


def test_model_within_vs_across_templates():
    rec = matches([(0, 1, 0, 0, 0), (1, 2, 0, 1, 1), (0, 3, 0, 2, 0), (2, 4, 0, 50, 0)])
    assert select_model(rec, ZERO_ANCHORS, 10, radius=5).tolist() == [0, 1, 3]
    assert select_model(rec, ZERO_ANCHORS, 10, radius=5, across_templates=True).tolist() == [0, 3]
    assert select_model(rec, ZERO_ANCHORS, 10, max_per_template=1, radius=5, across_templates=True).tolist() == [0, 3]


def test_model_top_k_truncation():
    rec = matches([(i % 3, 10 - i, 0, 40 * i, 0) for i in range(8)])
    assert select_model(rec, ZERO_ANCHORS, 3).tolist() == [7, 6, 5]
    assert select_model(rec, ZERO_ANCHORS, 3, max_per_template=1).tolist() == [7, 6, 5]
    assert select_model(rec, ZERO_ANCHORS, 4, max_per_template=1).tolist() == [7, 6, 5]
    assert select_model(rec, ZERO_ANCHORS, 1, radius=1000, across_templates=True).tolist() == [7]


def test_model_nan_orders_as_inf_and_ties_by_h():
    rec = matches([(0, np.nan, 0, 0, 0), (1, 1, 0, 0, 0), (2, np.inf, 0, 0, 0), (3, 0.5, 0, 0, 0)])
    assert select_model(rec, ZERO_ANCHORS, 10).tolist() == [3, 1, 0, 2]
    ties = matches([(0, 2, 0, 0, 0), (1, 1, 0, 0, 0), (2, 1, 0, 0, 0), (3, 2, 0, 0, 0)])
    assert select_model(ties, ZERO_ANCHORS, 10).tolist() == [1, 2, 0, 3]
    assert select_model(ties, ZERO_ANCHORS, 10, radius=1, across_templates=True).tolist() == [1]


def test_per_template_walk_equals_global_walk():
    rng = np.random.default_rng(2024)
    for trial in range(40):
        n_tmpl = int(rng.integers(1, 8))
        n = int(rng.integers(1, 120))
        rec = np.zeros(n, MATCH_DTYPE)
        rec["tmpl_idx"] = np.sort(rng.integers(0, n_tmpl, n))                      # hypothesis order groups templates
        rec["score"] = rng.choice(np.array([0.5, 1.0, 1.5, np.nan], F32), n) if trial % 4 == 0 else rng.uniform(0, 2, n).astype(F32)
        ang = rng.uniform(-math.pi, math.pi, n)
        rec["transform"][:, 0], rec["transform"][:, 1] = np.cos(ang), -np.sin(ang)
        rec["transform"][:, 3], rec["transform"][:, 4] = np.sin(ang), np.cos(ang)
        rec["transform"][:, 2], rec["transform"][:, 5] = rng.uniform(0, 60, n), rng.uniform(0, 60, n)
        anchors = rng.uniform(-20, 20, (n_tmpl, 2)).astype(F32)
        for cap in (0, 1, 2):
            for radius, max_angle in ((0.0, math.pi), (10.0, math.pi), (25.0, 0.5)):
                for k in (1, 5, n):
                    want = select_model(rec, anchors, k, cap, radius, max_angle)
                    got = per_template_model(rec, anchors, k, cap, radius, max_angle)
                    assert got.tolist() == want.tolist(), (trial, cap, radius, max_angle, k)
