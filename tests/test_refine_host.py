"""Pose refinement (fdcm_refine_matches, PoseRefinement): the numpy model of tests/models/refine.py pinned by known
answers, and the host hook fdcm_refine_poses against it bit for bit.  The rules are in include/fdcm_b200.h."""
import ctypes as C
import math

import numpy as np
import pytest

from openfdcm_b200 import _lib
from tests.models.refine import centre_index, grid_poses, level_table, valid_poses, walk, walk_order
from tests.util import F32


class Refine:
    def __init__(self, levels=3, rot_steps=4, rot_step=0.01, trans_steps=4, trans_step=1.0):
        self.levels, self.rot_steps, self.rot_step, self.trans_steps, self.trans_step = levels, rot_steps, rot_step, trans_steps, trans_step

    def params(self):
        return _lib.RefineParams(self.levels, self.rot_steps, self.rot_step, self.trans_steps, self.trans_step)


def hook_poses(c, anchor, r, level):
    NT = 2 * r.trans_steps + 1
    out = np.zeros((max(1, (2 * r.rot_steps + 1) * NT * NT), 6), F32)
    c = np.ascontiguousarray(c, F32).reshape(6)
    a = np.ascontiguousarray(anchor, F32).reshape(2)
    st = _lib.lib().fdcm_refine_poses(_lib.ptr(c), _lib.ptr(a), C.byref(r.params()), int(level), _lib.ptr(out))
    return st, out


def rot_mat(th, tx, ty):
    return np.array([math.cos(th), -math.sin(th), tx, math.sin(th), math.cos(th), ty], F32)


# ---- the pose grid ---------------------------------------------------------------------------------------------------
def test_zero_steps_give_only_the_centre():
    c = rot_mat(0.3, 10.5, -4.25)
    g = grid_poses(c, (3.0, -2.0), 0, 0, 0.01, 1.0, 0)
    assert g.shape == (1, 6) and g.tobytes() == c.tobytes()


def test_grid_centre_is_the_centre_bit_for_bit():
    rng = np.random.default_rng(1)
    for _ in range(50):
        c = rng.normal(size=6).astype(F32)
        for n_r, n_t in ((0, 3), (2, 0), (4, 4)):
            g = grid_poses(c, rng.normal(size=2) * 20, n_r, n_t, 0.05, 0.7, int(rng.integers(0, 4)))
            assert g[centre_index(n_r, n_t)].tobytes() == c.tobytes()


def test_level_table_is_host_double_cos_sin():
    ci, si, h = level_table(3, 0.01, 1.5, 2)
    for ir, i in enumerate(range(-3, 4)):
        assert ci[ir] == np.float32(math.cos(i * (float(F32(0.01)) / 4.0)))
        assert si[ir] == np.float32(math.sin(i * (float(F32(0.01)) / 4.0)))
    assert h == F32(0.375)


def test_composition_agrees_with_float64():
    rng = np.random.default_rng(2)
    for _ in range(40):
        th0 = rng.uniform(-math.pi, math.pi)
        c = rot_mat(th0, rng.uniform(0, 500), rng.uniform(0, 500))
        a = rng.uniform(-50, 50, 2)
        n_r, n_t, rs, ts, lv = 3, 2, 0.02, 0.5, int(rng.integers(0, 3))
        g = grid_poses(c, a, n_r, n_t, rs, ts, lv)
        c64 = c.astype(np.float64)
        p = np.array([c64[0] * a[0] + c64[1] * a[1] + c64[2], c64[3] * a[0] + c64[4] * a[1] + c64[5]])
        NT = 2 * n_t + 1
        h = ts / 2 ** lv
        for ir, i in enumerate(range(-n_r, n_r + 1)):
            th = i * rs / 2 ** lv
            Rr = np.array([[math.cos(th), -math.sin(th)], [math.sin(th), math.cos(th)]])
            M = Rr @ c64[[0, 1, 3, 4]].reshape(2, 2)
            t = Rr @ (c64[[2, 5]] - p) + p
            for kk, k in enumerate(range(-n_t, n_t + 1)):
                for jj, j in enumerate(range(-n_t, n_t + 1)):
                    want = np.array([M[0, 0], M[0, 1], t[0] + j * h, M[1, 0], M[1, 1], t[1] + k * h])
                    got = g[(ir * NT + kk) * NT + jj].astype(np.float64)
                    assert np.abs(got - want).max() <= 1e-5 * max(1.0, np.abs(want).max())


def test_pure_rotation_keeps_the_anchor():
    c = rot_mat(0.7, 321.25, 117.5)
    a = np.array([12.5, -30.0], F32)
    g = grid_poses(c, a, 4, 0, 0.05, 1.0, 0)
    anchor = lambda P: np.array([P[0] * a[0] + P[1] * a[1] + P[2], P[3] * a[0] + P[4] * a[1] + P[5]], np.float64)
    for P in g:
        assert np.abs(anchor(P) - anchor(c)).max() < 1e-3


def test_steps_halve_per_level():
    c = rot_mat(0.0, 100.0, 100.0)
    for lv in range(4):
        g = grid_poses(c, (0.0, 0.0), 1, 1, 0.08, 2.0, lv)
        assert g[centre_index(1, 1) + 1][2] - c[2] == F32(2.0 / 2 ** lv)   # (i, k, j) = (0, 0, 1)
        th = math.atan2(float(g[1][3]), float(g[1][0]))                     # (i, k, j) = (-1, -1, 0)
        assert abs(th - (-0.08 / 2 ** lv)) < 1e-6


# ---- the walk --------------------------------------------------------------------------------------------------------
def run_walk(scores, valid=None, n_r=1, n_t=1):
    n = (2 * n_r + 1) * (2 * n_t + 1) ** 2
    valid = np.ones(n, bool) if valid is None else valid
    return walk(np.zeros((n, 6), F32), valid, np.asarray(scores, F32), n_r, n_t)


def test_constant_score_keeps_the_centre():
    assert run_walk(np.full(27, 3.0)) == centre_index(1, 1)


def test_equal_minima_resolve_to_the_point_nearest_the_centre_then_the_earlier():
    assert walk_order(1, 1)[:4] == [centre_index(1, 1), 4, 10, 12]   # (0,0,0), then (-1,0,0), (0,-1,0), (0,0,-1)
    s = np.full(27, 5.0)
    s[[0, 22]] = 1.0             # (-1, -1, -1) and (1, 0, 0)
    assert run_walk(s) == 22
    s[4] = 1.0                   # (-1, 0, 0): as near as (1, 0, 0), earlier
    assert run_walk(s) == 4
    s[centre_index(1, 1)] = 1.0
    assert run_walk(s) == centre_index(1, 1)


def test_nan_loses_to_finite_and_ties_with_inf():
    s = np.full(27, np.nan)
    s[25] = 1e30
    assert run_walk(s) == 25
    s = np.full(27, np.inf)
    s[3] = np.nan
    assert run_walk(s) == centre_index(1, 1)
    s[centre_index(1, 1)] = np.nan
    assert run_walk(s) == centre_index(1, 1)


def test_invalid_centre_is_replaced_by_any_valid_pose():
    v = np.zeros(27, bool)
    v[26] = True
    s = np.full(27, 0.0)
    s[26] = np.nan
    assert run_walk(s, v) == 26
    assert run_walk(s, np.zeros(27, bool)) is None


def test_validity_boundary_is_exact():
    W, H, shift = 100, 80, (F32(2.5), F32(0.0))
    tmpl = np.array([[0.0], [0.0], [10.0], [5.0]], F32)   # one line from the origin
    x0 = -shift[0]                                         # end point exactly at 0
    x1 = F32(W - 1) - shift[0] - F32(10.0)                 # end point exactly at W - 1
    ident = lambda tx, ty: np.array([1, 0, tx, 0, 1, ty], F32)
    assert valid_poses(np.stack([ident(x0, 0.0), ident(x1, 0.0), ident(x0, F32(H - 1) - F32(5.0))]), tmpl, shift, W, H).all()
    below = np.nextafter(x0, F32(-np.inf))
    above = np.nextafter(x1, F32(np.inf))
    assert F32(0.0) + (shift[0] + below) < 0 and F32(10.0) + (shift[0] + above) > F32(W - 1)
    assert not valid_poses(np.stack([ident(below, 0.0), ident(above, 0.0), ident(x0, np.nextafter(F32(-0.0), F32(-1)))]), tmpl, shift,
                           W, H).any()
    nan = ident(10.0, 10.0)
    nan[1] = np.nan
    assert not valid_poses(nan[None], tmpl, shift, W, H)[0]
    assert valid_poses(ident(1e6, 1e6)[None], np.zeros((4, 0), F32), shift, W, H)[0]        # empty template: any pose
    assert not valid_poses(nan[None], np.zeros((4, 0), F32), shift, W, H)[0]


# ---- the host hook ---------------------------------------------------------------------------------------------------
def test_refine_poses_hook_equals_the_model():
    rng = np.random.default_rng(3)
    for case in range(60):
        r = Refine(int(rng.integers(1, 4)), int(rng.integers(0, 16)), float(rng.uniform(0, 0.2)), int(rng.integers(0, 16)),
                   float(rng.uniform(0, 3)))
        c = rot_mat(rng.uniform(-math.pi, math.pi), rng.uniform(-100, 900), rng.uniform(-100, 900))
        if case % 5 == 0:
            c = rng.normal(size=6).astype(F32) * F32(100)
        if case % 7 == 0:
            c[[0, 4]] = F32(-0.0)
        a = (rng.uniform(-80, 80, 2)).astype(F32)
        for lv in range(r.levels):
            st, got = hook_poses(c, a, r, lv)
            assert st == 0
            want = grid_poses(c, a, r.rot_steps, r.trans_steps, r.rot_step, r.trans_step, lv)
            assert got.tobytes() == want.tobytes(), f"case {case} level {lv}"


@pytest.mark.parametrize("bad", [dict(levels=0), dict(rot_steps=-1), dict(rot_steps=16), dict(trans_steps=16), dict(trans_steps=-1),
                                 dict(rot_step=-0.01), dict(rot_step=math.nan), dict(trans_step=math.inf), dict(trans_step=-1.0)])
def test_refine_poses_rejects_bad_parameters(bad):
    r = Refine(**{**dict(levels=2, rot_steps=1, rot_step=0.01, trans_steps=1, trans_step=1.0), **bad})
    st, _ = hook_poses(np.zeros(6, F32), np.zeros(2, F32), r, 0)
    assert st == _lib.FDCM_ERR_INVALID
    st = _lib.lib().fdcm_refine_poses(_lib.ptr(np.zeros(6, F32)), _lib.ptr(np.zeros(2, F32)), None, 0, _lib.ptr(np.zeros(6, F32)))
    assert st == _lib.FDCM_ERR_INVALID


def test_refine_poses_rejects_a_level_outside_the_walk():
    r = Refine(2, 0, 0.01, 0, 1.0)
    assert hook_poses(np.zeros(6, F32), np.zeros(2, F32), r, 2)[0] == _lib.FDCM_ERR_INVALID
    assert hook_poses(np.zeros(6, F32), np.zeros(2, F32), r, -1)[0] == _lib.FDCM_ERR_INVALID
