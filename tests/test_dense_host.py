"""Dense pose-grid search (fdcm_search_dense, DenseSearch): the numpy model of its rotations, grid, poses, cells and
records (tests/models/dense.py), pinned by known answers, and the host hook fdcm_dense_poses against it bit for bit.  The
rules are in include/fdcm_b200.h; tests/test_gpu_dense.py compares the device against this model.  No kernel is launched
here."""
import ctypes as C
import math

import numpy as np
import pytest

import openfdcm_b200 as fdcm
from openfdcm_b200 import _lib
from openfdcm_b200._lib import MATCH_DTYPE
from tests.helpers import dense_poses_hook
from tests.models.dense import dense_records, grid, grid_valid, output_model, poses, rot_table, rotate_template
from tests.models.refine import rotated, valid_poses
from tests.util import F32


def one_point(x=0.0, y=0.0):
    return np.array([[x], [y], [x], [y]], F32)


# ---- layout and rule 1 -----------------------------------------------------------------------------------------------
def test_dense_params_layout():
    assert C.sizeof(_lib.DenseParams) == 40
    assert [f[0] for f in _lib.DenseParams._fields_] == ["rotations", "rot_start", "rot_step", "stride", "cell", "roi_on", "roi"]
    assert _lib.DenseParams.roi.offset == 24


def test_default_rotations_cover_one_turn():
    d = fdcm.DenseSearch()
    assert (d.rotations, d.rot_start, d.stride, d.cell, d.roi) == (72, 0.0, 2, 8, None)
    assert d.rot_step == 2 * math.pi / 72
    (c,), (s,) = rot_table(d)
    assert c[0] == 1 and s[0] == 0 and abs(float(c[36]) + 1) < 1e-6 and abs(float(s[18]) - 1) < 1e-6
    assert fdcm.DenseSearch(10, rot_step=0.0).rot_step == 0.0


def test_rotation_table_is_host_double_cos_sin():
    d = fdcm.DenseSearch(5, rot_start=-0.3, rot_step=0.7)
    (c,), (s,) = rot_table(d)
    for r in range(5):
        th = float(F32(-0.3)) + r * float(F32(0.7))
        assert c[r] == F32(math.cos(th)) and s[r] == F32(math.sin(th))
        st, P, n, wh = dense_poses_hook(d, (0.0, 0.0), (0.0, 0.0), 3, 2, r)
        assert st == 0 and (P[:, 0] == c[r]).all() and (P[:, 3] == s[r]).all() and (P[:, 1] == -s[r]).all()


# ---- rule 2: the grid ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("roi,shift,want", [
    (None, (0.0, 0.0), (0, 0, 40, 30)),
    (None, (2.5, -1.25), (0, 0, 40, 30)),
    ((0.2, 1.0, 10.7, 5.3), (2.5, -1.25), (3, 0, 11, 5)),       # ceil(2.7) = 3, floor(13.2) = 13; y: ceil(-0.25) = 0, floor(4.05) = 4
    ((0.5, 1.25, 7.5, 4.25), (2.5, -1.25), (3, 0, 8, 4)),       # exact integers stay: [3, 10] x [0, 3]
    ((-100.0, -100.0, 1e6, 1e6), (2.5, -1.25), (0, 0, 40, 30)),  # clipped by the map
    ((30.0, 20.0, 1e6, 1e6), (2.5, 0.0), (33, 20, 7, 10)),      # clipped at the right and bottom
    ((40.0, 0.0, 50.0, 10.0), (0.0, 0.0), (0, 0, 0, 0)),        # right of the map
    ((0.0, -9.0, 10.0, -1.5), (0.0, 0.0), (0, 0, 0, 0)),        # above the map
    ((3.2, 0.0, 3.8, 5.0), (0.0, 0.0), (0, 0, 0, 0)),           # no pixel inside: ceil(3.2) > floor(3.8)
])
def test_grid_bounds(roi, shift, want):
    d = fdcm.DenseSearch(1, stride=1, roi=roi)
    assert grid(d, shift, 40, 30) == want
    st, P, n, wh = dense_poses_hook(d, (0.0, 0.0), shift, 40, 30, 0)
    assert st == 0 and wh == want[2:] and n == want[2] * want[3]
    if n:   # anchor (0, 0), identity: P2 = gx - shift_x
        assert P[0, 2] == F32(want[0]) - F32(shift[0]) and P[0, 5] == F32(want[1]) - F32(shift[1])


def test_empty_map_has_no_grid():
    for W, H in ((0, 0), (0, 5), (5, 0)):
        st, _, n, wh = dense_poses_hook(fdcm.DenseSearch(3, stride=1), (0.0, 0.0), (0.0, 0.0), W, H, 1)
        assert st == 0 and n == 0 and wh == (0, 0) or wh[0] * wh[1] == 0


def test_stride():
    for stride, want_nx in ((1, 17), (2, 9), (3, 6), (4, 5), (16, 2), (17, 1), (100, 1)):
        d = fdcm.DenseSearch(1, stride=stride)
        st, P, n, wh = dense_poses_hook(d, (0.0, 0.0), (0.0, 0.0), 17, 5, 0)
        assert st == 0 and wh[0] == want_nx
        gx = P.reshape(wh[1], wh[0], 6)[0, :, 2]
        assert gx.tolist() == [float(u * stride) for u in range(want_nx)]
        gy = P.reshape(wh[1], wh[0], 6)[:, 0, 5]
        assert gy.tolist() == [float(v * stride) for v in range(wh[1])]
    d = fdcm.DenseSearch(1, stride=3, roi=(2.0, 1.0, 12.0, 3.0))
    st, P, n, wh = dense_poses_hook(d, (0.0, 0.0), (0.0, 0.0), 17, 5, 0)
    assert wh == (4, 1) and P[:, 2].tolist() == [2.0, 5.0, 8.0, 11.0]


# ---- rule 5: cells, record order, ties -------------------------------------------------------------------------------
def bowl(cx, cy):
    """score_fn: squared distance of the translation from (cx, cy)."""
    return lambda Rt, tr: ((tr[:, 0] - F32(cx)) ** 2 + (tr[:, 1] - F32(cy)) ** 2).astype(F32)


def test_cells_and_record_order_with_partial_cells():
    """7 x 5 grid, cell 3: cells_x = 3 (the last one column wide), cells_y = 2 (the last two rows high)."""
    W, H = 7, 5
    d = fdcm.DenseSearch(2, rot_step=0.5, stride=1, cell=3)
    tmpls = [one_point(), one_point()]
    anchors = np.zeros((2, 2), F32)
    rec, valid, _ = dense_records(tmpls, anchors, d, (0.0, 0.0), W, H, bowl(4, 1), tmpl_idx_base=7)
    assert len(rec) == 2 * 2 * 2 * 3 and valid.all()
    cols = {0: [0, 1, 2], 1: [3, 4, 5], 2: [6]}
    rows = {0: [0, 1, 2], 1: [3, 4]}
    for t in range(2):
        for r in range(2):
            for cv in range(2):
                for cu in range(3):
                    h = ((t * 2 + r) * 2 + cv) * 3 + cu
                    x = min(cols[cu], key=lambda u: abs(u - 4))
                    y = min(rows[cv], key=lambda v: abs(v - 1))
                    T = rec[h]["transform"]
                    assert (T[2], T[5]) == (x, y), (t, r, cv, cu)
                    assert rec[h]["tmpl_idx"] == t + 7 and rec[h]["score"] == F32((x - 4) ** 2 + (y - 1) ** 2)
                    assert T[0] == rot_table(d)[0][0, r]


def test_ties_go_to_the_lowest_grid_index():
    d = fdcm.DenseSearch(1, stride=1, cell=3)
    rec, valid, _ = dense_records([one_point()], np.zeros((1, 2), F32), d, (0.0, 0.0), 7, 5, lambda Rt, tr: np.full(len(tr), 2.0, F32))
    # every cell keeps its top-left point
    assert [(float(T[2]), float(T[5])) for T in rec["transform"]] == [(0, 0), (3, 0), (6, 0), (0, 3), (3, 3), (6, 3)]


def test_nan_ties_with_inf_and_loses_to_finite():
    d = fdcm.DenseSearch(1, stride=1, cell=1000)   # one cell: the whole 4 x 1 grid, grid index = u

    def scores(vals):
        return lambda Rt, tr: np.array([vals[int(x)] for x in tr[:, 0]], F32)

    def best(vals):
        rec, valid, _ = dense_records([one_point()], np.zeros((1, 2), F32), d, (0.0, 0.0), 4, 1, scores(vals))
        assert len(rec) == 1 and valid[0]
        return int(rec[0]["transform"][2]), rec[0]["score"]

    nan, inf = math.nan, math.inf
    g, s = best([nan, inf, inf, nan])
    assert g == 0 and math.isnan(s)
    g, s = best([inf, nan, nan, inf])
    assert g == 0 and s == inf
    assert best([nan, inf, 1e30, nan]) == (2, F32(1e30))
    assert best([5.0, 3.0, 3.0, 4.0]) == (1, 3.0)


def test_invalid_poses_and_empty_templates_give_no_records():
    """A 2-px wide line fits a 4-px map at u = 0, 1 only; an empty template has no records at all."""
    d = fdcm.DenseSearch(1, stride=1, cell=1)
    tmpls = [np.array([[0.0], [0.0], [2.0], [0.0]], F32), np.zeros((4, 0), F32)]
    rec, valid, _ = dense_records(tmpls, np.zeros((2, 2), F32), d, (0.0, 0.0), 4, 2, bowl(0, 0))
    assert valid.tolist() == [True, True, False, False, True, True, False, False] + [False] * 8


def test_grid_validity_equals_the_refinement_rule():
    """grid_valid (separable in u and v) == valid_poses of refinement rule 4 on every pose."""
    rng = np.random.default_rng(11)
    for case in range(40):
        L = int(rng.integers(1, 6))
        tmpl = rng.uniform(-6, 6, (4, L)).astype(F32)
        if case % 5 == 0:
            tmpl[:, 0] = [F32(-0.0), 0.0, F32(-0.0), 3.0]
        anchor = rng.uniform(-3, 3, 2).astype(F32)
        shift = rng.uniform(-2, 2, 2).astype(F32)
        d = fdcm.DenseSearch(int(rng.integers(1, 9)), float(rng.uniform(-3, 3)), stride=int(rng.integers(1, 4)))
        W, H = int(rng.integers(1, 30)), int(rng.integers(1, 30))
        lx, ly, nx, ny = grid(d, shift, W, H)
        (cs,), (sn,) = rot_table(d)
        for r in range(d.rotations):
            P = poses(d, anchor, shift, W, H, r)
            want = valid_poses(P, tmpl, shift, W, H)
            assert (grid_valid(rotate_template(tmpl, cs[r], sn[r]), P, shift, W, H, nx, ny) == want).all(), (case, r)


# ---- rule 3: the identity at theta = 0 -------------------------------------------------------------------------------
def test_identity_rotation_uses_the_end_points_as_given():
    """A vertical line at x = -0 with a negative y: composing it through cos 0 and -sin 0 = -0 turns one x into +0, so dx
    changes sign and the slope goes from +inf to -inf (another orientation bin).  The dense rule keeps the end points."""
    tmpl = np.array([[-0.0], [-5.0], [-0.0], [3.0]], F32)
    (c,), (s,) = rot_table(fdcm.DenseSearch(1))
    assert c[0] == 1 and s[0] == 0
    kept = rotate_template(tmpl, c[0], s[0])
    assert kept.tobytes() == np.ascontiguousarray(tmpl.T).tobytes()
    composed = rotated(np.array([[c[0], -s[0], 0, s[0], c[0], 0]], F32), tmpl)[0]
    with np.errstate(divide="ignore"):
        slope = lambda R: (R[0, 3] - R[0, 1]) / (R[0, 2] - R[0, 0])
        assert slope(kept) == np.inf and slope(composed) == -np.inf
    # the transform itself is the general formula: (1, -0, qx - ax, 0, 1, qy - ay)
    st, P, n, wh = dense_poses_hook(fdcm.DenseSearch(1, stride=1), (1.5, -2.0), (0.25, 0.0), 4, 3, 0)
    assert st == 0 and np.signbit(P[:, 1]).all() and (P[:, 2] == P[:, 2]).all()
    assert P.reshape(3, 4, 6)[1, 2, 2] == (F32(2) - F32(0.25)) - F32(1.5) and P.reshape(3, 4, 6)[1, 2, 5] == F32(1) + F32(2.0)


# ---- the host hook ---------------------------------------------------------------------------------------------------
def test_dense_poses_hook_equals_the_model():
    rng = np.random.default_rng(3)
    for case in range(80):
        roi = None
        if case % 3 == 0:
            x0, y0 = rng.uniform(-20, 60, 2)
            roi = (float(x0), float(y0), float(x0 + rng.uniform(0, 50)), float(y0 + rng.uniform(0, 50)))
        d = fdcm.DenseSearch(int(rng.integers(1, 200)), float(rng.uniform(-7, 7)), float(rng.uniform(-0.5, 0.5)),
                             int(rng.integers(1, 7)), int(rng.integers(1, 20)), roi)
        if case % 10 == 0:
            d.rot_start, d.rot_step = 0.0, 0.0   # the identity in every rotation
        anchor = rng.uniform(-80, 80, 2).astype(F32)
        shift = (rng.uniform(-50, 50, 2) * (case % 4 != 1)).astype(F32)
        W, H = int(rng.integers(0, 70)), int(rng.integers(0, 70))
        for r in {0, int(rng.integers(0, d.rotations)), d.rotations - 1}:
            st, P, n, wh = dense_poses_hook(d, anchor, shift, W, H, r)
            want = poses(d, anchor, shift, W, H, r)
            assert st == 0 and wh == grid(d, shift, W, H)[2:] and n == len(want)
            assert P.tobytes() == want.tobytes(), f"case {case} rotation {r}"


def test_dense_poses_capacity():
    d = fdcm.DenseSearch(1, stride=1)
    st, _, n, wh = dense_poses_hook(d, (0.0, 0.0), (0.0, 0.0), 5, 4, 0, capacity=19)
    assert st == _lib.FDCM_ERR_CAPACITY and n == 20 and wh == (5, 4)
    assert dense_poses_hook(d, (0.0, 0.0), (0.0, 0.0), 5, 4, 0, capacity=20)[0] == 0


BAD = [dict(rotations=0), dict(rotations=4097), dict(rotations=-1), dict(stride=0), dict(stride=-2), dict(cell=0), dict(cell=-1),
       dict(rot_start=math.nan), dict(rot_start=math.inf), dict(rot_step=math.nan), dict(rot_step=-math.inf),
       dict(roi=(0.0, 0.0, math.nan, 5.0)), dict(roi=(-math.inf, 0.0, 5.0, 5.0)), dict(roi=(6.0, 0.0, 5.0, 5.0)),
       dict(roi=(0.0, 6.0, 5.0, 5.0))]


@pytest.mark.parametrize("bad", BAD)
def test_dense_poses_rejects_bad_parameters(bad):
    d = fdcm.DenseSearch(**{**dict(rotations=4, rot_step=0.1, stride=1, cell=2), **bad})
    out, n, wh = np.zeros((25, 6), F32), C.c_int64(0), np.zeros(2, np.int32)
    st = _lib.lib().fdcm_dense_poses(C.byref(d._params()), _lib.ptr(np.zeros(2, F32)), _lib.ptr(np.zeros(2, F32)), 5, 5, 0, _lib.ptr(out), 25,
                                     C.byref(n), _lib.ptr(wh))
    assert st == _lib.FDCM_ERR_INVALID
    assert b"dense search" in _lib.lib().fdcm_last_error()


def test_dense_poses_rejects_bad_arguments():
    d = fdcm.DenseSearch(4, stride=1)
    z = _lib.ptr(np.zeros(2, F32))
    out, n, wh = np.zeros((25, 6), F32), C.c_int64(0), np.zeros(2, np.int32)
    assert _lib.lib().fdcm_dense_poses(None, z, z, 5, 5, 0, _lib.ptr(out), 25, C.byref(n), _lib.ptr(wh)) == _lib.FDCM_ERR_INVALID
    for r in (-1, 4):
        assert dense_poses_hook(d, (0.0, 0.0), (0.0, 0.0), 5, 5, r)[0] == _lib.FDCM_ERR_INVALID
    assert dense_poses_hook(d, (0.0, 0.0), (0.0, 0.0), -1, 5, 0)[0] == _lib.FDCM_ERR_INVALID
    assert _lib.lib().fdcm_dense_poses(C.byref(d._params()), None, z, 5, 5, 0, _lib.ptr(out), 25, C.byref(n), _lib.ptr(wh)) == _lib.FDCM_ERR_INVALID
    with pytest.raises(ValueError):
        fdcm.DenseSearch(roi=(1.0, 2.0, 3.0))


def test_output_model_orders_by_score_then_record():
    rec = np.zeros(6, MATCH_DTYPE)
    rec["score"] = [3.0, np.nan, 1.0, 1.0, np.inf, 0.5]
    rec["tmpl_idx"] = [0, 0, 1, 1, 2, 2]
    valid = np.array([True, True, True, True, True, False])
    got = output_model(rec, valid, 10)
    # NaN orders as +inf: record 1 (NaN) before record 4 (+inf)
    assert got["score"].tolist()[:3] == [1.0, 1.0, 3.0] and math.isnan(got["score"][3]) and math.isinf(got["score"][4])
    assert output_model(rec, valid, 2).tobytes() == rec[[2, 3]].tobytes()
    sel = fdcm.DistinctMatches(max_per_template=1)
    assert output_model(rec, valid, 10, np.zeros((3, 2), F32), sel)["tmpl_idx"].tolist() == [1, 0, 2]


def test_cpp_search_dense_builds(tmp_path):
    """searchDense of include/openfdcm_b200/openfdcm_cuda.hpp compiles against the C ABI and links."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "dense.cpp"
    src.write_text(r'''
#include "openfdcm_b200/openfdcm_cuda.hpp"
#include <cstdio>
int main() {
    using namespace openfdcm::cuda;
    try {
        const LineArray scene{0.f, 0.f, 50.f, 0.f, 50.f, 0.f, 50.f, 40.f};
        const std::vector<LineArray> templates{LineArray{0.f, 0.f, 20.f, 0.f}};
        const Dt3Cuda fm = buildCudaFeaturemap(scene, Dt3CudaParameters{});
        DenseSearch dense;
        dense.rotations = 8;
        dense.hasRoi = true;
        dense.roi = {{0.f, 0.f, 40.f, 30.f}};
        const PoseRefinement refine{};
        const DistinctMatches select{1};
        const auto a = searchDense(fm, templates, dense, ExponentialPenalty{1.5f}, 5);
        const auto b = searchDense(fm, templates, dense, ExponentialPenalty{1.5f}, 5, select);
        const auto c = searchDense(fm, templates, dense, ExponentialPenalty{1.5f}, 5, &select, &refine);
        std::printf("%zu %zu %zu\n", a.size(), b.size(), c.size());
    } catch (const std::exception& e) {
        std::printf("%s\n", e.what());
        return 1;
    }
    return 0;
}
''')
    exe = tmp_path / "dense"
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Werror", "-I" + os.path.join(root, "include"), str(src),
                           "-L" + os.path.join(root, "openfdcm_b200"), "-lfdcm_b200", "-Wl,-rpath," + os.path.join(root, "openfdcm_b200"),
                           "-o", str(exe)])
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode in (0, 1) and r.stdout
