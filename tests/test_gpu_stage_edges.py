"""The dense pose-grid search, edge coverage and the pose fit at the edges of the map geometry and of their parameters:
tiny maps, scenes far from the origin, the exact / literal boundary, depths 1 to 64, coverage radius 16, fit parameters at
their limits, rule-3 ties that decide the fit, and crowded fit cells.

Every device output is byte-equal to the models of tests/models/, and every model input that other modules take from the
device comes from the CPU oracle here: pose scores from Dt3Cpu.evaluate, edge masks from the zero pixels of a stage-1
Dt3Cpu, scene bins from closest_orientation of the shifted scene.  A defect shared by the device evaluate, mask or bins
and a stage kernel cannot cancel out.

Each case asserts on the CPU that it reaches what it targets (a map narrower than a word, one fit cell, a dense cell that
straddles two 32-column chunks, equal fp32 translations of adjacent grid points, a tie that decides the fit, ...); the
last test asserts that the module reached all of them.
"""
import math

import numpy as np
import pytest

import openfdcm_b200 as fdcm
from oracle import fdcm_oracle as orc
from tests.helpers import (BOUNDARY, DIST, FAR, far_scene, map_templates, oracle_bins, oracle_masks, oracle_pose_score, oracle_scores,
                           pinned_scene)
from tests.models.coverage import Dilated, coverage_model
from tests.models.dense import dense_records, grid, grid_valid, output_model, penalised, poses, rot_table, rotate_template
from tests.models.fit import SceneLines, fit_model, line_samples
from tests.models.refine import rotated
from tests.util import F32, synth_templates

pytestmark = pytest.mark.gpu
PEN = fdcm.ExponentialPenalty(1.5)
SIDES = [1, 2, 3, 5, 8, 15, 16, 17, 31, 32, 33, 64, 65]
FIT_CELL = 16   # kFitCell: side of a cell of the fit's scene-line grid

TARGETS = {"word_narrower_than_radius", "w_mod32", "one_fit_cell", "partial_fit_cell", "dense_empty", "dense_valid",
           "equal_translations", "straddling_cell", "stride_beyond_map", "rotations_4096", "literal_map", "tol_all_planes",
           "tol_window", "depth_1", "depth_2", "depth_64", "edges_on_border", "tie_shared_end", "tie_midway", "crowded_cells",
           "min_inliers_all", "lines_beyond_corners"}
REACHED = set()


# ---- maps and references -------------------------------------------------------------------------------------------
class Pair:
    """A device map and its oracle, size and translation asserted equal; the stage-1 oracle (edge masks) on demand."""

    def __init__(self, scene, depth=30, padding=1.0, dist="L2"):
        gd, od = DIST[dist]
        self.scene, self.depth, self.padding, self.od = scene, depth, padding, od
        self.g = fdcm.build_cuda_featuremap(scene, fdcm.Dt3CudaParameters(depth, 5.0, padding, gd))
        self.c = orc.Dt3Cpu(scene, depth, 5.0, padding, od)
        assert (self.g.width, self.g.height, self.g.depth) == (self.c.W, self.c.H, self.c.depth)
        assert self.g.get_scene_translation().tobytes() == self.c.shift.tobytes(), (self.g.get_scene_translation(), self.c.shift)
        self._masks = None

    @property
    def masks(self):
        if self._masks is None:
            self._masks = oracle_masks(orc.Dt3Cpu(self.scene, self.depth, 5.0, self.padding, self.od, stage=1))
        return self._masks

    def scene_lines(self):
        return SceneLines.of(self.scene, self.c.shift, oracle_bins(self.c, self.scene), self.c.depth, self.c.W, self.c.H)


def dense_model(p, tmpls, d, g=None):
    return dense_records(tmpls, fdcm.get_template_anchors(tmpls), d, p.c.shift, p.c.W, p.c.H, oracle_scores(p.c), 0, g)


def check_dense(p, tmpls, d, g=None, what="", outputs=None):
    """search_dense (scales=g) against the dense model: no penalty and PEN; the plain top 1, 10 and every valid record
    (up to 500), and two distinct selections.  Returns (rec, valid, rs) of the model."""
    rec, valid, rs = dense_model(p, tmpls, d, g)
    anchors, lengths = fdcm.get_template_anchors(tmpls), fdcm.get_template_lengths(tmpls)
    tset = fdcm.TemplateSet(tmpls)
    n_valid = int(valid.sum())
    REACHED.add("dense_valid" if n_valid else "dense_empty")
    outs = outputs or ((1, None), (10, None), (min(max(n_valid, 1), 500), None), (10, fdcm.DistinctMatches(max_per_template=1)),
                       (10, fdcm.DistinctMatches(radius=6.0, max_angle=0.3, across_templates=True)))
    for pen in (None, PEN):
        prec = penalised(rec, valid, lengths, pen, g)
        for k, sel in outs:
            got = fdcm.search_dense(p.g, tset, d, pen, k, select=sel, scales=g)
            want = output_model(prec, valid, k, anchors, sel, 0, rs if g is not None else None)
            assert got.tobytes() == want.tobytes(), f"{what} {d} {g} {pen} k={k} {sel}: got {got[:3]} want {want[:3]}"
    return rec, valid, rs


def check_coverage(p, tmpls, matches, cov, what=""):
    got = fdcm.match_coverage(p.g, tmpls, matches, cov)
    want = coverage_model(Dilated(p.masks, cov.radius, cov.bin_tolerance), p.c.shift, tmpls, matches)
    bad = np.flatnonzero(got.view(np.uint32) != want.view(np.uint32))
    assert len(bad) == 0, f"{what} {cov}: {len(bad)} of {len(matches)} differ, first {bad[:5]}: {got[bad[:3]]} != {want[bad[:3]]}"
    return got


def fit_reference(sc, c, tmpls, matches, fit):
    return fit_model(sc, tmpls, fdcm.get_template_anchors(tmpls), matches, fit, oracle_pose_score(c))


def check_fit(p, tmpls, matches, fit, what="", sc=None):
    sc = sc or p.scene_lines()
    got, gst = fdcm.fit_matches(p.g, tmpls, matches, fit, return_stats=True)
    want, wst = fit_reference(sc, p.c, tmpls, matches, fit)
    bad = np.flatnonzero([a.tobytes() != b.tobytes() for a, b in zip(got, want)])
    assert len(bad) == 0, (what, fit, bad[:5], got[bad[:2]], want[bad[:2]])
    bad = np.flatnonzero([a.tobytes() != b.tobytes() for a, b in zip(gst, wst)])
    assert len(bad) == 0, (what, fit, "stats", bad[:5], gst[bad[:2]], wst[bad[:2]])
    return got, gst


def fit_cells(W, H):
    """(gx, gy) of the fit's grid; a partial cell when W or H is not a multiple of the cell side."""
    gx, gy = -(-W // FIT_CELL), -(-H // FIT_CELL)
    if gx == 1:
        REACHED.add("one_fit_cell")
    if W % FIT_CELL or H % FIT_CELL:
        REACHED.add("partial_fit_cell")
    return gx, gy


# ---- matches --------------------------------------------------------------------------------------------------------
def placed(c, tmpls, n, seed, scale=(1.0, 1.0)):
    """n matches per template at a random rotation (and scale), translated inside the range that keeps the rotated template
    in the map: its two ends (where the fp32 sums may fall just outside: invalid matches) and random points between; a
    template that does not fit gets one pose off the map."""
    rng = np.random.default_rng(seed)
    shift = c.shift.astype(np.float64)
    out = []
    for t, tmpl in enumerate(tmpls):
        for i in range(n):
            th, s = rng.uniform(-math.pi, math.pi), rng.uniform(*scale)
            T = np.array([s * math.cos(th), -s * math.sin(th), 0, s * math.sin(th), s * math.cos(th), 0], F32)
            R = rotated(T[None], tmpl)[0].astype(np.float64)
            lo = -shift - np.array([R[:, [0, 2]].min(), R[:, [1, 3]].min()])
            hi = np.array([c.W - 1.0, c.H - 1.0]) - shift - np.array([R[:, [0, 2]].max(), R[:, [1, 3]].max()])
            if (lo > hi).any():
                T[2], T[5] = F32(1e6), F32(0)
            else:
                T[2], T[5] = (lo if i % 4 == 0 else hi if i % 4 == 1 else rng.uniform(lo, hi)).astype(F32)
            out.append((t, 0.0, T))
    return np.array(out, fdcm.MATCH_DTYPE)


def dense_matches(rec, valid, n):
    """Up to n valid dense records, spread over the record order."""
    h = np.flatnonzero(valid)
    return rec[h[np.linspace(0, len(h) - 1, min(n, len(h))).astype(int)]] if len(h) else rec[:0]


# ---- 1. tiny maps ---------------------------------------------------------------------------------------------------
TINY_DENSE = fdcm.DenseSearch(8, rot_start=0.1, stride=1, cell=3)
TINY_SCALES = fdcm.ScaleGrid(3, 0.7, 1.4)


@pytest.mark.parametrize("side", SIDES)
def test_tiny_maps(side):
    scene = pinned_scene(side, 12, seed=side)
    p = Pair(scene)
    assert p.c.W == side
    tmpls = map_templates(side, seed=side + 1)
    big = tmpls[-1].reshape(4, -1)
    assert big[2].max() - big[0].min() > side, "the last template is larger than the map"
    what = f"side {side}"
    recs = []
    for g in (None, TINY_SCALES):
        rec, valid, _ = check_dense(p, tmpls, TINY_DENSE, g, what)
        assert not (rec[valid]["tmpl_idx"] == len(tmpls) - 1).any(), "a template larger than the map has no valid pose"
        recs.append(dense_matches(rec, valid, 40))
    m = np.concatenate(recs + [placed(p.c, tmpls, 6, seed=side)])
    if side % 32:
        REACHED.add("w_mod32")
    for r in (0, 2, 16):
        if r >= side:
            REACHED.add("word_narrower_than_radius")
        check_coverage(p, tmpls, m, fdcm.EdgeCoverage(r, 1), what)
    fit_cells(p.c.W, p.c.H)
    sc = p.scene_lines()
    check_fit(p, tmpls, m, fdcm.PoseFit(), what, sc)
    check_fit(p, tmpls, m, fdcm.PoseFit(scale_range=(0.8, 1.25)), what, sc)


# ---- 2. far from the origin -----------------------------------------------------------------------------------------
TEMPLATE_FAR = 2.5e7   # template coordinates beyond 2^24: their dense translations have an fp32 spacing of 2 px or more


def equal_adjacent_translations(p, tmpls, d, g=None):
    """Whether some template, scale and rotation has two adjacent valid grid points (in u or in v) with equal fp32
    translations: then the bisection meets a flat run of shift + tx(u) and the cell minimum a tie of equal scores."""
    lx, ly, nx, ny = grid(d, p.c.shift, p.c.W, p.c.H)
    A, B = rot_table(d, g)
    anchors = fdcm.get_template_anchors(tmpls)
    for t, tmpl in enumerate(tmpls):
        for k in range(A.shape[0]):
            for r in range(d.rotations):
                P = poses(d, anchors[t], p.c.shift, p.c.W, p.c.H, r, g, k)
                ok = grid_valid(rotate_template(tmpl, A[k, r], B[k, r]), P, p.c.shift, p.c.W, p.c.H, nx, ny).reshape(ny, nx)
                P = P.reshape(ny, nx, 6)
                if (ok[:, 1:] & ok[:, :-1] & (P[:, 1:, 2] == P[:, :-1, 2])).any():
                    return True
                if (ok[1:, :] & ok[:-1, :] & (P[1:, :, 5] == P[:-1, :, 5])).any():
                    return True
    return False


def far_templates(tmpls):
    """The templates moved to TEMPLATE_FAR in x and y (their anchors move with them)."""
    return [np.ascontiguousarray(np.asarray(t, np.float64) + TEMPLATE_FAR, F32) for t in tmpls]


FAR_CASES = [(o, pad) for o in FAR for pad in (1.0, 1.5)]


@pytest.mark.parametrize("offset,padding", FAR_CASES, ids=[f"{o:g}-pad{pad}" for o, pad in FAR_CASES])
def test_far_from_origin(offset, padding):
    scene, tmpls = far_scene(offset, "small")
    p = Pair(scene, padding=padding)
    what = f"offset {offset:g} padding {padding}"
    ftmpls = far_templates(tmpls[:3])
    d = fdcm.DenseSearch(6, rot_start=0.2, rot_step=0.05, stride=3, cell=5)
    # the far templates at stride 1 in a 48-px box about the map centre (scene coordinates)
    ctr = (np.array([p.c.W, p.c.H]) / 2.0 - p.c.shift.astype(np.float64)).tolist()
    dfar = fdcm.DenseSearch(6, rot_start=0.2, rot_step=0.05, stride=1, cell=5, roi=(ctr[0] - 24, ctr[1] - 24, ctr[0] + 24, ctr[1] + 24))
    g = fdcm.ScaleGrid(2, 1.0, 1.0 + 2.0 ** -20)
    assert equal_adjacent_translations(p, ftmpls, dfar), f"{what}: no adjacent grid points with equal translations"
    assert equal_adjacent_translations(p, ftmpls, dfar, g), f"{what} scaled: no adjacent grid points with equal translations"
    REACHED.add("equal_translations")
    recs = []
    for ts, dd in ((tmpls, d), (ftmpls, dfar)):
        for gg in (None, g):
            rec, valid, _ = check_dense(p, ts, dd, gg, what)
            assert valid.any()
            recs.append(dense_matches(rec, valid, 20))
    m = np.concatenate([recs[0], recs[1], placed(p.c, tmpls, 4, seed=int(offset))])
    for r, tol in ((0, 0), (3, 1), (16, 2)):
        check_coverage(p, tmpls, m, fdcm.EdgeCoverage(r, tol), what)
    check_coverage(p, ftmpls, np.concatenate([recs[2], recs[3]]), fdcm.EdgeCoverage(2, 1), what + " far templates")
    sc = p.scene_lines()
    for fit in (fdcm.PoseFit(max_distance=8.0), fdcm.PoseFit(max_distance=8.0, scale_range=(0.8, 1.25))):
        check_fit(p, tmpls, m, fit, what, sc)
        check_fit(p, ftmpls, np.concatenate([recs[2], recs[3]]), fit, what + " far templates", sc)


# ---- 3. the exact / literal boundary --------------------------------------------------------------------------------
@pytest.mark.parametrize("side", BOUNDARY)
def test_exact_literal_boundary(side):
    scene = pinned_scene(side, 40, seed=side)
    p = Pair(scene)
    assert p.c.W == side and p.g.info.exact_dt_path == (1 if side <= 2897 else 0)
    if side > 2897:
        REACHED.add("literal_map")
    what = f"side {side}"
    tmpls = map_templates(64, seed=side)
    sh = p.c.shift.astype(np.float64)
    # a region over the last 70 map pixels of both axes and past the map (its upper end is clamped to W - 1)
    roi = tuple(float(v) for v in (side - 70 - sh[0], side - 70 - sh[1], side + 10 - sh[0], side + 10 - sh[1]))
    d = fdcm.DenseSearch(4, rot_start=0.3, stride=2, cell=7, roi=roi)
    lx, ly, nx, ny = grid(d, p.c.shift, p.c.W, p.c.H)
    assert lx + (nx - 1) * d.stride >= side - 2 and nx * ny < 2000
    recs = []
    for g in (None, TINY_SCALES):
        rec, valid, _ = check_dense(p, tmpls, d, g, what)
        assert valid.any()
        recs.append(dense_matches(rec, valid, 20))
    m = np.concatenate(recs + [placed(p.c, tmpls, 4, seed=side)])
    check_coverage(p, tmpls, m, fdcm.EdgeCoverage(3, 1), what)
    check_coverage(p, tmpls, m, fdcm.EdgeCoverage(16, 0), what)
    sc = p.scene_lines()
    check_fit(p, tmpls, m, fdcm.PoseFit(max_distance=16.0), what, sc)
    check_fit(p, tmpls, m, fdcm.PoseFit(max_distance=16.0, scale_range=(0.8, 1.25)), what, sc)


# ---- 4. depth and parameter extremes ---------------------------------------------------------------------------------
def border_scene(side=100, n=40, seed=5):
    """The outline of [0, side-1]^2 and n random lines inside: at padding 1 edge pixels in the first and last map rows and
    columns, and a width that is not a multiple of 32."""
    rng = np.random.default_rng(seed)
    e = side - 1.0
    outline = np.array([[0, 0, e, 0], [e, 0, e, e], [e, e, 0, e], [0, e, 0, 0]], np.float64).T
    p1 = rng.uniform(0, e, (2, n))
    ang = rng.uniform(0, 2 * math.pi, n)
    p2 = np.clip(p1 + rng.uniform(3, side / 3, n) * np.stack([np.cos(ang), np.sin(ang)]), 0, e)
    return np.ascontiguousarray(np.concatenate([outline, np.concatenate([p1, p2])], axis=1), F32)


@pytest.mark.parametrize("depth", [1, 2, 7, 64])
def test_coverage_and_fit_depths(depth):
    scene = border_scene()
    p = Pair(scene, depth=depth)
    REACHED.add(f"depth_{depth}")
    assert p.c.W % 32 and p.masks[:, 0, :].any() and p.masks[:, -1, :].any() and p.masks[:, :, 0].any() and p.masks[:, :, -1].any()
    REACHED.add("edges_on_border")
    tmpls = map_templates(100, seed=depth)
    m = placed(p.c, tmpls, 12, seed=depth)
    what = f"depth {depth}"
    # bin tolerances on both sides of the switch 2 tol + 1 >= D (every plane) and, at D = 64, tol 31 and 32
    tols = sorted({0, 1, max(0, (depth - 1) // 2 - 1), (depth - 1) // 2, depth // 2, 32} if depth > 1 else {0, 1, 32})
    for tol in tols:
        REACHED.add("tol_all_planes" if 2 * tol + 1 >= depth else "tol_window")
        for r in (0, 16):
            check_coverage(p, tmpls, m, fdcm.EdgeCoverage(r, tol), what)
    sc = p.scene_lines()
    for tol in (0, 1, depth // 2):
        check_fit(p, tmpls, m, fdcm.PoseFit(bin_tolerance=tol, max_distance=6.0), what, sc)
        check_fit(p, tmpls, m, fdcm.PoseFit(bin_tolerance=tol, max_distance=6.0, scale_range=(0.8, 1.25)), what, sc)


def test_fit_parameter_extremes():
    scene = border_scene(side=120, n=60, seed=9)
    p = Pair(scene)
    tmpls = map_templates(100, seed=11)[:4]
    m = placed(p.c, tmpls, 6, seed=12)
    sc = p.scene_lines()
    extreme = dict(sample_step=0.5, iterations=100, bin_tolerance=32, max_distance=16.0, tolerance=0.0)
    for scale in (None, (0.5, 2.0)):
        check_fit(p, tmpls, m, fdcm.PoseFit(**extreme, scale_range=scale), "extremes", sc)
    # min_inliers equal to the sample count of the template: the fit iterates only while every sample is an inlier
    t = 0
    n = sum(len(line_samples(l, 0.5)[0]) for l in np.asarray(tmpls[t], F32).reshape(4, -1).T)
    one = m[m["tmpl_idx"] == t]
    for scale in (None, (0.5, 2.0)):
        got, st = check_fit(p, tmpls, one, fdcm.PoseFit(**{**extreme, "min_inliers": n}, scale_range=scale), "min_inliers", sc)
        assert (st["n_samples"][~np.isnan(got["score"])] == n).all()
    REACHED.add("min_inliers_all")


def test_coverage_radius_16_narrow_and_wide_words():
    """Radius 16 with funnel shifts across both neighbouring words on a map of 3 words whose last is partial."""
    scene = border_scene(side=75, n=30, seed=13)
    p = Pair(scene)
    assert p.c.W == 75 and p.c.W % 32
    tmpls = map_templates(75, seed=14)
    m = placed(p.c, tmpls, 16, seed=15)
    for tol in (0, 2):
        check_coverage(p, tmpls, m, fdcm.EdgeCoverage(16, tol), "side 75")


def straddles(ulo, uhi, cell):
    """Whether a cell of `cell` columns holds columns of two 32-column chunks of the valid range [ulo, uhi]."""
    for c0 in range((ulo // cell) * cell, uhi + 1, cell):
        a, b = max(c0, ulo), min(c0 + cell - 1, uhi)
        if a <= b and (a - ulo) // 32 != (b - ulo) // 32:
            return True
    return False


@pytest.mark.parametrize("cell", [31, 33, 64])
def test_dense_cells_across_chunks(cell):
    scene = pinned_scene(150, 40, seed=cell)
    p = Pair(scene)
    tmpls = map_templates(40, seed=cell)[:4]
    d = fdcm.DenseSearch(3, rot_start=0.4, rot_step=1.3, stride=1, cell=cell)
    rec, valid, _ = check_dense(p, tmpls, d, None, f"cell {cell}")
    check_dense(p, tmpls, d, fdcm.ScaleGrid(2, 0.9, 1.2), f"cell {cell}", outputs=((10, None), (50, None)))
    # the valid u range of some rotation has a cell that straddles two chunks
    lx, ly, nx, ny = grid(d, p.c.shift, p.c.W, p.c.H)
    A, B = rot_table(d)
    anchors = fdcm.get_template_anchors(tmpls)
    hit = False
    for t, tmpl in enumerate(tmpls):
        for r in range(d.rotations):
            P = poses(d, anchors[t], p.c.shift, p.c.W, p.c.H, r)
            ok = grid_valid(rotate_template(tmpl, A[0, r], B[0, r]), P, p.c.shift, p.c.W, p.c.H, nx, ny).reshape(ny, nx)
            us = np.flatnonzero(ok.any(axis=0))
            hit |= len(us) > 0 and straddles(int(us[0]), int(us[-1]), cell)
    assert hit and valid.any()
    REACHED.add("straddling_cell")


def test_dense_stride_beyond_map_and_4096_rotations():
    scene = pinned_scene(33, 12, seed=3)
    p = Pair(scene)
    tmpls = map_templates(33, seed=4)
    d = fdcm.DenseSearch(16, rot_step=0.4, stride=1000, cell=1)
    assert grid(d, p.c.shift, p.c.W, p.c.H)[2:] == (1, 1)
    check_dense(p, tmpls, d, None, "stride 1000")
    # a grid of 4096 rotations on a small map: the record count and every block of the dense kernel
    REACHED.add("stride_beyond_map")
    small = pinned_scene(17, 10, seed=5)
    p = Pair(small)
    tmpls = map_templates(17, seed=6)[:1]
    d = fdcm.DenseSearch(4096, rot_start=-math.pi, rot_step=2 * math.pi / 4096, stride=4, cell=2)
    rec, valid, _ = check_dense(p, tmpls, d, None, "4096 rotations", outputs=((10, None), (500, None),
                                                                               (10, fdcm.DistinctMatches(max_per_template=2))))
    assert valid.sum() > 1000
    REACHED.add("rotations_4096")


# ---- 5. rule-3 ties that decide the fit ------------------------------------------------------------------------------
def reversed_lines(sc):
    """The scene lines in reverse order: rule 3 on them takes the highest index among equal distances."""
    return SceneLines(sc.lines[::-1].copy(), sc.bins[::-1].copy(), sc.D, sc.shift, sc.W, sc.H)


def check_deciding_ties(p, tmpls, m, fit, what):
    """The fit against the model, and the model with the opposite tie rule differs: the ties decide some output."""
    sc = p.scene_lines()
    got, gst = check_fit(p, tmpls, m, fit, what, sc)
    other, ost = fit_reference(reversed_lines(sc), p.c, tmpls, m, fit)
    assert got.tobytes() != other.tobytes() or gst.tobytes() != ost.tobytes(), f"{what}: no tie decides the fit"


def test_ties_at_shared_end_points():
    """Polylines whose segments share end points; a template line outside each convex corner: its samples are nearest to
    the shared end point of both segments (u clamped to 1 on one, 0 on the other), at equal distances."""
    rng = np.random.default_rng(21)
    lines, tmpl_lines = [], []
    for q in range(6):
        c = np.array([40.0 + 60 * (q % 3), 40.0 + 70 * (q // 3)])
        a0 = rng.uniform(0, 2 * math.pi)
        turn = rng.uniform(0.3, 0.6)
        d1, d2 = np.array([math.cos(a0), math.sin(a0)]), np.array([math.cos(a0 + turn), math.sin(a0 + turn)])
        A, B, C = np.round(c - 20 * d1), np.round(c), np.round(c + 20 * d2)
        lines += [(*A, *B), (*B, *C)]
        # the outer bisector of the corner at B, 2 px out: a short template line across it
        out = -(d2 - d1) / np.linalg.norm(d2 - d1)
        m = B + 2.0 * out
        tang = np.array([-out[1], out[0]])
        tmpl_lines.append((*(m - 1.5 * tang), *(m + 1.5 * tang)))
    scene = np.asarray(lines, F32).T.copy()
    p = Pair(scene, padding=1.3)
    tmpl = np.asarray(tmpl_lines, F32).T.copy()
    m = np.zeros(1, fdcm.MATCH_DTYPE)
    m["transform"] = [1, 0, 0, 0, 1, 0]
    for fit in (fdcm.PoseFit(bin_tolerance=32, max_distance=4.0, min_inliers=3, iterations=3),
                fdcm.PoseFit(bin_tolerance=32, max_distance=4.0, min_inliers=3, iterations=3, scale_range=(0.8, 1.25))):
        check_deciding_ties(p, [tmpl], m, fit, "shared end points")
    REACHED.add("tie_shared_end")


def test_ties_midway_between_parallel_lines():
    """Scene squares 2 px inside and 2 px outside a template square at an integer pose: every sample of a side lies
    exactly midway between two parallel scene lines.  The lower index of each pair is the outer line on the top and left
    sides and the inner line on the bottom and right: the lower-index rule pulls the template up and left, the
    higher-index rule down and right."""
    sq = lambda a, b: [(a, a, b, a), (b, a, b, b), (b, b, a, b), (a, b, a, a)]   # top, right, bottom, left
    outer, inner = sq(20, 80), sq(24, 76)
    scene = np.asarray([outer[0], inner[1], inner[2], outer[3], inner[0], outer[1], outer[2], inner[3]], F32).T.copy()
    p = Pair(scene, padding=1.5)
    tmpl = np.asarray(sq(0, 56), F32).T.copy()
    sh = p.c.shift
    assert ((sh * 4) == np.round(sh * 4)).all(), "the shift keeps integer coordinates exact"
    m = np.zeros(2, fdcm.MATCH_DTYPE)
    m["transform"] = [[1, 0, 22, 0, 1, 22], [0, -1, 78, 1, 0, 22]]   # the square, and the square turned by 90 degrees
    for fit in (fdcm.PoseFit(max_distance=3.0, bin_tolerance=0, iterations=5),
                fdcm.PoseFit(max_distance=3.0, bin_tolerance=0, iterations=5, scale_range=(0.8, 1.25))):
        check_deciding_ties(p, [tmpl], m, fit, "midway")
    REACHED.add("tie_midway")


# ---- 6. crowded fit cells --------------------------------------------------------------------------------------------
def cell_counts(lines, reach, gx, gy):
    """The entries of every cell of the fit's grid (fit_line_cells: the cells whose centre lies within reach of a line)."""
    cnt = np.zeros(gx * gy, np.int64)
    cy, cx = np.divmod(np.arange(gx * gy), gx)
    px, py = (cx + 0.5) * FIT_CELL, (cy + 0.5) * FIT_CELL
    for ax, ay, bx, by in lines.astype(np.float64):
        dx, dy = bx - ax, by - ay
        l2 = dx * dx + dy * dy
        if not l2 > 0:
            continue
        u = np.clip(((px - ax) * dx + (py - ay) * dy) / l2, 0.0, 1.0)
        cnt += ((px - (ax + u * dx)) ** 2 + (py - (ay + u * dy)) ** 2 <= reach * reach)
    return cnt


def test_crowded_fit_cells():
    rng = np.random.default_rng(31)
    n = 2000
    p1 = rng.uniform(0, 199, (2, n))
    ang = rng.uniform(0, 2 * math.pi, n)
    p2 = np.clip(p1 + rng.uniform(0.5, 3.0, n) * np.stack([np.cos(ang), np.sin(ang)]), 0, 199)
    pins = np.array([[0, 0, 1, 0], [198, 199, 199, 199]], np.float64).T
    scene = np.ascontiguousarray(np.concatenate([np.concatenate([p1, p2]), pins], axis=1), F32)
    p = Pair(scene)
    assert p.c.W == 200
    sc = p.scene_lines()
    gx, gy = fit_cells(p.c.W, p.c.H)
    for md in (8.0, 16.0):
        cnt = cell_counts(sc.lines, md + 2.0 + 0.7072 * FIT_CELL, gx, gy)
        assert cnt.max() >= 100, cnt.max()
    REACHED.add("crowded_cells")
    tmpls = synth_templates(4, 8, 200, seed=32, max_len=60.0)
    m = placed(p.c, tmpls, 5, seed=33)
    for md in (8.0, 16.0):
        for scale in (None, (0.8, 1.25)):
            check_fit(p, tmpls, m, fdcm.PoseFit(max_distance=md, bin_tolerance=2, iterations=4, scale_range=scale), "crowded", sc)


def segment_distance(p, line):
    a, b = np.asarray(line[:2], np.float64), np.asarray(line[2:], np.float64)
    u = np.clip(np.dot(p - a, b - a) / np.dot(b - a, b - a), 0.0, 1.0)
    return float(np.linalg.norm(p - (a + u * (b - a))))


@pytest.mark.parametrize("md", [3.0, 8.0])
def test_fit_lines_beyond_cell_corners(md):
    """A sample in the corner of its fit cell whose only correspondence is a scene line beyond that corner: the line lies
    farther than max_distance + 2 + kFitCell / 2 from the cell's centre and within the grid's reach
    (max_distance + 2 + 0.7072 kFitCell), so a grid that reaches less than the cell's half-diagonal loses it."""
    delta = md - 0.4   # the scene line crosses the diagonal delta px beyond the corner; the last sample is 0.07 px inside
    lines, tmpl = [], []
    for cx, cy in ((2, 2), (5, 3), (8, 8), (3, 9)):
        K = np.array([(cx + 1.0) * FIT_CELL, (cy + 1.0) * FIT_CELL])
        f = K + delta / math.sqrt(2.0)
        lines.append((f[0] - 3, f[1] + 3, f[0] + 3, f[1] - 3))   # across the diagonal
        tmpl.append((K[0] - 4, K[1] - 4, K[0] - 0.05, K[1] - 0.05))   # along the diagonal, inside the cell
        centre = K - FIT_CELL / 2.0
        dist = segment_distance(centre, lines[-1])
        assert md + 2.0 + 0.5 * FIT_CELL < dist <= md + 2.0 + 0.7072 * FIT_CELL, dist
        assert segment_distance(np.array(tmpl[-1][2:]), lines[-1]) <= md
    pins = [(0, 0, 1, 0), (198, 199, 199, 199)]
    scene = np.asarray(lines + pins, F32).T.copy()
    p = Pair(scene)
    assert p.c.W == 200 and not p.c.shift.any(), "map coordinates are scene coordinates"
    tmpl = np.asarray(tmpl, F32).T.copy()
    m = np.zeros(1, fdcm.MATCH_DTYPE)
    m["transform"] = [1, 0, 0, 0, 1, 0]
    for scale in (None, (0.8, 1.25)):
        got, st = check_fit(p, [tmpl], m, fdcm.PoseFit(max_distance=md, bin_tolerance=32, min_inliers=3, iterations=3,
                                                       scale_range=scale), f"corners md {md}")
        assert st["n_inliers"][0] >= 3
    REACHED.add("lines_beyond_corners")


# ---- reach ----------------------------------------------------------------------------------------------------------
def test_every_target_reached():
    """Runs after the cases above (file order): together they must have reached every target."""
    if not REACHED:
        pytest.skip("no case of this module ran")
    assert TARGETS - REACHED == set(), f"targets never reached: {sorted(TARGETS - REACHED)}"
