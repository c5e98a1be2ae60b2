"""Match verification (fdcm_match_coverage, EdgeCoverage): the numpy model of the oriented edge coverage.  The rules are
in include/fdcm_b200.h."""
import numpy as np
from scipy.ndimage import maximum_filter

from openfdcm_b200 import _lib
from oracle import fdcm_oracle as orc
from tests.models.refine import rotated, valid_poses
from tests.util import F32


def table_bins(depth, lines):
    """Orientation bins of (n, 4) lines through the slope table the device uses (fdcm_orientation_bins' table path)."""
    lines = np.ascontiguousarray(lines, F32).reshape(-1, 4)
    n = lines.shape[0]
    a, b = np.zeros(max(n, 1), np.int32), np.zeros(max(n, 1), np.int32)
    if n:
        _lib.check(_lib.lib().fdcm_orientation_bins(int(depth), _lib.ptr(lines), n, _lib.ptr(a), _lib.ptr(b)))
    return b[:n]


def tolerance_planes(b, D, tol):
    """Rule 4: the planes q with min(|q - b|, D - |q - b|) <= tol."""
    q = np.arange(D)
    d = np.abs(q - b)
    return q[np.minimum(d, D - d) <= tol]


class Dilated:
    """Rule 4 on given masks (D, H, W): dilated(b)[y, x] holds iff a plane within the tolerance of b has an edge pixel in
    the (2r + 1)^2 window around (x, y), inside the map."""

    def __init__(self, masks, radius, tol):
        self.masks = np.asarray(masks).astype(bool)
        self.radius, self.tol = int(radius), int(tol)
        self.cache = {}

    def __call__(self, b):
        if b not in self.cache:
            D = self.masks.shape[0]
            m = self.masks[tolerance_planes(b, D, self.tol)].any(axis=0)
            self.cache[b] = maximum_filter(m, size=2 * self.radius + 1, mode="constant", cval=False)
        return self.cache[b]


def coverage_counts(dil, shift, tmpl, T):
    """Rules 1-5 for one match: (n_covered, n_total), or None when the coverage is NaN (rule 2)."""
    D, H, W = dil.masks.shape
    t = np.asarray(tmpl, F32).reshape(4, -1)
    L = t.shape[1]
    T = np.asarray(T, F32).reshape(6)
    if D == 0 or H == 0 or W == 0 or L == 0 or not valid_poses(T[None], t, shift, W, H)[0]:
        return None
    R = rotated(T[None], t)[0]                        # (L, 4) rotated end points
    bins = table_bins(D, R)
    with np.errstate(all="ignore"):
        ox, oy = F32(shift[0]) + T[2], F32(shift[1]) + T[5]
        M = np.stack([R[:, 0] + ox, R[:, 1] + oy, R[:, 2] + ox, R[:, 3] + oy], axis=1).astype(F32)
    covered = total = 0
    for q in range(L):
        px = orc.rasterize_line(M[q])                 # rows (x, y)
        assert ((px[:, 0] >= 0) & (px[:, 0] < W) & (px[:, 1] >= 0) & (px[:, 1] < H)).all()
        total += len(px)
        covered += int(dil(int(bins[q]))[px[:, 1], px[:, 0]].sum())
    return covered, total


def coverage_model(dil, shift, tmpls, matches, tmpl_idx_base=0):
    """Rule 5 for every match: float32 coverage, NaN where rule 2 says so."""
    out = np.full(len(matches), np.nan, F32)
    for i, m in enumerate(matches):
        c = coverage_counts(dil, shift, tmpls[int(m["tmpl_idx"]) - tmpl_idx_base], m["transform"])
        if c is not None:
            out[i] = F32(c[0]) / F32(c[1])
    return out


def filter_model(cov, min_coverage):
    """Rule 6: the records kept by the filter (NaN coverage is dropped)."""
    with np.errstate(invalid="ignore"):
        return cov >= F32(min_coverage)
