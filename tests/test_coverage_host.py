"""Match verification (fdcm_match_coverage, EdgeCoverage): the numpy model of the oriented edge coverage
(tests/models/coverage.py), pinned by known answers.  The rules are in include/fdcm_b200.h; tests/test_gpu_coverage.py
compares the device against this model byte for byte.  No kernel is launched here."""
import ctypes as C
import math

import numpy as np
import pytest

import openfdcm_b200 as fdcm
from openfdcm_b200 import _lib
from oracle import fdcm_oracle as orc
from tests.models.coverage import Dilated, coverage_counts, coverage_model, filter_model, table_bins, tolerance_planes
from tests.util import F32


# ---- known answers ---------------------------------------------------------------------------------------------------
IDENT = [1, 0, 0, 0, 1, 0]


def masks_with(D, H, W, pixels):
    m = np.zeros((D, H, W), np.uint8)
    for q, x, y in pixels:
        m[q, y, x] = 1
    return m


def one(masks, tmpl, T=IDENT, radius=0, tol=0, shift=(0.0, 0.0)):
    c = coverage_counts(Dilated(masks, radius, tol), shift, np.asarray(tmpl, F32).reshape(4, -1), T)
    return c


def test_coverage_params_layout():
    assert C.sizeof(_lib.CoverageParams) == 12
    assert [f[0] for f in _lib.CoverageParams._fields_] == ["radius", "bin_tolerance", "min_coverage"]
    e = fdcm.EdgeCoverage()
    assert (e.radius, e.bin_tolerance, e.min_coverage) == (2, 1, 0.0)


def test_horizontal_vertical_diagonal_and_degenerate_lines():
    D, H, W = 4, 20, 20
    bins = table_bins(D, np.array([[2, 5, 12, 5], [5, 2, 5, 12], [2, 2, 9, 9], [7, 7, 7, 7]], F32))
    # horizontal: 11 samples (2..12, 5); 6 of them on edges of its plane
    m = masks_with(D, H, W, [(bins[0], x, 5) for x in range(2, 8)])
    assert one(m, [2, 5, 12, 5]) == (6, 11)
    # vertical: 11 samples (5, 2..12); every one of them covered
    m = masks_with(D, H, W, [(bins[1], 5, y) for y in range(0, 20)])
    assert one(m, [5, 2, 5, 12]) == (11, 11)
    # diagonal: 8 samples (2..9, 2..9); covered on the diagonal only
    m = masks_with(D, H, W, [(bins[2], 4, 4), (bins[2], 4, 5)])
    assert one(m, [2, 2, 9, 9]) == (1, 8)
    # degenerate: one sample at the rounded point
    m = masks_with(D, H, W, [(bins[3], 7, 7)])
    assert one(m, [7.2, 6.8, 7.2, 6.8]) == (1, 1)
    assert one(np.zeros((D, H, W), np.uint8), [7, 7, 7, 7]) == (0, 1)


def test_samples_equal_the_build_raster():
    """The samples are the pixels the DT3 build draws for the same line (rasterizeLine, drawing.h:74-102)."""
    for line in ([3.4, 2.6, 17.9, 11.2], [15, 1, 2, 18], [0, 0, 19, 0], [4.5, 4.5, 4.5, 15.5]):
        px = orc.rasterize_line(np.array(line, F32))
        img = orc.draw_lines(np.zeros((20, 20), F32), np.array(line, F32).reshape(4, 1), 1.0)
        assert set(map(tuple, px.tolist())) == set(map(tuple, np.argwhere(img > 0)[:, ::-1].tolist()))


@pytest.mark.parametrize("radius", [0, 1, 3, 16])
def test_edge_at_radius_is_covered_and_at_radius_plus_one_is_not(radius):
    D, H, W = 2, 60, 60
    b = table_bins(D, np.array([[20, 30, 20, 30]], F32))[0]
    for dx, dy in ((radius, 0), (0, -radius), (radius, radius), (-radius, radius)):
        assert one(masks_with(D, H, W, [(b, 20 + dx, 30 + dy)]), [20, 30, 20, 30], radius=radius) == (1, 1)
    for dx, dy in ((radius + 1, 0), (0, radius + 1), (radius + 1, radius), (-radius - 1, -radius - 1)):
        assert one(masks_with(D, H, W, [(b, 20 + dx, 30 + dy)]), [20, 30, 20, 30], radius=radius) == (0, 1)


def test_tolerance_wraps_between_the_first_and_last_plane():
    D, H, W = 8, 10, 10
    line = [1, 5, 8, 5]                              # horizontal
    b = int(table_bins(D, np.array([line], F32))[0])
    other = (b - 1) % D                              # circular neighbour (D - 1 when b == 0)
    far = (b + D // 2) % D
    m = masks_with(D, H, W, [(other, x, 5) for x in range(1, 9)])
    assert one(m, line, tol=0) == (0, 8)
    assert one(m, line, tol=1) == (8, 8)
    assert set(tolerance_planes(0, D, 1).tolist()) == {0, 1, D - 1}
    assert set(tolerance_planes(D - 1, D, 1).tolist()) == {D - 2, D - 1, 0}
    m = masks_with(D, H, W, [(far, x, 5) for x in range(1, 9)])
    assert one(m, line, tol=D // 2 - 1) == (0, 8)
    for tol in (D // 2, D // 2 + 1, 32):             # tolerance >= D / 2: every plane
        assert tolerance_planes(b, D, tol).tolist() == list(range(D))
        assert one(m, line, tol=tol) == (8, 8)


def test_duplicate_samples_count_every_time():
    D, H, W = 2, 10, 10
    # the same line twice: every sample counts twice
    b = int(table_bins(D, np.array([[1, 1, 6, 1]], F32))[0])
    m = masks_with(D, H, W, [(b, 1, 1)])
    assert one(m, [[1, 1], [1, 1], [6, 6], [1, 1]]) == (2, 12)
    # two lines meeting at (5, 1): the shared pixel is a sample of both
    bh, bv = (int(v) for v in table_bins(D, np.array([[1, 1, 5, 1], [5, 1, 5, 4]], F32)))
    m = masks_with(D, H, W, [(bh, 5, 1), (bv, 5, 1)])
    assert one(m, [[1, 5], [1, 1], [5, 5], [1, 4]]) == (2, 9)


def test_validity_at_the_map_border():
    D, H, W = 2, 10, 12
    m = np.ones((D, H, W), np.uint8)
    assert one(m, [0, 0, 11, 9]) == (12, 12)
    assert one(m, [0, 0, 11, 9], T=[1, 0, 0.1, 0, 1, 0]) is None           # x = 11.1 > W - 1
    assert one(m, [0, 0, 11, 9], T=[1, 0, -0.001, 0, 1, 0]) is None        # x < 0
    assert one(m, [0, 0, 11, 9], T=[1, 0, 0, 0, 1, 0.0], shift=(0.0, 0.5)) is None
    assert one(m, [1, 1, 10, 8], T=[1, 0, -1, 0, 1, -1]) == (10, 10)        # exactly on the border after the shift


def test_nan_transform_and_empty_template_give_nan():
    D, H, W = 2, 10, 10
    m = np.ones((D, H, W), np.uint8)
    dil = Dilated(m, 1, 0)
    tmpls = [np.array([[1], [1], [5], [5]], F32), np.zeros((4, 0), F32)]
    rec = np.zeros(4, _lib.MATCH_DTYPE)
    rec["transform"] = IDENT
    rec["transform"][1, 2] = np.nan
    rec["transform"][2, 1] = np.nan                  # a NaN rotation entry (multiplied by y = 1)
    rec["tmpl_idx"] = [0, 0, 0, 1]
    got = coverage_model(dil, (0.0, 0.0), tmpls, rec)
    assert got[0] == F32(1) and np.isnan(got[1:]).all()
    assert np.isnan(coverage_model(Dilated(np.zeros((0, 0, 0), np.uint8), 1, 0), (0.0, 0.0), tmpls, rec[:1])).all()


def test_coverage_is_float32_division_and_the_filter_drops_nan():
    cov = np.array([F32(1) / F32(3), np.nan, 0.5, 0.0], F32)
    assert filter_model(cov, 0.5).tolist() == [False, False, True, False]
    assert filter_model(cov, F32(1) / F32(3)).tolist() == [True, False, True, False]


def test_bins_come_from_the_rotated_line():
    """A line rotated by 90 degrees takes the bin of the rotated slope, not of the template's."""
    D, H, W = 6, 30, 30
    line = [0, 0, 10, 0]
    T = [0, -1, 15, 1, 0, 5]                         # (x, y) -> (-y + 15, x + 5): vertical at x = 15
    bv = int(table_bins(D, np.array([[0, 0, 0, 10]], F32))[0])
    bh = int(table_bins(D, np.array([line], F32))[0])
    assert bv != bh
    m = masks_with(D, H, W, [(bv, 15, y) for y in range(5, 16)])
    assert one(m, line, T=T) == (11, 11)
    m = masks_with(D, H, W, [(bh, 15, y) for y in range(5, 16)])
    assert one(m, line, T=T) == (0, 11)


@pytest.mark.parametrize("bad", [dict(radius=-1), dict(radius=17), dict(bin_tolerance=-1), dict(bin_tolerance=33),
                                 dict(min_coverage=-0.01), dict(min_coverage=1.01), dict(min_coverage=math.nan)])
def test_match_coverage_rejects_bad_parameters_before_any_device_work(bad):
    p = _lib.CoverageParams(*[bad.get(k, d) for k, d in (("radius", 2), ("bin_tolerance", 1), ("min_coverage", 0.0))])
    st = _lib.lib().fdcm_match_coverage(None, None, 0, C.byref(p), None, 0, None)
    assert st == _lib.FDCM_ERR_INVALID
    msg = _lib.lib().fdcm_last_error().decode()
    assert any(s in msg for s in ("0..16", "0..32", "[0, 1]")), msg


def test_cpp_match_coverage_builds(tmp_path):
    """matchCoverage and the verified searchTopK / searchDense of include/openfdcm_b200/openfdcm_cuda.hpp compile and link."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "coverage.cpp"
    src.write_text(r'''
#include "openfdcm_b200/openfdcm_cuda.hpp"
#include <cstdio>
int main() {
    using namespace openfdcm::cuda;
    try {
        const LineArray scene{0.f, 0.f, 50.f, 0.f, 50.f, 0.f, 50.f, 40.f};
        const std::vector<LineArray> templates{LineArray{0.f, 0.f, 20.f, 0.f}};
        const Dt3Cuda fm = buildCudaFeaturemap(scene, Dt3CudaParameters{});
        const EdgeCoverage verify{2, 1, 0.5f};
        const auto a = searchTopK(DefaultSearch{4, 4}, BatchOptimize{10}, ExponentialPenalty{1.5f}, fm, templates, scene, 5, verify);
        const DistinctMatches select{1};
        const PoseRefinement refine{};
        const auto b = searchTopK(DefaultSearch{4, 4}, BatchOptimize{10}, ExponentialPenalty{1.5f}, fm, templates, scene, 5, &select, &refine,
                                  verify);
        DenseSearch dense;
        dense.rotations = 8;
        const auto c = searchDense(fm, templates, dense, ExponentialPenalty{1.5f}, 5, nullptr, nullptr, verify);
        const std::vector<float> cov = matchCoverage(fm, templates, a);
        const std::vector<float> cov2 = matchCoverage(fm, templates, b, EdgeCoverage{0, 0, 0.f});
        std::printf("%zu %zu %zu %zu %zu\n", a.size(), b.size(), c.size(), cov.size(), cov2.size());
    } catch (const std::exception& e) {
        std::printf("%s\n", e.what());
        return 1;
    }
    return 0;
}
''')
    exe = tmp_path / "coverage"
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Werror", "-I" + os.path.join(root, "include"), str(src),
                           "-L" + os.path.join(root, "openfdcm_b200"), "-lfdcm_b200", "-Wl,-rpath," + os.path.join(root, "openfdcm_b200"),
                           "-o", str(exe)])
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode in (0, 1) and r.stdout
