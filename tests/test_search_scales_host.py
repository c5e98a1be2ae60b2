"""Scale in the line-alignment search (fdcm_search_scales, search_topk / search_all with scales=ScaleGrid): the symbol in
the header and the library, and argument rejection before any device work.  The rules are in include/fdcm_b200.h;
tests/test_gpu_search_scales.py compares the device against the CPU oracle.  No kernel is launched here."""
import ctypes as C
import os
import re

import pytest

import openfdcm_b200 as fdcm
from openfdcm_b200 import _lib
from tests.helpers import dense_poses_hook

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BAD_GRIDS = [fdcm.ScaleGrid(0), fdcm.ScaleGrid(65), fdcm.ScaleGrid(2, 0.0, 1.0), fdcm.ScaleGrid(2, -1.0, 1.0), fdcm.ScaleGrid(2, float("nan"), 1.0),
             fdcm.ScaleGrid(2, float("inf"), 1.0), fdcm.ScaleGrid(2, 1.0, 0.0), fdcm.ScaleGrid(2, 1.0, -2.0), fdcm.ScaleGrid(2, 1.0, float("nan")),
             fdcm.ScaleGrid(64, 1.0, 1e10), fdcm.ScaleGrid(64, 1.0, 1e-10)]


def params(top_k=10):
    return _lib.SearchParams(4, 4, 10, 2, 1.5, top_k, 0, 0, 0.0, 0.0, 0.0, 0.0)


def call(p=None, g=None, select=None, refine=None, cov=None):
    n = C.c_int64(7)
    st = _lib.lib().fdcm_search_scales(None, None, None, 0, None if p is None else C.byref(p), None if g is None else C.byref(g._params()),
                                       None if select is None else C.byref(select._params()),
                                       None if refine is None else C.byref(refine._params()),
                                       None if cov is None else C.byref(cov._params()), None, 0, C.byref(n))
    return st, _lib.lib().fdcm_last_error().decode()


def test_header_and_library_export_the_symbol():
    with open(os.path.join(ROOT, "include", "fdcm_b200.h")) as f:
        h = f.read()
    assert re.search(r"fdcm_status fdcm_search_scales\(const fdcm_dt3\* map, const fdcm_templates\* templates", h)
    assert hasattr(_lib.lib(), "fdcm_search_scales")
    assert "fdcm_search_scales" in _lib.SIGNATURES
    assert _lib.lib().fdcm_abi_version() == 3


@pytest.mark.parametrize("g", BAD_GRIDS, ids=str)
def test_bad_grids_fail_with_the_dense_grid_messages(g):
    st, msg = call(params(), g)
    assert st == _lib.FDCM_ERR_INVALID
    want = dense_poses_hook(fdcm.DenseSearch(4), (0.0, 0.0), (0.0, 0.0), 10, 10, 0, capacity=0, g=g)[0]
    assert want == _lib.FDCM_ERR_INVALID
    assert msg == _lib.lib().fdcm_last_error().decode() and "scale" in msg


def test_null_arguments():
    g = fdcm.ScaleGrid(3, 0.9, 1.1)
    assert call(params(), None) == (_lib.FDCM_ERR_INVALID, "scales is null")
    assert call(None, g) == (_lib.FDCM_ERR_INVALID, "null argument")
    assert call(params(), g) == (_lib.FDCM_ERR_INVALID, "null argument")   # (no map, no templates)


@pytest.mark.parametrize("what", ["select", "refine", "cov"])
def test_select_refine_and_cov_need_top_k(what):
    arg = {"select": fdcm.DistinctMatches(max_per_template=1), "refine": fdcm.PoseRefinement(), "cov": fdcm.EdgeCoverage(min_coverage=0.5)}
    st, msg = call(params(top_k=0), fdcm.ScaleGrid(3, 0.9, 1.1), **{what: arg[what]})
    assert st == _lib.FDCM_ERR_INVALID and "top_k" in msg


@pytest.mark.parametrize("bad", [dict(select=fdcm.DistinctMatches(max_per_template=-1)), dict(refine=fdcm.PoseRefinement(levels=0)),
                                 dict(cov=fdcm.EdgeCoverage(radius=99)), dict(cov=fdcm.EdgeCoverage(min_coverage=2.0))], ids=str)
def test_bad_select_refine_and_cov_parameters(bad):
    st, _ = call(params(), fdcm.ScaleGrid(2, 0.9, 1.1), **bad)
    assert st == _lib.FDCM_ERR_INVALID


def test_python_entry_points_take_scales():
    import inspect
    for fn in (fdcm.search_topk, fdcm.search_all):
        assert inspect.signature(fn).parameters["scales"].default is None


def test_cpp_mirror_builds(tmp_path):
    """The C++ overloads taking a ScaleGrid compile against the header (not run: no device)."""
    src = tmp_path / "m.cpp"
    src.write_text('#include "openfdcm_b200/openfdcm_cuda.hpp"\n'
                   "using namespace openfdcm::cuda;\n"
                   "int main(int argc, char**) {\n"
                   "  if (argc < 5) return 0;\n"
                   "  Dt3Cuda fm = buildCudaFeaturemap(LineArray{}, Dt3CudaParameters{});\n"
                   "  std::vector<LineArray> t; LineArray s; ScaleGrid g{3, 0.9f, 1.1f}; DistinctMatches q{1};\n"
                   "  PoseRefinement r; EdgeCoverage c;\n"
                   "  auto a = search(DefaultMatch{}, DefaultSearch{4, 4}, BatchOptimize{10}, fm, t, s, g);\n"
                   "  auto b = searchTopK(DefaultSearch{4, 4}, BatchOptimize{10}, ExponentialPenalty{1.5f}, fm, t, s, 10, g, &q, &r, &c);\n"
                   "  return (int)(a.size() + b.size());\n"
                   "}\n")
    import subprocess
    r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-Wall", "-I" + os.path.join(ROOT, "include"), str(src)], capture_output=True,
                       text=True)
    assert r.returncode == 0, r.stderr
