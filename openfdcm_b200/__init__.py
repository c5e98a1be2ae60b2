"""openfdcm_b200 — B200-native drop-in for OpenFDCM's two hot paths.

Python surface mirrors the reference's pybind11 module `openfdcm`
(reference modules/python/src/matching.cpp:62-308, core.cpp:39-50): same class / function names
and argument meaning, with `Dt3CudaParameters` / `build_cuda_featuremap` / `Dt3Cuda` as the CUDA
feature map.  Line arrays are numpy (4, N) arrays (one column per line: x1,y1,x2,y2), any dtype,
converted to float32 exactly like pybind11's Eigen caster does for `core::LineArray`.

Everything computes through the C ABI of libfdcm_b200.so (include/fdcm_b200.h); there is no CPU
fallback.
"""
import ctypes as C
import enum
import math

import numpy as np

from . import _lib
from .io import read, write
from ._lib import MATCH_DTYPE, FdcmError, check, lib, ptr

__all__ = [
    "distance", "Dt3CudaParameters", "Dt3Cuda", "build_cuda_featuremap", "ThreadPool", "DefaultSearch", "ConcentricRangeStrategy",
    "BatchOptimize", "DefaultOptimize", "DefaultMatch", "DefaultPenalty", "ExponentialPenalty", "Match",
    "TemplateSet", "SceneBatch", "DistinctMatches", "PoseRefinement", "DenseSearch", "search", "search_topk", "search_dense",
    "refine_matches", "penalize", "get_template_lengths",
    "get_template_anchors", "sort_matches", "evaluate",
    "minmax_translation", "get_feature_size", "establish_search_strategy", "optimize", "read", "write", "FdcmError", "MATCH_DTYPE",
]


class distance(enum.IntEnum):
    """core::Distance (core/imgproc.h:148; python/src/core.cpp:45-49)."""
    L2 = 0
    L2_SQUARED = 1
    L1 = 2


def _records(lines):
    """(4,N) line array -> contiguous (N,4) float32 records."""
    a = np.asarray(lines, dtype=np.float32)
    if a.size == 0:
        return np.zeros((0, 4), np.float32)
    if a.ndim == 1 and a.size == 4:
        a = a.reshape(4, 1)
    if a.ndim != 2 or a.shape[0] != 4:
        raise ValueError(f"expected a (4,N) line array, got shape {a.shape}")
    return np.ascontiguousarray(a.T)


def _pack(templates):
    recs = [_records(t) for t in templates]
    off = np.zeros(len(recs) + 1, np.int32)
    for i, r in enumerate(recs):
        off[i + 1] = off[i] + r.shape[0]
    flat = np.concatenate(recs, axis=0) if recs else np.zeros((0, 4), np.float32)
    return np.ascontiguousarray(flat, np.float32), off


class Dt3CudaParameters:
    """Dt3CpuParameters (dt3cpu.h:34-42) + distance (python/src/matching.cpp:51-60), CUDA flavour."""

    def __init__(self, depth=30, dt3Coeff=5.0, padding=2.2, distance=distance.L2, device=0):
        self.depth = int(depth)
        self.dt3_coeff = float(dt3Coeff)
        self.padding = float(padding)
        self.distance = distance
        self.device = int(device)

    def __repr__(self):
        return f"<Dt3CudaParameters: depth={self.depth}, dt3_coeff={self.dt3_coeff}, padding={self.padding}>"


class Dt3Cuda:
    """Device-resident DT3 feature map: [depth][H][pitch] fp32 planes in HBM (mirrors Dt3Cpu, dt3cpu.h:46-63).
    Copies of the Python object share one ref-counted device handle (O(1), unlike FeatureMap's clone())."""

    def __init__(self, handle):
        self._h = C.c_void_p(handle)
        self._refresh()

    def _refresh(self):
        info = _lib.Dt3Info()
        check(lib().fdcm_dt3_get_info(self._h, C.byref(info)))
        self.info = info
        self.depth, self.width, self.height, self.pitch = info.depth, info.width, info.height, info.pitch
        self.device = info.device

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and lib is not None:   # (module globals are gone when the interpreter shuts down)
            lib().fdcm_dt3_release(h)

    def __copy__(self):
        check(lib().fdcm_dt3_retain(self._h))
        return Dt3Cuda(self._h.value)

    def get_scene_translation(self):
        return np.array(self.info.scene_translation[:], np.float32)

    def get_feature_size(self):
        return np.array([self.width, self.height], np.uint64)

    def angles(self):
        k = np.zeros(self.depth, np.float32)
        if self.depth:
            check(lib().fdcm_dt3_angles(self._h, ptr(k)))
        return k

    def plane(self, i):
        out = np.zeros((self.height, self.width), np.float32)
        check(lib().fdcm_dt3_download_plane(self._h, int(i), ptr(out)))
        return out

    def mask(self, i):
        out = np.zeros((self.height, self.width), np.uint8)
        check(lib().fdcm_dt3_download_mask(self._h, int(i), ptr(out)))
        return out

    def scene_bins(self):
        b = np.zeros(self.info.n_scene_lines, np.int32)
        if b.size:
            check(lib().fdcm_dt3_scene_bins(self._h, ptr(b)))
        return b

    def classify(self, lines):
        r = _records(lines)
        b = np.zeros(r.shape[0], np.int32)
        check(lib().fdcm_dt3_classify(self._h, ptr(r), r.shape[0], ptr(b)))
        return b

    def get_dt3_map(self):
        """{angle: H x W image} like Dt3Cpu::getDt3Map (downloads the whole map)."""
        return {float(a): self.plane(i) for i, a in enumerate(self.angles())}

    def device_ptr(self):
        p, n = C.c_void_p(0), C.c_uint64(0)
        check(lib().fdcm_dt3_device_ptr(self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def rebuild(self, scene, wait=True):
        r = _records(scene)
        check((lib().fdcm_dt3_rebuild if wait else lib().fdcm_dt3_rebuild_async)(self._h, ptr(r), r.shape[0]))
        self._refresh()

    def rerun(self, wait=True):
        check((lib().fdcm_dt3_rerun if wait else lib().fdcm_dt3_rerun_async)(self._h))

    def last_search_stats(self):
        st = _lib.SearchStats()
        check(lib().fdcm_search_last_stats(self._h, C.byref(st)))
        return {"n_hypotheses": st.n_hypotheses, "n_valid": st.n_valid, "n_evaluations": st.n_evaluations,
                "n_lookups": st.n_lookups}

    def last_hypotheses(self):
        n = C.c_int64(0)
        lib().fdcm_search_last_hypotheses(self._h, None, 0, C.byref(n))
        out = np.zeros((n.value, 4), np.int32)
        if n.value:
            check(lib().fdcm_search_last_hypotheses(self._h, ptr(out), n.value, C.byref(n)))
        return out

    def __repr__(self):
        t = self.info.scene_translation
        return f"<Dt3Cuda: scene translation=({t[0]}, {t[1]}), feature size=({self.width}, {self.height})>"


def build_cuda_featuremap(scene, params=None, pool=None, *, stage=0):
    """build_cpu_featuremap(scene, params, pool) (python/src/matching.cpp:116-130) on the GPU.
    `pool` is accepted for signature compatibility and ignored (the device is the pool)."""
    params = params or Dt3CudaParameters()
    p = _lib.Dt3Params(params.depth, params.dt3_coeff, params.padding, int(params.distance))
    r = _records(scene)
    h = C.c_void_p(0)
    check(lib().fdcm_dt3_build(ptr(r), r.shape[0], C.byref(p), params.device, int(stage), C.byref(h)))
    return Dt3Cuda(h.value)


class ThreadPool:
    """Placeholder for openfdcm.ThreadPool (python/src/matching.cpp:86-101): the CUDA strategies do not
    use host threads; kept so that reference call sites run unchanged."""

    def __init__(self, num_threads=0):
        self.num_threads = int(num_threads)

    def get_thread_count(self):
        return self.num_threads


class DefaultSearch:
    """searchstrategies/defaultsearch.h:53-66."""

    def __init__(self, max_tmpl_lines, max_scene_lines):
        self.max_tmpl_lines, self.max_scene_lines = int(max_tmpl_lines), int(max_scene_lines)

    def get_max_tmpl_lines(self):
        return self.max_tmpl_lines

    def get_max_scene_lines(self):
        return self.max_scene_lines


class ConcentricRangeStrategy(DefaultSearch):
    """searchstrategies/concentricrange.h:35-60: DefaultSearch on the scene lines whose centre lies in a radius band."""

    def __init__(self, max_tmpl_lines, max_scene_lines, center_position, low_boundary, high_boundary):
        super().__init__(max_tmpl_lines, max_scene_lines)
        c = np.asarray(center_position, np.float32).reshape(2)
        self.center_position = c
        self.low_boundary, self.high_boundary = float(low_boundary), float(high_boundary)

    def get_center_position(self):
        return self.center_position

    def get_low_radius_boundary(self):
        return self.low_boundary

    def get_high_radius_boundary(self):
        return self.high_boundary


class BatchOptimize:
    """optimizestrategies/batchoptimize.h:8-23 (pool / num_threads accepted and ignored)."""

    def __init__(self, batch_size, pool=None, num_threads=None):
        if int(batch_size) < 1:
            raise ValueError("batch_size must be >= 1")
        self.batch_size = int(batch_size)

    def get_batch_size(self):
        return self.batch_size


class DefaultOptimize:
    """optimizestrategies/defaultoptimize.h: step-1 line search == batches of one."""
    batch_size = 0

    def __init__(self, pool=None, num_threads=None):
        pass


class DefaultMatch:
    """matchstrategies/defaultmatch.h."""


class DefaultPenalty:
    kind, tau = 1, 0.0


class ExponentialPenalty:
    kind = 2

    def __init__(self, tau):
        self.tau = float(tau)

    def get_tau(self):
        return self.tau


class Match:
    """matching::Match (matchstrategy.h:35-44; python/src/matching.cpp:266-277)."""
    __slots__ = ("tmpl_idx", "score", "transform")

    def __init__(self, tmpl_idx, score, transform):
        self.tmpl_idx = int(tmpl_idx)
        self.score = float(score)
        self.transform = np.asarray(transform, np.float32).reshape(2, 3)

    def __repr__(self):
        return f"<Match tmplIdx={self.tmpl_idx}, score={self.score}, transform=\n{self.transform}>"


def _to_matches(rec):
    return [Match(r["tmpl_idx"], r["score"], r["transform"]) for r in rec]


def _to_records(matches):
    if isinstance(matches, np.ndarray) and matches.dtype == MATCH_DTYPE:
        return np.ascontiguousarray(matches).copy()
    rec = np.zeros(len(matches), MATCH_DTYPE)
    for i, m in enumerate(matches):
        rec[i] = (m.tmpl_idx, m.score, np.asarray(m.transform, np.float32).reshape(6))
    return rec


class TemplateSet:
    """Device-resident template set (upload once, search many scenes)."""

    def __init__(self, templates, device=0):
        flat, off = _pack(templates)
        self.n_tmpl = len(off) - 1
        self.n_lines = int(off[-1])
        self.max_lines = int(np.diff(off).max()) if self.n_tmpl else 0
        h = C.c_void_p(0)
        check(lib().fdcm_templates_create(ptr(flat), ptr(off), self.n_tmpl, int(device), C.byref(h)))
        self._h = h
        self.device = int(device)

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and lib is not None:   # (module globals are gone when the interpreter shuts down)
            lib().fdcm_templates_release(h)

    def lengths(self):
        out = np.zeros(self.n_tmpl, np.float32)
        if self.n_tmpl:
            check(lib().fdcm_templates_lengths(self._h, ptr(out)))
        return out


class DistinctMatches:
    """Distinct top-K (beyond the reference): from the matches in ascending (score, hypothesis) order, keep a match only
    while fewer than `top_k` are kept, fewer than `max_per_template` of its template are kept (0: no cap) and, with
    `radius` > 0, no kept match lies near it: template anchors (bounding-box centres) mapped by the two transforms within
    `radius` pixels and rotations within `max_angle` radians (>= pi: any rotation), counting kept matches of its own
    template only unless `across_templates` (at most top-k 1024 then).  Exact rules: include/fdcm_b200.h."""

    def __init__(self, max_per_template=0, radius=0.0, max_angle=math.pi, across_templates=False):
        self.max_per_template = int(max_per_template)
        self.radius = float(radius)
        self.max_angle = float(max_angle)
        self.across_templates = bool(across_templates)

    def _params(self):
        return _lib.SelectParams(self.max_per_template, self.radius, self.max_angle, 1 if self.across_templates else 0)

    def __repr__(self):
        return (f"<DistinctMatches: max_per_template={self.max_per_template}, radius={self.radius}, max_angle={self.max_angle}, "
                f"across_templates={self.across_templates}>")


class PoseRefinement:
    """Pose refinement (beyond the reference): around each match, `levels` coarse-to-fine grids of rotations
    i * rot_step / 2^l about the template anchor (|i| <= rot_steps) and translations (j, k) * trans_step / 2^l
    (|j|, |k| <= trans_steps); every level keeps the pose with the lowest evaluate<Dt3Cpu> score over all template lines,
    the centre on ties.  It minimises that score only: at sub-pixel and 0.01 rad scales the score is not lowest at the
    true pose, and refinement was measured to increase the error against known poses.  Exact rules: include/fdcm_b200.h."""

    def __init__(self, levels=3, rot_steps=4, rot_step=0.01, trans_steps=4, trans_step=1.0):
        self.levels = int(levels)
        self.rot_steps = int(rot_steps)
        self.rot_step = float(rot_step)
        self.trans_steps = int(trans_steps)
        self.trans_step = float(trans_step)

    def _params(self):
        return _lib.RefineParams(self.levels, self.rot_steps, self.rot_step, self.trans_steps, self.trans_step)

    def __repr__(self):
        return (f"<PoseRefinement: levels={self.levels}, rot_steps={self.rot_steps}, rot_step={self.rot_step}, "
                f"trans_steps={self.trans_steps}, trans_step={self.trans_step}>")


class DenseSearch:
    """Dense pose-grid search (beyond the reference): every template at `rotations` rotations rot_start + r * rot_step
    about its anchor (rot_step None: 2 pi / rotations) and at every `stride`-th map pixel of the map, or of the region
    roi = (x0, y0, x1, y1) in scene coordinates; each cell of cell x cell grid points keeps its best pose.  The grid is
    finite (pose error up to stride / 2 px and rot_step / 2 rad before refinement) and minimises the evaluate<Dt3Cpu>
    score, which is not lowest at the true pose at sub-pixel scales.  Exact rules: include/fdcm_b200.h."""

    def __init__(self, rotations=72, rot_start=0.0, rot_step=None, stride=2, cell=8, roi=None):
        self.rotations = int(rotations)
        self.rot_start = float(rot_start)
        if rot_step is None:   # one full turn (rotations < 1 is rejected by the search)
            rot_step = 2.0 * math.pi / self.rotations if self.rotations > 0 else 0.0
        self.rot_step = float(rot_step)
        self.stride = int(stride)
        self.cell = int(cell)
        self.roi = None if roi is None else tuple(float(v) for v in roi)
        if self.roi is not None and len(self.roi) != 4:
            raise ValueError("roi must be (x0, y0, x1, y1)")

    def _params(self):
        roi = self.roi or (0.0, 0.0, 0.0, 0.0)
        return _lib.DenseParams(self.rotations, self.rot_start, self.rot_step, self.stride, self.cell, 0 if self.roi is None else 1,
                                (C.c_float * 4)(*roi))

    def __repr__(self):
        return (f"<DenseSearch: rotations={self.rotations}, rot_start={self.rot_start}, rot_step={self.rot_step}, stride={self.stride}, "
                f"cell={self.cell}, roi={self.roi}>")


def _search_raw(featuremap, templates, scene, searcher, optimizer, penalty=None, top_k=0, tmpl_idx_base=0, select=None, refine=None):
    if not isinstance(featuremap, Dt3Cuda):
        raise TypeError("the CUDA search needs a Dt3Cuda feature map (build_cuda_featuremap)")
    tset = templates if isinstance(templates, TemplateSet) else TemplateSet(templates, featuremap.device)
    s = None if scene is None else _records(scene)   # None: the scene the map was built from, already resident
    conc = isinstance(searcher, ConcentricRangeStrategy)
    p = _lib.SearchParams(searcher.max_tmpl_lines, searcher.max_scene_lines, int(optimizer.batch_size),
                          0 if penalty is None else penalty.kind, 0.0 if penalty is None else float(penalty.tau),
                          int(top_k), int(tmpl_idx_base), 1 if conc else 0,
                          float(searcher.center_position[0]) if conc else 0.0, float(searcher.center_position[1]) if conc else 0.0,
                          searcher.low_boundary if conc else 0.0, searcher.high_boundary if conc else 0.0)
    if tset.n_tmpl == 0:
        return np.zeros(0, MATCH_DTYPE)
    cap = int(top_k) if top_k > 0 or select is not None else 2 * tset.n_tmpl * max(1, min(searcher.max_tmpl_lines, tset.max_lines)) * max(
        1, searcher.max_scene_lines)
    out = np.zeros(max(cap, 1), MATCH_DTYPE)
    n = C.c_int64(0)
    n_scene = _lib.FDCM_SCENE_RESIDENT if s is None else s.shape[0]
    if refine is not None:
        sp = None if select is None else C.byref(select._params())
        check(lib().fdcm_search_refine(featuremap._h, tset._h, ptr(s), n_scene, C.byref(p), sp, C.byref(refine._params()), ptr(out),
                                       out.shape[0], C.byref(n)))
    elif select is None:
        check(lib().fdcm_search(featuremap._h, tset._h, ptr(s), n_scene, C.byref(p), ptr(out), out.shape[0], C.byref(n)))
    else:
        sp = select._params()
        check(lib().fdcm_search_select(featuremap._h, tset._h, ptr(s), n_scene, C.byref(p), C.byref(sp), ptr(out), out.shape[0],
                                       C.byref(n)))
    return out[: n.value]


def search(matcher, searcher, optimizer, featuremap, templates, scene):
    """openfdcm.search (python/src/matching.cpp:279-289): every match in hypothesis order."""
    return _to_matches(_search_raw(featuremap, templates, scene, searcher, optimizer))


def search_topk(featuremap, templates, scene, searcher, optimizer, penalty=None, k=10, tmpl_idx_base=0, *, select=None, refine=None):
    """Fused search -> penalize -> top-k on the device; returns a MATCH_DTYPE record array (ascending score).
    select: a DistinctMatches for the distinct top-k (the kept matches in acceptance order, also ascending score).
    refine: a PoseRefinement applied to the selected matches on the device, equal to refine_matches of the unrefined
    result (same order: re-rank with sort_matches); it lowers the score, not the pose error (see PoseRefinement)."""
    return _search_raw(featuremap, templates, scene, searcher, optimizer, penalty, k, tmpl_idx_base, select, refine).copy()


def refine_matches(featuremap, templates, matches, refine, penalty=None, tmpl_idx_base=0):
    """Pose refinement of any match list against a feature map and a template set (list or TemplateSet); returns a
    MATCH_DTYPE array, entry i refining matches[i], scored like search_topk with the same penalty.  Each pose moves to the
    lowest evaluate<Dt3Cpu> score of its grid, which is not a more accurate pose (see PoseRefinement)."""
    if not isinstance(featuremap, Dt3Cuda):
        raise TypeError("refine_matches needs a Dt3Cuda feature map (build_cuda_featuremap)")
    tset = templates if isinstance(templates, TemplateSet) else TemplateSet(templates, featuremap.device)
    rec = _to_records(matches)
    out = np.zeros(max(rec.shape[0], 1), MATCH_DTYPE)
    st = lib().fdcm_refine_matches(featuremap._h, tset._h, int(tmpl_idx_base), 0 if penalty is None else penalty.kind,
                                   0.0 if penalty is None else float(penalty.tau), C.byref(refine._params()), ptr(rec), rec.shape[0],
                                   ptr(out))
    if st == _lib.FDCM_ERR_OUT_OF_RANGE:
        raise IndexError(lib().fdcm_last_error().decode())
    check(st)
    return out[: rec.shape[0]].copy()


def search_dense(featuremap, templates, dense, penalty=None, k=10, tmpl_idx_base=0, *, select=None, refine=None):
    """Dense pose-grid search on the device (see DenseSearch): the best pose of every (template, rotation, cell), then the
    top-k in ascending (score, record) order, or with select (a DistinctMatches) the distinct top-k, then with refine (a
    PoseRefinement) the refinement of those, equal to refine_matches of the unrefined result.  Returns a MATCH_DTYPE array."""
    if not isinstance(featuremap, Dt3Cuda):
        raise TypeError("search_dense needs a Dt3Cuda feature map (build_cuda_featuremap)")
    tset = templates if isinstance(templates, TemplateSet) else TemplateSet(templates, featuremap.device)
    out = np.zeros(max(int(k), 1), MATCH_DTYPE)
    n = C.c_int64(0)
    sp = None if select is None else C.byref(select._params())
    rp = None if refine is None else C.byref(refine._params())
    check(lib().fdcm_search_dense(featuremap._h, tset._h, C.byref(dense._params()), 0 if penalty is None else penalty.kind,
                                  0.0 if penalty is None else float(penalty.tau), int(k), int(tmpl_idx_base), sp, rp, ptr(out), out.shape[0],
                                  C.byref(n)))
    return out[: n.value].copy()


def search_all(featuremap, templates, scene, searcher, optimizer, penalty=None, tmpl_idx_base=0):
    """Every match (hypothesis order) as a MATCH_DTYPE record array, optionally penalised on the device."""
    return _search_raw(featuremap, templates, scene, searcher, optimizer, penalty, 0, tmpl_idx_base).copy()


class SceneBatch:
    """Multi-scene batches (BASELINE config 5): per scene a DT3 build + fused search / penalty / top-k against one
    resident TemplateSet, with the build of the next scene running under the search of the current one
    (fdcm_search_scenes)."""

    def __init__(self, params=None):
        params = params or Dt3CudaParameters()
        p = _lib.Dt3Params(params.depth, params.dt3_coeff, params.padding, int(params.distance))
        h = C.c_void_p(0)
        check(lib().fdcm_scene_batch_create(C.byref(p), params.device, C.byref(h)))
        self._h, self.device = h, params.device

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h and lib is not None:   # (module globals are gone when the interpreter shuts down)
            lib().fdcm_scene_batch_destroy(h)

    def search_topk(self, scenes, templates, searcher, optimizer, penalty=None, k=10, tmpl_idx_base=0, *, select=None):
        """-> list (one per scene) of MATCH_DTYPE arrays (ascending score); select: a DistinctMatches, like search_topk."""
        tset = templates if isinstance(templates, TemplateSet) else TemplateSet(templates, self.device)
        flat, off = _pack(scenes)
        p = _lib.SearchParams(searcher.max_tmpl_lines, searcher.max_scene_lines, int(optimizer.batch_size),
                              0 if penalty is None else penalty.kind, 0.0 if penalty is None else float(penalty.tau),
                              int(k), int(tmpl_idx_base), 0, 0.0, 0.0, 0.0, 0.0)
        n = len(off) - 1
        out = np.zeros((max(n, 1), int(k)), MATCH_DTYPE)
        cnt = np.zeros(max(n, 1), np.int32)
        if select is None:
            check(lib().fdcm_search_scenes(self._h, ptr(flat), ptr(off), n, tset._h, C.byref(p), ptr(out), ptr(cnt)))
        else:
            sp = select._params()
            check(lib().fdcm_search_scenes_select(self._h, ptr(flat), ptr(off), n, tset._h, C.byref(p), C.byref(sp), ptr(out), ptr(cnt)))
        return [out[i, : cnt[i]].copy() for i in range(n)]


def penalize(penalty, matches, templatelengths):
    """openfdcm.penalize (python/src/matching.cpp:291-297)."""
    rec = _to_records(matches)
    lengths = np.ascontiguousarray(templatelengths, np.float32)
    st = lib().fdcm_penalize(penalty.kind, float(penalty.tau), ptr(rec), rec.shape[0], ptr(lengths), lengths.shape[0])
    if st == _lib.FDCM_ERR_OUT_OF_RANGE:
        raise IndexError(lib().fdcm_last_error().decode())
    check(st)
    return rec if isinstance(matches, np.ndarray) else _to_matches(rec)


def get_template_lengths(templates):
    """openfdcm.get_template_lengths (core/math.h:319-324)."""
    flat, off = _pack(templates)
    out = np.zeros(len(off) - 1, np.float32)
    check(lib().fdcm_template_lengths(ptr(flat), ptr(off), len(off) - 1, ptr(out)))
    return out.tolist()


def get_template_anchors(templates):
    """Anchor of every template for DistinctMatches: the centre of the bounding box of its line end points, (0, 0) when
    empty; an (n_tmpl, 2) float32 array."""
    flat, off = _pack(templates)
    out = np.zeros((len(off) - 1, 2), np.float32)
    check(lib().fdcm_template_anchors(ptr(flat), ptr(off), len(off) - 1, ptr(out)))
    return out


def sort_matches(matches):
    """openfdcm.sort_matches (python/src/matching.cpp:302-307)."""
    rec = _to_records(matches)
    check(lib().fdcm_sort_matches(ptr(rec), rec.shape[0]))
    return rec if isinstance(matches, np.ndarray) else _to_matches(rec)


def get_feature_size(featuremap):
    """matching::getFeatureSize (featuremap.h:27-28)."""
    return featuremap.get_feature_size()


def minmax_translation(featuremap, tmpl, align_vec):
    """matching::minmaxTranslation (featuremap.h:38-40; dt3cpu.cpp:119-124)."""
    r = _records(tmpl)
    v = np.ascontiguousarray(align_vec, np.float32)
    out = np.zeros(2, np.float32)
    check(lib().fdcm_dt3_minmax_translation(featuremap._h, ptr(r), r.shape[0], ptr(v), ptr(out)))
    return out


def evaluate(featuremap, templates, translations):
    """matching::evaluate (featuremap.h:50-52; dt3cpu.cpp:126-179): list of per-template score lists."""
    flat, off = _pack(templates)
    tr = [np.ascontiguousarray(np.asarray(t, np.float32).reshape(-1, 2)) for t in translations]
    troff = np.zeros(len(tr) + 1, np.int32)
    for i, t in enumerate(tr):
        troff[i + 1] = troff[i] + t.shape[0]
    tflat = np.concatenate(tr, axis=0) if tr else np.zeros((0, 2), np.float32)
    tflat = np.ascontiguousarray(tflat, np.float32)
    scores = np.zeros(int(troff[-1]), np.float32)
    check(lib().fdcm_dt3_evaluate(featuremap._h, ptr(flat), ptr(off), len(off) - 1, ptr(tflat), ptr(troff), ptr(scores)))
    return [scores[troff[i]:troff[i + 1]].copy() for i in range(len(tr))]


def optimize(optimizer, templates, alignments, featuremap):
    """matching::optimize (optimizestrategy.h:62-64): list of None | (score, translation[2]) per template."""
    flat, off = _pack(templates)
    al = np.ascontiguousarray(np.asarray(alignments, np.float32).reshape(-1, 2))
    n = len(off) - 1
    if al.shape[0] != n:
        raise ValueError("templates and alignments must have the same length")
    has = np.zeros(n, np.uint8)
    sc = np.zeros(n, np.float32)
    tr = np.zeros((n, 2), np.float32)
    check(lib().fdcm_optimize(featuremap._h, ptr(flat), ptr(off), n, ptr(al), int(optimizer.batch_size), ptr(has), ptr(sc), ptr(tr)))
    return [(float(sc[i]), tr[i].copy()) if has[i] else None for i in range(n)]


def establish_search_strategy(searcher, tmpl, scene):
    """matching::establishSearchStrategy<DefaultSearch> (defaultsearch.cpp:29-49): (tmpl_line, scene_line) pairs."""
    t, s = _records(tmpl), _records(scene)
    cap = max(1, searcher.max_tmpl_lines * searcher.max_scene_lines)
    out = np.zeros((cap, 2), np.int32)
    n = C.c_int32(0)
    if isinstance(searcher, ConcentricRangeStrategy):
        check(lib().fdcm_concentric_search(ptr(t), t.shape[0], ptr(s), s.shape[0], searcher.max_tmpl_lines, searcher.max_scene_lines,
                                           float(searcher.center_position[0]), float(searcher.center_position[1]),
                                           searcher.low_boundary, searcher.high_boundary, ptr(out), cap, C.byref(n)))
    else:
        check(lib().fdcm_default_search(ptr(t), t.shape[0], ptr(s), s.shape[0], searcher.max_tmpl_lines,
                                        searcher.max_scene_lines, ptr(out), cap, C.byref(n)))
    return out[: n.value].copy()


def set_stream(device, cuda_stream):
    check(lib().fdcm_set_stream(int(device), C.c_void_p(cuda_stream) if cuda_stream else None))


def profile(enable=True, reset=False):
    if reset:
        check(lib().fdcm_profile_reset())
    check(lib().fdcm_profile_enable(1 if enable else 0))


def profile_report():
    n = C.c_int32(0)
    check(lib().fdcm_profile_count(C.byref(n)))
    out = {}
    for i in range(n.value):
        name = C.create_string_buffer(64)
        ms, cnt, by = C.c_double(0), C.c_int64(0), C.c_double(0)
        check(lib().fdcm_profile_get(i, name, 64, C.byref(ms), C.byref(cnt), C.byref(by)))
        out[name.value.decode()] = {"total_ms": ms.value, "launches": cnt.value, "bytes_per_launch": by.value}
    return out


def kernel_launch_count():
    return int(lib().fdcm_kernel_launch_count())
