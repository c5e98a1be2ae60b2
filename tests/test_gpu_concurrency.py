"""The library under concurrent use: caller streams, queued builds, host threads and profiling.

Every result is compared byte for byte, either with the same call made single-threaded on the library's own stream (itself
oracle-tested elsewhere) or with the oracle.  To make the orderings deterministic, a bounded spin kernel (torch.cuda._sleep,
calibrated once per module to SPIN_MS) is queued on the caller's stream first, so the library's work queues behind it.
Each case asserts that the spin was still running when the racing call was issued: a case whose window closed fails
instead of passing without having tested anything."""
import ctypes as C
import threading

import numpy as np
import pytest

import openfdcm_b200 as fdcm
from openfdcm_b200 import _lib
from oracle import fdcm_oracle as orc
from tests.util import F32, plant_instances, synth_scene, synth_templates

pytestmark = pytest.mark.gpu

DEV = 0
SPIN_MS = 250.0           # one spin; the calibration rejects anything that would measure 500 ms or more
JOIN_S = 120.0
P = fdcm.Dt3CudaParameters(30, 5.0, 1.5)
SEARCH, OPT, PEN = fdcm.DefaultSearch(4, 4), fdcm.BatchOptimize(10), fdcm.ExponentialPenalty(1.5)
SELECT = fdcm.DistinctMatches(max_per_template=2, radius=5.0)
REFINE = fdcm.PoseRefinement(levels=2, rot_steps=2, rot_step=0.01, trans_steps=2, trans_step=1.0)
DENSE = fdcm.DenseSearch(rotations=8, stride=4, cell=16)
PENALTIES = (None, fdcm.DefaultPenalty(), fdcm.ExponentialPenalty(1.5), fdcm.ExponentialPenalty(3.0))


# ---- helpers ---------------------------------------------------------------------------------
def canon(x):
    """Hashable byte image of a result (arrays by dtype, shape and bytes; floats by their bits)."""
    if isinstance(x, np.ndarray):
        return (x.dtype.str, x.shape, x.tobytes())
    if isinstance(x, (list, tuple)):
        return tuple(canon(v) for v in x)
    if isinstance(x, float):
        return np.float64(x).tobytes()
    return x


def same(a, b):
    return canon(a) == canon(b)


def planes(fm):
    return np.stack([fm.plane(d) for d in range(fm.depth)])


def masks(fm):
    return np.stack([fm.mask(d) for d in range(fm.depth)])


def top10(fm, tset, penalty=PEN, **kw):
    return fdcm.search_topk(fm, tset, None, SEARCH, OPT, penalty, k=10, **kw)


def oracle_top10(scene, tmpls):
    c = orc.Dt3Cpu(scene, 30, 5.0, 1.5)
    pen = orc.penalize(1, 1.5, c.search(tmpls, scene, 4, 4, batch=10), orc.template_lengths(tmpls))
    return pen[np.lexsort((np.arange(len(pen)), pen["score"]))[:10]]


def build(scene, params=P):
    return fdcm.build_cuda_featuremap(scene, params)


def join_all(threads):
    for t in threads:
        t.join(JOIN_S)
    alive = [t.name for t in threads if t.is_alive()]
    assert not alive, f"threads still running after {JOIN_S} s: {alive}"


def run_threads(fns):
    """Run every fn on its own thread, started together; -> (results, errors) in fn order."""
    res, err = [None] * len(fns), [None] * len(fns)
    go = threading.Barrier(len(fns))

    def body(i):
        try:
            go.wait(JOIN_S)
            res[i] = fns[i]()
        except BaseException as e:   # noqa: BLE001 (reported by the caller)
            err[i] = e

    threads = [threading.Thread(target=body, args=(i,), name=f"fdcm-test-{i}", daemon=True) for i in range(len(fns))]
    for t in threads:
        t.start()
    join_all(threads)
    return res, err


def raise_first(err):
    for e in err:
        if e is not None:
            raise e


class Spin:
    """A bounded spin kernel on a stream, and the check that it is still running."""

    def __init__(self, torch, cycles):
        self.torch, self.cycles = torch, cycles

    def hold(self, stream):
        with self.torch.cuda.stream(stream):
            self.torch.cuda._sleep(self.cycles)
        ev = self.torch.cuda.Event()
        ev.record(stream)
        return ev

    @staticmethod
    def held(ev, what):
        assert not ev.query(), (f"{what}: the spin on the caller's stream had already finished when the call was issued, so the "
                                "ordering was not exercised (the window closed; the host was slower than the spin)")


@pytest.fixture(scope="module")
def torch():
    import torch as t
    t.cuda.init()
    return t


@pytest.fixture(scope="module")
def spin(torch):
    s = torch.cuda.Stream(device=DEV)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    probe = 20_000_000
    with torch.cuda.stream(s):
        torch.cuda._sleep(1000)
        e0.record(s)
        torch.cuda._sleep(probe)
        e1.record(s)
    e1.synchronize()
    cycles = int(probe * SPIN_MS / max(e0.elapsed_time(e1), 1e-3))
    sp = Spin(torch, cycles)
    e0.record(s)
    sp.hold(s)
    e1.record(s)
    e1.synchronize()
    ms = e0.elapsed_time(e1)
    assert 0.4 * SPIN_MS < ms < 500.0, f"spin calibration: {cycles} cycles took {ms:.1f} ms"
    return sp


@pytest.fixture
def streams(torch):
    """New caller streams; the library is back on its own stream and the device idle afterwards."""
    made = []

    def new():
        made.append(torch.cuda.Stream(device=DEV))
        return made[-1]

    yield new
    fdcm.set_stream(DEV, None)
    torch.cuda.synchronize()


class Workload:
    """Three scenes of one line count and one map size, and a template set."""

    def __init__(self, w=320, h=240, n_scene=80, n_tmpl=12, n_lines=20, seed=71):
        self.tmpls = synth_templates(n_tmpl, n_lines, w, seed=seed)
        self.scenes = [plant_instances(synth_scene(w, h, n_scene, seed=seed + 10 * i + 1), self.tmpls, w, h, seed=seed + 10 * i + 2)
                       for i in range(3)]
        assert len({s.shape for s in self.scenes}) == 1
        self.X, self.Y, self.Z = self.scenes
        self.tset = fdcm.TemplateSet(self.tmpls, DEV)
        rng = np.random.default_rng(seed)
        self.placed = [(t.T.reshape(-1, 2) + np.array([w / 2, h / 2], F32)).reshape(-1, 4).T.astype(F32) for t in self.tmpls[:4]]
        self.trans = [rng.uniform(-20, 20, (9, 2)).astype(F32) for _ in self.placed]
        self.align = [np.array(v, F32) for v in ([1, 0], [0, 1], [0.6, 0.8], [-0.8, 0.6])]


@pytest.fixture(scope="module")
def wl(torch):
    w = Workload()
    fdcm.set_stream(DEV, None)
    sizes = {tuple(build(s).get_feature_size().tolist()) for s in w.scenes}
    assert len(sizes) == 1, sizes
    return w


# ---- A. every call on a held caller stream equals the call on the library's stream -----------------------------------
def _a_cases(w):
    """name -> (setup, act): setup() runs before the spin; act(state) races it and returns what is compared."""
    rm = lambda fm: top10(fm, w.tset)   # noqa: E731

    def rebuild(wait):
        def act(fm):
            fm.rebuild(w.X, wait=wait)
            return planes(fm), rm(fm)
        return (lambda: build(w.Z)), act

    def reruns(fm):
        for _ in range(3):
            fm.rerun(wait=False)
        return rm(fm)

    def search_host():
        import torch
        flat, off = fdcm._pack(w.tmpls)
        pin = lambda a: torch.from_numpy(a).pin_memory()   # noqa: E731
        return build(w.Z), pin(flat), pin(off), pin(fdcm._records(w.X))

    def search_host_act(st):
        fm, h_lines, h_off, h_scene = st
        L = fdcm.lib()
        fdcm.check(L.fdcm_dt3_rebuild_async(fm._h, h_scene.data_ptr(), h_scene.shape[0]))
        out, n = np.zeros(10, fdcm.MATCH_DTYPE), C.c_int64(0)
        p = _lib.SearchParams(4, 4, 10, PEN.kind, PEN.tau, 10, 0, 0, 0.0, 0.0, 0.0, 0.0)
        fdcm.check(L.fdcm_search_host(fm._h, h_lines.data_ptr(), h_off.data_ptr(), len(w.tmpls), None, _lib.FDCM_SCENE_RESIDENT,
                                      C.byref(p), fdcm.ptr(out), 10, C.byref(n)))
        return out[: n.value], rm(fm)

    def after_async_rebuild(fm):
        fm.rebuild(w.Y, wait=False)
        return planes(fm), masks(fm), fm.scene_bins()

    fmX = lambda: build(w.X)   # noqa: E731
    return {
        "build_cuda_featuremap": (lambda: None, lambda _: (lambda fm: (planes(fm), fm.scene_bins(), rm(fm)))(build(w.X))),
        "rebuild_wait": rebuild(True),
        "rebuild_async": rebuild(False),
        "rerun_async_x3_then_search": (fmX, reruns),
        "search_all": (fmX, lambda fm: fdcm.search_all(fm, w.tset, None, SEARCH, OPT, PEN)),
        "search_topk": (fmX, rm),
        "search_topk_select": (fmX, lambda fm: top10(fm, w.tset, select=SELECT)),
        "search_topk_refine": (fmX, lambda fm: top10(fm, w.tset, refine=REFINE)),
        "search_dense": (fmX, lambda fm: fdcm.search_dense(fm, w.tset, DENSE, PEN, k=10, select=SELECT, refine=REFINE)),
        "refine_matches": (lambda: (build(w.X), top10(build(w.X), w.tset)),
                           lambda st: fdcm.refine_matches(st[0], w.tset, st[1], REFINE, PEN)),
        "evaluate": (fmX, lambda fm: fdcm.evaluate(fm, w.placed, w.trans)),
        "minmax_translation": (fmX, lambda fm: [fdcm.minmax_translation(fm, t, v) for t, v in zip(w.placed, w.align)]),
        "classify": (fmX, lambda fm: fm.classify(w.Y)),
        "optimize": (fmX, lambda fm: fdcm.optimize(OPT, w.placed, w.align, fm)),
        "search_host_pinned": (search_host, search_host_act),
        "scene_batch": (lambda: fdcm.SceneBatch(P), lambda b: b.search_topk(w.scenes, w.tset, SEARCH, OPT, PEN, k=10)),
        "scene_batch_select": (lambda: fdcm.SceneBatch(P),
                               lambda b: b.search_topk(w.scenes, w.tset, SEARCH, OPT, PEN, k=10, select=SELECT)),
        "plane_mask_bins_after_async_rebuild": (fmX, after_async_rebuild),
    }


A_NAMES = list(_a_cases(None).keys())


@pytest.mark.parametrize("name", A_NAMES)
def test_caller_stream(name, wl, spin, streams, torch):
    setup, act = _a_cases(wl)[name]
    fdcm.set_stream(DEV, None)
    want = act(setup())
    S = streams()
    fdcm.set_stream(DEV, S.cuda_stream)
    state = setup()
    ev = spin.hold(S)
    spin.held(ev, name)
    got = act(state)
    torch.cuda.synchronize()
    fdcm.set_stream(DEV, None)
    assert same(got, want), f"{name}: the result on a held caller stream differs from the library stream's"


class _DevicePlanes:
    """A torch view of a map's planes through fdcm_dt3_device_ptr ([depth][height][pitch] fp32)."""

    def __init__(self, fm):
        p, n = fm.device_ptr()
        assert n == fm.depth * fm.height * fm.pitch * 4
        self.__cuda_array_interface__ = {"shape": (fm.depth, fm.height, fm.pitch), "typestr": "<f4", "data": (p, False),
                                         "strides": None, "version": 2}


def test_device_ptr_view_on_caller_stream(wl, spin, streams, torch):
    """A zero-copy reader on the stream the asynchronous rebuild and rerun were queued on sees the new map."""
    want = planes(build(wl.Y))
    fm = build(wl.X)
    S = streams()
    fdcm.set_stream(DEV, S.cuda_stream)
    ev = spin.hold(S)
    spin.held(ev, "rebuild(Y, wait=False)")
    fm.rebuild(wl.Y, wait=False)
    fm.rerun(wait=False)
    view = torch.as_tensor(_DevicePlanes(fm), device=f"cuda:{DEV}")
    with torch.cuda.stream(S):
        got = view[:, :, : fm.width].clone()
    spin.held(ev, "the read of the view")
    torch.cuda.synchronize()
    assert np.array_equal(got.cpu().numpy(), want)
    assert np.array_equal(planes(fm), want)


# ---- B. a stream switch after a queued build ---------------------------------------------------------------------------
B1_READERS = {
    "search_topk": lambda fm, w: top10(fm, w.tset),
    "search_dense": lambda fm, w: fdcm.search_dense(fm, w.tset, DENSE, PEN, k=10),
    "plane": lambda fm, w: planes(fm),
}


@pytest.mark.parametrize("target", ["other_stream", "library_stream"])
@pytest.mark.parametrize("reader", list(B1_READERS))
def test_stream_switch_after_async_rebuild(reader, target, wl, spin, streams):
    """rebuild(Y, wait=False) queued behind a spin on S1, then a call on S2 (or the library's stream) must see Y's map.
    X and Y have one line count and one map size, so a call that does not wait reads X's planes with Y's metadata."""
    read = B1_READERS[reader]
    fdcm.set_stream(DEV, None)
    want, want_x = read(build(wl.Y), wl), read(build(wl.X), wl)
    assert not same(want, want_x)
    fm = build(wl.X)
    S1, S2 = streams(), streams()
    fdcm.set_stream(DEV, S1.cuda_stream)
    ev = spin.hold(S1)
    spin.held(ev, "rebuild(Y, wait=False)")
    fm.rebuild(wl.Y, wait=False)
    fdcm.set_stream(DEV, S2.cuda_stream if target == "other_stream" else None)
    spin.held(ev, f"{reader} after the switch")
    got = read(fm, wl)
    fdcm.set_stream(DEV, None)
    assert not same(got, want_x), f"{reader} on the {target} read X's map: it was not ordered after the queued rebuild to Y"
    assert same(got, want), f"{reader} on the {target} after a queued rebuild to Y"


def test_two_writers_on_two_streams(wl, spin, streams, torch):
    """rebuild(Y, wait=False) queued behind a spin on S1, then rebuild(Z) on S2: the second build waits for the first,
    and the map ends as Z's.  (L1: the build runs on one stream; tiny maps of one size.)"""
    w, h = 64, 48
    tm = synth_templates(2, 6, w, seed=91)
    sc = [plant_instances(synth_scene(w, h, 12, seed=92 + i, min_len=3.0), tm, w, h, seed=95 + i, count=2) for i in range(3)]
    assert len({s.shape for s in sc}) == 1
    p1 = fdcm.Dt3CudaParameters(8, 5.0, 1.5, fdcm.distance.L1)
    fdcm.set_stream(DEV, None)
    ref = [build(s, p1) for s in sc]
    assert len({tuple(r.get_feature_size().tolist()) for r in ref}) == 1
    want = (planes(ref[2]), ref[2].scene_bins())
    c = orc.Dt3Cpu(sc[2], 8, 5.0, 1.5, orc.L1)
    assert np.array_equal(want[0], c.planes())
    fm = build(sc[0], p1)
    S1, S2 = streams(), streams()
    fdcm.set_stream(DEV, S1.cuda_stream)
    ev = spin.hold(S1)
    spin.held(ev, "rebuild(Y, wait=False)")
    fm.rebuild(sc[1], wait=False)
    fdcm.set_stream(DEV, S2.cuda_stream)
    spin.held(ev, "rebuild(Z) on the second stream")
    fm.rebuild(sc[2])
    torch.cuda.synchronize()
    fdcm.set_stream(DEV, None)
    assert same((planes(fm), fm.scene_bins()), want)


# ---- C. host threads ---------------------------------------------------------------------------------------------------
def _c1(wl, spin, S, variant, n_threads, torch, profile=False):
    """n_threads threads, each with its own map, one shared TemplateSet, a different penalty each; all calls queued on the
    held caller stream S.  profile: count only the threads' calls.  -> (want, got, window flags)"""
    kw = {"plain": {}, "select": {"select": SELECT}, "refine": {"refine": REFINE}}[variant]
    scenes = [wl.X, wl.Y, wl.Z, wl.X][:n_threads]
    fdcm.set_stream(DEV, None)
    maps = [build(s) for s in scenes]
    want = [top10(m, wl.tset, penalty=PENALTIES[i], **kw) for i, m in enumerate(maps)]
    if profile:
        fdcm.profile(True, reset=True)
    fdcm.set_stream(DEV, S.cuda_stream)
    ev = spin.hold(S)
    flags = [None] * n_threads

    def task(i):
        def f():
            flags[i] = not ev.query()
            return top10(maps[i], wl.tset, penalty=PENALTIES[i], **kw)
        return f

    got, err = run_threads([task(i) for i in range(n_threads)])
    torch.cuda.synchronize()
    fdcm.set_stream(DEV, None)
    raise_first(err)
    return want, got, flags


@pytest.mark.parametrize("variant", ["plain", "select", "refine"])
def test_threads_share_a_template_set_with_different_penalties(variant, wl, spin, streams, torch):
    want, got, flags = _c1(wl, spin, streams(), variant, 4, torch)
    assert all(flags), f"the spin had finished before the calls of threads {[i for i, f in enumerate(flags) if not f]} were issued"
    assert len({canon(x) for x in want}) == 4
    bad = [i for i in range(4) if not same(got[i], want[i])]
    assert not bad, f"{variant}: threads {bad} (penalties {[PENALTIES[i].__class__.__name__ if PENALTIES[i] else None for i in bad]}) " \
                    "got another thread's penalty"


@pytest.mark.parametrize("held", [False, True], ids=["library_stream", "held_caller_stream"])
def test_threads_on_one_map(held, wl, spin, streams, torch):
    """Several threads on one map and one set, mixing the search paths, refinement and evaluate: serialised per map."""
    fdcm.set_stream(DEV, None)
    fm = build(wl.X)
    base = top10(fm, wl.tset)
    calls = [
        lambda: top10(fm, wl.tset),
        lambda: top10(fm, wl.tset, select=SELECT),
        lambda: top10(fm, wl.tset, penalty=fdcm.ExponentialPenalty(3.0), refine=REFINE),
        lambda: fdcm.search_dense(fm, wl.tset, DENSE, fdcm.DefaultPenalty(), k=10, select=SELECT, refine=REFINE),
        lambda: fdcm.refine_matches(fm, wl.tset, base, REFINE, PEN),
        lambda: fdcm.evaluate(fm, wl.placed, wl.trans),
    ]
    want = [f() for f in calls]
    ev = None
    if held:
        S = streams()
        fdcm.set_stream(DEV, S.cuda_stream)
        ev = spin.hold(S)
    flags = []

    def repeat(f):
        def g():
            flags.append(ev is None or not ev.query())
            return [f() for _ in range(3)]
        return g

    got, err = run_threads([repeat(f) for f in calls])
    torch.cuda.synchronize()
    fdcm.set_stream(DEV, None)
    raise_first(err)
    if held:
        assert any(flags), "the spin had finished before any thread issued its first call"
    for i, (g, w_) in enumerate(zip(got, want)):
        assert all(same(x, w_) for x in g), f"call {i} on a map shared by {len(calls)} threads"


def test_rebuild_against_search_on_one_handle(wl, torch):
    """One thread rebuilds a handle to X and Y in turn (waiting and not), another searches its resident scene meanwhile:
    every result is the oracle's top-10 of X or of Y, never a mix."""
    want = {"X": oracle_top10(wl.X, wl.tmpls), "Y": oracle_top10(wl.Y, wl.tmpls)}
    assert not same(want["X"], want["Y"])
    fdcm.set_stream(DEV, None)
    fm = build(wl.X)
    assert same(top10(fm, wl.tset), want["X"])
    done = threading.Event()
    seen = []

    def rebuilder():
        try:
            for r in range(6):
                fm.rebuild(wl.Y if r % 2 == 0 else wl.X, wait=r % 4 < 2)
        finally:
            done.set()

    def searcher():
        while not done.is_set() or len(seen) < 8:
            g = top10(fm, wl.tset)
            seen.append("X" if same(g, want["X"]) else "Y" if same(g, want["Y"]) else g)
        return seen

    _, err = run_threads([rebuilder, searcher])
    raise_first(err)
    torn = [s for s in seen if not isinstance(s, str)]
    assert not torn, f"{len(torn)} of {len(seen)} searches equal neither X's nor Y's top-10, e.g. {torn[0]['tmpl_idx']}"
    assert same(top10(fm, wl.tset), want["X"])   # the last rebuild was to X


def test_last_error_is_per_thread(wl):
    """fdcm_last_error(): thread A fails (FDCM_ERR_INVALID) while thread B succeeds; each reads only its own message."""
    fm = build(wl.X)
    both = threading.Barrier(2)
    msg = {}

    def failing():
        with pytest.raises(fdcm.FdcmError) as e:
            top10(fm, wl.tset, select=fdcm.DistinctMatches(max_per_template=-1))
        assert e.value.status == _lib.FDCM_ERR_INVALID
        both.wait(JOIN_S)            # B succeeds now
        both.wait(JOIN_S)
        msg["A"] = fdcm.lib().fdcm_last_error().decode()

    def succeeding():
        both.wait(JOIN_S)            # after A's failure
        top10(fm, wl.tset)
        msg["B"] = fdcm.lib().fdcm_last_error().decode()
        both.wait(JOIN_S)

    _, err = run_threads([failing, succeeding])
    raise_first(err)
    assert "max_per_template" in msg["A"], msg
    assert msg["B"] == "", msg


def test_one_thread_per_device(wl, torch):
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip(f"one thread per device needs at least two devices; this machine has {n}")

    def on(dev):
        fm = fdcm.build_cuda_featuremap(wl.X, fdcm.Dt3CudaParameters(30, 5.0, 1.5, device=dev))
        ts = fdcm.TemplateSet(wl.tmpls, dev)
        return planes(fm)[::7], top10(fm, ts), top10(fm, ts, refine=REFINE), fdcm.search_dense(fm, ts, DENSE, PEN, k=10)

    want = [on(d) for d in range(n)]
    got, err = run_threads([lambda d=d: on(d) for d in range(n)])
    raise_first(err)
    for d in range(n):
        assert same(got[d], want[d]), f"device {d}"
        assert same(got[d], want[0]), f"device {d} against device 0"


# ---- D. profiling ------------------------------------------------------------------------------------------------------
@pytest.fixture
def profiling():
    fdcm.profile(True, reset=True)
    yield
    fdcm.profile(False, reset=True)


def test_profile_counts_scene_batch(profiling, torch):
    """Every scope of a profiled SceneBatch is counted once, also the next scene's build that runs under a search."""
    w, h, n = 640, 480, 6
    tm = synth_templates(12, 20, w, seed=81)
    scenes = [plant_instances(synth_scene(w, h, 200, seed=820 + i), tm, w, h, seed=840 + i) for i in range(n)]
    ts = fdcm.TemplateSet(tm, DEV)
    fdcm.set_stream(DEV, None)
    fdcm.profile(False)
    want = fdcm.SceneBatch(P).search_topk(scenes, ts, SEARCH, OPT, PEN, k=10)
    # the build kernels of these scenes, one build at a time
    fdcm.profile(True, reset=True)
    fm = build(scenes[0])
    for s in scenes[1:]:
        fm.rebuild(s)
    seq = fdcm.profile_report()
    assert seq["raster"]["launches"] == n, seq
    fdcm.profile(True, reset=True)
    got = fdcm.SceneBatch(P).search_topk(scenes, ts, SEARCH, OPT, PEN, k=10)
    torch.cuda.synchronize()
    rep = fdcm.profile_report()
    assert same(got, want)
    counts = {k: (rep.get(k, {}).get("launches", 0), v["launches"]) for k, v in seq.items()}
    assert all(a == b for a, b in counts.values()), f"build scopes counted (batch, one at a time): {counts}"
    assert rep["search"]["launches"] == n and rep["topk"]["launches"] == n, rep


def test_profile_counts_threads(profiling, wl, spin, streams, torch):
    """The C1 run with profiling on: one search and one top-K scope per thread, all resolved."""
    want, got, flags = _c1(wl, spin, streams(), "plain", 4, torch, profile=True)
    assert all(flags), flags
    assert all(same(a, b) for a, b in zip(got, want))
    rep = fdcm.profile_report()
    assert rep["search"]["launches"] == 4 and rep["topk"]["launches"] == 4, rep
