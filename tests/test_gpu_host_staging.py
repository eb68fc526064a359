"""OMEGA4_MEM_HOST staging of the plan, bars and plan-less entry points (omega4_combine, omega4_meter_frames,
omega4_meter_stats, omega4_rfft_batch, omega4_band_map, omega4_waterfall, omega4_bass_bars, omega4_bars_run): host
mode gives bit for bit what device mode gives on the same inputs, an object's staging buffers are reused across
call sizes without changing results, `mem` is validated, and the plan-less calls free what they stage."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MIB = 1 << 20


@pytest.fixture(scope="module")
def N():
    from omega4_b200 import _native
    _native.require_device()
    return _native


@pytest.fixture(scope="module")
def plan():
    from omega4_b200.plan import AnalysisPlan, BASELINE_CONFIGS
    p = AnalysisPlan(48000, BASELINE_CONFIGS, 512, device=0)
    yield p
    p.close()


def _bars_object():
    from omega4_b200.app.spectrum_post import SpectrumPostProcessor
    post = SpectrumPostProcessor()
    post._ensure()
    return post


@pytest.fixture(scope="module")
def bars():
    post = _bars_object()
    yield post
    post.close()


def _run(N, mem, call, data):
    """call(mem, p) with p[name] the address of data[name] in host memory (OMEGA4_MEM_HOST) or of a device copy
    (OMEGA4_MEM_DEVICE), None for None; returns every array as numpy after the call."""
    import torch
    if mem == N.MEM_HOST:
        bufs = {k: None if v is None else v.copy() for k, v in data.items()}
        rc = call(mem, {k: N.ptr(v) for k, v in bufs.items()})
    else:
        dev = {k: None if v is None else torch.from_numpy(v.copy()).cuda() for k, v in data.items()}
        rc = call(mem, {k: None if v is None else v.data_ptr() for k, v in dev.items()})
        torch.cuda.synchronize()
        bufs = {k: None if v is None else v.cpu().numpy() for k, v in dev.items()}
    N.check(rc, "host staging call")
    return bufs


def _host_equals_device(N, call, data, written, unspecified=()):
    """Runs both modes; every array but `unspecified` is bit-identical afterwards and each name in `written` was
    written."""
    h = _run(N, N.MEM_HOST, call, data)
    d = _run(N, N.MEM_DEVICE, call, data)
    for k, v in data.items():
        if v is not None and k not in unspecified:
            assert h[k].tobytes() == d[k].tobytes(), k
    for k in written:
        assert not np.array_equal(h[k], data[k]), f"{k} was not written"
    return h, d


def _fresh_state(state):
    """A call that starts a state fresh writes only part of it; in host mode the rest comes back unspecified."""
    return ("state",) if state == "fresh" else ()


def _carry_on_alike(N, make, *states):
    """A carried call from each state gives bit-identical outputs."""
    outs = [_run(N, N.MEM_HOST, *make(st)[:2]) for st in states]
    for k, v in outs[0].items():
        if k != "state" and v is not None:
            assert v.tobytes() == outs[1][k].tobytes(), k


def _mags(rng, *shape):
    return np.abs(rng.standard_normal(shape)).astype(np.float32)


# ------------------------------------------------------------------ the calls, each with seeded inputs
def _rfft(N, rng, window=True, complex_out=True, batch=5, n=2048):
    data = {"frames": rng.standard_normal((batch, n)).astype(np.float32),
            "mag": np.zeros((batch, n // 2 + 1), np.float32),
            "cx": np.zeros((batch, n // 2 + 1), np.complex64) if complex_out else None}
    win = np.hanning(n).astype(np.float32) if window else None

    def call(mem, p):
        return N.lib().omega4_rfft_batch(0, None, mem, p["frames"], batch, n, N.ptr(win), p["mag"], p["cx"])
    return call, data, [k for k in ("mag", "cx") if data[k] is not None]


def _band_map(N, rng, comp=True, db=1, rows=4, ln=700):
    bands = np.array([[0, 3], [3, 3], [10, 40], [40, 41], [100, 650], [690, 700], [650, 760]], np.int32)
    c = rng.uniform(0.5, 2.0, ln).astype(np.float32) if comp else None
    data = {"spec": _mags(rng, rows, ln), "out": np.zeros((rows, len(bands)), np.float32)}

    def call(mem, p):
        return N.lib().omega4_band_map(0, None, mem, p["spec"], rows, ln, N.ptr(bands), len(bands), N.ptr(c),
                                       p["out"], db)
    return call, data, ["out"]


def _waterfall_state(N, rng, n_ch, ln, lo, hi):
    """A carried state: what a fresh host-mode call over a few rows leaves."""
    st = np.zeros((n_ch, N.WATERFALL_STATE), np.float32)
    spec = _mags(rng, n_ch, 6, ln)
    db = np.empty((n_ch, 6, hi - lo), np.float32)
    N.check(N.lib().omega4_waterfall(0, None, N.MEM_HOST, N.ptr(spec), n_ch, 6, ln, lo, hi, 0, 1, 0.0, N.ptr(st), 1,
                                     N.ptr(db), None, None), "omega4_waterfall")
    return st


def _waterfall(N, rng, state="carried", rowstat=True, n_ch=3, n_rows=7, ln=1024, lo=5, hi=900):
    st = state if isinstance(state, np.ndarray) else None if state is None else (
        np.zeros((n_ch, N.WATERFALL_STATE), np.float32) if state == "fresh" else _waterfall_state(N, rng, n_ch, ln, lo, hi))
    data = {"spec": _mags(rng, n_ch, n_rows, ln), "state": st,
            "db": np.zeros((n_ch, n_rows, hi - lo), np.float32), "norm": np.zeros((n_ch, n_rows, hi - lo), np.float32),
            "rowstat": np.zeros((n_ch, n_rows, 4), np.float32) if rowstat else None}
    fresh = 1 if isinstance(state, str) and state == "fresh" else 0

    def call(mem, p):
        return N.lib().omega4_waterfall(0, None, mem, p["spec"], n_ch, n_rows, ln, lo, hi, 0, 1, 0.0, p["state"], fresh,
                                        p["db"], p["norm"], p["rowstat"])
    return call, data, ["db", "norm"] + (["rowstat"] if rowstat else []) + (["state"] if st is not None else [])


def _bass_bars(N, rng, state=True, n_ch=3, n_frames=4, n_bins=4097, n_bars=20):
    first = rng.integers(0, n_bins - 300, n_bars)
    count = rng.integers(0, 300, n_bars)
    count[3] = 0
    bins = np.ascontiguousarray(np.stack([first, count], 1).astype(np.int32))
    comp = rng.uniform(0.5, 2.0, n_bars).astype(np.float32)
    data = {"mag": _mags(rng, n_ch, n_frames, n_bins), "out": np.zeros((n_ch, n_frames, n_bars), np.float32),
            "state": rng.uniform(0.0, 1.0, (n_ch, n_bars)).astype(np.float32) if state else None}

    def call(mem, p):
        return N.lib().omega4_bass_bars(0, None, mem, p["mag"], n_ch, n_frames, n_bins, N.ptr(bins), N.ptr(comp),
                                        n_bars, p["state"], p["out"])
    return call, data, ["out"] + (["state"] if state else [])


def _meter_frames(N, rng, plan, weighted_only=False, n=5):
    w = plan.meter_window
    data = {"frames": (0.1 * rng.standard_normal((n, w))).astype(np.float64),
            "lufs": None if weighted_only else np.zeros(n), "tp": None if weighted_only else np.zeros(n),
            "w": np.zeros((n, w))}

    def call(mem, p):
        return N.lib().omega4_meter_frames(plan.handle, None, mem, p["frames"], n, p["lufs"], p["tp"], p["w"])
    return call, data, ["w"] + ([] if weighted_only else ["lufs", "tp"])


def _meter_stats(N, rng, plan, state="carried", n_ch=3, n=50):
    def series():
        return rng.uniform(-90.0, -10.0, (n_ch, n)), rng.uniform(-30.0, 0.0, (n_ch, n))
    st = state if isinstance(state, np.ndarray) else None
    if isinstance(state, str):
        st = np.zeros((n_ch, N.METER_STATE_DOUBLES))
        if state == "carried":
            li, tp = series()
            plan.meter_stats_host(li, tp, state=st, fresh=True)
    li, tp = series()
    data = {"li": li, "tp": tp, "state": st, "meters": np.zeros((n_ch, n, N.N_METERS), np.float32)}
    fresh = 1 if isinstance(state, str) and state == "fresh" else 0

    def call(mem, p):
        return N.lib().omega4_meter_stats(plan.handle, None, mem, p["li"], p["tp"], n_ch, n, 0, p["state"], p["meters"],
                                          fresh)
    return call, data, ["meters"] + (["state"] if st is not None else [])


def _combine(N, rng, plan, absent=(1,), rows=3):
    data = {f"m{r}": None if r in absent else _mags(rng, rows, n // 2 + 1) for r, n in enumerate(plan.sizes)}
    data["out"] = np.zeros((rows, plan.target_bins), np.float32)

    def call(mem, p):
        mags = N.ptr_array([p[f"m{r}"] for r in range(len(plan.sizes))])
        return N.lib().omega4_combine(plan.handle, None, mem, mags, rows, p["out"])
    return call, data, ["out"]


def _bars_run(N, rng, post, state="carried", peaks=True, n_ch=3, n_hops=5):
    nv = post.n_valid
    st = None
    if state is not None:
        st = np.zeros((n_ch, 1 + nv), np.float32)
        if state == "carried":
            st[:, 0] = 1.0
            st[:, 1:] = rng.uniform(0.0, 1.0, (n_ch, nv))
    data = {"spec": _mags(rng, n_ch, n_hops, post.bars), "state": st,
            "band": np.zeros((n_ch, n_hops, nv), np.float32),
            "peak": np.zeros((n_ch, n_hops, nv), np.float32) if peaks else None}
    fresh = 1 if isinstance(state, str) and state == "fresh" else 0

    def call(mem, p):
        return N.lib().omega4_bars_run(post._handle, None, mem, p["spec"], n_ch, n_hops, p["state"], fresh, p["band"],
                                       p["peak"])
    return call, data, ["band"] + (["peak"] if peaks else []) + (["state"] if st is not None else [])


# ------------------------------------------------------------------ host mode == device mode
@pytest.mark.parametrize("window", [True, False])
@pytest.mark.parametrize("complex_out", [True, False])
def test_rfft_batch_host_equals_device(N, window, complex_out):
    _host_equals_device(N, *_rfft(N, np.random.default_rng(1), window, complex_out))


@pytest.mark.parametrize("comp,db", [(True, 0), (False, 1), (True, 2)])
def test_band_map_host_equals_device(N, comp, db):
    _host_equals_device(N, *_band_map(N, np.random.default_rng(2), comp, db))


@pytest.mark.parametrize("state", [None, "fresh", "carried"])
@pytest.mark.parametrize("rowstat", [True, False])
def test_waterfall_host_equals_device(N, state, rowstat):
    h, d = _host_equals_device(N, *_waterfall(N, np.random.default_rng(3), state, rowstat), _fresh_state(state))
    if state == "fresh":
        _carry_on_alike(N, lambda st: _waterfall(N, np.random.default_rng(30), st, rowstat), h["state"], d["state"])


@pytest.mark.parametrize("state", [True, False])
def test_bass_bars_host_equals_device(N, state):
    _host_equals_device(N, *_bass_bars(N, np.random.default_rng(4), state))


@pytest.mark.parametrize("weighted_only", [True, False])
def test_meter_frames_host_equals_device(N, plan, weighted_only):
    _host_equals_device(N, *_meter_frames(N, np.random.default_rng(5), plan, weighted_only))


@pytest.mark.parametrize("state", [None, "fresh", "carried"])
def test_meter_stats_host_equals_device(N, plan, state):
    h, d = _host_equals_device(N, *_meter_stats(N, np.random.default_rng(6), plan, state), _fresh_state(state))
    if state == "fresh":
        _carry_on_alike(N, lambda st: _meter_stats(N, np.random.default_rng(60), plan, st), h["state"], d["state"])


@pytest.mark.parametrize("absent", [(), (1,), (0, 2)])
def test_combine_host_equals_device(N, plan, absent):
    _host_equals_device(N, *_combine(N, np.random.default_rng(7), plan, absent))


@pytest.mark.parametrize("state", [None, "fresh", "carried"])
@pytest.mark.parametrize("peaks", [True, False])
def test_bars_run_host_equals_device(N, bars, state, peaks):
    _host_equals_device(N, *_bars_run(N, np.random.default_rng(8), bars, state, peaks))


# ------------------------------------------------------------------ an object's staging buffers across sizes
def test_object_stages_reused_across_sizes(N):
    """Large, small, large host calls on one plan and one bars object (the plan's three calls interleaved, so they
    share its buffers) give what fresh objects give.  meter_stats runs without a state: one that started fresh holds
    unspecified values (_fresh_state), which the shared and the fresh plan need not agree on."""
    from omega4_b200.plan import AnalysisPlan, BASELINE_CONFIGS

    def calls(p, post, size, seed):
        big = size == "large"
        return [_combine(N, np.random.default_rng(seed), p, (1,), rows=40 if big else 1),
                _meter_frames(N, np.random.default_rng(seed + 1), p, False, n=70 if big else 1),
                _meter_stats(N, np.random.default_rng(seed + 2), p, None, n_ch=9 if big else 1, n=300 if big else 2),
                _meter_frames(N, np.random.default_rng(seed + 3), p, True, n=33 if big else 2),
                _bars_run(N, np.random.default_rng(seed + 4), post, "carried", True, n_ch=6 if big else 1,
                          n_hops=40 if big else 1)]

    shared, shared_post = AnalysisPlan(48000, BASELINE_CONFIGS, 512, device=0), _bars_object()
    try:
        for i, size in enumerate(["large", "small", "large"]):
            got = [_run(N, N.MEM_HOST, c, d) for c, d, _ in calls(shared, shared_post, size, 10 * i)]
            fresh, fresh_post = AnalysisPlan(48000, BASELINE_CONFIGS, 512, device=0), _bars_object()
            try:
                want = [_run(N, N.MEM_HOST, c, d) for c, d, _ in calls(fresh, fresh_post, size, 10 * i)]
            finally:
                fresh.close()
                fresh_post.close()
            for g, w in zip(got, want):
                for k in w:
                    if w[k] is not None:
                        assert g[k].tobytes() == w[k].tobytes(), (size, k)
    finally:
        shared.close()
        shared_post.close()


# ------------------------------------------------------------------ `mem` validation
def test_every_entry_point_rejects_a_bad_mem(N, plan, bars):
    """Valid device buffers, mem = 7: every call fails with a message naming `mem`."""
    import torch
    rng = np.random.default_rng(9)
    for name, (call, data, _) in [("rfft_batch", _rfft(N, rng)), ("band_map", _band_map(N, rng)),
                                  ("waterfall", _waterfall(N, rng)), ("bass_bars", _bass_bars(N, rng)),
                                  ("meter_frames", _meter_frames(N, rng, plan)),
                                  ("meter_stats", _meter_stats(N, rng, plan)), ("combine", _combine(N, rng, plan)),
                                  ("bars_run", _bars_run(N, rng, bars))]:
        dev = {k: None if v is None else torch.from_numpy(v).cuda() for k, v in data.items()}
        rc = call(7, {k: None if v is None else v.data_ptr() for k, v in dev.items()})
        torch.cuda.synchronize()
        assert rc < 0 and "mem" in N.last_error(), (name, rc, N.last_error())


# ------------------------------------------------------------------ plan-less calls free what they stage
@pytest.mark.parametrize("make", [_rfft, _band_map, _waterfall, _bass_bars], ids=lambda f: f.__name__.strip("_"))
def test_plan_less_host_calls_free_their_buffers(N, make):
    import torch
    rng = np.random.default_rng(10)
    sizes = {_rfft: dict(batch=64, n=8192), _band_map: dict(rows=512, ln=2048),
             _waterfall: dict(n_ch=8, n_rows=32, ln=4096, lo=5, hi=4000), _bass_bars: dict(n_ch=8, n_frames=32)}
    call, data, _ = make(N, rng, **sizes[make])
    host = {k: None if v is None else N.ptr(v) for k, v in data.items()}
    N.check(call(N.MEM_HOST, host), "warm-up")
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(200):
        N.check(call(N.MEM_HOST, host), "host call")
    torch.cuda.synchronize()
    free1 = torch.cuda.mem_get_info()[0]
    assert abs(free1 - free0) <= 2 * MIB, (free0 - free1) / MIB
