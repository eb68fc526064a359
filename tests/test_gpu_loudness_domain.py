"""The BS.1770-4 / EBU Tech 3342 loudness path (csrc/loudness_kernel.cuh) across its domain.

Summary: omega4_loudness_summary called directly, in host and device mode, on hand-built float32 momentary /
short-term series, against oracle/bs1770_np.py applied to the same float32 values in float64.  The loudness range
is a difference of two exact order statistics (the kernel's radix select), so it must equal
``np.float32(v[k_hi] - v[k_lo])`` bit for bit; the maxima are exact and I agrees within 1e-5 LU.  The series are
built where a select goes wrong: every survivor count 1 .. 64, ties, runs of consecutive float32 values, values
sharing their top 16 or 24 bits, mixed signs with +-0 and tiny magnitudes, NaN heads, -inf runs, the absolute
gate, empty and near-empty series, 10 h series, and row strides whose gap holds NaN, +inf and +100.  Every value
is kept at least 1e-3 LU from the relative gates, which kernel and oracle sum in a different order.

Push: seeded streams at 8, 22.05, 32, 44.1, 88.2 and 192 kHz, with 1, 3 and 32 channels and 1, 5, 33 and 257
streams, against the oracle at 0.01 LU; ragged pushes around the 100 ms sub-block and the 8-segment runs of the
chain kernel; tiles at unaligned addresses; the carried sample peak.  Plus the rejection of sample rates at which
the closed-form K-weighting is unstable."""
import ctypes as C

import numpy as np
import pytest

from oracle import bs1770_np as B
from test_gpu_loudness import compare_with_oracle, run_meter

gpu = pytest.mark.gpu

TOL_I = 1e-5
HDR, CH_DOUBLES = 30, 6              # carried state layout per stream (include/omega4_cuda.h)


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


@pytest.fixture(scope="module")
def loud():
    from omega4_b200 import loudness
    return loudness


@pytest.fixture(scope="module")
def handle(loud):
    h = loud._Handle(48000, np.ones(2), 0)
    yield h
    h.close()


# ------------------------------------------------------------------ summary on hand-built series
def f32(v):
    return np.asarray(v, dtype=np.float32)


def from_bits(u):
    return np.asarray(u, dtype=np.uint32).view(np.float32)


def _rel_gate(v, rel_lu):
    v = v[np.isfinite(v)]
    v = v[v > B.ABS_GATE]
    return None if v.size == 0 else (v, B._lufs(np.mean(10.0 ** ((v + 0.691) / 10.0))) + rel_lu)


def clear_of_relative_gates(m, s):
    """Whether every value above the absolute gate lies >= 1e-3 LU from the relative gate it meets."""
    for v, rel_lu in ((m, B.REL_GATE_I), (s, B.REL_GATE_LRA)):
        r = _rel_gate(np.asarray(v, np.float64), rel_lu)
        if r is not None and np.abs(r[0] - r[1]).min() < 1e-3:
            return False
    return True


def keep_clear(m, s):
    """Move the few values within 2e-3 LU of a relative gate 0.01 LU down (the gates move by far less)."""
    for v, rel_lu in ((m, B.REL_GATE_I), (s, B.REL_GATE_LRA)):
        r = _rel_gate(v.astype(np.float64), rel_lu)
        if r is not None:
            near = np.isfinite(v) & (np.abs(v.astype(np.float64) - r[1]) < 2e-3)
            v[near] -= np.float32(0.01)
    return m, s


def heads(m, s):
    """NaN heads as the push writes them: 3 momentary and 29 short-term steps."""
    m, s = f32(m).copy(), f32(s).copy()
    m[:3], s[:29] = np.nan, np.nan
    return m, s


def summary_series():
    """name -> (momentary, short_term) float32 of one stream."""
    rng = np.random.default_rng(5)
    out = {}
    for n in range(1, 65):                                   # every survivor count: distinct values, shuffled
        for seed in range(100):
            r = np.random.default_rng(1000 * n + seed)
            v = f32(-30.0 + r.permutation(n) * 0.37 + r.uniform(0.0, 0.3, n))
            if clear_of_relative_gates(v, v):
                break
        out[f"count{n}"] = (v, v)
    out["equal"] = heads(np.full(50, -23.0), np.full(80, -23.0))
    base = np.uint32(0xC1B800F0)                             # -23.000...f with the low byte at 0xF0
    run = from_bits(base - np.arange(300, dtype=np.uint32))  # 300 consecutive floats across two key bytes
    out["nextafter-run"] = (rng.permutation(run), rng.permutation(run))
    pos = from_bits(np.uint32(0x40A00000) + np.arange(300, dtype=np.uint32))   # 5.0f upwards
    out["nextafter-run-positive"] = (rng.permutation(pos), rng.permutation(pos))
    top24 = from_bits((np.uint32(0xC1B80000) & np.uint32(0xFFFFFF00)) | rng.integers(0, 256, 400).astype(np.uint32))
    top16 = from_bits(np.uint32(0xC1B80000) | rng.integers(0, 65536, 600).astype(np.uint32))
    out["top24"] = (top24, rng.permutation(top24))
    out["top16"] = (top16, rng.permutation(top16))
    mix = np.concatenate([[-5.0, 3.0, 0.0, -0.0, 1e-30, -1e-30, 1e-38, -1e-38, 1e-45, -1e-45, 12.5, 7.25, -2.0, 1.5],
                          rng.uniform(-8.0, 12.0, 120)])
    out["mixed-signs"] = (f32(rng.permutation(mix)), f32(rng.permutation(mix)))
    m, s = heads(rng.uniform(-40.0, -12.0, 400), rng.uniform(-40.0, -12.0, 400))
    m[100:110], s[150:190] = -np.inf, -np.inf
    out["nan-heads-inf-runs"] = (m, s)
    at = f32(np.concatenate([np.full(20, -70.0), np.full(20, np.nextafter(np.float32(-70.0), np.float32(0))),
                             rng.choice([-65.0, -60.5, -68.0], 60)]))
    out["absolute-gate"] = (rng.permutation(at), rng.permutation(at))
    for name, (m, s) in out.items():
        assert clear_of_relative_gates(m, s), name
    return out


def pack(series, stride=None, poison=False):
    """Series of different lengths -> [n_streams, stride] float32, NaN after each end (or NaN / +inf / +100 in
    the gap beyond n_steps when ``poison``); returns (M, S, n_steps)."""
    n_steps = max(len(m) for m, _ in series)
    stride = stride or n_steps
    M = np.full((len(series), stride), np.nan, np.float32)
    S = np.full_like(M, np.nan)
    if poison:
        gap = np.resize(np.array([np.nan, np.inf, 100.0], np.float32), stride - n_steps)
        M[:, n_steps:], S[:, n_steps:] = gap, gap[::-1]
    for i, (m, s) in enumerate(series):
        M[i, :len(m)], S[i, :len(s)] = m, s
    return M, S, n_steps


def summary(handle, torch, mode, M, S, n_steps):
    from omega4_b200 import _native as N
    lib = N.lib()
    n_streams, stride = M.shape
    if mode == "host":
        out = np.empty((n_streams, 4), np.float32)
        rc = lib.omega4_loudness_summary(handle.ptr, None, N.MEM_HOST, M.ctypes.data, S.ctypes.data, n_streams,
                                         n_steps, stride, out.ctypes.data)
        N.check(rc, "omega4_loudness_summary")
        return out
    dm, ds = torch.from_numpy(M).cuda(), torch.from_numpy(S).cuda()
    out = torch.empty((n_streams, 4), dtype=torch.float32, device="cuda")
    rc = lib.omega4_loudness_summary(handle.ptr, None, N.MEM_DEVICE, dm.data_ptr(), ds.data_ptr(), n_streams, n_steps,
                                     stride, out.data_ptr())
    N.check(rc, "omega4_loudness_summary")
    return out.cpu().numpy()


def check_summary(got, M, S, n_steps, labels):
    for i, label in enumerate(labels):
        m, s = M[i, :n_steps].astype(np.float64), S[i, :n_steps].astype(np.float64)
        I, lra = B.integrated(m), B.loudness_range(s)
        if np.isneginf(I):
            assert np.isneginf(got[i, 0]), (label, got[i])
        else:
            assert abs(float(got[i, 0]) - I) <= TOL_I, (label, "I", float(got[i, 0]), I)
        assert got[i, 1] == np.float32(lra), (label, "LRA", float(got[i, 1]), lra)
        for j, v in ((2, m), (3, s)):
            want = np.float32(B._nanmax(v))
            assert (np.isnan(want) and np.isnan(got[i, j])) or got[i, j] == want, (label, j, got[i, j], want)


SUMMARY = summary_series()


@gpu
@pytest.mark.parametrize("mode", ["host", "device"])
@pytest.mark.parametrize("poison", [False, True], ids=["dense", "poisoned-stride"])
def test_summary_hand_built_series(handle, torch, mode, poison):
    names = list(SUMMARY)
    n_steps = max(len(m) for m, _ in SUMMARY.values())
    M, S, n = pack([SUMMARY[k] for k in names], stride=n_steps + 13 if poison else None, poison=poison)
    got = summary(handle, torch, mode, M, S, n)
    check_summary(got, M, S, n, names)
    assert got[names.index("equal"), 1] == 0.0


@gpu
@pytest.mark.parametrize("mode", ["host", "device"])
@pytest.mark.parametrize("n_steps", [0, 1, 29, 30])
def test_summary_short_series(handle, torch, mode, n_steps):
    rng = np.random.default_rng(n_steps)
    series = [keep_clear(*heads(rng.uniform(-30.0, -15.0, n_steps), rng.uniform(-30.0, -15.0, n_steps))) for _ in range(3)]
    assert all(clear_of_relative_gates(m, s) for m, s in series)
    M, S, _ = pack(series, stride=max(n_steps, 1) + 5, poison=True)
    got = summary(handle, torch, mode, M, S, n_steps)
    check_summary(got, M, S, n_steps, [f"{n_steps} steps #{i}" for i in range(3)])
    if n_steps <= 29:
        assert np.all(got[:, 1] == 0.0) and np.isnan(got[:, 3]).all()
    if n_steps <= 3:
        assert np.isneginf(got[:, 0]).all() and np.isnan(got[:, 2]).all()


@gpu
@pytest.mark.parametrize("mode", ["host", "device"])
def test_summary_ten_hours(handle, torch, mode):
    """360 000 steps (10 h) for 4 streams."""
    rng = np.random.default_rng(36)
    n = 360000
    series = []
    for i in range(4):
        m, s = heads(rng.uniform(-45.0, -10.0, n) + 3.0 * i, rng.uniform(-45.0, -10.0, n) - 2.0 * i)
        m[1000 * (i + 1):1000 * (i + 1) + 5000] = -np.inf
        s[7000 * (i + 1):7000 * (i + 1) + 300] = -np.inf
        keep_clear(m, s)
        assert clear_of_relative_gates(m, s)
        series.append((m, s))
    M, S, _ = pack(series)
    check_summary(summary(handle, torch, mode, M, S, n), M, S, n, [f"10 h #{i}" for i in range(4)])


# ------------------------------------------------------------------ the push across its domain
def seeded_streams(n_streams, n_ch, seconds, fs, silent=(0, 1)):
    """Sweep + pink noise per (stream, channel), scaled to peak amplitudes log-spaced in 1e-4 .. 0.9, with the
    channel ``silent`` = (stream, channel) digitally zero."""
    from omega4_b200.batch.synth import synth_channel
    n = int(seconds * fs)
    amps = np.geomspace(1e-4, 0.9, n_streams * n_ch)
    np.random.default_rng(n_streams * 131 + n_ch).shuffle(amps)
    x = np.empty((n_streams, n_ch, n), np.float32)
    for s in range(n_streams):
        for c in range(n_ch):
            v = synth_channel(s, c, n, fs).astype(np.float64)
            x[s, c] = (v * (amps[s * n_ch + c] / np.abs(v).max())).astype(np.float32)
    x[silent] = 0.0
    return x


W3 = [1.0, 0.5, 1.41]
W32 = [0.0 if c % 7 == 3 else 1.0 + 0.05 * c for c in range(32)]
DOMAIN = [
    ("8k-mono-257", 257, 1, 10.0, 8000, "mono", [1.0]),
    ("22.05k-3ch-33", 33, 3, 10.0, 22050, W3, W3),
    ("32k-32ch-5", 5, 32, 6.0, 32000, W32, W32),
    ("44.1k-mono-33", 33, 1, 20.0, 44100, "mono", [1.0]),
    ("44.1k-3ch-5", 5, 3, 30.0, 44100, W3, W3),
    ("88.2k-3ch-5", 5, 3, 10.0, 88200, W3, W3),
    ("192k-32ch-1", 1, 32, 4.0, 192000, W32, W32),
]


@gpu
@pytest.mark.parametrize("name,n_streams,n_ch,seconds,fs,layout,weights", DOMAIN, ids=[c[0] for c in DOMAIN])
def test_push_domain_matches_oracle(loud, torch, name, n_streams, n_ch, seconds, fs, layout, weights):
    x = seeded_streams(n_streams, n_ch, seconds, fs, silent=(n_streams - 1, n_ch - 1))
    m, s, summ, meter = run_meter(loud, torch, x, fs, layout)
    ref, worst = compare_with_oracle(x, fs, weights, m, s, summ, name)
    st = meter._state.cpu().numpy()
    lin = st[:, HDR + CH_DOUBLES * np.arange(n_ch) + 5]
    assert np.array_equal(lin, np.abs(x).max(axis=2).astype(np.float64))     # the carried linear sample peak
    print(f"{name}: worst |GPU - oracle| " + ", ".join(f"{k} {v:.2e}" for k, v in worst.items()))


def ragged(sub):
    return [1, sub - 1, sub, sub + 1, 8 * sub - 1, 8 * sub, 8 * sub + 1, 9 * sub + 3]


def assert_cut_invariant(a, b, label):
    """The rule of test_tiling_invariance: equal above -70 LUFS within 1e-5, -inf only far below the gate."""
    assert np.array_equal(np.isnan(a), np.isnan(b)), label
    loud_ = (a > -70.0) | (b > -70.0)
    assert np.isfinite(a[loud_]).all() and np.isfinite(b[loud_]).all(), label
    if loud_.any():
        assert np.abs(a[loud_].astype(np.float64) - b[loud_]).max() <= 1e-5, label
    differ = np.isneginf(a) != np.isneginf(b)
    assert (np.maximum(a[differ], b[differ]) < -120.0).all(), (label, np.maximum(a[differ], b[differ]))


@gpu
@pytest.mark.parametrize("fs,n_ch,layout", [(44100, 1, "mono"), (22050, 3, W3), (8000, 32, W32)])
def test_ragged_pushes(loud, torch, fs, n_ch, layout):
    """Pushes of 1, sub - 1, sub, sub + 1, 8 sub - 1, 8 sub, 8 sub + 1 and 9 sub + 3 samples: every position of a
    sub-block boundary, of a chain kernel run of 8 segments and of its 100 ms warm-up."""
    x = seeded_streams(5, n_ch, 25.0, fs, silent=(4, 0))
    x[1, :, :3 * fs] = 0.0                             # leading digital silence
    x[0, :, 15 * fs:] = 0.0                            # a signal, then digital silence
    m1, s1, sum1, _ = run_meter(loud, torch, x, fs, layout)
    mt, st, sumt, _ = run_meter(loud, torch, x, fs, layout, tiles=ragged(fs // 10))
    assert_cut_invariant(m1, mt, "M")
    assert_cut_invariant(s1, st, "S")
    for k in ("integrated", "lra", "max_momentary", "max_short_term"):
        a, b = sum1[k].astype(np.float64), sumt[k].astype(np.float64)
        assert np.array_equal(np.isneginf(a), np.isneginf(b)) and np.array_equal(np.isnan(a), np.isnan(b)), (k, a, b)
        f = np.isfinite(a)
        assert np.abs(a[f] - b[f]).max(initial=0.0) <= 1e-5, k
    assert np.array_equal(sum1["sample_peak"], sumt["sample_peak"])


@gpu
def test_unaligned_device_tiles(loud, torch):
    """Tiles cut from a wider buffer at odd column offsets (base not 16-byte aligned, odd row stride) give exactly
    what the same tiles of a contiguous buffer give."""
    fs, n_ch = 44100, 3
    x = seeded_streams(5, n_ch, 12.0, fs)
    rows, n = 5 * n_ch, x.shape[2]
    tiles = [4411, 12345, 1, 77777, 4410, 9999]
    want_m, want_s, want_sum, _ = run_meter(loud, torch, x, fs, W3, tiles=tiles)
    wide = torch.full((rows, n + 11), float("nan"), dtype=torch.float32, device="cuda")
    off = 3
    wide[:, off:off + n] = torch.from_numpy(x.reshape(rows, n)).cuda()
    m = loud.LoudnessMeter(fs, W3, 5, max_seconds=n / fs + 1, device=0)
    pos, i = 0, 0
    while pos < n:
        t = min(tiles[i % len(tiles)], n - pos)
        view = wide[:, off + pos:off + pos + t]
        assert view.stride(0) == n + 11
        m.push(view)
        pos, i = pos + t, i + 1
    assert np.array_equal(m.momentary.cpu().numpy(), want_m, equal_nan=True)
    assert np.array_equal(m.short_term.cpu().numpy(), want_s, equal_nan=True)
    got = m.summary()
    for k in want_sum:
        assert np.array_equal(got[k], want_sum[k], equal_nan=True), k


# ------------------------------------------------------------------ sample rates
@pytest.mark.parametrize("fs", [0, 10, 1000, 3000, 7990, 44101, 48000.5, 192010, 384000, -48000, "48000"])
def test_python_rejects_unsupported_rates(loud, fs):
    """[8000, 192000] like the octave meter; below a few kHz the closed-form K-weighting is unstable (CPU only)."""
    with pytest.raises(ValueError):
        loud._check_rate(fs)
    with pytest.raises(ValueError):
        loud.program_loudness(np.zeros((1, 1, 4800), np.float32), fs, "mono")


@pytest.mark.parametrize("fs", [8000, 22050, 44100, 192000])
def test_python_accepts_supported_rates(loud, fs):
    assert loud._check_rate(fs) == fs and loud._check_rate(float(fs)) == fs


@gpu
def test_create_rejects_unstable_biquads():
    """omega4_loudness_create checks |a2| < 1 and |a1| < 1 + a2 for both sections, as omega4_octave_create does."""
    from omega4_b200 import _native as N
    lib = N.lib()
    dp = C.POINTER(C.c_double)
    w = np.ones(1)

    def create(fs, k):
        k = [np.ascontiguousarray(c, dtype=np.float64) for c in k]
        d = N.LoudnessDesc(fs, 1, w.ctypes.data_as(dp), *(c.ctypes.data_as(dp) for c in k), fs // 10)
        return lib.omega4_loudness_create(C.byref(d), 0), k

    for fs in (10, 1000, 3000):                         # poles of the closed form outside the unit circle
        h, _ = create(fs, B.k_weighting(fs))
        assert not h and "unit circle" in N.last_error(), fs
    sb, sa, hb, ha = B.k_weighting(48000)
    for bad in ([1.0, -2.0, 1.0], [1.0, 0.5, -1.0], [1.0, 1.6, 0.5], [2.0, -1.9, 0.9]):   # |a2| = 1, |a1| >= 1 + a2, a0 != 1
        for k in ((sb, bad, hb, ha), (sb, sa, hb, bad)):
            h, _ = create(48000, k)
            assert not h, bad
    for fs in (8000, 192000):
        h, _ = create(fs, B.k_weighting(fs))
        assert h, (fs, N.last_error())
        lib.omega4_loudness_destroy(h)
