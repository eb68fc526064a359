"""GPU checks of the BS.1770-4 / EBU Tech 3342 loudness path (omega4_b200.loudness, csrc/loudness_kernel.cuh)
against the float64 oracle (oracle/bs1770_np.py): EBU conformance cases, seeded sweep + pink streams at
48 and 96 kHz, invariance to how the stream is cut into pushes, host / device modes, state reset, bad
arguments and the kernels a push launches."""
import ctypes as C

import numpy as np
import pytest

from oracle import bs1770_np as B
from test_bs1770_oracle import CONFORMANCE, check_conformance, tech3341_case6, tech3341_case9, tone

pytestmark = pytest.mark.gpu

TOL_LU = 0.01
HDR, CH_DOUBLES = 30, 6              # carried state layout per stream (include/omega4_cuda.h)


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


@pytest.fixture(scope="module")
def loud():
    from omega4_b200 import loudness
    return loudness


def run_meter(loud, torch, x, fs, weights, tiles=None):
    """x [n_streams, C, n] float32 -> (momentary, short_term, summary dict, meter) through LoudnessMeter pushes."""
    n_streams, n_ch, n = x.shape
    m = loud.LoudnessMeter(fs, weights, n_streams, max_seconds=n / fs + 1, device=0)
    dev = torch.from_numpy(np.ascontiguousarray(x).reshape(n_streams * n_ch, n)).cuda()
    tiles, pos, i = tiles or [n], 0, 0
    while pos < n:                                       # cycle the tile pattern until the stream ends
        t = min(tiles[i % len(tiles)], n - pos)
        m.push(dev[:, pos:pos + t])
        pos, i = pos + t, i + 1
    summ = m.summary()
    return m.momentary.cpu().numpy(), m.short_term.cpu().numpy(), summ, m


def compare_series(got, ref, tol, label):
    """Finite values above -70 LUFS within tol; NaN and -inf positions identical.  Returns the worst error."""
    assert got.shape == ref.shape, (label, got.shape, ref.shape)
    assert np.array_equal(np.isnan(got), np.isnan(ref)), f"{label}: NaN positions differ"
    assert np.array_equal(np.isneginf(got), np.isneginf(ref)), f"{label}: -inf positions differ"
    sel = np.isfinite(ref) & (ref > -70.0)
    err = float(np.abs(got[sel].astype(np.float64) - ref[sel]).max()) if sel.any() else 0.0
    assert err <= tol, f"{label}: worst error {err} LU over {int(sel.sum())} values"
    return err


def compare_with_oracle(x, fs, weights, got_m, got_s, summ, label):
    ref = B.program_loudness(x, fs, weights)
    worst = {"M": compare_series(got_m, ref["momentary"], TOL_LU, label + " M"),
             "S": compare_series(got_s, ref["short_term"], TOL_LU, label + " S")}
    for key, rkey in (("integrated", "integrated"), ("lra", "lra"), ("max_momentary", "max_momentary"),
                      ("max_short_term", "max_short_term")):
        g, r = summ[key].astype(np.float64), ref[rkey].astype(np.float64)
        assert np.array_equal(np.isnan(g), np.isnan(r)) and np.array_equal(np.isneginf(g), np.isneginf(r)), (label, key, g, r)
        f = np.isfinite(r)
        worst[key] = float(np.abs(g[f] - r[f]).max()) if f.any() else 0.0
        assert worst[key] <= TOL_LU, (label, key, worst[key])
    return ref, worst


@pytest.mark.parametrize("name,segments,what,expected", CONFORMANCE, ids=[c[0] for c in CONFORMANCE])
def test_ebu_conformance(loud, torch, name, segments, what, expected):
    x = tone(segments).astype(np.float32)[None]
    m, s, summ, _ = run_meter(loud, torch, x, 48000, "stereo")
    r = {"momentary": m[0].astype(np.float64), "short_term": s[0].astype(np.float64),
         "integrated": float(summ["integrated"][0]), "lra": float(summ["lra"][0])}
    check_conformance(r, what, expected)
    compare_with_oracle(x, 48000, [1.0, 1.0], m, s, summ, name)


def test_ebu_3341_case6_and_case9(loud, torch):
    x, w = tech3341_case6()
    x = x.astype(np.float32)[None]
    m, s, summ, _ = run_meter(loud, torch, x, 48000, w)
    assert abs(summ["integrated"][0] + 23.0) <= 0.1
    compare_with_oracle(x, 48000, w, m, s, summ, "3341-6")
    x = tech3341_case9().astype(np.float32)[None]
    m, s, summ, _ = run_meter(loud, torch, x, 48000, "stereo")
    assert np.abs(s[0, 29:] + 23.0).max() <= 0.1
    compare_with_oracle(x, 48000, [1.0, 1.0], m, s, summ, "3341-9")


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


SEEDED = [
    ("stereo-48k", 32, 2, 60.0, 48000, "stereo", [1.0, 1.0]),
    ("5.1-48k", 1, 6, 60.0, 48000, "5.1", [1.0, 1.0, 1.0, 0.0, 1.41, 1.41]),
    ("8ch-96k", 4, 8, 30.0, 96000, [1.0, 1.0, 1.0, 0.0, 1.41, 1.41, 1.0, 1.0], [1.0, 1.0, 1.0, 0.0, 1.41, 1.41, 1.0, 1.0]),
]


@pytest.mark.parametrize("name,n_streams,n_ch,seconds,fs,layout,weights", SEEDED, ids=[c[0] for c in SEEDED])
def test_seeded_streams_match_oracle(loud, torch, name, n_streams, n_ch, seconds, fs, layout, weights):
    x = seeded_streams(n_streams, n_ch, seconds, fs)
    m, s, summ, meter = run_meter(loud, torch, x, fs, layout)
    ref, worst = compare_with_oracle(x, fs, weights, m, s, summ, name)
    # sample peak: the carried linear peak is exactly max |x| (float32), the dBFS value agrees to float32 rounding
    st = meter._state.cpu().numpy()
    lin = st[:, HDR + CH_DOUBLES * np.arange(n_ch) + 5]
    assert np.array_equal(lin, np.abs(x).max(axis=2).astype(np.float64))
    pk = summ["sample_peak"].astype(np.float64)
    assert np.array_equal(np.isneginf(pk), np.isneginf(ref["sample_peak"]))
    f = np.isfinite(ref["sample_peak"])
    assert np.abs(pk[f] - ref["sample_peak"][f]).max() <= 1e-4
    print(f"{name}: worst |GPU - oracle| " + ", ".join(f"{k} {v:.2e}" for k, v in worst.items()))


@pytest.mark.parametrize("fs", [48000, 96000])
def test_tiling_invariance(loud, torch, fs):
    """Above the -70 LUFS gate, series and summary do not depend on how the stream is cut into pushes.  Below it,
    after a signal stops, a sub-block can read -inf in one cut and a finite value far below the gate in another
    (include/omega4_cuda.h, omega4_loudness_push)."""
    x = seeded_streams(3, 2, 20.0, fs, silent=(2, 0))
    x[1, :, :3 * fs] = 0.0                             # leading digital silence: -inf momentary / short-term values
    x[0, :, 12 * fs:] = 0.0                            # a signal, then 8 s of digital silence
    m1, s1, sum1, _ = run_meter(loud, torch, x, fs, "stereo")
    mt, st, sumt, _ = run_meter(loud, torch, x, fs, "stereo", tiles=[1, 511, 4799, 4800, 4801, 77777, 9600, 12345])
    for a, b, label in ((m1, mt, "M"), (s1, st, "S")):
        assert np.array_equal(np.isnan(a), np.isnan(b)), label
        loud_ = (a > -70.0) | (b > -70.0)
        assert np.isfinite(a[loud_]).all() and np.isfinite(b[loud_]).all(), label
        assert np.abs(a[loud_].astype(np.float64) - b[loud_]).max() <= 1e-5, label
        differ = np.isneginf(a) != np.isneginf(b)
        assert (np.maximum(a[differ], b[differ]) < -120.0).all(), (label, np.maximum(a[differ], b[differ]))
    assert np.isneginf(m1[1, 3:30]).all() and np.isneginf(mt[1, 3:30]).all()
    assert np.isneginf(s1[1, 29]) and np.isneginf(st[1, 29])
    assert np.isneginf(m1[0, 140:]).any()                # 2 s into the silence (from step 120) a run restarted on zeros
    for k in ("integrated", "lra", "max_momentary", "max_short_term"):
        assert np.abs(sum1[k].astype(np.float64) - sumt[k]).max() <= 1e-5, k
    assert np.array_equal(sum1["sample_peak"], sumt["sample_peak"])


def test_host_and_device_modes_agree(loud, torch):
    x = seeded_streams(2, 2, 8.0, 48000)
    m, s, summ, _ = run_meter(loud, torch, x, 48000, "stereo")
    h = loud.program_loudness(x, 48000, "stereo")
    assert np.array_equal(h["momentary"], m, equal_nan=True) and np.array_equal(h["short_term"], s, equal_nan=True)
    for k in ("integrated", "lra", "max_momentary", "max_short_term", "sample_peak"):
        assert np.array_equal(h[k], summ[k], equal_nan=True), k


def test_reset_starts_streams_anew(loud, torch):
    x = seeded_streams(2, 2, 6.0, 48000)
    y = seeded_streams(2, 2, 5.0, 48000, silent=(1, 0)) * np.float32(0.5)
    _, _, fresh_sum, fresh = run_meter(loud, torch, y, 48000, "stereo")
    _, _, _, m = run_meter(loud, torch, x, 48000, "stereo")
    m.reset()
    assert m.steps == 0 and np.isneginf(m.summary()["sample_peak"]).all()
    m.push(torch.from_numpy(y.reshape(4, -1)).cuda())
    assert m.momentary.shape == fresh.momentary.shape
    assert torch.equal(torch.nan_to_num(m.momentary, 1.0), torch.nan_to_num(fresh.momentary, 1.0))
    again = m.summary()
    for k in fresh_sum:
        assert np.array_equal(again[k], fresh_sum[k], equal_nan=True), k


def test_bad_arguments_raise(loud, torch):
    from omega4_b200 import _native as N
    with pytest.raises(ValueError):
        loud.LoudnessMeter(44101, "stereo", 1, 1.0)
    with pytest.raises(ValueError):
        loud.LoudnessMeter(48000, [1.0, -1.0], 1, 1.0)
    with pytest.raises(ValueError):
        loud.LoudnessMeter(48000, "7.1", 1, 1.0)
    m = loud.LoudnessMeter(48000, "stereo", 2, 1.0)
    with pytest.raises(ValueError):
        m.push(torch.zeros((4, 100), dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        m.push(torch.zeros((3, 100), dtype=torch.float32, device="cuda"))
    with pytest.raises(ValueError):
        m.push(torch.zeros((4, 100), dtype=torch.float32))
    with pytest.raises(ValueError):
        m.push(torch.zeros((100, 4), dtype=torch.float32, device="cuda").t())
    with pytest.raises(ValueError):
        m.push(torch.zeros((4, 48000 + 4800), dtype=torch.float32, device="cuda"))   # beyond max_seconds
    with pytest.raises(ValueError):
        loud.program_loudness(np.zeros((1, 3, 4800), np.float32), 48000, "stereo")
    with pytest.raises(ValueError):
        loud.program_loudness(np.zeros((1, 2, 4800)), 48000, "stereo")
    with pytest.raises(ValueError):
        loud.program_loudness(np.zeros((2, 4800), np.float32), 48000, "mono")
    lib = N.lib()
    w = np.ones(2)
    k = [np.ascontiguousarray(c) for c in B.k_weighting(48000)]
    dp = C.POINTER(C.c_double)
    d = N.LoudnessDesc(48000, 2, w.ctypes.data_as(dp), *(c.ctypes.data_as(dp) for c in k), 4410)   # sub != fs / 10
    assert not lib.omega4_loudness_create(C.byref(d), 0)
    assert N.last_error()
    d.sub = 4800
    h = lib.omega4_loudness_create(C.byref(d), 0)
    assert h
    x = np.zeros((2, 4800), np.float32)
    rc = lib.omega4_loudness_push(h, None, N.MEM_HOST, x.ctypes.data, 4800, 1, 4800, None, 1, 1, None, None, None)
    assert rc < 0                                      # NULL state
    rc = lib.omega4_loudness_push(h, None, 7, x.ctypes.data, 4800, 1, 4800, x.ctypes.data, 1, 1, None, None, None)
    assert rc < 0 and "mem" in N.last_error()
    lib.omega4_loudness_destroy(h)


def test_push_launches_only_library_kernels(loud, torch):
    """A push is the library's two kernels writing straight into the meter's series (no torch or vendor kernel in
    between); a summary is one more."""
    m = loud.LoudnessMeter(48000, "stereo", 8, 10.0)
    tile = torch.randn((16, 48000), device="cuda") * 0.1
    torch.cuda.synchronize()
    before = m.launches
    m.push(tile)
    assert m.launches - before == 2
    m.push(tile[:, :777])
    assert m.launches - before == 4
    m.summary()
    assert m.launches - before == 5
    assert m.steps == (48000 + 777) // 4800 and m.momentary.data_ptr() == m._series_m.data_ptr()
