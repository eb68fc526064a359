"""GPU checks of the one-third-octave band-level path (omega4_b200.octave, csrc/octave_kernel.cuh) against the
float64 oracle (oracle/octave_np.py): seeded streams at 44.1, 48 and 96 kHz, tones at every mid-band frequency,
invariance to how a stream is cut into pushes, host / device modes, reset, the C ABI's acceptance of scipy's
own section pairing, bad arguments and the kernels a push launches."""
import ctypes as C

import numpy as np
import pytest
from scipy import signal

from oracle import octave_np as O

pytestmark = pytest.mark.gpu

TOL_DB = 1e-4
FLOOR_DB = -150.0                        # block levels below this are compared by their -inf pattern only


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


@pytest.fixture(scope="module")
def octave():
    from omega4_b200 import octave
    return octave


def run_meter(octave, torch, x, fs, tiles=None):
    """x [n_rows, n] float32 -> (levels, leq, max_level, meter) through ThirdOctaveMeter pushes."""
    n_rows, n = x.shape
    m = octave.ThirdOctaveMeter(fs, n_rows, max_seconds=n / fs + 1, device=0)
    dev = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    tiles, pos, i = tiles or [n], 0, 0
    while pos < n:                                        # cycle the tile pattern until the stream ends
        t = min(tiles[i % len(tiles)], n - pos)
        assert m.push(dev[:, pos:pos + t]) == (pos + t) // m.sub - pos // m.sub
        pos, i = pos + t, i + 1
    return m.levels.cpu().numpy(), m.leq.cpu().numpy(), m.max_level.cpu().numpy(), m


def compare(got, ref, label, floor=FLOOR_DB):
    """Values at or above ``floor`` within TOL_DB; -inf positions identical.  Returns the worst error (dB)."""
    assert got.shape == ref.shape, (label, got.shape, ref.shape)
    assert np.array_equal(np.isneginf(got), np.isneginf(ref)), f"{label}: -inf positions differ"
    assert not np.isnan(got).any() and not np.isposinf(got).any(), label
    sel = np.isfinite(ref) & (ref >= floor)
    err = float(np.abs(got[sel].astype(np.float64) - ref[sel]).max()) if sel.any() else 0.0
    assert err <= TOL_DB, f"{label}: worst error {err} dB over {int(sel.sum())} values"
    return err


def seeded_rows(n_rows, seconds, fs):
    """Sweep + pink noise rows (batch.synth) at peak amplitudes log-spaced in 1e-3 .. 0.9, then one digitally
    silent row and one row at 1e-4 peak amplitude."""
    from omega4_b200.batch.synth import synth_channel
    n = int(seconds * fs)
    amps = np.geomspace(1e-3, 0.9, n_rows)
    x = np.empty((n_rows + 2, n), np.float32)
    for r in range(n_rows):
        v = synth_channel(r // 2, r % 2, n, fs).astype(np.float64)
        x[r] = (v * (amps[r] / np.abs(v).max())).astype(np.float32)
    x[n_rows] = 0.0
    v = synth_channel(7, 1, n, fs).astype(np.float64)
    x[n_rows + 1] = (v * (1e-4 / np.abs(v).max())).astype(np.float32)
    return x


@pytest.mark.parametrize("fs", [44100, 48000, 96000])
def test_seeded_streams_match_oracle(octave, torch, fs):
    x = seeded_rows(6, 12.55 if fs < 96000 else 8.25, fs)          # ends inside a block: Leq sees the partial one
    lv, leq, lmax, m = run_meter(octave, torch, x, fs)
    ref = O.band_levels(x, fs)
    assert m.n_bands == ref["frequencies"].size and lv.shape[2] == m.n_bands + 1
    np.testing.assert_array_equal(m.nominal, ref["nominal"])
    np.testing.assert_allclose(m.frequencies, ref["frequencies"], rtol=1e-15)
    worst = {"levels": compare(lv, ref["levels"], f"{fs} levels"),
             "leq": compare(leq, ref["leq"], f"{fs} leq", floor=-np.inf),
             "max_level": compare(lmax, ref["max_level"], f"{fs} max_level", floor=-np.inf)}
    assert np.isneginf(lv[6]).all() and np.isneginf(leq[6]).all()         # the silent row
    assert np.isfinite(lv[7]).all()                                        # 1e-4 amplitude: every band has energy
    print(f"{fs} Hz: worst |GPU - oracle| " + ", ".join(f"{k} {v:.2e} dB" for k, v in worst.items()))


@pytest.mark.parametrize("fs", [44100, 48000, 96000])
def test_tone_at_every_mid_band_frequency(octave, torch, fs):
    """Row b holds a sine at band b's exact f_m: it reads its amplitude in its own band (energy mean of the
    blocks after 2 s, within 0.01 dB) and matches the oracle."""
    m0 = octave.ThirdOctaveMeter(fs, 1, 1.0)
    fm, nb = m0.frequencies, m0.n_bands
    m0.close()
    t = np.arange(int(4 * fs)) / fs
    amps = np.geomspace(1e-3, 1.0, nb)
    x = np.stack([a * np.sin(2 * np.pi * f * t) for a, f in zip(amps, fm)]).astype(np.float32)
    lv, leq, lmax, _ = run_meter(octave, torch, x, fs)
    for b in range(nb):
        got = 10 * np.log10(np.mean(10.0 ** (lv[b, 20:, b].astype(np.float64) / 10)))
        assert abs(got - 20 * np.log10(amps[b])) <= 0.01, (b, fm[b], got, 20 * np.log10(amps[b]))
    ref = O.band_levels(x, fs)
    compare(lv, ref["levels"], f"{fs} tones")
    compare(leq, ref["leq"], f"{fs} tones leq")          # far bands read a tone deep in their stop band


@pytest.mark.parametrize("fs", [48000, 96000])
def test_tiling_invariance(octave, torch, fs):
    """Ragged pushes give what one push gives: the carried state is exact, so the results are bit-identical
    (the test allows 1e-6 dB)."""
    x = seeded_rows(4, 6.0, fs)
    x[0, 3 * fs:] = 0.0                                   # a signal, then digital silence: its tail keeps ringing
    x[1, :2 * fs] = 0.0                                   # leading digital silence: -inf blocks
    one = run_meter(octave, torch, x, fs)
    cut = run_meter(octave, torch, x, fs, tiles=[1, 777, 4800, 48013, 5, 9600, 12345, 4799])
    for a, b, label in zip(one[:3], cut[:3], ("levels", "leq", "max_level")):
        assert np.array_equal(np.isneginf(a), np.isneginf(b)), label
        f = np.isfinite(a)
        d = float(np.abs(a[f].astype(np.float64) - b[f]).max())
        assert d <= 1e-6, (label, d)
        print(f"{fs} Hz {label}: worst difference between the two cuts {d:.1e} dB")
    assert np.isneginf(one[0][1, :20]).all() and np.isfinite(one[0][1, 20:]).all()
    # after the signal stops the overall column reads -inf while the 20 Hz band still rings
    assert np.isneginf(one[0][0, 30:, -1]).all() and np.isfinite(one[0][0, 30:32, 0]).all()


def test_host_and_device_modes_agree(octave, torch):
    x = seeded_rows(3, 3.37, 48000)
    lv, leq, lmax, _ = run_meter(octave, torch, x, 48000)
    h = octave.third_octave_levels(x, 48000)
    assert np.array_equal(h["levels"], lv) and np.array_equal(h["leq"], leq) and np.array_equal(h["max_level"], lmax)
    np.testing.assert_array_equal(h["nominal"][[0, -1]], [20, 20000])


def test_reset_starts_rows_anew(octave, torch):
    x = seeded_rows(2, 3.0, 48000)
    y = seeded_rows(2, 2.5, 48000) * np.float32(0.5)
    fresh = run_meter(octave, torch, y, 48000)
    _, _, _, m = run_meter(octave, torch, x, 48000)
    m.reset()
    assert m.steps == 0 and np.isneginf(m.leq.cpu().numpy()).all() and np.isneginf(m.max_level.cpu().numpy()).all()
    m.push(torch.from_numpy(y).cuda())
    assert m.levels.shape == fresh[3].levels.shape
    assert np.array_equal(m.levels.cpu().numpy(), fresh[0])
    assert np.array_equal(m.leq.cpu().numpy(), fresh[1]) and np.array_equal(m.max_level.cpu().numpy(), fresh[2])


def _abi_push(lib, N, sos, fs, x):
    """Host-mode push through the C ABI with an explicit section table -> (levels, leq)."""
    sos = np.ascontiguousarray(sos, dtype=np.float64)
    d = N.OctaveDesc(fs, sos.shape[0], sos.ctypes.data_as(C.POINTER(C.c_double)), fs // 10)
    h = lib.omega4_octave_create(C.byref(d), 0)
    assert h, N.last_error()
    try:
        rows, n = x.shape
        cols, steps = sos.shape[0] + 1, n // (fs // 10)
        state = np.zeros((rows, lib.omega4_octave_state_doubles(h)), np.float64)
        lv = np.zeros((rows, steps, cols), np.float32)
        leq = np.zeros((rows, cols), np.float32)
        rc = lib.omega4_octave_push(h, None, N.MEM_HOST, x.ctypes.data, n, rows, n, state.ctypes.data, 1, steps,
                                    lv.ctypes.data, leq.ctypes.data, None)
        N.check(rc, "omega4_octave_push")
        return lv, leq
    finally:
        lib.omega4_octave_destroy(h)


def test_abi_accepts_scipy_section_pairing(octave, torch):
    """scipy pairs the six zeros as g [1, -2, 1], [1, 0, -1], [1, 2, 1]; the kernel runs every section as
    [1, 0, -1] and the gain on the energy, which is the same cascade: it agrees with the package's table."""
    from omega4_b200 import _native as N, tables
    fs = 48000
    b = tables.third_octave_bands(fs)
    scipy_sos = np.stack([signal.butter(3, [f1, f2], btype="bandpass", fs=fs, output="sos")
                          for f1, f2 in zip(b["f1"], b["f2"])])
    x = seeded_rows(2, 2.0, fs)
    lib = N.lib()
    lv1, leq1 = _abi_push(lib, N, scipy_sos, fs, x)
    lv2, leq2 = _abi_push(lib, N, tables.third_octave_sos(fs), fs, x)
    compare(lv1, lv2.astype(np.float64), "scipy pairing")
    compare(leq1, leq2.astype(np.float64), "scipy pairing leq", floor=-np.inf)


def test_bad_arguments_raise(octave, torch):
    from omega4_b200 import _native as N, tables
    for fs in (44101, 7990, 200000, 48000.5):
        with pytest.raises(ValueError):
            octave.ThirdOctaveMeter(fs, 1, 1.0)
    with pytest.raises(ValueError):
        octave.ThirdOctaveMeter(48000, 0, 1.0)
    m = octave.ThirdOctaveMeter(48000, 2, 1.0)
    with pytest.raises(ValueError):
        m.push(torch.zeros((2, 100), dtype=torch.float32))                           # not CUDA
    with pytest.raises(ValueError):
        m.push(torch.zeros((2, 100), dtype=torch.float64, device="cuda"))            # float64
    with pytest.raises(ValueError):
        m.push(torch.zeros((3, 100), dtype=torch.float32, device="cuda"))            # wrong rows
    with pytest.raises(ValueError):
        m.push(torch.zeros((100, 2), dtype=torch.float32, device="cuda").t())        # time stride != 1
    with pytest.raises(ValueError):
        m.push(torch.zeros((2, 48000 + 4800), dtype=torch.float32, device="cuda"))   # beyond max_seconds
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            m.push(torch.zeros((2, 100), dtype=torch.float32, device="cuda:1"))      # wrong device
    m.dev = torch.device("cuda:1")        # on one GPU: pretend the meter lives elsewhere, so a cuda:0 tile is foreign
    with pytest.raises(ValueError):
        m.push(torch.zeros((2, 100), dtype=torch.float32, device="cuda:0"))
    with pytest.raises(ValueError):
        octave.third_octave_levels(np.zeros((2, 4800)), 48000)                       # float64
    with pytest.raises(ValueError):
        octave.third_octave_levels(np.zeros((1, 2, 4800), np.float32), 48000)        # not 2-D
    with pytest.raises(ValueError):
        octave.third_octave_levels(np.zeros((2, 4800), np.float32), 44105)           # bad rate
    lib = N.lib()
    sos = np.ascontiguousarray(tables.third_octave_sos(48000))
    dp = C.POINTER(C.c_double)
    d = N.OctaveDesc(48000, 31, sos.ctypes.data_as(dp), 4410)                         # sub != fs / 10
    assert not lib.omega4_octave_create(C.byref(d), 0) and N.last_error()
    d = N.OctaveDesc(48000, 32, sos.ctypes.data_as(dp), 4800)                         # too many bands
    assert not lib.omega4_octave_create(C.byref(d), 0)
    bad = sos.copy()
    bad[3, 1, 1] = 0.5                                                               # not a zero-pair numerator
    d = N.OctaveDesc(48000, 31, bad.ctypes.data_as(dp), 4800)
    assert not lib.omega4_octave_create(C.byref(d), 0) and "numerator" in N.last_error()
    bad = sos.copy()
    bad[0, 0, 5] = 1.0                                                               # pole on the unit circle
    d = N.OctaveDesc(48000, 31, bad.ctypes.data_as(dp), 4800)
    assert not lib.omega4_octave_create(C.byref(d), 0) and "unit circle" in N.last_error()
    d = N.OctaveDesc(48000, 31, sos.ctypes.data_as(dp), 4800)
    h = lib.omega4_octave_create(C.byref(d), 0)
    assert h
    x = np.zeros((2, 4800), np.float32)
    st = np.zeros((2, lib.omega4_octave_state_doubles(h)))
    lv = np.zeros((2, 1, 32), np.float32)
    assert lib.omega4_octave_push(h, None, N.MEM_HOST, x.ctypes.data, 4800, 2, 4800, None, 1, 1, None, None, None) < 0
    assert lib.omega4_octave_push(h, None, 7, x.ctypes.data, 4800, 2, 4800, st.ctypes.data, 1, 1, None, None, None) < 0
    assert "mem" in N.last_error()
    assert lib.omega4_octave_push(h, None, N.MEM_HOST, x.ctypes.data, 4000, 2, 4800, st.ctypes.data, 1, 1,
                                  None, None, None) < 0                              # ch_stride < n_samples
    assert lib.omega4_octave_push(h, None, N.MEM_HOST, x.ctypes.data + 2, 4800, 2, 4800, st.ctypes.data, 1, 1,
                                  None, None, None) < 0 and "aligned" in N.last_error()
    assert lib.omega4_octave_push(h, None, N.MEM_HOST, x.ctypes.data, 4800, 2, 4800, st.ctypes.data, 1, 0,
                                  lv.ctypes.data, None, None) < 0                    # out_stride below the count
    assert lib.omega4_octave_push(h, None, N.MEM_HOST, x.ctypes.data, 4800, 2, 4800, st.ctypes.data, 1, 1,
                                  lv.ctypes.data, None, None) == 0
    assert np.isneginf(lv).all()
    lib.omega4_octave_destroy(h)


def test_one_launch_per_push(octave, torch):
    """A push is the library's one kernel writing straight into the meter's series (no torch or vendor kernel in
    between), whatever the tile length."""
    m = octave.ThirdOctaveMeter(48000, 16, 10.0)
    tile = torch.randn((16, 48000), device="cuda") * 0.1
    torch.cuda.synchronize()
    before = m.launches
    m.push(tile)
    assert m.launches - before == 1
    m.push(tile[:, :777])
    assert m.launches - before == 2
    m.push(tile[:, :0])
    assert m.launches - before == 2
    assert m.steps == (48000 + 777) // 4800 and m.levels.data_ptr() == m._levels.data_ptr()
