"""GPU checks of the sound level meter (omega4_b200.slm, csrc/slm_kernel.cuh) against the float64 oracle
(oracle/slm_np.py): seeded rows at five sample rates, known answers for tones, decays and bursts, invariance to
how a stream is cut into pushes, host / device modes and row layouts, reset and capacity, exact percentiles, the
C ABI's rejections and the kernels a push and a query launch."""
import ctypes as C

import numpy as np
import pytest

from oracle import slm_np as O

pytestmark = pytest.mark.gpu

TOL_DB = 1e-4
FLOOR_DB = -150.0                        # values below this are compared by their -inf pattern only
PCTS = (0, 1, 5, 10, 50, 90, 95, 99, 100)


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


@pytest.fixture(scope="module")
def slm():
    from omega4_b200 import slm
    return slm


def run_meter(slm, torch, x, fs, tiles=None):
    """x [n_rows, n] float32 -> (levels, totals, state, meter) through SoundLevelMeter pushes."""
    n_rows, n = x.shape
    m = slm.SoundLevelMeter(fs, n_rows, max_seconds=n / fs + 1, device=0)
    dev = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    tiles, pos, i = tiles or [n], 0, 0
    while pos < n:                                        # cycle the tile pattern until the stream ends
        t = min(tiles[i % len(tiles)], n - pos)
        assert m.push(dev[:, pos:pos + t]) == (pos + t) // m.sub - pos // m.sub
        pos, i = pos + t, i + 1
    return m.levels.cpu().numpy(), m.totals.cpu().numpy(), m._state.cpu().numpy(), m


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
    """Sweep + pink rows (batch.synth) at peak amplitudes log-spaced in 1e-4 .. 0.9, then one digitally silent row
    and one row that falls silent for its last quarter."""
    from omega4_b200.batch.synth import synth_channel
    n = int(seconds * fs)
    amps = np.geomspace(1e-4, 0.9, n_rows)
    x = np.empty((n_rows + 2, n), np.float32)
    for r in range(n_rows):
        v = synth_channel(r // 2, r % 2, n, fs).astype(np.float64)
        x[r] = (v * (amps[r] / np.abs(v).max())).astype(np.float32)
    x[n_rows] = 0.0
    x[n_rows + 1] = x[n_rows - 1]
    x[n_rows + 1, 3 * n // 4:] = 0.0
    return x


def check_oracle(lv, tot, x, fs, label):
    ref = O.sound_levels(x, fs)
    return compare(lv, ref["levels"], f"{label} levels"), compare(tot, ref["totals"], f"{label} totals", -np.inf)


@pytest.mark.parametrize("fs", [8000, 44100, 48000, 96000, 192000])
def test_seeded_rows_match_oracle(slm, torch, fs):
    x = seeded_rows(6, 6.37 if fs < 96000 else 3.13, fs)           # ends inside a block: totals see the partial one
    lv, tot, _, m = run_meter(slm, torch, x, fs)
    assert lv.shape == (8, x.shape[1] // m.sub, 3, 6) and tot.shape == (8, 3, 4)
    e_lv, e_tot = check_oracle(lv, tot, x, fs, str(fs))
    assert np.isneginf(lv[6]).all() and np.isneginf(tot[6]).all()         # the silent row
    # the row that falls silent: its last block reads -inf in LZeq and LZpeak, while the A and C filters still
    # ring and F and S still decay
    assert np.isneginf(lv[7, -1, 2, [0, 5]]).all() and np.isfinite(lv[7, -1, :2]).all()
    assert np.isfinite(lv[7, :, :, 1:5]).all()
    print(f"{fs} Hz: worst |GPU - oracle| levels {e_lv:.2e} dB, totals {e_tot:.2e} dB")


def _tone(f, amp, seconds, fs, silence=0.0):
    t = np.arange(int(seconds * fs)) / fs
    x = amp * np.sin(2 * np.pi * f * t)
    return np.concatenate([x, np.zeros(int(silence * fs))]).astype(np.float32)


def test_known_answers(slm, torch):
    """The oracle's known answers through the GPU: a 1 kHz sine reads Leq 20 log10 a - 3.01 and Lpeak 20 log10 a
    in A, C and Z; LF and LS decay at 34.7 and 4.34 dB/s; 4 kHz bursts give LFmax - LF and LSmax - LS equal to
    10 log10(1 - e^(-T_b / tau))."""
    fs = 48000
    amps = (1.0, 0.1, 1e-3)
    x = np.stack([_tone(1000.0, a, 10.0, fs) for a in amps] + [_tone(1000.0, 0.5, 3.0, fs, silence=7.0)])
    lv, tot, _, _ = run_meter(slm, torch, x, fs)
    for r, a in enumerate(amps):
        want_eq = 20 * np.log10(a) - 10 * np.log10(2.0)
        assert np.abs(lv[r, 10:, :, 0] - want_eq).max() <= 0.01
        assert np.abs(lv[r, 10:, :, 5] - 20 * np.log10(a)).max() <= 0.01
        assert np.abs(lv[r, 80:, :, 4] - want_eq).max() <= 0.01
        assert np.abs(tot[r, :, 0] - want_eq).max() <= 0.01
    d = lv[3, :, 0].astype(np.float64)
    for q, tau, j0, j1 in ((3, 0.125, 31, 36), (4, 1.0, 31, 59)):
        rate = -(d[j1, q] - d[j0, q]) / ((j1 - j0) / 10.0)
        assert abs(rate / (10 * np.log10(np.e) / tau) - 1.0) <= 0.01, (q, rate)
    bursts = (1000, 500, 200, 100, 50, 20, 10)
    xb = np.zeros((len(bursts), 3 * fs), np.float32)
    for i, ms in enumerate(bursts):
        n_b = int(ms * fs / 1000)
        xb[i, fs:fs + n_b] = 0.5 * np.sin(2 * np.pi * 4000.0 * np.arange(n_b) / fs)
    m = slm.SoundLevelMeter(fs, 1, 10.0)
    m.push(torch.from_numpy(_tone(4000.0, 0.5, 8.0, fs)[None]).cuda())
    steady = m.levels.cpu().numpy()[0, -1].astype(np.float64)
    _, tb, _, _ = run_meter(slm, torch, xb, fs)
    for i, ms in enumerate(bursts):
        for q, tau in ((1, 0.125), (2, 1.0)):
            want = 10 * np.log10(1.0 - np.exp(-ms / 1000.0 / tau))
            got = tb[i, :, q] - steady[:, 3 if q == 1 else 4]
            assert np.abs(got - want).max() <= 0.1, (ms, tau, got, want)


@pytest.mark.parametrize("fs", [48000, 44100])
def test_tiling_is_bit_identical(slm, torch, fs):
    sub = fs // 10
    x = seeded_rows(3, 12.0, fs)
    one = run_meter(slm, torch, x, fs)
    cut = run_meter(slm, torch, x, fs, tiles=[1, sub - 1, sub + 1, 7919, 10 * fs, 33, 2 * sub])
    for a, b, label in zip(one[:3], cut[:3], ("levels", "totals", "state")):
        assert a.shape == b.shape and np.array_equal(a, b), label


def test_host_and_device_modes_and_layouts(slm, torch):
    fs = 48000
    base = seeded_rows(31, 2.05, fs)                                          # 33 rows
    for n_rows in (1, 31, 32, 33, 257):
        x = np.resize(base, (n_rows, base.shape[1])).astype(np.float32) * np.float32(0.999)
        lv, tot, _, _ = run_meter(slm, torch, x, fs)
        h = slm.sound_levels(x, fs, percentiles=PCTS)
        assert np.array_equal(h["levels"], lv) and np.array_equal(h["totals"], tot), n_rows
        m = slm.SoundLevelMeter(fs, n_rows, 3.0)
        # row stride > n and an address that is only float-aligned: a tile_view-like slice of a wider buffer
        wide = torch.zeros((n_rows, x.shape[1] + 37), dtype=torch.float32, device="cuda")
        wide[:, 3:3 + x.shape[1]] = torch.from_numpy(x).cuda()
        m.push(wide[:, 3:3 + x.shape[1]])
        assert np.array_equal(m.levels.cpu().numpy(), lv) and np.array_equal(m.totals.cpu().numpy(), tot), n_rows
        got = m.percentiles(PCTS).cpu().numpy()
        assert np.array_equal(got, h["percentiles"], equal_nan=True), n_rows
    check_oracle(lv[:8], tot[:8], x[:8], fs, "257 rows")


def test_reset_and_capacity(slm, torch):
    fs = 48000
    x = seeded_rows(2, 3.0, fs)
    y = seeded_rows(2, 2.5, fs) * np.float32(0.5)
    fresh = run_meter(slm, torch, y, fs)
    _, _, _, m = run_meter(slm, torch, x, fs)
    m.reset()
    assert m.steps == 0 and np.isneginf(m.totals.cpu().numpy()).all()
    assert np.isnan(m.percentiles([50]).cpu().numpy()).all()
    m.push(torch.from_numpy(y).cuda())
    assert np.array_equal(m.levels.cpu().numpy(), fresh[0]) and np.array_equal(m.totals.cpu().numpy(), fresh[1])
    m2 = slm.SoundLevelMeter(fs, 4, 1.0)
    m2.push(torch.zeros((4, 40000), dtype=torch.float32, device="cuda"))
    with pytest.raises(ValueError):
        m2.push(torch.zeros((4, 14000), dtype=torch.float32, device="cuda"))     # block 11 > 10 steps
    assert m2.push(torch.zeros((4, 8000), dtype=torch.float32, device="cuda")) == 2
    for fs_bad in (44101, 7990, 200000):
        with pytest.raises(ValueError):
            slm.SoundLevelMeter(fs_bad, 1, 1.0)


def test_percentiles_are_exact_order_statistics(slm, torch):
    fs = 8000
    x = seeded_rows(4, 30.0, fs)
    x[0, 4 * 800:9 * 800] = 0.0                                              # -inf blocks in row 0's LZeq / LZpeak
    lv, _, _, m = run_meter(slm, torch, x, fs)
    assert np.isneginf(lv[0, 4:9, 2, [0, 5]]).all()
    for w in m.WEIGHTINGS:
        for q in ("eq", "F", "Smax", "peak"):
            got = m.percentiles(PCTS, w, q).cpu().numpy()
            col = lv[:, :, m.WEIGHTINGS.index(w), m.QUANTITIES.index(q)]
            assert np.array_equal(got, O.percentiles(col, PCTS), equal_nan=True), (w, q)
    # short series through the C ABI in host mode: n_steps 0, 1, 2 and a crafted column with ties and -inf
    from omega4_b200 import _native as N
    lib = N.lib()
    series = np.full((2, 5, 3, 6), 7.0, np.float32)
    series[0, :, 1, 2] = [-np.inf, 3.0, 3.0, -np.inf, 1.5]
    series[1, :, 1, 2] = [2.0, -1.0, 2.0, 2.0, -np.inf]
    pct = np.array(PCTS, np.float64)
    for n_steps in (0, 1, 2, 5):
        out = np.zeros((2, pct.size), np.float32)
        assert lib.omega4_slm_percentiles(m._h.ptr, None, N.MEM_HOST, series.ctypes.data, 2, n_steps, 5, 8,
                                          pct.size, pct.ctypes.data, out.ctypes.data) == 0
        assert np.array_equal(out, O.percentiles(series[:, :n_steps, 1, 2], PCTS), equal_nan=True), n_steps


def test_abi_rejections(slm, torch):
    from omega4_b200 import _native as N, tables
    lib = N.lib()
    dp = C.POINTER(C.c_double)
    fs = 48000
    sa = np.ascontiguousarray(tables.iec61672_weighting_sos("A", fs))
    sc = np.ascontiguousarray(tables.iec61672_weighting_sos("C", fs))

    def create(a=sa, c=sc, rate=fs, sub=fs // 10):
        d = N.SlmDesc(rate, sub, a.ctypes.data_as(dp) if a is not None else None,
                      c.ctypes.data_as(dp) if c is not None else None)
        return lib.omega4_slm_create(C.byref(d), 0)

    assert not create(a=None) and not create(c=None)
    assert not create(rate=44101, sub=4410) and not create(sub=4410) and not create(rate=200000, sub=20000)
    bad = sa.copy(); bad[0, 1] = 0.5 * bad[0, 0]                              # not g [1, +-2, 1]
    assert not create(a=bad) and "numerator" in N.last_error()
    bad = sa.copy(); bad[0, 1] = -bad[0, 1]                                   # A with six zeros at z = 1
    assert not create(a=bad) and "zeros" in N.last_error()
    bad = sc.copy(); bad[1, 1] = -bad[1, 1]                                   # C with four zeros at z = -1
    assert not create(c=bad) and "zeros" in N.last_error()
    assert not create(a=np.ascontiguousarray(sa[[1, 2, 2]]))                 # A with six zeros at z = 1
    bad = sa.copy(); bad[2, 5] = 1.0                                          # |a2| = 1
    assert not create(a=bad) and "unit circle" in N.last_error()
    bad = sc.copy(); bad[0, 4] = -2.5; bad[0, 5] = 0.9                        # |a1| >= 1 + a2
    assert not create(c=bad) and "unit circle" in N.last_error()
    bad = sa.copy(); bad[1, 3] = 2.0                                          # a0 != 1
    assert not create(a=bad)
    h = create()
    assert h and lib.omega4_slm_state_doubles(h) == 41
    x = np.zeros((2, 4800), np.float32)
    st = np.zeros((2, 41))
    lv = np.zeros((2, 1, 3, 6), np.float32)
    tot = np.zeros((2, 3, 4), np.float32)
    H = N.MEM_HOST

    def push(samples=x.ctypes.data, ch=4800, rows=2, n=4800, state=st.ctypes.data, stride=1, levels=lv.ctypes.data,
             mem=H, handle=h):
        return lib.omega4_slm_push(handle, None, mem, samples, ch, rows, n, state, 1, stride, levels, tot.ctypes.data)

    assert push(handle=None) < 0 and push(samples=None) < 0 and push(state=None) < 0
    assert push(mem=7) < 0 and "mem" in N.last_error()
    assert push(rows=-1) < 0 and push(n=-1) < 0 and push(stride=-1) < 0
    assert push(ch=4000) < 0                                                  # ch_stride < n_samples
    assert push(samples=x.ctypes.data + 2) < 0 and "aligned" in N.last_error()
    assert push(stride=0) < 0 and "out_stride" in N.last_error()             # below the block count in host mode
    assert push(rows=0) == 0 and push(n=0) == 0
    assert push() == 0 and np.isneginf(lv).all() and np.isneginf(tot).all()
    pct = np.array([10.0, 90.0])
    out = np.zeros((2, 2), np.float32)

    def query(levels=lv.ctypes.data, rows=2, steps=1, stride=1, col=0, n_pct=2, p=pct, o=out.ctypes.data, mem=H,
              handle=h):
        return lib.omega4_slm_percentiles(handle, None, mem, levels, rows, steps, stride, col, n_pct,
                                          p.ctypes.data if p is not None else None, o)

    assert query(handle=None) < 0 and query(levels=None) < 0 and query(o=None) < 0 and query(p=None) < 0
    assert query(mem=7) < 0 and query(rows=-1) < 0 and query(steps=-1) < 0
    assert query(steps=2, stride=1) < 0                                      # stride < n_steps
    assert query(col=-1) < 0 and query(col=18) < 0 and "column" in N.last_error()
    assert query(n_pct=0) < 0 and query(n_pct=65, p=np.zeros(65)) < 0
    for bad in (np.array([10.0, 100.5]), np.array([-0.1, 5.0]), np.array([np.nan, 5.0])):
        assert query(p=bad) < 0 and "[0, 100]" in N.last_error()
    assert query(levels=lv.ctypes.data + 2) < 0 and "aligned" in N.last_error()
    assert query(col=17) == 0 and np.isneginf(out).all()
    lib.omega4_slm_destroy(h)
    m = slm.SoundLevelMeter(fs, 2, 1.0)
    for bad in ([101.0], [np.nan], []):
        with pytest.raises(ValueError):
            m.percentiles(bad)
    with pytest.raises(ValueError):
        m.percentiles([50], "B")
    with pytest.raises(ValueError):
        m.push(torch.zeros((2, 100), dtype=torch.float32))                    # not CUDA
    with pytest.raises(ValueError):
        m.push(torch.zeros((3, 100), dtype=torch.float32, device="cuda"))     # wrong rows
    with pytest.raises(ValueError):
        m.push(torch.zeros((100, 2), dtype=torch.float32, device="cuda").t())  # time stride != 1


def test_one_launch_per_push_and_query(slm, torch):
    m = slm.SoundLevelMeter(48000, 40, 10.0)
    tile = torch.randn((40, 48000), device="cuda") * 0.1
    torch.cuda.synchronize()
    before = m.launches
    m.push(tile)
    assert m.launches - before == 1
    m.push(tile[:, :777])
    assert m.launches - before == 2
    m.push(tile[:, :0])
    assert m.launches - before == 2
    m.percentiles((10, 50, 90), "C", "Fmax")
    assert m.launches - before == 3
    assert m.steps == (48000 + 777) // 4800 and m.levels.data_ptr() == m._levels.data_ptr()
