"""The push contract the three block meters share (include/omega4_cuda.h): loudness (omega4_b200.loudness),
one-third-octave levels (omega4_b200.octave) and the sound level meter (omega4_b200.slm).  A single-row tile
whose row stride torch reports as 1, a device-mode push whose out_stride is shorter than the blocks it
completes, and host-mode pointers that are not float / double aligned."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

FS = 48000
SUB = FS // 10
SENTINEL = 12345.0


def _loudness():
    from omega4_b200 import loudness

    def push(lib, m, mem, x, ch_stride, rows, n, state, out_stride, series):
        return lib.omega4_loudness_push(m._h.ptr, None, mem, x, ch_stride, rows, n, state, 1, out_stride,
                                        series[0], series[1], None)

    return {"make": lambda rows, seconds: loudness.LoudnessMeter(FS, "mono", rows, seconds),
            "results": lambda m: [m.momentary, m.short_term, m.sample_peak],
            "block": lambda m: (), "n_series": 2, "push": push}


def _octave():
    from omega4_b200 import octave

    def push(lib, m, mem, x, ch_stride, rows, n, state, out_stride, series):
        return lib.omega4_octave_push(m._h.ptr, None, mem, x, ch_stride, rows, n, state, 1, out_stride, series[0],
                                      None, None)

    return {"make": lambda rows, seconds: octave.ThirdOctaveMeter(FS, rows, seconds),
            "results": lambda m: [m.levels, m.leq, m.max_level],
            "block": lambda m: (m.n_bands + 1,), "n_series": 1, "push": push}


def _slm():
    from omega4_b200 import slm

    def push(lib, m, mem, x, ch_stride, rows, n, state, out_stride, series):
        return lib.omega4_slm_push(m._h.ptr, None, mem, x, ch_stride, rows, n, state, 1, out_stride, series[0], None)

    return {"make": lambda rows, seconds: slm.SoundLevelMeter(FS, rows, seconds),
            "results": lambda m: [m.levels, m.totals],
            "block": lambda m: (len(slm.WEIGHTINGS), len(slm.QUANTITIES)), "n_series": 1, "push": push}


METERS = {"loudness": _loudness, "octave": _octave, "slm": _slm}


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


@pytest.fixture(scope="module")
def lib():
    from omega4_b200 import _native as N
    return N.lib()


def noise(rows, n, seed=7):
    return (np.random.default_rng(seed).standard_normal((rows, n)) * 0.1).astype(np.float32)


@pytest.mark.parametrize("kind", sorted(METERS))
def test_single_row_tile_with_unit_row_stride(kind, torch):
    """torch gives a [1, n] view of an [n, 1] tensor the strides (1, 1); it is contiguous, and a push of it gives
    bit for bit what the push of a [1, n] tensor with strides (n, 1) gives."""
    M = METERS[kind]()
    n = int(2.37 * FS)
    x = noise(1, n)
    outs = []
    for single in (False, True):
        m = M["make"](1, 3.0)
        dev = torch.from_numpy(x[0]).cuda().reshape(n, 1).t() if single else torch.from_numpy(x).cuda()
        assert dev.shape == (1, n) and dev.is_contiguous() and dev.stride(0) == (1 if single else n)
        for a, b in ((0, 7 * SUB + 11), (7 * SUB + 11, n)):
            m.push(dev[:, a:b])
        outs.append([t.cpu().numpy() for t in M["results"](m)] + [m._state.cpu().numpy()])
    for got, want in zip(outs[1], outs[0]):
        assert got.shape == want.shape and np.array_equal(got, want, equal_nan=True), kind


@pytest.mark.parametrize("kind", sorted(METERS))
def test_device_push_writes_no_block_at_or_beyond_out_stride(kind, torch, lib):
    """A device-mode push of 2 rows completing 5 blocks with out_stride 2 writes blocks 0 and 1 of each row into
    columns 0 and 1, as a full-width push does, and nothing else of the 2 x 8 series buffer."""
    from omega4_b200 import _native as N
    M = METERS[kind]()
    rows, n = 2, 5 * SUB
    m = M["make"](rows, 1.0)
    x = torch.from_numpy(noise(rows, n)).cuda()
    block = M["block"](m)

    def push(out_stride, width):
        state = torch.zeros((rows, m._h.state_doubles), dtype=torch.float64, device="cuda")
        series = [torch.full((rows, width) + block, SENTINEL, dtype=torch.float32, device="cuda")
                  for _ in range(M["n_series"])]
        rc = M["push"](lib, m, N.MEM_DEVICE, x.data_ptr(), n, rows, n, state.data_ptr(), out_stride,
                       [s.data_ptr() for s in series])
        N.check(rc, kind)
        torch.cuda.synchronize()
        return [s.cpu().numpy() for s in series], state.cpu().numpy()

    full, full_state = push(5, 5)
    short, short_state = push(2, 8)
    for f, s in zip(full, short):
        flat = s.reshape((rows * 8,) + block)                 # row r of out_stride 2 starts at entry 2 r
        for r in range(rows):
            assert np.array_equal(flat[2 * r:2 * r + 2], f[r, :2], equal_nan=True), (kind, r)
        assert (flat[2 * rows:] == SENTINEL).all(), kind
    assert np.array_equal(short_state, full_state)


@pytest.mark.parametrize("kind", sorted(METERS))
def test_host_push_rejects_unaligned_samples_and_state(kind, lib):
    """Host mode: samples 2 bytes and state 4 bytes off their alignment are rejected.  Both come from arrays one
    element longer than the push needs, so nothing is read or written outside them either way."""
    from omega4_b200 import _native as N
    M = METERS[kind]()
    rows, n = 2, SUB
    m = M["make"](rows, 1.0)
    x = np.zeros(rows * n + 1, np.float32)
    st = np.zeros(rows * m._h.state_doubles + 1, np.float64)

    def push(xp, sp):
        return M["push"](lib, m, N.MEM_HOST, xp, n, rows, n, sp, 1, [None] * M["n_series"])

    assert push(x.ctypes.data, st.ctypes.data) == 0, N.last_error()
    assert push(x.ctypes.data + 2, st.ctypes.data) < 0 and "aligned" in N.last_error()
    assert push(x.ctypes.data, st.ctypes.data + 4) < 0 and "aligned" in N.last_error()
