"""CPU checks of the sound level meter's definitions: the closed-form A / C weighting sections
(tables.iec61672_weighting_sos) against scipy's bilinear design, the design's deviation from the analog curve,
known answers of the float64 oracle (oracle/slm_np.py) for tones, decays and bursts, the percentile rule and the
sample-rate rejection."""
import numpy as np
import pytest
from scipy import signal

from oracle import slm_np as O

RATES = (8000, 44100, 48000, 96000, 192000)
NOMINAL = (20, 25, 31.5, 40, 50, 63, 80, 100, 125, 160, 200, 250, 315, 400, 500, 630, 800, 1000, 1250, 1600,
           2000, 2500, 3150, 4000, 5000, 6300, 8000, 10000, 12500, 16000, 20000)


@pytest.fixture(scope="module")
def tables():
    from omega4_b200 import tables
    return tables


def _mag_db(sos, f, fs):
    """|H| in dB of a section cascade, evaluated in extended precision: near the low-frequency poles the float64
    evaluation of 1 + a1 z^-1 + a2 z^-2 alone is uncertain by about 1e-9 dB."""
    w = 2 * np.pi * np.asarray(f, dtype=np.longdouble) / np.longdouble(fs)
    zi = np.cos(w) - 1j * np.sin(w).astype(np.clongdouble)
    h = np.ones_like(zi)
    for b0, b1, b2, a0, a1, a2 in np.asarray(sos, dtype=np.longdouble):
        h *= (b0 + b1 * zi + b2 * zi * zi) / (a0 + a1 * zi + a2 * zi * zi)
    return (20.0 * np.log10(np.abs(h))).astype(np.float64)


@pytest.mark.parametrize("kind", ["A", "C"])
@pytest.mark.parametrize("fs", RATES)
def test_closed_form_matches_scipy_bilinear(tables, kind, fs):
    sos = tables.iec61672_weighting_sos(kind, fs)
    assert sos.shape == (3 if kind == "A" else 2, 6)
    np.testing.assert_array_equal(sos[:, 3], 1.0)
    # numerators g [1, +-2, 1]: A has four zeros at z = 1 and two at z = -1, C two and two
    m = sos[:, 1] / sos[:, 0]
    np.testing.assert_array_equal(sos[:, 2], sos[:, 0])
    assert sorted(m) == ([-2.0, -2.0, 2.0] if kind == "A" else [-2.0, 2.0])
    # denominators: scipy's bilinear poles, paired f4 f4 | f2 f3 | f1 f1, and the whole cascade's polynomial
    z, p, k = signal.bilinear_zpk(*O.analog_zpk(kind), fs)
    order = np.argsort(p.real)                                         # f4, f4, (f3, f2,) f1, f1
    p = p.real[order]
    pairs = [(p[0], p[1]), (p[-3], p[-4]), (p[-2], p[-1])] if kind == "A" else [(p[0], p[1]), (p[2], p[3])]
    for sec, (ra, rb) in zip(sos, pairs):
        want = np.array([-(ra + rb), ra * rb])
        assert np.all(np.abs(sec[4:] - want) <= 1e-12 * np.abs(want).max()), (sec[4:], want)
    den = np.array([1.0])
    for sec in sos:
        den = np.convolve(den, sec[3:])
    ref = np.poly(p)
    assert np.abs(den - ref).max() <= 1e-12 * np.abs(ref).max()
    # magnitude at every nominal one-third-octave frequency below Nyquist, and |H(1 kHz)| = 1
    f = np.array([v for v in NOMINAL if v < fs / 2])
    d = np.abs(_mag_db(sos, f, fs) - _mag_db(O.weighting_sos(kind, fs), f, fs))
    assert d.max() <= 1e-9, d.max()
    _, h = signal.sosfreqz(sos, worN=[1000.0], fs=fs)
    assert abs(abs(h[0]) - 1.0) <= 1e-12


# deviation (dB) of the bilinear A design from the analog curve (DESIGN.md section 4.9)
DEVIATION_FREQS = (100, 4000, 8000, 10000, 12500, 16000, 20000)
DEVIATION_A = {44100: (-0.005, -0.045, -0.66, -1.50, -3.37, -8.53, -24.5),
               48000: (-0.004, -0.038, -0.54, -1.22, -2.67, -6.43, -15.8),
               96000: (-0.001, -0.009, -0.12, -0.26, -0.53, -1.11, -2.10)}


def _decimals(v):
    s = f"{abs(v)}"
    return len(s.split(".")[1]) if "." in s else 0


@pytest.mark.parametrize("kind", ["A", "C"])
@pytest.mark.parametrize("fs", sorted(DEVIATION_A))
def test_deviation_table(tables, kind, fs):
    """The table in DESIGN.md section 4.9 (A's values; C's are within 0.005 dB of them), to the rounding of its
    last digit.  At 100 Hz and below the deviation is within the first column's value."""
    sos = tables.iec61672_weighting_sos(kind, fs)
    dev = _mag_db(sos, DEVIATION_FREQS, fs) - O.analog_db(kind, DEVIATION_FREQS)
    for f, got, want in zip(DEVIATION_FREQS, dev, DEVIATION_A[fs]):
        half = 0.5 * 10.0 ** -_decimals(want)
        slack = 0.005 if kind == "C" else 0.0
        assert abs(got - want) <= half + slack + 1e-12, (kind, fs, f, got, want)
    low = np.geomspace(10, 100, 20)
    assert np.abs(_mag_db(sos, low, fs) - O.analog_db(kind, low)).max() <= abs(DEVIATION_A[fs][0]) + 0.0005 + (
        0.005 if kind == "C" else 0.0)


def _tone(f, amp, seconds, fs, silence=0.0):
    t = np.arange(int(seconds * fs)) / fs
    x = amp * np.sin(2 * np.pi * f * t)
    return np.concatenate([x, np.zeros(int(silence * fs))])[None, :]


@pytest.mark.parametrize("amp", [1.0, 0.1, 1e-3])
def test_sine_reads_its_amplitude(amp):
    fs = 48000
    r = O.sound_levels(_tone(1000.0, amp, 10.0, fs), fs)
    lv = r["levels"][0]
    want_eq, want_pk = 20 * np.log10(amp) - 10 * np.log10(2.0), 20 * np.log10(amp)
    for w in range(3):
        assert np.abs(lv[10:, w, 0] - want_eq).max() <= 0.01                 # Leq of every block after 1 s
        assert np.abs(lv[10:, w, 5] - want_pk).max() <= 0.01                 # Lpeak
        assert np.abs(lv[10:, w, 3] - want_eq).max() <= 0.01                 # LF after 8 tau
        assert np.abs(lv[80:, w, 4] - want_eq).max() <= 0.01                 # LS after 8 tau
        assert abs(r["totals"][0, w, 0] - want_eq) <= 0.01
    assert abs(want_eq - (20 * np.log10(amp) - 3.0103)) < 1e-4


def test_decay_rates():
    """After the tone stops, LF and LS fall at 10 log10(e) / tau: 34.7 and 4.34 dB/s."""
    fs = 48000
    r = O.sound_levels(_tone(1000.0, 0.5, 3.0, fs, silence=3.0), fs)
    lv = r["levels"][0, :, 0]
    for q, tau, j0, j1 in ((3, 0.125, 31, 36), (4, 1.0, 31, 59)):
        rate = -(lv[j1, q] - lv[j0, q]) / ((j1 - j0) / 10.0)
        want = 10 * np.log10(np.e) / tau
        assert abs(rate / want - 1.0) <= 0.01, (q, rate, want)


@pytest.mark.parametrize("burst_ms", [1000, 500, 200, 100, 50, 20, 10])
def test_tone_burst_response(burst_ms):
    """A 4 kHz burst of T_b after silence: LFmax - LF,steady and LSmax - LS,steady equal 10 log10(1 - e^(-T_b/tau))
    within 0.1 dB (LF,steady and LS,steady: the continuous tone's level)."""
    fs = 48000
    amp = 0.5
    x = np.zeros((1, 3 * fs))
    n_b = int(burst_ms * fs / 1000)
    t = np.arange(n_b) / fs
    x[0, fs:fs + n_b] = amp * np.sin(2 * np.pi * 4000.0 * t)
    r = O.sound_levels(x, fs)["totals"][0]
    steady = O.sound_levels(_tone(4000.0, amp, 8.0, fs), fs)["levels"][0, -1]
    for w in range(3):
        for q, tq, tau in ((1, 4, 0.125), (2, 4, 1.0)):
            ref = steady[w, 3 if tau < 1 else 4]
            want = 10 * np.log10(1.0 - np.exp(-burst_ms / 1000.0 / tau))
            assert abs((r[w, q] - ref) - want) <= 0.1, (w, burst_ms, tau, r[w, q] - ref, want)


def test_percentile_rule():
    v = np.array([[3.0, 1.0, 2.0, 2.0, -np.inf, 5.0]], np.float32)
    got = O.percentiles(v, [0, 10, 50, 90, 100])
    s = np.sort(v[0])                                          # -inf, 1, 2, 2, 3, 5
    assert got[0, 0] == 5.0 and got[0, -1] == -np.inf          # L0 the maximum, L100 the minimum (-inf lowest)
    assert got[0, 1] == s[int(np.floor(0.9 * 5 + 0.5))] == 5.0 and got[0, 2] == s[int(np.floor(0.5 * 5 + 0.5))]
    # N = 90: (1 - 0.9) * 5 + 0.5 is just below 1 in float64, so the rank is 0, not 1
    assert O.percentile_rank(90, 6) == 0 and got[0, 3] == s[0]
    assert np.isnan(O.percentiles(np.zeros((2, 0), np.float32), [10, 90])).all()           # n = 0
    np.testing.assert_array_equal(O.percentiles(np.array([[7.0]]), [0, 50, 100]), [[7.0, 7.0, 7.0]])   # n = 1
    np.testing.assert_array_equal(O.percentiles(np.array([[4.0, 1.0]]), [0, 49, 50, 51, 100]),
                                  [[4.0, 4.0, 4.0, 1.0, 1.0]])                              # n = 2: 50 rounds up
    np.testing.assert_array_equal(O.percentiles(np.full((1, 9), 2.5), [0, 33, 100]), [[2.5, 2.5, 2.5]])  # ties


def test_rate_rejection(tables):
    for fs in (44101, 7990, 200000, 48000.5, "x"):
        with pytest.raises(ValueError):
            tables.iec61672_weighting_sos("A", fs)
    with pytest.raises(ValueError):
        tables.iec61672_weighting_sos("Z", 48000)
    with pytest.raises(ValueError):
        O.sound_levels(np.zeros((1, 100)), 44105)


def test_python_side_rejects_bad_queries():
    from omega4_b200 import slm
    assert slm._column("A", "eq") == 0 and slm._column("Z", "peak") == 17 and slm._column("C", "F") == 9
    for bad in (("B", "F"), ("A", "I")):
        with pytest.raises(ValueError):
            slm._column(*bad)
    for bad in ([], [101], [-1], [np.nan], list(range(65))):
        with pytest.raises(ValueError):
            slm._pct(bad)
    with pytest.raises(ValueError):
        slm.sound_levels(np.zeros((2, 4800)), 48000)                # float64
