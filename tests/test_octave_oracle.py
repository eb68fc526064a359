"""CPU checks of the one-third-octave band definitions: the host band table and closed-form Butterworth
band-pass sections (omega4_b200.tables) against scipy's own design, and the float64 oracle the GPU band-level
path is tested against (oracle/octave_np.py)."""
import numpy as np
import pytest
from scipy import signal

from omega4_b200 import tables
from oracle import octave_np as O

RATES = [8000, 44100, 48000, 96000]
BAND_COUNT = {8000: 23, 44100: 30, 48000: 31, 96000: 31, 192000: 31}


@pytest.mark.parametrize("fs", RATES + [192000])
def test_band_table(fs):
    b = tables.third_octave_bands(fs)
    n = BAND_COUNT[fs]
    assert b["fm"].size == n and list(b["x"]) == list(range(-17, -17 + n))
    np.testing.assert_allclose(b["fm"], 1000.0 * 10.0 ** (0.1 * b["x"]), rtol=1e-15)
    np.testing.assert_allclose(b["f1"] * b["f2"], b["fm"] ** 2, rtol=1e-14)
    np.testing.assert_allclose(b["f2"] / b["f1"], 10.0 ** 0.1, rtol=1e-14)
    assert (b["f2"] < fs / 2).all()
    r = O.bands(fs)                    # restated independently in the oracle
    for k in ("x", "fm", "f1", "f2", "nominal"):
        np.testing.assert_allclose(b[k], r[k], rtol=1e-15)


def test_nominal_labels():
    b = tables.third_octave_bands(48000)
    assert list(b["nominal"]) == [20, 25, 31.5, 40, 50, 63, 80, 100, 125, 160, 200, 250, 315, 400, 500, 630, 800,
                                  1000, 1250, 1600, 2000, 2500, 3150, 4000, 5000, 6300, 8000, 10000, 12500, 16000,
                                  20000]
    # the nominal label is the exact mid-band frequency rounded as IEC 61260-1 Annex E rounds it (within 3 %)
    assert (np.abs(b["nominal"] / b["fm"] - 1.0) < 0.03).all()
    assert list(tables.third_octave_bands(44100)["nominal"])[-1] == 16000
    assert list(tables.third_octave_bands(8000)["nominal"])[-1] == 3150


def _magnitude_db(k, n_plus, n_minus, poles, w):
    """|H(e^jw)| in dB from (gain, zeros at z = 1 and z = -1, poles), with |e^jw - 1| = 2 sin(w / 2) and
    |e^jw + 1| = 2 cos(w / 2) evaluated directly (a polynomial evaluation near z = 1 would cancel)."""
    e = np.exp(1j * w)[:, None]
    mag = abs(k) * (2 * np.sin(w / 2)) ** n_plus * (2 * np.cos(w / 2)) ** n_minus / np.prod(np.abs(e - poles[None]), 1)
    return 20 * np.log10(mag)


def _sos_poles(sos):
    """Poles of each section's z^2 + a1 z + a2 in closed form (complex pairs; np.roots is less accurate here)."""
    re = -sos[:, 4] / 2
    im = np.sqrt(sos[:, 5] - re * re)
    return np.concatenate([re + 1j * im, re - 1j * im])


def _sos_zero_counts(sos):
    """(zeros at z = 1, zeros at z = -1) of sections whose numerators are g [1, -2, 1], g [1, 2, 1] or g [1, 0, -1]."""
    plus = minus = 0
    for b0, b1, b2 in sos[:, :3]:
        if b1 == -2 * b0 and b2 == b0:
            plus += 2
        elif b1 == 2 * b0 and b2 == b0:
            minus += 2
        else:
            assert b1 == 0 and b2 == -b0, (b0, b1, b2)
            plus, minus = plus + 1, minus + 1
    return plus, minus


@pytest.mark.parametrize("fs", RATES + [192000])
def test_sos_matches_scipy_butter(fs):
    """The closed form designs the filter scipy.signal.butter(3, [f1, f2], "bandpass", fs=fs, output="sos")
    designs: magnitude within 1e-9 dB wherever above -120 dB on a dense log grid, poles within 1e-12 of
    scipy's zpk design.  Magnitudes come from the poles, the gain and the zeros at z = +-1 (a polynomial
    evaluation near z = 1 would itself lose ~1e-6 dB deep in the stop band)."""
    b = tables.third_octave_bands(fs)
    sos = tables.third_octave_sos(fs)
    assert sos.shape == (b["fm"].size, 3, 6) and sos.dtype == np.float64
    w = 2 * np.pi * np.geomspace(1.0, 0.999 * fs / 2, 6000) / fs
    worst_db = worst_pole = 0.0
    for i in range(sos.shape[0]):
        s = sos[i]
        assert (s[:, 3] == 1.0).all() and (s[:, 1] == 0.0).all() and (s[:, 2] == -s[:, 0]).all()   # g [1, 0, -1]
        sref = signal.butter(3, [b["f1"][i], b["f2"][i]], btype="bandpass", fs=fs, output="sos")
        assert _sos_zero_counts(sref) == (3, 3)
        ref = _magnitude_db(np.prod(sref[:, 0]), 3, 3, _sos_poles(sref), w)
        got = _magnitude_db(np.prod(s[:, 0]), 3, 3, _sos_poles(s), w)
        sel = ref > -120.0
        worst_db = max(worst_db, float(np.abs(got - ref)[sel].max()))
        z, p, k = signal.butter(3, [b["f1"][i], b["f2"][i]], btype="bandpass", fs=fs, output="zpk")
        assert sorted(z.real) == [-1, -1, -1, 1, 1, 1]
        mine = _sos_poles(s)                          # nearest-neighbour match: both are three conjugate pairs
        worst_pole = max(worst_pole, max(float(np.abs(mine - q).min()) for q in p))
    assert worst_db <= 1e-9, worst_db
    assert worst_pole <= 1e-12, worst_pole


@pytest.mark.parametrize("fs", RATES + [192000])
def test_edges_are_minus_3_db(fs):
    b = tables.third_octave_bands(fs)
    sos = tables.third_octave_sos(fs)
    for i in range(sos.shape[0]):
        _, h = signal.sosfreqz(sos[i], worN=[b["f1"][i], b["f2"][i], b["fm"][i]], fs=fs)
        db = 20 * np.log10(np.abs(h))
        assert np.abs(db[:2] + 10 * np.log10(2)).max() < 1e-7, (i, db)
        assert abs(db[2]) < 0.0044, (i, db)


@pytest.mark.parametrize("fs", [44100, 48000, 96000])
def test_oracle_tone_reads_its_amplitude(fs):
    """A sine of amplitude A at each f_m reads 20 log10 A in its own band: the energy mean of the 100 ms blocks
    after 2 s (a single block of a 20 Hz sine ripples by up to 0.19 dB: it holds two periods)."""
    b = O.bands(fs)
    t = np.arange(6 * fs) / fs
    amps = np.geomspace(1e-3, 0.9, b["fm"].size)
    x = np.stack([a * np.sin(2 * np.pi * f * t) for a, f in zip(amps, b["fm"])])
    r = O.band_levels(x, fs)
    for i, a in enumerate(amps):
        blocks = r["levels"][i, 20:, i]
        got = 10 * np.log10(np.mean(10.0 ** (blocks / 10)))
        assert abs(got - 20 * np.log10(a)) <= 0.01, (i, got, 20 * np.log10(a))
        # the band owns the tone: its neighbours read at least 10 dB lower
        for j in (i - 1, i + 1):
            if 0 <= j < b["fm"].size:
                assert r["leq"][i, j] < r["leq"][i, i] - 10.0
    # the overall column of a sine of amplitude A reads 20 log10 A over whole periods of the slowest tone
    assert abs(r["leq"][-1, -1] - 20 * np.log10(amps[-1])) < 1e-3


def test_oracle_silence_reads_minus_inf():
    r = O.band_levels(np.zeros((2, 48000 + 123), np.float32), 48000)
    for k in ("levels", "leq", "max_level"):
        assert np.isneginf(r[k]).all(), k
    assert r["levels"].shape == (2, 10, 32)
    x = np.zeros((1, 9600))
    x[0, 5000] = 0.5                                     # an impulse in block 1: block 0 stays silent
    r = O.band_levels(x, 48000)
    assert np.isneginf(r["levels"][0, 0]).all() and np.isfinite(r["levels"][0, 1]).all()
    assert np.isfinite(r["leq"]).all() and np.isfinite(r["max_level"]).all()


@pytest.mark.parametrize("fs", [0, 7990, 44101, 48000.5, 192010, 200000, -48000])
def test_bad_rates_raise(fs):
    with pytest.raises(ValueError):
        tables.third_octave_bands(fs)
    with pytest.raises(ValueError):
        tables.third_octave_sos(fs)
    with pytest.raises(ValueError):
        O.bands(fs)
