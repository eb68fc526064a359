"""CPU checks of the BS.1770-4 / EBU Tech 3341-3342 loudness definitions: the host K-weighting table and the
float64 oracle the GPU loudness path is tested against (EBU conformance cases synthesised as 1 kHz sines)."""
import numpy as np
import pytest

from omega4_b200 import tables
from oracle import bs1770_np as B

# BS.1770-4 Table 1 and Table 2 (48 kHz)
TABLE_48K = ([1.53512485958697, -2.69169618940638, 1.19839281085285],
             [1.0, -1.69065929318241, 0.73248077421585],
             [1.0, -2.0, 1.0],
             [1.0, -1.99004745483398, 0.99007225036621])


def tone(segments, fs=48000, n_ch=2, freq=1000.0):
    """1 kHz sine, each segment (dBFS of the peak amplitude, seconds), identical on n_ch channels -> [n_ch, n]."""
    parts = []
    for level, sec in segments:
        parts.append(np.full(int(round(sec * fs)), 10.0 ** (level / 20.0)))
    amp = np.concatenate(parts)
    x = amp * np.sin(2 * np.pi * freq * np.arange(amp.size) / fs)
    return np.repeat(x[None, :], n_ch, axis=0)


def test_k_weighting_table_48k():
    got = tables.bs1770_k_weighting(48000)
    for g, r in zip(got, TABLE_48K):
        np.testing.assert_allclose(g, r, rtol=0, atol=1e-12)


@pytest.mark.parametrize("fs", [44100, 48000, 96000])
def test_k_weighting_matches_oracle(fs):
    for g, r in zip(tables.bs1770_k_weighting(fs), B.k_weighting(fs)):
        np.testing.assert_allclose(g, r, rtol=0, atol=1e-15)


def test_layouts_and_weights():
    assert list(tables.bs1770_channel_weights("5.1")) == [1, 1, 1, 0, 1.41, 1.41]
    assert list(tables.bs1770_channel_weights("stereo", 2)) == [1, 1]
    assert "7.1" not in tables.BS1770_LAYOUTS
    for bad in ([1.0, np.nan], [-1.0], []):
        with pytest.raises(ValueError):
            tables.bs1770_channel_weights(bad)
    with pytest.raises(ValueError):
        tables.bs1770_channel_weights("stereo", 6)
    with pytest.raises(ValueError):
        tables.bs1770_channel_weights("7.1")


# (name, stereo 1 kHz segments (dBFS, seconds), what is checked, expected value)
CONFORMANCE = [
    ("3341-1", [(-23, 20)], "MSI", -23.0),
    ("3341-2", [(-33, 20)], "MSI", -33.0),
    ("3341-3", [(-36, 10), (-23, 60), (-36, 10)], "I", -23.0),
    ("3341-4", [(-72, 10), (-36, 10), (-23, 60), (-36, 10), (-72, 10)], "I", -23.0),
    ("3341-5", [(-26, 20), (-20, 20.1), (-26, 20)], "I", -23.0),
    ("3342-1", [(-20, 20), (-30, 20)], "LRA", 10.0),
    ("3342-2", [(-20, 20), (-15, 20)], "LRA", 5.0),
    ("3342-3", [(-40, 20), (-20, 20)], "LRA", 20.0),
    ("3342-4", [(-50, 20), (-35, 20), (-20, 20), (-35, 20), (-50, 20)], "LRA", 15.0),
]


def check_conformance(r, what, expected):
    if "M" in what:
        m = r["momentary"][~np.isnan(r["momentary"])]
        assert np.abs(m - expected).max() <= 0.1
    if "S" in what:
        s = r["short_term"][~np.isnan(r["short_term"])]
        assert np.abs(s - expected).max() <= 0.1
    if "I" in what:
        assert abs(r["integrated"] - expected) <= 0.1, r["integrated"]
    if what == "LRA":
        assert abs(r["lra"] - expected) <= 1.0, r["lra"]


@pytest.mark.parametrize("name,segments,what,expected", CONFORMANCE, ids=[c[0] for c in CONFORMANCE])
def test_oracle_ebu_conformance(name, segments, what, expected):
    r = B.stream_loudness(tone(segments), 48000, [1.0, 1.0])
    check_conformance(r, what, expected)


def tech3341_case6(fs=48000):
    """5.0: L, R at -28 dBFS, C at -24, Ls, Rs at -30, 20 s (weights 1, 1, 1, 1.41, 1.41)."""
    levels = [-28, -28, -24, -30, -30]
    return np.concatenate([tone([(lv, 20)], fs, 1) for lv in levels]), [1.0, 1.0, 1.0, 1.41, 1.41]


def test_oracle_ebu_3341_case6_five_channels():
    x, w = tech3341_case6()
    assert abs(B.stream_loudness(x, 48000, w)["integrated"] + 23.0) <= 0.1


def tech3341_case9(fs=48000):
    return tone([(-20, 1.34), (-30, 1.66)] * 5, fs)


def test_oracle_ebu_3341_case9_short_term():
    r = B.stream_loudness(tech3341_case9(), 48000, [1.0, 1.0])
    s = r["short_term"][29:]                         # S_j at the end of sub-block j, defined from 3 s on
    assert s.size > 100 and np.abs(s - (-23.0)).max() <= 0.1


def test_undefined_silent_and_steady_conventions():
    fs = 48000
    x = tone([(-20, 5)], fs)
    r = B.stream_loudness(x, fs, [1.0, 1.0])
    assert np.isnan(r["momentary"][:3]).all() and np.isfinite(r["momentary"][3:]).all()
    assert np.isnan(r["short_term"][:29]).all() and np.isfinite(r["short_term"][29:]).all()
    assert abs(r["lra"]) < 1e-9                        # a steady tone has no loudness range
    silent = np.zeros((2, 4 * fs))
    rs = B.stream_loudness(silent, fs, [1.0, 1.0])
    assert np.isneginf(rs["momentary"][3:]).all() and np.isneginf(rs["short_term"][29:]).all()
    assert np.isneginf(rs["integrated"]) and rs["lra"] == 0.0
    assert np.isneginf(rs["sample_peak"]).all() and rs["max_momentary"] == -np.inf
    short = B.stream_loudness(x[:, :fs // 5], fs, [1.0, 1.0])      # 200 ms: no momentary block yet
    assert np.isneginf(short["integrated"]) and np.isnan(short["max_momentary"])
    with pytest.raises(ValueError):
        B.subblock_energies(x, 44101, [1.0, 1.0])


def test_subblock_length_follows_sample_rate():
    for fs in (44100, 48000, 96000):
        x = tone([(-23, 1.0)], fs)
        assert B.subblock_energies(x, fs, [1.0, 1.0]).size == 10
