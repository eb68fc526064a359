"""Pin the numpy oracle (oracle/oracle_np.py) against fixtures produced by the UNMODIFIED
reference (oracle/gen_golden.py).  CPU only."""
import hashlib

import numpy as np
import pytest

from oracle import oracle_np as O

HOP, W = 512, 2048


# ---------------------------------------------------------------- windows / coefficients
@pytest.mark.parametrize("n", [2, 512, 1024, 2048, 8192])
def test_window_formulas_match_numpy(n):
    assert np.array_equal(O.np_blackman(n), np.blackman(n))
    assert np.array_equal(O.np_hamming(n), np.hamming(n))
    assert np.array_equal(O.np_hanning(n), np.hanning(n))


def test_kweighting_coefficients(golden):
    g = golden("meters_known.npz")
    c = O.k_weighting_coeffs(48000)
    for k in ("hp_b", "hp_a", "shelf_b", "shelf_a"):
        np.testing.assert_allclose(c[k], g[k], rtol=0, atol=2e-15)
    c96 = O.k_weighting_coeffs(96000)
    for k in ("hp_b", "hp_a", "shelf_b", "shelf_a"):
        np.testing.assert_allclose(c96[k], g[k + "96"], rtol=0, atol=2e-15)
    # SURVEY.md section 8 a12 probed values
    np.testing.assert_allclose(c["hp_a"], [1, -1.9929654642042134, 0.9929901199821451], atol=1e-14)
    np.testing.assert_allclose(c["shelf_a"], [1, -1.723776172762509, 0.7575469444788288], atol=1e-14)
    zi = O.lfilter_zi2(c["hp_b"], c["hp_a"])
    np.testing.assert_allclose(zi, [-c["hp_b"][0], c["hp_b"][0]], atol=1e-9)


def test_restated_iir_matches_scipy():
    sps = pytest.importorskip("scipy.signal")
    rng = np.random.default_rng(0)
    x = rng.standard_normal((3, 2048))
    c = O.k_weighting_coeffs(48000)
    for b, a in ((c["hp_b"], c["hp_a"]), (c["shelf_b"], c["shelf_a"])):
        np.testing.assert_allclose(O.lfilter_zi2(b, a), sps.lfilter_zi(b, a), atol=1e-10)
        np.testing.assert_allclose(O.filtfilt2(b, a, x), sps.filtfilt(b, a, x), rtol=0, atol=1e-11)
        bb, aa = sps.butter(2, (38.0 if b is c["hp_b"] else 1500.0) / 24000.0, btype="high")
        np.testing.assert_allclose(b, bb, atol=2e-15)
        np.testing.assert_allclose(a, aa, atol=2e-15)
    np.testing.assert_allclose(O.resample_fft(x, 4), sps.resample(x, 4 * 2048, axis=-1), atol=1e-12)
    sq = np.ones(480) * 0.9
    sq[::2] *= -1
    np.testing.assert_allclose(O.resample_fft(sq, 4), sps.resample(sq, 1920), atol=1e-12)


# ---------------------------------------------------------------- multi-resolution FFT
def _run_oracle_multires(x, sr, configs, T, keep=(), weighting=True):
    mr = O.OracleMultiResFFT(sr, 20000, configs)
    n_hops = len(x) // HOP
    comb = np.zeros((n_hops, T), np.float32)
    present = np.zeros((n_hops, len(mr.configs)), np.uint8)
    kept = {}
    for k in range(n_hops):
        res = mr.process_audio_chunk(x[k * HOP:(k + 1) * HOP], weighting)
        for i in res:
            present[k, i] = 1
        if res:
            comb[k] = mr.combine(res, T)[0]
        if k in keep:
            for i, m in res.items():
                kept[(k, i)] = m
    return comb, present, kept


def test_multires_baseline_sizes(golden):
    g = golden("multires_baseline.npz")
    keep = (0, 1, 3, 7, 15, 16, 50, 95)
    comb, present, kept = _run_oracle_multires(g["x"], 48000, O.BASELINE_CONFIGS, 512, keep)
    assert np.array_equal(present, g["present"])
    # readiness schedule: resolution N first appears at hop N/512 - 1
    assert [int(np.argmax(present[:, i])) for i in range(4)] == [15, 7, 3, 1]
    np.testing.assert_allclose(comb, g["combined"], rtol=2e-6, atol=1e-7)
    for (k, i), m in kept.items():
        ref = g[f"mag_h{k}_r{i}"]
        assert m.dtype == ref.dtype == np.float32
        np.testing.assert_allclose(m, ref, rtol=2e-6, atol=1e-6)
    comb_u, _, kept_u = _run_oracle_multires(g["x"], 48000, O.BASELINE_CONFIGS, 512, (50,), weighting=False)
    np.testing.assert_allclose(comb_u[50], g["combined_unweighted_h50"], rtol=2e-6, atol=1e-7)
    np.testing.assert_allclose(kept_u[(50, 0)], g["mag_h50_r0_unweighted"], rtol=2e-6, atol=1e-6)


def test_multires_default_config(golden):
    g = golden("multires_default.npz")
    comb, present, kept = _run_oracle_multires(g["x"], 48000, None, 1024, (6, 7, 47))
    assert np.array_equal(present, g["present"])
    np.testing.assert_allclose(comb, g["combined"], rtol=2e-6, atol=1e-7)
    for (k, i), m in kept.items():
        np.testing.assert_allclose(m, g[f"mag_h{k}_r{i}"], rtol=2e-6, atol=1e-6)


def test_multires_app_feed_oversize_chunks(golden):
    g = golden("multires_appfeed.npz")
    mr = O.OracleMultiResFFT(48000, 20000, None)
    for j, k in enumerate(range(3, 12)):
        res = mr.process_audio_chunk(g["frames"][j], True)
        assert sorted(res) == list(g[f"present_{k}"])
        np.testing.assert_allclose(mr.combine(res, 512)[0], g[f"combined_{k}"], rtol=2e-6, atol=1e-7)
        if k == 11:
            for i, m in res.items():
                np.testing.assert_allclose(m, g[f"mag_{k}_r{i}"], rtol=2e-6, atol=1e-6)


def test_multires_window_quirks(golden):
    g = golden("multires_windows.npz")
    wts = [str(w) for w in g["window_types"]]
    cfgs = [O.OracleFFTConfig(*c, window_type=wt) for c, wt in zip(O.BASELINE_CONFIGS, wts)]
    for i, c in enumerate(cfgs):
        assert np.array_equal(O.multires_window(c.window_type, c.fft_size), g[f"window_r{i}"])
    assert np.all(g["window_r0"] == 1.0)          # HANN -> np.hann missing -> rectangular
    x = golden("multires_baseline.npz")["x"][: int(g["n_samples"])]
    comb, _, kept = _run_oracle_multires(x, 48000, cfgs, 512, (23,))
    np.testing.assert_allclose(comb[23], g["combined_h23"], rtol=2e-6, atol=1e-7)
    for (k, i), m in kept.items():
        np.testing.assert_allclose(m, g[f"mag_h{k}_r{i}"], rtol=2e-6, atol=1e-6)


def test_multires_96k_six_resolutions(golden):
    g = golden("multires_96k.npz")
    cfgs = [(tuple(r), int(n), int(h), float(w)) for r, n, h, w in
            zip(g["cfg_ranges"], g["cfg_sizes"], g["cfg_hops"], g["cfg_weights"])]
    comb, present, kept = _run_oracle_multires(g["x"], 96000, cfgs, 512, (79,))
    assert np.array_equal(present, g["present"])
    np.testing.assert_allclose(comb[60:], g["combined_tail"], rtol=2e-6, atol=1e-7)
    for (k, i), m in kept.items():
        np.testing.assert_allclose(m, g[f"mag_h{k}_r{i}"], rtol=3e-6, atol=1e-5)


def test_combine_tables_reproduce_np_interp(golden):
    g = golden("multires_baseline.npz")
    mr = O.OracleMultiResFFT(48000, 20000, O.BASELINE_CONFIGS)
    tabs = O.combine_tables(48000, 20000, mr.configs, 512)
    assert [len(t[0]) for t in tabs] == [5, 20, 102, 384]      # SURVEY.md section 7 probe
    out = np.zeros(512)
    for i, (tidx, lo, frac) in enumerate(tabs):
        m = g[f"mag_h50_r{i}"].astype(np.float64)
        out[tidx] = m[lo] + (m[lo + 1] - m[lo]) * frac
    np.testing.assert_allclose(out, g["combined"][50], rtol=3e-6, atol=1e-7)


def test_ring_edge_cases():
    r = O.OracleRing(8)
    assert r.write(np.zeros(0)) is False and r.read_latest(4) is None
    r.write(np.arange(3, dtype=np.float32))
    assert r.read_latest(4) is None and r.read_latest(9) is None and r.read_latest(0) is None
    r.write(np.arange(3, 9, dtype=np.float32))                  # wraps
    assert list(r.read_latest(4)) == [5, 6, 7, 8]
    r.write(np.arange(100, 120, dtype=np.float32))             # oversize keeps the last 8
    assert list(r.read_latest(8)) == list(range(112, 120))
    with pytest.raises(ValueError):
        O.OracleFFTConfig((200, 100), 1024, 256, 1.0)
    with pytest.raises(ValueError):
        O.OracleFFTConfig((20, 200), 1000, 256, 1.0)
    with pytest.raises(ValueError):
        O.OracleMultiResFFT(48000, 30000)
    assert O.OracleMultiResFFT().process_audio_chunk(np.zeros(0)) == {}


# ---------------------------------------------------------------- batched FFT entry points
def test_batched_fft_entry_points(golden):
    g = golden("batched_fft.npz")
    for j, n in enumerate([16384, 4096, 2048, 2048, 1024]):
        r = O.batched_fft_cpu(g[f"in_{j}"], n)
        np.testing.assert_allclose(r["magnitude"], g[f"mag_{j}"], rtol=1e-5, atol=1e-4)
        np.testing.assert_allclose(r["complex"], g[f"cplx_{j}"], rtol=1e-5, atol=1e-4)
        assert np.array_equal(r["frequencies"], g[f"freq_{j}"])
        assert r["magnitude"].dtype == g[f"mag_{j}"].dtype
    for j, case in enumerate(g["w_cases"]):
        wt, ln, n = str(case).split(":")
        r = O.batched_fft_cpu(g[f"w_in_{j}"], int(n), wt)
        assert r["magnitude"].dtype == g[f"w_mag_{j}"].dtype == np.float64
        np.testing.assert_allclose(r["magnitude"], g[f"w_mag_{j}"], rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(r["complex"], g[f"w_cplx_{j}"], rtol=1e-12, atol=1e-12)
    r = O.batched_fft_cpu(g["app_in"], 2048)
    np.testing.assert_allclose(r["magnitude"], g["app_mag"], rtol=1e-12, atol=1e-13)
    for wt in ("hann", "hamming", "blackman"):
        mag, cplx = O.gpufft_compute_fft(g["g_in"], wt)
        np.testing.assert_allclose(mag, g[f"g_mag_{wt}"], rtol=1e-5, atol=1e-4)
        np.testing.assert_allclose(cplx, g[f"g_cplx_{wt}"], rtol=1e-5, atol=1e-4)
    np.testing.assert_allclose(O.gpufft_compute_fft(g["g_in_3000"], "hann")[0], g["g_mag_3000"], rtol=1e-5, atol=1e-4)
    m = O.gpufft_multi_resolution(g["gm_in"], {"bass": 8192, "mid": 4096, "high": 1024})
    for name in ("bass", "mid", "high"):
        np.testing.assert_allclose(m[name]["magnitude"], g[f"gm_mag_{name}"], rtol=1e-5, atol=1e-4)
        assert np.array_equal(m[name]["freqs"], g[f"gm_freqs_{name}"])


# ---------------------------------------------------------------- mel band mapping (bit exact)
KNOWN_HASHES = {  # SURVEY.md section 8 a9, sha256(int32 (start,end) array)[:16]
    "48000_2048_512": "9951968a2477a6eb", "48000_4096_512": "c2a393c27d5a0915",
    "48000_8192_512": "bc77c57968c01d00", "48000_1024_512": "82bb5527e0622094",
    "48000_4096_1024": "8e10536b9a9bb3bd", "96000_32768_512": "4d58d76d7eae1a5f",
}


def test_mel_band_indices_bit_exact(golden):
    g = golden("freq_mapper.npz")
    for combo in g["combos"]:
        combo = str(combo)
        sr, n, bars = (int(v) for v in combo.split("_"))
        bands = np.array(O.mel_band_indices(sr, n, bars), dtype=np.int32)
        assert np.array_equal(bands, g["bands_" + combo]), combo
        if combo in KNOWN_HASHES:
            assert hashlib.sha256(bands.tobytes()).hexdigest()[:16] == KNOWN_HASHES[combo]
        comp = O.compensation_curve(sr, n)
        np.testing.assert_allclose(comp, g["comp_" + combo], rtol=0, atol=1e-15)
        spec = g["spec_" + combo]
        blist = [tuple(b) for b in bands]
        np.testing.assert_allclose(O.map_spectrum_to_bars(spec, blist, bars, comp), g["bars_comp_" + combo], rtol=1e-6)
        np.testing.assert_allclose(O.map_spectrum_to_bars(spec, blist, bars, None), g["bars_raw_" + combo], rtol=1e-6)
        np.testing.assert_allclose(O.map_spectrum_to_bars(spec[:512], blist, bars, comp), g["bars_short_" + combo], rtol=1e-6)


# ---------------------------------------------------------------- meters
def test_meters_known_answers(golden):
    g = golden("meters_known.npz")
    m = O.OracleMetering(48000)
    r = m.calculate_lufs(g["sine_frame"])
    assert abs(r["momentary"] - float(g["sine_momentary"])) < 1e-9
    assert abs(r["true_peak"] - float(g["sine_true_peak"])) < 1e-9
    assert abs(r["momentary"] - (-16.491558806111666)) < 1e-6      # SURVEY.md section 8c probe (float32 sine there)
    assert abs(r["true_peak"] - (-6.020850533752008)) < 1e-6
    c = O.k_weighting_coeffs(48000)
    for name in ("sq480", "sq2048"):
        x = g[name]
        assert abs(float(O.true_peak_db(x[None])[0]) - float(g[name + "_tp"])) < 1e-9
        assert abs(float(O.lufs_instantaneous(x[None], c)[0]) - float(g[name + "_lufs"])) < 1e-9
    assert float(O.true_peak_db(np.zeros((1, W)))[0]) == float(g["zeros_tp"]) == -100.0
    assert float(O.lufs_instantaneous(np.zeros((1, W)), c)[0]) == float(g["zeros_lufs"]) == -100.0


def test_meters_stream_schedule(golden):
    g = golden("meters_stream.npz")
    x = g["x"]
    first, frames = O.meter_frames(x, HOP, W)
    assert first == int(g["first_hop"]) == 3
    c = O.k_weighting_coeffs(48000)
    inst = O.lufs_instantaneous(frames, c)
    tp = O.true_peak_db(frames)
    np.testing.assert_allclose(inst, g["lufs_inst"], rtol=0, atol=1e-9)
    np.testing.assert_allclose(tp, g["tp_db"], rtol=0, atol=1e-9)
    for k in (10, 44, 65, 85):
        np.testing.assert_allclose(O.apply_k_weighting(frames[k - first][None], c)[0], g[f"kweighted_h{k}"],
                                   rtol=0, atol=1e-12)
    assert np.all(inst[44 - first:46 - first] == -100.0)           # digital silence -> rms gate
    assert tp.max() > 0.0                                          # hot section crosses 0 dBTP
    st = O.OracleMeterStats()
    rows = np.array([(lambda d: [d[k] for k in O.METER_KEYS])(st.push(a, b)) for a, b in zip(inst, tp)])
    np.testing.assert_allclose(rows, g["meters"], rtol=0, atol=1e-9)
    full = O.analyze_channel(x, 48000, O.BASELINE_CONFIGS)
    np.testing.assert_allclose(full["meters"][first:], g["meters"], rtol=0, atol=1e-9)
    assert np.all(full["meters"][:first] == [-100, -100, -100, 0, -100])


def test_meters_long_statistics(golden):
    g = golden("meters_stats.npz")
    base, gains = g["base"], g["gains"]
    c = O.k_weighting_coeffs(48000)
    frames = gains[:, None] * base[np.arange(len(gains)) % 4]
    inst = np.concatenate([O.lufs_instantaneous(frames[s:s + 600], c) for s in range(0, len(frames), 600)])
    tp = np.concatenate([O.true_peak_db(frames[s:s + 600]) for s in range(0, len(frames), 600)])
    np.testing.assert_allclose(inst, g["lufs_inst"], rtol=0, atol=1e-9)
    np.testing.assert_allclose(tp, g["tp_db"], rtol=0, atol=1e-9)
    st = O.OracleMeterStats()
    rows = np.array([(lambda d: [d[k] for k in O.METER_KEYS])(st.push(a, b)) for a, b in zip(inst, tp)])
    np.testing.assert_allclose(rows, g["meters"], rtol=0, atol=1e-9)
    assert len(st.integ) == 3600                                   # the 60 s deque saturated
    assert (g["lufs_inst"] <= -70).sum() > 100                     # gate exercised


def test_ref_port_matches_oracle(golden):
    """The per-hop scipy-based port that bench.py times as the CPU baseline is the same function
    as the batched oracle (and therefore as the reference goldens)."""
    pytest.importorskip("scipy.signal")
    from oracle import ref_port
    g = golden("meters_stream.npz")
    x = g["x"][:60 * HOP]
    comb, meters = ref_port.run_channel(x)
    ref = O.analyze_channel(x, 48000, O.BASELINE_CONFIGS)
    np.testing.assert_allclose(comb, ref["combined"], rtol=2e-6, atol=1e-7)
    np.testing.assert_allclose(meters, ref["meters"], rtol=0, atol=1e-8)
    np.testing.assert_allclose(meters[3:], g["meters"][:57], rtol=0, atol=1e-8)
    r = ref_port.time_cpu_path(2, 2, 0.25, processes=2)
    assert r["value"] > 0 and r["cores"] == 2


# ---------------------------------------------------------------- section 8f rank 1: app post-processing
@pytest.mark.parametrize("variant,kw", [
    ("default", {}),
    ("normalized", {"normalization": True}),
    ("vocal", {"content_type": "vocal", "vocal_suppression": 0.5}),
    ("plain", {"freq_compensation": False, "smoothing": False}),
])
def test_app_post_processing_matches_reference_block(golden, variant, kw):
    """oracle OracleSpectrumPost vs omega4_main.py:992-1056 executed unmodified (gen_golden_next.py)."""
    g = golden("app_post.npz")
    cols = g["band_cols"]                                          # the fixture stores these of the 437 bands
    post = O.OracleSpectrumPost(512, **kw)
    assert np.array_equal(np.array(post.bands, dtype=np.int32), g["bands"])
    assert post.n_valid(512) == 437 and g["band_" + variant].shape == (len(g["combined"]), len(cols))
    for k, row in enumerate(g["combined"]):
        band, peak = post.process(row)
        np.testing.assert_allclose(peak[cols], g["peak_" + variant][k], rtol=0, atol=1.2e-7)
        np.testing.assert_allclose(band[cols], g["band_" + variant][k], rtol=0, atol=2.4e-7)
    assert float(g["band_default"].max()) == 1.0 and float(g["band_default"].min()) == 0.0


# ---------------------------------------------------------------- section 8f rank 2: A / C / Z weighting
def test_a_c_weighting_coefficients_and_frames(golden):
    """oracle closed-form Butterworth sections and apply_weighting vs the unmodified reference."""
    g = golden("meters_weighting.npz")
    for name, (b, a) in zip(("hp1", "hp2", "lp1", "lp2"), O.a_weighting_sections(48000)):
        np.testing.assert_allclose(b, g[f"A_{name}_b"], rtol=0, atol=3e-15)
        np.testing.assert_allclose(a, g[f"A_{name}_a"], rtol=0, atol=3e-15)
    for name, (b, a) in zip(("hp", "lp"), O.c_weighting_sections(48000)):
        np.testing.assert_allclose(b, g[f"C_{name}_b"], rtol=0, atol=3e-15)
        np.testing.assert_allclose(a, g[f"C_{name}_a"], rtol=0, atol=3e-15)
    x = g["x"]
    hops = list(g["weighted_hops"])
    frames = np.stack([x[(k + 1) * HOP - W:(k + 1) * HOP] * np.hanning(W) for k in range(3, len(x) // HOP)])
    for mode in ("A", "C", "Z"):
        w = O.apply_weighting(frames[[k - 3 for k in hops]], mode)
        assert np.abs(w - g[f"weighted_{mode}"]).max() <= 1e-11, mode
        li = O.lufs_instantaneous_mode(frames, mode)
        assert np.abs(li - g[f"lufs_inst_{mode}"]).max() <= 1e-9, mode
    # frames with rms < 1e-6 weigh to zeros in A and C (:158-160, :197-199) but pass through in Z
    quiet = frames[:1] * 1e-7
    assert np.all(O.apply_weighting(quiet, "A") == 0) and np.all(O.apply_weighting(quiet, "C") == 0)
    assert np.array_equal(O.apply_weighting(quiet, "Z"), quiet)


def test_restated_first_order_filtfilt_matches_scipy():
    sps = pytest.importorskip("scipy.signal")
    rng = np.random.default_rng(4)
    x = rng.standard_normal((2, 2048))
    for b, a in O.a_weighting_sections(48000):
        np.testing.assert_allclose(O.filtfilt_any(b, a, x), sps.filtfilt(b, a, x), rtol=0, atol=1e-9)   # 20.6 Hz poles: 1e-11 round-off


# ---------------------------------------------------------------- section 8f rank 3: bass zoom panel data side
def test_bass_zoom_bars_match_reference(golden):
    g = golden("bass_zoom.npz")
    ranges, groups = O.bass_mapping(48000)
    assert len(groups) == int(g["n_bars"]) == 31
    assert np.array_equal([x[0] for x in groups], g["bin_first"]) and np.array_equal([len(x) for x in groups], g["bin_count"])
    np.testing.assert_allclose(np.array(ranges), g["ranges"], rtol=0, atol=1e-12)
    bars = np.zeros(len(groups), np.float32)
    for fr, want in zip(g["frames"], g["bars"]):
        bars = O.bass_bars_step(fr.astype(np.float64), bars, ranges, groups)
        np.testing.assert_allclose(bars, want, rtol=0, atol=1e-7)


# ------------------------------------------------------------------ round 2 fixtures (oracle/gen_golden_r2.py)
def test_meters_96k_eight_channels(golden):
    """BASELINE configs[4] shape for the meters: ProfessionalMetering(96000) on 8 channels of s16le audio."""
    g = golden("meters_96k.npz")
    assert int(g["sample_rate"]) == 96000
    c = O.k_weighting_coeffs(96000)
    for k in ("hp_b", "hp_a", "shelf_b", "shelf_a"):
        np.testing.assert_allclose(c[k], g[k], rtol=0, atol=3e-15)
    x = g["x16"].astype(np.float32) / 32768.0                       # capture.py:574
    assert x.shape[0] == 8
    for ch in range(8):
        first, frames = O.meter_frames(x[ch], HOP, W)
        assert first == int(g["first_hop"])
        inst = O.lufs_instantaneous(frames, c)
        tp = O.true_peak_db(frames)
        np.testing.assert_allclose(inst, g["lufs_inst"][ch], rtol=0, atol=2e-9)
        np.testing.assert_allclose(tp, g["tp_db"][ch], rtol=0, atol=1e-9)
        np.testing.assert_allclose(O.apply_k_weighting(frames[40 - first][None], c)[0], g[f"kweighted_c{ch}_h40"],
                                   rtol=0, atol=1e-12)
        full = O.analyze_channel(x[ch], 96000, O.BASELINE_CONFIGS)
        np.testing.assert_allclose(full["meters"][first:], g["meters"][ch], rtol=0, atol=2e-9)
    assert np.all(g["lufs_inst"][1][23 - 3:30 - 3] == -100.0)       # digital silence -> rms gate
    assert g["tp_db"][2].max() > 0.0                                # the hot channel crosses 0 dBTP
    assert g["meters"][4][:, 2].max() == -100.0                     # a few LSB: never above the -70 gate


def test_waterfall_matches_reference(golden):
    g = golden("waterfall.npz")
    assert O.waterfall_freq_indices(48000, 2048) == tuple(g["freq_indices"])
    assert O.waterfall_freq_indices(96000, 4096) == tuple(g["freq_indices_96k_4096"])
    assert O.waterfall_freq_indices(22050, 1024) == tuple(g["freq_indices_22k_1024"])
    for tag, auto, gain in (("auto", True, 0.0), ("fixed", False, 0.0), ("auto_gain3", True, 3.0)):
        wf = O.OracleWaterfall(48000, 2048)
        wf.auto_gain, wf.gain_adjustment = auto, gain
        for k, spec in enumerate(g["spectra"]):
            row = wf.update(spec)
            # the reference works in float32: dB values up to 200 in magnitude carry ~1.5e-5 of rounding
            assert abs(wf.current_peak - g[f"peak_{tag}"][k]) < 1e-4 and abs(wf.current_floor - g[f"floor_{tag}"][k]) < 1e-4
            np.testing.assert_allclose(row, g[f"rows_{tag}"][k], rtol=0, atol=2e-6)
    assert O.OracleWaterfall().update(np.zeros(0)) is None
    np.testing.assert_allclose(O.magnitude_to_db_plus(g["spectra"][:8]), g["plugin_db"], rtol=0, atol=2e-5)


def test_multires_96k_adversarial_stream(golden):
    """Six resolutions up to 32768 at 96 kHz on a click / silence / full-scale-tone stream."""
    g = golden("multires_96k_stress.npz")
    cfgs = [(c[0], c[1], c[2], c[3]) for c in O.CONFIG5_96K]
    comb, present, kept = _run_oracle_multires(g["x"], 96000, cfgs, 512, (75, 130, 149))
    f0 = int(g["combined_first"])
    np.testing.assert_allclose(comb[f0:, :32], g["combined_low"], rtol=3e-6, atol=1e-9)
    for k in (75, 130, 149):
        np.testing.assert_allclose(comb[k], g[f"combined_h{k}"], rtol=3e-6, atol=1e-9)
        for i in (0, 1):
            np.testing.assert_allclose(kept[(k, i)][:64], g[f"mag_h{k}_r{i}"], rtol=3e-6, atol=1e-7)
