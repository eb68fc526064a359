"""GPU parity tests: the CUDA path (through the C ABI / the reference-shaped shims) against the
golden fixtures frozen from the unmodified reference and against the numpy oracle.

North-star tolerances (BASELINE.json): band-bin indices bit-exact, spectrum within 0.01 dB,
LUFS within 0.01 LU, true peak within 0.05 dBTP.  The asserted bounds below are those; the
measured errors are ~1e-4 dB / 1e-6 LU / 1e-5 dBTP (profiles/parity_r01.txt).
"""
import hashlib

import os

import numpy as np
import pytest

from conftest import assert_spectrum_close
from oracle import oracle_np as O

pytestmark = pytest.mark.gpu

TOL_DB = 0.01      # spectrum, dB
TOL_LU = 0.01      # LUFS
TOL_TP = 0.05      # dBTP
HOP, W = 512, 2048


@pytest.fixture(scope="module")
def plan():
    from omega4_b200.plan import AnalysisPlan, BASELINE_CONFIGS
    p = AnalysisPlan(48000, BASELINE_CONFIGS, 512)
    yield p
    p.close()


def _meters_close(got, ref, label=""):
    d = np.abs(np.asarray(got, np.float64) - np.asarray(ref, np.float64))
    assert d[..., :4].max() <= TOL_LU, f"{label} LUFS columns off by {d[..., :4].max(axis=tuple(range(d.ndim - 1)))}"
    assert d[..., 4].max() <= TOL_TP, f"{label} true peak off by {d[..., 4].max()}"


# ------------------------------------------------------------------ FFT primitive
@pytest.mark.parametrize("n", [512, 1024, 2048, 4096, 8192, 16384, 32768])
def test_rfft_batch_against_float64(n):
    from omega4_b200.plan import rfft_batch_host
    rng = np.random.default_rng(n)
    x = rng.standard_normal((7, n)).astype(np.float32)
    x[1] = 0.0                                           # all-zero frame
    x[2] = np.sin(2 * np.pi * 1000 * np.arange(n) / 48000)
    w = np.blackman(n).astype(np.float32)
    mag, cx = rfft_batch_host(x, w)
    ref = np.fft.rfft(x.astype(np.float64) * w, axis=1)
    scale = np.abs(ref).max(axis=1, keepdims=True) + 1e-30
    assert (np.abs(cx - ref) / scale).max() < 2e-6
    assert (np.abs(mag - np.abs(ref)) / scale).max() < 2e-6
    assert np.all(mag[1] == 0) and cx.dtype == np.complex64 and mag.shape == (7, n // 2 + 1)
    assert_spectrum_close(mag, np.abs(ref), TOL_DB, label=f"rfft {n}")
    mag2, none = rfft_batch_host(x, None, want_complex=False)       # rectangular window, magnitude only
    assert none is None
    assert_spectrum_close(mag2, np.abs(np.fft.rfft(x.astype(np.float64), axis=1)), TOL_DB)


def test_rfft_batch_rejects_unsupported_sizes():
    from omega4_b200 import Omega4CudaError
    from omega4_b200.plan import rfft_batch_host
    for n in (256, 3000, 65536):
        with pytest.raises(Omega4CudaError):
            rfft_batch_host(np.zeros((1, n), np.float32), None)


# ------------------------------------------------------------------ multi-resolution + combine
def test_multires_baseline_golden(plan, golden):
    g = golden("multires_baseline.npz")
    out = plan.analyze_host(g["x"][None, :], want_combined=True, want_magnitudes=True, want_meters=False)
    comb = out["combined"][0]
    assert comb.shape == g["combined"].shape
    assert np.array_equal(comb == 0, g["combined"] == 0)            # readiness schedule + orphan bin 0
    assert_spectrum_close(comb, g["combined"], TOL_DB, label="combined")
    for k in (0, 1, 3, 7, 15, 16, 50, 95):
        for r in range(4):
            key = f"mag_h{k}_r{r}"
            if key in g.files:
                assert_spectrum_close(out["magnitudes"][r][0, k], g[key], TOL_DB, label=key)
            else:
                assert np.all(out["magnitudes"][r][0, k] == 0)      # resolution not filled yet


def test_multires_unweighted(golden):
    from omega4_b200.plan import AnalysisPlan, BASELINE_CONFIGS
    g = golden("multires_baseline.npz")
    p = AnalysisPlan(48000, BASELINE_CONFIGS, 512, apply_weighting=False)
    out = p.analyze_host(g["x"][None, :], want_magnitudes=True, want_meters=False)
    assert_spectrum_close(out["combined"][0, 50], g["combined_unweighted_h50"], TOL_DB)
    assert_spectrum_close(out["magnitudes"][0][0, 50], g["mag_h50_r0_unweighted"], TOL_DB)
    p.close()


def test_multires_default_config_general_combine(golden):
    """Reference default (4096/2048/1024/1024, T=1024): ranges touch at 5000 Hz -> still disjoint
    on this grid; also run the general (CSR) combine on the returned magnitudes."""
    from omega4_b200.plan import AnalysisPlan, DEFAULT_CONFIGS
    g = golden("multires_default.npz")
    p = AnalysisPlan(48000, DEFAULT_CONFIGS, 1024)
    out = p.analyze_host(g["x"][None, :], want_magnitudes=True, want_meters=False)
    assert np.array_equal(out["combined"][0] == 0, g["combined"] == 0)
    assert_spectrum_close(out["combined"][0], g["combined"], TOL_DB, label="default combined")
    for k in (6, 7, 47):
        for r in range(4):
            key = f"mag_h{k}_r{r}"
            if key in g.files:
                assert_spectrum_close(out["magnitudes"][r][0, k], g[key], TOL_DB, label=key)
    rows = [m[0, 47:48] for m in out["magnitudes"]]
    again = p.combine_host(rows, 1)[0]
    assert_spectrum_close(again, g["combined"][47], TOL_DB, label="combine_host")
    partial = p.combine_host([None, rows[1], None, rows[3]], 1)[0]      # absent resolutions
    mr = O.OracleMultiResFFT(48000, 20000, None)
    ref = mr.combine({1: rows[1][0], 3: rows[3][0]}, 1024)[0]
    assert_spectrum_close(partial, ref, TOL_DB, label="partial combine")
    assert np.array_equal(partial == 0, ref == 0)
    p.close()


def test_multires_overlapping_ranges_use_general_path():
    """freq_ranges that overlap (two resolutions feed the same target bins): the fused epilogue is
    not applicable, the library falls back to magnitudes + CSR combine ON THE GPU."""
    from omega4_b200.plan import AnalysisPlan
    from omega4_b200.batch.synth import synth_channel
    cfg = [((20, 600), 4096, 512, 1.5, "blackman"), ((200, 3000), 2048, 512, 1.2, "hamming"),
           ((1000, 20000), 1024, 256, 1.0, "blackman")]
    x = synth_channel(7, 0, 24 * HOP)
    p = AnalysisPlan(48000, cfg, 512)
    out = p.analyze_host(x[None, :], want_meters=False)
    mr = O.OracleMultiResFFT(48000, 20000, [(c[0], c[1], c[2], c[3], c[4]) for c in cfg])
    for k in range(24):
        res = mr.process_audio_chunk(x[k * HOP:(k + 1) * HOP])
        ref = mr.combine(res, 512)[0] if res else np.zeros(512)
        assert_spectrum_close(out["combined"][0, k], ref, TOL_DB, label=f"overlap hop {k}")
    p.close()


def test_multires_window_quirks(golden):
    from omega4_b200.plan import AnalysisPlan, BASELINE_CONFIGS
    g = golden("multires_windows.npz")
    wts = [str(w) for w in g["window_types"]]
    cfg = [(c[0], c[1], c[2], c[3], wt) for c, wt in zip(BASELINE_CONFIGS, wts)]
    p = AnalysisPlan(48000, cfg, 512)
    for i in range(4):
        assert np.array_equal(p.windows[i], g[f"window_r{i}"])
    x = golden("multires_baseline.npz")["x"][: int(g["n_samples"])]
    out = p.analyze_host(x[None, :], want_magnitudes=True, want_meters=False)
    assert_spectrum_close(out["combined"][0, 23], g["combined_h23"], TOL_DB)
    for r in range(4):
        assert_spectrum_close(out["magnitudes"][r][0, 23], g[f"mag_h23_r{r}"], TOL_DB)
    p.close()


def test_multires_96k_six_resolutions(golden):
    from omega4_b200.plan import AnalysisPlan
    g = golden("multires_96k.npz")
    cfg = [(tuple(r), int(n), int(h), float(w), "blackman") for r, n, h, w in
           zip(g["cfg_ranges"], g["cfg_sizes"], g["cfg_hops"], g["cfg_weights"])]
    p = AnalysisPlan(96000, cfg, 512)
    out = p.analyze_host(g["x"][None, :], want_magnitudes=True, want_meters=False)
    assert_spectrum_close(out["combined"][0, 60:], g["combined_tail"], TOL_DB, label="96k combined")
    for r in range(6):
        assert_spectrum_close(out["magnitudes"][r][0, 79], g[f"mag_h79_r{r}"], TOL_DB, label=f"96k r{r}")
    present = (out["magnitudes"][0][0].max(axis=1) > 0)
    assert int(np.argmax(present)) == 63                              # 32768/512 - 1
    p.close()


# ------------------------------------------------------------------ hop-block partial DFT (fused, few-bin resolutions)
def _kernel_names(plan):
    return [n for n, _ in plan.kernel_times()]


def test_blockdft_path_matches_golden_and_full_fft(plan, golden):
    """Fused output only (no magnitudes): N = 8192 feeds 5 target bins from 10 FFT bins and N = 4096
    feeds 20 from 40, so the library evaluates them as hop-block partial DFTs -- by default as one
    3xTF32 tcgen05 GEMM (blockdft_tc_kernel.cuh), with OMEGA4_FLAG_NO_TENSOR as the fp32 CUDA-core GEMM
    for the 8192 alone (blockdft_kernel.cuh).  Same golden vectors; the full-FFT evaluation of the same
    call (OMEGA4_FLAG_NO_BLOCKDFT) must agree."""
    from omega4_b200 import _native as N
    g = golden("multires_baseline.npz")
    full = plan.analyze_host(g["x"][None, :], want_meters=False, flags=N.FLAG_TIME_KERNELS | N.FLAG_NO_BLOCKDFT)
    names = _kernel_names(plan)
    assert "multires_fft_8192" in names and not any(n.startswith("blockdft") for n in names)
    fullc = full["combined"][0]
    scale = fullc.max(axis=1, keepdims=True) + 1e-20
    for flags, want, absent in ((0, ("blockdft_tc_gemm", "blockdft_asm_8192", "blockdft_asm_4096"),
                                 ("multires_fft_8192", "multires_fft_4096", "blockdft_gemm")),
                                (N.FLAG_NO_TENSOR, ("blockdft_gemm", "blockdft_asm_8192", "multires_fft_4096"),
                                 ("multires_fft_8192", "blockdft_tc_gemm", "blockdft_asm_4096"))):
        out = plan.analyze_host(g["x"][None, :], want_meters=False, flags=N.FLAG_TIME_KERNELS | flags)
        names = _kernel_names(plan)
        assert all(w in names for w in want) and not any(a in names for a in absent), names
        comb = out["combined"][0]
        assert np.array_equal(comb == 0, g["combined"] == 0)
        assert_spectrum_close(comb, g["combined"], TOL_DB, label=f"blockdft flags={flags}")
        assert np.array_equal(fullc == 0, comb == 0)
        assert (np.abs(fullc - comb) / scale).max() < (2e-6 if flags else 2e-5)
        assert np.array_equal(fullc[:, 26:], comb[:, 26:])                  # 2048 / 1024 resolutions untouched


def test_blockdft_strong_tone_next_to_weak_content():
    """Worst case for the split-precision tensor-core GEMM: a full-scale 1 kHz tone leaking into the
    sparse low bins, which hold a tone 50 dB below it; float64 reference."""
    from omega4_b200 import _native as N
    from omega4_b200.plan import AnalysisPlan, BASELINE_CONFIGS
    n = 40 * HOP
    t = np.arange(n) / 48000.0
    x = (0.9 * np.sin(2 * np.pi * 1000.0 * t) + 0.9 * 10 ** (-50 / 20) * np.sin(2 * np.pi * 97.0 * t + 0.3)).astype(np.float32)
    mr = O.OracleMultiResFFT(48000, 20000, list(O.BASELINE_CONFIGS))
    for k in range(40):
        res = mr.process_audio_chunk(x[k * HOP:(k + 1) * HOP])
    # float64 evaluation of the same last frame
    ref64 = {}
    for i, c in enumerate(mr.configs):
        fr = x[n - c.fft_size:].astype(np.float64) * mr.windows[i].astype(np.float64)
        ref64[i] = (np.abs(np.fft.rfft(fr)) * mr.bin_weights(i)).astype(np.float64)
    want = mr.combine({i: v.astype(np.float32) for i, v in ref64.items()}, 512)[0]
    p = AnalysisPlan(48000, BASELINE_CONFIGS, 512)
    for flags in (0, N.FLAG_NO_TENSOR, N.FLAG_NO_BLOCKDFT):
        got = p.analyze_host(x[None, :], want_meters=False, flags=flags)["combined"][0, 39]
        assert_spectrum_close(got, want, TOL_DB, label=f"strong tone flags={flags}")
    p.close()


def test_blockdft_96k_default_and_window_variants(golden):
    from omega4_b200 import _native as N
    from omega4_b200.plan import AnalysisPlan, BASELINE_CONFIGS, DEFAULT_CONFIGS
    # 96 kHz, six resolutions: 32768 and 16384 share one GEMM
    g = golden("multires_96k.npz")
    cfg = [(tuple(r), int(n), int(h), float(w), "blackman") for r, n, h, w in
           zip(g["cfg_ranges"], g["cfg_sizes"], g["cfg_hops"], g["cfg_weights"])]
    p = AnalysisPlan(96000, cfg, 512)
    out = p.analyze_host(g["x"][None, :], want_meters=False, flags=N.FLAG_TIME_KERNELS)
    names = _kernel_names(p)
    assert "blockdft_asm_32768" in names and "blockdft_asm_16384" in names and "multires_fft_32768" not in names
    assert "blockdft_tc_gemm" in names
    assert_spectrum_close(out["combined"][0, 60:], g["combined_tail"], TOL_DB, label="96k blockdft")
    assert np.array_equal(out["combined"][0, 60:] == 0, g["combined_tail"] == 0)
    p.close()
    # reference default sizes, T = 1024: 4096 feeds 10 target bins from 20 FFT bins = 200 GEMM columns,
    # more than the FFT costs -> stays on the FFT kernel; T = 512 halves that and qualifies
    g = golden("multires_default.npz")
    p = AnalysisPlan(48000, DEFAULT_CONFIGS, 1024)
    out = p.analyze_host(g["x"][None, :], want_meters=False, flags=N.FLAG_TIME_KERNELS)
    assert "blockdft_gemm" not in _kernel_names(p) and "blockdft_tc_gemm" in _kernel_names(p)   # 200 columns: tensor cores only
    assert np.array_equal(out["combined"][0] == 0, g["combined"] == 0)
    assert_spectrum_close(out["combined"][0], g["combined"], TOL_DB, label="default blockdft")
    p.close()
    # rectangular ('hann' quirk) and hamming windows are cosine sums too
    g = golden("multires_windows.npz")
    wts = [str(w) for w in g["window_types"]]
    cfg = [(c[0], c[1], c[2], c[3], wt) for c, wt in zip(BASELINE_CONFIGS, wts)]
    x = golden("multires_baseline.npz")["x"][: int(g["n_samples"])]
    p = AnalysisPlan(48000, cfg, 512)
    for fl in (0, N.FLAG_NO_TENSOR):
        out = p.analyze_host(x[None, :], want_meters=False, flags=N.FLAG_TIME_KERNELS | fl)
        assert ("blockdft_gemm" if fl else "blockdft_tc_gemm") in _kernel_names(p)
        assert_spectrum_close(out["combined"][0, 23], g["combined_h23"], TOL_DB, label="window variants blockdft")
    p.close()
    # a window that is NOT a cosine sum: the exact-windowing operand (default) carries any window; the
    # cosine-sum formulation (OMEGA4_BLOCKDFT_FD=1) keeps the FFT path for it
    rng = np.random.default_rng(5)
    wins = [np.blackman(c[1]).astype(np.float32) for c in BASELINE_CONFIGS]
    wins[0] = (wins[0] * (1 + 0.01 * rng.standard_normal(8192))).astype(np.float32)
    mr = O.OracleMultiResFFT(48000, 20000, list(O.BASELINE_CONFIGS))
    mr.windows[0] = wins[0]
    for k in range(24):
        res = mr.process_audio_chunk(x[k * HOP:(k + 1) * HOP])
    want = mr.combine(res, 512)[0]
    for fd in (False, True):
        if fd:
            os.environ["OMEGA4_BLOCKDFT_FD"] = "1"
        try:
            p = AnalysisPlan(48000, BASELINE_CONFIGS, 512, windows=wins)
            out = p.analyze_host(x[None, :], want_meters=False, flags=N.FLAG_TIME_KERNELS)
            names = _kernel_names(p)
            if fd:
                assert "multires_fft_8192" in names and "blockdft_asm_8192" not in names and "blockdft_asm_4096" in names
            else:
                assert "blockdft_asm_8192" in names and "multires_fft_8192" not in names
            assert_spectrum_close(out["combined"][0, 23], want, TOL_DB, label="custom window")
            p.close()
        finally:
            os.environ.pop("OMEGA4_BLOCKDFT_FD", None)


def test_alternate_kernel_paths_stay_covered(golden):
    """The developer knobs select kernels the default path no longer runs: the float64-state K-weighting kernel in
    batch mode (OMEGA4_KW_F64=1) and the unfused frame assembly of the exact-windowing GEMM
    (OMEGA4_BLOCKDFT_UNFUSED=1, blockdft_sum_kernel).  Both must agree with the default path and the fixtures."""
    from omega4_b200 import _native as N
    from omega4_b200.plan import AnalysisPlan, BASELINE_CONFIGS
    g = golden("multires_baseline.npz")
    x = g["x"][None, : 120 * HOP]
    p = AnalysisPlan(48000, BASELINE_CONFIGS, 512)
    base = p.analyze_host(x, want_series=True, flags=N.FLAG_TIME_KERNELS)
    os.environ["OMEGA4_KW_F64"] = "1"
    try:
        f64 = p.analyze_host(x, want_series=True)
    finally:
        os.environ.pop("OMEGA4_KW_F64", None)
    m = np.isfinite(base["lufs_inst"][0]) & (base["lufs_inst"][0] > -99)
    assert m.sum() > 50
    assert np.abs(f64["lufs_inst"][0][m] - base["lufs_inst"][0][m]).max() < 2e-5      # float32 vs float64 state
    assert np.array_equal(f64["combined"], base["combined"])
    p.close()
    os.environ["OMEGA4_BLOCKDFT_UNFUSED"] = "1"
    try:
        p2 = AnalysisPlan(48000, BASELINE_CONFIGS, 512)
        unf = p2.analyze_host(x, want_meters=False, flags=N.FLAG_TIME_KERNELS)
        assert "blockdft_asm_8192" in _kernel_names(p2) and "blockdft_tc_gemm" in _kernel_names(p2)
        p2.close()
    finally:
        os.environ.pop("OMEGA4_BLOCKDFT_UNFUSED", None)
    # same GEMM, same additions in a different order: equal to float32 rounding of the frame sums
    scale = base["combined"][0].max(axis=1, keepdims=True) + 1e-20
    assert (np.abs(unf["combined"][0] - base["combined"][0]) / scale).max() < 2e-6


# ------------------------------------------------------------------ section 8f rank 1: app post-processing
TOL_BAR = 1e-5     # band_values live in [0, 1]; 0.01 dB on the spectrum is 5.8e-4 relative on a sqrt'd bar


def test_app_post_processing_golden_and_state():
    """omega4_bars_run vs omega4_main.py:992-1056 executed unmodified (tests/golden/app_post.npz)."""
    from omega4_b200.app.spectrum_post import SpectrumPostProcessor
    g = np.load(__import__("os").path.join(__import__("conftest").GOLDEN, "app_post.npz"))
    comb = g["combined"]
    cols = g["band_cols"]                                 # the fixture stores these of the 437 bands
    variants = {"default": {}, "normalized": {"normalization_enabled": True},
                "vocal": {"current_content_type": "vocal", "vocal_suppression": 0.5},
                "plain": {"freq_compensation_enabled": False, "smoothing_enabled": False}}
    for name, attrs in variants.items():
        post = SpectrumPostProcessor(512)
        for k, v in attrs.items():
            setattr(post, k, v)
        band, peak = post.process_host(comb[None], want_peaks=True)
        assert band.shape == (1, len(comb), 437)
        assert np.abs(peak[0][:, cols] - g["peak_" + name]).max() <= TOL_BAR, name
        assert np.abs(band[0][:, cols] - g["band_" + name]).max() <= TOL_BAR, name
        post.close()
    # frame-at-a-time (the application's call pattern, prev_band_values carried on the object)
    post = SpectrumPostProcessor(512)
    for k in range(20):
        b, p = post.process(comb[k])
        assert np.abs(b[cols] - g["band_default"][k]).max() <= TOL_BAR and np.abs(p[cols] - g["peak_default"][k]).max() <= TOL_BAR
    assert np.array_equal(post.prev_band_values, b)
    # tiles with carried state == one shot; channels independent
    one = post.process_host(np.stack([comb, comb[::-1]]))
    state = np.zeros((2, 1 + post.n_valid), np.float32)
    parts = [post.process_host(np.stack([comb, comb[::-1]])[:, s:s + 13], state=state) for s in range(0, len(comb), 13)]
    assert np.array_equal(np.concatenate(parts, axis=1), one)
    assert np.abs(one[0][:, cols] - g["band_default"]).max() <= TOL_BAR
    post.close()


def test_app_post_processing_long_rows_use_segments():
    """More than 512 hops per channel: the kernel cuts the rows into segments that rebuild the smoothing
    state by replaying the 128 rows before them -- identical to the sequential recurrence to 1e-9."""
    from omega4_b200.app.spectrum_post import SpectrumPostProcessor
    rng = np.random.default_rng(8)
    spec = np.abs(rng.standard_normal((2, 1300, 512))).astype(np.float32) * np.linspace(2.0, 0.01, 512, dtype=np.float32)
    spec[1, 600:640] = 0.0
    post = SpectrumPostProcessor(512)
    state = np.zeros((2, 1 + 437), np.float32)
    got = post.process_host(spec, state=state)
    for ch in range(2):
        ref = O.OracleSpectrumPost(512)
        want = np.stack([ref.process(row)[0] for row in spec[ch]])
        assert np.abs(got[ch] - want).max() <= TOL_BAR
        assert np.abs(state[ch, 1:] - want[-1]).max() <= TOL_BAR and state[ch, 0] == 1.0
    post.close()


def test_app_post_processing_resident_batch_against_oracle(plan):
    """Device-resident chain: analyze -> combined -> band_values, against the numpy oracle."""
    import torch
    from omega4_b200.app.spectrum_post import SpectrumPostProcessor
    from omega4_b200.batch.driver import analyze_resident
    from omega4_b200.batch.synth import synth_streams
    n_hops = 70
    x = synth_streams(2, 2, n_hops * HOP).reshape(4, -1)
    comb = torch.empty((4, n_hops, 512), device="cuda")
    analyze_resident(plan, torch.from_numpy(x).cuda(), combined=comb)
    post = SpectrumPostProcessor(512)
    post._ensure()
    bars = torch.empty((4, n_hops, post.n_valid), device="cuda")
    post.process_device(comb, bars)
    torch.cuda.synchronize()
    got = bars.cpu().numpy()
    c = comb.cpu().numpy()
    for ch in (0, 3):
        ref = O.OracleSpectrumPost(512)
        want = np.stack([ref.process(row)[0] for row in c[ch]])
        assert np.abs(got[ch] - want).max() <= TOL_BAR
    post.close()


# ------------------------------------------------------------------ section 8f rank 4: s16le wire format
def test_s16_interleaved_input_is_bit_identical_to_float_path(plan):
    """capture.py:571-574 decodes s16le as int16.astype(float32) / 32768 -- exact in float32, so the
    int16 entry point must reproduce the float32 entry point bit for bit (mono, stereo, 7.1)."""
    import torch
    rng = np.random.default_rng(21)
    n_hops = 40
    for il, n_streams in ((1, 3), (2, 2), (8, 1)):
        pcm = rng.integers(-32768, 32768, size=(n_streams, n_hops * HOP, il), dtype=np.int16)
        pcm[0, 5 * HOP:9 * HOP] = 0                                       # digital silence
        planar = (pcm.astype(np.float32) / 32768.0).transpose(0, 2, 1).reshape(n_streams * il, -1)
        ref = plan.analyze_host(planar)
        got = plan.analyze_s16_host(pcm)
        assert np.array_equal(got["combined"], ref["combined"]) and np.array_equal(got["meters"], ref["meters"])
        # device-resident int16, with carried history: second half of the clip as a tile
        d = torch.from_numpy(pcm.reshape(n_streams, -1)).cuda()
        comb = torch.empty((n_streams * il, n_hops, 512), device="cuda")
        met = torch.empty((n_streams * il, n_hops, 5), device="cuda")
        plan.analyze_s16_device(d, n_hops, il, combined=comb, meters=met)
        torch.cuda.synchronize()
        assert np.array_equal(comb.cpu().numpy(), ref["combined"]) and np.array_equal(met.cpu().numpy(), ref["meters"])
        h = 20
        tail = plan.analyze_s16_host(pcm, hist_frames=h * HOP, want_meters=False)
        assert np.array_equal(tail["combined"], plan.analyze_host(planar, hist_samples=h * HOP, want_meters=False)["combined"])
        assert np.array_equal(tail["combined"], ref["combined"][:, h:])      # 20 hops of history cover every window


def test_s16_decode_matches_capture_formula():
    rng = np.random.default_rng(2)
    pcm = rng.integers(-32768, 32768, size=4096, dtype=np.int16)
    want = np.frombuffer(pcm.tobytes(), dtype=np.int16).astype(np.float32) / 32768.0      # capture.py:574
    assert np.array_equal(want, pcm.astype(np.float32) * np.float32(1.0 / 32768.0))


def test_blockdft_edge_shapes_match_full_fft(plan):
    """Short inputs (fewer hops than the longest window has blocks), odd channel counts, padded row
    strides and carried history: the hop-block paths must agree with the full-FFT evaluation."""
    import torch
    from omega4_b200 import _native as N
    from omega4_b200.batch.synth import synth_streams
    for n_ch, n_hops in ((1, 1), (3, 3), (5, 15), (5, 16), (2, 17), (7, 300)):
        x = synth_streams(n_ch, 1, n_hops * HOP).reshape(n_ch, -1)
        ref = plan.analyze_host(x, want_meters=False, flags=N.FLAG_NO_BLOCKDFT)["combined"]
        scale = ref.max(axis=-1, keepdims=True) + 1e-20
        for fl in (0, N.FLAG_NO_TENSOR):
            got = plan.analyze_host(x, want_meters=False, flags=fl)["combined"]
            assert np.array_equal(got == 0, ref == 0), (n_ch, n_hops, fl)
            assert (np.abs(got - ref) / scale).max() < 2e-5, (n_ch, n_hops, fl)
    # padded row stride + history carried in front of the rows (device pointers)
    n_hops, hist = 40, 7680
    x = synth_streams(3, 1, hist + n_hops * HOP).reshape(3, -1)
    buf = torch.zeros((3, hist + n_hops * HOP + 64), device="cuda")
    buf[:, :x.shape[1]] = torch.from_numpy(x).cuda()
    outs = []
    for fl in (0, N.FLAG_NO_TENSOR, N.FLAG_NO_BLOCKDFT):
        comb = torch.empty((3, n_hops, 512), device="cuda")
        plan.analyze_device(buf, n_hops, hist_samples=hist, combined=comb, flags=fl)
        torch.cuda.synchronize()
        outs.append(comb.cpu().numpy())
    whole = plan.analyze_host(x, want_meters=False, flags=N.FLAG_NO_BLOCKDFT)["combined"][:, hist // HOP:]
    assert np.array_equal(outs[2], whole)                               # same frames, same FFT path: identical
    scale = whole.max(axis=-1, keepdims=True) + 1e-20
    assert (np.abs(outs[0] - whole) / scale).max() < 2e-5 and (np.abs(outs[1] - whole) / scale).max() < 2e-6
    assert np.all(outs[0][:, 0, 1:6] > 0)                                # the 8192 window is already full at hop 0


def test_new_entry_points_reject_bad_arguments(plan):
    import ctypes as C
    from omega4_b200 import _native as N, Omega4CudaError
    from omega4_b200.app.spectrum_post import SpectrumPostProcessor
    lib = N.lib()
    w = N.Weighting()
    w.n_sections = 5
    assert lib.omega4_plan_set_weighting(plan.handle, C.byref(w)) == -1
    w.n_sections = 1; w.order[0] = 3
    assert lib.omega4_plan_set_weighting(plan.handle, C.byref(w)) == -3
    w.order[0] = 2; w.blend = 1
    for j, v in enumerate((1.0, -1.9, 0.95)):
        w.a[0][j] = v; w.b[0][j] = v
    assert lib.omega4_plan_set_weighting(plan.handle, C.byref(w)) == -1          # blend needs two sections
    assert lib.omega4_plan_set_weighting(plan.handle, None) == 0                 # NULL restores K
    assert plan.analyze_s16_host(np.zeros((0, 512, 2), np.int16))["n_hops"] == 1
    assert plan.analyze_s16_host(np.zeros((2, 100), np.int16)).get("combined") is None   # less than one hop
    assert lib.omega4_analyze_s16(plan.handle, None, N.MEM_HOST, None, 0, 1, 2, 1, 0, None, None, None, None, None, None, 0) == -1
    post = SpectrumPostProcessor(512)
    with pytest.raises(Omega4CudaError):
        post.process(np.zeros(100, np.float32))
    d = N.BarsDesc()
    d.spectrum_len, d.n_bars = 512, 0
    assert not lib.omega4_bars_create(C.byref(d), 0) and b"bad bars descriptor" in lib.omega4_last_error()
    post.close()


# ------------------------------------------------------------------ section 8f rank 3: bass zoom panel data side
def test_bass_zoom_panel_golden(golden):
    """BassZoomPanel._process_bass_detail_internal (bass_zoom.py:141-214): Hann + zero-padded 8192-point
    rFFT (omega4_rfft_batch) and bar mean / compensation / dynamic scaling / compression / smoothing
    (omega4_bass_bars) against the reference's own bar values."""
    from omega4_b200.panels.bass_zoom import BassZoomPanel
    g = golden("bass_zoom.npz")
    p = BassZoomPanel(48000)
    assert p.bass_detail_bars == int(g["n_bars"]) and [x[0] for x in p.bass_bin_mapping] == list(g["bin_first"])
    np.testing.assert_allclose(np.array(p.bass_freq_ranges), g["ranges"], rtol=0, atol=1e-12)
    for k, (fr, want) in enumerate(zip(g["frames"], g["bars"])):           # frame at a time, state on the object
        p.update(fr)
        assert np.abs(p.bass_bar_values - want).max() <= TOL_BAR, k
    assert np.all(p.bass_peak_values >= p.bass_bar_values - 1e-6)
    # batch: all frames in one call, two channels (second one reversed in time), carried state
    frames = np.stack([g["frames"], g["frames"][::-1]])
    one = p.bar_values_batch(frames)
    assert np.abs(one[0] - g["bars"]).max() <= TOL_BAR
    state = np.zeros((2, p.bass_detail_bars), np.float32)
    parts = [p.bar_values_batch(frames[:, s:s + 10], state) for s in range(0, frames.shape[1], 10)]
    assert np.array_equal(np.concatenate(parts, axis=1), one)
    ranges, groups = O.bass_mapping(48000)
    bars = np.zeros(len(groups), np.float32)
    for j, fr in enumerate(frames[1]):
        bars = O.bass_bars_step(fr.astype(np.float64), bars, ranges, groups)
        assert np.abs(one[1, j] - bars).max() <= TOL_BAR


# ------------------------------------------------------------------ meters
def test_meters_stream_golden(plan, golden):
    g = golden("meters_stream.npz")
    out = plan.analyze_host(g["x"][None, :], want_combined=False, want_meters=True, want_series=True)
    f = int(g["first_hop"])
    assert np.abs(out["lufs_inst"][0, f:] - g["lufs_inst"]).max() <= TOL_LU
    assert np.abs(out["tp_db"][0, f:] - g["tp_db"]).max() <= TOL_TP
    _meters_close(out["meters"][0, f:], g["meters"], "stream")
    assert np.all(out["meters"][0, :f] == [-100, -100, -100, 0, -100])
    # much tighter than the gate in practice; the batch path evaluates the delayed true-peak phases in half precision
    # (truepeak16_kernel.cuh: ~0.01 dBTP), OMEGA4_FLAG_EXACT_TRUE_PEAK keeps them in float32
    assert np.abs(out["lufs_inst"][0, f:] - g["lufs_inst"]).max() < 1e-5
    assert np.abs(out["tp_db"][0, f:] - g["tp_db"]).max() < 0.03
    from omega4_b200 import _native as N
    ex = plan.analyze_host(g["x"][None, :], want_combined=False, want_meters=True, want_series=True, flags=N.FLAG_EXACT_TRUE_PEAK)
    assert np.abs(ex["tp_db"][0, f:] - g["tp_db"]).max() < 1e-3
    assert np.array_equal(ex["lufs_inst"], out["lufs_inst"])
    assert np.all(out["lufs_inst"][0, 44:46] == -100.0)               # digital silence -> rms gate


def test_meter_frames_and_long_statistics(plan, golden):
    from omega4_b200 import _native as N
    g = golden("meters_stats.npz")
    frames = g["gains"][:, None] * g["base"][np.arange(len(g["gains"])) % 4]
    li, tp, _ = plan.meter_frames_host(frames)
    assert np.abs(li - g["lufs_inst"]).max() <= TOL_LU and np.abs(tp - g["tp_db"]).max() <= TOL_TP
    assert np.abs(li - g["lufs_inst"]).max() < 1e-5
    state = np.zeros((1, N.METER_STATE_DOUBLES))
    m = plan.meter_stats_host(li, tp, state=state, fresh=True)[0]
    _meters_close(m, g["meters"], "long stats")
    assert int(state[0, 0]) == 3600 and int(state[0, 1]) == 60       # both windows saturated
    # tiled with carried state == one shot
    state = np.zeros((1, N.METER_STATE_DOUBLES))
    parts = [plan.meter_stats_host(li[s:s + 997], tp[s:s + 997], state=state, fresh=(s == 0))[0]
             for s in range(0, len(li), 997)]
    assert np.array_equal(np.concatenate(parts), m)


def test_meters_known_answers(plan, golden):
    g = golden("meters_known.npz")
    li, tp, w = plan.meter_frames_host(np.stack([g["sine_frame"], g["sq2048"], np.zeros(W)]), want_weighted=True)
    assert abs(li[0] - float(g["sine_momentary"])) <= 1e-5 and abs(tp[0] - float(g["sine_true_peak"])) <= 1e-3
    assert abs(li[1] - float(g["sq2048_lufs"])) <= 1e-5 and abs(tp[1] - float(g["sq2048_tp"])) <= 1e-3
    assert li[2] == -100.0 and tp[2] == -100.0 and np.all(w[2] == 0)
    c = O.k_weighting_coeffs(48000)
    ref = O.apply_k_weighting(np.stack([g["sine_frame"], g["sq2048"]]), c)
    assert np.abs(w[:2] - ref).max() < 1e-7


# ------------------------------------------------------------------ section 8f rank 2: A / C / Z weighting
@pytest.mark.parametrize("mode", ["A", "C", "Z"])
def test_meter_weighting_modes_golden(golden, mode):
    """ProfessionalMetering with weighting_mode A / C / Z (professional_meters.py:74-127, 155-229):
    cascades of first/second-order filtfilt sections through the same block-scan kernel."""
    from omega4_b200.panels.professional_meters import ProfessionalMetering
    from omega4_b200.plan import AnalysisPlan, BASELINE_CONFIGS
    g = golden("meters_weighting.npz")
    x = g["x"]
    m = ProfessionalMetering(48000)
    m.weighting_mode = mode
    hops = list(g["weighted_hops"])
    for k in range(3, len(x) // HOP):
        frame = x[(k + 1) * HOP - W:(k + 1) * HOP] * np.hanning(W)
        if k in hops:
            w = m.apply_weighting(frame)
            ref = g[f"weighted_{mode}"][hops.index(k)]
            assert np.abs(w - ref).max() <= 1e-7 * max(1.0, np.abs(ref).max()), (mode, k)
        d = m.calculate_lufs(frame)
        assert abs(m.lufs_momentary_history[-1] - g[f"lufs_inst_{mode}"][k - 3]) <= 1e-5, (mode, k)
        _meters_close([d[key] for key in O.METER_KEYS], g[f"meters_{mode}"][k - 3], f"{mode} hop {k}")
    quiet = x[:W] * np.hanning(W) * 1e-7                                 # rms gate: zeros in A / C, identity in Z
    wq = m.apply_weighting(quiet)
    assert np.array_equal(wq, quiet) if mode == "Z" else np.all(wq == 0)
    # the batch path with the plan switched to the same mode
    p = AnalysisPlan(48000, BASELINE_CONFIGS, 512)
    p.set_weighting(mode)
    out = p.analyze_host(x[None, :], want_combined=False, want_series=True)
    assert np.abs(out["lufs_inst"][0, 3:] - g[f"lufs_inst_{mode}"]).max() <= 1e-5
    _meters_close(out["meters"][0, 3:], g[f"meters_{mode}"], f"batch {mode}")
    p.set_weighting("K")
    k_out = p.analyze_host(x[None, :], want_combined=False, want_series=True)
    ref = O.analyze_channel(x, 48000, O.BASELINE_CONFIGS)
    assert np.abs(k_out["lufs_inst"][0, 3:] - ref["lufs_inst"][3:]).max() <= 1e-5        # back to K
    p.close()


# ------------------------------------------------------------------ reference-shaped shims
def test_shim_multires_chunks_and_appfeed(golden):
    from omega4_b200.audio.multi_resolution_fft import MultiResolutionFFT, FFTConfig, FFTResult, WindowType
    g = golden("multires_default.npz")
    mr = MultiResolutionFFT(48000)
    x = g["x"]
    for k in range(12):
        res = mr.process_audio_chunk(x[k * HOP:(k + 1) * HOP])
        assert sorted(res) == [i for i in range(4) if g["present"][k, i]]
        if res:
            comb, freqs = mr.combine_results_optimized(res, target_bins=1024)
            assert comb.dtype == np.float32 and freqs.dtype == np.float64 and len(freqs) == 1024
            assert_spectrum_close(comb, g["combined"][k], TOL_DB, label=f"shim hop {k}")
        for i, r in res.items():
            assert isinstance(r, FFTResult) and r.config_index == i and r.magnitude.dtype == np.float32
            if f"mag_h{k}_r{i}" in g.files:
                assert_spectrum_close(r.magnitude, g[f"mag_h{k}_r{i}"], TOL_DB)
    assert mr.process_audio_chunk(np.zeros(0)) == {} and mr.process_audio_chunk(None) == {}
    z, f = mr.combine_results_optimized({}, 64)
    assert z.dtype == np.float64 and np.all(z == 0) and len(f) == 64
    st = mr.get_processing_stats()
    assert st["total_calls"] == 12 and st["error_count"] == 0 and "avg_time_ms" in st
    mr.reset_all_buffers()
    assert mr.process_audio_chunk(x[:HOP]) == {}
    # app feed: 2048-sample Hann-windowed float64 frames -> oversize path of the 1024 rings
    ga = golden("multires_appfeed.npz")
    mr2 = MultiResolutionFFT(48000)
    for j, k in enumerate(range(3, 12)):
        res = mr2.process_audio_chunk(ga["frames"][j])
        assert sorted(res) == list(ga[f"present_{k}"])
        assert_spectrum_close(mr2.combine_results_optimized(res, 512)[0], ga[f"combined_{k}"], TOL_DB)
    # overwrite .configs and re-run the setup methods, the way the reference's users do
    gb = golden("multires_baseline.npz")
    mr3 = MultiResolutionFFT(48000)
    mr3.configs = [FFTConfig(fr, n, h, w, WindowType.BLACKMAN) for fr, n, h, w in O.BASELINE_CONFIGS]
    mr3._setup_windows(); mr3._setup_buffers(); mr3._setup_frequency_arrays(); mr3._setup_working_arrays()
    for k in range(17):
        res = mr3.process_audio_chunk(gb["x"][k * HOP:(k + 1) * HOP])
    assert sorted(res) == [0, 1, 2, 3]
    assert_spectrum_close(mr3.combine_results_optimized(res, 512)[0], gb["combined"][16], TOL_DB)
    with pytest.raises(ValueError):
        MultiResolutionFFT(48000, 30000)
    with pytest.raises(ValueError):
        FFTConfig((20, 200), 1000, 256, 1.0)


def test_shim_batched_and_gpu_fft(golden):
    from omega4_b200.optimization.batched_fft_processor import BatchedFFTProcessor, get_batched_fft_processor
    from omega4_b200.optimization.gpu_accelerated_fft import GPUAcceleratedFFT
    g = golden("batched_fft.npz")
    proc = BatchedFFTProcessor()
    ids = [proc.prepare_batch(f"panel{j}", g[f"in_{j}"], n) for j, n in enumerate([16384, 4096, 2048, 2048, 1024])]
    assert proc.process_batch() == 5
    res = proc.distribute_results()
    for j, rid in enumerate(ids):
        assert_spectrum_close(res[rid]["magnitude"], g[f"mag_{j}"], TOL_DB, label=f"batched {j}")
        scale = np.abs(g[f"cplx_{j}"]).max()
        assert np.abs(res[rid]["complex"] - g[f"cplx_{j}"]).max() / scale < 2e-6
        assert np.array_equal(res[rid]["frequencies"], g[f"freq_{j}"])
    assert proc.process_batch() == 0 and proc.distribute_results() == {}
    for j, case in enumerate(g["w_cases"]):
        wt, ln, n = str(case).split(":")
        rid = proc.prepare_batch("w", g[f"w_in_{j}"], int(n), wt)
        assert proc.process_batch() == 1
        r = proc.get_result_for_panel(rid)
        assert_spectrum_close(r["magnitude"], g[f"w_mag_{j}"], TOL_DB, label=str(case))
        assert proc.get_result_for_panel(rid) is None
    rid = proc.prepare_batch("main_spectrum", g["app_in"], 2048)          # the app's double-Hann request
    proc.process_batch()
    assert_spectrum_close(proc.distribute_results()[rid]["magnitude"], g["app_mag"], TOL_DB)
    st = proc.get_performance_stats()
    assert st["gpu_enabled"] is True and st["pending_requests"] == 0 and st["last_batch_size"] == 1
    assert get_batched_fft_processor() is get_batched_fft_processor()
    gf = GPUAcceleratedFFT()
    for wt in ("hann", "hamming", "blackman"):
        mag, cx = gf.compute_fft(g["g_in"], wt, True)
        assert_spectrum_close(mag, g[f"g_mag_{wt}"], TOL_DB)
        assert np.abs(cx - g[f"g_cplx_{wt}"]).max() / np.abs(g[f"g_cplx_{wt}"]).max() < 2e-6
    mag2, none = gf.compute_fft(g["g_in"], "hann", return_complex=False)  # cache hit path
    assert none is None and np.array_equal(mag2, gf.compute_fft(g["g_in"], "hann")[0])
    m = gf.compute_multi_resolution_fft(g["gm_in"], {"bass": 8192, "mid": 4096, "high": 1024})
    for name in ("bass", "mid", "high"):
        assert_spectrum_close(m[name]["magnitude"], g[f"gm_mag_{name}"], TOL_DB, label=name)
        assert np.array_equal(m[name]["freqs"], g[f"gm_freqs_{name}"])
    batch = np.stack([g["in_2"], g["in_3"]])
    cx = gf.process_fft_batch(batch, "hann")
    ref = np.fft.rfft(batch.astype(np.float64) * np.hanning(2048), axis=1)
    assert np.abs(cx - ref).max() / np.abs(ref).max() < 2e-6


def test_shim_freq_mapper_bit_exact_and_bars(golden):
    from omega4_b200.optimization.freq_mapper import PrecomputedFrequencyMapper
    g = golden("freq_mapper.npz")
    known = {"48000_2048_512": "9951968a2477a6eb", "48000_8192_512": "bc77c57968c01d00",
             "96000_32768_512": "4d58d76d7eae1a5f"}
    for combo in g["combos"]:
        combo = str(combo)
        sr, n, bars = (int(v) for v in combo.split("_"))
        fm = PrecomputedFrequencyMapper(sr, n, bars)
        b = np.array(fm.mapping.band_indices, dtype=np.int32)
        assert np.array_equal(b, g["bands_" + combo])                    # bit exact
        if combo in known:
            assert hashlib.sha256(b.tobytes()).hexdigest()[:16] == known[combo]
        spec = g["spec_" + combo]
        np.testing.assert_allclose(fm.map_spectrum_to_bars(spec, True), g["bars_comp_" + combo], rtol=2e-5, atol=1e-7)
        np.testing.assert_allclose(fm.map_spectrum_to_bars(spec, False), g["bars_raw_" + combo], rtol=2e-5, atol=1e-7)
        np.testing.assert_allclose(fm.map_spectrum_to_bars(spec[:512], True), g["bars_short_" + combo], rtol=2e-5, atol=1e-7)


def test_band_map_db_mode():
    from omega4_b200.plan import band_map_host
    rng = np.random.default_rng(3)
    spec = np.abs(rng.standard_normal((4, 513))).astype(np.float32)
    spec[0, :40] = 0
    bands = O.mel_band_indices(48000, 1024, 64)
    got = band_map_host(spec, bands, None, db=True)
    ref = np.stack([O.magnitude_to_db(O.map_spectrum_to_bars(s, bands, 64)) for s in spec])
    assert np.abs(got - ref).max() < 1e-3


def test_shim_professional_metering(golden):
    from omega4_b200.panels.professional_meters import ProfessionalMetering, ProfessionalMetersPanel
    from omega4_b200 import Omega4CudaError
    g = golden("meters_stream.npz")
    m = ProfessionalMetering(48000)
    x, f = g["x"], int(g["first_hop"])
    d0 = None
    for k in range(f, 60):
        frame = x[(k + 1) * HOP - W:(k + 1) * HOP] * np.hanning(W)
        assert abs(m.calculate_true_peak(frame) - g["tp_db"][k - f]) <= 1e-3
        d = m.calculate_lufs(frame)
        d0 = d0 or d
        assert d is d0                                                  # same mutable dict object
        _meters_close([d[key] for key in O.METER_KEYS], g["meters"][k - f], f"shim hop {k}")
    assert len(m.lufs_integrated_history) == 60 - f and len(m.peak_history) == 60 - f
    assert abs(m.lufs_momentary_history[-1] - g["lufs_inst"][59 - f]) < 1e-5
    assert m.calculate_lufs(np.zeros(0)) is d0 and m.calculate_true_peak(np.zeros(0)) == -100.0
    np.testing.assert_allclose(m.k_weighting_filter["hp_a"], golden("meters_known.npz")["hp_a"], atol=2e-15)
    with pytest.raises(Omega4CudaError):
        m.calculate_lufs(np.zeros(480))                                 # unsupported length: loud, no CPU path
    gp = golden("meters_panel.npz")
    p = ProfessionalMetersPanel(48000)
    assert p.get_results()["lufs"] is None
    for j, k in enumerate(range(int(gp["first_hop"]), 60)):
        p.update(gp["x"][(k + 1) * HOP - W:(k + 1) * HOP] * np.hanning(W))
        assert abs(p.peak_hold_value - gp["peak_hold"][j]) <= TOL_TP
        assert p.peak_hold_counter == gp["peak_hold_counter"][j]
        assert abs(p.transient_info["attack_time"] - gp["attack_time"][j]) < 1e-9
        assert p.transient_info["transients_detected"] == gp["transients"][j]
    np.testing.assert_allclose(np.array(p.level_history), gp["level_history"], atol=TOL_LU)
    np.testing.assert_allclose(p.get_level_histogram()[1], gp["histogram"], atol=0.02)


# ------------------------------------------------------------------ batch driver
def test_batch_driver_tiles_match_one_shot_and_oracle(plan):
    import torch
    from omega4_b200.batch.driver import StreamBatch, analyze_resident
    from omega4_b200.batch.synth import synth_streams
    n_hops = 90
    x = synth_streams(3, 2, n_hops * HOP).reshape(6, -1)
    xd = torch.from_numpy(x).cuda()
    comb = torch.empty((6, n_hops, 512), device="cuda")
    met = torch.empty((6, n_hops, 5), device="cuda")
    analyze_resident(plan, xd, combined=comb, meters=met)
    torch.cuda.synchronize()
    host = plan.analyze_host(x)
    assert np.array_equal(host["combined"], comb.cpu().numpy()) and np.array_equal(host["meters"], met.cpu().numpy())
    # time tiles with carried history + meter state: bit-identical to the one-shot run
    sb = StreamBatch(plan, 6, max_tile_hops=32)
    comb_t = torch.empty_like(comb)
    met_t = torch.empty_like(met)
    k = 0
    for nh in (32, 7, 32, 19):
        sb.tile_view(nh).copy_(xd[:, k * HOP:(k + nh) * HOP])
        c = torch.empty((6, nh, 512), device="cuda")
        m = torch.empty((6, nh, 5), device="cuda")
        sb.push(nh, combined=c, meters=m)
        comb_t[:, k:k + nh] = c
        met_t[:, k:k + nh] = m
        k += nh
    torch.cuda.synchronize()
    # spectra and LUFS columns are bit-identical; the true-peak kernel packs two consecutive frames into
    # one complex transform, so a different tiling pairs frames differently: same value to fp32 rounding
    assert k == n_hops and torch.equal(comb_t, comb) and torch.equal(met_t[..., :4], met[..., :4])
    # (half-precision delayed phases on the batch path: two evaluations of a frame in different lanes agree to ~0.01 dBTP)
    assert float((met_t[..., 4] - met[..., 4]).abs().max()) < 0.03
    # channels are independent: a single channel run alone gives the same rows
    solo = plan.analyze_host(x[4:5])
    assert np.array_equal(solo["combined"][0], host["combined"][4]) and np.array_equal(solo["meters"][0], host["meters"][4])
    # and the oracle agrees
    ref = O.analyze_channel(x[4], 48000, O.BASELINE_CONFIGS)
    assert_spectrum_close(host["combined"][4], ref["combined"], TOL_DB, label="driver vs oracle")
    _meters_close(host["meters"][4], ref["meters"], "driver vs oracle")


def test_device_synth_and_properties_at_scale(plan):
    """Size-independent properties on a larger HBM-resident batch (256 channels x 20 s):
    determinism, linearity of the spectrum in the input gain, +6.02 dB LUFS/TP shift, silence."""
    import torch
    from omega4_b200.batch.driver import device_synth, analyze_resident
    n_ch, n_hops = 256, 1875
    x = device_synth(n_ch // 2, 2, n_hops * HOP)
    assert torch.isfinite(x).all() and 0.2 < float(x.std()) < 0.6 and float(x.abs().max()) < 1.2
    assert not torch.equal(x[0], x[1]) and not torch.equal(x[0], x[2])
    comb = torch.empty((n_ch, n_hops, 512), device="cuda")
    met = torch.empty((n_ch, n_hops, 5), device="cuda")
    analyze_resident(plan, x, combined=comb, meters=met)
    comb2 = torch.empty_like(comb)
    met2 = torch.empty_like(met)
    analyze_resident(plan, x * 2.0, combined=comb2, meters=met2)
    torch.cuda.synchronize()
    assert torch.isfinite(comb).all() and torch.isfinite(met).all()
    assert float(((comb2 - 2 * comb).abs() / (comb.abs().amax(dim=-1, keepdim=True) + 1e-20)).max()) < 1e-5
    steady = slice(200, None)
    shift = 20 * np.log10(2.0)
    assert float((met2[:, steady, :3] - met[:, steady, :3] - shift).abs().max()) < 1e-3
    assert float((met2[:, steady, 4] - met[:, steady, 4] - shift).abs().max()) < 1e-3
    assert float((met2[:, steady, 3] - met[:, steady, 3]).abs().max()) < 1e-3       # range is gain invariant
    comb3 = torch.empty_like(comb)
    analyze_resident(plan, x, combined=comb3, meters=met2)
    torch.cuda.synchronize()
    assert torch.equal(comb3, comb) and torch.equal(met2, met)                      # deterministic
    x.zero_()
    analyze_resident(plan, x, combined=comb, meters=met)
    torch.cuda.synchronize()
    assert float(comb.abs().max()) == 0.0
    assert torch.equal(met[:, 3:], torch.tensor([-100., -100., -100., 0., -100.], device="cuda").expand(n_ch, n_hops - 3, 5))


def test_smoke_entry():
    import __graft_entry__ as ge
    ge.smoke()
