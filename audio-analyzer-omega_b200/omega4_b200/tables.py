"""Host-side tables that define the reference's behaviour (SURVEY.md section 7 step 3).

Windows, per-bin psychoacoustic weights, the np.interp segments of ``combine_results_optimized``,
mel band ``(start, end)`` pairs and the K-weighting coefficients are computed here with the same
numpy formulas the reference uses and handed to the CUDA library as DATA; that is what keeps the
index tables bit-exact and lets the kernels inherit the reference's quirks.
Paths cited are relative to the reference root.
"""
from __future__ import annotations

from typing import List, Sequence, Tuple

import numpy as np


# ------------------------------------------------------------------ windows
def multires_window(window_type: str, n: int) -> np.ndarray:
    """omega4/audio/multi_resolution_fft.py:171-193.  'hann' -> ``np.hann`` does not exist ->
    the except branch installs ones; 'blackman_harris' falls back to blackman."""
    wt = str(window_type).lower()
    if wt == "hann":
        return np.ones(n, dtype=np.float32)
    if wt == "hamming":
        return np.hamming(n).astype(np.float32)
    return np.blackman(n).astype(np.float32)


def batched_window(window_type: str, n: int) -> np.ndarray:
    """omega4/optimization/batched_fft_processor.py:101-117."""
    if window_type == "hann":
        return np.hanning(n).astype(np.float32)
    if window_type == "hamming":
        return np.hamming(n).astype(np.float32)
    if window_type == "blackman":
        return np.blackman(n).astype(np.float32)
    return np.ones(n, dtype=np.float32)


def gpufft_window(window_type: str, n: int) -> np.ndarray:
    """omega4/optimization/gpu_accelerated_fft.py:115-125 (anything but hann/hamming -> blackman)."""
    if window_type == "hann":
        return np.hanning(n).astype(np.float32)
    if window_type == "hamming":
        return np.hamming(n).astype(np.float32)
    return np.blackman(n).astype(np.float32)


# ------------------------------------------------------------------ multi-resolution tables
def psycho_weights(freqs: np.ndarray, freq_range: Tuple[float, float], weight: float) -> np.ndarray:
    """omega4/audio/multi_resolution_fft.py:304-326 (float32 in-place arithmetic)."""
    w = np.ones(len(freqs), dtype=np.float32)
    w.fill(weight)
    inr = (freqs >= freq_range[0]) & (freqs <= freq_range[1])
    w[inr & (freqs >= 60) & (freqs <= 120)] *= 1.8
    w[inr & (freqs >= 200) & (freqs <= 400)] *= 1.4
    w[inr & (freqs >= 2000) & (freqs <= 5000)] *= 1.2
    w[inr & (freqs >= 20) & (freqs <= 80)] *= 1.6
    return w


def combine_tables(sample_rate: int, max_freq: float, sizes: Sequence[int],
                   ranges: Sequence[Tuple[float, float]], target_bins: int):
    """np.interp segments of combine_results_optimized (multi_resolution_fft.py:353-391).

    Per resolution: (target index int32[], lower FFT bin int32[], fraction float32[]) such that
    interp = m[lo] + (m[lo+1] - m[lo]) * frac reproduces ``np.interp(target_subset, valid_freqs,
    valid_magnitude)`` including its clamping at both ends."""
    target_freqs = np.linspace(0, max_freq, target_bins)
    out = []
    for n, fr in zip(sizes, ranges):
        freqs = np.fft.rfftfreq(n, 1 / sample_rate)
        valid = np.where((freqs >= fr[0]) & (freqs <= fr[1]))[0]
        tidx = np.where((target_freqs >= fr[0]) & (target_freqs <= fr[1]))[0]
        if len(valid) < 2 or len(tidx) == 0:            # :373-374, :380-381
            out.append((np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0, np.float32)))
            continue
        vf = freqs[valid]
        x = target_freqs[tidx]
        j = np.searchsorted(vf, x, side="right") - 1
        lo = np.clip(j, 0, len(vf) - 2)
        frac = (x - vf[lo]) / (vf[lo + 1] - vf[lo])
        frac = np.where(j < 0, 0.0, frac)
        frac = np.where(j >= len(vf) - 1, 1.0, frac)
        out.append((tidx.astype(np.int32), (valid[0] + lo).astype(np.int32), frac.astype(np.float32)))
    return out


# ------------------------------------------------------------------ mel band mapping
def mel_band_indices(sample_rate: int, fft_size: int, num_bars: int) -> List[Tuple[int, int]]:
    """omega4/optimization/freq_mapper.py:83-124 -- must stay bit-exact (sha256 known answers in
    SURVEY.md section 8 a9), so it is computed with the same numpy scalar arithmetic."""
    binw = sample_rate / fft_size
    mel_min = 2595 * np.log10(1 + 20 / 700)
    mel_max = 2595 * np.log10(1 + 20000 / 700)
    mel_points = np.linspace(mel_min, mel_max, num_bars + 1)
    freq_points = [700 * (10 ** (mel / 2595) - 1) for mel in mel_points]
    freq_points[0] = max(20, freq_points[0])
    freq_points[-1] = min(20000, freq_points[-1])
    bands = []
    for i in range(num_bars):
        if i >= len(freq_points) - 1:
            break
        s = int(freq_points[i] / binw)
        e = int(freq_points[i + 1] / binw)
        if e <= s:
            e = s + 1
        s = max(0, min(s, fft_size // 2))
        e = max(s + 1, min(e, fft_size // 2 + 1))
        bands.append((s, e))
    return bands


def compensation_curve(frequencies: np.ndarray) -> np.ndarray:
    """omega4/optimization/freq_mapper.py:146-163."""
    f = np.asarray(frequencies, dtype=np.float64)
    c = np.ones_like(f)
    c = np.where((f > 0) & (f < 100), 1.0 + (100 - f) / 100 * 0.5, c)
    c = np.where((f >= 1000) & (f < 4000), 1.0 + (f - 1000) / 3000 * 0.3, c)
    c = np.where(f >= 4000, 1.3 - (f - 4000) / 16000 * 0.5, c)
    return c


def mel_scale_factors(frequencies: np.ndarray) -> np.ndarray:
    """omega4/optimization/freq_mapper.py:126-144."""
    f = np.asarray(frequencies, dtype=np.float64)
    return np.select([f < 250, f < 500, f < 2000, f < 6000], [1.5, 1.3, 1.1, 1.0], 0.9)


# ------------------------------------------------------------------ app-level post-processing
def app_compensation_gains(freqs: np.ndarray, content_type: str = "instrumental",
                           vocal_suppression: float = 0.0) -> np.ndarray:
    """Per-bin float32 gains of ProfessionalLiveAudioAnalyzer.apply_frequency_compensation
    (omega4_main.py:855-926): the in-place ``compensated[mask] *= g`` statements run on ones."""
    f = np.asarray(freqs)
    c = np.ones(len(f), dtype=np.float32)
    if content_type == "vocal":
        for m, g in ((f < 60, 0.15), ((f >= 60) & (f < 250), 0.2), ((f >= 250) & (f < 500), 0.6),
                     ((f >= 500) & (f < 2000), 1.5)):
            c[m] *= g
    else:
        for m, g in ((f < 60, 0.8), ((f >= 60) & (f < 250), 1.0), ((f >= 250) & (f < 500), 1.1),
                     ((f >= 500) & (f < 2000), 0.85)):
            c[m] *= g
    c[(f >= 2000) & (f < 6000)] *= 1.2
    c[(f >= 6000) & (f < 10000)] *= 0.8
    c[f >= 10000] *= 0.3
    if vocal_suppression > 0:
        c[(f >= 800) & (f < 4000)] *= (1.0 - vocal_suppression * 0.5)
    return c


def app_smoothing_factors(bands, sample_rate: int, fft_size_base: int) -> np.ndarray:
    """omega4_main.py:1043-1052: band start bin -> Hz -> 0.6 (< 250 Hz) / 0.75 (< 2 kHz) / 0.85."""
    hz = np.array([s for s, _e in bands], dtype=np.float64) * sample_rate / fft_size_base
    return np.where(hz < 250, 0.6, np.where(hz < 2000, 0.75, 0.85))


# ------------------------------------------------------------------ meters
def butter2_highpass(fc: float, fs: float):
    """scipy.signal.butter(2, fc/(fs/2), 'high') in closed form (bilinear transform with
    pre-warping) -- omega4/panels/professional_meters.py:54,62-64."""
    k = np.tan(np.pi * fc / fs)
    norm = 1.0 / (1.0 + np.sqrt(2.0) * k + k * k)
    b = np.array([1.0, -2.0, 1.0]) * norm
    a = np.array([1.0, 2.0 * (k * k - 1.0) * norm, (1.0 - np.sqrt(2.0) * k + k * k) * norm])
    return b, a


def k_weighting_coeffs(sample_rate: int) -> np.ndarray:
    """[hp_b, hp_a, shelf_b, shelf_a] flattened (12 doubles): 38 Hz and 1500 Hz Butterworth-2
    high-passes (professional_meters.py:48-72; shelf_gain there is computed but unused)."""
    hp_b, hp_a = butter2_highpass(38.0, sample_rate)
    sh_b, sh_a = butter2_highpass(1500.0, sample_rate)
    return np.concatenate([hp_b, hp_a, sh_b, sh_a]).astype(np.float64)


def butter_lowhigh(order: int, fc: float, fs: float, btype: str):
    """scipy.signal.butter(order, fc/(fs/2), btype), order 1 or 2, closed form (bilinear transform
    with pre-warping) -- the sections of professional_meters.py:88-99, 118-121."""
    k = np.tan(np.pi * fc / fs)
    if order == 1:
        a = np.array([1.0, (k - 1.0) / (k + 1.0)])
        b = (np.array([1.0, -1.0]) if btype == "high" else np.array([k, k])) / (1.0 + k)
        return b, a
    norm = 1.0 / (1.0 + np.sqrt(2.0) * k + k * k)
    a = np.array([1.0, 2.0 * (k * k - 1.0) * norm, (1.0 - np.sqrt(2.0) * k + k * k) * norm])
    b = (np.array([1.0, -2.0, 1.0]) if btype == "high" else np.array([1.0, 2.0, 1.0]) * k * k) * norm
    return b, a


def weighting_program(mode: str, sample_rate: int):
    """ProfessionalMetering.weighting_mode -> the cascade the CUDA meter kernel runs
    (professional_meters.py:74-127 filters, :129-229 application): dict with ``sections`` [(b, a)],
    ``blend`` (K's f + 0.3 (s - f)), ``rms_gate`` and ``gain``."""
    nyq = sample_rate / 2
    f1, f2, f3, f4 = 20.598997, 107.65265, 737.86223, 12194.217
    if mode == "K":
        return {"sections": [butter2_highpass(38.0, sample_rate), butter2_highpass(1500.0, sample_rate)],
                "blend": 1, "rms_gate": 1, "gain": 1.0}
    if mode == "A":
        return {"sections": [butter_lowhigh(2, f1, sample_rate, "high"), butter_lowhigh(1, f2, sample_rate, "high"),
                             butter_lowhigh(1, f3, sample_rate, "low"),
                             butter_lowhigh(2, min(f4 / nyq, 0.99) * nyq, sample_rate, "low")],
                "blend": 0, "rms_gate": 1, "gain": 2.5}
    if mode == "C":
        return {"sections": [butter_lowhigh(2, f1, sample_rate, "high"),
                             butter_lowhigh(2, min(f4 / nyq, 0.99) * nyq, sample_rate, "low")],
                "blend": 0, "rms_gate": 1, "gain": 1.0}
    return {"sections": [], "blend": 0, "rms_gate": 0, "gain": 1.0}       # 'Z' and anything else (:228-229)


# ------------------------------------------------------------------ ITU-R BS.1770-4 program loudness (extension)
#: channel weights G_c per stream layout (BS.1770-4 Table 3; 5.1 in L R C LFE Ls Rs order, LFE excluded).
#: There is no named 7.1 layout: its surround weights depend on speaker azimuth, so pass explicit weights.
BS1770_LAYOUTS = {
    "mono": (1.0,),
    "stereo": (1.0, 1.0),
    "5.1": (1.0, 1.0, 1.0, 0.0, 1.41, 1.41),
}


def bs1770_k_weighting(sample_rate: float) -> Tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray]:
    """(shelf_b, shelf_a, hp_b, hp_a), float64: the two K-weighting biquads of BS.1770-4 (high-shelf
    pre-filter, then the RLB high-pass) for any sample rate, from the bilinear-transform closed form whose
    parameters reproduce the standard's 48 kHz table to 1e-15."""
    fs = float(sample_rate)
    f0, G, Q = 1681.974450955533, 3.999843853973347, 0.7071752369554196
    K = np.tan(np.pi * f0 / fs)
    Vh = 10.0 ** (G / 20.0)
    Vb = Vh ** 0.4996667741545416
    a0 = 1.0 + K / Q + K * K
    shelf_b = np.array([Vh + Vb * K / Q + K * K, 2.0 * (K * K - Vh), Vh - Vb * K / Q + K * K]) / a0
    shelf_a = np.array([1.0, 2.0 * (K * K - 1.0) / a0, (1.0 - K / Q + K * K) / a0])
    f0, Q = 38.13547087602444, 0.5003270373238773
    K = np.tan(np.pi * f0 / fs)
    d = 1.0 + K / Q + K * K
    hp_b = np.array([1.0, -2.0, 1.0])
    hp_a = np.array([1.0, 2.0 * (K * K - 1.0) / d, (1.0 - K / Q + K * K) / d])
    return shelf_b, shelf_a, hp_b, hp_a


def bs1770_channel_weights(layout_or_weights, n_channels: int | None = None) -> np.ndarray:
    """float64 G_c from a layout name in ``BS1770_LAYOUTS`` or an explicit sequence of weights."""
    if isinstance(layout_or_weights, str):
        if layout_or_weights not in BS1770_LAYOUTS:
            raise ValueError(f"unknown layout {layout_or_weights!r}: one of {sorted(BS1770_LAYOUTS)} "
                             "or an explicit list of channel weights")
        w = np.array(BS1770_LAYOUTS[layout_or_weights], dtype=np.float64)
    else:
        w = np.asarray(layout_or_weights, dtype=np.float64).reshape(-1)
    if w.size < 1 or not np.all(np.isfinite(w)) or np.any(w < 0):
        raise ValueError("channel weights must be one or more finite values >= 0")
    if n_channels is not None and w.size != n_channels:
        raise ValueError(f"{w.size} channel weights for {n_channels} channels")
    return w


# ------------------------------------------------------------------ IEC 61260-1 one-third-octave bands (extension)
#: nominal mid-band frequencies (Hz) of the base-10 bands x = -17 .. 13 (IEC 61260-1 Annex E)
THIRD_OCTAVE_NOMINAL = (20, 25, 31.5, 40, 50, 63, 80, 100, 125, 160, 200, 250, 315, 400, 500, 630, 800,
                        1000, 1250, 1600, 2000, 2500, 3150, 4000, 5000, 6300, 8000, 10000, 12500, 16000, 20000)
THIRD_OCTAVE_X = tuple(range(-17, 14))
THIRD_OCTAVE_ORDER = 3                     # Butterworth prototype order: a 6th-order band-pass, three biquads


def check_octave_rate(sample_rate) -> int:
    """The sample rate as an int; raises ValueError unless it is an integer multiple of 10 in [8000, 192000]
    (100 ms blocks of fs / 10 samples)."""
    try:
        fs = int(sample_rate)
    except (TypeError, ValueError):
        raise ValueError(f"sample rate {sample_rate!r} must be an integer") from None
    if fs != sample_rate or fs % 10 or not 8000 <= fs <= 192000:
        raise ValueError(f"sample rate {sample_rate} must be an integer multiple of 10 in [8000, 192000]")
    return fs


def third_octave_bands(sample_rate) -> dict:
    """The one-third-octave bands below Nyquist: base-10 system, exact mid-band f_m = 1000 * 10^(x / 10),
    edges f_m * 10^(-/+ 1/20); a band is included iff its upper edge f2 < fs / 2 (31 bands at 48 and
    96 kHz, 30 at 44.1 kHz, 23 at 8 kHz).  Returns float64 / int arrays ``x``, ``fm``, ``f1``, ``f2`` and
    the nominal labels ``nominal``."""
    fs = check_octave_rate(sample_rate)
    x = np.array(THIRD_OCTAVE_X)
    fm = 1000.0 * 10.0 ** (0.1 * x)
    f1, f2 = fm * 10.0 ** -0.05, fm * 10.0 ** 0.05
    keep = f2 < fs / 2.0
    return {"x": x[keep], "fm": fm[keep], "f1": f1[keep], "f2": f2[keep],
            "nominal": np.array(THIRD_OCTAVE_NOMINAL, dtype=np.float64)[keep]}


def third_octave_sos(sample_rate) -> np.ndarray:
    """[n_bands][3][6] float64 second-order sections (b0 b1 b2 1 a1 a2) of the digital Butterworth band-pass
    of each band, the filter ``scipy.signal.butter(3, [f1, f2], btype="bandpass", fs=fs, output="sos")``
    designs, in closed form: analog prototype poles, low-pass to band-pass on the pre-warped edges,
    bilinear transform.  The arithmetic follows that design step for step (edges normalised to Nyquist,
    pre-warped as 4 tan(pi Wn / 2), bilinear map z = (4 + s) / (4 - s)), so the coefficients agree with
    scipy's to float64 rounding.  Each conjugate pole pair gets one zero pair (z = 1 and z = -1, numerator
    g * [1, 0, -1]); the three sections share the gain equally.  The gain is 1/sqrt(2) at f1 and f2."""
    fs = check_octave_rate(sample_rate)
    b = third_octave_bands(fs)
    N = THIRD_OCTAVE_ORDER
    proto = -np.exp(1j * np.pi * np.arange(-N + 1, N, 2) / (2 * N))     # left half-plane unit-circle poles
    sos = np.zeros((b["fm"].size, N, 6))
    for i, (f1, f2) in enumerate(zip(b["f1"], b["f2"])):
        w1, w2 = 4.0 * np.tan(np.pi * (2.0 * f1 / fs) / 2.0), 4.0 * np.tan(np.pi * (2.0 * f2 / fs) / 2.0)
        bw, w0 = w2 - w1, np.sqrt(w1 * w2)
        pl = proto * bw / 2.0
        root = np.sqrt(pl ** 2 - w0 ** 2)
        ps = np.concatenate([pl + root, pl - root])                        # 2N band-pass poles
        pz = (4.0 + ps) / (4.0 - ps)
        k = np.real(bw ** N * 4.0 ** N / np.prod(4.0 - ps))               # N zeros at s = 0, N at infinity
        upper = np.sort_complex(pz[pz.imag > 0])
        g = k ** (1.0 / N)
        for j, p in enumerate(upper):
            sos[i, j] = [g, 0.0, -g, 1.0, -(p + np.conj(p)).real, (p * np.conj(p)).real]
    return sos
