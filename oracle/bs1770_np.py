"""TEST INFRASTRUCTURE ONLY -- float64 numpy/scipy oracle of ITU-R BS.1770-4 program loudness and
EBU Tech 3342 loudness range, the reference the GPU loudness path (``omega4_b200.loudness``) is tested against.

This is NOT a port of the OMEGA-4 reference: the reference has no such path (its ``ProfessionalMetering`` is
not textbook BS.1770, SURVEY.md section 0.2).  It is written straight from the definitions pinned in
DESIGN.md section 4.7:

- K-weighting: the high-shelf then the high-pass biquad, ``scipy.signal.lfilter`` over the whole stream from
  zero initial state, coefficients from the closed form (``_k_weighting`` restates it here, independent of
  ``omega4_b200.tables``);
- 100 ms sub-blocks of ``sub = fs / 10`` samples, ``z_j = sum_c G_c sum_{n in j} y_c[n]^2``;
- momentary ``M_j = -0.691 + 10 log10(sum_{i=j-3..j} z_i / (4 sub))`` (NaN for j < 3), short-term ``S_j`` over
  ``i = j-29..j`` / ``(30 sub)`` (NaN for j < 29), -inf for zero energy;
- integrated loudness over the momentary blocks with the absolute gate (> -70 LUFS) and the relative gate
  (> 10 LU below the energy mean of the absolutely gated blocks), -inf when no block passes;
- loudness range over the short-term values: absolute gate > -70, relative gate > 20 LU below their energy
  mean, then ``v[floor(0.95 (n-1) + 0.5)] - v[floor(0.10 (n-1) + 0.5)]`` of the sorted survivors, 0 when n = 0;
- sample peak ``20 log10(max |x|)`` per channel (-inf for silence).
"""
from __future__ import annotations

from typing import Dict, Sequence

import numpy as np
from scipy.signal import lfilter

ABS_GATE = -70.0
REL_GATE_I = -10.0
REL_GATE_LRA = -20.0


def _k_weighting(fs: float):
    K = np.tan(np.pi * 1681.974450955533 / fs)
    Vh = 10.0 ** (3.999843853973347 / 20.0)
    Vb = Vh ** 0.4996667741545416
    Q = 0.7071752369554196
    a0 = 1.0 + K / Q + K * K
    shelf_b = np.array([Vh + Vb * K / Q + K * K, 2.0 * (K * K - Vh), Vh - Vb * K / Q + K * K]) / a0
    shelf_a = np.array([1.0, 2.0 * (K * K - 1.0) / a0, (1.0 - K / Q + K * K) / a0])
    K = np.tan(np.pi * 38.13547087602444 / fs)
    Q = 0.5003270373238773
    d = 1.0 + K / Q + K * K
    return shelf_b, shelf_a, np.array([1.0, -2.0, 1.0]), np.array([1.0, 2.0 * (K * K - 1.0) / d, (1.0 - K / Q + K * K) / d])


def k_weighting(fs: float):
    """(shelf_b, shelf_a, hp_b, hp_a) float64."""
    return _k_weighting(float(fs))


def _lufs(energy_per_sample):
    with np.errstate(divide="ignore"):
        return -0.691 + 10.0 * np.log10(energy_per_sample)


def subblock_energies(x: np.ndarray, fs: int, weights: Sequence[float]) -> np.ndarray:
    """x float [C, n] of one stream -> z [n // sub] weighted sub-block energies (float64)."""
    if fs % 10:
        raise ValueError("sample rate must be a multiple of 10")
    sub = fs // 10
    sb, sa, hb, ha = k_weighting(fs)
    x = np.asarray(x, dtype=np.float64)
    nb = x.shape[1] // sub
    z = np.zeros(nb)
    for c in range(x.shape[0]):
        y = lfilter(hb, ha, lfilter(sb, sa, x[c]))
        z += float(weights[c]) * (y[:nb * sub] ** 2).reshape(nb, sub).sum(axis=1)
    return z


def window_loudness(z: np.ndarray, sub: int, width: int) -> np.ndarray:
    """Loudness at the end of every sub-block over the last ``width`` sub-blocks (NaN before the window fills)."""
    out = np.full(len(z), np.nan)
    if len(z) >= width:
        s = np.array([z[j - width + 1:j + 1].sum() for j in range(width - 1, len(z))])
        out[width - 1:] = _lufs(s / (width * sub))
    return out


def integrated(momentary: np.ndarray) -> float:
    l = momentary[np.isfinite(momentary)]
    l = l[l > ABS_GATE]
    if l.size == 0:
        return -np.inf
    rel = _lufs(np.mean(10.0 ** ((l + 0.691) / 10.0))) + REL_GATE_I
    l = l[l > rel]
    if l.size == 0:
        return -np.inf
    return float(_lufs(np.mean(10.0 ** ((l + 0.691) / 10.0))))


def loudness_range(short_term: np.ndarray) -> float:
    v = short_term[np.isfinite(short_term)]
    v = v[v > ABS_GATE]
    if v.size == 0:
        return 0.0
    rel = _lufs(np.mean(10.0 ** ((v + 0.691) / 10.0))) + REL_GATE_LRA
    v = np.sort(v[v > rel])
    n = v.size
    if n == 0:
        return 0.0
    return float(v[int(np.floor(0.95 * (n - 1) + 0.5))] - v[int(np.floor(0.10 * (n - 1) + 0.5))])


def _nanmax(a: np.ndarray) -> float:
    a = a[~np.isnan(a)]
    return float(a.max()) if a.size else float("nan")


def stream_loudness(x: np.ndarray, fs: int, weights: Sequence[float]) -> Dict[str, object]:
    """One stream, x [C, n] -> M, S series (float64 LUFS per completed sub-block), I, LRA, max M, max S and
    the per-channel sample peak in dBFS."""
    sub = fs // 10
    z = subblock_energies(x, fs, weights)
    M = window_loudness(z, sub, 4)
    S = window_loudness(z, sub, 30)
    with np.errstate(divide="ignore"):
        peak = 20.0 * np.log10(np.abs(np.asarray(x)).max(axis=1).astype(np.float64)) if x.shape[1] else \
            np.full(x.shape[0], -np.inf)
    return {"z": z, "momentary": M, "short_term": S, "integrated": integrated(M), "lra": loudness_range(S),
            "max_momentary": _nanmax(M), "max_short_term": _nanmax(S), "sample_peak": peak}


def program_loudness(x: np.ndarray, fs: int, weights: Sequence[float]) -> Dict[str, np.ndarray]:
    """x [n_streams, C, n] -> the per-stream results of ``stream_loudness`` stacked."""
    rs = [stream_loudness(x[s], fs, weights) for s in range(x.shape[0])]
    return {k: np.stack([np.asarray(r[k]) for r in rs]) for k in rs[0]}
