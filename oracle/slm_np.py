"""TEST INFRASTRUCTURE ONLY -- float64 numpy/scipy oracle of the per-channel IEC 61672-1 sound level meter, the
reference the GPU path (``omega4_b200.slm``) is tested against.

This is NOT a port of the OMEGA-4 reference: the reference has no such path.  It is written straight from the
definitions pinned in DESIGN.md section 4.9 and does not import ``omega4_b200.tables``, so the GPU path and the
oracle are designed independently:

- frequency weightings A and C: the IEC 61672-1 Annex E analog prototypes (pole frequencies f1 .. f4 below;
  A: four zeros at s = 0 and poles -2 pi {f1, f1, f2, f3, f4, f4}; C: two zeros at s = 0 and poles
  -2 pi {f1, f1, f4, f4}), digitised by ``scipy.signal.bilinear_zpk`` without pre-warping, gain set to
  |H| = 1 at 1 kHz, run by ``scipy.signal.sosfilt`` over the whole row from zero state; Z is no filter;
- time weightings ``lfilter([1 - a], [1, -a], y^2)``, a = exp(-1 / (tau fs)), tau = 0.125 s (F) and 1 s (S);
- 100 ms blocks of ``sub = fs / 10`` samples from the stream start; per block and weighting Leq, LFmax, LSmax,
  LF, LS, Lpeak; per row and weighting over all samples Leq, LFmax, LSmax, Lpeak; all 10 log10 of an energy
  in dB re a mean square of 1.0 (-inf for zero);
- percentile levels by ``np.sort``: L_N = v[floor((1 - N / 100) (n - 1) + 0.5)], NaN for n = 0.
"""
from __future__ import annotations

from typing import Dict

import numpy as np
from scipy.signal import bilinear_zpk, freqz_zpk, lfilter, sosfilt, zpk2sos

F1, F2, F3, F4 = 20.598997, 107.65265, 737.86223, 12194.217
WEIGHTINGS = ("A", "C", "Z")
TAU = {"F": 0.125, "S": 1.0}


def check_rate(fs) -> int:
    if int(fs) != fs or int(fs) % 10 or not 8000 <= int(fs) <= 192000:
        raise ValueError(f"sample rate {fs} must be an integer multiple of 10 in [8000, 192000]")
    return int(fs)


def analog_zpk(kind: str):
    """(zeros, poles, gain 1) of the analog A or C weighting prototype."""
    if kind == "A":
        return np.zeros(4), -2.0 * np.pi * np.array([F1, F1, F2, F3, F4, F4]), 1.0
    if kind == "C":
        return np.zeros(2), -2.0 * np.pi * np.array([F1, F1, F4, F4]), 1.0
    raise ValueError(kind)


def weighting_sos(kind: str, fs) -> np.ndarray:
    """scipy's bilinear design of weighting ``kind`` at ``fs``, normalised to |H(1 kHz)| = 1."""
    z, p, k = bilinear_zpk(*analog_zpk(kind), check_rate(fs))
    _, h = freqz_zpk(z, p, k, worN=[1000.0], fs=fs)
    return zpk2sos(z, p, k / abs(h[0]))


def analog_db(kind: str, f) -> np.ndarray:
    """Magnitude (dB) of the analog prototype at f Hz, normalised to 0 dB at 1 kHz."""
    z, p, _ = analog_zpk(kind)

    def mag(fr):
        s = 2j * np.pi * np.asarray(fr, dtype=np.float64)
        return np.abs(np.prod(s[..., None] - z, axis=-1) / np.prod(s[..., None] - p, axis=-1))
    return 20.0 * np.log10(mag(f) / mag(1000.0))


def _db(e):
    with np.errstate(divide="ignore"):
        return 10.0 * np.log10(e)


def sound_levels(x: np.ndarray, fs) -> Dict[str, np.ndarray]:
    """x [n_rows, n] -> ``levels`` [n_rows, n // sub, 3, 6] (weighting A, C, Z; Leq, LFmax, LSmax, LF, LS, Lpeak)
    and ``totals`` [n_rows, 3, 4] (Leq, LFmax, LSmax, Lpeak), float64 dB."""
    fs = check_rate(fs)
    x = np.atleast_2d(np.asarray(x, dtype=np.float64))
    n_rows, n = x.shape
    sub = fs // 10
    steps = n // sub
    levels = np.zeros((n_rows, steps, 3, 6))
    totals = np.zeros((n_rows, 3, 4))
    for w, kind in enumerate(WEIGHTINGS):
        y = x if kind == "Z" else sosfilt(weighting_sos(kind, fs), x, axis=1)
        e = y * y
        v = {}
        for t, tau in TAU.items():
            a = np.exp(-1.0 / (tau * fs))
            v[t] = lfilter([1.0 - a], [1.0, -a], e, axis=1)

        def blocks(s):
            return s[:, :steps * sub].reshape(n_rows, steps, sub)
        levels[:, :, w, 0] = _db(blocks(e).sum(axis=2) / sub)
        levels[:, :, w, 1] = _db(blocks(v["F"]).max(axis=2) if steps else np.zeros((n_rows, 0)))
        levels[:, :, w, 2] = _db(blocks(v["S"]).max(axis=2) if steps else np.zeros((n_rows, 0)))
        levels[:, :, w, 3] = _db(v["F"][:, sub - 1:steps * sub:sub])
        levels[:, :, w, 4] = _db(v["S"][:, sub - 1:steps * sub:sub])
        with np.errstate(divide="ignore"):
            levels[:, :, w, 5] = 20.0 * np.log10(np.abs(blocks(y)).max(axis=2) if steps else np.zeros((n_rows, 0)))
        if n:
            totals[:, w, 0] = _db(e.sum(axis=1) / n)
            totals[:, w, 1] = _db(v["F"].max(axis=1))
            totals[:, w, 2] = _db(v["S"].max(axis=1))
            with np.errstate(divide="ignore"):
                totals[:, w, 3] = 20.0 * np.log10(np.abs(y).max(axis=1))
        else:
            totals[:, w] = -np.inf
    return {"levels": levels, "totals": totals}


def percentile_rank(N: float, n: int) -> int:
    """0-based ascending rank of L_N among n values."""
    return int(np.floor((1.0 - N / 100.0) * (n - 1) + 0.5))


def percentiles(series: np.ndarray, ns) -> np.ndarray:
    """series [n_rows, n] -> [n_rows, len(ns)] L_N by np.sort (-inf lowest); NaN for n = 0."""
    series = np.atleast_2d(np.asarray(series))
    n_rows, n = series.shape
    out = np.full((n_rows, len(ns)), np.nan, dtype=series.dtype)
    if n:
        v = np.sort(series, axis=1)
        for i, N in enumerate(ns):
            out[:, i] = v[:, percentile_rank(N, n)]
    return out
