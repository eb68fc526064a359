"""TEST INFRASTRUCTURE ONLY -- float64 numpy/scipy oracle of per-channel one-third-octave band levels, the
reference the GPU band-level path (``omega4_b200.octave``) is tested against.

This is NOT a port of the OMEGA-4 reference: the reference has no such path.  It is written straight from the
definitions pinned in DESIGN.md section 4.8, and it restates the band table here rather than importing
``omega4_b200.tables``, so the GPU path and the oracle are designed independently:

- bands of the base-10 system, x = -17 .. 13: f_m = 1000 * 10^(x / 10), f1 = f_m * 10^-0.05,
  f2 = f_m * 10^0.05, included iff f2 < fs / 2; the sample rate is an integer multiple of 10 in [8000, 192000];
- per band ``scipy.signal.butter(3, [f1, f2], btype="bandpass", fs=fs, output="sos")`` run by
  ``scipy.signal.sosfilt`` over the whole stream from zero state, in float64;
- 100 ms blocks of ``sub = fs / 10`` samples counted from the stream start; block level
  ``10 log10(2 / sub * sum y^2)`` dBFS (a full-scale sine in the band reads 0 dBFS), -inf for zero energy;
  one extra column, the overall level, is the same on the unfiltered input;
- ``leq = 10 log10(2 sum y^2 / T)`` over all T samples (including an incomplete last block) and ``max_level``,
  the largest completed-block level; both -inf when there is no energy (or no completed block, for max_level).
"""
from __future__ import annotations

from typing import Dict

import numpy as np
from scipy.signal import butter, sosfilt

NOMINAL = (20, 25, 31.5, 40, 50, 63, 80, 100, 125, 160, 200, 250, 315, 400, 500, 630, 800, 1000, 1250, 1600,
           2000, 2500, 3150, 4000, 5000, 6300, 8000, 10000, 12500, 16000, 20000)


def check_rate(fs) -> int:
    if int(fs) != fs or int(fs) % 10 or not 8000 <= int(fs) <= 192000:
        raise ValueError(f"sample rate {fs} must be an integer multiple of 10 in [8000, 192000]")
    return int(fs)


def bands(fs) -> Dict[str, np.ndarray]:
    """x, exact mid-band fm, edges f1 / f2 and nominal labels of the bands below fs / 2."""
    fs = check_rate(fs)
    out = {"x": [], "fm": [], "f1": [], "f2": [], "nominal": []}
    for i, x in enumerate(range(-17, 14)):
        fm = 1000.0 * 10.0 ** (x / 10.0)
        f1, f2 = fm / 10.0 ** 0.05, fm * 10.0 ** 0.05
        if f2 < fs / 2.0:
            for k, v in (("x", x), ("fm", fm), ("f1", f1), ("f2", f2), ("nominal", NOMINAL[i])):
                out[k].append(v)
    return {k: np.array(v, dtype=np.int64 if k == "x" else np.float64) for k, v in out.items()}


def band_sos(fs) -> list:
    b = bands(fs)
    return [butter(3, [f1, f2], btype="bandpass", fs=fs, output="sos") for f1, f2 in zip(b["f1"], b["f2"])]


def _db(e: np.ndarray) -> np.ndarray:
    with np.errstate(divide="ignore"):
        return 10.0 * np.log10(e)


def band_levels(x: np.ndarray, fs) -> Dict[str, np.ndarray]:
    """x [n_rows, n] -> ``levels`` [n_rows, n // sub, n_bands + 1] (last column: overall), ``leq`` and
    ``max_level`` [n_rows, n_bands + 1], all float64 dBFS, plus ``frequencies`` / ``nominal``."""
    fs = check_rate(fs)
    x = np.atleast_2d(np.asarray(x, dtype=np.float64))
    n_rows, n = x.shape
    sub = fs // 10
    steps = n // sub
    b = bands(fs)
    sos = band_sos(fs)
    nb = len(sos)
    blk = np.zeros((n_rows, steps, nb + 1))
    tot = np.zeros((n_rows, nb + 1))
    for k in range(nb + 1):
        y = sosfilt(sos[k], x, axis=1) if k < nb else x
        y2 = y * y
        blk[:, :, k] = y2[:, :steps * sub].reshape(n_rows, steps, sub).sum(axis=2)
        tot[:, k] = y2.sum(axis=1)
    levels = _db(2.0 / sub * blk)
    leq = _db(2.0 * tot / n) if n else np.full((n_rows, nb + 1), -np.inf)
    max_level = levels.max(axis=1) if steps else np.full((n_rows, nb + 1), -np.inf)
    return {"levels": levels, "leq": leq, "max_level": max_level, "frequencies": b["fm"], "nominal": b["nominal"]}
