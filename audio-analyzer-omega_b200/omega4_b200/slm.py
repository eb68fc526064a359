"""Per-channel IEC 61672-1 sound level meter on the GPU: A / C / Z frequency weighting, Fast / Slow time weighting,
Leq, Lmax, Lpeak and percentile levels.

An extension outside reference parity: the reference's A / C / Z meters filter each frame zero-phase with
Butterworth stand-ins and have no time weighting, so they are not levels; they stay as they are.  This module
is the sound level meter acoustics, noise and QC pipelines read next to ``LoudnessMeter`` and
``ThirdOctaveMeter``, on the same 100 ms blocks of the same tiles.  Per channel row (no channel summation) and
per weighting A, C and Z (A and C: the bilinear transform of the IEC 61672-1 Annex E prototypes,
``tables.iec61672_weighting_sos``; Z: no filter), with F (125 ms) and S (1 s) exponential time weighting run
continuously from silence, every completed 100 ms block gives the six ``QUANTITIES``: Leq, LFmax, LSmax, LF and
LS at the block end, and Lpeak.  Levels are in dB re a mean square of 1.0 (a full-scale sine reads Leq -3.01 dB;
the octave meter's dBFS reads 3.01 dB higher); add 20 log10(s / 20 uPa) for dB SPL when a sample of 1.0 is s
pascal.  Definitions: DESIGN.md section 4.9.  All arithmetic runs in libomega4_cuda (``omega4_slm_*``); there
is no CPU fallback.

    meter = SoundLevelMeter(48000, n_rows=2048, max_seconds=600)
    meter.push(tile)                      # float32 CUDA tensor [n_rows, n], e.g. StreamBatch.tile_view(n_hops)
    meter.levels                          # [n_rows, steps, 3, 6] device view (A, C, Z x QUANTITIES), dB
    meter.totals                          # [n_rows, 3, 4] device tensor: Leq, LFmax, LSmax, Lpeak since the start
    meter.percentiles((10, 50, 90))       # [n_rows, 3] LAF10, LAF50, LAF90 from LF sampled every 100 ms
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Sequence

import numpy as np

from . import _native as N
from . import tables
from ._blockmeter import BlockMeter, Handle, host_input

WEIGHTINGS = ("A", "C", "Z")
QUANTITIES = ("eq", "Fmax", "Smax", "F", "S", "peak")
TOTALS = ("eq", "Fmax", "Smax", "peak")


def _column(weighting: str, quantity: str) -> int:
    if weighting not in WEIGHTINGS:
        raise ValueError(f"weighting {weighting!r} must be one of {WEIGHTINGS}")
    if quantity not in QUANTITIES:
        raise ValueError(f"quantity {quantity!r} must be one of {QUANTITIES}")
    return WEIGHTINGS.index(weighting) * len(QUANTITIES) + QUANTITIES.index(quantity)


def _pct(ns: Sequence[float]) -> np.ndarray:
    p = np.ascontiguousarray(np.atleast_1d(np.asarray(ns, dtype=np.float64)))
    if p.ndim != 1 or not 1 <= p.size <= N.SLM_MAX_PCT:
        raise ValueError(f"give 1 .. {N.SLM_MAX_PCT} percentiles")
    if not np.all((p >= 0.0) & (p <= 100.0)):
        raise ValueError(f"percentiles must be in [0, 100], got {p}")
    return p


class _Handle(Handle):
    """Owns one omega4_slm object (sample rate, weighting coefficients, staging buffers)."""

    def __init__(self, fs: int, device: int):
        sa, sc = (np.ascontiguousarray(tables.iec61672_weighting_sos(k, fs), dtype=np.float64) for k in "AC")
        dp = C.POINTER(C.c_double)
        super().__init__("slm", N.SlmDesc(fs, fs // 10, sa.ctypes.data_as(dp), sc.ctypes.data_as(dp)), device)


class SoundLevelMeter(BlockMeter):
    """Sound level meter of ``n_rows`` channel rows, fed tile by tile with device tensors.

    ``max_seconds`` sizes the device series ``levels`` ([n_rows, steps, 3, 6], one step per completed 100 ms
    block).  Rows are independent channels.  F and S start from silence, so they read low for the first few
    time constants (0.125 s and 1 s).  ``launches`` counts one kernel per push and one per percentile query."""

    WEIGHTINGS = WEIGHTINGS
    QUANTITIES = QUANTITIES

    def __init__(self, sample_rate: int, n_rows: int, max_seconds: float, device: int = 0):
        import torch
        if int(n_rows) < 1:
            raise ValueError("n_rows must be >= 1")
        self.n_rows = int(n_rows)
        super().__init__(_Handle, sample_rate, self.n_rows, self.n_rows, max_seconds, device)
        nw, nq = len(WEIGHTINGS), len(QUANTITIES)
        self._levels = torch.full((self.n_rows, self.capacity, nw, nq), float("nan"), dtype=torch.float32,
                                  device=self.dev)
        self._totals = torch.full((self.n_rows, nw, len(TOTALS)), float("-inf"), dtype=torch.float32, device=self.dev)

    @property
    def levels(self):
        """[n_rows, steps, 3, 6] device view: per completed block and weighting (A, C, Z) Leq, LFmax, LSmax, LF,
        LS and Lpeak in dB (-inf for zero energy)."""
        return self._levels[:, :self.steps]

    @property
    def totals(self):
        """[n_rows, 3, 4] device tensor: per weighting Leq, LFmax, LSmax and Lpeak over all samples pushed since the
        last reset (an incomplete last block included); -inf before any energy."""
        return self._totals

    def reset(self) -> None:
        """Start every row anew from silence: the next push ignores the carried state and rewrites the series from
        step 0; ``totals`` read -inf until then."""
        self.samples = 0
        self._totals.fill_(float("-inf"))

    def push(self, tile, stream=None) -> int:
        """Continue every row by ``tile``: float32 CUDA tensor [n_rows, n] (unit stride along time, any row
        stride -- ``StreamBatch.tile_view`` qualifies).  Asynchronous on ``stream`` (default: torch's current
        stream).  Returns the number of 100 ms blocks this push completed."""
        n, row_stride, j0, done, s = self._tile(tile, stream)
        if n == 0:
            return 0
        cols = len(WEIGHTINGS) * len(QUANTITIES)
        rc = N.lib().omega4_slm_push(
            self._h.ptr, s, N.MEM_DEVICE, tile.data_ptr(), row_stride, self.n_rows, n, self._state.data_ptr(),
            1 if self.samples == 0 else 0, self.capacity, self._levels.data_ptr() + 4 * j0 * cols,
            self._totals.data_ptr())
        N.check(rc, "omega4_slm_push")
        self.samples += n
        return done

    def percentiles(self, ns: Sequence[float], weighting: str = "A", quantity: str = "F", stream=None):
        """[n_rows, len(ns)] device tensor: L_N, the level exceeded N % of the time, of series column (weighting,
        quantity) over the completed blocks, for each N in ``ns`` (in [0, 100]).  With the values sorted
        ascending, L_N = v[floor((1 - N / 100) (steps - 1) + 0.5)]: L_0 is the maximum, L_100 the minimum, -inf
        counts as the lowest; NaN before the first block.  The default column is LAF, which gives the customary
        LAF,N sampled every 100 ms.  One kernel launch."""
        import torch
        col = _column(weighting, quantity)
        p = _pct(ns)
        out = torch.empty((self.n_rows, p.size), dtype=torch.float32, device=self.dev)
        rc = N.lib().omega4_slm_percentiles(self._h.ptr, self._stream(stream), N.MEM_DEVICE, self._levels.data_ptr(),
                                            self.n_rows, self.steps, self.capacity, col, p.size, p.ctypes.data,
                                            out.data_ptr())
        N.check(rc, "omega4_slm_percentiles")
        return out


def sound_levels(x: np.ndarray, sample_rate: int, percentiles: Sequence[float] = (10, 50, 90),
                 device: int = 0) -> Dict[str, np.ndarray]:
    """Host convenience: x float32 [n_rows, n] -> numpy ``levels`` [n_rows, n // (sample_rate / 10), 3, 6],
    ``totals`` [n_rows, 3, 4] and ``percentiles`` [n_rows, len(percentiles)], the LAF,N of ``percentiles``
    (LAF sampled at every block end)."""
    fs = tables.check_meter_rate(sample_rate)
    x = host_input(x, 2, "[n_rows, n]")
    p = _pct(percentiles)
    n_rows, n = x.shape
    h = _Handle(fs, device)
    try:
        lib = N.lib()
        steps = n // (fs // 10)
        state = np.zeros((n_rows, h.state_doubles), np.float64)
        levels = np.full((n_rows, steps, len(WEIGHTINGS), len(QUANTITIES)), np.nan, np.float32)
        totals = np.full((n_rows, len(WEIGHTINGS), len(TOTALS)), -np.inf, np.float32)
        pct = np.full((n_rows, p.size), np.nan, np.float32)
        if n_rows and n:
            rc = lib.omega4_slm_push(h.ptr, None, N.MEM_HOST, x.ctypes.data, n, n_rows, n, state.ctypes.data, 1,
                                     steps, levels.ctypes.data, totals.ctypes.data)
            N.check(rc, "omega4_slm_push")
        if n_rows:
            rc = lib.omega4_slm_percentiles(h.ptr, None, N.MEM_HOST, levels.ctypes.data, n_rows, steps, steps,
                                            _column("A", "F"), p.size, p.ctypes.data, pct.ctypes.data)
            N.check(rc, "omega4_slm_percentiles")
        return {"levels": levels, "totals": totals, "percentiles": pct}
    finally:
        h.close()
