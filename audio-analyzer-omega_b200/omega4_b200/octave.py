"""Per-channel one-third-octave band levels (IEC 61260-1 base-10 bands, Butterworth band-pass) on the GPU.

An extension outside reference parity: the reference's spectrum is psychoacoustically weighted and
normalised, so none of its values is a level that compares between streams, files or tools.  This module
measures the real-time-analyser spectrum acousticians and broadcast QC read: per channel row, the bands
x = -17 .. 13 (20 Hz .. 20 kHz nominal) below Nyquist, each the 6th-order digital Butterworth band-pass
``tables.third_octave_sos`` designs, run continuously in float64, with the level of every 100 ms block in dBFS
(a full-scale sine in the band reads 0 dBFS), the overall level of the unfiltered input as one extra
column, and per column the running Leq and the largest block level.  The blocks are the 100 ms sub-blocks
of ``LoudnessMeter``, so one pipeline gets loudness and band levels on the same grid from the same tiles.
Definitions: DESIGN.md section 4.8.  All arithmetic runs in libomega4_cuda (``omega4_octave_*``); there is
no CPU fallback.

    meter = ThirdOctaveMeter(48000, n_rows=2048, max_seconds=600)
    meter.push(tile)              # float32 CUDA tensor [n_rows, n], e.g. StreamBatch.tile_view(n_hops)
    meter.levels                  # [n_rows, steps, n_bands + 1] device tensor (dBFS; last column: overall)
    meter.leq, meter.max_level    # [n_rows, n_bands + 1] device tensors
    meter.nominal                 # numpy nominal mid-band frequencies (Hz) of the band columns
"""
from __future__ import annotations

import ctypes as C
from typing import Dict

import numpy as np

from . import _native as N
from . import tables
from ._blockmeter import BlockMeter, Handle, host_input


class _Handle(Handle):
    """Owns one omega4_octave object (sample rate, band table, device coefficients)."""

    def __init__(self, fs: int, device: int):
        sos = np.ascontiguousarray(tables.third_octave_sos(fs), dtype=np.float64)
        super().__init__("octave", N.OctaveDesc(fs, sos.shape[0], sos.ctypes.data_as(C.POINTER(C.c_double)), fs // 10),
                         device)


class ThirdOctaveMeter(BlockMeter):
    """One-third-octave band levels of ``n_rows`` channel rows, fed tile by tile with device tensors.

    ``max_seconds`` sizes the device series ``levels`` ([n_rows, steps, n_bands + 1], one step per completed
    100 ms block).  Rows are independent channels: there is no summation over channels and no weighting.
    ``launches`` counts one kernel per push."""

    def __init__(self, sample_rate: int, n_rows: int, max_seconds: float, device: int = 0):
        import torch
        if int(n_rows) < 1:
            raise ValueError("n_rows must be >= 1")
        self.n_rows = int(n_rows)
        super().__init__(_Handle, sample_rate, self.n_rows, self.n_rows, max_seconds, device)
        self._bands = tables.third_octave_bands(self.sample_rate)
        self.n_bands = int(self._bands["fm"].size)
        cols = self.n_bands + 1
        self._levels = torch.full((self.n_rows, self.capacity, cols), float("nan"), dtype=torch.float32, device=self.dev)
        self._leq = torch.full((self.n_rows, cols), float("-inf"), dtype=torch.float32, device=self.dev)
        self._lmax = torch.full_like(self._leq, float("-inf"))

    @property
    def frequencies(self) -> np.ndarray:
        """Exact mid-band frequencies 1000 * 10^(x / 10) Hz of the band columns (numpy, n_bands)."""
        return self._bands["fm"].copy()

    @property
    def nominal(self) -> np.ndarray:
        """Nominal mid-band frequencies (20, 25, 31.5, ... Hz) of the band columns (numpy, n_bands)."""
        return self._bands["nominal"].copy()

    @property
    def levels(self):
        """[n_rows, steps, n_bands + 1] device view: the level of every completed block in dBFS (-inf for zero
        energy); column n_bands is the overall level of the unfiltered input."""
        return self._levels[:, :self.steps]

    @property
    def leq(self):
        """[n_rows, n_bands + 1] device tensor: 10 log10(2 sum y^2 / T) over all T samples pushed since the last
        reset (an incomplete last block included); -inf before any energy."""
        return self._leq

    @property
    def max_level(self):
        """[n_rows, n_bands + 1] device tensor: the largest completed-block level since the last reset."""
        return self._lmax

    def reset(self) -> None:
        """Start every row anew: the next push ignores the carried state and rewrites the series from step 0;
        ``leq`` and ``max_level`` read -inf until then."""
        self.samples = 0
        self._leq.fill_(float("-inf"))
        self._lmax.fill_(float("-inf"))

    def push(self, tile, stream=None) -> int:
        """Continue every row by ``tile``: float32 CUDA tensor [n_rows, n] (unit stride along time, any row
        stride -- ``StreamBatch.tile_view`` qualifies).  Asynchronous on ``stream`` (default: torch's current
        stream).  Returns the number of 100 ms blocks this push completed."""
        n, row_stride, j0, done, s = self._tile(tile, stream)
        if n == 0:
            return 0
        cols = self.n_bands + 1
        rc = N.lib().omega4_octave_push(
            self._h.ptr, s, N.MEM_DEVICE, tile.data_ptr(), row_stride, self.n_rows, n, self._state.data_ptr(),
            1 if self.samples == 0 else 0, self.capacity, self._levels.data_ptr() + 4 * j0 * cols,
            self._leq.data_ptr(), self._lmax.data_ptr())
        N.check(rc, "omega4_octave_push")
        self.samples += n
        return done


def third_octave_levels(x: np.ndarray, sample_rate: int, device: int = 0) -> Dict[str, np.ndarray]:
    """Host convenience: x float32 [n_rows, n] -> numpy ``levels`` [n_rows, n // (sample_rate / 10),
    n_bands + 1], ``leq`` and ``max_level`` [n_rows, n_bands + 1] (dBFS; last column: overall), and the band
    columns' ``frequencies`` and ``nominal`` mid-band frequencies."""
    fs = tables.check_meter_rate(sample_rate)
    x = host_input(x, 2, "[n_rows, n]")
    n_rows, n = x.shape
    bands = tables.third_octave_bands(fs)
    h = _Handle(fs, device)
    try:
        cols = bands["fm"].size + 1
        steps = n // (fs // 10)
        state = np.zeros((n_rows, h.state_doubles), np.float64)
        levels = np.full((n_rows, steps, cols), np.nan, np.float32)
        leq = np.full((n_rows, cols), -np.inf, np.float32)
        lmax = np.full_like(leq, -np.inf)
        if n_rows and n:
            rc = N.lib().omega4_octave_push(h.ptr, None, N.MEM_HOST, x.ctypes.data, n, n_rows, n, state.ctypes.data,
                                            1, steps, levels.ctypes.data, leq.ctypes.data, lmax.ctypes.data)
            N.check(rc, "omega4_octave_push")
        return {"levels": levels, "leq": leq, "max_level": lmax, "frequencies": bands["fm"],
                "nominal": bands["nominal"]}
    finally:
        h.close()
