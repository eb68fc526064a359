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


class _Handle:
    """Owns one omega4_octave object (sample rate, band table, device coefficients)."""

    def __init__(self, sample_rate, device: int):
        fs = tables.check_octave_rate(sample_rate)
        lib = N.lib()
        N.require_device()
        self.sample_rate, self.sub = fs, fs // 10
        self.bands = tables.third_octave_bands(fs)
        self._sos = np.ascontiguousarray(tables.third_octave_sos(fs), dtype=np.float64)
        self.n_bands = int(self._sos.shape[0])
        d = N.OctaveDesc()
        d.sample_rate, d.n_bands, d.sub = fs, self.n_bands, self.sub
        d.sos = self._sos.ctypes.data_as(C.POINTER(C.c_double))
        self.ptr = lib.omega4_octave_create(C.byref(d), int(device))
        if not self.ptr:
            raise N.Omega4CudaError(f"omega4_octave_create failed: {N.last_error()}")
        self.state_doubles = int(lib.omega4_octave_state_doubles(self.ptr))

    @property
    def launches(self) -> int:
        return int(N.lib().omega4_octave_launches(self.ptr))

    def close(self):
        if self.ptr:
            N.lib().omega4_octave_destroy(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ThirdOctaveMeter:
    """One-third-octave band levels of ``n_rows`` channel rows, fed tile by tile with device tensors.

    ``max_seconds`` sizes the device series ``levels`` ([n_rows, steps, n_bands + 1], one step per completed
    100 ms block).  Rows are independent channels: there is no summation over channels and no weighting."""

    def __init__(self, sample_rate: int, n_rows: int, max_seconds: float, device: int = 0):
        import torch
        fs = tables.check_octave_rate(sample_rate)
        if int(n_rows) < 1:
            raise ValueError("n_rows must be >= 1")
        if not max_seconds > 0:
            raise ValueError("max_seconds must be > 0")
        self._h = _Handle(fs, device)
        self.sample_rate, self.sub, self.n_rows, self.n_bands = fs, fs // 10, int(n_rows), self._h.n_bands
        self.capacity = int(np.ceil(float(max_seconds) * 10 - 1e-9))
        self.dev = torch.device(f"cuda:{device}")
        cols = self.n_bands + 1
        self._levels = torch.full((self.n_rows, self.capacity, cols), float("nan"), dtype=torch.float32, device=self.dev)
        self._leq = torch.full((self.n_rows, cols), float("-inf"), dtype=torch.float32, device=self.dev)
        self._lmax = torch.full_like(self._leq, float("-inf"))
        self._state = torch.zeros((self.n_rows, self._h.state_doubles), dtype=torch.float64, device=self.dev)
        self.samples = 0

    @property
    def frequencies(self) -> np.ndarray:
        """Exact mid-band frequencies 1000 * 10^(x / 10) Hz of the band columns (numpy, n_bands)."""
        return self._h.bands["fm"].copy()

    @property
    def nominal(self) -> np.ndarray:
        """Nominal mid-band frequencies (20, 25, 31.5, ... Hz) of the band columns (numpy, n_bands)."""
        return self._h.bands["nominal"].copy()

    @property
    def steps(self) -> int:
        """Completed 100 ms blocks per row so far."""
        return self.samples // self.sub

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

    @property
    def launches(self) -> int:
        """Kernels this meter's native object has launched (one per push)."""
        return self._h.launches

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
        import torch
        if not isinstance(tile, torch.Tensor) or not tile.is_cuda:
            raise ValueError("tile must be a CUDA tensor")
        if tile.dtype != torch.float32:
            raise ValueError(f"tile must be float32, got {tile.dtype}")
        if tile.dim() != 2 or tile.shape[0] != self.n_rows:
            raise ValueError(f"tile must be [{self.n_rows}, n], got {tuple(tile.shape)}")
        if tile.device != self.dev:
            raise ValueError(f"tile is on {tile.device}, the meter on {self.dev}")
        n = int(tile.shape[1])
        if n == 0:
            return 0
        if tile.stride(1) != 1:
            raise ValueError("tile rows must be contiguous along time")
        j0 = self.samples // self.sub
        done = (self.samples + n) // self.sub - j0
        if j0 + done > self.capacity:
            raise ValueError(f"push would exceed max_seconds ({self.capacity} steps); reset() or size the meter larger")
        s = stream if stream is not None else torch.cuda.current_stream(self.dev).cuda_stream
        cols = self.n_bands + 1
        rc = N.lib().omega4_octave_push(
            self._h.ptr, s, N.MEM_DEVICE, tile.data_ptr(), tile.stride(0), self.n_rows, n, self._state.data_ptr(),
            1 if self.samples == 0 else 0, self.capacity, self._levels.data_ptr() + 4 * j0 * cols,
            self._leq.data_ptr(), self._lmax.data_ptr())
        N.check(rc, "omega4_octave_push")
        self.samples += n
        return done

    def close(self) -> None:
        self._h.close()


def third_octave_levels(x: np.ndarray, sample_rate: int, device: int = 0) -> Dict[str, np.ndarray]:
    """Host convenience: x float32 [n_rows, n] -> numpy ``levels`` [n_rows, n // (sample_rate / 10),
    n_bands + 1], ``leq`` and ``max_level`` [n_rows, n_bands + 1] (dBFS; last column: overall), and the band
    columns' ``frequencies`` and ``nominal`` mid-band frequencies."""
    fs = tables.check_octave_rate(sample_rate)
    x = np.asarray(x)
    if x.dtype != np.float32:
        raise ValueError(f"x must be float32, got {x.dtype}")
    if x.ndim != 2:
        raise ValueError(f"x must be [n_rows, n], got shape {x.shape}")
    n_rows, n = x.shape
    h = _Handle(fs, device)
    try:
        cols = h.n_bands + 1
        xc = np.ascontiguousarray(x)
        steps = n // h.sub
        state = np.zeros((n_rows, h.state_doubles), np.float64)
        levels = np.full((n_rows, steps, cols), np.nan, np.float32)
        leq = np.full((n_rows, cols), -np.inf, np.float32)
        lmax = np.full_like(leq, -np.inf)
        if n_rows and n:
            rc = N.lib().omega4_octave_push(h.ptr, None, N.MEM_HOST, xc.ctypes.data, n, n_rows, n, state.ctypes.data,
                                            1, steps, levels.ctypes.data, leq.ctypes.data, lmax.ctypes.data)
            N.check(rc, "omega4_octave_push")
        return {"levels": levels, "leq": leq, "max_level": lmax, "frequencies": h.bands["fm"].copy(),
                "nominal": h.bands["nominal"].copy()}
    finally:
        h.close()
