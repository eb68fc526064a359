"""ITU-R BS.1770-4 program loudness and EBU Tech 3342 loudness range per stream, on the GPU.

An extension outside reference parity: OMEGA-4's ``ProfessionalMetering`` is not textbook BS.1770
(SURVEY.md section 0.2) and stays exactly as it is in ``AnalysisPlan`` / the five-column ``meters``.
This module measures what broadcast and streaming pipelines normalise to: per stream of C channels,
K-weighted sub-block energies summed over the channels with the layout's weights, momentary (400 ms)
and short-term (3 s) loudness every 100 ms, the gated integrated loudness, the loudness range and the
per-channel sample peak.  Definitions: DESIGN.md section 4.7.  All arithmetic runs in libomega4_cuda
(``omega4_loudness_*``); there is no CPU fallback.

    meter = LoudnessMeter(48000, "stereo", n_streams=1024, max_seconds=600)
    meter.push(tile)              # float32 CUDA tensor [n_streams * C, n], e.g. StreamBatch.tile_view(n_hops)
    meter.momentary               # [n_streams, steps] device tensor (LUFS)
    meter.summary()               # {"integrated", "lra", "max_momentary", "max_short_term", "sample_peak"}
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Sequence, Union

import numpy as np

from . import _native as N
from . import tables

SUMMARY_KEYS = ("integrated", "lra", "max_momentary", "max_short_term")


def _check_rate(sample_rate) -> int:
    fs = int(sample_rate)
    if fs != sample_rate or fs <= 0 or fs % 10:
        raise ValueError(f"sample rate {sample_rate} must be a positive integer multiple of 10 (100 ms sub-blocks)")
    return fs


class _Handle:
    """Owns one omega4_loudness object (sample rate, channel weights, K-weighting coefficients)."""

    def __init__(self, sample_rate: int, weights: np.ndarray, device: int):
        lib = N.lib()
        N.require_device()
        self.sample_rate, self.sub, self.channels = sample_rate, sample_rate // 10, int(weights.size)
        if self.channels > N.LOUDNESS_MAX_CH:
            raise ValueError(f"at most {N.LOUDNESS_MAX_CH} channels per stream, got {self.channels}")
        self._w = np.ascontiguousarray(weights, dtype=np.float64)
        self._k = [np.ascontiguousarray(c, dtype=np.float64) for c in tables.bs1770_k_weighting(sample_rate)]
        dp = C.POINTER(C.c_double)
        d = N.LoudnessDesc()
        d.sample_rate, d.channels, d.sub = sample_rate, self.channels, self.sub
        d.ch_weights = self._w.ctypes.data_as(dp)
        d.shelf_b, d.shelf_a, d.hp_b, d.hp_a = (k.ctypes.data_as(dp) for k in self._k)
        self.ptr = lib.omega4_loudness_create(C.byref(d), int(device))
        if not self.ptr:
            raise N.Omega4CudaError(f"omega4_loudness_create failed: {N.last_error()}")
        self.state_doubles = int(lib.omega4_loudness_state_doubles(self.ptr))

    @property
    def launches(self) -> int:
        return int(N.lib().omega4_loudness_launches(self.ptr))

    def close(self):
        if self.ptr:
            N.lib().omega4_loudness_destroy(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _summary_dict(out: np.ndarray, peak_db: np.ndarray) -> Dict[str, np.ndarray]:
    d = {k: out[:, i].copy() for i, k in enumerate(SUMMARY_KEYS)}
    d["sample_peak"] = peak_db
    return d


class LoudnessMeter:
    """Program loudness of ``n_streams`` streams of the same layout, fed tile by tile with device tensors.

    ``layout_or_weights``: "mono", "stereo", "5.1" (L R C LFE Ls Rs) or an explicit list of C channel
    weights (7.1 and other layouts).  ``max_seconds`` sizes the device series ``momentary`` / ``short_term``
    ([n_streams, steps], one step per completed 100 ms sub-block, NaN until the 400 ms / 3 s window fills)."""

    def __init__(self, sample_rate: int, layout_or_weights: Union[str, Sequence[float]], n_streams: int,
                 max_seconds: float, device: int = 0):
        import torch
        fs = _check_rate(sample_rate)
        w = tables.bs1770_channel_weights(layout_or_weights)
        if int(n_streams) < 1:
            raise ValueError("n_streams must be >= 1")
        if not max_seconds > 0:
            raise ValueError("max_seconds must be > 0")
        self._h = _Handle(fs, w, device)
        self.sample_rate, self.sub, self.channels, self.n_streams = fs, fs // 10, int(w.size), int(n_streams)
        self.capacity = int(np.ceil(float(max_seconds) * 10 - 1e-9))
        self.dev = torch.device(f"cuda:{device}")
        self._series_m = torch.full((self.n_streams, self.capacity), float("nan"), dtype=torch.float32, device=self.dev)
        self._series_s = torch.full_like(self._series_m, float("nan"))
        self._state = torch.zeros((self.n_streams, self._h.state_doubles), dtype=torch.float64, device=self.dev)
        self._peak = torch.full((self.n_streams, self.channels), float("-inf"), dtype=torch.float32, device=self.dev)
        self._out = torch.empty((self.n_streams, 4), dtype=torch.float32, device=self.dev)
        self.samples = 0

    @property
    def steps(self) -> int:
        """Completed 100 ms sub-blocks per stream so far."""
        return self.samples // self.sub

    @property
    def momentary(self):
        return self._series_m[:, :self.steps]

    @property
    def short_term(self):
        return self._series_s[:, :self.steps]

    @property
    def sample_peak(self):
        """[n_streams, C] device tensor: 20 log10(max |x|) in dBFS over everything pushed since the last reset
        (-inf for silence and before the first push)."""
        return self._peak

    @property
    def launches(self) -> int:
        """Kernels this meter's native object has launched (two per push, one per summary)."""
        return self._h.launches

    def reset(self) -> None:
        """Start every stream anew: the next push ignores the carried state and rewrites the series from step 0;
        the sample peaks read -inf until then."""
        self.samples = 0
        self._peak.fill_(float("-inf"))

    def push(self, tile, stream=None) -> int:
        """Continue every stream by ``tile``: float32 CUDA tensor [n_streams * C, n] (rows stream-major,
        unit stride along time, any row stride -- ``StreamBatch.tile_view`` qualifies).  Asynchronous on
        ``stream`` (default: torch's current stream).  Returns the number of steps this push completed."""
        import torch
        if not isinstance(tile, torch.Tensor) or not tile.is_cuda:
            raise ValueError("tile must be a CUDA tensor")
        if tile.dtype != torch.float32:
            raise ValueError(f"tile must be float32, got {tile.dtype}")
        if tile.dim() != 2 or tile.shape[0] != self.n_streams * self.channels:
            raise ValueError(f"tile must be [{self.n_streams * self.channels}, n], got {tuple(tile.shape)}")
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
        rc = N.lib().omega4_loudness_push(
            self._h.ptr, s, N.MEM_DEVICE, tile.data_ptr(), tile.stride(0), self.n_streams, n,
            self._state.data_ptr(), 1 if self.samples == 0 else 0, self.capacity,
            self._series_m.data_ptr() + 4 * j0, self._series_s.data_ptr() + 4 * j0, self._peak.data_ptr())
        N.check(rc, "omega4_loudness_push")
        self.samples += n
        return done

    def summary(self, stream=None) -> Dict[str, np.ndarray]:
        """Per stream (numpy arrays): ``integrated`` (LUFS, -inf when no block passes the gates), ``lra`` (LU),
        ``max_momentary``, ``max_short_term`` (NaN while undefined) and ``sample_peak`` [n_streams, C] (dBFS)."""
        import torch
        s = stream if stream is not None else torch.cuda.current_stream(self.dev).cuda_stream
        rc = N.lib().omega4_loudness_summary(self._h.ptr, s, N.MEM_DEVICE, self._series_m.data_ptr(),
                                             self._series_s.data_ptr(), self.n_streams, self.steps, self.capacity,
                                             self._out.data_ptr())
        N.check(rc, "omega4_loudness_summary")
        return _summary_dict(self._out.cpu().numpy(), self._peak.cpu().numpy())

    def close(self) -> None:
        self._h.close()


def program_loudness(x: np.ndarray, sample_rate: int, layout: Union[str, Sequence[float]] = "stereo",
                     device: int = 0) -> Dict[str, np.ndarray]:
    """Host convenience: x float32 [n_streams, C, n] -> the ``LoudnessMeter.summary`` dict plus the
    ``momentary`` / ``short_term`` series [n_streams, n // (sample_rate / 10)] as numpy arrays."""
    fs = _check_rate(sample_rate)
    x = np.asarray(x)
    if x.dtype != np.float32:
        raise ValueError(f"x must be float32, got {x.dtype}")
    if x.ndim != 3:
        raise ValueError(f"x must be [n_streams, C, n], got shape {x.shape}")
    n_streams, n_ch, n = x.shape
    w = tables.bs1770_channel_weights(layout, n_ch)
    h = _Handle(fs, w, device)
    try:
        xc = np.ascontiguousarray(x).reshape(n_streams * n_ch, n)
        steps = n // h.sub
        state = np.zeros((n_streams, h.state_doubles), np.float64)
        mom = np.full((n_streams, steps), np.nan, np.float32)
        sht = np.full_like(mom, np.nan)
        peak = np.full((n_streams, n_ch), -np.inf, np.float32)
        lib = N.lib()
        if n_streams and n:
            rc = lib.omega4_loudness_push(h.ptr, None, N.MEM_HOST, xc.ctypes.data, n, n_streams, n, state.ctypes.data,
                                          1, steps, mom.ctypes.data, sht.ctypes.data, peak.ctypes.data)
            N.check(rc, "omega4_loudness_push")
        out = np.empty((n_streams, 4), np.float32)
        rc = lib.omega4_loudness_summary(h.ptr, None, N.MEM_HOST, mom.ctypes.data, sht.ctypes.data, n_streams, steps,
                                         steps, out.ctypes.data)
        N.check(rc, "omega4_loudness_summary")
    finally:
        h.close()
    d = _summary_dict(out, peak)
    d["momentary"], d["short_term"] = mom, sht
    return d
