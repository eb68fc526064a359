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
from ._blockmeter import BlockMeter, Handle, host_input
from .tables import check_meter_rate as _check_rate

SUMMARY_KEYS = ("integrated", "lra", "max_momentary", "max_short_term")


class _Handle(Handle):
    """Owns one omega4_loudness object (sample rate, channel weights, K-weighting coefficients)."""

    def __init__(self, sample_rate: int, weights: np.ndarray, device: int):
        if weights.size > N.LOUDNESS_MAX_CH:
            raise ValueError(f"at most {N.LOUDNESS_MAX_CH} channels per stream, got {weights.size}")
        w = np.ascontiguousarray(weights, dtype=np.float64)
        k = [np.ascontiguousarray(c, dtype=np.float64) for c in tables.bs1770_k_weighting(sample_rate)]
        dp = C.POINTER(C.c_double)
        d = N.LoudnessDesc(sample_rate, w.size, w.ctypes.data_as(dp), *(c.ctypes.data_as(dp) for c in k),
                           sample_rate // 10)
        super().__init__("loudness", d, device)


def _summary_dict(out: np.ndarray, peak_db: np.ndarray) -> Dict[str, np.ndarray]:
    d = {k: out[:, i].copy() for i, k in enumerate(SUMMARY_KEYS)}
    d["sample_peak"] = peak_db
    return d


class LoudnessMeter(BlockMeter):
    """Program loudness of ``n_streams`` streams of the same layout, fed tile by tile with device tensors.

    ``layout_or_weights``: "mono", "stereo", "5.1" (L R C LFE Ls Rs) or an explicit list of C channel
    weights (7.1 and other layouts).  ``max_seconds`` sizes the device series ``momentary`` / ``short_term``
    ([n_streams, steps], one step per completed 100 ms sub-block, NaN until the 400 ms / 3 s window fills).
    ``launches`` counts two kernels per push and one per summary."""

    def __init__(self, sample_rate: int, layout_or_weights: Union[str, Sequence[float]], n_streams: int,
                 max_seconds: float, device: int = 0):
        import torch
        w = tables.bs1770_channel_weights(layout_or_weights)
        if int(n_streams) < 1:
            raise ValueError("n_streams must be >= 1")
        self.channels, self.n_streams = int(w.size), int(n_streams)
        super().__init__(lambda fs, dev: _Handle(fs, w, dev), sample_rate, self.n_streams * self.channels,
                         self.n_streams, max_seconds, device)
        self._series_m = torch.full((self.n_streams, self.capacity), float("nan"), dtype=torch.float32, device=self.dev)
        self._series_s = torch.full_like(self._series_m, float("nan"))
        self._peak = torch.full((self.n_streams, self.channels), float("-inf"), dtype=torch.float32, device=self.dev)
        self._out = torch.empty((self.n_streams, 4), dtype=torch.float32, device=self.dev)

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

    def reset(self) -> None:
        """Start every stream anew: the next push ignores the carried state and rewrites the series from step 0;
        the sample peaks read -inf until then."""
        self.samples = 0
        self._peak.fill_(float("-inf"))

    def push(self, tile, stream=None) -> int:
        """Continue every stream by ``tile``: float32 CUDA tensor [n_streams * C, n] (rows stream-major,
        unit stride along time, any row stride -- ``StreamBatch.tile_view`` qualifies).  Asynchronous on
        ``stream`` (default: torch's current stream).  Returns the number of steps this push completed."""
        n, row_stride, j0, done, s = self._tile(tile, stream)
        if n == 0:
            return 0
        rc = N.lib().omega4_loudness_push(
            self._h.ptr, s, N.MEM_DEVICE, tile.data_ptr(), row_stride, self.n_streams, n,
            self._state.data_ptr(), 1 if self.samples == 0 else 0, self.capacity,
            self._series_m.data_ptr() + 4 * j0, self._series_s.data_ptr() + 4 * j0, self._peak.data_ptr())
        N.check(rc, "omega4_loudness_push")
        self.samples += n
        return done

    def summary(self, stream=None) -> Dict[str, np.ndarray]:
        """Per stream (numpy arrays): ``integrated`` (LUFS, -inf when no block passes the gates), ``lra`` (LU),
        ``max_momentary``, ``max_short_term`` (NaN while undefined) and ``sample_peak`` [n_streams, C] (dBFS)."""
        rc = N.lib().omega4_loudness_summary(self._h.ptr, self._stream(stream), N.MEM_DEVICE,
                                             self._series_m.data_ptr(), self._series_s.data_ptr(), self.n_streams,
                                             self.steps, self.capacity, self._out.data_ptr())
        N.check(rc, "omega4_loudness_summary")
        return _summary_dict(self._out.cpu().numpy(), self._peak.cpu().numpy())


def program_loudness(x: np.ndarray, sample_rate: int, layout: Union[str, Sequence[float]] = "stereo",
                     device: int = 0) -> Dict[str, np.ndarray]:
    """Host convenience: x float32 [n_streams, C, n] -> the ``LoudnessMeter.summary`` dict plus the
    ``momentary`` / ``short_term`` series [n_streams, n // (sample_rate / 10)] as numpy arrays."""
    fs = _check_rate(sample_rate)
    x = host_input(x, 3, "[n_streams, C, n]")
    n_streams, n_ch, n = x.shape
    w = tables.bs1770_channel_weights(layout, n_ch)
    h = _Handle(fs, w, device)
    try:
        xc = x.reshape(n_streams * n_ch, n)
        steps = n // (fs // 10)
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
