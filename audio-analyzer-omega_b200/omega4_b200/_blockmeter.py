"""What the block meters share (``LoudnessMeter``, ``ThirdOctaveMeter``, ``SoundLevelMeter``): the native object,
the fields and checks of a meter fed tile by tile on the 100 ms grid, and the input checks of a push and of the
host conveniences.  The push contract itself is stated once in include/omega4_cuda.h."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as N
from . import tables


class Handle:
    """Owns one native ``omega4_<kind>`` object (kind ``loudness``, ``octave`` or ``slm``) created from ``desc``."""

    def __init__(self, kind: str, desc, device: int):
        lib = N.lib()
        N.require_device()
        self.kind = kind
        self.ptr = getattr(lib, f"omega4_{kind}_create")(C.byref(desc), int(device))
        if not self.ptr:
            raise N.Omega4CudaError(f"omega4_{kind}_create failed: {N.last_error()}")
        self.state_doubles = int(getattr(lib, f"omega4_{kind}_state_doubles")(self.ptr))

    @property
    def launches(self) -> int:
        return int(getattr(N.lib(), f"omega4_{self.kind}_launches")(self.ptr))

    def close(self):
        if self.ptr:
            getattr(N.lib(), f"omega4_{self.kind}_destroy")(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BlockMeter:
    """A meter of ``rows`` channel rows per tile with carried state [state_rows, state_doubles] on ``device``,
    completing one block per ``sub`` = sample_rate / 10 samples, with device series of ``capacity`` blocks
    (``max_seconds``).  ``open_handle(fs, device)`` creates the native object."""

    def __init__(self, open_handle, sample_rate, rows: int, state_rows: int, max_seconds: float, device: int):
        import torch
        fs = tables.check_meter_rate(sample_rate)
        if not max_seconds > 0:
            raise ValueError("max_seconds must be > 0")
        self._h = open_handle(fs, device)
        self.sample_rate, self.sub, self._rows = fs, fs // 10, rows
        self.capacity = int(np.ceil(float(max_seconds) * 10 - 1e-9))
        self.dev = torch.device(f"cuda:{device}")
        self._state = torch.zeros((state_rows, self._h.state_doubles), dtype=torch.float64, device=self.dev)
        self.samples = 0

    @property
    def steps(self) -> int:
        """Completed 100 ms blocks (steps of the series) so far."""
        return self.samples // self.sub

    @property
    def launches(self) -> int:
        """Kernels this meter's native object has launched."""
        return self._h.launches

    def close(self) -> None:
        self._h.close()

    def _stream(self, stream):
        import torch
        return stream if stream is not None else torch.cuda.current_stream(self.dev).cuda_stream

    def _tile(self, tile, stream):
        """Checks a push tile: float32 CUDA tensor [rows, n] on the meter's device, unit stride along time, its
        blocks within capacity.  Returns (n, row stride, first block j0, blocks completed, stream); n = 0 leaves
        nothing to push."""
        import torch
        if not isinstance(tile, torch.Tensor) or not tile.is_cuda:
            raise ValueError("tile must be a CUDA tensor")
        if tile.dtype != torch.float32:
            raise ValueError(f"tile must be float32, got {tile.dtype}")
        if tile.dim() != 2 or tile.shape[0] != self._rows:
            raise ValueError(f"tile must be [{self._rows}, n], got {tuple(tile.shape)}")
        if tile.device != self.dev:
            raise ValueError(f"tile is on {tile.device}, the meter on {self.dev}")
        n = int(tile.shape[1])
        if n == 0:
            return 0, n, 0, 0, None
        if tile.stride(1) != 1:
            raise ValueError("tile rows must be contiguous along time")
        j0 = self.samples // self.sub
        done = (self.samples + n) // self.sub - j0
        if j0 + done > self.capacity:
            raise ValueError(f"push would exceed max_seconds ({self.capacity} steps); reset() or size the meter larger")
        row_stride = tile.stride(0) if self._rows > 1 else n        # torch gives a single row any stride, even 0
        return n, row_stride, j0, done, self._stream(stream)


def host_input(x, ndim: int, shape: str) -> np.ndarray:
    """x as a C-contiguous float32 numpy array of ``ndim`` dimensions, named ``shape`` in the error."""
    x = np.asarray(x)
    if x.dtype != np.float32:
        raise ValueError(f"x must be float32, got {x.dtype}")
    if x.ndim != ndim:
        raise ValueError(f"x must be {shape}, got shape {x.shape}")
    return np.ascontiguousarray(x)
