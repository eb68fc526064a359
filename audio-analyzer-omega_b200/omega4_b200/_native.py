"""ctypes binding of libomega4_cuda.so (C ABI: include/omega4_cuda.h).

There is no CPU fallback anywhere in this package: if the library is missing, cannot be loaded
or reports no CUDA device, the call raises ``Omega4CudaError``.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from typing import Optional, Sequence

import numpy as np

LIB_NAME = "libomega4_cuda.so"
#: OMEGA4_CUDA_LIB: developer override for A/B measurements of two builds on the same box
LIB_PATH = os.environ.get("OMEGA4_CUDA_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), LIB_NAME)

OK = 0
MEM_HOST = 0
MEM_DEVICE = 1
MAX_RES = 8
METER_WINDOW = 2048
METER_STATE_DOUBLES = 8 + 3600 + 60
N_METERS = 5
FLAG_TIME_KERNELS = 1
FLAG_FRESH_METERS = 2
FLAG_CONCURRENT_METERS = 4
FLAG_NO_BLOCKDFT = 8
FLAG_NO_TENSOR = 16
FLAG_TENSOR = 32
FLAG_SERIAL_STATS = 64
FLAG_FRESH_BARS = 128
FLAG_EXACT_TRUE_PEAK = 256
ABI_VERSION = 4
WATERFALL_STATE = 41
LOUDNESS_MAX_CH = 32
OCTAVE_MAX_BANDS = 31

#: every symbol include/omega4_cuda.h declares (checked by tests/test_abi_symbols.py)
EXPORTS = (
    "omega4_abi_version", "omega4_last_error", "omega4_device_count",
    "omega4_plan_create", "omega4_plan_destroy", "omega4_analyze", "omega4_combine",
    "omega4_meter_frames", "omega4_meter_stats", "omega4_rfft_batch", "omega4_band_map",
    "omega4_synth_fill", "omega4_plan_launches", "omega4_plan_kernel_times",
    "omega4_analyze_s16", "omega4_plan_set_weighting", "omega4_bass_bars", "omega4_bars_create", "omega4_bars_destroy", "omega4_bars_count", "omega4_bars_run",
    "omega4_waterfall", "omega4_plan_set_gate_threshold",
    "omega4_analyze_io", "omega4_stream_hop", "omega4_meter_update",
    "omega4_loudness_create", "omega4_loudness_destroy", "omega4_loudness_state_doubles",
    "omega4_loudness_push", "omega4_loudness_summary", "omega4_loudness_launches",
    "omega4_octave_create", "omega4_octave_destroy", "omega4_octave_state_doubles", "omega4_octave_push",
    "omega4_octave_launches",
)


class Omega4CudaError(RuntimeError):
    pass


class PlanDesc(C.Structure):
    _fields_ = [
        ("sample_rate", C.c_int), ("hop", C.c_int), ("n_res", C.c_int),
        ("fft_sizes", C.POINTER(C.c_int)),
        ("windows", C.POINTER(C.c_float)),
        ("bin_weights", C.POINTER(C.c_float)),
        ("target_bins", C.c_int),
        ("tb_count", C.POINTER(C.c_int)),
        ("tb_idx", C.POINTER(C.c_int)),
        ("tb_lo", C.POINTER(C.c_int)),
        ("tb_frac", C.POINTER(C.c_float)),
        ("res_weight", C.POINTER(C.c_float)),
        ("meter_window", C.c_int),
        ("meter_hann", C.POINTER(C.c_double)),
        ("kw_coeffs", C.POINTER(C.c_double)),
        ("gate_threshold", C.c_double),
    ]


class Weighting(C.Structure):
    _fields_ = [
        ("n_sections", C.c_int), ("order", C.c_int * 4),
        ("b", (C.c_double * 3) * 4), ("a", (C.c_double * 3) * 4),
        ("blend", C.c_int), ("rms_gate", C.c_int), ("gain", C.c_double),
    ]


class BarsDesc(C.Structure):
    _fields_ = [
        ("spectrum_len", C.c_int), ("n_bars", C.c_int),
        ("bands", C.POINTER(C.c_int)),
        ("gain", C.POINTER(C.c_float)),
        ("smooth", C.POINTER(C.c_double)),
        ("percentile", C.c_double),
        ("scale", C.c_float),
        ("normalize_max", C.c_int),
    ]


class LoudnessDesc(C.Structure):
    """omega4_loudness_desc (include/omega4_cuda.h)."""
    _fields_ = [
        ("sample_rate", C.c_int), ("channels", C.c_int), ("ch_weights", C.POINTER(C.c_double)),
        ("shelf_b", C.POINTER(C.c_double)), ("shelf_a", C.POINTER(C.c_double)),
        ("hp_b", C.POINTER(C.c_double)), ("hp_a", C.POINTER(C.c_double)),
        ("sub", C.c_int),
    ]


class OctaveDesc(C.Structure):
    """omega4_octave_desc (include/omega4_cuda.h)."""
    _fields_ = [
        ("sample_rate", C.c_int), ("n_bands", C.c_int), ("sos", C.POINTER(C.c_double)), ("sub", C.c_int),
    ]


class IO(C.Structure):
    """omega4_io (include/omega4_cuda.h)."""
    _fields_ = [
        ("samples", C.c_void_p), ("frames_s16", C.c_void_p), ("n_interleaved", C.c_int),
        ("stride", C.c_longlong), ("n_ch", C.c_int), ("n_hops", C.c_int), ("hist", C.c_int),
        ("combined", C.c_void_p), ("magnitudes", C.POINTER(C.c_void_p)), ("meters", C.c_void_p),
        ("lufs_inst", C.c_void_p), ("tp_db", C.c_void_p), ("meter_state", C.c_void_p),
        ("bars", C.c_void_p), ("band_values", C.c_void_p), ("peak_values", C.c_void_p), ("bars_state", C.c_void_p),
        ("flags", C.c_int),
    ]


_lib = None
_lock = threading.Lock()


def lib() -> C.CDLL:
    """Load (once) and return the library; raises Omega4CudaError when it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise Omega4CudaError(
                f"{LIB_PATH} is missing -- build it with `python audio-analyzer-omega_b200/build.py` "
                "(nvcc, sm_100a). omega4_b200 has no CPU fallback.")
        try:
            l = C.CDLL(LIB_PATH)
        except OSError as e:
            raise Omega4CudaError(f"cannot load {LIB_PATH}: {e}") from e
        vp, ip, ll = C.c_void_p, C.c_int, C.c_longlong
        l.omega4_abi_version.restype = ip
        l.omega4_last_error.restype = C.c_char_p
        l.omega4_device_count.restype = ip
        l.omega4_plan_create.restype = vp
        l.omega4_plan_create.argtypes = [C.POINTER(PlanDesc), ip]
        l.omega4_plan_destroy.restype = None
        l.omega4_plan_destroy.argtypes = [vp]
        l.omega4_analyze.restype = ip
        l.omega4_analyze.argtypes = [vp, vp, ip, vp, ll, ip, ip, ip, vp, C.POINTER(vp), vp, vp, vp, vp, ip]
        l.omega4_analyze_s16.restype = ip
        l.omega4_analyze_s16.argtypes = [vp, vp, ip, vp, ll, ip, ip, ip, ip, vp, C.POINTER(vp), vp, vp, vp, vp, ip]
        l.omega4_plan_set_weighting.restype = ip
        l.omega4_plan_set_weighting.argtypes = [vp, C.POINTER(Weighting)]
        l.omega4_combine.restype = ip
        l.omega4_combine.argtypes = [vp, vp, ip, C.POINTER(vp), ip, vp]
        l.omega4_meter_frames.restype = ip
        l.omega4_meter_frames.argtypes = [vp, vp, ip, vp, ip, vp, vp, vp]
        l.omega4_meter_stats.restype = ip
        l.omega4_meter_stats.argtypes = [vp, vp, ip, vp, vp, ip, ip, ip, vp, vp, ip]
        l.omega4_rfft_batch.restype = ip
        l.omega4_rfft_batch.argtypes = [ip, vp, ip, vp, ip, ip, vp, vp, vp]
        l.omega4_band_map.restype = ip
        l.omega4_band_map.argtypes = [ip, vp, ip, vp, ip, ip, vp, ip, vp, vp, ip]
        l.omega4_analyze_io.restype = ip
        l.omega4_analyze_io.argtypes = [vp, vp, ip, C.POINTER(IO)]
        l.omega4_stream_hop.restype = ip
        l.omega4_stream_hop.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), vp]
        l.omega4_meter_update.restype = ip
        l.omega4_meter_update.argtypes = [vp, vp, vp, ip, vp, vp, vp]
        l.omega4_waterfall.restype = ip
        l.omega4_waterfall.argtypes = [ip, vp, ip, vp, ip, ip, ip, ip, ip, ip, ip, C.c_float, vp, ip, vp, vp, vp]
        l.omega4_plan_set_gate_threshold.restype = ip
        l.omega4_plan_set_gate_threshold.argtypes = [vp, C.c_double]
        l.omega4_bass_bars.restype = ip
        l.omega4_bass_bars.argtypes = [ip, vp, ip, vp, ip, ip, ip, vp, vp, ip, vp, vp]
        l.omega4_synth_fill.restype = ip
        l.omega4_synth_fill.argtypes = [ip, vp, vp, ip, ip, ll, ll, ip, ip, ll]
        l.omega4_plan_launches.restype = ll
        l.omega4_plan_launches.argtypes = [vp]
        l.omega4_plan_kernel_times.restype = ip
        l.omega4_plan_kernel_times.argtypes = [vp, vp, vp, ip]
        l.omega4_bars_create.restype = vp
        l.omega4_bars_create.argtypes = [C.POINTER(BarsDesc), ip]
        l.omega4_bars_destroy.restype = None
        l.omega4_bars_destroy.argtypes = [vp]
        l.omega4_bars_count.restype = ip
        l.omega4_bars_count.argtypes = [vp]
        l.omega4_bars_run.restype = ip
        l.omega4_bars_run.argtypes = [vp, vp, ip, vp, ip, ip, vp, ip, vp, vp]
        l.omega4_loudness_create.restype = vp
        l.omega4_loudness_create.argtypes = [C.POINTER(LoudnessDesc), ip]
        l.omega4_loudness_destroy.restype = None
        l.omega4_loudness_destroy.argtypes = [vp]
        l.omega4_loudness_state_doubles.restype = ip
        l.omega4_loudness_state_doubles.argtypes = [vp]
        l.omega4_loudness_push.restype = ip
        l.omega4_loudness_push.argtypes = [vp, vp, ip, vp, ll, ip, ll, vp, ip, ll, vp, vp, vp]
        l.omega4_loudness_summary.restype = ip
        l.omega4_loudness_summary.argtypes = [vp, vp, ip, vp, vp, ip, ip, ll, vp]
        l.omega4_loudness_launches.restype = ll
        l.omega4_loudness_launches.argtypes = [vp]
        l.omega4_octave_create.restype = vp
        l.omega4_octave_create.argtypes = [C.POINTER(OctaveDesc), ip]
        l.omega4_octave_destroy.restype = None
        l.omega4_octave_destroy.argtypes = [vp]
        l.omega4_octave_state_doubles.restype = ip
        l.omega4_octave_state_doubles.argtypes = [vp]
        l.omega4_octave_push.restype = ip
        l.omega4_octave_push.argtypes = [vp, vp, ip, vp, ll, ip, ll, vp, ip, ll, vp, vp, vp]
        l.omega4_octave_launches.restype = ll
        l.omega4_octave_launches.argtypes = [vp]
        if l.omega4_abi_version() != ABI_VERSION:
            raise Omega4CudaError(f"{LIB_NAME} ABI {l.omega4_abi_version()} != binding ABI {ABI_VERSION}")
        _lib = l
    return _lib


def last_error() -> str:
    return lib().omega4_last_error().decode("utf-8", "replace")


def check(rc: int, what: str = "omega4_cuda") -> None:
    if rc != OK:
        raise Omega4CudaError(f"{what} failed ({rc}): {last_error()}")


def require_device() -> int:
    n = lib().omega4_device_count()
    if n < 1:
        raise Omega4CudaError("no CUDA device visible: omega4_b200 has no CPU fallback")
    return n


def ptr(a) -> Optional[int]:
    """Address of a numpy array / torch tensor / None."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        return a.data_ptr()
    if isinstance(a, int):
        return a
    raise TypeError(f"cannot take the address of {type(a)}")


_DT = {"float32": 4, "float64": 8, "int16": 2, "int32": 4}


def checked(a, dtype: str, n_elems: Optional[int] = None, what: str = "buffer") -> Optional[int]:
    """Address of a numpy array / torch tensor after checking what the C side takes on trust: element type,
    C-contiguity and (when given) the element count.  None passes through."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        ok_dt, contiguous, count = a.dtype == np.dtype(dtype), a.flags["C_CONTIGUOUS"], a.size
    elif hasattr(a, "data_ptr"):
        ok_dt, contiguous, count = str(a.dtype).endswith(dtype), a.is_contiguous(), a.numel()
    else:
        raise TypeError(f"{what}: cannot take the address of {type(a)}")
    if not ok_dt:
        raise Omega4CudaError(f"{what} must be {dtype}, got {a.dtype}")
    if not contiguous:
        raise Omega4CudaError(f"{what} must be C-contiguous")
    if n_elems is not None and count < n_elems:
        raise Omega4CudaError(f"{what} holds {count} elements, the call needs {n_elems}")
    return ptr(a)


def ptr_array(items: Sequence) -> "C.Array":
    arr = (C.c_void_p * len(items))()
    for i, it in enumerate(items):
        arr[i] = ptr(it)
    return arr
