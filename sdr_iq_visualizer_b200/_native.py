"""ctypes binding of libspx (include/spx.h) -- the only door from Python to the CUDA kernels.

There is no CPU fallback: if the shared library cannot be loaded, or no CUDA device is present,
every compute entry point raises :class:`SpectralError`.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.environ.get("SPX_LIB") or os.path.join(CSRC, "libspx.so")   # SPX_LIB: an alternative build (kernel experiments)

OK, E_INVALID, E_CUDA, E_NOMEM, E_UNSUPPORTED, E_NODEVICE, E_BUSY = 0, -1, -2, -3, -4, -5, -6
WINDOW_RECT, WINDOW_HANN, WINDOW_BLACKMAN = 0, 1, 2
FMT_CF32, FMT_CI16 = 0, 1
MEM_HOST, MEM_DEVICE = 0, 1


class SpectralError(RuntimeError):
    """A libspx call failed (CUDA fault, bad argument, no device ...).  Deliberately NOT an OSError:
    the reference streamer treats OSError/Exception inside its read loop as a radio fault
    (/root/reference/app/sdr/streamer.py:134-174); callers can tell this one apart."""

    def __init__(self, code: int, message: str):
        super().__init__(f"libspx error {code}: {message}")
        self.code = code


class spx_device_info(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("sm_count", C.c_int32), ("cc_major", C.c_int32), ("cc_minor", C.c_int32),
                ("l2_bytes", C.c_int32), ("max_smem_optin", C.c_int32), ("total_mem", C.c_int64), ("name", C.c_char * 64)]


class spx_plan_config(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("device", C.c_int32), ("nfft", C.c_int32), ("hop", C.c_int32),
                ("window", C.c_int32), ("in_fmt", C.c_int32), ("in_scale", C.c_float), ("db_eps", C.c_float),
                ("variant", C.c_int32), ("reserved", C.c_int32)]


class spx_stft_args(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("mem", C.c_int32), ("in_", C.c_void_p), ("n_samples", C.c_int64),
                ("stream_stride", C.c_int64), ("n_streams", C.c_int32), ("accumulate", C.c_int32),
                ("db_rows", C.c_void_p), ("wf_rows", C.c_void_p), ("spec_rows", C.c_void_p),
                ("welch_acc", C.c_void_p), ("maxhold", C.c_void_p), ("vmin", C.c_float), ("vmax", C.c_float),
                ("stream", C.c_void_p), ("n_frames_out", C.c_int64), ("h2d_bytes_out", C.c_int64),
                ("d2h_bytes_out", C.c_int64), ("peer_outputs", C.c_int32), ("reserved", C.c_int32)]


class spx_pool_args(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("mode", C.c_int32), ("frames_per_row", C.c_int64),
                ("bins_per_col", C.c_int32), ("reserved", C.c_int32), ("first_frame", C.c_int64), ("n_rows", C.c_int64),
                ("acc", C.c_void_p)]


POOL_MEAN, POOL_MAX = 0, 1


class spx_ddc_config(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("device", C.c_int32), ("in_fmt", C.c_int32), ("in_scale", C.c_float),
                ("decim", C.c_int32), ("n_taps", C.c_int32), ("taps", C.c_void_p), ("phase_inc", C.c_int64)]


class spx_chan_config(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("device", C.c_int32), ("in_fmt", C.c_int32), ("in_scale", C.c_float),
                ("n_channels", C.c_int32), ("decim", C.c_int32), ("n_taps", C.c_int32), ("taps", C.c_void_p)]


class spx_features(C.Structure):
    _fields_ = [("n", C.c_int32), ("argmax", C.c_int32), ("peak_db", C.c_double), ("noise_floor_db", C.c_double),
                ("snr_db", C.c_double), ("adaptive_thr", C.c_double), ("p20_lo", C.c_double), ("p20_hi", C.c_double),
                ("min_distance_bins", C.c_int32), ("first_3db", C.c_int32), ("last_3db", C.c_int32),
                ("first_10db", C.c_int32), ("last_10db", C.c_int32), ("first_20db", C.c_int32),
                ("last_20db", C.c_int32), ("simple_first", C.c_int32), ("simple_last", C.c_int32),
                ("flatness", C.c_double), ("kurtosis", C.c_double), ("mean_db", C.c_double), ("std_db", C.c_double),
                ("n_candidates", C.c_int32), ("peak_count", C.c_int32), ("peak_spacing_std_bins", C.c_double),
                ("peaks_stored", C.c_int32), ("reserved", C.c_int32)]


class spx_region(C.Structure):
    _fields_ = [("row0", C.c_int32), ("row1", C.c_int32), ("col0", C.c_int32), ("col1", C.c_int32), ("n_cells", C.c_int64),
                ("peak_row", C.c_int32), ("peak_col", C.c_int32), ("peak_db", C.c_double), ("peak_floor_db", C.c_double),
                ("power_sum", C.c_double)]


class spx_ring_config(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("n_slots", C.c_int32), ("slot_samples", C.c_int64),
                ("want_wf_rows", C.c_int32), ("want_db_rows", C.c_int32), ("want_welch", C.c_int32),
                ("want_maxhold", C.c_int32), ("vmin", C.c_float), ("vmax", C.c_float), ("want_features", C.c_int32),
                ("reserved", C.c_int32), ("sample_rate", C.c_double)]


class spx_ring_result(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("reserved", C.c_int32), ("seq", C.c_int64), ("n_frames", C.c_int64),
                ("first_frame", C.c_int64), ("wf_rows", C.c_void_p), ("db_rows", C.c_void_p), ("welch_acc", C.c_void_p),
                ("maxhold", C.c_void_p), ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64), ("pxx_db", C.c_void_p),
                ("features", C.c_void_p)]


class spx_ring_stats_t(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("in_flight", C.c_int32), ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64),
                ("samples", C.c_int64), ("frames", C.c_int64), ("reserved", C.c_int64)]


class spx_feature_opts(C.Structure):
    _fields_ = [("drop_db", C.c_double * 3), ("peak_threshold_db", C.c_double), ("use_peak_threshold", C.c_int32),
                ("min_distance_bins", C.c_int32)]


# name -> (restype, argtypes); must list every symbol include/spx.h declares (tests check this)
_SIGNATURES = {
    "spx_abi_version": (C.c_int, []),
    "spx_last_error": (C.c_char_p, []),
    "spx_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "spx_get_device_info": (C.c_int, [C.c_int, C.POINTER(spx_device_info)]),
    "spx_frame_count": (C.c_int64, [C.c_int64, C.c_int32, C.c_int32]),
    "spx_host_alloc": (C.c_int, [C.POINTER(C.c_void_p), C.c_size_t]),
    "spx_host_alloc_wc": (C.c_int, [C.POINTER(C.c_void_p), C.c_size_t]),
    "spx_host_free": (C.c_int, [C.c_void_p]),
    "spx_host_register": (C.c_int, [C.c_void_p, C.c_size_t]),
    "spx_host_unregister": (C.c_int, [C.c_void_p]),
    "spx_device_alloc": (C.c_int, [C.c_int, C.POINTER(C.c_void_p), C.c_size_t]),
    "spx_device_free": (C.c_int, [C.c_int, C.c_void_p]),
    "spx_memcpy_h2d": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_size_t]),
    "spx_memcpy_d2h": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_size_t]),
    "spx_memcpy_d2h_async": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "spx_memset": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.c_size_t]),
    "spx_device_sync": (C.c_int, [C.c_int]),
    "spx_plan_create": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(spx_plan_config)]),
    "spx_plan_destroy": (C.c_int, [C.c_void_p]),
    "spx_plan_sync": (C.c_int, [C.c_void_p]),
    "spx_stft_exec": (C.c_int, [C.c_void_p, C.POINTER(spx_stft_args)]),
    "spx_stft_exec_persistence": (C.c_int, [C.c_void_p, C.POINTER(spx_stft_args), C.c_void_p]),
    "spx_stft_exec_pooled": (C.c_int, [C.c_void_p, C.POINTER(spx_stft_args), C.POINTER(spx_pool_args)]),
    "spx_pool_finalize": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int64, C.c_int64,
                                    C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_void_p]),
    "spx_ddc_create": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(spx_ddc_config)]),
    "spx_ddc_destroy": (C.c_int, [C.c_void_p]),
    "spx_ddc_sync": (C.c_int, [C.c_void_p]),
    "spx_ddc_exec": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.POINTER(C.c_int64),
                               C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.c_void_p]),
    "spx_chan_create": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(spx_chan_config)]),
    "spx_chan_destroy": (C.c_int, [C.c_void_p]),
    "spx_chan_sync": (C.c_int, [C.c_void_p]),
    "spx_chan_exec": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64,
                                C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.c_void_p]),
    "spx_stft_time": (C.c_int, [C.c_void_p, C.POINTER(spx_stft_args), C.c_int32, C.c_int32, C.c_int32,
                                C.POINTER(C.c_float)]),
    "spx_welch_finalize": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_double, C.c_void_p, C.c_void_p,
                                     C.c_void_p]),
    "spx_welch_finalize_batch": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int64, C.c_double, C.c_void_p,
                                           C.c_void_p, C.c_void_p]),
    "spx_classify_features": (C.c_int, [C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int64,
                                        C.POINTER(spx_features), C.c_void_p, C.c_int32, C.POINTER(spx_feature_opts),
                                        C.c_void_p]),
    "spx_classify_features_dev": (C.c_int, [C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_void_p,
                                            C.c_void_p, C.c_int32, C.POINTER(spx_feature_opts), C.c_void_p]),
    "spx_detect_regions": (C.c_int, [C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_double,
                                     C.c_int32, C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.c_void_p, C.c_void_p,
                                     C.c_void_p]),
    "spx_iq_hist2d": (C.c_int, [C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_double, C.c_int64, C.c_double,
                                C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]),
    "spx_frame_stats": (C.c_int, [C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_float, C.c_int64, C.c_int32,
                                  C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(C.c_int64), C.c_void_p]),
    "spx_ring_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_void_p, C.POINTER(spx_ring_config)]),
    "spx_ring_destroy": (C.c_int, [C.c_void_p]),
    "spx_ring_acquire": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
    "spx_ring_commit": (C.c_int, [C.c_void_p, C.c_int64]),
    "spx_ring_collect": (C.c_int, [C.c_void_p, C.POINTER(spx_ring_result)]),
    "spx_ring_release": (C.c_int, [C.c_void_p]),
    "spx_ring_stats": (C.c_int, [C.c_void_p, C.POINTER(spx_ring_stats_t)]),
    "spx_plan_window_sums": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "spx_plan_stream": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "spx_fp32_peak": (C.c_int, [C.c_int, C.POINTER(C.c_double)]),
    "spx_ipc_export": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p]),
    "spx_ipc_open": (C.c_int, [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    "spx_ipc_close": (C.c_int, [C.c_int, C.c_void_p]),
    "spx_memcpy_d2d_async": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "spx_stream_sync": (C.c_int, [C.c_int, C.c_void_p]),
    "spx_stream_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "spx_stream_destroy": (C.c_int, [C.c_int, C.c_void_p]),
    "spx_stream_wait_stream": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p]),
    "spx_copy_ceiling": (C.c_int, [C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t, C.c_int,
                                   C.POINTER(C.c_double)]),
    "spx_peer_reduce": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "spx_peer_push_rows": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "spx_nccl_unique_id": (C.c_int, [C.c_void_p]),
    "spx_nccl_init": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "spx_nccl_destroy": (C.c_int, [C.c_void_p]),
    "spx_allreduce_welch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64), C.c_void_p]),
    "spx_gather_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.POINTER(C.c_int64), C.c_int, C.c_void_p]),
    "spx_stream_frame_f64": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_double, C.c_double, C.c_void_p]),
    "spx_timer_create": (C.c_int, [C.c_int32, C.POINTER(C.c_void_p)]),
    "spx_timer_start": (C.c_int, [C.c_void_p, C.c_void_p]),
    "spx_timer_stop": (C.c_int, [C.c_void_p, C.c_void_p]),
    "spx_timer_elapsed_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "spx_timer_destroy": (C.c_int, [C.c_void_p]),
}

_lib = None
_lib_error = None          # a failed build / load is remembered: later calls raise at once instead of re-running make
_lock = threading.Lock()


def build(verbose: bool = False) -> str:
    """Compile csrc/*.cu into csrc/libspx.so for sm_100a (nvcc cross-compiles without a GPU)."""
    if shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc"):
        raise SpectralError(E_UNSUPPORTED, "nvcc not found: cannot build libspx.so")
    env = dict(os.environ)
    if shutil.which("nvcc") is None:
        env["PATH"] = "/usr/local/cuda/bin:" + env.get("PATH", "")
    jobs = str(max(1, min(8, os.cpu_count() or 1)))
    # one builder at a time across processes (one process per GPU may start on a tree without the .so): an exclusive
    # file lock around make; the Makefile links to a temporary name and renames, so a concurrent loader never sees a
    # half-written library
    import fcntl
    with open(os.path.join(CSRC, ".build.lock"), "w") as lock_fh:
        fcntl.flock(lock_fh, fcntl.LOCK_EX)
        try:
            res = subprocess.run(["make", "-C", CSRC, "-j", jobs], env=env, capture_output=True, text=True)
        finally:
            fcntl.flock(lock_fh, fcntl.LOCK_UN)
    if verbose or res.returncode != 0:
        print(res.stdout[-4000:])
        print(res.stderr[-4000:])
    if res.returncode != 0 or not os.path.exists(LIB_PATH):
        raise SpectralError(E_UNSUPPORTED, "building libspx.so failed:\n" + res.stderr[-2000:])
    return LIB_PATH


def lib() -> C.CDLL:
    """Load (building on first use if the .so is absent) and type the library."""
    global _lib, _lib_error
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if _lib_error is not None:      # do not rebuild / reload per call (e.g. per rx buffer in the streaming thread)
            raise SpectralError(E_UNSUPPORTED, _lib_error)
        try:
            if not os.path.exists(LIB_PATH):
                build()
            handle = C.CDLL(LIB_PATH)
        except SpectralError as e:
            _lib_error = f"libspx.so unavailable (cached failure; call _native.reset_load_failure() to retry): {e}"
            raise
        except OSError as e:  # missing extension is fatal: no fallback path exists
            _lib_error = f"cannot load {LIB_PATH} (cached failure; call _native.reset_load_failure() to retry): {e}"
            raise SpectralError(E_UNSUPPORTED, _lib_error) from e
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def reset_load_failure() -> None:
    """Forget a cached build / load failure so that the next call tries again (after fixing the toolchain)."""
    global _lib_error
    with _lock:
        _lib_error = None


def last_error() -> str:
    return (lib().spx_last_error() or b"").decode(errors="replace")


def check(rc: int) -> None:
    if rc != OK:
        raise SpectralError(rc, last_error())


def device_count() -> int:
    n = C.c_int(0)
    rc = lib().spx_device_count(C.byref(n))
    if rc == E_NODEVICE:
        return 0
    check(rc)
    return int(n.value)


def require_device() -> int:
    n = device_count()
    if n == 0:
        raise SpectralError(E_NODEVICE, "no CUDA device available; this package has no CPU fallback")
    return n


def device_info(device: int = 0) -> dict:
    info = spx_device_info()
    check(lib().spx_get_device_info(device, C.byref(info)))
    return {"name": info.name.decode(), "sm_count": info.sm_count, "cc": (info.cc_major, info.cc_minor),
            "l2_bytes": info.l2_bytes, "max_smem_optin": info.max_smem_optin, "total_mem": info.total_mem}


def fp32_peak_tflops(device: int = 0) -> float:
    """Measured FP32 FMA peak of the device (micro-kernel inside libspx), TFLOP/s."""
    v = C.c_double()
    check(lib().spx_fp32_peak(device, C.byref(v)))
    return float(v.value)


def frame_count(n_samples: int, nfft: int, hop: int) -> int:
    return int(lib().spx_frame_count(int(n_samples), int(nfft), int(hop)))


# ----------------------------------------------------------------------------- memory helpers
class _Pinned:
    """Owner of one cudaHostAlloc block, exposed to numpy through __array_interface__."""

    def __init__(self, nbytes: int, write_combined: bool = False):
        p = C.c_void_p()
        check((lib().spx_host_alloc_wc if write_combined else lib().spx_host_alloc)(C.byref(p), nbytes))
        self.ptr = p.value
        self.__array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (self.ptr, False), "version": 3}

    def __del__(self):
        try:
            if self.ptr and _lib is not None:
                _lib.spx_host_free(self.ptr)
                self.ptr = None
        except Exception:
            pass


def pinned_empty(shape, dtype, write_combined: bool = False) -> np.ndarray:
    """numpy array backed by page-locked host memory (cudaHostAlloc): makes the H2D/D2H legs of
    SPX_MEM_HOST execution truly asynchronous.  The block is freed when the last view dies.
    ``write_combined``: for input buffers the CPU only fills sequentially (never reads back)."""
    dtype = np.dtype(dtype)
    shape = tuple(int(v) for v in (shape if np.ndim(shape) else (shape,)))
    n = int(np.prod(shape))
    nbytes = max(1, n * dtype.itemsize)
    raw = np.asarray(_Pinned(nbytes, write_combined))
    return raw[: n * dtype.itemsize].view(dtype).reshape(shape)


class DeviceArray:
    """A typed device allocation owned by Python (cudaMalloc through libspx)."""

    def __init__(self, shape, dtype, device: int = 0, zero: bool = False):
        self.shape = tuple(int(s) for s in (shape if np.ndim(shape) else (shape,)))
        self.dtype = np.dtype(dtype)
        self.device = int(device)
        self.nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        p = C.c_void_p()
        check(lib().spx_device_alloc(self.device, C.byref(p), max(1, self.nbytes)))
        self.ptr = p.value
        if zero:
            self.zero_()

    @classmethod
    def from_host(cls, arr: np.ndarray, device: int = 0) -> "DeviceArray":
        arr = np.ascontiguousarray(arr)
        d = cls(arr.shape, arr.dtype, device)
        d.copy_from_host(arr)
        return d

    def copy_from_host(self, arr: np.ndarray) -> None:
        arr = np.ascontiguousarray(arr)
        if arr.nbytes != self.nbytes:
            raise ValueError("size mismatch")
        check(lib().spx_memcpy_h2d(self.device, self.ptr, arr.ctypes.data, self.nbytes))

    def to_host(self) -> np.ndarray:
        out = np.empty(self.shape, dtype=self.dtype)
        if self.nbytes:
            check(lib().spx_memcpy_d2h(self.device, out.ctypes.data, self.ptr, self.nbytes))
        return out

    def zero_(self) -> None:
        check(lib().spx_memset(self.device, self.ptr, 0, self.nbytes))

    def free(self) -> None:
        if getattr(self, "ptr", None):
            try:
                lib().spx_device_free(self.device, self.ptr)
            finally:
                self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class DeviceView:
    """A typed window into device memory this object does not own: a slice of a DeviceArray, or a peer
    GPU's buffer mapped with ``PeerBuffer``.  Accepted wherever a DeviceArray is."""

    def __init__(self, ptr: int, shape, dtype, device: int = 0, keep=None):
        self.ptr = int(ptr)
        self.shape = tuple(int(s) for s in (shape if np.ndim(shape) else (shape,)))
        self.dtype = np.dtype(dtype)
        self.device = int(device)
        self.nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        self._keep = keep

    def rows(self, r0: int, r1: int) -> "DeviceView":
        """Rows [r0, r1) of a 2-D view."""
        pitch = self.shape[1] * self.dtype.itemsize
        return DeviceView(self.ptr + r0 * pitch, (r1 - r0, self.shape[1]), self.dtype, self.device, self)


class PeerBuffer:
    """One device allocation shared between the ranks of a node (one process per GPU): the owner
    allocates and exports it (``handle``), the others map it with ``PeerBuffer.open`` and pass
    ``view()`` as an output of ``SpectralPlan.stft(..., peer_outputs=True)``; their kernels then write
    and reduce into the owner's HBM over NVLink."""

    def __init__(self, shape, dtype, device: int = 0):
        self.array = DeviceArray(shape, dtype, device, zero=True)
        self.shape, self.dtype, self.device = self.array.shape, self.array.dtype, device
        h = (C.c_ubyte * 64)()
        check(lib().spx_ipc_export(device, self.array.ptr, h))
        self.handle = bytes(h)
        self._mapped = None

    @classmethod
    def open(cls, handle: bytes, shape, dtype, device: int) -> "PeerBuffer":
        self = cls.__new__(cls)
        self.array = None
        self.shape = tuple(int(s) for s in (shape if np.ndim(shape) else (shape,)))
        self.dtype, self.device, self.handle = np.dtype(dtype), device, handle
        p = C.c_void_p()
        check(lib().spx_ipc_open(device, (C.c_ubyte * 64).from_buffer_copy(handle), C.byref(p)))
        self._mapped = p.value
        return self

    def view(self) -> DeviceView:
        ptr = self.array.ptr if self.array is not None else self._mapped
        return DeviceView(ptr, self.shape, self.dtype, self.device, self)

    def close(self) -> None:
        if self._mapped:
            lib().spx_ipc_close(self.device, self._mapped)
            self._mapped = None
        if self.array is not None:
            self.array.free()
            self.array = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DeviceTimer:
    """A pair of CUDA events recorded on a stream (spx_timer_*): device time of what ran in between."""

    def __init__(self, device: int = 0, stream: int = 0):
        self._h = C.c_void_p()
        self.stream = stream or None
        check(lib().spx_timer_create(device, C.byref(self._h)))

    def start(self) -> None:
        check(lib().spx_timer_start(self._h, self.stream))

    def stop(self) -> None:
        check(lib().spx_timer_stop(self._h, self.stream))

    def elapsed_ms(self) -> float:
        ms = C.c_float()
        check(lib().spx_timer_elapsed_ms(self._h, C.byref(ms)))
        return float(ms.value)

    def close(self) -> None:
        if self._h:
            lib().spx_timer_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class SideStream:
    """A non-blocking CUDA stream owned by Python, with the one ordering primitive callers need: ``after(other)`` makes
    this stream wait for what ``other`` (a cudaStream_t as int, or another SideStream) holds now."""

    def __init__(self, device: int = 0):
        self.device = int(device)
        h = C.c_void_p()
        check(lib().spx_stream_create(self.device, C.byref(h)))
        self.handle = int(h.value)

    @staticmethod
    def _h(s):
        return s.handle if isinstance(s, SideStream) else (s or None)

    def after(self, other) -> None:
        check(lib().spx_stream_wait_stream(self.device, self.handle, self._h(other)))

    def then(self, other) -> None:
        """``other`` waits for what this stream holds now."""
        check(lib().spx_stream_wait_stream(self.device, self._h(other), self.handle))

    def sync(self) -> None:
        check(lib().spx_stream_sync(self.device, self.handle))

    def close(self) -> None:
        if getattr(self, "handle", None):
            lib().spx_stream_destroy(self.device, self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def device_sync(device: int = 0) -> None:
    check(lib().spx_device_sync(device))


def as_ptr(x) -> tuple:
    """(pointer, mem) of a numpy array, DeviceArray, torch tensor or None."""
    if x is None:
        return None, None
    if isinstance(x, (DeviceArray, DeviceView)):
        return x.ptr, MEM_DEVICE
    if isinstance(x, np.ndarray):
        if not x.flags.c_contiguous:
            raise ValueError("array must be C-contiguous")
        return x.ctypes.data, MEM_HOST
    if hasattr(x, "data_ptr") and hasattr(x, "is_cuda"):  # torch tensor (plumbing only)
        if not x.is_contiguous():
            raise ValueError("tensor must be contiguous")
        return int(x.data_ptr()), (MEM_DEVICE if x.is_cuda else MEM_HOST)
    raise TypeError(f"unsupported buffer type {type(x)!r}")
