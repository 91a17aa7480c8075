"""Spectral hot path: host-side API over libspx (CUDA, sm_100a).  No CPU fallback.

This is the new ``app.processing.spectral`` module of the drop-in (SURVEY.md section 7): the
reference computes its spectrum inline in the streamer thread
(/root/reference/app/sdr/streamer.py:119-121) and, offline, through ``plt.psd``
(/root/reference/scripts/process_sigmf_data.py:188).  The functions here keep those semantics
(fftshift order, ``20*log10(|X| + 1e-12)``, mlab.psd normalisation) and add the overlapped STFT,
Welch / max-hold accumulators and uint8 waterfall rows of SURVEY.md section 8(a).

Arrays may be numpy (host; staged by the library through pinned memory), ``DeviceArray`` or
CUDA torch tensors (device; used in place on the given stream).
"""
from __future__ import annotations

import ctypes as C
import threading
import weakref
from dataclasses import dataclass
from typing import Optional

import numpy as np

from . import _native as nat
from ._native import (FMT_CF32, FMT_CI16, MEM_DEVICE, MEM_HOST, WINDOW_BLACKMAN, WINDOW_HANN, WINDOW_RECT,
                      DeviceArray, SpectralError, pinned_empty)

_WINDOWS = {"rect": WINDOW_RECT, "boxcar": WINDOW_RECT, "none": WINDOW_RECT, None: WINDOW_RECT,
            "hann": WINDOW_HANN, "hanning": WINDOW_HANN, "blackman": WINDOW_BLACKMAN}

DEFAULT_VARIANT = {}       # nfft -> kernel tuning variant (0 = library default everywhere)
DB_EPS_REFERENCE = 1e-12   # streamer.py:121
DB_EPS_LEGACY = 1e-10      # scripts/sdr_realtime_dash.py:73


def window_id(window) -> int:
    if isinstance(window, (int, np.integer)):
        if int(window) not in (0, 1, 2):
            raise ValueError(f"unknown window id {window}")
        return int(window)
    try:
        return _WINDOWS[window.lower() if isinstance(window, str) else window]
    except KeyError:
        raise ValueError(f"unknown window {window!r}") from None


def freq_axis(nfft: int, sample_rate: float, center_freq: float = 0.0) -> np.ndarray:
    """``fftshift(fftfreq(N, 1/fs)) + fc`` (streamer.py:120), float64.  Depends only on
    (N, fs, fc), so callers should cache it instead of rebuilding it per buffer."""
    return np.fft.fftshift(np.fft.fftfreq(int(nfft), 1 / sample_rate)) + center_freq


def pooled_freq_axis(nfft: int, bins_per_col: int, sample_rate: float, center_freq: float = 0.0) -> np.ndarray:
    """Frequency of each column of a pooled spectrogram (``SpectralPlan.stft(pool=(K, B, mode))``): the mean of the
    ``freq_axis`` frequencies of the B bins the column pools, float64 [nfft / B]."""
    nfft, b = int(nfft), int(bins_per_col)
    if b < 1 or nfft % b:
        raise ValueError(f"bins_per_col {b} must be >= 1 and divide nfft {nfft}")
    return freq_axis(nfft, sample_rate, center_freq).reshape(nfft // b, b).mean(axis=1)


_POOL_MODES = {"mean": nat.POOL_MEAN, "max": nat.POOL_MAX}


def pool_mode(mode) -> int:
    """SPX_POOL_* of "mean" (average detector) or "max" (peak detector)."""
    try:
        return _POOL_MODES[mode]
    except (KeyError, TypeError):
        raise ValueError(f"unknown pool mode {mode!r} (expected 'mean' or 'max')") from None


def _pool_shape(nfft: int, pool) -> tuple:
    """(K, B, mode id) of a ``pool=(K, B, mode)`` argument, checked."""
    try:
        K, B, mode = pool
    except (TypeError, ValueError):
        raise ValueError(f"pool must be (frames_per_row, bins_per_col, 'mean' | 'max'), got {pool!r}") from None
    K, B = int(K), int(B)
    if K < 1 or B < 1 or nfft % B:
        raise ValueError(f"pool: frames_per_row {K} must be >= 1, bins_per_col {B} >= 1 and a divisor of nfft {nfft}")
    return K, B, pool_mode(mode)


def _buffer_dtype_count(buf):
    """(numpy dtype, element count) of a numpy array, DeviceArray / DeviceView or torch tensor."""
    if isinstance(buf, np.ndarray):
        return buf.dtype, int(buf.size)
    if isinstance(buf, (DeviceArray, nat.DeviceView)):
        return np.dtype(buf.dtype), int(np.prod(buf.shape))
    if hasattr(buf, "data_ptr"):   # torch tensor: "torch.float32" -> float32
        return np.dtype(str(buf.dtype).replace("torch.", "")), int(buf.numel())
    raise TypeError(f"unsupported buffer type {type(buf)!r}")


def _check_buffer(buf, shape, dtype, name: str) -> None:
    """Caller-supplied output buffer: dtype and element count must be exactly what libspx will write."""
    want_dt, want_n = np.dtype(dtype), int(np.prod(shape))
    dt, n = _buffer_dtype_count(buf)
    if dt != want_dt or n != want_n:
        raise ValueError(f"{name}: expected {want_n} elements of {want_dt} (shape {tuple(shape)}), got {n} of {dt}")


@dataclass
class StftResult:
    n_frames: int
    n_streams: int
    db_rows: Optional[object] = None     # float32 [S*F, N]
    wf_rows: Optional[object] = None     # uint8   [S*F, N]
    spectrum: Optional[object] = None    # complex64 [S*F, N]
    welch_acc: Optional[object] = None   # float64 [S, N]
    maxhold: Optional[object] = None     # float32 [S, N]
    h2d_bytes: int = 0
    d2h_bytes: int = 0
    persistence: Optional[object] = None  # uint32  [S, 256, N] frames per waterfall level and bin
    pool_acc: Optional[object] = None     # float64 [S, G, N/B] pooled accumulator (finalise with pool_finalize)


class SpectralPlan:
    """One (nfft, hop, window, input format) configuration bound to one GPU.

    ``in_scale`` multiplies every sample (1.0 for the raw-integer stream path, 2**-15 for SigMF
    ``ci16_le``); ``db_eps`` is the epsilon of ``20*log10(|X| + eps)``.
    """

    def __init__(self, nfft: int, hop: Optional[int] = None, window="rect", in_fmt: int = FMT_CF32,
                 in_scale: float = 1.0, db_eps: float = DB_EPS_REFERENCE, device: int = 0, variant: int = 0):
        nat.require_device()
        self.nfft = int(nfft)
        self.hop = int(hop) if hop else self.nfft
        self.window = window_id(window)
        self.in_fmt = int(in_fmt)
        self.in_scale = float(in_scale)
        self.db_eps = float(db_eps)
        self.device = int(device)
        cfg = nat.spx_plan_config(C.sizeof(nat.spx_plan_config), self.device, self.nfft, self.hop, self.window,
                                  self.in_fmt, self.in_scale, self.db_eps, int(variant), 0)
        h = C.c_void_p()
        nat.check(nat.lib().spx_plan_create(C.byref(h), C.byref(cfg)))
        self._h = h
        self._rings = weakref.WeakSet()   # rings borrow the native plan: they are torn down first
        s2, s1 = C.c_double(), C.c_double()
        nat.check(nat.lib().spx_plan_window_sums(self._h, C.byref(s2), C.byref(s1)))
        self.sum_w2, self.sum_w = s2.value, s1.value

    # -- lifetime
    def close(self) -> None:
        for ring in list(getattr(self, "_rings", ())):
            ring.close()
        h, self._h = getattr(self, "_h", None), None
        if h:
            nat.lib().spx_plan_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def sync(self) -> None:
        nat.check(nat.lib().spx_plan_sync(self._h))

    def frame_count(self, n_samples: int) -> int:
        return nat.frame_count(n_samples, self.nfft, self.hop)

    # -- input marshalling
    def _host_input(self, x: np.ndarray) -> np.ndarray:
        x = np.asarray(x)
        if self.in_fmt == FMT_CI16:
            if x.dtype != np.int16:
                raise TypeError("ci16 plan needs int16 interleaved I,Q")
            return np.ascontiguousarray(x)
        if x.dtype == np.complex64:
            return np.ascontiguousarray(x)
        if np.iscomplexobj(x):
            # pyadi-iio rx() hands the stream path complex128 (streamer.py:114); complex64 holds
            # every int16-range value exactly
            return np.ascontiguousarray(x, dtype=np.complex64)
        if x.dtype == np.float32 and x.ndim >= 1 and x.shape[-1] == 2:
            return np.ascontiguousarray(x)
        return np.ascontiguousarray(x, dtype=np.complex64)

    def _samples_per_stream(self, x, n_streams: int) -> int:
        if isinstance(x, np.ndarray):
            total = x.size // 2 if (x.dtype == np.int16 or x.dtype == np.float32) else x.size
        elif isinstance(x, (DeviceArray, nat.DeviceView)):
            total = x.nbytes // (4 if self.in_fmt == FMT_CI16 else 8)
        else:
            total = x.numel() * x.element_size() // (4 if self.in_fmt == FMT_CI16 else 8)
        return total // n_streams

    # -- execution
    def stft(self, x, *, n_streams: int = 1, db_rows=False, wf_rows=False, spectrum=False, welch=False,
             maxhold=False, vmin: float = -100.0, vmax: float = 0.0, accumulate: bool = False,
             stream: int = 0, n_samples: Optional[int] = None, peer_outputs: int = 0, persistence=False,
             pool=None, pool_acc=True, pool_first_frame: int = 0, stream_stride: Optional[int] = None,
             _time=None) -> StftResult:
        """Windowed STFT of ``x`` (1 stream, or ``n_streams`` equal-length streams laid out back to
        back).  Each output flag is False (not wanted), True (allocate) or a caller buffer to fill
        (numpy for host input, DeviceArray / CUDA tensor for device input).

        ``persistence``: uint32 ``[n_streams, 256, nfft]``, for every bin the number of frames at each uint8 waterfall
        level of ``[vmin, vmax]`` (a persistence / density spectrum; every column sums to the frame count).  It is an
        accumulator like ``welch`` and ``maxhold``.  It does not need ``wf_rows``: without them the rows stay on the GPU.

        ``pool=(K, B, "mean" | "max")``: a pooled spectrogram (display detectors).  Row g pools the frames
        ``[g K, (g + 1) K)`` of global frame index (this call's frame 0 is ``pool_first_frame``), column c the bins
        ``[c B, (c + 1) B)``; "mean" sums the power of the cell, "max" keeps its largest dB value.  ``pool_acc`` is the
        float64 ``[n_streams, G, nfft / B]`` accumulator (True: allocate with G = ceil((pool_first_frame + F) / K)); it
        is an accumulator like ``welch``, so calls on consecutive pieces of a capture pool into one image, and
        ``pool_finalize`` turns it into dB and levels.  It does not need ``db_rows``: without them the rows stay on the
        GPU.

        ``stream_stride``: samples between the starts of consecutive streams (default: the stream length, streams back to
        back), e.g. the row pitch of a channel-major ``Channelizer`` output whose rows are longer than the samples used;
        ``n_samples`` then gives the samples per stream."""
        if persistence is not False and persistence is not None and _time is not None:
            raise ValueError("persistence cannot be timed with _time (spx_stft_time runs spx_stft_exec)")
        if pool is not None:
            if _time is not None:
                raise ValueError("pool cannot be timed with _time (spx_stft_time runs spx_stft_exec)")
            if persistence is not False and persistence is not None:
                raise ValueError("pool and persistence cannot be computed in one call")
            pK, pB, pmode = _pool_shape(self.nfft, pool)
            if int(pool_first_frame) < 0:
                raise ValueError("pool_first_frame must be >= 0")
        if isinstance(x, np.ndarray) or not (isinstance(x, (DeviceArray, nat.DeviceView)) or hasattr(x, "data_ptr")):
            x = self._host_input(x)
        in_ptr, mem = nat.as_ptr(x)
        L = int(n_samples) if n_samples is not None else self._samples_per_stream(x, n_streams)
        F = self.frame_count(L)
        rows = n_streams * F
        N = self.nfft

        def out(flag, shape, dtype, name, accumulator=False):
            if flag is False or flag is None:
                return None
            if flag is True:
                # library-allocated accumulators start from zero (``accumulate=True`` then means "add to nothing")
                if mem == MEM_HOST:
                    return np.zeros(shape, dtype) if accumulator else np.empty(shape, dtype)
                return DeviceArray(shape, dtype, self.device, zero=accumulator)
            p, m = nat.as_ptr(flag)
            if m != mem:
                raise ValueError("output buffers must live where the input lives")
            # libspx writes prod(shape) elements of ITS type through this pointer: a buffer of another size or dtype
            # would be overrun (or half filled) silently, so it is refused here
            _check_buffer(flag, shape, dtype, name)
            return flag

        o_db = out(db_rows, (rows, N), np.float32, "db_rows")
        o_wf = out(wf_rows, (rows, N), np.uint8, "wf_rows")
        o_sp = out(spectrum, (rows, N), np.complex64, "spectrum")
        o_we = out(welch, (n_streams, N), np.float64, "welch", accumulator=True)
        o_mh = out(maxhold, (n_streams, N), np.float32, "maxhold", accumulator=True)
        o_pe = out(persistence, (n_streams, 256, N), np.uint32, "persistence", accumulator=True)
        o_pool = None
        if pool is not None:
            C_ = N // pB
            if pool_acc is True:
                G = -(-(int(pool_first_frame) + F) // pK)
                # with accumulate=True a library-allocated accumulator adds to the mode's identity (0, or -inf for max)
                if accumulate:
                    ident = np.full((n_streams, G, C_), -np.inf if pmode == nat.POOL_MAX else 0.0)
                    o_pool = ident if mem == MEM_HOST else DeviceArray.from_host(ident, self.device)
                elif mem == MEM_HOST:
                    o_pool = np.empty((n_streams, G, C_), np.float64)
                else:
                    o_pool = DeviceArray((n_streams, G, C_), np.float64, self.device)
            else:
                if pool_acc is False or pool_acc is None:
                    raise ValueError("pool needs pool_acc (True or a buffer)")
                _, cnt = _buffer_dtype_count(pool_acc)
                G = cnt // max(1, n_streams * C_)
                o_pool = out(pool_acc, (n_streams, G, C_), np.float64, "pool_acc", accumulator=True)
            pa = nat.spx_pool_args(C.sizeof(nat.spx_pool_args), pmode, pK, pB, 0, int(pool_first_frame), G,
                                   nat.as_ptr(o_pool)[0])
        a = nat.spx_stft_args()
        a.struct_size = C.sizeof(nat.spx_stft_args)
        a.mem = mem
        a.in_ = in_ptr
        a.n_samples = L
        a.stream_stride = L if stream_stride is None else int(stream_stride)
        if a.stream_stride < L:
            raise ValueError(f"stream_stride {a.stream_stride} < samples per stream {L}")
        a.n_streams = n_streams
        a.accumulate = 1 if accumulate else 0
        a.db_rows = nat.as_ptr(o_db)[0]
        a.wf_rows = nat.as_ptr(o_wf)[0]
        a.spec_rows = nat.as_ptr(o_sp)[0]
        a.welch_acc = nat.as_ptr(o_we)[0]
        a.maxhold = nat.as_ptr(o_mh)[0]
        a.vmin, a.vmax = float(vmin), float(vmax)
        a.stream = stream or None
        a.peer_outputs = int(peer_outputs)   # bit 0: shared accumulators, bit 1: rows on a peer GPU (see spx.h)
        if _time is not None:
            warmup, iters, flush = _time
            ms = (C.c_float * iters)()
            nat.check(nat.lib().spx_stft_time(self._h, C.byref(a), warmup, iters, 1 if flush else 0, ms))
            self.last_times_ms = [float(v) for v in ms]
        elif o_pe is not None:
            nat.check(nat.lib().spx_stft_exec_persistence(self._h, C.byref(a), nat.as_ptr(o_pe)[0]))
        elif o_pool is not None:
            nat.check(nat.lib().spx_stft_exec_pooled(self._h, C.byref(a), C.byref(pa)))
        else:
            nat.check(nat.lib().spx_stft_exec(self._h, C.byref(a)))
        return StftResult(int(a.n_frames_out), n_streams, o_db, o_wf, o_sp, o_we, o_mh,
                          int(a.h2d_bytes_out), int(a.d2h_bytes_out), o_pe, o_pool)

    def time_stft(self, x, *, warmup: int = 3, iters: int = 10, flush_l2: bool = False, **kw):
        """Device-resident timing of the exact launch ``stft`` would make: CUDA events on the launch
        stream around each of ``iters`` launches after ``warmup`` untimed ones.  Returns
        (StftResult of the last launch, [ms per launch])."""
        res = self.stft(x, _time=(int(warmup), int(iters), bool(flush_l2)), **kw)
        return res, self.last_times_ms

    @property
    def stream(self) -> int:
        """cudaStream_t (as int) of the plan's compute stream, for ordering device-memory calls after its kernels."""
        st = C.c_void_p()
        nat.check(nat.lib().spx_plan_stream(self._h, C.byref(st)))
        return int(st.value or 0)

    def welch_finalize(self, welch_acc, n_frames: int, sample_rate: float, want_db: bool = True, pxx=None, pdb=None,
                       n_streams: int = 1, stream: int = 0):
        """mlab.psd density and its dB from an accumulated numerator (``n_streams`` accumulators laid out
        [n_streams][nfft], one launch).  ``pxx`` / ``pdb`` may be caller buffers (same memory space as
        ``welch_acc``) to avoid an allocation per call."""
        p, mem = nat.as_ptr(welch_acc)
        N = self.nfft * int(n_streams)
        _check_buffer(welch_acc, (N,), np.float64, "welch_acc")
        for name, buf in (("pxx", pxx), ("pdb", pdb)):
            if buf is not None:
                if nat.as_ptr(buf)[1] != mem:
                    raise ValueError(f"{name} must live where welch_acc lives")
                _check_buffer(buf, (N,), np.float64, name)
        if mem == MEM_HOST:
            pxx = np.empty(N, np.float64) if pxx is None else pxx
            pdb = (np.empty(N, np.float64) if want_db else None) if pdb is None else pdb
        else:
            pxx = DeviceArray((N,), np.float64, self.device) if pxx is None else pxx
            pdb = (DeviceArray((N,), np.float64, self.device) if want_db else None) if pdb is None else pdb
        nat.check(nat.lib().spx_welch_finalize_batch(self._h, mem, p, int(n_streams), int(n_frames), float(sample_rate),
                                                     nat.as_ptr(pxx)[0], nat.as_ptr(pdb)[0], stream or None))
        return pxx, pdb

    def pool_finalize(self, pool_acc, n_frames_total: int, frames_per_row: int, bins_per_col: int, mode="mean",
                      db: bool = True, wf: bool = False, vmin: float = -100.0, vmax: float = 0.0, n_streams: int = 1,
                      stream: int = 0):
        """Pooled dB (float32) and / or uint8 levels of ``[vmin, vmax]`` of an accumulator filled by
        ``stft(pool=(frames_per_row, bins_per_col, mode))`` over ``n_frames_total`` frames, both shaped
        ``[n_streams, G, nfft / B]`` with G = ceil(n_frames_total / K), in the accumulator's memory space.  Returns
        ``(db, levels)``; an output not asked for is None.  The levels are those of the returned float32 dB."""
        K, B, m = _pool_shape(self.nfft, (frames_per_row, bins_per_col, mode))
        F = int(n_frames_total)
        G = -(-F // K) if F > 0 else 0
        shape = (int(n_streams), G, self.nfft // B)
        _check_buffer(pool_acc, shape, np.float64, "pool_acc")
        p, mem = nat.as_ptr(pool_acc)

        def alloc(dtype):
            return np.empty(shape, dtype) if mem == MEM_HOST else DeviceArray(shape, dtype, self.device)
        o_db = alloc(np.float32) if db else None
        o_wf = alloc(np.uint8) if wf else None
        nat.check(nat.lib().spx_pool_finalize(self._h, mem, m, p, int(n_streams), G, F, K, B, nat.as_ptr(o_db)[0],
                                              nat.as_ptr(o_wf)[0], float(vmin), float(vmax), stream or None))
        return o_db, o_wf


# ----------------------------------------------------------------------------- plan cache + convenience
_plans: dict = {}
_plans_lock = threading.Lock()


def get_plan(nfft, hop=None, window="rect", in_fmt=FMT_CF32, in_scale=1.0, db_eps=DB_EPS_REFERENCE, device=0,
             variant=0) -> SpectralPlan:
    key = (int(nfft), int(hop or nfft), window_id(window), int(in_fmt), float(in_scale), float(db_eps), int(device), int(variant))
    with _plans_lock:
        pl = _plans.get(key)
        if pl is None:
            pl = SpectralPlan(*key[:2], window=key[2], in_fmt=key[3], in_scale=key[4], db_eps=key[5], device=key[6],
                              variant=key[7])
            _plans[key] = pl
        return pl


def clear_plans() -> None:
    with _plans_lock:
        for pl in _plans.values():
            pl.close()
        _plans.clear()


def stream_frame(samples, sample_rate: float, center_freq: float, eps: float = DB_EPS_REFERENCE, device: int = 0,
                 wf_range=None):
    """Drop-in for the three hot lines of the reference stream loop (streamer.py:119-121):
    returns ``(freqs, power_db)``, both float64[N] in fftshift order, for one rx buffer of any length.
    With ``wf_range=(vmin, vmax)`` the same launch also emits the uint8 waterfall row of the frame and the
    return value is ``(freqs, power_db, wf_row)``.

    Power-of-two buffers up to 8192 samples (the reference's default is 4096, streamer.py:10) run the float64 kernel
    (``spx_stream_frame_f64``): the reference computes this path in float64 and, at ~244 buffers/s, precision is what
    matters.  Other lengths go through the float32 plan (Bluestein / four-step kernels)."""
    x = np.asarray(samples)
    n = x.shape[0]
    if 2 <= n <= 8192 and (n & (n - 1)) == 0:
        nat.require_device()
        if x.dtype != np.complex64:
            x = np.ascontiguousarray(x, dtype=np.complex128)   # pyadi-iio rx() already returns complex128 (streamer.py:114)
        else:
            x = np.ascontiguousarray(x)
        pdb = np.empty(n, np.float64)
        wf = np.empty(n, np.uint8) if wf_range is not None else None
        vmin, vmax = (float(wf_range[0]), float(wf_range[1])) if wf_range is not None else (0.0, 1.0)
        nat.check(nat.lib().spx_stream_frame_f64(int(device), MEM_HOST, x.ctypes.data, 1 if x.dtype == np.complex128 else 0, n,
                                                  float(eps), pdb.ctypes.data, None, None if wf is None else wf.ctypes.data,
                                                  vmin, vmax, None))
        if wf is None:
            return freq_axis(n, sample_rate, center_freq), pdb
        return freq_axis(n, sample_rate, center_freq), pdb, wf
    pl = get_plan(n, n, "rect", FMT_CF32, 1.0, eps, device)
    if wf_range is None:
        res = pl.stft(x, db_rows=True)
        return freq_axis(n, sample_rate, center_freq), res.db_rows[0].astype(np.float64)
    res = pl.stft(x, db_rows=True, wf_rows=True, vmin=float(wf_range[0]), vmax=float(wf_range[1]))
    return freq_axis(n, sample_rate, center_freq), res.db_rows[0].astype(np.float64), res.wf_rows[0]


def welch_psd(x, nfft: int = 1024, hop: Optional[int] = None, window="hann", sample_rate: float = 1.0,
              center_freq: float = 0.0, in_fmt: int = FMT_CF32, in_scale: float = 1.0, device: int = 0):
    """``plt.psd(x, NFFT, Fs, Fc)`` semantics (process_sigmf_data.py:188): returns ``(freqs, Pxx)``
    with Pxx the two-sided density in fftshift order (plot ``10*log10(Pxx)``).  Input shorter than
    ``nfft`` is zero-padded to one frame, as mlab does."""
    pl = get_plan(nfft, hop or nfft, window, in_fmt, in_scale, DB_EPS_REFERENCE, device)
    x = pl._host_input(x)
    n = pl._samples_per_stream(x, 1)
    if n < nfft:
        pad = np.zeros(nfft * (2 if in_fmt == FMT_CI16 else 1), dtype=x.dtype)
        pad[: x.size] = x.reshape(-1)
        x = pad
    res = pl.stft(x, welch=True)
    pxx, _ = pl.welch_finalize(res.welch_acc[0], res.n_frames, sample_rate, want_db=False)
    return freq_axis(nfft, sample_rate, center_freq), pxx


def waterfall(x, nfft: int, hop: int, window="hann", vmin: float = -100.0, vmax: float = 0.0, in_fmt: int = FMT_CF32,
              in_scale: float = 1.0, device: int = 0) -> np.ndarray:
    """uint8 waterfall rows [F][N] (colormap indices; see viridis_lut)."""
    pl = get_plan(nfft, hop, window, in_fmt, in_scale, DB_EPS_REFERENCE, device)
    return pl.stft(x, wf_rows=True, vmin=vmin, vmax=vmax).wf_rows


_VIRIDIS = ["#440154", "#482878", "#3e4989", "#31688e", "#26828e", "#1f9e89", "#35b779", "#6ece58", "#b5de2b", "#fde725"]


def viridis_lut() -> np.ndarray:
    """256x3 uint8 table for the u8 rows: Plotly's 'Viridis' stops (callbacks.py:187), linear in RGB."""
    stops = np.array([[int(h[i:i + 2], 16) for i in (1, 3, 5)] for h in _VIRIDIS], dtype=np.float64)
    t = (np.arange(256) + 0.5) / 256.0
    pos = np.linspace(0.0, 1.0, len(stops))
    return np.floor(np.stack([np.interp(t, pos, stops[:, c]) for c in range(3)], axis=1) + 0.5).astype(np.uint8)
