"""Zoom: digital down-conversion (NCO mix + decimating FIR) on the GPU (libspx K9, ``spx_ddc_*`` in include/spx.h).

A ``DdcPlan`` shifts the band around ``shift_hz`` to 0 Hz, low-pass filters it and keeps every ``decim``-th sample.  Its
output is ordinary complex64 input at ``sample_rate / decim`` whose centre frequency is ``fc + plan.shift_hz``, so every
spectral product (``SpectralPlan.stft`` rows, Welch, max-hold, persistence, pooling, the classifier) applies to the
zoomed band unchanged.

Output m is ``np.convolve(mix, h, 'valid')[::decim][m]`` of the mixed input; with odd symmetric taps (the default design)
it belongs to time ``(first_sample + m decim + (T - 1) / 2) / fs``.  The default filter passes ``|f| <= 0.4 fs / decim``
free of aliasing (``usable_span_hz``); the outer 10 % of each side of the zoomed span is roll-off.  One stage takes up to
8192 taps (decim 256 with the default design); for more decimation cascade two plans, the second with ``shift_hz=0``.
Compute is libspx only (no CPU fallback); the filter design is numpy only.

A ``Channelizer`` does the M down-conversions of a uniform channel grid at once (a polyphase filter bank): channel j is the
``DdcPlan`` at shift ``(j - M/2) fs / M``, and its channel-major output feeds ``SpectralPlan.stft`` as M streams.
"""
from __future__ import annotations

import ctypes as C
import math
from fractions import Fraction
from typing import Optional

import numpy as np

from . import _native as nat
from ._native import FMT_CF32, FMT_CI16, MEM_HOST, DeviceArray
from .spectral import SpectralPlan, _check_buffer

MAX_TAPS = 8192
# one job of DdcPlan.exec_jobs (the layout of spx_ddc_job)
JOB_DTYPE = np.dtype([("first_sample", "<i8"), ("phase_inc", "<i8"), ("m0", "<i8"), ("n_out", "<i8"),
                      ("out_offset", "<i8")])


def kaiser_order(atten_db: float, width: float) -> tuple:
    """(numtaps, beta) of a Kaiser-window FIR (Kaiser's formulas, as scipy.signal.kaiserord): ``width`` is the transition
    width in units of the Nyquist frequency."""
    a = abs(float(atten_db))
    if a > 50:
        beta = 0.1102 * (a - 8.7)
    elif a > 21:
        beta = 0.5842 * (a - 21) ** 0.4 + 0.07886 * (a - 21)
    else:
        beta = 0.0
    return int(math.ceil((a - 7.95) / 2.285 / (math.pi * width) + 1)), beta


def design_taps(decim: int, atten_db: float = 80.0, transition: float = 0.2) -> np.ndarray:
    """Default anti-alias filter of a decimation by ``decim``: a Kaiser-windowed sinc with cutoff 0.5 / decim
    cycles/sample and a transition ``transition / decim`` wide, ``atten_db`` design attenuation, an odd length, unit DC
    gain (float64).  It equals ``scipy.signal.firwin(T, 1 / decim, window=('kaiser', beta))`` with T and beta from
    ``kaiserord(atten_db, 2 transition / decim)`` (T rounded up to odd).  The passband ``|f| <= (0.5 - transition / 2)
    fs / decim`` is free of aliasing; kaiserord is approximate, so the stopband is near but not at ``-atten_db``."""
    decim = int(decim)
    if decim < 1:
        raise ValueError(f"decim {decim} must be >= 1")
    if not 0 < transition < 1:
        raise ValueError(f"transition {transition} must be in (0, 1)")
    if decim == 1:
        return np.ones(1)
    T, beta = kaiser_order(atten_db, 2.0 * transition / decim)
    T += 1 - T % 2
    cutoff = 1.0 / decim                      # of the Nyquist frequency
    m = np.arange(T) - 0.5 * (T - 1)
    h = cutoff * np.sinc(cutoff * m) * np.kaiser(T, beta)
    return h / h.sum()


def phase_increment(shift_hz: float, sample_rate: float) -> tuple:
    """(phase_inc, actual shift in Hz): ``round(shift_hz / fs 2^64)`` as a two's-complement int64, computed exactly, and
    the shift it tunes, ``phase_inc fs / 2^64``.  +fs/2 and -fs/2 are the same increment, -2^63 (reported as -fs/2)."""
    fs = Fraction(sample_rate)
    if fs <= 0:
        raise ValueError("sample_rate must be > 0")
    v = round(Fraction(shift_hz) / fs * (1 << 64))
    inc = (v + (1 << 63)) % (1 << 64) - (1 << 63)
    return int(inc), float(Fraction(inc) * fs / (1 << 64))


class _FirHandle:
    """What ``DdcPlan`` and ``Channelizer`` share: the lifetime of a libspx FIR handle (``spx_<_native>_*``), ``sync``,
    the output count and the part of ``exec`` that marshals the input and calls libspx."""
    _native = ""   # the handle's libspx name: "ddc" or "chan"

    def _fn(self, name: str):
        return getattr(nat.lib(), f"spx_{self._native}_{name}")

    def _create(self, cfg) -> None:
        self._h = None
        nat.require_device()
        h = C.c_void_p()
        nat.check(self._fn("create")(C.byref(h), C.byref(cfg)))
        self._h = h

    @property
    def n_taps(self) -> int:
        return int(self.taps.size)

    @property
    def out_rate(self) -> float:
        return self.sample_rate / self.decim

    def out_count(self, n_samples: int) -> int:
        """(n - T) // decim + 1 outputs (per channel) of n input samples (0 if n < T)."""
        n = int(n_samples)
        return 0 if n < self.n_taps else (n - self.n_taps) // self.decim + 1

    def close(self) -> None:
        h, self._h = getattr(self, "_h", None), None
        if h:
            self._fn("destroy")(h)

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
        nat.check(self._fn("sync")(self._h))

    def _exec(self, x, out, first_sample, stream, n_samples):
        """exec of either handle; the subclass's ``_output(out, mem, n_out)`` allocates or checks the output and returns
        it with the libspx arguments that follow it."""
        if int(first_sample) < 0:
            raise ValueError("first_sample must be >= 0")
        if isinstance(x, np.ndarray) or not (isinstance(x, (DeviceArray, nat.DeviceView)) or hasattr(x, "data_ptr")):
            x = SpectralPlan._host_input(self, x)
        in_ptr, mem = nat.as_ptr(x)
        L = int(n_samples) if n_samples is not None else SpectralPlan._samples_per_stream(self, x, 1)
        if out is not True and nat.as_ptr(out)[1] != mem:
            raise ValueError("out must live where the input lives")
        out, out_args = self._output(out, mem, self.out_count(L))
        n, h2d, d2h = C.c_int64(), C.c_int64(), C.c_int64()
        nat.check(self._fn("exec")(self._h, mem, in_ptr, L, int(first_sample), nat.as_ptr(out)[0], *out_args, C.byref(n),
                                   C.byref(h2d), C.byref(d2h), stream or None))
        self.last_h2d_bytes, self.last_d2h_bytes = int(h2d.value), int(d2h.value)
        return out


def as_jobs(jobs) -> np.ndarray:
    """Jobs of ``DdcPlan.exec_jobs`` as a contiguous ``JOB_DTYPE`` array; ``phase_inc`` of tuples may be given mod 2^64."""
    if isinstance(jobs, np.ndarray) and jobs.dtype == JOB_DTYPE:
        return np.ascontiguousarray(jobs)
    rows = [tuple(int(v) for v in j) for j in jobs]
    rows = [(a, (p + (1 << 63)) % (1 << 64) - (1 << 63), m0, n, o) for a, p, m0, n, o in rows]
    return np.array(rows, dtype=JOB_DTYPE).reshape(-1)


class DdcPlan(_FirHandle):
    """NCO mix by ``-shift_hz``, FIR ``taps`` (default ``design_taps(decim)``) and decimation by ``decim`` of a
    ``sample_rate`` stream, on one GPU.  ``in_fmt`` / ``in_scale`` as in ``SpectralPlan``."""
    _native = "ddc"

    def __init__(self, sample_rate: float, shift_hz: float, decim: int, taps=None, in_fmt: int = FMT_CF32,
                 in_scale: float = 1.0, device: int = 0):
        self.sample_rate = float(sample_rate)
        self.decim = int(decim)
        if self.decim < 1:
            raise ValueError(f"decim {self.decim} must be >= 1")
        self.taps = design_taps(self.decim) if taps is None else np.ascontiguousarray(taps, dtype=np.float64).ravel()
        if not 1 <= self.taps.size <= MAX_TAPS:
            raise ValueError(f"{self.taps.size} taps: one stage takes 1 .. {MAX_TAPS}; for a larger decimation cascade "
                             "two DdcPlans, the second with shift_hz=0")
        if in_fmt not in (FMT_CF32, FMT_CI16):
            raise ValueError(f"unknown in_fmt {in_fmt}")
        self.phase_inc, self.shift_hz = phase_increment(shift_hz, self.sample_rate)
        self.in_fmt, self.in_scale, self.device = int(in_fmt), float(in_scale), int(device)
        self._create(nat.spx_ddc_config(C.sizeof(nat.spx_ddc_config), self.device, self.in_fmt, self.in_scale,
                                        self.decim, self.n_taps, self.taps.ctypes.data, self.phase_inc))

    @property
    def usable_span_hz(self) -> float:
        """Alias-free span of the output around its centre with the default filter: 0.8 fs / decim."""
        return 0.8 * self.out_rate

    def exec(self, x, out=True, first_sample: int = 0, stream: int = 0, n_samples: Optional[int] = None):
        """Outputs of ``x`` (numpy: staged through pinned pieces, returns numpy; DeviceArray / CUDA tensor: enqueued on
        ``stream``, returns a DeviceArray) as complex64 [M].  ``first_sample``: the global index of x's first sample, so
        that pieces of a capture that overlap by ``n_taps - decim`` samples give the outputs of one call.  ``out``: True
        (allocate) or a caller buffer of M complex64 in x's memory space."""
        return self._exec(x, out, first_sample, stream, n_samples)

    def exec_jobs(self, x_dev, jobs, out, in_first_sample: int = 0, stream: int = 0):
        """Many down-conversions of one device-resident capture in one launch (``spx_ddc_exec_jobs``): every job is this
        plan's DDC (taps, decimation, format) with its own NCO ``phase_inc`` and span.  Job ``(first_sample, phase_inc,
        m0, n_out, out_offset)`` writes its outputs ``m0 .. m0 + n_out - 1`` (output m of ``DdcPlan.exec`` on a plan with
        that increment called with ``first_sample``, bit for bit) to ``out[out_offset + m - m0]``.  ``x_dev``: DeviceArray /
        DeviceView / CUDA tensor whose sample 0 has global index ``in_first_sample``; every window a job reads must lie in
        it.  ``jobs``: a structured array of ``JOB_DTYPE`` or a list of 5-tuples.  ``out``: complex64 device buffer;
        the outputs of different jobs must not overlap, and elements no job writes are left untouched.  Enqueued on
        ``stream``; returns ``out``."""
        if isinstance(x_dev, np.ndarray) or not (isinstance(x_dev, (DeviceArray, nat.DeviceView)) or hasattr(x_dev, "data_ptr")):
            raise TypeError("exec_jobs takes device input (DeviceArray, DeviceView or a CUDA tensor)")
        jobs = as_jobs(jobs)
        in_ptr, _ = nat.as_ptr(x_dev)
        L = SpectralPlan._samples_per_stream(self, x_dev, 1)
        out_ptr, mem = nat.as_ptr(out)
        if mem == MEM_HOST:
            raise ValueError("out must be a device buffer")
        live = jobs[jobs["n_out"] > 0]
        need = int((live["out_offset"] + live["n_out"]).max()) if live.size else 0
        have = (out.numel() * out.element_size() if hasattr(out, "data_ptr") else out.nbytes) // 8
        if have < need:
            raise ValueError(f"out holds {have} complex64 outputs; the jobs write up to element {need - 1}")
        nat.check(nat.lib().spx_ddc_exec_jobs(self._h, in_ptr, L, int(in_first_sample), jobs.ctypes.data, len(jobs),
                                              out_ptr, stream or None))
        return out

    def _output(self, out, mem, M):
        if out is True:
            return (np.empty(M, np.complex64) if mem == MEM_HOST else DeviceArray((M,), np.complex64, self.device)), ()
        _check_buffer(out, (M,), np.complex64, "out")
        return out, ()


class Channelizer(_FirHandle):
    """Polyphase filter-bank channelizer (libspx K10, ``spx_chan_*``): splits a ``sample_rate`` stream into
    ``n_channels`` (M, a power of two in [16, 4096]) baseband channels in one pass on one GPU.  Channel j (fftshift order)
    is the ``DdcPlan`` at shift ``(j - M/2) fs / M`` with the same taps and decimation, centred at ``fc + (j - M/2) fs / M``
    and running at ``fs / decim``; a tone at its centre comes out at 0 Hz.

    ``decim``: M / 2 (2x oversampled, the default) or M (critically sampled).  Default taps: ``design_taps(M // 2,
    transition=0.5)`` for M / 2 (cutoff fs / M, the whole channel band |f| <= fs / (2M) alias-free) and ``design_taps(M)``
    for M (the usual compromise: |f| <= 0.4 fs / M alias-free, the channel edges roll off).  Up to 32 M caller taps."""
    _native = "chan"

    def __init__(self, sample_rate: float, n_channels: int, decim: Optional[int] = None, taps=None,
                 in_fmt: int = FMT_CF32, in_scale: float = 1.0, device: int = 0):
        self.sample_rate = float(sample_rate)
        M = int(n_channels)
        if M < 16 or M > 4096 or M & (M - 1):
            raise ValueError(f"n_channels {M} must be a power of two in [16, 4096]")
        self.n_channels = M
        self.decim = M // 2 if decim is None else int(decim)
        if self.decim not in (M, M // 2):
            raise ValueError(f"decim {self.decim} must be n_channels ({M}) or n_channels / 2")
        if taps is None:
            taps = design_taps(M // 2, transition=0.5) if self.decim == M // 2 else design_taps(M)
        self.taps = np.ascontiguousarray(taps, dtype=np.float64).ravel()
        if not 1 <= self.taps.size <= 32 * M:
            raise ValueError(f"{self.taps.size} taps: the channelizer takes 1 .. 32 n_channels = {32 * M}")
        if in_fmt not in (FMT_CF32, FMT_CI16):
            raise ValueError(f"unknown in_fmt {in_fmt}")
        self.in_fmt, self.in_scale, self.device = int(in_fmt), float(in_scale), int(device)
        self._create(nat.spx_chan_config(C.sizeof(nat.spx_chan_config), self.device, self.in_fmt, self.in_scale, M,
                                         self.decim, self.n_taps, self.taps.ctypes.data))

    def channel_freqs(self, center_freq: float = 0.0) -> np.ndarray:
        """Centre frequency of each channel, float64 [M] in fftshift order: fc + (j - M/2) fs / M."""
        M = self.n_channels
        return center_freq + (np.arange(M) - M // 2) * (self.sample_rate / M)

    def exec(self, x, first_sample: int = 0, out=True, stream: int = 0, n_samples: Optional[int] = None):
        """Channels of ``x`` as complex64 [M][n_out] (numpy input: staged through pinned pieces, returns numpy; DeviceArray
        / CUDA tensor: enqueued on ``stream``, returns a DeviceArray).  ``first_sample``: the global index of x's first
        sample, so that pieces that overlap by ``n_taps - decim`` samples give the outputs of one call.  ``out``: True
        (allocate) or a caller buffer [M][S] complex64 with S >= n_out in x's memory space; columns n_out .. S - 1 are
        left untouched."""
        return self._exec(x, out, first_sample, stream, n_samples)

    def _output(self, out, mem, n_out):
        M = self.n_channels
        if out is True:
            out = np.empty((M, n_out), np.complex64) if mem == MEM_HOST else DeviceArray((M, n_out), np.complex64,
                                                                                          self.device)
            return out, (max(n_out, 1),)
        shape = tuple(out.shape)
        if len(shape) != 2 or shape[0] != M or shape[1] < n_out:
            raise ValueError(f"out: expected shape ({M}, S) with S >= {n_out}, got {shape}")
        _check_buffer(out, shape, np.complex64, "out")
        return out, (max(shape[1], 1),)
