"""SigMF recordings in and out of the GPU spectral path (SURVEY.md section 8(f-3)).

The reference reads a recording with sigmf-python (``fromfile(base).read_samples()``,
/root/reference/scripts/process_sigmf_data.py:49-52), looks at the first 10 000 samples only
(:148,154) and hands them to ``plt.psd`` (:188); the dashboard writes ``cf32_le`` recordings
(/root/reference/app/dashboard/callbacks.py:285-311).  This module keeps those file conventions --

  * ``<base>.sigmf-meta``: JSON with ``global["core:datatype"]`` in {``cf32_le``, ``ci16_le``},
    ``global["core:sample_rate"]``, ``captures[0]["core:frequency"]``;
  * ``<base>.sigmf-data``: raw little-endian interleaved I,Q;
  * ``read_samples`` semantics of sigmf-python 1.2.x: ``ci16_le`` samples are scaled by 2**-15 and
    returned as complex64, ``cf32_le`` as is --

but memory-maps the data file and streams it through the fused STFT kernel in frame-aligned chunks
with (N - hop)-sample halos, so a capture of any length is processed without loading it whole and
without the 10 000-sample cap.  ``ci16_le`` files go to the GPU as int16 (4 B/sample over PCIe) and
are scaled by 2**-15 inside the kernel's window multiply.  Compute is libspx only (no CPU fallback).
"""
from __future__ import annotations

import io
import json
import os
import zipfile
from dataclasses import dataclass, field
from datetime import datetime, timezone
from typing import Iterator, Optional, Tuple

import numpy as np

from . import spectral as sp
from . import timedomain as td
from ._native import FMT_CF32, FMT_CI16

_DATATYPES = {"cf32_le": (np.dtype("<f4"), FMT_CF32, 1.0, 8), "ci16_le": (np.dtype("<i2"), FMT_CI16, 2.0 ** -15, 4)}
_EXTS = (".sigmf-data", ".sigmf-meta")


def resolve_base(path) -> str:
    """Base name of a recording given its data file, its meta file or the base itself
    (process_sigmf_data.py:35-44)."""
    p = os.fspath(path)
    for ext in _EXTS:
        if p.endswith(ext):
            return p[: -len(ext)]
    return p


@dataclass
class SigMFRecording:
    """A memory-mapped SigMF recording: metadata accessors + zero-copy sample access."""
    base: str
    meta: dict
    datatype: str
    raw: np.ndarray = field(repr=False)   # memmap: float32 [2L] (cf32_le) or int16 [2L] (ci16_le)

    # ---- metadata, named after the sigmf-python accessors the reference calls (:88-110,129-137)
    def get_global_info(self) -> dict:
        return dict(self.meta.get("global", {}))

    def get_global_field(self, key, default=None):
        return self.meta.get("global", {}).get(key, default)

    def get_captures(self) -> list:
        return list(self.meta.get("captures", []))

    def get_annotations(self) -> list:
        return list(self.meta.get("annotations", []))

    @property
    def sample_rate(self) -> float:
        return float(self.get_global_field("core:sample_rate", 1.0))

    @property
    def center_freq(self) -> float:
        caps = self.get_captures()
        return float(caps[0].get("core:frequency", 0.0)) if caps else 0.0

    @property
    def n_samples(self) -> int:
        return int(self.raw.shape[0] // 2)

    def __len__(self) -> int:
        return self.n_samples

    @property
    def in_fmt(self) -> int:
        return _DATATYPES[self.datatype][1]

    @property
    def in_scale(self) -> float:
        return _DATATYPES[self.datatype][2]

    @property
    def bytes_per_sample(self) -> int:
        return _DATATYPES[self.datatype][3]

    def frequency_info(self) -> dict:
        """get_frequency_info of the reference script (:125-145)."""
        info = {}
        fc = self.center_freq if self.get_captures() and "core:frequency" in self.get_captures()[0] else None
        if fc:
            info["center_frequency"] = fc
        fs = self.get_global_field("core:sample_rate")
        if fs:
            info["sample_rate"] = fs
            info["bandwidth"] = fs
            if fc:
                info["start_frequency"] = fc - fs / 2
                info["end_frequency"] = fc + fs / 2
        return info

    # ---- samples
    def raw_slice(self, start: int = 0, count: Optional[int] = None) -> np.ndarray:
        """Raw interleaved view (no copy, no scaling) of samples [start, start+count)."""
        stop = self.n_samples if count is None else min(self.n_samples, start + count)
        return self.raw[2 * start: 2 * stop]

    def read_samples(self, start: int = 0, count: Optional[int] = None) -> np.ndarray:
        """complex64, as sigmf-python's read_samples returns it (ci16_le scaled by 2**-15)."""
        r = self.raw_slice(start, count)
        if self.datatype == "cf32_le":
            return np.ascontiguousarray(r, dtype=np.float32).view(np.complex64)
        return (r.astype(np.float32) * np.float32(2.0 ** -15)).view(np.complex64)

    def frame_chunks(self, nfft: int, hop: int, max_chunk_samples: int = 1 << 26) -> Iterator[Tuple[int, int, np.ndarray]]:
        """Frame-aligned pieces of the capture: yields (first_frame, n_frames, raw view).  Consecutive
        pieces overlap by the (nfft - hop)-sample halo, so framing is identical to one pass over the file."""
        L = self.n_samples
        F = (L - nfft) // hop + 1 if L >= nfft else 0
        per = max(1, (max_chunk_samples - nfft) // hop + 1)
        f0 = 0
        while f0 < F:
            nf = min(per, F - f0)
            yield f0, nf, self.raw_slice(f0 * hop, (nf - 1) * hop + nfft)
            f0 += nf


def fromfile(path) -> SigMFRecording:
    """Open ``<base>.sigmf-meta`` + ``<base>.sigmf-data`` (same call name as sigmf-python's, :49)."""
    base = resolve_base(path)
    with open(base + ".sigmf-meta", "r") as fh:
        meta = json.load(fh)
    datatype = meta.get("global", {}).get("core:datatype")
    if datatype not in _DATATYPES:
        raise ValueError(f"unsupported core:datatype {datatype!r} (supported: {sorted(_DATATYPES)})")
    dt = _DATATYPES[datatype][0]
    data_path = base + ".sigmf-data"
    n = os.path.getsize(data_path) // dt.itemsize
    n -= n % 2
    raw = np.memmap(data_path, dtype=dt, mode="r", shape=(n,)) if n else np.zeros(0, dt)
    return SigMFRecording(base, meta, datatype, raw)


def build_metadata(sample_rate, center_freq, datatype: str = "cf32_le", hw: str = "", description: Optional[str] = None,
                   when: Optional[datetime] = None) -> dict:
    """The metadata dictionary the dashboard's recorder emits (callbacks.py:285-304)."""
    when = when or datetime.now(timezone.utc)
    return {
        "global": {
            "core:datatype": datatype,
            "core:sample_rate": int(sample_rate),
            "core:version": "1.0.0",
            "core:description": description or "SDR live stream sample from IQ Visualizer",
            "core:author": "SDR IQ Visualizer Dashboard",
            "core:recorder": "PlutoSDR via pyadi-iio",
            "core:hw": hw or "PlutoSDR",
            "core:license": "CC0-1.0",
        },
        "captures": [{"core:sample_start": 0, "core:frequency": int(center_freq),
                      "core:datetime": when.replace(tzinfo=None).isoformat() + "Z"}],
        "annotations": [],
    }


def _data_bytes(samples, datatype: str) -> bytes:
    a = np.asarray(samples)
    if datatype == "cf32_le":
        return np.ascontiguousarray(a, dtype=np.complex64).tobytes()      # callbacks.py:307-310
    if a.dtype == np.int16:
        return np.ascontiguousarray(a).astype("<i2", copy=False).tobytes()
    iq = np.empty(2 * a.size, dtype="<i2")
    iq[0::2] = np.clip(np.rint(a.real * 32768.0), -32768, 32767)
    iq[1::2] = np.clip(np.rint(a.imag * 32768.0), -32768, 32767)
    return iq.tobytes()


def write_recording(base, samples, sample_rate, center_freq, datatype: str = "cf32_le", **meta_kw) -> str:
    """Write ``<base>.sigmf-data`` / ``.sigmf-meta``.  ``samples``: complex array (any datatype) or
    interleaved int16 (``ci16_le``)."""
    if datatype not in _DATATYPES:
        raise ValueError(f"unsupported datatype {datatype!r}")
    base = resolve_base(base)
    with open(base + ".sigmf-data", "wb") as fh:
        fh.write(_data_bytes(samples, datatype))
    with open(base + ".sigmf-meta", "w") as fh:
        json.dump(build_metadata(sample_rate, center_freq, datatype, **meta_kw), fh, indent=2)
    return base


def recording_zip(samples, sample_rate, center_freq, base_filename: str, hw: str = "") -> bytes:
    """The zip the dashboard's "save" button downloads (callbacks.py:313-345): data + meta + README."""
    x = np.asarray(samples)
    meta = build_metadata(sample_rate, center_freq, "cf32_le", hw=hw)
    buf = io.BytesIO()
    with zipfile.ZipFile(buf, "w", zipfile.ZIP_DEFLATED) as z:
        z.writestr(f"{base_filename}.sigmf-data", _data_bytes(x, "cf32_le"))
        z.writestr(f"{base_filename}.sigmf-meta", json.dumps(meta, indent=2))
        z.writestr("README.txt",
                   "SigMF Recording from SDR IQ Visualizer\n"
                   f"Sample Rate: {sample_rate / 1e6:.2f} MHz\nCenter Frequency: {center_freq / 1e6:.2f} MHz\n"
                   f"Number of Samples: {x.size}\nDuration: {x.size / sample_rate:.3f} seconds\n"
                   f"Files: {base_filename}.sigmf-data (complex float32), {base_filename}.sigmf-meta (JSON)\n")
    return buf.getvalue()


@dataclass
class RecordingSpectra:
    freqs: np.ndarray                 # float64 [N], fftshift order, + center frequency
    pxx: np.ndarray                   # float64 [N] two-sided density (mlab.psd); plot 10*log10
    n_frames: int
    maxhold: Optional[np.ndarray] = None     # float32 [N] max_f |X|^2
    wf_rows: Optional[np.ndarray] = None     # uint8 [F, N]
    hist: Optional[np.ndarray] = None        # uint32 [bins, bins]
    sample_rate: float = 1.0
    center_freq: float = 0.0
    h2d_bytes: int = 0
    d2h_bytes: int = 0
    persistence: Optional[np.ndarray] = None  # uint32 [256, N] frames per waterfall level and bin
    overview_db: Optional[np.ndarray] = None  # float32 [G, N/B] pooled spectrogram (dB)
    overview_wf: Optional[np.ndarray] = None  # uint8 [G, N/B] its levels of [vmin, vmax]
    overview_frames_per_row: int = 0          # K
    overview_bins_per_col: int = 0            # B
    zoom: Optional[tuple] = None              # (actual shift Hz, decim D, taps T) when the spectra are of a zoomed band


def overview_pooling(n_frames: int, nfft: int, rows: int, cols: int) -> tuple:
    """(K, B) of an overview of about ``rows`` x ``cols`` pixels: K = ceil(F / rows) frames per row, B = the largest
    divisor of nfft that is <= nfft / cols bins per column (1 when cols > nfft)."""
    rows, cols, nfft = int(rows), int(cols), int(nfft)
    if rows < 1 or cols < 1:
        raise ValueError(f"overview: rows and cols must be >= 1, got {(rows, cols)}")
    K = max(1, -(-int(n_frames) // rows))
    top = max(1, nfft // cols)
    B = max(d for d in range(1, top + 1) if nfft % d == 0)
    return K, B


def process_recording(path_or_rec, nfft: int = 1024, hop: Optional[int] = None, window="hann", waterfall: bool = False,
                      vmin: float = -120.0, vmax: float = 0.0, maxhold: bool = True, hist_r: Optional[float] = None,
                      hist_bins: int = 256, max_samples: Optional[int] = None, max_chunk_samples: int = 1 << 26,
                      device: int = 0, persistence: bool = False, overview: Optional[tuple] = None,
                      overview_mode: str = "mean", zoom: Optional[tuple] = None, zoom_taps=None) -> RecordingSpectra:
    """The offline path of process_sigmf_data.py on the GPU, for the whole file: Welch PSD with
    ``plt.psd(data, NFFT, Fs, Fc)`` semantics (Hann, ``noverlap = nfft - hop``, default no overlap), plus
    optional max-hold, uint8 waterfall rows and the I/Q density histogram.  ``max_samples`` restores
    the reference's truncation (10 000 there) when wanted.  ``persistence``: the persistence spectrum of the whole
    capture (frames per waterfall level of ``[vmin, vmax]`` and bin, uint32 [256, N]), accumulated on the GPU over the
    file's chunks without bringing the F x N rows to the host (unless ``waterfall`` asks for them too).
    ``overview=(rows, cols)``: a pooled spectrogram of about that many pixels (``overview_pooling`` picks K and B;
    ``overview_mode`` "mean" or "max" detector), accumulated on the GPU over the file's chunks in the same way; its dB
    and levels of ``[vmin, vmax]`` are ``overview_db`` / ``overview_wf``.
    ``zoom=(center_hz, decim)``: analyse the band around the absolute RF frequency ``center_hz`` instead of the whole
    capture.  The file goes through a GPU down-converter (``ddc.DdcPlan``, default taps or ``zoom_taps``) chunk by chunk,
    and every product above is computed on the decimated stream; the result describes that stream (``sample_rate`` fs / D,
    ``center_freq`` fc + the tuned shift, ``freqs`` the zoomed axis, ``zoom`` = (shift, D, T))."""
    rec = path_or_rec if isinstance(path_or_rec, SigMFRecording) else fromfile(path_or_rec)
    hop = int(hop or nfft)
    if max_samples is not None and max_samples < rec.n_samples:
        rec = SigMFRecording(rec.base, rec.meta, rec.datatype, rec.raw[: 2 * max_samples])
    if zoom is not None:
        return _process_zoomed(rec, zoom, zoom_taps, nfft, hop, window, waterfall, vmin, vmax, maxhold, hist_r,
                               max_chunk_samples, device, persistence, overview, overview_mode)
    fs, fc = rec.sample_rate, rec.center_freq
    freqs = sp.freq_axis(nfft, fs, fc)
    L = rec.n_samples
    if overview is not None:
        sp.pool_mode(overview_mode)
        o_rows, o_cols = overview
    if persistence or overview is not None:
        sp.nat.require_device()   # no CPU fallback, whatever the file length
    if L < nfft:   # mlab zero-pads a short input to one frame
        f, pxx = sp.welch_psd(rec.raw_slice() if rec.in_fmt == FMT_CI16 else rec.read_samples(), nfft, hop, window, fs, fc,
                              in_fmt=rec.in_fmt, in_scale=rec.in_scale, device=device)
        # no full frame in the capture: the persistence spectrum counts none (the PSD's single frame is zero-padded)
        out = RecordingSpectra(f, pxx, 1, sample_rate=fs, center_freq=fc,
                               persistence=np.zeros((256, nfft), np.uint32) if persistence else None)
        if overview is not None:   # no full frame: an overview of no rows
            K, B = overview_pooling(0, nfft, o_rows, o_cols)
            out.overview_db = np.zeros((0, nfft // B), np.float32)
            out.overview_wf = np.zeros((0, nfft // B), np.uint8)
            out.overview_frames_per_row, out.overview_bins_per_col = K, B
        return out
    pl = sp.get_plan(nfft, hop, window, rec.in_fmt, rec.in_scale, sp.DB_EPS_REFERENCE, device)
    F = (L - nfft) // hop + 1
    welch = np.zeros((1, nfft), np.float64)
    mh = np.zeros((1, nfft), np.float32) if maxhold else False
    rows = np.empty((F, nfft), np.uint8) if waterfall else None
    hist = np.zeros((hist_bins, hist_bins), np.uint32) if hist_r is not None else None
    counts = np.zeros((1, 256, nfft), np.uint32) if persistence else False
    if overview is not None:
        K, B = overview_pooling(F, nfft, o_rows, o_cols)
        pool = (K, B, overview_mode)
        acc = np.empty((1, -(-F // K), nfft // B), np.float64)
    h2d = d2h = 0
    first = True
    for f0, nf, raw in rec.frame_chunks(nfft, hop, max_chunk_samples):
        x = raw if rec.in_fmt == FMT_CI16 else raw.view(np.complex64)
        # pooling and persistence cannot share a call: with both, the overview takes a call of its own
        both = persistence and overview is not None
        r = pl.stft(x, welch=welch, maxhold=mh, wf_rows=(rows[f0:f0 + nf] if waterfall else False), vmin=vmin, vmax=vmax,
                    persistence=counts, accumulate=not first,
                    **(dict(pool=pool, pool_acc=acc, pool_first_frame=f0) if overview is not None and not both else {}))
        h2d += r.h2d_bytes
        d2h += r.d2h_bytes
        if both:
            r = pl.stft(x, pool=pool, pool_acc=acc, pool_first_frame=f0, accumulate=not first)
            h2d += r.h2d_bytes
            d2h += r.d2h_bytes
        first = False
    if hist is not None:   # every sample once (no halo): the histogram is over the capture, not over frames
        step = max_chunk_samples
        for s0 in range(0, L, step):
            raw = rec.raw_slice(s0, step)
            x = raw if rec.in_fmt == FMT_CI16 else raw.view(np.complex64)
            td.iq_hist2d(x, hist_r, hist_bins, in_fmt=rec.in_fmt, in_scale=rec.in_scale, out=hist, accumulate=True, device=device)
    pxx, _ = pl.welch_finalize(welch[0], F, fs, want_db=False)
    out = RecordingSpectra(freqs, pxx, F, mh[0] if maxhold else None, rows, hist, fs, fc, h2d, d2h,
                           counts[0] if persistence else None)
    if overview is not None:
        o_db, o_wf = pl.pool_finalize(acc, F, K, B, overview_mode, db=True, wf=True, vmin=vmin, vmax=vmax)
        out.overview_db, out.overview_wf = o_db[0], o_wf[0]
        out.overview_frames_per_row, out.overview_bins_per_col = K, B
    return out


def _fir_chunk_runner(fir, rec, max_samples: int, st: int):
    """``run(raw, first_sample, out)``: FIR handle ``fir`` (``ddc.DdcPlan`` or ``ddc.Channelizer``) on a host chunk
    ``raw`` of ``rec`` (up to ``max_samples`` samples, global index of its first sample ``first_sample``) into the device
    buffer ``out``, on the plan stream ``st``.  The chunk is staged in one device buffer of the largest chunk's bytes;
    each run first waits for ``st``, so that the previous chunk's kernels are done with that buffer and with ``out``."""
    from ._native import DeviceArray, DeviceView
    nat, device = sp.nat, fir.device
    d_raw = DeviceArray((max_samples * rec.bytes_per_sample,), np.uint8, device)

    def run(raw, first_sample: int, out) -> None:
        raw = np.ascontiguousarray(raw)
        nat.check(nat.lib().spx_stream_sync(device, st))
        nat.check(nat.lib().spx_memcpy_h2d(device, d_raw.ptr, raw.ctypes.data, raw.nbytes))
        fir.exec(DeviceView(d_raw.ptr, raw.shape, raw.dtype, device), out=out, first_sample=first_sample, stream=st)
    return run


def _process_zoomed(rec, zoom, zoom_taps, nfft, hop, window, waterfall, vmin, vmax, maxhold, hist_r, max_chunk_samples,
                    device, persistence, overview, overview_mode) -> RecordingSpectra:
    """process_recording(zoom=...): each file chunk (``frame_chunks(T, D)``, halo T - D) is uploaded and down-converted
    into a device buffer right after the unframed tail of the decimated stream; the STFT runs on that buffer and its last
    unframed samples (fewer than nfft) are carried to the front of the other of two buffers for the next chunk."""
    from . import ddc as ddc_mod
    from ._native import DeviceArray, DeviceView
    nat = sp.nat
    if hist_r is not None:
        raise ValueError("hist_r is not supported with zoom (the I/Q histogram is of the whole capture)")
    center_hz, decim = zoom
    fs, fc = rec.sample_rate, rec.center_freq
    shift = float(center_hz) - fc
    if abs(shift) > fs / 2:
        raise ValueError(f"zoom centre {center_hz} Hz is {shift} Hz from the capture's centre {fc} Hz: |shift| must be "
                         f"<= fs/2 = {fs / 2} Hz")
    if overview is not None:
        sp.pool_mode(overview_mode)
        o_rows, o_cols = overview
    nat.require_device()
    dd = ddc_mod.DdcPlan(fs, shift, decim, zoom_taps, rec.in_fmt, rec.in_scale, device)
    T, D = dd.n_taps, dd.decim
    fs_z, fc_z = dd.out_rate, fc + dd.shift_hz
    info = (dd.shift_hz, D, T)
    M = dd.out_count(rec.n_samples)
    if M < nfft:   # no full frame of the decimated stream: mlab zero-pads to one frame
        y = dd.exec(rec.raw_slice() if rec.in_fmt == FMT_CI16 else rec.read_samples())
        dd.close()
        f, pxx = sp.welch_psd(y, nfft, hop, window, fs_z, fc_z, device=device)
        out = RecordingSpectra(f, pxx, 1, sample_rate=fs_z, center_freq=fc_z,
                               persistence=np.zeros((256, nfft), np.uint32) if persistence else None, zoom=info)
        if overview is not None:
            K, B = overview_pooling(0, nfft, o_rows, o_cols)
            out.overview_db = np.zeros((0, nfft // B), np.float32)
            out.overview_wf = np.zeros((0, nfft // B), np.uint8)
            out.overview_frames_per_row, out.overview_bins_per_col = K, B
        return out
    pl = sp.get_plan(nfft, hop, window, FMT_CF32, 1.0, sp.DB_EPS_REFERENCE, device)
    st = pl.stream
    F = (M - nfft) // hop + 1
    d_we = DeviceArray((1, nfft), np.float64, device)
    d_mh = DeviceArray((1, nfft), np.float32, device) if maxhold else False
    d_pc = DeviceArray((1, 256, nfft), np.uint32, device) if persistence else False
    rows = np.empty((F, nfft), np.uint8) if waterfall else None
    if overview is not None:
        K, B = overview_pooling(F, nfft, o_rows, o_cols)
        pool = (K, B, overview_mode)
        d_acc = DeviceArray((1, -(-F // K), nfft // B), np.float64, device)
    per = max(1, (max_chunk_samples - T) // D + 1)            # outputs per file chunk, at most
    bufs = [DeviceArray((nfft - 1 + per,), np.complex64, device) for _ in range(2)]
    run_chunk = _fir_chunk_runner(dd, rec, (per - 1) * D + T, st)
    both = persistence and overview is not None   # pooling and persistence cannot share a call
    carry = k = f0 = 0
    for m0, nm, raw in rec.frame_chunks(T, D, max_chunk_samples):
        buf, other = bufs[k & 1], bufs[(k + 1) & 1]
        k += 1
        run_chunk(raw, m0 * D, DeviceView(buf.ptr + 8 * carry, (nm,), np.complex64, device))
        n_avail = carry + nm
        nf = pl.frame_count(n_avail)
        if nf > 0:
            x = DeviceView(buf.ptr, (n_avail,), np.complex64, device)
            d_wf = DeviceArray((nf, nfft), np.uint8, device) if waterfall else False
            pool_kw = dict(pool=pool, pool_acc=d_acc, pool_first_frame=f0) if overview is not None else {}
            pl.stft(x, welch=d_we, maxhold=d_mh, wf_rows=d_wf, vmin=vmin, vmax=vmax, persistence=d_pc,
                    accumulate=f0 > 0, **({} if both else pool_kw))
            if both:
                pl.stft(x, accumulate=f0 > 0, **pool_kw)
            if waterfall:
                pl.sync()
                rows[f0:f0 + nf] = d_wf.to_host()
            f0 += nf
        consumed = nf * hop
        carry = n_avail - consumed
        if carry:
            nat.check(nat.lib().spx_memcpy_d2d_async(device, other.ptr, buf.ptr + 8 * consumed, 8 * carry, st))
    pxx, _ = pl.welch_finalize(d_we, F, fs_z, want_db=False)
    out = RecordingSpectra(sp.freq_axis(nfft, fs_z, fc_z), None, F, sample_rate=fs_z, center_freq=fc_z, wf_rows=rows,
                           zoom=info)
    if overview is not None:
        o_db, o_wf = pl.pool_finalize(d_acc, F, K, B, overview_mode, db=True, wf=True, vmin=vmin, vmax=vmax)
    pl.sync()
    out.pxx = pxx.to_host()
    out.maxhold = d_mh.to_host()[0] if maxhold else None
    out.persistence = d_pc.to_host()[0] if persistence else None
    if overview is not None:
        out.overview_db, out.overview_wf = o_db.to_host()[0], o_wf.to_host()[0]
        out.overview_frames_per_row, out.overview_bins_per_col = K, B
    dd.close()
    return out


@dataclass
class ChannelScan:
    """What ``scan_channels`` measured: one row per channel, channels in fftshift order (lowest frequency first)."""
    channel_freqs: np.ndarray      # float64 [M] RF centre of each channel
    out_rate: float                # channel sample rate fs / D
    freqs: np.ndarray              # float64 [nfft] baseband axis of one channel (add channel_freqs[j] for RF)
    pxx: np.ndarray                # float64 [M, nfft] Welch density of each channel (mlab.psd, two-sided)
    pxx_db: np.ndarray             # float64 [M, nfft] 10 log10 pxx
    maxhold: Optional[np.ndarray]  # float32 [M, nfft] max over frames of |X|^2
    n_frames: int                  # frames per channel
    measurements: list             # per channel: features.measure_batch dict of the measured band, plus bw3/10/20, spacing
    classification: list           # per channel: classify_signal_advanced's result dict (no temporal smoothing)
    band: tuple = (0, 0)           # bins [lo, hi) of each channel's spectrum that were measured and classified


def scan_channels(path_or_rec, n_channels: int = 64, decim: Optional[int] = None, nfft: int = 256, hop: Optional[int] = None,
                  window="hann", maxhold: bool = True, taps=None, max_chunk_samples: int = 1 << 24,
                  device: int = 0) -> ChannelScan:
    """Channel scan of a recording: which channels of the band are occupied, and by what.  The capture is split on the GPU
    into ``n_channels`` baseband channels (``ddc.Channelizer``, default decim n_channels / 2), and every channel gets a
    Welch spectrum (``nfft``, ``hop`` default nfft, ``window``), a max-hold, the classifier measurements and a verdict.

    The file is read chunk by chunk.  Each chunk yields ``nfft + (k - 1) hop`` channel outputs that start on an STFT frame
    boundary, so consecutive chunks overlap by ``(nfft - hop) D + (T - D)`` input samples, and the per-chunk STFT over the
    M channel streams accumulates the Welch sums and max-holds of one pass over the file.  With D = M / 2 only the centre
    nfft / 2 bins (the channel's own fs / M) are measured and classified, so that neighbours seen in the oversampled
    margin do not count; with D = M all bins are.  The classifier runs without its temporal smoothing: M channels are not
    one signal over time."""
    from . import classifier as cls_mod
    from . import ddc as ddc_mod
    from . import features
    from ._native import DeviceArray, DeviceView
    nat = sp.nat
    rec = path_or_rec if isinstance(path_or_rec, SigMFRecording) else fromfile(path_or_rec)
    nfft = int(nfft)
    hop = int(hop or nfft)
    nat.require_device()
    ch = ddc_mod.Channelizer(rec.sample_rate, n_channels, decim, taps, rec.in_fmt, rec.in_scale, device)
    try:
        M, D, T = ch.n_channels, ch.decim, ch.n_taps
        n_total = ch.out_count(rec.n_samples)
        F = (n_total - nfft) // hop + 1 if n_total >= nfft else 0
        if F == 0:
            raise ValueError(f"recording too short: {rec.n_samples} samples give {n_total} channel outputs, fewer than "
                             f"nfft = {nfft}")
        pl = sp.get_plan(nfft, hop, window, FMT_CF32, 1.0, sp.DB_EPS_REFERENCE, device)
        st = pl.stream
        kf = max(1, (((max_chunk_samples - T) // D + 1) - nfft) // hop + 1)   # frames per chunk
        S = (min(kf, F) - 1) * hop + nfft                                    # channel outputs of the largest chunk
        run_chunk = _fir_chunk_runner(ch, rec, (S - 1) * D + T, st)
        d_y = DeviceArray((M, S), np.complex64, device)
        d_we = DeviceArray((M, nfft), np.float64, device)
        d_mh = DeviceArray((M, nfft), np.float32, device) if maxhold else False
        for f0 in range(0, F, kf):
            nf = min(kf, F - f0)
            m0, n_y = f0 * hop, (nf - 1) * hop + nfft
            run_chunk(rec.raw_slice(m0 * D, (n_y - 1) * D + T), m0 * D, d_y)
            pl.stft(DeviceView(d_y.ptr, (M * S,), np.complex64, device), n_streams=M, stream_stride=S, n_samples=n_y,
                    welch=d_we, maxhold=d_mh, accumulate=f0 > 0, stream=st)
        pxx, pdb = pl.welch_finalize(DeviceView(d_we.ptr, (M * nfft,), np.float64, device), F, ch.out_rate, n_streams=M,
                                     stream=st)
        nat.check(nat.lib().spx_stream_sync(device, st))
        pxx, pdb = pxx.to_host().reshape(M, nfft), pdb.to_host().reshape(M, nfft)
        mh = d_mh.to_host() if maxhold else None
        freqs = sp.freq_axis(nfft, ch.out_rate, 0.0)
        chan_f = ch.channel_freqs(rec.center_freq)
    finally:
        ch.close()
    lo, hi = (nfft // 4, nfft - nfft // 4) if D == M // 2 else (0, nfft)
    band = np.ascontiguousarray(pdb[:, lo:hi])
    meas = features.measure_batch(band, device=device)
    out_m, out_c = [], []
    for j, m in enumerate(meas):
        fj = chan_f[j] + freqs[lo:hi]
        out_m.append(cls_mod.add_hz(fj, m))
        out_c.append(cls_mod.classify_from_measurements(fj, m, hi - lo, smooth=False))
    return ChannelScan(chan_f, ch.out_rate, freqs, pxx, pdb, mh, F, out_m, out_c, (lo, hi))


GENERATOR = "sdr_iq_visualizer_b200"


def region_annotation(region: dict, frames_per_row: int, bins_per_col: int, n_frames: int, nfft: int, hop: int,
                      sample_rate: float, center_freq: float, label: str = "signal") -> dict:
    """The SigMF annotation of a region of an overview whose row g pools frames [gK, min((g+1)K, F)) and column c bins
    [cB, (c+1)B) of an nfft-point STFT with hop `hop`.  Bin k covers [fc + (k - N/2 - 1/2) fs/N, fc + (k - N/2 + 1/2) fs/N);
    the samples are those of every frame of the region's rows."""
    K, B, F, N = int(frames_per_row), int(bins_per_col), int(n_frames), int(nfft)
    start = int(region["row0"]) * K * int(hop)
    last_frame = min((int(region["row1"]) + 1) * K, F) - 1
    df = float(sample_rate) / N
    return {
        "core:sample_start": start,
        "core:sample_count": last_frame * int(hop) + N - start,
        "core:freq_lower_edge": float(center_freq) + (int(region["col0"]) * B - N / 2 - 0.5) * df,
        "core:freq_upper_edge": float(center_freq) + ((int(region["col1"]) + 1) * B - N / 2 - 0.5) * df,
        "core:label": label,
        "core:comment": f"peak {region['peak_db'] - region['peak_floor_db']:.1f} dB above its row's noise floor",
        "core:generator": GENERATOR,
    }


def detect_signals(path_or_rec, nfft: int = 1024, hop: Optional[int] = None, window="hann", overview: tuple = (512, 1024),
                   overview_mode: str = "mean", threshold_db: float = 6.0, min_cells: int = 4, label: str = "signal",
                   device: int = 0):
    """Where in time and frequency a recording holds signals: the pooled overview of the whole file
    (``process_recording(..., overview=overview)``), its regions at least ``threshold_db`` above each row's noise floor
    (``detect.detect_regions``), and one SigMF annotation per region (``region_annotation``), sorted by sample_start.
    Returns ``(Detections, annotations)``; ``write_annotations`` stores the annotations with the recording."""
    from . import detect
    rec = path_or_rec if isinstance(path_or_rec, SigMFRecording) else fromfile(path_or_rec)
    hop = int(hop or nfft)
    out = process_recording(rec, nfft, hop, window, maxhold=False, overview=overview, overview_mode=overview_mode,
                            device=device)
    det = detect.detect_regions(out.overview_db, threshold_db, min_cells, device=device)
    K, B = out.overview_frames_per_row, out.overview_bins_per_col
    F = out.n_frames if out.overview_db.shape[0] else 0
    ann = [region_annotation(r, K, B, F, nfft, hop, rec.sample_rate, rec.center_freq, label) for r in det.regions]
    return det, sorted(ann, key=lambda a: a["core:sample_start"])


def write_annotations(path_or_rec, annotations) -> str:
    """Replace the ``annotations`` of a recording's ``<base>.sigmf-meta`` (sorted by core:sample_start, as SigMF asks),
    keeping every other field; the meta file is replaced atomically and the data file is not touched."""
    base = path_or_rec.base if isinstance(path_or_rec, SigMFRecording) else resolve_base(path_or_rec)
    meta_path = base + ".sigmf-meta"
    with open(meta_path, "r") as fh:
        meta = json.load(fh)
    meta["annotations"] = sorted((dict(a) for a in annotations), key=lambda a: a.get("core:sample_start", 0))
    tmp = f"{meta_path}.tmp.{os.getpid()}"
    try:
        with open(tmp, "w") as fh:
            json.dump(meta, fh, indent=2)
        os.replace(tmp, meta_path)
    finally:
        if os.path.exists(tmp):
            os.remove(tmp)
    if isinstance(path_or_rec, SigMFRecording):
        path_or_rec.meta["annotations"] = meta["annotations"]
    return base


def psd(path_or_rec, NFFT: int = 1024, noverlap: int = 0, max_samples: Optional[int] = None, device: int = 0):
    """``plt.psd(data, NFFT=1024, Fs=sample_rate, Fc=center_freq)`` of a recording (:188): returns
    ``(Pxx, freqs)`` in matplotlib's order."""
    out = process_recording(path_or_rec, NFFT, NFFT - noverlap, "hann", maxhold=False, max_samples=max_samples, device=device)
    return out.pxx, out.freqs
