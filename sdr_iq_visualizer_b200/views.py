"""Data side of the dashboard tick and of the chatbot's classify tool (SURVEY.md section 8(f-2), (f-4)).

The reference's ``update_graphs`` (/root/reference/app/dashboard/callbacks.py:95-243) rebuilds, every
300 ms, a float64 [100][N] waterfall array from a deque of rows (:176-190), scatters 2000 random
samples for the constellation (:199-214), finds peak markers with scipy (:150-153) and formats the
classifier line (:224-241).  The functions here produce the same *view data* from GPU results --
uint8 waterfall rows + a 256-entry LUT, an exact I/Q density histogram, GPU peak markers, the same
classifier text -- as plain numpy / dict payloads.  They import no plotting library: a Dash callback
wraps them in ``go.Heatmap`` / ``go.Image`` / ``go.Scatter`` (INTEGRATION.md shows the wiring).
"""
from __future__ import annotations

import threading
from typing import Optional

import numpy as np

from . import classifier as _classifier
from . import features as _features
from . import spectral as _spectral
from . import timedomain as _timedomain

WATERFALL_DEPTH = 100   # rows kept by the reference's deque (callbacks.py:19)


class WaterfallBlock:
    """Rolling block of the newest ``depth`` uint8 waterfall rows (ring buffer, no per-tick re-copy of
    float rows as at callbacks.py:182).  Rows are colormap indices for ``[vmin, vmax]`` dB."""

    def __init__(self, nfft: int, depth: int = WATERFALL_DEPTH, vmin: float = -20.0, vmax: float = 120.0):
        self.nfft, self.depth, self.vmin, self.vmax = int(nfft), int(depth), float(vmin), float(vmax)
        self._rows = np.zeros((self.depth, self.nfft), np.uint8)
        self._count = 0
        self._lock = threading.Lock()

    def push_rows(self, rows_u8) -> None:
        rows = np.asarray(rows_u8, dtype=np.uint8).reshape(-1, self.nfft)[-self.depth:]
        with self._lock:
            for r in rows:
                self._rows[self._count % self.depth] = r
                self._count += 1

    def push_db(self, power_db) -> None:
        """One float dB row from a frame dict that carries no ``wf_row`` (e.g. a dict built by other code): the
        display quantisation ``clip(floor((dB - vmin) * 256 / (vmax - vmin)), 0, 255)`` of SURVEY A7 applied to the
        ALREADY COMPUTED spectrum.  The streaming path does not come through here: with
        ``SDRDataStreamer.waterfall_range`` set, the kernel emits the uint8 row itself and ``push_rows`` takes it."""
        q = np.floor((np.asarray(power_db, dtype=np.float64) - self.vmin) * (256.0 / (self.vmax - self.vmin)))
        self.push_rows(np.clip(np.nan_to_num(q, nan=0.0, posinf=255.0, neginf=0.0), 0, 255).astype(np.uint8)[None, :])

    def __len__(self) -> int:
        return min(self._count, self.depth)

    def rows(self) -> np.ndarray:
        """uint8 [len, N], oldest row first (the order ``np.array(waterfall_data)`` has)."""
        with self._lock:
            n = len(self)
            if self._count <= self.depth:
                return self._rows[:n].copy()
            k = self._count % self.depth
            return np.concatenate([self._rows[k:], self._rows[:k]])

    def rgb(self) -> np.ndarray:
        """uint8 [len, N, 3] image through the Viridis LUT (for ``go.Image`` / PNG)."""
        return _spectral.viridis_lut()[self.rows()]

    def heatmap_payload(self, freqs_mhz=None) -> dict:
        """Arguments of the reference's ``go.Heatmap`` (:183-190) with a uint8 ``z`` and a fixed colour range."""
        z = self.rows()
        lut = _spectral.viridis_lut()
        scale = [[i / 255.0, "rgb(%d,%d,%d)" % tuple(lut[i])] for i in range(0, 256, 15)]
        return {"z": z, "x": freqs_mhz, "y": list(range(len(z))), "zmin": 0, "zmax": 255, "colorscale": scale,
                "db_range": (self.vmin, self.vmax)}


def persistence_payload(counts, n_frames: int, vmin: float, vmax: float, freqs_mhz=None) -> dict:
    """Arguments of a ``go.Heatmap`` of a persistence spectrum (``SpectralPlan.stft(persistence=...)``, one stream's
    uint32 [256, N] counts, or [1, 256, N]), in the style of ``WaterfallBlock.heatmap_payload``: ``z`` is the fraction of the
    ``n_frames`` frames at each level and bin (float32 [256, N], rows = levels), ``y`` the lower dB edge of each level
    (level q covers [vmin + q*D, vmin + (q+1)*D), D = (vmax - vmin)/256; level 0 also holds everything below vmin,
    level 255 everything above).  Decay and log colour scaling are left to the caller."""
    c = np.asarray(counts)
    if c.ndim == 3:   # [S][256][N]: one stream only, so that no stream is dropped unseen (pass counts[s] for the others)
        if c.shape[0] != 1:
            raise ValueError(f"counts: {c.shape[0]} streams; pass one stream's [256, N] counts")
        c = c[0]
    if c.ndim != 2 or c.shape[0] != 256:
        raise ValueError(f"counts: expected shape (256, N), got {c.shape}")
    z = c.astype(np.float32) / np.float32(max(int(n_frames), 1))
    y = vmin + np.arange(256, dtype=np.float64) * ((vmax - vmin) / 256.0)
    lut = _spectral.viridis_lut()
    scale = [[i / 255.0, "rgb(%d,%d,%d)" % tuple(lut[i])] for i in range(0, 256, 15)]
    return {"z": z, "x": freqs_mhz, "y": y, "zmin": 0.0, "zmax": 1.0, "colorscale": scale, "db_range": (vmin, vmax)}


def spectrogram_payload(db_or_levels, frames_per_row: int, hop: int, sample_rate: float, freqs_mhz=None,
                        vmin: float = -100.0, vmax: float = 0.0) -> dict:
    """Arguments of a ``go.Heatmap`` of a pooled spectrogram (``SpectralPlan.pool_finalize`` / ``process_recording(
    overview=...)``, one stream's [G, C] float32 dB or uint8 levels, or [1, G, C]), in the style of
    ``persistence_payload``: ``z`` as given (rows = pooled rows, oldest first), ``x`` the column frequencies
    (``spectral.pooled_freq_axis`` in MHz), ``y`` each row's start time in seconds, g * K * hop / fs.  dB is shown over
    [vmin, vmax], levels over [0, 255]."""
    z = np.asarray(db_or_levels)
    if z.ndim == 3:   # [S][G][C]: one stream only, so that no stream is dropped unseen
        if z.shape[0] != 1:
            raise ValueError(f"pooled rows: {z.shape[0]} streams; pass one stream's [G, C] rows")
        z = z[0]
    if z.ndim != 2:
        raise ValueError(f"pooled rows: expected shape (G, C), got {z.shape}")
    if int(frames_per_row) < 1 or int(hop) < 1 or not sample_rate > 0:
        raise ValueError("frames_per_row and hop must be >= 1 and sample_rate > 0")
    y = np.arange(z.shape[0], dtype=np.float64) * (int(frames_per_row) * int(hop) / float(sample_rate))
    levels = z.dtype == np.uint8
    lut = _spectral.viridis_lut()
    scale = [[i / 255.0, "rgb(%d,%d,%d)" % tuple(lut[i])] for i in range(0, 256, 15)]
    return {"z": z, "x": freqs_mhz, "y": y, "zmin": 0 if levels else vmin, "zmax": 255 if levels else vmax,
            "colorscale": scale, "db_range": (vmin, vmax)}


def constellation_density(samples, r: Optional[float] = None, bins: int = 256, in_fmt: int = _spectral.FMT_CF32,
                          in_scale: float = 1.0, device: int = 0) -> dict:
    """Exact I/Q density over ALL samples (kernel K4) instead of a random 2000-point scatter (:199-214).
    ``r`` defaults to the largest |I| or |Q| present (rounded up to a power of two)."""
    x = np.asarray(samples)
    if r is None:
        if in_fmt == _spectral.FMT_CI16:
            m = float(np.abs(x).max()) * in_scale if x.size else 1.0
        else:
            m = float(max(np.abs(x.real).max(), np.abs(x.imag).max())) if x.size else 1.0
        r = float(2.0 ** np.ceil(np.log2(max(m, 1e-30))))
    if in_fmt == _spectral.FMT_CF32 and x.dtype != np.complex64:
        x = x.astype(np.complex64)
    h = _timedomain.iq_hist2d(x, r, bins, in_fmt=in_fmt, in_scale=in_scale, device=device)
    edges = np.linspace(-r, r, bins + 1)
    centers = 0.5 * (edges[:-1] + edges[1:])
    return {"z": h.T, "x": centers, "y": centers, "r": r, "counts": h}   # z[j][i]: rows = Q, columns = I


def peak_markers(power_db, device: int = 0) -> np.ndarray:
    """Peak marker indices for the spectrum plot: the classifier's strict-local-maximum rule above its
    adaptive threshold (classifier.py:53,200-212) with the dashboard's spacing ``max(5, n // 200)``
    (:152).  Replaces ``scipy.signal.find_peaks(distance, prominence=3)`` -- same intent, GPU pick;
    the two rules differ on shoulders (prominence is not evaluated)."""
    p = np.asarray(power_db)
    if p.size < 3:
        return np.zeros(0, np.int64)
    m = _features.measure(p, device=device, min_distance_bins=max(5, p.size // 200))
    return np.asarray(m["peaks"], dtype=np.int64)


def classification_text(freqs, power_db) -> str:
    """The dashboard's classifier line (callbacks.py:224-241), same format and error text."""
    try:
        res = _classifier.classify_signal_advanced(freqs, power_db)
        feats = res.get('features', {})
        return (f"Detected: {res.get('label', 'Unknown')} (conf {res.get('confidence', 0.0):.2f}) — "
                f"OBW20={feats.get('bandwidth_hz_20db', 0.0) / 1e6:.2f}MHz SNR={feats.get('snr_db', 0.0):.1f}dB | "
                f"Flat {feats.get('spectral_flatness', 0.0):.2f} | Kurt {feats.get('spectral_kurtosis', 0.0):.2f} | "
                f"Peaks {feats.get('peak_count', 0)}\n{res.get('explanation', '')}")
    except Exception as e:  # the reference shows the failure instead of raising (:240-241)
        return f"Classification unavailable: {e}"


def classify_tool_text(data: Optional[dict]) -> dict:
    """The chatbot's ``classify_signal`` tool (chatbot.py:146-176) on a frame dict obtained with
    ``SDRDataStreamer.peek_latest()``: returns ``{'stats': str, 'include_graph': 'fd' | None}``."""
    if data is None:
        return {"stats": "No SDR data available yet. Please start streaming.", "include_graph": None}
    try:
        res = _classifier.classify_signal_advanced(data['freqs'], data['power_db'])
        feats = res.get('features', {})
        reasons = res.get('reasons', [])
        reason_text = "\n- " + "\n- ".join(reasons) if reasons else ""
        return {"stats": (f"Classification: {res.get('label', 'Unknown')} (conf {res.get('confidence', 0.0):.2f})\n"
                          f"OBW20={feats.get('bandwidth_hz_20db', 0.0) / 1e6:.2f} MHz, "
                          f"SNR={feats.get('snr_db', 0.0):.1f} dB{reason_text}"), "include_graph": 'fd'}
    except Exception as e:
        return {"stats": f"Classification error: {e}", "include_graph": 'fd'}


def dashboard_tick(data: Optional[dict], waterfall: WaterfallBlock, device: int = 0) -> Optional[dict]:
    """Everything one ``update_graphs`` tick needs from one frame dict (streamer.py:123-130), as data."""
    if data is None:
        return None
    samples, freqs, power_db = data['samples'], data['freqs'], data['power_db']
    if data.get('wf_row') is not None:
        waterfall.push_rows(data['wf_row'])      # quantised by the kernel (streamer.waterfall_range)
    else:
        waterfall.push_db(power_db)
    peaks = peak_markers(power_db, device=device)
    return {
        "time_ms": np.arange(len(samples)) / data['sample_rate'] * 1000,      # :114
        "i": np.real(samples), "q": np.imag(samples),
        "freqs_mhz": freqs / 1e6, "power_db": power_db,
        "peak_freqs_mhz": freqs[peaks] / 1e6, "peak_db": np.asarray(power_db)[peaks],
        "waterfall": waterfall.heatmap_payload(freqs / 1e6),
        "constellation": constellation_density(samples, device=device),
        "classification": classification_text(freqs, power_db),
    }
