"""Signal classification -- drop-in for /root/reference/app/processing/classifier.py.

Public surface kept: ``classify_signal_simple(freqs, power_db) -> str`` (classifier.py:15),
``classify_signal_advanced(freqs, power_db) -> dict`` (classifier.py:30, result keys :146-161), the
rolling ``_CLASS_HISTORY`` / ``_CONF_HISTORY`` deques (:5-6) and the private helper names
(:163-219).  All array work (max, percentile, masks, flatness/kurtosis moments, the peak scan that
is a Python loop in the reference) runs in one CUDA kernel (csrc/spx_features.cu); what remains
here is scalar: Hz from bin indices via the caller's ``freqs``, the ordered rule table and the
12-frame temporal smoothing.  No CPU fallback: without a GPU the calls raise ``SpectralError``.
"""
from __future__ import annotations

import threading
from collections import Counter, deque

import numpy as np

from . import features as _features

# rolling history for temporal smoothing (about the last 12 frames), shared like the reference's
_CLASS_HISTORY = deque(maxlen=12)
_CONF_HISTORY = deque(maxlen=12)
_HISTORY_LOCK = threading.Lock()  # dashboard, stream and chatbot threads all call in (SURVEY.md section 5)

_NO_DATA = {"label": "No Data", "confidence": 0.0, "features": {}, "explanation": "No spectrum data"}


def _span(freqs, first: int, last: int) -> float:
    if last < 0 or first < 0:
        return 0.0
    return float(freqs[last] - freqs[first])


def _spacing_std(freqs, peaks) -> float:
    if len(peaks) < 3:
        return 0.0
    pf = np.asarray(freqs)[np.asarray(peaks, dtype=np.int64)]
    return float(np.std(np.diff(pf)))


def add_hz(freqs, m: dict) -> dict:
    """Adds to a ``features.measure_batch`` result (with its peak list) the Hz quantities derived from the caller's
    frequency axis, un-rounded: occupied bandwidths bw3 / bw10 / bw20 and the peak-spacing sigma.  Returns ``m``."""
    m["bw3"] = _span(freqs, m["first_3db"], m["last_3db"])
    m["bw10"] = _span(freqs, m["first_10db"], m["last_10db"])
    m["bw20"] = _span(freqs, m["first_20db"], m["last_20db"])
    m["peak_spacing_std_hz"] = _spacing_std(freqs, m["peaks"])   # the list is complete (features.measure_batch raises otherwise)
    return m


def measure(freqs, power_db) -> dict:
    """GPU measurements + the Hz quantities derived from the caller's frequency axis (un-rounded)."""
    return add_hz(freqs, _features.measure(power_db))


def classify_signal_simple(freqs, power_db):
    if len(freqs) == 0:
        return "No Data"
    m = _features.measure(power_db)
    if m["simple_last"] < 0:
        return "Noise"
    bw = freqs[m["simple_last"]] - freqs[m["simple_first"]]
    if bw < 3e6:
        return "Narrowband"
    if bw > 15e6:
        return "Wideband"
    return "Unknown"


# ordered rule table: (predicate, label, confidence, reason) over the measurement namespace `v`
_RULES = [
    (lambda v: v.snr < 3,
     "Low SNR / Noise", lambda v: 0.45,
     lambda v: f"Low SNR ({v.snr:.1f} dB) below 3 dB threshold"),
    (lambda v: v.sfm > 0.85 and v.snr < 8 and v.occ > 0.5,
     "Broadband Noise / Hash", lambda v: 0.55,
     lambda v: f"High spectral flatness ({v.sfm:.2f}) with moderate SNR and broad occupancy ({v.occ:.2f})"),
    (lambda v: v.peaks == 1 and v.bw20 < 60e3 and v.sfm < 0.4,
     "CW Carrier", lambda v: 0.8 if v.snr > 6 else 0.6,
     lambda v: f"Single strong peak, OBW20 {v.bw20/1e3:.0f} kHz, flatness {v.sfm:.2f}"),
    (lambda v: 2 <= v.peaks <= 4 and v.bw20 < 600e3 and v.sfm < 0.55,
     "Multitone / FSK-like", lambda v: 0.7 if v.snr > 6 else 0.55,
     lambda v: f"Few peaks ({v.peaks}) with narrow OBW20 {v.bw20/1e3:.0f} kHz and low flatness {v.sfm:.2f}"),
    (lambda v: 88e6 <= v.mid <= 108e6 and 110e3 <= v.bw20 <= 300e3 and 0.15 < v.sfm < 0.6 and v.snr > 8,
     "FM Broadcast (candidate)", lambda v: 0.78,
     lambda v: "In FM band with plausible OBW and features"),
    (lambda v: v.bw20 > 10e6 and 0.25 < v.sfm < 0.9 and v.density > 0.02 and v.spacing / max(v.bw20, 1) < 0.12,
     "Wideband OFDM / Multi-carrier", lambda v: 0.82 if v.peaks > 20 else 0.7,
     lambda v: f"Wide OBW {v.bw20/1e6:.1f} MHz with many peaks ({v.peaks}) and regular spacing"),
    (lambda v: v.bw20 < 600e3 and v.snr > 4 and v.peaks <= 2 and v.sfm < 0.5,
     "Narrowband (voice)", lambda v: 0.65,
     lambda v: "Narrow OBW with few peaks and low flatness (voice-like)"),
    (lambda v: v.bw20 < 600e3 and v.snr > 4 and v.peaks > 4,
     "Channelized Narrowband", lambda v: 0.6,
     lambda v: "Narrow OBW with multiple peaks (channelized)"),
    (lambda v: v.bw20 < 600e3 and v.snr > 4,
     "Narrowband", lambda v: 0.55,
     lambda v: "Narrow OBW with moderate features"),
    (lambda v: v.occ > 0.6 and v.snr > 6 and v.density < 0.01 and 0.4 < v.sfm < 0.8,
     "Wideband Structured", lambda v: 0.55,
     lambda v: "High occupancy with structured spectrum (not noise)"),
]
_FALLBACKS = [
    (lambda v: v.snr > 10 and v.bw20 < 1e6, "Narrowband (generic)", "Fallback: strong SNR and narrow OBW"),
    (lambda v: v.snr > 10 and v.bw20 > 5e6, "Wideband (generic)", "Fallback: strong SNR and wide OBW"),
]


class _V:
    __slots__ = ("snr", "sfm", "kurt", "bw3", "bw10", "bw20", "peaks", "spacing", "density", "mid", "occ")


def _apply_rules(v):
    label, confidence, reasons = "Unknown", 0.25, []
    for pred, lab, conf, why in _RULES:
        if pred(v):
            label, confidence = lab, conf(v)
            reasons.append(why(v))
            break
    if label == "Unknown":
        for pred, lab, why in _FALLBACKS:
            if pred(v):
                label, confidence = lab, max(confidence, 0.5)
                reasons.append(why)
                break
    return label, confidence, reasons


def _smooth(label, confidence, reasons):
    """12-deep majority smoothing on the module-global history (classifier.py:125-139)."""
    with _HISTORY_LOCK:
        _CLASS_HISTORY.append(label)
        _CONF_HISTORY.append(confidence)
        counts = Counter(_CLASS_HISTORY)
        top_label, top_count = counts.most_common(1)[0]
        stability = top_count / len(_CLASS_HISTORY)
        if stability >= 0.5 and top_label != label:
            past = [c for l, c in zip(_CLASS_HISTORY, _CONF_HISTORY) if l == top_label]
            blended = (np.mean(past) + confidence) / 2
            label = top_label
            confidence = min(0.95, max(confidence, blended + 0.05 * stability))
            reasons.append(f"Temporal smoothing applied; adopting stable label '{top_label}' (stability {stability:.2f})")
        else:
            confidence = min(0.95, confidence + 0.05 * (counts[label] / len(_CLASS_HISTORY)))
    return label, confidence, stability


def classify_signal_advanced(freqs, power_db):
    """Return dict(label, confidence, features{...}, explanation, reasons) -- same keys, rounding and
    text as the reference (classifier.py:146-161)."""
    if len(freqs) == 0 or len(power_db) == 0:
        return dict(_NO_DATA)
    return classify_from_measurements(freqs, measure(freqs, power_db), len(power_db))


def with_hz(freqs, m: dict) -> dict:
    """Hz quantities for measurements that came back without a peak list (the ingest ring computes them on the
    device per Welch block): occupied bandwidths from the bin edges, peak-spacing sigma from its value in bins
    (the frequency axis is uniform)."""
    m = dict(m)
    m["bw3"] = _span(freqs, m["first_3db"], m["last_3db"])
    m["bw10"] = _span(freqs, m["first_10db"], m["last_10db"])
    m["bw20"] = _span(freqs, m["first_20db"], m["last_20db"])
    df = float(freqs[1] - freqs[0]) if len(freqs) > 1 else 0.0
    m["peak_spacing_std_hz"] = float(m.get("peak_spacing_std_bins", 0.0)) * df
    return m


def classify_from_measurements(freqs, m: dict, n_bins: int, smooth: bool = True):
    """Label rules + temporal smoothing (classifier.py:60-161) on measurements already taken (``measure`` or
    ``with_hz``): scalar host logic only.  ``smooth=False`` applies the rules alone and leaves the module-global history
    untouched, for spectra that are not one signal over time (e.g. the channels of a channel scan); the label and
    confidence are then the rule table's and the reported stability is 1."""
    power_db = range(n_bins)   # only its length is used below
    v = _V()
    v.snr, v.sfm, v.kurt = float(m["snr_db"]), float(m["flatness"]), float(m["kurtosis"])
    v.bw3, v.bw10, v.bw20 = m["bw3"], m["bw10"], m["bw20"]
    v.peaks = int(m["peak_count"])
    v.spacing = m["peak_spacing_std_hz"]
    v.density = v.peaks / max(len(power_db), 1)
    v.mid = float((freqs[0] + freqs[-1]) / 2.0)
    span_hz = float(freqs[-1] - freqs[0])
    v.occ = v.bw20 / span_hz if span_hz > 0 else 0.0

    label, confidence, reasons = _apply_rules(v)
    if smooth:
        label, confidence, stability = _smooth(label, confidence, reasons)
    else:
        stability = 1.0

    explanation = (
        f"SNR={v.snr:.1f} dB | peaks={v.peaks} (density {v.density:.3f}) | flat={v.sfm:.2f} | kurt={v.kurt:.2f} "
        f"| OBW20={v.bw20/1e6:.2f} MHz (OBW3={v.bw3/1e6:.3f} MHz) | spacingσ={v.spacing/1e3:.1f} kHz | stability={stability:.2f}"
    )
    return {
        "label": label,
        "confidence": round(confidence, 2),
        "features": {
            "bandwidth_hz_3db": float(v.bw3),
            "bandwidth_hz_10db": float(v.bw10),
            "bandwidth_hz_20db": float(v.bw20),
            "snr_db": float(round(v.snr, 2)),
            "spectral_flatness": float(round(v.sfm, 3)),
            "spectral_kurtosis": float(round(v.kurt, 3)),
            "peak_count": int(v.peaks),
            "peak_spacing_std_hz": float(v.spacing),
        },
        "explanation": explanation,
        "reasons": reasons,
    }


# ---- private helpers kept under the reference's names (classifier.py:163-219), GPU-backed
def _occupied_bandwidth(freqs, power_db, drop_db=20):
    if len(power_db) == 0:
        return 0.0
    m = _features.measure(power_db, drops=(float(drop_db), 10.0, 20.0))
    return _span(freqs, m["first_3db"], m["last_3db"])


def _estimate_noise_floor(power_db):
    return float(_features.measure(power_db)["noise_floor_db"])


def _estimate_snr(power_db):
    """Unused by the reference (classifier.py:172-177); kept for API completeness, scalar numpy."""
    if len(power_db) < 4:
        return 0.0
    return np.percentile(power_db, 95) - np.median(power_db)


def _spectral_flatness(power_db):
    return float(_features.measure(power_db)["flatness"])


def _spectral_kurtosis(power_db):
    return float(_features.measure(power_db)["kurtosis"])


def _find_peaks(power_db, threshold_db, min_distance_bins=5):
    if len(power_db) < 3:
        return []
    # reference loop (classifier.py:200-212): a distance <= 0 keeps EVERY strict local maximum, exactly like 1 or 2
    # (strict maxima are never adjacent); the kernel reads 0 as "use max(3, n//300)", so pass 1 for those
    md = int(min_distance_bins)
    m = _features.measure(power_db, peak_threshold_db=float(threshold_db), min_distance_bins=md if md >= 1 else 1)
    return list(m["peaks"])


def _peak_spacing_std(freqs, peak_idx):
    return _spacing_std(freqs, peak_idx)
