"""CPU oracle for the classifier feature path -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

float64 numpy restatement of the measurements taken by the reference's
``classify_signal_advanced`` / ``classify_signal_simple``
(/root/reference/app/processing/classifier.py:15-58,163-219), exposing the intermediate
values (noise floor, threshold, bin indices, peak list) that the CUDA feature kernel is
checked against.  The label rules / temporal smoothing (classifier.py:60-161) are scalar
host logic and are checked end-to-end against the imported reference instead.

Pinned by the reference's own outputs, stored: ``tests/golden/classifier_random.json``
(its helpers on random spectra with ties, ``tests/test_oracle.py::test_classifier_oracle_vs_reference_random``)
and ``tests/golden/classifier_cases.json`` generated from the reference by
``tests/golden/make_golden.py`` (includes SURVEY.md 8(c) KA-1 / KA-2).
"""
from __future__ import annotations

import numpy as np


def noise_floor(power_db) -> float:
    """20th percentile, numpy 'linear' interpolation (classifier.py:179-181)."""
    return float(np.percentile(np.asarray(power_db, dtype=np.float64), 20))


def occupied_edges(power_db, drop_db: float, strict: bool = False):
    """First/last bin index with p >= max - drop (classifier.py:163-170), or p > max - drop
    for the simple classifier (classifier.py:18-19).  Returns (first, last) or (-1, -1)."""
    p = np.asarray(power_db, dtype=np.float64)
    thr = np.max(p) - float(drop_db)
    mask = p > thr if strict else p >= thr
    idx = np.flatnonzero(mask)
    if idx.size == 0:
        return -1, -1
    return int(idx[0]), int(idx[-1])


def occupied_bandwidth(freqs, power_db, drop_db: float, strict: bool = False) -> float:
    a, b = occupied_edges(power_db, drop_db, strict)
    if a < 0:
        return 0.0
    f = np.asarray(freqs)
    return float(f[b] - f[a])


def spectral_flatness(power_db) -> float:
    """geometric/arithmetic mean of 10^(dB/10) clipped at 1e-15 (classifier.py:183-189)."""
    lin = np.maximum(10.0 ** (np.asarray(power_db, dtype=np.float64) / 10.0), 1e-15)
    g = float(np.exp(np.mean(np.log(lin))))
    a = float(np.mean(lin))
    return float(min(max(g / a, 0.0), 1.0))


def spectral_kurtosis(power_db) -> float:
    """Population 4th standardised moment of the dB values; 0 when sigma < 1e-9
    (classifier.py:191-198)."""
    x = np.asarray(power_db, dtype=np.float64)
    mu = float(np.mean(x))
    sd = float(np.std(x))
    if sd < 1e-9:
        return 0.0
    return float(np.mean(((x - mu) / sd) ** 4))


def peak_candidates(power_db, threshold_db: float) -> np.ndarray:
    """Strict interior local maxima above the threshold (the predicate of classifier.py:208)."""
    x = np.asarray(power_db, dtype=np.float64)
    if x.size < 3:
        return np.zeros(0, dtype=np.int64)
    mid = x[1:-1]
    ok = (mid > threshold_db) & (mid > x[:-2]) & (mid > x[2:])
    return np.flatnonzero(ok) + 1


def greedy_peaks(cand: np.ndarray, min_distance_bins: int) -> list:
    """Left-to-right greedy thinning: keep i when i - last_kept >= min_distance
    (classifier.py:205-211; the first candidate is always kept because last starts at
    -min_distance and i >= 1)."""
    kept = []
    last = -int(min_distance_bins)
    for i in cand.tolist():
        if i - last >= min_distance_bins:
            kept.append(i)
            last = i
    return kept


def peak_spacing_std(freqs, peaks) -> float:
    """std of successive peak-frequency differences, 0 for < 3 peaks (classifier.py:214-219)."""
    if len(peaks) < 3:
        return 0.0
    pf = np.asarray(freqs)[np.asarray(peaks, dtype=np.int64)]
    return float(np.std(np.diff(pf)))


def features(freqs, power_db) -> dict:
    """All measurements of classifier.py:45-58 with their intermediates (un-rounded)."""
    p = np.asarray(power_db, dtype=np.float64)
    f = np.asarray(freqs, dtype=np.float64)
    n = p.size
    nf = noise_floor(p)
    peak = float(np.max(p))
    snr = float(peak - nf)
    thr = max(nf + 5.0, peak - 0.9 * snr + 5.0)
    min_dist = max(3, n // 300)
    cand = peak_candidates(p, thr)
    peaks = greedy_peaks(cand, min_dist)
    edges = {d: occupied_edges(p, d) for d in (3, 10, 20)}
    return {
        "n": n,
        "noise_floor_db": nf,
        "peak_db": peak,
        "argmax": int(np.argmax(p)),
        "snr_db": snr,
        "adaptive_thr": float(thr),
        "min_distance_bins": int(min_dist),
        "edges": edges,
        "bw3": occupied_bandwidth(f, p, 3),
        "bw10": occupied_bandwidth(f, p, 10),
        "bw20": occupied_bandwidth(f, p, 20),
        "flatness": spectral_flatness(p),
        "kurtosis": spectral_kurtosis(p),
        "n_candidates": int(cand.size),
        "peaks": peaks,
        "peak_count": len(peaks),
        "peak_spacing_std_hz": peak_spacing_std(f, peaks),
        "simple_edges": occupied_edges(p, 20, strict=True),
    }
