"""Reference of signal detection (K11, include/spx.h spx_detect_regions), float64 numpy + scipy.

For a float32 dB image db[rows][cols]:
  floor[r]   = np.percentile(float64(db[r]), 20)          (NaN if the row holds a NaN, or is all -inf: inf - inf)
  mask[r][c] = float64(db[r][c]) >= floor[r] + threshold_db   (False for NaN cells and NaN floors)
  labels     = scipy.ndimage.label(mask, structure=np.ones((3, 3)))   8-connected, numbered in raster order of first cell
  filter     regions of fewer than min_cells cells get label 0; the rest are renumbered 1 .. n in the same order
  per region row0, row1, col0, col1 (inclusive box), n_cells, the peak (largest db, ties -> smallest raster index) with
             peak_db and peak_floor_db = floor[peak_row], and power_sum = sum of 10^(db/10) in float64."""
import numpy as np
from scipy import ndimage

STRUCTURE = np.ones((3, 3), bool)


def row_floors(db):
    a = np.asarray(db, np.float64)
    with np.errstate(invalid="ignore"):
        return np.array([np.percentile(row, 20) for row in a], np.float64).reshape(a.shape[0])


def mask_of(db, threshold_db, floors=None):
    a = np.asarray(db, np.float64)
    f = row_floors(db) if floors is None else floors
    with np.errstate(invalid="ignore"):
        return a >= (f + np.float64(threshold_db))[:, None]


def label(mask):
    """scipy's 8-connected labels of a boolean mask (int32) and the region count."""
    lab, n = ndimage.label(np.asarray(mask, bool), structure=STRUCTURE)
    return lab.astype(np.int32), int(n)


def detect(db, threshold_db=6.0, min_cells=4):
    """(regions, labels, floors): the region dicts in numbering order, int32 labels [rows, cols], float64 floors [rows]."""
    db = np.asarray(db, np.float32)
    rows, cols = db.shape
    floors = row_floors(db)
    lab, n = label(mask_of(db, threshold_db, floors))
    if n == 0:
        return [], lab, floors
    flat = lab.ravel()
    idx = np.flatnonzero(flat)
    k = flat[idx]
    v64 = db.ravel()[idx].astype(np.float64)
    n_cells = np.bincount(k, minlength=n + 1)[1:]
    power = np.bincount(k, weights=10.0 ** (v64 / 10.0), minlength=n + 1)[1:]
    # peak: per region the largest value (-0 == +0), then the smallest raster index
    o = np.lexsort((idx, -v64, k))
    first = np.searchsorted(k[o], np.arange(1, n + 1))
    peak = idx[o[first]]
    boxes = ndimage.find_objects(lab)
    keep = np.flatnonzero(n_cells >= min_cells)
    new = np.zeros(n + 1, np.int32)
    new[keep + 1] = np.arange(1, keep.size + 1, dtype=np.int32)
    regions = []
    for j in keep:
        sr, sc = boxes[j]
        p = int(peak[j])
        regions.append({
            "row0": sr.start, "row1": sr.stop - 1, "col0": sc.start, "col1": sc.stop - 1,
            "n_cells": int(n_cells[j]), "peak_row": p // cols, "peak_col": p % cols,
            "peak_db": float(db.ravel()[p]), "peak_floor_db": float(floors[p // cols]),
            "power_sum": float(power[j]),
        })
    return regions, new[lab], floors
