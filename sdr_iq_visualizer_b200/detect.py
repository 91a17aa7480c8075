"""Signal detection on a dB image (kernel K11, csrc/spx_detect.cu) -- host binding.

A region is an 8-connected set of cells at least ``threshold_db`` above their row's noise floor (the row's 20th
percentile, as the classifier measures it), with at least ``min_cells`` cells.  Regions are numbered in raster order of
their first cell, as ``scipy.ndimage.label`` numbers them; include/spx.h (spx_detect_regions) has the full definition.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional

import numpy as np

from . import _native as nat

REGION_FIELDS = [f[0] for f in nat.spx_region._fields_]


@dataclass
class Detections:
    regions: List[dict]            # one dict per region (REGION_FIELDS), in numbering order: region k has label k + 1
    row_floor_db: np.ndarray       # float64 [rows] the noise floor of every row
    labels: Optional[object]       # int32 [rows, cols] region labels (0: none), in the input's memory space; None unless asked
    n_total: int                   # regions found (always len(regions))


def _image(db):
    """(pointer, mem, rows, cols, stride, kind, keep) of a float32 dB image given as numpy, DeviceArray / DeviceView or
    torch tensor; rows must be contiguous, numpy input of another dtype is converted to float32."""
    if isinstance(db, (nat.DeviceArray, nat.DeviceView)):
        if db.dtype != np.float32 or len(db.shape) not in (1, 2):
            raise ValueError("a device image must be float32 [rows, cols]")
        rows, cols = (1, db.shape[0]) if len(db.shape) == 1 else db.shape
        return db.ptr, nat.MEM_DEVICE, rows, cols, cols, "device", db
    if hasattr(db, "data_ptr") and hasattr(db, "is_cuda"):   # torch tensor (plumbing only)
        import torch
        t = db if db.dim() == 2 else db.reshape(1, -1)
        if t.dtype != torch.float32 or t.dim() != 2:
            raise ValueError("a tensor image must be float32 [rows, cols]")
        if t.shape[1] > 1 and t.stride(1) != 1:
            t = t.contiguous()
        stride = t.stride(0) if t.shape[0] > 1 else t.shape[1]
        return int(t.data_ptr()), (nat.MEM_DEVICE if t.is_cuda else nat.MEM_HOST), t.shape[0], t.shape[1], stride, "torch", t
    a = np.asarray(db, np.float32)
    if a.ndim == 1:
        a = a[None, :]
    if a.ndim != 2:
        raise ValueError(f"the image must be 2-D, got shape {a.shape}")
    rows, cols = a.shape
    if (cols > 1 and a.strides[1] != 4) or a.strides[0] % 4 or (rows > 1 and a.strides[0] < 4 * cols):
        a = np.ascontiguousarray(a)
    stride = a.strides[0] // 4 if rows > 1 else cols
    return a.ctypes.data, nat.MEM_HOST, rows, cols, stride, "numpy", a


def detect_regions(db, threshold_db: float = 6.0, min_cells: int = 4, want_labels: bool = False, device: int = 0,
                   stream: int = 0) -> Detections:
    """Regions of ``db`` (float32 [rows, cols], one time slice per row, columns in fftshift order) at least
    ``threshold_db`` above their row's noise floor, of at least ``min_cells`` cells.  ``db`` is a numpy array (rows may
    be strided), a DeviceArray or a torch tensor; the labels come back in the same memory space.  The region list is
    never cut: when there are more regions than the first call has room for, the call is repeated with room for all."""
    nat.require_device()
    ptr, mem, rows, cols, stride, kind, keep = _image(db)
    labels = floors = None
    if kind == "torch" and mem == nat.MEM_DEVICE:
        import torch
        dev = keep.device
        if want_labels:
            labels = torch.empty((rows, cols), dtype=torch.int32, device=dev)
        floors = torch.empty((rows,), dtype=torch.float64, device=dev)
        l_ptr = int(labels.data_ptr()) if want_labels else None
        f_ptr = int(floors.data_ptr())
        stream = stream or torch.cuda.current_stream(dev).cuda_stream   # after the work that made the tensor
    elif mem == nat.MEM_DEVICE:
        if want_labels:
            labels = nat.DeviceArray((rows, cols), np.int32, device)
        floors = nat.DeviceArray((rows,), np.float64, device)
        l_ptr, f_ptr = (labels.ptr if want_labels else None), floors.ptr
    else:
        if want_labels:
            labels = np.empty((rows, cols), np.int32)
        floors = np.empty(rows, np.float64)
        l_ptr, f_ptr = (labels.ctypes.data if want_labels else None), floors.ctypes.data
    cap = 1024
    while True:
        out = (nat.spx_region * cap)()
        n = C.c_int32(0)
        nat.check(nat.lib().spx_detect_regions(device, mem, ptr, rows, cols, stride, float(threshold_db), int(min_cells), out,
                                               cap, C.byref(n), l_ptr, f_ptr, stream or None))
        if n.value <= cap:
            break
        cap = n.value
    regions = [{k: getattr(out[i], k) for k in REGION_FIELDS} for i in range(n.value)]
    if kind == "torch" and mem == nat.MEM_DEVICE:
        floors = floors.cpu().numpy()
    elif mem == nat.MEM_DEVICE:
        floors = floors.to_host()
    return Detections(regions, floors, labels, int(n.value))
