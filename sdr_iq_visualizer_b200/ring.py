"""Pinned ring-buffer ingest (csrc/spx_ring.cu): the high-rate replacement for the reference's queue of
per-buffer dicts (/root/reference/app/sdr/streamer.py:18,186-200).

    ring = StreamRing(plan, n_slots=4, slot_samples=1 << 22, wf_rows=True, welch=True, maxhold=True)
    buf = ring.acquire()          # numpy view of a page-locked slot: let the radio driver write into it
    buf[:2 * n] = raw_int16       # (or copy)
    ring.commit(n)                # enqueues H2D -> STFT -> D2H, returns immediately
    blk = ring.collect()          # oldest block: dict of numpy views of pinned result buffers
    ...use blk...; ring.release() # slot can be reused

Frames are continuous across slots; every slot is one Welch / max-hold block.  H2D / D2H byte counters
are reported separately in ``stats()``.  A commit is ordered with one-shot calls on the same plan that use its
scratch (N > 8192 or Bluestein lengths), on whatever stream they run: a ring can share a cached plan with them.

Ring depth: consecutive slots upload on two alternating streams.  A producer that keeps ``n_slots - 1`` commits in flight
reaches the PCIe copy ceiling with ``n_slots >= 6`` (0.94 - 1.00 of it on config 2); with 4 slots only one upload is in
flight at a time and ~10 % is lost (profiles/r02_e2e_ring_depth.jsonl).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as nat


class StreamRing:
    def __init__(self, plan, n_slots: int = 4, slot_samples: int = 1 << 22, wf_rows: bool = True, db_rows: bool = False,
                 welch: bool = True, maxhold: bool = True, vmin: float = -100.0, vmax: float = 0.0,
                 features: bool = False, sample_rate: float = 0.0):
        self.plan = plan  # keep the plan alive
        self.nfft = plan.nfft
        self.slot_samples = int(slot_samples)
        self._dtype = np.int16 if plan.in_fmt == nat.FMT_CI16 else np.complex64
        self._per_sample = 2 if plan.in_fmt == nat.FMT_CI16 else 1
        cfg = nat.spx_ring_config(C.sizeof(nat.spx_ring_config), int(n_slots), self.slot_samples, int(wf_rows), int(db_rows),
                                  int(welch), int(maxhold), float(vmin), float(vmax), int(features), 0, float(sample_rate))
        h = C.c_void_p()
        nat.check(nat.lib().spx_ring_create(C.byref(h), plan._h, C.byref(cfg)))
        self._h = h
        self._n_slots = int(n_slots)
        plan._rings.add(self)

    def close(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            nat.lib().spx_ring_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def acquire(self) -> np.ndarray:
        """Writable numpy view (int16 interleaved or complex64) of the next pinned slot."""
        p, cap = C.c_void_p(), C.c_int64()
        nat.check(nat.lib().spx_ring_acquire(self._h, C.byref(p), C.byref(cap)))
        n = int(cap.value) * self._per_sample
        buf = (C.c_char * (n * np.dtype(self._dtype).itemsize)).from_address(p.value)
        return np.frombuffer(buf, dtype=self._dtype, count=n)

    def commit(self, n_samples: int) -> None:
        nat.check(nat.lib().spx_ring_commit(self._h, int(n_samples)))

    def push(self, samples) -> None:
        """acquire + copy + commit for callers that already hold the samples in a numpy array."""
        a = np.ascontiguousarray(samples, dtype=self._dtype).reshape(-1)
        n = a.size // self._per_sample
        if n > self.slot_samples:
            raise ValueError("chunk larger than a slot")
        slot = self.acquire()
        slot[: a.size] = a
        self.commit(n)

    def collect(self) -> dict:
        """Block until the oldest committed slot is done; views stay valid until release()."""
        r = nat.spx_ring_result()
        nat.check(nat.lib().spx_ring_collect(self._h, C.byref(r)))
        F, N = int(r.n_frames), self.nfft

        def view(ptr, shape, dtype):
            if not ptr:
                return None
            n = int(np.prod(shape))
            if n == 0:
                return np.zeros(shape, dtype)
            buf = (C.c_char * (n * np.dtype(dtype).itemsize)).from_address(ptr)
            return np.frombuffer(buf, dtype=dtype, count=n).reshape(shape)

        feats = None
        if r.features:
            from .features import _to_dict
            feats = _to_dict(nat.spx_features.from_address(r.features), None)
        return {"features": feats, "pxx_db": view(r.pxx_db, (N,), np.float64),
                "seq": int(r.seq), "n_frames": F, "first_frame": int(r.first_frame),
                "wf_rows": view(r.wf_rows, (F, N), np.uint8), "db_rows": view(r.db_rows, (F, N), np.float32),
                "welch_acc": view(r.welch_acc, (N,), np.float64), "maxhold": view(r.maxhold, (N,), np.float32),
                "h2d_bytes": int(r.h2d_bytes), "d2h_bytes": int(r.d2h_bytes)}

    def release(self) -> None:
        nat.check(nat.lib().spx_ring_release(self._h))

    def stats(self) -> dict:
        s = nat.spx_ring_stats_t()
        nat.check(nat.lib().spx_ring_stats(self._h, C.byref(s)))
        return {"h2d_bytes": int(s.h2d_bytes), "d2h_bytes": int(s.d2h_bytes), "samples": int(s.samples),
                "frames": int(s.frames), "in_flight": int(s.in_flight)}
