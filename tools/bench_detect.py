"""Cost of signal detection (spx_detect_regions: K3 row floors + K11 labelling) on one GPU; prints one JSON line.

Workloads, each at about 5 % and 40 % of the cells above floor + threshold (the threshold is the matching quantile of
db - floor, read from the image):
  (O)  the detect_signals default: a 512 x 1024 overview, mean of 16 frames per cell (10 log10 of a Gamma(16) mean);
  (S)  a full-resolution 4096 x 4096 dB image: 4096 rows of a 4096-point Hann STFT of complex noise.
The image is device-resident.  Reported per workload:
  k3_us      the K3 floor step alone: spx_classify_features_dev over the image rows, CUDA events over many launches;
  k11_us     the K11 kernels of one call (det_*), and k3_in_call_us the K3 kernel in it, from torch.profiler records in a
             run of their own;
  call_us    host wall time of one whole call (it waits for the region table), no profiler.
HBM floor of K11: it must read the image once (4 B/cell) and, with labels, write them (4 B/cell).  Its passes move about
28 B/cell without labels (local: image + parents; flatten: parents read and written; assign: parents; stats: parents and
the image of the masked cells) and 36 B/cell with them; a 4096 x 4096 image (67 MB) and its parents fit the 126 MB L2.
The card's name and power limit are read in the same run.

    python tools/bench_detect.py [--steps 50] [--warmup 5] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

from tools.bench_persistence import gpu_name_power      # noqa: E402

HBM_GBPS = 6539.9


def overview_image(rows=512, cols=1024, seed=1):
    rng = np.random.default_rng(seed)
    return (10 * np.log10(rng.gamma(16.0, 1 / 16.0, size=(rows, cols)))).astype(np.float32)


def stft_image(rows=4096, n=4096, seed=2):
    from sdr_iq_visualizer_b200 import spectral as sp
    rng = np.random.default_rng(seed)
    x = ((rng.normal(size=rows * n) + 1j * rng.normal(size=rows * n)) * 0.01).astype(np.complex64)
    pl = sp.SpectralPlan(n, n, "hann", sp.FMT_CF32)
    db = pl.stft(x, db_rows=True).db_rows
    pl.close()
    return np.ascontiguousarray(db, np.float32)


def threshold_for(db, density):
    f = np.percentile(db.astype(np.float64), 20, axis=1)
    return float(np.quantile(db - f[:, None], 1.0 - density))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from sdr_iq_visualizer_b200 import _native as nat
    nat.require_device()
    lib = nat.lib()
    name, power = gpu_name_power()
    res = {"tool": "bench_detect", "gpu": name, "power_limit": power, "hbm_GBps": HBM_GBPS, "steps": args.steps,
           "warmup": args.warmup, "k11_bytes_per_cell": {"floor": 4, "floor_with_labels": 8, "passes": 28,
                                                         "passes_with_labels": 36}}
    images = {"O_512x1024": overview_image(), "S_4096x4096": stft_image()}
    for wname, db in images.items():
        rows, cols = db.shape
        d_db = nat.DeviceArray.from_host(db)
        d_lab = nat.DeviceArray((rows, cols), np.int32)
        d_feat = nat.DeviceArray((rows * C.sizeof(nat.spx_features),), np.uint8)
        cap = ((rows + 1) // 2) * ((cols + 1) // 2)
        out = (nat.spx_region * cap)()
        n = C.c_int32()
        for density in (0.05, 0.40):
            thr = threshold_for(db, density)
            key = f"{wname}_d{int(density * 100):02d}"

            def call(labels=True):
                nat.check(lib.spx_detect_regions(0, nat.MEM_DEVICE, d_db.ptr, rows, cols, cols, thr, 1, out, cap, C.byref(n),
                                                 d_lab.ptr if labels else None, None, None))

            def k3():
                nat.check(lib.spx_classify_features_dev(0, d_db.ptr, 0, cols, rows, cols, d_feat.ptr, None, 0, None, None))

            for _ in range(args.warmup):
                call()
                k3()
            nat.device_sync(0)
            frac = float(np.mean(d_lab.to_host() > 0))
            # K3 alone: events around many launches
            t = nat.DeviceTimer(0, 0)
            t.start()
            for _ in range(args.steps):
                k3()
            t.stop()
            k3_us = t.elapsed_ms() * 1e3 / args.steps
            t.close()
            # whole call, wall time
            call_us = {}
            for labels in (True, False):
                t0 = time.perf_counter()
                for _ in range(args.steps):
                    call(labels)
                call_us[labels] = (time.perf_counter() - t0) * 1e6 / args.steps
            # kernel times inside the call
            import torch
            from torch.autograd import DeviceType
            from torch.profiler import ProfilerActivity, profile
            torch.cuda.init()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(args.steps):
                    call()
                nat.device_sync(0)
            ev = [e for e in prof.events() if e.device_type == DeviceType.CUDA]
            k11 = sum(e.device_time_total for e in ev if "det_" in e.name) / args.steps
            k3_in = sum(e.device_time_total for e in ev if "features_kernel" in e.name) / args.steps
            per_kernel = {}
            for e in ev:
                if "det_" in e.name:
                    nm = e.name.split("det_")[1].split("_kernel")[0]
                    per_kernel[nm] = per_kernel.get(nm, 0.0) + e.device_time_total / args.steps
            floor_us = rows * cols * 8 / (HBM_GBPS * 1e3)
            res[key] = {"rows": rows, "cols": cols, "threshold_db": round(thr, 4), "mask_fraction": round(frac, 4),
                        "n_regions": n.value, "k3_us": round(k3_us, 2), "k3_in_call_us": round(k3_in, 2),
                        "k11_us": round(k11, 2), "k11_per_kernel_us": {k: round(v, 2) for k, v in per_kernel.items()},
                        "call_us": round(call_us[True], 1), "call_no_labels_us": round(call_us[False], 1),
                        "k11_hbm_floor_us_with_labels": round(floor_us, 2)}
        d_db.free()
        d_lab.free()
        d_feat.free()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
