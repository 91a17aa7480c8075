#!/usr/bin/env python3
"""GPU micro-benchmark of the fused STFT kernels over shapes, device-resident, CUDA events.
Run on the B200 box:  python tools/kernel_sweep.py [--quick]   (prints one JSON line per case)."""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sdr_iq_visualizer_b200 import _native as nat  # noqa: E402
from sdr_iq_visualizer_b200 import spectral as sp  # noqa: E402

HBM_GBS = 6539.9
try:
    HBM_GBS = json.load(open(os.path.join(os.path.dirname(__file__), "..", "MEASURED_PEAKS.json")))["hbm_gbs"]
except Exception:
    pass


def run_case(name, nfft, hop, window, fmt, L, outs, variant=0, iters=10, flush=False):
    rng = np.random.default_rng(1)
    if fmt == sp.FMT_CI16:
        host = rng.integers(-2047, 2048, size=2 * L, dtype=np.int16)
        in_b = 4
    else:
        host = (rng.standard_normal(2 * L).astype(np.float32)).view(np.complex64)
        in_b = 8
    x = nat.DeviceArray.from_host(host)
    pl = sp.SpectralPlan(nfft, hop, window, fmt, variant=variant)
    F = pl.frame_count(L)
    kw = {}
    out_b = 0
    if "db" in outs:
        kw["db_rows"] = nat.DeviceArray((F, nfft), np.float32); out_b += 4
    if "u8" in outs:
        kw["wf_rows"] = nat.DeviceArray((F, nfft), np.uint8); out_b += 1
    if "acc" in outs:
        kw["welch"] = nat.DeviceArray((1, nfft), np.float64); kw["maxhold"] = nat.DeviceArray((1, nfft), np.float32)
    res, ms = pl.time_stft(x, warmup=3, iters=iters, flush_l2=flush, vmin=-20.0, vmax=100.0, **kw)
    ms = np.array(ms)
    best, med = float(ms.min()), float(np.median(ms))
    bytes_per_sample = in_b + (nfft / hop) * out_b
    gsps = L / (med * 1e-3) / 1e9
    rec = {"case": name, "nfft": nfft, "hop": hop, "fmt": "ci16" if fmt else "cf32", "outs": outs, "variant": variant,
           "samples": L, "frames": F, "ms_med": round(med, 4), "ms_best": round(best, 4), "GSps": round(gsps, 2),
           "Gpts": round(F * nfft / (med * 1e-3) / 1e9, 1), "B_per_sample": bytes_per_sample,
           "hbm_frac": round(gsps * bytes_per_sample / HBM_GBS, 3)}
    print(json.dumps(rec), flush=True)
    pl.close()
    for v in kw.values():
        v.free()
    x.free()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--only4k", action="store_true")
    args = ap.parse_args()
    print(json.dumps(nat.device_info(0)))
    L = 1 << 24 if args.quick else 61_440_000
    run_case("C2 ci16 75% u8+acc", 4096, 1024, "hann", sp.FMT_CI16, L, ["u8", "acc"])
    run_case("headline cf32 hop=N f32", 4096, 4096, "hann", sp.FMT_CF32, L, ["db"])
    run_case("cf32 hop=N u8", 4096, 4096, "hann", sp.FMT_CF32, L, ["u8"])
    run_case("cf32 hop=N acc only", 4096, 4096, "hann", sp.FMT_CF32, L, ["acc"])
    run_case("cf32 50% f32", 4096, 2048, "hann", sp.FMT_CF32, L, ["db"])
    if args.only4k:
        return
    for n in (65536, 16384, 1 << 18):
        run_case(f"cf32 N={n} 50% u8+acc (C5 shape)", n, n // 2, "hann", sp.FMT_CF32, 1 << 26, ["u8", "acc"], 0, iters=5)
        run_case(f"cf32 N={n} hop=N f32", n, n, "hann", sp.FMT_CF32, 1 << 26, ["db"], 0, iters=5)
    for n in (256, 1024, 2048, 8192):
        run_case(f"cf32 N={n} 50% u8+acc", n, n // 2, "hann", sp.FMT_CF32, L, ["u8", "acc"], 0)
        run_case(f"cf32 N={n} hop=N f32", n, n, "hann", sp.FMT_CF32, L, ["db"], 0)


if __name__ == "__main__":
    main()
