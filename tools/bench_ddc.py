"""Cost of the zoom DDC (ddc.DdcPlan, K9 ddc_kernel) on one GPU; prints one JSON line.

Shapes:
  (Z1) the config-2 stream, 61.44 M ci16 samples, shift +7.3 MHz, D = 64, default taps (T = 1607);
  (Z2) the same with D = 256 (T = 6425);
  (Z3) 2^28 cf32 samples, D = 8 (T = 203);
  (chain) Z1 followed by an N = 4096 Hann 75 % STFT of the decimated stream (u8 rows, Welch, max-hold), against the plain
          config-2 step (the same STFT of the full-rate stream) in the same run;
  (host) one host-memory Z1 call (pinned input) against spx_copy_ceiling of its bytes.
Device-resident legs are timed with CUDA events after warm-up, alternating round by round; ddc_kernel alone comes from
torch.profiler records in a run of its own.

Algorithmic cost, from the shape alone: bytes per input sample = in_B + 8 / D (read the input, write the outputs);
flops per input sample = 4 T / D + 6 (a complex-by-real MAC is 4 flops, the mix 6; the NCO's sine and cosine are not
counted).  The kernel time is set against the HBM ceiling (6539.9 GB/s, DESIGN.md section 4) and the FP32 peak measured
by spx_fp32_peak in the same run; the larger of the two lower bounds names the binding one.  The card's name and power
limit are read in the same run.

    python tools/bench_ddc.py [--steps 20] [--warmup 3] [--out FILE]
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

from tools.bench_persistence import gpu_name_power   # noqa: E402

HBM_GBPS = 6539.9
FS = 61.44e6
SHIFT = 7.3e6


def cost(n, in_b, T, D):
    return {"bytes": n * (in_b + 8.0 / D), "flops": n * (4.0 * T / D + 6.0)}


def timed(legs, steps, warmup, nat, st):
    for fn in legs.values():
        for _ in range(warmup):
            fn()
    nat.device_sync(0)
    ms = {k: [] for k in legs}
    rounds = 2
    per = max(1, steps // rounds)
    for _ in range(rounds):
        for k, fn in legs.items():
            t = nat.DeviceTimer(0, st)
            t.start()
            for _ in range(per):
                fn()
            t.stop()
            ms[k].append(t.elapsed_ms() / per)
            t.close()
    return {k: (round(float(np.mean(v)), 4), [round(x, 4) for x in v]) for k, v in ms.items()}


def kernel_us(fn, steps, nat):
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    fn()
    nat.device_sync(0)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            fn()
        nat.device_sync(0)
    tot = sum(e.device_time_total for e in prof.events() if e.device_type == DeviceType.CUDA and "ddc_kernel" in e.name)
    return tot / steps


def roofline(c, us, peak_tflops):
    s = us * 1e-6
    t_mem = c["bytes"] / (HBM_GBPS * 1e9)
    t_fp = c["flops"] / (peak_tflops * 1e12)
    bind = "fp32" if t_fp >= t_mem else "hbm"
    return {"kernel_us": round(us, 2), "GB_per_s": round(c["bytes"] / s / 1e9, 1), "TFLOP_per_s": round(c["flops"] / s / 1e12, 2),
            "frac_of_hbm": round(t_mem / s, 3), "frac_of_fp32": round(t_fp / s, 3), "binding": bind,
            "frac_of_binding": round(max(t_mem, t_fp) / s, 3), "flops_per_sample": c["flops"] / c["samples"],
            "bytes_per_sample": c["bytes"] / c["samples"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    from sdr_iq_visualizer_b200 import _native as nat, ddc, spectral as sp, synth
    nat.require_device()
    name, power = gpu_name_power()
    peak = nat.fp32_peak_tflops(0)
    result = {"tool": "bench_ddc", "gpu": name, "power_limit": power, "fp32_peak_tflops": round(peak, 2),
              "hbm_GBps": HBM_GBPS, "steps": args.steps, "warmup": args.warmup,
              "cost_model": "bytes/sample = in_B + 8/D; flops/sample = 4T/D + 6 (sincos not counted)"}
    L2 = 61_440_000
    x2 = synth.tiled_ci16(L2, seed=2)
    d_x2 = nat.DeviceArray.from_host(x2)
    L3 = 1 << 28
    x3 = (synth.tiled_ci16(L3, seed=5).astype(np.float32) * np.float32(2.0 ** -10)).view(np.complex64)
    d_x3 = nat.DeviceArray.from_host(x3)
    del x3
    shapes = {"Z1": (d_x2, L2, sp.FMT_CI16, 2.0 ** -15, 64), "Z2": (d_x2, L2, sp.FMT_CI16, 2.0 ** -15, 256),
              "Z3": (d_x3, L3, sp.FMT_CF32, 1.0, 8)}
    # chain: Z1 + STFT of the decimated stream vs the plain config-2 step; every leg runs on the zoom STFT plan's stream,
    # so that one timer brackets it
    N, hop = 4096, 1024
    pz = sp.SpectralPlan(N, hop, "hann", sp.FMT_CF32)
    p2 = sp.SpectralPlan(N, hop, "hann", sp.FMT_CI16)
    st = pz.stream
    plans, outs, legs = {}, {}, {}
    for k, (d_x, L, fmt, scale, D) in shapes.items():
        p = ddc.DdcPlan(FS, SHIFT, D, in_fmt=fmt, in_scale=scale)
        plans[k] = p
        outs[k] = nat.DeviceArray((p.out_count(L),), np.complex64)
        legs[k] = (lambda p=p, d_x=d_x, o=outs[k]: p.exec(d_x, out=o, stream=st))
    Fz = pz.frame_count(outs["Z1"].shape[0])
    F2 = p2.frame_count(L2)
    wz, w2 = nat.DeviceArray((Fz, N), np.uint8), nat.DeviceArray((F2, N), np.uint8)
    acc = dict(welch=nat.DeviceArray((1, N), np.float64), maxhold=nat.DeviceArray((1, N), np.float32))
    legs["chain_Z1_stft"] = lambda: (legs["Z1"](), pz.stft(outs["Z1"], wf_rows=wz, vmin=20.0, vmax=130.0, **acc))
    legs["plain_c2_step"] = lambda: p2.stft(d_x2, wf_rows=w2, vmin=20.0, vmax=130.0, stream=st, **acc)
    res = timed(legs, args.steps, args.warmup, nat, st)
    for k, (ms, rounds) in res.items():
        result[k + "_ms"] = ms
        result[k + "_ms_rounds"] = rounds
    result["chain_frames"] = Fz
    for k, (d_x, L, fmt, scale, D) in shapes.items():
        in_b = 4 if fmt == sp.FMT_CI16 else 8
        c = dict(cost(L, in_b, plans[k].n_taps, D), samples=L)
        us = kernel_us(legs[k], 3, nat)
        r = roofline(c, us, peak)
        r.update({"samples": L, "fmt": "ci16" if fmt else "cf32", "decim": D, "taps": plans[k].n_taps,
                  "Gsamples_per_s_kernel": round(L / us / 1e3, 2),
                  "Gsamples_per_s_events": round(L / res[k][0] / 1e6, 2)})
        result[k] = r
    # one-shot host-memory call against the copy ceiling of the same bytes
    p = ddc.DdcPlan(FS, SHIFT, 64, in_fmt=sp.FMT_CI16, in_scale=2.0 ** -15)
    xin = nat.pinned_empty(x2.shape, x2.dtype)
    xin[:] = x2
    yo = nat.pinned_empty((p.out_count(L2),), np.complex64)
    p.exec(xin, out=yo)
    t0 = time.perf_counter()
    p.exec(xin, out=yo)
    wall = time.perf_counter() - t0
    sec = C.c_double()
    nat.check(nat.lib().spx_copy_ceiling(0, xin.ctypes.data, xin.nbytes, yo.ctypes.data, yo.nbytes,
                                         16 << 20, 5, C.byref(sec)))
    result["host_Z1"] = {"wall_ms": round(wall * 1e3, 2), "h2d_bytes": p.last_h2d_bytes, "d2h_bytes": p.last_d2h_bytes,
                         "copy_ceiling_ms": round(sec.value * 1e3, 2), "copy_ceiling_of": "input bytes up, output bytes down", "frac_of_copy_ceiling": round(sec.value / wall, 3)}
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
