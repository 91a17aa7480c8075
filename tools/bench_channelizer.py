"""Cost of the polyphase channelizer (ddc.Channelizer, K10 chan_kernel) on one GPU; prints one JSON line.

Shapes:
  (CH1) the config-2 stream, 61.44 M ci16 samples, M = 64, D = 32, default taps (T = 323);
  (CH2) 2^28 cf32 samples, M = 1024, D = 512 (T = 5141);
  (CH3) 2^28 cf32 samples, M = 1024, D = 1024, critically sampled (T = 25 697);
  (baseline) CH1 as 64 DdcPlan calls (K9, shifts (j - 32) fs / 64, the channelizer's taps and D), in the same run;
  (chain) CH1, then per channel an N = 256 Hann 50 % Welch and max-hold (one multi-stream STFT), the batched Welch
          finalize and 64 classifier measurements;
  (host) one host-memory CH1 call (pinned input and output) against spx_copy_ceiling of its bytes.
Device-resident legs are timed with CUDA events after warm-up, alternating round by round; chan_kernel alone comes from
torch.profiler records in a run of its own.

Algorithmic cost, from the shape alone: bytes per input sample = in_B + 8 M / D (read the input, write M / D complex64
outputs per sample); flops per input sample = (4 T + 5 M log2 M) / D (a complex-by-real MAC is 4 flops; an M-point FFT
5 M log2 M).  The kernel time is set against the HBM ceiling (6539.9 GB/s, DESIGN.md section 4) and the FP32 peak
measured by spx_fp32_peak in the same run; the larger of the two lower bounds names the binding one.  The card's name and
power limit are read in the same run.

    python tools/bench_channelizer.py [--steps 20] [--warmup 3] [--out FILE]
"""
import argparse
import ctypes as C
import json
import math
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

from tools.bench_ddc import HBM_GBPS, roofline, timed   # noqa: E402
from tools.bench_persistence import gpu_name_power      # noqa: E402

FS = 61.44e6


def cost(n, in_b, T, M, D):
    return {"bytes": n * (in_b + 8.0 * M / D), "flops": n * (4.0 * T + 5.0 * M * math.log2(M)) / D, "samples": n}


def kernel_us(fn, steps, nat, pat="chan_kernel"):
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
    tot = sum(e.device_time_total for e in prof.events() if e.device_type == DeviceType.CUDA and pat in e.name)
    return tot / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    from sdr_iq_visualizer_b200 import _native as nat, ddc, features, spectral as sp, synth
    nat.require_device()
    name, power = gpu_name_power()
    peak = nat.fp32_peak_tflops(0)
    result = {"tool": "bench_channelizer", "gpu": name, "power_limit": power, "fp32_peak_tflops": round(peak, 2),
              "hbm_GBps": HBM_GBPS, "steps": args.steps, "warmup": args.warmup,
              "cost_model": "bytes/sample = in_B + 8M/D; flops/sample = (4T + 5 M log2 M)/D"}
    L1 = 61_440_000
    x1 = synth.tiled_ci16(L1, seed=2)
    d_x1 = nat.DeviceArray.from_host(x1)
    L2 = 1 << 28
    x2 = (synth.tiled_ci16(L2, seed=5).astype(np.float32) * np.float32(2.0 ** -10)).view(np.complex64)
    d_x2 = nat.DeviceArray.from_host(x2)
    del x2
    shapes = {"CH1": (d_x1, L1, sp.FMT_CI16, 2.0 ** -15, 64, 32), "CH2": (d_x2, L2, sp.FMT_CF32, 1.0, 1024, 512),
              "CH3": (d_x2, L2, sp.FMT_CF32, 1.0, 1024, 1024)}
    N, hop = 256, 128
    pl = sp.SpectralPlan(N, hop, "hann", sp.FMT_CF32)
    st = pl.stream
    chans, outs, legs = {}, {}, {}
    for k, (d_x, L, fmt, scale, M, D) in shapes.items():
        ch = ddc.Channelizer(FS, M, D, in_fmt=fmt, in_scale=scale)
        chans[k] = ch
        outs[k] = nat.DeviceArray((M, ch.out_count(L)), np.complex64)
        legs[k] = (lambda ch=ch, d_x=d_x, o=outs[k]: ch.exec(d_x, out=o, stream=st))
    # baseline: the same 64 channels as 64 K9 calls
    c1 = chans["CH1"]
    ddcs = [ddc.DdcPlan(FS, (j - 32) * FS / 64, 32, taps=c1.taps, in_fmt=sp.FMT_CI16, in_scale=2.0 ** -15)
            for j in range(64)]
    n1 = c1.out_count(L1)
    y1 = outs["CH1"]

    def baseline():
        for j, dd in enumerate(ddcs):
            dd.exec(d_x1, out=nat.DeviceView(y1.ptr + 8 * n1 * j, (n1,), np.complex64), stream=st)
    legs["CH1_64_ddc_calls"] = baseline
    # chain: channelizer + per-channel Welch / max-hold + finalize + 64 measurements (device-resident)
    we = nat.DeviceArray((64, N), np.float64)
    mh = nat.DeviceArray((64, N), np.float32)
    pxx, pdb = nat.DeviceArray((64 * N,), np.float64), nat.DeviceArray((64 * N,), np.float64)
    fq = features.FeatureQueue(batch=64, stream=st)
    Fr = pl.frame_count(n1)

    def chain():
        legs["CH1"]()
        pl.stft(nat.DeviceView(y1.ptr, (64 * n1,), np.complex64), n_streams=64, stream_stride=n1, n_samples=n1,
                welch=we, maxhold=mh, stream=st)
        pl.welch_finalize(nat.DeviceView(we.ptr, (64 * N,), np.float64), Fr, FS / 32, pxx=pxx, pdb=pdb, n_streams=64,
                          stream=st)
        fq.enqueue(nat.DeviceView(pdb.ptr + 8 * (N // 4), (64, N // 2), np.float64), N // 2, stride=N)
    legs["CH1_chain"] = chain
    order = ["CH1", "CH1_64_ddc_calls", "CH1_chain", "CH2", "CH3"]
    res = timed({k: legs[k] for k in order}, args.steps, args.warmup, nat, st)
    for k, (ms, rounds) in res.items():
        result[k + "_ms"] = ms
        result[k + "_ms_rounds"] = rounds
    result["CH1_speedup_vs_64_ddc_calls"] = round(res["CH1_64_ddc_calls"][0] / res["CH1"][0], 2)
    result["CH1_chain_frames_per_channel"] = Fr
    for k, (d_x, L, fmt, scale, M, D) in shapes.items():
        ch = chans[k]
        c = cost(L, 4 if fmt == sp.FMT_CI16 else 8, ch.n_taps, M, D)
        us = kernel_us(legs[k], 3, nat)
        r = roofline(c, us, peak)
        r.update({"samples": L, "fmt": "ci16" if fmt else "cf32", "channels": M, "decim": D, "taps": ch.n_taps,
                  "Gsamples_per_s_kernel": round(L / us / 1e3, 2),
                  "Gsamples_per_s_events": round(L / res[k][0] / 1e6, 2)})
        result[k] = r
    # one-shot host-memory CH1 call against the copy ceiling of the same bytes
    xin = nat.pinned_empty(x1.shape, x1.dtype)
    xin[:] = x1
    yo = nat.pinned_empty((64, n1), np.complex64)
    c1.exec(xin, out=yo)
    t0 = time.perf_counter()
    c1.exec(xin, out=yo)
    wall = time.perf_counter() - t0
    sec = C.c_double()
    nat.check(nat.lib().spx_copy_ceiling(0, xin.ctypes.data, xin.nbytes, yo.ctypes.data, yo.nbytes, 16 << 20, 5,
                                         C.byref(sec)))
    result["host_CH1"] = {"wall_ms": round(wall * 1e3, 2), "h2d_bytes": c1.last_h2d_bytes, "d2h_bytes": c1.last_d2h_bytes,
                          "copy_ceiling_ms": round(sec.value * 1e3, 2), "copy_ceiling_of": "input bytes up, output bytes down",
                          "frac_of_copy_ceiling": round(sec.value / wall, 3)}
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
