"""Cost of the pooled spectrogram (SpectralPlan.stft(pool=...)) on one GPU; prints one JSON line.

Two shapes (those of tools/bench_persistence.py), each with device-resident legs timed with CUDA events on the plan's
stream after warm-up, alternating round by round:
  (a) uint8 rows + Welch + max-hold (what the pipeline computes today);
  (b) pooled mean + Welch + max-hold, no rows (plan-owned float row buffer, in batches);
  (c) pooled mean from the caller's float dB rows + Welch + max-hold;
  (b_max) leg (b) with the max detector.
Config-2 shape: 61.44 M ci16 samples, N = 4096 Hann, hop 1024, K x B = 600 x 4 -> 100 x 1024 (last row 597 frames).
Config-5 shape: 2^28 cf32 samples, N = 65536 Hann, hop 32768, K x B = 8 x 64 -> 1024 x 1024 (last row 7 frames).

Also: pool_kernel alone from torch.profiler records of leg (c) in a separate run (G bins/s, GB/s of dB rows read and
the fraction of 6539.9 GB/s, the HBM figure of DESIGN.md section 4), leg (b) for SPX_POOL_ROWS_BYTES of 32 / 64 / 128 /
256 MiB, and one-shot host-memory calls (pooled without rows vs uint8 rows: wall time, d2h_bytes).  The card's name and
power limit are read in the same run.

    python tools/bench_pooled.py [--steps 20] [--warmup 3] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

from tools.bench_persistence import gpu_name_power, shape_inputs   # noqa: E402

HBM_GBPS = 6539.9
POOL = {"c2": (600, 4), "c5": (8, 64)}
SWEEP_MIB = (32, 64, 128, 256)


def time_legs(pl, d_x, legs, vmin, vmax, steps, warmup, nat):
    st = pl.stream
    for kw in legs.values():
        for _ in range(warmup):
            pl.stft(d_x, vmin=vmin, vmax=vmax, **kw)
    pl.sync()
    ms = {k: [] for k in legs}
    rounds = 2
    per_round = max(1, steps // rounds)
    for _ in range(rounds):
        for k, kw in legs.items():
            t = nat.DeviceTimer(0, st)
            t.start()
            for _ in range(per_round):
                pl.stft(d_x, vmin=vmin, vmax=vmax, **kw)
            t.stop()
            ms[k].append(t.elapsed_ms() / per_round)
            t.close()
    return {k: (round(float(np.mean(v)), 4), [round(x, 4) for x in v]) for k, v in ms.items()}


def profile_pool(pl, d_x, kw, vmin, vmax, steps, nat):
    """Per-kernel device time of one leg from torch.profiler records (a run of its own)."""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    pl.stft(d_x, vmin=vmin, vmax=vmax, **kw)
    nat.device_sync(0)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            pl.stft(d_x, vmin=vmin, vmax=vmax, **kw)
        nat.device_sync(0)
    tot = {}
    for e in prof.events():
        if e.device_type == DeviceType.CUDA and "kernel" in e.name:
            key = "pool_kernel" if "pool_kernel<" in e.name else e.name.split("(")[0][:60]
            t, c = tot.get(key, (0.0, 0))
            tot[key] = (t + e.device_time_total, c + 1)     # microseconds
    return {k: {"us_per_step": round(t / steps, 2), "calls_per_step": c / steps} for k, (t, c) in tot.items()}


def run_shape(name, args, nat, sp):
    n, hop, fmt, L, vmin, vmax, d_x, x = shape_inputs(name, nat, sp)
    K, B = POOL[name]
    pl = sp.SpectralPlan(n, hop, "hann", fmt)
    F = pl.frame_count(L)
    G, C = -(-F // K), n // B
    d_wf = nat.DeviceArray((F, n), np.uint8)
    d_db = nat.DeviceArray((F, n), np.float32)
    d_we = nat.DeviceArray((1, n), np.float64)
    d_mh = nat.DeviceArray((1, n), np.float32)
    d_acc = nat.DeviceArray((1, G, C), np.float64)
    acc_kw = dict(pool_acc=d_acc, welch=d_we, maxhold=d_mh)
    legs = {
        "a_rows_welch_maxhold": dict(wf_rows=d_wf, welch=d_we, maxhold=d_mh),
        "b_pooled_mean_no_rows": dict(pool=(K, B, "mean"), **acc_kw),
        "c_pooled_mean_from_db_rows": dict(pool=(K, B, "mean"), db_rows=d_db, **acc_kw),
        "b_max_pooled_max_no_rows": dict(pool=(K, B, "max"), **acc_kw),
    }
    out = {"nfft": n, "hop": hop, "fmt": "ci16" if fmt else "cf32", "samples": L, "frames": F, "bins": F * n,
           "frames_per_row": K, "bins_per_col": B, "image": [G, C], "last_row_frames": F - (G - 1) * K}
    res = time_legs(pl, d_x, legs, vmin, vmax, args.steps, args.warmup, nat)
    for k, (m, rounds) in res.items():
        out[k + "_ms"] = m
        out[k + "_ms_rounds"] = rounds
    out["b_minus_a_ms"] = round(out["b_pooled_mean_no_rows_ms"] - out["a_rows_welch_maxhold_ms"], 4)
    # legs (b) and (c) pool the same frames (max: bit for bit)
    accs = {}
    for k in ("b_max_pooled_max_no_rows", "c_pooled_mean_from_db_rows", "b_pooled_mean_no_rows"):
        pl.stft(d_x, vmin=vmin, vmax=vmax, **legs[k])
        pl.sync()
        accs[k] = d_acc.to_host()
    b, c = accs["b_pooled_mean_no_rows"], accs["c_pooled_mean_from_db_rows"]
    out["mean_b_vs_c_max_rel"] = float(np.max(np.abs(b - c) / np.abs(c)))
    pl.stft(d_x, vmin=vmin, vmax=vmax, pool=(K, B, "max"), pool_acc=d_acc, db_rows=d_db)
    pl.sync()
    out["max_b_equal_from_rows"] = bool(np.array_equal(accs["b_max_pooled_max_no_rows"], d_acc.to_host()))
    prof = profile_pool(pl, d_x, legs["c_pooled_mean_from_db_rows"], vmin, vmax, 3, nat)
    pk = prof.get("pool_kernel")
    if pk:
        s = pk["us_per_step"] * 1e-6
        out["pool_kernel_us"] = pk["us_per_step"]
        out["pool_kernel_Gbins_per_s"] = round(F * n / s / 1e9, 1)
        out["pool_kernel_GB_per_s"] = round(F * n * 4 / s / 1e9, 1)
        out["pool_kernel_frac_of_hbm"] = round(F * n * 4 / s / 1e9 / HBM_GBPS, 3)
    out["kernels_leg_c"] = prof
    out["kernels_leg_b"] = profile_pool(pl, d_x, legs["b_pooled_mean_no_rows"], vmin, vmax, 3, nat)
    pl.close()
    for buf in (d_wf, d_db):
        buf.free()
    # SPX_POOL_ROWS_BYTES sweep of leg (b)
    sweep = {}
    for mib in SWEEP_MIB:
        os.environ["SPX_POOL_ROWS_BYTES"] = str(mib << 20)
        p2 = sp.SpectralPlan(n, hop, "hann", fmt)
        del os.environ["SPX_POOL_ROWS_BYTES"]
        r = time_legs(p2, d_x, {"b": legs["b_pooled_mean_no_rows"]}, vmin, vmax, args.steps, args.warmup, nat)["b"]
        sweep[f"{mib}MiB"] = {"ms": r[0], "ms_rounds": r[1]}
        p2.close()
    out["rows_bytes_sweep_leg_b"] = sweep
    d_x.free()
    out["host_one_shot"] = host_calls(n, hop, fmt, vmin, vmax, K, B, x, nat, sp)
    return out


def host_calls(n, hop, fmt, vmin, vmax, K, B, x, nat, sp):
    pl = sp.SpectralPlan(n, hop, "hann", fmt)
    xin = nat.pinned_empty(x.shape, x.dtype)
    xin[:] = x
    F = pl.frame_count(x.size // 2 if fmt else x.size)
    rows = nat.pinned_empty((F, n), np.uint8)
    res = {}
    for label, kw in (("u8_rows", dict(wf_rows=rows)), ("pooled_no_rows", dict(pool=(K, B, "mean")))):
        pl.stft(xin, welch=True, maxhold=True, vmin=vmin, vmax=vmax, **kw)   # warm-up
        t0 = time.perf_counter()
        r = pl.stft(xin, welch=True, maxhold=True, vmin=vmin, vmax=vmax, **kw)
        res[label] = {"wall_ms": round((time.perf_counter() - t0) * 1e3, 2), "d2h_bytes": r.d2h_bytes,
                      "h2d_bytes": r.h2d_bytes}
    pl.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    from sdr_iq_visualizer_b200 import _native as nat, spectral as sp
    nat.require_device()
    name, power = gpu_name_power()
    result = {"tool": "bench_pooled", "gpu": name, "power_limit": power, "steps": args.steps, "warmup": args.warmup}
    for shape in ("c2", "c5"):
        result[shape] = run_shape(shape, args, nat, sp)
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
