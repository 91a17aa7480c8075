"""Cost of the persistence spectrum (SpectralPlan.stft(persistence=...)) on one GPU; prints one JSON line.

Two shapes, each with three device-resident legs timed with CUDA events on the plan's stream (after warm-up):
  (a) uint8 rows + Welch + max-hold (what the pipeline computes today);
  (b) (a) + persistence counted from the caller's rows;
  (c) persistence + Welch + max-hold without rows (plan-owned row buffer, in batches).
Config-2 shape: 61.44 M ci16 samples, N = 4096 Hann, hop 1024, vmin 20, vmax 130.
Config-5 shape: 2^28 cf32 samples, N = 65536 Hann, hop 32768.

Also: the histogram kernel alone, from torch.profiler records of leg (b) in a separate run (bins/s and the fraction of
the shared-memory atomic lane rate in profiles/r02_atom_mix_micro.jsonl), and one-shot host-memory calls with and
without rows (wall time, d2h_bytes).  The card's name and power limit are read in the same run.

    python tools/bench_persistence.py [--steps 20] [--warmup 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def gpu_name_power():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        name, power = (v.strip() for v in out[0].split(","))
        return name, power
    except Exception as e:   # the numbers below are still device measurements; say that the card was not identified
        return f"unknown ({e})", "unknown"


def atom_rates():
    """ATOMS lane-operation rates of tools/micro/atom_mix.cu (round 2): distinct addresses per warp (dist 0) and the
    conflicting case (dist 1), G lane-ops/s on the whole GPU."""
    rates = {}
    with open(os.path.join(ROOT, "profiles", "r02_atom_mix_micro.jsonl")) as fh:
        for line in fh:
            r = json.loads(line)
            if r.get("mode") == "smem_atoms":
                rates[int(r["dist"])] = float(r["Gops_per_s"])
    return rates


def shape_inputs(name, nat, sp):
    from sdr_iq_visualizer_b200 import synth
    if name == "c2":
        n, hop, fmt, L, vmin, vmax = 4096, 1024, sp.FMT_CI16, 61_440_000, 20.0, 130.0
        x = synth.tiled_ci16(L, seed=2)
    else:
        n, hop, fmt, L, vmin, vmax = 65536, 32768, sp.FMT_CF32, 1 << 28, -40.0, 90.0
        x = (synth.tiled_ci16(L, seed=5).astype(np.float32) * np.float32(2.0 ** -10)).view(np.complex64)
    return n, hop, fmt, L, vmin, vmax, nat.DeviceArray.from_host(x), x


def time_legs(name, args, nat, sp):
    n, hop, fmt, L, vmin, vmax, d_x, x = shape_inputs(name, nat, sp)
    pl = sp.SpectralPlan(n, hop, "hann", fmt)
    F = pl.frame_count(L)
    d_wf = nat.DeviceArray((F, n), np.uint8)
    d_we = nat.DeviceArray((1, n), np.float64)
    d_mh = nat.DeviceArray((1, n), np.float32)
    d_pc = nat.DeviceArray((1, 256, n), np.uint32)
    legs = {
        "a_rows_welch_maxhold": dict(wf_rows=d_wf, welch=d_we, maxhold=d_mh),
        "b_rows_plus_persistence": dict(wf_rows=d_wf, welch=d_we, maxhold=d_mh, persistence=d_pc),
        "c_persistence_no_rows": dict(welch=d_we, maxhold=d_mh, persistence=d_pc),
    }
    st = pl.stream
    out = {"nfft": n, "hop": hop, "fmt": "ci16" if fmt else "cf32", "samples": L, "frames": F, "bins": F * n}
    # legs alternate round by round, so that drift of the shared host / card spreads over all three
    ms = {k: [] for k in legs}
    for k, kw in legs.items():
        for _ in range(args.warmup):
            pl.stft(d_x, vmin=vmin, vmax=vmax, **kw)
    pl.sync()
    rounds = 2
    per_round = max(1, args.steps // rounds)
    for _ in range(rounds):
        for k, kw in legs.items():
            t = nat.DeviceTimer(0, st)
            t.start()
            for _ in range(per_round):
                pl.stft(d_x, vmin=vmin, vmax=vmax, **kw)
            t.stop()
            ms[k].append(t.elapsed_ms() / per_round)
            t.close()
    for k in legs:
        out[k + "_ms"] = round(float(np.mean(ms[k])), 4)
        out[k + "_ms_rounds"] = [round(v, 4) for v in ms[k]]
    out["b_minus_a_ms"] = round(out["b_rows_plus_persistence_ms"] - out["a_rows_welch_maxhold_ms"], 4)
    out["c_minus_a_ms"] = round(out["c_persistence_no_rows_ms"] - out["a_rows_welch_maxhold_ms"], 4)
    # legs (b) and (c) compute the same counts (the plan's streams do not block the copy's stream: sync first)
    pl.stft(d_x, vmin=vmin, vmax=vmax, **legs["b_rows_plus_persistence"])
    pl.sync()
    c_b = d_pc.to_host()
    pl.stft(d_x, vmin=vmin, vmax=vmax, **legs["c_persistence_no_rows"])
    pl.sync()
    c_c = d_pc.to_host()
    out["counts_b_equal_c"] = bool(np.array_equal(c_b, c_c))
    out["column_sums_equal_F"] = bool((c_b.sum(axis=1) == F).all())
    return out, pl, d_x, x, legs, vmin, vmax


def profile_hist(pl, d_x, kw, vmin, vmax, steps, nat):
    """Per-kernel device time of leg (b) from torch.profiler records (a run of its own)."""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            pl.stft(d_x, vmin=vmin, vmax=vmax, **kw)
        nat.device_sync(0)
    tot = {}
    for e in prof.events():
        if e.device_type == DeviceType.CUDA and "kernel" in e.name:
            key = "persist_kernel" if "persist_kernel" in e.name else e.name.split("(")[0][:60]
            t, c = tot.get(key, (0.0, 0))
            tot[key] = (t + e.device_time_total, c + 1)     # microseconds
    return {k: {"us_per_call": round(t / c, 2), "calls": c} for k, (t, c) in tot.items()}


def host_calls(name, nat, sp, x):
    n, hop, fmt = (4096, 1024, sp.FMT_CI16) if name == "c2" else (65536, 32768, sp.FMT_CF32)
    vmin, vmax = (20.0, 130.0) if name == "c2" else (-40.0, 90.0)
    pl = sp.SpectralPlan(n, hop, "hann", fmt)
    xin = nat.pinned_empty(x.shape, x.dtype)
    xin[:] = x
    F = pl.frame_count(x.size // 2 if fmt else x.size)
    rows = nat.pinned_empty((F, n), np.uint8)
    res = {}
    for label, kw in (("rows", dict(wf_rows=rows)), ("no_rows", {})):
        pl.stft(xin, persistence=True, welch=True, maxhold=True, vmin=vmin, vmax=vmax, **kw)   # warm-up
        t0 = time.perf_counter()
        r = pl.stft(xin, persistence=True, welch=True, maxhold=True, vmin=vmin, vmax=vmax, **kw)
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
    rates = atom_rates()
    result = {"tool": "bench_persistence", "gpu": name, "power_limit": power, "steps": args.steps, "warmup": args.warmup}
    for shape in ("c2", "c5"):
        out, pl, d_x, x, legs, vmin, vmax = time_legs(shape, args, nat, sp)
        prof = profile_hist(pl, d_x, legs["b_rows_plus_persistence"], vmin, vmax, 3, nat)
        ph = prof.get("persist_kernel")
        if ph:
            bins_per_s = out["bins"] / (ph["us_per_call"] * 1e-6)
            out["persist_kernel_us"] = ph["us_per_call"]
            out["persist_kernel_Gbins_per_s"] = round(bins_per_s / 1e9, 1)
            out["persist_frac_of_atoms_rate_distinct"] = round(bins_per_s / (rates[0] * 1e9), 3)
            out["persist_frac_of_atoms_rate_conflicting"] = round(bins_per_s / (rates[1] * 1e9), 3)
        out["kernels_leg_b"] = prof
        pl.close()
        d_x.free()
        out["host_one_shot"] = host_calls(shape, nat, sp, x)
        result[shape] = out
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
