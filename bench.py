#!/usr/bin/env python3
"""bench.py -- IQ Msamples/s through windowed FFT -> PSD -> waterfall on B200 (BASELINE.json metric).

Workload (N = 1 GPU and per rank for N > 1): BASELINE config 2 -- one second of a 61.44 MS/s int16
IQ stream (61 440 000 samples), 4096-point Hann FFT with 75 % overlap (59 997 frames), producing the
uint8 waterfall rows, the Welch sum, the max-hold and the classifier features of the Welch PSD.
One "step" = one pass of that path over that batch.

  value   : whole-job Msamples/s with the input already resident in HBM (device buffers).
  e2e     : the same step through the pinned ingest ring of the C ABI (spx_ring_*: config 2 IS the ring-buffer
            stream): per 2^22-sample slot H2D -> fused STFT -> D2H of rows / Welch / max-hold / features, all inside
            the timed region; the producer writes in place (the slots are the DMA target).  The one-shot host-buffer
            call (spx_stft_exec, SPX_MEM_HOST) and the box's raw concurrent-copy ceiling are measured beside it.
  roofline: this shape transforms every sample four times, so FP32 binds (SURVEY.md 8(d)): achieved nominal TFLOP/s
            (5 N log2 N + 20 N per frame) over the CUDA-event duration of the fused STFT kernel vs the FP32 FMA peak
            measured in the same run; the HBM fraction (8 B/sample) and the HBM-bound headline shape are alongside.
  sustained: the same device-resident step looped for >= 2 s with NVML clock / power samples.
  sharded : the configs that shard (SURVEY.md 8(e)), strong scaling over the ranks of this run, parity-checked in
            the same run: config 5 (2^30-sample capture, 65536-pt, fused peer reduction; rows sharded or gathered
            to rank 0, NCCL all-reduce + gather as the baseline) and config 4 (64 streams x 2^24).
  cpu_baseline: the float64 numpy oracle (a port: the reference has no windowed/overlapped path)
            on a bounded slice, single core, timed on this box.

`--steps K` is the number of timed steps of each config-2 leg (device-resident, ring, one-shot call); the sustained
leg runs for >= 2 s instead (`--no-sustained` skips it).
`--dump-outputs DIR` writes what the device-resident step handed back in its last timed step as DIR/<name>.npy
(float32 / float64; the inputs are seeded, so two builds can be compared output for output).
`--impl reference` times the CPU oracle port with all host cores (multiprocessing over frame
blocks) on the same config and prints the same line with "impl": "reference".
Multi-GPU: config 2 is one ordered stream, so for `value` / `e2e` the ranks are independent replicas (one stream per
GPU, no data-path collective); the `sharded` block carries the configs with a real exchange step.
torch.distributed is the plumbing (barriers, IPC handles, tiny tensors).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (which may be read-only)

NFFT, HOP, FS, FC = 4096, 1024, 61.44e6, 2.4e9
L_STEP = 61_440_000
VMIN, VMAX = 20.0, 130.0
DUMP_ROWS = 2048                                  # seeded sample of the 59 997 waterfall rows: 32 MiB as float32
BYTES_PER_SAMPLE = 4 + (NFFT // HOP) * 1          # int16 IQ in + four u8 rows touched per sample
FLOP_PER_SAMPLE = (NFFT // HOP) * (5 * 12 + 20)   # SURVEY.md 8(d)
METRIC = "IQ Msamples/s through windowed FFT->PSD->waterfall"


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return json.load(fh), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


def synth_ci16(n, seed):
    """QPSK + CW tone + AWGN, 12-bit range int16 (SURVEY.md 8(d)); a 4 Mi-sample block tiled to n."""
    from sdr_iq_visualizer_b200 import synth
    return synth.tiled_ci16(n, seed)


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md clocks line):
    NVML in a thread every 5 ms; nvidia-smi --query-gpu as the fallback."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.sm, self.mask, self.max_mhz, self.power = [], 0, None, []
        self.pcie = []            # (link generation, width) seen while sampling: a downtrained link explains a low copy ceiling
        self.pcie_max = None
        self._stop = threading.Event()
        self._thr = None
        self._nvml = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = self.idx
            if vis:
                try:
                    phys = int(vis.split(",")[self.idx])
                except Exception:
                    phys = self.idx
            h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            try:
                self.pcie_max = (int(pynvml.nvmlDeviceGetMaxPcieLinkGeneration(h)), int(pynvml.nvmlDeviceGetMaxPcieLinkWidth(h)))
            except Exception:
                self.pcie_max = None
            self._nvml = (pynvml, h)
        except Exception:
            self._nvml = None
        self._thr = threading.Thread(target=self._run, daemon=True)
        self._thr.start()

    def _sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        out = subprocess.run(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=10).stdout.strip().split(",")
        self.sm.append(float(out[0])); self.max_mhz = float(out[1])
        for bit, v in zip((0x8, 0x40, 0x20, 0x4), out[2:6]):
            if v.strip().lower().startswith("active"):
                self.mask |= bit

    def _run(self):
        while not self._stop.is_set():
            try:
                if self._nvml:
                    nv, h = self._nvml
                    self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                    self.mask |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
                    self.power.append(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)
                    if len(self.sm) % 8 == 1:
                        self.pcie.append((int(nv.nvmlDeviceGetCurrPcieLinkGeneration(h)), int(nv.nvmlDeviceGetCurrPcieLinkWidth(h))))
                else:
                    self._sample_smi()
            except Exception:
                pass
            self._stop.wait(0.005)

    def stop(self):
        self._stop.set()
        if self._thr:
            self._thr.join(timeout=15)
        reasons = sorted(name for bit, name in self.REASONS.items() if self.mask & bit)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": reasons, "samples": len(self.sm), "source": "nvml" if self._nvml else "nvidia-smi",
                "power_w_max": round(max(self.power), 1) if self.power else None,
                "sm_mhz_min": float(min(self.sm)) if self.sm else None,
                "pcie_link": None if not self.pcie else {"gen_min": min(g for g, _ in self.pcie), "width_min": min(w for _, w in self.pcie),
                                                         "gen_max": self.pcie_max[0] if self.pcie_max else None,
                                                         "width_max": self.pcie_max[1] if self.pcie_max else None}}


def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local, dist


def barrier_max(dist, local, seconds):
    if dist is None:
        return seconds
    import torch
    t = torch.tensor([seconds], dtype=torch.float64, device=f"cuda:{local}")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def cpu_baseline_single(sample_log2=26):
    from oracle import pipeline_ref
    x = synth_ci16(1 << sample_log2, seed=2)
    best = 1e30
    for _ in range(2):
        t0 = time.perf_counter()
        pipeline_ref.c2_step(x, NFFT, HOP, "hann", FS, FC, VMIN, VMAX)
        best = min(best, time.perf_counter() - t0)
    return {"value": round((1 << sample_log2) / best / 1e6, 3), "unit": "Msamples/s", "cores": 1, "kind": "port",
            "sample": f"2^{sample_log2} int16 IQ samples of the config-2 step (float64 numpy oracle, best of 2), numpy {np.__version__}, "
                      f"{os.cpu_count()} host cores present"}


def run_reference(args):
    """CPU arm: the oracle port on all host cores, same config/metric."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    from oracle import pipeline_ref
    cores = os.cpu_count() or 1
    n = 1 << 23
    x = synth_ci16(n, seed=2)
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        for _ in range(args.warmup):
            pipeline_ref.c2_step_parallel(x, pool, cores, NFFT, HOP)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            acc, mx, F = pipeline_ref.c2_step_parallel(x, pool, cores, NFFT, HOP)
        dt = time.perf_counter() - t0
    v = round(n * args.steps / dt / 1e6, 3)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "Msamples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt / args.steps * 1e3, 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "config2: int16 IQ, 4096-pt Hann FFT, 75% overlap, u8 rows + Welch + max-hold (CPU oracle port)",
                       "nfft": NFFT, "hop": HOP, "samples_per_step": n},
            "cpu_baseline": {"value": v, "unit": "Msamples/s", "cores": cores, "kind": "port",
                             "sample": f"2^23-sample slice of the config-2 second per step, frame blocks over {cores} processes"},
            "e2e": {"value": v, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def numa_info(nat, local):
    """Where this rank's CPU threads and its GPU sit (the pinned buffers are first-touched after the affinity call)."""
    info = {}
    try:
        import pynvml
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[local]) if vis else local
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as fh:
            info["gpu_numa_node"] = int(fh.read().strip())
    except Exception:
        info["gpu_numa_node"] = None
    try:
        cpus = sorted(os.sched_getaffinity(0))
        info["cpu_affinity"] = f"{len(cpus)} cpus [{cpus[0]}..{cpus[-1]}]"
        nodes = set()
        for nd in os.listdir("/sys/devices/system/node"):
            if nd.startswith("node"):
                with open(f"/sys/devices/system/node/{nd}/cpulist") as fh:
                    rng = fh.read().strip()
                members = set()
                for part in rng.split(","):
                    if part:
                        a, _, b = part.partition("-")
                        members.update(range(int(a), int(b or a) + 1))
                if members & set(cpus):
                    nodes.add(int(nd[4:]))
        info["cpu_numa_nodes"] = sorted(nodes)
    except Exception:
        pass
    return info


def traffic_record(kernel_name):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture; refused (None) unless the capture
    names the kernel this run launched."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            t = json.load(fh)
        if t.get("kernel") != kernel_name:
            return None, f"profiles/traffic.json is for {t.get('kernel')!r}, this run launched {kernel_name!r}"
        return t.get("c2_stft_kernel_dram_bytes_per_launch"), f"{t.get('source')} (ncu --set full, commit {t.get('git_sha')})"
    except Exception as exc:
        return None, f"no traffic record: {exc}"


def dump_outputs(out_dir, wf_rows, welch_acc, maxhold, pxx, pdb, feat):
    """The outputs of one device-resident step as DIR/<name>.npy: a fixed, seeded sample of the uint8 waterfall rows
    (values as float32, row indices beside them), the Welch sum, max-hold, PSD, PSD in dB and the classifier features
    (the numeric fields of spx_features in declaration order)."""
    os.makedirs(out_dir, exist_ok=True)
    rows = wf_rows.to_host()
    idx = np.sort(np.random.default_rng(0).choice(rows.shape[0], min(DUMP_ROWS, rows.shape[0]), replace=False))
    out = {"wf_rows_sample": rows[idx].astype(np.float32), "wf_rows_sample_index": idx.astype(np.float64),
           "welch_acc": welch_acc.to_host().reshape(-1), "maxhold": maxhold.to_host().reshape(-1),
           "pxx": pxx.to_host(), "pxx_db": pdb.to_host(),
           "features": np.array([float(v) for k, v in feat.items() if k != "peaks"], np.float64)}
    for name, arr in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of each config-2 leg")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--variant", type=int, default=int(os.environ.get("SPX_VARIANT", "-1")))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sharded", action="store_true", help="skip the config-4 / config-5 strong-scaling block")
    ap.add_argument("--no-sustained", action="store_true")
    ap.add_argument("--no-views", action="store_true", help="skip the config-3 block (I/Q histogram, frame stats)")
    ap.add_argument("--sharded-log2", type=int, default=30, help="config-5 capture length (2^30 is BASELINE's size)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
        return

    rank, world, local, dist = dist_setup(args.gpus)
    try:  # keep this rank's pinned buffers and threads on the NUMA node its GPU hangs off
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[local]) if vis else local
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(phys))
    except Exception:
        pass
    from sdr_iq_visualizer_b200 import _native as nat
    from sdr_iq_visualizer_b200 import features, ring as ringmod, spectral as sp
    nat.require_device()
    dev = local
    peaks, peak_src = measured_peaks()
    numa = numa_info(nat, local)

    host_in = nat.pinned_empty(2 * L_STEP, np.int16)
    host_in[:] = synth_ci16(L_STEP, seed=2 + rank)
    variant = args.variant if args.variant >= 0 else sp.DEFAULT_VARIANT.get(NFFT, 0)
    pl = sp.SpectralPlan(NFFT, HOP, "hann", sp.FMT_CI16, device=dev, variant=variant)
    F = pl.frame_count(L_STEP)

    # ---------------- device-resident leg: every launch of a step goes to the plan's compute stream
    d_in = nat.DeviceArray.from_host(host_in, dev)
    d_wf = nat.DeviceArray((F, NFFT), np.uint8, dev)
    # two sets of Welch-block buffers: the classifier measurements of block k run on a side stream next to the STFT of
    # block k+1 (they are one latency-bound CTA; serialised behind the STFT kernel they were 8 % of the step)
    d_we = [nat.DeviceArray((1, NFFT), np.float64, dev) for _ in range(2)]
    d_mh = [nat.DeviceArray((1, NFFT), np.float32, dev) for _ in range(2)]
    d_pxx = [nat.DeviceArray((NFFT,), np.float64, dev) for _ in range(2)]
    d_pdb = [nat.DeviceArray((NFFT,), np.float64, dev) for _ in range(2)]
    d_we_flat = [nat.DeviceView(w.ptr, (NFFT,), np.float64, dev) for w in d_we]
    st = pl.stream
    side = [nat.SideStream(dev), nat.SideStream(dev)]     # one per buffer set: STFT k waits for the side work of step k-2 only
    total_timer = nat.DeviceTimer(dev, st)
    kernel_timers = [nat.DeviceTimer(dev, st) for _ in range(args.steps)]
    step_no = [0]

    def device_step(ktimer):
        # fused STFT launch on the plan's stream (bracketed by its own CUDA events when timed); Welch finalize + classifier
        # features of this block on the side stream behind it.  Buffer set b is reused two steps later: its STFT waits for
        # the side-stream work of step k-2 through the join below.
        b = step_no[0] & 1
        step_no[0] += 1
        side[b].then(st)        # the side work of step k-2 (same buffer set) precedes this STFT; step k-1's runs next to it
        if ktimer is not None:
            ktimer.start()
        res = pl.stft(d_in, wf_rows=d_wf, welch=d_we[b], maxhold=d_mh[b], vmin=VMIN, vmax=VMAX)
        if ktimer is not None:
            ktimer.stop()
        side[b].after(st)
        pl.welch_finalize(d_we_flat[b], res.n_frames, FS, pxx=d_pxx[b], pdb=d_pdb[b], stream=side[b].handle)
        # kernel + asynchronous copy of the result struct to pinned memory (the host never waits inside a step; results
        # are read after the loop)
        return fq[b].enqueue(d_pdb[b], NFFT), b

    def join_side():
        side[0].then(st)        # the timed region on `st` ends after the last blocks' measurements
        side[1].then(st)

    fq = [features.FeatureQueue(1, dev, sd_.handle, slots=max(args.steps, args.warmup, 1)) for sd_ in side]
    for _ in range(args.warmup):
        device_step(None)
    join_side()
    sampler = ClockSampler(dev)
    if dist is not None:
        dist.barrier()
    nat.device_sync(dev)
    sampler.start()
    total_timer.start()
    for i in range(args.steps):
        last_slot = device_step(kernel_timers[i])
    join_side()
    total_timer.stop()
    dt_dev = total_timer.elapsed_ms() * 1e-3
    nat.device_sync(dev)
    feat = fq[last_slot[1]].results(last_slot[0])[0]
    kernel_ms = [t.elapsed_ms() for t in kernel_timers]
    if args.dump_outputs and rank == 0:     # before the sustained leg overwrites these buffers
        b = last_slot[1]
        dump_outputs(args.dump_outputs, d_wf, d_we[b], d_mh[b], d_pxx[b], d_pdb[b], feat)
    dt_dev = barrier_max(dist, local, dt_dev)

    # ---------------- sustained leg: the same step back to back for >= 2 s (a 13 ms burst cannot show a power / thermal
    # limit); its own clock / power samples
    sustained = None
    if not args.no_sustained:
        n_sus = int(min(20000, max(args.steps, 2.2 / max(dt_dev / args.steps, 1e-5))))
        sus_sampler = ClockSampler(dev)
        sus_timer = nat.DeviceTimer(dev, st)
        if dist is not None:
            dist.barrier()
        nat.device_sync(dev)
        sus_sampler.start()
        sus_timer.start()
        for _ in range(n_sus):
            device_step(None)
        join_side()
        sus_timer.stop()
        dt_sus = sus_timer.elapsed_ms() * 1e-3
        nat.device_sync(dev)
        sus_clocks = sus_sampler.stop()
        dt_sus = barrier_max(dist, local, dt_sus)
        sustained = {"steps": n_sus, "seconds": round(dt_sus, 3), "value": round(world * L_STEP * n_sus / dt_sus / 1e6, 1),
                     "unit": "Msamples/s", "ms_per_step": round(dt_sus / n_sus * 1e3, 4), "clocks": sus_clocks,
                     "vs_burst": round((L_STEP * n_sus / dt_sus) / (L_STEP * args.steps / dt_dev), 4)}

    # ---------------- end-to-end leg 1: the pinned ingest ring (config 2 is the ring-buffer stream).  Per slot:
    # H2D of 2^22 samples -> fused STFT (+ Welch finalize + classifier features) -> D2H of the slot's rows, Welch sum,
    # max-hold, PSD and feature struct.  In-place producer: the pinned slots are where the radio DMA would land, so the
    # timed loop commits them without rewriting their contents (filled once, untimed, below).
    SLOT = 1 << 22
    n_full, tail = divmod(L_STEP, SLOT)
    slot_sizes = [SLOT] * n_full + ([tail] if tail else [])
    RING_SLOTS = 6      # five in flight + the one the producer fills: with fewer the two upload streams cannot both stay busy
    rg = ringmod.StreamRing(pl, n_slots=RING_SLOTS, slot_samples=SLOT, wf_rows=True, welch=True, maxhold=True, vmin=VMIN, vmax=VMAX,
                            features=True, sample_rate=FS)
    e2e_steps = args.steps

    ring_state = {"pending": 0, "last": None}

    def ring_pass(fill, drain):
        """One step = one second of the stream through the ring (slots are collected RING_SLOTS - 1 commits behind).  The stream is
        continuous: consecutive steps keep the pipeline full, only the end of the timed region drains it."""
        pos = 0
        for n in slot_sizes:
            buf = rg.acquire()
            if fill:
                buf[: 2 * n] = host_in[2 * pos: 2 * (pos + n)]      # memcpy producer (warm-up / comparison only)
            rg.commit(n)
            pos += n
            ring_state["pending"] += 1
            if ring_state["pending"] >= RING_SLOTS - 1:
                ring_state["last"] = rg.collect(); rg.release(); ring_state["pending"] -= 1
        while drain and ring_state["pending"]:
            ring_state["last"] = rg.collect(); rg.release(); ring_state["pending"] -= 1
        return ring_state["last"]

    t0 = time.perf_counter()
    ring_pass(True, True)
    dt_fill = time.perf_counter() - t0          # same pass with a single-threaded numpy memcpy producer, for the record
    ring_pass(False, True)
    st0 = rg.stats()
    if dist is not None:
        dist.barrier()
    nat.device_sync(dev)
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        blk = ring_pass(False, i == e2e_steps - 1)
    nat.device_sync(dev)
    dt_ring_local = time.perf_counter() - t0
    st1 = rg.stats()
    dt_ring = barrier_max(dist, local, dt_ring_local)
    ring_h2d = (st1["h2d_bytes"] - st0["h2d_bytes"]) // e2e_steps
    ring_d2h = (st1["d2h_bytes"] - st0["d2h_bytes"]) // e2e_steps
    feat_ring = blk["features"]
    rg.close()

    # ---------------- end-to-end leg 2: the one-shot host-buffer call (spx_stft_exec with SPX_MEM_HOST)
    h_wf = nat.pinned_empty((F, NFFT), np.uint8)
    h_we = nat.pinned_empty((1, NFFT), np.float64)
    h_mh = nat.pinned_empty((1, NFFT), np.float32)
    call_steps = args.steps

    def e2e_step():
        r = pl.stft(host_in, wf_rows=h_wf, welch=h_we, maxhold=h_mh, vmin=VMIN, vmax=VMAX)
        _, pdb = pl.welch_finalize(h_we[0], r.n_frames, FS)
        return r, features.measure(pdb, device=dev)

    for _ in range(2):
        r, feat_h = e2e_step()
    if dist is not None:
        dist.barrier()
    nat.device_sync(dev)
    t0 = time.perf_counter()
    for _ in range(call_steps):
        r, feat_h = e2e_step()
    nat.device_sync(dev)
    dt_call = barrier_max(dist, local, time.perf_counter() - t0)
    clocks = sampler.stop()     # sampled through the device-resident leg and both end-to-end legs

    # ---------------- the box's raw copy ceiling for exactly these bytes: the same pinned buffers, H2D and D2H at once on
    # two streams in 16 MiB pieces, nothing else running; every rank copies at the same time (as in the e2e legs)
    ceil_s = None
    try:
        import ctypes as C
        sec = C.c_double()
        if dist is not None:
            dist.barrier()
        nat.check(nat.lib().spx_copy_ceiling(dev, host_in.ctypes.data, host_in.nbytes, h_wf.ctypes.data, h_wf.nbytes,
                                             16 << 20, 3, C.byref(sec)))
        ceil_s = barrier_max(dist, local, float(sec.value))
    except Exception as exc:   # reported, never fatal
        print(f"copy ceiling probe failed: {exc}", file=sys.stderr)

    # ---------------- sharded configs (strong scaling over the ranks of this run), parity-checked in the same run
    sharded = None
    if not args.no_sharded:
        # free what the config-2 legs held before the 8 GiB captures are allocated
        pl.close(); d_in.free(); d_wf.free()
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import bench_sharded as bs
        ctx = bs.Ctx(rank, world, local, dist, strict=False)   # a failed check is reported in the line (and on stderr), loudly, not by losing the line
        block = bs.synth_block()
        lg = args.sharded_log2
        sharded = {"scaling": "strong", "n_gpus": world, "unit": "Msamples/s",
                   "c5": {"workload": f"config5: 2^{lg} cf32 samples, 65536-pt Hann, 50% overlap, u8 rows + Welch + max-hold; "
                                      "frame blocks with (N - hop)-sample halos per rank",
                          "reduce_only": bs.run_c5(ctx, "fused", "sharded", lg, 5, 2, True, block),
                          "gather_to_rank0": bs.run_c5(ctx, "fused", "gather", lg, 5, 2, True, block),
                          "nccl_allreduce_gather": bs.run_c5(ctx, "nccl", "gather", lg, 3, 2, True, block, measure_kernel=False)},
                   "c4": dict(bs.run_c4(ctx, 24, 64, 5, 2, True, block),
                              workload="config4: 64 streams x 2^24 cf32, 2048-pt Hann, 50% overlap, per-stream Welch PSD + classifier "
                                       "features; contiguous blocks of streams per rank")}

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---------------- context for the roofline: measured FP32 peak, and the HBM-bound headline shape of north_star
    # (cf32 in, hop = N, f32 dB rows: 12 B/sample, 80 nominal flop/sample) timed the same way on 61 440 000 samples
    # (492 MB in + 246 MB out per launch: several times the 126 MB L2, so no explicit flush)
    p32 = nat.fp32_peak_tflops(dev)
    Lh = L_STEP
    plh = sp.SpectralPlan(NFFT, NFFT, "hann", sp.FMT_CF32, device=dev)
    rngh = np.random.default_rng(1)
    d_xh = nat.DeviceArray.from_host(rngh.standard_normal(2 * Lh).astype(np.float32).view(np.complex64), dev)
    d_dbh = nat.DeviceArray((Lh // NFFT, NFFT), np.float32, dev)
    _, ms_h = plh.time_stft(d_xh, warmup=3, iters=10, flush_l2=False, db_rows=d_dbh)
    ms_h = float(np.median(ms_h))
    headline = {"shape": "cf32 in, 4096-pt Hann, hop = N, f32 dB rows (12 B/sample), 61 440 000 samples per launch (738 MB of traffic, "
                         "larger than L2; no flush)",
                "kernel_ms": round(ms_h, 4), "Msamples_per_s": round(Lh / (ms_h * 1e-3) / 1e6, 1),
                "achieved_gbs": round(Lh * 12 / (ms_h * 1e-3) / 1e9, 1),
                "frac_of_hbm_peak": round(Lh * 12 / (ms_h * 1e-3) / 1e9 / peaks["hbm_gbs"], 4)}
    plh.close(); d_xh.free(); d_dbh.free()

    # ---------------- config 3 (time-domain views): 2^24 cf32 samples -> 256 x 256 I/Q histogram and per-frame mean / peak power;
    # device time per call (CUDA events on the calls' stream, 16 calls back to back over 8 rotating copies = 1 GiB, so the
    # input is cold), counts checked against np.histogram2d on a 2^20-sample prefix in the same run
    views = None
    if not args.no_views:
        from sdr_iq_visualizer_b200 import timedomain as td
        L3 = 1 << 24
        x3 = (0.7 * np.random.default_rng(3).standard_normal(2 * L3, dtype=np.float32)).view(np.complex64)
        copies = [nat.DeviceArray.from_host(x3, dev) for _ in range(8)]
        d_h = nat.DeviceArray((256, 256), np.uint32, dev, zero=True)
        d_mp = (nat.DeviceArray((L3 // 4096,), np.float32, dev), nat.DeviceArray((L3 // 4096,), np.float32, dev))
        ss = nat.SideStream(dev)
        tm = nat.DeviceTimer(dev, ss.handle)

        def per_call_us(fn):
            best = None
            for rep in range(3):
                tm.start()
                for k in range(16):
                    fn(copies[k % 8])
                tm.stop()
                us = tm.elapsed_ms() / 16 * 1e3
                best = us if best is None or (rep > 0 and us < best) else best
            return best
        us_h = per_call_us(lambda d: td.iq_hist2d(d, 4.0, 256, out=d_h, device=dev, stream=ss.handle))
        us_f = per_call_us(lambda d: td.frame_stats(d, 4096, 4096, device=dev, stream=ss.handle, out=d_mp))
        pre = nat.DeviceView(copies[0].ptr, (1 << 20,), np.complex64, dev)
        td.iq_hist2d(pre, 4.0, 256, out=d_h, device=dev, stream=ss.handle)
        ss.sync()
        want = np.histogram2d(x3[: 1 << 20].real.astype(np.float64), x3[: 1 << 20].imag.astype(np.float64), bins=256,
                              range=[[-4.0, 4.0], [-4.0, 4.0]])[0].astype(np.uint32)
        views = {"workload": "config3: 2^24 cf32 samples (sigma 0.7, R = 4), 256 x 256 I/Q histogram; 4096-sample frames mean / peak power",
                 "hist2d_us_per_call": round(us_h, 2), "hist2d_frac_of_hbm_peak": round(L3 * 8 / (us_h * 1e-6) / 1e9 / peaks["hbm_gbs"], 4),
                 "frame_stats_us_per_call": round(us_f, 2), "frame_stats_frac_of_hbm_peak": round(L3 * 8 / (us_f * 1e-6) / 1e9 / peaks["hbm_gbs"], 4),
                 "timing": "CUDA events on the calls' stream, 16 calls back to back over 8 rotating copies (1 GiB: input cold)",
                 "check": "ok: counts equal np.histogram2d on a 2^20-sample prefix" if np.array_equal(d_h.to_host(), want)
                          else "FAILED: counts differ from np.histogram2d"}
        if not views["check"].startswith("ok"):
            print("CONFIG-3 HISTOGRAM CHECK FAILED", file=sys.stderr, flush=True)
        for c in copies:
            c.free()
        d_h.free(); d_mp[0].free(); d_mp[1].free()

    k_ms = float(np.mean(kernel_ms))
    achieved_gbs = L_STEP * BYTES_PER_SAMPLE / (k_ms * 1e-3) / 1e9
    achieved_tf = L_STEP * FLOP_PER_SAMPLE / (k_ms * 1e-3) / 1e12
    kernel_name = f"stft2_kernel<4096,ci16,acc> (K1v2) variant {variant}" if variant in (0, 20, 21, 22) else f"stft_kernel<4096,ci16,acc> variant {variant}"
    traffic, traffic_src = traffic_record(kernel_name)
    ring_gsps = world * L_STEP * e2e_steps / dt_ring
    e2e = {"value": round(ring_gsps / 1e6, 1), "unit": "Msamples/s",
           "h2d_bytes_per_step": int(ring_h2d), "d2h_bytes_per_step": int(ring_d2h), "steps": e2e_steps,
           "ms_per_step": round(dt_ring / e2e_steps * 1e3, 3),
           "h2d_gbs_per_gpu": round(ring_h2d * e2e_steps / dt_ring / 1e9, 2), "d2h_gbs_per_gpu": round(ring_d2h * e2e_steps / dt_ring / 1e9, 2),
           "path": "spx_ring_* (pinned ring, 6 slots x 2^22 samples, uploads on two alternating streams): per slot H2D -> fused STFT + Welch finalize + classifier "
                   "features -> D2H of rows / Welch / max-hold / PSD / features; in-place producer (slots are the DMA target)",
           "memcpy_producer_first_pass_ms": round(dt_fill * 1e3, 1),
           "one_shot_call": {"value": round(world * L_STEP * call_steps / dt_call / 1e6, 1), "ms_per_step": round(dt_call / call_steps * 1e3, 3),
                             "h2d_bytes_per_step": int(r.h2d_bytes + NFFT * 8), "d2h_bytes_per_step": int(r.d2h_bytes + NFFT * 8 + 160),
                             "path": "spx_stft_exec(SPX_MEM_HOST) on the whole second + spx_welch_finalize + spx_classify_features"},
           "numa": numa}
    if ceil_s:
        e2e["copy_ceiling"] = {"ms_per_step": round(ceil_s * 1e3, 3), "h2d_gbs_per_gpu": round(host_in.nbytes / ceil_s / 1e9, 2),
                               "d2h_gbs_per_gpu": round(h_wf.nbytes / ceil_s / 1e9, 2),
                               "how": "spx_copy_ceiling: the same pinned buffers, H2D + D2H at once, 16 MiB pieces, all ranks at once, max over ranks"}
        e2e["frac_of_copy_ceiling"] = round(ceil_s / (dt_ring / e2e_steps), 4)
        e2e["one_shot_call"]["frac_of_copy_ceiling"] = round(ceil_s / (dt_call / call_steps), 4)
    line = {
        "metric": METRIC, "value": round(world * L_STEP * args.steps / dt_dev / 1e6, 1), "unit": "Msamples/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt_dev / args.steps * 1e3, 4),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "config2: 61.44 MS/s int16 IQ (1 s = 61 440 000 samples per step per GPU), 4096-pt Hann FFT, "
                               "75% overlap -> u8 waterfall rows + Welch + max-hold + classifier features",
                   "nfft": NFFT, "hop": HOP, "frames_per_step": F, "kernel_variant": variant,
                   "l2": "step input (246 MB) + rows (246 MB) exceed the 126 MB L2; no explicit flush",
                   "timing": "CUDA events on the plan's compute stream around the K steps (max over ranks); "
                             "the STFT kernel additionally bracketed per launch",
                   "multi_gpu": "value / e2e: replicas only (one independent stream per GPU, no data-path collective); "
                                "the configs that shard are in `sharded` (strong scaling, fused peer reduction)",
                   "real_time_margin_x": round(L_STEP * args.steps / dt_dev / FS, 1)},
        "e2e": e2e,
        "gpu_launches": 3 * args.steps,
        "roofline": {"bound": "fp32", "achieved": round(achieved_tf, 2), "peak": round(p32, 2), "unit": "TFLOP/s",
                     "frac": round(achieved_tf / p32, 4), "traffic": traffic, "traffic_source": traffic_src,
                     "peak_source": "FP32 FMA micro-kernel measured in this run (MEASURED_PEAKS.json holds no FP32 figure)",
                     "flop_per_sample": FLOP_PER_SAMPLE,
                     "kernel": kernel_name, "kernel_ms": round(k_ms, 4),
                     "kernel_share_of_step": round(k_ms * args.steps / (dt_dev * 1e3), 3),
                     "hbm": {"achieved_gbs": round(achieved_gbs, 1), "peak_gbs": peaks["hbm_gbs"], "frac": round(achieved_gbs / peaks["hbm_gbs"], 4),
                             "bytes_per_sample": BYTES_PER_SAMPLE, "peak_source": peak_src},
                     "note": "this shape transforms every sample 4 times (75% overlap): 320 nominal flop/sample vs 8 B/sample, "
                             "so FP32 binds before HBM (SURVEY 8d); the HBM-bound shape of north_star is in headline_shape",
                     "headline_shape": headline},
        "clocks": clocks,
        "features": {"snr_db": round(feat["snr_db"], 2), "peak_count": feat["peak_count"],
                     "ring_snr_db": None if not feat_ring else round(feat_ring["snr_db"], 2)},
    }
    if sustained is not None:
        line["sustained"] = sustained
    if views is not None:
        line["views_c3"] = views
    if sharded is not None:
        line["sharded"] = sharded
        checks = [v.get("check", "") for v in list(sharded["c5"].values()) + [sharded["c4"]] if isinstance(v, dict)]
        line["sharded"]["parity"] = "ok" if all(c.startswith("ok") for c in checks) else "FAILED"
        if line["sharded"]["parity"] != "ok":
            print("SHARDED PARITY CHECK FAILED: " + "; ".join(checks), file=sys.stderr, flush=True)
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_single()
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
