"""Cost of signal extraction: the multi-job DDC (DdcPlan.exec_jobs, ddc_jobs_kernel) and sigmf_io.extract_signals on one
GPU; prints one JSON line.

Shapes:
  (X1) many small jobs: the config-2 capture, 61.44 M ci16 samples, 512 jobs of 120 000 samples each (1850 outputs) at
       D = 64, default taps (T = 1607), one exec_jobs call against 512 DdcPlan.exec calls on device views of the same
       spans;
  (X2) few long jobs: the same capture in 4 jobs at D = 64, against one DdcPlan.exec of the whole capture (K9's Z1);
  (call) extract_signals on a synthetic ci16 recording of 2^26 samples with 100 tone bursts, host wall time of the
       detection (detect_signals), of the extraction with classification (extract_signals on those annotations) and of
       the classification alone (measure_batch + the rule table on the returned spectra, repeated).
Device legs are timed with CUDA events after warm-up, alternating round by round; kernel times come from torch.profiler in
a run of their own.  Cost model as tools/bench_ddc.py: per input sample in_B + 8/D bytes and 4T/D + 6 flops (the NCO's
sine and cosine not counted), against the FP32 peak from spx_fp32_peak in the same run.  The card's name and power limit
are read in the same run.

    python tools/bench_extract.py [--steps 20] [--warmup 3] [--out FILE]
"""
import argparse
import json
import os
import shutil
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

from tools.bench_ddc import FS, cost, roofline, timed   # noqa: E402
from tools.bench_persistence import gpu_name_power   # noqa: E402


def kernel_us(fn, steps, nat, name):
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
    ev = [e for e in prof.events() if e.device_type == DeviceType.CUDA and name in e.name]
    return sum(e.device_time_total for e in ev) / steps, len(ev) // steps


def synth_bursts(L, n_bursts, fs, seed):
    """ci16 noise with n_bursts tone bursts on a 10 x (n_bursts / 10) time-frequency grid."""
    rng = np.random.default_rng(seed)
    x = (rng.normal(size=L) + 1j * rng.normal(size=L)).astype(np.complex64) * np.float32(0.01)
    rows = 10
    cols = n_bursts // rows
    seg = L // rows
    for k in range(n_bursts):
        r, c = divmod(k, cols)
        f = (c + 0.5) / cols - 0.5
        a, n = r * seg + seg // 8, seg * 3 // 4
        t = np.arange(a, a + n)
        x[a:a + n] += (0.05 * np.exp(2j * np.pi * f * t)).astype(np.complex64)
    iq = np.empty(2 * L, np.int16)
    iq[0::2] = np.clip(np.rint(x.real * 32768), -32768, 32767)
    iq[1::2] = np.clip(np.rint(x.imag * 32768), -32768, 32767)
    return iq


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    from sdr_iq_visualizer_b200 import _native as nat, classifier as cls_mod, ddc, features, sigmf_io as sio
    from sdr_iq_visualizer_b200 import spectral as sp, synth
    nat.require_device()
    name, power = gpu_name_power()
    peak = nat.fp32_peak_tflops(0)
    result = {"tool": "bench_extract", "gpu": name, "power_limit": power, "fp32_peak_tflops": round(peak, 2),
              "steps": args.steps, "warmup": args.warmup,
              "cost_model": "bytes/sample = in_B + 8/D; flops/sample = 4T/D + 6 (sincos not counted)"}
    L = 61_440_000
    D = 64
    d_x = nat.DeviceArray.from_host(synth.tiled_ci16(L, seed=2))
    st_plan = sp.SpectralPlan(1024, 1024, "hann", sp.FMT_CF32)
    st = st_plan.stream
    p = ddc.DdcPlan(FS, 7.3e6, D, in_fmt=sp.FMT_CI16, in_scale=2.0 ** -15)
    T = p.n_taps
    # X1: 512 spans of 120 000 samples, one NCO each
    span, n_jobs = 120_000, 512
    step = L // n_jobs
    n1 = p.out_count(span)
    incs = [ddc.phase_increment(((j * 0.618034) % 1.0 - 0.5) * FS, FS)[0] for j in range(n_jobs)]
    jobs1 = ddc.as_jobs([(j * step, incs[j], 0, n1, j * n1) for j in range(n_jobs)])
    out1 = nat.DeviceArray((n_jobs * n1,), np.complex64)
    views = [(nat.DeviceView(d_x.ptr + 4 * j * step, (2 * span,), np.int16),
              nat.DeviceView(out1.ptr + 8 * j * n1, (n1,), np.complex64), j * step) for j in range(n_jobs)]

    def x1_loop():
        for v, o, a in views:
            p.exec(v, out=o, first_sample=a, stream=st)
    # X2: 4 jobs over the whole capture against one K9 call
    q = L // 4
    jobs2, off = [], 0
    for j in range(4):
        n = p.out_count(min(L, (j + 1) * q + T - 1) - j * q)
        jobs2.append((j * q, p.phase_inc, 0, n, off))
        off += n
    jobs2 = ddc.as_jobs(jobs2)
    out2 = nat.DeviceArray((off,), np.complex64)
    out_z1 = nat.DeviceArray((p.out_count(L),), np.complex64)
    legs = {"X1_exec_jobs": lambda: p.exec_jobs(d_x, jobs1, out1, stream=st),
            "X1_per_job_loop": x1_loop,
            "X2_exec_jobs": lambda: p.exec_jobs(d_x, jobs2, out2, stream=st),
            "Z1_exec": lambda: p.exec(d_x, out=out_z1, stream=st)}
    res = timed(legs, args.steps, args.warmup, nat, st)
    for k, (ms, rounds) in res.items():
        result[k + "_ms"] = ms
        result[k + "_ms_rounds"] = rounds
    result["X1_speedup_over_loop"] = round(res["X1_per_job_loop"][0] / res["X1_exec_jobs"][0], 2)
    result["X2_rate_vs_Z1"] = round(res["Z1_exec"][0] / res["X2_exec_jobs"][0], 4)
    for k, samples, kname in (("X1_exec_jobs", n_jobs * span, "ddc_jobs_kernel"), ("X2_exec_jobs", L, "ddc_jobs_kernel"),
                              ("Z1_exec", L, "ddc_kernel"), ("X1_per_job_loop", n_jobs * span, "ddc_kernel")):
        us, launches = kernel_us(legs[k], 3, nat, kname)
        r = roofline(dict(cost(samples, 4, T, D), samples=samples), us, peak)
        r.update({"kernel": kname, "launches_per_call": launches, "samples": samples,
                  "Gsamples_per_s_kernel": round(samples / us / 1e3, 2),
                  "Gsamples_per_s_events": round(samples / res[k][0] / 1e6, 2)})
        result[k] = r
    p.close()
    del d_x, out1, out2, out_z1
    # the whole call on a recording of 2^26 samples with 100 bursts
    tmp = tempfile.mkdtemp(prefix="bench_extract_")
    try:
        fs_r, fc_r, Lr = 61.44e6, 2.4e9, 1 << 26
        base = sio.write_recording(os.path.join(tmp, "bursts"), synth_bursts(Lr, 100, fs_r, 7), fs_r, fc_r, "ci16_le")
        sio.detect_signals(base)                      # warm-up of every plan and kernel the call uses
        t0 = time.perf_counter()
        _, ann = sio.detect_signals(base)
        t1 = time.perf_counter()
        sigs = sio.extract_signals(base, ann)
        t2 = time.perf_counter()
        sigs = sio.extract_signals(base, ann)
        t3 = time.perf_counter()
        nfft = 256
        lo, hi = nfft // 4, nfft - nfft // 4
        live = [s for s in sigs if s.pxx is not None]
        band = np.array([10.0 * np.log10(s.pxx[lo:hi]) for s in live])
        t4 = time.perf_counter()
        meas = features.measure_batch(band) if live else []
        for s, m in zip(live, meas):
            fj = s.center_freq + sp.freq_axis(nfft, s.sample_rate, 0.0)[lo:hi]
            cls_mod.classify_from_measurements(fj, cls_mod.add_hz(fj, m), hi - lo, smooth=False)
        t5 = time.perf_counter()
        labels = {}
        for s in sigs:
            labels[str(s.label)] = labels.get(str(s.label), 0) + 1
        result["call"] = {"samples": Lr, "fmt": "ci16", "regions": len(ann),
                          "decims": sorted({s.decim for s in sigs}), "detect_ms": round((t1 - t0) * 1e3, 1),
                          "extract_and_classify_ms": [round((t2 - t1) * 1e3, 1), round((t3 - t2) * 1e3, 1)],
                          "classify_only_ms": round((t5 - t4) * 1e3, 1), "labels": labels}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
