#!/usr/bin/env python3
"""K1 (variant 12) vs the default K1v2 (variant 0) on the shapes that matter, device-resident, CUDA events (B200 box):
python tools/sweep_k1v2.py [12,0]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import kernel_sweep as ks
from sdr_iq_visualizer_b200 import spectral as sp
variants = [int(v) for v in (sys.argv[1].split(",") if len(sys.argv) > 1 else "12,0".split(","))]
L = 61_440_000
for v in variants:
    ks.run_case("C2 ci16 75% u8+acc", 4096, 1024, "hann", sp.FMT_CI16, L, ["u8", "acc"], v)
    ks.run_case("headline cf32 hop=N f32", 4096, 4096, "hann", sp.FMT_CF32, L, ["db"], v)
    ks.run_case("cf32 hop=N u8", 4096, 4096, "hann", sp.FMT_CF32, L, ["u8"], v)
    ks.run_case("cf32 50% f32", 4096, 2048, "hann", sp.FMT_CF32, L, ["db"], v)
    ks.run_case("C4 shape cf32 N=2048 50% acc", 2048, 1024, "hann", sp.FMT_CF32, L, ["acc"], v)
    ks.run_case("cf32 N=2048 hop=N f32", 2048, 2048, "hann", sp.FMT_CF32, L, ["db"], v)
    ks.run_case("C1 shape cf32 N=1024 50% u8+acc", 1024, 512, "hann", sp.FMT_CF32, L, ["u8", "acc"], v)
    ks.run_case("cf32 N=1024 hop=N f32", 1024, 1024, "hann", sp.FMT_CF32, L, ["db"], v)
