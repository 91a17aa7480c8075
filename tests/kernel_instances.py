"""Every kernel instance libspx.so builds, and the case that holds each one to the float64 oracle.

``inventory(lib)`` lists the instances of a built library (``cuobjdump -sass`` function names through ``cu++filt``);
``key(name)`` maps a demangled name, in cu++filt's form or in the CUDA profiler's, to one canonical key; ``CASES`` is the
table of GPU cases (tests/test_kernel_instances_gpu.py runs each once and checks that its ``expects`` launched);
``EXEMPT`` lists the only instances without a case.  tests/test_kernel_instances_cpu.py asserts that the union of all
``expects`` and ``EXEMPT`` is exactly the inventory, so a new template instance without a case fails on any machine.

No device calls here: the module imports on a CPU-only machine.
"""
from __future__ import annotations

import os
import re
import shutil
import subprocess

# bench.py's measurement kernels (FP32 peak probe, L2 flush); they compute nothing a user sees
EXEMPT = frozenset({"fp32_probe_kernel", "l2_flush_read_kernel"})

SMS = 148                  # streaming multiprocessors of a B200: the figure launch_stft_inst's chunking uses
# every K1 / K1v2 instance holds more than 64 registers per thread (cuobjdump -res-usage: 66 .. 128), so at most
# 65536 / 64 = 1024 of their threads are resident on an SM
MAX_THREADS_PER_SM = 1024

# outputs of an STFT call
ROWS = ("db_rows", "wf_rows", "spectrum")                       # every row output, no accumulators
ALL = ROWS + ("welch", "maxhold")
ACC = ("welch", "maxhold")
U8 = ("wf_rows",)
DB = ("db_rows",)


# ----------------------------------------------------------------------------- names
def _toolkit_bin(tool: str) -> str:
    """A CUDA toolkit binary, found the way _native.build finds nvcc: on PATH, else /usr/local/cuda/bin."""
    return shutil.which(tool) or os.path.join("/usr/local/cuda/bin", tool)


def inventory(lib_path: str) -> list:
    """Demangled names of every kernel (``Function :`` entry of ``cuobjdump -sass``) in the library."""
    sass = subprocess.run([_toolkit_bin("cuobjdump"), "-sass", lib_path], check=True, capture_output=True, text=True).stdout
    mangled = sorted({ln.split("Function :", 1)[1].strip() for ln in sass.splitlines() if "Function :" in ln})
    out = subprocess.run([_toolkit_bin("cu++filt")], input="\n".join(mangled) + "\n", check=True, capture_output=True,
                         text=True).stdout
    return [ln.strip() for ln in out.splitlines() if ln.strip()]


def key(name: str) -> str:
    """Canonical key of a demangled kernel name: no ``void ``, no ``spx::``, no parameter list, ints printed plainly,
    bools as true / false.  ``spx::stft2_kernel<(int)1024, (int)0, (bool)1, (int)2, (int)23>(spx::StftParams,
    CUtensorMap)`` and ``void spx::stft2_kernel<1024, 0, true, 2, 23>(spx::StftParams, CUtensorMap_st)`` both give
    ``stft2_kernel<1024, 0, true, 2, 23>``."""
    s = name.strip()
    if s.startswith("void "):
        s = s[5:]
    depth = 0
    for i, c in enumerate(s):                      # the parameter list: the first '(' outside the template arguments
        if c == "<":
            depth += 1
        elif c == ">":
            depth -= 1
        elif c == "(" and depth == 0:
            s = s[:i]
            break
    s = s.replace("spx::", "")
    s = re.sub(r"\(bool\)1\b", "true", s)
    s = re.sub(r"\(bool\)0\b", "false", s)
    s = re.sub(r"\((?:unsigned |signed )?(?:int|long|long long|short|char)\)(-?\d+)[uUlL]*", r"\1", s)
    s = re.sub(r"\s*,\s*", ", ", s)
    s = re.sub(r"\s*<\s*", "<", s)
    s = re.sub(r"\s*>", ">", s)
    return s.strip()


def _b(v: bool) -> str:
    return "true" if v else "false"


# ----------------------------------------------------------------------------- instance keys per family
def k1(n, fmt, acc, twm, occ, stage):
    """K1 ``stft_kernel<N, FMT, ACC, TWM, OCC, STAGE, TUNE_I2FP>`` (TWM: 0 L1 table, 1 registers, 2 shared memory)."""
    return f"stft_kernel<{n}, {fmt}, {_b(acc)}, {twm}, {occ}, {_b(stage)}, 1>"


def k1v2(n, fmt, acc, tune):
    return f"stft2_kernel<{n}, {fmt}, {_b(acc)}, 2, {tune}>"


def k2_cols(n, fmt, bulk):
    n1 = {14: 128, 15: 128, 16: 256, 17: 256, 18: 512, 19: 512, 20: 1024}[n.bit_length() - 1]
    return f"big_cols_kernel<{n1}, {n // n1}, {fmt}, {_b(bulk)}>"


def k2_rows(n, acc):
    n1 = {14: 128, 15: 128, 16: 256, 17: 256, 18: 512, 19: 512, 20: 1024}[n.bit_length() - 1]
    return f"big_rows_kernel<{n1}, {n // n1}, {_b(acc)}, true>"


# K1v2 output specialisations (spx_stft2_device.cuh: TUNE_*); T0 = TUNE_I2FP | TUNE_FMADFT | TUNE_QFMA
T0, L2PF, ONLY_U8, ONLY_DB, NO_ROWS = 7, 8, 16, 32, 64


# ----------------------------------------------------------------------------- frame counts
def k1_geometry(n):
    """(threads per CTA, frames in flight per CTA) of K1 at N (StftCfg<N>)."""
    t = n // 16
    fpc = 1 if t >= 256 else 256 // t
    return t * fpc, fpc


def k1v2_geometry(n):
    return 256, 4096 // n                   # Stft2Cfg<N, FMT>


def stft_frames(threads, fpc):
    """Frames of a K1 / K1v2 case.  launch_stft_inst gives each of W = SMs x occupancy x (frames per CTA) workers one chunk
    of ceil(F / W) frames.  The occupancy is at most 1024 / threads, so F = W_max + 1 puts at least 2 frames in every
    chunk at any occupancy: every worker's frame loop runs more than once, its accumulators are flushed from several
    frames, and the last chunk is short (for N = 4096, K1v2: W_max = 148 x 4 x 1 = 592, F = 593; for N = 16, K1:
    W_max = 148 x 4 x 256 = 151552)."""
    w_max = SMS * (MAX_THREADS_PER_SM // threads) * fpc
    return w_max + 1


def chunk_sizes(F, threads, fpc):
    """The frames per chunk launch_stft_inst picks at every occupancy the CTA size allows (the rows on both sides of
    each of their chunk boundaries are checked)."""
    out = set()
    for occ in range(1, MAX_THREADS_PER_SM // threads + 1):
        w = SMS * occ * fpc
        c = -(-F // w)
        if c > 256:
            waves = -(-c // 256)
            c = -(-c // waves)
        out.add(min(c, F))
    return sorted(out)


# ----------------------------------------------------------------------------- the case table
def _stft(cid, family, n, hop, fmt, outs, expects, frames, variant=0, kind="hann", geom=None):
    return dict(id=cid, family=family, n=n, hop=hop, fmt=fmt, outs=tuple(outs), variant=variant, kind=kind, frames=frames,
                geom=geom, mem="device", expects=frozenset(expects))


def _stft_cases():
    cases = []
    # K1, N = 16 .. 256: one twiddle mode, direct loads only (STAGE_WANTED is false below 512)
    for n in (16, 32, 64, 128, 256):
        g = k1_geometry(n)
        for fmt in (0, 1):
            for acc in (False, True):
                cases.append(_stft(f"K1 N={n} fmt={fmt} acc={acc}", "stft", n, n // 2 + 1, fmt, ALL if acc else ROWS,
                                   [k1(n, fmt, acc, 0, 2, False)], stft_frames(*g), geom=g))
    # K1 with staged (bulk-copy) input where hop * elt is a multiple of 16 bytes, direct loads where it is not.  At N =
    # 1024 / 2048 / 4096 K1v2 is the default, so the staged cases force K1 with variant 12 and the direct cases use a hop
    # that is not 128-byte aligned (K1v2 then falls back to K1 by itself).  N = 1024 builds the shared-memory twiddle
    # table without accumulators and the L1 table with them (spx_stft_1k2k.cu).
    k1_staged = {512: (0, 2, (False, True)), 1024: (None, 2, (False, True)), 2048: (0, 2, (False, True)),
                 4096: (1, 2, (False, True)), 8192: (0, 1, (False, True))}
    for n, (twm, occ, _) in k1_staged.items():
        g = k1_geometry(n)
        for fmt in (0, 1):
            for acc in (False, True):
                tw = (0 if acc else 2) if n == 1024 else twm
                for stage in (True, False):
                    hop = n // 2 if stage else n // 2 + 1
                    variant = 12 if stage and 1024 <= n <= 4096 else 0
                    cases.append(_stft(f"K1 N={n} fmt={fmt} acc={acc} {'staged' if stage else 'direct'}", "stft", n, hop,
                                       fmt, ALL if acc else ROWS, [k1(n, fmt, acc, tw, occ, stage)], stft_frames(*g),
                                       variant=variant, geom=g))
    # K1v2: the output set picks the specialisation (spx_stft2.cu launch_outs): u8 rows only, dB rows only, accumulators
    # only, or anything else (the generic kernel); each with and without accumulators.  cf32 N = 4096 takes the L2
    # prefetch kernels at hop >= 4096 and the strip kernel at hop = 1024, so its plain kernels run at hop 2048.
    out_sets = [(ROWS, T0, False), (ALL, T0, True), (U8, T0 | ONLY_U8, False), (U8 + ACC, T0 | ONLY_U8, True),
                (DB, T0 | ONLY_DB, False), (DB + ACC, T0 | ONLY_DB, True), (ACC, T0 | NO_ROWS, True)]
    for n in (1024, 2048, 4096):
        g = k1v2_geometry(n)
        for fmt in (0, 1):
            hops = [(n // 2, 0)] if not (n == 4096 and fmt == 0) else [(2048, 0), (4096, L2PF)]
            for hop, extra in hops:
                for outs, tune, acc in out_sets:
                    cases.append(_stft(f"K1v2 N={n} fmt={fmt} hop={hop} tune={tune | extra} acc={acc}", "stft", n, hop,
                                       fmt, outs, [k1v2(n, fmt, acc, tune | extra)], stft_frames(*g), geom=g))
    for acc in (False, True):
        cases.append(_stft(f"K1v2 strip acc={acc}", "stft", 4096, 1024, 0, ALL if acc else ROWS,
                           [f"stft2_strip_kernel<0, {_b(acc)}, 4, 2, 7>"], stft_frames(256, 1), geom=(256, 1)))
    # K2 (four-step, column kernel + row kernel), N = 2^14 .. 2^20.  Bulk copies need hop * elt to be a multiple of 16
    # bytes; dB rows keep N = 65536 off K2v2.  Each N: both formats, both copy modes, both row kernels.
    for e in range(14, 21):
        n = 1 << e
        frames = 6 if e >= 18 else 24
        for fmt, bulk, acc in ((0, True, True), (0, False, False), (1, True, False), (1, False, True)):
            hop = n // 2 if bulk else n // 2 + 1
            cases.append(_stft(f"K2 N={n} fmt={fmt} {'bulk' if bulk else 'direct'} acc={acc}", "stft", n, hop, fmt,
                               ALL if acc else ROWS, [k2_cols(n, fmt, bulk), k2_rows(n, acc)], frames))
    # K2v2 (N = 65536, outputs among u8 rows and accumulators, hop a multiple of 256): 41 frames over its lanes of 16 CTAs
    for fmt in (0, 1):
        for acc in (False, True):
            cases.append(_stft(f"K2v2 fmt={fmt} acc={acc}", "stft", 65536, 32768, fmt, U8 + ACC if acc else U8,
                               [f"big2_kernel<{_b(acc)}, {fmt}>"], 41))
    # Bluestein (N not a power of two): pre-chirp per format, post per accumulator flag
    for fmt, acc in ((0, True), (1, False)):
        cases.append(_stft(f"Bluestein N=3000 fmt={fmt} acc={acc}", "stft", 3000, 1500, fmt, ALL if acc else ROWS,
                           [f"blu_pre_kernel<{fmt}>", "blu_mul_kernel", f"blu_post_kernel<{_b(acc)}>"], 70))
    return cases


def _other_cases():
    cases = []
    for dtype in ("float64", "float32"):
        cases.append(dict(id=f"K3 features {dtype}", family="features", dtype=dtype,
                          expects=frozenset({f"features_kernel<{'double' if dtype == 'float64' else 'float'}>"})))
    # K4 histogram: shared-memory tables (> 4 CTAs: per-CTA tables merged) and the global-atomic kernel (bins 400 / 512)
    for fmt in (0, 1):
        cases.append(dict(id=f"K4 hist2d smem fmt={fmt}", family="hist2d", fmt=fmt, bins=256,
                          expects=frozenset({f"hist2d_smem_kernel<{fmt}>", "hist_merge_kernel", "hist_zero_kernel"})))
        cases.append(dict(id=f"K4 hist2d global fmt={fmt}", family="hist2d", fmt=fmt, bins=512 if fmt else 400,
                          expects=frozenset({f"hist2d_kernel<{fmt}>"})))
        cases.append(dict(id=f"K4 frame_stats fmt={fmt}", family="frame_stats", fmt=fmt,
                          expects=frozenset({f"frame_stats_kernel<{fmt}>"})))
    cases.append(dict(id="K6 stream_frame f64", family="stream_frame",
                      expects=frozenset({"stream_frame_f64_kernel<true>", "stream_frame_f64_kernel<false>"})))
    cases.append(dict(id="K7 persistence", family="persistence", expects=frozenset({"persist_kernel"})))
    for mode in ("mean", "max"):
        cases.append(dict(id=f"K8 pool {mode}", family="pool", mode=mode,
                          expects=frozenset({f"pool_kernel<{_b(mode == 'max')}>", "pool_finalize_kernel", "pool_fill_kernel"})))
    for fmt in (0, 1):
        cases.append(dict(id=f"K9 ddc fmt={fmt}", family="ddc", fmt=fmt,
                          expects=frozenset({f"ddc_kernel<{fmt}>", f"ddc_jobs_kernel<{fmt}>"})))
    for m in (16, 32, 64, 128, 256, 512, 1024, 2048, 4096):
        for fmt in (0, 1):
            cases.append(dict(id=f"K10 chan M={m} fmt={fmt}", family="chan", m=m, fmt=fmt, decim=m // 2, taps=None,
                              expects=frozenset({f"chan_kernel<{fmt}, {m}>"})))
        if 32 <= m <= 512:       # critically sampled with the longest window the handle takes
            fmt = (m.bit_length() - 1) % 2
            cases.append(dict(id=f"K10 chan M={m} fmt={fmt} D=M T=32M", family="chan", m=m, fmt=fmt, decim=m,
                              taps=32 * m, expects=frozenset({f"chan_kernel<{fmt}, {m}>"})))
    cases.append(dict(id="K11 detect", family="detect", expects=frozenset(
        {"det_local_kernel", "det_border_kernel", "det_flatten_kernel", "det_scan_kernel", "det_assign_kernel",
         "det_stats_kernel", "det_keep_kernel", "det_number_kernel", "det_relabel_kernel"})))
    cases.append(dict(id="welch_finalize", family="welch_finalize", expects=frozenset({"welch_finalize_kernel"})))
    cases.append(dict(id="ring carry", family="ring", expects=frozenset({"ring_carry_kernel"})))
    cases.append(dict(id="peer reduce", family="peer_reduce", expects=frozenset({"peer_reduce_kernel"})))
    return cases


CASES = _stft_cases() + _other_cases()


def covered() -> set:
    """Every key some case expects, plus the exempt ones."""
    out = set(EXEMPT)
    for c in CASES:
        out |= c["expects"]
    return out
