"""CPU tests of signal extraction: the multi-job DDC's work split (csrc/spx_ddc_device.cuh, run by the host harness
tests/emul/ddc_jobs_emul.cu), the region -> down-conversion planning of sigmf_io.signal_jobs and the chunk schedule of
sigmf_io.extract_signals."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

EMUL_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emul", "ddc_jobs_emul.cu")


@pytest.fixture(scope="module")
def walk_lib(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.fail("nvcc is needed to build the DDC work-split harness")
    so = str(tmp_path_factory.mktemp("ddc_walk") / "libddc_walk.so")
    subprocess.run([nvcc, "-std=c++17", "-O2", "-shared", "-Xcompiler", "-fPIC", "-gencode",
                    "arch=compute_100a,code=sm_100a", "-o", so, EMUL_SRC], check=True)
    lib = C.CDLL(so)
    lib.emul_job_walk.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_int64]
    lib.emul_job_walk.restype = C.c_int64
    return lib


def walk(lib, n_out, sub, grid):
    """The parts (cta, job, k0, k1) the CTAs of ddc_jobs_kernel walk for jobs of n_out outputs and sub-tiles of sub."""
    tile0 = np.concatenate([[0], np.cumsum([-(-n // sub) for n in n_out])]).astype(np.int64)
    cap = int(tile0[-1]) + 2 * grid + 8
    seg = np.zeros((cap, 4), np.int64)
    n = lib.emul_job_walk(tile0.ctypes.data, len(n_out), grid, seg.ctypes.data, cap)
    assert n <= cap
    return seg[:n]


def check_cover(n_out, sub, segs):
    cover = [np.zeros(n, np.int32) for n in n_out]
    for b, j, k0, k1 in segs:
        assert n_out[j] > 0 and 0 <= k0 < k1 <= -(-n_out[j] // sub)
        cover[j][k0 * sub: min(k1 * sub, n_out[j])] += 1
    for j, c in enumerate(cover):
        assert (c == 1).all(), (j, n_out[j])


@pytest.mark.parametrize("sub", [16, 64, 128, 256])
def test_job_walk_covers_every_output_once(walk_lib, sub):
    edge = [0, 1, sub - 1, sub, sub + 1]
    rng = np.random.default_rng(sub)
    tables = [edge, edge[::-1] * 3, [0, 0, 5, 0], [1] * 50, [sub * 7 + 3]]
    tables += [list(rng.choice(edge + [int(v) for v in rng.integers(0, 20 * sub, 8)], rng.integers(1, 300)))
               for _ in range(30)]
    crossed = 0
    for n_out in tables:
        n_sub = sum(-(-n // sub) for n in n_out)
        for grid in sorted({1, 2, 3, 7, 296, max(1, n_sub // 3), max(1, n_sub)}):
            if n_sub == 0:
                continue
            segs = walk(walk_lib, n_out, sub, min(grid, n_sub))
            check_cover(n_out, sub, segs)
            per_cta = np.bincount(segs[:, 0])
            crossed = max(crossed, int(per_cta.max()))
            # a CTA's parts follow each other: contiguous global sub-tiles, increasing jobs
            for b in np.unique(segs[:, 0]):
                s = segs[segs[:, 0] == b]
                assert (np.diff(s[:, 1]) > 0).all()
    assert crossed >= 3   # some CTA ran across two or more job boundaries


def test_job_of_skips_empty_jobs(walk_lib):
    segs = walk(walk_lib, [0, 3, 0, 0, 2, 0], 2, 1)
    assert [tuple(r) for r in segs] == [(0, 1, 0, 2), (0, 4, 0, 1)]


# ----------------------------------------------------------------------------- region -> job
def ann(start, count, lo, hi):
    return {"core:sample_start": start, "core:sample_count": count, "core:freq_lower_edge": lo, "core:freq_upper_edge": hi}


def test_signal_jobs_hand_computed():
    from sdr_iq_visualizer_b200 import ddc, sigmf_io as sio
    fs, fc, L = 1.024e6, 100e6, 10_000_000
    # bw 1 kHz: fs / D >= 2 kHz up to D = 512 -> clamped at 256
    (shift, inc, D, first, n), = sio.signal_jobs([ann(1_000_000, 100_000, fc + 1e3, fc + 2e3)], fs, fc, L)
    T = ddc.design_taps(256).size
    assert D == 256 and (inc, shift) == ddc.phase_increment(1.5e3, fs)
    assert first == 1_000_000 - (T - 1) // 2 and n == (100_000 + T - 1 - T) // 256 + 1
    # every power-of-two boundary: bw = fs / (2 D) gives D exactly, a hair more gives D / 2
    for D in (1, 2, 4, 8, 16, 32, 64, 128, 256):
        bw = fs / (2 * D)
        got = sio.signal_jobs([ann(0, 1000, fc - bw / 2, fc + bw / 2)], fs, fc, L)[0]
        assert got[2] == D and got[0] == 0.0 and got[1] == 0
        if D > 1:
            assert sio.signal_jobs([ann(0, 1000, fc - bw / 2, fc + bw / 2 + 1.0)], fs, fc, L)[0][2] == D // 2
    assert sio.signal_jobs([ann(0, 1000, fc, fc + 10.0)], fs, fc, L, max_decim=20)[0][2] == 16
    assert sio.signal_jobs([ann(0, 1000, fc - fs / 2, fc + fs / 2)], fs, fc, L)[0][2] == 1   # wider than fs / 2: D = 1


def test_signal_jobs_rejects_filters_over_one_stage():
    from sdr_iq_visualizer_b200 import sigmf_io as sio
    with pytest.raises(ValueError, match="8192"):
        sio.signal_jobs([], 1e6, 0.0, 100, max_decim=512)
    with pytest.raises(ValueError):
        sio.signal_jobs([], 1e6, 0.0, 100, max_decim=0)
    assert sio.signal_jobs([], 1e6, 0.0, 100, max_decim=511) == []


def test_signal_jobs_spans_and_shifts():
    from sdr_iq_visualizer_b200 import ddc, sigmf_io as sio
    fs, fc, L = 1e6, 0.0, 50_000
    T = ddc.design_taps(8).size     # 203
    bw = fs / 16                    # fs / D >= 2 bw: D = 8
    h = (T - 1) // 2
    jobs = sio.signal_jobs([ann(10, 1000, -bw / 2, bw / 2),             # clipped at 0
                            ann(L - 500, 500, -bw / 2, bw / 2),         # clipped at L
                            ann(20_000, 100, -bw / 2, bw / 2),          # not clipped
                            ann(30_000, 0, -bw / 2, bw / 2),            # len = 2h = T - 1 < T: no output
                            ann(5, 3, -bw / 2 - 2e5, bw / 2 - 2e5),     # negative shift, len < T
                            ann(0, L, fs / 2 - 1, fs / 2 + 1),          # +fs/2
                            ann(0, L, -fs / 2 - 1, -fs / 2 + 1)], fs, fc, L)  # -fs/2
    assert jobs[0][3] == 0 and jobs[0][4] == (10 + 1000 + h - T) // 8 + 1
    assert jobs[1][3] == L - 500 - h and jobs[1][4] == (500 + h - T) // 8 + 1
    assert jobs[2][3] == 20_000 - h and jobs[2][4] == (100 + 2 * h - T) // 8 + 1
    assert jobs[3][4] == 0 and jobs[4][4] == 0
    assert jobs[4][:2] == ddc.phase_increment(-2e5, fs)[::-1] and jobs[4][0] == -2e5
    assert jobs[5][1] == jobs[6][1] == -(1 << 63) and jobs[5][0] == jobs[6][0] == -fs / 2
    T256 = ddc.design_taps(256).size
    assert jobs[5][2] == 256 and jobs[5][3] == 0 and jobs[5][4] == (L - T256) // 256 + 1   # a 2 Hz band: D = 256


# ----------------------------------------------------------------------------- chunk schedule
@pytest.mark.parametrize("seed", range(12))
def test_extract_schedule_produces_each_output_once(seed):
    from sdr_iq_visualizer_b200 import sigmf_io as sio
    rng = np.random.default_rng(seed)
    L = int(rng.integers(1, 200_000))
    spans = []
    for _ in range(int(rng.integers(1, 40))):
        D = int(2 ** rng.integers(0, 9))
        T = int(rng.integers(1, 2000))
        first = int(rng.integers(0, L))
        n_max = (L - first - T) // D + 1 if L - first >= T else 0
        spans.append((first, int(rng.integers(0, n_max + 1)) if n_max > 0 and rng.random() < 0.9 else 0, D, T))
    chunk = int(rng.choice([1, 100, 4096, 50_000, 1 << 26]))
    got = [np.zeros(n, np.int32) for _, n, _, _ in spans]
    T_max = max([T for _, n, _, T in spans if n] or [1])
    prev = None
    for c0, c1, parts in sio.extract_schedule(spans, L, chunk):
        assert 0 <= c0 < c1 <= L and c1 - c0 <= max(chunk, T_max)
        if prev is not None:
            assert c0 > prev[0] and c0 >= prev[1] - (T_max - 1)
        prev = (c0, c1)
        for j, m0, n in parts:
            first, _, D, T = spans[j]
            assert n > 0 and first + m0 * D >= c0 and first + (m0 + n - 1) * D + T <= c1   # windows inside the chunk
            got[j][m0:m0 + n] += 1
    for g in got:
        assert (g == 1).all()


def test_as_jobs():
    from sdr_iq_visualizer_b200 import ddc
    j = ddc.as_jobs([(5, (1 << 64) - 1, 0, 3, 7), (0, 1 << 63, 2, 0, 0)])
    assert j.dtype == ddc.JOB_DTYPE and j["phase_inc"].tolist() == [-1, -(1 << 63)]
    assert j["first_sample"].tolist() == [5, 0] and j["out_offset"].tolist() == [7, 0]
    assert ddc.JOB_DTYPE.itemsize == 40
