"""CPU tests of the channelizer: the two statements of the float64 oracle against each other, K10's fold, index maps and
FFT phases (csrc/spx_chan_device.cuh, compiled for the host by tests/emul/chan_emul.cu) against the oracle and against
themselves under splits, and the host-side checks that run before any device call."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from tests import chan_ref as cr

EMUL_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emul", "chan_emul.cu")
FIRSTS = [0, 1, None, (1 << 40) + 5]          # None: M + 3


def _x(L, seed, fmt="cf32"):
    rng = np.random.default_rng(seed)
    xc = (rng.normal(size=L) + 1j * rng.normal(size=L)) * 0.3
    if fmt == "ci16":
        x = np.empty(2 * L, np.int16)
        x[0::2] = np.clip(np.rint(xc.real * 8000), -32768, 32767)
        x[1::2] = np.clip(np.rint(xc.imag * 8000), -32768, 32767)
        return x, 2.0 ** -15
    return xc.astype(np.complex64), 1.0


# ----------------------------------------------------------------------------- the oracle, written twice
@pytest.mark.parametrize("M", [16, 64])
@pytest.mark.parametrize("half", [True, False])
@pytest.mark.parametrize("first", FIRSTS)
@pytest.mark.parametrize("Tk", ["1", "M", "32M"])
def test_oracle_fold_fft_equals_ddc_loop(M, half, first, Tk):
    D = M // 2 if half else M
    T = {"1": 1, "M": M, "32M": 32 * M}[Tk]
    first = M + 3 if first is None else first
    rng = np.random.default_rng(M * 7 + T)
    h = rng.normal(size=T) / np.sqrt(T)
    x, _ = _x(T + 9 * D + 3, M + T)
    a = cr.channelize(x, h, M, D, first)
    b = cr.channelize_ddc(x, h, M, D, first)
    assert a.shape == b.shape == (M, cr.out_count(T + 9 * D + 3, T, D))
    assert np.abs(a - b).max() <= 1e-12 * cr.bound(h, x)


def test_oracle_phase_inc_exact():
    assert cr.phase_inc(0, 64) == -(1 << 63)            # c = -M/2: -fs/2
    assert cr.phase_inc(32, 64) == 0
    assert cr.phase_inc(33, 64) == 1 << 58
    assert cr.phase_inc(31, 64) == -(1 << 58)
    assert cr.channelize(np.zeros(5, np.complex64), np.ones(9), 16, 8).shape == (16, 0)


# ----------------------------------------------------------------------------- K10's math on the CPU
@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.fail("nvcc is needed to build the channelizer-math harness")
    so = str(tmp_path_factory.mktemp("chan_emul") / "libchan_emul.so")
    subprocess.run([nvcc, "-std=c++17", "-O2", "-shared", "-Xcompiler", "-fPIC", "-gencode",
                    "arch=compute_100a,code=sm_100a", "-o", so, EMUL_SRC], check=True)
    lib = C.CDLL(so)
    P = C.c_void_p
    lib.emul_chan.argtypes = [P, C.c_int, C.c_float, C.c_int64, C.c_uint64, P, C.c_int, C.c_int, C.c_int, P, C.c_int64, P,
                              C.c_int]
    lib.emul_chan.restype = C.c_int
    return lib


def emul_chan(lib, x, h, M, D, first=0, scale=1.0, fold=False, tb=0):
    """K10's outputs computed on the CPU, complex64 [M][n_out] (and the fold [n_out][M] with fold=True); tb > 0 folds
    each window in blocks of tb offsets, as the kernel's blocked mode does."""
    fmt = 1 if x.dtype == np.int16 else 0
    xv = np.ascontiguousarray(x)
    L = xv.size // 2 if fmt else xv.size
    hf = np.ascontiguousarray(h, np.float32)
    T = hf.size
    n_out = cr.out_count(L, T, D)
    out = np.zeros((M, n_out), np.complex64)
    fo = np.zeros((n_out, M), np.complex64) if fold else None
    rc = lib.emul_chan(xv.ctypes.data, fmt, np.float32(scale), L, first % (1 << 64), hf.ctypes.data, T, M, D,
                       out.ctypes.data, max(n_out, 1), fo.ctypes.data if fold else None, int(tb))
    assert rc == 0
    return (out, fo) if fold else out


@pytest.mark.parametrize("M", [16, 64])
@pytest.mark.parametrize("half", [True, False])
@pytest.mark.parametrize("first", FIRSTS)
@pytest.mark.parametrize("Tk", ["1", "M", "32M"])
def test_emul_matches_oracle(emul, M, half, first, Tk):
    D = M // 2 if half else M
    T = {"1": 1, "M": M, "32M": 32 * M}[Tk]
    first = M + 3 if first is None else first
    fmt = "ci16" if (M + T) % 2 else "cf32"
    rng = np.random.default_rng(M + 3 * T)
    h = rng.normal(size=T) / np.sqrt(T)
    x, scale = _x(T + 12 * D + 5, M * T, fmt)
    got = emul_chan(emul, x, h, M, D, first, scale)
    want = cr.channelize(x, h, M, D, first, scale)
    err = np.abs(got - want).max()
    assert err <= 1e-5 * cr.bound(h, x, scale), f"{err:.3e} vs bar {1e-5 * cr.bound(h, x, scale):.3e}"


@pytest.mark.parametrize("M,D", [(16, 8), (64, 64), (256, 128), (1024, 512), (4096, 2048)])
def test_emul_default_taps_larger_m(emul, M, D):
    """The FFT phases of every pass count (M up to 4096) with the default designs."""
    from sdr_iq_visualizer_b200 import ddc
    h = ddc.design_taps(M // 2, transition=0.5) if D == M // 2 else ddc.design_taps(M)
    x, scale = _x(h.size + 3 * D + 1, M)
    got = emul_chan(emul, x, h, M, D, 77, scale)
    want = cr.channelize(x, h, M, D, 77, scale)
    assert np.abs(got - want).max() <= 1e-5 * cr.bound(h, x, scale)


@pytest.mark.parametrize("M,D,T", [(16, 8, 81), (64, 32, 323), (64, 64, 2048)])
def test_emul_bit_identical_under_splits(emul, M, D, T):
    """Pieces cut at output boundaries with the T - D halo and their global first_sample give the outputs of one call."""
    rng = np.random.default_rng(T)
    h = rng.normal(size=T) / T
    x, _ = _x(T + 40 * D + 7, T)
    base = (1 << 40) + 5
    one = emul_chan(emul, x, h, M, D, base)
    n_out = one.shape[1]
    cuts = [0, 1, 7, n_out // 2 + 3, n_out - 1, n_out]
    parts = [emul_chan(emul, x[a * D: (b - 1) * D + T], h, M, D, base + a * D) for a, b in zip(cuts[:-1], cuts[1:])]
    assert np.array_equal(np.concatenate(parts, axis=1).view(np.uint32), one.view(np.uint32))


@pytest.mark.parametrize("M,D,T,tb", [(16, 16, 512, 48), (64, 64, 2048, 64), (64, 32, 2000, 448), (1024, 1024, 25697, 6144)])
def test_emul_blocked_fold_bit_identical(emul, M, D, T, tb):
    """Folding each window in blocks of tb offsets, partial sums carried from block to block (the kernel's mode for windows
    larger than shared memory), gives the bits of folding it at once."""
    rng = np.random.default_rng(T + tb)
    h = rng.normal(size=T) / np.sqrt(T)
    x, _ = _x(T + 6 * D + 1, T)
    whole, f_whole = emul_chan(emul, x, h, M, D, 12345, fold=True)
    blocked, f_blocked = emul_chan(emul, x, h, M, D, 12345, fold=True, tb=tb)
    assert np.array_equal(f_blocked.view(np.uint32), f_whole.view(np.uint32))
    assert np.array_equal(blocked.view(np.uint32), whole.view(np.uint32))


def test_emul_nan_poisons_covering_outputs(emul):
    M, D, T = 16, 8, 40
    x, _ = _x(400, 3)
    x[101] = np.nan
    y = emul_chan(emul, x, np.ones(T) / T, M, D, 5)
    m = np.arange(y.shape[1])
    covers = (m * D <= 101) & (101 <= m * D + T - 1)
    np.testing.assert_array_equal(np.isnan(y).all(axis=0), covers)   # every channel of a covering output
    assert not np.isnan(y[:, ~covers]).any()


# ----------------------------------------------------------------------------- host-side checks, no fallback
def _bare(M=64, D=32, T=33):
    from sdr_iq_visualizer_b200 import ddc
    p = ddc.Channelizer.__new__(ddc.Channelizer)
    p.sample_rate, p.n_channels, p.decim, p.taps = 61.44e6, M, D, np.ones(T) / T
    p.in_fmt, p.in_scale, p.device, p._h = 0, 1.0, 0, None
    return p


def test_python_side_argument_checks():
    from sdr_iq_visualizer_b200 import ddc
    p = _bare()
    assert p.out_count(32) == 0 and p.out_count(33) == 1 and p.out_count(33 + 64) == 3
    assert p.out_rate == 61.44e6 / 32
    f = p.channel_freqs(100e6)
    assert f.dtype == np.float64 and f.shape == (64,)
    assert f[32] == 100e6 and f[0] == 100e6 - 61.44e6 / 2 and f[33] - f[32] == 61.44e6 / 64
    x = np.zeros(200, np.complex64)
    with pytest.raises(ValueError, match="first_sample"):
        p.exec(x, first_sample=-1)
    with pytest.raises(ValueError, match="out"):
        p.exec(x, out=np.zeros((64, 4), np.complex64))      # n_out = 6
    with pytest.raises(ValueError, match="out"):
        p.exec(x, out=np.zeros((32, 6), np.complex64))
    with pytest.raises(ValueError, match="out"):
        p.exec(x, out=np.zeros((64, 6), np.complex128))
    for kw in (dict(n_channels=48), dict(n_channels=8), dict(n_channels=8192), dict(n_channels=64, decim=16),
               dict(n_channels=64, taps=np.ones(64 * 32 + 1)), dict(n_channels=64, taps=[]),
               dict(n_channels=64, in_fmt=7)):
        with pytest.raises(ValueError):
            ddc.Channelizer(1e6, **kw)


def test_default_designs():
    from sdr_iq_visualizer_b200 import ddc
    for M, T_half, T_crit in [(64, 323, 1607), (1024, 5141, 25697)]:
        assert ddc.design_taps(M // 2, transition=0.5).size == T_half
        assert ddc.design_taps(M).size == T_crit


def test_no_cpu_fallback():
    from sdr_iq_visualizer_b200 import _native as nat, ddc
    if nat.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(nat.SpectralError):
        ddc.Channelizer(1e6, 64)
