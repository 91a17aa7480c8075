"""CPU tests of the zoom DDC: the float64 reference against a brute-force loop, the default filter design against scipy,
the exact phase increment, K9's per-element math and summation order (csrc/spx_ddc_device.cuh, compiled for the host by
a harness of its own) against the reference, and the host-side checks that run before any device call."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from tests import ddc_ref as dr

EMUL_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emul", "ddc_emul.cu")


def _brute(x, h, D, inc, first):
    xc = dr.to_complex(x)
    T, L = len(h), xc.size
    M = (L - T) // D + 1 if L >= T else 0
    out = []
    for m in range(M):
        acc = 0j
        for k in range(T):
            n = m * D + T - 1 - k
            phi = ((first + n) * (inc % (1 << 64))) % (1 << 64)
            acc += h[k] * xc[n] * np.exp(-2j * np.pi * phi / 2.0 ** 64)
        out.append(acc)
    return np.array(out, np.complex128)


@pytest.mark.parametrize("L,T,D,inc,first", [(40, 7, 3, 123456789 << 32, 0),
                                             (30, 2, 5, -(1 << 61), 17),       # T < D, negative increment
                                             (12, 1, 1, 1 << 62, 0),           # T = 1, D = 1
                                             (5, 9, 2, 1 << 40, 0),            # L < T: no output
                                             (25, 5, 4, 0x9E3779B97F4A7C15 - (1 << 64), (1 << 63) - 10)])  # wraps
def test_ref_matches_brute_force(L, T, D, inc, first):
    rng = np.random.default_rng(L + T)
    x = (rng.normal(size=L) + 1j * rng.normal(size=L)).astype(np.complex64)
    h = rng.normal(size=T)
    got = dr.ddc(x, h, D, inc, first)
    want = _brute(x, h, D, inc, first)
    assert got.shape == want.shape == ((L - T) // D + 1 if L >= T else 0,)
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12)


def test_ref_phase_wraps_exactly():
    inc = 0x0123456789ABCDEF
    first = (1 << 63) + 5
    ph = dr.phases(4, first, inc)
    assert [int(v) for v in ph] == [((first + n) * inc) % (1 << 64) for n in range(4)]


# ----------------------------------------------------------------------------- default filter design
@pytest.mark.parametrize("D,T_want", [(2, 53), (8, 203), (64, 1607), (256, 6425)])
def test_design_taps_matches_scipy(D, T_want):
    signal = pytest.importorskip("scipy.signal")
    from sdr_iq_visualizer_b200 import ddc
    h = ddc.design_taps(D)
    T, beta = signal.kaiserord(80, 0.4 / D)
    T += 1 - T % 2
    assert h.size == T == T_want and beta == pytest.approx(7.857, abs=1e-3)
    assert (T, beta) == (ddc.kaiser_order(80, 0.4 / D)[0] + 1 - ddc.kaiser_order(80, 0.4 / D)[0] % 2,
                         ddc.kaiser_order(80, 0.4 / D)[1])
    np.testing.assert_allclose(h, signal.firwin(T, 1 / D, window=("kaiser", beta)), rtol=0, atol=1e-12)
    assert h.sum() == pytest.approx(1.0, abs=1e-14)
    # response: passband |f| <= 0.4 / D, stopband |f| >= 0.6 / D (cycles/sample)
    nf = 1 << 20 if D <= 64 else 1 << 22
    H = np.abs(np.fft.rfft(h, nf))
    f = np.arange(H.size) / nf
    with np.errstate(divide="ignore"):
        db = 20 * np.log10(H)
    pb = db[f <= 0.4 / D]
    assert np.abs(pb).max() <= 0.0011, f"passband ripple {np.abs(pb).max():.5f} dB"
    assert db[f >= 0.6 / D].max() <= -78.5


def test_design_taps_edges():
    from sdr_iq_visualizer_b200 import ddc
    np.testing.assert_array_equal(ddc.design_taps(1), [1.0])
    with pytest.raises(ValueError):
        ddc.design_taps(0)
    assert ddc.design_taps(400).size > ddc.MAX_TAPS     # one stage is not enough: cascade


# ----------------------------------------------------------------------------- phase increment
def test_phase_increment_exact():
    from sdr_iq_visualizer_b200 import ddc
    fs = 61.44e6
    inc, actual = ddc.phase_increment(7.3e6, fs)
    from fractions import Fraction
    assert inc == round(Fraction(7.3e6) / Fraction(fs) * (1 << 64))
    assert actual == pytest.approx(7.3e6, abs=fs / 2 ** 63)
    neg, a_neg = ddc.phase_increment(-7.3e6, fs)
    assert neg == -inc and a_neg == -actual
    assert ddc.phase_increment(0.0, fs) == (0, 0.0)
    assert ddc.phase_increment(fs / 2, fs) == (-(1 << 63), -fs / 2)
    assert ddc.phase_increment(-fs / 2, fs) == (-(1 << 63), -fs / 2)
    assert ddc.phase_increment(fs / 4, fs) == (1 << 62, fs / 4)
    with pytest.raises(ValueError):
        ddc.phase_increment(1.0, 0.0)


# ----------------------------------------------------------------------------- K9's math on the CPU
@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.fail("nvcc is needed to build the DDC-math harness")
    so = str(tmp_path_factory.mktemp("ddc_emul") / "libddc_emul.so")
    subprocess.run([nvcc, "-std=c++17", "-O2", "-shared", "-Xcompiler", "-fPIC", "-gencode",
                    "arch=compute_100a,code=sm_100a", "-o", so, EMUL_SRC], check=True)
    lib = C.CDLL(so)
    P = C.c_void_p
    lib.emul_cis.argtypes = [P, C.c_int64, P, P]
    lib.emul_ddc.argtypes = [P, C.c_int, C.c_float, C.c_int64, C.c_uint64, C.c_uint64, P, C.c_int, C.c_int, P]
    lib.emul_geom.argtypes = [C.c_int, P]
    return lib


def emul_ddc(lib, x, h, D, inc, first=0, scale=1.0):
    """K9's outputs computed on the CPU (x: complex64 or interleaved int16)."""
    fmt = 1 if x.dtype == np.int16 else 0
    xv = np.ascontiguousarray(x)
    L = xv.size // 2 if fmt else xv.size
    hf = np.ascontiguousarray(h, np.float32)
    T = hf.size
    M = (L - T) // D + 1 if L >= T else 0
    out = np.zeros(M, np.complex64)
    lib.emul_ddc(xv.ctypes.data, fmt, np.float32(scale), L, first % (1 << 64), int(inc) % (1 << 64), hf.ctypes.data, T, D,
                 out.ctypes.data)
    return out


def test_emul_cis(emul):
    rng = np.random.default_rng(3)
    ph = np.concatenate([rng.integers(0, 2 ** 63, 20000, dtype=np.uint64) * np.uint64(2),
                         np.array([0, 1 << 62, 1 << 63, 3 << 62, (1 << 64) - 1, (1 << 61) - 1, 1 << 61], np.uint64)])
    c = np.empty(ph.size, np.float32)
    s = np.empty(ph.size, np.float32)
    emul.emul_cis(ph.ctypes.data, ph.size, c.ctypes.data, s.ctypes.data)
    ang = 2 * np.pi * (ph.astype(np.float64) / 2.0 ** 64)
    assert np.abs(c - np.cos(ang)).max() < 3e-7 and np.abs(s - np.sin(ang)).max() < 3e-7
    assert c[-7] == 1.0 and s[-7] == 0.0      # phase 0: the identity, exactly


def test_emul_geometry(emul):
    g = np.zeros(4, np.int32)
    for D, want in [(1, (32, 1, 1, 8)), (4, (8, 1, 1, 8)), (64, (1, 2, 2, 4)), (256, (1, 8, 8, 1)), (3, (32, 3, 2, 4)),
                    (96, (1, 3, 2, 4))]:
        emul.emul_geom(D, g.ctypes.data)
        assert tuple(g) == want, D


@pytest.mark.parametrize("fmt", ["cf32", "ci16"])
@pytest.mark.parametrize("D,T", [(1, 1), (4, 33), (8, 203), (64, 1607), (3, 100), (1, 8192)])
def test_emul_matches_reference(emul, fmt, D, T):
    from sdr_iq_visualizer_b200 import ddc
    rng = np.random.default_rng(D * 1000 + T)
    L = T + 40 * D + 5
    xc = (rng.normal(size=L) + 1j * rng.normal(size=L)) * 0.3
    if fmt == "ci16":
        x = np.empty(2 * L, np.int16)
        x[0::2] = np.clip(np.rint(xc.real * 8000), -32768, 32767)
        x[1::2] = np.clip(np.rint(xc.imag * 8000), -32768, 32767)
        scale = 2.0 ** -15
    else:
        x, scale = xc.astype(np.complex64), 1.0
    h = ddc.design_taps(D) if T == ddc.design_taps(D).size else rng.normal(size=T) / T
    inc, _ = ddc.phase_increment(0.123456 * 61.44e6, 61.44e6)
    first = 123457
    got = emul_ddc(emul, x, h, D, inc, first, scale)
    want = dr.ddc(x, h, D, inc, first, scale)
    err = np.abs(got - want).max()
    assert err <= 1e-5 * dr.bound(h, x, scale), f"{err:.3e} vs bar {1e-5 * dr.bound(h, x, scale):.3e}"


def test_emul_exact_cases(emul):
    """h = [1], shift 0: x[::D] bit for bit; a NaN poisons only the outputs whose window covers it."""
    rng = np.random.default_rng(9)
    x = (rng.normal(size=101) + 1j * rng.normal(size=101)).astype(np.complex64)
    np.testing.assert_array_equal(emul_ddc(emul, x, [1.0], 4, 0), x[::4])
    x[50] = np.nan
    y = emul_ddc(emul, x, np.ones(7) / 7, 2, 1 << 60)
    bad = np.isnan(y)
    m = np.arange(y.size)
    np.testing.assert_array_equal(bad, (2 * m <= 50) & (50 <= 2 * m + 6))


# ----------------------------------------------------------------------------- host-side checks, no fallback
def _bare(D=4, T=9, fmt=0):
    from sdr_iq_visualizer_b200 import ddc
    p = ddc.DdcPlan.__new__(ddc.DdcPlan)
    p.sample_rate, p.decim, p.taps, p.in_fmt, p.in_scale, p.device, p._h = 1e6, D, np.ones(T) / T, fmt, 1.0, 0, None
    return p


def test_python_side_argument_checks():
    from sdr_iq_visualizer_b200 import ddc
    p = _bare()
    x = np.zeros(100, np.complex64)
    assert p.out_count(100) == 23 and p.out_count(8) == 0 and p.out_count(9) == 1
    with pytest.raises(ValueError, match="first_sample"):
        p.exec(x, first_sample=-1)
    with pytest.raises(ValueError, match="out"):
        p.exec(x, out=np.zeros(22, np.complex64))
    with pytest.raises(ValueError, match="out"):
        p.exec(x, out=np.zeros(23, np.complex128))
    for kw in (dict(decim=0), dict(decim=2, taps=np.ones(8193)), dict(decim=2, taps=[]), dict(decim=2, in_fmt=7)):
        with pytest.raises(ValueError):
            ddc.DdcPlan(1e6, 0.0, **kw)


def test_recording_zoom_checks(tmp_path):
    from sdr_iq_visualizer_b200 import sigmf_io
    base = sigmf_io.write_recording(str(tmp_path / "rec"), np.zeros(4096, np.complex64), 1e6, 100e6)
    with pytest.raises(ValueError, match="fs/2"):
        sigmf_io.process_recording(base, nfft=64, zoom=(100e6 + 0.6e6, 4))


def test_no_cpu_fallback(tmp_path):
    from sdr_iq_visualizer_b200 import _native as nat, ddc, sigmf_io
    if nat.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(nat.SpectralError):
        ddc.DdcPlan(1e6, 1e5, 4)
    base = sigmf_io.write_recording(str(tmp_path / "rec"), np.zeros(4096, np.complex64), 1e6, 0.0)
    with pytest.raises(nat.SpectralError):
        sigmf_io.process_recording(base, nfft=64, zoom=(1e5, 4))
