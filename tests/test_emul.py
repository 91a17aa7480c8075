"""CPU re-execution of the CUDA kernel's per-thread code (tests/emul) against the oracle.
Checks the Stockham index maps, padding, twiddle tables, fused epilogue and chunked accumulation
for every supported shared-memory FFT size -- without a GPU.  The emulator is test infrastructure;
the product never links it."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import spectral_ref as sref
from tests import parity

HERE = os.path.dirname(os.path.abspath(__file__))
EMUL_DIR = os.path.join(HERE, "emul")
EMUL_SO = os.path.join(EMUL_DIR, "libspx_emul.so")


@pytest.fixture(scope="session")
def emul():
    src = os.path.join(EMUL_DIR, "spx_emul.cu")
    csrc = os.path.join(os.path.dirname(HERE), "sdr_iq_visualizer_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in ("spx_fft_core.cuh", "spx_stft_device.cuh", "spx_stft2_device.cuh", "spx_big2_device.cuh", "spx_tables.h")]
    if not os.path.exists(EMUL_SO) or any(os.path.getmtime(d) > os.path.getmtime(EMUL_SO) for d in deps):
        nvcc = "nvcc" if subprocess.run(["which", "nvcc"], capture_output=True).returncode == 0 else "/usr/local/cuda/bin/nvcc"
        subprocess.run([nvcc, "-std=c++17", "-O2", "-shared", "-Xcompiler", "-fPIC", "-gencode",
                        "arch=compute_100a,code=sm_100a", "-o", EMUL_SO, src], check=True, cwd=EMUL_DIR)
    lib = C.CDLL(EMUL_SO)
    lib.spx_emul_stft.argtypes = [C.c_int] * 3 + [C.c_void_p, C.c_longlong, C.c_int, C.c_longlong, C.c_int, C.c_void_p,
                                                  C.c_float, C.c_float, C.c_float, C.c_int] + [C.c_void_p] * 5
    lib.spx_emul_plan.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    return lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def run_emul(lib, x, nfft, hop, kind, fmt=0, scale=1.0, tw_mode=0, n_streams=1, fpc=3, vmin=-60.0, vmax=60.0,
             eps=1e-12):
    L = (x.size // 2 if fmt == 1 else x.size) // n_streams
    F = sref.frame_count(L, nfft, hop)
    w = None
    if sref.window_id(kind) != 0 or scale != 1.0:
        w = (sref.window(kind, nfft) * scale).astype(np.float32)
    out = dict(db=np.zeros((n_streams * F, nfft), np.float32), wf=np.zeros((n_streams * F, nfft), np.uint8),
               spec=np.zeros((n_streams * F, nfft, 2), np.float32), welch=np.zeros((n_streams, nfft), np.float64),
               maxhold=np.zeros((n_streams, nfft), np.float32))
    rc = lib.spx_emul_stft(nfft, fmt, tw_mode, _p(x), L, n_streams, L, hop, _p(w), eps, vmin, vmax, fpc, _p(out["db"]),
                           _p(out["wf"]), _p(out["spec"]), _p(out["welch"]), _p(out["maxhold"]))
    assert rc == 0
    out["F"] = F
    out["win64"] = None if w is None else sref.window(kind, nfft) * scale
    return out


def oracle_power(x, nfft, hop, win64, fmt=0, n_streams=1):
    """float64 oracle with the float64 window of the reference (np.hanning via mlab, process_sigmf_data.py:188); the
    kernel's float32 window table is NOT fed back into the oracle."""
    xs = sref.as_complex128(x, fmt).reshape(n_streams, -1)
    w = np.ones(nfft) if win64 is None else win64
    rows = []
    for s in range(n_streams):
        fr = sref.frames(xs[s], nfft, hop)
        rows.append(sref.shift_bins(np.fft.fft(fr * w, axis=1)))
    return np.concatenate(rows, axis=0)


@pytest.mark.parametrize("nfft", [16, 32, 64, 128, 256, 512, 1024, 2048, 4096, 8192])
def test_plan_factorisation(emul, nfft):
    rad = (C.c_int * 5)()
    tws = C.c_int()
    p = emul.spx_emul_plan(nfft, rad, C.byref(tws))
    r = list(rad)[:p]
    assert r[0] == 16 and all(v in (2, 4, 8, 16) for v in r) and int(np.prod(r)) == nfft
    assert all(v == 0 for v in list(rad)[p:])


@pytest.mark.parametrize("nfft,hop,kind", [(16, 16, "rect"), (32, 8, "hann"), (64, 16, "blackman"), (128, 128, "hann"),
                                           (256, 64, "hann"), (512, 256, "blackman"), (1024, 512, "hann"),
                                           (2048, 1024, "hann"), (4096, 1024, "hann"), (8192, 4096, "hann")])
def test_emul_cf32_parity(emul, nfft, hop, kind):
    L = nfft + hop * 7 + 5  # ragged tail is dropped
    x = sref.synth_iq(L, seed=nfft + 1).astype(np.complex64)
    o = run_emul(emul, x, nfft, hop, kind)
    X = oracle_power(x, nfft, hop, o["win64"])
    P = X.real**2 + X.imag**2
    assert o["F"] == 8
    got = o["spec"][..., 0] + 1j * o["spec"][..., 1]
    assert np.abs(got - X).max() <= 4e-6 * np.sqrt(P.mean())
    parity.check_db_rows(o["db"], P, what=f"N={nfft}")
    parity.check_power(o["welch"][0], P.sum(axis=0), what="welch")
    parity.check_power(o["maxhold"][0], P.max(axis=0), what="maxhold")
    parity.check_u8(o["wf"], sref.amplitude_db(X), -60.0, 60.0, what="u8")


def test_emul_tone_lands_in_shifted_bin(emul):
    """fftshift order is an integer permutation: must be exact (streamer.py:119)."""
    n = 4096
    for k in (0, 1, 100, 2047, 2048, 4095):
        x = np.exp(2j * np.pi * k * np.arange(n) / n).astype(np.complex64)
        o = run_emul(emul, x, n, n, "rect")
        assert int(np.argmax(o["db"][0])) == (k + n // 2) % n


def test_emul_ci16_and_scale(emul):
    n, hop = 4096, 1024
    x = sref.to_ci16(sref.synth_iq(n + 9 * hop, seed=2))
    for scale in (1.0, 2.0**-15):
        o = run_emul(emul, x, n, hop, "hann", fmt=1, scale=scale, vmin=-40.0, vmax=120.0)
        X = oracle_power(x, n, hop, o["win64"], fmt=1)
        P = X.real**2 + X.imag**2
        parity.check_db_rows(o["db"], P, what=f"ci16 scale={scale}")
        parity.check_power(o["welch"][0], P.sum(axis=0), what="welch")


def test_emul_register_twiddles_match_table(emul):
    n, hop = 4096, 2048
    x = sref.synth_iq(n + 3 * hop, seed=4).astype(np.complex64)
    a = run_emul(emul, x, n, hop, "hann", tw_mode=0)
    b = run_emul(emul, x, n, hop, "hann", tw_mode=1)
    X = oracle_power(x, n, hop, a["win64"])
    P = X.real**2 + X.imag**2
    parity.check_db_rows(b["db"], P, what="TW_REG")
    assert np.abs(a["spec"] - b["spec"]).max() <= 2e-6 * np.sqrt(P.mean())


def test_emul_staged_input_matches_direct(emul):
    """pass 0 fed from the staging buffer (TMA path) == pass 0 fed from global memory."""
    n, hop = 4096, 1024
    x = sref.to_ci16(sref.synth_iq(n + 5 * hop, seed=6))
    a = run_emul(emul, x, n, hop, "hann", fmt=1, tw_mode=0)
    b = run_emul(emul, x, n, hop, "hann", fmt=1, tw_mode=0x10)
    np.testing.assert_array_equal(a["spec"], b["spec"])
    xc = sref.synth_iq(n + 5 * hop, seed=6).astype(np.complex64)
    a = run_emul(emul, xc, n, hop, "blackman", tw_mode=1)
    b = run_emul(emul, xc, n, hop, "blackman", tw_mode=0x11)
    np.testing.assert_array_equal(a["db"], b["db"])


def test_emul_multistream_chunking(emul):
    """chunks never cross a stream; accumulators are per stream (C4 layout)."""
    n, hop, S = 1024, 512, 3
    L = n + 10 * hop
    xs = np.concatenate([sref.synth_iq(L, seed=10 + s, snr_db=5 * (s + 1)) for s in range(S)]).astype(np.complex64)
    for fpc in (1, 4, 11, 64):
        o = run_emul(emul, xs, n, hop, "hann", n_streams=S, fpc=fpc)
        X = oracle_power(xs, n, hop, o["win64"], n_streams=S)
        P = (X.real**2 + X.imag**2).reshape(S, -1, n)
        for s in range(S):
            parity.check_power(o["welch"][s], P[s].sum(axis=0), what=f"welch s={s} fpc={fpc}")
            parity.check_power(o["maxhold"][s], P[s].max(axis=0), what=f"maxhold s={s}")


def test_emul_zero_input_is_minus_240_db(emul):
    o = run_emul(emul, np.zeros(4096, np.complex64), 4096, 4096, "rect")
    assert np.abs(o["db"] + 240.0).max() < 1e-3  # 20*log10(0 + 1e-12) (streamer.py:121)
    assert np.all(o["wf"] == 0)


# ----------------------------------------------------------------------------- K1v2: warp-local first exchange
K2 = 0x20


@pytest.mark.parametrize("nfft,hop,kind,fmt", [(4096, 1024, "hann", 0), (4096, 4096, "rect", 0), (4096, 2048, "blackman", 1),
                                               (2048, 1024, "hann", 0), (2048, 512, "hann", 1), (1024, 512, "hann", 0),
                                               (1024, 256, "blackman", 1)])
def test_emul_k1v2_parity(emul, nfft, hop, kind, fmt):
    """Phases of spx_stft2_device.cuh (swizzled staging, warp-local 16x16 tile, double-buffered column exchange) vs the
    float64 oracle: same bar as K1."""
    L = nfft + hop * 9 + 3
    xc = sref.synth_iq(L, seed=nfft + hop)
    x = sref.to_ci16(xc) if fmt else xc.astype(np.complex64)
    vmin, vmax = (0.0, 130.0) if fmt else (-60.0, 60.0)
    o = run_emul(emul, x, nfft, hop, kind, fmt=fmt, tw_mode=K2, vmin=vmin, vmax=vmax)
    X = oracle_power(x, nfft, hop, o["win64"], fmt=fmt)
    P = X.real**2 + X.imag**2
    assert o["F"] == 10
    got = o["spec"][..., 0] + 1j * o["spec"][..., 1]
    # the worst bin is the CW tone (|X| ~ 40 x rms): 4.2e-6 * rms there is 1e-7 of the bin; K1 with register twiddle
    # bases gives the identical figure on these inputs (same arithmetic, different data flow)
    assert np.abs(got - X).max() <= 5e-6 * np.sqrt(P.mean())
    if nfft == 4096:
        ref = run_emul(emul, x, nfft, hop, kind, fmt=fmt, tw_mode=1, vmin=vmin, vmax=vmax)
        np.testing.assert_array_equal(o["spec"], ref["spec"])      # bit-identical to K1 (TW_REG): only the data flow differs
        np.testing.assert_array_equal(o["wf"], ref["wf"])
    parity.check_db_rows(o["db"], P, what=f"K1v2 N={nfft}")
    parity.check_power(o["welch"][0], P.sum(axis=0), what="K1v2 welch")
    parity.check_power(o["maxhold"][0], P.max(axis=0), what="K1v2 maxhold")
    parity.check_u8(o["wf"], sref.amplitude_db(X), vmin, vmax, what="K1v2 u8")


@pytest.mark.parametrize("nfft,hop,kind,fmt", [(4096, 1024, "hann", 1), (4096, 4096, "rect", 0), (2048, 1024, "hann", 0), (1024, 512, "blackman", 0)])
def test_emul_k1v2_fma_form_dft(emul, nfft, hop, kind, fmt):
    """dft16_fma (no stand-alone W_16 multiplies, 144 instead of 160 operations): same parity bar, and its error against
    the float64 oracle is no worse than the plain radix-16 butterfly's.  The colormap index on the FMA pipe (TUNE_QFMA)
    is bit for bit the F2I one."""
    L = nfft + hop * 9 + 3
    xc = sref.synth_iq(L, seed=nfft + hop + 1)
    x = sref.to_ci16(xc) if fmt else xc.astype(np.complex64)
    vmin, vmax = (0.0, 130.0) if fmt else (-60.0, 60.0)
    o = run_emul(emul, x, nfft, hop, kind, fmt=fmt, tw_mode=K2 | 0x40, vmin=vmin, vmax=vmax)
    ref = run_emul(emul, x, nfft, hop, kind, fmt=fmt, tw_mode=K2, vmin=vmin, vmax=vmax)
    f2i = run_emul(emul, x, nfft, hop, kind, fmt=fmt, tw_mode=K2 | 0x80, vmin=vmin, vmax=vmax)
    np.testing.assert_array_equal(o["wf"], f2i["wf"])
    X = oracle_power(x, nfft, hop, o["win64"], fmt=fmt)
    P = X.real**2 + X.imag**2
    err = lambda r: np.sqrt((np.abs(r["spec"][..., 0] + 1j * r["spec"][..., 1] - X) ** 2).mean() / P.mean())
    assert err(o) <= 1.15 * err(ref) and err(o) < 2.5e-7
    parity.check_db_rows(o["db"], P, what=f"K1v2 fma N={nfft}")
    parity.check_power(o["welch"][0], P.sum(axis=0), what="K1v2 fma welch")
    parity.check_u8(o["wf"], sref.amplitude_db(X), vmin, vmax, what="K1v2 fma u8")


def test_emul_k1v2_tone_bins_and_multistream(emul):
    n = 4096
    for k in (0, 1, 17, 255, 256, 2047, 2048, 4095):        # integer permutation: exact (streamer.py:119)
        x = np.exp(2j * np.pi * k * np.arange(n) / n).astype(np.complex64)
        o = run_emul(emul, x, n, n, "rect", tw_mode=K2)
        assert int(np.argmax(o["db"][0])) == (k + n // 2) % n
    S, hop = 3, 1024
    L = n + 6 * hop
    xs = np.concatenate([sref.synth_iq(L, seed=20 + s, snr_db=5 * (s + 1)) for s in range(S)]).astype(np.complex64)
    o = run_emul(emul, xs, n, hop, "hann", n_streams=S, fpc=4, tw_mode=K2)
    X = oracle_power(xs, n, hop, o["win64"], n_streams=S)
    P = (X.real**2 + X.imag**2).reshape(S, -1, n)
    for s in range(S):
        parity.check_power(o["welch"][s], P[s].sum(axis=0), what=f"K1v2 welch s={s}")


# ----------------------------------------------------------------------------- K2v2: single-kernel 65536-point STFT
@pytest.mark.parametrize("tune", [0, 1])
def test_emul_big2_roles(emul, tune):
    """Roles A / B of spx_big2_device.cuh (column tiles -> twiddle -> scratch -> row tiles -> epilogue) against the
    float64 oracle on three overlapped 65536-point frames: uint8 rows, Welch sum, max-hold; a tone lands in its bin."""
    n, hop = 65536, 32768
    emul.spx_emul_big2.argtypes = [C.c_void_p, C.c_longlong, C.c_int, C.c_void_p] + [C.c_float] * 3 + [C.c_int] + [C.c_void_p] * 3
    L = n + 2 * hop + 100
    x = sref.synth_iq(L, seed=65, tone_cycles_per_sample=20000.37 / 65536).astype(np.complex64)
    w64 = sref.window("hann", n)
    w32 = w64.astype(np.float32)
    F = sref.frame_count(L, n, hop)
    wf = np.zeros((F, n), np.uint8)
    welch = np.zeros(n, np.float64)
    mh = np.zeros(n, np.float32)
    vmin, vmax = -20.0, 110.0
    assert emul.spx_emul_big2(_p(x), L, hop, _p(w32), 1e-12, vmin, vmax, tune, _p(wf), _p(welch), _p(mh)) == 0
    X = sref.shift_bins(sref.stft(sref.as_complex128(x), n, hop, "hann"))
    P = X.real**2 + X.imag**2
    assert F == 3 and X.shape == (3, n)
    parity.check_u8(wf, sref.amplitude_db(X), vmin, vmax, what=f"K2v2 u8 tune={tune}")
    parity.check_power(welch, P.sum(axis=0), what="K2v2 welch")
    parity.check_power(mh, P.max(axis=0), what="K2v2 maxhold")
    k = 12345
    tone = np.exp(2j * np.pi * k * np.arange(n) / n).astype(np.complex64)
    mh[:] = 0
    assert emul.spx_emul_big2(_p(tone), n, n, None, 1e-12, vmin, vmax, tune, None, None, _p(mh)) == 0
    assert int(np.argmax(mh)) == (k + n // 2) % n and abs(mh.max() / float(n) ** 2 - 1) < 1e-5


def test_emul_big2_ci16_column_tiles(emul):
    """K2v2 with int16 input: the {64 B x 256 rows} tile under CU_TENSOR_MAP_SWIZZLE_64B, int16 -> float, window * scale, then
    the same roles as cf32 -- against the float64 oracle on three overlapped 65536-point frames (SigMF scale 2^-15)."""
    n, hop = 65536, 32768
    emul.spx_emul_big2_ci16.argtypes = [C.c_void_p, C.c_longlong, C.c_int, C.c_void_p] + [C.c_float] * 3 + [C.c_void_p] * 3
    L = n + 2 * hop + 100
    raw = sref.to_ci16(sref.synth_iq(L, seed=66, tone_cycles_per_sample=20000.37 / 65536))
    scale = 2.0 ** -15
    w32 = (sref.window("hann", n) * scale).astype(np.float32)
    F = sref.frame_count(L, n, hop)
    wf = np.zeros((F, n), np.uint8)
    welch = np.zeros(n, np.float64)
    mh = np.zeros(n, np.float32)
    vmin, vmax = -80.0, 40.0
    assert emul.spx_emul_big2_ci16(_p(raw), L, hop, _p(w32), 1e-12, vmin, vmax, _p(wf), _p(welch), _p(mh)) == 0
    X = sref.shift_bins(sref.stft(sref.unpack_ci16(raw, scale), n, hop, "hann"))
    P = X.real**2 + X.imag**2
    parity.check_u8(wf, sref.amplitude_db(X), vmin, vmax, what="K2v2 ci16 u8")
    parity.check_power(welch, P.sum(axis=0), what="K2v2 ci16 welch")
    parity.check_power(mh, P.max(axis=0), what="K2v2 ci16 maxhold")
