"""CPU tests of the pooled spectrogram: the float64 reference against a brute-force loop, the kernels' per-element math
(csrc/spx_pool_device.cuh, compiled for the host by a harness of its own), the frequency axis, the dashboard payload, the
overview's choice of K and B, and the host-side checks that run before any device call.  No CPU fallback exists."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import spectral_ref as sref
from tests import pool_ref as pr

EMUL_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emul", "pool_emul.cu")


def _brute(P, K, B, mode, S=1):
    P = np.asarray(P, np.float64)
    N = P.shape[-1]
    P = P.reshape(S, -1, N)
    F = P.shape[1]
    G, Cn = -(-F // K), N // B
    out = np.empty((S, G, Cn))
    for s in range(S):
        for g in range(G):
            for c in range(Cn):
                vals = [P[s, f, j] for f in range(g * K, min((g + 1) * K, F)) for j in range(c * B, (c + 1) * B)]
                if mode == "mean":
                    out[s, g, c] = sum(vals) / len(vals)
                else:
                    ok = [v for v in vals if not np.isnan(v)]
                    out[s, g, c] = max(ok) if ok else np.nan
    return out


@pytest.mark.parametrize("mode", ["mean", "max"])
@pytest.mark.parametrize("F,N,K,B,S", [(10, 12, 3, 4, 1),     # partial last row (1 frame)
                                       (5, 8, 7, 2, 2),       # K > F: one partial row
                                       (9, 6, 2, 6, 1),       # B = N: a total-power strip
                                       (4, 5, 1, 1, 3),       # K = B = 1
                                       (0, 8, 3, 2, 2)])      # F = 0: no rows
def test_ref_matches_brute_force(mode, F, N, K, B, S):
    rng = np.random.default_rng(F * 100 + N)
    P = rng.exponential(1.0, (S * F, N))
    got = pr.pool_power(P, K, B, mode, S)
    assert got.shape == (S, -(-F // K), N // B)
    np.testing.assert_allclose(got, _brute(P, K, B, mode, S), rtol=1e-13)


def test_ref_nan_rules():
    P = np.ones((4, 4))
    P[1, 0] = np.nan            # one NaN frame value in cell (0, 0)
    P[2:4, 2:4] = np.nan        # cell (1, 1) all NaN
    mean = pr.pool_power(P, 2, 2, "mean")[0]
    mx = pr.pool_power(P, 2, 2, "max")[0]
    assert np.isnan(mean[0, 0]) and mean[0, 1] == 1.0 and np.isnan(mean[1, 1])
    assert mx[0, 0] == 1.0 and np.isnan(mx[1, 1])
    d = pr.pool_db(P, 2, 2, "max")[0]
    assert d[1, 1] == -np.inf and d[0, 0] == pytest.approx(20 * np.log10(1 + pr.EPS))
    assert np.isnan(pr.pool_db(P, 2, 2, "mean")[0, 0, 0])


def test_ref_db_rows_form():
    """K = B = 1 gives back the rows; max takes the rows' own maximum bit for bit; mean recovers the power."""
    rng = np.random.default_rng(1)
    P = rng.exponential(1e3, (12, 8))
    d32 = (20 * np.log10(np.sqrt(P) + pr.EPS)).astype(np.float32)
    np.testing.assert_array_equal(pr.pool_db_rows(d32, 1, 1, "max")[0].astype(np.float32), d32)
    np.testing.assert_allclose(pr.pool_db_rows(d32, 1, 1, "mean")[0], d32, atol=1e-5)
    mx = pr.pool_db_rows(d32, 5, 4, "max")[0]
    assert mx[0, 1] == d32[:5, 4:8].max() and mx[2, 0] == d32[10:, :4].max()
    np.testing.assert_allclose(pr.pool_db_rows(d32, 5, 4, "mean"), pr.pool_db(P, 5, 4, "mean"), atol=1e-4)
    nan_rows = d32.copy()
    nan_rows[:5] = np.nan
    assert (pr.pool_db_rows(nan_rows, 5, 4, "max")[0, 0] == -np.inf).all()


# ----------------------------------------------------------------------------- the kernels' math on the CPU
@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.fail("nvcc is needed to build the pooled-math harness")
    so = str(tmp_path_factory.mktemp("pool_emul") / "libpool_emul.so")
    subprocess.run([nvcc, "-std=c++17", "-O2", "-shared", "-Xcompiler", "-fPIC", "-gencode",
                    "arch=compute_100a,code=sm_100a", "-o", so, EMUL_SRC], check=True)
    lib = C.CDLL(so)
    P = C.c_void_p
    lib.emul_db_to_power.argtypes = [P, C.c_int64, C.c_float, P]
    lib.emul_mean_db.argtypes = [P, P, C.c_int64, C.c_int32, C.c_float, P]
    lib.emul_max_db.argtypes = [P, C.c_int64, P]
    lib.emul_level.argtypes = [P, C.c_int64, C.c_float, C.c_float, P]
    lib.emul_row_of.restype = C.c_int64
    lib.emul_row_of.argtypes = [C.c_int64, C.c_int64]
    lib.emul_col_of.argtypes = [C.c_int32, C.c_int32]
    lib.emul_row_frames.restype = C.c_int64
    lib.emul_row_frames.argtypes = [C.c_int64, C.c_int64, C.c_int64]
    return lib


def test_device_math_db_to_power(emul):
    d = np.concatenate([np.linspace(-260, 160, 5001), [np.nan, np.inf, -np.inf]]).astype(np.float32)
    out = np.empty_like(d)
    emul.emul_db_to_power(d.ctypes.data, d.size, np.float32(1e-12), out.ctypes.data)
    want = pr.db_to_power(d)
    fin = np.isfinite(d) & (want > 1e-18)   # amplitude >= 1000 eps: away from the cancellation against eps
    # float32 exponent: d / 20 is rounded to half an ulp, 2 ln(10) |d / 20| 2^-24 relative in power (3.6e-6 at 260 dB)
    np.testing.assert_allclose(out[fin], want[fin], rtol=5e-6)
    assert (out[d < -241] == 0).all()                 # below 20 log10(eps): clipped at zero power
    assert np.isnan(out[-3]) and out[-2] == np.inf and out[-1] == 0


def test_device_math_final_db_and_levels(emul):
    rng = np.random.default_rng(4)
    n = 4000
    s = rng.exponential(1e4, n) * rng.integers(1, 50, n)
    nf = rng.integers(1, 600, n).astype(np.int64)
    B = 4
    got = np.empty(n, np.float32)
    emul.emul_mean_db(s.ctypes.data, nf.ctypes.data, n, B, np.float32(1e-12), got.ctypes.data)
    want = (20 * np.log10(np.sqrt(s / (nf * B)) + pr.EPS)).astype(np.float32)
    np.testing.assert_array_equal(got, want)
    acc = np.concatenate([rng.normal(0, 80, 100).astype(np.float32).astype(np.float64), [-np.inf]])
    mx = np.empty(acc.size, np.float32)
    emul.emul_max_db(acc.ctypes.data, acc.size, mx.ctypes.data)
    np.testing.assert_array_equal(mx, acc.astype(np.float32))
    # levels: bit-exact against waterfall_u8 of the same float32 dB, ties, clips, NaN and infinities included
    vmin, vmax = -47.5, 61.25
    db = np.concatenate([rng.uniform(-80, 90, 20000), vmin + np.arange(257) * (vmax - vmin) / 256,
                         [np.nan, np.inf, -np.inf, vmin, vmax]]).astype(np.float32)
    q = np.empty(db.size, np.uint8)
    emul.emul_level(db.ctypes.data, db.size, np.float32(vmin), np.float32(vmax), q.ctypes.data)
    np.testing.assert_array_equal(q, sref.waterfall_u8(db, vmin, vmax))


def test_device_math_indices(emul):
    K, F = 600, 59_997
    assert emul.emul_row_of(599, K) == 0 and emul.emul_row_of(600, K) == 1 and emul.emul_row_of(F - 1, K) == 99
    assert emul.emul_row_frames(0, K, F) == 600 and emul.emul_row_frames(99, K, F) == 597
    assert emul.emul_row_frames(0, 10, 3) == 3
    assert emul.emul_col_of(7, 8) == 0 and emul.emul_col_of(8, 8) == 1 and emul.emul_col_of(999, 8) == 124


# ----------------------------------------------------------------------------- axes, payload, overview shape
def test_pooled_freq_axis():
    from sdr_iq_visualizer_b200 import spectral
    fs, fc = 61.44e6, 2.4e9
    f = spectral.freq_axis(4096, fs, fc)
    p = spectral.pooled_freq_axis(4096, 4, fs, fc)
    assert p.shape == (1024,)
    np.testing.assert_allclose(p, f.reshape(1024, 4).mean(axis=1))
    np.testing.assert_array_equal(spectral.pooled_freq_axis(4096, 1, fs, fc), f)
    assert spectral.pooled_freq_axis(1000, 1000, 1e6)[0] == pytest.approx(f.mean() * 0 + spectral.freq_axis(1000, 1e6).mean())
    with pytest.raises(ValueError):
        spectral.pooled_freq_axis(1000, 3, 1e6)


def test_spectrogram_payload():
    from sdr_iq_visualizer_b200 import views
    G, Cn, K, hop, fs = 5, 8, 600, 1024, 61.44e6
    db = np.linspace(-90, 10, G * Cn, dtype=np.float32).reshape(G, Cn)
    p = views.spectrogram_payload(db, K, hop, fs, freqs_mhz=np.arange(Cn) * 0.1, vmin=-100.0, vmax=0.0)
    assert p["z"] is db or np.array_equal(p["z"], db)
    np.testing.assert_allclose(p["y"], np.arange(G) * K * hop / fs)
    assert p["zmin"] == -100.0 and p["zmax"] == 0.0 and len(p["colorscale"]) > 2
    q = views.spectrogram_payload(np.zeros((1, G, Cn), np.uint8), K, hop, fs)
    assert q["z"].shape == (G, Cn) and q["zmin"] == 0 and q["zmax"] == 255
    with pytest.raises(ValueError, match="streams"):
        views.spectrogram_payload(np.zeros((2, G, Cn), np.float32), K, hop, fs)
    with pytest.raises(ValueError):
        views.spectrogram_payload(np.zeros(Cn, np.float32), K, hop, fs)


def test_overview_pooling_choice():
    from sdr_iq_visualizer_b200 import sigmf_io
    assert sigmf_io.overview_pooling(59_997, 4096, 100, 1024) == (600, 4)
    assert sigmf_io.overview_pooling(8191, 65536, 1024, 1024) == (8, 64)
    assert sigmf_io.overview_pooling(10, 1000, 3, 300) == (4, 2)       # 1000 / 300 = 3.3 -> largest divisor <= 3 is 2
    assert sigmf_io.overview_pooling(10, 1000, 20, 5000) == (1, 1)     # more columns than bins
    assert sigmf_io.overview_pooling(0, 64, 10, 10) == (1, 4)
    with pytest.raises(ValueError):
        sigmf_io.overview_pooling(10, 64, 0, 10)


# ----------------------------------------------------------------------------- host-side checks, no fallback
def _bare_plan(nfft=64, hop=64):
    """A SpectralPlan object without a native plan: enough for the checks stft() makes before calling libspx."""
    from sdr_iq_visualizer_b200 import spectral
    pl = spectral.SpectralPlan.__new__(spectral.SpectralPlan)
    pl.nfft, pl.hop, pl.in_fmt, pl.device, pl._h = nfft, hop, spectral.FMT_CF32, 0, None
    return pl


def test_python_side_argument_checks():
    pl = _bare_plan()
    x = np.zeros(64 * 4, np.complex64)
    for bad in [(0, 4, "mean"), (2, 0, "mean"), (2, 3, "mean"), (2, 4, "median"), (2, 4), None.__class__]:
        with pytest.raises(ValueError):
            pl.stft(x, pool=bad)
    with pytest.raises(ValueError, match="persistence"):
        pl.stft(x, pool=(2, 4, "mean"), persistence=True, vmin=-100.0, vmax=0.0)
    with pytest.raises(ValueError, match="_time"):
        pl.stft(x, pool=(2, 4, "max"), _time=(1, 1, False))
    with pytest.raises(ValueError, match="pool_first_frame"):
        pl.stft(x, pool=(2, 4, "max"), pool_first_frame=-1)
    with pytest.raises(ValueError, match="pool_acc"):   # F = 4, K = 2: [1, 2, 16] float64 expected
        pl.stft(x, pool=(2, 4, "mean"), pool_acc=np.zeros((1, 2, 15)))
    with pytest.raises(ValueError, match="pool_acc"):
        pl.stft(x, pool=(2, 4, "mean"), pool_acc=np.zeros((1, 2, 16), np.float32))
    with pytest.raises(ValueError, match="pool_acc"):
        pl.stft(x, pool=(2, 4, "mean"), pool_acc=False)
    with pytest.raises(ValueError, match="pool_acc"):
        pl.pool_finalize(np.zeros((1, 3, 16)), 4, 2, 4, "mean")      # ceil(4 / 2) = 2 rows, not 3


def _no_gpu():
    from sdr_iq_visualizer_b200 import _native as nat
    if nat.device_count() > 0:
        pytest.skip("a GPU is present")
    return nat


def test_no_cpu_fallback(tmp_path):
    nat = _no_gpu()
    from sdr_iq_visualizer_b200 import sigmf_io, spectral
    with pytest.raises(nat.SpectralError):
        spectral.SpectralPlan(1024).stft(np.zeros(4096, np.complex64), pool=(2, 4, "mean"))
    base = sigmf_io.write_recording(str(tmp_path / "rec"), np.zeros(4096, np.complex64), 1e6, 0.0)
    with pytest.raises(nat.SpectralError):
        sigmf_io.process_recording(base, nfft=256, overview=(4, 16))
    with pytest.raises(nat.SpectralError):   # shorter than one frame: still no fallback
        sigmf_io.process_recording(base, nfft=8192, overview=(4, 16))
