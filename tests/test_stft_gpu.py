"""GPU parity tests of the fused STFT path (K1) through the C ABI, against the float64 oracle and
the golden vectors generated from the reference.  Run on the B200 box: pytest -m gpu."""
import numpy as np
import pytest

from oracle import spectral_ref as sref
from tests import parity

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sp():
    from sdr_iq_visualizer_b200 import spectral
    from sdr_iq_visualizer_b200 import _native
    assert _native.device_count() > 0, "GPU tests need a CUDA device (no CPU fallback exists)"
    return spectral


def oracle_rows(x, nfft, hop, kind, fmt=0, scale=1.0, n_streams=1):
    xs = sref.as_complex128(x, fmt).reshape(n_streams, -1)
    w = sref.window(kind, nfft) * scale   # float64 window, as the reference's np.hanning (process_sigmf_data.py:188)
    out = []
    for s in range(n_streams):
        fr = sref.frames(xs[s], nfft, hop)
        for i in range(0, fr.shape[0], 1024):
            out.append(sref.shift_bins(np.fft.fft(fr[i:i + 1024] * w, axis=1)))
    return np.concatenate(out, axis=0) if out else np.zeros((0, nfft), complex)


def test_stream_frames_match_reference_golden(sp, golden_stream):
    """spectral.stream_frame == reference _stream_data outputs (streamer.py:119-121).  The drop-in runs the float64 kernel
    for these buffer sizes: every bin, above or below the noise floor, within 1e-9 dB of what the reference produced
    (the north_star bar is 1e-3 dB above the floor, 1e-4 relative below it)."""
    z, meta = golden_stream
    worst = 0.0
    for m in meta:
        k = m["key"]
        f, p = sp.stream_frame(z[k + "_samples"], m["sample_rate"], m["center_freq"])
        assert f.dtype == np.float64 and p.dtype == np.float64 and p.shape == (m["n"],)
        np.testing.assert_array_equal(f, z[k + "_freqs"])           # integer permutation + exact axis
        ref = z[k + "_power_db"]
        if np.all(ref == -240.0):
            np.testing.assert_array_equal(p, ref)
            continue
        # bins whose magnitude is comparable with eps = 1e-12 are excluded from the dB comparison only where the reference
        # itself is at its -240 dB clamp; everywhere else the comparison is on every bin
        err = np.abs(p - ref)
        worst = max(worst, float(err.max()))
        assert err.max() <= 1e-9, (k, float(err.max()))
        P = (10 ** (ref / 20) - 1e-12).clip(min=0) ** 2
        parity.check_db_rows(p[None, :], P[None, :], what=k + " (float64 stream kernel)")
        assert int(np.argmax(p)) == int(np.argmax(ref))
    parity._record("stream_f64", "golden stream frames", worst_abs_db_any_bin=worst)


def test_stream_frame_float32_plan_path_on_goldens(sp, golden_stream):
    """The same golden frames through the float32 STFT plan (the path a buffer size outside [2, 8192] or not a power of two
    takes, and the arithmetic of the batched kernels): the north_star tolerance, with the observed margin recorded."""
    z, meta = golden_stream
    for m in meta:
        k = m["key"]
        ref = z[k + "_power_db"]
        if np.all(ref == -240.0) or m["n"] < 16:
            continue
        pl = sp.get_plan(m["n"], m["n"], "rect", sp.FMT_CF32, 1.0, 1e-12, 0, variant=12)
        p = pl.stft(z[k + "_samples"], db_rows=True).db_rows[0].astype(np.float64)
        P = (10 ** (ref / 20) - 1e-12).clip(min=0) ** 2
        parity.check_db_rows(p[None, :], P[None, :], what=k + " (float32 plan, K1)")


@pytest.mark.parametrize("nfft,hop,kind", [(16, 16, "rect"), (32, 8, "hann"), (64, 16, "blackman"), (128, 128, "hann"),
                                           (256, 64, "hann"), (512, 256, "blackman"), (1024, 512, "hann"),
                                           (2048, 1024, "hann"), (4096, 1024, "hann"), (4096, 4096, "rect"),
                                           (8192, 4096, "hann"), (8192, 2048, "blackman")])
def test_cf32_host_parity(sp, nfft, hop, kind):
    L = nfft + hop * 37 + min(11, hop - 1)  # ragged tail, dropped
    x = sref.synth_iq(L, seed=nfft + hop).astype(np.complex64)
    pl = sp.SpectralPlan(nfft, hop, kind)
    r = pl.stft(x, db_rows=True, wf_rows=True, spectrum=True, welch=True, maxhold=True, vmin=-60.0, vmax=60.0)
    X = oracle_rows(x, nfft, hop, kind)
    P = X.real**2 + X.imag**2
    assert r.n_frames == 38 == X.shape[0]
    assert np.abs(r.spectrum - X).max() <= 4e-6 * np.sqrt(P.mean())
    parity.check_db_rows(r.db_rows, P, what=f"N={nfft}")
    parity.check_power(r.welch_acc[0], P.sum(axis=0), what="welch")
    parity.check_power(r.maxhold[0], P.max(axis=0), what="maxhold")
    parity.check_u8(r.wf_rows, sref.amplitude_db(X), -60.0, 60.0, what="u8")
    assert r.h2d_bytes == L * 8 and r.d2h_bytes > 0
    pl.close()


@pytest.mark.parametrize("fmt,hop,L", [(0, 4096, 4096 * 700 + 5), (0, 2048, 4096 + 2048 * 999), (1, 1024, 4096 + 1024 * 1500), (0, 4096, 4096)])
def test_4096_pipelined_rows_only_kernel(sp, fmt, hop, L):
    """variant 11: frame f+1's first pass overlapped with frame f's exchange (split-phase mbarriers); rows only.
    Several frames per CTA, a ragged tail, and the single-frame case."""
    n = 4096
    x = sref.synth_iq(L, seed=41)
    x = sref.to_ci16(x) if fmt else x.astype(np.complex64)
    pl = sp.SpectralPlan(n, hop, "hann", fmt, variant=11)
    ref = sp.SpectralPlan(n, hop, "hann", fmt, variant=12)     # K1 (round-1 default): same per-thread arithmetic
    vmin, vmax = (0.0, 130.0) if fmt else (-60.0, 60.0)
    r = pl.stft(x, db_rows=True, wf_rows=True, spectrum=True, vmin=vmin, vmax=vmax)
    r0 = ref.stft(x, db_rows=True, wf_rows=True, spectrum=True, vmin=vmin, vmax=vmax)
    assert r.n_frames == r0.n_frames == (L - n) // hop + 1
    np.testing.assert_array_equal(r.spectrum, r0.spectrum)      # same per-thread arithmetic, different schedule
    np.testing.assert_array_equal(r.db_rows, r0.db_rows)
    np.testing.assert_array_equal(r.wf_rows, r0.wf_rows)
    X = oracle_rows(x[: 2 * (n + 20 * hop)] if fmt else x[: n + 20 * hop], n, hop, "hann", fmt=fmt)
    parity.check_db_rows(r.db_rows[: X.shape[0]], X.real**2 + X.imag**2, what="pipelined")
    pl.close(); ref.close()


@pytest.mark.parametrize("variant", [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12])
def test_4096_kernel_variants_agree(sp, variant):
    n, hop = 4096, 1024
    x = sref.to_ci16(sref.synth_iq(n + 300 * hop, seed=77))
    pl = sp.SpectralPlan(n, hop, "hann", sp.FMT_CI16, variant=variant)
    r = pl.stft(x, db_rows=True, wf_rows=True, welch=True, maxhold=True, vmin=0.0, vmax=130.0)
    X = oracle_rows(x, n, hop, "hann", fmt=1)
    P = X.real**2 + X.imag**2
    parity.check_db_rows(r.db_rows, P, what=f"variant {variant}")
    parity.check_power(r.welch_acc[0], P.sum(axis=0), what="welch")
    parity.check_power(r.maxhold[0], P.max(axis=0), what="maxhold")
    parity.check_u8(r.wf_rows, sref.amplitude_db(X), 0.0, 130.0)
    pl.close()


@pytest.mark.parametrize("variant", [20, 21, 22])
@pytest.mark.parametrize("nfft,hop,kind,fmt", [(4096, 1024, "hann", 1), (4096, 4096, "rect", 0), (4096, 2048, "blackman", 0),
                                               (2048, 1024, "hann", 0), (2048, 512, "hann", 1), (1024, 512, "hann", 0),
                                               (1024, 256, "blackman", 1)])
def test_k1v2_warp_local_exchange_kernel(sp, variant, nfft, hop, kind, fmt):
    """K1v2 (spx_stft2_kernel.cuh: swizzled TMA tensor staging, warp-local first exchange, one barrier per frame; variant
    21 adds the FMA-form radix-16 DFT): oracle parity on many frames per CTA with a ragged tail; for N = 4096 variant 20
    is bit-identical to K1 (same arithmetic, different data flow)."""
    L = nfft + hop * 2999 + min(5, hop - 1)
    xc = sref.synth_iq(L, seed=nfft + hop + variant)
    x = sref.to_ci16(xc) if fmt else xc.astype(np.complex64)
    vmin, vmax = (0.0, 130.0) if fmt else (-60.0, 60.0)
    pl = sp.SpectralPlan(nfft, hop, kind, fmt, variant=variant)
    r = pl.stft(x, db_rows=True, wf_rows=True, spectrum=True, welch=True, maxhold=True, vmin=vmin, vmax=vmax)
    assert r.n_frames == 3000
    nchk = 64
    X = oracle_rows(x[: 2 * (nfft + (nchk - 1) * hop)] if fmt else x[: nfft + (nchk - 1) * hop], nfft, hop, kind, fmt=fmt)
    P = X.real**2 + X.imag**2
    assert np.abs(r.spectrum[:nchk] - X).max() <= 5e-6 * np.sqrt(P.mean())
    parity.check_db_rows(r.db_rows[:nchk], P, what=f"K1v2 v{variant} N={nfft}")
    parity.check_u8(r.wf_rows[:nchk], sref.amplitude_db(X), vmin, vmax, what=f"K1v2 v{variant} u8")
    ref = sp.SpectralPlan(nfft, hop, kind, fmt, variant=12)    # K1, the round-1 kernel
    r0 = ref.stft(x, db_rows=True, wf_rows=True, spectrum=True, welch=True, maxhold=True, vmin=vmin, vmax=vmax)
    if variant == 20 and nfft == 4096:
        np.testing.assert_array_equal(r.spectrum, r0.spectrum)
        np.testing.assert_array_equal(r.wf_rows, r0.wf_rows)
        np.testing.assert_array_equal(r.maxhold, r0.maxhold)
    else:   # every frame against K1 (itself oracle-checked above and elsewhere): tail frames, chunk flushes
        assert np.abs(r.spectrum - r0.spectrum).max() <= 4e-6 * np.sqrt(P.mean())
        assert np.abs(r.wf_rows.astype(np.int16) - r0.wf_rows.astype(np.int16)).max() <= 1
    parity.check_power(r.welch_acc[0], r0.welch_acc[0], what=f"K1v2 v{variant} welch vs K1", rel_tol=2e-5)
    parity.check_power(r.maxhold[0], r0.maxhold[0], what=f"K1v2 v{variant} maxhold vs K1", rel_tol=2e-5)
    if variant == 22:   # the FMA-pipe colormap index is bit-for-bit the F2I one
        alt = sp.SpectralPlan(nfft, hop, kind, fmt, variant=21)
        r1 = alt.stft(x, wf_rows=True, vmin=vmin, vmax=vmax)
        np.testing.assert_array_equal(r.wf_rows, r1.wf_rows)
        alt.close()
    pl.close(); ref.close()


def test_k1v2_multistream_and_unaligned_fallback(sp):
    """n_streams > 1 through the tensor map (stream stride a multiple of 128 bytes) and the fallback to K1 when the hop is
    not 128-byte aligned."""
    n, hop, S = 2048, 1024, 5
    L = n + 40 * hop
    xs = np.concatenate([sref.synth_iq(L, seed=30 + s, snr_db=4 * (s + 1)) for s in range(S)]).astype(np.complex64)
    pl = sp.SpectralPlan(n, hop, "hann", variant=20)
    r = pl.stft(xs, n_streams=S, welch=True, maxhold=True, db_rows=True)
    X = oracle_rows(xs, n, hop, "hann", n_streams=S)
    P = (X.real**2 + X.imag**2).reshape(S, -1, n)
    parity.check_db_rows(r.db_rows, P.reshape(-1, n), what="K1v2 streams")
    for s in range(S):
        parity.check_power(r.welch_acc[s], P[s].sum(axis=0), what=f"K1v2 welch s={s}")
        parity.check_power(r.maxhold[s], P[s].max(axis=0), what=f"K1v2 maxhold s={s}")
    pl.close()
    pl = sp.SpectralPlan(4096, 1023, "hann", variant=20)      # odd hop: frames are not 128-byte aligned -> K1 direct loads
    x = sref.synth_iq(4096 + 1023 * 20, seed=3).astype(np.complex64)
    r = pl.stft(x, db_rows=True)
    X = oracle_rows(x, 4096, 1023, "hann")
    parity.check_db_rows(r.db_rows, X.real**2 + X.imag**2, what="K1v2 fallback")
    pl.close()


def test_ci16_scale_sigmf(sp):
    """SigMF ci16_le autoscale 2^-15 (process_sigmf_data.py:52) vs raw stream values (streamer.py:114)."""
    n, hop = 1024, 512
    x = sref.to_ci16(sref.synth_iq(n + 40 * hop, seed=5))
    for scale in (1.0, 2.0**-15):
        pl = sp.SpectralPlan(n, hop, "hann", sp.FMT_CI16, in_scale=scale)
        r = pl.stft(x, db_rows=True, welch=True)
        X = oracle_rows(x, n, hop, "hann", fmt=1, scale=scale)
        P = X.real**2 + X.imag**2
        parity.check_db_rows(r.db_rows, P, what=f"scale {scale}")
        parity.check_power(r.welch_acc[0], P.sum(axis=0))
        pl.close()


def test_device_resident_equals_host_path(sp):
    from sdr_iq_visualizer_b200 import _native as nat
    n, hop = 2048, 512
    x = sref.synth_iq(n + 500 * hop, seed=9).astype(np.complex64)
    pl = sp.SpectralPlan(n, hop, "blackman")
    h = pl.stft(x, db_rows=True, wf_rows=True, welch=True, maxhold=True, vmin=-50, vmax=50)
    d = pl.stft(nat.DeviceArray.from_host(x), db_rows=True, wf_rows=True, welch=True, maxhold=True, vmin=-50, vmax=50)
    pl.sync()
    np.testing.assert_array_equal(h.db_rows, d.db_rows.to_host())
    np.testing.assert_array_equal(h.wf_rows, d.wf_rows.to_host())
    np.testing.assert_array_equal(h.maxhold, d.maxhold.to_host())
    np.testing.assert_allclose(h.welch_acc, d.welch_acc.to_host(), rtol=1e-12)  # fp64 atomics: order may differ
    pl.close()


def test_multistream_and_accumulate(sp):
    n, hop, S = 2048, 1024, 5
    L = n + 60 * hop
    xs = np.concatenate([sref.synth_iq(L, seed=100 + s, snr_db=5.0 * (s + 1)) for s in range(S)]).astype(np.complex64)
    pl = sp.SpectralPlan(n, hop, "hann")
    r = pl.stft(xs, n_streams=S, welch=True, maxhold=True, wf_rows=True, vmin=-40, vmax=60)
    X = oracle_rows(xs, n, hop, "hann", n_streams=S)
    P = (X.real**2 + X.imag**2).reshape(S, -1, n)
    assert r.n_frames == 61 and r.wf_rows.shape == (S * 61, n)
    for s in range(S):
        parity.check_power(r.welch_acc[s], P[s].sum(axis=0), what=f"stream {s}")
        parity.check_power(r.maxhold[s], P[s].max(axis=0))
    parity.check_u8(r.wf_rows, sref.amplitude_db(X), -40, 60)
    # accumulate=True continues the running Welch sum / max-hold (block-wise streaming use)
    half = (L // 2 // hop) * hop
    a = pl.stft(xs[:L][: half + n - hop], welch=True, maxhold=True)
    b = pl.stft(xs[:L][half:], welch=a.welch_acc, maxhold=a.maxhold, accumulate=True)
    assert a.n_frames + b.n_frames == 61
    parity.check_power(b.welch_acc[0], P[0].sum(axis=0), what="accumulated welch")
    parity.check_power(b.maxhold[0], P[0].max(axis=0), what="accumulated maxhold")
    pl.close()


def test_edge_cases(sp):
    pl = sp.SpectralPlan(1024, 512, "hann")
    r = pl.stft(np.zeros(100, np.complex64), db_rows=True, welch=True)   # shorter than one frame
    assert r.n_frames == 0 and r.db_rows.shape == (0, 1024) and np.all(r.welch_acc == 0)
    r = pl.stft(np.zeros(0, np.complex64), db_rows=True)
    assert r.n_frames == 0
    r = pl.stft(np.zeros(1024, np.complex64), db_rows=True, wf_rows=True)  # exactly one all-zero frame
    assert r.n_frames == 1 and np.abs(r.db_rows + 240.0).max() < 1e-3 and np.all(r.wf_rows == 0)
    with pytest.raises(sp.SpectralError):
        sp.SpectralPlan((1 << 19) + 2)  # beyond the supported non-power-of-two range
    with pytest.raises(sp.SpectralError):
        sp.SpectralPlan(0)
    with pytest.raises(sp.SpectralError):
        sp.SpectralPlan(1024, 2048)    # hop > nfft
    pl.close()
    # odd hop (not a divisor of N, frames start at unaligned samples)
    pl = sp.SpectralPlan(256, 77, "hann")
    x = sref.synth_iq(5000, seed=1).astype(np.complex64)
    r = pl.stft(x, db_rows=True)
    X = oracle_rows(x, 256, 77, "hann")
    parity.check_db_rows(r.db_rows, X.real**2 + X.imag**2)
    pl.close()


def test_welch_psd_matches_mlab_semantics(sp):
    """welch_psd == oracle restatement of plt.psd (process_sigmf_data.py:188): first 10 000 samples,
    NFFT=1024, noverlap=0, Hann."""
    x = sref.synth_iq(10000, seed=1).astype(np.complex64)
    f, pxx = sp.welch_psd(x, 1024, 1024, "hann", sample_rate=1e6, center_freq=2.4e9)
    fo, po = sref.welch_psd(x, 1024, 1024, "hann", 1e6, 2.4e9)
    np.testing.assert_array_equal(f, fo)
    parity.check_power(pxx, po, what="welch psd")
    # shorter than one frame: zero-padded to N like mlab
    f, pxx = sp.welch_psd(x[:300], 1024, 1024, "hann", 1e6, 0.0)
    fo, po = sref.welch_psd(x[:300], 1024, 1024, "hann", 1e6, 0.0)
    parity.check_power(pxx, po, what="zero-padded welch", rel_tol=2e-4)


def test_config1_full_size(sp):
    """BASELINE config 1: 2^20 cf32, N=1024 Hann, 50 % overlap -- full-array parity."""
    L, n, hop = 1 << 20, 1024, 512
    x = sref.synth_iq(L, seed=1).astype(np.complex64)
    pl = sp.SpectralPlan(n, hop, "hann")
    r = pl.stft(x, db_rows=True, wf_rows=True, welch=True, maxhold=True, vmin=-30.0, vmax=70.0)
    assert r.n_frames == 2047
    X = oracle_rows(x, n, hop, "hann")
    P = X.real**2 + X.imag**2
    parity.check_db_rows(r.db_rows, P, what="C1")
    parity.check_power(r.welch_acc[0], P.sum(axis=0), what="C1 welch")
    parity.check_power(r.maxhold[0], P.max(axis=0), what="C1 maxhold")
    parity.check_u8(r.wf_rows, sref.amplitude_db(X), -30.0, 70.0, what="C1 u8")
    pl.close()


def test_config2_slice_and_full_size_properties(sp):
    """BASELINE config 2: int16 @ 61.44 MS/s, N=4096, 75 % overlap.  Oracle parity on a 2^21-sample
    slice; at the full one-second size, size-independent properties (Parseval, block additivity)."""
    n, hop = 4096, 1024
    Ls = 1 << 21
    xs = sref.to_ci16(sref.synth_iq(Ls, seed=2))
    pl = sp.SpectralPlan(n, hop, "hann", sp.FMT_CI16)
    r = pl.stft(xs, db_rows=True, wf_rows=True, welch=True, maxhold=True, vmin=20.0, vmax=130.0)
    X = oracle_rows(xs, n, hop, "hann", fmt=1)
    P = X.real**2 + X.imag**2
    parity.check_db_rows(r.db_rows, P, what="C2 slice")
    parity.check_power(r.welch_acc[0], P.sum(axis=0), what="C2 welch")
    parity.check_power(r.maxhold[0], P.max(axis=0), what="C2 maxhold")
    parity.check_u8(r.wf_rows, sref.amplitude_db(X), 20.0, 130.0, what="C2 u8")
    # full size: 61.44 M samples (tile the slice; content does not matter for the properties)
    L = 61_440_000
    reps = -(-L // Ls)
    full = np.tile(xs.reshape(-1, 2), (reps, 1))[:L].reshape(-1)
    rf = pl.stft(full, welch=True, maxhold=True)
    assert rf.n_frames == 59_997
    # Parseval per frame summed over frames: sum_k sum_f |X_f[k]|^2 = N * sum_f sum_n |w[n] x_f[n]|^2
    w = sref.window("hann", n)   # float64 window (the kernel's float32 table differs by <= 6e-8 relative: inside 1e-6)
    iq = full.reshape(-1, 2).astype(np.float64)
    e = iq[:, 0] ** 2 + iq[:, 1] ** 2
    # sum over frames of sum_n w^2[n] e[f*hop+n]  via correlation of e with w^2 at stride hop
    w2 = w * w
    tot = 0.0
    for q in range(n // hop):
        seg = w2[q * hop:(q + 1) * hop]
        blocks = e[: (L // hop) * hop].reshape(-1, hop) @ seg          # per hop-block energy under this window quarter
        tot += blocks[q: q + rf.n_frames].sum()
    assert abs(rf.welch_acc.sum() - n * tot) <= 1e-6 * n * tot
    # block additivity: two halves with accumulate == one shot
    cut = (rf.n_frames // 2) * hop
    a = pl.stft(full[: 2 * (cut + n - hop)], welch=True, maxhold=True)
    b = pl.stft(full[2 * cut:], welch=a.welch_acc, maxhold=a.maxhold, accumulate=True)
    assert a.n_frames + b.n_frames == rf.n_frames
    np.testing.assert_allclose(b.welch_acc, rf.welch_acc, rtol=2e-6)  # fp32 partial sums per <=256-frame chunk
    np.testing.assert_array_equal(b.maxhold, rf.maxhold)
    pl.close()


@pytest.mark.parametrize("nfft,hop,kind,fmt", [(16384, 8192, "hann", 0), (32768, 32768, "blackman", 0),
                                               (65536, 32768, "hann", 0), (65536, 16384, "hann", 1),
                                               (131072, 65536, "hann", 0), (262144, 262144, "rect", 0),
                                               (1048576, 524288, "hann", 0)])
def test_large_n_four_step_parity(sp, nfft, hop, kind, fmt):
    """N >= 16384 runs as two fused kernels (columns + rows) through an L2-resident scratch."""
    F = 5 if nfft <= 131072 else 2
    L = nfft + hop * (F - 1) + 7
    x = sref.synth_iq(L, seed=nfft % 1000 + 3)
    x = sref.to_ci16(x) if fmt else x.astype(np.complex64)
    pl = sp.SpectralPlan(nfft, hop, kind, fmt)
    vmin, vmax = (20.0, 150.0) if fmt else (-40.0, 90.0)
    r = pl.stft(x, db_rows=True, wf_rows=True, spectrum=True, welch=True, maxhold=True, vmin=vmin, vmax=vmax)
    assert r.n_frames == F
    X = oracle_rows(x, nfft, hop, kind, fmt=fmt)
    P = X.real**2 + X.imag**2
    # fp32 FFT error: a floor relative to the frame's RMS bin level, a part relative to the bin itself, and
    # correlated-rounding spurs of the dominant tone (measured: -149 dBc at k0 + N/2 for N = 2^18)
    assert np.all(np.abs(r.spectrum - X) <= 6e-6 * np.sqrt(P.mean()) + 1e-6 * np.abs(X) + 1e-7 * np.abs(X).max())
    parity.check_db_rows(r.db_rows, P, what=f"N={nfft}")
    parity.check_power(r.welch_acc[0], P.sum(axis=0), what="welch")
    parity.check_power(r.maxhold[0], P.max(axis=0), what="maxhold")
    parity.check_u8(r.wf_rows, sref.amplitude_db(X), vmin, vmax, what="u8")
    pl.close()


def test_large_n_tone_bins_and_batches(sp):
    """integer bin placement for N = 65536: a pure tone at bin k lands at fftshift position (k + N/2) mod N, for bins at
    and around the 256-point sub-transform boundaries, DC, Nyquist and the last bin (one frame each, dB rows, K2).
    Batching through several scratch batches is tested in test_dispatch_paths_gpu.py."""
    n = 65536
    t = np.arange(n)
    pl = sp.SpectralPlan(n, n, "rect")
    for k in (0, 1, 255, 256, 257, 32767, 32768, 65535):
        x = np.exp(2j * np.pi * k * t / n).astype(np.complex64)
        r = pl.stft(x, db_rows=True)
        assert int(np.argmax(r.db_rows[0])) == (k + n // 2) % n
    pl.close()


def test_config5_prefix(sp):
    """BASELINE config 5 on a 2^23-sample prefix: N = 65536, Hann, 50 % overlap, u8 rows + Welch."""
    n, hop, L = 65536, 32768, 1 << 23
    x = sref.synth_iq(L, seed=5).astype(np.complex64)
    pl = sp.SpectralPlan(n, hop, "hann")
    r = pl.stft(x, wf_rows=True, welch=True, maxhold=True, vmin=-20.0, vmax=110.0)
    assert r.n_frames == 255
    X = oracle_rows(x, n, hop, "hann")
    P = X.real**2 + X.imag**2
    parity.check_power(r.welch_acc[0], P.sum(axis=0), what="C5 welch")
    parity.check_power(r.maxhold[0], P.max(axis=0), what="C5 maxhold")
    parity.check_u8(r.wf_rows, sref.amplitude_db(X), -20.0, 110.0, what="C5 u8")
    pl.close()


@pytest.mark.parametrize("hop,frames,kind,outs", [(32768, 1, "hann", "all"), (32768, 2, "hann", "all"), (32768, 19, "blackman", "all"),
                                                   (32768, 127, "hann", "all"), (65536, 40, "rect", "rows"), (16384, 90, "hann", "acc"),
                                                   (256, 37, "hann", "all")])
def test_k2v2_single_kernel_65536(sp, hop, frames, kind, outs):
    """K2v2 (spx_big2.cu: one persistent kernel, role A / role B per CTA, scratch resident in L2, counters between the
    16 CTAs of a lane): oracle parity and agreement with the two-kernel path (variant 1).  Frame counts below, at and above
    the lane count (single-frame lanes, uneven lanes, scratch slots wrapping around), hops down to 256 samples."""
    n = 65536
    L = n + hop * (frames - 1) + 77
    x = sref.synth_iq(L, seed=frames + hop, tone_cycles_per_sample=20000.37 / 65536).astype(np.complex64)
    vmin, vmax = -20.0, 110.0
    kw = dict(wf_rows=outs in ("all", "rows"), welch=outs in ("all", "acc"), maxhold=outs in ("all", "acc"), vmin=vmin, vmax=vmax)
    pl = sp.SpectralPlan(n, hop, kind)
    old = sp.SpectralPlan(n, hop, kind, variant=1)
    r, r0 = pl.stft(x, **kw), old.stft(x, **kw)
    assert r.n_frames == r0.n_frames == frames
    nchk = min(frames, 6)
    sel = sorted(set(range(nchk)) | set(range(max(0, frames - 3), frames)))
    X = np.stack([oracle_rows(x[f * hop: f * hop + n], n, n, kind)[0] for f in sel])
    if kw["wf_rows"]:
        parity.check_u8(r.wf_rows[sel], sref.amplitude_db(X), vmin, vmax, what=f"K2v2 u8 F={frames}")
        assert np.abs(r.wf_rows.astype(np.int16) - r0.wf_rows.astype(np.int16)).max() <= 1      # every row vs the two-kernel path
        assert (r.wf_rows != r0.wf_rows).mean() < 2e-3
    if kw["welch"]:
        parity.check_power(r.welch_acc[0], r0.welch_acc[0], what="K2v2 welch vs two-kernel path", rel_tol=1.5e-4)
        parity.check_power(r.maxhold[0], r0.maxhold[0], what="K2v2 maxhold vs two-kernel path", rel_tol=1.5e-4)
        if frames <= 6:
            P = X.real**2 + X.imag**2
            parity.check_power(r.welch_acc[0], P.sum(axis=0), what="K2v2 welch")
            parity.check_power(r.maxhold[0], P.max(axis=0), what="K2v2 maxhold")
    pl.close(); old.close()


@pytest.mark.parametrize("hop,frames,kind,scale", [(32768, 3, "hann", 1.0), (32768, 41, "blackman", 2.0**-15), (65536, 20, "rect", 1.0),
                                                   (16384, 70, "hann", 2.0**-11), (256, 25, "rect", 2.0**-15)])
def test_k2v2_int16_input(sp, hop, frames, kind, scale):
    """K2v2 on int16 I/Q (column tiles of 64 B under the 64-byte TMA swizzle, int16 -> float and window * scale fused on load):
    oracle parity on the first and last frames, agreement with the two-kernel path (variant 1) on every row."""
    from sdr_iq_visualizer_b200 import _native as nat
    n = 65536
    L = n + hop * (frames - 1) + 77
    raw = sref.to_ci16(sref.synth_iq(L, seed=frames + hop + 1, tone_cycles_per_sample=20000.37 / 65536))
    db_shift = 20.0 * np.log10(scale * 1024.0)
    vmin, vmax = -20.0 + db_shift, 110.0 + db_shift
    kw = dict(wf_rows=True, welch=True, maxhold=True, vmin=vmin, vmax=vmax)
    pl = sp.SpectralPlan(n, hop, kind, nat.FMT_CI16, in_scale=scale)
    old = sp.SpectralPlan(n, hop, kind, nat.FMT_CI16, in_scale=scale, variant=1)
    r, r0 = pl.stft(raw, **kw), old.stft(raw, **kw)
    assert r.n_frames == r0.n_frames == frames
    sel = sorted(set(range(min(frames, 3))) | set(range(max(0, frames - 2), frames)))
    xc = sref.unpack_ci16(raw, scale)
    X = np.stack([sref.shift_bins(sref.stft(xc[f * hop: f * hop + n], n, n, kind))[0] for f in sel])
    parity.check_u8(r.wf_rows[sel], sref.amplitude_db(X), vmin, vmax, what=f"K2v2 ci16 u8 F={frames}")
    assert np.abs(r.wf_rows.astype(np.int16) - r0.wf_rows.astype(np.int16)).max() <= 1
    assert (r.wf_rows != r0.wf_rows).mean() < 2e-3
    parity.check_power(r.welch_acc[0], r0.welch_acc[0], what="K2v2 ci16 welch vs two-kernel path", rel_tol=1.5e-4)
    parity.check_power(r.maxhold[0], r0.maxhold[0], what="K2v2 ci16 maxhold vs two-kernel path", rel_tol=1.5e-4)
    if frames <= 3:
        P = X.real**2 + X.imag**2
        parity.check_power(r.welch_acc[0], P.sum(axis=0), what="K2v2 ci16 welch")
        parity.check_power(r.maxhold[0], P.max(axis=0), what="K2v2 ci16 maxhold")
    pl.close(); old.close()


@pytest.mark.parametrize("nfft,hop,fmt,L", [(4096, 1024, 1, 300_000), (65536, 32768, 0, 1 << 21)])
def test_peer_output_pipeline_matches_direct_outputs(sp, monkeypatch, nfft, hop, fmt, L):
    """peer_outputs=True (multi-GPU capture shards): accumulators reduced with system-scope atomics, uint8 rows
    staged in frame pieces and pushed by the copy engine -- same rows and sums as the direct path.  World size 1
    here (the target is this GPU's own memory); tools/bench_sharded.py --check covers the IPC-mapped case."""
    from sdr_iq_visualizer_b200 import _native as nat, dist as sd
    monkeypatch.setenv("SPX_PEER_PIECE_BYTES", str(40 * nfft))           # 40-frame pieces: several pieces, ragged tail
    x = sref.synth_iq(L, seed=9)
    x = sref.to_ci16(x) if fmt else x.astype(np.complex64)
    pl = sp.SpectralPlan(nfft, hop, "hann", fmt)
    ref = pl.stft(x, wf_rows=True, welch=True, maxhold=True, vmin=-20.0, vmax=130.0)
    F = ref.n_frames
    d_in = nat.DeviceArray.from_host(x)
    sh = sd.capture_shard(L, nfft, hop, 0, 1)
    assert (sh.f0, sh.f1) == (0, F)
    tgt = sd.PeerReduceTarget(nfft, F, 0, 1, 0)
    for mode in (3, 3, 1):                                                 # staged + copy engine (twice: buffers and events are reused), then direct rows
        tgt.zero()
        nat.check(nat.lib().spx_memset(0, tgt.rows.ptr, 0, F * nfft))
        pl.stft(d_in, wf_rows=tgt.rows.rows(0, F), welch=tgt.welch, maxhold=tgt.maxhold, vmin=-20.0, vmax=130.0, accumulate=True,
                n_samples=L, peer_outputs=mode)
        pl.sync()
        rows = np.empty((F, nfft), np.uint8)
        nat.check(nat.lib().spx_memcpy_d2h(0, rows.ctypes.data, tgt.rows.ptr, rows.nbytes))
        np.testing.assert_array_equal(rows, ref.wf_rows)
        np.testing.assert_allclose(tgt.buffers["welch"].array.to_host(), ref.welch_acc, rtol=1e-6)  # fp32 partials regroup with the pieces
        np.testing.assert_array_equal(tgt.buffers["maxhold"].array.to_host(), ref.maxhold)
    tgt.zero()
    assert sd.fused_capture_step(pl, d_in, sh, tgt, -20.0, 130.0) == F      # the driver the sharded bench uses (owner: mode 1)
    pl.sync()
    np.testing.assert_allclose(tgt.buffers["welch"].array.to_host(), ref.welch_acc, rtol=1e-6)
    tgt.close()
    pl.close()


@pytest.mark.parametrize("nfft,hop,kind,fmt", [(1000, 1000, "rect", 0), (1000, 250, "hann", 1), (4095, 2048, "hann", 0),
                                               (4097, 4097, "blackman", 0), (7, 3, "rect", 0), (1, 1, "rect", 0),
                                               (12, 12, "hann", 0), (3000, 1500, "hann", 1), (100000, 50000, "hann", 0)])
def test_arbitrary_length_bluestein_parity(sp, nfft, hop, kind, fmt):
    """Frame lengths that are not a power of two (the reference's np.fft.fft takes any rx_buffer_size): Bluestein over
    the power-of-two kernels.  Same parity rules; fftshift follows numpy for odd N (out[j] = X[(j - N//2) mod N])."""
    F = 9 if nfft < 50000 else 3
    L = nfft + hop * (F - 1) + min(5, hop - 1)
    x = sref.synth_iq(L, seed=nfft % 97 + 1)
    x = sref.to_ci16(x) if fmt else x.astype(np.complex64)
    pl = sp.SpectralPlan(nfft, hop, kind, fmt)
    vmin, vmax = (20.0, 150.0) if fmt else (-40.0, 90.0)
    r = pl.stft(x, db_rows=True, wf_rows=True, spectrum=True, welch=True, maxhold=True, vmin=vmin, vmax=vmax)
    assert r.n_frames == F
    X = oracle_rows(x, nfft, hop, kind, fmt=fmt)
    P = X.real**2 + X.imag**2
    assert np.all(np.abs(r.spectrum - X) <= 6e-6 * np.sqrt(P.mean()) + 2e-6 * np.abs(X) + 1e-7 * np.abs(X).max())
    if nfft > 1:
        parity.check_db_rows(r.db_rows, P, what=f"N={nfft}")
        parity.check_power(r.welch_acc[0], P.sum(axis=0), what="welch")
        parity.check_power(r.maxhold[0], P.max(axis=0), what="maxhold")
        parity.check_u8(r.wf_rows, sref.amplitude_db(X), vmin, vmax, what="u8")
    pl.close()


def test_stream_frame_any_buffer_size(sp):
    """The drop-in for streamer.py:119-121 with rx_buffer_size = 1000 and 3001 (odd): freqs and power_db as numpy gives them."""
    rng = np.random.default_rng(4)
    for n in (1000, 3001):
        s = (rng.integers(-2047, 2048, n) + 1j * rng.integers(-2047, 2048, n)).astype(np.complex128)
        f, p = sp.stream_frame(s, 1e6, 2.4e9)
        f_ref, p_ref = sref.stream_frame(s, 1e6, 2.4e9)
        assert np.array_equal(f, f_ref)
        X = np.fft.fftshift(np.fft.fft(s))
        parity.check_db_rows(p[None, :], (X.real**2 + X.imag**2)[None, :], what=f"stream N={n}")


def test_non_finite_samples_and_extreme_values(sp):
    """NaN / Inf samples poison exactly the frames that contain them (as np.fft.fft does); the uint8 index of a NaN bin
    is 0; the max-hold skips NaN powers (fmax semantics, documented in spx.h); int16 full-scale values are exact."""
    n, hop = 1024, 512
    x = sref.synth_iq(n + hop * 9, seed=3).astype(np.complex64)
    x[3 * hop + 5] = np.nan                                   # inside frames 2 and 3 only
    pl = sp.SpectralPlan(n, hop, "hann")
    r = pl.stft(x, db_rows=True, wf_rows=True, maxhold=True, vmin=-60.0, vmax=60.0)
    bad = np.isnan(r.db_rows).all(axis=1)
    assert list(np.flatnonzero(bad)) == [2, 3] and not np.isnan(r.db_rows[~bad]).any()
    assert np.all(r.wf_rows[bad] == 0)
    good = np.delete(np.arange(r.n_frames), [2, 3])
    X = oracle_rows(x, n, hop, "hann")
    parity.check_db_rows(r.db_rows[good], (X.real**2 + X.imag**2)[good], what="frames without NaN")
    assert np.isfinite(r.maxhold).all()
    parity.check_power(r.maxhold[0], (X.real**2 + X.imag**2)[good].max(axis=0), what="max-hold skips NaN frames")
    pl.close()
    # int16 extremes, maximum overlap (hop = 1) on a short input
    raw = np.array([-32768, 32767] * 40 + [32767, -32768] * 40, np.int16)
    pl = sp.SpectralPlan(64, 1, "rect", sp.FMT_CI16)
    r = pl.stft(raw, spectrum=True, db_rows=True)
    assert r.n_frames == 80 - 64 + 1
    X = oracle_rows(raw, 64, 1, "rect", fmt=1)
    assert np.abs(r.spectrum - X).max() <= 4e-6 * np.abs(X).max()
    pl.close()


@pytest.mark.parametrize("n", [2, 4, 16, 64, 256, 1024, 4096, 8192])
def test_stream_frame_float64_kernel_vs_numpy(sp, n):
    """K6 (spx_stream_frame_f64): the reference's three lines (streamer.py:119-121) in float64 on the GPU, complex128 and
    complex64 input, any power-of-two buffer up to 8192 samples: within 1e-9 dB of numpy on every bin, exact frequency
    axis, uint8 row equal to the float64 definition except at exact ties."""
    rng = np.random.default_rng(n)
    x = np.rint(rng.normal(0, 300, n) + 1j * rng.normal(0, 300, n)) + 1500 * np.exp(2j * np.pi * 0.123 * np.arange(n))
    fs, fc = 2.5e6, 9.15e8
    f_ref, p_ref = sref.stream_frame(x, fs, fc)
    f, p, wf = sp.stream_frame(x, fs, fc, wf_range=(0.0, 140.0))
    np.testing.assert_array_equal(f, f_ref)
    assert p.dtype == np.float64 and np.abs(p - p_ref).max() <= 1e-9
    pre = (p_ref - 0.0) * 256.0 / 140.0
    want = np.clip(np.floor(pre), 0, 255).astype(np.uint8)
    assert np.all((wf == want) | (np.abs(pre - np.rint(pre)) < 1e-6))
    x32 = x.astype(np.complex64)
    _, p32 = sp.stream_frame(x32, fs, fc)
    _, p32_ref = sref.stream_frame(x32.astype(np.complex128), fs, fc)
    assert np.abs(p32 - p32_ref).max() <= 1e-9
    assert np.array_equal(sp.stream_frame(np.zeros(n, complex), fs, fc)[1], np.full(n, -240.0))


def test_copy_ceiling_probe_reports_a_plausible_rate():
    import ctypes as C
    from sdr_iq_visualizer_b200 import _native as nat
    a, b = nat.pinned_empty(32 << 20, np.uint8), nat.pinned_empty(32 << 20, np.uint8)
    a[:] = 1
    sec = C.c_double()
    nat.check(nat.lib().spx_copy_ceiling(0, a.ctypes.data, a.nbytes, b.ctypes.data, b.nbytes, 8 << 20, 2, C.byref(sec)))
    gbs = a.nbytes / sec.value / 1e9
    assert 1.0 < gbs < 200.0 and np.all(b == 0)      # the probe copies its own zeroed device buffer out


@pytest.mark.parametrize("hop,fmt,frames", [(1024, 1, 3000), (1024, 0, 1500), (2048, 0, 2000), (2048, 1, 777), (1024, 1, 5)])
def test_k1v2_strip_staging_variant_is_bit_identical(sp, hop, fmt, frames):
    """Variant 23 (ring of hop blocks in the staging buffer: a frame inside a chunk copies only its newest block): same
    arithmetic as the default kernel, so every output is bit-identical; chunk starts (whole-frame copies), ring
    wrap-around and short inputs are all exercised."""
    n = 4096
    L = n + hop * (frames - 1) + 3
    xc = sref.synth_iq(L, seed=hop + frames)
    x = sref.to_ci16(xc) if fmt else xc.astype(np.complex64)
    vmin, vmax = (0.0, 130.0) if fmt else (-60.0, 60.0)
    a = sp.SpectralPlan(n, hop, "hann", fmt, variant=23)
    b = sp.SpectralPlan(n, hop, "hann", fmt, variant=22)
    ra = a.stft(x, db_rows=True, wf_rows=True, welch=True, maxhold=True, vmin=vmin, vmax=vmax)
    rb = b.stft(x, db_rows=True, wf_rows=True, welch=True, maxhold=True, vmin=vmin, vmax=vmax)
    assert ra.n_frames == rb.n_frames == frames
    np.testing.assert_array_equal(ra.db_rows, rb.db_rows)
    np.testing.assert_array_equal(ra.wf_rows, rb.wf_rows)
    np.testing.assert_array_equal(ra.maxhold, rb.maxhold)
    np.testing.assert_allclose(ra.welch_acc, rb.welch_acc, rtol=1e-12)     # fp64 atomics: the order of the flushes may differ
    a.close(); b.close()
