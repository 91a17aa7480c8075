"""GPU tests of the polyphase channelizer (K10 chan_kernel): parity with the float64 oracle (tests/chan_ref.py), agreement
with K9 (DdcPlan) channel by channel, bit identity under chunking, between memory modes and with padding columns, the CPU
harness of K10's math, behaviour (tone at a channel centre, adjacent-channel suppression, NaN, empty calls, every error
code, a host call behind a device call), the chain into the multi-stream STFT and sigmf_io.scan_channels."""
import ctypes as C

import numpy as np
import pytest

from oracle import classifier_ref as cref
from oracle import spectral_ref as sref
from tests import chan_ref as cr, parity
from tests.test_channelizer_cpu import emul, emul_chan   # noqa: F401  (module fixture: K10's math built for the host)
from tests.test_dispatch_paths_gpu import launched

pytestmark = pytest.mark.gpu

FS = 61.44e6
FIRST = 1_000_003          # not a multiple of any M


def _mods():
    from sdr_iq_visualizer_b200 import _native as nat, ddc, sigmf_io, spectral as sp
    nat.require_device()
    return nat, ddc, sp, sigmf_io


def _signal(L, fmt, seed, tones=((0.11, 0.5), (-0.27, 0.2)), noise=0.05):
    rng = np.random.default_rng(seed)
    n = np.arange(L)
    x = sum(a * np.exp(2j * np.pi * f * n) for f, a in tones) + noise * (rng.normal(size=L) + 1j * rng.normal(size=L))
    if fmt == "ci16":
        return sref.to_ci16(x * 0.7), 2.0 ** -15
    return x.astype(np.complex64), 1.0


def _fmt(sp, fmt):
    return sp.FMT_CI16 if fmt == "ci16" else sp.FMT_CF32


def _host(h, arr):
    """A device result of a handle's call, after the handle's stream has finished it."""
    h.sync()
    return arr.to_host()


def _ran(names):
    assert any("chan_kernel" in nm for nm in names), sorted(set(names))


def _parity(got, want, h, x, scale, what):
    bar = 1e-5 * cr.bound(h, x, scale)
    err = float(np.abs(np.asarray(got, np.complex128) - want).max()) if want.size else 0.0
    parity._record("chan", what, outputs=int(want.size), worst_abs=err, bar=bar, margin=bar / err if err else None)
    assert got.shape == want.shape
    assert err <= bar, f"{what}: {err:.3e} > {bar:.3e}"


# default designs (both D; the critically sampled ones at M >= 1024 have windows larger than shared memory and run the
# blocked mode), caller taps at T = 1 and T = 32 M, and T < D (windows shorter than the hop)
SHAPES = [(16, 8, "default"), (64, 32, "default"), (64, 64, "default"), (1024, 512, "default"), (4096, 2048, "default"),
          (1024, 1024, "default"), (2048, 2048, "default"), (4096, 4096, "default"),
          (64, 32, "caller1"), (64, 32, "caller2048"), (1024, 512, "caller32768"),
          (16, 8, "caller4"), (4096, 2048, "caller1"), (4096, 2048, "caller1000")]


@pytest.mark.parametrize("fmt", ["cf32", "ci16"])
@pytest.mark.parametrize("mem", ["host", "device"])
@pytest.mark.parametrize("M,D,taps", SHAPES)
def test_parity(fmt, mem, M, D, taps):
    nat, ddc, sp, _ = _mods()
    rng = np.random.default_rng(M + D)
    h = None if taps == "default" else rng.normal(size=int(taps[6:])) / np.sqrt(int(taps[6:]))
    T = ddc.design_taps(M // 2, transition=0.5).size if h is None and D == M // 2 else \
        ddc.design_taps(M).size if h is None else h.size
    L = T + (12 if T > 20000 else 40 if M >= 1024 else 300) * D + 17
    x, scale = _signal(L, fmt, M + (fmt == "ci16"))
    ch = ddc.Channelizer(FS, M, D, taps=h, in_fmt=_fmt(sp, fmt), in_scale=scale)
    y, names = launched(lambda: ch.exec(x if mem == "host" else nat.DeviceArray.from_host(x), first_sample=FIRST))
    _ran(names)
    y = y if mem == "host" else y.to_host()
    _parity(y, cr.channelize(x, ch.taps, M, D, FIRST, scale), ch.taps, x, scale, f"{fmt} {mem} M={M} D={D} T={T}")
    ch.close()


@pytest.mark.parametrize("M,D", [(16, 8), (64, 32), (64, 64), (1024, 512)])   # every default shape with T <= 8192
def test_matches_ddc(M, D):
    """Channels 0, M/2 - 1, M/2 and M - 1 are K9 at shift (j - M/2) fs / M with the same taps and D."""
    nat, ddc, sp, _ = _mods()
    ch = ddc.Channelizer(FS, M, D)
    assert ch.n_taps <= ddc.MAX_TAPS
    x, _ = _signal(ch.n_taps + 200 * D + 5, "cf32", M)
    dx = nat.DeviceArray.from_host(x)
    y, names = launched(lambda: ch.exec(dx, first_sample=FIRST))   # launched() synchronises the device
    _ran(names)
    y = y.to_host()
    for j in (0, M // 2 - 1, M // 2, M - 1):
        with ddc.DdcPlan(FS, (j - M // 2) * FS / M, D, taps=ch.taps) as dd:
            assert dd.phase_inc == cr.phase_inc(j, M)
            yd = dd.exec(dx, first_sample=FIRST)
            dd.sync()
            yd = yd.to_host()
        _parity(y[j], yd.astype(np.complex128), ch.taps, x, 1.0, f"vs K9 M={M} D={D} j={j}")
    ch.close()


def test_matches_cpu_harness(emul):  # noqa: F811
    """The fold is K10's in the order spx_chan_device.cuh states; the FFT phases are the STFT's, whose complex multiplies
    the device build contracts into FMAs and the host build does not, so the harness agrees to float32 FFT rounding."""
    nat, ddc, sp, _ = _mods()
    for M, D, T, fmt in [(16, 8, 81, "cf32"), (64, 32, 323, "ci16"), (64, 64, 2048, "cf32"), (1024, 512, 5141, "ci16"),
                         (1024, 1024, 25697, "cf32"), (4096, 2048, 1000, "ci16")]:
        rng = np.random.default_rng(T)
        h = rng.normal(size=T) / np.sqrt(T)
        x, scale = _signal(T + 60 * D, fmt, T)
        ch = ddc.Channelizer(FS, M, D, taps=h, in_fmt=_fmt(sp, fmt), in_scale=scale)
        y = _host(ch, ch.exec(nat.DeviceArray.from_host(x), first_sample=77))
        want = emul_chan(emul, x, ch.taps, M, D, 77, scale)
        tol = 8 * np.log2(M) * 2.0 ** -24 * cr.bound(h, x, scale)
        err = float(np.abs(y.astype(np.complex128) - want).max())
        parity._record("chan_harness", f"M={M} D={D} T={T} {fmt}", worst_abs=err, tol=tol,
                       bit_identical_fraction=float(np.mean(y.view(np.uint64) == want.view(np.uint64))))
        assert err <= tol, (M, D, T, fmt, err, tol)
        ch.close()


@pytest.mark.parametrize("fmt", ["cf32", "ci16"])
@pytest.mark.parametrize("M,D", [(64, 32), (64, 64), (1024, 512), (1024, 1024)])
def test_chunking_bit_identical(fmt, M, D):
    nat, ddc, sp, _ = _mods()
    ch = ddc.Channelizer(FS, M, D, in_fmt=_fmt(sp, fmt))
    T = ch.n_taps
    x, _ = _signal(T + 900 * D + 3, fmt, 11)
    ew = 2 if fmt == "ci16" else 1
    base = 5 * 10 ** 9 + 3
    one = _host(ch, ch.exec(nat.DeviceArray.from_host(x), first_sample=base))
    n_out = one.shape[1]
    cuts = [0, 1, n_out // 3, n_out // 3 + 7, n_out - 2, n_out]
    parts = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        seg = x[ew * a * D: ew * ((b - 1) * D + T)]
        parts.append(_host(ch, ch.exec(nat.DeviceArray.from_host(seg), first_sample=base + a * D)))
    assert np.array_equal(np.concatenate(parts, axis=1).view(np.uint32), one.view(np.uint32))
    ch.close()


def test_host_pieces_and_padding(monkeypatch):
    """Host memory over several pieces equals device memory bit for bit; columns past n_out keep a sentinel."""
    nat, ddc, sp, _ = _mods()
    monkeypatch.setenv("SPX_H2D_PIECE_BYTES", "65536")
    x, scale = _signal(300_000, "ci16", 4)
    ch = ddc.Channelizer(FS, 64, 32, in_fmt=sp.FMT_CI16, in_scale=scale)
    n_out = ch.out_count(300_000)
    sentinel = np.complex64(complex(-7.25, 3.5))
    host = np.full((64, n_out + 5), sentinel, np.complex64)
    ch.exec(x, first_sample=9, out=host)
    assert ch.last_h2d_bytes > x.nbytes                           # several pieces with halos
    assert ch.last_d2h_bytes == 64 * n_out * 8
    dev = nat.DeviceArray.from_host(np.full((64, n_out + 3), sentinel, np.complex64))
    dev = _host(ch, ch.exec(nat.DeviceArray.from_host(x), first_sample=9, out=dev))
    assert np.array_equal(host[:, :n_out].view(np.uint32), dev[:, :n_out].view(np.uint32))
    assert (host[:, n_out:] == sentinel).all() and (dev[:, n_out:] == sentinel).all()
    ch.close()


def test_tone_at_channel_centre_and_suppression():
    nat, ddc, sp, _ = _mods()
    M, D = 64, 32
    k = 41                                       # c = 9
    f = (k - M // 2) / M                         # cycles/sample at the input rate
    ch = ddc.Channelizer(FS, M, D)
    x, _ = _signal(ch.n_taps + 400 * D, "cf32", 1, tones=((f, 0.5),), noise=0.0)
    y, names = launched(lambda: ch.exec(nat.DeviceArray.from_host(x), first_sample=FIRST))
    _ran(names)
    y = y.to_host()
    yk = y[k].astype(np.complex128)
    assert np.abs(np.abs(yk) - 0.5).max() < 1e-4                 # unit DC gain: the tone comes out at 0 Hz, constant
    assert np.abs(np.diff(np.angle(yk))).max() < 1e-4
    want = cr.channelize(x, ch.taps, M, D, FIRST)
    pk = np.mean(np.abs(yk) ** 2)
    for j in (k - 3, k + 3, 5):                                  # outside channel k's filter skirt
        sup = 10 * np.log10(pk / np.mean(np.abs(y[j].astype(np.complex128)) ** 2))
        sup_ref = 10 * np.log10(np.mean(np.abs(want[k]) ** 2) / np.mean(np.abs(want[j]) ** 2))
        parity._record("chan_suppression", f"channel {j} under {k} dB", got=float(sup), oracle=float(sup_ref))
        assert sup >= min(sup_ref - 1.0, 100.0), (j, sup, sup_ref)
    ch.close()


def test_nan_and_empty():
    nat, ddc, sp, _ = _mods()
    M, D = 16, 8
    ch = ddc.Channelizer(FS, M, D)
    T = ch.n_taps
    x, _ = _signal(5000, "cf32", 5)
    x[2001] = np.nan
    y = _host(ch, ch.exec(nat.DeviceArray.from_host(x)))
    m = np.arange(y.shape[1])
    covers = (m * D <= 2001) & (2001 <= m * D + T - 1)
    np.testing.assert_array_equal(np.isnan(y).all(axis=0), covers)
    assert not np.isnan(y[:, ~covers]).any()
    _, names = launched(lambda: (ch.exec(x[:T - 1]), ch.exec(nat.DeviceArray.from_host(x[:T - 1]))))
    assert not any("chan_kernel" in nm for nm in names)
    assert ch.exec(x[:T - 1]).shape == (M, 0)
    ch.close()


def test_errors():
    nat, ddc, sp, _ = _mods()
    lib = nat.lib()
    h = (C.c_double * 2048)(*([1.0] * 2048))

    def create(**kw):
        cfg = nat.spx_chan_config(C.sizeof(nat.spx_chan_config), 0, 0, 1.0, 64, 32, 65, C.cast(h, C.c_void_p))
        for key, v in kw.items():
            setattr(cfg, key, v)
        p = C.c_void_p()
        return lib.spx_chan_create(C.byref(p), C.byref(cfg)), p

    for kw in (dict(n_channels=48), dict(n_channels=8), dict(n_channels=8192), dict(decim=16), dict(decim=128),
               dict(n_taps=0), dict(n_taps=2049), dict(taps=None), dict(in_fmt=5), dict(device=99), dict(struct_size=4)):
        rc, _ = create(**kw)
        assert rc == nat.E_INVALID, kw
    big = (C.c_double * (32 * 4096))()
    rc, q = create(n_channels=4096, decim=4096, n_taps=32 * 4096, taps=C.cast(big, C.c_void_p))   # the longest window
    assert rc == nat.OK and lib.spx_chan_destroy(q) == nat.OK
    assert lib.spx_chan_create(None, None) == nat.E_INVALID
    rc, p = create()
    assert rc == nat.OK
    x = np.zeros(1000, np.complex64)
    out = np.zeros((64, 40), np.complex64)
    n = C.c_int64()
    ex = lib.spx_chan_exec
    X, O = x.ctypes.data, out.ctypes.data
    assert ex(p, 7, X, 1000, 0, O, 40, C.byref(n), None, None, None) == nat.E_INVALID
    assert ex(p, 0, X, -1, 0, O, 40, C.byref(n), None, None, None) == nat.E_INVALID
    assert ex(p, 0, X, 1000, -1, O, 40, C.byref(n), None, None, None) == nat.E_INVALID
    assert ex(p, 0, X, 1000, 0, O, 29, C.byref(n), None, None, None) == nat.E_INVALID and n.value == 30
    assert ex(p, 0, X, 1000, 0, None, 40, C.byref(n), None, None, None) == nat.E_INVALID
    assert ex(p, 0, None, 1000, 0, O, 40, C.byref(n), None, None, None) == nat.E_INVALID
    assert ex(p, 0, X + 2, 1000, 0, O, 40, C.byref(n), None, None, None) == nat.E_INVALID
    assert ex(p, 0, X, 1000, 0, O + 4, 40, C.byref(n), None, None, None) == nat.E_INVALID
    assert ex(p, 0, None, 64, 0, None, 0, C.byref(n), None, None, None) == nat.OK and n.value == 0
    assert ex(None, 0, X, 1000, 0, O, 40, C.byref(n), None, None, None) == nat.E_INVALID
    assert ex(p, 0, X, 1000, 0, O, 40, C.byref(n), None, None, None) == nat.OK and n.value == 30
    assert lib.spx_chan_sync(None) == nat.E_INVALID
    assert lib.spx_chan_sync(p) == nat.OK
    assert lib.spx_chan_destroy(p) == nat.OK


def test_host_call_behind_device_call_on_another_stream():
    nat, ddc, sp, _ = _mods()
    x, _ = _signal(2_000_000, "cf32", 6)
    ch = ddc.Channelizer(FS, 64, 32)
    side = nat.SideStream(0)
    d_out = ch.exec(nat.DeviceArray.from_host(x), stream=side.handle)   # enqueued only
    host = ch.exec(x)                                                   # queued behind it on the handle's own streams
    side.sync()
    assert np.array_equal(d_out.to_host().view(np.uint32), host.view(np.uint32))
    side.close()
    ch.close()


def _welch_ref(y, N, hop):
    w = np.hanning(N)
    F = (y.shape[-1] - N) // hop + 1
    fr = np.stack([y[..., f * hop: f * hop + N] * w for f in range(F)], axis=-2)
    P = np.abs(np.fft.fftshift(np.fft.fft(fr, axis=-1), axes=-1)) ** 2
    return P.sum(axis=-2), P.max(axis=-2), F


def test_chain_into_multistream_stft():
    nat, ddc, sp, _ = _mods()
    M, D, N, hop = 64, 32, 256, 128
    ch = ddc.Channelizer(FS, M, D)
    x, _ = _signal(ch.n_taps + (N + 40 * hop) * D, "cf32", 3, tones=((0.11, 0.5), (-0.27, 0.2), (9.1 / 64, 0.3)))
    n_out = ch.out_count(x.size)
    S = n_out + 13
    d_y = nat.DeviceArray((M, S), np.complex64)
    pl = sp.SpectralPlan(N, hop, "hann", sp.FMT_CF32)
    ch.exec(nat.DeviceArray.from_host(x), first_sample=FIRST, out=d_y, stream=pl.stream)
    r = pl.stft(nat.DeviceView(d_y.ptr, (M * S,), np.complex64), n_streams=M, stream_stride=S, n_samples=n_out,
                welch=True, maxhold=True)
    pl.sync()
    we, mh = r.welch_acc.to_host(), r.maxhold.to_host()
    ref_w, ref_m, F = _welch_ref(cr.channelize(x, ch.taps, M, D, FIRST), N, hop)
    assert r.n_frames == F
    for j in range(M):
        parity.check_power(we[j], ref_w[j], what=f"chain Welch channel {j}")
        parity.check_power(mh[j], ref_m[j], what=f"chain max-hold channel {j}")
    pl.close()
    ch.close()


@pytest.mark.parametrize("datatype", ["cf32_le", "ci16_le"])
def test_scan_channels(tmp_path, datatype):
    from sdr_iq_visualizer_b200 import classifier, synth
    nat, ddc, sp, sigmf_io = _mods()
    M, D, N, hop, fc = 16, 8, 64, 32, 2.4e9
    L = 300_000
    n = np.arange(L)
    k_tone, k_qpsk = 11, 4
    qpsk = synth.synth_iq(L, seed=3, snr_db=60.0, sps=64, tone_amp=0.0) * 0.3
    x = (0.4 * np.exp(2j * np.pi * (k_tone - M // 2) / M * n) + qpsk * np.exp(2j * np.pi * (k_qpsk - M // 2) / M * n)
         + 0.003 * (np.random.default_rng(2).normal(size=L) + 1j * np.random.default_rng(3).normal(size=L)))
    base = sigmf_io.write_recording(str(tmp_path / "scan"), x, FS, fc, datatype=datatype)
    rec = sigmf_io.fromfile(base)
    before = (list(classifier._CLASS_HISTORY), list(classifier._CONF_HISTORY))
    res, names = launched(lambda: sigmf_io.scan_channels(base, n_channels=M, nfft=N, hop=hop))
    _ran(names)
    assert (list(classifier._CLASS_HISTORY), list(classifier._CONF_HISTORY)) == before
    ch = ddc.Channelizer(FS, M, D, in_fmt=rec.in_fmt, in_scale=rec.in_scale)
    np.testing.assert_array_equal(res.channel_freqs, ch.channel_freqs(fc))
    assert res.out_rate == FS / D and res.band == (N // 4, N - N // 4)
    xin = np.ascontiguousarray(rec.raw_slice()) if datatype == "ci16_le" else rec.read_samples()
    y = cr.channelize(xin, ch.taps, M, D, 0, rec.in_scale)
    ref_w, _, F = _welch_ref(y, N, hop)
    assert res.n_frames == F
    pxx_ref = ref_w / (F * (FS / D) * np.sum(np.hanning(N) ** 2))
    for j in range(M):
        parity.check_power(res.pxx[j], pxx_ref[j], what=f"scan pxx channel {j}")
    lo, hi = res.band
    for j in range(M):
        pdb = res.pxx_db[j, lo:hi]
        fj = res.channel_freqs[j] + res.freqs[lo:hi]
        want = cref.features(fj, pdb)
        got = res.measurements[j]
        for key in ("noise_floor_db", "peak_db", "argmax", "snr_db", "peak_count", "n_candidates"):
            assert got[key] == want[key], (j, key)
        for d in (3, 10, 20):
            assert (got[f"first_{d}db"], got[f"last_{d}db"]) == want["edges"][d]
            assert got[f"bw{d}"] == want[f"bw{d}"]
        np.testing.assert_allclose(got["flatness"], want["flatness"], rtol=1e-11, atol=1e-300)
        np.testing.assert_allclose(got["kurtosis"], want["kurtosis"], rtol=1e-11, atol=1e-11)
        m_ref = dict(want, flatness=want["flatness"], kurtosis=want["kurtosis"])
        assert res.classification[j]["label"] == classifier.classify_from_measurements(fj, m_ref, hi - lo,
                                                                                     smooth=False)["label"]
    assert (list(classifier._CLASS_HISTORY), list(classifier._CONF_HISTORY)) == before
    snr = [m["snr_db"] for m in res.measurements]
    assert int(np.argmax(snr)) == k_tone
    assert int(np.argmax(res.pxx[k_tone])) == N // 2                   # the tone sits at the channel's centre bin
    parity._record("chan_scan_labels", datatype, tone=res.classification[k_tone]["label"],
                   qpsk=res.classification[k_qpsk]["label"], noise=res.classification[0]["label"])
    small = sigmf_io.scan_channels(base, n_channels=M, nfft=N, hop=hop, max_chunk_samples=3000)
    np.testing.assert_allclose(small.pxx, res.pxx, rtol=1e-12, atol=0)
    ch.close()
