"""GPU tests of the zoom DDC (K9 ddc_kernel): parity with the float64 oracle (tests/ddc_ref.py), exact cases, bit
identity under chunking and between memory modes and against the CPU harness of K9's math, the chain into the STFT,
process_recording(zoom=...), every error code and a host call queued behind a device call on another stream."""
import ctypes as C

import numpy as np
import pytest

from oracle import spectral_ref as sref
from tests import ddc_ref as dr, parity
from tests.test_ddc_cpu import emul, emul_ddc   # noqa: F401  (module fixture: K9's math built for the host)
from tests.test_dispatch_paths_gpu import launched

pytestmark = pytest.mark.gpu

FS = 61.44e6


def _mods():
    from sdr_iq_visualizer_b200 import _native as nat, ddc, sigmf_io, spectral as sp
    nat.require_device()
    return nat, ddc, sp, sigmf_io


def _signal(L, fmt, seed, tones=((0.11, 0.5), (-0.27, 0.2)), noise=0.05):
    """complex64 tones + noise, or interleaved int16 of it (in_scale 2^-15)."""
    rng = np.random.default_rng(seed)
    n = np.arange(L)
    x = sum(a * np.exp(2j * np.pi * f * n) for f, a in tones) + noise * (rng.normal(size=L) + 1j * rng.normal(size=L))
    if fmt == "ci16":
        return sref.to_ci16(x * 0.7), 2.0 ** -15
    return x.astype(np.complex64), 1.0


def _dev(nat, x):
    return nat.DeviceArray.from_host(x)


def _ran(names):
    assert any("ddc_kernel" in nm for nm in names), sorted(set(names))


def _parity(got, x, h, D, inc, scale, first=0, what=""):
    want = dr.ddc(x, h, D, inc, first, scale)
    bar = 1e-5 * dr.bound(h, x, scale)
    err = float(np.abs(np.asarray(got, np.complex128) - want).max()) if want.size else 0.0
    parity._record("ddc", what, outputs=int(want.size), worst_abs=err, bar=bar, margin=bar / err if err else None)
    assert got.shape == want.shape
    assert err <= bar, f"{what}: {err:.3e} > {bar:.3e}"


@pytest.mark.parametrize("fmt", ["cf32", "ci16"])
@pytest.mark.parametrize("mem", ["host", "device"])
@pytest.mark.parametrize("D,taps", [(1, "caller8192"), (4, "default"), (64, "default"), (256, "default"),
                                    (4, "caller77")])
def test_parity(fmt, mem, D, taps):
    nat, ddc, sp, _ = _mods()
    rng = np.random.default_rng(D)
    h = None if taps == "default" else rng.normal(size=int(taps[6:])) / np.sqrt(int(taps[6:]))
    T = ddc.design_taps(D).size if h is None else h.size
    L = T + 3000 * D + 17
    x, scale = _signal(L, fmt, D + (fmt == "ci16"))
    pl = ddc.DdcPlan(FS, 7.3e6, D, taps=h, in_fmt=sp.FMT_CI16 if fmt == "ci16" else sp.FMT_CF32, in_scale=scale)
    first = 1_000_003
    y, names = launched(lambda: pl.exec(x if mem == "host" else _dev(nat, x), first_sample=first))
    _ran(names)
    y = y if mem == "host" else y.to_host()
    _parity(y, x, pl.taps, D, pl.phase_inc, scale, first, f"{fmt} {mem} D={D} T={pl.n_taps}")
    pl.close()


def test_matches_cpu_harness_bit_for_bit(emul):  # noqa: F811
    """K9 computes each output in the order spx_ddc_device.cuh states: the GPU result equals the CPU harness's bits."""
    nat, ddc, sp, _ = _mods()
    for D, T, fmt in [(1, 8192, "cf32"), (3, 100, "ci16"), (64, 1607, "ci16"), (256, 6425, "cf32"), (96, 500, "cf32")]:
        rng = np.random.default_rng(T)
        h = ddc.design_taps(D) if ddc.design_taps(D).size == T else rng.normal(size=T)
        x, scale = _signal(T + 700 * D, fmt, T)
        pl = ddc.DdcPlan(FS, -3.1e6, D, taps=h, in_fmt=sp.FMT_CI16 if fmt == "ci16" else sp.FMT_CF32, in_scale=scale)
        y = pl.exec(_dev(nat, x), first_sample=77).to_host()
        want = emul_ddc(emul, x, pl.taps, D, pl.phase_inc, 77, scale)
        assert np.array_equal(y.view(np.uint32), want.view(np.uint32)), (D, T, fmt)
        pl.close()


def test_exact_cases():
    nat, ddc, sp, _ = _mods()
    x, _ = _signal(10_001, "cf32", 5)
    pl = ddc.DdcPlan(FS, 0.0, 4, taps=[1.0])
    y, names = launched(lambda: pl.exec(_dev(nat, x)).to_host())
    _ran(names)
    np.testing.assert_array_equal(y, x[::4])
    # misaligned device input: one sample past an aligned address
    big = _dev(nat, np.concatenate([[0], x]).astype(np.complex64))
    y1 = pl.exec(nat.DeviceView(big.ptr + 8, (x.size,), np.complex64)).to_host()
    np.testing.assert_array_equal(y1, x[::4])
    pl.close()
    # NaN poisons only the outputs whose window covers it
    h = ddc.design_taps(8)
    pl = ddc.DdcPlan(FS, 1e6, 8, in_fmt=sp.FMT_CF32)
    xn = x.copy()
    xn[5000] = np.nan
    y = pl.exec(_dev(nat, xn)).to_host()
    m = np.arange(y.size)
    covers = (8 * m <= 5000) & (5000 <= 8 * m + h.size - 1)
    np.testing.assert_array_equal(np.isnan(y.real), covers)
    assert not np.isnan(y[~covers]).any()
    # M = 0: nothing launched, an empty result
    assert pl.exec(x[:h.size - 1]).size == 0
    assert pl.exec(_dev(nat, x[:10])).shape == (0,)
    pl.close()


@pytest.mark.parametrize("fmt", ["cf32", "ci16"])
@pytest.mark.parametrize("D", [1, 64])
def test_chunking_bit_identical(fmt, D):
    nat, ddc, sp, _ = _mods()
    h = np.random.default_rng(1).normal(size=8192) / 90 if D == 1 else None
    pl = ddc.DdcPlan(FS, 7.3e6, D, taps=h, in_fmt=sp.FMT_CI16 if fmt == "ci16" else sp.FMT_CF32)
    T = pl.n_taps
    L = T + 20_000 * D + 3
    x, _ = _signal(L, fmt, 11)
    ew = 2 if fmt == "ci16" else 1
    base = 5 * 10 ** 9
    one = pl.exec(_dev(nat, x), first_sample=base).to_host()
    M = one.size
    cuts = [0, 1, M // 3, M // 3 + 7, M - 2, M]
    parts = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        seg = x[ew * a * D: ew * ((b - 1) * D + T)]
        parts.append(pl.exec(_dev(nat, seg), first_sample=base + a * D).to_host())
    assert np.array_equal(np.concatenate(parts).view(np.uint32), one.view(np.uint32))
    pl.close()


def test_host_pieces_bit_identical_to_device(monkeypatch):
    nat, ddc, sp, _ = _mods()
    monkeypatch.setenv("SPX_H2D_PIECE_BYTES", "65536")
    x, scale = _signal(300_000, "ci16", 4)
    pl = ddc.DdcPlan(FS, 2.5e6, 8, in_fmt=sp.FMT_CI16, in_scale=scale)
    host = pl.exec(x, first_sample=9)
    assert pl.last_h2d_bytes > x.nbytes       # several pieces with halos
    dev = pl.exec(_dev(nat, x), first_sample=9).to_host()
    assert np.array_equal(host.view(np.uint32), dev.view(np.uint32))
    pl.close()


def _welch_ref(y, N, hop):
    w = np.hanning(N)
    F = (y.size - N) // hop + 1
    fr = np.stack([y[f * hop: f * hop + N] * w for f in range(F)])
    return (np.abs(np.fft.fftshift(np.fft.fft(fr, axis=1), axes=1)) ** 2).sum(axis=0)


def test_chain_welch_and_alias_rejection():
    nat, ddc, sp, _ = _mods()
    D, N = 64, 1024
    fo = FS / D
    shift = 7.3e6
    # an in-band tone at +0.25 fo from the zoom centre, and one at +0.7 fo that aliases to -0.3 fo, inside the passband
    f_in, f_alias = 0.25 * fo, 0.7 * fo
    tones = (((shift + f_in) / FS, 0.3), ((shift + f_alias) / FS, 0.3))
    L = 64 * N * 40 + 2000
    dd = ddc.DdcPlan(FS, shift, D)
    pl = sp.SpectralPlan(N, N // 4, "hann", sp.FMT_CF32)
    freqs = sp.freq_axis(N, fo, 0.0)
    j_alias = int(np.argmin(np.abs(freqs - (f_alias - fo))))
    for noise in (3e-2, 0.0):
        x, _ = _signal(L, "cf32", 3, tones=tones, noise=noise)
        y, names = launched(lambda: dd.exec(_dev(nat, x)))
        _ran(names)
        welch = pl.stft(y, welch=True).welch_acc.to_host()[0]
        ref = _welch_ref(dr.ddc(x, dd.taps, D, dd.phase_inc), N, N // 4)
        if noise:
            parity.check_power(welch, ref, what="zoomed Welch vs oracle DDC + Welch")
            assert abs(freqs[int(np.argmax(welch))] - f_in) <= fo / N
        else:   # the alias bin: >= 78 dB under the in-band tone, as the oracle predicts
            sup = 10 * np.log10(welch.max() / welch[j_alias])
            sup_ref = 10 * np.log10(ref.max() / ref[j_alias])
            parity._record("ddc_alias", "alias suppression dB", got=float(sup), oracle=float(sup_ref))
            assert sup >= 78.0 and abs(sup - sup_ref) < 1.0, (sup, sup_ref)
    pl.close()
    dd.close()


@pytest.mark.parametrize("datatype", ["cf32_le", "ci16_le"])
def test_process_recording_zoom(tmp_path, datatype):
    nat, ddc, sp, sigmf_io = _mods()
    fc, shift, D, N, hop = 2.4e9, -5.0e6, 16, 256, 64
    x, _ = _signal(400_000, "cf32", 8, tones=((shift / FS + 0.002, 0.4), (0.3, 0.4)))
    base = sigmf_io.write_recording(str(tmp_path / "z"), x, FS, fc, datatype=datatype)
    rec = sigmf_io.fromfile(base)
    res, names = launched(lambda: sigmf_io.process_recording(base, nfft=N, hop=hop, waterfall=True, vmin=-120, vmax=0,
                                                               max_chunk_samples=50_000, zoom=(fc + shift, D),
                                                               persistence=True, overview=(8, 64)))
    _ran(names)
    dd = ddc.DdcPlan(FS, shift, D, in_fmt=rec.in_fmt, in_scale=rec.in_scale)
    xin = np.ascontiguousarray(rec.raw_slice()) if datatype == "ci16_le" else rec.read_samples()
    y = dd.exec(_dev(nat, xin))
    pl = sp.SpectralPlan(N, hop, "hann", sp.FMT_CF32)
    r = pl.stft(y, wf_rows=True, welch=True, maxhold=True, vmin=-120, vmax=0)
    F = r.n_frames
    assert res.n_frames == F and res.wf_rows.shape == (F, N)
    assert np.array_equal(res.wf_rows, r.wf_rows.to_host())
    pxx_ref, _ = pl.welch_finalize(r.welch_acc.to_host()[0], F, FS / D, want_db=False)
    np.testing.assert_allclose(res.pxx, pxx_ref, rtol=1e-12)
    np.testing.assert_array_equal(res.maxhold, r.maxhold.to_host()[0])
    assert res.persistence.sum(axis=0).tolist() == [F] * N
    assert res.sample_rate == FS / D and res.center_freq == fc + dd.shift_hz
    np.testing.assert_array_equal(res.freqs, sp.freq_axis(N, FS / D, fc + dd.shift_hz))
    assert res.zoom == (dd.shift_hz, D, dd.n_taps) and res.overview_db.shape[1] == N // res.overview_bins_per_col
    pl.close()
    dd.close()


def test_errors():
    nat, ddc, sp, _ = _mods()
    lib = nat.lib()
    h = (C.c_double * 3)(1.0, 2.0, 1.0)

    def create(**kw):
        cfg = nat.spx_ddc_config(C.sizeof(nat.spx_ddc_config), 0, 0, 1.0, 2, 3, C.cast(h, C.c_void_p), 0)
        for k, v in kw.items():
            setattr(cfg, k, v)
        p = C.c_void_p()
        return lib.spx_ddc_create(C.byref(p), C.byref(cfg)), p

    for kw in (dict(decim=0), dict(n_taps=0), dict(n_taps=8193), dict(taps=None), dict(in_fmt=5), dict(device=99),
               dict(struct_size=4)):
        rc, _ = create(**kw)
        assert rc == nat.E_INVALID, kw
    rc, _ = create(n_taps=8192, taps=C.cast((C.c_double * 8192)(), C.c_void_p), decim=4096)
    assert rc == nat.E_UNSUPPORTED
    assert lib.spx_ddc_create(None, None) == nat.E_INVALID
    rc, p = create()
    assert rc == nat.OK
    x = np.zeros(64, np.complex64)
    out = np.zeros(64, np.complex64)
    n = C.c_int64()
    ex = lib.spx_ddc_exec
    assert ex(p, 7, x.ctypes.data, 64, 0, out.ctypes.data, C.byref(n), None, None, None) == nat.E_INVALID
    assert ex(p, 0, x.ctypes.data, -1, 0, out.ctypes.data, C.byref(n), None, None, None) == nat.E_INVALID
    assert ex(p, 0, x.ctypes.data, 64, -1, out.ctypes.data, C.byref(n), None, None, None) == nat.E_INVALID
    assert ex(p, 0, x.ctypes.data, 64, 0, None, C.byref(n), None, None, None) == nat.E_INVALID
    assert ex(p, 0, None, 64, 0, out.ctypes.data, C.byref(n), None, None, None) == nat.E_INVALID
    assert ex(p, 0, x.ctypes.data + 2, 64, 0, out.ctypes.data, C.byref(n), None, None, None) == nat.E_INVALID
    assert ex(p, 0, x.ctypes.data, 64, 0, out.ctypes.data + 2, C.byref(n), None, None, None) == nat.E_INVALID
    assert ex(p, 0, None, 2, 0, None, C.byref(n), None, None, None) == nat.OK and n.value == 0
    assert ex(None, 0, x.ctypes.data, 64, 0, out.ctypes.data, C.byref(n), None, None, None) == nat.E_INVALID
    assert lib.spx_ddc_sync(None) == nat.E_INVALID
    assert lib.spx_ddc_sync(p) == nat.OK
    assert lib.spx_ddc_destroy(p) == nat.OK


def test_host_call_behind_device_call_on_another_stream():
    nat, ddc, sp, _ = _mods()
    x, _ = _signal(2_000_000, "cf32", 6)
    pl = ddc.DdcPlan(FS, 1e6, 64)
    side = nat.SideStream(0)
    d_x = _dev(nat, x)
    d_out = pl.exec(d_x, stream=side.handle)            # enqueued only
    host = pl.exec(x)                                    # queued behind it on the handle's own streams
    side.sync()
    assert np.array_equal(d_out.to_host().view(np.uint32), host.view(np.uint32))
    side.close()
    pl.close()
