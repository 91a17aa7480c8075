"""GPU tests of the pooled spectrogram (``SpectralPlan.stft(pool=...)`` / ``spx_stft_exec_pooled``, ``pool_finalize``):
waterfall rows of K frames x B bins pooled by ``pool_kernel`` with the mean or max detector.

Max mode keeps the largest float32 dB value of each cell, so it is checked bit for bit against ``tests.pool_ref`` of the
dB rows the same call returned; mean mode sums recovered power in float64 and is held to 5e-6 relative in power; levels
are bit-exact against ``waterfall_u8`` of the returned pooled dB.  The pooled dB also passes the dB-row parity rule against
the float64 oracle.  Every case asserts from the CUDA profiler's kernel names which STFT family ran and that the pooling
kernel ran."""
import ctypes as C

import numpy as np
import pytest

from oracle import spectral_ref as sref
from tests import parity
from tests import pool_ref as pr
from tests.test_dispatch_paths_gpu import K2_ROWS, _cut, _host, _iq, _oracle, count, launched
from tests.test_persistence_gpu import SHAPES, VRANGE, _input, _place

pytestmark = pytest.mark.gpu

POOL = r"\bpool_kernel<"
# float32 exponent of the power recovery (2 ln 10 |d/20| 2^-24, 3.6e-6 at 260 dB) plus float partial sums of 4 rows
MEAN_RTOL = 5e-6


def _family(name):
    """K2v2 has no float-row output: N = 65536 with pooling runs K2 (big_rows_kernel), as N = 16384 does."""
    n, hop, fmt, F, fam = SHAPES[name]
    return K2_ROWS if n >= 16384 else fam


@pytest.fixture(scope="module")
def sp():
    from sdr_iq_visualizer_b200 import _native, spectral
    assert _native.device_count() > 0, "GPU tests need a CUDA device (no CPU fallback exists)"
    return spectral


def _pw(db):
    return pr.db_to_power(np.asarray(db, np.float64))


def check_against_rows(got_db, db_rows, K, B, mode, S, what=""):
    """max: bit-identical to pool_ref of the call's rows; mean: <= MEAN_RTOL relative in power."""
    want = pr.pool_db_rows(db_rows, K, B, mode, S)
    got_db = np.asarray(got_db)
    assert got_db.shape == want.shape and got_db.dtype == np.float32, (got_db.shape, want.shape)
    if mode == "max":
        np.testing.assert_array_equal(got_db, want.astype(np.float32), err_msg=what)
        return 0.0
    pw, pw_ref = _pw(got_db), _pw(want)
    rel = float((np.abs(pw - pw_ref) / np.maximum(pw_ref, 1e-30)).max()) if pw.size else 0.0
    parity._record("pooled_mean_vs_rows", what, cells=int(pw.size), worst_rel_power=rel)
    assert rel <= MEAN_RTOL, f"{what}: {rel:.3e} relative in power"
    return rel


def _pooled_call(sp, pl, src, S, K, B, mode, vmin, vmax, **kw):
    r, names = launched(lambda: pl.stft(src, n_streams=S, pool=(K, B, mode), vmin=vmin, vmax=vmax, **kw))
    pl.sync()
    db, wf = pl.pool_finalize(r.pool_acc, r.n_frames, K, B, mode, db=True, wf=True, vmin=vmin, vmax=vmax, n_streams=S)
    pl.sync()
    return r, names, _host(db), _host(wf)


# ----------------------------------------------------------------------------- 1 + 2: against the call's rows and the oracle
@pytest.mark.parametrize("mem", ["host", "device"])
@pytest.mark.parametrize("S", [1, 3])
@pytest.mark.parametrize("name", sorted(SHAPES))
def test_pooled_matches_the_calls_rows(sp, name, S, mem):
    """One call with caller dB rows plus pooling, both detectors: max bit-identical, mean within 5e-6 in power, levels
    bit-identical to waterfall_u8 of the pooled dB.  With S = 1 on the device the pooled dB also passes the dB-row rule
    against pool_ref of the float64 oracle's power, and the levels the u8 rule."""
    n, hop, fmt, F, _ = SHAPES[name]
    fam = _family(name)
    vmin, vmax = VRANGE[fmt]
    x, L = _input(n, hop, fmt, max(F, 12), S, seed=n + S)
    F = sref.frame_count(L, n, hop)
    K = F // 3 + 1
    while F % K == 0:               # a partial last row
        K += 1
    B = 8
    pl = sp.SpectralPlan(n, hop, "hann", fmt)
    src = _place(x, mem)
    for mode in ("max", "mean"):
        r, names, db, wf = _pooled_call(sp, pl, src, S, K, B, mode, vmin, vmax, db_rows=True)
        assert r.n_frames == F and F % K != 0
        assert count(names, fam) > 0 and count(names, POOL) > 0, names
        rows = _host(r.db_rows)
        check_against_rows(db, rows, K, B, mode, S, what=f"{name} S={S} {mem} {mode}")
        np.testing.assert_array_equal(wf, sref.waterfall_u8(db, vmin, vmax))
        if S == 1 and mem == "device":
            X, _, _ = _oracle(x, n, hop, "hann", fmt, 1, list(range(F)))
            P = X.real ** 2 + X.imag ** 2
            ref_p = pr.pool_power(P, K, B, mode)[0]
            parity.check_db_rows(db[0], ref_p, eps=pr.EPS, what=f"pooled {mode} {name} vs float64")
            parity.check_u8(wf[0], pr.pool_db(P, K, B, mode)[0], vmin, vmax, what=f"pooled {mode} {name} u8")
    pl.close()


# ----------------------------------------------------------------------------- 3: batches and pieces
@pytest.mark.parametrize("mode", ["max", "mean"])
@pytest.mark.parametrize("mem", ["host", "device"])
@pytest.mark.parametrize("name", ["K1v2 ci16 4096", "K5 1000", "K2v2 65536"])
def test_batches_and_pieces(sp, monkeypatch, name, mem, mode):
    """Plan-owned float rows in batches of 5 frames (host: pieces of the H2D pipeline too): with K = 16 a row spans
    three or more batches, with K = 2 a batch spans several rows, and the last batch is short.  The accumulator matches
    the single-batch call with caller rows (max bit-identical), and a host call copies back only the accumulator."""
    n, hop, fmt, _, _ = SHAPES[name]
    fam = _family(name)
    vmin, vmax = VRANGE[fmt]
    S = 3 if mem == "device" else 1
    x, L = _input(n, hop, fmt, 53, S, seed=21)
    F = sref.frame_count(L, n, hop)
    src = _place(x, mem)
    ref_pl = sp.SpectralPlan(n, hop, "hann", fmt)
    fb = 5
    monkeypatch.setenv("SPX_POOL_ROWS_BYTES", str(S * n * 4 * fb))
    monkeypatch.setenv("SPX_H2D_PIECE_BYTES", str(max(65536, 12 * hop * (4 if fmt else 8))))
    pl = sp.SpectralPlan(n, hop, "hann", fmt)
    monkeypatch.delenv("SPX_POOL_ROWS_BYTES")
    monkeypatch.delenv("SPX_H2D_PIECE_BYTES")
    assert F % fb != 0
    for K in (16, 2):
        B = 8
        r0 = ref_pl.stft(src, n_streams=S, db_rows=True, pool=(K, B, mode))
        r, names = launched(lambda: pl.stft(src, n_streams=S, pool=(K, B, mode)))
        assert count(names, fam) > 0, names
        assert count(names, POOL) >= -(-F // fb), names
        a, a0 = _get(pl, r.pool_acc), _get(ref_pl, r0.pool_acc)
        if mode == "max":
            np.testing.assert_array_equal(a, a0)
        else:
            np.testing.assert_allclose(a, a0, rtol=1e-6)
        check_against_rows(pl.pool_finalize(a, F, K, B, mode, n_streams=S)[0], _host(r0.db_rows), K, B, mode, S,
                           what=f"batches {name} {mem} {mode} K={K}")
        if mem == "host":
            assert r.d2h_bytes == S * (-(-F // K)) * (n // B) * 8
            rw = pl.stft(src, pool=(K, B, mode), welch=True, wf_rows=True, vmin=vmin, vmax=vmax)
            assert rw.d2h_bytes == a.nbytes + n * 8 + F * n
            # the STFT writes dB rows too, so N = 65536 runs K2 here: compare with K2's uint8 rows
            want = ref_pl.stft(x, wf_rows=True, db_rows=True, vmin=vmin, vmax=vmax).wf_rows
            np.testing.assert_array_equal(rw.wf_rows, want)
    pl.close(); ref_pl.close()


def _get(pl, a):
    pl.sync()
    return _host(a)


# ----------------------------------------------------------------------------- 4: chunked calls
@pytest.mark.parametrize("mode", ["max", "mean"])
@pytest.mark.parametrize("mem", ["host", "device"])
def test_chunked_calls(sp, mem, mode):
    """Three calls on consecutive pieces of a capture (cut as SigMFRecording.frame_chunks cuts, in the middle of a pooled
    row), with pool_first_frame and accumulate=True, equal one call on the whole."""
    from sdr_iq_visualizer_b200 import _native as nat
    n, hop, fmt = 4096, 1024, 1
    F, K, B = 61, 7, 16
    x = _iq(n + hop * (F - 1), fmt, seed=5)
    cuts = [0, 17, 38, F]               # 17 and 38 are inside rows 2 and 5
    pl = sp.SpectralPlan(n, hop, "hann", fmt)
    whole = pl.stft(_place(x, mem), pool=(K, B, mode))
    G = -(-F // K)
    acc = np.empty((1, G, n // B)) if mem == "host" else nat.DeviceArray((1, G, n // B), np.float64)
    for i in range(3):
        f0, f1 = cuts[i], cuts[i + 1]
        piece = _cut(x, fmt, f0 * hop, (f1 - 1) * hop + n)
        r = pl.stft(_place(piece, mem), pool=(K, B, mode), pool_acc=acc, pool_first_frame=f0, accumulate=i > 0)
        assert r.n_frames == f1 - f0
    a, w = _get(pl, acc), _get(pl, whole.pool_acc)
    if mode == "max":
        np.testing.assert_array_equal(a, w)
    else:
        np.testing.assert_allclose(a, w, rtol=1e-6)   # float partials over other groupings of rows
    pl.close()


@pytest.mark.parametrize("fmt", [0, 1])
def test_process_recording_overview(sp, tmp_path, fmt):
    """process_recording(overview=...) over small chunks equals one device call on the whole file."""
    from sdr_iq_visualizer_b200 import _native as nat, sigmf_io
    n, hop = 1024, 256
    x = _iq(200_000, fmt, seed=9)
    dt = "ci16_le" if fmt else "cf32_le"
    base = sigmf_io.write_recording(str(tmp_path / f"cap{fmt}"), x, 1e6, 100e6, datatype=dt)
    vmin, vmax = -120.0, 0.0
    for mode in ("mean", "max"):
        rs = sigmf_io.process_recording(base, nfft=n, hop=hop, overview=(40, 100), overview_mode=mode, vmin=vmin,
                                        vmax=vmax, max_chunk_samples=30_000)
        K, B = rs.overview_frames_per_row, rs.overview_bins_per_col
        assert (K, B) == sigmf_io.overview_pooling(rs.n_frames, n, 40, 100)
        assert rs.wf_rows is None and rs.overview_db.shape == (-(-rs.n_frames // K), n // B)
        pl = sp.SpectralPlan(n, hop, "hann", fmt, in_scale=2.0 ** -15 if fmt else 1.0)
        r = pl.stft(nat.DeviceArray.from_host(x), pool=(K, B, mode))
        db, wf = pl.pool_finalize(r.pool_acc, r.n_frames, K, B, mode, wf=True, vmin=vmin, vmax=vmax)
        pl.sync()
        if mode == "max":
            np.testing.assert_array_equal(rs.overview_db, db.to_host()[0])
        else:
            np.testing.assert_allclose(_pw(rs.overview_db), _pw(db.to_host()[0]), rtol=1e-6)
        np.testing.assert_array_equal(rs.overview_wf, sref.waterfall_u8(rs.overview_db, vmin, vmax))
        pl.close()


# ----------------------------------------------------------------------------- 5: edges and errors
@pytest.mark.parametrize("mem", ["host", "device"])
def test_k_b_one_gives_the_rows(sp, mem):
    n, hop, fmt = 4096, 1024, 1
    x, L = _input(n, hop, fmt, 20, 1, seed=3)
    pl = sp.SpectralPlan(n, hop, "hann", fmt)
    for mode in ("max", "mean"):
        r, _, db, _ = _pooled_call(sp, pl, _place(x, mem), 1, 1, 1, mode, -40.0, 90.0, db_rows=True)
        rows = _host(r.db_rows)
        if mode == "max":
            np.testing.assert_array_equal(db[0], rows)
        else:
            assert np.abs(db[0].astype(np.float64) - rows).max() <= 2e-5
    pl.close()


@pytest.mark.parametrize("mem", ["host", "device"])
def test_edges(sp, mem):
    """K > F (one partial row), F = 0 (zero rows, no error), B = N (a total-power strip)."""
    n, hop = 1024, 512
    pl = sp.SpectralPlan(n, hop, "hann")
    x = _iq(n + hop * 9, 0, seed=4)
    for mode in ("max", "mean"):
        r, _, db, _ = _pooled_call(sp, pl, _place(x, mem), 1, 50, 4, mode, -40.0, 90.0, db_rows=True)
        assert db.shape == (1, 1, n // 4)
        check_against_rows(db, _host(r.db_rows), 50, 4, mode, 1, what=f"K > F {mode}")
        r, _, db, _ = _pooled_call(sp, pl, _place(x, mem), 1, 3, n, mode, -40.0, 90.0, db_rows=True)
        assert db.shape == (1, 4, 1)
        check_against_rows(db, _host(r.db_rows), 3, n, mode, 1, what=f"B = N {mode}")
        r, _, db, wf = _pooled_call(sp, pl, _place(x[: n - 1], mem), 1, 3, 4, mode, -40.0, 90.0)
        assert r.n_frames == 0 and db.shape == (1, 0, n // 4) and wf.shape == (1, 0, n // 4)
    pl.close()


def test_bluestein_bins_and_rejection(sp):
    from sdr_iq_visualizer_b200 import _native as nat
    n, hop = 1000, 250
    x, L = _input(n, hop, 0, 30, 1, seed=8)
    pl = sp.SpectralPlan(n, hop, "hann")
    for mode in ("max", "mean"):
        r, names, db, _ = _pooled_call(sp, pl, nat.DeviceArray.from_host(x), 1, 4, 8, mode, -40.0, 90.0, db_rows=True)
        assert count(names, SHAPES["K5 1000"][4]) > 0 and count(names, POOL) > 0
        check_against_rows(db, _host(r.db_rows), 4, 8, mode, 1, what=f"Bluestein {mode}")
    with pytest.raises(ValueError):
        pl.stft(x, pool=(4, 3, "mean"))
    a = nat.spx_stft_args(); a.struct_size = C.sizeof(nat.spx_stft_args)
    a.mem, a.in_, a.n_samples, a.stream_stride, a.n_streams = nat.MEM_HOST, x.ctypes.data, L, L, 1
    acc = np.zeros(1000)
    p = nat.spx_pool_args(C.sizeof(nat.spx_pool_args), 0, 4, 3, 0, 0, 8, acc.ctypes.data)
    assert nat.lib().spx_stft_exec_pooled(pl._h, C.byref(a), C.byref(p)) == nat.E_INVALID
    pl.close()


def test_nan_frame(sp):
    """A NaN input sample makes its frames' dB rows NaN: those mean rows are NaN, max rows skip them."""
    from sdr_iq_visualizer_b200 import _native as nat
    n, hop = 256, 256
    x = _iq(n * 8, 0, seed=6)
    x[3 * n + 5] = np.nan
    pl = sp.SpectralPlan(n, hop, "hann")
    for mode in ("max", "mean"):
        r, _, db, _ = _pooled_call(sp, pl, nat.DeviceArray.from_host(x), 1, 2, 4, mode, -40.0, 90.0, db_rows=True)
        rows = _host(r.db_rows)
        assert np.isnan(rows[3]).all()
        if mode == "mean":
            assert np.isnan(db[0, 1]).all() and not np.isnan(db[0, [0, 2, 3]]).any()
        else:
            np.testing.assert_array_equal(db[0, 1], rows[2].reshape(-1, 4).max(axis=1))
            check_against_rows(db, rows, 2, 4, mode, 1, what="NaN max")
    pl.close()


def test_errors(sp):
    from sdr_iq_visualizer_b200 import _native as nat
    n = 1024
    pl = sp.SpectralPlan(n, n, "hann")
    x = _iq(4 * n, 0, seed=2)
    acc = np.zeros((1, 4, n // 4))

    def call(mode=0, K=1, B=4, first=0, rows=4, size=None, peer=0, wf=None, vmin=-40.0, vmax=60.0, mem=nat.MEM_HOST,
             src=x, accp=acc):
        a = nat.spx_stft_args(); a.struct_size = C.sizeof(nat.spx_stft_args)
        a.mem, a.in_, a.n_samples, a.stream_stride, a.n_streams = mem, nat.as_ptr(src)[0], 4 * n, 4 * n, 1
        a.vmin, a.vmax, a.peer_outputs = vmin, vmax, peer
        a.wf_rows = wf
        p = nat.spx_pool_args(size or C.sizeof(nat.spx_pool_args), mode, K, B, 0, first, rows, nat.as_ptr(accp)[0])
        return nat.lib().spx_stft_exec_pooled(pl._h, C.byref(a), C.byref(p))

    assert call() == nat.OK
    for kw in (dict(K=0), dict(B=0), dict(B=3), dict(mode=2), dict(first=-1), dict(first=1), dict(rows=3),
               dict(size=8), dict(wf=np.zeros((4, n), np.uint8).ctypes.data, vmin=5.0, vmax=5.0)):
        assert call(**kw) == nat.E_INVALID, kw
    d_x, d_acc = nat.DeviceArray.from_host(x), nat.DeviceArray((1, 4, n // 4), np.float64)
    assert call(peer=1, mem=nat.MEM_DEVICE, src=d_x, accp=d_acc) == nat.E_UNSUPPORTED
    L = nat.lib()
    f = lambda **k: L.spx_pool_finalize(pl._h, nat.MEM_HOST, k.get("mode", 0), acc.ctypes.data, 1, k.get("rows", 4),
                                        4, 1, k.get("B", 4), None, k.get("wf", None), k.get("vmin", -40.0), 60.0, None)
    out = np.zeros(acc.size, np.uint8)
    assert f() == nat.OK
    for kw in (dict(rows=3), dict(rows=5), dict(B=3), dict(mode=7), dict(wf=out.ctypes.data, vmin=60.0)):
        assert f(**kw) == nat.E_INVALID, kw
    pl.close()


def test_queued_behind_a_device_call_on_another_stream(sp):
    """A pooled host-memory call (plan-owned row buffer, s_compute) right behind a device-resident pooled call on a side
    stream of the same plan, with no synchronisation in between: both results are right."""
    from sdr_iq_visualizer_b200 import _native as nat
    n, hop, fmt = 4096, 1024, 1
    x, L = _input(n, hop, fmt, 400, 1, seed=12)
    pl = sp.SpectralPlan(n, hop, "hann", fmt)
    ref = pl.stft(x, db_rows=True, pool=(9, 4, "max"))
    side = nat.SideStream()
    d_x = nat.DeviceArray.from_host(x)
    r1 = pl.stft(d_x, pool=(9, 4, "max"), stream=side.handle)
    r2 = pl.stft(x, pool=(9, 4, "max"))
    side.sync()
    np.testing.assert_array_equal(r1.pool_acc.to_host(), ref.pool_acc)
    np.testing.assert_array_equal(r2.pool_acc, ref.pool_acc)
    side.close()
    pl.close()
