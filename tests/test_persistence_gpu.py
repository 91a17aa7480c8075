"""GPU tests of the persistence spectrum (``SpectralPlan.stft(persistence=...)`` / ``spx_stft_exec_persistence``):
frames per uint8 waterfall level and bin, counted by ``persist_kernel``.

The counts are integers computed from the uint8 rows the same call produces, so they are checked bit-exactly against
``tests.persistence_ref.persistence`` of those rows; the rows themselves are held to the usual u8 parity rule against the float64
oracle.  Every case asserts from the CUDA profiler's kernel names which STFT family produced the rows and that the
histogram kernel ran."""
import ctypes as C

import numpy as np
import pytest

from oracle import spectral_ref as sref
from tests import parity
from tests import persistence_ref as pref
from tests.test_dispatch_paths_gpu import (BLU_PRE, K1_STAGED, K1V2, K2_COLS_BULK, K2V2, _cut, _host, _iq,
                                           _oracle, count, launched)

pytestmark = pytest.mark.gpu

PERSIST = r"\bpersist_kernel\b"
VRANGE = {0: (-40.0, 90.0), 1: (20.0, 130.0)}   # vmin, vmax per input format (cf32, ci16)

# name -> (nfft, hop, fmt, frames, family pattern)
SHAPES = {
    "K1v2 ci16 4096": (4096, 1024, 1, 40, K1V2),
    "K1v2 cf32 1024": (1024, 1024, 0, 60, K1V2),
    "K1 512": (512, 128, 0, 80, K1_STAGED),
    "K1 8192": (8192, 4096, 0, 20, K1_STAGED),
    "K2v2 65536": (65536, 32768, 0, 5, K2V2),
    "K2 16384": (16384, 8192, 0, 8, K2_COLS_BULK),
    "K5 1000": (1000, 250, 0, 30, BLU_PRE),
}


@pytest.fixture(scope="module")
def sp():
    from sdr_iq_visualizer_b200 import _native, spectral
    assert _native.device_count() > 0, "GPU tests need a CUDA device (no CPU fallback exists)"
    return spectral


def _input(n, hop, fmt, F, S, seed):
    """S streams of L samples, L a multiple of 256 so that every stream keeps the base alignment of the buffer."""
    L = -(-(n + hop * (F - 1)) // 256) * 256
    return _iq(L, fmt, seed, S=S), L


def _place(x, mem):
    from sdr_iq_visualizer_b200 import _native as nat
    return x if mem == "host" else nat.DeviceArray.from_host(x)


def _get(pl, a):
    """A result on the host once the plan's (non-blocking) streams are done with it."""
    pl.sync()
    return _host(a)


def _counts_of_rows(r, S):
    return pref.persistence(_host(r.wf_rows), S)


def _with_rows(sp, name, S, mem, seed=0):
    """One call with wf_rows and persistence; the counts must be the histogram of those very rows."""
    n, hop, fmt, F, fam = SHAPES[name]
    vmin, vmax = VRANGE[fmt]
    x, L = _input(n, hop, fmt, F, S, seed=n + S + seed)
    F = sref.frame_count(L, n, hop)   # L was rounded up
    pl = sp.SpectralPlan(n, hop, "hann", fmt)
    src = _place(x, mem)
    r, names = launched(lambda: pl.stft(src, n_streams=S, wf_rows=True, persistence=True, vmin=vmin, vmax=vmax))
    assert r.n_frames == F
    assert count(names, fam) > 0 and count(names, PERSIST) > 0, names
    c = _host(r.persistence)
    assert c.shape == (S, 256, n) and c.dtype == np.uint32
    np.testing.assert_array_equal(c, _counts_of_rows(r, S))
    np.testing.assert_array_equal(c.sum(axis=1), F)
    return pl, x, r, names


# ----------------------------------------------------------------------------- 1 + 2: bit-exact, and against float64
@pytest.mark.parametrize("mem", ["host", "device"])
@pytest.mark.parametrize("S", [1, 3])
@pytest.mark.parametrize("name", sorted(SHAPES))
def test_counts_match_the_calls_rows(sp, name, S, mem):
    """Counts equal persistence_ref.persistence of the rows the same call returned, for every family, S = 1 and 3, host and
    device memory.  With S = 1 on the device the rows also pass the u8 parity rule against the float64 oracle, and the
    counts differ from the histogram of the oracle's levels by at most two per accepted u8 mismatch in each column."""
    pl, x, r, _ = _with_rows(sp, name, S, mem)
    if S == 1 and mem == "device":
        n, hop, fmt, _, _ = SHAPES[name]
        F = r.n_frames
        vmin, vmax = VRANGE[fmt]
        X, _, _ = _oracle(x, n, hop, "hann", fmt, 1, list(range(F)))
        db = sref.amplitude_db(X)
        rows = _host(r.wf_rows)
        parity.check_u8(rows, db, vmin, vmax, what=f"persistence {name} u8")
        want = pref.persistence(sref.waterfall_u8(db, vmin, vmax))[0]
        l1 = np.abs(_host(r.persistence)[0].astype(np.int64) - want.astype(np.int64)).sum(axis=0)
        mism = (rows != sref.waterfall_u8(db, vmin, vmax)).sum(axis=0)
        parity._record("persistence", f"{name} vs float64 levels", bins=int(rows.size), worst_l1=int(l1.max()),
                       u8_mismatches=int(mism.sum()))
        assert (l1 <= 2 * mism).all()
    pl.close()


# ----------------------------------------------------------------------------- 3: scratch batches
@pytest.mark.parametrize("name,with_db", [("K1v2 ci16 4096", False), ("K2v2 65536", False), ("K5 1000", False),
                                          ("K1 512", True)])
def test_scratch_batches(sp, monkeypatch, name, with_db):
    """Device path without caller rows, S = 3, through a row buffer of 7 frames of all streams (two full batches and a
    short last one, or more): counts identical to the call with rows, the histogram kernel once per batch, the same
    STFT family.  With float rows the batches run one stream at a time."""
    from sdr_iq_visualizer_b200 import _native as nat
    S = 3
    n, hop, fmt, F, fam = SHAPES[name]
    F = max(F, 16)
    vmin, vmax = VRANGE[fmt]
    x, L = _input(n, hop, fmt, F, S, seed=7)
    F = sref.frame_count(L, n, hop)
    d_x = nat.DeviceArray.from_host(x)
    ref_pl = sp.SpectralPlan(n, hop, "hann", fmt)
    r0, names0 = launched(lambda: ref_pl.stft(d_x, n_streams=S, wf_rows=True, db_rows=with_db, welch=True,
                                              persistence=True, vmin=vmin, vmax=vmax))
    per = 1 if with_db else S
    fb = 7
    monkeypatch.setenv("SPX_PERSIST_ROWS_BYTES", str(per * n * fb))
    pl = sp.SpectralPlan(n, hop, "hann", fmt)
    monkeypatch.delenv("SPX_PERSIST_ROWS_BYTES")
    r, names = launched(lambda: pl.stft(d_x, n_streams=S, db_rows=with_db, welch=True, persistence=True, vmin=vmin,
                                        vmax=vmax))
    batches = -(-F // fb) * (S // per)
    assert r.n_frames == F and F % fb != 0 and batches >= 3
    assert count(names, PERSIST) == batches, names
    assert count(names, fam) > 0 and count(names0, fam) > 0, (names, names0)
    np.testing.assert_array_equal(r.persistence.to_host(), r0.persistence.to_host())
    np.testing.assert_array_equal(r.persistence.to_host(), _counts_of_rows(r0, S))
    np.testing.assert_allclose(r.welch_acc.to_host(), r0.welch_acc.to_host(), rtol=1e-6)
    if with_db:
        np.testing.assert_array_equal(r.db_rows.to_host(), r0.db_rows.to_host())
    pl.close(); ref_pl.close()


# ----------------------------------------------------------------------------- 4: host path without rows
@pytest.mark.parametrize("name", ["K1v2 ci16 4096", "K2v2 65536", "K5 1000"])
def test_host_path_without_rows(sp, name):
    """Host memory, no rows requested: the counts equal the call with rows, and only the counts (and the accumulators)
    come back over PCIe."""
    S = 3
    pl, x, r0, _ = _with_rows(sp, name, S, "host")
    n, hop, fmt, _, fam = SHAPES[name]
    vmin, vmax = VRANGE[fmt]
    r, names = launched(lambda: pl.stft(x, n_streams=S, persistence=True, vmin=vmin, vmax=vmax))
    assert count(names, fam) > 0 and count(names, PERSIST) > 0, names
    np.testing.assert_array_equal(r.persistence, r0.persistence)
    assert r.d2h_bytes == S * 256 * n * 4
    ra = pl.stft(x, n_streams=S, persistence=True, welch=True, maxhold=True, vmin=vmin, vmax=vmax)
    np.testing.assert_array_equal(ra.persistence, r0.persistence)
    assert ra.d2h_bytes == S * 256 * n * 4 + S * n * 8 + S * n * 4
    pl.close()


# ----------------------------------------------------------------------------- 5: accumulate
@pytest.mark.parametrize("mem", ["host", "device"])
def test_accumulate_halves(sp, mem):
    """Two calls on the halves of a capture, cut as SigMFRecording.frame_chunks cuts (the second half starts at its
    first frame and carries the N - hop halo), the second with accumulate=True, equal one call on the whole."""
    n, hop, fmt = 4096, 1024, 1
    vmin, vmax = VRANGE[fmt]
    F = 50
    x = _iq(n + hop * (F - 1), fmt, seed=5)
    F1 = 23
    a = _cut(x, fmt, 0, (F1 - 1) * hop + n)
    b = _cut(x, fmt, F1 * hop, n + hop * (F - 1))
    pl = sp.SpectralPlan(n, hop, "hann", fmt)
    whole = pl.stft(_place(x, mem), persistence=True, vmin=vmin, vmax=vmax)
    c = pl.stft(_place(a, mem), persistence=True, vmin=vmin, vmax=vmax).persistence
    r2 = pl.stft(_place(b, mem), persistence=c, accumulate=True, vmin=vmin, vmax=vmax)
    assert r2.n_frames == F - F1
    np.testing.assert_array_equal(_get(pl, c), _get(pl, whole.persistence))
    pl.close()


def test_process_recording_persistence(sp, tmp_path):
    """process_recording(persistence=True) over small chunks equals one plan call on the whole file, and the histogram
    of the waterfall rows it returns."""
    from sdr_iq_visualizer_b200 import sigmf_io
    n, hop = 1024, 256
    x = _iq(200_000, 1, seed=9)
    base = sigmf_io.write_recording(str(tmp_path / "cap"), x, 1e6, 100e6, datatype="ci16_le")
    vmin, vmax = -120.0, 0.0
    rs = sigmf_io.process_recording(base, nfft=n, hop=hop, persistence=True, waterfall=True, vmin=vmin, vmax=vmax,
                                    max_chunk_samples=30_000)
    pl = sp.SpectralPlan(n, hop, "hann", sp.FMT_CI16, in_scale=2.0 ** -15)
    r = pl.stft(x, persistence=True, vmin=vmin, vmax=vmax)
    assert rs.n_frames == r.n_frames and rs.persistence.shape == (256, n)
    np.testing.assert_array_equal(rs.persistence, r.persistence[0])
    np.testing.assert_array_equal(rs.persistence, pref.persistence(rs.wf_rows)[0])
    pl.close()


# ----------------------------------------------------------------------------- 6: worst-case contention
@pytest.mark.parametrize("mem", ["host", "device"])
def test_every_frame_in_one_level(sp, mem):
    """vmax below every value: every frame of every bin in level 255; vmin above every value: all in level 0.  Every
    lane of every warp then adds to the same level."""
    n, hop, fmt, S, F = 4096, 1024, 1, 3, 300
    x, L = _input(n, hop, fmt, F, S, seed=11)
    pl = sp.SpectralPlan(n, hop, "hann", fmt)
    src = _place(x, mem)
    F = sref.frame_count(L, n, hop)
    hi = _get(pl, pl.stft(src, n_streams=S, persistence=True, vmin=-400.0, vmax=-300.0).persistence)
    assert (hi[:, 255] == F).all() and hi[:, :255].sum() == 0
    lo = _get(pl, pl.stft(src, n_streams=S, persistence=True, vmin=400.0, vmax=500.0).persistence)
    assert (lo[:, 0] == F).all() and lo[:, 1:].sum() == 0
    pl.close()


def test_more_than_65535_frames_in_one_shared_counter(sp):
    """70 000 frames in level 255 counted by ONE shared-memory counter: N = 512 is 4 strips, and sm_count / 4 streams make
    a grid of one CTA per SM with a single chunk per strip (the chunk rule takes the fewest chunks that fill >= 90 % of
    the SMs), so each CTA counts all 70 000 frames of its columns itself.  A 16-bit counter would wrap."""
    from sdr_iq_visualizer_b200 import _native as nat
    n, hop, F = 512, 1, 70_000
    sm = nat.device_info()["sm_count"]
    S = sm // 4
    assert 4 * S >= 0.9 * sm
    x = _iq(n + hop * (F - 1), 0, seed=17, S=S)
    pl = sp.SpectralPlan(n, hop, "rect")
    r, names = launched(lambda: pl.stft(nat.DeviceArray.from_host(x), n_streams=S, wf_rows=True, persistence=True,
                                        vmin=-400.0, vmax=-300.0))
    assert r.n_frames == F and count(names, PERSIST) == 1, names
    c = r.persistence.to_host()
    assert (c[:, 255] == F).all() and c.sum() == S * F * n
    r.wf_rows.free()
    pl.close()


def test_more_than_65535_frames_in_one_column(sp):
    """N = 16, 70 000 frames, every one in level 255.  One strip, so the frames are split over ~130 chunks: this covers
    the global accumulation of the chunks past 2^16 (the shared counters stay below it; see the test above)."""
    from sdr_iq_visualizer_b200 import _native as nat
    n, F = 16, 70_000
    x = _iq(n * F, 0, seed=13)
    pl = sp.SpectralPlan(n, n, "rect")
    r, names = launched(lambda: pl.stft(nat.DeviceArray.from_host(x), persistence=True, vmin=-400.0, vmax=-300.0))
    assert count(names, PERSIST) > 0
    c = r.persistence.to_host()
    assert (c[0, 255] == F).all() and c.sum() == F * n
    pl.close()


# ----------------------------------------------------------------------------- 7: edges and errors
@pytest.mark.parametrize("mem", ["host", "device"])
@pytest.mark.parametrize("n", [1, 16, 1000])
def test_small_and_odd_lengths(sp, n, mem):
    """N = 1 and 16 (narrower than a warp's 128 columns) and 1000 (not a multiple of the strip width), F = 1 and more."""
    vmin, vmax = -40.0, 60.0
    pl = sp.SpectralPlan(n, n, "hann")
    for F in (1, 37):
        x = _iq(n * F, 0, seed=n + F)
        r = pl.stft(_place(x, mem), wf_rows=True, persistence=True, vmin=vmin, vmax=vmax)
        assert r.n_frames == F
        np.testing.assert_array_equal(_get(pl, r.persistence), _counts_of_rows(r, 1))
    pl.close()


@pytest.mark.parametrize("mem", ["host", "device"])
def test_zero_frames(sp, mem):
    """F = 0: the counts are zeroed, or left as they are with accumulate."""
    from sdr_iq_visualizer_b200 import _native as nat
    n = 256
    pl = sp.SpectralPlan(n, n, "hann")
    x = _iq(n - 1, 0, seed=1)
    full = np.full((1, 256, n), 7, np.uint32)
    buf = full.copy() if mem == "host" else nat.DeviceArray.from_host(full)
    r = pl.stft(_place(x, mem), persistence=buf, accumulate=True, vmin=-40.0, vmax=60.0)
    pl.sync()
    assert r.n_frames == 0
    np.testing.assert_array_equal(_host(buf), full)
    pl.stft(_place(x, mem), persistence=buf, vmin=-40.0, vmax=60.0)
    pl.sync()
    assert not _host(buf).any()
    pl.close()


def test_errors(sp):
    from sdr_iq_visualizer_b200 import _native as nat
    n = 1024
    pl = sp.SpectralPlan(n, n, "hann")
    x = _iq(4 * n, 0, seed=2)
    with pytest.raises(nat.SpectralError) as e:
        pl.stft(x, persistence=True, vmin=10.0, vmax=10.0)        # vmax <= vmin, even without wf_rows
    assert e.value.code == nat.E_INVALID
    with pytest.raises(nat.SpectralError) as e:
        pl.stft(nat.DeviceArray.from_host(x), persistence=True, welch=True, peer_outputs=1, vmin=-40.0, vmax=60.0)
    assert e.value.code == nat.E_UNSUPPORTED
    a = nat.spx_stft_args()
    a.struct_size = C.sizeof(nat.spx_stft_args)
    a.mem, a.in_, a.n_samples, a.stream_stride, a.n_streams = nat.MEM_HOST, x.ctypes.data, 4 * n, 4 * n, 1
    a.vmin, a.vmax = -40.0, 60.0
    assert nat.lib().spx_stft_exec_persistence(pl._h, C.byref(a), None) == nat.E_INVALID
    assert "counts" in nat.last_error()
    pl.close()
