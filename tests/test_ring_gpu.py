"""GPU tests of the pinned ring ingest (csrc/spx_ring.cu, ring.StreamRing) and the streamer's block mode on top of it.

Every STFT family runs inside a ring from a slot buffer that starts with the carried tail of the previous slot.  Each
slot is checked on its own: its rows, its Welch sum and its max-hold against the float64 oracle over exactly its frames,
its on-device measurements against the oracle density and `classifier_ref.features`, and its byte counters.  The rows
are also held bit for bit to one device-resident call over the whole input where both ran the same kernel instances."""
import ctypes as C

import numpy as np
import pytest

from oracle import classifier_ref as cref
from oracle import spectral_ref as sref
from tests import parity
from tests.test_dispatch_paths_gpu import (BLU_PRE, K1_DIRECT, K1_STAGED, K1V2, K2_COLS_BULK, K2_COLS_DIRECT, K2V2, VRANGE,
                                           _cut, _iq, check_oracle, count, launched)
from tests.test_stft_gpu import oracle_rows

pytestmark = pytest.mark.gpu

K1_ANY = r"\bstft_kernel<"
RATE = 1.0e6          # sample rate of the rings that measure features


@pytest.fixture(scope="module")
def sp():
    from sdr_iq_visualizer_b200 import spectral
    from sdr_iq_visualizer_b200 import _native
    assert _native.device_count() > 0, "GPU tests need a CUDA device (no CPU fallback exists)"
    return spectral


def _schedule(cap, hop):
    """Chunk sizes of one ring run: full slots, a 1-sample commit, commits shorter than a hop, an empty commit (its slot
    completes no frame), a half slot and a short tail."""
    return [cap, 1, max(1, hop // 3), 0, cap, 7, cap // 2 + 13, cap, max(1, hop - 1), cap, 5]


def _copy(b):
    return {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in b.items()}


def _drive(ring, x, fmt, chunks, n_slots):
    """Push `chunks` samples of x through the ring, keeping it full (acquire then fails with E_BUSY); every slot's result,
    copied before its release, in commit order."""
    from sdr_iq_visualizer_b200 import _native as nat
    blocks, pos, pending = [], 0, 0

    def take():
        blocks.append(_copy(ring.collect()))
        ring.release()

    for c in chunks:
        ring.push(_cut(x, fmt, pos, pos + c))
        pos += c
        pending += 1
        if pending == n_slots:
            with pytest.raises(nat.SpectralError) as e:
                ring.acquire()
            assert e.value.code == nat.E_BUSY
            take()
            pending -= 1
    while pending:
        take()
        pending -= 1
    return blocks


def _small_bytes(n, welch, maxhold, feats):
    """The slot's one-copy block of small results, laid out as spx_ring_create does."""
    from sdr_iq_visualizer_b200 import _native as nat
    b = (8 * n if welch else 0) + (8 * n if feats else 0) + (4 * n if maxhold else 0)
    return -(-b // 8) * 8 + (C.sizeof(nat.spx_features) if feats else 0)


def check_features(got, pdb, what):
    """The device measurements of a spectrum against the oracle's (test_classifier_gpu.test_random_spectra_vs_oracle)."""
    want = cref.features(np.arange(pdb.size, dtype=np.float64), pdb)
    assert got["n"] == want["n"], what
    for k in ("noise_floor_db", "peak_db", "argmax", "snr_db", "adaptive_thr", "min_distance_bins", "n_candidates",
              "peak_count"):
        assert got[k] == want[k], (what, k)
    for d in (3, 10, 20):
        assert (got[f"first_{d}db"], got[f"last_{d}db"]) == want["edges"][d], (what, d)
    assert (got["simple_first"], got["simple_last"]) == want["simple_edges"], what
    np.testing.assert_allclose(got["flatness"], want["flatness"], rtol=1e-11, atol=1e-300, err_msg=what)
    np.testing.assert_allclose(got["kurtosis"], want["kurtosis"], rtol=1e-11, atol=1e-11, err_msg=what)


def check_density(pdb, P, rate, sum_w2, what):
    """A slot's Welch PSD in dB against the oracle's mlab density of its frames: sum |X|^2 / (F fs sum w^2)."""
    parity.check_power(10.0 ** (pdb / 10.0), P.sum(axis=0) / (P.shape[0] * rate * sum_w2), what=what)


def check_slots(blocks, X, n, kind, fmt, outs, what):
    """Continuity of the slots, and each slot's rows and accumulators against the oracle rows X of its own frames."""
    P = X.real**2 + X.imag**2
    vmin, vmax = VRANGE[fmt]
    assert sum(b["n_frames"] for b in blocks) == X.shape[0], what
    assert any(b["n_frames"] == 0 for b in blocks), f"{what}: no slot without frames"
    f0 = 0
    for i, b in enumerate(blocks):
        nf = b["n_frames"]
        assert b["seq"] == i and b["first_frame"] == f0, (what, i)
        sl, w = slice(f0, f0 + nf), f"{what} slot {i} frames {f0}..{f0 + nf}"
        if "u8" in outs:
            assert b["wf_rows"].shape == (nf, n)
        if "db" in outs:
            assert b["db_rows"].shape == (nf, n)
        if nf == 0:
            # an empty slot still returns its accumulators: zero, whatever the slot held when it was last used
            assert not b["welch_acc"].any() and not b["maxhold"].any(), w
            assert b["features"] is None and b["pxx_db"] is None, w
        else:
            if "u8" in outs:
                parity.check_u8(b["wf_rows"], sref.amplitude_db(X[sl]), vmin, vmax, what=f"{w} u8")
            if "db" in outs:
                parity.check_db_rows(b["db_rows"], P[sl], what=f"{w} dB rows")
            parity.check_power(b["welch_acc"], P[sl].sum(axis=0), what=f"{w} welch")
            parity.check_power(b["maxhold"], P[sl].max(axis=0), what=f"{w} maxhold")
            if "feat" in outs:
                check_density(b["pxx_db"], P[sl], RATE, float((sref.window(kind, n) ** 2).sum()), f"{w} pxx")
                check_features(b["features"], b["pxx_db"], w)
        if "feat" not in outs:
            assert b["features"] is None and b["pxx_db"] is None
        d2h = nf * n * ("u8" in outs) + 4 * nf * n * ("db" in outs) + _small_bytes(n, True, True, "feat" in outs)
        assert b["d2h_bytes"] == d2h, (w, b["d2h_bytes"], d2h)
        f0 += nf


def _stft_instances(names):
    """The kernel template instances of the STFT itself (the feature kernel of a measuring ring left out)."""
    return {nm for nm in names if "<" in nm and "features_kernel" not in nm}


# n, hop, window, fmt, outputs, slot samples, slots, the family that must run in the ring, families that must not
RING_CASES = [
    (256, 77, "hann", 0, "u8 db", 4096, 4, K1_DIRECT, (K1_STAGED, K1V2)),        # odd hop: K1 with direct loads
    (512, 512, "rect", 1, "u8", 512, 3, K1_STAGED, (K1_DIRECT, K1V2)),           # hop == nfft, slot_samples == nfft
    (1024, 256, "blackman", 1, "u8 db", 8192, 4, K1V2, (K1_ANY,)),
    (2048, 512, "hann", 0, "u8", 16384, 3, K1V2, (K1_ANY,)),
    (4096, 1024, "hann", 1, "u8 db feat", 1 << 16, 3, K1V2, (K1_ANY,)),
    (4096, 1000, "hann", 0, "u8", 32768, 4, K1_ANY, (K1V2,)),                     # frames not 128-byte aligned: K1
    (8192, 2048, "blackman", 0, "u8 db", 32768, 3, K1_ANY, (K1V2,)),
    (16384, 8192, "hann", 0, "u8 db", 65536, 4, K2_COLS_BULK, (K2_COLS_DIRECT, K2V2)),   # 1 MiB scratch: 4 frames per batch
    (65536, 32768, "hann", 1, "u8 feat", 131072, 3, K2V2, (K2_COLS_BULK, K2_COLS_DIRECT)),
    (65536, 32768, "hann", 0, "db", 131072, 3, K2_COLS_BULK, (K2V2,)),            # K2v2 emits no float rows: K2
    (1000, 250, "hann", 1, "u8 db", 8000, 4, BLU_PRE, (K2V2, K2_COLS_BULK)),
    (1001, 1001, "rect", 0, "u8 feat", 4004, 2, BLU_PRE, (K2V2, K2_COLS_BULK)),   # odd N: the feature record's alignment
]


@pytest.mark.parametrize("n,hop,kind,fmt,outs,cap,n_slots,fam,absent", RING_CASES,
                         ids=[f"N{c[0]}-hop{c[1]}-{c[2]}-{'ci16' if c[3] else 'cf32'}-{c[4].replace(' ', '+')}" for c in RING_CASES])
def test_ring_matches_one_shot(sp, monkeypatch, n, hop, kind, fmt, outs, cap, n_slots, fam, absent):
    """One ring per dispatch family, fed an irregular schedule that keeps it full: every slot against the oracle over its
    own frames (rows, Welch sum, max-hold, measurements), the slots continuous, the counters exact; the family ran inside
    the ring; the rows bit-identical to one device-resident call over the whole input on a second plan when both ran
    the same kernel instances."""
    from sdr_iq_visualizer_b200 import _native as nat
    from sdr_iq_visualizer_b200.ring import StreamRing
    if n == 16384:
        monkeypatch.setenv("SPX_BIG_SCRATCH_BYTES", str(1 << 20))
    chunks = _schedule(cap, hop)
    L = sum(chunks)
    x = _iq(L, fmt, seed=n + hop + fmt)
    vmin, vmax = VRANGE[fmt]
    rows = dict(wf_rows="u8" in outs, db_rows="db" in outs)
    feats = "feat" in outs
    pl = sp.SpectralPlan(n, hop, kind, fmt)
    ref = sp.SpectralPlan(n, hop, kind, fmt)
    ring = StreamRing(pl, n_slots=n_slots, slot_samples=cap, **rows, welch=True, maxhold=True, vmin=vmin, vmax=vmax,
                      features=feats, sample_rate=RATE if feats else 0.0)
    blocks, names = launched(lambda: _drive(ring, x, fmt, chunks, n_slots))
    st = ring.stats()
    F = sref.frame_count(L, n, hop)
    elt = 4 if fmt else 8
    assert st == {"h2d_bytes": elt * L, "d2h_bytes": sum(b["d2h_bytes"] for b in blocks), "samples": L, "frames": F,
                  "in_flight": 0}
    assert len(blocks) == len(chunks)

    # the family ran inside the ring, once per batch of frames of every slot that has frames
    busy = [b["n_frames"] for b in blocks if b["n_frames"]]
    assert count(names, fam) > 0, names
    for pat in absent:
        assert count(names, pat) == 0, (pat, names)
    if fam == K2_COLS_BULK and n == 16384:
        assert count(names, fam) == sum(-(-f // 4) for f in busy), names
    elif fam in (K2V2, BLU_PRE):
        assert count(names, fam) == len(busy), names
    if feats:
        assert count(names, r"\bfeatures_kernel<") == len(busy), names

    X = oracle_rows(x, n, hop, kind, fmt=fmt)
    check_slots(blocks, X, n, kind, fmt, outs, what=f"ring N={n} hop={hop} {kind} fmt={fmt}")

    d_x = nat.DeviceArray.from_host(x)
    one, names0 = launched(lambda: ref.stft(d_x, **rows, welch=True, maxhold=True, vmin=vmin, vmax=vmax))
    assert one.n_frames == F
    inst, inst0 = _stft_instances(names), _stft_instances(names0)
    if inst == inst0 and len({nm.split("<")[0] for nm in inst}) == len(inst):
        # the same kernel instance computed every frame in both runs, from the same samples: the same bits
        for k, on in rows.items():
            if on:
                np.testing.assert_array_equal(np.concatenate([b[k] for b in blocks]), getattr(one, k).to_host(), err_msg=k)
    else:
        # a slot's frame count can pick another instance of the family (K1v2's strip kernel, occupancy variants) than the
        # whole run does, and those may round differently: both runs are then held to the oracle instead
        print("kernel instances differ:", sorted(inst ^ inst0))
        check_oracle(one, x, n, hop, kind, fmt, what=f"one-shot N={n} hop={hop}")
    ring.close(); pl.close(); ref.close()


def test_ring_errors(sp):
    """spx_ring_create's rejections, and E_BUSY / E_INVALID from acquire, commit, collect and release; the ring gives
    correct slots afterwards."""
    from sdr_iq_visualizer_b200 import _native as nat
    from sdr_iq_visualizer_b200.ring import StreamRing
    n, hop, cap = 1024, 256, 4096
    vmin, vmax = VRANGE[1]
    pl = sp.SpectralPlan(n, hop, "hann", sp.FMT_CI16)
    base = dict(n_slots=2, slot_samples=cap, wf_rows=True, welch=True, maxhold=True, vmin=vmin, vmax=vmax)
    for bad in (dict(n_slots=1), dict(n_slots=65), dict(slot_samples=n - 1), dict(vmin=vmax), dict(vmin=vmax + 1.0),
                dict(features=True, welch=False, sample_rate=RATE), dict(features=True, sample_rate=0.0)):
        with pytest.raises(nat.SpectralError) as e:
            StreamRing(pl, **{**base, **bad})
        assert e.value.code == nat.E_INVALID, bad
    cfg = nat.spx_ring_config(C.sizeof(nat.spx_ring_config) + 8, 2, cap, 1, 0, 1, 1, vmin, vmax, 0, 0, 0.0)
    h = C.c_void_p()
    assert nat.lib().spx_ring_create(C.byref(h), pl._h, C.byref(cfg)) == nat.E_INVALID and not h.value

    ring = StreamRing(pl, **base)

    def code(fn, *a):
        with pytest.raises(nat.SpectralError) as e:
            fn(*a)
        return e.value.code

    assert code(ring.collect) == nat.E_BUSY and code(ring.release) == nat.E_BUSY
    assert code(ring.commit, 10) == nat.E_INVALID                  # no slot acquired
    x = _iq(3 * cap, 1, seed=5)
    slot = ring.acquire()
    assert code(ring.commit, -1) == nat.E_INVALID and code(ring.commit, cap + 1) == nat.E_INVALID
    with pytest.raises(ValueError):
        ring.push(_cut(x, 1, 0, cap + 1))
    slot[: 2 * cap] = _cut(x, 1, 0, cap)                           # the acquired slot survived the rejected commits
    ring.commit(cap)
    ring.push(_cut(x, 1, cap, 2 * cap))
    assert code(ring.acquire) == nat.E_BUSY
    blocks = [_copy(ring.collect())]
    ring.release()
    ring.push(_cut(x, 1, 2 * cap, 3 * cap))
    blocks.append(_drain_one(ring))
    ring.push(np.zeros(0, np.int16))
    blocks += [_drain_one(ring), _drain_one(ring)]
    assert code(ring.collect) == nat.E_BUSY
    check_slots(blocks, oracle_rows(x, n, hop, "hann", fmt=1), n, "hann", 1, "u8", what="ring after errors")
    st = ring.stats()
    assert st["samples"] == 3 * cap and st["h2d_bytes"] == 4 * 3 * cap and st["in_flight"] == 0
    ring.close(); pl.close()


def _drain_one(ring):
    b = _copy(ring.collect())
    ring.release()
    return b


@pytest.mark.parametrize("order", ["one_shot_then_commit", "commit_then_one_shot"])
@pytest.mark.parametrize("n,hop,F1", [(16384, 8192, 300), (3000, 1500, 600)], ids=["K2", "Bluestein"])
def test_ring_commit_orders_with_one_shot_scratch(sp, monkeypatch, n, hop, F1, order):
    """A device-resident call on a caller stream and a ring commit on the same plan, enqueued back to back with no
    synchronisation in between, in either order.  Both use the plan's scratch (K2's two halves through a 1 MiB scratch:
    4 frames per batch, 75 batches on the caller stream; the Bluestein buffers); the commit waits for the call, and a
    call after a commit waits for the slot's kernels.  Both results against the oracle and against each run alone: rows
    and max-hold bit-identical, Welch to 1e-12.  One run cannot show that the race is gone (it may simply not have been
    hit); the ordering rests on reading the code, and this test holds the results of both orders."""
    from sdr_iq_visualizer_b200 import _native as nat
    from sdr_iq_visualizer_b200.ring import StreamRing
    monkeypatch.setenv("SPX_BIG_SCRATCH_BYTES", str(1 << 20))
    cap = n + 39 * hop                                              # 40 frames in the slot
    x = _iq(n + hop * (F1 - 1), 0, seed=n + 1)
    y = _iq(cap, 0, seed=n + 2)
    kw = dict(wf_rows=True, welch=True, maxhold=True, vmin=-40.0, vmax=90.0)
    pl = sp.SpectralPlan(n, hop, "hann")
    alone = sp.SpectralPlan(n, hop, "hann")
    side = nat.SideStream()
    d_x = nat.DeviceArray.from_host(x)
    outs = dict(wf_rows=nat.DeviceArray((F1, n), np.uint8), welch=nat.DeviceArray((1, n), np.float64),
                maxhold=nat.DeviceArray((1, n), np.float32))
    ring = StreamRing(pl, n_slots=2, slot_samples=cap, **kw)

    def both():
        if order == "one_shot_then_commit":
            rd = pl.stft(d_x, **{**kw, **outs}, stream=side.handle)
            ring.push(y)
        else:
            ring.push(y)
            rd = pl.stft(d_x, **{**kw, **outs}, stream=side.handle)
        side.sync()
        return rd, _drain_one(ring)

    (rd, b), names = launched(both)
    assert b["n_frames"] == 40 and rd.n_frames == F1
    if n == 16384:
        assert count(names, K2_COLS_BULK) == F1 // 4 + 40 // 4, names
    else:
        assert count(names, BLU_PRE) == 2, names
    check_oracle(rd, x, n, hop, "hann", 0, what=f"{order}: one-shot call")
    X = oracle_rows(y, n, hop, "hann")
    P = X.real**2 + X.imag**2
    parity.check_u8(b["wf_rows"], sref.amplitude_db(X), -40.0, 90.0, what=f"{order}: ring slot u8")
    parity.check_power(b["welch_acc"], P.sum(axis=0), what=f"{order}: ring slot welch")
    parity.check_power(b["maxhold"], P.max(axis=0), what=f"{order}: ring slot maxhold")

    ra = alone.stft(d_x, **kw)
    alone.sync()
    np.testing.assert_array_equal(rd.wf_rows.to_host(), ra.wf_rows.to_host())
    np.testing.assert_array_equal(rd.maxhold.to_host(), ra.maxhold.to_host())
    np.testing.assert_allclose(rd.welch_acc.to_host(), ra.welch_acc.to_host(), rtol=1e-12)
    ring_a = StreamRing(alone, n_slots=2, slot_samples=cap, **kw)
    ring_a.push(y)
    ba = _drain_one(ring_a)
    np.testing.assert_array_equal(b["wf_rows"], ba["wf_rows"])
    np.testing.assert_array_equal(b["maxhold"], ba["maxhold"])
    np.testing.assert_allclose(b["welch_acc"], ba["welch_acc"], rtol=1e-12)
    ring.close(); ring_a.close(); side.close(); alone.close(); pl.close()


def test_streamer_block_mode_matches_one_shot():
    """SURVEY 8(f-1): rx buffers -> pinned ring -> blocks of frames_per_block frames with u8 rows, Welch, running
    max-hold and on-device classifier measurements; identical to one pass over the concatenated stream, and every
    published block's PSD against the oracle density of its frames, its measurements against the oracle's of that PSD."""
    _streamer_blocks(4096, 0.75, 64, 40)


@pytest.mark.parametrize("n,fpb,nbuf", [(1000, 24, 40), (16384, 8, 24)], ids=["N1000", "N16384"])
def test_streamer_block_mode_other_families(n, fpb, nbuf):
    """The streamer's block mode at 50 % overlap on Bluestein (N = 1000) and on the four-step path (N = 16384), held to
    the same rules as at N = 4096."""
    _streamer_blocks(n, 0.5, fpb, nbuf)


def _streamer_blocks(n, overlap, fpb, nbuf):
    import sys
    from unittest.mock import MagicMock
    sys.modules.setdefault("adi", MagicMock())
    from app.processing import classifier as clf
    from app.sdr.streamer import SDRDataStreamer
    from sdr_iq_visualizer_b200 import features, spectral as sp
    hop = max(1, int(round(n * (1.0 - overlap))))
    rate = 61.44e6
    raw = sref.to_ci16(sref.synth_iq(nbuf * n, seed=33))
    x = raw[0::2].astype(np.float64) + 1j * raw[1::2].astype(np.float64)      # what pyadi-iio's rx() returns
    s = SDRDataStreamer(sample_rate=rate, center_freq=2_400_000_000)
    s.enable_block_mode(nfft=n, overlap=overlap, window="hann", frames_per_block=fpb, n_slots=3, vmin=20.0, vmax=130.0)
    blocks = []
    for b in range(nbuf):
        d = s.process_buffer(x[b * n:(b + 1) * n])
        assert set(d) >= {"time", "samples", "freqs", "power_db", "sample_rate", "center_freq"}
        blk = s.get_latest_block()
        if blk is not None and (not blocks or blk["seq"] != blocks[-1]["seq"]):
            blocks.append(blk)
    s.flush_blocks()
    blk = s.get_latest_block()
    if not blocks or blk["seq"] != blocks[-1]["seq"]:
        blocks.append(blk)
    assert len(blocks) >= 2
    st = s.get_status()
    assert st["ring"]["h2d_bytes"] == 4 * nbuf * n and st["blocks_done"] >= len(blocks)
    pl = sp.SpectralPlan(n, hop, "hann", sp.FMT_CI16)
    one = pl.stft(raw, wf_rows=True, welch=True, maxhold=True, vmin=20.0, vmax=130.0)
    sum_w2 = float((sref.window("hann", n) ** 2).sum())
    # the published blocks are a subsequence of all blocks (only the newest is kept): check each against its frames
    for blk in blocks:
        f0, nf = blk["first_frame"], blk["n_frames"]
        np.testing.assert_array_equal(blk["wf_rows"], one.wf_rows[f0:f0 + nf])
        seg = raw[2 * f0 * hop: 2 * ((f0 + nf - 1) * hop + n)]
        part = pl.stft(seg, welch=True)
        np.testing.assert_allclose(blk["welch_acc"], part.welch_acc[0], rtol=1e-6)
        _, pdb = pl.welch_finalize(blk["welch_acc"], nf, rate)
        np.testing.assert_allclose(blk["pxx_db"], pdb, rtol=0, atol=1e-9)
        X = oracle_rows(seg, n, hop, "hann", fmt=1)
        check_density(blk["pxx_db"], X.real**2 + X.imag**2, rate, sum_w2, f"streamer N={n} block {blk['seq']} pxx")
        check_features(blk["features"], blk["pxx_db"], f"streamer N={n} block {blk['seq']}")
        m = features.measure(blk["pxx_db"])
        for k in ("noise_floor_db", "snr_db", "first_20db", "last_20db", "flatness", "kurtosis", "peak_count"):
            assert blk["features"][k] == m[k], k
        clf._CLASS_HISTORY.clear(); clf._CONF_HISTORY.clear()
        want = clf.classify_signal_advanced(blk["freqs"], blk["pxx_db"])
        assert blk["classification"]["label"] is not None
        got_feats, want_feats = blk["classification"]["features"], want["features"]
        assert got_feats["snr_db"] == want_feats["snr_db"] and got_feats["bandwidth_hz_20db"] == want_feats["bandwidth_hz_20db"]
        assert abs(got_feats["peak_spacing_std_hz"] - want_feats["peak_spacing_std_hz"]) <= 1e-6 * max(1.0, want_feats["peak_spacing_std_hz"])
    last = blocks[-1]
    assert last["first_frame"] + last["n_frames"] == one.n_frames              # flush published the tail block
    np.testing.assert_array_equal(last["maxhold"], one.maxhold[0])              # running max-hold over every block
    clf._CLASS_HISTORY.clear(); clf._CONF_HISTORY.clear()
    s.disable_block_mode()
    pl.close()
