"""Every kernel instance libspx.so builds, held to the float64 oracle by name (tests/kernel_instances.py).

Each case of ``CASES`` runs once: its calls run under the CUDA profiler, the instances the case declares in ``expects``
must be among the kernels that ran, and every output of the calls is held to the float64 reference with the rule its
family's own tests use (tests/parity.py for the STFT outputs, chan_ref / ddc_ref / detect_ref / pool_ref /
persistence_ref, oracle/classifier_ref, oracle/spectral_ref).  tests/test_kernel_instances_cpu.py checks that the cases
cover every instance of the built library, so a green run of this module means every built instance was checked."""
import numpy as np
import pytest

from oracle import spectral_ref as sref
from tests import kernel_instances as ki, parity
from tests.test_dispatch_paths_gpu import VRANGE, check_oracle, launched as _launched

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def nat():
    from sdr_iq_visualizer_b200 import _native
    assert _native.device_count() > 0, "GPU tests need a CUDA device (no CPU fallback exists)"
    return _native


def launched(fn):
    """test_dispatch_paths_gpu.launched, with one torch kernel and a device synchronise at the start of the session: in a
    process that has already run other profiled tests, the profiler has been seen to drop the first activity of a
    session (a case's only kernel, or K2's column kernel), and that must not be a kernel a case declares."""
    import torch

    def run():
        torch.ones(1, device="cuda:0").add_(1.0)
        torch.cuda.synchronize(0)
        return fn()
    return _launched(run)


def _iq(L, fmt, seed):
    """tone + QPSK + noise (synth_iq); interleaved int16 for ci16 input."""
    x = sref.synth_iq(L, seed=seed)
    return sref.to_ci16(x) if fmt else x.astype(np.complex64)


def _ran(case, names):
    got = {ki.key(n) for n in names}
    missing = case["expects"] - got
    assert not missing, f"{case['id']}: expected instances did not run: {sorted(missing)}; ran {sorted(got)}"


def _sel(F, case, seed):
    """Rows checked: first and last frame, both sides of every chunk boundary near either end of the run for each chunk
    length the launcher can pick, and a seeded random sample."""
    sel = {0, 1, F - 2, F - 1}
    geom = case["geom"]
    for c in (ki.chunk_sizes(F, *geom) if geom else [max(1, F // 4)]):
        bounds = list(range(c, F, c))
        for b in bounds[:3] + bounds[-3:]:
            sel |= {b - 1, b}
    rng = np.random.default_rng(seed)
    sel |= set(rng.choice(F, size=min(F, 48), replace=False).tolist())
    return sorted(f for f in sel if 0 <= f < F)


# ----------------------------------------------------------------------------- STFT families (K1, K1v2, K2, K2v2, Bluestein)
def _run_stft(nat, case):
    from sdr_iq_visualizer_b200 import spectral as sp
    n, hop, fmt, F = case["n"], case["hop"], case["fmt"], case["frames"]
    L = n + hop * (F - 1) + 3
    x = _iq(L, fmt, seed=n + hop + fmt)
    vmin, vmax = VRANGE[fmt]
    pl = sp.SpectralPlan(n, hop, case["kind"], fmt, variant=case["variant"])
    d_x = nat.DeviceArray.from_host(x)
    outs = {k: True for k in case["outs"]}
    r, names = launched(lambda: pl.stft(d_x, **outs, vmin=vmin, vmax=vmax))
    pl.sync()
    _ran(case, names)
    assert r.n_frames == F
    for k in ("db_rows", "wf_rows", "spectrum", "welch", "maxhold"):
        attr = {"welch": "welch_acc"}.get(k, k)
        assert (getattr(r, attr) is not None) == (k in case["outs"]), k
    sel = _sel(F, case, seed=n + fmt)
    check_oracle(r, x, n, hop, case["kind"], fmt, sel=sel, what=case["id"])
    pl.close()


# ----------------------------------------------------------------------------- K3
def _run_features(nat, case):
    from sdr_iq_visualizer_b200 import features as feat
    from tests.test_features_edges_gpu import check, noisy
    dtype = np.float64 if case["dtype"] == "float64" else np.float32
    rows = [noisy(n, seed=n, dtype=dtype) for n in (4096, 4096, 4096)]
    rows[1][17] = rows[1].max() + 1.0                   # a second peak
    got, names = launched(lambda: feat.measure_batch(np.stack(rows)))
    _ran(case, names)
    for i, (g, r) in enumerate(zip(got, rows)):
        check(g, r, f"{case['id']} row {i}")


# ----------------------------------------------------------------------------- K4
def _run_hist2d(nat, case):
    from sdr_iq_visualizer_b200 import timedomain as td
    fmt, bins = case["fmt"], case["bins"]
    n = 3_000_001
    rng = np.random.default_rng(bins + fmt)
    if fmt:
        raw = rng.integers(-2048, 2048, 2 * n).astype(np.int16)
        raw[:8] = [-2048, -2048, 2047, 2047, 0, 0, -1, 1]                # both range edges and the centre
        r_range, scale = 2048.0, 1.0
        xc = sref.unpack_ci16(raw)
        src = raw
    else:
        xc = (0.6 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))).astype(np.complex64)
        xc[:6] = [2.0 + 2.0j, -2.0 - 2.0j, 0.0, 2.0000002 + 0j, np.nan + 0j, np.inf + 1j]   # edges, outside, non-finite
        r_range, scale = 2.0, 1.0
        src = xc
    d = nat.DeviceArray.from_host(src)
    h, names = launched(lambda: td.iq_hist2d(d, r_range, bins, in_fmt=fmt, in_scale=scale))
    _ran(case, names)
    want = sref.iq_hist2d(np.asarray(xc, np.complex128), r_range, bins)
    np.testing.assert_array_equal(h.to_host(), want)


def _run_frame_stats(nat, case):
    """NaN, +-inf (cf32) and full-scale int16 (ci16) samples; frame_len 7 with hop 9 (gaps between frames) over more
    frames than the 8 x SMs CTAs, so the grid-stride loop runs; frame_len 1; host and device memory."""
    from sdr_iq_visualizer_b200 import timedomain as td
    fmt = case["fmt"]
    F = 8 * ki.SMS * 2 + 37
    rng = np.random.default_rng(fmt + 5)
    calls = []
    for frame_len, hop in ((7, 9), (1, 1)):
        L = frame_len + hop * (F - 1)
        if fmt:
            raw = rng.integers(-32768, 32768, 2 * L).astype(np.int16)
            raw[:4] = [-32768, -32768, 32767, -32768]                    # I^2 + Q^2 = 2^31, and 2^31 - 2^16 + 1
            raw[2 * hop * 5: 2 * hop * 5 + 2] = [-32768, -32768]
            xc = sref.unpack_ci16(raw)
            src = raw
        else:
            xc = (100.0 * (rng.standard_normal(L) + 1j * rng.standard_normal(L))).astype(np.complex64)
            xc[hop * 3] = np.nan                                          # NaN at the start of frame 3
            xc[hop * 10 + frame_len - 1] = complex(1.0, np.nan)           # NaN Q at the end of frame 10
            xc[hop * 20] = complex(np.inf, 0.0)
            xc[hop * 21 + frame_len // 2] = complex(-np.inf, 5.0)
            xc[hop * 22] = complex(np.inf, np.nan)
            xc[hop * (F - 1)] = np.nan                                    # the last frame
            src = xc
        calls.append((frame_len, hop, xc, src))

    def run():
        out = []
        for frame_len, hop, xc, src in calls:
            out.append(td.frame_stats(src, frame_len, hop, in_fmt=fmt))                            # host memory
            d = nat.DeviceArray.from_host(src)
            mean, peak = td.frame_stats(d, frame_len, hop, in_fmt=fmt)                             # device memory
            nat.device_sync(0)
            out.append((mean.to_host(), peak.to_host()))
        return out

    got, names = launched(run)
    _ran(case, names)
    for i, (frame_len, hop, xc, _) in enumerate(calls):
        m_ref, p_ref = sref.frame_stats(np.asarray(xc, np.complex128), frame_len, hop)
        assert m_ref.size == F
        for mean, peak in got[2 * i: 2 * i + 2]:
            assert mean.shape == peak.shape == (F,)
            what = f"{case['id']} frame_len={frame_len}"
            np.testing.assert_array_equal(np.isnan(peak), np.isnan(p_ref), err_msg=f"{what}: NaN peaks")
            np.testing.assert_array_equal(np.isnan(mean), np.isnan(m_ref), err_msg=f"{what}: NaN means")
            p32 = p_ref.astype(np.float32)
            ok = ~np.isnan(p_ref)
            # the power is formed in float32: within one float32 ulp of the float64 power's rounding
            ulps = np.abs(peak[ok].view(np.int32).astype(np.int64) - p32[ok].view(np.int32).astype(np.int64))
            assert ulps.max() <= 1, f"{what}: peak {int(ulps.max())} ulp from float32(oracle)"
            fin = np.isfinite(m_ref)
            np.testing.assert_array_equal(mean[~fin & ~np.isnan(m_ref)], m_ref[~fin & ~np.isnan(m_ref)].astype(np.float32))
            np.testing.assert_allclose(mean[fin], m_ref[fin], rtol=2e-7, atol=0, err_msg=what)


# ----------------------------------------------------------------------------- K6
def _run_stream_frame(nat, case):
    from sdr_iq_visualizer_b200 import spectral as sp
    n = 4096
    rng = np.random.default_rng(n)
    x = np.rint(rng.normal(0, 300, n) + 1j * rng.normal(0, 300, n)) + 1500 * np.exp(2j * np.pi * 0.123 * np.arange(n))
    fs, fc = 2.5e6, 9.15e8
    (r64, r32), names = launched(lambda: (sp.stream_frame(x, fs, fc), sp.stream_frame(x.astype(np.complex64), fs, fc)))
    _ran(case, names)
    assert np.abs(r64[1] - sref.stream_frame(x, fs, fc)[1]).max() <= 1e-9
    assert np.abs(r32[1] - sref.stream_frame(x.astype(np.complex64).astype(np.complex128), fs, fc)[1]).max() <= 1e-9


# ----------------------------------------------------------------------------- K7 / K8
def _run_persistence(nat, case):
    from sdr_iq_visualizer_b200 import spectral as sp
    from tests import persistence_ref as pref
    n, hop, fmt, F = 4096, 1024, 1, 300
    x = _iq(n + hop * (F - 1), fmt, seed=7)
    vmin, vmax = VRANGE[fmt]
    pl = sp.SpectralPlan(n, hop, "hann", fmt)
    d_x = nat.DeviceArray.from_host(x)
    r, names = launched(lambda: pl.stft(d_x, wf_rows=True, persistence=True, vmin=vmin, vmax=vmax))
    pl.sync()
    _ran(case, names)
    rows = r.wf_rows.to_host()
    from tests.test_dispatch_paths_gpu import _oracle
    X, _, _ = _oracle(x, n, hop, "hann", fmt, 1, list(range(F)))
    parity.check_u8(rows, sref.amplitude_db(X), vmin, vmax, what=f"{case['id']} u8")
    np.testing.assert_array_equal(r.persistence.to_host(), pref.persistence(rows, 1))
    pl.close()


def _run_pool(nat, case):
    """Two calls on consecutive pieces pool into one accumulator (the second at pool_first_frame), then finalize."""
    from sdr_iq_visualizer_b200 import spectral as sp
    from tests import pool_ref as pr
    from tests.test_dispatch_paths_gpu import _oracle
    from tests.test_pooled_gpu import check_against_rows
    n, hop, fmt, F1, F2, K, B = 1024, 512, 0, 70, 53, 9, 8
    mode = case["mode"]
    vmin, vmax = VRANGE[fmt]
    F = F1 + F2
    x = _iq(n + hop * (F - 1), fmt, seed=11)
    pl = sp.SpectralPlan(n, hop, "hann", fmt)
    d_x = nat.DeviceArray.from_host(x)
    d_a = nat.DeviceView(d_x.ptr, (n + hop * (F1 - 1),), np.complex64, keep=d_x)
    d_b = nat.DeviceView(d_x.ptr + F1 * hop * 8, (n + hop * (F2 - 1),), np.complex64, keep=d_x)
    G = -(-F // K)
    acc = nat.DeviceArray((1, G, n // B), np.float64)

    def run():
        r1 = pl.stft(d_a, db_rows=True, pool=(K, B, mode), pool_acc=acc, vmin=vmin, vmax=vmax)
        r2 = pl.stft(d_b, db_rows=True, pool=(K, B, mode), pool_acc=acc, pool_first_frame=F1, accumulate=True,
                     vmin=vmin, vmax=vmax)
        pl.sync()
        db, wf = pl.pool_finalize(acc, F, K, B, mode, db=True, wf=True, vmin=vmin, vmax=vmax)
        pl.sync()
        return r1, r2, db.to_host(), wf.to_host()

    (r1, r2, db, wf), names = launched(run)
    _ran(case, names)
    rows = np.concatenate([r1.db_rows.to_host(), r2.db_rows.to_host()])
    check_against_rows(db, rows, K, B, mode, 1, what=case["id"])
    np.testing.assert_array_equal(wf, sref.waterfall_u8(db, vmin, vmax))
    X, _, _ = _oracle(x, n, hop, "hann", fmt, 1, list(range(F)))
    P = X.real ** 2 + X.imag ** 2
    parity.check_db_rows(db[0], pr.pool_power(P, K, B, mode)[0], eps=pr.EPS, what=f"{case['id']} vs float64")
    pl.close()


# ----------------------------------------------------------------------------- K9
def _run_ddc(nat, case):
    from sdr_iq_visualizer_b200 import ddc
    from tests import ddc_ref as dr
    fmt, fs, D, L = case["fmt"], 61.44e6, 8, 400_003
    x = _iq(L, fmt, seed=21 + fmt)
    scale = 1.0 / 1024 if fmt else 1.0
    p = ddc.DdcPlan(fs, 7.3e6, D, in_fmt=fmt, in_scale=scale)
    d_x = nat.DeviceArray.from_host(x)
    incs = [p.phase_inc, ddc.phase_increment(-11.1e6, fs)[0], ddc.phase_increment(3.0e5, fs)[0]]
    jobs = [(1000, incs[1], 0, 5000, 0), (0, incs[2], 17, 20000, 5000), (250_000, incs[0], 3, 9000, 25000)]
    out = nat.DeviceArray((34000,), np.complex64)

    def run():
        y = p.exec(d_x)
        p.exec_jobs(d_x, jobs, out)
        p.sync()
        return y.to_host(), out.to_host()

    (y, o), names = launched(run)
    _ran(case, names)
    bar = 1e-5 * dr.bound(p.taps, x, scale)
    want = dr.ddc(x, p.taps, D, p.phase_inc, 0, scale)
    assert y.shape == want.shape and np.abs(y - want).max() <= bar, case["id"]
    for first, inc, m0, n_out, off in jobs:
        # a job's outputs are those of DdcPlan.exec at its increment on the capture from its first sample
        w = dr.ddc(_cut(x, fmt, first, L), p.taps, D, inc, first, scale)[m0:m0 + n_out]
        assert w.size == n_out and np.abs(o[off:off + n_out] - w).max() <= bar, (case["id"], first)
    p.close()


def _cut(x, fmt, a, b):
    return x[2 * a: 2 * b] if fmt else x[a:b]


# ----------------------------------------------------------------------------- K10
def _run_chan(nat, case):
    from sdr_iq_visualizer_b200 import ddc
    from tests import chan_ref as cr
    M, D, fmt = case["m"], case["decim"], case["fmt"]
    taps = None
    if case["taps"]:
        taps = np.random.default_rng(M).normal(size=case["taps"]) / case["taps"]
    h = ddc.Channelizer(61.44e6, M, D, taps=taps, in_fmt=fmt, in_scale=1.0 / 1024 if fmt else 1.0)
    T = h.n_taps
    L = T + D * 3 * max(1, 65536 // M) + 5                               # several sub-tiles per channel
    x = _iq(L, fmt, seed=M + D + fmt)
    scale = 1.0 / 1024 if fmt else 1.0
    d_x = nat.DeviceArray.from_host(x)

    def run():
        y = h.exec(d_x, first_sample=12345)
        h.sync()
        return y.to_host()

    y, names = launched(run)
    _ran(case, names)
    want = cr.channelize(x, h.taps, M, D, first_sample=12345, in_scale=scale)
    bar = 1e-5 * cr.bound(h.taps, x, scale)
    assert y.shape == want.shape
    err = float(np.abs(y.astype(np.complex128) - want).max())
    assert err <= bar, f"{case['id']}: {err:.3e} > {bar:.3e}"
    h.close()


# ----------------------------------------------------------------------------- K11
def _run_detect(nat, case):
    from sdr_iq_visualizer_b200 import detect as det_mod
    from tests.test_detect_gpu import check, image
    db = image(200, 333, seed=5, smooth=True)                            # 7 x 11 tiles of 32 x 32
    d, names = launched(lambda: det_mod.detect_regions(db, 3.3, 3, want_labels=True))
    _ran(case, names)
    regions = check(d, db, 3.3, 3)
    assert len(regions) > 1


# ----------------------------------------------------------------------------- Welch finalize, ring carry, peer reduce
def _run_welch_finalize(nat, case):
    from sdr_iq_visualizer_b200 import spectral as sp
    n, hop, F, fs = 2048, 512, 400, 1.0e6
    x = _iq(n + hop * (F - 1), 0, seed=31)
    pl = sp.SpectralPlan(n, hop, "hann", 0)
    d_x = nat.DeviceArray.from_host(x)
    r = pl.stft(d_x, welch=True)
    pl.sync()
    (pxx, pdb), names = launched(lambda: pl.welch_finalize(r.welch_acc, F, fs))
    pl.sync()
    _ran(case, names)
    _, p_ref = sref.welch_psd(np.asarray(x, np.complex128), n, hop, "hann", fs)[:2]
    parity.check_power(pxx.to_host(), p_ref, what=f"{case['id']} pxx")
    assert np.abs(pdb.to_host() - 10 * np.log10(p_ref)).max() <= parity.DB_TOL
    pl.close()


def _run_ring(nat, case):
    from sdr_iq_visualizer_b200 import spectral as sp
    from sdr_iq_visualizer_b200.ring import StreamRing
    from tests.test_ring_gpu import _drive, _schedule, check_slots
    from tests.test_stft_gpu import oracle_rows
    n, hop, fmt, cap = 1024, 256, 1, 40_000
    chunks = _schedule(cap, hop)
    x = _iq(sum(chunks), fmt, seed=41)
    vmin, vmax = VRANGE[fmt]
    pl = sp.SpectralPlan(n, hop, "hann", fmt)
    ring = StreamRing(pl, n_slots=2, slot_samples=cap, wf_rows=True, welch=True, maxhold=True, vmin=vmin, vmax=vmax)
    blocks, names = launched(lambda: _drive(ring, x, fmt, chunks, 2))
    _ran(case, names)
    check_slots(blocks, oracle_rows(x, n, hop, "hann", fmt=fmt), n, "hann", fmt, ("u8",), what=case["id"])
    ring.close(); pl.close()


def _run_peer_reduce(nat, case):
    lib = nat.lib()
    N = 3 * 65536 + 17
    rng = np.random.default_rng(0)
    wl, ml = rng.random(N), rng.random(N).astype(np.float32)
    wo, mo = rng.random(N), rng.random(N).astype(np.float32)
    d = [nat.DeviceArray.from_host(a) for a in (wl, ml, wo, mo)]

    def run():
        nat.check(lib.spx_peer_reduce(0, d[0].ptr, d[1].ptr, d[2].ptr, d[3].ptr, N, None))
        nat.device_sync(0)

    _, names = launched(run)
    _ran(case, names)
    np.testing.assert_array_equal(d[2].to_host(), wo + wl)
    np.testing.assert_array_equal(d[3].to_host(), np.maximum(mo, ml))


RUNNERS = {"stft": _run_stft, "features": _run_features, "hist2d": _run_hist2d, "frame_stats": _run_frame_stats,
           "stream_frame": _run_stream_frame, "persistence": _run_persistence, "pool": _run_pool, "ddc": _run_ddc,
           "chan": _run_chan, "detect": _run_detect, "welch_finalize": _run_welch_finalize, "ring": _run_ring,
           "peer_reduce": _run_peer_reduce}


@pytest.mark.parametrize("case", ki.CASES, ids=[c["id"] for c in ki.CASES])
def test_instance(nat, case):
    RUNNERS[case["family"]](nat, case)
