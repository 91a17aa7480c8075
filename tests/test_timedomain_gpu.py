"""GPU tests of the time-domain views (K4): histogram counts bit-exact vs np.histogram2d, frame stats."""
import numpy as np
import pytest

from oracle import spectral_ref as sref

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def td():
    from sdr_iq_visualizer_b200 import timedomain, _native
    assert _native.device_count() > 0
    return timedomain


@pytest.mark.parametrize("r,bins", [(4.0, 256), (3.3, 256), (1.0, 64), (0.7, 100), (2.5, 1)])
def test_hist2d_cf32_bit_exact(td, r, bins):
    x = sref.synth_iq(1 << 18, seed=3).astype(np.complex64)
    # plant values exactly on edges, on the closed right edge, just outside, and NaN
    step = 2 * r / bins
    edges = np.linspace(-r, r, bins + 1)
    special = np.concatenate([edges, [np.nextafter(r, np.inf), np.nextafter(-r, -np.inf), r, -r, np.nan]]).astype(np.float32)
    x[: special.size] = special + 1j * special[::-1]
    h = td.iq_hist2d(x, r, bins)
    want = sref.iq_hist2d(x, r, bins)
    assert h.dtype == np.uint32 and h.shape == (bins, bins)
    np.testing.assert_array_equal(h, want)


def test_hist2d_ci16_and_accumulate(td):
    from sdr_iq_visualizer_b200 import _native as nat
    raw = sref.to_ci16(sref.synth_iq(1 << 18, seed=4))
    h = td.iq_hist2d(raw, 2048.0, 256, in_fmt=nat.FMT_CI16)
    want = sref.iq_hist2d(sref.unpack_ci16(raw), 2048.0, 256)
    np.testing.assert_array_equal(h, want)
    # scaled (SigMF ci16 autoscale) and non power-of-two range
    h2 = td.iq_hist2d(raw, 0.05, 256, in_fmt=nat.FMT_CI16, in_scale=2.0**-15)
    np.testing.assert_array_equal(h2, sref.iq_hist2d(sref.unpack_ci16(raw, 2.0**-15), 0.05, 256))
    # accumulate: two halves == whole; device-resident == host
    a = td.iq_hist2d(raw[: raw.size // 2], 2048.0, 256, in_fmt=nat.FMT_CI16)
    b = td.iq_hist2d(raw[raw.size // 2:], 2048.0, 256, in_fmt=nat.FMT_CI16, out=a, accumulate=True)
    np.testing.assert_array_equal(b, want)
    d = td.iq_hist2d(nat.DeviceArray.from_host(raw), 2048.0, 256, in_fmt=nat.FMT_CI16)
    nat.device_sync()
    np.testing.assert_array_equal(d.to_host(), want)


def test_config3_full_size(td):
    """BASELINE config 3: 16 Mi samples, 256x256 histogram (R = 4), 4096-sample frames."""
    L = 1 << 24
    x = sref.synth_iq(L, seed=3).astype(np.complex64)
    h = td.iq_hist2d(x, 4.0, 256)
    np.testing.assert_array_equal(h, sref.iq_hist2d(x, 4.0, 256))
    assert int(h.sum()) == L  # nothing falls outside R = 4 for this signal
    mean, peak = td.frame_stats(x, 4096, 4096)
    m_ref, p_ref = sref.frame_stats(x, 4096, 4096)
    assert mean.shape == (4096,)
    np.testing.assert_allclose(mean, m_ref, rtol=2e-7)
    np.testing.assert_allclose(peak, p_ref, rtol=2e-7)


def test_frame_stats_overlap_and_edges(td):
    from sdr_iq_visualizer_b200 import _native as nat
    x = sref.synth_iq(10_000, seed=8).astype(np.complex64)
    mean, peak = td.frame_stats(x, 1000, 300)
    m_ref, p_ref = sref.frame_stats(x, 1000, 300)
    assert mean.shape == m_ref.shape == (31,)
    np.testing.assert_allclose(mean, m_ref, rtol=2e-7)
    np.testing.assert_allclose(peak, p_ref, rtol=2e-7)
    mean, peak = td.frame_stats(x[:10], 1000)   # shorter than a frame
    assert mean.shape == (0,)
    raw = sref.to_ci16(x.astype(np.complex128))
    mean, peak = td.frame_stats(raw, 512, 512, in_fmt=nat.FMT_CI16)
    m_ref, p_ref = sref.frame_stats(sref.unpack_ci16(raw), 512, 512)
    np.testing.assert_allclose(mean, m_ref, rtol=2e-7)
    np.testing.assert_allclose(peak, p_ref, rtol=0)    # integers: exact


def test_hist2d_packed_counters_do_not_overflow_and_large_tables_fall_back(td):
    """Shared-memory path: every sample of a chunk in ONE bin (65 528 per chunk fits a 16-bit counter), odd bin
    counts (last packed word half used), unaligned device-side start (scalar loads); bins = 512 exceeds shared memory
    and takes the global-atomic kernel."""
    n = 1_000_003
    x = np.full(n, 0.3 - 0.2j, np.complex64)
    h = td.iq_hist2d(x, 1.0, 256)
    want = sref.iq_hist2d(x, 1.0, 256)
    assert h.sum() == n and np.array_equal(h, want) and h.max() == n
    rng = np.random.default_rng(8)
    y = (0.5 * (rng.standard_normal(300_001) + 1j * rng.standard_normal(300_001))).astype(np.complex64)
    for bins in (3, 255, 512):
        assert np.array_equal(td.iq_hist2d(y, 2.0, bins), sref.iq_hist2d(y, 2.0, bins)), bins
    assert np.array_equal(td.iq_hist2d(y[1:], 2.0, 256), sref.iq_hist2d(y[1:], 2.0, 256))   # host path re-stages: aligned again
    from sdr_iq_visualizer_b200 import _native as nat
    d = nat.DeviceArray.from_host(y)
    off = nat.DeviceView(d.ptr + 8, (y.size - 1,), np.complex64)                              # 8-byte offset: not 16-byte aligned
    got = td.iq_hist2d(off, 2.0, 256)
    nat.device_sync(0)                                                                        # device-memory calls are asynchronous
    assert np.array_equal(got.to_host(), sref.iq_hist2d(y[1:], 2.0, 256))


def test_hist2d_hot_counters_across_epochs_and_small_inputs(td):
    """One table per CTA for its whole share of the input: a CTA that meets the same bin in three or more epochs of
    32 760 samples must move the counter out before it can wrap (2^24 samples of two values -> ~113 k per CTA), the private
    tables are merged without atomics, and inputs of <= 4 epochs take the direct flush."""
    from sdr_iq_visualizer_b200 import _native as nat
    n = 1 << 24
    raw = np.empty(2 * n, np.int16)
    raw[0::2] = 100
    raw[1::2] = -7
    raw[2 * 5_000_000: 2 * 5_000_000 + 2 * 70_000: 2] = 101   # a second hot bin inside a few CTAs' shares
    rng = np.random.default_rng(21)
    idx = rng.integers(0, n, 50_000)
    raw[2 * idx] = rng.integers(-2047, 2048, idx.size).astype(np.int16)
    d = nat.DeviceArray.from_host(raw)
    h0 = nat.DeviceArray((256, 256), np.uint32, zero=True)
    got = td.iq_hist2d(d, 2048.0, 256, in_fmt=nat.FMT_CI16, out=h0)
    got = td.iq_hist2d(d, 2048.0, 256, in_fmt=nat.FMT_CI16, out=got, accumulate=True)        # twice: accumulate on the device
    nat.device_sync(0)
    i = raw[0::2].astype(np.float64)
    q = raw[1::2].astype(np.float64)
    want = np.histogram2d(i, q, bins=256, range=[[-2048.0, 2048.0]] * 2)[0].astype(np.uint32)
    assert np.array_equal(got.to_host(), 2 * want)
    assert int(want.max()) > 16_000_000
    for m in (1, 7, 32_759, 32_761, 4 * 32_760, 4 * 32_760 + 1, 5 * 32_760 + 3):                 # direct flush <-> merged tables
        x = sref.synth_iq(m, seed=m).astype(np.complex64)
        assert np.array_equal(td.iq_hist2d(x, 4.0, 256), sref.iq_hist2d(x, 4.0, 256)), m


@pytest.mark.parametrize("r,scale,bins", [(2048.0, 1.0, 256), (1.0, 2.0**-15, 256), (32768.0, 1.0, 256), (128.0, 1.0, 256),
                                          (64.0, 1.0, 256), (2048.0, 1.0, 64), (1000.0, 1.0, 250), (0.5, 2.0**-15, 192)])
def test_hist2d_ci16_integer_grid(td, r, scale, bins):
    """int16 input on a power-of-two bin grid (every product and edge exact: samples sit exactly ON edges, the estimate is
    shifted by half a grid step instead of using an edge zone) next to geometries that are not (1000 / 250, 192 bins):
    all int16 values, including start, stop (closed right edge), stop + 1 and the extremes."""
    from sdr_iq_visualizer_b200 import _native as nat
    rng = np.random.default_rng(int(r * 7) + bins)
    n = 1 << 18
    raw = rng.integers(-32768, 32768, 2 * n).astype(np.int16)
    k = int(round(r / scale))
    special = np.array([-k, k, -k - 1, k + 1, k - 1, -k + 1, 0, 1, -1, -32768, 32767], np.int64)
    special = special[(special >= -32768) & (special <= 32767)].astype(np.int16)
    raw[0:2 * special.size:2] = special
    raw[1:2 * special.size:2] = special[::-1]
    got = td.iq_hist2d(raw, r, bins, in_fmt=nat.FMT_CI16, in_scale=scale)
    want = sref.iq_hist2d(sref.unpack_ci16(raw, scale), r, bins)
    np.testing.assert_array_equal(got, want)
    assert got.sum() > 0


def test_hist2d_fuzz_against_numpy():
    """Randomised bins / range / scale / length / format with planted edge values, NaN, infinities and extremes
    (tools/fuzz_hist2d.py): every count equal to np.histogram2d."""
    import os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "fuzz_hist2d.py"), "120", "7"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "0 mismatches" in r.stdout


def test_plan_less_calls_on_every_device_and_bad_index(td):
    """The plan-less one-shot calls (histogram, frame stats, float64 stream frame, classifier measurements) keep their
    stream, staging and kernel set-up per device: on every device, after a first call on device 0, each returns exactly
    device 0's result, and a device index equal to the device count is rejected as an invalid argument."""
    from sdr_iq_visualizer_b200 import _native as nat, features, spectral
    n_dev = nat.device_count()
    x = sref.synth_iq(1 << 20, seed=17).astype(np.complex64)
    frame = x[:8192].astype(np.complex128)

    def run(dev):
        _, pdb = spectral.stream_frame(frame, 2.5e6, 9.15e8, device=dev)
        return (pdb, td.iq_hist2d(x, 4.0, 256, device=dev), td.frame_stats(x, 4096, 4096, device=dev),
                features.measure(pdb, device=dev))

    for call in (lambda: spectral.stream_frame(frame, 2.5e6, 9.15e8, device=n_dev),
                 lambda: td.iq_hist2d(x, 4.0, 256, device=n_dev),
                 lambda: td.frame_stats(x, 4096, 4096, device=n_dev),
                 lambda: features.measure(np.zeros(8192), device=n_dev)):
        with pytest.raises(nat.SpectralError) as e:
            call()
        assert e.value.code == nat.E_INVALID
    if n_dev < 2:
        pytest.skip("needs two GPUs")
    ref = run(0)
    for dev in range(n_dev):
        got = run(dev)
        np.testing.assert_array_equal(got[0], ref[0])
        np.testing.assert_array_equal(got[1], ref[1])
        np.testing.assert_array_equal(got[2][0], ref[2][0])
        np.testing.assert_array_equal(got[2][1], ref[2][1])
        assert got[3] == ref[3], dev
