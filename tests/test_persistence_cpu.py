"""CPU tests of the persistence spectrum (frames per uint8 waterfall level and bin): the oracle's definition on
hand-made rows, the shared-memory slot map of the kernel (restated in numpy), the dashboard payload, and the
host-side checks that run before any device call.  No CPU fallback exists: without a GPU the public entry points fail."""
import numpy as np
import pytest

from oracle import spectral_ref as sref
from tests import persistence_ref as pref

W = 128   # columns per strip of persist_kernel (csrc/spx_persist.cu)


def test_oracle_on_hand_made_rows():
    rows = np.array([[0, 255, 7], [0, 255, 7], [3, 0, 7], [0, 1, 8]], np.uint8)
    c = pref.persistence(rows)
    assert c.shape == (1, 256, 3) and c.dtype == np.uint32
    assert c[0, 0, 0] == 3 and c[0, 3, 0] == 1
    assert c[0, 255, 1] == 2 and c[0, 0, 1] == 1 and c[0, 1, 1] == 1
    assert c[0, 7, 2] == 3 and c[0, 8, 2] == 1
    np.testing.assert_array_equal(c.sum(axis=1), 4)
    assert int(c.sum()) == rows.size


def test_oracle_several_streams_and_column_sums():
    rng = np.random.default_rng(3)
    S, F, N = 3, 50, 37
    rows = rng.integers(0, 256, (S * F, N)).astype(np.uint8)
    c = pref.persistence(rows, S)
    assert c.shape == (S, 256, N)
    np.testing.assert_array_equal(c.sum(axis=1), F)
    for s in range(S):
        for j in (0, 17, N - 1):
            np.testing.assert_array_equal(c[s, :, j], np.bincount(rows[s * F:(s + 1) * F, j], minlength=256))


def test_oracle_nan_and_clip_levels():
    """Level 0 holds values below vmin and NaN, level 255 everything at or above vmax - D (A7 index)."""
    vmin, vmax = 20.0, 130.0
    d = (vmax - vmin) / 256
    db = np.array([[np.nan, -1e30, vmin - 1, vmin, vmin + d, vmax - d, vmax, 1e30, np.inf, -np.inf]])
    q = sref.waterfall_u8(db, vmin, vmax)
    np.testing.assert_array_equal(q[0], [0, 0, 0, 0, 1, 255, 255, 255, 255, 0])
    c = pref.persistence(np.repeat(q, 5, axis=0))
    assert c[0, 0, 0] == 5 and c[0, 0, 2] == 5 and c[0, 255, 6] == 5 and c[0, 1, 4] == 5


def test_oracle_zero_frames():
    c = pref.persistence(np.zeros((0, 16), np.uint8), 2)
    assert c.shape == (2, 256, 16) and not c.any()


def _slot(c):
    """persist_slot: column c of a 128-column strip -> counter slot within its level row."""
    return 32 * (c & 3) + (c >> 2)


def _col(p):
    """persist_col: the inverse."""
    return 4 * (p & 31) + (p >> 5)


def test_bank_map_is_a_permutation_and_conflict_free():
    c = np.arange(W)
    p = _slot(c)
    assert sorted(p) == list(range(W))
    np.testing.assert_array_equal(_col(p), c)
    np.testing.assert_array_equal(_slot(_col(c)), c)
    # lane l holds columns 4l .. 4l+3; for a fixed byte b the 32 lanes hit 32 distinct banks at ANY level q
    rng = np.random.default_rng(0)
    lanes = np.arange(32)
    for b in range(4):
        for _ in range(20):
            q = rng.integers(0, 256, 32)
            addr = q * W + _slot(4 * lanes + b)
            assert len(set(addr % 32)) == 32


def test_persistence_payload():
    from sdr_iq_visualizer_b200 import views
    N, F, vmin, vmax = 8, 40, -100.0, 0.0
    counts = np.zeros((256, N), np.uint32)
    counts[10] = 30
    counts[200] = 10
    p = views.persistence_payload(counts, F, vmin, vmax, freqs_mhz=np.arange(N) * 0.5)
    assert p["z"].dtype == np.float32 and p["z"].shape == (256, N)
    np.testing.assert_allclose(p["z"].sum(axis=0), 1.0)
    assert p["z"][10, 0] == np.float32(0.75) and p["z"][200, 3] == np.float32(0.25)
    assert len(p["y"]) == 256 and p["y"][0] == vmin and p["y"][1] == pytest.approx(vmin + (vmax - vmin) / 256)
    assert p["zmin"] == 0.0 and p["zmax"] == 1.0 and len(p["colorscale"]) > 2 and p["db_range"] == (vmin, vmax)
    # one stream of an [S][256][N] result is accepted as it is; F = 0 gives zeros, not NaN
    p0 = views.persistence_payload(np.zeros((1, 256, N), np.uint32), 0, vmin, vmax)
    assert not p0["z"].any()
    with pytest.raises(ValueError):
        views.persistence_payload(np.zeros((255, N), np.uint32), F, vmin, vmax)
    with pytest.raises(ValueError, match="streams"):     # several streams: the caller picks one
        views.persistence_payload(np.zeros((3, 256, N), np.uint32), F, vmin, vmax)


def _no_gpu():
    from sdr_iq_visualizer_b200 import _native as nat
    if nat.device_count() > 0:
        pytest.skip("a GPU is present")
    return nat


def test_no_cpu_fallback(tmp_path):
    nat = _no_gpu()
    from sdr_iq_visualizer_b200 import sigmf_io, spectral
    with pytest.raises(nat.SpectralError):
        spectral.SpectralPlan(1024).stft(np.zeros(4096, np.complex64), persistence=True, vmin=-100.0, vmax=0.0)
    base = sigmf_io.write_recording(str(tmp_path / "rec"), np.zeros(4096, np.complex64), 1e6, 0.0)
    with pytest.raises(nat.SpectralError):
        sigmf_io.process_recording(base, nfft=256, persistence=True)
    with pytest.raises(nat.SpectralError):   # shorter than one frame: still no fallback
        sigmf_io.process_recording(base, nfft=8192, persistence=True)


def _bare_plan(nfft=64, hop=64):
    """A SpectralPlan object without a native plan: enough for the checks stft() makes before calling libspx."""
    from sdr_iq_visualizer_b200 import spectral
    pl = spectral.SpectralPlan.__new__(spectral.SpectralPlan)
    pl.nfft, pl.hop, pl.in_fmt, pl.device, pl._h = nfft, hop, spectral.FMT_CF32, 0, None
    return pl


def test_python_side_buffer_checks():
    pl = _bare_plan()
    x = np.zeros(64 * 4, np.complex64)
    with pytest.raises(ValueError, match="persistence"):
        pl.stft(x, persistence=np.zeros((1, 256, 63), np.uint32), vmin=-100.0, vmax=0.0)
    with pytest.raises(ValueError, match="persistence"):
        pl.stft(x, persistence=np.zeros((1, 256, 64), np.int32), vmin=-100.0, vmax=0.0)
    with pytest.raises(ValueError, match="persistence"):
        pl.stft(x, n_streams=2, persistence=np.zeros((1, 256, 64), np.uint32), vmin=-100.0, vmax=0.0)
    with pytest.raises(ValueError, match="_time"):
        pl.stft(x, persistence=True, _time=(1, 1, False))
