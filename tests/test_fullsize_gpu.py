"""GPU tests at BASELINE.json's FULL sizes for the sharded configs, through size-independent properties
(SURVEY.md 8(c)/(d)): the captures are a synthetic block tiled on the device, so frames repeat with a known period and
the full-size result is determined by the oracle on one period.

  C5: 2^30 cf32 samples, 65536-pt Hann, 50 % overlap (32 767 frames, 2 GiB of rows)
  C4: 64 streams x 2^24 cf32 samples, 2048-pt Hann, 50 % overlap, per-stream Welch PSD + classifier features
"""
import numpy as np
import pytest

from oracle import classifier_ref as cref
from oracle import spectral_ref as sref
from tests import parity

pytestmark = pytest.mark.gpu


def _fill_tiled(nat, darr, block):
    lib, off = nat.lib(), 0
    while off < darr.nbytes:
        n = min(block.nbytes, darr.nbytes - off)
        nat.check(lib.spx_memcpy_h2d(darr.device, darr.ptr + off, block.ctypes.data, n))
        off += n


def _rows_to_host(nat, view, r0, r1, n):
    out = np.empty((r1 - r0, n), np.uint8)
    nat.check(nat.lib().spx_memcpy_d2h(view.device, out.ctypes.data, view.ptr + r0 * n, out.nbytes))
    return out


def test_config5_full_size_by_periodicity():
    from sdr_iq_visualizer_b200 import _native as nat, spectral as sp
    assert nat.device_count() > 0
    N, hop, L, B = 65536, 32768, 1 << 30, 1 << 22
    period = B // hop                                   # frames repeat every 128 frames
    block = sref.synth_iq(B, seed=5, tone_cycles_per_sample=20000.37 / 65536).astype(np.complex64)
    d_in = nat.DeviceArray((L,), np.complex64)
    _fill_tiled(nat, d_in, block)
    pl = sp.SpectralPlan(N, hop, "hann")
    F = pl.frame_count(L)
    assert F == 32767
    d_rows = nat.DeviceArray((F, N), np.uint8)
    r = pl.stft(d_in, wf_rows=d_rows, welch=True, maxhold=True, vmin=-20.0, vmax=110.0)
    pl.sync()
    assert r.n_frames == F
    # one period against the oracle (frames 0..127 see block + the first N - hop samples of the next copy)
    x1 = np.concatenate([block, block[: N - hop]])
    X = sref.shift_bins(sref.stft(sref.as_complex128(x1), N, hop, "hann"))
    assert X.shape[0] == period
    P = X.real**2 + X.imag**2
    first = _rows_to_host(nat, d_rows, 0, period, N)
    parity.check_u8(first, sref.amplitude_db(X), -20.0, 110.0, what="C5 first period")
    # periodicity: identical input frames give bit-identical rows wherever they sit in the capture (index map of the
    # batching, chunking and row placement at full size)
    for f in (period, 5 * period + 17, 100 * period + 127, F - 1 - ((F - 1) % period), F - 1):
        got = _rows_to_host(nat, d_rows, f, f + 1, N)
        assert np.array_equal(got[0], first[f % period]), f
    # Welch sum / max-hold over all 32 767 frames = the period's powers weighted by how often each frame occurs
    counts = np.bincount(np.arange(F) % period, minlength=period).astype(np.float64)
    parity.check_power(r.welch_acc.to_host()[0], (P * counts[:, None]).sum(axis=0), what="C5 full welch")
    parity.check_power(r.maxhold.to_host()[0], P.max(axis=0), what="C5 full maxhold")
    pl.close()


def test_config4_full_size_streams_and_features():
    from sdr_iq_visualizer_b200 import _native as nat, features, spectral as sp
    N, hop, Ls, S, B = 2048, 1024, 1 << 24, 64, 1 << 20
    period = B // hop
    base = sref.synth_iq(B, seed=100, tone_cycles_per_sample=300.37 / 2048).astype(np.complex64)
    d_in = nat.DeviceArray((S * Ls,), np.complex64)
    blocks = {}
    for s in range(S):
        blk = (np.roll(base, -(s * 4099)) * np.float32(1.0 + 0.01 * s)).astype(np.complex64)
        if s in (0, 31, 63):
            blocks[s] = blk
        _fill_tiled(nat, nat.DeviceView(d_in.ptr + s * Ls * 8, (Ls,), np.complex64), blk)
    pl = sp.SpectralPlan(N, hop, "hann")
    F = pl.frame_count(Ls)
    assert F == 16383
    r = pl.stft(d_in, n_streams=S, welch=True, maxhold=True, n_samples=Ls)
    pxx, pdb = pl.welch_finalize(r.welch_acc, F, 61.44e6, n_streams=S)
    feats = features.measure_batch(pdb, n=N, batch=S, stream=pl.stream)   # after the finalize on the plan's stream
    pxx_h = pxx.to_host().reshape(S, N)
    counts = np.bincount(np.arange(F) % period, minlength=period).astype(np.float64)
    w = sref.window("hann", N)
    fr = sref.freq_axis(N, 61.44e6, 0.0)
    for s, blk in blocks.items():
        x1 = np.concatenate([blk, blk[: N - hop]])
        X = sref.shift_bins(sref.stft(sref.as_complex128(x1), N, hop, "hann"))
        P = X.real**2 + X.imag**2
        want = (P * counts[:, None]).sum(axis=0) / F / (61.44e6 * np.sum(w**2))         # mlab.psd normalisation
        parity.check_power(pxx_h[s], want, what=f"C4 stream {s} welch psd")
        f = cref.features(fr, 10 * np.log10(want))
        m = feats[s]
        assert abs(m["snr_db"] - f["snr_db"]) < 2e-3 and abs(m["noise_floor_db"] - f["noise_floor_db"]) < 2e-3
        assert m["argmax"] == f["argmax"]
        for d in (3, 10, 20):                                                            # occupied-bandwidth edges: integer bins
            lo, hi = f["edges"][d]
            assert abs(m[f"first_{d}db"] - lo) <= 1 and abs(m[f"last_{d}db"] - hi) <= 1
    assert len({round(m["snr_db"], 3) for m in feats}) > 1                               # streams are distinct
    pl.close()
