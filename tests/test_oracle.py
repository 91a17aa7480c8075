"""CPU tests: the oracle against the reference's golden vectors and scipy.  No GPU needed."""
import json
import os

import numpy as np
import pytest
import scipy.signal

from oracle import classifier_ref as cref
from oracle import spectral_ref as sref

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_stream_frames_match_reference_golden(golden_stream):
    """oracle.stream_frame == reference SDRDataStreamer._stream_data (streamer.py:119-121)."""
    z, meta = golden_stream
    assert len(meta) == 9
    for m in meta:
        k = m["key"]
        f, p = sref.stream_frame(z[k + "_samples"], m["sample_rate"], m["center_freq"])
        np.testing.assert_array_equal(f, z[k + "_freqs"])
        np.testing.assert_array_equal(p, z[k + "_power_db"])
        # same thing through the generic STFT helpers (rect window, hop = N, one frame)
        rows = sref.stft_db_rows(z[k + "_samples"], m["n"], m["n"], sref.WINDOW_RECT)
        assert rows.shape == (1, m["n"])
        np.testing.assert_allclose(rows[0], z[k + "_power_db"], rtol=0, atol=1e-9)


def test_known_answers_ka3():
    """SURVEY.md 8(c) KA-3 frequency-axis values."""
    f = sref.freq_axis(4096, 61.44e6, 2.4e9)
    assert f[0] == 2.36928e9 and f[1] - f[0] == 15000.0
    f = sref.freq_axis(4096, 1e6, 2.4e9)
    assert f[0] == 2399500000.0 and f[-1] == 2400499755.859375 and f[1] - f[0] == 244.140625


def test_zero_buffer_gives_minus_240db(golden_stream):
    z, _ = golden_stream
    assert np.all(z["c0_2_power_db"] == -240.0)
    _, p = sref.stream_frame(np.zeros(64, complex), 1e6, 0)
    assert np.all(p == -240.0)


@pytest.mark.parametrize("nfft,hop,kind", [(1024, 1024, "hann"), (1024, 512, "hann"), (256, 64, "blackman"),
                                           (512, 512, "rect")])
def test_welch_matches_scipy(nfft, hop, kind):
    """mlab.psd restatement == scipy.signal.welch (the independent second anchor)."""
    x = sref.synth_iq(10000, seed=11)
    fs, fc = 1e6, 2.4e9
    f, pxx = sref.welch_psd(x, nfft, hop, kind, fs, fc)
    w = sref.window(kind, nfft)
    fsci, psci = scipy.signal.welch(x, fs, window=w, nperseg=nfft, noverlap=nfft - hop, detrend=False,
                                    return_onesided=False, scaling="density")
    np.testing.assert_allclose(pxx, np.fft.fftshift(psci), rtol=1e-12)
    np.testing.assert_allclose(f, np.fft.fftshift(fsci) + fc, rtol=0, atol=1e-3)
    # and the mean over spectrogram columns
    _, _, sxx = scipy.signal.spectrogram(x, fs, window=w, nperseg=nfft, noverlap=nfft - hop, detrend=False,
                                         return_onesided=False, scaling="density", mode="psd")
    np.testing.assert_allclose(pxx, np.fft.fftshift(sxx.mean(axis=1)), rtol=1e-12)


def test_framing_rules():
    assert sref.frame_count(2**20, 1024, 512) == 2047          # C1
    assert sref.frame_count(61_440_000, 4096, 1024) == 59_997  # C2
    assert sref.frame_count(2**30, 65536, 32768) == 32_767     # C5
    assert sref.frame_count(100, 1024, 512) == 0
    x = np.arange(20) + 0j
    fr = sref.frames(x, 8, 4)
    assert fr.shape == (4, 8) and fr[3, 0] == 12 and fr[3, -1] == 19
    assert sref.frames(x, 8, 5).shape == (3, 8)  # ragged tail dropped


def test_parseval_and_tone_bin():
    n = 4096
    x = sref.synth_iq(n, seed=3)
    p = sref.stft_power_rows(x, n, n, "rect")[0]
    np.testing.assert_allclose(p.sum(), n * np.sum(np.abs(x) ** 2), rtol=1e-12)
    t = np.exp(2j * np.pi * 100 * np.arange(n) / n)
    row = sref.stft_power_rows(t, n, n, "rect")[0]
    assert np.argmax(row) == n // 2 + 100 and abs(row.max() - n * n) < 1e-3


def test_unpack_ci16():
    raw = np.array([1, -2, 32767, -32768, 0, 5], dtype=np.int16)
    np.testing.assert_array_equal(sref.unpack_ci16(raw), np.array([1 - 2j, 32767 - 32768j, 5j]))
    np.testing.assert_array_equal(sref.unpack_ci16(raw, 2.0**-15), np.array([1 - 2j, 32767 - 32768j, 5j]) / 32768)


def test_waterfall_u8_rule():
    db = np.array([-200.0, -100.0, -99.99, -50.0, -0.01, 0.0, 10.0, -np.inf, np.nan])
    q = sref.waterfall_u8(db, -100.0, 0.0)
    np.testing.assert_array_equal(q, [0, 0, 0, 128, 255, 255, 255, 0, 0])
    lut = sref.viridis_lut()
    assert lut.shape == (256, 3) and tuple(lut[0]) == (0x44, 0x02, 0x55) or lut[0, 0] == 0x44
    assert tuple(lut[255])[0] >= 0xFC


def test_hist2d_edges():
    r = 4.0
    x = np.array([-4.0 - 4.0j, 4.0 + 4.0j, 0 + 0j, -1e-9 + 1e-9j, 4.0001 + 0j, 3.999 - 4.0j])
    h = sref.iq_hist2d(x, r)
    assert h.sum() == 5 and h[0, 0] == 1 and h[255, 255] == 1 and h[128, 128] == 1 and h[127, 128] == 1
    assert h[255, 0] == 1


def test_frame_stats():
    x = np.array([1 + 1j, 2 + 0j, 0 + 0j, 0 + 3j, 1 + 0j], dtype=complex)
    m, p = sref.frame_stats(x, 2, 2)
    np.testing.assert_allclose(m, [3.0, 4.5])
    np.testing.assert_allclose(p, [4.0, 9.0])


# ------------------------------------------------------------------ classifier oracle
def test_classifier_oracle_vs_golden(golden_classifier):
    z, res = golden_classifier
    for name, want in res["cases"].items():
        f, p = z[name + "_freqs"], z[name + "_power_db"]
        got = cref.features(f, p)
        assert got["noise_floor_db"] == want["noise_floor_db"], name
        assert got["adaptive_thr"] == want["adaptive_thr"], name
        assert got["peaks"] == want["peaks"], name
        assert [got["bw3"], got["bw10"], got["bw20"]] == want["bw"], name
        np.testing.assert_allclose(got["flatness"], want["flatness"], rtol=1e-13, atol=0, err_msg=name)
        np.testing.assert_allclose(got["kurtosis"], want["kurtosis"], rtol=1e-13, atol=0, err_msg=name)
        assert got["peak_spacing_std_hz"] == want["peak_spacing_std_hz"], name
        feats = want["advanced"]["features"]
        assert round(got["snr_db"], 2) == feats["snr_db"], name
        assert got["peak_count"] == feats["peak_count"], name


def test_known_answers_ka1_ka2(golden_classifier):
    """SURVEY.md 8(c) KA-1 / KA-2 values, via the oracle."""
    z, res = golden_classifier
    g = cref.features(z["ka1_cw_freqs"], z["ka1_cw_power_db"])
    assert abs(g["noise_floor_db"] - (-80.858940900062)) < 1e-9
    assert abs(g["adaptive_thr"] - (-69.773046810056)) < 1e-9
    assert g["peaks"] == [512] and g["min_distance_bins"] == 3
    assert g["bw3"] == 0.0 and abs(g["bw10"] - 1955.0342131108046) < 1e-6 and g["bw10"] == g["bw20"]
    assert abs(g["kurtosis"] - 282.091294420409) < 1e-6
    assert res["cases"]["ka1_cw"]["advanced"]["label"] == "CW Carrier"
    g = cref.features(z["ka2_wide_freqs"], z["ka2_wide_power_db"])
    assert (g["bw3"], g["bw10"], g["bw20"]) == (435000.0, 1485000.0, 23985000.0)
    assert g["peak_count"] == 2 and round(g["snr_db"], 2) == 41.36


def test_classifier_oracle_vs_reference_random():
    """Helper by helper against the reference's classifier on random spectra with ties (n = 3 ... 5000): its noise
    floor, peak pick, occupied bandwidths, flatness, kurtosis and peak spacing on these inputs are stored in
    tests/golden/classifier_random.{npz,json}."""
    z = np.load(os.path.join(GOLDEN, "classifier_random.npz"))
    with open(os.path.join(GOLDEN, "classifier_random.json")) as fh:
        cases = json.load(fh)["cases"]
    assert len(cases) == 28
    for want in cases:
        p = z[want["key"]] / 10.0       # dB rounded to 0.1 (forces ties), stored as int16 tenths
        assert p.size == want["n"]
        f = np.linspace(1e9, 1.02e9, p.size)
        g = cref.features(f, p)
        assert g["noise_floor_db"] == want["noise_floor_db"], want["key"]
        assert (g["adaptive_thr"], g["min_distance_bins"]) == (want["adaptive_thr"], want["min_distance_bins"]), want["key"]
        assert g["peaks"] == want["peaks"], want["key"]
        assert [g["bw3"], g["bw10"], g["bw20"]] == want["bw"], want["key"]
        assert abs(g["flatness"] - want["flatness"]) <= 1e-15, want["key"]
        assert abs(g["kurtosis"] - want["kurtosis"]) <= 1e-12 * max(1, abs(g["kurtosis"])), want["key"]
        assert g["peak_spacing_std_hz"] == want["peak_spacing_std_hz"], want["key"]
