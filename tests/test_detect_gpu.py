"""Signal detection on the GPU (K11, spx_detect_regions / detect.detect_regions / sigmf_io.detect_signals) against the
float64 oracle (tests/detect_ref.py): every integer field, the peaks, the floors and the labels exact, power_sum within
1e-9 relative; non-finite input; determinism; every SPX_E_INVALID case; and a synthetic recording end to end."""
import ctypes as C

import numpy as np
import pytest

from tests import detect_ref as dr

pytestmark = pytest.mark.gpu

EXACT = ["row0", "row1", "col0", "col1", "n_cells", "peak_row", "peak_col", "peak_db", "peak_floor_db"]


def image(rows, cols, seed, smooth=False):
    rng = np.random.default_rng(seed)
    a = rng.normal(size=(rows, cols))
    if smooth and rows > 2 and cols > 2:   # blobs rather than single cells
        a = (a + np.roll(a, 1, 0) + np.roll(a, 1, 1) + np.roll(a, (1, 1), (0, 1))) / 2
    return (a * 3 - 90).astype(np.float32)


THR_5, THR_40 = 7.5, 3.3    # ~5 % and ~40 % of the cells of image() above floor + threshold


def check(det, db, thr, min_cells, labels=True):
    regions, lab, floors = dr.detect(np.asarray(db), thr, min_cells)
    assert det.n_total == len(regions) == len(det.regions)
    np.testing.assert_array_equal(det.row_floor_db, floors)
    assert det.row_floor_db.view(np.uint64)[~np.isnan(floors)].tolist() == floors.view(np.uint64)[~np.isnan(floors)].tolist()
    for k, (g, w) in enumerate(zip(det.regions, regions)):
        assert {f: g[f] for f in EXACT} == {f: w[f] for f in EXACT}, k
        if np.isinf(w["power_sum"]):
            assert g["power_sum"] == w["power_sum"]
        else:
            assert abs(g["power_sum"] - w["power_sum"]) <= 1e-9 * abs(w["power_sum"]), k
    if labels:
        got = det.labels
        if hasattr(got, "to_host"):
            got = got.to_host()
        elif hasattr(got, "cpu"):
            got = got.cpu().numpy()
        np.testing.assert_array_equal(got, lab)
    return regions


def detect(*a, **k):
    from sdr_iq_visualizer_b200 import detect as det_mod
    return det_mod.detect_regions(*a, **k)


# ----------------------------------------------------------------------------- exact match
@pytest.mark.parametrize("shape", [(1, 1), (1, 4096), (4096, 1), (1000, 1024), (3, 1 << 20)])
@pytest.mark.parametrize("thr", [THR_5, THR_40])
def test_shapes_match_oracle(shape, thr):
    db = image(*shape, seed=shape[0] + shape[1], smooth=True)
    check(detect(db, thr, 4, want_labels=True), db, thr, 4)


@pytest.mark.parametrize("thr", [THR_5, THR_40])
def test_4096_square_matches_oracle(thr):
    db = image(4096, 4096, seed=4096)
    check(detect(db, thr, 1, want_labels=True), db, thr, 1)


def test_1x1_above_its_own_floor():
    db = np.array([[-3.0]], np.float32)
    det = detect(db, 0.0, 1, want_labels=True)
    assert det.n_total == 1 and det.regions[0]["peak_db"] == -3.0 and det.labels.tolist() == [[1]]
    assert detect(db, 0.5, 1).n_total == 0


@pytest.mark.parametrize("min_cells", [1, 4, 10 ** 9])
def test_min_cells(min_cells):
    db = image(300, 257, seed=9, smooth=True)
    regions = check(detect(db, THR_5, min_cells, want_labels=True), db, THR_5, min_cells)
    assert (len(regions) == 0) == (min_cells == 10 ** 9)


def test_strided_rows_host_and_torch():
    import torch
    big = image(200, 700, seed=3, smooth=True)
    view = big[:, 37:37 + 600]
    assert view.strides[0] == 700 * 4
    check(detect(view, THR_5, 4, want_labels=True), np.ascontiguousarray(view), THR_5, 4)
    t = torch.from_numpy(big).cuda()[:, 37:37 + 600]
    assert t.stride(0) == 700
    check(detect(t, THR_5, 4, want_labels=True), np.ascontiguousarray(view), THR_5, 4)


def test_memory_spaces_agree():
    import torch
    from sdr_iq_visualizer_b200 import _native as nat
    db = image(513, 1000, seed=21, smooth=True)
    res = [detect(db, THR_40, 4, want_labels=True),
           detect(nat.DeviceArray.from_host(db), THR_40, 4, want_labels=True),
           detect(torch.from_numpy(db).cuda(), THR_40, 4, want_labels=True),
           detect(torch.from_numpy(db), THR_40, 4, want_labels=True)]
    for r in res:
        check(r, db, THR_40, 4)


def _raw(img, thr_db, mc, n_cap, **kw):
    from sdr_iq_visualizer_b200 import _native as nat
    db = np.ascontiguousarray(img, np.float32)
    out = (nat.spx_region * max(n_cap, 1))()
    n = C.c_int32(-7)
    args = dict(device=0, mem=nat.MEM_HOST, db=db.ctypes.data, rows=db.shape[0], cols=db.shape[1], stride=db.shape[1],
                thr=float(thr_db), min_cells=mc, regions=out, cap=n_cap, n=C.byref(n), labels=None, floors=None)
    args.update(kw)
    rc = nat.lib().spx_detect_regions(args["device"], args["mem"], args["db"], args["rows"], args["cols"], args["stride"],
                                      args["thr"], args["min_cells"], args["regions"], args["cap"], args["n"],
                                      args["labels"], args["floors"], None)
    return rc, n.value, out


def test_max_regions_below_total():
    from sdr_iq_visualizer_b200 import detect as det_mod
    db = image(400, 512, seed=5, smooth=True)
    regions, _, _ = dr.detect(db, THR_5, 4)
    assert len(regions) > 10
    for cap in (0, 3, len(regions) - 1):
        rc, n, out = _raw(db, THR_5, 4, cap, regions=None if cap == 0 else (det_mod.nat.spx_region * cap)())
        assert rc == 0 and n == len(regions)
    rc, n, out = _raw(db, THR_5, 4, 3)
    got = [{f: getattr(out[i], f) for f in EXACT} for i in range(3)]
    assert got == [{f: r[f] for f in EXACT} for r in regions[:3]]


# ----------------------------------------------------------------------------- non-finite input
def test_non_finite_cells_and_rows():
    db = image(64, 300, seed=8, smooth=True)
    db[3, 10] = np.nan                     # row 3 has a NaN floor: drops out whole
    db[5, ::7] = np.nan                    # and row 5
    db[7, :] = -np.inf                     # all -inf: NaN floor
    db[9, 40] = np.inf                     # +inf: in the mask, infinite power
    db[11, 41] = -np.inf                   # -inf: never in the mask
    db[20, 100:104] = np.float32(-np.inf)
    det = detect(db, THR_5, 1, want_labels=True)
    check(det, db, THR_5, 1)
    assert np.isnan(det.row_floor_db[[3, 5, 7]]).all()
    lab = det.labels
    assert not lab[[3, 5, 7]].any() and lab[9, 40] > 0 and lab[11, 41] == 0
    assert det.regions[lab[9, 40] - 1]["peak_db"] == np.inf


def test_peak_ties():
    db = np.full((6, 40), -100.0, np.float32)
    db[1, 3:9] = -20.0                    # one flat region: the first cell is the peak
    db[3, 20] = -0.0
    db[3, 21] = 0.0                       # -0 and +0 tie: the first wins, with its own value
    db[4, 22] = 0.0
    db[2, 30], db[4, 30], db[3, 31] = 5.0, 5.0, 5.0   # three-way tie across rows, 8-connected through (3, 31)
    db[3, 29] = 5.0
    det = detect(db, 6.0, 1, want_labels=True)
    regions = check(det, db, 6.0, 1)
    by_col = {r["col0"]: r for r in det.regions}
    assert (by_col[3]["peak_row"], by_col[3]["peak_col"]) == (1, 3)
    tie = by_col[20]
    assert (tie["peak_row"], tie["peak_col"]) == (3, 20) and np.signbit(tie["peak_db"])
    assert (by_col[29]["peak_row"], by_col[29]["peak_col"]) == (2, 30)
    assert len(regions) == 3


def test_row_floors_match_measure_batch():
    from sdr_iq_visualizer_b200 import features
    db = image(300, 1000, seed=12)
    db[4, 7] = np.nan
    db[6] = -np.inf
    det = detect(db, THR_5, 4)
    want = np.array([m["noise_floor_db"] for m in features.measure_batch(db, want_peaks=False)])
    assert det.row_floor_db.tobytes() == want.tobytes()


# ----------------------------------------------------------------------------- determinism
def test_two_runs_identical_bytes():
    db = image(2048, 2048, seed=31, smooth=True)
    a = detect(db, THR_40, 2, want_labels=True)
    b = detect(db, THR_40, 2, want_labels=True)
    strip = lambda d: [{k: v for k, v in r.items() if k != "power_sum"} for r in d.regions]
    assert strip(a) == strip(b)
    assert a.labels.tobytes() == b.labels.tobytes() and a.row_floor_db.tobytes() == b.row_floor_db.tobytes()


# ----------------------------------------------------------------------------- errors
def test_invalid_arguments():
    from sdr_iq_visualizer_b200 import _native as nat
    db = image(8, 16, seed=1)
    cases = [dict(device=99), dict(device=-1), dict(mem=7), dict(rows=-1), dict(cols=-1), dict(stride=15),
             dict(min_cells=0), dict(cap=-1), dict(db=None), dict(n=None), dict(regions=None, cap=4),
             dict(rows=1 << 16, cols=1 << 16, stride=1 << 16), dict(rows=46341, cols=46341, stride=46341)]
    for kw in cases:
        rc, _, _ = _raw(db, 6.0, 4, 4, **kw)
        assert rc == nat.E_INVALID, kw
    assert "INT32_MAX" in nat.last_error()
    for shape in ((0, 16), (8, 0), (0, 0)):
        rc, n, _ = _raw(np.zeros(shape, np.float32), 6.0, 4, 4, stride=max(shape[1], 1))
        assert rc == 0 and n == 0
    with pytest.raises(nat.SpectralError):
        detect(db, 6.0, 0)


# ----------------------------------------------------------------------------- a recording end to end
FS, FC, NFFT, K, B = 1.024e6, 100e6, 1024, 16, 4      # 1 kHz bins; overview rows of 16 frames, columns of 4 bins
F = 512 * K


def synth_recording(seed):
    """Noise plus three bursts on frame boundaries (hop = nfft): a CW tone on a bin centre for the middle third, a QPSK
    burst band-limited to 100 kHz, and a linear chirp.  Returns the samples and the true (frame0, frame1, f_lo, f_hi)."""
    rng = np.random.default_rng(seed)
    L = F * NFFT
    x = ((rng.normal(size=L) + 1j * rng.normal(size=L)) * 0.01).astype(np.complex128)
    truth = []
    # CW: bin 810 = +298 kHz, frames [2736, 5456)
    f0, f1 = 2736, 5456
    n = np.arange(f0 * NFFT, f1 * NFFT)
    x[n] += 0.0171 * np.exp(2j * np.pi * 298e3 * n / FS)
    truth.append((f0, f1, FC + 298e3, FC + 298e3))
    # QPSK: 128 kbaud, brick-wall filtered to bins 266 .. 365 ([-246.5, -146.5] kHz), frames [1024, 3072)
    f0, f1 = 1024, 3072
    nb = (f1 - f0) * NFFT
    sym = (rng.integers(0, 2, nb // 8) * 2 - 1 + 1j * (rng.integers(0, 2, nb // 8) * 2 - 1)) / np.sqrt(2)
    y = np.fft.fft(np.repeat(sym, 8))
    y[np.abs(np.fft.fftfreq(nb, 1 / FS)) > 50e3] = 0
    y = np.fft.ifft(y)
    y *= 0.044 / np.sqrt(np.mean(np.abs(y) ** 2))
    n = np.arange(f0 * NFFT, f1 * NFFT)
    x[n] += y * np.exp(2j * np.pi * -196.5e3 * n / FS)
    truth.append((f0, f1, FC - 246.5e3, FC - 146.5e3))
    # chirp: -50 kHz (bin 462) to +149 kHz (bin 661), frames [4096, 7168)
    f0, f1 = 4096, 7168
    t = np.arange((f1 - f0) * NFFT) / FS
    rate = 199e3 / t[-1]
    x[f0 * NFFT:f1 * NFFT] += 0.0171 * np.exp(2j * np.pi * (-50e3 * t + 0.5 * rate * t * t))
    truth.append((f0, f1, FC - 50e3, FC + 149e3))
    return x, truth


@pytest.mark.parametrize("datatype", ["cf32_le", "ci16_le"])
def test_detect_signals_end_to_end(tmp_path, datatype):
    from sdr_iq_visualizer_b200 import sigmf_io as sio
    x, truth = synth_recording(17)
    base = sio.write_recording(str(tmp_path / "three"), x, FS, FC, datatype)
    det, ann = sio.detect_signals(base, nfft=NFFT, overview=(512, 1024 // B))
    assert len(ann) == 3, ann
    cell_t, cell_f = K * NFFT, B * FS / NFFT
    for f0, f1, lo, hi in truth:
        a = min(ann, key=lambda a: abs(a["core:sample_start"] - f0 * NFFT) + abs(a["core:freq_lower_edge"] - lo))
        assert abs(a["core:sample_start"] - f0 * NFFT) <= cell_t, (a, f0)
        assert abs(a["core:sample_count"] - (f1 - f0) * NFFT) <= cell_t, (a, f1)
        assert abs(a["core:freq_lower_edge"] - lo) <= cell_f and abs(a["core:freq_upper_edge"] - hi) <= cell_f, (a, lo, hi)
        assert a["core:label"] == "signal" and a["core:generator"] == "sdr_iq_visualizer_b200"
    assert [a["core:sample_start"] for a in ann] == sorted(a["core:sample_start"] for a in ann)
    sio.write_annotations(base, ann)
    assert sio.fromfile(base).get_annotations() == ann
    with pytest.raises(TypeError):
        sio.detect_signals(base, zoom=(FC, 4))
