"""CPU tests of signal detection: K11's labelling passes (csrc/spx_detect_device.cuh, run on the host by
tests/emul/detect_emul.cu in seeded random orders of tiles and cells) against scipy.ndimage.label, the peak key's order,
the oracle's numbering, the region -> SigMF annotation mapping and write_annotations."""
import ctypes as C
import json
import os
import shutil
import subprocess

import numpy as np
import pytest

from tests import detect_ref as dr

EMUL_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emul", "detect_emul.cu")
ORDERS = 20          # random union orders per mask


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.fail("nvcc is needed to build the labelling harness")
    so = str(tmp_path_factory.mktemp("detect_emul") / "libdetect_emul.so")
    subprocess.run([nvcc, "-std=c++17", "-O2", "-shared", "-Xcompiler", "-fPIC", "-gencode",
                    "arch=compute_100a,code=sm_100a", "-o", so, EMUL_SRC], check=True)
    lib = C.CDLL(so)
    lib.emul_label.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_void_p]
    lib.emul_label.restype = C.c_int
    lib.emul_peak_keys.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    lib.emul_peak_keys.restype = None
    return lib


def emul_label(lib, mask, tile=(32, 32), seed=0):
    m = np.ascontiguousarray(mask, np.uint8)
    rows, cols = m.shape
    out = np.zeros((rows, cols), np.int32)
    n = lib.emul_label(m.ctypes.data, rows, cols, tile[0], tile[1], seed, out.ctypes.data)
    return out, n


def check_orders(lib, mask, tiles=((32, 32),), orders=ORDERS, seed0=0):
    want, n_want = dr.label(mask)
    for tile in tiles:
        for k in range(orders):
            got, n = emul_label(lib, mask, tile, seed0 + 1000 * k + 7)
            assert n == n_want, (tile, k)
            np.testing.assert_array_equal(got, want, err_msg=f"tile {tile}, order {k}")


# ----------------------------------------------------------------------------- labels == scipy in any union order
@pytest.mark.parametrize("density", [0.1, 0.3, 0.41, 0.6, 0.9])
@pytest.mark.parametrize("shape", [(70, 90), (97, 64)])
def test_random_masks(emul, density, shape):
    rng = np.random.default_rng(int(density * 100) + shape[0])
    mask = rng.random(shape) < density
    check_orders(emul, mask, tiles=((32, 32), (8, 8), (5, 7), (1, 16)))


@pytest.mark.parametrize("shape", [(1, 1), (1, 300), (300, 1), (31, 31), (32, 32), (33, 33), (31, 33), (33, 31), (32, 65),
                                   (65, 32), (1, 33), (33, 1)])
@pytest.mark.parametrize("density", [0.41, 0.9])
def test_edge_shapes(emul, shape, density):
    rng = np.random.default_rng(shape[0] * 1009 + shape[1])
    mask = rng.random(shape) < density
    check_orders(emul, mask)


def serpentine(rows, cols):
    """One 1-cell-thick path: full lines on even rows, joined alternately at the right and the left end."""
    m = np.zeros((rows, cols), bool)
    m[0::2] = True
    for r in range(1, rows, 2):
        m[r, cols - 1 if (r // 2) % 2 == 0 else 0] = True
    return m


@pytest.mark.parametrize("transpose", [False, True])
def test_serpentine_crosses_tile_borders(emul, transpose):
    m = serpentine(129, 96)
    m = m.T.copy() if transpose else m
    assert dr.label(m)[1] == 1
    # with 8 x 8 tiles the path crosses a tile edge over a thousand times
    check_orders(emul, m, tiles=((32, 32), (8, 8), (3, 5)))


def test_checkerboard_is_one_region(emul):
    m = (np.add.outer(np.arange(70), np.arange(67)) % 2).astype(bool)
    assert dr.label(m)[1] == 1
    check_orders(emul, m, tiles=((32, 32), (4, 4)))


@pytest.mark.parametrize("fill", [False, True])
def test_all_false_all_true(emul, fill):
    m = np.full((65, 70), fill)
    check_orders(emul, m, tiles=((32, 32), (7, 9)), orders=3)
    assert emul_label(emul, m)[1] == int(fill)


def test_diagonal_chirp_stays_one_region(emul):
    m = np.zeros((100, 100), bool)
    m[np.arange(100), np.arange(100)] = True       # diagonal only: 8-connected, not 4-connected
    check_orders(emul, m, tiles=((32, 32), (8, 8)))
    assert emul_label(emul, m)[1] == 1


# ----------------------------------------------------------------------------- peak key: numpy's max, first index
def test_peak_key_order(emul):
    rng = np.random.default_rng(5)
    specials = np.array([0.0, -0.0, np.inf, -np.inf, 1e-45, -1e-45, 3.4e38, -3.4e38, 7.0, 7.0], np.float32)
    for trial in range(200):
        n = int(rng.integers(1, 40))
        v = rng.choice(np.concatenate([specials, rng.normal(size=5).astype(np.float32)]), size=n).astype(np.float32)
        idx = np.sort(rng.choice(1 << 20, size=n, replace=False)).astype(np.int32)
        keys = np.zeros(n, np.uint64)
        emul.emul_peak_keys(v.ctypes.data, idx.ctypes.data, n, keys.ctypes.data)
        assert int(np.argmax(keys)) == int(np.argmax(v.astype(np.float64))), (v, idx)


# ----------------------------------------------------------------------------- the oracle
def test_oracle_numbering_is_first_cell_order():
    rng = np.random.default_rng(11)
    for _ in range(50):
        lab, n = dr.label(rng.random((40, 50)) < rng.uniform(0.05, 0.7))
        firsts = [int(np.flatnonzero(lab.ravel() == k)[0]) for k in range(1, n + 1)]
        assert firsts == sorted(firsts)


def test_oracle_filter_and_floors():
    db = np.full((4, 10), -100.0, np.float32)
    db[0, 2:5] = -80.0          # 3 cells
    db[2, 0] = -70.0            # 1 cell
    db[1, 7:9] = -60.0          # 2 cells, diagonal to nothing
    db[3, 4] = np.nan           # row 3 drops out
    regions, labels, floors = dr.detect(db, 6.0, min_cells=2)
    assert np.isnan(floors[3]) and floors[0] == -100.0
    assert [(r["row0"], r["col0"], r["n_cells"]) for r in regions] == [(0, 2, 3), (1, 7, 2)]
    assert labels[2, 0] == 0 and labels[0, 3] == 1 and labels[1, 8] == 2 and not labels[3].any()
    assert regions[1]["peak_col"] == 7 and regions[1]["peak_db"] == -60.0


# ----------------------------------------------------------------------------- region -> SigMF annotation
def test_annotation_k1_b1():
    from sdr_iq_visualizer_b200 import sigmf_io as sio
    r = {"row0": 3, "row1": 5, "col0": 10, "col1": 12, "peak_db": -40.0, "peak_floor_db": -52.5}
    a = sio.region_annotation(r, 1, 1, 100, 64, 16, 6400.0, 1e6, "burst")
    # rows 3..5 are frames 3..5: samples [48, 5*16 + 64); bins 10..12 of 64 at 100 Hz
    assert a["core:sample_start"] == 48 and a["core:sample_count"] == 5 * 16 + 64 - 48
    assert a["core:freq_lower_edge"] == 1e6 + (10 - 32 - 0.5) * 100.0
    assert a["core:freq_upper_edge"] == 1e6 + (13 - 32 - 0.5) * 100.0
    assert a["core:label"] == "burst" and a["core:generator"] == "sdr_iq_visualizer_b200"
    assert "12.5 dB" in a["core:comment"]


def test_annotation_pooled_short_last_row():
    from sdr_iq_visualizer_b200 import sigmf_io as sio
    # F = 10 frames in rows of K = 4: row 2 holds frames 8 and 9 only; B = 8 bins per column of N = 256
    r = {"row0": 1, "row1": 2, "col0": 0, "col1": 31, "peak_db": 0.0, "peak_floor_db": 0.0}
    a = sio.region_annotation(r, 4, 8, 10, 256, 128, 1.024e6, 0.0)
    assert a["core:sample_start"] == 4 * 128
    assert a["core:sample_count"] == 9 * 128 + 256 - 4 * 128
    assert a["core:freq_lower_edge"] == (0 - 128 - 0.5) * 4000.0
    assert a["core:freq_upper_edge"] == (256 - 128 - 0.5) * 4000.0
    r1 = dict(r, row0=0, row1=0, col0=5, col1=5)
    b = sio.region_annotation(r1, 4, 8, 10, 256, 128, 1.024e6, 0.0)
    assert b["core:sample_count"] == 3 * 128 + 256
    assert b["core:freq_lower_edge"] == (40 - 128.5) * 4000.0 and b["core:freq_upper_edge"] == (48 - 128.5) * 4000.0


def test_write_annotations_round_trip(tmp_path):
    from sdr_iq_visualizer_b200 import sigmf_io as sio
    x = (np.arange(64) * (1 + 1j)).astype(np.complex64)
    base = sio.write_recording(str(tmp_path / "rec"), x, 1e6, 915e6, description="kept")
    data_before = open(base + ".sigmf-data", "rb").read()
    meta_before = json.load(open(base + ".sigmf-meta"))
    ann = [{"core:sample_start": 40, "core:sample_count": 8, "core:label": "b"},
           {"core:sample_start": 3, "core:sample_count": 5, "core:label": "a", "core:freq_lower_edge": 9.1e8}]
    sio.write_annotations(base + ".sigmf-data", ann)
    rec = sio.fromfile(base)
    assert [a["core:label"] for a in rec.get_annotations()] == ["a", "b"]
    assert rec.get_annotations()[0] == ann[1] and rec.get_annotations()[1] == ann[0]
    meta_after = json.load(open(base + ".sigmf-meta"))
    for k in ("global", "captures"):
        assert meta_after[k] == meta_before[k]
    assert set(meta_after) == set(meta_before)
    assert open(base + ".sigmf-data", "rb").read() == data_before
    assert sorted(os.listdir(tmp_path)) == ["rec.sigmf-data", "rec.sigmf-meta"]
    sio.write_annotations(rec, [])
    assert sio.fromfile(base).get_annotations() == [] and rec.get_annotations() == []


def test_no_cpu_fallback():
    from sdr_iq_visualizer_b200 import _native as nat, detect
    if nat.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(nat.SpectralError):
        detect.detect_regions(np.zeros((4, 4), np.float32))
