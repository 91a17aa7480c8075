"""Kernel K3 (csrc/spx_features.cu) at the inputs where an order-statistic and comparison kernel goes wrong: NaN of
either sign bit, +-inf, rows that are all non-finite, +-0.0, subnormals, +-MAX, values one ulp apart, the radix select's
early exit and next-distinct-key search, the peak ballot's 1024-bin tile boundaries, n = 2^20, option overrides and
strided batches from every memory form.  Every field of `spx_features` and the peak list are held to the oracle
(`oracle/classifier_ref.features`), and to plain numpy for the fields the oracle does not return.  float32 rows are
held to the oracle of their float64 widening.

Comparison rules (`check`): integers and indices exact; NaN-ness and the sign of an infinity match; the order
statistics, peak, SNR and threshold exact (-0.0 == 0.0 accepted); flatness and kurtosis to 1e-11 relative;
mean and std to 1e-12 relative plus the rounding bound of a sum of n terms taken in another order; the peak-spacing
sigma to 1e-9 relative."""
import ctypes as C

import numpy as np
import pytest

from oracle import classifier_ref as cref

pytestmark = pytest.mark.gpu

DTYPES = [np.float64, np.float32]
DT_IDS = ["f64", "f32"]
NEG_NAN = np.copysign(np.nan, -1.0)          # a NaN with the sign bit set
INT_FIELDS = ("n", "argmax", "min_distance_bins", "first_3db", "last_3db", "first_10db", "last_10db", "first_20db",
              "last_20db", "simple_first", "simple_last", "n_candidates", "peak_count")
EXACT_FIELDS = ("peak_db", "noise_floor_db", "snr_db", "adaptive_thr", "p20_lo", "p20_hi")


@pytest.fixture(scope="module")
def feat():
    from sdr_iq_visualizer_b200 import _native, features
    assert _native.device_count() > 0
    return features


def reference(p, drops=(3.0, 10.0, 20.0), peak_threshold_db=None, min_distance_bins=0):
    """Every spx_features field and the peak list of one spectrum, in float64: the oracle's measurements, its helpers
    for the option overrides, and numpy for p20_lo / p20_hi (np.sort puts every NaN last), mean, std and the
    peak-spacing sigma in bins."""
    p = np.asarray(p, dtype=np.float64)
    n = p.size
    with np.errstate(all="ignore"):
        w = cref.features(np.arange(n, dtype=np.float64), p)
        thr = w["adaptive_thr"] if peak_threshold_db is None else float(peak_threshold_db)
        md = w["min_distance_bins"] if min_distance_bins <= 0 else int(min_distance_bins)
        cand = cref.peak_candidates(p, thr)
        peaks = cref.greedy_peaks(cand, md)
        lo = int(np.floor((n - 1) * 0.2))
        s = np.sort(p)
        r = {"n": n, "argmax": w["argmax"], "peak_db": w["peak_db"], "noise_floor_db": w["noise_floor_db"],
             "snr_db": w["snr_db"], "adaptive_thr": thr, "p20_lo": float(s[lo]), "p20_hi": float(s[min(lo + 1, n - 1)]),
             "min_distance_bins": md, "flatness": w["flatness"], "kurtosis": w["kurtosis"],
             "mean_db": float(np.mean(p)), "std_db": float(np.std(p)), "n_candidates": int(cand.size),
             "peak_count": len(peaks), "peaks": peaks,
             "peak_spacing_std_bins": float(np.std(np.diff(peaks))) if len(peaks) >= 3 else 0.0}
        for name, d in zip((3, 10, 20), drops):
            r[f"first_{name}db"], r[f"last_{name}db"] = cref.occupied_edges(p, d)
        r["simple_first"], r["simple_last"] = cref.occupied_edges(p, drops[2], strict=True)
    return r


def _same(g, w):
    """Exact, NaN-aware; -0.0 == 0.0."""
    return (np.isnan(g) and np.isnan(w)) or g == w


def _close(g, w, rtol, atol=0.0):
    if not (np.isfinite(g) and np.isfinite(w)):
        return _same(g, w)
    return abs(g - w) <= rtol * abs(w) + atol


def check(got, p, what, peaks=True, moments=True, **opts):
    """Every field of a K3 result against `reference` of the float64 widening of spectrum p.  `moments=False` leaves
    out the sums (mean, std, flatness, kurtosis) for spectra with +-MAX, whose sums overflow or cancel depending on the
    order they are taken in; `peaks=False` for results measured without a peak list."""
    p = np.asarray(p, dtype=np.float64)
    want = reference(p, **opts)
    for k in INT_FIELDS:
        assert got[k] == want[k], (what, k, got[k], want[k])
    for k in EXACT_FIELDS:
        assert _same(got[k], want[k]), (what, k, got[k], want[k])
    if peaks:
        assert got["peaks"] == want["peaks"] and got["peaks_stored"] == want["peak_count"], what
    else:
        assert got["peaks"] == [] and got["peaks_stored"] == 0, what
    assert _close(got["peak_spacing_std_bins"], want["peak_spacing_std_bins"], 1e-9), what
    if moments:
        assert _close(got["flatness"], want["flatness"], 1e-11, 1e-300), (what, got["flatness"], want["flatness"])
        assert _close(got["kurtosis"], want["kurtosis"], 1e-11), (what, got["kurtosis"], want["kurtosis"])
        # the kernel sums n / 1024 terms per thread and then a 1024-leaf tree, numpy pairwise: the two roundings of a
        # sum of n terms differ by at most (n/1024 + 32) eps of the sum of magnitudes
        fin = p[np.isfinite(p)]
        atol = (p.size / 1024 + 32) * np.finfo(np.float64).eps * (float(np.mean(np.abs(fin))) if fin.size else 0.0)
        for k in ("mean_db", "std_db"):
            assert _close(got[k], want[k], 1e-12, atol), (what, k, got[k], want[k])


def measure_rows(feat, rows, dtype, **opts):
    rows = np.ascontiguousarray(np.asarray(rows, dtype=dtype))
    return feat.measure_batch(rows, **opts)


def check_rows(feat, rows, dtype, what, moments=True, **opts):
    rows = [np.asarray(r, dtype=dtype) for r in rows]
    by_n = {}
    for i, r in enumerate(rows):
        by_n.setdefault(r.size, []).append(i)
    for n, idx in by_n.items():
        got = measure_rows(feat, [rows[i] for i in idx], dtype, **opts)
        for g, i in zip(got, idx):
            check(g, rows[i], f"{what} row {i} n={n}", moments=moments, **opts)


def noisy(n, seed, dtype=np.float64):
    """normal(-80, 3) with a +40 dB carrier a quarter of the way in."""
    p = np.random.default_rng(seed).normal(-80.0, 3.0, n)
    if n >= 3:
        p[n // 4] += 40.0
    return p.astype(dtype)


# ---------------------------------------------------------------- non-finite values

@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("n", [1, 2, 3, 1023, 1024, 1025, 4096, 100_000])
def test_non_finite_planted(feat, n, dtype):
    """NaN of both sign bits, +inf and -inf planted at bin 0, bin n - 1, the argmax, beside it and at the rank of the
    20th percentile; mixed rows; rows that are all NaN, all +inf, all -inf, and one finite value among -inf."""
    base = noisy(n, n, dtype)
    b64 = base.astype(np.float64)
    am = int(np.argmax(b64))
    lo = int(np.floor((n - 1) * 0.2))
    at = sorted({0, n - 1, am, max(am - 1, 0), min(am + 1, n - 1), int(np.argsort(b64, kind="stable")[lo])})
    rows = []
    for v in (np.nan, NEG_NAN, np.inf, -np.inf):
        for i in at:
            r = base.copy()
            r[i] = v
            rows.append(r)
    rng = np.random.default_rng(n + 1)
    for vals in ((np.nan, np.inf, -np.inf), (NEG_NAN, -np.inf), (np.inf, -np.inf)):   # mixed, at random bins
        r = base.copy()
        k = min(n, 3 * len(vals))
        r[rng.permutation(n)[:k]] = np.resize(np.array(vals), k)
        rows.append(r)
    for v in (np.nan, NEG_NAN, np.inf, -np.inf):
        rows.append(np.full(n, v, dtype))
    r = np.full(n, -np.inf, dtype)
    r[n // 2] = -75.5                                            # one finite value among -inf
    rows.append(r)
    r = np.where(np.arange(n) % 2 == 0, np.nan, -np.inf).astype(dtype)   # NaN and -inf only
    rows.append(r)
    check_rows(feat, rows, dtype, f"non-finite {np.dtype(dtype).name}")


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_non_finite_table(feat, dtype):
    """The four spectra of the issue's table, with the values the oracle gives spelled out: a NaN bin makes the peak,
    the noise floor and the threshold NaN (no edges, no peaks) and the argmax the NaN's index; one +inf bin leaves the
    threshold at nf + 5 (Python's max with a NaN second term); all -inf gives argmax 0, edges (0, n - 1) and NaN
    kurtosis."""
    got = measure_rows(feat, table_spectra(dtype), dtype)
    nan_row, inf_row, ninf_row, all_ninf = got
    assert np.isnan(nan_row["peak_db"]) and nan_row["argmax"] == 7 and np.isnan(nan_row["noise_floor_db"])
    assert nan_row["first_3db"] == -1 and nan_row["n_candidates"] == 0 and np.isnan(nan_row["kurtosis"])
    assert inf_row["peak_db"] == np.inf and inf_row["argmax"] == 7 and (inf_row["first_3db"], inf_row["last_3db"]) == (7, 7)
    assert inf_row["adaptive_thr"] == inf_row["noise_floor_db"] + 5.0 and inf_row["n_candidates"] > 0
    assert ninf_row["argmax"] == 1000 and np.isfinite(ninf_row["flatness"]) and np.isnan(ninf_row["kurtosis"])
    assert all_ninf["peak_db"] == -np.inf and all_ninf["argmax"] == 0 and np.isnan(all_ninf["noise_floor_db"])
    assert (all_ninf["first_3db"], all_ninf["last_3db"]) == (0, 4095) and all_ninf["simple_last"] == -1
    assert np.isnan(all_ninf["kurtosis"])
    for g, p, name in zip(got, table_spectra(dtype), ("NaN at 7", "+inf at 7", "-inf at 7", "all -inf")):
        check(g, p, name)


def table_spectra(dtype=np.float64):
    p = np.random.default_rng(2024).normal(-80.0, 3.0, 4096)
    p[1000] += 40.0
    rows = []
    for v in (np.nan, np.inf, -np.inf):
        r = p.copy()
        r[7] = v
        rows.append(r)
    rows.append(np.full(4096, -np.inf))
    return [r.astype(dtype) for r in rows]


# ---------------------------------------------------------------- order statistics

def _ulps(v, k, dtype):
    """v moved k ulps (away from zero for positive k), in dtype."""
    it = np.int64 if np.dtype(dtype) == np.float64 else np.int32
    return (np.asarray(v, dtype).view(it) + np.asarray(k, it)).view(dtype)


def _order_rows(dtype, seed):
    rng = np.random.default_rng(seed)
    fi = np.finfo(dtype)
    n = 4096
    lo = int(np.floor((n - 1) * 0.2))
    rows, no_moments = [], []
    rows.append(_ulps(dtype(-80.1), rng.integers(0, 6, n), dtype))                 # ties one ulp apart
    rows.append(rng.permutation(_ulps(dtype(-80.1), np.arange(n), dtype)))         # n distinct consecutive values
    rows.append(rng.permutation(_ulps(dtype(3.0e-3), np.arange(n) - n // 2, dtype)))
    z = np.where(rng.random(n) < 0.5, -0.0, 0.0).astype(dtype)                    # +-0.0 mixture around the rank
    z[rng.permutation(n)[: lo - 10]] = -1.0
    z[rng.permutation(n)[: 50]] = 1.0
    rows.append(z)
    rows.append(np.where(rng.random(n) < 0.5, -0.0, 0.0).astype(dtype))
    tiny = fi.smallest_subnormal
    rows.append((rng.integers(-50, 51, n) * tiny).astype(dtype))                  # subnormals (and zeros)
    s = (rng.integers(-3, 4, n) * tiny).astype(dtype)
    s[rng.permutation(n)[:100]] = fi.tiny                                           # smallest normal beside them
    rows.append(s)
    rows.append(rng.normal(0.0, 3.0, n).astype(dtype))                              # crossing zero
    rows.append(np.round(rng.normal(0.0, 2.0, n)).astype(dtype))                    # crossing zero, heavy ties
    u = np.empty(n, dtype)                                                          # unique lo-th element, then ties
    u[:lo] = rng.normal(-90.0, 2.0, lo).astype(dtype) - 20
    u[lo] = dtype(-81.25)
    u[lo + 1:] = dtype(-70.5)
    rows.append(rng.permutation(u))
    t = u.copy()                                                                    # unique lo-th, unique lo+1-th, ties
    t[lo + 1] = dtype(-71.0)
    rows.append(rng.permutation(t))
    e = u.copy()                                                                    # ties across lo and lo + 1
    e[lo - 3: lo + 5] = dtype(-81.25)
    rows.append(rng.permutation(e))
    rows.append(np.full(n, -80.25, dtype))                                          # all equal (exact sums)
    rows.append(np.full(n, -73.1, dtype))                                           # all equal
    for r in rows:
        no_moments.append(False)
    m = rng.normal(-80.0, 3.0, n).astype(dtype)                                     # +-MAX
    m[rng.permutation(n)[: lo + 3]] = -fi.max
    m[rng.permutation(n)[:5]] = fi.max
    rows.append(m)
    m2 = rng.choice(np.array([-fi.max, fi.max, _ulps(-fi.max, -1, dtype), 0.0], dtype), n)
    rows.append(m2)
    no_moments += [True, True]
    return rows, no_moments


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_order_statistics(feat, dtype):
    """Noise floor and p20_lo / p20_hi exact (and every other field) on one-ulp steps, +-0.0, subnormals, +-MAX,
    zero-crossing spectra, a unique lo-th element followed by ties (the radix select's early exit and its next-distinct
    search), ties across the rank, all values equal, and n = 1 (lo + 1 == n) for finite, signed-zero and non-finite
    values."""
    rows, no_moments = _order_rows(dtype, 11)
    for i, (r, nm) in enumerate(zip(rows, no_moments)):
        got = measure_rows(feat, [r], dtype)[0]
        check(got, r, f"order row {i}", moments=not nm)
    ones = [np.array([v], dtype) for v in (-80.3, -0.0, 0.0, np.inf, -np.inf, np.nan, NEG_NAN, np.finfo(dtype).max)]
    got = measure_rows(feat, np.stack(ones), dtype)
    for g, r in zip(got, ones):
        check(g, r, f"n=1 value {r[0]}")


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("n", [1 << 20, (1 << 19) + 1])
def test_order_statistics_largest(feat, n, dtype):
    """The largest PSD a plan makes (2^20 bins) and 2^19 + 1: distinct values, ties at 0.1 dB, and a NaN among them."""
    rng = np.random.default_rng(n)
    a = rng.normal(-80.0, 3.0, n)
    a[rng.integers(0, n, 40)] += 35.0
    b = np.round(a, 1)
    c = a.copy()
    c[n - 2] = np.nan
    rows = [r.astype(dtype) for r in (a, b, c)]
    got = measure_rows(feat, rows, dtype)
    for i, (g, r) in enumerate(zip(got, rows)):
        check(g, r, f"n={n} row {i}")


# ---------------------------------------------------------------- kurtosis threshold

@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_kurtosis_threshold(feat, dtype):
    """sigma exactly 0 gives kurtosis 0, sigma well above 1e-9 gives the 4th moment.  Spectra whose sigma lies within
    rounding of 1e-9 are not compared: K3's block sum and numpy's pairwise sum round differently, so the two can fall
    on either side of the threshold."""
    rng = np.random.default_rng(5)
    n = 4096
    zero = [np.full(n, -80.0, dtype), np.zeros(n, dtype), np.full(7, 12.5, dtype)]
    got = measure_rows(feat, zero[:2], dtype) + measure_rows(feat, zero[2:], dtype)
    for g, r in zip(got, zero):
        assert g["std_db"] == 0.0 and g["kurtosis"] == 0.0, r[0]
        check(g, r, f"sigma 0, value {r[0]}")
    rows = [rng.normal(0.0, sd, n).astype(dtype) for sd in (1e-7, 1e-5, 1e-3, 1.0, 30.0)]
    rows.append(noisy(n, 6, dtype))
    for g, r in zip(measure_rows(feat, rows, dtype), rows):
        assert g["kurtosis"] > 1.0, float(np.std(r.astype(np.float64)))
        check(g, r, f"sigma {np.std(r.astype(np.float64)):.1e}")


# ---------------------------------------------------------------- peak pick

@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_peaks_on_tile_boundaries(feat, dtype):
    """Strict maxima at i = 1022 ... 1026 and 2047 / 2048 (either side of the ballot loop's 1024-bin tiles), at bins
    1 and n - 2, two maxima across a tile edge, and plateaus, which are not strict maxima."""
    n = 4096
    rows = []
    for i in (1, 1022, 1023, 1024, 1025, 1026, 2047, 2048, n - 2):
        r = np.full(n, -100.0)
        r[i] = -50.0
        rows.append(r)
    r = np.full(n, -100.0)
    r[[1023, 1025]] = -50.0
    r[1024] = -60.0
    rows.append(r)
    for a, b in ((1023, 1025), (2047, 2049), (1022, 1023), (0, 2)):                 # plateaus [a, b)
        r = np.full(n, -100.0)
        r[a:b] = -50.0
        r[3000] = -40.0
        rows.append(r)
    r = np.full(n, -100.0)
    r[1020:1030] = -100.0 + np.array([1, 2, 3, 4, 5, 6, 5, 4, 3, 2])               # maximum at 1025 on a slope
    rows.append(r)
    rows = [r.astype(dtype) for r in rows]
    check_rows(feat, rows, dtype, "tile boundaries")
    check_rows(feat, rows, dtype, "tile boundaries, threshold -90, distance 1", peak_threshold_db=-90.0,
               min_distance_bins=1)


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("md", [1, 2])
def test_alternating_maxima_full_size(feat, md, dtype):
    """Every odd bin a strict maximum at n = 2^20: (n + 1) // 2 is the peak list's capacity, and all of them survive
    a distance of 1 or 2."""
    n = 1 << 20
    p = np.random.default_rng(md).normal(-80.0, 1.0, n)
    p[1::2] += 20.0
    rows = [p.astype(dtype)]
    got = measure_rows(feat, rows, dtype, min_distance_bins=md)[0]
    assert got["peak_count"] == n // 2 - 1                     # bin n - 1 is not interior
    check(got, rows[0], f"alternating md={md}", min_distance_bins=md)
    got = measure_rows(feat, rows, dtype, min_distance_bins=md, peak_threshold_db=-1000.0)[0]
    check(got, rows[0], f"alternating md={md} thr -1000", min_distance_bins=md, peak_threshold_db=-1000.0)


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_peak_options(feat, dtype):
    """min_distance_bins greater than n (up to INT32_MAX: the first candidate is always kept), fixed thresholds
    (including -inf, +inf and NaN), and drops of (0, 0.5, 120)."""
    rows = [noisy(n, n + 3, dtype) for n in (5, 1000, 4096)]
    rows.append(table_spectra(dtype)[1])
    for md in (3, 4097, 2**31 - 1):
        for r in rows:
            check_rows(feat, [r], dtype, f"distance {md}", min_distance_bins=md)
    for thr in (-85.0, -60.0, -np.inf, np.inf, np.nan):
        check_rows(feat, rows, dtype, f"threshold {thr}", peak_threshold_db=thr)
    check_rows(feat, rows, dtype, "drops 0/0.5/120", drops=(0.0, 0.5, 120.0))
    check_rows(feat, table_spectra(dtype), dtype, "table, drops 0/0.5/120", drops=(0.0, 0.5, 120.0))


# ---------------------------------------------------------------- input forms

def _mixed_batch(n, dtype):
    rows = [noisy(n, 40 + i, dtype) for i in range(6)]
    rows[1][[5, n // 2]] = np.nan
    rows[2][[0, 17]] = -np.inf
    rows[3][:] = -np.inf
    rows[4][9] = NEG_NAN
    rows[5][n // 4] = np.inf
    return rows


def _same_result(a, b, what, keys=None):
    for k in keys or a:
        x, y = a[k], b[k]
        if isinstance(x, float):
            assert (np.isnan(x) and np.isnan(y)) or (x == y and np.signbit(x) == np.signbit(y)), (what, k, x, y)
        else:
            assert x == y, (what, k, x, y)


def _host_strided(buf, n, batch, stride, dtype):
    """spx_classify_features on host memory with stride > n (measure_batch packs numpy input densely)."""
    from sdr_iq_visualizer_b200 import _native as nat
    from sdr_iq_visualizer_b200.features import _to_dict
    out = (nat.spx_features * batch)()
    cap = n // 3 + 2
    peaks = np.zeros((batch, cap), np.int32)
    opts = nat.spx_feature_opts()
    opts.drop_db[0], opts.drop_db[1], opts.drop_db[2] = 3.0, 10.0, 20.0
    nat.check(nat.lib().spx_classify_features(0, nat.MEM_HOST, buf.ctypes.data, 0 if dtype == np.float32 else 1, n, batch,
                                              stride, out, peaks.ctypes.data, cap, C.byref(opts), None))
    return [_to_dict(out[b], peaks[b]) for b in range(batch)]


@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_input_forms_strided_batch(feat, dtype):
    """One batch mixing finite, NaN and -inf rows, stride > n, from host memory, a DeviceArray, a torch tensor and
    FeatureQueue: each row equals the same row measured alone, and the oracle."""
    import torch
    from sdr_iq_visualizer_b200 import _native as nat
    n, stride = 4096, 4096 + 37
    rows = _mixed_batch(n, dtype)
    batch = len(rows)
    buf = np.full((batch, stride), -1.0e3, dtype)                 # padding that would change every field if read
    for b, r in enumerate(rows):
        buf[b, :n] = r
    alone = [feat.measure(r) for r in rows]
    for a, r in zip(alone, rows):
        check(a, r, "alone")
    d = nat.DeviceArray.from_host(buf)
    t = torch.from_numpy(buf).cuda()
    forms = {"host": _host_strided(buf, n, batch, stride, dtype),
             "DeviceArray": feat.measure_batch(d, n=n, batch=batch, stride=stride),
             "torch": feat.measure_batch(t, n=n, batch=batch, stride=stride)}
    torch.cuda.synchronize()
    for name, got in forms.items():
        for b in range(batch):
            _same_result(got[b], alone[b], f"{name} row {b}")
    fq = feat.FeatureQueue(batch=batch, slots=2)
    slots = [fq.enqueue(d, n, stride=stride, dtype=dtype) for _ in range(2)]
    nat.device_sync(0)
    keys = [k for k in alone[0] if k not in ("peaks", "peaks_stored")]
    for s in slots:
        for b, g in enumerate(fq.results(s)):
            _same_result(g, alone[b], f"FeatureQueue slot {s} row {b}", keys)
            check(g, rows[b], f"FeatureQueue row {b}", peaks=False)


# ---------------------------------------------------------------- end to end

def _nan_equal(a, b):
    if isinstance(a, dict):
        return isinstance(b, dict) and a.keys() == b.keys() and all(_nan_equal(a[k], b[k]) for k in a)
    if isinstance(a, (list, tuple)):
        return type(a) is type(b) and len(a) == len(b) and all(_nan_equal(x, y) for x, y in zip(a, b))
    if isinstance(a, float) and isinstance(b, float) and np.isnan(a) and np.isnan(b):
        return True
    return type(a) is type(b) and a == b


def _rules_on_oracle(clf, f, p):
    """What classify_signal_advanced / _simple return when the rule table is applied to the oracle's measurements
    (and their Hz fields) instead of K3's."""
    with np.errstate(all="ignore"):
        w = cref.features(f, p)
    m = {"snr_db": w["snr_db"], "flatness": w["flatness"], "kurtosis": w["kurtosis"], "bw3": w["bw3"], "bw10": w["bw10"],
         "bw20": w["bw20"], "peak_count": w["peak_count"], "peak_spacing_std_hz": w["peak_spacing_std_hz"]}
    _clear(clf)
    adv = clf.classify_from_measurements(f, m, len(p))
    first, last = w["simple_edges"]
    if last < 0:
        simple = "Noise"
    else:
        bw = f[last] - f[first]
        simple = "Narrowband" if bw < 3e6 else ("Wideband" if bw > 15e6 else "Unknown")
    return adv, simple


def _clear(clf):
    clf._CLASS_HISTORY.clear()
    clf._CONF_HISTORY.clear()


def _check_classification(clf, f, p, what):
    want_adv, want_simple = _rules_on_oracle(clf, f, p)
    _clear(clf)
    got = clf.classify_signal_advanced(f, p)
    _clear(clf)
    assert _nan_equal(got, want_adv), (what, got, want_adv)
    assert clf.classify_signal_simple(f, p) == want_simple, what
    return got


def test_classifier_on_non_finite_spectra(feat):
    """classify_signal_advanced / _simple on the table's four spectra: label, confidence, features, explanation and
    reasons equal the rule table on the oracle's measurements (NaN-aware), e.g. `kurt=nan` in the explanation."""
    from sdr_iq_visualizer_b200 import classifier as clf
    f = np.linspace(2.40e9, 2.42e9, 4096)
    for p, name in zip(table_spectra(), ("NaN at 7", "+inf at 7", "-inf at 7", "all -inf")):
        got = _check_classification(clf, f, p, name)
        assert "kurt=nan" in got["explanation"], (name, got["explanation"])


def test_stream_frame_with_nan_sample(feat):
    """One NaN sample in an rx buffer: the float64 per-buffer frame is NaN in every bin, as numpy's, and the classifier
    measurements and labels of that frame follow the oracle."""
    from oracle import spectral_ref as sref
    from sdr_iq_visualizer_b200 import classifier as clf, spectral as sp
    x = sref.synth_iq(4096, seed=9).astype(np.complex128)
    x[1234] = np.nan
    fs, fc = 2.5e6, 9.15e8
    f, p = sp.stream_frame(x, fs, fc)
    with np.errstate(all="ignore"):
        f_ref, p_ref = sref.stream_frame(x, fs, fc)
    np.testing.assert_array_equal(f, f_ref)
    assert np.isnan(p).all() and np.isnan(p_ref).all()
    check(feat.measure(p), p, "stream_frame")
    _check_classification(clf, f, p, "stream_frame")


def test_ring_slot_with_nan_sample(feat):
    """A NaN in one slot's samples makes that slot's Welch PSD NaN in every bin (the density rule of the ring tests),
    and each slot's on-device measurements equal the oracle's of that slot's PSD."""
    from oracle import spectral_ref as sref
    from sdr_iq_visualizer_b200 import spectral as sp
    from sdr_iq_visualizer_b200.ring import StreamRing
    from tests.test_dispatch_paths_gpu import _iq
    from tests.test_ring_gpu import RATE, check_density
    from tests.test_stft_gpu import oracle_rows
    n, hop, cap = 1024, 256, 8192
    x = _iq(3 * cap, 0, seed=21)
    x[cap + cap // 2] = np.nan                                   # inside the second slot's frames only
    pl = sp.SpectralPlan(n, hop, "hann")
    ring = StreamRing(pl, n_slots=3, slot_samples=cap, wf_rows=False, welch=True, maxhold=True, features=True,
                      sample_rate=RATE)
    blocks = []
    try:
        for s in range(3):
            ring.push(x[s * cap:(s + 1) * cap])
            b = ring.collect()
            blocks.append({"n_frames": b["n_frames"], "pxx_db": b["pxx_db"].copy(), "features": dict(b["features"])})
            ring.release()
    finally:
        ring.close()
        pl.close()
    with np.errstate(all="ignore"):
        X = oracle_rows(x, n, hop, "hann")
        P = X.real**2 + X.imag**2
    sum_w2 = float((sref.window("hann", n) ** 2).sum())
    f0, poisoned = 0, []
    for i, b in enumerate(blocks):
        sl = slice(f0, f0 + b["n_frames"])
        f0 += b["n_frames"]
        if np.isnan(P[sl]).any():
            poisoned.append(i)
            assert np.isnan(b["pxx_db"]).all(), i
        else:
            check_density(b["pxx_db"], P[sl], RATE, sum_w2, f"slot {i} pxx")
        check(b["features"], b["pxx_db"], f"slot {i}", peaks=False)
    assert poisoned == [1]
    assert np.isnan(blocks[1]["features"]["noise_floor_db"]) and np.isnan(blocks[1]["features"]["peak_db"])
