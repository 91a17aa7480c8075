"""GPU parity tests of the STFT dispatch decisions that the per-family tests do not reach: K2 (two-kernel four-step path)
with several scratch batches and without bulk copies, N = 65536 falling back from K2v2 to K2, the per-stream loops of every
family, streams that fall back to another kernel inside one call, unaligned device input, Bluestein with several batches,
small host-pipeline pieces, and the scratch ordering between a device-resident call and a host-memory call.

Two plan-creation environment knobs make the batch and piece boundaries reachable at test sizes:
SPX_BIG_SCRATCH_BYTES (four-step scratch; frames per K2 batch = bytes / 2 / (N * 8)) and SPX_H2D_PIECE_BYTES (host
pipeline piece; max(bytes / sample size, 4 N) samples).  Every case proves that its path ran by the names of the kernels
the CUDA profiler saw, and checks every produced row and every stream's accumulators against the float64 oracle."""
import re

import numpy as np
import pytest

from oracle import spectral_ref as sref
from tests import parity
from tests.test_stft_gpu import oracle_rows

pytestmark = pytest.mark.gpu

ALL_OUTS = dict(db_rows=True, wf_rows=True, spectrum=True, welch=True, maxhold=True)
U8_ACC = dict(wf_rows=True, welch=True, maxhold=True)     # the outputs K2v2 serves (N = 65536)
VRANGE = {0: (-40.0, 90.0), 1: (20.0, 150.0)}              # vmin, vmax per input format (cf32, ci16)

# demangled kernel names (template arguments as the compiler prints them)
K1_STAGED = r"\bstft_kernel<\d+, \d+, (?:true|false), \d+, \d+, true"
K1_DIRECT = r"\bstft_kernel<\d+, \d+, (?:true|false), \d+, \d+, false"
K1V2 = r"\bstft2_(?:strip_)?kernel<"
K2_COLS_BULK = r"\bbig_cols_kernel<\d+, \d+, \d+, true>"
K2_COLS_DIRECT = r"\bbig_cols_kernel<\d+, \d+, \d+, false>"
K2_ROWS = r"\bbig_rows_kernel<"
K2V2 = r"\bbig2_kernel<"
BLU_PRE = r"\bblu_pre_kernel<"


@pytest.fixture(scope="module")
def sp():
    from sdr_iq_visualizer_b200 import spectral
    from sdr_iq_visualizer_b200 import _native
    assert _native.device_count() > 0, "GPU tests need a CUDA device (no CPU fallback exists)"
    return spectral


def launched(fn):
    """Run fn() under the CUDA profiler; return (its result, the names of the kernels launched, in order)."""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    from sdr_iq_visualizer_b200 import _native as nat
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        nat.device_sync(0)
    names = [e.name for e in prof.events() if e.device_type == DeviceType.CUDA and "kernel" in e.name]
    print("kernels:", sorted(set(names)))
    return out, names


def count(names, pat):
    return sum(1 for nm in names if re.search(pat, nm))


def _iq(L, fmt, seed, S=1):
    """S streams of L samples back to back: complex64, or interleaved int16 for ci16."""
    xc = np.concatenate([sref.synth_iq(L, seed=seed + s, snr_db=10.0 + 5.0 * s) for s in range(S)])
    return sref.to_ci16(xc) if fmt else xc.astype(np.complex64)


def _cut(x, fmt, a, b):
    """Samples [a, b) of a host input."""
    return x[2 * a: 2 * b] if fmt else x[a:b]


def _host(a):
    return a.to_host() if hasattr(a, "to_host") else a


def _oracle(x, n, hop, kind, fmt, S, sel):
    """float64 reference of an S-stream input: the rows of frames `sel` of every stream ([s][f] order), and every stream's
    Welch sum and max-hold over all its frames (accumulated in frame chunks to bound host memory)."""
    L = (x.size // 2 if fmt else x.size) // S
    F = sref.frame_count(L, n, hop)
    chunk = max(1, (1 << 22) // n)
    want = set(sel)
    rows, welch, mh = [], np.zeros((S, n)), np.zeros((S, n))
    for s in range(S):
        xs = _cut(x, fmt, s * L, (s + 1) * L)
        for f0 in range(0, F, chunk):
            f1 = min(F, f0 + chunk)
            X = oracle_rows(_cut(xs, fmt, f0 * hop, (f1 - 1) * hop + n), n, hop, kind, fmt=fmt)
            P = X.real**2 + X.imag**2
            welch[s] += P.sum(axis=0)
            mh[s] = np.maximum(mh[s], P.max(axis=0))
            rows.extend(X[f - f0] for f in range(f0, f1) if f in want)
    return np.array(rows), welch, mh


def check_oracle(r, x, n, hop, kind, fmt, S=1, sel=None, acc_times=1, what=""):
    """Every produced row of frames `sel` (all frames by default) of every stream, and every stream's accumulators
    (`acc_times` calls' worth of the same input), against the oracle."""
    F = r.n_frames
    sel = list(range(F)) if sel is None else sorted(set(sel))
    X, welch, mh = _oracle(x, n, hop, kind, fmt, S, sel)
    idx = [s * F + f for s in range(S) for f in sel]
    P = X.real**2 + X.imag**2
    vmin, vmax = VRANGE[fmt]
    if r.spectrum is not None:
        # the fp32 FFT bar of each family's own parity test (test_stft_gpu.py)
        if n & (n - 1) == 0 and n <= 8192:
            bound = 5e-6 * np.sqrt(P.mean())
        else:
            bound = 6e-6 * np.sqrt(P.mean()) + (1e-6 if n & (n - 1) == 0 else 2e-6) * np.abs(X) + 1e-7 * np.abs(X).max()
        ratio = np.abs(_host(r.spectrum)[idx] - X) / bound
        parity._record("spectrum", what, bins=int(X.size), worst_ratio_to_bound=float(ratio.max()))
        assert ratio.max() <= 1.0, f"{what}: spectrum error {ratio.max():.3f} x the bound"
    if r.db_rows is not None:
        parity.check_db_rows(_host(r.db_rows)[idx], P, what=f"{what} dB rows")
    if r.wf_rows is not None:
        parity.check_u8(_host(r.wf_rows)[idx], sref.amplitude_db(X), vmin, vmax, what=f"{what} u8")
    for s in range(S):
        if r.welch_acc is not None:
            parity.check_power(_host(r.welch_acc)[s], acc_times * welch[s], what=f"{what} welch s={s}")
        if r.maxhold is not None:
            parity.check_power(_host(r.maxhold)[s], mh[s], what=f"{what} maxhold s={s}")


def _edges(F, fb):
    """First and last frame and the frames on each side of every batch boundary."""
    sel = {0, F - 1}
    for b in range(fb, F, fb):
        sel |= {b - 1, b}
    return sorted(sel)


# ----------------------------------------------------------------------------- K2 scratch batches (two halves, aux stream)
@pytest.mark.parametrize("bulk", [True, False])
@pytest.mark.parametrize("fmt", [0, 1])
@pytest.mark.parametrize("n", [16384, 32768, 131072])
def test_k2_scratch_batches(sp, monkeypatch, n, fmt, bulk):
    """K2 through a 1 MiB scratch (fb = 4, 2, 1 frames per batch): one batch, exactly full halves, batches wrapping past
    the wait on the half that batch k-2 used, and a short last batch; accumulate=True on a second call.  A hop that is
    not a multiple of 16 bytes takes the column kernel without bulk copies.  Against the same plan at the default scratch
    (one batch): rows and max-hold bit-identical (same per-frame arithmetic), Welch within 1e-6 (fp32 partials regroup)."""
    elt = 4 if fmt else 8
    fb = max(1, (1 << 20) // 2 // (n * 8))
    hop = n // 2 if bulk else n // 2 + (2 if fmt else 1)
    assert ((hop * elt) % 16 == 0) == bulk
    monkeypatch.setenv("SPX_BIG_SCRATCH_BYTES", str(1 << 20))
    small = sp.SpectralPlan(n, hop, "hann", fmt)
    monkeypatch.delenv("SPX_BIG_SCRATCH_BYTES")
    ref = sp.SpectralPlan(n, hop, "hann", fmt)
    vmin, vmax = VRANGE[fmt]
    counts = sorted({F for F in (fb - 1, fb, fb + 1, 2 * fb + 1, 3 * fb + 2) if F >= 1})
    xall = _iq(n + hop * (counts[-1] - 1) + 5, fmt, seed=n // 1000 + fmt)
    for F in counts:
        x = _cut(xall, fmt, 0, n + hop * (F - 1) + 5)
        r, names = launched(lambda: small.stft(x, **ALL_OUTS, vmin=vmin, vmax=vmax))
        assert r.n_frames == F
        batches = -(-F // fb)
        assert count(names, K2_COLS_BULK if bulk else K2_COLS_DIRECT) == batches, names
        assert count(names, K2_COLS_DIRECT if bulk else K2_COLS_BULK) == 0 and count(names, K2_ROWS) == batches
        check_oracle(r, x, n, hop, "hann", fmt, what=f"K2 N={n} F={F} fb={fb}")
        r2 = small.stft(x, welch=r.welch_acc.copy(), maxhold=r.maxhold.copy(), accumulate=True)
        check_oracle(r2, x, n, hop, "hann", fmt, acc_times=2, what=f"K2 N={n} F={F} accumulate")
        r0 = ref.stft(x, **ALL_OUTS, vmin=vmin, vmax=vmax)
        for k in ("db_rows", "wf_rows", "spectrum", "maxhold"):
            np.testing.assert_array_equal(getattr(r, k), getattr(r0, k), err_msg=k)
        np.testing.assert_allclose(r.welch_acc, r0.welch_acc, rtol=1e-6)
    small.close(); ref.close()


def test_k2_real_batch_size_device_resident(sp):
    """Device-resident K2 at the default scratch: N = 16384 has 1536 frames per batch, so 1540 frames make a full batch
    and a 4-frame tail on the other half."""
    from sdr_iq_visualizer_b200 import _native as nat
    n, hop, F = 16384, 4096, 1540
    x = _iq(n + hop * (F - 1), 0, seed=15)
    pl = sp.SpectralPlan(n, hop, "hann")
    d_in = nat.DeviceArray.from_host(x)
    r, names = launched(lambda: pl.stft(d_in, db_rows=True, wf_rows=True, welch=True, maxhold=True, vmin=-40.0, vmax=90.0))
    assert r.n_frames == F
    assert count(names, K2_COLS_BULK) == 2 and count(names, K2_COLS_DIRECT) == 0, names
    check_oracle(r, x, n, hop, "hann", 0, sel=[0, 1, 2] + list(range(1533, 1540)), what="K2 real batch")
    pl.close()


# ----------------------------------------------------------------------------- N = 65536: K2v2 -> K2 fallbacks
@pytest.mark.parametrize("hop,fmt,offset", [(32896, 0, 0), (32896, 1, 0), (30001, 0, 0), (30001, 1, 0), (32768, 0, 8), (32768, 1, 4)])
def test_65536_falls_back_to_k2(sp, hop, fmt, offset):
    """N = 65536 with the outputs K2v2 serves, but a hop that is not a multiple of 256 samples (32896 is still a multiple of
    16 bytes: bulk copies; 30001 is not) or a device input `offset` bytes past a 16-byte boundary: K2 runs instead.
    Oracle parity, and the agreement bounds used for K2v2 against the two-kernel path (variant 1)."""
    from sdr_iq_visualizer_b200 import _native as nat
    n, F = 65536, 5
    elt = 4 if fmt else 8
    vmin, vmax = VRANGE[fmt]
    x = _iq(n + hop * (F - 1) + 77, fmt, seed=hop + fmt)
    pl = sp.SpectralPlan(n, hop, "hann", fmt)
    old = sp.SpectralPlan(n, hop, "hann", fmt, variant=1)
    if offset:
        pad = np.concatenate([np.zeros(offset // x.itemsize, x.dtype), x])
        d_pad = nat.DeviceArray.from_host(pad)
        src = nat.DeviceView(d_pad.ptr + offset, x.shape, x.dtype, keep=d_pad)
    else:
        src = x
    r, names = launched(lambda: pl.stft(src, **U8_ACC, vmin=vmin, vmax=vmax))
    assert r.n_frames == F
    bulk = offset == 0 and (hop * elt) % 16 == 0
    assert count(names, K2V2) == 0, names
    assert count(names, K2_COLS_BULK if bulk else K2_COLS_DIRECT) == 1 and count(names, K2_ROWS) == 1, names
    check_oracle(r, x, n, hop, "hann", fmt, what=f"65536 fallback hop={hop} +{offset}B")
    r0 = old.stft(x, **U8_ACC, vmin=vmin, vmax=vmax)
    wf = _host(r.wf_rows)
    assert np.abs(wf.astype(np.int16) - r0.wf_rows.astype(np.int16)).max() <= 1
    assert (wf != r0.wf_rows).mean() < 2e-3
    parity.check_power(_host(r.welch_acc)[0], r0.welch_acc[0], what="65536 fallback welch vs variant 1", rel_tol=1.5e-4)
    parity.check_power(_host(r.maxhold)[0], r0.maxhold[0], what="65536 fallback maxhold vs variant 1", rel_tol=1.5e-4)
    pl.close(); old.close()


# ----------------------------------------------------------------------------- several streams, every family
MS_FAMILIES = {512: (128, 40, K1_STAGED, K1_DIRECT), 4096: (1024, 20, K1V2, K1_DIRECT), 16384: (8192, 6, K2_COLS_BULK, K2_COLS_DIRECT),
               65536: (32768, 5, K2V2, K2_COLS_DIRECT), 1000: (250, 12, BLU_PRE, None), 100000: (50000, 3, BLU_PRE, None)}


@pytest.mark.parametrize("mem", ["host", "device"])
@pytest.mark.parametrize("odd", [False, True])
@pytest.mark.parametrize("n", sorted(MS_FAMILIES))
def test_three_streams_every_family(sp, n, odd, mem):
    """S = 3 streams of L samples.  L a multiple of 16 samples keeps every stream 128-byte aligned; an odd L puts streams
    1 and 2 eight bytes off.  The host pipeline and the per-stream loops of K2, K2v2 and Bluestein then run the fast
    kernel on stream 0 and the fallback on the others inside one call; a device-resident K1 / K1v2 launch covers all
    streams with one stride and falls back for all of them."""
    from sdr_iq_visualizer_b200 import _native as nat
    S = 3
    hop, F, fast, slow = MS_FAMILIES[n]
    L = -(-(n + hop * (F - 1) + 3) // 16) * 16 + (1 if odd else 0)
    x = _iq(L, 0, seed=n % 997, S=S)
    outs = U8_ACC if n == 65536 else ALL_OUTS
    pl = sp.SpectralPlan(n, hop, "hann")
    src = x if mem == "host" else nat.DeviceArray.from_host(x)
    r, names = launched(lambda: pl.stft(src, n_streams=S, **outs, vmin=-40.0, vmax=90.0))
    assert r.n_frames == F
    if slow is None:    # Bluestein reads the input with plain loads: one batch per stream
        assert count(names, fast) == S, names
    else:
        per_stream = mem == "host" or n >= 16384
        assert (count(names, fast) > 0) == (not odd or per_stream), names
        assert (count(names, slow) > 0) == odd, names
        if n == 65536:   # one K2v2 launch per 16-byte aligned stream (s * L * 8 bytes in), one K2 pair per other stream
            aligned = sum((s * L * 8) % 16 == 0 for s in range(S))
            assert count(names, fast) == aligned and count(names, slow) == S - aligned, names
    check_oracle(r, x, n, hop, "hann", 0, S=S, what=f"S={S} N={n} L={L} {mem}")
    pl.close()


# ----------------------------------------------------------------------------- unaligned device input
@pytest.mark.parametrize("fmt", [0, 1])
@pytest.mark.parametrize("n,hop,F", [(1024, 512, 60), (4096, 1024, 30), (65536, 32768, 4), (3000, 1500, 10)])
def test_unaligned_device_input(sp, n, hop, F, fmt):
    """A device view one sample past an aligned allocation (+8 bytes cf32, +4 bytes ci16): K1v2 falls back to K1 with
    direct loads, K2v2 to K2 without bulk copies; Bluestein reads with plain loads either way.  Against the oracle and
    against the same data in an aligned buffer (bit-identical where the kernel is the same; otherwise the bars the suite
    uses between K1v2 and K1, and between K2v2 and K2)."""
    from sdr_iq_visualizer_b200 import _native as nat
    vmin, vmax = VRANGE[fmt]
    x = _iq(n + hop * (F - 1) + 9, fmt, seed=n + fmt)
    per = 2 if fmt else 1
    d_al = nat.DeviceArray.from_host(x)
    d_pad = nat.DeviceArray.from_host(np.concatenate([np.zeros(per, x.dtype), x]))
    d_un = nat.DeviceView(d_pad.ptr + per * x.itemsize, x.shape, x.dtype, keep=d_pad)
    outs = U8_ACC if n == 65536 else ALL_OUTS
    pl = sp.SpectralPlan(n, hop, "hann", fmt)
    ra, names_a = launched(lambda: pl.stft(d_al, **outs, vmin=vmin, vmax=vmax))
    ru, names_u = launched(lambda: pl.stft(d_un, **outs, vmin=vmin, vmax=vmax))
    assert ra.n_frames == ru.n_frames == F
    check_oracle(ru, x, n, hop, "hann", fmt, what=f"unaligned N={n} fmt={fmt}")
    get = lambda res, k: _host(getattr(res, k))   # noqa: E731
    if n == 3000:
        assert count(names_a, BLU_PRE) == count(names_u, BLU_PRE) == 1
        for k in ("db_rows", "wf_rows", "spectrum", "maxhold"):
            np.testing.assert_array_equal(get(ru, k), get(ra, k), err_msg=k)
        np.testing.assert_allclose(get(ru, "welch_acc"), get(ra, "welch_acc"), rtol=1e-12)
    elif n == 65536:
        assert count(names_a, K2V2) == 1 and count(names_u, K2V2) == 0, (names_a, names_u)
        assert count(names_u, K2_COLS_DIRECT) == 1 and count(names_u, K2_COLS_BULK) == 0, names_u
        wa, wu = get(ra, "wf_rows"), get(ru, "wf_rows")
        assert np.abs(wu.astype(np.int16) - wa.astype(np.int16)).max() <= 1 and (wu != wa).mean() < 2e-3
        parity.check_power(get(ru, "welch_acc")[0], get(ra, "welch_acc")[0], what="unaligned K2 vs K2v2 welch", rel_tol=1.5e-4)
        parity.check_power(get(ru, "maxhold")[0], get(ra, "maxhold")[0], what="unaligned K2 vs K2v2 maxhold", rel_tol=1.5e-4)
    else:
        assert count(names_a, K1V2) >= 1 and count(names_a, K1_DIRECT) == 0, names_a
        assert count(names_u, K1_DIRECT) >= 1 and count(names_u, K1V2) == 0 and count(names_u, K1_STAGED) == 0, names_u
        X = get(ra, "spectrum")
        assert np.abs(get(ru, "spectrum") - X).max() <= 4e-6 * np.sqrt((np.abs(X) ** 2).mean())
        wa, wu = get(ra, "wf_rows"), get(ru, "wf_rows")
        assert np.abs(wu.astype(np.int16) - wa.astype(np.int16)).max() <= 1
        parity.check_power(get(ru, "welch_acc")[0], get(ra, "welch_acc")[0], what="unaligned K1 vs K1v2 welch", rel_tol=2e-5)
        parity.check_power(get(ru, "maxhold")[0], get(ra, "maxhold")[0], what="unaligned K1 vs K1v2 maxhold", rel_tol=2e-5)
    pl.close()


# ----------------------------------------------------------------------------- Bluestein batches
@pytest.mark.parametrize("F", [65, 129])
def test_bluestein_batches(sp, F):
    """N = 100000 (inner length M = 2^18): 64 frames per batch through the 128 MiB Bluestein buffers, so 65 and 129
    frames end in a one-frame batch.  Device-resident (the host pipeline would cut the run into its own pieces).  The
    frames around every batch boundary against the oracle; the whole run against each batch's frames run alone
    (the same launches: bit-identical rows and max-hold, Welch up to the order of fp64 atomics)."""
    from sdr_iq_visualizer_b200 import _native as nat
    n, hop, fb = 100000, 50000, 64
    x = _iq(n + hop * (F - 1), 0, seed=F)
    pl = sp.SpectralPlan(n, hop, "hann")
    d_in = nat.DeviceArray.from_host(x)
    kw = dict(db_rows=True, wf_rows=True, welch=True, maxhold=True, vmin=-40.0, vmax=90.0)
    r, names = launched(lambda: pl.stft(d_in, **kw))
    assert r.n_frames == F
    assert count(names, BLU_PRE) == -(-F // fb), names
    check_oracle(r, x, n, hop, "hann", 0, sel=_edges(F, fb), what=f"Bluestein F={F}")
    db, wf = r.db_rows.to_host(), r.wf_rows.to_host()
    welch, mh = np.zeros(n), np.zeros(n, np.float32)
    for b0 in range(0, F, fb):
        b1 = min(F, b0 + fb)
        view = nat.DeviceView(d_in.ptr + b0 * hop * 8, (n + hop * (b1 - b0 - 1),), np.complex64, keep=d_in)
        rb = pl.stft(view, **kw)
        pl.sync()
        np.testing.assert_array_equal(db[b0:b1], rb.db_rows.to_host())
        np.testing.assert_array_equal(wf[b0:b1], rb.wf_rows.to_host())
        welch += rb.welch_acc.to_host()[0]
        mh = np.maximum(mh, rb.maxhold.to_host()[0])
    np.testing.assert_allclose(r.welch_acc.to_host()[0], welch, rtol=1e-12)
    np.testing.assert_array_equal(r.maxhold.to_host()[0], mh)
    pl.close()


# ----------------------------------------------------------------------------- host pipeline pieces
def _stft_instances(names):
    return {nm for nm in names if "<" in nm}


@pytest.mark.parametrize("S", [1, 2])
@pytest.mark.parametrize("n,hop,fmt", [(256, 77, 0), (4096, 1024, 1), (4096, 1000, 0), (16384, 5000, 0), (3000, 1500, 0)])
def test_small_host_pieces(sp, monkeypatch, n, hop, fmt, S):
    """The host pipeline with 64 KiB pieces (max(64 KiB, 4 N samples)): pieces ramp up and down, frames straddle piece
    boundaries, each piece's base decides K1v2 against K1 again.  Against the oracle, and against the default-piece run
    (one piece): bit-identical rows where both runs launch one instance of each kernel template, the same set in both
    (every frame then ran the same code); Welch within 1e-6 (fp32 partials regroup with the pieces)."""
    elt = 4 if fmt else 8
    piece = max(65536 // elt, 4 * n)
    L = 12 * piece + 333
    x = _iq(L, fmt, seed=n + hop, S=S)
    vmin, vmax = VRANGE[fmt]
    monkeypatch.setenv("SPX_H2D_PIECE_BYTES", "65536")
    small = sp.SpectralPlan(n, hop, "hann", fmt)
    monkeypatch.delenv("SPX_H2D_PIECE_BYTES")
    ref = sp.SpectralPlan(n, hop, "hann", fmt)
    r, names = launched(lambda: small.stft(x, n_streams=S, **ALL_OUTS, vmin=vmin, vmax=vmax))
    r0, names0 = launched(lambda: ref.stft(x, n_streams=S, **ALL_OUTS, vmin=vmin, vmax=vmax))
    assert r.n_frames == r0.n_frames == sref.frame_count(L, n, hop)
    assert len(names) > len(names0), "64 KiB pieces must split the run into more launches"
    check_oracle(r, x, n, hop, "hann", fmt, S=S, what=f"pieces N={n} hop={hop} S={S}")
    inst, inst0 = _stft_instances(names), _stft_instances(names0)
    if inst == inst0 and len({nm.split("<")[0] for nm in inst}) == len(inst):
        for k in ("db_rows", "wf_rows", "spectrum", "maxhold"):
            np.testing.assert_array_equal(getattr(r, k), getattr(r0, k), err_msg=k)
    else:
        check_oracle(r0, x, n, hop, "hann", fmt, S=S, what=f"default pieces N={n} hop={hop} S={S}")
    np.testing.assert_allclose(r.welch_acc, r0.welch_acc, rtol=1e-6)
    small.close(); ref.close()


# ----------------------------------------------------------------------------- plan scratch across streams
def test_device_call_then_host_call_share_scratch(sp, monkeypatch):
    """A device-resident K2 call enqueued on a caller stream, then at once a host-memory call on the same plan: the host
    call must not overwrite the plan's four-step scratch while the device call's kernels still read it.  Both results
    against the oracle and against each call run alone."""
    from sdr_iq_visualizer_b200 import _native as nat
    monkeypatch.setenv("SPX_BIG_SCRATCH_BYTES", str(1 << 20))     # 4 frames per batch: 75 batches on the caller stream
    n, hop, F1, F2 = 16384, 8192, 300, 40
    x = _iq(n + hop * (F1 - 1), 0, seed=301)
    y = _iq(n + hop * (F2 - 1), 0, seed=302)
    kw = dict(wf_rows=True, welch=True, maxhold=True, vmin=-40.0, vmax=90.0)
    pl = sp.SpectralPlan(n, hop, "hann")
    side = nat.SideStream()
    d_x = nat.DeviceArray.from_host(x)
    outs = dict(wf_rows=nat.DeviceArray((F1, n), np.uint8), welch=nat.DeviceArray((1, n), np.float64),
                maxhold=nat.DeviceArray((1, n), np.float32))

    def both():
        rd = pl.stft(d_x, **{**kw, **outs}, stream=side.handle)
        rh = pl.stft(y, **kw)                                          # no synchronisation in between
        side.sync()
        return rd, rh

    (rd, rh), names = launched(both)
    assert count(names, K2_COLS_BULK) == F1 // 4 + F2 // 4, names
    check_oracle(rd, x, n, hop, "hann", 0, what="device call on a caller stream")
    check_oracle(rh, y, n, hop, "hann", 0, what="host call right after it")
    alone = sp.SpectralPlan(n, hop, "hann")
    ra = alone.stft(d_x, **kw)
    alone.sync()
    np.testing.assert_array_equal(rd.wf_rows.to_host(), ra.wf_rows.to_host())
    np.testing.assert_array_equal(rd.maxhold.to_host(), ra.maxhold.to_host())
    np.testing.assert_allclose(rd.welch_acc.to_host(), ra.welch_acc.to_host(), rtol=1e-12)
    rb = alone.stft(y, **kw)
    np.testing.assert_array_equal(rh.wf_rows, rb.wf_rows)
    np.testing.assert_array_equal(rh.maxhold, rb.maxhold)
    np.testing.assert_allclose(rh.welch_acc, rb.welch_acc, rtol=1e-12)
    side.close(); alone.close(); pl.close()
