"""GPU tests of the multi-job DDC (ddc_jobs_kernel, spx_ddc_exec_jobs / DdcPlan.exec_jobs) and of signal extraction
(sigmf_io.extract_signals): every job's outputs bit for bit against K9 (DdcPlan.exec) on the same span, split calls and
chunked input, untouched columns, NaN reach, parity with the float64 definition, every SPX_E_INVALID case, and a
three-signal recording end to end."""
import json
import os

import numpy as np
import pytest

from oracle import classifier_ref as cref
from tests import ddc_ref as dr
from tests.test_dispatch_paths_gpu import launched

pytestmark = pytest.mark.gpu

FS = 61.44e6
SENTINEL = np.uint32(0x7F8DEAD1)   # a NaN payload no output has


def _mods():
    from sdr_iq_visualizer_b200 import _native as nat, ddc, spectral as sp
    nat.require_device()
    return nat, ddc, sp


def sub_of(T, D):
    """SUB of K9's launch planning (spx_ddc.cu ddc_plan_launch), for choosing n_out around it."""
    low = D & -D
    g = min(low, 32)
    s, c = 32 // g, D // g
    wr = 1
    while wr * 2 <= c and wr * 2 <= 8:
        wr *= 2
    base = 16 * max(s, 8 // wr)

    def smem(sub):
        return ((T + 3) & ~3) * 4 + (sub * D + T - 1) * 8 + wr * sub * 8
    k = 1
    while base * (k + 1) * D <= 16384 and smem(base * (k + 1)) <= 110 << 10:
        k += 1
    return base * k


def signal(L, fmt, seed):
    rng = np.random.default_rng(seed)
    n = np.arange(L)
    x = 0.5 * np.exp(2j * np.pi * 0.11 * n) + 0.05 * (rng.normal(size=L) + 1j * rng.normal(size=L))
    if fmt == "ci16":
        from oracle import spectral_ref as sref
        return sref.to_ci16(x * 0.7), 2.0 ** -15
    return x.astype(np.complex64), 1.0


class Capture:
    """A device-resident capture whose sample 0 has global index `first`, and K9 references on spans of it."""

    def __init__(self, nat, ddc, sp, fmt, L, D, taps, first, seed):
        self.nat, self.ddc, self.sp = nat, ddc, sp
        self.x, self.scale = signal(L, fmt, seed)
        self.fmt = sp.FMT_CI16 if fmt == "ci16" else sp.FMT_CF32
        self.d_x = nat.DeviceArray.from_host(self.x)
        self.L, self.D, self.taps, self.first = L, D, taps, first
        self.plans = {}

    def plan(self, shift):
        if shift not in self.plans:
            self.plans[shift] = self.ddc.DdcPlan(FS, shift, self.D, self.taps, self.fmt, self.scale)
        return self.plans[shift]

    def view(self, a, n):
        """Samples [a, a + n) of the capture (global indices) as a device view."""
        ew = 2 if self.fmt == self.sp.FMT_CI16 else 1
        it = self.x.dtype.itemsize * ew
        return self.nat.DeviceView(self.d_x.ptr + (a - self.first) * it, (n * ew,), self.x.dtype)

    def k9(self, shift, first, m0, n):
        """Outputs m0 .. m0 + n - 1 of DdcPlan.exec on the capture from global sample `first` on."""
        p = self.plan(shift)
        T, D = p.n_taps, self.D
        y = p.exec(self.view(first, (m0 + n - 1) * D + T), first_sample=first)
        p.sync()   # the call ran on the handle's stream, which a plain copy does not wait for
        return y.to_host()[m0:m0 + n]

    def close(self):
        for p in self.plans.values():
            p.close()


SHIFTS = (0.0, FS / 2, 7.3e6, -3.123456789e6, 0.2718281828 * FS)   # phase_inc 0, -2^63, and odd ones


def make_jobs(cap, rng, n_jobs, gap=3):
    """Jobs of every kind: n_out of 1, SUB - 1, SUB, SUB + 1, many sub-tiles, windows ending at the capture's last
    sample, m0 > 0 and n_out = 0; shifts cycle through SHIFTS."""
    T, D = cap.plan(0.0).n_taps, cap.D
    sub = sub_of(T, D)
    top = (cap.L - T) // D + 1
    kinds = [1, sub - 1, sub, sub + 1, 5 * sub + 3, "end", 0, 2, "all"]
    jobs, refs, off = [], [], 0
    for i in range(n_jobs):
        kind = kinds[i % len(kinds)]
        shift = SHIFTS[i % len(SHIFTS)]
        if kind == "end":       # the last window ends at the last sample
            k = int(rng.integers(0, top))
            first = cap.first + cap.L - T - k * D
            avail = k + 1
            m0 = int(rng.integers(0, avail))
            n = avail - m0
        elif kind == "all":
            first, m0, n = cap.first, 0, top
        else:
            first = cap.first + int(rng.integers(0, cap.L - T + 1))
            avail = (cap.first + cap.L - first - T) // D + 1
            n = min(max(kind, 0), avail)
            m0 = int(rng.integers(0, avail - n + 1))
        inc = cap.plan(shift).phase_inc
        jobs.append((first, inc, m0, n, off))
        refs.append((shift, first, m0, n, off))
        off += n + gap
    return jobs, refs, off


def run_jobs(cap, jobs, n_total, x=None, in_first=None):
    nat = cap.nat
    out = nat.DeviceArray.from_host(np.full(2 * n_total, SENTINEL, np.uint32).view(np.complex64))
    p = cap.plan(0.0)
    _, names = launched(lambda: p.exec_jobs(cap.d_x if x is None else x, jobs, out,
                                            in_first_sample=cap.first if in_first is None else in_first))
    assert any("ddc_jobs_kernel" in nm for nm in names), sorted(set(names))
    p.sync()
    return out.to_host()


def check_against_k9(cap, got, refs, n_total):
    written = np.zeros(n_total, bool)
    for shift, first, m0, n, off in refs:
        want = cap.k9(shift, first, m0, n) if n else np.zeros(0, np.complex64)
        assert np.array_equal(got[off:off + n].view(np.uint32), want.view(np.uint32)), (shift, first, m0, n)
        written[off:off + n] = True
    assert (got[~written].view(np.uint32) == SENTINEL).all()   # columns no job writes are untouched


CASES = [(1, "default"), (4, "default"), (64, "default"), (256, "default"), (1, "caller8192"), (1024, "caller33")]


@pytest.mark.parametrize("fmt", ["cf32", "ci16"])
@pytest.mark.parametrize("D,taps", CASES)
def test_jobs_bit_identical_to_k9(fmt, D, taps):
    nat, ddc, sp = _mods()
    rng = np.random.default_rng(D)
    h = None if taps == "default" else rng.normal(size=int(taps[6:])) / np.sqrt(int(taps[6:]))
    T = ddc.design_taps(D).size if h is None else h.size
    cap = Capture(nat, ddc, sp, fmt, T + (6 * sub_of(T, D) + 50) * D + 17, D, h, 1_234_567, D + T)
    jobs, refs, n_total = make_jobs(cap, rng, 18)
    check_against_k9(cap, run_jobs(cap, jobs, n_total), refs, n_total)
    cap.close()


def test_thousand_jobs_and_one_job():
    nat, ddc, sp = _mods()
    rng = np.random.default_rng(1000)
    cap = Capture(nat, ddc, sp, "ci16", 400_000, 4, None, 77, 3)
    jobs, refs, n_total = make_jobs(cap, rng, 1000)
    check_against_k9(cap, run_jobs(cap, jobs, n_total), refs, n_total)
    one = [j for j, r in zip(jobs, refs) if r[3] > 1][:1]
    got = run_jobs(cap, one, one[0][3] + one[0][4] + 5)
    r = [r for r in refs if r[3] > 1][0]
    check_against_k9(cap, got, [r], one[0][3] + one[0][4] + 5)
    cap.close()


@pytest.mark.parametrize("fmt", ["cf32", "ci16"])
def test_split_calls_and_chunks_give_one_call(fmt):
    """m0 sub-ranges in separate calls, and the capture cut into overlapping device chunks, give one call's bits."""
    nat, ddc, sp = _mods()
    D = 64
    rng = np.random.default_rng(5)
    cap = Capture(nat, ddc, sp, fmt, 600_000, D, None, 10_000, 8)
    T = cap.plan(0.0).n_taps
    jobs, refs, n_total = make_jobs(cap, rng, 9)
    whole = run_jobs(cap, jobs, n_total)
    # the same jobs in three calls over m0 sub-ranges
    out = nat.DeviceArray.from_host(np.full(2 * n_total, SENTINEL, np.uint32).view(np.complex64))
    p = cap.plan(0.0)
    for part in range(3):
        sub = []
        for first, inc, m0, n, off in jobs:
            a, b = m0 + n * part // 3, m0 + n * (part + 1) // 3
            sub.append((first, inc, a, b - a, off + a - m0))
        p.exec_jobs(cap.d_x, sub, out, in_first_sample=cap.first)
    p.sync()
    assert np.array_equal(out.to_host().view(np.uint32), whole.view(np.uint32))
    # chunks of the capture overlapping by T - 1, each call given only the outputs whose windows it holds
    from sdr_iq_visualizer_b200 import sigmf_io as sio
    spans = [(first - cap.first, m0 + n, D, T) for first, _, m0, n, _ in jobs]
    out = nat.DeviceArray.from_host(np.full(2 * n_total, SENTINEL, np.uint32).view(np.complex64))
    for c0, c1, parts in sio.extract_schedule(spans, cap.L, 50_000):
        sub = []
        for j, a, n in parts:
            first, inc, m0, n_j, off = jobs[j]
            lo, hi = max(a, m0), min(a + n, m0 + n_j)
            if hi > lo:
                sub.append((first, inc, lo, hi - lo, off + lo - m0))
        p.exec_jobs(cap.view(cap.first + c0, c1 - c0), sub, out, in_first_sample=cap.first + c0)
    p.sync()
    assert np.array_equal(out.to_host().view(np.uint32), whole.view(np.uint32))
    cap.close()


def test_nan_reaches_only_covering_windows():
    nat, ddc, sp = _mods()
    D = 8
    cap = Capture(nat, ddc, sp, "cf32", 200_000, D, None, 0, 4)
    T = cap.plan(0.0).n_taps
    bad = 100_000
    cap.x[bad] = np.nan
    cap.d_x = nat.DeviceArray.from_host(cap.x)
    jobs = [(bad - 5000, cap.plan(7.3e6).phase_inc, 0, 1000, 0),       # its span holds the NaN
            (bad + 1, cap.plan(7.3e6).phase_inc, 0, 1000, 1000),       # starts right after it
            (bad - T - 1000 * D, cap.plan(0.0).phase_inc, 0, 1001, 2000)]  # its last window ends right before it
    got = run_jobs(cap, jobs, 3001)
    m = np.arange(1000)
    first = bad - 5000
    covers = (first + m * D <= bad) & (bad < first + m * D + T)
    assert covers.any()
    np.testing.assert_array_equal(np.isnan(got[:1000].real), covers)
    np.testing.assert_array_equal(np.isnan(got[:1000].imag), covers)
    assert not np.isnan(got[1000:3001].view(np.float32)).any()
    cap.close()


@pytest.mark.parametrize("fmt", ["cf32", "ci16"])
def test_parity_with_float64_definition(fmt):
    nat, ddc, sp = _mods()
    D = 16
    cap = Capture(nat, ddc, sp, fmt, 300_000, D, None, 999, 6)
    T = cap.plan(0.0).n_taps
    jobs, refs = [], []
    for i, (shift, a, n) in enumerate([(7.3e6, 0, 2000), (-20e6, 50_001, 700), (FS / 2, 299_999 - T - 99 * D, 100)]):
        jobs.append((cap.first + a, cap.plan(shift).phase_inc, 0, n, 3000 * i))
    got = run_jobs(cap, jobs, 9000)
    ew = 2 if fmt == "ci16" else 1
    h = cap.plan(0.0).taps
    for first, inc, _, n, off in jobs:
        a = first - cap.first
        seg = cap.x[ew * a: ew * (a + (n - 1) * D + T)]
        want = dr.ddc(seg, h, D, inc, first, cap.scale)
        err = np.abs(got[off:off + n].astype(np.complex128) - want).max()
        assert want.size == n and err <= 1e-5 * dr.bound(h, cap.x, cap.scale), err
    cap.close()


def test_errors_launch_nothing_and_leave_the_handle_usable():
    nat, ddc, sp = _mods()
    lib = nat.lib()
    D = 4
    cap = Capture(nat, ddc, sp, "cf32", 10_000, D, None, 100, 2)
    p = cap.plan(1e6)
    T = p.n_taps
    good = (150, p.phase_inc, 2, 50, 3)
    want = cap.k9(1e6, 150, 2, 50)
    out = nat.DeviceArray.from_host(np.full(2 * 60, SENTINEL, np.uint32).view(np.complex64))

    def call(jobs, in_ptr=None, n=cap.L, in_first=cap.first, out_ptr=None, n_jobs=None, handle=None):
        arr = ddc.as_jobs(jobs) if jobs is not None else None
        ptr = arr.ctypes.data if arr is not None and len(arr) else None
        return lib.spx_ddc_exec_jobs(p._h if handle is None else handle, cap.d_x.ptr if in_ptr is None else in_ptr, n,
                                     in_first, ptr, len(arr) if n_jobs is None else n_jobs,
                                     out.ptr if out_ptr is None else out_ptr, None)

    def still_good():
        out.copy_from_host(np.full(2 * 60, SENTINEL, np.uint32).view(np.complex64))
        assert call([good]) == nat.OK
        p.sync()
        got = out.to_host()
        assert np.array_equal(got[3:53].view(np.uint32), want.view(np.uint32))
        assert (got[:3].view(np.uint32) == SENTINEL).all() and (got[53:].view(np.uint32) == SENTINEL).all()

    f, inc, m0, n, o = good
    last_ok = (cap.first + cap.L - T - (m0 + n - 1) * D, inc, m0, n, o)     # window ends at the last sample
    assert call([last_ok]) == nat.OK
    bad = [dict(jobs=[(f, inc, m0, n, -1)]), dict(jobs=[(f, inc, -1, n, o)]), dict(jobs=[(f, inc, m0, -1, o)]),
           dict(jobs=[(-1, inc, m0, n, o)]),
           dict(jobs=[(cap.first - 1, inc, 0, n, o)]),                                # first window starts before in
           dict(jobs=[(last_ok[0] + 1, inc, m0, n, o)]),                              # last window ends after in
           dict(jobs=[good], n=-1), dict(jobs=[good], in_first=-1), dict(jobs=[good], n_jobs=-1),
           dict(jobs=[], n_jobs=1),                                                   # jobs NULL with n_jobs > 0
           dict(jobs=[good], in_ptr=0), dict(jobs=[good], out_ptr=0), dict(jobs=[good], in_ptr=cap.d_x.ptr + 2),
           dict(jobs=[good], out_ptr=out.ptr + 2), dict(jobs=[good, (f, inc, m0, n, -5)]),
           dict(jobs=[(f, inc, m0, 1 << 62, o)])]
    for kw in bad:
        assert call(**kw) == nat.E_INVALID, kw
        still_good()
    assert lib.spx_ddc_exec_jobs(None, cap.d_x.ptr, cap.L, cap.first, None, 0, out.ptr, None) == nat.E_INVALID
    # nothing to do: OK and nothing launched, even with NULL pointers
    assert call([(f, inc, m0, 0, o)], in_ptr=0, out_ptr=0) == nat.OK
    assert call([], n_jobs=0, in_ptr=0, out_ptr=0) == nat.OK
    with pytest.raises(ValueError):
        p.exec_jobs(cap.d_x, [(f, inc, m0, n, 20)], nat.DeviceArray((60,), np.complex64), in_first_sample=cap.first)
    with pytest.raises(TypeError):
        p.exec_jobs(cap.x, [good], out, in_first_sample=cap.first)
    still_good()
    cap.close()


# ----------------------------------------------------------------------------- a recording end to end
@pytest.mark.parametrize("datatype", ["cf32_le", "ci16_le"])
def test_extract_signals_end_to_end(tmp_path, datatype):
    from sdr_iq_visualizer_b200 import classifier as cls_mod, sigmf_io as sio, spectral as sp
    from tests.test_detect_gpu import B, FC, NFFT, synth_recording
    from tests.test_detect_gpu import FS as FS_R
    x, truth = synth_recording(17)
    base = sio.write_recording(str(tmp_path / "three"), x, FS_R, FC, datatype)
    data_before = open(base + ".sigmf-data", "rb").read()
    _, ann = sio.detect_signals(base, nfft=NFFT, overview=(512, 1024 // B))
    assert len(ann) == 3
    rec = sio.fromfile(base)
    plans = sio.signal_jobs(ann, FS_R, FC, rec.n_samples)
    out_dir = str(tmp_path / "sigs")
    nfft = 256
    sigs, names = launched(lambda: sio.extract_signals(base, ann, nfft=nfft, out_dir=out_dir, label_parent=True,
                                                       max_chunk_samples=1 << 20))
    assert any("ddc_jobs_kernel" in nm for nm in names)
    assert len(sigs) == 3
    for k, (s, a, (shift, inc, D, first, n)) in enumerate(zip(sigs, ann, plans)):
        assert s.annotation == a and s.decim == D and s.first_sample == first and s.iq.shape == (n,) and n > nfft
        assert s.sample_rate == FS_R / D and s.center_freq == FC + shift and s.n_taps == len(sio_taps(D))
        # the outputs cover the annotated span: output m belongs to time first + m D + (T - 1) / 2
        h = (s.n_taps - 1) // 2
        assert first + h == a["core:sample_start"]
        assert first + (n - 1) * D + h >= a["core:sample_start"] + a["core:sample_count"] - D
        # files read back as the returned IQ, with the stated meta
        r = sio.fromfile(os.path.join(out_dir, f"three.sig{k}"))
        assert np.array_equal(r.read_samples().view(np.uint32), s.iq.view(np.uint32))
        assert r.sample_rate == s.sample_rate and r.center_freq == s.center_freq
        assert r.get_global_field("core:sample_rate") == (int(s.sample_rate) if s.sample_rate.is_integer() else s.sample_rate)
        assert "three" in r.get_global_field("core:description")
        assert r.get_annotations()[0]["core:label"] == s.label and r.get_annotations()[0]["core:sample_count"] == n
        # measurements: the oracle on the returned spectrum's centre half
        lo, hi = nfft // 4, nfft - nfft // 4
        pdb = 10.0 * np.log10(s.pxx[lo:hi])
        fj = s.center_freq + sp.freq_axis(nfft, s.sample_rate, 0.0)[lo:hi]
        w = cref.features(fj, pdb)
        m = s.measurements
        for key in ("n", "argmax", "min_distance_bins", "n_candidates", "peak_count"):
            assert m[key] == w[key], key
        for key in ("noise_floor_db", "peak_db", "snr_db", "adaptive_thr"):
            assert m[key] == w[key], key
        assert m["peaks"] == w["peaks"]
        assert (m["first_3db"], m["last_3db"]) == w["edges"][3] and (m["first_20db"], m["last_20db"]) == w["edges"][20]
        assert abs(m["flatness"] - w["flatness"]) <= 1e-11 and abs(m["kurtosis"] - w["kurtosis"]) <= 1e-11
        assert s.label == cls_mod.classify_from_measurements(fj, w, hi - lo, smooth=False)["label"]
    # the CW tone: its baseband peak at 298 kHz - the shift, within a bin
    tone = min(sigs, key=lambda s: abs(s.center_freq - (FC + 298e3)))
    f = sp.freq_axis(nfft, tone.sample_rate, 0.0)
    assert abs(f[int(np.argmax(tone.pxx))] - (FC + 298e3 - tone.center_freq)) <= tone.sample_rate / nfft
    # the parent: relabelled annotations, the data file untouched
    assert open(base + ".sigmf-data", "rb").read() == data_before
    got = sio.fromfile(base).get_annotations()
    assert [g["core:label"] for g in got] == [s.label for s in sigs]
    assert [{k: v for k, v in g.items() if k != "core:label"} for g in got] == \
        [{k: v for k, v in a.items() if k != "core:label"} for a in ann]
    print("labels", datatype, [(round(s.center_freq - FC), s.decim, s.label) for s in sigs])


def sio_taps(D):
    from sdr_iq_visualizer_b200 import ddc
    return ddc.design_taps(D)


def test_extract_signals_detects_by_default_and_reports_empty_regions(tmp_path):
    from sdr_iq_visualizer_b200 import sigmf_io as sio
    from tests.test_detect_gpu import FC, synth_recording
    from tests.test_detect_gpu import FS as FS_R
    x, _ = synth_recording(17)
    base = sio.write_recording(str(tmp_path / "three"), x[: 1 << 21], FS_R, FC)
    _, ann = sio.detect_signals(base)
    sigs = sio.extract_signals(base)
    assert [s.annotation for s in sigs] == ann
    empty = dict(ann[0]) if ann else {"core:freq_lower_edge": FC, "core:freq_upper_edge": FC + 10.0}
    empty.update({"core:sample_start": 10, "core:sample_count": 5})
    s = sio.extract_signals(base, [empty], out_dir=str(tmp_path / "e"))
    assert s[0].iq.shape == (0,) and s[0].pxx is None and s[0].label is None
    meta = json.load(open(str(tmp_path / "e" / "three.sig0.sigmf-meta")))
    assert "core:label" not in meta["annotations"][0]
