"""CPU tests of the drop-in boundary: the streamer surface of `app.sdr.streamer` behaves like the
reference's, the C ABI exports every symbol include/spx.h declares, and the product fails
loudly without a GPU (no CPU fallback)."""
import hashlib
import os
import re
import sys
from unittest.mock import MagicMock

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFERENCE_TEST_CLASSIFIER_SHA256 = "81b5422a44e9c1b337f15d66b1cca256576cb665007569d4318e57a9e3123678"


def test_abi_exports_every_declared_symbol():
    from sdr_iq_visualizer_b200 import _native as nat
    hdr = open(os.path.join(ROOT, "include", "spx.h")).read()
    declared = set(re.findall(r"SPX_API\s+[\w\s\*]+?\b(spx_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 25
    lib = nat.lib()
    for name in declared:
        assert hasattr(lib, name), f"libspx.so does not export {name}"
    assert declared == set(nat._SIGNATURES), declared ^ set(nat._SIGNATURES)
    assert lib.spx_abi_version() == 3
    assert lib.spx_frame_count(61_440_000, 4096, 1024) == 59_997


def test_no_cpu_fallback_without_gpu():
    from sdr_iq_visualizer_b200 import _native as nat
    if nat.device_count() > 0:
        pytest.skip("a GPU is present")
    from sdr_iq_visualizer_b200 import classifier, spectral, timedomain
    with pytest.raises(nat.SpectralError):
        spectral.SpectralPlan(1024)
    with pytest.raises(nat.SpectralError):
        spectral.stream_frame(np.zeros(64, complex), 1e6, 0.0)
    with pytest.raises(nat.SpectralError):
        classifier.classify_signal_advanced(np.arange(8.0), np.zeros(8))
    with pytest.raises(nat.SpectralError):
        timedomain.iq_hist2d(np.zeros(8, np.complex64), 1.0)
    # empty input never reaches the device and answers like the reference (classifier.py:16-17,41-42)
    assert classifier.classify_signal_simple(np.array([]), np.array([])) == "No Data"
    assert classifier.classify_signal_advanced(np.array([]), np.array([]))["label"] == "No Data"


def test_plan_create_accepts_only_the_documented_variants():
    """spx_plan_config.variant is 0, 1, 12 or 22 for every nfft; any other value is refused with SPX_E_INVALID before a
    device is looked for, so the check holds with or without a GPU."""
    import ctypes as C
    from sdr_iq_visualizer_b200 import _native as nat
    has_gpu = nat.device_count() > 0
    for nfft in (256, 1000, 4096, 65536):
        for variant in (0, 1, 12, 22, -1, 2, 5, 11, 20, 21, 23):
            cfg = nat.spx_plan_config(C.sizeof(nat.spx_plan_config), 0, nfft, nfft // 4, nat.WINDOW_HANN, nat.FMT_CI16,
                                      1.0, 1e-12, variant, 0)
            h = C.c_void_p()
            rc = nat.lib().spx_plan_create(C.byref(h), C.byref(cfg))
            if variant in (0, 1, 12, 22):
                assert rc == (nat.OK if has_gpu else nat.E_NODEVICE), (nfft, variant, nat.last_error())
                if h.value:
                    nat.check(nat.lib().spx_plan_destroy(h))
            else:
                assert rc == nat.E_INVALID and h.value is None, (nfft, variant)
                assert f"unknown variant {variant}: accepted values are 0, 1, 12 and 22" in nat.last_error()


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "sdr_iq_visualizer_b200")
    for base in (pkg, os.path.join(ROOT, "app")):
        for dirpath, _, files in os.walk(base):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h")):
                    text = open(os.path.join(dirpath, f)).read()
                    assert "oracle" not in text.replace("oracle's", ""), f"{f} mentions the oracle"


def test_streamer_drop_in_surface():
    sys.modules.setdefault("adi", MagicMock())
    from app.sdr.streamer import SDRDataStreamer, sdr_streamer
    s = SDRDataStreamer()
    assert (s.uri, s.sample_rate, s.center_freq, s.rx_lo, s.rx_rf_bandwidth, s.rx_buffer_size) == \
        ("ip:192.168.2.1", 1_000_000, 2_400_000_000, 2_400_000_000, 4_000_000, 4096)
    assert s.sdr is None and s.running is False and s.thread is None and s.connected is False
    assert isinstance(sdr_streamer, SDRDataStreamer)
    for i in range(130):                       # drop-oldest bounded queue
        s._push({"i": i})
    assert s.data_queue.qsize() == 100
    # reference semantics (streamer.py:196-200): one frame per call, oldest first; the newest only on request
    assert s.get_latest_data() == {"i": 30} and s.get_latest_data() == {"i": 31}
    assert s.get_newest_data() == {"i": 129} and s.get_latest_data() is None
    st = s.get_status()
    assert {"connected", "running", "queue_size", "last_success_age_ms", "total_frames"} <= set(st)


def test_streamer_compute_error_is_not_a_radio_fault(monkeypatch):
    """SpectralError inside the loop must not count toward the reconnect logic (SURVEY.md section 5)."""
    sys.modules.setdefault("adi", MagicMock())
    from sdr_iq_visualizer_b200 import streamer as st
    s = st.SDRDataStreamer()
    calls = {"n": 0}

    class Radio:
        def rx(self_inner):
            calls["n"] += 1
            if calls["n"] >= 5:
                s.running = False
            return np.zeros(64, complex)

    def boom(*a, **k):
        raise st.SpectralError(-2, "injected")

    monkeypatch.setattr(st.spectral, "stream_frame", boom)
    monkeypatch.setattr(s, "_attempt_reconnect", lambda *a, **k: pytest.fail("reconnect attempted"))
    s.sdr, s.connected, s.running = Radio(), True, True
    s._stream_data()
    assert s.compute_errors == 5 and s.total_frames == 0 and s.connected is True
    assert s.get_status()["compute_state"] == "degraded" and "injected" in s.get_status()["compute_last_error"]


def test_streamer_any_processing_exception_is_a_compute_fault_and_stops_after_limit(monkeypatch):
    """A ValueError out of process_buffer is not a radio fault either; the stream stops after COMPUTE_FAULT_LIMIT
    consecutive compute failures instead of spinning, and says so in get_status()."""
    sys.modules.setdefault("adi", MagicMock())
    from sdr_iq_visualizer_b200 import streamer as st
    s = st.SDRDataStreamer()
    s.COMPUTE_FAULT_LIMIT = 4
    monkeypatch.setattr(st.time, "sleep", lambda *_: None)

    class Radio:
        def rx(self_inner):
            return np.zeros(64, complex)

    monkeypatch.setattr(s, "process_buffer", lambda *_: (_ for _ in ()).throw(ValueError("bad shape")))
    monkeypatch.setattr(s, "_attempt_reconnect", lambda *a, **k: pytest.fail("reconnect attempted"))
    s.sdr, s.connected, s.running = Radio(), True, True
    s._stream_data()
    st_ = s.get_status()
    assert s.running is False and s.connected is True
    assert st_["compute_state"] == "failed" and st_["compute_errors"] == 4 and "ValueError" in st_["compute_last_error"]


def test_two_consumers_share_the_queue_like_the_reference():
    """Dashboard tick (callbacks.py:104) and chatbot tool (chatbot.py:149) both call get_latest_data(): each call
    consumes one frame, so a second consumer still finds data after the first one ran."""
    sys.modules.setdefault("adi", MagicMock())
    from app.sdr.streamer import SDRDataStreamer
    s = SDRDataStreamer()
    for i in range(3):
        s._push({"i": i})
    assert s.get_latest_data() == {"i": 0}      # dashboard
    assert s.get_latest_data() == {"i": 1}      # chatbot right after it: not starved
    assert s.peek_latest() == {"i": 2} and s.data_queue.qsize() == 1


def test_vendored_reference_test_is_verbatim():
    """tests/golden/reference_test_classifier.py is the reference's tests/test_classifier.py byte for byte: the digest
    is the reference file's SHA-256."""
    here = os.path.join(os.path.dirname(__file__), "golden", "reference_test_classifier.py")
    with open(here, "rb") as fh:
        assert hashlib.sha256(fh.read()).hexdigest() == REFERENCE_TEST_CLASSIFIER_SHA256


def test_failed_library_load_is_cached(monkeypatch, tmp_path):
    """A missing / unbuildable libspx.so raises at once on every later call instead of re-running make per call."""
    from sdr_iq_visualizer_b200 import _native as nat
    calls = {"n": 0}

    def failing_build(*a, **k):
        calls["n"] += 1
        raise nat.SpectralError(nat.E_UNSUPPORTED, "injected build failure")

    monkeypatch.setattr(nat, "_lib", None)
    monkeypatch.setattr(nat, "_lib_error", None)
    monkeypatch.setattr(nat, "LIB_PATH", str(tmp_path / "absent.so"))
    monkeypatch.setattr(nat, "build", failing_build)
    for _ in range(3):
        with pytest.raises(nat.SpectralError):
            nat.lib()
    assert calls["n"] == 1
    nat.reset_load_failure()
    with pytest.raises(nat.SpectralError):
        nat.lib()
    assert calls["n"] == 2


def test_output_buffers_are_validated():
    """Caller-supplied outputs of the wrong size / dtype are refused before libspx writes through them."""
    from sdr_iq_visualizer_b200 import spectral
    spectral._check_buffer(np.empty((3, 8), np.float32), (3, 8), np.float32, "db_rows")
    with pytest.raises(ValueError):
        spectral._check_buffer(np.empty((3, 8), np.float64), (3, 8), np.float32, "db_rows")
    with pytest.raises(ValueError):
        spectral._check_buffer(np.empty((2, 8), np.float32), (3, 8), np.float32, "db_rows")
    import torch
    spectral._check_buffer(torch.empty((3, 8), dtype=torch.uint8), (3, 8), np.uint8, "wf_rows")
    with pytest.raises(ValueError):
        spectral._check_buffer(torch.empty((3, 8), dtype=torch.float64), (3, 8), np.float32, "maxhold")
