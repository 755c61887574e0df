"""bench.py's clock sampler against a fake NVML (no GPU): samples inside the timed window only, throttle bits decoded,
CUDA_VISIBLE_DEVICES honoured; and the nvidia-smi fallback when NVML is unusable."""
import importlib
import sys
import time
import types


def _fake_nvml(reason_bits=0x4):
    m = types.ModuleType("pynvml")
    m.NVML_CLOCK_SM = 1
    m.seen_index = []
    m.nvmlInit = lambda: None
    m.nvmlDeviceGetHandleByIndex = lambda i: (m.seen_index.append(i), ("h", i))[1]
    m.nvmlDeviceGetMaxClockInfo = lambda h, c: 1965
    m.nvmlDeviceGetClockInfo = lambda h, c: 1900
    m.nvmlDeviceGetCurrentClocksEventReasons = lambda h: reason_bits
    return m


def test_nvml_sampler_window_and_reasons(monkeypatch):
    fake = _fake_nvml()
    monkeypatch.setitem(sys.modules, "pynvml", fake)
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "3,5")
    bench = importlib.import_module("bench")
    s = bench.ClockSampler(1)
    s.start()
    time.sleep(0.03)
    t0 = time.time()
    time.sleep(0.05)
    t1 = time.time()
    time.sleep(0.02)
    out = s.stop(t0, t1)
    assert fake.seen_index == [5]
    assert out["sm_mhz"] == 1900.0 and out["sm_max_mhz"] == 1965.0
    assert out["reasons"] == ["sw_power_cap"]
    assert 5 <= out["samples"] <= 40, out          # ~2 ms period over a 50 ms window, none from outside it
    assert out["samples_in_timed_region"] == out["samples"] and "note" not in out


def test_nvml_sampler_extension_is_reported(monkeypatch):
    """Too few samples inside the timed region: the caller keeps the load up and passes the extended end; the result
    says so and keeps the in-region count separate."""
    monkeypatch.setitem(sys.modules, "pynvml", _fake_nvml(0))
    monkeypatch.delenv("CUDA_VISIBLE_DEVICES", raising=False)
    bench = importlib.import_module("bench")
    s = bench.ClockSampler(0)
    s.start()
    t0 = time.time()
    t1 = t0 + 0.0005                               # a "timed region" shorter than one sampling period
    time.sleep(0.05)
    assert 0 <= s.count(t0, t1) < 3
    t_ext = time.time()
    out = s.stop(t0, t1, t_ext)
    assert out["samples_in_timed_region"] < 3 <= out["samples"] and "note" in out and out["reasons"] == []


def test_sampler_falls_back_when_nvml_is_unusable(monkeypatch, tmp_path):
    broken = types.ModuleType("pynvml")

    def boom():
        raise RuntimeError("no driver")

    broken.nvmlInit = boom
    monkeypatch.setitem(sys.modules, "pynvml", broken)
    monkeypatch.setenv("PATH", str(tmp_path))      # and no nvidia-smi, even on a GPU machine
    bench = importlib.import_module("bench")
    s = bench.ClockSampler(0)
    s.start()                                      # nvidia-smi is absent too: both paths must degrade quietly
    out = s.stop(time.time() - 1, time.time())
    assert out["sm_mhz"] is None and "samples" in out or out["reasons"]
