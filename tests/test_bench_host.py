"""CPU: host-side pieces of bench.py that need no GPU."""
import importlib.util
import os
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


class _FakeNvml:
    NVML_CLOCK_SM = 0
    nvmlClocksThrottleReasonGpuIdle = 1
    nvmlClocksThrottleReasonSwPowerCap = 4
    nvmlClocksEventReasonSwThermalSlowdown = 32

    def __init__(self, reasons):
        self.calls, self.reasons = 0, reasons

    def nvmlDeviceGetClockInfo(self, h, c):
        self.calls += 1
        return 1965

    def nvmlDeviceGetCurrentClocksThrottleReasons(self, h):
        return self.reasons


def _sampler(b, nv):
    cs = b.ClockSampler.__new__(b.ClockSampler)
    cs.index, cs.samples, cs.reasons, cs._stop, cs.max_mhz, cs.nv, cs.h = 0, [], set(), threading.Event(), 1965, nv, None
    return cs


def test_clock_sampler_takes_few_samples_and_reports_reasons():
    """NVML polling serialises with the CUDA driver (it doubled the measured multi-GPU step): one sample 50 ms into the
    region, then one per second; a region shorter than that still gets one sample."""
    b = _bench()
    nv = _FakeNvml(4)
    cs = _sampler(b, nv)
    with cs:
        time.sleep(0.3)
    assert nv.calls == 1 and cs.summary() == {"sm_mhz": 1965.0, "sm_max_mhz": 1965, "reasons": ["SwPowerCap"]}
    nv2 = _FakeNvml(0)
    cs2 = _sampler(b, nv2)
    with cs2:
        pass
    assert nv2.calls == 1 and cs2.summary()["reasons"] == []


def test_dist_info_reads_torchrun_environment(monkeypatch):
    b = _bench()
    monkeypatch.setenv("RANK", "3"); monkeypatch.setenv("WORLD_SIZE", "8"); monkeypatch.setenv("LOCAL_RANK", "3")
    assert b.dist_info() == (3, 8, 3)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        monkeypatch.delenv(k)
    assert b.dist_info() == (0, 1, 0)


def test_dump_outputs_writes_float_arrays_within_the_limit(tmp_path):
    import numpy as np
    import pytest
    b = _bench()
    pose = np.linspace(0, 1, 14).reshape(2, 7)
    b.dump_outputs(str(tmp_path / "d"), {"pose": pose, "train": np.array([[-1, 999]], np.int32),
                                         "dist": np.array([0.5], np.float32), "big": np.array([2 ** 30], np.int64)})
    got = {n: np.load(tmp_path / "d" / f"{n}.npy") for n in ("pose", "train", "dist", "big")}
    assert got["pose"].dtype == np.float64 and np.array_equal(got["pose"], pose)
    assert got["train"].dtype == np.float32 and got["train"].tolist() == [[-1.0, 999.0]]
    assert got["dist"].dtype == np.float32 and got["big"].dtype == np.float64 and got["big"][0] == 2 ** 30
    with pytest.raises(ValueError):
        b.dump_outputs(str(tmp_path / "e"), {"x": np.zeros(b.DUMP_LIMIT_BYTES // 4 + 1, np.float32)})
    assert not (tmp_path / "e").exists()
