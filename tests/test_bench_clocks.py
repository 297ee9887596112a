"""CPU: bench.py's clock sampler.  A timed region of the bench is a few hundred ms, so the sampler runs from
before the warm-up and keeps only the samples stamped inside the timed windows; these tests pin that windowing,
the throttle-reason decoding, and the nvidia-smi child path (a stand-in `nvidia-smi` script on PATH, NVML kept out)."""
import os
import stat
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _sampler():
    import bench
    return bench.ClockSampler(0, None)


def test_nvml_samples_are_windowed_and_reasons_decoded():
    c = _sampler()
    c.max_mhz = 1965
    c.windows = [[1.0, 2.0], [3.0, 4.0]]
    rows = [(0.5, 300, 0x8),            # before the first window: an idle clock and a slowdown that must not count
            (1.5, 1950, 0x4), (1.6, 1960, 0), (2.5, 210, 0x40), (3.5, 1965, 0)]
    out = c.summary(rows, [])
    assert out["samples"] == 3 and out["sm_mhz"] == 1960 and out["sm_max_mhz"] == 1965
    assert out["reasons"] == ["sw_power_cap"] and out["window"] == "timed regions"
    assert out["source"].startswith("nvml")


def test_thermal_and_hw_slowdown_bits():
    c = _sampler()
    c.windows = [[0.0, 10.0]]
    out = c.summary([(1.0, 1000, 0x8 | 0x20 | 0x40)], [])
    assert out["reasons"] == ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"]


def test_smi_fallback_and_warmup_fallback():
    c = _sampler()
    c.windows = [[1.0, 2.0]]
    smi = [(0.5, 1000, 1965, []), (1.5, 1900, 1965, ["sw_power_cap"])]
    out = c.summary([], smi)
    assert out["samples"] == 1 and out["sm_mhz"] == 1900 and out["reasons"] == ["sw_power_cap"]
    # nothing inside the window: warm-up samples are used and the line says so; later samples are not
    out = c.summary([], [(0.5, 1000, 1965, []), (0.7, 1900, 1965, []), (9.0, 100, 1965, ["hw_slowdown"])])
    assert out["window"] == "warm-up + timed regions" and out["samples"] == 2 and out["reasons"] == []


def test_no_source_reports_unavailable():
    c = _sampler()
    c.windows = [[1.0, 2.0]]
    out = c.summary([], [])
    assert out == {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"], "samples": 0}


def test_nvidia_smi_child_path(tmp_path, monkeypatch):
    fake = tmp_path / "nvidia-smi"
    fake.write_text("#!/bin/sh\nwhile true; do echo '1965, 1965, Not Active, Not Active, Not Active, Active'; sleep 0.02; done\n")
    fake.chmod(fake.stat().st_mode | stat.S_IEXEC)
    monkeypatch.setenv("PATH", f"{tmp_path}:{os.environ['PATH']}")
    c = _sampler()

    def no_nvml():
        raise RuntimeError("NVML unavailable")
    monkeypatch.setattr(c, "_nvml_open", no_nvml)   # where a GPU is, NVML would win over the child this test is about
    c.start()
    time.sleep(0.15)                    # "warm-up"
    c.begin()
    time.sleep(0.25)
    c.end()
    out = c.stop()
    assert out["samples"] >= 3 and out["sm_mhz"] == 1965 and out["sm_max_mhz"] == 1965
    assert out["reasons"] == ["sw_power_cap"] and out["window"] == "timed regions"
