"""bench.py's host-side pieces that need no GPU: the clock sampler (NVML in-process, nvidia-smi per sample as the fallback), the
workload descriptions of the four BASELINE configs, the peak lookup."""
import importlib
import json
import os
import stat
import sys
import time
import types

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture()
def bench(monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py"])
    sys.path.insert(0, ROOT)
    mod = importlib.import_module("bench")
    return importlib.reload(mod)


def _fake_nvml(reason_mask=0x4, fail_init=False):
    m = types.ModuleType("pynvml")
    m.NVML_CLOCK_SM = 1

    def init():
        if fail_init:
            raise RuntimeError("no driver")
    m.nvmlInit = init
    m.nvmlShutdown = lambda: None

    def by_uuid(u):
        raise RuntimeError("unknown uuid")
    m.nvmlDeviceGetHandleByUUID = by_uuid
    m.nvmlDeviceGetHandleByIndex = lambda i: ("handle", i)
    m.nvmlDeviceGetMaxClockInfo = lambda h, c: 1965
    m.nvmlDeviceGetClockInfo = lambda h, c: 1950
    m.nvmlDeviceGetCurrentClocksEventReasons = lambda h: reason_mask
    return m


def test_clock_sampler_reads_nvml_in_process(bench, monkeypatch):
    monkeypatch.setitem(sys.modules, "pynvml", _fake_nvml(reason_mask=0x4 | 0x40))
    cs = bench.ClockSampler(0, "not-a-real-uuid")     # unknown uuid: falls back to the index
    cs.start()
    time.sleep(0.35)
    out = cs.summary()
    assert out["source"] == "nvml" and out["samples"] >= 3
    assert out["sm_mhz"] == 1950 and out["sm_max_mhz"] == 1965
    assert out["reasons"] == ["hw_thermal_slowdown", "sw_power_cap"]


def test_clock_sampler_falls_back_to_nvidia_smi(bench, monkeypatch, tmp_path):
    monkeypatch.setitem(sys.modules, "pynvml", _fake_nvml(fail_init=True))
    smi = tmp_path / "nvidia-smi"
    smi.write_text("#!/bin/bash\necho '1965, 1965, 412.5, Not Active, Not Active, Not Active, Active'\n")
    smi.chmod(smi.stat().st_mode | stat.S_IEXEC)
    monkeypatch.setenv("PATH", str(tmp_path) + os.pathsep + os.environ["PATH"])
    cs = bench.ClockSampler(0)
    cs.start()
    time.sleep(0.5)
    out = cs.summary()
    assert out["source"] == "nvidia-smi" and out["samples"] >= 1
    assert out["sm_mhz"] == 1965 and out["reasons"] == ["sw_power_cap"]


def test_workload_descriptions_cover_the_baseline_configs(bench):
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert sorted(bench.CONFIGS) == ["c2", "c3", "c4", "c5"] and len(base["configs"]) == 5   # configs[0] is the CPU-only n = 10 case
    for name, c in bench.CONFIGS.items():
        w = bench.workload_config(name)
        assert w["n"] == c["n"] and w["m"] == c["m"] and w["line_search"] == c["ls"] and "BASELINE.json configs[" in w["workload"]
    assert bench.CONFIGS["c2"]["n"] == 10_000_000 and bench.CONFIGS["c2"]["m"] == 10 and bench.CONFIGS["c2"]["ls"] == "MoreThuente"
    assert bench.CONFIGS["c3"]["m"] == 20 and bench.CONFIGS["c3"]["ls"] == "Bracketing"
    assert bench.workload_config("c5")["batch"] == 64


def test_peak_lookup(bench):
    peak, src = bench.load_peaks()
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        assert peak == float(json.load(open(path))["hbm_gbs"]) and src.startswith("measured")
    else:
        assert peak == 6650.0 and src.startswith("fallback")


def test_dump_outputs_writes_float64_and_a_fixed_sample(bench, tmp_path):
    import numpy as np
    x = np.arange(bench.DUMP_SAMPLE + 1000, dtype=np.float64)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"x": x, "fx": 1.5, "niter": [22, 23]})
    a = np.load(tmp_path / "a" / "x.npy")
    assert a.dtype == np.float64 and a.size == bench.DUMP_SAMPLE and np.all(np.diff(a) > 0)   # distinct entries of x, in order
    assert np.array_equal(a, np.load(tmp_path / "b" / "x.npy"))
    assert np.load(tmp_path / "a" / "fx.npy") == 1.5 and np.load(tmp_path / "a" / "niter.npy").tolist() == [22.0, 23.0]
    small = np.arange(10.0)
    bench.dump_outputs(str(tmp_path / "c"), {"x": small})
    assert np.array_equal(np.load(tmp_path / "c" / "x.npy"), small)


def test_parse_args_steps_and_dump_outputs(bench):
    assert bench.parse_args(["--steps", "7"]).steps == 7
    assert bench.parse_args(["--dump-outputs", "out"]).dump_outputs == "out"
    with pytest.raises(SystemExit):
        bench.parse_args(["--steps", "0"])


def test_cpu_leg_builds_its_checker_outside_the_tree(bench):
    """The timing build of the checker goes to a temporary directory: bench.py writes nothing into the tree."""
    before = sorted(os.listdir(os.path.join(ROOT, "oracle")))
    po, orc = bench.load_oracle()
    assert not orc.path.startswith(ROOT + os.sep) and not os.path.exists(orc.path)
    assert sorted(os.listdir(os.path.join(ROOT, "oracle"))) == before
    assert orc.lbfgs(po.OBJ_ROSENBROCK_PAIRED, [0.0] * 10, po.LS_MORE_THUENTE, orc.default_param())["niter"] == 21
