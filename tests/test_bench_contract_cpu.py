"""bench.py's reference arm and sampler plumbing on a GPU-less box (the driver runs `bench.py --impl reference` and parses one
JSON line; a typo there would only show at round end)."""
import json
import os
import subprocess
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env_extra=None):
    env = dict(os.environ)
    env.update(env_extra or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, env=env,
                          timeout=600)


def test_reference_arm_prints_one_contract_line():
    r = _run(["--impl", "reference", "--encoder", "vits", "--size", "126", "--steps", "1", "--warmup", "0", "--gpus", "1"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "images/sec" and d["unit"] == "images/s" and d["higher_is_better"]
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1 and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    r = _run(["--impl", "reference", "--encoder", "vits", "--size", "126", "--steps", "1", "--warmup", "0", "--gpus", "2"],
             {"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and not [l for l in r.stdout.splitlines() if l.startswith("{")]


def test_product_arm_refuses_to_run_without_a_gpu():
    r = _run(["--steps", "1"], {"CUDA_VISIBLE_DEVICES": ""})   # no visible device, also on a GPU machine
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_steps_below_one_are_refused():
    r = _run(["--impl", "reference", "--encoder", "vits", "--size", "126", "--steps", "0", "--warmup", "0"])
    assert r.returncode != 0 and "--steps" in r.stderr


def test_reference_arm_dumps_the_same_last_step_output_every_run(tmp_path):
    import numpy as np
    got = []
    for run in ("a", "b"):
        r = _run(["--impl", "reference", "--encoder", "vits", "--size", "126", "--steps", "2", "--warmup", "0",
                  "--dump-outputs", str(tmp_path / run)])
        assert r.returncode == 0, r.stderr[-2000:]
        d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])
        assert d["steps"] == 2 and d["dump_outputs"]["file"] == "depth.npy" and not d["dump_outputs"]["sampled"]
        got.append(np.load(tmp_path / run / "depth.npy"))
    assert got[0].dtype == np.float32 and got[0].shape == (1, 1, 126, 126) and np.isfinite(got[0]).all()
    assert np.array_equal(got[0], got[1])


def test_dump_outputs_samples_a_large_output_the_same_way_every_time(tmp_path):
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    out = torch.arange(1000, dtype=torch.float32).view(10, 1, 10, 10)
    info = bench.dump_outputs(torch, out, str(tmp_path / "a.npy"), 400)
    bench.dump_outputs(torch, out, str(tmp_path / "b.npy"), 400)
    a = np.load(tmp_path / "a.npy")
    assert info["sampled"] and info["elements"] == 100 and info["shape"] == [10, 1, 10, 10]
    assert a.dtype == np.float32 and a.nbytes <= 400 and a.shape == (100,)
    assert np.array_equal(a, np.load(tmp_path / "b.npy")) and (np.diff(a) > 0).all()   # distinct elements, index order
    info = bench.dump_outputs(torch, out, str(tmp_path / "c.npy"), 4000)
    assert not info["sampled"] and np.array_equal(np.load(tmp_path / "c.npy"), out.numpy())


def test_nvml_sampler_report_with_a_fake_nvml(monkeypatch):
    """NvmlSampler against a stand-in pynvml: samples inside [mark_begin, mark_end] only, median clock, reasons decoded
    from the bit mask (sw_power_cap kept and named, hw bits named), and a clean 'unavailable' report when NVML is missing."""
    sys.path.insert(0, ROOT)
    import bench
    import time

    fake = types.ModuleType("pynvml")
    fake.NVML_CLOCK_SM = 1
    fake.nvmlClocksThrottleReasonHwSlowdown = 0x8
    fake.nvmlClocksThrottleReasonHwThermalSlowdown = 0x40
    fake.nvmlClocksThrottleReasonSwThermalSlowdown = 0x20
    fake.nvmlClocksThrottleReasonSwPowerCap = 0x4
    fake.nvmlClocksThrottleReasonHwPowerBrakeSlowdown = 0x80
    fake.nvmlClocksThrottleReasonSyncBoost = 0x10
    fake.nvmlInit = lambda: None
    fake.nvmlDeviceGetHandleByUUID = lambda u: "h"
    fake.nvmlDeviceGetMaxClockInfo = lambda h, c: 1965
    fake.nvmlDeviceGetClockInfo = lambda h, c: 1500
    fake.nvmlDeviceGetPowerUsage = lambda h: 990000
    fake.nvmlDeviceGetCurrentClocksEventReasons = lambda h: 0x4
    monkeypatch.setitem(sys.modules, "pynvml", fake)
    s = bench.NvmlSampler("GPU-x")
    s.start()
    assert s.ok
    time.sleep(0.25)
    s.mark_begin()
    time.sleep(0.35)
    s.mark_end()
    rep = s.stop()
    assert rep["sm_mhz"] == 1500.0 and rep["sm_max_mhz"] == 1965.0 and rep["reasons"] == ["sw_power_cap"]
    assert 2 <= rep["samples"] <= 5 and abs(rep["power_w_max"] - 990.0) < 1e-6

    broken = types.ModuleType("pynvml")
    monkeypatch.setitem(sys.modules, "pynvml", broken)   # no nvmlInit -> start() must not raise
    s2 = bench.NvmlSampler("GPU-x")
    s2.start()
    assert not s2.ok and s2.stop()["reasons"] == ["NVML unavailable"]
