"""bench.py host-side pieces that can be checked without a GPU: the clock sampler
(against a fake `nvidia-smi`), the reference arm's one-line contract, the output dump and
the argument checks."""
import json
import os
import stat
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FAKE = """#!/bin/bash
sleep 0.05
i=0
while true; do
  if [ $i -ge 12 ] && [ $i -le 14 ]; then
    echo "0, 1500, 1965, 990.0, 0x4, Not Active, Not Active, Not Active, Active"
  else
    echo "0, $((1900 + i)), 1965, 600.0, 0x0, Not Active, Not Active, Not Active, Not Active"
  fi
  i=$((i+1)); sleep 0.02
done
"""


def test_clock_sampler_windows(tmp_path, monkeypatch):
    import bench
    fake = tmp_path / "nvidia-smi"
    fake.write_text(FAKE)
    fake.chmod(fake.stat().st_mode | stat.S_IEXEC)
    monkeypatch.setenv("PATH", str(tmp_path) + os.pathsep + os.environ["PATH"])
    s = bench.ClockSampler(0, period_ms=20)
    s.start()
    time.sleep(0.22)                                   # warm-up: process already streaming
    t0 = time.time()
    time.sleep(0.30)                                   # the "timed region"
    t1 = time.time()
    time.sleep(0.05)
    r = s.stop(t0, t1)
    assert r["window"] == "timed region" and 8 <= r["samples"] < r["samples_total"]
    assert r["sm_max_mhz"] == 1965.0 and 1500 <= r["sm_mhz"] <= 1965 and r["period_ms"] == 20
    assert r["reasons"] == ["sw_power_cap"] and r["power_w_max"] == 990.0
    # a timed region shorter than the sampling period: nearest samples under the same load
    s = bench.ClockSampler(0)
    s.start()
    time.sleep(0.2)
    t0 = time.time()
    r = s.stop(t0, t0 + 1e-4)
    assert r["samples"] >= 1 and "warm-up" in r["window"] and r["sm_mhz"] is not None
    # no nvidia-smi on the machine
    monkeypatch.setenv("PATH", str(tmp_path / "nothing"))
    s = bench.ClockSampler(0)
    s.start()
    assert s.stop(0, 1)["reasons"] == ["nvidia-smi unavailable"]


def test_reference_arm_prints_one_json_line_per_job():
    env = dict(os.environ, RANK="0", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                        "--gpus", "2"], env=env, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0
    rec = json.loads(r.stdout.strip())
    assert rec["impl"] == "reference" and rec["unavailable"]
    env["RANK"] = "1"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                        "--gpus", "2"], env=env, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_types_names_and_size_limit(tmp_path):
    import numpy as np
    import torch
    import bench
    out = {"loss": torch.tensor(2.5), "state/h": torch.ones(3, 4, dtype=torch.bfloat16),
           "ids": torch.arange(5), "big": torch.arange(40000, dtype=torch.float64),
           "step": 7, "note": "not an array"}
    got = bench.dump_outputs(out, str(tmp_path / "a"), limit=64 << 10)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["big.npy", "ids.npy", "loss.npy", "state_h.npy", "step.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 << 10
    loss = np.load(tmp_path / "a" / "loss.npy")
    assert loss.dtype == np.float32 and loss.shape == () and float(loss) == 2.5
    h = np.load(tmp_path / "a" / "state_h.npy")
    assert h.dtype == np.float32 and h.shape == (3, 4) and (h == 1).all()
    assert np.load(tmp_path / "a" / "ids.npy").dtype == np.float64
    assert float(np.load(tmp_path / "a" / "step.npy")) == 7.0
    # the large array is a sample of its elements: same positions on every call
    big = np.load(tmp_path / "a" / "big.npy")
    assert got["big"]["shape"] == [40000] and got["big"]["stored"] == big.size < 40000
    assert (np.diff(big) > 0).all() and (big == big.astype(np.int64)).all()
    bench.dump_outputs(out, str(tmp_path / "b"), limit=64 << 10)
    assert (np.load(tmp_path / "b" / "big.npy") == big).all()
    # under the limit nothing is sampled
    got = bench.dump_outputs({"big": out["big"]}, str(tmp_path / "c"))
    assert got["big"]["stored"] == 40000
    assert (np.load(tmp_path / "c" / "big.npy") == np.arange(40000)).all()


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "--steps" in r.stderr
