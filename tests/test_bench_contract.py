"""bench.py contract checks: the reference arm prints one JSON line with the agreed keys (no GPU needed), and
--dump-outputs writes the outputs of the timed steps (GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--cpu-rows", "256"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.split("\n") if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "examples/s" and d["higher_is_better"] is True
    for k in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data",
              "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["vs_baseline"] is None and d["dtype"] == "f32" and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["value"] > 0 and "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                         capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs(tmp_path):
    d = tmp_path / "dump"
    B, steps, warmup = 2048, 2, 3
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(warmup),
                          "--batch", str(B), "--no-sweep", "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(d)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.split("\n") if l.startswith("{")][-1])
    assert line["steps"] == steps
    got = {f[:-4]: np.load(d / f) for f in os.listdir(d)}
    assert set(got) == {"progress", "fea_cnt", "w", "sqrt_g", "z", "has_V", "V", "V_cg"}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(os.path.getsize(d / f) for f in os.listdir(d)) <= 64 << 20
    assert got["progress"][4] == (warmup + steps) * B          # nrows: every warm-up and timed step ran once
    n = len(got["w"])
    assert n > 1000 and got["V"].shape == got["V_cg"].shape == (n, 64)
    assert np.all(got["has_V"] == 1) and np.all(got["fea_cnt"] > 0)     # default hyper: every key owns a V row
