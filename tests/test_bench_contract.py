"""CPU: bench.py's reference arm runs without a GPU and prints the contract's JSON line; the product arm refuses to run
without a B200 instead of falling back.  GPU: --dump-outputs writes what the last timed step computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT


def run_bench(*args, timeout=300):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=timeout,
                          cwd=ROOT)


def test_reference_arm_prints_the_contract_line():
    r = run_bench("--impl", "reference", "--steps", "2", "--warmup", "1", "--workload", "embedding")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1                                            # ONE JSON line
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "train samples/s" and d["unit"] == "samples/s"
    assert d["higher_is_better"] is True and d["steps"] == 2 and d["warmup"] == 1 and d["gpu_launches"] == 0
    assert d["value"] > 0 and abs(d["value"] - 128 * 1e3 / d["ms_per_step"]) <= 1e-6 * d["value"]
    assert d["config"]["workload"].startswith("embedding (config/embedding.yaml)") and d["config"]["params"] == 23608320
    cb = d["cpu_baseline"]
    live = os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "codae", "model"))
    assert cb["kind"] == ("reference" if live else "port")            # the unmodified reference classes when installed, else the port
    assert cb["cores"] == (os.cpu_count() or 1) and cb["value"] == d["value"] and "steps of 128 rows" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["vs_baseline"] is None and d["dtype"] == "f32" and d["data"] == "synthetic"


def test_reference_arm_port_and_live_reference_agree_on_the_workload():
    """CODAE_CPU_ARM=port forces the oracle port; both arms time the same step (same shapes, same batch) and report the kind."""
    env = dict(os.environ, CODAE_CPU_ARM="port")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--workload", "modanet"], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["cpu_baseline"]["kind"] == "port" and "steps of 32 rows" in d["cpu_baseline"]["sample"]


def test_default_workload_is_the_polyvore_shaped_step():
    """The default bench line is quoted on BASELINE.json configs[3] (10 x Linear(4096, 4096), B = 8192 per GPU); its CPU arm
    times a bounded 2048-row sample of that batch."""
    r = run_bench("--impl", "reference", "--steps", "1", "--warmup", "0", timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["config"]["workload"].startswith("polyvore (config/polyvore_multislot.yaml): 10 x Linear, io=4096, B=8192/GPU")
    assert d["config"]["params"] == 167813120 and "2048 rows (of the 8192-row batch)" in d["cpu_baseline"]["sample"]
    assert abs(d["value"] - 2048 * 1e3 / d["ms_per_step"]) <= 1e-6 * d["value"]


def test_reference_arm_other_ranks_exit_silently():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "2", "--warmup", "1"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    """--dump-outputs writes float32 / float64 arrays, under 64 MB in all, of the last timed step: its loss is the JSON line's
    loss_last_step, and the rows monitor counts exactly the warm-up and --steps steps."""
    out = tmp_path / "dump"
    r = run_bench("--workload", "embedding", "--steps", "5", "--warmup", "3", "--no-secondary", "--no-scoring", "--no-cpu",
                  "--dump-outputs", str(out), timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    a = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert sorted(a) == ["gradients", "loss", "monitors", "parameters", "reconstruction"]
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert float(a["loss"][0]) == d["loss_last_step"] and d["steps"] == 5
    assert a["monitors"][2] == 128 * (3 + 5)
    assert a["reconstruction"].shape == (128, 1536) and np.isfinite(a["reconstruction"]).all()
    assert a["parameters"].shape == a["gradients"].shape == (1 << 22,) and np.abs(a["gradients"]).max() > 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_product_arm_refuses_to_run_without_a_gpu():
    r = run_bench("--steps", "1", "--warmup", "0", timeout=120)
    assert r.returncode != 0 and "no CPU fallback" in r.stderr
