"""bench.py contract checks.  Without a GPU: the reference arm (CPU port on a bounded sample) prints one JSON line with
the required keys; under torchrun only rank 0 prints.  On the GPU: --dump-outputs writes what the timed path returned."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = ["impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"]


def _check(line):
    j = json.loads(line)
    for k in REQUIRED:
        assert k in j, k
    assert j["impl"] == "reference" and j["metric"] == "Gauss-Newton steps/sec" and j["unit"] == "GN steps/s"
    assert j["dtype"] == "f64" and j["higher_is_better"] is True and j["vs_baseline"] is None
    assert j["e2e"] == {"value": j["value"], "unit": j["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = j["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and "sample" in cb and cb["value"] == j["value"] and j["value"] > 0
    assert "workload" in j["config"]
    assert cb["extrapolated"] is True and j["same_config"] is False          # the workload size itself is never run on the CPU
    big = cb["measured_at_largest_size"]
    assert big["N_domain"] == 300 and big["steps_per_s"] > 0


def test_reference_arm_single_process():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--cpu_sample_N", "200", "--cpu_big_N", "300", "--N_domain", "2000"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-1500:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    _check(lines[0])


def test_reference_arm_under_torchrun_only_rank0_prints():
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                          "--master-port", "29631", os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "0", "--cpu_sample_N", "200", "--cpu_big_N", "300", "--N_domain", "2000"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-1500:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    _check(lines[0])
    assert json.loads(lines[0])["n_gpus"] == 2


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(tmp_path):
    """--dump-outputs writes the loss history, GN iterate, solution vector and collocation errors of the last timed step
    in float64; they are the numbers the JSON line of the same run reports."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--N_domain", "2000",
                          "--nugget", "1e-8", "--skip_cpu_baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-1500:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j["steps"] == 2
    d = {n: np.load(tmp_path / f"{n}.npy") for n in ("loss_hist", "sol", "sol_vec", "pts_err")}
    assert all(v.dtype == np.float64 for v in d.values())
    N, M = j["config"]["n"], j["config"]["M"]
    assert d["loss_hist"].shape == (5,) and d["sol"].shape == (N,) and d["sol_vec"].shape == (M,) and d["pts_err"].shape == (N,)
    assert d["loss_hist"][-1] == j["result"]["final_loss"] and d["pts_err"].max() == j["result"]["pts_max_err"]
