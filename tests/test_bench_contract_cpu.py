"""bench.py contract on the CPU side: the reference arm (`--impl reference`, the oracle port timed on the host cores)
prints exactly one JSON line with the keys the driver reads, under plain python and under torchrun with two ranks
(rank 0 prints, the other exits 0 without work).  The b200 arm needs a GPU (tests/test_*_gpu.py + the driver)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ["impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
        "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"]


def _check(line, n_gpus):
    d = json.loads(line)
    for k in KEYS:
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "gicp_scans_per_sec" and d["unit"] == "scans/s"
    assert d["n_gpus"] == n_gpus and d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["value"] > 0 and abs(d["ms_per_step"] - 1000.0 / d["value"]) < 1e-6 * d["ms_per_step"] + 1e-9
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-800:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    _check(lines[0], 1)


def test_reference_arm_under_torchrun_rank0_only():
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.join(ROOT, "bench.py"),
                        "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-800:]
    lines = [l for l in r.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1
    _check(lines[0], 2)


def test_dump_outputs_refused_without_the_b200_arm(tmp_path):
    """--dump-outputs writes what the b200 arm's timed path returned; the CPU arm refuses it instead of ignoring it"""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path)],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=120, cwd=ROOT)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and not r.stdout.strip()
    assert os.listdir(tmp_path) == []


def test_reference_arm_c3_contract_line():
    """--config c3 (scan-to-submap, BASELINE configs[2]): same contract line; the CPU arm keeps the submap's kd-tree and
    covariances between scans, like the reference does while setInputTarget is not called again"""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "c3", "--impl", "reference", "--steps", "1",
                        "--warmup", "1", "--stream-scans", "3"],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-800:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    _check(lines[0], 1)
    d = json.loads(lines[0])
    assert d["config"]["name"] == "c3" and "500000-point submap" in d["config"]["workload"] and "corr 0.2" in d["config"]["workload"]
