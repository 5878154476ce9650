"""bench.py --dump-outputs: after the timed steps the outputs of the last one are written as float32 / float64 .npy
files, and two runs with the same arguments write the same arrays (the inputs come from fixed seeds), so two builds
can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import conftest

pytestmark = pytest.mark.gpu

# c3 at its smallest: the one-scan step of the blocking calls, the align result plus the filtered cloud
ARGS = ["--config", "c3", "--steps", "2", "--warmup", "1", "--stream-scans", "3", "--no-cpu-baseline"]
NAMES = ["converged", "delta", "filtered_cloud", "final_transformation", "iterations", "n_correspondences", "n_filtered"]


def _run(out):
    r = subprocess.run([sys.executable, os.path.join(conftest.ROOT, "bench.py")] + ARGS + ["--dump-outputs", str(out)],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900, cwd=conftest.ROOT)
    assert r.returncode == 0, r.stderr[-800:]
    line = json.loads([l for l in r.stdout.splitlines() if l.strip()][-1])
    return line, {f[:-len(".npy")]: np.load(os.path.join(out, f)) for f in sorted(os.listdir(out))}


def test_dump_outputs_repeat_bit_for_bit(tmp_path):
    line, a = _run(tmp_path / "a")
    _, b = _run(tmp_path / "b")
    assert line["steps"] == 2
    assert sorted(a) == NAMES and sorted(b) == NAMES
    for k, v in a.items():
        assert v.dtype in (np.float32, np.float64), k
        assert np.array_equal(v, b[k]), k
    assert a["final_transformation"].shape == (1, 4, 4) and a["converged"][0] == 1
    assert a["filtered_cloud"].shape == (int(a["n_filtered"][0]), 4) and np.isfinite(a["filtered_cloud"]).all()
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
