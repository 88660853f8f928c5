"""bench.py's GPU arm on a B200 (`pytest -m gpu`): a short run with --dump-outputs prints one JSON line for the requested
number of timed steps and leaves the loss of that line and every model-A parameter as float32 arrays within 64 MB."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import icap_loader

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pkg = icap_loader.load()


def test_dump_outputs(tmp_path):
    import bench
    out = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "1",
           "--no-decode", "--no-cpu-baseline", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["steps"] == 3
    names = [n for n in pkg.param_layout(pkg.ModelConfig(**bench.MODEL_A)) if not n.endswith("pos_table")]
    assert sorted(os.listdir(out)) == sorted(["loss.npy"] + [f"param.{n}.npy" for n in names])
    arrays = [np.load(out / f) for f in os.listdir(out)]
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in arrays)
    assert sum(a.nbytes for a in arrays) <= 64 << 20
    assert float(np.load(out / "loss.npy")[0]) == d["final_loss"]
