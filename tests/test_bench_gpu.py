"""bench.py on the GPU: --steps sets the timed steps and --dump-outputs writes what the last of them computed, the same
from run to run with the same arguments (BASELINE.json configs[0], a small workload, in a subprocess each time)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--config", "cfg1", "--steps", str(steps),
                        "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_bench_dumps_the_last_timed_step_reproducibly(tmp_path):
    d = _bench(tmp_path / "a", 3)
    assert d["steps"] == 3 and d["dump_outputs"]["bytes"] <= 64 << 20
    files = sorted(os.listdir(tmp_path / "a"))
    assert len(files) == d["dump_outputs"]["files"]
    a = {f: np.load(tmp_path / "a" / f) for f in files}
    assert all(x.dtype == np.float32 and np.isfinite(x).all() for x in a.values())
    for f in ("loss.npy", "masked_lm_loss.npy", "next_sentence_loss.npy", "seq_relationship_score.npy",
              "grad.bert.encoder.layer.1.output.dense.weight.npy", "grad.bert.embeddings.projection.weight.npy"):
        assert f in a, f
    assert a["loss.npy"] > 0 and np.abs(a["grad.bert.encoder.layer.1.output.dense.weight.npy"]).max() > 0
    _bench(tmp_path / "b", 3)
    assert sorted(os.listdir(tmp_path / "b")) == files
    for f in files:   # same inputs, same dropout masks; the kernels may only reorder fp32 sums
        b = np.load(tmp_path / "b" / f)
        assert b.shape == a[f].shape, f
        assert np.abs(b - a[f]).max() <= 1e-3 * max(np.abs(a[f]).max(), 1e-12), f
