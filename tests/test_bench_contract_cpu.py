"""bench.py contract checks that need no GPU: the reference arm (`--impl reference`, the oracle port timed on host
cores) prints ONE JSON line with the keys the driver reads; per-GPU batch of the configs BASELINE.json quotes as 8-GPU
global batches."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "cfg1", "--steps", "1",
                        "--warmup", "1", "--cpu-sample", "2"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "pairs/s"
    for k in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config",
              "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"]
    assert d["steps"] == 1 and d["cpu_baseline"]["spread"]["steps"] == 1   # --steps is the number of timed steps
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]


def test_dump_outputs_writes_float32_seeded_samples_within_64_mb(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    torch.manual_seed(0)
    model = torch.nn.Sequential(torch.nn.Embedding(30522, 768), torch.nn.Linear(768, 768))  # 94 MB of fp32 gradient
    for p in model.parameters():
        p.grad = torch.randn_like(p)
    outputs = {"loss": torch.tensor(1.5), "seq_relationship_score": torch.randn(4, 2).bfloat16()}
    n, total = bench.dump_outputs(str(tmp_path / "a"), outputs, model)
    files = sorted(os.listdir(tmp_path / "a"))
    assert n == len(files) == 5 and total <= 64 << 20
    assert files == ["grad.0.weight.npy", "grad.1.bias.npy", "grad.1.weight.npy", "loss.npy", "seq_relationship_score.npy"]
    a = {f: np.load(tmp_path / "a" / f) for f in files}
    assert all(x.dtype == np.float32 for x in a.values())
    assert a["loss.npy"] == 1.5 and np.array_equal(a["seq_relationship_score.npy"], outputs["seq_relationship_score"].float().numpy())
    assert np.array_equal(a["grad.1.weight.npy"], model[1].weight.grad.reshape(-1).numpy())   # small enough: whole
    big = a["grad.0.weight.npy"]
    assert 0 < big.size < model[0].weight.numel() and np.isin(big, model[0].weight.grad.numpy()).all()
    bench.dump_outputs(str(tmp_path / "b"), outputs, model)
    assert all(np.array_equal(np.load(tmp_path / "b" / f), a[f]) for f in files)   # the same positions every time


def test_per_gpu_batch_of_the_eight_gpu_configs():
    sys.path.insert(0, ROOT)
    import bench
    assert bench.build_cfg("cfg2")["B"] == 256          # quoted on 1 GPU
    assert bench.build_cfg("cfg3")["B"] == 512 // 8     # global batch over 8 data-parallel ranks
    assert bench.build_cfg("cfg4")["B"] == 256 // 8
    assert bench.build_cfg("cfg5")["B"] == 1024 // 8
    assert bench.build_cfg("cfg5", 16)["B"] == 16
    assert "configs[4]" in bench.workload_name(bench.build_cfg("cfg5"))
