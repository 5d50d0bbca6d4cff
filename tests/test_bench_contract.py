"""bench.py's driver contract on the CPU: the reference arm (`--impl reference`, the reference's torch path on the host cores)
prints exactly ONE JSON line on stdout with the keys the driver reads.  (The GPU arm needs a B200; its line is checked by the
driver itself.)"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, OMP_NUM_THREADS="2")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c2", "--model", "lightgcn",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, p.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "epoch_s" and d["unit"] == "s" and d["higher_is_better"] is False
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["config"]["workload"].startswith("c2:")
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and d["dtype"] == "f32"


def test_other_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--workload", "c2",
                        "--model", "lightgcn", "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=120, env=env, cwd=ROOT)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_dump_outputs_writes_small_arrays_whole_and_a_repeatable_sample_of_large_ones(tmp_path, monkeypatch):
    import numpy as np
    import torch

    import bench

    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    monkeypatch.setattr(bench, "DUMP_WHOLE_BYTES", 1 << 16)
    model = torch.nn.Module()
    model.emb = torch.nn.Parameter(torch.randn(20_000, 64))  # 5 MB: sampled
    model.lin = torch.nn.Linear(64, 64)                       # 16 KB: whole
    losses = torch.tensor([0.5, 0.25])
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), losses, model, 0, 1)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["loss.npy", "param.emb.npy", "param.lin.bias.npy", "param.lin.weight.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= (1 << 20) + 128 * len(files)
    for f in files:
        assert np.load(tmp_path / "a" / f).tobytes() == np.load(tmp_path / "b" / f).tobytes(), f
    assert np.array_equal(np.load(tmp_path / "a" / "loss.npy"), losses.numpy())
    assert np.array_equal(np.load(tmp_path / "a" / "param.lin.weight.npy"), model.lin.weight.detach().numpy())
    emb, full = np.load(tmp_path / "a" / "param.emb.npy"), model.emb.detach().numpy()
    assert emb.dtype == np.float32 and 1000 < emb.shape[0] < full.shape[0] and emb.shape[1] == 64
    rows = [int(np.nonzero((full == r).all(1))[0][0]) for r in emb[:50]]
    assert rows == sorted(rows)
