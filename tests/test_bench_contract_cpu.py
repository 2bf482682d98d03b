"""bench.py contract checks that need no GPU: the reference arm (`--impl reference`: the oracle port timed on the host
cores) prints ONE JSON line with the keys the driver reads, rank != 0 under torchrun prints nothing, and the
algorithmic-byte formula is SURVEY.md 8(d)'s."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, env=e,
                          timeout=600, cwd=ROOT)


def test_reference_arm_prints_one_contract_line():
    r = run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--tokens", "512"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "tokens/s" and d["higher_is_better"] is True and d["scaling"] == "weak"
    assert d["metric"] == "byte-mix embedding fwd+bwd tokens/sec" and d["value"] > 0 and d["vs_baseline"] is None
    assert d["config"]["workload"] == "mot-sum-124M-48k" and d["dtype"] == "bf16" and d["data"] == "synthetic"
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "tokens" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_reference_arm_other_ranks_stay_silent():
    r = run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"], env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_steps_below_one_are_refused():
    r = run(["--impl", "reference", "--steps", "0"])
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr


def test_dump_outputs_stays_in_budget_and_samples_the_same_rows(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import numpy as np
    import torch
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 40_000)
    big = torch.arange(3000, dtype=torch.float32)[:, None].repeat(1, 8)     # every element holds its row number
    small = torch.randn(5, 4, dtype=torch.float64)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"big": big, "small": small, "scalar": torch.tensor(2.5)})
    a, b = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert a.dtype == np.float32 and np.array_equal(a, b)
    rows = a[:, 0].astype(np.int64)
    assert 0 < len(rows) < 3000 and np.all(np.diff(rows) > 0) and np.array_equal(a, big.float().numpy()[rows])
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), small.numpy())                  # float64 kept, whole
    assert np.load(tmp_path / "a" / "scalar.npy").tolist() == [2.5]
    assert sum(np.load(p).nbytes for p in (tmp_path / "a").iterdir()) <= 40_000


def test_algorithmic_bytes_follow_survey_8d():
    sys.path.insert(0, ROOT)
    import bench
    w = dict(bench.WORKLOADS["mot-sum-124M-48k"])
    fwd, bwd, Do = bench.algorithmic_bytes(w)
    N, Dt, bd, bpt, e, V, Vb = 49152, 768, 48, 16, 2, 50257, 458
    assert Do == Dt
    assert fwd == N * (4 + 4 * bpt + Dt * e + Do * e) + Vb * bd * e
    assert bwd == N * (Do * e + 4 + 4 * bpt + Dt * e) + V * Dt * e + Vb * bd * e
    assert abs((fwd + bwd) / 1e6 - 386.0) < 1.0          # the 386 MB per step DESIGN.md quotes


def test_arms_share_one_config_dict():
    """The driver compares the arms' `config`: ours, the CPU reference arm and the PyTorch-on-GPU arm describe the workload
    with the same dictionary (the full per-GPU batch in every arm)."""
    sys.path.insert(0, ROOT)
    import argparse
    import bench
    args = argparse.Namespace(dist="uniform")
    w = dict(bench.WORKLOADS["mot-sum-124M-48k"], name="mot-sum-124M-48k")
    c1, c2 = bench.main_config(w, args, 1), bench.main_config(w, args, 1)
    assert c1 == c2 and c1["tokens_per_gpu_per_step"] == 49152 and c1["parallelism"] == "dp1"
    assert bench.main_config(w, args, 8)["parallelism"].startswith("dp8")
    r = run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--tokens", "256"])
    d = json.loads(r.stdout.strip().splitlines()[-1])
    w["N"] = 256
    assert d["config"] == bench.main_config(w, args, 1)                # the reference arm prints exactly that dictionary
    assert "full per-GPU batch" in d["cpu_baseline"]["sample"] and "tokens_to_bytes" in d["cpu_baseline"]["sample"]
