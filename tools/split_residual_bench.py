"""The split residual of runs/71081 (V3g) at its shipped shape: the fused front (MoTSplitResidualEmbedding: one gather, one
backward) against the three-call composition it replaced (V3c + tok-only + bytes-only mot_embed launches, autograd adding
the two dense token-table gradients), alternated in one process.

    python tools/split_residual_bench.py [--tokens 65536] [--steps 50] [--warmup 10] [--rounds 5] [--out result.json]

Per arm: fwd+bwd step time from CUDA events (median over rounds of the mean over steps; every round runs both arms), and
the max-abs difference of the two arms' outputs and gradients on the same inputs.  Prints one JSON line with the card
name and power limit.  Working set: 103 MB token table + 3 x 134 MB of outputs and as many upstream gradients, larger than
the 126 MB L2."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "mixture-of-tokenizers_b200")]

import mot_b200  # noqa: E402
from mot_b200 import MixSpec  # noqa: E402

V, VB, D, BD = 50257, 458, 1024, 64   # runs/71081: GPT-2 vocabulary, 1024 = 16 x 64, byte vocabulary 458


def three_calls(m, tok, ids):
    Et, Eb = m.embed_tokens.weight, m.embed_bytes.weight
    x0t = mot_b200.mot_embed(tok, None, Et, None, MixSpec(combine="tok_only", tok_norm=True, out_norm=False))
    x0b = mot_b200.mot_embed(None, ids, None, Eb, MixSpec(combine="bytes_only", byte_norm=True, out_norm=False,
                                                          slot_major=True), bpt=m.bpt)
    x = mot_b200.mot_embed(tok, ids, Et, Eb, MixSpec(**mot_b200.RUN_VARIANTS["V3c"]), bpt=m.bpt, lam=m.lambdas.flip(0))
    return x[None], x0t[None], x0b[None]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tokens", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("split_residual_bench: needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    m = mot_b200.MoTSplitResidualEmbedding(V, VB, D, BD, D // BD).to(dev).bfloat16()
    g = torch.Generator(device=dev).manual_seed(1)
    tok = torch.randint(0, V, (a.tokens,), generator=g, device=dev, dtype=torch.int32)
    ids = torch.randint(0, VB, (m.bpt, a.tokens), generator=g, device=dev, dtype=torch.int32)
    grads = [torch.randn(1, a.tokens, D, generator=g, device=dev).bfloat16() for _ in range(3)]
    arms = {"fused": lambda: m(tok, ids), "three_calls": lambda: three_calls(m, tok, ids)}

    def step(fn):
        for p in m.parameters():
            p.grad = None
        outs = fn()
        torch.autograd.backward(list(outs), grads)
        return outs

    # the two arms on the same inputs
    res = {}
    for name, fn in arms.items():
        outs = step(fn)
        res[name] = [o.float() for o in outs] + [p.grad.float() for p in m.parameters()]
    names = ["x", "x0t", "x0b"] + [n + ".grad" for n, _ in m.named_parameters()]
    maxabs = {n: float((u - v).abs().max()) for n, u, v in zip(names, res["fused"], res["three_calls"])}
    del res

    times = {k: [] for k in arms}
    for name, fn in arms.items():
        for _ in range(a.warmup):
            step(fn)
    for _ in range(a.rounds):
        for name, fn in arms.items():
            for _ in range(a.warmup):
                step(fn)
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for _ in range(a.steps):
                step(fn)
            t1.record()
            t1.synchronize()
            times[name].append(t0.elapsed_time(t1) * 1000.0 / a.steps)
    gpu, power = card()
    out = {"tool": "split_residual_bench", "gpu": gpu, "power_limit": power, "tokens": a.tokens, "V": V, "D": D,
           "dtype": "bf16", "steps": a.steps, "rounds": a.rounds,
           "step_us": {k: round(statistics.median(v), 1) for k, v in times.items()},
           "step_us_rounds": {k: [round(x, 1) for x in v] for k, v in times.items()},
           "max_abs_fused_vs_three_calls": maxabs}
    out["speedup"] = round(out["step_us"]["three_calls"] / out["step_us"]["fused"], 3)
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
