"""Token-only byte mix against the explicit integer pipeline, on seeded inputs.

    python tools/ttb_pull_bench.py [--steps 20] [--rounds 5] [--out DIR]

For each workload two arms run the same training step (forward + backward of the embedding front):
  explicit   : create_batch's byte part (ttb_expand -> pull_from_left / pull_from_right -> slices) feeding the
               explicit-id kernels;
  token-only : the same call with token ids alone (and, for right pulls, the window's last column as the lookahead);
               the kernels derive the pulled ids from the ttb table.
The arms alternate inside one process (rounds x steps each, CUDA events, median round reported).  A separate
torch.profiler pass sums the device time per kernel group.  Workloads: mot-proj-spt-64k (pull_in), mot-proj-spt-addpp-64k,
both again with padding_in="right" (-right), and the MoT-sum front (V3) at 48K tokens with pulled ids.  Needs a CUDA
device; there is no CPU path.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", "mixture-of-tokenizers_b200"))

import torch  # noqa: E402

import mot_b200  # noqa: E402
from mot_b200 import data as D  # noqa: E402

V_TOK, V_BYTE, PAD, EOT = 50257, 458, 456, 457


def make_ttb(bpt: int, dev, side: str = "left") -> torch.Tensor:
    """int16 table padded on `side`: 1..8 bytes per token (GPT-2 tokens are short), the end-of-text row all EOT."""
    g = torch.Generator().manual_seed(0)
    t = torch.full((V_TOK, bpt), PAD, dtype=torch.int16)
    lens = torch.randint(1, 9, (V_TOK,), generator=g)
    vals = torch.randint(0, 256, (V_TOK, bpt), generator=g).to(torch.int16)
    if side == "left":
        mask = torch.arange(bpt)[None, :] >= (bpt - lens)[:, None]
    else:
        mask = torch.arange(bpt)[None, :] < lens[:, None]
    t[mask] = vals[mask]
    t[V_TOK - 1] = EOT
    return t.to(dev)


def make_tokens(B: int, S: int, dev) -> torch.Tensor:
    g = torch.Generator().manual_seed(1)
    tok = torch.randint(0, V_TOK - 1, (B, S), generator=g)
    tok[torch.rand(B, S, generator=g) < 1e-3] = V_TOK - 1      # a document boundary every ~1000 tokens
    return tok.to(torch.int32).to(dev)


def workloads(dev):
    bpt = 16
    ttb = make_ttb(bpt, dev)
    out = {}
    for name, pair, side in (("mot-proj-spt-64k", False, "left"), ("mot-proj-spt-addpp-64k", True, "left"),
                             ("mot-proj-spt-64k-right", False, "right"), ("mot-proj-spt-addpp-64k-right", True, "right")):
        torch.manual_seed(0)
        tab = ttb if side == "left" else make_ttb(bpt, dev, "right")
        mod = mot_b200.SptByteMixEmbedding(V_TOK, V_BYTE, 256, 48, 1024, bpt, pull_in=True, add_padded_and_pulled=pair,
                                           ttb=tab, padding_in=side).to(dev)
        mod.embed.bfloat16()
        toks = make_tokens(64, 1025, dev)                     # [B, S+1] as the loader yields them
        gout = torch.randn(64, 1024, 1024, device=dev, dtype=torch.bfloat16)

        def explicit(mod=mod, toks=toks, gout=gout, tab=tab, side=side):
            ti, bp, bl, _ = D.create_batch(toks, tab, None, bpt, pull_in=True, padding_in=side)
            mod(ti, bp, bl).backward(gout)

        def token_only(mod=mod, toks=toks, gout=gout, tab=tab, side=side):
            ti, _, _, _, nxt = D.create_batch(toks, tab, None, bpt, pull_in=True, padding_in=side, byte_ids=False,
                                              next_tokens=True)
            mod(ti, next_tokens=nxt if side == "right" else None).backward(gout)
        out[name] = (mod, explicit, token_only)

    torch.manual_seed(0)
    mod = mot_b200.MoTEmbedding(V_TOK, V_BYTE, 768, 48, bpt, variant="V3", ttb=ttb, pull_in=True).to(dev).to(torch.bfloat16)
    tok = make_tokens(1, 49152, dev)[0]
    gout = torch.randn(1, 49152, 768, device=dev, dtype=torch.bfloat16)

    def explicit_sum():
        ids = mot_b200.pull_from_left(mot_b200.ttb_expand(tok[None], ttb), bpt).view(bpt, -1)
        mod(tok, ids).backward(gout)

    def token_only_sum():
        mod(tok).backward(gout)
    out["mot-sum-124M-48k-pulled"] = (mod, explicit_sum, token_only_sum)
    return out


def time_arms(arms, steps: int, rounds: int):
    for f in arms.values():                                   # warm-up: every shape, every kernel
        for _ in range(3):
            f()
    torch.cuda.synchronize()
    res = {k: [] for k in arms}
    for _ in range(rounds):
        for k, f in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                f()
            e1.record()
            torch.cuda.synchronize()
            res[k].append(e0.elapsed_time(e1) / steps)
    return {k: {"ms_median": statistics.median(v), "ms_min": min(v), "ms_max": max(v)} for k, v in res.items()}


GROUPS = (("fwd", ("mot_fwd_kernel", "mot_pair_fwd")), ("bwd", ("mot_bwd_kernel", "mot_bwd_sum_kernel", "mot_pair_bwd")),
          ("integer", ("ttb_expand", "pull_")))


def kernel_times(f, steps: int):
    from torch.profiler import ProfilerActivity, profile
    f()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            f()
        torch.cuda.synchronize()
    sums = {g: 0.0 for g, _ in GROUPS}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
        for g, keys in GROUPS:
            if any(k in e.key for k in keys):
                sums[g] += t / 1000.0 / steps                # us -> ms per step
    return sums


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ttb_pull_bench: needs a CUDA device")
    dev = torch.device("cuda:0")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    report = {"gpu": gpu, "workloads": {}}
    for name, (mod, explicit, token_only) in workloads(dev).items():
        steps = time_arms({"explicit": explicit, "token_only": token_only}, args.steps, args.rounds)
        kern = {"explicit": kernel_times(explicit, 5), "token_only": kernel_times(token_only, 5)}
        report["workloads"][name] = {"step": steps, "kernels_ms": kern}
        print(json.dumps({name: report["workloads"][name]}), flush=True)
    print(json.dumps({"gpu": gpu}))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "ttb_pull_bench.json"), "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
