"""Data-parallel step of the embedding front plus the three value embeddings (runs/7:252,308), four ways of exchanging
their gradients.  Run under torchrun on one node:

    torchrun --nproc-per-node N tools/dp_value_embeds_bench.py [--rounds 7] [--steps 20] [--shapes 768,1024]

One step = MoTEmbedding V3 forward + TokenValueEmbeddings(3) forward, backward of both, and the gradient exchange.
Shapes: 768/48 at 49152 tokens per GPU (the 124M model) and 1024/64 at 65536 (what runs/71 ships), each with uniform
and with Zipf token ids (bench.make_tokens: Zipf(1.0) over a seeded permutation, an EOT about every 800 tokens).
Arms, alternated round by round in one process:
  (a) rows  : one bucket [token table | 3 value tables | byte table], row_tables=4, touched-rows exchange
  (b) dense : the same bucket exchanged whole by the library's kernel (sparse_rows=False, what MOT_DP_DENSE=1 selects)
  (c) ref   : the reference's way: the front's own bucket + dist.all_reduce(AVG) on each value-embedding gradient
  (d) nccl  : everything in one bucket in ordinary memory (symmetric=False): one NCCL all-reduce
Per arm: the step time (median over rounds of the mean of `--steps` steps, slowest rank), the exchange alone (CUDA
events around the exchange inside the step: it includes the wait for the slowest rank at the entry barrier), tokens/s,
and for (a) the union density of the row bitmap.  Last, a value check of every arm: the exchanged gradients against an
fp32 NCCL average of the ranks' own gradients.  Rank 0 prints the card name and power limit and one JSON line per
shape and distribution."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "mixture-of-tokenizers_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch
import torch.distributed as dist

import mot_b200
from mot_b200 import dp
from bench import V_BYTE, V_TOK, make_tokens

SHAPES = {768: dict(Dt=768, bd=48, N=49152), 1024: dict(Dt=1024, bd=64, N=65536)}
BPT = 16


def card():
    try:
        pl = subprocess.run(["nvidia-smi", f"--id={torch.cuda.current_device()}", "--query-gpu=power.limit",
                             "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        pl = f"unknown ({type(e).__name__})"
    return torch.cuda.get_device_name(), pl


class Arm:
    def __init__(self, name, front, ve, dev):
        self.name, self.front, self.ve = name, front, ve
        self.params = [front.embed_tokens.weight, *(m.weight for m in ve.value_embeds), front.embed_bytes.weight]
        if name in ("rows", "dense"):
            self.bucket = dp.GradBucket(self.params, symmetric=True, row_tables=4, sparse_rows=(name == "rows"))
            if self.bucket._symm is None:
                raise SystemExit("dp_value_embeds_bench: no symmetric memory on this node")
            assert self.bucket.sparse_rows == (name == "rows"), "touched-rows exchange unavailable at this world size"
        elif name == "ref":
            self.bucket = dp.GradBucket(self.params[:1] + self.params[-1:], symmetric=True)
        else:
            self.bucket = dp.GradBucket(self.params, symmetric=False)

    def attach(self):
        self.front.attach_grad_bucket(self.bucket)
        self.ve.grad_bucket = None if self.name == "ref" else self.bucket

    def exchange(self):
        self.bucket.all_reduce_avg()
        if self.name == "ref":
            for m in self.ve.value_embeds:
                dist.all_reduce(m.weight.grad, op=dist.ReduceOp.AVG)


def run_shape(D, dist_name, args, rank, world, dev):
    cfg = SHAPES[D]
    Dt, bd, N = cfg["Dt"], cfg["bd"], cfg["N"]
    torch.manual_seed(0)
    front = mot_b200.MoTEmbedding(V_TOK, V_BYTE, Dt, bd, BPT, variant="V3").to(dev).bfloat16()
    ve = mot_b200.TokenValueEmbeddings(V_TOK, Dt, 3).to(dev).bfloat16()
    dp.broadcast_params([*front.parameters(), *ve.parameters()])
    tok = make_tokens(N, dist_name, 12345 + rank, dev)
    g = torch.Generator(device=dev).manual_seed(7 + rank)
    ids = torch.randint(0, V_BYTE, (BPT, N), generator=g, device=dev, dtype=torch.int32)
    go = torch.randn(1, N, Dt, generator=g, device=dev).bfloat16()
    gvs = [torch.randn(N, Dt, generator=g, device=dev).bfloat16() for _ in range(3)]
    arms = [Arm(n, front, ve, dev) for n in ("rows", "dense", "ref", "nccl")]

    def step(arm, ev=None):
        for p in arm.params:
            p.grad = None
        torch.autograd.backward([front(tok, ids), *ve(tok)], [go, *gvs])
        if ev is not None:
            ev[0].record()
        arm.exchange()
        if ev is not None:
            ev[1].record()

    def slowest(x):
        t = torch.tensor([x], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    step_ms = {a.name: [] for a in arms}
    xchg_ms = {a.name: [] for a in arms}
    for a in arms:
        a.attach()
        for _ in range(args.warmup):
            step(a)
    for _ in range(args.rounds):
        for a in arms:
            a.attach()
            dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                step(a)
            e1.record()
            torch.cuda.synchronize()
            step_ms[a.name].append(slowest(e0.elapsed_time(e1) / args.steps))
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
            dist.barrier()
            for ev in evs:
                step(a, ev)
            torch.cuda.synchronize()
            xchg_ms[a.name].append(slowest(statistics.median(x.elapsed_time(y) for x, y in evs)))

    # union density of the row bitmap (arm a) and the value check of every arm
    res = {"shape": f"{Dt}/{bd}", "tokens_per_gpu": N, "dist": dist_name, "world": world,
           "bucket_mb": arms[0].bucket.flat.numel() * 2 / 1e6, "arms": {}}
    for a in arms:
        a.attach()
        for p in a.params:
            p.grad = None
        torch.autograd.backward([front(tok, ids), *ve(tok)], [go, *gvs])
        want = [p.grad.float() for p in a.params]
        for w in want:
            dist.all_reduce(w, op=dist.ReduceOp.SUM)
            w /= world
        if a.name == "rows":
            hit = ((a.bucket.bitmap[:, None] >> torch.arange(32, device=dev, dtype=torch.int32)) & 1).reshape(-1)[:V_TOK]
            hit = hit.contiguous()
            dist.all_reduce(hit, op=dist.ReduceOp.MAX)
            res["rows_union_density"] = float(hit.float().mean())
        a.exchange()
        torch.cuda.synchronize()
        err = slowest(max(float((p.grad.float() - w).abs().max() / w.abs().max().clamp_min(1e-30))
                          for p, w in zip(a.params, want)))
        ms = statistics.median(step_ms[a.name])
        res["arms"][a.name] = {"step_ms_median": ms, "step_ms_rounds": step_ms[a.name],
                               "exchange_ms_median": statistics.median(xchg_ms[a.name]),
                               "tokens_per_sec": world * N / (ms * 1e-3),
                               "max_rel_err_vs_fp32_nccl": err, "check": "ok" if err <= 2.0 ** -7 else "FAILED"}
    front.grad_bucket = ve.grad_bucket = None
    del arms
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--shapes", default="768,1024")
    ap.add_argument("--dists", default="uniform,zipf")
    args = ap.parse_args()
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    try:
        name, pl = card()
        if rank == 0:
            print(f"# {world} x {name}, power limit {pl}; median of {args.rounds} rounds x {args.steps} steps, "
                  "arms alternated", flush=True)
        for D in (int(s) for s in args.shapes.split(",")):
            for dist_name in args.dists.split(","):
                res = run_shape(D, dist_name, args, rank, world, dev)
                res["card"], res["power_limit"] = name, pl
                if rank == 0:
                    a = res["arms"]
                    print(f"# {res['shape']} {dist_name}: step (a) rows {a['rows']['step_ms_median']:.3f} ms, "
                          f"(b) dense {a['dense']['step_ms_median']:.3f}, (c) ref {a['ref']['step_ms_median']:.3f}, "
                          f"(d) nccl {a['nccl']['step_ms_median']:.3f}; union density "
                          f"{res.get('rows_union_density', float('nan')):.3f}", flush=True)
                    print(json.dumps(res), flush=True)
    finally:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
