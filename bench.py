#!/usr/bin/env python
"""bench.py -- byte-mix embedding fwd+bwd throughput (tokens/s) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one forward + one backward of the fused byte-mix embedding over one
synthetic batch (per GPU), plus -- for N > 1 -- the all-reduce(AVG) of the dense
token / byte embedding gradients (the one exchange step of the path,
spt/train_gpt.py:1320-1321, runs/7:697-700).  Prints ONE JSON line (rank 0).

`value`   : tokens/s, whole job, inputs resident in HBM, CUDA-event timed.
`e2e`     : same metric through the module API with token / byte ids in pinned host memory
            (H2D every step) and a D2H read of the byte-embedding gradient every step.
`roofline`: the dominant kernel (backward) timed with CUDA events recorded by the library
            immediately around that kernel on its launch stream, against MEASURED_PEAKS.json.
`cpu_baseline`: the oracle port of the reference (eager torch CPU, all host cores) on a bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "mixture-of-tokenizers_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch

V_TOK, V_BYTE = 50257, 458

# name -> config.  N = tokens per GPU per step.
WORKLOADS = {
    # BASELINE.json configs[2]: modded-nanogpt 124M byte-mix embedding, 48K tokens/GPU/step, bf16.
    # MoT-sum (runs/71:228-230,312-314) at model_dim 768 = 16 bytes x 48.
    "mot-sum-124M-48k": dict(variant="V3", N=49152, Dt=768, bd=48, bpt=16, dtype="bf16"),
    # what the reference runs ship (runs/71:496,500-501): 64K tokens, 1024 = 16 x 64
    "mot-sum-medium-64k": dict(variant="V3", N=65536, Dt=1024, bd=64, bpt=16, dtype="bf16"),
    "mot-sum-medium-48k": dict(variant="V3", N=49152, Dt=1024, bd=64, bpt=16, dtype="bf16"),
    "mot-sum-1m": dict(variant="V3", N=1048576, Dt=1024, bd=64, bpt=16, dtype="bf16"),
    "mot-concat-711": dict(variant="V4", N=65536, Dt=512, bd=32, bpt=16, dtype="bf16"),
    "mot-norm-lambdas-71041": dict(variant="V3d", N=65536, Dt=1024, bd=64, bpt=16, dtype="bf16"),
    # concat + dense projection (tensor-core bound): runs/7 (1024/64 -> 1024, K = 2048, runs/7:496-503) and the
    # scaled-pre-train default (256/48 -> 1024, K = 1024, B=64 x S=1024 per GPU, spt/train_gpt.py:822)
    "mot-proj-runs7-64k": dict(variant="V1", N=65536, Dt=1024, bd=64, bpt=16, Do=1024, dtype="bf16"),
    "mot-proj-spt-64k": dict(variant="V1", N=65536, Dt=256, bd=48, bpt=16, Do=1024, dtype="bf16"),
    # BASELINE.json configs[3] "16/32 bytes-per-token padding": 32 bytes per token (K = 256 + 32 x 48 = 1792; runs/71072 is
    # the only reference script with bpt 32, spt/train_gpt.py:922 admits 16/18/20)
    "mot-proj-spt-bpt32-64k": dict(variant="V1", N=65536, Dt=256, bd=48, bpt=32, Do=1024, dtype="bf16"),
    # scaled-pre-train with --add-padded-and-pulled (spt/train_gpt.py:371-379): two int64 id tensors, rows summed before
    # the per-byte norm (mot_byte_pair_*), same projection
    "mot-proj-spt-addpp-64k": dict(variant="V1", N=65536, Dt=256, bd=48, bpt=16, Do=1024, dtype="bf16", pair=True),
    # SURVEY 8(f)-2: the three value embeddings gathered with the same token ids (runs/7:252,308), dense grads
    "value-embeds-64k": dict(variant="VE", N=65536, Dt=1024, bd=0, bpt=0, dtype="bf16", tables=3),
    # BASELINE.json configs[1]: mathblations digit mixin (mathblations/model.py:256-268): B=1024, S=11, dpt 4,
    # vocab 10003, 256/256 -> K = 1280 -> 256, fp32 parameters, TF32 matmul; launch-latency bound
    "mathblations-concat": dict(variant="V8", N=1024 * 11, Dt=256, bd=256, bpt=4, Do=256, dtype="f32"),
}
DEFAULT_WORKLOAD = "mot-sum-124M-48k"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", choices=["ours", "reference", "torch-gpu"], default="ours")
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--tokens", type=int, default=0, help="override tokens per GPU per step")
    ap.add_argument("--dist", choices=["uniform", "zipf"], default="uniform",
                    help="token id distribution: uniform = the reference's own warm-up generator (runs/7:633-635)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-torch-gpu", action="store_true", help="skip the PyTorch-on-the-same-GPU arm (eager + torch.compile)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (output, gradients) as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return a


DUMP_BYTES = 60 << 20   # data of all files; leaves room for the .npy headers under 64 MB


def dump_outputs(path, arrays, seed=0):
    """Write each tensor of `arrays` as <path>/<name>.npy in float32 (float64 stays float64), DUMP_BYTES in all.  The
    smallest go first and are written whole; a tensor larger than an even share of what is left keeps a sample of its
    rows (leading dimension), the same sorted rows on every run, so two builds can be compared output for output."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    left, items = DUMP_BYTES, sorted(arrays.items(), key=lambda kv: kv[1].numel())
    for i, (name, t) in enumerate(items):
        t = t.detach().reshape(-1) if t.dim() == 0 else t.detach()
        dt = torch.float64 if t.dtype == torch.float64 else torch.float32
        row_bytes = max(1, t[0].numel()) * dt.itemsize
        keep = min(t.shape[0], left // (len(items) - i) // row_bytes)
        if keep < t.shape[0]:
            rows = np.sort(np.random.default_rng(seed).choice(t.shape[0], keep, replace=False))
            t = t.index_select(0, torch.from_numpy(rows).to(t.device))
        a = t.to(dt).cpu().numpy()
        np.save(os.path.join(path, f"{name}.npy"), a)
        left -= a.nbytes


def workload_config(args):
    w = dict(WORKLOADS[args.workload])
    if args.tokens:
        w["N"] = args.tokens
    w["name"] = args.workload
    return w


def algorithmic_bytes(w):
    """BASELINE.md section 3 (ids given as a tensor, R = 1 because the mixed row is normalised)."""
    e = 2 if w["dtype"] == "bf16" else 4
    N, Dt, bd, bpt = w["N"], w["Dt"], w["bd"], w["bpt"]
    Do = {"V3": Dt, "V3d": Dt, "V4": Dt + bpt * bd, "V1": w.get("Do", Dt)}[w["variant"]]
    fwd = N * (4 + 4 * bpt + Dt * e + Do * e) + V_BYTE * bd * e
    bwd = N * (Do * e + 4 + 4 * bpt + Dt * e) + V_TOK * Dt * e + V_BYTE * bd * e
    return fwd, bwd, Do


def main_config(w, args, world):
    """`config` of the JSON line: a pure function of the workload and the launch, identical for --impl ours / reference /
    torch-gpu (what differs between the arms is reported beside it, never inside it)."""
    e = 2 if w["dtype"] == "bf16" else 4
    Do = algorithmic_bytes(w)[2]
    return {"workload": w["name"], "variant": w["variant"], "tokens_per_gpu_per_step": w["N"], "token_dim": w["Dt"],
            "byte_dim": w["bd"], "bytes_per_token": w["bpt"], "out_dim": Do, "token_dist": args.dist,
            "byte_ids": "uniform randint(0,458), given as a tensor (runs/7:635 layout)",
            "l2": f"working set {(2 * V_TOK * w['Dt'] * e + 2 * w['N'] * Do * e) / 1e6:.0f} MB > 126 MB L2, no flush",
            "parallelism": f"dp{world}" + (", tables replicated, one exchange (average) of the dense table gradients per step"
                                           if world > 1 else "")}


def make_tokens(N, dist, seed, device="cpu"):
    g = torch.Generator().manual_seed(seed)
    if dist == "uniform":
        return torch.randint(0, V_TOK - 1, (N,), generator=g, dtype=torch.int32).to(device)
    # Zipf(1.0) over a seeded permutation of the vocabulary, EOT every ~800 tokens ("FineWeb-shape")
    ranks = torch.arange(1, V_TOK, dtype=torch.float64)
    p = (1.0 / ranks)
    p /= p.sum()
    perm = torch.randperm(V_TOK - 1, generator=g)
    toks = perm[torch.multinomial(p, N, replacement=True, generator=g)].int()
    eot = torch.rand(N, generator=g) < 1.0 / 800
    toks[eot] = V_TOK - 1
    return toks.to(device)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_traffic(workload, kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu capture of this workload (profiles/traffic.json)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[workload][kernel]
    except Exception:
        return None


def measured_tensor_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(path))["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained: kernel timed inside a long step)"
    except Exception:
        return 1400.0, "fallback (B200_PROFILING.md ~1.4 PFLOP/s sustained)"


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            d = json.load(open(path))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ----------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference path, eager torch on the host cores
# ----------------------------------------------------------------------------------------------
def cpu_reference_step_fn(w, n_sample, seed=12345):
    from oracle import mot_oracle as O
    g = torch.Generator().manual_seed(seed)
    if w["variant"] == "VE":   # the value embeddings: plain gathers + dense grads (runs/7:252,308)
        dt = torch.bfloat16
        toks = torch.randint(0, V_TOK - 1, (n_sample,), generator=g, dtype=torch.int32)
        tables = [torch.randn(V_TOK, w["Dt"], generator=g).to(dt) for _ in range(w["tables"])]
        gouts = [torch.randn(n_sample, w["Dt"], generator=g).to(dt) for _ in range(w["tables"])]
        return lambda: O.value_embeds_fwd_bwd(toks, tables, gouts, math_dtype=dt)
    spec = O.VARIANTS[w["variant"]][0]
    Dt, bd, bpt = w["Dt"], w["bd"], w["bpt"]
    Do = algorithmic_bytes(w)[2]
    dt = torch.bfloat16 if w["dtype"] == "bf16" else torch.float32
    toks = torch.randint(0, V_TOK - 1, (n_sample,), generator=g, dtype=torch.int32)
    slot_major = w["variant"].startswith("V3")
    Do = w.get("Do", Do)
    ids = torch.randint(0, V_BYTE, (bpt, n_sample) if slot_major else (1, n_sample * bpt), generator=g, dtype=torch.int32)
    E_tok = torch.randn(V_TOK, Dt, generator=g).to(dt)   # nn.Embedding N(0,1) -> bf16 (train_gpt.py:1124-1126)
    E_byte = torch.randn(V_BYTE, bd, generator=g).to(dt)
    gout = torch.randn(n_sample, Do, generator=g).to(dt)
    kw = dict(bpt=bpt, slot_major=slot_major)
    if w["variant"] == "V1":
        K = Dt + bpt * bd
        kw["W"] = ((torch.rand(w["Do"], K, generator=g) * 2 - 1) * (3 ** 0.5) * 0.5 * K ** -0.5).to(dt)
    if w["variant"] in ("V3c", "V3d"):
        kw["lam_tok"], kw["lam_byte"] = torch.tensor(0.5), torch.tensor(0.5)
    if w.get("pair"):
        kw["byte_ids2"] = torch.randint(0, V_BYTE, (1, n_sample * bpt), generator=g, dtype=torch.int32)

    import numpy as np
    ttb = torch.randint(0, V_BYTE, (V_TOK, max(bpt, 1)), generator=g).to(torch.int16).numpy()   # synthetic table, uniform ids

    def step():
        # the loader's per-step expansion (runs/7:477-485: tokens_to_bytes, then `.view(bpt, -1)` for the sum runs) ...
        flat = O.tokens_to_bytes(toks.numpy(), ttb)
        ids_step = torch.from_numpy(np.ascontiguousarray(flat.reshape(bpt, -1) if slot_major else flat).astype(np.int32))
        # ... and the model front: the reference computes in the parameter dtype (eager bf16); math_dtype=dt reproduces that cost
        O.mot_embed_fwd_bwd(spec, toks, ids_step if ids_step.shape == ids.shape else ids, E_tok, E_byte, gout, math_dtype=dt, **kw)
    return step


def time_cpu_reference(w, steps, warmup, budget_s=20.0, n_sample=None):
    """The oracle port on the host cores.  n_sample=None: the FULL per-GPU batch of the workload (same config as the GPU
    arm); the number of timed steps is bounded by `budget_s` seconds (budget_s=None: exactly `steps`)."""
    torch.set_num_threads(os.cpu_count() or 1)
    n_sample = w["N"] if n_sample is None else min(w["N"], n_sample)
    step = cpu_reference_step_fn(w, n_sample)
    for _ in range(max(1, min(warmup, 3))):
        step()
    t0 = time.perf_counter(); step(); one = time.perf_counter() - t0
    reps = steps if budget_s is None else max(1, min(steps, int(budget_s / max(one, 1e-6))))
    t0 = time.perf_counter()
    for _ in range(reps):
        step()
    dt = (time.perf_counter() - t0) / reps
    return {"value": n_sample / dt, "unit": "tokens/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{reps} steps of {n_sample} tokens ({'the full per-GPU batch' if n_sample == w['N'] else 'a sample'} of the "
                      f"same workload): oracle/mot_oracle.py, eager torch {w['dtype']} on CPU, per step: tokens_to_bytes through "
                      f"the ttb table (runs/7:477-485) + fwd + bwd incl. the dense [50257,{w['Dt']}] gradient",
            "ms_per_step": dt * 1e3, "n_sample": n_sample, "steps": reps, "warmup": max(1, min(warmup, 3))}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    w = workload_config(args)
    r = time_cpu_reference(w, args.steps, args.warmup, budget_s=None)
    cfg = main_config(w, args, world) if w["variant"] in ("V3", "V3d", "V4") else \
        {"workload": w["name"], "variant": w["variant"], "tokens_per_gpu_per_step": w["N"], "token_dim": w["Dt"],
         "byte_dim": w["bd"], "bytes_per_token": w["bpt"]}
    line = {"impl": "reference", "metric": "byte-mix embedding fwd+bwd tokens/sec", "value": r["value"], "unit": "tokens/s",
            "n_gpus": args.gpus, "steps": r["steps"], "warmup": r["warmup"], "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": w["dtype"], "data": "synthetic",
            "config": cfg,
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# PyTorch on the same B200: the reference's own lines restated with torch ops on device="cuda" (SURVEY 2.3: "the bar is
# PyTorch 2.11's eager / torch.compile of the same lines on the same B200").  Written out here (not imported from oracle/).
# ----------------------------------------------------------------------------------------------
def torch_gpu_step_fn(w, dev, seed=12345):
    import torch.nn.functional as F
    g = torch.Generator(device=dev).manual_seed(seed)
    dt = torch.bfloat16 if w["dtype"] == "bf16" else torch.float32
    N, Dt, bd, bpt = w["N"], w["Dt"], w["bd"], w["bpt"]
    Do = algorithmic_bytes(w)[2]
    embed_tokens = torch.nn.Embedding(V_TOK, Dt, device=dev, dtype=dt)
    embed_bytes = torch.nn.Embedding(V_BYTE, bd, device=dev, dtype=dt)
    tok = torch.randint(0, V_TOK - 1, (N,), generator=g, device=dev, dtype=torch.int32)
    slot_major = w["variant"].startswith("V3")
    ids = torch.randint(0, V_BYTE, (bpt, N) if slot_major else (1, N * bpt), generator=g, device=dev, dtype=torch.int32)
    gout = torch.randn(1, N, Do, generator=g, device=dev).to(dt)
    scalars = torch.nn.Parameter(torch.tensor([0.5, 0.5], device=dev))

    def norm(x):                                   # runs/71:132-133
        return F.rms_norm(x, (x.size(-1),))

    def model(token_inputs, byte_inputs):
        if w["variant"] == "V3":                   # runs/71:228-230,312-314
            x_toks = embed_tokens(token_inputs)[None]
            x_bytes = embed_bytes(byte_inputs).squeeze()
            return norm(x_toks + torch.cat([b for b in x_bytes], dim=-1)[None])
        if w["variant"] == "V3d":                  # runs/71041:226-228,311-313
            x_toks = norm(embed_tokens(token_inputs)[None]) * scalars[-1]
            x_bytes = norm(embed_bytes(byte_inputs).squeeze()) * scalars[-2]
            return norm(x_toks + torch.cat([b for b in x_bytes], dim=-1)[None])
        if w["variant"] == "V4":                   # runs/711:224-232,314-316
            x_toks = embed_tokens(token_inputs)[None]
            x_bytes = embed_bytes(byte_inputs).squeeze()[None]
            B, T, _ = x_toks.shape
            return norm(torch.cat([x_toks, x_bytes.view(B, T, -1)], dim=-1))
        raise SystemExit(f"torch-gpu arm: no restatement for variant {w['variant']}")

    params = [embed_tokens.weight, embed_bytes.weight] + ([scalars] if w["variant"] == "V3d" else [])

    def make_step(fn):
        def step():
            for p_ in params:
                p_.grad = None
            fn(tok, ids).backward(gout)
        return step
    return make_step(model), make_step(torch.compile(model, dynamic=False)), params


def time_torch_gpu(w, dev, steps=20, warmup=5):
    """ms per fwd+bwd step of the PyTorch restatement, eager and torch.compile(dynamic=False) (the reference's setting,
    runs/7:623), CUDA-event timed after warm-up (the compile happens in the warm-up)."""
    eager, compiled, _ = torch_gpu_step_fn(w, dev)
    out = {"what": "the reference's forward lines restated with torch ops on the same GPU (nn.Embedding gathers, cat, add, "
                   "F.rms_norm) + autograd backward incl. the dense embedding gradients; inputs resident in HBM",
           "torch": torch.__version__}
    for name, fn in (("eager", eager), ("compiled", compiled)):
        try:
            for _ in range(warmup):
                fn()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(steps):
                fn()
            b.record(); torch.cuda.synchronize()
            ms = a.elapsed_time(b) / steps
            out[f"{name}_ms_per_step"] = ms
            out[f"{name}_tokens_per_sec"] = w["N"] / (ms * 1e-3)
        except Exception as e:  # noqa: BLE001 - an arm that cannot run is reported, not fatal
            out[f"{name}_error"] = f"{type(e).__name__}: {str(e)[:200]}"
    return out


def run_torch_gpu(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    w = workload_config(args)
    r = time_torch_gpu(w, dev, steps=args.steps, warmup=max(3, min(args.warmup, 10)))
    best = min(v for k, v in r.items() if k.endswith("_ms_per_step"))
    line = {"impl": "torch-gpu", "metric": "byte-mix embedding fwd+bwd tokens/sec", "value": w["N"] / (best * 1e-3), "unit": "tokens/s",
            "n_gpus": 1, "steps": args.steps, "warmup": max(3, min(args.warmup, 10)), "ms_per_step": best,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": w["dtype"], "data": "synthetic",
            "config": main_config(w, args, world), "torch_gpu": r, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    import mot_b200
    from mot_b200 import ops, _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group(backend="nccl", device_id=dev)
    w = workload_config(args)
    N, Dt, bd, bpt = w["N"], w["Dt"], w["bd"], w["bpt"]
    dt = torch.bfloat16 if w["dtype"] == "bf16" else torch.float32
    esz = 2 if dt == torch.bfloat16 else 4
    A_fwd, A_bwd, Do = algorithmic_bytes(w)
    spec_kw = dict(mot_b200.RUN_VARIANTS[w["variant"]])
    slot_major = spec_kw.get("slot_major", False)
    spec = mot_b200.MixSpec(**spec_kw)

    # ---- synthetic inputs, resident in HBM (rank r owns its own shard of the stream: seed + rank) ----
    g = torch.Generator(device=dev).manual_seed(12345)       # tables identical on every rank (replicas)
    E_tok = torch.randn(V_TOK, Dt, generator=g, device=dev).to(dt)
    E_byte = torch.randn(V_BYTE, bd, generator=g, device=dev).to(dt)
    gd = torch.Generator(device=dev).manual_seed(12345 + 1000 * (rank + 1))
    tok_host = make_tokens(N, args.dist, 12345 + rank).pin_memory()
    tok = tok_host.to(dev)
    ids_shape = (bpt, N) if slot_major else (1, N * bpt)
    ids = torch.randint(0, V_BYTE, ids_shape, generator=gd, device=dev, dtype=torch.int32)  # runs/7:635
    ids_host = ids.cpu().pin_memory()
    gout = torch.randn(N, Do, generator=gd, device=dev).to(dt)
    lam = torch.tensor([0.5, 0.5], device=dev) if w["variant"] in ("V3c", "V3d") else None
    out = torch.empty(N, Do, dtype=dt, device=dev)
    # what F.rms_norm's autograd node keeps: the forward result and rstd (read by the saved-output backward of the
    # MoT-sum variant; the other variants rebuild the mixed row and ignore them)
    rstd = None   # allocated below once the descriptor exists: only where the library would use it
    # one flat gradient bucket [gE_tok | gE_byte] the backward writes into -> a single NCCL all-reduce (SURVEY 2.3 C2)
    from mot_b200 import dp
    bucket = dp.GradBucket([torch.nn.Parameter(E_tok, requires_grad=False), torch.nn.Parameter(E_byte, requires_grad=False)],
                           symmetric="auto" if world > 1 else False)
    gE_tok, gE_byte = bucket.views()
    g_lam = torch.empty(2, dtype=torch.float32, device=dev) if lam is not None else None
    desc = ops.make_desc(spec, N, E_tok, E_byte, bpt, ids=ids, ttb=None, has_lam=lam is not None, seq_len=N)
    if ops.embed_bwd_uses_saved(desc):
        rstd = torch.empty(N, dtype=torch.float32, device=dev)
    # N > 1: where the bucket lives in symmetric memory and the variant has the saved-output backward, the step is a
    # PIPELINE: the backward walks the vocabulary in slabs and the rows of slab k are averaged across ranks on the
    # exchange stream while slab k + 1 is computed (mot_embed_bwd_slab + mot_dp_exchange); else one exchange after it.
    n_slabs = bucket.n_slabs if (world > 1 and bucket.pipelined and rstd is not None and not os.environ.get("MOT_DP_NO_OVERLAP")) else 1
    if n_slabs > 1:
        desc = ops.make_desc(spec, N, E_tok, E_byte, bpt, ids=ids, ttb=None, has_lam=lam is not None, seq_len=N, dp_slabs=n_slabs)
    ws = ops.acquire_workspace(desc, dev)   # kept across steps: every completed backward leaves it clean (no memset)
    main_stream = torch.cuda.current_stream(dev)

    def compute_step(exchange=True):
        # the same call sequence as mot_b200.mot_embed + autograd: the backward plan (counting sort of the token ids)
        # is launched on a side stream beside the forward kernel, the backward waits for it
        ops.embed_plan_async(desc, tok, ws, dev)
        ops.embed_forward_out(desc, tok, ids, None, E_tok, E_byte, lam, out, rstd=rstd)
        ops.embed_plan_join(ws, dev)
        if n_slabs > 1:
            for k in range(n_slabs):
                ops.embed_backward_slab_out(desc, tok, ids, None, E_tok, E_byte, lam, gout, out, rstd, gE_tok, gE_byte, g_lam,
                                            ws.buf, k, n_slabs, reserve_sms=bucket.reserve_sms if k > 0 else 0, plan_joined=True)
                if exchange:
                    lo, hi = ops.slab_rows(V_TOK, k, n_slabs)
                    bucket.exchange_async(lo * Dt, hi * Dt if k < n_slabs - 1 else bucket.flat.numel(), last=(k == n_slabs - 1))
            ws.clean = True
            if exchange:
                bucket.wait()
            return
        ops.embed_backward_out(desc, tok, ids, None, E_tok, E_byte, lam, gout, gE_tok, gE_byte, g_lam, ws.buf,
                               plan_ready=True, ws_clean=True, out_saved=out if rstd is not None else None, rstd=rstd,
                               plan_joined=True)
        ws.clean = True
        if world > 1 and exchange:
            bucket.mark_rows(desc, ws.buf)      # touched-rows exchange (no-op where the bucket does not offer it)
            bucket.all_reduce_avg()

    def step():
        compute_step(True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    lib = _lib.lib()
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()

    # ---- timed region: exactly K steps, device-timed, clocks sampled meanwhile ----
    K = args.steps
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    mot_b200.reset_launch_count()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        step()
    e1.record()
    barrier()
    launches = mot_b200.launch_count()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"out": out, "grad_embed_tokens": gE_tok, "grad_embed_bytes": gE_byte,
                                         **({"grad_lambdas": g_lam} if g_lam is not None else {})})
    ms_total = e0.elapsed_time(e1)
    t = torch.tensor([ms_total], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / K
    value = world * N / (ms_step * 1e-3)

    # ---- instrumented pass (same K steps again, clocks still sampled): the library records CUDA event pairs on the
    #      launch stream immediately around the main forward / backward kernel.  Kept out of the timed region above
    #      because an event between two launches disables their programmatic-dependent-launch overlap. ----
    fwd_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    bwd_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for a, b in fwd_ev + bwd_ev:  # materialise the cudaEvent_t handles
        a.record(); b.record()
    barrier()
    for i in range(K):
        lib.mot_profile_events(fwd_ev[i][0].cuda_event, fwd_ev[i][1].cuda_event, bwd_ev[i][0].cuda_event, bwd_ev[i][1].cuda_event)
        step()
    barrier()
    lib.mot_profile_events(None, None, None, None)
    clocks = sampler.stop() if rank == 0 else None
    fwd_ms = sum(a.elapsed_time(b) for a, b in fwd_ev) / K
    bwd_ms = sum(a.elapsed_time(b) for a, b in bwd_ev) / K

    # ---- N > 1: the exchange alone, the compute alone, and a value check of the exchanged bucket ----
    dp_info = None
    if world > 1:
        def timed(fn, reps):
            for _ in range(3):
                fn()
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                fn()
            b.record()
            barrier()
            t_ = torch.tensor([a.elapsed_time(b) / reps], device=dev)
            dist.all_reduce(t_, op=dist.ReduceOp.MAX)
            return float(t_.item())
        ar_ms = timed(bucket.all_reduce_avg, max(10, K // 4))                 # the whole bucket, one (dense) exchange
        ar_rows_ms = timed(lambda: (bucket.mark_rows(desc, ws.buf), bucket.all_reduce_avg()), max(10, K // 4)) \
            if bucket.sparse_rows else None                                   # bitmap + touched-rows exchange
        comp_ms = timed(lambda: compute_step(False), max(10, K // 4))         # fwd + bwd (slabs), no exchange
        nccl_buf = bucket.flat.clone()
        nccl_ms = timed(lambda: dist.all_reduce(nccl_buf, op=dist.ReduceOp.AVG), max(10, K // 4))
        # value check: one more step, then rank-local gradients averaged in fp32 by NCCL
        compute_step(False)
        torch.cuda.synchronize()
        want = bucket.flat.float()
        dist.all_reduce(want, op=dist.ReduceOp.SUM)
        want /= world
        step()
        torch.cuda.synchronize()
        err = float((bucket.flat.float() - want).abs().max() / want.abs().max().clamp_min(1e-30))
        errt = torch.tensor([err], device=dev)
        dist.all_reduce(errt, op=dist.ReduceOp.MAX)
        union_density = None
        if bucket.sparse_rows:
            rows_hit = ((bucket.bitmap[:, None] >> torch.arange(32, device=dev, dtype=torch.int32)) & 1).reshape(-1)[:V_TOK].contiguous()
            dist.all_reduce(rows_hit, op=dist.ReduceOp.MAX)        # NCCL has no bitwise OR: one int per row
            union_density = float(rows_hit.float().mean())
        dp_info = {"exchange": bucket.algo + (" (touched rows only)" if bucket.sparse_rows else ""), "rows_union_density": union_density,
                   "n_slabs": n_slabs, "reserve_sms": bucket.reserve_sms if n_slabs > 1 else 0,
                   "allreduce_ms": ar_ms, "touched_rows_allreduce_ms": ar_rows_ms, "nccl_allreduce_ms": nccl_ms, "compute_only_ms": comp_ms,
                   "bucket_mb": bucket.flat.numel() * esz / 1e6,
                   "allreduce_algbw_gbs": bucket.flat.numel() * esz / (ar_ms * 1e-3) / 1e9,
                   "exposed_exchange_ms": ms_step - comp_ms,
                   "kernel_only_tokens_per_sec": world * N / (comp_ms * 1e-3),
                   "bucket_max_rel_err_vs_fp32_nccl": float(errt.item()), "bucket_check": "ok" if float(errt.item()) <= 2.0 ** -7 else "FAILED"}
        if dp_info["bucket_check"] != "ok":
            print(f"bench: exchanged bucket differs from the fp32 NCCL reference by {float(errt.item()):.3e}", file=sys.stderr)

    # ---- e2e: module API, ids in pinned host memory, H2D every step, D2H of the byte-table gradient ----
    e2e = None
    if not args.no_e2e:
        mod = mot_b200.MoTEmbedding(V_TOK, V_BYTE, Dt, bd, bpt, variant=w["variant"]).to(dev).to(dt)
        with torch.no_grad():
            mod.embed_tokens.weight.copy_(E_tok); mod.embed_bytes.weight.copy_(E_byte)
        mod_bucket = mod.attach_grad_bucket()
        res_host = torch.empty(V_BYTE, bd, dtype=dt).pin_memory()
        # the caller's inputs are the token ids (what the reference's loader hands over, runs/7:468-474); the byte ids are
        # expanded from them on the device like runs/7:477-485 does (tokens_to_bytes through the ttb table, then the
        # `.view(bpt, -1)` of runs/71:479 for the sum variants).  Synthetic table: uniform ids, int16.
        ttb_tab = torch.randint(0, V_BYTE, (V_TOK, bpt), generator=gd, device=dev, dtype=torch.int32).to(torch.int16)

        def e2e_step():
            for p_ in mod.parameters():
                p_.grad = None
            t_in = tok_host.to(dev, non_blocking=True)
            b_in = mot_b200.ttb_expand(t_in, ttb_tab, out_dtype=torch.int32)
            b_in = b_in.view(bpt, -1) if slot_major else b_in
            x = mod(t_in, b_in)
            x.backward(gout.view_as(x))
            if world > 1:
                mod_bucket.all_reduce_avg()
            res_host.copy_(mod.embed_bytes.weight.grad, non_blocking=True)
            torch.cuda.current_stream().synchronize()   # the caller reads the result on the host every step

        for _ in range(max(3, args.warmup // 4)):
            e2e_step()
        barrier()
        # The same call through torch.cuda.make_graphed_callables (one CUDA graph for the forward incl. the byte-id
        # expansion and the sort plan, one for the backward): most of the eager step is host time (Python, autograd
        # engine, ctypes) around 92 us of kernels.  Used only if capture succeeds AND a replayed step reproduces the eager
        # gradients (within the bf16 bar: the fp32 accumulation order of duplicates differs run to run); otherwise the
        # eager call stays (MOT_E2E_EAGER=1 forces it).
        e2e_api = "eager"
        eager_mod = mod
        if world == 1 and not os.environ.get("MOT_E2E_EAGER"):
            try:
                class _Front(torch.nn.Module):
                    def __init__(self, emb):
                        super().__init__()
                        self.emb = emb

                    def forward(self, t_in):
                        if os.environ.get("MOT_E2E_FAIL") and torch.cuda.is_current_stream_capturing():
                            raise RuntimeError("injected failure inside the capture (fallback test)")
                        b_in = mot_b200.ttb_expand(t_in, ttb_tab, out_dtype=torch.int32)
                        return self.emb(t_in, b_in.view(bpt, -1) if slot_major else b_in)

                eager_ref = mod.embed_bytes.weight.grad.clone()
                eager_ref_t = mod.embed_tokens.weight.grad.clone()
                # a fresh module (no autograd state from the eager steps); gradients come back through autograd
                mod = mot_b200.MoTEmbedding(V_TOK, V_BYTE, Dt, bd, bpt, variant=w["variant"]).to(dev).to(dt)
                with torch.no_grad():
                    mod.embed_tokens.weight.copy_(E_tok); mod.embed_bytes.weight.copy_(E_byte)
                def rel(a, b):
                    return float((a.float() - b.float()).abs().max()) / max(float(b.float().abs().max()), 1e-30)

                def check_against_eager(what):
                    errs = (rel(mod.embed_tokens.weight.grad, eager_ref_t), rel(mod.embed_bytes.weight.grad, eager_ref))
                    # two bf16 results of fp32 sums taken in different orders may differ by one bf16 ulp (2^-7 of an element)
                    if not all(e <= 2.0 ** -6 for e in errs):     # also false for NaN
                        raise RuntimeError(f"{what} does not reproduce the eager gradients (normalised max-abs {errs})")

                front_mod = _Front(mod)
                whole = None
                if not os.environ.get("MOT_E2E_NO_WHOLE_GRAPH"):
                    # The whole step as ONE CUDA graph (PyTorch's "whole network capture"): H2D copy of the token ids from
                    # the pinned host buffer, byte-id expansion, forward, autograd backward, D2H read of the byte-table
                    # gradient.  The user's call is graph.replay() + a stream synchronize.
                    try:
                        t_static = torch.empty_like(tok)
                        side = torch.cuda.Stream(device=dev)
                        side.wait_stream(torch.cuda.current_stream(dev))
                        with torch.cuda.stream(side):            # warm-up on a side stream, as the capture recipe asks
                            for _ in range(3):
                                for p_ in mod.parameters():
                                    p_.grad = None
                                t_static.copy_(tok_host, non_blocking=True)
                                xw = front_mod(t_static)
                                xw.backward(gout.view_as(xw))
                        torch.cuda.current_stream(dev).wait_stream(side)
                        torch.cuda.synchronize()
                        for p_ in mod.parameters():
                            p_.grad = None                       # the capture allocates the gradients in the graph's pool
                        whole = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(whole):
                            t_static.copy_(tok_host, non_blocking=True)
                            xg = front_mod(t_static)
                            xg.backward(gout.view_as(xg))
                            res_host.copy_(mod.embed_bytes.weight.grad, non_blocking=True)

                        def e2e_step():   # noqa: F811
                            whole.replay()
                            torch.cuda.current_stream().synchronize()

                        e2e_step()
                        check_against_eager("the whole-step graph")
                        for _ in range(3):
                            e2e_step()
                        e2e_api = "one CUDA graph for the whole step (torch.cuda.graph around H2D + forward + backward + D2H)"
                    except Exception as e:  # noqa: BLE001
                        print(f"bench: whole-step graph unavailable ({type(e).__name__}: {e}); trying make_graphed_callables", file=sys.stderr)
                        whole = None
                        for p_ in mod.parameters():
                            p_.grad = None
                if whole is None:
                    front = torch.cuda.make_graphed_callables(front_mod, (tok.clone(),))

                    def e2e_step():   # noqa: F811
                        for p_ in mod.parameters():
                            p_.grad = None
                        x = front(tok_host.to(dev, non_blocking=True))
                        x.backward(gout.view_as(x))
                        res_host.copy_(mod.embed_bytes.weight.grad, non_blocking=True)
                        torch.cuda.current_stream().synchronize()

                    e2e_step()
                    check_against_eager("the graphed step")
                    for _ in range(3):
                        e2e_step()
                    e2e_api = "cuda-graphed (torch.cuda.make_graphed_callables)"
            except Exception as e:  # noqa: BLE001 - any capture problem: keep the eager call
                print(f"bench: graphed e2e unavailable ({type(e).__name__}: {e}); eager call kept", file=sys.stderr)
                e2e_api = "eager"
                mod = eager_mod

                def e2e_step():   # noqa: F811
                    for p_ in mod.parameters():
                        p_.grad = None
                    t_in = tok_host.to(dev, non_blocking=True)
                    b_in = mot_b200.ttb_expand(t_in, ttb_tab, out_dtype=torch.int32)
                    x = mod(t_in, b_in.view(bpt, -1) if slot_major else b_in)
                    x.backward(gout.view_as(x))
                    res_host.copy_(mod.embed_bytes.weight.grad, non_blocking=True)
                    torch.cuda.current_stream().synchronize()
                for _ in range(3):
                    e2e_step()
        barrier()
        Ke = max(10, K // 4)
        t0 = time.perf_counter()
        for _ in range(Ke):
            e2e_step()
        barrier()
        t_e = torch.tensor([(time.perf_counter() - t0) / Ke], device=dev)
        if world > 1:
            dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
        e2e = {"value": world * N / float(t_e.item()), "unit": "tokens/s",
               "h2d_bytes_per_step": tok_host.numel() * 4,
               "d2h_bytes_per_step": res_host.numel() * esz, "ms_per_step": float(t_e.item()) * 1e3,
               "api": "token ids from pinned host memory -> mot_b200.ttb_expand -> MoTEmbedding.forward + autograd backward "
                      "-> byte-table gradient read back; " + e2e_api, "steps": Ke}

    if rank == 0:
        peak, peak_src = measured_peaks()
        dom_bytes, dom_ms, dom = (A_bwd, bwd_ms, "mot_bwd_sum_kernel" if rstd is not None else "mot_bwd_kernel") if bwd_ms >= fwd_ms else (A_fwd, fwd_ms, "mot_fwd_kernel")
        achieved = dom_bytes / (dom_ms * 1e-3) / 1e9
        line = {
            "metric": "byte-mix embedding fwd+bwd tokens/sec", "value": value, "unit": "tokens/s", "n_gpus": world,
            "steps": K, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": w["dtype"], "data": "synthetic",
            "config": main_config(w, args, world),
            "exchange": (f"{bucket.algo}" + (f", {n_slabs} vocabulary slabs beside the backward" if n_slabs > 1 else ", after the backward")) if world > 1 else None,
            "tokens_per_sec_per_gpu": value / world,
            "kernel_ms": {"fwd": fwd_ms, "bwd_main": bwd_ms},
            "step_hbm_gbs": (A_fwd + A_bwd) / (ms_step * 1e-3) / 1e9,
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "frac_of_8TBs_spec": achieved / 8000.0,
                         "traffic": measured_traffic(w["name"], dom),
                         "algorithmic_bytes_per_launch": dom_bytes, "kernel_ms": dom_ms, "peak_source": peak_src,
                         "timing": "CUDA event pairs around the kernel on its launch stream, averaged over a second "
                                   "pass of the same K steps (events between launches would disable PDL overlap in the timed region)",
                         "fwd": {"achieved": A_fwd / (fwd_ms * 1e-3) / 1e9, "bytes": A_fwd, "ms": fwd_ms},
                         "bwd": {"achieved": A_bwd / (bwd_ms * 1e-3) / 1e9, "bytes": A_bwd, "ms": bwd_ms}},
            "gpu_launches": int(launches), "clocks": clocks,
        }
        if e2e is not None:
            line["e2e"] = e2e
        if dp_info is not None:
            line["dp"] = dp_info
        if world == 1 and not args.no_torch_gpu:
            line["torch_gpu"] = time_torch_gpu(w, dev)
        if world == 1 and not args.no_cpu_baseline:
            r = time_cpu_reference(w, steps=50, warmup=2, budget_s=20.0)
            line["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------
# GPU arm, concat + dense projection workloads (tensor-core bound)
# ----------------------------------------------------------------------------------------------
def run_proj(args):
    import torch.distributed as dist
    import mot_b200
    from mot_b200 import ops, dp

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group(backend="nccl", device_id=dev)
    w = workload_config(args)
    N, Dt, bd, bpt, Do = w["N"], w["Dt"], w["bd"], w["bpt"], w["Do"]
    K = Dt + bpt * bd
    dt = torch.bfloat16
    g = torch.Generator(device=dev).manual_seed(12345)
    E_tok = torch.randn(V_TOK, Dt, generator=g, device=dev).to(dt)
    E_byte = torch.randn(V_BYTE, bd, generator=g, device=dev).to(dt)
    W = ((torch.rand(Do, K, generator=g, device=dev) * 2 - 1) * (3 ** 0.5) * 0.5 * K ** -0.5).to(dt)
    gd = torch.Generator(device=dev).manual_seed(12345 + 1000 * (rank + 1))
    tok_host = make_tokens(N, args.dist, 12345 + rank).pin_memory()
    tok = tok_host.to(dev)
    ids = torch.randint(0, V_BYTE, (1, N * bpt), generator=gd, device=dev, dtype=torch.int32)
    ids_host = ids.cpu().pin_memory()
    gout = torch.randn(N, Do, generator=gd, device=dev).to(dt)
    pair = bool(w.get("pair"))
    if pair:   # spt ids are int64 [B, S*bpt]; the token columns come from a tok-only launch over strided rows
        ids = ids.long()
        ids2 = torch.randint(0, V_BYTE, (1, N * bpt), generator=gd, device=dev)
        ids_host, ids2_host = ids.cpu().pin_memory(), ids2.cpu().pin_memory()
        spec = mot_b200.MixSpec(combine="tok_only", tok_norm=True, out_norm=False)
        desc = ops.make_desc(spec, N, E_tok, None, 0, ids=None, ttb=None, has_lam=False, row_stride=K, col_offset=0)
    else:
        spec = mot_b200.MixSpec(combine="concat", tok_norm=True, byte_norm=True, out_norm=False)   # the [tok | bytes] operand
        desc = ops.make_desc(spec, N, E_tok, E_byte, bpt, ids=ids, ttb=None, has_lam=False)
    ws = ops.acquire_workspace(desc, dev)

    def gather_A():
        if pair:
            ops.embed_forward_out(desc, tok, None, None, E_tok, None, None, A)
            ops.byte_pair_forward_out(ids, ids2, bpt, E_byte, A, Dt)
        else:
            ops.embed_forward_out(desc, tok, ids, None, E_tok, E_byte, None, A)

    def scatter_dA():
        if pair:
            ops.embed_backward_out(desc, tok, None, None, E_tok, None, None, dA, gE_tok, None, None, ws.buf,
                                   plan_ready=True, ws_clean=True)
            ops.byte_pair_backward_out(ids, ids2, bpt, E_byte, dA, Dt, gE_byte)
        else:
            ops.embed_backward_out(desc, tok, ids, None, E_tok, E_byte, None, dA, gE_tok, gE_byte, None, ws.buf,
                                   plan_ready=True, ws_clean=True)
    A = torch.empty(N, K, dtype=dt, device=dev)
    dA = torch.empty(N, K, dtype=dt, device=dev)
    Y, out, dY = (torch.empty(N, Do, dtype=dt, device=dev) for _ in range(3))
    dW32 = torch.empty(Do, K, dtype=torch.float32, device=dev)
    bucket = dp.GradBucket([torch.nn.Parameter(E_tok, requires_grad=False), torch.nn.Parameter(E_byte, requires_grad=False),
                            torch.nn.Parameter(W, requires_grad=False)])
    gE_tok, gE_byte, gW = bucket.views()
    ev = {k: [] for k in ("fwd", "dx", "dw")}

    def timed(key, fn, record):
        if not record:
            return fn()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        ev[key].append((a, b))

    def step(record=False):
        # forward: fused gather of [tok | bytes] -> tcgen05 projection -> rms_norm   (runs/7:317-319,233-234)
        ops.embed_plan_async(desc, tok, ws, dev)
        gather_A()
        timed("fwd", lambda: ops.linear_forward_out(A, W, Y), record)
        ops.rmsnorm_forward_out(Y, out)
        # backward: norm bwd -> dW, dX on the tensor cores -> fused scatter into the dense table gradients
        ops.rmsnorm_backward_out(Y, gout, dY)
        # the [N, K] operand of the forward is kept (like mot_b200.mot_embed_proj; MOT_PROJ_REGATHER=1 gathers it again)
        if os.environ.get("MOT_PROJ_REGATHER"):
            gather_A()
        timed("dw", lambda: ops.linear_bwd_weight_out(dY, A, dW32, gW), record)
        timed("dx", lambda: ops.linear_bwd_input_out(dY, W, dA), record)
        ops.embed_plan_join(ws, dev)
        scatter_dA()
        ws.clean = True
        if world > 1:
            bucket.all_reduce_avg()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    K_steps = args.steps
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start(); time.sleep(0.3)
    mot_b200.reset_launch_count()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K_steps):
        step()
    e1.record()
    barrier()
    launches = mot_b200.launch_count()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"out": out, "grad_embed_tokens": gE_tok, "grad_embed_bytes": gE_byte, "grad_proj": gW})
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / K_steps
    value = world * N / (ms_step * 1e-3)
    for _ in range(K_steps):       # instrumented pass: events around the three GEMM calls
        step(record=True)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    gemm_ms = {k: sum(a.elapsed_time(b) for a, b in v) / len(v) for k, v in ev.items()}

    e2e = None
    if not args.no_e2e:
        if pair:
            mod = mot_b200.SptByteMixEmbedding(V_TOK, V_BYTE, Dt, bd, Do, bpt, pull_in=True, add_padded_and_pulled=True).to(dev)
            mod.embed.bfloat16()
            mod.embed_bytes = mod.embed.embed_bytes
        else:
            mod = mot_b200.MoTProjEmbedding(V_TOK, V_BYTE, Dt, bd, Do, bpt, variant="V1").to(dev).to(dt)
        res_host = torch.empty(V_BYTE, bd, dtype=dt).pin_memory()

        def e2e_step():
            for p_ in mod.parameters():
                p_.grad = None
            if pair:
                x = mod(tok_host.to(dev, non_blocking=True).view(64, -1), ids_host.to(dev, non_blocking=True).view(64, -1),
                        ids2_host.to(dev, non_blocking=True).view(64, -1))
            else:
                x = mod(tok_host.to(dev, non_blocking=True), ids_host.to(dev, non_blocking=True))
            x.backward(gout.view_as(x))
            if world > 1:
                for p_ in mod.parameters():
                    dist.all_reduce(p_.grad, op=dist.ReduceOp.AVG)
            res_host.copy_(mod.embed_bytes.weight.grad, non_blocking=True)
            torch.cuda.current_stream().synchronize()

        for _ in range(3):
            e2e_step()
        barrier()
        Ke = max(10, K_steps // 4)
        t0 = time.perf_counter()
        for _ in range(Ke):
            e2e_step()
        barrier()
        t_e = torch.tensor([(time.perf_counter() - t0) / Ke], device=dev)
        if world > 1:
            dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
        e2e = {"value": world * N / float(t_e.item()), "unit": "tokens/s",
               "h2d_bytes_per_step": tok_host.numel() * 4 + ids_host.numel() * ids_host.element_size() * (2 if pair else 1),
               "d2h_bytes_per_step": res_host.numel() * 2, "ms_per_step": float(t_e.item()) * 1e3,
               "api": ("mot_b200.SptByteMixEmbedding(add_padded_and_pulled=True)" if pair else "mot_b200.MoTProjEmbedding") +
                      ".forward + autograd backward", "steps": Ke}

    if rank == 0:
        peak, peak_src = measured_tensor_peak()
        flops = 2.0 * N * K * Do
        tot_ms = sum(gemm_ms.values())
        achieved = 3 * flops / (tot_ms * 1e-3) / 1e12
        line = {
            "metric": "byte-mix embedding fwd+bwd tokens/sec", "value": value, "unit": "tokens/s", "n_gpus": world,
            "steps": K_steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": w["name"],
                       "variant": ("V1b padded+pulled byte rows summed before the norm (spt/train_gpt.py:371-379,439-443)" if pair
                                   else "V1 concat+projection (runs/7:226-234,317-319)"),
                       "tokens_per_gpu_per_step": N, "token_dim": Dt, "byte_dim": bd, "bytes_per_token": bpt, "in_dim": K,
                       "out_dim": Do, "token_dist": args.dist, "l2": "working set > 126 MB L2, no flush",
                       "parallelism": f"dp{world}" + (", one flat-bucket NCCL all-reduce(AVG) per step" if world > 1 else "")},
            "tokens_per_sec_per_gpu": value / world,
            "kernel_ms": {"linear_fwd": gemm_ms["fwd"], "linear_bwd_input": gemm_ms["dx"], "linear_bwd_weight": gemm_ms["dw"]},
            "roofline": {"bound": "tensor", "kernel": "mot_gemm_kernel (fwd + dX + dW)", "achieved": achieved, "peak": peak,
                         "unit": "TFLOP/s", "frac": achieved / peak, "traffic": None, "flops_per_launch": flops,
                         "peak_source": peak_src,
                         "per_kernel_tflops": {k: flops / (v * 1e-3) / 1e12 for k, v in gemm_ms.items()},
                         "timing": "CUDA event pairs around each projection call in a second pass of the same K steps"},
            "gpu_launches": int(launches), "clocks": clocks,
        }
        if e2e is not None:
            line["e2e"] = e2e
        if world == 1 and not args.no_cpu_baseline:
            r = time_cpu_reference(w, steps=20, warmup=1, budget_s=15.0)
            line["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_value_embeds(args):
    """SURVEY 8(f)-2: `ve = [value_embed(token_inputs) for value_embed in self.value_embeds]` (runs/7:252,308) forward and
    the three dense gradient scatters, one token sort shared by all tables.  HBM bound."""
    import mot_b200
    from mot_b200 import ops, _lib
    if int(os.environ.get("WORLD_SIZE", "1")) != 1:
        raise SystemExit("bench.py: the value-embeds workload is a single-GPU kernel measurement")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    w = workload_config(args)
    N, D, T = w["N"], w["Dt"], w["tables"]
    dt = torch.bfloat16
    g = torch.Generator(device=dev).manual_seed(12345)
    tables = [torch.randn(V_TOK, D, generator=g, device=dev).to(dt) for _ in range(T)]
    gouts = [torch.randn(N, D, generator=g, device=dev).to(dt) for _ in range(T)]
    tok_host = make_tokens(N, args.dist, 12345).pin_memory()
    tok = tok_host.to(dev)
    outs = [torch.empty(N, D, dtype=dt, device=dev) for _ in range(T)]
    grads = [torch.empty_like(E) for E in tables]
    desc = ops.make_desc(mot_b200.MixSpec(combine="tok_only", out_norm=False), N, tables[0], None, 0, ids=None, ttb=None, has_lam=False)
    ws = ops.acquire_workspace(desc, dev)

    def step():
        ops.embed_plan_async(desc, tok, ws, dev)
        for E, o in zip(tables, outs):
            ops.embed_forward_out(desc, tok, None, None, E, None, None, o)
        ops.embed_plan_join(ws, dev)
        for E, go, gE in zip(tables, gouts, grads):
            ops.embed_backward_out(desc, tok, None, None, E, None, None, go, gE, None, None, ws.buf, plan_ready=True, ws_clean=True)
        ws.clean = True

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    K = args.steps
    sampler = ClockSampler(0)
    sampler.start(); time.sleep(0.3)
    mot_b200.reset_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        step()
    e1.record()
    torch.cuda.synchronize()
    launches = mot_b200.launch_count()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {**{f"out_{i}": o for i, o in enumerate(outs)},
                                         **{f"grad_value_embeds_{i}": gE for i, gE in enumerate(grads)}})
    ms_step = e0.elapsed_time(e1) / K
    # instrumented pass: event pairs around the main backward kernel of every scatter (3 per step -> the last one wins;
    # use one step per pair)
    lib = _lib.lib()
    bwd_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for a, b in bwd_ev:
        a.record(); b.record()
    torch.cuda.synchronize()
    for i in range(K):
        ops.embed_plan_async(desc, tok, ws, dev)
        ops.embed_plan_join(ws, dev)
        lib.mot_profile_events(None, None, bwd_ev[i][0].cuda_event, bwd_ev[i][1].cuda_event)
        ops.embed_backward_out(desc, tok, None, None, tables[0], None, None, gouts[0], grads[0], None, None, ws.buf,
                               plan_ready=True, ws_clean=True)
        lib.mot_profile_events(None, None, None, None)
    torch.cuda.synchronize()
    clocks = sampler.stop()
    bwd_ms = sum(a.elapsed_time(b) for a, b in bwd_ev) / K
    e = 2
    A_bwd1 = N * (D * e + 8) + V_TOK * D * e          # one table: upstream rows + sorted stream in, dense gradient out (R = 0)
    A_step = T * (N * (4 + 2 * D * e) + A_bwd1)       # forward: ids + table row in, row out
    mod = mot_b200.TokenValueEmbeddings(V_TOK, D, T).to(dev).to(dt)
    res_host = torch.empty(16, D, dtype=dt).pin_memory()

    def e2e_step():
        for p_ in mod.parameters():
            p_.grad = None
        ve = mod(tok_host.to(dev, non_blocking=True))
        torch.autograd.backward(ve, gouts)
        res_host.copy_(mod.value_embeds[0].weight.grad[:16], non_blocking=True)
        torch.cuda.current_stream().synchronize()

    for _ in range(3):
        e2e_step()
    Ke = max(10, K // 4)
    t0 = time.perf_counter()
    for _ in range(Ke):
        e2e_step()
    t_e = (time.perf_counter() - t0) / Ke
    peak, peak_src = measured_peaks()
    line = {"metric": "byte-mix embedding fwd+bwd tokens/sec", "value": N / (ms_step * 1e-3), "unit": "tokens/s", "n_gpus": 1,
            "steps": K, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": w["name"], "variant": "value embeddings: 3 plain gathers sharing the token ids (runs/7:252,308)",
                       "tokens_per_gpu_per_step": N, "tables": T, "dim": D, "token_dist": args.dist,
                       "l2": "working set > 126 MB L2, no flush", "parallelism": "dp1"},
            "step_hbm_gbs": A_step / (ms_step * 1e-3) / 1e9,
            "roofline": {"bound": "hbm", "kernel": "mot_bwd_kernel (plain gather: no token rows)", "achieved": A_bwd1 / (bwd_ms * 1e-3) / 1e9,
                         "peak": peak, "unit": "GB/s", "frac": A_bwd1 / (bwd_ms * 1e-3) / 1e9 / peak, "traffic": None,
                         "algorithmic_bytes_per_launch": A_bwd1, "kernel_ms": bwd_ms, "peak_source": peak_src},
            "gpu_launches": int(launches), "clocks": clocks,
            "e2e": {"value": N / t_e, "unit": "tokens/s", "h2d_bytes_per_step": tok_host.numel() * 4,
                    "d2h_bytes_per_step": res_host.numel() * 2, "ms_per_step": t_e * 1e3,
                    "api": "mot_b200.TokenValueEmbeddings.forward + autograd backward", "steps": Ke}}
    print(json.dumps(line), flush=True)


def run_mathblations(args):
    """Config 2: the whole module step (digits expansion + fused gather + TF32 projection, forward and backward)."""
    import mot_b200
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        raise SystemExit("mathblations-concat is a 1-GPU configuration (BASELINE.json configs[1])")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    w = workload_config(args)
    B, S, dpt, V = 1024, 11, w["bpt"], 10003
    g = torch.Generator().manual_seed(12345)
    idx_host = torch.randint(0, 10000, (B, S), generator=g)
    idx_host[torch.rand(B, S, generator=g) < 0.2] = 10000
    idx_host = idx_host.pin_memory()
    torch.manual_seed(12345)     # the module's initial weights and gout: the same inputs on every run
    m = mot_b200.DigitMixinEmbedding(V, w["Dt"], w["bd"], dpt).to(dev)
    gout = torch.randn(B, S, w["Do"], device=dev)
    res_host = torch.empty(14, w["bd"]).pin_memory()
    idx = idx_host.to(dev)

    def step(e2e=False):
        for p_ in m.parameters():
            p_.grad = None
        t = idx_host.to(dev, non_blocking=True) if e2e else idx
        digits = mot_b200.tokens_to_digits(t, dpt, 10000, 10001, 10002).view(B, S * dpt)
        y = m(t, digits)
        y.backward(gout)
        if e2e:
            res_host.copy_(m.dte.weight.grad, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        return y

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    sampler = ClockSampler(0); sampler.start(); time.sleep(0.3)
    mot_b200.reset_launch_count()
    K = args.steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        y = step()
    e1.record(); torch.cuda.synchronize()
    launches = mot_b200.launch_count()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"out": y, **{"grad_" + n.replace(".", "_"): p_.grad for n, p_ in m.named_parameters()}})
    ms_step = e0.elapsed_time(e1) / K
    t0 = time.perf_counter()
    for _ in range(K):
        step(e2e=True)
    t_e = (time.perf_counter() - t0) / K
    clocks = sampler.stop()
    N, Kd, Do = w["N"], w["Dt"] + dpt * w["bd"], w["Do"]
    peak, peak_src = measured_tensor_peak()
    flops = 6.0 * N * Kd * Do
    line = {"metric": "byte-mix embedding fwd+bwd tokens/sec", "value": N / (ms_step * 1e-3), "unit": "tokens/s", "n_gpus": 1,
            "steps": K, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 (tf32 tensor cores)", "data": "synthetic",
            "config": {"workload": w["name"], "variant": "V8 digits concat + linear with bias (mathblations/model.py:256-268)",
                       "batch": B, "seq": S, "digits_per_token": dpt, "n_embd_tok": w["Dt"], "n_embd_digit": w["bd"],
                       "l2": "working set fits L2: launch-latency bound configuration, reported as us/step", "parallelism": "dp1"},
            "us_per_step": ms_step * 1e3,
            "roofline": {"bound": "tensor", "kernel": "mot_gemm_kernel<float> (fwd + dX + dW)", "achieved": flops / (ms_step * 1e-3) / 1e12,
                         "peak": peak, "unit": "TFLOP/s", "frac": flops / (ms_step * 1e-3) / 1e12 / peak, "traffic": None,
                         "peak_source": peak_src + "; whole-step time: the step is launch-latency bound, not tensor bound"},
            "gpu_launches": int(launches), "clocks": clocks,
            "e2e": {"value": N / t_e, "unit": "tokens/s", "h2d_bytes_per_step": idx_host.numel() * 8,
                    "d2h_bytes_per_step": res_host.numel() * 4, "ms_per_step": t_e * 1e3,
                    "api": "mot_b200.tokens_to_digits + DigitMixinEmbedding.forward + autograd backward", "steps": K}}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    elif a.impl == "torch-gpu":
        run_torch_gpu(a)
    elif WORKLOADS[a.workload]["variant"] == "V1":
        run_proj(a)
    elif WORKLOADS[a.workload]["variant"] == "V8":
        run_mathblations(a)
    elif WORKLOADS[a.workload]["variant"] == "VE":
        run_value_embeds(a)
    else:
        run_ours(a)
