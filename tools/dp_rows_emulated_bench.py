"""Touched-rows exchange kernel with the ranks emulated on ONE GPU (every rank's copy is a buffer of the same device, one
stream per rank, 8 CTAs per rank so that all of them are resident and meet at the barriers):

    python tools/dp_rows_emulated_bench.py OLD_LIB.so NEW_LIB.so

* the one-table call (mot_dp_exchange_rows, 50257 x 768 bf16 + a dense tail) of two builds of the library, alternated;
* the four-table call of NEW (mot_dp_exchange_rows_multi, [256 | 3 x 768]) against four one-table calls.
Uniform-like bitmaps (62 % of the rows per rank).  The copies are in HBM, so this times the kernel's own work, not
NVLink: it compares builds and call shapes, it does not predict a multi-GPU step."""
import ctypes as C
import json
import os
import subprocess
import sys
import time

import torch
DEV = torch.device("cuda", 0)
P = C.c_void_p
def load(path):
    L = C.CDLL(path)
    L.mot_dp_exchange_rows.argtypes = [P, P, P, P, C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_int64, C.c_int64,
                                       C.c_int64, C.c_int32, C.c_uint32, C.c_int32, P]
    return L
class T(C.Structure):
    _fields_ = [("byte_offset", C.c_int64), ("row_bytes", C.c_int32), ("reserved", C.c_int32)]
def setup(world, V, widths, dense, density, seed=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    offs, n = [], 0
    for w in widths:
        offs.append(n); n += V * w
    dlo = n; n += dense
    words = (V + 31) // 32
    bm_off = n * 2
    total = n + (words * 4 + 15) // 16 * 8
    bits = torch.rand(world, V, generator=g, device=DEV) < density
    bufs = []
    for r in range(world):
        b = torch.zeros(total, dtype=torch.bfloat16, device=DEV)
        for o, w in zip(offs, widths):
            b[o:o + V * w].view(V, w).copy_(torch.randn(V, w, generator=g, device=DEV).bfloat16().masked_fill(~bits[r, :, None], 0.0))
        wv = torch.zeros(words * 32, dtype=torch.int64, device=DEV); wv[:V] = bits[r].long()
        packed = (wv.view(words, 32) << torch.arange(32, device=DEV)).sum(1)
        b.view(torch.uint8)[bm_off:bm_off + 4 * words].copy_(packed.bitwise_and(0xFFFFFFFF).to(torch.int32).view(torch.uint8))
        bufs.append(b)
    st = dict(bufs=bufs, offs=offs, dlo=dlo, dense=dense, bm_off=bm_off, widths=widths, V=V, world=world,
              union=float(bits.any(0).float().mean()))
    st["peers"] = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device=DEV)
    st["pads_mem"] = [torch.zeros(9216 // 4, dtype=torch.int32, device=DEV) for _ in range(world)]
    st["pads"] = torch.tensor([p.data_ptr() for p in st["pads_mem"]], dtype=torch.int64, device=DEV)
    st["works"] = [torch.zeros(64, dtype=torch.int32, device=DEV) for _ in range(world)]
    st["streams"] = [torch.cuda.Stream(device=DEV) for _ in range(world)]
    st["epoch"] = 1
    return st
def run_one(L, st, k):
    """one-table exchange of table k, dense tail only with the last table"""
    for r in reversed(range(st["world"])):
        last = k == len(st["widths"]) - 1
        rc = L.mot_dp_exchange_rows(None, st["peers"].data_ptr(), st["pads"].data_ptr(), st["works"][r].data_ptr(), r, st["world"],
                                    st["offs"][k] * 2, st["V"], st["widths"][k] * 2, st["bm_off"], st["dlo"] * 2,
                                    st["dense"] * 2 if last else 0, 0, st["epoch"], 1, st["streams"][r].cuda_stream)
        assert rc == 0, rc
    st["epoch"] += 2
def run_multi(L, st):
    tabs = (T * len(st["widths"]))(*[T(o * 2, w * 2, 0) for o, w in zip(st["offs"], st["widths"])])
    for r in reversed(range(st["world"])):
        rc = L.mot_dp_exchange_rows_multi(None, P(st["peers"].data_ptr()), P(st["pads"].data_ptr()), P(st["works"][r].data_ptr()),
                                          r, st["world"], tabs, len(st["widths"]), st["V"], C.c_int64(st["bm_off"]),
                                          C.c_int64(st["dlo"] * 2), C.c_int64(st["dense"] * 2), 0, C.c_uint32(st["epoch"]), 1,
                                          P(st["streams"][r].cuda_stream))
        assert rc == 0, rc
    st["epoch"] += 2
def timed(fn, iters=50):
    for _ in range(5): fn()
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(iters): fn()
    torch.cuda.synchronize(); return (time.perf_counter() - t0) / iters * 1e6
os.environ["MOT_AR_BLOCKS"] = "8"     # all ranks' CTAs resident together on the one GPU
old, new = load(sys.argv[1]), load(sys.argv[2])
new.mot_dp_exchange_rows_multi.restype = C.c_int
pl = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
print("#", torch.cuda.get_device_name(), f"power limit {pl} - ranks emulated on one GPU, 8 CTAs per rank: HBM, not NVLink")
for world in (2, 4):
    st = setup(world, 50257, [768], 458 * 48, 0.62)
    res = {"parent": [], "new": []}
    for rnd in range(5):
        res["parent"].append(timed(lambda: run_one(old, st, 0)))
        res["new"].append(timed(lambda: run_one(new, st, 0)))
    print(json.dumps({"world": world, "case": "one table 50257x768 bf16 + 458x48 dense", "union": st["union"],
                      "parent_us": [round(x, 1) for x in res["parent"]], "new_us": [round(x, 1) for x in res["new"]]}))
    del st
    st = setup(world, 50257, [256, 768, 768, 768], 458 * 16, 0.62)
    m, s = [], []
    for rnd in range(5):
        m.append(timed(lambda: run_multi(new, st), 20))
        s.append(timed(lambda: [run_one(new, st, k) for k in range(4)], 20))
    print(json.dumps({"world": world, "case": "4 tables 256+3x768 bf16: one multi call vs four one-table calls", "union": st["union"],
                      "multi_us": [round(x, 1) for x in m], "four_calls_us": [round(x, 1) for x in s]}))
    del st
