"""The peer-to-peer touched-rows exchange over several row tables, on ONE GPU: 2 and 4 ranks emulated in one process.

Each "rank" is an ordinary device buffer of the same GPU; the peer-pointer array lists all of them, every rank has its
own signal pad and work area, and the ranks' kernels run on separate streams (8 CTAs each, so that all of them are
resident together and meet at the barriers).  The kernel cannot tell this from peers over NVLink, so this checks its
arithmetic on any box: the multi-GPU test (tests/test_gpu_dp_rows.py) needs 2+ GPUs and skips below that.

Bucket: [table 0: 256 wide | tables 1-3: 768 wide | dense tail | bitmap], bf16 and fp32.  Each rank's rows are nonzero
exactly where its bitmap bit is set (the precondition of the exchange).  Expected, bit for bit: rows of the union and the
dense tail = the fp32 sum in rank order times 1/world, rounded to the bucket dtype; every other row untouched; every
rank's copy the same.  The one-table entry point is checked the same way."""
import ctypes as C
import os

import pytest
import torch

from mot_b200 import _lib as L

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)


def _expected(copies, world):
    acc = torch.zeros_like(copies[0], dtype=torch.float32)
    for c in copies:
        acc += c.float()
    return (acc * (1.0 / world)).to(copies[0].dtype)


def _run(world, dtype, widths, n_rows=5000, dense=4096, seed=0, one_table_call=False):
    g = torch.Generator(device=DEV).manual_seed(seed)
    esz = torch.empty(0, dtype=dtype).element_size()
    offs, n = [], 0
    for w in widths:
        offs.append(n)
        n += n_rows * w
    dense_lo = n
    n += dense
    bm_words = (n_rows + 31) // 32
    bm_off = n * esz
    total = n + (bm_words * 4 + 15) // 16 * 16 // esz
    bits = torch.rand(world, n_rows, generator=g, device=DEV) < 0.3
    bits[:, : n_rows // 7] = False                             # rows nobody gathered
    bufs = []
    for r in range(world):
        b = torch.zeros(total, dtype=dtype, device=DEV)
        for o, w in zip(offs, widths):
            t = b[o:o + n_rows * w].view(n_rows, w)
            t.copy_(torch.randn(n_rows, w, generator=g, device=DEV).to(dtype).masked_fill(~bits[r, :, None], 0.0))
        b[dense_lo:dense_lo + dense].copy_(torch.randn(dense, generator=g, device=DEV).to(dtype))
        words = torch.zeros(bm_words * 32, dtype=torch.int64, device=DEV)
        words[:n_rows] = bits[r].long()
        packed = (words.view(bm_words, 32) << torch.arange(32, device=DEV)).sum(1)
        b.view(torch.uint8)[bm_off:bm_off + 4 * bm_words].copy_(
            packed.to(torch.int64).bitwise_and(0xFFFFFFFF).to(torch.int32).view(torch.uint8))
        bufs.append(b)
    want = _expected([b[:n] for b in bufs], world)
    union = bits.any(0)
    for o, w in zip(offs, widths):                                 # rows outside the union are not touched
        t = want[o:o + n_rows * w].view(n_rows, w)
        t[~union] = bufs[0][o:o + n_rows * w].view(n_rows, w)[~union]
    peers = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device=DEV)
    pads_mem = [torch.zeros(9216 // 4, dtype=torch.int32, device=DEV) for _ in range(world)]
    pads = torch.tensor([p.data_ptr() for p in pads_mem], dtype=torch.int64, device=DEV)
    works = [torch.zeros(64, dtype=torch.int32, device=DEV) for _ in range(world)]
    streams = [torch.cuda.Stream(device=DEV) for _ in range(world)]
    tables = (L.MotRowTable * len(widths))(*[L.MotRowTable(o * esz, w * esz, 0) for o, w in zip(offs, widths)])
    dt = L.BF16 if dtype == torch.bfloat16 else L.F32
    torch.cuda.synchronize()
    os.environ["MOT_AR_BLOCKS"] = "8"
    try:
        for r in reversed(range(world)):
            if one_table_call:
                rc = L.lib().mot_dp_exchange_rows(None, C.c_void_p(peers.data_ptr()), C.c_void_p(pads.data_ptr()),
                                                  C.c_void_p(works[r].data_ptr()), r, world, 0, n_rows, widths[0] * esz,
                                                  bm_off, dense_lo * esz, dense * esz, dt, 1, L.DP_P2P,
                                                  C.c_void_p(streams[r].cuda_stream))
            else:
                rc = L.lib().mot_dp_exchange_rows_multi(None, C.c_void_p(peers.data_ptr()), C.c_void_p(pads.data_ptr()),
                                                        C.c_void_p(works[r].data_ptr()), r, world, tables, len(widths),
                                                        n_rows, bm_off, dense_lo * esz, dense * esz, dt, 1, L.DP_P2P,
                                                        C.c_void_p(streams[r].cuda_stream))
            assert rc == L.OK, L.lib().mot_strerror(rc)
    finally:
        del os.environ["MOT_AR_BLOCKS"]
    torch.cuda.synchronize()
    return bufs, want, n, union


@pytest.mark.parametrize("world", [2, 4])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_multi_table_rows_exchange_two_widths(world, dtype):
    bufs, want, n, union = _run(world, dtype, [256, 768, 768, 768])
    assert bool(union.any()) and not bool(union.all())
    for r, b in enumerate(bufs):
        assert torch.equal(b[:n].view(torch.uint8), want.view(torch.uint8)), f"rank {r}"


@pytest.mark.parametrize("world", [2, 4])
def test_one_table_call_is_the_same_kernel(world):
    bufs, want, n, _ = _run(world, torch.bfloat16, [1024], seed=1, one_table_call=True)
    for r, b in enumerate(bufs):
        assert torch.equal(b[:n].view(torch.uint8), want.view(torch.uint8)), f"rank {r}"
