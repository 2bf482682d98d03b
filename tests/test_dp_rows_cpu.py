"""CPU checks of the touched-rows exchange over several row tables: the argument checks of mot_dp_exchange_rows_multi
(all returned before any CUDA call) and the layout of a GradBucket whose first k parameters are row tables, in one
process and over gloo at world 2."""
import ctypes as C
import os
import socket
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "mixture-of-tokenizers_b200"))

from mot_b200 import _lib as L  # noqa: E402
from mot_b200 import dp  # noqa: E402

V = 1000                     # rows of every table; bitmap = 32 words
FAKE = C.c_void_p(4096)      # never dereferenced: every call below fails its checks first


def _tables(*specs):
    """(byte offset, row bytes[, reserved]) per table -> a host array of MotRowTable"""
    return (L.MotRowTable * len(specs))(*[L.MotRowTable(*s) if len(s) == 3 else L.MotRowTable(*s, 0) for s in specs])


def _call(tables, n_tables, n_rows=V, bm=None, dense_lo=None, dense_bytes=0, rank=0, world=2, dtype=L.BF16,
          algo=L.DP_P2P, pads=FAKE, work=FAKE, mc=FAKE, peers=FAKE):
    bm = 16 << 20 if bm is None else bm
    dense_lo = 32 << 20 if dense_lo is None else dense_lo
    return L.lib().mot_dp_exchange_rows_multi(mc, peers, pads, work, rank, world, tables, n_tables, n_rows, bm, dense_lo,
                                              dense_bytes, dtype, 1, algo, None)


def test_exchange_rows_multi_error_codes_without_a_device():
    two = _tables((0, 512), (V * 512, 1536))
    # n_tables outside 1 .. MOT_DP_MAX_ROW_TABLES, no table array, reserved field set
    assert _call(two, 0) == L.ERR_BAD_ARG
    assert _call(two, -1) == L.ERR_BAD_ARG
    nine = (L.MotRowTable * 9)(*[L.MotRowTable(i * V * 16, 16, 0) for i in range(9)])
    assert _call(nine, 9) == L.ERR_BAD_ARG
    assert L.DP_MAX_ROW_TABLES == 8
    assert _call(None, 2) == L.ERR_BAD_ARG
    assert _call(_tables((0, 512, 1), (V * 512, 1536)), 2) == L.ERR_BAD_ARG
    # sizes and process arguments
    assert _call(_tables((0, 0), (V * 512, 1536)), 2) == L.ERR_BAD_ARG            # empty rows
    assert _call(_tables((-16, 512), (V * 512, 1536)), 2) == L.ERR_BAD_ARG        # negative offset
    assert _call(two, 2, n_rows=-1) == L.ERR_BAD_ARG
    assert _call(two, 2, dense_bytes=-16) == L.ERR_BAD_ARG
    assert _call(two, 2, rank=2) == L.ERR_BAD_ARG
    assert _call(two, 2, pads=None) == L.ERR_BAD_ARG
    assert _call(two, 2, algo=L.DP_NVLS, mc=None) == L.ERR_BAD_ARG
    assert _call(two, 2, algo=L.DP_P2P, peers=None) == L.ERR_BAD_ARG
    # misaligned offsets or widths
    assert _call(_tables((0, 520), (V * 528, 1536)), 2) == L.ERR_MISALIGNED      # row of 520 bytes
    assert _call(_tables((0, 512), (V * 512 + 8, 1536)), 2) == L.ERR_MISALIGNED  # offset of table 1
    assert _call(two, 2, dense_lo=(32 << 20) + 8, dense_bytes=16) == L.ERR_MISALIGNED
    assert _call(two, 2, dense_bytes=24) == L.ERR_MISALIGNED
    assert _call(two, 2, bm=(16 << 20) + 2) == L.ERR_MISALIGNED
    # overlapping ranges: two tables, a table and the dense range, a table and the bitmap, the bitmap and the dense range
    assert _call(_tables((0, 512), (V * 512 - 16, 1536)), 2) == L.ERR_BAD_ARG
    assert _call(two, 2, dense_lo=V * 512 + 16, dense_bytes=64) == L.ERR_BAD_ARG
    assert _call(two, 2, bm=V * 512 + 64) == L.ERR_BAD_ARG
    assert _call(two, 2, bm=(32 << 20) + 16, dense_bytes=4096) == L.ERR_BAD_ARG
    # unsupported: peer-to-peer exists for 2 and 4 ranks, dtypes bf16 / fp32
    assert _call(two, 2, world=8, rank=0) == L.ERR_UNSUPPORTED
    assert _call(two, 2, world=3, rank=0) == L.ERR_UNSUPPORTED
    assert _call(two, 2, dtype=7) == L.ERR_UNSUPPORTED
    assert _call(two, 2, algo=5) == L.ERR_UNSUPPORTED
    # the one-table entry point is the same call with one table: same checks
    lib = L.lib()
    assert lib.mot_dp_exchange_rows(FAKE, FAKE, FAKE, FAKE, 0, 2, 0, V, 520, 16 << 20, 32 << 20, 0, L.BF16, 1, L.DP_P2P,
                                    None) == L.ERR_MISALIGNED
    assert lib.mot_dp_exchange_rows(FAKE, FAKE, FAKE, FAKE, 0, 2, 0, V, 512, 16 << 20, 64, 4096, L.BF16, 1, L.DP_P2P,
                                    None) == L.ERR_BAD_ARG                       # dense range inside the table
    assert lib.mot_dp_exchange_rows(FAKE, FAKE, FAKE, FAKE, 0, 8, 0, V, 512, 16 << 20, 32 << 20, 0, L.BF16, 1, L.DP_P2P,
                                    None) == L.ERR_UNSUPPORTED


def _check_row_bucket_layout():
    """Front token table [V, 128] + three value tables [V, 384] + the byte table, bf16: the row tables lead the
    bucket back to back, the dense range starts at the byte table."""
    tok = torch.nn.Parameter(torch.zeros(V, 128, dtype=torch.bfloat16))
    ves = [torch.nn.Parameter(torch.zeros(V, 384, dtype=torch.bfloat16)) for _ in range(3)]
    byte = torch.nn.Parameter(torch.zeros(458, 8, dtype=torch.bfloat16))
    b = dp.GradBucket([tok, *ves, byte], row_tables=4)
    assert b.row_tables == 4 and b.offsets == [0, V * 128, V * 512, V * 896, V * 1280]
    assert b.flat.numel() == V * 1280 + 458 * 8
    for p, v in zip(b.params, b.views()):
        assert v.shape == p.shape and v.is_contiguous()
    assert b.view_of(ves[1]).data_ptr() == b.flat.data_ptr() + 2 * V * 512
    tabs, dense_lo, dense_bytes = b.rows_layout()
    assert tabs == [(0, 256), (V * 256, 768), (V * 1024, 768), (V * 1792, 768)]
    assert dense_lo == V * 2560 and dense_bytes == 458 * 8 * 2
    assert all(b.is_row_table(t) for t in (tok, *ves)) and not b.is_row_table(byte) and b.holds(byte)
    # the default: one row table (params[0]), everything after it dense -- today's layout
    b1 = dp.GradBucket([tok, *ves, byte])
    assert b1.row_tables == 1 and b1.offsets == b.offsets
    assert b1.rows_layout() == ([(0, 256)], V * 256, (V * 1280 + 458 * 8 - V * 128) * 2)
    assert b1.is_row_table(tok) and not b1.is_row_table(ves[0])
    # a bucket of row tables only: empty dense range
    bv = dp.GradBucket(ves, row_tables=3)
    assert bv.rows_layout()[1:] == (V * 3 * 768, 0)
    return b


def _check_row_bucket_refusals():
    tok = torch.nn.Parameter(torch.zeros(V, 128, dtype=torch.bfloat16))
    with pytest.raises(ValueError, match="share"):
        dp.GradBucket([tok, torch.nn.Parameter(torch.zeros(V + 1, 128, dtype=torch.bfloat16))], row_tables=2)
    with pytest.raises(ValueError, match="2-D"):
        dp.GradBucket([tok, torch.nn.Parameter(torch.zeros(V * 128, dtype=torch.bfloat16))], row_tables=2)
    with pytest.raises(ValueError, match="16 bytes"):
        dp.GradBucket([tok, torch.nn.Parameter(torch.zeros(V, 12, dtype=torch.bfloat16))], row_tables=2)
    with pytest.raises(ValueError, match="16 bytes"):     # 12 fp32 = 48 bytes, but 24 bytes in a bf16 bucket
        dp.GradBucket([tok, torch.nn.Parameter(torch.zeros(V, 12))], dtype=torch.bfloat16, row_tables=2)
    with pytest.raises(ValueError, match="row_tables"):
        dp.GradBucket([tok], row_tables=2)
    with pytest.raises(ValueError, match="row_tables"):
        dp.GradBucket([tok], row_tables=0)
    many = [torch.nn.Parameter(torch.zeros(V, 8, dtype=torch.bfloat16)) for _ in range(9)]
    with pytest.raises(ValueError, match="row_tables"):
        dp.GradBucket(many, row_tables=9)
    dp.GradBucket(many, row_tables=8)


def test_row_table_bucket_layout_and_refusals():
    _check_row_bucket_layout()
    _check_row_bucket_refusals()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, q):
    sys.path.insert(0, os.path.join(ROOT, "mixture-of-tokenizers_b200"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        b = _check_row_bucket_layout()
        _check_row_bucket_refusals()
        assert b._symm is None and b.algo == "nccl" and not b.sparse_rows       # gloo: ordinary memory, one collective
        for i, v in enumerate(b.views()):
            v.fill_(float((rank + 1) * (i + 1)))
        b.attach()
        b.all_reduce_avg()
        for i, p in enumerate(b.params):
            assert torch.equal(p.grad.float(), torch.full(p.shape, 1.5 * (i + 1))), i    # mean of (i+1), 2(i+1)
        q.put((rank, "ok"))
    except Exception as e:  # pragma: no cover
        q.put((rank, repr(e)))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(120)
def test_row_table_bucket_world2_gloo():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=100) for _ in procs]
    for p in procs:
        p.join(timeout=30)
    assert sorted(res) == [(0, "ok"), (1, "ok")], res
