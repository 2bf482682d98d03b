"""The split residual's gradient bucket across ranks: needs >= 2 CUDA devices with NVLink peers (skipped otherwise).

One process per GPU (NCCL rendezvous on 127.0.0.1), 2 or 4 ranks.  A bucket [token table | byte table] attached with
MoTSplitResidualEmbedding.attach_grad_bucket() is averaged with bucket.all_reduce_avg() (the touched-rows exchange where
the box offers it) and compared with an fp32 NCCL average of the gradients of an identical module without a bucket:
every table and the lambdas within 2^-7, rows no rank gathered exactly zero, every rank holding the same bits."""
import os
import socket
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
V, VB, D, BD, N = 50257, 458, 1024, 64, 16384


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _nerr(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))


def _worker(rank, world, port, q):
    import torch.distributed as dist
    for p in (ROOT, os.path.join(ROOT, "mixture-of-tokenizers_b200")):
        sys.path.insert(0, p)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        import mot_b200
        from mot_b200 import dp

        def module(dtype):
            torch.manual_seed(0)
            m = mot_b200.MoTSplitResidualEmbedding(V, VB, D, BD, D // BD).to(dev)
            m.embed_tokens.to(dtype), m.embed_bytes.to(dtype)
            dp.broadcast_params(list(m.parameters()))
            return m

        for dtype in (torch.bfloat16, torch.float32):
            m, ref = module(dtype), module(dtype)
            bucket = m.attach_grad_bucket()
            g = torch.Generator(device=dev).manual_seed(100 + rank)          # every rank its own shard
            tok = torch.randint(0, V // 2, (N,), generator=g, device=dev, dtype=torch.int32)
            ids = torch.randint(0, VB, (m.bpt, N), generator=g, device=dev, dtype=torch.int32)
            grads = [torch.randn(1, N, D, generator=g, device=dev).to(dtype) for _ in range(3)]
            torch.autograd.backward(list(m(tok, ids)), grads)
            torch.autograd.backward(list(ref(tok, ids)), grads)
            bucket.all_reduce_avg()
            dist.all_reduce(m.lambdas.grad, op=dist.ReduceOp.AVG)
            want = [p.grad.float() for p in ref.parameters()]
            for w in want:
                dist.all_reduce(w, op=dist.ReduceOp.SUM)
                w /= world
            torch.cuda.synchronize()
            for (name, p), w in zip(m.named_parameters(), want):
                assert _nerr(p.grad, w) <= 2.0 ** -7, (str(dtype), name, _nerr(p.grad, w))
            assert float(m.embed_tokens.weight.grad[V // 2:].abs().max()) == 0.0
            mine = bucket.flat.clone().view(torch.uint8)
            other = mine.clone()
            dist.broadcast(other, src=0)
            assert torch.equal(mine, other), (str(dtype), "ranks disagree")
            del bucket, m, ref
        q.put((rank, "ok"))
    except Exception as e:  # pragma: no cover
        import traceback
        q.put((rank, "FAIL " + repr(e) + "\n" + traceback.format_exc()))
    finally:
        try:
            dist.destroy_process_group()
        except Exception:
            pass


@pytest.mark.timeout(900)
def test_split_residual_bucket_exchange_multi_gpu():
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 CUDA devices; a 1-GPU machine skips it")
    world = 4 if n >= 4 else 2
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=800) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert all(r[1].startswith("ok") for r in res), res
