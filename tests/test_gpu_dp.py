"""The data-parallel exchange of the path on real GPUs (SURVEY 8 A9 / 8e): needs >= 2 CUDA devices with NVLink peers
(skipped otherwise; the host logic runs over gloo in test_dp_gloo.py).

Spawns one process per GPU (NCCL rendezvous on 127.0.0.1) and checks, against an fp32 NCCL all-reduce of the same data:
  * mot_dp_exchange over the whole bucket, P2P and (where the switch offers multicast) NVLS, bf16 and fp32;
  * the same bucket exchanged as ranges on the exchange stream (exchange_async + wait), ragged range sizes;
  * the pipelined training step: vocabulary-slab backward + per-slab exchange == one-piece backward + one exchange,
    and == the average of the ranks' own gradients.
Reference: one dist.all_reduce(param.grad, AVG) per parameter (spt/train_gpt.py:1320-1321, runs/7:697-711)."""
import os
import socket
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


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
        from mot_b200 import dp, ops
        notes = []
        algos = ["p2p"] if world in (2, 4, 8) else []
        probe = dp.GradBucket([torch.nn.Parameter(torch.zeros(64, 8, device=dev), requires_grad=False)], symmetric=True)
        if probe._symm is None:
            q.put((rank, "skip: no symmetric memory"))
            return
        if probe._symm.multicast_ptr != 0:
            algos.append("nvls")
        for algo in algos:
            os.environ["MOT_DP_ALGO"] = algo
            for dtype, shapes in [(torch.bfloat16, [(50257, 64), (458, 48)]), (torch.float32, [(1000, 40), (14, 8)])]:
                params = [torch.nn.Parameter(torch.empty(s, dtype=dtype, device=dev), requires_grad=False) for s in shapes]
                b = dp.GradBucket(params, symmetric=True, n_slabs=4)
                assert b._symm is not None and b.algo == algo, (b.algo, algo)
                g = torch.Generator(device=dev).manual_seed(100 + rank)
                src = torch.randn(b.flat.numel(), generator=g, device=dev).to(dtype)
                ref = src.float()
                dist.all_reduce(ref, op=dist.ReduceOp.SUM)
                ref /= world
                tol = 2.0 ** -7 if dtype == torch.bfloat16 else 1e-6
                for trial in range(3):                      # whole bucket, repeatedly (epochs keep growing)
                    b.flat.copy_(src)
                    b.all_reduce_avg()
                    torch.cuda.synchronize()
                    assert _nerr(b.flat, ref) <= tol, (algo, dtype, trial, _nerr(b.flat, ref))
                # ragged ranges on the exchange stream
                n = b.flat.numel()
                cuts = sorted({0, 8 * 101, min(8 * 5000, n // 4 // 8 * 8), n // 2 // 8 * 8, n})
                for trial in range(2):
                    b.flat.copy_(src)
                    for i in range(len(cuts) - 1):
                        b.exchange_async(cuts[i], cuts[i + 1], last=(i == len(cuts) - 2))
                    b.all_reduce_avg()                      # pending ranges: joins, does not exchange again
                    torch.cuda.synchronize()
                    assert _nerr(b.flat, ref) <= tol, (algo, dtype, "ranges", _nerr(b.flat, ref))
                # every rank holds the same bits (the averaged values are computed once, by the owner of the sub-slice)
                mine = b.flat.clone().view(torch.uint8)      # raw bytes: NCCL broadcasts uint8
                other = mine.clone()
                dist.broadcast(other, src=0)
                assert torch.equal(mine, other), (algo, dtype, "ranks disagree")
            notes.append(algo)
        # ---- the pipelined step of the MoT-sum module against the one-piece step, with every exchange the box offers
        #      (peer-to-peer at 2 / 4 ranks moves only the rows each PEER gathered, NVLS the rows of the union) ----
        for step_algo in algos:
            os.environ["MOT_DP_ALGO"] = step_algo
            V, Dt, bd, bpt, N = 50257, 256, 16, 16, 20000
            res = {}
            for n_slabs in (1, 4):
                torch.manual_seed(0)
                m = mot_b200.MoTEmbedding(V, 458, Dt, bd, bpt, variant="V3").to(dev).bfloat16()
                dp.broadcast_params(m.parameters())
                bucket = m.attach_grad_bucket(dp.GradBucket([m.embed_tokens.weight, m.embed_bytes.weight], symmetric=True,
                                                            n_slabs=n_slabs))
                assert bucket.pipelined == (n_slabs > 1)
                g = torch.Generator(device=dev).manual_seed(7 + rank)        # every rank its own shard of the batch
                tok = torch.randint(0, V, (N,), generator=g, device=dev, dtype=torch.int32)
                ids = torch.randint(0, 458, (bpt, N), generator=g, device=dev, dtype=torch.int32)
                go = torch.randn(1, N, Dt, generator=g, device=dev).bfloat16()
                for step in range(2):
                    for p_ in m.parameters():
                        p_.grad = None
                    m(tok, ids).backward(go)
                    bucket.all_reduce_avg()
                torch.cuda.synchronize()
                res[n_slabs] = (m.embed_tokens.weight.grad.clone(), m.embed_bytes.weight.grad.clone())
                if n_slabs == 1:
                    assert bucket.sparse_rows == (step_algo == "nvls" or world in (2, 4)), "touched-rows exchange availability"
                    seen = torch.zeros(V, dtype=torch.int32, device=dev)
                    seen[tok.long()] = 1
                    dist.all_reduce(seen, op=dist.ReduceOp.MAX)
                    nobody = seen == 0                      # rows no rank gathered: exactly zero, never exchanged
                    assert bool(nobody.any()) and float(res[1][0][nobody].abs().max()) == 0.0
                    mine = res[1][0].clone().view(torch.uint8)       # every rank holds the same bits
                    other = mine.clone()
                    dist.broadcast(other, src=0)
                    assert torch.equal(mine, other), (step_algo, "ranks disagree after the touched-rows exchange")
                if n_slabs == 1:   # fp32 reference: average of the ranks' own (un-exchanged) gradients
                    m2 = mot_b200.MoTEmbedding(V, 458, Dt, bd, bpt, variant="V3").to(dev).bfloat16()
                    m2.load_state_dict(m.state_dict())
                    m2(tok, ids).backward(go)
                    want = [m2.embed_tokens.weight.grad.float(), m2.embed_bytes.weight.grad.float()]
                    for w in want:
                        dist.all_reduce(w, op=dist.ReduceOp.SUM)
                        w /= world
                    assert _nerr(res[1][0], want[0]) <= 2.0 ** -7 and _nerr(res[1][1], want[1]) <= 2.0 ** -7
            assert _nerr(res[4][0], res[1][0]) <= 2.0 ** -7 and _nerr(res[4][1], res[1][1]) <= 2.0 ** -7
        q.put((rank, "ok " + "+".join(notes)))
    except Exception as e:  # pragma: no cover
        import traceback
        q.put((rank, "FAIL " + repr(e) + "\n" + traceback.format_exc()))
    finally:
        try:
            dist.destroy_process_group()
        except Exception:
            pass


@pytest.mark.timeout(600)
def test_exchange_kernels_and_pipelined_step_multi_gpu():
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 CUDA devices with NVLink peers; a 1-GPU machine skips it")
    world = 8 if n >= 8 else (4 if n >= 4 else 2)
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=500) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    if all(r[1].startswith("skip") for r in res):
        pytest.skip(res[0][1])
    assert all(r[1].startswith("ok") for r in res), res
