"""The touched-rows exchange of one bucket holding the front's token table and the three value embeddings (runs/7:252,308)
on real GPUs: needs >= 2 CUDA devices with NVLink peers (skipped otherwise; CUDA_VISIBLE_DEVICES picks the count).

One process per GPU (NCCL rendezvous on 127.0.0.1).  The bucket is [token table 256 wide | 3 value tables 768 wide |
byte table]: two row widths, one bitmap.  For every exchange the box offers (peer-to-peer at 2 / 4 ranks, NVLS where
the switch has multicast), bf16 and fp32, uniform and Zipf token ids, it checks against an fp32 NCCL average of the
ranks' own gradients:
  * every table within 2^-7 (normalised);
  * rows that no rank gathered are exactly zero in all four row tables;
  * every rank holds the same bits;
  * two micro-batches with different token sets before one all_reduce_avg() equal the dense average (the bitmap is the
    union of every backward since the last exchange, also when autograd adds the second gradient to the first)."""
import os
import socket
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
V, V_BYTE, DT, BD, BPT, DV, N = 50257, 458, 256, 16, 16, 768, 16384


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _nerr(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))


def _tokens(dist, n, lo, hi, g, dev):
    """ids in [lo, hi): uniform, or Zipf(1.0) over a seeded permutation of the range"""
    if dist == "uniform":
        return torch.randint(lo, hi, (n,), generator=g, device=dev, dtype=torch.int32)
    p = 1.0 / torch.arange(1, hi - lo + 1, device=dev, dtype=torch.float64)
    perm = torch.randperm(hi - lo, generator=torch.Generator(device=dev).manual_seed(11), device=dev)
    return (perm[torch.multinomial(p, n, replacement=True, generator=g)] + lo).int()


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
        algos = ["p2p"] if world in (2, 4) else []
        probe = dp.GradBucket([torch.nn.Parameter(torch.zeros(64, 8, device=dev), requires_grad=False)], symmetric=True)
        if probe._symm is None:
            q.put((rank, "skip: no symmetric memory"))
            return
        if probe._symm.multicast_ptr != 0:
            algos.append("nvls")
        if not algos:
            q.put((rank, f"skip: no touched-rows exchange at {world} ranks without multicast"))
            return

        def modules(dtype):
            torch.manual_seed(0)
            front = mot_b200.MoTEmbedding(V, V_BYTE, DT, BD, BPT, variant="V3").to(dev).to(dtype)
            ve = mot_b200.TokenValueEmbeddings(V, DV, 3).to(dev).to(dtype)
            dp.broadcast_params([*front.parameters(), *ve.parameters()])
            return front, ve, [front.embed_tokens.weight, *(m.weight for m in ve.value_embeds), front.embed_bytes.weight]

        def backward(front, ve, tok, seed, dtype):
            g = torch.Generator(device=dev).manual_seed(seed)
            ids = torch.randint(0, V_BYTE, (BPT, tok.numel()), generator=g, device=dev, dtype=torch.int32)
            go = torch.randn(1, tok.numel(), DT, generator=g, device=dev).to(dtype)
            gvs = [torch.randn(tok.numel(), DV, generator=g, device=dev).to(dtype) for _ in range(3)]
            torch.autograd.backward([front(tok, ids), *ve(tok)], [go, *gvs])

        notes = []
        for algo in algos:
            os.environ["MOT_DP_ALGO"] = algo
            for dtype in (torch.bfloat16, torch.float32):
                front, ve, params = modules(dtype)
                ref_front, ref_ve, ref_params = modules(dtype)
                bucket = dp.GradBucket(params, symmetric=True, row_tables=4)
                assert bucket.algo == algo and bucket.sparse_rows, (bucket.algo, algo, bucket.sparse_rows)
                front.attach_grad_bucket(bucket)
                ve.attach_grad_bucket(bucket)
                for dist_name in ("uniform", "zipf"):
                    g = torch.Generator(device=dev).manual_seed(1000 + rank)      # every rank its own shard
                    # micro-batch sets: the whole vocabulary, then two halves (different token sets per micro-batch)
                    for case, batches in (("one batch", [(0, V)]), ("two micro-batches", [(0, V // 2), (V // 2, V)])):
                        toks = [_tokens(dist_name, N, lo, hi, g, dev) for lo, hi in batches]
                        for p in (*params, *ref_params):
                            p.grad = None
                        for i, tok in enumerate(toks):
                            backward(front, ve, tok, 50 + 10 * rank + i, dtype)
                            backward(ref_front, ref_ve, tok, 50 + 10 * rank + i, dtype)
                        bucket.all_reduce_avg()
                        want = [p.grad.float() for p in ref_params]
                        for w in want:
                            dist.all_reduce(w, op=dist.ReduceOp.SUM)
                            w /= world
                        torch.cuda.synchronize()
                        what = (algo, str(dtype), dist_name, case)
                        for i, (p, w) in enumerate(zip(params, want)):
                            assert p.grad.data_ptr() == bucket.view_of(p).data_ptr(), (what, i)
                            assert _nerr(p.grad, w) <= 2.0 ** -7, (what, i, _nerr(p.grad, w))
                        seen = torch.zeros(V, dtype=torch.int32, device=dev)
                        for tok in toks:
                            seen[tok.long()] = 1
                        dist.all_reduce(seen, op=dist.ReduceOp.MAX)
                        nobody = seen == 0
                        assert bool(nobody.any()), what
                        for i, p in enumerate(params[:4]):
                            assert float(p.grad[nobody].abs().max()) == 0.0, (what, i)
                        mine = bucket.flat.clone().view(torch.uint8)
                        other = mine.clone()
                        dist.broadcast(other, src=0)
                        assert torch.equal(mine, other), (what, "ranks disagree")
                del bucket, front, ve, ref_front, ref_ve, params, ref_params
            notes.append(algo)
        q.put((rank, "ok " + "+".join(notes)))
    except Exception as e:  # pragma: no cover
        import traceback
        q.put((rank, "FAIL " + repr(e) + "\n" + traceback.format_exc()))
    finally:
        try:
            dist.destroy_process_group()
        except Exception:
            pass


@pytest.mark.timeout(900)
def test_touched_rows_exchange_of_front_and_value_embeddings_multi_gpu():
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
    res = [q.get(timeout=800) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    if all(r[1].startswith("skip") for r in res):
        pytest.skip(res[0][1])
    assert all(r[1].startswith("ok") for r in res), res
