"""The fused split residual (runs/71081:302-304,315, V3g) on the GPU: one kernel writes (x, x0t, x0b), one backward takes
the three upstream gradients.

  * forward: bitwise equal to the three separate launches it replaces (V3c, tok-only + token norm, bytes-only + per-byte
    norm), also above 56832 tokens (stream chunks of more than one 32-entry batch in the backward);
  * gradients: one rounding to the table dtype, so the single-rounding bar of the other gradient tests against the
    oracle, for every combination of unused x0t / x0b;
  * token ids alone (ttb=, pull_in=): the forward of the explicit ids of ttb_expand -> pull_from_left -> .view(bpt, -1);
  * gradient bucket: the views receive the gradients of a run without a bucket and the touched rows are the batch's;
  * torch.compile(fullgraph=True) and one captured CUDA-graph step."""
import pytest
import torch

from oracle import mot_oracle as O

pytestmark = pytest.mark.gpu

TOL = {torch.float32: 1e-5, torch.bfloat16: 2.0 ** -8}
DEV = torch.device("cuda", 0)
VB = 458


def nerr(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def make(V, D, bd, dtype, seed=0, **kw):
    import mot_b200
    torch.manual_seed(seed)
    m = mot_b200.MoTSplitResidualEmbedding(V, VB, D, bd, D // bd, **kw).to(DEV)
    m.embed_tokens.to(dtype), m.embed_bytes.to(dtype)
    with torch.no_grad():
        m.lambdas.copy_(torch.tensor([0.4, 0.7]))
    return m


def three_calls(m, tok, ids):
    """The composition the fused front replaces, through the public mot_embed."""
    import mot_b200
    from mot_b200 import MixSpec
    Et, Eb = m.embed_tokens.weight, m.embed_bytes.weight
    x0t = mot_b200.mot_embed(tok, None, Et, None, MixSpec(combine="tok_only", tok_norm=True, out_norm=False))
    x0b = mot_b200.mot_embed(None, ids, None, Eb, MixSpec(combine="bytes_only", byte_norm=True, out_norm=False,
                                                          slot_major=True), bpt=m.bpt)
    x = mot_b200.mot_embed(tok, ids, Et, Eb, MixSpec(**mot_b200.RUN_VARIANTS["V3c"]), bpt=m.bpt, lam=m.lambdas.flip(0))
    return x, x0t, x0b


def inputs(V, D, bpt, N, dtype, seed=1):
    g = torch.Generator(device=DEV).manual_seed(seed)
    tok = torch.randint(0, V, (N,), generator=g, device=DEV, dtype=torch.int32)
    ids = torch.randint(0, VB, (bpt, N), generator=g, device=DEV, dtype=torch.int32)
    grads = [torch.randn(1, N, D, generator=g, device=DEV).to(dtype) for _ in range(3)]
    return tok, ids, grads


@pytest.mark.parametrize("dtype,V,D,bd,N", [
    (torch.bfloat16, 50257, 1024, 64, 65536),     # runs/71081's shape
    (torch.bfloat16, 400, 512, 32, 777),
    (torch.float32, 50257, 1024, 64, 60000),
    (torch.float32, 400, 512, 32, 777),
])
def test_forward_is_bitwise_the_three_launches(dtype, V, D, bd, N):
    m = make(V, D, bd, dtype)
    tok, ids, _ = inputs(V, D, m.bpt, N, dtype)
    with torch.no_grad():
        got = m(tok, ids)
        want = three_calls(m, tok, ids)
    for g, w, name in zip(got, want, ("x", "x0t", "x0b")):
        assert g.shape == (1, N, D) and g.dtype == dtype
        assert torch.equal(g[0], w), name


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("use_t,use_b", [(True, True), (True, False), (False, True), (False, False)])
def test_gradients_single_rounding_vs_oracle(dtype, use_t, use_b):
    V, D, bd, N = 400, 512, 32, 777
    m = make(V, D, bd, dtype)
    tok, ids, grads = inputs(V, D, m.bpt, N, dtype, seed=5)
    if not use_t:
        grads[1] = torch.zeros_like(grads[1])
    if not use_b:
        grads[2] = torch.zeros_like(grads[2])
    lam = m.lambdas.detach().cpu()
    _, want = O.split_residual_fwd_bwd(tok.cpu(), ids.cpu(), m.embed_tokens.weight.detach().cpu(),
                                       m.embed_bytes.weight.detach().cpu(), lam[1], lam[0],
                                       [g[0].cpu() for g in grads], bpt=m.bpt)
    x, x0t, x0b = m(tok, ids)
    used = [(x, grads[0])] + ([(x0t, grads[1])] if use_t else []) + ([(x0b, grads[2])] if use_b else [])
    torch.autograd.backward([o for o, _ in used], [g for _, g in used])
    torch.cuda.synchronize()
    tol = TOL[dtype]
    assert nerr(m.embed_tokens.weight.grad, want["E_tok"]) <= tol, nerr(m.embed_tokens.weight.grad, want["E_tok"])
    assert nerr(m.embed_bytes.weight.grad, want["E_byte"]) <= tol, nerr(m.embed_bytes.weight.grad, want["E_byte"])
    got_l = m.lambdas.grad.cpu().double()
    ref_l = torch.stack([want["lam_byte"], want["lam_tok"]]).double()
    assert float((got_l - ref_l).abs().max() / ref_l.abs().max()) <= (1e-4 if dtype == torch.float32 else tol)


def test_gradients_past_the_ring_refill_boundary():
    """65536 tokens over a 2000-row vocabulary: stream chunks of several batches, rows straddling chunks."""
    dtype, V, D, bd, N = torch.bfloat16, 2000, 1024, 64, 65536
    m = make(V, D, bd, dtype)
    tok, ids, grads = inputs(V, D, m.bpt, N, dtype, seed=7)
    lam = m.lambdas.detach().cpu()
    _, want = O.split_residual_fwd_bwd(tok.cpu(), ids.cpu(), m.embed_tokens.weight.detach().cpu(),
                                       m.embed_bytes.weight.detach().cpu(), lam[1], lam[0],
                                       [g[0].cpu() for g in grads], bpt=m.bpt)
    torch.autograd.backward(list(m(tok, ids)), grads)
    torch.cuda.synchronize()
    assert nerr(m.embed_tokens.weight.grad, want["E_tok"]) <= TOL[dtype]
    assert nerr(m.embed_bytes.weight.grad, want["E_byte"]) <= TOL[dtype]


def _ttb(V, bpt, seed=3):
    g = torch.Generator().manual_seed(seed)
    t = torch.full((V, bpt), O.PAD_BYTE, dtype=torch.int64)
    lens = torch.randint(0, bpt + 1, (V,), generator=g)
    for v in range(V):
        n = int(lens[v])
        if n:
            t[v, bpt - n:] = torch.randint(0, 256, (n,), generator=g)
    t[:20] = O.EOT_BYTE
    return t.to(torch.int16).to(DEV)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("pull", [False, True])
def test_token_ids_alone(dtype, pull):
    import mot_b200
    V, D, bd, N = 3000, 1024, 64, 4096
    ttb = _ttb(V, D // bd)
    m = make(V, D, bd, dtype, ttb=ttb, pull_in=pull)
    ref = make(V, D, bd, dtype)
    ref.load_state_dict(m.state_dict())
    tok, _, grads = inputs(V, D, m.bpt, N, dtype, seed=9)
    tok[::97] = 5                                                     # EOT tokens inside the row
    flat = mot_b200.ttb_expand(tok, ttb)
    if pull:
        flat = mot_b200.pull_from_left(flat, m.bpt)
    ids = flat.view(m.bpt, -1)
    got, want = m(tok), ref(tok, ids)
    for g, w in zip(got, want):
        assert torch.equal(g, w)
    torch.autograd.backward(list(got), grads)
    torch.autograd.backward(list(want), grads)
    for a, b in zip(m.parameters(), ref.parameters()):
        assert nerr(a.grad, b.grad) <= TOL[dtype]


def test_grad_bucket_views_and_touched_rows():
    from mot_b200 import dp
    dtype, V, D, bd, N = torch.bfloat16, 50257, 1024, 64, 16384
    m, ref = make(V, D, bd, dtype), make(V, D, bd, dtype)
    g = torch.Generator(device=DEV).manual_seed(4)
    tok = torch.randperm(V, generator=g, device=DEV)[:N].int()        # distinct ids: the gradients are bit-repeatable
    ids = torch.randint(0, VB, (m.bpt, N), generator=g, device=DEV, dtype=torch.int32)
    grads = [torch.randn(1, N, D, generator=g, device=DEV).to(dtype) for _ in range(3)]
    bucket = m.attach_grad_bucket()
    assert isinstance(bucket, dp.GradBucket)
    # the touched-rows bitmap of a symmetric-memory bucket, emulated on one GPU (ordinary memory, no exchange)
    bucket.sparse_rows, bucket.bitmap = True, torch.zeros((V + 31) // 32, dtype=torch.int32, device=DEV)
    torch.autograd.backward(list(m(tok, ids)), grads)
    torch.autograd.backward(list(ref(tok, ids)), grads)
    torch.cuda.synchronize()
    for p in (m.embed_tokens.weight, m.embed_bytes.weight):
        assert p.grad.data_ptr() == bucket.view_of(p).data_ptr()
    assert torch.equal(m.embed_tokens.weight.grad, ref.embed_tokens.weight.grad)      # one occurrence per row: exact
    assert nerr(m.embed_bytes.weight.grad, ref.embed_bytes.weight.grad) <= TOL[dtype]  # fp32 atomics in any order
    bits = bucket.bitmap.view(torch.uint8).cpu()
    rows = torch.zeros(((V + 31) // 32) * 32, dtype=torch.bool)
    rows[tok.long().cpu()] = True
    want = torch.zeros_like(bits)
    for k in range(8):
        want |= (rows.view(-1, 8)[:, k].to(torch.uint8) << k)
    assert torch.equal(bits, want)


def test_grad_bucket_shared_with_value_embeddings():
    """One bucket [front token table | 3 value tables | byte table], row_tables=4: every table's gradient lands in its
    view, the same as without the bucket."""
    import mot_b200
    from mot_b200 import dp
    dtype, V, D, bd, N = torch.bfloat16, 50257, 1024, 64, 8192
    m, ref = make(V, D, bd, dtype), make(V, D, bd, dtype)
    ve = mot_b200.TokenValueEmbeddings(V, D).to(DEV).to(dtype)
    g = torch.Generator(device=DEV).manual_seed(6)
    tok = torch.randperm(V, generator=g, device=DEV)[:N].int()
    ids = torch.randint(0, VB, (m.bpt, N), generator=g, device=DEV, dtype=torch.int32)
    grads = [torch.randn(1, N, D, generator=g, device=DEV).to(dtype) for _ in range(3)]
    bucket = dp.GradBucket([m.embed_tokens.weight, *(t.weight for t in ve.value_embeds), m.embed_bytes.weight],
                           row_tables=4)
    assert m.attach_grad_bucket(bucket) is bucket and ve.attach_grad_bucket(bucket) is bucket
    torch.autograd.backward(list(m(tok, ids)), grads)
    torch.autograd.backward(list(ref(tok, ids)), grads)
    torch.cuda.synchronize()
    assert m.embed_tokens.weight.grad.data_ptr() == bucket.view_of(m.embed_tokens.weight).data_ptr()
    assert torch.equal(m.embed_tokens.weight.grad, ref.embed_tokens.weight.grad)
    assert nerr(m.embed_bytes.weight.grad, ref.embed_bytes.weight.grad) <= TOL[dtype]
    assert nerr(m.lambdas.grad, ref.lambdas.grad) <= TOL[dtype]


class _Net(torch.nn.Module):
    def __init__(self, front):
        super().__init__()
        self.front = front

    def forward(self, tok, ids):
        x, x0t, x0b = self.front(tok, ids)
        return (x.float() * 2 + x0t.float() - x0b.float()).sum()


def test_torch_compile_fullgraph():
    dtype, V, D, bd, N = torch.bfloat16, 1000, 1024, 64, 2048
    m, ref = make(V, D, bd, dtype), make(V, D, bd, dtype)
    tok, ids, _ = inputs(V, D, m.bpt, N, dtype)
    torch._dynamo.reset()
    net = torch.compile(_Net(m), fullgraph=True, dynamic=False)
    loss = net(tok, ids)
    loss.backward()
    want = _Net(ref)(tok, ids)
    want.backward()
    assert nerr(loss, want) <= 1e-6                  # same kernels; the compiled graph may sum the rows in another order
    for a, b in zip(m.parameters(), ref.parameters()):
        assert nerr(a.grad, b.grad) <= TOL[dtype]


def test_cuda_graph_step_reproduces_eager():
    dtype, V, D, bd, N = torch.bfloat16, 50257, 1024, 64, 16384
    m = make(V, D, bd, dtype)
    tok, ids, grads = inputs(V, D, m.bpt, N, dtype, seed=11)

    def step():
        for p in m.parameters():
            p.grad = None
        outs = m(tok, ids)
        torch.autograd.backward(list(outs), grads)
        return outs

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs_c = step()
    graph.replay()
    torch.cuda.synchronize()
    got = [o.clone() for o in outs_c] + [p.grad.clone() for p in m.parameters()]
    outs = step()
    torch.cuda.synchronize()
    for a, b in zip(got[:3], outs):
        assert torch.equal(a, b)
    for a, p in zip(got[3:], m.parameters()):
        assert nerr(a, p.grad) <= TOL[dtype]
