"""Value embeddings with a gradient bucket on one GPU (no process group: the bucket is ordinary memory and the exchange
a no-op): the backward writes each table's dense gradient straight into its bucket view, with the same bits as without
a bucket; a second backward before the exchange adds to it; a table whose output got no gradient keeps grad None.

Bit-for-bit comparisons use batches without repeated token ids: the fp32 order in which the repeats of one id are summed
follows the sort plan's atomic cursor and is not repeatable run to run (DESIGN 4.4), with or without a bucket.  Batches
with repeats are compared at the 2^-8 bar of the other gradient tests."""
import pytest
import torch

import mot_b200
from mot_b200 import dp

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)


def _pair(V=50257, D=768, n_tables=3, dtype=torch.bfloat16):
    torch.manual_seed(0)
    a = mot_b200.TokenValueEmbeddings(V, D, n_tables).to(DEV).to(dtype)
    b = mot_b200.TokenValueEmbeddings(V, D, n_tables).to(DEV).to(dtype)
    b.load_state_dict(a.state_dict())
    return a, b


def _nerr(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))


def _inputs(V, D, n, n_out, seed, distinct=True):
    g = torch.Generator(device=DEV).manual_seed(seed)
    tok = torch.randperm(V, generator=g, device=DEV)[:n].int() if distinct else \
        torch.randint(0, V, (n,), generator=g, device=DEV, dtype=torch.int32)
    gos = [torch.randn(n, D, generator=g, device=DEV).bfloat16() for _ in range(n_out)]
    return tok, gos


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_bucket_gradients_are_the_views_and_bit_identical(dtype):
    V, D, n = 50257, 768, 16384
    ref, mod = _pair(V, D, 3, dtype)
    bucket = mod.attach_grad_bucket()
    assert bucket.row_tables == 3 and bucket.params == [m.weight for m in mod.value_embeds]
    tok, gos = _inputs(V, D, n, 3, 1)
    torch.autograd.backward(ref(tok), [g.to(dtype) for g in gos])
    torch.autograd.backward(mod(tok), [g.to(dtype) for g in gos])
    for mr, mb in zip(ref.value_embeds, mod.value_embeds):
        assert mb.weight.grad.data_ptr() == bucket.view_of(mb.weight).data_ptr()
        assert torch.equal(mb.weight.grad, mr.weight.grad)
    # a second backward before the exchange adds to the bucket view (autograd accumulates into param.grad)
    tok2, gos2 = _inputs(V, D, n, 3, 2)
    torch.autograd.backward(ref(tok2), [g.to(dtype) for g in gos2])
    torch.autograd.backward(mod(tok2), [g.to(dtype) for g in gos2])
    for mr, mb in zip(ref.value_embeds, mod.value_embeds):
        assert mb.weight.grad.data_ptr() == bucket.view_of(mb.weight).data_ptr()
        assert torch.equal(mb.weight.grad, mr.weight.grad)
    # repeated ids: the same values up to the summation order of the repeats
    for m in (*ref.value_embeds, *mod.value_embeds):
        m.weight.grad = None
    tok3, gos3 = _inputs(V, D, 4 * n, 3, 4, distinct=False)
    torch.autograd.backward(ref(tok3), [g.to(dtype) for g in gos3])
    torch.autograd.backward(mod(tok3), [g.to(dtype) for g in gos3])
    for mr, mb in zip(ref.value_embeds, mod.value_embeds):
        assert mb.weight.grad.data_ptr() == bucket.view_of(mb.weight).data_ptr()
        assert _nerr(mb.weight.grad, mr.weight.grad) <= 2.0 ** -8
    assert bucket.all_reduce_avg() is None                  # no process group: nothing to exchange
    torch.cuda.synchronize()


def test_table_without_output_gradient_keeps_grad_none():
    V, D, n = 5000, 256, 4096
    ref, mod = _pair(V, D, 3)
    mod.attach_grad_bucket()
    tok, gos = _inputs(V, D, n, 3, 3)
    outs_r, outs_b = ref(tok), mod(tok)
    torch.autograd.backward([outs_r[0], outs_r[2]], [gos[0], gos[2]])
    torch.autograd.backward([outs_b[0], outs_b[2]], [gos[0], gos[2]])
    assert mod.value_embeds[1].weight.grad is None
    g_ref = ref.value_embeds[1].weight.grad         # without a bucket: None, or zeros where autograd materialised them
    assert g_ref is None or not bool(g_ref.any())
    for i in (0, 2):
        assert torch.equal(mod.value_embeds[i].weight.grad, ref.value_embeds[i].weight.grad)


def test_front_and_value_embeddings_share_one_bucket():
    """The documented call: the front's token table and the value tables as row tables, the byte table dense behind
    them; every gradient lands in its view with the bits of the bucket-less modules."""
    V, Dt, bd, bpt, D, n = 50257, 256, 16, 16, 768, 8192
    torch.manual_seed(0)
    front = mot_b200.MoTEmbedding(V, 458, Dt, bd, bpt, variant="V3").to(DEV).bfloat16()
    front_ref = mot_b200.MoTEmbedding(V, 458, Dt, bd, bpt, variant="V3").to(DEV).bfloat16()
    front_ref.load_state_dict(front.state_dict())
    ve_ref, ve = _pair(V, D, 3)
    bucket = dp.GradBucket([front.embed_tokens.weight, *(m.weight for m in ve.value_embeds), front.embed_bytes.weight],
                           row_tables=4)
    front.attach_grad_bucket(bucket)
    ve.attach_grad_bucket(bucket)
    g = torch.Generator(device=DEV).manual_seed(5)
    tok = torch.randperm(V, generator=g, device=DEV)[:n].int()
    ids = torch.randint(0, 458, (bpt, n), generator=g, device=DEV, dtype=torch.int32)
    go = torch.randn(1, n, Dt, generator=g, device=DEV).bfloat16()
    gvs = [torch.randn(n, D, generator=g, device=DEV).bfloat16() for _ in range(3)]
    for f, v in ((front_ref, ve_ref), (front, ve)):
        torch.autograd.backward([f(tok, ids), *v(tok)], [go, *gvs])
    params = [front.embed_tokens.weight, *(m.weight for m in ve.value_embeds), front.embed_bytes.weight]
    refs = [front_ref.embed_tokens.weight, *(m.weight for m in ve_ref.value_embeds), front_ref.embed_bytes.weight]
    for i, (p, r) in enumerate(zip(params, refs)):
        assert p.grad.data_ptr() == bucket.view_of(p).data_ptr()
        if 1 <= i <= 3:
            assert torch.equal(p.grad, r.grad), i
        else:          # the byte table sums many repeats of each byte id: see the module docstring
            assert _nerr(p.grad, r.grad) <= 2.0 ** -8, i
