"""torch.compile / compiled-autograd interplay of the drop-in modules, and parity of the torch.library operator path.

The reference wraps the whole model in torch.compile(model, dynamic=False) (scaled-pre-train/train_gpt.py:1195; runs/7:623)
and the runs enable compiled autograd (runs/7:32).  A model that contains the mot_b200 modules must trace with ZERO graph
breaks (fullgraph=True) and give the eager results."""
import pytest
import torch
from torch import nn

import mot_b200

pytestmark = pytest.mark.gpu


def dev():
    return torch.device("cuda:0")


def nerr(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


class TinyRuns(nn.Module):
    """GPT.forward's front of the sum runs (runs/71:312-314) followed by a trainable head."""

    def __init__(self, variant="V3"):
        super().__init__()
        self.emb = mot_b200.MoTEmbedding(2000, 458, 512, 32, 16, variant=variant)
        self.ve = mot_b200.TokenValueEmbeddings(2000, 512, n_tables=2)
        self.head = nn.Linear(512, 16)

    def forward(self, tok, ids, target):
        x = self.emb(tok, ids)
        ve = self.ve(tok)
        x = x + 0.1 * ve[0][None] + 0.2 * ve[1][None]
        return nn.functional.cross_entropy(self.head(x.float()).view(-1, 16), target)


class TinySpt(nn.Module):
    """scaled-pre-train's embed + byte_mixin pair (train_gpt.py:605-606) followed by a head."""

    def __init__(self, addpp=False):
        super().__init__()
        self.front = mot_b200.SptByteMixEmbedding(1500, 458, 64, 16, 256, bytes_per_token=16, add_padded_and_pulled=addpp)
        self.head = nn.Linear(256, 16)

    def forward(self, tok, padded, pulled, target):
        x = self.front(tok, padded, pulled)
        return nn.functional.cross_entropy(self.head(x.float()).view(-1, 16), target)


def _grads(model):
    return {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None}


def _runs_inputs(d):
    g = torch.Generator(device="cuda").manual_seed(4)
    N = 1024
    return (torch.randint(0, 2000, (N,), generator=g, device=d, dtype=torch.int32),
            torch.randint(0, 458, (16, N), generator=g, device=d, dtype=torch.int32),
            torch.randint(0, 16, (N,), generator=g, device=d))


@pytest.mark.parametrize("variant", ["V3", "V3d"])
def test_custom_op_path_equals_function_path(variant):
    d = dev()
    torch.manual_seed(0)
    m = TinyRuns(variant).to(d)
    m.emb.bfloat16(); m.ve.bfloat16()
    args = _runs_inputs(d)
    res = {}
    for mode in (None, True):        # eager autograd.Function path, then forced torch.ops.mot_b200 path
        mot_b200.set_custom_ops(mode)
        try:
            m.zero_grad(set_to_none=True)
            loss = m(*args)
            loss.backward()
            res[mode] = (loss.detach().clone(), _grads(m))
        finally:
            mot_b200.set_custom_ops(None)
    assert abs(float(res[None][0]) - float(res[True][0])) <= 1e-6 * abs(float(res[None][0]))
    assert res[None][1].keys() == res[True][1].keys() and len(res[True][1]) >= 5
    for k in res[None][1]:
        assert nerr(res[True][1][k], res[None][1][k]) <= 2.0 ** -8, k


@pytest.mark.parametrize("addpp", [False, True])
def test_custom_op_path_projection_and_others(addpp):
    d = dev()
    torch.manual_seed(1)
    m = TinySpt(addpp).to(d)
    m.front.embed.bfloat16()
    g = torch.Generator(device="cuda").manual_seed(5)
    tok = torch.randint(0, 1500, (4, 128), generator=g, device=d, dtype=torch.int32)
    padded = torch.randint(0, 458, (4, 128 * 16), generator=g, device=d)
    pulled = torch.randint(0, 458, (4, 128 * 16), generator=g, device=d)
    tgt = torch.randint(0, 16, (4 * 128,), generator=g, device=d)
    res = {}
    for mode in (None, True):
        mot_b200.set_custom_ops(mode)
        try:
            m.zero_grad(set_to_none=True)
            loss = m(tok, padded, pulled, tgt)
            loss.backward()
            res[mode] = (float(loss), _grads(m))
        finally:
            mot_b200.set_custom_ops(None)
    assert abs(res[None][0] - res[True][0]) <= 1e-5 * abs(res[None][0])
    for k in res[None][1]:
        assert nerr(res[True][1][k], res[None][1][k]) <= 2.0 ** -8, k
    assert res[True][1]["front.byte_mixin.mixin.mixin.weight"].dtype == torch.float32   # fp32 master-weight gradient
    # mathblations' digit mixin (fp32 tables on the TF32 path, projection bias: colsum_out and the bias gradient) and
    # value embeddings with one frozen table (the want_mask of tok_gather_bwd)
    dm = mot_b200.DigitMixinEmbedding(1000, 64, 64, 4).to(d)
    ve = mot_b200.TokenValueEmbeddings(1500, 128, n_tables=3).to(d).bfloat16()
    ve.value_embeds[1].weight.requires_grad_(False)
    idx = torch.randint(0, 1000, (8, 11), generator=g, device=d)
    digits = torch.randint(0, 14, (8, 11 * 4), generator=g, device=d)
    go_dm = torch.randn(8, 11, 64, generator=g, device=d)
    go_ve = [torch.randn(4, 128, 128, generator=g, device=d).bfloat16() for _ in range(3)]
    res = {}
    for mode in (None, True):
        mot_b200.set_custom_ops(mode)
        try:
            dm.zero_grad(set_to_none=True)
            ve.zero_grad(set_to_none=True)
            loss = (dm(idx, digits) * go_dm).sum()
            loss = loss + sum((o.float() * go.float()).sum() for o, go in zip(ve(tok), go_ve))
            loss.backward()
            res[mode] = (float(loss), {**_grads(dm), **{"ve." + k: v for k, v in _grads(ve).items()}})
        finally:
            mot_b200.set_custom_ops(None)
    assert abs(res[None][0] - res[True][0]) <= 1e-5 * abs(res[None][0])
    assert res[None][1].keys() == res[True][1].keys()
    assert "digit_mixin.fc.bias" in res[True][1] and "ve.value_embeds.1.weight" not in res[True][1]
    for k in res[None][1]:
        assert nerr(res[True][1][k], res[None][1][k]) <= 2.0 ** -8, k
    # byte-FC variant, digits, integer ops and the expand through the operators
    mot_b200.set_custom_ops(True)
    try:
        fc = mot_b200.MoTByteFcEmbedding(800, 458, 512, 32, 16).to(d).bfloat16()
        t1 = torch.randint(0, 800, (300,), generator=g, device=d, dtype=torch.int32)
        i1 = torch.randint(0, 458, (16, 300), generator=g, device=d, dtype=torch.int32)
        go = torch.randn(1, 300, 512, generator=g, device=d).bfloat16()
        fc(t1, i1).backward(go)
        got = _grads(fc)
        mot_b200.set_custom_ops(None)
        fc.zero_grad(set_to_none=True)
        fc(t1, i1).backward(go)
        for k, v in _grads(fc).items():
            assert nerr(got[k], v) <= 2.0 ** -8, k
        mot_b200.set_custom_ops(True)
        tab = torch.randint(0, 457, (800, 16), generator=g, device=d).to(torch.int16)
        b_ops = mot_b200.ttb_expand(t1, tab)
        p_ops = mot_b200.pull_from_left(b_ops, 16)
        dg_ops = mot_b200.tokens_to_digits(t1, 4, 10000, 10001, 10002)
        mot_b200.set_custom_ops(None)
        assert torch.equal(b_ops, mot_b200.ttb_expand(t1, tab)) and torch.equal(p_ops, mot_b200.pull_from_left(b_ops, 16))
        assert torch.equal(dg_ops, mot_b200.tokens_to_digits(t1, 4, 10000, 10001, 10002))
    finally:
        mot_b200.set_custom_ops(None)


def _compile_and_compare(model, args, compiled_autograd=False):
    import torch._dynamo
    torch._dynamo.reset()
    model.zero_grad(set_to_none=True)
    loss_e = model(*args)
    loss_e.backward()
    want = (float(loss_e), _grads(model))
    model.zero_grad(set_to_none=True)
    cm = torch.compile(model, dynamic=False, fullgraph=True)          # fullgraph: any graph break raises
    if compiled_autograd:
        with torch._dynamo.utils.maybe_enable_compiled_autograd(True, fullgraph=True, dynamic=False):
            loss_c = cm(*args)
            loss_c.backward()
    else:
        loss_c = cm(*args)
        loss_c.backward()
    got = (float(loss_c), _grads(model))
    assert abs(got[0] - want[0]) <= 1e-4 * abs(want[0]), (got[0], want[0])
    assert got[1].keys() == want[1].keys()
    for k in want[1]:
        assert nerr(got[1][k], want[1][k]) <= 2.0 ** -7, k
    # second call: no recompilation, same numbers
    model.zero_grad(set_to_none=True)
    cm(*args).backward()
    for k in want[1]:
        assert nerr(_grads(model)[k], want[1][k]) <= 2.0 ** -7, k


def test_torch_compile_fullgraph_runs_front():
    d = dev()
    torch.manual_seed(0)
    m = TinyRuns("V3").to(d)
    m.emb.bfloat16(); m.ve.bfloat16()
    _compile_and_compare(m, _runs_inputs(d))


def test_torch_compile_fullgraph_spt_front():
    d = dev()
    torch.manual_seed(0)
    m = TinySpt().to(d)
    m.front.embed.bfloat16()
    g = torch.Generator(device="cuda").manual_seed(5)
    args = (torch.randint(0, 1500, (4, 128), generator=g, device=d, dtype=torch.int32), None,
            torch.randint(0, 458, (4, 128 * 16), generator=g, device=d), torch.randint(0, 16, (512,), generator=g, device=d))
    _compile_and_compare(m, args)


def test_torch_compile_with_compiled_autograd():
    """runs/7:32 sets torch._dynamo.config.compiled_autograd = True."""
    d = dev()
    torch.manual_seed(0)
    m = TinyRuns("V3d").to(d)
    m.emb.bfloat16(); m.ve.bfloat16()
    _compile_and_compare(m, _runs_inputs(d), compiled_autograd=True)


def test_opcheck_schemas_and_fakes():
    d = dev()
    g = torch.Generator(device="cuda").manual_seed(2)
    N, V, bpt, bd = 128, 300, 16, 16
    tok = torch.randint(0, V, (N,), generator=g, device=d, dtype=torch.int32)
    ids = torch.randint(0, 458, (bpt, N), generator=g, device=d, dtype=torch.int32)
    Et = torch.randn(V, 256, generator=g, device=d).bfloat16().requires_grad_(True)
    Eb = torch.randn(458, bd, generator=g, device=d).bfloat16().requires_grad_(True)
    code = mot_b200._library.pack_spec(mot_b200.MixSpec(combine="add", slot_major=True))
    # schema + fake-tensor consistency (values of the workspace output depend on atomic order: no value comparison)
    torch.library.opcheck(torch.ops.mot_b200.embed.default, (tok, ids, None, Et, Eb, None, code, bpt, 0, mot_b200.FP32_EPS, True),
                          test_utils=("test_schema", "test_faketensor"))
    x = torch.randn(6, 64, generator=g, device=d).bfloat16().requires_grad_(True)
    torch.library.opcheck(torch.ops.mot_b200.mixout_copy.default, (x, 4))
    tab = torch.randint(0, 457, (V, bpt), generator=g, device=d).to(torch.int16)
    torch.library.opcheck(torch.ops.mot_b200.ttb_expand.default, (tok, tab, True))
