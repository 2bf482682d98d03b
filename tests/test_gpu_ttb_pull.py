"""Pulled byte ids derived from the ttb table inside the kernels (MOT_F_TTB_PULL_LEFT): every front called with token
ids alone must equal the same front called with the explicit ids of ttb_expand -> pull_from_left -> slices."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

PAD, EOT = 456, 457
V, VB = 3000, 458


def dev():
    return torch.device("cuda:0")


def make_ttb(bpt, kind, seed=0):
    """A left-padded [V, bpt] table with the rows the pull has to survive: all-EOT rows, all-pad rows (tokens that add no
    byte), pads inside a row, full rows.  kind: int16 | f32 (plus junk fractional / huge values in some rows, as in
    float rows missing from the JSON) | bf16 (ids > 256 rounded by the cast, so 457 reads back as 456)."""
    g = torch.Generator().manual_seed(seed)
    t = torch.full((V, bpt), PAD, dtype=torch.int64)
    lens = torch.randint(0, 6, (V,), generator=g)
    for v in range(V):
        n = int(lens[v])
        if n:
            t[v, bpt - n:] = torch.randint(0, 256, (n,), generator=g)
    t[:40] = EOT                                     # EOT rows
    t[40:100] = PAD                                  # rows without a byte
    t[100:140, 0] = 300                              # a byte before the pads
    t[140:200] = torch.randint(0, 456, (60, bpt), generator=g)   # full rows
    if kind == "int16":
        return t.to(torch.int16).to(dev())
    f = t.to(torch.float32)
    if kind == "f32":
        f[200:220] += 0.75                           # truncated like .to(int64)
        f[220:230, -1] = 1.0e6                       # out of the int16 range: the pulled stream keeps its low 16 bits
        f[230:240, -1] = -3.5
        return f.to(dev())
    return f.to(torch.bfloat16).to(dev())


def make_tokens(B, S, seed=0):
    """Rows with runs of EOT tokens, more than 32 consecutive byte-less tokens (so the 32-token window of the kernel is
    short of bytes and has to continue), and segments much longer than bpt tokens."""
    g = torch.Generator().manual_seed(seed + 1)
    tok = torch.randint(100, V, (B, S), generator=g)
    for b in range(B):
        tok[b, 5:9] = torch.randint(0, 40, (4,), generator=g)          # an EOT run
        tok[b, 20:70] = torch.randint(40, 100, (50,), generator=g)     # 50 byte-less tokens
        tok[b, 0] = 45                                                 # the row starts byte-less
        tok[b, S // 2] = 3                                             # an EOT mid row
        tok[b, S - 40:S - 3] = torch.randint(40, 100, (37,), generator=g)
    return tok.to(torch.int32).to(dev())


def explicit_pulled(tok, ttb, bpt):
    import mot_b200
    full = mot_b200.ttb_expand(tok, ttb)                              # [B, S*bpt] int64
    return mot_b200.pull_from_left(full, bpt), full


@pytest.mark.parametrize("bpt", [8, 16, 18, 20, 32])
@pytest.mark.parametrize("kind", ["int16", "f32", "bf16"])
def test_derived_ids_equal_pull_from_left(bpt, kind):
    """The ids themselves: bytes-only, fp32 table with E_byte[v, 0] = v and no norm, so column k*8 of the output is the
    clamped id of slot k."""
    import mot_b200
    ttb = make_ttb(bpt, kind)
    tok = make_tokens(3, 256)
    pulled, _ = explicit_pulled(tok, ttb, bpt)
    E = torch.zeros(VB, 8, device=dev())
    E[:, 0] = torch.arange(VB, device=dev(), dtype=torch.float32)
    spec = mot_b200.MixSpec(combine="bytes_only", out_norm=False, ttb_pull=True)
    out = mot_b200.mot_embed(tok, None, None, E, spec, bpt=bpt, ttb=ttb, seq_len=tok.shape[1])
    got = out.view(-1, bpt, 8)[:, :, 0].long()
    want = pulled.view(-1, bpt).clamp(0, VB - 1)
    assert torch.equal(got, want)


def test_derived_ids_match_reference_golden(golden_dir):
    """Against the reference's own pull_from_left outputs (tests/golden/integer_path.npz)."""
    import mot_b200
    g = np.load(os.path.join(golden_dir, "integer_path.npz"))
    tab = np.load(os.path.join(golden_dir, "ttb_8_left_pad.npz"))["table"]
    full = np.full((50257, 8), PAD, dtype=np.float32)
    full[:50256] = tab
    full[50256] = EOT
    ttb = torch.from_numpy(full).to(dev())
    E = torch.zeros(VB, 8, device=dev())
    E[:, 0] = torch.arange(VB, device=dev(), dtype=torch.float32)
    spec = mot_b200.MixSpec(combine="bytes_only", out_norm=False, ttb_pull=True)
    for case in "abcd":
        tok = torch.from_numpy(g[f"{case}_tokens"]).to(dev())
        out = mot_b200.mot_embed(tok, None, None, E, spec, bpt=8, ttb=ttb, seq_len=tok.shape[1])
        got = out.view(tok.shape[0], -1, 8)[:, :, 0].long().cpu().numpy()
        assert np.array_equal(got, g[f"{case}_pull_from_left"]), case


def _grads(params):
    return [p.grad.detach().clone() for p in params]


def _zero(params):
    for p in params:
        p.grad = None


def _close(a, b):
    for x, y in zip(a, b):
        tol = 2e-2 if x.dtype == torch.bfloat16 else 1e-4
        torch.testing.assert_close(x.float(), y.float(), rtol=tol, atol=tol * max(1.0, float(y.float().abs().max())))


@pytest.mark.parametrize("variant,bpt,kind", [("V3", 16, "int16"), ("V3", 16, "bf16"), ("V3d", 16, "f32"),
                                              ("V3b", 8, "int16"), ("V4", 20, "int16"), ("V5", 18, "f32")])
def test_mot_fronts_token_only_equal_explicit(variant, bpt, kind):
    """MoTEmbedding (runs): one row of T tokens, the `.view(bpt,-1)` scramble for the slot-major variants."""
    import mot_b200
    from mot_b200.modules import RUN_VARIANTS
    torch.manual_seed(0)
    T = 2048
    td, bd = (768, 48) if variant != "V4" and bpt == 16 else (bpt * 32, 32)
    ttb = make_ttb(bpt, kind)
    tok = make_tokens(1, T)[0]
    m = mot_b200.MoTEmbedding(V, VB, td, bd, bytes_per_token=bpt, variant=variant, ttb=ttb, pull_in=True)
    m = m.to(dev()).to(torch.bfloat16)
    m.ttb = ttb                                    # .to(bfloat16) also cast a float ttb buffer; keep the table under test
    pulled, _ = explicit_pulled(tok[None], ttb, bpt)
    ids = pulled.view(bpt, -1) if RUN_VARIANTS[variant].get("slot_major") else pulled
    params = [p for p in m.parameters()]
    ref = m(tok, ids.int())
    g = torch.randn_like(ref)
    ref.backward(g)
    gr = _grads(params)
    _zero(params)
    out = m(tok)
    assert torch.equal(out, ref)
    out.backward(g)
    _close(_grads(params), gr)


@pytest.mark.parametrize("variant,bpt,kind", [("V1", 16, "int16"), ("V2", 16, "bf16"), ("V1", 32, "f32")])
def test_proj_fronts_token_only_equal_explicit(variant, bpt, kind):
    import mot_b200
    torch.manual_seed(0)
    T = 1024
    ttb = make_ttb(bpt, kind)
    tok = make_tokens(1, T)[0]
    m = mot_b200.MoTProjEmbedding(V, VB, 256, 32, 512, bytes_per_token=bpt, variant=variant, ttb=ttb, pull_in=True)
    m = m.to(dev())
    m.embed_tokens.to(torch.bfloat16)
    m.embed_bytes.to(torch.bfloat16)
    pulled, _ = explicit_pulled(tok[None], ttb, bpt)
    ids = pulled.view(bpt, -1) if variant == "V2" else pulled
    params = list(m.parameters())
    ref = m(tok, ids.int())
    g = torch.randn_like(ref)
    ref.backward(g)
    gr = _grads(params)
    _zero(params)
    out = m(tok)
    assert torch.equal(out, ref)
    out.backward(g)
    _close(_grads(params), gr)


def _spt(pull_in, addpp, bpt, kind, B=4, S=512):
    import mot_b200
    torch.manual_seed(0)
    ttb = make_ttb(bpt, kind)
    m = mot_b200.SptByteMixEmbedding(V, VB, 256, 32, 512, bytes_per_token=bpt, pull_in=pull_in,
                                     add_padded_and_pulled=addpp, ttb=ttb).to(dev())
    tok = make_tokens(B, S)
    pulled, full = explicit_pulled(tok, ttb, bpt)
    return m, tok, full, pulled


@pytest.mark.parametrize("pull_in,addpp,bpt,kind", [(True, False, 16, "int16"), (False, False, 16, "int16"),
                                                    (True, True, 16, "int16"), (True, True, 20, "f32"),
                                                    (True, False, 32, "bf16"), (True, True, 8, "bf16")])
def test_spt_token_only_equal_explicit(pull_in, addpp, bpt, kind):
    m, tok, full, pulled = _spt(pull_in, addpp, bpt, kind)
    params = list(m.parameters())
    ref = m(tok, full, pulled)
    g = torch.randn_like(ref)
    ref.backward(g)
    gr = _grads(params)
    _zero(params)
    out = m(tok)
    assert torch.equal(out, ref)
    out.backward(g)
    _close(_grads(params), gr)


def test_byte_fc_token_only_equal_explicit():
    import mot_b200
    torch.manual_seed(0)
    bpt, T = 16, 1024
    ttb = make_ttb(bpt, "int16")
    tok = make_tokens(1, T)[0]
    m = mot_b200.MoTByteFcEmbedding(V, VB, 512, 32, bytes_per_token=bpt).to(dev())
    m.embed_tokens.to(torch.bfloat16)
    m.embed_bytes.to(torch.bfloat16)
    pulled, _ = explicit_pulled(tok[None], ttb, bpt)
    Et, Eb, W = m.embed_tokens.weight, m.embed_bytes.weight, m.byte_fc
    ref = mot_b200.mot_embed_byte_fc(tok, pulled.view(bpt, -1).int(), Et, Eb, W, bpt=bpt)
    g = torch.randn_like(ref)
    ref.backward(g)
    gr = _grads([Et, Eb, W])
    _zero([Et, Eb, W])
    out = mot_b200.mot_embed_byte_fc(tok, None, Et, Eb, W, bpt=bpt, ttb=ttb, seq_len=T, ttb_pull=True)
    assert torch.equal(out, ref)
    out.backward(g)
    _close(_grads([Et, Eb, W]), gr)


def test_right_pull_refused_before_launch():
    import mot_b200
    ttb = make_ttb(16, "int16")
    m = mot_b200.SptByteMixEmbedding(V, VB, 256, 32, 512, bytes_per_token=16, ttb=ttb, padding_in="right").to(dev())
    n0 = mot_b200.ops.launch_count()
    with pytest.raises(NotImplementedError):
        m(make_tokens(2, 128))
    assert mot_b200.ops.launch_count() == n0


def test_custom_op_path_and_compile():
    """The torch.library path (the one torch.compile sees) equals the eager path, under fullgraph compile too."""
    import mot_b200
    from mot_b200 import _library
    m, tok, full, pulled = _spt(True, True, 16, "int16", B=2, S=256)
    ref = m(tok)
    _library.set_custom_ops(True)
    try:
        assert torch.equal(m(tok), ref)
    finally:
        _library.set_custom_ops(None)
    cm = torch.compile(m, fullgraph=True, dynamic=False)
    out = cm(tok)
    assert torch.equal(out, ref)
    out.sum().backward()
    assert m.embed.embed_bytes.weight.grad is not None


def test_cuda_graph_capture():
    import mot_b200
    ttb = make_ttb(16, "int16")
    tok = make_tokens(1, 2048)[0]
    m = mot_b200.MoTEmbedding(V, VB, 768, 48, variant="V3", ttb=ttb, pull_in=True).to(dev()).to(torch.bfloat16)
    for p in m.parameters():
        p.requires_grad_(False)
    ref = m(tok).clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        m(tok)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = m(tok)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, ref)


def test_create_batch_token_ids_only():
    from mot_b200 import data as D
    ttb = make_ttb(16, "int16")
    toks = make_tokens(2, 129)
    ti, bp, bl, tg = D.create_batch(toks, ttb, None, 16, byte_ids=False)
    assert bp is None and bl is None
    assert torch.equal(ti, toks[:, :-1]) and torch.equal(tg, toks[:, 1:])
