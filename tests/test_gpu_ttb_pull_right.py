"""Right-pulled byte ids derived from the ttb table inside the kernels (MOT_F_TTB_PULL_RIGHT, with the one-token lookahead
of MOT_F_TTB_NEXT_TOK): every front called with token ids (and the lookahead) must equal the same front called with the
explicit ids of ttb_expand -> pull_from_right over the window of S + 1 tokens -> the first S*bpt columns."""
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
    """A right-padded [V, bpt] table: all-EOT rows (0..39), byte-less rows (40..99), a byte after the pads (100..139),
    full rows (140..199).  kind: int16 | f32 (with truncated and out-of-range junk values) | bf16 (457 reads back as 456,
    so the EOT test never fires)."""
    g = torch.Generator().manual_seed(seed)
    t = torch.full((V, bpt), PAD, dtype=torch.int64)
    lens = torch.randint(0, 6, (V,), generator=g)
    for v in range(V):
        n = int(lens[v])
        if n:
            t[v, :n] = torch.randint(0, 256, (n,), generator=g)
    t[:40] = EOT
    t[40:100] = PAD
    t[100:140, -1] = 300
    t[140:200] = torch.randint(0, 456, (60, bpt), generator=g)
    if kind == "int16":
        return t.to(torch.int16).to(dev())
    f = t.to(torch.float32)
    if kind == "f32":
        f[200:220] += 0.75
        f[220:230, 0] = 1.0e6
        f[230:240, 0] = -3.5
        return f.to(dev())
    return f.to(torch.bfloat16).to(dev())


def make_window(B, S, seed=0):
    """[B, S + 1] windows whose rows hold the adversarial cases: EOT runs, more than 32 byte-less tokens just before the
    row end, an EOT as the last input token, an EOT / a byte-less token as the lookahead, and a segment whose only bytes
    come from the lookahead."""
    g = torch.Generator().manual_seed(seed + 1)
    w = torch.randint(100, V, (B, S + 1), generator=g)
    for b in range(B):
        w[b, 5:9] = torch.randint(0, 40, (4,), generator=g)                  # an EOT run
        w[b, S // 2] = 3                                                     # an EOT mid row
        w[b, S - 40:S] = torch.randint(40, 100, (40,), generator=g)          # 40 byte-less tokens before the row end
        case = b % 4
        if case == 0:
            w[b, S - 1] = 7                                                  # EOT as the last input token
        elif case == 1:
            w[b, S] = 11                                                     # EOT as the lookahead
        elif case == 2:
            w[b, S] = 60                                                     # byte-less lookahead
        # case 3: the byte-less tail's segment takes its only bytes from the lookahead (a full row, 140..199)
        if case == 3:
            w[b, S] = 150
    return w.to(torch.int32).to(dev())


def explicit_right(window, ttb, bpt, lookahead=True):
    """pull_from_right over the whole window, its last token dropped; without the lookahead over the S tokens."""
    import mot_b200
    S = window.shape[1] - 1
    src = window if lookahead else window[:, :S]
    full = mot_b200.ttb_expand(src.contiguous(), ttb)
    return mot_b200.pull_from_right(full, bpt)[:, :S * bpt].contiguous(), full[:, :S * bpt].contiguous()


def _id_table():
    E = torch.zeros(VB, 8, device=dev())
    E[:, 0] = torch.arange(VB, device=dev(), dtype=torch.float32)
    return E


def _derived(tok, ttb, bpt, S, nxt):
    import mot_b200
    spec = mot_b200.MixSpec(combine="bytes_only", out_norm=False, ttb_pull=True, ttb_pull_side="right")
    out = mot_b200.mot_embed(tok, None, None, _id_table(), spec, bpt=bpt, ttb=ttb, seq_len=S, next_tokens=nxt)
    return out.view(-1, bpt, 8)[:, :, 0].long()


@pytest.mark.parametrize("bpt", [8, 16, 18, 20, 32])
@pytest.mark.parametrize("kind", ["int16", "f32", "bf16"])
def test_derived_ids_equal_pull_from_right(bpt, kind):
    """The ids themselves (bytes-only, fp32 table with E[v, 0] = v, no norm), with and without the lookahead."""
    ttb = make_ttb(bpt, kind)
    S = 256
    w = make_window(4, S)
    tok = w[:, :S].contiguous()
    for lookahead in (True, False):
        pulled, _ = explicit_right(w, ttb, bpt, lookahead)
        got = _derived(tok, ttb, bpt, S, w[:, S] if lookahead else None)
        assert torch.equal(got, pulled.view(-1, bpt).clamp(0, VB - 1)), lookahead


@pytest.mark.parametrize("kind", ["int16", "bf16"])
def test_seq_len_one(kind):
    """Rows of one token: the pull sees the token and its lookahead only."""
    bpt = 16
    ttb = make_ttb(bpt, kind)
    ar = torch.arange(64, device=dev(), dtype=torch.int32)
    w = torch.stack((ar * 13 % 240, ar * 37 % 240), dim=1).contiguous()   # EOT, byte-less and full tokens and lookaheads
    for lookahead in (True, False):
        pulled, _ = explicit_right(w, ttb, bpt, lookahead)
        got = _derived(w[:, :1].contiguous(), ttb, bpt, 1, w[:, 1] if lookahead else None)
        assert torch.equal(got, pulled.view(-1, bpt).clamp(0, VB - 1)), lookahead


def _golden_right_ttb(golden_dir):
    tab = np.load(os.path.join(golden_dir, "ttb_8_left_pad.npz"))["table"]
    full = np.full((50257, 8), PAD, dtype=np.int16)
    full[:50256] = tab
    full[50256] = EOT
    right = np.full_like(full, PAD)
    for v in range(full.shape[0]):                       # the right-padded table as make_golden.py derives it
        ch = full[v][full[v] != PAD]
        right[v, :len(ch)] = ch
    return torch.from_numpy(right).to(dev())


def test_derived_ids_match_reference_golden(golden_dir):
    """Against the reference's own pull_from_right outputs (tests/golden/integer_path.npz): tokens[:, :-1] in,
    tokens[:, -1] as the lookahead."""
    g = np.load(os.path.join(golden_dir, "integer_path.npz"))
    ttb = _golden_right_ttb(golden_dir)
    for case in "abcd":
        toks = torch.from_numpy(g[f"{case}_tokens"]).to(dev())
        S = toks.shape[1] - 1
        got = _derived(toks[:, :S].contiguous(), ttb, 8, S, toks[:, S])
        assert np.array_equal(got.view(toks.shape[0], -1).cpu().numpy(), g[f"{case}_pull_from_right"][:, :-8]), case


def _grads(params):
    return [p.grad.detach().clone() for p in params]


def _zero(params):
    for p in params:
        p.grad = None


def _close(a, b):
    for x, y in zip(a, b):
        tol = 2e-2 if x.dtype == torch.bfloat16 else 1e-4
        torch.testing.assert_close(x.float(), y.float(), rtol=tol, atol=tol * max(1.0, float(y.float().abs().max())))


def _spt(addpp, bpt, kind, B=4, S=512):
    import mot_b200
    torch.manual_seed(0)
    ttb = make_ttb(bpt, kind)
    m = mot_b200.SptByteMixEmbedding(V, VB, 256, 32, 512, bytes_per_token=bpt, pull_in=True,
                                     add_padded_and_pulled=addpp, ttb=ttb, padding_in="right").to(dev())
    w = make_window(B, S)
    return m, w, ttb


@pytest.mark.parametrize("addpp,bpt,kind", [(False, 16, "int16"), (True, 16, "int16"), (False, 20, "f32"),
                                            (True, 8, "bf16"), (False, 32, "bf16")])
def test_spt_token_only_equal_create_batch(addpp, bpt, kind):
    """forward(tokens, next_tokens=window[:, -1]) against the explicit create_batch(padding_in="right") call."""
    from mot_b200 import data as D
    m, w, ttb = _spt(addpp, bpt, kind)
    ti, bpad, bpul, _, nxt = D.create_batch(w, ttb, None, bpt, padding_in="right", next_tokens=True)
    params = list(m.parameters())
    ref = m(ti, bpad, bpul)
    g = torch.randn_like(ref)
    ref.backward(g)
    gr = _grads(params)
    _zero(params)
    out = m(ti, next_tokens=nxt)
    assert torch.equal(out, ref)
    out.backward(g)
    _close(_grads(params), gr)


@pytest.mark.parametrize("variant,bpt,kind", [("V3", 16, "int16"), ("V3d", 16, "f32"), ("V4", 20, "int16"),
                                              ("V5", 18, "bf16")])
def test_mot_embed_token_only_equal_explicit(variant, bpt, kind):
    """mot_embed over one row of T tokens: V3 (saved-output backward) and V3d (lambdas) under the `.view(bpt,-1)`
    scramble, V4 and V5 token-major."""
    import mot_b200
    from mot_b200.modules import RUN_VARIANTS
    torch.manual_seed(0)
    T = 2048
    ttb = make_ttb(bpt, kind)
    w = make_window(1, T)
    tok, nxt = w[0, :T].contiguous(), w[:, T]
    pulled, _ = explicit_right(w, ttb, bpt)
    kw = RUN_VARIANTS[variant]
    slot_major = kw.get("slot_major", False)
    bd = 48 if bpt == 16 else 32
    td = bpt * bd
    Et = torch.randn(V, td, device=dev(), dtype=torch.bfloat16, requires_grad=variant != "V5")
    Eb = torch.randn(VB, bd, device=dev(), dtype=torch.bfloat16, requires_grad=True)
    lam = torch.tensor([0.6, 0.4], device=dev(), requires_grad=True) if variant == "V3d" else None
    params = [p for p in (Et if variant != "V5" else None, Eb, lam) if p is not None]
    E_tok = Et if variant != "V5" else None
    ids = pulled.view(bpt, -1) if slot_major else pulled
    ref = mot_b200.mot_embed(tok if E_tok is not None else None, ids.int(), E_tok, Eb, mot_b200.MixSpec(**kw), bpt=bpt,
                             lam=lam)
    g = torch.randn_like(ref)
    ref.backward(g)
    gr = _grads(params)
    _zero(params)
    spec = mot_b200.MixSpec(**{**kw, "slot_major": False, "ttb_scramble": slot_major, "ttb_pull": True,
                               "ttb_pull_side": "right"})
    out = mot_b200.mot_embed(tok, None, E_tok, Eb, spec, bpt=bpt, lam=lam, ttb=ttb, seq_len=T, next_tokens=nxt)
    assert torch.equal(out, ref)
    out.backward(g)
    _close(_grads(params), gr)


def test_byte_fc_token_only_equal_explicit():
    import mot_b200
    torch.manual_seed(0)
    bpt, T = 16, 1024
    ttb = make_ttb(bpt, "int16")
    w = make_window(1, T)
    tok, nxt = w[0, :T].contiguous(), w[:, T]
    m = mot_b200.MoTByteFcEmbedding(V, VB, 512, 32, bytes_per_token=bpt).to(dev())
    m.embed_tokens.to(torch.bfloat16)
    m.embed_bytes.to(torch.bfloat16)
    pulled, _ = explicit_right(w, ttb, bpt)
    Et, Eb, W = m.embed_tokens.weight, m.embed_bytes.weight, m.byte_fc
    ref = mot_b200.mot_embed_byte_fc(tok, pulled.view(bpt, -1).int(), Et, Eb, W, bpt=bpt)
    g = torch.randn_like(ref)
    ref.backward(g)
    gr = _grads([Et, Eb, W])
    _zero([Et, Eb, W])
    out = mot_b200.mot_embed_byte_fc(tok, None, Et, Eb, W, bpt=bpt, ttb=ttb, seq_len=T, ttb_pull=True,
                                     ttb_pull_side="right", next_tokens=nxt)
    assert torch.equal(out, ref)
    out.backward(g)
    _close(_grads([Et, Eb, W]), gr)


def test_custom_op_path_and_compile():
    """The torch.library path equals the eager path, forward and gradients, and runs under fullgraph compile."""
    from mot_b200 import _library
    m, w, ttb = _spt(True, 16, "int16", B=2, S=256)
    tok, nxt = w[:, :256].contiguous(), w[:, 256].contiguous()
    params = list(m.parameters())
    ref = m(tok, next_tokens=nxt)
    ref.sum().backward()
    gr = _grads(params)
    _zero(params)
    _library.set_custom_ops(True)
    try:
        out = m(tok, next_tokens=nxt)
        assert torch.equal(out, ref)
        out.sum().backward()
        _close(_grads(params), gr)
    finally:
        _library.set_custom_ops(None)
    _zero(params)
    cm = torch.compile(m, fullgraph=True, dynamic=False)
    out = cm(tok, next_tokens=nxt)
    assert torch.equal(out, ref)
    out.sum().backward()
    _close(_grads(params), gr)


def test_cuda_graph_capture():
    import mot_b200
    bpt, T = 16, 2048
    ttb = make_ttb(bpt, "int16")
    w = make_window(1, T)
    tok, nxt = w[0, :T].contiguous(), w[:, T].contiguous()
    E_tok = torch.randn(V, 768, device=dev(), dtype=torch.bfloat16)
    E_byte = torch.randn(VB, 48, device=dev(), dtype=torch.bfloat16)
    spec = mot_b200.MixSpec(combine="add", ttb_scramble=True, ttb_pull=True, ttb_pull_side="right")

    def run():
        return mot_b200.mot_embed(tok, None, E_tok, E_byte, spec, bpt=bpt, ttb=ttb, seq_len=T, next_tokens=nxt)

    ref = run().clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        run()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = run()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, ref)


def test_bad_next_tokens_refused_before_launch():
    import mot_b200
    bpt, S = 16, 128
    ttb = make_ttb(bpt, "int16")
    w = make_window(2, S)
    tok = w[:, :S].contiguous()
    E = _id_table()
    right = mot_b200.MixSpec(combine="bytes_only", out_norm=False, ttb_pull=True, ttb_pull_side="right")
    left = mot_b200.MixSpec(combine="bytes_only", out_norm=False, ttb_pull=True)
    bad = [(right, w[:, S:].reshape(-1)[:1], RuntimeError), (right, w[:, S].float(), NotImplementedError),
           (right, w[:, S].cpu(), RuntimeError), (left, w[:, S], RuntimeError)]
    n0 = mot_b200.ops.launch_count()
    for spec, nxt, exc in bad:
        with pytest.raises(exc):
            mot_b200.mot_embed(tok, None, None, E, spec, bpt=bpt, ttb=ttb, seq_len=S, next_tokens=nxt)
    assert mot_b200.ops.launch_count() == n0


def test_create_batch_next_tokens():
    from mot_b200 import data as D
    ttb = make_ttb(16, "int16")
    w = make_window(2, 128)
    for key in [(True, True, True, True), (True, False, True, True), (True, True, True, False), (True, True, False, False),
                (False, False, True, True), (False, False, True, False), (True, False, False, False),
                (False, False, False, False)]:
        bi, pi, bo, po = key
        kw = dict(byte_in=bi, pull_in=pi, byte_out=bo, pull_out=po, padding_in="right", padding_out="right")
        base = D.create_batch(w, ttb, ttb, 16, **kw)
        got = D.create_batch(w, ttb, ttb, 16, next_tokens=True, **kw)
        assert len(base) == 4 and len(got) == 5
        for a, b in zip(base, got[:4]):
            assert (a is None and b is None) or torch.equal(a, b)
        assert got[4].dtype == torch.int32 and torch.equal(got[4], w[:, -1])
