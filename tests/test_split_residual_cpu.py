"""The split residual (runs/71081, V3g) without a GPU: the C ABI's refusals (all decided before any CUDA call), the
schemas and fake implementations of mot_b200::split_residual / split_residual_bwd, and the module's ttb= / pull_in=
checks."""
import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode

import mot_b200
from mot_b200 import _lib as L

V3C = L.F_TOK_NORM | L.F_BYTE_NORM | L.F_HAS_LAMBDAS


def desc(**kw):
    base = dict(abi_version=L.ABI_VERSION, dtype=L.BF16, n_tokens=4096, seq_len=0, tok_vocab=50257, byte_vocab=458, bpt=16,
                tok_dim=1024, byte_dim=64, out_dim=1024, combine=L.ADD, flags=V3C | L.F_SLOT_MAJOR, ttb_dtype=0, eps=1e-7)
    base.update(kw)
    return L.MotDesc(**base)


A = 1 << 20           # an aligned stand-in device address (never dereferenced: every call below fails validation)


def fwd(d, **kw):
    args = dict(tok=A, ids=A, ttb=None, E_tok=A, E_byte=A, lam=A, x=A, x0t=A, x0b=A)
    args.update(kw)
    return L.lib().mot_split_residual_fwd(d, *args.values(), None)


def bwd(d, **kw):
    args = dict(tok=A, ids=A, ttb=None, E_tok=A, E_byte=A, lam=A, gx=A, gx0t=None, gx0b=None, gE_tok=A, gE_byte=A, g_lam=A,
                ws=A)
    args.update(kw)
    vals = list(args.values())
    return L.lib().mot_split_residual_bwd(d, *vals[:13], 1 << 30, 0, None)


def test_symbols_are_exported():
    assert {"mot_split_residual_fwd", "mot_split_residual_bwd"} <= set(L.exported_symbols())


@pytest.mark.parametrize("bad", [
    dict(flags=V3C | L.F_OUT_NORM | L.F_SLOT_MAJOR),                   # V3d: output norm
    dict(flags=L.F_TOK_NORM | L.F_BYTE_NORM | L.F_SLOT_MAJOR),         # V3b: no lambdas
    dict(flags=L.F_OUT_NORM | L.F_SLOT_MAJOR),                         # V3
    dict(combine=L.CONCAT, tok_dim=1024, out_dim=2048),
    dict(row_stride=2048),
    dict(flags=V3C | L.F_IDS_FROM_TTB | L.F_TTB_SCRAMBLE | L.F_TTB_PULL_RIGHT, seq_len=1024),
])
def test_non_v3c_descriptors_are_refused(bad):
    assert fwd(desc(**bad)) == L.ERR_BAD_ARG
    assert bwd(desc(**bad)) == L.ERR_BAD_ARG


@pytest.mark.parametrize("null", ["x", "x0t", "x0b", "tok", "E_tok", "E_byte", "lam", "ids"])
def test_forward_null_pointers(null):
    assert fwd(desc(), **{null: None}) == L.ERR_BAD_ARG
    assert fwd(desc(flags=V3C | L.F_IDS_FROM_TTB | L.F_TTB_SCRAMBLE, seq_len=4096), ids=None, ttb=None) == L.ERR_BAD_ARG


@pytest.mark.parametrize("null", ["gx", "tok", "E_tok", "E_byte", "lam", "gE_tok", "gE_byte", "g_lam", "ws"])
def test_backward_null_pointers(null):
    assert bwd(desc(), **{null: None}) == L.ERR_BAD_ARG


def test_misaligned_outputs_and_gradients():
    assert fwd(desc(), x0t=A + 8) == L.ERR_MISALIGNED
    assert fwd(desc(), x0b=A + 2) == L.ERR_MISALIGNED
    assert bwd(desc(), gx0t=A + 8) == L.ERR_MISALIGNED
    assert bwd(desc(), gx0b=A + 4) == L.ERR_MISALIGNED


def test_empty_batch_writes_nothing():
    assert fwd(desc(n_tokens=0), x=None, x0t=None, x0b=None) == L.OK


def test_module_ttb_and_pull_in_checks():
    ttb = torch.zeros(100, 16, dtype=torch.int16)
    m = mot_b200.MoTSplitResidualEmbedding(100, 458, 1024, 64, 16, ttb=ttb, pull_in=True)
    assert m.pull_in and m.ttb is ttb and "ttb" not in m.state_dict()
    assert {n for n, _ in m.named_parameters()} == {"lambdas", "embed_tokens.weight", "embed_bytes.weight"}
    with pytest.raises(ValueError, match="pull_in"):
        mot_b200.MoTSplitResidualEmbedding(100, 458, 1024, 64, 16, pull_in=True)
    with pytest.raises(ValueError, match="ttb"):
        mot_b200.MoTSplitResidualEmbedding(100, 458, 1024, 64, 16, ttb=torch.zeros(100, 8, dtype=torch.int16))
    with pytest.raises(ValueError, match="ttb"):
        mot_b200.MoTSplitResidualEmbedding(100, 458, 1024, 64, 16, ttb=torch.zeros(100, 16, dtype=torch.int64))
    with pytest.raises(RuntimeError, match="ttb"):
        mot_b200.MoTSplitResidualEmbedding(100, 458, 1024, 64, 16)(torch.zeros(8, dtype=torch.int32))


def test_operator_schemas():
    fw = torch.ops.mot_b200.split_residual.default._schema
    bw = torch.ops.mot_b200.split_residual_bwd.default._schema
    assert fw.name == "mot_b200::split_residual" and len(fw.returns) == 4
    assert [a.name for a in fw.arguments] == ["tok", "ids", "ttb", "E_tok", "E_byte", "lam", "spec", "bpt", "seq_len", "eps",
                                              "plan"]
    assert bw.name == "mot_b200::split_residual_bwd" and len(bw.returns) == 3
    assert [a.name for a in bw.arguments][:3] == ["gx", "gx0t", "gx0b"]
    assert all(str(a.type) == "Optional[Tensor]" for a in bw.arguments[:3])


@pytest.mark.parametrize("derive", [False, True])
def test_fake_implementations(derive):
    mot_b200.set_custom_ops(True)
    try:
        with FakeTensorMode():
            d = "cuda"
            N, V, bpt, bd = 2048, 1000, 16, 64
            tok = torch.empty(N, dtype=torch.int32, device=d)
            ids = None if derive else torch.empty(bpt, N, dtype=torch.int32, device=d)
            ttb = torch.empty(V, bpt, dtype=torch.int16, device=d) if derive else None
            Et = torch.empty(V, bpt * bd, dtype=torch.bfloat16, device=d, requires_grad=True)
            Eb = torch.empty(458, bd, dtype=torch.bfloat16, device=d, requires_grad=True)
            lam = torch.empty(2, device=d, requires_grad=True)
            outs = mot_b200.split_residual(tok, ids, Et, Eb, lam, bpt=bpt, ttb=ttb, seq_len=N, pull=derive)
            assert len(outs) == 3
            for o in outs:
                assert o.shape == (N, bpt * bd) and o.dtype == torch.bfloat16
            assert "split_residual" in type(outs[0].grad_fn).__name__
            spec = mot_b200._library.pack_spec(mot_b200.ops._resid_spec(derive, derive, mot_b200.FP32_EPS))
            r = torch.ops.mot_b200.split_residual(tok, ids, ttb, Et, Eb, lam.detach(), spec, bpt, N, mot_b200.FP32_EPS, True)
            assert r[3].dtype == torch.uint8 and r[3].numel() > N * 8       # the planned workspace travels as a tensor
            g = torch.empty(N, bpt * bd, dtype=torch.bfloat16, device=d)
            gt, gb, gl = torch.ops.mot_b200.split_residual_bwd(g, None, g, tok, ids, ttb, Et.detach(), Eb.detach(),
                                                               lam.detach(), r[3], spec, bpt, N, mot_b200.FP32_EPS)
            assert gt.shape == Et.shape and gb.shape == Eb.shape and gl.shape == (2,) and gl.dtype == torch.float32
    finally:
        mot_b200.set_custom_ops(None)
