"""The token-only call form (pulled byte ids derived from the ttb table inside the kernels), checked without a GPU: the
C ABI flag and descriptor fields, the spec code of the operators, the refusals, and the fake shapes the operators report
to torch.compile.  The right pull (test_ttb_pull_right_cpu.py) shares this file's descriptor, tensor and fake-shape
helpers."""
import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode

import mot_b200
from mot_b200 import _lib as L
from mot_b200 import ops
from mot_b200._library import pack_spec, unpack_spec


def _desc(side="left", **kw):
    """A valid token-only descriptor with a pull from `side`; fields overridden by kw."""
    base = dict(abi_version=L.ABI_VERSION, dtype=L.BF16, n_tokens=4096, seq_len=1024, tok_vocab=50257, byte_vocab=458,
                bpt=16, tok_dim=768, byte_dim=48, out_dim=768, combine=L.ADD,
                flags=L.F_OUT_NORM | L.F_IDS_FROM_TTB | (L.F_TTB_PULL_LEFT if side == "left" else L.F_TTB_PULL_RIGHT),
                ttb_dtype=L.TTB_I16, eps=1e-7, pad_id=456, eot_id=457)
    base.update(kw)
    return L.MotDesc(**base)


def test_flag_and_abi_v7():
    assert L.ABI_VERSION == 7 and L.lib().mot_abi_version() == 7
    assert L.F_TTB_PULL_LEFT == 1 << 9
    names = [f[0] for f in L.MotDesc._fields_]
    assert names[-2:] == ["pad_id", "eot_id"]
    for fn in ("mot_byte_pair_fwd", "mot_byte_pair_bwd"):
        assert hasattr(L.lib(), fn)


def test_validation_of_the_pull_flag():
    ws = L.lib().mot_embed_workspace_bytes
    assert ws(_desc()) > 0
    assert ws(_desc(flags=_desc().flags | L.F_TTB_SCRAMBLE)) > 0
    assert ws(_desc(seq_len=0)) == 0                    # rows are needed
    assert ws(_desc(seq_len=1000)) == 0                 # n_tokens % seq_len != 0
    assert ws(_desc(bpt=33, tok_dim=33 * 8, byte_dim=8, out_dim=33 * 8)) == 0
    assert ws(_desc(pad_id=70000)) == 0                 # the pulled stream holds int16 ids
    assert ws(_desc(combine=L.BYTES_ONLY, tok_vocab=0, tok_dim=0)) == 0   # the ttb rows are needed to derive ids
    # descriptors valid without the flag keep their verdict
    plain = _desc(flags=L.F_OUT_NORM | L.F_IDS_FROM_TTB)
    assert ws(plain) > 0 and ws(_desc(flags=L.F_OUT_NORM, seq_len=0)) > 0
    assert ws(_desc(flags=L.F_OUT_NORM | L.F_IDS_FROM_TTB, seq_len=0)) > 0


def test_make_desc_sets_flag_and_ids():
    E_tok, E_byte = torch.empty(100, 64), torch.empty(458, 16)
    ttb = torch.empty(100, 4, dtype=torch.int16)
    spec = mot_b200.MixSpec(combine="add", ttb_scramble=True, ttb_pull=True)
    d = ops.make_desc(spec, 64, E_tok, E_byte, 4, ids=None, ttb=ttb, has_lam=False, seq_len=32)
    assert d.flags & L.F_IDS_FROM_TTB and d.flags & L.F_TTB_SCRAMBLE and d.flags & L.F_TTB_PULL_LEFT
    assert (d.pad_id, d.eot_id) == (456, 457)
    d = ops.make_desc(spec, 64, E_tok, E_byte, 4, ids=torch.empty(64 * 4, dtype=torch.int64), ttb=None, has_lam=False)
    assert not d.flags & L.F_TTB_PULL_LEFT
    d = ops.make_desc(mot_b200.MixSpec(combine="bytes_only", out_norm=False, ttb_pull=True), 64, None, E_byte, 4, ids=None,
                      ttb=ttb, has_lam=False, seq_len=32)
    assert d.tok_vocab == 100


@pytest.mark.parametrize("pull", [False, True])
def test_spec_round_trip(pull):
    spec = mot_b200.MixSpec(combine="concat", tok_norm=True, byte_norm=True, ttb_scramble=True, ttb_pull=pull)
    code = pack_spec(spec)
    assert bool(code & 1024) == pull
    assert unpack_spec(code, spec.eps) == spec


def test_right_pull_refused():
    ttb = torch.full((100, 16), 456, dtype=torch.int16)
    m = mot_b200.SptByteMixEmbedding(100, 458, 64, 16, 64, ttb=ttb, padding_in="right")
    with pytest.raises(NotImplementedError, match="right-padded"):
        m(torch.zeros(2, 8, dtype=torch.int32))
    with pytest.raises(ValueError):
        mot_b200.SptByteMixEmbedding(100, 458, 64, 16, 64, padding_in="middle")


N, V, VB, BPT, BD, S = 64, 100, 458, 4, 16, 16
R = N // S


def _t(*shape, dtype=torch.bfloat16, grad=False):
    return torch.empty(*shape, dtype=dtype, device="cuda", requires_grad=grad)


def test_bad_seq_len_refused_before_launch():
    with FakeTensorMode():
        Et, Eb, W = _t(V, 64, grad=True), _t(VB, BD, grad=True), _t(32, 64 + BPT * BD, grad=True)
        ttb = _t(V, BPT, dtype=torch.int16)
        spec = mot_b200.MixSpec(combine="concat", tok_norm=True, byte_norm=True, ttb_pull=True)
        for sl in (0, 48):
            with pytest.raises(RuntimeError, match="seq_len"):
                mot_b200.mot_embed_proj(_t(N, dtype=torch.int32), None, Et, Eb, W, spec, bpt=BPT, ttb=ttb, seq_len=sl)
        with pytest.raises(RuntimeError, match="seq_len"):
            mot_b200.mot_embed_byte_fc(_t(N, dtype=torch.int32), None, _t(V, 64), Eb, _t(64, 64), bpt=BPT, ttb=ttb,
                                       seq_len=0, ttb_pull=True)


def check_fake_shapes(side: str) -> None:
    """The operators with `ttb` (ids=None) report the shapes of their outputs; a right pull also passes its lookahead
    next_tok, one token per row of S."""
    with FakeTensorMode():
        tok = _t(N, dtype=torch.int32)
        nxt = (_t(R, dtype=torch.int32),) if side == "right" else ()
        ttb = _t(V, BPT, dtype=torch.int16)
        Et, Eb = _t(V, 64), _t(VB, BD)
        W = _t(32, 64 + BPT * BD, dtype=torch.float32)
        spec = pack_spec(mot_b200.MixSpec(combine="concat", tok_norm=True, byte_norm=True, ttb_pull=True,
                                          ttb_pull_side=side))
        for pair in (False, True):
            out, Y, w_c, ws = torch.ops.mot_b200.embed_proj(tok, None, None, Et, Eb, W, None, spec, BPT, 1e-7, True, ttb, S,
                                                            pair, *nxt)
            assert out.shape == (N, 32) and Y.shape == (N, 32) and w_c.shape == W.shape and ws.numel() > 0
            gt, gb, gW, gbias = torch.ops.mot_b200.embed_proj_bwd(out, tok, None, None, Et, Eb, W, w_c, Y, ws, spec, BPT,
                                                                  1e-7, False, ttb, S, pair, *nxt)
            assert gt.shape == Et.shape and gb.shape == Eb.shape and gW.shape == W.shape and gbias.numel() == 0
        spec_b = pack_spec(mot_b200.MixSpec(combine="bytes_only", out_norm=False, ttb_scramble=True, ttb_pull=True,
                                            ttb_pull_side=side))
        Wf = _t(64, 64)
        out, Y, w_c, ws = torch.ops.mot_b200.embed_byte_fc(tok, None, Et, Eb, Wf, spec_b, BPT, 1e-7, True, ttb, S, *nxt)
        assert out.shape == (N, 64) and Y.shape == (N, 64) and w_c.numel() == 0
        gt, gb, gW = torch.ops.mot_b200.embed_byte_fc_bwd(out, tok, None, Et, Eb, Wf, w_c, Y, ws, spec_b, BPT, 1e-7, ttb, S,
                                                          *nxt)
        assert gt.shape == Et.shape and gb.shape == Eb.shape and gW.shape == Wf.shape
        Ea = _t(V, BPT * BD)
        spec_e = pack_spec(mot_b200.MixSpec(combine="add", ttb_pull=True, ttb_pull_side=side))
        out, rstd, ws = torch.ops.mot_b200.embed(tok, None, ttb, Ea, Eb, None, spec_e, BPT, S, 1e-7, True, *nxt)
        assert out.shape == (N, BPT * BD) and ws.numel() > 0
        gt, gb, gl = torch.ops.mot_b200.embed_bwd(out, tok, None, ttb, Ea, Eb, None, out, rstd, ws, spec_e, BPT, S, 1e-7,
                                                  *nxt)
        assert gt.shape == Ea.shape and gb.shape == Eb.shape and gl.numel() == 0


def test_fake_shapes_with_ttb():
    check_fake_shapes("left")
