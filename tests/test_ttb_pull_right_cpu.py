"""Right pulls from token ids alone (MOT_F_TTB_PULL_RIGHT, with the lookahead tail of MOT_F_TTB_NEXT_TOK), checked
without a GPU: the flag values, the library's verdict on the new flag combinations, the spec code, the fake shapes of
the operators with `next_tok`, and the refusals of a bad `next_tokens` on both dispatch paths."""
import dataclasses

import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode

import mot_b200
from mot_b200 import _lib as L
from mot_b200 import ops
from mot_b200._library import pack_spec, unpack_spec
from test_ttb_pull_cpu import BD, BPT, N, R, S, V, VB, _desc, _t, check_fake_shapes


def test_flag_values_and_descriptor_symbols():
    assert L.F_TTB_PULL_RIGHT == 1 << 10 and L.F_TTB_NEXT_TOK == 1 << 11
    assert L.ABI_VERSION == 7 and L.lib().mot_abi_version() == 7
    for fn in ("mot_byte_pair_fwd", "mot_byte_pair_bwd"):   # the direction is a flag of their descriptor
        assert hasattr(L.lib(), fn) and L._SIGNATURES[fn][1][0] is L.C.POINTER(L.MotDesc)
    assert not hasattr(L.lib(), "mot_byte_pair_ttb_fwd") and not hasattr(L.lib(), "mot_byte_pair_ttb_bwd")


def test_validation_of_the_right_pull_flags():
    ws = L.lib().mot_embed_workspace_bytes
    right, nxt = _desc("right").flags, _desc("right").flags | L.F_TTB_NEXT_TOK
    assert ws(_desc("right")) > 0 and ws(_desc("right", flags=nxt)) > 0
    assert ws(_desc("right", flags=nxt | L.F_TTB_SCRAMBLE)) > 0
    assert ws(_desc("right", flags=right | L.F_TTB_PULL_LEFT)) == 0                  # both directions
    assert ws(_desc(flags=L.F_OUT_NORM | L.F_IDS_FROM_TTB | L.F_TTB_PULL_LEFT | L.F_TTB_NEXT_TOK)) == 0
    assert ws(_desc(flags=L.F_OUT_NORM | L.F_IDS_FROM_TTB | L.F_TTB_NEXT_TOK)) == 0  # a lookahead without a right pull
    assert ws(_desc("right", seq_len=0)) == 0 and ws(_desc("right", seq_len=1000)) == 0   # rows as for the left pull
    assert ws(_desc("right", pad_id=70000)) == 0 and ws(_desc("right", eot_id=-40000)) == 0
    assert ws(_desc("right", combine=L.BYTES_ONLY, tok_vocab=0, tok_dim=0, flags=nxt)) == 0
    assert ws(_desc("right", bpt=33, tok_dim=33 * 8, byte_dim=8, out_dim=33 * 8)) == 0


def _pair_desc(flags, **kw):
    """A pair descriptor (bytes-only, per-byte norm, derived ids' fields set) with no positions; fields overridden by kw."""
    base = dict(abi_version=L.ABI_VERSION, dtype=L.BF16, n_tokens=0, seq_len=16, tok_vocab=100, byte_vocab=458, bpt=4,
                byte_dim=16, out_dim=64, combine=L.BYTES_ONLY, flags=flags, ttb_dtype=L.TTB_I16, eps=1e-7, row_stride=64,
                pad_id=456, eot_id=457)
    base.update(kw)
    return L.MotDesc(**base)


def test_pair_descriptor_refuses_bad_flags():
    # checked before anything else: no pointer is dereferenced, no device is needed (no positions: accepted is MOT_OK)
    fwd, bwd = L.lib().mot_byte_pair_fwd, L.lib().mot_byte_pair_bwd
    norm, ttb = L.F_BYTE_NORM, L.F_BYTE_NORM | L.F_IDS_FROM_TTB
    left, right, nxt = L.F_TTB_PULL_LEFT, L.F_TTB_PULL_RIGHT, L.F_TTB_NEXT_TOK
    good = (norm, norm | L.F_IDS_I64, ttb | left, ttb | right, ttb | right | nxt)
    for flags in good:
        assert fwd(_pair_desc(flags), *[None] * 7) == L.OK
    bad = [ttb | f for f in (0, left | right, left | nxt, nxt, right | L.F_TTB_SCRAMBLE)]   # the former `flags` argument
    bad += [f | extra for f in good for extra in (L.F_TOK_NORM, L.F_OUT_NORM, L.F_BYTES_FIRST, L.F_SLOT_MAJOR,
                                                  L.F_HAS_LAMBDAS, L.F_TTB_SCRAMBLE)]
    bad += [norm | f for f in (left, right, right | nxt, nxt)]   # pulls without derived ids
    bad += [f & ~L.F_BYTE_NORM for f in good] + [ttb | left | L.F_IDS_I64]
    for flags in bad:
        assert fwd(_pair_desc(flags), *[None] * 7) == L.ERR_BAD_ARG, hex(flags)
        assert bwd(_pair_desc(flags), *[None] * 8, 0, None) == L.ERR_BAD_ARG, hex(flags)
    # another combine, with a descriptor the fused kernels accept
    for combine, tok_dim, out_dim in ((L.ADD, 64, 64), (L.CONCAT, 64, 128), (L.TOK_ONLY, 64, 64), (L.MEAN, 16, 16)):
        d = _pair_desc(ttb | left, combine=combine, tok_dim=tok_dim, out_dim=out_dim, row_stride=out_dim)
        assert L.lib().mot_embed_workspace_bytes(d) > 0
        assert fwd(d, *[None] * 7) == L.ERR_BAD_ARG and bwd(d, *[None] * 8, 0, None) == L.ERR_BAD_ARG


def test_make_desc_sets_the_right_flags():
    E_tok, E_byte = torch.empty(100, 64), torch.empty(458, 16)
    ttb = torch.empty(100, 4, dtype=torch.int16)
    spec = mot_b200.MixSpec(combine="add", ttb_pull=True, ttb_pull_side="right")
    d = ops.make_desc(spec, 64, E_tok, E_byte, 4, ids=None, ttb=ttb, has_lam=False, seq_len=32)
    assert d.flags & L.F_TTB_PULL_RIGHT and not d.flags & (L.F_TTB_PULL_LEFT | L.F_TTB_NEXT_TOK)
    d = ops.make_desc(spec, 64, E_tok, E_byte, 4, ids=None, ttb=ttb, has_lam=False, seq_len=32, next_tok=True)
    assert d.flags & L.F_TTB_PULL_RIGHT and d.flags & L.F_TTB_NEXT_TOK
    d = ops.make_desc(spec, 64, E_tok, E_byte, 4, ids=torch.empty(256, dtype=torch.int64), ttb=None, has_lam=False)
    assert not d.flags & (L.F_TTB_PULL_LEFT | L.F_TTB_PULL_RIGHT | L.F_TTB_NEXT_TOK)


@pytest.mark.parametrize("side", ["left", "right"])
@pytest.mark.parametrize("pull", [False, True])
def test_spec_round_trip(pull, side):
    spec = mot_b200.MixSpec(combine="concat", tok_norm=True, byte_norm=True, ttb_scramble=True, ttb_pull=pull,
                            ttb_pull_side=side)
    code = pack_spec(spec)
    assert bool(code & 2048) == (side == "right")
    assert unpack_spec(code, spec.eps) == spec


def test_invalid_pull_side():
    with pytest.raises(ValueError, match="ttb_pull_side"):
        mot_b200.MixSpec(ttb_pull=True, ttb_pull_side="up")
    with pytest.raises(ValueError, match="ttb_pull_side"):
        mot_b200.mot_embed_byte_fc(torch.zeros(8, dtype=torch.int32), None, torch.empty(10, 64), torch.empty(458, 16),
                                   torch.empty(64, 64), bpt=4, ttb_pull=True, ttb_pull_side="middle")


def test_right_pull_without_lookahead_still_refused():
    ttb = torch.full((100, 16), 456, dtype=torch.int16)
    m = mot_b200.SptByteMixEmbedding(100, 458, 64, 16, 64, ttb=ttb, padding_in="right")
    with pytest.raises(NotImplementedError, match="next_tokens="):
        m(torch.zeros(2, 8, dtype=torch.int32))


def test_fake_shapes_with_next_tok():
    check_fake_shapes("right")


_RIGHT = mot_b200.MixSpec(combine="concat", tok_norm=True, byte_norm=True, ttb_pull=True, ttb_pull_side="right")
_LEFT = mot_b200.MixSpec(combine="concat", tok_norm=True, byte_norm=True, ttb_pull=True)


def _proj(nxt, spec=_RIGHT, pair=False):
    Et, Eb = _t(V, 64, grad=True), _t(VB, BD, grad=True)
    return mot_b200.mot_embed_proj(_t(N, dtype=torch.int64), None, Et, Eb, _t(32, 64 + BPT * BD, grad=True), spec,
                                   bpt=BPT, ttb=_t(V, BPT, dtype=torch.int16), seq_len=S, padded_and_pulled=pair,
                                   next_tokens=nxt)


def _embed(nxt, spec=mot_b200.MixSpec(combine="add", ttb_pull=True, ttb_pull_side="right")):
    return mot_b200.mot_embed(_t(N, dtype=torch.int32), None, _t(V, BPT * BD, grad=True), _t(VB, BD, grad=True), spec,
                              bpt=BPT, ttb=_t(V, BPT, dtype=torch.int16), seq_len=S, next_tokens=nxt)


def _byte_fc(nxt, side="right"):
    return mot_b200.mot_embed_byte_fc(_t(N, dtype=torch.int32), None, _t(V, 64, grad=True), _t(VB, BD, grad=True),
                                      _t(64, 64, grad=True), bpt=BPT, ttb=_t(V, BPT, dtype=torch.int16), seq_len=S,
                                      ttb_pull=True, ttb_pull_side=side, next_tokens=nxt)


def _nxt(count=R, dtype=torch.int32, device="cuda"):
    return torch.empty(count, dtype=dtype, device=device)


# case -> (call, exception type, a piece of its message)
CASES = {
    "embed_count": (lambda: _embed(_nxt(R + 1)), RuntimeError, "one per row"),
    "embed_dtype": (lambda: _embed(_nxt(dtype=torch.float32)), NotImplementedError, "next_tokens must be int32"),
    "embed_device": (lambda: _embed(_nxt(device="cpu")), RuntimeError, "CUDA device"),
    "embed_left": (lambda: _embed(_nxt(), mot_b200.MixSpec(combine="add", ttb_pull=True)), RuntimeError,
                   "lookahead of a right pull"),
    "embed_no_pull": (lambda: _embed(_nxt(), mot_b200.MixSpec(combine="add")), RuntimeError, "lookahead of a right pull"),
    "proj_count": (lambda: _proj(_nxt(R - 1)), RuntimeError, "one per row"),
    "proj_dtype": (lambda: _proj(_nxt(dtype=torch.int16)), NotImplementedError, "next_tokens must be int32"),
    "proj_left": (lambda: _proj(_nxt(), _LEFT), RuntimeError, "lookahead of a right pull"),
    "proj_pair_left": (lambda: _proj(_nxt(), dataclasses.replace(_LEFT, ttb_pull=False), pair=True), RuntimeError,
                       "lookahead of a right pull"),
    "proj_pair_count": (lambda: _proj(_nxt(2 * R), dataclasses.replace(_RIGHT, ttb_pull=False), pair=True),
                        RuntimeError, "one per row"),
    "byte_fc_count": (lambda: _byte_fc(_nxt(1)), RuntimeError, "one per row"),
    "byte_fc_device": (lambda: _byte_fc(_nxt(device="cpu")), RuntimeError, "CUDA device"),
    "byte_fc_left": (lambda: _byte_fc(_nxt(), side="left"), RuntimeError, "lookahead of a right pull"),
}


def _raised(call):
    try:
        call()
    except Exception as e:   # noqa: BLE001 -- the exception itself is the result
        return type(e), str(e)
    return None


@pytest.mark.parametrize("case", sorted(CASES))
def test_both_paths_refuse_bad_next_tokens_alike(case):
    call, exc, text = CASES[case]
    got = {}
    for custom_ops in (False, True):
        mot_b200.set_custom_ops(custom_ops)
        try:
            with FakeTensorMode():
                got[custom_ops] = _raised(call)
        finally:
            mot_b200.set_custom_ops(None)
    assert got[False] is not None and got[False][0] is exc and text in got[False][1], got[False]
    assert got[True] == got[False]
