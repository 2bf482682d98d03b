"""CPU-side checks of the C-ABI library and the host logic: the library loads without a GPU,
exports every symbol include/mot_b200.h declares, validates arguments before touching the
device, and the Python host side refuses CPU tensors (no fallback)."""
import ctypes as C
import os
import re

import pytest
import torch

import mot_b200
from mot_b200 import _lib as L
from mot_b200 import ops

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    src = open(os.path.join(ROOT, "include", "mot_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(mot_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    lib = L.lib()
    names = header_functions()
    assert "mot_embed_fwd" in names and "mot_embed_bwd" in names and "mot_ttb_expand" in names
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/mot_b200.h but not exported"
    assert sorted(L.exported_symbols()) == names, "ctypes signature table out of sync with the header"
    assert lib.mot_abi_version() == L.ABI_VERSION


def test_library_has_no_torch_dependency():
    out = os.popen(f"ldd {L.LIB_PATH}").read()
    assert "libtorch" not in out and "libc10" not in out, out


def test_strerror_and_codes():
    lib = L.lib()
    assert lib.mot_strerror(0) == b"ok"
    for rc in range(1, 7):
        assert len(lib.mot_strerror(rc)) > 3
    assert lib.mot_strerror(99) == b"unknown error"
    with pytest.raises(NotImplementedError):
        L.check(L.ERR_UNSUPPORTED, "x")
    with pytest.raises(RuntimeError):
        L.check(L.ERR_BAD_ARG, "x")


def desc(**kw):
    base = dict(abi_version=L.ABI_VERSION, dtype=L.BF16, n_tokens=49152, seq_len=0, tok_vocab=50257, byte_vocab=458, bpt=16,
                tok_dim=768, byte_dim=48, out_dim=768, combine=L.ADD, flags=L.F_OUT_NORM, ttb_dtype=0, eps=1e-7)
    base.update(kw)
    return L.MotDesc(**base)


def test_workspace_sizes_and_validation_v7():
    lib = L.lib()
    ws = lib.mot_embed_workspace_bytes(desc())
    assert 0 < ws < 64 << 20 and ws % 256 == 0
    assert lib.mot_embed_workspace_bytes(desc(n_tokens=1 << 20, tok_dim=1024, byte_dim=64, out_dim=1024)) < 256 << 20
    # inconsistent dims -> 0 bytes / error codes, all before any CUDA call
    assert lib.mot_embed_workspace_bytes(desc(out_dim=1024)) == 0
    assert lib.mot_embed_workspace_bytes(desc(abi_version=L.ABI_VERSION + 1)) == 0
    null = None
    assert lib.mot_embed_fwd(desc(out_dim=1024), null, null, null, null, null, null, null, null) == L.ERR_BAD_ARG
    assert lib.mot_embed_fwd(desc(byte_dim=44, tok_dim=704, out_dim=704), null, null, null, null, null, null, null, null) == L.ERR_MISALIGNED
    assert lib.mot_embed_fwd(desc(dtype=5), null, null, null, null, null, null, null, null) == L.ERR_UNSUPPORTED
    assert lib.mot_embed_fwd(desc(), null, null, null, null, null, null, null, null) == L.ERR_BAD_ARG  # null pointers
    assert lib.mot_embed_fwd(desc(out_dim=4096, tok_dim=4096, byte_dim=256), null, null, null, null, null, null, null, null) == L.ERR_UNSUPPORTED
    assert lib.mot_ttb_expand(null, 4, null, 10, 8, 0, null, 0, null) == L.ERR_BAD_ARG
    assert lib.mot_ttb_expand(null, 0, null, 10, 8, 0, null, 0, null) == L.OK  # empty input: nothing to do
    assert lib.mot_embed_bwd(desc(), *([null] * 11), 0, 0, null) == L.ERR_BAD_ARG


def test_make_desc_maps_the_variant_catalogue():
    E_tok = torch.empty(50257, 768, dtype=torch.bfloat16)
    E_byte = torch.empty(458, 48, dtype=torch.bfloat16)
    ids32 = torch.empty(16, 64, dtype=torch.int32)
    d = ops.make_desc(mot_b200.MixSpec(combine="add", slot_major=True), 64, E_tok, E_byte, 16, ids=ids32, ttb=None, has_lam=False)
    assert (d.combine, d.out_dim, d.tok_dim, d.byte_dim) == (L.ADD, 768, 768, 48)
    assert d.flags == L.F_OUT_NORM | L.F_SLOT_MAJOR
    d = ops.make_desc(mot_b200.MixSpec(combine="concat", tok_norm=True, byte_norm=True, out_norm=False), 64, E_tok, E_byte, 16,
                      ids=ids32.long(), ttb=None, has_lam=True)
    assert d.out_dim == 768 + 16 * 48
    assert d.flags == L.F_TOK_NORM | L.F_BYTE_NORM | L.F_IDS_I64 | L.F_HAS_LAMBDAS
    ttb = torch.empty(50257, 16, dtype=torch.int16)
    d = ops.make_desc(mot_b200.MixSpec(combine="add", ttb_scramble=True), 64, E_tok, E_byte, 16, ids=None, ttb=ttb, has_lam=False, seq_len=64)
    assert d.flags & L.F_IDS_FROM_TTB and d.flags & L.F_TTB_SCRAMBLE and d.ttb_dtype == L.TTB_I16 and d.seq_len == 64
    with pytest.raises(NotImplementedError):
        ops.make_desc(mot_b200.MixSpec(), 64, E_tok.half(), E_byte.half(), 16, ids=ids32, ttb=None, has_lam=False)
    with pytest.raises(NotImplementedError):
        ops.make_desc(mot_b200.MixSpec(combine="cross_attn"), 64, E_tok, E_byte, 16, ids=ids32, ttb=None, has_lam=False)


def test_cpu_tensors_are_refused_not_emulated():
    E_tok = torch.randn(10, 128).bfloat16()
    E_byte = torch.randn(458, 8).bfloat16()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        mot_b200.mot_embed(torch.zeros(4, dtype=torch.int32), torch.zeros(4, 16, dtype=torch.int32), E_tok, E_byte,
                           mot_b200.MixSpec(), bpt=16)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        mot_b200.ttb_expand(torch.zeros(4, dtype=torch.int32), torch.zeros(10, 8, dtype=torch.int16))


def test_module_keeps_reference_parameter_names():
    m = mot_b200.MoTEmbedding(50257, 458, 1024, 64, 16, variant="V3")
    assert [n for n, _ in m.named_parameters()] == ["embed_tokens.weight", "embed_bytes.weight"]
    assert tuple(m.embed_tokens.weight.shape) == (50257, 1024) and tuple(m.embed_bytes.weight.shape) == (458, 64)
    m = mot_b200.MoTEmbedding(50257, 458, 1024, 64, 16, variant="V3d")
    assert "lambdas" in dict(m.named_parameters())
    with pytest.raises(NotImplementedError):
        mot_b200.MoTEmbedding(50257, 458, 1024, 64, 16, variant="cross_attn")


def test_value_embedding_modules_keep_reference_names_and_refuse_cpu():
    m = mot_b200.TokenValueEmbeddings(50257, 64)
    assert [n for n, _ in m.named_parameters()] == [f"value_embeds.{i}.weight" for i in range(3)]   # runs/7:252
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(5, dtype=torch.int32))
    m9 = mot_b200.MoTValueEmbeddings(1000, 458, 64, 16, 16)                                          # runs/9:252-254
    names = [n for n, _ in m9.named_parameters()]
    assert names[:3] == [f"value_embeds_toks.{i}.weight" for i in range(3)]
    assert names[3:6] == [f"value_embeds_bytes.{i}.weight" for i in range(3)]
    assert names[6:] == [f"value_byte_mixin_weights.{i}" for i in range(3)]
    assert tuple(m9.value_byte_mixin_weights[0].shape) == (64, 64 + 16 * 16) and m9.value_byte_mixin_weights[0].dtype == torch.bfloat16
    m51 = mot_b200.MoTByteFcEmbedding(1000, 458, 512, 32, 16)                                         # runs/71051:253
    assert tuple(m51.byte_fc.shape) == (512, 512) and m51.byte_fc.dtype == torch.bfloat16
    m81 = mot_b200.MoTSplitResidualEmbedding(1000, 458, 512, 32, 16)                                  # runs/71081
    assert [n for n, _ in m81.named_parameters()] == ["lambdas", "embed_tokens.weight", "embed_bytes.weight"]
    with pytest.raises(ValueError):
        mot_b200.MoTSplitResidualEmbedding(1000, 458, 512, 48, 16)


def test_saved_backward_query_needs_no_device():
    lib = L.lib()
    assert lib.mot_embed_bwd_uses_saved(desc()) == 1                       # MoT-sum 768 = 16 x 48, 48K tokens
    assert lib.mot_embed_bwd_uses_saved(desc(n_tokens=1 << 20)) == 0      # > 4 positions per vocabulary row
    assert lib.mot_embed_bwd_uses_saved(desc(flags=L.F_OUT_NORM | L.F_TOK_NORM)) == 0
    assert lib.mot_embed_bwd_uses_saved(desc(combine=L.CONCAT, out_dim=768 + 16 * 48)) == 0
    assert lib.mot_embed_bwd_uses_saved(desc(abi_version=9)) == 0


def test_new_entry_points_validate_descriptors_before_touching_the_device():
    lib = L.lib()
    null = None
    # byte-pair kernels (spt/train_gpt.py:371-379): sizes, alignment and dtype are checked first
    def pair_desc(n=4, bpt=16, bd=48, dtype=L.BF16, ld=256 + 16 * 48, col=256):
        return L.MotDesc(abi_version=L.ABI_VERSION, dtype=dtype, n_tokens=n, byte_vocab=458, bpt=bpt, byte_dim=bd,
                         out_dim=bpt * bd, combine=L.BYTES_ONLY, flags=L.F_BYTE_NORM | L.F_IDS_I64, eps=1e-7,
                         row_stride=ld, col_offset=col)

    def pair_fwd(**kw):
        return lib.mot_byte_pair_fwd(pair_desc(**kw), null, null, null, null, null, null, null)
    assert pair_fwd() == L.ERR_BAD_ARG                       # null pointers
    assert pair_fwd(n=0) == L.OK                             # empty batch: nothing to do
    assert pair_fwd(bd=44) == L.ERR_MISALIGNED
    assert pair_fwd(col=4) == L.ERR_MISALIGNED
    assert pair_fwd(ld=256) == L.ERR_BAD_ARG                 # rows narrower than col + bpt*bd
    assert pair_fwd(bpt=33) == L.ERR_BAD_ARG
    assert pair_fwd(dtype=7) == L.ERR_UNSUPPORTED
    assert lib.mot_byte_pair_workspace_bytes(458, 48) == 16 * 458 * 48 * 4 and lib.mot_byte_pair_workspace_bytes(0, 48) == 0
    assert lib.mot_byte_pair_bwd(pair_desc(), null, null, null, null, null, null, null, null, 0, null) == L.ERR_BAD_ARG
    # uint16 -> int32 widening of shard tokens
    assert lib.mot_tokens_widen_u16(null, 0, null, null) == L.OK
    assert lib.mot_tokens_widen_u16(null, 8, null, null) == L.ERR_BAD_ARG
    assert lib.mot_tokens_widen_u16(null, -1, null, null) == L.ERR_BAD_ARG
    # extended forward / backward: the dense addend is refused with a split concat or strided rows, never dropped
    one = C.c_void_p(16)
    split = desc(combine=L.CONCAT, out_dim=768 + 16 * 48, flags=L.F_TOK_NORM | L.F_BYTE_NORM)
    assert lib.mot_embed_fwd_ex(split, null, null, null, null, null, null, one, null, null, null) == L.ERR_UNSUPPORTED
    strided = desc(combine=L.TOK_ONLY, out_dim=768, byte_dim=8, row_stride=2048, col_offset=0)
    assert lib.mot_embed_fwd_ex(strided, null, null, null, null, null, null, one, null, null, null) == L.ERR_UNSUPPORTED
    assert lib.mot_embed_workspace_bytes(desc(row_stride=512)) == 0          # rows narrower than out_dim
    assert lib.mot_embed_workspace_bytes(desc(row_stride=1024, col_offset=4)) == 0
    assert lib.mot_embed_workspace_bytes(desc(row_stride=1024, col_offset=256)) > 0
