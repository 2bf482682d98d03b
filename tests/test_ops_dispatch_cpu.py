"""Argument checks of the fused entry points, checked without a GPU: the autograd.Function path (eager) and the
torch.ops.mot_b200 path (torch.compile, MOT_CUSTOM_OPS=1) refuse the same malformed inputs with the same exception type
and message.  Run on fake CUDA tensors: every check raises before a kernel is launched."""
import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode

import mot_b200

N, V, VB, BPT, BD = 64, 100, 458, 4, 16
D = BPT * BD


def _t(*shape, dtype=torch.bfloat16, grad=False):
    return torch.empty(*shape, dtype=dtype, device="cuda", requires_grad=grad)


def _tok():
    return _t(N, dtype=torch.int64)


def _ids(count=N * BPT, dtype=torch.int64):
    return _t(1, count, dtype=dtype)


def _tables(dt_tok=torch.bfloat16, dt_byte=torch.bfloat16):
    return _t(V, D, dtype=dt_tok, grad=True), _t(VB, BD, dtype=dt_byte, grad=True)


_ADD = mot_b200.MixSpec(combine="add")
_CONCAT = mot_b200.MixSpec(combine="concat", tok_norm=True, byte_norm=True)


def _proj(ids=None, tables=None, W=None, bias=None, ids2=None, spec=_CONCAT):
    Et, Eb = tables or _tables()
    W = W if W is not None else _t(32, D + BPT * BD, grad=True)
    return mot_b200.mot_embed_proj(_tok(), ids if ids is not None else _ids(), Et, Eb, W, spec, bpt=BPT, bias=bias,
                                   byte_ids2=ids2)


def _byte_fc(ids=None, tables=None, W=None):
    Et, Eb = tables or _tables()
    W = W if W is not None else _t(D, D, grad=True)
    return mot_b200.mot_embed_byte_fc(_tok(), ids if ids is not None else _ids(), Et, Eb, W, bpt=BPT)


# case -> (call, exception type, a piece of its message)
CASES = {
    "embed_id_count": (lambda: mot_b200.mot_embed(_tok(), _ids(N * BPT - 1), *_tables(), _ADD, bpt=BPT),
                       RuntimeError, "byte ids have"),
    "embed_float_ids": (lambda: mot_b200.mot_embed(_tok(), _ids(dtype=torch.float32), *_tables(), _ADD, bpt=BPT),
                        NotImplementedError, "byte ids must be int32 or int64"),
    "embed_table_dtypes": (lambda: mot_b200.mot_embed(_tok(), _ids(), *_tables(dt_byte=torch.float32), _ADD, bpt=BPT),
                           NotImplementedError, "must share one dtype"),
    "proj_id_count": (lambda: _proj(ids=_ids(N * BPT + 1)), RuntimeError, "byte ids have"),
    "proj_float_ids": (lambda: _proj(ids=_ids(dtype=torch.float32)), NotImplementedError, "int32 or int64"),
    "proj_table_dtypes": (lambda: _proj(tables=_tables(dt_byte=torch.float32)), NotImplementedError,
                          "must both be bf16 or both fp32"),
    "proj_weight_shape": (lambda: _proj(W=_t(32, D, grad=True)), RuntimeError, "projection weight is"),
    "proj_bias_dtype": (lambda: _proj(bias=_t(32, grad=True)), NotImplementedError, "bias must be fp32"),
    "proj_ids2_spec": (lambda: _proj(ids2=_ids(), spec=mot_b200.MixSpec(combine="concat", tok_norm=True)),
                       NotImplementedError, "padded+pulled"),
    "proj_ids2_size": (lambda: _proj(ids2=_ids(N * BPT * 2)), RuntimeError, "two byte-id tensors"),
    "byte_fc_id_count": (lambda: _byte_fc(ids=_ids(N * BPT - 2)), RuntimeError, "byte-FC mix needs"),
    "byte_fc_float_ids": (lambda: _byte_fc(ids=_ids(dtype=torch.float32)), NotImplementedError, "int32 or int64"),
    "byte_fc_table_dtypes": (lambda: _byte_fc(tables=_tables(dt_tok=torch.float32)), NotImplementedError,
                             "must both be bf16 or both fp32"),
    "byte_fc_weight_not_square": (lambda: _byte_fc(W=_t(D, D + 1, grad=True)), RuntimeError, "square [D, D] weight"),
    "tok_gather_shapes": (lambda: mot_b200.tok_gather(_tok(), _t(V, 64, grad=True), _t(V, 32, grad=True)),
                          NotImplementedError, "share one [V, D] shape and dtype"),
    "tok_gather_dtypes": (lambda: mot_b200.tok_gather(_tok(), _t(V, 64, grad=True), _t(V, 64, dtype=torch.float32)),
                          NotImplementedError, "share one [V, D] shape and dtype"),
    "tok_gather_no_table": (lambda: mot_b200.tok_gather(_tok()), RuntimeError, "need at least one table"),
}


def _raised(call):
    try:
        call()
    except Exception as e:   # noqa: BLE001 -- the exception itself is the result
        return type(e), str(e)
    return None


@pytest.mark.parametrize("case", sorted(CASES))
def test_both_paths_refuse_alike(case):
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
