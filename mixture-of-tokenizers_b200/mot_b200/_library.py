"""torch.library registration of the path's operators (`torch.ops.mot_b200.*`).

Both reference trees wrap the whole model in `torch.compile(model, dynamic=False)`
(scaled-pre-train/train_gpt.py:1195; runs/7:623) and the runs also enable compiled autograd (runs/7:32).  A ctypes call
inside an `autograd.Function` is opaque to Dynamo (graph break; `fullgraph=True` raises), so every entry point of the
library is ALSO registered as a custom operator with a fake (meta) implementation and a registered autograd formula:
Dynamo / AOTAutograd / compiled autograd then see one opaque node per call and the drop-in stays a one-line module swap.

Dispatch rule (`custom_ops_wanted`): while Dynamo is tracing (`torch.compiler.is_compiling()`) the public functions of
`mot_b200.ops` route through these operators; in eager mode they keep the `autograd.Function`s, whose host overhead is
about half (one Python autograd node instead of dispatcher -> Python kernel -> autograd.Function -> redispatch).
`MOT_CUSTOM_OPS=1` / `set_custom_ops(True)` force the operator path in eager mode too (tests run both).

The operators are functional: the backward workspace (sort plan + accumulators) is an OUTPUT tensor of the forward
operator and an input of the backward operator, allocated fresh and zeroed per call; the plan still runs on the side
stream beside the forward kernel and rejoins before the operator returns (so no event outlives the call and the
operators are CUDA-graph capturable as they are).  The kernels are the same C-ABI entry points either way.
"""
from __future__ import annotations

import os
from typing import List, Optional, Tuple

import torch
from torch import Tensor

from . import ops as O   # ops imports this module at its end: the name resolves from sys.modules

_FORCE: Optional[bool] = {"1": True, "0": False}.get(os.environ.get("MOT_CUSTOM_OPS", ""), None)


def set_custom_ops(mode: Optional[bool]) -> None:
    """True: always route through torch.ops.mot_b200; False: never (even under torch.compile: graph breaks);
    None (default): only while Dynamo is tracing."""
    global _FORCE
    _FORCE = mode


def custom_ops_wanted() -> bool:
    if _FORCE is not None:
        return _FORCE
    return torch.compiler.is_compiling()


# ---------------------------------------------------------------------------------------------------------------
# MixSpec <-> int (operator schemas carry ints, floats, bools and tensors)
# ---------------------------------------------------------------------------------------------------------------
_COMBINE_NAMES = tuple(O._COMBINE)   # the combine mode is its index in this order (bits 0-3 of the code)


def pack_spec(spec) -> int:
    return (_COMBINE_NAMES.index(spec.combine) | (16 if spec.tok_norm else 0) | (32 if spec.byte_norm else 0) |
            (64 if spec.out_norm else 0) | (128 if spec.bytes_first else 0) | (256 if spec.slot_major else 0) |
            (512 if spec.ttb_scramble else 0) | (1024 if spec.ttb_pull else 0) |
            (2048 if spec.ttb_pull_side == "right" else 0))


def unpack_spec(code: int, eps: float):
    return O.MixSpec(combine=_COMBINE_NAMES[code & 15], tok_norm=bool(code & 16), byte_norm=bool(code & 32),
                     out_norm=bool(code & 64), bytes_first=bool(code & 128), slot_major=bool(code & 256),
                     ttb_scramble=bool(code & 512), ttb_pull=bool(code & 1024), eps=eps,
                     ttb_pull_side="right" if code & 2048 else "left")


_PLANNERS: dict = {}


def _plan_beside(desc, tok: Tensor, dev) -> Tensor:
    """A fresh workspace with the sort plan of `tok`, started on the side stream (fork after everything queued on the
    current stream; the library zeroes the head of the fresh buffer there first).  The caller launches its forward
    kernels and then calls _rejoin()."""
    ws = _PLANNERS.get(dev.index)
    if ws is None:   # one per device; the operators share its fork / join events, never its buffer
        ws = _PLANNERS[dev.index] = O.Workspace(None, dev)
    ws.buf = torch.empty(O.embed_workspace_bytes(desc), dtype=torch.uint8, device=dev)
    O.embed_plan_async(desc, tok, ws, dev)         # ws.clean stays False: the plan clears the fresh buffer
    buf, ws.buf = ws.buf, None
    return buf


def _rejoin(dev) -> None:
    O.embed_plan_join(_PLANNERS[dev.index], dev)


def _bwd_workspace(ws: Tensor, desc, dev) -> Tuple[Tensor, bool]:
    """-> (workspace, plan_ready): the forward's planned workspace (left clean by the plan), else a fresh one."""
    if ws.numel() > 0:
        return ws, True
    return torch.empty(O.embed_workspace_bytes(desc), dtype=torch.uint8, device=dev), False


def _empty(dev, dtype=torch.uint8) -> Tensor:
    return torch.empty(0, dtype=dtype, device=dev)


# ---------------------------------------------------------------------------------------------------------------
# mot_b200::embed  (fused gather + pool + combine + norm; every variant without a dense projection)
# ---------------------------------------------------------------------------------------------------------------
@torch.library.custom_op("mot_b200::embed", mutates_args=(), device_types="cuda")
def embed_op(tok: Optional[Tensor], ids: Optional[Tensor], ttb: Optional[Tensor], E_tok: Optional[Tensor],
             E_byte: Optional[Tensor], lam: Optional[Tensor], spec: int, bpt: int, seq_len: int, eps: float,
             plan: bool, next_tok: Optional[Tensor] = None) -> Tuple[Tensor, Tensor, Tensor]:
    """-> (out [n, out_dim], rstd [n] fp32 or [0], workspace uint8 or [0]).  next_tok: the lookahead of a right pull."""
    tok, desc = O._ids_desc(unpack_spec(spec, eps), bpt, seq_len, tok, next_tok, ids, ttb, E_tok, E_byte, lam is not None)
    n, ref = desc.n_tokens, (E_tok if E_tok is not None else E_byte)
    dev = ref.device
    out = torch.empty((n, desc.out_dim), dtype=ref.dtype, device=dev)
    planned = plan and tok is not None and n > 0
    ws = _plan_beside(desc, tok, dev) if planned else _empty(dev)
    keep = plan and n > 0 and O.embed_bwd_uses_saved(desc)
    rstd = torch.empty(n if keep else 0, dtype=torch.float32, device=dev)
    O.embed_forward_out(desc, tok, ids, ttb, E_tok, E_byte, lam, out, rstd=rstd if keep else None)
    if planned:
        _rejoin(dev)
    return out, rstd, ws


@embed_op.register_fake
def _(tok, ids, ttb, E_tok, E_byte, lam, spec, bpt, seq_len, eps, plan, next_tok=None):
    tok, desc = O._ids_desc(unpack_spec(spec, eps), bpt, seq_len, tok, next_tok, ids, ttb, E_tok, E_byte, lam is not None)
    n, ref = desc.n_tokens, (E_tok if E_tok is not None else E_byte)
    planned = plan and tok is not None and n > 0
    keep = plan and n > 0 and O.embed_bwd_uses_saved(desc)
    return (ref.new_empty((n, desc.out_dim)), ref.new_empty((n if keep else 0,), dtype=torch.float32),
            ref.new_empty((O.embed_workspace_bytes(desc) if planned else 0,), dtype=torch.uint8))


@torch.library.custom_op("mot_b200::embed_bwd", mutates_args=(), device_types="cuda")
def embed_bwd_op(grad_out: Tensor, tok: Optional[Tensor], ids: Optional[Tensor], ttb: Optional[Tensor],
                 E_tok: Optional[Tensor], E_byte: Optional[Tensor], lam: Optional[Tensor], out_saved: Optional[Tensor],
                 rstd: Tensor, ws: Tensor, spec: int, bpt: int, seq_len: int, eps: float,
                 next_tok: Optional[Tensor] = None) -> Tuple[Tensor, Tensor, Tensor]:
    """-> (gE_tok dense or [0], gE_byte dense or [0], g_lam fp32 [2] or [0])."""
    tok, desc = O._ids_desc(unpack_spec(spec, eps), bpt, seq_len, tok, next_tok, ids, ttb, E_tok, E_byte, lam is not None)
    n, ref = desc.n_tokens, (E_tok if E_tok is not None else E_byte)
    dev = ref.device
    g = grad_out.reshape(n, desc.out_dim)
    g = (g if g.dtype == ref.dtype else g.to(ref.dtype)).contiguous()
    gE_tok = torch.empty_like(E_tok) if E_tok is not None else _empty(dev, ref.dtype)
    gE_byte = torch.empty_like(E_byte) if E_byte is not None else _empty(dev, ref.dtype)
    g_lam = torch.empty(2 if lam is not None else 0, dtype=torch.float32, device=dev)
    ws, planned = _bwd_workspace(ws, desc, dev)
    keep = rstd.numel() > 0 and out_saved is not None
    O.embed_backward_out(desc, tok, ids, ttb, E_tok, E_byte, lam, g, gE_tok if E_tok is not None else None,
                         gE_byte if E_byte is not None else None, g_lam if lam is not None else None, ws,
                         plan_ready=planned, ws_clean=planned, out_saved=out_saved if keep else None,
                         rstd=rstd if keep else None, plan_joined=planned)
    return gE_tok, gE_byte, g_lam


@embed_bwd_op.register_fake
def _(grad_out, tok, ids, ttb, E_tok, E_byte, lam, out_saved, rstd, ws, spec, bpt, seq_len, eps, next_tok=None):
    ref = E_tok if E_tok is not None else E_byte
    return (torch.empty_like(E_tok) if E_tok is not None else ref.new_empty((0,)),
            torch.empty_like(E_byte) if E_byte is not None else ref.new_empty((0,)),
            ref.new_empty((2 if lam is not None else 0,), dtype=torch.float32))


def _embed_setup(ctx, inputs, output):
    tok, ids, ttb, E_tok, E_byte, lam, spec, bpt, seq_len, eps, plan, next_tok = inputs
    out, rstd, ws = output
    ctx.save_for_backward(tok, ids, ttb, E_tok, E_byte, lam, out if rstd.numel() > 0 else None, rstd, ws, next_tok)
    ctx.cfg = (spec, bpt, seq_len, eps)


def _embed_backward(ctx, g_out, g_rstd, g_ws):
    tok, ids, ttb, E_tok, E_byte, lam, out, rstd, ws, next_tok = ctx.saved_tensors
    gt, gb, gl = torch.ops.mot_b200.embed_bwd(g_out, tok, ids, ttb, E_tok, E_byte, lam, out, rstd, ws, *ctx.cfg, next_tok)
    return (None, None, None, gt if E_tok is not None else None, gb if E_byte is not None else None,
            gl if lam is not None else None, None, None, None, None, None, None)


embed_op.register_autograd(_embed_backward, setup_context=_embed_setup)


# ---------------------------------------------------------------------------------------------------------------
# mot_b200::tok_gather  (several tables gathered with the same token ids: the value embeddings)
# ---------------------------------------------------------------------------------------------------------------
@torch.library.custom_op("mot_b200::tok_gather", mutates_args=(), device_types="cuda")
def tok_gather_op(tok: Tensor, tables: List[Tensor], plan: bool) -> List[Tensor]:
    """-> [tables[0][tok], ..., tables[k-1][tok], workspace]."""
    dev = tok.device
    desc = O._gather_desc(tok, tables[0])
    planned = plan and tok.numel() > 0
    ws = _plan_beside(desc, tok, dev) if planned else _empty(dev)
    outs = O._gather_forward(desc, tok, tables, dev)
    if planned:
        _rejoin(dev)
    return outs + [ws]


@tok_gather_op.register_fake
def _(tok, tables, plan):
    n = tok.numel()
    desc = O._gather_desc(tok, tables[0])
    outs = [E.new_empty((n, E.shape[1])) for E in tables]
    return outs + [tok.new_empty((O.embed_workspace_bytes(desc) if plan and n > 0 else 0,), dtype=torch.uint8)]


@torch.library.custom_op("mot_b200::tok_gather_bwd", mutates_args=(), device_types="cuda")
def tok_gather_bwd_op(tok: Tensor, tables: List[Tensor], grads: List[Tensor], ws: Tensor, want_mask: int) -> List[Tensor]:
    """Dense gradients of the tables whose bit is set in want_mask ([0]-sized placeholders for the others); one sort
    plan serves every scatter."""
    dev = tok.device
    desc = O._gather_desc(tok, tables[0])
    ws, planned = _bwd_workspace(ws, desc, dev)
    want = [(want_mask >> i) & 1 for i in range(len(tables))]
    gEs = O._gather_backward(desc, tok, tables, grads, want, ws, planned, planned)
    return [gE if gE is not None else _empty(dev, E.dtype) for gE, E in zip(gEs, tables)]


@tok_gather_bwd_op.register_fake
def _(tok, tables, grads, ws, want_mask):
    return [torch.empty_like(E) if (want_mask >> i) & 1 else E.new_empty((0,)) for i, E in enumerate(tables)]


def _tok_gather_setup(ctx, inputs, output):
    tok, tables, plan = inputs
    ctx.n_tables = len(tables)
    ctx.save_for_backward(tok, output[-1], *tables)


def _tok_gather_backward(ctx, grads):
    tok, ws, *tables = ctx.saved_tensors
    want = 0
    for i in range(ctx.n_tables):
        if ctx.needs_input_grad[1][i] if isinstance(ctx.needs_input_grad[1], (list, tuple)) else ctx.needs_input_grad[1]:
            want |= 1 << i
    gs = [g if g is not None else torch.zeros((tok.numel(), E.shape[1]), dtype=E.dtype, device=E.device)
          for g, E in zip(grads[:ctx.n_tables], tables)]
    out = torch.ops.mot_b200.tok_gather_bwd(tok, list(tables), gs, ws, want)
    return None, [o if (want >> i) & 1 else None for i, o in enumerate(out)], None


tok_gather_op.register_autograd(_tok_gather_backward, setup_context=_tok_gather_setup)


# ---------------------------------------------------------------------------------------------------------------
# mot_b200::embed_proj  (concat + dense projection variants, tcgen05)
# ---------------------------------------------------------------------------------------------------------------
@torch.library.custom_op("mot_b200::embed_proj", mutates_args=(), device_types="cuda")
def embed_proj_op(tok: Tensor, ids: Optional[Tensor], ids2: Optional[Tensor], E_tok: Tensor, E_byte: Tensor, W: Tensor,
                  bias: Optional[Tensor], spec: int, bpt: int, eps: float, plan: bool, ttb: Optional[Tensor] = None,
                  seq_len: int = 0, ttb_pair: bool = False,
                  next_tok: Optional[Tensor] = None) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """-> (out [n, Do], Y = the product before the row norm or [0], W in the compute dtype or [0], workspace or [0]).
    ids=None with `ttb`: the byte ids come from the table inside the kernels; next_tok: the lookahead of a right pull."""
    dev, cdt = E_tok.device, E_tok.dtype
    sp = unpack_spec(spec, eps)
    tok, desc, desc_pair = O._proj_descs(sp, bpt, seq_len, tok, next_tok, ids, ids2, ttb, ttb_pair, E_tok, E_byte)
    w_c = W if W.dtype == cdt else O.cast_out(W, cdt)
    planned = plan and tok.numel() > 0
    ws = _plan_beside(desc, tok, dev) if planned else _empty(dev)
    out, Y, _ = O._proj_forward(sp, desc, desc_pair, tok, ids, ids2, ttb, E_tok, E_byte, w_c, bias, False)
    if planned:
        _rejoin(dev)
    return out, (Y if sp.out_norm else _empty(dev, cdt)), (w_c if w_c is not W else _empty(dev, cdt)), ws


@embed_proj_op.register_fake
def _(tok, ids, ids2, E_tok, E_byte, W, bias, spec, bpt, eps, plan, ttb=None, seq_len=0, ttb_pair=False, next_tok=None):
    sp = unpack_spec(spec, eps)
    tok, desc, _ = O._proj_descs(sp, bpt, seq_len, tok, next_tok, ids, ids2, ttb, ttb_pair, E_tok, E_byte)
    n, cdt = tok.numel(), E_tok.dtype
    out = E_tok.new_empty((n, W.shape[0]))
    Y = E_tok.new_empty((n, W.shape[0]) if sp.out_norm else (0,))
    w_c = E_tok.new_empty(tuple(W.shape) if W.dtype != cdt else (0,))
    return out, Y, w_c, E_tok.new_empty((O.embed_workspace_bytes(desc) if plan and n > 0 else 0,), dtype=torch.uint8)


@torch.library.custom_op("mot_b200::embed_proj_bwd", mutates_args=(), device_types="cuda")
def embed_proj_bwd_op(grad_out: Tensor, tok: Tensor, ids: Optional[Tensor], ids2: Optional[Tensor], E_tok: Tensor,
                      E_byte: Tensor, W: Tensor, w_c: Tensor, Y: Tensor, ws: Tensor, spec: int, bpt: int, eps: float,
                      has_bias: bool, ttb: Optional[Tensor] = None, seq_len: int = 0,
                      ttb_pair: bool = False, next_tok: Optional[Tensor] = None) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """-> (gE_tok, gE_byte, gW in W's dtype, g_bias fp32 [Do] or [0])."""
    dev = E_tok.device
    sp = unpack_spec(spec, eps)
    tok, desc, desc_pair = O._proj_descs(sp, bpt, seq_len, tok, next_tok, ids, ids2, ttb, ttb_pair, E_tok, E_byte)
    dA, gW, g_bias = O._proj_backward(sp, desc, desc_pair, tok, ids, ids2, ttb, E_tok, E_byte,
                                      w_c if w_c.numel() > 0 else W, W.dtype, has_bias, Y, None,   # operand gathered again
                                      grad_out)
    ws, planned = _bwd_workspace(ws, desc, dev)
    gE_tok, gE_byte = O._scatter_operand(desc, desc_pair, tok, ids, ids2, ttb, E_tok, E_byte, dA, ws, planned, planned)
    return gE_tok, gE_byte, gW, (g_bias if has_bias else _empty(dev, torch.float32))


@embed_proj_bwd_op.register_fake
def _(grad_out, tok, ids, ids2, E_tok, E_byte, W, w_c, Y, ws, spec, bpt, eps, has_bias, ttb=None, seq_len=0, ttb_pair=False,
      next_tok=None):
    return (torch.empty_like(E_tok), torch.empty_like(E_byte), torch.empty_like(W),
            E_tok.new_empty((W.shape[0] if has_bias else 0,), dtype=torch.float32))


def _proj_setup(ctx, inputs, output):
    tok, ids, ids2, E_tok, E_byte, W, bias, spec, bpt, eps, plan, ttb, seq_len, ttb_pair, next_tok = inputs
    out, Y, w_c, ws = output
    ctx.save_for_backward(tok, ids, ids2, E_tok, E_byte, W, w_c, Y, ws, ttb, next_tok)
    ctx.cfg = (spec, bpt, eps, bias is not None)
    ctx.ttb_cfg = (seq_len, ttb_pair)
    ctx.bias_dtype = bias.dtype if bias is not None else None


def _proj_backward(ctx, g_out, g_Y, g_wc, g_ws):
    tok, ids, ids2, E_tok, E_byte, W, w_c, Y, ws, ttb, next_tok = ctx.saved_tensors
    gt, gb, gW, gbias = torch.ops.mot_b200.embed_proj_bwd(g_out, tok, ids, ids2, E_tok, E_byte, W, w_c, Y, ws, *ctx.cfg,
                                                          ttb, *ctx.ttb_cfg, next_tok)
    return (None, None, None, gt, gb, gW, gbias.to(ctx.bias_dtype) if ctx.cfg[3] else None, None, None, None, None,
            None, None, None, None)


embed_proj_op.register_autograd(_proj_backward, setup_context=_proj_setup)


# ---------------------------------------------------------------------------------------------------------------
# mot_b200::embed_byte_fc  (runs/71051: norm(tok + F.linear(cat(bytes), byte_fc)))
# ---------------------------------------------------------------------------------------------------------------
@torch.library.custom_op("mot_b200::embed_byte_fc", mutates_args=(), device_types="cuda")
def embed_byte_fc_op(tok: Tensor, ids: Optional[Tensor], E_tok: Tensor, E_byte: Tensor, W: Tensor, spec_b: int, bpt: int,
                     eps: float, plan: bool, ttb: Optional[Tensor] = None, seq_len: int = 0,
                     next_tok: Optional[Tensor] = None) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """-> (out [n, D], Y = the byte-FC product, W in the compute dtype or [0], workspace or [0]).  ids=None with `ttb`:
    the byte ids come from the table inside the kernels; next_tok: the lookahead of a right pull."""
    dev, cdt = E_tok.device, E_tok.dtype
    tok, desc_b, desc_t = O._fc_descs(unpack_spec(spec_b, eps), bpt, seq_len, tok, next_tok, ids, ttb, E_tok, E_byte)
    w_c = W if W.dtype == cdt else O.cast_out(W, cdt)
    planned = plan and tok.numel() > 0
    ws = _plan_beside(desc_t, tok, dev) if planned else _empty(dev)
    out, Y = O._byte_fc_forward(desc_b, desc_t, tok, ids, E_tok, E_byte, w_c, ttb)
    if planned:
        _rejoin(dev)
    return out, Y, (w_c if w_c is not W else _empty(dev, cdt)), ws


@embed_byte_fc_op.register_fake
def _(tok, ids, E_tok, E_byte, W, spec_b, bpt, eps, plan, ttb=None, seq_len=0, next_tok=None):
    tok, _, desc_t = O._fc_descs(unpack_spec(spec_b, eps), bpt, seq_len, tok, next_tok, ids, ttb, E_tok, E_byte)
    n, D = tok.numel(), E_tok.shape[1]
    return (E_tok.new_empty((n, D)), E_tok.new_empty((n, D)), E_tok.new_empty(tuple(W.shape) if W.dtype != E_tok.dtype else (0,)),
            E_tok.new_empty((O.embed_workspace_bytes(desc_t) if plan and n > 0 else 0,), dtype=torch.uint8))


@torch.library.custom_op("mot_b200::embed_byte_fc_bwd", mutates_args=(), device_types="cuda")
def embed_byte_fc_bwd_op(grad_out: Tensor, tok: Tensor, ids: Optional[Tensor], E_tok: Tensor, E_byte: Tensor, W: Tensor,
                         w_c: Tensor, Y: Tensor, ws: Tensor, spec_b: int, bpt: int, eps: float,
                         ttb: Optional[Tensor] = None, seq_len: int = 0,
                         next_tok: Optional[Tensor] = None) -> Tuple[Tensor, Tensor, Tensor]:
    dev = E_tok.device
    tok, desc_b, desc_t = O._fc_descs(unpack_spec(spec_b, eps), bpt, seq_len, tok, next_tok, ids, ttb, E_tok, E_byte)
    ws, planned = _bwd_workspace(ws, desc_t, dev)
    wsb = torch.empty(O.embed_workspace_bytes(desc_b), dtype=torch.uint8, device=dev)
    return O._byte_fc_backward(desc_b, desc_t, tok, ids, E_tok, E_byte, w_c if w_c.numel() > 0 else W, W.dtype, Y,
                               grad_out, ws, planned, planned, wsb, False, ttb)


@embed_byte_fc_bwd_op.register_fake
def _(grad_out, tok, ids, E_tok, E_byte, W, w_c, Y, ws, spec_b, bpt, eps, ttb=None, seq_len=0, next_tok=None):
    return torch.empty_like(E_tok), torch.empty_like(E_byte), torch.empty_like(W)


def _fc_setup(ctx, inputs, output):
    tok, ids, E_tok, E_byte, W, spec_b, bpt, eps, plan, ttb, seq_len, next_tok = inputs
    out, Y, w_c, ws = output
    ctx.save_for_backward(tok, ids, E_tok, E_byte, W, w_c, Y, ws, ttb, next_tok)
    ctx.cfg = (spec_b, bpt, eps)
    ctx.seq_len = seq_len


def _fc_backward(ctx, g_out, g_Y, g_wc, g_ws):
    tok, ids, E_tok, E_byte, W, w_c, Y, ws, ttb, next_tok = ctx.saved_tensors
    gt, gb, gW = torch.ops.mot_b200.embed_byte_fc_bwd(g_out, tok, ids, E_tok, E_byte, W, w_c, Y, ws, *ctx.cfg, ttb,
                                                      ctx.seq_len, next_tok)
    return None, None, gt, gb, gW, None, None, None, None, None, None, None


embed_byte_fc_op.register_autograd(_fc_backward, setup_context=_fc_setup)


# ---------------------------------------------------------------------------------------------------------------
# integer half and the output-side expand
# ---------------------------------------------------------------------------------------------------------------
@torch.library.custom_op("mot_b200::ttb_expand", mutates_args=(), device_types="cuda")
def ttb_expand_op(tok: Tensor, ttb: Tensor, out_i64: bool) -> Tensor:
    """-> [n, bpt] int64 / int32 (tokens_to_bytes, spt/data_creation.py:61-67)."""
    return O._ttb_expand_impl(tok, ttb, torch.int64 if out_i64 else torch.int32)


@ttb_expand_op.register_fake
def _(tok, ttb, out_i64):
    return tok.new_empty((tok.numel(), ttb.shape[1]), dtype=torch.int64 if out_i64 else torch.int32)


@torch.library.custom_op("mot_b200::pull", mutates_args=(), device_types="cuda")
def pull_op(byte_tensor: Tensor, bpt: int, pad_byte: int, eot_byte: int, from_right: bool) -> Tensor:
    return O._pull_impl(byte_tensor, bpt, pad_byte, eot_byte, from_right)


@pull_op.register_fake
def _(byte_tensor, bpt, pad_byte, eot_byte, from_right):
    return torch.empty_like(byte_tensor)


@torch.library.custom_op("mot_b200::tokens_to_digits", mutates_args=(), device_types="cuda")
def tokens_to_digits_op(tok: Tensor, dpt: int, op_token: int, eq_token: int, pad_token: int, out_i64: bool) -> Tensor:
    return O._tokens_to_digits_impl(tok, dpt, op_token, eq_token, pad_token, torch.int64 if out_i64 else torch.int32)


@tokens_to_digits_op.register_fake
def _(tok, dpt, op_token, eq_token, pad_token, out_i64):
    return tok.new_empty((tok.numel() * dpt,), dtype=torch.int64 if out_i64 else torch.int32)


@torch.library.custom_op("mot_b200::mixout_copy", mutates_args=(), device_types="cuda")
def mixout_copy_op(x: Tensor, bpt: int) -> Tensor:
    """[rows, D] -> [rows*bpt, D]: every row repeated bpt times (ByteMixoutCopy, spt/train_gpt.py:493)."""
    return O._mixout_copy_impl(x, bpt, backward=False)


@mixout_copy_op.register_fake
def _(x, bpt):
    return x.new_empty((x.shape[0] * bpt, x.shape[1]))


@torch.library.custom_op("mot_b200::mixout_copy_bwd", mutates_args=(), device_types="cuda")
def mixout_copy_bwd_op(grad_y: Tensor, bpt: int) -> Tensor:
    return O._mixout_copy_impl(grad_y, bpt, backward=True)


@mixout_copy_bwd_op.register_fake
def _(grad_y, bpt):
    return grad_y.new_empty((grad_y.shape[0] // bpt, grad_y.shape[1]))


def _mixout_setup(ctx, inputs, output):
    ctx.bpt = inputs[1]


def _mixout_backward(ctx, g):
    return torch.ops.mot_b200.mixout_copy_bwd(g.contiguous(), ctx.bpt), None


mixout_copy_op.register_autograd(_mixout_backward, setup_context=_mixout_setup)
