"""Functional API over libmot_b200.so: ttb expansion and the fused byte-mix
embedding with autograd.  Tensors must live on a CUDA (B200) device; CPU tensors
raise -- there is no fallback path."""
from __future__ import annotations

import dataclasses
from typing import Optional

import torch

from torch._subclasses.fake_tensor import FakeTensor

from . import _lib as L

FP32_EPS = float(torch.finfo(torch.float32).eps)  # F.rms_norm's default eps (train_gpt.py:172-173)

_COMBINE = {"add": L.ADD, "concat": L.CONCAT, "tok_only": L.TOK_ONLY, "bytes_only": L.BYTES_ONLY, "mean": L.MEAN}
_DTYPE = {torch.bfloat16: L.BF16, torch.float32: L.F32}
_TTB_DTYPE = {torch.int16: L.TTB_I16, torch.float32: L.TTB_F32, torch.bfloat16: L.TTB_BF16}


@dataclasses.dataclass(frozen=True)
class MixSpec:
    """Which member of the mixin catalogue (SURVEY.md 2.4) the fused kernel computes."""
    combine: str = "add"          # add | concat | tok_only | bytes_only | mean
    tok_norm: bool = False        # rms_norm(E_tok[tok])            runs/7:317
    byte_norm: bool = False       # rms_norm(E_byte[id]) per byte   runs/7:318
    out_norm: bool = True         # rms_norm(mixed row)             runs/71:230
    bytes_first: bool = False     # concat order [bytes | tok]      mathblations/model.py:267
    slot_major: bool = False      # byte ids are [bpt, T]           runs/71:479
    ttb_scramble: bool = False    # ids from ttb with the `.view(bpt,-1)` index map
    ttb_pull: bool = False        # ids from ttb: the pulled ids of pull_from_left over rows of seq_len tokens
    eps: float = FP32_EPS
    ttb_pull_side: str = "left"   # with ttb_pull: "left" (pull_from_left) or "right" (pull_from_right)

    def __post_init__(self):
        if self.ttb_pull_side not in ("left", "right"):
            raise ValueError(f"ttb_pull_side must be 'left' or 'right', got {self.ttb_pull_side!r}")


def _require_cuda(*tensors) -> torch.device:
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("mot_b200: tensors must be on a CUDA device (no CPU fallback)")
        if dev is not None and t.device != dev:
            raise RuntimeError("mot_b200: tensors are on different devices")
        dev = t.device
    return dev


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


_ABSENT = torch.empty(0)   # placeholder for "no tensor" in save_for_backward (one object, not one allocation per call)
_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)   # the cudaStream_t itself, no Stream object built


def _stream(dev) -> int:
    """cudaStream_t of torch's current stream on `dev` (called several times per step: torch.cuda.current_stream()
    costs ~15 us of host time per call, the raw getter well under one)."""
    if _raw_stream is not None and dev.index is not None:
        return _raw_stream(dev.index)
    return torch.cuda.current_stream(dev).cuda_stream


class _on_device:
    """`with torch.cuda.device(dev)` only when dev is not already current (the common case costs one integer compare)."""
    __slots__ = ("dev", "prev")

    def __init__(self, dev):
        self.dev = dev

    def __enter__(self):
        self.prev = torch.cuda.current_device()
        if self.dev.index is not None and self.dev.index != self.prev:
            torch.cuda.set_device(self.dev)
        else:
            self.prev = -1

    def __exit__(self, *exc):
        if self.prev >= 0:
            torch.cuda.set_device(self.prev)
        return False


def _ttb_expand_impl(tok: torch.Tensor, ttb: torch.Tensor, out_dtype: torch.dtype) -> torch.Tensor:
    dev = tok.device
    V, bpt = ttb.shape
    n = tok.numel()
    out = torch.empty((n, bpt), dtype=out_dtype, device=dev)
    with _on_device(dev):
        rc = L.lib().mot_ttb_expand(_ptr(tok), n, _ptr(ttb), V, bpt, _TTB_DTYPE[ttb.dtype], _ptr(out),
                                    1 if out_dtype == torch.int64 else 0, _stream(dev))
    L.check(rc, "mot_ttb_expand")
    return out


def ttb_expand(tokens: torch.Tensor, ttb: torch.Tensor, out_dtype: torch.dtype = torch.int64) -> torch.Tensor:
    """tokens_to_bytes (spt/data_creation.py:61-67): [B,T] -> [B, T*bpt], [T] -> [1, T*bpt].

    `ttb` is the [V, bpt] table: int16 (native) or the reference's float containers (fp32
    nn.Embedding weight, or the bf16-cast weight of the runs with its id-rounding quirk)."""
    _require_cuda(tokens, ttb)
    if ttb.dtype not in _TTB_DTYPE or ttb.dim() != 2:
        raise NotImplementedError(f"mot_b200.ttb_expand: ttb must be a 2-D int16/float32/bfloat16 table, got {ttb.dtype}")
    if out_dtype not in (torch.int64, torch.int32):
        raise NotImplementedError("mot_b200.ttb_expand: out_dtype must be int64 or int32")
    tok = tokens.to(torch.int32).contiguous().reshape(-1)
    ttb = ttb.contiguous()
    if _custom_ops_wanted():
        out = torch.ops.mot_b200.ttb_expand(tok, ttb, out_dtype == torch.int64)
    else:
        out = _ttb_expand_impl(tok, ttb, out_dtype)
    if tokens.dim() == 2:
        return out.view(tokens.shape[0], -1)
    return out.view(1, -1)


def _tokens_to_digits_impl(t: torch.Tensor, dpt: int, op_token: int, eq_token: int, pad_token: int,
                           out_dtype: torch.dtype) -> torch.Tensor:
    dev = t.device
    out = torch.empty(t.numel() * dpt, dtype=out_dtype, device=dev)
    with _on_device(dev):
        rc = L.lib().mot_tokens_to_digits(_ptr(t), t.numel(), 1 if t.dtype == torch.int64 else 0, dpt,
                                          op_token, eq_token, pad_token, _ptr(out), 1 if out_dtype == torch.int64 else 0,
                                          _stream(dev))
    L.check(rc, "mot_tokens_to_digits")
    return out


def tokens_to_digits(tokens: torch.Tensor, max_digits_per_token: int, op_token: int, eq_token: int, pad_token: int,
                     out_dtype: torch.dtype = torch.int64) -> torch.Tensor:
    """GenerateEquations.tokens_to_digits (mathblations/data.py:92-109) on the device: [n] -> [n * dpt]."""
    _require_cuda(tokens)
    if tokens.dtype not in (torch.int32, torch.int64) or out_dtype not in (torch.int32, torch.int64):
        raise NotImplementedError("mot_b200.tokens_to_digits: int32 / int64 only")
    t = tokens.reshape(-1).contiguous()
    if _custom_ops_wanted():
        return torch.ops.mot_b200.tokens_to_digits(t, max_digits_per_token, op_token, eq_token, pad_token,
                                                   out_dtype == torch.int64)
    return _tokens_to_digits_impl(t, max_digits_per_token, op_token, eq_token, pad_token, out_dtype)


def _pull_impl(x: torch.Tensor, bytes_per_token: int, pad_byte: int, eot_byte: int, from_right: bool) -> torch.Tensor:
    dev = x.device
    B, TB = x.shape
    out = torch.empty_like(x)
    T = TB // bytes_per_token
    if B * T == 0:
        return out
    ws = torch.empty(int(L.lib().mot_pull_workspace_bytes(B, T, bytes_per_token)), dtype=torch.uint8, device=dev)
    with _on_device(dev):
        rc = L.lib().mot_pull(_ptr(x), _ptr(out), B, T, bytes_per_token, 1 if x.dtype == torch.int64 else 0, pad_byte,
                              eot_byte, 1 if from_right else 0, _ptr(ws), ws.numel(), _stream(dev))
    L.check(rc, "mot_pull")
    return out


def _pull(byte_tensor: torch.Tensor, bytes_per_token: int, pad_byte: int, eot_byte: int, from_right: bool) -> torch.Tensor:
    _require_cuda(byte_tensor)
    if byte_tensor.dtype not in (torch.int32, torch.int64) or byte_tensor.dim() != 2:
        raise NotImplementedError("mot_b200.pull: byte_tensor must be a 2-D int32 / int64 tensor [B, T*bpt]")
    if byte_tensor.shape[1] % bytes_per_token:
        raise RuntimeError("T must be divisible by bytes_per_token")   # the reference's assert (data_creation.py:189)
    x = byte_tensor.contiguous()
    if _custom_ops_wanted():
        return torch.ops.mot_b200.pull(x, bytes_per_token, pad_byte, eot_byte, from_right)
    return _pull_impl(x, bytes_per_token, pad_byte, eot_byte, from_right)


def pull_from_left(byte_tensor: torch.Tensor, bytes_per_token: int, pad_byte: int = 456, eot_byte: int = 457) -> torch.Tensor:
    """spt/data_creation.py:179-305 (== runs/7:351-428), same signature: every non-EOT token receives the last
    bytes_per_token non-pad bytes of its segment up to and including itself, right-aligned.  No host syncs."""
    return _pull(byte_tensor, bytes_per_token, pad_byte, eot_byte, False)


def pull_from_right(byte_tensor: torch.Tensor, bytes_per_token: int, pad_byte: int = 456, eot_byte: int = 457) -> torch.Tensor:
    """spt/data_creation.py:71-176: the first bytes_per_token non-pad bytes of tokens t, t+1, ... before the next EOT."""
    return _pull(byte_tensor, bytes_per_token, pad_byte, eot_byte, True)


PAD_ID, EOT_ID = 456, 457   # pad and end-of-text byte of the ttb tables (spt/data_creation.py; pull_from_left's defaults)


def _pull_flags(side: str, next_tok: bool) -> int:
    """MOT_F_TTB_PULL_LEFT / _RIGHT (+ MOT_F_TTB_NEXT_TOK: the lookahead tail after the token ids) of a pull from `side`."""
    if side == "left":
        return L.F_TTB_PULL_LEFT
    return L.F_TTB_PULL_RIGHT | (L.F_TTB_NEXT_TOK if next_tok else 0)


def make_desc(spec: MixSpec, n_tokens: int, E_tok, E_byte, bpt: int, *, ids: Optional[torch.Tensor],
              ttb: Optional[torch.Tensor], has_lam: bool, seq_len: int = 0, row_stride: int = 0,
              col_offset: int = 0, dp_slabs: int = 0, pad_id: int = PAD_ID, eot_id: int = EOT_ID,
              next_tok: bool = False) -> L.MotDesc:
    ref = E_tok if E_tok is not None else E_byte
    if ref.dtype not in _DTYPE:
        raise NotImplementedError(f"mot_b200: embedding dtype {ref.dtype} is not supported (bf16 / fp32 only)")
    if spec.combine not in _COMBINE:
        raise NotImplementedError(f"mot_b200: unknown combine mode {spec.combine!r}")
    has_tok, has_bytes = spec.combine != "bytes_only", spec.combine != "tok_only"
    Dt = E_tok.shape[1] if has_tok else 0
    bd = E_byte.shape[1] if has_bytes else 0
    if spec.combine in ("add", "tok_only", "mean"):
        Do = Dt
    elif spec.combine == "concat":
        Do = Dt + bpt * bd
    else:
        Do = bpt * bd
    flags = 0
    flags |= L.F_TOK_NORM if spec.tok_norm else 0
    flags |= L.F_BYTE_NORM if spec.byte_norm else 0
    flags |= L.F_OUT_NORM if spec.out_norm else 0
    flags |= L.F_BYTES_FIRST if spec.bytes_first else 0
    flags |= L.F_HAS_LAMBDAS if has_lam else 0
    ttb_dtype = 0
    if has_bytes:
        if ids is None:
            flags |= L.F_IDS_FROM_TTB
            flags |= L.F_TTB_SCRAMBLE if spec.ttb_scramble else 0
            flags |= _pull_flags(spec.ttb_pull_side, next_tok) if spec.ttb_pull else 0
            ttb_dtype = _TTB_DTYPE[ttb.dtype]
        else:
            flags |= L.F_SLOT_MAJOR if spec.slot_major else 0
            flags |= L.F_IDS_I64 if ids.dtype == torch.int64 else 0
    # without a token table the token ids still index the ttb table when the kernels derive the byte ids from it
    tok_vocab = E_tok.shape[0] if has_tok else (ttb.shape[0] if has_bytes and ids is None else 0)
    return L.MotDesc(L.ABI_VERSION, _DTYPE[ref.dtype], n_tokens, seq_len,
                     tok_vocab, E_byte.shape[0] if has_bytes else 0, bpt if has_bytes else 0,
                     Dt, bd, Do, _COMBINE[spec.combine], flags, ttb_dtype, spec.eps, row_stride, col_offset, dp_slabs,
                     pad_id, eot_id)


def embed_forward_out(desc: L.MotDesc, tok, ids, ttb, E_tok, E_byte, lam, out, stream: Optional[int] = None,
                      rstd: Optional[torch.Tensor] = None, addend: Optional[torch.Tensor] = None) -> None:
    """mot_embed_fwd on caller-allocated tensors (no allocation, no sync; CUDA-graph capturable).  `rstd` (fp32
    [n_tokens]) additionally keeps the reciprocal rms of every mixed row for the saved-output backward; `addend`
    ([n_tokens, out_dim]) is added to the mixed row before the output norm (mot_embed_fwd_ex)."""
    dev = out.device
    with _on_device(dev):
        if rstd is None and addend is None:
            rc = L.lib().mot_embed_fwd(desc, _ptr(tok), _ptr(ids), _ptr(ttb), _ptr(E_tok), _ptr(E_byte), _ptr(lam),
                                       _ptr(out), _stream(dev) if stream is None else stream)
        else:
            rc = L.lib().mot_embed_fwd_ex(desc, _ptr(tok), _ptr(ids), _ptr(ttb), _ptr(E_tok), _ptr(E_byte), _ptr(lam),
                                          _ptr(addend), _ptr(out), _ptr(rstd), _stream(dev) if stream is None else stream)
    L.check(rc, "mot_embed_fwd")


def embed_bwd_uses_saved(desc: L.MotDesc) -> bool:
    """Whether mot_embed_bwd_ex would read the kept forward result for this descriptor (MoT-sum, moderate N)."""
    return bool(L.lib().mot_embed_bwd_uses_saved(desc))


def embed_workspace_bytes(desc: L.MotDesc) -> int:
    return int(L.lib().mot_embed_workspace_bytes(desc))


def embed_workspace_init(desc: L.MotDesc, ws) -> None:
    """Zero the head of a fresh workspace once; afterwards every completed backward leaves it clean (MOT_WS_CLEAN)."""
    dev = ws.device
    with _on_device(dev):
        rc = L.lib().mot_embed_workspace_init(desc, _ptr(ws), ws.numel(), _stream(dev))
    L.check(rc, "mot_embed_workspace_init")


def embed_plan(desc: L.MotDesc, tok, ws, ws_clean: bool = False) -> None:
    dev = ws.device
    with _on_device(dev):
        rc = L.lib().mot_embed_plan(desc, _ptr(tok), _ptr(ws), ws.numel(), L.WS_CLEAN if ws_clean else 0, _stream(dev))
    L.check(rc, "mot_embed_plan")


def embed_backward_out(desc: L.MotDesc, tok, ids, ttb, E_tok, E_byte, lam, grad_out, gE_tok, gE_byte, g_lam, ws,
                       plan_ready: bool = False, ws_clean: bool = False, stream: Optional[int] = None,
                       out_saved: Optional[torch.Tensor] = None, rstd: Optional[torch.Tensor] = None,
                       addend: Optional[torch.Tensor] = None, d_addend: Optional[torch.Tensor] = None,
                       plan_joined: bool = False) -> None:
    """mot_embed_bwd on caller-allocated tensors; gE_tok / gE_byte are fully overwritten.  `ws_clean`: the caller
    vouches that the head of `ws` is zero (fresh from embed_workspace_init or left by a completed backward).
    `plan_joined`: the plan ran on the side stream and this stream waited for its event (MOT_WS_PLAN_JOINED).
    `out_saved` + `rstd` (what embed_forward_out(..., rstd=) produced) and `addend` / `d_addend`: mot_embed_bwd_ex."""
    dev = grad_out.device
    flags = (L.WS_PLAN_READY if plan_ready else 0) | (L.WS_CLEAN if ws_clean else 0) | \
        (L.WS_PLAN_JOINED if plan_ready and plan_joined else 0)
    with _on_device(dev):
        if (out_saved is None or rstd is None) and addend is None and d_addend is None:
            rc = L.lib().mot_embed_bwd(desc, _ptr(tok), _ptr(ids), _ptr(ttb), _ptr(E_tok), _ptr(E_byte), _ptr(lam),
                                       _ptr(grad_out), _ptr(gE_tok), _ptr(gE_byte), _ptr(g_lam), _ptr(ws), ws.numel(),
                                       flags, _stream(dev) if stream is None else stream)
        else:
            rc = L.lib().mot_embed_bwd_ex(desc, _ptr(tok), _ptr(ids), _ptr(ttb), _ptr(E_tok), _ptr(E_byte), _ptr(lam),
                                          _ptr(addend), _ptr(grad_out), _ptr(out_saved), _ptr(rstd), _ptr(gE_tok),
                                          _ptr(gE_byte), _ptr(g_lam), _ptr(d_addend), _ptr(ws), ws.numel(), flags,
                                          _stream(dev) if stream is None else stream)
    L.check(rc, "mot_embed_bwd")


def embed_backward_slab_out(desc: L.MotDesc, tok, ids, ttb, E_tok, E_byte, lam, grad_out, out_saved, rstd, gE_tok, gE_byte,
                            g_lam, ws, slab: int, n_slabs: int, *, reserve_sms: int = 0, plan_ready: bool = True,
                            ws_clean: bool = True, plan_joined: bool = False, stream: Optional[int] = None) -> None:
    """mot_embed_bwd_slab: slab `slab` of `n_slabs` of the backward (rows slab_rows(...) of gE_tok are final once its
    kernels have run; gE_byte / g_lam after the last slab).  desc must have been made with dp_slabs=n_slabs."""
    dev = grad_out.device
    flags = (L.WS_PLAN_READY if plan_ready else 0) | (L.WS_CLEAN if ws_clean else 0) | \
        (L.WS_PLAN_JOINED if plan_ready and plan_joined else 0)
    with _on_device(dev):
        rc = L.lib().mot_embed_bwd_slab(desc, _ptr(tok), _ptr(ids), _ptr(ttb), _ptr(E_tok), _ptr(E_byte), _ptr(lam),
                                        _ptr(grad_out), _ptr(out_saved), _ptr(rstd), _ptr(gE_tok), _ptr(gE_byte), _ptr(g_lam),
                                        _ptr(ws), ws.numel(), flags, slab, n_slabs, reserve_sms,
                                        _stream(dev) if stream is None else stream)
    L.check(rc, "mot_embed_bwd_slab")


def slab_rows(tok_vocab: int, slab: int, n_slabs: int):
    """Rows [lo, hi) of the token table that slab `slab` of `n_slabs` owns (mot_embed_slab_rows)."""
    import ctypes as C
    lo, hi = C.c_int32(), C.c_int32()
    L.check(L.lib().mot_embed_slab_rows(tok_vocab, slab, n_slabs, C.byref(lo), C.byref(hi)), "mot_embed_slab_rows")
    return lo.value, hi.value


class Workspace:
    """A backward workspace that remembers whether the library left it clean (so the steady-state step needs no
    memset), plus the fork / join events of the plan that runs on the side stream.  Instances are recycled through a
    pool per (device, table geometry)."""

    def __init__(self, key, dev):
        self.key = key
        self.buf: Optional[torch.Tensor] = None
        self.clean = False
        self.ev_fork, self.ev_join = torch.cuda.Event(), torch.cuda.Event()
        cur = torch.cuda.current_stream(dev)
        self.ev_fork.record(cur)   # materialise the cudaEvent_t handles
        self.ev_join.record(cur)
        self.pending = False       # a plan was launched on the side stream and no backward has consumed it yet

    def reserve(self, desc: L.MotDesc, dev) -> torch.Tensor:
        need = embed_workspace_bytes(desc)
        if self.buf is None or self.buf.numel() < need or self.buf.device != dev:
            self.buf = torch.empty(need, dtype=torch.uint8, device=dev)
            self.clean = False
        return self.buf

    def take_clean(self) -> bool:
        """Whether the head of buf is zero; the buffer counts as dirty until a completed backward marks it clean."""
        clean, self.clean = self.clean, False
        return clean

    def __del__(self):   # dropped with a plan in flight (forward without backward): keep the allocator off the buffer
        try:
            if self.pending and self.buf is not None:
                self.buf.record_stream(side_stream(self.buf.device))
        except Exception:
            pass


_WS_POOL: dict = {}
_SIDE_STREAMS: dict = {}


def acquire_workspace(desc: L.MotDesc, dev) -> Workspace:
    # the zeroed head of the workspace (histogram | byte accumulators | one fp32 slot per stream chunk) is laid out by the
    # table geometry AND by (n_tokens, tok_dim): a buffer is only "clean" for the exact layout it was last used with
    key = (dev.index, desc.tok_vocab, desc.byte_vocab, desc.byte_dim, desc.combine, desc.n_tokens, desc.tok_dim, desc.dp_slabs)
    free = _WS_POOL.get(key)
    if free is None:
        free = _WS_POOL[key] = []
    ws = free.pop() if free else Workspace(key, dev)
    ws.reserve(desc, dev)
    return ws


def release_workspace(ws: Workspace) -> None:
    free = _WS_POOL.setdefault(ws.key, [])
    if len(free) < 4:
        free.append(ws)


def side_stream(dev) -> torch.cuda.Stream:
    """Per-device stream on which the backward plan (a counting sort of the token ids) runs beside the forward."""
    st = _SIDE_STREAMS.get(dev.index)
    if st is None:
        st = _SIDE_STREAMS[dev.index] = torch.cuda.Stream(device=dev)
    return st


def embed_plan_async(desc: L.MotDesc, tok, ws: Workspace, dev, stream: Optional[int] = None) -> None:
    """mot_embed_plan_async: fork from the current stream, run the plan on the side stream, record ws.ev_join.  The
    backward waits for it with embed_plan_join()."""
    clean = ws.take_clean()
    with _on_device(dev):
        rc = L.lib().mot_embed_plan_async(desc, _ptr(tok), _ptr(ws.buf), ws.buf.numel(), L.WS_CLEAN if clean else 0,
                                          _stream(dev) if stream is None else stream, side_stream(dev).cuda_stream,
                                          ws.ev_fork.cuda_event, ws.ev_join.cuda_event)
    L.check(rc, "mot_embed_plan_async")
    ws.pending = True


def embed_plan_join_if_capturing(ws: Optional[Workspace], dev, stream: Optional[int] = None) -> None:
    """Inside a CUDA-graph capture (torch.cuda.graph / make_graphed_callables) the side stream must rejoin before the
    capture of the forward ends; the graph keeps plan and forward concurrent.  Called by every forward that forked."""
    if ws is not None and ws.pending and torch.cuda.is_current_stream_capturing():
        embed_plan_join(ws, dev, stream)


def embed_plan_join(ws: Workspace, dev, stream: Optional[int] = None) -> None:
    rc = L.lib().mot_stream_wait_event(_stream(dev) if stream is None else stream, ws.ev_join.cuda_event)
    L.check(rc, "mot_stream_wait_event")
    ws.pending = False


def _planned_workspace(desc: L.MotDesc, tok, dev, stream: Optional[int] = None) -> Workspace:
    """A pooled workspace with the backward's sort plan of `tok` started on the side stream, beside the forward."""
    ws = acquire_workspace(desc, dev)
    embed_plan_async(desc, tok, ws, dev, stream)
    return ws


def _take_workspace(ws: Optional[Workspace], desc: L.MotDesc, dev, stream: Optional[int] = None):
    """The workspace of an eager backward -> (ws, plan_ready, ws_clean): the one its forward planned in (joined here
    unless a captured forward joined at its own end), else one from the pool.  Hand it back with _return_workspace."""
    if ws is None:
        ws = acquire_workspace(desc, dev)
        return ws, False, ws.take_clean()
    if ws.pending:
        embed_plan_join(ws, dev, stream)
    return ws, True, True     # the plan ran on a clean (or freshly cleared) workspace and leaves it clean


def _return_workspace(ws: Workspace) -> None:
    ws.clean = True           # every completed backward leaves the head of the workspace zeroed
    release_workspace(ws)


# ------------------------------------------------------------------------------------------------------------
# argument checks shared by both dispatch paths (autograd.Function and torch.ops.mot_b200)
# ------------------------------------------------------------------------------------------------------------
def _tok_i32(tokens: torch.Tensor) -> torch.Tensor:
    """Token ids as the kernels read them: flat, contiguous int32."""
    tok = tokens.reshape(-1)
    return (tok if tok.dtype == torch.int32 else tok.to(torch.int32)).contiguous()


def _id_args(spec: MixSpec, bpt: int, tokens, byte_ids, ttb, seq_len: int, next_tokens, byte_ids2=None,
             ttb_pair: bool = False):
    """Where the byte ids of a front come from, checked once for every front -> (tok, ids, ids2, ttb, next_tok).

    Explicit `byte_ids` (with `byte_ids2`: the second id tensor of `--add-padded-and-pulled`), or byte_ids=None with the
    [V, bpt] table `ttb`: the kernels derive the padded ids, the pulled ones under spec.ttb_pull, both sets with ttb_pair.
    next_tokens (a right pull's lookahead) comes back with tok as views of ONE int32 buffer [tok | next], so that the
    kernels find token seq_len of row r at tok[n + r] (MOT_F_TTB_NEXT_TOK) while the plan and the gathers see n tokens."""
    tok = _tok_i32(tokens) if tokens is not None else None
    if byte_ids is None and ttb is None and spec.combine != "tok_only":
        raise RuntimeError("mot_b200: need byte ids or a ttb table")
    pull = spec.ttb_pull or ttb_pair
    if next_tokens is not None and (tok is None or byte_ids is not None or ttb is None or not pull
                                    or spec.ttb_pull_side != "right"):
        raise RuntimeError("mot_b200: next_tokens= is the lookahead of a right pull (ttb ids with ttb_pull_side='right')")
    pair = ttb_pair if byte_ids is None else byte_ids2 is not None
    if pair and (not spec.byte_norm or spec.slot_major or spec.bytes_first or (ttb_pair and spec.ttb_scramble)):
        raise NotImplementedError("mot_b200: the padded+pulled sum exists only with per-byte norms, token-major "
                                  "ids and [tok | bytes] order (spt/train_gpt.py:371-379,442-443)")
    if byte_ids is not None:
        if byte_ids.dtype not in (torch.int32, torch.int64):
            raise NotImplementedError("mot_b200: byte ids must be int32 or int64")
        ids = byte_ids.contiguous()
        n = tok.numel() if tok is not None else ids.numel() // bpt
        if ids.numel() != n * bpt:
            raise RuntimeError(f"mot_b200: byte ids have {ids.numel()} entries, expected {n}*{bpt}")
        ids2 = byte_ids2.contiguous() if pair else None
        if pair and (ids2.dtype != ids.dtype or ids2.numel() != ids.numel()):
            raise RuntimeError("mot_b200: the two byte-id tensors must share dtype and size")
        return tok, ids, ids2, None, None
    if ttb is None:
        return tok, None, None, None, None
    if ttb.dtype not in _TTB_DTYPE or ttb.dim() != 2:
        raise NotImplementedError(f"mot_b200: ttb must be a 2-D int16/float32/bfloat16 table, got {ttb.dtype}")
    if pull and (seq_len <= 0 or tok.numel() % seq_len):
        raise RuntimeError(f"mot_b200: pulled ids need rows of seq_len tokens (seq_len={seq_len}, {tok.numel()} tokens)")
    if next_tokens is None:
        return tok, None, None, ttb.contiguous(), None
    if next_tokens.dtype not in (torch.int32, torch.int64):
        raise NotImplementedError("mot_b200: next_tokens must be int32 or int64")
    n, rows = tok.numel(), tok.numel() // seq_len
    if next_tokens.numel() != rows:
        raise RuntimeError(f"mot_b200: next_tokens has {next_tokens.numel()} entries, expected one per row ({rows})")
    buf = torch.cat((tok, next_tokens.reshape(-1).to(torch.int32)))
    return buf[:n], None, None, ttb.contiguous(), buf[n:]


def _tok_next(tok: torch.Tensor, next_tok: Optional[torch.Tensor]) -> torch.Tensor:
    """Token ids whose lookahead follows them in memory (the operators receive tok and next_tok as two tensors; _id_args
    made them views of one buffer, which a traced graph may not keep).  A fake tensor only carries its shape."""
    if next_tok is None or next_tok.numel() == 0 or isinstance(tok, FakeTensor):
        return tok
    if next_tok.data_ptr() == tok.data_ptr() + 4 * tok.numel():
        return tok
    return torch.cat((tok, next_tok))[:tok.numel()]


def _ids_desc(spec: MixSpec, bpt: int, seq_len: int, tok, next_tok, ids, ttb, E_tok, E_byte, has_lam: bool = False,
              row_stride: int = 0, col_offset: int = 0):
    """-> (tok, desc): the descriptor of the gather that reads the byte ids (explicit `ids`, else derived from `ttb` over
    rows of seq_len tokens, with the lookahead next_tok behind tok); tok with next_tok behind it in memory."""
    tok = _tok_next(tok, next_tok)
    n = tok.numel() if tok is not None else ids.numel() // bpt
    return tok, make_desc(spec, n, E_tok, E_byte, bpt, ids=ids, ttb=ttb, has_lam=has_lam, seq_len=seq_len,
                          row_stride=row_stride, col_offset=col_offset, next_tok=next_tok is not None)


def _require_chain_dtype(E_tok: torch.Tensor, E_byte: torch.Tensor) -> None:
    """The projection chains compute in the table dtype: bf16, or fp32 on the TF32 tensor-core path."""
    if E_tok.dtype not in (torch.bfloat16, torch.float32) or E_byte.dtype != E_tok.dtype:
        raise NotImplementedError("mot_b200: token and byte tables must both be bf16 or both fp32")


def _embed_args(spec: MixSpec, bpt: int, tokens, byte_ids, ttb, E_tok, E_byte, lam, seq_len: int, next_tokens):
    """mot_embed's arguments checked and normalised -> (dev, tok, ids, ttb, E_tok, E_byte, next_tok)."""
    dev = _require_cuda(tokens, byte_ids, ttb, E_tok, E_byte, lam, next_tokens)
    tok, ids, _, ttb, nxt = _id_args(spec, bpt, tokens, byte_ids, ttb, seq_len, next_tokens)
    E_tok = E_tok.contiguous() if E_tok is not None else None
    E_byte = E_byte.contiguous() if E_byte is not None else None
    if E_tok is not None and E_byte is not None and E_tok.dtype != E_byte.dtype:
        raise NotImplementedError("mot_b200: token and byte tables must share one dtype")
    return dev, tok, ids, ttb, E_tok, E_byte, nxt


class _MotEmbedFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, desc: L.MotDesc, dev, tok, ids, ttb, E_tok, E_byte, lam, grad_bufs=None):
        # optional ((param_tok, view_tok), (param_byte, view_byte)): views of a dp.GradBucket that become param.grad
        ctx.grad_bufs = grad_bufs
        lam_c = lam.detach().to(torch.float32).contiguous() if lam is not None else None
        n = desc.n_tokens
        # data-parallel pipeline: a bucket that holds exactly [token table | byte table] in symmetric memory lets the
        # backward run as vocabulary slabs with the exchange of slab k beside the backward of slab k + 1
        ctx.dp_bucket = None
        bucket = grad_bufs[2] if grad_bufs is not None and len(grad_bufs) > 2 else None
        if bucket is not None and bucket.pipelined and n > 0 and E_tok is not None and E_byte is not None \
                and len(bucket.params) == 2 and bucket.params[0] is grad_bufs[0][0] and bucket.params[1] is grad_bufs[1][0] \
                and bool(L.lib().mot_embed_bwd_uses_saved(desc)):
            desc = L.MotDesc.from_buffer_copy(desc)
            desc.dp_slabs = bucket.n_slabs
            ctx.dp_bucket = bucket
        ref = E_tok if E_tok is not None else E_byte
        out = torch.empty((n, desc.out_dim), dtype=ref.dtype, device=dev)
        # the backward needs the positions grouped by token id: start that sort now, beside the forward kernel
        st = _stream(dev)
        needs_grad = any(ctx.needs_input_grad[5:8])   # E_tok, E_byte, lam
        ctx.ws = _planned_workspace(desc, tok, dev, st) if needs_grad and tok is not None and n > 0 else None
        # MoT-sum (runs/71): keep what rms_norm's autograd node keeps (its result and rstd); the backward then reads two
        # rows per occurrence instead of rebuilding the mixed row (mot_embed_bwd_ex)
        keep = needs_grad and n > 0 and bool(L.lib().mot_embed_bwd_uses_saved(desc))
        rstd = torch.empty(n, dtype=torch.float32, device=dev) if keep else None
        embed_forward_out(desc, tok, ids, ttb, E_tok, E_byte, lam_c, out, st, rstd=rstd)
        embed_plan_join_if_capturing(ctx.ws, dev, st)
        ctx.desc, ctx.dev = desc, dev
        saved = (tok, ids, ttb, E_tok, E_byte, lam_c, out if keep else None, rstd)
        ctx.save_for_backward(*[t if t is not None else _ABSENT for t in saved])
        ctx.present = [t is not None for t in saved]
        ctx.lam_dtype = lam.dtype if lam is not None else None
        return out

    @staticmethod
    def backward(ctx, grad_out):
        saved = [t if ok else None for t, ok in zip(ctx.saved_tensors, ctx.present)]
        tok, ids, ttb, E_tok, E_byte, lam, out_saved, rstd = saved
        desc, dev = ctx.desc, ctx.dev
        g = grad_out.contiguous()
        if g.dtype != (E_tok if E_tok is not None else E_byte).dtype:
            g = g.to((E_tok if E_tok is not None else E_byte).dtype)
        direct = [None, None]
        if ctx.grad_bufs is not None:
            # the kernels overwrite every row, so they can write straight into the caller's flat bucket; the view is
            # installed as param.grad here (autograd would clone a view).  With a gradient already accumulated on the
            # parameter the normal path is taken and autograd adds to it.
            for i, (pv, E) in enumerate(zip(ctx.grad_bufs, (E_tok, E_byte))):
                if pv is not None and E is not None and pv[0].grad is None:
                    view = pv[1]
                    if view.dtype != E.dtype or view.shape != E.shape or not view.is_contiguous() or view.device != E.device:
                        raise TypeError("mot_b200: the gradient-bucket view of a table must match its dtype, shape and "
                                        f"device and be contiguous (table {tuple(E.shape)} {E.dtype}, view "
                                        f"{tuple(view.shape)} {view.dtype})")
                    direct[i] = pv
        gE_tok = direct[0][1] if direct[0] is not None else (torch.empty_like(E_tok) if E_tok is not None else None)
        gE_byte = direct[1][1] if direct[1] is not None else (torch.empty_like(E_byte) if E_byte is not None else None)
        g_lam = torch.empty(2, dtype=torch.float32, device=dev) if lam is not None else None
        st = _stream(dev)
        ws, planned, clean = _take_workspace(ctx.ws, desc, dev, st)
        bucket = ctx.dp_bucket
        if bucket is not None and direct[0] is not None and direct[1] is not None and out_saved is not None \
                and not torch.cuda.is_current_stream_capturing():
            # slab k of the vocabulary, then its rows of the bucket go to the exchange stream while slab k + 1 is computed;
            # the byte table (finished by the last slab) travels with the last range.  bucket.all_reduce_avg() / wait() joins.
            K, V_, Dt_ = bucket.n_slabs, E_tok.shape[0], E_tok.shape[1]
            for k in range(K):
                embed_backward_slab_out(desc, tok, ids, ttb, E_tok, E_byte, lam, g, out_saved, rstd, gE_tok, gE_byte, g_lam,
                                        ws.buf, k, K, reserve_sms=bucket.reserve_sms if k > 0 else 0,
                                        plan_ready=planned or k > 0, ws_clean=clean or k > 0, plan_joined=planned, stream=st)
                lo, hi = slab_rows(V_, k, K)
                bucket.exchange_async(lo * Dt_, hi * Dt_ if k < K - 1 else bucket.flat.numel(), last=(k == K - 1))
        else:
            embed_backward_out(desc, tok, ids, ttb, E_tok, E_byte, lam, g, gE_tok, gE_byte, g_lam, ws.buf,
                               plan_ready=planned, ws_clean=clean, stream=st, out_saved=out_saved, rstd=rstd,
                               plan_joined=planned)
        if ctx.grad_bufs is not None and len(ctx.grad_bufs) > 2 and ctx.grad_bufs[0] is not None and tok is not None:
            bk, p_tok = ctx.grad_bufs[2], ctx.grad_bufs[0][0]
            if bk is not None and bk.sparse_rows and bk.is_row_table(p_tok) and not bk._pending:
                # the rows this batch gathered, also when autograd adds this gradient to an existing one: the exchange
                # moves only the union of every backward since the last exchange
                bk.mark_rows(desc, ws.buf, fresh=(p_tok,) if direct[0] is not None else ())
        ctx.ws = None
        _return_workspace(ws)
        if g_lam is not None:
            g_lam = g_lam.to(ctx.lam_dtype)
        if direct[0] is not None:
            direct[0][0].grad, gE_tok = gE_tok, None
        if direct[1] is not None:
            direct[1][0].grad, gE_byte = gE_byte, None
        return None, None, None, None, None, gE_tok, gE_byte, g_lam, None


def mot_embed(tokens: Optional[torch.Tensor], byte_ids: Optional[torch.Tensor], E_tok: Optional[torch.Tensor],
              E_byte: Optional[torch.Tensor], spec: MixSpec, *, bpt: int = 16, lam: Optional[torch.Tensor] = None,
              ttb: Optional[torch.Tensor] = None, seq_len: int = 0, grad_bufs=None,
              next_tokens: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Fused gather + pool + combine + norm.  Returns [n_tokens, out_dim] in the table dtype.

    tokens   int32/int64 [..] (flattened); byte_ids int32/int64 with n_tokens*bpt entries, token-major
    ([.., T*bpt]) or slot-major ([bpt, T], spec.slot_major); byte_ids=None derives the ids from `ttb`
    inside the kernel.  lam = float tensor [2] = (lam_tok, lam_byte) or None.  grad_bufs = optional
    ((param, view), (param, view)) pairs for the token / byte table: the backward writes the dense gradient into `view`
    (a slice of a dp.GradBucket) and installs it as `param.grad`.  next_tokens: with spec.ttb_pull and
    ttb_pull_side="right", token seq_len of every row ([n_tokens / seq_len], the last column of the loader's window of
    seq_len + 1 tokens), which the right pull of the row's last tokens reads; without it the row ends at its last input."""
    dev, tok, ids, ttb_c, E_tok_c, E_byte_c, nxt = _embed_args(spec, bpt, tokens, byte_ids, ttb, E_tok, E_byte, lam,
                                                               seq_len, next_tokens)
    if grad_bufs is None and _custom_ops_wanted():
        lam32 = lam.to(torch.float32).contiguous() if lam is not None else None   # differentiable cast
        need = torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in (E_tok, E_byte, lam))
        return torch.ops.mot_b200.embed(tok, ids, ttb_c, E_tok_c, E_byte_c, lam32, pack_spec(spec), bpt, seq_len,
                                        float(spec.eps), need, nxt)[0]
    tok, desc = _ids_desc(spec, bpt, seq_len, tok, nxt, ids, ttb_c, E_tok_c, E_byte_c, has_lam=lam is not None)
    return _MotEmbedFn.apply(desc, dev, tok, ids, ttb_c, E_tok_c, E_byte_c, lam, grad_bufs)


# ------------------------------------------------------------------------------------------------------------
# several tables gathered with the same token ids (the value embeddings, runs/7:252,308; spt/train_gpt.py:566,600)
# ------------------------------------------------------------------------------------------------------------
_GATHER_SPEC = MixSpec(combine="tok_only", out_norm=False)


def _gather_args(tokens, tables):
    """tok_gather's arguments checked and normalised -> (dev, tok, tables)."""
    dev = _require_cuda(tokens, *tables)
    if not tables:
        raise RuntimeError("mot_b200.tok_gather: need at least one table")
    shape, dtype = tables[0].shape, tables[0].dtype
    for E in tables:
        if E.shape != shape or E.dtype != dtype or E.dim() != 2:
            raise NotImplementedError("mot_b200.tok_gather: tables must share one [V, D] shape and dtype")
    return dev, _tok_i32(tokens), [E.contiguous() for E in tables]


def _gather_desc(tok, table) -> L.MotDesc:
    return make_desc(_GATHER_SPEC, tok.numel(), table, None, 0, ids=None, ttb=None, has_lam=False)


def _gather_forward(desc: L.MotDesc, tok, tables, dev, stream: Optional[int] = None):
    outs = []
    for E in tables:
        out = torch.empty((tok.numel(), E.shape[1]), dtype=E.dtype, device=dev)
        embed_forward_out(desc, tok, None, None, E, None, None, out, stream)
        outs.append(out)
    return outs


def _gather_backward(desc: L.MotDesc, tok, tables, grads, want, ws_buf, plan_ready: bool, ws_clean: bool,
                     stream: Optional[int] = None, outs=None):
    """Dense gradients of the tables whose `want` entry is true (None for the others), one scatter launch each; the
    first one finds the plan in place or builds it, and every one leaves the accumulators zeroed.  outs[i], where given,
    is the tensor table i's gradient is written into (a gradient-bucket view), else a new one."""
    gEs = []
    for i, (E, g, w) in enumerate(zip(tables, grads, want)):
        if not w:
            gEs.append(None)
            continue
        g = g.reshape(-1, E.shape[1]).to(E.dtype).contiguous()
        gE = outs[i] if outs is not None and outs[i] is not None else torch.empty_like(E)
        embed_backward_out(desc, tok, None, None, E, None, None, g, gE, None, None, ws_buf,
                           plan_ready=plan_ready, ws_clean=ws_clean, stream=stream)
        plan_ready, ws_clean = True, True
        gEs.append(gE)
    return gEs


class _TokGatherFn(torch.autograd.Function):
    """outs[i] = tables[i][tokens]: plain gathers (no norm) of same-shaped tables.  The backward needs the positions
    grouped by token id once for all tables: one sort plan (started beside the first forward gather), one scatter
    launch per table reusing it (MOT_WS_PLAN_READY); the dense gradients need no token rows (R = 0).
    grad_bucket = optional (dp.GradBucket, the table parameters): the gradient of a table the bucket holds is written
    into its bucket view, which becomes param.grad, and the rows of the batch are marked for the touched-rows exchange."""

    @staticmethod
    def forward(ctx, dev, tok, grad_bucket, *tables):
        if grad_bucket is not None:      # an output without gradient leaves its table's grad None, not a view of zeros
            ctx.set_materialize_grads(False)
        desc = _gather_desc(tok, tables[0])
        st = _stream(dev)
        ctx.ws = _planned_workspace(desc, tok, dev, st) if any(ctx.needs_input_grad[3:]) and tok.numel() > 0 else None
        outs = _gather_forward(desc, tok, tables, dev, st)
        embed_plan_join_if_capturing(ctx.ws, dev, st)
        ctx.desc, ctx.dev, ctx.grad_bucket = desc, dev, grad_bucket
        ctx.save_for_backward(tok, *tables)
        return tuple(outs)

    @staticmethod
    def backward(ctx, *grad_outs):
        tok, *Es = ctx.saved_tensors
        st = _stream(ctx.dev)
        ws, planned, clean = _take_workspace(ctx.ws, ctx.desc, ctx.dev, st)
        want = [g is not None and ctx.needs_input_grad[3 + i] for i, g in enumerate(grad_outs)]
        direct = [None] * len(Es)
        if ctx.grad_bucket is not None:
            # as in _MotEmbedFn: the scatter overwrites every row, so it writes straight into the bucket; with a
            # gradient already on the parameter the normal path is taken and autograd adds to it
            bk, params = ctx.grad_bucket
            for i, (p, E) in enumerate(zip(params, Es)):
                if want[i] and p.grad is None and bk.holds(p):
                    view = bk.view_of(p)
                    if view.dtype != E.dtype or view.shape != E.shape or not view.is_contiguous() or view.device != E.device:
                        raise TypeError("mot_b200: the gradient-bucket view of a table must match its dtype, shape and "
                                        f"device and be contiguous (table {tuple(E.shape)} {E.dtype}, view "
                                        f"{tuple(view.shape)} {view.dtype})")
                    direct[i] = view
        grads = _gather_backward(ctx.desc, tok, Es, grad_outs, want, ws.buf, planned, clean, st, outs=direct)
        if ctx.grad_bucket is not None:
            bk, params = ctx.grad_bucket
            if bk.sparse_rows and not bk._pending and tok.numel() > 0 \
                    and any(w and bk.is_row_table(p) for w, p in zip(want, params)):
                bk.mark_rows(ctx.desc, ws.buf,
                             fresh=[p for p, d in zip(params, direct) if d is not None and bk.is_row_table(p)])
            for i, p in enumerate(params):
                if direct[i] is not None:
                    p.grad, grads[i] = direct[i], None
        ctx.ws = None
        _return_workspace(ws)
        return (None, None, None, *grads)


def tok_gather(tokens: torch.Tensor, *tables: torch.Tensor, grad_bucket=None):
    """`[E(tokens) for E in tables]` (the value embeddings of runs/7:308 / spt/train_gpt.py:600): returns a tuple of
    [n_tokens, D] tensors; dense gradients, one token sort shared by every table.  grad_bucket = optional
    dp.GradBucket holding the tables: the backward writes their gradients into it and marks the gathered rows."""
    dev, tok, Es = _gather_args(tokens, tables)
    if grad_bucket is None and _custom_ops_wanted():
        need = torch.is_grad_enabled() and any(E.requires_grad for E in tables)
        return tuple(torch.ops.mot_b200.tok_gather(tok, Es, need)[:-1])
    return _TokGatherFn.apply(dev, tok, (grad_bucket, tables) if grad_bucket is not None else None, *Es)


# ------------------------------------------------------------------------------------------------------------
# concat + dense projection variants (V1 runs/7:226-234,317-319 and spt/train_gpt.py:439-443; V2 runs/72:227-230)
# ------------------------------------------------------------------------------------------------------------
def _gemm_dtype(*ts) -> int:
    """Operand dtype of the projection kernels: all bf16 (kind::f16) or all fp32 (read in place on the TF32 path)."""
    dts = {t.dtype for t in ts if t is not None}
    if dts == {torch.bfloat16}:
        return L.BF16
    if dts == {torch.float32}:
        return L.F32
    raise NotImplementedError(f"mot_b200: the tcgen05 projection kernels take all-bf16 or all-fp32 operands, got {sorted(map(str, dts))}")


def _linear_ws(n: int, in_dim: int, out_dim: int, dt: int, dev) -> Optional[torch.Tensor]:
    need = int(L.lib().mot_linear_workspace_bytes(n, in_dim, out_dim, dt))
    return torch.empty(need, dtype=torch.uint8, device=dev) if need else None


def linear_forward_out(x, w, y, bias=None) -> None:
    """y[n, Do] = x[n, K] . w[Do, K]^T (+ bias): mot_linear_fwd (tcgen05).  bf16 operands -> y bf16 or fp32; fp32
    operands (TF32 tensor cores) -> y fp32."""
    dt = _gemm_dtype(x, w)
    dev = _require_cuda(x, w, y, bias)
    n, K = x.shape
    if dt == L.F32 and y.dtype != torch.float32:
        raise NotImplementedError("mot_b200: fp32 operands produce an fp32 result")
    with _on_device(dev):
        rc = L.lib().mot_linear_fwd(_ptr(x), _ptr(w), _ptr(bias), _ptr(y), n, K, w.shape[0], dt,
                                    1 if y.dtype == torch.float32 else 0, _stream(dev))
    L.check(rc, "mot_linear_fwd")


def linear_bwd_input_out(dy, w, dx) -> None:
    """dx[n, K] = dy[n, Do] . w[Do, K]: mot_linear_bwd_input (w read in place as an MN-major operand)."""
    dt = _gemm_dtype(dy, w, dx)
    dev = _require_cuda(dy, w, dx)
    ws = _linear_ws(dy.shape[0], w.shape[1], w.shape[0], dt, dev)
    with _on_device(dev):
        rc = L.lib().mot_linear_bwd_input(_ptr(dy), _ptr(w), _ptr(dx), dy.shape[0], w.shape[1], w.shape[0], dt,
                                          _ptr(ws), ws.numel() if ws is not None else 0, _stream(dev))
    L.check(rc, "mot_linear_bwd_input")


def linear_bwd_weight_out(dy, x, dw_f32, dw_bf16=None) -> None:
    """dw[Do, K] = dy^T . x reduced in fp32 (split over the tokens), optionally also cast to bf16."""
    dt = _gemm_dtype(dy, x)
    dev = _require_cuda(dy, x, dw_f32, dw_bf16)
    ws = _linear_ws(dy.shape[0], x.shape[1], dy.shape[1], dt, dev)
    with _on_device(dev):
        rc = L.lib().mot_linear_bwd_weight(_ptr(dy), _ptr(x), _ptr(dw_f32), _ptr(dw_bf16), dy.shape[0], x.shape[1],
                                           dy.shape[1], dt, _ptr(ws), ws.numel() if ws is not None else 0, _stream(dev))
    L.check(rc, "mot_linear_bwd_weight")


def rmsnorm_forward_out(y, out, eps: float = FP32_EPS) -> None:
    dev = _require_cuda(y, out)
    with _on_device(dev):
        rc = L.lib().mot_rmsnorm_fwd(_ptr(y), _ptr(out), y.shape[0], y.shape[1], _DTYPE[y.dtype], eps, _stream(dev))
    L.check(rc, "mot_rmsnorm_fwd")


def rmsnorm_backward_out(y, grad_out, dy, eps: float = FP32_EPS) -> None:
    dev = _require_cuda(y, grad_out, dy)
    with _on_device(dev):
        rc = L.lib().mot_rmsnorm_bwd(_ptr(y), _ptr(grad_out), _ptr(dy), y.shape[0], y.shape[1], _DTYPE[y.dtype], eps,
                                     _stream(dev))
    L.check(rc, "mot_rmsnorm_bwd")


def _pair_desc(n: int, bpt: int, E_byte, row_stride: int, col_offset: int, eps: float, *, ids=None, ttb=None,
               seq_len: int = 0, pull_side: str = "left", next_tok: bool = False) -> L.MotDesc:
    """The descriptor of the padded+pulled byte pair (mot_byte_pair_fwd/bwd): bytes-only with the per-byte norm, written
    into the columns [col_offset, col_offset + bpt*bd) of rows of row_stride elements.  Explicit `ids` (their dtype gives
    the width), else both id sets derived from `ttb` over rows of seq_len tokens with a pull from pull_side.  Built
    directly rather than through make_desc: the eager step calls it twice, and its host time adds to the step."""
    flags, tok_vocab, ttb_dtype = L.F_BYTE_NORM, 0, 0
    if ids is not None:
        flags |= L.F_IDS_I64 if ids.dtype == torch.int64 else 0
    else:
        flags |= L.F_IDS_FROM_TTB | _pull_flags(pull_side, next_tok)
        tok_vocab, ttb_dtype = ttb.shape[0], _TTB_DTYPE[ttb.dtype]
    Vb, bd = E_byte.shape
    return L.MotDesc(L.ABI_VERSION, _DTYPE[E_byte.dtype], n, seq_len, tok_vocab, Vb, bpt, 0, bd, bpt * bd, L.BYTES_ONLY, flags,
                     ttb_dtype, eps, row_stride, col_offset, 0, PAD_ID, EOT_ID)


def pair_forward_out(desc: L.MotDesc, tok, ids_a, ids_b, ttb, E_byte, out) -> None:
    """mot_byte_pair_fwd: out[:, col + k*bd : +bd] = rms_norm(E_byte[a[:, k]] + E_byte[b[:, k]]) (spt/train_gpt.py:371-379)
    in the byte columns that desc (_pair_desc) locates; (a, b) = (ids_a, ids_b), or the padded and the pulled ids of
    `tok` derived from `ttb` inside the kernel."""
    dev = _require_cuda(tok, ids_a, ids_b, ttb, E_byte, out)
    with _on_device(dev):
        rc = L.lib().mot_byte_pair_fwd(desc, _ptr(tok), _ptr(ids_a), _ptr(ids_b), _ptr(ttb), _ptr(E_byte), _ptr(out),
                                       _stream(dev))
    L.check(rc, "mot_byte_pair_fwd")


def pair_backward_out(desc: L.MotDesc, tok, ids_a, ids_b, ttb, E_byte, grad_rows, gE_byte) -> None:
    """mot_byte_pair_bwd: dense gE_byte from the byte columns of grad_rows that desc locates."""
    dev = _require_cuda(tok, ids_a, ids_b, ttb, E_byte, grad_rows, gE_byte)
    ws = torch.empty(int(L.lib().mot_byte_pair_workspace_bytes(desc.byte_vocab, desc.byte_dim)), dtype=torch.uint8,
                     device=dev)
    with _on_device(dev):
        rc = L.lib().mot_byte_pair_bwd(desc, _ptr(tok), _ptr(ids_a), _ptr(ids_b), _ptr(ttb), _ptr(E_byte), _ptr(grad_rows),
                                       _ptr(gE_byte), _ptr(ws), ws.numel(), _stream(dev))
    L.check(rc, "mot_byte_pair_bwd")


def byte_pair_forward_out(ids_a, ids_b, bpt: int, E_byte, out, col_offset: int, eps: float = FP32_EPS) -> None:
    """pair_forward_out with explicit ids into the byte columns [col_offset, col_offset + bpt*bd) of the [n, K] operand
    `out`."""
    desc = _pair_desc(out.shape[0], bpt, E_byte, out.stride(0), col_offset, eps, ids=ids_a)
    pair_forward_out(desc, None, ids_a, ids_b, None, E_byte, out)


def byte_pair_backward_out(ids_a, ids_b, bpt: int, E_byte, grad_rows, col_offset: int, gE_byte, eps: float = FP32_EPS) -> None:
    """pair_backward_out with explicit ids: dense gE_byte from the byte columns of grad_rows [n, K]."""
    desc = _pair_desc(grad_rows.shape[0], bpt, E_byte, grad_rows.stride(0), col_offset, eps, ids=ids_a)
    pair_backward_out(desc, None, ids_a, ids_b, None, E_byte, grad_rows, gE_byte)


def cast_out(w: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """CastedLinear's per-call `self.weight.type_as(x)` (spt/train_gpt.py:185-186) inside the library: fp32 -> bf16
    (mot_cast_f32_bf16).  Same dtype: returned as is."""
    w = w.detach()
    if w.dtype == dtype:
        return w.contiguous()
    if w.dtype != torch.float32 or dtype != torch.bfloat16:
        raise NotImplementedError(f"mot_b200: projection weight {w.dtype} with {dtype} tables is not supported "
                                  "(bf16 weight, or fp32 master weight cast to bf16 per call)")
    dev = _require_cuda(w)
    w = w.contiguous()
    out = torch.empty(w.shape, dtype=torch.bfloat16, device=dev)
    with _on_device(dev):
        rc = L.lib().mot_cast_f32_bf16(_ptr(w), _ptr(out), w.numel(), _stream(dev))
    L.check(rc, "mot_cast_f32_bf16")
    return out


def colsum_out(x: torch.Tensor) -> torch.Tensor:
    """fp32 column sums of x [n, dim]: the bias gradient of F.linear (mot_colsum, fixed summation order)."""
    dev = _require_cuda(x)
    x = x.contiguous()
    out = torch.empty(x.shape[1], dtype=torch.float32, device=dev)
    with _on_device(dev):
        rc = L.lib().mot_colsum(_ptr(x), _ptr(out), x.shape[0], x.shape[1], _DTYPE[x.dtype], _stream(dev))
    L.check(rc, "mot_colsum")
    return out


def _mixout_copy_impl(x: torch.Tensor, bpt: int, backward: bool) -> torch.Tensor:
    dev = x.device
    rows, D = x.shape
    n = rows // bpt if backward else rows
    out = torch.empty((n if backward else n * bpt, D), dtype=x.dtype, device=dev)
    with _on_device(dev):
        fn = L.lib().mot_mixout_copy_bwd if backward else L.lib().mot_mixout_copy_fwd
        rc = fn(_ptr(x), _ptr(out), n, D, bpt, _DTYPE[x.dtype], _stream(dev))
    L.check(rc, "mot_mixout_copy_bwd" if backward else "mot_mixout_copy_fwd")
    return out


class _MixoutCopyFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x2d, bpt):
        ctx.bpt = bpt
        return _mixout_copy_impl(x2d, bpt, backward=False)

    @staticmethod
    def backward(ctx, g):
        return _mixout_copy_impl(g.contiguous(), ctx.bpt, backward=True), None


def mixout_copy(x: torch.Tensor, bytes_per_token: int) -> torch.Tensor:
    """ByteMixoutCopy's expand (spt/train_gpt.py:493): `einops.repeat(x, "... T D -> ... (T bpt) D")`; the backward sums
    the bpt copies of every row in fp32."""
    _require_cuda(x)
    if x.dtype not in _DTYPE:
        raise NotImplementedError(f"mot_b200.mixout_copy: dtype {x.dtype} is not supported (bf16 / fp32 only)")
    lead, T, D = x.shape[:-2], x.shape[-2], x.shape[-1]
    x2 = x.contiguous().view(-1, D)
    if _custom_ops_wanted():
        y = torch.ops.mot_b200.mixout_copy(x2, bytes_per_token)
    else:
        y = _MixoutCopyFn.apply(x2, bytes_per_token)
    return y.view(*lead, T * bytes_per_token, D)


def mixout_split(x: torch.Tensor, bytes_per_token: int) -> torch.Tensor:
    """ByteMixoutSplit's expand (spt/train_gpt.py:516): `rearrange(x, "... T (bpt D) -> ... (T bpt) D")` is a view of
    contiguous rows: no kernel, no copy."""
    lead, T, D = x.shape[:-2], x.shape[-2], x.shape[-1]
    if D % bytes_per_token:
        raise RuntimeError("model_dim must be divisible by bytes_per_token")   # spt/train_gpt.py:502
    return x.contiguous().view(*lead, T * bytes_per_token, D // bytes_per_token)


_PROJ_KEEP_OPERAND = not __import__("os").environ.get("MOT_PROJ_REGATHER")


def _proj_args(spec: MixSpec, bpt: int, tokens, byte_ids, E_tok, E_byte, W, bias, byte_ids2, ttb, seq_len: int,
               ttb_pair: bool, next_tokens):
    """mot_embed_proj's arguments checked and normalised -> (dev, tok, ids, ids2, E_tok, E_byte, ttb, next_tok)."""
    dev = _require_cuda(tokens, byte_ids, E_tok, E_byte, W, bias, byte_ids2, ttb, next_tokens)
    _require_chain_dtype(E_tok, E_byte)
    tok, ids, ids2, ttb, nxt = _id_args(spec, bpt, tokens, byte_ids, ttb, seq_len, next_tokens, byte_ids2, ttb_pair)
    K = E_tok.shape[1] + bpt * E_byte.shape[1]
    if W.shape[1] != K:
        raise RuntimeError(f"mot_b200: projection weight is {tuple(W.shape)}, expected [{W.shape[0]}, {K}]")
    if bias is not None and bias.dtype != torch.float32:
        raise NotImplementedError("mot_b200: the projection bias must be fp32 (mathblations/model.py:261)")
    return dev, tok, ids, ids2, E_tok.contiguous(), E_byte.contiguous(), ttb, nxt


def _proj_descs(spec: MixSpec, bpt: int, seq_len: int, tok, next_tok, ids, ids2, ttb, ttb_pair: bool, E_tok, E_byte):
    """-> (tok, desc, desc_pair): desc gathers the [n, K] operand, the concat of both tables.  With a pair (`ids2`, or
    ttb_pair: the padded and the pulled ids from `ttb`) desc gathers only the operand's token columns, with row stride K,
    and desc_pair (bytes-only, per-byte norm) describes the byte columns that the pair kernels write.  Without a pair
    desc_pair is None."""
    if ids2 is None and not ttb_pair:
        tok, desc = _ids_desc(dataclasses.replace(spec, combine="concat", out_norm=False), bpt, seq_len, tok, next_tok,
                              ids, ttb, E_tok, E_byte)
        return tok, desc, None
    K = E_tok.shape[1] + bpt * E_byte.shape[1]
    tok = _tok_next(tok, next_tok)
    desc_pair = _pair_desc(tok.numel(), bpt, E_byte, K, E_tok.shape[1], spec.eps, ids=ids, ttb=ttb, seq_len=seq_len,
                           pull_side=spec.ttb_pull_side, next_tok=next_tok is not None)
    desc = make_desc(MixSpec(combine="tok_only", tok_norm=spec.tok_norm, out_norm=False, eps=spec.eps), tok.numel(),
                     E_tok, None, 0, ids=None, ttb=None, has_lam=False, row_stride=K, col_offset=0)
    return tok, desc, desc_pair


def _gather_operand(desc: L.MotDesc, desc_pair: Optional[L.MotDesc], tok, ids, ids2, ttb, E_tok, E_byte, A) -> None:
    if desc_pair is None:
        embed_forward_out(desc, tok, ids, ttb, E_tok, E_byte, None, A)
    elif tok.numel() > 0:
        embed_forward_out(desc, tok, None, None, E_tok, None, None, A)
        pair_forward_out(desc_pair, tok, ids, ids2, ttb, E_byte, A)


def _scatter_operand(desc: L.MotDesc, desc_pair: Optional[L.MotDesc], tok, ids, ids2, ttb, E_tok, E_byte, dA, ws_buf,
                     plan_ready: bool, ws_clean: bool):
    """The backward of _gather_operand: dense (gE_tok, gE_byte) from the operand's gradient dA."""
    gE_tok, gE_byte = torch.empty_like(E_tok), torch.empty_like(E_byte)
    if desc_pair is None:
        embed_backward_out(desc, tok, ids, ttb, E_tok, E_byte, None, dA, gE_tok, gE_byte, None, ws_buf,
                           plan_ready=plan_ready, ws_clean=ws_clean)
    else:   # token columns through the sorted-stream scatter, byte columns through the pair kernel
        embed_backward_out(desc, tok, None, None, E_tok, None, None, dA, gE_tok, None, None, ws_buf,
                           plan_ready=plan_ready, ws_clean=ws_clean)
        pair_backward_out(desc_pair, tok, ids, ids2, ttb, E_byte, dA, gE_byte)
    return gE_tok, gE_byte


def _proj_forward(spec: MixSpec, desc: L.MotDesc, desc_pair: Optional[L.MotDesc], tok, ids, ids2, ttb, E_tok, E_byte, w_c,
                  bias, keep_operand: bool):
    """-> (out, Y, A): Y = A . w_c^T (+ bias) with the gathered [n, K] operand A (None unless keep_operand), out = the
    row norm of Y under spec.out_norm, else Y itself.  w_c: the weight in the table dtype."""
    n, (Do, K), dev, cdt = tok.numel(), w_c.shape, E_tok.device, E_tok.dtype
    A = torch.empty((n, K), dtype=cdt, device=dev)
    _gather_operand(desc, desc_pair, tok, ids, ids2, ttb, E_tok, E_byte, A)
    Y = torch.empty((n, Do), dtype=cdt, device=dev)
    linear_forward_out(A, w_c, Y, bias.contiguous() if bias is not None else None)
    if not keep_operand:
        A = None
    if spec.out_norm:
        out = torch.empty_like(Y)
        rmsnorm_forward_out(Y, out, spec.eps)
    else:
        out = Y
    return out, Y, A


def _proj_backward(spec: MixSpec, desc: L.MotDesc, desc_pair: Optional[L.MotDesc], tok, ids, ids2, ttb, E_tok, E_byte, w_c,
                   w_dtype, has_bias: bool, Y, A, grad_out):
    """The backward of _proj_forward down to the operand -> (dA, gW in w_dtype, g_bias fp32 or None).  A: the forward's
    operand if it was kept, else None (gathered again here)."""
    n, (Do, K), dev, cdt = tok.numel(), w_c.shape, E_tok.device, E_tok.dtype
    g = grad_out.reshape(n, Do).to(cdt).contiguous()
    if spec.out_norm:
        dY = torch.empty_like(Y)
        rmsnorm_backward_out(Y, g, dY, spec.eps)
    else:
        dY = g
    g_bias = colsum_out(dY) if has_bias else None
    if A is not None:
        dA = torch.empty((n, K), dtype=cdt, device=dev)                   # a saved tensor is never overwritten
    else:
        A = torch.empty((n, K), dtype=cdt, device=dev)
        _gather_operand(desc, desc_pair, tok, ids, ids2, ttb, E_tok, E_byte, A)
        dA = A                                                            # dX may overwrite the private copy
    dW32 = torch.empty((Do, K), dtype=torch.float32, device=dev)
    dW16 = torch.empty((Do, K), dtype=torch.bfloat16, device=dev) if w_dtype == torch.bfloat16 else None
    linear_bwd_weight_out(dY, A, dW32, dW16)
    linear_bwd_input_out(dY, w_c, dA)
    return dA, (dW16 if dW16 is not None else dW32), g_bias      # cast_out admits bf16 or fp32 weights only


class _MotEmbedProjFn(torch.autograd.Function):
    """out = f_out( [tok | bytes] . W^T + bias ): the fused gather builds the [n, K] operand (mot_embed_fwd, CONCAT),
    the projection runs on the tensor cores (mot_linear_fwd), the row norm after it is a separate HBM-bound pass over
    the bf16 product (the reference also rounds F.linear's output to bf16 before its rms_norm).  The [n, K] operand is
    kept for the backward (n*K*2 bytes: 268 MB at 64K x 2048, small on 180 GB; saves one gather pass, ~0.1 ms of a 1.2 ms
    step); MOT_PROJ_REGATHER=1 gathers it again instead (the round-1 behaviour, for memory-tight callers)."""

    @staticmethod
    def forward(ctx, spec: MixSpec, desc: L.MotDesc, desc_pair: Optional[L.MotDesc], dev, tok, ids, ids2, E_tok, E_byte, W,
                bias, ttb=None):
        w16 = cast_out(W, E_tok.dtype)                         # CastedLinear: W.type_as(x) (spt/train_gpt.py:186)
        ctx.ws = _planned_workspace(desc, tok, dev) if any(ctx.needs_input_grad[7:9]) and tok.numel() > 0 else None
        keep_A = _PROJ_KEEP_OPERAND and any(ctx.needs_input_grad[7:11])
        out, Y, A = _proj_forward(spec, desc, desc_pair, tok, ids, ids2, ttb, E_tok, E_byte, w16, bias, keep_A)
        embed_plan_join_if_capturing(ctx.ws, dev)
        ctx.desc, ctx.desc_pair, ctx.dev, ctx.spec = desc, desc_pair, dev, spec
        ctx.w_dtype, ctx.has_bias = W.dtype, bias is not None
        ctx.present = (ids is not None, ids2 is not None, keep_A, ttb is not None)
        ctx.save_for_backward(tok, *[t if t is not None else _ABSENT for t in (ids, ids2, A if keep_A else None, ttb)],
                              E_tok, E_byte, w16, Y)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        tok, ids, ids2, A, ttb, E_tok, E_byte, w16, Y = ctx.saved_tensors
        ids, ids2, A, ttb = [t if ok else None for t, ok in zip((ids, ids2, A, ttb), ctx.present)]
        desc, desc_pair, dev = ctx.desc, ctx.desc_pair, ctx.dev
        dA, gW, g_bias = _proj_backward(ctx.spec, desc, desc_pair, tok, ids, ids2, ttb, E_tok, E_byte, w16, ctx.w_dtype,
                                        ctx.has_bias, Y, A, grad_out)
        ws, planned, clean = _take_workspace(ctx.ws, desc, dev)
        gE_tok, gE_byte = _scatter_operand(desc, desc_pair, tok, ids, ids2, ttb, E_tok, E_byte, dA, ws.buf, planned, clean)
        ctx.ws = None
        _return_workspace(ws)
        return None, None, None, None, None, None, None, gE_tok, gE_byte, gW, g_bias, None


def _byte_fc_args(spec_b: MixSpec, bpt: int, tokens, byte_ids, E_tok, E_byte, W, ttb, seq_len: int, next_tokens):
    """mot_embed_byte_fc's arguments checked and normalised -> (dev, tok, ids, E_tok, E_byte, ttb, next_tok)."""
    dev = _require_cuda(tokens, byte_ids, E_tok, E_byte, W, ttb, next_tokens)
    _require_chain_dtype(E_tok, E_byte)
    D = E_tok.shape[1]
    if (byte_ids is not None and byte_ids.numel() != tokens.numel() * bpt) or bpt * E_byte.shape[1] != D \
            or tuple(W.shape) != (D, D):
        raise RuntimeError("mot_b200: byte-FC mix needs bpt*byte_dim == token_dim and a square [D, D] weight")
    tok, ids, _, ttb, nxt = _id_args(spec_b, bpt, tokens, byte_ids, ttb, seq_len, next_tokens)
    return dev, tok, ids, E_tok.contiguous(), E_byte.contiguous(), ttb, nxt


def _fc_descs(spec_b: MixSpec, bpt: int, seq_len: int, tok, next_tok, ids, ttb, E_tok, E_byte):
    """-> (tok, desc_b, desc_t): the bytes-only gather of the product's operand; the token gather + addend + norm."""
    tok, desc_b = _ids_desc(spec_b, bpt, seq_len, tok, next_tok, ids, ttb, None, E_byte)
    return tok, desc_b, make_desc(MixSpec(combine="tok_only", out_norm=True, eps=spec_b.eps), tok.numel(), E_tok, None, 0,
                                  ids=None, ttb=None, has_lam=False)


def _byte_fc_forward(desc_b: L.MotDesc, desc_t: L.MotDesc, tok, ids, E_tok, E_byte, w_c, ttb=None):
    """-> (out, Y): Y = C . w_c^T with C the bytes-only gather (not kept), out = norm(E_tok[tok] + Y)."""
    n, D, dev, cdt = tok.numel(), E_tok.shape[1], E_tok.device, E_tok.dtype
    C = torch.empty((n, D), dtype=cdt, device=dev)
    embed_forward_out(desc_b, tok if ttb is not None else None, ids, ttb, None, E_byte, None, C)
    Y = torch.empty((n, D), dtype=cdt, device=dev)
    linear_forward_out(C, w_c, Y)
    del C
    out = torch.empty((n, D), dtype=cdt, device=dev)
    if n > 0:
        embed_forward_out(desc_t, tok, None, None, E_tok, None, None, out, addend=Y)
    return out, Y


def _byte_fc_backward(desc_b: L.MotDesc, desc_t: L.MotDesc, tok, ids, E_tok, E_byte, w_c, w_dtype, Y, grad_out,
                      ws_buf, plan_ready: bool, ws_clean: bool, wsb_buf, wsb_clean: bool, ttb=None):
    """-> (gE_tok, gE_byte, gW in w_dtype).  ws_*: the workspace of the token scatter; wsb_*: the workspace of the
    bytes-only scatter, which is never planned ahead."""
    (n, D), dev, cdt = Y.shape, Y.device, Y.dtype
    g = grad_out.reshape(n, D).to(cdt).contiguous()
    gE_tok, gE_byte = torch.empty_like(E_tok), torch.empty_like(E_byte)
    dY = torch.empty_like(Y)
    embed_backward_out(desc_t, tok, None, None, E_tok, None, None, g, gE_tok, None, None, ws_buf,
                       plan_ready=plan_ready, ws_clean=ws_clean, addend=Y, d_addend=dY)
    C = torch.empty((n, D), dtype=cdt, device=dev)
    tok_b = tok if ttb is not None else None                                     # the bytes-only gather reads tokens only to derive ids
    embed_forward_out(desc_b, tok_b, ids, ttb, None, E_byte, None, C)            # gathered again, not kept
    dW32 = torch.empty((D, D), dtype=torch.float32, device=dev)
    dW16 = torch.empty((D, D), dtype=torch.bfloat16, device=dev) if w_dtype == torch.bfloat16 else None
    linear_bwd_weight_out(dY, C, dW32, dW16)
    linear_bwd_input_out(dY, w_c, C)                                             # dC overwrites the operand buffer
    embed_backward_out(desc_b, tok_b, ids, ttb, None, E_byte, None, C, None, gE_byte, None, wsb_buf,
                       plan_ready=False, ws_clean=wsb_clean)
    return gE_tok, gE_byte, (dW16 if dW16 is not None else dW32)


class _MotEmbedByteFcFn(torch.autograd.Function):
    """runs/71051:226-229,312-314 (V3f): out = norm(embed_tokens(tok) + F.linear(cat_k embed_bytes(ids_k), byte_fc)).
    Forward: bytes-only gather of the [n, D] operand (ids in the `.view(bpt,-1)` order), tcgen05 product, then the fused
    token gather + add + rms-norm (mot_embed_fwd_ex with the product as dense addend).  Backward: the fused kernel
    scatters d z into the token table and writes it densely as the gradient of the product; dW, dX on the tensor
    cores; bytes-only scatter.  The operand is gathered again in the backward, not kept."""

    @staticmethod
    def forward(ctx, desc_b: L.MotDesc, desc_t: L.MotDesc, dev, tok, ids, E_tok, E_byte, W, ttb=None):
        w16 = cast_out(W, E_tok.dtype)
        ctx.ws = _planned_workspace(desc_t, tok, dev) if ctx.needs_input_grad[5] and tok.numel() > 0 else None
        out, Y = _byte_fc_forward(desc_b, desc_t, tok, ids, E_tok, E_byte, w16, ttb)
        embed_plan_join_if_capturing(ctx.ws, dev)
        ctx.desc_b, ctx.desc_t, ctx.dev, ctx.w_dtype = desc_b, desc_t, dev, W.dtype
        ctx.present = (ids is not None, ttb is not None)
        ctx.save_for_backward(tok, ids if ids is not None else _ABSENT, ttb if ttb is not None else _ABSENT,
                              E_tok, E_byte, w16, Y)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        tok, ids, ttb, E_tok, E_byte, w16, Y = ctx.saved_tensors
        ids, ttb = [t if ok else None for t, ok in zip((ids, ttb), ctx.present)]
        ws, planned, clean = _take_workspace(ctx.ws, ctx.desc_t, ctx.dev)
        wsb, _, clean_b = _take_workspace(None, ctx.desc_b, ctx.dev)
        gE_tok, gE_byte, gW = _byte_fc_backward(ctx.desc_b, ctx.desc_t, tok, ids, E_tok, E_byte, w16, ctx.w_dtype, Y,
                                                grad_out, ws.buf, planned, clean, wsb.buf, clean_b, ttb)
        ctx.ws = None
        _return_workspace(ws)
        _return_workspace(wsb)
        return None, None, None, None, None, gE_tok, gE_byte, gW, None


def mot_embed_byte_fc(tokens: torch.Tensor, byte_ids: Optional[torch.Tensor], E_tok: torch.Tensor, E_byte: torch.Tensor,
                      W_fc: torch.Tensor, *, bpt: int = 16, slot_major: bool = True, eps: float = FP32_EPS,
                      ttb: Optional[torch.Tensor] = None, seq_len: int = 0, ttb_pull: bool = False,
                      ttb_pull_side: str = "left", next_tokens: Optional[torch.Tensor] = None) -> torch.Tensor:
    """`norm(token_embs + F.linear(cat(byte_embs), byte_fc))` (runs/71051:226-229,312-314): [n_tokens, D].
    byte_ids=None: the ids come from `ttb` inside the kernels (rows of seq_len tokens; the `.view(bpt,-1)` order under
    slot_major), the pulled ids of pull_from_left with ttb_pull (pull_from_right with ttb_pull_side="right", whose
    lookahead `next_tokens` holds token seq_len of every row, as in mot_embed)."""
    spec_b = MixSpec(combine="bytes_only", out_norm=False, slot_major=slot_major and byte_ids is not None,
                     ttb_scramble=slot_major and byte_ids is None, ttb_pull=ttb_pull and byte_ids is None, eps=eps,
                     ttb_pull_side=ttb_pull_side)
    dev, tok, ids, E_tok_c, E_byte_c, ttb_c, nxt = _byte_fc_args(spec_b, bpt, tokens, byte_ids, E_tok, E_byte, W_fc, ttb,
                                                                 seq_len, next_tokens)
    if _custom_ops_wanted():
        need = torch.is_grad_enabled() and any(t.requires_grad for t in (E_tok, E_byte, W_fc))
        return torch.ops.mot_b200.embed_byte_fc(tok, ids, E_tok_c, E_byte_c, W_fc.contiguous(), pack_spec(spec_b), bpt,
                                                float(eps), need, ttb_c, seq_len, nxt)[0]
    tok, desc_b, desc_t = _fc_descs(spec_b, bpt, seq_len, tok, nxt, ids, ttb_c, E_tok_c, E_byte_c)
    return _MotEmbedByteFcFn.apply(desc_b, desc_t, dev, tok, ids, E_tok_c, E_byte_c, W_fc, ttb_c)


def mot_embed_proj(tokens: torch.Tensor, byte_ids: Optional[torch.Tensor], E_tok: torch.Tensor, E_byte: torch.Tensor,
                   W: torch.Tensor, spec: MixSpec, *, bpt: int = 16, bias: Optional[torch.Tensor] = None,
                   byte_ids2: Optional[torch.Tensor] = None, ttb: Optional[torch.Tensor] = None, seq_len: int = 0,
                   padded_and_pulled: bool = False, next_tokens: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Concat + dense projection variants: `norm(F.linear(cat([f(tok), f(bytes)]), W))` (runs/7:226-234, runs/72,
    spt/train_gpt.py:439-443).  spec.tok_norm / byte_norm are the per-input norms, spec.out_norm the norm after the
    projection, spec.bytes_first the operand order.  Tables bf16 with W bf16 (runs) or an fp32 master (spt: cast per
    call, gradient returned in fp32); or everything fp32 (mathblations: TF32 tensor cores).  byte_ids2: the second id
    tensor of `--add-padded-and-pulled` (spt/train_gpt.py:371-379), rows summed before the per-byte norm.  Returns
    [n_tokens, W.shape[0]] in the table dtype.

    Token-only form: byte_ids=None with the [V, bpt] table `ttb` derives the ids inside the kernels -- the padded ids, or
    with spec.ttb_pull the pulled ids of pull_from_left over rows of `seq_len` tokens; padded_and_pulled=True derives
    both sets of `--add-padded-and-pulled`.  spec.ttb_pull_side="right": pull_from_right, with the lookahead
    `next_tokens` (token seq_len of every row, as in mot_embed)."""
    ttb_pair = padded_and_pulled and byte_ids is None
    dev, tok, ids, ids2, E_tok_c, E_byte_c, ttb_c, nxt = _proj_args(spec, bpt, tokens, byte_ids, E_tok, E_byte, W, bias,
                                                                    byte_ids2, ttb, seq_len, ttb_pair, next_tokens)
    if _custom_ops_wanted():
        need = torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in (E_tok, E_byte, W, bias))
        return torch.ops.mot_b200.embed_proj(tok, ids, ids2, E_tok_c, E_byte_c, W.contiguous(), bias, pack_spec(spec), bpt,
                                             float(spec.eps), need, ttb_c, seq_len, ttb_pair, nxt)[0]
    tok, desc, desc_pair = _proj_descs(spec, bpt, seq_len, tok, nxt, ids, ids2, ttb_c, ttb_pair, E_tok_c, E_byte_c)
    return _MotEmbedProjFn.apply(spec, desc, desc_pair, dev, tok, ids, ids2, E_tok_c, E_byte_c, W, bias, ttb_c)


def launch_count() -> int:
    return int(L.lib().mot_launch_count())


def reset_launch_count() -> None:
    L.lib().mot_launch_count_reset()


# torch.library registration of the same entry points (torch.compile / compiled autograd see opaque operators)
from ._library import custom_ops_wanted as _custom_ops_wanted, pack_spec, set_custom_ops  # noqa: E402,F401
