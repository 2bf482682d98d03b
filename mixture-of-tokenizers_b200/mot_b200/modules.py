"""Drop-in nn.Modules with the reference's parameter names and forward signatures,
backed by the fused CUDA path (no PyTorch fallback).

Reference call sites:
  * modded-nanogpt runs:  `x_toks = embed_tokens(token_inputs)[None]; x_bytes = embed_bytes(byte_inputs)...;
    x = mixin_bytes(x_toks, x_bytes[, W])`  (runs/71:312-314, runs/7:317-319, ...)
  * scaled-pre-train:     `xt, xb = self.embed(tokens, bytes_padded, bytes_pulled); x = self.byte_mixin(xt, xb)`
    (spt/train_gpt.py:605-606)
  * mathblations:         `x = self.digit_mixin(self.wte(idx), self.dte(digits))` (mathblations/model.py:323-327)
"""
from __future__ import annotations

import dataclasses
from typing import Optional

import torch
from torch import nn

from .ops import _TTB_DTYPE, MixSpec, mot_embed, mot_embed_byte_fc, mot_embed_proj, split_residual, tok_gather

# variant name -> MixSpec kwargs (SURVEY.md 2.4; `slot_major` is the `.view(bpt,-1)` id layout of the sum runs)
RUN_VARIANTS = {
    "V0": dict(combine="tok_only"),
    "V3": dict(combine="add", slot_major=True),                                                  # runs/71
    "V3b": dict(combine="add", tok_norm=True, byte_norm=True, out_norm=False, slot_major=True),  # runs/73
    "V3c": dict(combine="add", tok_norm=True, byte_norm=True, out_norm=False, slot_major=True),  # runs/74 (+lambdas)
    "V3d": dict(combine="add", tok_norm=True, byte_norm=True, out_norm=True, slot_major=True),   # runs/71041 (+lambdas)
    "V3e": dict(combine="add", tok_norm=True, byte_norm=True, out_norm=True, slot_major=True),   # runs/71042-44 (lambdas / their sum)
    "V4": dict(combine="concat"),                                                                # runs/711
    "V5": dict(combine="bytes_only"),                                                            # runs/4
}
_LAMBDA_VARIANTS = ("V3c", "V3d", "V3e")
# (byte, token) initial values of the two trailing `scalars` entries per run (runs/74:259; runs/71043:252-259; runs/71044)
LAMBDA_INIT = {"run74": (0.5, 0.5), "run71042": (0.5, 0.5), "run71043": (0.01, 0.99), "run71044": (0.4, 0.6)}


class MoTEmbedding(nn.Module):
    """The embedding front of the modded-nanogpt MoT runs: parameters `embed_tokens.weight`,
    `embed_bytes.weight` (and `lambdas` = the two trailing entries of the reference's `scalars`,
    [byte, token] order as in runs/74:259,314-315); forward(token_inputs [T] int32,
    byte_inputs int32 [bpt, T] or [1, T*bpt]) -> [1, T, model_dim].  With byte_inputs=None and a ttb
    table the byte ids are derived inside the kernel: the padded ids, or with pull_in=True the pulled ids of
    pull_from_left over the T tokens."""

    def __init__(self, token_vocab_size: int, byte_vocab_size: int, token_dim: int, byte_dim: int,
                 bytes_per_token: int = 16, variant: str = "V3", ttb: Optional[torch.Tensor] = None,
                 lambda_init=(0.5, 0.5), pull_in: bool = False):
        super().__init__()
        if variant not in RUN_VARIANTS:
            raise NotImplementedError(f"mot_b200: variant {variant!r} has no fused kernel")
        self.variant, self.bpt, self.pull_in = variant, bytes_per_token, pull_in
        self.spec = MixSpec(**RUN_VARIANTS[variant])
        self.embed_tokens = nn.Embedding(token_vocab_size, token_dim) if variant != "V5" else None
        self.embed_bytes = nn.Embedding(byte_vocab_size, byte_dim) if variant != "V0" else None
        self.lambdas = nn.Parameter(torch.tensor([float(lambda_init[0]), float(lambda_init[1])])) \
            if variant in _LAMBDA_VARIANTS else None
        self.register_buffer("ttb", ttb, persistent=False)
        self.grad_bucket = None

    def attach_grad_bucket(self, bucket=None):
        """Data parallelism: let the backward kernels write `embed_tokens.weight.grad` / `embed_bytes.weight.grad`
        straight into one flat bucket, so the per-parameter all-reduces of the reference (runs/7:697-700) become a
        single `bucket.all_reduce_avg()`.  The bucket may hold more tables (the value embeddings: see
        TokenValueEmbeddings.attach_grad_bucket); the rows of the batch are marked whenever the token table is one of
        its row tables.  Call after the module is on its device and in its final dtype."""
        from .dp import GradBucket
        tables = [m.weight for m in (self.embed_tokens, self.embed_bytes) if m is not None]
        self.grad_bucket = bucket if bucket is not None else GradBucket(tables, symmetric="auto")
        return self.grad_bucket

    def forward(self, token_inputs: torch.Tensor, byte_inputs: Optional[torch.Tensor] = None) -> torch.Tensor:
        assert token_inputs.ndim == 1  # runs/71:300
        lam = None
        if self.lambdas is not None:  # kernel order (tok, byte); parameter order (byte, tok) like scalars[-2], scalars[-1]
            lam = self.lambdas.flip(0)
            if self.variant == "V3e":  # runs/71042:311-313: both scalars divided by their sum
                lam = lam / lam.sum()
        spec = self.spec
        if byte_inputs is None and self.embed_bytes is not None:
            spec = MixSpec(**{**RUN_VARIANTS[self.variant], "slot_major": False,
                              "ttb_scramble": RUN_VARIANTS[self.variant].get("slot_major", False), "ttb_pull": self.pull_in})
        derive = byte_inputs is None and self.embed_bytes is not None   # the ids come from the tokens and the ttb table
        x = mot_embed(token_inputs if self.embed_tokens is not None or derive else None, byte_inputs,
                      self.embed_tokens.weight if self.embed_tokens is not None else None,
                      self.embed_bytes.weight if self.embed_bytes is not None else None,
                      spec, bpt=self.bpt, lam=lam, ttb=self.ttb if byte_inputs is None else None,
                      seq_len=token_inputs.numel(), grad_bufs=self._grad_bufs())
        return x[None]

    def _grad_bufs(self):
        if self.grad_bucket is None:
            return None
        b = self.grad_bucket
        tw = self.embed_tokens.weight if self.embed_tokens is not None else None
        bw = self.embed_bytes.weight if self.embed_bytes is not None else None
        return ((tw, b.view_of(tw)) if tw is not None else None, (bw, b.view_of(bw)) if bw is not None else None, b)


# variant name -> MixSpec kwargs of the concat + dense projection family
PROJ_VARIANTS = {
    "V1": dict(combine="concat", tok_norm=True, byte_norm=True, out_norm=True),                  # runs/7:226-234,317-319
    "V2": dict(combine="concat", tok_norm=False, byte_norm=False, out_norm=True, slot_major=True),  # runs/72:227-230,313-315
}


def _init_linear_(w: torch.Tensor) -> torch.Tensor:
    """CastedLinear.reset_parameters (spt/train_gpt.py:179-183): uniform +-sqrt(3)*0.5*in^-0.5."""
    bound = (3 ** 0.5) * 0.5 * (w.shape[1] ** -0.5)
    with torch.no_grad():
        return w.uniform_(-bound, bound)


class MoTProjEmbedding(nn.Module):
    """The concat + projection front of the modded-nanogpt runs (runs/7, 72, 75-79): parameters `embed_tokens.weight`,
    `embed_bytes.weight`, `byte_mixin_weight` [model_dim, token_dim + bpt*byte_dim] (bf16 like runs/7:249).
    forward(token_inputs [T] int32, byte_inputs int32 [1, T*bpt] (V1) or [bpt, T] (V2)) -> [1, T, model_dim]:
    fused gather of the [tok | bytes] operand, tcgen05 projection, rms_norm.  With a ttb table, byte_inputs=None derives
    the ids inside the kernels (the pulled ids of pull_from_left over the T tokens with pull_in=True)."""

    def __init__(self, token_vocab_size: int, byte_vocab_size: int, token_dim: int, byte_dim: int, model_dim: int,
                 bytes_per_token: int = 16, variant: str = "V1", ttb: Optional[torch.Tensor] = None, pull_in: bool = False):
        super().__init__()
        if variant not in PROJ_VARIANTS:
            raise NotImplementedError(f"mot_b200: projection variant {variant!r} has no fused kernel")
        self.variant, self.bpt = variant, bytes_per_token
        self.spec = MixSpec(**PROJ_VARIANTS[variant])
        self.embed_tokens = nn.Embedding(token_vocab_size, token_dim)
        self.embed_bytes = nn.Embedding(byte_vocab_size, byte_dim)
        self.byte_mixin_weight = nn.Parameter(
            _init_linear_(torch.empty(model_dim, token_dim + bytes_per_token * byte_dim)).bfloat16())
        self.register_buffer("ttb", ttb, persistent=False)
        self.pull_in = pull_in

    def forward(self, token_inputs: torch.Tensor, byte_inputs: Optional[torch.Tensor] = None) -> torch.Tensor:
        assert token_inputs.ndim == 1  # runs/7:305
        spec = self.spec
        if byte_inputs is None:
            spec = MixSpec(**{**PROJ_VARIANTS[self.variant], "slot_major": False,
                              "ttb_scramble": PROJ_VARIANTS[self.variant].get("slot_major", False), "ttb_pull": self.pull_in})
        x = mot_embed_proj(token_inputs, byte_inputs, self.embed_tokens.weight, self.embed_bytes.weight,
                           self.byte_mixin_weight, spec, bpt=self.bpt, ttb=self.ttb if byte_inputs is None else None,
                           seq_len=token_inputs.numel())
        return x[None]


class MoTByteFcEmbedding(nn.Module):
    """runs/71051:226-229,253,312-314 (V3f): parameters `embed_tokens.weight`, `embed_bytes.weight`, `byte_fc`
    [model_dim, model_dim] bf16; forward(token_inputs [T], byte_inputs [bpt, T]) ->
    norm(embed_tokens(tok) + F.linear(cat(embed_bytes(bytes)), byte_fc)) as [1, T, model_dim]."""

    def __init__(self, token_vocab_size: int, byte_vocab_size: int, model_dim: int, byte_dim: int, bytes_per_token: int = 16):
        super().__init__()
        if byte_dim * bytes_per_token != model_dim:
            raise ValueError("MoTByteFcEmbedding: bytes_per_token * byte_dim must equal model_dim (runs/71051:500-501)")
        self.bpt = bytes_per_token
        self.embed_tokens = nn.Embedding(token_vocab_size, model_dim)
        self.embed_bytes = nn.Embedding(byte_vocab_size, byte_dim)
        self.byte_fc = nn.Parameter(_init_linear_(torch.empty(model_dim, model_dim)).bfloat16())

    def forward(self, token_inputs: torch.Tensor, byte_inputs: torch.Tensor) -> torch.Tensor:
        assert token_inputs.ndim == 1
        x = mot_embed_byte_fc(token_inputs, byte_inputs, self.embed_tokens.weight, self.embed_bytes.weight, self.byte_fc,
                              bpt=self.bpt)
        return x[None]


class MoTSplitResidualEmbedding(nn.Module):
    """runs/71081:302-304,315 (V3g): the token and byte halves are kept apart for the per-block residuals.
    forward(token_inputs [T], byte_inputs [bpt, T]) -> (x, x0t, x0b), each [1, T, model_dim], with
    x0t = norm(embed_tokens(tok)), x0b = the per-byte-normed bytes concatenated in the `.view(bpt,-1)` order and
    x = lam_tok * x0t + lam_byte * x0b.  Parameters `embed_tokens.weight`, `embed_bytes.weight`, `lambdas` ([byte,
    token] = the reference's scalars[-2], scalars[-1]).  One fused kernel writes the three outputs and one backward
    takes the gradients of all three uses (model_dim 512 or 1024).  With byte_inputs=None and a ttb table the byte ids
    are derived inside the kernels: the padded ids, or with pull_in=True the pulled ids of pull_from_left over the T
    tokens."""

    def __init__(self, token_vocab_size: int, byte_vocab_size: int, model_dim: int, byte_dim: int, bytes_per_token: int = 16,
                 ttb: Optional[torch.Tensor] = None, pull_in: bool = False):
        super().__init__()
        if byte_dim * bytes_per_token != model_dim:
            raise ValueError("MoTSplitResidualEmbedding: bytes_per_token * byte_dim must equal model_dim (runs/71081:500-501)")
        if ttb is not None and (ttb.dim() != 2 or ttb.shape[1] != bytes_per_token or ttb.dtype not in _TTB_DTYPE):
            raise ValueError(f"MoTSplitResidualEmbedding: ttb must be a [V, {bytes_per_token}] int16 / float32 / bfloat16 "
                             f"table, got {tuple(ttb.shape)} {ttb.dtype}")
        if pull_in and ttb is None:
            raise ValueError("MoTSplitResidualEmbedding: pull_in=True derives the pulled ids from a ttb table: pass ttb=")
        self.bpt, self.pull_in = bytes_per_token, pull_in
        self.embed_tokens = nn.Embedding(token_vocab_size, model_dim)
        self.embed_bytes = nn.Embedding(byte_vocab_size, byte_dim)
        self.lambdas = nn.Parameter(torch.tensor([0.5, 0.5]))
        self.register_buffer("ttb", ttb, persistent=False)
        self.grad_bucket = None

    def attach_grad_bucket(self, bucket=None):
        """Data parallelism, as MoTEmbedding.attach_grad_bucket: the backward writes `embed_tokens.weight.grad` and
        `embed_bytes.weight.grad` straight into one flat bucket (default: a bucket of these two tables) and marks the
        rows of the batch when the token table is one of its row tables, so one `bucket.all_reduce_avg()` moves only the
        rows some rank gathered.  Call after the module is on its device and in its final dtype."""
        from .dp import GradBucket
        self.grad_bucket = bucket if bucket is not None else \
            GradBucket([self.embed_tokens.weight, self.embed_bytes.weight], symmetric="auto")
        return self.grad_bucket

    def forward(self, token_inputs: torch.Tensor, byte_inputs: Optional[torch.Tensor] = None):
        assert token_inputs.ndim == 1
        if byte_inputs is None and self.ttb is None:
            raise RuntimeError("MoTSplitResidualEmbedding: byte_inputs=None derives the ids from a ttb table: pass ttb=")
        Et, Eb, b = self.embed_tokens.weight, self.embed_bytes.weight, self.grad_bucket
        x, x0t, x0b = split_residual(token_inputs, byte_inputs, Et, Eb, self.lambdas.flip(0), bpt=self.bpt,
                                     ttb=self.ttb if byte_inputs is None else None, seq_len=token_inputs.numel(),
                                     pull=self.pull_in, grad_bufs=((Et, b.view_of(Et)), (Eb, b.view_of(Eb)), b)
                                     if b is not None else None)
        return x[None], x0t[None], x0b[None]


class TokenValueEmbeddings(nn.Module):
    """The value embeddings that share the token ids with the embedding front (SURVEY 8f-2): parameters
    `value_embeds.{0,1,2}.weight` [vocab, model_dim] (runs/7:252; spt/train_gpt.py:566); forward(token_inputs) ->
    `[value_embed(token_inputs) for value_embed in self.value_embeds]` (runs/7:308; spt/train_gpt.py:600).  One token
    sort serves the three dense gradient scatters."""

    def __init__(self, vocab_size: int, model_dim: int, n_tables: int = 3):
        super().__init__()
        self.value_embeds = nn.ModuleList([nn.Embedding(vocab_size, model_dim) for _ in range(n_tables)])
        self.grad_bucket = None

    def attach_grad_bucket(self, bucket=None):
        """Data parallelism: the backward writes the dense gradients of the tables straight into `bucket` (default: a
        bucket of these tables, all of them row tables) and marks the gathered rows, so that the per-table all-reduces
        of the reference (runs/7:697-700) become one `bucket.all_reduce_avg()` that moves only the rows some rank
        gathered.  A bucket shared with the front lists its token table and these tables as its row tables:
        `GradBucket([front.embed_tokens.weight, *(m.weight for m in ve.value_embeds), front.embed_bytes.weight],
        row_tables=4)`.  Call after the module is on its device and in its final dtype."""
        from .dp import GradBucket
        tables = [m.weight for m in self.value_embeds]
        self.grad_bucket = bucket if bucket is not None else GradBucket(tables, symmetric="auto", row_tables=len(tables))
        return self.grad_bucket

    def forward(self, token_inputs: torch.Tensor):
        outs = tok_gather(token_inputs, *[m.weight for m in self.value_embeds], grad_bucket=self.grad_bucket)
        return [o.view(*token_inputs.shape, -1) for o in outs]


class MoTValueEmbeddings(nn.Module):
    """runs/9_mot-in_mot-valemb.py:252-254,311-313 (V6): three value embeddings, each a concat + projection mix of a
    token table and a byte table.  Parameters `value_embeds_toks.{i}.weight` [token_vocab, token_dim],
    `value_embeds_bytes.{i}.weight` [token_vocab, byte_dim] (the reference sizes the byte value tables by the TOKEN
    vocabulary; only the first byte_vocab rows are ever indexed) and `value_byte_mixin_weights.{i}`
    [token_dim, token_dim + bpt*byte_dim] bf16.  forward(token_inputs [T], byte_inputs [1, T*bpt]) -> list of three
    [1, T, token_dim]."""

    def __init__(self, token_vocab_size: int, byte_vocab_size: int, token_dim: int, byte_dim: int,
                 bytes_per_token: int = 16, n_tables: int = 3):
        super().__init__()
        self.bpt, self.byte_vocab = bytes_per_token, byte_vocab_size
        self.value_embeds_toks = nn.ModuleList([nn.Embedding(token_vocab_size, token_dim) for _ in range(n_tables)])
        self.value_embeds_bytes = nn.ModuleList([nn.Embedding(token_vocab_size, byte_dim) for _ in range(n_tables)])
        self.value_byte_mixin_weights = nn.ParameterList(
            [nn.Parameter(_init_linear_(torch.empty(token_dim, token_dim + bytes_per_token * byte_dim)).bfloat16())
             for _ in range(n_tables)])
        self.spec = MixSpec(**PROJ_VARIANTS["V1"])

    def forward(self, token_inputs: torch.Tensor, byte_inputs: torch.Tensor):
        assert token_inputs.ndim == 1
        outs = []
        for et, eb, w in zip(self.value_embeds_toks, self.value_embeds_bytes, self.value_byte_mixin_weights):
            # rows >= byte_vocab of the byte value table are never gathered: hand the kernels the live rows (autograd
            # pads their gradient back to the full table with zeros, like the reference's dense embedding backward)
            outs.append(mot_embed_proj(token_inputs, byte_inputs, et.weight, eb.weight[:self.byte_vocab], w, self.spec,
                                       bpt=self.bpt)[None])
        return outs


class _Holder(nn.Module):
    """Parameter container that only exists to reproduce the reference's state-dict keys."""


class SptByteMixEmbedding(nn.Module):
    """scaled-pre-train's `FlexibleEmbedding` + `ByteMixin(concat)` pair (spt/train_gpt.py:327-379,430-443,560-565)
    fused behind the same call: forward(tokens [B,S] int32, byte_tensor [B,S*bpt] int64 | None,
    byte_tensor_pulled [B,S*bpt] int64 | None) -> x [B,S,model_dim], the value `self.byte_mixin(*self.embed(...))`
    has at spt/train_gpt.py:605-606.  State-dict keys match the reference: `embed.embed_tokens.weight`,
    `embed.embed_bytes.weight`, `byte_mixin.mixin.mixin.weight` (fp32 master, cast to bf16 per call like
    CastedLinear, gradient returned in fp32).  byte_mixin_method "noop" gives norm(embed_tokens(tokens)).
    add_padded_and_pulled=True sums the padded and the pulled byte rows before the per-byte norm (:371-379).
    With the input ttb table `ttb` ([V, bpt], padded on the `padding_in` side), forward(tokens) alone derives the byte
    ids inside the kernels (both byte tensors None): the pulled ids of every row of S tokens with pull_in, else the
    padded ids.  A right pull (padding_in="right") reads a token's bytes from the tokens after it, so the last input
    tokens of a row need token S of the loader's window: forward(tokens, next_tokens=window[:, -1]) ([B]).
    Refused (no fallback): cross_attn, byte self-attention; a right pull from token ids without next_tokens."""

    def __init__(self, vocab_size: int, byte_vocab_size: int, token_dim: int, byte_dim: int, model_dim: int,
                 bytes_per_token: int = 16, byte_mixin_method: str = "concat", pull_in: bool = True,
                 add_padded_and_pulled: bool = False, use_byte_self_attn: bool = False,
                 ttb: Optional[torch.Tensor] = None, padding_in: str = "left"):
        super().__init__()
        if byte_mixin_method not in ("concat", "noop"):
            raise NotImplementedError(f"mot_b200: byte_mixin_method={byte_mixin_method!r} is attention pooling, "
                                      "not a gather/pool; it has no kernel here (no fallback)")
        if use_byte_self_attn:
            raise NotImplementedError("mot_b200: use_byte_self_attn=True is not supported (no fallback)")
        self.method, self.bpt, self.pull_in = byte_mixin_method, bytes_per_token, pull_in
        self.add_padded_and_pulled = bool(add_padded_and_pulled) and pull_in and byte_mixin_method == "concat"  # :334-341
        self.embed = _Holder()
        self.embed.embed_tokens = nn.Embedding(vocab_size, token_dim if byte_mixin_method != "noop" else model_dim)
        self.byte_mixin = _Holder()
        if byte_mixin_method == "concat":
            self.embed.embed_bytes = nn.Embedding(byte_vocab_size, byte_dim)
            self.byte_mixin.mixin = _Holder()
            self.byte_mixin.mixin.mixin = _Holder()
            self.byte_mixin.mixin.mixin.weight = nn.Parameter(
                _init_linear_(torch.empty(model_dim, token_dim + bytes_per_token * byte_dim)))
        self.spec = MixSpec(combine="concat", tok_norm=True, byte_norm=True, out_norm=True)
        if padding_in not in ("left", "right"):
            raise ValueError(f"padding_in must be 'left' or 'right', got {padding_in!r}")
        self.padding_in = padding_in
        self.register_buffer("ttb", ttb, persistent=False)

    def forward(self, tokens: torch.Tensor, byte_tensor: Optional[torch.Tensor] = None,
                byte_tensor_pulled: Optional[torch.Tensor] = None, *,
                next_tokens: Optional[torch.Tensor] = None) -> torch.Tensor:
        B, S = tokens.shape
        if self.method == "noop":   # _forward_tokens, :342-348
            x = mot_embed(tokens, None, self.embed.embed_tokens.weight, None, MixSpec(combine="tok_only"))
            return x.view(B, S, -1)
        if byte_tensor is None and byte_tensor_pulled is None and self.ttb is not None:
            return self._forward_from_tokens(tokens, next_tokens)
        ids = byte_tensor_pulled if self.pull_in else byte_tensor   # _forward_bytes_pulled / _padded, :350-369
        if ids is None:
            raise RuntimeError("mot_b200: byte ids are required (byte_tensor_pulled with pull_in, else byte_tensor)")
        ids2 = None
        if self.add_padded_and_pulled:                              # _forward_bytes_padded_and_pulled, :371-379
            if byte_tensor is None:
                raise RuntimeError("mot_b200: add_padded_and_pulled needs byte_tensor and byte_tensor_pulled")
            ids, ids2 = byte_tensor, byte_tensor_pulled
        x = mot_embed_proj(tokens, ids, self.embed.embed_tokens.weight, self.embed.embed_bytes.weight,
                           self.byte_mixin.mixin.mixin.weight, self.spec, bpt=self.bpt, byte_ids2=ids2)
        return x.view(B, S, -1)

    def _forward_from_tokens(self, tokens: torch.Tensor, next_tokens: Optional[torch.Tensor]) -> torch.Tensor:
        B, S = tokens.shape
        if self.pull_in and self.padding_in == "right" and next_tokens is None:
            raise NotImplementedError("mot_b200: pulled ids of right-padded rows need the token after the last input; "
                                      "pass next_tokens= (the last column of the loader's window) or byte_tensor_pulled")
        spec = dataclasses.replace(self.spec, ttb_pull=self.pull_in and not self.add_padded_and_pulled,
                                   ttb_pull_side=self.padding_in)
        x = mot_embed_proj(tokens, None, self.embed.embed_tokens.weight, self.embed.embed_bytes.weight,
                           self.byte_mixin.mixin.mixin.weight, spec, bpt=self.bpt, ttb=self.ttb, seq_len=S,
                           padded_and_pulled=self.add_padded_and_pulled, next_tokens=next_tokens)
        return x.view(B, S, -1)


class DigitMixinEmbedding(nn.Module):
    """mathblations' `wte` + `dte` + `DigitMixinConcat` (mathblations/model.py:304-305,256-268,323-327) fused behind one
    call: forward(idx [B,S] int64, digits [B, S*dpt] int64) -> `digit_mixin(wte(idx), dte(digits))` = fc([digits | tok])
    with bias, no norms, fp32 parameters on the TF32 tensor-core path (main.py:522 sets matmul precision 'high').
    State-dict keys as in the reference GPT: `wte.weight`, `dte.weight`, `digit_mixin.fc.weight`, `digit_mixin.fc.bias`.
    `digit_mixin_method="cross_attn"` and `use_digit_self_attn` are refused (attention, not a gather/pool)."""

    def __init__(self, vocab_size: int, n_embd_tok: int, n_embd_digit: int, length_factor: int,
                 digit_mixin_method: str = "concat", use_digit_self_attn: bool = False, n_digit_vocab: int = 14):
        super().__init__()
        if digit_mixin_method != "concat" or use_digit_self_attn:
            raise NotImplementedError("mot_b200: only the concat digit mixin without digit self-attention has a kernel")
        self.dpt = length_factor
        self.wte = nn.Embedding(vocab_size, n_embd_tok)
        self.dte = nn.Embedding(n_digit_vocab, n_embd_digit)
        self.digit_mixin = _Holder()
        self.digit_mixin.fc = nn.Linear(n_embd_tok + n_embd_digit * length_factor, n_embd_tok)
        self.spec = MixSpec(combine="concat", out_norm=False, bytes_first=True)

    def forward(self, idx: torch.Tensor, digits: torch.Tensor) -> torch.Tensor:
        B, S = idx.shape
        x = mot_embed_proj(idx, digits, self.wte.weight, self.dte.weight, self.digit_mixin.fc.weight, self.spec,
                           bpt=self.dpt, bias=self.digit_mixin.fc.bias)
        return x.view(B, S, -1)
