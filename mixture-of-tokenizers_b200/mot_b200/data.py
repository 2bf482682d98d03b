"""The data side of the path (SURVEY 8f-4 and the batch builder between the loader and the embedding): shard files ->
pinned host tokens -> device -> (toks_in, bytes_padded_in, bytes_pulled_in, targets), with the ttb expansion and the
byte pulls on the device through libmot_b200 (no host loops, no host syncs).

Reference: `_load_data_shard` / `load_data_shard` / `distributed_data_generator` (spt/train_gpt.py:628-806); the eight
`_create_data_from_toks_*` closures (:686-764); shard format of modded-nanogpt/data/fineweb.py:28-50 (256 x int32
header: magic 20240520, version 1, token count; then uint16 tokens, or int32 for the pre-expanded `bytes/` shards)."""
from __future__ import annotations

import glob
import os
import random
from typing import Iterator, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import _lib as L
from .ops import _on_device, _ptr, _require_cuda, _stream, pull_from_left, pull_from_right, ttb_expand

SHARD_MAGIC, SHARD_VERSION, HEADER_INTS = 20240520, 1, 256


def write_data_shard(path: str, tokens: np.ndarray) -> None:
    """The writer side of the format (modded-nanogpt/data/fineweb.py:28-50), used by the tests and for synthetic shards."""
    tokens = np.asarray(tokens)
    if tokens.dtype not in (np.uint16, np.int32):
        raise TypeError("shard tokens are uint16 (token shards) or int32 (`bytes/` shards)")
    header = np.zeros(HEADER_INTS, dtype=np.int32)
    header[0], header[1], header[2] = SHARD_MAGIC, SHARD_VERSION, tokens.size
    with open(path, "wb") as f:
        f.write(header.tobytes())
        f.write(tokens.tobytes())


def load_data_shard(path: str, dtype: Optional[torch.dtype] = None, pin_memory: bool = True) -> torch.Tensor:
    """`_load_data_shard` (spt/train_gpt.py:628-638): header checked with the reference's assertions, tokens read
    straight into (pinned) host memory.  Unlike the reference the tokens keep their on-disk dtype (uint16): they are
    widened on the device (`tokens_to_device`), not on the host."""
    if dtype is None:
        dtype = torch.int32 if "bytes/" in str(path).replace(os.sep, "/") else torch.uint16   # :645
    with open(path, "rb", buffering=0) as f:
        header = np.frombuffer(f.read(HEADER_INTS * 4), dtype=np.int32)
        assert header.size == HEADER_INTS and header[0] == SHARD_MAGIC, \
            f"magic number mismatch in the data .bin file: {header[0] if header.size else None}"
        assert header[1] == SHARD_VERSION, f"unsupported version, expected 1 but got {header[1]}"
        num_tokens = int(header[2])
        tokens = torch.empty(num_tokens, dtype=dtype, pin_memory=pin_memory and torch.cuda.is_available())
        got = f.readinto(tokens.numpy())
        assert got == num_tokens * tokens.element_size(), "number of tokens read does not match header"
    return tokens


def tokens_to_device(tokens: torch.Tensor, device) -> torch.Tensor:
    """Host tokens (uint16 or int32, any shape) -> int32 on `device`.  uint16 is uploaded as is (2 bytes per token over
    PCIe) and widened by mot_tokens_widen_u16."""
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("mot_b200: tensors must be on a CUDA device (no CPU fallback)")
    if tokens.dtype == torch.int32:
        return tokens.to(dev, non_blocking=True)
    if tokens.dtype != torch.uint16:
        raise NotImplementedError("mot_b200.tokens_to_device: uint16 or int32 tokens")
    src = tokens.contiguous().to(dev, non_blocking=True)
    out = torch.empty(src.shape, dtype=torch.int32, device=dev)
    if src.numel():
        with _on_device(dev):
            rc = L.lib().mot_tokens_widen_u16(_ptr(src), src.numel(), _ptr(out), _stream(dev))
        L.check(rc, "mot_tokens_widen_u16")
    return out


def create_batch(toks: torch.Tensor, ttb_in: Optional[torch.Tensor], ttb_out: Optional[torch.Tensor], bytes_per_token: int, *,
                 byte_in: bool = True, pull_in: bool = True, byte_out: bool = False, pull_out: bool = False,
                 padding_in: str = "left", padding_out: str = "left", pad_byte: int = 456, eot_byte: int = 457,
                 byte_ids: bool = True, next_tokens: bool = False):
    """The `_create_data_from_toks_*` family (spt/train_gpt.py:686-764) for toks [B, S+1] on the device ->
    (toks_in [B,S], bytes_padded_in [B,S*bpt] | None, bytes_pulled_in | None, targets).  (byte_in, pull_in, byte_out,
    pull_out) = (byte_mixin_method != "noop", pull_in, byte_mixout_method != "noop", pull_out) as at :766-779; invalid
    combinations raise KeyError like the reference's dict lookup.  byte_ids=False skips the input byte tensors (both
    None): a loader then ships token ids only and the embedding derives the ids from its ttb table.  next_tokens=True
    appends a fifth element, the window's last column toks[:, -1] as int32 [B]: the lookahead a right pull of token ids
    alone needs (with byte_out the targets hold byte ids, so this is the only place the caller gets that token)."""
    _require_cuda(toks, ttb_in, ttb_out)
    key = (bool(byte_in), bool(pull_in), bool(byte_out), bool(pull_out))
    valid = {(True, True, True, True), (True, False, True, True), (True, True, True, False), (True, True, False, False),
             (False, False, True, True), (False, False, True, False), (True, False, False, False), (False, False, False, False)}
    if key not in valid:
        raise KeyError(key)
    bpt = bytes_per_token
    pull = {"left": pull_from_left, "right": pull_from_right}
    bytes_padded_in = bytes_pulled_in = None
    if byte_in and byte_ids:
        full = ttb_expand(toks, ttb_in)                                                # tokens_to_bytes(toks, ttb_in)
        if pull_in:
            bytes_pulled_in = pull[padding_in](full, bpt, pad_byte, eot_byte)[:, :-bpt].contiguous()
        bytes_padded_in = full[:, :-bpt].contiguous()
    if byte_out:
        out_full = ttb_expand(toks, ttb_out)
        if pull_out:
            out_full = pull[padding_out](out_full, bpt, pad_byte, eot_byte)
        targets = out_full[:, bpt:].contiguous()
    else:
        targets = toks[:, 1:].contiguous()
    if next_tokens:
        return (toks[:, :-1].contiguous(), bytes_padded_in, bytes_pulled_in, targets,
                toks[:, -1].to(torch.int32).contiguous())
    return toks[:, :-1].contiguous(), bytes_padded_in, bytes_pulled_in, targets


def distributed_data_generator(filename_patterns: Union[str, Sequence[str]], seq_len: int, batch_size: int, rank: int,
                               world_size: int, *, bytes_per_token: int, ttb_in: Optional[torch.Tensor] = None,
                               ttb_out: Optional[torch.Tensor] = None, byte_in: bool = True, pull_in: bool = True,
                               byte_out: bool = False, pull_out: bool = False, padding_in: str = "left",
                               padding_out: str = "left", device="cuda", seed: int = 12345,
                               byte_ids: bool = True, next_tokens: bool = False) -> Iterator[Tuple]:
    """`distributed_data_generator` (spt/train_gpt.py:651-806): same shard order (sorted glob, `random.seed(seed)`
    shuffle), same windows (rank r takes `data[pos + r*local : pos + (r+1)*local]` viewed as [-1, seq_len+1]), batches
    built by create_batch on the device (byte_ids=False: token ids only; next_tokens=True: the fifth element, the
    lookahead of a right pull).  Raises StopIteration when the shards run out, like the reference."""
    if isinstance(filename_patterns, str):
        filename_patterns = [filename_patterns]
    files: List[str] = []
    for pat in filename_patterns:
        files.extend(sorted(glob.glob(pat)))
    rng = random.Random(seed)       # the reference seeds the global generator; same sequence, no global side effect
    rng.shuffle(files)
    assert batch_size % world_size == 0
    local_seq_len = seq_len + 1
    local_batch_size = (batch_size * local_seq_len) // world_size
    file_iter = iter(files)

    def next_shard() -> torch.Tensor:
        while True:
            f = next(file_iter)
            try:
                return load_data_shard(f)
            except AssertionError:
                pass

    try:
        data, pos = next_shard(), 0
    except StopIteration:
        return
    while True:
        if pos + batch_size * local_seq_len + 1 >= len(data):
            try:   # :799-801 verbatim: the new shard is appended to the WHOLE old buffer and the cursor restarts at 0
                data, pos = torch.cat([data, next_shard()]), 0
            except StopIteration:
                return
        window = data[pos + rank * local_batch_size:][:local_batch_size].view(-1, local_seq_len)
        pos += batch_size * local_seq_len
        yield create_batch(tokens_to_device(window, device), ttb_in, ttb_out, bytes_per_token, byte_in=byte_in, pull_in=pull_in,
                           byte_out=byte_out, pull_out=pull_out, padding_in=padding_in, padding_out=padding_out,
                           byte_ids=byte_ids, next_tokens=next_tokens)
