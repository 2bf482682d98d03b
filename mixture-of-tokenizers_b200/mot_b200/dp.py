"""Data-parallel plumbing of the path (the reference's only parallelism, SURVEY 2.2): tables are replicated, the
batch is sharded by rank, and the dense gradients of the three tensors the path owns are averaged across ranks.

Reference: `dist.broadcast(param, 0)` for every parameter at start (spt/train_gpt.py:1127-1128; runs/7:571-572) and one
`dist.all_reduce(param.grad, op=AVG)` per parameter per step (spt/train_gpt.py:1320-1321; runs/7:697-700).  Here the
gradients of the path live in ONE flat bucket `[embed_tokens.grad | embed_bytes.grad | mixin.grad ...]` that the
backward kernels write into directly, so the exchange is a single NCCL all-reduce (NVLS on NVSwitch) with no packing
copy.  Pure torch.distributed host logic: works with any backend (the CPU tests run it over gloo)."""
from __future__ import annotations

import os
import warnings
from typing import Iterable, List, Optional

import torch
import torch.distributed as dist


def shard_for_rank(tokens: torch.Tensor, pos: int, local: int, rank: int) -> torch.Tensor:
    """The reference's batch sharding: rank r takes tokens[pos + r*local : pos + (r+1)*local] (runs/7:468-474)."""
    return tokens[pos + rank * local: pos + (rank + 1) * local]


def broadcast_params(params: Iterable[torch.Tensor], src: int = 0, group=None) -> None:
    """Replicate the tables from rank `src` once (spt/train_gpt.py:1127-1128)."""
    if not (dist.is_available() and dist.is_initialized()):
        return
    for p in params:
        dist.broadcast(p.detach(), src, group=group)


def pick_algo(world: int, has_multicast: bool) -> str:
    """Which exchange runs the gradient bucket of this path (77 MB bf16 at the 124M shape) at `world` ranks of one
    NVSwitch node.  Per GPU and direction the in-switch reduction (NVLS) moves S (1 + 1/n) bytes, the peer-to-peer
    two-shot 2 S (n - 1) / n: P2P is less at n = 2, NVLS from n = 4 on; NCCL remains for everything else (no symmetric
    memory, other world sizes).  Measured on 8 x B200: profiles/r2_dp.md.  MOT_DP_ALGO=nvls|p2p|nccl forces one."""
    forced = os.environ.get("MOT_DP_ALGO", "").lower()
    if os.environ.get("MOT_DP_NCCL"):
        forced = "nccl"
    if forced in ("nvls", "p2p", "nccl"):
        if forced == "nvls" and not has_multicast:
            return "nccl"
        if forced == "p2p" and world not in (2, 4, 8):
            return "nccl"
        return forced
    if world == 2:
        return "p2p"
    if has_multicast and world >= 3:
        return "nvls"
    if world in (4, 8):
        return "p2p"
    return "nccl"


def default_slabs(world: int) -> int:
    """Vocabulary slabs of the pipelined step (mot_embed_bwd_slab + exchange_async): 1 = the backward in one piece, then one
    exchange.  Every extra slab costs a backward launch (ramp + tail, ~8 us) and an exchange launch with its entry
    barrier and drain (~12 us), and the exchange traffic slows the backward it runs beside.  Measured at 48K tokens /
    77 MB bucket (profiles/r2_dp.md): 2 ranks 254 / 258 / 274 us per step with 1 / 2 / 4 slabs, 8 ranks 289 / 299 / 328 us:
    the exchange (150-200 us) is twice the compute step (92 us) and link-bound, so hiding the 52 us backward behind it
    buys less than the slicing costs.  The default is therefore one piece; MOT_DP_SLABS=n / GradBucket(n_slabs=n) turn
    the pipeline on (it pays when the compute step is long against the per-slab overheads)."""
    return 1


_DP_STREAMS: dict = {}


def dp_stream(dev) -> torch.cuda.Stream:
    """Per-device stream on which the exchange kernels run beside the backward (high priority: its few CTAs should get
    their SMs as soon as a slab is ready)."""
    st = _DP_STREAMS.get(dev.index)
    if st is None:
        st = _DP_STREAMS[dev.index] = torch.cuda.Stream(device=dev, priority=-1)
    return st


class GradBucket:
    """One flat buffer holding the gradients of `params` back to back (each slice 16-byte aligned), with a view per
    parameter.  `views()` are handed to the backward kernels as their dense-gradient outputs (mot_embed_bwd
    overwrites every row, so no zeroing is needed), `attach()` points `param.grad` at them, `all_reduce_avg()`
    averages the whole bucket across ranks in one collective.

    With symmetric memory (CUDA, NVLink peers) the exchange is the library's own kernel (`mot_dp_exchange`: NVLS
    in-switch reduction or peer-to-peer two-shot) and can run as a PIPELINE beside the backward: the backward walks the
    vocabulary in `n_slabs` slabs (mot_embed_bwd_slab), `exchange_async(lo, hi, last)` averages the rows of a finished
    slab on a second stream while the next slab is computed, `wait()` joins.  This is the overlap the reference gets
    from its asynchronous per-parameter all-reduces (runs/7:697-711), inside the path.

    Touched-rows exchange: the first `row_tables` parameters are `[V, D_i]` tables gathered with the same token ids (the
    front's token table and the value embeddings, runs/7:252,308).  The backwards publish the rows their batch gathered
    (`mark_rows`) into one bitmap behind the bucket, and the exchange moves only the rows some rank gathered, in every
    row table at once; the parameters after them are exchanged dense."""

    def __init__(self, params: Iterable[torch.nn.Parameter], dtype: Optional[torch.dtype] = None, symmetric="auto",
                 group=None, n_slabs: Optional[int] = None, reserve_sms: int = 8, sparse_rows="auto", row_tables: int = 1):
        """symmetric=True / "auto" (CUDA, initialised process group with more than one rank): allocate the bucket in
        symmetric memory so that the library's own exchange kernels apply; False: ordinary memory, NCCL.
        row_tables=k > 1: params[:k] are 2-D tables of one row count V, indexed by the same token ids, with rows of a
        multiple of 16 bytes (ValueError otherwise); one bitmap of V bits covers all of them."""
        self.params: List[torch.nn.Parameter] = list(params)
        if not self.params:
            raise ValueError("GradBucket needs at least one parameter")
        self.dtype = dtype or self.params[0].dtype
        dev = self.params[0].device
        esz = torch.empty(0, dtype=self.dtype).element_size()
        align = max(1, 16 // esz)
        from ._lib import DP_MAX_ROW_TABLES
        self.row_tables = int(row_tables)
        if not 1 <= self.row_tables <= min(len(self.params), DP_MAX_ROW_TABLES):
            raise ValueError(f"GradBucket: row_tables={row_tables} must be 1 .. min(len(params), {DP_MAX_ROW_TABLES})")
        if self.row_tables > 1:
            tabs = self.params[:self.row_tables]
            if any(t.dim() != 2 for t in tabs):
                raise ValueError("GradBucket: row tables must be 2-D [V, D] tables")
            if len({t.shape[0] for t in tabs}) != 1:
                raise ValueError("GradBucket: row tables must share their row count V (one bitmap of token ids)")
            if any(t.shape[1] * esz % 16 for t in tabs):
                raise ValueError("GradBucket: row-table rows must be a multiple of 16 bytes")
        self.offsets, n = [], 0
        for p in self.params:
            if p.device != dev:
                raise ValueError("GradBucket: parameters on different devices")
            self.offsets.append(n)
            n += (p.numel() + align - 1) // align * align
        self._symm = None
        self._epoch = 1
        self.algo = "nccl"
        self.n_slabs = 1
        self.reserve_sms = int(reserve_sms)
        self._ev = None
        self._pending = False
        self.sparse_rows = False          # touched-rows exchange of params[:row_tables] ([V, D_i] tables) available
        self.bitmap = None
        self._rows_ready = False          # a mark since the last exchange: the bitmap holds this rank's rows
        self._fresh = set()               # ids of the row tables a backward overwrote since the last exchange
        self._bits_new = None             # the rows of a later mark, ORed into the bitmap
        n = (n + align - 1) // align * align
        # room for the touched-rows bitmap of the row tables behind the gradients (same symmetric allocation)
        words = (self.params[0].shape[0] + 31) // 32 if self.params[0].dim() == 2 else 0
        extra = (words * 4 + 15) // 16 * 16 // esz
        self.flat = None
        have_group = dist.is_available() and dist.is_initialized()
        world = dist.get_world_size(group) if have_group else 1
        if symmetric and dev.type == "cuda" and have_group and world > 1 and group is None \
                and self.dtype in (torch.bfloat16, torch.float32) and pick_algo(world, True) != "nccl":
            # Symmetric memory needs NVLink peers (and NVSwitch multicast for NVLS) and a driver with fabric support; where
            # it is missing the bucket is ordinary device memory and the exchange is NCCL's all-reduce (a library
            # collective on the same data, not a different code path for the kernels).
            try:
                import torch.distributed._symmetric_memory as symm_mem
                full = symm_mem.empty(n + extra, dtype=self.dtype, device=dev)
                full.zero_()
                hdl = symm_mem.rendezvous(full, dist.group.WORLD)
                algo = pick_algo(world, hdl.multicast_ptr != 0)
                if algo != "nccl":
                    self._full = full
                    self.flat, self._symm, self.algo = full[:n], hdl, algo
                    want_sparse = sparse_rows if sparse_rows != "auto" else not os.environ.get("MOT_DP_DENSE")
                    if want_sparse and words > 0 and (algo == "nvls" or world in (2, 4)) \
                            and all(t.is_contiguous() for t in self.params[:self.row_tables]):
                        self.sparse_rows = True
                        self.bitmap = full[n:].view(torch.int32)[:words]
                        self._bitmap_off = n * esz
                    self.n_slabs = max(1, int(os.environ.get("MOT_DP_SLABS", n_slabs if n_slabs is not None
                                                             else default_slabs(world))))
                    self._ev = torch.cuda.Event()
                    self._work = torch.zeros(64, dtype=torch.int32, device=dev)   # tile counters of the exchange launches
            except Exception as e:  # noqa: BLE001 - any allocator / rendezvous failure means "no symmetric memory here"
                warnings.warn(f"GradBucket: symmetric memory unavailable ({type(e).__name__}: {e}); using NCCL")
                self.flat = None
                self._symm = None
        if self.flat is None:
            self.flat = torch.zeros(n, dtype=self.dtype, device=dev)
        self._views = [self.flat[o:o + p.numel()].view(p.shape) for o, p in zip(self.offsets, self.params)]

    # ------------------------------------------------------------------------------------------------ views
    def views(self) -> List[torch.Tensor]:
        return self._views

    def view_of(self, param: torch.nn.Parameter) -> torch.Tensor:
        for p, v in zip(self.params, self._views):
            if p is param:
                return v
        raise KeyError("parameter is not in this bucket")

    def offset_of(self, param: torch.nn.Parameter) -> int:
        for p, o in zip(self.params, self.offsets):
            if p is param:
                return o
        raise KeyError("parameter is not in this bucket")

    def holds(self, param: torch.nn.Parameter) -> bool:
        return any(p is param for p in self.params)

    def is_row_table(self, param: torch.nn.Parameter) -> bool:
        return any(p is param for p in self.params[:self.row_tables])

    def attach(self) -> None:
        """param.grad = its slice of the bucket (grads of a different dtype are copied in, e.g. an fp32 master-weight
        gradient into a bf16 bucket is NOT done silently: dtypes must match)."""
        for p, v in zip(self.params, self._views):
            if p.grad is not None and p.grad.data_ptr() != v.data_ptr():
                if p.grad.dtype != self.dtype:
                    raise TypeError("GradBucket: gradient dtype differs from the bucket dtype")
                v.copy_(p.grad)
                self._fresh.discard(id(p))      # rows no bitmap describes: the next exchange is dense
            p.grad = v

    # ------------------------------------------------------------------------------------------------ exchange
    @property
    def pipelined(self) -> bool:
        """The exchange can run slab by slab beside the backward (own kernels over symmetric memory)."""
        return self._symm is not None and self.n_slabs > 1

    def _exchange(self, lo: int, hi: int, last: bool, stream: int) -> None:
        from . import _lib as L
        h = self._symm
        esz = self.flat.element_size()
        rc = L.lib().mot_dp_exchange(h.multicast_ptr if self.algo == "nvls" else None,
                                     h.buffer_ptrs_dev if self.algo == "p2p" else None, h.signal_pad_ptrs_dev,
                                     self._work.data_ptr(), h.rank,
                                     h.world_size, lo * esz, (hi - lo) * esz,
                                     L.BF16 if self.dtype == torch.bfloat16 else L.F32, self._epoch, 1 if last else 0,
                                     L.DP_NVLS if self.algo == "nvls" else L.DP_P2P, stream)
        L.check(rc, "mot_dp_exchange")
        self._epoch = (self._epoch + (2 if last else 1)) & 0xFFFFFFFF

    def mark_rows(self, desc, ws_buf: torch.Tensor, fresh: Iterable[torch.nn.Parameter] = ()) -> None:
        """Publish the rows of the row tables this rank's batch gathered (from the sort plan in `ws_buf`) for the
        touched-rows exchange; call after a backward that produced a row table's gradient, on its stream.  The next
        all_reduce_avg() then moves only the rows some rank gathered (rows that are zero everywhere stay as they are).
        The first mark after an exchange writes the bitmap, later ones (micro-batches, several modules) are ORed into
        it.  `fresh`: the row tables whose bucket view this backward overwrote.  A row table whose `.grad` is its view
        and was not overwritten since the last exchange holds rows no bitmap describes: that exchange is dense."""
        if not self.sparse_rows:
            return
        if desc.tok_vocab != self.params[0].shape[0]:
            raise ValueError(f"GradBucket.mark_rows: a plan over {desc.tok_vocab} rows for row tables of "
                             f"{self.params[0].shape[0]}")
        from . import _lib as L
        dev = self.flat.device
        merge = self._rows_ready
        if merge and self._bits_new is None:
            self._bits_new = torch.empty_like(self.bitmap)
        dst = self._bits_new if merge else self.bitmap
        with torch.cuda.device(dev):
            rc = L.lib().mot_embed_touched_rows(desc, ws_buf.data_ptr(), ws_buf.numel(), dst.data_ptr(),
                                                torch.cuda.current_stream(dev).cuda_stream)
            L.check(rc, "mot_embed_touched_rows")
            if merge:
                self.bitmap.bitwise_or_(self._bits_new)
        self._rows_ready = True
        self._fresh.update(id(p) for p in fresh)

    def _rows_describe_bucket(self) -> bool:
        """Every row table whose gradient is its bucket view was overwritten by a backward since the last exchange, so
        its nonzero rows are all in this rank's bitmap (the precondition of the touched-rows exchange)."""
        for p, v in zip(self.params[:self.row_tables], self._views):
            if p.grad is not None and p.grad.data_ptr() == v.data_ptr() and id(p) not in self._fresh:
                return False
        return True

    def rows_layout(self):
        """Byte layout of the touched-rows exchange -> ([(byte offset, row bytes) per row table], dense byte offset,
        dense bytes): the row tables lead the bucket, everything from params[row_tables] on is exchanged dense."""
        esz, k = self.flat.element_size(), self.row_tables
        tabs = [(o * esz, p.shape[1] * esz) for o, p in zip(self.offsets[:k], self.params[:k])]
        dense_lo = self.offsets[k] if len(self.offsets) > k else self.flat.numel()
        return tabs, dense_lo * esz, (self.flat.numel() - dense_lo) * esz

    def _exchange_rows(self, stream: int) -> None:
        from . import _lib as L
        h = self._symm
        tabs, dense_lo, dense_bytes = self.rows_layout()
        tables = (L.MotRowTable * len(tabs))(*[L.MotRowTable(o, rb, 0) for o, rb in tabs])
        rc = L.lib().mot_dp_exchange_rows_multi(h.multicast_ptr if self.algo == "nvls" else None,
                                                h.buffer_ptrs_dev if self.algo == "p2p" else None, h.signal_pad_ptrs_dev,
                                                self._work.data_ptr(), h.rank, h.world_size, tables, len(tabs),
                                                self.params[0].shape[0], self._bitmap_off, dense_lo, dense_bytes,
                                                L.BF16 if self.dtype == torch.bfloat16 else L.F32, self._epoch,
                                                L.DP_NVLS if self.algo == "nvls" else L.DP_P2P, stream)
        L.check(rc, "mot_dp_exchange_rows_multi")
        self._epoch = (self._epoch + 2) & 0xFFFFFFFF

    def exchange_async(self, lo: int, hi: int, last: bool) -> None:
        """Average elements [lo, hi) of the bucket (multiples of 16 bytes) across ranks on the exchange stream, ordered
        after everything queued on the current stream (the backward of that slab).  Every rank issues the same calls;
        the final range of a step passes last=True.  `wait()` joins the exchange stream into the current one."""
        if self._symm is None:
            raise RuntimeError("GradBucket.exchange_async needs the symmetric-memory bucket (own exchange kernels)")
        dev = self.flat.device
        cur = torch.cuda.current_stream(dev)
        side = dp_stream(dev)
        self._ev.record(cur)
        side.wait_event(self._ev)
        with torch.cuda.device(dev):
            self._exchange(lo, hi, last, side.cuda_stream)
        self._pending = True

    def wait(self) -> None:
        """The current stream waits for the exchange stream (no host synchronisation)."""
        if self._pending:
            dev = self.flat.device
            torch.cuda.current_stream(dev).wait_stream(dp_stream(dev))
            self._pending = False

    def all_reduce_avg(self, group=None, async_op: bool = False):
        """Average the whole bucket across ranks.  AVG = SUM / world_size (gloo has no AVG reduce op).  If the backward
        already exchanged its slabs (exchange_async) this only joins the exchange stream."""
        if not (dist.is_available() and dist.is_initialized()):
            return None
        world = dist.get_world_size(group)
        if self._symm is not None:
            if async_op or group is not None:
                raise NotImplementedError("GradBucket: the symmetric-memory exchange is stream-ordered on the whole world "
                                          "(async_op / sub-groups are NCCL features: build the bucket with symmetric=False)")
            rows = self._rows_ready and self._rows_describe_bucket()
            self._rows_ready = False
            self._fresh.clear()
            if self._pending:          # the slabs are already in flight on the exchange stream
                self.wait()
                return None
            dev = self.flat.device
            with torch.cuda.device(dev):
                if rows:                   # the backwards published their row bitmap: move only the rows of the union
                    self._exchange_rows(torch.cuda.current_stream(dev).cuda_stream)
                else:
                    self._exchange(0, self.flat.numel(), True, torch.cuda.current_stream(dev).cuda_stream)
            return None
        if dist.get_backend(group) == "nccl":
            return dist.all_reduce(self.flat, op=dist.ReduceOp.AVG, group=group, async_op=async_op)
        work = dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, group=group, async_op=False)
        self.flat.div_(world)
        return work
