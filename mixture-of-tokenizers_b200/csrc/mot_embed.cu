// Host side of the fused byte-mix embedding: validation, workspace layout, plan, C ABI.
#include <algorithm>

#include "mot_embed_bwd_sum.cuh"

namespace mot {

// ======================================================================================
// Backward plan: group positions by token id (counting sort over the vocabulary)
// ======================================================================================
__global__ void plan_hist_kernel(const int32_t* tok, long long N, int V, int* cnt) {
  pdl_launch_dependents();
  pdl_wait();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x)
    atomicAdd(&cnt[clampi(ld_g(tok + i), V - 1)], 1);
}

// Exclusive scan of the histogram -> segment offsets.  One 256-thread CTA per 1024-entry tile (four entries per
// thread): each CTA first sums every entry in front of its tile (coalesced 16-byte loads, all L2 hits), then scans
// its own tile with warp shuffles.  Small CTAs with few registers so that the plan can run beside the forward
// kernel on a second stream.
constexpr int kScanTile = 1024;
__global__ void __launch_bounds__(256) plan_scan_kernel(EmbedParams p) {
  __shared__ int wsum[8];
  __shared__ int wcarry[8];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int base = blockIdx.x * kScanTile;  // multiple of 4: the tile starts 16-byte aligned
  pdl_launch_dependents();
  pdl_wait();
  int carry = 0;
  for (int v = tid * 4; v < base; v += 256 * 4) {
    const int4 c = *reinterpret_cast<const int4*>(p.cnt + v);
    carry += c.x + c.y + c.z + c.w;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) carry += __shfl_xor_sync(0xffffffffu, carry, o);
  if (lane == 0) wcarry[warp] = carry;
  const int v0 = base + tid * 4;
  int c[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) c[j] = v0 + j < p.V ? p.cnt[v0 + j] : 0;
  const int mine = c[0] + c[1] + c[2] + c[3];
  int inc = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) wsum[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int cr = lane < 8 ? wcarry[lane] : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cr += __shfl_xor_sync(0xffffffffu, cr, o);
    const int w = lane < 8 ? wsum[lane] : 0;
    int wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi += t;
    }
    if (lane < 8) wsum[lane] = cr + wi - w;  // exclusive warp offset including the carry-in
  }
  __syncthreads();
  int ex = wsum[warp] + inc - mine;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (v0 + j < p.V) p.off[v0 + j] = ex;
    ex += c[j];
    if (v0 + j == p.V - 1) p.off[p.V] = ex;
  }
}

// Scatter every position into its token's segment of the stream (cursor = cnt, counted back down to 0).
// Leaves cnt all zero again (part of the self-cleaning workspace contract, MOT_WS_CLEAN).
__global__ void plan_fill_kernel(EmbedParams p) {
  pdl_launch_dependents();
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < p.N) {
    const int v = clampi(ld_g(p.tok + i), p.V - 1);
    const int slot = atomicSub(&p.cnt[v], 1) - 1;
    const int at = p.off[v] + slot;
    p.order[at] = (int)i;
    p.stok[at] = v;
  }
}

// Bitmap of the vocabulary rows this batch gathered (bit v of word v / 32 = off[v+1] > off[v]), for the touched-rows
// exchange of the data-parallel step (mot_dp_exchange_rows).  One warp per word.
__global__ void __launch_bounds__(256) plan_rowmap_kernel(const int* off, int V, uint32_t* bitmap) {
  pdl_launch_dependents();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int words = (V + 31) >> 5;
  for (int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < words; w += (gridDim.x * blockDim.x) >> 5) {
    const int v = (w << 5) + lane;
    const bool hit = v < V && ld_g(off + v + 1) > ld_g(off + v);
    const unsigned m = __ballot_sync(0xffffffffu, hit);
    if (lane == 0) bitmap[w] = m;
  }
}

__global__ void mot_lam_store_kernel(float* acc, float* g_lam) {
  pdl_launch_dependents();
  pdl_wait();
  if (threadIdx.x < 2) {
    g_lam[threadIdx.x] = acc[threadIdx.x];
    acc[threadIdx.x] = 0.f;  // self-cleaning workspace
  }
}

// ======================================================================================
// Host side
// ======================================================================================
// Stream chunk size: one chunk per backward warp of a full B200 (148 SMs x warps per CTA), so that every warp walks
// the same number of stream entries; chunks longer than one 32-entry batch are whole batches.  (A constant, not the
// current device's SM count: the workspace layout must not depend on the device.)
static int stream_chunk(long long n_tokens, int warps_per_cta) {
  const long long warps = 148LL * warps_per_cta;
  long long R = (n_tokens + warps - 1) / warps;
  if (R < 1) R = 1;
  if (R > 32) R = (R + 31) / 32 * 32;
  return (int)R;
}

// Chunk size when the backward runs as `n_slabs` vocabulary slabs beside the gradient exchange (mot_embed_bwd_slab): one
// chunk per warp of a launch that leaves up to 16 SMs to the exchange kernel, for a slab holding 1 / n_slabs of the
// stream (uniform token ids; a slab with more entries walks several chunks per warp).  A pure function of
// (n_tokens, n_slabs): the workspace layout depends on it.
constexpr int kDpReserveMax = 16;
static int stream_chunk_slab(long long n_tokens, int n_slabs, int warps_per_cta) {
  const long long warps = (148LL - kDpReserveMax) * warps_per_cta;
  const long long per_slab = (n_tokens + n_slabs - 1) / n_slabs;
  long long R = (per_slab + warps - 1) / warps;
  if (R < 1) R = 1;
  if (R > 32) R = (R + 31) / 32 * 32;
  return (int)R;
}

// The rules every descriptor obeys, the byte pair's too (mot_pair.cu).
int validate_desc(const MotDesc* d) {
  if (!d) return MOT_ERR_BAD_ARG;
  if (d->abi_version != MOT_B200_ABI_VERSION) return MOT_ERR_BAD_ARG;
  if (d->dtype != MOT_BF16 && d->dtype != MOT_F32) return MOT_ERR_UNSUPPORTED;
  if (d->n_tokens < 0 || d->n_tokens > 0x7fffffffLL) return MOT_ERR_BAD_ARG;
  if (d->combine < MOT_ADD || d->combine > MOT_MEAN) return MOT_ERR_UNSUPPORTED;
  const bool has_tok = d->combine != MOT_BYTES_ONLY, has_bytes = d->combine != MOT_TOK_ONLY;
  if (has_tok && (d->tok_vocab <= 0 || d->tok_dim <= 0)) return MOT_ERR_BAD_ARG;
  if (has_tok && d->tok_dim % 8) return MOT_ERR_MISALIGNED;
  if (has_bytes) {
    if (d->byte_vocab <= 0 || d->byte_dim <= 0 || d->bpt <= 0 || d->bpt > 32) return MOT_ERR_BAD_ARG;
    if (d->byte_dim % 8) return MOT_ERR_MISALIGNED;
  }
  if (d->out_dim <= 0 || d->out_dim % 8) return MOT_ERR_MISALIGNED;
  const long long db = (long long)d->bpt * d->byte_dim;
  switch (d->combine) {
    case MOT_ADD: if (d->tok_dim != db || d->out_dim != d->tok_dim) return MOT_ERR_BAD_ARG; break;
    case MOT_CONCAT: if (d->out_dim != d->tok_dim + db) return MOT_ERR_BAD_ARG; break;
    case MOT_TOK_ONLY: if (d->out_dim != d->tok_dim) return MOT_ERR_BAD_ARG; break;
    case MOT_BYTES_ONLY: if (d->out_dim != db) return MOT_ERR_BAD_ARG; break;
    case MOT_MEAN: if (d->byte_dim != d->tok_dim || d->out_dim != d->tok_dim) return MOT_ERR_BAD_ARG; break;
  }
  if (d->row_stride != 0 || d->col_offset != 0) {  // a column slice of wider rows
    const long long ld = d->row_stride ? d->row_stride : d->out_dim;
    if (d->col_offset < 0 || ld < (long long)d->col_offset + d->out_dim || ld > 0x7fffffffLL) return MOT_ERR_BAD_ARG;
    if (ld % 8 || d->col_offset % 8) return MOT_ERR_MISALIGNED;
  }
  if (d->dp_slabs < 0 || d->dp_slabs > 64) return MOT_ERR_BAD_ARG;
  if ((d->flags & MOT_F_TTB_PULL_LEFT) && (d->flags & MOT_F_TTB_PULL_RIGHT)) return MOT_ERR_BAD_ARG;
  if ((d->flags & MOT_F_TTB_NEXT_TOK) && !(d->flags & MOT_F_TTB_PULL_RIGHT)) return MOT_ERR_BAD_ARG;
  if ((d->flags & MOT_F_IDS_FROM_TTB) && has_bytes) {
    if (d->ttb_dtype < MOT_TTB_I16 || d->ttb_dtype > MOT_TTB_BF16) return MOT_ERR_UNSUPPORTED;
    if (d->flags & (MOT_F_TTB_SCRAMBLE | MOT_F_TTB_PULL_LEFT | MOT_F_TTB_PULL_RIGHT))
      if (d->seq_len <= 0 || d->n_tokens % d->seq_len) return MOT_ERR_BAD_ARG;
    if (d->flags & (MOT_F_TTB_PULL_LEFT | MOT_F_TTB_PULL_RIGHT)) {
      if (d->tok_vocab <= 0) return MOT_ERR_BAD_ARG;  // rows of the ttb table, also without a token table
      if (d->pad_id != (int16_t)d->pad_id || d->eot_id != (int16_t)d->eot_id) return MOT_ERR_BAD_ARG;  // int16, as in mot_pull
    }
  }
  return MOT_OK;
}

// validate_desc plus the capacity of the fused kernels.
static int validate(const MotDesc* d) {
  if (int rc = validate_desc(d)) return rc;
  if ((d->flags & MOT_F_BYTE_NORM) && d->combine != MOT_TOK_ONLY && d->byte_dim > 256) return MOT_ERR_UNSUPPORTED;
  // a lane holds at most 8 chunks of 8 elements per launch: 2048 columns.  A concat without a norm over the whole row
  // runs as two launches (concat_splits), so the cap applies to each half: the widest reference operand
  // (spt/experiments100_000steps.sh: 1024 + 16 x 128 = 3072 columns) fits.
  constexpr int kMaxCols = 8 * 32 * 8;
  if (d->combine == MOT_CONCAT && !(d->flags & (MOT_F_OUT_NORM | MOT_F_HAS_LAMBDAS))) {
    if (d->tok_dim > kMaxCols || (long long)d->bpt * d->byte_dim > kMaxCols) return MOT_ERR_UNSUPPORTED;
  } else if (d->out_dim > kMaxCols) {
    return MOT_ERR_UNSUPPORTED;
  }
  return MOT_OK;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

static void fill_params(const MotDesc* d, EmbedParams& p) {
  p = EmbedParams{};
  p.N = d->n_tokens;
  p.T = d->seq_len > 0 ? d->seq_len : (d->n_tokens > 0 ? d->n_tokens : 1);
  p.V = d->tok_vocab;
  p.Vb = d->combine == MOT_TOK_ONLY ? 0 : d->byte_vocab;
  p.bpt = d->combine == MOT_TOK_ONLY ? 0 : d->bpt;
  p.Dt = d->combine == MOT_BYTES_ONLY ? 0 : d->tok_dim;
  p.bd = d->combine == MOT_TOK_ONLY ? 8 : d->byte_dim;
  p.Do = d->out_dim;
  p.combine = d->combine;
  p.flags = d->flags;
  p.ttb_dtype = d->ttb_dtype;
  p.pad_eot = (d->pad_id & 0xffff) | (d->eot_id << 16);
  p.n_chunks = d->out_dim / kChunk;
  p.io_ld = d->row_stride ? d->row_stride : d->out_dim;
  p.io_col = d->col_offset;
  p.eps = d->eps;
  p.R = stream_chunk(d->n_tokens, kBwdThreads / 32);  // the saved-output kernel re-chunks for its own CTA size
  p.n_rep = kByteRep;
  p.stages = 4;
  p.tab_smem = 1;
  p.v_lo = 0;
  p.v_hi = p.V;
  p.last_slab = 1;
}

// A concat without a norm over the concatenated row and without lambdas (the [tok | bytes] operand of the projection
// variants, runs/7:226-232) is two independent halves: columns [0, Dt) depend on the token only, the rest on the byte
// ids only.  They run as a tok-only and a bytes-only launch over the strided rows: half the row per lane (no register
// spills at 2048-wide rows), and the bytes half needs neither the token rows nor the sorted stream.
static bool concat_splits(const MotDesc* d) {
  return d->combine == MOT_CONCAT && !(d->flags & (MOT_F_OUT_NORM | MOT_F_HAS_LAMBDAS));
}
static void split_params(const MotDesc* d, EmbedParams& pt, EmbedParams& pb) {
  const int db = d->bpt * d->byte_dim;
  const bool bytes_first = (d->flags & MOT_F_BYTES_FIRST) != 0;
  MotDesc dt = *d, dbd = *d;
  dt.combine = MOT_TOK_ONLY;
  dt.out_dim = d->tok_dim;
  dt.flags = d->flags & MOT_F_TOK_NORM;
  dbd.combine = MOT_BYTES_ONLY;
  dbd.out_dim = db;
  dbd.flags = d->flags & ~(MOT_F_TOK_NORM | MOT_F_BYTES_FIRST);
  fill_params(&dt, pt);
  fill_params(&dbd, pb);
  pt.io_ld = pb.io_ld = d->row_stride ? d->row_stride : d->out_dim;
  pt.io_col = d->col_offset + (bytes_first ? db : 0);
  pb.io_col = d->col_offset + (bytes_first ? 0 : d->tok_dim);
}

struct WsLayout {
  size_t cnt, byte_acc, lam_acc, partial, zero_end, off, order, stok, total;
};

static WsLayout ws_layout(const EmbedParams& p, int dp_slabs = 0) {
  WsLayout w{};
  const long long V = p.V > 0 ? p.V : 1, N = p.N > 0 ? p.N : 1;
  // one fp32 slot per stream chunk, sized for the finest chunking in use (recompute / saved-output kernel / the slabs of
  // the data-parallel pipeline when the descriptor announces them)
  int r_min = std::min(p.R, stream_chunk(N, kSumThreads / 32));
  if (dp_slabs > 1) r_min = std::min(r_min, stream_chunk_slab(N, dp_slabs, kSumThreads / 32));
  const long long n_stream_chunks = (N + r_min - 1) / r_min;
  size_t o = 0;
  auto take = [&](size_t bytes) {
    size_t at = o;
    o = align_up(o + bytes, 256);
    return at;
  };
  // zeroed region first: cnt | byte_acc | lam_acc | partial (one memset, only when the caller does not pass MOT_WS_CLEAN)
  w.cnt = take((size_t)V * 4);
  w.byte_acc = take((size_t)p.n_rep * (p.Vb > 0 ? p.Vb : 1) * p.bd * 4);
  w.lam_acc = take(16);
  w.partial = take((size_t)n_stream_chunks * (p.Dt > 0 ? p.Dt : 8) * 4);
  w.zero_end = o;
  w.off = take((size_t)(V + 1) * 4);
  w.order = take((size_t)N * 4);
  w.stok = take((size_t)N * 4);
  w.total = o;
  return w;
}

static void bind_ws(EmbedParams& p, const WsLayout& w, void* ws) {
  char* b = reinterpret_cast<char*>(ws);
  p.cnt = reinterpret_cast<int*>(b + w.cnt);
  p.byte_acc = reinterpret_cast<float*>(b + w.byte_acc);
  p.lam_acc = reinterpret_cast<float*>(b + w.lam_acc);
  p.off = reinterpret_cast<int*>(b + w.off);
  p.order = reinterpret_cast<int*>(b + w.order);
  p.stok = reinterpret_cast<int*>(b + w.stok);
  p.partial = reinterpret_cast<float*>(b + w.partial);
  p.chk = chk_record();
  p.n_slots = (int)((w.zero_end - w.partial) / ((size_t)(p.Dt > 0 ? p.Dt : 8) * 4));
}

static int run_plan(const EmbedParams& p, cudaStream_t s) {
  if (p.combine == MOT_BYTES_ONLY || p.N == 0) return MOT_OK;
  long long hb = (p.N + 255) / 256;
  if (hb > 2048) hb = 2048;
  launch_pdl(plan_hist_kernel, dim3((unsigned)hb), dim3(256), 0, s, p.tok, p.N, p.V, p.cnt);
  launch_pdl(plan_scan_kernel, dim3((unsigned)((p.V + kScanTile - 1) / kScanTile)), dim3(256), 0, s, p);
  launch_pdl(plan_fill_kernel, dim3((unsigned)((p.N + 255) / 256)), dim3(256), 0, s, p);
  count_launch(3);
  return check_launch();
}

}  // namespace mot

using namespace mot;

extern "C" size_t mot_embed_workspace_bytes(const MotDesc* d) {
  if (validate(d) != MOT_OK) return 0;
  EmbedParams p;
  fill_params(d, p);
  return ws_layout(p, d->dp_slabs).total;
}

extern "C" int mot_embed_fwd(const MotDesc* d, const int32_t* tok, const void* byte_ids, const void* ttb,
                             const void* E_tok, const void* E_byte, const float* lam, void* out, void* stream) {
  return mot_embed_fwd_ex(d, tok, byte_ids, ttb, E_tok, E_byte, lam, nullptr, out, nullptr, stream);
}

extern "C" int mot_embed_fwd_ex(const MotDesc* d, const int32_t* tok, const void* byte_ids, const void* ttb,
                                const void* E_tok, const void* E_byte, const float* lam, const void* addend, void* out,
                                float* rstd_out, void* stream) {
  if (int rc = validate(d)) return rc;
  if (addend && (concat_splits(d) || d->row_stride != 0 || d->col_offset != 0)) return MOT_ERR_UNSUPPORTED;
  if (!aligned16(addend)) return MOT_ERR_MISALIGNED;
  if (d->n_tokens == 0) return MOT_OK;  // empty batch: nothing to write (empty tensors have null pointers)
  const bool has_tok = d->combine != MOT_BYTES_ONLY, has_bytes = d->combine != MOT_TOK_ONLY;
  if (!out || (has_tok && (!tok || !E_tok)) || (has_bytes && !E_byte)) return MOT_ERR_BAD_ARG;
  if (has_bytes) {
    if (d->flags & MOT_F_IDS_FROM_TTB) { if (!ttb || !tok) return MOT_ERR_BAD_ARG; }
    else if (!byte_ids) return MOT_ERR_BAD_ARG;
  }
  if ((d->flags & MOT_F_HAS_LAMBDAS) && !lam) return MOT_ERR_BAD_ARG;
  if (!aligned16(out) || !aligned16(E_tok) || !aligned16(E_byte)) return MOT_ERR_MISALIGNED;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (concat_splits(d)) {
    EmbedParams pt, pb;
    split_params(d, pt, pb);
    for (EmbedParams* q : {&pt, &pb}) {
      q->tok = tok; q->ids = byte_ids; q->ttb = ttb; q->E_tok = E_tok; q->E_byte = E_byte; q->lam = lam; q->out = out;
      if (int rc = d->dtype == MOT_BF16 ? dispatch_fwd_bf16(*q, s) : dispatch_fwd_f32(*q, s)) return rc;
    }
    return MOT_OK;
  }
  EmbedParams p;
  fill_params(d, p);
  p.tok = tok; p.ids = byte_ids; p.ttb = ttb; p.E_tok = E_tok; p.E_byte = E_byte; p.lam = lam; p.out = out;
  p.rstd_out = (d->flags & MOT_F_OUT_NORM) ? rstd_out : nullptr;
  p.addend = addend;
  if (addend) return d->dtype == MOT_BF16 ? dispatch_fwd_addend_bf16(p, s) : dispatch_fwd_addend_f32(p, s);
  return d->dtype == MOT_BF16 ? dispatch_fwd_bf16(p, s) : dispatch_fwd_f32(p, s);
}

extern "C" int mot_embed_workspace_init(const MotDesc* d, void* workspace, size_t ws_bytes, void* stream) {
  if (int rc = validate(d)) return rc;
  if (!workspace) return MOT_ERR_BAD_ARG;
  EmbedParams p;
  fill_params(d, p);
  const WsLayout w = ws_layout(p, d->dp_slabs);
  if (ws_bytes < w.total) return MOT_ERR_WORKSPACE;
  if (cudaMemsetAsync(workspace, 0, w.zero_end, reinterpret_cast<cudaStream_t>(stream)) != cudaSuccess) return check_launch();
  return MOT_OK;
}

extern "C" int mot_embed_plan(const MotDesc* d, const int32_t* tok, void* workspace, size_t ws_bytes, int32_t ws_flags,
                              void* stream) {
  if (int rc = validate(d)) return rc;
  if (!workspace) return MOT_ERR_BAD_ARG;
  if (d->combine != MOT_BYTES_ONLY && !tok) return MOT_ERR_BAD_ARG;
  EmbedParams p;
  fill_params(d, p);
  const WsLayout w = ws_layout(p, d->dp_slabs);
  if (ws_bytes < w.total) return MOT_ERR_WORKSPACE;
  if (!aligned16(workspace)) return MOT_ERR_MISALIGNED;
  bind_ws(p, w, workspace);
  p.tok = tok;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  // zero cnt | byte_acc | lam_acc (contiguous at the head of the workspace) unless the caller vouches for it
  if (!(ws_flags & MOT_WS_CLEAN) && cudaMemsetAsync(workspace, 0, w.zero_end, s) != cudaSuccess) return check_launch();
  return run_plan(p, s);
}

extern "C" int mot_embed_plan_async(const MotDesc* d, const int32_t* tok, void* workspace, size_t ws_bytes, int32_t ws_flags,
                                    void* main_stream, void* side_stream, void* ev_fork, void* ev_join) {
  if (!side_stream || !ev_fork || !ev_join) return MOT_ERR_BAD_ARG;
  cudaStream_t ms = reinterpret_cast<cudaStream_t>(main_stream), ss = reinterpret_cast<cudaStream_t>(side_stream);
  cudaEvent_t ef = reinterpret_cast<cudaEvent_t>(ev_fork), ej = reinterpret_cast<cudaEvent_t>(ev_join);
  // fork: the plan starts after everything already queued on the main stream (token ids ready, the previous
  // backward done with the workspace) and runs beside whatever the caller queues next (the forward kernel)
  if (cudaEventRecord(ef, ms) != cudaSuccess || cudaStreamWaitEvent(ss, ef, 0) != cudaSuccess) return check_launch();
  if (int rc = mot_embed_plan(d, tok, workspace, ws_bytes, ws_flags, side_stream)) return rc;
  if (cudaEventRecord(ej, ss) != cudaSuccess) return check_launch();
  return MOT_OK;
}

extern "C" int mot_stream_wait_event(void* stream, void* event) {
  if (!event) return MOT_ERR_BAD_ARG;
  if (cudaStreamWaitEvent(reinterpret_cast<cudaStream_t>(stream), reinterpret_cast<cudaEvent_t>(event), 0) != cudaSuccess)
    return check_launch();
  return MOT_OK;
}

// Would mot_embed_bwd_ex run the saved-output kernel for this descriptor?  (variant, width with an instantiation,
// and few enough positions per vocabulary row, see below)
static bool saved_path_applies(const MotDesc* d, const EmbedParams& p) {
  static const bool no_saved = getenv("MOT_NO_SAVED_BWD") != nullptr;  // debug knob (A/B timing)
  if (no_saved || concat_splits(d) || pick_mode(p, kBwdCW) != 1 || p.io_ld != p.Do || p.io_col != 0) return false;
  const int cpl = p.Do / (32 * kBwdCW);
  if (!(cpl == 4 || cpl == 6 || cpl == 8 || (d->dtype == MOT_F32 && cpl == 2))) return false;
  // Beyond ~4 positions per vocabulary row the recompute kernel wins: its token rows are re-read from L2 (the
  // sorted stream visits a row's occurrences back to back) while the saved rows are all distinct HBM reads
  // (768 = 16 x 48 bf16, V = 50257: 131K tokens 118 vs 132 us, 262K 225 vs 218 us, 1M 921 vs 795 us; profiles/r1_experiments.md).
  return p.N <= 4LL * p.V;
}

extern "C" int mot_embed_bwd_uses_saved(const MotDesc* d) {
  if (validate(d) != MOT_OK) return 0;
  EmbedParams p;
  fill_params(d, p);
  return saved_path_applies(d, p) ? 1 : 0;
}

extern "C" int mot_embed_bwd(const MotDesc* d, const int32_t* tok, const void* byte_ids, const void* ttb,
                             const void* E_tok, const void* E_byte, const float* lam, const void* grad_out,
                             void* gE_tok, void* gE_byte, float* g_lam, void* workspace, size_t ws_bytes,
                             int32_t ws_flags, void* stream) {
  return mot_embed_bwd_ex(d, tok, byte_ids, ttb, E_tok, E_byte, lam, nullptr, grad_out, nullptr, nullptr, gE_tok, gE_byte,
                          g_lam, nullptr, workspace, ws_bytes, ws_flags, stream);
}

static int embed_bwd_impl(const MotDesc* d, const int32_t* tok, const void* byte_ids, const void* ttb,
                          const void* E_tok, const void* E_byte, const float* lam, const void* addend,
                          const void* grad_out, const void* out_saved, const float* rstd_saved, void* gE_tok,
                          void* gE_byte, float* g_lam, void* d_addend, void* workspace, size_t ws_bytes,
                          int32_t ws_flags, int slab, int n_slabs, int reserve_sms, void* stream) {
  const bool plan_ready = (ws_flags & MOT_WS_PLAN_READY) != 0, ws_clean = (ws_flags & MOT_WS_CLEAN) != 0;
  if (int rc = validate(d)) return rc;
  const bool slabbed = n_slabs > 1;
  if (n_slabs < 1 || slab < 0 || slab >= n_slabs || reserve_sms < 0 || reserve_sms > kDpReserveMax) return MOT_ERR_BAD_ARG;
  if (slabbed && (d->dp_slabs != n_slabs || (slab > 0 && !plan_ready))) return MOT_ERR_BAD_ARG;
  if (slabbed && d->n_tokens == 0) return MOT_ERR_UNSUPPORTED;
  const bool has_tok = d->combine != MOT_BYTES_ONLY, has_bytes = d->combine != MOT_TOK_ONLY;
  if (has_tok && !gE_tok) return MOT_ERR_BAD_ARG;
  if (has_bytes && !gE_byte) return MOT_ERR_BAD_ARG;
  if ((addend || d_addend) && (concat_splits(d) || d->row_stride != 0 || d->col_offset != 0)) return MOT_ERR_UNSUPPORTED;
  if (d_addend && (d->flags & MOT_F_OUT_NORM) && !addend) return MOT_ERR_BAD_ARG;  // d z needs z: the addend itself
  if (!aligned16(addend) || !aligned16(d_addend)) return MOT_ERR_MISALIGNED;
  if (!aligned16(gE_tok) || !aligned16(gE_byte)) return MOT_ERR_MISALIGNED;
  if (d->n_tokens == 0) {  // nothing gathered: dense zero grads
    cudaStream_t s0 = reinterpret_cast<cudaStream_t>(stream);
    const size_t esz0 = d->dtype == MOT_BF16 ? 2 : 4;
    if (has_tok && cudaMemsetAsync(gE_tok, 0, (size_t)d->tok_vocab * d->tok_dim * esz0, s0) != cudaSuccess) return check_launch();
    if (has_bytes && cudaMemsetAsync(gE_byte, 0, (size_t)d->byte_vocab * d->byte_dim * esz0, s0) != cudaSuccess) return check_launch();
    if (g_lam && cudaMemsetAsync(g_lam, 0, 8, s0) != cudaSuccess) return check_launch();
    return MOT_OK;
  }
  if (!grad_out || !workspace) return MOT_ERR_BAD_ARG;
  if (has_tok && (!tok || !E_tok)) return MOT_ERR_BAD_ARG;
  if (has_bytes && !E_byte) return MOT_ERR_BAD_ARG;
  if (has_bytes) {
    if (d->flags & MOT_F_IDS_FROM_TTB) { if (!ttb || !tok) return MOT_ERR_BAD_ARG; }
    else if (!byte_ids) return MOT_ERR_BAD_ARG;
  }
  if ((d->flags & MOT_F_HAS_LAMBDAS) && (!lam || !g_lam)) return MOT_ERR_BAD_ARG;
  if (!aligned16(grad_out) || !aligned16(E_tok) || !aligned16(E_byte) || !aligned16(gE_tok) || !aligned16(gE_byte) ||
      !aligned16(workspace))
    return MOT_ERR_MISALIGNED;
  EmbedParams p;
  fill_params(d, p);
  const WsLayout w = ws_layout(p, d->dp_slabs);
  if (ws_bytes < w.total) return MOT_ERR_WORKSPACE;
  bind_ws(p, w, workspace);
  p.tok = tok; p.ids = byte_ids; p.ttb = ttb; p.E_tok = E_tok; p.E_byte = E_byte; p.lam = lam;
  p.gout = grad_out; p.gE_tok = gE_tok; p.gE_byte = gE_byte; p.g_lam = g_lam;
  p.addend = addend; p.d_addend = d_addend;
  p.plan_early = (plan_ready && (ws_flags & MOT_WS_PLAN_JOINED)) ? 1 : 0;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (slabbed) {
    // rows [V k / n, V (k+1) / n) of the dense token gradient; the byte table and the lambdas finish with the last slab
    p.v_lo = (int)((long long)p.V * slab / n_slabs);
    p.v_hi = (int)((long long)p.V * (slab + 1) / n_slabs);
    p.last_slab = slab == n_slabs - 1;
    p.grid_cap = 148 - reserve_sms;
  }
  if (!plan_ready) {
    if (!ws_clean && cudaMemsetAsync(workspace, 0, w.zero_end, s) != cudaSuccess) return check_launch();
    if (int rc = run_plan(p, s)) return rc;
  } else if (!ws_clean) {  // plan kept from mot_embed_plan(): only the accumulators need clearing
    if (cudaMemsetAsync(reinterpret_cast<char*>(workspace) + w.byte_acc, 0, w.zero_end - w.byte_acc, s) != cudaSuccess)
      return check_launch();
  }
  int rc = MOT_OK;
  if (slabbed && concat_splits(d)) return MOT_ERR_UNSUPPORTED;
  if (concat_splits(d)) {
    EmbedParams pt, pb;
    split_params(d, pt, pb);
    for (EmbedParams* q : {&pt, &pb}) {
      bind_ws(*q, w, workspace);
      q->tok = tok; q->ids = byte_ids; q->ttb = ttb; q->E_tok = E_tok; q->E_byte = E_byte; q->lam = lam;
      q->gout = grad_out; q->gE_tok = gE_tok; q->gE_byte = gE_byte; q->g_lam = g_lam;
      q->R = p.R;  // one stream chunking for both halves and the finalize pass
      if ((rc = d->dtype == MOT_BF16 ? dispatch_bwd_bf16(*q, s) : dispatch_bwd_f32(*q, s))) return rc;
    }
  } else {
    // the MoT-sum variant with the forward result kept: the saved-output kernel (mot_embed_bwd_sum.cuh); every other
    // case recomputes the mixed row
    rc = -1;
    if (out_saved && rstd_saved && !addend && !d_addend && saved_path_applies(d, p)) {
      if (!aligned16(out_saved)) return MOT_ERR_MISALIGNED;
      p.out_saved = out_saved;
      p.rstd = rstd_saved;
      const int r_default = p.R;
      // the finalize pass below reads the same p.R
      p.R = slabbed ? stream_chunk_slab(p.N, n_slabs, kSumThreads / 32) : stream_chunk(p.N, kSumThreads / 32);
      rc = d->dtype == MOT_BF16 ? dispatch_bwd_sum_bf16(p, s) : dispatch_bwd_sum_f32(p, s);
      if (rc < 0) p.R = r_default;
    }
    if (slabbed && rc < 0) return MOT_ERR_UNSUPPORTED;  // only the saved-output kernel walks a vocabulary slab
    if (rc < 0 && (addend || d_addend)) rc = d->dtype == MOT_BF16 ? dispatch_bwd_addend_bf16(p, s) : dispatch_bwd_addend_f32(p, s);
    if (rc < 0) rc = d->dtype == MOT_BF16 ? dispatch_bwd_bf16(p, s) : dispatch_bwd_f32(p, s);
  }
  if (rc) return rc;
  int sms = 0, optin = 0;
  device_props(&sms, &optin);
  {  // one warp per task (chunk boundary or byte row), 8 warps per CTA
    const long long tasks = (has_tok ? (p.N + p.R - 1) / p.R : 0) + p.Vb;
    long long fb = (tasks + 7) / 8;
    if (fb > 8LL * sms) fb = 8LL * sms;
    if (fb < 1) fb = 1;
    p.trace = g_trace ? g_trace + 2 * 4096 * 64 : nullptr;
    rc = d->dtype == MOT_BF16 ? launch_finalize_bf16(p, (int)fb, s) : launch_finalize_f32(p, (int)fb, s);
  }
  if (rc) return rc;
  if ((d->flags & MOT_F_HAS_LAMBDAS) && g_lam && p.last_slab) {
    launch_pdl(mot_lam_store_kernel, dim3(1), dim3(32), 0, s, p.lam_acc, g_lam);
    count_launch();
  }
  return check_launch();
}

extern "C" int mot_embed_bwd_ex(const MotDesc* d, const int32_t* tok, const void* byte_ids, const void* ttb,
                                const void* E_tok, const void* E_byte, const float* lam, const void* addend,
                                const void* grad_out, const void* out_saved, const float* rstd_saved, void* gE_tok,
                                void* gE_byte, float* g_lam, void* d_addend, void* workspace, size_t ws_bytes,
                                int32_t ws_flags, void* stream) {
  return embed_bwd_impl(d, tok, byte_ids, ttb, E_tok, E_byte, lam, addend, grad_out, out_saved, rstd_saved, gE_tok, gE_byte,
                        g_lam, d_addend, workspace, ws_bytes, ws_flags, 0, 1, 0, stream);
}

extern "C" int mot_embed_bwd_slab(const MotDesc* d, const int32_t* tok, const void* byte_ids, const void* ttb,
                                  const void* E_tok, const void* E_byte, const float* lam, const void* grad_out,
                                  const void* out_saved, const float* rstd_saved, void* gE_tok, void* gE_byte, float* g_lam,
                                  void* workspace, size_t ws_bytes, int32_t ws_flags, int32_t slab, int32_t n_slabs,
                                  int32_t reserve_sms, void* stream) {
  return embed_bwd_impl(d, tok, byte_ids, ttb, E_tok, E_byte, lam, nullptr, grad_out, out_saved, rstd_saved, gE_tok, gE_byte,
                        g_lam, nullptr, workspace, ws_bytes, ws_flags, slab, n_slabs, reserve_sms, stream);
}

extern "C" int mot_embed_slab_rows(int32_t tok_vocab, int32_t slab, int32_t n_slabs, int32_t* row_lo, int32_t* row_hi) {
  if (tok_vocab <= 0 || n_slabs < 1 || slab < 0 || slab >= n_slabs || !row_lo || !row_hi) return MOT_ERR_BAD_ARG;
  *row_lo = (int32_t)((long long)tok_vocab * slab / n_slabs);
  *row_hi = (int32_t)((long long)tok_vocab * (slab + 1) / n_slabs);
  return MOT_OK;
}

extern "C" int mot_embed_touched_rows(const MotDesc* d, const void* workspace, size_t ws_bytes, uint32_t* bitmap, void* stream) {
  if (int rc = validate(d)) return rc;
  if (d->combine == MOT_BYTES_ONLY) return MOT_ERR_UNSUPPORTED;
  if (!workspace || !bitmap) return MOT_ERR_BAD_ARG;
  EmbedParams p;
  fill_params(d, p);
  const WsLayout w = ws_layout(p, d->dp_slabs);
  if (ws_bytes < w.total) return MOT_ERR_WORKSPACE;
  bind_ws(p, w, const_cast<void*>(workspace));
  const int words = (p.V + 31) / 32;
  launch_pdl(plan_rowmap_kernel, dim3((unsigned)((words + 7) / 8)), dim3(256), 0, reinterpret_cast<cudaStream_t>(stream),
             (const int*)p.off, (int)p.V, bitmap);
  count_launch();
  return check_launch();
}
