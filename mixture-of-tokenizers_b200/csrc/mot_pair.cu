// Byte half of scaled-pre-train's `--add-padded-and-pulled` embedding (spt/train_gpt.py:371-379, flag :949-951):
//     byte_embs = norm(embed_bytes(byte_tensor) + embed_bytes(byte_tensor_pulled))        (norm over byte_dim, per byte)
// i.e. two gathers per (position, slot) summed BEFORE the rms-norm, so the scale depends on the id PAIR and cannot be
// precomputed per table row the way the single-gather kernels do.  Rows are written as the byte columns of the
// [tok | bytes] projection operand (spt/train_gpt.py:442-443) -- token-major ids, strided output rows.
//
// Layout / execution: E_byte (<= 117 KB) is staged once per CTA in shared memory with bulk async copies; persistent
// CTAs, a warp owns one position at a time; a slot's byte_dim elements belong to a group of G adjacent lanes
// (G = largest power of two <= 32 / bpt), lane h of the group owning the 8-element chunks h, h+G, ...; the per-slot
// sums of squares / dot products are G-lane butterfly reductions; adjacent lanes touch adjacent 16-byte chunks, so
// every 32-byte sector of the output row is written whole.  HBM-bound: per position 2*bpt ids + bpt*bd*e output bytes
// (forward) / the same read of the upstream gradient plus 2*bpt*bd fp32 REDs into L2-resident replicas (backward).
#include <type_traits>

#include "mot_embed_kernels.cuh"

namespace mot {

struct PairParams {
  const void* ids_a;
  const void* ids_b;
  const void* E_byte;
  void* out;         // forward: [N, ld] rows, this kernel writes columns [col, col + bpt*bd)
  const void* gout;  // backward: same geometry
  float* acc;        // backward: [n_rep][Vb*bd] fp32, zero on entry
  long long N, ld;
  int col, Vb, bpt, bd, ids_i64, n_rep, G;
  float eps;
};
// Both id sets derived from the token ids (a padded, b pulled).  A separate type, so that the kernels of explicit ids keep
// their parameter block.
struct PairTtbParams : PairParams {
  PullSrc ttb;
};
// The same with the pulled ids of pull_from_right (MOT_F_TTB_PULL_RIGHT): its own kernel instantiations.
struct PairTtbRightParams : PairTtbParams {};
template <typename P>
constexpr bool kPairTtb = std::is_base_of_v<PairTtbParams, P>;

constexpr int kPairThreads = 512;

template <typename T>
__device__ __forceinline__ void pair_stage_table(const PairParams& p, T* tab, uint64_t* bar) {
  const uint32_t bytes = (uint32_t)p.Vb * p.bd * sizeof(T);
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    fence_mbar_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    mbar_expect_tx(bar, bytes);
    for (uint32_t done = 0; done < bytes;) {
      const uint32_t n = min(bytes - done, 32768u);
      bulk_g2s(reinterpret_cast<char*>(tab) + done, reinterpret_cast<const char*>(p.E_byte) + done, n, bar);
      done += n;
    }
  }
  mbar_wait(bar, 0);
}

__device__ __forceinline__ int pair_load_id(const void* ids, int i64, long long idx, int hi) {
  const int v = i64 ? (int)ld_g(reinterpret_cast<const long long*>(ids) + idx) : ld_g(reinterpret_cast<const int*>(ids) + idx);
  return clampi(v, hi);
}

// Byte ids (ia, ib) of this lane's slot at position pos derived from the token ids: padded ids for a, pulled ids for b.
// Warp collective; clamped; 0 on inactive lanes.
template <typename P>
__device__ __forceinline__ void pair_ttb_ids(const P& p, long long pos, int slot, bool active, int& ia, int& ib) {
  const int lane = lane_id();
  const int tv = clampi(ld_g(p.ttb.tok + pos), p.ttb.V - 1);
  const int a = lane < p.bpt ? ttb_raw(p.ttb.ttb, p.ttb.ttb_dtype, tv, p.bpt, lane) : 0;
  const int b = pulled_row_warp<std::is_same_v<P, PairTtbRightParams>>(p.ttb, (int)pos);
  ia = clampi(__shfl_sync(0xffffffffu, a, slot & 31), p.Vb - 1);
  ib = clampi(__shfl_sync(0xffffffffu, b, slot & 31), p.Vb - 1);
  if (!active) ia = ib = 0;
}

template <int G>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = G >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// MAXJ = 8-element chunks per lane (ceil(bd / 8 / G))
template <typename T, int G, int MAXJ, typename P>
__global__ void __launch_bounds__(kPairThreads, MAXJ <= 4 ? 2 : 1) mot_pair_fwd_kernel(const P p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ uint64_t tab_bar;
  T* tab = reinterpret_cast<T*>(smem_raw);
  pdl_launch_dependents();
  pdl_wait();
  pair_stage_table<T>(p, tab, &tab_bar);
  const int lane = lane_id(), warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int slot = lane / G, h = lane % G;
  const bool active = slot < p.bpt;
  const int nch = p.bd / kChunk;
  const float inv_bd = 1.f / (float)p.bd;
  T* out = reinterpret_cast<T*>(p.out);
  const long long W = (long long)gridDim.x * nw;
  for (long long pos = (long long)warp * gridDim.x + blockIdx.x; pos < p.N; pos += W) {
    int ia = 0, ib = 0;
    if constexpr (kPairTtb<P>) {
      pair_ttb_ids(p, pos, slot, active, ia, ib);
    } else if (active) {
      ia = pair_load_id(p.ids_a, p.ids_i64, pos * p.bpt + slot, p.Vb - 1);
      ib = pair_load_id(p.ids_b, p.ids_i64, pos * p.bpt + slot, p.Vb - 1);
    }
    float a[MAXJ][8];
    float ss = 0.f;
#pragma unroll
    for (int j = 0; j < MAXJ; ++j) {
      const int c = j * G + h;
      if (active && c < nch) {
        float b[8];
        Vec8<T>::unpack(Vec8<T>::lds_raw(tab + (size_t)ia * p.bd + c * kChunk), a[j]);
        Vec8<T>::unpack(Vec8<T>::lds_raw(tab + (size_t)ib * p.bd + c * kChunk), b);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          a[j][e] += b[e];
          ss += a[j][e] * a[j][e];
        }
      }
    }
    ss = group_sum<G>(ss);
    const float r = rsqrtf(ss * inv_bd + p.eps);
    T* orow = out + (size_t)pos * p.ld + p.col + (size_t)slot * p.bd;
#pragma unroll
    for (int j = 0; j < MAXJ; ++j) {
      const int c = j * G + h;
      if (active && c < nch) {
#pragma unroll
        for (int e = 0; e < 8; ++e) a[j][e] *= r;
        Vec8<T>::stg(orow + c * kChunk, a[j]);
      }
    }
  }
}

// Backward: with s = E[ia] + E[ib], r = rsqrt(mean(s^2) + eps): ds = r*g - s * r^3 * mean(g.s); both gathered rows
// receive ds (fp32 RED.v4 into one of n_rep L2-resident replicas; mot_bwd_finalize_kernel sums and casts them).
// Two passes over the slot (reduce, then scatter) so that nothing of the row is held across the reduction.
template <typename T, int G, int MAXJ, typename P>
__global__ void __launch_bounds__(kPairThreads, MAXJ <= 4 ? 2 : 1) mot_pair_bwd_kernel(const P p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ uint64_t tab_bar;
  T* tab = reinterpret_cast<T*>(smem_raw);
  pdl_launch_dependents();
  pdl_wait();
  pair_stage_table<T>(p, tab, &tab_bar);
  const int lane = lane_id(), warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int slot = lane / G, h = lane % G;
  const bool active = slot < p.bpt;
  const int nch = p.bd / kChunk;
  const float inv_bd = 1.f / (float)p.bd;
  const T* gout = reinterpret_cast<const T*>(p.gout);
  const int gw = warp * gridDim.x + blockIdx.x;
  float* acc = p.acc + (size_t)(gw % p.n_rep) * p.Vb * p.bd;
  const long long W = (long long)gridDim.x * nw;
  for (long long pos = gw; pos < p.N; pos += W) {
    int ia = 0, ib = 0;
    if constexpr (kPairTtb<P>) {
      pair_ttb_ids(p, pos, slot, active, ia, ib);
    } else if (active) {
      ia = pair_load_id(p.ids_a, p.ids_i64, pos * p.bpt + slot, p.Vb - 1);
      ib = pair_load_id(p.ids_b, p.ids_i64, pos * p.bpt + slot, p.Vb - 1);
    }
    const T* grow = gout + (size_t)pos * p.ld + p.col + (size_t)slot * p.bd;
    float ss = 0.f, dot = 0.f;
#pragma unroll
    for (int j = 0; j < MAXJ; ++j) {
      const int c = j * G + h;
      if (active && c < nch) {
        float a[8], b[8], g[8];
        Vec8<T>::unpack(Vec8<T>::lds_raw(tab + (size_t)ia * p.bd + c * kChunk), a);
        Vec8<T>::unpack(Vec8<T>::lds_raw(tab + (size_t)ib * p.bd + c * kChunk), b);
        Vec8<T>::unpack(Vec8<T>::ldg_raw(grow + c * kChunk), g);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          a[e] += b[e];
          ss += a[e] * a[e];
          dot += g[e] * a[e];
        }
      }
    }
    ss = group_sum<G>(ss);
    dot = group_sum<G>(dot);
    const float r = rsqrtf(ss * inv_bd + p.eps);
    const float coef = r * r * r * dot * inv_bd;
#pragma unroll
    for (int j = 0; j < MAXJ; ++j) {
      const int c = j * G + h;
      if (active && c < nch) {
        float a[8], b[8], g[8];
        Vec8<T>::unpack(Vec8<T>::lds_raw(tab + (size_t)ia * p.bd + c * kChunk), a);
        Vec8<T>::unpack(Vec8<T>::lds_raw(tab + (size_t)ib * p.bd + c * kChunk), b);
        Vec8<T>::unpack(Vec8<T>::ldg_raw(grow + c * kChunk), g);   // second read of the 16/32 bytes: L2 hit
        float lo[4], hi4[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          lo[e] = r * g[e] - coef * (a[e] + b[e]);
          hi4[e] = r * g[e + 4] - coef * (a[e + 4] + b[e + 4]);
        }
        float* da = acc + (size_t)ia * p.bd + c * kChunk;
        float* db = acc + (size_t)ib * p.bd + c * kChunk;
        gmem_add4(da, lo);
        gmem_add4(da + 4, hi4);
        gmem_add4(db, lo);
        gmem_add4(db + 4, hi4);
      }
    }
  }
}

template <typename T, int G, int MAXJ, typename P>
static int launch_pair(const P& p, bool backward, cudaStream_t s) {
  int sms = 0, optin = 0;
  if (int rc = device_props(&sms, &optin)) return rc;
  const size_t smem = align_up((size_t)p.Vb * p.bd * sizeof(T), 128);
  if (smem + 1024 > (size_t)optin) return MOT_ERR_UNSUPPORTED;  // table does not fit in shared memory
  long long blocks = (p.N + kPairThreads / 32 - 1) / (kPairThreads / 32);
  const int per_sm = (MAXJ <= 4 && 2 * (smem + 1024) <= (size_t)optin) ? 2 : 1;  // two CTAs per SM while two tables fit
  if (blocks > (long long)per_sm * sms) blocks = (long long)per_sm * sms;
  if (blocks < 1) blocks = 1;
  if (backward) {
    auto kern = mot_pair_bwd_kernel<T, G, MAXJ, P>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return check_launch();
    launch_pdl(kern, dim3((unsigned)blocks), dim3(kPairThreads), smem, s, p);
  } else {
    auto kern = mot_pair_fwd_kernel<T, G, MAXJ, P>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return check_launch();
    launch_pdl(kern, dim3((unsigned)blocks), dim3(kPairThreads), smem, s, p);
  }
  count_launch();
  return check_launch();
}

template <typename T, typename P>
static int dispatch_pair(const P& p, bool backward, cudaStream_t s) {
  const int per_lane = (p.bd / kChunk + p.G - 1) / p.G;  // 8-element chunks per lane
  const int mj = per_lane <= 4 ? 4 : 8;
  if (per_lane > 8) return MOT_ERR_UNSUPPORTED;
#define MOT_PAIR_CASE(GG)                                                     \
  case GG:                                                                    \
    return mj == 4 ? launch_pair<T, GG, 4>(p, backward, s) : launch_pair<T, GG, 8>(p, backward, s);
  switch (p.G) {
    MOT_PAIR_CASE(1)
    MOT_PAIR_CASE(2)
    MOT_PAIR_CASE(4)
    MOT_PAIR_CASE(8)
  }
#undef MOT_PAIR_CASE
  return MOT_ERR_UNSUPPORTED;
}

static int pair_ttb_validate(const int32_t* tok, const void* ttb, int32_t tok_vocab, int32_t ttb_dtype, int64_t seq_len,
                             int64_t n) {
  if (ttb_dtype < MOT_TTB_I16 || ttb_dtype > MOT_TTB_BF16) return MOT_ERR_UNSUPPORTED;
  if (tok_vocab <= 0 || seq_len <= 0 || n % seq_len) return MOT_ERR_BAD_ARG;
  if (n > 0 && (!tok || !ttb)) return MOT_ERR_BAD_ARG;
  return MOT_OK;
}

static int pair_validate(const void* ids_a, const void* ids_b, int64_t n, int32_t bpt, const void* E_byte, int32_t Vb,
                         int32_t bd, int32_t dtype, const void* rows, int64_t row_stride, int32_t col_offset) {
  if (dtype != MOT_BF16 && dtype != MOT_F32) return MOT_ERR_UNSUPPORTED;
  if (n < 0 || n > 0x7fffffffLL || bpt <= 0 || bpt > 32 || Vb <= 0 || bd <= 0) return MOT_ERR_BAD_ARG;
  if (bd % 8 || row_stride % 8 || col_offset % 8) return MOT_ERR_MISALIGNED;
  if (col_offset < 0 || row_stride < (int64_t)col_offset + (int64_t)bpt * bd) return MOT_ERR_BAD_ARG;
  if (n == 0) return MOT_OK;
  if (!ids_a || !ids_b || !E_byte || !rows) return MOT_ERR_BAD_ARG;
  if ((reinterpret_cast<uintptr_t>(E_byte) | reinterpret_cast<uintptr_t>(rows)) & 15u) return MOT_ERR_MISALIGNED;
  return MOT_OK;
}

static void pair_fill(PairParams& p, const void* ids_a, const void* ids_b, int32_t ids_i64, int64_t n, int32_t bpt,
                      const void* E_byte, int32_t Vb, int32_t bd, float eps, int64_t row_stride, int32_t col_offset) {
  p = PairParams{};
  p.ids_a = ids_a; p.ids_b = ids_b; p.E_byte = E_byte;
  p.N = n; p.ld = row_stride; p.col = col_offset;
  p.Vb = Vb; p.bpt = bpt; p.bd = bd; p.ids_i64 = ids_i64 != 0; p.n_rep = kByteRep; p.eps = eps;
  int G = 1;
  while (G * 2 * bpt <= 32 && G * 2 <= bd / kChunk) G *= 2;  // lanes per slot: power of two, at most one lane per chunk
  p.G = G;
}

}  // namespace mot

using namespace mot;

template <typename P>
static int pair_fwd(const P& p, int32_t dtype, void* stream) {
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  return dtype == MOT_BF16 ? dispatch_pair<__nv_bfloat16>(p, false, s) : dispatch_pair<float>(p, false, s);
}

template <typename P>
static int pair_bwd(P& p, int32_t dtype, void* gE_byte, void* workspace, size_t ws_bytes, void* stream) {
  if (!gE_byte) return MOT_ERR_BAD_ARG;
  if (reinterpret_cast<uintptr_t>(gE_byte) & 15u) return MOT_ERR_MISALIGNED;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const size_t esz = dtype == MOT_BF16 ? 2 : 4;
  if (p.N == 0) {  // nothing gathered: dense zero gradient
    if (cudaMemsetAsync(gE_byte, 0, (size_t)p.Vb * p.bd * esz, s) != cudaSuccess) return check_launch();
    return MOT_OK;
  }
  const size_t need = mot_byte_pair_workspace_bytes(p.Vb, p.bd);
  if (!workspace || ws_bytes < need) return MOT_ERR_WORKSPACE;
  if (reinterpret_cast<uintptr_t>(workspace) & 15u) return MOT_ERR_MISALIGNED;
  if (cudaMemsetAsync(workspace, 0, need, s) != cudaSuccess) return check_launch();
  p.acc = reinterpret_cast<float*>(workspace);
  if (int rc = dtype == MOT_BF16 ? dispatch_pair<__nv_bfloat16>(p, true, s) : dispatch_pair<float>(p, true, s)) return rc;
  // sum the replicas and cast (the norm backward already happened per occurrence: no MOT_F_BYTE_NORM here)
  EmbedParams q{};
  q.combine = MOT_BYTES_ONLY;
  q.N = p.N; q.R = 32; q.Vb = p.Vb; q.bd = p.bd; q.bpt = p.bpt; q.Do = p.bpt * p.bd;
  q.n_rep = kByteRep; q.byte_acc = p.acc; q.E_byte = p.E_byte; q.gE_byte = gE_byte; q.eps = p.eps;
  q.last_slab = 1;  // the byte rows are this launch's only work
  const int fb = (p.Vb + 7) / 8;
  return dtype == MOT_BF16 ? launch_finalize_bf16(q, fb, s) : launch_finalize_f32(q, fb, s);
}

// flags: MOT_F_TTB_PULL_LEFT, or MOT_F_TTB_PULL_RIGHT with or without MOT_F_TTB_NEXT_TOK (the tail tok[n + r]).
static PullSrc pair_pull_src(const int32_t* tok, const void* ttb, int32_t tok_vocab, int32_t ttb_dtype, int64_t seq_len,
                             int32_t pad_id, int32_t eot_id, int64_t n, int32_t bpt, int32_t flags) {
  return PullSrc{tok, ttb, seq_len, tok_vocab, bpt, ttb_dtype, pad_id, eot_id, 0,
                 (flags & MOT_F_TTB_NEXT_TOK) ? tok + n : nullptr};
}
static bool pair_pull_flags_ok(int32_t flags) {
  return flags == MOT_F_TTB_PULL_LEFT || flags == MOT_F_TTB_PULL_RIGHT ||
         flags == (MOT_F_TTB_PULL_RIGHT | MOT_F_TTB_NEXT_TOK);
}

extern "C" int mot_byte_pair_fwd(const void* ids_a, const void* ids_b, int32_t ids_i64, int64_t n_tokens, int32_t bpt,
                                 const void* E_byte, int32_t byte_vocab, int32_t byte_dim, int32_t dtype, float eps,
                                 void* out, int64_t row_stride, int32_t col_offset, void* stream) {
  if (int rc = pair_validate(ids_a, ids_b, n_tokens, bpt, E_byte, byte_vocab, byte_dim, dtype, out, row_stride, col_offset)) return rc;
  if (n_tokens == 0) return MOT_OK;
  PairParams p;
  pair_fill(p, ids_a, ids_b, ids_i64, n_tokens, bpt, E_byte, byte_vocab, byte_dim, eps, row_stride, col_offset);
  p.out = out;
  return pair_fwd(p, dtype, stream);
}

extern "C" size_t mot_byte_pair_workspace_bytes(int32_t byte_vocab, int32_t byte_dim) {
  if (byte_vocab <= 0 || byte_dim <= 0) return 0;
  return align_up((size_t)kByteRep * byte_vocab * byte_dim * 4, 256);
}

extern "C" int mot_byte_pair_bwd(const void* ids_a, const void* ids_b, int32_t ids_i64, int64_t n_tokens, int32_t bpt,
                                 const void* E_byte, int32_t byte_vocab, int32_t byte_dim, int32_t dtype, float eps,
                                 const void* grad_out, int64_t row_stride, int32_t col_offset, void* gE_byte,
                                 void* workspace, size_t ws_bytes, void* stream) {
  if (int rc = pair_validate(ids_a, ids_b, n_tokens, bpt, E_byte, byte_vocab, byte_dim, dtype, grad_out, row_stride, col_offset))
    return rc;
  PairParams p;
  pair_fill(p, ids_a, ids_b, ids_i64, n_tokens, bpt, E_byte, byte_vocab, byte_dim, eps, row_stride, col_offset);
  p.gout = grad_out;
  return pair_bwd(p, dtype, gE_byte, workspace, ws_bytes, stream);
}

// The id tensors' null checks of pair_validate do not apply here: a non-null placeholder stands in for them.
extern "C" int mot_byte_pair_ttb_fwd(const int32_t* tok, const void* ttb, int32_t tok_vocab, int32_t ttb_dtype,
                                     int64_t seq_len, int32_t pad_id, int32_t eot_id, int64_t n_tokens, int32_t bpt,
                                     const void* E_byte, int32_t byte_vocab, int32_t byte_dim, int32_t dtype, float eps,
                                     void* out, int64_t row_stride, int32_t col_offset, int32_t flags, void* stream) {
  if (!pair_pull_flags_ok(flags)) return MOT_ERR_BAD_ARG;
  if (int rc = pair_ttb_validate(tok, ttb, tok_vocab, ttb_dtype, seq_len, n_tokens)) return rc;
  if (int rc = pair_validate(tok, tok, n_tokens, bpt, E_byte, byte_vocab, byte_dim, dtype, out, row_stride, col_offset)) return rc;
  if (n_tokens == 0) return MOT_OK;
  const auto run = [&](auto p) {
    pair_fill(p, nullptr, nullptr, 0, n_tokens, bpt, E_byte, byte_vocab, byte_dim, eps, row_stride, col_offset);
    p.ttb = pair_pull_src(tok, ttb, tok_vocab, ttb_dtype, seq_len, pad_id, eot_id, n_tokens, bpt, flags);
    p.out = out;
    return pair_fwd(p, dtype, stream);
  };
  return (flags & MOT_F_TTB_PULL_RIGHT) ? run(PairTtbRightParams{}) : run(PairTtbParams{});
}

extern "C" int mot_byte_pair_ttb_bwd(const int32_t* tok, const void* ttb, int32_t tok_vocab, int32_t ttb_dtype,
                                     int64_t seq_len, int32_t pad_id, int32_t eot_id, int64_t n_tokens, int32_t bpt,
                                     const void* E_byte, int32_t byte_vocab, int32_t byte_dim, int32_t dtype, float eps,
                                     const void* grad_out, int64_t row_stride, int32_t col_offset, void* gE_byte,
                                     void* workspace, size_t ws_bytes, int32_t flags, void* stream) {
  if (!pair_pull_flags_ok(flags)) return MOT_ERR_BAD_ARG;
  if (int rc = pair_ttb_validate(tok, ttb, tok_vocab, ttb_dtype, seq_len, n_tokens)) return rc;
  if (int rc = pair_validate(tok, tok, n_tokens, bpt, E_byte, byte_vocab, byte_dim, dtype, grad_out, row_stride, col_offset))
    return rc;
  const auto run = [&](auto p) {
    pair_fill(p, nullptr, nullptr, 0, n_tokens, bpt, E_byte, byte_vocab, byte_dim, eps, row_stride, col_offset);
    p.ttb = pair_pull_src(tok, ttb, tok_vocab, ttb_dtype, seq_len, pad_id, eot_id, n_tokens, bpt, flags);
    p.gout = grad_out;
    return pair_bwd(p, dtype, gE_byte, workspace, ws_bytes, stream);
  };
  return (flags & MOT_F_TTB_PULL_RIGHT) ? run(PairTtbRightParams{}) : run(PairTtbParams{});
}
