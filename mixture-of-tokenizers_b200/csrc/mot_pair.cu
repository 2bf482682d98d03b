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
// their parameter block (and with it their register counts).
struct PairTtbParams : PairParams {
  PullSrc ttb;
};
template <int PULL>
using PairArgs = std::conditional_t<PULL == kNoPull, PairParams, PairTtbParams>;

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
template <int PULL>
__device__ __forceinline__ void pair_ttb_ids(const PairTtbParams& p, long long pos, int slot, bool active, int& ia, int& ib) {
  const int lane = lane_id();
  const int tv = clampi(ld_g(p.ttb.tok + pos), p.ttb.V - 1);
  const int a = lane < p.bpt ? ttb_raw(p.ttb.ttb, p.ttb.ttb_dtype, tv, p.bpt, lane) : 0;
  const int b = pulled_row_warp<PULL == kPullRight>(p.ttb, (int)pos);
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

// MAXJ = 8-element chunks per lane (ceil(bd / 8 / G)); PULL: kNoPull loads the ids, kPullLeft / kPullRight derive them
template <typename T, int G, int MAXJ, int PULL>
__global__ void __launch_bounds__(kPairThreads, MAXJ <= 4 ? 2 : 1) mot_pair_fwd_kernel(const PairArgs<PULL> p) {
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
    if constexpr (PULL != kNoPull) {
      pair_ttb_ids<PULL>(p, pos, slot, active, ia, ib);
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
template <typename T, int G, int MAXJ, int PULL>
__global__ void __launch_bounds__(kPairThreads, MAXJ <= 4 ? 2 : 1) mot_pair_bwd_kernel(const PairArgs<PULL> p) {
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
    if constexpr (PULL != kNoPull) {
      pair_ttb_ids<PULL>(p, pos, slot, active, ia, ib);
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

template <typename T, int G, int MAXJ, int PULL>
static int launch_pair(const PairTtbParams& p, bool backward, cudaStream_t s) {
  int sms = 0, optin = 0;
  if (int rc = device_props(&sms, &optin)) return rc;
  const size_t smem = align_up((size_t)p.Vb * p.bd * sizeof(T), 128);
  if (smem + 1024 > (size_t)optin) return MOT_ERR_UNSUPPORTED;  // table does not fit in shared memory
  long long blocks = (p.N + kPairThreads / 32 - 1) / (kPairThreads / 32);
  const int per_sm = (MAXJ <= 4 && 2 * (smem + 1024) <= (size_t)optin) ? 2 : 1;  // two CTAs per SM while two tables fit
  if (blocks > (long long)per_sm * sms) blocks = (long long)per_sm * sms;
  if (blocks < 1) blocks = 1;
  if (backward) {
    auto kern = mot_pair_bwd_kernel<T, G, MAXJ, PULL>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return check_launch();
    launch_pdl(kern, dim3((unsigned)blocks), dim3(kPairThreads), smem, s, p);
  } else {
    auto kern = mot_pair_fwd_kernel<T, G, MAXJ, PULL>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return check_launch();
    launch_pdl(kern, dim3((unsigned)blocks), dim3(kPairThreads), smem, s, p);
  }
  count_launch();
  return check_launch();
}

template <typename T, int PULL>
static int dispatch_pair(const PairTtbParams& p, bool backward, cudaStream_t s) {
  const int per_lane = (p.bd / kChunk + p.G - 1) / p.G;  // 8-element chunks per lane
  const int mj = per_lane <= 4 ? 4 : 8;
  if (per_lane > 8) return MOT_ERR_UNSUPPORTED;
#define MOT_PAIR_CASE(GG)                                                     \
  case GG:                                                                    \
    return mj == 4 ? launch_pair<T, GG, 4, PULL>(p, backward, s) : launch_pair<T, GG, 8, PULL>(p, backward, s);
  switch (p.G) {
    MOT_PAIR_CASE(1)
    MOT_PAIR_CASE(2)
    MOT_PAIR_CASE(4)
    MOT_PAIR_CASE(8)
  }
#undef MOT_PAIR_CASE
  return MOT_ERR_UNSUPPORTED;
}

// The instantiation of the descriptor's dtype and id source.
static int run_pair(const MotDesc* d, const PairTtbParams& p, bool backward, cudaStream_t s) {
  const bool bf16 = d->dtype == MOT_BF16;
  if (d->flags & MOT_F_TTB_PULL_LEFT)
    return bf16 ? dispatch_pair<__nv_bfloat16, kPullLeft>(p, backward, s) : dispatch_pair<float, kPullLeft>(p, backward, s);
  if (d->flags & MOT_F_TTB_PULL_RIGHT)
    return bf16 ? dispatch_pair<__nv_bfloat16, kPullRight>(p, backward, s) : dispatch_pair<float, kPullRight>(p, backward, s);
  return bf16 ? dispatch_pair<__nv_bfloat16, kNoPull>(p, backward, s) : dispatch_pair<float, kNoPull>(p, backward, s);
}

int validate_desc(const MotDesc* d);  // mot_embed.cu: the rules every descriptor obeys

// A pair descriptor (mot_b200.h): bytes-only with the per-byte norm; explicit ids (MOT_F_IDS_I64 gives their width), or
// ids derived from the ttb table with exactly one pull, the right one optionally with its lookahead.
static int pair_check(const MotDesc* d) {
  constexpr int32_t kPull = MOT_F_TTB_PULL_LEFT | MOT_F_TTB_PULL_RIGHT;
  if (d->combine != MOT_BYTES_ONLY || !(d->flags & MOT_F_BYTE_NORM)) return MOT_ERR_BAD_ARG;
  const int32_t ids = d->flags & ~MOT_F_BYTE_NORM;
  const bool ok = (ids & MOT_F_IDS_FROM_TTB) ? (ids & kPull) && !(ids & ~(MOT_F_IDS_FROM_TTB | kPull | MOT_F_TTB_NEXT_TOK))
                                             : !(ids & ~MOT_F_IDS_I64);
  return ok ? MOT_OK : MOT_ERR_BAD_ARG;
}

// Everything both entry points check before they touch the device; `rows` is out (forward) or grad_out (backward).
static int pair_args(const MotDesc* d, const int32_t* tok, const void* ids_a, const void* ids_b, const void* ttb,
                     const void* E_byte, const void* rows) {
  if (int rc = validate_desc(d)) return rc;
  if (int rc = pair_check(d)) return rc;
  if (d->n_tokens == 0) return MOT_OK;
  const bool derived = (d->flags & MOT_F_IDS_FROM_TTB) != 0;
  if ((derived ? !tok || !ttb : !ids_a || !ids_b) || !E_byte || !rows) return MOT_ERR_BAD_ARG;
  if ((reinterpret_cast<uintptr_t>(E_byte) | reinterpret_cast<uintptr_t>(rows)) & 15u) return MOT_ERR_MISALIGNED;
  return MOT_OK;
}

static PairTtbParams pair_params(const MotDesc* d, const int32_t* tok, const void* ids_a, const void* ids_b,
                                 const void* ttb, const void* E_byte) {
  PairTtbParams p{};
  p.ids_a = ids_a; p.ids_b = ids_b; p.E_byte = E_byte;
  p.N = d->n_tokens; p.ld = d->row_stride ? d->row_stride : d->out_dim; p.col = d->col_offset;
  p.Vb = d->byte_vocab; p.bpt = d->bpt; p.bd = d->byte_dim; p.ids_i64 = (d->flags & MOT_F_IDS_I64) != 0;
  p.n_rep = kByteRep; p.eps = d->eps;
  int G = 1;
  while (G * 2 * p.bpt <= 32 && G * 2 <= p.bd / kChunk) G *= 2;  // lanes per slot: power of two, at most one lane per chunk
  p.G = G;
  if (d->flags & MOT_F_IDS_FROM_TTB)
    p.ttb = PullSrc{tok, ttb, d->seq_len, d->tok_vocab, d->bpt, d->ttb_dtype, d->pad_id, d->eot_id, 0,
                    (d->flags & MOT_F_TTB_NEXT_TOK) ? tok + d->n_tokens : nullptr};
  return p;
}

}  // namespace mot

using namespace mot;

extern "C" int mot_byte_pair_fwd(const MotDesc* d, const int32_t* tok, const void* ids_a, const void* ids_b, const void* ttb,
                                 const void* E_byte, void* out, void* stream) {
  if (int rc = pair_args(d, tok, ids_a, ids_b, ttb, E_byte, out)) return rc;
  if (d->n_tokens == 0) return MOT_OK;
  PairTtbParams p = pair_params(d, tok, ids_a, ids_b, ttb, E_byte);
  p.out = out;
  return run_pair(d, p, false, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" size_t mot_byte_pair_workspace_bytes(int32_t byte_vocab, int32_t byte_dim) {
  if (byte_vocab <= 0 || byte_dim <= 0) return 0;
  return align_up((size_t)kByteRep * byte_vocab * byte_dim * 4, 256);
}

extern "C" int mot_byte_pair_bwd(const MotDesc* d, const int32_t* tok, const void* ids_a, const void* ids_b, const void* ttb,
                                 const void* E_byte, const void* grad_out, void* gE_byte, void* workspace, size_t ws_bytes,
                                 void* stream) {
  if (int rc = pair_args(d, tok, ids_a, ids_b, ttb, E_byte, grad_out)) return rc;
  if (!gE_byte) return MOT_ERR_BAD_ARG;
  if (reinterpret_cast<uintptr_t>(gE_byte) & 15u) return MOT_ERR_MISALIGNED;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const size_t esz = d->dtype == MOT_BF16 ? 2 : 4;
  if (d->n_tokens == 0) {  // nothing gathered: dense zero gradient
    if (cudaMemsetAsync(gE_byte, 0, (size_t)d->byte_vocab * d->byte_dim * esz, s) != cudaSuccess) return check_launch();
    return MOT_OK;
  }
  const size_t need = mot_byte_pair_workspace_bytes(d->byte_vocab, d->byte_dim);
  if (!workspace || ws_bytes < need) return MOT_ERR_WORKSPACE;
  if (reinterpret_cast<uintptr_t>(workspace) & 15u) return MOT_ERR_MISALIGNED;
  if (cudaMemsetAsync(workspace, 0, need, s) != cudaSuccess) return check_launch();
  PairTtbParams p = pair_params(d, tok, ids_a, ids_b, ttb, E_byte);
  p.gout = grad_out;
  p.acc = reinterpret_cast<float*>(workspace);
  if (int rc = run_pair(d, p, true, s)) return rc;
  // sum the replicas and cast (the norm backward already happened per occurrence: no MOT_F_BYTE_NORM here)
  EmbedParams q{};
  q.combine = MOT_BYTES_ONLY;
  q.N = p.N; q.R = 32; q.Vb = p.Vb; q.bd = p.bd; q.bpt = p.bpt; q.Do = p.bpt * p.bd;
  q.n_rep = kByteRep; q.byte_acc = p.acc; q.E_byte = p.E_byte; q.gE_byte = gE_byte; q.eps = p.eps;
  q.last_slab = 1;  // the byte rows are this launch's only work
  const int fb = (p.Vb + 7) / 8;
  return d->dtype == MOT_BF16 ? launch_finalize_bf16(q, fb, s) : launch_finalize_f32(q, fb, s);
}
