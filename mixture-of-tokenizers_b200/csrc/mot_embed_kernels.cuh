// Fused byte-mix embedding forward / backward for sm_100a.
//
// Replaces (reference, read-only at /root/reference in the build container):
//   forward : runs/71:312-314 + mixin_bytes :228-230 and the other gather/pool/add/norm variants
//             of SURVEY.md 2.4; spt/train_gpt.py:342-379 (+ the cat of :443 as GEMM A operand)
//   backward: the autograd graph of those lines: rms_norm backward, split, and two
//             embedding_dense_backward scatter-adds producing DENSE [V,Dt] / [Vb,bd] grads.
//
// Data layout in HBM: E_tok [V,Dt], E_byte [Vb,bd], out / grad_out [N,Do] row-major, element type T
// (bf16 or fp32); token ids int32 [N]; byte ids int32/int64, token-major [N,bpt] or slot-major [bpt,N];
// ttb table [V,bpt] int16 (or the reference's fp32 / bf16 float containers).
//
// Execution model (both kernels): persistent CTAs, one per SM.  A warp owns one position (forward) or
// one occurrence of the token-sorted stream (backward) at a time; a lane owns chunks of 8 consecutive
// elements (chunk c = it*32 + lane -> every warp-wide access is a contiguous 512 B segment).  The rows
// a warp needs next (token row; grad row + token row) are fetched by ONE lane with 1-D bulk async copies
// (cp.async.bulk, the TMA engine) into a per-warp ring of shared-memory stages guarded by mbarriers, so
// several KB per warp are in flight without holding registers.  The byte table (<= 117 KB) is staged in
// shared memory once per CTA the same way.  HBM streams: token rows, grad rows, output rows, dense grad.
#pragma once
#include <cstdlib>

#include "mot_common.cuh"

namespace mot {

// forward CTA: compiled for up to 1024 threads (<= 64 registers), launched with 24 warps, which leaves a quarter of the
// register file to kernels on other streams (the backward plan runs beside the forward)
constexpr int kFwdThreads = 768;
#ifndef MOT_BWD_THREADS
#define MOT_BWD_THREADS 384
#endif
constexpr int kBwdThreads = MOT_BWD_THREADS;
#ifndef MOT_BYTE_REP
#define MOT_BYTE_REP 16
#endif
constexpr int kByteRep = MOT_BYTE_REP;  // replicas of the fp32 byte-grad accumulator (spreads hot byte ids over L2 atomic units)

struct EmbedParams {
  const int32_t* tok;
  const void* ids;
  const void* ttb;
  const void* E_tok;
  const void* E_byte;
  const float* lam;
  void* out;
  float* rstd_out;  // optional [N]: reciprocal rms of every mixed row (out_norm), kept for the saved-output backward
  // backward
  const void* gout;
  const void* out_saved;  // optional: the forward result and its rstd (mot_embed_bwd_ex)
  const float* rstd;
  const void* addend;     // optional dense [N, Do] rows added to the mixed row before the output norm (runs/71051:228-229)
  void* d_addend;         // backward: receives d(mixed row) [N, Do], the gradient of `addend`
  void* gE_tok;
  void* gE_byte;
  float* g_lam;
  // plan / workspace views
  int* cnt;         // [V]     histogram, doubles as fill cursor
  int* off;         // [V+1]   exclusive scan of cnt
  int* order;       // [N]     positions grouped by token id (the token-sorted stream)
  int* stok;        // [N]     token id of every stream entry
  float* partial;   // [n_stream_chunks, Dt] fp32 slots, zero on entry: sums of the rows that straddle chunk boundaries
  float* byte_acc;  // [n_rep, Vb*bd] fp32, zeroed per call
  float* lam_acc;   // [2]; the int behind them (lam_acc + 2) is the zero-fill work counter of the saved-output backward
  long long N, T;
  long long io_ld;  // row stride (elements) of `out` (forward) / `gout` (backward); Do unless the call is one half of a split concat
  int io_col;       // first column of this kernel's slice inside those rows
  int V, Vb, bpt, Dt, bd, Do, combine, flags, ttb_dtype;
  int n_chunks;  // Do / 8
  int R;         // stream entries per chunk (multiple of 32)
  int n_rep;     // replicas of the byte-grad accumulator (spreads hot byte ids over L2 atomic units)
  int stages;    // ring depth per warp
  int tab_smem;  // 1: byte table staged in shared memory; 0: too large, rows read through L1/L2
  int v_lo, v_hi;  // vocabulary rows [v_lo, v_hi) this launch is responsible for (a slab of the data-parallel pipeline; the
                   // whole table: 0, V)
  int grid_cap;    // > 0: launch at most this many CTAs (SMs left to the exchange kernel that runs beside a slab)
  int last_slab;   // finalize: 1 = also finish the byte table and the lambdas (the last / only slab)
  int plan_early;  // 1: the sort plan was complete before this kernel was launched (event join): its arrays may be read
                   //    before griddepcontrol.wait
  float eps;
  long long* trace;  // MOT_TRACE builds: per-warp time stamps (nullptr: off)
  long long* chk;    // MOT_CHECK builds: violation record
  int n_slots;       // fp32 slots of `partial` (MOT_CHECK builds verify every slot index against it)
  int pad_eot;      // MOT_F_TTB_PULL_LEFT / _RIGHT: pad byte | end-of-text byte << 16 (int16 each; fits the struct's tail padding)
};

struct ChunkMap {
  int toff;  // element offset in the token row, -1: chunk has no token part
  int slot;  // byte slot, -1: no byte part, -2: mean over all slots
  int boff;  // element offset inside the byte row
};

template <int CW>
__device__ __forceinline__ ChunkMap chunk_map(const EmbedParams& p, int c) {
  ChunkMap m{-1, -1, 0};
  if (c * CW >= p.Do) return m;
  const int e = c * CW;
  switch (p.combine) {
    case MOT_ADD:
      m.toff = e;
      m.slot = e / p.bd;
      m.boff = e - m.slot * p.bd;
      break;
    case MOT_CONCAT: {
      const int db = p.bpt * p.bd;
      int eb = -1;
      if (p.flags & MOT_F_BYTES_FIRST) {
        if (e < db) eb = e; else m.toff = e - db;
      } else {
        if (e < p.Dt) m.toff = e; else eb = e - p.Dt;
      }
      if (eb >= 0) {
        m.slot = eb / p.bd;
        m.boff = eb - m.slot * p.bd;
      }
    } break;
    case MOT_TOK_ONLY:
      m.toff = e;
      break;
    case MOT_BYTES_ONLY:
      m.slot = e / p.bd;
      m.boff = e - m.slot * p.bd;
      break;
    case MOT_MEAN:
      m.toff = e;
      m.slot = -2;
      m.boff = e;
      break;
  }
  return m;
}

__device__ __forceinline__ int clampi(int v, int hi) { return min(max(v, 0), hi); }
// row * width as ONE 32 x 32 -> 64 bit multiply (both factors are non-negative and < 2^31: validated on the host)
__device__ __forceinline__ size_t mul_u32(int a, int b) { return (size_t)(unsigned)a * (unsigned)b; }

// RAW byte id of (position, slot); slot < bpt.  The caller clamps it with clamp_id() where it is consumed,
// one iteration later, so the load's latency is not exposed at the load site (the pipeline issues in order).
// Out-of-range ids are clamped (the reference device-asserts).
__device__ __forceinline__ int fetch_id(const EmbedParams& p, long long pos, int slot) {
  int id;
  if (p.flags & MOT_F_IDS_FROM_TTB) {
    long long tokpos = pos;
    int k = slot;
    if (p.flags & MOT_F_TTB_SCRAMBLE) {  // runs/71:479: flat byte i*T + s of the row
      const long long row = pos / p.T, s = pos - row * p.T;
      const long long f = (long long)slot * p.T + s;
      tokpos = row * p.T + f / p.bpt;
      k = (int)(f % p.bpt);
    }
    const int tv = clampi(ld_g(p.tok + tokpos), p.V - 1);
    const size_t e = (size_t)tv * p.bpt + k;
    if (p.ttb_dtype == MOT_TTB_I16) id = ld_g(reinterpret_cast<const short*>(p.ttb) + e);
    else if (p.ttb_dtype == MOT_TTB_F32) id = (int)ld_g(reinterpret_cast<const float*>(p.ttb) + e);
    else id = (int)__bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p.ttb)[e]);
  } else {
    const long long idx = (p.flags & MOT_F_SLOT_MAJOR) ? (long long)slot * p.N + pos : pos * p.bpt + slot;
    id = (p.flags & MOT_F_IDS_I64) ? (int)ld_g(reinterpret_cast<const long long*>(p.ids) + idx)
                                   : ld_g(reinterpret_cast<const int*>(p.ids) + idx);
  }
  return id;
}
__device__ __forceinline__ int clamp_id(const EmbedParams& p, int id) { return clampi(id, p.Vb - 1); }

// ---- pulled ids derived from the token ids (MOT_F_TTB_PULL_LEFT) ----
// Entry k of ttb row tv as mot_ttb_expand writes it (float rows truncated to int64) and mot_pull reads it back (int).
__device__ __forceinline__ int ttb_raw(const void* ttb, int ttb_dtype, int tv, int bpt, int k) {
  const size_t e = (size_t)tv * bpt + k;
  if (ttb_dtype == MOT_TTB_I16) return ld_g(reinterpret_cast<const short*>(ttb) + e);
  if (ttb_dtype == MOT_TTB_F32) return (int)(long long)ld_g(reinterpret_cast<const float*>(ttb) + e);
  return (int)(long long)__bfloat162float(reinterpret_cast<const __nv_bfloat16*>(ttb)[e]);
}

struct PullSrc {
  const int32_t* tok;
  const void* ttb;
  long long T;  // tokens per row
  int V, bpt, ttb_dtype, pad, eot, scramble;
  const int32_t* next;  // right pulls with MOT_F_TTB_NEXT_TOK: next[r] = token T of row r (the lookahead); else nullptr
};

// Non-pad count of ttb row tv; eot = every entry is the EOT byte (mot_pull's pull_count_kernel).
__device__ __forceinline__ int ttb_row_count(const PullSrc& q, int tv, bool& eot) {
  int cnt = 0, n_eot = 0;
  for (int k = 0; k < q.bpt; ++k) {
    const int id = ttb_raw(q.ttb, q.ttb_dtype, tv, q.bpt, k);
    cnt += id != q.pad;
    n_eot += id == q.eot;
  }
  eot = n_eot == q.bpt;
  return cnt;
}
// Non-pad byte fi of ttb row tv as mot_pull's compacted stream keeps it (int16, hence the (short)); res if none.
__device__ __forceinline__ void ttb_nth_byte(const PullSrc& q, int tv, int fi, int& res) {
  for (int k = 0; k < q.bpt; ++k) {
    const int id = ttb_raw(q.ttb, q.ttb_dtype, tv, q.bpt, k);
    if (id != q.pad && fi-- == 0) {
      res = (int)(short)id;
      break;
    }
  }
}

// The bpt pulled ids of token t (pull_from_left over its row of T tokens, mot_pull.cu), computed by one warp without
// the pulled tensor: lane k < bpt returns slot k.  Raw values: pads and EOT are detected on them, the caller clamps.
// Lanes take tokens t, t-1, ..., t-31 of the row, each its non-pad count and EOT flag from its ttb row; the segment
// ends (going back) at an EOT token or the row start; an inclusive scan of the counts gives every token the range of
// backward byte indices it holds, and slot k receives backward index bpt - k.  Tokens with no non-pad byte can leave
// the 32-token window short of bpt bytes: the next window continues.  Integer work, bit-exact with mot_pull, whose
// compacted stream keeps the bytes as int16 (ttb_nth_byte).
__device__ __forceinline__ int pulled_ids_warp(const PullSrc q, int t) {
  const int lane = lane_id();
  const int row0 = (int)(t - t % q.T);
  const int want = q.bpt - lane;  // backward index (1 = last byte of the segment) of this lane's slot
  int res = q.pad, acc = 0;
  for (int base = t;; base -= 32) {
    const int j = base - lane;
    const bool valid = j >= row0;
    int cnt = 0, tv = 0;
    bool eot = false;
    if (valid) {
      tv = clampi(ld_g(q.tok + j), q.V - 1);
      cnt = ttb_row_count(q, tv, eot);
    }
    if (base == t && __shfl_sync(0xffffffffu, eot, 0)) return q.eot;  // EOT tokens pass through unchanged
    const unsigned stop = __ballot_sync(0xffffffffu, !valid || eot);
    const int f = stop ? __ffs(stop) - 1 : 32;  // lanes [0, f) belong to the segment
    if (lane >= f) cnt = 0;
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += u;
    }
    incl += acc;
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    int l = 0;  // first lane whose inclusive count reaches `want`
#pragma unroll
    for (int step = 16; step > 0; step >>= 1)
      if (__shfl_sync(0xffffffffu, incl, l + step - 1) < want) l += step;
    const int o_tv = __shfl_sync(0xffffffffu, tv, l), o_incl = __shfl_sync(0xffffffffu, incl, l);
    if (lane < q.bpt && want > acc && want <= total)  // index of the byte among the owner's non-pad bytes, in row order
      ttb_nth_byte(q, o_tv, o_incl - want, res);
    if (total >= q.bpt || f < 32) return res;
    acc = total;
  }
}

// The mirror image for pull_from_right (mot_pull.cu reads the row backwards): token t receives the first min(bpt, n)
// non-pad bytes of tokens t, t+1, ... before the next EOT token or the row end, left-aligned.  Lanes take tokens t,
// t+1, ..., t+31; the row ends after token T-1, or after the lookahead q.next[row] (read as token T) when there is one;
// the segment ends (going forward) before the first EOT token or the row end; the inclusive scan gives every token the
// range of forward byte indices it holds, and slot k receives forward index k + 1.
__device__ __forceinline__ int pulled_ids_right_warp(const PullSrc q, int t) {
  const int lane = lane_id();
  const int row = (int)(t / q.T);
  const int row_end = (int)((row + 1) * q.T);        // first index past the row's own tokens
  const int end = row_end + (q.next ? 1 : 0);        // index row_end reads the lookahead
  const int want = lane + 1;                         // forward index (1 = first byte of the segment) of this slot
  int res = q.pad, acc = 0;
  for (int base = t;; base += 32) {
    const int j = base + lane;
    const bool valid = j < end;
    int cnt = 0, tv = 0;
    bool eot = false;
    if (valid) {
      tv = clampi(j < row_end ? ld_g(q.tok + j) : ld_g(q.next + row), q.V - 1);
      cnt = ttb_row_count(q, tv, eot);
    }
    if (base == t && __shfl_sync(0xffffffffu, eot, 0)) return q.eot;  // EOT tokens pass through unchanged
    const unsigned stop = __ballot_sync(0xffffffffu, !valid || eot);
    const int f = stop ? __ffs(stop) - 1 : 32;  // lanes [0, f) belong to the segment
    if (lane >= f) cnt = 0;
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += u;
    }
    incl += acc;
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    int l = 0;  // first lane whose inclusive count reaches `want`
#pragma unroll
    for (int step = 16; step > 0; step >>= 1)
      if (__shfl_sync(0xffffffffu, incl, l + step - 1) < want) l += step;
    const int o_tv = __shfl_sync(0xffffffffu, tv, l), o_incl = __shfl_sync(0xffffffffu, incl, l);
    const int o_cnt = __shfl_sync(0xffffffffu, cnt, l);
    if (lane < q.bpt && want > acc && want <= total)  // index of the byte among the owner's non-pad bytes, in row order
      ttb_nth_byte(q, o_tv, want - (o_incl - o_cnt) - 1, res);
    if (total >= q.bpt || f < 32) return res;
    acc = total;
  }
}

// The pulled row of token t; the direction is a compile-time value, so that each instantiation carries one routine.
template <bool RIGHT>
__device__ __forceinline__ int pulled_row_warp(const PullSrc q, int t) {
  if constexpr (RIGHT) return pulled_ids_right_warp(q, t);
  else return pulled_ids_warp(q, t);
}

// Pulled id of this lane's slot at position pos (warp collective).  With the `.view(bpt,-1)` scramble every slot lane
// reads another token: the warp derives the pulled row of each of them in turn.
template <bool RIGHT>
__device__ __forceinline__ int fetch_pulled_id(const PullSrc q, int pos) {
  const int lane = lane_id();
  if (!q.scramble) return pulled_row_warp<RIGHT>(q, pos);
  const long long row = pos / q.T, s = pos - row * q.T;
  const long long f = (long long)min(lane, q.bpt - 1) * q.T + s;
  const int tokpos = (int)(row * q.T + f / q.bpt), k = (int)(f % q.bpt);
  int id = 0;
  for (int r = 0; r < q.bpt; ++r) {
    const int v = pulled_row_warp<RIGHT>(q, __shfl_sync(0xffffffffu, tokpos, r));
    const int got = __shfl_sync(0xffffffffu, v, __shfl_sync(0xffffffffu, k, r));
    if (lane == r) id = got;
  }
  return id;
}

// Per-lane view of the byte-id source, set up once: one multiply-add + load per position.
struct IdSrc {
  const char* base;      // address of (position 0, slot = lane) for id tensors
  unsigned pos_stride;   // bytes between consecutive positions (<= 8 * 32)
  int kind;              // 0: int32 tensor, 1: int64 tensor, 2: derived from the ttb table
};
__device__ __forceinline__ IdSrc make_id_src(const EmbedParams& p, int slot) {
  IdSrc s;
  const int esz = (p.flags & MOT_F_IDS_I64) ? 8 : 4;
  s.kind = (p.flags & MOT_F_IDS_FROM_TTB) ? 2 : ((p.flags & MOT_F_IDS_I64) ? 1 : 0);
  const bool sm = (p.flags & MOT_F_SLOT_MAJOR) != 0;
  s.base = reinterpret_cast<const char*>(p.ids) + (sm ? (long long)slot * p.N : (long long)slot) * esz;
  s.pos_stride = (unsigned)((sm ? 1 : p.bpt) * esz);
  return s;
}
__device__ __forceinline__ int load_raw_id(const EmbedParams& p, const IdSrc& s, int pos, int slot) {
  if (s.kind == 2) return fetch_id(p, pos, slot);
  const char* a = s.base + (unsigned long long)(unsigned)pos * s.pos_stride;  // one 32 x 32 -> 64 multiply-add
  return s.kind == 1 ? (int)ld_g(reinterpret_cast<const long long*>(a)) : ld_g(reinterpret_cast<const int*>(a));
}
// The kernels' PULL template value: kNoPull loads the byte ids (tensor or ttb rows); kPullLeft / kPullRight derive the
// pulled ids in the kernel, every id load being the warp collective fetch_pulled_id (the kNoPull instantiations carry
// none of its code, and each pulled instantiation one direction).
constexpr int kNoPull = 0, kPullLeft = 1, kPullRight = 2;
inline int ids_pulled(const EmbedParams& p) {
  if (!(p.flags & MOT_F_IDS_FROM_TTB) || p.bpt <= 0) return kNoPull;
  if (p.flags & MOT_F_TTB_PULL_LEFT) return kPullLeft;
  return (p.flags & MOT_F_TTB_PULL_RIGHT) ? kPullRight : kNoPull;
}
// Raw pulled id of this lane's slot (0 on lanes that hold no slot).  Every lane of the warp must call it.
// The lookahead tail of MOT_F_TTB_NEXT_TOK follows the N token ids.
template <int PULL>
__device__ __forceinline__ int pulled_lane_id(const EmbedParams& p, int pos, bool id_lane) {
  const int32_t* next = (PULL == kPullRight && (p.flags & MOT_F_TTB_NEXT_TOK)) ? p.tok + p.N : nullptr;
  const int id = fetch_pulled_id<PULL == kPullRight>(
      PullSrc{p.tok, p.ttb, p.T, p.V, p.bpt, p.ttb_dtype, (short)(p.pad_eot & 0xffff), p.pad_eot >> 16,
              (p.flags & MOT_F_TTB_SCRAMBLE) ? 1 : 0, next}, pos);
  return id_lane ? id : 0;
}

// Compile-time specialisation of the variant flags.  MODE 0: everything decided at run time (all variants);
// MODE 1: the MoT-sum fast path (runs/71): combine == ADD, out_norm only, no lambdas;
// MODE 4: MODE 0 plus a dense [N, Do] addend to the mixed row and its gradient (runs/71051:226-229);
// MODE 2 / 3: the two halves of the split [tok | bytes] concat operand of the projection variants (runs/7:226-232):
//   2 = tok-only rows with the per-input token norm, 3 = bytes-only rows with the per-byte norm (neither has a norm
//   over the mixed row, so the backward needs no reduction and keeps nothing of the row in registers).
// MODE 0 and MODE 4 decide every variant flag at run time; MODE 4 additionally handles the dense addend (kept out of
// MODE 0 so that the common kernels do not carry its registers)
#define MOT_RT(M) ((M) == 0 || (M) == 4)
// MODE 5: plain token gather (no norm, no lambdas): the value embeddings (runs/7:308);
// MODE 6: pure concat with the output norm only (runs/711:224-232), token / byte columns decided per chunk;
// MODE 16 + f: the ADD family with its flags fixed at compile time, f = tok_norm | byte_norm << 1 | out_norm << 2 |
//   lambdas << 3 (runs/73: f = 3, runs/74: 11, runs/71041..66: 15), byte table in shared memory.  The run-time-flag
//   kernel spends most of its instructions re-deciding these per chunk (2350 warp instructions per occurrence at
//   1024 columns, profiles/r1_bwd_generic_ncu.txt).
#define MOT_ADDFAM(M) ((M) >= 16)
#define MOT_ADDFLAG(M, bit) (MOT_ADDFAM(M) && (((M) - 16) & (bit)) != 0)
template <int MODE>
struct Cfg {
  __device__ __forceinline__ static bool tok_norm(const EmbedParams& p) {
    return MODE == 2 || MOT_ADDFLAG(MODE, 1) || (MOT_RT(MODE) && (p.flags & MOT_F_TOK_NORM));
  }
  __device__ __forceinline__ static bool byte_scale(const EmbedParams& p) {
    return MODE == 3 || MOT_ADDFLAG(MODE, 2 | 8) ||
           (MOT_RT(MODE) && ((p.flags & (MOT_F_BYTE_NORM | MOT_F_HAS_LAMBDAS)) || p.combine == MOT_MEAN));
  }
  __device__ __forceinline__ static bool has_lam(const EmbedParams& p) {
    return MOT_ADDFLAG(MODE, 8) || (MOT_RT(MODE) && (p.flags & MOT_F_HAS_LAMBDAS));
  }
  __device__ __forceinline__ static bool out_norm(const EmbedParams& p) {
    return MODE == 1 || MODE == 6 || MOT_ADDFLAG(MODE, 4) || (MOT_RT(MODE) && (p.flags & MOT_F_OUT_NORM));
  }
  __device__ __forceinline__ static bool has_tok(const EmbedParams& p) {
    return MODE == 1 || MODE == 2 || MODE == 5 || MODE == 6 || MOT_ADDFAM(MODE) || (MOT_RT(MODE) && p.combine != MOT_BYTES_ONLY);
  }
  __device__ __forceinline__ static bool has_bytes(const EmbedParams& p) {
    return MODE == 1 || MODE == 3 || MODE == 6 || MOT_ADDFAM(MODE) || (MOT_RT(MODE) && p.combine != MOT_TOK_ONLY);
  }
  __device__ __forceinline__ static bool mean(const EmbedParams& p) { return MOT_RT(MODE) && p.combine == MOT_MEAN; }
  // the token part / the byte part carries a scale that is not identically 1 (a norm or a lambda)
  static constexpr bool kTokScaled = MOT_RT(MODE) || MODE == 2 || MOT_ADDFLAG(MODE, 1 | 8);
  static constexpr bool kLam = MOT_RT(MODE) || MOT_ADDFLAG(MODE, 8);
};
inline int pick_mode(const EmbedParams& p, int cw) {
  if (p.addend != nullptr || p.d_addend != nullptr) return 4;  // the dense addend has its own instantiations
  const int f = p.flags & (MOT_F_TOK_NORM | MOT_F_BYTE_NORM | MOT_F_OUT_NORM | MOT_F_HAS_LAMBDAS);
  if (p.Do % (32 * cw) != 0) return 0;
  if (p.combine == MOT_ADD && f == MOT_F_OUT_NORM && p.tab_smem) return 1;
  if (p.combine == MOT_ADD && p.tab_smem)
    return 16 + ((f & MOT_F_TOK_NORM) ? 1 : 0) + ((f & MOT_F_BYTE_NORM) ? 2 : 0) + ((f & MOT_F_OUT_NORM) ? 4 : 0) +
           ((f & MOT_F_HAS_LAMBDAS) ? 8 : 0);
  if (p.combine == MOT_TOK_ONLY && f == 0) return 5;
  if (p.combine == MOT_CONCAT && f == MOT_F_OUT_NORM && p.tab_smem) return 6;
  if (p.combine == MOT_TOK_ONLY && f == MOT_F_TOK_NORM) return 2;
  if (p.combine == MOT_BYTES_ONLY && f == MOT_F_BYTE_NORM && p.tab_smem) return 3;
  return 0;
}

#define MOT_TOK_OK(it) (MODE == 1 || MODE == 2 || MODE == 5 || MOT_ADDFAM(MODE) || ((MOT_RT(MODE) || MODE == 6) && cm[it].toff >= 0))
#define MOT_BYTE_OK(it) (MODE == 1 || MODE == 3 || MOT_ADDFAM(MODE) || ((MOT_RT(MODE) || MODE == 6) && cm[it].slot >= 0))
// element offset of chunk `it` in the token row: affine (base + immediate addressing) on the fast path
#define MOT_TOFF(it) ((MODE == 1 || MODE == 2 || MODE == 5 || MOT_ADDFAM(MODE)) ? ((it) * 32 + lane) * CW : cm[it].toff)
#define MOT_CHUNK_OK(it) (!MOT_RT(MODE) || ((it) * 32 + lane) * CW < p.Do)

template <typename T, int MODE = 0, int CW = 8>
__device__ __forceinline__ typename Vec<T, CW>::Raw tab_load(const EmbedParams& p, const T* tab, size_t off) {
  if (MODE == 1 || MODE == 3 || MODE == 6 || MOT_ADDFAM(MODE)) return Vec<T, CW>::lds_raw(tab + off);  // only dispatched when the table fits
  return p.tab_smem ? Vec<T, CW>::lds_raw(tab + off) : Vec<T, CW>::ldg_raw(reinterpret_cast<const T*>(p.E_byte) + off);
}

// Stage E_byte into shared memory (bulk async copies of <= 32 KB) and compute the per-row rms scale
// of byte_norm: rs[r] = rsqrt(mean(row^2) + eps), or 1.  Ends with __syncthreads().  need_rs == false (a variant that
// never scales byte rows: the MoT-sum fast path) skips the scale pass: every thread has waited on the copy barrier
// itself, which is all the table reads need.
template <typename T>
__device__ __forceinline__ void issue_byte_table(const EmbedParams& p, T* tab, uint64_t* bar) {
  if (p.tab_smem && threadIdx.x == 0) {
    const uint32_t bytes = (uint32_t)p.Vb * p.bd * sizeof(T);
    mbar_expect_tx(bar, bytes);
    for (uint32_t done = 0; done < bytes;) {
      const uint32_t n = min(bytes - done, 32768u);
      bulk_g2s(reinterpret_cast<char*>(tab) + done, reinterpret_cast<const char*>(p.E_byte) + done, n, bar);
      done += n;
    }
  }
}
template <typename T>
__device__ void stage_byte_table(const EmbedParams& p, T* tab, float* rs, uint64_t* bar, bool need_rs, bool issued = false) {
  if (p.tab_smem) {
    if (!issued) issue_byte_table<T>(p, tab, bar);
    mbar_wait(bar, 0);
  }
  if (!need_rs) return;
  const int warp = threadIdx.x >> 5, nw = blockDim.x >> 5, lane = lane_id();
  const bool bn = (p.flags & MOT_F_BYTE_NORM) != 0;
  for (int r = warp; r < p.Vb; r += nw) {
    float ss = 0.f;
    if (bn) {
      for (int c = lane; c < p.bd / kChunk; c += 32) {
        float v[8];
        Vec8<T>::unpack(tab_load<T>(p, tab, (size_t)r * p.bd + c * kChunk), v);
#pragma unroll
        for (int e = 0; e < 8; ++e) ss += v[e] * v[e];
      }
      ss = warp_sum(ss);
    }
    if (lane == 0) rs[r] = bn ? rsqrtf(ss / (float)p.bd + p.eps) : 1.f;
  }
  __syncthreads();
}

__host__ __device__ inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Shared-memory layout shared by both kernels:
//   [rs: Vb floats][byte table (if tab_smem)][ring barriers: warps*stages u64][ring: warps*stages*stage_bytes]
struct SmemLayout {
  size_t rs, tab, bars, ring, stage_bytes, g_bytes, total;
};
__host__ __device__ inline SmemLayout smem_layout(const EmbedParams& p, size_t esz, int warps, bool backward) {
  SmemLayout L{};
  const bool has_bytes = p.combine != MOT_TOK_ONLY, has_tok = p.combine != MOT_BYTES_ONLY;
  size_t o = 0;
  L.rs = o;
  o += has_bytes ? align_up((size_t)p.Vb * 4, 128) : 0;
  L.tab = o;
  o += (has_bytes && p.tab_smem) ? align_up((size_t)p.Vb * p.bd * esz, 128) : 0;
  L.bars = o;
  o += align_up((size_t)warps * p.stages * 8, 128);
  L.ring = o;
  L.g_bytes = backward ? align_up((size_t)p.Do * esz, 128) : 0;
  L.stage_bytes = L.g_bytes + (has_tok ? align_up((size_t)p.Dt * esz, 128) : 0);
  o += (size_t)warps * p.stages * L.stage_bytes;
  L.total = o;
  return L;
}

// fp32 accumulate of 4 consecutive values into the L2-resident scratch: one RED.E.ADD.F32x4 (no return value, no
// dependency chain).  A warp-wide instruction covers 512 contiguous bytes per byte row piece: the L2 atomic units work
// per 32-byte sector, so two lanes fill one sector per request (tools/ubench/red_bench.cu: 28.8 us for the 37.7 M adds
// of the 48K-token workload, against 49.0 us when a lane owns 8 consecutive floats and issues two half-sector REDs;
// shared-memory fp32 atomics are CAS spin loops, 47.3 us).
__device__ __forceinline__ void gmem_add4(float* a, const float (&v)[4]) {
#ifdef MOT_EXPERIMENT_NO_RED
  if (v[0] == 12345.678f) a[0] = v[1];
  return;
#endif
  atomicAdd(reinterpret_cast<float4*>(a), make_float4(v[0], v[1], v[2], v[3]));
}

// ======================================================================================
// Forward
// ======================================================================================
template <typename T, int CPL, int MODE, int NT, int PULL>
__global__ void __launch_bounds__(NT, 1) mot_fwd_kernel(const EmbedParams p) {
  using C = Cfg<MODE>;
  constexpr int CW = 8;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ uint64_t tab_bar;
  const int lane = lane_id();
  const int warp = threadIdx.x >> 5;
  const int nw = blockDim.x >> 5;
  const SmemLayout L = smem_layout(p, sizeof(T), nw, false);
  float* rs = reinterpret_cast<float*>(smem_raw + L.rs);
  T* tab = reinterpret_cast<T*>(smem_raw + L.tab);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + L.bars) + warp * p.stages;
  unsigned char* ring = smem_raw + L.ring + (size_t)warp * p.stages * L.stage_bytes;
  const bool has_tok = C::has_tok(p), has_bytes = C::has_bytes(p);
  const int D = p.stages;

  if (threadIdx.x == 0) mbar_init(&tab_bar, 1);
  if (lane == 0)
    for (int s = 0; s < D; ++s) mbar_init(bars + s, 1);
  fence_mbar_init();
  pdl_launch_dependents();
  __syncthreads();
  const int gw = warp * gridDim.x + blockIdx.x;  // interleaved over the CTAs: every SM gets the same share +-1
                                                 // (n_tokens < 2^31, validated on the host: 32-bit position math)
  MOT_STAMP(p.trace, gw, 0);
  pdl_wait();  // nothing above touches global memory
  MOT_STAMP(p.trace, gw, 1);

  const int stride = gridDim.x * nw;
  const int Ni = (int)p.N;
  const int n_i = gw < Ni ? (Ni - gw + stride - 1) / stride : 0;  // positions of this warp
  const T* E_tok = reinterpret_cast<const T*>(p.E_tok);
  const uint32_t row_bytes = (uint32_t)p.Dt * sizeof(T);

  // the byte table first (one elected thread, no dependent loads in front of it), then the ring prologue: the token rows
  // are in flight while the table arrives
  if (has_bytes) issue_byte_table<T>(p, tab, &tab_bar);
  int tok_ahead = 0;  // lane 0: raw token id of position i + D
  if (has_tok && lane == 0) {
    for (int i = 0; i < D && i < n_i; ++i) {
      const int tv = clampi(ld_g(p.tok + gw + i * stride), p.V - 1);
      mbar_expect_tx(bars + i, row_bytes);
      bulk_g2s(ring + (size_t)i * L.stage_bytes, E_tok + mul_u32(tv, p.Dt), row_bytes, bars + i);
    }
    if (D < n_i) tok_ahead = ld_g(p.tok + gw + D * stride);  // raw; clamped where it is used
  }
  MOT_STAMP(p.trace, gw, 2);
  if (has_bytes) stage_byte_table<T>(p, tab, rs, &tab_bar, C::byte_scale(p), /*issued=*/true);
  MOT_STAMP(p.trace, gw, 3);

  ChunkMap cm[CPL];
#pragma unroll
  for (int it = 0; it < CPL; ++it) cm[it] = chunk_map<CW>(p, it * 32 + lane);

  float lam_t = 1.f, lam_b = 1.f;
  if (C::has_lam(p)) {
    lam_t = ld_g(p.lam);
    lam_b = ld_g(p.lam + 1);
  }
  if (C::mean(p)) lam_b /= (float)p.bpt;
  T* out = reinterpret_cast<T*>(p.out);
  const bool tok_norm = C::tok_norm(p), out_norm = C::out_norm(p), byte_scale = C::byte_scale(p);

  const float inv_Dt = 1.f / (float)(p.Dt > 0 ? p.Dt : 1), inv_Do = 1.f / (float)p.Do;
  const bool id_lane = has_bytes && lane < p.bpt;
  const IdSrc idsrc = make_id_src(p, lane);
  // raw byte ids are fetched two positions ahead and clamped where they are consumed
  int id_n1, id_n2;
  if constexpr (PULL) {
    id_n1 = n_i > 0 ? pulled_lane_id<PULL>(p, gw, id_lane) : 0;
    id_n2 = n_i > 1 ? pulled_lane_id<PULL>(p, gw + stride, id_lane) : 0;
  } else {
    id_n1 = (id_lane && n_i > 0) ? load_raw_id(p, idsrc, gw, lane) : 0;
    id_n2 = (id_lane && n_i > 1) ? load_raw_id(p, idsrc, gw + stride, lane) : 0;
  }
  int s = 0;
  uint32_t parity = 0;
  int pos = gw;
  for (int i = 0; i < n_i; ++i, pos += stride) {
    const int idreg = clamp_id(p, id_n1);
    id_n1 = id_n2;
    if constexpr (PULL) {
      if (i + 2 < n_i) id_n2 = pulled_lane_id<PULL>(p, pos + 2 * stride, id_lane);
    } else {
      if (id_lane && i + 2 < n_i) id_n2 = load_raw_id(p, idsrc, pos + 2 * stride, lane);
    }

    float x[CPL][8];
    float ss_t = 0.f;
    if (has_tok) {
      mbar_wait(bars + s, parity);
      MOT_STAMP(p.trace, gw, 5 + i);
      const T* trow = reinterpret_cast<const T*>(ring + (size_t)s * L.stage_bytes);
#pragma unroll
      for (int it = 0; it < CPL; ++it) {
        if (MOT_TOK_OK(it)) {
          Vec8<T>::unpack(Vec8<T>::lds_raw(trow + MOT_TOFF(it)), x[it]);
          if (tok_norm) {
#pragma unroll
            for (int e = 0; e < 8; ++e) ss_t += x[it][e] * x[it][e];
          }
        } else {
#pragma unroll
          for (int e = 0; e < 8; ++e) x[it][e] = 0.f;
        }
      }
    } else {
#pragma unroll
      for (int it = 0; it < CPL; ++it)
#pragma unroll
        for (int e = 0; e < 8; ++e) x[it][e] = 0.f;
    }
    float tscale = lam_t;
    if (tok_norm) {
      ss_t = warp_sum(ss_t);
      tscale *= rsqrtf(ss_t * inv_Dt + p.eps);
    }
    float ss = 0.f;
#pragma unroll
    for (int it = 0; it < CPL; ++it) {
      if (C::kTokScaled) {
#pragma unroll
        for (int e = 0; e < 8; ++e) x[it][e] *= tscale;
      }
      if (has_bytes) {
        if (C::mean(p)) {
          for (int k = 0; k < p.bpt; ++k) {
            const int id = __shfl_sync(0xffffffffu, idreg, k);
            if (cm[it].slot == -2) {
              float b[8];
              Vec8<T>::unpack(tab_load<T, MODE>(p, tab, (unsigned)(id * p.bd + cm[it].boff)), b);
              const float bs = lam_b * rs[id];
#pragma unroll
              for (int e = 0; e < 8; ++e) x[it][e] += bs * b[e];
            }
          }
        } else {
          const int id = __shfl_sync(0xffffffffu, idreg, cm[it].slot & 31);
          if (MOT_BYTE_OK(it)) {
            float b[8];
            Vec8<T>::unpack(tab_load<T, MODE>(p, tab, (unsigned)(id * p.bd + cm[it].boff)), b);
            if (byte_scale) {
              const float bs = lam_b * rs[id];
#pragma unroll
              for (int e = 0; e < 8; ++e) x[it][e] += bs * b[e];
            } else {
#pragma unroll
              for (int e = 0; e < 8; ++e) x[it][e] += b[e];
            }
          }
        }
      }
      if (MODE == 4 && p.addend != nullptr && MOT_CHUNK_OK(it)) {
        float ad[8];
        Vec8<T>::unpack(Vec8<T>::ldg_raw(reinterpret_cast<const T*>(p.addend) + (size_t)pos * p.Do + (size_t)(it * 32 + lane) * kChunk), ad);
#pragma unroll
        for (int e = 0; e < 8; ++e) x[it][e] += ad[e];
      }
      if (out_norm) {
#pragma unroll
        for (int e = 0; e < 8; ++e) ss += x[it][e] * x[it][e];
      }
    }
    float oscale = 1.f;
    if (out_norm) {
      ss = warp_sum(ss);  // every lane has consumed its shared-memory reads here: the stage can be refilled
      oscale = rsqrtf(ss * inv_Do + p.eps);
      if (p.rstd_out != nullptr && lane == 0) p.rstd_out[pos] = oscale;
    } else {
      __syncwarp();
    }
    if (has_tok && lane == 0 && i + D < n_i) {
      mbar_expect_tx(bars + s, row_bytes);
      bulk_g2s(ring + (size_t)s * L.stage_bytes, E_tok + mul_u32(clampi(tok_ahead, p.V - 1), p.Dt), row_bytes, bars + s);
      if (i + D + 1 < n_i) tok_ahead = ld_g(p.tok + pos + (D + 1) * stride);
    }
    if (++s == D) {
      s = 0;
      parity ^= 1u;
    }
    T* orow = out + mul_u32(pos, (int)p.io_ld) + p.io_col;
#pragma unroll
    for (int it = 0; it < CPL; ++it) {
      if (MOT_CHUNK_OK(it)) {
        if (out_norm) {
#pragma unroll
          for (int e = 0; e < 8; ++e) x[it][e] *= oscale;
        }
        Vec8<T>::stg(orow + (size_t)(it * 32 + lane) * kChunk, x[it]);
      }
    }
  }
  MOT_STAMP(p.trace, gw, 62);
#ifdef MOT_TRACE
  if (p.trace != nullptr && lane == 0) p.trace[(size_t)gw * 64 + 63] = n_i;
#endif
}

// ======================================================================================
// Backward
// ======================================================================================
// The backward kernel uses 4-element chunks (CW = 4): chunk c = it*32 + lane, so every warp-wide access is a contiguous
// 256 B (bf16) / 512 B (fp32) segment and the byte-gradient REDs fill whole 32-byte sectors (see gmem_add4).
constexpr int kBwdCW = 4;

// Finish one token row: Du = sum over its occurrences of d z[token part]; tv = the raw token row (shared or
// global memory); writes d E_tok[v] and returns <Du, that> (the row's contribution to d lam_tok).
template <typename T, int CPL, int MODE>
__device__ __forceinline__ float finish_tok_row(const EmbedParams& p, const ChunkMap (&cm)[CPL], int v, float (&Du)[CPL][kBwdCW],
                                                const T* trow_smem, float lam_t) {
  using C = Cfg<MODE>;
  constexpr int CW = kBwdCW;
  using V = Vec<T, CW>;
  const int lane = lane_id();
  const bool tok_norm = C::tok_norm(p);
  const bool need_t = tok_norm || C::has_lam(p);
  float dot = 0.f, ss = 0.f;  // <Du, tv>, |tv|^2
  if (need_t) {
#pragma unroll
    for (int it = 0; it < CPL; ++it) {
      if (MOT_TOK_OK(it)) {
        float tv[CW];
        V::unpack(V::lds_raw(trow_smem + MOT_TOFF(it)), tv);
#pragma unroll
        for (int e = 0; e < CW; ++e) {
          dot += Du[it][e] * tv[e];
          ss += tv[e] * tv[e];
        }
      }
    }
    warp_sum2(dot, ss);
  }
  const float r_t = tok_norm ? rsqrtf(ss / (float)p.Dt + p.eps) : 1.f;
  // d that = lam_t * Du ; dt = r_t * d that - tv * r_t^3 * mean(d that . tv)
  const float a = lam_t * r_t;
  const float b = tok_norm ? lam_t * r_t * r_t * r_t * dot / (float)p.Dt : 0.f;
  T* grow = reinterpret_cast<T*>(p.gE_tok) + mul_u32(v, p.Dt);
#pragma unroll
  for (int it = 0; it < CPL; ++it) {
    if (MOT_TOK_OK(it)) {
      float o[CW];
      if (tok_norm) {
        float tv[CW];
        V::unpack(V::lds_raw(trow_smem + MOT_TOFF(it)), tv);
#pragma unroll
        for (int e = 0; e < CW; ++e) o[e] = a * Du[it][e] - b * tv[e];
      } else if (C::kLam) {
#pragma unroll
        for (int e = 0; e < CW; ++e) o[e] = a * Du[it][e];
      } else {
#pragma unroll
        for (int e = 0; e < CW; ++e) o[e] = Du[it][e];
      }
      V::stg(grow + MOT_TOFF(it), o);
    }
  }
  return r_t * dot;
}

// One batch of the token-sorted stream: up to 32 consecutive entries, one per lane.
struct Batch {
  int pos, v;      // per lane: position and token id of entry `lane`
  int cnt;         // valid entries (0: the stream is exhausted)
  int chunk, sub;  // stream chunk and batch index inside the chunk
};

// CTA size of the backward: 12 warps; the widest ADD-family kernel with an output norm (32 columns per lane kept for the
// mixed row and the accumulator) runs 8 warps so that it fits the register file without spilling.
#ifndef MOT_WIDE_STATIC_THREADS
#define MOT_WIDE_STATIC_THREADS 256
#endif
template <int CPL, int MODE>
constexpr int bwd_threads() { return (MOT_ADDFLAG(MODE, 4) && CPL >= 8) ? MOT_WIDE_STATIC_THREADS : kBwdThreads; }

template <typename T, int CPL, int MODE, int PULL>
__global__ void __launch_bounds__((bwd_threads<CPL, MODE>()), 1) mot_bwd_kernel(const EmbedParams p) {
  using C = Cfg<MODE>;
  constexpr int CW = kBwdCW;
  using V = Vec<T, CW>;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ uint64_t tab_bar;
  const int lane = lane_id();
  const int warp = threadIdx.x >> 5;
  const int nw = blockDim.x >> 5;
  const SmemLayout L = smem_layout(p, sizeof(T), nw, true);
  float* rs = reinterpret_cast<float*>(smem_raw + L.rs);
  T* tab = reinterpret_cast<T*>(smem_raw + L.tab);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + L.bars) + warp * p.stages;
  unsigned char* ring = smem_raw + L.ring + (size_t)warp * p.stages * L.stage_bytes;
  const bool has_tok = C::has_tok(p), has_bytes = C::has_bytes(p);
  const int D = p.stages;

  if (threadIdx.x == 0) mbar_init(&tab_bar, 1);
  if (lane == 0)
    for (int s = 0; s < D; ++s) mbar_init(bars + s, 1);
  fence_mbar_init();
  pdl_launch_dependents();
  __syncthreads();
  pdl_wait();  // nothing above touches global memory

  const int gw = warp * gridDim.x + blockIdx.x;  // interleaved over the CTAs
  const int W = gridDim.x * nw;
  const T* E_tok = reinterpret_cast<const T*>(p.E_tok);
  const T* gout = reinterpret_cast<const T*>(p.gout);
  const uint32_t g_bytes = (uint32_t)p.Do * sizeof(T);
  // the token row itself is only needed where the backward goes through a norm or a lambda (a plain gather, e.g. the
  // value embeddings of runs/7:308, has d E[v] = sum of the upstream rows: R = 0 in SURVEY 8d's byte count)
  const bool need_trow = has_tok && (C::tok_norm(p) || C::out_norm(p) || C::has_lam(p));
  const uint32_t t_bytes = need_trow ? (uint32_t)p.Dt * sizeof(T) : 0u;

  // ---- the warp's share of the token-sorted stream: chunks gw, gw+W, ... of R entries (gw is interleaved over the
  //      CTAs, so every SM gets the same number of chunks +-1), walked in batches of 32 entries (one per lane) ----
  const int Ni = (int)p.N;  // n_tokens < 2^31 (validated on the host): 32-bit stream math
  const int n_stream_chunks = (Ni + p.R - 1) / p.R;
  int nx_chunk = gw, nx_sub = 0;    // the next batch to load
  auto load_next = [&](Batch& b) {
    b.pos = 0;
    b.v = -1;
    b.cnt = 0;
    b.chunk = -1;
    b.sub = 0;
    if (nx_chunk >= n_stream_chunks) return;
    const int a = nx_chunk * p.R + nx_sub * 32;  // < Ni by construction
    const int c_end = min(nx_chunk * p.R + p.R, Ni);
    const int left = c_end - a;
    b.cnt = left < 32 ? left : 32;
    b.chunk = nx_chunk;
    b.sub = nx_sub;
    if (lane < b.cnt) {
      if (has_tok) {
        b.pos = ld_g(p.order + a + lane);
        b.v = ld_g(p.stok + a + lane);
      } else {
        b.pos = a + lane;  // bytes-only: no token table, the stream is the position order
        b.v = 0;
      }
    }
    if (a + 32 >= c_end) {
      nx_chunk += W;
      nx_sub = 0;
    } else {
      ++nx_sub;
    }
  };
  Batch A, B;
  load_next(A);
  load_next(B);

  // ---- ring: occurrence n of this warp lives in stage n % D ----
  int issued = 0, consumed = 0;  // occurrences of this warp (< 2^31)
  int is = 0;                    // stage of the next issue  (issued % D)
  int cs = 0;                    // stage of the next consume (consumed % D)
  int ps = 0;                    // stage of the previous consume
  uint32_t cpar = 0;             // mbarrier parity of the next consume ((consumed / D) & 1)
  int iw = 0, ik = 0;            // issue cursor: batch (0 = A, 1 = B) and entry
  auto try_issue = [&]() -> bool {
    for (;;) {
      const int cnt = iw ? B.cnt : A.cnt;
      if (ik < cnt) break;
      if (iw == 1) return false;  // ran past the prefetched batch: wait for the consumer to advance
      iw = 1;
      ik = 0;
    }
    if (lane == ik) {  // the lane that holds entry ik of the batch issues its two row copies (no broadcast needed)
      const int pos = iw ? B.pos : A.pos, v = iw ? B.v : A.v;
      unsigned char* st = ring + (size_t)is * L.stage_bytes;
      mbar_expect_tx(bars + is, g_bytes + t_bytes);
      bulk_g2s(st, gout + mul_u32(pos, (int)p.io_ld) + p.io_col, g_bytes, bars + is);
      if (need_trow) bulk_g2s(st + L.g_bytes, E_tok + mul_u32(v, p.Dt), t_bytes, bars + is);
    }
    ++issued;
    if (++is == D) is = 0;
    ++ik;
    return true;
  };
  while (issued < D && try_issue()) {
  }

  if (has_bytes) stage_byte_table<T>(p, tab, rs, &tab_bar, C::byte_scale(p));  // ring prologue already in flight

  ChunkMap cm[CPL];
#pragma unroll
  for (int it = 0; it < CPL; ++it) cm[it] = chunk_map<CW>(p, it * 32 + lane);

  const bool has_lam = C::has_lam(p);
  float lam_t = 1.f, lam_b = 1.f;
  if (has_lam) {
    lam_t = ld_g(p.lam);
    lam_b = ld_g(p.lam + 1);
  }
  const float inv_pool = C::mean(p) ? 1.f / (float)p.bpt : 1.f;
  const float lam_b_eff = lam_b * inv_pool;
  const bool tok_norm = C::tok_norm(p), out_norm = C::out_norm(p), byte_scale = C::byte_scale(p);
  float dlam_t = 0.f, dlam_b = 0.f;  // per-lane partials
  float* accp = p.byte_acc + (size_t)(gw % p.n_rep) * p.Vb * p.bd;
  const float inv_Dt = 1.f / (float)(p.Dt > 0 ? p.Dt : 1), inv_Do = 1.f / (float)p.Do;
  const bool id_lane = has_bytes && lane < p.bpt;
  const IdSrc idsrc = make_id_src(p, lane);

  // ---- phase Z: rows nobody gathered get zeros (the dense-grad contract of the reference) ----
  if (has_tok) {
    T* G = reinterpret_cast<T*>(p.gE_tok);
    const float zero[CW] = {0.f, 0.f, 0.f, 0.f};
    for (int vb = gw * 32; vb < p.V; vb += W * 32) {
      const int v = vb + lane;
      const bool empty = v < p.V && (ld_g(p.off + v + 1) - ld_g(p.off + v)) == 0;
      unsigned m = __ballot_sync(0xffffffffu, empty);
      while (m) {
        const int j = __ffs(m) - 1;
        m &= m - 1;
        T* row = G + mul_u32(vb + j, p.Dt);
        for (int c = lane; c < p.Dt / CW; c += 32) V::stg(row + c * CW, zero);
      }
    }
  }

  // ---- phase S: the stream ----
  float Du[CPL][CW];
#pragma unroll
  for (int it = 0; it < CPL; ++it)
#pragma unroll
    for (int e = 0; e < CW; ++e) Du[it][e] = 0.f;
  int cur_v = -1;
  bool seg_lead = false;  // current row segment started at the chunk start and continues a row of the previous chunk
  float tscale = lam_t;   // lam_t * r_t of the current row

  // flush the current row segment: direct write if the whole row lies inside this chunk, else fp32 RED into its slot
  auto flush = [&](bool trail) {
    const T* trow = reinterpret_cast<const T*>(ring + (size_t)ps * L.stage_bytes + L.g_bytes);
    if (!seg_lead && !trail) {
      const float d = finish_tok_row<T, CPL, MODE>(p, cm, cur_v, Du, trow, lam_t);
      if (lane == 0) dlam_t += d;
    } else {
      // the row continues in another chunk: add this segment into the fp32 slot of the row's FIRST chunk (a chunk is
      // the first chunk of at most one such row: its last one).  Hot rows spread over many chunks meet there through
      // the L2 atomic units; the finalize kernel reads the one slot, writes the row and zeroes the slot again.
      const int c_first = ld_g(p.off + cur_v) / p.R;
      float* prow = p.partial + mul_u32(c_first, p.Dt);
#pragma unroll
      for (int it = 0; it < CPL; ++it) {
        if (MOT_TOK_OK(it))
          atomicAdd(reinterpret_cast<float4*>(prow + MOT_TOFF(it)), make_float4(Du[it][0], Du[it][1], Du[it][2], Du[it][3]));
      }
    }
#pragma unroll
    for (int it = 0; it < CPL; ++it)
#pragma unroll
      for (int e = 0; e < CW; ++e) Du[it][e] = 0.f;
  };

  while (A.cnt > 0) {
    const int chunk = A.chunk;
    const int a = chunk * p.R + A.sub * 32;
    const bool chunk_first = A.sub == 0, chunk_last = a + 32 >= min(chunk * p.R + p.R, Ni);
    int v_before = -1;
    if (has_tok && chunk_first && a > 0) v_before = ld_g(p.stok + a - 1);
    const int pos_first = __shfl_sync(0xffffffffu, A.pos, 0);  // warp collective: outside lane-dependent branches
    int id_next;
    if constexpr (PULL) id_next = pulled_lane_id<PULL>(p, pos_first, id_lane);
    else id_next = id_lane ? load_raw_id(p, idsrc, pos_first, lane) : 0;
    for (int k = 0; k < A.cnt; ++k) {
      const int v = __shfl_sync(0xffffffffu, A.v, k);
      const int pos_k = __shfl_sync(0xffffffffu, A.pos, k);  // position of this occurrence (dense addend rows)
      const bool new_row = has_tok && v != cur_v;
      if (new_row) {  // flush BEFORE refilling the ring: the old row's token row sits in stage (consumed-1) % D
        if (cur_v >= 0) flush(false);
        seg_lead = chunk_first && k == 0 && v == v_before;
        cur_v = v;
      }
      if (issued - consumed < D) try_issue();  // one stage was freed by the previous occurrence
      const int idreg = clamp_id(p, id_next);
      const int pos_ahead = __shfl_sync(0xffffffffu, A.pos, (k + 1) & 31);
      if constexpr (PULL) {
        if (k + 1 < A.cnt) id_next = pulled_lane_id<PULL>(p, pos_ahead, id_lane);
      } else {
        if (id_lane && k + 1 < A.cnt) id_next = load_raw_id(p, idsrc, pos_ahead, lane);
      }

      mbar_wait(bars + cs, cpar);
      ++consumed;
      const T* grow = reinterpret_cast<const T*>(ring + (size_t)cs * L.stage_bytes);
      const T* trow = reinterpret_cast<const T*>(ring + (size_t)cs * L.stage_bytes + L.g_bytes);
      ps = cs;
      if (++cs == D) {
        cs = 0;
        cpar ^= 1u;
      }

      if (new_row && tok_norm) {
        float ss_t = 0.f;
#pragma unroll
        for (int it = 0; it < CPL; ++it) {
          if (MOT_TOK_OK(it)) {
            float tv[CW];
            V::unpack(V::lds_raw(trow + MOT_TOFF(it)), tv);
#pragma unroll
            for (int e = 0; e < CW; ++e) ss_t += tv[e] * tv[e];
          }
        }
        ss_t = warp_sum(ss_t);
        tscale = lam_t * rsqrtf(ss_t * inv_Dt + p.eps);
      }

      int idv[CPL];  // byte id of this lane's slot per chunk (warp collective: outside lane-dependent branches)
#pragma unroll
      for (int it = 0; it < CPL; ++it) idv[it] = has_bytes ? __shfl_sync(0xffffffffu, idreg, cm[it].slot & 31) : 0;
      // z = tscale * t + lam_b * rs * b
      float z[CPL][CW];  // mixed row of this occurrence (only with out_norm)
      float ss = 0.f, gz = 0.f;
      if (out_norm) {
#pragma unroll
      for (int it = 0; it < CPL; ++it) {
        if (has_tok && MOT_TOK_OK(it)) {
          V::unpack(V::lds_raw(trow + MOT_TOFF(it)), z[it]);
          if (C::kTokScaled) {
#pragma unroll
            for (int e = 0; e < CW; ++e) z[it][e] *= tscale;
          }
        } else {
#pragma unroll
          for (int e = 0; e < CW; ++e) z[it][e] = 0.f;
        }
        if (has_bytes) {
          if (C::mean(p)) {
            for (int kk = 0; kk < p.bpt; ++kk) {
              const int id = __shfl_sync(0xffffffffu, idreg, kk);
              if (cm[it].slot == -2) {
                float b[CW];
                V::unpack(tab_load<T, MODE, CW>(p, tab, (unsigned)(id * p.bd + cm[it].boff)), b);
                const float bs = lam_b_eff * rs[id];
#pragma unroll
                for (int e = 0; e < CW; ++e) z[it][e] += bs * b[e];
              }
            }
          } else {
            const int id = idv[it];
            if (MOT_BYTE_OK(it)) {
              float b[CW];
              V::unpack(tab_load<T, MODE, CW>(p, tab, (unsigned)(id * p.bd + cm[it].boff)), b);
              if (byte_scale) {
                const float bs = lam_b_eff * rs[id];
#pragma unroll
                for (int e = 0; e < CW; ++e) z[it][e] += bs * b[e];
              } else {
#pragma unroll
                for (int e = 0; e < CW; ++e) z[it][e] += b[e];
              }
            }
          }
        }
        if (MODE == 4 && p.addend != nullptr && MOT_CHUNK_OK(it)) {
          float ad[CW];
          V::unpack(V::ldg_raw(reinterpret_cast<const T*>(p.addend) + (size_t)pos_k * p.Do + (size_t)(it * 32 + lane) * CW), ad);
#pragma unroll
          for (int e = 0; e < CW; ++e) z[it][e] += ad[e];
        }
        if (MOT_CHUNK_OK(it)) {
          float g4[CW];  // not kept across the reduction: the second pass reads the staged row again (registers)
          V::unpack(V::lds_raw(grow + (size_t)(it * 32 + lane) * CW), g4);
#pragma unroll
          for (int e = 0; e < CW; ++e) {
            ss += z[it][e] * z[it][e];
            gz += g4[e] * z[it][e];
          }
        }
      }
      }
      float r_o = 1.f, coef = 0.f;
      if (out_norm) {
        warp_sum2(ss, gz);
        r_o = rsqrtf(ss * inv_Do + p.eps);
        coef = r_o * r_o * r_o * gz * inv_Do;
      }
#pragma unroll
      for (int it = 0; it < CPL; ++it) {
        const bool valid = MOT_CHUNK_OK(it);  // lane-dependent: no warp collectives under it
        float dz[CW];
        if (valid) {
          if (out_norm) {
            float g4[CW];
            V::unpack(V::lds_raw(grow + (size_t)(it * 32 + lane) * CW), g4);
#pragma unroll
            for (int e = 0; e < CW; ++e) dz[e] = r_o * g4[e] - coef * z[it][e];
          } else {  // no norm over the mixed row: dz is the upstream gradient itself
            V::unpack(V::lds_raw(grow + (size_t)(it * 32 + lane) * CW), dz);
          }
          if (MOT_TOK_OK(it)) {
#pragma unroll
            for (int e = 0; e < CW; ++e) Du[it][e] += dz[e];
          }
          if (MODE == 4 && p.d_addend != nullptr)
            V::stg(reinterpret_cast<T*>(p.d_addend) + (size_t)pos_k * p.Do + (size_t)(it * 32 + lane) * CW, dz);
        } else {
#pragma unroll
          for (int e = 0; e < CW; ++e) dz[e] = 0.f;
        }
        if (has_bytes) {
          if (C::mean(p)) {
            for (int kk = 0; kk < p.bpt; ++kk) {
              const int id = __shfl_sync(0xffffffffu, idreg, kk);
              if (valid && cm[it].slot == -2) {
                if (has_lam) {
                  float b[CW];
                  V::unpack(tab_load<T, MODE, CW>(p, tab, (unsigned)(id * p.bd + cm[it].boff)), b);
                  const float r = rs[id] * inv_pool;
#pragma unroll
                  for (int e = 0; e < CW; ++e) dlam_b += dz[e] * r * b[e];
                }
                float dzs[CW];
#pragma unroll
                for (int e = 0; e < CW; ++e) dzs[e] = dz[e] * lam_b_eff;
                gmem_add4(accp + (unsigned)(id * p.bd + cm[it].boff), dzs);
              }
            }
          } else if (valid && MOT_BYTE_OK(it)) {
            const int id = idv[it];
            if (has_lam) {  // d lam_byte += <dz, bhat>
              float b[CW];
              V::unpack(tab_load<T, MODE, CW>(p, tab, (unsigned)(id * p.bd + cm[it].boff)), b);
              const float r = rs[id];
#pragma unroll
              for (int e = 0; e < CW; ++e) dlam_b += dz[e] * r * b[e];
            }
            if (C::kLam) {
#pragma unroll
              for (int e = 0; e < CW; ++e) dz[e] *= lam_b_eff;
            }
            gmem_add4(accp + (unsigned)(id * p.bd + cm[it].boff), dz);
          }
        }
      }
      __syncwarp();  // shared-memory reads of this stage are done (values consumed above)
    }
    // at the end of a chunk the open row segment is flushed
    if (chunk_last && has_tok && cur_v >= 0) {
      const int b_end = chunk * p.R + p.R;
      const bool trail = b_end < Ni && ld_g(p.stok + b_end) == cur_v;
      flush(trail);
      cur_v = -1;
      seg_lead = false;
    }
    // advance: A <- B, prefetch the batch after
    A = B;
    if (iw == 1) iw = 0; else ik = 0;
    load_next(B);
    // the issue cursor may have been waiting for this batch.  An open row whose flush reads its token row (token norm /
    // lambdas) still needs the most recently consumed stage `ps`: the refill must leave that one stage alone until the
    // flush at the next row change (the issue order fills the OLDEST free stage first, so keeping one stage free is
    // keeping `ps`).  Without this a row ending exactly at a 32-entry batch boundary inside a chunk (chunks longer than
    // one batch: more than 56832 tokens) was normalised against a half-overwritten token row.
    const int hold = (cur_v >= 0 && need_trow && (tok_norm || has_lam)) ? 1 : 0;
    while (issued - consumed < D - hold && try_issue()) {
    }
  }

  // ---- lambda partials ----
  if (has_lam) {
    dlam_t = warp_sum(dlam_t);
    dlam_b = warp_sum(dlam_b);
    if (lane == 0) {
      atomicAdd(p.lam_acc, dlam_t);
      atomicAdd(p.lam_acc + 1, dlam_b);
    }
  }
}

// Finalize: (a) token rows that straddle stream-chunk boundaries: sum their fp32 partials in stream order,
// apply the token-norm backward, write the row; (b) byte table: sum the accumulator replicas, apply the
// byte-norm backward, cast; (c) lambda partials of (a).
template <typename T>
__global__ void __launch_bounds__(256) mot_bwd_finalize_kernel(const EmbedParams p) {
  pdl_launch_dependents();
  MOT_STAMP(p.trace, (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) & 4095, 0);
  pdl_wait();
  const int lane = lane_id();
  const int nw = blockDim.x >> 5;
  const int gw = blockIdx.x * nw + (threadIdx.x >> 5);
  MOT_STAMP(p.trace, gw & 4095, 1);
  const int W = gridDim.x * nw;
  const bool has_tok = p.combine != MOT_BYTES_ONLY;
  const bool has_bytes = p.combine != MOT_TOK_ONLY;
  const bool has_lam = (p.flags & MOT_F_HAS_LAMBDAS) != 0;
  float lam_t = 1.f;
  if (has_lam) lam_t = ld_g(p.lam);
  float dlam_t = 0.f;
  if (blockIdx.x == 0 && threadIdx.x == 0 && p.lam_acc != nullptr)
    reinterpret_cast<int*>(p.lam_acc)[2] = 0;  // zero-fill work counter of the saved-output backward (self-cleaning)
  if (has_tok) {
    const bool tok_norm = (p.flags & MOT_F_TOK_NORM) != 0;
    // chunk boundaries strictly inside this launch's part of the stream [off[v_lo], off[v_hi]) (the whole stream unless
    // the backward runs as vocabulary slabs): a slab starts and ends on a row boundary, so no row crosses it
    const long long a0 = ld_g(p.off + p.v_lo), a1 = ld_g(p.off + p.v_hi);
    const long long c_lo = a0 / p.R, c_hi = (a1 + p.R - 1) / p.R;
    const T* E_tok = reinterpret_cast<const T*>(p.E_tok);
    T* G = reinterpret_cast<T*>(p.gE_tok);
    MOT_ASSERT(a0 >= 0 && a0 <= a1 && a1 <= p.N, "finalize stream range", a0, a1);
    for (long long c0 = c_lo + gw; c0 + 1 < c_hi; c0 += W) {
      MOT_ASSERT(c0 >= 0 && c0 < p.n_slots, "finalize slot", c0, p.n_slots);
      const long long bnd = (c0 + 1) * (long long)p.R;  // first stream entry of chunk c0 + 1
      MOT_ASSERT(bnd > 0 && bnd < p.N, "finalize boundary", bnd, p.N);
      const int v = ld_g(p.stok + bnd - 1);
      MOT_ASSERT(v >= 0 && v < p.V, "finalize token", v, p.V);
      if (ld_g(p.stok + bnd) != v) continue;                  // no row crosses this boundary
      if (ld_g(p.off + v) < c0 * (long long)p.R) continue;    // the row started in an earlier chunk: not ours
      float* prow = p.partial + (size_t)c0 * p.Dt;             // all segments of the row were added here
      const T* trow = E_tok + (size_t)v * p.Dt;
      float dot = 0.f, ss = 0.f;
      // pass 0 (only when the token-norm backward or d lam_tok need <Du, t> and |t|^2), pass 1 writes the row
      for (int pass = (tok_norm || has_lam) ? 0 : 1; pass < 2; ++pass) {
        const float r_t = tok_norm ? rsqrtf(ss / (float)p.Dt + p.eps) : 1.f;
        const float a_ = lam_t * r_t;
        const float b_ = tok_norm ? lam_t * r_t * r_t * r_t * dot / (float)p.Dt : 0.f;
        float dacc = 0.f, sacc = 0.f;
        for (int c = lane; c < p.Dt / kChunk; c += 32) {
          float tv[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, du[8];
          if (tok_norm || has_lam) Vec8<T>::unpack(Vec8<T>::ldg_raw(trow + c * kChunk), tv);
          float* pr = prow + c * kChunk;
          const float4 x = *reinterpret_cast<const float4*>(pr), y = *reinterpret_cast<const float4*>(pr + 4);
          du[0] = x.x; du[1] = x.y; du[2] = x.z; du[3] = x.w; du[4] = y.x; du[5] = y.y; du[6] = y.z; du[7] = y.w;
          if (pass == 0) {
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              dacc += du[e] * tv[e];
              sacc += tv[e] * tv[e];
            }
          } else {
            float o[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) o[e] = a_ * du[e] - b_ * tv[e];
            Vec8<T>::stg(G + (size_t)v * p.Dt + c * kChunk, o);
            // leave the slot zeroed for the next call (self-cleaning workspace, MOT_WS_CLEAN)
            *reinterpret_cast<float4*>(pr) = make_float4(0.f, 0.f, 0.f, 0.f);
            *reinterpret_cast<float4*>(pr + 4) = make_float4(0.f, 0.f, 0.f, 0.f);
          }
        }
        if (pass == 0) {
          warp_sum2(dacc, sacc);
          dot = dacc;
          ss = sacc;
          if (lane == 0) dlam_t += (tok_norm ? rsqrtf(ss / (float)p.Dt + p.eps) : 1.f) * dot;
        }
      }
    }
  }
  if (has_bytes && p.last_slab) {
    // One warp per byte row.  The row has nc = bd / 8 chunks of 8 elements and kByteRep replicas: lane = group * nc + c
    // owns chunk c of the replicas {group, group + G, ...} (G = 32 / nc lane groups), so every replica load of the row is
    // in flight at once (one L2 round trip instead of one per 8 replicas with 6 of 32 lanes working: the byte rows were
    // the critical path of this kernel, 5-6.6 us of 6.6, profiles/r2_timeline.md); the groups then meet through shuffles.
    const bool bn = (p.flags & MOT_F_BYTE_NORM) != 0;
    const T* E_byte = reinterpret_cast<const T*>(p.E_byte);
    T* G = reinterpret_cast<T*>(p.gE_byte);
    const size_t rep_stride = (size_t)p.Vb * p.bd;
    const int nc = p.bd / kChunk;  // <= 32 (bd <= 256, validated on the host for byte_norm; wider rows take the slow loop)
    // byte rows are handed out from the LAST warp of the grid backwards (the chunk boundaries above from the first
    // forwards), so a grid of (boundaries + Vb) warps gives one task per warp
    for (int r = W - 1 - gw; r < p.Vb; r += W) {
      if (nc <= 32) {
        const int ngrp = 32 / nc;                    // lane groups (>= 1)
        const int grp = lane / nc, c = lane - grp * nc;
        const bool live = grp < ngrp;
        float a[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (live) {
          float* base = p.byte_acc + (size_t)r * p.bd + c * kChunk;
          // replicas grp, grp + G, grp + 2G, ...: four per trip (bd <= 64: one trip covers all 16)
#pragma unroll 1
          for (int j0 = 0; grp + j0 * ngrp < kByteRep; j0 += 4) {
            float4 x[4], y[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int rep = grp + (j0 + j) * ngrp;
              if (rep < kByteRep) {
                x[j] = *reinterpret_cast<const float4*>(base + rep * rep_stride);
                y[j] = *reinterpret_cast<const float4*>(base + rep * rep_stride + 4);
              }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int rep = grp + (j0 + j) * ngrp;
              if (rep < kByteRep) {  // zeroed again for the next call (the workspace cleans itself, MOT_WS_CLEAN)
                *reinterpret_cast<float4*>(base + rep * rep_stride) = make_float4(0.f, 0.f, 0.f, 0.f);
                *reinterpret_cast<float4*>(base + rep * rep_stride + 4) = make_float4(0.f, 0.f, 0.f, 0.f);
                a[0] += x[j].x; a[1] += x[j].y; a[2] += x[j].z; a[3] += x[j].w;
                a[4] += y[j].x; a[5] += y[j].y; a[6] += y[j].z; a[7] += y[j].w;
              }
            }
          }
        }
        // group g adds into group 0: lane c receives from lanes c + g * nc (fixed order: deterministic given the replicas)
        for (int g2 = 1; g2 < ngrp; ++g2) {
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float o_ = __shfl_sync(0xffffffffu, a[e], (lane + g2 * nc) & 31);
            if (lane < nc) a[e] += o_;
          }
        }
        float ev[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        const bool owner = lane < nc;
        if (bn && owner) Vec8<T>::unpack(Vec8<T>::ldg_raw(E_byte + (size_t)r * p.bd + c * kChunk), ev);
        float rsr = 1.f, b_ = 0.f;
        if (bn) {
          float dot = 0.f, ss = 0.f;
          if (owner) {
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              dot += a[e] * ev[e];
              ss += ev[e] * ev[e];
            }
          }
          warp_sum2(dot, ss);
          rsr = rsqrtf(ss / (float)p.bd + p.eps);
          b_ = rsr * rsr * rsr * dot / (float)p.bd;
        }
        if (owner) {
          float o[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) o[e] = rsr * a[e] - b_ * ev[e];
          Vec8<T>::stg(G + (size_t)r * p.bd + c * kChunk, o);
        }
      } else {
        // rows wider than 256 elements (no byte norm: refused on the host): one lane per chunk, replicas in turn
        for (int c0 = 0; c0 < nc; c0 += 32) {
          const int c = c0 + lane;
          if (c >= nc) continue;
          float a[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
          float* base = p.byte_acc + (size_t)r * p.bd + c * kChunk;
          for (int rep = 0; rep < kByteRep; ++rep) {
            const float4 x = *reinterpret_cast<const float4*>(base + rep * rep_stride);
            const float4 y = *reinterpret_cast<const float4*>(base + rep * rep_stride + 4);
            *reinterpret_cast<float4*>(base + rep * rep_stride) = make_float4(0.f, 0.f, 0.f, 0.f);
            *reinterpret_cast<float4*>(base + rep * rep_stride + 4) = make_float4(0.f, 0.f, 0.f, 0.f);
            a[0] += x.x; a[1] += x.y; a[2] += x.z; a[3] += x.w; a[4] += y.x; a[5] += y.y; a[6] += y.z; a[7] += y.w;
          }
          Vec8<T>::stg(G + (size_t)r * p.bd + c * kChunk, a);
        }
      }
    }
  }
  if (has_lam) {
    dlam_t = warp_sum(dlam_t);
    if (lane == 0 && dlam_t != 0.f) atomicAdd(p.lam_acc, dlam_t);
  }
  MOT_STAMP(p.trace, gw & 4095, 62);
}

// ======================================================================================
// Launchers
// ======================================================================================
// Pick the ring depth and whether the byte table fits next to it; returns dynamic smem bytes or 0.
inline size_t plan_smem(EmbedParams& p, size_t esz, int warps, bool backward, int optin) {
  static const char* env_st = getenv("MOT_STAGES");  // debug knob
  const int want = env_st ? atoi(env_st) : 2;  // measured: 2 stages per warp are as fast as 4 (profiles/r1_experiments.md)
  p.tab_smem = 1;
  for (int tab = 1; tab >= 0; --tab) {
    p.tab_smem = tab;
    for (int st = want; st >= 2; --st) {
      p.stages = st;
      const SmemLayout L = smem_layout(p, esz, warps, backward);
      if (L.total + 1024 <= (size_t)optin) return L.total;
    }
  }
  return 0;
}

template <typename T, int CPL, int MODE, int PULL = kNoPull>
static int launch_fwd(const EmbedParams& p_in, cudaStream_t s) {
  if constexpr (PULL == kNoPull && MODE != 2 && MODE != 5) {
    if (const int k = ids_pulled(p_in))
      return k == kPullLeft ? launch_fwd<T, CPL, MODE, kPullLeft>(p_in, s) : launch_fwd<T, CPL, MODE, kPullRight>(p_in, s);
  }
  int sms = 0, optin = 0;
  if (int rc = device_props(&sms, &optin)) return rc;
  EmbedParams p = p_in;
  // Rows up to 3 x 256 elements: compiled for <= 64 registers, launched with 24 warps.  Wider rows hold more of the
  // row per lane: compiled for <= 128 registers, 16 warps (no spills; measured as fast at 1024 elements).
  constexpr int NT = CPL * sizeof(T) <= 6 ? 1024 : 512;
  static const char* env_thr = getenv("MOT_FWD_THREADS");  // debug knob
  int threads = env_thr ? atoi(env_thr) : (NT == 1024 ? kFwdThreads : 512);
  if (threads > NT) threads = NT;
  size_t smem = 0;
  for (; threads >= 256; threads = threads > 512 ? threads - 256 : threads >> 1) {
    smem = plan_smem(p, sizeof(T), threads / 32, false, optin);
    if (smem != 0 && (p.tab_smem || p.combine == MOT_TOK_ONLY || threads == 256)) break;
  }
  if (smem == 0) return MOT_ERR_UNSUPPORTED;
  if ((MODE == 1 || MOT_ADDFAM(MODE)) && !p.tab_smem) return launch_fwd<T, CPL, 0, PULL>(p_in, s);  // fast paths assume the table in smem
  p.trace = g_trace;
  auto kern = mot_fwd_kernel<T, CPL, MODE, NT, PULL>;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return check_launch();
  const long long warps_needed = p.N;
  long long blocks = (warps_needed + (threads / 32) - 1) / (threads / 32);
  if (blocks > sms) blocks = sms;
  if (blocks < 1) blocks = 1;
  if (g_prof_fwd_start) cudaEventRecord(g_prof_fwd_start, s);
  launch_pdl(kern, dim3((unsigned)blocks), dim3(threads), smem, s, p);
  if (g_prof_fwd_stop) cudaEventRecord(g_prof_fwd_stop, s);
  count_launch();
  return check_launch();
}

template <typename T, int CPL, int MODE, int PULL = kNoPull>
static int launch_bwd(const EmbedParams& p_in, cudaStream_t s) {
  if constexpr (PULL == kNoPull && MODE != 2 && MODE != 5) {
    if (const int k = ids_pulled(p_in))
      return k == kPullLeft ? launch_bwd<T, CPL, MODE, kPullLeft>(p_in, s) : launch_bwd<T, CPL, MODE, kPullRight>(p_in, s);
  }
  int sms = 0, optin = 0;
  if (int rc = device_props(&sms, &optin)) return rc;
  EmbedParams p = p_in;
  constexpr int NT = bwd_threads<CPL, MODE>();
  const size_t smem = plan_smem(p, sizeof(T), NT / 32, true, optin);
  if (smem == 0) return MOT_ERR_UNSUPPORTED;
  if ((MODE == 1 || MODE == 3 || MODE == 6 || MOT_ADDFAM(MODE)) && !p.tab_smem) return launch_bwd<T, CPL, 0, PULL>(p_in, s);  // fast paths assume the table in smem
  auto kern = mot_bwd_kernel<T, CPL, MODE, PULL>;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return check_launch();
  if (g_prof_start) cudaEventRecord(g_prof_start, s);
  launch_pdl(kern, dim3((unsigned)sms), dim3(NT), smem, s, p);
  if (g_prof_stop) cudaEventRecord(g_prof_stop, s);
  count_launch();
  return check_launch();
}

// per-translation-unit dispatchers (one TU per element type so nvcc compiles them in parallel)
int dispatch_fwd_bf16(const EmbedParams& p, cudaStream_t s);
int dispatch_fwd_f32(const EmbedParams& p, cudaStream_t s);
int dispatch_bwd_bf16(const EmbedParams& p, cudaStream_t s);
int dispatch_bwd_f32(const EmbedParams& p, cudaStream_t s);
int dispatch_bwd_split_bf16(const EmbedParams& p, int mode, cudaStream_t s);  // MODE 2 / 3 instantiations
int dispatch_fwd_static_bf16(const EmbedParams& p, int mode, cudaStream_t s);  // MODE 16+f forward instantiations; -1: none
int dispatch_bwd_static_bf16(const EmbedParams& p, int mode, cudaStream_t s);  // MODE 5 / 16+f instantiations; -1: none
int dispatch_bwd_gather_bf16(const EmbedParams& p, cudaStream_t s);
int dispatch_bwd_concat_bf16(const EmbedParams& p, cudaStream_t s);
int dispatch_bwd_sum_bf16(const EmbedParams& p, cudaStream_t s);  // saved-output MoT-sum kernel; -1: not applicable
int dispatch_bwd_sum_f32(const EmbedParams& p, cudaStream_t s);
int dispatch_fwd_addend_bf16(const EmbedParams& p, cudaStream_t s);  // MODE 4 instantiations
int dispatch_fwd_addend_f32(const EmbedParams& p, cudaStream_t s);
int dispatch_bwd_addend_bf16(const EmbedParams& p, cudaStream_t s);
int dispatch_bwd_addend_f32(const EmbedParams& p, cudaStream_t s);
int launch_finalize_bf16(const EmbedParams& p, int blocks, cudaStream_t s);
int launch_finalize_f32(const EmbedParams& p, int blocks, cudaStream_t s);

}  // namespace mot
