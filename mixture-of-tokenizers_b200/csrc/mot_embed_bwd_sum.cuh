// Backward of the MoT-sum variant (runs/71:228-230,312-314: out = rms_norm(E_tok[tok] + concat_k E_byte[id_k])) from the
// SAVED forward result: the autograd graph of F.rms_norm keeps its output side, so the backward does not have to
// rebuild the mixed row z = t + C'.  With o = out (= z * r) and r = rstd saved by the forward,
//     dz = r * g - z * r^3 * mean(g . z) = r * g - o * (r * mean(g . o)),
// so an occurrence needs two rows (g and o, both indexed by the POSITION) instead of three (g, the token row and
// bpt byte rows), no byte table in shared memory and no second reduction.  Same HBM bytes as the recompute kernel
// (the out row replaces the token row), about half the instructions (profiles/r1_bwd_sum_ncu.txt).
//
// Work split, ring and scatter are those of mot_bwd_kernel (mot_embed_kernels.cuh): persistent CTAs, a warp owns whole
// chunks of the token-sorted stream, one lane per 4-element chunk of the row, rows arrive through a per-warp ring of
// 1-D bulk copies, token rows are written once (rows that straddle stream chunks go through the fp32 slot of their
// first chunk and the finalize kernel), byte gradients are RED.v4.f32 into L2-resident replicas.
#pragma once
#include "mot_embed_kernels.cuh"

namespace mot {

// Threads per CTA of the saved-output kernel and its body shape.  Two passes over the staged rows (reduce, then
// re-read and scatter) keep only the token-gradient accumulator in registers across the warp reduction, which lets
// more warps share the SM; one pass keeps both rows unpacked (12 warps).
#ifndef MOT_SUM_THREADS
#define MOT_SUM_THREADS 384
#endif
#ifndef MOT_SUM_TWO_PASS
#define MOT_SUM_TWO_PASS 0
#endif
// Byte gradients through the TMA engine: the warp writes dz (fp32) over the ring stage it has just consumed and the lanes
// that hold the byte ids each hand one slot (bd floats) to cp.reduce.async.bulk...add.f32, which adds it into the L2-resident
// accumulator replica.  The SM issues bpt bulk operations per occurrence instead of 32 x CPL RED.128, no id shuffles, and
// the reductions drain beside the next occurrence; the stage is refilled one occurrence later (when the bulk group has
// read it).  Measurements: profiles/r2_experiments.md.
#ifndef MOT_SUM_BULK_RED
#define MOT_SUM_BULK_RED 0
#endif
constexpr int kSumThreads = MOT_SUM_THREADS;

struct SumSmem {
  size_t bars, ring, row_bytes, stage_bytes, total;
};
__host__ __device__ inline SumSmem sum_smem(int Do, size_t esz, int warps, int stages) {
  SumSmem L{};
  L.bars = 0;
  L.ring = align_up((size_t)warps * stages * 8, 128);
  L.row_bytes = align_up((size_t)Do * esz, 128);
  L.stage_bytes = 2 * L.row_bytes;  // [grad row | saved out row]
  L.total = L.ring + (size_t)warps * stages * L.stage_bytes;
  return L;
}

// mbarrier / bulk-copy helpers on 32-bit shared addresses (no generic -> shared conversion per call)
__device__ __forceinline__ void mbar_expect_tx_s(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait_s(uint32_t bar, uint32_t phase) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}\n" ::"r"(bar),
      "r"(phase)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s_s(uint32_t dst, const void* gmem_src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(gmem_src), "r"(bytes), "r"(bar)
               : "memory");
}

// One batch of the token-sorted stream: up to 32 consecutive entries of one stream chunk, one per lane.
struct SumBatch {
  int pos, v;  // per lane: position and token id of entry `lane`
  float r;     // per lane: saved rstd of that position
  int cnt;     // valid entries (0: the stream is exhausted)
  int a;       // stream index of entry 0
  int flags;   // bit 0: first batch of its chunk, bit 1: last batch of its chunk
  int v_prev;  // first batch: token id of the stream entry before the chunk (-1: none)
  int v_next;  // last batch: token id of the stream entry after the chunk (-1: none)
};

template <typename T, int CPL, int PULL>
__global__ void __launch_bounds__(kSumThreads, 1) mot_bwd_sum_kernel(const EmbedParams p) {
  constexpr int CW = kBwdCW;
  using V = Vec<T, CW>;
  constexpr unsigned kFull = 0xffffffffu;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int lane = lane_id();
  const int warp = threadIdx.x >> 5;
  const int nw = blockDim.x >> 5;
  const int D = p.stages;
  const SumSmem L = sum_smem(p.Do, sizeof(T), nw, D);
  const uint32_t bars_s = smem_u32(smem_raw + L.bars) + (uint32_t)(warp * D) * 8u;
  const uint32_t stage_bytes = (uint32_t)L.stage_bytes, row_off = (uint32_t)L.row_bytes;
  unsigned char* ring = smem_raw + L.ring + (size_t)warp * D * L.stage_bytes;
  const uint32_t ring_s = smem_u32(ring);

  if (lane == 0)
    for (int s = 0; s < D; ++s) mbar_init(reinterpret_cast<uint64_t*>(smem_raw + L.bars) + warp * D + s, 1);
  fence_mbar_init();
  pdl_launch_dependents();
  __syncthreads();
  const int gw = warp * gridDim.x + blockIdx.x;  // interleaved over the CTAs: every SM gets the same share +-1
  MOT_STAMP(p.trace, gw, 0);
  // The sort plan (order / stok / off) was finished before this kernel was launched when the caller joined it through an
  // event (plan_early): the first two batches of the stream are fetched while the predecessor kernel is still draining.
  // Everything the predecessor may have written (rstd, the saved output, the upstream gradient) waits for
  // griddepcontrol.wait.
  if (!p.plan_early) pdl_wait();

  const int W = gridDim.x * nw;
  const int Ni = (int)p.N, R = p.R;  // n_tokens < 2^31 (validated on the host): 32-bit stream math
  const char* gout = reinterpret_cast<const char*>(p.gout);
  const char* osv = reinterpret_cast<const char*>(p.out_saved);
  const uint32_t row_bytes = (uint32_t)p.Do * sizeof(T);  // rows of gout / out_saved are contiguous (never a split concat)

  // ---- this launch's part of the stream: the entries of the vocabulary rows [v_lo, v_hi), i.e. [a0, a1) (the whole
  //      stream unless the backward runs as slabs of the data-parallel pipeline).  Chunks keep their GLOBAL numbering
  //      (chunk c = entries [c R, (c+1) R)), clipped to [a0, a1): a slab starts and ends on a row boundary.
  const int a0 = ld_g(p.off + p.v_lo), a1 = ld_g(p.off + p.v_hi);
  const int c_lo = a0 / R, c_hi = (a1 + R - 1) / R;
  MOT_ASSERT(a0 >= 0 && a0 <= a1 && a1 <= Ni, "stream range", a0, a1);
  MOT_ASSERT(p.v_lo >= 0 && p.v_lo <= p.v_hi && p.v_hi <= p.V, "row range", p.v_lo, p.v_hi);

  // ---- the warp's share: chunks c_lo + gw, c_lo + gw + W, ... walked in batches of <= 32 entries ----
  int nx_chunk = c_lo + gw, nx_a = max(nx_chunk * R, a0);  // the next batch to load
  auto load_next = [&](SumBatch& b, bool with_r) {
    b.pos = 0;
    b.v = -1;
    b.r = 0.f;
    b.cnt = 0;
    b.a = 0;
    b.flags = 0;
    b.v_prev = -1;
    b.v_next = -1;
    if (nx_chunk >= c_hi) return;
    const int c0 = max(nx_chunk * R, a0), c_end = min(nx_chunk * R + R, a1);
    const int a = nx_a, left = c_end - a;
    b.a = a;
    b.cnt = left < 32 ? left : 32;
    MOT_ASSERT(a >= a0 && a + b.cnt <= a1 && b.cnt >= 0, "batch range", a, b.cnt);
    if (lane < b.cnt) {
      b.pos = ld_g(p.order + a + lane);
      b.v = ld_g(p.stok + a + lane);
      MOT_ASSERT(b.pos >= 0 && b.pos < Ni, "position", b.pos, a + lane);
      MOT_ASSERT(b.v >= p.v_lo && b.v < p.v_hi, "token row", b.v, a + lane);
      if (with_r) b.r = ld_g(p.rstd + b.pos);
    }
    if (a == c0) {
      b.flags |= 1;
      if (a > 0) b.v_prev = ld_g(p.stok + a - 1);
    }
    if (left <= 32) {
      b.flags |= 2;
      if (c_end < Ni) b.v_next = ld_g(p.stok + c_end);
      nx_chunk += W;
      nx_a = nx_chunk < c_hi ? max(nx_chunk * R, a0) : 0;
    } else {
      nx_a = a + 32;
    }
  };
  SumBatch A, B;
  load_next(A, !p.plan_early);
  load_next(B, !p.plan_early);
  if (p.plan_early) {
    pdl_wait();
    if (lane < A.cnt) A.r = ld_g(p.rstd + A.pos);
    if (lane < B.cnt) B.r = ld_g(p.rstd + B.pos);
  }
  MOT_STAMP(p.trace, gw, 1);
  MOT_STAMP(p.trace, gw, 2);

  // ---- ring: occurrence n of this warp lives in stage n % D ----
  int inflight = 0;    // issued - consumed
  int is = 0, cs = 0;  // stage of the next issue / the next consume
  uint32_t cpar = 0;   // mbarrier parity of the next consume
  int iw = 0, ik = 0;  // issue cursor: batch (0 = A, 1 = B) and entry
  auto try_issue = [&]() -> bool {
    int cnt = iw ? B.cnt : A.cnt;
    if (ik >= cnt) {
      if (iw == 1 || B.cnt == 0) return false;  // ran past the prefetched batch / end of the stream
      iw = 1;
      ik = 0;
    }
    if (lane == ik) {  // the lane that holds the entry issues its two row copies (no broadcast needed)
      const unsigned long long goff = (unsigned long long)(unsigned)(iw ? B.pos : A.pos) * row_bytes;
      const uint32_t st = ring_s + (uint32_t)is * stage_bytes, bar = bars_s + (uint32_t)is * 8u;
      mbar_expect_tx_s(bar, 2u * row_bytes);
      bulk_g2s_s(st, gout + goff, row_bytes, bar);
#ifdef MOT_X_SUM_NO_OCOPY
      bulk_g2s_s(st + row_off, gout + goff, row_bytes, bar);  // same row twice: half the gather traffic
#else
      bulk_g2s_s(st + row_off, osv + goff, row_bytes, bar);
#endif
    }
    ++inflight;
    if (++is == D) is = 0;
    ++ik;
    return true;
  };
  while (inflight < D && try_issue()) {
  }
  MOT_STAMP(p.trace, gw, 3);

  // ---- per-lane constants: byte slot and accumulator offset of each of the lane's chunks ----
#if !MOT_SUM_BULK_RED || MOT_SUM_TWO_PASS
  int slot[CPL];
  unsigned boff4[CPL];  // byte offset of the lane's chunk inside a row of the fp32 accumulator
#pragma unroll
  for (int it = 0; it < CPL; ++it) {
    const int e = (it * 32 + lane) * CW;
    slot[it] = e / p.bd;
    boff4[it] = (unsigned)(e - slot[it] * p.bd) * 4u;
    asm volatile("" : "+r"(slot[it]), "+r"(boff4[it]));  // keep them in registers (no 64-bit rematerialisation per use)
  }
#else
  bool red_pending = false;  // the previous occurrence's stage still feeds its bulk reductions (released one occurrence later)
#endif
  const unsigned bd4 = (unsigned)p.bd * 4u;
  char* accp = reinterpret_cast<char*>(p.byte_acc + (size_t)(gw % p.n_rep) * p.Vb * p.bd);
  const float inv_Do = 1.f / (float)p.Do;
  const bool id_lane = lane < p.bpt;
  const IdSrc idsrc = make_id_src(p, lane);
  T* G = reinterpret_cast<T*>(p.gE_tok);

  MOT_STAMP(p.trace, gw, 4);
  // ---- phase S: the stream ----
#ifdef MOT_TRACE
  int n_occ = 0;
#endif
  float Du[CPL][CW];
#pragma unroll
  for (int it = 0; it < CPL; ++it)
#pragma unroll
    for (int e = 0; e < CW; ++e) Du[it][e] = 0.f;
  int cur_v = -1;
  bool seg_lead = false;  // the open row segment started at the chunk start and continues a row of the previous chunk

  // close the open row segment: direct write if the whole row lies inside this chunk, else fp32 RED into the slot of the
  // row's FIRST chunk (hot rows spread over many chunks meet there; the finalize kernel writes the row)
  auto flush = [&](bool partial_row) {
    if (!partial_row) {
#ifndef MOT_X_SUM_NO_FLUSH
      MOT_ASSERT(cur_v >= p.v_lo && cur_v < p.v_hi, "flush row", cur_v, p.v_hi);
      T* grow = G + (size_t)(unsigned)cur_v * (unsigned)p.Dt;
#pragma unroll
      for (int it = 0; it < CPL; ++it) V::stg(grow + (it * 32 + lane) * CW, Du[it]);
#endif
    } else {
      const int c_first = ld_g(p.off + cur_v) / R;
      MOT_ASSERT(c_first >= 0 && c_first < p.n_slots, "partial slot", c_first, p.n_slots);
      float* prow = p.partial + (size_t)(unsigned)c_first * (unsigned)p.Dt;
#pragma unroll
      for (int it = 0; it < CPL; ++it)
        atomicAdd(reinterpret_cast<float4*>(prow + (it * 32 + lane) * CW), make_float4(Du[it][0], Du[it][1], Du[it][2], Du[it][3]));
    }
#pragma unroll
    for (int it = 0; it < CPL; ++it)
#pragma unroll
      for (int e = 0; e < CW; ++e) Du[it][e] = 0.f;
  };

  int id_next = 0;  // raw byte id (lane = slot) of the next occurrence, fetched one occurrence ahead
  if (A.cnt > 0) {
    const int pos0 = __shfl_sync(kFull, A.pos, 0);
    if constexpr (PULL) id_next = pulled_lane_id<PULL>(p, pos0, id_lane);
    else if (id_lane) id_next = load_raw_id(p, idsrc, pos0, lane);
  }
  while (A.cnt > 0) {
    const int cnt = A.cnt;
    for (int k = 0; k < cnt; ++k) {
      const int v = __shfl_sync(kFull, A.v, k);
      const float r = __shfl_sync(kFull, A.r, k);
      if (v != cur_v) {
        if (cur_v >= 0) flush(seg_lead);
        seg_lead = k == 0 && (A.flags & 1) && v == A.v_prev;
        cur_v = v;
      }
      const int idreg = clamp_id(p, id_next);
      {  // byte ids of the next occurrence (the first entry of the next batch after the last one of this batch)
        const bool more = k + 1 < cnt;  // warp-uniform
        const int pos_n = __shfl_sync(kFull, more ? A.pos : B.pos, more ? k + 1 : 0);
        if constexpr (PULL) {
          if (more || B.cnt > 0) id_next = pulled_lane_id<PULL>(p, pos_n, id_lane);
        } else {
          if (id_lane && (more || B.cnt > 0)) id_next = load_raw_id(p, idsrc, pos_n, lane);
        }
      }

      mbar_wait_s(bars_s + (uint32_t)cs * 8u, cpar);
#ifdef MOT_TRACE
      MOT_STAMP(p.trace, gw, 5 + n_occ);
      ++n_occ;
#endif
      const T* grow = reinterpret_cast<const T*>(ring + (size_t)cs * stage_bytes);
      const T* orow = reinterpret_cast<const T*>(ring + (size_t)cs * stage_bytes + row_off);
#if MOT_SUM_BULK_RED
      float* dzrow = reinterpret_cast<float*>(ring + (size_t)cs * stage_bytes);  // dz (fp32) overwrites [g | o] in place
      const uint32_t dz_s = ring_s + (uint32_t)cs * stage_bytes;
#endif
      if (++cs == D) {
        cs = 0;
        cpar ^= 1u;
      }
#if MOT_SUM_TWO_PASS
      float gzp[CW] = {0.f, 0.f, 0.f, 0.f};  // independent partial sums: no serial dependency chain over the row
#pragma unroll
      for (int it = 0; it < CPL; ++it) {
        float g[CW], o[CW];
        V::unpack(V::lds_raw(grow + (it * 32 + lane) * CW), g);
        V::unpack(V::lds_raw(orow + (it * 32 + lane) * CW), o);
#pragma unroll
        for (int e = 0; e < CW; ++e) gzp[e] += g[e] * o[e];
      }
      float gz = (gzp[0] + gzp[1]) + (gzp[2] + gzp[3]);
      gz = warp_sum(gz);
      const float c = r * gz * inv_Do;
#ifdef MOT_X_SUM_NO_MATH
      if (c == 12345.678f)
#endif
#pragma unroll
      for (int it = 0; it < CPL; ++it) {
        const int id = __shfl_sync(kFull, idreg, slot[it]);
        float g[CW], o[CW], dz[CW];
        V::unpack(V::lds_raw(grow + (it * 32 + lane) * CW), g);
        V::unpack(V::lds_raw(orow + (it * 32 + lane) * CW), o);
#pragma unroll
        for (int e = 0; e < CW; ++e) {
          dz[e] = r * g[e] - c * o[e];
          Du[it][e] += dz[e];
        }
        gmem_add4(reinterpret_cast<float*>(accp + ((unsigned)id * bd4 + boff4[it])), dz);
      }
      __syncwarp();  // every lane has its second-pass shared-memory reads in registers: the stage can be refilled
      --inflight;
      try_issue();
#else
      float g[CPL][CW], o[CPL][CW];
      float gzp[CW] = {0.f, 0.f, 0.f, 0.f};  // independent partial sums: no serial dependency chain over the row
#pragma unroll
      for (int it = 0; it < CPL; ++it) {
        V::unpack(V::lds_raw(grow + (it * 32 + lane) * CW), g[it]);
        V::unpack(V::lds_raw(orow + (it * 32 + lane) * CW), o[it]);
#pragma unroll
        for (int e = 0; e < CW; ++e) gzp[e] += g[it][e] * o[it][e];
      }
      float gz = (gzp[0] + gzp[1]) + (gzp[2] + gzp[3]);
      gz = warp_sum(gz);  // every lane has its shared-memory reads in registers here: the stage can be refilled
#if !MOT_SUM_BULK_RED
      --inflight;
      try_issue();
#endif
      const float c = r * gz * inv_Do;
#ifdef MOT_X_SUM_NO_MATH
      if (c == 12345.678f)
#endif
#pragma unroll
      for (int it = 0; it < CPL; ++it) {
#if !MOT_SUM_BULK_RED
        const int id = __shfl_sync(kFull, idreg, slot[it]);
#endif
        float dz[CW];
#pragma unroll
        for (int e = 0; e < CW; ++e) {
          dz[e] = r * g[it][e] - c * o[it][e];
          Du[it][e] += dz[e];
        }
#if MOT_SUM_BULK_RED
        *reinterpret_cast<float4*>(dzrow + (it * 32 + lane) * CW) = make_float4(dz[0], dz[1], dz[2], dz[3]);
#else
        MOT_ASSERT(id >= 0 && id < p.Vb, "byte id", id, p.Vb);
        gmem_add4(reinterpret_cast<float*>(accp + ((unsigned)id * bd4 + boff4[it])), dz);
#endif
      }
#if MOT_SUM_BULK_RED
      // generic-proxy writes of dz -> visible to the async proxy, then one bulk reduction per byte slot (lane = slot)
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if (id_lane) {
        MOT_ASSERT(idreg >= 0 && idreg < p.Vb, "byte id", idreg, p.Vb);
#ifndef MOT_EXPERIMENT_NO_RED
        asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f32 [%0], [%1], %2;" ::"l"(accp + (unsigned)idreg * bd4),
                     "r"(dz_s + (unsigned)lane * bd4), "r"(bd4)
                     : "memory");
#endif
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        // every group but the one just committed has finished READING its stage: the previous occurrence's stage is free
        asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
      }
      __syncwarp();
      if (red_pending) {
        --inflight;
        try_issue();
      }
      red_pending = true;
#endif
#endif
    }
    if (A.flags & 2) {  // end of the chunk: close the open row segment
      if (cur_v >= 0) flush(seg_lead || A.v_next == cur_v);
      cur_v = -1;
      seg_lead = false;
    }
    // advance: A <- B, prefetch the batch after
    A = B;
    if (iw == 1) iw = 0; else ik = 0;
    load_next(B, true);
    while (inflight < D && try_issue()) {  // the issue cursor may have been waiting for this batch
    }
  }
  MOT_STAMP(p.trace, gw, 61);

  // ---- phase Z (after the stream): rows nobody gathered get zeros (the dense-grad contract of the reference).  Blocks of
  //      32 vocabulary rows are handed out by a global counter, so the warps that finish their stream first take the
  //      zero fill (13 % of the kernel's HBM traffic at 48K tokens) while the slower ones are still streaming: the fill is
  //      the load balancer of the kernel instead of a serial prologue in front of the first row copy.  The finalize
  //      kernel resets the counter (self-cleaning workspace).
#ifndef MOT_X_SUM_NO_ZERO
  {
    const float zero[CW] = {0.f, 0.f, 0.f, 0.f};
    int* zctr = reinterpret_cast<int*>(p.lam_acc) + 2;
    const int n_blocks = (p.v_hi - p.v_lo + 31) >> 5;
    auto grab = [&]() -> int {
      int b = 0;
      if (lane == 0) b = atomicAdd(zctr, 1);
      return __shfl_sync(kFull, b, 0);
    };
    int nb = grab();
    while (nb < n_blocks) {
      const int vb = p.v_lo + (nb << 5);
      const int v = vb + lane;
      const bool empty = v < p.v_hi && (ld_g(p.off + v + 1) - ld_g(p.off + v)) == 0;
      nb = grab();  // the next block's ticket travels while this block is written
      unsigned m = __ballot_sync(kFull, empty);
      while (m) {
        const int j = __ffs(m) - 1;
        m &= m - 1;
        MOT_ASSERT(vb + j >= p.v_lo && vb + j < p.v_hi, "zero row", vb + j, p.v_hi);
        T* row = G + (size_t)(unsigned)(vb + j) * (unsigned)p.Dt;
#pragma unroll
        for (int it = 0; it < CPL; ++it) V::stg(row + (it * 32 + lane) * CW, zero);
      }
    }
  }
#endif
  MOT_STAMP(p.trace, gw, 62);
#if MOT_SUM_BULK_RED && !MOT_SUM_TWO_PASS
  // the bulk reductions drained beside the zero fill; they must be complete (and the ring intact) when the thread exits
  if (id_lane) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
#endif
#ifdef MOT_TRACE
  if (p.trace != nullptr && lane == 0) p.trace[(size_t)gw * 64 + 63] = n_occ;
#endif
}

template <typename T, int CPL, int PULL = kNoPull>
static int launch_bwd_sum(const EmbedParams& p_in, cudaStream_t s) {
  if constexpr (PULL == kNoPull) {
    if (const int k = ids_pulled(p_in))
      return k == kPullLeft ? launch_bwd_sum<T, CPL, kPullLeft>(p_in, s) : launch_bwd_sum<T, CPL, kPullRight>(p_in, s);
  }
  int sms = 0, optin = 0;
  if (int rc = device_props(&sms, &optin)) return rc;
  EmbedParams p = p_in;
  static const char* env_st = getenv("MOT_SUM_STAGES");  // debug knob
  int want = env_st ? atoi(env_st) : 4;
  if (want < 2) want = 2;
  size_t smem = 0;
  for (int st = want; st >= 2; --st) {
    const SumSmem L = sum_smem(p.Do, sizeof(T), kSumThreads / 32, st);
    if (L.total + 1024 <= (size_t)optin) {
      p.stages = st;
      smem = L.total;
      break;
    }
  }
  if (smem == 0) return MOT_ERR_UNSUPPORTED;
  p.trace = g_trace ? g_trace + 4096 * 64 : nullptr;
  auto kern = mot_bwd_sum_kernel<T, CPL, PULL>;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return check_launch();
  if (g_prof_start) cudaEventRecord(g_prof_start, s);
  const int ctas = (p.grid_cap > 0 && p.grid_cap < sms) ? p.grid_cap : sms;
  launch_pdl(kern, dim3((unsigned)ctas), dim3(kSumThreads), smem, s, p);
  if (g_prof_stop) cudaEventRecord(g_prof_stop, s);
  count_launch();
  return check_launch();
}

// The saved-output kernel applies to the MoT-sum fast path (pick_mode == 1) when the caller kept out and rstd.
inline bool sum_path_ok(const EmbedParams& p) {
  return p.out_saved != nullptr && p.rstd != nullptr && pick_mode(p, kBwdCW) == 1 && p.io_ld == p.Do && p.io_col == 0 &&
         !(p.flags & MOT_F_IDS_FROM_TTB && p.ttb == nullptr);
}

}  // namespace mot
