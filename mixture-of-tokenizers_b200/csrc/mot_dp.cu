// The one exchange step of the path: average the dense gradients of the replicated tables across the data-parallel
// ranks (reference: one dist.all_reduce(param.grad, AVG) per parameter, spt/train_gpt.py:1320-1321, runs/7:697-700;
// the runs launch them asynchronously and wait per optimizer, runs/7:697-711).
//
// The flat gradient bucket the backward kernels write lives in symmetric memory: every rank can address every rank's
// copy (peer pointers over NVLink 5 / NVSwitch) and, where the switch offers it, all copies through ONE multicast
// address (NVLS).  The exchange works on byte RANGES of the bucket so that it can run slab by slab beside the
// backward (mot_embed_bwd_slab): range k is exchanged on a second stream while the backward of slab k + 1 runs.
//
// One kernel per rank and range, two-shot: rank r owns sub-slice r of the range,
//   barrier   (signal pads, release / acquire at system scope): every rank's backward has written the range
//   NVLS    : multimem.ld_reduce pulls the sub-slice from ALL copies, summed inside the switch with fp32 accumulation;
//             scale by 1 / world; multimem.st pushes the averaged values back to ALL copies.  Per GPU and direction
//             about (1 + 1/world) range sizes cross NVLink, independent of the number of ranks.
//   P2P     : the sub-slice is read from every rank's copy through the peer pointers (rank order: one fixed fp32
//             summation order, the same value everywhere), averaged, and written to every copy.  2 (world-1)/world
//             range sizes per direction: less than NVLS's (1 + 1/world) at 2 ranks, the same at ... never again, so
//             the library picks P2P at 2 ranks, NVLS from 4 on (measured: profiles/r2_dp.md).
//   barrier   only after the LAST range of a step: the ranges of one step touch disjoint addresses, and a rank's next
//             step cannot write the bucket before its own last exchange kernel has passed that barrier.
#include <cstdlib>

#include "mot_common.cuh"

namespace mot {

constexpr int kArThreads = 1024;
constexpr int kArMaxBlocksNvls = 8;   // measured best for the in-switch reduction (8 ranks: 8 CTAs 195 us, 36 CTAs 219 us)
constexpr int kArMaxBlocksP2p = 32;   // 512-thread CTAs (up to 64 data registers per thread in flight)
constexpr int kPadSlots = 9216 / 4;   // torch's signal pad: 9216 bytes of uint32 slots

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// Block b of every rank meets block b of every other rank: lane r tells rank r "rank `rank` reached `target`", then
// waits until rank r said the same.  The slots only grow (signed-difference compare: wrap safe), so nothing is ever
// reset, and a block that did not take part in an earlier, smaller launch simply jumps to the current target.
__device__ __forceinline__ void rank_barrier(uint32_t* const* pads, int rank, int world, uint32_t target) {
  __syncthreads();
  if ((int)threadIdx.x < world) {
    __threadfence_system();
    st_release_sys(pads[threadIdx.x] + blockIdx.x * world + rank, target);
    const uint32_t* mine = pads[rank] + blockIdx.x * world + threadIdx.x;
    while ((int32_t)(ld_acquire_sys(mine) - target) < 0) {
    }
  }
  __syncthreads();
}

__device__ __forceinline__ void scale_vec(uint32_t (&r)[4], float inv, bool bf16) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (bf16) {
      float lo_f, hi_f;
      bf16x2_to_f32(r[j], lo_f, hi_f);
      r[j] = f32x2_to_bf16x2(lo_f * inv, hi_f * inv);
    } else {
      r[j] = __float_as_uint(__uint_as_float(r[j]) * inv);
    }
  }
}

template <bool BF16, int kUnroll>
__global__ void __launch_bounds__(kUnroll > 8 ? 512 : 1024) nvls_allreduce_avg_kernel(char* mc, uint32_t* const* pads, int rank, int world,
                                                                        long long vec_lo, long long n_vec /* 16-byte vectors */,
                                                                        uint32_t epoch, int last, unsigned* work, long long* trace) {
  pdl_launch_dependents();
  MOT_STAMP(trace, blockIdx.x, 0);
  pdl_wait();  // the local backward / finalize kernels of this range have completed: this rank's copy is final
  MOT_STAMP(trace, blockIdx.x, 1);
  if (blockIdx.x == 0 && threadIdx.x == 0) work[(epoch + 1u) & 63u] = work[(epoch + 2u) & 63u] = 0u;
  work += epoch & 63u;
  rank_barrier(pads, rank, world, epoch);
  MOT_STAMP(trace, blockIdx.x, 2);
  const long long per = (n_vec + world - 1) / world;
  const long long lo = vec_lo + per * rank, hi = min(lo + per, vec_lo + n_vec);
  const float inv = 1.f / (float)world;
  // The sub-slice is handed out in tiles of blockDim x kUnroll vectors by a counter (work[0], zeroed by the launch): the
  // CTAs do not run at the same speed (8 ranks, 77 MB, static split: the first CTA finishes at 122 us, the last at 161 us;
  // profiles/r2_dp.md) and the slowest one sets the exit barrier.  kUnroll independent 16-byte reductions are in flight per
  // thread: one switch round trip is microseconds, the link wants megabytes outstanding.
  __shared__ long long tile_s[2];
  const long long tile_vecs = (long long)blockDim.x * kUnroll;
  if (threadIdx.x == 0) tile_s[0] = (long long)atomicAdd(work, 1u);
  __syncthreads();
  for (int it = 0;; ++it) {
    const long long base = lo + tile_s[it & 1] * tile_vecs;
    if (base >= hi) break;
    if (threadIdx.x == 0) tile_s[(it + 1) & 1] = (long long)atomicAdd(work, 1u);  // the next ticket travels while this tile moves
    const long long i0 = base + threadIdx.x;
    uint32_t r[kUnroll][4];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const long long i = i0 + (long long)u * blockDim.x;
      if (i < hi) {
        char* a = mc + i * 16;
        if (BF16)
          asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.v4.bf16x2 {%0,%1,%2,%3}, [%4];"
                       : "=r"(r[u][0]), "=r"(r[u][1]), "=r"(r[u][2]), "=r"(r[u][3]) : "l"(a) : "memory");
        else
          asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
                       : "=r"(r[u][0]), "=r"(r[u][1]), "=r"(r[u][2]), "=r"(r[u][3]) : "l"(a) : "memory");
      }
    }
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const long long i = i0 + (long long)u * blockDim.x;
      if (i < hi) {
        scale_vec(r[u], inv, BF16);
        asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(mc + i * 16), "r"(r[u][0]), "r"(r[u][1]),
                     "r"(r[u][2]), "r"(r[u][3])
                     : "memory");
      }
    }
    __syncthreads();
  }
  MOT_STAMP(trace, blockIdx.x, 3);
  if (last) rank_barrier(pads, rank, world, epoch + 1u);
  MOT_STAMP(trace, blockIdx.x, 4);
}

__device__ __forceinline__ void ld_sys_16(const char* p, uint32_t (&r)[4]) {
  asm volatile("ld.relaxed.sys.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "l"(p) : "memory");
}
__device__ __forceinline__ void st_sys_16(char* p, const uint32_t (&r)[4]) {
  asm volatile("st.relaxed.sys.global.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]) : "memory");
}

// Peer-to-peer two-shot: WORLD copies are read and written through the peer pointers.  kUnroll x WORLD 16-byte loads in
// flight per thread (an NVLink round trip is about 2 us: a rank needs megabytes outstanding to fill 900 GB/s).
template <bool BF16, int WORLD, int kUnroll>
__global__ void __launch_bounds__(512) p2p_allreduce_avg_kernel(char* const* peers, uint32_t* const* pads, int rank,
                                                                       long long vec_lo, long long n_vec, uint32_t epoch, int last,
                                                                       unsigned* work, long long* trace) {
  pdl_launch_dependents();
  MOT_STAMP(trace, blockIdx.x, 0);
  pdl_wait();
  MOT_STAMP(trace, blockIdx.x, 1);
  if (blockIdx.x == 0 && threadIdx.x == 0) work[(epoch + 1u) & 63u] = work[(epoch + 2u) & 63u] = 0u;
  work += epoch & 63u;
  rank_barrier(pads, rank, WORLD, epoch);
  MOT_STAMP(trace, blockIdx.x, 2);
  char* P[WORLD];
#pragma unroll
  for (int q = 0; q < WORLD; ++q) P[q] = peers[q];
  const long long per = (n_vec + WORLD - 1) / WORLD;
  const long long lo = vec_lo + per * rank, hi = min(lo + per, vec_lo + n_vec);
  const float inv = 1.f / (float)WORLD;
  __shared__ long long tile_s[2];
  const long long tile_vecs = (long long)blockDim.x * kUnroll;
  if (threadIdx.x == 0) tile_s[0] = (long long)atomicAdd(work, 1u);
  __syncthreads();
  for (int it = 0;; ++it) {  // tiles handed out by a counter, like the NVLS kernel
    const long long base = lo + tile_s[it & 1] * tile_vecs;
    if (base >= hi) break;
    if (threadIdx.x == 0) tile_s[(it + 1) & 1] = (long long)atomicAdd(work, 1u);
    const long long i0 = base + threadIdx.x;
    uint32_t v[kUnroll][WORLD][4];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const long long i = i0 + (long long)u * blockDim.x;
      if (i < hi) {
#pragma unroll
        for (int q = 0; q < WORLD; ++q) ld_sys_16(P[q] + i * 16, v[u][q]);
      }
    }
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const long long i = i0 + (long long)u * blockDim.x;
      if (i < hi) {
        uint32_t r[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (BF16) {  // fp32 accumulation in rank order 0 .. WORLD-1: the same value on every rank, run to run
            float a = 0.f, b = 0.f;
#pragma unroll
            for (int q = 0; q < WORLD; ++q) {
              float lo_f, hi_f;
              bf16x2_to_f32(v[u][q][j], lo_f, hi_f);
              a += lo_f;
              b += hi_f;
            }
            r[j] = f32x2_to_bf16x2(a * inv, b * inv);
          } else {
            float a = 0.f;
#pragma unroll
            for (int q = 0; q < WORLD; ++q) a += __uint_as_float(v[u][q][j]);
            r[j] = __float_as_uint(a * inv);
          }
        }
#pragma unroll
        for (int q = 0; q < WORLD; ++q) st_sys_16(P[q] + i * 16, r);
      }
    }
    __syncthreads();
  }
  MOT_STAMP(trace, blockIdx.x, 3);
  if (last) rank_barrier(pads, rank, WORLD, epoch + 1u);
  MOT_STAMP(trace, blockIdx.x, 4);
}

template <bool BF16, int WORLD>
static void launch_p2p(int unroll, dim3 g, dim3 b, cudaStream_t s, char* const* peers, uint32_t* const* pads, int rank,
                       long long vec_lo, long long n_vec, uint32_t epoch, int last, unsigned* work, long long* trace) {
  if (unroll >= 4 && WORLD <= 4)
    launch_pdl(p2p_allreduce_avg_kernel<BF16, WORLD, 4>, g, b, 0, s, peers, pads, rank, vec_lo, n_vec, epoch, last, work, trace);
  else if (unroll >= 2 && WORLD <= 8)
    launch_pdl(p2p_allreduce_avg_kernel<BF16, WORLD, 2>, g, b, 0, s, peers, pads, rank, vec_lo, n_vec, epoch, last, work, trace);
  else
    launch_pdl(p2p_allreduce_avg_kernel<BF16, WORLD, 1>, g, b, 0, s, peers, pads, rank, vec_lo, n_vec, epoch, last, work, trace);
}


// ---- touched-rows exchange ------------------------------------------------------------------------------------------
// The dense token gradient has a row of zeros for every token the rank's batch did not contain, and a row that is zero on
// EVERY rank needs no exchange at all: it is already correct everywhere.  Each rank publishes a bitmap of the rows its
// backward gathered (mot_embed_touched_rows, from the sort plan) next to the bucket; the exchange ORs the bitmaps through
// the same fabric (multimem.ld_reduce.or / peer loads) and moves only the rows of the union.  Uniform synthetic ids at 48K
// tokens touch 62 % of the vocabulary per rank (union 86 % at 2 ranks, ~100 % from 4 ranks on: no gain there); Zipf /
// real text touches 20-30 % per rank.  Work unit: 64 rows (two bitmap words), handed out by the tile counter; a warp owns a
// row, its lanes the row's 16-byte vectors.
//
// Several tables indexed by the same token ids (the front's token table and the value embeddings, runs/7:252,308) share
// one bitmap: row v of every table is touched exactly when token v was gathered.  A warp moves row v of ALL tables, one
// table after the other, with the same rows in flight.
constexpr int kRowsPerTile = 64;
constexpr int kMaxVecPerLane = 4;  // rows up to 32 x 4 x 16 = 2048 bytes in one trip; wider rows loop
constexpr int kMaxRowWords = 2048; // bitmap words of one rank's rows held in shared memory (65536 rows per rank)

struct RowTables {                          // a kernel parameter: no device array, no copy
  long long vec_off[MOT_DP_MAX_ROW_TABLES];  // bucket vector (16 bytes) of row 0 of table t
  int row_vecs[MOT_DP_MAX_ROW_TABLES];       // vectors per row of table t
  int n;
};

// Table t of the parameter struct, selected with compile-time indices (a run-time index would copy the struct to local
// memory).  NT = the compile-time bound of the table count: NT = 1 is the one-table exchange, compiled to the code
// (addresses, summation order, registers) of the single-table kernel it replaced.
template <int NT>
__device__ __forceinline__ void row_table(const RowTables& T, int t, long long& vec_off, int& row_vecs) {
  vec_off = T.vec_off[0];
  row_vecs = T.row_vecs[0];
#pragma unroll
  for (int k = 1; k < NT; ++k)
    if (k == t) {
      vec_off = T.vec_off[k];
      row_vecs = T.row_vecs[k];
    }
}

template <bool BF16, bool NVLS, int WORLD, int NT>
__global__ void __launch_bounds__(NVLS ? 1024 : 512) rows_allreduce_avg_kernel(char* mc, char* const* peers, uint32_t* const* pads, int rank, int world,
                                                                 const RowTables T, int n_rows, long long bm_off,
                                                                 long long dense_vec_lo, long long dense_vecs, uint32_t epoch,
                                                                 unsigned* work, int peer_bits, long long* trace) {
  pdl_launch_dependents();
  MOT_STAMP(trace, blockIdx.x, 0);
  pdl_wait();
  MOT_STAMP(trace, blockIdx.x, 1);
  if (blockIdx.x == 0 && threadIdx.x == 0) work[(epoch + 1u) & 63u] = work[(epoch + 2u) & 63u] = 0u;
  work += epoch & 63u;
  rank_barrier(pads, rank, world, epoch);
  MOT_STAMP(trace, blockIdx.x, 2);
  char* P[WORLD];
  if (!NVLS) {
#pragma unroll
    for (int q = 0; q < WORLD; ++q) P[q] = peers[q];
  }
  const float inv = 1.f / (float)world;
  // rows of this rank: a multiple of 32 per rank, so that a bitmap word belongs to one rank
  const int per = ((n_rows + world - 1) / world + 31) / 32 * 32;
  const int r_lo = min(per * rank, n_rows), r_hi = min(r_lo + per, n_rows);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __shared__ long long tile_s[2];
  __shared__ uint32_t bits_all[kMaxRowWords];   // union bitmap of this rank's rows, fetched once (one fabric round trip)
  // peer-to-peer: the bitmap of every rank as well.  A row a rank did not gather is a row of zeros in that rank's copy (the
  // dense-gradient contract of the backward), so it is not read at all: the pull phase moves the rows each PEER gathered
  // (62 % of the table per rank for uniform ids at 48K tokens), the push phase the rows of the union (86 % at 2 ranks).
  __shared__ uint32_t bits_rank[NVLS ? 1 : WORLD][NVLS ? 1 : kMaxRowWords];
  auto or_word = [&](int w_local, int w) -> uint32_t {  // union over the ranks of bitmap word w
    uint32_t v = 0;
    if (NVLS) {
      asm volatile("multimem.ld_reduce.relaxed.sys.global.or.b32 %0, [%1];" : "=r"(v) : "l"(mc + bm_off + (long long)w * 4) : "memory");
    } else {
#pragma unroll
      for (int q = 0; q < WORLD; ++q) {
        uint32_t x;
        asm volatile("ld.relaxed.sys.global.b32 %0, [%1];" : "=r"(x) : "l"(P[q] + bm_off + (long long)w * 4) : "memory");
        bits_rank[q][w_local] = peer_bits ? x : 0xffffffffu;
        v |= x;
      }
    }
    return v;
  };
  if (threadIdx.x == 0) tile_s[0] = (long long)atomicAdd(work, 1u);
  for (int w = threadIdx.x; w < (r_hi - r_lo + 31) / 32; w += blockDim.x) bits_all[w] = or_word(w, (r_lo >> 5) + w);
  __syncthreads();
  for (int it = 0;; ++it) {
    const long long row0 = (long long)r_lo + tile_s[it & 1] * kRowsPerTile;
    if (row0 >= r_hi) break;
    if (threadIdx.x == 0) tile_s[(it + 1) & 1] = (long long)atomicAdd(work, 1u);
    const uint32_t* bits_t = bits_all + ((row0 - r_lo) >> 5);
    // a warp owns rows warp, warp + nw, ... of the tile; RPW of them are in flight together: every load of those rows is
    // issued before the first value is used (an NVLink round trip is ~2 us; with one row at a time the peer-to-peer
    // version ran at 250 GB/s)
    constexpr int RPW = NVLS ? 2 : (WORLD <= 2 ? 2 : 1);
    for (int rr0 = warp; rr0 < kRowsPerTile; rr0 += nw * RPW) {
      long long rows[RPW];
      bool act[RPW];
      uint32_t has[RPW];  // peer-to-peer: bit q = rank q gathered the row (its copy is read), else its copy is zeros
#pragma unroll
      for (int q2 = 0; q2 < RPW; ++q2) {
        const int rr = rr0 + q2 * nw;
        const long long row = row0 + rr;
        act[q2] = rr < kRowsPerTile && row < r_hi && ((bits_t[rr >> 5] >> (rr & 31)) & 1u);
        rows[q2] = row;
        has[q2] = 0u;
        if (!NVLS && act[q2]) {
          const int wl = (int)((row0 - r_lo) >> 5) + (rr >> 5);
#pragma unroll
          for (int q = 0; q < WORLD; ++q) has[q2] |= ((bits_rank[q][wl] >> (rr & 31)) & 1u) << q;
        }
      }
      for (int t = 0; t < (NT == 1 ? 1 : T.n); ++t) {
        long long vec_off;
        int row_vecs;
        row_table<NT>(T, t, vec_off, row_vecs);
        long long vrow[RPW];
  #pragma unroll
        for (int q2 = 0; q2 < RPW; ++q2) vrow[q2] = vec_off + rows[q2] * row_vecs;
        for (int j0 = 0; j0 < row_vecs; j0 += 32 * kMaxVecPerLane) {
          if (NVLS) {
            uint32_t r[RPW][kMaxVecPerLane][4];
  #pragma unroll
            for (int q2 = 0; q2 < RPW; ++q2)
  #pragma unroll
              for (int u = 0; u < kMaxVecPerLane; ++u) {
                const int j = j0 + u * 32 + lane;
                if (act[q2] && j < row_vecs) {
                  char* a = mc + (vrow[q2] + j) * 16;
                  if (BF16)
                    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.v4.bf16x2 {%0,%1,%2,%3}, [%4];"
                                 : "=r"(r[q2][u][0]), "=r"(r[q2][u][1]), "=r"(r[q2][u][2]), "=r"(r[q2][u][3]) : "l"(a) : "memory");
                  else
                    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
                                 : "=r"(r[q2][u][0]), "=r"(r[q2][u][1]), "=r"(r[q2][u][2]), "=r"(r[q2][u][3]) : "l"(a) : "memory");
                }
              }
  #pragma unroll
            for (int q2 = 0; q2 < RPW; ++q2)
  #pragma unroll
              for (int u = 0; u < kMaxVecPerLane; ++u) {
                const int j = j0 + u * 32 + lane;
                if (act[q2] && j < row_vecs) {
                  scale_vec(r[q2][u], inv, BF16);
                  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(mc + (vrow[q2] + j) * 16),
                               "r"(r[q2][u][0]), "r"(r[q2][u][1]), "r"(r[q2][u][2]), "r"(r[q2][u][3]) : "memory");
                }
              }
          } else {
            uint32_t v[RPW][kMaxVecPerLane][WORLD][4];
  #pragma unroll
            for (int q2 = 0; q2 < RPW; ++q2)
  #pragma unroll
              for (int u = 0; u < kMaxVecPerLane; ++u) {
                const int j = j0 + u * 32 + lane;
                if (act[q2] && j < row_vecs) {
  #pragma unroll
                  for (int q = 0; q < WORLD; ++q) {
                    if ((has[q2] >> q) & 1u) {
                      ld_sys_16(P[q] + (vrow[q2] + j) * 16, v[q2][u][q]);
                    } else {
                      v[q2][u][q][0] = v[q2][u][q][1] = v[q2][u][q][2] = v[q2][u][q][3] = 0u;  // +0.0 in bf16x2 and fp32 alike
                    }
                  }
                }
              }
  #pragma unroll
            for (int q2 = 0; q2 < RPW; ++q2)
  #pragma unroll
              for (int u = 0; u < kMaxVecPerLane; ++u) {
                const int j = j0 + u * 32 + lane;
                if (act[q2] && j < row_vecs) {
                  uint32_t r[4];
  #pragma unroll
                  for (int k = 0; k < 4; ++k) {
                    if (BF16) {
                      float a = 0.f, b = 0.f;
  #pragma unroll
                      for (int q = 0; q < WORLD; ++q) {
                        float lo_f, hi_f;
                        bf16x2_to_f32(v[q2][u][q][k], lo_f, hi_f);
                        a += lo_f;
                        b += hi_f;
                      }
                      r[k] = f32x2_to_bf16x2(a * inv, b * inv);
                    } else {
                      float a = 0.f;
  #pragma unroll
                      for (int q = 0; q < WORLD; ++q) a += __uint_as_float(v[q2][u][q][k]);
                      r[k] = __float_as_uint(a * inv);
                    }
                  }
  #pragma unroll
                  for (int q = 0; q < WORLD; ++q) st_sys_16(P[q] + (vrow[q2] + j) * 16, r);
                }
              }
          }
        }
      }
    }
    __syncthreads();
  }
  // the rest of the bucket (byte table, anything else): dense, this rank's share, a static stride loop (it is small)
  {
    const long long dper = (dense_vecs + world - 1) / world;
    const long long lo = dense_vec_lo + dper * rank, hi = min(lo + dper, dense_vec_lo + dense_vecs);
    for (long long i = lo + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += (long long)gridDim.x * blockDim.x) {
      uint32_t r[4];
      if (NVLS) {
        if (BF16)
          asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.v4.bf16x2 {%0,%1,%2,%3}, [%4];"
                       : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "l"(mc + i * 16) : "memory");
        else
          asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
                       : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "l"(mc + i * 16) : "memory");
        scale_vec(r, inv, BF16);
        asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(mc + i * 16), "r"(r[0]), "r"(r[1]), "r"(r[2]),
                     "r"(r[3]) : "memory");
      } else {
        uint32_t v[WORLD][4];
#pragma unroll
        for (int q = 0; q < WORLD; ++q) ld_sys_16(P[q] + i * 16, v[q]);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          if (BF16) {
            float a = 0.f, b = 0.f;
#pragma unroll
            for (int q = 0; q < WORLD; ++q) {
              float lo_f, hi_f;
              bf16x2_to_f32(v[q][k], lo_f, hi_f);
              a += lo_f;
              b += hi_f;
            }
            r[k] = f32x2_to_bf16x2(a * inv, b * inv);
          } else {
            float a = 0.f;
#pragma unroll
            for (int q = 0; q < WORLD; ++q) a += __uint_as_float(v[q][k]);
            r[k] = __float_as_uint(a * inv);
          }
        }
#pragma unroll
        for (int q = 0; q < WORLD; ++q) st_sys_16(P[q] + i * 16, r);
      }
    }
  }
  MOT_STAMP(trace, blockIdx.x, 3);
  rank_barrier(pads, rank, world, epoch + 1u);
  MOT_STAMP(trace, blockIdx.x, 4);
}

}  // namespace mot

using namespace mot;

extern "C" int mot_dp_exchange(void* multicast_ptr, void* const* peer_ptrs_dev, void* const* signal_pads_dev, void* work_area,
                               int32_t rank, int32_t world, int64_t byte_offset, int64_t n_bytes, int32_t dtype, uint32_t epoch,
                               int32_t last, int32_t algo, void* stream) {
  if (!signal_pads_dev || !work_area || world < 1 || rank < 0 || rank >= world || n_bytes < 0 || byte_offset < 0) return MOT_ERR_BAD_ARG;
  if (dtype != MOT_BF16 && dtype != MOT_F32) return MOT_ERR_UNSUPPORTED;
  if (algo == MOT_DP_NVLS && !multicast_ptr) return MOT_ERR_BAD_ARG;
  if (algo == MOT_DP_P2P && !peer_ptrs_dev) return MOT_ERR_BAD_ARG;
  if (algo != MOT_DP_NVLS && algo != MOT_DP_P2P) return MOT_ERR_UNSUPPORTED;
  if (algo == MOT_DP_P2P && world != 2 && world != 4 && world != 8) return MOT_ERR_UNSUPPORTED;
  if ((reinterpret_cast<uintptr_t>(multicast_ptr) & 15u) || (n_bytes & 15) || (byte_offset & 15)) return MOT_ERR_MISALIGNED;
  if (world > 16) return MOT_ERR_UNSUPPORTED;
  if (n_bytes == 0 && !last) return MOT_OK;
  int sms = 0, optin = 0;
  if (int rc = device_props(&sms, &optin)) return rc;
  const long long n_vec = n_bytes / 16, vec_lo = byte_offset / 16;
  const char* env_b = getenv("MOT_AR_BLOCKS");    // debug knobs, read per call so that one process can sweep them
  const char* env_t = getenv("MOT_AR_THREADS");
  const char* env_u = getenv("MOT_AR_UNROLL");
  int threads = env_t ? atoi(env_t) : kArThreads;
  if (threads < 32 || threads > 1024 || threads % 32) threads = kArThreads;
  const int unroll = env_u ? atoi(env_u) : (algo == MOT_DP_NVLS ? 8 : 4);
  if (threads > 512 && (algo == MOT_DP_P2P || unroll > 8)) threads = 512;   // those kernels are compiled for 512 threads
  long long max_blocks = env_b ? atoi(env_b) : (algo == MOT_DP_NVLS ? kArMaxBlocksNvls : kArMaxBlocksP2p);
  if (max_blocks < 1) max_blocks = 1;
  if (max_blocks * world > kPadSlots) max_blocks = kPadSlots / world;   // signal-pad slots: blocks x world uint32
  long long blocks = (n_vec / world + threads * 4 - 1) / (threads * 4);
  if (blocks > max_blocks) blocks = max_blocks;
  if (blocks < 1) blocks = 1;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  uint32_t* const* pads = reinterpret_cast<uint32_t* const*>(signal_pads_dev);
  const dim3 g((unsigned)blocks), b(threads);
  const bool bf = dtype == MOT_BF16;
  const int lastf = last ? 1 : 0;
  // MOT_TRACE builds: block stamps of consecutive exchange launches go to consecutive 64-block regions behind the
  // forward / backward / finalize regions of the trace buffer
  // tile counter of this launch: word (epoch mod 64) of the caller's zero-initialised work area; every launch zeroes the
  // two words its successors may use (epoch + 1, epoch + 2), so no memset sits between the kernels of the stream
  unsigned* work = reinterpret_cast<unsigned*>(work_area);
  static int trace_seq = 0;
  long long* trace = g_trace ? g_trace + (3 * 4096 + (size_t)(trace_seq++ % 16) * 64) * 64 : nullptr;
  if (algo == MOT_DP_NVLS) {
    char* mc = reinterpret_cast<char*>(multicast_ptr);
    if (bf) {
      if (unroll == 4) launch_pdl(nvls_allreduce_avg_kernel<true, 4>, g, b, 0, s, mc, pads, (int)rank, (int)world, vec_lo, n_vec, epoch, lastf, work, trace);
      else if (unroll == 16) launch_pdl(nvls_allreduce_avg_kernel<true, 16>, g, b, 0, s, mc, pads, (int)rank, (int)world, vec_lo, n_vec, epoch, lastf, work, trace);
      else launch_pdl(nvls_allreduce_avg_kernel<true, 8>, g, b, 0, s, mc, pads, (int)rank, (int)world, vec_lo, n_vec, epoch, lastf, work, trace);
    } else {
      if (unroll == 4) launch_pdl(nvls_allreduce_avg_kernel<false, 4>, g, b, 0, s, mc, pads, (int)rank, (int)world, vec_lo, n_vec, epoch, lastf, work, trace);
      else launch_pdl(nvls_allreduce_avg_kernel<false, 8>, g, b, 0, s, mc, pads, (int)rank, (int)world, vec_lo, n_vec, epoch, lastf, work, trace);
    }
  } else {
    char* const* peers = reinterpret_cast<char* const*>(peer_ptrs_dev);
    if (world == 2) {
      if (bf) launch_p2p<true, 2>(unroll, g, b, s, peers, pads, rank, vec_lo, n_vec, epoch, lastf, work, trace);
      else launch_p2p<false, 2>(unroll, g, b, s, peers, pads, rank, vec_lo, n_vec, epoch, lastf, work, trace);
    } else if (world == 4) {
      if (bf) launch_p2p<true, 4>(unroll, g, b, s, peers, pads, rank, vec_lo, n_vec, epoch, lastf, work, trace);
      else launch_p2p<false, 4>(unroll, g, b, s, peers, pads, rank, vec_lo, n_vec, epoch, lastf, work, trace);
    } else {
      if (bf) launch_p2p<true, 8>(unroll, g, b, s, peers, pads, rank, vec_lo, n_vec, epoch, lastf, work, trace);
      else launch_p2p<false, 8>(unroll, g, b, s, peers, pads, rank, vec_lo, n_vec, epoch, lastf, work, trace);
    }
  }
  count_launch();
  return check_launch();
}

// The whole bucket in one call (round-1 entry point): one range, both barriers.  `epoch` grows by TWO per call.
extern "C" int mot_dp_allreduce_avg(void* multicast_ptr, void* const* signal_pads_dev, void* work_area, int32_t rank, int32_t world,
                                    int64_t n_bytes, int32_t dtype, uint32_t epoch, void* stream) {
  if (!multicast_ptr) return MOT_ERR_BAD_ARG;
  return mot_dp_exchange(multicast_ptr, nullptr, signal_pads_dev, work_area, rank, world, 0, n_bytes, dtype, epoch, 1, MOT_DP_NVLS,
                         stream);
}

static bool ranges_overlap(long long a_lo, long long a_n, long long b_lo, long long b_n) {
  return a_n > 0 && b_n > 0 && a_lo < b_lo + b_n && b_lo < a_lo + a_n;
}

extern "C" int mot_dp_exchange_rows_multi(void* multicast_ptr, void* const* peer_ptrs_dev, void* const* signal_pads_dev,
                                          void* work_area, int32_t rank, int32_t world, const MotRowTable* tables,
                                          int32_t n_tables, int32_t n_rows, int64_t bitmap_byte_offset,
                                          int64_t dense_byte_offset, int64_t dense_bytes, int32_t dtype, uint32_t epoch,
                                          int32_t algo, void* stream) {
  if (!signal_pads_dev || !work_area || world < 1 || rank < 0 || rank >= world || n_rows < 0 || dense_bytes < 0)
    return MOT_ERR_BAD_ARG;
  if (!tables || n_tables < 1 || n_tables > MOT_DP_MAX_ROW_TABLES) return MOT_ERR_BAD_ARG;
  for (int t = 0; t < n_tables; ++t)
    if (tables[t].row_bytes <= 0 || tables[t].byte_offset < 0 || tables[t].reserved != 0) return MOT_ERR_BAD_ARG;
  if (bitmap_byte_offset < 0 || dense_byte_offset < 0) return MOT_ERR_BAD_ARG;
  if (dtype != MOT_BF16 && dtype != MOT_F32) return MOT_ERR_UNSUPPORTED;
  if (algo == MOT_DP_NVLS && !multicast_ptr) return MOT_ERR_BAD_ARG;
  if (algo == MOT_DP_P2P && !peer_ptrs_dev) return MOT_ERR_BAD_ARG;
  if (algo != MOT_DP_NVLS && algo != MOT_DP_P2P) return MOT_ERR_UNSUPPORTED;
  if (algo == MOT_DP_P2P && world != 2 && world != 4) return MOT_ERR_UNSUPPORTED;
  if (world > 16) return MOT_ERR_UNSUPPORTED;
  if (((n_rows + world - 1) / world + 31) / 32 + 1 > kMaxRowWords) return MOT_ERR_UNSUPPORTED;
  for (int t = 0; t < n_tables; ++t)
    if ((tables[t].row_bytes & 15) || (tables[t].byte_offset & 15)) return MOT_ERR_MISALIGNED;
  if ((bitmap_byte_offset & 3) || (dense_byte_offset & 15) || (dense_bytes & 15)) return MOT_ERR_MISALIGNED;
  // the kernel reads the bitmap and rewrites the tables and the dense range in place: no byte may belong to two of them
  const long long bm_bytes = ((long long)n_rows + 31) / 32 * 4;
  RowTables T{};
  T.n = n_tables;
  for (int t = 0; t < n_tables; ++t) {
    const long long lo = tables[t].byte_offset, nb = (long long)n_rows * tables[t].row_bytes;
    if (ranges_overlap(lo, nb, dense_byte_offset, dense_bytes) || ranges_overlap(lo, nb, bitmap_byte_offset, bm_bytes))
      return MOT_ERR_BAD_ARG;
    for (int u = 0; u < t; ++u)
      if (ranges_overlap(lo, nb, tables[u].byte_offset, (long long)n_rows * tables[u].row_bytes)) return MOT_ERR_BAD_ARG;
    T.vec_off[t] = lo / 16;
    T.row_vecs[t] = tables[t].row_bytes / 16;
  }
  if (ranges_overlap(bitmap_byte_offset, bm_bytes, dense_byte_offset, dense_bytes)) return MOT_ERR_BAD_ARG;
  int sms = 0, optin = 0;
  if (int rc = device_props(&sms, &optin)) return rc;
  const char* env_b = getenv("MOT_AR_BLOCKS");
  const char* env_pb = getenv("MOT_DP_PEER_BITS");   // debug knob: 0 = read every copy of a union row (round-2 behaviour)
  const int peer_bits = env_pb ? atoi(env_pb) : 1;
  long long blocks = env_b ? atoi(env_b) : (algo == MOT_DP_NVLS ? kArMaxBlocksNvls : kArMaxBlocksP2p);
  if (blocks < 1) blocks = 1;
  if (blocks * world > kPadSlots) blocks = kPadSlots / world;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  uint32_t* const* pads = reinterpret_cast<uint32_t* const*>(signal_pads_dev);
  unsigned* work = reinterpret_cast<unsigned*>(work_area);
  static int trace_seq = 0;
  long long* trace = g_trace ? g_trace + (3 * 4096 + (size_t)(trace_seq++ % 16) * 64) * 64 : nullptr;
  char* mc = reinterpret_cast<char*>(multicast_ptr);
  char* const* peers = reinterpret_cast<char* const*>(peer_ptrs_dev);
  const dim3 g((unsigned)blocks), b(algo == MOT_DP_NVLS ? 1024 : 512);
  const long long dlo = dense_byte_offset / 16, dn = dense_bytes / 16;
  const bool bf = dtype == MOT_BF16;
  // one table: the table loop compiled away (NT = 1); several: bounded by MOT_DP_MAX_ROW_TABLES, the count read at run time
#define MOT_ROWS_LAUNCH(BF, NV, WD, NT)                                                                                       \
  launch_pdl(rows_allreduce_avg_kernel<BF, NV, WD, NT>, g, b, 0, s, mc, peers, pads, (int)rank, (int)world, T, (int)n_rows,   \
             (long long)bitmap_byte_offset, dlo, dn, epoch, work, peer_bits, trace)
#define MOT_ROWS_LAUNCH_NT(BF, NV, WD) \
  do { if (n_tables == 1) MOT_ROWS_LAUNCH(BF, NV, WD, 1); else MOT_ROWS_LAUNCH(BF, NV, WD, MOT_DP_MAX_ROW_TABLES); } while (0)
  if (algo == MOT_DP_NVLS) {
    if (bf) MOT_ROWS_LAUNCH_NT(true, true, 1); else MOT_ROWS_LAUNCH_NT(false, true, 1);
  } else if (world == 2) {
    if (bf) MOT_ROWS_LAUNCH_NT(true, false, 2); else MOT_ROWS_LAUNCH_NT(false, false, 2);
  } else {
    if (bf) MOT_ROWS_LAUNCH_NT(true, false, 4); else MOT_ROWS_LAUNCH_NT(false, false, 4);
  }
#undef MOT_ROWS_LAUNCH_NT
#undef MOT_ROWS_LAUNCH
  count_launch();
  return check_launch();
}

extern "C" int mot_dp_exchange_rows(void* multicast_ptr, void* const* peer_ptrs_dev, void* const* signal_pads_dev, void* work_area,
                                    int32_t rank, int32_t world, int64_t table_byte_offset, int32_t n_rows, int32_t row_bytes,
                                    int64_t bitmap_byte_offset, int64_t dense_byte_offset, int64_t dense_bytes, int32_t dtype,
                                    uint32_t epoch, int32_t algo, void* stream) {
  const MotRowTable table = {table_byte_offset, row_bytes, 0};
  return mot_dp_exchange_rows_multi(multicast_ptr, peer_ptrs_dev, signal_pads_dev, work_area, rank, world, &table, 1, n_rows,
                                    bitmap_byte_offset, dense_byte_offset, dense_bytes, dtype, epoch, algo, stream);
}
