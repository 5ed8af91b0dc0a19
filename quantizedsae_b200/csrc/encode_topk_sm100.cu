// Fused encoder GEMM + per-row top-k candidate selection for sm_100a.
//
//   z[b, h] = sum_d x[b, d] * W[h, d] + bias[h]           (nn.Linear, sae/binary.py:82-84,92)
//   per row b keep the k largest z[b, :]                   (Tensor.topk,  sae/binary.py:94)
//
// One CTA owns BM = 128 rows of x (resident in shared memory for the whole sweep) and streams W
// through a TMA/mbarrier ring in tiles of BN = 256 latents x BK = 64. One thread issues
// tcgen05.mma (UMMA 128x256x16, bf16 in, fp32 accumulate) into one of two 256-column TMEM
// accumulators while eight epilogue warps drain the other with tcgen05.ld. The dense [B, H]
// pre-activation is never written.
//
// Selection in the epilogue. Thread (row, column-half) sees its row's values 32 columns at a
// time, column j of every chunk forming "class" j. It keeps in registers the running largest
// (or two largest) value of each class; with 32 classes x m values per class there are 32*m seen
// values >= T = min_j (m-th largest of class j), so T is a lower bound of the row's k-th largest
// for every k <= 32*m -- one FMNMX per element, no memory, no sorting. Values >= T (about 4k per
// row survive in total) are appended to a per-(row, sub-stream) buffer in global memory; stores
// are gated by a warp vote so they are only issued when a survivor exists. A buffer that runs
// full is filtered in place against the current T (bit-serial bisection to the exact k-th value
// is the fallback when filtering does not help, e.g. floods of equal values after ReLU).
// select_topk.cu merges the sub-streams of a row, sharpened by max_s T_s.
//
// The latent axis can be split over `n_splits` CTAs per row block (grid.x) to fill the 148 SMs
// at small batch; every (split, column-half) is an independent sub-stream.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include "kernels.h"
#include "ptx_sm100.cuh"
#include "tmap_cache.cuh"
#include "topk_common.cuh"

namespace qsae {

TmapCache& tmap_cache() {
  static TmapCache cache;
  return cache;
}

namespace {

constexpr int BM = kEncBM;         // rows of x per CTA (UMMA M)
constexpr int BN = kEncBN;         // latents per tile (UMMA N)
constexpr int BK = 64;             // one 128-byte swizzle atom of bf16
constexpr int UMMA_K = 16;
constexpr int kStagesSparse = 3;   // W ring depth, selection epilogues
constexpr int kStagesDense = 2;    // W ring depth when the epilogue needs a store staging area
// Defaults from B200 measurements (DESIGN.md 5.1): the dense epilogue gains 17 % from cta_group::2
// pairs (3-stage ring next to the staging area, half the W bytes per SM); the selection epilogues lose
// 5 % with pairs (the leader's MMA waits for the slower of two epilogues) and gain 2 % from multicast
// at large batch.
constexpr int kDefaultClusterDense = 2;
// dense epilogue: one XOR-swizzled transposition tile per warp, 32 rows of 128 bytes (pairs) or 64 bytes
__host__ __device__ constexpr int dense_stage_bytes(bool wide) { return wide ? 32 * 128 : 32 * 64; }
constexpr int kABytesPerChunk = BM * BK * 2;   // 16 KiB
constexpr int kBBytesPerStage = BN * BK * 2;   // 32 KiB
// warps: 0 TMA, 1 MMA, 2 TMEM alloc, 3 bias, 4.. epilogue (8 warps, 128 columns of a tile each).
// Measured for the dense epilogue: 16 warps of 64 columns are not faster (237 vs 227 us at B = 4096);
// the store phase is bound by the SM's store path to L2 (~25 B/clk per SM, DESIGN.md 5.1), not by
// the latency of an epilogue warp.
__host__ __device__ constexpr int epi_warps(bool dense) { return 8; }
__host__ __device__ constexpr int cta_threads(bool dense) { return 128 + epi_warps(dense) * 32; }
constexpr int kTmemCols = 512;                  // 2 accumulators x 256 columns

constexpr int kMaxPieces = 8;   // pieces of one CTA's range: ceil(range / tiles per row block) + 1 at most, i.e. 2 when there are
                                // fewer row blocks than CTAs (every range-scheduled sweep on 148 SMs); checked by encode_pick_range
struct SmemLayout {
  uint32_t a_off, b_off, staging_off, bias_off, share_off, bar_off, tmem_ptr_off, piece_off, total;
};
// pair (cta_group::2): a CTA keeps only its half of every W stage (16 KiB), which pays for deeper rings
__host__ __device__ constexpr int ring_stages(bool dense, bool pair) {
  return pair ? 4 : (dense ? kStagesDense : kStagesSparse);
}
__host__ __device__ constexpr int stage_bytes(bool pair) { return pair ? kBBytesPerStage / 2 : kBBytesPerStage; }
__host__ __device__ inline SmemLayout smem_layout(int k_chunks, bool dense, bool pair) {
  SmemLayout L;
  const int stages = ring_stages(dense, pair);
  L.a_off = 0;
  L.b_off = L.a_off + k_chunks * kABytesPerChunk;
  L.staging_off = L.b_off + stages * stage_bytes(pair);   // 1024-byte aligned (swizzled TMA store source)
  L.bias_off = L.staging_off + (dense ? epi_warps(true) * dense_stage_bytes(pair) : 0);
  L.share_off = L.bias_off + 2 * BN * 4;         // partner thresholds, 2 x 128 x bf16
  L.bar_off = L.share_off + 2 * BM * 2;
  L.tmem_ptr_off = L.bar_off + 8 * (1 + 2 * stages + 9);
  L.piece_off = L.tmem_ptr_off + 16;
  L.total = L.piece_off + 16 + kMaxPieces * 32;
  return L;
}

// float -> bf16 bits rounded toward -inf (a lower bound stays a lower bound)
__device__ __forceinline__ uint16_t bf16_floor_bits(float f) {
  uint32_t u = __float_as_uint(f);
  if (u & 0x80000000u) u += 0xFFFFu;  // negative: grow the magnitude
  return static_cast<uint16_t>(u >> 16);
}
__device__ __forceinline__ float bf16_bits_to_float(uint16_t b) {
  return __uint_as_float(static_cast<uint32_t>(b) << 16);
}

// smallest float strictly greater than f (f finite or -inf)
__device__ __forceinline__ float next_above(float f) { return key_to_float(float_to_key(f) + 1u); }

// Overflow handling for the 32 buffers owned by this warp's lanes (lane r owns `buf`, `cnt`, and
// the inclusive survivor threshold `thr`). Every buffer more than half full is filtered in place
// against its owner's threshold (insertion order preserved); if that leaves it nearly full it is
// cut to its exact k largest and the threshold moves just above the k-th value (after an exact
// cut, later values equal to the k-th lose on column order).
static __device__ __noinline__ void relieve_warp_buffers(uint2* buf, int& cnt, float& thr,
                                                         float& valid_bound, int k, int cap, int lane) {
  const unsigned full = 0xffffffffu;
  const unsigned lt_mask = (1u << lane) - 1u;
  constexpr int BATCH = 8;
  __syncwarp();
#pragma unroll 1
  for (int r = 0; r < 32; ++r) {
    const int n = __shfl_sync(full, cnt, r);
    if (n <= (cap >> 1)) continue;
    const float t_in = __shfl_sync(full, thr, r);
    uint2* rb = reinterpret_cast<uint2*>(
        __shfl_sync(full, reinterpret_cast<unsigned long long>(buf), r));
    int out = 0;
#pragma unroll 1
    for (int base = 0; base < n; base += 32 * BATCH) {
      uint2 t[BATCH];
#pragma unroll
      for (int i = 0; i < BATCH; ++i) {  // BATCH independent loads in flight
        const int e = base + i * 32 + lane;
        t[i] = (e < n) ? rb[e] : make_uint2(0u, 0u);
      }
#pragma unroll
      for (int i = 0; i < BATCH; ++i) {  // writes land at or before the slots already loaded
        const int e = base + i * 32 + lane;
        const bool keep = (e < n) && (__uint_as_float(t[i].x) >= t_in);
        const unsigned b = __ballot_sync(full, keep);
        if (keep) rb[out + __popc(b & lt_mask)] = t[i];
        out += __popc(b);
      }
    }
    float t_out = t_in;
    float kth = -INFINITY;
    if (out > cap - 96 && out > k) {
      __syncwarp();
      out = warp_compact_row_generic(rb, out, k, lane, &kth);
      t_out = fmaxf(t_in, next_above(kth));
    }
    if (lane == r) {
      cnt = out;
      thr = t_out;
      valid_bound = fmaxf(valid_bound, kth);  // the k-th value itself stays an inclusive bound
    }
  }
  __syncwarp();
}

// v[j] for a per-lane dynamic j: 31 selects (registers cannot be indexed dynamically)
__device__ __forceinline__ float pick32(const float (&v)[32], int j) {
  float a[16], b[8], c[4], d[2];
#pragma unroll
  for (int i = 0; i < 16; ++i) a[i] = (j & 16) ? v[i + 16] : v[i];
#pragma unroll
  for (int i = 0; i < 8; ++i) b[i] = (j & 8) ? a[i + 8] : a[i];
#pragma unroll
  for (int i = 0; i < 4; ++i) c[i] = (j & 4) ? b[i + 4] : b[i];
#pragma unroll
  for (int i = 0; i < 2; ++i) d[i] = (j & 2) ? c[i + 2] : c[i];
  return (j & 1) ? d[1] : d[0];
}

// MODE 0: no class bound (any k <= kMaxK; bisection only)      MODE 1: top-1 per class, k <= 32
// MODE 2: top-2 per class, k <= 64       MODE 3: top-2 per class shared with the partner thread
//                                                 handling the other column half, k <= 128
// MODE 4: fixed prior threshold per row (p.prior), no class bookkeeping
// MODE 5: no survivor buffers at all: every thread keeps the two largest values of each of the 32 column
//         classes of its sub-stream in registers and writes these kTopM = 64 values to p.top_out (sample pre-pass)
// One PIECE of a CTA's work: n_my_tiles tiles starting at tile_begin against the x rows [m0, m0 + 128). A CTA of
// the (split, row block) grid has one piece; a CTA of the range schedule (see Piece below) up to three, and calls
// this once per piece: all selection state is per piece. tt0 = tiles this CTA has processed before the piece (the
// accumulator / barrier phases run on across pieces); sub_base + half = the piece's sub-stream among the row's
// p.nsub survivor lists; zero_from >= 0: this is the last piece of its row block and the lists from zero_from on
// are unused for these rows (their counts are cleared for the merge).
template <int MODE>
__device__ __forceinline__ void epilogue_loop(const EncodeLaunch& p, int n_my_tiles, int tile_begin,
                                              int sub_base, int m0, int tt0, int zero_from, int e, int lane,
                                              uint32_t tmem_base, const float* bias_smem, uint16_t* share,
                                              uint64_t* tmem_full, uint64_t* tmem_empty,
                                              uint64_t* bias_full, uint64_t* pair_empty) {
  const unsigned full = 0xffffffffu;
  const int quad = e & 3;       // TMEM lanes 32*quad .. +31 (hardware: warp_id % 4)
  const int half = e >> 2;      // columns [half*128, half*128+128) of the tile
  const int row_in_tile = quad * 32 + lane;
  const int row = m0 + row_in_tile;
  const bool row_ok = row < p.B;
  const int nsub = p.nsub;
  const int sub = sub_base + half;
  const int cap = p.cap;
  const size_t slot = static_cast<size_t>(row_ok ? row : 0) * nsub + sub;
  uint2* buf = reinterpret_cast<uint2*>(p.cand) + slot * cap;
  int cnt = 0;
  const int k = p.k_sel;
  const uint32_t lane_taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);

  // a value survives iff v >= thr (inclusive; starts at the lowest finite float so that the
  // -inf used to mask out-of-range columns never survives)
  float thr = row_ok ? -3.402823466e+38f : INFINITY;
  float valid_bound = -INFINITY;  // inclusive lower bound of the k-th largest, reported to the merge
  float tm[MODE == 5 ? kTopM : 1];
#pragma unroll
  for (int i = 0; i < (MODE == 5 ? kTopM : 1); ++i) tm[i] = -INFINITY;
  if (MODE == 4 && row_ok) {
    // prior threshold: the m-th largest pre-activation of a sample of this row's latents
    // (itself one of the row's values). Tight, but only probably <= the k-th largest: the merge
    // kernel verifies it by counting survivors and sends the rare failing row to the rescue path.
    thr = fmaxf(thr, p.prior != nullptr ? __ldg(p.prior + static_cast<size_t>(row) * p.prior_stride) : p.prior_const);
    valid_bound = thr;
  }
  constexpr bool kClasses = (MODE >= 1 && MODE <= 3);
  constexpr bool kTop2 = (MODE == 2 || MODE == 3);
  float top1[kClasses ? 32 : 1];
  float top2[kTop2 ? 32 : 1];
  const float init = row_ok ? -INFINITY : INFINITY;
#pragma unroll
  for (int j = 0; j < (kClasses ? 32 : 1); ++j) top1[j] = init;
#pragma unroll
  for (int j = 0; j < (kTop2 ? 32 : 1); ++j) top2[j] = init;

  for (int t = 0; t < n_my_tiles; ++t) {
    const int acc = (tt0 + t) & 1;
    const uint32_t ph = ((tt0 + t) >> 1) & 1;
    mbar_wait(&tmem_full[acc], ph);
    mbar_wait(&bias_full[acc], ph);
    tc_fence_after();
    const int n_tile = (tile_begin + t) * BN + half * 128;
    const float4* bias4 = reinterpret_cast<const float4*>(bias_smem + acc * BN + half * 128);
#pragma unroll 1
    for (int c = 0; c < 4; ++c) {
      uint32_t r[32];
      tmem_ld_32x32b_x32(lane_taddr + acc * BN + half * 128 + c * 32, r);
      tmem_ld_wait();
      const int col0 = n_tile + c * 32;
      float v[32];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 b = bias4[c * 8 + j];
        v[4 * j + 0] = __uint_as_float(r[4 * j + 0]) + b.x;
        v[4 * j + 1] = __uint_as_float(r[4 * j + 1]) + b.y;
        v[4 * j + 2] = __uint_as_float(r[4 * j + 2]) + b.z;
        v[4 * j + 3] = __uint_as_float(r[4 * j + 3]) + b.w;
      }
      if (p.act == 1) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
      }
      if (col0 + 32 > p.H) {  // last, partial tile only
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (col0 + j >= p.H) v[j] = -INFINITY;
      }
      if (p.debug_z != nullptr && row_ok) {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (col0 + j < p.H) p.debug_z[static_cast<size_t>(row) * p.H + col0 + j] = v[j];
      }
      if constexpr (kClasses) {
        // class maxima and the bound they imply
        float bound;
        if constexpr (MODE == 1) {
#pragma unroll
          for (int j = 0; j < 32; ++j) top1[j] = fmaxf(top1[j], v[j]);
          bound = top1[0];
#pragma unroll
          for (int j = 1; j < 32; ++j) bound = fminf(bound, top1[j]);
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            top2[j] = fmaxf(top2[j], fminf(top1[j], v[j]));
            top1[j] = fmaxf(top1[j], v[j]);
          }
          bound = top2[0];
#pragma unroll
          for (int j = 1; j < 32; ++j) bound = fminf(bound, top2[j]);
        }
        if constexpr (MODE == 3) {
          // exchange with the thread on the other column half of this row; a stale partner
          // value is an older, lower bound and therefore still valid
          share[half * BM + row_in_tile] = bf16_floor_bits(bound);
          bound = fminf(bound, bf16_bits_to_float(share[(half ^ 1) * BM + row_in_tile]));
        }
        if (row_ok) { thr = fmaxf(thr, bound); valid_bound = fmaxf(valid_bound, bound); }
      }
      // survivors: per-lane hit mask, then rounds in which every lane with a pending hit stores
      // one entry. Scattered stores cost one LSU transaction per lane, so the number of store
      // instructions per chunk (= max hits of any lane) is what matters, not the ALU work.
      uint32_t hits = 0u;
      if constexpr (MODE == 5) {
        // sample pre-pass: the two largest values of each of the 32 column classes (column mod 32), three
        // FMNMX per element and no data-dependent work. The m-th largest of a row's 2 x 32 x nsub kept values is a
        // lower bound of the m-th largest sampled value (they are distinct elements) and equals it unless three of
        // the row's top m fall into one class (~3 % of the rows at m = 10 over 64 classes). The first version kept
        // an exact sorted top-16 list per thread (25 K warp instructions per tile against 9 K in the main sweep,
        // pre-pass 157 us); one maximum per class is cheaper still but too loose (see DESIGN.md 5.1).
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          tm[32 + j] = fmaxf(tm[32 + j], fminf(tm[j], v[j]));
          tm[j] = fmaxf(tm[j], v[j]);
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) hits |= (v[j] >= thr) ? (1u << j) : 0u;
        while (__any_sync(full, hits != 0u)) {
          if (hits != 0u) {
            const int j = __ffs(hits) - 1;
            hits &= hits - 1u;
            buf[cnt] = make_uint2(__float_as_uint(pick32(v, j)), static_cast<uint32_t>(col0 + j));
            ++cnt;
          }
        }
        if (__any_sync(full, cnt > cap - 32)) {
          if (MODE == 4 && k <= 0) {
            // threshold-only use (q_sae: every value above the threshold is wanted): a full
            // buffer cannot be cut, so stop collecting and report the overflow
            if (cnt > cap - 32) {
              thr = INFINITY;
              if (p.overflow != nullptr) atomicExch(p.overflow, 1);
            }
          } else {
            relieve_warp_buffers(buf, cnt, thr, valid_bound, k, cap, lane);
          }
        }
      }
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) {
      mbar_arrive(&tmem_empty[acc]);
      if (pair_empty != nullptr) mbar_arrive_cluster(&pair_empty[acc], 0);   // the leader's MMA thread waits for both CTAs
    }
  }
  if constexpr (MODE == 5) {
    if (row_ok) {
      float4* dst = reinterpret_cast<float4*>(p.top_out + slot * kTopM);
#pragma unroll
      for (int i = 0; i < kTopM / 4; ++i)
        dst[i] = make_float4(tm[4 * i], tm[4 * i + 1], tm[4 * i + 2], tm[4 * i + 3]);
      if (zero_from >= 0 && half == 0) {   // range schedule: the row block's unused lists hold no values
        const float4 ninf = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
        for (int s2 = zero_from; s2 < nsub; ++s2) {
          float4* z = reinterpret_cast<float4*>(p.top_out + (static_cast<size_t>(row) * nsub + s2) * kTopM);
#pragma unroll
          for (int i = 0; i < kTopM / 4; ++i) z[i] = ninf;
        }
      }
    }
  } else if (row_ok) {
    p.cand_cnt[slot] = cnt;
    p.cand_thr[slot] = valid_bound;
    if (zero_from >= 0 && half == 0) {
      for (int s2 = zero_from; s2 < nsub; ++s2) {
        p.cand_cnt[static_cast<size_t>(row) * nsub + s2] = 0;
        p.cand_thr[static_cast<size_t>(row) * nsub + s2] = -INFINITY;
      }
    }
  }
}

// MODE 4 on its own: the epilogue of the specialised sweep (SEL == 4 below). It keeps exactly the survivor lists of
// epilogue_loop<4> (same threshold, same column order, same counts and bounds) and has no debug paths. Compiled
// without the other modes' per-class registers, it has room for a pipelined TMEM drain: chunk c + 1's tcgen05.ld is
// in flight while chunk c is compared and its survivors stored (tcgen05.wait::ld waits for every outstanding load of
// the thread, so the wait for chunk c + 1 comes after chunk c's work). The chunk loop is unrolled so that the
// two load buffers never have to be copied while a load is landing in one of them.
__device__ __forceinline__ void epilogue_prior(const EncodeLaunch& p, int n_my_tiles, int tile_begin, int sub_base, int m0,
                                               int tt0, int zero_from, int e, int lane, uint32_t tmem_base,
                                               const float* bias_smem, uint64_t* tmem_full, uint64_t* tmem_empty,
                                               uint64_t* bias_full, uint64_t* pair_empty) {
  const unsigned full = 0xffffffffu;
  const int quad = e & 3;       // TMEM lanes 32*quad .. +31 (hardware: warp_id % 4)
  const int half = e >> 2;      // columns [half*128, half*128+128) of the tile
  const int row = m0 + quad * 32 + lane;
  const bool row_ok = row < p.B;
  const int nsub = p.nsub;
  const int cap = p.cap;
  const int k = p.k_sel;
  const size_t slot = static_cast<size_t>(row_ok ? row : 0) * nsub + sub_base + half;
  uint2* buf = reinterpret_cast<uint2*>(p.cand) + slot * cap;
  int cnt = 0;
  const uint32_t half_taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + half * 128;

  // as in epilogue_loop<4>: a value survives iff v >= thr, thr = max(lowest finite float, prior of the row)
  float thr = INFINITY;
  float valid_bound = -INFINITY;
  if (row_ok) {
    thr = fmaxf(-3.402823466e+38f, p.prior != nullptr ? __ldg(p.prior + static_cast<size_t>(row) * p.prior_stride) : p.prior_const);
    valid_bound = thr;
  }

  for (int t = 0; t < n_my_tiles; ++t) {
    const int acc = (tt0 + t) & 1;
    const uint32_t ph = ((tt0 + t) >> 1) & 1;
    mbar_wait(&tmem_full[acc], ph);
    mbar_wait(&bias_full[acc], ph);
    tc_fence_after();
    const int n_tile = (tile_begin + t) * BN + half * 128;
    const float4* bias4 = reinterpret_cast<const float4*>(bias_smem + acc * BN + half * 128);
    const uint32_t taddr = half_taddr + acc * BN;
    uint32_t r[2][32];
    tmem_ld_32x32b_x32(taddr, r[0]);
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      uint32_t (&rc)[32] = r[c & 1];
      tmem_ld_wait(rc);                                              // chunk c has landed; nothing else is in flight
      if (c < 3) tmem_ld_32x32b_x32(taddr + (c + 1) * 32, r[(c + 1) & 1]);
      const int col0 = n_tile + c * 32;
      float v[32];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 b = bias4[c * 8 + j];
        v[4 * j + 0] = __uint_as_float(rc[4 * j + 0]) + b.x;
        v[4 * j + 1] = __uint_as_float(rc[4 * j + 1]) + b.y;
        v[4 * j + 2] = __uint_as_float(rc[4 * j + 2]) + b.z;
        v[4 * j + 3] = __uint_as_float(rc[4 * j + 3]) + b.w;
      }
      if (p.act == 1) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
      }
      if (col0 + 32 > p.H) {  // last, partial tile only
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (col0 + j >= p.H) v[j] = -INFINITY;
      }
      uint32_t hits = 0u;
#pragma unroll
      for (int j = 0; j < 32; ++j) hits |= (v[j] >= thr) ? (1u << j) : 0u;
      while (__any_sync(full, hits != 0u)) {
        if (hits != 0u) {
          const int j = __ffs(hits) - 1;
          hits &= hits - 1u;
          buf[cnt] = make_uint2(__float_as_uint(pick32(v, j)), static_cast<uint32_t>(col0 + j));
          ++cnt;
        }
      }
      if (__any_sync(full, cnt > cap - 32)) {
        if (k <= 0) {
          // threshold-only use (q_sae): a full buffer cannot be cut, so stop collecting and report the overflow
          if (cnt > cap - 32) {
            thr = INFINITY;
            if (p.overflow != nullptr) atomicExch(p.overflow, 1);
          }
        } else {
          // the call may save and restore registers: let the next chunk land first. It takes its in / out
          // arguments by address, so they are copies: cnt, thr and valid_bound stay in registers on the common path.
          if (c < 3) tmem_ld_wait(r[(c + 1) & 1]);
          int cnt_r = cnt;
          float thr_r = thr, bound_r = valid_bound;
          relieve_warp_buffers(buf, cnt_r, thr_r, bound_r, k, cap, lane);
          cnt = cnt_r; thr = thr_r; valid_bound = bound_r;
        }
      }
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) {
      mbar_arrive(&tmem_empty[acc]);
      if (pair_empty != nullptr) mbar_arrive_cluster(&pair_empty[acc], 0);   // the leader's MMA thread waits for both CTAs
    }
  }
  if (row_ok) {
    p.cand_cnt[slot] = cnt;
    p.cand_thr[slot] = valid_bound;
    if (zero_from >= 0 && half == 0) {
      for (int s2 = zero_from; s2 < nsub; ++s2) {
        p.cand_cnt[static_cast<size_t>(row) * nsub + s2] = 0;
        p.cand_thr[static_cast<size_t>(row) * nsub + s2] = -INFINITY;
      }
    }
  }
}

// ---- range schedule --------------------------------------------------------------------------------------
// Small batches do not fill the machine with (split, row block) CTAs: B = 4096 gives 32 row blocks x 4 splits = 128
// CTAs on 148 SMs. With p.range_g > 0 the grid is range_g CTAs (one per SM) and the U = row_blocks x n_tiles tile
// units, in row-block-major order, are cut into range_g contiguous ranges of (almost) equal length: CTA g sweeps
// units [g U / G, (g + 1) U / G). A range that crosses a row-block boundary is processed in pieces, the x tile
// being reloaded in between (the producer waits for the MMAs that still read the old one); every piece is a
// sub-stream pair of its row block, numbered by the CTA's position among the CTAs that touch the block.
struct Piece {
  int rb, tile0, n, sub_base, zero_from;
};
__host__ __device__ inline long long range_start(long long g, long long U, long long G) { return g * U / G; }
// the CTA whose range contains unit u: the largest g with g U / G <= u
__host__ __device__ inline int range_owner(long long u, long long U, long long G) {
  return static_cast<int>(((u + 1) * G - 1) / U);
}
struct PieceIter {
  long long u, u_end, U, G;
  int n_tiles, g;
  bool legacy, done;
  Piece legacy_piece;
  __device__ bool next(Piece& pc) {
    if (legacy) {
      if (done) return false;
      done = true;
      pc = legacy_piece;
      return pc.n > 0;
    }
    if (u >= u_end) return false;
    const int rb = static_cast<int>(u / n_tiles);
    const int t0 = static_cast<int>(u - static_cast<long long>(rb) * n_tiles);
    const long long left = u_end - u;
    const int n = static_cast<int>(left < n_tiles - t0 ? left : n_tiles - t0);
    const long long first_u = static_cast<long long>(rb) * n_tiles;
    const int g_first = range_owner(first_u, U, G);
    pc.rb = rb; pc.tile0 = t0; pc.n = n;
    pc.sub_base = 2 * (g - g_first);
    pc.zero_from = (t0 + n == n_tiles) ? pc.sub_base + 2 : -1;
    u += n;
    return true;
  }
};

__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  const __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&t);
}

__device__ __forceinline__ uint4 ld_shared_v4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}

// Dense epilogue (t_sae: the reference returns the dense ReLU latents, sae/ternary.py:116-122).
// Each epilogue warp turns its 32 rows x 32 columns of the accumulator into
//   h fp32                 (p.dense_flags & 1)   the module's first return value
//   h_hi = bf16(h)         (p.dense_flags & 2)   A operand of the decoder GEMM
//   h_lo = bf16(h - h_hi)  (p.dense_flags & 4)   second A operand (h_hi + h_lo carries 16 mantissa bits)
// The accumulator arrives one row per lane; an XOR-swizzled shared-memory tile (16-byte chunk c of
// row r at c ^ (r % 8) for 128-byte rows, c ^ ((r / 2) % 4) for 64-byte rows: conflict-free both for the
// lane-per-row writes and for the row-contiguous reads) turns that into 16-byte global stores in which
// every warp instruction writes whole 128-byte (fp32) or 64-byte (bf16) row segments. The L1 data pipe
// is the resource to spare here: it also feeds the UMMA operand reads (ncu: 73 % busy, half of it bank
// conflicts, with a padded-row layout). (A first version issued cp.async.bulk.tensor stores from a swizzled staging tile; the TMA
// engine handled its 64-byte-wide boxes at ~16 B/clk per SM and the store time added to the sweep
// instead of hiding behind it: 225 us vs 110 us with the stores masked off at B = 4096.)
// WIDE: 36-word fp32 staging rows (32 columns at a time); otherwise the fp32 tile goes through the
// 20-word bf16 layout in two 16-column halves (the single-CTA variant has no shared memory to spare).
template <bool WIDE>
__device__ __forceinline__ void epilogue_dense(const EncodeLaunch& p, int n_my_tiles, int tile_begin, int m0, int tt0, int e,
                                               int lane, uint32_t tmem_base, const float* bias_smem, uint8_t* staging,
                                               uint64_t* tmem_full, uint64_t* tmem_empty, uint64_t* bias_full,
                                               uint64_t* pair_empty) {
  constexpr int kColsPerWarp = BN / (epi_warps(true) / 4);   // 128
  const int quad = e & 3;          // TMEM lanes 32*quad .. +31 (hardware: warp_id % 4)
  const int cgrp = e >> 2;         // columns [cgrp * 128, +128) of the tile
  const int row0 = m0 + quad * 32;
  const bool warp_live = row0 < p.B;
  const uint32_t st = smem_u32(staging + e * dense_stage_bytes(WIDE));
  const uint32_t lane_taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
  const int flags = p.dense_flags;
  const size_t H = static_cast<size_t>(p.H);
  // read-back roles: fp32 -- 8 lanes per row, 4 rows per instruction; bf16 -- 4 lanes per row, 8 rows
  const int f_row = lane >> 3, f_col = (lane & 7) * 4;
  const int h_row = lane >> 2, h_col = (lane & 3) * 8;

  // act == 2: activity counts of the current level, flushed (one atomic per warp) when the level changes
  unsigned n_act = 0u;
  int cur_lvl = 0;
  auto flush_level_count = [&]() {
    const unsigned tot = __reduce_add_sync(0xffffffffu, n_act);
    if (lane == 0 && tot != 0u) atomicAdd(p.step_level_count + cur_lvl, static_cast<unsigned long long>(tot));
    n_act = 0u;
  };

  for (int t = 0; t < n_my_tiles; ++t) {
    const int acc = (tt0 + t) & 1;
    const uint32_t ph = ((tt0 + t) >> 1) & 1;
    mbar_wait(&tmem_full[acc], ph);
    mbar_wait(&bias_full[acc], ph);
    tc_fence_after();
    const int n_tile = (tile_begin + t) * BN + cgrp * kColsPerWarp;
    const float4* bias4 = reinterpret_cast<const float4*>(bias_smem + acc * BN + cgrp * kColsPerWarp);
    if (p.act == 2) {   // the warp's 128 columns of a tile lie in one level (boundaries are multiples of 128)
      int lvl = 0;
      while (lvl + 1 < p.step_n_levels && n_tile >= __ldg(p.step_level_start + lvl + 1)) ++lvl;
      if (lvl != cur_lvl) {
        flush_level_count();
        cur_lvl = lvl;
      }
    }
#pragma unroll 1
    for (int c = 0; c < kColsPerWarp / 32; ++c) {
      uint32_t r[32];
      tmem_ld_32x32b_x32(lane_taddr + acc * BN + cgrp * kColsPerWarp + c * 32, r);
      tmem_ld_wait();
      const int col0 = n_tile + c * 32;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 b = bias4[c * 8 + j];
        r[4 * j + 0] = __float_as_uint(__uint_as_float(r[4 * j + 0]) + b.x);
        r[4 * j + 1] = __float_as_uint(__uint_as_float(r[4 * j + 1]) + b.y);
        r[4 * j + 2] = __float_as_uint(__uint_as_float(r[4 * j + 2]) + b.z);
        r[4 * j + 3] = __float_as_uint(__uint_as_float(r[4 * j + 3]) + b.w);
      }
      if (p.act == 1) {
#pragma unroll
        for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(fmaxf(__uint_as_float(r[j]), 0.f));
      }
      if (!warp_live || col0 >= p.H) continue;  // warp-uniform
      uint32_t act_bits = 0u;   // act == 2: bit j = column col0 + j of this lane's row is active
      if (p.act == 2) {
        // q_sae dense path: r = active ? scale[col] : 0 (the A operand of the level GEMMs; hi / lo leave below)
        const float4* sc4 = reinterpret_cast<const float4*>(p.step_scale + col0);
        unsigned n = 0u;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 s = __ldg(sc4 + j);
          const bool a0 = __uint_as_float(r[4 * j + 0]) >= p.step_thr, a1 = __uint_as_float(r[4 * j + 1]) >= p.step_thr;
          const bool a2 = __uint_as_float(r[4 * j + 2]) >= p.step_thr, a3 = __uint_as_float(r[4 * j + 3]) >= p.step_thr;
          n += (a0 ? 1u : 0u) + (a1 ? 1u : 0u) + (a2 ? 1u : 0u) + (a3 ? 1u : 0u);
          act_bits |= ((a0 ? 1u : 0u) | (a1 ? 2u : 0u) | (a2 ? 4u : 0u) | (a3 ? 8u : 0u)) << (4 * j);
          r[4 * j + 0] = a0 ? __float_as_uint(s.x) : 0u;
          r[4 * j + 1] = a1 ? __float_as_uint(s.y) : 0u;
          r[4 * j + 2] = a2 ? __float_as_uint(s.z) : 0u;
          r[4 * j + 3] = a3 ? __float_as_uint(s.w) : 0u;
        }
        if (row0 + lane < p.B) n_act += n;
      }
      if constexpr (WIDE) {
        if (p.act == 3) {
          // ReLU backward at the forward's output (streamed-operand kernel only, no bias): out = (acc + gate_add) *
          // (gate > 0); torch masks on the returned h and selects, so a non-finite acc where h <= 0 gives 0. gate /
          // gate_add do not depend on the accumulator: four rows of both are loaded before any of them is used (a load
          // per row in turn left the kernel latency-bound). The warp's 32 rows are summed per column (p.gate_colsum +=
          // sum_b out: the bias gradient, one atomic per column and warp). The transformation runs in the
          // row-contiguous read-back layout, where gate and gate_add are read coalesced.
          __syncwarp();
#pragma unroll
          for (int q = 0; q < 8; ++q)
            st_shared_v4(st + lane * 128 + ((q ^ (lane & 7)) << 4), r[4 * q], r[4 * q + 1], r[4 * q + 2], r[4 * q + 3]);
          __syncwarp();
          const int cc = col0 + f_col;
          float4 cs = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int j0 = 0; j0 < 8; j0 += 4) {
            float4 hv[4], av[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int rr = 4 * (j0 + i) + f_row;
              const bool ok = row0 + rr < p.B && cc < p.H;
              const size_t off = static_cast<size_t>(row0 + rr) * H + cc;
              hv[i] = ok ? __ldg(reinterpret_cast<const float4*>(p.gate + off)) : make_float4(0.f, 0.f, 0.f, 0.f);
              av[i] = ok && p.gate_add != nullptr ? __ldg(reinterpret_cast<const float4*>(p.gate_add + off))
                                                  : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int rr = 4 * (j0 + i) + f_row;
              if (row0 + rr >= p.B || cc >= p.H) continue;
              const size_t off = static_cast<size_t>(row0 + rr) * H + cc;
              const uint4 u = ld_shared_v4(st + rr * 128 + (((lane & 7) ^ (rr & 7)) << 4));
              float4 v = make_float4(__uint_as_float(u.x) + av[i].x, __uint_as_float(u.y) + av[i].y,
                                     __uint_as_float(u.z) + av[i].z, __uint_as_float(u.w) + av[i].w);
              v.x = hv[i].x > 0.f ? v.x : 0.f; v.y = hv[i].y > 0.f ? v.y : 0.f;
              v.z = hv[i].z > 0.f ? v.z : 0.f; v.w = hv[i].w > 0.f ? v.w : 0.f;
              cs.x += v.x; cs.y += v.y; cs.z += v.z; cs.w += v.w;
              if (flags & 1) *reinterpret_cast<float4*>(p.out_f32 + off) = v;
              if (flags & 2)
                *reinterpret_cast<uint2*>(p.out_hi + off) = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
            }
          }
          if (p.gate_colsum != nullptr) {   // lanes l, l + 8, l + 16, l + 24 hold the same four columns
#pragma unroll
            for (int sh = 8; sh <= 16; sh <<= 1) {
              cs.x += __shfl_xor_sync(0xffffffffu, cs.x, sh);
              cs.y += __shfl_xor_sync(0xffffffffu, cs.y, sh);
              cs.z += __shfl_xor_sync(0xffffffffu, cs.z, sh);
              cs.w += __shfl_xor_sync(0xffffffffu, cs.w, sh);
            }
            if (lane < 8 && cc < p.H) {
              atomicAdd(p.gate_colsum + cc, cs.x);
              atomicAdd(p.gate_colsum + cc + 1, cs.y);
              atomicAdd(p.gate_colsum + cc + 2, cs.z);
              atomicAdd(p.gate_colsum + cc + 3, cs.w);
            }
          }
          continue;
        }
      }
      if (flags & 1) {
        if constexpr (WIDE) {
          __syncwarp();                            // the previous tile's readers are done
#pragma unroll
          for (int q = 0; q < 8; ++q)
            st_shared_v4(st + lane * 128 + ((q ^ (lane & 7)) << 4), r[4 * q], r[4 * q + 1], r[4 * q + 2], r[4 * q + 3]);
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int rr = 4 * j + f_row;
            const uint4 v = ld_shared_v4(st + rr * 128 + (((lane & 7) ^ (rr & 7)) << 4));
            if (row0 + rr < p.B && col0 + f_col < p.H)
              *reinterpret_cast<uint4*>(p.out_f32 + static_cast<size_t>(row0 + rr) * H + col0 + f_col) = v;
          }
        } else {
#pragma unroll
          for (int hf = 0; hf < 2; ++hf) {         // 16 columns at a time through the 80-byte-row layout
            __syncwarp();
#pragma unroll
            for (int q = 0; q < 4; ++q)
              st_shared_v4(st + lane * 64 + ((q ^ ((lane >> 1) & 3)) << 4), r[16 * hf + 4 * q], r[16 * hf + 4 * q + 1],
                           r[16 * hf + 4 * q + 2], r[16 * hf + 4 * q + 3]);
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int rr = 8 * j + h_row;
              const int cc = col0 + 16 * hf + (lane & 3) * 4;
              const uint4 v = ld_shared_v4(st + rr * 64 + (((lane & 3) ^ ((rr >> 1) & 3)) << 4));
              if (row0 + rr < p.B && cc < p.H)
                *reinterpret_cast<uint4*>(p.out_f32 + static_cast<size_t>(row0 + rr) * H + cc) = v;
            }
          }
        }
      }
      if (flags & 6) {
        uint32_t hi[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) hi[j] = pack_bf16x2(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1]));
        if (flags & 2) {
          __syncwarp();
#pragma unroll
          for (int q = 0; q < 4; ++q)
            st_shared_v4(st + lane * 64 + ((q ^ ((lane >> 1) & 3)) << 4), hi[4 * q], hi[4 * q + 1], hi[4 * q + 2], hi[4 * q + 3]);
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int rr = 8 * j + h_row;
            const uint4 v = ld_shared_v4(st + rr * 64 + (((lane & 3) ^ ((rr >> 1) & 3)) << 4));
            if (row0 + rr < p.B && col0 + h_col < p.H)
              *reinterpret_cast<uint4*>(p.out_hi + static_cast<size_t>(row0 + rr) * H + col0 + h_col) = v;
          }
        }
        if (flags & 4) {
          uint32_t lo[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float a = __uint_as_float(r[2 * j]), b = __uint_as_float(r[2 * j + 1]);
            const float ah = __uint_as_float(hi[j] << 16), bh = __uint_as_float(hi[j] & 0xFFFF0000u);
            lo[j] = pack_bf16x2(a - ah, b - bh);
          }
          __syncwarp();
#pragma unroll
          for (int q = 0; q < 4; ++q)
            st_shared_v4(st + lane * 64 + ((q ^ ((lane >> 1) & 3)) << 4), lo[4 * q], lo[4 * q + 1], lo[4 * q + 2], lo[4 * q + 3]);
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int rr = 8 * j + h_row;
            const uint4 v = ld_shared_v4(st + rr * 64 + (((lane & 3) ^ ((rr >> 1) & 3)) << 4));
            if (row0 + rr < p.B && col0 + h_col < p.H)
              *reinterpret_cast<uint4*>(p.out_lo + static_cast<size_t>(row0 + rr) * H + col0 + h_col) = v;
          }
        }
      }
      if (p.act == 2 && p.step_mask != nullptr) {
        // activity mask of the same decisions: bf16 1.0 (0x3F80) / 0, through the staging layout of the bf16 outputs
        uint32_t mk[16];
#pragma unroll
        for (int j = 0; j < 16; ++j)
          mk[j] = (((act_bits >> (2 * j)) & 1u) ? 0x3F80u : 0u) | (((act_bits >> (2 * j + 1)) & 1u) ? 0x3F800000u : 0u);
        __syncwarp();
#pragma unroll
        for (int q = 0; q < 4; ++q)
          st_shared_v4(st + lane * 64 + ((q ^ ((lane >> 1) & 3)) << 4), mk[4 * q], mk[4 * q + 1], mk[4 * q + 2], mk[4 * q + 3]);
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int rr = 8 * j + h_row;
          const uint4 v = ld_shared_v4(st + rr * 64 + (((lane & 3) ^ ((rr >> 1) & 3)) << 4));
          if (row0 + rr < p.B && col0 + h_col < p.H)
            *reinterpret_cast<uint4*>(p.step_mask + static_cast<size_t>(row0 + rr) * p.step_mask_pitch + col0 + h_col) = v;
        }
      }
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) {
      mbar_arrive(&tmem_empty[acc]);
      if (pair_empty != nullptr) mbar_arrive_cluster(&pair_empty[acc], 0);
    }
  }
  if (p.act == 2) flush_level_count();
}

// one piece of the epilogue role: dense epilogue, the prior-threshold epilogue of the specialised sweep (SEL == 4), or
// the selection mode of this launch
template <bool DENSE, bool PAIR, int SEL>
__device__ __forceinline__ void run_epilogue_piece(const EncodeLaunch& p, int n, int tile0, int sub_base, int m0, int tt0,
                                                   int zero_from, int e, int lane, uint32_t tmem_base, const float* bias_smem,
                                                   uint16_t* share, uint8_t* staging, uint64_t* tmem_full, uint64_t* tmem_empty,
                                                   uint64_t* bias_full, uint64_t* pe) {
  if constexpr (DENSE) {
    epilogue_dense<PAIR>(p, n, tile0, m0, tt0, e, lane, tmem_base, bias_smem, staging, tmem_full, tmem_empty, bias_full, pe);
  } else if constexpr (SEL == 4) {
    epilogue_prior(p, n, tile0, sub_base, m0, tt0, zero_from, e, lane, tmem_base, bias_smem, tmem_full, tmem_empty, bias_full, pe);
  } else {
    switch (p.mode) {
      case 1:
        epilogue_loop<1>(p, n, tile0, sub_base, m0, tt0, zero_from, e, lane, tmem_base, bias_smem, share, tmem_full, tmem_empty, bias_full, pe);
        break;
      case 2:
        epilogue_loop<2>(p, n, tile0, sub_base, m0, tt0, zero_from, e, lane, tmem_base, bias_smem, share, tmem_full, tmem_empty, bias_full, pe);
        break;
      case 3:
        epilogue_loop<3>(p, n, tile0, sub_base, m0, tt0, zero_from, e, lane, tmem_base, bias_smem, share, tmem_full, tmem_empty, bias_full, pe);
        break;
      case 4:
        epilogue_loop<4>(p, n, tile0, sub_base, m0, tt0, zero_from, e, lane, tmem_base, bias_smem, share, tmem_full, tmem_empty, bias_full, pe);
        break;
      case 5:
        epilogue_loop<5>(p, n, tile0, sub_base, m0, tt0, zero_from, e, lane, tmem_base, bias_smem, share, tmem_full, tmem_empty, bias_full, pe);
        break;
      default:
        epilogue_loop<0>(p, n, tile0, sub_base, m0, tt0, zero_from, e, lane, tmem_base, bias_smem, share, tmem_full, tmem_empty, bias_full, pe);
        break;
    }
  }
}

// CL = 0: one CTA per 128 rows.
// CL = 1 (multicast): clusters of two CTAs along the row-block axis sweep the same W tiles in
//   lockstep; each CTA fetches half of every 256 x 64 stage (128 latents) and TMA-multicasts it into
//   both CTAs' rings, so the pair reads W from L2 once instead of twice. MMAs stay per CTA.
// CL = 2 (pair, cta_group::2): the two CTAs execute ONE tcgen05.mma of M = 256. Each keeps its own
//   128 rows of x and only ITS half of every W stage (16 KiB instead of 32), the leader (rank 0)
//   issues the MMAs and commits, every TMA load credits the leader's barriers, both epilogues drain
//   their own 128 accumulator rows from their own TMEM. Halves the W bytes per SM (L2 -> SM traffic
//   and shared-memory reads) and frees 16 KiB per stage: 4-stage ring for the selection epilogues,
//   3 stages next to the store staging area for the dense epilogue.
// SEL = -1: the selection mode is p.mode, chosen at run time; SEL = 4: prior threshold only (epilogue_prior). Producer,
//   MMA and bias roles are the same for both.
template <int K_CHUNKS, bool DENSE, int CL, int SEL>
__global__ void __launch_bounds__(cta_threads(DENSE), 1)
encode_topk_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_w, EncodeLaunch p) {
  constexpr bool MCAST = CL == 1;
  constexpr bool PAIR = CL >= 2;            // CL = 3: cta_group::2 pairs ON the range schedule (sparse sweeps, small batches)
  constexpr int kStages = ring_stages(DENSE, PAIR);
  constexpr int kStageBytes = stage_bytes(PAIR);
  extern __shared__ __align__(1024) uint8_t smem[];
  const SmemLayout L = smem_layout(K_CHUNKS, DENSE, PAIR);
  uint8_t* a_smem = smem + L.a_off;
  uint8_t* b_smem = smem + L.b_off;
  float* bias_smem = reinterpret_cast<float*>(smem + L.bias_off);
  uint16_t* share = reinterpret_cast<uint16_t*>(smem + L.share_off);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.bar_off);
  uint64_t* a_full = bars;
  uint64_t* full = bars + 1;
  uint64_t* empty = full + kStages;
  uint64_t* tmem_full = empty + kStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* bias_full = tmem_empty + 2;
  uint64_t* pair_empty = bias_full + 2;     // leader only: both CTAs' epilogues released accumulator a
  uint64_t* a_empty = pair_empty + 2;       // every MMA of the finished piece has completed (the x tile may be replaced)
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + L.tmem_ptr_off);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // range schedule (single-CTA variant only): one CTA per SM sweeps a contiguous range of tile units
  const bool ranged = (CL == 0 || CL == 3) && p.range_g > 0;
  // cluster variants pair two row blocks along grid.x (CTA pairs must be adjacent in x)
  const int split = ranged ? 0 : ((CL != 0) ? blockIdx.y : blockIdx.x);
  const int m0_grid = ranged ? 0 : ((CL != 0) ? blockIdx.x : blockIdx.y) * BM;
  const uint32_t cta_rank = (CL != 0) ? cluster_ctarank() : 0u;
  const bool leader = cta_rank == 0u;
  // the CTA's pieces, computed once by thread 0 (64-bit divisions) and read from shared memory by every role
  int* piece_n = reinterpret_cast<int*>(smem + L.piece_off);
  Piece* piece_tab = reinterpret_cast<Piece*>(smem + L.piece_off + 16);
  if (threadIdx.x == 0) {
    PieceIter it;
    it.legacy = !ranged;
    it.done = false;
    it.n_tiles = p.n_tiles;
    // pair variant: the units are (pair of row blocks, tile); both CTAs of a pair walk the same range
    it.g = (CL == 3) ? blockIdx.x / 2 : blockIdx.x;
    it.U = static_cast<long long>(((p.B + BM - 1) / BM) / (CL == 3 ? 2 : 1)) * p.n_tiles;
    it.G = ranged ? p.range_g : 1;
    it.u = ranged ? range_start(it.g, it.U, it.G) : 0;
    it.u_end = ranged ? range_start(it.g + 1, it.U, it.G) : 0;
    const int tile_begin = split * p.tiles_per_split;
    const int tile_end = min(p.n_tiles, tile_begin + p.tiles_per_split);
    it.legacy_piece.rb = m0_grid / BM;
    it.legacy_piece.tile0 = tile_begin;
    it.legacy_piece.n = max(0, tile_end - tile_begin);
    it.legacy_piece.sub_base = split * 2;
    it.legacy_piece.zero_from = -1;
    int n = 0;
    Piece pc;
    while (it.next(pc)) {
      if (n == kMaxPieces) {
        printf("qsae: more than %d pieces in one CTA's tile range\n", kMaxPieces);
        __trap();
      }
      if (CL == 3) pc.rb = 2 * pc.rb + static_cast<int>(cta_rank);   // my row block of the pair
      piece_tab[n++] = pc;
    }
    *piece_n = n;
  }
  if (threadIdx.x == 0) {
    if ((smem_u32(smem) & 1023u) != 0u) {
      printf("qsae: dynamic shared memory is not 1024-byte aligned\n");
      __trap();
    }
    mbar_init(a_full, 1);
    mbar_init(a_empty, 1);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], MCAST ? 2 : 1);   // multicast: both CTAs' MMAs must have released the stage
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], epi_warps(DENSE));
      mbar_init(&bias_full[a], 1);
      mbar_init(&pair_empty[a], 2 * epi_warps(DENSE));
    }
    fence_mbar_init();
    fence_proxy_async_smem();
  }
  if (threadIdx.x < 2 * BM) share[threadIdx.x] = 0xFF80u;  // bf16 -inf
  if (warp == 2) {
    if constexpr (PAIR) tmem_alloc_pair<kTmemCols>(tmem_ptr);
    else tmem_alloc<kTmemCols>(tmem_ptr);
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (CL != 0) cluster_sync_all();   // the peer's barriers exist before anything signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ------------------------------------------------------------- TMA producer
    if (lane == 0) {
      tma_prefetch_desc(&tmap_x);
      tma_prefetch_desc(&tmap_w);
      const int n_pieces = *piece_n;
      int stage = 0;
      uint32_t phase = 0;
      for (int pi = 0; pi < n_pieces; ++pi) {
        const Piece pc = piece_tab[pi];
        const int m0 = pc.rb * BM;
        // a new x tile may only land once every MMA that reads the previous one has completed
        if (pi > 0) mbar_wait(a_empty, static_cast<uint32_t>(pi - 1) & 1u);
        if constexpr (PAIR) {
          // both x tiles and both halves of every W stage are credited to the leader's barriers
          const uint32_t a_full_leader = mapa_u32(smem_u32(a_full), 0);
          if (leader) mbar_arrive_expect_tx(a_full, 2 * K_CHUNKS * kABytesPerChunk);
#pragma unroll
          for (int kc = 0; kc < K_CHUNKS; ++kc)
            tma_load_2d_pair(a_smem + kc * kABytesPerChunk, &tmap_x, a_full_leader, kc * BK, m0, kPolicyEvictFirst);
        } else {
          mbar_arrive_expect_tx(a_full, K_CHUNKS * kABytesPerChunk);
#pragma unroll
          for (int kc = 0; kc < K_CHUNKS; ++kc)
            tma_load_2d(a_smem + kc * kABytesPerChunk, &tmap_x, a_full, kc * BK, m0, kPolicyEvictFirst);
        }
        for (int t = 0; t < pc.n; ++t) {
          const int n0 = (pc.tile0 + t) * BN;
#pragma unroll 1
          for (int kc = 0; kc < K_CHUNKS; ++kc) {
            mbar_wait(&empty[stage], phase ^ 1u);
            if constexpr (PAIR) {
              if (leader) mbar_arrive_expect_tx(&full[stage], kBBytesPerStage);   // 16 KiB from each CTA
              tma_load_2d_pair(b_smem + stage * kStageBytes, &tmap_w, mapa_u32(smem_u32(&full[stage]), 0), kc * BK,
                               n0 + static_cast<int>(cta_rank) * (BN / 2), kPolicyEvictLast);
            } else if constexpr (MCAST) {
              mbar_arrive_expect_tx(&full[stage], kBBytesPerStage);
              // my half of the stage lands in both CTAs; the other half arrives from the peer
              tma_load_2d_mcast(b_smem + stage * kBBytesPerStage + cta_rank * (kBBytesPerStage / 2), &tmap_w,
                                &full[stage], kc * BK, n0 + static_cast<int>(cta_rank) * (BN / 2), 0x3, kPolicyEvictLast);
            } else {
              mbar_arrive_expect_tx(&full[stage], kBBytesPerStage);
              tma_load_2d(b_smem + stage * kBBytesPerStage, &tmap_w, &full[stage], kc * BK, n0, kPolicyEvictLast);
            }
            if (++stage == kStages) { stage = 0; phase ^= 1u; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------- MMA issuer (pair: the leader only)
    if (lane == 0 && (!PAIR || leader)) {
      constexpr uint32_t idesc = umma_idesc_bf16_f32(PAIR ? 2 * BM : BM, BN);
      const uint64_t a_desc0 = umma_desc_kmajor_sw128(smem_u32(a_smem));
      const uint64_t b_desc0 = umma_desc_kmajor_sw128(smem_u32(b_smem));
      const int n_pieces = *piece_n;
      int tt = 0;
      int stage = 0;
      uint32_t phase = 0;
      for (int pi = 0; pi < n_pieces; ++pi) {
        const Piece pc = piece_tab[pi];
        mbar_wait(a_full, static_cast<uint32_t>(pi) & 1u);
        tc_fence_after();
        for (int t = 0; t < pc.n; ++t, ++tt) {
          const int acc = tt & 1;
          mbar_wait(PAIR ? &pair_empty[acc] : &tmem_empty[acc], ((tt >> 1) & 1) ^ 1u);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + acc * BN;
#pragma unroll 1
          for (int kc = 0; kc < K_CHUNKS; ++kc) {
            mbar_wait(&full[stage], phase);
            tc_fence_after();
            const uint64_t a_desc = a_desc0 + static_cast<uint64_t>((kc * kABytesPerChunk) >> 4);
            const uint64_t b_desc = b_desc0 + static_cast<uint64_t>((stage * kStageBytes) >> 4);
#pragma unroll
            for (int ks = 0; ks < BK / UMMA_K; ++ks) {
              // advance 16 elements = 32 bytes along K inside the swizzle atom: +2 in the
              // (address >> 4) field of the descriptor
              if constexpr (PAIR) umma_f16_ss_pair(d_tmem, a_desc + ks * 2, b_desc + ks * 2, idesc, (kc | ks) != 0 ? 1u : 0u);
              else umma_f16_ss(d_tmem, a_desc + ks * 2, b_desc + ks * 2, idesc, (kc | ks) != 0 ? 1u : 0u);
            }
            if constexpr (PAIR) {
              umma_commit_pair(&empty[stage], 0x3);
              if (kc == K_CHUNKS - 1) umma_commit_pair(&tmem_full[acc], 0x3);
            } else {
              if constexpr (MCAST) umma_commit_mcast(&empty[stage], 0x3);
              else umma_commit(&empty[stage]);
              if (kc == K_CHUNKS - 1) umma_commit(&tmem_full[acc]);
            }
            if (++stage == kStages) { stage = 0; phase ^= 1u; }
          }
        }
        if constexpr (CL == 0) umma_commit(a_empty);   // the piece's MMAs no longer read the x tile once this fires
        if constexpr (CL == 3) umma_commit_pair(a_empty, 0x3);   // ... in either CTA of the pair
      }
    }
  } else if (warp == 3) {
    // ------------------------------------------------------------- bias tile loader
    const int n_pieces = *piece_n;
    int tt = 0;
    for (int pi = 0; pi < n_pieces; ++pi) {
      const Piece pc = piece_tab[pi];
      for (int t = 0; t < pc.n; ++t, ++tt) {
        const int acc = tt & 1;
        mbar_wait(&tmem_empty[acc], ((tt >> 1) & 1) ^ 1u);
        const int n0 = (pc.tile0 + t) * BN;
#pragma unroll
        for (int i = 0; i < BN / 32; ++i) {
          const int c = i * 32 + lane;
          bias_smem[acc * BN + c] = (p.bias != nullptr && n0 + c < p.H) ? __ldg(p.bias + n0 + c) : 0.f;
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&bias_full[acc]);
      }
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------- epilogue / selection
    const int e = warp - 4;
    uint64_t* pe = PAIR ? pair_empty : nullptr;
    if constexpr (CL == 1 || CL == 2) {
      // these cluster variants never run the range schedule: one piece, its constants known at compile time (keeps the
      // epilogue's register allocation where it was before pieces existed: the B = 65536 sweep lost 7 % otherwise)
      const int tile_begin = split * p.tiles_per_split;
      const int n = max(0, min(p.n_tiles, tile_begin + p.tiles_per_split) - tile_begin);
      if (n > 0) run_epilogue_piece<DENSE, PAIR, SEL>(p, n, tile_begin, split * 2, m0_grid, 0, -1, e, lane, tmem_base, bias_smem, share, smem + L.staging_off,
                                                 tmem_full, tmem_empty, bias_full, pe);
    } else {
      const int n_pieces = *piece_n;
      int tt0 = 0;
#pragma unroll 1
      for (int pi = 0; pi < n_pieces; ++pi) {
        const Piece pc = piece_tab[pi];
        run_epilogue_piece<DENSE, PAIR, SEL>(p, pc.n, pc.tile0, pc.sub_base, pc.rb * BM, tt0, pc.zero_from, e, lane, tmem_base, bias_smem, share,
                                        smem + L.staging_off, tmem_full, tmem_empty, bias_full, pe);
        tt0 += pc.n;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if constexpr (CL != 0) cluster_sync_all();   // no CTA leaves while its peer may still write into it
  tc_fence_after();
  if (warp == 2) {
    if constexpr (PAIR) tmem_dealloc_pair<kTmemCols>(tmem_base);
    else tmem_dealloc<kTmemCols>(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------------------------
// encode_dense_split_kernel: the fp32-accurate dense encoder (exact mode of t_sae / of the q_sae dense path) in ONE
// launch. x = xh + xm + xl and W = wh + wm + wl (bf16 parts, both sums exact); the six partial products above 2^-24
// are contracted into the SAME TMEM accumulator, smallest first:
//     xl wh, xm wm, xh wl, xm wh, xh wm, xh wh        (K = 6 D in effect)
// so the dense fp32 output is written once (three launches that read-modify-wrote it took 2054 us against 595 us at
// B = 4096, profiles/r2s3_measurements.md 1). No x tile is resident: every ring stage carries one 128 x 64 chunk of an
// x part next to the CTA's half (128 latents) of the matching W chunk, the cta_group::2 pair executes M = 256 MMAs
// (CL = 2 of the kernel above), and the epilogue is the same dense epilogue (bias + activation, fp32 / hi / lo).
// The MMAs of a tile take six times as long as its drain, so the stores hide behind the tensor pipe here.
// Six 32 KiB stages next to the 32 KiB store staging area: 231.6 KB, all the shared memory a CTA can have (five stages:
// 620 us at B = 4096, H = 32768; six: 595 us -- this kernel is bound by the tensor pipe, and ring depth shows).
constexpr int kSplitStages = 6;
static_assert(kSplitStages * (kABytesPerChunk + kBBytesPerStage / 2) + 8 * 4096 + 2 * kEncBN * 4 + 8 * (2 * kSplitStages + 8) + 16
                  <= 227 * 1024, "encode_dense_split_kernel: shared memory budget");
constexpr int kSplitStageBytes = kABytesPerChunk + kBBytesPerStage / 2;   // 32 KiB: x chunk | my half of the W chunk
__host__ __device__ inline SmemLayout split_smem_layout() {
  SmemLayout L;
  L.a_off = 0;
  L.b_off = 0;
  L.staging_off = kSplitStages * kSplitStageBytes;
  L.bias_off = L.staging_off + epi_warps(true) * dense_stage_bytes(true);
  L.share_off = L.bias_off + 2 * BN * 4;
  L.bar_off = L.share_off;
  L.tmem_ptr_off = L.bar_off + 8 * (2 * kSplitStages + 8);
  L.piece_off = L.tmem_ptr_off + 16;
  L.total = L.piece_off;
  return L;
}

__global__ void __launch_bounds__(cta_threads(true), 1)
encode_dense_split_kernel(const __grid_constant__ CUtensorMap tmap_xh, const __grid_constant__ CUtensorMap tmap_xm,
                          const __grid_constant__ CUtensorMap tmap_xl, const __grid_constant__ CUtensorMap tmap_wh,
                          const __grid_constant__ CUtensorMap tmap_wm, const __grid_constant__ CUtensorMap tmap_wl,
                          EncodeLaunch p, int k_chunks, int n_prod, uint32_t prods) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const SmemLayout L = split_smem_layout();
  uint8_t* ring = smem;
  float* bias_smem = reinterpret_cast<float*>(smem + L.bias_off);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.bar_off);
  uint64_t* full = bars;
  uint64_t* empty = full + kSplitStages;
  uint64_t* tmem_full = empty + kSplitStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* bias_full = tmem_empty + 2;
  uint64_t* pair_empty = bias_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + L.tmem_ptr_off);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = cluster_ctarank();
  const bool leader = cta_rank == 0u;
  // Range schedule: the units are (pair of row blocks, tile) in row-block-major order; pair g of the gridDim.x / 2
  // pairs sweeps the contiguous units [u0, u1). Nothing is resident per row block, so a range may cross row blocks
  // freely and every pair gets the same number of units (+-1).
  const int n_tiles = p.n_tiles;
  const long long U = static_cast<long long>(((p.B + BM - 1) / BM + 1) / 2) * n_tiles;
  const long long G = gridDim.x / 2;
  const long long u0 = range_start(blockIdx.x / 2, U, G);
  const int n_my = static_cast<int>(range_start(blockIdx.x / 2 + 1, U, G) - u0);
  const int rbp0 = static_cast<int>(u0 / n_tiles);
  const int tile0 = static_cast<int>(u0 - static_cast<long long>(rbp0) * n_tiles);
  // products: (x part, W part) of product i = ((prods >> 4i + 2) & 3, (prods >> 4i) & 3), see the launcher.
  // n_prod = 6: the split-operand product; n_prod = 3: three x parts against one W part; n_prod = 1: only xh wh (the
  // single bf16 product of the fast-mode t_sae backward)
  const int k_iters = n_prod * k_chunks;

  if (threadIdx.x == 0) {
    if ((smem_u32(smem) & 1023u) != 0u) {
      printf("qsae: dynamic shared memory is not 1024-byte aligned\n");
      __trap();
    }
    for (int s = 0; s < kSplitStages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], epi_warps(true));
      mbar_init(&bias_full[a], 1);
      mbar_init(&pair_empty[a], 2 * epi_warps(true));
    }
    fence_mbar_init();
    fence_proxy_async_smem();
  }
  if (warp == 2) tmem_alloc_pair<kTmemCols>(tmem_ptr);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    if (lane == 0) {
      tma_prefetch_desc(&tmap_xh);
      tma_prefetch_desc(&tmap_wh);
      int stage = 0;
      uint32_t phase = 0;
      int rbp = rbp0, tile = tile0;
      for (int t = 0; t < n_my; ++t) {
        const int m0 = (2 * rbp + static_cast<int>(cta_rank)) * BM;
        const int n0 = tile * BN + static_cast<int>(cta_rank) * (BN / 2);
#pragma unroll 1
        for (int it = 0; it < k_iters; ++it) {
          const int pi = it / k_chunks, kc = it - pi * k_chunks;
          const uint32_t pr = prods >> (4 * pi);
          const uint32_t xi = (pr >> 2) & 3u, wi = pr & 3u;
          const CUtensorMap* tx = (xi == 2) ? &tmap_xl : (xi == 1 ? &tmap_xm : &tmap_xh);
          const CUtensorMap* tw = (wi == 2) ? &tmap_wl : (wi == 1 ? &tmap_wm : &tmap_wh);
          mbar_wait(&empty[stage], phase ^ 1u);
          const uint32_t full_leader = mapa_u32(smem_u32(&full[stage]), 0);
          if (leader) mbar_arrive_expect_tx(&full[stage], 2 * kSplitStageBytes);   // 32 KiB from each CTA
          uint8_t* dst = ring + stage * kSplitStageBytes;
          tma_load_2d_pair(dst, tx, full_leader, kc * BK, m0, kPolicyEvictLast);
          tma_load_2d_pair(dst + kABytesPerChunk, tw, full_leader, kc * BK, n0, kPolicyEvictLast);
          if (++stage == kSplitStages) { stage = 0; phase ^= 1u; }
        }
        if (++tile == n_tiles) { tile = 0; ++rbp; }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && leader) {
      constexpr uint32_t idesc = umma_idesc_bf16_f32(2 * BM, BN);
      const uint64_t a_desc0 = umma_desc_kmajor_sw128(smem_u32(ring));
      const uint64_t b_desc0 = umma_desc_kmajor_sw128(smem_u32(ring + kABytesPerChunk));
      int stage = 0;
      uint32_t phase = 0;
      for (int t = 0; t < n_my; ++t) {
        const int acc = t & 1;
        mbar_wait(&pair_empty[acc], ((t >> 1) & 1) ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
#pragma unroll 1
        for (int it = 0; it < k_iters; ++it) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint64_t so = static_cast<uint64_t>((stage * kSplitStageBytes) >> 4);
#pragma unroll
          for (int ks = 0; ks < BK / UMMA_K; ++ks)
            umma_f16_ss_pair(d_tmem, a_desc0 + so + ks * 2, b_desc0 + so + ks * 2, idesc, (it | ks) != 0 ? 1u : 0u);
          umma_commit_pair(&empty[stage], 0x3);
          if (it == k_iters - 1) umma_commit_pair(&tmem_full[acc], 0x3);
          if (++stage == kSplitStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 3) {
    int tile = tile0;
    for (int t = 0; t < n_my; ++t) {
      const int acc = t & 1;
      mbar_wait(&tmem_empty[acc], ((t >> 1) & 1) ^ 1u);
      const int n0 = tile * BN;
#pragma unroll
      for (int i = 0; i < BN / 32; ++i) {
        const int c = i * 32 + lane;
        bias_smem[acc * BN + c] = (p.bias != nullptr && n0 + c < p.H) ? __ldg(p.bias + n0 + c) : 0.f;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&bias_full[acc]);
      if (++tile == n_tiles) tile = 0;
    }
  } else if (warp >= 4) {
    // one call of the dense epilogue per row-block pair the range touches
    int rbp = rbp0, tile = tile0, done = 0;
#pragma unroll 1
    while (done < n_my) {
      const int n = min(n_my - done, n_tiles - tile);
      epilogue_dense<true>(p, n, tile, (2 * rbp + static_cast<int>(cta_rank)) * BM, done, warp - 4, lane, tmem_base, bias_smem,
                           smem + L.staging_off, tmem_full, tmem_empty, bias_full, pair_empty);
      done += n;
      tile = 0;
      ++rbp;
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  if (warp == 2) tmem_dealloc_pair<kTmemCols>(tmem_base);
}

// ---------------------------------------------------------------------------------------------------------
// prior_prep_kernel: cast + sample pre-pass + prior threshold in one launch (small batches; kernels.h PrepLaunch).
//
// Round 1 ran three launches before the sweep (cast 5 us, pre-pass 13.5 us, a sorting prior kernel 15 us at
// B = 4096: a quarter of the step). Here one cluster of NS CTAs per 128-row block does all of it:
//   * the eight epilogue warps read x in fp32, round it to bf16 and store it in the 128-byte-swizzled K-major
//     layout the UMMA descriptors expect (the layout TMA would have produced); CTA 0 of the cluster also writes the
//     row-major bf16 copy the sweep loads by TMA;
//   * the CTA contracts the x tile against ITS tiles of the sampled dictionary rows (TMA ring -> tcgen05.mma ->
//     TMEM, as in the sweep) and every epilogue thread keeps one running maximum per column class (column mod 32):
//     one FMNMX per element;
//   * the class maxima go to a padded shared-memory tile, the cluster synchronises, and CTA c computes the priors of
//     rows [128 c / NS, 128 (c + 1) / NS): a warp reads the row's NS x 64 maxima from all CTAs (distributed shared
//     memory) and bisects for the m-th largest.
// The m-th largest class maximum is a lower bound of the m-th largest sampled value (distinct elements) and equals
// it unless two of the row's top m fall into one of the 64 NS classes (17 % of the rows at m = 10, NS = 4: one rank
// looser, ~3 % more survivors). The sweep's result never depends on it (count check + exact rescue).
// ---------------------------------------------------------------------------------------------------------
constexpr int kPrepStages = 3;   // the exchange tile aliases the x operand (dead once the MMAs are done), which pays for the third stage
constexpr int kPrepPitch = 65;   // floats per row of the exchange tile: 2 x 32 class maxima + 1 (conflict-free both ways)

struct PrepSmem { uint32_t a_off, b_off, exch_off, bar_off, tmem_ptr_off, total; };
__host__ __device__ inline PrepSmem prep_smem_layout(int k_chunks) {
  PrepSmem L;
  L.a_off = 0;
  L.b_off = k_chunks * kABytesPerChunk;
  // class maxima over the x operand when it is large enough (k_chunks >= 3: 48 KB >= 33 KB), else behind the ring
  const uint32_t exch_bytes = ((BM * kPrepPitch * 4 + 15) / 16) * 16;
  const uint32_t ring_end = L.b_off + kPrepStages * kBBytesPerStage;
  const bool alias = static_cast<uint32_t>(k_chunks) * kABytesPerChunk >= exch_bytes;
  L.exch_off = alias ? L.a_off : ring_end;
  L.bar_off = alias ? ring_end : ring_end + exch_bytes;
  L.tmem_ptr_off = L.bar_off + 8 * (k_chunks + 2 * kPrepStages + 4);
  L.total = L.tmem_ptr_off + 16;
  return L;
}

template <int K_CHUNKS, int NS>
__global__ void __launch_bounds__(384, 1)
prior_prep_kernel(const __grid_constant__ CUtensorMap tmap_w, PrepLaunch p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const PrepSmem L = prep_smem_layout(K_CHUNKS);
  uint8_t* a_smem = smem + L.a_off;
  uint8_t* b_smem = smem + L.b_off;
  float* exch = reinterpret_cast<float*>(smem + L.exch_off);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.bar_off);
  uint64_t* a_full = bars;                            // one per 64-column chunk of x: the MMAs start on chunk 0
  uint64_t* full = bars + K_CHUNKS;                   // while the later chunks are still being converted
  uint64_t* empty = full + kPrepStages;
  uint64_t* tmem_full = empty + kPrepStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(smem + L.tmem_ptr_off);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();            // == blockIdx.x: the cluster spans grid.x
  const int m0 = blockIdx.y * BM;
  const int n_tiles = (p.n_sample + BN - 1) / BN;
  const int tiles_per_cta = (n_tiles + NS - 1) / NS;
  const int tile_begin = static_cast<int>(rank) * tiles_per_cta;
  const int n_my_tiles = max(0, min(n_tiles, tile_begin + tiles_per_cta) - tile_begin);

  if (threadIdx.x == 0) {
    if ((smem_u32(smem) & 1023u) != 0u) {
      printf("qsae: dynamic shared memory is not 1024-byte aligned\n");
      __trap();
    }
    for (int kc = 0; kc < K_CHUNKS; ++kc) mbar_init(&a_full[kc], 12);   // one arrival per converting warp
    for (int s = 0; s < kPrepStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tmem_full[a], 1); mbar_init(&tmem_empty[a], 8); }
    fence_mbar_init();
    fence_proxy_async_smem();
    if (p.zero_counters != nullptr && blockIdx.x == 0 && blockIdx.y == 0) {
      for (int i = 0; i < kPriorCounters; ++i) p.zero_counters[i] = 0;
    }
  }
  if (warp == 2) tmem_alloc<kTmemCols>(tmem_ptr);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  // ------------------------------------------------------------- x -> bf16 operand (all twelve warps)
  // unit = 8 consecutive columns of one row = one 16-byte swizzle unit; consecutive threads take consecutive units,
  // so a warp reads 1 KB of one fp32 row and writes 4 x 128 contiguous bytes of shared memory. 16 loads of 16 bytes
  // in flight per thread (96 KB per SM): the copy is bound by latency x bytes in flight, not by bandwidth.
  if (warp == 0 && lane == 0 && n_my_tiles > 0) {
    // the first W stages travel while x is being converted
    tma_prefetch_desc(&tmap_w);
    for (int st0 = 0; st0 < kPrepStages && st0 < K_CHUNKS; ++st0) {
      mbar_arrive_expect_tx(&full[st0], kBBytesPerStage);
      tma_load_2d(b_smem + st0 * kBBytesPerStage, &tmap_w, &full[st0], st0 * BK, tile_begin * BN, kPolicyEvictLast);
    }
  }
  {
    // chunk-major order: unit u = (chunk u / 1024, row (u % 1024) / 8, 16-byte unit u % 8), so that the first chunks
    // of the operand are complete (and their barrier arrives) while the later ones are still in flight
    constexpr int kUnitsPerChunk = BM * 8;
    constexpr int kUnits = K_CHUNKS * kUnitsPerChunk;
    const bool write_global = rank == 0u;
    constexpr int BATCH = 8;
    constexpr int kPerIter = 384 * BATCH;              // 3 chunks per iteration
    static_assert(kPerIter % kUnitsPerChunk == 0, "an iteration must cover whole chunks");
#pragma unroll 1
    for (int u0 = threadIdx.x; u0 < kUnits; u0 += kPerIter) {
      float4 lo[BATCH], hi[BATCH];
#pragma unroll
      for (int i = 0; i < BATCH; ++i) {
        const int u = u0 + i * 384;
        const int kc = u / kUnitsPerChunk, r = (u % kUnitsPerChunk) >> 3, c8 = kc * BK + (u & 7) * 8;
        lo[i] = hi[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (u < kUnits && m0 + r < p.B && c8 < p.D) {
          const float4* src = reinterpret_cast<const float4*>(p.x_f32 + static_cast<size_t>(m0 + r) * p.D + c8);
          lo[i] = __ldg(src);
          hi[i] = __ldg(src + 1);
        }
      }
#pragma unroll
      for (int i = 0; i < BATCH; ++i) {
        const int u = u0 + i * 384;
        if (u >= kUnits) continue;
        const int kc = u / kUnitsPerChunk, r = (u % kUnitsPerChunk) >> 3, j = u & 7;
        const uint32_t w0 = pack_bf16x2(lo[i].x, lo[i].y), w1 = pack_bf16x2(lo[i].z, lo[i].w);
        const uint32_t w2 = pack_bf16x2(hi[i].x, hi[i].y), w3 = pack_bf16x2(hi[i].z, hi[i].w);
        st_shared_v4(smem_u32(a_smem) + kc * kABytesPerChunk + r * 128 + ((j ^ (r & 7)) << 4), w0, w1, w2, w3);
        const int c8 = kc * BK + j * 8;
        if (write_global && m0 + r < p.B && c8 < p.D)
          *reinterpret_cast<uint4*>(p.x_bf16 + static_cast<size_t>(m0 + r) * p.D + c8) = make_uint4(w0, w1, w2, w3);
      }
      fence_proxy_async_smem();     // generic-proxy stores -> visible to the tensor-core (async proxy) reads
      __syncwarp();
      if (lane == 0) {
        const int c_begin = (u0 - static_cast<int>(threadIdx.x)) / kUnitsPerChunk;
        const int c_end = min(K_CHUNKS, c_begin + kPerIter / kUnitsPerChunk);
        for (int kc = c_begin; kc < c_end; ++kc) mbar_arrive(&a_full[kc]);
      }
    }
  }

  // The class maxima are written over the x operand. A CTA with tiles writes them after its last accumulator is
  // complete (every MMA has read the operand); a CTA without tiles must see all twelve warps' conversion stores first.
  if (n_my_tiles == 0) __syncthreads();

  if (warp == 0) {
    // ------------------------------------------------------------- TMA producer: my tiles of the sampled rows
    if (lane == 0 && n_my_tiles > 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = 0; t < n_my_tiles; ++t) {
        const int n0 = (tile_begin + t) * BN;
#pragma unroll 1
        for (int kc = 0; kc < K_CHUNKS; ++kc) {
          if (t > 0 || kc >= kPrepStages) {     // the first stages were issued before the conversion
            mbar_wait(&empty[stage], phase ^ 1u);
            mbar_arrive_expect_tx(&full[stage], kBBytesPerStage);
            tma_load_2d(b_smem + stage * kBBytesPerStage, &tmap_w, &full[stage], kc * BK, n0, kPolicyEvictLast);
          }
          if (++stage == kPrepStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------- MMA issuer
    if (lane == 0 && n_my_tiles > 0) {
      constexpr uint32_t idesc = umma_idesc_bf16_f32(BM, BN);
      const uint64_t a_desc0 = umma_desc_kmajor_sw128(smem_u32(a_smem));
      const uint64_t b_desc0 = umma_desc_kmajor_sw128(smem_u32(b_smem));
      int stage = 0;
      uint32_t phase = 0;
      for (int t = 0; t < n_my_tiles; ++t) {
        const int acc = t & 1;
        mbar_wait(&tmem_empty[acc], ((t >> 1) & 1) ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
#pragma unroll 1
        for (int kc = 0; kc < K_CHUNKS; ++kc) {
          if (t == 0) mbar_wait(&a_full[kc], 0);     // this chunk of the x operand has been converted
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint64_t a_desc = a_desc0 + static_cast<uint64_t>((kc * kABytesPerChunk) >> 4);
          const uint64_t b_desc = b_desc0 + static_cast<uint64_t>((stage * kBBytesPerStage) >> 4);
#pragma unroll
          for (int ks = 0; ks < BK / UMMA_K; ++ks)
            umma_f16_ss(d_tmem, a_desc + ks * 2, b_desc + ks * 2, idesc, (kc | ks) != 0 ? 1u : 0u);
          umma_commit(&empty[stage]);
          if (kc == K_CHUNKS - 1) umma_commit(&tmem_full[acc]);
          if (++stage == kPrepStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------- class maxima of my sample tiles
    const int e = warp - 4;
    const int quad = e & 3;       // TMEM lanes 32*quad .. +31 (hardware: warp_id % 4)
    const int half = e >> 2;      // columns [half*128, half*128+128) of the tile
    const int row_in_tile = quad * 32 + lane;
    const uint32_t lane_taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    float top[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) top[j] = -INFINITY;
    for (int t = 0; t < n_my_tiles; ++t) {
      const int acc = t & 1;
      mbar_wait(&tmem_full[acc], (t >> 1) & 1);
      tc_fence_after();
      const int n_tile = (tile_begin + t) * BN + half * 128;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        uint32_t r[32];
        tmem_ld_32x32b_x32(lane_taddr + acc * BN + half * 128 + c * 32, r);
        tmem_ld_wait();
        const int col0 = n_tile + c * 32;
        if (col0 + 32 <= p.n_sample) {
          const float4* bias4 = reinterpret_cast<const float4*>(p.bias + col0);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 b = __ldg(bias4 + j);
            float v0 = __uint_as_float(r[4 * j + 0]) + b.x, v1 = __uint_as_float(r[4 * j + 1]) + b.y;
            float v2 = __uint_as_float(r[4 * j + 2]) + b.z, v3 = __uint_as_float(r[4 * j + 3]) + b.w;
            if (p.act == 1) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); v2 = fmaxf(v2, 0.f); v3 = fmaxf(v3, 0.f); }
            top[4 * j + 0] = fmaxf(top[4 * j + 0], v0);
            top[4 * j + 1] = fmaxf(top[4 * j + 1], v1);
            top[4 * j + 2] = fmaxf(top[4 * j + 2], v2);
            top[4 * j + 3] = fmaxf(top[4 * j + 3], v3);
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            if (col0 + j < p.n_sample) {
              float v = __uint_as_float(r[j]) + __ldg(p.bias + col0 + j);
              if (p.act == 1) v = fmaxf(v, 0.f);
              top[j] = fmaxf(top[j], v);
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);
    }
    // row-major padded tile: thread (row, half) writes 32 consecutive floats; lanes = rows, pitch 65 words
#pragma unroll
    for (int j = 0; j < 32; ++j) exch[row_in_tile * kPrepPitch + half * 32 + j] = top[j];
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();          // every CTA's class maxima are in place (release / acquire at cluster scope)

  // ------------------------------------------------------------- priors of my share of the row block
  {
    constexpr int kRowsPerCta = BM / NS;
    constexpr int NV = 2 * NS;                 // values per lane: NS CTAs x 2 column halves, class = lane
    const unsigned fullmask = 0xffffffffu;
    for (int rr = warp; rr < kRowsPerCta; rr += 12) {
      const int r = static_cast<int>(rank) * kRowsPerCta + rr;
      const int row = m0 + r;
      if (row >= p.B) continue;               // warp-uniform
      uint32_t key[NV];
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const uint32_t addr = smem_u32(exch + r * kPrepPitch + (i & 1) * 32 + lane);
        key[i] = float_to_key(ld_dsmem_f32(addr, static_cast<uint32_t>(i >> 1)));
      }
      // m-th largest of the 32 NV keys: m rounds of "take the maximum, retire every key equal to it". Equal keys
      // retire together, so with ties the result is at most the true m-th largest: still a valid lower bound.
      uint32_t T = 0u;
#pragma unroll 1
      for (int round = 0; round < p.m; ++round) {
        uint32_t mx = key[0];
#pragma unroll
        for (int i = 1; i < NV; ++i) mx = max(mx, key[i]);
        T = __reduce_max_sync(fullmask, mx);
#pragma unroll
        for (int i = 0; i < NV; ++i) key[i] = (key[i] == T) ? 0u : key[i];
      }
      if (lane == 0) p.prior[row] = key_to_float(T);
    }
  }

  cluster_sync_all();          // no CTA leaves while a peer may still read its class maxima
  tc_fence_after();
  if (warp == 2) tmem_dealloc<kTmemCols>(tmem_base);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* ptr = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) !=
          cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(ptr);
  return fn;
}

// row-major [rows, cols] -> 2D tensor map with a {box_cols x box_rows} box
bool make_tmap_2d(CUtensorMap* map, CUtensorMapDataType dtype, int elem_bytes, const void* base, int rows, int cols,
                  int box_cols, int box_rows, CUtensorMapSwizzle swizzle) {
  EncodeTiledFn enc = get_encode_tiled();
  if (!enc) return false;
  const TmapKey key{base, static_cast<unsigned long long>(rows), static_cast<unsigned long long>(cols),
                    static_cast<unsigned long long>(cols) * elem_bytes, static_cast<unsigned int>(box_cols),
                    static_cast<unsigned int>(box_rows), static_cast<int>(dtype), static_cast<int>(swizzle), tmap_current_device()};
  return tmap_cache().get(key, map, [&](CUtensorMap* m) {
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(cols) * elem_bytes};
    cuuint32_t box[2] = {static_cast<cuuint32_t>(box_cols), static_cast<cuuint32_t>(box_rows)};
    cuuint32_t estr[2] = {1, 1};
    return enc(m, dtype, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle,
               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
  });
}
// bf16 operand tile: {64 x box_rows} box, 128-byte swizzle
bool make_tmap_bf16(CUtensorMap* map, const void* base, int rows, int cols, int box_rows) {
  return make_tmap_2d(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, rows, cols, BK, box_rows,
                      CU_TENSOR_MAP_SWIZZLE_128B);
}

template <int K_CHUNKS, bool DENSE, int CL, int SEL>
cudaError_t launch_k(const CUtensorMap& tx, const CUtensorMap& tw, const EncodeLaunch& p, cudaStream_t stream) {
  const SmemLayout L = smem_layout(K_CHUNKS, DENSE, CL >= 2);
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(encode_topk_kernel<K_CHUNKS, DENSE, CL, SEL>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, L.total);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  dim3 grid(p.n_splits, (p.B + BM - 1) / BM);
  if (CL == 0 && p.range_g > 0) grid = dim3(p.range_g, 1);
  if constexpr (CL != 0) {
    // whole clusters along x; the padding CTA sweeps zero rows and writes nothing
    grid = dim3(((p.B + BM - 1) / BM + 1) / 2 * 2, p.n_splits);
    if (CL == 3) grid = dim3(2 * p.range_g, 1);   // range_g pairs, one CTA per SM
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(cta_threads(DENSE));
    cfg.dynamicSmemBytes = L.total;
    cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, encode_topk_kernel<K_CHUNKS, DENSE, CL, SEL>, tx, tw, p);
  } else {
    encode_topk_kernel<K_CHUNKS, DENSE, CL, SEL><<<grid, cta_threads(DENSE), L.total, stream>>>(tx, tw, p);
    return cudaGetLastError();
  }
}

template <bool DENSE, int SEL>
cudaError_t launch_kc(const CUtensorMap& tx, const CUtensorMap& tw, const EncodeLaunch& p, cudaStream_t stream) {
  switch ((p.D + BK - 1) / BK) {
    case 1: return launch_k<1, DENSE, 0, SEL>(tx, tw, p, stream);
    case 2: return launch_k<2, DENSE, 0, SEL>(tx, tw, p, stream);
    case 3: return launch_k<3, DENSE, 0, SEL>(tx, tw, p, stream);
    case 4: return launch_k<4, DENSE, 0, SEL>(tx, tw, p, stream);
    case 5: return launch_k<5, DENSE, 0, SEL>(tx, tw, p, stream);
    case 6: return launch_k<6, DENSE, 0, SEL>(tx, tw, p, stream);
    case 7: return launch_k<7, DENSE, 0, SEL>(tx, tw, p, stream);
    default:   // the headline width: the cluster variants exist here (launch_any has checked D <= 512)
      if constexpr (!DENSE) {   // the dense epilogue has the single-CTA and the cta_group::2 variants only
        if (p.cluster == 3) return launch_k<8, DENSE, 3, SEL>(tx, tw, p, stream);
        if (p.cluster == 1) return launch_k<8, DENSE, 1, SEL>(tx, tw, p, stream);
      }
      if (p.cluster == 2) return launch_k<8, DENSE, 2, SEL>(tx, tw, p, stream);
      return launch_k<8, DENSE, 0, SEL>(tx, tw, p, stream);
  }
}

// Prior-threshold sweeps (mode 4) run on the kernel compiled for that mode alone unless QSAE_ENCODE_SPECIALISED=0;
// the dense dump (debug_z) exists in the generic kernel only.
template <bool DENSE>
const char* launch_any(const CUtensorMap& tx, const CUtensorMap& tw, const EncodeLaunch& p, cudaStream_t stream) {
  const int kc = (p.D + BK - 1) / BK;
  if (kc < 1 || kc > 8) return "D must be <= 512";
  if (p.cluster == 3 && kc != 8) return "the pair range schedule exists for D > 448 only";
  cudaError_t e;
  if constexpr (!DENSE) {
    if (p.mode == 4 && p.debug_z == nullptr && tuning().encode_specialised != 0)
      e = launch_kc<false, 4>(tx, tw, p, stream);
    else
      e = launch_kc<false, -1>(tx, tw, p, stream);
  } else {
    e = launch_kc<true, -1>(tx, tw, p, stream);
  }
  return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
}

// Cluster variant of a launch: 0 single CTA, 1 multicast pair, 2 cta_group::2 pair. Pairs need two row
// blocks. QSAE_ENCODE_CLUSTER overrides the default (tests and tuning experiments).
int pick_cluster(const EncodeLaunch& p, int dflt) {
  if (tuning().encode_cluster >= 0) dflt = tuning().encode_cluster;
  if (dflt < 0 || dflt > 2 || p.D <= 448 || p.B <= BM) return 0;
  return dflt;
}

}  // namespace

int encode_pick_splits(int B, int H, int num_sms) {
  const int m_tiles = (B + BM - 1) / BM;
  const int n_tiles = (H + BN - 1) / BN;
  int best_s = 1;
  double best = -1.0;
  for (int s = 1; s <= kMaxSplits && s <= n_tiles; s *= 2) {
    const long units = static_cast<long>(m_tiles) * s;
    const long waves = (units + num_sms - 1) / num_sms;
    const int tps = (n_tiles + s - 1) / s;
    // fraction of SM-time doing useful tiles: wave fill x split balance
    const double eff = (static_cast<double>(units) / (waves * num_sms)) *
                       (static_cast<double>(n_tiles) / (static_cast<double>(tps) * s));
    if (eff > best * 1.03) { best = eff; best_s = s; }
  }
  // no split without tiles (9 tiles over 8 splits of 2 leave 3 empty): the cluster variants launch no epilogue for an
  // empty split, so its survivor-list counts would never be written. The same tile ranges over fewer splits.
  const int tps = (n_tiles + best_s - 1) / best_s;
  return (n_tiles + tps - 1) / tps;
}

int encode_pick_range(int B, int H, int num_sms, int* nsub, int* pair) {
  *nsub = 0;
  if (pair) *pair = 0;
  if (tuning().encode_range == 0 || B >= 16384) return 0;   // large batches: the multicast pairs take over
  const long long m_tiles = (B + BM - 1) / BM;
  const long long n_tiles = (H + BN - 1) / BN;
  const long long U = m_tiles * n_tiles;
  const int s = encode_pick_splits(B, H, num_sms);
  const long long units = m_tiles * s;
  const long long waves = (units + num_sms - 1) / num_sms;
  const long long tps = (n_tiles + s - 1) / s;
  const double eff = (static_cast<double>(units) / (waves * num_sms)) *
                     (static_cast<double>(n_tiles) / (static_cast<double>(tps) * s));
  if (eff >= 0.95 || U < 2ll * num_sms) return 0;
  // cta_group::2 pairs on the range schedule: the units are (pair of row blocks, tile), one pair per two SMs. Halves the
  // W bytes every SM pulls from L2 (the single-CTA sweep runs at the L2 slice limit: 3.5 us per tile against 3.1 us
  // for the pair). Needs whole pairs of full row blocks.
  const bool use_pair = pair != nullptr && tuning().encode_range_pair != 0 && (B % (2 * BM)) == 0 && (num_sms % 2) == 0 &&
                        (H % BN) == 0 && U / 2 >= num_sms;
  const long long G = use_pair ? num_sms / 2 : num_sms;
  const long long rbs = use_pair ? m_tiles / 2 : m_tiles;
  const long long Ur = rbs * n_tiles;
  int max_pieces = 1;
  for (long long rb = 0; rb < rbs; ++rb) {
    const int pieces = range_owner(rb * n_tiles + n_tiles - 1, Ur, G) - range_owner(rb * n_tiles, Ur, G) + 1;
    if (pieces > max_pieces) max_pieces = pieces;
  }
  if (2 * max_pieces > 32) return 0;   // the warp-level merge reads at most 32 lists per row
  const long long range_len = (Ur + G - 1) / G;
  if ((range_len + n_tiles - 1) / n_tiles + 1 > kMaxPieces) return 0;   // pieces of one CTA's range (its piece table)
  *nsub = 2 * max_pieces;
  if (pair) *pair = use_pair ? 1 : 0;
  return static_cast<int>(G);
}

void encode_pick_mode(int k_sel, int* mode, int* cap) {
  *cap = kCandCapMax;
  if (k_sel <= 32) *mode = 1;
  else if (k_sel <= 64) *mode = 2;
  else if (k_sel <= 128) *mode = 3;
  else *mode = 0;
}

// tensor map of W with the box the cluster variant loads (256 latents, or 128 per CTA of a pair)
const char* make_w_map(CUtensorMap* tw, const uint16_t* w_bf16, const EncodeLaunch& p) {
  if (!make_tmap_bf16(tw, w_bf16, p.H, p.D, p.cluster ? BN / 2 : BN)) return "cuTensorMapEncodeTiled(W) failed";
  return nullptr;
}

const char* encode_topk_launch(const uint16_t* x_bf16, const uint16_t* w_bf16, EncodeLaunch p,
                               cudaStream_t stream) {
  CUtensorMap tx;
  if (!make_tmap_bf16(&tx, x_bf16, p.B, p.D, BM)) return "cuTensorMapEncodeTiled(x) failed";
  p.dense_flags = 0;
  p.cluster = p.range_g > 0 ? (p.range_pair ? 3 : 0) : pick_cluster(p, p.B >= 16384 ? 1 : 0);
  CUtensorMap tw;
  if (const char* err = make_w_map(&tw, w_bf16, p)) return err;
  return launch_any<false>(tx, tw, p, stream);
}

const char* encode_dense_tc_launch(const uint16_t* x_bf16, const uint16_t* w_bf16, EncodeLaunch p, float* out_f32,
                                   uint16_t* out_hi, uint16_t* out_lo, cudaStream_t stream) {
  if ((p.H % 8) != 0) return "dense tensor-core encoder needs H % 8 == 0";
  if ((reinterpret_cast<uintptr_t>(out_f32) | reinterpret_cast<uintptr_t>(out_hi) | reinterpret_cast<uintptr_t>(out_lo)) & 15)
    return "dense tensor-core encoder: outputs must be 16-byte aligned";
  if (p.act == 2 && (!p.step_scale || !p.step_level_start || !p.step_level_count || (p.H % 128) != 0))
    return "dense encoder: the step-operand epilogue needs scale / levels / counts and H % 128 == 0";
  if (p.act == 3) return "dense encoder: the ReLU-backward epilogue runs on the streamed-operand kernel only";
  CUtensorMap tx;
  if (!make_tmap_bf16(&tx, x_bf16, p.B, p.D, BM)) return "cuTensorMapEncodeTiled(x) failed";
  p.out_f32 = out_f32; p.out_hi = out_hi; p.out_lo = out_lo;
  p.dense_flags = (out_f32 ? 1 : 0) | (out_hi ? 2 : 0) | (out_lo ? 4 : 0);
  if (p.dense_flags == 0) return "dense encoder: no output requested";
  p.range_g = 0;
  p.cluster = pick_cluster(p, kDefaultClusterDense);
  if (p.cluster == 1) p.cluster = kDefaultClusterDense;   // no multicast variant: it gained nothing here (DESIGN.md 5.1)
  CUtensorMap tw;
  if (const char* err = make_w_map(&tw, w_bf16, p)) return err;
  return launch_any<true>(tx, tw, p, stream);
}

const char* encode_dense_split_launch(const uint16_t* const* x_parts, const uint16_t* const* w_parts, int n_parts, EncodeLaunch p,
                                      float* out_f32, uint16_t* out_hi, uint16_t* out_lo, int num_sms, cudaStream_t stream,
                                      int n_w_parts) {
  if (n_w_parts == 0) n_w_parts = n_parts;
  if (n_parts != 1 && n_parts != 3) return "dense tensor-core encoder (streamed operands): 1 or 3 parts per operand";
  if (n_w_parts != n_parts && !(n_parts == 3 && n_w_parts == 1))
    return "dense tensor-core encoder (streamed operands): 1 x 1, 3 x 3 or 3 x 1 parts";
  if ((p.H % 8) != 0) return "dense tensor-core encoder needs H % 8 == 0";
  if (p.act == 3 && (!p.gate || out_lo || p.bias != nullptr))
    return "dense encoder: the ReLU-backward epilogue needs the gate, writes fp32 and / or bf16 hi, and takes no bias";
  if ((reinterpret_cast<uintptr_t>(out_f32) | reinterpret_cast<uintptr_t>(out_hi) | reinterpret_cast<uintptr_t>(out_lo)) & 15)
    return "dense tensor-core encoder: outputs must be 16-byte aligned";
  if (p.act == 2 && (!p.step_scale || !p.step_level_start || !p.step_level_count || (p.H % 128) != 0))
    return "dense encoder: the step-operand epilogue needs scale / levels / counts and H % 128 == 0";
  p.out_f32 = out_f32; p.out_hi = out_hi; p.out_lo = out_lo;
  p.range_g = 0;
  p.cluster = 2;
  p.dense_flags = (out_f32 ? 1 : 0) | (out_hi ? 2 : 0) | (out_lo ? 4 : 0);
  if (p.dense_flags == 0) return "dense encoder: no output requested";
  CUtensorMap tx[3], tw[3];
  for (int i = 0; i < 3; ++i) {
    if (!make_tmap_bf16(&tx[i], x_parts[i < n_parts ? i : 0], p.B, p.D, BM)) return "cuTensorMapEncodeTiled(x part) failed";
    if (!make_tmap_bf16(&tw[i], w_parts[i < n_w_parts ? i : 0], p.H, p.D, BN / 2)) return "cuTensorMapEncodeTiled(W part) failed";
  }
  // product list (x part, W part), smallest first: 3 x 3: xl wh, xm wm, xh wl, xm wh, xh wm, xh wh;
  // 3 x 1: xl wh, xm wh, xh wh; 1 x 1: xh wh
  static const uint32_t kSix[6][2] = {{2, 0}, {1, 1}, {0, 2}, {1, 0}, {0, 1}, {0, 0}};
  static const uint32_t kThree[3][2] = {{2, 0}, {1, 0}, {0, 0}};
  int n_prod = 1;
  uint32_t prods = 0u;
  if (n_parts == 3) {
    n_prod = n_w_parts == 3 ? 6 : 3;
    for (int i = 0; i < n_prod; ++i) {
      const uint32_t* pr = n_prod == 6 ? kSix[i] : kThree[i];
      prods |= ((pr[0] << 2) | pr[1]) << (4 * i);
    }
  }
  const SmemLayout L = split_smem_layout();
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(encode_dense_split_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, L.total);
    if (e != cudaSuccess) return cudaGetErrorString(e);
    attr_set = true;
  }
  cudaLaunchConfig_t cfg = {};
  // range schedule over CTA pairs: one pair per two SMs, or one per unit when there are fewer units than that
  const long long units = static_cast<long long>(((p.B + BM - 1) / BM + 1) / 2) * p.n_tiles;
  int n_pairs = num_sms / 2;
  if (units < n_pairs) n_pairs = static_cast<int>(units);
  cfg.gridDim = dim3(2 * n_pairs, 1);
  cfg.blockDim = dim3(cta_threads(true));
  cfg.dynamicSmemBytes = L.total;
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  const int k_chunks = (p.D + BK - 1) / BK;
  cudaError_t e = cudaLaunchKernelEx(&cfg, encode_dense_split_kernel, tx[0], tx[1], tx[2], tw[0], tw[1], tw[2], p, k_chunks,
                                     n_prod, prods);
  return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
}


namespace {
template <int K_CHUNKS, int NS>
cudaError_t launch_prep(const CUtensorMap& tw, const PrepLaunch& p, cudaStream_t stream) {
  const PrepSmem L = prep_smem_layout(K_CHUNKS);
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(prior_prep_kernel<K_CHUNKS, NS>, cudaFuncAttributeMaxDynamicSharedMemorySize, L.total);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(NS, (p.B + BM - 1) / BM);
  cfg.blockDim = dim3(384);
  cfg.dynamicSmemBytes = L.total;
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = NS;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, prior_prep_kernel<K_CHUNKS, NS>, tw, p);
}
}  // namespace

int prior_prep_pick_ns(int B, int D, int n_sample, int m, int num_sms) {
  if (tuning().prior_prep == 0) return 0;   // always the separate cast / pre-pass / prior kernels
  if (D != 512 && D != 256) return 0;                  // instantiated widths (the benchmark shapes)
  if (n_sample < 512 || m < 1 || m > 32) return 0;
  const int m_tiles = (B + BM - 1) / BM;
  const int n_tiles = (n_sample + BN - 1) / BN;
  if (4 * m_tiles <= num_sms - num_sms % 4 && n_tiles >= 4) return 4;
  if (2 * m_tiles <= num_sms - num_sms % 2 && n_tiles >= 2) return 2;
  return 0;
}

const char* prior_prep_launch(const uint16_t* w_sample, const PrepLaunch& p, cudaStream_t stream) {
  CUtensorMap tw;
  if (!make_tmap_bf16(&tw, w_sample, p.n_sample, p.D, BN)) return "cuTensorMapEncodeTiled(W sample) failed";
  cudaError_t e;
  if (p.D == 512 && p.ns == 4) e = launch_prep<8, 4>(tw, p, stream);
  else if (p.D == 512 && p.ns == 2) e = launch_prep<8, 2>(tw, p, stream);
  else if (p.D == 256 && p.ns == 4) e = launch_prep<4, 4>(tw, p, stream);
  else if (p.D == 256 && p.ns == 2) e = launch_prep<4, 2>(tw, p, stream);
  else return "prior_prep: unsupported shape";
  return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
}

}  // namespace qsae
