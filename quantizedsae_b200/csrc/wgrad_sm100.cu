// Weight-gradient GEMM for sm_100a:  C[M, N] = sum_k A(k, m) B(k, n),  bf16 operands, fp32 accumulation in TMEM.
//
// The backward of a dense layer contracts over the batch (t_sae, training.py): grad encoder.0.weight = gz^T x [H, D]
// and grad decoder.weight = g^T h [D, H]. Both operands are the row-major batch tensors as they are, A = [K, M] and
// B = [K, N]: MN-major UMMA operands, so no [B, H] tensor is ever transposed. A TMA box of 64 columns x 64 batch rows
// with the 128-byte swizzle lands as one MN-major column of atoms (64 rows of 128 B); a stage holds two such columns
// of A (128 rows of the output) and four of B (256 columns). The batch is K and may have any length: TMA zero-fills
// the tail rows, and columns past M or N.
//
// A may instead be K-major, [M, K] row-major (x.grad = gz W_enc contracts over H, and gz is [B, H]).
//
// Products: a list of (A part, B part) pairs contracted into the SAME accumulator. Fast mode is one bf16 product;
// exact mode splits both fp32 operands into three bf16 parts and keeps the six partial products above 2^-24,
// smallest first (the order of encode_dense_split_kernel).
//
// Persistent CTAs over 128 x 256 output tiles (the dimension with fewer tiles runs fastest, so the CTAs working at
// the same time share the slice of the large operand in L2), a 4-stage ring of 48 KiB stages, and two TMEM
// accumulators: the epilogue drains tile t while the MMAs of tile t + 1 run.
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include "kernels.h"
#include "ptx_sm100.cuh"
#include "tmap_cache.cuh"

namespace qsae {

namespace {

constexpr int BM = 128, BN = 256, BK = 64, UMMA_K = 16;
constexpr int kABytes = BM * BK * 2;        // 16 KiB: two MN columns of 64 rows x 128 B (or 128 K-major rows)
constexpr int kBBytes = BN * BK * 2;        // 32 KiB: four MN columns
constexpr int kColBytes = BK * 128;         // one MN column of atoms: 64 K rows x 128 B
constexpr int kStageBytes = kABytes + kBBytes;
constexpr int kStages = 4;
constexpr int kThreads = 256;               // warps: 0 TMA, 1 MMA, 2 TMEM alloc, 3 idle, 4-7 epilogue
constexpr int kTmemCols = 2 * BN;           // two accumulators
constexpr int kBarOff = kStages * kStageBytes;
constexpr int kSmem = kBarOff + 8 * (2 * kStages + 4) + 16;
static_assert(kSmem <= 227 * 1024, "wgrad_kernel: shared memory budget");

struct WgradParams {
  int M, N;
  int m_tiles, n_tiles;
  int k_chunks;          // ceil(K / 64)
  int n_prod;
  uint32_t prods;        // product i: A part (prods >> 4i + 2) & 3, B part (prods >> 4i) & 3
  int a_kmajor;
  int m_fast;            // tile u -> (u % m_tiles, u / m_tiles), else (u / n_tiles, u % n_tiles)
  float* c;              // [M, N] row-major
};

template <bool A_KMAJOR>
__global__ void __launch_bounds__(kThreads, 1)
wgrad_kernel(const __grid_constant__ CUtensorMap ta0, const __grid_constant__ CUtensorMap ta1,
             const __grid_constant__ CUtensorMap ta2, const __grid_constant__ CUtensorMap tb0,
             const __grid_constant__ CUtensorMap tb1, const __grid_constant__ CUtensorMap tb2, WgradParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kBarOff);
  uint64_t* full = bars;
  uint64_t* empty = bars + kStages;
  uint64_t* tmem_full = bars + 2 * kStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_units = p.m_tiles * p.n_tiles;
  const int k_iters = p.n_prod * p.k_chunks;
  auto tile_of = [&](int u, int* m0, int* n0) {
    const int mt = p.m_fast ? u % p.m_tiles : u / p.n_tiles;
    const int nt = p.m_fast ? u / p.m_tiles : u % p.n_tiles;
    *m0 = mt * BM;
    *n0 = nt * BN;
  };

  if (threadIdx.x == 0) {
    if ((smem_u32(smem) & 1023u) != 0u) {
      printf("qsae: dynamic shared memory is not 1024-byte aligned\n");
      __trap();
    }
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], 4);
    }
    fence_mbar_init();
    fence_proxy_async_smem();
  }
  if (warp == 2) tmem_alloc<kTmemCols>(tmem_ptr);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    if (lane == 0) {
      tma_prefetch_desc(&ta0);
      tma_prefetch_desc(&tb0);
      int stage = 0;
      uint32_t phase = 0;
      for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
        int m0, n0;
        tile_of(u, &m0, &n0);
#pragma unroll 1
        for (int it = 0; it < k_iters; ++it) {
          const int pi = it / p.k_chunks, kc = it - pi * p.k_chunks;
          const uint32_t pr = p.prods >> (4 * pi);
          const int ai = (pr >> 2) & 3, bi = pr & 3;
          const CUtensorMap* ta = ai == 0 ? &ta0 : (ai == 1 ? &ta1 : &ta2);
          const CUtensorMap* tb = bi == 0 ? &tb0 : (bi == 1 ? &tb1 : &tb2);
          mbar_wait(&empty[stage], phase ^ 1u);
          uint8_t* st = smem + stage * kStageBytes;
          mbar_arrive_expect_tx(&full[stage], kStageBytes);
          const int k0 = kc * BK;
          if constexpr (A_KMAJOR) {
            tma_load_2d(st, ta, &full[stage], k0, m0, kPolicyEvictNormal);
          } else {
#pragma unroll
            for (int c = 0; c < BM / 64; ++c) tma_load_2d(st + c * kColBytes, ta, &full[stage], m0 + 64 * c, k0, kPolicyEvictNormal);
          }
#pragma unroll
          for (int c = 0; c < BN / 64; ++c)
            tma_load_2d(st + kABytes + c * kColBytes, tb, &full[stage], n0 + 64 * c, k0, kPolicyEvictNormal);
          if (++stage == kStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16_f32_major(BM, BN, !A_KMAJOR, true);
      int stage = 0;
      uint32_t phase = 0;
      int t = 0;
      for (int u = blockIdx.x; u < n_units; u += gridDim.x, ++t) {
        const int acc = t & 1;
        mbar_wait(&tmem_empty[acc], ((t >> 1) & 1) ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
#pragma unroll 1
        for (int it = 0; it < k_iters; ++it) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint32_t st = smem_u32(smem + stage * kStageBytes);
          const uint64_t a_desc = A_KMAJOR ? umma_desc_kmajor_sw128(st) : umma_desc_mnmajor_sw128(st, kColBytes);
          const uint64_t b_desc = umma_desc_mnmajor_sw128(st + kABytes, kColBytes);
#pragma unroll
          for (int ks = 0; ks < BK / UMMA_K; ++ks) {
            // K-major: 16 elements = 32 B along the row; MN-major: 16 K rows = two 1024-byte atoms
            const uint64_t a_step = A_KMAJOR ? 2u * ks : static_cast<uint64_t>(ks) * (2048 >> 4);
            umma_f16_ss(d_tmem, a_desc + a_step, b_desc + static_cast<uint64_t>(ks) * (2048 >> 4), idesc,
                        (it | ks) != 0 ? 1u : 0u);
          }
          umma_commit(&empty[stage]);
          if (it == k_iters - 1) umma_commit(&tmem_full[acc]);
          if (++stage == kStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp >= 4) {
    const int quad = warp - 4;   // TMEM lanes 32 quad .. +31 (warp_id % 4)
    const uint32_t lane_taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    int t = 0;
    for (int u = blockIdx.x; u < n_units; u += gridDim.x, ++t) {
      int m0, n0;
      tile_of(u, &m0, &n0);
      const int acc = t & 1;
      mbar_wait(&tmem_full[acc], (t >> 1) & 1);
      tc_fence_after();
      const int row = m0 + quad * 32 + lane;
      float* dst = p.c + static_cast<size_t>(row) * p.N;
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 32) {
        if (n0 + c0 >= p.N) break;   // warp-uniform
        uint32_t r[32];
        tmem_ld_32x32b_x32(lane_taddr + acc * BN + c0, r);
        tmem_ld_wait();
        if (row < p.M) {
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            if (n0 + c0 + j < p.N)   // N % 8 == 0
              *reinterpret_cast<uint4*>(dst + n0 + c0 + j) = make_uint4(r[j], r[j + 1], r[j + 2], r[j + 3]);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 2) tmem_dealloc<kTmemCols>(tmem_base);
}

// ---- Co-activation counts of a dense activity mask: cooc[H, H] int32 += M^T M, M [K, H] bf16 0/1 (the analysis
// consumers' dense route, analysis.py). The producer and MMA warps are those of wgrad_kernel with A = B = M (both
// MN-major, one product); the schedule and the epilogue differ:
//   - only the 128 x 256 tiles that reach the upper triangle (some n >= m) are computed, column by column of tiles
//     (m fastest: the CTAs working at the same time share the 256-column slice of M in L2);
//   - the epilogue reads the exact integer counts (products of 0/1 summed in fp32: exact up to 2^24 rows) and, for
//     every element with n >= m, adds it to cooc[m, n] and, when n > m, to cooc[n, m] -- one writer per element and
//     launch, so no atomics, the result is bit-deterministic and complete after every launch. Lanes hold consecutive
//     rows m, so the mirrored read-modify-writes are coalesced 128-byte rows. The diagonal also goes to counts[m].
//   - eight epilogue warps (two per TMEM lane quarter, 128 columns each) keep enough loads in flight for the
//     read-modify-write to hide behind the MMAs of the next tile at K = 4096.
constexpr int kCoThreads = 384;             // warps: 0 TMA, 1 MMA, 2 TMEM alloc, 3 idle, 4-11 epilogue
constexpr int kCoEpiWarps = 8;

struct CoactParams {
  int H;
  int m_tiles;
  int k_chunks;
  int n_units;           // tiles that reach the upper triangle
  int32_t* c;            // [H, H]
  long long* counts;     // [H] or null
};

// unit u -> tile (m0, n0): columns of tiles in order, tile column nt holding row tiles 0 .. min(2 nt + 2, m_tiles) - 1
__device__ __forceinline__ void coact_tile_of(int u, int m_tiles, int* m0, int* n0) {
  int nt = 0;
  for (;;) {
    const int c = min(2 * nt + 2, m_tiles);
    if (u < c) break;
    u -= c;
    ++nt;
  }
  *m0 = u * BM;
  *n0 = nt * BN;
}

__global__ void __launch_bounds__(kCoThreads, 1)
coactivation_dense_kernel(const __grid_constant__ CUtensorMap tm, CoactParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kBarOff);
  uint64_t* full = bars;
  uint64_t* empty = bars + kStages;
  uint64_t* tmem_full = bars + 2 * kStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    if ((smem_u32(smem) & 1023u) != 0u) {
      printf("qsae: dynamic shared memory is not 1024-byte aligned\n");
      __trap();
    }
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], kCoEpiWarps);
    }
    fence_mbar_init();
    fence_proxy_async_smem();
  }
  if (warp == 2) tmem_alloc<kTmemCols>(tmem_ptr);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    if (lane == 0) {
      tma_prefetch_desc(&tm);
      int stage = 0;
      uint32_t phase = 0;
      for (int u = blockIdx.x; u < p.n_units; u += gridDim.x) {
        int m0, n0;
        coact_tile_of(u, p.m_tiles, &m0, &n0);
#pragma unroll 1
        for (int kc = 0; kc < p.k_chunks; ++kc) {
          mbar_wait(&empty[stage], phase ^ 1u);
          uint8_t* st = smem + stage * kStageBytes;
          mbar_arrive_expect_tx(&full[stage], kStageBytes);
          const int k0 = kc * BK;
#pragma unroll
          for (int c = 0; c < BM / 64; ++c) tma_load_2d(st + c * kColBytes, &tm, &full[stage], m0 + 64 * c, k0, kPolicyEvictNormal);
#pragma unroll
          for (int c = 0; c < BN / 64; ++c)
            tma_load_2d(st + kABytes + c * kColBytes, &tm, &full[stage], n0 + 64 * c, k0, kPolicyEvictNormal);
          if (++stage == kStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16_f32_major(BM, BN, true, true);
      int stage = 0;
      uint32_t phase = 0;
      int t = 0;
      for (int u = blockIdx.x; u < p.n_units; u += gridDim.x, ++t) {
        const int acc = t & 1;
        mbar_wait(&tmem_empty[acc], ((t >> 1) & 1) ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
#pragma unroll 1
        for (int kc = 0; kc < p.k_chunks; ++kc) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint32_t st = smem_u32(smem + stage * kStageBytes);
          const uint64_t a_desc = umma_desc_mnmajor_sw128(st, kColBytes);
          const uint64_t b_desc = umma_desc_mnmajor_sw128(st + kABytes, kColBytes);
#pragma unroll
          for (int ks = 0; ks < BK / UMMA_K; ++ks) {
            const uint64_t step = static_cast<uint64_t>(ks) * (2048 >> 4);   // 16 K rows = two 1024-byte atoms
            umma_f16_ss(d_tmem, a_desc + step, b_desc + step, idesc, (kc | ks) != 0 ? 1u : 0u);
          }
          umma_commit(&empty[stage]);
          if (kc == p.k_chunks - 1) umma_commit(&tmem_full[acc]);
          if (++stage == kStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp >= 4) {
    const int e = warp - 4;
    const int quad = e & 3;                    // TMEM lanes 32 quad .. +31 (warp_id % 4)
    const int cbase = (e >> 2) * (BN / 2);     // this warp's 128 columns of the tile
    const uint32_t lane_taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    const size_t H = static_cast<size_t>(p.H);
    int t = 0;
    for (int u = blockIdx.x; u < p.n_units; u += gridDim.x, ++t) {
      int m0, n0;
      coact_tile_of(u, p.m_tiles, &m0, &n0);
      const int acc = t & 1;
      mbar_wait(&tmem_full[acc], (t >> 1) & 1);
      tc_fence_after();
      const int wrow0 = m0 + quad * 32;
      const int m = wrow0 + lane;
      const bool row_ok = m < p.H;
#pragma unroll 1
      for (int c0 = cbase; c0 < cbase + BN / 2; c0 += 32) {
        const int nc = n0 + c0;
        if (nc >= p.H) break;                       // warp-uniform
        if (nc + 31 < wrow0 || wrow0 >= p.H) continue;   // wholly below the diagonal for every row of the warp
        uint32_t r[32];
        tmem_ld_32x32b_x32(lane_taddr + acc * BN + c0, r);
        tmem_ld_wait();
        int* v = reinterpret_cast<int*>(r);       // exact integer counts, in place
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __float2int_rn(__uint_as_float(r[j]));
        // cooc[m, n] for n >= m: the lane's own row, 16-byte groups (H % 8 == 0: a group is inside [0, H) or past it)
        int32_t* drow = p.c + static_cast<size_t>(m) * H + nc;
        int4 old[8];
#pragma unroll
        for (int q = 0; q < 8; ++q)
          old[q] = (row_ok && nc + 4 * q + 3 >= m && nc + 4 * q < p.H) ? *reinterpret_cast<const int4*>(drow + 4 * q)
                                                                        : make_int4(0, 0, 0, 0);
        // cooc[n, m] for n > m: column j of the tile is a row of cooc, the warp's 32 rows m are 32 consecutive ints;
        // 16 columns at a time, their loads issued together with the row's
        int mir[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          const int n = nc + j;
          mir[j] = (row_ok && n > m && n < p.H) ? p.c[static_cast<size_t>(n) * H + m] : 0;
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const int n = nc + 4 * q;
          if (!row_ok || n + 3 < m || n >= p.H) continue;
          if (n >= m) {
            *reinterpret_cast<int4*>(drow + 4 * q) =
                make_int4(old[q].x + v[4 * q], old[q].y + v[4 * q + 1], old[q].z + v[4 * q + 2], old[q].w + v[4 * q + 3]);
          } else {                                  // the group holding the diagonal: elements n + i >= m only
            if (n + 1 >= m) drow[4 * q + 1] = old[q].y + v[4 * q + 1];
            if (n + 2 >= m) drow[4 * q + 2] = old[q].z + v[4 * q + 2];
            drow[4 * q + 3] = old[q].w + v[4 * q + 3];
          }
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          if (h == 1) {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const int n = nc + 16 + j;
              mir[j] = (row_ok && n > m && n < p.H) ? p.c[static_cast<size_t>(n) * H + m] : 0;
            }
          }
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int n = nc + 16 * h + j;
            if (row_ok && n > m && n < p.H) p.c[static_cast<size_t>(n) * H + m] = mir[j] + v[16 * h + j];
          }
        }
        if (p.counts != nullptr && row_ok && m >= nc && m < nc + 32) {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (nc + j == m) p.counts[m] += v[j];
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 2) tmem_dealloc<kTmemCols>(tmem_base);
}

// ---- STE backward of the q_sae level decoder from a dense activity mask (training.py, dense route):
//   M[h, :] = sum_b a[b, h] g_level(h)[b, :]      (a: bf16 0/1 mask [B, H], g_l: d loss / d result[l] [B, D])
//   grad_w[h, d] += alpha[h] M[h, d] s(w[h, d]) (1 - s(w[h, d])), the same for the mirror
// (the STE term of matryoshka_grad_finish_kernel, train.cu, with M never written to memory). The producer and MMA
// warps are those of wgrad_kernel (A = the mask, MN-major; B = the gradient parts, MN-major); schedule and epilogue
// differ:
//   - B is one stacked bf16 tensor [n_levels B, D] per part: level l's K rows start at l B. The TMA zero-fills mask
//     rows past B, so whatever the B tile holds there (the next level's first rows) adds nothing;
//   - a work unit is (128-row tile, level, 256-column tile), one for each level the row tile intersects (level
//     boundaries may fall anywhere); a unit's epilogue writes only its level's rows, so each element has one writer:
//     no atomics, and the result is bit-deterministic. Segments (row tile, level) run in row order; the dimension
//     with fewer tiles runs fastest;
//   - products: mask x each bf16 part of g into one accumulator (1 or 3; the mask is exact in bf16);
//   - eight epilogue warps (two per TMEM lane quarter, 128 columns each) read w, w_mirror and both .grad rows
//     while the next unit's MMAs run.
struct SteDenseParams {
  int H, D, B;
  int m_tiles, n_tiles, n_segs, k_chunks;
  int n_prod;
  uint32_t prods;        // as WgradParams (A part always 0: the mask)
  int n_fast;            // unit u -> (segment u / n_tiles, n tile u % n_tiles), else (u % n_segs, u / n_segs)
  int n_levels;
  int start[9];          // level l owns rows [start[l], start[l + 1])
  const float* w;
  const float* wm;
  const float* alpha;
  float* gw;
  float* gwm;
};

// segments (row tile, non-empty level intersecting it) before row tile mt
__host__ __device__ inline int ste_seg_first(const int* start, int n_levels, int mt) {
  int s = 0;
  for (int l = 0; l < n_levels; ++l) {
    if (start[l] >= start[l + 1]) continue;
    const int lo = start[l] / BM, hi = (start[l + 1] - 1) / BM + 1;   // row tiles [lo, hi) of level l
    const int e = hi < mt ? hi : mt;
    if (e > lo) s += e - lo;
  }
  return s;
}

// segment index -> (row tile, level); a tile holds at most n_levels segments, so the search is short
__device__ __forceinline__ void ste_seg_of(const SteDenseParams& p, int s, int* mt, int* level) {
  int t = s < p.m_tiles - 1 ? s : p.m_tiles - 1;
  int f = ste_seg_first(p.start, p.n_levels, t);
  while (f > s) f = ste_seg_first(p.start, p.n_levels, --t);
  int j = s - f;
  const int r0 = t * BM, r1 = r0 + BM;
  int lv = 0;
  for (int l = 0; l < p.n_levels; ++l) {
    if (p.start[l] < p.start[l + 1] && p.start[l] < r1 && p.start[l + 1] > r0) {
      if (j == 0) { lv = l; break; }
      --j;
    }
  }
  *mt = t;
  *level = lv;
}

__device__ __forceinline__ void ste_unit(const SteDenseParams& p, int u, int* m0, int* n0, int* level) {
  const int s = p.n_fast ? u / p.n_tiles : u % p.n_segs;
  const int nt = p.n_fast ? u % p.n_tiles : u / p.n_segs;
  int mt;
  ste_seg_of(p, s, &mt, level);
  *m0 = mt * BM;
  *n0 = nt * BN;
}

// the literal fp32 logistic of train.cu (this file is compiled without fast-math as well)
__device__ __forceinline__ float ste_logistic(float w) { return 1.0f / (1.0f + expf(-w)); }

__global__ void __launch_bounds__(kCoThreads, 1)
matryoshka_ste_dense_kernel(const __grid_constant__ CUtensorMap tm, const __grid_constant__ CUtensorMap tg0,
                            const __grid_constant__ CUtensorMap tg1, const __grid_constant__ CUtensorMap tg2,
                            const __grid_constant__ SteDenseParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kBarOff);
  uint64_t* full = bars;
  uint64_t* empty = bars + kStages;
  uint64_t* tmem_full = bars + 2 * kStages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_units = p.n_segs * p.n_tiles;
  const int k_iters = p.n_prod * p.k_chunks;
  if (threadIdx.x == 0) {
    if ((smem_u32(smem) & 1023u) != 0u) {
      printf("qsae: dynamic shared memory is not 1024-byte aligned\n");
      __trap();
    }
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], kCoEpiWarps);
    }
    fence_mbar_init();
    fence_proxy_async_smem();
  }
  if (warp == 2) tmem_alloc<kTmemCols>(tmem_ptr);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    if (lane == 0) {
      tma_prefetch_desc(&tm);
      tma_prefetch_desc(&tg0);
      int stage = 0;
      uint32_t phase = 0;
      for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
        int m0, n0, level;
        ste_unit(p, u, &m0, &n0, &level);
        const int kbase = level * p.B;
#pragma unroll 1
        for (int it = 0; it < k_iters; ++it) {
          const int pi = it / p.k_chunks, kc = it - pi * p.k_chunks;
          const int bi = (p.prods >> (4 * pi)) & 3;
          const CUtensorMap* tg = bi == 0 ? &tg0 : (bi == 1 ? &tg1 : &tg2);
          mbar_wait(&empty[stage], phase ^ 1u);
          uint8_t* st = smem + stage * kStageBytes;
          mbar_arrive_expect_tx(&full[stage], kStageBytes);
          const int k0 = kc * BK;
#pragma unroll
          for (int c = 0; c < BM / 64; ++c) tma_load_2d(st + c * kColBytes, &tm, &full[stage], m0 + 64 * c, k0, kPolicyEvictNormal);
#pragma unroll
          for (int c = 0; c < BN / 64; ++c)
            tma_load_2d(st + kABytes + c * kColBytes, tg, &full[stage], n0 + 64 * c, kbase + k0, kPolicyEvictNormal);
          if (++stage == kStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16_f32_major(BM, BN, true, true);
      int stage = 0;
      uint32_t phase = 0;
      int t = 0;
      for (int u = blockIdx.x; u < n_units; u += gridDim.x, ++t) {
        const int acc = t & 1;
        mbar_wait(&tmem_empty[acc], ((t >> 1) & 1) ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
#pragma unroll 1
        for (int it = 0; it < k_iters; ++it) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint32_t st = smem_u32(smem + stage * kStageBytes);
          const uint64_t a_desc = umma_desc_mnmajor_sw128(st, kColBytes);
          const uint64_t b_desc = umma_desc_mnmajor_sw128(st + kABytes, kColBytes);
#pragma unroll
          for (int ks = 0; ks < BK / UMMA_K; ++ks) {
            const uint64_t step = static_cast<uint64_t>(ks) * (2048 >> 4);   // 16 K rows = two 1024-byte atoms
            umma_f16_ss(d_tmem, a_desc + step, b_desc + step, idesc, (it | ks) != 0 ? 1u : 0u);
          }
          umma_commit(&empty[stage]);
          if (it == k_iters - 1) umma_commit(&tmem_full[acc]);
          if (++stage == kStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp >= 4) {
    const int e = warp - 4;
    const int quad = e & 3;                    // TMEM lanes 32 quad .. +31 (warp_id % 4)
    const int cbase = (e >> 2) * (BN / 2);     // this warp's 128 columns of the tile
    const uint32_t lane_taddr = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    int t = 0;
    for (int u = blockIdx.x; u < n_units; u += gridDim.x, ++t) {
      int m0, n0, level;
      ste_unit(p, u, &m0, &n0, &level);
      const int acc = t & 1;
      mbar_wait(&tmem_full[acc], (t >> 1) & 1);
      tc_fence_after();
      const int row = m0 + quad * 32 + lane;
      const bool row_ok = row >= p.start[level] && row < p.start[level + 1];
      if (__ballot_sync(0xffffffffu, row_ok) != 0u) {
        const float a = row_ok ? p.alpha[row] : 0.f;
        const size_t roff = static_cast<size_t>(row) * p.D;
#pragma unroll 1
        for (int c0 = cbase; c0 < cbase + BN / 2; c0 += 32) {
          const int nc = n0 + c0;
          if (nc >= p.D) break;                 // warp-uniform; D % 16 == 0
          uint32_t r[32];
          tmem_ld_32x32b_x32(lane_taddr + acc * BN + c0, r);
          tmem_ld_wait();
          if (!row_ok) continue;
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int cc = nc + 16 * h;
            if (cc >= p.D) break;
            float4 w4[4], wm4[4], g4[4], gm4[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              w4[q] = *reinterpret_cast<const float4*>(p.w + roff + cc + 4 * q);
              wm4[q] = *reinterpret_cast<const float4*>(p.wm + roff + cc + 4 * q);
              g4[q] = *reinterpret_cast<const float4*>(p.gw + roff + cc + 4 * q);
              gm4[q] = *reinterpret_cast<const float4*>(p.gwm + roff + cc + 4 * q);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float* wv = reinterpret_cast<const float*>(&w4[q]);
              const float* wmv = reinterpret_cast<const float*>(&wm4[q]);
              float* gv = reinterpret_cast<float*>(&g4[q]);
              float* gmv = reinterpret_cast<float*>(&gm4[q]);
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const float up = a * __uint_as_float(r[16 * h + 4 * q + i]);
                const float s = ste_logistic(wv[i]), sm = ste_logistic(wmv[i]);
                gv[i] += up * (s * (1.f - s));
                gmv[i] += up * (sm * (1.f - sm));
              }
              *reinterpret_cast<float4*>(p.gw + roff + cc + 4 * q) = g4[q];
              *reinterpret_cast<float4*>(p.gwm + roff + cc + 4 * q) = gm4[q];
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 2) tmem_dealloc<kTmemCols>(tmem_base);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// row-major bf16 [rows, cols] with a {64 x box_rows} box, 128-byte swizzle
bool make_tmap(CUtensorMap* map, const void* base, int rows, int cols, int box_rows) {
  static EncodeTiledFn enc = nullptr;
  if (!enc) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      return false;
    enc = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  const TmapKey key{base, static_cast<unsigned long long>(rows), static_cast<unsigned long long>(cols),
                    static_cast<unsigned long long>(cols) * 2, static_cast<unsigned int>(BK), static_cast<unsigned int>(box_rows),
                    static_cast<int>(CU_TENSOR_MAP_DATA_TYPE_BFLOAT16), static_cast<int>(CU_TENSOR_MAP_SWIZZLE_128B),
                    tmap_current_device()};
  EncodeTiledFn fn = enc;
  return tmap_cache().get(key, map, [&](CUtensorMap* m) {
    cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
    cuuint64_t strides[1] = {static_cast<cuuint64_t>(cols) * 2};
    cuuint32_t box[2] = {BK, static_cast<cuuint32_t>(box_rows)};
    cuuint32_t estr[2] = {1, 1};
    return fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
  });
}

template <bool A_KMAJOR>
cudaError_t launch(const CUtensorMap* ta, const CUtensorMap* tb, const WgradParams& p, int grid, cudaStream_t stream) {
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(wgrad_kernel<A_KMAJOR>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
    if (e != cudaSuccess) return e;
    attr = true;
  }
  wgrad_kernel<A_KMAJOR><<<grid, kThreads, kSmem, stream>>>(ta[0], ta[1], ta[2], tb[0], tb[1], tb[2], p);
  return cudaGetLastError();
}

}  // namespace

const char* wgrad_launch(const uint16_t* const* a_parts, const uint16_t* const* b_parts, int n_parts, int M, int N, int K,
                         bool a_kmajor, float* c, int num_sms, cudaStream_t stream) {
  if (n_parts != 1 && n_parts != 3) return "wgrad: 1 or 3 parts per operand";
  if (M <= 0 || N <= 0 || K <= 0 || (N % 8) != 0) return "wgrad: M, N, K must be positive and N a multiple of 8";
  if (a_kmajor ? (K % 8) != 0 : (M % 8) != 0) return "wgrad: the row pitch of A (M, or K when A is K-major) must be a multiple of 8";
  CUtensorMap ta[3], tb[3];
  for (int i = 0; i < 3; ++i) {
    const int j = i < n_parts ? i : 0;
    const bool ok_a = a_kmajor ? make_tmap(&ta[i], a_parts[j], M, K, BM) : make_tmap(&ta[i], a_parts[j], K, M, BK);
    if (!ok_a) return "cuTensorMapEncodeTiled(wgrad A) failed";
    if (!make_tmap(&tb[i], b_parts[j], K, N, BK)) return "cuTensorMapEncodeTiled(wgrad B) failed";
  }
  WgradParams p;
  p.M = M; p.N = N;
  p.m_tiles = (M + BM - 1) / BM;
  p.n_tiles = (N + BN - 1) / BN;
  p.k_chunks = (K + BK - 1) / BK;
  if (n_parts == 1) {
    p.n_prod = 1;
    p.prods = 0u;
  } else {
    // (A part, B part), smallest first: lo hi, mid mid, hi lo, mid hi, hi mid, hi hi
    const uint32_t pairs[6][2] = {{2, 0}, {1, 1}, {0, 2}, {1, 0}, {0, 1}, {0, 0}};
    p.n_prod = 6;
    p.prods = 0u;
    for (int i = 0; i < 6; ++i) p.prods |= ((pairs[i][0] << 2) | pairs[i][1]) << (4 * i);
  }
  p.a_kmajor = a_kmajor ? 1 : 0;
  p.m_fast = p.m_tiles <= p.n_tiles ? 1 : 0;
  p.c = c;
  const int units = p.m_tiles * p.n_tiles;
  const int grid = units < num_sms ? units : num_sms;
  const cudaError_t e = a_kmajor ? launch<true>(ta, tb, p, grid, stream) : launch<false>(ta, tb, p, grid, stream);
  return cuda_err(e);
}

const char* coactivation_dense_launch(const uint16_t* mask, int K, int H, int32_t* cooc, long long* counts, int num_sms,
                                      cudaStream_t stream) {
  if (K <= 0 || H <= 0 || (H % 8) != 0) return "coactivation_dense: K and H must be positive and H a multiple of 8";
  if (K > (1 << 24)) return "coactivation_dense: at most 2^24 rows per launch (fp32 counts are exact up to 2^24)";
  CUtensorMap tm;
  if (!make_tmap(&tm, mask, K, H, BK)) return "cuTensorMapEncodeTiled(coactivation mask) failed";
  CoactParams p;
  p.H = H;
  p.m_tiles = (H + BM - 1) / BM;
  p.k_chunks = (K + BK - 1) / BK;
  p.n_units = 0;
  for (int nt = 0; nt < (H + BN - 1) / BN; ++nt) p.n_units += 2 * nt + 2 < p.m_tiles ? 2 * nt + 2 : p.m_tiles;
  p.c = cooc;
  p.counts = counts;
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(coactivation_dense_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
    if (e != cudaSuccess) return cuda_err(e);
    attr = true;
  }
  const int grid = p.n_units < num_sms ? p.n_units : num_sms;
  coactivation_dense_kernel<<<grid, kCoThreads, kSmem, stream>>>(tm, p);
  return cuda_err(cudaGetLastError());
}

const char* matryoshka_ste_dense_launch(const uint16_t* mask, int B, int H, int D, const uint16_t* const* g_parts, int n_parts,
                                        const int* level_start, int n_levels, const float* w, const float* w_mirror,
                                        const float* alpha, float* grad_w, float* grad_w_mirror, int num_sms,
                                        cudaStream_t stream) {
  if (n_parts != 1 && n_parts != 3) return "matryoshka_ste_dense: 1 or 3 parts of the gradients";
  if (n_levels < 1 || n_levels > 8) return "matryoshka_ste_dense: 1..8 levels";
  if (B <= 0 || H <= 0 || (H % 8) != 0 || D <= 0 || (D % 16) != 0)
    return "matryoshka_ste_dense: B, H, D must be positive, H a multiple of 8 and D of 16";
  CUtensorMap tm, tg[3];
  if (!make_tmap(&tm, mask, B, H, BK)) return "cuTensorMapEncodeTiled(ste mask) failed";
  for (int i = 0; i < 3; ++i)
    if (!make_tmap(&tg[i], g_parts[i < n_parts ? i : 0], n_levels * B, D, BK)) return "cuTensorMapEncodeTiled(ste gradients) failed";
  SteDenseParams p;
  p.H = H; p.D = D; p.B = B;
  p.m_tiles = (H + BM - 1) / BM;
  p.n_tiles = (D + BN - 1) / BN;
  p.k_chunks = (B + BK - 1) / BK;
  p.n_levels = n_levels;
  for (int i = 0; i < 9; ++i) p.start[i] = level_start[i <= n_levels ? i : n_levels];
  p.n_segs = ste_seg_first(p.start, n_levels, p.m_tiles);
  if (n_parts == 1) {
    p.n_prod = 1;
    p.prods = 0u;
  } else {
    // mask x (lo, mid, hi): smallest first
    p.n_prod = 3;
    p.prods = 2u | (1u << 4) | (0u << 8);
  }
  p.n_fast = p.n_tiles <= p.n_segs ? 1 : 0;
  p.w = w; p.wm = w_mirror; p.alpha = alpha; p.gw = grad_w; p.gwm = grad_w_mirror;
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(matryoshka_ste_dense_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
    if (e != cudaSuccess) return cuda_err(e);
    attr = true;
  }
  const int units = p.n_segs * p.n_tiles;
  const int grid = units < num_sms ? units : num_sms;
  matryoshka_ste_dense_kernel<<<grid, kCoThreads, kSmem, stream>>>(tm, tg[0], tg[1], tg[2], p);
  return cuda_err(cudaGetLastError());
}

}  // namespace qsae
