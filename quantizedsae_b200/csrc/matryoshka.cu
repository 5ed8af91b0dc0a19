// q_sae (QuantizedMatryoshkaDecoder, sae/quantized_matryoshka.py:47-143) on a packed dictionary.
//
// Reference per level i (latent rows [start_i, start_i + size_i)):
//   S = +1 where sigmoid(w) >= 0.5 else -1, for weight and weight_mirror          (:67-80)
//   T = S + S_mirror in {-2, 0, +2}
//   scale[h] = 2^(n_bits - i - 2) * quant_step / (||T[h,:]||_2 + 1e-8)            (:82-91)
//   a[b,h]  = latent[b,h] > 0.5 (latent = sigmoid(z), i.e. z > 0)                 (:99)
//   recon  += (scale * a) @ T ; + bias once at level 0 ; result[i] = recon         (:121-129)
//   latent_group[i] = mean_b sum_{h in level i} a[b,h]                             (:127)
//
// Packed form: 2 bits per entry (bit0 = non-zero, bit1 = negative; value = +-2), 16 entries per
// 32-bit word, [H, D/16] words (128 B per row at D = 512) + one fp32 scale per row.
// The decoder consumes the encoder's survivor lists directly (the active latents of a row, any
// order): warp per token, level accumulators in shared memory, cumulative outputs.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "kernels.h"

namespace qsae {

namespace {

__device__ __forceinline__ float logistic(float w) { return 1.0f / (1.0f + expf(-w)); }

// one warp per dictionary row; lane handles 16 consecutive features per trip
__global__ void __launch_bounds__(256)
pack_matryoshka_kernel(const float* __restrict__ w, const float* __restrict__ wm, int H, int D,
                       const int* __restrict__ level_start, const float* __restrict__ level_factor,
                       int n_levels, uint32_t* __restrict__ packed, float* __restrict__ scale) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = blockIdx.x * 8 + warp;
  if (h >= H) return;
  const int words = D >> 4;
  int nnz = 0;
  for (int wd = lane; wd < words; wd += 32) {
    uint32_t bits = 0u;
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      const size_t o = static_cast<size_t>(h) * D + wd * 16 + q;
      const int s = (logistic(w[o]) >= 0.5f) ? 1 : -1;
      const int sm = (logistic(wm[o]) >= 0.5f) ? 1 : -1;
      const int t = s + sm;                     // -2, 0, +2
      const uint32_t code = (t != 0 ? 1u : 0u) | (t < 0 ? 2u : 0u);
      bits |= code << (2 * q);
      nnz += (t != 0);
    }
    packed[static_cast<size_t>(h) * words + wd] = bits;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) nnz += __shfl_xor_sync(0xffffffffu, nnz, o);
  if (lane == 0) {
    int lvl = 0;
    while (lvl + 1 < n_levels && h >= level_start[lvl + 1]) ++lvl;
    const float norm = sqrtf(static_cast<float>(4 * nnz));  // ||T||_2, T entries are +-2
    scale[h] = level_factor[lvl] / (norm + 1e-8f);
  }
}

// max_h ||w[h,:]||_2 (for the rounding-error band of the bf16 activity test), non-negative float max
__global__ void __launch_bounds__(256)
max_row_norm_kernel(const float* __restrict__ w, int H, int D, float* __restrict__ out) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = blockIdx.x * 8 + warp;
  if (h >= H) return;
  float s = 0.f;
  for (int d = lane; d < D; d += 32) { const float v = w[static_cast<size_t>(h) * D + d]; s = fmaf(v, v, s); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) atomicMax(reinterpret_cast<unsigned*>(out), __float_as_uint(sqrtf(s)));
}

// thr[b] = thr_value - band_b, band_b = 2^-8 ||x_b||_2 max_h||w_h||_2 (+1 %): an upper bound of
// |z_bf16 - z_fp32| (each operand carries <= 2^-9 relative rounding error), so every latent that
// is active in fp32 survives the tensor-core sweep and is then decided exactly by re-scoring
__global__ void __launch_bounds__(256)
row_threshold_kernel(const float* __restrict__ x, int B, int D, const float* __restrict__ wmax, float thr_value,
                     float* __restrict__ thr) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * 8 + warp;
  if (b >= B) return;
  float s = 0.f;
  for (int d = lane; d < D; d += 32) { const float v = x[static_cast<size_t>(b) * D + d]; s = fmaf(v, v, s); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) thr[b] = thr_value - (1.01f * 0.00390625f * sqrtf(s) * (*wmax) + 1e-6f);
}

// ---- dense fallback (rows with more active latents than the survivor lists hold, e.g. an untrained
// model with ~50 % activity): the level sums become tensor-core GEMMs over K ranges of H.

// packed codes [H, D/16] -> T^T bf16 [D, H]; 32 x 32 tiles through shared memory, coalesced both ways
__global__ void unpack_matryoshka_t_kernel(const uint32_t* __restrict__ packed, int H, int D,
                                           uint16_t* __restrict__ t_bf16) {
  __shared__ uint16_t tile[32][33];
  const int h0 = blockIdx.x * 32, d0 = blockIdx.y * 32;   // D % 16 == 0: a tile covers two code words per row
  const int words = D >> 4;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int h = h0 + i, d = d0 + threadIdx.x;
    uint16_t v = 0;
    if (h < H && d < D) {
      const uint32_t code = (packed[static_cast<size_t>(h) * words + (d >> 4)] >> (2 * (d & 15))) & 3u;
      v = (code & 1u) ? ((code & 2u) ? 0xC000u : 0x4000u) : 0u;   // -2.0 / +2.0 / 0 in bf16
    }
    tile[i][threadIdx.x] = v;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int d = d0 + i, h = h0 + threadIdx.x;
    if (d < D && h < H) t_bf16[static_cast<size_t>(d) * H + h] = tile[threadIdx.x][i];
  }
}

// a[b, h] = (z[b, h] >= thr) ? scale[h] : 0, as bf16 hi + lo (hi + lo = scale to 2^-17); per-level activity counts;
// with a mask, also mask[b * mask_pitch + h] = bf16 (z[b, h] >= thr) (the activity itself: a zero scale is still active).
// HBM-streaming (4 B read, 4 B written per element): 8 consecutive latents per thread through 16-byte accesses. A
// group's count is added once per warp when the warp's groups lie inside one level (the usual case), else per lane;
// a group that straddles a level boundary (boundaries need not be multiples of 8) is counted element by element.
__global__ void __launch_bounds__(256)
matryoshka_dense_operand_kernel(const float* __restrict__ z, int B, int H, const float* __restrict__ scale, float thr,
                                const int* __restrict__ level_start, int n_levels, uint16_t* __restrict__ a_hi,
                                uint16_t* __restrict__ a_lo, unsigned* __restrict__ count_partial /* [gridDim.x, 32] */,
                                uint16_t* __restrict__ mask, int mask_pitch) {
  __shared__ unsigned s_cnt[32];
  __shared__ int s_start[33];
  if (threadIdx.x < 32) s_cnt[threadIdx.x] = 0u;
  if (threadIdx.x <= n_levels) s_start[threadIdx.x] = level_start[threadIdx.x];
  __syncthreads();
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const unsigned h8 = static_cast<unsigned>(H >> 3);
  const size_t groups = static_cast<size_t>(B) * h8;
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  const size_t first = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  // whole warps iterate together (the tail lanes of the last iteration carry an empty group)
  for (size_t g0 = first - lane; g0 < groups; g0 += stride) {
    const size_t g = g0 + lane;
    const bool live = g < groups;
    int lvl = -1;
    int h = 0;
    unsigned n_act = 0u, act_bits = 0u;
    bool straddle = false;
    if (live) {
      h = static_cast<int>(g % h8) << 3;
      const float4 z0 = __ldcs(reinterpret_cast<const float4*>(z + g * 8));
      const float4 z1 = __ldcs(reinterpret_cast<const float4*>(z + g * 8) + 1);
      const float4 s0 = __ldg(reinterpret_cast<const float4*>(scale + h));
      const float4 s1 = __ldg(reinterpret_cast<const float4*>(scale + h) + 1);
      const float zv[8] = {z0.x, z0.y, z0.z, z0.w, z1.x, z1.y, z1.z, z1.w};
      const float sv[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
      uint32_t hi[4], lo[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const bool a0 = zv[2 * i] >= thr, a1 = zv[2 * i + 1] >= thr;
        n_act += (a0 ? 1u : 0u) + (a1 ? 1u : 0u);
        act_bits |= (a0 ? 1u : 0u) << (2 * i) | (a1 ? 1u : 0u) << (2 * i + 1);
        const float v0 = a0 ? sv[2 * i] : 0.f, v1 = a1 ? sv[2 * i + 1] : 0.f;
        const __nv_bfloat162 hh = __floats2bfloat162_rn(v0, v1);
        const __nv_bfloat162 ll = __floats2bfloat162_rn(v0 - __bfloat162float(hh.x), v1 - __bfloat162float(hh.y));
        hi[i] = *reinterpret_cast<const uint32_t*>(&hh);
        lo[i] = *reinterpret_cast<const uint32_t*>(&ll);
      }
      *reinterpret_cast<uint4*>(a_hi + g * 8) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
      *reinterpret_cast<uint4*>(a_lo + g * 8) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
      if (mask != nullptr) {
        uint32_t mk[4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
          mk[i] = (((act_bits >> (2 * i)) & 1u) ? 0x3F80u : 0u) | (((act_bits >> (2 * i + 1)) & 1u) ? 0x3F800000u : 0u);
        *reinterpret_cast<uint4*>(mask + (g / h8) * static_cast<size_t>(mask_pitch) + h) = make_uint4(mk[0], mk[1], mk[2], mk[3]);
      }
      lvl = 0;
      while (lvl + 1 < n_levels && h >= s_start[lvl + 1]) ++lvl;
      straddle = lvl + 1 < n_levels && h + 8 > s_start[lvl + 1];
    }
    const int lvl0 = __shfl_sync(full, lvl, 0);
    if (__all_sync(full, lvl == lvl0 && !straddle)) {
      const unsigned tot = __reduce_add_sync(full, n_act);
      if (lane == 0 && tot != 0u) atomicAdd(&s_cnt[lvl0], tot);
    } else if (!straddle) {
      if (n_act != 0u) atomicAdd(&s_cnt[lvl], n_act);
    } else {
      for (int i = 0; i < 8; ++i) {
        while (lvl + 1 < n_levels && h + i >= s_start[lvl + 1]) ++lvl;
        if ((act_bits >> i) & 1u) atomicAdd(&s_cnt[lvl], 1u);
      }
    }
  }
  __syncthreads();
  if (threadIdx.x < 32) count_partial[static_cast<size_t>(blockIdx.x) * 32 + threadIdx.x] = s_cnt[threadIdx.x];
}

// The dense level GEMMs run over the cuts c_l = floor8(level_start[l + 1]), because a TMA base address must be 16-byte
// aligned: their chain leaves R[l] = bias + sum over h < c_l in result[l] for every level whose range [c_{l-1}, c_l)
// is not empty. This kernel completes every level:
//   result[l] = R[m] + sum over h in [c_l, level_start[l + 1]) of (a_hi + a_lo)[b, h] T[h, :],
// m = the last level <= l that had a GEMM (none: R = bias). The at most 7 leftover columns of level l lie in level
// l + 1's GEMM range, so they go to result[l] only. Block per row, thread per output feature, levels in order.
__global__ void __launch_bounds__(128)
matryoshka_dense_tail_kernel(const uint16_t* __restrict__ a_hi, const uint16_t* __restrict__ a_lo,
                             const uint16_t* __restrict__ t_bf16 /* [D, H] */, const int* __restrict__ level_start,
                             int n_levels, int B, int H, int D, const float* __restrict__ bias,
                             float* __restrict__ result /* [n_levels, B, D] */) {
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
      float chain = bias != nullptr ? __ldg(bias + d) : 0.f;
      int c_prev = 0;
      for (int l = 0; l < n_levels; ++l) {
        const int end = __ldg(level_start + l + 1), c = end & ~7;
        float* out = result + (static_cast<size_t>(l) * B + b) * D + d;
        if (c > c_prev) chain = *out;
        float tail = 0.f;
        if (end > c) {
          const uint4 hv = __ldg(reinterpret_cast<const uint4*>(a_hi + static_cast<size_t>(b) * H + c));
          const uint4 lv = __ldg(reinterpret_cast<const uint4*>(a_lo + static_cast<size_t>(b) * H + c));
          const uint4 tv = __ldg(reinterpret_cast<const uint4*>(t_bf16 + static_cast<size_t>(d) * H + c));
          const uint32_t hw[4] = {hv.x, hv.y, hv.z, hv.w}, lw[4] = {lv.x, lv.y, lv.z, lv.w}, tw[4] = {tv.x, tv.y, tv.z, tv.w};
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int sh = (j & 1) ? 0 : 16;   // bf16 j of a word: low half for even j
            const float a = __uint_as_float((hw[j >> 1] << sh) & 0xFFFF0000u) + __uint_as_float((lw[j >> 1] << sh) & 0xFFFF0000u);
            const float t = __uint_as_float((tw[j >> 1] << sh) & 0xFFFF0000u);
            if (c + j < end) tail = fmaf(a, t, tail);
          }
        }
        *out = chain + tail;
        c_prev = c;
      }
    }
  }
}

constexpr int kMatWarps = 4;

// Sparse level decoder: warp per token row (persistent grid), one 32-bit code word = 16 features per
// lane (D <= 512). The outputs are CUMULATIVE over the levels and every survivor list is sorted by column
// (a sub-stream sweeps its tiles in ascending order), so the row is processed level by level with ONE
// running accumulator: for level l every list is scanned from its cursor up to the level's last column,
// then result[l] = bias + running sum is written. (The first version kept one accumulator set per level,
// 64 + registers per thread: 143 registers, 12 warps per SM, issue slots 31 % busy.) The level test is
// warp-uniform. Activity counts are kept in registers over all rows of a warp and leave through a
// [warps, n_levels] partial array that a second kernel sums: tens of thousands of atomics on n_levels
// addresses serialise in L2 (measured: 3.9 ms of a 5.7 ms forward at B = 65536 before this change).
template <int NL, int BPS = 6>
__global__ void __launch_bounds__(kMatWarps * 32, BPS)
decode_matryoshka_kernel(const uint2* __restrict__ cand, const int* __restrict__ cand_cnt, int nsub,
                         int cap, int B, const uint32_t* __restrict__ packed,
                         const float* __restrict__ scale, const int* __restrict__ level_start,
                         int n_levels, int H, int D, const float* __restrict__ bias,
                         float* __restrict__ result /* [n_levels, B, D] */,
                         unsigned long long* __restrict__ level_count /* [n_levels], += */,
                         const float* __restrict__ x_f32, const float* __restrict__ w_f32,
                         const float* __restrict__ b_enc, float thr_value, int exact,
                         int32_t* __restrict__ active_idx /* [B, active_cap] or null */, int active_cap,
                         int* __restrict__ active_cnt /* [B] */,
                         const float* __restrict__ resid_in /* [B, D] or null */, float* __restrict__ resid_out /* [B, D] */,
                         const int* __restrict__ poison_flag /* != 0: the sweep overflowed a survivor list */) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const unsigned full = 0xffffffffu;
  // A sweep whose survivor lists overflowed has dropped active latents: every output of this call becomes NaN, so a
  // caller that reads the overflow flag lazily (no host synchronisation per forward) can never use a wrong result
  const float poison = (poison_flag != nullptr && *poison_flag != 0) ? __uint_as_float(0x7FC00000u) : 0.f;
  const int words = D >> 4;                 // <= 32: lane `l` owns word l (features 16 l .. 16 l + 15)
  const bool has_word = lane < words;
  unsigned cnt[NL];
#pragma unroll
  for (int l = 0; l < NL; ++l) cnt[l] = 0u;

  for (int row = blockIdx.x * kMatWarps + warp; row < B; row += gridDim.x * kMatWarps) {
    float run[16];   // bias + sum over the active latents of the levels processed so far
#pragma unroll
    for (int q = 0; q < 16; ++q) run[q] = (bias && has_word) ? __ldg(bias + lane * 16 + q) : 0.f;
    float4 xr[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int d = c * 128 + lane * 4;
      xr[c] = (exact && d < D) ? *reinterpret_cast<const float4*>(x_f32 + static_cast<size_t>(row) * D + d)
                               : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    // lane s keeps the length and the cursor of list s (nsub <= 32)
    const int my_c = (lane < nsub) ? min(cand_cnt[static_cast<size_t>(row) * nsub + lane], cap) : 0;
    int my_cur = 0;
    int n_act = 0;   // warp-uniform: active latents of this row (exported for the analysis consumers)
#pragma unroll
    for (int l = 0; l < NL; ++l) {
      if (l < n_levels) {
        const int col_end = (l + 1 < n_levels) ? __ldg(level_start + l + 1) : 0x7fffffff;   // first column of the next level
        for (int s = 0; s < nsub; ++s) {
          const int c = __shfl_sync(full, my_c, s);
          int cur = __shfl_sync(full, my_cur, s);
          const uint2* src = cand + (static_cast<size_t>(row) * nsub + s) * cap;
          bool level_done = false;
          while (cur < c && !level_done) {
            const int e = cur + lane;
            const int my_col = (e < c) ? static_cast<int>(src[e].y) : 0x7fffffff;
            // entries of this chunk that belong to the level: a prefix (the list is sorted by column)
            const unsigned in_level = __ballot_sync(full, my_col < col_end);
            const int m = __popc(in_level);             // in_level is a low-bit prefix mask
            level_done = m < 32;
            // two candidates per trip: their dictionary rows and scales are fetched together
            for (int j = 0; j < m; j += 2) {
              int col[2];
              bool ok[2];
              col[0] = __shfl_sync(full, my_col, j);
              col[1] = __shfl_sync(full, my_col, min(j + 1, 31));
              ok[0] = col[0] >= 0 && col[0] < H;
              ok[1] = (j + 1 < m) && col[1] >= 0 && col[1] < H;
              if (exact) {  // the sweep kept a rounding-error band below the threshold: decide in fp32
                float a[2] = {0.f, 0.f};
#pragma unroll
                for (int t = 0; t < 2; ++t) {
                  if (ok[t]) {   // warp-uniform
                    const float* wrow = w_f32 + static_cast<size_t>(col[t]) * D;
#pragma unroll
                    for (int cc = 0; cc < 4; ++cc) {
                      const int d = cc * 128 + lane * 4;
                      if (d < D) {
                        const float4 u = __ldg(reinterpret_cast<const float4*>(wrow + d));
                        a[t] = fmaf(xr[cc].x, u.x, a[t]); a[t] = fmaf(xr[cc].y, u.y, a[t]);
                        a[t] = fmaf(xr[cc].z, u.z, a[t]); a[t] = fmaf(xr[cc].w, u.w, a[t]);
                      }
                    }
                  }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                  a[0] += __shfl_xor_sync(full, a[0], o);
                  a[1] += __shfl_xor_sync(full, a[1], o);
                }
#pragma unroll
                for (int t = 0; t < 2; ++t)
                  if (ok[t]) ok[t] = (a[t] + __ldg(b_enc + col[t]) >= thr_value);
              }
              float s2[2];
              uint32_t bits[2];
#pragma unroll
              for (int t = 0; t < 2; ++t) {
                s2[t] = ok[t] ? 2.f * __ldg(scale + col[t]) : 0.f;
                bits[t] = (ok[t] && has_word) ? __ldg(packed + static_cast<size_t>(col[t]) * words + lane) : 0u;
              }
#pragma unroll
              for (int t = 0; t < 2; ++t) {
                if (ok[t]) {   // warp-uniform
                  if (active_idx != nullptr) {
                    if (lane == 0 && n_act < active_cap) active_idx[static_cast<size_t>(row) * active_cap + n_act] = col[t];
                    ++n_act;
                  }
                  ++cnt[l];
                }
#pragma unroll
                for (int q = 0; q < 16; ++q) {
                  const float mag = ((bits[t] >> (2 * q)) & 1u) ? s2[t] : 0.f;
                  run[q] += ((bits[t] >> (2 * q + 1)) & 1u) ? -mag : mag;
                }
              }
            }
            cur += m;
          }
          if (lane == s) my_cur = cur;
        }
        if (has_word) {   // cumulative output of this level
          float4* dst = reinterpret_cast<float4*>(result + (static_cast<size_t>(l) * B + row) * D + lane * 16);
#pragma unroll
          for (int q = 0; q < 4; ++q)
            dst[q] = make_float4(run[4 * q] + poison, run[4 * q + 1] + poison, run[4 * q + 2] + poison, run[4 * q + 3] + poison);
        }
      }
    }
    if (active_idx != nullptr && lane == 0) active_cnt[row] = n_act;
    // rq_sae: the next stage's input, (residual - reconstruction) * 2 (sae/residual_quantized.py:67), from the
    // final reconstruction still in registers
    if (resid_out != nullptr && has_word) {
      const float4* rin = reinterpret_cast<const float4*>(resid_in + static_cast<size_t>(row) * D + lane * 16);
      float4* rout = reinterpret_cast<float4*>(resid_out + static_cast<size_t>(row) * D + lane * 16);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 r = rin[q];
        rout[q] = make_float4((r.x - run[4 * q]) * 2.f + poison, (r.y - run[4 * q + 1]) * 2.f + poison,
                              (r.z - run[4 * q + 2]) * 2.f + poison, (r.w - run[4 * q + 3]) * 2.f + poison);
      }
    }
  }
  // activity counts: the block's warps add up in shared memory, then one 64-bit atomic per level and block (a few
  // thousand integer atomics on n_levels addresses per launch; the sum is exact, so the order does not matter).
  // Round 1 summed a [warps, n_levels] partial array in a second, single-block kernel: 12.7 us at any batch size.
  __shared__ unsigned s_cnt[kMatWarps][NL];
  if (lane == 0) {
#pragma unroll
    for (int l = 0; l < NL; ++l) s_cnt[warp][l] = cnt[l];
  }
  __syncthreads();
  if (threadIdx.x < NL && threadIdx.x < n_levels) {
    unsigned long long t = 0ull;
#pragma unroll
    for (int w = 0; w < kMatWarps; ++w) t += s_cnt[w][threadIdx.x];
    if (t != 0ull) atomicAdd(level_count + threadIdx.x, t);
  }
}

// level_count[l] += sum over the partial rows (one block per level; fixed order)
__global__ void __launch_bounds__(256)
sum_level_counts_kernel(const unsigned* __restrict__ partial, int n_rows, int stride, int n_levels,
                        unsigned long long* __restrict__ level_count) {
  __shared__ unsigned long long s[256];
  const int l = blockIdx.x;
  unsigned long long a = 0ull;
  for (int r = threadIdx.x; r < n_rows; r += blockDim.x) a += partial[static_cast<size_t>(r) * stride + l];
  s[threadIdx.x] = a;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) level_count[l] += s[0];
}

}  // namespace

const char* pack_matryoshka_launch(const float* w, const float* wm, int H, int D, const int* level_start,
                                   const float* level_factor, int n_levels, uint32_t* packed, float* scale,
                                   cudaStream_t stream) {
  pack_matryoshka_kernel<<<(H + 7) / 8, 256, 0, stream>>>(w, wm, H, D, level_start, level_factor, n_levels,
                                                          packed, scale);
  return cuda_err(cudaGetLastError());
}

const char* unpack_matryoshka_t_launch(const uint32_t* packed, int H, int D, uint16_t* t_bf16, cudaStream_t stream) {
  dim3 grid((H + 31) / 32, (D + 31) / 32), block(32, 8);
  unpack_matryoshka_t_kernel<<<grid, block, 0, stream>>>(packed, H, D, t_bf16);
  return cuda_err(cudaGetLastError());
}

size_t matryoshka_dense_operand_scratch_bytes() { return static_cast<size_t>(148) * 16 * 32 * sizeof(unsigned); }

const char* matryoshka_dense_operand_launch(const float* z, int B, int H, const float* scale, float thr,
                                            const int* level_start, int n_levels, uint16_t* a_hi, uint16_t* a_lo,
                                            unsigned long long* level_count, void* scratch, cudaStream_t stream,
                                            uint16_t* mask, int mask_pitch) {
  if ((H % 8) != 0) return "matryoshka_dense_operand: H must be a multiple of 8";
  if (mask != nullptr && ((mask_pitch % 8) != 0 || (reinterpret_cast<uintptr_t>(mask) & 15) != 0))
    return "matryoshka_dense_operand: the mask needs 16-byte aligned rows";
  if (n_levels > 32) return "matryoshka_dense_operand: at most 32 levels";
  size_t g = (static_cast<size_t>(B) * (H / 8) + 255) / 256;
  if (g > 148 * 16) g = 148 * 16;
  unsigned* partial = static_cast<unsigned*>(scratch);
  matryoshka_dense_operand_kernel<<<static_cast<int>(g), 256, 0, stream>>>(z, B, H, scale, thr, level_start, n_levels,
                                                                           a_hi, a_lo, partial, mask, mask_pitch);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cudaGetErrorString(e);
  count_launches(1);
  sum_level_counts_kernel<<<n_levels, 256, 0, stream>>>(partial, static_cast<int>(g), 32, n_levels, level_count);
  return cuda_err(cudaGetLastError());
}

const char* matryoshka_dense_tail_launch(const uint16_t* a_hi, const uint16_t* a_lo, const uint16_t* t_bf16,
                                        const int* level_start, int n_levels, int B, int H, int D, const float* bias,
                                        float* result, cudaStream_t stream) {
  if ((H % 8) != 0) return "matryoshka_dense_tail: H must be a multiple of 8";
  const int g = B < 148 * 16 ? B : 148 * 16;
  matryoshka_dense_tail_kernel<<<g, 128, 0, stream>>>(a_hi, a_lo, t_bf16, level_start, n_levels, B, H, D, bias, result);
  return cuda_err(cudaGetLastError());
}

const char* max_row_norm_launch(const float* w, int H, int D, float* out, cudaStream_t stream) {
  cudaError_t e = cudaMemsetAsync(out, 0, sizeof(float), stream);
  if (e != cudaSuccess) return cudaGetErrorString(e);
  max_row_norm_kernel<<<(H + 7) / 8, 256, 0, stream>>>(w, H, D, out);
  return cuda_err(cudaGetLastError());
}

const char* row_threshold_launch(const float* x, int B, int D, const float* wmax, float thr_value, float* thr,
                                 cudaStream_t stream) {
  row_threshold_kernel<<<(B + 7) / 8, 256, 0, stream>>>(x, B, D, wmax, thr_value, thr);
  return cuda_err(cudaGetLastError());
}

size_t decode_matryoshka_scratch_bytes(int num_sms) {
  return static_cast<size_t>(num_sms) * 8 * kMatWarps * 8 * sizeof(unsigned);
}

const char* decode_matryoshka_launch(const void* cand, const int* cand_cnt, int nsub, int cap, int B,
                                     const uint32_t* packed, const float* scale, const int* level_start,
                                     int n_levels, int H, int D, const float* bias, float* result,
                                     unsigned long long* level_count, const float* x_f32, const float* w_f32,
                                     const float* b_enc, float thr_value, int exact, void* scratch, int num_sms,
                                     cudaStream_t stream, int32_t* active_idx, int active_cap, int* active_cnt,
                                     const float* resid_in, float* resid_out, const int* poison_flag) {
  if (n_levels > 8) return "decode_matryoshka: at most 8 levels (n_bits <= 8)";
  if (D > 512 || (D % 16) != 0) return "decode_matryoshka: D must be a multiple of 16, <= 512";
  // Resident blocks per SM (launch bounds). Six (80 registers) is the fastest steady state; a batch whose rows fit one
  // wave of 7 or 8 blocks per SM but not of 6 (B = 4096 on 148 SMs: 27.7 rows per SM against 24 warps) would run two
  // half-empty waves of a latency-bound kernel, so it takes the smallest occupancy that holds every row at once.
  int bps = 6;
  const long long rows_per_wave6 = static_cast<long long>(num_sms) * 6 * kMatWarps;
  if (B > rows_per_wave6 && B <= static_cast<long long>(num_sms) * 7 * kMatWarps) bps = 7;
  else if (B > rows_per_wave6 && B <= static_cast<long long>(num_sms) * 8 * kMatWarps) bps = 8;
  int blocks = (B + kMatWarps - 1) / kMatWarps;
  if (blocks > num_sms * bps) blocks = num_sms * bps;   // = resident blocks
  (void)scratch;   // round 1: per-warp partial counts for a second kernel; the counts now leave through atomics
  const uint2* c2 = reinterpret_cast<const uint2*>(cand);
#define QSAE_MAT_B(NL, BPS) \
  decode_matryoshka_kernel<NL, BPS><<<blocks, kMatWarps * 32, 0, stream>>>(c2, cand_cnt, nsub, cap, B, packed, scale, level_start, \
      n_levels, H, D, bias, result, level_count, x_f32, w_f32, b_enc, thr_value, exact, active_idx, active_cap, active_cnt, \
      resid_in, resid_out, poison_flag)
#define QSAE_MAT(NL) \
  do { if (bps == 8) QSAE_MAT_B(NL, 8); else if (bps == 7) QSAE_MAT_B(NL, 7); else QSAE_MAT_B(NL, 6); } while (0)
  if (n_levels <= 1) QSAE_MAT(1);
  else if (n_levels <= 2) QSAE_MAT(2);
  else if (n_levels <= 4) QSAE_MAT(4);
  else QSAE_MAT(8);
#undef QSAE_MAT_B
#undef QSAE_MAT
  return cuda_err(cudaGetLastError());
}

}  // namespace qsae
