// Training-side kernels adjacent to the forward (SURVEY 8f-4). The reference gets all of this from eager autograd
// over dense [B, H] latents and dense [H, D n_bits] soft-bit tensors; here every piece works on the sparse forward
// quantities (top-k values / indices, active lists) and streams each weight matrix exactly once:
//   * rows_scatter_add / rows_gather_dot / column_sum: the sparse outer products and row dots of the b_sae
//     decoder and encoder backward (sae/binary.py:24-47, 91-103 under loss.backward());
//   * bsae_logit_grad: chain rule through the sigmoid bits + the polarize_loss gradient (sae/binary.py:26-43);
//   * matryoshka_scatter / matryoshka_grad_finish: STE backward of the q_sae level decoder wrt weight and
//     weight_mirror (sae/quantized_matryoshka.py:94-121) and apply_secant_grad (:145-190);
//   * mask_column_count: z2 of the same backward from a dense activity mask (the product itself runs on the tensor
//     cores, wgrad_sm100.cu);
//   * radix select + apply kernels: STEWeights.init_mask / update_mask (RigL drop / grow, sae/ternary.py:27-87) and
//     mask_grad (:89-90);
//   * bwd_* kernels: the deterministic latent-major backward of baseline_sae (sae/baseline.py:17-40), and with
//     bsae_latent_reduce_kernel the deterministic b_sae backward (the logit chain rule fused into the reduction).
// All HBM-bound elementwise / scatter work: no tensor cores. Compiled without fast-math: the logistic is the literal
// 1 / (1 + expf(-w)) the packing kernels use, so Bsign here equals the sign packed for the forward.
#include <cuda_runtime.h>
#include <stdint.h>

#include "kernels.h"

namespace qsae {

namespace {

__device__ __forceinline__ float logistic(float w) { return 1.0f / (1.0f + expf(-w)); }

// one 16-byte reduction into global memory (sm_90+): four fp32 adds in one L2 transaction
__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// ---------------------------------------------------------------------------------------------
// dst[idx[b,j], :] += scale * coef[b,j] * src[b, :]   (+ dst_col[idx[b,j]] += scale * coef[b,j])
// One warp per row b: the row of src stays in registers (NCH float4 per lane), each list entry is NCH 16-byte
// reductions per lane. Atomic order is not fixed: results agree with a serial sum to fp32 rounding.
// ---------------------------------------------------------------------------------------------
template <int NCH>
__global__ void __launch_bounds__(256)
rows_scatter_add_kernel(const float* __restrict__ coef, const int32_t* __restrict__ idx, const float* __restrict__ src,
                        int B, int k, int D, int H, float scale, float* __restrict__ dst, float* __restrict__ dst_col) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int nchunk = D >> 2;
  for (int row = warp; row < B; row += nwarps) {
    float4 s[NCH > 0 ? NCH : 1];
    if (NCH > 0) {
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        const int q = lane + 32 * c;
        s[c] = q < nchunk ? reinterpret_cast<const float4*>(src + static_cast<size_t>(row) * D)[q] : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    for (int j0 = 0; j0 < k; j0 += 32) {
      const int jl = j0 + lane;
      const int my_h = jl < k ? idx[static_cast<size_t>(row) * k + jl] : -1;
      const float my_c = (jl < k && coef != nullptr) ? coef[static_cast<size_t>(row) * k + jl] : 1.0f;
      const int nj = min(32, k - j0);
      for (int j = 0; j < nj; ++j) {
        const int h = __shfl_sync(0xffffffffu, my_h, j);
        const float c = scale * __shfl_sync(0xffffffffu, my_c, j);
        if (h < 0 || h >= H || c == 0.f) continue;
        float* drow = dst + static_cast<size_t>(h) * D;
        if (NCH > 0) {
#pragma unroll
          for (int cc = 0; cc < NCH; ++cc) {
            const int q = lane + 32 * cc;
            if (q < nchunk) red_add_v4(drow + 4 * q, c * s[cc].x, c * s[cc].y, c * s[cc].z, c * s[cc].w);
          }
        } else {
          for (int d = lane; d < D; d += 32) atomicAdd(drow + d, c * src[static_cast<size_t>(row) * D + d]);
        }
        if (dst_col != nullptr && lane == 0) atomicAdd(dst_col + h, c);
      }
    }
  }
}

// out[b,j] = scale * <g[b,:], rows[idx[b,j], :]>  (0 for empty entries). Warp per row b, deterministic.
__global__ void __launch_bounds__(256)
rows_gather_dot_kernel(const float* __restrict__ g, const float* __restrict__ rows, const int32_t* __restrict__ idx,
                       int B, int k, int D, int H, float scale, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const bool vec = (D & 3) == 0;
  for (int row = warp; row < B; row += nwarps) {
    const float* grow = g + static_cast<size_t>(row) * D;
    for (int j = 0; j < k; ++j) {
      const int h = idx[static_cast<size_t>(row) * k + j];
      float acc = 0.f;
      if (h >= 0 && h < H) {
        const float* r = rows + static_cast<size_t>(h) * D;
        if (vec) {
          for (int q = lane; q < (D >> 2); q += 32) {
            const float4 a = reinterpret_cast<const float4*>(grow)[q];
            const float4 b = reinterpret_cast<const float4*>(r)[q];
            acc += a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w;
          }
        } else {
          for (int d = lane; d < D; d += 32) acc += grow[d] * r[d];
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if (lane == 0) out[static_cast<size_t>(row) * k + j] = scale * acc;
    }
  }
}

// out[c] += scale * sum_r src[r, c]. blockDim (32, 8): 128-byte row segments per warp; partial sums join by atomics.
__global__ void __launch_bounds__(256)
column_sum_kernel(const float* __restrict__ src, int R, int C, float scale, float* __restrict__ out) {
  __shared__ float part[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  float acc = 0.f;
  if (c < C)
    for (int r = blockIdx.y * 8 + threadIdx.y; r < R; r += gridDim.y * 8) acc += src[static_cast<size_t>(r) * C + c];
  part[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += part[i][threadIdx.x];
    atomicAdd(out + c, scale * t);
  }
}

// ---------------------------------------------------------------------------------------------
// b_sae: grad_logits[h, d n + i] (+)= (G[h,d] c_i + gp 2^i (1 - 2p) / N) p (1 - p)     (sae/binary.py:26-43)
// One thread per group of four consecutive logits of a row (n_bits in {1, 2, 4, 8, ...}: a group never straddles
// rows because D n_bits % 4 == 0 on this path; the launcher falls back to VEC = 1 otherwise).
// gp: device scalar (upstream gradient of polarize_loss, e.g. polarize_lambda) or NULL = gp_host.
// ---------------------------------------------------------------------------------------------
// The three helpers below are the whole per-element formula; bsae_latent_reduce_kernel (the deterministic backward)
// calls the same ones, so both paths give the same bits for the same G. The logistic uses the fast exponential /
// reciprocal (relative error ~1e-6: a gradient, not a thresholded bit -- the packing kernels keep the exact form).
// gp / N, N = H D n_bits: the polarize gradient's scale, divided once per thread
__device__ __forceinline__ float bsae_polarize_scale(const float* gp_dev, float gp_host, int H, int cols) {
  return (gp_dev != nullptr ? *gp_dev : gp_host) / static_cast<float>(static_cast<double>(H) * cols);
}

// bit i of n: its coefficient c_i (2^i, the sign bit -2^(n-1)) and gp 2^i
__device__ __forceinline__ void bsae_bit_consts(int i, int n_bits, float gp, float& ci, float& gpw) {
  const float pw = static_cast<float>(1u << i);
  ci = (i == n_bits - 1) ? -pw : pw;
  gpw = gp * pw;
}

__device__ __forceinline__ float bsae_logit_grad_value(float w, float up, float ci, float gpw) {
  const float p = __frcp_rn(1.0f + __expf(-w));
  return (up * ci + gpw * (1.f - 2.f * p)) * (p * (1.f - p));
}

// blockIdx.x / threadIdx.x pick the group of VEC consecutive logits of a row, blockIdx.y strides over the rows: bit
// index, bit weight and dictionary column are per-thread constants.
template <int VEC>
__global__ void __launch_bounds__(256)
bsae_logit_grad_kernel(const float* __restrict__ logits, const float* __restrict__ G, int H, int D, int n_bits,
                       const float* __restrict__ gp_dev, float gp_host, int accumulate, float* __restrict__ grad) {
  const int cols = D * n_bits;
  const int groups = cols / VEC;
  const int cg = blockIdx.x * blockDim.x + threadIdx.x;
  if (cg >= groups) return;
  const float gp = bsae_polarize_scale(gp_dev, gp_host, H, cols);
  int dcol[VEC];
  float ci[VEC], gpw[VEC];
#pragma unroll
  for (int u = 0; u < VEC; ++u) {
    const int col = cg * VEC + u;
    dcol[u] = col / n_bits;
    bsae_bit_consts(col - dcol[u] * n_bits, n_bits, gp, ci[u], gpw[u]);
  }
  constexpr int R = 2;                                // rows in flight per thread
  for (int h0 = blockIdx.y; h0 < H; h0 += R * gridDim.y) {
    float w[R][VEC], up0[R][VEC], old[R][VEC];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int h = h0 + r * gridDim.y;
      if (h >= H) continue;
      const size_t e = static_cast<size_t>(h) * groups + cg;
      if (VEC == 4) {
        const float4 v = reinterpret_cast<const float4*>(logits)[e];
        w[r][0] = v.x; w[r][1 % VEC] = v.y; w[r][2 % VEC] = v.z; w[r][3 % VEC] = v.w;
        if (accumulate) {
          const float4 o = reinterpret_cast<const float4*>(grad)[e];
          old[r][0] = o.x; old[r][1 % VEC] = o.y; old[r][2 % VEC] = o.z; old[r][3 % VEC] = o.w;
        }
      } else {
        w[r][0] = logits[e];
        if (accumulate) old[r][0] = grad[e];
      }
#pragma unroll
      for (int u = 0; u < VEC; ++u) up0[r][u] = G != nullptr ? G[static_cast<size_t>(h) * D + dcol[u]] : 0.f;
    }
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int h = h0 + r * gridDim.y;
      if (h >= H) continue;
      const size_t e = static_cast<size_t>(h) * groups + cg;
      float o[VEC];
#pragma unroll
      for (int u = 0; u < VEC; ++u) {
        o[u] = bsae_logit_grad_value(w[r][u], up0[r][u], ci[u], gpw[u]);
        if (accumulate) o[u] += old[r][u];
      }
      if (VEC == 4) reinterpret_cast<float4*>(grad)[e] = make_float4(o[0], o[1 % VEC], o[2 % VEC], o[3 % VEC]);
      else grad[e] = o[0];
    }
  }
}

// ---------------------------------------------------------------------------------------------
// q_sae: M[h,:] += g_level(h)[b,:] for every active (b, h); z2[h] += 1                (quantized_matryoshka.py:121,137)
// Warp per row b over its active list (idx [B, cap], empty = -1, as exported by qsae_matryoshka_forward_active).
// ---------------------------------------------------------------------------------------------
struct LevelPtrs {
  const float* g[8];
  int start[9];
  int n;
};

__global__ void __launch_bounds__(256)
matryoshka_scatter_kernel(const int32_t* __restrict__ idx, int B, int cap, int H, int D, LevelPtrs lv,
                          float* __restrict__ M, int32_t* __restrict__ z2) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int nchunk = D >> 2;
  for (int row = warp; row < B; row += nwarps) {
    for (int j0 = 0; j0 < cap; j0 += 32) {
      const int jl = j0 + lane;
      const int my_h = jl < cap ? idx[static_cast<size_t>(row) * cap + jl] : -1;
      if (__ballot_sync(0xffffffffu, my_h >= 0) == 0u) continue;
      for (int j = 0; j < 32; ++j) {
        const int h = __shfl_sync(0xffffffffu, my_h, j);
        if (h < 0 || h >= H) continue;
        int l = 0;
        while (l + 1 < lv.n && h >= lv.start[l + 1]) ++l;
        const float* grow = lv.g[l] + static_cast<size_t>(row) * D;
        float* drow = M + static_cast<size_t>(h) * D;
        if ((D & 3) == 0) {
          for (int q = lane; q < nchunk; q += 32) {
            const float4 s = reinterpret_cast<const float4*>(grow)[q];
            red_add_v4(drow + 4 * q, s.x, s.y, s.z, s.w);
          }
        } else {
          for (int d = lane; d < D; d += 32) atomicAdd(drow + d, grow[d]);
        }
        if (lane == 0) atomicAdd(z2 + h, 1);
      }
    }
  }
}

// grad_W[h,d]  += (ste ? alpha[h] M[h,d] : 0  -  (secant ? c m(h) z2[h] alpha[h]^2 Bsign(W[h,d]) : 0)) s'(W[h,d])
// and the same for weight_mirror                                     (quantized_matryoshka.py:94-95, 167-189)
__global__ void __launch_bounds__(256)
matryoshka_grad_finish_kernel(const float* __restrict__ W, const float* __restrict__ Wm, const float* __restrict__ M,
                              const int32_t* __restrict__ z2, const float* __restrict__ alpha, LevelPtrs lv, int H, int D,
                              float c, int joint_bits, float* __restrict__ gW, float* __restrict__ gWm) {
  const size_t total = static_cast<size_t>(H) * D;
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  for (size_t e = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; e < total; e += stride) {
    const int h = static_cast<int>(e / D);
    const float a = alpha[h];
    float sec = 0.f;
    if (z2 != nullptr) {
      float m = 1.f;
      if (joint_bits > 0) {
        int l = 0;
        while (l + 1 < lv.n && h >= lv.start[l + 1]) ++l;
        m = static_cast<float>(joint_bits - l);
      }
      sec = c * m * static_cast<float>(z2[h]) * a * a;
    }
    const float up = M != nullptr ? a * M[e] : 0.f;
    const float p = logistic(W[e]), pm = logistic(Wm[e]);
    gW[e] += (up - (p >= 0.5f ? sec : -sec)) * (p * (1.f - p));
    gWm[e] += (up - (pm >= 0.5f ? sec : -sec)) * (pm * (1.f - pm));
  }
}

// z2[h] += #{b : mask[b,h] != 0} for a bf16 0/1 activity mask [B, H] (the dense route's z2, :137): 8 columns per
// thread (16-byte loads, a warp reads 512 consecutive bytes of a row), a slice of the rows per grid row, one integer
// atomic per column and slice -- exact, and the same bits in any order.
__global__ void __launch_bounds__(256)
mask_column_count_kernel(const uint16_t* __restrict__ mask, int B, int H, int rows_per, int32_t* __restrict__ z2) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (8 * g >= H) return;
  const int r0 = blockIdx.y * rows_per;
  const int r1 = min(B, r0 + rows_per);
  int c[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const uint16_t* col = mask + 8 * static_cast<size_t>(g);
#pragma unroll 4
  for (int r = r0; r < r1; ++r) {
    const uint4 v = __ldcs(reinterpret_cast<const uint4*>(col + static_cast<size_t>(r) * H));
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      c[2 * q] += (w[q] & 0x7fffu) != 0u;
      c[2 * q + 1] += (w[q] & 0x7fff0000u) != 0u;
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j)
    if (c[j] != 0) atomicAdd(z2 + 8 * g + j, c[j]);
}

// ---------------------------------------------------------------------------------------------
// RigL (sae/ternary.py:27-87): exact k-th order statistics over D H elements by a three-pass radix select on the
// fp32 bit patterns (non-negative floats order like their bits), then elementwise apply kernels. No host sync.
// ---------------------------------------------------------------------------------------------
constexpr int kSelBins = 2048;

struct SelectState {
  unsigned int prefix;        // bits of the k-th smallest transformed key found so far
  unsigned int prefix_mask;   // which bits of `prefix` are decided
  unsigned long long k;       // rank (1-based) still to locate inside the current prefix; after the last pass:
                              // how many elements EQUAL to the threshold belong to the selection
  unsigned int hist[kSelBins];
};

enum SelectMode {
  kSelAbsActive = 0,     // key = |w[i]| over mask[i] != 0, k-th smallest            (update_mask drop, :66-67)
  kSelAbsAll = 1,        // key = |w[i]| over all i, k-th smallest                   (init_mask, :32-33)
  kSelScoreInactive = 2  // key = |dmean[i / H]| |amean[i % H]| over mask[i] == 0, k-th LARGEST (grow, :76-82)
};

struct SelectSrc {
  const float* w;
  const float* mask;
  const float* amean;   // [H]
  const float* dmean;   // [D]
  int H;
  size_t n;
};

template <int MODE>
__device__ __forceinline__ bool select_key(const SelectSrc& s, size_t i, unsigned int* key) {
  if (MODE == kSelAbsActive) {
    if (s.mask[i] == 0.f) return false;
    *key = __float_as_uint(fabsf(s.w[i]));
    return true;
  }
  if (MODE == kSelAbsAll) {
    *key = __float_as_uint(fabsf(s.w[i]));
    return true;
  }
  if (s.mask[i] != 0.f) return false;
  const size_t d = i / static_cast<size_t>(s.H);
  const int h = static_cast<int>(i - d * s.H);
  *key = ~__float_as_uint(fabsf(s.dmean[d]) * fabsf(s.amean[h]));   // largest first
  return true;
}

// Four consecutive elements [4 g, 4 g + 4) with 16-byte loads (the launcher guarantees n % 4 == 0, H % 4 == 0 and
// 16-byte aligned arrays, so the four share their row d of the score matrix). -> 4-bit mask of valid elements.
template <int MODE>
__device__ __forceinline__ unsigned int select_keys4(const SelectSrc& s, size_t g, unsigned int (&key)[4]) {
  unsigned int valid = 0u;
  if (MODE == kSelAbsActive || MODE == kSelAbsAll) {
    const float4 w = reinterpret_cast<const float4*>(s.w)[g];
    key[0] = __float_as_uint(fabsf(w.x)); key[1] = __float_as_uint(fabsf(w.y));
    key[2] = __float_as_uint(fabsf(w.z)); key[3] = __float_as_uint(fabsf(w.w));
    if (MODE == kSelAbsAll) return 0xfu;
    const float4 m = reinterpret_cast<const float4*>(s.mask)[g];
    valid = (m.x != 0.f ? 1u : 0u) | (m.y != 0.f ? 2u : 0u) | (m.z != 0.f ? 4u : 0u) | (m.w != 0.f ? 8u : 0u);
    return valid;
  }
  const float4 m = reinterpret_cast<const float4*>(s.mask)[g];
  valid = (m.x == 0.f ? 1u : 0u) | (m.y == 0.f ? 2u : 0u) | (m.z == 0.f ? 4u : 0u) | (m.w == 0.f ? 8u : 0u);
  if (valid == 0u) return 0u;
  const unsigned int first = static_cast<unsigned int>(g) * 4u;          // n < 2^32 (checked by the C ABI)
  const unsigned int d = first / static_cast<unsigned int>(s.H);
  const unsigned int h = first - d * static_cast<unsigned int>(s.H);
  const float dm = fabsf(s.dmean[d]);
  const float4 a = *reinterpret_cast<const float4*>(s.amean + h);
  key[0] = ~__float_as_uint(dm * fabsf(a.x)); key[1] = ~__float_as_uint(dm * fabsf(a.y));
  key[2] = ~__float_as_uint(dm * fabsf(a.z)); key[3] = ~__float_as_uint(dm * fabsf(a.w));
  return valid;
}

// The first pass sees a few exponent bins only (all |w| of a layer share their leading bits): lanes that hit the same
// bin are merged with __match_any_sync and one lane adds the group's count. Four independent elements per thread and
// trip keep enough loads in flight to stream at HBM rate.
template <int MODE, bool VEC>
__global__ void __launch_bounds__(256)
select_hist_kernel(SelectSrc s, int shift, int bits, SelectState* st) {
  __shared__ unsigned int h[kSelBins];
  for (int i = threadIdx.x; i < kSelBins; i += blockDim.x) h[i] = 0;
  __syncthreads();
  const unsigned int prefix = st->prefix, pmask = st->prefix_mask;
  const unsigned int dmask = (1u << bits) - 1u;
  const int lane = threadIdx.x & 31;
  constexpr int E = VEC ? 4 : 1;            // elements per group
  constexpr int U = VEC ? 2 : 4;            // groups in flight per thread and trip
  const size_t ng = s.n / E;
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  const size_t first = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  for (size_t base = first - lane; base < ng; base += U * stride) {      // warp-uniform trip count
    unsigned int bin[U][E];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const size_t g = base + lane + u * stride;
      unsigned int key[4] = {0u, 0u, 0u, 0u};
      unsigned int valid = 0u;
      if (g < ng) {
        if (VEC) valid = select_keys4<MODE>(s, g, key);
        else valid = select_key<MODE>(s, g, &key[0]) ? 1u : 0u;
      }
#pragma unroll
      for (int e = 0; e < E; ++e)
        bin[u][e] = (((valid >> e) & 1u) && (key[e] & pmask) == prefix) ? ((key[e] >> shift) & dmask) : 0xffffffffu;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
#pragma unroll
      for (int e = 0; e < E; ++e) {
        if (__ballot_sync(0xffffffffu, bin[u][e] != 0xffffffffu) == 0u) continue;
        const unsigned int peers = __match_any_sync(0xffffffffu, bin[u][e]);
        if (bin[u][e] != 0xffffffffu && lane == __ffs(peers) - 1) atomicAdd(&h[bin[u][e]], static_cast<unsigned int>(__popc(peers)));
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kSelBins; i += blockDim.x)
    if (h[i] != 0u) atomicAdd(&st->hist[i], h[i]);
}

__global__ void select_init_kernel(SelectState* st, unsigned long long k) {
  if (threadIdx.x == 0) { st->prefix = 0; st->prefix_mask = 0; st->k = k; }
  for (int i = threadIdx.x; i < kSelBins; i += blockDim.x) st->hist[i] = 0;
}

// Exclusive prefix sums of 2048 counters held 8 per thread by a block of 256 threads (64-bit: 2^32 elements may tie).
__device__ __forceinline__ unsigned long long block_exclusive_scan_256(unsigned long long local, unsigned long long* total) {
  __shared__ unsigned long long warp_tot[8];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  unsigned long long incl = local;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) warp_tot[wid] = incl;
  __syncthreads();
  unsigned long long base = 0, all = 0;
#pragma unroll
  for (int w = 0; w < 8; ++w) {
    if (w < wid) base += warp_tot[w];
    all += warp_tot[w];
  }
  __syncthreads();
  *total = all;
  return base + incl - local;
}

// the bin that holds rank k (block of 256 threads, 8 bins each), then clear the histogram for the next pass
__global__ void __launch_bounds__(256) select_pick_kernel(int shift, int bits, SelectState* st) {
  const int nb = 1 << bits;
  unsigned int c[8];
  unsigned long long local = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int b = threadIdx.x * 8 + j;
    c[j] = b < nb ? st->hist[b] : 0u;
    local += c[j];
  }
  const unsigned long long k = st->k;
  unsigned long long total;
  unsigned long long cum = block_exclusive_scan_256(local, &total);
  __syncthreads();                                   // everybody has read st->k and the histogram
  if (k != ~0ull && total < k) {                     // fewer than k candidates: everything is selected
    if (threadIdx.x == 0) {
      st->k = ~0ull;
      st->prefix |= static_cast<unsigned int>(nb - 1) << shift;
      st->prefix_mask |= ((1u << bits) - 1u) << shift;
    }
  } else if (k == ~0ull) {
    if (threadIdx.x == 0) {
      st->prefix |= static_cast<unsigned int>(nb - 1) << shift;
      st->prefix_mask |= ((1u << bits) - 1u) << shift;
    }
  } else if (cum < k && k <= cum + local) {          // exactly one thread owns rank k
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (cum + c[j] >= k) {
        st->k = k - cum;
        st->prefix |= static_cast<unsigned int>(threadIdx.x * 8 + j) << shift;
        st->prefix_mask |= ((1u << bits) - 1u) << shift;
        break;
      }
      cum += c[j];
    }
  }
  for (int i = threadIdx.x; i < kSelBins; i += blockDim.x) st->hist[i] = 0;
}

// drop (:68-69): active &= !(|w| <= threshold) -- every tie at the threshold goes
__global__ void __launch_bounds__(256)
rigl_drop_apply_kernel(const float* __restrict__ w, float* __restrict__ mask, size_t n, int vec, const SelectState* st) {
  const unsigned int thr = st->prefix;
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (vec) {
    for (size_t g = tid; g < n / 4; g += stride) {
      const float4 ww = reinterpret_cast<const float4*>(w)[g];
      float4 m = reinterpret_cast<float4*>(mask)[g];
      bool ch = false;
      if (m.x != 0.f && __float_as_uint(fabsf(ww.x)) <= thr) { m.x = 0.f; ch = true; }
      if (m.y != 0.f && __float_as_uint(fabsf(ww.y)) <= thr) { m.y = 0.f; ch = true; }
      if (m.z != 0.f && __float_as_uint(fabsf(ww.z)) <= thr) { m.z = 0.f; ch = true; }
      if (m.w != 0.f && __float_as_uint(fabsf(ww.w)) <= thr) { m.w = 0.f; ch = true; }
      if (ch) reinterpret_cast<float4*>(mask)[g] = m;
    }
    return;
  }
  for (size_t i = tid; i < n; i += stride)
    if (mask[i] != 0.f && __float_as_uint(fabsf(w[i])) <= thr) mask[i] = 0.f;
}

// Tie-ranked apply: elements with key < T are selected, of those == T the first st->k by flat index.
// Every block owns a contiguous range; ties are counted per block, scanned by one block, ranked inside the range.
template <int MODE, bool VEC>
__global__ void __launch_bounds__(256)
select_tie_count_kernel(SelectSrc s, size_t per_block, const SelectState* st, unsigned int* tie_count) {
  __shared__ unsigned int total;
  if (threadIdx.x == 0) total = 0;
  __syncthreads();
  const unsigned int T = st->prefix;
  const size_t lo = static_cast<size_t>(blockIdx.x) * per_block;          // per_block is a multiple of 256 (and of 4)
  const size_t hi = lo + per_block < s.n ? lo + per_block : s.n;
  unsigned int c = 0;
  if (VEC) {
    for (size_t g = lo / 4 + threadIdx.x; g < hi / 4; g += blockDim.x) {
      unsigned int key[4];
      const unsigned int valid = select_keys4<MODE>(s, g, key);
#pragma unroll
      for (int e = 0; e < 4; ++e) c += (((valid >> e) & 1u) && key[e] == T) ? 1u : 0u;
    }
  } else {
    for (size_t i = lo + threadIdx.x; i < hi; i += blockDim.x) {
      unsigned int key;
      if (select_key<MODE>(s, i, &key) && key == T) ++c;
    }
  }
  if (c) atomicAdd(&total, c);
  __syncthreads();
  if (threadIdx.x == 0) tie_count[blockIdx.x] = total;
}

// exclusive prefix of the per-block tie counts (at most 2048 blocks), total in [nblocks]
__global__ void __launch_bounds__(256) select_tie_scan_kernel(unsigned int* tie_count, int nblocks) {
  unsigned int c[8];
  unsigned long long local = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int b = threadIdx.x * 8 + j;
    c[j] = b < nblocks ? tie_count[b] : 0u;
    local += c[j];
  }
  unsigned long long total;
  unsigned long long run = block_exclusive_scan_256(local, &total);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int b = threadIdx.x * 8 + j;
    if (b < nblocks) tie_count[b] = run > 0xffffffffull ? 0xffffffffu : static_cast<unsigned int>(run);
    run += c[j];
  }
  if (threadIdx.x == 0) tie_count[nblocks] = total > 0xffffffffull ? 0xffffffffu : static_cast<unsigned int>(total);
}

// selected -> new_value in mask (init_mask: 0, grow: 1); then weight *= mask over the whole range (:39, :86-87)
template <int MODE, bool VEC>
__global__ void __launch_bounds__(256)
select_apply_kernel(SelectSrc s, size_t per_block, const SelectState* st, const unsigned int* tie_base,
                    float new_value, float* __restrict__ mask, float* __restrict__ weight) {
  __shared__ unsigned int warp_cnt[8];
  __shared__ unsigned int running;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (threadIdx.x == 0) running = tie_base[blockIdx.x];
  __syncthreads();
  const unsigned int T = st->prefix;
  const unsigned long long take = st->k;
  const size_t lo = static_cast<size_t>(blockIdx.x) * per_block;
  const size_t hi = lo + per_block < s.n ? lo + per_block : s.n;
  if (VEC && tie_base[blockIdx.x + 1] == tie_base[blockIdx.x]) {
    // no element of this range sits exactly on the threshold (the usual case): plain elementwise pass, 16-byte accesses
    for (size_t g = lo / 4 + threadIdx.x; g < hi / 4; g += blockDim.x) {
      unsigned int key[4];
      const unsigned int valid = select_keys4<MODE>(s, g, key);
      float4 m = reinterpret_cast<float4*>(mask)[g];
      float* mm = reinterpret_cast<float*>(&m);
      bool ch = false, any_zero = false;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (((valid >> e) & 1u) && key[e] < T) { mm[e] = new_value; ch = true; }
        any_zero |= mm[e] == 0.f;
      }
      if (ch) reinterpret_cast<float4*>(mask)[g] = m;
      if (weight != nullptr && any_zero) {
        float4 w = reinterpret_cast<float4*>(weight)[g];
        if (m.x == 0.f) w.x = 0.f * w.x;
        if (m.y == 0.f) w.y = 0.f * w.y;
        if (m.z == 0.f) w.z = 0.f * w.z;
        if (m.w == 0.f) w.w = 0.f * w.w;
        reinterpret_cast<float4*>(weight)[g] = w;
      }
    }
    return;
  }
  if (tie_base[blockIdx.x + 1] == tie_base[blockIdx.x]) {
    // no element of this range sits exactly on the threshold (the usual case): plain elementwise pass
    for (size_t i = lo + threadIdx.x; i < hi; i += blockDim.x) {
      unsigned int key = 0;
      float m = mask[i];
      if (select_key<MODE>(s, i, &key) && key < T) { m = new_value; mask[i] = m; }
      if (weight != nullptr && m == 0.f) weight[i] = 0.f * weight[i];
    }
    return;
  }
  for (size_t base = lo; base < hi; base += blockDim.x) {
    const size_t i = base + threadIdx.x;
    unsigned int key = 0;
    const bool valid = i < hi && select_key<MODE>(s, i, &key);
    const bool tie = valid && key == T;
    const unsigned int bal = __ballot_sync(0xffffffffu, tie);
    if (lane == 0) warp_cnt[wid] = __popc(bal);
    __syncthreads();
    unsigned int off = running;
    for (int w2 = 0; w2 < wid; ++w2) off += warp_cnt[w2];
    const unsigned int rank = off + __popc(bal & ((1u << lane) - 1u));
    const bool sel = valid && (key < T || (tie && static_cast<unsigned long long>(rank) < take));
    if (i < hi) {
      float m = mask[i];
      if (sel) { m = new_value; mask[i] = m; }
      if (weight != nullptr && m == 0.f) weight[i] = 0.f * weight[i];   // weight *= mask (keeps the sign of zero / NaN like the reference)
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      unsigned int t = 0;
      for (int w2 = 0; w2 < 8; ++w2) t += warp_cnt[w2];
      running += t;
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(256)
mul_inplace_kernel(float* __restrict__ a, const float* __restrict__ b, size_t n) {
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) a[i] *= b[i];
}

int grid_for(size_t work_items, int threads, int max_blocks) {
  size_t g = (work_items + threads - 1) / threads;
  if (g < 1) g = 1;
  if (g > static_cast<size_t>(max_blocks)) g = max_blocks;
  return static_cast<int>(g);
}

// 16-byte accesses over groups of four consecutive elements are possible
bool select_vec_ok(const SelectSrc& s) {
  auto al = [](const void* p) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  return (s.n & 3) == 0 && (s.H & 3) == 0 && al(s.w) && al(s.mask) && al(s.amean);
}

template <int MODE>
const char* run_select(const SelectSrc& s, unsigned long long k, SelectState* st, int sms, cudaStream_t stream) {
  select_init_kernel<<<1, 256, 0, stream>>>(st, k);
  const int grid = grid_for(s.n, 256 * 8, sms * 8);
  const int shifts[3] = {21, 10, 0}, bits[3] = {11, 11, 10};
  for (int p = 0; p < 3; ++p) {
    if (select_vec_ok(s)) select_hist_kernel<MODE, true><<<grid, 256, 0, stream>>>(s, shifts[p], bits[p], st);
    else select_hist_kernel<MODE, false><<<grid, 256, 0, stream>>>(s, shifts[p], bits[p], st);
    select_pick_kernel<<<1, 256, 0, stream>>>(shifts[p], bits[p], st);
  }
  count_launches(7);
  return cuda_err(cudaGetLastError());
}

template <int MODE>
const char* run_tie_apply(const SelectSrc& s, const SelectState* st, unsigned int* tie_scratch, int nblocks,
                          float new_value, float* mask, float* weight, cudaStream_t stream) {
  size_t per = (s.n + nblocks - 1) / nblocks;
  per = (per + 255) / 256 * 256;
  const int nb = static_cast<int>((s.n + per - 1) / per);
  if (select_vec_ok(s)) select_tie_count_kernel<MODE, true><<<nb, 256, 0, stream>>>(s, per, st, tie_scratch);
  else select_tie_count_kernel<MODE, false><<<nb, 256, 0, stream>>>(s, per, st, tie_scratch);
  select_tie_scan_kernel<<<1, 256, 0, stream>>>(tie_scratch, nb);
  if (select_vec_ok(s)) select_apply_kernel<MODE, true><<<nb, 256, 0, stream>>>(s, per, st, tie_scratch, new_value, mask, weight);
  else select_apply_kernel<MODE, false><<<nb, 256, 0, stream>>>(s, per, st, tie_scratch, new_value, mask, weight);
  count_launches(3);
  return cuda_err(cudaGetLastError());
}

}  // namespace

const char* rows_scatter_add_launch(const float* coef, const int32_t* idx, const float* src, int B, int k, int D, int H,
                                    float scale, float* dst, float* dst_col, cudaStream_t stream) {
  if (B == 0 || k == 0) return nullptr;
  const int grid = grid_for(static_cast<size_t>(B) * 32, 256, 148 * 8);
  const int nch = (D & 3) == 0 ? (D / 4 + 31) / 32 : 0;
  switch (nch <= 4 ? nch : 0) {
    case 1: rows_scatter_add_kernel<1><<<grid, 256, 0, stream>>>(coef, idx, src, B, k, D, H, scale, dst, dst_col); break;
    case 2: rows_scatter_add_kernel<2><<<grid, 256, 0, stream>>>(coef, idx, src, B, k, D, H, scale, dst, dst_col); break;
    case 3: rows_scatter_add_kernel<3><<<grid, 256, 0, stream>>>(coef, idx, src, B, k, D, H, scale, dst, dst_col); break;
    case 4: rows_scatter_add_kernel<4><<<grid, 256, 0, stream>>>(coef, idx, src, B, k, D, H, scale, dst, dst_col); break;
    default: rows_scatter_add_kernel<0><<<grid, 256, 0, stream>>>(coef, idx, src, B, k, D, H, scale, dst, dst_col); break;
  }
  return cuda_err(cudaGetLastError());
}

const char* rows_gather_dot_launch(const float* g, const float* rows, const int32_t* idx, int B, int k, int D, int H,
                                   float scale, float* out, cudaStream_t stream) {
  if (B == 0 || k == 0) return nullptr;
  const int grid = grid_for(static_cast<size_t>(B) * 32, 256, 148 * 8);
  rows_gather_dot_kernel<<<grid, 256, 0, stream>>>(g, rows, idx, B, k, D, H, scale, out);
  return cuda_err(cudaGetLastError());
}

const char* column_sum_launch(const float* src, int R, int C, float scale, float* out, cudaStream_t stream) {
  if (R == 0 || C == 0) return nullptr;
  const int gx = (C + 31) / 32;
  int gy = (R + 127) / 128;
  const int cap = (148 * 8 + gx - 1) / gx;
  if (gy > cap) gy = cap;
  if (gy < 1) gy = 1;
  column_sum_kernel<<<dim3(gx, gy), dim3(32, 8), 0, stream>>>(src, R, C, scale, out);
  return cuda_err(cudaGetLastError());
}

const char* bsae_logit_grad_launch(const float* logits, const float* G, int H, int D, int n_bits, const float* gp_dev,
                                   float gp_host, int accumulate, float* grad, cudaStream_t stream) {
  const size_t cols = static_cast<size_t>(D) * n_bits;
  const size_t n = static_cast<size_t>(H) * cols;
  if (n == 0) return nullptr;
  const bool vec = (cols & 3) == 0 && ((reinterpret_cast<uintptr_t>(logits) | reinterpret_cast<uintptr_t>(grad)) & 15) == 0;
  const size_t groups = vec ? cols / 4 : cols;
  const int gx = static_cast<int>((groups + 255) / 256);
  int gy = (148 * 16 + gx - 1) / gx;             // ~16 blocks per SM; every block walks H / gy rows
  if (gy > H) gy = H;
  if (gy > 65535) gy = 65535;
  if (vec)
    bsae_logit_grad_kernel<4><<<dim3(gx, gy), 256, 0, stream>>>(logits, G, H, D, n_bits, gp_dev, gp_host, accumulate, grad);
  else
    bsae_logit_grad_kernel<1><<<dim3(gx, gy), 256, 0, stream>>>(logits, G, H, D, n_bits, gp_dev, gp_host, accumulate, grad);
  return cuda_err(cudaGetLastError());
}

static bool fill_levels(LevelPtrs* lv, const float* const* g_levels, const int* level_start, int n_levels) {
  if (n_levels < 1 || n_levels > 8) return false;
  lv->n = n_levels;
  for (int i = 0; i < 8; ++i) lv->g[i] = (g_levels != nullptr && i < n_levels) ? g_levels[i] : nullptr;
  for (int i = 0; i <= n_levels; ++i) lv->start[i] = level_start[i];
  for (int i = n_levels + 1; i < 9; ++i) lv->start[i] = level_start[n_levels];
  return true;
}

const char* matryoshka_scatter_launch(const int32_t* idx, int B, int cap, int H, int D, const float* const* g_levels,
                                      const int* level_start, int n_levels, float* M, int32_t* z2, cudaStream_t stream) {
  LevelPtrs lv;
  if (!fill_levels(&lv, g_levels, level_start, n_levels)) return "matryoshka backward: 1..8 levels";
  if (B == 0 || cap == 0) return nullptr;
  matryoshka_scatter_kernel<<<grid_for(static_cast<size_t>(B) * 32, 256, 148 * 8), 256, 0, stream>>>(idx, B, cap, H, D, lv, M, z2);
  return cuda_err(cudaGetLastError());
}

const char* matryoshka_grad_finish_launch(const float* W, const float* Wm, const float* M, const int32_t* z2,
                                          const float* alpha, const int* level_start, int n_levels, int H, int D, float c,
                                          int joint_bits, float* gW, float* gWm, cudaStream_t stream) {
  LevelPtrs lv;
  if (!fill_levels(&lv, nullptr, level_start, n_levels)) return "matryoshka backward: 1..8 levels";
  const size_t n = static_cast<size_t>(H) * D;
  if (n == 0) return nullptr;
  matryoshka_grad_finish_kernel<<<grid_for(n, 256, 148 * 16), 256, 0, stream>>>(W, Wm, M, z2, alpha, lv, H, D, c, joint_bits, gW, gWm);
  return cuda_err(cudaGetLastError());
}

const char* mask_column_count_launch(const uint16_t* mask, int B, int H, int32_t* z2, cudaStream_t stream) {
  if (B <= 0 || H <= 0) return nullptr;
  const int gx = (H / 8 + 255) / 256;
  int gy = (148 * 8 + gx - 1) / gx;              // ~8 blocks per SM
  if (gy > B) gy = B;
  if (gy > 65535) gy = 65535;
  const int rows_per = (B + gy - 1) / gy;
  gy = (B + rows_per - 1) / rows_per;
  mask_column_count_kernel<<<dim3(gx, gy), 256, 0, stream>>>(mask, B, H, rows_per, z2);
  return cuda_err(cudaGetLastError());
}

size_t rigl_workspace_bytes(int sms) {
  return 1024 + sizeof(SelectState) + (static_cast<size_t>(sms) * 8 + 2) * sizeof(unsigned int);
}

const char* rigl_init_mask_launch(float* weight, float* mask, int D, int H, unsigned long long n_inactive, void* ws, int sms,
                                  cudaStream_t stream) {
  SelectSrc s{weight, mask, nullptr, nullptr, H, static_cast<size_t>(D) * H};
  SelectState* st = reinterpret_cast<SelectState*>(ws);
  unsigned int* tie = reinterpret_cast<unsigned int*>(reinterpret_cast<char*>(ws) + ((sizeof(SelectState) + 255) / 256 * 256));
  if (n_inactive == 0) return nullptr;
  const char* e = run_select<kSelAbsAll>(s, n_inactive, st, sms, stream);
  if (e) return e;
  return run_tie_apply<kSelAbsAll>(s, st, tie, sms * 8, 0.f, mask, weight, stream);
}

const char* rigl_update_mask_launch(float* weight, float* mask, const float* amean, const float* dmean, int D, int H,
                                    unsigned long long n_drop, unsigned long long n_grow, void* ws, int sms,
                                    cudaStream_t stream) {
  SelectSrc s{weight, mask, amean, dmean, H, static_cast<size_t>(D) * H};
  SelectState* st = reinterpret_cast<SelectState*>(ws);
  unsigned int* tie = reinterpret_cast<unsigned int*>(reinterpret_cast<char*>(ws) + ((sizeof(SelectState) + 255) / 256 * 256));
  if (n_drop > 0) {
    const char* e = run_select<kSelAbsActive>(s, n_drop, st, sms, stream);
    if (e) return e;
    rigl_drop_apply_kernel<<<grid_for(s.n, 256 * 4, sms * 8), 256, 0, stream>>>(weight, mask, s.n, select_vec_ok(s) ? 1 : 0, st);
    count_launches(1);
  }
  if (n_grow > 0 && amean != nullptr && dmean != nullptr) {
    const char* e = run_select<kSelScoreInactive>(s, n_grow, st, sms, stream);
    if (e) return e;
    return run_tie_apply<kSelScoreInactive>(s, st, tie, sms * 8, 1.f, mask, weight, stream);
  }
  // no grow step: still weight *= mask (:87)
  mul_inplace_kernel<<<grid_for(s.n, 256 * 4, sms * 8), 256, 0, stream>>>(weight, mask, s.n);
  count_launches(1);
  return cuda_err(cudaGetLastError());
}

const char* mul_inplace_launch(float* a, const float* b, size_t n, cudaStream_t stream) {
  if (n == 0) return nullptr;
  mul_inplace_kernel<<<grid_for(n, 256 * 4, 148 * 8), 256, 0, stream>>>(a, b, n);
  return cuda_err(cudaGetLastError());
}

// ---------------------------------------------------------------------------------------------
// baseline_sae backward (sae/baseline.py:17-40 under loss.backward(): Linear -> top-k -> scatter -> Linear).
// With g = d loss / d recon and gv[b,j] = <g[b,:], W_dec[:, idx[b,j]]> + g_h[b, idx[b,j]]:
//   grad W_enc[h,:] = sum gv x[b,:],  grad b_enc[h] = sum gv,  grad W_dec[:,h] = sum v g[b,:]
// over the rows b that selected h; grad b_dec = column sums of g; grad x = gv W_enc (decode_rows_f32).
// The B k entries are grouped by latent with a stable radix sort of the row-major entries (b ascends inside a
// latent), so every gradient element has one writer and a summation order fixed by the inputs alone: the whole
// backward is bit-deterministic, with no float atomics and no [H, D] scratch matrices.
// ---------------------------------------------------------------------------------------------
namespace {

constexpr int kBwdChunk = 256;   // entries one warp reduces directly; longer latents are split into chunks of this size
constexpr int kBwdTile = 32;     // consecutive latents per block of the reduction: grad W_dec leaves in [D, 32] segments
constexpr int kSortThreads = 256, kSortItems = 16, kSortTile = kSortThreads * kSortItems, kRadix = 256;
constexpr int kColParts = 256;   // most partial rows of the two-level column sum

__device__ __forceinline__ int clamp_key(int h, int H) { return static_cast<unsigned>(h) < static_cast<unsigned>(H) ? h : H; }

// gv[b,j] = scale <g[b,:], rows[idx[b,j],:]> + g_h term (0 for an index outside [0, H)); cnt[h] += 1 per selection.
// Warp per row, the row of g in registers, butterfly reductions: the same bits in every lane and on every run.
// baseline_sae passes scale 1 (the product is exact, so its bits are those of the plain dot), b_sae the step q.
template <int NCH>
__global__ void __launch_bounds__(256)
bwd_latent_grad_kernel(const float* __restrict__ g, const float* __restrict__ rows, const int32_t* __restrict__ idx,
                       const float* __restrict__ gh_dense, const float* __restrict__ gh_vals, int B, int k, int D, int H,
                       float scale, float* __restrict__ gv, int* __restrict__ cnt) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int nchunk = D >> 2;
  for (int row = warp; row < B; row += nwarps) {
    float4 gr[NCH];
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const int q = lane + 32 * c;
      gr[c] = q < nchunk ? reinterpret_cast<const float4*>(g + static_cast<size_t>(row) * D)[q] : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    for (int j0 = 0; j0 < k; j0 += 32) {
      const int jl = j0 + lane;
      const size_t e = static_cast<size_t>(row) * k + jl;
      const int my_h = jl < k ? idx[e] : -1;
      const bool ok = static_cast<unsigned>(my_h) < static_cast<unsigned>(H);
      float my_gh = 0.f;
      if (ok && gh_vals != nullptr) my_gh = gh_vals[e];
      else if (ok && gh_dense != nullptr) my_gh = gh_dense[static_cast<size_t>(row) * H + my_h];
      float my_dot = 0.f;
      const int nj = min(32, k - j0);
      for (int j = 0; j < nj; ++j) {
        const int h = __shfl_sync(0xffffffffu, my_h, j);
        if (static_cast<unsigned>(h) >= static_cast<unsigned>(H)) continue;
        const float4* r = reinterpret_cast<const float4*>(rows + static_cast<size_t>(h) * D);
        float acc = 0.f;
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          const int q = lane + 32 * c;
          if (q < nchunk) {
            const float4 w = r[q];
            acc += gr[c].x * w.x + gr[c].y * w.y + gr[c].z * w.z + gr[c].w * w.w;
          }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == j) my_dot = acc;
      }
      if (jl < k) {
        gv[e] = ok ? scale * my_dot + my_gh : 0.f;
        if (ok) atomicAdd(cnt + my_h, 1);     // integer counts: exact in any order
      }
    }
  }
}

// Exclusive prefix sums by one block of 1024 threads (each owns a contiguous run): out[0..n], out[n] = total.
// CHUNKED: the values are the chunk counts of the per-latent entry counts in[] (latents longer than kBwdChunk only).
// May run in place (in == out): every thread reads and writes only its own run.
template <bool CHUNKED>
__global__ void __launch_bounds__(1024) bwd_scan_kernel(const int* in, int n, int* out) {
  __shared__ int warp_tot[32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int per = (n + 1023) / 1024;
  const int lo = min(n, threadIdx.x * per), hi = min(n, lo + per);
  auto value = [&](int i) {
    const int c = in[i];
    return CHUNKED ? (c > kBwdChunk ? (c + kBwdChunk - 1) / kBwdChunk : 0) : c;
  };
  int local = 0;
  for (int i = lo; i < hi; ++i) local += value(i);
  int incl = local;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) warp_tot[wid] = incl;
  __syncthreads();
  int base = 0, all = 0;
  for (int w = 0; w < 32; ++w) {
    if (w < wid) base += warp_tot[w];
    all += warp_tot[w];
  }
  int run = base + incl - local;
  for (int i = lo; i < hi; ++i) {
    const int v = value(i);
    out[i] = run;
    run += v;
  }
  if (threadIdx.x == 0) out[n] = all;
}

// radix sort of the entries by latent, 8 bits per pass: digit counts of one tile of kSortTile entries, digit-major
// [kRadix][ntiles] so that one exclusive scan gives every (digit, tile) its first output position
__global__ void __launch_bounds__(kSortThreads)
bwd_sort_hist_kernel(const int32_t* __restrict__ keys, int n, int H, int shift, int ntiles, int* __restrict__ hist) {
  __shared__ int h[kRadix];
  h[threadIdx.x] = 0;
  __syncthreads();
  const int base = blockIdx.x * kSortTile;
  for (int i = threadIdx.x; i < kSortTile; i += kSortThreads)
    if (base + i < n) atomicAdd(&h[(clamp_key(keys[base + i], H) >> shift) & (kRadix - 1)], 1);
  __syncthreads();
  hist[threadIdx.x * ntiles + blockIdx.x] = h[threadIdx.x];
}

// Stable scatter of one tile: rounds of 256 consecutive entries in order; inside a round the rank of an entry among
// its digit's is its warp's earlier lanes (match_any) plus the earlier warps' counts. Intermediate passes move
// (key, entry); the last one writes the records {b, v, gv} the reduction reads.
template <bool LAST>
__global__ void __launch_bounds__(kSortThreads)
bwd_sort_scatter_kernel(const int32_t* __restrict__ keys, const int* __restrict__ src_e, int n, int H, int shift, int ntiles,
                        const int* __restrict__ hist_off, int* __restrict__ keys_out, int* __restrict__ e_out, int k,
                        const float* __restrict__ vals, const float* __restrict__ gv, int* __restrict__ ent_b,
                        float* __restrict__ ent_v, float* __restrict__ ent_g) {
  constexpr int kWarps = kSortThreads / 32;
  __shared__ int run[kRadix];
  __shared__ int wcnt[kWarps][kRadix];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  run[threadIdx.x] = hist_off[threadIdx.x * ntiles + blockIdx.x];
#pragma unroll
  for (int w = 0; w < kWarps; ++w) wcnt[w][threadIdx.x] = 0;
  __syncthreads();
  const int base = blockIdx.x * kSortTile;
  for (int r = 0; r < kSortItems; ++r) {
    const int i = base + r * kSortThreads + threadIdx.x;
    const bool valid = i < n;
    const int key = valid ? clamp_key(keys[i], H) : 0;
    const int d = valid ? (key >> shift) & (kRadix - 1) : -1;
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    const int lt = __popc(peers & ((1u << lane) - 1u));
    if (valid && lt == 0) wcnt[wid][d] = __popc(peers);
    __syncthreads();
    if (valid) {
      int pos = run[d] + lt;
      for (int w = 0; w < wid; ++w) pos += wcnt[w][d];
      const int e = src_e != nullptr ? src_e[i] : i;
      if (LAST) {
        ent_b[pos] = e / k;
        ent_v[pos] = vals[e];
        ent_g[pos] = gv[e];
      } else {
        keys_out[pos] = key;
        e_out[pos] = e;
      }
    }
    __syncthreads();
    int s = 0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) {
      s += wcnt[w][threadIdx.x];
      wcnt[w][threadIdx.x] = 0;
    }
    run[threadIdx.x] += s;
    __syncthreads();
  }
}

// aWe += sum gv x[b,:], aWd += sum v g[b,:], sbe += sum gv over the records [lo, hi), in record order
template <int NCH>
__device__ __forceinline__ void bwd_reduce_entries(int lo, int hi, const int* __restrict__ ent_b, const float* __restrict__ ent_v,
                                                   const float* __restrict__ ent_g, const float4* __restrict__ x4,
                                                   const float4* __restrict__ g4, int nchunk, int lane, float4 (&aWe)[NCH],
                                                   float4 (&aWd)[NCH], float& sbe) {
  for (int e0 = lo; e0 < hi; e0 += 32) {
    const int my = e0 + lane;
    const int my_b = my < hi ? ent_b[my] : 0;
    const float my_v = my < hi ? ent_v[my] : 0.f;
    const float my_g = my < hi ? ent_g[my] : 0.f;
    const int n = min(32, hi - e0);
#pragma unroll 4
    for (int j = 0; j < n; ++j) {
      const int b = __shfl_sync(0xffffffffu, my_b, j);
      const float v = __shfl_sync(0xffffffffu, my_v, j);
      const float gg = __shfl_sync(0xffffffffu, my_g, j);
      sbe += gg;
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        const int q = lane + 32 * c;
        if (q < nchunk) {
          const float4 xr = x4[static_cast<size_t>(b) * nchunk + q];
          const float4 gr = g4[static_cast<size_t>(b) * nchunk + q];
          aWe[c].x = fmaf(gg, xr.x, aWe[c].x); aWe[c].y = fmaf(gg, xr.y, aWe[c].y);
          aWe[c].z = fmaf(gg, xr.z, aWe[c].z); aWe[c].w = fmaf(gg, xr.w, aWe[c].w);
          aWd[c].x = fmaf(v, gr.x, aWd[c].x); aWd[c].y = fmaf(v, gr.y, aWd[c].y);
          aWd[c].z = fmaf(v, gr.z, aWd[c].z); aWd[c].w = fmaf(v, gr.w, aWd[c].w);
        }
      }
    }
  }
}

__device__ __forceinline__ void add4(float4& a, const float4 b) { a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }

// Partials of the latents with more than kBwdChunk entries: warp per chunk q (chunks of latent h are
// [coff[h], coff[h+1]), entries [off[h] + c kBwdChunk, ...)). part[q] = {We partial [D], Wd partial [D], be, pad}.
template <int NCH>
__global__ void __launch_bounds__(256)
bwd_chunk_kernel(const int* __restrict__ off, const int* __restrict__ coff, int H, const int* __restrict__ ent_b,
                 const float* __restrict__ ent_v, const float* __restrict__ ent_g, const float* __restrict__ x,
                 const float* __restrict__ g, int D, float* __restrict__ part) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int nchunk = D >> 2;
  const size_t pitch = 2 * static_cast<size_t>(D) + 4;
  const int total = coff[H];
  for (int q = warp; q < total; q += nwarps) {
    int lo_h = 0, hi_h = H;                    // the last h with coff[h] <= q
    while (hi_h - lo_h > 1) {
      const int mid = (lo_h + hi_h) >> 1;
      if (coff[mid] <= q) lo_h = mid;
      else hi_h = mid;
    }
    const int h = lo_h;
    const int lo = off[h] + (q - coff[h]) * kBwdChunk;
    const int hi = min(off[h + 1], lo + kBwdChunk);
    float4 aWe[NCH], aWd[NCH];
#pragma unroll
    for (int c = 0; c < NCH; ++c) aWe[c] = aWd[c] = make_float4(0.f, 0.f, 0.f, 0.f);
    float sbe = 0.f;
    bwd_reduce_entries<NCH>(lo, hi, ent_b, ent_v, ent_g, reinterpret_cast<const float4*>(x), reinterpret_cast<const float4*>(g),
                            nchunk, lane, aWe, aWd, sbe);
    float* p = part + static_cast<size_t>(q) * pitch;
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const int q4 = lane + 32 * c;
      if (q4 < nchunk) {
        reinterpret_cast<float4*>(p)[q4] = aWe[c];
        reinterpret_cast<float4*>(p + D)[q4] = aWd[c];
      }
    }
    if (lane == 0) p[2 * D] = sbe;
  }
}

// One warp's sums for latent h: aWe = sum gv x, aWd = sum v g, sbe = sum gv over the rows that selected h. A latent
// with at most kBwdChunk entries is reduced from its records, a longer one sums its chunk partials in chunk order;
// a latent nobody selected gets exact zeros.
template <int NCH>
__device__ __forceinline__ void bwd_latent_sums(int h, const int* __restrict__ off, const int* __restrict__ coff,
                                                const int* __restrict__ ent_b, const float* __restrict__ ent_v,
                                                const float* __restrict__ ent_g, const float* __restrict__ x,
                                                const float* __restrict__ g, int D, const float* __restrict__ part, int lane,
                                                float4 (&aWe)[NCH], float4 (&aWd)[NCH], float& sbe) {
  const int nchunk = D >> 2;
  const size_t pitch = 2 * static_cast<size_t>(D) + 4;
#pragma unroll
  for (int c = 0; c < NCH; ++c) aWe[c] = aWd[c] = make_float4(0.f, 0.f, 0.f, 0.f);
  sbe = 0.f;
  const int lo = off[h], hi = off[h + 1];
  if (hi - lo <= kBwdChunk) {
    bwd_reduce_entries<NCH>(lo, hi, ent_b, ent_v, ent_g, reinterpret_cast<const float4*>(x),
                            reinterpret_cast<const float4*>(g), nchunk, lane, aWe, aWd, sbe);
  } else {
    for (int q = coff[h]; q < coff[h + 1]; ++q) {
      const float* p = part + static_cast<size_t>(q) * pitch;
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        const int q4 = lane + 32 * c;
        if (q4 < nchunk) {
          add4(aWe[c], reinterpret_cast<const float4*>(p)[q4]);
          add4(aWd[c], reinterpret_cast<const float4*>(p + D)[q4]);
        }
      }
      sbe += p[2 * D];
    }
  }
}

// Latent-major reduction: block of 8 warps over kBwdTile consecutive latents, warp per latent. grad W_enc rows
// and grad b_enc leave directly; the grad W_dec columns are staged in shared memory [kBwdTile][D + 1] and leave as
// [D, kBwdTile] row segments.
template <int NCH>
__global__ void __launch_bounds__(256)
bwd_latent_reduce_kernel(const int* __restrict__ off, const int* __restrict__ coff, int H, const int* __restrict__ ent_b,
                         const float* __restrict__ ent_v, const float* __restrict__ ent_g, const float* __restrict__ x,
                         const float* __restrict__ g, int D, const float* __restrict__ part, float* __restrict__ gWe,
                         float* __restrict__ gbe, float* __restrict__ gWd) {
  extern __shared__ float stage[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int nchunk = D >> 2;
  const int h0 = blockIdx.x * kBwdTile;
  const int nl = min(kBwdTile, H - h0);
  for (int l = wid; l < nl; l += blockDim.x >> 5) {
    const int h = h0 + l;
    float4 aWe[NCH], aWd[NCH];
    float sbe;
    bwd_latent_sums<NCH>(h, off, coff, ent_b, ent_v, ent_g, x, g, D, part, lane, aWe, aWd, sbe);
    float* srow = stage + static_cast<size_t>(l) * (D + 1);
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const int q4 = lane + 32 * c;
      if (q4 < nchunk) {
        reinterpret_cast<float4*>(gWe + static_cast<size_t>(h) * D)[q4] = aWe[c];
        srow[4 * q4] = aWd[c].x; srow[4 * q4 + 1] = aWd[c].y; srow[4 * q4 + 2] = aWd[c].z; srow[4 * q4 + 3] = aWd[c].w;
      }
    }
    if (lane == 0) gbe[h] = sbe;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < D * kBwdTile; i += blockDim.x) {
    const int d = i / kBwdTile, l = i - d * kBwdTile;
    if (l < nl) gWd[static_cast<size_t>(d) * H + h0 + l] = stage[static_cast<size_t>(l) * (D + 1) + d];
  }
}

// b_sae latent-major pass: warp per latent h, 8 latents per block. From the sums of bwd_latent_sums:
//   grad W_enc[h,:] = sum gv x, grad b_enc[h] = sum gv,  G[h,:] = q sum v g  (d loss / d int_w, never in memory)
//   grad_logits[h, d n + i] = (G[h,d] c_i + gp 2^i (1 - 2p) / N) p (1 - p)   (the bsae_logit_grad formula)
// G's row is staged in the warp's slice of shared memory so that the logit row streams in coalesced 16-byte groups,
// exactly as bsae_logit_grad reads it. Each logit is read once and each output element has one writer; a latent
// nobody selected has G = 0 and gets the polarize-only gradient and exact zeros in grad W_enc / grad b_enc.
constexpr int kBsaeWarps = 8;
constexpr int kBsaeUnroll = 4;   // 16-byte logit loads in flight per lane

template <int NCH>
__global__ void __launch_bounds__(32 * kBsaeWarps)
bsae_latent_reduce_kernel(const int* __restrict__ off, const int* __restrict__ coff, int H, const int* __restrict__ ent_b,
                          const float* __restrict__ ent_v, const float* __restrict__ ent_g, const float* __restrict__ x,
                          const float* __restrict__ g, int D, const float* __restrict__ part, float q,
                          const float* __restrict__ logits, int n_bits, const float* __restrict__ gp_dev, float gp_host,
                          float* __restrict__ gWe, float* __restrict__ gbe, float* __restrict__ glog) {
  __shared__ float4 sG[kBsaeWarps][NCH * 32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int h = blockIdx.x * kBsaeWarps + wid;
  if (h >= H) return;                             // warp-uniform; the block never synchronises
  const int nchunk = D >> 2;
  float4 aWe[NCH], aWd[NCH];
  float sbe;
  bwd_latent_sums<NCH>(h, off, coff, ent_b, ent_v, ent_g, x, g, D, part, lane, aWe, aWd, sbe);
#pragma unroll
  for (int c = 0; c < NCH; ++c) {
    const int q4 = lane + 32 * c;
    if (q4 < nchunk) {
      reinterpret_cast<float4*>(gWe + static_cast<size_t>(h) * D)[q4] = aWe[c];
      sG[wid][q4] = make_float4(q * aWd[c].x, q * aWd[c].y, q * aWd[c].z, q * aWd[c].w);
    }
  }
  if (lane == 0) gbe[h] = sbe;
  __syncwarp();
  const float* Gs = reinterpret_cast<const float*>(sG[wid]);
  const int cols = D * n_bits, groups = cols >> 2;     // D % 8 == 0: a row is whole 16-byte groups
  const float gp = bsae_polarize_scale(gp_dev, gp_host, H, cols);
  const float4* lrow = reinterpret_cast<const float4*>(logits + static_cast<size_t>(h) * cols);
  float4* grow = reinterpret_cast<float4*>(glog + static_cast<size_t>(h) * cols);
  for (int c0 = lane; c0 < groups; c0 += 32 * kBsaeUnroll) {
    float4 w[kBsaeUnroll];
#pragma unroll
    for (int u = 0; u < kBsaeUnroll; ++u) {
      const int cg = c0 + 32 * u;
      if (cg < groups) w[u] = lrow[cg];
    }
#pragma unroll
    for (int u = 0; u < kBsaeUnroll; ++u) {
      const int cg = c0 + 32 * u;
      if (cg >= groups) continue;
      const int col = 4 * cg;
      int d = col / n_bits, i = col - d * n_bits;
      const float wv[4] = {w[u].x, w[u].y, w[u].z, w[u].w};
      float o[4];
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        float ci, gpw;
        bsae_bit_consts(i, n_bits, gp, ci, gpw);
        o[t] = bsae_logit_grad_value(wv[t], Gs[d], ci, gpw);
        if (++i == n_bits) { i = 0; ++d; }
      }
      grow[cg] = make_float4(o[0], o[1], o[2], o[3]);
    }
  }
}

// grad b_dec = column sums of g [B, D] in a fixed order: partial sums over fixed row slices, then the partials in order
__global__ void __launch_bounds__(128)
bwd_colsum_part_kernel(const float* __restrict__ g, int B, int D, int rows_per, float* __restrict__ part) {
  const int t = threadIdx.x, nchunk = D >> 2;
  if (t >= nchunk) return;
  const int r0 = blockIdx.x * rows_per, r1 = min(B, r0 + rows_per);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int r = r0; r < r1; ++r) add4(acc, reinterpret_cast<const float4*>(g)[static_cast<size_t>(r) * nchunk + t]);
  reinterpret_cast<float4*>(part)[static_cast<size_t>(blockIdx.x) * nchunk + t] = acc;
}

__global__ void __launch_bounds__(128) bwd_colsum_final_kernel(const float* __restrict__ part, int nparts, int D, float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= D) return;
  float s = 0.f;
#pragma unroll 8
  for (int p = 0; p < nparts; ++p) s += part[static_cast<size_t>(p) * D + c];
  out[c] = s;
}

// workspace of both latent-major backwards (baseline_sae and b_sae need the same regions)
struct BaselineBwdLayout {
  int n, ntiles, npasses, max_chunks, col_rows, col_parts;
  size_t gv, cnt, off, coff, hist, keys[2], ent[2], eb, ev, eg, part, colpart, total;
};

BaselineBwdLayout baseline_bwd_layout(int B, int H, int D, int k) {
  BaselineBwdLayout L{};
  L.n = B * k;
  L.ntiles = (L.n + kSortTile - 1) / kSortTile;
  const int key_bits = 32 - __builtin_clz(static_cast<unsigned>(H));    // keys run over [0, H]: H marks a bad index
  L.npasses = (key_bits + 7) / 8;
  // a latent with c > kBwdChunk entries has ceil(c / kBwdChunk) < 2 c / kBwdChunk chunks
  L.max_chunks = static_cast<int>(2 * (static_cast<long long>(L.n) / kBwdChunk) + 1);
  L.col_rows = B > 0 ? (B + kColParts - 1) / kColParts : 1;
  if (L.col_rows < 32) L.col_rows = 32;
  L.col_parts = B > 0 ? (B + L.col_rows - 1) / L.col_rows : 0;
  const size_t n = static_cast<size_t>(L.n);
  size_t o = 0;
  auto take = [&](size_t bytes) {
    const size_t s = o;
    o = (o + bytes + 255) / 256 * 256;
    return s;
  };
  L.gv = take(n * 4);
  L.cnt = take((static_cast<size_t>(H) + 1) * 4);
  L.off = take((static_cast<size_t>(H) + 1) * 4);
  L.coff = take((static_cast<size_t>(H) + 1) * 4);
  L.hist = take((static_cast<size_t>(kRadix) * L.ntiles + 1) * 4);
  for (int i = 0; i < 2; ++i) {
    L.keys[i] = take(n * 4);
    L.ent[i] = take(n * 4);
  }
  L.eb = take(n * 4);
  L.ev = take(n * 4);
  L.eg = take(n * 4);
  L.part = take(static_cast<size_t>(L.max_chunks) * (2 * static_cast<size_t>(D) + 4) * 4);
  L.colpart = take(static_cast<size_t>(L.col_parts) * D * 4);
  L.total = o;
  return L;
}

// one warp per possible chunk (the device-side total decides which run): no host synchronisation
template <int NCH>
void bwd_chunk_launch(const BaselineBwdLayout& L, uint8_t* ws, int H, int D, const float* x, const float* g, cudaStream_t stream) {
  bwd_chunk_kernel<NCH><<<grid_for(static_cast<size_t>(L.max_chunks) * 32, 256, 148 * 8), 256, 0, stream>>>(
      reinterpret_cast<const int*>(ws + L.off), reinterpret_cast<const int*>(ws + L.coff), H,
      reinterpret_cast<const int*>(ws + L.eb), reinterpret_cast<const float*>(ws + L.ev),
      reinterpret_cast<const float*>(ws + L.eg), x, g, D, reinterpret_cast<float*>(ws + L.part));
}

template <int NCH>
void bwd_reduce_launches(const BaselineBwdLayout& L, uint8_t* ws, int H, int D, const float* x, const float* g, float* gWe,
                         float* gbe, float* gWd, cudaStream_t stream) {
  bwd_chunk_launch<NCH>(L, ws, H, D, x, g, stream);
  const size_t smem = static_cast<size_t>(kBwdTile) * (D + 1) * sizeof(float);
  cudaFuncSetAttribute(bwd_latent_reduce_kernel<NCH>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
  bwd_latent_reduce_kernel<NCH><<<(H + kBwdTile - 1) / kBwdTile, 256, smem, stream>>>(
      reinterpret_cast<const int*>(ws + L.off), reinterpret_cast<const int*>(ws + L.coff), H,
      reinterpret_cast<const int*>(ws + L.eb), reinterpret_cast<const float*>(ws + L.ev),
      reinterpret_cast<const float*>(ws + L.eg), x, g, D, reinterpret_cast<const float*>(ws + L.part), gWe, gbe, gWd);
}

template <int NCH>
void bsae_reduce_launches(const BaselineBwdLayout& L, uint8_t* ws, int H, int D, const float* x, const float* g, float q,
                          const float* logits, int n_bits, const float* gp_dev, float gp_host, float* gWe, float* gbe,
                          float* glog, cudaStream_t stream) {
  bwd_chunk_launch<NCH>(L, ws, H, D, x, g, stream);
  bsae_latent_reduce_kernel<NCH><<<(H + kBsaeWarps - 1) / kBsaeWarps, 32 * kBsaeWarps, 0, stream>>>(
      reinterpret_cast<const int*>(ws + L.off), reinterpret_cast<const int*>(ws + L.coff), H,
      reinterpret_cast<const int*>(ws + L.eb), reinterpret_cast<const float*>(ws + L.ev),
      reinterpret_cast<const float*>(ws + L.eg), x, g, D, reinterpret_cast<const float*>(ws + L.part), q, logits, n_bits,
      gp_dev, gp_host, gWe, gbe, glog);
}

// The first steps of both latent-major backwards:
//   1. gv = scale <g, rows[h]> + g_h term at each kept entry, and the per-latent counts;
//   2. CSC offsets of the entries and of the chunks of long latents;
//   3. stable radix sort of the row-major entries by latent -> records {b, v, gv}, latent-major.
const char* bwd_group_by_latent(const BaselineBwdLayout& L, uint8_t* ws, const float* g, const float* rows, const int32_t* idx,
                                const float* vals, const float* g_h, const float* g_vals, int B, int H, int D, int k,
                                float scale, int* launches, cudaStream_t stream) {
  float* gv = reinterpret_cast<float*>(ws + L.gv);
  int* cnt = reinterpret_cast<int*>(ws + L.cnt);
  int* hist = reinterpret_cast<int*>(ws + L.hist);
  const cudaError_t e = cudaMemsetAsync(cnt, 0, static_cast<size_t>(H) * 4, stream);
  if (e != cudaSuccess) return cudaGetErrorString(e);
  const int grid_rows = grid_for(static_cast<size_t>(B) * 32, 256, 148 * 8);
  switch ((D / 4 + 31) / 32) {
    case 1: bwd_latent_grad_kernel<1><<<grid_rows, 256, 0, stream>>>(g, rows, idx, g_h, g_vals, B, k, D, H, scale, gv, cnt); break;
    case 2: bwd_latent_grad_kernel<2><<<grid_rows, 256, 0, stream>>>(g, rows, idx, g_h, g_vals, B, k, D, H, scale, gv, cnt); break;
    case 3: bwd_latent_grad_kernel<3><<<grid_rows, 256, 0, stream>>>(g, rows, idx, g_h, g_vals, B, k, D, H, scale, gv, cnt); break;
    default: bwd_latent_grad_kernel<4><<<grid_rows, 256, 0, stream>>>(g, rows, idx, g_h, g_vals, B, k, D, H, scale, gv, cnt); break;
  }
  bwd_scan_kernel<false><<<1, 1024, 0, stream>>>(cnt, H, reinterpret_cast<int*>(ws + L.off));
  bwd_scan_kernel<true><<<1, 1024, 0, stream>>>(cnt, H, reinterpret_cast<int*>(ws + L.coff));
  *launches += 3;
  const int32_t* keys_in = idx;
  const int* e_in = nullptr;
  for (int p = 0; p < L.npasses; ++p) {
    const int shift = 8 * p;
    const bool last = p == L.npasses - 1;
    bwd_sort_hist_kernel<<<L.ntiles, kSortThreads, 0, stream>>>(keys_in, L.n, H, shift, L.ntiles, hist);
    bwd_scan_kernel<false><<<1, 1024, 0, stream>>>(hist, kRadix * L.ntiles, hist);
    int* keys_out = reinterpret_cast<int*>(ws + L.keys[p & 1]);
    int* e_out = reinterpret_cast<int*>(ws + L.ent[p & 1]);
    if (last)
      bwd_sort_scatter_kernel<true><<<L.ntiles, kSortThreads, 0, stream>>>(
          keys_in, e_in, L.n, H, shift, L.ntiles, hist, nullptr, nullptr, k, vals, gv, reinterpret_cast<int*>(ws + L.eb),
          reinterpret_cast<float*>(ws + L.ev), reinterpret_cast<float*>(ws + L.eg));
    else
      bwd_sort_scatter_kernel<false><<<L.ntiles, kSortThreads, 0, stream>>>(
          keys_in, e_in, L.n, H, shift, L.ntiles, hist, keys_out, e_out, k, nullptr, nullptr, nullptr, nullptr, nullptr);
    keys_in = keys_out;
    e_in = e_out;
    *launches += 3;
  }
  return nullptr;
}

// grad b_dec = column sums of g, then grad x = gv W_enc over the kept entries (the sparse decoder over the encoder rows)
const char* bwd_tail_launches(const BaselineBwdLayout& L, uint8_t* ws, const float* g, const int32_t* idx, const float* w_enc,
                              int B, int H, int D, int k, float* gbd, float* gx, int* launches, cudaStream_t stream) {
  float* colpart = reinterpret_cast<float*>(ws + L.colpart);
  bwd_colsum_part_kernel<<<L.col_parts, 128, 0, stream>>>(g, B, D, L.col_rows, colpart);
  bwd_colsum_final_kernel<<<(D + 127) / 128, 128, 0, stream>>>(colpart, L.col_parts, D, gbd);
  *launches += 2;
  if (gx != nullptr) {
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cudaGetErrorString(e);
    const char* err = decode_f32_launch(reinterpret_cast<const float*>(ws + L.gv), idx, B, k, w_enc, H, D, 1.0f, nullptr, gx, 0, stream);
    if (err != nullptr) return err;
    ++*launches;
  }
  return nullptr;
}

}  // namespace

size_t baseline_backward_workspace_bytes(int B, int H, int D, int k) { return baseline_bwd_layout(B, H, D, k).total; }

const char* baseline_backward_launch(const float* x, const float* vals, const int32_t* idx, const float* g,
                                     const float* g_h, const float* g_vals, const float* w_enc, const float* dec_rows, int B,
                                     int H, int D, int k, float* gWe, float* gbe, float* gWd, float* gbd, float* gx, void* workspace,
                                     cudaStream_t stream) {
  const BaselineBwdLayout L = baseline_bwd_layout(B, H, D, k);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  int launches = 0;
  const char* err = bwd_group_by_latent(L, ws, g, dec_rows, idx, vals, g_h, g_vals, B, H, D, k, 1.0f, &launches, stream);
  if (err != nullptr) return err;
  // 4. latent-major reduction: grad W_enc, grad b_enc, grad W_dec
  switch ((D / 4 + 31) / 32) {
    case 1: bwd_reduce_launches<1>(L, ws, H, D, x, g, gWe, gbe, gWd, stream); break;
    case 2: bwd_reduce_launches<2>(L, ws, H, D, x, g, gWe, gbe, gWd, stream); break;
    case 3: bwd_reduce_launches<3>(L, ws, H, D, x, g, gWe, gbe, gWd, stream); break;
    default: bwd_reduce_launches<4>(L, ws, H, D, x, g, gWe, gbe, gWd, stream); break;
  }
  launches += 2;
  // 5, 6. grad b_dec, grad x
  err = bwd_tail_launches(L, ws, g, idx, w_enc, B, H, D, k, gbd, gx, &launches, stream);
  if (err != nullptr) return err;
  count_launches(launches);
  return cuda_err(cudaGetLastError());
}

// b_sae (sae/binary.py:24-47, 91-103): the baseline's steps with gv = q <g, soft_rows[h]>, the soft rows in place of
// W_dec^T, and the b_sae pass in place of the grad W_dec reduction; the same workspace layout.
const char* bsae_backward_launch(const float* x, const float* vals, const int32_t* idx, const float* g, const float* soft_rows,
                                 const float* logits, float q, const float* gp_dev, float gp_host, const float* w_enc, int B,
                                 int H, int D, int k, int n_bits, float* gWe, float* gbe, float* glog, float* gbd, float* gx,
                                 void* workspace, cudaStream_t stream) {
  const BaselineBwdLayout L = baseline_bwd_layout(B, H, D, k);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  int launches = 0;
  const char* err = bwd_group_by_latent(L, ws, g, soft_rows, idx, vals, nullptr, nullptr, B, H, D, k, q, &launches, stream);
  if (err != nullptr) return err;
  switch ((D / 4 + 31) / 32) {
    case 1: bsae_reduce_launches<1>(L, ws, H, D, x, g, q, logits, n_bits, gp_dev, gp_host, gWe, gbe, glog, stream); break;
    case 2: bsae_reduce_launches<2>(L, ws, H, D, x, g, q, logits, n_bits, gp_dev, gp_host, gWe, gbe, glog, stream); break;
    case 3: bsae_reduce_launches<3>(L, ws, H, D, x, g, q, logits, n_bits, gp_dev, gp_host, gWe, gbe, glog, stream); break;
    default: bsae_reduce_launches<4>(L, ws, H, D, x, g, q, logits, n_bits, gp_dev, gp_host, gWe, gbe, glog, stream); break;
  }
  launches += 2;
  err = bwd_tail_launches(L, ws, g, idx, w_enc, B, H, D, k, gbd, gx, &launches, stream);
  if (err != nullptr) return err;
  count_launches(launches);
  return cuda_err(cudaGetLastError());
}

}  // namespace qsae
