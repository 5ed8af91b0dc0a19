// One-time weight preparation kernels (all HBM-bound streaming passes):
//   fp32 -> bf16 cast, bit-plane logits -> packed two's-complement dictionary (+ polarize stats),
//   soft (sigmoid) dequantisation, fp32 transpose.
// Compiled WITHOUT fast-math: the logistic must be the literal 1 / (1 + expf(-w)) that
// torch evaluates (sae/binary.py:26,52) so the strict 0.5 threshold lands identically.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "kernels.h"

namespace qsae {

namespace {

__device__ __forceinline__ float logistic(float w) { return 1.0f / (1.0f + expf(-w)); }

__global__ void cast_bf16_kernel(const float* __restrict__ src, uint16_t* __restrict__ dst, size_t n) {
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  const size_t n4 = n / 4;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 v = reinterpret_cast<const float4*>(src)[i];
    __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y);
    __nv_bfloat162 hi = __floats2bfloat162_rn(v.z, v.w);
    uint2 o;
    o.x = *reinterpret_cast<uint32_t*>(&lo);
    o.y = *reinterpret_cast<uint32_t*>(&hi);
    reinterpret_cast<uint2*>(dst)[i] = o;
  }
  for (size_t i = n4 * 4 + static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
    __nv_bfloat16 b = __float2bfloat16_rn(src[i]);
    dst[i] = *reinterpret_cast<uint16_t*>(&b);
  }
}

__global__ void upcast_bf16_kernel(const uint16_t* __restrict__ src, float* __restrict__ dst, size_t n) {
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  const size_t n4 = n / 4;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const uint2 v = reinterpret_cast<const uint2*>(src)[i];
    reinterpret_cast<float4*>(dst)[i] = make_float4(__uint_as_float(v.x << 16), __uint_as_float(v.x & 0xFFFF0000u),
                                                    __uint_as_float(v.y << 16), __uint_as_float(v.y & 0xFFFF0000u));
  }
  for (size_t i = n4 * 4 + static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride)
    dst[i] = __uint_as_float(static_cast<uint32_t>(src[i]) << 16);
}

// One thread per output feature (h, d): reads its n_bits logits, emits the integer.
// Threads of a warp read consecutive features, i.e. a contiguous 32*n_bits*4-byte span.
template <bool kNibble>
__global__ void pack_bitplanes_kernel(const float* __restrict__ logits, int H, int D, int n_bits,
                                      uint8_t* __restrict__ packed, double* stats) {
  const size_t total = static_cast<size_t>(H) * D;
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  double pol = 0.0;
  float gap = 0.f;
  // the trip count is warp-uniform (decided on the warp's first feature) because of the shuffle
  for (size_t f0 = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
       f0 - (threadIdx.x & 31) < total; f0 += stride) {
    const bool in = f0 < total;
    int value = 0;
    if (in) {
      const float* lp = logits + f0 * n_bits;
      float polf = 0.f;
      for (int i = 0; i < n_bits; ++i) {
        const float p = logistic(lp[i]);
        const int bit = p > 0.5f ? 1 : 0;
        const int w = 1 << i;
        value += (i == n_bits - 1) ? -bit * w : bit * w;
        polf += p * (1.0f - p) * static_cast<float>(w);
        gap = fmaxf(gap, fabsf(p - static_cast<float>(bit)));
      }
      pol += static_cast<double>(polf);
    }
    if (kNibble) {
      // features 2j (low nibble) and 2j+1 (high nibble) sit in adjacent lanes; D is even
      const int nib = value & 0xF;
      const int other = __shfl_down_sync(0xffffffffu, nib, 1);
      if (in && (f0 & 1) == 0) packed[f0 >> 1] = static_cast<uint8_t>(nib | (other << 4));
    } else {
      if (in) packed[f0] = static_cast<uint8_t>(static_cast<int8_t>(value));
    }
  }
  if (stats != nullptr) {
    // block reduce, one atomic pair per block
    __shared__ double s_pol[32];
    __shared__ float s_gap[32];
    for (int o = 16; o > 0; o >>= 1) {
      pol += __shfl_xor_sync(0xffffffffu, pol, o);
      gap = fmaxf(gap, __shfl_xor_sync(0xffffffffu, gap, o));
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { s_pol[warp] = pol; s_gap[warp] = gap; }
    __syncthreads();
    if (warp == 0) {
      const int nw = blockDim.x >> 5;
      pol = lane < nw ? s_pol[lane] : 0.0;
      gap = lane < nw ? s_gap[lane] : 0.f;
      for (int o = 16; o > 0; o >>= 1) {
        pol += __shfl_xor_sync(0xffffffffu, pol, o);
        gap = fmaxf(gap, __shfl_xor_sync(0xffffffffu, gap, o));
      }
      if (lane == 0) {
        atomicAdd(&stats[0], pol);
        // non-negative doubles order like their bit patterns
        atomicMax(reinterpret_cast<unsigned long long*>(&stats[1]),
                  static_cast<unsigned long long>(__double_as_longlong(static_cast<double>(gap))));
      }
    }
  }
}

__global__ void dequant_soft_kernel(const float* __restrict__ logits, size_t total, int n_bits,
                                    float* __restrict__ rows) {
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  for (size_t f = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; f < total; f += stride) {
    const float* lp = logits + f * n_bits;
    float acc = 0.f;
    for (int i = 0; i < n_bits; ++i) {
      const float c = static_cast<float>(1 << i);
      // separate multiply and add (no FMA contraction): matches (p * c).sum(-1) in fp32
      acc = __fadd_rn(acc, __fmul_rn(logistic(lp[i]), (i == n_bits - 1) ? -c : c));
    }
    rows[f] = acc;
  }
}

// hi = bf16(v), lo = bf16(v - hi): hi + lo carries 16 mantissa bits of v
__global__ void split_bf16_kernel(const float* __restrict__ src, uint16_t* __restrict__ hi, uint16_t* __restrict__ lo,
                                  size_t n) {
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  const size_t n4 = n / 4;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 v = reinterpret_cast<const float4*>(src)[i];
    const __nv_bfloat162 h0 = __floats2bfloat162_rn(v.x, v.y), h1 = __floats2bfloat162_rn(v.z, v.w);
    uint2 o;
    o.x = *reinterpret_cast<const uint32_t*>(&h0);
    o.y = *reinterpret_cast<const uint32_t*>(&h1);
    reinterpret_cast<uint2*>(hi)[i] = o;
    if (lo != nullptr) {
      const float2 f0 = __bfloat1622float2(h0), f1 = __bfloat1622float2(h1);
      const __nv_bfloat162 l0 = __floats2bfloat162_rn(v.x - f0.x, v.y - f0.y);
      const __nv_bfloat162 l1 = __floats2bfloat162_rn(v.z - f1.x, v.w - f1.y);
      o.x = *reinterpret_cast<const uint32_t*>(&l0);
      o.y = *reinterpret_cast<const uint32_t*>(&l1);
      reinterpret_cast<uint2*>(lo)[i] = o;
    }
  }
  for (size_t i = n4 * 4 + static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
    const __nv_bfloat16 h = __float2bfloat16_rn(src[i]);
    hi[i] = *reinterpret_cast<const uint16_t*>(&h);
    if (lo != nullptr) {
      const __nv_bfloat16 l = __float2bfloat16_rn(src[i] - __bfloat162float(h));
      lo[i] = *reinterpret_cast<const uint16_t*>(&l);
    }
  }
}

// hi = bf16(v), mid = bf16(v - hi), lo = bf16(v - hi - mid): the three parts sum to v exactly
// (8 + 8 + 8 mantissa bits; both subtractions are exact in fp32)
__global__ void split_bf16x3_kernel(const float* __restrict__ src, uint16_t* __restrict__ hi, uint16_t* __restrict__ mid,
                                    uint16_t* __restrict__ lo, size_t n) {
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
    const float v = src[i];
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    const float r1 = v - __bfloat162float(h);
    const __nv_bfloat16 m = __float2bfloat16_rn(r1);
    const float r2 = r1 - __bfloat162float(m);
    const __nv_bfloat16 l = __float2bfloat16_rn(r2);
    hi[i] = *reinterpret_cast<const uint16_t*>(&h);
    if (mid != nullptr) mid[i] = *reinterpret_cast<const uint16_t*>(&m);
    if (lo != nullptr) lo[i] = *reinterpret_cast<const uint16_t*>(&l);
  }
}

// STEWeights hard weights (sae/ternary.py:46-49): sign(w) * (|w| >= threshold) in {-1, 0, +1}.
// 32 x 32 tiles of w [D, H]: bf16 in place ([D, H], K-major B operand of the decoder GEMM) and
// transposed int8 rows ([H, D], gather layout of the sparse decoder) and / or transposed bf16 ([H, D], K-major B
// operand of the t_sae backward's g T).
__global__ void pack_ternary_kernel(const float* __restrict__ w, int D, int H, float threshold,
                                    uint16_t* __restrict__ t_bf16, int8_t* __restrict__ t_rows, uint16_t* __restrict__ t_t_bf16) {
  __shared__ int8_t tile[32][33];
  const int h0 = blockIdx.x * 32, d0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int d = d0 + i, h = h0 + threadIdx.x;
    int8_t t = 0;
    if (d < D && h < H) {
      const float v = w[static_cast<size_t>(d) * H + h];
      t = (fabsf(v) >= threshold) ? (v > 0.f ? 1 : (v < 0.f ? -1 : 0)) : 0;
      if (t_bf16 != nullptr)
        t_bf16[static_cast<size_t>(d) * H + h] = t == 0 ? 0x0000u : (t > 0 ? 0x3F80u : 0xBF80u);
    }
    tile[i][threadIdx.x] = t;
  }
  if (t_rows == nullptr && t_t_bf16 == nullptr) return;
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int h = h0 + i, d = d0 + threadIdx.x;
    if (h < H && d < D) {
      const int8_t t = tile[threadIdx.x][i];
      if (t_rows != nullptr) t_rows[static_cast<size_t>(h) * D + d] = t;
      if (t_t_bf16 != nullptr) t_t_bf16[static_cast<size_t>(h) * D + d] = t == 0 ? 0x0000u : (t > 0 ? 0x3F80u : 0xBF80u);
    }
  }
}

// rq_sae residual step (sae/residual_quantized.py:67): out = (r - recon) * 2
__global__ void residual_update_kernel(const float* __restrict__ r, const float* __restrict__ recon, size_t n,
                                       float* __restrict__ out) {
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  const size_t n4 = n / 4;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 a = reinterpret_cast<const float4*>(r)[i], b = reinterpret_cast<const float4*>(recon)[i];
    reinterpret_cast<float4*>(out)[i] = make_float4((a.x - b.x) * 2.f, (a.y - b.y) * 2.f, (a.z - b.z) * 2.f, (a.w - b.w) * 2.f);
  }
  for (size_t i = n4 * 4 + static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride)
    out[i] = (r[i] - recon[i]) * 2.f;
}

__global__ void transpose_kernel(const float* __restrict__ src, int R, int C, float* __restrict__ dst) {
  __shared__ float tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < R && c < C) ? src[static_cast<size_t>(r) * C + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (r < R && c < C) dst[static_cast<size_t>(c) * R + r] = tile[threadIdx.x][i];
  }
}

// Stratified pseudo-random sample of dictionary rows: sample i is drawn from the i-th of n_sample
// equal slices of [0, H) at a hashed offset, so the sample is spread over the whole dictionary
// without following any period the latent ordering may have.
__host__ __device__ inline int sample_row_index(int i, int H, int n_sample) {
  const long long lo = static_cast<long long>(i) * H / n_sample;
  const long long hi = static_cast<long long>(i + 1) * H / n_sample;
  uint32_t h = static_cast<uint32_t>(i) * 2654435761u;
  h ^= h >> 15; h *= 2246822519u; h ^= h >> 13;
  const long long span = hi - lo > 0 ? hi - lo : 1;
  return static_cast<int>(lo + static_cast<long long>(h % static_cast<uint32_t>(span)));
}

__global__ void sample_rows_kernel(const uint16_t* __restrict__ w, const float* __restrict__ bias, int H,
                                   int D, int n_sample, uint16_t* __restrict__ ws, float* __restrict__ bs) {
  const int i = blockIdx.x;
  const int src = sample_row_index(i, H, n_sample);
  for (int d = threadIdx.x; d < D; d += blockDim.x)
    ws[static_cast<size_t>(i) * D + d] = w[static_cast<size_t>(src) * D + d];
  if (threadIdx.x == 0) bs[i] = bias[src];
}

int grid_for(size_t n, int block, int cap = 148 * 16) {
  size_t g = (n + block - 1) / block;
  if (g > static_cast<size_t>(cap)) g = cap;
  if (g < 1) g = 1;
  return static_cast<int>(g);
}

}  // namespace

const char* cast_bf16_launch(const float* src, uint16_t* dst, size_t n, cudaStream_t stream) {
  cast_bf16_kernel<<<grid_for(n / 4 + 1, 256), 256, 0, stream>>>(src, dst, n);
  return cuda_err(cudaGetLastError());
}

const char* upcast_bf16_launch(const uint16_t* src, float* dst, size_t n, cudaStream_t stream) {
  upcast_bf16_kernel<<<grid_for(n / 4 + 1, 256), 256, 0, stream>>>(src, dst, n);
  return cuda_err(cudaGetLastError());
}

const char* pack_bitplanes_launch(const float* logits, int H, int D, int n_bits, uint8_t* packed,
                                  double* stats, cudaStream_t stream) {
  const size_t total = static_cast<size_t>(H) * D;
  const int grid = grid_for(total, 256);
  if (n_bits <= 4)
    pack_bitplanes_kernel<true><<<grid, 256, 0, stream>>>(logits, H, D, n_bits, packed, stats);
  else
    pack_bitplanes_kernel<false><<<grid, 256, 0, stream>>>(logits, H, D, n_bits, packed, stats);
  return cuda_err(cudaGetLastError());
}

const char* dequant_soft_launch(const float* logits, int H, int D, int n_bits, float* rows,
                                cudaStream_t stream) {
  const size_t total = static_cast<size_t>(H) * D;
  dequant_soft_kernel<<<grid_for(total, 256), 256, 0, stream>>>(logits, total, n_bits, rows);
  return cuda_err(cudaGetLastError());
}

const char* sample_rows_launch(const uint16_t* w_bf16, const float* bias, int H, int D, int n_sample,
                               uint16_t* w_sample, float* b_sample, cudaStream_t stream) {
  sample_rows_kernel<<<n_sample, 128, 0, stream>>>(w_bf16, bias, H, D, n_sample, w_sample, b_sample);
  return cuda_err(cudaGetLastError());
}

const char* residual_update_launch(const float* r, const float* recon, size_t n, float* out, cudaStream_t stream) {
  residual_update_kernel<<<grid_for(n / 4 + 1, 256), 256, 0, stream>>>(r, recon, n, out);
  return cuda_err(cudaGetLastError());
}

const char* split_bf16x3_launch(const float* src, uint16_t* hi, uint16_t* mid, uint16_t* lo, size_t n, cudaStream_t stream) {
  split_bf16x3_kernel<<<grid_for(n, 256), 256, 0, stream>>>(src, hi, mid, lo, n);
  return cuda_err(cudaGetLastError());
}

const char* split_bf16_launch(const float* src, uint16_t* hi, uint16_t* lo, size_t n, cudaStream_t stream) {
  split_bf16_kernel<<<grid_for(n / 4 + 1, 256), 256, 0, stream>>>(src, hi, lo, n);
  return cuda_err(cudaGetLastError());
}

const char* pack_ternary_launch(const float* w, int D, int H, float threshold, uint16_t* t_bf16, int8_t* t_rows,
                                cudaStream_t stream, uint16_t* t_t_bf16) {
  dim3 grid((H + 31) / 32, (D + 31) / 32), block(32, 8);
  pack_ternary_kernel<<<grid, block, 0, stream>>>(w, D, H, threshold, t_bf16, t_rows, t_t_bf16);
  return cuda_err(cudaGetLastError());
}

const char* transpose_launch(const float* src, int R, int C, float* dst, cudaStream_t stream) {
  dim3 grid((C + 31) / 32, (R + 31) / 32), block(32, 8);
  transpose_kernel<<<grid, block, 0, stream>>>(src, R, C, dst);
  return cuda_err(cudaGetLastError());
}

}  // namespace qsae
