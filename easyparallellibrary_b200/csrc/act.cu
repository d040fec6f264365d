// Fused bias + GELU (tanh approximation, as GPT-2/BERT use) forward and backward, plus bias-gradient
// column reduction.  Element-wise, HBM-bound; in the GEMM path these run as the tcgen05 epilogue
// (gemm_tcgen05.cu), the stand-alone kernels serve non-GEMM call sites and are the numerics reference.
#include "epl_common.cuh"
#include <algorithm>

namespace epl {

EPL_DEVICE float gelu_tanh(float x) {
  const float k0 = 0.7978845608028654f, k1 = 0.044715f;
  float u = k0 * (x + k1 * x * x * x);
  return 0.5f * x * (1.f + tanhf(u));
}
EPL_DEVICE float gelu_tanh_grad(float x) {
  const float k0 = 0.7978845608028654f, k1 = 0.044715f;
  float u = k0 * (x + k1 * x * x * x);
  float t = tanhf(u);
  return 0.5f * (1.f + t) + 0.5f * x * (1.f - t * t) * k0 * (1.f + 3.f * k1 * x * x);
}

// y = gelu(x + bias); pre = x + bias (optional, saved for backward).  x:[rows, D], bias:[D]
template <typename T, bool kSavePre>
__global__ void __launch_bounds__(256) bias_gelu_fwd_kernel(const T* __restrict__ x, const T* __restrict__ bias,
                                                            T* __restrict__ y, T* __restrict__ pre, int64_t nvec, int dvec) {
  constexpr int E = 16 / sizeof(T);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += stride) {
    Vec<T, E> xv = ld_vec<T, E>(x + i * E);
    Vec<T, E> o, p;
    if (bias != nullptr) {
      Vec<T, E> bv = ld_vec<T, E>(bias + (i % dvec) * E);
#pragma unroll
      for (int e = 0; e < E; ++e) {
        float h = to_f32<T>(xv.v[e]) + to_f32<T>(bv.v[e]);
        p.v[e] = from_f32<T>(h);
        o.v[e] = from_f32<T>(gelu_tanh(to_f32<T>(p.v[e])));
      }
    } else {
#pragma unroll
      for (int e = 0; e < E; ++e) { p.v[e] = xv.v[e]; o.v[e] = from_f32<T>(gelu_tanh(to_f32<T>(xv.v[e]))); }
    }
    st_vec<T, E>(y + i * E, o);
    if constexpr (kSavePre) st_vec<T, E>(pre + i * E, p);
  }
}

// dpre = dy * gelu'(pre)
template <typename T>
__global__ void __launch_bounds__(256) gelu_bwd_kernel(const T* __restrict__ pre, const T* __restrict__ dy,
                                                       T* __restrict__ dpre, int64_t nvec) {
  constexpr int E = 16 / sizeof(T);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += stride) {
    Vec<T, E> pv = ld_vec<T, E>(pre + i * E);
    Vec<T, E> dv = ld_vec<T, E>(dy + i * E);
    Vec<T, E> o;
#pragma unroll
    for (int e = 0; e < E; ++e) o.v[e] = from_f32<T>(to_f32<T>(dv.v[e]) * gelu_tanh_grad(to_f32<T>(pv.v[e])));
    st_vec<T, E>(dpre + i * E, o);
  }
}

// column sums: scratch[blockIdx.y][d] = sum over this CTA's rows of x[r][d].  Block (32, 8): thread x owns 16 bytes of
// consecutive columns, rows are strided over threadIdx.y and blockIdx.y; per-CTA smem reduction, one partial per column per
// CTA row, summed in row order by finish_colsum_kernel (no atomics: the result does not depend on which CTA finishes first).
template <typename T>
__global__ void __launch_bounds__(256) colsum_kernel(const T* __restrict__ x, float* __restrict__ scratch, int rows, int D) {
  constexpr int E = 16 / sizeof(T);
  const int col = (blockIdx.x * 32 + threadIdx.x) * E;
  float acc[E];
#pragma unroll
  for (int e = 0; e < E; ++e) acc[e] = 0.f;
  if (col < D) {
    const int step = gridDim.y * 8;
    int r = blockIdx.y * 8 + threadIdx.y;
    for (; r + 3 * step < rows; r += 4 * step) {          // four independent 16-byte loads in flight per thread
      Vec<T, E> v0 = ld_vec<T, E>(x + (size_t)r * D + col);
      Vec<T, E> v1 = ld_vec<T, E>(x + (size_t)(r + step) * D + col);
      Vec<T, E> v2 = ld_vec<T, E>(x + (size_t)(r + 2 * step) * D + col);
      Vec<T, E> v3 = ld_vec<T, E>(x + (size_t)(r + 3 * step) * D + col);
#pragma unroll
      for (int e = 0; e < E; ++e) acc[e] += (to_f32<T>(v0.v[e]) + to_f32<T>(v1.v[e])) + (to_f32<T>(v2.v[e]) + to_f32<T>(v3.v[e]));
    }
    for (; r < rows; r += step) {
      Vec<T, E> v = ld_vec<T, E>(x + (size_t)r * D + col);
#pragma unroll
      for (int e = 0; e < E; ++e) acc[e] += to_f32<T>(v.v[e]);
    }
  }
  __shared__ float s[8][32 * E + 1];
#pragma unroll
  for (int e = 0; e < E; ++e) s[threadIdx.y][threadIdx.x * E + e] = acc[e];
  __syncthreads();
  for (int c = threadIdx.y * 32 + threadIdx.x; c < 32 * E; c += 256) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += s[k][c];
    const int gc = blockIdx.x * 32 * E + c;
    if (gc < D) scratch[(size_t)blockIdx.y * D + gc] = t;
  }
}

// out[d] = sum over the partial rows of scratch[.][d] in a fixed order: block (32, 8), thread (x, y) adds rows y, y + 8, ...
// of column x in row order, then the eight sums are added in y order.
template <typename T>
__global__ void __launch_bounds__(256) finish_colsum_kernel(const float* __restrict__ scratch, T* __restrict__ out, int D, int parts,
                                                            int accumulate) {
  __shared__ float s[8][33];
  const int d = blockIdx.x * 32 + threadIdx.x;
  float v = 0.f;
  if (d < D) {
#pragma unroll 4
    for (int y = threadIdx.y; y < parts; y += 8) v += scratch[(size_t)y * D + d];
  }
  s[threadIdx.y][threadIdx.x] = v;
  __syncthreads();
  if (threadIdx.y == 0 && d < D) {
    float t = s[0][threadIdx.x];
#pragma unroll
    for (int k = 1; k < 8; ++k) t += s[k][threadIdx.x];
    if (accumulate) t += to_f32<T>(out[d]);
    out[d] = from_f32<T>(t);
  }
}

// y = a + b (residual add), 16-byte vectors
template <typename T>
__global__ void __launch_bounds__(256) add_kernel(const T* __restrict__ a, const T* __restrict__ b, T* __restrict__ y, int64_t nvec) {
  constexpr int E = 16 / sizeof(T);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += stride) {
    Vec<T, E> av = ld_vec<T, E>(a + i * E), bv = ld_vec<T, E>(b + i * E), o;
#pragma unroll
    for (int e = 0; e < E; ++e) o.v[e] = from_f32<T>(to_f32<T>(av.v[e]) + to_f32<T>(bv.v[e]));
    st_vec<T, E>(y + i * E, o);
  }
}

static int grid_for(int64_t nvec) { return (int)std::max<int64_t>(1, std::min<int64_t>((nvec + 255) / 256, (int64_t)kNumSMs * 16)); }

}  // namespace epl
using namespace epl;

#define BY_DTYPE(dtype, ...)                                           \
  if (dtype == EPL_F32) { using T = float; __VA_ARGS__; }              \
  else if (dtype == EPL_BF16) { using T = __nv_bfloat16; __VA_ARGS__; }\
  else { using T = __half; __VA_ARGS__; }

// n = rows*D elements; D and n must be multiples of 16/sizeof(T)
extern "C" int epl_bias_gelu_fwd(const void* x, const void* bias, void* y, void* pre, int64_t n, int D, int dtype, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  BY_DTYPE(dtype, {
    constexpr int E = 16 / sizeof(T);
    int64_t nvec = n / E;
    if (pre) bias_gelu_fwd_kernel<T, true><<<grid_for(nvec), 256, 0, st>>>((const T*)x, (const T*)bias, (T*)y, (T*)pre, nvec, D / E);
    else bias_gelu_fwd_kernel<T, false><<<grid_for(nvec), 256, 0, st>>>((const T*)x, (const T*)bias, (T*)y, nullptr, nvec, D / E);
  });
  return EPL_CHECK_LAUNCH();
}

extern "C" int epl_gelu_bwd(const void* pre, const void* dy, void* dpre, int64_t n, int dtype, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  BY_DTYPE(dtype, {
    constexpr int E = 16 / sizeof(T);
    int64_t nvec = n / E;
    gelu_bwd_kernel<T><<<grid_for(nvec), 256, 0, st>>>((const T*)pre, (const T*)dy, (T*)dpre, nvec);
  });
  return EPL_CHECK_LAUNCH();
}

// CTA rows of the colsum grid = rows of fp32[D] partials the caller provides as scratch
extern "C" int epl_colsum_parts(int rows, int D, int dtype) {
  const int E = 16 / (dtype == 0 ? 4 : 2);
  const int gx = (D + 32 * E - 1) / (32 * E);
  return std::max(1, std::min((rows + 31) / 32, (8 * kNumSMs + gx - 1) / gx));
}

// scratch: fp32 [epl_colsum_parts(rows, D, dtype), D]
extern "C" int epl_colsum(const void* x, void* out, void* scratch, int rows, int D, int dtype, int accumulate, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  const int parts = epl_colsum_parts(rows, D, dtype);
  BY_DTYPE(dtype, {
    constexpr int E = 16 / sizeof(T);
    const int gx = (D + 32 * E - 1) / (32 * E);
    dim3 block(32, 8), grid(gx, parts);
    colsum_kernel<T><<<grid, block, 0, st>>>((const T*)x, (float*)scratch, rows, D);
    finish_colsum_kernel<T><<<(D + 31) / 32, dim3(32, 8), 0, st>>>((const float*)scratch, (T*)out, D, parts, accumulate);
  });
  return EPL_CHECK_LAUNCH();
}

extern "C" int epl_add(const void* a, const void* b, void* y, int64_t n, int dtype, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  BY_DTYPE(dtype, {
    constexpr int E = 16 / sizeof(T);
    int64_t nvec = n / E;
    add_kernel<T><<<grid_for(nvec), 256, 0, st>>>((const T*)a, (const T*)b, (T*)y, nvec);
  });
  return EPL_CHECK_LAUNCH();
}

// ---------------------------------------------------------------------------------------------------------
// Per-tensor e4m3 quantisation for the fp8 GEMM path (amp.level = "fp8"): pass 1 = absolute maximum, pass 2 = scale by
// 448 / amax, saturate, cast; the de-quantisation factor amax / 448 is left in device memory for the GEMM epilogue (no host
// round trip).
// ---------------------------------------------------------------------------------------------------------
#include <cuda_fp8.h>
namespace epl {
template <typename T>
__global__ void __launch_bounds__(256) amax_kernel(const T* __restrict__ x, int64_t n, uint32_t* __restrict__ amax_bits) {
  float m = 0.f;
  const int64_t nvec = n >> 3, stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += stride) {
    Vec<T, 8> v = ld_vec<T, 8>(x + 8 * i);
#pragma unroll
    for (int j = 0; j < 8; ++j) m = fmaxf(m, fabsf(to_f32<T>(v.v[j])));
  }
  for (int64_t i = (nvec << 3) + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) m = fmaxf(m, fabsf(to_f32<T>(x[i])));
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0) atomicMax(amax_bits, __float_as_uint(m));      // non-negative floats order like their bit patterns
}

template <typename T>
__global__ void __launch_bounds__(256) cast_e4m3_kernel(const T* __restrict__ x, int64_t n, const uint32_t* __restrict__ amax_bits,
                                                         uint8_t* __restrict__ out, float* __restrict__ inv_scale) {
  const float amax = fmaxf(__uint_as_float(*amax_bits), 1e-12f);
  const float s = 448.f / amax;
  if (blockIdx.x == 0 && threadIdx.x == 0) *inv_scale = amax / 448.f;
  const int64_t nvec = n >> 3, stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += stride) {
    Vec<T, 8> v = ld_vec<T, 8>(x + 8 * i);
    uint32_t w[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const __nv_fp8x2_storage_t lo = __nv_cvt_float2_to_fp8x2(make_float2(to_f32<T>(v.v[4 * h]) * s, to_f32<T>(v.v[4 * h + 1]) * s), __NV_SATFINITE, __NV_E4M3);
      const __nv_fp8x2_storage_t hi = __nv_cvt_float2_to_fp8x2(make_float2(to_f32<T>(v.v[4 * h + 2]) * s, to_f32<T>(v.v[4 * h + 3]) * s), __NV_SATFINITE, __NV_E4M3);
      w[h] = (uint32_t)lo | ((uint32_t)hi << 16);
    }
    *reinterpret_cast<uint2*>(out + 8 * i) = make_uint2(w[0], w[1]);
  }
  for (int64_t i = (nvec << 3) + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    out[i] = (uint8_t)__nv_cvt_float_to_fp8(to_f32<T>(x[i]) * s, __NV_SATFINITE, __NV_E4M3);
}
}  // namespace epl

// x: n elements (bf16 / fp16 / fp32, 16-byte aligned), out: n bytes (8-byte aligned), amax_scratch: one uint32 (zeroed here),
// inv_scale: one float.
extern "C" int epl_quantize_e4m3(const void* x, int dtype, int64_t n, void* out, void* amax_scratch, void* inv_scale, void* stream) {
  using namespace epl;
  cudaStream_t st = (cudaStream_t)stream;
  cudaMemsetAsync(amax_scratch, 0, 4, st);
  int blocks = (int)std::min<int64_t>((n / 8 + 255) / 256 + 1, (int64_t)kNumSMs * 8);
  if (dtype == EPL_BF16) {
    amax_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>((const __nv_bfloat16*)x, n, (uint32_t*)amax_scratch);
    cast_e4m3_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>((const __nv_bfloat16*)x, n, (const uint32_t*)amax_scratch, (uint8_t*)out, (float*)inv_scale);
  } else if (dtype == EPL_F16) {
    amax_kernel<__half><<<blocks, 256, 0, st>>>((const __half*)x, n, (uint32_t*)amax_scratch);
    cast_e4m3_kernel<__half><<<blocks, 256, 0, st>>>((const __half*)x, n, (const uint32_t*)amax_scratch, (uint8_t*)out, (float*)inv_scale);
  } else {
    amax_kernel<float><<<blocks, 256, 0, st>>>((const float*)x, n, (uint32_t*)amax_scratch);
    cast_e4m3_kernel<float><<<blocks, 256, 0, st>>>((const float*)x, n, (const uint32_t*)amax_scratch, (uint8_t*)out, (float*)inv_scale);
  }
  return EPL_CHECK_LAUNCH();
}
