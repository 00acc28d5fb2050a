// Reductions / elementwise kernels of the projection and MLP backward (row N1 of SURVEY.md 8(f)):
//   * colsum: bias gradient db[c] = sum_m dy[m][c]   (ATen's generic reduce ran at ~1.3 TB/s here)
//   * gelu_bwd_colsum: dh = dy * gelu'(h) (exact erf GELU, timm Mlp / nn.GELU of models/vit.py:118)
//     with the fc1 bias gradient sum_m dh[m][c] accumulated in the same pass.
#include "common.cuh"
#include "kernels.h"

namespace vrr {

namespace {

constexpr int kCsThreads = 256;   // 32 column-quads x 8 row lanes
constexpr int kCsRows = 256;      // rows per CTA

// 16-byte loads, eight of them in flight per thread: thread = VEC consecutive columns (8 bf16 / 4 fp32) x rows
// rl, rl + 16, ...; CTA = 16 column groups x 16 row lanes over kCsRows rows; grid (ceil(C / (16 VEC)), ceil(M / 256)).
// (The first version read 8 bytes per thread and row with a rolled loop: 38 us average over the step's bias
// gradients where the HBM floor is 24 us.)
template <typename T>
struct CsVec;
template <>
struct CsVec<float> {
  static constexpr int kVec = 4;
  using Raw = float4;
  static __device__ __forceinline__ void add(float (&acc)[4], const float4& v) {
    acc[0] += v.x; acc[1] += v.y; acc[2] += v.z; acc[3] += v.w;
  }
};
template <>
struct CsVec<__nv_bfloat16> {
  static constexpr int kVec = 8;
  using Raw = uint4;
  static __device__ __forceinline__ void add(float (&acc)[8], const uint4& v) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[e]));
      acc[2 * e] += f.x; acc[2 * e + 1] += f.y;
    }
  }
};
template <>
struct CsVec<__half> {
  static constexpr int kVec = 8;
  using Raw = uint4;
  static __device__ __forceinline__ void add(float (&acc)[8], const uint4& v) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[e]));
      acc[2 * e] += f.x; acc[2 * e + 1] += f.y;
    }
  }
};

template <typename T>
__global__ void __launch_bounds__(kCsThreads) colsum_vec_kernel(const T* __restrict__ x, float* __restrict__ out, int M, int C) {
  constexpr int VEC = CsVec<T>::kVec;
  using Raw = typename CsVec<T>::Raw;
  __shared__ float part[16][16 * VEC + 1];
  const int cg = threadIdx.x & 15, rl = threadIdx.x >> 4;
  const int c = (blockIdx.x * 16 + cg) * VEC;
  const int r0 = blockIdx.y * kCsRows + rl, r1 = min(M, blockIdx.y * kCsRows + kCsRows);
  float acc[VEC];
#pragma unroll
  for (int e = 0; e < VEC; ++e) acc[e] = 0.f;
  if (c < C) {
    const T* p = x + (size_t)r0 * C + c;
    int r = r0;
    for (; r + 7 * 16 < r1; r += 8 * 16, p += (size_t)8 * 16 * C) {
      Raw v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = *reinterpret_cast<const Raw*>(p + (size_t)k * 16 * C);
#pragma unroll
      for (int k = 0; k < 8; ++k) CsVec<T>::add(acc, v[k]);
    }
    for (; r < r1; r += 16, p += (size_t)16 * C) CsVec<T>::add(acc, *reinterpret_cast<const Raw*>(p));
  }
#pragma unroll
  for (int e = 0; e < VEC; ++e) part[rl][cg * VEC + e] = acc[e];
  __syncthreads();
  if (threadIdx.x < 16 * VEC) {
    const int col = blockIdx.x * 16 * VEC + threadIdx.x;
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k) s += part[k][threadIdx.x];
    if (col < C) atomicAdd(out + col, s);
  }
}

// grid (ceil(C / 128), ceil(M / kCsRows)); thread = 4 consecutive columns x strided rows
template <typename T>
__global__ void __launch_bounds__(kCsThreads) colsum_kernel(const T* __restrict__ x, float* __restrict__ out, int M, int C) {
  __shared__ float4 part[8][32];
  const int cq = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int c = blockIdx.x * 128 + cq * 4;
  const int r0 = blockIdx.y * kCsRows, r1 = min(M, r0 + kCsRows);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (c < C) {
    for (int r = r0 + rl; r < r1; r += 8) {
      const float4 v = ld4(x + (size_t)r * C + c);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
  }
  part[rl][cq] = acc;
  __syncthreads();
  if (rl == 0 && c < C) {
#pragma unroll
    for (int k = 1; k < 8; ++k) {
      const float4 v = part[k][cq];
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    atomicAdd(out + c + 0, acc.x);
    atomicAdd(out + c + 1, acc.y);
    atomicAdd(out + c + 2, acc.z);
    atomicAdd(out + c + 3, acc.w);
  }
}

// Any alignment (a view at an odd offset into a larger buffer): grid (ceil(C / 32), ceil(M / kCsRows)); thread = one
// column x rows rl, rl + 8, ...; element loads, a warp reads 32 consecutive columns of a row.
template <typename T>
__global__ void __launch_bounds__(kCsThreads) colsum_scalar_kernel(const T* __restrict__ x, float* __restrict__ out, int M,
                                                                   int C) {
  __shared__ float part[8][32];
  const int cl = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cl;
  const int r0 = blockIdx.y * kCsRows, r1 = min(M, r0 + kCsRows);
  float acc = 0.f;
  if (c < C)
    for (int r = r0 + rl; r < r1; r += 8) acc += Elem<T>::ld(x + (size_t)r * C + c);
  part[rl][cl] = acc;
  __syncthreads();
  if (rl == 0 && c < C) {
#pragma unroll
    for (int k = 1; k < 8; ++k) acc += part[k][cl];
    atomicAdd(out + c, acc);
  }
}

__device__ __forceinline__ float gelu_grad(float h) {
  // d/dh [ 0.5 h (1 + erf(h / sqrt 2)) ] = Phi(h) + h * phi(h),  phi(h) = exp(-h^2/2) / sqrt(2 pi).
  // erf by Abramowitz-Stegun 7.1.26 (|error| <= 1.5e-7): erf(z) = 1 - (a1 t + .. + a5 t^5) exp(-z^2),
  // t = 1 / (1 + 0.3275911 z), z = |h| / sqrt 2 - its exponential exp(-z^2) = exp(-h^2/2) is the one
  // phi(h) needs, so the whole derivative costs one MUFU.EX2, one MUFU.RCP and ~12 FMA-pipe ops
  // (libm erff alone is ~3x that, which made this kernel issue-bound instead of HBM-bound).
  const float e = __expf(-0.5f * h * h);
  const float z = fabsf(h) * 0.70710678118654752f;
  const float t = __fdividef(1.f, fmaf(0.3275911f, z, 1.f));
  float poly = fmaf(1.061405429f, t, -1.453152027f);
  poly = fmaf(poly, t, 1.421413741f);
  poly = fmaf(poly, t, -0.284496736f);
  poly = fmaf(poly, t, 0.254829592f);
  const float erf_abs = fmaf(-poly * t, e, 1.f);           // erf(|h| / sqrt 2)
  const float cdf = 0.5f * (1.f + copysignf(erf_abs, h));  // Phi(h)
  return fmaf(h * 0.3989422804014327f, e, cdf);
}

template <typename T>
__global__ void __launch_bounds__(kCsThreads) gelu_bwd_colsum_kernel(const T* __restrict__ dy, const T* __restrict__ h,
                                                                     T* __restrict__ dh, float* __restrict__ db, int M,
                                                                     int C) {
  __shared__ float4 part[8][32];
  const int cq = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int c = blockIdx.x * 128 + cq * 4;
  const int r0 = blockIdx.y * kCsRows, r1 = min(M, r0 + kCsRows);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (c < C) {
    for (int r = r0 + rl; r < r1; r += 8) {
      const size_t o = (size_t)r * C + c;
      const float4 g = ld4(dy + o), hv = ld4(h + o);
      float4 d;
      d.x = g.x * gelu_grad(hv.x);
      d.y = g.y * gelu_grad(hv.y);
      d.z = g.z * gelu_grad(hv.z);
      d.w = g.w * gelu_grad(hv.w);
      st4(dh + o, d);
      // the bias gradient sums the values as stored (rounded to T), like autograd's sum over dh
      T q[4];
      Elem<T>::st(&q[0], d.x); Elem<T>::st(&q[1], d.y); Elem<T>::st(&q[2], d.z); Elem<T>::st(&q[3], d.w);
      acc.x += Elem<T>::ld(&q[0]); acc.y += Elem<T>::ld(&q[1]); acc.z += Elem<T>::ld(&q[2]); acc.w += Elem<T>::ld(&q[3]);
    }
  }
  part[rl][cq] = acc;
  __syncthreads();
  if (rl == 0 && c < C) {
#pragma unroll
    for (int k = 1; k < 8; ++k) {
      const float4 v = part[k][cq];
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    atomicAdd(db + c + 0, acc.x);
    atomicAdd(db + c + 1, acc.y);
    atomicAdd(db + c + 2, acc.z);
    atomicAdd(db + c + 3, acc.w);
  }
}

// SIMT-family fallbacks of the GEMM epilogues VRR_EPI_BIAS_GELU_GRAD / VRR_EPI_MUL (fp32, odd shapes, forced SIMT)
template <typename T>
__global__ void gelu_grad_inplace_kernel(T* __restrict__ h, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    Elem<T>::st(h + i, gelu_grad(Elem<T>::ld(h + i)));
}
template <typename T>
__global__ void mul_inplace_kernel(T* __restrict__ c, const T* __restrict__ m, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    Elem<T>::st(c + i, Elem<T>::ld(c + i) * Elem<T>::ld(m + i));
}

// One thread per group of 8 elements (one Philox call).  c <- T(c * f); c2 (h on entry) <- T(T(gelu'(h)) * f).
template <typename T>
__global__ void drop_gelu_kernel(T* __restrict__ c, T* __restrict__ c2, int M, int N, const DropView dv) {
  const uint2 key = dv.key();
  const size_t groups = (size_t)M * N / 8;
  for (size_t gi = (size_t)blockIdx.x * blockDim.x + threadIdx.x; gi < groups; gi += (size_t)gridDim.x * blockDim.x) {
    const int m = (int)(gi * 8 / N), n = (int)(gi * 8 - (size_t)m * N);
    const float4 f0 = dv.factor4(key, m, n, N, dv.s), f1 = dv.factor4(key, m, n + 4, N, dv.s);
    const float f[8] = {f0.x, f0.y, f0.z, f0.w, f1.x, f1.y, f1.z, f1.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      T* pc = c + gi * 8 + j;
      Elem<T>::st(pc, Elem<T>::ld(pc) * f[j]);
      if (c2) {
        T* p2 = c2 + gi * 8 + j;
        Elem<T>::st(p2, Elem<T>::round(gelu_grad(Elem<T>::ld(p2))) * f[j]);
      }
    }
  }
}

// keep[m][n] (element mask alone) and keep_path[b] (stochastic depth per image), 1 = kept
__global__ void dropout_mask_kernel(const DropView dv, uint8_t* __restrict__ keep, uint8_t* __restrict__ keep_path,
                                    int M, int E, int images) {
  const uint2 key = dv.key();
  const size_t groups = keep ? (size_t)M * E / 8 : 0;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t gi = (size_t)blockIdx.x * blockDim.x + threadIdx.x; gi < groups; gi += stride) {
    const int m = (int)(gi * 8 / E), n = (int)(gi * 8 - (size_t)m * E);
    const float4 f0 = dv.factor4(key, m, n, E, 1.f), f1 = dv.factor4(key, m, n + 4, E, 1.f);
    uint2 w;
    w.x = (f0.x != 0.f ? 1u : 0u) | (f0.y != 0.f ? 1u << 8 : 0u) | (f0.z != 0.f ? 1u << 16 : 0u) | (f0.w != 0.f ? 1u << 24 : 0u);
    w.y = (f1.x != 0.f ? 1u : 0u) | (f1.y != 0.f ? 1u << 8 : 0u) | (f1.z != 0.f ? 1u << 16 : 0u) | (f1.w != 0.f ? 1u << 24 : 0u);
    *reinterpret_cast<uint2*>(keep + gi * 8) = w;
  }
  if (keep_path)
    for (size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x; b < (size_t)images; b += stride)
      keep_path[b] = dv.row_factor(key, (int)b * dv.rows_per_sample) != 0.f ? 1 : 0;
}

}  // namespace

int drop_gelu_inplace(void* c, void* c2, int M, int N, int dtype, const DropView& dv, cudaStream_t st) {
  const size_t groups = (size_t)M * N / 8;
  const int grid = (int)((groups + 255) / 256 < 148 * 8 ? (groups + 255) / 256 : 148 * 8);
  if (dtype == VRR_F32) drop_gelu_kernel<float><<<grid, 256, 0, st>>>((float*)c, (float*)c2, M, N, dv);
  else if (dtype == VRR_BF16) drop_gelu_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>((__nv_bfloat16*)c, (__nv_bfloat16*)c2, M, N, dv);
  else drop_gelu_kernel<__half><<<grid, 256, 0, st>>>((__half*)c, (__half*)c2, M, N, dv);
  VRR_LAUNCHED();
  return VRR_OK;
}

int dropout_mask(const DropView& dv, uint8_t* keep, uint8_t* keep_path, int M, int E, cudaStream_t st) {
  const int images = dv.rows_per_sample > 0 ? ceil_div(M, dv.rows_per_sample) : 0;
  const size_t work = keep ? (size_t)M * E / 8 : (size_t)images;
  const int grid = (int)((work + 255) / 256 < 148 * 8 ? (work + 255) / 256 : 148 * 8);
  dropout_mask_kernel<<<grid, 256, 0, st>>>(dv, keep, keep_path, M, E, keep_path ? images : 0);
  VRR_LAUNCHED();
  return VRR_OK;
}

int gelu_grad_inplace(void* h, size_t n, int dtype, cudaStream_t st) {
  const int grid = (int)((n + 255) / 256 < 148 * 8 ? (n + 255) / 256 : 148 * 8);
  if (dtype == VRR_F32) gelu_grad_inplace_kernel<float><<<grid, 256, 0, st>>>((float*)h, n);
  else if (dtype == VRR_BF16) gelu_grad_inplace_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>((__nv_bfloat16*)h, n);
  else gelu_grad_inplace_kernel<__half><<<grid, 256, 0, st>>>((__half*)h, n);
  VRR_LAUNCHED();
  return VRR_OK;
}

int mul_inplace(void* c, const void* m, size_t n, int dtype, cudaStream_t st) {
  const int grid = (int)((n + 255) / 256 < 148 * 8 ? (n + 255) / 256 : 148 * 8);
  if (dtype == VRR_F32) mul_inplace_kernel<float><<<grid, 256, 0, st>>>((float*)c, (const float*)m, n);
  else if (dtype == VRR_BF16) mul_inplace_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>((__nv_bfloat16*)c, (const __nv_bfloat16*)m, n);
  else mul_inplace_kernel<__half><<<grid, 256, 0, st>>>((__half*)c, (const __half*)m, n);
  VRR_LAUNCHED();
  return VRR_OK;
}

int colsum(const void* x, float* out, int M, int C, int dtype, cudaStream_t st) {
  VRR_REQUIRE(C % 4 == 0, VRR_ERR_UNSUPPORTED, "colsum: C = %d must be a multiple of 4", C);
  VRR_CUDA(cudaMemsetAsync(out, 0, (size_t)C * sizeof(float), st));
  const int vec = dtype == VRR_F32 ? 4 : 8;
  if (C % vec == 0 && ((uintptr_t)x & 15) == 0) {
    dim3 grid(ceil_div(C, 16 * vec), ceil_div(M, kCsRows));
    if (dtype == VRR_F32) colsum_vec_kernel<float><<<grid, kCsThreads, 0, st>>>((const float*)x, out, M, C);
    else if (dtype == VRR_BF16) colsum_vec_kernel<__nv_bfloat16><<<grid, kCsThreads, 0, st>>>((const __nv_bfloat16*)x, out, M, C);
    else colsum_vec_kernel<__half><<<grid, kCsThreads, 0, st>>>((const __half*)x, out, M, C);
    VRR_LAUNCHED();
    return VRR_OK;
  }
  // colsum_kernel reads 4 elements at a time (16 bytes fp32, 8 bytes bf16 / fp16): a base address off that grid takes the
  // element-wise kernel
  if (((uintptr_t)x & (dtype == VRR_F32 ? 15 : 7)) != 0) {
    dim3 grid(ceil_div(C, 32), ceil_div(M, kCsRows));
    if (dtype == VRR_F32) colsum_scalar_kernel<float><<<grid, kCsThreads, 0, st>>>((const float*)x, out, M, C);
    else if (dtype == VRR_BF16) colsum_scalar_kernel<__nv_bfloat16><<<grid, kCsThreads, 0, st>>>((const __nv_bfloat16*)x, out, M, C);
    else colsum_scalar_kernel<__half><<<grid, kCsThreads, 0, st>>>((const __half*)x, out, M, C);
    VRR_LAUNCHED();
    return VRR_OK;
  }
  dim3 grid(ceil_div(C, 128), ceil_div(M, kCsRows));
  if (dtype == VRR_F32) colsum_kernel<float><<<grid, kCsThreads, 0, st>>>((const float*)x, out, M, C);
  else if (dtype == VRR_BF16) colsum_kernel<__nv_bfloat16><<<grid, kCsThreads, 0, st>>>((const __nv_bfloat16*)x, out, M, C);
  else colsum_kernel<__half><<<grid, kCsThreads, 0, st>>>((const __half*)x, out, M, C);
  VRR_LAUNCHED();
  return VRR_OK;
}

int gelu_bwd_colsum(const void* dy, const void* h, void* dh, float* db, int M, int C, int dtype, cudaStream_t st) {
  VRR_REQUIRE(C % 4 == 0, VRR_ERR_UNSUPPORTED, "gelu_bwd: C = %d must be a multiple of 4", C);
  VRR_CUDA(cudaMemsetAsync(db, 0, (size_t)C * sizeof(float), st));
  dim3 grid(ceil_div(C, 128), ceil_div(M, kCsRows));
  if (dtype == VRR_F32)
    gelu_bwd_colsum_kernel<float><<<grid, kCsThreads, 0, st>>>((const float*)dy, (const float*)h, (float*)dh, db, M, C);
  else if (dtype == VRR_BF16)
    gelu_bwd_colsum_kernel<__nv_bfloat16><<<grid, kCsThreads, 0, st>>>((const __nv_bfloat16*)dy, (const __nv_bfloat16*)h,
                                                                      (__nv_bfloat16*)dh, db, M, C);
  else
    gelu_bwd_colsum_kernel<__half><<<grid, kCsThreads, 0, st>>>((const __half*)dy, (const __half*)h, (__half*)dh, db, M, C);
  VRR_LAUNCHED();
  return VRR_OK;
}

}  // namespace vrr
