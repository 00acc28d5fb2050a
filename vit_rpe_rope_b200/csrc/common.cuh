// Shared host/device helpers for libvrr_b200.so (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "../../include/vrr.h"

namespace vrr {

// ---- error reporting -------------------------------------------------------------------------
void set_error(const char* fmt, ...);
extern std::atomic<uint64_t> g_launches;
extern std::atomic<int> g_impl;

#define VRR_REQUIRE(cond, code, ...)      \
  do {                                    \
    if (!(cond)) {                        \
      ::vrr::set_error(__VA_ARGS__);      \
      return (code);                      \
    }                                     \
  } while (0)

#define VRR_CUDA(expr)                                                              \
  do {                                                                              \
    cudaError_t e__ = (expr);                                                       \
    if (e__ != cudaSuccess) {                                                       \
      ::vrr::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__),     \
                       __FILE__, __LINE__);                                         \
      return VRR_ERR_CUDA;                                                          \
    }                                                                               \
  } while (0)

// Call after every kernel launch: counts it and surfaces launch-configuration errors.
#define VRR_LAUNCHED()                                   \
  do {                                                   \
    ::vrr::g_launches.fetch_add(1, std::memory_order_relaxed); \
    VRR_CUDA(cudaGetLastError());                        \
  } while (0)

int require_device();  // VRR_OK or VRR_ERR_NO_DEVICE (state cached per device ordinal)
int sm_count();        // SM count of the current device
extern std::atomic<uint64_t> g_family_launches[3];  // indexed by vrr_impl: dispatches per kernel family
bool first_use_on_device(std::atomic<unsigned char>* flags);  // flags: static array [64], one per device

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (kernel, device).
#define VRR_SMEM_ATTR_ONCE(kernel, bytes)                                                              \
  do {                                                                                                 \
    static std::atomic<unsigned char> flags__[64];                                                     \
    if (::vrr::first_use_on_device(flags__))                                                           \
      VRR_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes))); \
  } while (0)
#define VRR_COUNT_FAMILY(f) ::vrr::g_family_launches[(f)].fetch_add(1, std::memory_order_relaxed)

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
// bf16 and fp16 run the same kernels (the tcgen05 family where the shape allows): "a 16-bit dtype"
static inline bool is16(int dtype) { return dtype == VRR_BF16 || dtype == VRR_F16; }

// ---- element type traits -----------------------------------------------------------------------
template <typename T>
struct Elem;
template <>
struct Elem<float> {
  static __device__ __forceinline__ float ld(const float* p) { return *p; }
  static __device__ __forceinline__ void st(float* p, float v) { *p = v; }
  static __device__ __forceinline__ float round(float v) { return v; }
};
template <>
struct Elem<__nv_bfloat16> {
  static __device__ __forceinline__ float ld(const __nv_bfloat16* p) { return __bfloat162float(*p); }
  static __device__ __forceinline__ void st(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
  static __device__ __forceinline__ float round(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }
};
template <>
struct Elem<__half> {
  static __device__ __forceinline__ float ld(const __half* p) { return __half2float(*p); }
  static __device__ __forceinline__ void st(__half* p, float v) { *p = __float2half_rn(v); }
  static __device__ __forceinline__ float round(float v) { return __half2float(__float2half_rn(v)); }
};

// Load 4 consecutive elements (16B-aligned for float, 8B for bf16 / fp16) as floats.
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 ld4(const __nv_bfloat16* p) {
  uint2 raw = *reinterpret_cast<const uint2*>(p);
  __nv_bfloat162 a = *reinterpret_cast<__nv_bfloat162*>(&raw.x);
  __nv_bfloat162 b = *reinterpret_cast<__nv_bfloat162*>(&raw.y);
  float2 fa = __bfloat1622float2(a), fb = __bfloat1622float2(b);
  return make_float4(fa.x, fa.y, fb.x, fb.y);
}
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void st4(__nv_bfloat16* p, float4 v) {
  __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
  uint2 raw;
  raw.x = *reinterpret_cast<uint32_t*>(&a);
  raw.y = *reinterpret_cast<uint32_t*>(&b);
  *reinterpret_cast<uint2*>(p) = raw;
}
__device__ __forceinline__ float4 ld4(const __half* p) {
  uint2 raw = *reinterpret_cast<const uint2*>(p);
  float2 fa = __half22float2(*reinterpret_cast<__half2*>(&raw.x)), fb = __half22float2(*reinterpret_cast<__half2*>(&raw.y));
  return make_float4(fa.x, fa.y, fb.x, fb.y);
}
__device__ __forceinline__ void st4(__half* p, float4 v) {
  __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
  uint2 raw;
  raw.x = *reinterpret_cast<uint32_t*>(&a);
  raw.y = *reinterpret_cast<uint32_t*>(&b);
  *reinterpret_cast<uint2*>(p) = raw;
}

// ---- counter-based randomness for dropout / stochastic depth (vrr_drop_desc) ----------------------------
// Philox4x32-10 (Salmon et al., SC'11; the Random123 constants).  Counter {g lo, g hi, site, stream}, key = the 64-bit
// seed (low word first).  Element (m, n) of an [M][E] site (E % 8 == 0) is group g = (m E + n) / 8 of stream 0 and
// uses 16-bit half (n & 1) of output word (n % 8) >> 1; image b's stochastic-depth decision is the low half of word
// 0 of counter {b, 0, site, 1}.  Kept iff the 16 bits are below the threshold t = round((1 - p) 65536).
// oracle/philox_np.py restates all of it.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r) {
      k.x += 0x9E3779B9u;
      k.y += 0xBB67AE85u;
    }
    const uint32_t lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
    const uint32_t lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
  }
  return c;
}

// Device-side view of vrr_drop_desc.  A threshold of 65536 keeps everything and draws nothing.
struct DropView {
  const unsigned long long* seed;
  uint32_t t, t_path;     // element / stochastic-depth keep thresholds
  float s;                // (1 / (1 - p)) * (1 / (1 - p_path)), formed in fp32
  int rows_per_sample, site;
  __device__ __forceinline__ uint2 key() const {
    const unsigned long long k = *seed;
    return make_uint2((uint32_t)k, (uint32_t)(k >> 32));
  }
  // factor of row m before the element mask: s, or 0 when the row's image is dropped
  __device__ __forceinline__ float row_factor(uint2 k, int m) const {
    if (t_path >= 65536u) return s;
    const uint4 r = philox4x32_10(make_uint4((uint32_t)(m / rows_per_sample), 0u, (uint32_t)site, 1u), k);
    return (r.x & 0xFFFFu) < t_path ? s : 0.f;
  }
  __device__ __forceinline__ uint4 bits(uint2 k, unsigned long long g) const {
    return philox4x32_10(make_uint4((uint32_t)g, (uint32_t)(g >> 32), (uint32_t)site, 0u), k);
  }
  // factors of elements (m, n .. n + 3), n % 4 == 0, given the row factor fr
  __device__ __forceinline__ float4 factor4(uint2 k, int m, int n, int E, float fr) const {
    if (t >= 65536u) return make_float4(fr, fr, fr, fr);
    const uint4 r = bits(k, ((unsigned long long)m * E + n) >> 3);
    const uint32_t w0 = (n & 4) ? r.z : r.x, w1 = (n & 4) ? r.w : r.y;
    return make_float4((w0 & 0xFFFFu) < t ? fr : 0.f, (w0 >> 16) < t ? fr : 0.f, (w1 & 0xFFFFu) < t ? fr : 0.f,
                       (w1 >> 16) < t ? fr : 0.f);
  }
  __device__ __forceinline__ float factor(uint2 k, int m, int n, int E, float fr) const {
    if (t >= 65536u) return fr;
    const uint4 r = bits(k, ((unsigned long long)m * E + n) >> 3);
    const int j = n & 7;
    const uint32_t w = j < 2 ? r.x : (j < 4 ? r.y : (j < 6 ? r.z : r.w));
    return ((j & 1) ? (w >> 16) : (w & 0xFFFFu)) < t ? fr : 0.f;
  }
};
// SiLU of a SwiGLU Mlp (vrr_gemm_swiglu) and its derivative, sigma = 1 / (1 + 2^(-g log2 e)) on the MUFU unit:
//   s = silu(g) = g sigma,  ds = silu'(g) = sigma + s (1 - sigma).
// ex2.approx (relative error <= 2^-22) of an argument rounded to fp32 (relative error of the exponential
// <= |g| 2^-24) and rcp.approx (<= 1 ulp) give |s - silu(g)| <= 2^-20 (1 + |g|) |silu(g)| + 2^-126 (1 + |g|) and
// |ds - silu'(g)| <= 2^-20 (1 + |g|) (sigma + |silu(g)| (1 - sigma)) + 2^-126 (1 + |g|) for finite g
// (tests/test_swiglu_gpu.py); the absolute term is sigma flushed to zero below the fp32 normal range (g < -87.3).
// g -> -inf: the exponential overflows to +inf, sigma = 0, s = -0, ds = 0.
__device__ __forceinline__ void silu_and_grad(float g, float& s, float& ds) {
  float e, sig;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(__fmul_rn(g, -1.4426950408889634f)));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(sig) : "f"(__fadd_rn(e, 1.f)));
  s = __fmul_rn(g, sig);
  ds = __fmaf_rn(s, __fadd_rn(1.f, -sig), sig);
}

__device__ __forceinline__ float4 mul4_rn(float4 a, float4 f) {
  return make_float4(__fmul_rn(a.x, f.x), __fmul_rn(a.y, f.y), __fmul_rn(a.z, f.z), __fmul_rn(a.w, f.w));
}

// QK-norm (vrr_qkv_rope_norm_fwd / _bwd): the LayerNorm of one q or k head row of n = Dh channels, in fp32.
//   mean = (sum x) / n, var = (sum (x - mean)^2) / n (biased), rstd = rsqrtf(var + eps); each sum runs in four
//   interleaved partials (channel 4i + e adds into partial e), combined as (p0 + p1) + (p2 + p3).
// xhat and y are formed without contraction: the backward recomputes the y the forward rotated, bit for bit.
__device__ __forceinline__ float qk_norm_xhat(float x, float mean, float rstd) { return __fmul_rn(__fsub_rn(x, mean), rstd); }
__device__ __forceinline__ float qk_norm_y(float xhat, float g, float b) { return __fmaf_rn(xhat, g, b); }
__device__ __forceinline__ float2 qk_norm_stats(const float* x, int n, float eps) {
  const float inv = 1.f / (float)n;  // n is a power of two: exact
  float p[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int i = 0; i < n; i += 4)
#pragma unroll
    for (int e = 0; e < 4; ++e) p[e] = __fadd_rn(p[e], x[i + e]);
  const float mean = __fmul_rn(__fadd_rn(__fadd_rn(p[0], p[1]), __fadd_rn(p[2], p[3])), inv);
#pragma unroll
  for (int e = 0; e < 4; ++e) p[e] = 0.f;
#pragma unroll
  for (int i = 0; i < n; i += 4)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float d = __fsub_rn(x[i + e], mean);
      p[e] = __fmaf_rn(d, d, p[e]);
    }
  const float var = __fmul_rn(__fadd_rn(__fadd_rn(p[0], p[1]), __fadd_rn(p[2], p[3])), inv);
  return make_float2(mean, rsqrtf(__fadd_rn(var, eps)));
}

// vrr_drop_desc -> DropView (validated); `*active` = false when the desc draws nothing (NULL, or both
// probabilities 0): the caller then runs the plain kernels.
int drop_view(const vrr_drop_desc* d, int M, int E, DropView* v, bool* active);

// ---- logit bias evaluated on the fly -------------------------------------------------------------
// Device-side view of vrr_bias_desc for one head.  `lut` lives in shared memory:
//   TABLE: the head's table row, lut[i - j + N - 1]
//   POLY : lut[d] = sum_k coef[k] * d^k for d in [0, 2g-2] (power-sum order of the reference,
//          models/positional_encoding.py:145-148), 0 on the cls row/column.
struct BiasView {
  int mode, n, grid;
  const float* lut;
  __device__ __forceinline__ int index(int i, int j) const {
    if (mode == VRR_BIAS_TABLE) return i - j + n - 1;
    // POLY; caller guarantees i, j >= 1
    int pi = i - 1, pj = j - 1;
    int yi = pi % grid, xi = pi / grid, yj = pj % grid, xj = pj / grid;
    return abs(yi - yj) + abs(xi - xj);
  }
  __device__ __forceinline__ float at(int i, int j) const {
    if (mode == VRR_BIAS_NONE) return 0.f;
    if (mode == VRR_BIAS_POLY && (i == 0 || j == 0)) return 0.f;
    return lut[index(i, j)];
  }
};

// Number of LUT entries a CTA keeps in shared memory for one head.
static inline int bias_lut_len(const vrr_bias_desc* b, int n) {
  if (!b || b->mode == VRR_BIAS_NONE) return 0;
  if (b->mode == VRR_BIAS_TABLE) return 2 * n - 1;
  return 2 * b->grid - 1;
}

// Fill the per-head LUT (all threads of the CTA participate; caller syncs afterwards).
__device__ __forceinline__ void fill_bias_lut(float* lut, int mode, const float* param, int heads,
                                              int len, int grid, int n, int h) {
  if (mode == VRR_BIAS_TABLE) {
    const float* row = param + (size_t)h * len;
    for (int t = threadIdx.x; t < 2 * n - 1; t += blockDim.x) lut[t] = row[t];
  } else if (mode == VRR_BIAS_POLY) {
    const float* c = param + (size_t)(heads == 1 ? 0 : h) * len;
    for (int d = threadIdx.x; d < 2 * grid - 1; d += blockDim.x) {
      float x = (float)d, pw = 1.f, acc = 0.f;
      for (int k = 0; k < len; ++k) {
        acc = fmaf(pw, c[k], acc);
        pw *= x;
      }
      lut[d] = acc;
    }
  }
}

}  // namespace vrr
