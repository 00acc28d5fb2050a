// RoPE rotate-half kernels that are not GEMM epilogues:
//   * backward of the fused QKV+RoPE epilogue: un-rotate the plane gradients into the token
//     layout [B*N][3E] the two projection-backward GEMMs consume, and reduce d_cos / d_sin over
//     the batch (autograd of models/rope_utils.py:22-35 and of the cat/split at vit.py:56-68);
//   * the stand-alone public apply_rotary_emb (models/rope_utils.py:3-37).
#include "common.cuh"
#include "kernels.h"

namespace vrr {

// One thread = VEC consecutive channels dd..dd+VEC-1 of the first half (and their partners dd+Dh/2..)
// of one (head, token), looping over a chunk of the batch: 16-byte loads/stores throughout.
template <typename T, int VEC>
struct VecIO;
template <>
struct VecIO<float, 4> {
  using Raw = float4;
  static __device__ __forceinline__ void cvt(const float4& x, float (&v)[4]) {
    v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w;
  }
  static __device__ __forceinline__ void ld(const float* p, float (&v)[4]) {
    cvt(*reinterpret_cast<const float4*>(p), v);
  }
  static __device__ __forceinline__ void st(float* p, const float (&v)[4]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  }
};
template <>
struct VecIO<__nv_bfloat16, 8> {
  using Raw = uint4;
  static __device__ __forceinline__ void cvt(const uint4& x, float (&v)[8]) {
    const uint32_t w[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[e]));
      v[2 * e] = f.x; v[2 * e + 1] = f.y;
    }
  }
  static __device__ __forceinline__ void ld(const __nv_bfloat16* p, float (&v)[8]) {
    cvt(*reinterpret_cast<const uint4*>(p), v);
  }
  static __device__ __forceinline__ void st(__nv_bfloat16* p, const float (&v)[8]) {
    uint4 x;
    __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]), b = __floats2bfloat162_rn(v[2], v[3]);
    __nv_bfloat162 c = __floats2bfloat162_rn(v[4], v[5]), d = __floats2bfloat162_rn(v[6], v[7]);
    x.x = *reinterpret_cast<uint32_t*>(&a); x.y = *reinterpret_cast<uint32_t*>(&b);
    x.z = *reinterpret_cast<uint32_t*>(&c); x.w = *reinterpret_cast<uint32_t*>(&d);
    *reinterpret_cast<uint4*>(p) = x;
  }
};
template <>
struct VecIO<__half, 8> {
  using Raw = uint4;
  static __device__ __forceinline__ void cvt(const uint4& x, float (&v)[8]) {
    const uint32_t w[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[e]));
      v[2 * e] = f.x; v[2 * e + 1] = f.y;
    }
  }
  static __device__ __forceinline__ void ld(const __half* p, float (&v)[8]) {
    cvt(*reinterpret_cast<const uint4*>(p), v);
  }
  static __device__ __forceinline__ void st(__half* p, const float (&v)[8]) {
    uint4 x;
    __half2 a = __floats2half2_rn(v[0], v[1]), b = __floats2half2_rn(v[2], v[3]);
    __half2 c = __floats2half2_rn(v[4], v[5]), d = __floats2half2_rn(v[6], v[7]);
    x.x = *reinterpret_cast<uint32_t*>(&a); x.y = *reinterpret_cast<uint32_t*>(&b);
    x.z = *reinterpret_cast<uint32_t*>(&c); x.w = *reinterpret_cast<uint32_t*>(&d);
    *reinterpret_cast<uint4*>(p) = x;
  }
};

// NORM (vrr_qkv_rope_norm_bwd): `planes` is qk_pre [2][B][H][N][Dh] (x, the q / k rows before the norm) and the
// LayerNorm backward of each q / k row follows the un-rotation: with dy the un-rotated row, xhat = (x - mean) rstd,
//   d_qkv = T(rstd (g dy - mean(g dy) - xhat mean(g dy xhat))),  d_g += dy xhat,  d_b += dy,
// and d_cos / d_sin take y = xhat g + b (recomputed as the forward formed it) for the un-rotated value.  The two row
// means are an nv-lane shuffle (the nv threads of a row are adjacent lanes of one warp).  d_g / d_b: per-thread sums
// over its images, then reduced over the warp (lanes with the same channels) and the block (shared memory) before
// one fp32 atomic per column per block: 4 Dh x gridDim.x x gridDim.y atomics per launch.  No thread returns early:
// the block reduction needs them all.
struct NormBwdView {
  const float2* stats;  // [2][B][H][N] {mean, rstd}
  const float* w[2];    // q_norm / k_norm weight, bias [Dh]
  const float* b[2];
  float* dw[2];         // [Dh] each, zeroed; NULL: no parameter gradients
  float* db[2];
};

template <typename T, int VEC, bool NORM>
__global__ void qkv_rope_bwd_kernel(const T* __restrict__ d_planes, const T* __restrict__ planes,
                                    const float* __restrict__ cos_tab, const float* __restrict__ sin_tab,
                                    T* __restrict__ d_qkv, float* d_cos, float* d_sin, int B, int N,
                                    int E, int H, int Dh, int npre, int rope_mode, int b_chunk, const NormBwdView nb) {
  const int hd = Dh >> 1, nv = hd / VEC;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if constexpr (!NORM) {
    if (idx >= H * N * nv) return;
  }
  const bool live = idx < H * N * nv;
  const int dd = (idx % nv) * VEC, t = (idx / nv) % N, h = idx / (nv * N);
  const int b0 = blockIdx.y * b_chunk, b1 = (NORM && !live) ? b0 : min(B, b0 + b_chunk);
  const size_t plane = (size_t)B * H * N * Dh;
  const bool rot = rope_mode != VRR_ROPE_NONE && t >= npre && (!NORM || live);  // prefix rows (cls, registers) are never rotated
  float c[VEC], s[VEC], acc_c[VEC], acc_s[VEC];
  size_t tab = 0;
#pragma unroll
  for (int e = 0; e < VEC; ++e) { c[e] = 1.f; s[e] = 0.f; acc_c[e] = 0.f; acc_s[e] = 0.f; }
  if (rot) {
    tab = ((size_t)(rope_mode == VRR_ROPE_MIXED ? h * (N - npre) : 0) + (t - npre)) * hd + dd;
#pragma unroll
    for (int e = 0; e < VEC; ++e) { c[e] = cos_tab[tab + e]; s[e] = sin_tab[tab + e]; }
  }
  const bool want_cs = rot && d_cos != nullptr;
  // All ten 16-byte loads of one image are issued before the first use (raw, converted when consumed): with the
  // loads interleaved with the stores a thread had 32 bytes in flight and the kernel ran at a third of the HBM rate.
  using Raw = typename VecIO<T, VEC>::Raw;
  [[maybe_unused]] float pg[2][2 * VEC], pb[2][2 * VEC];  // NORM: this thread's d_g / d_b of channels dd.., hd + dd..
  if constexpr (NORM) {
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int e = 0; e < 2 * VEC; ++e) { pg[i][e] = 0.f; pb[i][e] = 0.f; }
  }
  for (int b = b0; b < b1; ++b) {
    const size_t src = (((size_t)b * H + h) * N + t) * Dh + dd;
    T* dst = d_qkv + ((size_t)b * N + t) * (3 * E) + h * Dh + dd;
    Raw rg[3][2], rx[2][2];
    [[maybe_unused]] float2 st[2];
#pragma unroll
    for (int which = 0; which < 3; ++which) {
      rg[which][0] = *reinterpret_cast<const Raw*>(d_planes + which * plane + src);
      rg[which][1] = *reinterpret_cast<const Raw*>(d_planes + which * plane + src + hd);
    }
    if (NORM || want_cs) {
#pragma unroll
      for (int which = 0; which < 2; ++which) {
        rx[which][0] = *reinterpret_cast<const Raw*>(planes + which * plane + src);
        rx[which][1] = *reinterpret_cast<const Raw*>(planes + which * plane + src + hd);
      }
    }
    if constexpr (NORM) {
#pragma unroll
      for (int which = 0; which < 2; ++which) st[which] = nb.stats[(((size_t)which * B + b) * H + h) * N + t];
    }
#pragma unroll
    for (int which = 0; which < 2; ++which) {
      float g1[VEC], g2[VEC], o1[VEC], o2[VEC];
      VecIO<T, VEC>::cvt(rg[which][0], g1);
      VecIO<T, VEC>::cvt(rg[which][1], g2);
#pragma unroll
      for (int e = 0; e < VEC; ++e) {
        o1[e] = g1[e] * c[e] + g2[e] * s[e];
        o2[e] = g2[e] * c[e] - g1[e] * s[e];
      }
      if constexpr (NORM) {
        // o = dy; x -> xhat; the two row sums over the Dh channels of the nv adjacent lanes
        float x1[VEC], x2[VEC], w1[VEC], w2[VEC];
        VecIO<T, VEC>::cvt(rx[which][0], x1);
        VecIO<T, VEC>::cvt(rx[which][1], x2);
        const float* wp = nb.w[which] + dd;
#pragma unroll
        for (int e = 0; e < VEC; ++e) { w1[e] = __ldg(wp + e); w2[e] = __ldg(wp + hd + e); }
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
          x1[e] = qk_norm_xhat(x1[e], st[which].x, st[which].y);
          x2[e] = qk_norm_xhat(x2[e], st[which].x, st[which].y);
          const float a1 = w1[e] * o1[e], a2 = w2[e] * o2[e];
          s1 += a1 + a2;
          s2 += a1 * x1[e] + a2 * x2[e];
        }
        const unsigned gmask = (0xFFFFFFFFu >> (32 - nv)) << ((threadIdx.x & 31) & ~(nv - 1));
        for (int o = 1; o < nv; o <<= 1) {
          s1 += __shfl_xor_sync(gmask, s1, o);
          s2 += __shfl_xor_sync(gmask, s2, o);
        }
        const float inv = 1.f / (float)Dh, m1 = s1 * inv, m2 = s2 * inv;
        float d1[VEC], d2[VEC];
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
          d1[e] = st[which].y * (w1[e] * o1[e] - m1 - x1[e] * m2);
          d2[e] = st[which].y * (w2[e] * o2[e] - m1 - x2[e] * m2);
          pg[which][e] += o1[e] * x1[e];
          pg[which][VEC + e] += o2[e] * x2[e];
          pb[which][e] += o1[e];
          pb[which][VEC + e] += o2[e];
        }
        VecIO<T, VEC>::st(dst + which * E, d1);
        VecIO<T, VEC>::st(dst + which * E + hd, d2);
        if (want_cs) {
          const float* bp = nb.b[which] + dd;
#pragma unroll
          for (int e = 0; e < VEC; ++e) {
            const float y1 = qk_norm_y(x1[e], w1[e], __ldg(bp + e)), y2 = qk_norm_y(x2[e], w2[e], __ldg(bp + hd + e));
            acc_c[e] += g1[e] * y1 + g2[e] * y2;
            acc_s[e] += g2[e] * y1 - g1[e] * y2;
          }
        }
      } else {
        VecIO<T, VEC>::st(dst + which * E, o1);
        VecIO<T, VEC>::st(dst + which * E + hd, o2);
        if (want_cs) {
          float r1[VEC], r2[VEC];
          VecIO<T, VEC>::cvt(rx[which][0], r1);
          VecIO<T, VEC>::cvt(rx[which][1], r2);
#pragma unroll
          for (int e = 0; e < VEC; ++e) {
            const float x1 = r1[e] * c[e] + r2[e] * s[e], x2 = r2[e] * c[e] - r1[e] * s[e];  // un-rotated
            acc_c[e] += g1[e] * x1 + g2[e] * x2;
            acc_s[e] += g2[e] * x1 - g1[e] * x2;
          }
        }
      }
    }
    *reinterpret_cast<Raw*>(dst + 2 * E) = rg[2][0];
    *reinterpret_cast<Raw*>(dst + 2 * E + hd) = rg[2][1];
  }
  if (want_cs) {
#pragma unroll
    for (int e = 0; e < VEC; ++e) {
      atomicAdd(d_cos + tab + e, acc_c[e]);
      atomicAdd(d_sin + tab + e, acc_s[e]);
    }
  }
  if constexpr (NORM) {
    if (nb.dw[0] == nullptr) return;  // uniform over the launch
    __shared__ float red[4][64];      // [q_w, q_b, k_w, k_b][channel], Dh <= 64
    for (int i = threadIdx.x; i < 4 * 64; i += blockDim.x) red[i >> 6][i & 63] = 0.f;
    __syncthreads();
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int e = 0; e < 2 * VEC; ++e) {
        float vg = pg[i][e], vb = pb[i][e];
        for (int o = nv; o < 32; o <<= 1) {  // lanes l, l + nv, .. hold the same channels
          vg += __shfl_xor_sync(0xFFFFFFFFu, vg, o);
          vb += __shfl_xor_sync(0xFFFFFFFFu, vb, o);
        }
        if (lane < nv) {
          const int ch = (e < VEC ? 0 : hd) + dd + (e & (VEC - 1));
          atomicAdd(&red[2 * i][ch], vg);
          atomicAdd(&red[2 * i + 1][ch], vb);
        }
      }
    __syncthreads();
    for (int i = threadIdx.x; i < 4 * Dh; i += blockDim.x) {
      const int k = i / Dh, ch = i - k * Dh;
      float* out = (k & 1) ? nb.db[k >> 1] : nb.dw[k >> 1];
      atomicAdd(out + ch, red[k][ch]);
    }
  }
}

int qkv_rope_bwd(const void* d_planes, const void* planes, const float* cos_tab, const float* sin_tab,
                 void* d_qkv, float* d_cos, float* d_sin, int B, int N, int E, int H, int npre, int rope_mode,
                 int dtype, cudaStream_t st) {
  const int Dh = E / H, hd = Dh / 2;
  if (rope_mode == VRR_ROPE_NONE) d_cos = d_sin = nullptr;
  if (d_cos) {
    size_t n = (size_t)(rope_mode == VRR_ROPE_MIXED ? H : 1) * (N - npre) * hd * sizeof(float);
    if (reinterpret_cast<char*>(d_sin) == reinterpret_cast<char*>(d_cos) + n) {  // halves of one buffer: one memset node
      VRR_CUDA(cudaMemsetAsync(d_cos, 0, 2 * n, st));
    } else {
      VRR_CUDA(cudaMemsetAsync(d_cos, 0, n, st));
      VRR_CUDA(cudaMemsetAsync(d_sin, 0, n, st));
    }
  }
  const int vec = dtype == VRR_F32 ? 4 : 8;
  VRR_REQUIRE(hd % vec == 0, VRR_ERR_UNSUPPORTED, "qkv_rope_bwd: head dim %d too small for %d-wide access", Dh, vec);
  VRR_REQUIRE(((uintptr_t)d_planes & 15) == 0 && ((uintptr_t)planes & 15) == 0 && ((uintptr_t)d_qkv & 15) == 0,
              VRR_ERR_INVALID_ARG, "qkv_rope_bwd: pointers must be 16-byte aligned");
  const int threads = 128, blocks = ceil_div(H * N * (hd / vec), threads);
  int chunks = 1;
  while (chunks < B && blocks * chunks < 8 * sm_count()) chunks *= 2;
  const int b_chunk = ceil_div(B, chunks);
  dim3 grid(blocks, ceil_div(B, b_chunk));
  const NormBwdView nb = {};
  if (dtype == VRR_F32)
    qkv_rope_bwd_kernel<float, 4, false><<<grid, threads, 0, st>>>((const float*)d_planes, (const float*)planes, cos_tab,
                                                                  sin_tab, (float*)d_qkv, d_cos, d_sin, B, N, E, H, Dh,
                                                                  npre, rope_mode, b_chunk, nb);
  else if (dtype == VRR_BF16)
    qkv_rope_bwd_kernel<__nv_bfloat16, 8, false><<<grid, threads, 0, st>>>(
        (const __nv_bfloat16*)d_planes, (const __nv_bfloat16*)planes, cos_tab, sin_tab,
        (__nv_bfloat16*)d_qkv, d_cos, d_sin, B, N, E, H, Dh, npre, rope_mode, b_chunk, nb);
  else
    qkv_rope_bwd_kernel<__half, 8, false><<<grid, threads, 0, st>>>((const __half*)d_planes, (const __half*)planes, cos_tab,
                                                                   sin_tab, (__half*)d_qkv, d_cos, d_sin, B, N, E, H, Dh,
                                                                   npre, rope_mode, b_chunk, nb);
  VRR_LAUNCHED();
  return VRR_OK;
}

int qkv_rope_norm_bwd(const void* d_planes, const QkNormArgs& qn, const float* cos_tab, const float* sin_tab, void* d_qkv,
                      float* d_cos, float* d_sin, const QkNormGrads& gr, int B, int N, int E, int H, int npre, int rope_mode,
                      int dtype, cudaStream_t st) {
  const int Dh = E / H, hd = Dh / 2;
  if (rope_mode == VRR_ROPE_NONE) d_cos = d_sin = nullptr;
  if (d_cos) {
    size_t n = (size_t)(rope_mode == VRR_ROPE_MIXED ? H : 1) * (N - npre) * hd * sizeof(float);
    if (reinterpret_cast<char*>(d_sin) == reinterpret_cast<char*>(d_cos) + n) {
      VRR_CUDA(cudaMemsetAsync(d_cos, 0, 2 * n, st));
    } else {
      VRR_CUDA(cudaMemsetAsync(d_cos, 0, n, st));
      VRR_CUDA(cudaMemsetAsync(d_sin, 0, n, st));
    }
  }
  if (gr.d_qn_w) {
    const size_t n = (size_t)Dh * sizeof(float);
    if (gr.d_qn_b == gr.d_qn_w + Dh && gr.d_kn_w == gr.d_qn_w + 2 * Dh && gr.d_kn_b == gr.d_qn_w + 3 * Dh) {  // one buffer
      VRR_CUDA(cudaMemsetAsync(gr.d_qn_w, 0, 4 * n, st));
    } else {
      for (float* p : {gr.d_qn_w, gr.d_qn_b, gr.d_kn_w, gr.d_kn_b}) VRR_CUDA(cudaMemsetAsync(p, 0, n, st));
    }
  }
  const int vec = dtype == VRR_F32 ? 4 : 8;
  VRR_REQUIRE(hd % vec == 0 && Dh <= 64, VRR_ERR_UNSUPPORTED, "qkv_rope_norm_bwd: head dim %d unsupported for %d-wide access",
              Dh, vec);
  VRR_REQUIRE(((uintptr_t)d_planes & 15) == 0 && ((uintptr_t)qn.qk_pre & 15) == 0 && ((uintptr_t)d_qkv & 15) == 0 &&
                  ((uintptr_t)qn.qk_stats & 7) == 0,
              VRR_ERR_INVALID_ARG, "qkv_rope_norm_bwd: pointers must be 16-byte aligned (qk_stats 8)");
  const int threads = 128, blocks = ceil_div(H * N * (hd / vec), threads);
  int chunks = 1;
  while (chunks < B && blocks * chunks < 8 * sm_count()) chunks *= 2;
  const int b_chunk = ceil_div(B, chunks);
  dim3 grid(blocks, ceil_div(B, b_chunk));
  const NormBwdView nb = {reinterpret_cast<const float2*>(qn.qk_stats), {qn.qn_w, qn.kn_w}, {qn.qn_b, qn.kn_b},
                          {gr.d_qn_w, gr.d_kn_w}, {gr.d_qn_b, gr.d_kn_b}};
  if (dtype == VRR_F32)
    qkv_rope_bwd_kernel<float, 4, true><<<grid, threads, 0, st>>>((const float*)d_planes, (const float*)qn.qk_pre, cos_tab,
                                                                 sin_tab, (float*)d_qkv, d_cos, d_sin, B, N, E, H, Dh, npre,
                                                                 rope_mode, b_chunk, nb);
  else if (dtype == VRR_BF16)
    qkv_rope_bwd_kernel<__nv_bfloat16, 8, true><<<grid, threads, 0, st>>>(
        (const __nv_bfloat16*)d_planes, (const __nv_bfloat16*)qn.qk_pre, cos_tab, sin_tab, (__nv_bfloat16*)d_qkv, d_cos,
        d_sin, B, N, E, H, Dh, npre, rope_mode, b_chunk, nb);
  else
    qkv_rope_bwd_kernel<__half, 8, true><<<grid, threads, 0, st>>>((const __half*)d_planes, (const __half*)qn.qk_pre, cos_tab,
                                                                  sin_tab, (__half*)d_qkv, d_cos, d_sin, B, N, E, H, Dh, npre,
                                                                  rope_mode, b_chunk, nb);
  VRR_LAUNCHED();
  return VRR_OK;
}

// cos / sin tables [heads][rows][hd] -> packed[heads][hd / 2][rows] of float4 {cos[2q], sin[2q], cos[2q+1], sin[2q+1]}:
// the layout the QKV GEMM epilogue reads.  There a LANE is a token row, so with the row-major tables one 16-byte load
// instruction touched 32 different 128-byte lines (the table row of every lane) and the L1 tag stage, not the math,
// set the epilogue's pace (ViT-B: 189 us with rope-mixed against 131 us without rotation); with rows innermost a
// load instruction covers 512 contiguous bytes.
__global__ void rope_pack_tables_kernel(const float* __restrict__ cos_tab, const float* __restrict__ sin_tab,
                                        float4* __restrict__ packed, int heads, int rows, int hd) {
  const int quads = hd >> 1;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= heads * quads * rows) return;
  const int t = idx % rows, q = (idx / rows) % quads, h = idx / (rows * quads);
  const size_t src = ((size_t)h * rows + t) * hd + 2 * q;
  packed[idx] = make_float4(cos_tab[src], sin_tab[src], cos_tab[src + 1], sin_tab[src + 1]);
}

int rope_pack_tables(const float* cos_tab, const float* sin_tab, float* packed, int heads, int rows, int hd, cudaStream_t st) {
  VRR_REQUIRE(hd % 2 == 0 && ((uintptr_t)packed & 15) == 0, VRR_ERR_INVALID_ARG,
              "rope_pack_tables: half head dim must be even and `packed` 16-byte aligned");
  const int total = heads * (hd / 2) * rows;
  rope_pack_tables_kernel<<<ceil_div(total, 256), 256, 0, st>>>(cos_tab, sin_tab, reinterpret_cast<float4*>(packed), heads, rows, hd);
  VRR_LAUNCHED();
  return VRR_OK;
}

template <typename T>
__global__ void rope_apply_kernel(const T* __restrict__ q_in, const T* __restrict__ k_in,
                                  const float* __restrict__ cos_tab, const float* __restrict__ sin_tab,
                                  T* __restrict__ q_out, T* __restrict__ k_out, int B, int H, int Nr,
                                  int Dh, int rope_mode, int inverse) {
  const int hd = Dh >> 1;
  const size_t total = (size_t)B * H * Nr * hd;
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int dd = idx % hd;
  const size_t row = idx / hd;  // (b*H + h)*Nr + t
  const int t = row % Nr, h = (row / Nr) % H;
  const size_t tab = ((size_t)(rope_mode == VRR_ROPE_MIXED ? h * Nr : 0) + t) * hd + dd;
  const float c = cos_tab[tab], s = inverse ? -sin_tab[tab] : sin_tab[tab];
  const size_t o = row * Dh + dd;
  const float q1 = Elem<T>::ld(q_in + o), q2 = Elem<T>::ld(q_in + o + hd);
  const float k1 = Elem<T>::ld(k_in + o), k2 = Elem<T>::ld(k_in + o + hd);
  Elem<T>::st(q_out + o, q1 * c - q2 * s);
  Elem<T>::st(q_out + o + hd, q1 * s + q2 * c);
  Elem<T>::st(k_out + o, k1 * c - k2 * s);
  Elem<T>::st(k_out + o + hd, k1 * s + k2 * c);
}

int rope_apply(const void* q_in, const void* k_in, const float* cos_tab, const float* sin_tab,
               void* q_out, void* k_out, int B, int H, int Nr, int Dh, int rope_mode, int inverse,
               int dtype, cudaStream_t st) {
  const size_t total = (size_t)B * H * Nr * (Dh / 2);
  const int threads = 256;
  const unsigned blocks = (unsigned)((total + threads - 1) / threads);
  if (dtype == VRR_F32)
    rope_apply_kernel<float><<<blocks, threads, 0, st>>>((const float*)q_in, (const float*)k_in, cos_tab, sin_tab,
                                                        (float*)q_out, (float*)k_out, B, H, Nr, Dh, rope_mode, inverse);
  else if (dtype == VRR_BF16)
    rope_apply_kernel<__nv_bfloat16><<<blocks, threads, 0, st>>>(
        (const __nv_bfloat16*)q_in, (const __nv_bfloat16*)k_in, cos_tab, sin_tab, (__nv_bfloat16*)q_out,
        (__nv_bfloat16*)k_out, B, H, Nr, Dh, rope_mode, inverse);
  else
    rope_apply_kernel<__half><<<blocks, threads, 0, st>>>((const __half*)q_in, (const __half*)k_in, cos_tab, sin_tab,
                                                         (__half*)q_out, (__half*)k_out, B, H, Nr, Dh, rope_mode, inverse);
  VRR_LAUNCHED();
  return VRR_OK;
}

// Gradient of the stand-alone rotate-half w.r.t. its tables: d_cos = sum (g1 x1 + g2 x2),
// d_sin = sum (g2 x1 - g1 x2) over q and k, over the batch (and over heads for the head-shared axial
// table).  One thread per table entry, a plain loop over what it sums: deterministic, no atomics.
template <typename T>
__global__ void rope_table_grad_kernel(const T* __restrict__ q_in, const T* __restrict__ k_in,
                                       const T* __restrict__ dq, const T* __restrict__ dk, float* __restrict__ d_cos,
                                       float* __restrict__ d_sin, int B, int H, int Nr, int Dh, int rope_mode) {
  const int hd = Dh >> 1;
  const int heads_tab = rope_mode == VRR_ROPE_MIXED ? H : 1;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= heads_tab * Nr * hd) return;
  const int dd = idx % hd, t = (idx / hd) % Nr, ht = idx / (hd * Nr);
  const int h0 = rope_mode == VRR_ROPE_MIXED ? ht : 0, h1 = rope_mode == VRR_ROPE_MIXED ? ht + 1 : H;
  float ac = 0.f, as = 0.f;
  for (int b = 0; b < B; ++b)
    for (int h = h0; h < h1; ++h) {
      const size_t o = (((size_t)b * H + h) * Nr + t) * Dh + dd;
      const float q1 = Elem<T>::ld(q_in + o), q2 = Elem<T>::ld(q_in + o + hd);
      const float k1 = Elem<T>::ld(k_in + o), k2 = Elem<T>::ld(k_in + o + hd);
      const float gq1 = Elem<T>::ld(dq + o), gq2 = Elem<T>::ld(dq + o + hd);
      const float gk1 = Elem<T>::ld(dk + o), gk2 = Elem<T>::ld(dk + o + hd);
      ac += gq1 * q1 + gq2 * q2 + gk1 * k1 + gk2 * k2;
      as += gq2 * q1 - gq1 * q2 + gk2 * k1 - gk1 * k2;
    }
  d_cos[idx] = ac;
  d_sin[idx] = as;
}

int rope_table_grad(const void* q_in, const void* k_in, const void* dq, const void* dk, float* d_cos, float* d_sin,
                    int B, int H, int Nr, int Dh, int rope_mode, int dtype, cudaStream_t st) {
  const int total = (rope_mode == VRR_ROPE_MIXED ? H : 1) * Nr * (Dh / 2);
  const int threads = 128, blocks = ceil_div(total, threads);
  if (dtype == VRR_F32)
    rope_table_grad_kernel<float><<<blocks, threads, 0, st>>>((const float*)q_in, (const float*)k_in, (const float*)dq,
                                                             (const float*)dk, d_cos, d_sin, B, H, Nr, Dh, rope_mode);
  else if (dtype == VRR_BF16)
    rope_table_grad_kernel<__nv_bfloat16><<<blocks, threads, 0, st>>>(
        (const __nv_bfloat16*)q_in, (const __nv_bfloat16*)k_in, (const __nv_bfloat16*)dq, (const __nv_bfloat16*)dk,
        d_cos, d_sin, B, H, Nr, Dh, rope_mode);
  else
    rope_table_grad_kernel<__half><<<blocks, threads, 0, st>>>((const __half*)q_in, (const __half*)k_in, (const __half*)dq,
                                                              (const __half*)dk, d_cos, d_sin, B, H, Nr, Dh, rope_mode);
  VRR_LAUNCHED();
  return VRR_OK;
}

}  // namespace vrr
