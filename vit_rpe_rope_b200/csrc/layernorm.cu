// LayerNorm forward / backward for the token stream (row N1 of SURVEY.md section 8(f): the first
// "next" component after the attention path).  Replaces nn.LayerNorm at models/vit.py:113,117,122,124,
// 210 of the reference: y = (x - mean) * rstd * gamma + beta over the last dimension, eps 1e-5.
//
// Why a kernel of our own: under autocast the reference's LayerNorm runs in fp32 and every consumer
// (qkv / fc1 GEMM) then casts its output to bf16 - two extra passes over [B*N, E]; and ATen's
// gamma/beta-gradient kernel alone was 14 % of the ViT-B/16 training step (profiles/r1_summary.md).
// Here the forward writes the consumer's dtype directly (same rounding point as the reference: fp32
// math, one rounding to bf16) and the backward produces dx, dgamma, dbeta in ONE pass over dy and x.
//
// One warp per row, rows grid-strided over a persistent grid; the row (<= a few KB) is re-read from
// L1 for the second pass instead of being held in registers, so any E works.  HBM-bound:
//   fwd  : read x, write y                      (E*(sx + sy) bytes per row)
//   bwd  : read dy, x, write dx                 (E*(sy + sx + sx) bytes per row)
#include "common.cuh"
#include "kernels.h"

namespace vrr {

namespace {

constexpr int kLnWarps = 8;
static int g_ln_bwd_minb = 3;  // register-resident add_ln_bwd at E >= 768: 3 = 12 warps x 1 CTA/SM (E = 768), 1 = 8 x 1, 2 = 8 x 2 (spills)
static int g_ln_reg = 1;       // 0: generic multi-pass kernels only (option "ln_reg")

// resident CTAs per SM the backward's shared-memory partials allow (`rows` x warps x E floats per CTA)
static inline int ln_bwd_ctas_per_sm(int E, int rows = 2) {
  const size_t per_cta = (size_t)rows * kLnWarps * E * sizeof(float) + 1024;
  int n = (int)((200 * 1024) / per_cta);
  return n < 1 ? 1 : (n > 6 ? 6 : n);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// DROP (add+LayerNorm): 0 plain; 1 stochastic depth only (one factor per row); 2 element masks (and stochastic depth).
// Factors of elements (m, n .. n + 3) / (m, n) given the row factor fr.
template <int DROP>
__device__ __forceinline__ float4 drop_f4(const DropView& dv, uint2 k, int m, int n, int E, float fr) {
  if constexpr (DROP == 1) return make_float4(fr, fr, fr, fr);
  else return dv.factor4(k, m, n, E, fr);
}
template <int DROP>
__device__ __forceinline__ float drop_f1(const DropView& dv, uint2 k, int m, int n, int E, float fr) {
  if constexpr (DROP == 1) return fr;
  else return dv.factor(k, m, n, E, fr);
}

// VEC = 4: E % 128 == 0, 16-byte (fp32) / 8-byte (bf16) accesses; VEC = 1: any E.
template <typename TX, typename TY, int VEC>
__global__ void __launch_bounds__(kLnWarps * 32)
ln_fwd_kernel(const TX* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
              TY* __restrict__ y, float* __restrict__ mean_out, float* __restrict__ rstd_out, int M, int E,
              float eps) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float inv_e = 1.f / (float)E;
  for (int row = blockIdx.x * kLnWarps + warp; row < M; row += gridDim.x * kLnWarps) {
    const TX* xr = x + (size_t)row * E;
    TY* yr = y + (size_t)row * E;
    float s = 0.f;
    if (VEC == 4) {
      for (int c = lane * 4; c < E; c += 128) {
        const float4 v = ld4(xr + c);
        s += (v.x + v.y) + (v.z + v.w);
      }
    } else {
      for (int c = lane; c < E; c += 32) s += Elem<TX>::ld(xr + c);
    }
    const float mean = warp_sum(s) * inv_e;
    float q = 0.f;
    if (VEC == 4) {
      for (int c = lane * 4; c < E; c += 128) {
        const float4 v = ld4(xr + c);
        const float a = v.x - mean, b = v.y - mean, cc = v.z - mean, d = v.w - mean;
        q += (a * a + b * b) + (cc * cc + d * d);
      }
    } else {
      for (int c = lane; c < E; c += 32) {
        const float a = Elem<TX>::ld(xr + c) - mean;
        q += a * a;
      }
    }
    const float rstd = rsqrtf(warp_sum(q) * inv_e + eps);
    if (VEC == 4) {
      for (int c = lane * 4; c < E; c += 128) {
        const float4 v = ld4(xr + c), g = ld4(gamma + c), b = ld4(beta + c);
        float4 o;
        o.x = (v.x - mean) * rstd * g.x + b.x;
        o.y = (v.y - mean) * rstd * g.y + b.y;
        o.z = (v.z - mean) * rstd * g.z + b.z;
        o.w = (v.w - mean) * rstd * g.w + b.w;
        st4(yr + c, o);
      }
    } else {
      for (int c = lane; c < E; c += 32)
        Elem<TY>::st(yr + c, (Elem<TX>::ld(xr + c) - mean) * rstd * gamma[c] + beta[c]);
    }
    if (lane == 0) {
      mean_out[row] = mean;
      rstd_out[row] = rstd;
    }
  }
}

// dx = rstd * (g*gamma - mean(g*gamma) - xhat * mean(g*gamma*xhat));  dgamma += g*xhat;  dbeta += g.
// Per-warp column partials live in shared memory ([warps][E] x 2); flushed with one atomicAdd per column
// per CTA at the end.
template <typename TX, typename TY, int VEC>
__global__ void __launch_bounds__(kLnWarps * 32)
ln_bwd_kernel(const TY* __restrict__ dy, const TX* __restrict__ x, const float* __restrict__ gamma,
              const float* __restrict__ mean_in, const float* __restrict__ rstd_in, TX* __restrict__ dx,
              float* __restrict__ dgamma, float* __restrict__ dbeta, int M, int E) {
  extern __shared__ __align__(16) float ln_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* pg = ln_smem + (size_t)warp * E;                      // this warp's dgamma partial
  float* pb = ln_smem + (size_t)(kLnWarps + warp) * E;         // this warp's dbeta partial
  for (int c = lane; c < E; c += 32) {
    pg[c] = 0.f;
    pb[c] = 0.f;
  }
  __syncwarp();
  const float inv_e = 1.f / (float)E;
  for (int row = blockIdx.x * kLnWarps + warp; row < M; row += gridDim.x * kLnWarps) {
    const TY* gr = dy + (size_t)row * E;
    const TX* xr = x + (size_t)row * E;
    TX* dr = dx + (size_t)row * E;
    const float mean = mean_in[row], rstd = rstd_in[row];
    float s1 = 0.f, s2 = 0.f;
    if (VEC == 4) {
      for (int c = lane * 4; c < E; c += 128) {
        const float4 g = ld4(gr + c), v = ld4(xr + c), w = ld4(gamma + c);
        const float gw[4] = {g.x * w.x, g.y * w.y, g.z * w.z, g.w * w.w};
        const float xh[4] = {(v.x - mean) * rstd, (v.y - mean) * rstd, (v.z - mean) * rstd, (v.w - mean) * rstd};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          s1 += gw[e];
          s2 = fmaf(gw[e], xh[e], s2);
        }
      }
    } else {
      for (int c = lane; c < E; c += 32) {
        const float gw = Elem<TY>::ld(gr + c) * gamma[c], xh = (Elem<TX>::ld(xr + c) - mean) * rstd;
        s1 += gw;
        s2 = fmaf(gw, xh, s2);
      }
    }
    const float c1 = warp_sum(s1) * inv_e, c2 = warp_sum(s2) * inv_e;
    if (VEC == 4) {
      for (int c = lane * 4; c < E; c += 128) {
        const float4 g = ld4(gr + c), v = ld4(xr + c), w = ld4(gamma + c);
        const float gv[4] = {g.x, g.y, g.z, g.w}, wv[4] = {w.x, w.y, w.z, w.w};
        const float xh[4] = {(v.x - mean) * rstd, (v.y - mean) * rstd, (v.z - mean) * rstd, (v.w - mean) * rstd};
        float o[4];
        float4 ag = *reinterpret_cast<float4*>(pg + c), ab = *reinterpret_cast<float4*>(pb + c);
        float agv[4] = {ag.x, ag.y, ag.z, ag.w}, abv[4] = {ab.x, ab.y, ab.z, ab.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          o[e] = rstd * (gv[e] * wv[e] - c1 - xh[e] * c2);
          agv[e] = fmaf(gv[e], xh[e], agv[e]);
          abv[e] += gv[e];
        }
        st4(dr + c, make_float4(o[0], o[1], o[2], o[3]));
        *reinterpret_cast<float4*>(pg + c) = make_float4(agv[0], agv[1], agv[2], agv[3]);
        *reinterpret_cast<float4*>(pb + c) = make_float4(abv[0], abv[1], abv[2], abv[3]);
      }
    } else {
      for (int c = lane; c < E; c += 32) {
        const float g = Elem<TY>::ld(gr + c), xh = (Elem<TX>::ld(xr + c) - mean) * rstd;
        Elem<TX>::st(dr + c, rstd * (g * gamma[c] - c1 - xh * c2));
        pg[c] = fmaf(g, xh, pg[c]);
        pb[c] += g;
      }
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < E; c += kLnWarps * 32) {
    float sg = 0.f, sb = 0.f;
#pragma unroll
    for (int w = 0; w < kLnWarps; ++w) {
      sg += ln_smem[(size_t)w * E + c];
      sb += ln_smem[(size_t)(kLnWarps + w) * E + c];
    }
    atomicAdd(dgamma + c, sg);
    atomicAdd(dbeta + c, sb);
  }
}

template <typename TX, typename TY>
int ln_fwd_t(const void* x, const float* gamma, const float* beta, void* y, float* mean, float* rstd, int M, int E,
             float eps, cudaStream_t st) {
  const int grid = min(ceil_div(M, kLnWarps), 8 * sm_count());
  if (E % 128 == 0)
    ln_fwd_kernel<TX, TY, 4><<<grid, kLnWarps * 32, 0, st>>>((const TX*)x, gamma, beta, (TY*)y, mean, rstd, M, E, eps);
  else
    ln_fwd_kernel<TX, TY, 1><<<grid, kLnWarps * 32, 0, st>>>((const TX*)x, gamma, beta, (TY*)y, mean, rstd, M, E, eps);
  VRR_LAUNCHED();
  return VRR_OK;
}

template <typename TX, typename TY, int VEC>
int ln_bwd_launch(const void* dy, const void* x, const float* gamma, const float* mean, const float* rstd, void* dx,
                  float* dgamma, float* dbeta, int M, int E, cudaStream_t st) {
  const size_t smem = (size_t)2 * kLnWarps * E * sizeof(float);
  auto kern = ln_bwd_kernel<TX, TY, VEC>;
  VRR_SMEM_ATTR_ONCE(kern, 160 * 1024);
  const int grid = min(ceil_div(M, kLnWarps), ln_bwd_ctas_per_sm(E) * sm_count());
  kern<<<grid, kLnWarps * 32, smem, st>>>((const TY*)dy, (const TX*)x, gamma, mean, rstd, (TX*)dx, dgamma, dbeta, M, E);
  VRR_LAUNCHED();
  return VRR_OK;
}

template <typename TX, typename TY>
int ln_bwd_t(const void* dy, const void* x, const float* gamma, const float* mean, const float* rstd, void* dx,
             float* dgamma, float* dbeta, int M, int E, cudaStream_t st) {
  if (dbeta == dgamma + E) {  // the two rows of one [2][E] buffer (what ops.py allocates): one memset node instead of two
    VRR_CUDA(cudaMemsetAsync(dgamma, 0, (size_t)2 * E * sizeof(float), st));
  } else {
    VRR_CUDA(cudaMemsetAsync(dgamma, 0, (size_t)E * sizeof(float), st));
    VRR_CUDA(cudaMemsetAsync(dbeta, 0, (size_t)E * sizeof(float), st));
  }
  if (E % 128 == 0) return ln_bwd_launch<TX, TY, 4>(dy, x, gamma, mean, rstd, dx, dgamma, dbeta, M, E, st);
  return ln_bwd_launch<TX, TY, 1>(dy, x, gamma, mean, rstd, dx, dgamma, dbeta, M, E, st);
}

// ---- fused residual add + LayerNorm (pre-LN transformer: x_new = x + branch; y = LN(x_new)) ----------
// forward : reads x (fp32) and branch, writes x_new (fp32) and y.
// backward: dx = d_xnew + LN'(dy) written as fp32 (gradient of the residual input) AND in the branch's
//           dtype (gradient of the branch: the same values) - the autograd add and the cast disappear.
// DROP != 0: the branch is multiplied by its dropout / stochastic-depth factor f (DropView) as it is read, in every pass.
// LS: then by the LayerScale vector ls[E], b' = fl(fl(f * branch) * ls[c]) (each product rounded, never contracted).
// The LS kernels declare one resident CTA per SM as the minimum (a minimum of 0 is no declaration, today's kernels):
// without it ptxas aims at a lower register count and spills a few bytes in some of them.
template <typename TB, typename TY, int VEC, int DROP, bool LS>
__global__ void __launch_bounds__(kLnWarps * 32, LS ? 1 : 0)
add_ln_fwd_kernel(const float* __restrict__ x, const TB* __restrict__ branch, float* __restrict__ x_new,
                  const float* __restrict__ gamma, const float* __restrict__ beta, TY* __restrict__ y,
                  float* __restrict__ mean_out, float* __restrict__ rstd_out, int M, int E, float eps, const DropView dv,
                  const float* __restrict__ ls) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float inv_e = 1.f / (float)E;
  [[maybe_unused]] uint2 key;
  if constexpr (DROP) key = dv.key();
  for (int row = blockIdx.x * kLnWarps + warp; row < M; row += gridDim.x * kLnWarps) {
    const float* xr = x + (size_t)row * E;
    const TB* br = branch + (size_t)row * E;
    float* nr = x_new + (size_t)row * E;
    TY* yr = y + (size_t)row * E;
    [[maybe_unused]] float fr = 1.f;
    if constexpr (DROP) fr = dv.row_factor(key, row);
    auto ldb4 = [&](int c) {
      float4 b = ld4(br + c);
      if constexpr (DROP) b = mul4_rn(b, drop_f4<DROP>(dv, key, row, c, E, fr));
      if constexpr (LS) b = mul4_rn(b, ld4(ls + c));
      return b;
    };
    auto ldb1 = [&](int c) {
      float b = Elem<TB>::ld(br + c);
      if constexpr (DROP) b = __fmul_rn(b, drop_f1<DROP>(dv, key, row, c, E, fr));
      if constexpr (LS) b = __fmul_rn(b, ls[c]);
      return b;
    };
    float s = 0.f;
    if (VEC == 4) {
      for (int c = lane * 4; c < E; c += 128) {
        const float4 a = ld4(xr + c), b = ldb4(c);
        const float4 v = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
        st4(nr + c, v);
        s += (v.x + v.y) + (v.z + v.w);
      }
    } else {
      for (int c = lane; c < E; c += 32) {
        const float v = xr[c] + ldb1(c);
        nr[c] = v;
        s += v;
      }
    }
    const float mean = warp_sum(s) * inv_e;
    float q = 0.f;
    if (VEC == 4) {
      for (int c = lane * 4; c < E; c += 128) {
        const float4 a = ld4(xr + c), b = ldb4(c);
        const float d0 = a.x + b.x - mean, d1 = a.y + b.y - mean, d2 = a.z + b.z - mean, d3 = a.w + b.w - mean;
        q += (d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3);
      }
    } else {
      for (int c = lane; c < E; c += 32) {
        const float d = xr[c] + ldb1(c) - mean;
        q += d * d;
      }
    }
    const float rstd = rsqrtf(warp_sum(q) * inv_e + eps);
    if (VEC == 4) {
      for (int c = lane * 4; c < E; c += 128) {
        const float4 a = ld4(xr + c), b = ldb4(c), g = ld4(gamma + c), bt = ld4(beta + c);
        float4 o;
        o.x = (a.x + b.x - mean) * rstd * g.x + bt.x;
        o.y = (a.y + b.y - mean) * rstd * g.y + bt.y;
        o.z = (a.z + b.z - mean) * rstd * g.z + bt.z;
        o.w = (a.w + b.w - mean) * rstd * g.w + bt.w;
        st4(yr + c, o);
      }
    } else {
      for (int c = lane; c < E; c += 32)
        Elem<TY>::st(yr + c, (xr[c] + ldb1(c) - mean) * rstd * gamma[c] + beta[c]);
    }
    if (lane == 0) {
      mean_out[row] = mean;
      rstd_out[row] = rstd;
    }
  }
}

// DROP != 0: d_branch = dx * f (the factor of the forward, regenerated)
// LS: d_branch = fl(fl(dx * f) * ls[c]); with d_ls, d_ls[c] = sum_rows fl(dx * f) * branch (a third [warps][E] partial)
template <typename TB, typename TY, int VEC, int DROP, bool LS>
__global__ void __launch_bounds__(kLnWarps * 32)
add_ln_bwd_kernel(const TY* __restrict__ dy, const float* __restrict__ d_xnew, const float* __restrict__ x_new,
                  const float* __restrict__ gamma, const float* __restrict__ mean_in,
                  const float* __restrict__ rstd_in, float* __restrict__ dx, TB* __restrict__ d_branch,
                  float* __restrict__ dgamma, float* __restrict__ dbeta, int M, int E, const DropView dv,
                  const float* __restrict__ ls, const TB* __restrict__ branch, float* __restrict__ d_ls) {
  extern __shared__ __align__(16) float ln_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* pg = ln_smem + (size_t)warp * E;
  float* pb = ln_smem + (size_t)(kLnWarps + warp) * E;
  [[maybe_unused]] float* pl = ln_smem + (size_t)(2 * kLnWarps + warp) * E;  // LS: this warp's d_ls partial
  for (int c = lane; c < E; c += 32) {
    pg[c] = 0.f;
    pb[c] = 0.f;
    if constexpr (LS) pl[c] = 0.f;
  }
  __syncwarp();
  const float inv_e = 1.f / (float)E;
  [[maybe_unused]] uint2 key;
  if constexpr (DROP) key = dv.key();
  for (int row = blockIdx.x * kLnWarps + warp; row < M; row += gridDim.x * kLnWarps) {
    const TY* gr = dy + (size_t)row * E;
    const float* xr = x_new + (size_t)row * E;
    const float* rr = d_xnew ? d_xnew + (size_t)row * E : nullptr;
    [[maybe_unused]] float fr = 1.f;
    if constexpr (DROP) fr = dv.row_factor(key, row);
    float* dr = dx + (size_t)row * E;
    TB* br = d_branch + (size_t)row * E;
    [[maybe_unused]] const TB* xb = LS && d_ls ? branch + (size_t)row * E : nullptr;
    const float mean = mean_in[row], rstd = rstd_in[row];
    float s1 = 0.f, s2 = 0.f;
    if (VEC == 4) {
      for (int c = lane * 4; c < E; c += 128) {
        const float4 g = ld4(gr + c), v = ld4(xr + c), w = ld4(gamma + c);
        const float gw[4] = {g.x * w.x, g.y * w.y, g.z * w.z, g.w * w.w};
        const float xh[4] = {(v.x - mean) * rstd, (v.y - mean) * rstd, (v.z - mean) * rstd, (v.w - mean) * rstd};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          s1 += gw[e];
          s2 = fmaf(gw[e], xh[e], s2);
        }
      }
    } else {
      for (int c = lane; c < E; c += 32) {
        const float gw = Elem<TY>::ld(gr + c) * gamma[c], xh = (xr[c] - mean) * rstd;
        s1 += gw;
        s2 = fmaf(gw, xh, s2);
      }
    }
    const float c1 = warp_sum(s1) * inv_e, c2 = warp_sum(s2) * inv_e;
    if (VEC == 4) {
      for (int c = lane * 4; c < E; c += 128) {
        const float4 g = ld4(gr + c), v = ld4(xr + c), w = ld4(gamma + c);
        const float4 r = rr ? ld4(rr + c) : make_float4(0.f, 0.f, 0.f, 0.f);
        const float gv[4] = {g.x, g.y, g.z, g.w}, wv[4] = {w.x, w.y, w.z, w.w}, rv[4] = {r.x, r.y, r.z, r.w};
        const float xh[4] = {(v.x - mean) * rstd, (v.y - mean) * rstd, (v.z - mean) * rstd, (v.w - mean) * rstd};
        float o[4];
        float4 ag = *reinterpret_cast<float4*>(pg + c), ab = *reinterpret_cast<float4*>(pb + c);
        float agv[4] = {ag.x, ag.y, ag.z, ag.w}, abv[4] = {ab.x, ab.y, ab.z, ab.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          o[e] = rv[e] + rstd * (gv[e] * wv[e] - c1 - xh[e] * c2);
          agv[e] = fmaf(gv[e], xh[e], agv[e]);
          abv[e] += gv[e];
        }
        const float4 ov = make_float4(o[0], o[1], o[2], o[3]);
        st4(dr + c, ov);
        float4 t = ov;
        if constexpr (DROP) t = mul4_rn(ov, drop_f4<DROP>(dv, key, row, c, E, fr));
        if constexpr (LS) {
          st4(br + c, mul4_rn(t, ld4(ls + c)));
          if (xb) {
            const float4 bv = ld4(xb + c);
            float4 al = *reinterpret_cast<float4*>(pl + c);
            al = make_float4(fmaf(t.x, bv.x, al.x), fmaf(t.y, bv.y, al.y), fmaf(t.z, bv.z, al.z), fmaf(t.w, bv.w, al.w));
            *reinterpret_cast<float4*>(pl + c) = al;
          }
        } else {
          st4(br + c, t);
        }
        *reinterpret_cast<float4*>(pg + c) = make_float4(agv[0], agv[1], agv[2], agv[3]);
        *reinterpret_cast<float4*>(pb + c) = make_float4(abv[0], abv[1], abv[2], abv[3]);
      }
    } else {
      for (int c = lane; c < E; c += 32) {
        const float g = Elem<TY>::ld(gr + c), xh = (xr[c] - mean) * rstd;
        const float o = (rr ? rr[c] : 0.f) + rstd * (g * gamma[c] - c1 - xh * c2);
        dr[c] = o;
        float t = o;
        if constexpr (DROP) t = __fmul_rn(o, drop_f1<DROP>(dv, key, row, c, E, fr));
        if constexpr (LS) {
          Elem<TB>::st(br + c, __fmul_rn(t, ls[c]));
          if (xb) pl[c] = fmaf(t, Elem<TB>::ld(xb + c), pl[c]);
        } else {
          Elem<TB>::st(br + c, t);
        }
        pg[c] = fmaf(g, xh, pg[c]);
        pb[c] += g;
      }
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < E; c += kLnWarps * 32) {
    float sg = 0.f, sb = 0.f;
#pragma unroll
    for (int w = 0; w < kLnWarps; ++w) {
      sg += ln_smem[(size_t)w * E + c];
      sb += ln_smem[(size_t)(kLnWarps + w) * E + c];
    }
    atomicAdd(dgamma + c, sg);
    atomicAdd(dbeta + c, sb);
    if constexpr (LS) {
      if (d_ls) {
        float sl = 0.f;
#pragma unroll
        for (int w = 0; w < kLnWarps; ++w) sl += ln_smem[(size_t)(2 * kLnWarps + w) * E + c];
        atomicAdd(d_ls + c, sl);
      }
    }
  }
}

// ---- register-resident rows (E = 128 NV, NV <= 8: ViT-B 768, ViT-L 1024) ---------------------------------------
// The generic kernels above re-read the row from L1 for every pass (three passes forward, two backward) and keep
// the gamma / beta gradient partials in shared memory with a read-modify-write per element and row: 99 / 138 us at
// ViT-B where the HBM floor is 71 / 95 us.  Here a lane keeps its NV float4 of the row in registers across the
// passes and its slice of the dgamma / dbeta partial sums in registers across ROWS (a lane owns the same columns
// for every row), touching shared memory once per CTA for the cross-warp reduction.  Same operation order per
// element as the generic kernels, so the results are bit-identical to them.
template <typename TB, typename TY, int NV, int DROP, bool LS>
__global__ void __launch_bounds__(kLnWarps * 32, LS ? 1 : 0)  // see add_ln_fwd_kernel
add_ln_fwd_reg_kernel(const float* __restrict__ x, const TB* __restrict__ branch, float* __restrict__ x_new,
                      const float* __restrict__ gamma, const float* __restrict__ beta, TY* __restrict__ y,
                      float* __restrict__ mean_out, float* __restrict__ rstd_out, int M, float eps, const DropView dv,
                      const float* __restrict__ ls) {
  constexpr int E = NV * 128;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float inv_e = 1.f / (float)E;
  float4 g[NV], bt[NV];
  [[maybe_unused]] float4 lsv[LS ? NV : 1];
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    g[i] = ld4(gamma + lane * 4 + i * 128);
    bt[i] = ld4(beta + lane * 4 + i * 128);
    if constexpr (LS) lsv[i] = ld4(ls + lane * 4 + i * 128);
  }
  [[maybe_unused]] uint2 key;
  if constexpr (DROP) key = dv.key();
  for (int row = blockIdx.x * kLnWarps + warp; row < M; row += gridDim.x * kLnWarps) {
    const float* xr = x + (size_t)row * E + lane * 4;
    const TB* br = branch + (size_t)row * E + lane * 4;
    float* nr = x_new + (size_t)row * E + lane * 4;
    TY* yr = y + (size_t)row * E + lane * 4;
    float4 v[NV];
    float s = 0.f;
    [[maybe_unused]] float fr = 1.f;
    if constexpr (DROP) fr = dv.row_factor(key, row);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const float4 a = ld4(xr + i * 128);
      float4 b = ld4(br + i * 128);
      if constexpr (DROP) b = mul4_rn(b, drop_f4<DROP>(dv, key, row, lane * 4 + i * 128, E, fr));
      if constexpr (LS) b = mul4_rn(b, lsv[i]);
      v[i] = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
    }
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      st4(nr + i * 128, v[i]);
      s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
    const float mean = warp_sum(s) * inv_e;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const float d0 = v[i].x - mean, d1 = v[i].y - mean, d2 = v[i].z - mean, d3 = v[i].w - mean;
      q += (d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3);
    }
    const float rstd = rsqrtf(warp_sum(q) * inv_e + eps);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      float4 o;
      o.x = (v[i].x - mean) * rstd * g[i].x + bt[i].x;
      o.y = (v[i].y - mean) * rstd * g[i].y + bt[i].y;
      o.z = (v[i].z - mean) * rstd * g[i].z + bt[i].z;
      o.w = (v[i].w - mean) * rstd * g[i].w + bt[i].w;
      st4(yr + i * 128, o);
    }
    if (lane == 0) {
      mean_out[row] = mean;
      rstd_out[row] = rstd;
    }
  }
}

// LS: the d_ls partial of a lane's columns accumulates in that lane's slots of the third [WARPS][E] shared row (no
// synchronisation: a lane owns the same columns for every row) - in registers it would not fit next to pg / pb at NV 8.
template <typename TB, typename TY, int NV, int WARPS, int MINB, int DROP, bool LS>
__global__ void __launch_bounds__(WARPS * 32, MINB)
add_ln_bwd_reg_kernel(const TY* __restrict__ dy, const float* __restrict__ d_xnew, const float* __restrict__ x_new,
                      const float* __restrict__ gamma, const float* __restrict__ mean_in, const float* __restrict__ rstd_in,
                      float* __restrict__ dx, TB* __restrict__ d_branch, float* __restrict__ dgamma,
                      float* __restrict__ dbeta, int M, const DropView dv, const float* __restrict__ ls,
                      const TB* __restrict__ branch, float* __restrict__ d_ls) {
  constexpr int E = NV * 128;
  extern __shared__ __align__(16) float ln_smem[];  // [2 (+1 LS)][WARPS][E]; pg / pb used once at the end
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float inv_e = 1.f / (float)E;
  float4 pg[NV], pb[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) pg[i] = pb[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  [[maybe_unused]] float* pl = ln_smem + (size_t)(2 * WARPS + warp) * E + lane * 4;
  if constexpr (LS) {
#pragma unroll
    for (int i = 0; i < NV; ++i) *reinterpret_cast<float4*>(pl + i * 128) = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  [[maybe_unused]] uint2 key;
  if constexpr (DROP) key = dv.key();
  for (int row = blockIdx.x * WARPS + warp; row < M; row += gridDim.x * WARPS) {
    const TY* gr = dy + (size_t)row * E + lane * 4;
    const float* xr = x_new + (size_t)row * E + lane * 4;
    const float* rr = d_xnew ? d_xnew + (size_t)row * E + lane * 4 : nullptr;
    float* dr = dx + (size_t)row * E + lane * 4;
    TB* br = d_branch + (size_t)row * E + lane * 4;
    [[maybe_unused]] const TB* xb = LS && d_ls ? branch + (size_t)row * E + lane * 4 : nullptr;
    const float mean = mean_in[row], rstd = rstd_in[row];
    float4 g[NV], xh[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      g[i] = ld4(gr + i * 128);
      xh[i] = ld4(xr + i * 128);
    }
    // the row's factor and (DROP == 2) keep bits (4 per float4), drawn while its loads are in flight: at one CTA of
    // 12 warps per SM the Philox rounds were exposed when they ran in the output loop
    [[maybe_unused]] float fr = 1.f;
    if constexpr (DROP) fr = dv.row_factor(key, row);
    [[maybe_unused]] uint32_t kb = 0;
    if constexpr (DROP == 2) {
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const float4 f = dv.factor4(key, row, lane * 4 + i * 128, E, 1.f);
        kb |= ((f.x != 0.f ? 1u : 0u) | (f.y != 0.f ? 2u : 0u) | (f.z != 0.f ? 4u : 0u) | (f.w != 0.f ? 8u : 0u)) << (4 * i);
      }
    }
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const float4 w = __ldg(reinterpret_cast<const float4*>(gamma + lane * 4 + i * 128));
      xh[i] = make_float4((xh[i].x - mean) * rstd, (xh[i].y - mean) * rstd, (xh[i].z - mean) * rstd, (xh[i].w - mean) * rstd);
      const float gw[4] = {g[i].x * w.x, g[i].y * w.y, g[i].z * w.z, g[i].w * w.w};
      const float xv[4] = {xh[i].x, xh[i].y, xh[i].z, xh[i].w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        s1 += gw[e];
        s2 = fmaf(gw[e], xv[e], s2);
      }
    }
    const float c1 = warp_sum(s1) * inv_e, c2 = warp_sum(s2) * inv_e;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const float4 w = __ldg(reinterpret_cast<const float4*>(gamma + lane * 4 + i * 128));
      const float4 r = rr ? ld4(rr + i * 128) : make_float4(0.f, 0.f, 0.f, 0.f);
      float4 o;
      o.x = r.x + rstd * (g[i].x * w.x - c1 - xh[i].x * c2);
      o.y = r.y + rstd * (g[i].y * w.y - c1 - xh[i].y * c2);
      o.z = r.z + rstd * (g[i].z * w.z - c1 - xh[i].z * c2);
      o.w = r.w + rstd * (g[i].w * w.w - c1 - xh[i].w * c2);
      st4(dr + i * 128, o);
      if constexpr (LS) {
        float4 t = o;
        if constexpr (DROP == 1) {
          t = mul4_rn(o, make_float4(fr, fr, fr, fr));
        } else if constexpr (DROP == 2) {
          const uint32_t b4 = kb >> (4 * i);
          t = mul4_rn(o, make_float4(b4 & 1u ? fr : 0.f, b4 & 2u ? fr : 0.f, b4 & 4u ? fr : 0.f, b4 & 8u ? fr : 0.f));
        }
        st4(br + i * 128, mul4_rn(t, __ldg(reinterpret_cast<const float4*>(ls + lane * 4 + i * 128))));
        if (xb) {
          const float4 bv = ld4(xb + i * 128);
          float4 al = *reinterpret_cast<float4*>(pl + i * 128);
          al = make_float4(fmaf(t.x, bv.x, al.x), fmaf(t.y, bv.y, al.y), fmaf(t.z, bv.z, al.z), fmaf(t.w, bv.w, al.w));
          *reinterpret_cast<float4*>(pl + i * 128) = al;
        }
      } else if constexpr (DROP == 1) {
        st4(br + i * 128, mul4_rn(o, make_float4(fr, fr, fr, fr)));
      } else if constexpr (DROP == 2) {
        const uint32_t b4 = kb >> (4 * i);
        st4(br + i * 128, mul4_rn(o, make_float4(b4 & 1u ? fr : 0.f, b4 & 2u ? fr : 0.f, b4 & 4u ? fr : 0.f, b4 & 8u ? fr : 0.f)));
      } else {
        st4(br + i * 128, o);
      }
      pg[i].x = fmaf(g[i].x, xh[i].x, pg[i].x);
      pg[i].y = fmaf(g[i].y, xh[i].y, pg[i].y);
      pg[i].z = fmaf(g[i].z, xh[i].z, pg[i].z);
      pg[i].w = fmaf(g[i].w, xh[i].w, pg[i].w);
      pb[i].x += g[i].x;
      pb[i].y += g[i].y;
      pb[i].z += g[i].z;
      pb[i].w += g[i].w;
    }
  }
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    *reinterpret_cast<float4*>(ln_smem + (size_t)warp * E + lane * 4 + i * 128) = pg[i];
    *reinterpret_cast<float4*>(ln_smem + (size_t)(WARPS + warp) * E + lane * 4 + i * 128) = pb[i];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < E; c += WARPS * 32) {
    float sg = 0.f, sb = 0.f;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) {
      sg += ln_smem[(size_t)w * E + c];
      sb += ln_smem[(size_t)(WARPS + w) * E + c];
    }
    atomicAdd(dgamma + c, sg);
    atomicAdd(dbeta + c, sb);
    if constexpr (LS) {
      if (d_ls) {
        float sl = 0.f;
#pragma unroll
        for (int w = 0; w < WARPS; ++w) sl += ln_smem[(size_t)(2 * WARPS + w) * E + c];
        atomicAdd(d_ls + c, sl);
      }
    }
  }
}

template <typename TB, typename TY, int DROP, bool LS>
int add_ln_fwd_t(const float* x, const void* branch, float* x_new, const float* gamma, const float* beta, void* y,
                 float* mean, float* rstd, int M, int E, float eps, const DropView& dv, const float* ls, cudaStream_t st) {
  const int grid = min(ceil_div(M, kLnWarps), 8 * sm_count());
#define VRR_LN_REG(NV)                                                                                                \
  if (g_ln_reg && E == NV * 128) { \
    const int g2 = min(ceil_div(M, kLnWarps), 4 * sm_count());                                                        \
    add_ln_fwd_reg_kernel<TB, TY, NV, DROP, LS><<<g2, kLnWarps * 32, 0, st>>>(x, (const TB*)branch, x_new, gamma,     \
                                                                              beta, (TY*)y, mean, rstd, M, eps, dv, ls); \
    VRR_LAUNCHED();                                                                                                   \
    return VRR_OK;                                                                                                    \
  }
  VRR_LN_REG(6) VRR_LN_REG(8) VRR_LN_REG(4) VRR_LN_REG(2)
#undef VRR_LN_REG
  if (E % 128 == 0)
    add_ln_fwd_kernel<TB, TY, 4, DROP, LS><<<grid, kLnWarps * 32, 0, st>>>(x, (const TB*)branch, x_new, gamma, beta, (TY*)y, mean, rstd, M, E, eps, dv, ls);
  else
    add_ln_fwd_kernel<TB, TY, 1, DROP, LS><<<grid, kLnWarps * 32, 0, st>>>(x, (const TB*)branch, x_new, gamma, beta, (TY*)y, mean, rstd, M, E, eps, dv, ls);
  VRR_LAUNCHED();
  return VRR_OK;
}

template <typename TB, typename TY, int VEC, int DROP, bool LS>
int add_ln_bwd_launch(const void* dy, const float* d_xnew, const float* x_new, const float* gamma, const float* mean,
                      const float* rstd, float* dx, void* d_branch, float* dgamma, float* dbeta, int M, int E,
                      const DropView& dv, const float* ls, const void* branch, float* d_ls, cudaStream_t st) {
  const size_t smem = (size_t)(LS ? 3 : 2) * kLnWarps * E * sizeof(float);
  auto kern = add_ln_bwd_kernel<TB, TY, VEC, DROP, LS>;
  VRR_SMEM_ATTR_ONCE(kern, 160 * 1024);
  const int grid = min(ceil_div(M, kLnWarps), ln_bwd_ctas_per_sm(E, LS ? 3 : 2) * sm_count());
  kern<<<grid, kLnWarps * 32, smem, st>>>((const TY*)dy, d_xnew, x_new, gamma, mean, rstd, dx, (TB*)d_branch, dgamma, dbeta, M, E, dv,
                                          ls, (const TB*)branch, d_ls);
  VRR_LAUNCHED();
  return VRR_OK;
}

template <typename TB, typename TY, int DROP, bool LS>
int add_ln_bwd_t(const void* dy, const float* d_xnew, const float* x_new, const float* gamma, const float* mean,
                 const float* rstd, float* dx, void* d_branch, float* dgamma, float* dbeta, int M, int E,
                 const DropView& dv, const float* ls, const void* branch, float* d_ls, cudaStream_t st) {
  // the rows of one [2][E] (or, with d_ls, [3][E]) buffer (what ops.py allocates): one memset node
  const bool three = d_ls && dbeta == dgamma + E && d_ls == dgamma + 2 * E;
  if (dbeta == dgamma + E) {
    VRR_CUDA(cudaMemsetAsync(dgamma, 0, (size_t)(three ? 3 : 2) * E * sizeof(float), st));
  } else {
    VRR_CUDA(cudaMemsetAsync(dgamma, 0, (size_t)E * sizeof(float), st));
    VRR_CUDA(cudaMemsetAsync(dbeta, 0, (size_t)E * sizeof(float), st));
  }
  if (d_ls && !three) VRR_CUDA(cudaMemsetAsync(d_ls, 0, (size_t)E * sizeof(float), st));
#define VRR_LN_BWD_GO(NV, W, B)                                                                                          \
  auto kern = add_ln_bwd_reg_kernel<TB, TY, NV, W, B, DROP, LS>;                                                       \
  VRR_SMEM_ATTR_ONCE(kern, 160 * 1024);                                                                                \
  const int grid = min(ceil_div(M, W), B * sm_count());                                                                \
  kern<<<grid, W * 32, (size_t)(LS ? 3 : 2) * W * E * sizeof(float), st>>>((const TY*)dy, d_xnew, x_new, gamma, mean,  \
                                                                           rstd, dx, (TB*)d_branch, dgamma, dbeta, M,   \
                                                                           dv, ls, (const TB*)branch, d_ls);
  // LS: its own launch shape, the one that compiles without spills for every dtype and DROP (12 x 1 spills at NV 6 with
  // an fp32 branch, 8 x 2 at NV >= 4); ln_bwd_minb does not apply
#define VRR_LN_REG(NV)                                                                                                  \
  if (g_ln_reg && E == NV * 128) { \
    if constexpr (LS) {                                                                                                 \
      if constexpr (NV <= 2) {                                                                                                  \
        VRR_LN_BWD_GO(NV, 8, 2)                                                                                         \
      } else {                                                                                                          \
        VRR_LN_BWD_GO(NV, 8, 1)                                                                                         \
      }                                                                                                                 \
    } else if (NV <= 4 || g_ln_bwd_minb == 2) {                                                                                \
      VRR_LN_BWD_GO(NV, 8, 2)                                                                                              \
    } else if (g_ln_bwd_minb == 1 || NV > 6) {                                                                               \
      VRR_LN_BWD_GO(NV, 8, 1)                                                                                              \
    } else {                                                                                                            \
      VRR_LN_BWD_GO(NV, 12, 1)                                                                                             \
    }                                                                                                                   \
    VRR_LAUNCHED();                                                                                                     \
    return VRR_OK;                                                                                                      \
  }
  VRR_LN_REG(6) VRR_LN_REG(8) VRR_LN_REG(4) VRR_LN_REG(2)
#undef VRR_LN_REG
  if (E % 128 == 0)
    return add_ln_bwd_launch<TB, TY, 4, DROP, LS>(dy, d_xnew, x_new, gamma, mean, rstd, dx, d_branch, dgamma, dbeta, M, E, dv,
                                                  ls, branch, d_ls, st);
  return add_ln_bwd_launch<TB, TY, 1, DROP, LS>(dy, d_xnew, x_new, gamma, mean, rstd, dx, d_branch, dgamma, dbeta, M, E, dv,
                                                ls, branch, d_ls, st);
}

}  // namespace

int layernorm_fwd(const void* x, const float* gamma, const float* beta, void* y, float* mean, float* rstd, int M, int E,
                  float eps, int x_dtype, int y_dtype, cudaStream_t st) {
  VRR_REQUIRE((size_t)2 * kLnWarps * E * sizeof(float) <= 160 * 1024, VRR_ERR_UNSUPPORTED,
              "layernorm: E = %d too large (max 2560)", E);
  if (x_dtype == VRR_F32 && y_dtype == VRR_F32) return ln_fwd_t<float, float>(x, gamma, beta, y, mean, rstd, M, E, eps, st);
  if (x_dtype == VRR_F32 && y_dtype == VRR_BF16) return ln_fwd_t<float, __nv_bfloat16>(x, gamma, beta, y, mean, rstd, M, E, eps, st);
  if (x_dtype == VRR_BF16 && y_dtype == VRR_BF16)
    return ln_fwd_t<__nv_bfloat16, __nv_bfloat16>(x, gamma, beta, y, mean, rstd, M, E, eps, st);
  if (x_dtype == VRR_F32 && y_dtype == VRR_F16) return ln_fwd_t<float, __half>(x, gamma, beta, y, mean, rstd, M, E, eps, st);
  if (x_dtype == VRR_F16 && y_dtype == VRR_F16) return ln_fwd_t<__half, __half>(x, gamma, beta, y, mean, rstd, M, E, eps, st);
  set_error("layernorm_fwd: unsupported dtype combination (x %d, y %d)", x_dtype, y_dtype);
  return VRR_ERR_UNSUPPORTED;
}

int layernorm_bwd(const void* dy, const void* x, const float* gamma, const float* mean, const float* rstd, void* dx,
                  float* dgamma, float* dbeta, int M, int E, int x_dtype, int y_dtype, cudaStream_t st) {
  VRR_REQUIRE((size_t)2 * kLnWarps * E * sizeof(float) <= 160 * 1024, VRR_ERR_UNSUPPORTED,
              "layernorm: E = %d too large (max 2560)", E);
  if (x_dtype == VRR_F32 && y_dtype == VRR_F32) return ln_bwd_t<float, float>(dy, x, gamma, mean, rstd, dx, dgamma, dbeta, M, E, st);
  if (x_dtype == VRR_F32 && y_dtype == VRR_BF16)
    return ln_bwd_t<float, __nv_bfloat16>(dy, x, gamma, mean, rstd, dx, dgamma, dbeta, M, E, st);
  if (x_dtype == VRR_BF16 && y_dtype == VRR_BF16)
    return ln_bwd_t<__nv_bfloat16, __nv_bfloat16>(dy, x, gamma, mean, rstd, dx, dgamma, dbeta, M, E, st);
  if (x_dtype == VRR_F32 && y_dtype == VRR_F16)
    return ln_bwd_t<float, __half>(dy, x, gamma, mean, rstd, dx, dgamma, dbeta, M, E, st);
  if (x_dtype == VRR_F16 && y_dtype == VRR_F16)
    return ln_bwd_t<__half, __half>(dy, x, gamma, mean, rstd, dx, dgamma, dbeta, M, E, st);
  set_error("layernorm_bwd: unsupported dtype combination (x %d, y %d)", x_dtype, y_dtype);
  return VRR_ERR_UNSUPPORTED;
}

template <int DROP, bool LS>
static int add_layernorm_fwd_d(const void* x, const void* branch, void* x_new, const float* gamma, const float* beta,
                               void* y, float* mean, float* rstd, int M, int E, float eps, int branch_dtype, int y_dtype,
                               const DropView& dv, const float* ls, cudaStream_t st) {
  VRR_REQUIRE((size_t)2 * kLnWarps * E * sizeof(float) <= 160 * 1024, VRR_ERR_UNSUPPORTED,
              "add_layernorm: E = %d too large (max 2560)", E);
#define ARGS (const float*)x, branch, (float*)x_new, gamma, beta, y, mean, rstd, M, E, eps, dv, ls, st
  if (branch_dtype == VRR_F32 && y_dtype == VRR_F32) return add_ln_fwd_t<float, float, DROP, LS>(ARGS);
  if (branch_dtype == VRR_BF16 && y_dtype == VRR_BF16) return add_ln_fwd_t<__nv_bfloat16, __nv_bfloat16, DROP, LS>(ARGS);
  if (branch_dtype == VRR_F32 && y_dtype == VRR_BF16) return add_ln_fwd_t<float, __nv_bfloat16, DROP, LS>(ARGS);
  if (branch_dtype == VRR_F16 && y_dtype == VRR_F16) return add_ln_fwd_t<__half, __half, DROP, LS>(ARGS);
  if (branch_dtype == VRR_F32 && y_dtype == VRR_F16) return add_ln_fwd_t<float, __half, DROP, LS>(ARGS);
#undef ARGS
  set_error("add_layernorm_fwd: unsupported dtype combination (branch %d, y %d)", branch_dtype, y_dtype);
  return VRR_ERR_UNSUPPORTED;
}

template <int DROP, bool LS>
static int add_layernorm_bwd_d(const void* dy, const void* d_xnew, const void* x_new, const float* gamma,
                               const float* mean, const float* rstd, void* dx, void* d_branch, float* dgamma,
                               float* dbeta, int M, int E, int branch_dtype, int y_dtype, const DropView& dv,
                               const float* ls, const void* branch, float* d_ls, cudaStream_t st) {
  VRR_REQUIRE((size_t)(LS ? 3 : 2) * kLnWarps * E * sizeof(float) <= 160 * 1024, VRR_ERR_UNSUPPORTED,
              "add_layernorm: E = %d too large (max %d)", E, LS ? 1706 : 2560);
#define ARGS dy, (const float*)d_xnew, (const float*)x_new, gamma, mean, rstd, (float*)dx, d_branch, dgamma, dbeta, M, E, dv, \
             ls, branch, d_ls, st
  if (branch_dtype == VRR_F32 && y_dtype == VRR_F32) return add_ln_bwd_t<float, float, DROP, LS>(ARGS);
  if (branch_dtype == VRR_BF16 && y_dtype == VRR_BF16) return add_ln_bwd_t<__nv_bfloat16, __nv_bfloat16, DROP, LS>(ARGS);
  if (branch_dtype == VRR_F32 && y_dtype == VRR_BF16) return add_ln_bwd_t<float, __nv_bfloat16, DROP, LS>(ARGS);
  if (branch_dtype == VRR_F16 && y_dtype == VRR_F16) return add_ln_bwd_t<__half, __half, DROP, LS>(ARGS);
  if (branch_dtype == VRR_F32 && y_dtype == VRR_F16) return add_ln_bwd_t<float, __half, DROP, LS>(ARGS);
#undef ARGS
  set_error("add_layernorm_bwd: unsupported dtype combination (branch %d, y %d)", branch_dtype, y_dtype);
  return VRR_ERR_UNSUPPORTED;
}

template <bool LS>
static int add_layernorm_fwd_l(const void* x, const void* branch, void* x_new, const float* gamma, const float* beta,
                               void* y, float* mean, float* rstd, int M, int E, float eps, int branch_dtype, int y_dtype,
                               const vrr_drop_desc* drop, const float* ls, cudaStream_t st) {
  DropView dv = {};
  bool active = false;
  if (int rc = drop_view(drop, M, E, &dv, &active)) return rc;
#define ARGS x, branch, x_new, gamma, beta, y, mean, rstd, M, E, eps, branch_dtype, y_dtype, dv, ls, st
  if (active && dv.t < 65536u) return add_layernorm_fwd_d<2, LS>(ARGS);
  if (active) return add_layernorm_fwd_d<1, LS>(ARGS);
  return add_layernorm_fwd_d<0, LS>(ARGS);
#undef ARGS
}

template <bool LS>
static int add_layernorm_bwd_l(const void* dy, const void* d_xnew, const void* x_new, const float* gamma,
                               const float* mean, const float* rstd, void* dx, void* d_branch, float* dgamma,
                               float* dbeta, int M, int E, int branch_dtype, int y_dtype, const vrr_drop_desc* drop,
                               const float* ls, const void* branch, float* d_ls, cudaStream_t st) {
  DropView dv = {};
  bool active = false;
  if (int rc = drop_view(drop, M, E, &dv, &active)) return rc;
#define ARGS dy, d_xnew, x_new, gamma, mean, rstd, dx, d_branch, dgamma, dbeta, M, E, branch_dtype, y_dtype, dv, ls, branch, d_ls, st
  if (active && dv.t < 65536u) return add_layernorm_bwd_d<2, LS>(ARGS);
  if (active) return add_layernorm_bwd_d<1, LS>(ARGS);
  return add_layernorm_bwd_d<0, LS>(ARGS);
#undef ARGS
}

int add_layernorm_fwd(const void* x, const void* branch, void* x_new, const float* gamma, const float* beta, void* y,
                      float* mean, float* rstd, int M, int E, float eps, int branch_dtype, int y_dtype,
                      const vrr_drop_desc* drop, const float* ls, cudaStream_t st) {
  if (ls)
    return add_layernorm_fwd_l<true>(x, branch, x_new, gamma, beta, y, mean, rstd, M, E, eps, branch_dtype, y_dtype, drop, ls, st);
  return add_layernorm_fwd_l<false>(x, branch, x_new, gamma, beta, y, mean, rstd, M, E, eps, branch_dtype, y_dtype, drop,
                                    nullptr, st);
}

int add_layernorm_bwd(const void* dy, const void* d_xnew, const void* x_new, const float* gamma, const float* mean,
                      const float* rstd, void* dx, void* d_branch, float* dgamma, float* dbeta, int M, int E,
                      int branch_dtype, int y_dtype, const vrr_drop_desc* drop, const float* ls, const void* branch,
                      float* d_ls, cudaStream_t st) {
  if (ls)
    return add_layernorm_bwd_l<true>(dy, d_xnew, x_new, gamma, mean, rstd, dx, d_branch, dgamma, dbeta, M, E, branch_dtype,
                                     y_dtype, drop, ls, branch, d_ls, st);
  return add_layernorm_bwd_l<false>(dy, d_xnew, x_new, gamma, mean, rstd, dx, d_branch, dgamma, dbeta, M, E, branch_dtype,
                                    y_dtype, drop, nullptr, nullptr, nullptr, st);
}

void layernorm_set_option(int which, int value) {
  if (which == 0) g_ln_reg = value != 0;
  if (which == 1) g_ln_bwd_minb = value;
}

}  // namespace vrr
