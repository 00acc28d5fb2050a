// bf16 / fp16 GEMMs of the ViT hot path on tcgen05 tensor cores with CTA PAIRS (cta_group::2), all operand
// layouts, fused epilogues.  T (Elem16) is the element type of the operands and of every 16-bit output.  One kernel template serves
//   * the QKV projection with the RoPE rotate-half epilogue         (models/vit.py:47-68)
//   * the patch-embedding GEMM                                      (models/vit.py:164,248-254)
//   * out-proj / fc1(+bias+GELU) / fc2 / head forward               (models/vit.py:91,118,285)
//   * every projection backward: dX = dY . W  and  dW = dY^T . X    (autograd of the above)
//
// C[M][N] = op(A)[M][K] . op(B)[K][N], fp32 accumulation in TMEM.
//   A_MN = 0: A stored [M][K] (K-major);  A_MN = 1: A stored [K][M] (MN-major, i.e. A^T is given)
//   B_MN = 0: B stored [N][K] (K-major, a Linear weight); B_MN = 1: B stored [K][N]
//
// A cluster of two CTAs (one per SM of a TPC) computes a 256 x BN tile: each CTA stages ITS 128 rows of
// op(A) and ITS half (BN/2 columns) of op(B) with TMA (128-byte swizzle), the leader CTA's MMA thread
// issues tcgen05.mma.cta_group::2 (M 256, N BN, K 16) which reads both CTAs' shared memory, and each CTA's
// TMEM receives its 128 rows x BN columns.  Per SM and per MMA this halves the shared-memory operand
// traffic (8 KB read per 128 tensor-clocks instead of 12 KB) - the 1-CTA kernel of round 1 was bound by
// shared-memory bandwidth (TMA fill + operand reads) at ~45 % of the tensor peak.
//
// Persistent: gridDim.x / 2 clusters loop over work units (m-tile, n-tile, k-split); warp roles
//   warp 0        TMA producer (one lane), kStages-deep ring, completes on the LEADER's full barrier
//   warp 1        TMEM allocator (both CTAs) + MMA issuer (leader only); accumulators double-buffered
//   warps 2..9    epilogue: tcgen05.ld -> registers -> (bias / GELU / RoPE) -> swizzled shared staging
//                 -> TMA store / TMA reduce-add (fp32 split-K), or a direct mapped store (planes, tokens)
//
// The bias of the BIAS epilogue is rounded to T before it is added for an fp32 C too (vrr.h: "cast to `dtype`
// first"); the fp32-C path once added the unrounded fp32 value.  tests/test_kernels_at_scale.py pins both C types
// bit for bit with biases off the bf16 grid.
#include <string.h>

#include <type_traits>

#include "common.cuh"
#include "kernels.h"
#include "tc_common.cuh"

namespace vrr {

using namespace tc;

namespace {

constexpr int kPM = 128;                              // rows of op(A) per CTA
constexpr int kPK = 64;                               // K elements per pipeline stage
constexpr int kEpiWarps = 8;
constexpr int kPairThreads = 64 + 32 * kEpiWarps;     // 320
constexpr int kWarpStaging = 8192;                    // two [32 rows][128 B] swizzled buffers per epilogue warp
constexpr int kSmemBudget = 232448;                   // 227 KB

struct PairShape {
  int M, N, K;
  int tiles_m, tiles_n, splits, num_k;
};

// ---------------------------------------------------------------------------------------------------
// Epilogues.  kTma = false: functor called per (row, 64-column chunk) with the fp32 accumulators.
// ---------------------------------------------------------------------------------------------------
// kPlaneStore: the functor only transforms the 64 accumulators of (row m, head chunk n0) in registers; the kernel
// rounds them to T, stages 32 rows x 128 B per warp in swizzled shared memory and writes them with TMA through a
// 3-D map of planes[3 B H][N][64]; the one warp tile in N / 32 that runs into the next image falls back to per-thread
// row stores.  A thread writing its own 128-byte row touched 32 lines per store instruction and made
// this GEMM 1.7x slower than the plain one.
template <typename T>
struct QkvRopeEpi2 {
  static constexpr bool kTma = false;
  static constexpr bool kPlaneStore = true;
  static constexpr bool kDrop = false;
  T* planes;
  const float *cos_tab, *sin_tab;
  const float4* packed;  // rope_pack_tables layout [heads][16][N - npre], or null
  int B, N, E, H, rope_mode;
  int npre;  // prefix tokens (cls, registers): rows t >= npre are rotated by table row t - npre
  __device__ __forceinline__ void rotate(int m, int n0, float (&f)[64]) const {
    const int hd = 32;
    const int b = m / N, t = m - b * N;
    const int which = n0 / E, h = (n0 - which * E) >> 6;
    if (rope_mode != VRR_ROPE_NONE && which < 2 && t >= npre && b < B && packed != nullptr) {
      // lanes = consecutive token rows = consecutive float4 of the packed table: coalesced 512-byte requests
      const float4* pk = packed + (size_t)(rope_mode == VRR_ROPE_MIXED ? h * 16 : 0) * (N - npre) + (t - npre);
#pragma unroll
      for (int q = 0; q < 16; ++q) {
        const float4 v = __ldg(pk + (size_t)q * (N - npre));  // {cos[2q], sin[2q], cos[2q+1], sin[2q+1]}
        const float x1 = f[2 * q], x2 = f[2 * q + hd], y1 = f[2 * q + 1], y2 = f[2 * q + 1 + hd];
        f[2 * q] = x1 * v.x - x2 * v.y;
        f[2 * q + hd] = x1 * v.y + x2 * v.x;
        f[2 * q + 1] = y1 * v.z - y2 * v.w;
        f[2 * q + 1 + hd] = y1 * v.w + y2 * v.z;
      }
    } else if (rope_mode != VRR_ROPE_NONE && which < 2 && t >= npre && b < B) {
      const size_t base = ((size_t)(rope_mode == VRR_ROPE_MIXED ? h * (N - npre) : 0) + (t - npre)) * hd;
      const float4* c4 = reinterpret_cast<const float4*>(cos_tab + base);
      const float4* s4 = reinterpret_cast<const float4*>(sin_tab + base);
#pragma unroll
      for (int q4 = 0; q4 < 8; ++q4) {
        const float4 c = __ldg(c4 + q4), s = __ldg(s4 + q4);
        const float cc[4] = {c.x, c.y, c.z, c.w}, ss[4] = {s.x, s.y, s.z, s.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int d = q4 * 4 + e;
          const float x1 = f[d], x2 = f[d + hd];
          f[d] = x1 * cc[e] - x2 * ss[e];
          f[d + hd] = x1 * ss[e] + x2 * cc[e];
        }
      }
    }
  }
  // plane index (third map coordinate) of the head chunk n0 for image b
  __device__ __forceinline__ int plane_of(int b, int n0) const {
    const int which = n0 / E, h = (n0 - which * E) >> 6;
    return (which * B + b) * H + h;
  }
  static constexpr bool kNorm = false;
};

// QkvRopeEpi2 with QK-norm (vrr_qkv_rope_norm_fwd).  Per q / k head chunk the kernel rounds the 64 accumulators to T
// (x), stores x to qk_pre (the map tmap_c2, same plane index as planes: its planes are planes' first 2 B H) through the
// staging slot before the final tile's, then normalize() writes {mean, rstd} and replaces x by y = xhat g + b; rotate()
// and the plane store follow as without the norm.  qk_pre / qk_stats null: inference, nothing saved.
template <typename T>
struct QkvNormRopeEpi2 : QkvRopeEpi2<T> {
  static constexpr bool kNorm = true;
  T* qk_pre;         // [2][B][H][N][64]
  float2* qk_stats;  // [2][B][H][N]
  const float4 *qn_w, *qn_b, *kn_w, *kn_b;  // [64] each
  float eps;
  __device__ __forceinline__ void normalize(int m, int n0, bool store, float (&f)[64]) const {
    const float2 st = qk_norm_stats(f, 64, eps);
    if (store && qk_stats != nullptr) {
      const int b = m / this->N, t = m - b * this->N;
      qk_stats[(size_t)this->plane_of(b, n0) * this->N + t] = st;  // lanes = consecutive rows: coalesced
    }
    const bool k = n0 >= this->E;
    const float4 *gw = k ? kn_w : qn_w, *gb = k ? kn_b : qn_b;  // warp-uniform: broadcast loads
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      const float4 g = __ldg(gw + q), bb = __ldg(gb + q);
      f[4 * q + 0] = qk_norm_y(qk_norm_xhat(f[4 * q + 0], st.x, st.y), g.x, bb.x);
      f[4 * q + 1] = qk_norm_y(qk_norm_xhat(f[4 * q + 1], st.x, st.y), g.y, bb.y);
      f[4 * q + 2] = qk_norm_y(qk_norm_xhat(f[4 * q + 2], st.x, st.y), g.z, bb.z);
      f[4 * q + 3] = qk_norm_y(qk_norm_xhat(f[4 * q + 3], st.x, st.y), g.w, bb.w);
    }
  }
};

// One row of 64 values as T: into the swizzled [32 rows][128 B] staging buffer at row_base (lane = row), or straight to
// global memory.
template <typename T>
__device__ __forceinline__ void stage_row64(uint32_t row_base, uint32_t sw, const float (&f)[64]) {
#pragma unroll
  for (int c8 = 0; c8 < 8; ++c8)
    st_shared_v4(row_base + (((uint32_t)c8 ^ sw) << 4), Elem16<T>::pack2(f[c8 * 8 + 0], f[c8 * 8 + 1]),
                 Elem16<T>::pack2(f[c8 * 8 + 2], f[c8 * 8 + 3]), Elem16<T>::pack2(f[c8 * 8 + 4], f[c8 * 8 + 5]),
                 Elem16<T>::pack2(f[c8 * 8 + 6], f[c8 * 8 + 7]));
}
template <typename T>
__device__ __forceinline__ void store_row64(T* dst, const float (&f)[64]) {
#pragma unroll
  for (int v8 = 0; v8 < 8; ++v8) {
    uint4 wv;
    wv.x = Elem16<T>::pack2(f[v8 * 8 + 0], f[v8 * 8 + 1]);
    wv.y = Elem16<T>::pack2(f[v8 * 8 + 2], f[v8 * 8 + 3]);
    wv.z = Elem16<T>::pack2(f[v8 * 8 + 4], f[v8 * 8 + 5]);
    wv.w = Elem16<T>::pack2(f[v8 * 8 + 6], f[v8 * 8 + 7]);
    *reinterpret_cast<uint4*>(dst + v8 * 8) = wv;
  }
}

// tokens[b][npre+p][n] = round_T(acc + bias[n]) (+ pos[p][n]); TT = token-stream type
template <typename T, typename TT>
struct PatchEmbedEpi2 {
  static constexpr bool kTma = false;
  static constexpr bool kPlaneStore = false;
  static constexpr bool kDrop = false;
  TT* tokens;
  const T* bias;
  const TT* pos;  // may be null
  int Np, E;
  int rows;  // token rows per image (npre + Np); `tokens` points at row npre of image 0
  __device__ __forceinline__ void operator()(int m, int n0, float (&f)[64]) const {
    const int b = m / Np, p = m - b * Np;
    TT* dst = tokens + ((size_t)b * rows + p) * E + n0;
    const TT* prow = pos ? pos + (size_t)p * E + n0 : nullptr;
#pragma unroll
    for (int v4 = 0; v4 < 16; ++v4) {
      const float4 bv = ld4(bias + n0 + v4 * 4);
      float4 o;
      o.x = Elem16<T>::round(f[v4 * 4 + 0] + bv.x);
      o.y = Elem16<T>::round(f[v4 * 4 + 1] + bv.y);
      o.z = Elem16<T>::round(f[v4 * 4 + 2] + bv.z);
      o.w = Elem16<T>::round(f[v4 * 4 + 3] + bv.w);
      if (prow) {
        const float4 pv = ld4(prow + v4 * 4);
        o.x += pv.x; o.y += pv.y; o.z += pv.z; o.w += pv.w;
      }
      st4(dst + v4 * 4, o);
    }
  }
};

// Row-major C through shared staging + TMA store.  Runtime (warp-uniform) switches keep the number of
// template instances small.
template <typename T>
struct StoreEpi {
  static constexpr bool kTma = true;
  static constexpr bool kPlaneStore = false;
  static constexpr bool kDrop = false;
  const float* bias;  // fp32 [N] or null; rounded to T first for either C type (autocast casts the bias)
  int out_f32;        // C element type: 0 T, 1 fp32
  int reduce;         // fp32 only: C += tile via TMA reduce-add (split-K partial sums / gradient accumulation)
  int gelu;           // T only.  1: C = h = T(acc + bias), C2 = T(gelu(h)) (exact erf GELU);
                      //         2: C = T(gelu(h)), C2 = T(gelu'(h)) - what an Mlp backward needs instead of h
                      //         3: C = T(gelu(h)) only (inference): its own code path, one TMA store per chunk
  const T* mul;       // T C only, or null: C = T(acc * mul[m][n]) (mul is [M][N] like C): d_act * gelu'(h)
  float* colsum;      // T plain / bias / mul paths, or null: colsum[n] += sum_m C[m][n] (values as stored; atomics)
};

// fc1 with element dropout (vrr_gemm_ex_drop): gelu 2 or 3 as above, every output then T(T(value) * f).  A type of its
// own, so that its epilogue branch is compiled into its own kernels and leaves the registers of the others alone.
template <typename T>
struct StoreEpiDrop : StoreEpi<T> {
  static constexpr bool kDrop = true;
  DropView dv;
};

// fc1 of a packed SwiGLU Mlp (vrr_gemm_swiglu).  The CTA pair stages gate rows (rank 0) and the matching value rows
// (rank 1) of w1 through one 3-D map [2][H][K], so TMEM columns [0, BN/2) of the tile hold g and [BN/2, BN) hold v
// for the same BN/2 output columns, and a ragged last tile is zero-filled within its half.  The epilogue writes act
// (tmap_c) and the two halves of aux (tmap_c2 / tmap_c3: maps over aux[:, :H] / aux[:, H:], row stride 2H) - or act
// alone when with_aux is 0.  Three [32 rows][128 B] staging buffers per warp.
template <typename T, bool DROP>
struct SwiGluEpi {
  static constexpr int kSwiGlu = 1;
  static constexpr int kStagingBytes = 12288;
  static constexpr bool kDrop = DROP;
  const float* bias;  // fp32 [2H]: gate biases, then value biases
  int with_aux;
  DropView dv;        // DROP only: mask of act [M][H]
};

// fc2's dX with the SwiGLU backward (vrr_gemm_swiglu_bwd): dA = dy . w2 stays in registers and is multiplied by the
// two multiplier tiles aux[:, n..] and aux[:, H+n..] into the halves of dh (tmap_c / tmap_c2); fc1's bias gradient
// is the column sums of both staged tiles (fp32 atomics, as StoreEpi::colsum).
template <typename T>
struct SwiGluBwdEpi {
  static constexpr int kSwiGlu = 2;
  const T* aux;   // [M][2H]
  float* colsum;  // [2H], zeroed by the caller
};

// SwiGluKind<Epi>::value: 0 for the epilogues above these two, else their kSwiGlu.  Staging<Epi>::kBytes: shared
// memory per epilogue warp.
template <class E, class = void>
struct SwiGluKind { static constexpr int value = 0; };
template <class E>
struct SwiGluKind<E, std::void_t<decltype(E::kSwiGlu)>> { static constexpr int value = E::kSwiGlu; };
template <class E, class = void>
struct Staging { static constexpr int kBytes = kWarpStaging; };
template <class E>
struct Staging<E, std::void_t<decltype(E::kStagingBytes)>> { static constexpr int kBytes = E::kStagingBytes; };

// gelu(h) and d gelu / dh for TWO values at a time on the packed fp32x2 pipe (fma.rn.f32x2, sm_100): the epilogue of
// fc1 is bound by its instruction count (128 x 256 outputs per CTA against ~6 100 tensor-clocks of MMA per tile), and
// the scalar version (~20 FMA-pipe ops per element) made the GEMM run at half the speed of the plain one.
//   Phi(h) = 1 - erfc(|h| / sqrt 2) / 2 (h >= 0), erfc / 2 otherwise; erfc(z) = (a1 t + .. + a5 t^5) exp(-z^2),
//   t = 1 / (1 + p z) (Abramowitz-Stegun 7.1.26, |error| <= 1.5e-7); gelu = h Phi, gelu' = Phi + h phi(h) with
//   phi(h) = exp(-h^2 / 2) / sqrt(2 pi) - the same exponential.
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void gelu_and_grad2(float2 h, float2& g, float2& dg) {
  const float2 hh = __fmul2_rn(h, h);
  const float2 ea = __fmul2_rn(hh, make_float2(-0.72134752044448170f, -0.72134752044448170f));
  const float2 e = make_float2(ex2(ea.x), ex2(ea.y));  // exp(-h^2 / 2)
  const float2 za = make_float2(fabsf(h.x), fabsf(h.y));
  const float2 den = __ffma2_rn(za, make_float2(0.23164190f, 0.23164190f), make_float2(1.f, 1.f));  // 1 + p |h| / sqrt 2
  const float2 t = make_float2(rcp_approx(den.x), rcp_approx(den.y));
  // coefficients pre-multiplied by 1/2
  float2 poly = __ffma2_rn(make_float2(0.5307027145f, 0.5307027145f), t, make_float2(-0.7265760135f, -0.7265760135f));
  poly = __ffma2_rn(poly, t, make_float2(0.7107068705f, 0.7107068705f));
  poly = __ffma2_rn(poly, t, make_float2(-0.142248368f, -0.142248368f));
  poly = __ffma2_rn(poly, t, make_float2(0.127414796f, 0.127414796f));
  const float2 q = __fmul2_rn(__fmul2_rn(poly, t), e);  // erfc(|h| / sqrt 2) / 2
  const float2 om = __ffma2_rn(q, make_float2(-1.f, -1.f), make_float2(1.f, 1.f));
  const float2 cdf = make_float2(h.x >= 0.f ? om.x : q.x, h.y >= 0.f ? om.y : q.y);  // Phi(h)
  g = __fmul2_rn(h, cdf);
  dg = __ffma2_rn(__fmul2_rn(h, e), make_float2(0.3989422804014327f, 0.3989422804014327f), cdf);
}

// gelu(h) alone, packed to a pair of T (same Phi(h) as above)
template <typename T>
__device__ __forceinline__ uint32_t gelu_only2(float2 h) {
  const float2 hh = __fmul2_rn(h, h);
  const float2 ea = __fmul2_rn(hh, make_float2(-0.72134752044448170f, -0.72134752044448170f));
  const float2 e = make_float2(ex2(ea.x), ex2(ea.y));
  const float2 za = make_float2(fabsf(h.x), fabsf(h.y));
  const float2 den = __ffma2_rn(za, make_float2(0.23164190f, 0.23164190f), make_float2(1.f, 1.f));
  const float2 t = make_float2(rcp_approx(den.x), rcp_approx(den.y));
  float2 poly = __ffma2_rn(make_float2(0.5307027145f, 0.5307027145f), t, make_float2(-0.7265760135f, -0.7265760135f));
  poly = __ffma2_rn(poly, t, make_float2(0.7107068705f, 0.7107068705f));
  poly = __ffma2_rn(poly, t, make_float2(-0.142248368f, -0.142248368f));
  poly = __ffma2_rn(poly, t, make_float2(0.127414796f, 0.127414796f));
  const float2 q = __fmul2_rn(__fmul2_rn(poly, t), e);
  const float2 om = __ffma2_rn(q, make_float2(-1.f, -1.f), make_float2(1.f, 1.f));
  const float2 g = __fmul2_rn(h, make_float2(h.x >= 0.f ? om.x : q.x, h.y >= 0.f ? om.y : q.y));
  return Elem16<T>::pack2(g.x, g.y);
}

// ---------------------------------------------------------------------------------------------------
template <typename T, int BN, bool A_MN, bool B_MN, class Epi>
__global__ void __launch_bounds__(kPairThreads, 1)
gemm_pair_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                 const __grid_constant__ CUtensorMap tmap_c, const __grid_constant__ CUtensorMap tmap_c2,
                 const __grid_constant__ CUtensorMap tmap_c3, const PairShape g, const Epi epi) {
  constexpr int kBHalf = BN / 2;
  constexpr int kABytes = kPM * kPK * 2;
  constexpr int kBBytes = kBHalf * kPK * 2;
  constexpr int kStageBytes = kABytes + kBBytes;
  constexpr int kStg = Staging<Epi>::kBytes;
  constexpr int kSwi = SwiGluKind<Epi>::value;
  constexpr int kStages = (kSmemBudget - 1024 - kEpiWarps * kStg - 512) / kStageBytes;
  constexpr uint32_t kTmemCols = 2 * BN;  // two accumulator stages (256 or 512: powers of two)
  static_assert(kStages >= 3, "pipeline too shallow");
  static_assert(kSwi != 1 || (BN == 256 && !A_MN && !B_MN), "the SwiGLU forward pairs 128 gate with 128 value columns");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* staging = smem + kStages * kStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(staging + kEpiWarps * kStg);
  uint64_t* bar_full = bars;                              // [kStages] leader's: both CTAs' TMA -> MMA
  uint64_t* bar_empty = bars + kStages;                   // [kStages] per CTA: MMA retired -> own TMA producer
  uint64_t* bar_acc_full = bars + 2 * kStages;            // [2] per CTA: accumulator ready -> own epilogue
  uint64_t* bar_acc_empty = bars + 2 * kStages + 2;       // [2] leader's: both CTAs' epilogues -> MMA
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int num_clusters = gridDim.x >> 1, cluster_id = blockIdx.x >> 1;
  const int total_units = g.tiles_m * g.tiles_n * g.splits;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&bar_full[s], 2);   // one arrive.expect_tx per CTA of the pair
      mbar_init(&bar_empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&bar_acc_full[a], 1);
      mbar_init(&bar_acc_empty[a], 2 * kEpiWarps);  // one elected lane per epilogue warp, both CTAs
    }
    fence_mbar_init();
  }
  __syncwarp();
  if (warp == 1) tmem_alloc_pair(tmem_slot, kTmemCols);
  tc_fence_before();
  cluster_sync();  // both CTAs: barriers initialised, TMEM allocated, before any cross-CTA signal
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ====================================== TMA producer (both CTAs) ======================================
    if (lane == 0) {
      tma_prefetch_desc(&tmap_a);
      tma_prefetch_desc(&tmap_b);
      int stage = 0;
      uint32_t phase = 0;
      for (int unit = cluster_id; unit < total_units; unit += num_clusters) {
        const int split = unit % g.splits, t = unit / g.splits;
        const int n_blk = t % g.tiles_n, m_blk = t / g.tiles_n;
        const int kb0 = (int)((long long)split * g.num_k / g.splits), kb1 = (int)((long long)(split + 1) * g.num_k / g.splits);
        const int m_row0 = m_blk * (2 * kPM) + (int)rank * kPM;
        [[maybe_unused]] const int n_row0 = n_blk * BN + (int)rank * kBHalf;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait_cluster(&bar_empty[stage], phase ^ 1);
          const uint32_t full_leader = mapa(smem_u32(&bar_full[stage]), 0);
          mbar_expect_tx_cluster(full_leader, kStageBytes);
          uint8_t* sa = smem + stage * kStageBytes;
          uint8_t* sb = sa + kABytes;
          if (!A_MN) {
            tma_load_2d_pair(sa, &tmap_a, full_leader, kb * kPK, m_row0);
          } else {
#pragma unroll
            for (int j = 0; j < kPM / 64; ++j) tma_load_2d_pair(sa + j * 8192, &tmap_a, full_leader, m_row0 + 64 * j, kb * kPK);
          }
          if constexpr (kSwi == 1) {  // rank 0: gate rows, rank 1: the value rows of the same output columns
            tma_load_3d_pair(sb, &tmap_b, full_leader, kb * kPK, n_blk * kBHalf, (int)rank);
          } else if (!B_MN) {
            tma_load_2d_pair(sb, &tmap_b, full_leader, kb * kPK, n_row0);
          } else {
#pragma unroll
            for (int j = 0; j < kBHalf / 64; ++j) tma_load_2d_pair(sb + j * 8192, &tmap_b, full_leader, n_row0 + 64 * j, kb * kPK);
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ====================================== MMA issuer (leader CTA only) ==================================
    if (rank == 0 && lane == 0) {
      constexpr uint32_t idesc = idesc_16<T>(2 * kPM, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
      constexpr uint32_t adv_a = A_MN ? 128 : 2, adv_b = B_MN ? 128 : 2;  // descriptor units (16 B) per K = 16
      int stage = 0, acc = 0;
      uint32_t phase = 0, acc_phase = 0;
      for (int unit = cluster_id; unit < total_units; unit += num_clusters) {
        const int split = unit % g.splits;
        const int kb0 = (int)((long long)split * g.num_k / g.splits), kb1 = (int)((long long)(split + 1) * g.num_k / g.splits);
        mbar_wait_cluster(&bar_acc_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait_cluster(&bar_full[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * kStageBytes);
          const uint64_t da = A_MN ? smem_desc_sw128_ex(sa, 8192, 1024) : smem_desc_sw128(sa);
          const uint64_t db = B_MN ? smem_desc_sw128_ex(sa + kABytes, 8192, 1024) : smem_desc_sw128(sa + kABytes);
#pragma unroll
          for (int k = 0; k < kPK / 16; ++k)
            mma_ss_pair(d_tmem, da + adv_a * k, db + adv_b * k, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          mma_commit_pair(&bar_empty[stage], 3);  // both CTAs' producers may refill the slot when these retire
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        mma_commit_pair(&bar_acc_full[acc], 3);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if constexpr (kSwi == 1) {
    // ============================ SwiGLU fc1 epilogue (both CTAs): act and aux from (g, v) ===============
    // Warp half `chalf` takes output columns [64 chalf, 64 chalf + 64) of the tile: g at TMEM column c, v at
    // BN/2 + c; two halves of 32 columns, every 8 columns stored to the three swizzled staging buffers as soon as
    // they are computed (holding them for a later flush spilled registers).
    const int ew = warp - 2, quad = warp & 3, chalf = ew >> 2;
    uint8_t* my_stage = staging + ew * kStg;
    const uint32_t sw = (uint32_t)(lane & 7);
    const uint32_t row_base = smem_u32(my_stage) + (uint32_t)lane * 128u;
    const int H = g.N;
    [[maybe_unused]] uint2 key;
    if constexpr (Epi::kDrop) key = epi.dv.key();
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int unit = cluster_id; unit < total_units; unit += num_clusters) {
      const int n_blk = unit % g.tiles_n, m_blk = unit / g.tiles_n;  // one k-split
      const int m_warp0 = m_blk * (2 * kPM) + (int)rank * kPM + quad * 32;
      const int m = m_warp0 + lane;
      const int n0 = n_blk * kBHalf + chalf * 64;
      mbar_wait_cluster(&bar_acc_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t tg = tmem_base + ((uint32_t)(quad * 32) << 16) + acc * BN + chalf * 64;
      if (lane == 0) bulk_wait_read<0>();  // the previous unit's stores have left the staging buffers
      __syncwarp();
#pragma unroll 1
      for (int hf = 0; hf < 2; ++hf) {
        uint32_t v[64];
        __syncwarp();
        tmem_ld32(tg + hf * 32, *reinterpret_cast<uint32_t(*)[32]>(&v[0]));
        tmem_ld32(tg + kBHalf + hf * 32, *reinterpret_cast<uint32_t(*)[32]>(&v[32]));
        tmem_wait_ld();
        if (hf == 1) {  // this warp has read everything it needs from the accumulator stage
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(mapa(smem_u32(&bar_acc_empty[acc]), 0));
        }
        const float* fa = reinterpret_cast<const float*>(v);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint32_t oa[4], og[4], ov[4];
          const int nb = max(min(n0 + hf * 32 + q * 8, H - 8), 0);  // H % 8 == 0; columns past H are clipped
          const float4 bg0 = __ldg(reinterpret_cast<const float4*>(epi.bias + nb));
          const float4 bg1 = __ldg(reinterpret_cast<const float4*>(epi.bias + nb + 4));
          const float4 bv0 = __ldg(reinterpret_cast<const float4*>(epi.bias + H + nb));
          const float4 bv1 = __ldg(reinterpret_cast<const float4*>(epi.bias + H + nb + 4));
          // the biases as T (F.linear's cast), packed in pairs
          const uint32_t bgp[4] = {Elem16<T>::pack2(bg0.x, bg0.y), Elem16<T>::pack2(bg0.z, bg0.w), Elem16<T>::pack2(bg1.x, bg1.y),
                                   Elem16<T>::pack2(bg1.z, bg1.w)};
          const uint32_t bvp[4] = {Elem16<T>::pack2(bv0.x, bv0.y), Elem16<T>::pack2(bv0.z, bv0.w), Elem16<T>::pack2(bv1.x, bv1.y),
                                   Elem16<T>::pack2(bv1.z, bv1.w)};
          [[maybe_unused]] uint32_t rw[4];
          if constexpr (Epi::kDrop) {
            const uint4 r = epi.dv.bits(key, ((unsigned long long)m * (unsigned)H + (unsigned)nb) >> 3);
            rw[0] = r.x; rw[1] = r.y; rw[2] = r.z; rw[3] = r.w;
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            float a[2], lo[2], hi[2];
            const float2 bg2 = Elem16<T>::unpack2(bgp[j]), bv2 = Elem16<T>::unpack2(bvp[j]);
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const int c = q * 8 + 2 * j + e;
              const float gg = Elem16<T>::round(fa[c] + (e ? bg2.y : bg2.x));
              const float vv = Elem16<T>::round(fa[32 + c] + (e ? bv2.y : bv2.x));
              float s, ds;
              silu_and_grad(gg, s, ds);
              const float sr = Elem16<T>::round(s);
              a[e] = Elem16<T>::round(__fmul_rn(sr, vv));
              lo[e] = __fmul_rn(vv, ds);
              hi[e] = sr;
              if constexpr (Epi::kDrop) {
                const float f = ((e ? (rw[j] >> 16) : (rw[j] & 0xFFFFu)) < epi.dv.t) ? epi.dv.s : 0.f;
                a[e] = __fmul_rn(a[e], f);
                lo[e] = __fmul_rn(lo[e], f);
                hi[e] = __fmul_rn(hi[e], f);
              }
            }
            oa[j] = Elem16<T>::pack2(a[0], a[1]);
            og[j] = Elem16<T>::pack2(lo[0], lo[1]);
            ov[j] = Elem16<T>::pack2(hi[0], hi[1]);
          }
          const uint32_t off = (((uint32_t)(hf * 4 + q) ^ sw) << 4);
          st_shared_v4(row_base + off, oa[0], oa[1], oa[2], oa[3]);
          if (epi.with_aux) {
            st_shared_v4(row_base + 4096u + off, og[0], og[1], og[2], og[3]);
            st_shared_v4(row_base + 8192u + off, ov[0], ov[1], ov[2], ov[3]);
          }
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        if (n0 < H && m_warp0 < g.M) {
          tma_store_2d(&tmap_c, my_stage, n0, m_warp0);
          if (epi.with_aux) {
            tma_store_2d(&tmap_c2, my_stage + 4096, n0, m_warp0);
            tma_store_2d(&tmap_c3, my_stage + 8192, n0, m_warp0);
          }
        }
        bulk_commit();
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    if (lane == 0) bulk_wait<0>();
  } else if constexpr (kSwi == 2) {
    // ==================== SwiGLU backward epilogue (both CTAs): dh halves and fc1's bias gradient ===============
    const int ew = warp - 2, quad = warp & 3, chalf = ew >> 2;
    constexpr int kChunks = BN / 2 / 64;
    uint8_t* my_stage = staging + ew * kStg;
    const uint32_t stage_u32 = smem_u32(my_stage);
    const uint32_t sw = (uint32_t)(lane & 7);
    const uint32_t row_base = stage_u32 + (uint32_t)lane * 128u;
    const int H = g.N;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int unit = cluster_id; unit < total_units; unit += num_clusters) {
      const int n_blk = unit % g.tiles_n, m_blk = unit / g.tiles_n;  // one k-split
      const int m_warp0 = m_blk * (2 * kPM) + (int)rank * kPM + quad * 32;
      mbar_wait_cluster(&bar_acc_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t trow = tmem_base + ((uint32_t)(quad * 32) << 16) + acc * BN + chalf * (BN / 2);
#pragma unroll 1
      for (int c = 0; c < kChunks; ++c) {
        const int n0 = n_blk * BN + chalf * (BN / 2) + c * 64;
        // the warp's [32 rows][64] tiles of aux[:, n0..] and aux[:, H + n0..], loaded coalesced (as StoreEpi::mul)
        // while the TMEM load is in flight
        uint4 ml[8], mh[8];
        const int nb = max(min(n0 + (lane & 7) * 8, H - 8), 0);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int mr = min(m_warp0 + i * 4 + (lane >> 3), g.M - 1);
          const T* p = epi.aux + (size_t)mr * 2 * H + nb;
          ml[i] = __ldg(reinterpret_cast<const uint4*>(p));
          mh[i] = __ldg(reinterpret_cast<const uint4*>(p + H));
        }
        // "lane = row" through the two staging buffers (the previous chunk's stores have been read) BEFORE the TMEM
        // load: the multipliers and the 64 accumulators held together spilled registers
        if (lane == 0) bulk_wait_read<0>();
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const uint32_t r = (uint32_t)(i * 4 + (lane >> 3));
          const uint32_t off = r * 128u + ((((uint32_t)lane & 7u) ^ (r & 7u)) << 4);
          st_shared_v4(stage_u32 + off, ml[i].x, ml[i].y, ml[i].z, ml[i].w);
          st_shared_v4(stage_u32 + 4096u + off, mh[i].x, mh[i].y, mh[i].z, mh[i].w);
        }
        uint32_t v[64];
        __syncwarp();
        tmem_ld32(trow + c * 64, *reinterpret_cast<uint32_t(*)[32]>(&v[0]));
        tmem_ld32(trow + c * 64 + 32, *reinterpret_cast<uint32_t(*)[32]>(&v[32]));
        tmem_wait_ld();
        if (c == kChunks - 1) {  // this warp has read everything it needs from the accumulator stage
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(mapa(smem_u32(&bar_acc_empty[acc]), 0));
        }
        const float* fa = reinterpret_cast<const float*>(v);
#pragma unroll
        for (int c8 = 0; c8 < 8; ++c8) {  // each lane reads and overwrites its own row's chunk: no other lane touches it
          const uint32_t off = (((uint32_t)c8 ^ sw) << 4);
          const uint4 ml4 = ld_shared_v4(row_base + off), mh4 = ld_shared_v4(row_base + 4096u + off);
          const uint32_t wl[4] = {ml4.x, ml4.y, ml4.z, ml4.w}, wh[4] = {mh4.x, mh4.y, mh4.z, mh4.w};
          uint32_t ol[4], oh[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float2 a2 = make_float2(fa[c8 * 8 + 2 * j], fa[c8 * 8 + 2 * j + 1]);
            const float2 l2 = Elem16<T>::unpack2(wl[j]), h2 = Elem16<T>::unpack2(wh[j]);
            ol[j] = Elem16<T>::pack2(__fmul_rn(a2.x, l2.x), __fmul_rn(a2.y, l2.y));
            oh[j] = Elem16<T>::pack2(__fmul_rn(a2.x, h2.x), __fmul_rn(a2.y, h2.y));
          }
          st_shared_v4(row_base + off, ol[0], ol[1], ol[2], ol[3]);
          st_shared_v4(row_base + 4096u + off, oh[0], oh[1], oh[2], oh[3]);
        }
        fence_proxy_async_smem();
        __syncwarp();
        const bool store_ok = n0 < H && m_warp0 < g.M;
        if (lane == 0) {
          if (store_ok) {
            tma_store_2d(&tmap_c, my_stage, n0, m_warp0);
            tma_store_2d(&tmap_c2, my_stage + 4096, n0, m_warp0);
          }
          bulk_commit();
        }
        if (store_ok) {
          // column sums of both tiles as stored (rows past M hold zeros: their dy rows were zero-filled)
          float s0 = 0.f, s1 = 0.f, t0 = 0.f, t1 = 0.f;
          const uint32_t cbase = stage_u32 + ((uint32_t)lane & 3u) * 4u;
#pragma unroll 8
          for (uint32_t r = 0; r < 32; ++r) {
            const uint32_t off = r * 128u + ((((uint32_t)lane >> 2) ^ (r & 7u)) << 4);
            const float2 l2 = Elem16<T>::unpack2(ld_shared_u32(cbase + off));
            const float2 h2 = Elem16<T>::unpack2(ld_shared_u32(cbase + 4096u + off));
            s0 += l2.x; s1 += l2.y; t0 += h2.x; t1 += h2.y;
          }
          const int col = n0 + 2 * lane;
          if (col < H) {
            atomicAdd(epi.colsum + col, s0);
            atomicAdd(epi.colsum + col + 1, s1);
            atomicAdd(epi.colsum + H + col, t0);
            atomicAdd(epi.colsum + H + col + 1, t1);
          }
        }
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    if (lane == 0) bulk_wait<0>();
  } else {
    // ====================================== epilogue (both CTAs) ==========================================
    const int ew = warp - 2;
    const int quad = warp & 3;          // TMEM lane quadrant this warp may access
    const int chalf = ew >> 2;          // which half of the tile's columns
    constexpr int kChunks = BN / 2 / 64;
    uint8_t* my_stage = staging + ew * kWarpStaging;
    const uint32_t stage_u32 = smem_u32(my_stage);
    int acc = 0;
    uint32_t acc_phase = 0;
    uint32_t chunk_counter = 0;
    for (int unit = cluster_id; unit < total_units; unit += num_clusters) {
      const int t = unit / g.splits;
      const bool first_split = (unit - t * g.splits) == 0;  // the bias joins exactly one of the k-splits
      const int n_blk = t % g.tiles_n, m_blk = t / g.tiles_n;
      const int m_warp0 = m_blk * (2 * kPM) + (int)rank * kPM + quad * 32;
      const int m = m_warp0 + lane;
      mbar_wait_cluster(&bar_acc_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t trow = tmem_base + ((uint32_t)(quad * 32) << 16) + acc * BN + chalf * (BN / 2);
#pragma unroll 1
      for (int c = 0; c < kChunks; ++c) {
        uint32_t v[64];
        // StoreEpi::mul: the warp's [32 rows][64] multiplier tile.  Loaded COALESCED (instruction i = rows 4i..4i+3,
        // eight lanes x 16 bytes per row; a lane reading its own row touched 32 lines per instruction) while the TMEM
        // load is in flight, then turned into "lane = row" through the swizzled staging buffer this chunk's output
        // will use (its previous TMA store has been read: bulk_wait_read<1>).
        [[maybe_unused]] uint4 mv[8];
        [[maybe_unused]] bool with_mul = false;
        if constexpr (Epi::kTma && !Epi::kDrop) {
          with_mul = epi.mul != nullptr;
          if (with_mul) {
            const int n0m = n_blk * BN + chalf * (BN / 2) + c * 64;
            const int nb = max(min(n0m + (lane & 7) * 8, g.N - 8), 0);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int mr = min(m_warp0 + i * 4 + (lane >> 3), g.M - 1);
              mv[i] = __ldg(reinterpret_cast<const uint4*>(epi.mul + (size_t)mr * g.N + nb));
            }
          }
        }
        __syncwarp();  // tcgen05.ld is .sync.aligned
        tmem_ld32(trow + c * 64, *reinterpret_cast<uint32_t(*)[32]>(&v[0]));
        tmem_ld32(trow + c * 64 + 32, *reinterpret_cast<uint32_t(*)[32]>(&v[32]));
        if constexpr (Epi::kTma && !Epi::kDrop) {
          if (with_mul) {
            const uint32_t tbuf = stage_u32 + (chunk_counter & 1u) * 4096u;
            if (lane == 0) bulk_wait_read<1>();
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const uint32_t r = (uint32_t)(i * 4 + (lane >> 3));
              st_shared_v4(tbuf + r * 128u + ((((uint32_t)lane & 7u) ^ (r & 7u)) << 4), mv[i].x, mv[i].y, mv[i].z, mv[i].w);
            }
            __syncwarp();
#pragma unroll
            for (int c8 = 0; c8 < 8; ++c8)
              mv[c8] = ld_shared_v4(tbuf + (uint32_t)lane * 128u + ((((uint32_t)c8) ^ ((uint32_t)lane & 7u)) << 4));
          }
        }
        tmem_wait_ld();
        if (c == kChunks - 1) {  // this warp has read everything it needs from the accumulator stage
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(mapa(smem_u32(&bar_acc_empty[acc]), 0));
        }
        const int n0 = n_blk * BN + chalf * (BN / 2) + c * 64;
        float(&f)[64] = *reinterpret_cast<float(*)[64]>(v);
        if constexpr (Epi::kPlaneStore) {
          if constexpr (Epi::kNorm) {
            if (n0 < 2 * epi.E) {  // a q or k head (warp-uniform)
#pragma unroll
              for (int i = 0; i < 64; ++i) f[i] = Elem16<T>::round(f[i]);
              const int pb0 = m_warp0 / epi.N, pt0 = m_warp0 - pb0 * epi.N;
              const bool p_in_range = m_warp0 < g.M;
              if (epi.qk_pre != nullptr) {
                // staged in any case; the warp tile that runs into the next image copies each lane's own row out of the
                // staging buffer (row stores straight from the registers spilled at BN = 256)
                const bool whole = pt0 + 32 <= epi.N || !p_in_range;
                const uint32_t sw = (uint32_t)(lane & 7);
                const uint32_t buf = (chunk_counter & 1u) * 4096u, row_base = stage_u32 + buf + (uint32_t)lane * 128u;
                if (lane == 0) bulk_wait_read<1>();
                __syncwarp();
                stage_row64<T>(row_base, sw, f);
                if (whole) {
                  fence_proxy_async_smem();
                  __syncwarp();
                } else if (m < g.M) {
                  const int b = m / epi.N, t = m - b * epi.N;
                  uint4* dst = reinterpret_cast<uint4*>(epi.qk_pre + ((size_t)epi.plane_of(b, n0) * epi.N + t) * 64);
#pragma unroll
                  for (int c8 = 0; c8 < 8; ++c8) dst[c8] = ld_shared_v4(row_base + (((uint32_t)c8 ^ sw) << 4));
                }
                if (lane == 0) {
                  if (whole && p_in_range) tma_store_3d(&tmap_c2, my_stage + buf, 0, pt0, epi.plane_of(pb0, n0));
                  bulk_commit();  // a group in either case: the ring's bulk_wait_read<1> counts one per slot use
                }
                ++chunk_counter;
              }
              epi.normalize(m, n0, m < g.M, f);
            }
          }
          epi.rotate(m, n0, f);
          const int b0 = m_warp0 / epi.N, t0 = m_warp0 - b0 * epi.N;
          const bool in_range = n0 < g.N && m_warp0 < g.M;
          if (t0 + 32 <= epi.N || !in_range) {
            // the warp's 32 rows lie in one image: swizzled staging + one TMA store
            const uint32_t buf = (chunk_counter & 1u) * 4096u;
            if (lane == 0) bulk_wait_read<1>();
            __syncwarp();
            stage_row64<T>(stage_u32 + buf + (uint32_t)lane * 128u, (uint32_t)(lane & 7), f);
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              if (in_range) tma_store_3d(&tmap_c, my_stage + buf, 0, t0, epi.plane_of(b0, n0));
              bulk_commit();
            }
            ++chunk_counter;
          } else if (m < g.M) {
            // the rows run into the next image (one warp tile in N / 32; TMA stores take no negative coordinates -
            // "illegal instruction" - and a box cannot be shortened): each thread stores its own row
            const int b = m / epi.N, t = m - b * epi.N;
            store_row64<T>(epi.planes + ((size_t)epi.plane_of(b, n0) * epi.N + t) * 64, f);
          }
        } else if constexpr (!Epi::kTma) {
          if (m < g.M && n0 < g.N) epi(m, n0, f);
        } else {
          const bool store_ok = (n0 < g.N) && (m_warp0 < g.M);
          const uint32_t sw = (uint32_t)(lane & 7);
          const uint32_t row_base = stage_u32 + (uint32_t)lane * 128u;
          if (Epi::kDrop || !epi.out_f32) {
            // ---- 16-bit C (T) ----
            if constexpr (Epi::kDrop) {
              // fc1 with dropout: (gelu(h), gelu'(h)) or gelu(h) alone, each rounded to T and multiplied by the keep
              // factor of its element; one Philox call per 8 columns covers a group of the mask.  Computed in two
              // halves of 32 columns, as in the two-output branch below.
              const uint2 key = epi.dv.key();
              const bool two = epi.gelu == 2;
#pragma unroll
              for (int hf = 0; hf < 2; ++hf) {
                uint32_t o0[16], o1[16];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  const int c8 = hf * 4 + q;
                  const int nb = min(n0 + c8 * 8, g.N - 8);
                  const float4 b0 = __ldg(reinterpret_cast<const float4*>(epi.bias + nb));
                  const float4 b1 = __ldg(reinterpret_cast<const float4*>(epi.bias + nb + 4));
                  const uint32_t br[4] = {Elem16<T>::pack2(b0.x, b0.y), Elem16<T>::pack2(b0.z, b0.w), Elem16<T>::pack2(b1.x, b1.y), Elem16<T>::pack2(b1.z, b1.w)};
                  const uint4 r = epi.dv.bits(key, ((unsigned long long)m * (unsigned)g.N + (unsigned)nb) >> 3);
                  const uint32_t rw[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
                  for (int j = 0; j < 4; ++j) {
                    const float2 bb = Elem16<T>::unpack2(br[j]);
                    const float2 hs = __fadd2_rn(make_float2(f[c8 * 8 + 2 * j], f[c8 * 8 + 2 * j + 1]), bb);
                    const float2 hr = Elem16<T>::unpack2(Elem16<T>::pack2(hs.x, hs.y));
                    const float f0 = (rw[j] & 0xFFFFu) < epi.dv.t ? epi.dv.s : 0.f;
                    const float f1 = (rw[j] >> 16) < epi.dv.t ? epi.dv.s : 0.f;
                    if (two) {
                      float2 gl, dg;
                      gelu_and_grad2(hr, gl, dg);
                      const float2 gr = Elem16<T>::unpack2(Elem16<T>::pack2(gl.x, gl.y));
                      const float2 dr = Elem16<T>::unpack2(Elem16<T>::pack2(dg.x, dg.y));
                      o0[q * 4 + j] = Elem16<T>::pack2(__fmul_rn(gr.x, f0), __fmul_rn(gr.y, f1));
                      o1[q * 4 + j] = Elem16<T>::pack2(__fmul_rn(dr.x, f0), __fmul_rn(dr.y, f1));
                    } else {
                      const float2 gr = Elem16<T>::unpack2(gelu_only2<T>(hr));
                      o0[q * 4 + j] = Elem16<T>::pack2(__fmul_rn(gr.x, f0), __fmul_rn(gr.y, f1));
                    }
                  }
                }
                if (hf == 0) {
                  if (lane == 0) bulk_wait_read<0>();
                  __syncwarp();
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  const uint32_t off = (((uint32_t)(hf * 4 + q) ^ sw) << 4);
                  st_shared_v4(row_base + off, o0[q * 4], o0[q * 4 + 1], o0[q * 4 + 2], o0[q * 4 + 3]);
                  if (two) st_shared_v4(row_base + 4096u + off, o1[q * 4], o1[q * 4 + 1], o1[q * 4 + 2], o1[q * 4 + 3]);
                }
              }
              fence_proxy_async_smem();
              __syncwarp();
              if (lane == 0) {
                if (store_ok) {
                  tma_store_2d(&tmap_c, my_stage, n0, m_warp0);
                  if (two) tma_store_2d(&tmap_c2, my_stage + 4096, n0, m_warp0);
                }
                bulk_commit();
              }
            } else if (epi.gelu == 3) {
              // inference: gelu(h) alone.  Its own branch - folding it into the two-output code below cost that path
              // 50 us per launch (register allocation of the o0 / o1 arrays).
              uint32_t o0[32];
#pragma unroll
              for (int c8 = 0; c8 < 8; ++c8) {
                const int nb = min(n0 + c8 * 8, g.N - 8);
                const float4 b0 = __ldg(reinterpret_cast<const float4*>(epi.bias + nb));
                const float4 b1 = __ldg(reinterpret_cast<const float4*>(epi.bias + nb + 4));
                const uint32_t br[4] = {Elem16<T>::pack2(b0.x, b0.y), Elem16<T>::pack2(b0.z, b0.w), Elem16<T>::pack2(b1.x, b1.y), Elem16<T>::pack2(b1.z, b1.w)};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  const float2 bb = Elem16<T>::unpack2(br[j]);
                  const float2 hs = __fadd2_rn(make_float2(f[c8 * 8 + 2 * j], f[c8 * 8 + 2 * j + 1]), bb);
                  const uint32_t hw = Elem16<T>::pack2(hs.x, hs.y);
                  o0[c8 * 4 + j] = gelu_only2<T>(Elem16<T>::unpack2(hw));
                }
              }
              const uint32_t buf = (chunk_counter & 1u) * 4096u;
              if (lane == 0) bulk_wait_read<1>();
              __syncwarp();
#pragma unroll
              for (int c8 = 0; c8 < 8; ++c8)
                st_shared_v4(row_base + buf + (((uint32_t)c8 ^ sw) << 4), o0[c8 * 4], o0[c8 * 4 + 1], o0[c8 * 4 + 2],
                             o0[c8 * 4 + 3]);
              fence_proxy_async_smem();
              __syncwarp();
              if (lane == 0) {
                if (store_ok) tma_store_2d(&tmap_c, my_stage + buf, n0, m_warp0);
                bulk_commit();
              }
            } else if (epi.gelu != 0) {
              // two outputs: (h, gelu(h)) or (gelu(h), gelu'(h)).  Computed and flushed to the staging buffers in two
              // halves of 32 columns: the profile of the one-piece version was 58 % fixed-latency dependency stalls
              // (`stall_wait`) - with 64 packed outputs held next to the 64 accumulators ptxas had no registers left
              // to interleave the per-pair chains.  The first half is computed BEFORE the wait for the previous
              // chunk's TMA stores.
#pragma unroll
              for (int hf = 0; hf < 2; ++hf) {
                uint32_t o0[16], o1[16];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  const int c8 = hf * 4 + q;
                  const int nb = min(n0 + c8 * 8, g.N - 8);  // N % 8 == 0; clamp keeps the tail read in bounds
                  const float4 b0 = __ldg(reinterpret_cast<const float4*>(epi.bias + nb));
                  const float4 b1 = __ldg(reinterpret_cast<const float4*>(epi.bias + nb + 4));
                  const uint32_t br[4] = {Elem16<T>::pack2(b0.x, b0.y), Elem16<T>::pack2(b0.z, b0.w), Elem16<T>::pack2(b1.x, b1.y), Elem16<T>::pack2(b1.z, b1.w)};
#pragma unroll
                  for (int j = 0; j < 4; ++j) {
                    const float2 bb = Elem16<T>::unpack2(br[j]);  // bias as T
                    const float2 hs = __fadd2_rn(make_float2(f[c8 * 8 + 2 * j], f[c8 * 8 + 2 * j + 1]), bb);
                    const uint32_t hw = Elem16<T>::pack2(hs.x, hs.y);
                    const float2 hr = Elem16<T>::unpack2(hw);  // h as stored
                    float2 gl, dg;
                    gelu_and_grad2(hr, gl, dg);
                    if (epi.gelu == 1) {
                      o0[q * 4 + j] = hw;
                      o1[q * 4 + j] = Elem16<T>::pack2(gl.x, gl.y);
                    } else {
                      o0[q * 4 + j] = Elem16<T>::pack2(gl.x, gl.y);
                      o1[q * 4 + j] = Elem16<T>::pack2(dg.x, dg.y);
                    }
                  }
                }
                if (hf == 0) {
                  if (lane == 0) bulk_wait_read<0>();
                  __syncwarp();
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  const uint32_t off = (((uint32_t)(hf * 4 + q) ^ sw) << 4);
                  st_shared_v4(row_base + off, o0[q * 4], o0[q * 4 + 1], o0[q * 4 + 2], o0[q * 4 + 3]);
                  st_shared_v4(row_base + 4096u + off, o1[q * 4], o1[q * 4 + 1], o1[q * 4 + 2], o1[q * 4 + 3]);
                }
              }
              fence_proxy_async_smem();
              __syncwarp();
              if (lane == 0) {
                if (store_ok) {
                  tma_store_2d(&tmap_c, my_stage, n0, m_warp0);
                  tma_store_2d(&tmap_c2, my_stage + 4096, n0, m_warp0);
                }
                bulk_commit();
              }
            } else {
              const uint32_t buf = (chunk_counter & 1u) * 4096u;
              if (lane == 0) bulk_wait_read<1>();
              __syncwarp();
#pragma unroll
              for (int c8 = 0; c8 < 8; ++c8) {
                float x[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) x[j] = f[c8 * 8 + j];
                if (epi.bias != nullptr) {
                  const int nb = min(n0 + c8 * 8, g.N - 8);
                  const float4 b0 = __ldg(reinterpret_cast<const float4*>(epi.bias + nb));
                  const float4 b1 = __ldg(reinterpret_cast<const float4*>(epi.bias + nb + 4));
                  const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                  for (int j = 0; j < 8; ++j) x[j] += Elem16<T>::round(bb[j]);
                }
                if (epi.mul != nullptr) {
                  const uint32_t mw[4] = {mv[c8].x, mv[c8].y, mv[c8].z, mv[c8].w};
#pragma unroll
                  for (int j = 0; j < 4; ++j) {
                    const float2 m2 = Elem16<T>::unpack2(mw[j]);
                    x[2 * j] *= m2.x;
                    x[2 * j + 1] *= m2.y;
                  }
                }
                st_shared_v4(row_base + buf + (((uint32_t)c8 ^ sw) << 4), Elem16<T>::pack2(x[0], x[1]), Elem16<T>::pack2(x[2], x[3]),
                             Elem16<T>::pack2(x[4], x[5]), Elem16<T>::pack2(x[6], x[7]));
              }
              fence_proxy_async_smem();
              __syncwarp();
              if (lane == 0) {
                if (store_ok) tma_store_2d(&tmap_c, my_stage + buf, n0, m_warp0);
                bulk_commit();
              }
              if (epi.colsum != nullptr && store_ok) {
                // bias gradient of the layer that produced A: column sums of the tile AS STORED (T), read back from
                // the staging buffer while the TMA store drains it; lane = column pair, conflict-free under the swizzle
                // (rows past M hold zeros: their A rows were zero-filled)
                float s0 = 0.f, s1 = 0.f;
                const uint32_t cbase = stage_u32 + buf + ((uint32_t)lane & 3u) * 4u;
#pragma unroll 8
                for (uint32_t r = 0; r < 32; ++r) {
                  const uint32_t wv = ld_shared_u32(cbase + r * 128u + ((((uint32_t)lane >> 2) ^ (r & 7u)) << 4));
                  const float2 v2 = Elem16<T>::unpack2(wv);
                  s0 += v2.x;
                  s1 += v2.y;
                }
                const int col = n0 + 2 * lane;
                if (col < g.N) {
                  atomicAdd(epi.colsum + col, s0);
                  atomicAdd(epi.colsum + col + 1, s1);
                }
              }
            }
          } else {
            // ---- fp32 C: two [32 rows][32 floats] boxes per 64-column chunk ----
            if (lane == 0) bulk_wait_read<0>();
            __syncwarp();
#pragma unroll
            for (int hb = 0; hb < 2; ++hb) {
#pragma unroll
              for (int c4 = 0; c4 < 8; ++c4) {
                float x[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) x[j] = f[hb * 32 + c4 * 4 + j];
                if (epi.bias != nullptr && first_split) {
                  const int nb = min(n0 + hb * 32 + c4 * 4, g.N - 4);
                  const float4 b0 = __ldg(reinterpret_cast<const float4*>(epi.bias + nb));
                  x[0] += Elem16<T>::round(b0.x); x[1] += Elem16<T>::round(b0.y); x[2] += Elem16<T>::round(b0.z); x[3] += Elem16<T>::round(b0.w);
                }
                st_shared_v4(row_base + hb * 4096u + (((uint32_t)c4 ^ sw) << 4), __float_as_uint(x[0]), __float_as_uint(x[1]),
                             __float_as_uint(x[2]), __float_as_uint(x[3]));
              }
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              if (store_ok) {
#pragma unroll
                for (int hb = 0; hb < 2; ++hb) {
                  if (n0 + hb * 32 < g.N) {
                    if (epi.reduce) tma_reduce_add_2d(&tmap_c, my_stage + hb * 4096, n0 + hb * 32, m_warp0);
                    else tma_store_2d(&tmap_c, my_stage + hb * 4096, n0 + hb * 32, m_warp0);
                  }
                }
              }
              bulk_commit();
            }
          }
          ++chunk_counter;
        }
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    if constexpr (Epi::kTma || Epi::kPlaneStore) {
      if (lane == 0) bulk_wait<0>();  // all stores of this warp have been written
    }
  }
  __syncwarp();
  tc_fence_before();
  cluster_sync();  // nobody signals the peer's barriers / reads its shared memory after this point
  if (warp == 1) tmem_dealloc_pair(tmem_base, kTmemCols);
}

template <int BN, int STG>
constexpr size_t pair_smem_bytes() {
  constexpr int stage = kPM * kPK * 2 + (BN / 2) * kPK * 2;
  constexpr int stages = (kSmemBudget - 1024 - kEpiWarps * STG - 512) / stage;
  return 1024 + (size_t)stages * stage + kEpiWarps * STG + 512;
}

// Pick the k-split count for accumulate/reduce GEMMs so that the work units fill whole waves of clusters.
int pick_splits(int tiles, int num_k, int clusters) {
  if (tiles >= 2 * clusters) return 1;
  int best = 1;
  double best_cost = 1e30;
  const int max_s = num_k / 8 > 0 ? num_k / 8 : 1;
  for (int s = 1; s <= max_s && s <= 64; ++s) {
    const int units = tiles * s;
    const int waves = (units + clusters - 1) / clusters;
    // cost ~ time: waves x per-unit k-work, plus a per-unit epilogue charge (~6 k-blocks worth)
    const double cost = (double)waves * ((double)num_k / s + 6.0);
    if (cost < best_cost - 1e-9) { best_cost = cost; best = s; }
  }
  return best;
}

// Launch on prebuilt maps (tc3_: a third output map, read by the SwiGLU forward only).
template <typename T, int BN, bool A_MN, bool B_MN, class Epi>
int launch_pair_maps(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc_, const CUtensorMap& tc2_,
                     const CUtensorMap& tc3_, const PairShape& g, const Epi& epi, cudaStream_t st) {
  constexpr size_t smem = pair_smem_bytes<BN, Staging<Epi>::kBytes>();
  auto kern = gemm_pair_kernel<T, BN, A_MN, B_MN, Epi>;
  VRR_SMEM_ATTR_ONCE(kern, smem);
  const int clusters_max = sm_count() / 2;
  const long long units = (long long)g.tiles_m * g.tiles_n * g.splits;
  const int clusters = (int)(units < clusters_max ? units : clusters_max);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * clusters);
  cfg.blockDim = dim3(kPairThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  VRR_CUDA(cudaLaunchKernelEx(&cfg, kern, ta, tb, tc_, tc2_, tc3_, g, epi));
  VRR_LAUNCHED();
  return VRR_OK;
}

template <typename T, int BN, bool A_MN, bool B_MN, class Epi>
int launch_pair(const void* a, const void* b, int M, int N, int K, int splits, const CUtensorMap& tc_, const CUtensorMap& tc2_,
                const Epi& epi, cudaStream_t st) {
  CUtensorMap ta, tb;
  if (!A_MN) { if (int rc = make_tmap_2d(&ta, a, Elem16<T>::kTmap, (uint64_t)M, (uint64_t)K, (uint64_t)K * 2, kPM, 64)) return rc; }
  else       { if (int rc = make_tmap_2d(&ta, a, Elem16<T>::kTmap, (uint64_t)K, (uint64_t)M, (uint64_t)M * 2, 64, 64)) return rc; }
  if (!B_MN) { if (int rc = make_tmap_2d(&tb, b, Elem16<T>::kTmap, (uint64_t)N, (uint64_t)K, (uint64_t)K * 2, BN / 2, 64)) return rc; }
  else       { if (int rc = make_tmap_2d(&tb, b, Elem16<T>::kTmap, (uint64_t)K, (uint64_t)N, (uint64_t)N * 2, 64, 64)) return rc; }
  PairShape g;
  g.M = M; g.N = N; g.K = K;
  g.tiles_m = ceil_div(M, 2 * kPM);
  g.tiles_n = ceil_div(N, BN);
  g.num_k = ceil_div(K, kPK);
  g.splits = splits < 1 ? 1 : (splits > g.num_k ? g.num_k : splits);
  return launch_pair_maps<T, BN, A_MN, B_MN, Epi>(ta, tb, tc_, tc2_, tc2_, g, epi, st);
}

template <typename T, bool A_MN, bool B_MN>
int launch_store(const void* a, const void* b, void* c, void* c2, const float* bias, int M, int N, int K, int c_f32,
                 int epilogue, int accumulate, float* colsum, cudaStream_t st) {
  StoreEpi<T> epi;
  epi.colsum = colsum;
  epi.bias = (epilogue != VRR_EPI_NONE && epilogue != VRR_EPI_MUL) ? bias : nullptr;
  epi.out_f32 = c_f32;
  epi.gelu = epilogue == VRR_EPI_BIAS_GELU ? 1 : (epilogue == VRR_EPI_BIAS_GELU_GRAD ? 2 : (epilogue == VRR_EPI_BIAS_GELU_ACT ? 3 : 0));
  epi.mul = epilogue == VRR_EPI_MUL ? (const T*)c2 : nullptr;
  if (epilogue == VRR_EPI_MUL) epi.bias = nullptr;
  const int tiles = ceil_div(M, 2 * kPM) * ceil_div(N, N > 128 ? 256 : 128);
  int splits = 1;
  if (c_f32) splits = pick_splits(tiles, ceil_div(K, kPK), sm_count() / 2);
  epi.reduce = (c_f32 && (accumulate || splits > 1)) ? 1 : 0;
  if (c_f32 && !accumulate && splits > 1) VRR_CUDA(cudaMemsetAsync(c, 0, (size_t)M * N * sizeof(float), st));
  CUtensorMap tc_, tc2_;
  if (c_f32) {
    if (int rc = make_tmap_2d(&tc_, c, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (uint64_t)M, (uint64_t)N, (uint64_t)N * 4, 32, 32)) return rc;
    tc2_ = tc_;
  } else {
    if (int rc = make_tmap_2d(&tc_, c, Elem16<T>::kTmap, (uint64_t)M, (uint64_t)N, (uint64_t)N * 2, 32, 64)) return rc;
    tc2_ = tc_;
    if (epi.gelu == 1 || epi.gelu == 2)
      if (int rc = make_tmap_2d(&tc2_, c2, Elem16<T>::kTmap, (uint64_t)M, (uint64_t)N, (uint64_t)N * 2, 32, 64)) return rc;
  }
  if (N > 128) return launch_pair<T, 256, A_MN, B_MN, StoreEpi<T>>(a, b, M, N, K, splits, tc_, tc2_, epi, st);
  return launch_pair<T, 128, A_MN, B_MN, StoreEpi<T>>(a, b, M, N, K, splits, tc_, tc2_, epi, st);
}

template <typename T>
int launch_store_drop(const void* a, const void* b, void* c, void* c2, const float* bias, int M, int N, int K, int epilogue,
                      const DropView& dv, cudaStream_t st) {
  StoreEpiDrop<T> epi = {};
  epi.bias = bias;
  epi.gelu = epilogue == VRR_EPI_BIAS_GELU_GRAD ? 2 : 3;
  epi.dv = dv;
  CUtensorMap tc_, tc2_;
  if (int rc = make_tmap_2d(&tc_, c, Elem16<T>::kTmap, (uint64_t)M, (uint64_t)N, (uint64_t)N * 2, 32, 64)) return rc;
  tc2_ = tc_;
  if (epi.gelu == 2)
    if (int rc = make_tmap_2d(&tc2_, c2, Elem16<T>::kTmap, (uint64_t)M, (uint64_t)N, (uint64_t)N * 2, 32, 64)) return rc;
  if (N > 128) return launch_pair<T, 256, false, false, StoreEpiDrop<T>>(a, b, M, N, K, 1, tc_, tc2_, epi, st);
  return launch_pair<T, 128, false, false, StoreEpiDrop<T>>(a, b, M, N, K, 1, tc_, tc2_, epi, st);
}

// unfold(images)[m][k], m = b*Np + py*gw + px, k = c*P*P + i*P + j  ->  TO (bf16 / fp16); 8 consecutive j per thread
template <typename TI, typename TO>
__global__ void patch_unfold_kernel(const TI* __restrict__ img, TO* __restrict__ out, int B, int C, int Hi,
                                    int Wi, int P, int gw, int Np) {
  const int K8 = C * P * P / 8;
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)B * Np * K8) return;
  const int k8 = (int)(idx % K8);
  const size_t m = idx / K8;
  const int b = (int)(m / Np), p = (int)(m - (size_t)b * Np), py = p / gw, px = p - py * gw;
  const int k = k8 * 8, c = k / (P * P), r = k - c * P * P, i = r / P, j = r - i * P;
  const TI* src = img + (((size_t)b * C + c) * Hi + (py * P + i)) * Wi + (px * P + j);
  float4 lo = ld4(src), hi = ld4(src + 4);
  TO* dst = out + m * (size_t)(K8 * 8) + k;
  st4(dst, lo);
  st4(dst + 4, hi);
}

}  // namespace

// 16-bit operands; TMA needs 16-byte row strides: the CONTIGUOUS dimension of every operand and of C must be a
// multiple of 8 elements (4 for an fp32 C); the other dimensions are free (ragged tiles are zero-filled / clipped).
// A 16-bit C has the operands' type.
bool gemm_tc_supported(int M, int N, int K, int trans_a, int trans_b, int dtype, int c_dtype, int epilogue) {
  if (M < 1 || N < 1 || K < 1) return false;
  if (!is16(dtype)) return false;
  if ((trans_a ? M : K) % 8 != 0) return false;   // A stored [K][M] or [M][K]
  if ((trans_b ? K : N) % 8 != 0) return false;   // B stored [N][K] or [K][N]
  if (c_dtype == dtype ? (N % 8 != 0) : (N % 4 != 0)) return false;
  if (c_dtype != VRR_F32 && c_dtype != dtype) return false;
  if (epilogue >= VRR_EPI_BIAS_GELU && c_dtype != dtype) return false;
  if (epilogue != VRR_EPI_NONE && N % 8 != 0) return false;  // vector loads of the bias / the multiplier
  if ((long long)M * N >= (1ll << 40)) return false;
  return true;
}

template <typename T>
static int gemm_tc_t(const void* a, const void* b, void* c, void* c2, const float* bias, int M, int N, int K, int trans_a,
                     int trans_b, int c_f32, int epilogue, int accumulate, cudaStream_t st, float* colsum) {
  const bool a_mn = trans_a != 0, b_mn = trans_b == 0;
  if (!a_mn && !b_mn) return launch_store<T, false, false>(a, b, c, c2, bias, M, N, K, c_f32, epilogue, accumulate, colsum, st);
  if (!a_mn && b_mn) return launch_store<T, false, true>(a, b, c, c2, bias, M, N, K, c_f32, epilogue, accumulate, colsum, st);
  if (a_mn && b_mn) return launch_store<T, true, true>(a, b, c, c2, bias, M, N, K, c_f32, epilogue, accumulate, colsum, st);
  return launch_store<T, true, false>(a, b, c, c2, bias, M, N, K, c_f32, epilogue, accumulate, colsum, st);
}

int gemm_tc(const void* a, const void* b, void* c, void* c2, const float* bias, int M, int N, int K, int trans_a,
            int trans_b, int dtype, int c_dtype, int epilogue, int accumulate, cudaStream_t st, float* colsum) {
  VRR_REQUIRE(is16(dtype) && (c_dtype == VRR_F32 || c_dtype == dtype), VRR_ERR_UNSUPPORTED,
              "gemm (tcgen05): operands must be bf16 or fp16 and C fp32 or the operands' type (got %d / %d)", dtype, c_dtype);
  VRR_REQUIRE(colsum == nullptr || (c_dtype == dtype && epilogue != VRR_EPI_BIAS_GELU && epilogue != VRR_EPI_BIAS_GELU_GRAD &&
                                    epilogue != VRR_EPI_BIAS_GELU_ACT),
              VRR_ERR_UNSUPPORTED, "gemm (tcgen05): column sums come with the 16-bit plain / bias / multiply epilogues only");
  VRR_REQUIRE((((uintptr_t)a | (uintptr_t)b | (uintptr_t)c | (uintptr_t)c2) & 15) == 0, VRR_ERR_INVALID_ARG,
              "gemm (tcgen05): a / b / c must be 16-byte aligned");
  VRR_REQUIRE(epilogue == VRR_EPI_NONE || epilogue == VRR_EPI_MUL || (bias != nullptr && ((uintptr_t)bias & 15) == 0),
              VRR_ERR_INVALID_ARG, "gemm (tcgen05): the bias epilogues need a 16-byte aligned fp32 bias");
  VRR_REQUIRE(epilogue < VRR_EPI_BIAS_GELU || epilogue == VRR_EPI_BIAS_GELU_ACT || c2 != nullptr, VRR_ERR_INVALID_ARG,
              "gemm (tcgen05): the two-output GELU epilogues and MUL need c2");
  VRR_REQUIRE(!accumulate || c_dtype == VRR_F32, VRR_ERR_UNSUPPORTED, "gemm (tcgen05): accumulate needs an fp32 C");
  const int c_f32 = c_dtype == VRR_F32;
  if (dtype == VRR_F16)
    return gemm_tc_t<__half>(a, b, c, c2, bias, M, N, K, trans_a, trans_b, c_f32, epilogue, accumulate, st, colsum);
  return gemm_tc_t<__nv_bfloat16>(a, b, c, c2, bias, M, N, K, trans_a, trans_b, c_f32, epilogue, accumulate, st, colsum);
}

int gemm_tc_drop(const void* a, const void* b, void* c, void* c2, const float* bias, int M, int N, int K, int dtype,
                 int epilogue, const DropView& dv, cudaStream_t st) {
  VRR_REQUIRE(is16(dtype) && (epilogue == VRR_EPI_BIAS_GELU_GRAD || epilogue == VRR_EPI_BIAS_GELU_ACT), VRR_ERR_UNSUPPORTED,
              "gemm (tcgen05, dropout): 16-bit operands and the BIAS_GELU_GRAD / BIAS_GELU_ACT epilogues only");
  VRR_REQUIRE(gemm_tc_supported(M, N, K, 0, 1, dtype, dtype, epilogue), VRR_ERR_UNSUPPORTED,
              "gemm (tcgen05, dropout): unsupported shape M=%d N=%d K=%d", M, N, K);
  if (dtype == VRR_F16) return launch_store_drop<__half>(a, b, c, c2, bias, M, N, K, epilogue, dv, st);
  return launch_store_drop<__nv_bfloat16>(a, b, c, c2, bias, M, N, K, epilogue, dv, st);
}

// ---- SwiGLU Mlp: fc1 with the gated activation, fc2's dX with its backward ----------------------------------
template <typename T, bool DROP>
static int swiglu_tc_t(const void* x, const void* w1, const float* b1, void* act, void* aux, int M, int H, int K,
                       const DropView& dv, cudaStream_t st) {
  SwiGluEpi<T, DROP> epi = {};
  epi.bias = b1;
  epi.with_aux = aux != nullptr;
  epi.dv = dv;
  CUtensorMap ta, tb, tc_, tc2_, tc3_;
  if (int rc = make_tmap_2d(&ta, x, Elem16<T>::kTmap, (uint64_t)M, (uint64_t)K, (uint64_t)K * 2, kPM, 64)) return rc;
  // w1 [2][H][K]: box [1][128 rows][64]; plane 0 = gate rows, plane 1 = value rows
  if (int rc = make_tmap_3d(&tb, w1, Elem16<T>::kTmap, (uint64_t)K, (uint64_t)H, 2, (uint64_t)K * 2, (uint64_t)H * K * 2, 64, 128))
    return rc;
  if (int rc = make_tmap_2d(&tc_, act, Elem16<T>::kTmap, (uint64_t)M, (uint64_t)H, (uint64_t)H * 2, 32, 64)) return rc;
  tc2_ = tc3_ = tc_;
  if (aux) {
    if (int rc = make_tmap_2d(&tc2_, aux, Elem16<T>::kTmap, (uint64_t)M, (uint64_t)H, (uint64_t)H * 4, 32, 64)) return rc;
    if (int rc = make_tmap_2d(&tc3_, (const T*)aux + H, Elem16<T>::kTmap, (uint64_t)M, (uint64_t)H, (uint64_t)H * 4, 32, 64))
      return rc;
  }
  PairShape g;
  g.M = M; g.N = H; g.K = K;
  g.tiles_m = ceil_div(M, 2 * kPM);
  g.tiles_n = ceil_div(H, 128);
  g.num_k = ceil_div(K, kPK);
  g.splits = 1;
  return launch_pair_maps<T, 256, false, false, SwiGluEpi<T, DROP>>(ta, tb, tc_, tc2_, tc3_, g, epi, st);
}

int gemm_tc_swiglu(const void* x, const void* w1, const float* b1, void* act, void* aux, int M, int H, int K, int dtype,
                   const DropView* dv, cudaStream_t st) {
  if (dtype == VRR_F16) {
    if (dv) return swiglu_tc_t<__half, true>(x, w1, b1, act, aux, M, H, K, *dv, st);
    return swiglu_tc_t<__half, false>(x, w1, b1, act, aux, M, H, K, DropView{}, st);
  }
  if (dv) return swiglu_tc_t<__nv_bfloat16, true>(x, w1, b1, act, aux, M, H, K, *dv, st);
  return swiglu_tc_t<__nv_bfloat16, false>(x, w1, b1, act, aux, M, H, K, DropView{}, st);
}

template <typename T>
static int swiglu_bwd_tc_t(const void* dy, const void* w2, const void* aux, void* dh, float* db1, int M, int H, int K,
                           cudaStream_t st) {
  SwiGluBwdEpi<T> epi{(const T*)aux, db1};
  CUtensorMap tc_, tc2_;  // the halves of dh [M][2H]
  if (int rc = make_tmap_2d(&tc_, dh, Elem16<T>::kTmap, (uint64_t)M, (uint64_t)H, (uint64_t)H * 4, 32, 64)) return rc;
  if (int rc = make_tmap_2d(&tc2_, (T*)dh + H, Elem16<T>::kTmap, (uint64_t)M, (uint64_t)H, (uint64_t)H * 4, 32, 64)) return rc;
  VRR_CUDA(cudaMemsetAsync(db1, 0, (size_t)2 * H * sizeof(float), st));
  // dA = dy [M][K] . w2 [K][H]: w2 is fc2.weight, stored [K][N] (B_MN)
  if (H > 128) return launch_pair<T, 256, false, true, SwiGluBwdEpi<T>>(dy, w2, M, H, K, 1, tc_, tc2_, epi, st);
  return launch_pair<T, 128, false, true, SwiGluBwdEpi<T>>(dy, w2, M, H, K, 1, tc_, tc2_, epi, st);
}

int gemm_tc_swiglu_bwd(const void* dy, const void* w2, const void* aux, void* dh, float* db1, int M, int H, int K, int dtype,
                       cudaStream_t st) {
  if (dtype == VRR_F16) return swiglu_bwd_tc_t<__half>(dy, w2, aux, dh, db1, M, H, K, st);
  return swiglu_bwd_tc_t<__nv_bfloat16>(dy, w2, aux, dh, db1, M, H, K, st);
}

// ---- QKV projection + RoPE epilogue on the CTA-pair kernel -----------------------------------------------
bool qkv_rope_fwd_tc_supported(int B, int N, int E, int H) {
  if (H <= 0 || E % H != 0 || E / H != 64) return false;
  if ((long long)B * N >= (1ll << 31) / 4) return false;
  return true;
}

template <typename T>
static int qkv_rope_fwd_tc2_t(const void* x, const void* w, const float* cos_tab, const float* sin_tab, const float* packed,
                              void* planes, int B, int N, int E, int H, int npre, int rope_mode, cudaStream_t st) {
  QkvRopeEpi2<T> epi{(T*)planes, cos_tab, sin_tab, reinterpret_cast<const float4*>(packed), B, N, E, H, rope_mode, npre};
  CUtensorMap tplanes;  // planes[3 B H][N][64] of T, box = [1][32 rows][64]
  if (int rc = make_tmap_3d(&tplanes, planes, Elem16<T>::kTmap, 64, (uint64_t)N, (uint64_t)3 * B * H, 128, (uint64_t)N * 128,
                            64, 32))
    return rc;
  // 64-column chunks are whole heads (3E = 192 H); a ragged last n-tile is clipped by the n0 < N test
  if (3 * E > 128) return launch_pair<T, 256, false, false, QkvRopeEpi2<T>>(x, w, B * N, 3 * E, E, 1, tplanes, tplanes, epi, st);
  return launch_pair<T, 128, false, false, QkvRopeEpi2<T>>(x, w, B * N, 3 * E, E, 1, tplanes, tplanes, epi, st);
}

template <typename T>
static int qkv_rope_norm_fwd_tc2_t(const void* x, const void* w, const float* cos_tab, const float* sin_tab,
                                   const float* packed, void* planes, int B, int N, int E, int H, int npre, int rope_mode,
                                   const QkNormArgs& qn, cudaStream_t st) {
  QkvNormRopeEpi2<T> epi{{(T*)planes, cos_tab, sin_tab, reinterpret_cast<const float4*>(packed), B, N, E, H, rope_mode, npre},
                         (T*)qn.qk_pre, reinterpret_cast<float2*>(qn.qk_stats), reinterpret_cast<const float4*>(qn.qn_w),
                         reinterpret_cast<const float4*>(qn.qn_b), reinterpret_cast<const float4*>(qn.kn_w),
                         reinterpret_cast<const float4*>(qn.kn_b), qn.eps};
  CUtensorMap tplanes, tpre;  // planes[3 B H][N][64] and qk_pre[2 B H][N][64] of T, box = [1][32 rows][64]
  if (int rc = make_tmap_3d(&tplanes, planes, Elem16<T>::kTmap, 64, (uint64_t)N, (uint64_t)3 * B * H, 128, (uint64_t)N * 128,
                            64, 32))
    return rc;
  tpre = tplanes;
  if (qn.qk_pre != nullptr)
    if (int rc = make_tmap_3d(&tpre, qn.qk_pre, Elem16<T>::kTmap, 64, (uint64_t)N, (uint64_t)2 * B * H, 128, (uint64_t)N * 128,
                              64, 32))
      return rc;
  if (3 * E > 128) return launch_pair<T, 256, false, false, QkvNormRopeEpi2<T>>(x, w, B * N, 3 * E, E, 1, tplanes, tpre, epi, st);
  return launch_pair<T, 128, false, false, QkvNormRopeEpi2<T>>(x, w, B * N, 3 * E, E, 1, tplanes, tpre, epi, st);
}

int qkv_rope_fwd_tc2(const void* x, const void* w, const float* cos_tab, const float* sin_tab, const float* packed,
                     void* planes, int B, int N, int E, int H, int npre, int rope_mode, int dtype, cudaStream_t st,
                     const QkNormArgs* qn) {
  VRR_REQUIRE(((uintptr_t)x & 15) == 0 && ((uintptr_t)w & 15) == 0 && ((uintptr_t)planes & 15) == 0,
              VRR_ERR_INVALID_ARG, "qkv_rope_fwd (tcgen05): x / w / planes must be 16-byte aligned");
  if (rope_mode != VRR_ROPE_NONE)
    VRR_REQUIRE(((uintptr_t)cos_tab & 15) == 0 && ((uintptr_t)sin_tab & 15) == 0, VRR_ERR_INVALID_ARG,
                "qkv_rope_fwd (tcgen05): cos / sin must be 16-byte aligned");
  VRR_REQUIRE(((uintptr_t)packed & 15) == 0, VRR_ERR_INVALID_ARG, "qkv_rope_fwd (tcgen05): packed table must be 16-byte aligned");
  if (qn != nullptr) {
    VRR_REQUIRE((((uintptr_t)qn->qn_w | (uintptr_t)qn->qn_b | (uintptr_t)qn->kn_w | (uintptr_t)qn->kn_b | (uintptr_t)qn->qk_pre) & 15) == 0 &&
                    ((uintptr_t)qn->qk_stats & 7) == 0,
                VRR_ERR_INVALID_ARG, "qkv_rope_norm_fwd (tcgen05): norm tensors and qk_pre must be 16-byte aligned, qk_stats 8");
    if (dtype == VRR_F16)
      return qkv_rope_norm_fwd_tc2_t<__half>(x, w, cos_tab, sin_tab, packed, planes, B, N, E, H, npre, rope_mode, *qn, st);
    return qkv_rope_norm_fwd_tc2_t<__nv_bfloat16>(x, w, cos_tab, sin_tab, packed, planes, B, N, E, H, npre, rope_mode, *qn, st);
  }
  if (dtype == VRR_F16) return qkv_rope_fwd_tc2_t<__half>(x, w, cos_tab, sin_tab, packed, planes, B, N, E, H, npre, rope_mode, st);
  return qkv_rope_fwd_tc2_t<__nv_bfloat16>(x, w, cos_tab, sin_tab, packed, planes, B, N, E, H, npre, rope_mode, st);
}

// ---- patch embedding: unfold pre-pass (fused fp32 -> 16-bit cast) + the CTA-pair kernel -------------------
bool patch_embed_tc_supported(int B, int C, int Hi, int Wi, int P, int E) {
  const int K = C * P * P;
  if (P % 8 != 0 || Wi % 4 != 0 || K % 64 != 0 || E % 64 != 0) return false;
  if ((long long)B * (Hi / P) * (Wi / P) >= (1ll << 31) / 4) return false;
  return true;
}
size_t patch_embed_tc_workspace_bytes(int B, int C, int Hi, int Wi, int P) {
  return (size_t)B * (Hi / P) * (Wi / P) * C * P * P * 2;
}
int patch_unfold(const void* images, void* out, int B, int C, int Hi, int Wi, int P, int img_dtype, int out_dtype,
                 cudaStream_t st) {
  const int gw = Wi / P, Np = (Hi / P) * gw;
  VRR_REQUIRE(P % 8 == 0 && Wi % 4 == 0, VRR_ERR_UNSUPPORTED, "patch_unfold: needs P %% 8 == 0 and Wi %% 4 == 0");
  VRR_REQUIRE(((uintptr_t)images & 15) == 0 && ((uintptr_t)out & 15) == 0, VRR_ERR_INVALID_ARG,
              "patch_unfold: pointers must be 16-byte aligned");
  VRR_REQUIRE(is16(out_dtype) && (img_dtype == VRR_F32 || img_dtype == out_dtype), VRR_ERR_INVALID_ARG,
              "patch_unfold: images %d cannot be unfolded into dtype %d", img_dtype, out_dtype);
  const size_t total = (size_t)B * Np * (C * P * P / 8);
  const unsigned blocks = (unsigned)((total + 255) / 256);
  if (out_dtype == VRR_BF16) {
    if (img_dtype == VRR_F32)
      patch_unfold_kernel<float, __nv_bfloat16><<<blocks, 256, 0, st>>>((const float*)images, (__nv_bfloat16*)out, B, C, Hi,
                                                                         Wi, P, gw, Np);
    else
      patch_unfold_kernel<__nv_bfloat16, __nv_bfloat16><<<blocks, 256, 0, st>>>((const __nv_bfloat16*)images,
                                                                                 (__nv_bfloat16*)out, B, C, Hi, Wi, P, gw, Np);
  } else {
    if (img_dtype == VRR_F32)
      patch_unfold_kernel<float, __half><<<blocks, 256, 0, st>>>((const float*)images, (__half*)out, B, C, Hi, Wi, P, gw, Np);
    else
      patch_unfold_kernel<__half, __half><<<blocks, 256, 0, st>>>((const __half*)images, (__half*)out, B, C, Hi, Wi, P, gw, Np);
  }
  VRR_LAUNCHED();
  return VRR_OK;
}

template <typename T, typename TT>
static int patch_embed_gemm(const void* workspace, const void* weight, const void* bias, const void* pos, void* tokens, int M,
                            int E, int K, int Np, int npre, cudaStream_t st) {
  CUtensorMap dummy;  // PatchEmbedEpi2 stores its rows directly: no C map
  memset(&dummy, 0, sizeof(dummy));
  PatchEmbedEpi2<T, TT> epi{(TT*)tokens + (size_t)npre * E, (const T*)bias, (const TT*)pos, Np, E, Np + npre};
  if (E > 128) return launch_pair<T, 256, false, false, PatchEmbedEpi2<T, TT>>(workspace, weight, M, E, K, 1, dummy, dummy, epi, st);
  return launch_pair<T, 128, false, false, PatchEmbedEpi2<T, TT>>(workspace, weight, M, E, K, 1, dummy, dummy, epi, st);
}

int patch_embed_fwd_tc(const void* images, const void* weight, const void* bias, const void* pos, void* tokens,
                       void* workspace, int B, int C, int Hi, int Wi, int P, int E, int npre, int img_dtype, int dtype,
                       int tok_dtype, cudaStream_t st) {
  const int Np = (Hi / P) * (Wi / P), K = C * P * P, M = B * Np;
  if (int rc = patch_unfold(images, workspace, B, C, Hi, Wi, P, img_dtype, dtype, st)) return rc;
  if (dtype == VRR_F16) {
    if (tok_dtype == VRR_F32) return patch_embed_gemm<__half, float>(workspace, weight, bias, pos, tokens, M, E, K, Np, npre, st);
    return patch_embed_gemm<__half, __half>(workspace, weight, bias, pos, tokens, M, E, K, Np, npre, st);
  }
  if (tok_dtype == VRR_F32) return patch_embed_gemm<__nv_bfloat16, float>(workspace, weight, bias, pos, tokens, M, E, K, Np, npre, st);
  return patch_embed_gemm<__nv_bfloat16, __nv_bfloat16>(workspace, weight, bias, pos, tokens, M, E, K, Np, npre, st);
}

}  // namespace vrr
