// SIMT (FFMA) tiled GEMM with pluggable operand loaders and epilogues.
//
// fp32 product path for the three projections on the hot path (tcgen05 has no fp32 MMA and the
// fp32 parity bar is 1e-5), and the bf16 path for shapes the tcgen05 GEMM does not cover:
//   * QKV projection with the RoPE rotate-half epilogue writing [3][B][H][N][Dh] planes
//     (models/vit.py:47-68 + models/rope_utils.py:22-35 in one kernel);
//   * patch embedding as unfold(im2col-on-the-fly) x weight^T + bias (+ absolute pos_embed),
//     written straight into token rows 1.. (models/vit.py:164,248-258);
//   * the plain GEMMs of the projection backward (dX, dW) and the patch-embed weight gradient.
//
// 64x64 output tile, BK = 16, 256 threads, 4x4 register micro-tile, fp32 accumulation.
#include <type_traits>

#include "common.cuh"
#include "kernels.h"

namespace vrr {

constexpr int BM = 64, BN = 64, BK = 16, GT = 256;
constexpr int LDS_ = BM + 4;  // padded leading dimension of the k-major operand tiles

// ---- operand loaders: element (row, k) of a logical [rows][K] operand ---------------------------
template <typename T>
struct StridedOperand {
  const T* p;
  long long s_row, s_k;
  __device__ __forceinline__ float operator()(int r, int k) const {
    return Elem<T>::ld(p + (long long)r * s_row + (long long)k * s_k);
  }
  // four consecutive elements along the contiguous dimension (k when s_k == 1, the row index when s_row == 1)
  static constexpr bool kVec = true;
  __device__ __forceinline__ bool vec_ok() const {
    const long long other = s_k == 1 ? s_row : s_k;
    return (s_k == 1 || s_row == 1) && (other & 3) == 0 && ((uintptr_t)p & 15) == 0;
  }
  __device__ __forceinline__ float4 ld4k(int r, int k) const { return ld4(p + (long long)r * s_row + k); }   // s_k == 1
  __device__ __forceinline__ float4 ld4r(int r, int k) const { return ld4(p + (long long)k * s_k + r); }     // s_row == 1
};

// A[m][k] of unfold(images): m = b*Np + p (p = py*gw + px), k = c*P*P + i*P + j
// TI = storage type of the images; ROUND = round each pixel to bf16 first (bf16 arithmetic on fp32
// images, i.e. the reference's autocast cast of the conv input fused into the load).
// ROUND: the image is rounded to the conv dtype TR on load (fp32 images under autocast)
template <typename TI, bool ROUND, typename TR>
struct Im2colOperand {
  static constexpr bool kVec = false;
  const TI* img;
  int C, Hi, Wi, P, gw, Np;
  __device__ __forceinline__ float operator()(int m, int k) const {
    int b = m / Np, p = m - b * Np, py = p / gw, px = p - py * gw;
    int c = k / (P * P), r = k - c * P * P, i = r / P, j = r - i * P;
    float v = Elem<TI>::ld(img + (((long long)b * C + c) * Hi + (py * P + i)) * Wi + (px * P + j));
    return ROUND ? Elem<TR>::round(v) : v;
  }
};

// A'[e][m] = d_tokens[b][npre+p][e] for the patch-embed weight gradient (m = b*Np + p)
template <typename T>
struct PatchGradOperand {
  static constexpr bool kVec = false;
  const T* dtok;
  int Np, E, rows;  // rows = npre + Np token rows per image; dtok points at row npre of image 0
  __device__ __forceinline__ float operator()(int e, int m) const {
    int b = m / Np, p = m - b * Np;
    return Elem<T>::ld(dtok + ((long long)b * rows + p) * E + e);
  }
};

template <typename Inner>
struct SwapArgs {  // view an operand (r,k) as (k,r)
  static constexpr bool kVec = false;
  Inner in;
  __device__ __forceinline__ float operator()(int r, int k) const { return in(k, r); }
};

// ---- epilogues ------------------------------------------------------------------------------
template <typename T>
struct StoreEpilogue {
  T* c;
  long long ldc;
  __device__ __forceinline__ void operator()(int m, int n, float v, const float*, int) const {
    Elem<T>::st(c + (long long)m * ldc + n, v);
  }
};
// Linear-layer epilogue: c = round_T(acc + bias[n]) (bias cast to T first, like F.linear on T tensors);
// optionally c2 = gelu(c) with the exact erf GELU.
template <typename T>
struct BiasEpilogue {
  T* c;
  T* c2;
  const float* bias;
  long long ldc;
  int gelu;
  __device__ __forceinline__ void operator()(int m, int n, float v, const float*, int) const {
    float b = bias[n];
    if (sizeof(T) == 2) b = Elem<T>::round(b);
    T r;
    Elem<T>::st(&r, v + b);
    if (gelu != 2) c[(long long)m * ldc + n] = r;
    if (gelu) {  // 1: c = h, c2 = gelu(h);  2: c = gelu(h) only (inference)
      const float h = Elem<T>::ld(&r);
      Elem<T>::st((gelu == 2 ? c : c2) + (long long)m * ldc + n, 0.5f * h * (1.f + erff(h * 0.70710678118654752f)));
    }
  }
};
struct AtomicEpilogue {  // split-K accumulation into a zeroed fp32 C
  float* c;
  long long ldc;
  __device__ __forceinline__ void operator()(int m, int n, float v, const float*, int) const {
    atomicAdd(c + (long long)m * ldc + n, v);
  }
};

template <typename T>
struct QkvRopeEpilogue {
  static constexpr bool kRowPrep = false;
  T* planes;
  const float *cos_tab, *sin_tab;
  int B, N, E, H, Dh, rope_mode;
  int npre, rows;  // prefix tokens (never rotated); row t >= npre uses table row t - npre of rows = N - npre
  __device__ __forceinline__ void operator()(int m, int n, float v, const float* crow, int n0) const {
    const int which = n / E, r = n - which * E, h = r / Dh, d = r - h * Dh;
    const int b = m / N, t = m - b * N;
    if (rope_mode != VRR_ROPE_NONE && which < 2 && t >= npre) {
      const int hd = Dh >> 1, dd = d < hd ? d : d - hd;
      const size_t idx = ((size_t)(rope_mode == VRR_ROPE_MIXED ? h * rows : 0) + (t - npre)) * hd + dd;
      const float c = cos_tab[idx], s = sin_tab[idx];
      const float other = crow[(d < hd ? n + hd : n - hd) - n0];
      v = d < hd ? v * c - other * s : other * s + v * c;
    }
    Elem<T>::st(planes + ((((size_t)which * B + b) * H + h) * N + t) * Dh + d, v);
  }
};

// QkvRopeEpilogue with QK-norm (vrr_qkv_rope_norm_fwd).  prep() runs once per (row, head) of the staged tile before
// the per-element pass: for a q / k head it rounds the Dh accumulators to T (x), saves x and {mean, rstd}, and
// overwrites the staged row with y = xhat g + b, which the per-element pass then rotates and stores.
template <typename T>
struct QkvNormRopeEpilogue : QkvRopeEpilogue<T> {
  static constexpr bool kRowPrep = true;
  QkNormArgs qn;
  __device__ __forceinline__ void prep(int m, int n, float* seg) const {
    const int Dh = this->Dh, which = n / this->E;
    if (which == 2) return;
    const int h = (n - which * this->E) / Dh, b = m / this->N, t = m - b * this->N;
    for (int j = 0; j < Dh; ++j) seg[j] = Elem<T>::round(seg[j]);
    const float2 st = qk_norm_stats(seg, Dh, qn.eps);
    const size_t row = (((size_t)which * this->B + b) * this->H + h) * this->N + t;
    if (qn.qk_pre != nullptr) {
      T* pre = (T*)qn.qk_pre + row * Dh;
      for (int j = 0; j < Dh; ++j) Elem<T>::st(pre + j, seg[j]);
      reinterpret_cast<float2*>(qn.qk_stats)[row] = st;
    }
    const float *g = which ? qn.kn_w : qn.qn_w, *bb = which ? qn.kn_b : qn.qn_b;
    for (int j = 0; j < Dh; ++j) seg[j] = qk_norm_y(qk_norm_xhat(seg[j], st.x, st.y), g[j], bb[j]);
  }
};

// Epilogues with kRowPrep: prep(m, n, row segment) once per (row, head) of the staged tile (COLS columns, 64 rows),
// after the tile is in shared memory and before the per-element pass.
template <class Epi, class = void>
struct HasRowPrep { static constexpr bool value = false; };
template <class Epi>
struct HasRowPrep<Epi, std::void_t<decltype(Epi::kRowPrep)>> { static constexpr bool value = Epi::kRowPrep; };
template <class Epi, int COLS>
__device__ __forceinline__ void row_prep(const Epi& epi, float* Cs, int m0, int n0, int M, int N) {
  if constexpr (HasRowPrep<Epi>::value) {
    const int segs = COLS / epi.Dh;
    for (int s = threadIdx.x; s < 64 * segs; s += GT) {
      const int r = s / segs, c0 = (s - r * segs) * epi.Dh;
      if (m0 + r < M && n0 + c0 < N) epi.prep(m0 + r, n0 + c0, Cs + r * (COLS + 1) + c0);
    }
    __syncthreads();
  }
}

// T: element type of images / weight / bias (the conv arithmetic); TT: element type of the token
// stream (prefix tokens, pos_embed, tokens).  Under autocast T = bf16 and TT = fp32, which reproduces
// the reference's semantics: conv output rounded to bf16, then cat with the fp32 cls token promotes
// to fp32 and the absolute table is added in fp32 (vit.py:248-258).
template <typename T, typename TT>
struct PatchEmbedEpilogue {
  TT* tokens;
  const T* bias;
  const TT* pos;  // may be null
  int Np, E, npre;
  __device__ __forceinline__ void operator()(int m, int n, float v, const float*, int) const {
    const int b = m / Np, p = m - b * Np;
    T rounded;
    Elem<T>::st(&rounded, v + Elem<T>::ld(bias + n));  // conv (+bias) in the conv dtype
    float out = Elem<T>::ld(&rounded);
    if (pos) out += Elem<TT>::ld(pos + (size_t)p * E + n);
    Elem<TT>::st(tokens + ((size_t)b * (Np + npre) + npre + p) * E + n, out);
  }
};

// ---- kernel -----------------------------------------------------------------------------------
// C[m][n] = sum_k A(m,k) * Bop(n,k).  A_KC / B_KC: the operand is contiguous along k in memory
// (chooses the thread->element mapping of the global loads so that they coalesce).
template <typename AOp, typename BOp, typename Epi, bool A_KC, bool B_KC>
__global__ void __launch_bounds__(GT) gemm_simt_kernel(AOp A, BOp Bop, Epi epi, int M, int N, int K,
                                                       int k_per_split) {
  __shared__ __align__(16) float smem[BM * (BN + 1)];
  float* As = smem;               // [BK][LDS_]
  float* Bs = smem + BK * LDS_;   // [BK][LDS_]
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int k_begin = blockIdx.z * k_per_split, k_end = min(K, k_begin + k_per_split);
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int k0 = k_begin; k0 < k_end; k0 += BK) {
    // global -> shared (4 elements of each operand per thread)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      int r, k;
      if (A_KC) { r = tid >> 2; k = (tid & 3) * 4 + e; } else { r = (tid & 15) * 4 + e; k = tid >> 4; }
      float v = (m0 + r < M && k0 + k < k_end) ? A(m0 + r, k0 + k) : 0.f;
      As[k * LDS_ + r] = v;
      if (B_KC) { r = tid >> 2; k = (tid & 3) * 4 + e; } else { r = (tid & 15) * 4 + e; k = tid >> 4; }
      v = (n0 + r < N && k0 + k < k_end) ? Bop(n0 + r, k0 + k) : 0.f;
      Bs[k * LDS_ + r] = v;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      float4 a = *reinterpret_cast<const float4*>(As + k * LDS_ + ty * 4);
      float4 b = *reinterpret_cast<const float4*>(Bs + k * LDS_ + tx * 4);
      const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
  // stage the tile so that epilogues can see a whole output row (RoPE pairs d, d + Dh/2)
  float* Cs = smem;  // [BM][BN + 1]
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) Cs[(ty * 4 + i) * (BN + 1) + tx * 4 + j] = acc[i][j];
  __syncthreads();
  row_prep<Epi, BN>(epi, Cs, m0, n0, M, N);
  for (int e = tid; e < BM * BN; e += GT) {
    const int r = e / BN, c = e - r * BN;
    if (m0 + r < M && n0 + c < N) epi(m0 + r, n0 + c, Cs[r * (BN + 1) + c], Cs + r * (BN + 1), n0);
  }
}

// ---- 128 x 128 tile variant ------------------------------------------------------------------------
// The 64 x 64 kernel above is bound by shared-memory bandwidth (two LDS.128 per 16 FFMA) and by its scalar,
// un-pipelined global loads: 25 TFLOP/s on the ViT-Tiny shapes (8320 x 768 x 192), a third of the FFMA roof and
// slower than cuBLAS SGEMM - which made the fp32 configurations slower than the reference's own GPU path.  Here
// each thread owns an 8 x 8 micro-tile as 2 x 2 blocks of 4 x 4 (four LDS.128 per 64 FFMA), the operand tiles are
// double-buffered in shared memory with the next tile's global loads (128-bit when the operand is a plain
// row-major matrix) in flight during the FFMAs, and the output tile is staged 64 rows at a time for the row-aware
// epilogues.
constexpr int TM = 128, TN = 128, TK = 16;
constexpr int TLD = TM + 4;

// ROWS = 128 or 64 rows of the operand tile; every thread moves ROWS / 16 elements per k-tile.
//   KC  (operand contiguous along k): element e of half h -> (r = tid >> 2 + 64 h, k = 4 (tid & 3) + e)
//   !KC (contiguous along the row index): ROWS = 128: (r = 4 (tid & 31) + e, k = tid >> 5 + 8 h); ROWS = 64: (r = 4 (tid & 15) + e, k = tid >> 4)
template <typename Op, bool KC, int ROWS>
__device__ __forceinline__ void load_tile(const Op& op, bool vec, int row0, int nrows, int k0, int k_end, int tid,
                                          float (&reg)[ROWS / 16]) {
  constexpr int H = ROWS / 64;
#pragma unroll
  for (int h = 0; h < H; ++h) {
    int r, k;
    if (KC) { r = (tid >> 2) + h * 64; k = (tid & 3) * 4; }
    else if (ROWS == 128) { r = (tid & 31) * 4; k = (tid >> 5) + h * 8; }
    else { r = (tid & 15) * 4; k = tid >> 4; }
    bool done = false;
    if constexpr (Op::kVec) {
      if (vec && (KC ? (row0 + r < nrows && k0 + k + 3 < k_end) : (row0 + r + 3 < nrows && k0 + k < k_end))) {
        const float4 v = KC ? op.ld4k(row0 + r, k0 + k) : op.ld4r(row0 + r, k0 + k);
        reg[h * 4 + 0] = v.x; reg[h * 4 + 1] = v.y; reg[h * 4 + 2] = v.z; reg[h * 4 + 3] = v.w;
        done = true;
      }
    }
    if (!done) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int rr = KC ? r : r + e, kk = KC ? k + e : k;
        reg[h * 4 + e] = (row0 + rr < nrows && k0 + kk < k_end) ? op(row0 + rr, k0 + kk) : 0.f;
      }
    }
  }
}
template <bool KC, int ROWS>
__device__ __forceinline__ void store_tile(float* S, int tid, const float (&reg)[ROWS / 16]) {  // S: [TK][TLD], k-major
  constexpr int H = ROWS / 64;
#pragma unroll
  for (int h = 0; h < H; ++h) {
    if (KC) {
      const int r = (tid >> 2) + h * 64, k = (tid & 3) * 4;
#pragma unroll
      for (int e = 0; e < 4; ++e) S[(k + e) * TLD + r] = reg[h * 4 + e];
    } else {
      const int r = ROWS == 128 ? (tid & 31) * 4 : (tid & 15) * 4, k = ROWS == 128 ? (tid >> 5) + h * 8 : tid >> 4;
      *reinterpret_cast<float4*>(S + k * TLD + r) = make_float4(reg[h * 4], reg[h * 4 + 1], reg[h * 4 + 2], reg[h * 4 + 3]);
    }
  }
}

// NB = 1 or 2 blocks of 64 output columns (tile 128 x 64 or 128 x 128)
template <typename AOp, typename BOp, typename Epi, bool A_KC, bool B_KC, int NB>
__global__ void __launch_bounds__(GT, 2) gemm_simt128_kernel(AOp A, BOp Bop, Epi epi, int M, int N, int K, int k_per_split) {
  constexpr int TNN = 64 * NB;
  __shared__ __align__(16) float smem[4 * TK * TLD];  // A[2][TK][TLD] | B[2][TK][TLD]; reused as C staging [64][TNN + 1]
  static_assert(4 * TK * TLD >= 64 * (TN + 1), "C staging does not fit");
  float* As = smem;
  float* Bs = smem + 2 * TK * TLD;
  const int m0 = blockIdx.y * TM, n0 = blockIdx.x * TNN;
  const int k_begin = blockIdx.z * k_per_split, k_end = min(K, k_begin + k_per_split);
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  bool avec = false, bvec = false;
  if constexpr (AOp::kVec) avec = A.vec_ok() && (A_KC ? A.s_k == 1 : A.s_row == 1);
  if constexpr (BOp::kVec) bvec = Bop.vec_ok() && (B_KC ? Bop.s_k == 1 : Bop.s_row == 1);

  float acc[2][NB][4][4];
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < NB; ++b)
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[a][b][i][j] = 0.f;

  float ra[8], rb[4 * NB];
  load_tile<AOp, A_KC, 128>(A, avec, m0, M, k_begin, k_end, tid, ra);
  load_tile<BOp, B_KC, TNN>(Bop, bvec, n0, N, k_begin, k_end, tid, rb);
  store_tile<A_KC, 128>(As, tid, ra);
  store_tile<B_KC, TNN>(Bs, tid, rb);
  __syncthreads();
  int buf = 0;
  for (int k0 = k_begin; k0 < k_end; k0 += TK) {
    const bool more = k0 + TK < k_end;
    if (more) {  // next tile's global loads in flight during the FFMAs
      load_tile<AOp, A_KC, 128>(A, avec, m0, M, k0 + TK, k_end, tid, ra);
      load_tile<BOp, B_KC, TNN>(Bop, bvec, n0, N, k0 + TK, k_end, tid, rb);
    }
    const float* Ac = As + buf * TK * TLD;
    const float* Bc = Bs + buf * TK * TLD;
#pragma unroll
    for (int k = 0; k < TK; ++k) {
      float av[2][4], bv[NB][4];
#pragma unroll
      for (int a = 0; a < 2; ++a) {
        const float4 v = *reinterpret_cast<const float4*>(Ac + k * TLD + a * 64 + ty * 4);
        av[a][0] = v.x; av[a][1] = v.y; av[a][2] = v.z; av[a][3] = v.w;
      }
#pragma unroll
      for (int b = 0; b < NB; ++b) {
        const float4 v = *reinterpret_cast<const float4*>(Bc + k * TLD + b * 64 + tx * 4);
        bv[b][0] = v.x; bv[b][1] = v.y; bv[b][2] = v.z; bv[b][3] = v.w;
      }
#pragma unroll
      for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < NB; ++b)
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[a][b][i][j] = fmaf(av[a][i], bv[b][j], acc[a][b][i][j]);
    }
    if (more) {
      store_tile<A_KC, 128>(As + (buf ^ 1) * TK * TLD, tid, ra);
      store_tile<B_KC, TNN>(Bs + (buf ^ 1) * TK * TLD, tid, rb);
    }
    __syncthreads();
    buf ^= 1;
  }
  // epilogue: 64 rows of the tile at a time through shared memory (row-aware epilogues see a whole output row)
  float* Cs = smem;  // [64][TNN + 1]
#pragma unroll
  for (int a = 0; a < 2; ++a) {
#pragma unroll
    for (int b = 0; b < NB; ++b)
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) Cs[(ty * 4 + i) * (TNN + 1) + b * 64 + tx * 4 + j] = acc[a][b][i][j];
    __syncthreads();
    row_prep<Epi, TNN>(epi, Cs, m0 + a * 64, n0, M, N);
    for (int e = tid; e < 64 * TNN; e += GT) {
      const int r = e / TNN, c = e - r * TNN;
      const int m = m0 + a * 64 + r;
      if (m < M && n0 + c < N) epi(m, n0 + c, Cs[r * (TNN + 1) + c], Cs + r * (TNN + 1), n0);
    }
    __syncthreads();
  }
}

std::atomic<int> g_simt_tile{128};  // 128: the 128 x 128 kernel when the problem has at least one full tile; 64: always 64 x 64

template <typename AOp, typename BOp, typename Epi, bool A_KC, bool B_KC>
static int launch_gemm(AOp A, BOp Bop, Epi epi, int M, int N, int K, int splits, cudaStream_t st) {
  if (g_simt_tile.load() == 128 && M >= TM && N >= 64) {
    // 128 x 128 tiles unless the last one would be at most half full (192, 576 columns, ...): then 128 x 64
    const int rem = N % TN;
    const bool narrow = N < TN || (rem > 0 && rem <= 64);
    int kps = ceil_div(ceil_div(K, splits), TK) * TK;
    if (narrow) {
      dim3 grid(ceil_div(N, 64), ceil_div(M, TM), splits);
      gemm_simt128_kernel<AOp, BOp, Epi, A_KC, B_KC, 1><<<grid, GT, 0, st>>>(A, Bop, epi, M, N, K, kps);
    } else {
      dim3 grid(ceil_div(N, TN), ceil_div(M, TM), splits);
      gemm_simt128_kernel<AOp, BOp, Epi, A_KC, B_KC, 2><<<grid, GT, 0, st>>>(A, Bop, epi, M, N, K, kps);
    }
    VRR_LAUNCHED();
    return VRR_OK;
  }
  dim3 grid(ceil_div(N, BN), ceil_div(M, BM), splits);
  int kps = ceil_div(ceil_div(K, splits), BK) * BK;
  gemm_simt_kernel<AOp, BOp, Epi, A_KC, B_KC><<<grid, GT, 0, st>>>(A, Bop, epi, M, N, K, kps);
  VRR_LAUNCHED();
  return VRR_OK;
}

// ---- QKV projection + RoPE epilogue -----------------------------------------------------------
template <typename T>
static int qkv_rope_fwd_t(const void* x, const void* w, const float* cos_tab, const float* sin_tab,
                          void* planes, int B, int N, int E, int H, int npre, int rope_mode, cudaStream_t st) {
  StridedOperand<T> A{(const T*)x, E, 1}, W{(const T*)w, E, 1};
  QkvRopeEpilogue<T> epi{(T*)planes, cos_tab, sin_tab, B, N, E, H, E / H, rope_mode, npre, N - npre};
  return launch_gemm<StridedOperand<T>, StridedOperand<T>, QkvRopeEpilogue<T>, true, true>(
      A, W, epi, B * N, 3 * E, E, 1, st);
}
template <typename T>
static int qkv_rope_norm_fwd_t(const void* x, const void* w, const float* cos_tab, const float* sin_tab, void* planes, int B,
                               int N, int E, int H, int npre, int rope_mode, const QkNormArgs& qn, cudaStream_t st) {
  StridedOperand<T> A{(const T*)x, E, 1}, W{(const T*)w, E, 1};
  QkvNormRopeEpilogue<T> epi{{(T*)planes, cos_tab, sin_tab, B, N, E, H, E / H, rope_mode, npre, N - npre}, qn};
  return launch_gemm<StridedOperand<T>, StridedOperand<T>, QkvNormRopeEpilogue<T>, true, true>(A, W, epi, B * N, 3 * E, E, 1, st);
}
int qkv_rope_fwd_simt(const void* x, const void* w, const float* cos_tab, const float* sin_tab,
                      void* planes, int B, int N, int E, int H, int npre, int rope_mode, int dtype,
                      cudaStream_t st, const QkNormArgs* qn) {
  if (qn != nullptr) {
    if (dtype == VRR_F32) return qkv_rope_norm_fwd_t<float>(x, w, cos_tab, sin_tab, planes, B, N, E, H, npre, rope_mode, *qn, st);
    if (dtype == VRR_BF16)
      return qkv_rope_norm_fwd_t<__nv_bfloat16>(x, w, cos_tab, sin_tab, planes, B, N, E, H, npre, rope_mode, *qn, st);
    return qkv_rope_norm_fwd_t<__half>(x, w, cos_tab, sin_tab, planes, B, N, E, H, npre, rope_mode, *qn, st);
  }
  if (dtype == VRR_F32) return qkv_rope_fwd_t<float>(x, w, cos_tab, sin_tab, planes, B, N, E, H, npre, rope_mode, st);
  if (dtype == VRR_BF16) return qkv_rope_fwd_t<__nv_bfloat16>(x, w, cos_tab, sin_tab, planes, B, N, E, H, npre, rope_mode, st);
  return qkv_rope_fwd_t<__half>(x, w, cos_tab, sin_tab, planes, B, N, E, H, npre, rope_mode, st);
}

// ---- plain GEMM -------------------------------------------------------------------------------
// C[M][N] = op(A) . op(B), row-major; op(A) is [M][K], op(B) is [K][N].
template <typename T, typename TC>
static int gemm_t(const void* a, const void* b, void* c, int M, int N, int K, int ta, int tb,
                  cudaStream_t st) {
  // A(m,k): !ta -> a[m*K + k] (k contiguous) ; ta -> a[k*M + m] (m contiguous)
  StridedOperand<T> A = ta ? StridedOperand<T>{(const T*)a, 1, M} : StridedOperand<T>{(const T*)a, K, 1};
  // Bop(n,k) = op(B)[k][n]: !tb -> b[k*N + n] (n contiguous) ; tb -> b[n*K + k] (k contiguous)
  StridedOperand<T> Bo = tb ? StridedOperand<T>{(const T*)b, K, 1} : StridedOperand<T>{(const T*)b, 1, N};
  const bool big = g_simt_tile.load() == 128 && M >= TM && N >= 64;
  const bool narrow = N < TN || (N % TN > 0 && N % TN <= 64);
  const int tiles = big ? ceil_div(M, TM) * ceil_div(N, narrow ? 64 : TN) : ceil_div(M, BM) * ceil_div(N, BN);
  int splits = 1;
  if (sizeof(TC) == 4) {
    const int want = 2 * sm_count();
    if (tiles < want && K >= 8 * BK) splits = min(ceil_div(want, tiles), K / (4 * BK));
    if (splits < 1) splits = 1;
  }
#define GO(AKC, BKC)                                                                              \
  do {                                                                                            \
    if (splits > 1) {                                                                             \
      VRR_CUDA(cudaMemsetAsync(c, 0, (size_t)M * N * sizeof(float), st));                         \
      return launch_gemm<StridedOperand<T>, StridedOperand<T>, AtomicEpilogue, AKC, BKC>(         \
          A, Bo, AtomicEpilogue{(float*)c, N}, M, N, K, splits, st);                              \
    }                                                                                             \
    return launch_gemm<StridedOperand<T>, StridedOperand<T>, StoreEpilogue<TC>, AKC, BKC>(        \
        A, Bo, StoreEpilogue<TC>{(TC*)c, N}, M, N, K, 1, st);                                     \
  } while (0)
  if (!ta && tb) GO(true, true);
  if (!ta && !tb) GO(true, false);
  if (ta && tb) GO(false, true);
  GO(false, false);
#undef GO
}
template <typename T>
static int gemm_bias_t(const void* a, const void* b, void* c, void* c2, const float* bias, int M, int N, int K, int ta,
                       int tb, int gelu, cudaStream_t st) {
  StridedOperand<T> A = ta ? StridedOperand<T>{(const T*)a, 1, M} : StridedOperand<T>{(const T*)a, K, 1};
  StridedOperand<T> Bo = tb ? StridedOperand<T>{(const T*)b, K, 1} : StridedOperand<T>{(const T*)b, 1, N};
  BiasEpilogue<T> epi{(T*)c, (T*)c2, bias, N, gelu};
  if (!ta && tb) return launch_gemm<StridedOperand<T>, StridedOperand<T>, BiasEpilogue<T>, true, true>(A, Bo, epi, M, N, K, 1, st);
  if (!ta && !tb) return launch_gemm<StridedOperand<T>, StridedOperand<T>, BiasEpilogue<T>, true, false>(A, Bo, epi, M, N, K, 1, st);
  if (ta && tb) return launch_gemm<StridedOperand<T>, StridedOperand<T>, BiasEpilogue<T>, false, true>(A, Bo, epi, M, N, K, 1, st);
  return launch_gemm<StridedOperand<T>, StridedOperand<T>, BiasEpilogue<T>, false, false>(A, Bo, epi, M, N, K, 1, st);
}
// C = round(op(A).op(B) + bias) (+ C2 = gelu(C)); C has the operands' element type.
int gemm_simt_bias(const void* a, const void* b, void* c, void* c2, const float* bias, int M, int N, int K, int ta, int tb,
                   int dtype, int gelu, cudaStream_t st) {
  if (dtype == VRR_F32) return gemm_bias_t<float>(a, b, c, c2, bias, M, N, K, ta, tb, gelu, st);
  if (dtype == VRR_BF16) return gemm_bias_t<__nv_bfloat16>(a, b, c, c2, bias, M, N, K, ta, tb, gelu, st);
  return gemm_bias_t<__half>(a, b, c, c2, bias, M, N, K, ta, tb, gelu, st);
}

// ---- SwiGLU Mlp (vrr_gemm_swiglu / vrr_gemm_swiglu_bwd) ---------------------------------------------------
// fc1: logical output column n of block n / 64 pairs gate row j = 32 (n / 64) + (n % 32) of w1 [2H][K] (n % 64 < 32)
// with value row H + j (n % 64 >= 32), so every 64-column block of a tile (both tile widths are multiples of 64) holds
// the g and v of 32 output columns; rows j >= H read as zeros.
template <typename T>
struct SwiGluPairOperand {
  static constexpr bool kVec = true;
  const T* w;
  int H, K;
  __device__ __forceinline__ int row(int n) const {
    const int j = (n >> 6) * 32 + (n & 31);
    return j < H ? ((n & 32) ? H + j : j) : -1;
  }
  __device__ __forceinline__ float operator()(int n, int k) const {
    const int r = row(n);
    return r < 0 ? 0.f : Elem<T>::ld(w + (long long)r * K + k);
  }
  __device__ __forceinline__ bool vec_ok() const { return (K & 3) == 0 && ((uintptr_t)w & 15) == 0; }
  __device__ __forceinline__ float4 ld4k(int n, int k) const {
    const int r = row(n);
    return r < 0 ? make_float4(0.f, 0.f, 0.f, 0.f) : ld4(w + (long long)r * K + k);
  }
  __device__ __forceinline__ float4 ld4r(int n, int k) const {
    return make_float4((*this)(n, k), (*this)(n + 1, k), (*this)(n + 2, k), (*this)(n + 3, k));
  }
  static constexpr long long s_k = 1, s_row = 0;  // k-contiguous (the launcher's vectorisation test)
};
// g = T(acc + T(b1[j])), v = T(acc' + T(b1[H + j])), s = T(silu(g)); act = T(T(s v) f); aux = [T(v silu'(g) f) | T(s f)]
template <typename T>
struct SwiGluEpilogue {
  T* act;
  T* aux;  // [M][2H] or null (act only)
  const float* bias;
  int H;
  int drop;  // 0: f = 1, no product taken
  DropView dv;
  __device__ __forceinline__ void operator()(int m, int n, float acc, const float* crow, int n0) const {
    if (n & 32) return;  // the value column: handled with its gate column
    const int j = (n >> 6) * 32 + (n & 31);
    if (j >= H) return;
    const float g = Elem<T>::round(acc + Elem<T>::round(bias[j]));
    const float v = Elem<T>::round(crow[n + 32 - n0] + Elem<T>::round(bias[H + j]));
    float s, ds;
    silu_and_grad(g, s, ds);
    const float sr = Elem<T>::round(s);
    float a = Elem<T>::round(__fmul_rn(sr, v)), lo = __fmul_rn(v, ds), hi = sr;
    if (drop) {
      const float f = dv.factor(dv.key(), m, j, H, dv.s);
      a = __fmul_rn(a, f);
      lo = __fmul_rn(lo, f);
      hi = __fmul_rn(hi, f);
    }
    Elem<T>::st(act + (long long)m * H + j, a);
    if (aux) {
      Elem<T>::st(aux + (long long)m * 2 * H + j, lo);
      Elem<T>::st(aux + (long long)m * 2 * H + H + j, hi);
    }
  }
};
// dh[m][j] = T(dA aux[m][j]), dh[m][H + j] = T(dA aux[m][H + j]) for the fp32 accumulator dA of (m, j)
template <typename T>
struct SwiGluBwdEpilogue {
  T* dh;
  const T* aux;
  int H;
  __device__ __forceinline__ void operator()(int m, int j, float acc, const float*, int) const {
    const long long o = (long long)m * 2 * H + j;
    Elem<T>::st(dh + o, __fmul_rn(acc, Elem<T>::ld(aux + o)));
    Elem<T>::st(dh + o + H, __fmul_rn(acc, Elem<T>::ld(aux + o + H)));
  }
};

template <typename T>
static int swiglu_simt_t(const void* x, const void* w1, const float* b1, void* act, void* aux, int M, int H, int K,
                         const DropView* dv, cudaStream_t st) {
  StridedOperand<T> A{(const T*)x, K, 1};
  SwiGluPairOperand<T> Bo{(const T*)w1, H, K};
  SwiGluEpilogue<T> epi{(T*)act, (T*)aux, b1, H, dv != nullptr, dv ? *dv : DropView{}};
  return launch_gemm<StridedOperand<T>, SwiGluPairOperand<T>, SwiGluEpilogue<T>, true, true>(A, Bo, epi, M, 64 * ceil_div(H, 32),
                                                                                            K, 1, st);
}
int swiglu_simt(const void* x, const void* w1, const float* b1, void* act, void* aux, int M, int H, int K, int dtype,
                const DropView* dv, cudaStream_t st) {
  if (dtype == VRR_F32) return swiglu_simt_t<float>(x, w1, b1, act, aux, M, H, K, dv, st);
  if (dtype == VRR_BF16) return swiglu_simt_t<__nv_bfloat16>(x, w1, b1, act, aux, M, H, K, dv, st);
  return swiglu_simt_t<__half>(x, w1, b1, act, aux, M, H, K, dv, st);
}

template <typename T>
static int swiglu_bwd_simt_t(const void* dy, const void* w2, const void* aux, void* dh, int M, int H, int K, cudaStream_t st) {
  StridedOperand<T> A{(const T*)dy, K, 1};
  StridedOperand<T> Bo{(const T*)w2, 1, H};  // op(B)[k][n] = w2[k][n]: fc2.weight [K][H]
  SwiGluBwdEpilogue<T> epi{(T*)dh, (const T*)aux, H};
  return launch_gemm<StridedOperand<T>, StridedOperand<T>, SwiGluBwdEpilogue<T>, true, false>(A, Bo, epi, M, H, K, 1, st);
}
int swiglu_bwd_simt(const void* dy, const void* w2, const void* aux, void* dh, int M, int H, int K, int dtype, cudaStream_t st) {
  if (dtype == VRR_F32) return swiglu_bwd_simt_t<float>(dy, w2, aux, dh, M, H, K, st);
  if (dtype == VRR_BF16) return swiglu_bwd_simt_t<__nv_bfloat16>(dy, w2, aux, dh, M, H, K, st);
  return swiglu_bwd_simt_t<__half>(dy, w2, aux, dh, M, H, K, st);
}

void gemm_simt_set_tile(int v) { g_simt_tile.store(v == 64 ? 64 : 128); }

int gemm_simt(const void* a, const void* b, void* c, int M, int N, int K, int ta, int tb, int dtype,
              int c_dtype, cudaStream_t st) {
  if (dtype == VRR_F32 && c_dtype == VRR_F32) return gemm_t<float, float>(a, b, c, M, N, K, ta, tb, st);
  if (dtype == VRR_BF16 && c_dtype == VRR_F32) return gemm_t<__nv_bfloat16, float>(a, b, c, M, N, K, ta, tb, st);
  if (dtype == VRR_BF16 && c_dtype == VRR_BF16)
    return gemm_t<__nv_bfloat16, __nv_bfloat16>(a, b, c, M, N, K, ta, tb, st);
  if (dtype == VRR_F16 && c_dtype == VRR_F32) return gemm_t<__half, float>(a, b, c, M, N, K, ta, tb, st);
  if (dtype == VRR_F16 && c_dtype == VRR_F16) return gemm_t<__half, __half>(a, b, c, M, N, K, ta, tb, st);
  set_error("vrr_gemm: unsupported dtype combination (%d -> %d)", dtype, c_dtype);
  return VRR_ERR_UNSUPPORTED;
}

// ---- patch embedding --------------------------------------------------------------------------
int patch_prefix_rows(void* tokens, const void* prefix, int B, int Np, int E, int npre, int tok_dtype, cudaStream_t st);
// tokens[b][t][:] = prefix[t][:] for the npre prefix rows (cls, then the registers) of every image
template <typename T>
__global__ void prefix_rows_kernel(T* tokens, const T* prefix, int B, int Np, int E, int npre) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * npre * E) return;
  int b = idx / (npre * E), r = idx - b * (npre * E);
  tokens[(size_t)b * (Np + npre) * E + r] = prefix[r];
}

template <typename TI, typename T, typename TT>
static int patch_fwd_t(const void* images, const void* weight, const void* bias, const void* prefix,
                       const void* pos, void* tokens, int B, int C, int Hi, int Wi, int P, int E, int npre,
                       cudaStream_t st) {
  constexpr bool kRound = sizeof(TI) == 4 && sizeof(T) == 2;
  using AOp = Im2colOperand<TI, kRound, T>;
  const int gh = Hi / P, gw = Wi / P, Np = gh * gw, Kd = C * P * P;
  AOp A{(const TI*)images, C, Hi, Wi, P, gw, Np};
  StridedOperand<T> W{(const T*)weight, Kd, 1};
  PatchEmbedEpilogue<T, TT> epi{(TT*)tokens, (const T*)bias, (const TT*)pos, Np, E, npre};
  int rc = launch_gemm<AOp, StridedOperand<T>, PatchEmbedEpilogue<T, TT>, true, true>(
      A, W, epi, B * Np, E, Kd, 1, st);
  if (rc) return rc;
  return patch_prefix_rows(tokens, prefix, B, Np, E, npre, sizeof(TT) == 4 ? VRR_F32 : (std::is_same<TT, __half>::value ? VRR_F16 : VRR_BF16),
                        st);
}
int patch_prefix_rows(void* tokens, const void* prefix, int B, int Np, int E, int npre, int tok_dtype, cudaStream_t st) {
  const int blocks = ceil_div(B * npre * E, 256);
  if (tok_dtype == VRR_F32)
    prefix_rows_kernel<float><<<blocks, 256, 0, st>>>((float*)tokens, (const float*)prefix, B, Np, E, npre);
  else if (tok_dtype == VRR_BF16)
    prefix_rows_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>((__nv_bfloat16*)tokens, (const __nv_bfloat16*)prefix, B, Np, E,
                                                              npre);
  else
    prefix_rows_kernel<__half><<<blocks, 256, 0, st>>>((__half*)tokens, (const __half*)prefix, B, Np, E, npre);
  VRR_LAUNCHED();
  return VRR_OK;
}
int patch_embed_fwd_simt(const void* images, const void* weight, const void* bias, const void* prefix,
                         const void* pos, void* tokens, int B, int C, int Hi, int Wi, int P, int E, int npre,
                         int img_dtype, int dtype, int tok_dtype, cudaStream_t st) {
#define ARGS images, weight, bias, prefix, pos, tokens, B, C, Hi, Wi, P, E, npre, st
  if (img_dtype == VRR_F32 && dtype == VRR_F32 && tok_dtype == VRR_F32) return patch_fwd_t<float, float, float>(ARGS);
  if (img_dtype == VRR_F32 && dtype == VRR_BF16 && tok_dtype == VRR_F32) return patch_fwd_t<float, __nv_bfloat16, float>(ARGS);
  if (img_dtype == VRR_BF16 && dtype == VRR_BF16 && tok_dtype == VRR_F32) return patch_fwd_t<__nv_bfloat16, __nv_bfloat16, float>(ARGS);
  if (img_dtype == VRR_BF16 && dtype == VRR_BF16 && tok_dtype == VRR_BF16)
    return patch_fwd_t<__nv_bfloat16, __nv_bfloat16, __nv_bfloat16>(ARGS);
  if (img_dtype == VRR_F32 && dtype == VRR_F16 && tok_dtype == VRR_F32) return patch_fwd_t<float, __half, float>(ARGS);
  if (img_dtype == VRR_F16 && dtype == VRR_F16 && tok_dtype == VRR_F32) return patch_fwd_t<__half, __half, float>(ARGS);
  if (img_dtype == VRR_F16 && dtype == VRR_F16 && tok_dtype == VRR_F16) return patch_fwd_t<__half, __half, __half>(ARGS);
#undef ARGS
  set_error("patch_embed_fwd: unsupported dtype combination (images %d, weights %d, tokens %d)", img_dtype, dtype, tok_dtype);
  return VRR_ERR_UNSUPPORTED;
}

// s[t][e] = sum_b d_tokens[b][t][e]  ->  d_prefix (t < npre), d_pos (t >= npre), d_bias (sum over t >= npre)
template <typename T>
__global__ void token_batch_sum_kernel(const T* __restrict__ dtok, float* d_bias, float* d_prefix,
                                       float* d_pos, int B, int Np, int E, int npre) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (Np + npre) * E) return;
  int t = idx / E, e = idx - t * E;
  float s = 0.f;
  for (int b = 0; b < B; ++b) s += Elem<T>::ld(dtok + ((size_t)b * (Np + npre) + t) * E + e);
  if (t < npre) {
    d_prefix[idx] = s;
  } else {
    if (d_pos) d_pos[(size_t)(t - npre) * E + e] = s;
    atomicAdd(d_bias + e, s);
  }
}

template <typename TI, bool ROUND, typename TT, typename TR>
static int patch_bwd_t(const void* images, const void* d_tokens, float* d_weight, float* d_bias,
                       float* d_prefix, float* d_pos, int B, int C, int Hi, int Wi, int P, int E, int npre,
                       cudaStream_t st) {
  const int gh = Hi / P, gw = Wi / P, Np = gh * gw, Kd = C * P * P, Mtok = B * Np;
  VRR_CUDA(cudaMemsetAsync(d_bias, 0, (size_t)E * sizeof(float), st));
  token_batch_sum_kernel<TT><<<ceil_div((Np + npre) * E, 256), 256, 0, st>>>((const TT*)d_tokens, d_bias, d_prefix, d_pos, B,
                                                                              Np, E, npre);
  VRR_LAUNCHED();
  if (!d_weight) return VRR_OK;  // caller computes the weight gradient itself (plain library GEMM)
  // d_weight[e][k] = sum_m d_tokens[m][e] * unfold(images)[m][k]   (reduction over m = tokens)
  using BOp = SwapArgs<Im2colOperand<TI, ROUND, TR>>;
  PatchGradOperand<TT> A{(const TT*)d_tokens + (size_t)npre * E, Np, E, Np + npre};
  BOp Bo{Im2colOperand<TI, ROUND, TR>{(const TI*)images, C, Hi, Wi, P, gw, Np}};
  const int tiles = ceil_div(E, BM) * ceil_div(Kd, BN);
  int splits = max(1, min(ceil_div(2 * sm_count(), tiles), Mtok / (4 * BK)));
  VRR_CUDA(cudaMemsetAsync(d_weight, 0, (size_t)E * Kd * sizeof(float), st));
  return launch_gemm<PatchGradOperand<TT>, BOp, AtomicEpilogue, false, false>(
      A, Bo, AtomicEpilogue{d_weight, Kd}, E, Kd, Mtok, splits, st);
}
int patch_embed_bwd_simt(const void* images, const void* d_tokens, float* d_weight, float* d_bias,
                         float* d_prefix, float* d_pos, int B, int C, int Hi, int Wi, int P, int E, int npre,
                         int img_dtype, int dtype, int tok_dtype, cudaStream_t st) {
#define ARGS images, d_tokens, d_weight, d_bias, d_prefix, d_pos, B, C, Hi, Wi, P, E, npre, st
  using bf16 = __nv_bfloat16;
  if (img_dtype == VRR_F32 && dtype == VRR_F32 && tok_dtype == VRR_F32) return patch_bwd_t<float, false, float, float>(ARGS);
  if (img_dtype == VRR_F32 && dtype == VRR_BF16 && tok_dtype == VRR_F32) return patch_bwd_t<float, true, float, bf16>(ARGS);
  if (img_dtype == VRR_BF16 && dtype == VRR_BF16 && tok_dtype == VRR_F32) return patch_bwd_t<bf16, false, float, bf16>(ARGS);
  if (img_dtype == VRR_BF16 && dtype == VRR_BF16 && tok_dtype == VRR_BF16) return patch_bwd_t<bf16, false, bf16, bf16>(ARGS);
  if (img_dtype == VRR_F32 && dtype == VRR_F16 && tok_dtype == VRR_F32) return patch_bwd_t<float, true, float, __half>(ARGS);
  if (img_dtype == VRR_F16 && dtype == VRR_F16 && tok_dtype == VRR_F32) return patch_bwd_t<__half, false, float, __half>(ARGS);
  if (img_dtype == VRR_F16 && dtype == VRR_F16 && tok_dtype == VRR_F16) return patch_bwd_t<__half, false, __half, __half>(ARGS);
#undef ARGS
  set_error("patch_embed_bwd: unsupported dtype combination (images %d, weights %d, tokens %d)", img_dtype, dtype, tok_dtype);
  return VRR_ERR_UNSUPPORTED;
}

}  // namespace vrr
