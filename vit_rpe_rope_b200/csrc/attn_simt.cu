// SIMT (FFMA) fused attention, forward and backward, fp32 math with fp32 or bf16 I/O.
//
// This is the fp32 product path (tcgen05 has no fp32 MMA and the fp32 parity bar is 1e-5) and the
// bf16 path for shapes the tcgen05 kernels do not cover.  Replaces models/vit.py:71-88 of the
// reference (q k^T * scale + bias -> softmax -> . v -> merge heads) without ever materialising the
// [B,H,N,N] logits; the relative-position table / polynomial bias is looked up in a per-head LUT
// held in shared memory.
//
// Work decomposition: one CTA = 64 rows (query rows for fwd / dQ, key rows for dK,dV) of one
// (image, head); two threads per row, each owning alternate 4-wide chunks of the head dimension
// (so that the pair's float4 shared-memory reads are adjacent -> conflict free); the streamed
// operand (K,V for fwd / dQ; Q,dO for dK,dV) goes through shared memory in tiles of 32 rows and is
// read as warp-wide broadcasts.
#include "common.cuh"

namespace vrr {

constexpr int kRows = 64;     // rows per CTA
constexpr int kThreads = 128; // two threads per row
constexpr int kTile = 32;     // streamed rows per shared-memory tile

template <int DH>
struct HalfDims {
  static constexpr int HD = DH / 2;   // elements owned by one thread of the pair
  static constexpr int NC = DH / 8;   // 4-wide chunks owned by one thread
  // element offset of this thread's chunk c
  static __device__ __forceinline__ int off(int c, int half) { return 8 * c + 4 * half; }
};

template <typename T, int DH>
__device__ __forceinline__ void load_half_row(const T* row, int half, float (&dst)[DH / 2]) {
#pragma unroll
  for (int c = 0; c < DH / 8; ++c) {
    float4 v = ld4(row + HalfDims<DH>::off(c, half));
    dst[4 * c + 0] = v.x; dst[4 * c + 1] = v.y; dst[4 * c + 2] = v.z; dst[4 * c + 3] = v.w;
  }
}
template <typename T, int DH>
__device__ __forceinline__ void store_half_row(T* row, int half, const float (&src)[DH / 2], float mul) {
#pragma unroll
  for (int c = 0; c < DH / 8; ++c) {
    st4(row + HalfDims<DH>::off(c, half),
        make_float4(src[4 * c] * mul, src[4 * c + 1] * mul, src[4 * c + 2] * mul, src[4 * c + 3] * mul));
  }
}
template <int DH>
__device__ __forceinline__ float half_dot(const float (&a)[DH / 2], const float* srow, int half) {
  float acc = 0.f;
#pragma unroll
  for (int c = 0; c < DH / 8; ++c) {
    float4 v = *reinterpret_cast<const float4*>(srow + HalfDims<DH>::off(c, half));
    acc = fmaf(a[4 * c + 0], v.x, acc); acc = fmaf(a[4 * c + 1], v.y, acc);
    acc = fmaf(a[4 * c + 2], v.z, acc); acc = fmaf(a[4 * c + 3], v.w, acc);
  }
  return acc;
}
template <int DH>
__device__ __forceinline__ void half_axpy(float (&acc)[DH / 2], float a, const float* srow, int half) {
#pragma unroll
  for (int c = 0; c < DH / 8; ++c) {
    float4 v = *reinterpret_cast<const float4*>(srow + HalfDims<DH>::off(c, half));
    acc[4 * c + 0] = fmaf(a, v.x, acc[4 * c + 0]); acc[4 * c + 1] = fmaf(a, v.y, acc[4 * c + 1]);
    acc[4 * c + 2] = fmaf(a, v.z, acc[4 * c + 2]); acc[4 * c + 3] = fmaf(a, v.w, acc[4 * c + 3]);
  }
}
__device__ __forceinline__ float pair_sum(float v) { return v + __shfl_xor_sync(0xffffffffu, v, 1); }

// Cooperative copy of `rows` consecutive DH-wide rows (contiguous in global memory) into a shared
// tile of kTile rows; rows past `rows` are zero-filled.
template <typename T, int DH>
__device__ __forceinline__ void load_tile(float* stile, const T* g, int rows) {
  constexpr int V4 = kTile * DH / 4;
  for (int v = threadIdx.x; v < V4; v += kThreads) {
    int r = (v * 4) / DH;
    float4 x = (r < rows) ? ld4(g + (size_t)v * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
    *reinterpret_cast<float4*>(stile + v * 4) = x;
  }
}

struct AttnShape {
  int B, H, N;
  float scale;
  int bias_mode, bias_heads, bias_len, bias_grid;
  const float* bias_param;
  int poly_pw;  // dQ kernel, polynomial bias of degree <= 3: per-thread power sums instead of the shared histogram
};

// Positional bias of (own token, streamed token).  Relative table: index i - j + N - 1; polynomial: LUT over the L1
// grid distance.  The own token's grid coordinates are computed once per thread and the streamed tile's once per
// tile (32 entries of shared memory): the first version divided twice per ELEMENT, which made the polynomial mode
// 1.4x (forward) to 1.7x (backward) slower than the table mode at ViT-Tiny.
struct RowBias {
  int mode, n;
  const float* lut;
  const int* tyx;  // POLY: (y << 8 | x) of the streamed tile's tokens
  int self, ys, xs;
  bool self_is_query;
  __device__ __forceinline__ void init(int mode_, int n_, int grid, const float* lut_, const int* tyx_, int self_, bool q) {
    mode = mode_; n = n_; lut = lut_; tyx = tyx_; self = self_; self_is_query = q;
    const int ps = self_ > 0 ? self_ - 1 : 0;
    ys = grid > 0 ? ps % grid : 0;
    xs = grid > 0 ? ps / grid : 0;
  }
  // call by every thread right after the tile loads, before the __syncthreads that publishes the tile
  __device__ __forceinline__ void fill_tile(int* tyx_w, int j0, int grid) const {
    if (mode == VRR_BIAS_POLY && threadIdx.x < kTile) {
      const int t = j0 + (int)threadIdx.x, pt = t > 0 ? t - 1 : 0;
      tyx_w[threadIdx.x] = ((pt % grid) << 8) | (pt / grid);
    }
  }
  __device__ __forceinline__ int index(int other, int jl) const {
    if (mode == VRR_BIAS_TABLE) return (self_is_query ? self - other : other - self) + n - 1;
    const int yx = tyx[jl];
    return abs(ys - (yx >> 8)) + abs(xs - (yx & 255));
  }
  __device__ __forceinline__ float at(int other, int jl) const {
    if (mode == VRR_BIAS_NONE) return 0.f;
    if (mode == VRR_BIAS_POLY && (self == 0 || other == 0)) return 0.f;
    return lut[index(other, jl)];
  }
};

// ------------------------------------------------------------------------------------------ forward
template <typename T, int DH>
__global__ void __launch_bounds__(kThreads) attn_fwd_simt_kernel(const T* __restrict__ planes,
                                                                 T* __restrict__ out,
                                                                 float* __restrict__ lse, AttnShape sh) {
  extern __shared__ __align__(16) float smem[];
  float* Ks = smem;
  float* Vs = Ks + kTile * DH;
  int* tyx = reinterpret_cast<int*>(Vs + kTile * DH);
  float* lut = reinterpret_cast<float*>(tyx + kTile);

  const int bh = blockIdx.y, b = bh / sh.H, h = bh % sh.H, N = sh.N;
  const int half = threadIdx.x & 1;
  const int i = blockIdx.x * kRows + (threadIdx.x >> 1);
  const int ic = min(i, N - 1);
  const size_t plane = (size_t)sh.B * sh.H * N * DH;
  const T* qg = planes + ((size_t)bh * N) * DH;
  const T* kg = qg + plane;
  const T* vg = kg + plane;

  fill_bias_lut(lut, sh.bias_mode, sh.bias_param, sh.bias_heads, sh.bias_len, sh.bias_grid, N, h);
  RowBias bias;
  bias.init(sh.bias_mode, N, sh.bias_grid, lut, tyx, ic, true);

  float q[DH / 2], acc[DH / 2];
  load_half_row<T, DH>(qg + (size_t)ic * DH, half, q);
#pragma unroll
  for (int d = 0; d < DH / 2; ++d) acc[d] = 0.f;
  float m = -INFINITY, l = 0.f;

  for (int j0 = 0; j0 < N; j0 += kTile) {
    const int rows = min(kTile, N - j0);
    __syncthreads();
    load_tile<T, DH>(Ks, kg + (size_t)j0 * DH, rows);
    load_tile<T, DH>(Vs, vg + (size_t)j0 * DH, rows);
    bias.fill_tile(tyx, j0, sh.bias_grid);
    __syncthreads();
    float s[kTile];
    float tmax = -INFINITY;
#pragma unroll
    for (int j = 0; j < kTile; ++j) {
      float d = pair_sum(half_dot<DH>(q, Ks + j * DH, half));
      float v = (j < rows) ? d * sh.scale + bias.at(j0 + j, j) : -INFINITY;
      s[j] = v;
      tmax = fmaxf(tmax, v);
    }
    const float m_new = fmaxf(m, tmax);
    const float corr = __expf(m - m_new);  // m == -inf on the first tile -> 0
    l *= corr;
#pragma unroll
    for (int d = 0; d < DH / 2; ++d) acc[d] *= corr;
#pragma unroll
    for (int j = 0; j < kTile; ++j) {
      float p = expf(s[j] - m_new);
      l += p;
      half_axpy<DH>(acc, p, Vs + j * DH, half);
    }
    m = m_new;
  }
  if (i < N) {
    const float inv = 1.f / l;
    store_half_row<T, DH>(out + ((size_t)b * N + i) * (sh.H * DH) + h * DH, half, acc, inv);
    if (half == 0) lse[(size_t)bh * N + i] = m + logf(l);
  }
}

// ------------------------------------------------------------------------------------------ dQ
// Row owner = query i.  Streams K,V.  Also produces delta_i = sum_d dO_i O_i (written for the
// dK,dV kernel) and the histogram of dS over LUT indices (gradient of the table / polynomial).
template <typename T, int DH>
__global__ void __launch_bounds__(kThreads) attn_bwd_dq_simt_kernel(
    const T* __restrict__ planes, const T* __restrict__ out, const T* __restrict__ d_out,
    const float* __restrict__ lse, T* __restrict__ d_planes, float* __restrict__ delta,
    float* __restrict__ d_lut, AttnShape sh) {
  extern __shared__ __align__(16) float smem[];
  float* Ks = smem;
  float* Vs = Ks + kTile * DH;
  int* tyx = reinterpret_cast<int*>(Vs + kTile * DH);
  float* lut = reinterpret_cast<float*>(tyx + kTile);
  const int lut_len = (sh.bias_mode == VRR_BIAS_TABLE) ? 2 * sh.N - 1
                      : (sh.bias_mode == VRR_BIAS_POLY ? 2 * sh.bias_grid - 1 : 0);
  float* hist = lut + lut_len;

  const int bh = blockIdx.y, b = bh / sh.H, h = bh % sh.H, N = sh.N, E = sh.H * DH;
  const int half = threadIdx.x & 1;
  const int i = blockIdx.x * kRows + (threadIdx.x >> 1);
  const int ic = min(i, N - 1);
  const bool live = i < N;
  const size_t plane = (size_t)sh.B * sh.H * N * DH;
  const T* qg = planes + ((size_t)bh * N) * DH;
  const T* kg = qg + plane;
  const T* vg = kg + plane;

  fill_bias_lut(lut, sh.bias_mode, sh.bias_param, sh.bias_heads, sh.bias_len, sh.bias_grid, N, h);
  for (int t = threadIdx.x; t < lut_len; t += kThreads) hist[t] = 0.f;
  RowBias bias;
  bias.init(sh.bias_mode, N, sh.bias_grid, lut, tyx, ic, true);
  float pw0 = 0.f, pw1 = 0.f, pw2 = 0.f, pw3 = 0.f;  // poly_pw: sum of dS * distance^k over this thread's elements

  float q[DH / 2], go[DH / 2], dq[DH / 2];
  load_half_row<T, DH>(qg + (size_t)ic * DH, half, q);
  load_half_row<T, DH>(d_out + ((size_t)b * N + ic) * E + h * DH, half, go);
  float dl;
  {
    float o[DH / 2];
    load_half_row<T, DH>(out + ((size_t)b * N + ic) * E + h * DH, half, o);
    float a = 0.f;
#pragma unroll
    for (int d = 0; d < DH / 2; ++d) a = fmaf(go[d], o[d], a);
    dl = pair_sum(a);
  }
  const float li = lse[(size_t)bh * N + ic];
  if (live && half == 0) delta[(size_t)bh * N + i] = dl;
#pragma unroll
  for (int d = 0; d < DH / 2; ++d) dq[d] = 0.f;

  for (int j0 = 0; j0 < N; j0 += kTile) {
    const int rows = min(kTile, N - j0);
    __syncthreads();
    load_tile<T, DH>(Ks, kg + (size_t)j0 * DH, rows);
    load_tile<T, DH>(Vs, vg + (size_t)j0 * DH, rows);
    bias.fill_tile(tyx, j0, sh.bias_grid);
    __syncthreads();
#pragma unroll 4
    for (int j = 0; j < kTile; ++j) {
      float s = pair_sum(half_dot<DH>(q, Ks + j * DH, half));
      float dp = pair_sum(half_dot<DH>(go, Vs + j * DH, half));
      const int jj = j0 + j;
      const bool ok = live && j < rows;
      float p = ok ? expf(s * sh.scale + bias.at(jj, j) - li) : 0.f;
      float ds = p * (dp - dl);
      half_axpy<DH>(dq, ds, Ks + j * DH, half);
      if (ok && half == 0 && sh.bias_mode != VRR_BIAS_NONE &&
          !(sh.bias_mode == VRR_BIAS_POLY && (ic == 0 || jj == 0))) {
        if (sh.poly_pw) {  // d_coef[k] = sum dS * distance^k: no atomics in the loop (15 bins, every thread of the CTA)
          const float dist = (float)bias.index(jj, j);
          pw0 += ds;
          const float w1 = ds * dist;
          pw1 += w1;
          const float w2 = w1 * dist;
          pw2 += w2;
          pw3 = fmaf(w2, dist, pw3);
        } else {
          atomicAdd(&hist[bias.index(jj, j)], ds);
        }
      }
    }
  }
  if (live) store_half_row<T, DH>(d_planes + ((size_t)bh * N + i) * DH, half, dq, sh.scale);
  if (sh.poly_pw) {  // warp sums -> hist[0..3] (which the tail below adds to d_lut[h][0..3])
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      pw0 += __shfl_xor_sync(0xffffffffu, pw0, o);
      pw1 += __shfl_xor_sync(0xffffffffu, pw1, o);
      pw2 += __shfl_xor_sync(0xffffffffu, pw2, o);
      pw3 += __shfl_xor_sync(0xffffffffu, pw3, o);
    }
    if ((threadIdx.x & 31) == 0) {
      atomicAdd(&hist[0], pw0);
      atomicAdd(&hist[1], pw1);
      atomicAdd(&hist[2], pw2);
      atomicAdd(&hist[3], pw3);
    }
  }
  if (lut_len) {
    __syncthreads();
    float* dst = d_lut + (size_t)h * lut_len;
    for (int t = threadIdx.x; t < lut_len; t += kThreads) {
      float v = hist[t];
      if (v != 0.f) atomicAdd(dst + t, v);
    }
  }
}

// ------------------------------------------------------------------------------------------ dK, dV
// Row owner = key j.  Streams Q, dO (+ lse, delta).
template <typename T, int DH>
__global__ void __launch_bounds__(kThreads) attn_bwd_dkv_simt_kernel(
    const T* __restrict__ planes, const T* __restrict__ d_out, const float* __restrict__ lse,
    const float* __restrict__ delta, T* __restrict__ d_planes, AttnShape sh) {
  extern __shared__ __align__(16) float smem[];
  float* Qs = smem;
  float* Gs = Qs + kTile * DH;   // dO tile
  float* Ls = Gs + kTile * DH;   // lse tile
  float* Ds = Ls + kTile;        // delta tile
  int* tyx = reinterpret_cast<int*>(Ds + kTile);
  float* lut = reinterpret_cast<float*>(tyx + kTile);

  const int bh = blockIdx.y, b = bh / sh.H, h = bh % sh.H, N = sh.N, E = sh.H * DH;
  const int half = threadIdx.x & 1;
  const int j = blockIdx.x * kRows + (threadIdx.x >> 1);
  const int jc = min(j, N - 1);
  const bool live = j < N;
  const size_t plane = (size_t)sh.B * sh.H * N * DH;
  const T* qg = planes + ((size_t)bh * N) * DH;
  const T* kg = qg + plane;
  const T* vg = kg + plane;

  fill_bias_lut(lut, sh.bias_mode, sh.bias_param, sh.bias_heads, sh.bias_len, sh.bias_grid, N, h);
  RowBias bias;
  bias.init(sh.bias_mode, N, sh.bias_grid, lut, tyx, jc, false);

  float k[DH / 2], v[DH / 2], dk[DH / 2], dv[DH / 2];
  load_half_row<T, DH>(kg + (size_t)jc * DH, half, k);
  load_half_row<T, DH>(vg + (size_t)jc * DH, half, v);
#pragma unroll
  for (int d = 0; d < DH / 2; ++d) dk[d] = dv[d] = 0.f;

  for (int i0 = 0; i0 < N; i0 += kTile) {
    const int rows = min(kTile, N - i0);
    __syncthreads();
    load_tile<T, DH>(Qs, qg + (size_t)i0 * DH, rows);
    // dO rows are strided by E in [B,N,E]
    for (int t = threadIdx.x; t < kTile * DH / 4; t += kThreads) {
      int r = (t * 4) / DH, c = (t * 4) % DH;
      float4 x = (r < rows) ? ld4(d_out + ((size_t)b * N + i0 + r) * E + h * DH + c)
                            : make_float4(0.f, 0.f, 0.f, 0.f);
      *reinterpret_cast<float4*>(Gs + t * 4) = x;
    }
    if (threadIdx.x < kTile) {
      int r = threadIdx.x;
      Ls[r] = (r < rows) ? lse[(size_t)bh * N + i0 + r] : 0.f;
      Ds[r] = (r < rows) ? delta[(size_t)bh * N + i0 + r] : 0.f;
    }
    bias.fill_tile(tyx, i0, sh.bias_grid);
    __syncthreads();
#pragma unroll 4
    for (int r = 0; r < kTile; ++r) {
      float s = pair_sum(half_dot<DH>(k, Qs + r * DH, half));
      float dp = pair_sum(half_dot<DH>(v, Gs + r * DH, half));
      const bool ok = live && r < rows;
      float p = ok ? expf(s * sh.scale + bias.at(i0 + r, r) - Ls[r]) : 0.f;
      float ds = p * (dp - Ds[r]);
      half_axpy<DH>(dv, p, Gs + r * DH, half);
      half_axpy<DH>(dk, ds, Qs + r * DH, half);
    }
  }
  if (live) {
    store_half_row<T, DH>(d_planes + plane + ((size_t)bh * N + j) * DH, half, dk, sh.scale);
    store_half_row<T, DH>(d_planes + 2 * plane + ((size_t)bh * N + j) * DH, half, dv, 1.f);
  }
}

// d_coef[hc][k] = sum over heads (if shared) and distances of d_lut[h][d] * d^k
// (pw_mode: d_lut[h][k] already holds sum dS * distance^k - only the heads are summed)
__global__ void poly_coef_grad_kernel(const float* __restrict__ d_lut, float* __restrict__ d_coef,
                                      int H, int coef_heads, int len, int lut_len, int pw_mode) {
  int hc = blockIdx.x, k = threadIdx.x;
  if (k >= len) return;
  double acc = 0.0;
  for (int h = 0; h < H; ++h) {
    if (coef_heads != 1 && h != hc) continue;
    if (pw_mode) {
      acc += (double)d_lut[(size_t)h * lut_len + k];
      continue;
    }
    for (int d = 0; d < lut_len; ++d) {
      double pw = 1.0;
      for (int e = 0; e < k; ++e) pw *= (double)d;
      acc += (double)d_lut[(size_t)h * lut_len + d] * pw;
    }
  }
  d_coef[hc * len + k] = (float)acc;
}

// ------------------------------------------------------------------------------------------ host
static AttnShape make_shape(int B, int H, int N, float scale, const vrr_bias_desc* bias) {
  AttnShape sh{B, H, N, scale, VRR_BIAS_NONE, 0, 0, 0, nullptr, 0};
  if (bias && bias->mode != VRR_BIAS_NONE) {
    sh.bias_mode = bias->mode; sh.bias_heads = bias->heads; sh.bias_len = bias->len;
    sh.bias_grid = bias->grid; sh.bias_param = bias->param;
  }
  return sh;
}

template <typename T, int DH>
static int fwd_launch(const void* planes, const vrr_bias_desc* bias, void* out, float* lse, int B,
                      int H, int N, float scale, cudaStream_t st) {
  AttnShape sh = make_shape(B, H, N, scale, bias);
  size_t smem = (size_t)(2 * kTile * DH + kTile + bias_lut_len(bias, N)) * sizeof(float);
  auto kern = attn_fwd_simt_kernel<T, DH>;
  if (smem > 48 * 1024) VRR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid(ceil_div(N, kRows), B * H);
  kern<<<grid, kThreads, smem, st>>>((const T*)planes, (T*)out, lse, sh);
  VRR_LAUNCHED();
  return VRR_OK;
}

template <typename T, int DH>
static int bwd_launch(const void* planes, const vrr_bias_desc* bias, const void* out,
                      const void* d_out, const float* lse, void* d_planes, float* d_bias_param,
                      float* delta, float* d_lut_ws, int B, int H, int N, float scale,
                      cudaStream_t st) {
  AttnShape sh = make_shape(B, H, N, scale, bias);
  const int lut_len = bias_lut_len(bias, N);
  float* d_lut = nullptr;
  if (lut_len) {
    // TABLE: the LUT *is* the table row, so the histogram lands directly in d_bias_param.
    d_lut = (sh.bias_mode == VRR_BIAS_TABLE) ? d_bias_param : d_lut_ws;
    VRR_CUDA(cudaMemsetAsync(d_lut, 0, (size_t)H * lut_len * sizeof(float), st));
  }
  // polynomial of degree <= 3 (the reference's default): per-thread power sums; the histogram needs >= 4 bins to carry them
  sh.poly_pw = (sh.bias_mode == VRR_BIAS_POLY && sh.bias_len <= 4 && lut_len >= 4) ? 1 : 0;
  dim3 grid(ceil_div(N, kRows), B * H);
  {
    size_t smem = (size_t)(2 * kTile * DH + kTile + 2 * lut_len) * sizeof(float);
    auto kern = attn_bwd_dq_simt_kernel<T, DH>;
    if (smem > 48 * 1024) VRR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, kThreads, smem, st>>>((const T*)planes, (const T*)out, (const T*)d_out, lse,
                                       (T*)d_planes, delta, d_lut, sh);
    VRR_LAUNCHED();
  }
  {
    size_t smem = (size_t)(2 * kTile * DH + 3 * kTile + lut_len) * sizeof(float);
    auto kern = attn_bwd_dkv_simt_kernel<T, DH>;
    if (smem > 48 * 1024) VRR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, kThreads, smem, st>>>((const T*)planes, (const T*)d_out, lse, delta, (T*)d_planes, sh);
    VRR_LAUNCHED();
  }
  if (sh.bias_mode == VRR_BIAS_POLY) {
    poly_coef_grad_kernel<<<bias->heads, 32, 0, st>>>(d_lut, d_bias_param, H, bias->heads, bias->len, lut_len, sh.poly_pw);
    VRR_LAUNCHED();
  }
  return VRR_OK;
}

#define VRR_DISPATCH_T_DH(dtype, DHv, CALL)                                      \
  do {                                                                           \
    if ((dtype) == VRR_F32) {                                                    \
      if ((DHv) == 16) return CALL(float, 16);                                   \
      if ((DHv) == 32) return CALL(float, 32);                                   \
      if ((DHv) == 64) return CALL(float, 64);                                   \
    } else if ((dtype) == VRR_BF16) {                                            \
      if ((DHv) == 16) return CALL(__nv_bfloat16, 16);                           \
      if ((DHv) == 32) return CALL(__nv_bfloat16, 32);                           \
      if ((DHv) == 64) return CALL(__nv_bfloat16, 64);                           \
    } else {                                                                     \
      if ((DHv) == 16) return CALL(__half, 16);                                  \
      if ((DHv) == 32) return CALL(__half, 32);                                  \
      if ((DHv) == 64) return CALL(__half, 64);                                  \
    }                                                                            \
  } while (0)

int attn_fwd_simt(const void* planes, const vrr_bias_desc* bias, void* out, float* lse, int B, int H,
                  int N, int Dh, float scale, int dtype, cudaStream_t st) {
#define CALL(T, D) fwd_launch<T, D>(planes, bias, out, lse, B, H, N, scale, st)
  VRR_DISPATCH_T_DH(dtype, Dh, CALL);
#undef CALL
  set_error("attn_fwd: head dim %d unsupported (16, 32, 64)", Dh);
  return VRR_ERR_UNSUPPORTED;
}

int attn_bwd_simt(const void* planes, const vrr_bias_desc* bias, const void* out, const void* d_out,
                  const float* lse, void* d_planes, float* d_bias_param, float* delta,
                  float* d_lut_ws, int B, int H, int N, int Dh, float scale, int dtype,
                  cudaStream_t st) {
#define CALL(T, D) \
  bwd_launch<T, D>(planes, bias, out, d_out, lse, d_planes, d_bias_param, delta, d_lut_ws, B, H, N, scale, st)
  VRR_DISPATCH_T_DH(dtype, Dh, CALL);
#undef CALL
  set_error("attn_bwd: head dim %d unsupported (16, 32, 64)", Dh);
  return VRR_ERR_UNSUPPORTED;
}

}  // namespace vrr
