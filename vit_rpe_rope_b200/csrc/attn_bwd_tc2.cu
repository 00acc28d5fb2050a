// Fused attention backward for every case the whole-sequence kernel (attn_bwd_ws.cu) does not take: the bias modes
// and N > 208.  Two kernels with the tiled forward's pipeline - a dedicated issuer warp (TMA + every tcgen05.mma),
// 32-row streamed tiles, double-buffered S / dP accumulators in TMEM so the issuer computes tile t+1 while the four
// row-owner warps work on tile t, dS / P written back in place (bf16 / fp16) and consumed from TMEM by the
// accumulating MMAs.
//
//  dQ kernel  (CTA = 128 query rows):  TMEM cols  S[2] 0..63 | dP[2] 64..127 | dQ 128..191
//       S = Q K_t^T, dP = dO V_t^T  ->  thread: P = exp2(S*c + bias - lse), dS = P (dP - delta)
//       -> dS (T) over S buffer  ->  dQ += dS K_t.   Also delta, and the bias gradients:
//       relative table: each warp transposes its 32x32 dS block through shared memory and every lane
//       sums two diagonals (conflict-free, 33-float pitch) -> 2 shared atomics per lane per tile;
//       polynomial: per-thread power sums.
//  dK/dV kernel (CTA = 128 key rows):  TMEM cols  S^T[2] 0..63 | dP^T[2] 64..127 | dV 128..191 | dK 192..255
//       S^T = K Q_t^T, dP^T = V dO_t^T -> thread: P^T, dS^T -> T in place -> dV += P^T dO_t, dK += dS^T Q_t.
#include "common.cuh"
#include "kernels.h"
#include "tc_common.cuh"

namespace vrr {

using namespace tc;

namespace {

constexpr int kRows = 128;   // rows (TMEM lanes) per CTA
constexpr int kT = 32;       // streamed rows per tile
constexpr int kSt = 6;       // ring depth
constexpr int kDh = 64;
constexpr int kTileB = kT * kDh * 2;      // 4 KB
constexpr int kResB = kRows * kDh * 2;    // 16 KB
constexpr int kThreads = 160;
constexpr uint32_t kTmemCols = 256;
constexpr float kLog2e = 1.4426950408889634f;

struct Bwd2Params {
  const void *out, *d_out;  // element type T of the kernels
  const float* lse;
  float* delta;
  void* d_planes;           // T
  const float* bias_param;
  float* d_bias_param;
  int B, H, N;
  float scale, scale_log2;
  int bias_heads, bias_len, bias_grid;
  int lut_floats;
};

template <int BIAS>
__device__ __forceinline__ void fill_lut2(float* lut, uint16_t* key_yx, const Bwd2Params& p, int h, int tid) {
  if (BIAS == VRR_BIAS_TABLE) {
    const float* row = p.bias_param + (size_t)h * p.bias_len;
    for (int t = tid; t < p.bias_len; t += 128) lut[t] = row[t] * kLog2e;
  } else if (BIAS == VRR_BIAS_POLY) {
    const float* c = p.bias_param + (size_t)(p.bias_heads == 1 ? 0 : h) * p.bias_len;
    for (int d = tid; d < 2 * p.bias_grid - 1; d += 128) {
      float x = (float)d, pw = 1.f, acc = 0.f;
      for (int k = 0; k < p.bias_len; ++k) {
        acc = fmaf(pw, c[k], acc);
        pw *= x;
      }
      lut[d] = acc * kLog2e;
    }
    for (int t = tid; t < p.N; t += 128) {
      const int pt = t > 0 ? t - 1 : 0;
      key_yx[t] = (uint16_t)(((pt % p.bias_grid) << 8) | (pt / p.bias_grid));
    }
  }
}

template <typename T>
__device__ __forceinline__ void store_row64(T* dst, const uint32_t (&lo)[32], const uint32_t (&hi)[32], float mul) {
#pragma unroll
  for (int v8 = 0; v8 < 8; ++v8) {
    const uint32_t* src = v8 < 4 ? &lo[v8 * 8] : &hi[(v8 - 4) * 8];
    uint4 w;
    w.x = Elem16<T>::pack2(__uint_as_float(src[0]) * mul, __uint_as_float(src[1]) * mul);
    w.y = Elem16<T>::pack2(__uint_as_float(src[2]) * mul, __uint_as_float(src[3]) * mul);
    w.z = Elem16<T>::pack2(__uint_as_float(src[4]) * mul, __uint_as_float(src[5]) * mul);
    w.w = Elem16<T>::pack2(__uint_as_float(src[6]) * mul, __uint_as_float(src[7]) * mul);
    *reinterpret_cast<uint4*>(dst + v8 * 8) = w;
  }
}

// ============================================================================================ dQ
template <typename T, int BIAS>
__global__ void __launch_bounds__(kThreads, 2)
attn_bwd_dq_tc2_kernel(const __grid_constant__ CUtensorMap tmap_pl, const __grid_constant__ CUtensorMap tmap_do,
                       const Bwd2Params p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;
  uint8_t* sG = sQ + kResB;                 // dO rows of this CTA
  uint8_t* sK = sG + kResB;                 // K ring [kSt][4 KB]
  uint8_t* sV = sK + kSt * kTileB;          // V ring [kSt][4 KB]
  float* lut = reinterpret_cast<float*>(sV + kSt * kTileB);
  float* hist = lut + p.lut_floats;                                         // TABLE: 2N-1 bins
  const int hist_floats = (BIAS == VRR_BIAS_TABLE) ? ((2 * p.N - 1 + 3) & ~3) : 0;
  float* xpose = hist + hist_floats;                                        // TABLE: [4 warps][32][33]
  const int xpose_floats = (BIAS == VRR_BIAS_TABLE) ? 4 * 32 * 33 : 0;
  uint16_t* key_yx = reinterpret_cast<uint16_t*>(xpose + xpose_floats);
  const int key_yx_bytes = (BIAS == VRR_BIAS_POLY) ? ((p.N * 2 + 15) & ~15) : 0;
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(key_yx) + key_yx_bytes);
  uint64_t* bar_kfull = bars;
  uint64_t* bar_vfull = bars + kSt;
  uint64_t* bar_kempty = bars + 2 * kSt;    // dQ MMA of the tile retired (K is read by S and by dQ)
  uint64_t* bar_vempty = bars + 3 * kSt;    // dP MMA of the tile retired
  uint64_t* bar_q = bars + 4 * kSt;
  uint64_t* bar_s = bars + 4 * kSt + 1;     // [2] S and dP of the tile ready
  uint64_t* bar_p = bars + 4 * kSt + 3;     // [2] dS stored (128 arrivals)
  uint64_t* bar_done = bars + 4 * kSt + 5;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4 * kSt + 6);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N = p.N, H = p.H, E = H * kDh;
  const int bh = blockIdx.y, b = bh / H, h = bh - b * H;
  const int m0 = blockIdx.x * kRows;
  const int ntiles = (N + kT - 1) / kT;
  const int BHN = p.B * H * N;

  if (warp == 4) {
    if (tid == 128) {
      for (int s = 0; s < kSt; ++s) {
        mbar_init(&bar_kfull[s], 1);
        mbar_init(&bar_vfull[s], 1);
        mbar_init(&bar_kempty[s], 1);
        mbar_init(&bar_vempty[s], 1);
      }
      mbar_init(bar_q, 1);
      for (int s = 0; s < 2; ++s) {
        mbar_init(&bar_s[s], 1);
        mbar_init(&bar_p[s], 128);
      }
      mbar_init(bar_done, 1);
      fence_mbar_init();
    }
    __syncwarp();
    if (elect_one()) {
      tma_prefetch_desc(&tmap_pl);
      tma_prefetch_desc(&tmap_do);
      mbar_expect_tx(bar_q, 2 * kResB);
#pragma unroll
      for (int r = 0; r < kRows / kT; ++r) {
        tma_load_2d(sQ + r * kTileB, &tmap_pl, bar_q, 0, bh * N + m0 + r * kT);
        tma_load_2d(sG + r * kTileB, &tmap_do, bar_q, h * kDh, b * N + m0 + r * kT);
      }
      for (int s = 0; s < kSt && s < ntiles; ++s) {
        mbar_expect_tx(&bar_kfull[s], kTileB);
        tma_load_2d(sK + s * kTileB, &tmap_pl, &bar_kfull[s], 0, BHN + bh * N + s * kT);
        mbar_expect_tx(&bar_vfull[s], kTileB);
        tma_load_2d(sV + s * kTileB, &tmap_pl, &bar_vfull[s], 0, 2 * BHN + bh * N + s * kT);
      }
    }
    __syncwarp();
    tmem_alloc(tmem_slot, kTmemCols);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 4) {
    // =========================================== issuer ===========================================
    const uint64_t desc_q = smem_desc_sw128(smem_u32(sQ));
    const uint64_t desc_g = smem_desc_sw128(smem_u32(sG));
    constexpr uint32_t idesc_s = idesc_16<T>(kRows, kT, 0, 0);
    constexpr uint32_t idesc_q = idesc_16<T>(kRows, kDh, 0, 1);
    auto issue_s_dp = [&](int t) {  // S(t), dP(t) into buffer t & 1
      const int st = t % kSt;
      mbar_wait(&bar_kfull[st], (uint32_t)((t / kSt) & 1));
      mbar_wait(&bar_vfull[st], (uint32_t)((t / kSt) & 1));
      tc_fence_after();
      if (elect_one()) {
        const uint64_t dk = smem_desc_sw128(smem_u32(sK + st * kTileB));
        const uint64_t dv = smem_desc_sw128(smem_u32(sV + st * kTileB));
        const uint32_t cs = tmem_base + (t & 1) * kT, cp = tmem_base + 64 + (t & 1) * kT;
#pragma unroll
        for (int k = 0; k < 4; ++k) mma_ss(cs, desc_q + 2 * k, dk + 2 * k, idesc_s, k > 0);
#pragma unroll
        for (int k = 0; k < 4; ++k) mma_ss(cp, desc_g + 2 * k, dv + 2 * k, idesc_s, k > 0);
        mma_commit(&bar_s[t & 1]);
        mma_commit(&bar_vempty[st]);
      }
      __syncwarp();
    };
    mbar_wait(bar_q, 0);
    issue_s_dp(0);
    for (int t = 0; t < ntiles; ++t) {
      const int st = t % kSt;
      if (t + 1 < ntiles) issue_s_dp(t + 1);
      if (t + kSt < ntiles) {  // V(t) was consumed by dP(t): refill its stage
        mbar_wait(&bar_vempty[st], (uint32_t)((t / kSt) & 1));
        if (elect_one()) {
          mbar_expect_tx(&bar_vfull[st], kTileB);
          tma_load_2d(sV + st * kTileB, &tmap_pl, &bar_vfull[st], 0, 2 * BHN + bh * N + (t + kSt) * kT);
        }
        __syncwarp();
      }
      mbar_wait(&bar_p[t & 1], (uint32_t)((t >> 1) & 1));
      tc_fence_after();
      if (elect_one()) {
        const uint64_t dk = smem_desc_sw128(smem_u32(sK + st * kTileB));
        const uint32_t a = tmem_base + (t & 1) * kT;
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) mma_ts(tmem_base + 128, a + kk * 8, dk + 128 * kk, idesc_q, (t | kk) != 0);
        mma_commit(&bar_kempty[st]);
        if (t == ntiles - 1) mma_commit(bar_done);
      }
      __syncwarp();
      if (t >= 1 && t - 1 + kSt < ntiles) {  // K(t-1) was last read by dQ(t-1): refill its stage
        const int sp = (t - 1) % kSt;
        mbar_wait(&bar_kempty[sp], (uint32_t)(((t - 1) / kSt) & 1));
        if (elect_one()) {
          mbar_expect_tx(&bar_kfull[sp], kTileB);
          tma_load_2d(sK + sp * kTileB, &tmap_pl, &bar_kfull[sp], 0, BHN + bh * N + (t - 1 + kSt) * kT);
        }
        __syncwarp();
      }
    }
  } else {
    // =========================================== row owners =======================================
    const int i = m0 + tid;
    const int ic = min(i, N - 1);
    const bool live = i < N;
    const bool warp_active = (m0 + warp * 32) < N;
    const uint32_t tmem_row = tmem_base + ((uint32_t)(warp * 32) << 16);
    fill_lut2<BIAS>(lut, key_yx, p, h, tid);
    if (BIAS == VRR_BIAS_TABLE)
      for (int t = tid; t < 2 * N - 1; t += 128) hist[t] = 0.f;
    float lse2 = 0.f, delta = 0.f;
    {
      const size_t off = ((size_t)b * N + ic) * E + h * kDh;
      const uint4* o4 = reinterpret_cast<const uint4*>(static_cast<const T*>(p.out) + off);
      const uint4* g4 = reinterpret_cast<const uint4*>(static_cast<const T*>(p.d_out) + off);
#pragma unroll
      for (int v8 = 0; v8 < 8; ++v8) {
        const uint4 ov = __ldg(o4 + v8), gv = __ldg(g4 + v8);
        const uint32_t ow[4] = {ov.x, ov.y, ov.z, ov.w}, gw[4] = {gv.x, gv.y, gv.z, gv.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 of = Elem16<T>::unpack2(ow[e]);
          const float2 gf = Elem16<T>::unpack2(gw[e]);
          delta = fmaf(of.x, gf.x, delta);
          delta = fmaf(of.y, gf.y, delta);
        }
      }
      lse2 = p.lse[(size_t)bh * N + ic] * kLog2e;
      if (live) p.delta[(size_t)bh * N + i] = delta;
    }
    int yi = 0, xi = 0;
    if (BIAS == VRR_BIAS_POLY) {
      const int pi = ic > 0 ? ic - 1 : 0;
      yi = pi % p.bias_grid;
      xi = pi / p.bias_grid;
    }
    if (BIAS != VRR_BIAS_NONE) asm volatile("bar.sync 1, 128;" ::: "memory");
    float pw0 = 0.f, pw1 = 0.f, pw2 = 0.f, pw3 = 0.f;
    float* xp = xpose + warp * (32 * 33);

    for (int t = 0; t < ntiles; ++t) {
      const int sb = t & 1;
      const int nvalid = min(kT, N - t * kT);
      mbar_wait(&bar_s[sb], (uint32_t)((t >> 1) & 1));
      tc_fence_after();
      if (warp_active) {
        uint32_t sr[32], dr[32], packed[16];
        tmem_ld32(tmem_row + sb * kT, sr);
        tmem_ld32(tmem_row + 64 + sb * kT, dr);
        tmem_wait_ld();
#pragma unroll
        for (int e = 0; e < kT; ++e) {
          const int j = t * kT + e;
          float x = fmaf(__uint_as_float(sr[e]), p.scale_log2, -lse2);
          float dist_f = 0.f;
          if (BIAS == VRR_BIAS_TABLE) {
            x += lut[min(max(ic - j + N - 1, 0), 2 * N - 2)];
          } else if (BIAS == VRR_BIAS_POLY) {
            const int yx = key_yx[min(j, N - 1)];
            const int dist = abs(yi - (yx >> 8)) + abs(xi - (yx & 255));
            dist_f = (float)dist;
            x += (ic == 0 || j == 0) ? 0.f : lut[dist];
          }
          const float pr = (live && e < nvalid) ? ex2(x) : 0.f;
          const float ds = pr * (__uint_as_float(dr[e]) - delta);
          if (BIAS == VRR_BIAS_TABLE) {
            xp[lane * 33 + e] = ds;
          } else if (BIAS == VRR_BIAS_POLY) {
            const float w = (ic == 0 || j == 0) ? 0.f : ds;
            pw0 += w;
            const float w1 = w * dist_f;
            pw1 += w1;
            const float w2 = w1 * dist_f;
            pw2 += w2;
            pw3 = fmaf(w2, dist_f, pw3);
          }
          if (e & 1) packed[e >> 1] = Elem16<T>::pack2(__uint_as_float(sr[e - 1]), ds);
          else sr[e] = __float_as_uint(ds);
        }
        tmem_st16(tmem_row + sb * kT, packed);  // dS (pairs of T) over this S buffer
        if (BIAS == VRR_BIAS_TABLE) {
          // diagonal sums of the warp's 32x32 dS block: element (r, c) lies on diagonal r - c; lane l
          // owns diagonal l (rows l.., cols 0..) and diagonal l-32 (rows 0.., cols 32-l..): 32 elements.
          __syncwarp();
          float d1 = 0.f, d2 = 0.f;
          for (int k = 0; k + lane < 32; ++k) d1 += xp[(lane + k) * 33 + k];
          for (int k = 0; k < lane; ++k) d2 += xp[k * 33 + (k + 32 - lane)];
          const int base_bin = (m0 + warp * 32) - t * kT + N - 1;  // bin of diagonal 0
          const int b1 = base_bin + lane, b2 = base_bin + lane - 32;
          if (b1 >= 0 && b1 <= 2 * N - 2) atomicAdd(&hist[b1], d1);
          if (lane > 0 && b2 >= 0 && b2 <= 2 * N - 2) atomicAdd(&hist[b2], d2);
          __syncwarp();
        }
        tmem_wait_st();
      }
      tc_fence_before();
      mbar_arrive(&bar_p[sb]);
    }

    mbar_wait(bar_done, 0);
    tc_fence_after();
    if (warp_active) {
      uint32_t lo[32], hi[32];
      tmem_ld32(tmem_row + 128, lo);
      tmem_ld32(tmem_row + 160, hi);
      tmem_wait_ld();
      if (live) store_row64(static_cast<T*>(p.d_planes) + ((size_t)bh * N + i) * kDh, lo, hi, p.scale);
    }
    if (BIAS == VRR_BIAS_TABLE) {
      asm volatile("bar.sync 1, 128;" ::: "memory");
      float* dst = p.d_bias_param + (size_t)h * (2 * N - 1);
      for (int t = tid; t < 2 * N - 1; t += 128) {
        const float v = hist[t];
        if (v != 0.f) atomicAdd(dst + t, v);
      }
    } else if (BIAS == VRR_BIAS_POLY) {
      float v[4] = {pw0, pw1, pw2, pw3};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
      }
      if (lane == 0) {
        float* dst = p.d_bias_param + (size_t)(p.bias_heads == 1 ? 0 : h) * p.bias_len;
        for (int k = 0; k < p.bias_len && k < 4; ++k) atomicAdd(dst + k, v[k]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem_base, kTmemCols);
}

// ============================================================================================ dK, dV
template <typename T, int BIAS>
__global__ void __launch_bounds__(kThreads, 2)
attn_bwd_dkv_tc2_kernel(const __grid_constant__ CUtensorMap tmap_pl, const __grid_constant__ CUtensorMap tmap_do,
                        const Bwd2Params p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sK = smem;
  uint8_t* sV = sK + kResB;
  uint8_t* sQr = sV + kResB;                // Q ring  [kSt][4 KB]
  uint8_t* sGr = sQr + kSt * kTileB;        // dO ring [kSt][4 KB]
  const int npad = ((p.N + kT - 1) / kT) * kT;
  float2* stats = reinterpret_cast<float2*>(sGr + kSt * kTileB);  // [npad] (lse*log2e, delta)
  float* lut = reinterpret_cast<float*>(stats + npad);
  uint16_t* key_yx = reinterpret_cast<uint16_t*>(lut + p.lut_floats);
  const int key_yx_bytes = (BIAS == VRR_BIAS_POLY) ? ((p.N * 2 + 15) & ~15) : 0;
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(key_yx) + key_yx_bytes);
  uint64_t* bar_full = bars;              // [kSt] Q and dO tile landed
  uint64_t* bar_empty = bars + kSt;       // [kSt] dV / dK MMAs of the tile retired
  uint64_t* bar_kv = bars + 2 * kSt;
  uint64_t* bar_s = bars + 2 * kSt + 1;   // [2]
  uint64_t* bar_p = bars + 2 * kSt + 3;   // [2]
  uint64_t* bar_done = bars + 2 * kSt + 5;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kSt + 6);

  const int tid = threadIdx.x, warp = tid >> 5;
  const int N = p.N, H = p.H;
  const int bh = blockIdx.y, b = bh / H, h = bh - b * H;
  const int j0 = blockIdx.x * kRows;
  const int ntiles = (N + kT - 1) / kT;
  const int BHN = p.B * H * N;

  if (warp == 4) {
    if (tid == 128) {
      for (int s = 0; s < kSt; ++s) {
        mbar_init(&bar_full[s], 1);
        mbar_init(&bar_empty[s], 1);
      }
      mbar_init(bar_kv, 1);
      for (int s = 0; s < 2; ++s) {
        mbar_init(&bar_s[s], 1);
        mbar_init(&bar_p[s], 128);
      }
      mbar_init(bar_done, 1);
      fence_mbar_init();
    }
    __syncwarp();
    if (elect_one()) {
      tma_prefetch_desc(&tmap_pl);
      tma_prefetch_desc(&tmap_do);
      mbar_expect_tx(bar_kv, 2 * kResB);
#pragma unroll
      for (int r = 0; r < kRows / kT; ++r) {
        tma_load_2d(sK + r * kTileB, &tmap_pl, bar_kv, 0, BHN + bh * N + j0 + r * kT);
        tma_load_2d(sV + r * kTileB, &tmap_pl, bar_kv, 0, 2 * BHN + bh * N + j0 + r * kT);
      }
      for (int s = 0; s < kSt && s < ntiles; ++s) {
        mbar_expect_tx(&bar_full[s], 2 * kTileB);
        tma_load_2d(sQr + s * kTileB, &tmap_pl, &bar_full[s], 0, bh * N + s * kT);
        tma_load_2d(sGr + s * kTileB, &tmap_do, &bar_full[s], h * kDh, b * N + s * kT);
      }
    }
    __syncwarp();
    tmem_alloc(tmem_slot, kTmemCols);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 4) {
    const uint64_t desc_k = smem_desc_sw128(smem_u32(sK));
    const uint64_t desc_v = smem_desc_sw128(smem_u32(sV));
    constexpr uint32_t idesc_s = idesc_16<T>(kRows, kT, 0, 0);
    constexpr uint32_t idesc_acc = idesc_16<T>(kRows, kDh, 0, 1);
    auto issue_st = [&](int t) {  // S^T(t), dP^T(t) into buffer t & 1
      const int st = t % kSt;
      mbar_wait(&bar_full[st], (uint32_t)((t / kSt) & 1));
      tc_fence_after();
      if (elect_one()) {
        const uint64_t dq = smem_desc_sw128(smem_u32(sQr + st * kTileB));
        const uint64_t dg = smem_desc_sw128(smem_u32(sGr + st * kTileB));
        const uint32_t cs = tmem_base + (t & 1) * kT, cp = tmem_base + 64 + (t & 1) * kT;
#pragma unroll
        for (int k = 0; k < 4; ++k) mma_ss(cs, desc_k + 2 * k, dq + 2 * k, idesc_s, k > 0);
#pragma unroll
        for (int k = 0; k < 4; ++k) mma_ss(cp, desc_v + 2 * k, dg + 2 * k, idesc_s, k > 0);
        mma_commit(&bar_s[t & 1]);
      }
      __syncwarp();
    };
    mbar_wait(bar_kv, 0);
    issue_st(0);
    for (int t = 0; t < ntiles; ++t) {
      const int st = t % kSt;
      if (t + 1 < ntiles) issue_st(t + 1);
      mbar_wait(&bar_p[t & 1], (uint32_t)((t >> 1) & 1));
      tc_fence_after();
      if (elect_one()) {
        const uint64_t dq = smem_desc_sw128(smem_u32(sQr + st * kTileB));
        const uint64_t dg = smem_desc_sw128(smem_u32(sGr + st * kTileB));
        const uint32_t ap = tmem_base + (t & 1) * kT, ad = tmem_base + 64 + (t & 1) * kT;
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) mma_ts(tmem_base + 128, ap + kk * 8, dg + 128 * kk, idesc_acc, (t | kk) != 0);  // dV
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) mma_ts(tmem_base + 192, ad + kk * 8, dq + 128 * kk, idesc_acc, (t | kk) != 0);  // dK
        mma_commit(&bar_empty[st]);
        if (t == ntiles - 1) mma_commit(bar_done);
      }
      __syncwarp();
      if (t >= 1 && t - 1 + kSt < ntiles) {
        const int sp = (t - 1) % kSt, tn = t - 1 + kSt;
        mbar_wait(&bar_empty[sp], (uint32_t)(((t - 1) / kSt) & 1));
        if (elect_one()) {
          mbar_expect_tx(&bar_full[sp], 2 * kTileB);
          tma_load_2d(sQr + sp * kTileB, &tmap_pl, &bar_full[sp], 0, bh * N + tn * kT);
          tma_load_2d(sGr + sp * kTileB, &tmap_do, &bar_full[sp], h * kDh, b * N + tn * kT);
        }
        __syncwarp();
      }
    }
  } else {
    const int j = j0 + tid;
    const int jc = min(j, N - 1);
    const bool live = j < N;
    const bool warp_active = (j0 + warp * 32) < N;
    const uint32_t tmem_row = tmem_base + ((uint32_t)(warp * 32) << 16);
    fill_lut2<BIAS>(lut, key_yx, p, h, tid);
    for (int t = tid; t < npad; t += 128) {
      float2 v;
      v.x = t < N ? p.lse[(size_t)bh * N + t] * kLog2e : INFINITY;  // +inf -> P = 0 for padded queries
      v.y = t < N ? p.delta[(size_t)bh * N + t] : 0.f;
      stats[t] = v;
    }
    int yj = 0, xj = 0;
    if (BIAS == VRR_BIAS_POLY) {
      const int pj = jc > 0 ? jc - 1 : 0;
      yj = pj % p.bias_grid;
      xj = pj / p.bias_grid;
    }
    asm volatile("bar.sync 1, 128;" ::: "memory");

    for (int t = 0; t < ntiles; ++t) {
      const int sb = t & 1;
      mbar_wait(&bar_s[sb], (uint32_t)((t >> 1) & 1));
      tc_fence_after();
      if (warp_active) {
        uint32_t sr[32], dr[32], pp[16], pd[16];
        tmem_ld32(tmem_row + sb * kT, sr);
        tmem_ld32(tmem_row + 64 + sb * kT, dr);
        tmem_wait_ld();
#pragma unroll
        for (int e = 0; e < kT; ++e) {
          const int i = t * kT + e;  // query index = accumulator column
          const float2 stt = stats[i];
          float x = fmaf(__uint_as_float(sr[e]), p.scale_log2, -stt.x);
          if (BIAS == VRR_BIAS_TABLE) {
            x += lut[min(max(i - jc + N - 1, 0), 2 * N - 2)];
          } else if (BIAS == VRR_BIAS_POLY) {
            const int yx = key_yx[min(i, N - 1)];
            const int dist = abs(yj - (yx >> 8)) + abs(xj - (yx & 255));
            x += (i == 0 || jc == 0) ? 0.f : lut[dist];
          }
          const float pr = ex2(x);
          const float ds = pr * (__uint_as_float(dr[e]) - stt.y);
          if (e & 1) {
            pp[e >> 1] = Elem16<T>::pack2(__uint_as_float(sr[e - 1]), pr);
            pd[e >> 1] = Elem16<T>::pack2(__uint_as_float(dr[e - 1]), ds);
          } else {
            sr[e] = __float_as_uint(pr);
            dr[e] = __float_as_uint(ds);
          }
        }
        tmem_st16(tmem_row + sb * kT, pp);        // P^T  over S^T
        tmem_st16(tmem_row + 64 + sb * kT, pd);   // dS^T over dP^T
        tmem_wait_st();
      }
      tc_fence_before();
      mbar_arrive(&bar_p[sb]);
    }

    mbar_wait(bar_done, 0);
    tc_fence_after();
    if (warp_active) {
      uint32_t lo[32], hi[32];
      const size_t plane = (size_t)BHN * kDh;
      tmem_ld32(tmem_row + 128, lo);
      tmem_ld32(tmem_row + 160, hi);
      tmem_wait_ld();
      if (live) store_row64(static_cast<T*>(p.d_planes) + 2 * plane + ((size_t)bh * N + j) * kDh, lo, hi, 1.f);
      __syncwarp();
      tmem_ld32(tmem_row + 192, lo);
      tmem_ld32(tmem_row + 224, hi);
      tmem_wait_ld();
      if (live) store_row64(static_cast<T*>(p.d_planes) + plane + ((size_t)bh * N + j) * kDh, lo, hi, p.scale);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem_base, kTmemCols);
}

size_t bwd2_smem_bytes(int N, const vrr_bias_desc* bias, int* lut_floats, bool dkv) {
  int lf = 0;
  const int mode = bias ? bias->mode : VRR_BIAS_NONE;
  if (mode == VRR_BIAS_TABLE) lf = 2 * N - 1;
  else if (mode == VRR_BIAS_POLY) lf = 2 * bias->grid - 1;
  lf = (lf + 3) & ~3;
  if (lut_floats) *lut_floats = lf;
  size_t extra = (size_t)lf * 4;
  if (mode == VRR_BIAS_POLY) extra += (size_t)((N * 2 + 15) & ~15);
  if (dkv) extra += (size_t)(((N + kT - 1) / kT) * kT) * 8;
  else if (mode == VRR_BIAS_TABLE) extra += (size_t)((2 * N - 1 + 3) & ~3) * 4 + 4 * 32 * 33 * 4;
  return 1024 + 2 * kResB + (size_t)2 * kSt * kTileB + extra + (4 * kSt + 8) * 8 + 16;
}

}  // namespace

bool attn_bwd_tc2_supported(int B, int H, int N, int Dh, const vrr_bias_desc* bias) {
  if (Dh != kDh || N < 1) return false;
  if ((long long)3 * B * H * N >= (1ll << 31)) return false;
  const int mode = bias ? bias->mode : VRR_BIAS_NONE;
  if (mode == VRR_BIAS_POLY && (bias->grid > 255 || bias->len > 4)) return false;
  // up to 113 KB keeps two CTAs per SM; the relative table at >= ~900 tokens needs more and runs one CTA per SM
  return bwd2_smem_bytes(N, bias, nullptr, false) <= 200 * 1024 && bwd2_smem_bytes(N, bias, nullptr, true) <= 200 * 1024;
}

template <typename T>
static int attn_bwd_tc2_t(const void* planes, const vrr_bias_desc* bias, const void* out, const void* d_out, const float* lse,
                          void* d_planes, float* d_bias_param, float* delta, int B, int H, int N, float scale,
                          cudaStream_t st) {
  VRR_REQUIRE(((uintptr_t)planes & 15) == 0 && ((uintptr_t)out & 15) == 0 && ((uintptr_t)d_out & 15) == 0 &&
                  ((uintptr_t)d_planes & 15) == 0,
              VRR_ERR_INVALID_ARG, "attn_bwd (tcgen05): planes / out / d_out / d_planes must be 16-byte aligned");
  const int E = H * kDh;
  CUtensorMap tm_pl, tm_do;
  if (int rc = make_tmap_2d(&tm_pl, planes, Elem16<T>::kTmap, (uint64_t)3 * B * H * N, kDh, kDh * 2, kT, 64)) return rc;
  if (int rc = make_tmap_2d(&tm_do, d_out, Elem16<T>::kTmap, (uint64_t)B * N, (uint64_t)E, (uint64_t)E * 2, kT, 64)) return rc;
  Bwd2Params p;
  p.out = out;
  p.d_out = d_out;
  p.lse = lse;
  p.delta = delta;
  p.d_planes = d_planes;
  p.B = B; p.H = H; p.N = N;
  p.scale = scale;
  p.scale_log2 = scale * kLog2e;
  const int mode = bias ? bias->mode : VRR_BIAS_NONE;
  p.bias_param = mode != VRR_BIAS_NONE ? bias->param : nullptr;
  p.d_bias_param = d_bias_param;
  p.bias_heads = mode != VRR_BIAS_NONE ? bias->heads : 0;
  p.bias_len = mode != VRR_BIAS_NONE ? bias->len : 0;
  p.bias_grid = mode != VRR_BIAS_NONE ? bias->grid : 0;
  if (mode != VRR_BIAS_NONE)
    VRR_CUDA(cudaMemsetAsync(d_bias_param, 0, (size_t)bias->heads * bias->len * sizeof(float), st));
  dim3 grid(ceil_div(N, kRows), B * H);
  const size_t smem_q = bwd2_smem_bytes(N, bias, &p.lut_floats, false);
  const size_t smem_kv = bwd2_smem_bytes(N, bias, &p.lut_floats, true);
#define LAUNCH(MODE)                                                                                             \
  do {                                                                                                           \
    VRR_SMEM_ATTR_ONCE((attn_bwd_dq_tc2_kernel<T, MODE>), 200 * 1024);                                           \
    VRR_SMEM_ATTR_ONCE((attn_bwd_dkv_tc2_kernel<T, MODE>), 200 * 1024);                                          \
    attn_bwd_dq_tc2_kernel<T, MODE><<<grid, kThreads, smem_q, st>>>(tm_pl, tm_do, p);                            \
    VRR_LAUNCHED();                                                                                              \
    attn_bwd_dkv_tc2_kernel<T, MODE><<<grid, kThreads, smem_kv, st>>>(tm_pl, tm_do, p);                          \
    VRR_LAUNCHED();                                                                                              \
  } while (0)
  if (mode == VRR_BIAS_TABLE) LAUNCH(VRR_BIAS_TABLE);
  else if (mode == VRR_BIAS_POLY) LAUNCH(VRR_BIAS_POLY);
  else LAUNCH(VRR_BIAS_NONE);
#undef LAUNCH
  return VRR_OK;
}

int attn_bwd_tc2(const void* planes, const vrr_bias_desc* bias, const void* out, const void* d_out, const float* lse,
                 void* d_planes, float* d_bias_param, float* delta, int B, int H, int N, int Dh, float scale, int dtype,
                 cudaStream_t st) {
  (void)Dh;
  if (dtype == VRR_F16)
    return attn_bwd_tc2_t<__half>(planes, bias, out, d_out, lse, d_planes, d_bias_param, delta, B, H, N, scale, st);
  return attn_bwd_tc2_t<__nv_bfloat16>(planes, bias, out, d_out, lse, d_planes, d_bias_param, delta, B, H, N, scale, st);
}

}  // namespace vrr
