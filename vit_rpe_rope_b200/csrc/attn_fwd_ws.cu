// Fused attention forward with a relative-table or polynomial bias for SHORT sequences (N <= 256: the 65..197-token
// ViT configurations), the whole sequence resident per item.  Replaces models/vit.py:71-88 of the reference
// (S = q k^T * scale (+ bias) -> softmax -> . v -> merge heads) without materialising S or P in HBM.
//
// Why a separate kernel.  clock64 timelines of the streaming kernel (attn_tc.cu, and of a persistent two-group
// variant of it that was measured and dropped: 147 us against 141 us) at 197 tokens
// showed the time going to per-tile fixed costs, not to math: every 64-key tile costs the issuer ~4 mbarrier waits
// (~90 cycles each even when already complete), ~16 small tcgen05.mma (N = 64: 32-48 cycles each at issue) and ~7
// commits, and costs each softmax thread a wait / fence / arrive round trip - more than the tile's exponentials.
// With the whole sequence resident the item needs ONE round trip:
//   * persistent grid, one CTA per SM, work item = one (image, head); Q, K, V of the next item are prefetched by
//     TMA into the other half of shared memory while the current one is processed;
//   * two softmax warpgroups (rows 0..127 and 128..255; thread = query row = TMEM lane), each with its OWN issuer
//     warp, so the groups drift out of phase and one group's exponentials overlap the other's MMAs and epilogue;
//   * S = Q K^T for a 128-row tile against ALL keys is 4 tcgen05.mma (M 128, N = round16(N) <= 256, K 16) into
//     TMEM columns [0, N); the softmax is exact two-pass (row max, then exponentials) straight out of TMEM - no
//     online rescaling; P (bf16 / fp16) is written in place over S; O = P V is N/16 tcgen05.mma with A = P from TMEM into
//     columns [192, 256), which S no longer needs by then;
//   * epilogue: O / l -> bf16 / fp16 -> 128-byte-swizzled staging -> one TMA store per warp through a 3-D map of
//     out[B][N][E] (rows past N are clipped by the hardware), so every global write is a full line.
// Bias: the head's relative-position table row is staged by a TMA bulk copy issued by the producer warp one item
// ahead (positional_encoding.py:58-75,93); the polynomial bias is a per-head distance LUT (:127-171).
#include "common.cuh"
#include "kernels.h"
#include "tc_common.cuh"

namespace vrr {

using namespace tc;

namespace {

constexpr int kDh = 64;
constexpr int kBoxBytes = 64 * kDh * 2;     // one TMA box: 64 rows x 128 B
constexpr int kSeqBytes = 256 * kDh * 2;    // 32 KB: up to 256 rows of Q, K or V
constexpr int kThreads = 384;               // warps 0-3 / 4-7 softmax groups, 8 producer, 9 / 10 issuers, 11 idle
constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kColO = 192;
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;
constexpr int kNumBars = 16;
constexpr int kSmemMax = 232448;

struct WsParams {
  float* lse;
  const float* bias_param;
  int B, H, N;
  float scale_log2;
  int bias_heads, bias_len, bias_grid;
  int lut_floats;   // floats of ONE group-private LUT
  int raw_floats;   // TABLE: floats of the TMA staging buffer
  int total_items;
};

__device__ __forceinline__ void table_span(const WsParams& p, int h, size_t& row_b, size_t& a0, size_t& a1) {
  row_b = (size_t)h * p.bias_len * 4;
  const size_t row_e = row_b + (size_t)p.bias_len * 4;
  const size_t tot = (size_t)p.bias_heads * p.bias_len * 4;
  a0 = row_b & ~size_t(15);
  a1 = (row_e + 15) & ~size_t(15);
  if (a1 > (tot & ~size_t(15))) a1 = tot & ~size_t(15);
}

// Walk the accumulator row of this thread in 32-column chunks (+ an optional 16-column tail).  Control flow is
// warp-uniform.  Deliberately a rolled loop with one register buffer: the straight-line double-buffered version
// made ptxas hoist loads until it needed 254 registers (the 384-thread CTA allows 168).
template <class F>
__device__ __forceinline__ void for_chunks(uint32_t t_s, int nch32, bool tail16, F& f) {
#pragma unroll 1
  for (int c = 0; c < nch32; ++c) {
    uint32_t buf[32];
    tmem_ld32(t_s + c * 32, buf);
    tmem_wait_ld();
    f.template run<32>(buf, c * 32);
  }
  if (tail16) {
    uint32_t t[16];
    tmem_ld16(t_s + nch32 * 32, t);
    tmem_wait_ld();
    f.template run<16>(t, nch32 * 32);
  }
}

// pass 1: mask, scale + bias (written back to TMEM for pass 2), row max
template <int BIAS>
struct Pass1 {
  const WsParams& p;
  uint32_t t_s;
  int i, yi, xi;
  const float* lut;
  const uint16_t* key_yx;
  float tm[4];
  template <int W>
  __device__ __forceinline__ void run(uint32_t (&s)[W], int j0) {
    const bool full = j0 + W <= p.N;  // warp-uniform: only the last chunk has keys past the sequence
#pragma unroll
    for (int jl = 0; jl < W; ++jl) {
      const int j = j0 + jl;
      float bsv;
      if (BIAS == VRR_BIAS_TABLE) {
        bsv = lut[min(max(i - j + p.N - 1, 0), 2 * p.N - 2)];
      } else {
        const int yx = key_yx[min(j, p.N - 1)];
        const int dist = abs(yi - (yx >> 8)) + abs(xi - (yx & 255));
        bsv = (i == 0 || j == 0) ? 0.f : lut[dist];
      }
      const float v = (full || j < p.N) ? fmaf(__uint_as_float(s[jl]), p.scale_log2, bsv) : -INFINITY;
      s[jl] = __float_as_uint(v);
      tm[jl & 3] = fmaxf(tm[jl & 3], v);
    }
    if constexpr (W == 32) tmem_st32(t_s + j0, s);
    else tmem_st16(t_s + j0, s);
  }
};

// pass 2: exponentials against the row max, row sum, P (pairs of T) written in place over S; masked keys hold -inf
// from pass 1
template <typename T>
struct Pass2 {
  uint32_t t_s;
  float neg_m;
  float ls[2];
  template <int W>
  __device__ __forceinline__ void run(const uint32_t (&s)[W], int j0) {
#pragma unroll
    for (int q = 0; q < W / 16; ++q) {
      uint32_t packed[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int jl = q * 16 + 2 * e;
        const float p0 = ex2(__uint_as_float(s[jl]) + neg_m), p1 = ex2(__uint_as_float(s[jl + 1]) + neg_m);
        ls[0] += p0;
        ls[1] += p1;
        packed[e] = Elem16<T>::pack2(p0, p1);
      }
      tmem_st8(t_s + (j0 >> 1) + q * 8, packed);
    }
  }
};

template <typename T, int BIAS>
__global__ void __launch_bounds__(kThreads, 1)
attn_fwd_ws_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap_out,
                   const __grid_constant__ WsParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;                               // [256 rows][128 B]
  uint8_t* sK = sQ + kSeqBytes;                     // [2 items][256 rows][128 B]
  uint8_t* sV = sK + 2 * kSeqBytes;                 // [2 items][256 rows][128 B]
  uint8_t* sOut = sV + 2 * kSeqBytes;               // [8 warps][32 rows][128 B] swizzled staging for the TMA store
  float* lut_raw = reinterpret_cast<float*>(sOut + 8 * 4096);
  float* lut_wg = lut_raw + p.raw_floats;
  uint16_t* key_yx = reinterpret_cast<uint16_t*>(lut_wg + 2 * p.lut_floats);
  const int key_yx_bytes = (BIAS == VRR_BIAS_POLY) ? ((p.N * 2 + 15) & ~15) : 0;
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(key_yx) + key_yx_bytes);
  uint64_t* bar_qfull = bars;            // Q landed
  uint64_t* bar_qempty = bars + 1;       // S MMAs of every group retired -> Q reusable
  uint64_t* bar_kvfull = bars + 2;       // [2] K and V of the item landed
  uint64_t* bar_kvempty = bars + 4;      // [2] PV MMAs of every group retired
  uint64_t* bar_sfull = bars + 6;        // [2 groups] S ready
  uint64_t* bar_pfull = bars + 8;        // [2] P stored (128 arrivals)
  uint64_t* bar_ofull = bars + 10;       // [2] O ready
  uint64_t* bar_oempty = bars + 12;      // [2] epilogue has read O (128 arrivals): the group's TMEM is free
  uint64_t* bar_lutfull = bars + 14;
  uint64_t* bar_lutempty = bars + 15;    // 256 arrivals
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kNumBars);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N = p.N, H = p.H;
  const int total = p.total_items;
  const int BHN = p.B * H * N;
  const int npad = (N + 15) & ~15;       // MMA N of S, K extent of PV
  const int nbox = (N + 63) >> 6;
  const int nwg = N > 128 ? 2 : 1;

  if (tid == 0) {
    mbar_init(bar_qfull, 1);
    mbar_init(bar_qempty, nwg);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&bar_kvfull[s], 1);
      mbar_init(&bar_kvempty[s], nwg);
      mbar_init(&bar_sfull[s], 1);
      mbar_init(&bar_pfull[s], 128);
      mbar_init(&bar_ofull[s], 1);
      mbar_init(&bar_oempty[s], 128);
    }
    mbar_init(bar_lutfull, 1);
    mbar_init(bar_lutempty, 256);
    fence_mbar_init();
  }
  if (BIAS == VRR_BIAS_POLY) {
    for (int t = tid; t < N; t += kThreads) {
      const int pt = t > 0 ? t - 1 : 0;
      key_yx[t] = (uint16_t)(((pt % p.bias_grid) << 8) | (pt / p.bias_grid));
    }
  }
  __syncwarp();
  if (warp == 8) tmem_alloc(tmem_slot, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // Producer / issuer warps run converged and issue under elect_one(): ptxas then keeps descriptors in uniform
  // registers and emits back-to-back UTCHMMA / UTMALDG (under `if (lane == 0)` every one of them is wrapped in an
  // elect-and-branch loop costing ~100 cycles).
  if (warp == 8) {
    // ============================================ TMA producer ============================================
    if (elect_one()) {
      tma_prefetch_desc(&tmap);
      tma_prefetch_desc(&tmap_out);
    }
    __syncwarp();
    int k = 0;
    for (int bh = blockIdx.x; bh < total; bh += gridDim.x, ++k) {
      const int kb = k & 1;
      mbar_wait(&bar_kvempty[kb], (uint32_t)(((k >> 1) & 1) ^ 1));
      if (elect_one()) {
        mbar_expect_tx(&bar_kvfull[kb], (uint32_t)(2 * nbox) * kBoxBytes);
        for (int j = 0; j < nbox; ++j)
          tma_load_2d(sK + kb * kSeqBytes + j * kBoxBytes, &tmap, &bar_kvfull[kb], 0, BHN + bh * N + j * 64);
        for (int j = 0; j < nbox; ++j)
          tma_load_2d(sV + kb * kSeqBytes + j * kBoxBytes, &tmap, &bar_kvfull[kb], 0, 2 * BHN + bh * N + j * 64);
      }
      __syncwarp();
      if (BIAS == VRR_BIAS_TABLE) {
        mbar_wait(bar_lutempty, (uint32_t)((k & 1) ^ 1));
        size_t row_b, a0, a1;
        table_span(p, bh % H, row_b, a0, a1);
        if (elect_one()) {
          if (a1 > a0) {
            mbar_expect_tx(bar_lutfull, (uint32_t)(a1 - a0));
            bulk_load_1d(lut_raw, reinterpret_cast<const uint8_t*>(p.bias_param) + a0, (uint32_t)(a1 - a0), bar_lutfull);
          } else {
            mbar_arrive(bar_lutfull);
          }
        }
        __syncwarp();
      }
      mbar_wait(bar_qempty, (uint32_t)((k & 1) ^ 1));
      if (elect_one()) {
        mbar_expect_tx(bar_qfull, (uint32_t)nbox * kBoxBytes);
        for (int j = 0; j < nbox; ++j) tma_load_2d(sQ + j * kBoxBytes, &tmap, bar_qfull, 0, bh * N + j * 64);
      }
      __syncwarp();
    }
  } else if (warp == 9 || warp == 10) {
    // ============================================ MMA issuer of group w ===================================
    const int w = warp - 9;
    if (w < nwg) {
      const uint32_t tmem_w = tmem_base + (uint32_t)(w * 256);
      const uint32_t idesc_s = idesc_16<T>(128, npad, 0, 0);
      constexpr uint32_t idesc_o = idesc_16<T>(128, kDh, 0, 1);
      const uint64_t dq = smem_desc_sw128(smem_u32(sQ + w * (128 * kDh * 2)));
      const int ksteps = npad >> 4;
      int k = 0;
      for (int bh = blockIdx.x; bh < total; bh += gridDim.x, ++k) {
        const int kb = k & 1;
        const uint32_t par = (uint32_t)(k & 1);
        mbar_wait(bar_qfull, par);
        mbar_wait(&bar_kvfull[kb], (uint32_t)((k >> 1) & 1));
        mbar_wait(&bar_oempty[w], par ^ 1);  // the epilogue of the previous item has read O: the group's TMEM is free
        tc_fence_after();
        if (elect_one()) {
          const uint64_t dk = smem_desc_sw128(smem_u32(sK + kb * kSeqBytes));
#pragma unroll
          for (int kk = 0; kk < kDh / 16; ++kk) mma_ss(tmem_w, dq + 2 * kk, dk + 2 * kk, idesc_s, kk > 0);
          mma_commit(&bar_sfull[w]);
          mma_commit(bar_qempty);
        }
        __syncwarp();
        mbar_wait(&bar_pfull[w], par);
        tc_fence_after();
        if (elect_one()) {
          const uint64_t dv = smem_desc_sw128(smem_u32(sV + kb * kSeqBytes));
#pragma unroll
          for (int kk = 0; kk < 16; ++kk)
            if (kk < ksteps) mma_ts(tmem_w + kColO, tmem_w + kk * 8, dv + 128 * kk, idesc_o, kk > 0);
          mma_commit(&bar_ofull[w]);
          mma_commit(&bar_kvempty[kb]);
        }
        __syncwarp();
      }
    }
  } else if (warp < 8) {
    // ============================================ softmax groups ==========================================
    const int w = warp >> 2, wq = warp & 3, r = tid & 127;
    const int i = w * 128 + r;
    const bool active = w < nwg;
    const bool warp_active = (w * 128 + wq * 32) < N;
    const uint32_t tmem_row = tmem_base + (uint32_t)(w * 256) + ((uint32_t)(wq * 32) << 16);
    float* lut = lut_wg + w * p.lut_floats;
    uint8_t* my_stage = sOut + warp * 4096;
    const int nch32 = npad >> 5;
    const bool tail16 = (npad & 31) != 0;
    bool lut_valid = false;
    const bool store_leader = elect_one();  // the same lane issues, commits and waits for this warp's TMA stores
    int yi = 0, xi = 0;
    if (BIAS == VRR_BIAS_POLY) {
      const int pi = i > 0 ? i - 1 : 0;
      yi = pi % p.bias_grid;
      xi = pi / p.bias_grid;
    }
    int k = 0;
    for (int bh = blockIdx.x; bh < total; bh += gridDim.x, ++k) {
      const int b = bh / H, h = bh - b * H;
      const uint32_t par = (uint32_t)(k & 1);
      if (BIAS == VRR_BIAS_TABLE) {
        mbar_wait(bar_lutfull, par);
        if (active) {
          size_t row_b, a0, a1;
          table_span(p, h, row_b, a0, a1);
          const int have = a1 > row_b ? (int)((a1 - row_b) / 4) : 0;  // elements the bulk copy delivered
          const float* src = lut_raw + (row_b - a0) / 4;
          const float* grow = p.bias_param + (size_t)h * p.bias_len;
          asm volatile("bar.sync %0, 128;" ::"r"(1 + w) : "memory");  // every row of the group left the previous item
          for (int t = r; t < p.bias_len; t += 128) lut[t] = (t < have ? src[t] : __ldg(grow + t)) * kLog2e;
        }
        mbar_arrive(bar_lutempty);
        if (active) asm volatile("bar.sync %0, 128;" ::"r"(1 + w) : "memory");
      } else if (BIAS == VRR_BIAS_POLY) {
        if (active && (!lut_valid || p.bias_heads > 1)) {
          const float* c = p.bias_param + (size_t)(p.bias_heads == 1 ? 0 : h) * p.bias_len;
          asm volatile("bar.sync %0, 128;" ::"r"(1 + w) : "memory");
          for (int d = r; d < 2 * p.bias_grid - 1; d += 128) {
            float x = (float)d, pw = 1.f, acc = 0.f;
            for (int q = 0; q < p.bias_len; ++q) {
              acc = fmaf(pw, c[q], acc);
              pw *= x;
            }
            lut[d] = acc * kLog2e;
          }
          asm volatile("bar.sync %0, 128;" ::"r"(1 + w) : "memory");
          lut_valid = true;
        }
      }
      if (!active) continue;

      mbar_wait(&bar_sfull[w], par);
      tc_fence_after();
      float m_row = 0.f, l_row = 1.f;
      if (warp_active) {
        Pass1<BIAS> p1{p, tmem_row, i, yi, xi, lut, key_yx, {-INFINITY, -INFINITY, -INFINITY, -INFINITY}};
        for_chunks(tmem_row, nch32, tail16, p1);
        m_row = fmaxf(fmaxf(p1.tm[0], p1.tm[1]), fmaxf(p1.tm[2], p1.tm[3]));
        tmem_wait_st();
        Pass2<T> p2{tmem_row, -m_row, {0.f, 0.f}};
        for_chunks(tmem_row, nch32, tail16, p2);
        l_row = p2.ls[0] + p2.ls[1];
        tmem_wait_st();
      }
      tc_fence_before();
      mbar_arrive(&bar_pfull[w]);

      // ---- epilogue: O / l -> T -> swizzled staging -> TMA store; lse ---------------------------
      mbar_wait(&bar_ofull[w], par);
      tc_fence_after();
      uint32_t olo[32], ohi[32];
      if (warp_active) {
        tmem_ld32(tmem_row + kColO, olo);
        tmem_ld32(tmem_row + kColO + 32, ohi);
        tmem_wait_ld();
      }
      tc_fence_before();
      mbar_arrive(&bar_oempty[w]);
      if (warp_active) {
        const float inv = 1.f / l_row;
        if (store_leader) bulk_wait_read<0>();  // the previous item's store has finished reading the staging buffer
        __syncwarp();
        const uint32_t row_base = smem_u32(my_stage) + (uint32_t)lane * 128u;
        const uint32_t sw = (uint32_t)(lane & 7);
#pragma unroll
        for (int c8 = 0; c8 < 4; ++c8)
          st_shared_v4(row_base + (((uint32_t)c8 ^ sw) << 4),
                       Elem16<T>::pack2(__uint_as_float(olo[c8 * 8 + 0]) * inv, __uint_as_float(olo[c8 * 8 + 1]) * inv),
                       Elem16<T>::pack2(__uint_as_float(olo[c8 * 8 + 2]) * inv, __uint_as_float(olo[c8 * 8 + 3]) * inv),
                       Elem16<T>::pack2(__uint_as_float(olo[c8 * 8 + 4]) * inv, __uint_as_float(olo[c8 * 8 + 5]) * inv),
                       Elem16<T>::pack2(__uint_as_float(olo[c8 * 8 + 6]) * inv, __uint_as_float(olo[c8 * 8 + 7]) * inv));
#pragma unroll
        for (int c8 = 0; c8 < 4; ++c8)
          st_shared_v4(row_base + (((uint32_t)(c8 + 4) ^ sw) << 4),
                       Elem16<T>::pack2(__uint_as_float(ohi[c8 * 8 + 0]) * inv, __uint_as_float(ohi[c8 * 8 + 1]) * inv),
                       Elem16<T>::pack2(__uint_as_float(ohi[c8 * 8 + 2]) * inv, __uint_as_float(ohi[c8 * 8 + 3]) * inv),
                       Elem16<T>::pack2(__uint_as_float(ohi[c8 * 8 + 4]) * inv, __uint_as_float(ohi[c8 * 8 + 5]) * inv),
                       Elem16<T>::pack2(__uint_as_float(ohi[c8 * 8 + 6]) * inv, __uint_as_float(ohi[c8 * 8 + 7]) * inv));
        fence_proxy_async_smem();
        __syncwarp();
        if (store_leader) {
          tma_store_3d(&tmap_out, my_stage, h * kDh, w * 128 + wq * 32, b);
          bulk_commit();
        }
        if (i < N) p.lse[(size_t)bh * N + i] = (m_row + log2f(l_row)) * kLn2;
      }
    }
    if (warp_active && store_leader) bulk_wait<0>();  // stores complete before the CTA (and its shared memory) goes away
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) tmem_dealloc(tmem_base, kTmemCols);
}

size_t ws_smem_bytes(int N, const vrr_bias_desc* bias, int* lut_floats, int* raw_floats) {
  int lf = 0, rf = 0;
  const int mode = bias->mode;
  if (mode == VRR_BIAS_TABLE) {
    lf = (2 * N - 1 + 3) & ~3;
    rf = (2 * N - 1 + 8 + 3) & ~3;  // + slack for the aligned span
  } else {
    lf = (2 * bias->grid - 1 + 3) & ~3;
  }
  if (lut_floats) *lut_floats = lf;
  if (raw_floats) *raw_floats = rf;
  const size_t yx = mode == VRR_BIAS_POLY ? (size_t)((N * 2 + 15) & ~15) : 0;
  return 1024 + (size_t)5 * kSeqBytes + 8 * 4096 + (size_t)(rf + 2 * lf) * 4 + yx + (size_t)kNumBars * 8 + 16;
}

template <typename T, int MODE>
int ws_launch(const CUtensorMap& tmap, const CUtensorMap& tmap_out, const WsParams& p, int grid, size_t smem,
              cudaStream_t st) {
  VRR_SMEM_ATTR_ONCE((attn_fwd_ws_kernel<T, MODE>), kSmemMax);
  attn_fwd_ws_kernel<T, MODE><<<grid, kThreads, smem, st>>>(tmap, tmap_out, p);
  VRR_LAUNCHED();
  return VRR_OK;
}

}  // namespace

bool attn_fwd_ws_supported(int B, int H, int N, int Dh, const vrr_bias_desc* bias) {
  if (!bias || bias->mode == VRR_BIAS_NONE) return false;  // attn_fwd_tc4_kernel is faster without bias
  if (Dh != kDh || N < 1 || N > 256) return false;
  if ((long long)3 * B * H * N >= (1ll << 31)) return false;
  if (bias->mode == VRR_BIAS_POLY && bias->grid > 255) return false;
  return ws_smem_bytes(N, bias, nullptr, nullptr) <= (size_t)kSmemMax;
}

template <typename T>
static int attn_fwd_ws_t(const void* planes, const vrr_bias_desc* bias, void* out, float* lse, int B, int H, int N,
                         float scale, cudaStream_t st) {
  VRR_REQUIRE(((uintptr_t)planes & 15) == 0 && ((uintptr_t)out & 15) == 0, VRR_ERR_INVALID_ARG,
              "attn_fwd (tcgen05): planes/out must be 16-byte aligned");
  CUtensorMap tmap, tmap_out;
  if (int rc = make_tmap_2d(&tmap, planes, Elem16<T>::kTmap, (uint64_t)3 * B * H * N, kDh, kDh * 2, 64, 64)) return rc;
  const uint64_t E = (uint64_t)H * kDh;
  if (int rc = make_tmap_3d(&tmap_out, out, Elem16<T>::kTmap, E, (uint64_t)N, (uint64_t)B, E * 2, (uint64_t)N * E * 2, kDh, 32))
    return rc;
  WsParams p;
  p.lse = lse;
  p.B = B; p.H = H; p.N = N;
  p.scale_log2 = scale * kLog2e;
  const int mode = bias->mode;  // a bias: attn_fwd_ws_supported
  p.bias_param = bias->param;
  p.bias_heads = bias->heads;
  p.bias_len = bias->len;
  p.bias_grid = bias->grid;
  if (mode == VRR_BIAS_TABLE)
    VRR_REQUIRE(((uintptr_t)bias->param & 15) == 0, VRR_ERR_INVALID_ARG, "attn_fwd (tcgen05): bias table must be 16-byte aligned");
  p.total_items = B * H;
  const size_t smem = ws_smem_bytes(N, bias, &p.lut_floats, &p.raw_floats);
  const int grid = p.total_items < sm_count() ? p.total_items : sm_count();
  if (mode == VRR_BIAS_TABLE) return ws_launch<T, VRR_BIAS_TABLE>(tmap, tmap_out, p, grid, smem, st);
  return ws_launch<T, VRR_BIAS_POLY>(tmap, tmap_out, p, grid, smem, st);
}

int attn_fwd_ws(const void* planes, const vrr_bias_desc* bias, void* out, float* lse, int B, int H, int N, int Dh,
                float scale, int dtype, cudaStream_t st) {
  (void)Dh;
  if (dtype == VRR_F16) return attn_fwd_ws_t<__half>(planes, bias, out, lse, B, H, N, scale, st);
  return attn_fwd_ws_t<__nv_bfloat16>(planes, bias, out, lse, B, H, N, scale, st);
}

}  // namespace vrr
