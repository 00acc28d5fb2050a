// Fused attention forward on the 5th-generation tensor cores (tcgen05 + TMEM), bf16 or fp16, head dim 64, tiled over
// the keys: every N without bias, and N > 256 with a bias (attn_fwd_ws.cu takes the shorter biased sequences).
//
// Replaces models/vit.py:71-88 of the reference: S = q k^T * scale (+ relative-position table /
// polynomial bias) -> softmax -> . v -> merge heads, without materialising S or P in HBM.
//
// Both kernels: one CTA = 128 query rows of one (image, head), 160 threads - warps 0-3 softmax (thread t = query
// row t = TMEM lane t), warp 4 the issuer of every TMA load and tcgen05.mma.  Q and 64-key K / V tiles arrive by
// TMA (128-byte swizzle); S = Q K^T and O += P V (P from TMEM) accumulate in TMEM, O across all key tiles, with a
// lazy online-softmax rescale; epilogue O / l -> bf16 / fp16 -> out[b][i][h*64 ..], lse.
//   * attn_fwd_tc4_kernel (no bias): one S buffer, 2-stage ring, 128 TMEM columns, ~50 KB of shared memory, four
//     CTAs per SM;
//   * attn_fwd_tc2_kernel (relative table / polynomial bias): double-buffered S, 4-stage ring, 256 TMEM columns,
//     the bias row staged in shared memory (table row by a TMA bulk copy, polynomial as a distance LUT), two CTAs
//     per SM.
#include "common.cuh"
#include "kernels.h"
#include "tc_common.cuh"

namespace vrr {

using namespace tc;

namespace {

constexpr int kM = 128;       // query rows per CTA
constexpr int kDh = 64;
constexpr int kQBytes = kM * kDh * 2;  // 16 KB
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

struct FwdParams {
  void* out;  // element type T of the kernel
  float* lse;
  const float* bias_param;
  int B, H, N;
  float scale_log2;  // scale * log2(e)
  int bias_heads, bias_len, bias_grid;
  int lut_floats;    // shared-memory floats reserved for the LUT (incl. alignment slack)
  long long* dbg;    // optional phase timestamps (clock64) of one CTA, 8 per key tile; NULL in production
};

// =====================================================================================================
// attn_fwd_tc2_kernel (bias modes): a dedicated issuer warp, double-buffered S, O accumulated in TMEM.
//   warps 0-3 : softmax, thread t = query row t = TMEM lane t
//   warp 4    : issuer - TMA loads and every tcgen05.mma, descriptors kept warp-uniform
// 64-key tiles.  TMEM: S/P buffer 0 = cols [0,64), buffer 1 = [64,128), O = [128,192).
// The issuer runs one S tile ahead: S(t+1) = Q K(t+1)^T executes while the softmax warps work on
// tile t, and O += P(t) V(t) accumulates in TMEM across ALL key tiles, so the softmax warps never
// read O until the epilogue.  The running max only has to be a *reference* for exp2: it is updated
// (and O, l rescaled through tcgen05.ld/st) only when a row's tile max exceeds it by more than 2^8
// - P <= 256 is harmless in bf16, fp16 and fp32 - which after the first tile is rare.
constexpr int kV2KT = 64, kV2Stages = 4, kV2Threads = 160;
constexpr uint32_t kV2TmemCols = 256, kV2ColO = 128;
constexpr float kRescaleThreshold = 8.0f;  // log2 units
constexpr int kV2NumBars = 4 * kV2Stages + 9;

template <typename T, int BIAS>
__global__ void __launch_bounds__(kV2Threads, 2)
attn_fwd_tc2_kernel(const __grid_constant__ CUtensorMap tmap, const FwdParams p) {
  constexpr int kKT = kV2KT, kStages = kV2Stages;
  constexpr int kTileBytes = kKT * kDh * 2;  // 8 KB
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + kQBytes;                   // K ring [kStages][8 KB]
  uint8_t* sV = sK + kStages * kTileBytes;      // V ring [kStages][8 KB] (separate: K frees much earlier)
  float* lut_raw = reinterpret_cast<float*>(sV + kStages * kTileBytes);
  uint16_t* key_yx = reinterpret_cast<uint16_t*>(lut_raw + p.lut_floats);
  const int key_yx_bytes = (BIAS == VRR_BIAS_POLY) ? ((p.N * 2 + 15) & ~15) : 0;
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(key_yx) + key_yx_bytes);
  uint64_t* bar_kfull = bars;                   // [kStages] TMA K tile landed
  uint64_t* bar_vfull = bars + kStages;         // [kStages] TMA V tile landed
  uint64_t* bar_kempty = bars + 2 * kStages;    // [kStages] S(t) retired  -> K stage reusable
  uint64_t* bar_vempty = bars + 3 * kStages;    // [kStages] PV(t) retired -> V stage reusable
  uint64_t* bar_q = bars + 4 * kStages;
  uint64_t* bar_s = bars + 4 * kStages + 1;     // [2] S buffer ready (issuer commit -> softmax)
  uint64_t* bar_p = bars + 4 * kStages + 3;     // [2] P buffer ready (128 softmax arrivals -> issuer)
  uint64_t* bar_o = bars + 4 * kStages + 5;     // PV(t) retired (one phase per tile)
  uint64_t* bar_lut = bars + 4 * kStages + 6;
  // the LAST PV retired.  A separate single-phase barrier: a softmax thread does not observe every
  // phase of bar_o, so after its last arrival bar_o may be two phases behind and a parity wait on it
  // would alias (return early).
  uint64_t* bar_done = bars + 4 * kStages + 7;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4 * kStages + 8);

  const int tid = threadIdx.x, warp = tid >> 5;
  const int N = p.N, H = p.H;
  const int bh = blockIdx.y, b = bh / H, h = bh - b * H;
  const int m0 = blockIdx.x * kM;
  const int ntiles = (N + kKT - 1) / kKT;
  const int BHN = p.B * H * N;

  if (warp == 4) {
    // barriers first, then the TMA prologue, THEN the TMEM allocation: the loads' latency overlaps
    // the allocation and the LUT fill of the softmax warps
    if (tid == 128) {
      for (int s = 0; s < kStages; ++s) {
        mbar_init(&bar_kfull[s], 1);
        mbar_init(&bar_vfull[s], 1);
        mbar_init(&bar_kempty[s], 1);
        mbar_init(&bar_vempty[s], 1);
      }
      mbar_init(bar_done, 1);
      mbar_init(bar_q, 1);
      for (int s = 0; s < 2; ++s) {
        mbar_init(&bar_s[s], 1);
        mbar_init(&bar_p[s], 128);
      }
      mbar_init(bar_o, 1);
      mbar_init(bar_lut, 1);
      fence_mbar_init();
    }
    __syncwarp();
    if (elect_one()) {
      tma_prefetch_desc(&tmap);
      mbar_expect_tx(bar_q, kQBytes);
      tma_load_2d(sQ, &tmap, bar_q, 0, bh * N + m0);
      tma_load_2d(sQ + kTileBytes, &tmap, bar_q, 0, bh * N + m0 + kKT);
      for (int s = 0; s < kStages && s < ntiles; ++s) {
        mbar_expect_tx(&bar_kfull[s], kTileBytes);
        tma_load_2d(sK + s * kTileBytes, &tmap, &bar_kfull[s], 0, BHN + bh * N + s * kKT);
      }
      for (int s = 0; s < kStages && s < ntiles; ++s) {
        mbar_expect_tx(&bar_vfull[s], kTileBytes);
        tma_load_2d(sV + s * kTileBytes, &tmap, &bar_vfull[s], 0, 2 * BHN + bh * N + s * kKT);
      }
      if (BIAS == VRR_BIAS_TABLE) {
        // TMA bulk copy of the head's table row (rows of 2N-1 floats are not 16-byte aligned in general:
        // copy the enclosing aligned span that stays inside the table; the softmax warps patch the tail)
        const size_t row_b = (size_t)h * p.bias_len * 4, row_e = row_b + (size_t)p.bias_len * 4;
        const size_t tot = (size_t)p.bias_heads * p.bias_len * 4;
        const size_t a0 = row_b & ~size_t(15);
        size_t a1 = (row_e + 15) & ~size_t(15);
        if (a1 > (tot & ~size_t(15))) a1 = tot & ~size_t(15);
        if (a1 > a0) {
          mbar_expect_tx(bar_lut, (uint32_t)(a1 - a0));
          bulk_load_1d(lut_raw, reinterpret_cast<const uint8_t*>(p.bias_param) + a0, (uint32_t)(a1 - a0), bar_lut);
        } else {
          mbar_arrive(bar_lut);
        }
      }
    }
    __syncwarp();
    tmem_alloc(tmem_slot, kV2TmemCols);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 4) {
    // =========================================== issuer ===========================================
    const uint64_t desc_q = smem_desc_sw128(smem_u32(sQ));
    constexpr uint32_t idesc_s = idesc_16<T>(kM, kKT, 0, 0);
    constexpr uint32_t idesc_o = idesc_16<T>(kM, kDh, 0, 1);
    // S(0)
    mbar_wait(bar_q, 0);
    mbar_wait(&bar_kfull[0], 0);
    tc_fence_after();
    if (elect_one()) {
      const uint64_t desc_k = smem_desc_sw128(smem_u32(sK));
#pragma unroll
      for (int k = 0; k < kDh / 16; ++k) mma_ss(tmem_base, desc_q + 2 * k, desc_k + 2 * k, idesc_s, k > 0);
      mma_commit(&bar_s[0]);
      mma_commit(&bar_kempty[0]);
    }
    __syncwarp();
    for (int t = 0; t < ntiles; ++t) {
      const int stage = t % kStages;
      const uint32_t use_parity = (uint32_t)((t / kStages) & 1);
      if (t + 1 < ntiles) {  // run one S tile ahead, into the other S buffer
        const int sn = (t + 1) % kStages;
        mbar_wait(&bar_kfull[sn], (uint32_t)(((t + 1) / kStages) & 1));
        tc_fence_after();
        if (elect_one()) {
          const uint64_t desc_k = smem_desc_sw128(smem_u32(sK + sn * kTileBytes));
          const uint32_t d = tmem_base + ((t + 1) & 1) * kKT;
#pragma unroll
          for (int k = 0; k < kDh / 16; ++k) mma_ss(d, desc_q + 2 * k, desc_k + 2 * k, idesc_s, k > 0);
          mma_commit(&bar_s[(t + 1) & 1]);
          mma_commit(&bar_kempty[sn]);
        }
        __syncwarp();
      }
      // K(t) was consumed by S(t) (issued one iteration ago): refill its stage with K(t + kStages)
      if (t + kStages < ntiles) {
        mbar_wait(&bar_kempty[stage], use_parity);
        if (elect_one()) {
          mbar_expect_tx(&bar_kfull[stage], kTileBytes);
          tma_load_2d(sK + stage * kTileBytes, &tmap, &bar_kfull[stage], 0, BHN + bh * N + (t + kStages) * kKT);
        }
        __syncwarp();
      }
      // O += P(t) V(t)
      mbar_wait(&bar_vfull[stage], use_parity);
      mbar_wait(&bar_p[t & 1], (uint32_t)((t >> 1) & 1));
      tc_fence_after();
      if (elect_one()) {
        const uint64_t desc_v = smem_desc_sw128(smem_u32(sV + stage * kTileBytes));
        const uint32_t a = tmem_base + (t & 1) * kKT;
        const int nvalid = min(kKT, N - t * kKT);
        const int ksteps = (nvalid + 15) >> 4;
        for (int kk = 0; kk < ksteps; ++kk)
          mma_ts(tmem_base + kV2ColO, a + kk * 8, desc_v + 128 * kk, idesc_o, (t | kk) != 0);
        mma_commit(&bar_vempty[stage]);
        mma_commit(bar_o);
        if (t == ntiles - 1) mma_commit(bar_done);
      }
      __syncwarp();
      // V(t-1) was consumed by PV(t-1) (retired by now): refill its stage with V(t - 1 + kStages)
      if (t >= 1 && t - 1 + kStages < ntiles) {
        const int sp = (t - 1) % kStages;
        mbar_wait(&bar_vempty[sp], (uint32_t)(((t - 1) / kStages) & 1));
        if (elect_one()) {
          mbar_expect_tx(&bar_vfull[sp], kTileBytes);
          tma_load_2d(sV + sp * kTileBytes, &tmap, &bar_vfull[sp], 0, 2 * BHN + bh * N + (t - 1 + kStages) * kKT);
        }
        __syncwarp();
      }
    }
  } else {
    // =========================================== softmax ==========================================
    const int i = m0 + tid;
    const bool warp_active = (m0 + warp * 32) < N;
    const uint32_t tmem_row = tmem_base + ((uint32_t)(warp * 32) << 16);
    const float* lut = lut_raw;
    int yi = 0, xi = 0;
    if (BIAS == VRR_BIAS_TABLE) {
      const size_t row_b = (size_t)h * p.bias_len * 4, row_e = row_b + (size_t)p.bias_len * 4;
      const size_t tot = (size_t)p.bias_heads * p.bias_len * 4;
      const size_t a0 = row_b & ~size_t(15);
      size_t a1 = (row_e + 15) & ~size_t(15);
      if (a1 > (tot & ~size_t(15))) a1 = tot & ~size_t(15);
      const int have = a1 > row_b ? (int)((a1 - row_b) / 4) : 0;  // elements the bulk copy delivered
      float* lw = lut_raw + (row_b - a0) / 4;
      lut = lw;
      const float* grow = p.bias_param + (size_t)h * p.bias_len;
      mbar_wait(bar_lut, 0);
      for (int t = tid; t < p.bias_len; t += 128) lw[t] = (t < have ? lw[t] : grow[t]) * kLog2e;
      asm volatile("bar.sync 1, 128;" ::: "memory");
    } else if (BIAS == VRR_BIAS_POLY) {
      const float* c = p.bias_param + (size_t)(p.bias_heads == 1 ? 0 : h) * p.bias_len;
      for (int d = tid; d < 2 * p.bias_grid - 1; d += 128) {
        float x = (float)d, pw = 1.f, acc = 0.f;
        for (int k = 0; k < p.bias_len; ++k) {
          acc = fmaf(pw, c[k], acc);
          pw *= x;
        }
        lut_raw[d] = acc * kLog2e;
      }
      for (int t = tid; t < N; t += 128) {
        int pt = t > 0 ? t - 1 : 0;
        key_yx[t] = (uint16_t)(((pt % p.bias_grid) << 8) | (pt / p.bias_grid));
      }
      const int pi = i > 0 ? i - 1 : 0;
      yi = pi % p.bias_grid;
      xi = pi / p.bias_grid;
      asm volatile("bar.sync 1, 128;" ::: "memory");
    }

    float m_ref = -INFINITY, l_run = 0.f;
    for (int t = 0; t < ntiles; ++t) {
      const int sb = t & 1;
      const int nvalid = min(kKT, N - t * kKT);
      const bool dbg_on = p.dbg != nullptr && tid == 0 && blockIdx.x == 0 && blockIdx.y == gridDim.y / 2 && t < 8;
      long long* dbg = dbg_on ? p.dbg + t * 8 : nullptr;
      if (dbg_on) dbg[0] = clock64();
      mbar_wait(&bar_s[sb], (uint32_t)((t >> 1) & 1));
      tc_fence_after();
      if (dbg_on) dbg[1] = clock64();
      if (warp_active) {
        uint32_t sraw[kKT];
        tmem_ld32(tmem_row + sb * kKT, *reinterpret_cast<uint32_t(*)[32]>(&sraw[0]));
        tmem_ld32(tmem_row + sb * kKT + 32, *reinterpret_cast<uint32_t(*)[32]>(&sraw[32]));
        tmem_wait_ld();
        if (dbg_on) dbg[2] = clock64();
        if (nvalid < kKT) {
#pragma unroll
          for (int jl = 0; jl < kKT; ++jl)
            if (jl >= nvalid) sraw[jl] = 0xff800000u;  // -inf
        }
        float tmax = -INFINITY;
#pragma unroll
        for (int jl = 0; jl < kKT; ++jl) {
          const int j = t * kKT + jl;
          float bsv;
          if (BIAS == VRR_BIAS_TABLE) {
            bsv = lut[min(max(i - j + N - 1, 0), 2 * N - 2)];
          } else {
            const int yx = key_yx[min(j, N - 1)];
            const int dist = abs(yi - (yx >> 8)) + abs(xi - (yx & 255));
            bsv = (i == 0 || j == 0) ? 0.f : lut[dist];
          }
          const float v = fmaf(__uint_as_float(sraw[jl]), p.scale_log2, bsv);
          sraw[jl] = __float_as_uint(v);
          tmax = fmaxf(tmax, v);
        }
        if (dbg_on) dbg[3] = clock64();
        // reference-max update: warp-uniform decision (tcgen05.ld/st are warp-collective)
        const bool jump = tmax > m_ref + kRescaleThreshold;
        if (__any_sync(0xffffffffu, jump)) {
          const float m_new = fmaxf(m_ref, tmax);
          if (t > 0) {
            const float f = ex2(m_ref - m_new);  // 1 for rows whose reference did not move
            l_run *= f;
            // PV(t-1) retired.  Safe parity wait: S(t) was committed after PV(t-2), so having passed
            // bar_s(t) this thread knows bar_o is at phase t-1 or t - never further behind.
            mbar_wait(bar_o, (uint32_t)((t - 1) & 1));
            tc_fence_after();
#pragma unroll
            for (int half = 0; half < 2; ++half) {
              uint32_t o[32];
              tmem_ld32(tmem_row + kV2ColO + half * 32, o);
              tmem_wait_ld();
#pragma unroll
              for (int d = 0; d < 32; ++d) o[d] = __float_as_uint(__uint_as_float(o[d]) * f);
              tmem_st32(tmem_row + kV2ColO + half * 32, o);
            }
          }
          m_ref = m_new;
        }
        const float neg_m = -m_ref;
#pragma unroll
        for (int c = 0; c < kKT / 32; ++c) {
          uint32_t packed[16];
#pragma unroll
          for (int e = 0; e < 16; ++e) {
            const float a0 = __uint_as_float(sraw[c * 32 + 2 * e]), a1 = __uint_as_float(sraw[c * 32 + 2 * e + 1]);
            const float p0 = ex2(a0 + neg_m);
            const float p1 = ex2(a1 + neg_m);
            l_run += p0 + p1;
            packed[e] = Elem16<T>::pack2(p0, p1);
          }
          tmem_st16(tmem_row + sb * kKT + c * 16, packed);  // P over the first half of this S buffer
        }
        if (dbg_on) dbg[4] = clock64();
        tmem_wait_st();
      }
      tc_fence_before();
      mbar_arrive(&bar_p[sb]);
      if (dbg_on) dbg[5] = clock64();
    }

    // ---- epilogue: O / l -------------------------------------------------------------------------
    mbar_wait(bar_done, 0);
    tc_fence_after();
    if (warp_active) {
      uint32_t lo[32], hi[32];
      tmem_ld32(tmem_row + kV2ColO, lo);
      tmem_ld32(tmem_row + kV2ColO + 32, hi);
      tmem_wait_ld();
      if (i < N) {
        const float inv = 1.f / l_run;
        T* dst = static_cast<T*>(p.out) + ((size_t)b * N + i) * (size_t)(H * kDh) + h * kDh;
#pragma unroll
        for (int v8 = 0; v8 < 8; ++v8) {
          const uint32_t* src = v8 < 4 ? &lo[v8 * 8] : &hi[(v8 - 4) * 8];
          uint4 w;
          w.x = Elem16<T>::pack2(__uint_as_float(src[0]) * inv, __uint_as_float(src[1]) * inv);
          w.y = Elem16<T>::pack2(__uint_as_float(src[2]) * inv, __uint_as_float(src[3]) * inv);
          w.z = Elem16<T>::pack2(__uint_as_float(src[4]) * inv, __uint_as_float(src[5]) * inv);
          w.w = Elem16<T>::pack2(__uint_as_float(src[6]) * inv, __uint_as_float(src[7]) * inv);
          *reinterpret_cast<uint4*>(dst + v8 * 8) = w;
        }
        p.lse[(size_t)bh * N + i] = (m_ref + log2f(l_run)) * kLn2;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem_base, kV2TmemCols);
}

// =====================================================================================================
// attn_fwd_tc4_kernel (no bias, every N): the same tile loop with HALF the on-chip footprint per CTA and four CTAs
// per SM.  attn_fwd_tc2_kernel's layout at 1025 tokens runs at ~45 % of the exponential (MUFU) roof: with two CTAs
// per SM a scheduler holds two softmax warps, and each of them spends about half of a tile waiting (S barrier, tcgen05.ld,
// tcgen05.st, P barrier).  Here a CTA keeps ONE S buffer (P written in place, the next S issued right behind the PV
// MMA that reads it - the tensor pipe executes in issue order), a 2-stage K / V ring and 128 TMEM columns (S/P
// [0,64), O [64,128)), so four CTAs = four independent streams share an SM: a stream's barrier and tensor-pipe
// latencies are covered by the other three.  Registers are capped at ~100 by the residency, so a softmax thread
// walks its row twice (max pass, exp pass) in 16-column chunks re-read from TMEM, the next chunk's tcgen05.ld in
// flight behind the current one's arithmetic; scale-and-subtract and the row sum run on the packed fp32x2 pipe.
constexpr int kV4Stages = 2, kV4Threads = 160;
constexpr uint32_t kV4TmemCols = 128, kV4ColO = 64;
constexpr int kV4NumBars = 4 * kV4Stages + 4;
// pairs out of every 8 whose exponential takes the FMA-pipe polynomial (tc::ex2_poly2) instead of MUFU.EX2; of the
// shares 0..4, 2 was the fastest at 577 and 1025 tokens (profiles/r2_attn_long_probe.txt)
constexpr int kPolyPairs = 2;

__device__ __forceinline__ float v4_max16(const uint32_t (&r)[16], float mx) {
#pragma unroll
  for (int e = 0; e < 16; e += 2) mx = fmaxf(mx, fmaxf(__uint_as_float(r[e]), __uint_as_float(r[e + 1])));
  return mx;
}
template <bool FULL>
__device__ __forceinline__ float v4_max16m(const uint32_t (&r)[16], float mx, int first, int nvalid) {
  if constexpr (FULL) {
    return v4_max16(r, mx);
  } else {
#pragma unroll
    for (int e = 0; e < 16; ++e)
      if (first + e < nvalid) mx = fmaxf(mx, __uint_as_float(r[e]));
    return mx;
  }
}
// P = 2^(s * scale - m) for 16 scores -> 8 packed pairs of T; the row sum accumulates in l2.  kPolyPairs of the 8 pairs
// take the polynomial, the others MUFU.EX2.
template <typename T, bool FULL>
__device__ __forceinline__ void v4_exp16(const uint32_t (&r)[16], uint32_t (&pk)[8], float2 sc2, float2 nm2, float2& l2,
                                         int first, int nvalid) {
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const float2 x = __ffma2_rn(make_float2(__uint_as_float(r[2 * e]), __uint_as_float(r[2 * e + 1])), sc2, nm2);
    // spread the polynomial pairs between the MUFU ones: e * kPolyPairs / 8 steps at the chosen pairs
    const bool poly = ((e + 1) * kPolyPairs) / 8 != (e * kPolyPairs) / 8;
    float2 pv = poly ? ex2_poly2(x) : make_float2(ex2(x.x), ex2(x.y));
    if (!FULL) {
      if (first + 2 * e >= nvalid) pv.x = 0.f;
      if (first + 2 * e + 1 >= nvalid) pv.y = 0.f;
    }
    l2 = __fadd2_rn(l2, pv);
    pk[e] = Elem16<T>::pack2(pv.x, pv.y);
  }
}

// one key tile of one query row: lazy reference-max update, then P over the first 32 of the 64 columns S occupied
template <typename T, bool FULL>
__device__ __forceinline__ void v4_tile(uint32_t trow, int nvalid, int t, float scale_log2, float& m_ref, float& l_run) {
  uint32_t ab[32];
  uint32_t(&a)[16] = *reinterpret_cast<uint32_t(*)[16]>(&ab[0]);
  uint32_t(&b)[16] = *reinterpret_cast<uint32_t(*)[16]>(&ab[16]);
  // ---- pass 1: tile max (two 32-column loads: one TMEM round trip less than four 16-column ones) ----
  // The ragged LAST tile (every ViT sequence is 64 k + a few tokens: 65, 197, 577, 1025) was issued as a narrow MMA of
  // nc = round16(nvalid) columns and is walked in nc / 16 chunks only.
  float tmax = -INFINITY;
  const int nchunks = FULL ? 4 : (nvalid + 15) >> 4;
  if (FULL) {
    tmem_ld32(trow, ab);
    tmem_wait_ld();
    tmax = v4_max16(a, tmax);
    tmax = v4_max16(b, tmax);
    tmem_ld32(trow + 32, ab);
    tmem_wait_ld();
    tmax = v4_max16(a, tmax);
    tmax = v4_max16(b, tmax);
  } else {
    for (int c = 0; c < nchunks; ++c) {
      tmem_ld16(trow + c * 16, a);
      tmem_wait_ld();
      tmax = v4_max16m<false>(a, tmax, c * 16, nvalid);
    }
  }
  tmax *= scale_log2;
  tmem_ld16(trow, a);  // first chunk of pass 2
  const bool jump = tmax > m_ref + kRescaleThreshold;
  if (__any_sync(0xffffffffu, jump)) {
    const float m_new = fmaxf(m_ref, tmax);
    if (t > 0) {
      // PV(t-1) has retired: bar_s(t) was committed behind it
      const float f = ex2(m_ref - m_new);  // 1 for rows whose reference did not move
      l_run *= f;
      tmem_wait_ld();
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        tmem_ld16(trow + kV4ColO + q * 16, b);
        tmem_wait_ld();
#pragma unroll
        for (int d = 0; d < 16; ++d) b[d] = __float_as_uint(__uint_as_float(b[d]) * f);
        tmem_st16(trow + kV4ColO + q * 16, b);
      }
    }
    m_ref = m_new;
  }
  // ---- pass 2 ----
  const float2 sc2 = make_float2(scale_log2, scale_log2), nm2 = make_float2(-m_ref, -m_ref);
  float2 l2 = make_float2(0.f, 0.f);
  uint32_t pk[8];
  if (FULL) {
    tmem_wait_ld();
    tmem_ld16(trow + 16, b);
    v4_exp16<T, true>(a, pk, sc2, nm2, l2, 0, nvalid);
    tmem_st8(trow, pk);  // columns [0,8): scores already consumed
    tmem_wait_ld();
    tmem_ld16(trow + 32, a);
    v4_exp16<T, true>(b, pk, sc2, nm2, l2, 16, nvalid);
    tmem_st8(trow + 8, pk);
    tmem_wait_ld();
    tmem_ld16(trow + 48, b);
    v4_exp16<T, true>(a, pk, sc2, nm2, l2, 32, nvalid);
    tmem_st8(trow + 16, pk);
    tmem_wait_ld();
    v4_exp16<T, true>(b, pk, sc2, nm2, l2, 48, nvalid);
    tmem_st8(trow + 24, pk);
  } else {
    for (int c = 0; c < nchunks; ++c) {
      if (c > 0) tmem_ld16(trow + c * 16, a);
      tmem_wait_ld();
      v4_exp16<T, false>(a, pk, sc2, nm2, l2, c * 16, nvalid);
      tmem_st8(trow + c * 8, pk);  // columns [8c, 8c+8) lie below every chunk still to be read
    }
  }
  l_run += l2.x + l2.y;
  tmem_wait_st();
}

template <typename T>
__global__ void __launch_bounds__(kV4Threads, 4)
attn_fwd_tc4_kernel(const __grid_constant__ CUtensorMap tmap, const FwdParams p) {
  constexpr int kKT = kV2KT, kStages = kV4Stages;
  constexpr int kTileBytes = kKT * kDh * 2;  // 8 KB
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + kQBytes;
  uint8_t* sV = sK + kStages * kTileBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sV + kStages * kTileBytes);
  uint64_t* bar_kfull = bars;                 // [2] TMA K tile landed
  uint64_t* bar_vfull = bars + kStages;       // [2] TMA V tile landed
  uint64_t* bar_kempty = bars + 2 * kStages;  // [2] S(t) retired  -> K stage reusable
  uint64_t* bar_vempty = bars + 3 * kStages;  // [2] PV(t) retired -> V stage reusable
  uint64_t* bar_q = bars + 4 * kStages;
  uint64_t* bar_s = bars + 4 * kStages + 1;   // S(t) ready - and, committed behind it, PV(t-1) retired
  uint64_t* bar_p = bars + 4 * kStages + 2;   // P(t) written (128 softmax arrivals)
  uint64_t* bar_done = bars + 4 * kStages + 3;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kV4NumBars);

  const int tid = threadIdx.x, warp = tid >> 5;
  const int N = p.N, H = p.H;
  const int bh = blockIdx.y, b = bh / H, h = bh - b * H;
  const int m0 = blockIdx.x * kM;
  const int ntiles = (N + kKT - 1) / kKT;
  const int BHN = p.B * H * N;

  if (warp == 4) {
    if (tid == 128) {
      for (int s = 0; s < kStages; ++s) {
        mbar_init(&bar_kfull[s], 1);
        mbar_init(&bar_vfull[s], 1);
        mbar_init(&bar_kempty[s], 1);
        mbar_init(&bar_vempty[s], 1);
      }
      mbar_init(bar_q, 1);
      mbar_init(bar_s, 1);
      mbar_init(bar_p, 4);  // one elected lane per softmax warp
      mbar_init(bar_done, 1);
      fence_mbar_init();
    }
    __syncwarp();
    if (elect_one()) {
      tma_prefetch_desc(&tmap);
      mbar_expect_tx(bar_q, kQBytes);
      tma_load_2d(sQ, &tmap, bar_q, 0, bh * N + m0);
      tma_load_2d(sQ + kTileBytes, &tmap, bar_q, 0, bh * N + m0 + kKT);
      for (int s = 0; s < kStages && s < ntiles; ++s) {
        mbar_expect_tx(&bar_kfull[s], kTileBytes);
        tma_load_2d(sK + s * kTileBytes, &tmap, &bar_kfull[s], 0, BHN + bh * N + s * kKT);
      }
      for (int s = 0; s < kStages && s < ntiles; ++s) {
        mbar_expect_tx(&bar_vfull[s], kTileBytes);
        tma_load_2d(sV + s * kTileBytes, &tmap, &bar_vfull[s], 0, 2 * BHN + bh * N + s * kKT);
      }
    }
    __syncwarp();
    tmem_alloc(tmem_slot, kV4TmemCols);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 4) {
    // =========================================== issuer ===========================================
    const uint64_t desc_q = smem_desc_sw128(smem_u32(sQ));
    constexpr uint32_t idesc_s = idesc_16<T>(kM, kKT, 0, 0);
    constexpr uint32_t idesc_o = idesc_16<T>(kM, kDh, 0, 1);
    mbar_wait(bar_q, 0);
    mbar_wait(&bar_kfull[0], 0);
    tc_fence_after();
    // the ragged last tile is a narrow MMA: N = round16(valid keys) instead of 64
    const int last_cols = (N - (ntiles - 1) * kKT + 15) & ~15;
    const uint32_t idesc_s_last = idesc_16<T>(kM, last_cols, 0, 0);
    if (elect_one()) {
      const uint64_t desc_k = smem_desc_sw128(smem_u32(sK));
      const uint32_t id0 = ntiles == 1 ? idesc_s_last : idesc_s;
#pragma unroll
      for (int k = 0; k < kDh / 16; ++k) mma_ss(tmem_base, desc_q + 2 * k, desc_k + 2 * k, id0, k > 0);
      mma_commit(bar_s);
      mma_commit(&bar_kempty[0]);
    }
    __syncwarp();
    for (int t = 0; t < ntiles; ++t) {
      const int stage = t & 1;
      const uint32_t use_parity = (uint32_t)((t >> 1) & 1);
      // S(t) has been issued: once it retires its K stage takes K(t + 2); PV(t-1)'s V stage takes V(t + 1)
      if (t + kStages < ntiles) {
        mbar_wait(&bar_kempty[stage], use_parity);
        if (elect_one()) {
          mbar_expect_tx(&bar_kfull[stage], kTileBytes);
          tma_load_2d(sK + stage * kTileBytes, &tmap, &bar_kfull[stage], 0, BHN + bh * N + (t + kStages) * kKT);
        }
        __syncwarp();
      }
      if (t >= 1 && t + 1 < ntiles) {
        const int sp = (t - 1) & 1;
        mbar_wait(&bar_vempty[sp], (uint32_t)(((t - 1) >> 1) & 1));
        if (elect_one()) {
          mbar_expect_tx(&bar_vfull[sp], kTileBytes);
          tma_load_2d(sV + sp * kTileBytes, &tmap, &bar_vfull[sp], 0, 2 * BHN + bh * N + (t + 1) * kKT);
        }
        __syncwarp();
      }
      // O += P(t) V(t), and S(t+1) right behind it into the columns P(t) occupies
      mbar_wait(&bar_vfull[stage], use_parity);
      if (t + 1 < ntiles) mbar_wait(&bar_kfull[(t + 1) & 1], (uint32_t)(((t + 1) >> 1) & 1));
      mbar_wait(bar_p, (uint32_t)(t & 1));
      tc_fence_after();
      if (elect_one()) {
        const uint64_t desc_v = smem_desc_sw128(smem_u32(sV + stage * kTileBytes));
        const int nvalid = min(kKT, N - t * kKT);
        const int ksteps = (nvalid + 15) >> 4;
        for (int kk = 0; kk < ksteps; ++kk)
          mma_ts(tmem_base + kV4ColO, tmem_base + kk * 8, desc_v + 128 * kk, idesc_o, (t | kk) != 0);
        mma_commit(&bar_vempty[stage]);
        if (t + 1 < ntiles) {
          const uint64_t desc_k = smem_desc_sw128(smem_u32(sK + ((t + 1) & 1) * kTileBytes));
          const uint32_t idn = (t + 2 == ntiles) ? idesc_s_last : idesc_s;
#pragma unroll
          for (int k = 0; k < kDh / 16; ++k) mma_ss(tmem_base, desc_q + 2 * k, desc_k + 2 * k, idn, k > 0);
          mma_commit(bar_s);
          mma_commit(&bar_kempty[(t + 1) & 1]);
        } else {
          mma_commit(bar_done);
        }
      }
      __syncwarp();
    }
  } else {
    // =========================================== softmax ==========================================
    const int i = m0 + tid;
    const bool warp_active = (m0 + warp * 32) < N;
    const uint32_t tmem_row = tmem_base + ((uint32_t)(warp * 32) << 16);
    float m_ref = -INFINITY, l_run = 0.f;
    for (int t = 0; t < ntiles; ++t) {
      const int nvalid = min(kKT, N - t * kKT);
      mbar_wait(bar_s, (uint32_t)(t & 1));
      tc_fence_after();
      if (warp_active) {
        if (nvalid == kKT) v4_tile<T, true>(tmem_row, nvalid, t, p.scale_log2, m_ref, l_run);
        else v4_tile<T, false>(tmem_row, nvalid, t, p.scale_log2, m_ref, l_run);
      }
      tc_fence_before();
      __syncwarp();
      if (elect_one()) mbar_arrive(bar_p);
    }

    // ---- epilogue: O / l -------------------------------------------------------------------------
    mbar_wait(bar_done, 0);
    tc_fence_after();
    if (warp_active) {
      const float inv = 1.f / l_run;
      T* dst = static_cast<T*>(p.out) + ((size_t)b * N + min(i, N - 1)) * (size_t)(H * kDh) + h * kDh;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t o[32];
        tmem_ld32(tmem_row + kV4ColO + half * 32, o);
        tmem_wait_ld();
        if (i < N) {
#pragma unroll
          for (int v8 = 0; v8 < 4; ++v8) {
            uint4 w;
            w.x = Elem16<T>::pack2(__uint_as_float(o[v8 * 8 + 0]) * inv, __uint_as_float(o[v8 * 8 + 1]) * inv);
            w.y = Elem16<T>::pack2(__uint_as_float(o[v8 * 8 + 2]) * inv, __uint_as_float(o[v8 * 8 + 3]) * inv);
            w.z = Elem16<T>::pack2(__uint_as_float(o[v8 * 8 + 4]) * inv, __uint_as_float(o[v8 * 8 + 5]) * inv);
            w.w = Elem16<T>::pack2(__uint_as_float(o[v8 * 8 + 6]) * inv, __uint_as_float(o[v8 * 8 + 7]) * inv);
            *reinterpret_cast<uint4*>(dst + half * 32 + v8 * 8) = w;
          }
        }
      }
      if (i < N) p.lse[(size_t)bh * N + i] = (m_ref + log2f(l_run)) * kLn2;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem_base, kV4TmemCols);
}

constexpr size_t kFwd4SmemBytes = 1024 + (size_t)kQBytes + (size_t)2 * kV4Stages * kV2KT * kDh * 2 + (size_t)kV4NumBars * 8 + 16;

size_t fwd2_smem_bytes(int N, const vrr_bias_desc* bias, int* lut_floats) {
  int lf = 0;
  if (bias && bias->mode == VRR_BIAS_TABLE) lf = 2 * N - 1 + 8;  // + slack for the aligned span
  else if (bias && bias->mode == VRR_BIAS_POLY) lf = 2 * bias->grid - 1;
  lf = (lf + 3) & ~3;
  if (lut_floats) *lut_floats = lf;
  size_t yx = (bias && bias->mode == VRR_BIAS_POLY) ? (size_t)((N * 2 + 15) & ~15) : 0;
  return 1024 + (size_t)kQBytes + (size_t)2 * kV2Stages * kV2KT * kDh * 2 + (size_t)lf * 4 + yx + (size_t)kV2NumBars * 8 + 16;
}

std::atomic<long long*> g_fwd_dbg{nullptr};

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode = nullptr;

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link against libcuda), looked up once
int encode_tiled(EncodeTiledFn* fn_out) {
  if (!g_encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    VRR_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    VRR_REQUIRE(fn && qres == cudaDriverEntryPointSuccess, VRR_ERR_CUDA, "cuTensorMapEncodeTiled not available");
    g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  }
  *fn_out = g_encode;
  return VRR_OK;
}

}  // namespace

int make_tmap_2d(CUtensorMap* map, const void* base, CUtensorMapDataType dtype, uint64_t rows, uint64_t cols,
                 uint64_t row_stride_bytes, uint32_t box_rows, uint32_t box_cols) {
  EncodeTiledFn encode;
  if (int rc = encode_tiled(&encode)) return rc;
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {row_stride_bytes};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode(map, dtype, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  VRR_REQUIRE(r == CUDA_SUCCESS, VRR_ERR_CUDA,
              "cuTensorMapEncodeTiled failed with CUresult %d (rows %llu cols %llu stride %llu box %ux%u)", (int)r,
              (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)row_stride_bytes, box_rows, box_cols);
  return VRR_OK;
}

int make_tmap_3d(CUtensorMap* map, const void* base, CUtensorMapDataType dtype, uint64_t d0, uint64_t d1, uint64_t d2,
                 uint64_t stride1_bytes, uint64_t stride2_bytes, uint32_t box0, uint32_t box1, int swizzle128) {
  EncodeTiledFn encode;
  if (int rc = encode_tiled(&encode)) return rc;
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {stride1_bytes, stride2_bytes};
  cuuint32_t box[3] = {box0, box1, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = encode(map, dtype, 3, const_cast<void*>(base), dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                      CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  VRR_REQUIRE(r == CUDA_SUCCESS, VRR_ERR_CUDA, "cuTensorMapEncodeTiled (3-D) failed with CUresult %d", (int)r);
  return VRR_OK;
}

bool attn_fwd_tc_supported(int B, int H, int N, int Dh, const vrr_bias_desc* bias) {
  if (Dh != kDh || N < 1) return false;
  if ((long long)3 * B * H * N >= (1ll << 31)) return false;
  if (bias && bias->mode == VRR_BIAS_POLY && bias->grid > 255) return false;
  return fwd2_smem_bytes(N, bias, nullptr) <= 110 * 1024;
}

void attn_fwd_tc_set_debug(long long* buf) { g_fwd_dbg.store(buf); }

template <typename T, int MODE>
static int fwd2_launch_tc(const CUtensorMap& tmap, const FwdParams& p, dim3 grid, size_t smem, cudaStream_t st) {
  VRR_SMEM_ATTR_ONCE((attn_fwd_tc2_kernel<T, MODE>), 110 * 1024);
  attn_fwd_tc2_kernel<T, MODE><<<grid, kV2Threads, smem, st>>>(tmap, p);
  VRR_LAUNCHED();
  return VRR_OK;
}

template <typename T>
static int attn_fwd_tc_t(const void* planes, const vrr_bias_desc* bias, void* out, float* lse, int B, int H, int N,
                         float scale, cudaStream_t st) {
  VRR_REQUIRE(((uintptr_t)planes & 15) == 0 && ((uintptr_t)out & 15) == 0, VRR_ERR_INVALID_ARG,
              "attn_fwd (tcgen05): planes/out must be 16-byte aligned");
  CUtensorMap tmap;
  if (int rc = make_tmap_2d(&tmap, planes, Elem16<T>::kTmap, (uint64_t)3 * B * H * N, kDh, kDh * 2, kV2KT, 64)) return rc;
  FwdParams p;
  p.out = out;
  p.lse = lse;
  p.B = B; p.H = H; p.N = N;
  p.scale_log2 = scale * kLog2e;
  p.dbg = g_fwd_dbg.load();
  const int mode = bias ? bias->mode : VRR_BIAS_NONE;
  p.bias_param = mode != VRR_BIAS_NONE ? bias->param : nullptr;
  p.bias_heads = mode != VRR_BIAS_NONE ? bias->heads : 0;
  p.bias_len = mode != VRR_BIAS_NONE ? bias->len : 0;
  p.bias_grid = mode != VRR_BIAS_NONE ? bias->grid : 0;
  if (mode == VRR_BIAS_TABLE)
    VRR_REQUIRE(((uintptr_t)bias->param & 15) == 0, VRR_ERR_INVALID_ARG, "attn_fwd (tcgen05): bias table must be 16-byte aligned");
  dim3 grid(ceil_div(N, kM), B * H);
  if (mode == VRR_BIAS_NONE) {
    // the bias modes stay on attn_fwd_tc2_kernel: evaluating the bias in both passes made the four-CTA kernel slower
    // there (577 tokens: table 118 vs 82 us, polynomial 175 vs 108 us)
    p.lut_floats = 0;
    VRR_SMEM_ATTR_ONCE(attn_fwd_tc4_kernel<T>, 64 * 1024);
    attn_fwd_tc4_kernel<T><<<grid, kV4Threads, kFwd4SmemBytes, st>>>(tmap, p);
    VRR_LAUNCHED();
    return VRR_OK;
  }
  const size_t smem2 = fwd2_smem_bytes(N, bias, &p.lut_floats);
  if (mode == VRR_BIAS_TABLE) return fwd2_launch_tc<T, VRR_BIAS_TABLE>(tmap, p, grid, smem2, st);
  return fwd2_launch_tc<T, VRR_BIAS_POLY>(tmap, p, grid, smem2, st);
}

int attn_fwd_tc(const void* planes, const vrr_bias_desc* bias, void* out, float* lse, int B, int H, int N, int Dh,
                float scale, int dtype, cudaStream_t st) {
  (void)Dh;
  if (dtype == VRR_F16) return attn_fwd_tc_t<__half>(planes, bias, out, lse, B, H, N, scale, st);
  return attn_fwd_tc_t<__nv_bfloat16>(planes, bias, out, lse, B, H, N, scale, st);
}

}  // namespace vrr
