// Fused attention backward for SHORT sequences (round16(N) <= 208: the 65..197-token ViT configurations), one
// persistent kernel: the whole-sequence variant.  Autograd of models/vit.py:71-88 of the reference (SURVEY row A18):
//   P = softmax(S), dV = P^T dO, dP = dO V^T, dS = P o (dP - delta), dQ = scale dS K, dK = scale dS^T Q.
//
// attn_bwd_tc2.cu is two kernels (dQ; dK/dV) that each read Q, K, V, dO from HBM (1.44x the algorithmic
// traffic, measured) and walk the sequence in 32-row tiles: ten small tcgen05.mma, four mbarrier round trips and a
// CTA prologue per tile.  Here
//   * one CTA per SM loops over work items (image, head); Q, K, V, dO of the NEXT item are prefetched by TMA into the
//     other half of shared memory (2 x 4 x N x 128 B) while the current one is processed: every operand is read from
//     HBM exactly once per launch;
//   * an item is a set of LANE TILES (128 TMEM lanes against all columns):
//       dQ tile  (lane = query row i):  S = Q K^T, dP = dO V^T  ->  dS            ->  dQ = dS K
//       dKV tile (lane = key j):        S^T = K Q^T, dP^T = V dO^T -> P^T, dS^T   ->  dV = P^T dO, dK = dS^T Q
//     processed in two or three COLUMN GROUPS (128 columns, then <= 96 / <= 64) of large tcgen05.mma (N up to 128)
//     with ONE softmax-side round trip each, instead of one per 32 columns;
//   * the two compute warpgroups are independent streams: each owns half of TMEM (256 columns), its own issuer warp
//     and its own lane tiles (group w: the dQ tiles of parity w and the dKV tiles of parity 1 - w), so one group's
//     exponentials overlap the other's MMAs and epilogue;
//   * per stream TMEM: S at [0,128), dP at [128,256) for the first column group; P / dS are written back in place
//     (bf16 / fp16) and consumed from TMEM by the accumulating MMAs; the accumulators live in columns the group has already
//     consumed (dQ or dV at [192,256), dK at [64,128)); later column groups reuse [0,96) / [96,192) (dQ) or
//     [0,64) / [128,192) (dKV) - the tensor pipe executes in issue order, so a group's S MMAs may be issued right
//     behind the accumulating MMAs that read the columns they overwrite;
//   * delta = rowsum(dO o O) and lse*log2(e) of the NEXT item are computed by a helper warp into shared memory
//     while the current item runs (rows past N get lse = +inf -> P = 0).
// Bias modes (relative table / polynomial) stay on attn_bwd_tc2.cu: a version of this kernel with the bias in the exponent
// of both orientations and the gradients taken in the dQ tiles (systolic diagonal sums into a shared histogram;
// per-thread power sums) was built and was correct, but its per-element extras made it slower than attn_bwd_tc2.cu
// (relative table 1 104 us against 856 us, polynomial 716 us against 627 us at ViT-B) - not kept.
//
// Measured alternatives (ViT-B/16-224, B = 256; this kernel: 303 us, attn_bwd_tc2.cu: 399 us):
//   * one stream of all eight warps walking double-buffered 96-column groups with a TMA-store epilogue: 315 us - the
//     S / dP waits disappear but twelve small groups per item cost as much in per-group overhead;
//   * staging the outputs through 1 KB of shared memory per warp for coalesced stores: no gain (the 8-row rounds
//     serialise); 32-byte TMA boxes need 4 KB per warp, which two resident items do not leave;
//   * a second register buffer to keep the next chunk's tcgen05.ld in flight: slower (2 620 -> 3 400 cycles per 128
//     columns).  The exponentials run at ~50-60 % of the MUFU roof (16 ex2 / clk / SM, scripts/ubench/mufu.cu) -
//     P is evaluated twice per element (once per orientation), which is the price of keeping dS out of shared memory;
//   * process16 on the packed fp32x2 pipe (fma / add / mul .f32x2): 349 us (132 registers instead of 113), and on top of
//     it a share of the exponentials by the FMA-pipe polynomial tc::ex2_poly2: +5 us per pair of eight (350 -> 371 us
//     at 6 of 8) - the column groups are bound by instruction issue and register traffic, not by MUFU throughput;
//   * two 16-column chunks per loop iteration (four tcgen05.ld in flight, 168 registers, no spills): 308 us - no gain.
#include "common.cuh"
#include "kernels.h"
#include "tc_common.cuh"

namespace vrr {

using namespace tc;

namespace {

constexpr int kDh = 64;
constexpr int kThreads = 384;   // warps 0-3 / 4-7 compute streams, 8 producer, 9 / 10 issuers, 11 statistics helper
constexpr uint32_t kTmemCols = 512;
constexpr float kLog2e = 1.4426950408889634f;
constexpr int kNumBars = 14;
constexpr int kSmemMax = 232448;

struct BwsParams {
  const void* out;  // element type T of the kernel
  const float* lse;
  void* d_planes;   // T
  int B, H, N;
  float scale, scale_log2;
  int total_items;
  long long* dbg;
};

__device__ __forceinline__ void dbg_stamp(const BwsParams& p, int region, int idx) {
  if (p.dbg != nullptr && blockIdx.x == 0 && idx < 256) p.dbg[region * 256 + idx] = clock64();
}

// Store this thread's row (64 fp32 channels in two 32-register halves) as 128 bytes of T.
template <typename T>
__device__ __forceinline__ void store_row(T* dst, const uint32_t (&lo)[32], const uint32_t (&hi)[32], float mul) {
#pragma unroll
  for (int v8 = 0; v8 < 4; ++v8) {
    uint4 w;
    w.x = Elem16<T>::pack2(__uint_as_float(lo[v8 * 8 + 0]) * mul, __uint_as_float(lo[v8 * 8 + 1]) * mul);
    w.y = Elem16<T>::pack2(__uint_as_float(lo[v8 * 8 + 2]) * mul, __uint_as_float(lo[v8 * 8 + 3]) * mul);
    w.z = Elem16<T>::pack2(__uint_as_float(lo[v8 * 8 + 4]) * mul, __uint_as_float(lo[v8 * 8 + 5]) * mul);
    w.w = Elem16<T>::pack2(__uint_as_float(lo[v8 * 8 + 6]) * mul, __uint_as_float(lo[v8 * 8 + 7]) * mul);
    *reinterpret_cast<uint4*>(dst + v8 * 8) = w;
  }
#pragma unroll
  for (int v8 = 0; v8 < 4; ++v8) {
    uint4 w;
    w.x = Elem16<T>::pack2(__uint_as_float(hi[v8 * 8 + 0]) * mul, __uint_as_float(hi[v8 * 8 + 1]) * mul);
    w.y = Elem16<T>::pack2(__uint_as_float(hi[v8 * 8 + 2]) * mul, __uint_as_float(hi[v8 * 8 + 3]) * mul);
    w.z = Elem16<T>::pack2(__uint_as_float(hi[v8 * 8 + 4]) * mul, __uint_as_float(hi[v8 * 8 + 5]) * mul);
    w.w = Elem16<T>::pack2(__uint_as_float(hi[v8 * 8 + 6]) * mul, __uint_as_float(hi[v8 * 8 + 7]) * mul);
    *reinterpret_cast<uint4*>(dst + 32 + v8 * 8) = w;
  }
}

// One column group of a lane tile for one thread (= one TMEM lane), 16 accumulator columns at a time with the NEXT
// 16 columns' tcgen05.ld in flight while the current ones are processed (two register buffers, A / B).
//   DQ  (lane = query row i, column = key j):  dS = exp2(S c - lse2_i) (dP - delta_i), keys past N masked;
//        dS (pairs of T) written over the S columns.
//   !DQ (lane = key j, column = query row i):  per-column (lse2_i, delta_i) from shared memory (lse2 = +inf past N
//        -> P = 0);  P^T (T) over the S^T columns, dS^T (T) over the dP^T columns.
template <typename T, bool DQ>
__device__ __forceinline__ void process16(const BwsParams& p, const uint32_t (&s)[16], const uint32_t (&d)[16], uint32_t t_dst_p,
                                          uint32_t t_dst_ds, int col0, float neg_lse2, float delta, const float4* stats2) {
  uint32_t pp[8], pd[8];
  if (DQ) {
    const bool full = col0 + 16 <= p.N;
#pragma unroll
    for (int e = 0; e < 16; e += 2) {
      float p0 = ex2(fmaf(__uint_as_float(s[e]), p.scale_log2, neg_lse2));
      float p1 = ex2(fmaf(__uint_as_float(s[e + 1]), p.scale_log2, neg_lse2));
      if (!full) {
        p0 = col0 + e < p.N ? p0 : 0.f;
        p1 = col0 + e + 1 < p.N ? p1 : 0.f;
      }
      pd[e >> 1] = Elem16<T>::pack2(p0 * (__uint_as_float(d[e]) - delta), p1 * (__uint_as_float(d[e + 1]) - delta));
    }
    tmem_st8(t_dst_p, pd);
  } else {
#pragma unroll
    for (int e = 0; e < 16; e += 2) {
      const float4 st = stats2[e >> 1];  // (lse2, delta) of rows col0+e and col0+e+1
      const float p0 = ex2(fmaf(__uint_as_float(s[e]), p.scale_log2, -st.x));
      const float p1 = ex2(fmaf(__uint_as_float(s[e + 1]), p.scale_log2, -st.z));
      pp[e >> 1] = Elem16<T>::pack2(p0, p1);
      pd[e >> 1] = Elem16<T>::pack2(p0 * (__uint_as_float(d[e]) - st.y), p1 * (__uint_as_float(d[e + 1]) - st.w));
    }
    tmem_st8(t_dst_p, pp);
    tmem_st8(t_dst_ds, pd);
  }
}

template <typename T, bool DQ>
__device__ __forceinline__ void process_group(const BwsParams& p, uint32_t t_s, uint32_t t_dp, int n16, int col0, float neg_lse2,
                                              float delta, const float4* stats2) {
  // (a version with the next chunk's tcgen05.ld in flight behind a second register buffer measured SLOWER: 3 400 vs
  // 2 620 cycles per 128 columns - the group is bound by the exponentials, not by the TMEM latency)
#pragma unroll 1
  for (int c = 0; c < n16; ++c) {
    uint32_t s[16], d[16];
    tmem_ld16(t_s + c * 16, s);
    tmem_ld16(t_dp + c * 16, d);
    tmem_wait_ld();
    process16<T, DQ>(p, s, d, t_s + c * 8, t_dp + c * 8, col0 + c * 16, neg_lse2, delta, stats2 + c * 8);
  }
}

// Column groups of a lane tile: (start column, width, TMEM offset of dP): 128 columns, then <= 96 (dQ) / <= 64 (dKV).
// Same functions on the issuer and the compute side.
struct ColGroup {
  int c0, cw, dp_off;
};
__device__ __forceinline__ int num_groups(bool is_dq, int npad) {
  if (npad <= 128) return 1;
  const int step = is_dq ? 96 : 64;
  return 1 + (npad - 128 + step - 1) / step;
}
__device__ __forceinline__ ColGroup group_at(bool is_dq, int npad, int gi) {
  ColGroup g;
  if (gi == 0) {
    g.c0 = 0;
    g.cw = npad < 128 ? npad : 128;
    g.dp_off = 128;
  } else {
    const int step = is_dq ? 96 : 64;
    g.c0 = 128 + (gi - 1) * step;
    g.cw = npad - g.c0 < step ? npad - g.c0 : step;
    g.dp_off = is_dq ? 96 : 128;
  }
  return g;
}

template <typename T>
__global__ void __launch_bounds__(kThreads, 1)
attn_bwd_ws_kernel(const __grid_constant__ CUtensorMap tm_pl64, const __grid_constant__ CUtensorMap tm_pl16,
                   const __grid_constant__ CUtensorMap tm_do64, const __grid_constant__ CUtensorMap tm_do16,
                   const __grid_constant__ BwsParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int N = p.N, H = p.H, E = H * kDh;
  const int npad = (N + 15) & ~15;
  const int tbytes = npad * 128;                   // one tensor of one item (multiple of 2048)
  const int slot_bytes = 4 * tbytes;               // Q | K | V | dO
  float2* stats = reinterpret_cast<float2*>(smem + 2 * slot_bytes);   // [2 items][256] (lse * log2e, delta)
  uint64_t* bars = reinterpret_cast<uint64_t*>(stats + 512);
  uint64_t* bar_full = bars;              // [2] item data landed
  uint64_t* bar_empty = bars + 2;         // [2] last MMA of the item retired in both streams -> slot reusable
  uint64_t* bar_sfull = bars + 4;         // [2 streams] S and dP of the column group ready
  uint64_t* bar_pfull = bars + 6;         // [2 streams] P / dS of the column group stored (128 arrivals)
  uint64_t* bar_accfull = bars + 8;       // [2 streams] accumulators of the lane tile ready
  uint64_t* bar_accempty = bars + 10;     // [2 streams] epilogue has read them (128 arrivals)
  uint64_t* bar_stfull = bars + 12;       // [2] statistics of the item written (32 arrivals)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + kNumBars);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int total = p.total_items;
  const int BHN = p.B * H * N;
  const int ntile = (N + 127) >> 7;                // 128-lane tiles of rows / of keys

  if (tid == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(&bar_full[s], 1);
      mbar_init(&bar_empty[s], 2);
      mbar_init(&bar_sfull[s], 1);
      mbar_init(&bar_pfull[s], 128);
      mbar_init(&bar_accfull[s], 1);
      mbar_init(&bar_accempty[s], 128);
      mbar_init(&bar_stfull[s], 32);
    }
    fence_mbar_init();
  }
  __syncwarp();
  if (warp == 8) tmem_alloc(tmem_slot, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // NB: with 230 KB of shared memory the L1 that would absorb register spills is nearly gone - a 184-byte stack frame
  // cost ~5 000 cycles per lane tile (measured).  Keep `ptxas -v` at 0 spill bytes for this kernel.
  if (warp == 8) {
    // ============================================ TMA producer ============================================
    if (elect_one()) {
      tma_prefetch_desc(&tm_pl64);
      tma_prefetch_desc(&tm_pl16);
      tma_prefetch_desc(&tm_do64);
      tma_prefetch_desc(&tm_do16);
    }
    __syncwarp();
    const int nb64 = npad >> 6, nb16 = (npad & 63) >> 4;
    int k = 0;
    for (int bh = blockIdx.x; bh < total; bh += gridDim.x, ++k) {
      const int sl = k & 1;
      const int b = bh / H, h = bh - b * H;
      mbar_wait(&bar_empty[sl], (uint32_t)(((k >> 1) & 1) ^ 1));
      if (elect_one()) {
        uint8_t* base = smem + sl * slot_bytes;
        mbar_expect_tx(&bar_full[sl], (uint32_t)slot_bytes);
#pragma unroll 1
        for (int t = 0; t < 3; ++t) {  // Q, K, V planes
          uint8_t* dst = base + t * tbytes;
          const int row0 = t * BHN + bh * N;
          for (int j = 0; j < nb64; ++j) tma_load_2d(dst + j * 8192, &tm_pl64, &bar_full[sl], 0, row0 + j * 64);
          for (int j = 0; j < nb16; ++j)
            tma_load_2d(dst + nb64 * 8192 + j * 2048, &tm_pl16, &bar_full[sl], 0, row0 + nb64 * 64 + j * 16);
        }
        uint8_t* dst = base + 3 * tbytes;  // dO rows of image b, columns of head h
        for (int j = 0; j < nb64; ++j) tma_load_2d(dst + j * 8192, &tm_do64, &bar_full[sl], h * kDh, b * N + j * 64);
        for (int j = 0; j < nb16; ++j)
          tma_load_2d(dst + nb64 * 8192 + j * 2048, &tm_do16, &bar_full[sl], h * kDh, b * N + nb64 * 64 + j * 16);
      }
      __syncwarp();
    }
  } else if (warp == 9 || warp == 10) {
    // ============================================ MMA issuer of stream w ==================================
    const int w = warp - 9;
    const uint32_t tw = tmem_base + (uint32_t)(w * 256);
    const uint32_t smem_b = smem_u32(smem);
    constexpr uint32_t idesc_acc = idesc_16<T>(128, kDh, 0, 1);
    uint32_t ng = 0, nt = 0;  // column groups / lane tiles issued so far by this stream (barrier phases)
    int k = 0;
    for (int bh = blockIdx.x; bh < total; bh += gridDim.x, ++k) {
      const int sl = k & 1;
      const uint32_t q_b = smem_b + sl * slot_bytes, k_b = q_b + tbytes, v_b = k_b + tbytes, g_b = v_b + tbytes;
      mbar_wait(&bar_full[sl], (uint32_t)((k >> 1) & 1));
      for (int lt = 0; lt < 2 * ntile; ++lt) {
        const bool is_dq = lt < ntile;
        const int tile = is_dq ? lt : lt - ntile;
        if (((tile & 1) == w) != is_dq) continue;  // stream w: dQ tiles of parity w, dKV tiles of parity 1 - w
        // lanes: dQ tile -> Q / dO rows of the tile against K / V;  dKV tile -> K / V rows against Q / dO
        const uint32_t a_s = (is_dq ? q_b : k_b) + tile * 16384, a_p = (is_dq ? g_b : v_b) + tile * 16384;
        const uint32_t b_s = is_dq ? k_b : q_b, b_p = is_dq ? v_b : g_b;
        mbar_wait(&bar_accempty[w], (nt & 1) ^ 1);  // the previous lane tile's epilogue has read its accumulators
        tc_fence_after();
        const int ngr = num_groups(is_dq, npad);
        for (int gi = 0; gi < ngr; ++gi) {
          const ColGroup g = group_at(is_dq, npad, gi);
          const bool first = gi == 0;
          const bool last = gi == ngr - 1;
          if (elect_one()) {
            const uint32_t idesc = idesc_16<T>(128, g.cw, 0, 0);
            const uint64_t das = smem_desc_sw128(a_s), dap = smem_desc_sw128(a_p);
            const uint64_t dbs = smem_desc_sw128(b_s + g.c0 * 128), dbp = smem_desc_sw128(b_p + g.c0 * 128);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) mma_ss(tw, das + 2 * kk, dbs + 2 * kk, idesc, kk > 0);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) mma_ss(tw + g.dp_off, dap + 2 * kk, dbp + 2 * kk, idesc, kk > 0);
            mma_commit(&bar_sfull[w]);
          }
          __syncwarp();
          mbar_wait(&bar_pfull[w], ng & 1);
          tc_fence_after();
          if (elect_one()) {
            const int ksteps = g.cw >> 4;
            const uint32_t adv = (uint32_t)(128 * (g.c0 >> 4));
            if (is_dq) {
              const uint64_t dk = smem_desc_sw128(k_b) + adv;
              for (int kk = 0; kk < ksteps; ++kk)  // dQ += dS K
                mma_ts(tw + 192, tw + kk * 8, dk + 128 * kk, idesc_acc, (!first || kk > 0) ? 1u : 0u);
            } else {
              const uint64_t dg = smem_desc_sw128(g_b) + adv, dq = smem_desc_sw128(q_b) + adv;
              for (int kk = 0; kk < ksteps; ++kk)  // dV += P^T dO
                mma_ts(tw + 192, tw + kk * 8, dg + 128 * kk, idesc_acc, (!first || kk > 0) ? 1u : 0u);
              for (int kk = 0; kk < ksteps; ++kk)  // dK += dS^T Q
                mma_ts(tw + 64, tw + g.dp_off + kk * 8, dq + 128 * kk, idesc_acc, (!first || kk > 0) ? 1u : 0u);
            }
            if (last) mma_commit(&bar_accfull[w]);
          }
          __syncwarp();
          ++ng;
        }
        ++nt;
      }
      // every MMA of this stream that reads the slot has been issued: its retirement releases the slot
      if (elect_one()) mma_commit(&bar_empty[sl]);
      __syncwarp();
    }
  } else if (warp == 11) {
    // ============================================ statistics helper =======================================
    // stats[k & 1][i] = (lse_i * log2 e, delta_i = sum_d dO[i][d] O[i][d]) for the rows of item k, one item ahead
    int k = 0;
    for (int bh = blockIdx.x; bh < total; bh += gridDim.x, ++k) {
      const int sl = k & 1;
      const int b = bh / H, h = bh - b * H;
      float2* st = stats + sl * 256;
      const uint8_t* sG = smem + sl * slot_bytes + 3 * tbytes;
      mbar_wait(&bar_full[sl], (uint32_t)((k >> 1) & 1));
#pragma unroll 1
      for (int r0 = 0; r0 < 256; r0 += 32) {
        const int i = r0 + lane;
        float2 v = make_float2(INFINITY, 0.f);
        if (i < N) {
          const uint4* o4 = reinterpret_cast<const uint4*>(static_cast<const T*>(p.out) + ((size_t)b * N + i) * E + h * kDh);
          const uint8_t* grow = sG + i * 128;
          float acc = 0.f;
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            const uint4 ov = __ldg(o4 + c);
            const uint4 gv = *reinterpret_cast<const uint4*>(grow + ((c ^ (i & 7)) << 4));
            const uint32_t ow[4] = {ov.x, ov.y, ov.z, ov.w}, gw[4] = {gv.x, gv.y, gv.z, gv.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 of = Elem16<T>::unpack2(ow[e]);
              const float2 gf = Elem16<T>::unpack2(gw[e]);
              acc = fmaf(of.x, gf.x, acc);
              acc = fmaf(of.y, gf.y, acc);
            }
          }
          v = make_float2(p.lse[(size_t)bh * N + i] * kLog2e, acc);
        }
        st[i] = v;
      }
      mbar_arrive(&bar_stfull[sl]);
    }
  } else if (warp < 8) {
    // ============================================ compute streams =========================================
    const int w = warp >> 2, wq = warp & 3;
    const int lrow = wq * 32 + lane;  // TMEM lane of this thread
    const uint32_t trow = tmem_base + (uint32_t)(w * 256) + ((uint32_t)(wq * 32) << 16);
    const size_t plane = (size_t)BHN * kDh;
    const bool dbg_on = p.dbg != nullptr && (tid & 127) == 0;
    uint32_t ng = 0, nt = 0;
    int k = 0;
    for (int bh = blockIdx.x; bh < total; bh += gridDim.x, ++k) {
      const int sl = k & 1;
      const float2* st = stats + sl * 256;
      mbar_wait(&bar_stfull[sl], (uint32_t)((k >> 1) & 1));
      for (int lt = 0; lt < 2 * ntile; ++lt) {
        const bool is_dq = lt < ntile;
        const int tile = is_dq ? lt : lt - ntile;
        if (((tile & 1) == w) != is_dq) continue;
        const int idx = tile * 128 + lrow;             // query row (dQ tile) / key (dKV tile) of this thread
        const bool warp_live = tile * 128 + wq * 32 < N;
        const float2 mine = st[min(idx, 255)];
        const float neg_lse2 = -mine.x, delta = mine.y;
        const int ngr = num_groups(is_dq, npad);
#pragma unroll 1
        for (int gi = 0; gi < ngr; ++gi) {
          const ColGroup g = group_at(is_dq, npad, gi);
          if (dbg_on) dbg_stamp(p, w, (int)ng * 4 + 0);
          mbar_wait(&bar_sfull[w], ng & 1);
          tc_fence_after();
          if (dbg_on) dbg_stamp(p, w, (int)ng * 4 + 1);
          if (warp_live) {
            const float4* st2 = reinterpret_cast<const float4*>(st + g.c0);
            if (is_dq) process_group<T, true>(p, trow, trow + g.dp_off, g.cw >> 4, g.c0, neg_lse2, delta, st2);
            else process_group<T, false>(p, trow, trow + g.dp_off, g.cw >> 4, g.c0, neg_lse2, delta, st2);
            tmem_wait_st();
          }
          tc_fence_before();
          mbar_arrive(&bar_pfull[w]);
          if (dbg_on) dbg_stamp(p, w, (int)ng * 4 + 2);
          ++ng;
        }
        // ---- epilogue of the lane tile -------------------------------------------------------------------
        mbar_wait(&bar_accfull[w], nt & 1);
        tc_fence_after();
        if (dbg_on) dbg_stamp(p, w, (int)(ng - 1) * 4 + 3);
        if (warp_live) {
          // (ld, arrive, store) in ONE scope: with the loads and the uses in differently-predicated blocks ptxas kept
          // the 64 accumulator registers in local memory
          {
            uint32_t a0[32], a1[32];
            if (dbg_on && w == 0) dbg_stamp(p, 3, (int)nt * 4 + 0);
            tmem_ld32(trow + 192, a0);  // dQ or dV
            tmem_ld32(trow + 224, a1);
            tmem_wait_ld();
            if (dbg_on && w == 0) dbg_stamp(p, 3, (int)nt * 4 + 1);
            if (is_dq) {
              tc_fence_before();
              mbar_arrive(&bar_accempty[w]);
            }
            if (idx < N) store_row(static_cast<T*>(p.d_planes) + (is_dq ? 0 : 2) * plane + ((size_t)bh * N + idx) * kDh, a0, a1, is_dq ? p.scale : 1.f);
            if (dbg_on && w == 0) dbg_stamp(p, 3, (int)nt * 4 + 2);
          }
          if (!is_dq) {
            uint32_t b0[32], b1[32];
            tmem_ld32(trow + 64, b0);  // dK
            tmem_ld32(trow + 96, b1);
            tmem_wait_ld();
            tc_fence_before();
            mbar_arrive(&bar_accempty[w]);
            if (idx < N) store_row(static_cast<T*>(p.d_planes) + plane + ((size_t)bh * N + idx) * kDh, b0, b1, p.scale);
            if (dbg_on && w == 0) dbg_stamp(p, 3, (int)nt * 4 + 3);
          }
        } else {
          tc_fence_before();
          mbar_arrive(&bar_accempty[w]);
        }
        ++nt;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) tmem_dealloc(tmem_base, kTmemCols);
}

// The 128-row A operand of a pass starts at row tile * 128 of a tensor that holds round16(N) rows: the tensor core
// reads up to 127 rows (16 KB) past it - harmless garbage for lanes that are never stored, but the bytes must exist:
// a 16 KB tail (holding the statistics and the barriers) follows the last slot.
size_t bws_smem_bytes(int N) {
  const int npad = (N + 15) & ~15;
  static_assert(512 * 8 + kNumBars * 8 + 16 <= 16384, "tail too small");
  return 1024 + (size_t)2 * 4 * npad * 128 + 16384;
}

std::atomic<long long*> g_bws_dbg{nullptr};

}  // namespace

void attn_bwd_ws_set_debug(long long* buf) { g_bws_dbg.store(buf); }

bool attn_bwd_ws_supported(int B, int H, int N, int Dh, const vrr_bias_desc* bias) {
  if (Dh != kDh || N < 1 || N > 256) return false;
  if (bias && bias->mode != VRR_BIAS_NONE) return false;
  if ((long long)3 * B * H * N >= (1ll << 31)) return false;
  return bws_smem_bytes(N) <= (size_t)kSmemMax;
}

template <typename T>
static int attn_bwd_ws_t(const void* planes, const void* out, const void* d_out, const float* lse, void* d_planes, int B,
                         int H, int N, float scale, cudaStream_t st) {
  VRR_REQUIRE(((uintptr_t)planes & 15) == 0 && ((uintptr_t)out & 15) == 0 && ((uintptr_t)d_out & 15) == 0 &&
                  ((uintptr_t)d_planes & 15) == 0,
              VRR_ERR_INVALID_ARG, "attn_bwd (tcgen05): planes / out / d_out / d_planes must be 16-byte aligned");
  const int E = H * kDh;
  CUtensorMap tm_pl64, tm_pl16, tm_do64, tm_do16;
  if (int rc = make_tmap_2d(&tm_pl64, planes, Elem16<T>::kTmap, (uint64_t)3 * B * H * N, kDh, kDh * 2, 64, 64)) return rc;
  if (int rc = make_tmap_2d(&tm_pl16, planes, Elem16<T>::kTmap, (uint64_t)3 * B * H * N, kDh, kDh * 2, 16, 64)) return rc;
  if (int rc = make_tmap_2d(&tm_do64, d_out, Elem16<T>::kTmap, (uint64_t)B * N, (uint64_t)E, (uint64_t)E * 2, 64, 64)) return rc;
  if (int rc = make_tmap_2d(&tm_do16, d_out, Elem16<T>::kTmap, (uint64_t)B * N, (uint64_t)E, (uint64_t)E * 2, 16, 64)) return rc;
  BwsParams p;
  p.out = out;
  p.lse = lse;
  p.d_planes = d_planes;
  p.B = B; p.H = H; p.N = N;
  p.scale = scale;
  p.scale_log2 = scale * kLog2e;
  p.total_items = B * H;
  p.dbg = g_bws_dbg.load();
  const size_t smem = bws_smem_bytes(N);
  const int grid = p.total_items < sm_count() ? p.total_items : sm_count();
  VRR_SMEM_ATTR_ONCE(attn_bwd_ws_kernel<T>, kSmemMax);
  attn_bwd_ws_kernel<T><<<grid, kThreads, smem, st>>>(tm_pl64, tm_pl16, tm_do64, tm_do16, p);
  VRR_LAUNCHED();
  return VRR_OK;
}

int attn_bwd_ws(const void* planes, const void* out, const void* d_out, const float* lse, void* d_planes, int B, int H,
                int N, int Dh, float scale, int dtype, cudaStream_t st) {
  (void)Dh;
  if (dtype == VRR_F16) return attn_bwd_ws_t<__half>(planes, out, d_out, lse, d_planes, B, H, N, scale, st);
  return attn_bwd_ws_t<__nv_bfloat16>(planes, out, d_out, lse, d_planes, B, H, N, scale, st);
}

}  // namespace vrr
