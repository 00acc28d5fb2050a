/*
 * vrr.h - C ABI of libvrr_b200.so: the B200 (sm_100a) ViT attention hot path of
 * zhengyk19/vit-rpe-rope.
 *
 * The reference is pure Python/PyTorch and has NO FFI / plugin boundary of its own
 * (SURVEY.md section 8, row B1): its boundary is the Python module API of models/.  This header
 * is therefore the boundary a maintainer would bind from that API (INTEGRATION.md shows the
 * ctypes stub).  Each entry point names the reference code (file:line under /root/reference) it
 * replaces.
 *
 * Conventions (all entry points)
 *   - plain pointers and sizes only: no torch / pybind / C++ types cross this boundary;
 *   - every data pointer is a DEVICE pointer on the current CUDA device (sm_100); the library
 *     never allocates, never synchronises, never throws; all work is enqueued on `stream`
 *     (a cudaStream_t passed as void*; NULL = legacy default stream);
 *   - return value: VRR_OK (0) or a negative vrr_status; vrr_last_error() gives the reason;
 *   - tensors are dense row-major with the shapes documented per argument; `dtype` selects the
 *     element type of activations/weights (VRR_F32, VRR_BF16 or VRR_F16).  Where an entry point takes several
 *     dtypes, bf16 and fp16 never meet in one call (VRR_ERR_INVALID_ARG); each pairs with fp32 in exactly the
 *     combinations documented for bf16, and fp16 runs the same kernels as bf16.  Position tables (cos/sin, bias
 *     table, polynomial coefficients), softmax statistics and all parameter-gradient outputs that
 *     are reductions (d_table, d_coef, d_cos, d_sin) are ALWAYS fp32;
 *   - there is no CPU path: on a machine without an sm_100 device every compute entry point
 *     returns VRR_ERR_NO_DEVICE.
 *
 * Token / head geometry: B images, N tokens per image, E = H * Dh channels, H heads of Dh channels.  Dh must be
 * one of 16, 32, 64 (the tcgen05 bf16 / fp16 kernels need Dh == 64).  An image's token stream is
 *   [cls, reg_0 .. reg_{R-1}, patch_0 .. patch_{Np-1}]      (timm / DINOv2 order, n_prefix = 1 + R, N = n_prefix + Np)
 * with the Np patches in raster order.  The n_prefix prefix tokens (the cls token and R register tokens) get no
 * absolute position embedding and are never rotated; patch p sits at token row n_prefix + p.  The *_prefix entry
 * points take n_prefix (1 <= n_prefix <= N, else VRR_ERR_INVALID_ARG); the others are those entry points at
 * n_prefix = 1 (no registers: token 0 is the cls token, tokens 1..N-1 the patches).
 *
 * "qkv planes": one buffer [3][B][H][N][Dh] holding q (rotated when RoPE is on), k (likewise), v.
 */
#ifndef VRR_H_
#define VRR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VRR_ABI_VERSION 1

typedef enum {
  VRR_OK = 0,
  VRR_ERR_INVALID_ARG = -1,   /* null pointer, bad enum, inconsistent sizes            */
  VRR_ERR_UNSUPPORTED = -2,   /* shape/dtype outside what the kernels implement         */
  VRR_ERR_NO_DEVICE = -3,     /* no CUDA device, or the current device is not sm_100    */
  VRR_ERR_CUDA = -4,          /* a CUDA runtime/driver call failed (see vrr_last_error) */
  VRR_ERR_WORKSPACE = -5      /* workspace too small (see vrr_*_workspace_bytes)        */
} vrr_status;

/* fp16 (IEEE binary16) results that overflow are +-inf, never a clamped finite value (mixed-precision training
 * with a loss scaler detects the overflow from them). */
typedef enum { VRR_F32 = 0, VRR_BF16 = 1, VRR_F16 = 2 } vrr_dtype;

/* RoPE variants of models/vit.py:51-68.  AXIAL: cos/sin are [N-n_prefix][Dh/2] shared by all heads
 * (positional_encoding.py:216-245).  MIXED: cos/sin are [H][N-n_prefix][Dh/2]
 * (positional_encoding.py:313-351).  Prefix tokens (cls, registers) are never rotated (vit.py:56-57); token row
 * t >= n_prefix is rotated by table row t - n_prefix. */
typedef enum { VRR_ROPE_NONE = 0, VRR_ROPE_AXIAL = 1, VRR_ROPE_MIXED = 2 } vrr_rope_mode;

/* Additive logit bias of models/vit.py:73-81.
 * TABLE: relative-position table [H][2N-1]; bias[h][i][j] = table[h][i - j + N - 1]
 *        (positional_encoding.py:58-75,93).
 * POLY : polynomial in the L1 patch distance, coef [Hc][degree+1] with Hc = 1 (shared) or H;
 *        bias[h][i][j] = sum_k coef[k] * d^k for i,j >= 1, 0 on the cls row/column, with
 *        d = |(i-1)%g - (j-1)%g| + |(i-1)/g - (j-1)/g| (positional_encoding.py:127-171). */
typedef enum { VRR_BIAS_NONE = 0, VRR_BIAS_TABLE = 1, VRR_BIAS_POLY = 2 } vrr_bias_mode;

/* Kernel family selection for the bf16 / fp16 attention, QKV, GEMM and patch-embedding kernels.
 * AUTO picks the tcgen05 (tensor core, TMEM) kernels whenever the shape allows and the SIMT kernels
 * otherwise (fp16 exactly where bf16 would); the other two
 * force one family (tests use them to cross-check).  fp32 always runs the SIMT FFMA kernels:
 * tcgen05 has no fp32 MMA and the fp32 parity bar is 1e-5. */
typedef enum { VRR_IMPL_AUTO = 0, VRR_IMPL_SIMT = 1, VRR_IMPL_TCGEN05 = 2 } vrr_impl;

/* Epilogues of vrr_gemm_ex (Linear layers, models/vit.py:91,118,285). */
typedef enum {
  VRR_EPI_NONE = 0,
  VRR_EPI_BIAS = 1,            /* c = acc + bias                                                              */
  VRR_EPI_BIAS_GELU = 2,       /* c = h = acc + bias, c2 = gelu(h)            (exact erf GELU, timm Mlp)        */
  VRR_EPI_BIAS_GELU_GRAD = 3,  /* c = gelu(h), c2 = d gelu / dh (h)           (what the Mlp backward needs)     */
  VRR_EPI_MUL = 4,             /* c = acc * c2[m][n]; c2 is an INPUT [M][N]   (d_act * gelu'(h) in fc2's dX)    */
  VRR_EPI_BIAS_GELU_ACT = 5    /* c = gelu(acc + bias), c2 unused             (the Mlp under torch.no_grad)     */
} vrr_epilogue;

typedef struct {
  int32_t mode;        /* vrr_bias_mode                                                  */
  int32_t heads;       /* rows of `param`: H for TABLE; 1 or H for POLY                  */
  int32_t len;         /* columns of `param`: 2N-1 for TABLE; degree+1 for POLY          */
  int32_t grid;        /* POLY: patch grid side g (N-1 == g*g); ignored otherwise        */
  const float* param;  /* fp32 [heads][len]; NULL when mode == NONE                      */
} vrr_bias_desc;

/* Element dropout and stochastic depth (timm DropPath) applied inside the kernels that already read the data.
 * Random numbers are Philox4x32-10 with key = *seed (low word = key[0]) and counter {g lo32, g hi32, site, stream}:
 *   element (m, n) of an [M][E] site (E % 8 == 0): stream 0, g = (m E + n) / 8, 16-bit half (n & 1) (low half first)
 *     of output word (n % 8) >> 1; kept iff that value < round((1 - p) 65536);
 *   image b (rows b N .. b N + N - 1, N = rows_per_sample): stream 1, counter {b, 0, site, 1}; kept iff the low 16
 *     bits of word 0 < round((1 - p_path) 65536).
 * An element's factor is f = keep * keep_path(b) * s with s = (1 / (1 - p)) * (1 / (1 - p_path)) formed in fp32.
 * A probability of 0 draws nothing for it.  The seed is read on the device, so a captured CUDA graph that refills
 * it before the kernels gets fresh masks on every replay.  oracle/philox_np.py restates the masks. */
typedef struct {
  float p;                  /* element dropout probability, [0, 1)                            */
  float p_path;             /* stochastic-depth probability per image, [0, 1); 0 where unused  */
  int32_t rows_per_sample;  /* token rows per image (N): image of row m = m / rows_per_sample   */
  int32_t site;             /* Philox counter word 2                                          */
  const uint64_t* seed;     /* DEVICE pointer to the 64-bit Philox key                        */
} vrr_drop_desc;

/* ---- library ------------------------------------------------------------------------------- */
int vrr_abi_version(void);
const char* vrr_last_error(void);          /* thread-local, valid until the next call           */
int vrr_device_ok(void);                   /* 1 if the current device is sm_100, else 0         */
int vrr_set_impl(int impl);                /* vrr_impl; process-wide; returns previous value    */
/* Number of kernel launches issued by this library since load (for bench.py's gpu_launches). */
uint64_t vrr_launch_count(void);
/* Dispatch counters per kernel family (VRR_IMPL_SIMT or VRR_IMPL_TCGEN05): how many of the entry
 * points that choose between the two families (patch_embed_fwd, qkv_rope_fwd, attn_fwd, attn_bwd, gemm)
 * took that family since load.  Lets a caller (and the parity tests) assert which family ran under
 * VRR_IMPL_AUTO instead of trusting the selection silently. */
uint64_t vrr_family_count(int family);
/* Tuning switches (process-wide), kept for A/B measurements: "ln_reg" (0 = generic multi-pass LayerNorm kernels only;
 * the tests use them as the bit-exact reference for the register-resident ones), "ln_bwd_minb" (1 / 2 / 3: launch
 * shape of the register-resident add+LayerNorm backward), "simt_gemm_tile" (128 / 64: tile of the fp32 FFMA GEMM).
 * Any other name returns VRR_ERR_INVALID_ARG. */
int vrr_set_option(const char* name, int value);
/* Debug: CTA 0 of the next attention launches records clock64() phase stamps of its producer, issuer and
 * softmax roles into `device_buf` (1024 x int64, zero it first); NULL switches it off. */
int vrr_debug_timestamps(void* device_buf);

/* ---- (c) patch embedding: models/vit.py:164,248-258 ---------------------------------------- */
/* tokens[b][0][:]   = cls_token
 * tokens[b][1+p][:] = round_dtype(conv_weight[E][C*P*P] . unfold(images)[b][p][:] + conv_bias) (+ pos_embed[p])
 * images [B][C][Hi][Wi]                                            : element type `img_dtype`
 * weight [E][C][P][P], bias [E]                                    : element type `dtype` (the conv arithmetic)
 * cls_token [E], pos_embed, tokens [B][Np+1][E]                    : element type `tok_dtype`
 * pos_embed: NULL, or the absolute table [>= Np][E] (positional_encoding.py:37-40: added to patch
 * rows only).  (img fp32, dtype bf16, tok fp32) is the reference's autocast semantics: the image is
 * rounded to bf16 on load, the conv result is bf16, and the concatenation with the fp32 cls token
 * promotes the stream to fp32; fp16 in place of every bf16 gives the float16-autocast semantics.  The 16-bit
 * tensor-core path (P % 8 == 0, C*P*P % 64 == 0, E % 64 == 0)
 * unfolds the patches into `workspace` (vrr_patch_embed_workspace_bytes, 256-byte aligned) and runs
 * a tcgen05 GEMM; otherwise workspace may be NULL. */
size_t vrr_patch_embed_workspace_bytes(int B, int C, int Hi, int Wi, int P, int E, int dtype);
int vrr_patch_embed_fwd(const void* images, const void* weight, const void* bias,
                        const void* cls_token, const void* pos_embed, void* tokens, void* workspace,
                        size_t workspace_bytes, int B, int C, int Hi, int Wi, int P, int E,
                        int img_dtype, int dtype, int tok_dtype, void* stream);
/* The same with n_prefix prefix tokens (cls, then registers):
 *   tokens[b][t][:]          = prefix_tokens[t][:]                 for t < n_prefix
 *   tokens[b][n_prefix+p][:] = the patch row p above (+ pos_embed[p])
 * prefix_tokens [n_prefix][E] and tokens [B][n_prefix+Np][E] are of `tok_dtype`.  n_prefix = 1 is
 * vrr_patch_embed_fwd. */
int vrr_patch_embed_fwd_prefix(const void* images, const void* weight, const void* bias, const void* prefix_tokens,
                               int n_prefix, const void* pos_embed, void* tokens, void* workspace,
                               size_t workspace_bytes, int B, int C, int Hi, int Wi, int P, int E, int img_dtype,
                               int dtype, int tok_dtype, void* stream);
/* out[b*Np + p][c*P*P + i*P + j] = bf16(images[b][c][py*P+i][px*P+j]): the im2col matrix of the
 * stride-P convolution (needs P % 8 == 0).  Used by the forward above and by callers that take the
 * weight gradient with a plain library GEMM. */
int vrr_patch_unfold(const void* images, void* out, int B, int C, int Hi, int Wi, int P,
                     int img_dtype, void* stream);
/* The same with an explicit output element type `out_dtype` (VRR_BF16 or VRR_F16); images are fp32 or
 * `out_dtype`. */
int vrr_patch_unfold_ex(const void* images, void* out, int B, int C, int Hi, int Wi, int P,
                        int img_dtype, int out_dtype, void* stream);
/* d_tokens [B][Np+1][E] (`tok_dtype`).  Parameter gradients are reductions and ALWAYS fp32:
 * d_weight [E][C*P*P] (or NULL: skip it), d_bias [E], d_cls [E], d_pos [Np][E] or NULL; written (not
 * accumulated).  Images need no gradient (train.py:109-115). */
int vrr_patch_embed_bwd(const void* images, const void* d_tokens, void* d_weight, void* d_bias,
                        void* d_cls, void* d_pos, int B, int C, int Hi, int Wi, int P, int E,
                        int img_dtype, int dtype, int tok_dtype, void* stream);
/* The same with n_prefix prefix tokens: d_tokens [B][n_prefix+Np][E]; d_prefix fp32 [n_prefix][E] with
 * d_prefix[t] = sum_b d_tokens[b][t]; d_pos, d_bias and d_weight come from the rows t >= n_prefix.  n_prefix = 1 is
 * vrr_patch_embed_bwd. */
int vrr_patch_embed_bwd_prefix(const void* images, const void* d_tokens, void* d_weight, void* d_bias, void* d_prefix,
                               int n_prefix, void* d_pos, int B, int C, int Hi, int Wi, int P, int E, int img_dtype,
                               int dtype, int tok_dtype, void* stream);

/* ---- (a) QKV projection with RoPE epilogue: models/vit.py:47-68, rope_utils.py:3-37 -------- */
/* planes = split_heads(x . w_qkv^T) with q,k rows 1.. rotated by (cos,sin) in the epilogue (n_prefix = 1).
 * x [B*N][E], w_qkv [3E][E] (row order (3,H,Dh), vit.py:47), cos/sin fp32 (see vrr_rope_mode),
 * planes [3][B][H][N][Dh]. */
int vrr_qkv_rope_fwd(const void* x, const void* w_qkv, const float* cos_tab, const float* sin_tab,
                     void* planes, int B, int N, int E, int H, int rope_mode, int dtype,
                     void* stream);
/* Optional fast path for the tables: `packed` = vrr_rope_pack_tables(cos_tab, sin_tab) of the SAME tables,
 * [heads][half_dim/2][rows] float4 {cos[2q], sin[2q], cos[2q+1], sin[2q+1]} (heads = H for rope-mixed, 1 for
 * rope-axial; rows = N-n_prefix; half_dim = Dh/2).  In the tcgen05 epilogue a lane is a token row: with the row-major tables
 * one load instruction touches 32 cache lines, with the packed table 4 (ViT-B rope-mixed: 189 -> ~140 us).  Results
 * are bit-identical.  `packed` may be NULL (= vrr_qkv_rope_fwd); cos_tab / sin_tab are still required (the SIMT
 * family reads them). */
int vrr_rope_pack_tables(const float* cos_tab, const float* sin_tab, float* packed, int heads, int rows,
                         int half_dim, void* stream);
int vrr_qkv_rope_fwd_packed(const void* x, const void* w_qkv, const float* cos_tab, const float* sin_tab,
                            const float* packed, void* planes, int B, int N, int E, int H, int rope_mode,
                            int dtype, void* stream);
/* vrr_qkv_rope_fwd_packed with n_prefix prefix tokens: q,k rows t >= n_prefix are rotated by table row t - n_prefix
 * (cos/sin and `packed` have N - n_prefix rows); rows t < n_prefix and all of v are stored as computed. */
int vrr_qkv_rope_fwd_prefix(const void* x, const void* w_qkv, const float* cos_tab, const float* sin_tab,
                            const float* packed, void* planes, int B, int N, int E, int H, int n_prefix, int rope_mode,
                            int dtype, void* stream);
/* Backward of the epilogue: un-rotates d_planes into token layout and reduces the table grads.
 * d_planes [3][B][H][N][Dh] (grads w.r.t. rotated q,k and v), planes = forward output,
 * d_qkv [B*N][3E] (gradient of x . w_qkv^T, ready for the two plain GEMMs dX = d_qkv . W and
 * dW = d_qkv^T . x), d_cos/d_sin fp32 with the shape of cos/sin or NULL (skipped), written. */
int vrr_qkv_rope_bwd(const void* d_planes, const void* planes, const float* cos_tab,
                     const float* sin_tab, void* d_qkv, float* d_cos, float* d_sin, int B, int N,
                     int E, int H, int rope_mode, int dtype, void* stream);
/* The same with n_prefix prefix tokens: rows t >= n_prefix are un-rotated with table row t - n_prefix and feed
 * d_cos / d_sin there ([..][N-n_prefix][Dh/2]); prefix rows pass through. */
int vrr_qkv_rope_bwd_prefix(const void* d_planes, const void* planes, const float* cos_tab, const float* sin_tab,
                            void* d_qkv, float* d_cos, float* d_sin, int B, int N, int E, int H, int n_prefix,
                            int rope_mode, int dtype, void* stream);

/* QK-norm (timm's Attention(qk_norm=True); ViT-22B): a LayerNorm over the Dh channels of every q and k head row,
 * including the prefix rows, before RoPE.  q_norm and k_norm are affine with weight / bias qn_w, qn_b / kn_w, kn_b
 * (fp32 [Dh], shared by all heads, all required) and one `eps`.  For every token row and head, with T = `dtype`:
 *   1. x = T(acc), the projection rounded to T (nn.Linear's output under autocast; x = acc for fp32);
 *   2. mean = sum(x) / Dh, var = sum((x - mean)^2) / Dh (biased), rstd = rsqrtf(var + eps), all in fp32;
 *      xhat = (x - mean) * rstd and y = xhat * g + b, each without FMA contraction of the subtraction and product;
 *   3. rows t >= n_prefix: y rotated by RoPE in fp32 as in vrr_qkv_rope_fwd_prefix;
 *   4. the result rounded to T once.  The v plane is the plain projection, as without the norm.
 * (Without the norm the q / k rows are rotated from the unrounded accumulator: step 1 is what the backward saves.)
 * Saved outputs (both or neither; NULL: inference): qk_pre [2][B][H][N][Dh] of T, the x of q (plane 0) and k
 * (plane 1) in the layout of planes; qk_stats fp32 [2][B][H][N][2] = {mean, rstd}.  Arguments and kernel family
 * choice are those of vrr_qkv_rope_fwd_prefix.  qk_pre / the norm tensors must be 16-byte aligned. */
int vrr_qkv_rope_norm_fwd(const void* x, const void* w_qkv, const float* cos_tab, const float* sin_tab, const float* packed,
                          void* planes, int B, int N, int E, int H, int n_prefix, int rope_mode, int dtype, const float* qn_w,
                          const float* qn_b, const float* kn_w, const float* kn_b, float eps, void* qk_pre, float* qk_stats,
                          void* stream);
/* Backward of vrr_qkv_rope_norm_fwd from its saved outputs.  Per q / k row, dy = the un-rotated d_planes row in fp32
 * (d_planes itself on prefix rows), xhat recomputed from qk_pre / qk_stats as in the forward:
 *   d_qkv = T(rstd (g dy - mean(g dy) - xhat mean(g dy xhat)))   (v columns: d_planes[2] unchanged)
 *   d_g = sum dy xhat, d_b = sum dy over images, tokens and heads (fp32 atomics: reproducible to ~1e-6, not bitwise)
 *   d_cos / d_sin as in vrr_qkv_rope_bwd_prefix with the un-rotated value y = xhat g + b, recomputed bit for bit.
 * d_qn_w, d_qn_b, d_kn_w, d_kn_b [Dh] are written (not accumulated): all four or none; d_cos / d_sin both or neither. */
int vrr_qkv_rope_norm_bwd(const void* d_planes, const void* qk_pre, const float* qk_stats, const float* cos_tab,
                          const float* sin_tab, const float* qn_w, const float* qn_b, const float* kn_w, const float* kn_b,
                          void* d_qkv, float* d_cos, float* d_sin, float* d_qn_w, float* d_qn_b, float* d_kn_w,
                          float* d_kn_b, int B, int N, int E, int H, int n_prefix, int rope_mode, int dtype, void* stream);

/* Stand-alone rotate-half of rope_utils.py:3-37 (the public apply_rotary_emb): q,k [B][H][Nr][Dh]
 * dense, cos/sin fp32 [Nr][Dh/2] (AXIAL) or [H][Nr][Dh/2] (MIXED); every row is rotated.
 * inverse != 0 applies the transpose rotation (the gradient w.r.t. q,k). */
int vrr_rope_apply(const void* q_in, const void* k_in, const float* cos_tab, const float* sin_tab,
                   void* q_out, void* k_out, int B, int H, int Nr, int Dh, int rope_mode,
                   int inverse, int dtype, void* stream);

/* Gradient of vrr_rope_apply (inverse == 0) w.r.t. its tables: d_cos, d_sin fp32 with the shape of
 * cos/sin, written (not accumulated); q_in, k_in = the un-rotated inputs, dq, dk = gradients w.r.t. the
 * rotated outputs.  Deterministic (no atomics). */
int vrr_rope_table_grad(const void* q_in, const void* k_in, const void* dq, const void* dk, float* d_cos,
                        float* d_sin, int B, int H, int Nr, int Dh, int rope_mode, int dtype, void* stream);

/* Plain GEMM used by the backward of the projection: C = op(A) . op(B), row-major operands,
 * op(A) is [M][K] (trans_a: A is stored [K][M]), op(B) is [K][N] (trans_b: B is stored [N][K]).
 * `dtype` is the element type of A and B, `c_dtype` that of C (fp32 C is allowed for bf16 / fp16 inputs:
 * weight gradients).  fp32 accumulation always. */
int vrr_gemm(const void* a, const void* b, void* c, int M, int N, int K, int trans_a, int trans_b,
             int dtype, int c_dtype, void* stream);

/* GEMM of the Linear layers of the path and of their backward, with fused epilogues:
 * C[M][N] = op(A).op(B) with the vrr_gemm operand conventions; `dtype` = element type of A and B.
 *   forward  y = x.W^T (+b)        : trans_a 0, trans_b 1   (models/vit.py:47,91,118,285)
 *   backward dX = dY.W             : trans_a 0, trans_b 0
 *   backward dW = dY^T.X           : trans_a 1, trans_b 0, c_dtype VRR_F32
 * epilogue (vrr_epilogue): BIAS adds the fp32 `bias[N]` (cast to `dtype` first, like F.linear on `dtype`
 * tensors) before the single rounding to c_dtype; BIAS_GELU additionally writes C2 = gelu(C), exact erf GELU
 * (timm Mlp, act_layer=nn.GELU); BIAS_GELU_GRAD writes C = gelu(h) and C2 = gelu'(h) for h = round(acc + bias)
 * (h itself is not stored: the Mlp backward only needs gelu'); MUL multiplies by the INPUT matrix C2[M][N]
 * before rounding (fc2's dX fused with the GELU backward: dh = (dy . W2) * gelu'(h)).  accumulate != 0 (fp32 C, tcgen05 kernel only): C += result.
 * bf16 or fp16 operands with N % 8 == 0, K % 8 == 0 (and M % 8 == 0 when trans_a) and 16-byte aligned pointers run
 * the tcgen05 CTA-pair kernel (cta_group::2, TMA in, TMA store / reduce-add out; fp32 C is split over K and
 * combined by TMA reduce-add, so its summation order is not deterministic); everything else (fp32 operands,
 * odd shapes, a pointer that is not 16-byte aligned, e.g. a view at an offset into a larger buffer) runs the
 * FFMA kernel.  vrr_set_impl() forces a family (VRR_IMPL_TCGEN05 with a case the tcgen05 kernel cannot take:
 * VRR_ERR_UNSUPPORTED); vrr_family_count() reports it.  The same dispatch applies to vrr_gemm_mul_colsum. */
int vrr_gemm_ex(const void* a, const void* b, void* c, void* c2, const float* bias, int M, int N, int K,
                int trans_a, int trans_b, int dtype, int c_dtype, int epilogue, int accumulate, void* stream);

/* ---- (b) fused attention: models/vit.py:71-88 ---------------------------------------------- */
/* out = merge_heads(softmax(q k^T * scale + bias) v), lse = log-sum-exp of the logits.
 * planes [3][B][H][N][Dh], out [B][N][H*Dh], lse fp32 [B][H][N].  scale = Dh^-0.5 (vit.py:32),
 * applied after q k^T and before the bias (vit.py:71,75). */
int vrr_attn_fwd(const void* planes, const vrr_bias_desc* bias, void* out, float* lse, int B,
                 int H, int N, int Dh, float scale, int dtype, void* stream);
size_t vrr_attn_bwd_workspace_bytes(int B, int H, int N, int Dh, const vrr_bias_desc* bias);
/* d_planes [3][B][H][N][Dh] (dq, dk, dv w.r.t. the planes), written.
 * d_bias_param fp32 [bias->heads][bias->len] or NULL: gradient of the table / coefficients summed
 * over the batch, written (not accumulated).  workspace: device scratch of at least
 * vrr_attn_bwd_workspace_bytes() bytes. */
int vrr_attn_bwd(const void* planes, const vrr_bias_desc* bias, const void* out, const void* d_out,
                 const float* lse, void* d_planes, float* d_bias_param, void* workspace,
                 size_t workspace_bytes, int B, int H, int N, int Dh, float scale, int dtype,
                 void* stream);

/* ---- (f) N1, first "next" row: LayerNorm of the token stream, models/vit.py:113,117,122,124,210 - */
/* y = (x - mean) * rstd * gamma + beta over the last dimension (nn.LayerNorm, biased variance, eps
 * inside the sqrt).  x [M][E] (`x_dtype`), y [M][E] (`y_dtype`: the consumer GEMM's dtype, so that
 * under autocast the fp32 -> bf16 cast of the reference is fused into the store), gamma/beta fp32 [E],
 * mean/rstd fp32 [M] (saved for the backward). */
int vrr_layernorm_fwd(const void* x, const float* gamma, const float* beta, void* y, float* mean,
                      float* rstd, int M, int E, float eps, int x_dtype, int y_dtype, void* stream);
/* dx [M][E] (`x_dtype`), dgamma/dbeta fp32 [E] (written, not accumulated), from dy [M][E] (`y_dtype`). */
int vrr_layernorm_bwd(const void* dy, const void* x, const float* gamma, const float* mean,
                      const float* rstd, void* dx, float* dgamma, float* dbeta, int M, int E,
                      int x_dtype, int y_dtype, void* stream);

/* Fused residual add + LayerNorm of the pre-LN block (models/vit.py:122-124: x = x + branch; the next
 * sub-block starts with norm(x)):  x_new = x + branch (fp32, written);  y = LayerNorm(x_new).
 * x, x_new fp32 [M][E]; branch `branch_dtype`; y `y_dtype`. */
int vrr_add_layernorm_fwd(const void* x, const void* branch, void* x_new, const float* gamma,
                          const float* beta, void* y, float* mean, float* rstd, int M, int E, float eps,
                          int branch_dtype, int y_dtype, void* stream);
/* g = d_xnew + LayerNorm'(dy): written as fp32 `dx` (gradient of x) and in `branch_dtype` as `d_branch`
 * (gradient of branch - the same values); d_xnew may be NULL (no other consumer of x_new). */
int vrr_add_layernorm_bwd(const void* dy, const void* d_xnew, const void* x_new, const float* gamma,
                          const float* mean, const float* rstd, void* dx, void* d_branch, float* dgamma,
                          float* dbeta, int M, int E, int branch_dtype, int y_dtype, void* stream);

/* The same with dropout / stochastic depth on the branch (Block with proj_drop / Mlp drop2 and DropPath):
 *   forward : x_new = x + f * branch (the product rounded to fp32, never contracted into the add), so x_new, y,
 *             mean and rstd are bit-identical to vrr_add_layernorm_fwd fed the fp32 branch f * branch;
 *   backward: dx as vrr_add_layernorm_bwd; d_branch = round_to_branch_dtype(dx * f), the masks regenerated from the
 *             same desc (nothing is stored between the passes).
 * The element masks are indexed by (row, column) of the [M][E] stream (E % 8 == 0 when p > 0).  `drop` NULL, or
 * p == p_path == 0, is exactly the entry point above. */
int vrr_add_layernorm_drop_fwd(const void* x, const void* branch, void* x_new, const float* gamma,
                               const float* beta, void* y, float* mean, float* rstd, int M, int E, float eps,
                               int branch_dtype, int y_dtype, const vrr_drop_desc* drop, void* stream);
int vrr_add_layernorm_drop_bwd(const void* dy, const void* d_xnew, const void* x_new, const float* gamma,
                               const float* mean, const float* rstd, void* dx, void* d_branch, float* dgamma,
                               float* dbeta, int M, int E, int branch_dtype, int y_dtype,
                               const vrr_drop_desc* drop, void* stream);

/* The same with LayerScale on the branch (timm's LayerScale, Block(init_values): x = x + drop_path(ls * branch)).
 * ls fp32 [E].  f is the factor of `drop` as above; without a desc (drop NULL) no f product is taken.  Every product
 * is rounded to fp32 and never contracted into the add:
 *   forward : b' = fl(fl(f * branch) * ls[c]); x_new = x + b'; y = LayerNorm(x_new).  x_new, y, mean and rstd are
 *             bit-identical to vrr_add_layernorm_fwd fed the fp32 branch b'.  Without dropout b' = fl(branch * ls),
 *             torch's product of a 16-bit tensor and an fp32 parameter;
 *   backward: dx as vrr_add_layernorm_bwd; d_branch = round_to_branch_dtype(fl(fl(dx * f) * ls[c]));
 *             d_ls[c] = sum_m fl(dx * f)[m][c] * float(branch[m][c]), an fp32 column sum (written, not accumulated;
 *             like dgamma / dbeta its summation order is not fixed).  `branch` is the forward's branch input
 *             (`branch_dtype`); it is read only when d_ls is not NULL.
 * d_ls non-NULL needs ls and branch (VRR_ERR_INVALID_ARG otherwise).  ls NULL is exactly the _drop_ entry points
 * (branch and d_ls are then not used).  With ls the backward keeps a third [warps][E] partial in shared memory:
 * E <= 1706 (VRR_ERR_UNSUPPORTED beyond). */
int vrr_add_layernorm_ls_fwd(const void* x, const void* branch, void* x_new, const float* gamma,
                             const float* beta, void* y, float* mean, float* rstd, int M, int E, float eps,
                             int branch_dtype, int y_dtype, const vrr_drop_desc* drop, const float* ls,
                             void* stream);
int vrr_add_layernorm_ls_bwd(const void* dy, const void* d_xnew, const void* x_new, const float* gamma,
                             const float* mean, const float* rstd, void* dx, void* d_branch, float* dgamma,
                             float* dbeta, int M, int E, int branch_dtype, int y_dtype,
                             const vrr_drop_desc* drop, const float* ls, const void* branch, float* d_ls,
                             void* stream);

/* vrr_gemm_ex with element dropout on the GELU outputs (fc1 of an Mlp with drop1 > 0), for the epilogues
 * VRR_EPI_BIAS_GELU_GRAD (C = T(T(gelu(h)) * f), C2 = T(T(gelu'(h)) * f)) and VRR_EPI_BIAS_GELU_ACT
 * (C = T(T(gelu(h)) * f)), T = `dtype`; `drop->p_path` must be 0.  The mask is indexed by (m, n) of C (N % 8 == 0).
 * This is torch's rounding of Dropout on a 16-bit tensor, and fc2's dX through VRR_EPI_MUL then yields
 * (dy . W2) * gelu'(h) * f: Dropout's backward.  The tcgen05 kernel takes the Linear-forward layout (trans_a 0,
 * trans_b 1) under the vrr_gemm_ex conditions; everything else runs the SIMT route. */
int vrr_gemm_ex_drop(const void* a, const void* b, void* c, void* c2, const float* bias, int M, int N, int K,
                     int trans_a, int trans_b, int dtype, int c_dtype, int epilogue, int accumulate,
                     const vrr_drop_desc* drop, void* stream);

/* The decisions the kernels above take for `drop`: keep_u8 [M][E] (1 kept, 0 dropped; the element mask alone) and
 * keep_path_u8 [ceil(M / rows_per_sample)] (the stochastic-depth decision per image); either may be NULL.  A
 * probability of 0 writes all ones. */
int vrr_dropout_mask(const vrr_drop_desc* drop, void* keep_u8, void* keep_path_u8, int M, int E, void* stream);

/* fc2's input gradient with the GELU backward and fc1's bias gradient fused (autograd of timm Mlp, vit.py:118):
 *   c[m][n] = (op(a) . op(b))[m][n] * mul[m][n]   (`dtype`, as VRR_EPI_MUL)
 *   col_sums[n] = sum_m c[m][n]                   (fp32 [N], written; sums the values AS STORED, like autograd's
 *                                                  sum over the bf16 / fp16 tensor)
 * bf16 / fp16 on the tcgen05 kernel: the epilogue adds the column sums of each staged tile (fp32 atomics - summation
 * order not deterministic); otherwise vrr_gemm_ex(VRR_EPI_MUL) followed by vrr_colsum. */
int vrr_gemm_mul_colsum(const void* a, const void* b, void* c, const void* mul, float* col_sums, int M, int N,
                        int K, int trans_a, int trans_b, int dtype, void* stream);

/* fc1 of a packed SwiGLU Mlp (timm's SwiGLUPacked: fc2(silu(x W_g^T + b_g) * (x W_v^T + b_v))), T = `dtype`.
 * x [M][K], w1 [2H][K] (fc1.weight: gate rows [0, H), then value rows [H, 2H)), b1 fp32 [2H]; act [M][H];
 * aux [M][2H] or NULL (torch.no_grad: act only).  For output column j (rounding as torch on T tensors):
 *   g = T(acc_j + T(b1[j])),  v = T(acc_{H+j} + T(b1[H+j]))                 (F.linear)
 *   s = T(silu(g))                                                          (nn.SiLU)
 *   act[m][j]     = T(T(s * v) * f)                                         (the product, then Dropout)
 *   aux[m][j]     = T(fl(v * silu'(g)) * f)                                 (d act / d g)
 *   aux[m][H + j] = T(s * f)                                                (d act / d v)
 * Every product is an fp32 multiply rounded to nearest; silu and silu' carry the error bound documented in
 * csrc/common.cuh (relative 2^-20 (1 + |g|), plus 2^-126 (1 + |g|) absolute where sigma underflows).  f is the factor of `drop` for element (m, j) of act [M][H] (as
 * vrr_gemm_ex_drop: p_path must be 0, the mask groups need H % 8 == 0); drop NULL or p == 0: f = 1 and no product is
 * taken.  bf16 / fp16 with H % 8 == 0, K % 8 == 0 and 16-byte aligned pointers run the tcgen05 kernel (gate and value
 * columns paired in one accumulator tile); everything else, fp32 included, the FFMA kernel with the same arithmetic.
 * vrr_set_impl / vrr_family_count as for vrr_gemm_ex.  No workspace. */
int vrr_gemm_swiglu(const void* x, const void* w1, const float* b1, void* act, void* aux, int M, int H, int K,
                    int dtype, const vrr_drop_desc* drop, void* stream);
/* fc2's dX with the SwiGLU backward and fc1's bias gradient: dA = dy [M][K] . w2 [K][H] (fc2.weight) in fp32, then
 *   dh [M][2H]:  dh[m][j] = T(dA[m][j] * aux[m][j]),  dh[m][H + j] = T(dA[m][j] * aux[m][H + j])
 *   db1 fp32 [2H] = column sums of dh as stored (written; tcgen05: fp32 atomics, summation order not fixed).
 * dh is then the gradient of fc1's output (dX = dh . w1 and dW1 = dh^T x are plain vrr_gemm_ex calls).  H % 2 == 0.
 * Dispatch as vrr_gemm_swiglu; the FFMA route is the GEMM with the products in its epilogue, then vrr_colsum. */
int vrr_gemm_swiglu_bwd(const void* dy, const void* w2, const void* aux, void* dh, float* db1, int M, int H,
                        int K, int dtype, void* stream);

/* Bias gradient of a Linear layer (out-proj vit.py:91, Mlp fc1/fc2 vit.py:118, head vit.py:285):
 * out[c] = sum_m x[m][c], fp32 [C] (written); x [M][C] `dtype`, C % 4 == 0, any element-aligned address (a view
 * at an offset into a larger buffer takes an element-wise kernel). */
int vrr_colsum(const void* x, float* out, int M, int C, int dtype, void* stream);
/* Backward of the exact (erf) GELU between fc1 and fc2 of the Mlp (vit.py:118, act_layer=nn.GELU):
 * dh = dy * gelu'(h), written in `dtype`, and db[c] = sum_m dh[m][c] (fp32, written) - the fc1 bias
 * gradient - in the same pass.  dy, h, dh [M][C]. */
int vrr_gelu_bwd(const void* dy, const void* h, void* dh, float* db, int M, int C, int dtype, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VRR_H_ */
