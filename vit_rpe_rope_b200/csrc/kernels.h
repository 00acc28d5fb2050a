// Internal kernel-launcher declarations shared by the translation units of libvrr_b200.so.
#pragma once
#include <cuda_runtime.h>

#include "../../include/vrr.h"

namespace vrr {

struct DropView;  // common.cuh

// attn_simt.cu
int attn_fwd_simt(const void* planes, const vrr_bias_desc* bias, void* out, float* lse, int B, int H, int N,
                  int Dh, float scale, int dtype, cudaStream_t st);
int attn_bwd_simt(const void* planes, const vrr_bias_desc* bias, const void* out, const void* d_out,
                  const float* lse, void* d_planes, float* d_bias_param, float* delta, float* d_lut_ws, int B,
                  int H, int N, int Dh, float scale, int dtype, cudaStream_t st);

// The tcgen05 launchers below take `dtype` VRR_BF16 or VRR_F16 (the operands' and the 16-bit outputs' element type).

// attn_tc.cu (tcgen05 / TMEM, Dh == 64; tiled over 64-key tiles): without bias attn_fwd_tc4_kernel (four CTAs
// per SM), with a bias attn_fwd_tc2_kernel (two CTAs per SM)
bool attn_fwd_tc_supported(int B, int H, int N, int Dh, const vrr_bias_desc* bias);
void attn_fwd_tc_set_debug(long long* buf);
int attn_fwd_tc(const void* planes, const vrr_bias_desc* bias, void* out, float* lse, int B, int H, int N,
                int Dh, float scale, int dtype, cudaStream_t st);

// attn_fwd_ws.cu (whole-sequence forward with a bias for N <= 256: persistent, one round trip per (image, head))
bool attn_fwd_ws_supported(int B, int H, int N, int Dh, const vrr_bias_desc* bias);
int attn_fwd_ws(const void* planes, const vrr_bias_desc* bias, void* out, float* lse, int B, int H, int N, int Dh,
                float scale, int dtype, cudaStream_t st);

// attn_bwd_tc2.cu (dQ and dK/dV kernels: issuer warp, double-buffered 32-row tiles; every case attn_bwd_ws.cu does
// not take)
bool attn_bwd_tc2_supported(int B, int H, int N, int Dh, const vrr_bias_desc* bias);
int attn_bwd_tc2(const void* planes, const vrr_bias_desc* bias, const void* out, const void* d_out, const float* lse,
                 void* d_planes, float* d_bias_param, float* delta, int B, int H, int N, int Dh, float scale,
                 int dtype, cudaStream_t st);

// attn_bwd_ws.cu (whole-sequence fused backward for N <= 256, no bias: one persistent kernel, operands read once)
bool attn_bwd_ws_supported(int B, int H, int N, int Dh, const vrr_bias_desc* bias);
void attn_bwd_ws_set_debug(long long* buf);
int attn_bwd_ws(const void* planes, const void* out, const void* d_out, const float* lse, void* d_planes, int B, int H,
                int N, int Dh, float scale, int dtype, cudaStream_t st);

// QK-norm of the QKV+RoPE forward (vrr_qkv_rope_norm_fwd): fp32 [Dh] affine parameters of q_norm / k_norm, eps, and
// the saved outputs qk_pre [2][B][H][N][Dh] (the compute type) and qk_stats [2][B][H][N][2] {mean, rstd}, or both NULL
struct QkNormArgs {
  const float *qn_w, *qn_b, *kn_w, *kn_b;
  float eps;
  void* qk_pre;
  float* qk_stats;
};

// gemm_simt.cu
void layernorm_set_option(int which, int value);  // 0: ln_reg, 1: ln_bwd_minb
void gemm_simt_set_tile(int v);  // 128 (default): 128 x 128 double-buffered kernel for problems with a full tile; 64: 64 x 64 always
// npre: prefix tokens per image (token rows 0..npre-1: cls, then registers); they are never rotated, and the patch
// rows t >= npre use table row t - npre
int qkv_rope_fwd_simt(const void* x, const void* w, const float* cos_tab, const float* sin_tab, void* planes,
                      int B, int N, int E, int H, int npre, int rope_mode, int dtype, cudaStream_t st,
                      const QkNormArgs* qn = nullptr);
int gemm_simt(const void* a, const void* b, void* c, int M, int N, int K, int ta, int tb, int dtype,
              int c_dtype, cudaStream_t st);
int gemm_simt_bias(const void* a, const void* b, void* c, void* c2, const float* bias, int M, int N, int K, int ta, int tb,
                   int dtype, int gelu, cudaStream_t st);
int patch_embed_fwd_simt(const void* images, const void* weight, const void* bias, const void* prefix,
                         const void* pos, void* tokens, int B, int C, int Hi, int Wi, int P, int E, int npre,
                         int img_dtype, int dtype, int tok_dtype, cudaStream_t st);
int patch_embed_bwd_simt(const void* images, const void* d_tokens, float* d_weight, float* d_bias, float* d_prefix,
                         float* d_pos, int B, int C, int Hi, int Wi, int P, int E, int npre, int img_dtype, int dtype,
                         int tok_dtype, cudaStream_t st);
// SwiGLU Mlp on the FFMA kernels (any H, K; dv NULL: no dropout; aux NULL: act only).  The backward writes dh only.
int swiglu_simt(const void* x, const void* w1, const float* b1, void* act, void* aux, int M, int H, int K, int dtype,
                const DropView* dv, cudaStream_t st);
int swiglu_bwd_simt(const void* dy, const void* w2, const void* aux, void* dh, int M, int H, int K, int dtype, cudaStream_t st);
int patch_prefix_rows(void* tokens, const void* prefix, int B, int Np, int E, int npre, int tok_dtype, cudaStream_t st);

// gemm_tc2.cu (tcgen05 CTA pairs, cta_group::2: every operand layout, TMA-store epilogues)
bool gemm_tc_supported(int M, int N, int K, int trans_a, int trans_b, int dtype, int c_dtype, int epilogue);
int gemm_tc(const void* a, const void* b, void* c, void* c2, const float* bias, int M, int N, int K, int trans_a,
            int trans_b, int dtype, int c_dtype, int epilogue, int accumulate, cudaStream_t st, float* colsum = nullptr);
// fc1 with element dropout on the GELU outputs (VRR_EPI_BIAS_GELU_GRAD / _ACT, trans_a 0, trans_b 1, C of dtype)
int gemm_tc_drop(const void* a, const void* b, void* c, void* c2, const float* bias, int M, int N, int K, int dtype,
                 int epilogue, const DropView& dv, cudaStream_t st);
// SwiGLU Mlp (vrr.h: vrr_gemm_swiglu / vrr_gemm_swiglu_bwd): 16-bit, H % 8 == 0, K % 8 == 0, 16-byte aligned pointers.
// dv NULL: no dropout; aux NULL: act only.  The backward writes db1 (it zeroes it first).
int gemm_tc_swiglu(const void* x, const void* w1, const float* b1, void* act, void* aux, int M, int H, int K, int dtype,
                   const DropView* dv, cudaStream_t st);
int gemm_tc_swiglu_bwd(const void* dy, const void* w2, const void* aux, void* dh, float* db1, int M, int H, int K, int dtype,
                       cudaStream_t st);
// colsum (16-bit C, plain / bias / multiply epilogues): colsum[n] += sum_m C[m][n] of the values as stored; zeroed by the caller
int rope_pack_tables(const float* cos_tab, const float* sin_tab, float* packed, int heads, int rows, int hd, cudaStream_t st);
bool qkv_rope_fwd_tc_supported(int B, int N, int E, int H);
// `packed`: optional output of rope_pack_tables for the same tables (NULL: the epilogue reads cos_tab / sin_tab)
int qkv_rope_fwd_tc2(const void* x, const void* w, const float* cos_tab, const float* sin_tab, const float* packed, void* planes, int B, int N,
                     int E, int H, int npre, int rope_mode, int dtype, cudaStream_t st, const QkNormArgs* qn = nullptr);

bool patch_embed_tc_supported(int B, int C, int Hi, int Wi, int P, int E);
size_t patch_embed_tc_workspace_bytes(int B, int C, int Hi, int Wi, int P);
// out_dtype: VRR_BF16 or VRR_F16; images fp32 or of out_dtype
int patch_unfold(const void* images, void* out, int B, int C, int Hi, int Wi, int P, int img_dtype, int out_dtype,
                 cudaStream_t st);
int patch_embed_fwd_tc(const void* images, const void* weight, const void* bias, const void* pos, void* tokens,
                       void* workspace, int B, int C, int Hi, int Wi, int P, int E, int npre, int img_dtype, int dtype,
                       int tok_dtype, cudaStream_t st);

// layernorm.cu
int layernorm_fwd(const void* x, const float* gamma, const float* beta, void* y, float* mean, float* rstd, int M, int E,
                  float eps, int x_dtype, int y_dtype, cudaStream_t st);
int layernorm_bwd(const void* dy, const void* x, const float* gamma, const float* mean, const float* rstd, void* dx,
                  float* dgamma, float* dbeta, int M, int E, int x_dtype, int y_dtype, cudaStream_t st);

// drop: NULL or a desc that draws nothing runs the plain kernels; ls: NULL runs the kernels without LayerScale
// (branch and d_ls are then ignored); d_ls NULL: no LayerScale gradient (branch is not read)
int add_layernorm_fwd(const void* x, const void* branch, void* x_new, const float* gamma, const float* beta, void* y,
                      float* mean, float* rstd, int M, int E, float eps, int branch_dtype, int y_dtype,
                      const vrr_drop_desc* drop, const float* ls, cudaStream_t st);
int add_layernorm_bwd(const void* dy, const void* d_xnew, const void* x_new, const float* gamma, const float* mean,
                      const float* rstd, void* dx, void* d_branch, float* dgamma, float* dbeta, int M, int E,
                      int branch_dtype, int y_dtype, const vrr_drop_desc* drop, const float* ls, const void* branch,
                      float* d_ls, cudaStream_t st);

// elementwise.cu
int colsum(const void* x, float* out, int M, int C, int dtype, cudaStream_t st);
int gelu_bwd_colsum(const void* dy, const void* h, void* dh, float* db, int M, int C, int dtype, cudaStream_t st);
int gelu_grad_inplace(void* h, size_t n, int dtype, cudaStream_t st);            // h <- d gelu / dh (h)
int mul_inplace(void* c, const void* m, size_t n, int dtype, cudaStream_t st);  // c <- c * m
// c <- T(c * f) and, when c2 is given, c2 <- T(T(gelu'(c2)) * f) (SIMT route of vrr_gemm_ex_drop); c, c2 [M][N]
int drop_gelu_inplace(void* c, void* c2, int M, int N, int dtype, const DropView& dv, cudaStream_t st);
int dropout_mask(const DropView& dv, uint8_t* keep, uint8_t* keep_path, int M, int E, cudaStream_t st);

// rope.cu
int qkv_rope_bwd(const void* d_planes, const void* planes, const float* cos_tab, const float* sin_tab,
                 void* d_qkv, float* d_cos, float* d_sin, int B, int N, int E, int H, int npre, int rope_mode, int dtype,
                 cudaStream_t st);
// QK-norm backward (vrr_qkv_rope_norm_bwd): qn->qk_pre / qk_stats are the forward's saved outputs; d_w / d_b
// [q, k] are written (zeroed here, atomically reduced), or all NULL
struct QkNormGrads {
  float *d_qn_w, *d_qn_b, *d_kn_w, *d_kn_b;
};
int qkv_rope_norm_bwd(const void* d_planes, const QkNormArgs& qn, const float* cos_tab, const float* sin_tab, void* d_qkv,
                      float* d_cos, float* d_sin, const QkNormGrads& grads, int B, int N, int E, int H, int npre,
                      int rope_mode, int dtype, cudaStream_t st);
int rope_apply(const void* q_in, const void* k_in, const float* cos_tab, const float* sin_tab, void* q_out,
               void* k_out, int B, int H, int Nr, int Dh, int rope_mode, int inverse, int dtype, cudaStream_t st);

int rope_table_grad(const void* q_in, const void* k_in, const void* dq, const void* dk, float* d_cos, float* d_sin,
                    int B, int H, int Nr, int Dh, int rope_mode, int dtype, cudaStream_t st);

}  // namespace vrr
