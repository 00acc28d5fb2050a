// extern "C" entry points of libvrr_b200.so (see include/vrr.h): argument validation, kernel
// family selection, workspace carving.  No allocation, no synchronisation, no exceptions.
#include <stdarg.h>
#include <string.h>

#include "common.cuh"
#include "kernels.h"

namespace vrr {

static thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};
std::atomic<int> g_impl{VRR_IMPL_AUTO};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// Per-DEVICE state (a process may drive several GPUs): 0 unknown, 1 ok, -1 not sm_100.  Plain
// atomics: racing first calls on one device compute the same values.
constexpr int kMaxDevices = 64;
static std::atomic<int> g_dev_state[kMaxDevices];
static std::atomic<int> g_dev_sms[kMaxDevices];
std::atomic<uint64_t> g_family_launches[3];  // [VRR_IMPL_SIMT], [VRR_IMPL_TCGEN05] dispatch counters

int current_device() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    cudaGetLastError();
    return -1;
  }
  return dev;
}

int require_device() {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("no CUDA device: %s", cudaGetErrorString(e));
    return VRR_ERR_NO_DEVICE;
  }
  if (dev < 0 || dev >= kMaxDevices) {
    set_error("device ordinal %d out of range", dev);
    return VRR_ERR_NO_DEVICE;
  }
  // Driver-API calls made by the launchers (cuTensorMapEncodeTiled) need the primary context CURRENT in the
  // calling thread.  A runtime call that touches the device binds it; cudaGetDevice does not.  PyTorch's autograd
  // worker threads reach this library without one when their allocations are served from the caching allocator
  // (observed: CUDA_ERROR_INVALID_CONTEXT from the first backward of a process) - bind once per thread.
  static thread_local int bound_dev = -1;
  if (bound_dev != dev) {
    e = cudaFree(nullptr);
    if (e != cudaSuccess) {
      cudaGetLastError();
      set_error("cannot initialise the CUDA context of device %d: %s", dev, cudaGetErrorString(e));
      return VRR_ERR_NO_DEVICE;
    }
    bound_dev = dev;
  }
  const int state = g_dev_state[dev].load(std::memory_order_acquire);
  if (state == 1) return VRR_OK;
  int major = 0, minor = 0, sms = 0;
  e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("cudaDeviceGetAttribute: %s", cudaGetErrorString(e));
    return VRR_ERR_NO_DEVICE;
  }
  if (major != 10) {
    set_error("device %d is sm_%d%d; libvrr_b200 is built for sm_100a only (no fallback path)", dev, major, minor);
    g_dev_state[dev].store(-1, std::memory_order_release);
    return VRR_ERR_NO_DEVICE;
  }
  g_dev_sms[dev].store(sms, std::memory_order_relaxed);
  g_dev_state[dev].store(1, std::memory_order_release);
  return VRR_OK;
}
int sm_count() {
  const int dev = current_device();
  const int n = (dev >= 0 && dev < kMaxDevices) ? g_dev_sms[dev].load(std::memory_order_relaxed) : 0;
  return n > 0 ? n : 148;
}

// One-time per (kernel, device) attribute set-up: `flags` is a function-local static array.
bool first_use_on_device(std::atomic<unsigned char>* flags) {
  const int dev = current_device();
  if (dev < 0 || dev >= kMaxDevices) return true;
  return flags[dev].exchange(1, std::memory_order_acq_rel) == 0;
}

static bool dtype_ok(int d) { return d == VRR_F32 || d == VRR_BF16 || d == VRR_F16; }
// bf16 and fp16 never meet in one call (each pairs with fp32 only)
static bool no_mix(int a, int b, int c = VRR_F32) {
  const bool bf = a == VRR_BF16 || b == VRR_BF16 || c == VRR_BF16, hf = a == VRR_F16 || b == VRR_F16 || c == VRR_F16;
  return !(bf && hf);
}
static bool gemm_ptrs_aligned16(const void* a, const void* b, const void* c, const void* c2, const void* bias) {
  return (((uintptr_t)a | (uintptr_t)b | (uintptr_t)c | (uintptr_t)c2 | (uintptr_t)bias) & 15) == 0;
}
static bool dh_ok(int dh) { return dh == 16 || dh == 32 || dh == 64; }
// 1 <= n_prefix <= N, and the prefix rows of the batch indexable by the 32-bit index of the prefix-rows kernel
static bool prefix_ok(int n_prefix, long long N, int B, int E) {
  return n_prefix >= 1 && n_prefix <= N && (long long)B * n_prefix * E < (1ll << 31);
}

static int check_bias(const vrr_bias_desc* b, int H, int N) {
  if (!b || b->mode == VRR_BIAS_NONE) return VRR_OK;
  VRR_REQUIRE(b->param != nullptr, VRR_ERR_INVALID_ARG, "bias: param is NULL");
  if (b->mode == VRR_BIAS_TABLE) {
    VRR_REQUIRE(b->heads == H && b->len == 2 * N - 1, VRR_ERR_INVALID_ARG,
                "bias table must be [H=%d][2N-1=%d], got [%d][%d] (the relative table is tied to the "
                "construction-time token count)", H, 2 * N - 1, b->heads, b->len);
  } else if (b->mode == VRR_BIAS_POLY) {
    VRR_REQUIRE((b->heads == 1 || b->heads == H) && b->len >= 1 && b->len <= 16, VRR_ERR_INVALID_ARG,
                "poly coefficients must be [1 or H][1..16], got [%d][%d]", b->heads, b->len);
    VRR_REQUIRE(b->grid >= 1 && b->grid * b->grid == N - 1, VRR_ERR_INVALID_ARG,
                "poly bias needs N-1 == grid^2 (N=%d, grid=%d)", N, b->grid);
  } else {
    set_error("bias: unknown mode %d", b->mode);
    return VRR_ERR_INVALID_ARG;
  }
  return VRR_OK;
}

static uint32_t keep_threshold(float p) { return (uint32_t)llrint((1.0 - (double)p) * 65536.0); }

int drop_view(const vrr_drop_desc* d, int M, int E, DropView* v, bool* active) {
  (void)M;
  *active = false;
  if (!d) return VRR_OK;
  VRR_REQUIRE(d->p >= 0.f && d->p < 1.f && d->p_path >= 0.f && d->p_path < 1.f, VRR_ERR_INVALID_ARG,
              "drop desc: probabilities must lie in [0, 1) (p %g, p_path %g)", (double)d->p, (double)d->p_path);
  if (d->p == 0.f && d->p_path == 0.f) return VRR_OK;
  VRR_REQUIRE(d->seed != nullptr && ((uintptr_t)d->seed & 7) == 0, VRR_ERR_INVALID_ARG,
              "drop desc: seed must be an 8-byte aligned device pointer");
  VRR_REQUIRE(d->p == 0.f || E % 8 == 0, VRR_ERR_UNSUPPORTED, "drop desc: element dropout needs E %% 8 == 0 (E = %d)", E);
  VRR_REQUIRE(d->p_path == 0.f || d->rows_per_sample > 0, VRR_ERR_INVALID_ARG,
              "drop desc: stochastic depth needs rows_per_sample > 0");
  v->seed = reinterpret_cast<const unsigned long long*>(d->seed);
  v->t = keep_threshold(d->p);
  v->t_path = keep_threshold(d->p_path);
  v->s = (1.f / (1.f - d->p)) * (1.f / (1.f - d->p_path));
  v->rows_per_sample = d->rows_per_sample > 0 ? d->rows_per_sample : 1;
  v->site = d->site;
  *active = true;
  return VRR_OK;
}

}  // namespace vrr

using namespace vrr;

extern "C" {

int vrr_abi_version(void) { return VRR_ABI_VERSION; }
const char* vrr_last_error(void) { return g_err; }
int vrr_device_ok(void) { return require_device() == VRR_OK ? 1 : 0; }
int vrr_set_impl(int impl) {
  if (impl < VRR_IMPL_AUTO || impl > VRR_IMPL_TCGEN05) return g_impl.load();
  return g_impl.exchange(impl);
}
uint64_t vrr_launch_count(void) { return g_launches.load(); }
uint64_t vrr_family_count(int family) {
  if (family != VRR_IMPL_SIMT && family != VRR_IMPL_TCGEN05) return 0;
  return g_family_launches[family].load();
}
int vrr_debug_timestamps(void* device_buf) {  /* 64 x int64 device buffer, or NULL to switch off */
  attn_fwd_tc_set_debug((long long*)device_buf);
  attn_bwd_ws_set_debug((long long*)device_buf);
  return VRR_OK;
}
int vrr_set_option(const char* name, int value) {
  if (!name) return VRR_ERR_INVALID_ARG;
  if (!strcmp(name, "simt_gemm_tile")) { gemm_simt_set_tile(value); return VRR_OK; }
  if (!strcmp(name, "ln_reg")) { layernorm_set_option(0, value); return VRR_OK; }
  if (!strcmp(name, "ln_bwd_minb")) { layernorm_set_option(1, value); return VRR_OK; }
  set_error("vrr_set_option: unknown option '%s'", name);
  return VRR_ERR_INVALID_ARG;
}

size_t vrr_patch_embed_workspace_bytes(int B, int C, int Hi, int Wi, int P, int E, int dtype) {
  if (!is16(dtype) || P <= 0 || !patch_embed_tc_supported(B, C, Hi, Wi, P, E)) return 0;
  return patch_embed_tc_workspace_bytes(B, C, Hi, Wi, P);
}

int vrr_patch_embed_fwd(const void* images, const void* weight, const void* bias, const void* cls_token,
                        const void* pos_embed, void* tokens, void* workspace, size_t workspace_bytes, int B, int C,
                        int Hi, int Wi, int P, int E, int img_dtype, int dtype, int tok_dtype, void* stream) {
  return vrr_patch_embed_fwd_prefix(images, weight, bias, cls_token, 1, pos_embed, tokens, workspace, workspace_bytes, B, C,
                                    Hi, Wi, P, E, img_dtype, dtype, tok_dtype, stream);
}

int vrr_patch_embed_fwd_prefix(const void* images, const void* weight, const void* bias, const void* prefix_tokens,
                               int n_prefix, const void* pos_embed, void* tokens, void* workspace, size_t workspace_bytes,
                               int B, int C, int Hi, int Wi, int P, int E, int img_dtype, int dtype, int tok_dtype,
                               void* stream) {
  VRR_REQUIRE(images && weight && bias && prefix_tokens && tokens, VRR_ERR_INVALID_ARG, "patch_embed_fwd: NULL pointer");
  VRR_REQUIRE(dtype_ok(dtype) && dtype_ok(tok_dtype) && dtype_ok(img_dtype) && no_mix(img_dtype, dtype, tok_dtype),
              VRR_ERR_INVALID_ARG, "patch_embed_fwd: bad dtype %d/%d/%d", img_dtype, dtype, tok_dtype);
  VRR_REQUIRE(B > 0 && C > 0 && P > 0 && E > 0 && Hi >= P && Wi >= P, VRR_ERR_INVALID_ARG,
              "patch_embed_fwd: bad sizes B=%d C=%d Hi=%d Wi=%d P=%d E=%d", B, C, Hi, Wi, P, E);
  const int Np = (Hi / P) * (Wi / P);
  VRR_REQUIRE(prefix_ok(n_prefix, Np + (long long)n_prefix, B, E), VRR_ERR_INVALID_ARG,
              "patch_embed_fwd: n_prefix %d must lie in [1, N] (N = n_prefix + %d patches)", n_prefix, Np);
  if (int rc = require_device()) return rc;
  const int impl = g_impl.load();
  if (is16(dtype) && impl != VRR_IMPL_SIMT && patch_embed_tc_supported(B, C, Hi, Wi, P, E)) {
    const size_t need = patch_embed_tc_workspace_bytes(B, C, Hi, Wi, P);
    VRR_REQUIRE(workspace && workspace_bytes >= need, VRR_ERR_WORKSPACE,
                "patch_embed_fwd: workspace %zu < %zu bytes (vrr_patch_embed_workspace_bytes)", workspace_bytes, need);
    VRR_REQUIRE(((uintptr_t)workspace & 255) == 0, VRR_ERR_INVALID_ARG, "patch_embed_fwd: workspace must be 256-byte aligned");
    VRR_COUNT_FAMILY(VRR_IMPL_TCGEN05);
    if (int rc = patch_embed_fwd_tc(images, weight, bias, pos_embed, tokens, workspace, B, C, Hi, Wi, P, E, n_prefix,
                                    img_dtype, dtype, tok_dtype, (cudaStream_t)stream))
      return rc;
    return patch_prefix_rows(tokens, prefix_tokens, B, Np, E, n_prefix, tok_dtype, (cudaStream_t)stream);
  }
  VRR_REQUIRE(impl != VRR_IMPL_TCGEN05 || !is16(dtype), VRR_ERR_UNSUPPORTED,
              "patch_embed_fwd: tcgen05 kernel forced but shape unsupported (P %% 8, C*P*P %% 64, E %% 64)");
  VRR_COUNT_FAMILY(VRR_IMPL_SIMT);
  return patch_embed_fwd_simt(images, weight, bias, prefix_tokens, pos_embed, tokens, B, C, Hi, Wi, P, E, n_prefix,
                              img_dtype, dtype, tok_dtype, (cudaStream_t)stream);
}

int vrr_patch_unfold(const void* images, void* out, int B, int C, int Hi, int Wi, int P, int img_dtype, void* stream) {
  VRR_REQUIRE(images && out, VRR_ERR_INVALID_ARG, "patch_unfold: NULL pointer");
  VRR_REQUIRE(img_dtype == VRR_F32 || img_dtype == VRR_BF16, VRR_ERR_INVALID_ARG, "patch_unfold: bad dtype %d", img_dtype);
  VRR_REQUIRE(B > 0 && C > 0 && P > 0 && Hi >= P && Wi >= P, VRR_ERR_INVALID_ARG, "patch_unfold: bad sizes");
  if (int rc = require_device()) return rc;
  return patch_unfold(images, out, B, C, Hi, Wi, P, img_dtype, VRR_BF16, (cudaStream_t)stream);
}

int vrr_patch_unfold_ex(const void* images, void* out, int B, int C, int Hi, int Wi, int P, int img_dtype, int out_dtype,
                        void* stream) {
  VRR_REQUIRE(images && out, VRR_ERR_INVALID_ARG, "patch_unfold_ex: NULL pointer");
  VRR_REQUIRE(is16(out_dtype) && (img_dtype == VRR_F32 || img_dtype == out_dtype), VRR_ERR_INVALID_ARG,
              "patch_unfold_ex: bad dtype %d -> %d", img_dtype, out_dtype);
  VRR_REQUIRE(B > 0 && C > 0 && P > 0 && Hi >= P && Wi >= P, VRR_ERR_INVALID_ARG, "patch_unfold_ex: bad sizes");
  if (int rc = require_device()) return rc;
  return patch_unfold(images, out, B, C, Hi, Wi, P, img_dtype, out_dtype, (cudaStream_t)stream);
}

int vrr_patch_embed_bwd(const void* images, const void* d_tokens, void* d_weight, void* d_bias, void* d_cls,
                        void* d_pos, int B, int C, int Hi, int Wi, int P, int E, int img_dtype, int dtype,
                        int tok_dtype, void* stream) {
  return vrr_patch_embed_bwd_prefix(images, d_tokens, d_weight, d_bias, d_cls, 1, d_pos, B, C, Hi, Wi, P, E, img_dtype,
                                    dtype, tok_dtype, stream);
}

int vrr_patch_embed_bwd_prefix(const void* images, const void* d_tokens, void* d_weight, void* d_bias, void* d_prefix,
                               int n_prefix, void* d_pos, int B, int C, int Hi, int Wi, int P, int E, int img_dtype,
                               int dtype, int tok_dtype, void* stream) {
  VRR_REQUIRE(images && d_tokens && d_bias && d_prefix, VRR_ERR_INVALID_ARG, "patch_embed_bwd: NULL pointer");
  VRR_REQUIRE(dtype_ok(dtype) && dtype_ok(tok_dtype) && dtype_ok(img_dtype) && no_mix(img_dtype, dtype, tok_dtype),
              VRR_ERR_INVALID_ARG, "patch_embed_bwd: bad dtype %d/%d/%d", img_dtype, dtype, tok_dtype);
  VRR_REQUIRE(B > 0 && C > 0 && P > 0 && E > 0 && Hi >= P && Wi >= P, VRR_ERR_INVALID_ARG,
              "patch_embed_bwd: bad sizes");
  const int Np = (Hi / P) * (Wi / P);
  VRR_REQUIRE(prefix_ok(n_prefix, Np + (long long)n_prefix, B, E), VRR_ERR_INVALID_ARG,
              "patch_embed_bwd: n_prefix %d must lie in [1, N] (N = n_prefix + %d patches)", n_prefix, Np);
  if (int rc = require_device()) return rc;
  return patch_embed_bwd_simt(images, d_tokens, (float*)d_weight, (float*)d_bias, (float*)d_prefix, (float*)d_pos, B,
                              C, Hi, Wi, P, E, n_prefix, img_dtype, dtype, tok_dtype, (cudaStream_t)stream);
}

int vrr_qkv_rope_fwd(const void* x, const void* w_qkv, const float* cos_tab, const float* sin_tab, void* planes,
                     int B, int N, int E, int H, int rope_mode, int dtype, void* stream) {
  return vrr_qkv_rope_fwd_packed(x, w_qkv, cos_tab, sin_tab, nullptr, planes, B, N, E, H, rope_mode, dtype, stream);
}

int vrr_rope_pack_tables(const float* cos_tab, const float* sin_tab, float* packed, int heads, int rows, int half_dim,
                         void* stream) {
  VRR_REQUIRE(cos_tab && sin_tab && packed, VRR_ERR_INVALID_ARG, "rope_pack_tables: NULL pointer");
  VRR_REQUIRE(heads > 0 && rows > 0 && half_dim > 0, VRR_ERR_INVALID_ARG, "rope_pack_tables: bad sizes");
  if (int rc = require_device()) return rc;
  return rope_pack_tables(cos_tab, sin_tab, packed, heads, rows, half_dim, (cudaStream_t)stream);
}

int vrr_qkv_rope_fwd_packed(const void* x, const void* w_qkv, const float* cos_tab, const float* sin_tab,
                            const float* packed, void* planes, int B, int N, int E, int H, int rope_mode, int dtype,
                            void* stream) {
  return vrr_qkv_rope_fwd_prefix(x, w_qkv, cos_tab, sin_tab, packed, planes, B, N, E, H, 1, rope_mode, dtype, stream);
}

int vrr_qkv_rope_fwd_prefix(const void* x, const void* w_qkv, const float* cos_tab, const float* sin_tab,
                            const float* packed, void* planes, int B, int N, int E, int H, int n_prefix, int rope_mode,
                            int dtype, void* stream) {
  VRR_REQUIRE(x && w_qkv && planes, VRR_ERR_INVALID_ARG, "qkv_rope_fwd: NULL pointer");
  VRR_REQUIRE(dtype_ok(dtype), VRR_ERR_INVALID_ARG, "qkv_rope_fwd: bad dtype %d", dtype);
  VRR_REQUIRE(rope_mode >= VRR_ROPE_NONE && rope_mode <= VRR_ROPE_MIXED, VRR_ERR_INVALID_ARG,
              "qkv_rope_fwd: bad rope_mode %d", rope_mode);
  VRR_REQUIRE(rope_mode == VRR_ROPE_NONE || (cos_tab && sin_tab), VRR_ERR_INVALID_ARG,
              "qkv_rope_fwd: cos/sin required for rope_mode %d", rope_mode);
  VRR_REQUIRE(B > 0 && N > 0 && H > 0 && E > 0 && E % H == 0, VRR_ERR_INVALID_ARG, "qkv_rope_fwd: bad sizes");
  VRR_REQUIRE(n_prefix >= 1 && n_prefix <= N, VRR_ERR_INVALID_ARG, "qkv_rope_fwd: n_prefix %d must lie in [1, N = %d]",
              n_prefix, N);
  VRR_REQUIRE(dh_ok(E / H), VRR_ERR_UNSUPPORTED, "qkv_rope_fwd: head dim %d unsupported (16, 32, 64)", E / H);
  if (int rc = require_device()) return rc;
  const int impl = g_impl.load();
  if (is16(dtype) && impl != VRR_IMPL_SIMT && qkv_rope_fwd_tc_supported(B, N, E, H)) {
    VRR_COUNT_FAMILY(VRR_IMPL_TCGEN05);
    return qkv_rope_fwd_tc2(x, w_qkv, cos_tab, sin_tab, packed, planes, B, N, E, H, n_prefix, rope_mode, dtype,
                            (cudaStream_t)stream);
  }
  VRR_REQUIRE(impl != VRR_IMPL_TCGEN05, VRR_ERR_UNSUPPORTED,
              "qkv_rope_fwd: tcgen05 kernel forced but shape/dtype unsupported (bf16 or fp16, Dh=64, E%%64==0)");
  VRR_COUNT_FAMILY(VRR_IMPL_SIMT);
  return qkv_rope_fwd_simt(x, w_qkv, cos_tab, sin_tab, planes, B, N, E, H, n_prefix, rope_mode, dtype, (cudaStream_t)stream);
}

int vrr_qkv_rope_bwd(const void* d_planes, const void* planes, const float* cos_tab, const float* sin_tab,
                     void* d_qkv, float* d_cos, float* d_sin, int B, int N, int E, int H, int rope_mode,
                     int dtype, void* stream) {
  return vrr_qkv_rope_bwd_prefix(d_planes, planes, cos_tab, sin_tab, d_qkv, d_cos, d_sin, B, N, E, H, 1, rope_mode, dtype,
                                 stream);
}

int vrr_qkv_rope_bwd_prefix(const void* d_planes, const void* planes, const float* cos_tab, const float* sin_tab,
                            void* d_qkv, float* d_cos, float* d_sin, int B, int N, int E, int H, int n_prefix,
                            int rope_mode, int dtype, void* stream) {
  VRR_REQUIRE(d_planes && planes && d_qkv, VRR_ERR_INVALID_ARG, "qkv_rope_bwd: NULL pointer");
  VRR_REQUIRE(dtype_ok(dtype), VRR_ERR_INVALID_ARG, "qkv_rope_bwd: bad dtype %d", dtype);
  VRR_REQUIRE(rope_mode >= VRR_ROPE_NONE && rope_mode <= VRR_ROPE_MIXED, VRR_ERR_INVALID_ARG,
              "qkv_rope_bwd: bad rope_mode %d", rope_mode);
  VRR_REQUIRE(rope_mode == VRR_ROPE_NONE || (cos_tab && sin_tab), VRR_ERR_INVALID_ARG,
              "qkv_rope_bwd: cos/sin required");
  VRR_REQUIRE((d_cos == nullptr) == (d_sin == nullptr), VRR_ERR_INVALID_ARG,
              "qkv_rope_bwd: d_cos and d_sin must both be given or both NULL");
  VRR_REQUIRE(B > 0 && N > 0 && H > 0 && E > 0 && E % H == 0 && dh_ok(E / H), VRR_ERR_INVALID_ARG,
              "qkv_rope_bwd: bad sizes");
  VRR_REQUIRE(n_prefix >= 1 && n_prefix <= N, VRR_ERR_INVALID_ARG, "qkv_rope_bwd: n_prefix %d must lie in [1, N = %d]",
              n_prefix, N);
  if (int rc = require_device()) return rc;
  return qkv_rope_bwd(d_planes, planes, cos_tab, sin_tab, d_qkv, d_cos, d_sin, B, N, E, H, n_prefix, rope_mode, dtype,
                      (cudaStream_t)stream);
}

int vrr_qkv_rope_norm_fwd(const void* x, const void* w_qkv, const float* cos_tab, const float* sin_tab, const float* packed,
                          void* planes, int B, int N, int E, int H, int n_prefix, int rope_mode, int dtype, const float* qn_w,
                          const float* qn_b, const float* kn_w, const float* kn_b, float eps, void* qk_pre, float* qk_stats,
                          void* stream) {
  VRR_REQUIRE(x && w_qkv && planes, VRR_ERR_INVALID_ARG, "qkv_rope_norm_fwd: NULL pointer");
  VRR_REQUIRE(qn_w && qn_b && kn_w && kn_b, VRR_ERR_INVALID_ARG, "qkv_rope_norm_fwd: q_norm / k_norm weight and bias are required");
  VRR_REQUIRE((qk_pre == nullptr) == (qk_stats == nullptr), VRR_ERR_INVALID_ARG,
              "qkv_rope_norm_fwd: qk_pre and qk_stats must both be given or both NULL");
  VRR_REQUIRE(eps >= 0.f, VRR_ERR_INVALID_ARG, "qkv_rope_norm_fwd: eps must be >= 0");
  VRR_REQUIRE(dtype_ok(dtype), VRR_ERR_INVALID_ARG, "qkv_rope_norm_fwd: bad dtype %d", dtype);
  VRR_REQUIRE(rope_mode >= VRR_ROPE_NONE && rope_mode <= VRR_ROPE_MIXED, VRR_ERR_INVALID_ARG,
              "qkv_rope_norm_fwd: bad rope_mode %d", rope_mode);
  VRR_REQUIRE(rope_mode == VRR_ROPE_NONE || (cos_tab && sin_tab), VRR_ERR_INVALID_ARG,
              "qkv_rope_norm_fwd: cos/sin required for rope_mode %d", rope_mode);
  VRR_REQUIRE(B > 0 && N > 0 && H > 0 && E > 0 && E % H == 0, VRR_ERR_INVALID_ARG, "qkv_rope_norm_fwd: bad sizes");
  VRR_REQUIRE(n_prefix >= 1 && n_prefix <= N, VRR_ERR_INVALID_ARG,
              "qkv_rope_norm_fwd: n_prefix %d must lie in [1, N = %d]", n_prefix, N);
  VRR_REQUIRE(dh_ok(E / H), VRR_ERR_UNSUPPORTED, "qkv_rope_norm_fwd: head dim %d unsupported (16, 32, 64)", E / H);
  if (int rc = require_device()) return rc;
  const QkNormArgs qn = {qn_w, qn_b, kn_w, kn_b, eps, qk_pre, qk_stats};
  const int impl = g_impl.load();
  if (is16(dtype) && impl != VRR_IMPL_SIMT && qkv_rope_fwd_tc_supported(B, N, E, H)) {
    VRR_COUNT_FAMILY(VRR_IMPL_TCGEN05);
    return qkv_rope_fwd_tc2(x, w_qkv, cos_tab, sin_tab, packed, planes, B, N, E, H, n_prefix, rope_mode, dtype,
                            (cudaStream_t)stream, &qn);
  }
  VRR_REQUIRE(impl != VRR_IMPL_TCGEN05, VRR_ERR_UNSUPPORTED,
              "qkv_rope_norm_fwd: tcgen05 kernel forced but shape/dtype unsupported (bf16 or fp16, Dh=64, E%%64==0)");
  VRR_COUNT_FAMILY(VRR_IMPL_SIMT);
  return qkv_rope_fwd_simt(x, w_qkv, cos_tab, sin_tab, planes, B, N, E, H, n_prefix, rope_mode, dtype, (cudaStream_t)stream,
                           &qn);
}

int vrr_qkv_rope_norm_bwd(const void* d_planes, const void* qk_pre, const float* qk_stats, const float* cos_tab,
                          const float* sin_tab, const float* qn_w, const float* qn_b, const float* kn_w, const float* kn_b,
                          void* d_qkv, float* d_cos, float* d_sin, float* d_qn_w, float* d_qn_b, float* d_kn_w,
                          float* d_kn_b, int B, int N, int E, int H, int n_prefix, int rope_mode, int dtype, void* stream) {
  VRR_REQUIRE(d_planes && qk_pre && qk_stats && d_qkv, VRR_ERR_INVALID_ARG, "qkv_rope_norm_bwd: NULL pointer");
  VRR_REQUIRE(qn_w && qn_b && kn_w && kn_b, VRR_ERR_INVALID_ARG, "qkv_rope_norm_bwd: q_norm / k_norm weight and bias are required");
  VRR_REQUIRE((d_cos == nullptr) == (d_sin == nullptr), VRR_ERR_INVALID_ARG,
              "qkv_rope_norm_bwd: d_cos and d_sin must both be given or both NULL");
  const int n_grads = (d_qn_w != nullptr) + (d_qn_b != nullptr) + (d_kn_w != nullptr) + (d_kn_b != nullptr);
  VRR_REQUIRE(n_grads == 0 || n_grads == 4, VRR_ERR_INVALID_ARG,
              "qkv_rope_norm_bwd: d_qn_w, d_qn_b, d_kn_w and d_kn_b must all be given or all NULL");
  VRR_REQUIRE(dtype_ok(dtype), VRR_ERR_INVALID_ARG, "qkv_rope_norm_bwd: bad dtype %d", dtype);
  VRR_REQUIRE(rope_mode >= VRR_ROPE_NONE && rope_mode <= VRR_ROPE_MIXED, VRR_ERR_INVALID_ARG,
              "qkv_rope_norm_bwd: bad rope_mode %d", rope_mode);
  VRR_REQUIRE(rope_mode == VRR_ROPE_NONE || (cos_tab && sin_tab), VRR_ERR_INVALID_ARG, "qkv_rope_norm_bwd: cos/sin required");
  VRR_REQUIRE(B > 0 && N > 0 && H > 0 && E > 0 && E % H == 0 && dh_ok(E / H), VRR_ERR_INVALID_ARG,
              "qkv_rope_norm_bwd: bad sizes");
  VRR_REQUIRE(n_prefix >= 1 && n_prefix <= N, VRR_ERR_INVALID_ARG,
              "qkv_rope_norm_bwd: n_prefix %d must lie in [1, N = %d]", n_prefix, N);
  if (int rc = require_device()) return rc;
  const QkNormArgs qn = {qn_w, qn_b, kn_w, kn_b, 0.f, const_cast<void*>(qk_pre), const_cast<float*>(qk_stats)};
  const QkNormGrads gr = {d_qn_w, d_qn_b, d_kn_w, d_kn_b};
  return qkv_rope_norm_bwd(d_planes, qn, cos_tab, sin_tab, d_qkv, d_cos, d_sin, gr, B, N, E, H, n_prefix, rope_mode, dtype,
                           (cudaStream_t)stream);
}

int vrr_rope_apply(const void* q_in, const void* k_in, const float* cos_tab, const float* sin_tab, void* q_out,
                   void* k_out, int B, int H, int Nr, int Dh, int rope_mode, int inverse, int dtype,
                   void* stream) {
  VRR_REQUIRE(q_in && k_in && cos_tab && sin_tab && q_out && k_out, VRR_ERR_INVALID_ARG, "rope_apply: NULL pointer");
  VRR_REQUIRE(dtype_ok(dtype), VRR_ERR_INVALID_ARG, "rope_apply: bad dtype %d", dtype);
  VRR_REQUIRE(rope_mode == VRR_ROPE_AXIAL || rope_mode == VRR_ROPE_MIXED, VRR_ERR_INVALID_ARG,
              "rope_apply: bad rope_mode %d", rope_mode);
  VRR_REQUIRE(B > 0 && H > 0 && Nr > 0 && Dh > 0 && Dh % 2 == 0, VRR_ERR_INVALID_ARG, "rope_apply: bad sizes");
  if (int rc = require_device()) return rc;
  return rope_apply(q_in, k_in, cos_tab, sin_tab, q_out, k_out, B, H, Nr, Dh, rope_mode, inverse, dtype,
                    (cudaStream_t)stream);
}

int vrr_rope_table_grad(const void* q_in, const void* k_in, const void* dq, const void* dk, float* d_cos,
                        float* d_sin, int B, int H, int Nr, int Dh, int rope_mode, int dtype, void* stream) {
  VRR_REQUIRE(q_in && k_in && dq && dk && d_cos && d_sin, VRR_ERR_INVALID_ARG, "rope_table_grad: NULL pointer");
  VRR_REQUIRE(dtype_ok(dtype), VRR_ERR_INVALID_ARG, "rope_table_grad: bad dtype %d", dtype);
  VRR_REQUIRE(rope_mode == VRR_ROPE_AXIAL || rope_mode == VRR_ROPE_MIXED, VRR_ERR_INVALID_ARG,
              "rope_table_grad: bad rope_mode %d", rope_mode);
  VRR_REQUIRE(B > 0 && H > 0 && Nr > 0 && Dh > 0 && Dh % 2 == 0, VRR_ERR_INVALID_ARG, "rope_table_grad: bad sizes");
  if (int rc = require_device()) return rc;
  return rope_table_grad(q_in, k_in, dq, dk, d_cos, d_sin, B, H, Nr, Dh, rope_mode, dtype, (cudaStream_t)stream);
}

int vrr_gemm(const void* a, const void* b, void* c, int M, int N, int K, int trans_a, int trans_b, int dtype,
             int c_dtype, void* stream) {
  VRR_REQUIRE(a && b && c, VRR_ERR_INVALID_ARG, "gemm: NULL pointer");
  VRR_REQUIRE(M > 0 && N > 0 && K > 0, VRR_ERR_INVALID_ARG, "gemm: bad sizes");
  VRR_REQUIRE(dtype_ok(dtype) && dtype_ok(c_dtype) && no_mix(dtype, c_dtype), VRR_ERR_INVALID_ARG, "gemm: bad dtype %d/%d",
              dtype, c_dtype);
  if (int rc = require_device()) return rc;
  return gemm_simt(a, b, c, M, N, K, trans_a, trans_b, dtype, c_dtype, (cudaStream_t)stream);
}

int vrr_gemm_ex(const void* a, const void* b, void* c, void* c2, const float* bias, int M, int N, int K, int trans_a,
                int trans_b, int dtype, int c_dtype, int epilogue, int accumulate, void* stream) {
  VRR_REQUIRE(a && b && c, VRR_ERR_INVALID_ARG, "gemm_ex: NULL pointer");
  VRR_REQUIRE(M > 0 && N > 0 && K > 0, VRR_ERR_INVALID_ARG, "gemm_ex: bad sizes");
  VRR_REQUIRE(dtype_ok(dtype) && dtype_ok(c_dtype) && no_mix(dtype, c_dtype), VRR_ERR_INVALID_ARG, "gemm_ex: bad dtype %d/%d",
              dtype, c_dtype);
  VRR_REQUIRE(epilogue >= VRR_EPI_NONE && epilogue <= VRR_EPI_BIAS_GELU_ACT, VRR_ERR_INVALID_ARG, "gemm_ex: bad epilogue %d",
              epilogue);
  VRR_REQUIRE(epilogue == VRR_EPI_NONE || epilogue == VRR_EPI_MUL || bias, VRR_ERR_INVALID_ARG,
              "gemm_ex: the bias epilogues need `bias`");
  VRR_REQUIRE(epilogue < VRR_EPI_BIAS_GELU || epilogue == VRR_EPI_BIAS_GELU_ACT || c2, VRR_ERR_INVALID_ARG,
              "gemm_ex: the two-output GELU epilogues and MUL need `c2`");
  if (int rc = require_device()) return rc;
  const int impl = g_impl.load();
  // TMA needs 16-byte aligned base addresses: a view at an odd offset into a larger buffer runs the SIMT kernel
  const bool uses_c2 = epilogue == VRR_EPI_BIAS_GELU || epilogue == VRR_EPI_BIAS_GELU_GRAD || epilogue == VRR_EPI_MUL;
  const bool uses_bias = epilogue != VRR_EPI_NONE && epilogue != VRR_EPI_MUL;
  const bool aligned = gemm_ptrs_aligned16(a, b, c, uses_c2 ? c2 : nullptr, uses_bias ? bias : nullptr);
  if (is16(dtype) && impl != VRR_IMPL_SIMT && aligned && gemm_tc_supported(M, N, K, trans_a, trans_b, dtype, c_dtype, epilogue)) {
    VRR_COUNT_FAMILY(VRR_IMPL_TCGEN05);
    return gemm_tc(a, b, c, c2, bias, M, N, K, trans_a, trans_b, dtype, c_dtype, epilogue, accumulate, (cudaStream_t)stream);
  }
  VRR_REQUIRE(impl != VRR_IMPL_TCGEN05 || !is16(dtype), VRR_ERR_UNSUPPORTED,
              "gemm_ex: tcgen05 kernel forced but M=%d N=%d K=%d (trans %d/%d) needs N %% 8 == 0, K %% 8 == 0 "
              "(M %% 8 == 0 when trans_a) and 16-byte aligned pointers", M, N, K, trans_a, trans_b);
  VRR_REQUIRE(!accumulate, VRR_ERR_UNSUPPORTED, "gemm_ex: accumulate is implemented by the tcgen05 kernel only");
  VRR_COUNT_FAMILY(VRR_IMPL_SIMT);
  if (epilogue == VRR_EPI_MUL) {
    VRR_REQUIRE(c_dtype == dtype, VRR_ERR_UNSUPPORTED, "gemm_ex (SIMT): the MUL epilogue needs c_dtype == dtype");
    if (int rc = gemm_simt(a, b, c, M, N, K, trans_a, trans_b, dtype, c_dtype, (cudaStream_t)stream)) return rc;
    return mul_inplace(c, c2, (size_t)M * N, c_dtype, (cudaStream_t)stream);
  }
  if (epilogue != VRR_EPI_NONE) {
    VRR_REQUIRE(c_dtype == dtype, VRR_ERR_UNSUPPORTED, "gemm_ex (SIMT): the bias epilogues need c_dtype == dtype");
    if (epilogue == VRR_EPI_BIAS_GELU_GRAD) {  // (h, gelu(h)) into (c2, c), then c2 <- gelu'(h)
      if (int rc = gemm_simt_bias(a, b, c2, c, bias, M, N, K, trans_a, trans_b, dtype, 1, (cudaStream_t)stream)) return rc;
      return gelu_grad_inplace(c2, (size_t)M * N, dtype, (cudaStream_t)stream);
    }
    return gemm_simt_bias(a, b, c, c2, bias, M, N, K, trans_a, trans_b, dtype,
                          epilogue == VRR_EPI_BIAS_GELU ? 1 : (epilogue == VRR_EPI_BIAS_GELU_ACT ? 2 : 0), (cudaStream_t)stream);
  }
  return gemm_simt(a, b, c, M, N, K, trans_a, trans_b, dtype, c_dtype, (cudaStream_t)stream);
}

int vrr_gemm_ex_drop(const void* a, const void* b, void* c, void* c2, const float* bias, int M, int N, int K,
                     int trans_a, int trans_b, int dtype, int c_dtype, int epilogue, int accumulate,
                     const vrr_drop_desc* drop, void* stream) {
  VRR_REQUIRE(epilogue == VRR_EPI_BIAS_GELU_GRAD || epilogue == VRR_EPI_BIAS_GELU_ACT, VRR_ERR_INVALID_ARG,
              "gemm_ex_drop: epilogue %d (only BIAS_GELU_GRAD and BIAS_GELU_ACT take dropout)", epilogue);
  VRR_REQUIRE(!drop || drop->p_path == 0.f, VRR_ERR_INVALID_ARG, "gemm_ex_drop: p_path must be 0");
  DropView dv = {};
  bool active = false;
  if (int rc = drop_view(drop, M, N, &dv, &active)) return rc;
  if (!active) return vrr_gemm_ex(a, b, c, c2, bias, M, N, K, trans_a, trans_b, dtype, c_dtype, epilogue, accumulate, stream);
  VRR_REQUIRE(a && b && c && bias, VRR_ERR_INVALID_ARG, "gemm_ex_drop: NULL pointer");
  VRR_REQUIRE(epilogue == VRR_EPI_BIAS_GELU_ACT || c2, VRR_ERR_INVALID_ARG, "gemm_ex_drop: BIAS_GELU_GRAD needs `c2`");
  VRR_REQUIRE(M > 0 && N > 0 && K > 0, VRR_ERR_INVALID_ARG, "gemm_ex_drop: bad sizes");
  VRR_REQUIRE(dtype_ok(dtype) && c_dtype == dtype, VRR_ERR_INVALID_ARG, "gemm_ex_drop: bad dtype %d/%d (C has the operands' type)",
              dtype, c_dtype);
  VRR_REQUIRE(!accumulate, VRR_ERR_UNSUPPORTED, "gemm_ex_drop: accumulate needs an fp32 C");
  if (int rc = require_device()) return rc;
  const int impl = g_impl.load();
  const bool grad = epilogue == VRR_EPI_BIAS_GELU_GRAD;
  const bool aligned = gemm_ptrs_aligned16(a, b, c, grad ? c2 : nullptr, bias);
  const bool tc_ok = is16(dtype) && aligned && trans_a == 0 && trans_b == 1 &&
                     gemm_tc_supported(M, N, K, trans_a, trans_b, dtype, c_dtype, epilogue);
  if (impl != VRR_IMPL_SIMT && tc_ok) {
    VRR_COUNT_FAMILY(VRR_IMPL_TCGEN05);
    return gemm_tc_drop(a, b, c, grad ? c2 : nullptr, bias, M, N, K, dtype, epilogue, dv, (cudaStream_t)stream);
  }
  VRR_REQUIRE(impl != VRR_IMPL_TCGEN05 || !is16(dtype), VRR_ERR_UNSUPPORTED,
              "gemm_ex_drop: tcgen05 kernel forced but the case needs trans_a 0, trans_b 1, N %% 8 == 0, K %% 8 == 0 "
              "and 16-byte aligned pointers");
  VRR_COUNT_FAMILY(VRR_IMPL_SIMT);
  if (grad) {  // (h, gelu(h)) into (c2, c); then c <- T(c f), c2 <- T(T(gelu'(h)) f)
    if (int rc = gemm_simt_bias(a, b, c2, c, bias, M, N, K, trans_a, trans_b, dtype, 1, (cudaStream_t)stream)) return rc;
  } else {
    if (int rc = gemm_simt_bias(a, b, c, nullptr, bias, M, N, K, trans_a, trans_b, dtype, 2, (cudaStream_t)stream)) return rc;
  }
  return drop_gelu_inplace(c, grad ? c2 : nullptr, M, N, dtype, dv, (cudaStream_t)stream);
}

int vrr_gemm_mul_colsum(const void* a, const void* b, void* c, const void* mul, float* col_sums, int M, int N, int K,
                        int trans_a, int trans_b, int dtype, void* stream) {
  VRR_REQUIRE(a && b && c && mul && col_sums, VRR_ERR_INVALID_ARG, "gemm_mul_colsum: NULL pointer");
  VRR_REQUIRE(M > 0 && N > 0 && K > 0 && N % 4 == 0, VRR_ERR_INVALID_ARG, "gemm_mul_colsum: bad sizes (N %% 4 == 0)");
  VRR_REQUIRE(dtype_ok(dtype), VRR_ERR_INVALID_ARG, "gemm_mul_colsum: bad dtype %d", dtype);
  if (int rc = require_device()) return rc;
  const int impl = g_impl.load();
  if (is16(dtype) && impl != VRR_IMPL_SIMT && gemm_ptrs_aligned16(a, b, c, mul, nullptr) &&
      gemm_tc_supported(M, N, K, trans_a, trans_b, dtype, dtype, VRR_EPI_MUL)) {
    VRR_COUNT_FAMILY(VRR_IMPL_TCGEN05);
    VRR_CUDA(cudaMemsetAsync(col_sums, 0, (size_t)N * sizeof(float), (cudaStream_t)stream));
    return gemm_tc(a, b, c, const_cast<void*>(mul), nullptr, M, N, K, trans_a, trans_b, dtype, dtype, VRR_EPI_MUL, 0,
                   (cudaStream_t)stream, col_sums);
  }
  if (int rc = vrr_gemm_ex(a, b, c, const_cast<void*>(mul), nullptr, M, N, K, trans_a, trans_b, dtype, dtype, VRR_EPI_MUL, 0, stream))
    return rc;
  return colsum(c, col_sums, M, N, dtype, (cudaStream_t)stream);
}

// tcgen05 SwiGLU kernels: 16-bit, H and K multiples of 8 (TMA row strides, the 8-column bias / mask groups), pointers
// 16-byte aligned (the value half of aux / dh starts H elements into each row)
static bool swiglu_tc_ok(int dtype, int M, int H, int K, const void* p0, const void* p1, const void* p2, const void* p3,
                         const void* p4) {
  return is16(dtype) && H % 8 == 0 && K % 8 == 0 && (long long)M * 2 * H < (1ll << 40) &&
         ((((uintptr_t)p0 | (uintptr_t)p1 | (uintptr_t)p2 | (uintptr_t)p3 | (uintptr_t)p4)) & 15) == 0;
}

int vrr_gemm_swiglu(const void* x, const void* w1, const float* b1, void* act, void* aux, int M, int H, int K, int dtype,
                    const vrr_drop_desc* drop, void* stream) {
  VRR_REQUIRE(x && w1 && b1 && act, VRR_ERR_INVALID_ARG, "gemm_swiglu: NULL pointer");
  VRR_REQUIRE(M > 0 && H > 0 && K > 0, VRR_ERR_INVALID_ARG, "gemm_swiglu: bad sizes M=%d H=%d K=%d", M, H, K);
  VRR_REQUIRE(dtype_ok(dtype), VRR_ERR_INVALID_ARG, "gemm_swiglu: bad dtype %d", dtype);
  VRR_REQUIRE(!drop || drop->p_path == 0.f, VRR_ERR_INVALID_ARG, "gemm_swiglu: p_path must be 0");
  DropView dv = {};
  bool active = false;
  if (int rc = drop_view(drop, M, H, &dv, &active)) return rc;
  if (int rc = require_device()) return rc;
  const int impl = g_impl.load();
  if (impl != VRR_IMPL_SIMT && swiglu_tc_ok(dtype, M, H, K, x, w1, b1, act, aux)) {
    VRR_COUNT_FAMILY(VRR_IMPL_TCGEN05);
    return gemm_tc_swiglu(x, w1, b1, act, aux, M, H, K, dtype, active ? &dv : nullptr, (cudaStream_t)stream);
  }
  VRR_REQUIRE(impl != VRR_IMPL_TCGEN05 || !is16(dtype), VRR_ERR_UNSUPPORTED,
              "gemm_swiglu: tcgen05 kernel forced but M=%d H=%d K=%d needs H %% 8 == 0, K %% 8 == 0 and 16-byte aligned "
              "pointers", M, H, K);
  VRR_COUNT_FAMILY(VRR_IMPL_SIMT);
  return swiglu_simt(x, w1, b1, act, aux, M, H, K, dtype, active ? &dv : nullptr, (cudaStream_t)stream);
}

int vrr_gemm_swiglu_bwd(const void* dy, const void* w2, const void* aux, void* dh, float* db1, int M, int H, int K, int dtype,
                        void* stream) {
  VRR_REQUIRE(dy && w2 && aux && dh && db1, VRR_ERR_INVALID_ARG, "gemm_swiglu_bwd: NULL pointer");
  VRR_REQUIRE(M > 0 && H > 0 && K > 0 && H % 2 == 0, VRR_ERR_INVALID_ARG,
              "gemm_swiglu_bwd: bad sizes M=%d H=%d K=%d (H %% 2 == 0)", M, H, K);
  VRR_REQUIRE(dtype_ok(dtype), VRR_ERR_INVALID_ARG, "gemm_swiglu_bwd: bad dtype %d", dtype);
  if (int rc = require_device()) return rc;
  const int impl = g_impl.load();
  if (impl != VRR_IMPL_SIMT && swiglu_tc_ok(dtype, M, H, K, dy, w2, aux, dh, db1)) {
    VRR_COUNT_FAMILY(VRR_IMPL_TCGEN05);
    return gemm_tc_swiglu_bwd(dy, w2, aux, dh, db1, M, H, K, dtype, (cudaStream_t)stream);
  }
  VRR_REQUIRE(impl != VRR_IMPL_TCGEN05 || !is16(dtype), VRR_ERR_UNSUPPORTED,
              "gemm_swiglu_bwd: tcgen05 kernel forced but M=%d H=%d K=%d needs H %% 8 == 0, K %% 8 == 0 and 16-byte "
              "aligned pointers", M, H, K);
  VRR_COUNT_FAMILY(VRR_IMPL_SIMT);
  if (int rc = swiglu_bwd_simt(dy, w2, aux, dh, M, H, K, dtype, (cudaStream_t)stream)) return rc;
  return colsum(dh, db1, M, 2 * H, dtype, (cudaStream_t)stream);
}

int vrr_attn_fwd(const void* planes, const vrr_bias_desc* bias, void* out, float* lse, int B, int H, int N,
                 int Dh, float scale, int dtype, void* stream) {
  VRR_REQUIRE(planes && out && lse, VRR_ERR_INVALID_ARG, "attn_fwd: NULL pointer");
  VRR_REQUIRE(dtype_ok(dtype), VRR_ERR_INVALID_ARG, "attn_fwd: bad dtype %d", dtype);
  VRR_REQUIRE(B > 0 && H > 0 && N > 0, VRR_ERR_INVALID_ARG, "attn_fwd: bad sizes");
  VRR_REQUIRE(dh_ok(Dh), VRR_ERR_UNSUPPORTED, "attn_fwd: head dim %d unsupported (16, 32, 64)", Dh);
  if (int rc = check_bias(bias, H, N)) return rc;
  if (int rc = require_device()) return rc;
  const int impl = g_impl.load();
  if (is16(dtype) && impl != VRR_IMPL_SIMT && attn_fwd_tc_supported(B, H, N, Dh, bias)) {
    VRR_COUNT_FAMILY(VRR_IMPL_TCGEN05);
    // with a bias, N <= 256: the whole-sequence kernel; otherwise the tiled kernels (four CTAs per SM without bias)
    if (attn_fwd_ws_supported(B, H, N, Dh, bias))
      return attn_fwd_ws(planes, bias, out, lse, B, H, N, Dh, scale, dtype, (cudaStream_t)stream);
    return attn_fwd_tc(planes, bias, out, lse, B, H, N, Dh, scale, dtype, (cudaStream_t)stream);
  }
  VRR_REQUIRE(impl != VRR_IMPL_TCGEN05, VRR_ERR_UNSUPPORTED,
              "attn_fwd: tcgen05 kernel forced but shape/dtype unsupported (bf16 or fp16, Dh=64)");
  VRR_COUNT_FAMILY(VRR_IMPL_SIMT);
  return attn_fwd_simt(planes, bias, out, lse, B, H, N, Dh, scale, dtype, (cudaStream_t)stream);
}

size_t vrr_attn_bwd_workspace_bytes(int B, int H, int N, int Dh, const vrr_bias_desc* bias) {
  (void)Dh;
  size_t delta = (size_t)B * H * N * sizeof(float);
  size_t lut = (size_t)H * (size_t)bias_lut_len(bias, N) * sizeof(float);
  return ((delta + 255) / 256) * 256 + ((lut + 255) / 256) * 256 + 256;
}

int vrr_attn_bwd(const void* planes, const vrr_bias_desc* bias, const void* out, const void* d_out,
                 const float* lse, void* d_planes, float* d_bias_param, void* workspace, size_t workspace_bytes,
                 int B, int H, int N, int Dh, float scale, int dtype, void* stream) {
  VRR_REQUIRE(planes && out && d_out && lse && d_planes && workspace, VRR_ERR_INVALID_ARG, "attn_bwd: NULL pointer");
  VRR_REQUIRE(dtype_ok(dtype), VRR_ERR_INVALID_ARG, "attn_bwd: bad dtype %d", dtype);
  VRR_REQUIRE(B > 0 && H > 0 && N > 0, VRR_ERR_INVALID_ARG, "attn_bwd: bad sizes");
  VRR_REQUIRE(dh_ok(Dh), VRR_ERR_UNSUPPORTED, "attn_bwd: head dim %d unsupported (16, 32, 64)", Dh);
  if (int rc = check_bias(bias, H, N)) return rc;
  const bool has_bias = bias && bias->mode != VRR_BIAS_NONE;
  VRR_REQUIRE(!has_bias || d_bias_param, VRR_ERR_INVALID_ARG, "attn_bwd: d_bias_param required with a bias");
  VRR_REQUIRE(workspace_bytes >= vrr_attn_bwd_workspace_bytes(B, H, N, Dh, bias), VRR_ERR_WORKSPACE,
              "attn_bwd: workspace %zu < %zu bytes", workspace_bytes, vrr_attn_bwd_workspace_bytes(B, H, N, Dh, bias));
  VRR_REQUIRE(((uintptr_t)workspace & 255) == 0, VRR_ERR_INVALID_ARG, "attn_bwd: workspace must be 256-byte aligned");
  if (int rc = require_device()) return rc;
  float* delta = (float*)workspace;
  size_t delta_bytes = (((size_t)B * H * N * sizeof(float) + 255) / 256) * 256;
  float* d_lut = (float*)((char*)workspace + delta_bytes);
  const int impl = g_impl.load();
  if (is16(dtype) && impl != VRR_IMPL_SIMT && attn_bwd_tc2_supported(B, H, N, Dh, bias)) {
    VRR_COUNT_FAMILY(VRR_IMPL_TCGEN05);
    if (attn_bwd_ws_supported(B, H, N, Dh, bias))  // short sequences, no bias: the whole-sequence kernel
      return attn_bwd_ws(planes, out, d_out, lse, d_planes, B, H, N, Dh, scale, dtype, (cudaStream_t)stream);
    return attn_bwd_tc2(planes, bias, out, d_out, lse, d_planes, d_bias_param, delta, B, H, N, Dh, scale, dtype,
                        (cudaStream_t)stream);
  }
  // e.g. polynomial degree > 3 (the tcgen05 kernel keeps 4 power sums per thread): explicit under
  // VRR_IMPL_TCGEN05, and visible to AUTO callers through vrr_family_count(VRR_IMPL_SIMT)
  VRR_REQUIRE(impl != VRR_IMPL_TCGEN05, VRR_ERR_UNSUPPORTED,
              "attn_bwd: tcgen05 kernel forced but shape/dtype unsupported (bf16 or fp16, Dh=64, poly degree <= 3)");
  VRR_COUNT_FAMILY(VRR_IMPL_SIMT);
  return attn_bwd_simt(planes, bias, out, d_out, lse, d_planes, d_bias_param, delta, d_lut, B, H, N, Dh, scale,
                       dtype, (cudaStream_t)stream);
}

int vrr_layernorm_fwd(const void* x, const float* gamma, const float* beta, void* y, float* mean, float* rstd, int M,
                      int E, float eps, int x_dtype, int y_dtype, void* stream) {
  VRR_REQUIRE(x && gamma && beta && y && mean && rstd, VRR_ERR_INVALID_ARG, "layernorm_fwd: NULL pointer");
  VRR_REQUIRE(dtype_ok(x_dtype) && dtype_ok(y_dtype) && no_mix(x_dtype, y_dtype), VRR_ERR_INVALID_ARG, "layernorm_fwd: bad dtype");
  VRR_REQUIRE(M > 0 && E > 0, VRR_ERR_INVALID_ARG, "layernorm_fwd: bad sizes");
  VRR_REQUIRE((((uintptr_t)x | (uintptr_t)y | (uintptr_t)gamma | (uintptr_t)beta) & 15) == 0, VRR_ERR_INVALID_ARG,
              "layernorm_fwd: pointers must be 16-byte aligned");
  if (int rc = require_device()) return rc;
  return layernorm_fwd(x, gamma, beta, y, mean, rstd, M, E, eps, x_dtype, y_dtype, (cudaStream_t)stream);
}

int vrr_layernorm_bwd(const void* dy, const void* x, const float* gamma, const float* mean, const float* rstd,
                      void* dx, float* dgamma, float* dbeta, int M, int E, int x_dtype, int y_dtype, void* stream) {
  VRR_REQUIRE(dy && x && gamma && mean && rstd && dx && dgamma && dbeta, VRR_ERR_INVALID_ARG, "layernorm_bwd: NULL pointer");
  VRR_REQUIRE(dtype_ok(x_dtype) && dtype_ok(y_dtype) && no_mix(x_dtype, y_dtype), VRR_ERR_INVALID_ARG, "layernorm_bwd: bad dtype");
  VRR_REQUIRE(M > 0 && E > 0, VRR_ERR_INVALID_ARG, "layernorm_bwd: bad sizes");
  VRR_REQUIRE((((uintptr_t)x | (uintptr_t)dy | (uintptr_t)dx | (uintptr_t)gamma) & 15) == 0, VRR_ERR_INVALID_ARG,
              "layernorm_bwd: pointers must be 16-byte aligned");
  if (int rc = require_device()) return rc;
  return layernorm_bwd(dy, x, gamma, mean, rstd, dx, dgamma, dbeta, M, E, x_dtype, y_dtype, (cudaStream_t)stream);
}

int vrr_add_layernorm_fwd(const void* x, const void* branch, void* x_new, const float* gamma, const float* beta,
                          void* y, float* mean, float* rstd, int M, int E, float eps, int branch_dtype, int y_dtype,
                          void* stream) {
  VRR_REQUIRE(x && branch && x_new && gamma && beta && y && mean && rstd, VRR_ERR_INVALID_ARG, "add_layernorm_fwd: NULL pointer");
  VRR_REQUIRE(dtype_ok(branch_dtype) && dtype_ok(y_dtype) && no_mix(branch_dtype, y_dtype), VRR_ERR_INVALID_ARG,
              "add_layernorm_fwd: bad dtype");
  VRR_REQUIRE(M > 0 && E > 0, VRR_ERR_INVALID_ARG, "add_layernorm_fwd: bad sizes");
  VRR_REQUIRE((((uintptr_t)x | (uintptr_t)branch | (uintptr_t)x_new | (uintptr_t)y | (uintptr_t)gamma | (uintptr_t)beta) & 15) == 0,
              VRR_ERR_INVALID_ARG, "add_layernorm_fwd: pointers must be 16-byte aligned");
  if (int rc = require_device()) return rc;
  return add_layernorm_fwd(x, branch, x_new, gamma, beta, y, mean, rstd, M, E, eps, branch_dtype, y_dtype, nullptr,
                           nullptr, (cudaStream_t)stream);
}

int vrr_add_layernorm_drop_fwd(const void* x, const void* branch, void* x_new, const float* gamma, const float* beta,
                               void* y, float* mean, float* rstd, int M, int E, float eps, int branch_dtype, int y_dtype,
                               const vrr_drop_desc* drop, void* stream) {
  VRR_REQUIRE(x && branch && x_new && gamma && beta && y && mean && rstd, VRR_ERR_INVALID_ARG, "add_layernorm_drop_fwd: NULL pointer");
  VRR_REQUIRE(dtype_ok(branch_dtype) && dtype_ok(y_dtype) && no_mix(branch_dtype, y_dtype), VRR_ERR_INVALID_ARG,
              "add_layernorm_drop_fwd: bad dtype");
  VRR_REQUIRE(M > 0 && E > 0, VRR_ERR_INVALID_ARG, "add_layernorm_drop_fwd: bad sizes");
  VRR_REQUIRE((((uintptr_t)x | (uintptr_t)branch | (uintptr_t)x_new | (uintptr_t)y | (uintptr_t)gamma | (uintptr_t)beta) & 15) == 0,
              VRR_ERR_INVALID_ARG, "add_layernorm_drop_fwd: pointers must be 16-byte aligned");
  if (int rc = require_device()) return rc;
  return add_layernorm_fwd(x, branch, x_new, gamma, beta, y, mean, rstd, M, E, eps, branch_dtype, y_dtype, drop,
                           nullptr, (cudaStream_t)stream);
}

int vrr_add_layernorm_bwd(const void* dy, const void* d_xnew, const void* x_new, const float* gamma, const float* mean,
                          const float* rstd, void* dx, void* d_branch, float* dgamma, float* dbeta, int M, int E,
                          int branch_dtype, int y_dtype, void* stream) {
  VRR_REQUIRE(dy && x_new && gamma && mean && rstd && dx && d_branch && dgamma && dbeta, VRR_ERR_INVALID_ARG,
              "add_layernorm_bwd: NULL pointer");
  VRR_REQUIRE(dtype_ok(branch_dtype) && dtype_ok(y_dtype) && no_mix(branch_dtype, y_dtype), VRR_ERR_INVALID_ARG,
              "add_layernorm_bwd: bad dtype");
  VRR_REQUIRE(M > 0 && E > 0, VRR_ERR_INVALID_ARG, "add_layernorm_bwd: bad sizes");
  VRR_REQUIRE((((uintptr_t)dy | (uintptr_t)d_xnew | (uintptr_t)x_new | (uintptr_t)dx | (uintptr_t)d_branch | (uintptr_t)gamma) & 15) == 0,
              VRR_ERR_INVALID_ARG, "add_layernorm_bwd: pointers must be 16-byte aligned");
  if (int rc = require_device()) return rc;
  return add_layernorm_bwd(dy, d_xnew, x_new, gamma, mean, rstd, dx, d_branch, dgamma, dbeta, M, E, branch_dtype,
                           y_dtype, nullptr, nullptr, nullptr, nullptr, (cudaStream_t)stream);
}

int vrr_add_layernorm_drop_bwd(const void* dy, const void* d_xnew, const void* x_new, const float* gamma,
                               const float* mean, const float* rstd, void* dx, void* d_branch, float* dgamma,
                               float* dbeta, int M, int E, int branch_dtype, int y_dtype, const vrr_drop_desc* drop,
                               void* stream) {
  VRR_REQUIRE(dy && x_new && gamma && mean && rstd && dx && d_branch && dgamma && dbeta, VRR_ERR_INVALID_ARG,
              "add_layernorm_drop_bwd: NULL pointer");
  VRR_REQUIRE(dtype_ok(branch_dtype) && dtype_ok(y_dtype) && no_mix(branch_dtype, y_dtype), VRR_ERR_INVALID_ARG,
              "add_layernorm_drop_bwd: bad dtype");
  VRR_REQUIRE(M > 0 && E > 0, VRR_ERR_INVALID_ARG, "add_layernorm_drop_bwd: bad sizes");
  VRR_REQUIRE((((uintptr_t)dy | (uintptr_t)d_xnew | (uintptr_t)x_new | (uintptr_t)dx | (uintptr_t)d_branch | (uintptr_t)gamma) & 15) == 0,
              VRR_ERR_INVALID_ARG, "add_layernorm_drop_bwd: pointers must be 16-byte aligned");
  if (int rc = require_device()) return rc;
  return add_layernorm_bwd(dy, d_xnew, x_new, gamma, mean, rstd, dx, d_branch, dgamma, dbeta, M, E, branch_dtype,
                           y_dtype, drop, nullptr, nullptr, nullptr, (cudaStream_t)stream);
}

int vrr_add_layernorm_ls_fwd(const void* x, const void* branch, void* x_new, const float* gamma, const float* beta,
                             void* y, float* mean, float* rstd, int M, int E, float eps, int branch_dtype, int y_dtype,
                             const vrr_drop_desc* drop, const float* ls, void* stream) {
  VRR_REQUIRE(x && branch && x_new && gamma && beta && y && mean && rstd, VRR_ERR_INVALID_ARG, "add_layernorm_ls_fwd: NULL pointer");
  VRR_REQUIRE(dtype_ok(branch_dtype) && dtype_ok(y_dtype) && no_mix(branch_dtype, y_dtype), VRR_ERR_INVALID_ARG,
              "add_layernorm_ls_fwd: bad dtype");
  VRR_REQUIRE(M > 0 && E > 0, VRR_ERR_INVALID_ARG, "add_layernorm_ls_fwd: bad sizes");
  VRR_REQUIRE((((uintptr_t)x | (uintptr_t)branch | (uintptr_t)x_new | (uintptr_t)y | (uintptr_t)gamma | (uintptr_t)beta |
                (uintptr_t)ls) & 15) == 0,
              VRR_ERR_INVALID_ARG, "add_layernorm_ls_fwd: pointers must be 16-byte aligned");
  if (int rc = require_device()) return rc;
  return add_layernorm_fwd(x, branch, x_new, gamma, beta, y, mean, rstd, M, E, eps, branch_dtype, y_dtype, drop, ls,
                           (cudaStream_t)stream);
}

int vrr_add_layernorm_ls_bwd(const void* dy, const void* d_xnew, const void* x_new, const float* gamma,
                             const float* mean, const float* rstd, void* dx, void* d_branch, float* dgamma,
                             float* dbeta, int M, int E, int branch_dtype, int y_dtype, const vrr_drop_desc* drop,
                             const float* ls, const void* branch, float* d_ls, void* stream) {
  VRR_REQUIRE(dy && x_new && gamma && mean && rstd && dx && d_branch && dgamma && dbeta, VRR_ERR_INVALID_ARG,
              "add_layernorm_ls_bwd: NULL pointer");
  VRR_REQUIRE(!d_ls || (ls && branch), VRR_ERR_INVALID_ARG, "add_layernorm_ls_bwd: d_ls needs ls and branch");
  VRR_REQUIRE(dtype_ok(branch_dtype) && dtype_ok(y_dtype) && no_mix(branch_dtype, y_dtype), VRR_ERR_INVALID_ARG,
              "add_layernorm_ls_bwd: bad dtype");
  VRR_REQUIRE(M > 0 && E > 0, VRR_ERR_INVALID_ARG, "add_layernorm_ls_bwd: bad sizes");
  VRR_REQUIRE((((uintptr_t)dy | (uintptr_t)d_xnew | (uintptr_t)x_new | (uintptr_t)dx | (uintptr_t)d_branch | (uintptr_t)gamma |
                (uintptr_t)ls | (uintptr_t)branch) & 15) == 0,
              VRR_ERR_INVALID_ARG, "add_layernorm_ls_bwd: pointers must be 16-byte aligned");
  if (int rc = require_device()) return rc;
  return add_layernorm_bwd(dy, d_xnew, x_new, gamma, mean, rstd, dx, d_branch, dgamma, dbeta, M, E, branch_dtype,
                           y_dtype, drop, ls, branch, d_ls, (cudaStream_t)stream);
}

int vrr_dropout_mask(const vrr_drop_desc* drop, void* keep_u8, void* keep_path_u8, int M, int E, void* stream) {
  VRR_REQUIRE(drop && drop->seed, VRR_ERR_INVALID_ARG, "dropout_mask: NULL desc or seed");
  VRR_REQUIRE(M > 0 && E > 0 && E % 8 == 0, VRR_ERR_INVALID_ARG, "dropout_mask: bad sizes (E %% 8 == 0)");
  VRR_REQUIRE(!keep_path_u8 || drop->rows_per_sample > 0, VRR_ERR_INVALID_ARG,
              "dropout_mask: keep_path needs rows_per_sample > 0");
  VRR_REQUIRE(((uintptr_t)keep_u8 & 7) == 0, VRR_ERR_INVALID_ARG, "dropout_mask: keep_u8 must be 8-byte aligned");
  DropView dv = {};
  bool active = false;
  if (int rc = drop_view(drop, M, E, &dv, &active)) return rc;
  if (!active) {  // nothing dropped: the same DropView with thresholds that keep everything
    dv.seed = reinterpret_cast<const unsigned long long*>(drop->seed);
    dv.t = dv.t_path = 65536u;
    dv.s = 1.f;
    dv.rows_per_sample = drop->rows_per_sample > 0 ? drop->rows_per_sample : 1;
    dv.site = drop->site;
  }
  if (int rc = require_device()) return rc;
  if (!keep_u8 && !keep_path_u8) return VRR_OK;
  return dropout_mask(dv, (uint8_t*)keep_u8, (uint8_t*)keep_path_u8, M, E, (cudaStream_t)stream);
}

int vrr_colsum(const void* x, float* out, int M, int C, int dtype, void* stream) {
  VRR_REQUIRE(x && out, VRR_ERR_INVALID_ARG, "colsum: NULL pointer");
  VRR_REQUIRE(dtype_ok(dtype) && M > 0 && C > 0, VRR_ERR_INVALID_ARG, "colsum: bad arguments");
  if (int rc = require_device()) return rc;
  return colsum(x, out, M, C, dtype, (cudaStream_t)stream);
}

int vrr_gelu_bwd(const void* dy, const void* h, void* dh, float* db, int M, int C, int dtype, void* stream) {
  VRR_REQUIRE(dy && h && dh && db, VRR_ERR_INVALID_ARG, "gelu_bwd: NULL pointer");
  VRR_REQUIRE(dtype_ok(dtype) && M > 0 && C > 0, VRR_ERR_INVALID_ARG, "gelu_bwd: bad arguments");
  VRR_REQUIRE((((uintptr_t)dy | (uintptr_t)h | (uintptr_t)dh) & 15) == 0, VRR_ERR_INVALID_ARG,
              "gelu_bwd: pointers must be 16-byte aligned");
  if (int rc = require_device()) return rc;
  return gelu_bwd_colsum(dy, h, dh, db, M, C, dtype, (cudaStream_t)stream);
}

}  // extern "C"
