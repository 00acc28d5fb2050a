"""ctypes binding of ``libvrr_b200.so`` (C ABI declared in ``include/vrr.h``).

The library is built in-tree by ``__graft_entry__.build()`` (``nvcc -gencode
arch=compute_100a,code=sm_100a``) into ``vit_rpe_rope_b200/lib/``.  There is no
fallback: if the shared object is missing, or the current device is not sm_100,
every op raises.
"""
import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_int32, c_size_t, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libvrr_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "vrr.h")

VRR_F32, VRR_BF16, VRR_F16 = 0, 1, 2
ROPE_NONE, ROPE_AXIAL, ROPE_MIXED = 0, 1, 2
BIAS_NONE, BIAS_TABLE, BIAS_POLY = 0, 1, 2
IMPL_AUTO, IMPL_SIMT, IMPL_TCGEN05 = 0, 1, 2
EPI_NONE, EPI_BIAS, EPI_BIAS_GELU, EPI_BIAS_GELU_GRAD, EPI_MUL, EPI_BIAS_GELU_ACT = 0, 1, 2, 3, 4, 5

STATUS_NAMES = {0: "VRR_OK", -1: "VRR_ERR_INVALID_ARG", -2: "VRR_ERR_UNSUPPORTED",
                -3: "VRR_ERR_NO_DEVICE", -4: "VRR_ERR_CUDA", -5: "VRR_ERR_WORKSPACE"}


class BiasDesc(Structure):
    """``vrr_bias_desc`` of include/vrr.h."""
    _fields_ = [("mode", c_int32), ("heads", c_int32), ("len", c_int32), ("grid", c_int32),
                ("param", c_void_p)]


class DropDesc(Structure):
    """``vrr_drop_desc`` of include/vrr.h (``seed``: device pointer to the 64-bit Philox key)."""
    _fields_ = [("p", c_float), ("p_path", c_float), ("rows_per_sample", c_int32), ("site", c_int32),
                ("seed", c_void_p)]


# name -> (restype, argtypes); must list every function include/vrr.h declares
# (tests/test_c_abi.py parses the header and checks this table and the .so against it).
SIGNATURES = {
    "vrr_abi_version": (c_int, []),
    "vrr_last_error": (c_char_p, []),
    "vrr_device_ok": (c_int, []),
    "vrr_set_impl": (c_int, [c_int]),
    "vrr_launch_count": (c_uint64, []),
    "vrr_family_count": (c_uint64, [c_int]),
    "vrr_set_option": (c_int, [c_char_p, c_int]),
    "vrr_debug_timestamps": (c_int, [c_void_p]),
    "vrr_patch_embed_workspace_bytes": (c_size_t, [c_int] * 7),
    "vrr_patch_embed_fwd": (c_int, [c_void_p] * 7 + [c_size_t] + [c_int] * 9 + [c_void_p]),
    "vrr_patch_unfold": (c_int, [c_void_p] * 2 + [c_int] * 6 + [c_void_p]),
    "vrr_patch_unfold_ex": (c_int, [c_void_p] * 2 + [c_int] * 7 + [c_void_p]),
    "vrr_patch_embed_bwd": (c_int, [c_void_p] * 6 + [c_int] * 9 + [c_void_p]),
    "vrr_patch_embed_fwd_prefix": (c_int, [c_void_p] * 4 + [c_int] + [c_void_p] * 3 + [c_size_t] + [c_int] * 9
                                   + [c_void_p]),
    "vrr_patch_embed_bwd_prefix": (c_int, [c_void_p] * 5 + [c_int] + [c_void_p] + [c_int] * 9 + [c_void_p]),
    "vrr_qkv_rope_fwd": (c_int, [c_void_p] * 5 + [c_int] * 6 + [c_void_p]),
    "vrr_qkv_rope_fwd_packed": (c_int, [c_void_p] * 6 + [c_int] * 6 + [c_void_p]),
    "vrr_rope_pack_tables": (c_int, [c_void_p] * 3 + [c_int] * 3 + [c_void_p]),
    "vrr_qkv_rope_bwd": (c_int, [c_void_p] * 7 + [c_int] * 6 + [c_void_p]),
    "vrr_qkv_rope_fwd_prefix": (c_int, [c_void_p] * 6 + [c_int] * 7 + [c_void_p]),
    "vrr_qkv_rope_bwd_prefix": (c_int, [c_void_p] * 7 + [c_int] * 7 + [c_void_p]),
    "vrr_qkv_rope_norm_fwd": (c_int, [c_void_p] * 6 + [c_int] * 7 + [c_void_p] * 4 + [c_float] + [c_void_p] * 3),
    "vrr_qkv_rope_norm_bwd": (c_int, [c_void_p] * 16 + [c_int] * 7 + [c_void_p]),
    "vrr_rope_apply": (c_int, [c_void_p] * 6 + [c_int] * 7 + [c_void_p]),
    "vrr_rope_table_grad": (c_int, [c_void_p] * 6 + [c_int] * 6 + [c_void_p]),
    "vrr_gemm": (c_int, [c_void_p] * 3 + [c_int] * 7 + [c_void_p]),
    "vrr_gemm_ex": (c_int, [c_void_p] * 5 + [c_int] * 9 + [c_void_p]),
    "vrr_layernorm_fwd": (c_int, [c_void_p] * 6 + [c_int, c_int, c_float, c_int, c_int, c_void_p]),
    "vrr_layernorm_bwd": (c_int, [c_void_p] * 8 + [c_int] * 4 + [c_void_p]),
    "vrr_add_layernorm_fwd": (c_int, [c_void_p] * 8 + [c_int, c_int, c_float, c_int, c_int, c_void_p]),
    "vrr_add_layernorm_bwd": (c_int, [c_void_p] * 10 + [c_int] * 4 + [c_void_p]),
    "vrr_add_layernorm_drop_fwd": (c_int, [c_void_p] * 8 + [c_int, c_int, c_float, c_int, c_int, POINTER(DropDesc),
                                                           c_void_p]),
    "vrr_add_layernorm_drop_bwd": (c_int, [c_void_p] * 10 + [c_int] * 4 + [POINTER(DropDesc), c_void_p]),
    "vrr_add_layernorm_ls_fwd": (c_int, [c_void_p] * 8 + [c_int, c_int, c_float, c_int, c_int, POINTER(DropDesc),
                                                         c_void_p, c_void_p]),
    "vrr_add_layernorm_ls_bwd": (c_int, [c_void_p] * 10 + [c_int] * 4 + [POINTER(DropDesc)] + [c_void_p] * 4),
    "vrr_gemm_ex_drop": (c_int, [c_void_p] * 5 + [c_int] * 9 + [POINTER(DropDesc), c_void_p]),
    "vrr_dropout_mask": (c_int, [POINTER(DropDesc), c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "vrr_colsum": (c_int, [c_void_p] * 2 + [c_int] * 3 + [c_void_p]),
    "vrr_gemm_mul_colsum": (c_int, [c_void_p] * 5 + [c_int] * 6 + [c_void_p]),
    "vrr_gelu_bwd": (c_int, [c_void_p] * 4 + [c_int] * 3 + [c_void_p]),
    "vrr_gemm_swiglu": (c_int, [c_void_p] * 5 + [c_int] * 4 + [POINTER(DropDesc), c_void_p]),
    "vrr_gemm_swiglu_bwd": (c_int, [c_void_p] * 5 + [c_int] * 4 + [c_void_p]),
    "vrr_attn_fwd": (c_int, [c_void_p, POINTER(BiasDesc), c_void_p, c_void_p] + [c_int] * 4
                     + [c_float, c_int, c_void_p]),
    "vrr_attn_bwd_workspace_bytes": (c_size_t, [c_int] * 4 + [POINTER(BiasDesc)]),
    "vrr_attn_bwd": (c_int, [c_void_p, POINTER(BiasDesc)] + [c_void_p] * 6 + [c_size_t] + [c_int] * 4
                     + [c_float, c_int, c_void_p]),
}

_lib = None


def load():
    """dlopen the library once and attach the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  vit_rpe_rope_b200 has no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    if lib.vrr_abi_version() != 1:
        raise ImportError(f"libvrr_b200.so ABI {lib.vrr_abi_version()} != 1: rebuild")
    _lib = lib
    # Debug switch (never set by the product): force one kernel family for the bf16 / fp16 kernels.
    forced = os.environ.get("VRR_IMPL", "").lower()
    if forced in ("simt", "tcgen05"):
        lib.vrr_set_impl(IMPL_SIMT if forced == "simt" else IMPL_TCGEN05)
    return lib


def last_error() -> str:
    return (load().vrr_last_error() or b"").decode("utf-8", "replace")


def check(rc: int, what: str):
    if rc != 0:
        raise RuntimeError(f"{what}: {STATUS_NAMES.get(rc, rc)}: {last_error()}")


def launch_count() -> int:
    return int(load().vrr_launch_count())


def family_count(family: int) -> int:
    """Dispatches that took the SIMT (IMPL_SIMT) or tcgen05 (IMPL_TCGEN05) kernel family since load."""
    return int(load().vrr_family_count(int(family)))


def set_impl(impl: int) -> int:
    return int(load().vrr_set_impl(int(impl)))
