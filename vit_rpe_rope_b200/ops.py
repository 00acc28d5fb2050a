"""Autograd bindings of the libvrr_b200 kernels (host side of the C ABI).

Each ``torch.autograd.Function`` here is the product implementation of one stretch of the
reference's ``Attention.forward`` / ``forward_features`` (citations: /root/reference):

* :class:`PatchEmbedFn`      - models/vit.py:164,248-258 (conv patch embed, cls / register concat, absolute add)
* :class:`QkvRopeFn`         - models/vit.py:47-68 + models/rope_utils.py:22-35
* :class:`FusedAttentionFn`  - models/vit.py:71-88

PyTorch is used for device memory, streams and autograd plumbing only; all arithmetic on these
paths runs in the hand-written sm_100a kernels.  CUDA only - CPU tensors raise.
"""
import ctypes
import os
import weakref

import torch

from . import _lib

_DT = {torch.float32: _lib.VRR_F32, torch.bfloat16: _lib.VRR_BF16, torch.float16: _lib.VRR_F16}
# the 16-bit compute dtypes: both run the same kernels (tcgen05 where the shape allows) and the same fusions
_LP16 = (torch.bfloat16, torch.float16)


def compute_dtype(x: torch.Tensor) -> torch.dtype:
    """Element type the kernels run in: the autocast dtype inside ``torch.autocast('cuda')`` (bf16, or fp16 - the
    default of ``torch.autocast('cuda')``; how the build defines "bf16 training", SURVEY.md row O4), else the tensor's
    own dtype."""
    dt = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else x.dtype
    if dt not in _DT:
        raise TypeError(f"vit_rpe_rope_b200 kernels support float32, bfloat16 and float16, got {dt}")
    return dt


def _require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError(
                "vit_rpe_rope_b200 runs on CUDA sm_100 devices only (no CPU fallback); got a "
                f"{t.device} tensor")


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _f32c(t):
    return None if t is None else t.detach().to(torch.float32).contiguous()


# ---- low-precision weight cache ---------------------------------------------------------------------
# Under autocast the reference re-casts every fp32 weight to bf16 / fp16 in every forward (~60 small cast kernels per
# ViT-B step).  Here the model asks once per forward: the 16-bit copies of all its GEMM weights are refreshed by
# ONE multi-tensor copy, and only when a master weight changed (its version counter moved) - i.e. once per
# optimizer step.  The GEMM Functions take the fp32 master (it receives the fp32 weight gradient straight from
# the dW GEMM) plus this copy.
_LP = {}  # id(param) -> [weakref(param), version at last refresh, low-precision copy]


def refresh_lp_weights(params, dt):
    src, dst = [], []
    capturing = torch.cuda.is_current_stream_capturing()
    for p in params:
        if p.dtype == dt or not p.is_cuda:
            continue
        ent = _LP.get(id(p))
        if ent is None or ent[0]() is not p or ent[2].device != p.device or ent[2].dtype != dt or ent[2].shape != p.shape:
            ent = [weakref.ref(p), -1, torch.empty_like(p, dtype=dt, memory_format=torch.contiguous_format)]
            _LP[id(p)] = ent
        if capturing or ent[1] != p._version:  # a captured step must always contain its own refresh
            src.append(p.detach())
            dst.append(ent[2])
            ent[1] = p._version
    if dst:
        torch._foreach_copy_(dst, src)
    if len(_LP) > 4096:  # drop entries of dead parameters
        for k in [k for k, e in _LP.items() if e[0]() is None]:
            del _LP[k]


def lp_weight(p, dt):
    """The cached ``dt`` copy of parameter ``p`` if :func:`refresh_lp_weights` holds a current one, else None."""
    ent = _LP.get(id(p))
    if ent is None or ent[0]() is not p or ent[2].dtype != dt or ent[1] != p._version or ent[2].device != p.device:
        return None
    return ent[2]


# bench.py sets this to a list to time individual kernel launches with CUDA events recorded on the
# launching (current) stream; None (default) adds no overhead.
PROFILE_EVENTS = None


class _timed:
    def __init__(self, name):
        self.name = name

    def __enter__(self):
        if PROFILE_EVENTS is not None:
            self.start = torch.cuda.Event(enable_timing=True)
            self.start.record()

    def __exit__(self, *exc):
        if PROFILE_EVENTS is not None:
            end = torch.cuda.Event(enable_timing=True)
            end.record()
            PROFILE_EVENTS.append((self.name, self.start, end))
        return False


# ------------------------------------------------------------------------------------------------
class PatchEmbedFn(torch.autograd.Function):
    """tokens[B, P+Np, E] from images: the P prefix rows (cls, then register tokens) + unfold + GEMM + bias
    (+ absolute pos_embed on the patch rows).

    weight / bias carry the conv dtype; prefix_tokens ([..., P, E], e.g. the [1, 1, E] cls token) / pos_embed / tokens
    the token-stream dtype (fp32 under autocast, like the reference's cat with the fp32 cls token); images may stay
    fp32 when the conv runs in bf16 / fp16 - the rounding is fused into the kernel's load."""

    @staticmethod
    def forward(ctx, images, weight, bias, prefix_tokens, pos_embed, patch):
        _require_cuda(images, weight, bias, prefix_tokens, pos_embed)
        lib = _lib.load()
        B, C, Hi, Wi = images.shape
        E = weight.shape[0]
        idt, dt, tdt = images.dtype, weight.dtype, prefix_tokens.dtype
        if bias.dtype != dt or (pos_embed is not None and pos_embed.dtype != tdt):
            raise TypeError("patch_embed: weight/bias must share a dtype, prefix_tokens/pos_embed another")
        if idt != dt and not (idt == torch.float32 and dt in _LP16):
            raise TypeError(f"patch_embed: images {idt} with weights {dt} is not supported")
        if prefix_tokens.numel() == 0 or prefix_tokens.numel() % E or prefix_tokens.shape[-1] != E:
            raise RuntimeError(f"patch_embed: prefix tokens {tuple(prefix_tokens.shape)} are not [..., n_prefix, {E}]")
        images = images.contiguous()
        w = weight.detach().contiguous()
        b = bias.detach().contiguous()
        prefix = prefix_tokens.detach().reshape(-1, E).contiguous()
        n_prefix = prefix.shape[0]
        Np = (Hi // patch) * (Wi // patch)
        pos = None
        if pos_embed is not None:
            if pos_embed.shape[-2] < Np:
                raise RuntimeError(f"absolute pos_embed has {pos_embed.shape[-2]} rows, need {Np}")
            pos = pos_embed.detach().reshape(-1, E).contiguous()
        tokens = torch.empty(B, n_prefix + Np, E, device=images.device, dtype=tdt)
        ws_bytes = int(lib.vrr_patch_embed_workspace_bytes(B, C, Hi, Wi, patch, E, _DT[dt]))
        ws = torch.empty(ws_bytes, device=images.device, dtype=torch.uint8) if ws_bytes else None
        with torch.cuda.device(images.device), _timed("patch_embed_fwd"):
            _lib.check(lib.vrr_patch_embed_fwd_prefix(_ptr(images), _ptr(w), _ptr(b), _ptr(prefix), n_prefix, _ptr(pos),
                                                      _ptr(tokens), _ptr(ws), ws_bytes, B, C, Hi, Wi, patch, E, _DT[idt],
                                                      _DT[dt], _DT[tdt], _stream()), "vrr_patch_embed_fwd_prefix")
        if ctx.needs_input_grad[0]:
            ctx.w_for_dimg = w
        # the tcgen05 path's workspace IS unfold(images) [B*Np][C*P*P] in dt: the weight-gradient GEMM reuses it
        ctx.unfolded = ws if (ws is not None and ws_bytes == B * Np * C * patch * patch * 2) else None
        ctx.save_for_backward(images)
        ctx.meta = (B, C, Hi, Wi, patch, E, Np, n_prefix, pos_embed.shape if pos_embed is not None else None,
                    weight.shape, prefix_tokens.shape, idt, dt, tdt)
        return tokens

    @staticmethod
    def backward(ctx, d_tokens):
        lib = _lib.load()
        (images,) = ctx.saved_tensors
        B, C, Hi, Wi, patch, E, Np, n_prefix, pos_shape, w_shape, prefix_shape, idt, dt, tdt = ctx.meta
        d_tokens = d_tokens.contiguous()
        dev = images.device
        K = C * patch * patch
        # bf16 / fp16: the weight gradient is the GEMM d_tokens^T . unfold(images) on the tcgen05 kernel (fp32 result,
        # split over the B*Np rows); fp32: the library's FFMA split-K GEMM with the unfold fused in.
        own_dw = not (dt in _LP16 and patch % 8 == 0 and Wi % 4 == 0 and E % 8 == 0)
        d_w = torch.empty(E, K, device=dev, dtype=torch.float32) if own_dw else None
        d_b = torch.empty(E, device=dev, dtype=torch.float32)
        d_prefix = torch.empty(n_prefix, E, device=dev, dtype=torch.float32)
        d_pos_rows = torch.empty(Np, E, device=dev, dtype=torch.float32) if pos_shape is not None else None
        with torch.cuda.device(dev), _timed("patch_embed_bwd"):
            _lib.check(lib.vrr_patch_embed_bwd_prefix(_ptr(images), _ptr(d_tokens), _ptr(d_w), _ptr(d_b), _ptr(d_prefix),
                                                      n_prefix, _ptr(d_pos_rows), B, C, Hi, Wi, patch, E, _DT[idt], _DT[dt],
                                                      _DT[tdt], _stream()), "vrr_patch_embed_bwd_prefix")
            if not own_dw:
                if ctx.unfolded is not None:
                    unf = ctx.unfolded.view(dt).view(B * Np, K)
                else:
                    unf = torch.empty(B * Np, K, device=dev, dtype=dt)
                    _lib.check(lib.vrr_patch_unfold_ex(_ptr(images), _ptr(unf), B, C, Hi, Wi, patch, _DT[idt], _DT[dt],
                                                       _stream()), "vrr_patch_unfold_ex")
                # cast first: one strided read + packed 16-bit write (reshaping the fp32 slice first copied 154 MB twice)
                g = d_tokens[:, n_prefix:, :].to(dt).reshape(B * Np, E)
                d_w = _gemm(g, unf, True, False, torch.float32, name="patch_dw")
        d_pos = None
        if pos_shape is not None:
            d_pos = torch.zeros(pos_shape, device=dev, dtype=tdt)
            d_pos.view(-1, E)[:Np] = d_pos_rows.to(tdt)
        return (None, d_w.view(w_shape).to(dt), d_b.to(dt), d_prefix.view(prefix_shape).to(tdt), d_pos, None)


def patch_embed(images, weight, bias, prefix_tokens, pos_embed, patch):
    """Conv weights are cast to the compute dtype (autograd-tracked casts keep fp32 master grads);
    under autocast the token stream (prefix tokens, pos, output) stays fp32 as in the reference, and fp32 images
    are passed as they are (rounded to bf16 / fp16 inside the kernel).  ``prefix_tokens``: ``[1, n_prefix, E]``, the
    cls token followed by the register tokens (``torch.cat((cls_token, reg_token), 1)``); its gradient is the batch
    sum of the prefix rows' gradients."""
    dt = compute_dtype(images)
    tdt = torch.float32 if torch.is_autocast_enabled("cuda") else dt
    if not (images.dtype == torch.float32 and dt in _LP16):
        images = images.to(dt)
    return PatchEmbedFn.apply(images, weight.to(dt), bias.to(dt), prefix_tokens.to(tdt),
                              None if pos_embed is None else pos_embed.to(tdt), patch)


# ------------------------------------------------------------------------------------------------
def _rope_args(cos, sin, H, N, Dh, n_prefix=1):
    """Classify the (cos, sin) pair the way ``reshape_for_broadcast`` does (rope_utils.py:39-66).  The tables cover
    the N - n_prefix patch tokens; the prefix tokens (cls, registers) are not rotated."""
    if cos is None:
        return _lib.ROPE_NONE
    if cos.shape != sin.shape:
        raise RuntimeError(f"cos {tuple(cos.shape)} and sin {tuple(sin.shape)} differ")
    rows = N - n_prefix
    if cos.ndim == 2:
        mode, want = _lib.ROPE_AXIAL, (rows, Dh // 2)
    elif cos.ndim == 3:
        mode, want = _lib.ROPE_MIXED, (H, rows, Dh // 2)
    else:
        raise ValueError(f"Unexpected tensor shapes: {cos.shape} vs {(1, H, rows, Dh)}")
    if tuple(cos.shape) != want:
        raise RuntimeError(f"RoPE table shape {tuple(cos.shape)} does not broadcast against the "
                           f"{rows} patch tokens x {H} heads x {Dh} channels (expected {want})")
    return mode


_packed_cache = {}  # device index -> (key, cos32, sin32, packed); the table tensors are held so their storage stays theirs


def _packed_tables(cos32, sin32):
    """``vrr_rope_pack_tables`` of the fp32 tables ([heads][half/2][rows] float4), computed once per table pair: every
    block of a forward pass receives the SAME cos / sin storage (one shared PE module), so the repack runs once per
    step (and once inside a captured graph).  Keyed on storage address + version counter; the cache keeps the tables
    alive, so an address cannot be recycled for other data while its entry exists."""
    dev = cos32.device.index
    try:
        key = (cos32.data_ptr(), sin32.data_ptr(), cos32._version, sin32._version, tuple(cos32.shape))
    except RuntimeError:  # tensors made under torch.inference_mode() carry no version counter: repack every call
        key = None
    hit = _packed_cache.get(dev)
    if key is not None and hit is not None and hit[0] == key:
        return hit[3]
    heads = cos32.shape[0] if cos32.ndim == 3 else 1
    rows, half = cos32.shape[-2], cos32.shape[-1]
    packed = torch.empty(heads, half // 2, rows, 4, device=cos32.device, dtype=torch.float32)
    _lib.check(_lib.load().vrr_rope_pack_tables(_ptr(cos32), _ptr(sin32), _ptr(packed), heads, rows, half, _stream()),
               "vrr_rope_pack_tables")
    if key is not None:
        _packed_cache[dev] = (key, cos32, sin32, packed)
    return packed


class QkvRopeFn(torch.autograd.Function):
    """planes[3, B, H, N, Dh] = split_heads(x @ w_qkv^T), q/k rows n_prefix.. rotated in the GEMM epilogue; with QK-norm
    (``qn_w`` .. ``kn_b`` given) every q / k head row is layer-normalised first (``vrr_qkv_rope_norm_fwd``)."""

    @staticmethod
    def forward(ctx, x, w_qkv, cos, sin, num_heads, w_lp=None, n_prefix=1, qn_w=None, qn_b=None, kn_w=None, kn_b=None,
                eps=1e-5):
        """``w_qkv`` receives the gradient (fp32 master weight or a tensor already in x's dtype); ``w_lp`` is an
        optional ready-made copy of it in x's dtype (the model's 16-bit weight cache).  ``n_prefix``: the leading
        token rows that are never rotated (cls and register tokens); row t >= n_prefix uses table row t - n_prefix.
        ``qn_w, qn_b, kn_w, kn_b``: the [Dh] weight and bias of q_norm / k_norm (all four or none), with ``eps``."""
        _require_cuda(x, w_qkv, cos, sin, qn_w, qn_b, kn_w, kn_b)
        lib = _lib.load()
        B, N, E = x.shape
        H, Dh = num_heads, E // num_heads
        mode = _rope_args(cos, sin, H, N, Dh, n_prefix)
        x = x.contiguous()
        w = (w_lp if w_lp is not None else w_qkv.detach().to(x.dtype)).detach().contiguous()
        ctx.w_grad_dtype = w_qkv.dtype
        cos32, sin32 = _f32c(cos), _f32c(sin)
        planes = torch.empty(3, B, H, N, Dh, device=x.device, dtype=x.dtype)
        norm = qn_w is not None
        with torch.cuda.device(x.device):
            packed = None
            if mode != _lib.ROPE_NONE and x.dtype in _LP16 and Dh == 64:  # the tcgen05 epilogue's table layout
                packed = _packed_tables(cos32, sin32)
            if not norm:
                with _timed("qkv_rope_fwd"):
                    _lib.check(lib.vrr_qkv_rope_fwd_prefix(_ptr(x), _ptr(w), _ptr(cos32), _ptr(sin32), _ptr(packed),
                                                           _ptr(planes), B, N, E, H, n_prefix, mode, _DT[x.dtype], _stream()),
                               "vrr_qkv_rope_fwd_prefix")
                ctx.save_for_backward(x, w, planes, cos32, sin32)
                ctx.meta = (B, N, E, H, n_prefix, mode, None if cos is None else (cos.dtype, sin.dtype))
                ctx.norm = None
                return planes
            nt = [_f32c(t) for t in (qn_w, qn_b, kn_w, kn_b)]
            grad = any(ctx.needs_input_grad)
            qk_pre = torch.empty(2, B, H, N, Dh, device=x.device, dtype=x.dtype) if grad else None  # inference: no saves
            qk_stats = torch.empty(2, B, H, N, 2, device=x.device, dtype=torch.float32) if grad else None
            with _timed("qkv_rope_fwd"):
                _lib.check(lib.vrr_qkv_rope_norm_fwd(_ptr(x), _ptr(w), _ptr(cos32), _ptr(sin32), _ptr(packed), _ptr(planes),
                                                     B, N, E, H, n_prefix, mode, _DT[x.dtype], *map(_ptr, nt), float(eps),
                                                     _ptr(qk_pre), _ptr(qk_stats), _stream()), "vrr_qkv_rope_norm_fwd")
        if grad:
            ctx.save_for_backward(x, w, qk_pre, qk_stats, cos32, sin32, *nt)
            ctx.meta = (B, N, E, H, n_prefix, mode, None if cos is None else (cos.dtype, sin.dtype))
            ctx.norm = tuple(t.dtype for t in (qn_w, qn_b, kn_w, kn_b))
        return planes

    @staticmethod
    def backward(ctx, d_planes):
        lib = _lib.load()
        if ctx.norm is None:
            x, w, planes, cos32, sin32 = ctx.saved_tensors
        else:
            x, w, qk_pre, qk_stats, cos32, sin32, *nt = ctx.saved_tensors
        B, N, E, H, n_prefix, mode, cs_dtypes = ctx.meta
        d_planes = d_planes.contiguous()
        dev, dt = x.device, x.dtype
        need_cs = mode != _lib.ROPE_NONE and (ctx.needs_input_grad[2] or ctx.needs_input_grad[3])
        d_cos = d_sin = None
        if need_cs:  # halves of one buffer: zeroed by one memset
            d_cs = torch.empty((2,) + tuple(cos32.shape), device=dev, dtype=torch.float32)
            d_cos, d_sin = d_cs[0], d_cs[1]
        d_qkv = torch.empty(B * N, 3 * E, device=dev, dtype=dt)
        d_norm = [None] * 4
        with torch.cuda.device(dev):
            if ctx.norm is None:
                with _timed("qkv_rope_bwd"):
                    _lib.check(lib.vrr_qkv_rope_bwd_prefix(_ptr(d_planes), _ptr(planes), _ptr(cos32), _ptr(sin32),
                                                           _ptr(d_qkv), _ptr(d_cos), _ptr(d_sin), B, N, E, H, n_prefix, mode,
                                                           _DT[dt], _stream()), "vrr_qkv_rope_bwd_prefix")
            else:
                if any(ctx.needs_input_grad[7:11]):  # rows of one buffer: zeroed by one memset
                    d_norm = list(torch.empty(4, E // H, device=dev, dtype=torch.float32))
                with _timed("qkv_rope_bwd"):
                    _lib.check(lib.vrr_qkv_rope_norm_bwd(_ptr(d_planes), _ptr(qk_pre), _ptr(qk_stats), _ptr(cos32),
                                                         _ptr(sin32), *map(_ptr, nt), _ptr(d_qkv), _ptr(d_cos), _ptr(d_sin),
                                                         *map(_ptr, d_norm), B, N, E, H, n_prefix, mode, _DT[dt],
                                                         _stream()), "vrr_qkv_rope_norm_bwd")
                d_norm = [None if g is None else g.to(t) for g, t in zip(d_norm, ctx.norm)]
            dx = dw = None
            if ctx.needs_input_grad[0]:
                dx = _gemm(d_qkv, w, False, False, dt, name="qkv_dx").view(B, N, E)            # [BN,3E] . [3E,E]
            if ctx.needs_input_grad[1]:
                dw = _gemm(d_qkv, x.view(B * N, E), True, False, ctx.w_grad_dtype, name="qkv_dw")  # [3E,BN] . [BN,E]
        if need_cs:
            d_cos, d_sin = d_cos.to(cs_dtypes[0]), d_sin.to(cs_dtypes[1])
        return (dx, dw, d_cos, d_sin, None, None, None, *d_norm, None)


def _gemm(a, b, trans_a, trans_b, out_dtype, bias=None, epilogue=_lib.EPI_NONE, out2=False, name="gemm", aux=None,
          drop=None):
    """C = op(A) . op(B) in the library's kernels (``vrr_gemm_ex``) - no cuBLAS anywhere on the path.

    op(A) is [M][K] (trans_a: A stored [K][M]); op(B) is [K][N] (trans_b: B stored [N][K]).  bf16 / fp16 operands
    run the tcgen05 CTA-pair kernel (fp32 accumulation; result in ``out_dtype``: the operands' type, or fp32 for
    weight gradients), fp32 operands the exact-fp32 FFMA kernel (no TF32).  ``epilogue``: fused ``+ bias`` or
    ``+ bias, GELU`` (``out2``: second output - gelu(C) for EPI_BIAS_GELU; EPI_BIAS_GELU_GRAD returns
    (gelu(h), gelu'(h)) instead; EPI_BIAS_GELU_ACT returns gelu(h) alone); ``aux``: the [M][N] multiplier of EPI_MUL;
    ``drop``: element dropout on the GELU outputs of those two epilogues (``vrr_gemm_ex_drop``)."""
    lib = _lib.load()
    M = a.shape[1] if trans_a else a.shape[0]
    K = a.shape[0] if trans_a else a.shape[1]
    N = b.shape[0] if trans_b else b.shape[1]
    a, b = a.contiguous(), b.contiguous()
    c = torch.empty(M, N, device=a.device, dtype=out_dtype)
    c2 = torch.empty_like(c) if out2 else (aux.contiguous() if aux is not None else None)
    bias32 = _f32c(bias) if bias is not None and epilogue != _lib.EPI_NONE else None
    with _timed(name):
        if drop is None:
            _lib.check(lib.vrr_gemm_ex(_ptr(a), _ptr(b), _ptr(c), _ptr(c2), _ptr(bias32), M, N, K, int(trans_a), int(trans_b),
                                       _DT[a.dtype], _DT[out_dtype], int(epilogue), 0, _stream()), "vrr_gemm_ex")
        else:
            d = _drop_desc(drop)
            _lib.check(lib.vrr_gemm_ex_drop(_ptr(a), _ptr(b), _ptr(c), _ptr(c2), _ptr(bias32), M, N, K, int(trans_a),
                                            int(trans_b), _DT[a.dtype], _DT[out_dtype], int(epilogue), 0, ctypes.byref(d),
                                            _stream()), "vrr_gemm_ex_drop")
    return (c, c2) if out2 else c


def qkv_rope(x, w_qkv, cos, sin, num_heads, w_lp=None, n_prefix=1, q_norm=None, k_norm=None):
    """``n_prefix``: the leading token rows that RoPE leaves alone (the cls token and any register tokens).
    ``q_norm`` / ``k_norm``: QK-norm, two affine ``nn.LayerNorm((Dh,))`` with one eps (:func:`check_qk_norm`), or None."""
    dt = compute_dtype(x)
    if w_lp is not None and w_lp.dtype != dt:
        w_lp = None
    if q_norm is None and k_norm is None:
        return QkvRopeFn.apply(x.to(dt), w_qkv, cos, sin, num_heads, w_lp, n_prefix)
    check_qk_norm(q_norm, k_norm, x.shape[-1] // num_heads)
    return QkvRopeFn.apply(x.to(dt), w_qkv, cos, sin, num_heads, w_lp, n_prefix, q_norm.weight, q_norm.bias, k_norm.weight,
                           k_norm.bias, q_norm.eps)


def check_qk_norm(q_norm, k_norm, head_dim):
    """The QK-norm the fused QKV kernels implement: q_norm and k_norm are affine ``nn.LayerNorm((head_dim,))`` with a
    bias and the same eps.  Anything else (an RMSNorm, a LayerNorm without affine or bias) raises NotImplementedError."""
    for name, m in (("q_norm", q_norm), ("k_norm", k_norm)):
        if not (type(m) is torch.nn.LayerNorm and m.elementwise_affine and m.bias is not None
                and tuple(m.normalized_shape) == (head_dim,)):
            raise NotImplementedError(f"qk_norm: {name} is {m!r}; the fused QKV+RoPE kernel implements an affine "
                                      f"nn.LayerNorm(({head_dim},)) with weight and bias only")
    if q_norm.eps != k_norm.eps:
        raise NotImplementedError(f"qk_norm: q_norm.eps {q_norm.eps} != k_norm.eps {k_norm.eps}; the fused kernel takes one eps")


# ------------------------------------------------------------------------------------------------
class FusedAttentionFn(torch.autograd.Function):
    """out[B, N, E] = merge_heads(softmax(q k^T * scale + bias) v) from the qkv planes."""

    @staticmethod
    def forward(ctx, planes, bias_param, bias_mode, bias_grid, scale):
        _require_cuda(planes, bias_param)
        lib = _lib.load()
        _, B, H, N, Dh = planes.shape
        planes = planes.contiguous()
        bp = _f32c(bias_param)
        desc = _bias_desc(bias_mode, bp, bias_grid)
        out = torch.empty(B, N, H * Dh, device=planes.device, dtype=planes.dtype)
        lse = torch.empty(B, H, N, device=planes.device, dtype=torch.float32)
        with torch.cuda.device(planes.device), _timed("attn_fwd"):
            _lib.check(lib.vrr_attn_fwd(_ptr(planes), ctypes.byref(desc), _ptr(out), _ptr(lse), B, H, N, Dh,
                                        float(scale), _DT[planes.dtype], _stream()), "vrr_attn_fwd")
        ctx.save_for_backward(planes, out, lse, bp)
        ctx.meta = (B, H, N, Dh, float(scale), bias_mode, bias_grid,
                    None if bias_param is None else (bias_param.shape, bias_param.dtype))
        return out

    @staticmethod
    def backward(ctx, d_out):
        lib = _lib.load()
        planes, out, lse, bp = ctx.saved_tensors
        B, H, N, Dh, scale, bias_mode, bias_grid, bp_meta = ctx.meta
        d_out = d_out.contiguous()
        dev = planes.device
        desc = _bias_desc(bias_mode, bp, bias_grid)
        d_planes = torch.empty_like(planes)
        d_bp = torch.empty_like(bp) if bp is not None else None
        ws_bytes = int(lib.vrr_attn_bwd_workspace_bytes(B, H, N, Dh, ctypes.byref(desc)))
        ws = torch.empty(ws_bytes, device=dev, dtype=torch.uint8)
        with torch.cuda.device(dev), _timed("attn_bwd"):
            _lib.check(lib.vrr_attn_bwd(_ptr(planes), ctypes.byref(desc), _ptr(out), _ptr(d_out), _ptr(lse),
                                        _ptr(d_planes), _ptr(d_bp), _ptr(ws), ws_bytes, B, H, N, Dh, scale,
                                        _DT[planes.dtype], _stream()), "vrr_attn_bwd")
        if d_bp is not None:
            d_bp = d_bp.view(bp_meta[0]).to(bp_meta[1])
        return d_planes, d_bp, None, None, None


def _bias_desc(mode, param32, grid):
    d = _lib.BiasDesc()
    d.mode = mode
    if mode == _lib.BIAS_NONE:
        d.heads = d.len = d.grid = 0
        d.param = None
        return d
    p2 = param32.reshape(-1, param32.shape[-1])
    d.heads, d.len, d.grid = p2.shape[0], p2.shape[1], int(grid)
    d.param = param32.data_ptr()
    return d


def fused_attention(planes, scale, bias_mode=_lib.BIAS_NONE, bias_param=None, bias_grid=0):
    return FusedAttentionFn.apply(planes, bias_param, bias_mode, bias_grid, scale)


# ------------------------------------------------------------------------------------------------
class LayerNormFn(torch.autograd.Function):
    """y = LayerNorm(x) over the last dim, written directly in the consumer's dtype (fp32 statistics)."""

    @staticmethod
    def forward(ctx, x, weight, bias, eps, out_dtype):
        _require_cuda(x, weight, bias)
        lib = _lib.load()
        E = x.shape[-1]
        x2 = x.contiguous().view(-1, E)
        M = x2.shape[0]
        w32, b32 = _f32c(weight), _f32c(bias)
        y = torch.empty(M, E, device=x.device, dtype=out_dtype)
        mean = torch.empty(M, device=x.device, dtype=torch.float32)
        rstd = torch.empty(M, device=x.device, dtype=torch.float32)
        with torch.cuda.device(x.device), _timed("layernorm_fwd"):
            _lib.check(lib.vrr_layernorm_fwd(_ptr(x2), _ptr(w32), _ptr(b32), _ptr(y), _ptr(mean), _ptr(rstd), M, E,
                                             float(eps), _DT[x2.dtype], _DT[out_dtype], _stream()),
                       "vrr_layernorm_fwd")
        ctx.save_for_backward(x2, w32, mean, rstd)
        ctx.meta = (x.shape, weight.dtype, bias.dtype, out_dtype)
        return y.view(x.shape)

    @staticmethod
    def backward(ctx, dy):
        lib = _lib.load()
        x2, w32, mean, rstd = ctx.saved_tensors
        shape, w_dtype, b_dtype, out_dtype = ctx.meta
        M, E = x2.shape
        dy2 = dy.contiguous().view(M, E)
        if dy2.dtype != out_dtype:
            dy2 = dy2.to(out_dtype)
        dx = torch.empty_like(x2)
        dgb = torch.empty(2, E, device=x2.device, dtype=torch.float32)  # one buffer: zeroed by one memset
        dg, db = dgb[0], dgb[1]
        with torch.cuda.device(x2.device), _timed("layernorm_bwd"):
            _lib.check(lib.vrr_layernorm_bwd(_ptr(dy2), _ptr(x2), _ptr(w32), _ptr(mean), _ptr(rstd), _ptr(dx), _ptr(dg),
                                             _ptr(db), M, E, _DT[x2.dtype], _DT[out_dtype], _stream()),
                       "vrr_layernorm_bwd")
        return dx.view(shape), dg.to(w_dtype), db.to(b_dtype), None, None


# ------------------------------------------------------------------------------------------------
# Dropout / stochastic depth inside the kernels (vrr_drop_desc).  A site is described by the tuple
# ``(p, p_path, rows_per_sample, site, seed)``: element probability, per-image probability, token rows per image, the
# Philox counter word naming the site within one forward, and the int64 device tensor holding the key.  None = off.
def new_seed(device):
    """One 64-bit Philox key drawn on the device from torch's CUDA generator (graph-safe: a captured step draws a
    fresh key on every replay)."""
    return torch.randint(-2 ** 63, 2 ** 63 - 1, (1,), device=device, dtype=torch.int64)


def _drop_desc(drop):
    p, p_path, rows, site, seed = drop
    d = _lib.DropDesc()
    d.p, d.p_path, d.rows_per_sample, d.site = float(p), float(p_path), int(rows), int(site)
    d.seed = seed.data_ptr()
    return d


def drop_scale(p, p_path):
    """The kernels' factor of a kept element: (1 / (1 - p)) * (1 / (1 - p_path)) formed in fp32."""
    one = torch.ones((), dtype=torch.float32)
    return ((one / (one - torch.tensor(p, dtype=torch.float32))) * (one / (one - torch.tensor(p_path, dtype=torch.float32)))).item()


def dropout_mask(drop, M, E):
    """(keep [M, E] uint8 or None when p == 0, keep_path [ceil(M / rows)] uint8 or None when p_path == 0): the
    decisions the kernels take for ``drop`` (``vrr_dropout_mask``)."""
    p, p_path, rows, site, seed = drop
    dev = seed.device
    keep = torch.empty(M, E, device=dev, dtype=torch.uint8) if p > 0 else None
    keep_path = torch.empty(-(-M // rows), device=dev, dtype=torch.uint8) if p_path > 0 else None
    d = _drop_desc(drop)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().vrr_dropout_mask(ctypes.byref(d), _ptr(keep), _ptr(keep_path), M, E, _stream()),
                   "vrr_dropout_mask")
    return keep, keep_path


def branch_factor(drop, B, N, E, cls_only=False):
    """f [B, N, E] fp32 (cls_only: [B, 1, E], token rows b*N): the factor each element of a [B*N, E] branch gets at
    site ``drop`` (keep * keep_path * s), for the residual add the kernels do not take (the model's last one)."""
    p, p_path = drop[0], drop[1]
    keep, keep_path = dropout_mask(drop, B * N, E)
    f = torch.full((B, 1 if cls_only else N, E), drop_scale(p, p_path), device=drop[4].device, dtype=torch.float32)
    if keep is not None:
        k = keep.view(B, N, E)
        f = f * (k[:, :1] if cls_only else k)
    if keep_path is not None:
        f = f * keep_path[:B].view(B, 1, 1)
    return f


class AddLayerNormFn(torch.autograd.Function):
    """(x_new, y) = (x + branch, LayerNorm(x + branch)): the residual add of one sub-block fused with the
    LayerNorm that opens the next one; the backward emits the residual-stream gradient (fp32) and the
    branch gradient (branch dtype) from a single pass.  ``drop``: the branch's dropout / stochastic-depth site
    (x_new = x + f * branch; the masks are regenerated in the backward), or None.  ``ls``: a LayerScale vector [E]
    (x_new = x + (f * branch) * ls, each product rounded to fp32), or None; its gradient is a column reduction of the
    same pass, for which the branch is saved only when ``ls`` needs one."""

    @staticmethod
    def forward(ctx, x, branch, weight, bias, eps, out_dtype, drop=None, ls=None):
        _require_cuda(x, branch, weight, bias)
        lib = _lib.load()
        E = x.shape[-1]
        x2 = x.contiguous().view(-1, E)
        b2 = branch.contiguous().view(-1, E)
        M = x2.shape[0]
        w32, b32 = _f32c(weight), _f32c(bias)
        x_new = torch.empty_like(x2)
        y = torch.empty(M, E, device=x.device, dtype=out_dtype)
        mean = torch.empty(M, device=x.device, dtype=torch.float32)
        rstd = torch.empty(M, device=x.device, dtype=torch.float32)
        ls32 = _f32c(ls)
        with torch.cuda.device(x.device), _timed("add_layernorm_fwd"):
            if ls is not None:
                d = _drop_desc(drop) if drop is not None else None
                _lib.check(lib.vrr_add_layernorm_ls_fwd(_ptr(x2), _ptr(b2), _ptr(x_new), _ptr(w32), _ptr(b32), _ptr(y),
                                                        _ptr(mean), _ptr(rstd), M, E, float(eps), _DT[b2.dtype],
                                                        _DT[out_dtype], ctypes.byref(d) if d is not None else None,
                                                        _ptr(ls32), _stream()), "vrr_add_layernorm_ls_fwd")
            elif drop is None:
                _lib.check(lib.vrr_add_layernorm_fwd(_ptr(x2), _ptr(b2), _ptr(x_new), _ptr(w32), _ptr(b32), _ptr(y),
                                                     _ptr(mean), _ptr(rstd), M, E, float(eps), _DT[b2.dtype],
                                                     _DT[out_dtype], _stream()), "vrr_add_layernorm_fwd")
            else:
                d = _drop_desc(drop)
                _lib.check(lib.vrr_add_layernorm_drop_fwd(_ptr(x2), _ptr(b2), _ptr(x_new), _ptr(w32), _ptr(b32), _ptr(y),
                                                          _ptr(mean), _ptr(rstd), M, E, float(eps), _DT[b2.dtype],
                                                          _DT[out_dtype], ctypes.byref(d), _stream()),
                           "vrr_add_layernorm_drop_fwd")
        ctx.drop = drop  # holds the seed tensor: the backward regenerates the masks from it
        ls_grad = ls is not None and ctx.needs_input_grad[7]
        ctx.save_for_backward(x_new, w32, mean, rstd, ls32, b2 if ls_grad else None)
        ctx.meta = (x.shape, weight.dtype, bias.dtype, out_dtype, b2.dtype, None if ls is None else ls.dtype)
        return x_new.view(x.shape), y.view(x.shape)

    @staticmethod
    def backward(ctx, d_xnew, d_y):
        lib = _lib.load()
        x_new, w32, mean, rstd, ls32, b2 = ctx.saved_tensors
        shape, w_dtype, b_dtype, out_dtype, br_dtype, ls_dtype = ctx.meta
        M, E = x_new.shape
        if d_y is None:
            d_y = torch.zeros(M, E, device=x_new.device, dtype=out_dtype)
        dy2 = d_y.contiguous().view(M, E)
        if dy2.dtype != out_dtype:
            dy2 = dy2.to(out_dtype)
        dr2 = None
        if d_xnew is not None:
            dr2 = d_xnew.contiguous().view(M, E)
            if dr2.dtype != torch.float32:
                dr2 = dr2.float()
        dx = torch.empty_like(x_new)
        d_branch = torch.empty(M, E, device=x_new.device, dtype=br_dtype)
        # one buffer: the library zeroes its rows (gamma, beta and the LayerScale gradient) with one memset
        dgb = torch.empty(2 if b2 is None else 3, E, device=x_new.device, dtype=torch.float32)
        dg, db = dgb[0], dgb[1]
        d_ls = dgb[2] if b2 is not None else None
        with torch.cuda.device(x_new.device), _timed("add_layernorm_bwd"):
            if ls32 is not None:
                d = _drop_desc(ctx.drop) if ctx.drop is not None else None
                _lib.check(lib.vrr_add_layernorm_ls_bwd(_ptr(dy2), _ptr(dr2), _ptr(x_new), _ptr(w32), _ptr(mean),
                                                        _ptr(rstd), _ptr(dx), _ptr(d_branch), _ptr(dg), _ptr(db), M, E,
                                                        _DT[br_dtype], _DT[out_dtype],
                                                        ctypes.byref(d) if d is not None else None, _ptr(ls32),
                                                        _ptr(b2), _ptr(d_ls), _stream()), "vrr_add_layernorm_ls_bwd")
            elif ctx.drop is None:
                _lib.check(lib.vrr_add_layernorm_bwd(_ptr(dy2), _ptr(dr2), _ptr(x_new), _ptr(w32), _ptr(mean), _ptr(rstd),
                                                     _ptr(dx), _ptr(d_branch), _ptr(dg), _ptr(db), M, E, _DT[br_dtype],
                                                     _DT[out_dtype], _stream()), "vrr_add_layernorm_bwd")
            else:
                d = _drop_desc(ctx.drop)
                _lib.check(lib.vrr_add_layernorm_drop_bwd(_ptr(dy2), _ptr(dr2), _ptr(x_new), _ptr(w32), _ptr(mean),
                                                          _ptr(rstd), _ptr(dx), _ptr(d_branch), _ptr(dg), _ptr(db), M, E,
                                                          _DT[br_dtype], _DT[out_dtype], ctypes.byref(d), _stream()),
                           "vrr_add_layernorm_drop_bwd")
        return (dx.view(shape), d_branch.view(shape), dg.to(w_dtype), db.to(b_dtype), None, None, None,
                None if d_ls is None else d_ls.to(ls_dtype))


def can_fuse_add_layer_norm(x, norm) -> bool:
    """The fused add+LayerNorm kernels need an fp32 residual stream and a plain affine last-dim LayerNorm."""
    return (x.is_cuda and x.dtype == torch.float32 and type(norm) is torch.nn.LayerNorm and norm.elementwise_affine
            and norm.bias is not None and tuple(norm.normalized_shape) == (x.shape[-1],))


def add_layer_norm(x, branch, norm: torch.nn.LayerNorm, drop=None, ls=None):
    """``x_new = x + (f * branch) * ls; y = norm(x_new)`` in one kernel (see :class:`AddLayerNormFn`); f = 1 when
    ``drop`` is None, and no LayerScale product when ``ls`` (a LayerScale's ``gamma`` [E]) is None."""
    out_dtype = compute_dtype(x)
    if branch.dtype not in (torch.float32, out_dtype):
        branch = branch.to(out_dtype)
    return AddLayerNormFn.apply(x, branch, norm.weight, norm.bias, norm.eps, out_dtype, drop, ls)


def layer_norm(x, norm: torch.nn.LayerNorm):
    """``norm(x)`` for an ``nn.LayerNorm`` over the last dimension, output in the compute dtype
    (bf16 / fp16 under autocast: the reference's LayerNorm-then-cast, fused).  Falls through to the module
    itself for anything that is not a plain affine last-dim LayerNorm (a caller-supplied norm_layer)."""
    if (type(norm) is not torch.nn.LayerNorm or not norm.elementwise_affine or norm.bias is None
            or tuple(norm.normalized_shape) != (x.shape[-1],)):
        return norm(x)
    out_dtype = compute_dtype(x)
    if x.dtype in _LP16 and out_dtype != x.dtype:
        x = x.float()
    return LayerNormFn.apply(x, norm.weight, norm.bias, norm.eps, out_dtype)


# ------------------------------------------------------------------------------------------------
def _colsum(t2d):
    lib = _lib.load()
    M, C = t2d.shape
    out = torch.empty(C, device=t2d.device, dtype=torch.float32)
    _lib.check(lib.vrr_colsum(_ptr(t2d), _ptr(out), M, C, _DT[t2d.dtype], _stream()), "vrr_colsum")
    return out


class LinearFn(torch.autograd.Function):
    """y = x W^T + b (out-proj / head, models/vit.py:91,285).  bf16 / fp16: forward GEMM with the bias in its
    epilogue, dX and dW (fp32, straight into the master-weight gradient) on the tcgen05 CTA-pair kernel;
    bias gradient on the column-sum kernel.  ``w`` / ``b`` receive the gradients (fp32 masters or tensors in
    x's dtype); ``w_lp`` is an optional ready-made copy of ``w`` in x's dtype."""

    @staticmethod
    def forward(ctx, x, w, b, w_lp=None):
        _require_cuda(x, w, b)
        dt = x.dtype
        wl = (w_lp if w_lp is not None else w.detach().to(dt)).detach()
        x2 = x.reshape(-1, x.shape[-1])
        y = _gemm(x2, wl, False, True, dt, bias=b, epilogue=_lib.EPI_BIAS if b is not None else _lib.EPI_NONE,
                  name="linear_fwd")
        ctx.save_for_backward(x2, wl)
        ctx.meta = (x.shape, w.dtype, None if b is None else b.dtype)
        return y.view(*x.shape[:-1], wl.shape[0])

    @staticmethod
    def backward(ctx, dy):
        x2, wl = ctx.saved_tensors
        x_shape, w_dtype, b_dtype = ctx.meta
        dy2 = dy.contiguous().view(-1, dy.shape[-1])
        if dy2.dtype != x2.dtype:
            dy2 = dy2.to(x2.dtype)
        dx = dw = db = None
        with torch.cuda.device(dy.device):
            if ctx.needs_input_grad[0]:
                dx = _gemm(dy2, wl, False, False, x2.dtype, name="linear_dx").view(x_shape)
            if ctx.needs_input_grad[1]:
                dw = _gemm(dy2, x2, True, False, w_dtype, name="linear_dw")
            if b_dtype is not None and ctx.needs_input_grad[2]:
                with _timed("colsum"):
                    db = _colsum(dy2).to(b_dtype)
        return dx, dw, db, None


_FUSE_DB1 = os.environ.get("VRR_FUSE_DB1", "1") != "0"  # A/B switch: fc1's bias gradient inside fc2's dX GEMM


class MlpFn(torch.autograd.Function):
    """fc1 -> exact GELU -> fc2 (timm Mlp, models/vit.py:118).  fc1's GEMM epilogue adds the bias and writes BOTH
    gelu(h) and gelu'(h) (h itself is never stored: the backward only needs the derivative); fc2 adds its bias.
    Backward = four GEMMs on the same kernel (dW in fp32); the GELU backward is the epilogue of fc2's dX GEMM
    (dh = (dy . W2) * gelu'(h)), the two bias gradients are column sums."""

    @staticmethod
    def forward(ctx, x, w1, b1, w2, b2, w1_lp=None, w2_lp=None, drop1=None):
        """``drop1``: element dropout on the GELU output (a site with p_path 0), applied in fc1's epilogue to gelu(h)
        and gelu'(h) alike - the backward below is then Dropout's backward unchanged."""
        _require_cuda(x, w1, b1, w2, b2)
        dt = x.dtype
        w1l = (w1_lp if w1_lp is not None else w1.detach().to(dt)).detach()
        w2l = (w2_lp if w2_lp is not None else w2.detach().to(dt)).detach()
        x2 = x.reshape(-1, x.shape[-1])
        if not any(ctx.needs_input_grad):  # inference: the activation alone - one output stream instead of two
            a = _gemm(x2, w1l, False, True, dt, bias=b1, epilogue=_lib.EPI_BIAS_GELU_ACT, name="fc1_fwd", drop=drop1)
            y = _gemm(a, w2l, False, True, dt, bias=b2, epilogue=_lib.EPI_BIAS, name="fc2_fwd")
            return y.view(*x.shape[:-1], w2l.shape[0])
        a, gp = _gemm(x2, w1l, False, True, dt, bias=b1, epilogue=_lib.EPI_BIAS_GELU_GRAD, out2=True, name="fc1_fwd",
                      drop=drop1)
        y = _gemm(a, w2l, False, True, dt, bias=b2, epilogue=_lib.EPI_BIAS, name="fc2_fwd")
        ctx.save_for_backward(x2, gp, a, w1l, w2l)
        ctx.meta = (x.shape, w1.dtype, b1.dtype, w2.dtype, b2.dtype)
        return y.view(*x.shape[:-1], w2l.shape[0])

    @staticmethod
    def backward(ctx, dy):
        x2, gp, a2, w1l, w2l = ctx.saved_tensors
        x_shape, w1_dt, b1_dt, w2_dt, b2_dt = ctx.meta
        dy2 = dy.contiguous().view(-1, dy.shape[-1])
        if dy2.dtype != x2.dtype:
            dy2 = dy2.to(x2.dtype)
        with torch.cuda.device(dy.device):
            # dh = (dy . W2) * gelu'(h) with fc1's bias gradient (column sums of dh as stored, like autograd's sum
            # over the rounded tensor) accumulated by the same GEMM's epilogue
            if _FUSE_DB1:
                lib = _lib.load()
                M, N, K = dy2.shape[0], w2l.shape[1], dy2.shape[1]
                dh = torch.empty(M, N, device=dy2.device, dtype=x2.dtype)
                db1 = torch.empty(N, device=dy2.device, dtype=torch.float32)
                with _timed("fc2_dx"):
                    _lib.check(lib.vrr_gemm_mul_colsum(_ptr(dy2), _ptr(w2l), _ptr(dh), _ptr(gp), _ptr(db1), M, N, K, 0, 0,
                                                       _DT[x2.dtype], _stream()), "vrr_gemm_mul_colsum")
                db1 = db1.to(b1_dt)
            else:
                dh = _gemm(dy2, w2l, False, False, x2.dtype, epilogue=_lib.EPI_MUL, aux=gp, name="fc2_dx")
                with _timed("colsum"):
                    db1 = _colsum(dh).to(b1_dt)
            dw2 = _gemm(dy2, a2, True, False, w2_dt, name="fc2_dw")
            with _timed("colsum"):
                db2 = _colsum(dy2).to(b2_dt)
            dx = _gemm(dh, w1l, False, False, x2.dtype, name="fc1_dx").view(x_shape)
            dw1 = _gemm(dh, x2, True, False, w1_dt, name="fc1_dw")
        return dx, dw1, db1, dw2, db2, None, None, None


def linear(x, lin: torch.nn.Linear, w_lp=None):
    """``lin(x)`` through :class:`LinearFn` (CUDA, bias, supported dtype, width % 4 == 0) else the module."""
    if not (x.is_cuda and lin.bias is not None and lin.out_features % 4 == 0 and x.dtype in _DT):
        return lin(x)
    dt = compute_dtype(x)
    if w_lp is not None and w_lp.dtype != dt:
        w_lp = None
    return LinearFn.apply(x.to(dt), lin.weight, lin.bias, w_lp)


def mlp(x, fc1: torch.nn.Linear, fc2: torch.nn.Linear, w1_lp=None, w2_lp=None, drop1=None):
    dt = compute_dtype(x)
    if w1_lp is not None and (w1_lp.dtype != dt or w2_lp is None or w2_lp.dtype != dt):
        w1_lp = w2_lp = None
    return MlpFn.apply(x.to(dt), fc1.weight, fc1.bias, fc2.weight, fc2.bias, w1_lp, w2_lp, drop1)


def can_fuse_mlp(x, m) -> bool:
    """fc1 -> exact GELU -> fc2 with biases; fc1's dropout (drop1) runs in its epilogue when its hidden width is a
    multiple of 8 (the mask's groups), and the caller applies drop2 (nn.Dropout, or the next add+LayerNorm)."""
    act = getattr(m, "act", None)
    p1 = getattr(m.drop1, "p", 0.0) if isinstance(m.drop1, torch.nn.Dropout) else None
    return (x.is_cuda and x.dtype in _DT and type(act) is torch.nn.GELU and getattr(act, "approximate", "none") == "none"
            and m.fc1.bias is not None and m.fc2.bias is not None and m.fc1.out_features % 4 == 0
            and m.fc2.out_features % 4 == 0 and p1 is not None and (p1 == 0.0 or m.fc1.out_features % 8 == 0)
            and isinstance(m.drop2, (torch.nn.Dropout, torch.nn.Identity)))


class SwiGLUMlpFn(torch.autograd.Function):
    """fc1 -> SwiGLU -> fc2 (timm ``SwiGLUPacked``: ``fc2(silu(x W_g^T + b_g) * (x W_v^T + b_v))``, fc1.weight holding
    the gate rows then the value rows).  fc1's GEMM pairs each gate column with its value column and writes the
    activation and both partial derivatives (``vrr_gemm_swiglu``); fc2 adds its bias.  Backward: fc2's dX GEMM applies
    the SwiGLU backward and sums fc1's bias gradient (``vrr_gemm_swiglu_bwd``); dW2, dX and dW1 are plain GEMMs."""

    @staticmethod
    def forward(ctx, x, w1, b1, w2, b2, w1_lp=None, w2_lp=None, drop1=None):
        """``drop1``: element dropout on the activation (a site with p_path 0), applied in fc1's epilogue to the
        activation and to both derivatives - the backward is then Dropout's backward unchanged."""
        _require_cuda(x, w1, b1, w2, b2)
        lib = _lib.load()
        dt = x.dtype
        w1l = (w1_lp if w1_lp is not None else w1.detach().to(dt)).detach().contiguous()
        w2l = (w2_lp if w2_lp is not None else w2.detach().to(dt)).detach().contiguous()
        x2 = x.reshape(-1, x.shape[-1]).contiguous()
        M, K, H = x2.shape[0], x2.shape[1], w1l.shape[0] // 2
        b1_32 = _f32c(b1)
        grad = any(ctx.needs_input_grad)
        act = torch.empty(M, H, device=x.device, dtype=dt)
        aux = torch.empty(M, 2 * H, device=x.device, dtype=dt) if grad else None  # inference: the activation alone
        d = _drop_desc(drop1) if drop1 is not None else None
        with torch.cuda.device(x.device), _timed("fc1_fwd"):
            _lib.check(lib.vrr_gemm_swiglu(_ptr(x2), _ptr(w1l), _ptr(b1_32), _ptr(act), _ptr(aux), M, H, K, _DT[dt],
                                           ctypes.byref(d) if d is not None else None, _stream()), "vrr_gemm_swiglu")
        y = _gemm(act, w2l, False, True, dt, bias=b2, epilogue=_lib.EPI_BIAS, name="fc2_fwd")
        if grad:
            ctx.save_for_backward(x2, aux, act, w1l, w2l)
            ctx.meta = (x.shape, w1.dtype, b1.dtype, w2.dtype, b2.dtype)
        return y.view(*x.shape[:-1], w2l.shape[0])

    @staticmethod
    def backward(ctx, dy):
        x2, aux, act, w1l, w2l = ctx.saved_tensors
        x_shape, w1_dt, b1_dt, w2_dt, b2_dt = ctx.meta
        lib = _lib.load()
        dy2 = dy.contiguous().view(-1, dy.shape[-1])
        if dy2.dtype != x2.dtype:
            dy2 = dy2.to(x2.dtype)
        M, K, H = dy2.shape[0], dy2.shape[1], act.shape[1]
        with torch.cuda.device(dy.device):
            dh = torch.empty(M, 2 * H, device=dy2.device, dtype=x2.dtype)
            db1 = torch.empty(2 * H, device=dy2.device, dtype=torch.float32)
            with _timed("fc2_dx"):
                _lib.check(lib.vrr_gemm_swiglu_bwd(_ptr(dy2), _ptr(w2l), _ptr(aux), _ptr(dh), _ptr(db1), M, H, K,
                                                   _DT[x2.dtype], _stream()), "vrr_gemm_swiglu_bwd")
            dw2 = _gemm(dy2, act, True, False, w2_dt, name="fc2_dw")
            with _timed("colsum"):
                db2 = _colsum(dy2).to(b2_dt)
            dx = _gemm(dh, w1l, False, False, x2.dtype, name="fc1_dx").view(x_shape)
            dw1 = _gemm(dh, x2, True, False, w1_dt, name="fc1_dw")
        return dx, dw1, db1.to(b1_dt), dw2, db2, None, None, None


def swiglu_mlp(x, fc1: torch.nn.Linear, fc2: torch.nn.Linear, w1_lp=None, w2_lp=None, drop1=None):
    dt = compute_dtype(x)
    if w1_lp is not None and (w1_lp.dtype != dt or w2_lp is None or w2_lp.dtype != dt):
        w1_lp = w2_lp = None
    return SwiGLUMlpFn.apply(x.to(dt), fc1.weight, fc1.bias, fc2.weight, fc2.bias, w1_lp, w2_lp, drop1)


def can_fuse_swiglu(x, m) -> bool:
    """timm's SwiGLUPacked: SiLU on the first half of fc1's output (gate_last False), no norm inside, both biases; the
    hidden width H is even and fc2's output width a multiple of 4 (the bias-gradient kernels), and H % 8 == 0 when
    drop1 is on (the mask's groups).  The caller applies drop2."""
    p1 = getattr(m.drop1, "p", 0.0) if isinstance(m.drop1, torch.nn.Dropout) else None
    H = m.fc1.out_features // 2
    return (x.is_cuda and x.dtype in _DT and type(m.act) is torch.nn.SiLU and not m.gate_last
            and type(m.norm) is torch.nn.Identity and m.fc1.bias is not None and m.fc2.bias is not None
            and m.fc1.out_features % 2 == 0 and H % 2 == 0 and m.fc2.in_features == H and m.fc2.out_features % 4 == 0
            and p1 is not None and (p1 == 0.0 or H % 8 == 0) and isinstance(m.drop2, (torch.nn.Dropout, torch.nn.Identity)))


# ------------------------------------------------------------------------------------------------
class RopeApplyFn(torch.autograd.Function):
    """Stand-alone rotate-half of q and k (public ``apply_rotary_emb``, rope_utils.py:3-37)."""

    @staticmethod
    def forward(ctx, q, k, cos, sin):
        _require_cuda(q, k, cos, sin)
        lib = _lib.load()
        B, H, Nr, Dh = q.shape
        cos_b = torch.broadcast_to(cos, (1, cos.shape[1], Nr, Dh // 2))[0] if cos.ndim == 4 else cos
        sin_b = torch.broadcast_to(sin, (1, sin.shape[1], Nr, Dh // 2))[0] if sin.ndim == 4 else sin
        if cos_b.ndim == 3 and cos_b.shape[0] == 1:
            cos_b, sin_b = cos_b[0], sin_b[0]
        mode = _lib.ROPE_AXIAL if cos_b.ndim == 2 else _lib.ROPE_MIXED
        want = (Nr, Dh // 2) if mode == _lib.ROPE_AXIAL else (H, Nr, Dh // 2)
        if tuple(cos_b.shape) != want or tuple(sin_b.shape) != want:
            raise RuntimeError(f"cos/sin {tuple(cos.shape)} do not broadcast against q {tuple(q.shape)}")
        q, k = q.contiguous(), k.contiguous()
        c32, s32 = _f32c(cos_b), _f32c(sin_b)
        qo, ko = torch.empty_like(q), torch.empty_like(k)
        with torch.cuda.device(q.device):
            _lib.check(lib.vrr_rope_apply(_ptr(q), _ptr(k), _ptr(c32), _ptr(s32), _ptr(qo), _ptr(ko), B, H, Nr, Dh,
                                          mode, 0, _DT[q.dtype], _stream()), "vrr_rope_apply")
        need_tab = ctx.needs_input_grad[2] or ctx.needs_input_grad[3]
        ctx.save_for_backward(c32, s32, *((q, k) if need_tab else ()))
        ctx.meta = (B, H, Nr, Dh, mode, cos.shape, sin.shape, cos.dtype, sin.dtype)
        return qo, ko

    @staticmethod
    def backward(ctx, dq, dk):
        lib = _lib.load()
        c32, s32 = ctx.saved_tensors[:2]
        B, H, Nr, Dh, mode, cos_shape, sin_shape, cos_dt, sin_dt = ctx.meta
        dq, dk = dq.contiguous(), dk.contiguous()
        gq, gk = torch.empty_like(dq), torch.empty_like(dk)
        d_cos = d_sin = None
        with torch.cuda.device(dq.device):
            _lib.check(lib.vrr_rope_apply(_ptr(dq), _ptr(dk), _ptr(c32), _ptr(s32), _ptr(gq), _ptr(gk), B, H, Nr,
                                          Dh, mode, 1, _DT[dq.dtype], _stream()), "vrr_rope_apply")
            if len(ctx.saved_tensors) == 4:  # the tables are differentiable too (RoPEMixed.freqs feeds them)
                q, k = ctx.saved_tensors[2:]
                d_cos, d_sin = torch.empty_like(c32), torch.empty_like(s32)
                _lib.check(lib.vrr_rope_table_grad(_ptr(q), _ptr(k), _ptr(dq), _ptr(dk), _ptr(d_cos), _ptr(d_sin), B, H,
                                                   Nr, Dh, mode, _DT[dq.dtype], _stream()), "vrr_rope_table_grad")
                # undo the broadcast of reshape_for_broadcast: sum_to_size restores [1, 1|H, Nr, Dh/2] / the raw shape
                d_cos = d_cos.reshape((1,) * (len(cos_shape) - d_cos.ndim) + tuple(d_cos.shape)).sum_to_size(cos_shape).to(cos_dt)
                d_sin = d_sin.reshape((1,) * (len(sin_shape) - d_sin.ndim) + tuple(d_sin.shape)).sum_to_size(sin_shape).to(sin_dt)
        return gq, gk, (d_cos if ctx.needs_input_grad[2] else None), (d_sin if ctx.needs_input_grad[3] else None)
