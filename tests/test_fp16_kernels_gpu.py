"""The fp16 instantiations of the kernels, through the C ABI (VRR_F16), with the conventions of test_kernels_at_scale.py
and test_streaming_kernels_at_scale.py: every output pre-filled with NaN, shapes sized from the SM count so that a
GEMM cluster takes >= 4 units and an attention CTA >= 3 items, and every head-dim-64 case asserting through
vrr_family_count that the tcgen05 family ran.

* GEMMs with small-integer operands are exact in fp16 and in fp32 accumulation, so their results are compared BIT FOR
  BIT with the float64 product rounded once by numpy's ``astype(np.float16)``.
* Attention is checked per item against float64 torch with bounds of a few fp16 unit roundoffs (2^-11), where the bf16
  tests use 2^-8, set from the worst errors measured on a B200 (out 1.4, d_planes 1.9 unit roundoffs): rounding P,
  dS or the output to bf16 in the fp16 kernels moves out / d_planes to 2.1e-3 .. 3.9e-3 and fails them.
* fp16 overflows must come out as +-inf (torch.amp.GradScaler skips a step on them), never as a clamped 65504.
"""
import ctypes

import numpy as np
import pytest
import torch

from test_kernels_at_scale import (LAYOUTS, _bias_case, _clusters, _dparam_ref, _gelu64, _m_for_units, _p,
                                   _per_item, _pick_splits, _ref, _regime_shape, _sms, _st, _tiles)
from test_parity_gpu import report, tcgen05_must_run
from test_streaming_kernels_at_scale import _rope_ref_bwd
from vit_rpe_rope_b200 import _lib

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
HF = torch.float16
NAN = float("nan")
U16 = 2.0 ** -11  # fp16 unit roundoff


def _lib_():
    return _lib.load()


def _ints(shape, r, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randint(-r, r + 1, shape, generator=g, device=DEV).to(HF)


def _acc64(a, b, ta, tb):
    acc = (a.t() if ta else a).double() @ (b.t() if tb else b).double()
    assert acc.abs().max().item() < 2 ** 22
    return acc


def _to16(x64):
    """float64 -> fp16 with numpy's single rounding (the documented rounding of the kernels)."""
    return torch.from_numpy(x64.cpu().numpy().astype(np.float16)).to(DEV)


def _gemm(a, b, c, m, n, k, ta, tb, c_dtype, epi=_lib.EPI_NONE, c2=None, bias=None):
    return _lib_().vrr_gemm_ex(_p(a), _p(b), _p(c), _p(c2), _p(bias), m, n, k, ta, tb, _lib.VRR_F16, c_dtype, epi, 0,
                               _st())


def _check_exact(m, n, k, ta, tb, c_f32, epi=_lib.EPI_NONE, seed=0):
    a = _ints((k, m) if ta else (m, k), 1 if k > 1000 else 3, seed)
    b = _ints((n, k) if tb else (k, n), 1 if k > 1000 else 3, seed + 1)
    bias = ((torch.arange(n, device=DEV) % 7) - 3).float() + 1.0 / 3.0 if epi == _lib.EPI_BIAS else None
    c = torch.full((m, n), NAN, device=DEV, dtype=torch.float32 if c_f32 else HF)
    rc = _gemm(a, b, c, m, n, k, ta, tb, _lib.VRR_F32 if c_f32 else _lib.VRR_F16, epi, bias=bias)
    assert rc == 0, _lib.last_error()
    want = _acc64(a, b, ta, tb)
    if bias is not None:  # the bias is cast to fp16 first (F.linear on fp16 tensors)
        want = want + bias.to(HF).double()
    want = want.float() if c_f32 else _to16(want)
    if not torch.equal(c, want):
        bad = (c != want).nonzero()[0].tolist()
        return f"M {m} N {n} K {k} trans {ta}{tb} c_f32 {c_f32} epi {epi}: first difference at {bad}"
    return None


# ------------------------------------------------------------------------------------------------ GEMM

@pytest.mark.parametrize("c_f32", [0, 1])
@pytest.mark.parametrize("ta,tb", LAYOUTS)
def test_fp16_gemm_integer_exact_ragged(ta, tb, c_f32):
    """Every layout x C type at ragged M and across the BN 128 -> 256 switch (N 128 / 136), plain and BIAS."""
    ms = [248, 264] if ta else [255, 257]
    failures = []
    with tcgen05_must_run():
        for m in ms:
            for n in (128, 136, 264):
                for k in (72, 520):
                    for epi in (_lib.EPI_NONE, _lib.EPI_BIAS):
                        msg = _check_exact(m, n, k, ta, tb, c_f32, epi, seed=m + n + k)
                        if msg:
                            failures.append(msg)
    assert not failures, "\n".join(failures[:10])


@pytest.mark.parametrize("ta,tb", LAYOUTS)
def test_fp16_gemm_integer_exact_many_units(ta, tb):
    """>= 4 work units per cluster, fp16 C, plain and BIAS: the whole output bit for bit."""
    n, k = 768, 768
    m = _m_for_units(n, 4)
    assert _tiles(m, n) >= 4 * _clusters()
    with tcgen05_must_run():
        for epi in (_lib.EPI_NONE, _lib.EPI_BIAS):
            msg = _check_exact(m, n, k, ta, tb, 0, epi, seed=3)
            assert msg is None, msg


@pytest.mark.parametrize("regime", ["no_split", "split_one_wave", "split_multi_wave"])
def test_fp16_gemm_fp32_split_k_regimes_exact(regime):
    """fp32 C (weight gradients) in each split-K regime of pick_splits: partial sums reduce-added, still exact."""
    m, n, k = _regime_shape(regime)
    splits = _pick_splits(_tiles(m, n), -(-k // 64), _clusters())
    assert (splits == 1) == (regime == "no_split")
    with tcgen05_must_run():
        msg = _check_exact(m, n, k, 1, 0, 1, seed=11)
    assert msg is None, msg


def test_fp16_gemm_mul_colsum_exact():
    """MUL epilogue (fc2's dX with gelu') and the fused fp32 column sums of the fp16 values as stored."""
    n, k = 768, 256
    m = _m_for_units(n, 4)
    a, b = _ints((m, k), 2, 21), _ints((k, n), 2, 22)
    mul = _ints((m, n), 2, 23)
    c = torch.full((m, n), NAN, device=DEV, dtype=HF)
    cs = torch.full((n,), NAN, device=DEV)
    with tcgen05_must_run():
        _lib.check(_lib_().vrr_gemm_mul_colsum(_p(a), _p(b), _p(c), _p(mul), _p(cs), m, n, k, 0, 0, _lib.VRR_F16, _st()),
                   "gemm_mul_colsum")
    want = _to16(_acc64(a, b, 0, 0) * mul.double())
    assert torch.equal(c, want)
    assert torch.equal(cs.double(), want.double().sum(0))  # |sums| < 2^24: exact in any order


def test_fp16_qkv_and_patch_embed_direct_stores_exact():
    """The direct-store epilogues: QKV planes (no RoPE) and the patch-embedding tokens (fp32 images rounded to fp16 on
    load, fp32 token stream, absolute pos added after the fp16 rounding)."""
    lib = _lib_()
    b, n, e, h = -(-4 * _clusters() * 256 // 197) // 3 + 1, 197, 192, 3
    x = _ints((b * n, e), 2, 31)
    w = _ints((3 * e, e), 2, 32)
    planes = torch.full((3, b, h, n, 64), NAN, device=DEV, dtype=HF)
    with tcgen05_must_run():
        _lib.check(lib.vrr_qkv_rope_fwd(_p(x), _p(w), None, None, _p(planes), b, n, e, h, _lib.ROPE_NONE, _lib.VRR_F16,
                                        _st()), "qkv_rope_fwd")
    want = _to16(x.double() @ w.double().t()).view(b, n, 3, h, 64).permute(2, 0, 3, 1, 4)
    assert torch.equal(planes, want)

    bsz, c, size, p, e = 16 * _clusters(), 3, 64, 8, 128  # 64 tokens per image: >= 4 units per cluster
    g = torch.Generator(device=DEV).manual_seed(33)
    img = torch.randint(-8, 9, (bsz, c, size, size), generator=g, device=DEV).float() / 4 + 1.0 / 3.0  # off the fp16 grid
    wt = _ints((e, c, p, p), 1, 34)
    bias = _ints((e,), 3, 35)
    cls = torch.randn(e, device=DEV)
    pos = torch.randint(-4, 5, (64, e), generator=g, device=DEV).float() / 8
    np_ = (size // p) ** 2
    tok = torch.full((bsz, np_ + 1, e), NAN, device=DEV)
    ws_bytes = lib.vrr_patch_embed_workspace_bytes(bsz, c, size, size, p, e, _lib.VRR_F16)
    assert ws_bytes > 0
    ws = torch.empty(ws_bytes, device=DEV, dtype=torch.uint8)
    with tcgen05_must_run():
        _lib.check(lib.vrr_patch_embed_fwd(_p(img), _p(wt), _p(bias), _p(cls), _p(pos), _p(tok), _p(ws), ws_bytes, bsz, c,
                                           size, size, p, e, _lib.VRR_F32, _lib.VRR_F16, _lib.VRR_F32, _st()),
                   "patch_embed_fwd")
    unf = img.to(HF).double().unfold(2, p, p).unfold(3, p, p).permute(0, 2, 3, 1, 4, 5).reshape(bsz * np_, c * p * p)
    conv = _to16(unf @ wt.double().reshape(e, -1).t() + bias.double()).float().view(bsz, np_, e)
    assert torch.equal(tok[:, 1:], conv + pos[:np_])
    assert torch.equal(tok[:, 0], cls.expand(bsz, e))
    # the workspace is unfold(images) in fp16, and vrr_patch_unfold_ex reproduces it
    unf2 = torch.full((bsz * np_, c * p * p), NAN, device=DEV, dtype=HF)
    _lib.check(lib.vrr_patch_unfold_ex(_p(img), _p(unf2), bsz, c, size, size, p, _lib.VRR_F32, _lib.VRR_F16, _st()),
               "patch_unfold_ex")
    assert torch.equal(unf2, ws.view(HF).view_as(unf2)) and torch.equal(unf2.double(), unf)


def _fp16_ulp(y):
    y = y.double().abs()
    _, e = torch.frexp(y.clamp_min(2.0 ** -14))
    return torch.ldexp(torch.ones_like(y), (e - 11).to(torch.int64))  # 2^-24 below the normal range


def test_fp16_gelu_epilogue_sweep_vs_float64():
    """BIAS_GELU / BIAS_GELU_GRAD / BIAS_GELU_ACT over every normal fp16 h in [-8, 8] (acc = h exactly): h back bit for
    bit; gelu(h), gelu'(h) within one fp16 ulp plus the method's error (A&S 7.1.26 |d erfc| <= 1.5e-7, i.e. a few fp16
    ulps of the tiny far-negative-tail results, fp32 rcp / ex2 approximations); the three epilogues agree."""
    bits = torch.arange(0x0400, 0x4801, dtype=torch.int32)  # 2^-14 .. 8.0
    pos = bits.to(torch.int16).view(HF)
    hv = torch.cat([torch.zeros(1, dtype=HF), pos, -pos]).to(DEV)
    m, n, k = hv.numel(), 8, 8
    a = torch.zeros(m, k, device=DEV, dtype=HF)
    a[:, 0] = hv
    b = torch.zeros(n, k, device=DEV, dtype=HF)
    b[:, 0] = 1.0
    bias = torch.zeros(n, device=DEV)
    outs = {}
    with tcgen05_must_run():
        for epi in (_lib.EPI_BIAS_GELU, _lib.EPI_BIAS_GELU_GRAD, _lib.EPI_BIAS_GELU_ACT):
            c = torch.full((m, n), NAN, device=DEV, dtype=HF)
            c2 = torch.full((m, n), NAN, device=DEV, dtype=HF)
            _lib.check(_gemm(a, b, c, m, n, k, 0, 1, _lib.VRR_F16, epi, c2=c2, bias=bias), f"epilogue {epi}")
            outs[epi] = (c, c2)
    h_out, gelu_a = outs[_lib.EPI_BIAS_GELU]
    gelu_b, dgelu = outs[_lib.EPI_BIAS_GELU_GRAD]
    assert torch.equal(h_out, hv[:, None].expand(m, n))
    assert torch.equal(gelu_a, gelu_b) and torch.equal(outs[_lib.EPI_BIAS_GELU_ACT][0], gelu_b)
    g, dg, cdf, pdf = _gelu64(hv.float())
    ah, tail = hv.double().abs(), torch.minimum(cdf, 1.0 - cdf)
    bg = _fp16_ulp(g) + ah * (0.75e-7 + 2.0 ** -21 * tail + 2.0 ** -23)
    bdg = _fp16_ulp(dg) + 0.75e-7 + 2.0 ** -21 * (tail + ah * pdf) + 2.0 ** -23
    eg, edg = (gelu_b[:, 0].double() - g).abs(), (dgelu[:, 0].double() - dg).abs()
    ulps_g, ulps_dg = (eg / _fp16_ulp(g)).max().item(), (edg / _fp16_ulp(dg)).max().item()
    rg, rdg = (eg / bg).max().item(), (edg / bdg).max().item()
    report(f"fp16 gelu sweep ({m} values): gelu worst {ulps_g:.2f} fp16 ulp ({rg:.2f} of bound), gelu' worst "
           f"{ulps_dg:.2f} ulp ({rdg:.2f} of bound)")
    worst = int((eg / bg).argmax())
    assert rg <= 1.0, ("gelu", hv[worst].item(), gelu_b[worst, 0].item(), g[worst].item())
    worst = int((edg / bdg).argmax())
    assert rdg <= 1.0, ("gelu'", hv[worst].item(), dgelu[worst, 0].item(), dg[worst].item())


# ------------------------------------------------------------------------------------------------ attention

def _planes(b, h, n, seed, dh=64):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randn(3, b, h, n, dh, generator=g, device=DEV) * 0.8).to(HF)


def _fwd(planes, desc):
    _, b, h, n, dh = planes.shape
    out = torch.full((b, n, h * dh), NAN, device=DEV, dtype=HF)
    lse = torch.full((b, h, n), NAN, device=DEV)
    _lib.check(_lib_().vrr_attn_fwd(_p(planes), None if desc is None else ctypes.byref(desc), _p(out), _p(lse), b, h, n,
                                    dh, ctypes.c_float(dh ** -0.5), _lib.VRR_F16, _st()), "attn_fwd")
    return out, lse


def _bwd(planes, desc, param, out, d_out, lse):
    lib = _lib_()
    _, b, h, n, dh = planes.shape
    dref = None if desc is None else ctypes.byref(desc)
    ws_bytes = lib.vrr_attn_bwd_workspace_bytes(b, h, n, dh, dref)
    ws = torch.empty(ws_bytes, device=DEV, dtype=torch.uint8)
    d_planes = torch.full_like(planes, NAN)
    d_param = None if param is None else torch.full_like(param, NAN)
    _lib.check(lib.vrr_attn_bwd(_p(planes), dref, _p(out), _p(d_out), _p(lse), _p(d_planes), _p(d_param), _p(ws), ws_bytes,
                                b, h, n, dh, ctypes.c_float(dh ** -0.5), _lib.VRR_F16, _st()), "attn_bwd")
    return d_planes, d_param


# Per-item bounds relative to the item's max.  Measured worst on a B200 over every case below: out 7.0e-4 (1.4 U16),
# d_planes 9.0e-4 (1.9 U16), d_param 4e-6.  A bf16 rounding of P in the forward gives ~2.1e-3 on out, of P or dS in the
# backward ~2.4e-3 .. 3.7e-3 on d_planes, of the stored output ~3.5e-3: all above these bounds.
OUT_TOL, GRAD_TOL, PARAM_TOL = 3 * U16, 4 * U16, 4 * U16


def _check_attention(kind, b, h, n, seed):
    desc, param, bias64 = _bias_case(kind, h, n, seed)
    planes = _planes(b, h, n, seed)
    g = torch.Generator(device=DEV).manual_seed(seed + 1)
    d_out = (torch.randn(b, n, h * 64, generator=g, device=DEV) * 0.5).to(HF)
    with tcgen05_must_run():
        out, lse = _fwd(planes, desc)
        d_planes, d_param = _bwd(planes, desc, param, out, d_out, lse)
    o, lse_ref, grads, dbias = _ref(planes, bias64, d_out, out)
    e_out = _per_item(out.view(b, n, h, 64).permute(0, 2, 1, 3), o, (2, 3))
    e_lse = ((lse.double() - lse_ref).abs() / lse_ref.abs().clamp_min(1.0)).amax(2)
    e_grad = _per_item(d_planes, grads, (3, 4))
    tag = f"fp16 {kind} B={b} H={h} N={n}"
    report(f"attention {tag}: worst per-item out {e_out.max().item():.2e} lse {e_lse.max().item():.2e} "
           f"grad {e_grad.max().item():.2e}")
    assert torch.isfinite(out).all() and torch.isfinite(lse).all() and torch.isfinite(d_planes).all(), tag
    assert e_out.max().item() <= OUT_TOL, (tag, "out", e_out.max().item())
    assert e_lse.max().item() <= 1e-4, (tag, "lse", e_lse.max().item())
    assert e_grad.max().item() <= GRAD_TOL, (tag, "d_planes", e_grad.max().item())
    if param is not None:
        want = _dparam_ref(kind, dbias, n)
        e_p = _per_item(d_param.view_as(want), want, (1,) if want.dim() == 2 else (0,))
        report(f"attention {tag}: worst per-head d_param {e_p.max().item():.2e}")
        assert e_p.max().item() <= PARAM_TOL, (tag, "d_param", e_p.max().item())


# every N reaching a different forward / backward kernel; the polynomial bias needs N - 1 = g^2
ATTN_CASES = ([(kind, n) for kind in ("none", "table") for n in (65, 197, 208, 209, 256, 257, 577, 1025)]
              + [(kind, n) for kind in ("poly", "poly_perhead") for n in (65, 197, 226, 257, 577, 1025)])


@pytest.mark.parametrize("kind,n", ATTN_CASES)
def test_fp16_attention_vs_float64(kind, n):
    """Every bias mode at every N that reaches a different forward / backward kernel, fwd + bwd + lse + d_param per
    item against float64; the batch gives every persistent CTA >= 3 items at N <= 256."""
    h = 4
    b = -(-3 * _sms() // h) if n <= 257 else 2
    _check_attention(kind, b, h, n, seed=n + 7)


@pytest.mark.parametrize("kind,n", [("table", 197), ("poly", 197), ("none", 197), ("table", 257), ("none", 577)])
def test_fp16_attention_batch_invariance_bitwise(kind, n):
    """An image computed inside a batch of >= 3 x SM items equals, bit for bit, the same image computed alone: every
    forward kernel and both backward kernels in fp16."""
    h = 12
    b = -(-3 * _sms() // h)
    desc, param, _ = _bias_case(kind, h, n, seed=n)
    planes = _planes(b, h, n, seed=61)
    g = torch.Generator(device=DEV).manual_seed(62)
    d_out = (torch.randn(b, n, h * 64, generator=g, device=DEV) * 0.5).to(HF)
    with tcgen05_must_run():
        out, lse = _fwd(planes, desc)
        d_planes, _ = _bwd(planes, desc, param, out, d_out, lse)
        for img in (0, b // 2, b - 1):
            one = planes[:, img:img + 1].contiguous()
            o1, l1 = _fwd(one, desc)
            assert torch.equal(o1[0], out[img]) and torch.equal(l1[0], lse[img]), ("forward", img)
            dp1, _ = _bwd(one, desc, param, out[img:img + 1].contiguous(), d_out[img:img + 1].contiguous(),
                          lse[img:img + 1].contiguous())
            assert torch.equal(dp1[:, 0], d_planes[:, img]), ("backward", img)


@pytest.mark.parametrize("n", [65, 197])
@pytest.mark.parametrize("dh", [16, 32])
def test_fp16_simt_attention(dh, n):
    """Head dims 16 and 32 (the reference's ViT-Tiny under fp16 autocast) run the SIMT kernels in fp16: out, lse, dQ,
    dK, dV per item and d_table per head against float64, with the bounds of the tcgen05 cases."""
    b, h = 4, 3
    planes = _planes(b, h, n, 81, dh)
    desc, param, bias64 = _bias_case("table", h, n, seed=3)
    g = torch.Generator(device=DEV).manual_seed(82)
    d_out = (torch.randn(b, n, h * dh, generator=g, device=DEV) * 0.5).to(HF)
    simt0 = _lib.family_count(_lib.IMPL_SIMT)
    out, lse = _fwd(planes, desc)
    d_planes, d_param = _bwd(planes, desc, param, out, d_out, lse)
    assert _lib.family_count(_lib.IMPL_SIMT) == simt0 + 2
    sc = dh ** -0.5
    q, k, v = planes.double().unbind(0)
    s = q @ k.transpose(-1, -2) * sc + bias64[None]
    lse_ref = torch.logsumexp(s, -1)
    p = torch.exp(s - lse_ref[..., None])
    o = p @ v
    do = d_out.double().view(b, n, h, dh).permute(0, 2, 1, 3)
    ob = out.double().view(b, n, h, dh).permute(0, 2, 1, 3)
    ds = p * (do @ v.transpose(-1, -2) - (do * ob).sum(-1, keepdim=True))
    grads = torch.stack([ds @ k * sc, ds.transpose(-1, -2) @ q * sc, p.transpose(-1, -2) @ do])
    e_out = _per_item(ob, o, (2, 3))
    e_lse = ((lse.double() - lse_ref).abs() / lse_ref.abs().clamp_min(1.0)).max().item()
    e_grad = _per_item(d_planes, grads, (3, 4))
    e_tab = _per_item(d_param, _dparam_ref("table", ds.sum(0), n), (1,))
    report(f"attention fp16 SIMT Dh={dh} N={n}: worst per-item out {e_out.max().item():.2e} lse {e_lse:.2e} "
           f"grad {e_grad.max().item():.2e} d_table {e_tab.max().item():.2e}")
    assert e_out.max().item() <= OUT_TOL and e_lse <= 1e-4
    assert e_grad.max().item() <= GRAD_TOL, e_grad.amax((1, 2))
    assert e_tab.max().item() <= PARAM_TOL, e_tab


def test_fp16_backward_overflow_is_inf_never_clamped():
    """Gradients past fp16's range: dS > 65504 (written to TMEM as the MMA's fp16 A operand) gives non-finite dQ / dK,
    and a dV or dQ whose fp32 accumulator exceeds 65504 (from finite dS) is stored as +inf, not 65504 - in both
    backward kernels."""
    for n in (197, 257):  # whole-sequence backward / two-kernel backward
        b, h = 2, 2
        planes = torch.zeros(3, b, h, n, 64, device=DEV, dtype=HF)
        planes[0] = 1.0                      # q
        planes[1, :, :, 0] = 2.0             # k: every query attends to keys 0 and 1 (P ~ 0.5 each)
        planes[1, :, :, 1] = 2.0
        planes[2, :, :, 0] = 1.0             # v0 = +1, v1 = -1: O = 0, dP_i0 = dO . v0 = 64 * 3e4
        planes[2, :, :, 1] = -1.0
        d_out = torch.full((b, n, h * 64), 30000.0, device=DEV, dtype=HF)
        with tcgen05_must_run():
            out, lse = _fwd(planes, None)
            d_planes, _ = _bwd(planes, None, None, out, d_out, lse)
        assert not torch.isfinite(d_planes[0]).all() and not torch.isfinite(d_planes[1]).all(), n
        dv0 = d_planes[2, :, :, 0]  # sum_i P_i0 dO_i ~ n / 2 * 3e4 > 65504
        assert torch.isinf(dv0).all() and (dv0 > 0).all(), (n, dv0.flatten()[:4])
        assert (d_planes.abs() != 65504).all(), n
    # dQ: dS stays finite (~300) but the fp32 dQ accumulator passes 65504 - the stored dQ must be +inf
    for n in (197, 257):
        b, h = 2, 2
        planes = torch.zeros(3, b, h, n, 64, device=DEV, dtype=HF)
        planes[0, ..., :32] = 1.0              # q = 1 on the first 32 channels
        planes[1, :, :, 0:2, :32] = 2.0        # keys 0 and 1 score 8, the others 0: P ~ 0.48 each
        planes[1, :, :, 0, 32:] = 2000.0       # k0 - k1 = 4000 on the last 32 channels, which q does not see
        planes[1, :, :, 1, 32:] = -2000.0
        planes[2, :, :, 0] = 1.0               # v0 = +1, v1 = -1: O = 0, dS_i0 = -dS_i1 ~ 0.48 * 64 * 10
        planes[2, :, :, 1] = -1.0
        d_out = torch.full((b, n, h * 64), 10.0, device=DEV, dtype=HF)
        with tcgen05_must_run():
            out, lse = _fwd(planes, None)
            d_planes, _ = _bwd(planes, None, None, out, d_out, lse)
        dq_hi = d_planes[0, ..., 32:]          # 0.125 * (dS_i0 - dS_i1) * 2000 ~ 1.5e5
        assert torch.isinf(dq_hi).all() and (dq_hi > 0).all(), (n, dq_hi.flatten()[:4])
        assert torch.isfinite(d_planes[0, ..., :32]).all() and torch.isfinite(d_planes[1:]).all(), n


# ------------------------------------------------------------------------------------------------ streaming kernels

def _ln_ints(m, e, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randint(-8, 9, (m, e), generator=g, device=DEV).float()


@pytest.mark.parametrize("e", [192, 768, 1024])
def test_fp16_layernorm_rows_and_param_grads(e):
    """LayerNorm and add+LayerNorm with fp16 y / branch: rows identical across the launch variants and when computed
    alone; dgamma / dbeta exact with integer data (mean / rstd fixed to exact values)."""
    lib = _lib_()
    m = 3 * 8 * _sms() + 5
    x = torch.randn(m, e, device=DEV) * 2 + 0.5
    gamma, beta = torch.randn(e, device=DEV), torch.randn(e, device=DEV)
    outs = []
    for reg in (1, 0):
        lib.vrr_set_option(b"ln_reg", reg)
        y = torch.full((m, e), NAN, device=DEV, dtype=HF)
        mean, rstd = torch.empty(m, device=DEV), torch.empty(m, device=DEV)
        _lib.check(lib.vrr_layernorm_fwd(_p(x), _p(gamma), _p(beta), _p(y), _p(mean), _p(rstd), m, e, ctypes.c_float(1e-5),
                                         _lib.VRR_F32, _lib.VRR_F16, _st()), "ln fwd")
        outs.append(y)
    lib.vrr_set_option(b"ln_reg", 1)
    assert torch.equal(outs[0], outs[1])
    y1 = torch.full((1, e), NAN, device=DEV, dtype=HF)
    m1, r1 = torch.empty(1, device=DEV), torch.empty(1, device=DEV)
    _lib.check(lib.vrr_layernorm_fwd(_p(x[7:8].contiguous()), _p(gamma), _p(beta), _p(y1), _p(m1), _p(r1), 1, e,
                                     ctypes.c_float(1e-5), _lib.VRR_F32, _lib.VRR_F16, _st()), "ln fwd one row")
    assert torch.equal(y1[0], outs[0][7])
    ref = torch.nn.functional.layer_norm(x.double(), (e,), gamma.double(), beta.double(), 1e-5)
    assert (outs[0].double() - ref).abs().max().item() <= 2 * U16 * ref.abs().max().item()

    # add+LayerNorm, fp16 branch: x_new = x + branch exact in fp32 for small integers; rows alone == rows in batch
    br = _ln_ints(m, e, 5).to(HF)
    xi = _ln_ints(m, e, 6)
    res = []
    for rows in ((0, m), (9, 10)):
        r0, r1_ = rows
        mm = r1_ - r0
        xn = torch.full((mm, e), NAN, device=DEV)
        y = torch.full((mm, e), NAN, device=DEV, dtype=HF)
        mu, rs = torch.empty(mm, device=DEV), torch.empty(mm, device=DEV)
        _lib.check(lib.vrr_add_layernorm_fwd(_p(xi[r0:r1_].contiguous()), _p(br[r0:r1_].contiguous()), _p(xn), _p(gamma),
                                             _p(beta), _p(y), _p(mu), _p(rs), mm, e, ctypes.c_float(1e-5), _lib.VRR_F16,
                                             _lib.VRR_F16, _st()), "add ln fwd")
        res.append((xn, y))
    assert torch.equal(res[0][0], xi + br.float()) and torch.equal(res[1][1][0], res[0][1][9])

    # backward: dgamma / dbeta exact with integer x, dy and mean, rstd = 1/4
    dy = _ln_ints(m, e, 7).to(HF)
    mean = torch.randint(-2, 3, (m,), device=DEV).float()
    rstd = torch.full((m,), 0.25, device=DEV)
    dx = torch.full((m, e), NAN, device=DEV)
    dgb = torch.full((2, e), NAN, device=DEV)
    _lib.check(lib.vrr_layernorm_bwd(_p(dy), _p(xi), _p(gamma), _p(mean), _p(rstd), _p(dx), _p(dgb[0]), _p(dgb[1]), m, e,
                                     _lib.VRR_F32, _lib.VRR_F16, _st()), "ln bwd")
    xhat = (xi.double() - mean.double()[:, None]) * 0.25
    assert torch.equal(dgb[0].double(), (dy.double() * xhat).sum(0)) and torch.equal(dgb[1].double(), dy.double().sum(0))
    d_branch = torch.full((m, e), NAN, device=DEV, dtype=HF)
    dgb2 = torch.full((2, e), NAN, device=DEV)
    _lib.check(lib.vrr_add_layernorm_bwd(_p(dy), None, _p(xi), _p(gamma), _p(mean), _p(rstd), _p(dx), _p(d_branch),
                                         _p(dgb2[0]), _p(dgb2[1]), m, e, _lib.VRR_F16, _lib.VRR_F16, _st()), "add ln bwd")
    assert torch.equal(dgb2, dgb) and torch.equal(d_branch, dx.to(HF))


def test_fp16_rope_backward_and_tables_exact():
    """d_qkv, d_cos and d_sin of the QKV/RoPE backward on a 1/4 grid (exact in fp32 sums) with >= 4 images per
    thread; vrr_rope_apply and vrr_rope_table_grad in fp16."""
    lib = _lib_()
    h, n, dh = 12, 197, 64
    e = h * dh
    b = 4 * 8 * _sms() * 128 // (h * n * 8) + 4
    g = torch.Generator(device=DEV).manual_seed(91)
    q4 = lambda shape: (torch.randint(-4, 5, shape, generator=g, device=DEV).float() / 4)  # noqa: E731
    d_planes, planes = (q4((3, b, h, n, dh)) * 4).to(HF), (q4((3, b, h, n, dh)) * 4).to(HF)  # integers in [-4, 4]
    cos, sin = q4((h, n - 1, dh // 2)), q4((h, n - 1, dh // 2))
    d_qkv = torch.full((b * n, 3 * e), NAN, device=DEV, dtype=HF)
    d_cs = torch.full((2, h, n - 1, dh // 2), NAN, device=DEV)
    _lib.check(lib.vrr_qkv_rope_bwd(_p(d_planes), _p(planes), _p(cos), _p(sin), _p(d_qkv), _p(d_cs[0]), _p(d_cs[1]), b, n,
                                    e, h, _lib.ROPE_MIXED, _lib.VRR_F16, _st()), "qkv_rope_bwd")
    want, tc, ts = _rope_ref_bwd(d_planes, planes, cos, sin, "mixed", b, n, e, h)
    assert torch.equal(d_qkv.double(), want)  # values on a 1/16 grid below 8: exact in fp16
    assert torch.equal(d_cs[0].double(), tc.sum((0, 1))) and torch.equal(d_cs[1].double(), ts.sum((0, 1)))
    hd = dh // 2

    # stand-alone rotate-half and its table gradient
    qi, ki = q4((2, h, 64, dh)).to(HF), q4((2, h, 64, dh)).to(HF)
    ct, st_ = q4((h, 64, hd)), q4((h, 64, hd))
    qo, ko = torch.full_like(qi, NAN), torch.full_like(ki, NAN)
    _lib.check(lib.vrr_rope_apply(_p(qi), _p(ki), _p(ct), _p(st_), _p(qo), _p(ko), 2, h, 64, dh, _lib.ROPE_MIXED, 0,
                                  _lib.VRR_F16, _st()), "rope_apply")
    x1, x2 = qi.double()[..., :hd], qi.double()[..., hd:]
    want_q = torch.cat([x1 * ct.double() - x2 * st_.double(), x1 * st_.double() + x2 * ct.double()], -1)
    assert torch.equal(qo.double(), _to16(want_q).double())
    dq, dk = q4((2, h, 64, dh)).to(HF), q4((2, h, 64, dh)).to(HF)
    dc, dsn = torch.full_like(ct, NAN), torch.full_like(st_, NAN)
    _lib.check(lib.vrr_rope_table_grad(_p(qi), _p(ki), _p(dq), _p(dk), _p(dc), _p(dsn), 2, h, 64, dh, _lib.ROPE_MIXED,
                                       _lib.VRR_F16, _st()), "rope_table_grad")
    wc = torch.zeros(h, 64, hd, dtype=torch.float64, device=DEV)
    ws = torch.zeros_like(wc)
    for inp, gr in ((qi, dq), (ki, dk)):
        a1, a2 = inp.double()[..., :hd], inp.double()[..., hd:]
        g1, g2 = gr.double()[..., :hd], gr.double()[..., hd:]
        wc += (g1 * a1 + g2 * a2).sum(0)
        ws += (g2 * a1 - g1 * a2).sum(0)
    assert torch.equal(dc.double(), wc) and torch.equal(dsn.double(), ws)


def test_fp16_colsum_gelu_bwd_and_patch_embed_bwd():
    """vrr_colsum (aligned and element-offset views), vrr_gelu_bwd and the patch-embedding backward in fp16."""
    lib = _lib_()
    m, c = 8 * _sms() + 3, 768
    x = _ints((m + 1, c), 4, 101)
    for view in (x[:m], x.view(-1)[1:1 + m * c].view(m, c)):
        out = torch.full((c,), NAN, device=DEV)
        _lib.check(lib.vrr_colsum(_p(view), _p(out), m, c, _lib.VRR_F16, _st()), "colsum")
        assert torch.equal(out.double(), view.double().sum(0))
    g = torch.Generator(device=DEV).manual_seed(102)
    dy = (torch.randn(m, c, generator=g, device=DEV)).to(HF)
    hh = (torch.randn(m, c, generator=g, device=DEV) * 2).to(HF)
    dh = torch.full((m, c), NAN, device=DEV, dtype=HF)
    db = torch.full((c,), NAN, device=DEV)
    _lib.check(lib.vrr_gelu_bwd(_p(dy), _p(hh), _p(dh), _p(db), m, c, _lib.VRR_F16, _st()), "gelu_bwd")
    _, dg, _, _ = _gelu64(hh.float())
    want = dy.double() * dg
    assert (dh.double() - want).abs().max().item() <= 2 * U16 * want.abs().max().item()
    assert (db.double() - dh.double().sum(0)).abs().max().item() <= 1e-5 * dh.double().abs().sum(0).max().item()

    bsz, ch, size, p, e = 2 * _sms(), 3, 32, 8, 64
    np_ = (size // p) ** 2
    dtok = _ints((bsz, np_ + 1, e), 3, 103)
    img = _ints((bsz, ch, size, size), 2, 104)
    d_w = torch.full((e, ch * p * p), NAN, device=DEV)
    d_b, d_cls = torch.full((e,), NAN, device=DEV), torch.full((e,), NAN, device=DEV)
    d_pos = torch.full((np_, e), NAN, device=DEV)
    _lib.check(lib.vrr_patch_embed_bwd(_p(img), _p(dtok), _p(d_w), _p(d_b), _p(d_cls), _p(d_pos), bsz, ch, size, size, p, e,
                                       _lib.VRR_F16, _lib.VRR_F16, _lib.VRR_F16, _st()), "patch_embed_bwd")
    t = dtok.double()
    unf = img.double().unfold(2, p, p).unfold(3, p, p).permute(0, 2, 3, 1, 4, 5).reshape(bsz * np_, -1)
    assert torch.equal(d_cls.double(), t[:, 0].sum(0)) and torch.equal(d_pos.double(), t[:, 1:].sum(0))
    assert torch.equal(d_b.double(), t[:, 1:].sum((0, 1)))
    assert torch.equal(d_w.double(), t[:, 1:].reshape(-1, e).t() @ unf)


def test_fp16_mixing_with_bf16_is_rejected():
    """bf16 and fp16 never meet in one call."""
    lib = _lib_()
    a = torch.zeros(8, 8, device=DEV, dtype=HF)
    c = torch.zeros(8, 8, device=DEV, dtype=torch.bfloat16)
    assert lib.vrr_gemm_ex(_p(a), _p(a), _p(c), None, None, 8, 8, 8, 0, 1, _lib.VRR_F16, _lib.VRR_BF16, 0, 0, _st()) == -1
    x = torch.zeros(8, 64, device=DEV, dtype=HF)
    y = torch.zeros(8, 64, device=DEV, dtype=torch.bfloat16)
    s = torch.zeros(64, device=DEV)
    assert lib.vrr_layernorm_fwd(_p(x), _p(s), _p(s), _p(y), _p(s), _p(s), 8, 64, ctypes.c_float(1e-5), _lib.VRR_F16,
                                 _lib.VRR_BF16, _st()) == -1
