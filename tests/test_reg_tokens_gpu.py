"""Register tokens on the device: the prefix-aware patch-embedding and QKV+RoPE kernels bit for bit, and the model with
registers against an fp32 oracle that places them as timm / DINOv2 do.

Kernel checks use the equivalence the C ABI states: a QKV+RoPE call with ``n_prefix = P`` and tables ``T`` is the
``n_prefix = 1`` call fed ``T`` with ``P - 1`` identity rows (cos 1, sin 0) prepended, because a rotation by (1, 0) is
exact.  The patch embedding uses integer data, exact in any summation order, against float64 sums.  Outputs are
pre-filled with NaN and shapes are sized from the device so that every GEMM cluster takes several work units.
"""
import math

import pytest
import torch
import torch.nn.functional as F

import train
from oracle import vit_torch as V
from vit_rpe_rope_b200 import VisionTransformer, _lib, ops
from vit_rpe_rope_b200.runtime import GraphedInference

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
BF, HF, F32 = torch.bfloat16, torch.float16, torch.float32
DT = {F32: _lib.VRR_F32, BF: _lib.VRR_BF16, HF: _lib.VRR_F16}
NAN = float("nan")
PREFIXES = [1, 2, 5]


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _p(t):
    return ops._ptr(t)


def _st():
    return ops._stream()


def _nan(shape, dtype=F32):
    return torch.full(shape, NAN, device=DEV, dtype=dtype)


def _ints(shape, lo, hi, dtype, gen):
    return torch.randint(lo, hi + 1, shape, generator=gen).to(dtype).to(DEV)


class _impl:
    def __init__(self, impl):
        self.impl = impl

    def __enter__(self):
        self.prev = _lib.set_impl(self.impl)

    def __exit__(self, *exc):
        _lib.set_impl(self.prev)
        return False


# ===================================================================================== QKV + RoPE
# (dtype, family, packed tables): tcgen05 bf16 / fp16 with both table layouts, and the SIMT fp32 kernel
QKV_CASES = [(BF, _lib.IMPL_TCGEN05, True), (BF, _lib.IMPL_TCGEN05, False), (HF, _lib.IMPL_TCGEN05, True),
             (HF, _lib.IMPL_TCGEN05, False), (F32, _lib.IMPL_AUTO, False)]
QKV_IDS = ["bf16-packed", "bf16-rowmajor", "f16-packed", "f16-rowmajor", "f32-simt"]


def _qkv_shape(P, dtype):
    H, Dh = 2, 64
    E = H * Dh
    N = 64 + P  # 8 x 8 patches
    if dtype == F32:
        B = 64
    else:  # 256-row tiles x 2 column tiles (3E = 384): >= 4 work units per CTA pair
        B = math.ceil(4 * (_sms() // 2) * 256 / 2 / N)
    return B, N, E, H, Dh


def _tables(mode, H, rows, Dh, gen, integer=False):
    shape = (rows, Dh // 2) if mode == _lib.ROPE_AXIAL else (H, rows, Dh // 2)
    if integer:  # values whose products and sums are exact in fp32
        vals = torch.tensor([-1.0, -0.5, 0.0, 0.5, 1.0])
        c = vals[torch.randint(0, 5, shape, generator=gen)]
        s = vals[torch.randint(0, 5, shape, generator=gen)]
    else:
        a = torch.rand(shape, generator=gen) * 6.2832
        c, s = torch.cos(a), torch.sin(a)
    return c.to(DEV).contiguous(), s.to(DEV).contiguous()


def _padded(cos, sin, P, mode):
    """(cos, sin) with P - 1 identity rows (cos 1, sin 0) prepended."""
    ax = 0 if mode == _lib.ROPE_AXIAL else 1
    shp = list(cos.shape)
    shp[ax] = P - 1
    one = torch.ones(shp, device=DEV)
    zero = torch.zeros(shp, device=DEV)
    return torch.cat((one, cos), ax).contiguous(), torch.cat((zero, sin), ax).contiguous()


def _pack(cos, sin, mode):
    heads = cos.shape[0] if mode == _lib.ROPE_MIXED else 1
    rows, half = cos.shape[-2], cos.shape[-1]
    out = torch.empty(heads, half // 2, rows, 4, device=DEV)
    _lib.check(_lib.load().vrr_rope_pack_tables(_p(cos), _p(sin), _p(out), heads, rows, half, _st()), "pack")
    return out


def _qkv_fwd(x, w, cos, sin, packed, B, N, E, H, P, mode, dtype, old=False):
    lib = _lib.load()
    planes = _nan((3, B, H, N, E // H), dtype)
    if old:
        rc = lib.vrr_qkv_rope_fwd_packed(_p(x), _p(w), _p(cos), _p(sin), _p(packed), _p(planes), B, N, E, H, mode,
                                         DT[dtype], _st())
    else:
        rc = lib.vrr_qkv_rope_fwd_prefix(_p(x), _p(w), _p(cos), _p(sin), _p(packed), _p(planes), B, N, E, H, P, mode,
                                         DT[dtype], _st())
    _lib.check(rc, "qkv_rope_fwd")
    return planes


@pytest.mark.parametrize("P", PREFIXES)
@pytest.mark.parametrize("mode", [_lib.ROPE_AXIAL, _lib.ROPE_MIXED], ids=["axial", "mixed"])
@pytest.mark.parametrize("dtype,impl,packed", QKV_CASES, ids=QKV_IDS)
def test_qkv_forward_prefix_is_identity_padded_tables(dtype, impl, packed, mode, P):
    B, N, E, H, Dh = _qkv_shape(P, dtype)
    g = torch.Generator().manual_seed(P * 10 + mode)
    x = (torch.randn(B * N, E, generator=g) * 0.5).to(dtype).to(DEV)
    w = (torch.randn(3 * E, E, generator=g) * 0.05).to(dtype).to(DEV)
    cos, sin = _tables(mode, H, N - P, Dh, g)
    cpad, spad = _padded(cos, sin, P, mode)
    pk = _pack(cos, sin, mode) if packed else None
    pkpad = _pack(cpad, spad, mode) if packed else None
    fam = _lib.family_count(_lib.IMPL_TCGEN05)
    with _impl(impl):
        got = _qkv_fwd(x, w, cos, sin, pk, B, N, E, H, P, mode, dtype)
        want = _qkv_fwd(x, w, cpad, spad, pkpad, B, N, E, H, 1, mode, dtype, old=True)
    torch.cuda.synchronize()
    if impl == _lib.IMPL_TCGEN05:
        assert _lib.family_count(_lib.IMPL_TCGEN05) - fam == 2
    assert not got.isnan().any()
    assert torch.equal(got, want)
    # the prefix rows of q and k, and all of v, are the plain projection: unchanged by the tables
    cos2, sin2 = _tables(mode, H, N - P, Dh, g)
    with _impl(impl):
        other = _qkv_fwd(x, w, cos2, sin2, _pack(cos2, sin2, mode) if packed else None, B, N, E, H, P, mode, dtype)
    assert torch.equal(other[:, :, :, :P], got[:, :, :, :P]) and torch.equal(other[2], got[2])


def _qkv_bwd(dpl, pl, cos, sin, B, N, E, H, P, mode, dtype, old=False):
    lib = _lib.load()
    d_qkv = _nan((B * N, 3 * E), dtype)
    d_cos, d_sin = _nan(tuple(cos.shape)), _nan(tuple(cos.shape))
    if old:
        rc = lib.vrr_qkv_rope_bwd(_p(dpl), _p(pl), _p(cos), _p(sin), _p(d_qkv), _p(d_cos), _p(d_sin), B, N, E, H, mode,
                                  DT[dtype], _st())
    else:
        rc = lib.vrr_qkv_rope_bwd_prefix(_p(dpl), _p(pl), _p(cos), _p(sin), _p(d_qkv), _p(d_cos), _p(d_sin), B, N, E, H,
                                         P, mode, DT[dtype], _st())
    _lib.check(rc, "qkv_rope_bwd")
    return d_qkv, d_cos, d_sin


@pytest.mark.parametrize("P", PREFIXES)
@pytest.mark.parametrize("mode", [_lib.ROPE_AXIAL, _lib.ROPE_MIXED], ids=["axial", "mixed"])
@pytest.mark.parametrize("dtype", [BF, HF, F32], ids=["bf16", "f16", "f32"])
def test_qkv_backward_prefix_is_identity_padded_tables(dtype, mode, P):
    """Integer-valued data and tables from {0, +-0.5, +-1}: d_cos / d_sin (fp32 atomics) are exact in any order."""
    B, N, E, H, Dh = _qkv_shape(P, BF)
    g = torch.Generator().manual_seed(100 + P * 10 + mode)
    dpl = _ints((3, B, H, N, Dh), -3, 3, dtype, g)
    pl = _ints((3, B, H, N, Dh), -3, 3, dtype, g)
    cos, sin = _tables(mode, H, N - P, Dh, g, integer=True)
    cpad, spad = _padded(cos, sin, P, mode)
    got = _qkv_bwd(dpl, pl, cos, sin, B, N, E, H, P, mode, dtype)
    want = _qkv_bwd(dpl, pl, cpad, spad, B, N, E, H, 1, mode, dtype, old=True)
    assert not got[0].isnan().any() and not got[1].isnan().any()
    assert torch.equal(got[0], want[0])
    ax = 0 if mode == _lib.ROPE_AXIAL else 1
    for a, b in ((got[1], want[1]), (got[2], want[2])):
        assert torch.equal(a, b.narrow(ax, P - 1, N - P))


# ===================================================================================== patch embedding
def _patch_case(P, dtype, tdt, seed):
    """Integer images, weights, bias, prefix and table; B sized for >= 4 work units per CTA pair (E 128: one column
    tile, 256-row tiles).  Sparse weights keep every conv output below 256 in magnitude: exact in bf16 and fp16."""
    C, S, PS, E = 3, 64, 16, 128
    Np = (S // PS) ** 2
    B = math.ceil(4 * (_sms() // 2) * 256 / Np) if dtype != F32 else 64
    g = torch.Generator().manual_seed(seed)
    img = torch.randint(-2, 3, (B, C, S, S), generator=g).float()
    w = torch.randint(-1, 2, (E, C, PS, PS), generator=g).float() * (torch.rand(E, C, PS, PS, generator=g) < 0.02)
    bias = torch.randint(-4, 5, (E,), generator=g).float()
    prefix = torch.randint(-9, 10, (P, E), generator=g).float()
    pos = torch.randint(-3, 4, (Np + 3, E), generator=g).float()
    return dict(C=C, S=S, PS=PS, E=E, Np=Np, B=B, img=img, w=w, bias=bias, prefix=prefix, pos=pos)


def _patch_fwd(c, P, dtype, tdt, old=False, pos=True):
    lib = _lib.load()
    B, C, S, PS, E, Np = c["B"], c["C"], c["S"], c["PS"], c["E"], c["Np"]
    img = c["img"].to(DEV)  # fp32 images: rounded to the conv dtype on load
    w, b = c["w"].to(dtype).to(DEV), c["bias"].to(dtype).to(DEV)
    pre, pe = c["prefix"].to(tdt).to(DEV), c["pos"].to(tdt).to(DEV) if pos else None
    tokens = _nan((B, P + Np, E), tdt)
    ws_bytes = int(lib.vrr_patch_embed_workspace_bytes(B, C, S, S, PS, E, DT[dtype]))
    ws = torch.empty(max(ws_bytes, 1), device=DEV, dtype=torch.uint8)
    if old:
        rc = lib.vrr_patch_embed_fwd(_p(img), _p(w), _p(b), _p(pre), _p(pe), _p(tokens), _p(ws), ws_bytes, B, C, S, S,
                                     PS, E, DT[F32], DT[dtype], DT[tdt], _st())
    else:
        rc = lib.vrr_patch_embed_fwd_prefix(_p(img), _p(w), _p(b), _p(pre), P, _p(pe), _p(tokens), _p(ws), ws_bytes, B,
                                            C, S, S, PS, E, DT[F32], DT[dtype], DT[tdt], _st())
    _lib.check(rc, "patch_embed_fwd")
    return tokens


def _patch_bwd(c, P, dtype, tdt, d_tok, old=False):
    lib = _lib.load()
    B, C, S, PS, E, Np = c["B"], c["C"], c["S"], c["PS"], c["E"], c["Np"]
    idt = F32 if tdt == F32 else dtype  # 16-bit token gradients pair with 16-bit images
    img = c["img"].to(idt).to(DEV)
    K = C * PS * PS
    d_w, d_b, d_pre, d_pos = _nan((E, K)), _nan((E,)), _nan((P, E)), _nan((Np, E))
    if old:
        rc = lib.vrr_patch_embed_bwd(_p(img), _p(d_tok), _p(d_w), _p(d_b), _p(d_pre), _p(d_pos), B, C, S, S, PS, E,
                                     DT[idt], DT[dtype], DT[tdt], _st())
    else:
        rc = lib.vrr_patch_embed_bwd_prefix(_p(img), _p(d_tok), _p(d_w), _p(d_b), _p(d_pre), P, _p(d_pos), B, C, S, S,
                                            PS, E, DT[idt], DT[dtype], DT[tdt], _st())
    _lib.check(rc, "patch_embed_bwd")
    return d_w, d_b, d_pre, d_pos


def _unfold64(c):
    B, C, S, PS = c["B"], c["C"], c["S"], c["PS"]
    u = c["img"].double().reshape(B, C, S // PS, PS, S // PS, PS).permute(0, 2, 4, 1, 3, 5)
    return u.reshape(B * c["Np"], C * PS * PS)


# (conv dtype, token dtype): the tcgen05 kernel under bf16 / fp16 autocast and with 16-bit tokens, and fp32 SIMT
PATCH_CASES = [(BF, F32), (HF, F32), (BF, BF), (F32, F32)]
PATCH_IDS = ["bf16-tokf32", "f16-tokf32", "bf16-tokbf16", "f32"]


@pytest.mark.parametrize("P", PREFIXES)
@pytest.mark.parametrize("dtype,tdt", PATCH_CASES, ids=PATCH_IDS)
def test_patch_embed_prefix_integer_exact(dtype, tdt, P):
    c = _patch_case(P, dtype, tdt, seed=P)
    B, E, Np = c["B"], c["E"], c["Np"]
    fam = _lib.family_count(_lib.IMPL_TCGEN05)
    tokens = _patch_fwd(c, P, dtype, tdt)
    torch.cuda.synchronize()
    if dtype != F32:
        assert _lib.family_count(_lib.IMPL_TCGEN05) - fam == 1
    conv = (_unfold64(c) @ c["w"].double().reshape(E, -1).t() + c["bias"].double()).reshape(B, Np, E)
    want = torch.empty(B, P + Np, E, dtype=torch.float64)
    want[:, :P] = c["prefix"].double()
    want[:, P:] = conv + c["pos"].double()[:Np]
    assert torch.equal(tokens.double().cpu(), want)

    g = torch.Generator().manual_seed(50 + P)
    d_tok = _ints((B, P + Np, E), -3, 3, tdt, g)
    d_w, d_b, d_pre, d_pos = _patch_bwd(c, P, dtype, tdt, d_tok)
    dt64 = d_tok.double().cpu()
    assert torch.equal(d_pre.double().cpu(), dt64[:, :P].sum(0))
    assert torch.equal(d_pos.double().cpu(), dt64[:, P:].sum(0))
    assert torch.equal(d_b.double().cpu(), dt64[:, P:].sum((0, 1)))
    assert torch.equal(d_w.double().cpu(), dt64[:, P:].reshape(B * Np, E).t() @ _unfold64(c))


@pytest.mark.parametrize("dtype,tdt", PATCH_CASES, ids=PATCH_IDS)
def test_prefix_entry_points_at_one_are_the_old_ones(dtype, tdt):
    c = _patch_case(1, dtype, tdt, seed=9)
    cf = dict(c, img=c["img"] + torch.rand(c["img"].shape) * 0.5)  # non-integer: the same bits, not merely exact sums
    for pos in (True, False):
        assert torch.equal(_patch_fwd(cf, 1, dtype, tdt, pos=pos), _patch_fwd(cf, 1, dtype, tdt, old=True, pos=pos))
    g = torch.Generator().manual_seed(3)  # integer backward: the split-K weight gradient is exact in any order
    d_tok = _ints((c["B"], 1 + c["Np"], c["E"]), -3, 3, tdt, g)
    for a, b in zip(_patch_bwd(c, 1, dtype, tdt, d_tok), _patch_bwd(c, 1, dtype, tdt, d_tok, old=True)):
        assert torch.equal(a, b)
    qd = dtype if dtype != F32 else F32
    B, N, E, H, Dh = _qkv_shape(1, qd)
    x = (torch.randn(B * N, E, generator=g) * 0.5).to(qd).to(DEV)
    w = (torch.randn(3 * E, E, generator=g) * 0.05).to(qd).to(DEV)
    for mode in (_lib.ROPE_NONE, _lib.ROPE_AXIAL, _lib.ROPE_MIXED):
        cos, sin = _tables(mode if mode else _lib.ROPE_AXIAL, H, N - 1, Dh, g)
        pk = _pack(cos, sin, mode if mode else _lib.ROPE_AXIAL) if qd != F32 and mode else None
        assert torch.equal(_qkv_fwd(x, w, cos, sin, pk, B, N, E, H, 1, mode, qd),
                           _qkv_fwd(x, w, cos, sin, pk, B, N, E, H, 1, mode, qd, old=True))
        dpl = _ints((3, B, H, N, Dh), -3, 3, qd, g)
        ci, si = _tables(mode if mode else _lib.ROPE_AXIAL, H, N - 1, Dh, g, integer=True)  # atomics: exact sums
        got = _qkv_bwd(dpl, dpl.flip(0).contiguous(), ci, si, B, N, E, H, 1, mode, qd)
        want = _qkv_bwd(dpl, dpl.flip(0).contiguous(), ci, si, B, N, E, H, 1, mode, qd, old=True)
        assert torch.equal(got[0], want[0])
        if mode != _lib.ROPE_NONE:  # without rotation the table gradients are not written
            assert torch.equal(got[1], want[1]) and torch.equal(got[2], want[2])


# ===================================================================================== model vs oracle
def _ref_attention(cfg, p, pre, x, rope, npre):
    """oracle/vit_torch.attention with `npre` unrotated prefix tokens."""
    b, n, c = x.shape
    h, dh = cfg.num_heads, cfg.head_dim
    qkv = F.linear(x, p[pre + "qkv.weight"]).reshape(b, n, 3, h, dh).permute(2, 0, 3, 1, 4)
    q, k, v = qkv[0], qkv[1], qkv[2]
    if rope is not None:
        qr, kr = V.rotate_half_pair(q[:, :, npre:], k[:, :, npre:], V.expand_cs(rope[0]), V.expand_cs(rope[1]))
        q = torch.cat([q[:, :, :npre], qr], dim=2)
        k = torch.cat([k[:, :, :npre], kr], dim=2)
    att = ((q @ k.transpose(-2, -1)) * dh ** -0.5).softmax(dim=-1)
    out = (att @ v).transpose(1, 2).reshape(b, n, c)
    return F.linear(out, p[pre + "proj.weight"], p[pre + "proj.bias"])


def _ref_forward(cfg, p, images, sites=None):
    """[cls, registers, patches] through oracle/vit_torch's layers; `sites`: replayed dropout factors per block."""
    b, _, hh, ww = images.shape
    e = cfg.embed_dim
    x = F.conv2d(images, p["patch_embed.weight"], p["patch_embed.bias"], stride=cfg.patch_size)
    gh, gw = hh // cfg.patch_size, ww // cfg.patch_size
    prefix = [p["cls_token"].expand(b, -1, -1)] + ([p["reg_token"].expand(b, -1, -1)] if "reg_token" in p else [])
    npre = sum(t.shape[1] for t in prefix)
    x = torch.cat(prefix + [x.flatten(2).transpose(1, 2)], dim=1)
    if cfg.pos_encoding == "absolute":
        x = torch.cat([x[:, :npre], x[:, npre:] + p["pos_embed.pos_embed"][:, : gh * gw]], dim=1)
    rope = None
    if cfg.pos_encoding == "rope-axial":
        rope = V.axial_cos_sin(p["pos_embed.inv_freq"], gh * gw)
    elif cfg.pos_encoding == "rope-mixed":
        rope = V.mixed_cos_sin(p["pos_embed.freqs"], gh * gw)
    mul = lambda t, f: t if f is None else t * f
    for i in range(cfg.depth):
        pre = f"blocks.{i}."
        fa, f1, f2 = sites[i] if sites is not None else (None, None, None)
        y = F.layer_norm(x, (e,), p[pre + "norm1.weight"], p[pre + "norm1.bias"], 1e-5)
        x = x + mul(_ref_attention(cfg, p, pre + "attn.", y, rope, npre), fa)
        y = F.layer_norm(x, (e,), p[pre + "norm2.weight"], p[pre + "norm2.bias"], 1e-5)
        h = mul(F.gelu(F.linear(y, p[pre + "mlp.fc1.weight"], p[pre + "mlp.fc1.bias"])), f1)
        x = x + mul(F.linear(h, p[pre + "mlp.fc2.weight"], p[pre + "mlp.fc2.bias"]), f2)
    x = F.layer_norm(x, (e,), p["norm.weight"], p["norm.bias"], 1e-5)
    return F.linear(x[:, 0], p["head.weight"], p["head.bias"])


def _cfg(kw):
    return V.VitConfig(**{k: v for k, v in kw.items() if k not in ("reg_tokens", "drop_rate", "drop_path_rate")})


def _build(kw, seed=0):
    torch.manual_seed(seed)
    model = VisionTransformer(**kw)
    with torch.no_grad():  # make zero / tiny initialised paths live
        model.cls_token.normal_(std=0.02)
        if kw.get("reg_tokens", 0):
            model.reg_token.normal_(std=0.02)
        for n, prm in model.named_parameters():
            if n.endswith(".bias"):
                prm.normal_(std=0.02)
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    return model.to(DEV), sd


def _check(model, logits, ref, p, bar, flat):
    got = logits.detach().float().cpu()
    ref = ref.detach()
    if flat:
        err = ((got - ref).abs().max() / ref.abs().max()).item()
    else:
        err = (got - ref).abs().max().item() / max(1.0, ref.abs().max().item())
    assert err <= bar, ("logits", err)
    names = set()
    for name, prm in model.named_parameters():
        want = p[name].grad if name in p else None
        if want is None:
            continue
        names.add(name)
        d = (prm.grad.detach().float().cpu() - want).abs().max()
        e = (d / want.abs().max().clamp_min(1e-30)).item() if flat else d.item() / max(1.0, want.abs().max().item())
        assert e <= bar, (name, e)
    assert "reg_token" in names or "reg_token" not in p


def _model_case(kw, images, labels, amp=None, bar=1e-5, flat=False, tc=False):
    model, sd = _build(kw)
    fam = (_lib.family_count(_lib.IMPL_TCGEN05), _lib.family_count(_lib.IMPL_SIMT))
    with torch.autocast("cuda", dtype=amp or BF, enabled=amp is not None):
        logits = model(images.to(DEV))
        loss = F.cross_entropy(logits.float(), labels.to(DEV))
    loss.backward()
    torch.cuda.synchronize()
    if tc:
        assert _lib.family_count(_lib.IMPL_TCGEN05) > fam[0] and _lib.family_count(_lib.IMPL_SIMT) == fam[1]
    p = V.params_from_state_dict(sd)
    ref = _ref_forward(_cfg(kw), p, images)
    F.cross_entropy(ref, labels).backward()
    _check(model, logits, ref, p, bar, flat)


RMODES = ["none", "absolute", "rope-axial", "rope-mixed"]
TINY = dict(img_size=32, patch_size=4, in_chans=3, num_classes=10, embed_dim=192, depth=3, num_heads=3)
CFG3 = dict(img_size=224, patch_size=16, in_chans=3, num_classes=1000, embed_dim=768, depth=2, num_heads=12)


@pytest.mark.parametrize("R", [1, 4])
@pytest.mark.parametrize("mode", RMODES)
def test_vit_tiny_with_registers_fp32(mode, R):
    torch.manual_seed(1)
    images, labels = torch.randn(8, 3, 32, 32), torch.randint(0, 10, (8,))
    _model_case(dict(TINY, pos_encoding=mode, reg_tokens=R), images, labels)


@pytest.mark.parametrize("R", [1, 4])
@pytest.mark.parametrize("mode", RMODES)
def test_cfg3_geometry_with_registers_bf16(mode, R):
    """ViT-B/16-224 geometry: 197 + R tokens (201 at R = 4), the tcgen05 family throughout."""
    torch.manual_seed(2)
    images, labels = torch.randn(4, 3, 224, 224), torch.randint(0, 1000, (4,))
    _model_case(dict(CFG3, pos_encoding=mode, reg_tokens=R), images, labels, amp=BF, bar=2e-2, flat=True, tc=True)


def test_registers_under_fp16_autocast():
    torch.manual_seed(3)
    images, labels = torch.randn(4, 3, 224, 224), torch.randint(0, 1000, (4,))
    _model_case(dict(CFG3, pos_encoding="rope-mixed", reg_tokens=4), images, labels, amp=HF, bar=2e-2, flat=True, tc=True)


def test_registers_with_resolution_extrapolation_bf16():
    """Built at 224, fed 512 px in eval: 1024 patches + 5 prefix tokens = 1029."""
    kw = dict(CFG3, pos_encoding="rope-mixed", reg_tokens=4)
    model, sd = _build(kw)
    model.eval()
    torch.manual_seed(4)
    images = torch.randn(2, 3, 512, 512)
    with torch.no_grad(), torch.autocast("cuda", dtype=BF):
        logits = model(images.to(DEV))
    with torch.no_grad():
        ref = _ref_forward(_cfg(kw), V.params_from_state_dict(sd, requires_grad=False), images)
    err = ((logits.float().cpu() - ref).abs().max() / ref.abs().max()).item()
    assert err <= 2e-2, err


def test_registers_with_dropout_and_stochastic_depth_fp32():
    kw = dict(TINY, pos_encoding="rope-mixed", reg_tokens=4, drop_rate=0.1, drop_path_rate=0.1)
    model, sd = _build(kw)
    model.train()
    B, N = 8, 64 + 5
    torch.manual_seed(5)
    images, labels = torch.randn(B, 3, 32, 32), torch.randint(0, 10, (B,))
    logits = model(images.to(DEV))
    F.cross_entropy(logits, labels.to(DEV)).backward()
    seed, E = model._drop_seed, kw["embed_dim"]
    sites = []
    for i, blk in enumerate(model.blocks):
        pp = getattr(blk.drop_path, "drop_prob", 0.0)
        Hd = blk.mlp.fc1.out_features
        sites.append((ops.branch_factor((0.1, pp, N, 3 * i, seed), B, N, E).cpu(),
                      ops.branch_factor((0.1, 0.0, N, 3 * i + 1, seed), B, N, Hd).cpu(),
                      ops.branch_factor((0.1, pp, N, 3 * i + 2, seed), B, N, E).cpu()))
    assert any((f == 0).any() for s in sites for f in s)
    p = V.params_from_state_dict(sd)
    ref = _ref_forward(_cfg(kw), p, images, sites)
    F.cross_entropy(ref, labels).backward()
    _check(model, logits, ref, p, 1e-5, False)


@pytest.mark.parametrize("amp", [None, BF], ids=["f32", "bf16"])
def test_zero_registers_change_nothing(amp):
    kw = dict(TINY if amp is None else dict(CFG3, num_classes=10), pos_encoding="rope-mixed")
    torch.manual_seed(0)
    base = VisionTransformer(**kw).to(DEV)
    torch.manual_seed(0)
    zero = VisionTransformer(**kw, reg_tokens=0).to(DEV)
    images = torch.randn(4, 3, kw["img_size"], kw["img_size"], device=DEV)
    outs = []
    for m in (base, zero):
        before = _lib.launch_count()
        with torch.autocast("cuda", dtype=BF, enabled=amp is not None):
            logits = m(images)
            logits.float().sum().backward()
        torch.cuda.synchronize()
        outs.append((logits.detach(), _lib.launch_count() - before))
    assert outs[0][1] == outs[1][1]
    assert torch.equal(outs[0][0], outs[1][0])


def test_graphed_inference_with_registers():
    kw = dict(img_size=64, patch_size=8, in_chans=3, num_classes=10, embed_dim=256, depth=2, num_heads=4,
              pos_encoding="rope-mixed", reg_tokens=4)
    model, _ = _build(kw)
    model.eval()
    runner = GraphedInference(model, (4, 3, 96, 96), torch.device(DEV), bf16=True)
    assert runner.graph is not None
    g = torch.Generator().manual_seed(7)
    for _ in range(2):
        x = torch.randn(4, 3, 96, 96, generator=g).to(DEV)
        got = runner.run(x).float().clone()
        with torch.no_grad(), torch.autocast("cuda", dtype=BF):
            want = model(x).float()
        assert torch.equal(got, want)
    runner.close()


def test_train_cli_with_registers_learns_and_reloads(tmp_path):
    argv = ["--dataset", "cifar10", "--pos_encoding", "rope-mixed", "--epochs", "2", "--batch_size", "32", "--synthetic",
            "--synthetic_size", "256", "--max_steps", "8", "--log_dir", str(tmp_path / "logs"), "--ckpt_dir",
            str(tmp_path / "ck"), "--amp", "bf16", "--embed_dim", "128", "--num_heads", "2", "--depth", "2",
            "--reg_tokens", "4"]
    log_file, ckpt = train.main(argv)
    rows = [r.split(",") for r in open(log_file).read().strip().splitlines()[1:]]
    assert len(rows) == 2 and all(math.isfinite(float(r[1])) for r in rows)
    assert float(rows[1][1]) < float(rows[0][1]), rows  # the training loss falls
    sd = torch.load(ckpt, map_location="cpu")
    assert sd["reg_token"].shape == (1, 4, 128)
    m = VisionTransformer(img_size=32, patch_size=4, in_chans=3, num_classes=10, embed_dim=128, depth=2, num_heads=2,
                          pos_encoding="rope-mixed", reg_tokens=4)
    m.load_state_dict(sd, strict=True)
