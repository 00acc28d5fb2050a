"""QK-norm on the device: ``vrr_qkv_rope_norm_fwd`` / ``_bwd`` against the contract of include/vrr.h, and the model
with ``qk_norm=True`` against an fp32 oracle that applies timm's ``q_norm`` / ``k_norm`` before RoPE.

Forward: integer x and W make the accumulator exact, so the saved pre-norm rows must be its rounding bit for bit; the
statistics and the normalised, rotated planes are held to a bound derived from the kernels' operation order against
float64.  Backward: integer data, integer means, rstd = 2^-k, integer affine parameters and tables on a half grid make
every product and sum exact in fp32, so all outputs must equal the float64 result (d_qkv after its one rounding).
Outputs are pre-filled with NaN; the GEMM shapes give every CTA pair at least four work units, the backward shapes at
least four images per thread, and N = 65 and 197 put warp tiles across image boundaries.
"""
import math

import pytest
import torch
import torch.nn.functional as F

import train
from oracle import vit_torch as V
from vit_rpe_rope_b200 import VisionTransformer, _lib, ops
from vit_rpe_rope_b200.dp import BucketedDataParallel
from vit_rpe_rope_b200.models.vit import SwiGLUPacked
from vit_rpe_rope_b200.runtime import GraphedInference, GraphedTrainStep

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
BF, HF, F32 = torch.bfloat16, torch.float16, torch.float32
DT = {F32: _lib.VRR_F32, BF: _lib.VRR_BF16, HF: _lib.VRR_F16}
TC, SIMT = _lib.IMPL_TCGEN05, _lib.IMPL_SIMT
NAN = float("nan")
U = 2.0 ** -24
U_T = {F32: 2.0 ** -24, BF: 2.0 ** -8, HF: 2.0 ** -11}      # unit roundoff of the output type
TINY_T = {F32: 2.0 ** -150, BF: 2.0 ** -134, HF: 2.0 ** -25}  # half the smallest subnormal
MODES3 = [_lib.ROPE_NONE, _lib.ROPE_AXIAL, _lib.ROPE_MIXED]
EPS = 1e-5


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _p(t):
    return ops._ptr(t)


def _st():
    return ops._stream()


def _nan(shape, dtype=F32):
    return torch.full(shape, NAN, device=DEV, dtype=dtype)


def _ints(shape, lo, hi, gen):
    return torch.randint(lo, hi + 1, shape, generator=gen).double()


def _gam(k):
    return k * U / (1 - k * U)


class _impl:
    def __init__(self, impl):
        self.impl = impl

    def __enter__(self):
        self.prev = _lib.set_impl(self.impl)

    def __exit__(self, *exc):
        _lib.set_impl(self.prev)
        return False


def _tables(mode, H, rows, Dh, gen, half_grid=False):
    m = mode if mode != _lib.ROPE_NONE else _lib.ROPE_AXIAL
    shape = (rows, Dh // 2) if m == _lib.ROPE_AXIAL else (H, rows, Dh // 2)
    if half_grid:  # products and sums exact in fp32
        vals = torch.tensor([-1.0, -0.5, 0.0, 0.5, 1.0])
        c, s = vals[torch.randint(0, 5, shape, generator=gen)], vals[torch.randint(0, 5, shape, generator=gen)]
    else:
        a = torch.rand(shape, generator=gen) * 6.2832
        c, s = torch.cos(a), torch.sin(a)
    return c.contiguous(), s.contiguous()


def _pack(cos, sin, mode):
    heads = cos.shape[0] if mode == _lib.ROPE_MIXED else 1
    rows, half = cos.shape[-2], cos.shape[-1]
    out = torch.empty(heads, half // 2, rows, 4, device=DEV)
    _lib.check(_lib.load().vrr_rope_pack_tables(_p(cos), _p(sin), _p(out), heads, rows, half, _st()), "pack")
    return out


def _cs_rows(cos, sin, mode, H, N, P):
    """[H][N][Dh/2] float64 tables per token row, identity on the P prefix rows."""
    c, s = cos.double(), sin.double()
    if mode == _lib.ROPE_AXIAL:
        c, s = c.expand(H, -1, -1), s.expand(H, -1, -1)
    one = torch.ones(H, P, c.shape[-1], dtype=torch.float64)
    if mode == _lib.ROPE_NONE:
        return one.new_ones(H, N, c.shape[-1]), one.new_zeros(H, N, c.shape[-1])
    return torch.cat((one, c), 1), torch.cat((one * 0, s), 1)


# ===================================================================================== forward kernel
# (dtype, Dh, family): tcgen05 bf16 / fp16 (Dh 64), FFMA fp32 at every head dim, FFMA bf16 at Dh 16 / 32
FWD_CASES = [(BF, 64, TC), (HF, 64, TC), (F32, 16, SIMT), (F32, 32, SIMT), (F32, 64, SIMT), (BF, 16, SIMT), (BF, 32, SIMT)]
FWD_IDS = ["bf16-tc", "f16-tc", "f32-dh16", "f32-dh32", "f32-dh64", "bf16-simt-dh16", "bf16-simt-dh32"]


def _fwd_shape(N, dtype, fam):
    E = 128
    if fam == TC:  # 256-row tiles x 2 column tiles (3E = 384): >= 4 work units per CTA pair
        B = math.ceil(4 * (_sms() // 2) * 256 / 2 / N)
    else:
        B = 24
    return B, E


def _norm_fwd(x, w, cos, sin, pk, qn, B, N, E, H, P, mode, dtype, saved=True):
    Dh = E // H
    planes = _nan((3, B, H, N, Dh), dtype)
    pre = _nan((2, B, H, N, Dh), dtype) if saved else None
    stats = _nan((2, B, H, N, 2)) if saved else None
    rc = _lib.load().vrr_qkv_rope_norm_fwd(_p(x), _p(w), _p(cos), _p(sin), _p(pk), _p(planes), B, N, E, H, P, mode,
                                           DT[dtype], *map(_p, qn), EPS, _p(pre), _p(stats), _st())
    _lib.check(rc, "vrr_qkv_rope_norm_fwd")
    return planes, pre, stats


def _fwd_bounds(x, dtype):
    """Per-row bounds of |mean - mean64| and of the relative error of rstd (x: [.., Dh] float64 of the rounded rows)."""
    n = x.shape[-1]
    mean64 = x.mean(-1, keepdim=True)
    dt = x - mean64
    var64 = (dt * dt).mean(-1, keepdim=True)
    em = _gam(n // 4 + 1) * x.abs().sum(-1, keepdim=True) / n
    delta = em + U * (dt.abs() + em)
    ev = ((delta * (2 * dt.abs() + delta)).sum(-1, keepdim=True)
          + _gam(n // 4 + 1) * ((dt.abs() + delta) ** 2).sum(-1, keepdim=True)) / n
    rel_v = (ev + U * (var64 + EPS + ev)) / (var64 + EPS)
    q = rel_v / (2 * (1 - rel_v))
    rel_r = q + 4 * U * (1 + q)  # rsqrtf: 2 ulp
    return mean64, var64, em, delta, rel_r


@pytest.mark.parametrize("P", [1, 5])
@pytest.mark.parametrize("N", [65, 197])
@pytest.mark.parametrize("dtype,Dh,fam", FWD_CASES, ids=FWD_IDS)
def test_forward_against_float64(dtype, Dh, fam, N, P):
    B, E = _fwd_shape(N, dtype, fam)
    H = E // Dh
    g = torch.Generator().manual_seed(N * 10 + P + Dh)
    x64 = _ints((B * N, E), -2, 2, g)
    w64 = _ints((3 * E, E), -2, 2, g)
    qn64 = [torch.randn(Dh, generator=g).double() * 0.5 + (1.0 if i % 2 == 0 else 0.0) for i in range(4)]
    x, w = x64.to(dtype).to(DEV), w64.to(dtype).to(DEV)
    qn = [t.float().to(DEV) for t in qn64]
    acc = (x64 @ w64.t()).reshape(B, N, 3, H, Dh).permute(2, 0, 3, 1, 4)  # exact
    xr = acc[:2].float().to(dtype).double()  # x = T(acc)
    mean64, var64, em, delta, rel_r = _fwd_bounds(xr, dtype)
    rstd64 = 1.0 / torch.sqrt(var64 + EPS)
    worst = {"mean": 0.0, "rstd": 0.0, "planes": 0.0}
    for mode in MODES3:
        cos, sin = _tables(mode, H, N - P, Dh, g)
        layouts = [None] if mode == _lib.ROPE_NONE or fam != TC else ["packed", "rowmajor"]
        for lay in layouts:
            cd, sd = cos.to(DEV), sin.to(DEV)
            pk = _pack(cd, sd, mode) if lay == "packed" else None
            before = _lib.family_count(TC)
            with _impl(fam):
                planes, pre, stats = _norm_fwd(x, w, cd, sd, pk, qn, B, N, E, H, P, mode, dtype)
                inf, _, _ = _norm_fwd(x, w, cd, sd, pk, qn, B, N, E, H, P, mode, dtype, saved=False)
                plain = _nan((3, B, H, N, Dh), dtype)
                _lib.check(_lib.load().vrr_qkv_rope_fwd_prefix(_p(x), _p(w), _p(cd), _p(sd), _p(pk), _p(plain), B, N, E, H,
                                                               P, mode, DT[dtype], _st()), "fwd_prefix")
            torch.cuda.synchronize()
            assert (_lib.family_count(TC) - before == 3) == (fam == TC)
            assert torch.equal(pre.double().cpu(), xr)           # the saved rows: T(acc) bit for bit
            assert torch.equal(inf, planes)                      # inference writes the same planes
            assert torch.equal(planes[2], plain[2])              # v: the plain projection
            st = stats.double().cpu()
            err_m = (st[..., 0:1] - mean64).abs()
            assert (err_m <= em).all()
            err_r = (st[..., 1:2] - rstd64).abs()
            assert (err_r <= rel_r * rstd64).all()
            worst["mean"] = max(worst["mean"], (err_m / em.clamp_min(1e-300)).max().item())
            worst["rstd"] = max(worst["rstd"], (err_r / (rel_r * rstd64)).max().item())
            # y = xhat g + b in float64, then the rotation; bounds follow the kernels' order (vrr.h)
            gq = torch.stack((qn64[0], qn64[2])).view(2, 1, 1, 1, Dh)
            bq = torch.stack((qn64[1], qn64[3])).view(2, 1, 1, 1, Dh)
            dt = xr - mean64
            xh = dt * rstd64
            ex = delta * rstd64 * (1 + rel_r) + dt.abs() * rstd64 * rel_r
            ex = ex + U * (xh.abs() + ex)
            y = xh * gq + bq
            ey = gq.abs() * ex
            ey = ey + U * (y.abs() + ey)
            c, s = _cs_rows(cos, sin, mode, H, N, P)
            c, s = c.view(1, 1, H, N, Dh // 2), s.view(1, 1, H, N, Dh // 2)
            hd = Dh // 2
            y1, y2, e1, e2 = y[..., :hd], y[..., hd:], ey[..., :hd], ey[..., hd:]
            r = torch.cat((y1 * c - y2 * s, y1 * s + y2 * c), -1)
            rot = torch.cat((c.abs() * e1 + s.abs() * e2 + _gam(2) * ((y1 * c).abs() + (y2 * s).abs() + e1 + e2),
                             s.abs() * e1 + c.abs() * e2 + _gam(2) * ((y1 * s).abs() + (y2 * c).abs() + e1 + e2)), -1)
            er = rot if mode != _lib.ROPE_NONE else ey
            bound = er + U_T[dtype] * (r.abs() + er) + TINY_T[dtype]
            err = (planes[:2].double().cpu() - r).abs()
            assert (err <= bound).all(), (err / bound).max().item()
            worst["planes"] = max(worst["planes"], (err / bound).max().item())
    print(f"\nqk_norm fwd {dtype} Dh {Dh} N {N} P {P}: worst err / bound "
          + ", ".join(f"{k} {v:.3f}" for k, v in worst.items()))


# ===================================================================================== backward kernel
BWD_CASES = [(BF, 64), (HF, 64), (F32, 64), (F32, 32), (F32, 16), (BF, 32), (BF, 16)]
BWD_IDS = ["bf16-dh64", "f16-dh64", "f32-dh64", "f32-dh32", "f32-dh16", "bf16-dh32", "bf16-dh16"]


def _bwd_launch(B, N, H, Dh, dtype):
    """The launcher's grid (rope.cu: qkv_rope_norm_bwd): images per thread."""
    vec = 4 if dtype == F32 else 8
    blocks = math.ceil(H * N * (Dh // 2 // vec) / 128)
    chunks = 1
    while chunks < B and blocks * chunks < 8 * _sms():
        chunks *= 2
    return math.ceil(B / chunks)


@pytest.mark.parametrize("P", [1, 5])
@pytest.mark.parametrize("N", [65, 197])
@pytest.mark.parametrize("dtype,Dh", BWD_CASES, ids=BWD_IDS)
def test_backward_exact(dtype, Dh, N, P):
    E = 128
    H = E // Dh
    B = 16
    while _bwd_launch(B, N, H, Dh, dtype) < 4:
        B *= 2
    assert _bwd_launch(B, N, H, Dh, dtype) >= 4
    g = torch.Generator().manual_seed(200 + N + P + Dh)
    dpl64 = _ints((3, B, H, N, Dh), -3, 3, g)
    pre64 = _ints((2, B, H, N, Dh), -3, 3, g)
    mean64 = _ints((2, B, H, N, 1), -1, 1, g)
    rstd64 = 2.0 ** -_ints((2, B, H, N, 1), 0, 1, g)
    qn64 = [_ints((Dh,), -2, 2, g) for _ in range(4)]
    stats = torch.cat((mean64, rstd64), -1).float().to(DEV)
    dpl, pre = dpl64.to(dtype).to(DEV), pre64.to(dtype).to(DEV)
    qn = [t.float().to(DEV) for t in qn64]
    gw = torch.stack((qn64[0], qn64[2])).view(2, 1, 1, 1, Dh)
    gb = torch.stack((qn64[1], qn64[3])).view(2, 1, 1, 1, Dh)
    hd = Dh // 2
    for mode in MODES3:
        cos, sin = _tables(mode, H, N - P, Dh, g, half_grid=True)
        cd, sd = cos.to(DEV), sin.to(DEV)
        d_qkv = _nan((B * N, 3 * E), dtype)
        d_cs = _nan((2,) + tuple(cos.shape))
        d_norm = _nan((4, Dh))
        cs = (d_cs[0], d_cs[1]) if mode != _lib.ROPE_NONE else (None, None)
        rc = _lib.load().vrr_qkv_rope_norm_bwd(_p(dpl), _p(pre), _p(stats), _p(cd), _p(sd), *map(_p, qn),
                                               _p(d_qkv), *map(_p, cs), *map(_p, d_norm), B, N, E, H, P, mode, DT[dtype],
                                               _st())
        _lib.check(rc, "vrr_qkv_rope_norm_bwd")
        torch.cuda.synchronize()
        c, s = _cs_rows(cos, sin, mode, H, N, P)
        c, s = c.view(1, 1, H, N, hd), s.view(1, 1, H, N, hd)
        g1, g2 = dpl64[:2, ..., :hd], dpl64[:2, ..., hd:]
        dy = torch.cat((g1 * c + g2 * s, g2 * c - g1 * s), -1)  # un-rotated (prefix rows: d_planes)
        xh = (pre64 - mean64) * rstd64
        a = gw * dy
        m1, m2 = a.mean(-1, keepdim=True), (a * xh).mean(-1, keepdim=True)
        dx = rstd64 * (a - m1 - xh * m2)
        want = torch.cat((dx, dpl64[2:]), 0)  # [3, B, H, N, Dh]
        want = want.permute(1, 3, 0, 2, 4).reshape(B * N, 3 * E).float().to(dtype)
        assert torch.equal(d_qkv.cpu(), want)
        dn = d_norm.double().cpu()
        for i in range(2):
            assert torch.equal(dn[2 * i], (dy[i] * xh[i]).sum((0, 1, 2)))
            assert torch.equal(dn[2 * i + 1], dy[i].sum((0, 1, 2)))
        if mode != _lib.ROPE_NONE:
            y = xh * gw + gb
            y1, y2 = y[..., :hd], y[..., hd:]
            dc = (g1 * y1 + g2 * y2)[:, :, :, P:].sum((0, 1))  # [H, N - P, hd]
            ds = (g2 * y1 - g1 * y2)[:, :, :, P:].sum((0, 1))
            if mode == _lib.ROPE_AXIAL:
                dc, ds = dc.sum(0), ds.sum(0)
            assert torch.equal(d_cs[0].double().cpu(), dc) and torch.equal(d_cs[1].double().cpu(), ds)


def test_backward_without_parameter_gradients_writes_the_same_d_qkv():
    B, N, E, H, P, dtype = 64, 65, 128, 2, 1, BF
    g = torch.Generator().manual_seed(9)
    dpl = _ints((3, B, H, N, 64), -3, 3, g).to(dtype).to(DEV)
    pre = _ints((2, B, H, N, 64), -3, 3, g).to(dtype).to(DEV)
    stats = torch.cat((_ints((2, B, H, N, 1), -1, 1, g), torch.ones(2, B, H, N, 1).double()), -1).float().to(DEV)
    qn = [_ints((64,), -2, 2, g).float().to(DEV) for _ in range(4)]
    outs = []
    for with_grads in (True, False):
        d_qkv = _nan((B * N, 3 * E), dtype)
        dn = list(_nan((4, 64))) if with_grads else [None] * 4
        _lib.check(_lib.load().vrr_qkv_rope_norm_bwd(_p(dpl), _p(pre), _p(stats), None, None, *map(_p, qn), _p(d_qkv),
                                                     None, None, *map(_p, dn), B, N, E, H, P, _lib.ROPE_NONE, DT[dtype],
                                                     _st()), "bwd")
        outs.append(d_qkv)
    assert torch.equal(outs[0], outs[1])


# ===================================================================================== model vs oracle
def _ref_attention(cfg, p, pre, x, rope, npre):
    """oracle/vit_torch.attention with q_norm / k_norm (when their parameters are in p) before RoPE and `npre`
    unrotated prefix tokens."""
    b, n, c = x.shape
    h, dh = cfg.num_heads, cfg.head_dim
    qkv = F.linear(x, p[pre + "qkv.weight"]).reshape(b, n, 3, h, dh).permute(2, 0, 3, 1, 4)
    q, k, v = qkv[0], qkv[1], qkv[2]
    if pre + "q_norm.weight" in p:
        qk = []
        for name, t in (("q_norm", q), ("k_norm", k)):
            y = F.layer_norm(t, (dh,), p[pre + name + ".weight"], p[pre + name + ".bias"], 1e-5)
            if y.requires_grad and not torch.is_autocast_enabled("cpu"):  # the fp32 oracle's magnitudes
                _scale_hook(y, F.layer_norm(t.detach(), (dh,), eps=1e-5), pre + name)
            qk.append(y)
        q, k = qk
    if rope is not None:
        qr, kr = V.rotate_half_pair(q[:, :, npre:], k[:, :, npre:], V.expand_cs(rope[0]), V.expand_cs(rope[1]))
        q = torch.cat([q[:, :, :npre], qr], dim=2)
        k = torch.cat([k[:, :, :npre], kr], dim=2)
    att = (q @ k.transpose(-2, -1)) * dh ** -0.5
    if cfg.pos_encoding == "relative":
        att = att + V.relative_bias(p["pos_embed.relative_position_bias_table"], p["pos_embed.relative_position_index"])
    elif cfg.pos_encoding == "polynomial":
        att = att + V.poly_bias(p["pos_embed.coefficients"], cfg.num_patches, h, cfg.poly_shared_heads)
    out = (att.softmax(dim=-1) @ v).transpose(1, 2).reshape(b, n, c)
    return F.linear(out, p[pre + "proj.weight"], p[pre + "proj.bias"])


_SCALES = {}  # "blocks.{i}.attn.q_norm.weight" -> max over channels of sum |dy xhat| (".bias": sum |dy|), fp32 oracle


def _scale_hook(y, xhat, key):
    """The magnitudes the q_norm / k_norm gradients are sums of (over every row of every head and image)."""
    def hook(dy):
        _SCALES[key + ".weight"] = (dy * xhat).abs().sum((0, 1, 2)).max().item()
        _SCALES[key + ".bias"] = dy.abs().sum((0, 1, 2)).max().item()
    y.register_hook(hook)


def _ref_forward(cfg, p, images, sites=None):
    """oracle/vit_torch's forward with QK-norm; registers, LayerScale and the SwiGLU MLP when their parameters are in
    p; `sites`: replayed dropout factors per block."""
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
        x = x + mul(mul(_ref_attention(cfg, p, pre + "attn.", y, rope, npre), fa), p.get(pre + "ls1.gamma"))
        y = F.layer_norm(x, (e,), p[pre + "norm2.weight"], p[pre + "norm2.bias"], 1e-5)
        h = F.linear(y, p[pre + "mlp.fc1.weight"], p[pre + "mlp.fc1.bias"])
        if p[pre + "mlp.fc2.weight"].shape[1] * 2 == h.shape[-1]:  # SwiGLUPacked
            gate, val = h.chunk(2, dim=-1)
            h = F.silu(gate) * val
        else:
            h = F.gelu(h)
        x = x + mul(mul(F.linear(mul(h, f1), p[pre + "mlp.fc2.weight"], p[pre + "mlp.fc2.bias"]), f2),
                    p.get(pre + "ls2.gamma"))
    x = F.layer_norm(x, (e,), p["norm.weight"], p["norm.bias"], 1e-5)
    return F.linear(x[:, 0], p["head.weight"], p["head.bias"])


def _cfg(kw):
    return V.VitConfig(**{k: v for k, v in kw.items() if k not in ("reg_tokens", "drop_rate", "drop_path_rate",
                                                                   "init_values", "mlp_layer", "qk_norm")})


def _build(kw, seed=0):
    torch.manual_seed(seed)
    model = VisionTransformer(**kw)
    with torch.no_grad():  # make zero / one initialised paths live; a swapped or mis-indexed g or b shows
        model.cls_token.normal_(std=0.02)
        if kw.get("reg_tokens", 0):
            model.reg_token.normal_(std=0.02)
        for n, prm in model.named_parameters():
            if n.endswith("_norm.weight"):  # q_norm / k_norm: randomised around their initial (1, 0)
                prm.uniform_(0.75, 1.25)
            elif n.endswith("_norm.bias"):
                prm.normal_(std=0.2)
            elif n.endswith(".bias"):
                prm.normal_(std=0.02)
            if n.endswith(".gamma"):
                prm.uniform_(0.25, 1.0)
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    return model.to(DEV), sd


def _check(model, logits, ref, p, bar, flat, p16=None, ref16=None):
    """Logits and every parameter gradient against the fp32 oracle: within `bar` of the largest reference value
    (flat) or of max(1, it).  In the 16-bit cases (p16 / ref16: the same oracle run under torch's 16-bit autocast)
    gradients that are sums which cancel lose most of their digits in any 16-bit evaluation - softmax-backward rows
    sum to zero, so the polynomial / table bias and RoPE frequency gradients cancel, and without RoPE the k_norm bias
    gradient is zero in exact arithmetic.  There a value may instead differ from the fp32 oracle by up to twice what
    torch's own 16-bit computation does, and the q_norm / k_norm gradients are measured against the magnitude of
    their summands (`bar` times max over channels of sum |dy xhat|, sum |dy|)."""
    def within(name, got, want, want16):
        d = (got - want).abs().max().item()
        if flat and name in _SCALES:
            return d <= bar * _SCALES[name], d / _SCALES[name]
        e = d / max(want.abs().max().item(), 1e-30) if flat else d / max(1.0, want.abs().max().item())
        return e <= bar or (want16 is not None and d <= 2 * (want16.float() - want).abs().max().item()), e

    ok, e = within("logits", logits.detach().float().cpu(), ref.detach(), None if ref16 is None else ref16.detach())
    assert ok, ("logits", e)
    names = set()
    for name, prm in model.named_parameters():
        want = p[name].grad if name in p else None
        if want is None:
            continue
        names.add(name)
        ok, e = within(name, prm.grad.detach().float().cpu(), want, None if p16 is None else p16[name].grad)
        assert ok, (name, e)
    norms = {n for n in p if "_norm." in n}
    assert norms and norms <= names  # every q_norm / k_norm gradient was compared


def _model_case(kw, images, labels, amp=None, bar=1e-5, flat=False, tc=False):
    model, sd = _build(dict(kw, qk_norm=True))
    fam = (_lib.family_count(TC), _lib.family_count(SIMT))
    with torch.autocast("cuda", dtype=amp or BF, enabled=amp is not None):
        logits = model(images.to(DEV))
        loss = F.cross_entropy(logits.float(), labels.to(DEV))
    loss.backward()
    torch.cuda.synchronize()
    if tc:
        assert _lib.family_count(TC) > fam[0] and _lib.family_count(SIMT) == fam[1]
    p = V.params_from_state_dict(sd)
    _SCALES.clear()
    ref = _ref_forward(_cfg(kw), p, images)
    F.cross_entropy(ref, labels).backward()
    assert {n for n in p if "_norm." in n} <= set(_SCALES)
    p16 = ref16 = None
    if amp is not None:
        p16 = V.params_from_state_dict(sd)
        with torch.autocast("cpu", dtype=amp):
            ref16 = _ref_forward(_cfg(kw), p16, images)
            loss16 = F.cross_entropy(ref16.float(), labels)
        loss16.backward()
    _check(model, logits, ref, p, bar, flat, p16, ref16)


MODES = ["none", "absolute", "relative", "polynomial", "rope-axial", "rope-mixed"]
TINY = dict(img_size=32, patch_size=4, in_chans=3, num_classes=10, embed_dim=192, depth=3, num_heads=3)
HD64 = dict(img_size=64, patch_size=8, in_chans=3, num_classes=10, embed_dim=256, depth=2, num_heads=4)
CFG3 = dict(img_size=224, patch_size=16, in_chans=3, num_classes=1000, embed_dim=768, depth=2, num_heads=12)


@pytest.mark.parametrize("mode", MODES)
def test_vit_tiny_with_qk_norm_fp32(mode):
    torch.manual_seed(1)
    images, labels = torch.randn(8, 3, 32, 32), torch.randint(0, 10, (8,))
    _model_case(dict(TINY, pos_encoding=mode), images, labels)


@pytest.mark.parametrize("mode", MODES)
def test_head_dim_64_with_qk_norm_bf16(mode):
    torch.manual_seed(2)
    images, labels = torch.randn(8, 3, 64, 64), torch.randint(0, 10, (8,))
    _model_case(dict(HD64, pos_encoding=mode), images, labels, amp=BF, bar=2e-2, flat=True, tc=True)


@pytest.mark.parametrize("mode", ["relative", "rope-mixed"])
def test_cfg3_geometry_with_qk_norm_bf16(mode):
    torch.manual_seed(3)
    images, labels = torch.randn(4, 3, 224, 224), torch.randint(0, 1000, (4,))
    _model_case(dict(CFG3, pos_encoding=mode), images, labels, amp=BF, bar=2e-2, flat=True, tc=True)


def test_qk_norm_under_fp16_autocast():
    torch.manual_seed(4)
    images, labels = torch.randn(4, 3, 224, 224), torch.randint(0, 1000, (4,))
    _model_case(dict(CFG3, pos_encoding="rope-axial"), images, labels, amp=HF, bar=2e-2, flat=True, tc=True)


def test_qk_norm_with_registers_layer_scale_swiglu_and_dropout_fp32():
    kw = dict(TINY, pos_encoding="rope-mixed", reg_tokens=4, init_values=1e-5, mlp_layer=SwiGLUPacked, mlp_ratio=5.33334,
              drop_rate=0.1, drop_path_rate=0.1, qk_norm=True)
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
        Hd = blk.mlp.fc2.in_features
        sites.append((ops.branch_factor((0.1, pp, N, 3 * i, seed), B, N, E).cpu(),
                      ops.branch_factor((0.1, 0.0, N, 3 * i + 1, seed), B, N, Hd).cpu(),
                      ops.branch_factor((0.1, pp, N, 3 * i + 2, seed), B, N, E).cpu()))
    assert all((s[1] == 0).any() for s in sites)
    p = V.params_from_state_dict(sd)
    ref = _ref_forward(_cfg(kw), p, images, sites)
    F.cross_entropy(ref, labels).backward()
    _check(model, logits, ref, p, 1e-5, False)


@pytest.mark.parametrize("amp", [None, BF], ids=["f32", "bf16"])
def test_qk_norm_false_changes_nothing(amp):
    kw = dict(TINY if amp is None else HD64, pos_encoding="rope-mixed")
    torch.manual_seed(0)
    base = VisionTransformer(**kw).to(DEV)
    torch.manual_seed(0)
    off = VisionTransformer(**kw, qk_norm=False).to(DEV)
    images = torch.randn(4, 3, kw["img_size"], kw["img_size"], device=DEV)
    outs = []
    for m in (base, off):
        before = _lib.launch_count()
        with torch.autocast("cuda", dtype=BF, enabled=amp is not None):
            logits = m(images)
            logits.float().sum().backward()
        torch.cuda.synchronize()
        outs.append((logits.detach(), _lib.launch_count() - before))
    assert outs[0][1] == outs[1][1] and torch.equal(outs[0][0], outs[1][0])


def test_graphed_inference_with_qk_norm():
    model, _ = _build(dict(HD64, pos_encoding="rope-mixed", reg_tokens=4, qk_norm=True))
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


def test_graphed_train_step_with_qk_norm():
    kw = dict(TINY, pos_encoding="rope-axial", qk_norm=True)
    model, _ = _build(kw)
    dp = BucketedDataParallel(model, bucket_mb=32.0)
    opt = torch.optim.AdamW(model.parameters(), lr=1e-4, weight_decay=0.01, fused=True, capturable=True)
    B = 16
    images, labels = torch.randn(B, 3, 32, 32, device=DEV), torch.randint(0, 10, (B,), device=DEV)
    runner = GraphedTrainStep(dp, opt, tuple(images.shape), 10, torch.device(DEV), bf16=False, use_graph=True)
    runner.prepare(images, labels)
    assert runner.graph is not None
    cfg = _cfg(kw)
    for _ in range(2):
        sd = {k: v.detach().clone().cpu() for k, v in model.state_dict().items()}
        loss = runner.run().item()
        ref = F.cross_entropy(_ref_forward(cfg, V.params_from_state_dict(sd, requires_grad=False), images.cpu()),
                              labels.cpu()).item()
        assert abs(loss - ref) <= 1e-5 * max(1.0, abs(ref)), (loss, ref)
    runner.close()


@pytest.mark.parametrize("amp", ["bf16", "fp16"])
def test_train_cli_with_qk_norm_learns_and_reloads(tmp_path, amp):
    argv = ["--dataset", "cifar10", "--pos_encoding", "rope-mixed", "--epochs", "2", "--batch_size", "32", "--synthetic",
            "--synthetic_size", "256", "--max_steps", "8", "--log_dir", str(tmp_path / "logs"), "--ckpt_dir",
            str(tmp_path / "ck"), "--amp", amp, "--embed_dim", "128", "--num_heads", "2", "--depth", "2", "--qk_norm"]
    log_file, ckpt = train.main(argv)
    rows = [r.split(",") for r in open(log_file).read().strip().splitlines()[1:]]
    assert len(rows) == 2 and all(math.isfinite(float(r[1])) for r in rows)
    assert float(rows[1][1]) < float(rows[0][1]), rows  # the training loss falls
    sd = torch.load(ckpt, map_location="cpu")
    assert sd["blocks.1.attn.k_norm.bias"].shape == (64,)
    m = VisionTransformer(img_size=32, patch_size=4, in_chans=3, num_classes=10, embed_dim=128, depth=2, num_heads=2,
                          pos_encoding="rope-mixed", qk_norm=True)
    m.load_state_dict(sd, strict=True)
