"""SwiGLU MLP on the device: ``vrr_gemm_swiglu`` / ``vrr_gemm_swiglu_bwd`` against the contract of include/vrr.h, and
the model with ``mlp_layer=SwiGLUPacked`` against an fp32 oracle with a SwiGLU block.

Kernels are called through the C ABI with NaN-filled outputs.  Integer operands make every accumulator exact, so the
gate and value ``g = T(acc + T(b))``, ``v`` and the products are checked bit for bit: ``act`` against ``T(s * v)``
with the kernel's own ``s = aux[:, H:]``, and ``aux[:, H:]`` against ``g`` itself where ``silu(g)`` rounds to ``g``
(g >= 16).  SiLU and its derivative are checked against float64 within the bound documented in csrc/common.cuh,
with the accumulator driven to chosen values (one-hot rows of x select a column of w1).  Shapes span more work units
than the grid has clusters, with ragged M, H (not a multiple of 128) and K.  The process-wide family selection is
restored in ``finally``.
"""
import ctypes
import math

import pytest
import torch
import torch.nn.functional as F

import train
from oracle import vit_torch as V
from vit_rpe_rope_b200 import VisionTransformer, _lib, ops
from vit_rpe_rope_b200.dp import BucketedDataParallel
from vit_rpe_rope_b200.models.vit import GluMlp, Mlp, SwiGLUPacked
from vit_rpe_rope_b200.runtime import GraphedInference, GraphedTrainStep

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
BF, HF, F32 = torch.bfloat16, torch.float16, torch.float32
DT = {F32: _lib.VRR_F32, BF: _lib.VRR_BF16, HF: _lib.VRR_F16}
NAN = float("nan")
EPS_SILU = 2.0 ** -20
FTZ = 2.0 ** -126  # sigma flushed to zero below the fp32 normal range: absolute error <= FTZ (1 + |g|)
UNIT = {F32: 2.0 ** -24, BF: 2.0 ** -8, HF: 2.0 ** -11}  # unit roundoff of the stored type
TINIEST = {F32: 1e-38, BF: 1e-38, HF: 2.0 ** -24}


def _p(t):
    return ops._ptr(t)


def _nan(shape, dtype):
    return torch.full(shape, NAN, device=DEV, dtype=dtype)


def _bits_equal(a, b):
    a, b = a.contiguous(), b.contiguous()
    assert a.dtype == b.dtype and a.shape == b.shape
    w = {4: torch.int32, 2: torch.int16}[a.element_size()]
    return torch.equal(a.view(w), b.view(w))


def _desc(drop):
    return None if drop is None else ctypes.byref(ops._drop_desc(drop))


def _fwd(x, w1, b1, H, aux=True, drop=None):
    M, K = x.shape
    act = _nan((M, H), x.dtype)
    a = _nan((M, 2 * H), x.dtype) if aux else None
    rc = _lib.load().vrr_gemm_swiglu(_p(x), _p(w1), _p(b1), _p(act), _p(a), M, H, K, DT[x.dtype], _desc(drop),
                                     ops._stream())
    _lib.check(rc, "vrr_gemm_swiglu")
    torch.cuda.synchronize()
    return act, a


def _bwd(dy, w2, aux):
    M, K = dy.shape
    H = w2.shape[1]
    dh = _nan((M, 2 * H), dy.dtype)
    db1 = _nan((2 * H,), F32)
    _lib.check(_lib.load().vrr_gemm_swiglu_bwd(_p(dy), _p(w2), _p(aux), _p(dh), _p(db1), M, H, K, DT[dy.dtype],
                                               ops._stream()), "vrr_gemm_swiglu_bwd")
    torch.cuda.synchronize()
    return dh, db1


def _family(dtype):
    return _lib.IMPL_SIMT if dtype == F32 else _lib.IMPL_TCGEN05


def _counted(dtype, fn):
    fam = _family(dtype)
    other = _lib.IMPL_TCGEN05 if fam == _lib.IMPL_SIMT else _lib.IMPL_SIMT
    before = (_lib.family_count(fam), _lib.family_count(other))
    out = fn()
    assert _lib.family_count(fam) == before[0] + 1 and _lib.family_count(other) == before[1]
    return out


def _silu64(g):
    sig = 1.0 / (1.0 + torch.exp(-g))
    return g * sig, sig + g * sig * (1.0 - sig), sig


def _within(got, want, bound, dtype):
    """|got - want| <= bound + rounding of `want` to the stored type."""
    err = (got.double() - want).abs()
    lim = bound + UNIT[dtype] * want.abs() + TINIEST[dtype]
    bad = err > lim
    assert not bad.any(), (err[bad][:5], want[bad][:5])


# ===================================================================================== SiLU
@pytest.mark.parametrize("dtype", [F32, HF, BF])
def test_silu_and_its_derivative_against_float64(dtype):
    """One-hot rows of x pick column m % K of w1: the gate accumulator is exactly the chosen value, v is 1."""
    H, K, M = 512, 16, 2048
    vals = torch.linspace(-40.0, 40.0, H * K, dtype=torch.float64)
    vals = torch.cat([vals[: H * K - 8], torch.tensor([0.0, -0.0, 1e-3, -1e-3, 88.5, -88.5, 100.0, -100.0],
                                                      dtype=torch.float64)])
    wg = vals.view(H, K).to(dtype)
    w1 = torch.cat([wg, torch.ones(H, K, dtype=dtype)]).to(DEV)
    x = F.one_hot(torch.arange(M) % K, K).to(dtype).to(DEV)
    b1 = torch.zeros(2 * H, device=DEV)
    act, aux = _counted(dtype, lambda: _fwd(x, w1, b1, H))
    g = wg.double().t()[torch.arange(M) % K]  # [M][H]: g[m][j] = wg[j][m % K]
    s, ds, sig = _silu64(g)
    bs = EPS_SILU * (1 + g.abs()) * s.abs() + FTZ * (1 + g.abs())
    bds = EPS_SILU * (1 + g.abs()) * (sig + s.abs() * (1 - sig)) + FTZ * (1 + g.abs())
    _within(aux[:, H:].cpu(), s, bs, dtype)  # fp32: the kernel's values themselves; else their rounding to T
    _within(aux[:, :H].cpu(), ds, bds, dtype)
    assert _bits_equal(act, aux[:, H:])  # v = 1: T(s * 1) = s


# ===================================================================================== forward, integer operands
SHAPES = [(4133, 520, 136), (700, 2048, 768), (37, 24, 8)]


def _int_case(M, H, K, dtype, seed, big_gate=False):
    g = torch.Generator().manual_seed(seed)
    if big_gate:  # g = acc + 16 with acc in [0, K]: silu(g) rounds to g in bf16 / fp16
        x = torch.randint(0, 2, (M, K), generator=g).to(dtype)
        wg = torch.randint(0, 2, (H, K), generator=g).to(dtype)
        bg = torch.full((H,), 16.0)
    else:
        x = torch.randint(-2, 3, (M, K), generator=g).to(dtype)
        wg = torch.randint(-2, 3, (H, K), generator=g).to(dtype)
        bg = torch.randint(-3, 4, (H,), generator=g).float()
    wv = torch.randint(-2, 3, (H, K), generator=g).to(dtype)
    bv = torch.randint(-3, 4, (H,), generator=g).float()
    w1 = torch.cat([wg, wv])
    b1 = torch.cat([bg, bv])
    gref = (x.double() @ wg.double().t() + bg.double()).to(dtype)  # exact accumulators, one rounding to T
    vref = (x.double() @ wv.double().t() + bv.double()).to(dtype)
    return x.to(DEV), w1.to(DEV), b1.to(DEV), gref, vref


@pytest.mark.parametrize("dtype", [BF, HF, F32])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_forward_on_integers(shape, dtype):
    M, H, K = shape
    if dtype != F32 and (H % 8 or K % 8):
        pytest.skip("tcgen05 shapes")
    x, w1, b1, gref, vref = _int_case(M, H, K, dtype, seed=M + H)
    act, aux = _counted(dtype, lambda: _fwd(x, w1, b1, H))
    act, aux = act.cpu(), aux.cpu()
    s = aux[:, H:]
    assert _bits_equal(act, (s.float() * vref.float()).to(dtype))  # act = T(s v) with the kernel's s, bit for bit
    s64, ds64, sig = _silu64(gref.double())
    ga, va = 1 + gref.double().abs(), vref.double().abs()
    _within(s, s64, EPS_SILU * ga * s64.abs() + FTZ * ga, dtype)
    _within(aux[:, :H], vref.double() * ds64,
            va * (EPS_SILU * ga * (sig + s64.abs() * (1 - sig)) + FTZ * ga) + 2 * UNIT[F32] * (va * ds64.abs()), dtype)
    act_only, none = _fwd(x, w1, b1, H, aux=False)  # torch.no_grad: the same act, nothing else
    assert none is None and _bits_equal(act_only.cpu(), act)


@pytest.mark.parametrize("dtype", [BF, HF])
@pytest.mark.parametrize("shape", SHAPES[:2], ids=lambda s: "x".join(map(str, s)))
def test_gate_and_value_bit_for_bit(shape, dtype):
    """silu(g) rounds to g for g >= 16: aux[:, H:] IS the gate, and act = T(g v) exposes the value."""
    M, H, K = shape
    x, w1, b1, gref, vref = _int_case(M, H, K, dtype, seed=7, big_gate=True)
    act, aux = _fwd(x, w1, b1, H)
    assert _bits_equal(aux[:, H:].cpu(), gref)
    assert _bits_equal(act.cpu(), (gref.float() * vref.float()).to(dtype))


@pytest.mark.parametrize("dtype", [BF, F32])
def test_forward_dropout_replays_the_mask(dtype):
    M, H, K = 1500, 264, 64
    x, w1, b1, _, _ = _int_case(M, H, K, dtype, seed=11)
    p, seed = 0.25, torch.tensor([123456789], device=DEV, dtype=torch.int64)
    drop = (p, 0.0, 1, 7, seed)
    act0, aux0 = _fwd(x, w1, b1, H)
    act1, aux1 = _counted(dtype, lambda: _fwd(x, w1, b1, H, drop=drop))
    keep, _ = ops.dropout_mask(drop, M, H)
    f = keep.float() * ops.drop_scale(p, 0.0)
    assert 0.6 < keep.float().mean().item() < 0.9
    assert _bits_equal(act1, (act0.float() * f).to(dtype))                        # T(T(s v) f)
    assert _bits_equal(aux1[:, H:], (aux0[:, H:].float() * f).to(dtype))          # T(s f)
    lo0, lo1 = aux0[:, :H].float(), aux1[:, :H].float()
    assert torch.equal(lo1 == 0, (keep == 0) | (lo0 == 0))
    assert ((lo1 - lo0 * f).abs() <= 3 * UNIT[dtype] * (lo0 * f).abs()).all()    # T(fl(v silu') f) vs T(T(..) f)
    # no dropout desc and p = 0 are the plain kernel
    act2, aux2 = _fwd(x, w1, b1, H, drop=(0.0, 0.0, 1, 7, seed))
    assert _bits_equal(act2, act0) and _bits_equal(aux2, aux0)


# ===================================================================================== backward
@pytest.mark.parametrize("dtype", [BF, HF, F32])
@pytest.mark.parametrize("shape", [(4133, 520, 136), (900, 2048, 768), (300, 64, 40), (53, 6, 10)],
                         ids=lambda s: "x".join(map(str, s)))
def test_backward_on_integers(shape, dtype):
    M, H, K = shape
    if dtype != F32 and (H % 8 or K % 8):
        pytest.skip("tcgen05 shapes")
    g = torch.Generator().manual_seed(M + K)
    dy = torch.randint(-2, 3, (M, K), generator=g).to(dtype)
    w2 = torch.randint(-1, 2, (K, H), generator=g).to(dtype)  # fc2.weight [E][H]
    aux = torch.randint(-3, 4, (M, 2 * H), generator=g).to(dtype)
    dh, db1 = _counted(dtype, lambda: _bwd(dy.to(DEV), w2.to(DEV), aux.to(DEV)))
    dA = (dy.double() @ w2.double()).float()  # exact
    want = (torch.cat([dA, dA], 1) * aux.float()).to(dtype)
    assert _bits_equal(dh.cpu(), want)
    assert torch.equal(db1.cpu().double(), want.double().sum(0))  # integer partial sums: exact in any order


# ===================================================================================== dispatch and arguments
def test_dispatch_and_arguments():
    lib = _lib.load()
    x = torch.ones(64, 24, device=DEV, dtype=BF)
    w1 = torch.ones(24, 24, device=DEV, dtype=BF)  # H = 12: not a tcgen05 shape
    b1 = torch.zeros(24, device=DEV)
    act, aux = _nan((64, 12), BF), _nan((64, 24), BF)
    prev = _lib.set_impl(_lib.IMPL_TCGEN05)
    try:
        rc = lib.vrr_gemm_swiglu(_p(x), _p(w1), _p(b1), _p(act), _p(aux), 64, 12, 24, _lib.VRR_BF16, None, ops._stream())
        assert rc == -2  # VRR_ERR_UNSUPPORTED
        rc = lib.vrr_gemm_swiglu_bwd(_p(x), _p(w1), _p(aux), _p(aux), _p(b1), 64, 12, 24, _lib.VRR_BF16, ops._stream())
        assert rc == -2
        _lib.set_impl(_lib.IMPL_SIMT)
        _counted(F32, lambda: _fwd(x, w1, b1, 12))  # a forced SIMT family takes it
    finally:
        _lib.set_impl(prev)
    bad = [
        (None, w1, b1, act, aux, 64, 12, 24, _lib.VRR_BF16, None),
        (x, w1, None, act, aux, 64, 12, 24, _lib.VRR_BF16, None),
        (x, w1, b1, act, aux, 0, 12, 24, _lib.VRR_BF16, None),
        (x, w1, b1, act, aux, 64, 12, 24, 7, None),
        (x, w1, b1, act, aux, 64, 12, 24, _lib.VRR_BF16,
         (0.1, 0.1, 1, 0, torch.zeros(1, device=DEV, dtype=torch.int64))),  # p_path must be 0
    ]
    for a in bad:
        args = [(_p(t) if isinstance(t, torch.Tensor) else t) for t in a[:9]]
        assert lib.vrr_gemm_swiglu(*args, _desc(a[9]), ops._stream()) == -1
    assert lib.vrr_gemm_swiglu_bwd(_p(x), _p(w1), None, _p(aux), _p(b1), 64, 12, 24, _lib.VRR_BF16, ops._stream()) == -1
    assert lib.vrr_gemm_swiglu_bwd(_p(x), _p(w1), _p(aux), _p(aux), _p(b1), 64, 11, 24, _lib.VRR_BF16, ops._stream()) == -1


# ===================================================================================== model vs oracle
def _ref_attention(cfg, p, pre, x, rope, npre):
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
    """oracle/vit_torch's forward with timm's SwiGLUPacked block: fc2(silu(h[:, :H]) * h[:, H:]) for h = fc1(y);
    LayerScale and registers when their parameters are in p; `sites`: replayed dropout factors per block."""
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
        if npre == 1 and cfg.pos_encoding in ("relative", "polynomial"):
            a = V.attention(cfg, p, pre + "attn.", y, "pos_embed.", rope)
        else:
            a = _ref_attention(cfg, p, pre + "attn.", y, rope, npre)
        x = x + mul(mul(a, fa), p.get(pre + "ls1.gamma"))
        y = F.layer_norm(x, (e,), p[pre + "norm2.weight"], p[pre + "norm2.bias"], 1e-5)
        gate, val = F.linear(y, p[pre + "mlp.fc1.weight"], p[pre + "mlp.fc1.bias"]).chunk(2, dim=-1)
        h = mul(F.silu(gate) * val, f1)
        x = x + mul(mul(F.linear(h, p[pre + "mlp.fc2.weight"], p[pre + "mlp.fc2.bias"]), f2), p.get(pre + "ls2.gamma"))
    x = F.layer_norm(x, (e,), p["norm.weight"], p["norm.bias"], 1e-5)
    return F.linear(x[:, 0], p["head.weight"], p["head.bias"])


def _cfg(kw):
    return V.VitConfig(**{k: v for k, v in kw.items()
                          if k not in ("reg_tokens", "drop_rate", "drop_path_rate", "init_values", "mlp_layer")})


def _build(kw, seed=0):
    torch.manual_seed(seed)
    model = VisionTransformer(**kw)
    with torch.no_grad():  # make zero-initialised paths live
        model.cls_token.normal_(std=0.02)
        if kw.get("reg_tokens", 0):
            model.reg_token.normal_(std=0.02)
        for n, prm in model.named_parameters():
            if n.endswith(".bias"):
                prm.normal_(std=0.02)
            if n.endswith(".gamma"):
                prm.uniform_(0.25, 1.0)
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
    assert {n for n in p if ".mlp.fc" in n} <= names  # every SwiGLU parameter gradient was compared


def _model_case(kw, images, labels, amp=None, bar=1e-5, flat=False, tc=False):
    model, sd = _build(kw)
    assert all(type(b.mlp) is GluMlp for b in model.blocks)
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


MODES = ["none", "absolute", "relative", "polynomial", "rope-axial", "rope-mixed"]
SW = dict(mlp_layer=SwiGLUPacked, mlp_ratio=5.33334)  # E = 192, 768: fc1 1024, 4096 (the GELU MLP's parameters)
TINY = dict(img_size=32, patch_size=4, in_chans=3, num_classes=10, embed_dim=192, depth=3, num_heads=3, **SW)
HD64 = dict(img_size=64, patch_size=8, in_chans=3, num_classes=10, embed_dim=256, depth=2, num_heads=4, **dict(SW, mlp_ratio=5.5))
CFG3 = dict(img_size=224, patch_size=16, in_chans=3, num_classes=1000, embed_dim=768, depth=2, num_heads=12, **SW)


@pytest.mark.parametrize("mode", MODES)
def test_vit_tiny_with_swiglu_fp32(mode):
    torch.manual_seed(1)
    images, labels = torch.randn(8, 3, 32, 32), torch.randint(0, 10, (8,))
    _model_case(dict(TINY, pos_encoding=mode), images, labels)


@pytest.mark.parametrize("mode", MODES)
def test_head_dim_64_with_swiglu_bf16(mode):
    torch.manual_seed(2)
    images, labels = torch.randn(8, 3, 64, 64), torch.randint(0, 10, (8,))
    _model_case(dict(HD64, pos_encoding=mode), images, labels, amp=BF, bar=2e-2, flat=True, tc=True)


def test_swiglu_under_fp16_autocast():
    torch.manual_seed(4)
    images, labels = torch.randn(4, 3, 224, 224), torch.randint(0, 1000, (4,))
    _model_case(dict(CFG3, pos_encoding="rope-mixed"), images, labels, amp=HF, bar=2e-2, flat=True, tc=True)


def test_swiglu_with_layer_scale_and_registers_fp32():
    torch.manual_seed(5)
    images, labels = torch.randn(8, 3, 32, 32), torch.randint(0, 10, (8,))
    _model_case(dict(TINY, pos_encoding="rope-mixed", reg_tokens=4, init_values=1e-5), images, labels)


def test_swiglu_with_dropout_and_stochastic_depth_fp32():
    kw = dict(TINY, pos_encoding="rope-mixed", drop_rate=0.1, drop_path_rate=0.1)
    model, sd = _build(kw)
    model.train()
    B, N = 8, 65
    torch.manual_seed(6)
    images, labels = torch.randn(B, 3, 32, 32), torch.randint(0, 10, (B,))
    logits = model(images.to(DEV))
    F.cross_entropy(logits, labels.to(DEV)).backward()
    seed, E = model._drop_seed, kw["embed_dim"]
    sites = []
    for i, blk in enumerate(model.blocks):
        pp = getattr(blk.drop_path, "drop_prob", 0.0)
        Hd = blk.mlp.fc2.in_features  # drop1 acts on the [B N, H] product
        sites.append((ops.branch_factor((0.1, pp, N, 3 * i, seed), B, N, E).cpu(),
                      ops.branch_factor((0.1, 0.0, N, 3 * i + 1, seed), B, N, Hd).cpu(),
                      ops.branch_factor((0.1, pp, N, 3 * i + 2, seed), B, N, E).cpu()))
    assert all((s[1] == 0).any() for s in sites)
    p = V.params_from_state_dict(sd)
    ref = _ref_forward(_cfg(kw), p, images, sites)
    F.cross_entropy(ref, labels).backward()
    _check(model, logits, ref, p, 1e-5, False)


def test_swiglu_runs_the_fused_loop():
    model, _ = _build(dict(TINY, pos_encoding="rope-mixed"))
    x = torch.randn(2, 3, 32, 32, device=DEV)
    assert model._fusable(ops.patch_embed(x, model.patch_embed.weight, model.patch_embed.bias, model.cls_token, None,
                                          model.patch_size))
    ops.PROFILE_EVENTS = []
    try:
        model(x).sum().backward()
        names = [e[0] for e in ops.PROFILE_EVENTS]
    finally:
        ops.PROFILE_EVENTS = None
    depth = len(model.blocks)
    assert names.count("fc1_fwd") == depth and names.count("fc2_dx") == depth
    assert names.count("add_layernorm_fwd") == 2 * depth - 1  # the fused loop, not Block.forward


@pytest.mark.parametrize("amp", [None, BF], ids=["f32", "bf16"])
def test_mlp_layer_mlp_changes_nothing(amp):
    kw = dict(TINY if amp is None else HD64, pos_encoding="rope-mixed")
    kw = {k: v for k, v in kw.items() if k not in SW}
    torch.manual_seed(0)
    base = VisionTransformer(**kw).to(DEV)
    torch.manual_seed(0)
    explicit = VisionTransformer(**kw, mlp_layer=Mlp).to(DEV)
    images = torch.randn(4, 3, kw["img_size"], kw["img_size"], device=DEV)
    outs = []
    for m in (base, explicit):
        before = _lib.launch_count()
        with torch.autocast("cuda", dtype=BF, enabled=amp is not None):
            logits = m(images)
        torch.cuda.synchronize()
        outs.append((logits.detach(), _lib.launch_count() - before))
    assert outs[0][1] == outs[1][1] and torch.equal(outs[0][0], outs[1][0])


def test_graphed_inference_with_swiglu():
    model, _ = _build(dict(HD64, pos_encoding="rope-mixed"))
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


def test_graphed_train_step_with_swiglu():
    kw = dict(TINY, pos_encoding="rope-axial")
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


def test_train_cli_with_swiglu_learns_and_reloads(tmp_path):
    argv = ["--dataset", "cifar10", "--pos_encoding", "rope-mixed", "--epochs", "2", "--batch_size", "32", "--synthetic",
            "--synthetic_size", "256", "--max_steps", "8", "--log_dir", str(tmp_path / "logs"), "--ckpt_dir",
            str(tmp_path / "ck"), "--amp", "bf16", "--embed_dim", "128", "--num_heads", "2", "--depth", "2",
            "--mlp_layer", "swiglu", "--mlp_ratio", "5"]
    log_file, ckpt = train.main(argv)
    rows = [r.split(",") for r in open(log_file).read().strip().splitlines()[1:]]
    assert len(rows) == 2 and all(math.isfinite(float(r[1])) for r in rows)
    assert float(rows[1][1]) < float(rows[0][1]), rows  # the training loss falls
    sd = torch.load(ckpt, map_location="cpu")
    assert tuple(sd["blocks.0.mlp.fc1.weight"].shape) == (640, 128) and tuple(sd["blocks.0.mlp.fc2.weight"].shape) == (128, 320)
    m = VisionTransformer(img_size=32, patch_size=4, in_chans=3, num_classes=10, embed_dim=128, depth=2, num_heads=2,
                          pos_encoding="rope-mixed", mlp_layer=SwiGLUPacked, mlp_ratio=5.0)
    m.load_state_dict(sd, strict=True)
