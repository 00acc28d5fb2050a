"""LayerScale on the device: the add+LayerNorm kernels that apply it and reduce its gradient, and the model against
the fp32 oracle with LayerScale.

Kernels are called through the C ABI with NaN-filled outputs at shapes sized from the device (several rows per warp of
the largest grid) and compared BIT FOR BIT with the plain kernels fed the already-scaled fp32 branch
(b' = fl(fl(f * branch) * ls), the contract of include/vrr.h).  The LayerScale gradient is a column sum whose order is
not fixed: it is checked exactly on integer data whose every partial sum is exact in fp32, and within a summation
bound on random data.  The model's gammas are randomised after construction: at 1e-5 a mishandled branch would hide
under the tolerance.  Process-wide options are restored in ``finally``.
"""
import ctypes
import math

import pytest
import torch
import torch.nn.functional as F

import train
from oracle import vit_torch as V
from vit_rpe_rope_b200 import VisionTransformer, _lib, ops
from vit_rpe_rope_b200.models.vit import LayerScale
from vit_rpe_rope_b200.runtime import GraphedInference

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
BF, HF, F32 = torch.bfloat16, torch.float16, torch.float32
DT = {F32: _lib.VRR_F32, BF: _lib.VRR_BF16, HF: _lib.VRR_F16}
NAN = float("nan")


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _p(t):
    return ops._ptr(t)


def _st():
    return ops._stream()


def _seed(value):
    return torch.tensor([value], device=DEV, dtype=torch.int64)


def _nan(shape, dtype=F32):
    return torch.full(shape, NAN, device=DEV, dtype=dtype)


def _bits_equal(a, b):
    a, b = a.contiguous(), b.contiguous()
    assert a.dtype == b.dtype and a.shape == b.shape
    w = {4: torch.int32, 2: torch.int16}[a.element_size()]
    return torch.equal(a.view(w), b.view(w))


def _set_option(name, value):
    _lib.check(_lib.load().vrr_set_option(name.encode(), int(value)), name)


def _desc(drop):
    return None if drop is None else ctypes.byref(ops._drop_desc(drop))


# ===================================================================================== add + LayerNorm
def _fwd(x, br, gamma, beta, y_dtype, drop=None, ls=None, entry="ls"):
    """entry: "ls" (vrr_add_layernorm_ls_fwd), "drop" or "plain"."""
    lib = _lib.load()
    M, E = x.shape
    x_new, y = _nan((M, E)), _nan((M, E), y_dtype)
    mean, rstd = _nan((M,)), _nan((M,))
    args = (_p(x), _p(br), _p(x_new), _p(gamma), _p(beta), _p(y), _p(mean), _p(rstd), M, E, 1e-5, DT[br.dtype],
            DT[y_dtype])
    if entry == "ls":
        rc = lib.vrr_add_layernorm_ls_fwd(*args, _desc(drop), _p(ls), _st())
    elif entry == "drop":
        rc = lib.vrr_add_layernorm_drop_fwd(*args, _desc(drop), _st())
    else:
        rc = lib.vrr_add_layernorm_fwd(*args, _st())
    _lib.check(rc, "add_layernorm fwd")
    return x_new, y, mean, rstd


def _bwd(dy, dxn, x_new, gamma, mean, rstd, br_dtype, drop=None, ls=None, branch=None, d_ls=True, entry="ls"):
    """-> dx, d_branch, [3][E] (dgamma, dbeta, d_ls: the last row stays NaN when d_ls is not asked for)."""
    lib = _lib.load()
    M, E = x_new.shape
    dx, dbr, dgb = _nan((M, E)), _nan((M, E), br_dtype), _nan((3, E))
    args = (_p(dy), _p(dxn), _p(x_new), _p(gamma), _p(mean), _p(rstd), _p(dx), _p(dbr), _p(dgb[0]), _p(dgb[1]), M, E,
            DT[br_dtype], DT[dy.dtype])
    if entry == "ls":
        rc = lib.vrr_add_layernorm_ls_bwd(*args, _desc(drop), _p(ls), _p(branch), _p(dgb[2]) if d_ls else None, _st())
    elif entry == "drop":
        rc = lib.vrr_add_layernorm_drop_bwd(*args, _desc(drop), _st())
    else:
        rc = lib.vrr_add_layernorm_bwd(*args, _st())
    _lib.check(rc, "add_layernorm bwd")
    return dx, dbr, dgb


# (E, ln_reg, ln_bwd_minb): register-resident NV 2/4/6/8 with every backward launch shape, generic VEC 4 and VEC 1
VARIANTS = [(256, 1, 3), (512, 1, 2), (768, 1, 3), (768, 1, 1), (768, 1, 2), (1024, 1, 3), (1024, 1, 2),
            (768, 0, 3), (640, 1, 3), (192, 1, 3)]
DROPS = [None, (0.0, 0.3, 197, 4), (0.2, 0.1, 197, 5)]  # none, stochastic depth only, element + path


def _rows(N=197):
    return N * max(8, 3 * 4 * 8 * _sms() // N)  # whole images; ~3 rows per warp of the largest grid (4 CTAs x 8 warps)


@pytest.mark.parametrize("E,ln_reg,minb", VARIANTS)
@pytest.mark.parametrize("bdt", [F32, BF, HF], ids=["f32", "bf16", "f16"])
def test_add_layernorm_ls_is_the_plain_kernel_fed_the_scaled_branch(E, ln_reg, minb, bdt):
    N, M = 197, _rows()
    g = torch.Generator(device=DEV).manual_seed(E + 7)
    x = torch.randn(M, E, device=DEV, generator=g)
    br = torch.randn(M, E, device=DEV, generator=g).to(bdt)
    gamma, beta = 1 + 0.1 * torch.randn(E, device=DEV, generator=g), 0.1 * torch.randn(E, device=DEV, generator=g)
    ls = 0.25 + 0.75 * torch.rand(E, device=DEV, generator=g)
    ydt = F32 if bdt == F32 else bdt
    dy = torch.randn(M, E, device=DEV, generator=g).to(ydt)
    dxn = torch.randn(M, E, device=DEV, generator=g)
    try:
        _set_option("ln_reg", ln_reg)
        _set_option("ln_bwd_minb", minb)
        for dd in DROPS:
            drop = None if dd is None else dd + (_seed(0x5EED0 + E),)
            f = None if drop is None else ops.branch_factor(drop, M // N, N, E).view(M, E)
            fb = br.float() if f is None else br.float() * f
            ref = _fwd(x, fb * ls, gamma, beta, ydt, entry="plain")
            got = _fwd(x, br, gamma, beta, ydt, drop, ls)
            for r, o in zip(ref, got):
                assert _bits_equal(o, r), dd
            rdx, _, rdgb = _bwd(dy, dxn, ref[0], gamma, ref[2], ref[3], F32, entry="plain")
            gdx, gdbr, gdgb = _bwd(dy, dxn, got[0], gamma, got[2], got[3], bdt, drop, ls, br)
            t = rdx if f is None else rdx * f  # fl(dx * f)
            assert _bits_equal(gdx, rdx), dd
            assert _bits_equal(gdbr, (t * ls).to(bdt)), dd
            # dgamma / dbeta / d_ls: fp32 column sums whose order across CTAs is not fixed - bounded by the sums of |terms|
            xh = (ref[0].double() - ref[2].double()[:, None]) * ref[3].double()[:, None]
            terms = t.double() * br.double()
            want = torch.stack([rdgb[0].double(), rdgb[1].double(), terms.sum(0)])
            scale = torch.stack([(dy.double() * xh).abs().sum(0), dy.double().abs().sum(0), terms.abs().sum(0)])
            assert ((gdgb.double() - want).abs() <= 2e-5 * scale).all(), dd
            # without d_ls the branch is not read: same dx / d_branch, the d_ls row untouched
            ndx, ndbr, ndgb = _bwd(dy, dxn, got[0], gamma, got[2], got[3], bdt, drop, ls, None, d_ls=False)
            assert _bits_equal(ndx, gdx) and _bits_equal(ndbr, gdbr) and torch.isnan(ndgb[2]).all()
        # ls NULL is exactly the drop / plain entry points
        for dd in (None, DROPS[2]):
            drop = None if dd is None else dd + (_seed(3),)
            a = _fwd(x, br, gamma, beta, ydt, drop, None)
            b = _fwd(x, br, gamma, beta, ydt, drop, entry="drop" if drop else "plain")
            assert all(_bits_equal(u, v) for u, v in zip(a, b))
            ga = _bwd(dy, dxn, a[0], gamma, a[2], a[3], bdt, drop, None, None, d_ls=False)
            gb = _bwd(dy, dxn, a[0], gamma, a[2], a[3], bdt, drop, entry="drop" if drop else "plain")
            assert _bits_equal(ga[0], gb[0]) and _bits_equal(ga[1], gb[1])
    finally:
        _set_option("ln_reg", 1)
        _set_option("ln_bwd_minb", 3)


@pytest.mark.parametrize("E,ln_reg,minb", VARIANTS)
@pytest.mark.parametrize("bdt", [F32, BF, HF], ids=["f32", "bf16", "f16"])
def test_ls_gradient_is_exact_on_integers(E, ln_reg, minb, bdt):
    """dy = 0 makes dx == d_xnew exactly; integer d_xnew and branch with p = p_path = 0.5 (f in {0, 4}) keep every
    partial sum an integer below 2^24, so d_ls is exact in any summation order and equals the float64 sum."""
    N, M = 197, _rows()
    g = torch.Generator(device=DEV).manual_seed(E + 11)
    x = torch.randn(M, E, device=DEV, generator=g)
    br = torch.randint(-8, 9, (M, E), device=DEV, generator=g).to(bdt)
    dxn = torch.randint(-8, 9, (M, E), device=DEV, generator=g).float()
    gamma, beta = 1 + 0.1 * torch.randn(E, device=DEV, generator=g), 0.1 * torch.randn(E, device=DEV, generator=g)
    ls = 0.25 + 0.75 * torch.rand(E, device=DEV, generator=g)
    ydt = F32 if bdt == F32 else bdt
    dy = torch.zeros(M, E, device=DEV, dtype=ydt)
    drop = (0.5, 0.5, N, 9, _seed(0xABCDEF + E))
    assert M * 4 * 64 < 2 ** 24
    try:
        _set_option("ln_reg", ln_reg)
        _set_option("ln_bwd_minb", minb)
        fw = _fwd(x, br, gamma, beta, ydt, drop, ls)
        dx, dbr, dgb = _bwd(dy, dxn, fw[0], gamma, fw[2], fw[3], bdt, drop, ls, br)
        assert torch.equal(dx, dxn)
        f = ops.branch_factor(drop, M // N, N, E).view(M, E)
        assert set(f.unique().tolist()) == {0.0, 4.0}
        want = ((dxn * f).double() * br.double()).sum(0)
        assert torch.equal(dgb[2].double(), want)
    finally:
        _set_option("ln_reg", 1)
        _set_option("ln_bwd_minb", 3)


# ===================================================================================== model vs oracle
def _ref_attention(cfg, p, pre, x, rope, npre):
    """oracle/vit_torch.attention with `npre` unrotated prefix tokens (rotary or no bias)."""
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
    """timm's block order with LayerScale: x = x + ls1(f_attn * attn(norm1(x))); x = x + ls2(f_mlp * mlp(norm2(x)));
    registers when "reg_token" is in p; `sites`: replayed dropout factors per block."""
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
        if npre == 1:
            a = V.attention(cfg, p, pre + "attn.", y, "pos_embed.", rope)
        else:
            a = _ref_attention(cfg, p, pre + "attn.", y, rope, npre)
        x = x + mul(mul(a, fa), p.get(pre + "ls1.gamma"))
        y = F.layer_norm(x, (e,), p[pre + "norm2.weight"], p[pre + "norm2.bias"], 1e-5)
        h = mul(F.gelu(F.linear(y, p[pre + "mlp.fc1.weight"], p[pre + "mlp.fc1.bias"])), f1)
        x = x + mul(mul(F.linear(h, p[pre + "mlp.fc2.weight"], p[pre + "mlp.fc2.bias"]), f2), p.get(pre + "ls2.gamma"))
    x = F.layer_norm(x, (e,), p["norm.weight"], p["norm.bias"], 1e-5)
    return F.linear(x[:, 0], p["head.weight"], p["head.bias"])


def _cfg(kw):
    return V.VitConfig(**{k: v for k, v in kw.items()
                          if k not in ("reg_tokens", "drop_rate", "drop_path_rate", "init_values")})


def _build(kw, seed=0):
    torch.manual_seed(seed)
    model = VisionTransformer(**kw)
    with torch.no_grad():  # make zero / tiny initialised paths live; gammas far from 1e-5 and from each other
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
    gammas = {n for n in p if n.endswith(".gamma") and n.startswith("blocks.")}
    assert gammas and gammas <= names  # every LayerScale gradient was compared


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


MODES = ["none", "absolute", "relative", "polynomial", "rope-axial", "rope-mixed"]
TINY = dict(img_size=32, patch_size=4, in_chans=3, num_classes=10, embed_dim=192, depth=3, num_heads=3)
HD64 = dict(img_size=64, patch_size=8, in_chans=3, num_classes=10, embed_dim=256, depth=2, num_heads=4)
CFG3 = dict(img_size=224, patch_size=16, in_chans=3, num_classes=1000, embed_dim=768, depth=2, num_heads=12)


@pytest.mark.parametrize("mode", MODES)
def test_vit_tiny_with_layer_scale_fp32(mode):
    torch.manual_seed(1)
    images, labels = torch.randn(8, 3, 32, 32), torch.randint(0, 10, (8,))
    _model_case(dict(TINY, pos_encoding=mode, init_values=1e-5), images, labels)


@pytest.mark.parametrize("mode", MODES)
def test_head_dim_64_with_layer_scale_bf16(mode):
    torch.manual_seed(2)
    images, labels = torch.randn(8, 3, 64, 64), torch.randint(0, 10, (8,))
    _model_case(dict(HD64, pos_encoding=mode, init_values=1e-5), images, labels, amp=BF, bar=2e-2, flat=True, tc=True)


@pytest.mark.parametrize("mode", ["absolute", "rope-mixed"])
def test_cfg3_geometry_with_layer_scale_bf16(mode):
    torch.manual_seed(3)
    images, labels = torch.randn(4, 3, 224, 224), torch.randint(0, 1000, (4,))
    _model_case(dict(CFG3, pos_encoding=mode, init_values=1e-5), images, labels, amp=BF, bar=2e-2, flat=True, tc=True)


def test_layer_scale_under_fp16_autocast():
    torch.manual_seed(4)
    images, labels = torch.randn(4, 3, 224, 224), torch.randint(0, 1000, (4,))
    _model_case(dict(CFG3, pos_encoding="rope-mixed", init_values=1e-5), images, labels, amp=HF, bar=2e-2, flat=True,
                tc=True)


def test_layer_scale_with_registers_fp32():
    torch.manual_seed(5)
    images, labels = torch.randn(8, 3, 32, 32), torch.randint(0, 10, (8,))
    _model_case(dict(TINY, pos_encoding="rope-mixed", reg_tokens=4, init_values=1e-5), images, labels)


@pytest.mark.parametrize("R", [0, 4])
def test_layer_scale_with_dropout_and_stochastic_depth_fp32(R):
    kw = dict(TINY, pos_encoding="rope-mixed", reg_tokens=R, drop_rate=0.1, drop_path_rate=0.1, init_values=1e-5)
    model, sd = _build(kw)
    model.train()
    B, N = 8, 64 + 1 + R
    torch.manual_seed(6)
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


def test_forward_features_last_add_matches_forward():
    """forward() adds only the cls row of the last residual; forward_features() the whole stream, in the same order."""
    kw = dict(TINY, pos_encoding="rope-mixed", init_values=1e-5)
    model, _ = _build(kw)
    model.eval()
    x = torch.randn(4, 3, 32, 32, device=DEV)
    with torch.no_grad():
        feats = model.forward_features(x)
        y = ops.layer_norm(feats[:, 0], model.norm)
        want = ops.linear(y, model.head, ops.lp_weight(model.head.weight, F32))
        assert torch.equal(model(x), want)


@pytest.mark.parametrize("amp", [None, BF], ids=["f32", "bf16"])
def test_init_values_none_changes_nothing(amp):
    kw = dict(TINY if amp is None else dict(CFG3, num_classes=10), pos_encoding="rope-mixed")
    torch.manual_seed(0)
    base = VisionTransformer(**kw).to(DEV)
    torch.manual_seed(0)
    none = VisionTransformer(**kw, init_values=None).to(DEV)
    images = torch.randn(4, 3, kw["img_size"], kw["img_size"], device=DEV)
    outs = []
    for m in (base, none):
        before = _lib.launch_count()
        with torch.autocast("cuda", dtype=BF, enabled=amp is not None):
            logits = m(images)
            logits.float().sum().backward()
        torch.cuda.synchronize()
        outs.append((logits.detach(), _lib.launch_count() - before, dict(m.named_parameters())))
    assert outs[0][1] == outs[1][1]
    assert torch.equal(outs[0][0], outs[1][0])
    assert list(outs[0][2]) == list(outs[1][2])
    # The backward's batch reductions (LayerNorm gamma / beta, bias column sums, the RoPE table gradient) add fp32
    # partials with atomics in hardware-scheduled order: two backward passes of one and the same model agree to ~1e-6,
    # not bit for bit (DESIGN section 2, "Determinism"), so the gradients are held to that reproducibility.
    for name, p in outs[0][2].items():
        a, b = p.grad.float(), outs[1][2][name].grad.float()
        assert (a - b).abs().max() <= 1e-5 * b.abs().max(), name


def test_layer_scale_runs_the_fused_loop():
    model, _ = _build(dict(TINY, pos_encoding="rope-mixed", init_values=1e-5))
    x = torch.randn(2, 3, 32, 32, device=DEV)
    assert model._fusable(ops.patch_embed(x, model.patch_embed.weight, model.patch_embed.bias, model.cls_token, None,
                                          model.patch_size))
    assert all(type(b.ls1) is LayerScale and type(b.ls2) is LayerScale for b in model.blocks)


def test_graphed_inference_with_layer_scale():
    kw = dict(HD64, pos_encoding="rope-mixed", init_values=1e-5)
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


@pytest.mark.parametrize("amp", ["bf16", "fp16"])
def test_train_cli_with_layer_scale_learns_and_reloads(tmp_path, amp):
    argv = ["--dataset", "cifar10", "--pos_encoding", "rope-mixed", "--epochs", "2", "--batch_size", "32", "--synthetic",
            "--synthetic_size", "256", "--max_steps", "8", "--log_dir", str(tmp_path / "logs"), "--ckpt_dir",
            str(tmp_path / "ck"), "--amp", amp, "--embed_dim", "128", "--num_heads", "2", "--depth", "2",
            "--init_values", "1e-5"]
    log_file, ckpt = train.main(argv)
    rows = [r.split(",") for r in open(log_file).read().strip().splitlines()[1:]]
    assert len(rows) == 2 and all(math.isfinite(float(r[1])) for r in rows)
    assert float(rows[1][1]) < float(rows[0][1]), rows  # the training loss falls
    sd = torch.load(ckpt, map_location="cpu")
    assert sd["blocks.0.ls1.gamma"].shape == (128,) and not torch.equal(sd["blocks.1.ls2.gamma"], torch.full((128,), 1e-5))
    m = VisionTransformer(img_size=32, patch_size=4, in_chans=3, num_classes=10, embed_dim=128, depth=2, num_heads=2,
                          pos_encoding="rope-mixed", init_values=1e-5)
    m.load_state_dict(sd, strict=True)
