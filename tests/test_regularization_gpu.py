"""Dropout and stochastic depth on the device: the masks, the add+LayerNorm and fc1 kernels that apply them, and the
model against the fp32 oracle with the same masks replayed.

The masks come from ``vrr_dropout_mask`` and are pinned to ``oracle/philox_np.py`` bit for bit; every kernel that
applies them is compared BIT FOR BIT with the plain kernel fed the already-multiplied input (the contract of
include/vrr.h), at shapes sized from the device so that every warp / cluster handles several rows or tiles.  Output
buffers are pre-filled with NaN; process-wide options are restored in ``finally``.
"""
import ctypes
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import train
from oracle import philox_np
from oracle import vit_torch as V
from vit_rpe_rope_b200 import VisionTransformer, _lib, ops
from vit_rpe_rope_b200.dp import BucketedDataParallel
from vit_rpe_rope_b200.runtime import GraphedTrainStep

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


# ===================================================================================== masks
SEEDS = [0x0123456789ABCDEF, -0x5A5A5A5A12345678, 0x7FFFFFFF00000001]


@pytest.mark.parametrize("E", [192, 768, 1024, 3072])
def test_dropout_mask_matches_philox_np(E):
    M = 4 * _sms() + 37  # ragged
    for seed in SEEDS:
        for site, p, pp, rows in [(0, 0.1, 0.0, 1), (5, 0.5, 0.2, 7), (35, 0.3, 0.1, 197)]:
            s = _seed(seed)
            keep, keep_path = ops.dropout_mask((p, pp, rows, site, s), M, E)
            want = philox_np.element_mask(seed, site, p, M, E)
            assert np.array_equal(keep.cpu().numpy().astype(bool), want), (seed, site, E)
            if pp > 0:
                wp = philox_np.path_mask(seed, site, pp, -(-M // rows))
                assert np.array_equal(keep_path.cpu().numpy().astype(bool), wp), (seed, site)


@pytest.mark.parametrize("p", [0.1, 0.5])
def test_kept_fraction_and_independence(p):
    M, E = 16384, 768  # 1.26e7 elements
    s = _seed(SEEDS[0])
    a, _ = ops.dropout_mask((p, 0.0, 1, 1, s), M, E)
    b, _ = ops.dropout_mask((p, 0.0, 1, 2, s), M, E)
    n = M * E
    q = 1 - philox_np.threshold(p) / 65536
    kept = a.double().mean().item()
    assert abs(kept - (1 - q)) <= 5 * math.sqrt(q * (1 - q) / n)
    # two sites, and adjacent columns of one site, agree at the rate of independent coins
    agree_rate = (1 - q) ** 2 + q ** 2
    for x, y, cnt in [(a, b, n), (a[:, 0::2], a[:, 1::2], n // 2)]:
        agree = (x == y).double().mean().item()
        assert abs(agree - agree_rate) <= 5 * math.sqrt(agree_rate * (1 - agree_rate) / cnt)


# ===================================================================================== add + LayerNorm
def _set_option(name, value):
    _lib.check(_lib.load().vrr_set_option(name.encode(), int(value)), name)


def _add_ln(x, br, gamma, beta, y_dtype, drop=None):
    lib = _lib.load()
    M, E = x.shape
    x_new, y = _nan((M, E)), _nan((M, E), y_dtype)
    mean, rstd = _nan((M,)), _nan((M,))
    if drop == "null":  # the drop entry point with a NULL desc
        rc = lib.vrr_add_layernorm_drop_fwd(_p(x), _p(br), _p(x_new), _p(gamma), _p(beta), _p(y), _p(mean), _p(rstd),
                                            M, E, 1e-5, DT[br.dtype], DT[y_dtype], None, _st())
    elif drop is None:
        rc = lib.vrr_add_layernorm_fwd(_p(x), _p(br), _p(x_new), _p(gamma), _p(beta), _p(y), _p(mean), _p(rstd), M, E,
                                       1e-5, DT[br.dtype], DT[y_dtype], _st())
    else:
        d = ops._drop_desc(drop) if not isinstance(drop, _lib.DropDesc) else drop
        rc = lib.vrr_add_layernorm_drop_fwd(_p(x), _p(br), _p(x_new), _p(gamma), _p(beta), _p(y), _p(mean), _p(rstd),
                                            M, E, 1e-5, DT[br.dtype], DT[y_dtype], ctypes.byref(d), _st())
    _lib.check(rc, "add_layernorm fwd")
    return x_new, y, mean, rstd


def _add_ln_bwd(dy, dxn, x_new, gamma, mean, rstd, br_dtype, drop=None):
    lib = _lib.load()
    M, E = x_new.shape
    dx, dbr, dgb = _nan((M, E)), _nan((M, E), br_dtype), _nan((2, E))
    if drop is None:
        rc = lib.vrr_add_layernorm_bwd(_p(dy), _p(dxn), _p(x_new), _p(gamma), _p(mean), _p(rstd), _p(dx), _p(dbr),
                                       _p(dgb[0]), _p(dgb[1]), M, E, DT[br_dtype], DT[dy.dtype], _st())
    else:
        d = ops._drop_desc(drop) if not isinstance(drop, _lib.DropDesc) else drop
        rc = lib.vrr_add_layernorm_drop_bwd(_p(dy), _p(dxn), _p(x_new), _p(gamma), _p(mean), _p(rstd), _p(dx),
                                            _p(dbr), _p(dgb[0]), _p(dgb[1]), M, E, DT[br_dtype], DT[dy.dtype],
                                            ctypes.byref(d), _st())
    _lib.check(rc, "add_layernorm bwd")
    return dx, dbr, dgb


# (E, ln_reg, ln_bwd_minb): register-resident NV 2/4/6/8 with every backward launch shape, generic VEC 4 and VEC 1
VARIANTS = [(256, 1, 3), (512, 1, 2), (768, 1, 3), (768, 1, 1), (768, 1, 2), (1024, 1, 3), (1024, 1, 2),
            (768, 0, 3), (640, 1, 3), (192, 1, 3)]


@pytest.mark.parametrize("E,ln_reg,minb", VARIANTS)
@pytest.mark.parametrize("bdt", [F32, BF, HF], ids=["f32", "bf16", "f16"])
def test_add_layernorm_drop_is_the_plain_kernel_fed_f_times_branch(E, ln_reg, minb, bdt):
    N = 197
    M = N * max(8, 3 * 4 * 8 * _sms() // N)  # whole images; ~3 rows per warp of the largest grid (4 CTAs x 8 warps / SM)
    g = torch.Generator(device=DEV).manual_seed(E)
    x = torch.randn(M, E, device=DEV, generator=g)
    br = torch.randn(M, E, device=DEV, generator=g).to(bdt)
    gamma, beta = 1 + 0.1 * torch.randn(E, device=DEV, generator=g), 0.1 * torch.randn(E, device=DEV, generator=g)
    ydt = F32 if bdt == F32 else bdt
    dy = torch.randn(M, E, device=DEV, generator=g).to(ydt)
    dxn = torch.randn(M, E, device=DEV, generator=g)
    try:
        _set_option("ln_reg", ln_reg)
        _set_option("ln_bwd_minb", minb)
        for p, pp, site in [(0.1, 0.0, 3), (0.0, 0.3, 4), (0.2, 0.1, 5)]:
            drop = (p, pp, N, site, _seed(SEEDS[1]))
            f = ops.branch_factor(drop, M // N, N, E).view(M, E)
            ref = _add_ln(x, br.float() * f, gamma, beta, ydt)
            got = _add_ln(x, br, gamma, beta, ydt, drop)
            for r, o in zip(ref, got):
                assert _bits_equal(o, r), (p, pp)
            rdx, _, rdgb = _add_ln_bwd(dy, dxn, ref[0], gamma, ref[2], ref[3], F32)
            gdx, gdbr, gdgb = _add_ln_bwd(dy, dxn, got[0], gamma, got[2], got[3], bdt, drop)
            assert _bits_equal(gdx, rdx)
            assert _bits_equal(gdbr, (rdx * f).to(bdt))
            # dgamma / dbeta: fp32 sums over the rows whose order across CTAs is not fixed - bounded by the sums of |terms|
            xh = (ref[0].double() - ref[2].double()[:, None]) * ref[3].double()[:, None]
            scale = torch.stack([(dy.double() * xh).abs().sum(0), dy.double().abs().sum(0)])
            assert ((gdgb.double() - rdgb.double()).abs() <= 2e-5 * scale).all()
        # p == 0 and a NULL desc are the plain entry point
        zero = (0.0, 0.0, N, 1, _seed(1))
        for drop in (zero, "null"):
            a, b = _add_ln(x, br, gamma, beta, ydt, drop), _add_ln(x, br, gamma, beta, ydt)
            assert all(_bits_equal(u, v) for u, v in zip(a, b))
        plain = _add_ln_bwd(dy, dxn, a[0], gamma, a[2], a[3], bdt)
        zd = _add_ln_bwd(dy, dxn, a[0], gamma, a[2], a[3], bdt, zero)
        assert _bits_equal(zd[0], plain[0]) and _bits_equal(zd[1], plain[1])
    finally:
        _set_option("ln_reg", 1)
        _set_option("ln_bwd_minb", 3)


def test_add_layernorm_drop_rejects_bad_descs():
    lib = _lib.load()
    M, E = 64, 768
    x, br, gamma, beta = _nan((M, E)), _nan((M, E)), _nan((E,)), _nan((E,))
    for drop in [(1.0, 0.0, 1, 0, _seed(1)), (0.1, -0.1, 1, 0, _seed(1)), (0.0, 0.1, 0, 0, _seed(1))]:
        d = ops._drop_desc(drop)
        rc = lib.vrr_add_layernorm_drop_fwd(_p(x), _p(br), _p(x), _p(gamma), _p(beta), _p(x), _p(x), _p(x), M, E,
                                            1e-5, 0, 0, ctypes.byref(d), _st())
        assert rc == -1, drop
    d = ops._drop_desc((0.1, 0.0, 1, 0, _seed(1)))
    x2 = _nan((M, 100))
    rc = lib.vrr_add_layernorm_drop_fwd(_p(x2), _p(x2), _p(x2), _p(gamma), _p(beta), _p(x2), _p(x2), _p(x2), M, 100,
                                        1e-5, 0, 0, ctypes.byref(d), _st())
    assert rc == -2  # element masks need E % 8 == 0


# ===================================================================================== fc1
@pytest.mark.parametrize("impl", [_lib.IMPL_TCGEN05, _lib.IMPL_SIMT], ids=["tcgen05", "simt"])
@pytest.mark.parametrize("dt", [BF, HF, F32], ids=["bf16", "f16", "f32"])
@pytest.mark.parametrize("epi", [_lib.EPI_BIAS_GELU_GRAD, _lib.EPI_BIAS_GELU_ACT], ids=["grad", "act"])
def test_fc1_dropout_epilogue(impl, dt, epi):
    if dt == F32 and impl == _lib.IMPL_TCGEN05:
        pytest.skip("fp32 always runs the SIMT kernels")
    lib = _lib.load()
    sms = _sms()
    M, N, K = (2 * 128) * (sms // 12 + 1) + 40, 3072, 768  # more 256 x 256 tiles than clusters, ragged M
    if dt == F32 or impl == _lib.IMPL_SIMT:
        M = 2 * 128 * 3 + 40
    g = torch.Generator(device=DEV).manual_seed(7)
    a = (torch.randn(M, K, device=DEV, generator=g) * 0.5).to(dt)
    w = (torch.randn(N, K, device=DEV, generator=g) * 0.05).to(dt)
    bias = torch.randn(N, device=DEV, generator=g) * 0.3
    grad = epi == _lib.EPI_BIAS_GELU_GRAD

    def run(drop):
        c, c2 = _nan((M, N), dt), (_nan((M, N), dt) if grad else None)
        if drop is None:
            rc = lib.vrr_gemm_ex(_p(a), _p(w), _p(c), _p(c2), _p(bias), M, N, K, 0, 1, DT[dt], DT[dt], epi, 0, _st())
        else:
            d = ops._drop_desc(drop)
            rc = lib.vrr_gemm_ex_drop(_p(a), _p(w), _p(c), _p(c2), _p(bias), M, N, K, 0, 1, DT[dt], DT[dt], epi, 0,
                                      ctypes.byref(d), _st())
        _lib.check(rc, "gemm")
        return c, c2

    prev = _lib.set_impl(impl)
    try:
        fam0 = _lib.family_count(impl)
        ref = run(None)
        drop = (0.1, 0.0, 1, 7, _seed(SEEDS[2]))
        got = run(drop)
        torch.cuda.synchronize()
        assert _lib.family_count(impl) - fam0 == 2, "the forced kernel family must have run"
        keep, _ = ops.dropout_mask(drop, M, N)
        f = keep.float() * ops.drop_scale(0.1, 0.0)
        assert _bits_equal(got[0], (ref[0].float() * f).to(dt))
        if grad:
            assert _bits_equal(got[1], (ref[1].float() * f).to(dt))
        zero = run((0.0, 0.0, 1, 7, _seed(3)))
        assert _bits_equal(zero[0], ref[0])
    finally:
        _lib.set_impl(prev)


# ===================================================================================== model
def _sites_of(model, B, N):
    """Per block (f_attn [B,N,E], f_fc1 [B,N,4E], f_mlp [B,N,E]) (CPU, fp32, or None) of the last training forward."""
    seed = model._drop_seed
    E = model.embed_dim
    out = []
    for i, blk in enumerate(model.blocks):
        pp = getattr(blk.drop_path, "drop_prob", 0.0)
        pa, p1, p2 = blk.attn.proj_drop.p, blk.mlp.drop1.p, blk.mlp.drop2.p
        H = blk.mlp.fc1.out_features
        fa = ops.branch_factor((pa, pp, N, 3 * i, seed), B, N, E).cpu() if (pa or pp) else None
        f1 = ops.branch_factor((p1, 0.0, N, 3 * i + 1, seed), B, N, H).cpu() if p1 else None
        f2 = ops.branch_factor((p2, pp, N, 3 * i + 2, seed), B, N, E).cpu() if (p2 or pp) else None
        out.append((fa, f1, f2))
    return out


def _oracle_forward(cfg, p, images, sites):
    """oracle/vit_torch.forward with the block branches multiplied by the replayed factors."""
    b, _, hh, ww = images.shape
    e = cfg.embed_dim
    x = F.conv2d(images, p["patch_embed.weight"], p["patch_embed.bias"], stride=cfg.patch_size)
    gh, gw = hh // cfg.patch_size, ww // cfg.patch_size
    x = torch.cat((p["cls_token"].expand(b, -1, -1), x.flatten(2).transpose(1, 2)), dim=1)
    if cfg.pos_encoding == "absolute":
        x[:, 1:] = x[:, 1:] + p["pos_embed.pos_embed"][:, : x.size(1) - 1]
    rope = None
    if cfg.pos_encoding == "rope-axial":
        rope = V.axial_cos_sin(p["pos_embed.inv_freq"], gh * gw)
    elif cfg.pos_encoding == "rope-mixed":
        rope = V.mixed_cos_sin(p["pos_embed.freqs"], gh * gw)
    mul = lambda t, f: t if f is None else t * f
    for i in range(cfg.depth):
        pre = f"blocks.{i}."
        fa, f1, f2 = sites[i]
        y = F.layer_norm(x, (e,), p[pre + "norm1.weight"], p[pre + "norm1.bias"], 1e-5)
        x = x + mul(V.attention(cfg, p, pre + "attn.", y, "pos_embed.", rope), fa)
        y = F.layer_norm(x, (e,), p[pre + "norm2.weight"], p[pre + "norm2.bias"], 1e-5)
        h = mul(F.gelu(F.linear(y, p[pre + "mlp.fc1.weight"], p[pre + "mlp.fc1.bias"])), f1)
        x = x + mul(F.linear(h, p[pre + "mlp.fc2.weight"], p[pre + "mlp.fc2.bias"]), f2)
    x = F.layer_norm(x, (e,), p["norm.weight"], p["norm.bias"], 1e-5)
    return F.linear(x[:, 0], p["head.weight"], p["head.bias"])


TINY = dict(img_size=32, patch_size=4, in_chans=3, num_classes=10, embed_dim=192, depth=3, num_heads=6)
CFG3 = dict(img_size=64, patch_size=8, in_chans=3, num_classes=10, embed_dim=256, depth=2, num_heads=4)


@pytest.mark.parametrize("mode", ["rope-mixed", "relative", "polynomial"])
@pytest.mark.parametrize("amp", [None, BF], ids=["f32", "bf16"])
def test_model_with_dropout_matches_the_oracle(mode, amp):
    kw = dict(TINY if amp is None else CFG3, pos_encoding=mode)
    torch.manual_seed(0)
    model = VisionTransformer(**kw, drop_rate=0.1, drop_path_rate=0.1)
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    model = model.to(DEV).train()
    B = 8
    images, labels = torch.randn(B, 3, kw["img_size"], kw["img_size"]), torch.randint(0, 10, (B,))
    with torch.autocast("cuda", dtype=BF, enabled=amp is not None):
        logits = model(images.to(DEV))
        loss = F.cross_entropy(logits.float(), labels.to(DEV))
    loss.backward()
    N = (kw["img_size"] // kw["patch_size"]) ** 2 + 1
    sites = _sites_of(model, B, N)
    assert any(s is not None and (s == 0).any() for blk in sites for s in blk), "no element was dropped"
    cfg = V.VitConfig(**kw)
    p = V.params_from_state_dict(sd)
    ref = _oracle_forward(cfg, p, images, sites)
    F.cross_entropy(ref, labels).backward()
    got = logits.detach().float().cpu()
    if amp is None:
        err = (got - ref.detach()).abs().max().item()
        assert err <= 1e-5 * max(1.0, ref.abs().max().item()), err
        for name, prm in model.named_parameters():
            want = p[name].grad
            e = (prm.grad.detach().cpu() - want).abs().max().item() / max(1.0, want.abs().max().item())
            assert e <= 1e-5, (name, e)
    else:
        err = ((got - ref.detach()).abs().max() / ref.detach().abs().max()).item()
        assert err <= 2e-2, err
        for name, prm in model.named_parameters():
            want = p[name].grad
            e = ((prm.grad.detach().cpu() - want).abs().max() / want.abs().max().clamp_min(1e-30)).item()
            assert e <= 2e-2, (name, e)
    # forward() takes the cls rows of the last residual add alone: same bits as forward_features + norm + head
    torch.manual_seed(5)
    with torch.no_grad(), torch.autocast("cuda", dtype=BF, enabled=amp is not None):
        l1 = model(images.to(DEV))
        torch.manual_seed(5)
        feats = model.forward_features(images.to(DEV))
        l2 = ops.linear(ops.layer_norm(feats[:, 0], model.norm), model.head)
    assert _bits_equal(l1, l2)


def _run(model, images, labels, amp):
    model.zero_grad(set_to_none=True)
    before = _lib.launch_count()
    with torch.autocast("cuda", dtype=BF, enabled=amp):
        logits = model(images)
        loss = F.cross_entropy(logits.float(), labels)
    loss.backward()
    torch.cuda.synchronize()
    return logits.detach(), [q.grad.clone() for q in model.parameters()], _lib.launch_count() - before


@pytest.mark.parametrize("amp", [False, True], ids=["f32", "bf16"])
def test_no_change_when_off(amp):
    """Rates left at 0 in training, and any rates in eval mode, run exactly the kernels of a model built without them:
    the same launches and the same logits bit for bit; gradients agree to the last bits the fp32 atomics of the
    reductions leave open."""
    kw = dict(CFG3 if amp else TINY, pos_encoding="rope-mixed")
    torch.manual_seed(0)
    base = VisionTransformer(**kw).to(DEV)
    zero = VisionTransformer(**kw, drop_rate=0.0, drop_path_rate=0.0).to(DEV)
    on = VisionTransformer(**kw, drop_rate=0.1, drop_path_rate=0.1).to(DEV)
    zero.load_state_dict(base.state_dict())
    on.load_state_dict(base.state_dict())
    images = torch.randn(8, 3, kw["img_size"], kw["img_size"], device=DEV)
    labels = torch.randint(0, 10, (8,), device=DEV)
    for ref_model, model in ((base.train(), zero.train()), (base.eval(), on.eval())):
        ref = _run(ref_model, images, labels, amp)
        rng = torch.cuda.get_rng_state()
        got = _run(model, images, labels, amp)
        assert torch.equal(rng, torch.cuda.get_rng_state()), "no seed is drawn"
        assert got[2] == ref[2], (got[2], ref[2])
        assert _bits_equal(got[0].float(), ref[0].float())
        for a, b in zip(got[1], ref[1]):
            assert (a - b).abs().max().item() <= 1e-5 * b.abs().max().item()


def test_eager_training_forwards_are_reproducible():
    kw = dict(TINY, pos_encoding="relative")
    torch.manual_seed(0)
    model = VisionTransformer(**kw, drop_rate=0.1, drop_path_rate=0.1).to(DEV).train()
    images = torch.randn(8, 3, 32, 32, device=DEV)
    outs = []
    for _ in range(2):
        torch.manual_seed(11)
        with torch.no_grad():
            outs.append(model(images))
    assert _bits_equal(outs[0], outs[1])
    with torch.no_grad():
        third = model(images)
    assert not torch.equal(third, outs[0]), "a new forward draws a new key"


def test_cuda_graph_replays_draw_fresh_masks():
    kw = dict(TINY, pos_encoding="rope-axial")
    torch.manual_seed(0)
    model = VisionTransformer(**kw, drop_rate=0.1, drop_path_rate=0.1).to(DEV)
    dp = BucketedDataParallel(model, bucket_mb=32.0)
    opt = torch.optim.AdamW(model.parameters(), lr=1e-4, weight_decay=0.01, fused=True, capturable=True)
    B = 16
    images, labels = torch.randn(B, 3, 32, 32, device=DEV), torch.randint(0, 10, (B,), device=DEV)
    runner = GraphedTrainStep(dp, opt, tuple(images.shape), 10, torch.device(DEV), bf16=False, use_graph=True)
    runner.prepare(images, labels)
    assert runner.graph is not None
    N = 65
    cfg = V.VitConfig(**kw)
    seeds = []
    for _ in range(2):
        sd = {k: v.detach().clone().cpu() for k, v in model.state_dict().items()}
        loss = runner.run().item()
        seeds.append(int(model._drop_seed.item()))
        sites = _sites_of(model, B, N)
        ref = F.cross_entropy(_oracle_forward(cfg, V.params_from_state_dict(sd, requires_grad=False), images.cpu(), sites),
                              labels.cpu()).item()
        assert abs(loss - ref) <= 1e-5 * max(1.0, abs(ref)), (loss, ref)
    assert seeds[0] != seeds[1]
    runner.close()


@pytest.mark.parametrize("amp", ["bf16", "fp16"])
def test_train_cli_with_regularisers(tmp_path, amp):
    argv = ["--dataset", "cifar10", "--pos_encoding", "rope-mixed", "--epochs", "1", "--batch_size", "32", "--synthetic",
            "--synthetic_size", "128", "--max_steps", "3", "--log_dir", str(tmp_path / "logs"), "--ckpt_dir",
            str(tmp_path / "ck"), "--amp", amp, "--embed_dim", "128", "--num_heads", "2", "--depth", "2",
            "--drop_rate", "0.1", "--drop_path_rate", "0.1"]
    log_file, ckpt = train.main(argv)
    rows = open(log_file).read().strip().splitlines()
    assert len(rows) == 2 and all(math.isfinite(float(v)) for v in rows[1].split(",")[1:3])
