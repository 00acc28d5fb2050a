"""GPU parity tests: the CUDA path (through the C ABI) against the oracle and the golden fixtures.

Tolerances (BASELINE.json north_star): index / coordinate tables bit-exact (CPU tests); logits and
gradients max-abs <= 1e-5 in fp32 and <= 2e-2 relative in bf16.

* fp32: ``err_scaled`` = max|a-b| / max(1, max|b|) must be <= 1e-5 (the north-star absolute bar, scaled
  up only for tensors whose own magnitude exceeds 1), AND - because most gradients are far below 1 in
  magnitude, where an absolute bar alone is weak - ``err_rel`` = max|a-b| / max|b| must be <=
  FP32_REL_TOL (summation-order noise of fp32 reductions over 1e3..1e5 terms stays well inside it).
* bf16: ``err_rel`` <= 2e-2, flat, against the fp32 oracle, for logits and every gradient tensor (the
  reference's own autocast run is measured beside it and reported, but buys no allowance).
* every bf16 head-dim-64 case asserts that the tcgen05 kernel family ran (``vrr_family_count``).

Observed worst errors are appended to ``gpurun_out/parity_report.txt`` (when that directory exists).
"""
import ctypes
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import attention_np as A
from oracle import tables_np as T
from oracle import vit_torch as V
from vit_rpe_rope_b200 import _lib, models, ops
from vit_rpe_rope_b200.models.vit import Attention, VisionTransformer

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
MODES = ("none", "absolute", "relative", "polynomial", "rope-axial", "rope-mixed")
MODEL_TAGS = ["none", "absolute", "relative", "polynomial", "polynomial_perhead", "rope_axial", "rope_mixed"]
FP32_TOL = 1e-5
FP32_REL_TOL = 5e-5
BF16_TOL = 2e-2
DEV = "cuda:0"
_REPORT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out", "parity_report.txt")


def report(line):
    if os.path.isdir(os.path.dirname(_REPORT)):
        with open(_REPORT, "a") as f:
            f.write(line + "\n")


class tcgen05_must_run:
    """Context: the wrapped calls must dispatch to the tcgen05 family and never to the SIMT family."""

    def __enter__(self):
        self.tc0, self.simt0 = _lib.family_count(_lib.IMPL_TCGEN05), _lib.family_count(_lib.IMPL_SIMT)
        return self

    def __exit__(self, et, ev, tb):
        if et is None:
            assert _lib.family_count(_lib.IMPL_TCGEN05) > self.tc0, "no tcgen05 kernel was dispatched"
            assert _lib.family_count(_lib.IMPL_SIMT) == self.simt0, "a SIMT kernel ran where tcgen05 was expected"
        return False


def check_fp32(got, want, what=""):
    ea, er = err_scaled(got, want), err_rel(got, want)
    report(f"fp32 {what}: scaled {ea:.2e} rel {er:.2e}")
    assert ea <= FP32_TOL, (what, ea)
    assert er <= FP32_REL_TOL, (what, er)


def check_bf16(got, want32, ref16=None, what=""):
    e_mine = err_rel(got, want32)
    e_ref = err_rel(ref16, want32) if ref16 is not None else 0.0
    bound = BF16_TOL
    report(f"bf16 {what}: mine {e_mine:.2e} ref-autocast {e_ref:.2e} bound {bound:.2e}")
    assert e_mine <= bound, (what, e_mine, e_ref)


@pytest.fixture(autouse=True, scope="module")
def _no_tf32():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield


def err_scaled(got, want):
    got = torch.as_tensor(got).detach().double().cpu()
    want = torch.as_tensor(want).detach().double().cpu()
    assert got.shape == want.shape, (got.shape, want.shape)
    return (got - want).abs().max().item() / max(1.0, want.abs().max().item())


def err_rel(got, want):
    got = torch.as_tensor(got).detach().double().cpu()
    want = torch.as_tensor(want).detach().double().cpu()
    assert got.shape == want.shape, (got.shape, want.shape)
    return (got - want).abs().max().item() / max(want.abs().max().item(), 1e-30)


# ------------------------------------------------------------------------------------- golden: model

@pytest.mark.parametrize("tag", MODEL_TAGS)
def test_model_vs_reference_golden_fp32(tag):
    """Small ViT: logits, loss and every parameter gradient against outputs of the reference itself."""
    z = np.load(os.path.join(GOLDEN, f"model_{tag}.npz"))
    kw = eval(str(z["kwargs"]))  # noqa: S307
    model = VisionTransformer(**kw)
    model.load_state_dict({k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd.")}, strict=True)
    model = model.to(DEV)
    before = _lib.launch_count()
    logits = model(torch.from_numpy(z["images"]).to(DEV))
    loss = F.cross_entropy(logits, torch.from_numpy(z["labels"]).to(DEV))
    loss.backward()
    assert _lib.launch_count() > before, "no libvrr kernel was launched"
    check_fp32(logits, z["logits"], f"golden {tag} logits")
    assert abs(loss.item() - float(z["loss"])) <= FP32_TOL
    checked = 0
    for name, p in model.named_parameters():
        assert p.grad is not None, name
        check_fp32(p.grad, z["grad." + name], f"golden {tag} {name}")
        checked += 1
    assert checked == sum(1 for k in z.files if k.startswith("grad.") and ".attn.pos_encoding." not in k)


# ------------------------------------------------------------------------------------- golden: attention

@pytest.mark.parametrize("tag", [t for t in MODEL_TAGS if t != "absolute"])
def test_attention_module_vs_reference_golden_fp32(tag):
    z = np.load(os.path.join(GOLDEN, f"attn_{tag}.npz"))
    heads, n = 3, 65
    e = z["x"].shape[-1]
    attn = Attention(e, num_heads=heads)
    mode = {"none": "none", "relative": "relative", "polynomial": "polynomial", "polynomial_perhead": "polynomial",
            "rope_axial": "rope-axial", "rope_mixed": "rope-mixed"}[tag]
    pe = {"none": models.NoPositionalEncoding(),
          "relative": models.RelativePositionalEncoding(n - 1, heads),
          "polynomial": models.PolynomialRPE(n - 1, 3, heads, tag == "polynomial"),
          "rope-axial": models.RoPEAxial(e // heads, 100.0),
          "rope-mixed": models.RoPEMixed(e // heads, heads, 100.0)}[mode]
    attn.set_pos_encoding(pe)
    attn.load_state_dict({k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd.")}, strict=True)
    attn = attn.to(DEV)
    x = torch.from_numpy(z["x"]).to(DEV).requires_grad_(True)
    freqs = pe.get_freqs_cis(n - 1, DEV) if mode.startswith("rope") else None
    if freqs is not None:
        assert err_scaled(freqs[0], z["cos"]) <= 2e-6 and err_scaled(freqs[1], z["sin"]) <= 2e-6
    y = attn(x, freqs_cis=freqs)
    (y * torch.from_numpy(z["dy"]).to(DEV)).sum().backward()
    check_fp32(y, z["y"], f"golden attn {tag} y")
    check_fp32(x.grad, z["dx"], f"golden attn {tag} dx")
    for name, p in attn.named_parameters():
        check_fp32(p.grad, z["grad." + name], f"golden attn {tag} {name}")


# ------------------------------------------------------------------------------------- oracle: ViT-Tiny

def _tiny_kwargs(mode, **over):
    kw = dict(img_size=32, patch_size=4, in_chans=3, num_classes=10, embed_dim=192, depth=6, num_heads=6,
              pos_encoding=mode)
    kw.update(over)
    return kw


def _build_pair(kw, seed=0):
    torch.manual_seed(seed)
    model = VisionTransformer(**kw)
    with torch.no_grad():  # make zero-initialised paths live
        model.cls_token.normal_(std=0.02)
        for n, p in model.named_parameters():
            if n.endswith(".bias"):
                p.normal_(std=0.02)
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    return model.to(DEV), sd


def _oracle_run(kw, sd, images, labels, device="cpu", autocast=False):
    cfg = V.VitConfig(**kw)
    p = V.params_from_state_dict(sd, device=device)
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
        logits = V.forward(cfg, p, images.to(device))
        loss = F.cross_entropy(logits.float(), labels.to(device))
    loss.backward()
    return logits.detach(), {k: v.grad for k, v in p.items() if v.is_floating_point() and v.grad is not None}


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("chans", [3, 1])
def test_vit_tiny_fp32_vs_oracle(mode, chans):
    """BASELINE configs[0]/[1]: ViT-Tiny (65 tokens, Dh 32), CIFAR- and MNIST-shaped, every mode."""
    kw = _tiny_kwargs(mode, in_chans=chans)
    model, sd = _build_pair(kw)
    torch.manual_seed(1)
    images, labels = torch.randn(8, chans, 32, 32), torch.randint(0, 10, (8,))
    logits = model(images.to(DEV))
    F.cross_entropy(logits, labels.to(DEV)).backward()
    want, grads = _oracle_run(kw, sd, images, labels)
    check_fp32(logits, want, f"{kw['pos_encoding']} logits")
    for name, p in model.named_parameters():
        check_fp32(p.grad, grads[name], f"{kw['pos_encoding']} {name}")


def test_vit_tiny_polynomial_per_head_fp32():
    kw = _tiny_kwargs("polynomial", poly_shared_heads=False, depth=2)
    model, sd = _build_pair(kw)
    with torch.no_grad():
        model.pos_embed.coefficients.mul_(0.3)
    sd = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}
    images, labels = torch.randn(4, 3, 32, 32), torch.randint(0, 10, (4,))
    logits = model(images.to(DEV))
    F.cross_entropy(logits, labels.to(DEV)).backward()
    want, grads = _oracle_run(kw, sd, images, labels)
    check_fp32(logits, want, f"{kw['pos_encoding']} logits")
    for name, p in model.named_parameters():
        check_fp32(p.grad, grads[name], f"{kw['pos_encoding']} {name}")


@pytest.mark.parametrize("mode", ["none", "absolute", "rope-axial", "rope-mixed"])
def test_resolution_extrapolation_fp32(mode):
    """vit.py:249,265: the token count follows the INPUT; rope / none / absolute accept larger images."""
    kw = _tiny_kwargs(mode, depth=2)
    model, sd = _build_pair(kw)
    images, labels = torch.randn(2, 3, 64, 64), torch.randint(0, 10, (2,))
    logits = model(images.to(DEV))
    F.cross_entropy(logits, labels.to(DEV)).backward()
    want, grads = _oracle_run(kw, sd, images, labels)
    check_fp32(logits, want, f"{kw['pos_encoding']} logits")
    for name, p in model.named_parameters():
        check_fp32(p.grad, grads[name], f"{kw['pos_encoding']} {name}")


@pytest.mark.parametrize("mode", ["relative", "polynomial"])
def test_fixed_size_bias_rejects_other_resolutions(mode):
    """Reference behaviour (SURVEY aux table): relative / polynomial fail when N != construction N."""
    model, _ = _build_pair(_tiny_kwargs(mode, depth=1))
    with pytest.raises(RuntimeError):
        model(torch.randn(1, 3, 64, 64, device=DEV))


# ------------------------------------------------------------------------------------- bf16 (autocast)

def _bf16_model_case(kw, batch, size, train=True, seed=2):
    model, sd = _build_pair(kw)
    torch.manual_seed(seed)
    images = torch.randn(batch, kw["in_chans"], size, size)
    labels = torch.randint(0, kw["num_classes"], (batch,))
    if not train:
        model.eval()
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16), tcgen05_must_run():
            logits = model(images.to(DEV))
        cfg = V.VitConfig(**kw)
        with torch.no_grad():
            p32 = V.params_from_state_dict(sd, device=DEV, requires_grad=False)
            want32 = V.forward(cfg, p32, images.to(DEV))
            with torch.autocast("cuda", dtype=torch.bfloat16):
                want16 = V.forward(cfg, p32, images.to(DEV))
        check_bf16(logits.float(), want32, want16.float(), f"{kw['pos_encoding']} N={(size // kw['patch_size']) ** 2 + 1} logits (eval)")
        return
    with tcgen05_must_run():
        with torch.autocast("cuda", dtype=torch.bfloat16):
            logits = model(images.to(DEV))
            loss = F.cross_entropy(logits.float(), labels.to(DEV))
        loss.backward()
    want32, grads32 = _oracle_run(kw, sd, images, labels, device=DEV)
    want16, grads16 = _oracle_run(kw, sd, images, labels, device=DEV, autocast=True)
    tag = f"{kw['pos_encoding']} E={kw['embed_dim']} N={(size // kw['patch_size']) ** 2 + 1}"
    check_bf16(logits.float(), want32, want16.float(), f"{tag} logits")
    for name, p in model.named_parameters():
        assert p.grad.dtype == torch.float32
        check_bf16(p.grad, grads32[name], grads16[name], f"{tag} {name}")


@pytest.mark.parametrize("mode", MODES)
def test_vit_bf16_autocast_vs_reference_semantics(mode):
    """bf16 = the reference ops under torch.autocast('cuda', bfloat16) with fp32 master weights
    (SURVEY row O4).  Head dim 64 (ViT-B geometry, shortened): the tcgen05 kernels must be the ones
    that run.  Logits and every gradient within 2e-2 relative of the fp32 oracle (see module docstring)."""
    kw = dict(img_size=64, patch_size=8, in_chans=3, num_classes=10, embed_dim=256, depth=2, num_heads=4,
              pos_encoding=mode)
    _bf16_model_case(kw, batch=16, size=64)


@pytest.mark.parametrize("mode", ["rope-mixed", "relative", "polynomial"])
def test_cfg3_geometry_bf16(mode):
    """BASELINE configs[2] geometry (ViT-B/16-224: 12 heads x 64, 197 tokens, E 768), depth 2, batch 4."""
    kw = dict(img_size=224, patch_size=16, in_chans=3, num_classes=1000, embed_dim=768, depth=2, num_heads=12,
              pos_encoding=mode)
    _bf16_model_case(kw, batch=4, size=224)


def test_cfg4_geometry_bf16():
    """BASELINE configs[3] geometry (ViT-L/16-384: 16 heads x 64, 577 tokens, E 1024, rope-axial), depth 1."""
    kw = dict(img_size=384, patch_size=16, in_chans=3, num_classes=1000, embed_dim=1024, depth=1, num_heads=16,
              pos_encoding="rope-axial")
    _bf16_model_case(kw, batch=2, size=384)


def test_cfg5_resolution_extrapolation_inference_bf16():
    """BASELINE configs[4]: ViT-B/16 rope-mixed built at 224, fed 512x512 (1025 tokens), eval + no_grad
    (reference resolution path: models/vit.py:249,265)."""
    kw = dict(img_size=224, patch_size=16, in_chans=3, num_classes=1000, embed_dim=768, depth=2, num_heads=12,
              pos_encoding="rope-mixed")
    _bf16_model_case(kw, batch=2, size=512, train=False)


def test_graphed_inference_replays_the_eager_forward():
    """runtime.GraphedInference: the captured forward returns what the eager forward returns, for fresh inputs
    (the RoPE tables and their packed copy are rebuilt inside the graph), and counts its launches."""
    from vit_rpe_rope_b200.models.vit import VisionTransformer
    from vit_rpe_rope_b200.runtime import GraphedInference
    torch.manual_seed(0)
    model = VisionTransformer(img_size=64, patch_size=8, in_chans=3, num_classes=10, embed_dim=256, depth=2, num_heads=4,
                              pos_encoding="rope-mixed").to(DEV).eval()
    runner = GraphedInference(model, (4, 3, 96, 96), torch.device(DEV), bf16=True)  # 145 tokens: resolution extrapolation
    assert runner.graph is not None and runner.launches_per_step > 0
    g = torch.Generator().manual_seed(7)
    for _ in range(3):
        x = torch.randn(4, 3, 96, 96, generator=g).to(DEV)
        got = runner.run(x).float().clone()
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            want = model(x).float()
        assert torch.equal(got, want)
        with torch.inference_mode(), torch.autocast("cuda", dtype=torch.bfloat16):
            assert torch.equal(model(x).float(), want)  # inference tensors (no version counters) take the same path
    runner.close()


# ------------------------------------------------------------------------------------- kernels vs numpy

def _planes(b, h, n, d, dtype, seed=0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(3, b, h, n, d, generator=g) * 0.8).to(dtype)


def _bias_case(kind, h, n, seed=0):
    g = torch.Generator().manual_seed(seed + 5)
    if kind == "none":
        return _lib.BIAS_NONE, None, 0, None
    if kind == "table":
        tab = torch.randn(h, 2 * n - 1, generator=g) * 0.5
        return _lib.BIAS_TABLE, tab, 0, T.relative_bias(tab.numpy().astype(np.float64), n)
    shared = kind == "poly"
    grid = int(round((n - 1) ** 0.5))
    # coefficient k scaled by (2g)^-k so that |bias| stays O(1) at every grid size: with |bias| in the
    # hundreds the softmax is one-hot and dS = P*(dP - delta) is pure cancellation in ANY fp32
    # implementation (the reference included), which would make the d_coef comparison meaningless.
    span = torch.tensor([float(max(2 * grid - 2, 1)) ** -k for k in range(4)])
    coef = (torch.randn(4, generator=g) if shared else torch.randn(h, 4, generator=g)) * 0.7 * span
    return _lib.BIAS_POLY, coef, grid, T.poly_bias(coef.numpy(), n - 1, h).astype(np.float64)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("n,d", [(1, 16), (2, 32), (17, 16), (65, 32), (65, 64), (197, 64), (200, 64), (257, 64),
                                 (577, 64), (1025, 64)])
@pytest.mark.parametrize("kind", ["none", "table", "poly", "poly_perhead"])
def test_attention_kernels_vs_numpy(dtype, n, d, kind):
    """Fused attention fwd + bwd vs float64 numpy, ragged and edge sizes: N = 1, N not a multiple of any
    tile, N > one tile, and the cfg4 / cfg5 sequence lengths (577 = 10 key tiles, 1025 = 17: every
    K/V ring stage and mbarrier parity wraps several times).  bf16 with head dim 64 must take the
    tcgen05 family."""
    if kind.startswith("poly") and int(round((n - 1) ** 0.5)) ** 2 != n - 1:
        pytest.skip("polynomial bias needs a square patch grid")
    if kind.startswith("poly") and n == 1:
        pytest.skip("no patches")
    b, h = (2, 3) if n <= 257 else (1, 2)
    mode, param, grid, bias_np = _bias_case(kind, h, n)
    planes = _planes(b, h, n, d, dtype).to(DEV).requires_grad_(True)
    prm = None if param is None else param.to(DEV).requires_grad_(True)
    scale = d ** -0.5
    g = torch.Generator().manual_seed(9)
    d_out = torch.randn(b, n, h * d, generator=g).to(dtype)
    import contextlib
    with (tcgen05_must_run() if (dtype == torch.bfloat16 and d == 64) else contextlib.nullcontext()):
        out = ops.fused_attention(planes, scale, mode, prm, grid)
        out.backward(d_out.to(DEV))
    pl = planes.detach().double().cpu().numpy()
    o_np, _, _, _ = A.attention_forward(pl[0], pl[1], pl[2], scale, bias_np)
    # the backward re-reads the STORED output (bf16-rounded in bf16 mode) for delta = rowsum(dO*O)
    gr = A.attention_backward(d_out.double().numpy(), pl[0], pl[1], pl[2], scale, bias_np,
                              out=out.detach().double().cpu().numpy())
    tol = FP32_TOL if dtype == torch.float32 else BF16_TOL
    e = err_scaled if dtype == torch.float32 else err_rel
    assert e(out.float(), o_np) <= tol
    want = np.stack([gr["dq"], gr["dk"], gr["dv"]])
    assert e(planes.grad.float(), want) <= tol
    if kind == "table":
        assert e(prm.grad, A.dtable_from_dbias(gr["dbias"])) <= tol
    if kind.startswith("poly"):
        # d_coef[k] = sum over B*H*N^2 terms of dS * d^k: for k = 3 the terms are ~1e4 x larger than the
        # bf16-rounded dS noise of the k = 0 column, all summed into one [..,4] tensor whose max is the
        # k = 3 entry -> a 2x allowance in bf16; flat in fp32
        e_c = e(prm.grad, A.dcoef_from_dbias(gr["dbias"], 3, shared=(kind == "poly")))
        report(f"attn kernel {dtype} n={n} {kind}: d_coef err {e_c:.2e}")
        assert e_c <= (tol if dtype == torch.float32 else 2 * tol)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("rope", ["none", "axial", "mixed"])
@pytest.mark.parametrize("b,n,e,h", [(2, 17, 32, 2), (3, 65, 192, 6), (2, 197, 256, 4), (1, 5, 64, 1)])
def test_qkv_rope_kernel_vs_numpy(dtype, rope, b, n, e, h):
    """QKV projection + RoPE epilogue fwd/bwd vs float64 numpy (rotate-half pairs (d, d+Dh/2), cls row
    un-rotated), including d_cos / d_sin."""
    if rope != "none" and int(round((n - 1) ** 0.5)) ** 2 != n - 1:
        pytest.skip("square grid only")
    dh = e // h
    g = torch.Generator().manual_seed(3)
    x = torch.randn(b, n, e, generator=g).to(dtype)
    w = (torch.randn(3 * e, e, generator=g) * e ** -0.5).to(dtype)
    cos = sin = None
    if rope != "none":
        shape = (n - 1, dh // 2) if rope == "axial" else (h, n - 1, dh // 2)
        ang = torch.rand(*shape, generator=g) * 6.0
        cos, sin = torch.cos(ang), torch.sin(ang)
    xs, ws = x.to(DEV).requires_grad_(True), w.to(DEV).requires_grad_(True)
    cs = None if cos is None else cos.to(DEV).requires_grad_(True)
    sn = None if sin is None else sin.to(DEV).requires_grad_(True)
    planes = ops.QkvRopeFn.apply(xs, ws, cs, sn, h)
    d_pl = torch.randn(3, b, h, n, dh, generator=g).to(dtype)
    planes.backward(d_pl.to(DEV))
    # float64 restatement
    xd, wd = x.double().numpy(), w.double().numpy()
    qkv = (xd @ wd.T).reshape(b, n, 3, h, dh).transpose(2, 0, 3, 1, 4)
    q, k, v = qkv[0], qkv[1], qkv[2]
    if cos is not None:
        qr, kr = A.apply_rope_skip_cls(q, k, cos.numpy(), sin.numpy())
    else:
        qr, kr = q, k
    tol = FP32_TOL if dtype == torch.float32 else BF16_TOL
    e_ = err_scaled if dtype == torch.float32 else err_rel
    assert e_(planes.float(), np.stack([qr, kr, v])) <= tol
    gpl = d_pl.double().numpy()
    dq, dk, dv = gpl[0].copy(), gpl[1].copy(), gpl[2]
    if cos is not None:
        c, s = A._bcast_cs(cos.double().numpy()), A._bcast_cs(sin.double().numpy())
        d2 = dh // 2
        dc = np.zeros((b, h, n - 1, d2))
        ds_ = np.zeros((b, h, n - 1, d2))
        for x0, g0 in ((q, gpl[0]), (k, gpl[1])):
            x1, x2 = x0[:, :, 1:, :d2], x0[:, :, 1:, d2:]
            g1, g2 = g0[:, :, 1:, :d2], g0[:, :, 1:, d2:]
            dc += g1 * x1 + g2 * x2
            ds_ += -g1 * x2 + g2 * x1
        dq[:, :, 1:] = A.rotate_half_inverse(gpl[0][:, :, 1:], c, s)
        dk[:, :, 1:] = A.rotate_half_inverse(gpl[1][:, :, 1:], c, s)
        red = (0,) if rope == "mixed" else (0, 1)
        e_c, e_s = e_(cs.grad, dc.sum(red)), e_(sn.grad, ds_.sum(red))
        report(f"qkv_rope {dtype} {rope} b={b} n={n} e={e}: d_cos {e_c:.2e} d_sin {e_s:.2e}")
        assert e_c <= tol and e_s <= tol
    dqkv = np.stack([dq, dk, dv]).transpose(1, 3, 0, 2, 4).reshape(b * n, 3 * e)
    e_x, e_w = e_(xs.grad.float(), (dqkv @ wd).reshape(b, n, e)), e_(ws.grad.float(), dqkv.T @ xd.reshape(b * n, e))
    report(f"qkv_rope {dtype} {rope} b={b} n={n} e={e}: dx {e_x:.2e} dw {e_w:.2e}")
    assert e_x <= tol and e_w <= tol


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("b,c,hw,p,e,absolute", [(2, 3, 16, 4, 32, False), (3, 1, 32, 4, 192, True),
                                                  (2, 3, 64, 16, 128, True), (1, 3, 24, 8, 80, False)])
def test_patch_embed_kernel_vs_conv2d(dtype, b, c, hw, p, e, absolute):
    g = torch.Generator().manual_seed(4)
    img = torch.randn(b, c, hw, hw, generator=g).to(dtype)
    w = (torch.randn(e, c, p, p, generator=g) * 0.1).to(dtype)
    bias = (torch.randn(e, generator=g) * 0.1).to(dtype)
    cls = (torch.randn(1, 1, e, generator=g) * 0.1).to(dtype)
    pos = (torch.randn(1, 100, e, generator=g) * 0.1).to(dtype) if absolute else None
    leaves = [t.to(DEV).requires_grad_(True) if t is not None else None for t in (w, bias, cls, pos)]
    tok = ops.PatchEmbedFn.apply(img.to(DEV), *leaves, p)
    d_tok = torch.randn(tok.shape, generator=g).to(dtype)
    tok.backward(d_tok.to(DEV))
    ref_leaves = [t.double().requires_grad_(True) if t is not None else None for t in (w, bias, cls, pos)]
    y = F.conv2d(img.double(), ref_leaves[0], ref_leaves[1], stride=p).flatten(2).transpose(1, 2)
    y = torch.cat([ref_leaves[2].expand(b, -1, -1), y], dim=1)
    if absolute:
        y = torch.cat([y[:, :1], y[:, 1:] + ref_leaves[3][:, : y.shape[1] - 1]], dim=1)
    y.backward(d_tok.double())
    tol = FP32_TOL if dtype == torch.float32 else BF16_TOL
    e_ = err_scaled if dtype == torch.float32 else err_rel
    assert e_(tok.float(), y) <= tol
    for got, want in zip(leaves, ref_leaves):
        if got is not None:
            assert e_(got.grad.float(), want.grad) <= tol


@pytest.mark.parametrize("xdt,ydt", [(torch.float32, torch.float32), (torch.float32, torch.bfloat16),
                                     (torch.bfloat16, torch.bfloat16)])
@pytest.mark.parametrize("m,e", [(1, 32), (7, 48), (130, 192), (515, 768), (64, 1024), (3, 100)])
def test_layernorm_kernel_vs_torch(xdt, ydt, m, e):
    """LayerNorm fwd/bwd (N1) vs float64 F.layer_norm: any width (vectorised when E % 128 == 0), the
    autocast combination fp32 in / bf16 out, gamma / beta gradients reduced over all rows."""
    g = torch.Generator().manual_seed(e + m)
    x = (torch.randn(m, e, generator=g) * 1.7 + 0.3).to(xdt)
    w = torch.randn(e, generator=g) * 0.5 + 1.0
    b = torch.randn(e, generator=g) * 0.2
    dy = torch.randn(m, e, generator=g).to(ydt)
    xs = x.to(DEV).requires_grad_(True)
    ws, bs = w.to(DEV).requires_grad_(True), b.to(DEV).requires_grad_(True)
    y = ops.LayerNormFn.apply(xs, ws, bs, 1e-5, ydt)
    assert y.dtype == ydt
    y.backward(dy.to(DEV))
    xr = x.double().requires_grad_(True)
    wr, br = w.double().requires_grad_(True), b.double().requires_grad_(True)
    yr = F.layer_norm(xr, (e,), wr, br, 1e-5)
    yr.backward(dy.double())
    exact = xdt == torch.float32 and ydt == torch.float32
    tol, err = (FP32_TOL, err_scaled) if exact else (BF16_TOL, err_rel)
    assert err(y.float(), yr) <= tol
    assert err(xs.grad.float(), xr.grad) <= tol
    assert err(ws.grad, wr.grad) <= (tol if exact else 1e-3 + tol)
    assert err(bs.grad, br.grad) <= tol


@pytest.mark.parametrize("bdt,ydt", [(torch.float32, torch.float32), (torch.bfloat16, torch.bfloat16),
                                     (torch.float32, torch.bfloat16)])
@pytest.mark.parametrize("m,e", [(5, 48), (130, 192), (515, 768), (3, 100)])
def test_add_layernorm_kernel_vs_torch(bdt, ydt, m, e):
    """Fused residual add + LayerNorm: x_new = x + branch, y = LN(x_new); both outputs feed gradients."""
    g = torch.Generator().manual_seed(e * 3 + m)
    x = torch.randn(m, e, generator=g) * 1.3
    br = (torch.randn(m, e, generator=g) * 0.7).to(bdt)
    w = torch.randn(e, generator=g) * 0.5 + 1.0
    b = torch.randn(e, generator=g) * 0.2
    d_xn = torch.randn(m, e, generator=g)
    d_y = torch.randn(m, e, generator=g).to(ydt)
    leaves = [t.to(DEV).requires_grad_(True) for t in (x, br, w, b)]
    x_new, y = ops.AddLayerNormFn.apply(leaves[0], leaves[1], leaves[2], leaves[3], 1e-5, ydt)
    torch.autograd.backward([x_new, y], [d_xn.to(DEV), d_y.to(DEV)])
    ref = [t.double().requires_grad_(True) for t in (x, br, w, b)]
    xn_r = ref[0] + ref[1]
    y_r = F.layer_norm(xn_r, (e,), ref[2], ref[3], 1e-5)
    torch.autograd.backward([xn_r, y_r], [d_xn.double(), d_y.double()])
    exact = bdt == torch.float32 and ydt == torch.float32
    tol, err = (FP32_TOL, err_scaled) if exact else (BF16_TOL, err_rel)
    assert err(x_new, xn_r) <= FP32_TOL and x_new.dtype == torch.float32
    assert err(y.float(), y_r) <= tol
    assert err(leaves[0].grad, ref[0].grad) <= tol
    assert err(leaves[1].grad.float(), ref[1].grad) <= tol and leaves[1].grad.dtype == bdt
    assert err(leaves[2].grad, ref[2].grad) <= (tol if exact else 1e-3 + tol)
    assert err(leaves[3].grad, ref[3].grad) <= tol


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("m,e,hid", [(7, 32, 128), (197 * 3, 192, 768), (130, 96, 100)])
def test_mlp_and_linear_functions_vs_torch(dtype, m, e, hid):
    """MlpFn / LinearFn (cuBLAS GEMMs + gelu-backward / column-sum kernels) vs float64 autograd."""
    g = torch.Generator().manual_seed(m + hid)
    x = torch.randn(m, e, generator=g).to(dtype)
    w1, b1 = (torch.randn(hid, e, generator=g) * e ** -0.5).to(dtype), (torch.randn(hid, generator=g) * 0.1).to(dtype)
    w2, b2 = (torch.randn(e, hid, generator=g) * hid ** -0.5).to(dtype), (torch.randn(e, generator=g) * 0.1).to(dtype)
    dy = torch.randn(m, e, generator=g).to(dtype)
    leaves = [t.to(DEV).requires_grad_(True) for t in (x, w1, b1, w2, b2)]
    y = ops.MlpFn.apply(*leaves)
    y.backward(dy.to(DEV))
    ref = [t.double().requires_grad_(True) for t in (x, w1, b1, w2, b2)]
    yr = F.linear(F.gelu(F.linear(ref[0], ref[1], ref[2])), ref[3], ref[4])
    yr.backward(dy.double())
    tol, err = (2e-5, err_scaled) if dtype == torch.float32 else (BF16_TOL, err_rel)
    assert err(y.float(), yr) <= tol
    for got, want in zip(leaves, ref):
        assert err(got.grad.float(), want.grad) <= tol
    lin_leaves = [t.to(DEV).requires_grad_(True) for t in (x, w1, b1)]
    z = ops.LinearFn.apply(*lin_leaves)
    dz = torch.randn(m, hid, generator=g).to(dtype)
    z.backward(dz.to(DEV))
    lref = [t.double().requires_grad_(True) for t in (x, w1, b1)]
    F.linear(*lref).backward(dz.double())
    for got, want in zip(lin_leaves, lref):
        assert err(got.grad.float(), want.grad) <= tol


@pytest.mark.parametrize("rope", ["axial", "mixed"])
def test_apply_rotary_emb_public_function(rope):
    b, h, n, d = 2, 3, 16, 32
    g = torch.Generator().manual_seed(6)
    q, k = torch.randn(b, h, n, d, generator=g), torch.randn(b, h, n, d, generator=g)
    ang = torch.rand(*((n, d // 2) if rope == "axial" else (h, n, d // 2)), generator=g) * 6
    cos, sin = torch.cos(ang), torch.sin(ang)
    qd, kd = q.to(DEV).requires_grad_(True), k.to(DEV).requires_grad_(True)
    tgt = qd
    qo, ko = models.apply_rotary_emb(qd, kd, models.reshape_for_broadcast(cos.to(DEV), tgt),
                                     models.reshape_for_broadcast(sin.to(DEV), tgt))
    c, s = A._bcast_cs(cos.double().numpy()), A._bcast_cs(sin.double().numpy())
    assert err_scaled(qo, A.rotate_half(q.double().numpy(), c, s)) <= FP32_TOL
    assert err_scaled(ko, A.rotate_half(k.double().numpy(), c, s)) <= FP32_TOL
    (qo.sum() + 2 * ko.sum()).backward()
    ones = np.ones((b, h, n, d))
    assert err_scaled(qd.grad, A.rotate_half_inverse(ones, c, s)) <= FP32_TOL
    assert err_scaled(kd.grad, 2 * A.rotate_half_inverse(ones, c, s)) <= FP32_TOL
    # the tables are differentiable too (the reference's rope_utils is plain torch arithmetic): autograd of
    # the same expression in float64
    cr, sr = cos.double().requires_grad_(True), sin.double().requires_grad_(True)
    qr, kr = q.double(), k.double()
    cb = cr if rope == "mixed" else cr[None]
    sb = sr if rope == "mixed" else sr[None]
    h2 = d // 2

    def rot(x):
        return torch.cat([x[..., :h2] * cb - x[..., h2:] * sb, x[..., :h2] * sb + x[..., h2:] * cb], dim=-1)

    wq, wk = torch.randn(b, h, n, d, generator=g).double(), torch.randn(b, h, n, d, generator=g).double()
    ((rot(qr) * wq).sum() + (rot(kr) * wk).sum()).backward()
    cd, sd_ = cos.to(DEV).requires_grad_(True), sin.to(DEV).requires_grad_(True)
    qo2, ko2 = models.apply_rotary_emb(q.to(DEV), k.to(DEV), models.reshape_for_broadcast(cd, tgt),
                                       models.reshape_for_broadcast(sd_, tgt))
    ((qo2 * wq.float().to(DEV)).sum() + (ko2 * wk.float().to(DEV)).sum()).backward()
    assert cd.grad is not None and cd.grad.shape == cos.shape
    check_fp32(cd.grad, cr.grad, f"apply_rotary_emb {rope} d_cos")
    check_fp32(sd_.grad, sr.grad, f"apply_rotary_emb {rope} d_sin")


@pytest.mark.parametrize("ta,tb", [(0, 0), (0, 1), (1, 0), (1, 1)])
@pytest.mark.parametrize("m,n,k", [(64, 64, 64), (130, 70, 33), (576, 192, 520), (5, 3, 1000)])
def test_plain_gemm_fp32(ta, tb, m, n, k):
    lib = _lib.load()
    g = torch.Generator().manual_seed(8)
    a = torch.randn((k, m) if ta else (m, k), generator=g).to(DEV)
    b = torch.randn((n, k) if tb else (k, n), generator=g).to(DEV)
    c = torch.empty(m, n, device=DEV)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = lib.vrr_gemm(ctypes.c_void_p(a.data_ptr()), ctypes.c_void_p(b.data_ptr()), ctypes.c_void_p(c.data_ptr()),
                      m, n, k, ta, tb, 0, 0, st)
    assert rc == 0, _lib.last_error()
    want = (a.t() if ta else a).double() @ (b.t() if tb else b).double()
    assert err_scaled(c, want) <= FP32_TOL


# ------------------------------------------------------------------------------------- full-size properties

@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("kind", ["none", "table", "poly"])
def test_attention_properties_at_vitb_size(dtype, kind):
    """BASELINE full size (ViT-B/16-224 geometry: 197 tokens, 12 heads, Dh 64; batch shortened to 32):
    size-independent properties instead of an oracle run.
      * softmax rows sum to 1: with V == 1 the output is exactly 1 (to rounding);
      * linearity in V: attn(q,k,a*v1 + v2) == a*attn(q,k,v1) + attn(q,k,v2);
      * lse is the log-sum-exp: re-deriving one row on the host matches."""
    b, h, n, d = 32, 12, 197, 64
    mode, param, grid, bias_np = _bias_case(kind, h, n)
    prm = None if param is None else param.to(DEV)
    planes = _planes(b, h, n, d, dtype, seed=11).to(DEV)
    scale = d ** -0.5
    ones = planes.clone()
    ones[2] = 1.0
    out1 = ops.fused_attention(ones, scale, mode, prm, grid)
    tol = 1e-5 if dtype == torch.float32 else 1e-2
    assert (out1.float() - 1.0).abs().max().item() <= tol
    v2 = _planes(b, h, n, d, dtype, seed=12)[2].to(DEV)
    pa, pb, pc = planes.clone(), planes.clone(), planes.clone()
    pb[2] = v2
    pc[2] = (0.5 * planes[2].float() + v2.float()).to(dtype)
    oa, ob, oc = (ops.fused_attention(p_, scale, mode, prm, grid).float() for p_ in (pa, pb, pc))
    lin_tol = 2e-5 if dtype == torch.float32 else 4e-2
    assert (oc - (0.5 * oa + ob)).abs().max().item() <= lin_tol
    # one row re-derived in float64
    pl = planes[:, 3, 5].double().cpu().numpy()  # [3, N, D]
    s = pl[0] @ pl[1].T * scale + (0 if bias_np is None else bias_np[5])
    p_ = np.exp(s - s.max(-1, keepdims=True))
    o_row = (p_ / p_.sum(-1, keepdims=True)) @ pl[2]
    got = oa[3].reshape(n, h, d)[:, 5].double().cpu().numpy()
    e = np.abs(got - o_row).max() / max(1.0, np.abs(o_row).max())
    assert e <= (FP32_TOL if dtype == torch.float32 else BF16_TOL)


# ------------------------------------------------------------------------------------- persistent kernels

def _set_option(name, value):
    _lib.check(_lib.load().vrr_set_option(name.encode(), int(value)), f"vrr_set_option({name})")


@pytest.mark.parametrize("b,h,n", [(30, 12, 197), (40, 8, 65), (2, 3, 130), (171, 2, 197)])
def test_persistent_backward_many_items_per_cta(b, h, n):
    """Without bias at N <= 208 the forward is attn_fwd_tc4_kernel (one CTA per 128-row tile, four per SM) and the
    backward the persistent whole-sequence kernel (attn_bwd_ws.cu): with more (image, head) items than SMs every
    backward CTA walks several items through its double-buffered shared memory, TMEM and barrier phases.
    fwd + bwd of ALL items against float64 numpy, error checked per item (rotating-buffer bugs only show from the
    second item on), and bit-for-bit run-to-run reproducibility of the forward (no atomics on this path)."""
    d = 64
    planes = _planes(b, h, n, d, torch.bfloat16, seed=21).to(DEV).requires_grad_(True)
    g = torch.Generator().manual_seed(22)
    d_out = (torch.randn(b, n, h * d, generator=g) * 0.5).to(torch.bfloat16)
    scale = d ** -0.5
    with tcgen05_must_run():
        out = ops.fused_attention(planes, scale)
        out.backward(d_out.to(DEV))
    out2 = ops.fused_attention(planes.detach(), scale)
    assert torch.equal(out, out2), "forward is not reproducible run to run"
    pl = planes.detach().double().cpu().numpy()
    o_np, _, _, _ = A.attention_forward(pl[0], pl[1], pl[2], scale, None)
    gr = A.attention_backward(d_out.double().numpy(), pl[0], pl[1], pl[2], scale, None, out=out.detach().double().cpu().numpy())
    assert torch.isfinite(planes.grad).all()
    assert err_rel(out.float(), o_np) <= BF16_TOL
    # per item: a wrong item hides in a global max-norm when its neighbours are right
    got = planes.grad.float().cpu().numpy().reshape(3, b * h, n, d)
    want = np.stack([gr["dq"], gr["dk"], gr["dv"]]).reshape(3, b * h, n, d)
    per_item = np.abs(got - want).max(axis=(2, 3)) / np.maximum(np.abs(want).max(axis=(2, 3)), 1e-6)
    report(f"persistent attention b={b} h={h} n={n}: worst per-item grad err {per_item.max():.2e}")
    assert per_item.max() <= 2 * BF16_TOL, (np.unravel_index(per_item.argmax(), per_item.shape), per_item.max())


@pytest.mark.parametrize("rope", ["axial", "mixed"])
@pytest.mark.parametrize("b,n,e,h", [(3, 197, 768, 12), (2, 50, 128, 2), (5, 65, 192, 3), (32, 197, 768, 12)])
def test_qkv_rope_packed_tables_bit_identical(rope, b, n, e, h):
    """vrr_rope_pack_tables + vrr_qkv_rope_fwd_packed (coalesced table reads in the tcgen05 epilogue) against
    vrr_qkv_rope_fwd on the same inputs: bit-identical planes; and the Python-side cache notices a table that changed
    in place."""
    lib = _lib.load()
    dh = e // h
    g = torch.Generator().manual_seed(11)
    x = torch.randn(b, n, e, generator=g).to(torch.bfloat16).to(DEV)
    w = (torch.randn(3 * e, e, generator=g) * e ** -0.5).to(torch.bfloat16).to(DEV)
    heads = h if rope == "mixed" else 1
    ang = torch.rand(heads, n - 1, dh // 2, generator=g) * 6.0
    cos, sin = torch.cos(ang).to(DEV), torch.sin(ang).to(DEV)
    mode = _lib.ROPE_MIXED if rope == "mixed" else _lib.ROPE_AXIAL
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())
    plain = torch.empty(3, b, h, n, dh, device=DEV, dtype=torch.bfloat16)
    fast = torch.empty_like(plain)
    packed = torch.empty(heads, dh // 4, n - 1, 4, device=DEV)
    with tcgen05_must_run():
        _lib.check(lib.vrr_qkv_rope_fwd(p(x), p(w), p(cos), p(sin), p(plain), b, n, e, h, mode, 1, st), "plain")
    _lib.check(lib.vrr_rope_pack_tables(p(cos), p(sin), p(packed), heads, n - 1, dh // 2, st), "pack")
    want = torch.stack([cos[..., 0::2], sin[..., 0::2], cos[..., 1::2], sin[..., 1::2]], dim=-1).permute(0, 2, 1, 3)
    assert torch.equal(packed, want.contiguous())
    with tcgen05_must_run():
        _lib.check(lib.vrr_qkv_rope_fwd_packed(p(x), p(w), p(cos), p(sin), p(packed), p(fast), b, n, e, h, mode, 1, st), "packed")
    assert torch.equal(plain, fast)
    # host mirror: same storage + same version -> cached; an in-place change -> repacked
    cs = cos if rope == "mixed" else cos[0]
    sn = sin if rope == "mixed" else sin[0]
    out1 = ops.QkvRopeFn.apply(x, w, cs, sn, h)
    assert torch.equal(out1, plain)
    cs.mul_(-1.0)
    out2 = ops.QkvRopeFn.apply(x, w, cs, sn, h)
    _lib.check(lib.vrr_qkv_rope_fwd(p(x), p(w), p(cos), p(sin), p(plain), b, n, e, h, mode, 1, st), "plain")
    assert torch.equal(out2, plain) and not torch.equal(out1, out2)
    with torch.inference_mode():  # inference tensors have no version counter: the cache must step aside, not raise
        ang2 = torch.rand(heads, n - 1, dh // 2, device=DEV) * 6.0
        c2, s2 = torch.cos(ang2), torch.sin(ang2)
        out3 = ops.QkvRopeFn.apply(x, w, c2 if rope == "mixed" else c2[0], s2 if rope == "mixed" else s2[0], h)
    _lib.check(lib.vrr_qkv_rope_fwd(p(x), p(w), p(c2), p(s2), p(plain), b, n, e, h, mode, 1, st), "plain")
    assert torch.equal(out3, plain)


@pytest.mark.parametrize("b,h,n", [(2, 3, 257), (1, 2, 577), (3, 2, 641), (1, 2, 1025)])
def test_long_sequence_forward_vs_oracle(b, h, n):
    """N > 256 without bias: the four-CTAs-per-SM forward (single S buffer, chunked TMEM re-reads, 2 of every 8
    exponential pairs by polynomial on the FMA pipe) against the float64 numpy oracle; ragged last key tile
    (n % 64 = 1) and ragged last row tile."""
    d = 64
    planes = _planes(b, h, n, d, torch.bfloat16, seed=41).to(DEV)
    pl = planes.double().cpu().numpy()
    want, _, _, _ = A.attention_forward(pl[0], pl[1], pl[2], d ** -0.5, None)  # [B, N, H*D]
    with tcgen05_must_run():
        out = ops.fused_attention(planes, d ** -0.5)
    e = err_rel(out.float(), want)
    report(f"long forward b={b} h={h} n={n}: err {e:.2e}")
    assert e <= 1e-2, e


@pytest.mark.parametrize("m,n,k", [(394, 3072, 768), (130, 104, 72), (1000, 256, 520), (6304, 3072, 768)])
def test_gemm_epilogues_gelu_grad_and_mul(m, n, k):
    """VRR_EPI_BIAS_GELU_GRAD (c = gelu(h), c2 = gelu'(h), h = bf16(a.b^T + bias)) and VRR_EPI_MUL (c = (a.b) * c2),
    the pair that replaces the stand-alone GELU backward: against torch in fp32 on the bf16-rounded h."""
    g = torch.Generator().manual_seed(5)
    a = (torch.randn(m, k, generator=g) * 0.5).to(torch.bfloat16).to(DEV)
    w = (torch.randn(n, k, generator=g) * k ** -0.5).to(torch.bfloat16).to(DEV)
    bias = torch.randn(n, generator=g).to(DEV)
    with tcgen05_must_run():
        act, gp = ops._gemm(a, w, False, True, torch.bfloat16, bias=bias, epilogue=_lib.EPI_BIAS_GELU_GRAD, out2=True)
    h = (a.float() @ w.float().t() + bias.to(torch.bfloat16).float()).to(torch.bfloat16).float().requires_grad_(True)
    ref = F.gelu(h)
    ref.sum().backward()
    assert err_rel(act.float(), ref.detach().cpu().numpy()) <= 1e-2
    assert err_rel(gp.float(), h.grad.cpu().numpy()) <= 1e-2
    with tcgen05_must_run():  # the inference epilogue: the same activation, alone
        act_only = ops._gemm(a, w, False, True, torch.bfloat16, bias=bias, epilogue=_lib.EPI_BIAS_GELU_ACT)
    assert torch.equal(act_only, act)
    a32, w32 = a.float(), w.float()  # SIMT family (fp32): c = gelu(h) alone against torch
    act32 = ops._gemm(a32, w32, False, True, torch.float32, bias=bias, epilogue=_lib.EPI_BIAS_GELU_ACT)
    assert err_rel(act32, F.gelu(a32 @ w32.t() + bias).cpu().numpy()) <= 1e-5
    dy = (torch.randn(m, n, generator=g) * 0.5).to(torch.bfloat16).to(DEV)
    w2 = (torch.randn(n, k, generator=g) * n ** -0.5).to(torch.bfloat16).to(DEV)  # dX = dy . w2 -> [m, k]
    mul = torch.randn(m, k, generator=g).to(torch.bfloat16).to(DEV)
    with tcgen05_must_run():
        dx = ops._gemm(dy, w2, False, False, torch.bfloat16, epilogue=_lib.EPI_MUL, aux=mul)
    want = (dy.float() @ w2.float()) * mul.float()
    assert err_rel(dx.float(), want.cpu().numpy()) <= 1e-2
    # the same GEMM with the column sums of its output (fc1's bias gradient) from the epilogue
    lib = _lib.load()
    dx2 = torch.empty_like(dx)
    sums = torch.full((k,), float("nan"), device=DEV)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    with tcgen05_must_run():
        _lib.check(lib.vrr_gemm_mul_colsum(p(dy), p(w2), p(dx2), p(mul), p(sums), m, k, n, 0, 0, 1, st), "mul_colsum")
    assert torch.equal(dx2, dx)
    assert err_rel(sums, dx.float().sum(0).cpu().numpy()) <= 1e-5
    dy32, w32_, mul32 = dy.float(), w2.float(), mul.float()  # SIMT family: same entry point, fp32
    dx32 = torch.empty(m, k, device=DEV)
    _lib.check(lib.vrr_gemm_mul_colsum(p(dy32), p(w32_), p(dx32), p(mul32), p(sums), m, k, n, 0, 0, 0, st), "mul_colsum f32")
    assert err_rel(dx32, want.cpu().numpy()) <= 1e-5
    assert err_rel(sums, dx32.sum(0).cpu().numpy()) <= 1e-5
