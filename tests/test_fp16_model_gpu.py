"""The model under float16 autocast: ``torch.autocast("cuda")`` (whose CUDA default is float16) and
``torch.amp.GradScaler``, the most common mixed-precision recipe, against the fp32 oracle.

Each logit and gradient must pass two bars: the flat 2e-2 relative bar of the bf16 tests, and a bar relative to the
reference's own error under the same autocast (``err <= 2 * err_ref16 + FP16_SLACK``).  The second one is what fp16
buys over bf16; rounding any GEMM or attention output to bf16 first does not pass it.
"""
import csv
import os

import pytest
import torch
import torch.nn.functional as F

import train
from oracle import vit_torch as V
from test_parity_gpu import BF16_TOL, MODES, _build_pair, _tiny_kwargs, err_rel, report, tcgen05_must_run
from vit_rpe_rope_b200 import VisionTransformer

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
FP16_SLACK = 2e-3


def check_fp16(got, want32, ref16, what):
    e_mine, e_ref = err_rel(got, want32), err_rel(ref16, want32)
    bound = min(BF16_TOL, 2 * e_ref + FP16_SLACK)
    report(f"fp16 {what}: mine {e_mine:.2e} ref-autocast {e_ref:.2e} bound {bound:.2e}")
    assert e_mine <= bound, (what, e_mine, e_ref)


def _oracle(kw, sd, images, labels, autocast):
    cfg = V.VitConfig(**kw)
    p = V.params_from_state_dict(sd, device=DEV)
    with torch.autocast("cuda", dtype=torch.float16, enabled=autocast):
        logits = V.forward(cfg, p, images.to(DEV))
        loss = F.cross_entropy(logits.float(), labels.to(DEV))
    loss.backward()
    return logits.detach().float(), {k: v.grad for k, v in p.items() if v.is_floating_point() and v.grad is not None}


def _fp16_model_case(kw, batch, size, train_=True, seed=2, tcgen05=True):
    model, sd = _build_pair(kw)
    torch.manual_seed(seed)
    images = torch.randn(batch, kw["in_chans"], size, size)
    labels = torch.randint(0, kw["num_classes"], (batch,))
    tag = f"{kw['pos_encoding']} E={kw['embed_dim']} H={kw['num_heads']} N={(size // kw['patch_size']) ** 2 + 1}"
    must = tcgen05_must_run() if tcgen05 else _Nothing()
    if not train_:
        model.eval()
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16), must:
            logits = model(images.to(DEV))
        cfg = V.VitConfig(**kw)
        with torch.no_grad():
            p32 = V.params_from_state_dict(sd, device=DEV, requires_grad=False)
            want32 = V.forward(cfg, p32, images.to(DEV))
            with torch.autocast("cuda", dtype=torch.float16):
                want16 = V.forward(cfg, p32, images.to(DEV)).float()
        check_fp16(logits.float(), want32, want16, f"{tag} logits (eval)")
        return
    with must:
        with torch.autocast("cuda", dtype=torch.float16):
            logits = model(images.to(DEV))
            loss = F.cross_entropy(logits.float(), labels.to(DEV))
        loss.backward()
    want32, grads32 = _oracle(kw, sd, images, labels, autocast=False)
    want16, grads16 = _oracle(kw, sd, images, labels, autocast=True)
    check_fp16(logits.float(), want32, want16, f"{tag} logits")
    for name, p in model.named_parameters():
        assert p.grad.dtype == torch.float32
        check_fp16(p.grad, grads32[name], grads16[name], f"{tag} {name}")


class _Nothing:
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


@pytest.mark.parametrize("mode", MODES)
def test_vit_fp16_autocast_head_dim_64(mode):
    """All six modes at the 64-wide-head geometry: the tcgen05 kernels in fp16."""
    kw = dict(img_size=64, patch_size=8, in_chans=3, num_classes=10, embed_dim=256, depth=2, num_heads=4,
              pos_encoding=mode)
    _fp16_model_case(kw, batch=16, size=64)


@pytest.mark.parametrize("mode", ["rope-mixed", "relative", "polynomial"])
def test_cfg3_geometry_fp16(mode):
    kw = dict(img_size=224, patch_size=16, in_chans=3, num_classes=1000, embed_dim=768, depth=2, num_heads=12,
              pos_encoding=mode)
    _fp16_model_case(kw, batch=4, size=224)


def test_cfg4_geometry_fp16():
    kw = dict(img_size=384, patch_size=16, in_chans=3, num_classes=1000, embed_dim=1024, depth=1, num_heads=16,
              pos_encoding="rope-axial")
    _fp16_model_case(kw, batch=2, size=384)


def test_cfg5_inference_1025_tokens_fp16():
    kw = dict(img_size=224, patch_size=16, in_chans=3, num_classes=1000, embed_dim=768, depth=2, num_heads=12,
              pos_encoding="rope-mixed")
    _fp16_model_case(kw, batch=2, size=512, train_=False)


@pytest.mark.parametrize("mode", MODES)
def test_reference_vit_tiny_fp16(mode):
    """The reference's default ViT-Tiny (head dim 32): SIMT attention in fp16, tcgen05 GEMMs where they fit."""
    kw = _tiny_kwargs(mode, in_chans=3)
    _fp16_model_case(kw, batch=8, size=kw["img_size"], tcgen05=False)


def test_default_autocast_dtype_is_fp16():
    """``torch.autocast("cuda")`` without a dtype equals dtype=torch.float16: the forward bit for bit, and every
    gradient within the run-to-run spread of two dtype=torch.float16 backwards (the fp32 weight gradients are split
    over K and combined by reduce-adds, and the bias / table gradients by atomics, so their last bits vary from run to
    run; a bf16 backward would differ by ~1e-2)."""
    kw = dict(img_size=64, patch_size=8, in_chans=3, num_classes=10, embed_dim=256, depth=1, num_heads=4,
              pos_encoding="relative")
    model, _ = _build_pair(kw)
    x = torch.randn(8, 3, 64, 64, device=DEV)
    runs = []
    for ctx in (lambda: torch.autocast("cuda"), lambda: torch.autocast("cuda", dtype=torch.float16),
                lambda: torch.autocast("cuda", dtype=torch.float16)):
        model.zero_grad(set_to_none=True)
        with ctx(), tcgen05_must_run():
            y = model(x)
        y.float().square().mean().backward()
        runs.append((y.detach().clone(), [p.grad.clone() for p in model.parameters()]))
    assert y.dtype == torch.float16
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[1][0], runs[2][0])
    for (name, _), g0, g1, g2 in zip(model.named_parameters(), runs[0][1], runs[1][1], runs[2][1]):
        spread = (g1 - g2).abs().max().item()
        assert (g0 - g1).abs().max().item() <= 2 * spread + 1e-7 * g1.abs().max().item(), name


def _scaler_step(model, opt, scaler, x, y):
    opt.zero_grad(set_to_none=True)
    with torch.autocast("cuda", dtype=torch.float16):
        loss = F.cross_entropy(model(x).float(), y)
    scaler.scale(loss).backward()
    scaler.unscale_(opt)
    finite = all(torch.isfinite(p.grad).all().item() for p in model.parameters() if p.grad is not None)
    scaler.step(opt)
    scaler.update()
    return finite


def test_grad_scaler_normal_scale_and_overflow_skip():
    kw = dict(img_size=64, patch_size=8, in_chans=3, num_classes=10, embed_dim=256, depth=2, num_heads=4,
              pos_encoding="relative")
    model, _ = _build_pair(kw)
    opt = torch.optim.AdamW(model.parameters(), lr=1e-4)
    g = torch.Generator().manual_seed(3)
    x = torch.randn(16, 3, 64, 64, generator=g).to(DEV)
    y = torch.randint(0, 10, (16,), generator=g).to(DEV)
    # a normal scale: finite gradients, the scale never drops
    scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 10)
    for _ in range(3):
        with tcgen05_must_run():
            assert _scaler_step(model, opt, scaler, x, y)
        assert scaler.get_scale() >= 2.0 ** 10
    # 2^60: the first step overflows (fp16 gradients become inf, not a clamped finite value), is skipped, scale halves
    before = [p.detach().clone() for p in model.parameters()]
    scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 60)
    assert not _scaler_step(model, opt, scaler, x, y)
    assert scaler.get_scale() == 2.0 ** 59
    assert all(torch.equal(a, p.detach()) for a, p in zip(before, model.parameters()))


def test_training_run_amp_fp16(tmp_path):
    """train.py --amp fp16 (autocast float16 + GradScaler): three synthetic epochs at head dim 64; the loss falls and
    the checkpoint strict-loads into a fresh VisionTransformer."""
    mode = "rope-mixed"
    argv = ["--dataset", "cifar10", "--pos_encoding", mode, "--epochs", "3", "--batch_size", "64", "--synthetic",
            "--synthetic_size", "512", "--log_dir", str(tmp_path / "logs"), "--ckpt_dir", str(tmp_path / "ck"),
            "--amp", "fp16", "--embed_dim", "128", "--num_heads", "2", "--depth", "2"]
    log_file, ckpt = train.main(argv)
    rows = list(csv.reader(open(log_file)))
    assert rows[0] == ["epoch", "train_loss", "train_acc", "test_loss", "test_acc", "best_acc"]
    losses = [float(r[1]) for r in rows[1:]]
    assert len(losses) == 3 and losses[-1] < losses[0], losses
    assert os.path.basename(ckpt) == f"cifar10_{mode}_best.pth"
    VisionTransformer(img_size=32, patch_size=4, in_chans=3, num_classes=10, pos_encoding=mode, embed_dim=128,
                      num_heads=2, depth=2).load_state_dict(torch.load(ckpt), strict=True)


def test_graphed_inference_fp16_replays_the_eager_forward():
    from vit_rpe_rope_b200.runtime import GraphedInference
    torch.manual_seed(0)
    model = VisionTransformer(img_size=64, patch_size=8, in_chans=3, num_classes=10, embed_dim=256, depth=2, num_heads=4,
                              pos_encoding="rope-mixed").to(DEV).eval()
    runner = GraphedInference(model, (4, 3, 96, 96), torch.device(DEV), amp_dtype=torch.float16)
    assert runner.graph is not None
    g = torch.Generator().manual_seed(7)
    for _ in range(3):
        x = torch.randn(4, 3, 96, 96, generator=g).to(DEV)
        got = runner.run(x).clone()
        assert got.dtype == torch.float16
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
            want = model(x)
        assert torch.equal(got, want)
    runner.close()
