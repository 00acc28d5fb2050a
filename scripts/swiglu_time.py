"""Cost of the SwiGLU MLP against the GELU MLP in the training step, and of its fused kernels against the unfused
composition (one process, one GPU).

1. ViT-B/16-224 rope-mixed bf16 at batch 256, the whole step (forward, backward, AdamW) captured in one CUDA graph as
   bench.py captures it, for ``Mlp`` (mlp_ratio 4) and ``SwiGLUPacked`` (mlp_ratio 5.33334: fc1 768 -> 4096, fc2
   2048 -> 768, the GELU MLP's parameters and FLOPs) in alternating windows; then the per-launch medians of fc1_fwd,
   fc2_dx, fc1_dx and fc1_dw of each from eager steps through the ``ops._timed`` hooks.
2. At the same shapes (M = 256 x 197 tokens, K = 768, H = 2048), CUDA events around repeated launches of
     fused forward   vrr_gemm_swiglu (act and aux from one GEMM)
     unfused forward vrr_gemm_ex(EPI_BIAS) to h [M][2H], then an elementwise pass h -> act, aux
     fused backward  vrr_gemm_swiglu_bwd (dh and fc1's bias gradient from fc2's dX GEMM)
     unfused backward the plain dX GEMM to dA [M][H], then an elementwise pass dA, aux -> dh, db1
   The elementwise passes are timed as torch ops and also bounded below by their HBM traffic at 7.7 TB/s (the HGX B200
   data-sheet bandwidth of one GPU): the fused kernel is compared with GEMM + that floor, the cheapest any separate
   pass could be.  Every operand set is larger than the 126 MB L2.
The card's name and power limit are read in the same run.

    python scripts/swiglu_time.py [--steps 20] [--rounds 5] [--out result.json]
"""
import argparse
import json
import os
import statistics
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from dropout_time import card, time_window  # noqa: E402
from vit_rpe_rope_b200 import VisionTransformer, _lib, ops  # noqa: E402
from vit_rpe_rope_b200.dp import BucketedDataParallel  # noqa: E402
from vit_rpe_rope_b200.models.vit import Mlp, SwiGLUPacked  # noqa: E402
from vit_rpe_rope_b200.runtime import GraphedTrainStep  # noqa: E402

VITB = dict(img_size=224, patch_size=16, in_chans=3, num_classes=1000, embed_dim=768, depth=12, num_heads=12,
            pos_encoding="rope-mixed")
SETTINGS = {"gelu_mlp": dict(mlp_layer=Mlp, mlp_ratio=4.0), "swiglu_packed": dict(mlp_layer=SwiGLUPacked, mlp_ratio=5.33334)}
KERNELS = ("fc1_fwd", "fc2_dx", "fc1_dx", "fc1_dw")
HBM_BYTES_PER_S = 7.7e12


def make_runner(kw, batch, dev):
    torch.manual_seed(0)
    model = VisionTransformer(**VITB, **kw).to(dev)
    dp = BucketedDataParallel(model, bucket_mb=32.0)
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3, weight_decay=0.01, fused=True, capturable=True)
    g = torch.Generator().manual_seed(1234)
    images = torch.randn(batch, 3, 224, 224, generator=g).to(dev)
    labels = torch.randint(0, 1000, (batch,), generator=g).to(dev)
    runner = GraphedTrainStep(dp, opt, tuple(images.shape), 1000, dev, bf16=True, use_graph=True)
    runner.prepare(images, labels)
    return runner


def kernel_times(runner, steps):
    ops.PROFILE_EVENTS = []
    for _ in range(steps):
        runner._eager_step()
    torch.cuda.synchronize()
    events, ops.PROFILE_EVENTS = ops.PROFILE_EVENTS, None
    per = {}
    for name, a, b in events:
        if name in KERNELS:
            per.setdefault(name, []).append(a.elapsed_time(b) * 1e3)
    return {k: {"median_us": statistics.median(v), "launches_per_step": len(v) // steps} for k, v in per.items()}


def time_us(fn, reps=20, windows=5):
    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(windows):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1) * 1e3 / reps)
    return statistics.median(out)


def fused_vs_unfused(dev, batch):
    lib, st = _lib.load(), ops._stream
    M, K, H = batch * 197, 768, 2048
    bf = torch.bfloat16
    g = torch.Generator(device=dev).manual_seed(5)
    x = torch.randn(M, K, device=dev, generator=g).to(bf)
    w1 = (torch.randn(2 * H, K, device=dev, generator=g) * 0.02).to(bf)
    b1 = torch.randn(2 * H, device=dev, generator=g) * 0.02
    w2 = (torch.randn(K, H, device=dev, generator=g) * 0.02).to(bf)
    dy = torch.randn(M, K, device=dev, generator=g).to(bf)
    act, aux = torch.empty(M, H, device=dev, dtype=bf), torch.empty(M, 2 * H, device=dev, dtype=bf)
    dh, db1 = torch.empty(M, 2 * H, device=dev, dtype=bf), torch.empty(2 * H, device=dev)
    p = ops._ptr

    def fused_fwd():
        _lib.check(lib.vrr_gemm_swiglu(p(x), p(w1), p(b1), p(act), p(aux), M, H, K, _lib.VRR_BF16, None, st()), "swiglu")

    def fused_bwd():
        _lib.check(lib.vrr_gemm_swiglu_bwd(p(dy), p(w2), p(aux), p(dh), p(db1), M, H, K, _lib.VRR_BF16, st()), "swiglu_bwd")

    h = ops._gemm(x, w1, False, True, bf, bias=b1, epilogue=_lib.EPI_BIAS)
    dA = ops._gemm(dy, w2, False, False, bf)

    def fwd_elementwise():
        gate, val = h.chunk(2, -1)
        s = F.silu(gate)
        torch.mul(s, val, out=act)
        sig = torch.sigmoid(gate)
        aux[:, :H] = val * (sig + s * (1 - sig))
        aux[:, H:] = s

    def bwd_elementwise():
        torch.mul(dA.repeat(1, 2), aux, out=dh)
        db1.copy_(dh.float().sum(0))

    fam = _lib.family_count(_lib.IMPL_TCGEN05)
    res = {
        "shape": {"M": M, "K": K, "H": H},
        "fused_fwd_us": time_us(fused_fwd),
        "bias_gemm_to_2H_us": time_us(lambda: ops._gemm(x, w1, False, True, bf, bias=b1, epilogue=_lib.EPI_BIAS)),
        "fwd_elementwise_torch_us": time_us(fwd_elementwise),
        "fwd_elementwise_hbm_floor_us": M * (2 * H + 3 * H) * 2 / HBM_BYTES_PER_S * 1e6,  # read h, write act + aux
        "fused_bwd_us": time_us(fused_bwd),
        "dx_gemm_to_H_us": time_us(lambda: ops._gemm(dy, w2, False, False, bf)),
        "bwd_elementwise_torch_us": time_us(bwd_elementwise),
        "bwd_elementwise_hbm_floor_us": M * (H + 2 * H + 2 * H) * 2 / HBM_BYTES_PER_S * 1e6,  # read dA, aux, write dh
    }
    assert _lib.family_count(_lib.IMPL_TCGEN05) > fam
    res["fwd_unfused_floor_us"] = res["bias_gemm_to_2H_us"] + res["fwd_elementwise_hbm_floor_us"]
    res["bwd_unfused_floor_us"] = res["dx_gemm_to_H_us"] + res["bwd_elementwise_hbm_floor_us"]
    res["fused_fwd_beats_unfused"] = res["fused_fwd_us"] < res["fwd_unfused_floor_us"]
    res["fused_bwd_beats_unfused"] = res["fused_bwd_us"] < res["bwd_unfused_floor_us"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--out", type=str, default="")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    runners = {name: make_runner(kw, args.batch, dev) for name, kw in SETTINGS.items()}
    ms = {name: [] for name in SETTINGS}
    for _ in range(args.rounds):  # alternating windows
        for name in SETTINGS:
            ms[name].append(time_window(runners[name], args.steps))
    rows = {}
    for name in SETTINGS:
        m = statistics.median(ms[name])
        rows[name] = {"ms_per_step": m, "ms_windows": ms[name], "images_per_s": args.batch / (m / 1e3),
                      "kernels": kernel_times(runners[name], 3)}
        runners[name].graph = None
    del runners
    torch.cuda.empty_cache()
    res = {"card": card(), "torch": torch.__version__, "vitb16_224_rope_mixed_bf16_b%d" % args.batch: rows,
           "step_time_swiglu_over_gelu": rows["swiglu_packed"]["ms_per_step"] / rows["gelu_mlp"]["ms_per_step"],
           "fc1_fused_vs_unfused": fused_vs_unfused(dev, args.batch)}
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
