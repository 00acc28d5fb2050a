"""Cost of QK-norm in the training step (one process, one GPU).

ViT-B/16-224 rope-mixed bf16 at batch 256, the whole step (forward, backward, AdamW) captured in one CUDA graph as
bench.py captures it, timed for qk_norm False and True in alternating windows; then the per-launch times of the QKV
forward (qkv_rope_fwd: the GEMM with its RoPE / QK-norm epilogue) and of its backward kernel (qkv_rope_bwd) of each
setting from eager steps through the ``ops._timed`` hooks.  The card's name and power limit are read in the same run.

    python scripts/qk_norm_time.py [--steps 20] [--rounds 5] [--out result.json]
"""
import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from dropout_time import card, time_window  # noqa: E402
from vit_rpe_rope_b200 import VisionTransformer, ops  # noqa: E402
from vit_rpe_rope_b200.dp import BucketedDataParallel  # noqa: E402
from vit_rpe_rope_b200.runtime import GraphedTrainStep  # noqa: E402

VITB = dict(img_size=224, patch_size=16, in_chans=3, num_classes=1000, embed_dim=768, depth=12, num_heads=12,
            pos_encoding="rope-mixed")
KERNELS = ("qkv_rope_fwd", "qkv_rope_bwd")


def make_runner(qk_norm, batch, dev):
    torch.manual_seed(0)
    model = VisionTransformer(**VITB, qk_norm=qk_norm).to(dev)
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--out", type=str, default="")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    settings = (False, True)
    runners = {s: make_runner(s, args.batch, dev) for s in settings}
    ms = {s: [] for s in settings}
    for _ in range(args.rounds):
        for s in settings:
            ms[s].append(time_window(runners[s], args.steps))
    rows = []
    for s in settings:
        m = statistics.median(ms[s])
        rows.append({"qk_norm": s, "ms_per_step": m, "ms_windows": ms[s], "images_per_s": args.batch / (m / 1e3),
                     "kernels": kernel_times(runners[s], 3)})
        runners[s].graph = None
    res = {"card": card(), "torch": torch.__version__, "vitb16_224_rope_mixed_bf16": rows,
           "step_cost_of_qk_norm": rows[1]["ms_per_step"] / rows[0]["ms_per_step"] - 1}
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
