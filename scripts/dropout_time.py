"""Cost of dropout and stochastic depth in the training step (one process, one GPU).

ViT-B/16-224 rope-mixed bf16 at batch 256, the whole step (forward, backward, AdamW) captured in one CUDA graph as
bench.py captures it, timed for (drop_path_rate, drop_rate) = (0, 0), (0.1, 0), (0.1, 0.1) in alternating windows;
then the per-launch times of add_layernorm_fwd / _bwd and fc1_fwd of each setting from eager steps through the
``ops._timed`` hooks; then ViT-Tiny fp32 (rope-axial, batch 128) at (0, 0) and (0.1, 0.1).  The card's name and
power limit are read in the same run.

    python scripts/dropout_time.py [--steps 20] [--rounds 5] [--out result.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from vit_rpe_rope_b200 import VisionTransformer, ops  # noqa: E402
from vit_rpe_rope_b200.dp import BucketedDataParallel  # noqa: E402
from vit_rpe_rope_b200.runtime import GraphedTrainStep  # noqa: E402

VITB = dict(img_size=224, patch_size=16, in_chans=3, num_classes=1000, embed_dim=768, depth=12, num_heads=12,
            pos_encoding="rope-mixed")
TINY = dict(img_size=32, patch_size=4, in_chans=3, num_classes=10, embed_dim=192, depth=6, num_heads=6,
            pos_encoding="rope-axial")
KERNELS = ("add_layernorm_fwd", "add_layernorm_bwd", "fc1_fwd")


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as e:  # pragma: no cover
        return {"name": torch.cuda.get_device_name(), "power_limit": f"unavailable ({type(e).__name__})"}


def make_runner(cfg, batch, bf16, dpr, dr, dev):
    torch.manual_seed(0)
    model = VisionTransformer(**cfg, drop_rate=dr, drop_path_rate=dpr).to(dev)
    dp = BucketedDataParallel(model, bucket_mb=32.0)
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3, weight_decay=0.01, fused=True, capturable=True)
    g = torch.Generator().manual_seed(1234)
    images = torch.randn(batch, cfg["in_chans"], cfg["img_size"], cfg["img_size"], generator=g).to(dev)
    labels = torch.randint(0, cfg["num_classes"], (batch,), generator=g).to(dev)
    runner = GraphedTrainStep(dp, opt, tuple(images.shape), cfg["num_classes"], dev, bf16=bf16, use_graph=True)
    runner.prepare(images, labels)
    return runner


def time_window(runner, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    runner.run()
    e0.record()
    for _ in range(steps):
        runner.run()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


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


def sweep(cfg, batch, bf16, settings, steps, rounds, dev):
    runners = {s: make_runner(cfg, batch, bf16, s[0], s[1], dev) for s in settings}
    ms = {s: [] for s in settings}
    for _ in range(rounds):
        for s in settings:
            ms[s].append(time_window(runners[s], steps))
    out = []
    for s in settings:
        m = statistics.median(ms[s])
        out.append({"drop_path_rate": s[0], "drop_rate": s[1], "ms_per_step": m, "ms_windows": ms[s],
                    "images_per_s": batch / (m / 1e3), "kernels": kernel_times(runners[s], 3)})
        runners[s].graph = None
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", type=str, default="")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    res = {"card": card(), "torch": torch.__version__,
           "vitb16_224_rope_mixed_bf16_b256": sweep(VITB, 256, True, [(0.0, 0.0), (0.1, 0.0), (0.1, 0.1)],
                                                    args.steps, args.rounds, dev),
           "vit_tiny_rope_axial_fp32_b128": sweep(TINY, 128, False, [(0.0, 0.0), (0.1, 0.1)], args.steps, args.rounds,
                                                  dev)}
    print(json.dumps(res, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
