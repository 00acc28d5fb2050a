"""bf16 against fp16 autocast on the same kernels, alternated in one process.

Times (CUDA events, eager, fresh random inputs, after warm-up), for each dtype in turn, `--rounds` times:
  * the ViT-B/16-224 rope-mixed training step, batch 256, WITHOUT GradScaler (the kernels compared like for like);
  * the same step with torch.amp.GradScaler (fp16 only: its cost over the plain step);
  * the ViT-L/16-384 rope-axial training step, batch 64;
  * the ViT-B/16 forward at 512 px (1025 tokens), batch 64, no_grad;
and the per-kernel times of attn_fwd, attn_bwd, qkv_rope_fwd and fc1_fwd inside the ViT-B step (ops.PROFILE_EVENTS).
Prints the card's name and power limit (read-only nvidia-smi query) first.  Usage:
    python scripts/amp_dtype_time.py [--rounds 3] [--steps 10]
"""
import argparse
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vit_rpe_rope_b200 import VisionTransformer, ops  # noqa: E402

VITB = dict(img_size=224, patch_size=16, in_chans=3, num_classes=1000, embed_dim=768, depth=12, num_heads=12,
            pos_encoding="rope-mixed")
VITL = dict(img_size=384, patch_size=16, in_chans=3, num_classes=1000, embed_dim=1024, depth=24, num_heads=16,
            pos_encoding="rope-axial")
KERNELS = ("attn_fwd", "attn_bwd", "qkv_rope_fwd", "fc1_fwd")


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f"nvidia-smi unavailable ({e})"


class Step:
    def __init__(self, kw, batch, size, train, dtype, scaler):
        torch.manual_seed(0)
        self.model = VisionTransformer(**kw).cuda()
        self.opt = torch.optim.AdamW(self.model.parameters(), lr=1e-4) if train else None
        self.scaler = torch.amp.GradScaler("cuda") if scaler else None
        self.train, self.dtype = train, dtype
        self.x = torch.randn(batch, 3, size, size, device="cuda")
        self.y = torch.randint(0, kw["num_classes"], (batch,), device="cuda")

    def __call__(self):
        if not self.train:
            with torch.no_grad(), torch.autocast("cuda", dtype=self.dtype):
                return self.model(self.x)
        self.opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=self.dtype):
            loss = F.cross_entropy(self.model(self.x).float(), self.y)
        if self.scaler is not None:
            self.scaler.scale(loss).backward()
            self.scaler.step(self.opt)
            self.scaler.update()
        else:
            loss.backward()
            self.opt.step()
        return loss


def time_ms(fn, steps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / steps


def kernel_us(fn):
    ops.PROFILE_EVENTS = []
    fn()
    torch.cuda.synchronize()
    acc = {}
    for name, s, e in ops.PROFILE_EVENTS:
        if name in KERNELS:
            acc[name] = acc.get(name, 0.0) + s.elapsed_time(e) * 1000.0
    ops.PROFILE_EVENTS = None
    return acc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    args = ap.parse_args()
    print("card:", card())
    dts = {"bf16": torch.bfloat16, "fp16": torch.float16}
    cases = [("vitb16-224 step", VITB, 256, 224, True, False), ("vitb16-224 step+GradScaler", VITB, 256, 224, True, True),
             ("vitl16-384 step", VITL, 64, 384, True, False), ("vitb16-512 infer", VITB, 64, 512, False, False)]
    res = {}
    for r in range(args.rounds):
        for name, kw, batch, size, train, scaler in cases:
            for tag, dt in dts.items():
                if scaler and tag == "bf16":
                    continue
                step = Step(kw, batch, size, train, dt, scaler)
                ms = time_ms(step, args.steps)
                res.setdefault((name, tag), []).append(ms)
                if name == "vitb16-224 step":
                    for k, us in kernel_us(step).items():
                        res.setdefault((f"  {k} (sum per step)", tag), []).append(us / 1000.0)
                del step
                torch.cuda.empty_cache()
        print(f"round {r + 1}/{args.rounds} done", flush=True)
    print(f"{'case':34s} {'dtype':5s} {'ms per step (each round)':>40s}")
    for (name, tag), v in res.items():
        print(f"{name:34s} {tag:5s} " + "  ".join(f"{x:9.3f}" for x in v) + f"   min {min(v):.3f}")


if __name__ == "__main__":
    main()
