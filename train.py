"""Training entry point with the command line, log and checkpoint conventions of the reference's ``train.py``
(/root/reference/train.py:20-56 arguments, :167-171 CSV header, :199-213 best-checkpoint + per-epoch row), running the
B200 kernels of this repository through the drop-in ``VisionTransformer``.

Same flags and defaults; same files: ``<log_dir>/<dataset>_<pos_encoding>_<timestamp>.csv`` with the columns
``epoch, train_loss, train_acc, test_loss, test_acc, best_acc`` and ``<ckpt_dir>/<dataset>_<pos_encoding>_best.pth``
holding ``model.state_dict()`` (loadable by the reference and vice versa: the key layout is the reference's, see
tests/test_host_api.py).  Same loop: AdamW(lr, weight_decay), CosineAnnealingLR(T_max = epochs), CrossEntropyLoss.

Additions (all off by default, so a reference command line behaves like the reference):
  --amp bf16         run the step under torch.autocast(bfloat16) - the tcgen05 kernels (head dim 64)
  --amp fp16         run the step under torch.autocast(float16) with torch.amp.GradScaler (loss scaling; a step whose
                     gradients overflow is skipped and the scale lowered) - the same kernels in fp16
  --synthetic        class-conditional synthetic images instead of MNIST / CIFAR-10.  Chosen automatically when the
                     dataset is not on disk: this repository never downloads anything.
  --max_steps N      stop every epoch after N batches (smoke runs)
  --drop_rate P      dropout on every block's attention projection and Mlp (timm's drop_rate)
  --drop_path_rate P stochastic depth, linearly from 0 at the first block to P at the last (timm's drop_path_rate)
  --reg_tokens R     R register tokens after the cls token (timm's reg_tokens; not with relative / polynomial)
  --init_values V    LayerScale in every block, gamma initialised to V (timm's init_values, e.g. 1e-5 as in DeiT III)
  --mlp_layer swiglu every block's MLP is timm's SwiGLUPacked (fc2(silu(x W_g + b_g) * (x W_v + b_v))) instead of Mlp
  --qk_norm          QK-norm in every attention: LayerNorm of each q / k head row before RoPE (timm's qk_norm)
  --mlp_ratio R      fc1's width over embed_dim (default 4; 5.33334 gives a SwiGLU MLP the GELU MLP's parameters)
There is no CPU path: a CUDA sm_100 device is required.
"""
import argparse
import csv
import os
import sys
import time
from datetime import datetime

import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from vit_rpe_rope_b200.models.vit import Mlp, SwiGLUPacked, VisionTransformer  # noqa: E402

MODES = ["none", "absolute", "relative", "polynomial", "rope-axial", "rope-mixed"]


def get_args(argv=None):
    p = argparse.ArgumentParser(description="Vision Transformer Training (B200 kernels)")
    p.add_argument("--log_dir", type=str, default="logs")
    p.add_argument("--ckpt_dir", type=str, default="checkpoints")
    p.add_argument("--dataset", type=str, default="mnist", choices=["mnist", "cifar10"])
    p.add_argument("--pos_encoding", type=str, default="absolute", choices=MODES)
    p.add_argument("--rope_theta", type=float, default=100.0)
    p.add_argument("--poly_degree", type=int, default=3)
    p.add_argument("--poly_shared_heads", action="store_true", default=True)
    p.add_argument("--no-poly_shared_heads", action="store_false", dest="poly_shared_heads")
    p.add_argument("--batch_size", type=int, default=128)
    p.add_argument("--epochs", type=int, default=25)
    p.add_argument("--lr", type=float, default=0.001)
    p.add_argument("--weight_decay", type=float, default=0.01)
    p.add_argument("--img_size", type=int, default=32)
    p.add_argument("--patch_size", type=int, default=4)
    p.add_argument("--embed_dim", type=int, default=192)
    p.add_argument("--depth", type=int, default=6)
    p.add_argument("--num_heads", type=int, default=6)
    # additions
    p.add_argument("--amp", type=str, default="none", choices=["none", "bf16", "fp16"])
    p.add_argument("--synthetic", action="store_true")
    p.add_argument("--synthetic_size", type=int, default=4096, help="training images of the synthetic set")
    p.add_argument("--max_steps", type=int, default=0)
    p.add_argument("--data_root", type=str, default="./data")
    p.add_argument("--seed", type=int, default=0)
    p.add_argument("--drop_rate", type=float, default=0.0, help="proj / Mlp dropout of every block")
    p.add_argument("--drop_path_rate", type=float, default=0.0,
                   help="stochastic depth of the last block (linearly from 0 over the depth, timm's rule)")
    p.add_argument("--reg_tokens", type=int, default=0, help="register tokens after the cls token")
    p.add_argument("--init_values", type=float, default=None, help="LayerScale initial value (default: no LayerScale)")
    p.add_argument("--mlp_layer", type=str, default="mlp", choices=["mlp", "swiglu"], help="Mlp (GELU) or SwiGLUPacked")
    p.add_argument("--qk_norm", action="store_true", help="LayerNorm of each q / k head row before RoPE")
    p.add_argument("--mlp_ratio", type=float, default=4.0, help="fc1 width / embed_dim")
    return p.parse_args(argv)


class SyntheticImages(torch.utils.data.Dataset):
    """Ten fixed random class templates plus noise: learnable, deterministic, needs no files."""

    def __init__(self, n, chans, size, num_classes=10, seed=0):
        g = torch.Generator().manual_seed(seed)
        self.templates = torch.randn(num_classes, chans, size, size, generator=torch.Generator().manual_seed(1234))
        self.labels = torch.randint(0, num_classes, (n,), generator=g)
        self.noise = torch.randn(n, chans, size, size, generator=g)

    def __len__(self):
        return self.labels.numel()

    def __getitem__(self, i):
        y = int(self.labels[i])
        return self.templates[y] + 0.7 * self.noise[i], y


def get_dataset(args):
    """(train_loader, test_loader, num_classes, in_chans); MNIST is 1 x HxW, CIFAR-10 3 x HxW, both resized to img_size."""
    in_chans = 1 if args.dataset == "mnist" else 3
    train_set = test_set = None
    if not args.synthetic:
        try:
            from torchvision import datasets, transforms
            norm = ((0.1307,), (0.3081,)) if args.dataset == "mnist" else ((0.4914, 0.4822, 0.4465), (0.2023, 0.1994, 0.2010))
            tf = transforms.Compose([transforms.Resize(args.img_size), transforms.ToTensor(), transforms.Normalize(*norm)])
            cls = datasets.MNIST if args.dataset == "mnist" else datasets.CIFAR10
            train_set = cls(root=args.data_root, train=True, download=False, transform=tf)
            test_set = cls(root=args.data_root, train=False, download=False, transform=tf)
        except Exception as e:  # not on disk (or no torchvision): never download
            print(f"[train.py] {args.dataset} not available under {args.data_root} ({type(e).__name__}); using --synthetic data")
    if train_set is None:
        train_set = SyntheticImages(args.synthetic_size, in_chans, args.img_size, seed=args.seed)
        test_set = SyntheticImages(max(args.synthetic_size // 4, args.batch_size), in_chans, args.img_size, seed=args.seed + 1)
    mk = lambda ds, shuffle: torch.utils.data.DataLoader(ds, batch_size=args.batch_size, shuffle=shuffle, num_workers=0,
                                                         pin_memory=True, drop_last=False)
    return mk(train_set, True), mk(test_set, False), 10, in_chans


def run_epoch(model, loader, criterion, optimizer, device, amp, max_steps, amp_dtype=torch.bfloat16, scaler=None):
    """One pass; trains when ``optimizer`` is given.  Returns (mean batch loss, accuracy %) like the reference's
    train() / test() (train.py:97-155); the loss / accuracy counters stay on the device until the end of the pass.
    ``amp``: autocast to ``amp_dtype``; ``scaler``: a torch.amp.GradScaler for the backward and the optimizer step."""
    training = optimizer is not None
    model.train(training)
    loss_sum = torch.zeros((), device=device)
    correct = torch.zeros((), device=device, dtype=torch.long)
    total, batches = 0, 0
    with torch.set_grad_enabled(training):
        for images, labels in loader:
            images, labels = images.to(device, non_blocking=True), labels.to(device, non_blocking=True)
            if training:
                optimizer.zero_grad()
            with torch.autocast("cuda", dtype=amp_dtype, enabled=amp):
                outputs = model(images)
                loss = criterion(outputs.float(), labels)
            if training and scaler is not None:
                scaler.scale(loss).backward()
                scaler.step(optimizer)
                scaler.update()
            elif training:
                loss.backward()
                optimizer.step()
            loss_sum += loss.detach()
            correct += (outputs.argmax(1) == labels).sum()
            total += labels.numel()
            batches += 1
            if max_steps and batches >= max_steps:
                break
    return float(loss_sum) / max(batches, 1), 100.0 * int(correct) / max(total, 1)


def main(argv=None):
    args = get_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("train.py: a CUDA sm_100 device is required (this implementation has no CPU path)")
    device = torch.device("cuda")
    torch.manual_seed(args.seed)
    os.makedirs(args.log_dir, exist_ok=True)
    os.makedirs(args.ckpt_dir, exist_ok=True)
    stamp = datetime.now().strftime("%Y%m%d_%H%M%S")
    log_file = os.path.join(args.log_dir, f"{args.dataset}_{args.pos_encoding}_{stamp}.csv")
    with open(log_file, "w", newline="") as f:
        csv.writer(f).writerow(["epoch", "train_loss", "train_acc", "test_loss", "test_acc", "best_acc"])
    train_loader, test_loader, num_classes, in_chans = get_dataset(args)
    model = VisionTransformer(img_size=args.img_size, patch_size=args.patch_size, in_chans=in_chans, num_classes=num_classes,
                              embed_dim=args.embed_dim, depth=args.depth, num_heads=args.num_heads,
                              pos_encoding=args.pos_encoding, rope_theta=args.rope_theta, poly_degree=args.poly_degree,
                              poly_shared_heads=args.poly_shared_heads, drop_rate=args.drop_rate,
                              drop_path_rate=args.drop_path_rate, reg_tokens=args.reg_tokens,
                              init_values=args.init_values, mlp_ratio=args.mlp_ratio,
                              mlp_layer=SwiGLUPacked if args.mlp_layer == "swiglu" else Mlp,
                              qk_norm=args.qk_norm).to(device)
    criterion = nn.CrossEntropyLoss()
    optimizer = torch.optim.AdamW(model.parameters(), lr=args.lr, weight_decay=args.weight_decay)
    scheduler = torch.optim.lr_scheduler.CosineAnnealingLR(optimizer, T_max=args.epochs)
    amp = args.amp != "none"
    amp_dtype = torch.float16 if args.amp == "fp16" else torch.bfloat16
    scaler = torch.amp.GradScaler("cuda") if args.amp == "fp16" else None
    best_acc, ckpt = 0.0, os.path.join(args.ckpt_dir, f"{args.dataset}_{args.pos_encoding}_best.pth")
    for epoch in range(args.epochs):
        t0 = time.time()
        train_loss, train_acc = run_epoch(model, train_loader, criterion, optimizer, device, amp, args.max_steps, amp_dtype,
                                          scaler)
        test_loss, test_acc = run_epoch(model, test_loader, criterion, None, device, amp, args.max_steps, amp_dtype)
        scheduler.step()
        if test_acc > best_acc:
            best_acc = test_acc
            torch.save(model.state_dict(), ckpt)
        with open(log_file, "a", newline="") as f:
            csv.writer(f).writerow([epoch + 1, train_loss, train_acc, test_loss, test_acc, best_acc])
        print(f"Epoch {epoch + 1}/{args.epochs}: train loss {train_loss:.4f} acc {train_acc:.2f}% | test loss {test_loss:.4f} "
              f"acc {test_acc:.2f}% | best {best_acc:.2f}% | {time.time() - t0:.1f} s")
    return log_file, ckpt


if __name__ == "__main__":
    main()
