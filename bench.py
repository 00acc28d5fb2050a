#!/usr/bin/env python
"""bench.py - ViT images/sec (fwd + CE + bwd + AdamW) on the B200 attention hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl ours|reference]
                    [--dump-outputs DIR]

One process per GPU (torchrun sets RANK / LOCAL_RANK / WORLD_SIZE for N > 1).  Prints ONE JSON
line on rank 0.  A "step" is the reference's training step (train.py:108-116: zero_grad -> forward
-> CrossEntropyLoss -> backward -> AdamW.step) on one synthetic batch.

Keys: ``value`` = whole-job images/s with the batch already resident in HBM; ``e2e`` = the same
metric through the public module API with pinned-host inputs copied H2D and the loss read back
every step; ``roofline`` = the fused attention forward kernel, timed per launch with CUDA events
inside the timed region, against its binding roof; ``cpu_baseline`` = the oracle port of the
reference (oracle/vit_torch.py, torch CPU fp32) timed on this box's host cores on a bounded
sample; ``clocks`` = nvidia-smi SM clock / throttle reasons sampled during the timed region.
``--impl reference`` times that CPU path alone (rank 0 only).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # a benchmark run leaves the (possibly read-only) tree as it found it

WORKLOADS = {
    # BASELINE.json configs[2]: the configuration the metric's "fused-attn % of tensor-core peak" and
    # the north_star targets are quoted on; fits one GPU.  1000 classes (free choice, SURVEY row M2).
    "vitb16-224-rope-mixed-bf16": dict(
        model=dict(img_size=224, patch_size=16, in_chans=3, num_classes=1000, embed_dim=768, depth=12,
                   num_heads=12, pos_encoding="rope-mixed"),
        batch=256, dtype="bf16", train=True, cpu_sample_batch=8),
    # configs[0] / configs[1]: ViT-Tiny fp32
    "vit-tiny-rope-axial-fp32": dict(
        model=dict(img_size=32, patch_size=4, in_chans=3, num_classes=10, embed_dim=192, depth=6, num_heads=6,
                   pos_encoding="rope-axial"),
        batch=128, dtype="f32", train=True, cpu_sample_batch=128),
    "vit-tiny-polynomial-fp32": dict(
        model=dict(img_size=32, patch_size=4, in_chans=1, num_classes=10, embed_dim=192, depth=6, num_heads=6,
                   pos_encoding="polynomial"),
        batch=128, dtype="f32", train=True, cpu_sample_batch=128),
    "vit-tiny-relative-fp32": dict(
        model=dict(img_size=32, patch_size=4, in_chans=3, num_classes=10, embed_dim=192, depth=6, num_heads=6,
                   pos_encoding="relative"),
        batch=128, dtype="f32", train=True, cpu_sample_batch=128),
    # configs[3]: ViT-L/16-384 rope-axial bf16, batch 64/GPU (BASELINE leaves it open; SURVEY row M2)
    "vitl16-384-rope-axial-bf16": dict(
        model=dict(img_size=384, patch_size=16, in_chans=3, num_classes=1000, embed_dim=1024, depth=24,
                   num_heads=16, pos_encoding="rope-axial"),
        batch=64, dtype="bf16", train=True, cpu_sample_batch=2),
    # configs[4]: ViT-B/16 built at 224, fed 512x512 (1025 tokens), inference
    "vitb16-512-rope-mixed-infer-bf16": dict(
        model=dict(img_size=224, patch_size=16, in_chans=3, num_classes=1000, embed_dim=768, depth=12,
                   num_heads=12, pos_encoding="rope-mixed"),
        batch=64, dtype="bf16", train=False, input_size=512, cpu_sample_batch=2),
}
DEFAULT_WORKLOAD = "vitb16-224-rope-mixed-bf16"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch override")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-reference-gpu", action="store_true",
                    help="skip timing the reference's eager PyTorch path (oracle port) on the same GPU")
    ap.add_argument("--attn-impl", default="auto", choices=["auto", "simt", "tcgen05"])
    ap.add_argument("--no-graph", action="store_true", help="issue the training step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (float32), for comparing builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the timed GPU path: it needs --impl ours")
    return args


# ------------------------------------------------------------------------------------------------ helpers

def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], bf16_tflops=p["bf16_tflops"],
                    bf16_tflops_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


def load_traffic():
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the hot-path kernels, taken
    from the committed `ncu --set full` capture summarised in profiles/traffic.json (keyed by workload)."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.isfile(path):
        with open(path) as f:
            return json.load(f)
    return {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (profiling recipe's clocks line)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self.stop_flag, self.thread = index, [], threading.Event(), None

    def _run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 6:
                    self.samples.append((float(f[0]), float(f[1]), f[2:6]))
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def start(self):
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def stop(self):
        self.stop_flag.set()
        if self.thread:
            self.thread.join(timeout=6)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        reasons = sorted({n for _, _, fl in self.samples for n, v in zip(self.NAMES, fl) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(s[0] for s in self.samples), "sm_max_mhz": self.samples[0][1],
                "reasons": reasons, "samples": len(self.samples)}


DUMP_ELEMENTS = 8 << 20  # float32 elements in one --dump-outputs directory (32 MB)


def dump_outputs(out_dir, train, model, runner, inf_runner):
    """What a caller of the timed step holds after its last step, as ``out_dir/<name>.npy`` in float32.
    Training: ``loss`` and every updated parameter as ``param.<name>``, a tensor larger than its even share
    of DUMP_ELEMENTS as a fixed seeded sample of its elements (same positions in every run of a workload).
    Inference: ``logits``.  The inputs are the same in every run; the training values are not bit-stable,
    because some backward reductions sum in no fixed order (include/vrr.h) and every step builds on the last,
    so compare two builds with a tolerance."""
    import numpy as np
    if train:
        arrays = {"loss": runner.static_loss}
        params = list(model.named_parameters())
        share = DUMP_ELEMENTS // len(params)
        g = torch.Generator().manual_seed(0)
        for name, p in params:
            flat = p.detach().reshape(-1)
            if flat.numel() > share:
                flat = flat[torch.randperm(flat.numel(), generator=g)[:share].sort().values.to(flat.device)]
            arrays["param." + name] = flat
    else:
        arrays = {"logits": inf_runner.static_out}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def attn_algorithmic(model_cfg, tokens):
    """Per image, per layer (BASELINE.md section 4): fwd flops 4*N^2*E; min bytes (bf16) 8*N*E + 4*H*N."""
    e, h = model_cfg["embed_dim"], model_cfg["num_heads"]
    return 4.0 * tokens * tokens * e, 8.0 * tokens * e + 4.0 * h * tokens


def model_flops_per_image(model_cfg, tokens, train):
    e, depth, p, c = model_cfg["embed_dim"], model_cfg["depth"], model_cfg["patch_size"], model_cfg["in_chans"]
    fwd = depth * (24.0 * tokens * e * e + 4.0 * tokens * tokens * e) + 2.0 * (tokens - 1) * c * p * p * e \
        + 2.0 * e * model_cfg["num_classes"]
    return fwd * (3.0 if train else 1.0)


# ------------------------------------------------------------------------------------------------ CPU arm

def cpu_reference_run(wl, steps, warmup):
    """The reference's CPU path (oracle port, torch fp32, all host threads) on a bounded sample."""
    from oracle import vit_torch as V
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    cfg = V.VitConfig(**wl["model"])
    bs = wl["cpu_sample_batch"]
    size = wl.get("input_size", cfg.img_size)
    params = V.params_from_state_dict(V.init_state_dict(cfg, seed=0), requires_grad=wl["train"])
    g = torch.Generator().manual_seed(0)
    images = torch.randn(bs, cfg.in_chans, size, size, generator=g)
    labels = torch.randint(0, cfg.num_classes, (bs,), generator=g)
    opt = torch.optim.AdamW([p for p in params.values() if p.requires_grad], lr=1e-3, weight_decay=0.01) \
        if wl["train"] else None

    def step():
        if wl["train"]:
            V.train_step(cfg, params, opt, images, labels)
        else:
            with torch.no_grad():
                V.forward(cfg, params, images)

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return dict(value=bs * steps / dt, unit="images/s", cores=threads, kind="port",
                sample=f"{steps} steps of batch {bs} (of the workload's {wl['batch']}/GPU), fp32, "
                       f"torch {torch.__version__} CPU, {threads} threads"), dt / steps * 1e3


def gpu_reference_run(wl, batch, dev, steps, warmup):
    """The reference's own eager PyTorch path (oracle port: the same torch ops in the same order) on THIS
    GPU at the workload's full batch and dtype (bf16 = torch.autocast, fp32 master weights) - the bar a
    user of the reference on a B200 would see (train.py:108-116 with device='cuda').  A baseline like
    cpu_baseline: reported, never on the product path."""
    from oracle import vit_torch as V
    cfg = V.VitConfig(**wl["model"])
    size = wl.get("input_size", cfg.img_size)
    bf16 = wl["dtype"] == "bf16"
    try:
        params = V.params_from_state_dict(V.init_state_dict(cfg, seed=0), requires_grad=wl["train"], device=dev)
        g = torch.Generator().manual_seed(0)
        images = torch.randn(batch, cfg.in_chans, size, size, generator=g).to(dev)
        labels = torch.randint(0, cfg.num_classes, (batch,), generator=g).to(dev)
        opt = torch.optim.AdamW([p for p in params.values() if p.requires_grad], lr=1e-3, weight_decay=0.01, fused=True) \
            if wl["train"] else None

        def step():
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=bf16):
                if wl["train"]:
                    opt.zero_grad()
                    loss = F.cross_entropy(V.forward(cfg, params, images).float(), labels)
                    loss.backward()
                    opt.step()
                else:
                    with torch.no_grad():
                        V.forward(cfg, params, images)

        for _ in range(warmup):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        return {"value": batch / (ms / 1e3), "unit": "images/s", "ms_per_step": ms, "batch": batch, "steps": steps,
                "kind": "port of the reference's eager path (oracle/vit_torch.py) on the same B200, "
                        + ("bf16 autocast" if bf16 else "fp32 (TF32 off)") + ", eager launches, torch " + torch.__version__}
    except torch.OutOfMemoryError as e:  # pragma: no cover
        return {"unavailable": f"out of memory at batch {batch}: {str(e)[:80]}"}


def run_reference_arm(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = max(1, min(args.steps, 5)), max(1, min(args.warmup, 2))
    cb, ms = cpu_reference_run(wl, steps, warmup)
    line = {"impl": "reference", "metric": "ViT images/sec fwd+bwd", "value": cb["value"], "unit": "images/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, **wl["model"], "batch_per_step": wl["cpu_sample_batch"],
                       "train": wl["train"]},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm

def main():
    args = parse_args()
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference_arm(args, wl)
        return

    import torch.distributed as dist
    from vit_rpe_rope_b200 import VisionTransformer, _lib, ops
    from vit_rpe_rope_b200.dp import BucketedDataParallel
    from vit_rpe_rope_b200.runtime import GraphedInference, GraphedTrainStep

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # The step (incl. the bucketed NCCL all-reduces) is captured into one CUDA graph at every world size.
    # Round 1's multi-rank captures worked; what stalled was process-group teardown with the graph still
    # alive - see teardown() below.
    use_graph = not args.no_graph
    if world > 1:
        import datetime
        import faulthandler
        import signal
        faulthandler.enable()
        signal.signal(signal.SIGALRM, lambda *_: (sys.stderr.write(
            "bench.py: multi-rank run made no progress for 300 s - aborting instead of hanging\n"), os._exit(3)))
        signal.alarm(300)
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=120))
    _lib.load()
    _lib.set_impl({"auto": _lib.IMPL_AUTO, "simt": _lib.IMPL_SIMT, "tcgen05": _lib.IMPL_TCGEN05}[args.attn_impl])
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False

    mcfg = wl["model"]
    batch = args.batch or wl["batch"]
    size = wl.get("input_size", mcfg["img_size"])
    tokens = (size // mcfg["patch_size"]) ** 2 + 1
    bf16 = wl["dtype"] == "bf16"
    torch.manual_seed(0)
    model = VisionTransformer(**mcfg).to(dev)
    train = wl["train"]
    dp = BucketedDataParallel(model, bucket_mb=32.0) if train else None
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3, weight_decay=0.01, fused=True, capturable=use_graph) \
        if train else None
    if not train:
        model.eval()

    g = torch.Generator().manual_seed(1234 + rank)
    host_images = torch.randn(batch, mcfg["in_chans"], size, size, generator=g).pin_memory()
    host_labels = torch.randint(0, mcfg["num_classes"], (batch,), generator=g).pin_memory()
    dev_images, dev_labels = host_images.to(dev), host_labels.to(dev)

    runner = None
    if train:
        runner = GraphedTrainStep(dp, opt, tuple(host_images.shape), mcfg["num_classes"], dev, bf16=bf16,
                                  use_graph=use_graph, warmup=max(3, args.warmup))
        runner.prepare(dev_images, dev_labels)

    inf_runner = None
    if not train:
        inf_runner = GraphedInference(model, tuple(host_images.shape), dev, bf16=bf16, use_graph=use_graph,
                                      warmup=max(3, args.warmup))

    def infer(images):
        return inf_runner.run(images)

    def infer_eager(images):
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16, enabled=bf16):
            return model(images)

    if inf_runner is not None:
        inf_runner.static_images.copy_(dev_images)  # `value`: the batch is already where the captured forward reads it

    def step_resident():
        return runner.run() if train else inf_runner.run()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    for _ in range(args.warmup):
        step_resident()

    # ---- timed region 1: device-resident inputs -> `value`
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    launches0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step_resident()
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if use_graph:
        gpu_launches = (runner.launches_per_step if train else inf_runner.launches_per_step) * args.steps
    else:
        gpu_launches = _lib.launch_count() - launches0
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    if args.dump_outputs and rank == 0:  # before the passes below step the model further
        dump_outputs(args.dump_outputs, train, model, runner, inf_runner)

    # ---- per-launch kernel timing (CUDA events on the launching stream) -> `roofline`.  A graph replay has
    # no host-side launch sites, so the same K steps are issued eagerly once more with events around
    # every libvrr launch; the kernels and their inputs are identical to the timed region's.
    ops.PROFILE_EVENTS = []
    for _ in range(args.steps):
        runner._eager_step() if train else infer_eager(dev_images)
    torch.cuda.synchronize()
    events, ops.PROFILE_EVENTS = ops.PROFILE_EVENTS, None
    kernel_ms = {}
    for name, a, b in events:
        kernel_ms.setdefault(name, []).append(a.elapsed_time(b))

    # ---- timed region 2: end to end through the public API with pinned-host inputs -> `e2e`.
    # Every step copies its batch H2D from pinned memory and its loss / logits D2H, all inside the timed
    # region; the copies run on a side stream one batch ahead (runtime.GraphedTrainStep.feed / step_fed)
    # so they overlap the previous step instead of serialising with it.
    if train:
        def e2e_loop(n):
            runner.feed(host_images, host_labels)
            last_ = None
            for i in range(n):
                if i + 1 < n:
                    runner.feed(host_images, host_labels)      # batch i+1 travels while step i runs
                last_ = runner.step_fed()                      # returns the loss of step i-1 (already on the host)
            return runner.last_loss()                          # the final step's loss: read inside the region
    else:
        copy_stream = torch.cuda.Stream(device=dev)
        stage = [torch.empty_like(dev_images) for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        free = [torch.cuda.Event() for _ in range(2)]
        host_out = torch.zeros(2, batch, mcfg["num_classes"], dtype=torch.float32).pin_memory()
        out_ev = [torch.cuda.Event() for _ in range(2)]

        def feed_inf(i):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(free[i & 1])
                stage[i & 1].copy_(host_images, non_blocking=True)
                ready[i & 1].record(copy_stream)

        def e2e_loop(n):
            cur = torch.cuda.current_stream()
            for ev in free:
                ev.record(cur)
            feed_inf(0)
            for i in range(n):
                if i + 1 < n:
                    feed_inf(i + 1)
                cur.wait_event(ready[i & 1])
                o = infer(stage[i & 1])
                free[i & 1].record(cur)
                if i >= 2:
                    out_ev[i & 1].synchronize()
                host_out[i & 1].copy_(o.float(), non_blocking=True)
                out_ev[i & 1].record(cur)
            out_ev[(n - 1) & 1].synchronize()
            return float(host_out[(n - 1) & 1][0, 0])

    e2e_loop(2)
    barrier()
    e0.record()
    last = e2e_loop(args.steps)
    e1.record()
    barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    h2d = host_images.numel() * host_images.element_size() + host_labels.numel() * host_labels.element_size()
    out = None if train else infer(dev_images)

    def teardown():
        """Drop the captured graph (it references NCCL work) BEFORE the process group goes: round 1's
        multi-rank runs had printed their result and then stalled inside destroy_process_group()."""
        if runner is not None:
            runner.close()
        if inf_runner is not None:
            inf_runner.close()
        if world > 1:
            import signal
            sys.stdout.flush()
            signal.signal(signal.SIGALRM, lambda *_: os._exit(0))  # result is already printed: never hang at exit
            signal.alarm(30)
            torch.cuda.synchronize()
            dist.barrier()
            dist.destroy_process_group()
            signal.alarm(0)

    if world > 1:
        import signal
        signal.alarm(0)
    if rank != 0:
        teardown()
        return

    peaks = load_peaks()
    value = world * batch * args.steps / (ms_total / 1e3)
    e2e_value = world * batch * args.steps / (ms_e2e / 1e3)
    # ---- rooflines of the hot-path kernels.  Algorithmic work per launch (SURVEY.md section 8 row M4, DESIGN.md
    # section 5): attention core fwd 4*N^2*E flop and 8*N*E + 4*H*N bytes (bf16) per image, bwd twice that;
    # QKV projection 6*N*E^2 flop per image.  `roofline` (the contract key) is the DOMINANT hot-path kernel
    # (largest share of the step); the others are listed under `rooflines`.
    flops_img, bytes_img = attn_algorithmic(mcfg, tokens)
    traffic_tab = load_traffic().get(args.workload, {})
    ridge = peaks["bf16_tflops_sustained"] * 1e3 / peaks["hbm_gbs"]
    esz = 1.0 if bf16 else 2.0
    algo = {"attn_fwd": (flops_img * batch, bytes_img * batch * esz),
            "attn_bwd": (2 * flops_img * batch, 2 * bytes_img * batch * esz)}
    e_, n_ = mcfg["embed_dim"], tokens
    algo["qkv_rope_fwd"] = (6.0 * n_ * e_ * e_ * batch, (n_ * e_ + 3 * e_ * e_ / batch + 3 * n_ * e_) * 2.0 * esz * batch)
    rooflines, extra = {}, {}
    for name, arr in kernel_ms.items():
        avg_ms = statistics.mean(arr)
        extra[name] = {"avg_launch_ms": avg_ms, "launches": len(arr), "share_of_step": avg_ms * len(arr) / args.steps / (ms_total / args.steps)}
        if name not in algo:
            continue
        flops, byts = algo[name]
        tf, gbs = flops / avg_ms / 1e9, byts / avg_ms / 1e6
        if flops / byts < ridge or not bf16:
            r = {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"]}
        else:
            r = {"bound": "tensor", "achieved": tf, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                 "frac": tf / peaks["bf16_tflops_sustained"]}
        r.update({"traffic": traffic_tab.get(name), "kernel": "vrr_" + name,
                  "timed": "CUDA events around every launch, eager re-issue of the same K steps",
                  "avg_launch_ms": avg_ms, "launches_timed": len(arr), "algorithmic_flops_per_launch": flops,
                  "algorithmic_bytes_per_launch": byts, "tflops": tf,
                  "frac_of_bf16_sustained_peak": tf / peaks["bf16_tflops_sustained"],
                  "frac_of_bf16_burst_peak": tf / peaks["bf16_tflops"],
                  "peak_source": peaks["source"] + ": HBM copy bandwidth; bf16 sustained figure (kernel timed inside a long step)",
                  "traffic_source": traffic_tab.get("_source")})
        rooflines[name] = r
    roofline = None
    if rooflines:
        dominant = max(rooflines, key=lambda k: extra[k]["share_of_step"])
        roofline = rooflines[dominant]
    step_tflops = model_flops_per_image(mcfg, tokens, train) * value / 1e12

    cpu_baseline = None
    reference_gpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu_baseline, _ = cpu_reference_run(wl, steps=3, warmup=1)
    if world == 1 and not args.no_reference_gpu:
        if runner is not None:
            runner.close()
            runner = None
        del dp, opt, model
        torch.cuda.empty_cache()
        reference_gpu = gpu_reference_run(wl, batch, dev, steps=min(args.steps, 5), warmup=2)

    line = {
        "metric": "ViT images/sec fwd+bwd", "value": value, "unit": "images/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": wl["dtype"], "data": "synthetic",
        "config": {"workload": args.workload, **mcfg, "tokens": tokens, "batch_per_gpu": batch,
                   "global_batch": batch * world, "train": train, "optimizer": "AdamW(lr=1e-3, wd=0.01)" if train else None,
                   "parallelism": f"dp{world}", "l2": "inputs+activations per step exceed the 126 MB L2 (no flush needed)",
                   "attn_impl": args.attn_impl, "cuda_graph": bool(use_graph)},
        "e2e": {"value": e2e_value, "unit": "images/s", "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4 if train else int(out.numel() * 4)},
        "gpu_launches": int(gpu_launches),
        "roofline": roofline, "rooflines": rooflines, "hot_path_kernels": extra, "model_tflops": step_tflops,
        "mfu_vs_bf16_sustained": step_tflops / (world * peaks["bf16_tflops_sustained"]) if bf16 else None,
        "cpu_baseline": cpu_baseline, "reference_gpu": reference_gpu, "clocks": clocks, "last_result": last,
    }
    print(json.dumps(line), flush=True)
    teardown()


if __name__ == "__main__":
    main()
