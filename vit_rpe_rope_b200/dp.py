"""Batch data-parallel training for the ViT hot path: one process per GPU, one NCCL communicator,
gradients all-reduced in flat buckets that overlap with the rest of backward (SURVEY.md row G1).

The reference has no multi-GPU code; images are independent units, so forward/backward need no
exchange and the single collective is the gradient mean before ``optimizer.step``.  Design:

* parameters are grouped into flat fp32 buckets (~``bucket_mb`` each) in *reverse registration
  order* - the order backward produces their gradients; parameters whose gradient only completes
  at the very end of backward (the shared PE parameter that every block feeds, the cls and
  register tokens, the patch projection, an absolute table) go into the last bucket;
* default (``dp.zero_grad()``): ``param.grad`` is dropped, autograd then ADOPTS the gradient tensors the backward
  kernels produce (no ``grad += dW`` pass, no zero-fill of 345 MB per step: ~220 small ATen launches and ~0.9 ms of
  a 38 ms ViT-B step); when the last parameter of a bucket has its gradient, ONE multi-tensor copy gathers them
  into the flat bucket and ``param.grad`` is re-bound to the bucket slices (world size 1: nothing is copied at
  all).  ``dp.zero_grad(set_to_none=False)`` keeps the other style: ``param.grad`` stays a view into its (zeroed)
  bucket and gradients accumulate straight into bucket memory;
* a post-accumulate hook marks a parameter as seen for this step; when the last parameter of a
  bucket has been seen the bucket is all-reduced asynchronously with ``ReduceOp.AVG`` (NCCL runs it
  on its own stream, behind an event on the compute stream) while backward keeps computing earlier
  layers.  Backends without AVG (gloo, the CPU tests) pre-scale by 1/world and SUM;
* ``sync()`` (called before the optimizer step) makes the compute stream wait for the collectives
  and re-arms the buckets for the next step.

Works with any zeroing style, including the reference loop's ``optimizer.zero_grad()`` (train.py:111): whatever
``p.grad`` is when its bucket completes - bucket slice or a tensor of autograd's - ends up in the bucket before the
collective.  Gradient accumulation over several backwards: wrap all but the
last one in ``with dp.no_sync():``.

Works unchanged on CPU tensors with the ``gloo`` backend (tests/test_dp_gloo.py, world_size 2).
"""
import contextlib
from typing import List

import torch
import torch.distributed as dist


class _Bucket:
    def __init__(self, params, device, dtype):
        self.params = params
        self.numel = sum(p.numel() for p in params)
        self.flat = torch.zeros(self.numel, device=device, dtype=dtype)
        self.views = {}
        self.seen = set()
        self.work = None
        self.reduced = False
        off = 0
        for p in params:
            v = self.flat[off:off + p.numel()].view_as(p)
            self.views[id(p)] = v
            p.grad = v
            off += p.numel()


class BucketedDataParallel(torch.nn.Module):
    def __init__(self, module: torch.nn.Module, bucket_mb: float = 32.0, process_group=None,
                 broadcast_from_rank0: bool = True):
        super().__init__()
        self.module = module
        self.group = process_group
        self.world = dist.get_world_size(process_group) if dist.is_initialized() else 1
        backend = dist.get_backend(process_group) if dist.is_initialized() else ""
        self._use_avg = str(backend).lower() == "nccl"
        self._sync_enabled = True
        params = [p for p in module.parameters() if p.requires_grad]
        if not params:
            raise ValueError("module has no trainable parameters")
        if broadcast_from_rank0 and self.world > 1:
            for t in list(module.parameters()) + list(module.buffers()):
                dist.broadcast(t.data, src=0, group=process_group)
        late_ids = self._late_parameter_ids(module)
        early = [p for p in reversed(params) if id(p) not in late_ids]
        late = [p for p in reversed(params) if id(p) in late_ids]
        cap = int(bucket_mb * (1 << 20) / 4)
        self.buckets: List[_Bucket] = []
        for group in self._split(early, cap) + ([late] if late else []):
            self.buckets.append(_Bucket(group, group[0].device, group[0].dtype))
        self._bucket_of = {}
        for b in self.buckets:
            for p in b.params:
                self._bucket_of[id(p)] = b
                p.register_post_accumulate_grad_hook(self._on_grad)
        self.allreduce_bytes = sum(b.numel for b in self.buckets) * 4

    @staticmethod
    def _late_parameter_ids(module):
        """Parameters whose gradient is complete only when backward reaches the stem."""
        late = set()
        for name, p in module.named_parameters():
            if name.startswith(("pos_embed.", "patch_embed.")) or name in ("cls_token", "reg_token"):
                late.add(id(p))
        return late

    @staticmethod
    def _split(params, cap):
        groups, cur, size = [], [], 0
        for p in params:
            if cur and (size + p.numel() > cap or p.dtype != cur[0].dtype):
                groups.append(cur)
                cur, size = [], 0
            cur.append(p)
            size += p.numel()
        if cur:
            groups.append(cur)
        return groups

    def _on_grad(self, p):
        b = self._bucket_of[id(p)]
        if b.reduced:
            raise RuntimeError("a gradient arrived for a bucket that was already all-reduced in this step; "
                               "wrap all but the last backward of an accumulation step in dp.no_sync()")
        if not self._sync_enabled:
            return
        b.seen.add(id(p))
        if len(b.seen) == len(b.params):
            self._launch(b)

    def _launch(self, b):
        b.reduced = True
        if self.world <= 1:
            return  # single process: the gradients stay wherever autograd put them
        # gather the gradients that are not (any more) slices of the flat bucket: one multi-tensor copy
        src, dst = [], []
        for p in b.params:
            v = b.views[id(p)]
            if p.grad.data_ptr() != v.data_ptr() or p.grad.dtype != v.dtype:
                src.append(p.grad if p.grad.dtype == v.dtype else p.grad.to(v.dtype))
                dst.append(v)
        if src:
            torch._foreach_copy_(dst, src)
            for p in b.params:
                p.grad = b.views[id(p)]
        if self._use_avg:
            b.work = dist.all_reduce(b.flat, op=dist.ReduceOp.AVG, group=self.group, async_op=True)
        else:
            b.flat.mul_(1.0 / self.world)
            b.work = dist.all_reduce(b.flat, op=dist.ReduceOp.SUM, group=self.group, async_op=True)

    @contextlib.contextmanager
    def no_sync(self):
        """Backwards inside this context only accumulate locally (gradient accumulation)."""
        prev, self._sync_enabled = self._sync_enabled, False
        try:
            yield
        finally:
            self._sync_enabled = prev

    def forward(self, *args, **kwargs):
        return self.module(*args, **kwargs)

    def zero_grad(self, set_to_none: bool = True):
        """``set_to_none=True`` (default): drop the gradients - autograd adopts the tensors the next backward produces.
        ``False``: zero the flat buckets in place and keep ``param.grad`` bound to their slices."""
        for b in self.buckets:
            if set_to_none:
                for p in b.params:
                    p.grad = None
            else:
                b.flat.zero_()
                for p in b.params:
                    if p.grad is None or p.grad.data_ptr() != b.views[id(p)].data_ptr():
                        p.grad = b.views[id(p)]
            self._rearm(b)

    @staticmethod
    def _rearm(b):
        b.seen.clear()
        b.work = None
        b.reduced = False

    def sync(self):
        """Wait for every bucket's all-reduce (call after ``backward``, before ``optimizer.step``) and
        re-arm the buckets for the next step."""
        missing = [b for b in self.buckets if not b.reduced]
        if missing and self.world > 1:
            names = {id(p): n for n, p in self.module.named_parameters()}
            absent = [names.get(id(p), "?") for b in missing for p in b.params if id(p) not in b.seen]
            raise RuntimeError(f"{len(missing)} gradient bucket(s) were never all-reduced: no gradient reached "
                               f"{absent[:6]}{'...' if len(absent) > 6 else ''} in this step (unused parameter, or "
                               "every backward of the step ran under no_sync())")
        for b in self.buckets:
            if b.work is not None:
                b.work.wait()
            self._rearm(b)
