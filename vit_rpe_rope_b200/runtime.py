"""Training-step runner: the whole step (zero_grad -> forward -> loss -> backward -> all-reduce ->
AdamW) captured once into a CUDA graph and replayed; host batches are prefetched on a copy stream.

The reference's step (train.py:108-116) is ~900 kernel launches for ViT-B/16; issued eagerly from
Python they leave the GPU idle a few % of the step.  B200-first: no tracing compiler - the eager step,
which already runs the hand-written kernels through the C ABI on the current stream, is captured with
``torch.cuda.graph`` (kernel parameters incl. the TMA tensor maps are baked into the graph; every
buffer lives in the graph's private pool, the gradient buckets of ``BucketedDataParallel`` are
persistent) and replayed with one launch.  The bucketed NCCL all-reduces are captured with it (the
collectives become graph nodes on NCCL's stream), so the same graph serves 1..8 ranks.

End-to-end path (``feed`` / ``step_fed``): batch t+1 travels host -> device on a side stream into one
of two staging buffers while step t runs; at the start of step t+1 a device-to-device copy moves it into
the graph's static input buffers (0.1 ms for a 154 MB batch) and the loss of step t is copied to pinned
host memory asynchronously and read one step later - the H2D copy (2.8 ms over PCIe 5) and the loss
read-back no longer serialise with the 44 ms step.

Teardown (``close``): a captured graph keeps NCCL work objects alive; destroying the process group
while it exists stalled round 1's multi-GPU runs at exit.  ``close()`` drops the graph, synchronises
and only then may the caller destroy the process group.
"""
import torch
import torch.nn.functional as F

from . import _lib
from .dp import BucketedDataParallel


class GraphedTrainStep:
    def __init__(self, dp: BucketedDataParallel, optimizer: torch.optim.Optimizer, images_shape, num_classes,
                 device, bf16: bool = True, use_graph: bool = True, warmup: int = 3):
        self.dp, self.opt, self.bf16, self.device = dp, optimizer, bf16, device
        self.static_images = torch.zeros(images_shape, device=device, dtype=torch.float32)
        self.static_labels = torch.zeros(images_shape[0], device=device, dtype=torch.long)
        self.static_loss = torch.zeros((), device=device, dtype=torch.float32)
        self.num_classes = num_classes
        self.graph = None
        self.launches_per_step = 0
        self._warmup = warmup
        self._use_graph = use_graph
        # end-to-end feeding: two staging slots filled by the copy stream
        self._copy_stream = None
        self._stage = None
        self._flip_in = 0   # next slot the copy stream fills
        self._flip_out = 0  # next slot the compute stream consumes
        self._host_loss = None
        self._loss_events = None
        self._steps_fed = 0

    def _eager_step(self):
        self.dp.zero_grad()
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=self.bf16):
            logits = self.dp(self.static_images)
            loss = F.cross_entropy(logits.float(), self.static_labels)
        loss.backward()
        self.dp.sync()
        self.opt.step()
        self.static_loss.copy_(loss.detach())

    def prepare(self, images, labels):
        """Warm up (allocator, cuBLAS workspaces, one-time kernel attributes, NCCL channels) and capture."""
        self.load(images, labels)
        if not self._use_graph:
            for _ in range(self._warmup):
                before = _lib.launch_count()
                self._eager_step()
                self.launches_per_step = _lib.launch_count() - before
            torch.cuda.synchronize()
            return
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(self._warmup):
                before = _lib.launch_count()
                self._eager_step()
                self.launches_per_step = _lib.launch_count() - before
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self._eager_step()
        torch.cuda.synchronize()

    def load(self, images, labels):
        self.static_images.copy_(images, non_blocking=True)
        self.static_labels.copy_(labels, non_blocking=True)

    def run(self):
        """One training step on whatever is in the static input buffers; returns the (device) loss."""
        if self.graph is not None:
            self.graph.replay()
        else:
            self._eager_step()
        return self.static_loss

    # ---- end-to-end feeding ----------------------------------------------------------------------
    def _init_feed(self):
        self._copy_stream = torch.cuda.Stream(device=self.device)
        self._stage = []
        for _ in range(2):
            self._stage.append(dict(images=torch.empty_like(self.static_images), labels=torch.empty_like(self.static_labels),
                                    ready=torch.cuda.Event(), free=torch.cuda.Event()))
            self._stage[-1]["free"].record(torch.cuda.current_stream())
        self._host_loss = torch.zeros(2, dtype=torch.float32).pin_memory()
        self._loss_events = [torch.cuda.Event(), torch.cuda.Event()]

    def feed(self, host_images, host_labels):
        """Start the H2D copy of the NEXT batch (pinned host tensors) on the copy stream."""
        if self._stage is None:
            self._init_feed()
        slot = self._stage[self._flip_in]
        self._flip_in ^= 1
        with torch.cuda.stream(self._copy_stream):
            self._copy_stream.wait_event(slot["free"])  # its previous contents were consumed
            slot["images"].copy_(host_images, non_blocking=True)
            slot["labels"].copy_(host_labels, non_blocking=True)
            slot["ready"].record(self._copy_stream)

    def step_fed(self):
        """Run one step on the oldest fed batch.  Returns the loss of the PREVIOUS fed step as a Python
        float (None for the first): its D2H copy was issued a step ago, so this read does not stall."""
        cur = torch.cuda.current_stream()
        slot = self._stage[self._flip_out]
        self._flip_out ^= 1
        cur.wait_event(slot["ready"])
        self.static_images.copy_(slot["images"], non_blocking=True)
        self.static_labels.copy_(slot["labels"], non_blocking=True)
        slot["free"].record(cur)
        self.run()
        k = self._steps_fed & 1
        prev = None
        if self._steps_fed > 0:
            self._loss_events[k ^ 1].synchronize()
            prev = float(self._host_loss[k ^ 1])
        self._host_loss[k:k + 1].copy_(self.static_loss.reshape(1), non_blocking=True)
        self._loss_events[k].record(cur)
        self._steps_fed += 1
        return prev

    def last_loss(self):
        """Loss of the most recent ``step_fed`` (blocks until its copy has landed)."""
        k = (self._steps_fed - 1) & 1
        self._loss_events[k].synchronize()
        return float(self._host_loss[k])

    def close(self):
        """Release the captured graph (and the NCCL work it references) before the process group goes."""
        torch.cuda.synchronize()
        self.graph = None
        torch.cuda.synchronize()


class GraphedInference:
    """``model(images)`` under ``no_grad`` (and autocast to ``amp_dtype``, bf16 by default) captured once and replayed
    with one launch: at small batches the ~90 launches of a ViT-B forward cost more than the kernels (batch 1 at 1025
    tokens: 4.5 ms eager).  ``bf16=False`` runs without autocast (fp32).  ``run(images)`` copies the batch into the
    graph's static input and returns the static output tensor."""

    def __init__(self, model, images_shape, device, bf16: bool = True, use_graph: bool = True, warmup: int = 3,
                 amp_dtype: torch.dtype = torch.bfloat16):
        if amp_dtype not in (torch.bfloat16, torch.float16):
            raise ValueError(f"GraphedInference: amp_dtype must be torch.bfloat16 or torch.float16, got {amp_dtype}")
        self.model, self.bf16, self.amp_dtype, self.device = model, bf16, amp_dtype, device
        self.static_images = torch.zeros(images_shape, device=device, dtype=torch.float32)
        self.static_out = None
        self.graph = None
        self.launches_per_step = 0
        side = torch.cuda.Stream(device=device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(max(1, warmup)):
                before = _lib.launch_count()
                self.static_out = self._eager()
                self.launches_per_step = _lib.launch_count() - before
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        if use_graph:
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self.static_out = self._eager()
            torch.cuda.synchronize()

    def _eager(self):
        with torch.no_grad(), torch.autocast("cuda", dtype=self.amp_dtype, enabled=self.bf16):
            return self.model(self.static_images)

    def run(self, images=None):
        if images is not None and images is not self.static_images:
            self.static_images.copy_(images, non_blocking=True)
        if self.graph is not None:
            self.graph.replay()
        else:
            self.static_out = self._eager()
        return self.static_out

    def close(self):
        torch.cuda.synchronize()
        self.graph = None
        torch.cuda.synchronize()

