"""One CUDA graph for a whole training step.

At the step size of the reference's own yaml (options/nerf_lm_adapt_gan.yaml:28,117-118: 8 patches x 256 rays x 64 samples) the
kernels of a texture-learner step take ~0.9 ms while Python needs ~1.9 ms to issue them (18 C-ABI launches, the loss glue, autograd
bookkeeping and the engine's `torch.optim.Adam`, model/nerf_adapt_st_gan.py:62-69,117-126) -- the step is launch-bound.  Every
texpose_b200 entry point launches on the caller's stream, never synchronises and never allocates outside torch's caching allocator,
so the step -- `Graph.render(mode='train')`, `Graph.compute_loss`, `summarize_loss`, `backward()`, `optimizer.step()` and the re-pack
of the bf16 weight images that the updated weights require -- can be captured once and replayed as ONE graph launch:
0.97 ms instead of 1.88 ms per step on a B200 (scripts/yaml_step_time.py; the unmodified reference needs 17 ms).

    step = GraphedStep(fn, optimizer, static=dict(coords=coords, image=image, ...))
    for batch in loader:
        out = step(coords=batch.coords, image=batch.image, ...)      # copies into the static buffers, replays

Capturable steps (each tested replay == eager, bit for bit: tests/test_gpu_train_graph.py, test_gpu_graph_pretrain.py,
test_gpu_graph_fp32.py):
  * adaptation `model.nerf_adapt_st_gan.Graph`, opt.b200.mlp 'bf16' / 'auto' (lock-step forward + fused heads backward, or the
    staged kernels) and 'fp32' with fp32_engine = 'tc' (split save + split staged heads backward);
  * pre-training `model.nerf_pretrain.Graph` (and nerf_pretrain_env), opt.b200.mlp 'bf16' / 'auto' and 'fp32' with
    fp32_engine = 'tc' (mlp_tc_plain: the trunk trains).
Static inputs -- everything the step reads that changes between steps, allocated once and passed in `static`: the adaptation
step's patch coordinates, image and mask; the pre-training step's ray subset (`Graph.get_ray_idx` draws it with torch.randperm:
call it eagerly, outside the graph, so the random stream is the reference's, and pass `var.ray_idx`), image, obj_mask,
erode_mask, depth_gt; and for either engine pose, intr, z_near / z_far whenever they change per batch.  View matrices: the bf16
modes build them on the device in one launch (tp_view_matrices), the fp32 mode with torch.linalg.inv_ex, which is captured as
it stands.  With camera.HOST_MATRICES (K^-1 / pose^-1 inverted on the CPU, a synchronisation) compute them eagerly with
`camera.view_matrices` and pass them as a static `view=(kinv, pinv)` to `Graph.render`; capturing the host inversion raises.

Requirements (checked where they can be): the optimizer is capturable (`torch.optim.Adam(..., capturable=True)`); `fn` reads its
inputs from the static tensors, takes no data-dependent Python branch and makes no host read-back; shapes are fixed.  What
would freeze a host decision into the graph raises while capturing, naming the option: opt.b200.rng = 'philox' (its seed is drawn
on the host: use 'torch', whose generator advances on every replay), opt.b200.nan_guard (reads back), mlp_tc32.check_range
(reads back), camera.HOST_MATRICES without `view`, and an ops.device_table miss (a host upload).  The warm-up iterations are real
training steps on the inputs present in the static buffers.

Weight caches: the packed weight images are keyed by the parameters' addresses and `_version`.  A replay changes the weights
without Python seeing it, so the step bumps the version counter of every parameter the optimizer updates before the capture
(every pack launch is then recorded in the graph, never skipped on a stale key) and after every replay (an eager render between
replays re-packs from the weights the replays wrote).

Data-parallel: call the gradient exchange inside `fn` after `backward()`.  `parallel.PeerGradExchange(params, capturable=True)`
keeps its epoch on the device, so every replay runs a new exchange and nothing NCCL-side is captured; its warm-up calls here are
eager exchanges on the same counter, so every rank must build its GraphedStep (same `warmup`) and replay in the same sequence.
A `PeerGradExchange` without `capturable` refuses to be captured.  `parallel.GradBucket` captures the NCCL allreduce instead; a
process group whose communicator lives in a graph does not tear down cleanly.
"""
from __future__ import annotations

from typing import Callable, Dict, Optional

import torch
from torch.autograd.graph import increment_version


def refuse_capture(option: str, reason: str):
    """Raises when the current stream is capturing a CUDA graph: the caller is about to decide something on the host (`reason`)
    that a replay would repeat with the captured value instead of deciding it again."""
    if torch.cuda.is_available() and torch.cuda.is_current_stream_capturing():
        raise RuntimeError(f"{option} cannot be captured in a CUDA graph: {reason}")


class GraphedStep:

    def __init__(self, fn: Callable[[], object], optimizer: Optional[torch.optim.Optimizer] = None,
                 static: Optional[Dict[str, torch.Tensor]] = None, warmup: int = 3):
        if not torch.cuda.is_available():
            raise RuntimeError("GraphedStep needs a CUDA device (texpose_b200 has no CPU path)")
        if optimizer is not None:
            for group in optimizer.param_groups:
                if "capturable" in group and not group["capturable"]:
                    raise ValueError("the optimizer step is part of the captured graph: construct it with capturable=True")
        self.static = dict(static or {})
        for k, v in self.static.items():
            if not (isinstance(v, torch.Tensor) and v.is_cuda):
                raise ValueError(f"static input {k!r} must be a CUDA tensor")
        self.optimizer = optimizer
        self.warmup_steps = int(warmup)
        self._trained = [p for group in optimizer.param_groups for p in group["params"]] if optimizer is not None else []

        def one():
            out = fn()
            if optimizer is not None:
                optimizer.step()
            return out

        # warm-up on a side stream (torch's capture recipe): lazy initialisation -- optimizer state, packed weight images, cached
        # descriptor tables (ops.device_table uploads from host memory on a miss, which a capture does not allow) -- happens here
        current = torch.cuda.current_stream()
        side = torch.cuda.Stream()
        side.wait_stream(current)
        with torch.cuda.stream(side):
            for _ in range(max(1, self.warmup_steps)):
                if optimizer is not None:
                    optimizer.zero_grad(set_to_none=True)
                one()
        current.wait_stream(side)
        # gradients are created inside the capture, from the graph's private pool; a replay overwrites them in place
        if optimizer is not None:
            optimizer.zero_grad(set_to_none=True)
        increment_version(self._trained)        # no weight cache may hit during the capture: every pack launch is recorded
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.out = one()
        self.replays = 0

    def __call__(self, **inputs):
        """Copies `inputs` into the static buffers of the same names and replays the step; returns the captured outputs (static
        tensors, overwritten by the next call)."""
        for k, v in inputs.items():
            if k not in self.static:
                raise KeyError(f"{k!r} is not a static input of this step (have {sorted(self.static)})")
            dst = self.static[k]
            if tuple(v.shape) != tuple(dst.shape):
                raise ValueError(f"static input {k!r} has shape {tuple(dst.shape)}; got {tuple(v.shape)} (a graph has fixed shapes)")
            dst.copy_(v, non_blocking=True)
        self.graph.replay()
        increment_version(self._trained)        # the replay rewrote the weights: version-keyed caches must re-pack
        self.replays += 1
        return self.out
