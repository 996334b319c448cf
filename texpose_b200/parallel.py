"""Multi-GPU plumbing for the render path: one process per GPU, torch.distributed (NCCL over NVLink/NVSwitch).

The reference is single-GPU (options.py:112).  The path shards naturally (SURVEY.md 8e):
  * rendering: views (or contiguous row blocks of one frame) are partitioned across ranks, no exchange;
    an optional all_gather collects the 56 B/ray outputs;
  * training: data-parallel over patches; ONE exchange per step -- the mean over the ranks of a flat fp32 buffer with
    the head + embedding gradients (~1.7 MB).  Two implementations with the same interface:
      GradBucket        torch.distributed allreduce (NCCL on GPUs; gloo in the CPU tests),
      PeerGradExchange  one kernel over CUDA-IPC peer windows (NVLink loads/stores, csrc/peer.cu): ranks of ONE node,
                        result bit-identical on every rank (fixed rank-order sum).
Samples of one ray are never split (scan dependence).
"""
from __future__ import annotations

import ctypes
from typing import Iterable, List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist

from . import _C


def shard_range(n: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous [begin, end) of `n` items for `rank`; sizes differ by at most one, order preserved."""
    base, rem = divmod(n, world)
    begin = rank * base + min(rank, rem)
    return begin, begin + base + (1 if rank < rem else 0)


def shard_views(n_views: int, rank: int, world: int) -> List[int]:
    b, e = shard_range(n_views, rank, world)
    return list(range(b, e))


def shard_rays(n_rays: int, rank: int, world: int, align: int = 1) -> Tuple[int, int]:
    """Row-block partition of one frame's rays; `align` keeps shard boundaries on multiples (e.g. image rows)."""
    units = (n_rays + align - 1) // align
    b, e = shard_range(units, rank, world)
    return min(b * align, n_rays), min(e * align, n_rays)


class GradBucket:
    """Flat fp32 buffer over the trainable parameters (heads + latent embeddings): one allreduce per step."""

    def __init__(self, params: Iterable[torch.nn.Parameter]):
        self.params = [p for p in params if p.requires_grad]
        self.sizes = [p.numel() for p in self.params]
        total = sum(self.sizes)
        dev = self.params[0].device if self.params else torch.device("cpu")
        self.flat = torch.zeros(total, dtype=torch.float32, device=dev)

    def pack(self, into: Optional[torch.Tensor] = None):
        """One launch: concatenate the gradients into the flat buffer (missing gradients count as zero)."""
        if into is None:
            into = self.flat
        base = into.untyped_storage().data_ptr()
        parts = []
        for p in self.params:
            g = p.grad if p.grad is not None else torch.zeros_like(p)
            if g.untyped_storage().data_ptr() == base:      # a view left by the previous unpack, accumulated into: no aliasing
                g = g.clone()
            parts.append(g.reshape(-1))
        if parts:
            torch.cat(parts, out=into)
        return into

    def unpack(self):
        """No copy back: every .grad becomes a view into the reduced flat buffer."""
        off = 0
        for p, n in zip(self.params, self.sizes):
            p.grad = self.flat[off:off + n].view_as(p)
            off += n

    def allreduce_mean(self, group=None):
        """Mean over the ranks of every gradient (per-shard losses are means): one concatenation, one allreduce."""
        if not (dist.is_available() and dist.is_initialized()):
            return
        world = dist.get_world_size(group)
        if world == 1:
            return
        self.pack()
        if dist.get_backend(group) == "nccl":
            dist.all_reduce(self.flat, op=dist.ReduceOp.AVG, group=group)
        else:                                       # gloo (CPU tests) has no AVG
            dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, group=group)
            self.flat.div_(world)
        self.unpack()


class _DeviceSpan:
    """fp32 view of raw device memory for torch.as_tensor (CUDA array interface); keeps the owning window alive."""

    def __init__(self, ptr: int, n: int, owner):
        self.owner = owner
        self.__cuda_array_interface__ = dict(shape=(n,), typestr="<f4", data=(ptr, False), version=3, strides=None)


class PeerWindow:
    """One rank's exchange window (csrc/peer.cu): [1 KB header | data buffer 0 | data buffer 1] in cudaMalloc'ed memory that
    peer processes open through its 64-byte CUDA IPC handle.  `buffers[k]` are fp32 tensors over the two data buffers."""

    def __init__(self, n_floats: int, device):
        lib = _C.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("PeerWindow lives in GPU memory (texpose_b200 has no CPU path)")
        self.n = int(n_floats)
        self.bytes = int(lib.tp_peer_window_bytes(self.n))
        ptr = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            _C.check(lib.tp_peer_window_create(self.bytes, ctypes.byref(ptr)), "tp_peer_window_create")
        self.ptr = int(ptr.value)
        self._imported = []
        self.buffers = [torch.as_tensor(_DeviceSpan(self.ptr + int(lib.tp_peer_data_offset(self.n, k)), max(self.n, 1), self),
                                        device=self.device)[:self.n] for k in (0, 1)]

    def handle(self) -> bytes:
        buf = ctypes.create_string_buffer(64)
        with torch.cuda.device(self.device):
            _C.check(_C.load().tp_peer_window_export(self.ptr, buf), "tp_peer_window_export")
        return buf.raw

    def open_peer(self, handle: bytes) -> int:
        """Device pointer of a peer process' window in this process (peer access is enabled on first use)."""
        out = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            _C.check(_C.load().tp_peer_window_import(ctypes.create_string_buffer(handle, 64), ctypes.byref(out)),
                     "tp_peer_window_import")
        self._imported.append(int(out.value))
        return int(out.value)

    def status(self) -> int:
        """0 = healthy; otherwise the epoch at which a peer failed to arrive within the timeout (synchronising read)."""
        st = ctypes.c_uint32(0)
        with torch.cuda.device(self.device):
            _C.check(_C.load().tp_peer_status(self.ptr, ctypes.byref(st)), "tp_peer_status")
        return int(st.value)

    def close(self):
        lib = _C.load()
        if self.ptr:
            with torch.cuda.device(self.device):
                torch.cuda.synchronize()
                for q in self._imported:
                    lib.tp_peer_window_release(q)
                lib.tp_peer_window_destroy(self.ptr)
            self.ptr, self._imported, self.buffers = 0, [], []


def peer_allreduce_mean(window_ptrs: Sequence[int], rank: int, n_floats: int, epoch: int, out: torch.Tensor,
                        grid_ctas: int = 0, timeout_ms: int = 0, stream=None):
    """out[:n] = mean over the windows of data buffer (epoch & 1), summed in rank order (tp_peer_allreduce_mean)."""
    if not out.is_cuda or out.dtype != torch.float32 or out.numel() < (n_floats + 3) // 4 * 4:
        raise RuntimeError("peer_allreduce_mean: `out` must be a CUDA fp32 tensor of at least n rounded up to 4 floats")
    arr = (ctypes.c_void_p * len(window_ptrs))(*window_ptrs)
    st = stream if stream is not None else torch.cuda.current_stream(out.device)
    with torch.cuda.device(out.device):
        _C.call("tp_peer_allreduce_mean", arr, len(window_ptrs), rank, n_floats, epoch, out.data_ptr(), grid_ctas,
                timeout_ms, st.cuda_stream)


def peer_stage(window_ptr: int, n_floats: int, src: torch.Tensor, stream=None):
    """Data buffer (e+1)&1 of the local window <- src[:n], then the window's device epoch e becomes e+1 (tp_peer_stage)."""
    if not src.is_cuda or src.dtype != torch.float32 or not src.is_contiguous() or src.numel() < n_floats:
        raise RuntimeError("peer_stage: `src` must be a contiguous CUDA fp32 tensor of at least n floats")
    st = stream if stream is not None else torch.cuda.current_stream(src.device)
    with torch.cuda.device(src.device):
        _C.call("tp_peer_stage", window_ptr, n_floats, src.data_ptr(), st.cuda_stream)


def peer_allreduce_mean_dev(window_ptrs: Sequence[int], rank: int, n_floats: int, out: torch.Tensor,
                            grid_ctas: int = 0, timeout_ms: int = 0, stream=None):
    """peer_allreduce_mean with the epoch read from the local window's device epoch (tp_peer_allreduce_mean_dev)."""
    if not out.is_cuda or out.dtype != torch.float32 or out.numel() < (n_floats + 3) // 4 * 4:
        raise RuntimeError("peer_allreduce_mean_dev: `out` must be a CUDA fp32 tensor of at least n rounded up to 4 floats")
    arr = (ctypes.c_void_p * len(window_ptrs))(*window_ptrs)
    st = stream if stream is not None else torch.cuda.current_stream(out.device)
    with torch.cuda.device(out.device):
        _C.call("tp_peer_allreduce_mean_dev", arr, len(window_ptrs), rank, n_floats, out.data_ptr(), grid_ctas,
                timeout_ms, st.cuda_stream)


class PeerGradExchange(GradBucket):
    """GradBucket whose exchange is ONE kernel over NVLink peer memory instead of a library allreduce.

    Set-up (once): every rank creates a window, the 64-byte IPC handles travel through `all_gather_object`, every rank opens
    its peers' windows.  Per step: one `cat` packs the gradients into the local window's buffer of the step's parity, one
    launch publishes / waits / reduces, `.grad`s become views of the reduced buffer.  All ranks must sit on one node with
    peer access (NVLink / NVSwitch); anything else raises at set-up -- there is no silent fallback to the allreduce.

    capturable=True makes `allreduce_mean()` capturable in a CUDA graph (e.g. inside `train_graph.GraphedStep`, like
    `torch.optim.Adam(capturable=True)`): the epoch and the parity buffer are then chosen on the device, not on the host.
    Each call, eager or replayed, is one `cat` into a fixed local staging buffer, `tp_peer_stage` (copy into the window's
    buffer of the next device epoch and advance it), `tp_peer_allreduce_mean_dev` into `flat`, and the views of `unpack()`.
    Eager calls and replays advance the same device counter, so every rank must make the same sequence of exchanges --
    counting GraphedStep's eager warm-up steps -- as it must make the same sequence of calls without a graph.  Without
    capturable, a call made while the current stream is capturing raises: the host epoch would be frozen into the graph."""

    def __init__(self, params: Iterable[torch.nn.Parameter], group=None, timeout_ms: int = 10000, capturable: bool = False):
        super().__init__(params)
        if not (dist.is_available() and dist.is_initialized()):
            raise RuntimeError("PeerGradExchange needs an initialised process group (use GradBucket for a single process)")
        dev = self.flat.device
        self.group, self.timeout_ms = group, int(timeout_ms)
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.n = self.flat.numel()
        self.window = PeerWindow(self.n, dev)
        handles = [None] * self.world
        dist.all_gather_object(handles, self.window.handle(), group=group)
        self.ptrs = [self.window.ptr if r == self.rank else self.window.open_peer(h) for r, h in enumerate(handles)]
        self.flat = torch.zeros((self.n + 3) // 4 * 4, dtype=torch.float32, device=dev)    # the reduced gradients land here
        self.epoch = 0
        self.capturable = bool(capturable)
        self.staging = torch.zeros_like(self.flat) if self.capturable else None
        torch.cuda.synchronize(dev)
        dist.barrier(group)          # every window exists, is zeroed and is open everywhere before the first publish

    def allreduce_mean(self, group=None):
        if self.capturable:
            self.pack(into=self.staging[:self.n])
            peer_stage(self.window.ptr, self.n, self.staging)
            peer_allreduce_mean_dev(self.ptrs, self.rank, self.n, self.flat, timeout_ms=self.timeout_ms)
            self.unpack()
            return
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError("PeerGradExchange.allreduce_mean() is being captured in a CUDA graph, which would freeze its "
                               "host-chosen epoch: construct the exchange with capturable=True")
        self.epoch += 1
        self.pack(into=self.window.buffers[self.epoch & 1])
        peer_allreduce_mean(self.ptrs, self.rank, self.n, self.epoch, self.flat, timeout_ms=self.timeout_ms)
        self.unpack()

    def check(self):
        """Raises if a peer ever missed an exchange (reads one status word back: call it off the hot path)."""
        bad = self.window.status()
        if bad:
            raise RuntimeError(f"PeerGradExchange: a peer did not arrive at epoch {bad} within {self.timeout_ms} ms")

    def close(self):
        if dist.is_initialized():
            torch.cuda.synchronize(self.flat.device)
            dist.barrier(self.group)     # nobody unmaps a window a peer may still be reading
        self.window.close()


PER_RAY_KEYS = ("rgb", "rgb_static", "rgb_transient", "depth", "opacity", "opacity_static", "opacity_transient", "uncert")
PRETRAIN_KEYS = ("rgb", "depth", "opacity")      # the per-ray outputs of the pre-training engine (model.nerf_pretrain.Graph)
_PER_RAY_CHANNELS = dict(rgb=3, rgb_static=3, rgb_transient=3, depth=1, opacity=1, opacity_static=1, opacity_transient=1, uncert=1)


def frame_layout(n_rays: int, keys: Sequence[str] = PER_RAY_KEYS):
    """Float offsets of the per-ray frame buffers inside one data buffer of the gather window: {key: (offset, channels)},
    total floats.  Every buffer starts on a 64-float (256 B) boundary."""
    off, out = 0, {}
    for k in keys:
        c = _PER_RAY_CHANNELS[k]
        out[k] = (off, c)
        off += (n_rays * c + 63) // 64 * 64
    return out, off


def peer_barrier(window_ptrs: Sequence[int], rank: int, epoch: int, device, timeout_ms: int = 0, stream=None):
    arr = (ctypes.c_void_p * len(window_ptrs))(*window_ptrs)
    st = stream if stream is not None else torch.cuda.current_stream(device)
    with torch.cuda.device(device):
        _C.call("tp_peer_barrier", arr, len(window_ptrs), rank, epoch, timeout_ms, st.cuda_stream)


class FrameGather:
    """ONE frame rendered by all ranks of a node (the north-star's 480x640x128 frame at 1/2/4/8 GPUs; the reference is
    single-GPU, options.py:112).  Rank r renders the row block shard_rays(HW, r, world, align=W) with the graph's render launch
    (`graph._render_fused`: the lock-step or the staged kernel's; keys=PRETRAIN_KEYS for the pre-training engine),
    whose compositing epilogue stores the 56 B/ray outputs STRAIGHT INTO THE ROOT RANK'S FRAME BUFFERS -- a CUDA-IPC window, so
    the stores of ranks != root travel over NVLink as they are produced: the gather is the kernel's own output write, there
    is no collective and no staging copy.  One tiny barrier kernel per frame (tp_peer_barrier) publishes completion.

    Frame e lands in data buffer e & 1 of the root's window, so the root may still read frame e while frame e+1 is rendered;
    buffer e & 1 is rewritten by frame e+2, which no rank starts before the root has passed barrier e+1 -- i.e. after whatever
    the root enqueued on its stream between the two barriers (its reads of frame e).  Per-sample tensors (alpha_*, density:
    16 B/sample) are not gathered: a rank that wants them for its rows passes them in `local_keys`."""

    def __init__(self, opt, keys: Sequence[str] = PER_RAY_KEYS, root: int = 0, group=None, timeout_ms: int = 10000, device=None):
        self.keys = tuple(keys)
        self.H, self.W = int(opt.H), int(opt.W)
        self.HW = self.H * self.W
        self.layout, self.n = frame_layout(self.HW, self.keys)
        self.group, self.root, self.timeout_ms = group, int(root), int(timeout_ms)
        distributed = dist.is_available() and dist.is_initialized()
        self.rank = dist.get_rank(group) if distributed else 0
        self.world = dist.get_world_size(group) if distributed else 1
        self.device = torch.device(device if device is not None else opt.device)
        self.window = PeerWindow(self.n, self.device)
        if self.world > 1:
            handles = [None] * self.world
            dist.all_gather_object(handles, self.window.handle(), group=group)
            self.ptrs = [self.window.ptr if r == self.rank else self.window.open_peer(h) for r, h in enumerate(handles)]
        else:
            self.ptrs = [self.window.ptr]
        self.epoch = 0
        lib = _C.load()
        self._data_off = [int(lib.tp_peer_data_offset(self.n, k)) for k in (0, 1)]
        self.rows = shard_rays(self.HW, self.rank, self.world, align=self.W)
        torch.cuda.synchronize(self.device)
        if self.world > 1:
            dist.barrier(group)

    def frame_views(self, parity: int):
        """The root's view of one data buffer: {key: [1, HW, C] tensor} (valid on the root after the frame's barrier)."""
        buf = self.window.buffers[parity]
        return {k: buf[o:o + self.HW * c].view(1, self.HW, c) for k, (o, c) in self.layout.items()}

    def render(self, graph, opt, pose, intr, depth_range, sample_idx=None, mode="val", local_keys: Sequence[str] = ()):
        """Renders this rank's row block of the frame of view `pose` ([1,3,4]) and gathers it.  Returns (frame, local): `frame` =
        {key: [1,HW,C]} on the root (None elsewhere), `local` = the `local_keys` outputs of this rank's rows."""
        if len(pose) != 1:
            raise ValueError("FrameGather renders one view per call")
        missing = [k for k in tuple(self.keys) + tuple(local_keys) if k not in getattr(graph, "RENDER_KEYS", ())]
        if missing:
            raise ValueError(f"{type(graph).__module__}.{type(graph).__name__} does not render {missing} "
                             f"(it renders {getattr(graph, 'RENDER_KEYS', ())})")
        self.epoch += 1
        par = self.epoch & 1
        b, e = self.rows
        base = self.ptrs[self.root] + self._data_off[par]
        out_ptrs = {k: base + 4 * (o + b * c) for k, (o, c) in self.layout.items()}
        local = graph._render_fused(opt, pose, intr, range(b, e), depth_range, sample_idx, mode,
                                    want=tuple(self.keys) + tuple(local_keys), out_ptrs=out_ptrs)
        peer_barrier(self.ptrs, self.rank, self.epoch, self.device, timeout_ms=self.timeout_ms)
        return (self.frame_views(par) if self.rank == self.root else None), local

    def check(self):
        bad = self.window.status()
        if bad:
            raise RuntimeError(f"FrameGather: a rank did not finish frame {bad} within {self.timeout_ms} ms")

    def close(self):
        if self.world > 1 and dist.is_initialized():
            torch.cuda.synchronize(self.device)
            dist.barrier(self.group)
        self.window.close()


def gather_ray_outputs(local: torch.Tensor, sizes: Sequence[int], group=None) -> torch.Tensor:
    """all_gather of per-ray outputs [R_local, C] from uneven contiguous shards -> [sum(sizes), C] on every rank."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return local
    world = dist.get_world_size(group)
    m = max(sizes)
    pad = torch.zeros(m, *local.shape[1:], dtype=local.dtype, device=local.device)
    pad[:local.shape[0]] = local
    outs = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(outs, pad, group=group)
    return torch.cat([o[:n] for o, n in zip(outs, sizes)], dim=0)
