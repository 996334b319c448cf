#!/usr/bin/env python
"""Benchmark of the TexPose render hot path on B200 (contract: see the task's bench.py section).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1], "C2"): LineMOD-duck-shaped synthetic full-frame render, 480x640 rays x 128
samples, static + transient + light heads, random-init (seed 0) weights, bf16 tensor-core MLP.  One step = ONE frame.
  N = 1   the frame through the public API (Graph.nerf_forward(mode='val')): one fused render launch.
  N > 1   the SAME frame, row blocks sharded over the ranks (strong scaling: BASELINE `metric` "480x640 render ms/frame
          at 1/2/4/8 B200"): every rank's fused launch stores its 56 B/ray outputs straight into rank 0's frame buffers
          over NVLink peer memory (parallel.FrameGather), one barrier kernel per frame; no collective.
          The round-1 weak-scaling number (one view per GPU) is kept as the `weak_views` block.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W, NS = 480, 640, 128
FLOP_PER_SAMPLE_FWD = 1_821_184          # SURVEY.md 8d (dense, unpadded)
FLOP_PER_SAMPLE_BWD = 1_399_808          # SURVEY.md 8d: backward with the trunk frozen
FLOP_PER_SAMPLE_FWD_BWD = FLOP_PER_SAMPLE_FWD + FLOP_PER_SAMPLE_BWD
METRIC, UNIT = "ray-samples/sec", "samples/s"
WORKLOAD = "C2 LineMOD-duck synthetic full-frame render 480x640x128, static+transient+light heads"
REF_CHUNK0 = 230 * W                     # the reference arm's 2048-ray chunks start in the object rows of the frame


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-rays", type=int, default=2048, help="rays per step of the bounded CPU sample (the reference's own "
                                                               "chunk size, opt.nerf.rand_rays)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--no-parity-frame", action="store_true", help="skip the fp32-parity-mode frame (split-fp16 kernel vs SIMT)")
    ap.add_argument("--no-weak", action="store_true", help="N > 1: skip the one-view-per-GPU block")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


def so_sha16():
    from texpose_b200 import _C
    try:
        return hashlib.sha256(open(_C.LIB_PATH, "rb").read()).hexdigest()[:16]
    except OSError:
        return None


def src_sha16():
    """Hash of the kernel sources + the C-ABI header: identifies a build across recompilations (nvcc's output is not bit-reproducible)."""
    from texpose_b200 import _C
    h = hashlib.sha256()
    files = sorted(os.path.join(_C.CSRC, f) for f in os.listdir(_C.CSRC) if f.endswith((".cu", ".cuh"))) + [_C.HEADER]
    for f in files:
        h.update(os.path.basename(f).encode())
        h.update(open(f, "rb").read())
    return h.hexdigest()[:16]


# ---------------------------------------------------------------------------------------------- reference arm

def frame_inputs(dev="cpu"):
    """Seeded C2 inputs (SURVEY 8d): pose seed 0, LineMOD K, AABB sample bounds of the padded duck box."""
    from oracle import texpose_oracle as O
    from texpose_b200 import synth
    pose, intr = synth.poses([0]), synth.intrinsics(1)
    c, r = O.get_center_and_ray(pose, intr, H, W)
    lo, hi = synth.padded_aabb()
    tn, tf, v = O.aabb_ray_intersection(lo, hi, c, r)
    zn, zf = O.box_bounds_to_range(tn, tf, v, *synth.BG_RANGE)
    t = lambda x: x.to(dev)
    return t(pose), t(intr), (t(zn)[:, :, None], t(zf)[:, :, None])


def reference_graph(device):
    """The REAL reference (unmodified sources from /root/reference or baseline/_ref): Graph of model/nerf_adapt_st_gan.py with
    the nerf_lm_adapt_gan.yaml options at the C2 sample count.  None when no copy of the reference is present."""
    from oracle import ref_import
    if not ref_import.available():
        return None
    ns = ref_import.load()
    opt = ref_import.load_yaml_opt("nerf_lm_adapt_gan", H, W, device=device)
    opt.nerf.sample_intvs = NS
    g = ref_import.build_graph(ns, opt, n_images=8, seed=0).to(device)
    return ns, opt, g


def cpu_reference_step(n_rays, threads):
    """One step of the CPU arm = one chunk of the reference's own render_by_slices loop (model/nerf_adapt_st_gan.py:640-650):
    Graph.render(mode='val') on `n_rays` consecutive rays of the C2 frame, fp32, all host threads.  The real reference when a
    copy is present (kind 'reference'), else the oracle port.  Returns (step, samples per step, kind, description)."""
    import torch
    torch.set_num_threads(threads)
    ref = reference_graph("cpu")
    pose, intr, dr = frame_inputs("cpu")
    state = {"c": 0}
    if ref is not None:
        from oracle import ref_import
        ns, opt, g = ref

        def step():
            c0 = REF_CHUNK0 + (state["c"] % 16) * n_rays
            state["c"] += 1
            idx = torch.arange(c0, c0 + n_rays)[None]
            with ref_import.cpu_shim(), torch.no_grad():
                state["out"] = g.render(opt, pose, intr=intr, ray_idx=idx, depth_range=dr, sample_idx=None, mode="val")

        return step, n_rays * NS, "reference", (f"the unmodified reference (model/nerf_adapt_st_gan.py Graph.render, mode='val') on {n_rays} "
                                                f"consecutive rays x {NS} samples of the C2 frame per step = one chunk of its own "
                                                f"render_by_slices loop, fp32, torch CPU ops on {threads} threads")
    from oracle import texpose_oracle as O
    from texpose_b200 import synth
    from texpose_b200.config import adapt_gan_opt
    from texpose_b200.layers.nerf_static_transient_light import NeRF
    torch.manual_seed(0)
    m = NeRF(adapt_gan_opt())
    L = lambda ml: [(l.weight.detach(), l.bias.detach()) for l in ml]
    feat, rgb, trans = L(m.mlp_feat), L(m.mlp_rgb), L(m.mlp_trans)
    lt, ll = synth.latents(1)

    def step():
        c0 = REF_CHUNK0 + (state["c"] % 16) * n_rays
        state["c"] += 1
        with torch.no_grad():
            c, r = O.get_center_and_ray(pose, intr, H, W)
            idx = torch.arange(c0, c0 + n_rays)[None]
            rand = torch.rand(1, n_rays, NS, 1)
            state["out"] = O.render_stl(O.gather_rays(c, idx), O.gather_rays(r, idx), dr[0][:, idx[0], 0], dr[1][:, idx[0], 0], rand, NS,
                                        lt, ll, feat, rgb, trans)

    return step, n_rays * NS, "port", (f"oracle port of the reference path (no copy of the reference on this box) on {n_rays} consecutive rays x "
                                      f"{NS} samples per step, fp32, {threads} threads")


def eager_gpu_sample(dev, n_chunks=8):
    """The meaningful "before" on the same B200: the reference's stock eager path (Graph.render in its own 2048-ray chunks, full-
    frame ray generation per chunk, cuBLAS fp32) -- the real reference when a copy is present, else the oracle port."""
    import torch
    ref = reference_graph(str(dev))
    pose, intr, dr = frame_inputs(dev)
    chunk = 2048
    if ref is not None:
        ns, opt, g = ref
        kind = "reference"

        def run():
            with torch.no_grad():
                for c in range(n_chunks):
                    idx = torch.arange(REF_CHUNK0 + c * chunk, REF_CHUNK0 + (c + 1) * chunk, device=dev)[None]
                    g.render(opt, pose, intr=intr, ray_idx=idx, depth_range=dr, sample_idx=None, mode="val")
    else:
        from oracle import texpose_oracle as O
        from texpose_b200 import synth
        from texpose_b200.config import adapt_gan_opt
        from texpose_b200.layers.nerf_static_transient_light import NeRF
        torch.manual_seed(0)
        m = NeRF(adapt_gan_opt()).to(dev)
        L = lambda ml: [(l.weight.detach(), l.bias.detach()) for l in ml]
        feat, rgb, trans = L(m.mlp_feat), L(m.mlp_rgb), L(m.mlp_trans)
        lt, ll = [t.to(dev) for t in synth.latents(1)]
        kind = "port"

        def run():
            with torch.no_grad():
                for c in range(n_chunks):
                    cen, ray = O.get_center_and_ray(pose, intr, H, W)
                    idx = torch.arange(REF_CHUNK0 + c * chunk, REF_CHUNK0 + (c + 1) * chunk, device=dev)[None]
                    rand = torch.rand(1, chunk, NS, 1, device=dev)
                    O.render_stl(O.gather_rays(cen, idx), O.gather_rays(ray, idx), dr[0][:, idx[0], 0], dr[1][:, idx[0], 0], rand, NS, lt,
                                 ll, feat, rgb, trans)
    run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    return dict(value=n_chunks * chunk * NS / (ms * 1e-3), unit=UNIT, kind=kind,
                sample=f"{n_chunks} chunks x {chunk} rays x {NS} samples through Graph.render(mode='val') of the "
                       f"{'unmodified reference' if kind == 'reference' else 'oracle port'}, eager torch ops on this GPU, fp32",
                ms_per_frame_extrapolated=ms * (H * W / (n_chunks * chunk)))


def run_reference(args, rank):
    import torch
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    step, samples, kind, desc = cpu_reference_step(args.cpu_rays, threads)
    for _ in range(max(1, min(args.warmup, 2))):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    val = samples / dt
    line = dict(metric=METRIC, value=val, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=dt * 1e3, higher_is_better=True, scaling="strong" if args.gpus > 1 else "weak", vs_baseline=None,
                dtype="f32", data="synthetic", impl="reference",
                config=dict(workload=WORKLOAD + " (bounded CPU sample)", rays_per_step=args.cpu_rays, samples_per_ray=NS),
                cpu_baseline=dict(value=val, unit=UNIT, cores=threads, kind=kind, sample=desc),
                e2e=dict(value=val, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                torch_threads=torch.get_num_threads())
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------- clocks sampler

class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms",
                                          "20", "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                smax = max(smax, float(f[1]))
                if t0 <= t <= t1:
                    sm.append(float(f[0]))
                    for n, v in zip(names, f[3:7]):
                        if v.lower().startswith("active"):
                            reasons.add(n)
            except ValueError:
                continue
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=smax or None, reasons=sorted(reasons),
                    samples=len(sm))


class CallTimer:
    """CUDA events around C-ABI calls (on the launching stream): per-entry-point device time of an instrumented pass."""

    def __init__(self, names=None):
        from texpose_b200 import _C
        self._C, self.names, self.events, self.orig = _C, names, [], _C.call

    def __enter__(self):
        import torch

        def call(name, *a):
            if self.names is None or name in self.names:
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record()
                self.orig(name, *a)
                a1.record()
                self.events.append((name, a0, a1))
            else:
                self.orig(name, *a)

        self._C.call = call
        return self

    def __exit__(self, *exc):
        self._C.call = self.orig
        return False

    def per_call_ms(self):
        import torch
        torch.cuda.synchronize()
        out = {}
        for name, a0, a1 in self.events:
            out.setdefault(name, []).append(a0.elapsed_time(a1))
        return out


def kernel_ms_of_timed_steps(call_ms, steps, warmup):
    """Device time per step of one entry point from the per-call event times of `warmup + steps` iterations: the calls of the
    last `steps` iterations, summed per step.  None when the calls do not divide evenly over the iterations."""
    total = steps + warmup
    if total <= 0 or steps <= 0 or not call_ms or len(call_ms) % total:
        return None
    per = len(call_ms) // total
    return sum(call_ms[-per * steps:]) / steps


DUMP_LIMIT_BYTES = 64 << 20     # all arrays of one --dump-outputs directory
DUMP_WHOLE_BYTES = 8 << 20      # larger arrays are stored at DUMP_RAYS rays
DUMP_RAYS = 8192


def dump_outputs(out_dir, outputs, n_rays):
    """Writes every tensor of `outputs` as out_dir/<name>.npy: floating point as float32 (float64 stays), integers as float64.
    An array over DUMP_WHOLE_BYTES (the per-sample outputs [1, rays, samples, ...], 0.65 GB a frame) is stored at DUMP_RAYS rays drawn
    with a fixed seed, listed in sample_ray_idx.npy.  The bench's inputs are seeded, so the same arguments write the same files
    and two builds can be compared array by array.  Returns the bytes written."""
    import numpy as np
    import torch
    pick = torch.randperm(n_rays, generator=torch.Generator().manual_seed(0))[:DUMP_RAYS].sort().values
    arrays = {}
    for name, t in outputs.items():
        if not isinstance(t, torch.Tensor):
            continue
        dtype = torch.float32 if t.is_floating_point() and t.dtype != torch.float64 else torch.float64
        t = t.detach()
        if t.numel() * dtype.itemsize > DUMP_WHOLE_BYTES:
            if t.dim() < 2 or t.shape[1] != n_rays:
                raise ValueError(f"--dump-outputs: {name} {tuple(t.shape)} is too large to store whole and has no ray dimension")
            t = t.index_select(1, pick.to(t.device))
            arrays["sample_ray_idx"] = pick.to(torch.float64)
        arrays[name] = t.to("cpu", dtype)
    total = sum(a.numel() * a.element_size() for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES} byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())
    return total


# ---------------------------------------------------------------------------------------------- our arm

def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from texpose_b200 import _C, compute_box, parallel, synth
    from texpose_b200.config import AttrDict, adapt_gan_opt
    from texpose_b200.model.nerf_adapt_st_gan import Graph

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py --impl ours needs a CUDA device (texpose_b200 has no CPU path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # stdout carries exactly one JSON line: NCCL prints its version banner to stdout while the communicator is created
        # (NCCL_DEBUG=VERSION / WARN), so file descriptor 1 points at stderr until the first collective has run
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    _C.build()
    pk = peaks()

    opt = adapt_gan_opt(H=H, W=W, sample_intvs=NS, device=str(dev))
    opt.b200 = AttrDict(mlp="bf16", rng="philox")
    torch.manual_seed(0)
    g = Graph(opt, n_train_images=8).to(dev)
    g.eval()
    lo, hi = [t.to(dev) for t in synth.padded_aabb()]

    def view_inputs(seed):
        pose_h = synth.poses([seed]).pin_memory()
        intr_h = synth.intrinsics(1).pin_memory()
        zn, zf = compute_box.box_range(pose_h.to(dev), intr_h.to(dev), lo, hi, H, W, *synth.BG_RANGE)
        return pose_h, intr_h, zn, zf

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, sampler=False):
        for _ in range(warmup):
            fn()
        barrier()
        cs = ClockSampler(local_rank) if sampler else None
        if cs:
            time.sleep(0.25)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        t1 = time.perf_counter()
        ms = e0.elapsed_time(e1) / steps
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms, (cs.stop(t0, t1) if cs else None)

    # ---- the frame: view 0 on every rank (N > 1: the ranks share it)
    pose_h, intr_h, zn, zf = view_inputs(0)
    zn_h, zf_h = zn.cpu().pin_memory(), zf.cpu().pin_memory()
    mask_h = torch.ones(1, H, W).pin_memory()
    pose_d, intr_d = pose_h.to(dev), intr_h.to(dev)
    idx0 = torch.zeros(1, dtype=torch.long, device=dev)
    var_dev = AttrDict(pose=pose_d, intr=intr_d, z_near=zn, z_far=zf, obj_mask=mask_h.to(dev), idx=idx0)
    out_h = dict(rgb=torch.empty(1, H * W, 3).pin_memory(), depth=torch.empty(1, H * W, 1).pin_memory(),
                 opacity=torch.empty(1, H * W, 1).pin_memory(), uncert=torch.empty(1, H * W, 1).pin_memory())
    samples_per_frame = H * W * NS

    if world == 1:
        rows = (0, H * W)
        gather = None

        def step_resident():
            with torch.no_grad():
                return g.nerf_forward(opt, AttrDict(var_dev), mode="val")

        def step_e2e():
            with torch.no_grad():
                var = AttrDict(pose=pose_h.to(dev, non_blocking=True), intr=intr_h.to(dev, non_blocking=True),
                               z_near=zn_h.to(dev, non_blocking=True), z_far=zf_h.to(dev, non_blocking=True),
                               obj_mask=mask_h.to(dev, non_blocking=True), idx=idx0)
                ret = g.nerf_forward(opt, var, mode="val")
                for k, buf in out_h.items():
                    buf.copy_(ret[k], non_blocking=True)
            return ret

        h2d = sum(t.numel() * t.element_size() for t in (pose_h, intr_h, zn_h, zf_h, mask_h))
        d2h = sum(t.numel() * t.element_size() for t in out_h.values())
    else:
        gather = parallel.FrameGather(opt, device=dev)
        rows = gather.rows
        dr_dev = (zn[:, :, None], zf[:, :, None])
        zn_e2e, zf_e2e = torch.zeros_like(zn), torch.zeros_like(zf)      # e2e: only this rank's rows are uploaded

        def step_resident():
            with torch.no_grad():
                return gather.render(g, opt, pose_d, intr_d, dr_dev)

        def step_e2e():
            b, e = rows
            with torch.no_grad():
                p_d, i_d = pose_h.to(dev, non_blocking=True), intr_h.to(dev, non_blocking=True)
                zn_e2e[:, b:e].copy_(zn_h[:, b:e], non_blocking=True)
                zf_e2e[:, b:e].copy_(zf_h[:, b:e], non_blocking=True)
                frame, _ = gather.render(g, opt, p_d, i_d, (zn_e2e[:, :, None], zf_e2e[:, :, None]))
                if frame is not None:
                    for k, buf in out_h.items():
                        buf.copy_(frame[k], non_blocking=True)

        h2d_local = (pose_h.numel() + intr_h.numel() + 2 * (rows[1] - rows[0])) * 4
        t = torch.tensor([float(h2d_local)], device=dev)
        dist.all_reduce(t)
        h2d = int(t.item())
        d2h = sum(t.numel() * t.element_size() for t in out_h.values())      # rank 0 reads the gathered frame back

    last = {}

    def step_timed():
        last["ret"] = step_resident()

    _C.launch_counts.clear()
    # CUDA events around the fused launch INSIDE the timed region (two event records per step on the launching stream): the kernel
    # time of the roofline and the step time of the headline come from the same iterations, so kernel <= step by construction
    with CallTimer({"tp_render_fused_forward"}) as ct:
        ms, clocks = timed(step_timed, args.steps, args.warmup, sampler=True)
    if args.dump_outputs and rank == 0:
        # written before any later block renders again: N > 1 returns views of the frame buffers the next gathers overwrite
        frame = last["ret"] if world == 1 else last["ret"][0]
        nbytes = dump_outputs(args.dump_outputs, frame, H * W)
        print(f"bench.py: wrote {nbytes / 2 ** 20:.1f} MiB of step {args.steps} outputs to {args.dump_outputs}", file=sys.stderr)
    per_step = {k: v // (args.steps + args.warmup) for k, v in _C.launch_counts.items() if v >= args.steps + args.warmup}
    launches = sum(per_step.values()) * args.steps
    k_ms = kernel_ms_of_timed_steps(ct.per_call_ms().get("tp_render_fused_forward", []), args.steps, args.warmup)
    if k_ms is None:      # (not expected: a step that did not launch the fused kernel a whole number of times) an instrumented pass of its own
        with CallTimer({"tp_render_fused_forward"}) as ct:
            for _ in range(min(args.steps, 5)):
                step_resident()
        kms = ct.per_call_ms()["tp_render_fused_forward"]
        k_ms = sum(kms) / min(args.steps, 5)
    local_samples = (rows[1] - rows[0]) * NS
    achieved_tf = FLOP_PER_SAMPLE_FWD * local_samples / (k_ms * 1e-3) / 1e12
    if gather is not None:
        gather.check()

    ms_e2e, _ = timed(step_e2e, args.steps, max(1, args.warmup // 2))
    # the same frame through the multi-kernel path the fused launch replaces (raygen, gathers, depths, bias table, per-sample MLP
    # launch, compositing: 9 launches, 4.2 GB of HBM traffic) -- reported beside the headline, same box, same process
    multi = None
    if world == 1:
        opt_mk = AttrDict(opt)
        opt_mk.b200 = AttrDict(opt.b200)
        opt_mk.b200.fused_render = False

        def step_multi():
            with torch.no_grad():
                return g.nerf_forward(opt_mk, AttrDict(var_dev), mode="val")

        _C.launch_counts.clear()
        ms_mk, _ = timed(step_multi, max(3, args.steps // 2), 2)
        n_mk = max(3, args.steps // 2) + 2
        multi = dict(ms_per_frame=ms_mk, value=samples_per_frame / (ms_mk * 1e-3), unit=UNIT,
                     launches_per_frame=sum(v // n_mk for v in _C.launch_counts.values()),
                     note="multi-kernel path (opt.b200.fused_render = False): per-sample tensors and the bias table go through HBM")
    # the same frame in the fp32-parity mode (<= 1e-4 against the reference): split-fp16 tensor-core kernel (three MMA passes per
    # K step, csrc/mlp_tc_split.cu) against the SIMT FFMA kernels it replaces for rendering -- same box, same process
    parity = None
    if world == 1 and not args.no_parity_frame:
        def parity_step(engine):
            o = AttrDict(opt)
            o.b200 = AttrDict(opt.b200)
            o.b200.mlp, o.b200.fp32_engine = "fp32", engine

            def step():
                with torch.no_grad():
                    return g.nerf_forward(o, AttrDict(var_dev), mode="val")
            return step

        ms_tc, _ = timed(parity_step("auto"), 3, 1)
        with CallTimer({"tp_tc32_forward"}) as ct32:
            parity_step("auto")()
        k32 = sum(ct32.per_call_ms()["tp_tc32_forward"])
        ms_simt, _ = timed(parity_step("simt"), 1, 1)
        tf32 = 3 * FLOP_PER_SAMPLE_FWD * samples_per_frame / (k32 * 1e-3) / 1e12
        parity = dict(ms_per_frame=ms_tc, value=samples_per_frame / (ms_tc * 1e-3), unit=UNIT, simt_ms_per_frame=ms_simt,
                      speedup_vs_simt=ms_simt / ms_tc, kernel="tcs::nerf_forward_split_kernel", kernel_ms_per_frame=k32,
                      launches_of_kernel_per_frame=len(ct32.per_call_ms()["tp_tc32_forward"]),
                      executed_tflops=tf32, frac_of_sustained_tensor_peak=tf32 / pk["tf_sustained"],
                      note="fp32-parity mode: operands carried as hi + lo fp16, three tcgen05 passes per K step (executed FLOPs = 3 x "
                           "algorithmic); tolerance 1e-4 (tests/test_gpu_tc32.py)")
    # SURVEY 8 (f4): depth + NOCS maps of a 20 480-face mesh at the frame size (tp_mesh_render: project, clear, raster, resolve)
    raster = None
    if world == 1:
        from texpose_b200.tools import mvrenderer
        mv, mf = [t.to(dev) for t in synth.icosphere(5, 0.6)]
        nocs = mvrenderer.nocs_coordinates(mv)
        rows8 = synth.poses(list(range(8))).reshape(8, 12).to(dev)
        K8 = intr_d.expand(8, 3, 3).contiguous()
        ms_r1, _ = timed(lambda: mvrenderer.render_mesh(mv, mf, nocs, rows8[:1], K8[:1], H, W), 20, 3)
        ms_r8, _ = timed(lambda: mvrenderer.render_mesh(mv, mf, nocs, rows8, K8, H, W), 20, 3)
        bytes_view = mv.numel() * 4 * 2 + mf.numel() * 4 + H * W * (8 + 8 + 4 + 12)
        raster = dict(workload="depth + NOCS of a 20 480-face icosphere, 480x640", ms_per_view_b1=ms_r1, ms_per_view_b8=ms_r8 / 8,
                      algorithmic_bytes_per_view=bytes_view, hbm_gbs_b8=8 * bytes_view / (ms_r8 * 1e-3) / 1e9, hbm_peak=pk["hbm"],
                      note="10 MB per view: four launches in the launch-latency regime; views batch into the same four launches")
    value = samples_per_frame / (ms * 1e-3)
    e2e_value = samples_per_frame / (ms_e2e * 1e-3)

    weak = None
    if world > 1 and not args.no_weak:
        # round-1 mode for continuity: every rank renders its OWN view (seed = rank), no exchange at all
        p_h, i_h, zn_r, zf_r = view_inputs(rank)
        var_r = AttrDict(pose=p_h.to(dev), intr=i_h.to(dev), z_near=zn_r, z_far=zf_r, obj_mask=mask_h.to(dev), idx=idx0)

        def step_view():
            with torch.no_grad():
                return g.nerf_forward(opt, AttrDict(var_r), mode="val")

        ms_w, _ = timed(step_view, max(3, args.steps // 2), 2)
        weak = dict(workload="one 480x640x128 view per GPU per step (views sharded across ranks, no exchange)", scaling="weak",
                    value=world * samples_per_frame / (ms_w * 1e-3), unit=UNIT, ms_per_step=ms_w)

    train = None
    if not args.no_train:
        train = bench_train(args, g, opt, dev, world, timed, pk)
    if gather is not None:
        gather.close()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # DRAM bytes of the fused launch from ncu (`scripts/collect_profiles.sh`), valid only for the build it was measured on
    traffic, traffic_note = None, "no ncu capture for this build (scripts/collect_profiles.sh writes profiles/r02_render_traffic.json)"
    tpath = os.path.join(ROOT, "profiles", "r02_render_traffic.json")
    if os.path.exists(tpath) and world == 1:
        try:
            tj = json.load(open(tpath))
            if tj.get("so_sha16") == so_sha16() or (tj.get("src_sha16") and tj.get("src_sha16") == src_sha16()):
                traffic, traffic_note = tj.get("dram_bytes_per_launch"), (f"ncu dram__bytes_read+write of this build (sources "
                                                                          f"{tj.get('src_sha16')}, .so {tj.get('so_sha16')})")
            else:
                traffic_note = (f"profiles/r02_render_traffic.json was measured on sources {tj.get('src_sha16')} / .so {tj.get('so_sha16')}, "
                                f"this is {src_sha16()} / {so_sha16()}")
        except Exception:
            pass

    sharding = "1 GPU" if world == 1 else (f"one frame, {world} row blocks of {(rows[1] - rows[0]) // W} image rows; per-ray outputs stored into "
                                          f"rank 0's frame buffers over NVLink peer memory by the fused launch, one barrier kernel per frame")
    l2 = ("per-frame working set 0.65 GB of per-sample outputs (alpha, density) + 20 MB per-ray I/O >> 126 MB L2: inputs larger than "
          "L2, no flush needed") if world == 1 else ("per-ray outputs only (17 MB per frame, written once over NVLink); the 2 MB weight "
                                                     "image stays L2-resident by design")
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
                ms_per_step=ms, higher_is_better=True, scaling="strong" if world > 1 else "weak", vs_baseline=None, dtype="bf16",
                data="synthetic", impl="ours",
                config=dict(workload=WORKLOAD + f", ONE frame per step ({sharding})",
                            rays_per_step=H * W, samples_per_ray=NS, ms_per_frame=ms, mlp="bf16 tcgen05, fp32 accumulate",
                            weights="random-init seed 0 (Xavier, as the reference)", rng="in-kernel Philox jitter", l2=l2),
                roofline=dict(bound="tensor", achieved=achieved_tf, peak=pk["tf_sustained"], unit="TFLOP/s",
                              frac=achieved_tf / pk["tf_sustained"], traffic=traffic, traffic_note=traffic_note,
                              kernel="tc::nerf_stl_forward_kernel<1,17,3> (fused render launch)",
                              kernel_ms=k_ms, kernel_share_of_step=k_ms / ms, peak_source=f"{pk['src']} bf16 sustained",
                              flop_per_sample=FLOP_PER_SAMPLE_FWD, samples_per_launch=local_samples),
                e2e=dict(value=e2e_value, unit=UNIT, h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h, ms_per_step=ms_e2e),
                gpu_launches=launches, launches_per_step=per_step, clocks=clocks, so_sha16=so_sha16(), src_sha16=src_sha16())
    if multi:
        line["multi_kernel_frame"] = multi
    if parity:
        line["fp32_parity_frame"] = parity
    if raster:
        line["mesh_rasteriser"] = raster
    if weak:
        line["weak_views"] = weak
    if train:
        line["train_step"] = train
    if not args.no_cpu_baseline and world == 1:
        try:
            line["eager_gpu_baseline"] = eager_gpu_sample(dev)
        except Exception as e:  # noqa: BLE001  (context only; never fails the bench)
            line["eager_gpu_baseline"] = dict(error=str(e)[:200])
        threads = os.cpu_count() or 1
        cstep, csamples, kind, desc = cpu_reference_step(args.cpu_rays, threads)
        cstep()
        times = []
        t_end = time.perf_counter() + 20.0
        while len(times) < 12 and (len(times) < 3 or time.perf_counter() < t_end):
            t0 = time.perf_counter()
            cstep()
            times.append(time.perf_counter() - t0)
        line["cpu_baseline"] = dict(value=csamples / (sum(times) / len(times)), unit=UNIT, cores=threads, kind=kind,
                                    sample=desc + f"; mean of {len(times)} steps after one warm-up")
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def bench_train(args, g, opt, dev, world, timed, pk):
    """C3: texture-learner step, 16 patches of 16x16 rays x 128 samples per GPU, fwd + bwd (+ grad exchange)."""
    import torch
    import torch.distributed as dist
    from texpose_b200 import compute_box, parallel, synth
    from texpose_b200.config import AttrDict, adapt_gan_opt
    from texpose_b200.model.base import summarize_loss
    B, P = 16, 16
    opt_t = adapt_gan_opt(H=128, W=128, sample_intvs=NS, device=str(dev))
    opt_t.b200 = AttrDict(mlp="bf16", rng="philox")
    pose = synth.poses(list(range(B))).to(dev)
    K = torch.tensor([[572.4114, 0, 64 - 572.4114 * 0.3 / 8], [0, 573.57043, 64 + 573.57043 * 0.2 / 8], [0, 0, 1]])
    intr = K.repeat(B, 1, 1).to(dev)
    lo, hi = [t.to(dev) for t in synth.padded_aabb()]
    zn, zf = compute_box.box_range(pose, intr, lo, hi, 128, 128, *synth.BG_RANGE)
    coords, _ = synth.patch_coords(B, P, seed=2)
    coords = coords.to(dev)
    idx = torch.arange(B, device=dev) % 8
    image = torch.rand(B, 3, 128, 128, device=dev)
    mask = (torch.rand(B, 128, 128, device=dev) > 0.3).float()
    params = [p for p in g.parameters() if p.requires_grad]
    # the one exchange of the path: N > 1 -> one kernel over NVLink peer windows (csrc/peer.cu); the NCCL allreduce of the same
    # bucket is timed beside it
    exchange = parallel.PeerGradExchange(params) if world > 1 else parallel.GradBucket(params)
    g.train()
    # the engine's own optimizer (model/nerf_adapt_st_gan.py:62-69: torch.optim.Adam over nerf + the two latent tables, optim.lr 1e-3).
    # It changes the weights every step, so every timed step also re-packs the bf16 weight images, as real training does.
    optim = torch.optim.Adam([dict(params=g.nerf.parameters(), lr=1.e-3)])
    optim.add_param_group(dict(params=g.latent_vars_light.parameters(), lr=1.e-3))
    optim.add_param_group(dict(params=g.latent_vars_trans.parameters(), lr=1.e-3))

    def make_step(bucket, optimizer=True):
        def step():
            for p in params:
                p.grad = None
            ret = g.render(opt_t, pose, intr=intr, ray_idx=coords, depth_range=(zn[:, :, None], zf[:, :, None]),
                           sample_idx=idx, mode="train")
            var = AttrDict(idx=idx, image=image, obj_mask=mask, ray_idx=coords)
            var.update(ret)
            loss = g.compute_loss(opt_t, var, mode="train")      # patch gather + render / uncert / trans_reg terms, fused
            summarize_loss(opt_t, var, loss)["all"].backward()   # seeds formed on the device in the backward
            if bucket is not None:
                bucket.allreduce_mean()
            if optimizer:
                optim.step()
        return step

    n_steps = max(10, args.steps)       # 2.4 ms each: enough steps for the max-over-ranks time to settle
    ms, _ = timed(make_step(exchange), n_steps, 3)
    ms_fb, _ = timed(make_step(exchange, optimizer=False), n_steps, 2)      # forward + backward alone (weights unchanged: nothing re-packed)
    samples = B * P * P * NS
    tf = FLOP_PER_SAMPLE_FWD_BWD * samples / (ms * 1e-3) / 1e12
    tf_fb = FLOP_PER_SAMPLE_FWD_BWD * samples / (ms_fb * 1e-3) / 1e12
    out = dict(workload="C3 train step: 4096 rays x 128 samples per GPU, fused patch loss, bf16 tcgen05 fwd + bwd (dX chain with thin "
                        "gradients, dW GEMMs), grad exchange, Adam step of the engine (heads + latents) and the re-pack of the weight images",
               value=world * samples / (ms * 1e-3), unit="samples/s", ms_per_step=ms, grad_exchange_bytes=exchange.flat.numel() * 4,
               grad_exchange="none (1 GPU)" if world == 1 else "one-kernel rank-order mean over CUDA-IPC peer windows (NVLink)",
               optimizer="torch.optim.Adam as model/nerf_adapt_st_gan.py:62-69 builds it, inside the timed step",
               tflops_per_gpu=tf, flop_per_sample=FLOP_PER_SAMPLE_FWD_BWD, frac_of_sustained_bf16=tf / pk["tf_sustained"],
               fwd_bwd_only=dict(ms_per_step=ms_fb, tflops_per_gpu=tf_fb, frac_of_sustained_bf16=tf_fb / pk["tf_sustained"],
                                 note="same step without optimizer.step(): forward + loss + backward + exchange"))
    # per-entry-point device time of the step (CUDA events around every C-ABI call, a pass of its own) and the roofline of the
    # two calls that carry the work; algorithmic bytes per 128-sample tile from DESIGN.md section 4 (K2 / K2b)
    step = make_step(None)
    with CallTimer() as ct:
        for _ in range(5):
            step()
    per = {k: sum(v) / 5 for k, v in ct.per_call_ms().items()}
    tiles = samples / 128
    fwd_ms, bwd_ms = per.get("tp_tc_nerf_stl_forward", 0.0), per.get("tp_tc_heads_backward", 0.0)
    fwd_bytes = tiles * (7 * 65536 + 4 * 4096) + samples * 36               # activation save + bitmasks + per-sample outputs
    bwd_bytes = tiles * ((2 * 65536 + 4 * 4096 + 6 * 65536) + 13 * 65536)   # chain: in + dz out; dW GEMMs: dz + activations in

    def roof(entry, t_ms, flop, nbytes, bound):
        if not t_ms:
            return dict(entry=entry, ms=None)
        tfs, gbs = flop * samples / (t_ms * 1e-3) / 1e12, nbytes / (t_ms * 1e-3) / 1e9
        return dict(entry=entry, ms=t_ms, bound=bound, achieved=tfs, unit="TFLOP/s", peak=pk["tf_sustained"], frac=tfs / pk["tf_sustained"],
                    hbm_gbs=gbs, hbm_peak=pk["hbm"], hbm_frac=gbs / pk["hbm"], algorithmic_bytes=nbytes)

    out["train_roofline"] = [
        roof("tp_tc_nerf_stl_forward (training launch: forward + activation save)", fwd_ms, FLOP_PER_SAMPLE_FWD, fwd_bytes, "tensor"),
        roof("tp_tc_heads_backward (dX chain + thin gradients, finish, six dW GEMMs, reduce: 5 launches)", bwd_ms, FLOP_PER_SAMPLE_BWD,
             bwd_bytes, "tensor + hbm"),
    ]
    out["entry_point_ms"] = {k: round(v, 4) for k, v in sorted(per.items(), key=lambda kv: -kv[1])}
    if world == 1:
        out["plain_model_train_step"] = bench_plain_train(dev, timed, samples)
        try:
            out["cuda_graph_step"] = bench_graphed_steps(g, dev, timed)
        except Exception as e:  # noqa: BLE001  (an extra block; never fails the bench)
            out["cuda_graph_step"] = dict(error=repr(e)[:300])
    if world > 1:
        exchange.check()
        # the exchanged gradients must equal the NCCL allreduce of the same bucket: one more step, then both exchanges
        make_step(None)()
        ref_bucket = parallel.GradBucket(params)
        ref_bucket.pack()
        dist.all_reduce(ref_bucket.flat, op=dist.ReduceOp.SUM)
        want = ref_bucket.flat / world
        exchange.allreduce_mean()
        got = exchange.flat[:want.numel()]
        err, scale = float((got - want).abs().max()), float(want.abs().max())
        out["exchange_vs_nccl_allreduce"] = dict(max_abs_diff=err, max_abs_value=scale,
                                                 note="peer-window rank-order mean vs NCCL SUM / world of the same packed gradients")
        if not err <= 1e-5 * max(scale, 1e-30) + 1e-12:
            raise RuntimeError(f"peer exchange differs from the NCCL allreduce: {err} (scale {scale})")
        ms_nccl, _ = timed(make_step(parallel.GradBucket(params)), n_steps, 3)
        out["ms_per_step_nccl_allreduce"] = ms_nccl
        # the exchange alone, back to back (gradients already in place): device time per call, max over ranks
        for p in params:
            p.grad = torch.ones_like(p)
        out["exchange_only_us"] = {"peer": 1e3 * timed(exchange.allreduce_mean, 50, 5)[0],
                                   "nccl": 1e3 * timed(parallel.GradBucket(params).allreduce_mean, 50, 5)[0]}
        exchange.check()
        exchange.close()
    g.eval()
    return out


def bench_graphed_steps(g, dev, timed):
    """The whole training step -- render, fused loss, backward, Adam, weight re-pack -- captured once as a CUDA graph
    (texpose_b200.train_graph.GraphedStep) beside the eager step, at BASELINE's C3 shape and at the step size of
    options/nerf_lm_adapt_gan.yaml itself (8 patches x 256 rays x 64 samples), where Python cannot issue the launches as fast as the
    GPU retires them."""
    import torch
    from texpose_b200 import compute_box, synth
    from texpose_b200.config import AttrDict, adapt_gan_opt
    from texpose_b200.model.base import summarize_loss
    from texpose_b200.train_graph import GraphedStep
    res = {}
    for name, B, P, N in (("c3_16x256x128", 16, 16, NS), ("yaml_8x256x64", 8, 16, 64)):
        o = adapt_gan_opt(H=128, W=128, sample_intvs=N, device=str(dev))
        o.batch_size = B
        o.b200 = AttrDict(mlp="bf16", rng="torch")       # torch.rand jitter: graph-safe (the Philox mode draws its seed on the host)
        pose = synth.poses(list(range(B))).to(dev)
        K = torch.tensor([[572.4114, 0, 64 - 572.4114 * 0.3 / 8], [0, 573.57043, 64 + 573.57043 * 0.2 / 8], [0, 0, 1]])
        intr = K.repeat(B, 1, 1).to(dev)
        lo, hi = [t.to(dev) for t in synth.padded_aabb()]
        zn, zf = compute_box.box_range(pose, intr, lo, hi, 128, 128, *synth.BG_RANGE)
        coords = synth.patch_coords(B, P, seed=2)[0].to(dev)
        idx = torch.arange(B, device=dev) % 8
        image = torch.rand(B, 3, 128, 128, device=dev)
        mask = (torch.rand(B, 128, 128, device=dev) > 0.3).float()

        def adam(capturable):
            op = torch.optim.Adam([dict(params=g.nerf.parameters(), lr=1.e-3)], capturable=capturable)
            op.add_param_group(dict(params=g.latent_vars_light.parameters(), lr=1.e-3))
            op.add_param_group(dict(params=g.latent_vars_trans.parameters(), lr=1.e-3))
            return op

        def fwd_bwd():
            ret = g.render(o, pose, intr=intr, ray_idx=coords, depth_range=(zn[:, :, None], zf[:, :, None]), sample_idx=idx, mode="train")
            var = AttrDict(idx=idx, image=image, obj_mask=mask, ray_idx=coords)
            var.update(ret)
            total = summarize_loss(o, var, g.compute_loss(o, var, mode="train"))["all"]
            total.backward()
            return total

        eager_optim = adam(False)

        def eager():
            eager_optim.zero_grad(set_to_none=True)
            fwd_bwd()
            eager_optim.step()

        ms_eager, _ = timed(eager, 20, 3)
        step = GraphedStep(fwd_bwd, adam(True), static=dict(coords=coords, image=image, mask=mask), warmup=3)
        ms_graph, _ = timed(lambda: step(coords=coords, image=image), 20, 3)      # inputs copied into the static buffers every step
        n = B * P * P * N
        res[name] = dict(samples_per_step=n, eager_ms_per_step=ms_eager, graph_ms_per_step=ms_graph,
                         graph_samples_per_s=n / (ms_graph * 1e-3), speedup=ms_eager / ms_graph)
    res["note"] = ("whole step (render, fused loss, backward, Adam, weight re-pack) replayed as one CUDA graph; bit-identical to the eager "
                   "run (tests/test_gpu_train_graph.py)")
    return res


def bench_plain_train(dev, timed, samples):
    """layers/nerf.py (options/nerf_lm_env.yaml) at the C3 shape: forward + composite + backward of every trunk / head parameter,
    tensor-core path (single-pass staged forward with saved activations, staged dX chain, dW GEMMs) vs the SIMT fp32 kernels."""
    import torch
    from texpose_b200.config import AttrDict, env_opt
    from texpose_b200.layers.nerf import NeRF as PlainNeRF
    B, R, N = 16, 256, NS
    g = torch.Generator().manual_seed(0)
    center = (torch.randn(B, R, 3, generator=g) * 0.02 + torch.tensor([0.3, 0.2, -0.8])).to(dev)
    ray = (torch.randn(B, R, 3, generator=g) * 0.1 + torch.tensor([0.0, 0.0, 1.0])).to(dev)
    depth = ((torch.rand(B, R, N, 1, generator=g) + torch.arange(N)[None, None, :, None]) / N * 1.2 + 0.2).to(dev)
    image = torch.rand(B, R, 3, generator=g).to(dev)
    res = {}
    for mode, steps in (("bf16", 10), ("fp32", 2)):
        opt = env_opt(device=str(dev))
        opt.b200 = AttrDict(mlp=mode)
        torch.manual_seed(0)
        m = PlainNeRF(opt).to(dev)

        optim = torch.optim.Adam([dict(params=m.parameters(), lr=1.e-3)])      # model/nerf_pretrain.py:59-62

        def step():
            optim.zero_grad()
            rgb_s, sig = m.forward_samples(opt, center, ray, depth, mode="train")
            ((m.composite(opt, ray, rgb_s, sig, depth)[0] - image) ** 2).mean().backward()
            optim.step()

        res[mode] = timed(step, steps, 2)[0]
    return dict(workload="plain NeRF (8 x 256 trunk, 286 -> 128 -> 3 head), 4096 rays x 128 samples, fwd + composite + bwd of all parameters "
                         "+ Adam step",
                ms_per_step=res["bf16"], value=samples / (res["bf16"] * 1e-3), unit="samples/s", simt_fp32_ms_per_step=res["fp32"],
                speedup_vs_simt=res["fp32"] / res["bf16"])


def main():
    args = parse()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
