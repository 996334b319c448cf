"""Frame time of mask-prior eval frames: the existing Graph.nerf_forward(mode='eval_noalign') (render_by_slices: per view a host
`nonzero`, one render launch and eleven scatters into defaults) against Graph.render_masked (one list build, one defaults fill,
one render launch for all B views).

    python scripts/masked_render_time.py [--frames 4] [--rounds 3] [--out profiles/r05_masked_render_n1.log]

Synthetic C2 views (synth.poses([0|3|5|...]), 480 x 640), object mask = the pixels whose ray hits the padded AABB; N = 128 and 64,
B = 1 and 8, opt.b200.mlp = 'bf16' and 'fp32'; midpoint depths, so both paths compute the same frame (the largest difference is
printed: 0 in bf16, where both run the lock-step render launch; in fp32 nerf_forward runs the multi-kernel path and render_masked the
staged render launch, whose compositing sums in another order).
The two paths alternate round by round after a warm-up of both, timed with CUDA events over `frames` frames per round.
With several GPUs, eval frames through parallel.FrameGather at 1 / 2 / 4 / 8 ranks (one process per GPU) and the per-rank
object pixels of row blocks against the per-rank list slots; on a one-GPU box those lines say "not measured".
The card's name and power limit are read in the same run (nvidia-smi --query-gpu, read-only)."""
from __future__ import annotations

import argparse
import os
import socket
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

H, W = 480, 640
SEEDS = [0, 3, 5, 0, 3, 5, 0, 3]


def _setup(mlp, N, B, dev):
    from texpose_b200 import compute_box, ops, synth
    from texpose_b200.config import AttrDict, adapt_gan_opt
    from texpose_b200.model.nerf_adapt_st_gan import Graph
    opt = adapt_gan_opt(H=H, W=W, sample_intvs=N, device=str(dev))
    opt.b200 = AttrDict(mlp=mlp)
    opt.nerf.sample_stratified = False
    torch.manual_seed(0)
    g = Graph(opt, n_train_images=8).to(dev).eval()
    pose, intr = synth.poses(SEEDS[:B]).to(dev), synth.intrinsics(B).to(dev)
    lo, hi = [t.to(dev) for t in synth.padded_aabb()]
    zn, zf = compute_box.box_range(pose, intr, lo, hi, H, W, *synth.BG_RANGE)
    from texpose_b200 import camera
    kinv, pinv = camera.view_matrices(pose, intr)
    center, ray = ops.raygen(kinv, pinv, H, W, 0.5)
    _, _, valid = ops.aabb_intersect(lo.reshape(1, 3), hi.reshape(1, 3), center, ray)
    mask = valid.float()
    from texpose_b200.config import AttrDict as AD
    var = AD(pose=pose, intr=intr, z_near=zn, z_far=zf, obj_mask=mask.view(B, H * W, 1), pose_anchor=synth.poses([0, 3, 5, 7]).to(dev))
    return opt, g, var, mask


def _time(fn, frames):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(frames):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / frames


def single_gpu(frames, rounds, log):
    dev = torch.device("cuda", 0)
    keys = ("rgb", "rgb_static", "depth", "opacity", "uncert", "alpha_static", "density")
    for mlp in ("bf16", "fp32"):
        for N in (128, 64):
            for B in (1, 8):
                opt, g, var, mask = _setup(mlp, N, B, dev)
                idx = torch.zeros(B, dtype=torch.int64, device=dev) if B > 1 else torch.tensor(0, device=dev)
                dr = (var.z_near[:, :, None], var.z_far[:, :, None])
                with torch.no_grad():
                    def old():
                        g.nerf_forward(opt, var, mode="eval_noalign")

                    def new():
                        return g.render_masked(opt, var.pose, var.intr, dr, mask, sample_idx=idx, mode="eval_noalign")
                    torch.manual_seed(1)
                    old()
                    torch.manual_seed(1)
                    R_dist = __import__("texpose_b200.model.nerf_adapt_st_gan", fromlist=["x"]).rotation_distance(
                        var.pose[:, None, :3, :3], var.pose_anchor[None, :, :3, :3])
                    k = int(opt.render.N_candidate)
                    idx = torch.topk(R_dist, k=k, dim=1, largest=False, sorted=True)[1][:, int(torch.randperm(k)[0])]
                    if B == 1:
                        idx = idx[0]
                    got = new()
                    diff = max(float((got[key] - var[key]).abs().max()) for key in keys)
                    note = ""
                    if B > 1:      # the same views one call each: K^-1 is then inverted per view, as render_by_slices does
                        per_view = [g.render_masked(opt, var.pose[i:i + 1], var.intr[i:i + 1], tuple(d[i:i + 1] for d in dr), mask[i:i + 1],
                                                    sample_idx=idx[i], mode="eval_noalign") for i in range(B)]
                        d1 = max(float((torch.cat([r[key] for r in per_view]) - var[key]).abs().max()) for key in keys)
                        kb = torch.linalg.inv_ex(var.intr.float())[0]
                        ks = torch.cat([torch.linalg.inv_ex(var.intr[i:i + 1].float())[0] for i in range(B)])
                        note = (f"; views rendered one call each: max |difference| {d1:.2e}; batched vs per-view K^-1 (torch) "
                                f"max |difference| {float((kb - ks).abs().max()):.2e}")
                    t_old, t_new = [], []
                    for _ in range(rounds):
                        torch.manual_seed(1)
                        t_old.append(_time(old, frames))
                        t_new.append(_time(new, frames))
                    n_obj = int(mask.sum().item())
                    log(f"{mlp:4s} N={N:3d} B={B}: object pixels {n_obj} ({100.0 * n_obj / (B * H * W):.1f} %); "
                        f"nerf_forward(eval_noalign) {min(t_old):8.2f} ms/frame-batch (rounds {', '.join(f'{t:.2f}' for t in t_old)}); "
                        f"render_masked {min(t_new):8.2f} ms (rounds {', '.join(f'{t:.2f}' for t in t_new)}); "
                        f"speed-up {min(t_old) / min(t_new):.2f}x; max |difference| of the outputs {diff:.2e}{note}")
                del g
                torch.cuda.empty_cache()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gather_worker(rank, world, port, frames, rounds, out):
    import torch.distributed as dist
    from texpose_b200 import ops, parallel
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        for mlp in ("bf16", "fp32"):
            opt, g, var, mask = _setup(mlp, 128, 1, dev)
            dr = (var.z_near[:, :, None], var.z_far[:, :, None])
            fg = parallel.FrameGather(opt, device=dev, timeout_ms=60000)
            idx = torch.tensor(0, device=dev)
            with torch.no_grad():
                def frame():
                    fg.render(g, opt, var.pose, var.intr, dr, sample_idx=idx, mode="eval", object_mask=mask)
                frame()
                torch.cuda.synchronize(dev)
                ts = []
                for _ in range(rounds):
                    dist.barrier()
                    ts.append(_time(frame, frames))
                fg.check()
                b, e = fg.rows
                rows_obj = int(mask[0, b:e].sum().item())
                _, n_slots, _ = ops.mask_ray_list(mask, 128)
                T = int(n_slots.item()) // 2
                slots = (T * (rank + 1) // world - T * rank // world) * 2
            out[(mlp, rank)] = (min(ts), rows_obj, slots)
            fg.close()
    finally:
        dist.destroy_process_group()


def multi_gpu(frames, rounds, log):
    import torch.multiprocessing as mp
    n = torch.cuda.device_count()
    for world in (1, 2, 4, 8):
        if world > n:
            log(f"FrameGather eval frame at {world} ranks: not measured ({n} GPU{'s' if n > 1 else ''} on this box)")
            continue
        mgr = mp.Manager()
        out = mgr.dict()
        mp.spawn(_gather_worker, args=(world, _free_port(), frames, rounds, out), nprocs=world, join=True)
        for mlp in ("bf16", "fp32"):
            t = max(out[(mlp, r)][0] for r in range(world))
            rows = [out[(mlp, r)][1] for r in range(world)]
            slots = [out[(mlp, r)][2] for r in range(world)]
            log(f"FrameGather eval frame, {mlp}, N=128, {world} ranks: {t:.2f} ms/frame (slowest rank); object pixels of the row "
                f"blocks {rows} (max/mean {max(rows) / max(1e-9, sum(rows) / world):.2f}); list slots per rank {slots}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=4)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("masked_render_time.py measures on the GPU; no CUDA device found")
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip()
    log(f"GPUs (name, power limit, max SM clock): {q.splitlines() if q else 'unknown'}")
    log(f"torch {torch.__version__}, {H}x{W}, frames per round {a.frames}, rounds {a.rounds}")
    single_gpu(a.frames, a.rounds, log)
    multi_gpu(a.frames, a.rounds, log)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
