"""Frame time of the staged kernel's render launch (tp_tc32_render_forward) against the multi-kernel frame it can replace.

    python scripts/staged_render_time.py [--frames 6] [--rounds 3] [--out DIR]

Per configuration, in one process: the multi-kernel frame Graph.render_by_slices(mode='val') (raygen, bounds, sample_depth, per-ray
bias table, tp_tc32_forward / the lock-step kernel, compositing) and the one-launch frame parallel.FrameGather.render at world 1,
alternated round by round after a warm-up of both, timed with CUDA events over `frames` frames per round.  Configurations:
  c2_parity       adaptation Graph, nerf_lm_adapt_gan.yaml model, 480 x 640 x 128, opt.b200.mlp = 'fp32' (<= 1e-4 mode)
  pretrain_bf16   pre-training Graph, nerf_lm_env.yaml plain model, 480 x 640 x 64, 'bf16' (multi-kernel: the lock-step kernel;
                  one launch: the staged kernel's single pass)
  pretrain_fp32   the same in the <= 1e-4 mode
FrameGather at 2 / 4 / 8 ranks: one process per GPU, where that many GPUs exist; otherwise the line says "not measured".
The card's name, power limit and SM clock limit are read in the same run (nvidia-smi --query-gpu, read-only)."""
from __future__ import annotations

import argparse
import os
import socket
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

H, W = 480, 640
CONFIGS = {"c2_parity": ("adapt", "fp32", 128), "pretrain_bf16": ("pretrain", "bf16", 64), "pretrain_fp32": ("pretrain", "fp32", 64)}


def _setup(name, dev):
    from texpose_b200 import compute_box, parallel, synth
    from texpose_b200.config import AttrDict, adapt_gan_opt, env_opt
    from texpose_b200.model.nerf_adapt_st_gan import Graph as AdaptGraph
    from texpose_b200.model.nerf_pretrain import Graph as PretrainGraph
    engine, mlp, N = CONFIGS[name]
    opt = (adapt_gan_opt if engine == "adapt" else env_opt)(H=H, W=W, sample_intvs=N, device=str(dev))
    opt.b200 = AttrDict(mlp=mlp)
    opt.nerf.sample_stratified = False      # midpoints: both frames see the same depths, so their outputs can be compared
    torch.manual_seed(0)
    g = (AdaptGraph(opt, n_train_images=2) if engine == "adapt" else PretrainGraph(opt)).to(dev).eval()
    pose, intr = synth.poses([0]).to(dev), synth.intrinsics(1).to(dev)
    lo, hi = [t.to(dev) for t in synth.padded_aabb()]
    zn, zf = compute_box.box_range(pose, intr, lo, hi, H, W, *synth.BG_RANGE)
    keys = parallel.PER_RAY_KEYS if engine == "adapt" else parallel.PRETRAIN_KEYS
    return opt, g, pose, intr, (zn[:, :, None], zf[:, :, None]), keys


def _time(fn, frames):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(frames):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / frames


def single_gpu(name, frames, rounds, log):
    from texpose_b200 import parallel
    dev = torch.device("cuda", 0)
    opt, g, pose, intr, dr, keys = _setup(name, dev)
    fg = parallel.FrameGather(opt, keys=keys, device=dev)
    multi = lambda: g.render_by_slices(opt, pose, intr=intr, depth_range=dr, mode="val")
    one = lambda: fg.render(g, opt, pose, intr, dr)
    with torch.no_grad():
        for fn in (multi, one):      # warm-up: module loads, weight images, scratch buffers
            fn()
            fn()
        torch.cuda.synchronize()
        t_multi, t_one = [], []
        for _ in range(rounds):
            t_multi.append(_time(multi, frames))
            t_one.append(_time(one, frames))
        a = multi()
        frame, _ = one()
        torch.cuda.synchronize()
        diff = max(float((frame[k] - a[k]).abs().max()) for k in keys)
    fg.close()
    log(f"{name}: multi-kernel render_by_slices {min(t_multi):8.2f} ms/frame (rounds {', '.join(f'{t:.2f}' for t in t_multi)})")
    log(f"{name}: FrameGather world 1        {min(t_one):8.2f} ms/frame (rounds {', '.join(f'{t:.2f}' for t in t_one)})"
        f"  speed-up {min(t_multi) / min(t_one):.3f}x  max|diff| of the per-ray outputs {diff:.2e}")
    return min(t_one)


def _worker(rank, world, port, name, frames, rounds, ret):
    import torch.distributed as dist
    from texpose_b200 import parallel
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        opt, g, pose, intr, dr, keys = _setup(name, dev)
        fg = parallel.FrameGather(opt, keys=keys, device=dev, timeout_ms=60000)
        one = lambda: fg.render(g, opt, pose, intr, dr)
        with torch.no_grad():
            one()
            one()
            torch.cuda.synchronize()
            dist.barrier()
            times = [_time(one, frames) for _ in range(rounds)]      # every rank's frames end at the root's barrier
        fg.check()
        fg.close()
        if rank == 0:
            ret["ms"] = min(times)
    finally:
        dist.destroy_process_group()


def multi_gpu(name, world, frames, rounds):
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, port, name, frames, rounds, ret), nprocs=world, join=True)
    return ret["ms"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=6)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--configs", default=",".join(CONFIGS))
    ap.add_argument("--out", default=None, help="directory of the log (one file per configuration)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("staged_render_time.py measures on a GPU; none is visible")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    n_gpu = torch.cuda.device_count()
    for name in args.configs.split(","):
        lines = []

        def log(s):
            print(s, flush=True)
            lines.append(s)

        log(f"# scripts/staged_render_time.py --frames {args.frames} --rounds {args.rounds}  ({time.strftime('%Y-%m-%d %H:%M:%S')})")
        for i, c in enumerate(card):
            log(f"# GPU {i}: {c}  (name, power limit, max SM clock)")
        engine, mlp, N = CONFIGS[name]
        log(f"# {name}: {engine} engine, {H} x {W} x {N}, opt.b200.mlp = {mlp!r}; CUDA-event time per frame, best of the rounds")
        t1 = single_gpu(name, args.frames, args.rounds, log)
        for world in (2, 4, 8):
            if world > n_gpu:
                log(f"{name}: FrameGather world {world}: not measured ({n_gpu} GPU(s) visible)")
                continue
            t = multi_gpu(name, world, args.frames, args.rounds)
            log(f"{name}: FrameGather world {world}        {t:8.2f} ms/frame  scaling {t1 / t:.2f}x over world 1")
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, f"r04_staged_render_{name}.log"), "w") as f:
                f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
