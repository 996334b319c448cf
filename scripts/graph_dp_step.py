"""Data-parallel texture-learner step at the reference yaml's step size (8 patches x 256 rays x 64 samples PER GPU), one process per
GPU, three arms: eager (render, fused loss, backward, NCCL gradient allreduce of parallel.GradBucket, Adam); the same step captured
as one CUDA graph per rank (texpose_b200.train_graph.GraphedStep) with the NCCL allreduce inside the capture; and the same step
captured with the peer-window exchange parallel.PeerGradExchange(capturable=True) inside the capture instead.  Checks that all
ranks hold the same weights afterwards.  torchrun --nproc-per-node N scripts/graph_dp_step.py [--arms eager,nccl_graph,peer_graph].
Never a benchmark.

A process group whose NCCL communicator was captured into a live CUDA graph does not tear down cleanly (a run hung in
destroy_process_group), so a run with the nccl_graph arm leaves through os._exit; a run without it tears the group down normally."""
import argparse
import os
import subprocess
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from texpose_b200 import compute_box, parallel, synth  # noqa: E402
from texpose_b200.config import AttrDict, adapt_gan_opt  # noqa: E402
from texpose_b200.model.base import summarize_loss  # noqa: E402
from texpose_b200.model.nerf_adapt_st_gan import Graph  # noqa: E402
from texpose_b200.train_graph import GraphedStep  # noqa: E402

ARMS = ("eager", "nccl_graph", "peer_graph")
ap = argparse.ArgumentParser()
ap.add_argument("--arms", default=",".join(ARMS))
ap.add_argument("--steps", type=int, default=200)
args = ap.parse_args()
arms = [a for a in args.arms.split(",") if a]
if not set(arms) <= set(ARMS):
    raise SystemExit(f"--arms: choose from {ARMS}")

rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if world > 1:
    dist.init_process_group("nccl", device_id=dev)
elif "peer_graph" in arms:              # PeerGradExchange sets up through a process group: a single-process one, no sockets
    dist.init_process_group("gloo", store=dist.HashStore(), rank=0, world_size=1)
B, P, N = 8, 16, 64
opt = adapt_gan_opt(H=128, W=128, sample_intvs=N, device=str(dev))
opt.batch_size = B
opt.b200 = AttrDict(mlp="bf16", rng="torch")
pose = synth.poses(list(range(rank * B, rank * B + B))).to(dev)            # every rank its own views and patches
K = torch.tensor([[572.4114, 0, 64 - 572.4114 * 0.3 / 8], [0, 573.57043, 64 + 573.57043 * 0.2 / 8], [0, 0, 1]])
intr = K.repeat(B, 1, 1).to(dev)
lo, hi = [t.to(dev) for t in synth.padded_aabb()]
zn, zf = compute_box.box_range(pose, intr, lo, hi, 128, 128, *synth.BG_RANGE)
coords = synth.patch_coords(B, P, seed=2 + rank)[0].to(dev)
idx = torch.arange(B, device=dev)
gen = torch.Generator().manual_seed(10 + rank)
image = torch.rand(B, 3, 128, 128, generator=gen).to(dev)
mask = (torch.rand(B, 128, 128, generator=gen) > 0.3).float().to(dev)


def build(capturable, peer=False):
    torch.manual_seed(0)                                                   # same weights on every rank
    g = Graph(opt, n_train_images=B).to(dev).train()
    op = torch.optim.Adam([dict(params=g.nerf.parameters(), lr=1.e-3)], capturable=capturable)
    op.add_param_group(dict(params=g.latent_vars_light.parameters(), lr=1.e-3))
    op.add_param_group(dict(params=g.latent_vars_trans.parameters(), lr=1.e-3))
    params = [p for p in g.parameters() if p.requires_grad]
    bucket = parallel.PeerGradExchange(params, capturable=True) if peer else parallel.GradBucket(params)

    def fwd_bwd():
        ret = g.render(opt, pose, intr=intr, ray_idx=coords, depth_range=(zn[:, :, None], zf[:, :, None]), sample_idx=idx, mode="train")
        var = AttrDict(idx=idx, image=image, obj_mask=mask, ray_idx=coords)
        var.update(ret)
        total = summarize_loss(opt, var, g.compute_loss(opt, var, mode="train"))["all"]
        total.backward()
        bucket.allreduce_mean()
        return total

    return g, op, fwd_bwd, bucket


def timed(fn, steps=args.steps, warm=5):
    for _ in range(warm):
        fn()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / steps], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t)


def spread(g):
    """max over parameters of |mine - rank 0's|"""
    worst = 0.0
    for p in g.parameters():
        ref = p.detach().clone()
        if world > 1:
            dist.broadcast(ref, 0)
        worst = max(worst, float((ref - p.detach()).abs().max()))
    return worst


results = []
for arm in arms:
    if arm == "eager":
        g, op, fb, _ = build(False)

        def run(op=op, fb=fb):
            op.zero_grad(set_to_none=True)
            fb()
            op.step()
    else:
        g, op, fb, bucket = build(True, peer=arm == "peer_graph")
        step = GraphedStep(fb, op, static=dict(coords=coords, image=image, mask=mask), warmup=3)
        run = lambda step=step: step(coords=coords, image=image, mask=mask)     # noqa: E731
    ms = timed(run)
    results.append((arm, ms, spread(g)))
    if arm == "peer_graph":
        bucket.check()
        bucket.close()
if rank == 0:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(local)],
                       capture_output=True, text=True)
    n = world * B * P * P * N
    print(f"{world} x {torch.cuda.get_device_name(dev)} (nvidia-smi name, power limit: {q.stdout.strip() or 'unavailable'})")
    print(f"{B} x {P * P} rays x {N} samples per GPU and step, gradient exchange inside the step, {args.steps} timed steps:")
    if world == 1:
        print("  (1 process: GradBucket returns without an exchange, so eager / nccl_graph run no exchange; peer_graph runs its"
              " stage + one-rank exchange)")
    for arm, ms, s in results:
        print(f"  {arm:<10} {ms:.3f} ms per step ({n / ms / 1e3:.1f} M samples/s), weights differ across ranks by at most {s!r}")
sys.stdout.flush()
torch.cuda.synchronize()
if world > 1:
    dist.barrier()
    torch.cuda.synchronize()
if "nccl_graph" in arms and world > 1:
    os._exit(0)            # a captured NCCL communicator: leave without the teardown (module docstring)
if dist.is_initialized():
    dist.destroy_process_group()
if rank == 0:
    print("process group destroyed normally")
