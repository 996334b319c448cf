"""Eager vs one-CUDA-graph training steps (texpose_b200.train_graph.GraphedStep), one process, warmed shapes, CUDA events:
  * the pre-training step (model.nerf_pretrain.Graph, options/nerf_lm_env.yaml: 2048 rays x 64 samples, trunk and head train) in
    bf16 and in the <= 1e-4 mode on the tensor cores (opt.b200.mlp = 'fp32', fp32_engine = 'tc');
  * the adaptation step in the <= 1e-4 mode at the yaml size (8 patches x 256 rays x 64 samples).
Best of 3 rounds, eager and graphed alternated within each round.  The eager step is what a training loop issues per step:
render(mode='train'), compute_loss, backward, Adam.  The graphed step copies the batch into the static buffers and replays;
the pre-training ray subset (get_ray_idx, torch.randperm) is drawn eagerly in both arms.  Prints the GPU name and power limit.
Never a benchmark; the log goes to profiles/r07_graph_train_time.log."""
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from texpose_b200 import compute_box, synth  # noqa: E402
from texpose_b200.config import AttrDict, adapt_gan_opt, env_opt  # noqa: E402
from texpose_b200.model import nerf_adapt_st_gan, nerf_pretrain  # noqa: E402
from texpose_b200.model.base import summarize_loss  # noqa: E402
from texpose_b200.train_graph import GraphedStep  # noqa: E402

dev = "cuda:0"
H, W = 480, 640
STEPS, ROUNDS = 50, 3


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def timed(fn, steps=STEPS):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(steps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def scene(B):
    pose = synth.poses(list(range(B))).to(dev)
    intr = synth.intrinsics(B).to(dev)
    lo, hi = [t.to(dev) for t in synth.padded_aabb()]
    zn, zf = compute_box.box_range(pose, intr, lo, hi, H, W, *synth.BG_RANGE)
    return pose, intr, zn, zf


def pretrain_arms(b200):
    B = 2
    opt = env_opt(H=H, W=W, sample_intvs=64, device=dev)
    opt.nerf.rand_rays = 2048
    opt.loss_weight = AttrDict(render=0, mask=-1, depth=-1)
    opt.data.erode_mask_loss = False
    opt.b200 = AttrDict(b200, rng="torch")
    pose, intr, zn, zf = scene(B)
    gen = torch.Generator().manual_seed(3)
    fixed = dict(image=torch.rand(B, 3, H, W, generator=gen).to(dev), obj_mask=(zf < 29).view(B, H, W).float(),
                 depth_gt=(7.5 + torch.rand(B, H, W, generator=gen)).to(dev))
    idx = torch.arange(B, device=dev)

    def make():
        torch.manual_seed(0)
        g = nerf_pretrain.Graph(opt).to(dev).train()
        optim = torch.optim.Adam(g.nerf.parameters(), lr=5e-4, capturable=True)
        static = dict(ray_idx=nerf_pretrain.Graph.get_ray_idx(opt, AttrDict(idx=[0] * B)).ray_idx)

        def fn():
            var = AttrDict(idx=idx, pose=pose, intr=intr, z_near=zn, z_far=zf, ray_idx=static["ray_idx"], **fixed)
            var.update(g.render(opt, pose, intr=intr, ray_idx=var.ray_idx, depth_range=(zn[:, :, None], zf[:, :, None]), mode="train"))
            loss = g.compute_loss(opt, var, mode="train")
            total = sum(10 ** float(opt.loss_weight[k]) * loss[k] for k in loss)
            total.backward()
            return total
        return g, optim, static, fn

    rays = lambda: nerf_pretrain.Graph.get_ray_idx(opt, AttrDict(idx=[0] * B)).ray_idx      # forward()'s draw, eager in both arms
    _, optim_e, static_e, fn_e = make()

    def eager(i):
        static_e["ray_idx"] = rays()
        optim_e.zero_grad(set_to_none=True)
        fn_e()
        optim_e.step()

    _, optim_g, static_g, fn_g = make()
    step = GraphedStep(fn_g, optim_g, static=static_g, warmup=3)

    def graphed(i):
        step(ray_idx=rays())
    return eager, graphed


def adapt_arms(b200):
    B, P = 8, 16
    opt = adapt_gan_opt(H=H, W=W, sample_intvs=64, device=dev)
    opt.batch_size, opt.patch_size = B, P
    opt.b200 = AttrDict(b200, rng="torch")
    pose, intr, zn, zf = scene(B)
    gen = torch.Generator().manual_seed(4)
    image = torch.rand(B, 3, H, W, generator=gen).to(dev)
    mask = (zf < 29).view(B, H, W).float()
    idx = torch.arange(B, device=dev)

    def make():
        torch.manual_seed(0)
        g = nerf_adapt_st_gan.Graph(opt, n_train_images=B).to(dev).train()
        optim = torch.optim.Adam([dict(params=g.nerf.parameters(), lr=1.e-3)], capturable=True)
        optim.add_param_group(dict(params=g.latent_vars_light.parameters(), lr=1.e-3))
        optim.add_param_group(dict(params=g.latent_vars_trans.parameters(), lr=1.e-3))
        static = dict(coords=synth.patch_coords(B, P, seed=5)[0].to(dev))

        def fn():
            ret = g.render(opt, pose, intr=intr, ray_idx=static["coords"], depth_range=(zn[:, :, None], zf[:, :, None]),
                           sample_idx=idx, mode="train")
            var = AttrDict(idx=idx, image=image, obj_mask=mask, ray_idx=static["coords"])
            var.update(ret)
            total = summarize_loss(opt, var, g.compute_loss(opt, var, mode="train"))["all"]
            total.backward()
            return total
        return g, optim, static, fn

    coords = [synth.patch_coords(B, P, seed=10 + i)[0].to(dev) for i in range(8)]
    _, optim_e, static_e, fn_e = make()

    def eager(i):
        static_e["coords"].copy_(coords[i % 8])
        optim_e.zero_grad(set_to_none=True)
        fn_e()
        optim_e.step()

    _, optim_g, static_g, fn_g = make()
    step = GraphedStep(fn_g, optim_g, static=static_g, warmup=3)

    def graphed(i):
        step(coords=coords[i % 8])
    return eager, graphed


def main():
    print("GPU:", gpu_info())
    print(f"torch {torch.__version__}, {STEPS} steps per timed window, best of {ROUNDS} rounds, eager / graphed alternated")
    cases = [("pre-training step, 2048 rays x 64 samples, bf16", lambda: pretrain_arms(dict(mlp="bf16"))),
             ("pre-training step, 2048 rays x 64 samples, fp32 on the tensor cores", lambda: pretrain_arms(dict(mlp="fp32", fp32_engine="tc"))),
             ("adaptation step, 8 x 256 rays x 64 samples, fp32 on the tensor cores",
              lambda: adapt_arms(dict(mlp="fp32", fp32_engine="tc")))]
    for name, build in cases:
        eager, graphed = build()
        for i in range(5):          # warm every shape of both arms
            eager(i)
            graphed(i)
        te, tg = [], []
        for _ in range(ROUNDS):
            te.append(timed(eager))
            tg.append(timed(graphed))
        print(f"{name}: eager {min(te):.3f} ms, one graph {min(tg):.3f} ms, x{min(te) / min(tg):.2f}   "
              f"(rounds: eager {', '.join(f'{t:.3f}' for t in te)}; graph {', '.join(f'{t:.3f}' for t in tg)})")
        del eager, graphed
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
    if torch.cuda.device_count() < 2:
        print(f"data-parallel arm (2 / 4 / 8 GPUs): not measured ({torch.cuda.device_count()} GPU in this run)")
    else:
        print("data-parallel arm (2 / 4 / 8 GPUs): not measured by this script (one process)")


if __name__ == "__main__":
    main()
