"""Training step in the <= 1e-4 mode (opt.b200.mlp = 'fp32') with opt.b200.fp32_engine = 'simt' and 'tc', alternating, on three cases:
  * the pre-training engine's Graph step (model/nerf_pretrain.py; options/nerf_lm_env.yaml shapes: 2048 rays x 64 samples,
    forward + compute_loss + backward),
  * the plain model (layers/nerf.py) at 16 x 256 rays x 128 samples (forward_samples + composite + backward),
  * the static / transient / light model (yaml architecture, frozen trunk) at C3, 16 x 256 x 128, with the 1/u^2 loss.
Each case is warmed up per engine, then timed in rounds that alternate the engines (device-synchronised, CUDA events).  Needs no
reference sources.  Never a benchmark; numbers go to DESIGN.md.

    python scripts/fp32_train_time.py [--rounds 3] [--steps 5]
"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from texpose_b200 import compute_box, synth  # noqa: E402
from texpose_b200.config import AttrDict, adapt_gan_opt, env_opt  # noqa: E402

dev = "cuda:0"
ENGINES = ("simt", "tc")


def gpu_line():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi unavailable"
    return f"{torch.cuda.get_device_name(0)} | {q}"


def pretrain_case():
    from texpose_b200.model.nerf_pretrain import Graph
    H, W, B = 480, 640, 2
    pose = synth.poses([0, 1]).to(dev)
    intr = synth.intrinsics(B).to(dev)
    lo, hi = [t.to(dev) for t in synth.padded_aabb()]
    zn, zf = compute_box.box_range(pose, intr, lo, hi, H, W, *synth.BG_RANGE)
    gen = torch.Generator().manual_seed(3)
    var0 = dict(idx=torch.arange(B), pose=pose, pose_init=pose, intr=intr, z_near=zn, z_far=zf,
                image=torch.rand(B, 3, H, W, generator=gen).to(dev), obj_mask=(zf < 29).view(B, H, W).float(),
                depth_gt=(7.5 + torch.rand(B, H, W, generator=gen)).to(dev))
    steps = {}
    for engine in ENGINES:
        opt = env_opt(H=H, W=W, sample_intvs=64, device=dev)
        opt.nerf.rand_rays = 2048
        opt.loss_weight = AttrDict(render=0, mask=-1, depth=-1)
        opt.data.erode_mask_loss = False
        opt.b200 = AttrDict(mlp="fp32", fp32_engine=engine)
        torch.manual_seed(0)
        g = Graph(opt).to(dev)

        def step(g=g, opt=opt):
            for p in g.parameters():
                p.grad = None
            var = g.forward(opt, AttrDict(var0), mode="train")
            loss = g.compute_loss(opt, var, mode="train")
            sum(10 ** float(opt.loss_weight[k]) * loss[k] for k in loss).backward()

        steps[engine] = step
    return "pre-training Graph step, 2048 x 64", steps


def _c3_inputs():
    B, R, N = 16, 256, 128
    g = torch.Generator().manual_seed(0)
    center = (torch.randn(B, R, 3, generator=g) * 0.02 + torch.tensor([0.3, 0.2, -0.8])).to(dev)
    ray = (torch.randn(B, R, 3, generator=g) * 0.1 + torch.tensor([0.0, 0.0, 1.0])).to(dev)
    depth = ((torch.rand(B, R, N, 1, generator=g) + torch.arange(N)[None, None, :, None]) / N * 1.2 + 0.2).to(dev)
    image = torch.rand(B, R, 3, generator=g).to(dev)
    return center, ray, depth, image


def plain_case():
    from texpose_b200.layers.nerf import NeRF
    center, ray, depth, image = _c3_inputs()
    steps = {}
    for engine in ENGINES:
        opt = env_opt(device=dev)
        opt.b200 = AttrDict(mlp="fp32", fp32_engine=engine)
        torch.manual_seed(0)
        m = NeRF(opt).to(dev)

        def step(m=m, opt=opt):
            for p in m.parameters():
                p.grad = None
            rgb_s, sig = m.forward_samples(opt, center, ray, depth, mode="train")
            comp = m.composite(opt, ray, rgb_s, sig, depth)
            (((comp[0] - image) ** 2).mean() + 0.1 * comp[1].mean() + 0.01 * sig.mean()).backward()

        steps[engine] = step
    return "plain model step, 16 x 256 x 128", steps


def stl_case():
    from texpose_b200.layers.nerf_static_transient_light import NeRF
    center, ray, depth, image = _c3_inputs()
    B = center.shape[0]
    lt, ll = [t.to(dev) for t in synth.latents(B)]
    steps = {}
    for engine in ENGINES:
        opt = adapt_gan_opt(device=dev)
        opt.b200 = AttrDict(mlp="fp32", fp32_engine=engine)
        torch.manual_seed(0)
        m = NeRF(opt).to(dev)
        for p in m.mlp_feat.parameters():
            p.requires_grad_(False)
        lt_g, ll_g = lt.clone().requires_grad_(True), ll.clone().requires_grad_(True)

        def step(m=m, opt=opt, lt_g=lt_g, ll_g=ll_g):
            for p in list(m.parameters()) + [lt_g, ll_g]:
                p.grad = None
            s = m.forward_samples(opt, center, ray, depth, lt_g, ll_g, mode="train")
            comp = m.composite(opt, ray, *s[:2], depth, s[2])
            rgb, unc = comp[0], comp[8]
            (((image - rgb) ** 2 / unc ** 2).mean() + (5 + torch.log(unc ** 2).mean() / 2) + 0.01 * s[1][..., -1].mean()).backward()

        steps[engine] = step
    return "static/transient/light step (yaml), 16 x 256 x 128", steps


def timed(fn, steps):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    a = ap.parse_args()
    print("GPU:", gpu_line())
    for make in (pretrain_case, plain_case, stl_case):
        name, steps = make()
        for engine in ENGINES:
            for _ in range(a.warmup):
                steps[engine]()
        ms = {e: [] for e in ENGINES}
        for _ in range(a.rounds):
            for engine in ENGINES:
                ms[engine].append(timed(steps[engine], a.steps))
        best = {e: min(v) for e, v in ms.items()}
        print(f"{name}: " + ", ".join(f"{e} {best[e]:.2f} ms (rounds: {' '.join(f'{x:.2f}' for x in ms[e])})" for e in ENGINES)
              + f"  -> tc / simt = {best['tc'] / best['simt']:.2f}", flush=True)
        del steps
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
