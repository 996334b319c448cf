"""BASELINE.json configs[2] ("C3") as a parity problem: texture-learner step on 16 patches of 16x16 rays x 128 samples,
8 latent rows, bf16 tensor-core MLP with the fused composite / loss backward -- the CUDA path and the CPU oracle on the same
seeded inputs.  Shared by the C3 parity test and the data-parallel equivalence test (test infrastructure only)."""
import torch

from oracle import texpose_oracle as O
from texpose_b200 import camera, compute_box, synth
from texpose_b200.config import AttrDict, adapt_gan_opt
from texpose_b200.model import base
from texpose_b200.model.nerf_adapt_st_gan import Graph

B, P, N, H, W, N_LATENT_ROWS = 16, 16, 128, 128, 128, 8


def inputs():
    pose = synth.poses(list(range(B)))
    K = torch.tensor([[572.4114, 0, W / 2 - 572.4114 * 0.3 / 8], [0, 573.57043, H / 2 + 573.57043 * 0.2 / 8], [0, 0, 1]])
    intr = K.repeat(B, 1, 1)
    coords, _ = synth.patch_coords(B, P, seed=2)
    g = torch.Generator().manual_seed(8)
    image = torch.rand(B, 3, H, W, generator=g)
    mask = (torch.rand(B, H, W, generator=g) > 0.3).float()
    idx = torch.arange(B) % N_LATENT_ROWS
    return AttrDict(pose=pose, intr=intr, coords=coords, image=image, mask=mask, idx=idx)


def graph(dev, precision="bf16"):
    opt = adapt_gan_opt(H=H, W=W, sample_intvs=N, device=dev)
    opt.b200 = AttrDict(mlp=precision)
    opt.batch_size, opt.patch_size = B, P
    torch.manual_seed(0)
    return opt, Graph(opt, n_train_images=N_LATENT_ROWS).to(dev)


def named_trainables(g):
    out = list(g.nerf.mlp_rgb.named_parameters(prefix="mlp_rgb")) + list(g.nerf.mlp_trans.named_parameters(prefix="mlp_trans"))
    return out + [("latent_vars_trans.weight", g.latent_vars_trans.weight), ("latent_vars_light.weight", g.latent_vars_light.weight)]


def cuda_step(opt, g, inp, images, dev, seed):
    """One training step of the CUDA path on the images `images` (a slice of the batch).  Returns ({name: grad}, rand, loss)."""
    sl = images
    pose, intr = inp.pose[sl].to(dev), inp.intr[sl].to(dev)
    lo, hi = [t.to(dev) for t in synth.padded_aabb()]
    coords = inp.coords[sl].to(dev)
    idx = inp.idx[sl].to(dev)
    for _, p in named_trainables(g):
        p.grad = None
    n = len(idx)
    # K^-1 / pose^-1 with the CPU reference's LAPACK bits, so rays and bounds are bit-identical to the oracle's (the 2^9 pi
    # positional encoding amplifies an ulp of difference in a ray to ~1e-3 at the outputs: DESIGN.md section 2)
    host_matrices = camera.HOST_MATRICES
    camera.HOST_MATRICES = True
    try:
        zn, zf = compute_box.box_range(pose, intr, lo, hi, H, W, *synth.BG_RANGE)
        torch.manual_seed(seed)
        ret = g.render(opt, pose, intr=intr, ray_idx=coords, depth_range=(zn[:, :, None], zf[:, :, None]), sample_idx=idx, mode="train")
    finally:
        camera.HOST_MATRICES = host_matrices
    torch.manual_seed(seed)
    rand = torch.rand(n, P * P, N, 1, device=dev).cpu()          # the draw Graph.sample_depth just made (:690)
    var = AttrDict(idx=idx, image=inp.image[sl].to(dev), obj_mask=inp.mask[sl].to(dev), ray_idx=coords)
    var.update(ret)
    loss = base.summarize_loss(opt, var, g.compute_loss(opt, var, mode="train"))
    loss["all"].backward()
    return {k: p.grad.detach().clone() for k, p in named_trainables(g)}, rand, {k: float(v.detach()) for k, v in loss.items()}, (zn.cpu(), zf.cpu())


def oracle_step(g, inp, images, rand, keep=None):
    """The same step through the CPU oracle (fp32): rays, bounds, depths, MLP, composite, losses, autograd.  `keep` [n, P*P, N]
    (0 / 1): the per-sample seeds of the masked samples are zeroed (the gradient without their contribution)."""
    if keep is not None:
        from tests.gradcheck import cotangent_mask
        real = O.nerf_stl_forward

        def masked(*a, **kw):
            rgb, dens, unc = real(*a, **kw)
            return (cotangent_mask(rgb, keep[..., None, None]), cotangent_mask(dens, keep[..., None]),
                    cotangent_mask(unc, keep[..., None]))
        O.nerf_stl_forward = masked
        try:
            return oracle_step(g, inp, images, rand)
        finally:
            O.nerf_stl_forward = real
    sl = images
    cpu = {k: p.detach().cpu().clone().requires_grad_(True) for k, p in named_trainables(g)}
    feat = [(l.weight.detach().cpu(), l.bias.detach().cpu()) for l in g.nerf.mlp_feat]
    rl = [(cpu[f"mlp_rgb.{i}.weight"], cpu[f"mlp_rgb.{i}.bias"]) for i in range(4)]
    tl = [(cpu[f"mlp_trans.{i}.weight"], cpu[f"mlp_trans.{i}.bias"]) for i in range(4)]
    pose, intr, coords = inp.pose[sl], inp.intr[sl], inp.coords[sl]
    n = len(pose)
    c, r = O.get_center_and_ray(pose, intr, H, W)
    lo, hi = synth.padded_aabb()
    tn, tf, v = O.aabb_ray_intersection(lo, hi, c, r)
    zn, zf = O.box_bounds_to_range(tn, tf, v, *synth.BG_RANGE)
    center, ray = O.patch_rays(coords, pose, intr, H, W)
    pzn, pzf = O.patch_bounds(coords, zn, zf, H, W)
    center, ray = center.reshape(n, P * P, 3), ray.reshape(n, P * P, 3)
    idx = inp.idx[sl]
    out = O.render_stl(center, ray, pzn.reshape(n, P * P), pzf.reshape(n, P * P), rand, N, cpu["latent_vars_trans.weight"][idx],
                       cpu["latent_vars_light.weight"][idx], feat, rl, tl)
    losses = O.patch_losses(inp.image[sl], inp.mask[sl], coords, out["rgb"], out["uncert"], out["density"], 0.0, 0.0, -2.0)
    losses["all"].backward()
    grads = {k: (p.grad if p.grad is not None else torch.zeros_like(p)) for k, p in cpu.items()}
    return grads, {k: float(losses[k].detach()) for k in ("render", "uncert", "trans_reg", "all")}, (zn, zf)
