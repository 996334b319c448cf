"""Smoke-sized run of every hand-written synchronisation protocol, for compute-sanitizer (memcheck / racecheck / synccheck):
the fused forward kernel in its three launch kinds (render <17,3>, per-sample inference <17,1>, training <17,2> with the
activation save), the static-only instantiations, the fused backward chain + dW GEMM kernels, the fused loss, and the peer-window
exchange / barrier kernels with two "ranks" on one device.
usage: compute-sanitizer --tool racecheck python scripts/sanitize_target.py [what ...]   (what: render train split plain peer; default render train split plain)"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from texpose_b200 import compute_box, parallel, synth  # noqa: E402
from texpose_b200.config import AttrDict, adapt_gan_opt  # noqa: E402
from texpose_b200.model.base import summarize_loss  # noqa: E402
from texpose_b200.model.nerf_adapt_st_gan import Graph  # noqa: E402

what = set(sys.argv[1:]) or {"render", "train", "split", "plain"}      # "peer" needs concurrent kernels: the tool serialises launches of one process
dev = "cuda:0"
H, W, N = 12, 64, 128            # 768 rays x 128 samples = 384 super-tiles: every CTA runs 2-3 of them
opt = adapt_gan_opt(H=H, W=W, sample_intvs=N, device=dev)
opt.b200 = AttrDict(mlp="bf16", rng="philox")
torch.manual_seed(0)
g = Graph(opt, n_train_images=4).to(dev)
pose, intr = synth.poses([0, 1]).to(dev), synth.intrinsics(2).to(dev).clone()
intr[:, :2] *= 0.1
lo, hi = [t.to(dev) for t in synth.padded_aabb()]
zn, zf = compute_box.box_range(pose, intr, lo, hi, H, W, *synth.BG_RANGE)
dr = (zn[:, :, None], zf[:, :, None])

if "render1" in what:      # the per-sample inference launch alone (multi-kernel path)
    with torch.no_grad():
        o2 = AttrDict(opt); o2.b200 = AttrDict(opt.b200); o2.b200.fused_render = False
        b = g.render(o2, pose, intr=intr, ray_idx=range(0, H * W), depth_range=dr, mode="val")
    torch.cuda.synchronize()
    print("render1 ok", float(b.rgb.sum()))

if "render" in what:
    with torch.no_grad():
        a = g.render(opt, pose, intr=intr, ray_idx=range(0, H * W), depth_range=dr, mode="val")                   # <17,3>
        o2 = AttrDict(opt); o2.b200 = AttrDict(opt.b200); o2.b200.fused_render = False
        b = g.render(o2, pose, intr=intr, ray_idx=range(0, H * W), depth_range=dr, mode="val")                    # <17,1> + composite
        o3 = AttrDict(opt); o3.b200 = AttrDict(opt.b200); o3.b200.static_only = True
        c = g.render(o3, pose[:1], intr=intr[:1], ray_idx=range(0, H * W), depth_range=(dr[0][:1], dr[1][:1]), sample_idx=torch.tensor(0, device=dev), mode="eval")   # <13,3>
        opt64 = adapt_gan_opt(H=H, W=W, sample_intvs=64, device=dev); opt64.b200 = AttrDict(mlp="bf16", rng="torch")
        d = g.render(opt64, pose, intr=intr, ray_idx=torch.randperm(H * W, device=dev)[None, :300].expand(2, -1).contiguous(), depth_range=dr, mode="val")   # 2 rays per tile
    torch.cuda.synchronize()
    print("render ok", float(a.rgb.sum()), float(b.rgb.sum()), float(c.rgb_static.sum()), float(d.rgb.sum()))

if "split" in what:
    # fp32-parity split-fp16 kernel (csrc/mlp_tc_split.cu): full stage list (park + reload), static-only list, ragged tail tile
    o32 = AttrDict(opt); o32.b200 = AttrDict(mlp="fp32", rng="philox")
    with torch.no_grad():
        a = g.render(o32, pose, intr=intr, ray_idx=range(0, H * W), depth_range=dr, mode="val")
        o33 = AttrDict(o32); o33.b200 = AttrDict(o32.b200); o33.b200.static_only = True
        b = g.render(o33, pose[:1], intr=intr[:1], ray_idx=range(0, H * W - 5), depth_range=(dr[0][:1], dr[1][:1]), sample_idx=torch.tensor(0, device=dev), mode="eval")
    torch.cuda.synchronize()
    print("split ok", float(a.rgb.sum()), float(b.rgb_static.sum()))

if "plain" in what:
    # plain-model training on the tensor cores: single-pass forward with activation save, staged dX chain, dW GEMM; mesh rasteriser
    from texpose_b200.config import env_opt
    from texpose_b200.layers.nerf import NeRF as PlainNeRF
    from texpose_b200.tools import mvrenderer
    oe = env_opt(device=dev); oe.b200 = AttrDict(mlp="bf16")
    pm = PlainNeRF(oe).to(dev)
    gg = torch.Generator().manual_seed(0)
    c_ = (torch.randn(2, 100, 3, generator=gg) * 0.02 + torch.tensor([0.3, 0.2, -0.8])).to(dev)
    r_ = (torch.randn(2, 100, 3, generator=gg) * 0.1 + torch.tensor([0.0, 0.0, 1.0])).to(dev)
    d_ = ((torch.rand(2, 100, 48, 1, generator=gg) + torch.arange(48)[None, None, :, None]) / 48 * 1.2 + 0.2).to(dev)
    rgb_s, sig = pm.forward_samples(oe, c_, r_, d_, mode="train")
    (rgb_s.square().mean() + sig.mean()).backward()
    mv, mf = [t.to(dev) for t in synth.icosphere(3, 0.6)]
    out, dep, _ = mvrenderer.render_mesh(mv, mf, mvrenderer.nocs_coordinates(mv), synth.poses([0, 1]).reshape(2, 12).to(dev), synth.intrinsics(2).to(dev) * torch.tensor([0.2, 0.2, 1.0], device=dev)[:, None], 96, 128)
    torch.cuda.synchronize()
    print("plain ok", float(pm.mlp_feat[0].weight.grad.abs().sum()), float(dep.max()))

if "train" in what:
    B, P = 4, 16
    opt_t = adapt_gan_opt(H=64, W=64, sample_intvs=N, device=dev)
    opt_t.b200 = AttrDict(mlp="bf16", rng="philox")
    pose_t = synth.poses(list(range(B))).to(dev)
    K = torch.tensor([[572.4114, 0, 32 - 572.4114 * 0.3 / 8], [0, 573.57043, 32 + 573.57043 * 0.2 / 8], [0, 0, 1]])
    intr_t = K.repeat(B, 1, 1).to(dev)
    zn_t, zf_t = compute_box.box_range(pose_t, intr_t, lo, hi, 64, 64, *synth.BG_RANGE)
    coords = synth.patch_coords(B, P, seed=2)[0].to(dev)
    idx = torch.arange(B, device=dev)
    var = AttrDict(idx=idx, image=torch.rand(B, 3, 64, 64, device=dev), obj_mask=(torch.rand(B, 64, 64, device=dev) > 0.3).float(), ray_idx=coords)
    g.train()
    ret = g.render(opt_t, pose_t, intr=intr_t, ray_idx=coords, depth_range=(zn_t[:, :, None], zf_t[:, :, None]), sample_idx=idx, mode="train")   # <17,2>
    var.update(ret)
    summarize_loss(opt_t, var, g.compute_loss(opt_t, var, mode="train"))["all"].backward()      # chain + dW + finish kernels
    torch.cuda.synchronize()
    print("train ok", float(g.nerf.mlp_trans[3].weight.grad.abs().sum()))

if "peer" in what:
    n = 100003
    ndev = 1          # both "ranks" on this device (two GPUs: tests/test_gpu_peer.py::test_two_processes_through_cuda_ipc under
    devs = [torch.device("cuda", 0)] * 2      # compute-sanitizer --target-processes all)
    wins = [parallel.PeerWindow(n, d) for d in devs]
    ptrs = [w.ptr for w in wins]
    outs = [torch.empty((n + 3) // 4 * 4, device=d) for d in devs]
    streams = [torch.cuda.Stream(d) for d in devs]
    for e in (1, 2, 3):
        for r in range(2):
            wins[r].buffers[e & 1].copy_(torch.full((n,), float(r + e), device=devs[r]))
        for d in devs:
            torch.cuda.synchronize(d)
        for r in (1, 0):
            parallel.peer_allreduce_mean(ptrs, r, n, e, outs[r], grid_ctas=8, timeout_ms=20000, stream=streams[r])
            parallel.peer_barrier(ptrs, r, e, devs[r], timeout_ms=20000, stream=streams[r])
        for d in devs:
            torch.cuda.synchronize(d)
        assert all(w.status() == 0 for w in wins)
        assert float(outs[0][:n].min()) == float(outs[1][:n].max()) == (1 + e + 2 + e) / 2
    for w in wins:
        w.close()
    print("peer ok on", ndev, "device(s)")
