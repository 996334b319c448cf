"""Mask-prior eval frames in one launch (Graph.render_masked): the device-built object-pixel list (tp_mask_ray_list), the
background defaults (tp_mask_defaults), the list mode of both render launches against the per-view eval path and the full-frame
launch, CUDA-graph capture, and the object-balanced multi-GPU eval frame (parallel.FrameGather with an object mask)."""
import os
import socket
import time

import pytest
import torch

from texpose_b200 import _C, compute_box, ops, synth
from texpose_b200.config import AttrDict, adapt_gan_opt
from texpose_b200.model.nerf_adapt_st_gan import Graph

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
KEYS = Graph.RENDER_KEYS
ARCH_SINGLE = dict(layers_feat=[None] + [256] * 6, skip=[2], layers_rgb=[None, 256, 256, 3], layers_trans=[None, 256, 256, 5])
PER_VIEW = ("tp_render_fused_forward", "tp_tc32_render_forward")


def _reference_list(mask, N):
    """(entries, counts) of the list format from (mask[b] > 0).nonzero() per view."""
    u = 256 // N
    B, HW = mask.shape
    out, counts = [], []
    for b in range(B):
        idx = (mask[b] > 0).nonzero(as_tuple=True)[0].cpu() + b * HW
        counts.append(len(idx))
        pad = (-len(idx)) % u
        out.append(torch.cat([idx, torch.full((pad,), ~(b * HW), dtype=torch.int64)]))
    return torch.cat(out), torch.tensor(counts)


def _masks():
    gen = torch.Generator().manual_seed(3)
    ragged = (torch.rand(3, 24 * 40, generator=gen) < torch.tensor([[0.3], [0.0], [0.07]])).float()
    ones = torch.ones(1, 37 * 11)
    single = torch.zeros(2, 500)
    single[1, 321] = 1.0
    signed = torch.randn(2, 1000, generator=gen)
    signed[0, ::7] = 0.0
    signed[1, ::5] = -0.0
    frame = torch.zeros(1, 480, 640)
    frame[0, 200:290, 250:400] = 1.0
    frame[0, 10, 10] = 2.0
    return [ragged, ones, single, signed, frame.reshape(1, -1)]


@pytest.mark.parametrize("N", [32, 64, 128])
def test_mask_ray_list_equals_nonzero_per_view(N):
    for mask in _masks():
        mask = mask.to(DEV)
        lst, n_slots, counts = ops.mask_ray_list(mask, N)
        want, want_counts = _reference_list(mask, N)
        n = int(n_slots.item())
        u = 256 // N
        assert n == sum((int(c) + u - 1) // u * u for c in want_counts)
        assert torch.equal(lst[:n].cpu(), want)
        assert torch.equal(counts.cpu(), want_counts)


def _graph(mlp, N, H, W, arch=None, static_only=False):
    opt = adapt_gan_opt(H=H, W=W, sample_intvs=N, device=DEV)
    for k, v in (arch or {}).items():
        opt.arch[k] = v
    opt.nerf.sample_stratified = False
    opt.b200 = AttrDict(mlp=mlp, static_only=static_only)
    torch.manual_seed(0)
    g = Graph(opt, n_train_images=4).to(DEV).eval()
    gen = torch.Generator().manual_seed(12)
    with torch.no_grad():
        for lin in [l for ml in (g.nerf.mlp_feat, g.nerf.mlp_rgb, g.nerf.mlp_trans) for l in ml]:
            lin.bias.copy_(torch.randn(lin.bias.shape, generator=gen).mul_(0.2).to(DEV))
    opt.render.transient = "sample"
    return opt, g


def _views(B, H, W, scale, seeds=None):
    pose, intr = synth.poses(seeds or list(range(0, 3 * B, 3))).to(DEV), synth.intrinsics(B).to(DEV).clone()
    intr[:, :2] *= scale
    lo, hi = [t.to(DEV) for t in synth.padded_aabb()]
    zn, zf = compute_box.box_range(pose, intr, lo, hi, H, W, *synth.BG_RANGE)
    return pose, intr, (zn[:, :, None], zf[:, :, None])


def _ragged_mask(B, HW, seed=4):
    gen = torch.Generator().manual_seed(seed)
    m = (torch.rand(B, HW, generator=gen) < torch.linspace(0.4, 0.05, B)[:, None]).float()
    m[1] = 0.0          # one empty view
    return m.to(DEV)


def _per_view_render_launch(g, opt, pose, intr, dr, mask, sample_idx):
    """render_by_slices' mask-prior branch (defaults, then per view the object pixels' nonzero() and one render launch, scattered)
    with Graph._render_fused as the per-view render."""
    B, HW, N = len(pose), opt.H * opt.W, opt.nerf.sample_intvs
    out = {k: torch.zeros(B, HW, 3, device=DEV) if "rgb" in k else torch.ones(B, HW, N, device=DEV) if "alpha" in k
           else torch.ones(B, HW, N, 2, device=DEV) if k == "density"
           else torch.full((B, HW, 1), float(opt.nerf.min_uncert), device=DEV) if k == "uncert" else torch.zeros(B, HW, 1, device=DEV)
           for k in KEYS}
    for b in range(B):
        idx = (mask[b] > 0).nonzero(as_tuple=True)[0]
        if len(idx) == 0:
            continue
        sl = slice(b, b + 1)
        ret = g._render_fused(opt, pose[sl], intr[sl], idx[None], tuple(d[sl] for d in dr), sample_idx[b], "eval")
        for k in KEYS:
            out[k][b, idx] = ret[k][0]
    return out


CASES = [("bf16", 32, None, False), ("bf16", 64, None, False), ("bf16", 128, None, False), ("bf16", 64, None, True),
         ("fp32", 64, None, False), ("bf16", 64, ARCH_SINGLE, False)]


@pytest.mark.parametrize("mlp,N,arch,static_only", CASES)
def test_render_masked_equals_the_per_view_eval_path(mlp, N, arch, static_only):
    H, W, B = 24, 40, 3
    opt, g = _graph(mlp, N, H, W, arch, static_only)
    # the per-view path inverts K per view: torch's batched inverse of B views may differ from it in the last bit, the kernel's does not
    opt.b200.view_matrices = "kernel"
    pose, intr, dr = _views(B, H, W, 0.06)
    mask = _ragged_mask(B, H * W)
    sample_idx = torch.tensor([2, 0, 3], device=DEV)
    list_entry = "tp_render_fused_forward_list" if mlp == "bf16" and arch is None else "tp_tc32_render_forward_list"
    with torch.no_grad():
        if g.nerf.fused_render_applies(opt, "eval"):      # K2r: render_by_slices' eval branch runs the render launch per view
            want = g.render_by_slices(opt, pose, intr=intr, depth_range=dr, object_mask=mask, sample_idx=sample_idx, mode="eval")
        else:      # render_by_slices runs the multi-kernel path here: the same branch with the staged render launch per view
            want = _per_view_render_launch(g, opt, pose, intr, dr, mask, sample_idx)
        _C.launch_counts.clear()
        got = g.render_masked(opt, pose, intr, dr, mask, sample_idx=sample_idx, mode="eval")
    assert _C.launch_counts.get(list_entry) == 1, dict(_C.launch_counts)
    assert not any(k in _C.launch_counts for k in PER_VIEW), dict(_C.launch_counts)
    for k in KEYS:
        assert got[k].shape == want[k].shape, k
        assert torch.equal(got[k], want[k]), (k, float((got[k] - want[k]).abs().max()))


@pytest.mark.parametrize("rng", ["torch", "philox"])
@pytest.mark.parametrize("mlp", ["bf16", "fp32"])
def test_stratified_jitter_equals_the_full_frame_launch(rng, mlp):
    H, W, B, N = 24, 40, 2, 64
    opt, g = _graph(mlp, N, H, W)
    opt.nerf.sample_stratified = True
    opt.b200.rng = rng
    pose, intr, dr = _views(B, H, W, 0.06)
    mask = _ragged_mask(B, H * W)
    mask[1, 5:300] = 1.0
    sample_idx = torch.tensor([1, 2], device=DEV)
    with torch.no_grad():
        torch.manual_seed(77)
        got = g.render_masked(opt, pose, intr, dr, mask, sample_idx=sample_idx)
        torch.manual_seed(77)
        full = g._render_fused(opt, pose, intr, range(0, H * W), dr, sample_idx, "eval")
    obj = mask > 0
    defaults = dict(rgb=0.0, rgb_static=0.0, rgb_transient=0.0, depth=0.0, opacity=0.0, opacity_static=0.0, opacity_transient=0.0,
                    uncert=float(opt.nerf.min_uncert), alpha_static=1.0, alpha_transient=1.0, density=1.0)
    for k in KEYS:
        assert torch.equal(got[k][obj], full[k][obj]), k
        assert (got[k][~obj] == defaults[k]).all(), k


def test_render_masked_is_captured_in_a_cuda_graph():
    H, W, B, N = 24, 40, 2, 64
    opt, g = _graph("bf16", N, H, W)
    opt.nerf.sample_stratified = True
    pose, intr, dr = _views(B, H, W, 0.06)
    s_pose, s_intr = pose.clone(), intr.clone()
    s_zn, s_zf = dr[0].clone(), dr[1].clone()
    s_mask = _ragged_mask(B, H * W)
    sample_idx = torch.tensor([1, 2], device=DEV)
    with torch.no_grad():
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                g.render_masked(opt, s_pose, s_intr, (s_zn, s_zf), s_mask, sample_idx=sample_idx)
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out = g.render_masked(opt, s_pose, s_intr, (s_zn, s_zf), s_mask, sample_idx=sample_idx)
        for seeds, mseed in (([1, 4], 9), ([6, 2], 10)):
            pose2, intr2, dr2 = _views(B, H, W, 0.06, seeds)
            mask2 = _ragged_mask(B, H * W, mseed)
            s_pose.copy_(pose2); s_intr.copy_(intr2); s_zn.copy_(dr2[0]); s_zf.copy_(dr2[1]); s_mask.copy_(mask2)
            torch.manual_seed(mseed)
            graph.replay()
            torch.manual_seed(mseed)
            eager = g.render_masked(opt, pose2, intr2, dr2, mask2, sample_idx=sample_idx)
            for k in KEYS:
                assert torch.equal(out[k], eager[k]), k


def test_render_masked_at_size_equals_nerf_forward_eval():
    H, W, N = 480, 640, 128
    opt, g = _graph("bf16", N, H, W)
    opt.render.transient = "zero"
    pose, intr, dr = _views(1, H, W, 1.0, [3])
    zn, zf = dr[0][..., 0], dr[1][..., 0]
    mask = (zf < synth.BG_RANGE[1]).float() if (zf < synth.BG_RANGE[1]).any() else torch.zeros_like(zf)
    mask[0, 200 * W + 300:200 * W + 420] = 1.0
    var = AttrDict(pose=pose, intr=intr, z_near=zn, z_far=zf, obj_mask=mask.view(1, H * W, 1),
                   pose_anchor=synth.poses([0, 3, 5, 7]).to(DEV))
    with torch.no_grad():
        torch.manual_seed(5)
        g.nerf_forward(opt, var, mode="eval_noalign")
        torch.manual_seed(5)
        from texpose_b200.model.nerf_adapt_st_gan import rotation_distance
        R_dist = rotation_distance(var.pose[:, None, :3, :3], var.pose_anchor[None, :, :3, :3])
        k = int(opt.render.N_candidate)
        idx = torch.topk(R_dist, k=k, dim=1, largest=False, sorted=True)[1][:, int(torch.randperm(k)[0])][0]
        got = g.render_masked(opt, pose, intr, dr, mask, sample_idx=idx, mode="eval_noalign")
    for key in KEYS:
        assert torch.equal(got[key], var[key]), key


# ------------------------------------------------------------------------------------------ eval frames across ranks
GH, GW, GN = 32, 64, 64


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gather_worker(rank, world, port, ret):
    import torch.distributed as dist
    from texpose_b200 import parallel
    from texpose_b200.model.nerf_pretrain import Graph as PretrainGraph
    from texpose_b200.config import env_opt
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", rank % torch.cuda.device_count())
    torch.cuda.set_device(dev)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    ok = True
    try:
        lo, hi = [t.to(dev) for t in synth.padded_aabb()]
        for mlp in ("bf16", "fp32"):
            opt = adapt_gan_opt(H=GH, W=GW, sample_intvs=GN, device=str(dev))
            opt.nerf.sample_stratified = False
            opt.b200 = AttrDict(mlp=mlp)
            torch.manual_seed(0)
            g = Graph(opt, n_train_images=2).to(dev).eval()
            fg = parallel.FrameGather(opt, device=dev, timeout_ms=30000)
            try:
                for seed in (0, 3, 5):          # three frames: both window buffers, one reused
                    pose, intr = synth.poses([seed]).to(dev), synth.intrinsics(1).to(dev).clone()
                    intr[:, :2] *= 0.1
                    zn, zf = compute_box.box_range(pose, intr, lo, hi, GH, GW, *synth.BG_RANGE)
                    dr = (zn[:, :, None], zf[:, :, None])
                    mask = torch.zeros(1, GH * GW, device=dev)
                    mask[0, 5 * GW + 10:5 * GW + 40] = 1.0
                    mask[0, 20 * GW:21 * GW] = 1.0
                    mask[0, 7 + seed] = 1.0
                    sidx = torch.tensor(1, device=dev)
                    with torch.no_grad():
                        got, _ = fg.render(g, opt, pose, intr, dr, sample_idx=sidx, mode="eval", object_mask=mask)
                        torch.cuda.synchronize(dev)
                        fg.check()
                        # what each rank writes: its share rendered into a NaN-filled frame of its own
                        mine = torch.full((GH * GW,), float("nan"), device=dev)
                        g.render_masked(opt, pose, intr, dr, mask, sample_idx=sidx, mode="eval", want=("depth",),
                                        out_ptrs={"depth": mine.data_ptr()}, shard=(rank, world))
                        written = [None] * world
                        dist.all_gather_object(written, (~mine.isnan()).cpu())
                        obj = (mask[0] > 0).cpu()
                        times = torch.stack(written).int().sum(0)
                        ok = ok and bool((times == 1).all())      # every frame position written once, by one rank
                        u = 256 // GN
                        n_obj = [int((w & obj).sum()) for w in written]
                        ok = ok and max(abs(n - int(obj.sum()) / world) for n in n_obj) <= 2 * u      # balanced by object pixels
                        lo_r, hi_r = fg.rows
                        ok = ok and bool(written[rank][~obj].eq(torch.zeros(GH * GW, dtype=torch.bool).index_fill_(
                            0, torch.arange(lo_r, hi_r), True)[~obj]).all())      # background: this rank's row block
                        if rank == 0:
                            want = g.render_masked(opt, pose, intr, dr, mask, sample_idx=sidx, mode="eval")      # the world-1 frame
                            for k in parallel.PER_RAY_KEYS:
                                ok = ok and torch.equal(got[k], want[k])
                        else:
                            assert got is None
                        if mlp == "bf16" and seed == 0:
                            for bad in (lambda: fg.render(g, opt, pose, intr, dr, mode="eval", object_mask=mask,
                                                          local_keys=("density",)),
                                        lambda: fg.render(PretrainGraph(env_opt(H=GH, W=GW, sample_intvs=GN, device=str(dev))),
                                                          opt, pose, intr, dr, object_mask=mask)):
                                try:
                                    bad()
                                    ok = False
                                except ValueError:
                                    pass
            finally:
                fg.close()
        ret[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_frame_gather_eval_frames_equal_the_world_1_frame(world):
    import torch.multiprocessing as mp
    _C.build()
    mgr = mp.Manager()
    ret = mgr.dict()
    ctx = mp.spawn(_gather_worker, args=(world, _free_port(), ret), nprocs=world, join=False)
    deadline = time.time() + 400
    done = False
    while not done and time.time() < deadline:
        done = ctx.join(timeout=5)
    if not done:
        for p in ctx.processes:
            if p.is_alive():
                p.terminate()
        pytest.fail("frame-gather workers did not finish")
    assert all(ret.get(r) for r in range(world)), dict(ret)
