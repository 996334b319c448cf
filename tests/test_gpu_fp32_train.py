"""The <= 1e-4 training step on the tensor cores (opt.b200.mlp = 'fp32', opt.b200.fp32_engine = 'tc'): split-fp16 forward that
saves the activations as bf16 hi + lo images (tp_tc32_forward_split_save), split dX chain (tp_tc_chain_backward_split), dW GEMMs
and thin helpers on the hi / lo images.  Every gradient against the CPU oracle's fp32 autograd (or the SIMT fp32 step) within
1e-4 max-abs, the launch route, determinism, exact scale invariance, the pre-training Graph against the reference fixture, and
the routes that must stay on SIMT."""
import pytest
import torch

from oracle import texpose_oracle as O
from texpose_b200 import _C, synth
from texpose_b200.config import AttrDict, adapt_gan_opt, env_opt
from texpose_b200.layers import nerf, nerf_static_transient_light
from tests.test_gpu_tc import _c1_inputs

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-4
TC = AttrDict(mlp="fp32", fp32_engine="tc")


def _opt(make, b200, arch=None, **kw):
    opt = make(**kw)
    for k, v in (arch or {}).items():
        opt.arch[k] = v
    opt.b200 = AttrDict(b200)
    return opt


def _plain_models(arch=None, seed=0):
    opt = _opt(env_opt, TC, arch, device=DEV)
    torch.manual_seed(seed)
    m = nerf.NeRF(opt).to(DEV)
    gen = torch.Generator().manual_seed(7)
    with torch.no_grad():
        for lin in list(m.mlp_feat) + list(m.mlp_rgb):
            lin.bias.copy_(torch.randn(lin.bias.shape, generator=gen).mul_(0.2).to(DEV))
    cpu = nerf.NeRF(_opt(env_opt, {}, arch))
    cpu.load_state_dict(m.state_dict())
    return opt, m, cpu


def _plain_loss(rgb, depth, opacity, sigma, image, mask):
    return (mask * (image - rgb) ** 2).sum() / (mask.sum() + 1e-5) + 0.1 * depth.mean() + 0.05 * opacity.mean() + 0.01 * sigma.mean()


def _plain_vs_oracle(opt, m, cpu, R, N, use_forward_samples=True):
    """One training step of the plain model on the GPU and on the oracle -> (rgb error, composite error, worst gradient error)."""
    center, ray, depth = _c1_inputs(R=R, N=N, seed_pose=1)
    g = torch.Generator().manual_seed(9)
    image, mask = torch.rand(1, R, 3, generator=g), (torch.rand(1, R, 1, generator=g) > 0.3).float()
    fl = [(l.weight, l.bias) for l in cpu.mlp_feat]
    rl = [(l.weight, l.bias) for l in cpu.mlp_rgb]
    pts = O.points_from_depth(center, ray, depth)
    unit = torch.nn.functional.normalize(ray, dim=-1)[..., None, :].expand_as(pts)
    rgb_s, sig = O.nerf_plain_forward(pts, unit, fl, rl)
    comp = O.composite_plain(ray, rgb_s, sig, depth)
    _plain_loss(comp[0], comp[1], comp[2], sig, image, mask).backward()
    if use_forward_samples:
        rgb_g, sig_g = m.forward_samples(opt, center.to(DEV), ray.to(DEV), depth.to(DEV), mode="train")
    else:
        rgb_g, sig_g = m.forward(opt, pts.to(DEV), unit.to(DEV), mode="train")
    comp_g = m.composite(opt, ray.to(DEV), rgb_g, sig_g, depth.to(DEV))
    _plain_loss(comp_g[0], comp_g[1], comp_g[2], sig_g, image.to(DEV), mask.to(DEV)).backward()
    worst = 0.0
    for (n, a), b in zip(list(m.mlp_feat.named_parameters(prefix="mlp_feat")) + list(m.mlp_rgb.named_parameters(prefix="mlp_rgb")),
                         list(cpu.mlp_feat.parameters()) + list(cpu.mlp_rgb.parameters())):
        assert a.grad is not None and a.grad.shape == b.grad.shape, n
        err = (a.grad.cpu() - b.grad).abs().max().item()
        print(f"  {n:22s} |grad|max {b.grad.abs().max().item():9.3e}  max-abs err {err:9.3e}")
        worst = max(worst, err)
    out = max((rgb_g.cpu() - rgb_s).abs().max().item(), (sig_g.cpu() - sig).abs().max().item())
    return out, (comp_g[0].cpu() - comp[0]).abs().max().item(), worst


@pytest.mark.parametrize("R,N", [(256, 64), (300, 24)])
def test_plain_fp32_step_on_tensor_cores_vs_oracle(R, N):
    opt, m, cpu = _plain_models()
    assert m.trains_on_tensor_cores(opt)
    _C.launch_counts.clear()
    out, comp, worst = _plain_vs_oracle(opt, m, cpu, R, N)
    counts = dict(_C.launch_counts)
    print(f"plain {R}x{N}, fp32 step on the tensor cores: outputs {out:.2e}, composite {comp:.2e}, worst gradient {worst:.2e}")
    assert counts.get("tp_tc32_forward_split_save") == 1 and counts.get("tp_tc_chain_backward_split") == 1, counts
    assert "tp_tc32_forward" not in counts and "tp_tc_chain_backward" not in counts
    assert "tp_linear_forward" not in counts and "tp_linear_backward_input" not in counts
    assert out <= TOL and comp <= TOL and worst <= TOL


def _c3_inputs():
    B, R, N = 16, 256, 128
    g = torch.Generator().manual_seed(0)
    center = (torch.randn(B, R, 3, generator=g) * 0.02 + torch.tensor([0.3, 0.2, -0.8])).to(DEV)
    ray = (torch.randn(B, R, 3, generator=g) * 0.1 + torch.tensor([0.0, 0.0, 1.0])).to(DEV)
    depth = ((torch.rand(B, R, N, 1, generator=g) + torch.arange(N)[None, None, :, None]) / N * 1.2 + 0.2).to(DEV)
    image = torch.rand(B, R, 3, generator=g).to(DEV)
    return center, ray, depth, image


def _plain_grads(m, o, inputs, scale=1.0):
    center, ray, depth, image = inputs
    for p in m.parameters():
        p.grad = None
    rgb_s, sig = m.forward_samples(o, center, ray, depth, mode="train")
    comp = m.composite(o, ray, rgb_s, sig, depth)
    ((((comp[0] - image) ** 2).mean() + 0.1 * comp[1].mean() + 0.01 * sig.mean()) * scale).backward()
    return [p.grad.clone() for p in m.parameters()]


def test_plain_fp32_step_at_the_c3_shape_matches_simt_and_repeats_bit_for_bit():
    inputs = _c3_inputs()
    opt, m, _ = _plain_models()
    simt = _opt(env_opt, dict(mlp="fp32", fp32_engine="simt"), device=DEV)
    a, a2, ref = _plain_grads(m, opt, inputs), _plain_grads(m, opt, inputs), _plain_grads(m, simt, inputs)
    worst = 0.0
    for (n, _), x, x2, y in zip(m.named_parameters(), a, a2, ref):
        assert torch.equal(x, x2), n
        err = (x - y).abs().max().item()
        worst = max(worst, err)
        assert err <= TOL, (n, err, y.abs().max().item())
    print(f"plain 16x256x128: tensor-core fp32 step vs SIMT fp32 step, worst gradient max-abs {worst:.2e}")


def test_gradients_scale_exactly_with_the_loss():
    """No operand format depends on magnitude: the gradients of loss * 2^-20 are 2^-20 x those of loss, bit for bit."""
    center, ray, depth = [t.to(DEV) for t in _c1_inputs(R=256, N=64, seed_pose=1)]
    image = torch.rand(1, 256, 3, generator=torch.Generator().manual_seed(9)).to(DEV)
    opt, m, _ = _plain_models()
    a = _plain_grads(m, opt, (center, ray, depth, image))
    b = _plain_grads(m, opt, (center, ray, depth, image), scale=2.0 ** -20)
    for (n, _), x, y in zip(m.named_parameters(), a, b):
        assert torch.equal(x * 2.0 ** -20, y), n


STL_ARCHS = [
    {},
    dict(layers_feat=[None] + [256] * 6, skip=[2], layers_rgb=[None, 256, 256, 3], layers_trans=[None, 256, 256, 5]),
    dict(layers_feat=[None] + [256] * 8, skip=[4], layers_rgb=[None, 256, 3], layers_trans=[None, 256, 256, 256, 256, 5]),
]


@pytest.mark.parametrize("arch", STL_ARCHS, ids=["yaml", "6x256-skip2", "rgb1-trans4"])
def test_static_transient_light_fp32_step_on_tensor_cores_vs_oracle(arch):
    R, N = 256, 64
    center, ray, depth = _c1_inputs(R=R, N=N, seed_pose=1)
    lt, ll = synth.latents(1)
    opt = _opt(adapt_gan_opt, TC, arch, device=DEV)
    torch.manual_seed(0)
    m = nerf_static_transient_light.NeRF(opt).to(DEV)
    gen = torch.Generator().manual_seed(12)
    with torch.no_grad():
        for lin in list(m.mlp_feat) + list(m.mlp_rgb) + list(m.mlp_trans):
            lin.bias.copy_(torch.randn(lin.bias.shape, generator=gen).mul_(0.2).to(DEV))
    cpu = nerf_static_transient_light.NeRF(_opt(adapt_gan_opt, {}, arch))
    cpu.load_state_dict(m.state_dict())
    g = torch.Generator().manual_seed(9)
    image = torch.rand(1, R, 3, generator=g)
    mask = (torch.rand(1, R, 1, generator=g) > 0.3).float()

    def loss_of(comp, dens, image, mask):
        rgb, unc = comp[0], comp[8]
        return (mask * ((image - rgb) ** 2 / unc ** 2)).sum() / (mask.sum() + 1e-5) + (5 + torch.log(unc ** 2).mean() / 2) \
            + 0.01 * dens[..., -1].mean()

    lt_o, ll_o = lt.clone().requires_grad_(True), ll.clone().requires_grad_(True)
    fl = [(l.weight.detach(), l.bias.detach()) for l in cpu.mlp_feat]
    rl = [(l.weight, l.bias) for l in cpu.mlp_rgb]
    tl = [(l.weight, l.bias) for l in cpu.mlp_trans]
    pts = O.points_from_depth(center, ray, depth)
    unit = torch.nn.functional.normalize(ray, dim=-1)[..., None, :].expand_as(pts)
    ref_s = O.nerf_stl_forward(pts, unit, lt_o, ll_o, fl, rl, tl, skip=tuple(opt.arch.skip))
    loss_of(O.composite_stl(ray, *ref_s[:2], depth, ref_s[2], 0.05), ref_s[1], image, mask).backward()

    lt_g, ll_g = lt.to(DEV).requires_grad_(True), ll.to(DEV).requires_grad_(True)
    _C.launch_counts.clear()
    got_s = m.forward_samples(opt, center.to(DEV), ray.to(DEV), depth.to(DEV), lt_g, ll_g, mode="train")
    comp = m.composite(opt, ray.to(DEV), *got_s[:2], depth.to(DEV), got_s[2])
    loss_of(comp, got_s[1], image.to(DEV), mask.to(DEV)).backward()
    counts = dict(_C.launch_counts)
    assert counts.get("tp_tc32_forward_split_save") == 1 and counts.get("tp_tc_chain_backward_split") == 2, counts
    # no SIMT GEMM of a 256-wide layer: no SIMT forward, and the SIMT input-gradient GEMMs are the two latents' (<= 48 columns)
    assert "tp_linear_forward" not in counts and counts.get("tp_linear_backward_input", 0) <= 2, counts
    assert all(p.grad is None for p in m.mlp_feat.parameters())           # the trunk stays frozen
    pairs = [("latent_trans", lt_g.grad.cpu(), lt_o.grad), ("latent_light", ll_g.grad.cpu(), ll_o.grad)]
    names = [n for n, _ in list(m.mlp_rgb.named_parameters(prefix="mlp_rgb")) + list(m.mlp_trans.named_parameters(prefix="mlp_trans"))]
    for n, a, b in zip(names, list(m.mlp_rgb.parameters()) + list(m.mlp_trans.parameters()),
                       list(cpu.mlp_rgb.parameters()) + list(cpu.mlp_trans.parameters())):
        pairs.append((n, a.grad.cpu(), b.grad))
    worst = 0.0
    for n, a, b in pairs:
        err = (a - b).abs().max().item()
        print(f"  {n:22s} |grad|max {b.abs().max().item():9.3e}  max-abs err {err:9.3e}")
        assert a.shape == b.shape
        worst = max(worst, err)
    print(f"static/transient/light {arch or 'yaml'}: worst gradient max-abs error {worst:.2e}")
    assert worst <= TOL


def test_pretrain_graph_fp32_tc_step_matches_the_real_reference(golden, monkeypatch):
    """Fixture `pretrain` (model/nerf_pretrain.py Graph of the unmodified reference), the pattern of
    test_gpu_pretrain_graph.test_train_step_and_val_frame_match_the_real_reference, with the step on the split kernels."""
    from texpose_b200 import camera
    from texpose_b200.model.nerf_pretrain import Graph
    camera.HOST_MATRICES = True
    try:
        g = golden("pretrain")
        B, R = g.ray_idx.shape
        opt = env_opt(H=int(g.H), W=int(g.W), sample_intvs=int(g.N), device=DEV)
        opt.nerf.rand_rays = B * R
        opt.loss_weight = AttrDict(render=0, mask=-1, depth=-1)
        opt.data.erode_mask_loss = False
        opt.b200 = AttrDict(TC)
        torch.manual_seed(0)
        gr = Graph(opt).to(DEV)
        var = AttrDict(idx=torch.arange(B), pose=g.pose.to(DEV), pose_init=g.pose.to(DEV), intr=g.intr.to(DEV),
                       z_near=g.z_near.to(DEV), z_far=g.z_far.to(DEV), image=g.image.to(DEV), obj_mask=g.obj_mask.to(DEV),
                       depth_gt=g.depth_gt.to(DEV))
        real_randperm, real_rand = torch.randperm, torch.rand
        perm = torch.cat([g.ray_idx[0], torch.zeros(int(g.H) * int(g.W) - R, dtype=torch.long)]).to(DEV)
        monkeypatch.setattr(torch, "randperm", lambda n, **kw: perm if n == int(g.H) * int(g.W) else real_randperm(n, **kw))
        monkeypatch.setattr(torch, "rand", lambda *s, **kw: g.rand.to(DEV) if tuple(s) == tuple(g.rand.shape) else real_rand(*s, **kw))
        _C.launch_counts.clear()
        var = gr.forward(opt, var, mode="train")
        loss = gr.compute_loss(opt, var, mode="train")
        monkeypatch.undo()
        assert torch.equal(var.ray_idx.cpu(), g.ray_idx)
        sum(10 ** float(opt.loss_weight[k]) * loss[k] for k in loss).backward()
        assert _C.launch_counts.get("tp_tc32_forward_split_save") == 1 and _C.launch_counts.get("tp_tc_chain_backward_split") == 1
        errs = {k: (var[k].cpu() - g["o_" + k]).abs().max().item() for k in ("rgb", "depth", "opacity")}
        errs.update({"l_" + k: abs(loss[k].item() - float(g["l_" + k])) for k in ("render", "mask", "depth")})
        worst, mag = 0.0, 0.0
        for n, p in gr.nerf.named_parameters():
            got = p.grad if p.grad.numel() <= 2048 else p.grad[:, ::8][::8]
            worst = max(worst, (got.cpu() - g["g/" + n]).abs().max().item())
            mag = max(mag, g["g/" + n].abs().max().item())
        errs["grad"] = worst
        print("pretrain Graph, fp32 step on the tensor cores, vs the real reference:", {k: f"{v:.2e}" for k, v in errs.items()},
              f"gradient error relative to max |grad| {mag:.3e}: {worst / mag:.2e}")
        for k, e in errs.items():
            assert e <= TOL, (k, e)
    finally:
        camera.HOST_MATRICES = False


@pytest.mark.parametrize("engine", [None, "simt"])
def test_fp32_training_without_tc_engine_stays_on_simt(engine):
    opt, m, _ = _plain_models()
    opt.b200 = AttrDict(mlp="fp32", fp32_engine=engine)
    assert not m.trains_on_tensor_cores(opt)
    center, ray, depth = [t.to(DEV) for t in _c1_inputs(R=128, N=32)]
    _C.launch_counts.clear()
    rgb, sig = m.forward_samples(opt, center, ray, depth, mode="train")
    (rgb.square().mean() + sig.mean()).backward()
    counts = dict(_C.launch_counts)
    assert counts.get("tp_linear_forward", 0) > 0 and counts.get("tp_linear_backward_input", 0) > 0, counts
    assert not any(k.startswith("tp_tc") for k in counts), counts


def test_tc_engine_unsupported_architecture_and_explicit_points_train_on_simt():
    # an rgb head of two hidden layers is not a shape the plain tensor-core step implements
    arch = dict(layers_rgb=[None, 128, 128, 3])
    opt, m, cpu = _plain_models(arch)
    assert not m.trains_on_tensor_cores(opt)
    _C.launch_counts.clear()
    out, comp, worst = _plain_vs_oracle(opt, m, cpu, 256, 64)
    assert _C.launch_counts.get("tp_linear_forward", 0) > 0 and "tp_tc_chain_backward_split" not in _C.launch_counts
    print(f"'tc' engine, unsupported head: SIMT step, outputs {out:.2e}, worst gradient {worst:.2e}")
    assert out <= TOL and worst <= TOL
    # explicit points (NeRF.forward) with the supported architecture
    opt, m, cpu = _plain_models()
    _C.launch_counts.clear()
    out, comp, worst = _plain_vs_oracle(opt, m, cpu, 256, 64, use_forward_samples=False)
    assert _C.launch_counts.get("tp_linear_forward", 0) > 0 and not any(k.startswith("tp_tc") for k in _C.launch_counts)
    print(f"'tc' engine, explicit points: SIMT step, outputs {out:.2e}, worst gradient {worst:.2e}")
    assert out <= TOL and worst <= TOL
