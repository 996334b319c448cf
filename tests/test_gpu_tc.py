"""bf16 tensor-core path (csrc/mlp_tc.cu, tcgen05/TMEM) parity: BASELINE.json configs[0]-shaped case -- 1024 synthetic
AABB-bounded rays x 64 samples -- against the fp32 oracle.  Tolerance 1e-2 max-abs on rendered rgb/depth/opacity and
on gradients of the mean-normalised losses (north_star, bf16 MLP path)."""
import pytest
import torch

from oracle import texpose_oracle as O
from texpose_b200 import _C, synth
from texpose_b200.config import AttrDict, adapt_gan_opt
from texpose_b200.layers.nerf_static_transient_light import NeRF
from tests.conftest import layer_list

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-2


def _c1_inputs(R=1024, N=64, seed_pose=0):
    pose, intr = synth.poses([seed_pose]), synth.intrinsics(1)
    c, r = O.get_center_and_ray(pose, intr, 480, 640)
    lo, hi = synth.padded_aabb()
    tn, tf, v = O.aabb_ray_intersection(lo, hi, c, r)
    idx = v[0].nonzero()[:, 0][:R][None]                        # first R valid rays (SURVEY 8d, C1)
    g = torch.Generator().manual_seed(3)
    rand = torch.rand(1, R, N, 1, generator=g)
    depth = O.sample_depth(tn[:, idx[0]], tf[:, idx[0]], N, rand)
    return O.gather_rays(c, idx), O.gather_rays(r, idx), depth


def _module(precision):
    opt = adapt_gan_opt(device=DEV)
    opt.b200 = AttrDict(mlp=precision)
    torch.manual_seed(0)
    return opt, NeRF(opt).to(DEV)


def test_c1_forward_render_bf16_vs_oracle():
    center, ray, depth = _c1_inputs()
    lt, ll = synth.latents(1)
    opt, m = _module("bf16")
    cpu = NeRF(adapt_gan_opt())
    cpu.load_state_dict(m.state_dict())
    pts = O.points_from_depth(center, ray, depth)
    unit = torch.nn.functional.normalize(ray, dim=-1)[..., None, :].expand_as(pts)
    ref_s = O.nerf_stl_forward(pts, unit, lt, ll, layer_list(cpu.mlp_feat), layer_list(cpu.mlp_rgb), layer_list(cpu.mlp_trans))
    ref = O.composite_stl(ray, *ref_s[:2], depth, ref_s[2], 0.05)
    with torch.no_grad():
        got_s = m.forward_samples(opt, center.to(DEV), ray.to(DEV), depth.to(DEV), lt.to(DEV), ll.to(DEV), mode="val")
        got = m.composite(opt, ray.to(DEV), *got_s[:2], depth.to(DEV), got_s[2])
    names = ["rgb", "rgb_static", "rgb_transient", "depth", "opacity", "opacity_static", "opacity_transient", "prob",
             "uncert", "alpha_static", "alpha_transient"]
    errs = {k: (a.cpu() - b).abs().max().item() for k, a, b in zip(names, got, ref)}
    print("bf16 render max-abs errors:", {k: f"{v:.2e}" for k, v in errs.items()})
    for k in ("rgb", "rgb_static", "rgb_transient", "depth", "opacity", "opacity_static", "opacity_transient"):
        assert errs[k] <= TOL, (k, errs[k])
    # uncert is not bounded by 1 (it reaches 1.8 on these rays): 1.1e-2 = 0.6 % of its range, set by the bf16 trunk (with an
    # exact trunk the same head arithmetic gives 6.7e-3; DESIGN.md section 2) -- held to 1.5e-2
    assert errs["uncert"] <= 1.5e-2, errs["uncert"]
    # per-sample head outputs: bounded quantities within 1e-2, raw densities within 2 % of their range
    assert (got_s[0].cpu() - ref_s[0]).abs().max() <= 2e-2
    assert (got_s[1].cpu() - ref_s[1]).abs().max() <= 0.02 * ref_s[1].abs().max()


def test_bf16_matches_fp32_kernels_on_ragged_batch():
    """Two images, 37 rays x 24 samples (S = 1776: not a multiple of the 256-sample super-tile; rays straddle tiles)."""
    B, R, N = 2, 37, 24
    g = torch.Generator().manual_seed(4)
    center = (torch.randn(B, R, 3, generator=g) * 0.02 + torch.tensor([0.3, 0.2, -0.8])).to(DEV)
    ray = (torch.randn(B, R, 3, generator=g) * 0.1 + torch.tensor([0.0, 0.0, 1.0])).to(DEV)
    depth = ((torch.rand(B, R, N, 1, generator=g) + torch.arange(N)[None, None, :, None]) / N * 1.2 + 0.2).to(DEV)
    lt, ll = [t.to(DEV) for t in synth.latents(B)]
    opt16, m = _module("bf16")
    opt32 = adapt_gan_opt(device=DEV)
    with torch.no_grad():
        gen = torch.Generator().manual_seed(12)       # non-zero biases: they travel inside the packed weight image
        for lin in list(m.mlp_feat) + list(m.mlp_rgb) + list(m.mlp_trans):
            lin.bias.copy_(torch.randn(lin.bias.shape, generator=gen).mul_(0.3).to(DEV))
        a = m.forward_samples(opt16, center, ray, depth, lt, ll, mode="val")
        b = m.forward_samples(opt32, center, ray, depth, lt, ll, mode="val")
    assert a[0].shape == (B, R, N, 3, 2) and a[1].shape == (B, R, N, 2) and a[2].shape == (B, R, N, 1)
    assert (a[0] - b[0]).abs().max() <= 2e-2
    assert (a[1] - b[1]).abs().max() <= 0.03 * b[1].abs().max()
    assert (a[2] - b[2]).abs().max() <= 0.03 * b[2].abs().max()
    # weights changed in place -> packed image must be rebuilt (param._version key)
    with torch.no_grad():
        m.mlp_rgb[3].bias.add_(0.5)
        c = m.forward_samples(opt16, center, ray, depth, lt, ll, mode="val")
        d = m.forward_samples(opt32, center, ray, depth, lt, ll, mode="val")
    assert (c[0][..., 0] - a[0][..., 0]).abs().max() > 0.05
    assert (c[0] - d[0]).abs().max() <= 2e-2


def test_c3_shape_gradients_bf16():
    """fwd (tensor cores) + bwd of the three loss seeds with mean-normalised losses; grads within 1e-2 of the oracle."""
    R, N = 256, 64
    center, ray, depth = _c1_inputs(R=R, N=N, seed_pose=1)
    lt, ll = synth.latents(1)
    opt, m = _module("bf16")
    cpu = NeRF(adapt_gan_opt())
    cpu.load_state_dict(m.state_dict())
    g = torch.Generator().manual_seed(9)
    image = torch.rand(1, R, 3, generator=g)
    mask = (torch.rand(1, R, 1, generator=g) > 0.3).float()

    def loss_of(comp, dens, image, mask):
        rgb, unc = comp[0], comp[8]
        return (mask * ((image - rgb) ** 2 / unc ** 2)).sum() / (mask.sum() + 1e-5) + (5 + torch.log(unc ** 2).mean() / 2) \
            + 0.01 * dens[..., -1].mean()

    lt_o, ll_o = lt.clone().requires_grad_(True), ll.clone().requires_grad_(True)
    for p in list(cpu.mlp_rgb.parameters()) + list(cpu.mlp_trans.parameters()):
        p.requires_grad_(True)
    rl = [(l.weight, l.bias) for l in cpu.mlp_rgb]
    tl = [(l.weight, l.bias) for l in cpu.mlp_trans]
    pts = O.points_from_depth(center, ray, depth)
    unit = torch.nn.functional.normalize(ray, dim=-1)[..., None, :].expand_as(pts)
    ref_s = O.nerf_stl_forward(pts, unit, lt_o, ll_o, layer_list(cpu.mlp_feat), rl, tl)
    loss_of(O.composite_stl(ray, *ref_s[:2], depth, ref_s[2], 0.05), ref_s[1], image, mask).backward()

    lt_g, ll_g = lt.to(DEV).requires_grad_(True), ll.to(DEV).requires_grad_(True)
    got_s = m.forward_samples(opt, center.to(DEV), ray.to(DEV), depth.to(DEV), lt_g, ll_g, mode="train")
    comp = m.composite(opt, ray.to(DEV), *got_s[:2], depth.to(DEV), got_s[2])
    loss_of(comp, got_s[1], image.to(DEV), mask.to(DEV)).backward()
    pairs = [("latent_trans", lt_g.grad.cpu(), lt_o.grad), ("latent_light", ll_g.grad.cpu(), ll_o.grad)]
    names = [n for n, _ in list(m.mlp_rgb.named_parameters(prefix="mlp_rgb")) + list(m.mlp_trans.named_parameters(prefix="mlp_trans"))]
    for n, a, b in zip(names, list(m.mlp_rgb.parameters()) + list(m.mlp_trans.parameters()),
                       list(cpu.mlp_rgb.parameters()) + list(cpu.mlp_trans.parameters())):
        pairs.append((n, a.grad.cpu(), b.grad))
    worst, gmax = 0.0, 0.0
    for n, a, b in pairs:
        err, mag = (a - b).abs().max().item(), b.abs().max().item()
        print(f"  {n:22s} |grad|max {mag:9.3e}  max-abs err {err:9.3e}  ({100 * err / max(mag, 1e-12):5.2f} % of max)")
        worst, gmax = max(worst, err), max(gmax, mag)
    print(f"bf16 fwd gradient max-abs error {worst:.2e} (largest gradient entry {gmax:.2e})")
    # north_star: 1e-2 max-abs with the bf16 MLP path, for gradients of the reference's mean-normalised losses -- every tensor,
    # no relative carve-out (the output layers carry their weights as bf16 hi + lo rows: the systematic rounding of those few
    # rows was the dominant term for mlp_trans.3.weight, whose entries reach 1.86; DESIGN.md section 2)
    for n, a, b in pairs:
        err = (a - b).abs().max().item()
        assert err <= TOL, (n, err)


@pytest.mark.parametrize("B,R,N", [(3, 50, 48), (2, 1200, 32), (16, 256, 128)])
def test_fused_backward_matches_fp32_kernels(B, R, N):
    """tp_tc_heads_backward (thin gradients on the tensor pipe inside the dX chain kernel, 5 launches) against the fp32 SIMT
    backward on multi-image / ragged batches: every head and latent gradient within the bf16 contract, bit-identical repeats."""
    from texpose_b200 import mlp_tc_bwd
    S = B * R * N
    assert mlp_tc_bwd.fused_supported(S, R * N)
    g = torch.Generator().manual_seed(11)
    center = (torch.randn(B, R, 3, generator=g) * 0.02 + torch.tensor([0.3, 0.2, -0.8])).to(DEV)
    ray = (torch.randn(B, R, 3, generator=g) * 0.1 + torch.tensor([0.0, 0.0, 1.0])).to(DEV)
    depth = ((torch.rand(B, R, N, 1, generator=g) + torch.arange(N)[None, None, :, None]) / N * 1.2 + 0.2).to(DEV)
    lt0, ll0 = synth.latents(B)
    image = torch.rand(B, R, 3, generator=g).to(DEV)

    def grads(m, opt):
        for p in m.parameters():
            p.grad = None
        lt, ll = lt0.to(DEV).requires_grad_(True), ll0.to(DEV).requires_grad_(True)
        out = m.forward_samples(opt, center, ray, depth, lt, ll, mode="train")
        comp = m.composite(opt, ray, *out[:2], depth, out[2])
        loss = ((image - comp[0]) ** 2 / comp[8] ** 2).mean() + torch.log(comp[8] ** 2).mean() + 0.01 * out[1][..., -1].mean()
        loss.backward()
        named = list(m.mlp_rgb.named_parameters(prefix="mlp_rgb")) + list(m.mlp_trans.named_parameters(prefix="mlp_trans"))
        return [("latent_trans", lt.grad.clone()), ("latent_light", ll.grad.clone())] + [(n, p.grad.clone()) for n, p in named]

    opt16, m16 = _module("bf16")
    _C.launch_counts.clear()
    a = grads(m16, opt16)
    assert _C.launch_counts.get("tp_tc_heads_backward", 0) == 1 and "tp_tc_chain_backward" not in _C.launch_counts
    opt32, m32 = _module("fp32")
    b = grads(m32, opt32)
    worst = 0.0
    for (n, x), (_, y) in zip(a, b):
        err, mag = (x - y).abs().max().item(), y.abs().max().item()
        print(f"  {n:22s} |grad|max {mag:9.3e}  fused-vs-fp32 {err:9.3e}")
        assert x.shape == y.shape and torch.isfinite(x).all()
        assert err <= max(1e-3, 0.02 * mag) and err <= TOL, (n, err, mag)
        worst = max(worst, err)
    print(f"B,R,N = {B},{R},{N}: worst fused-vs-fp32 gradient max-abs error {worst:.2e}")
    # deterministic: fixed-order reductions everywhere
    c = grads(m16, opt16)
    for (n, x), (_, y) in zip(a, c):
        assert torch.equal(x, y), n


def test_backward_falls_back_when_images_are_tiny():
    """Images of 32 samples: a CTA's tile range would touch more than four of them -> tp_tc_heads_backward is not applicable,
    so the forward already routes the batch to the staged kernels (single-pass forward with saved activations, staged dX
    chain); gradients still match the fp32 kernels within the bf16 tolerance."""
    from texpose_b200 import mlp_tc_bwd
    B, R, N = 64, 4, 8
    assert not mlp_tc_bwd.fused_supported(B * R * N, R * N)
    g = torch.Generator().manual_seed(2)
    center = (torch.randn(B, R, 3, generator=g) * 0.02 + torch.tensor([0.3, 0.2, -0.8])).to(DEV)
    ray = (torch.randn(B, R, 3, generator=g) * 0.1 + torch.tensor([0.0, 0.0, 1.0])).to(DEV)
    depth = ((torch.rand(B, R, N, 1, generator=g) + torch.arange(N)[None, None, :, None]) / N * 1.2 + 0.2).to(DEV)
    lt0, ll0 = synth.latents(B)
    res = {}
    for prec in ("bf16", "fp32"):
        opt, m = _module(prec)
        lt, ll = lt0.to(DEV).requires_grad_(True), ll0.to(DEV).requires_grad_(True)
        _C.launch_counts.clear()
        out = m.forward_samples(opt, center, ray, depth, lt, ll, mode="train")
        (out[0].mean() + out[1][..., 1].mean() + out[2].mean()).backward()
        if prec == "bf16":
            assert _C.launch_counts.get("tp_tc32_forward") == 1 and _C.launch_counts.get("tp_tc_chain_backward") == 2
            assert "tp_tc_nerf_stl_forward" not in _C.launch_counts and "tp_tc_heads_backward" not in _C.launch_counts
        res[prec] = [lt.grad, ll.grad] + [p.grad for p in list(m.mlp_rgb.parameters()) + list(m.mlp_trans.parameters())]
    for a, b in zip(res["bf16"], res["fp32"]):
        assert (a - b).abs().max() <= max(1e-3, 0.02 * b.abs().max().item())


@pytest.mark.parametrize("layers_rgb", [[None, 128, 3], [None, 256, 256, 256, 3], [None, 192, 96, 3]])
def test_plain_nerf_renders_on_tensor_cores(layers_rgb):
    """layers/nerf.py in rendering mode (no gradient): the plain model runs through the fused tcgen05 kernel as a padded
    static/transient/light layer image (identity pass-through layers, zero transient head) and stays within the bf16
    contract (<= 1e-2 on rendered rgb / depth / opacity) of its own fp32 kernels; with gradients enabled it keeps using them."""
    from texpose_b200.config import env_opt
    from texpose_b200.layers.nerf import NeRF as PlainNeRF
    opt = env_opt(device=DEV, sample_intvs=64)
    opt.arch.layers_rgb = layers_rgb
    opt.b200 = AttrDict(mlp="bf16")
    torch.manual_seed(1)
    m = PlainNeRF(opt).to(DEV)
    with torch.no_grad():
        for l in list(m.mlp_feat) + list(m.mlp_rgb):
            l.bias.normal_(0.0, 0.05)
    B, R, N = 2, 150, 64
    g = torch.Generator().manual_seed(9)
    center = (torch.randn(B, R, 3, generator=g) * 0.02 + torch.tensor([0.3, 0.2, -8.0])).to(DEV)
    ray = (torch.randn(B, R, 3, generator=g) * 0.05 + torch.tensor([0.0, 0.0, 1.0])).to(DEV)
    depth = ((torch.rand(B, R, N, 1, generator=g) + torch.arange(N)[None, None, :, None]) / N * 2.5 + 6.7).to(DEV)
    assert not m.uses_tensor_cores(opt)                     # parameters want gradients and grad mode is on
    with torch.no_grad():
        assert m.uses_tensor_cores(opt)
        rgb_s, den = m.forward_samples(opt, center, ray, depth, mode="val")
        out = m.composite(opt, ray, rgb_s, den, depth)
        opt32 = env_opt(device=DEV, sample_intvs=64)
        opt32.arch.layers_rgb = layers_rgb
        opt32.b200 = AttrDict(mlp="fp32")
        rgb_32, den_32 = m.forward_samples(opt32, center, ray, depth, mode="val")
        out32 = m.composite(opt32, ray, rgb_32, den_32, depth)
    assert rgb_s.shape == (B, R, N, 3) and den.shape == (B, R, N) and rgb_s.is_contiguous()
    for k in range(3):                                      # rgb, depth, opacity
        assert (out[k] - out32[k]).abs().max() <= 1e-2, (k, (out[k] - out32[k]).abs().max())
    assert (rgb_s - rgb_32).abs().max() <= 3e-2
    # a parameter update must reach the packed image
    with torch.no_grad():
        m.mlp_rgb[-1].bias.add_(0.5)
        rgb_2, _ = m.forward_samples(opt, center, ray, depth, mode="val")
    assert (rgb_2 - rgb_s).abs().max() > 1e-3


def test_static_only_eval_render_matches_the_static_outputs_bit_for_bit():
    """opt.b200.static_only (honoured in mode='eval' on the fused kernel): the stage list stops after the rgb head.  The static
    per-sample outputs and everything composited from them (rgb_static, depth, opacity_static -- what Model.evaluate_full
    uses, model/nerf_adapt_st_gan.py:341-362) are bit-identical to the full launch; the transient outputs are zeros."""
    opt, m = _module("bf16")
    B, R, N = 2, 333, opt.nerf.sample_intvs
    g = torch.Generator().manual_seed(21)
    center = (torch.randn(B, R, 3, generator=g) * 0.02 + torch.tensor([0.3, 0.2, -8.0])).to(DEV)
    ray = (torch.randn(B, R, 3, generator=g) * 0.05 + torch.tensor([0.0, 0.0, 1.0])).to(DEV)
    depth = ((torch.rand(B, R, N, 1, generator=g) + torch.arange(N)[None, None, :, None]) / N * 2.5 + 6.7).to(DEV)
    lt, ll = [t.to(DEV) for t in synth.latents(B)]
    opt_s, _ = _module("bf16")
    opt_s.b200.static_only = True
    with torch.no_grad():
        full = m.forward_samples(opt, center, ray, depth, lt, ll, mode="eval")
        stat = m.forward_samples(opt_s, center, ray, depth, lt, ll, mode="eval")
        val = m.forward_samples(opt_s, center, ray, depth, lt, ll, mode="val")       # only eval honours the switch
        c_full = m.composite(opt, ray, *full[:2], depth, full[2])
        c_stat = m.composite(opt_s, ray, *stat[:2], depth, stat[2])
    assert torch.equal(val[0], full[0]) and torch.equal(val[2], full[2])
    assert torch.equal(stat[0][..., 0], full[0][..., 0]) and torch.equal(stat[1][..., 0], full[1][..., 0])
    assert float(stat[0][..., 1].abs().max()) == 0.0 and float(stat[1][..., 1].abs().max()) == 0.0
    assert float(stat[2].abs().max()) == 0.0
    for k in (1, 3, 5):          # rgb_static, depth, opacity_static
        assert torch.equal(c_stat[k], c_full[k]), k
