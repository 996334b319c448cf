"""Training step of the plain model (layers/nerf.py:61-99, options/nerf_lm_env.yaml) on the tensor cores: single-pass bf16
forward with saved activations (csrc/mlp_tc_split.cu), staged dX chain through head and trunk (csrc/mlp_tc_chain.cu), dW GEMMs
on the tile images -- every parameter gradient against the CPU oracle's autograd, bf16 contract (<= 1e-2 max-abs for the
mean-normalised loss), plus the launch accounting that shows the SIMT kernels are out of the step."""
import pytest
import torch

from oracle import texpose_oracle as O
from texpose_b200 import _C
from texpose_b200.config import AttrDict, env_opt
from texpose_b200.layers.nerf import NeRF
from tests import bf16_reference as BR
from tests import gradcheck as G
from tests.test_gpu_tc import _c1_inputs, _check_grads

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-2
# relative bounds beside TOL (max-abs / max|grad|, error norm / norm), 2x the worst measured on one B200
# (profiles/r06_pytest_grads.log).  Oracle step: against the exact oracle the largest-entry error is 5.2e-2 (bound
# REL_EXACT_MAX), but the trunk's early layers sit up to 7.7 % off in norm -- as far as the float64 reference that rounds to bf16
# where the step rounds (tests/bf16_reference.py) sits from the exact oracle: bf16 rounding through eight trunk layers, not the
# kernels.  Against that reference the step measures 7.7e-3 and 1.0e-2, held in both measures (REL_ORACLE).  vs SIMT 128 x 32 9.99e-3, 9.97e-3; C3 shape vs
# SIMT 1.22e-2, 2.23e-2
REL_EXACT_MAX = 0.10
REL_ORACLE = (0.015, 0.020, 0.0)
REL_SIMT = (0.019, 0.019, 0.0)
REL_C3 = (0.024, 0.044, 0.0)


def _models(seed=0):
    opt = env_opt(device=DEV)
    opt.b200 = AttrDict(mlp="bf16")
    torch.manual_seed(seed)
    m = NeRF(opt).to(DEV)
    gen = torch.Generator().manual_seed(7)
    with torch.no_grad():
        for lin in list(m.mlp_feat) + list(m.mlp_rgb):
            lin.bias.copy_(torch.randn(lin.bias.shape, generator=gen).mul_(0.2).to(DEV))
    cpu = NeRF(env_opt())
    cpu.load_state_dict(m.state_dict())
    return opt, m, cpu


def _loss(rgb, depth, opacity, sigma, image, mask):
    return (mask * (image - rgb) ** 2).sum() / (mask.sum() + 1e-5) + 0.1 * depth.mean() + 0.05 * opacity.mean() + 0.01 * sigma.mean()


@pytest.mark.parametrize("R,N", [(256, 64), (300, 24)])
def test_plain_training_step_gradients_vs_oracle(R, N):
    center, ray, depth = _c1_inputs(R=R, N=N, seed_pose=1)
    opt, m, cpu = _models()
    g = torch.Generator().manual_seed(9)
    image, mask = torch.rand(1, R, 3, generator=g), (torch.rand(1, R, 1, generator=g) > 0.3).float()
    # ---- oracle (CPU, fp32, autograd)
    fl = [(l.weight, l.bias) for l in cpu.mlp_feat]
    rl = [(l.weight, l.bias) for l in cpu.mlp_rgb]
    pts = O.points_from_depth(center, ray, depth)
    unit = torch.nn.functional.normalize(ray, dim=-1)[..., None, :].expand_as(pts)
    rgb_s, sig = O.nerf_plain_forward(pts, unit, fl, rl)
    comp = O.composite_plain(ray, rgb_s, sig, depth)
    _loss(comp[0], comp[1], comp[2], sig, image, mask).backward()
    # ---- tensor cores
    assert m.trains_on_tensor_cores(opt)
    _C.launch_counts.clear()
    rgb_g, sig_g = m.forward_samples(opt, center.to(DEV), ray.to(DEV), depth.to(DEV), mode="train")
    comp_g = m.composite(opt, ray.to(DEV), rgb_g, sig_g, depth.to(DEV))
    _loss(comp_g[0], comp_g[1], comp_g[2], sig_g, image.to(DEV), mask.to(DEV)).backward()
    assert _C.launch_counts.get("tp_tc32_forward") == 1 and _C.launch_counts.get("tp_tc_chain_backward") == 1
    assert _C.launch_counts.get("tp_tc_dw_gemm") == 1 and "tp_linear_forward" not in _C.launch_counts
    assert "tp_linear_backward_input" not in _C.launch_counts
    assert (rgb_g.cpu() - rgb_s).abs().max() <= 2e-2 and (comp_g[0].cpu() - comp[0]).abs().max() <= TOL
    # ---- the bf16-rounding reference (float64, rounded where the step rounds: tests/bf16_reference.py), same loss
    P = [(l.weight.detach().double().requires_grad_(True), l.bias.detach().double().requires_grad_(True))
         for l in list(cpu.mlp_feat) + list(cpu.mlp_rgb)]
    rgb_r, sig_r = BR.plain_forward(pts.double(), unit.double(), P[:len(cpu.mlp_feat)], P[len(cpu.mlp_feat):])
    comp_r = O.composite_plain(ray.double(), rgb_r, sig_r, depth.double())
    _loss(comp_r[0], comp_r[1], comp_r[2], sig_r, image.double(), mask.double()).backward()
    ref = [t.grad for pair in P for t in pair]
    pairs, gap = [], 0.0
    for (n, a), b, r in zip(list(m.mlp_feat.named_parameters(prefix="mlp_feat")) + list(m.mlp_rgb.named_parameters(prefix="mlp_rgb")),
                            list(cpu.mlp_feat.parameters()) + list(cpu.mlp_rgb.parameters()), ref):
        assert a.grad is not None and a.grad.shape == b.grad.shape, n
        # the exact oracle: the north-star absolute bound and the largest-entry bound
        err, (e_max, _) = float((a.grad.cpu() - b.grad).abs().max()), G.rel_errors(a.grad, b.grad)
        assert err <= TOL and e_max <= REL_EXACT_MAX, (n, err, e_max)
        gap = max(gap, G.rel_errors(r, b.grad.double())[1])
        pairs.append((n, a.grad, r))
    print(f"plain {R}x{N}: bf16-rounding reference vs exact oracle, worst error norm / norm {gap:.3e}")
    _check_grads(f"plain {R}x{N} tensor-core step vs bf16-rounding reference", pairs, REL_ORACLE)


def test_plain_training_is_deterministic_and_fp32_mode_keeps_simt():
    center, ray, depth = [t.to(DEV) for t in _c1_inputs(R=128, N=32)]
    opt, m, _ = _models()

    def grads(o):
        for p in m.parameters():
            p.grad = None
        rgb, sig = m.forward_samples(o, center, ray, depth, mode="train")
        (rgb.square().mean() + sig.mean()).backward()
        return [p.grad.clone() for p in m.parameters()]

    a, b = grads(opt), grads(opt)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    o32 = env_opt(device=DEV)
    o32.b200 = AttrDict(mlp="fp32")
    _C.launch_counts.clear()
    c = grads(o32)
    assert "tp_tc_chain_backward" not in _C.launch_counts and _C.launch_counts.get("tp_linear_forward", 0) > 0
    _check_grads("plain 128x32 tensor-core vs SIMT", [(n, x, y) for (n, _), x, y in zip(m.named_parameters(), a, c)], REL_SIMT)


def test_chain_stage_list_is_validated():
    from texpose_b200 import ops
    lib = _C.load()
    z = torch.zeros(1 << 16, device=DEV)
    img = torch.zeros(9 * 16384, dtype=torch.uint8, device=DEV)

    def run(rows, thin1=None):
        st = torch.tensor(rows, dtype=torch.int32)
        return lib.tp_tc_chain_backward(ops._p(z), 3, thin1, 1, 128, ops._p(img), 9, ops._p(st), len(rows), ops._p(img), 2, ops._p(img), 2, None)

    assert run([[0, 0, 0, 0, 0, 0], [-1, 0, 1, 8, 1, 1]]) == 0
    assert run([[-1, 0, 1, 8, 0, 0]]) == -1                      # the first stage reads an A tile nobody wrote
    assert run([[1, 0, 0, 0, 0, 0]]) == -1                       # thin operand 1 is absent
    assert run([[0, 0, 0, 0, 0, 0], [-1, 0, 4, 8, 1, 1]]) == -1  # chunks beyond the image
    assert run([[0, 0, 0, 0, 2, 0]]) == -1                       # mask slot beyond the saved images
    torch.cuda.synchronize()


def test_plain_training_step_at_the_c3_shape_matches_the_simt_step():
    """16 x 256 rays x 128 samples (BASELINE C3 shape) of the plain model: tensor-core step against the fp32 SIMT step, every
    gradient within the bf16 contract, and the step is deterministic."""
    B, R, N = 16, 256, 128
    g = torch.Generator().manual_seed(0)
    center = (torch.randn(B, R, 3, generator=g) * 0.02 + torch.tensor([0.3, 0.2, -0.8])).to(DEV)
    ray = (torch.randn(B, R, 3, generator=g) * 0.1 + torch.tensor([0.0, 0.0, 1.0])).to(DEV)
    depth = ((torch.rand(B, R, N, 1, generator=g) + torch.arange(N)[None, None, :, None]) / N * 1.2 + 0.2).to(DEV)
    image = torch.rand(B, R, 3, generator=g).to(DEV)
    opt, m, _ = _models()
    o32 = env_opt(device=DEV)
    o32.b200 = AttrDict(mlp="fp32")

    def grads(o):
        for p in m.parameters():
            p.grad = None
        rgb_s, sig = m.forward_samples(o, center, ray, depth, mode="train")
        comp = m.composite(o, ray, rgb_s, sig, depth)
        (((comp[0] - image) ** 2).mean() + 0.1 * comp[1].mean() + 0.01 * sig.mean()).backward()
        return [p.grad.clone() for p in m.parameters()]

    a, a2, ref = grads(opt), grads(opt), grads(o32)
    for (n, _), x, x2 in zip(m.named_parameters(), a, a2):
        assert torch.equal(x, x2), n
    _check_grads("plain C3 shape tensor-core vs SIMT", [(n, x, y) for (n, _), x, y in zip(m.named_parameters(), a, ref)], REL_C3)
