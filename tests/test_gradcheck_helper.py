"""The relative gradient checks of tests/gradcheck.py reject the kernel bugs an absolute 1e-2 bound lets through.

At a small static/transient/light problem (3 images of 10 rays x 24 samples: S = 720, a partial last tile of 80 samples; a latent
table of 4 rows, image i on row i) the oracle's fp32 gradients are taken, then mutated the way a wrong reduction kernel would
mutate them.  The helper, at the loosest bounds the bf16 tests may use (10 % max-abs, 5 % norm, 5 % per latent row), must reject
every mutant and accept the oracle plus noise at the bf16 kernels' measured error level."""
import pytest
import torch

from oracle import texpose_oracle as O
from texpose_b200 import synth
from texpose_b200.config import adapt_gan_opt
from texpose_b200.layers.nerf_static_transient_light import NeRF
from tests import gradcheck as G
from tests.conftest import layer_list

B, R, N, ROWS = 3, 10, 24, 4
S = B * R * N
REL_MAX, REL_NORM, REL_ROW = 0.10, 0.05, 0.05          # the caps of the bf16 contract's relative checks
IDX = torch.arange(B)                                  # image i -> latent row i; row 3 is never touched


def _oracle_grads(keep=None):
    """{name: grad} of a C3-like loss; `keep` [B,R,N] (0 / 1) zeroes the per-sample seeds of the samples it masks."""
    g = torch.Generator().manual_seed(5)
    center = torch.randn(B, R, 3, generator=g) * 0.02 + torch.tensor([0.3, 0.2, -0.8])
    ray = torch.randn(B, R, 3, generator=g) * 0.1 + torch.tensor([0.0, 0.0, 1.0])
    depth = (torch.rand(B, R, N, 1, generator=g) + torch.arange(N)[None, None, :, None]) / N * 1.2 + 0.2
    image = torch.rand(B, R, 3, generator=g)
    torch.manual_seed(0)
    cpu = NeRF(adapt_gan_opt())
    lt_tab = (torch.randn(ROWS, 16, generator=g) * 0.5).requires_grad_(True)
    ll_tab = (torch.randn(ROWS, 48, generator=g) * 0.5).requires_grad_(True)
    for p in list(cpu.mlp_rgb.parameters()) + list(cpu.mlp_trans.parameters()):
        p.requires_grad_(True)
    rl = [(l.weight, l.bias) for l in cpu.mlp_rgb]
    tl = [(l.weight, l.bias) for l in cpu.mlp_trans]
    pts = O.points_from_depth(center, ray, depth)
    unit = torch.nn.functional.normalize(ray, dim=-1)[..., None, :].expand_as(pts)
    rgb, dens, unc = O.nerf_stl_forward(pts, unit, lt_tab[IDX], ll_tab[IDX], layer_list(cpu.mlp_feat), rl, tl)
    if keep is not None:
        rgb = G.cotangent_mask(rgb, keep[..., None, None])
        dens = G.cotangent_mask(dens, keep[..., None])
        unc = G.cotangent_mask(unc, keep[..., None])
    comp = O.composite_stl(ray, rgb, dens, depth, unc, 0.05)
    loss = ((image - comp[0]) ** 2 / comp[8] ** 2).mean() + torch.log(comp[8] ** 2).mean() + 0.01 * dens[..., -1].mean()
    loss.backward()
    out = {"latent_trans": lt_tab.grad, "latent_light": ll_tab.grad}
    for n, p in list(cpu.mlp_rgb.named_parameters(prefix="mlp_rgb")) + list(cpu.mlp_trans.named_parameters(prefix="mlp_trans")):
        out[n] = p.grad
    return {k: v.detach().clone() for k, v in out.items()}


@pytest.fixture(scope="module")
def want():
    return _oracle_grads()


def _accepts(got, want):
    try:
        for k in want:
            if k.startswith("latent"):
                G.assert_latent_rows(got[k], want[k], IDX.tolist(), REL_ROW, name=k)
            G.assert_grad_close(k, got[k], want[k], rel_max=REL_MAX, rel_norm=REL_NORM)
    except AssertionError as e:
        print("  rejected:", e)
        return False
    return True


def _dropped(keep):
    return _oracle_grads(keep)


def _keep_all_but(sample_lo, sample_hi):
    keep = torch.ones(S)
    keep[sample_lo:sample_hi] = 0
    return keep.view(B, R, N)


def test_the_oracle_itself_and_noise_at_the_measured_level_are_accepted(want):
    assert _accepts(want, want)
    # the worst bf16 kernel errors measured: 8.9 % of max|grad| (max-abs), 4.7 % of the norm, 4.85 % of a latent row's norm
    g = torch.Generator().manual_seed(1)
    noisy = {}
    for k, w in want.items():
        n = torch.randn(w.shape, generator=g)
        d = n / n.abs().max() * (0.089 * float(w.abs().max()))
        d = d * min(1.0, 0.047 * float(w.norm()) / float(d.norm()))
        if k.startswith("latent"):      # per-row budget; untouched rows stay exactly zero
            d[ROWS - 1] = 0
            d = d * min(1.0, min(0.0485 * float(w[r].norm()) / max(float(d[r].norm()), 1e-30) for r in range(B)))
        noisy[k] = w + d
    assert _accepts(noisy, want)


def test_absolute_bound_alone_lets_a_zeroed_latent_gradient_pass(want):
    """The gap the relative checks close: the per-image latent gradients here are far below the 1e-2 absolute bound, so a zeroed
    table passes `max|got - want| <= 1e-2`; the relative check rejects it."""
    zero = torch.zeros_like(want["latent_light"])
    assert float((zero - want["latent_light"]).abs().max()) <= 1e-2
    assert not _accepts({**want, "latent_light": zero}, want)


@pytest.mark.parametrize("mutant", ["zeroed", "halved", "rows_swapped", "image_dropped", "last_tile_dropped"])
def test_every_mutant_is_rejected(want, mutant):
    if mutant == "zeroed":
        cases = [{**want, k: torch.zeros_like(want[k])} for k in want]
    elif mutant == "halved":
        cases = [{**want, k: want[k] * 0.5} for k in want]
    elif mutant == "rows_swapped":
        cases = [{**want, k: G.swap_rows(want[k], 0, 1)} for k in ("latent_trans", "latent_light")]
    elif mutant == "image_dropped":                                   # the middle image's seed zeroed
        cases = [_dropped(_keep_all_but(R * N, 2 * R * N))]
    else:                                                              # the samples of the last, partial 128-row tile
        cases = [_dropped(_keep_all_but((S - 1) // 128 * 128, S))]
    assert S % 128 != 0
    for got in cases:
        assert not _accepts(got, want), mutant


def test_the_bf16_rounding_reference_is_the_oracle_without_rounding():
    """tests/bf16_reference.py computes the oracle's plain model when its rounding is off (so it is the same operation), and its
    rounding moves the gradients by the bf16 scale, not more."""
    from tests import bf16_reference as BR
    from texpose_b200.config import env_opt
    from texpose_b200.layers.nerf import NeRF as PlainNeRF
    g = torch.Generator().manual_seed(3)
    center = torch.randn(2, 5, 3, generator=g) * 0.02 + torch.tensor([0.3, 0.2, -0.8])
    ray = torch.randn(2, 5, 3, generator=g) * 0.1 + torch.tensor([0.0, 0.0, 1.0])
    depth = (torch.rand(2, 5, 24, 1, generator=g) + torch.arange(24)[None, None, :, None]) / 24 * 1.2 + 0.2
    torch.manual_seed(0)
    m = PlainNeRF(env_opt())
    pts = O.points_from_depth(center, ray, depth)
    unit = torch.nn.functional.normalize(ray, dim=-1)[..., None, :].expand_as(pts)
    seeds = (torch.rand(2, 5, 24, 3, generator=g).double(), torch.rand(2, 5, 24, generator=g).double())

    def grads(fn, **kw):
        P = [(l.weight.detach().double().requires_grad_(True), l.bias.detach().double().requires_grad_(True))
             for l in list(m.mlp_feat) + list(m.mlp_rgb)]
        fl, rl = P[:len(m.mlp_feat)], P[len(m.mlp_feat):]
        rgb, den = fn(pts.double(), unit.double(), fl, rl, **kw)
        ((rgb * seeds[0]).sum() + (den * seeds[1]).sum()).backward()
        return [t.grad for pair in P for t in pair]

    real = O.positional_encoding
    try:
        O.positional_encoding = lambda x, L: real(x.float(), L).to(x.dtype)
        exact = grads(O.nerf_plain_forward)
    finally:
        O.positional_encoding = real
    off = grads(BR.plain_forward, rounding=False)
    on = grads(BR.plain_forward, rounding=True)
    for a, b, c in zip(exact, off, on):
        assert float((a - b).abs().max()) <= 1e-12 * max(1.0, float(a.abs().max()))
        e = G.rel_errors(c, a)[1]
        assert 0 < e < 0.2, e
