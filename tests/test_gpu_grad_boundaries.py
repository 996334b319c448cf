"""Gradients of losses seeded only at the edges of the tensor-core backward's bookkeeping, against the oracle's autograd in
float64.  A loss that touches every sample averages a misplaced tile, ray or image away; here the per-sample cotangent is
non-zero only on
  (a) the last, partial 128-row tile,
  (b) one image in the middle of a batch whose image boundaries fall inside tiles (R * N not a multiple of 128),
  (c) one ray that straddles a tile boundary (N = 24: ray 5 covers samples 120 - 143; N = 12: ray 10 covers 120 - 131),
for each of the four backward engines, and the launch counts show which one ran (the plain model against the float64
reference that rounds to bf16 where its step rounds, tests/bf16_reference.py -- against the exact oracle its trunk's early
layers sit 3.7-12 % off in norm from bf16 rounding alone):
  fused        tp_tc_heads_backward after the lock-step forward (fused_supported),
  staged_bf16  single-pass forward with save + tp_tc_chain_backward (images of 24 samples: fused_supported is false),
  split        the <= 1e-4 mode (opt.b200.fp32_engine = 'tc'): split-save forward + tp_tc_chain_backward_split,
  plain        the plain model's staged chain (trunk and head trainable).
Every head (and, for the plain model, trunk) gradient within the relative bounds of tests/gradcheck.py; the per-image latent
tables row by row, and rows of images the seed does not touch exactly zero.  The oracle runs in float64 on the float32 points
and the reference's float32 positional encoding (the argument rounded as the reference and the kernels round it).

Measured on one B200 (profiles/r06_pytest_grads.log): worst relative errors per engine beside REL.  The seeds are positive, as a
loss that pulls every output the same way gives them; with random signs the gradients are sums with heavy cancellation, whose
relative error is the bf16 rounding times the cancellation factor (up to 30 % measured)."""
import pytest
import torch

from oracle import texpose_oracle as O
from texpose_b200 import _C, mlp_tc_bwd, synth
from texpose_b200.config import AttrDict, adapt_gan_opt, env_opt
from texpose_b200.layers import nerf, nerf_static_transient_light
from tests import bf16_reference as BR
from tests import gradcheck as G

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

ENGINES = {
    "fused": dict(model="stl", b200=dict(mlp="bf16"), shape=(3, 50, 24), counts={"tp_tc_heads_backward": 1},
                  absent=("tp_tc_chain_backward",)),
    "staged_bf16": dict(model="stl", b200=dict(mlp="bf16"), shape=(30, 2, 12),
                        counts={"tp_tc32_forward": 1, "tp_tc_chain_backward": 2}, absent=("tp_tc_heads_backward",)),
    "split": dict(model="stl", b200=dict(mlp="fp32", fp32_engine="tc"), shape=(3, 50, 24),
                  counts={"tp_tc32_forward_split_save": 1, "tp_tc_chain_backward_split": 2}, absent=("tp_linear_forward",)),
    "plain": dict(model="plain", b200=dict(mlp="bf16"), shape=(3, 50, 24),
                  counts={"tp_tc32_forward": 1, "tp_tc_chain_backward": 1}, absent=("tp_linear_forward",)),
}
# (max-abs error / max|grad|, error norm / norm, latent row error / row norm).  Worst measured over the seeds on one B200:
#   fused        7.7e-2, 3.6e-2, 3.6e-2 (last tile)
#   staged_bf16  8.9e-2, 4.7e-2, 4.4e-2 (straddling ray; last two tiles)
#   split        5.7e-4, 1.8e-4, 1.7e-4 (middle image)
#   plain        5.3e-2, 3.5e-2, -      (last tile; against the bf16-rounding reference, which itself sits 3.7-12 % in norm from
#                                        the exact oracle: 12 % under the 16-sample last-tile seed)
# bf16 bounds are 2x those, but at most 10 % / 5 % / 5 %
REL = {
    "fused": (0.10, 0.05, 0.05),
    "staged_bf16": (0.10, 0.05, 0.05),
    "split": (1e-3, 3.6e-4, 3.4e-4),
    "plain": (0.10, 0.05, 0.0),
}


def _region(kind, B, R, N):
    """Flat sample indices [S] (bool) where the seed is non-zero."""
    S, P = B * R * N, R * N
    keep = torch.zeros(S, dtype=torch.bool)
    if kind == "last_tile":
        assert S % 128 != 0
        keep[(S - 1) // 128 * 128:] = True
    elif kind == "last_two_tiles":
        keep[((S - 1) // 128 - 1) * 128:] = True
    elif kind == "middle_image":
        j = min((j for j in range(1, B - 1) if (j * P) % 128 and ((j + 1) * P) % 128), key=lambda j: abs(j - B // 2))
        keep[j * P:(j + 1) * P] = True
    elif kind == "straddling_ray":
        assert 128 % N != 0
        r = 128 // N
        keep[r * N:(r + 1) * N] = True
        assert r * N < 128 < (r + 1) * N
    return keep


def _problem(engine):
    e = ENGINES[engine]
    B, R, N = e["shape"]
    g = torch.Generator().manual_seed(11)
    center = torch.randn(B, R, 3, generator=g) * 0.02 + torch.tensor([0.3, 0.2, -0.8])
    ray = torch.randn(B, R, 3, generator=g) * 0.1 + torch.tensor([0.0, 0.0, 1.0])
    depth = (torch.rand(B, R, N, 1, generator=g) + torch.arange(N)[None, None, :, None]) / N * 1.2 + 0.2
    if e["model"] == "stl":
        opt = adapt_gan_opt(device=DEV)
        opt.b200 = AttrDict(e["b200"])
        torch.manual_seed(0)
        m = nerf_static_transient_light.NeRF(opt).to(DEV)
        heads = list(m.mlp_rgb.named_parameters(prefix="mlp_rgb")) + list(m.mlp_trans.named_parameters(prefix="mlp_trans"))
    else:
        opt = env_opt(device=DEV)
        opt.b200 = AttrDict(e["b200"])
        torch.manual_seed(0)
        m = nerf.NeRF(opt).to(DEV)
        heads = list(m.mlp_feat.named_parameters(prefix="mlp_feat")) + list(m.mlp_rgb.named_parameters(prefix="mlp_rgb"))
    gen = torch.Generator().manual_seed(12)
    with torch.no_grad():
        for lin in m.modules():
            if isinstance(lin, torch.nn.Linear):
                lin.bias.copy_(torch.randn(lin.bias.shape, generator=gen).mul_(0.2).to(DEV))
    lt, ll = synth.latents(B)
    w = [torch.rand(B, R, N, 3, 2, generator=g) + 0.5, torch.rand(B, R, N, 2, generator=g) + 0.5, torch.rand(B, R, N, 1, generator=g) + 0.5]
    if e["model"] == "plain":
        w = [w[0][..., 0], w[1][..., 0]]
    return dict(e=e, opt=opt, m=m, heads=heads, center=center, ray=ray, depth=depth, lt=lt, ll=ll, w=w)


def _seeds(pb, keep):
    B, R, N = pb["e"]["shape"]
    k = keep.view(B, R, N).double()
    return [wi.double() * k.view(B, R, N, *([1] * (wi.dim() - 3))) for wi in pb["w"]]


def _kernel(pb, seeds):
    m, opt = pb["m"], pb["opt"]
    for p in m.parameters():
        p.grad = None
    center, ray, depth = pb["center"].to(DEV), pb["ray"].to(DEV), pb["depth"].to(DEV)
    _C.launch_counts.clear()
    if pb["e"]["model"] == "stl":
        lt, ll = pb["lt"].to(DEV).requires_grad_(True), pb["ll"].to(DEV).requires_grad_(True)
        out = m.forward_samples(opt, center, ray, depth, lt, ll, mode="train")
    else:
        out = m.forward_samples(opt, center, ray, depth, mode="train")
    sum((o * s.float().to(DEV)).sum() for o, s in zip(out, seeds)).backward()
    counts = dict(_C.launch_counts)
    got = {n: p.grad.detach().cpu() for n, p in pb["heads"]}
    if pb["e"]["model"] == "stl":
        got.update(latent_trans=lt.grad.detach().cpu(), latent_light=ll.grad.detach().cpu())
    return got, counts


def _oracle(pb, seeds, monkeypatch, bf16=False):
    """float64 autograd of the same loss; the encoding as the reference computes it (float32 argument and sin / cos).  bf16: the
    plain model through tests/bf16_reference.py, rounded to bf16 where its tensor-core step rounds."""
    real = O.positional_encoding
    monkeypatch.setattr(O, "positional_encoding", lambda x, L: real(x.float(), L).to(x.dtype))
    m = pb["m"]
    pts = O.points_from_depth(pb["center"], pb["ray"], pb["depth"])                     # float32, as the kernels form them
    unit = torch.nn.functional.normalize(pb["ray"], dim=-1)[..., None, :].expand_as(pts)
    pts, unit = pts.double(), unit.double()
    P = {n: p.detach().cpu().double().requires_grad_(True) for n, p in pb["heads"]}
    layers = lambda prefix, ml: [(P.get(f"{prefix}.{i}.weight", l.weight.detach().cpu().double()),
                                  P.get(f"{prefix}.{i}.bias", l.bias.detach().cpu().double())) for i, l in enumerate(ml)]
    if pb["e"]["model"] == "stl":
        lt, ll = pb["lt"].double().requires_grad_(True), pb["ll"].double().requires_grad_(True)
        out = O.nerf_stl_forward(pts, unit, lt, ll, layers("mlp_feat", m.mlp_feat), layers("mlp_rgb", m.mlp_rgb),
                                 layers("mlp_trans", m.mlp_trans))
    else:
        fwd = BR.plain_forward if bf16 else O.nerf_plain_forward
        out = fwd(pts, unit, layers("mlp_feat", m.mlp_feat), layers("mlp_rgb", m.mlp_rgb))
    sum((o * s).sum() for o, s in zip(out, seeds)).backward()
    monkeypatch.setattr(O, "positional_encoding", real)
    want = {n: (p.grad if p.grad is not None else torch.zeros_like(p)) for n, p in P.items()}
    if pb["e"]["model"] == "stl":
        want.update(latent_trans=lt.grad, latent_light=ll.grad)
    return want


def _check(tag, got, want, rows_used, rel):
    worst = [0.0, 0.0, 0.0]
    for n in want:
        e = G.assert_grad_close(n, got[n], want[n], rel_max=rel[0], rel_norm=rel[1], tag=tag)
        r = G.assert_latent_rows(got[n], want[n], rows_used, rel[2], name=n, tag=tag) if n.startswith("latent") else 0.0
        worst = [max(x, y) for x, y in zip(worst, (e[0], e[1], r))]
    print(f"{tag}: worst relative errors: max-abs {worst[0]:.3e}, norm {worst[1]:.3e}, latent row {worst[2]:.3e}")
    return worst


def _run(engine, kind, monkeypatch):
    pb = _problem(engine)
    B, R, N = pb["e"]["shape"]
    keep = _region(kind, B, R, N)
    seeds = _seeds(pb, keep)
    got, counts = _kernel(pb, seeds)
    for k, v in pb["e"]["counts"].items():
        assert counts.get(k) == v, (engine, counts)
    for k in pb["e"]["absent"]:
        assert k not in counts, (engine, counts)
    if engine in ("fused", "staged_bf16"):
        assert mlp_tc_bwd.fused_supported(B * R * N, R * N) == (engine == "fused")
    want = _oracle(pb, seeds, monkeypatch, bf16=engine == "plain")
    if engine == "plain":            # what bf16 rounding alone costs: the exact oracle against the bf16-rounding reference
        exact = _oracle(pb, seeds, monkeypatch)
        gap = max(G.rel_errors(want[n], exact[n])[1] for n in want)
        print(f"plain/{kind}: bf16-rounding reference vs exact oracle, worst error norm / norm {gap:.3e}")
    rows_used = sorted({int(i) for i in (keep.view(B, R * N).any(dim=1)).nonzero()[:, 0]})
    return pb, keep, got, want, rows_used


@pytest.mark.parametrize("kind", ["last_tile", "middle_image", "straddling_ray"])
@pytest.mark.parametrize("engine", list(ENGINES))
def test_boundary_seeded_gradients_vs_float64_oracle(engine, kind, monkeypatch):
    pb, keep, got, want, rows_used = _run(engine, kind, monkeypatch)
    B, R, N = pb["e"]["shape"]
    print(f"{engine} {B}x{R}x{N}, seed on {kind}: samples {int(keep.nonzero()[0])}..{int(keep.nonzero()[-1])}, images {rows_used}")
    _check(f"{engine}/{kind}", got, want, rows_used, REL[engine])


@pytest.mark.parametrize("engine", list(ENGINES))
def test_dropped_last_partial_tile_is_rejected(engine, monkeypatch):
    """Seed on the last two tiles; the kernel's gradients pass, and the same gradients moved by the oracle's difference for a
    dropped last partial tile (its seeds zeroed) are rejected."""
    pb, keep, got, want, rows_used = _run(engine, "last_two_tiles", monkeypatch)
    B, R, N = pb["e"]["shape"]
    S = B * R * N
    _check(f"{engine}/last_two_tiles", got, want, rows_used, REL[engine])
    keep_drop = keep.clone()
    keep_drop[(S - 1) // 128 * 128:] = False
    dropped = _oracle(pb, _seeds(pb, keep_drop), monkeypatch, bf16=engine == "plain")
    mutant = {n: got[n] + (dropped[n] - want[n]).float() for n in got}
    with pytest.raises(AssertionError):
        _check(f"{engine}/last_two_tiles, last tile dropped", mutant, want, rows_used, REL[engine])
