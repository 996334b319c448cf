"""CPU emulation of the operand formats a <= 1e-4 tensor-core backward could use (DESIGN.md §2, split backward).

Every Linear layer's backward is recomputed in float64 with its operands rounded where the kernels round them:
    dX = dz W      and      dW = dz^T x      (dz, W and the saved activation x each carried in the candidate format,
                                               the products of the two smallest parts dropped, as the MMA passes drop them)
    db = sum dz    (the column sums read the same dz images)
The forward and every other backward step are the oracle's fp32 autograd (the split forward's own error is measured on the GPU),
so what is left is the error the backward's operand format adds.  It is compared with the oracle's fp32 autograd ("vs fp32") and
with the same backward computed in float64 without rounding ("vs exact"), at the shapes and losses of tests/test_gpu_fp32_train.py.

Formats:
    bf16x2   bf16 hi + lo, three passes (16 significand bits, fp32 exponent range)
    bf16x3   bf16 hi + mid + lo, six passes (24 bits)
    fp16x2s  fp16 hi + lo, dz scaled by a power of two so that max |dz| of the layer sits at 2^14, three passes
    fp16x2   fp16 hi + lo unscaled (the forward's format; shown because it is what a copy of the forward would do)

    python scripts/split_bwd_emulation.py
"""
from __future__ import annotations

import os
import sys
import types

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import texpose_oracle as O  # noqa: E402
from texpose_b200 import synth  # noqa: E402
from texpose_b200.config import adapt_gan_opt, env_opt  # noqa: E402


def _parts(x, fmt):
    if fmt == "bf16x3":
        hi = x.to(torch.bfloat16).double()
        mid = (x - hi).to(torch.bfloat16).double()
        return [hi, mid, (x - hi - mid).to(torch.bfloat16).double()]
    dt = torch.bfloat16 if fmt == "bf16x2" else torch.float16
    hi = x.to(dt).double()
    return [hi, (x - hi).to(dt).double()]


def _scale(dz, fmt):
    if fmt != "fp16x2s":
        return 1.0
    m = dz.abs().max().item()
    return 1.0 if m == 0 else 2.0 ** (14 - torch.tensor(m).log2().floor().item())


def _mm(a, b, fmt, sa=1.0):
    """a @ b with both operands in `fmt`, the MMA passes of the kernels: part i x part j for i + j < number of parts."""
    pa, pb = _parts(a * sa, fmt), _parts(b, fmt)
    n = len(pa)
    out = sum(pa[i] @ pb[j] for i in range(n) for j in range(n) if i + j < n)
    return out / sa


class _Linear(torch.autograd.Function):
    fmt = "exact"

    @staticmethod
    def forward(ctx, x, W, b):
        ctx.save_for_backward(x, W)
        return F.linear(x, W, b)

    @staticmethod
    def backward(ctx, dz):
        x, W = (t.double() for t in ctx.saved_tensors)
        fmt = _Linear.fmt
        shape = x.shape
        dz2, x2 = dz.double().reshape(-1, dz.shape[-1]), x.reshape(-1, shape[-1])
        if fmt == "exact":
            return (dz2 @ W).reshape(shape).float(), (dz2.t() @ x2).float(), dz2.sum(0).float()
        s = _scale(dz2, fmt)
        dx = _mm(dz2, W, fmt, s).reshape(shape)
        dW = _mm(dz2.t().contiguous(), x2, fmt, s)
        db = sum(_parts(dz2 * s, fmt)).sum(0) / s
        return dx.float(), dW.float(), db.float()


_FNS = types.SimpleNamespace(**{k: getattr(F, k) for k in dir(F) if not k.startswith("_")})
_FNS.linear = lambda x, W, b: _Linear.apply(x, W, b)


def _inputs(R, N):
    pose, intr = synth.poses([1]), synth.intrinsics(1)
    c, r = O.get_center_and_ray(pose, intr, 480, 640)
    lo, hi = synth.padded_aabb()
    tn, tf, v = O.aabb_ray_intersection(lo, hi, c, r)
    idx = v[0].nonzero()[:, 0][:R][None]
    rand = torch.rand(1, R, N, 1, generator=torch.Generator().manual_seed(3))
    depth = O.sample_depth(tn[:, idx[0]], tf[:, idx[0]], N, rand)
    return O.gather_rays(c, idx), O.gather_rays(r, idx), depth


def _plain_case(R, N):
    from texpose_b200.layers.nerf import NeRF
    torch.manual_seed(0)
    m = NeRF(env_opt())
    gen = torch.Generator().manual_seed(7)
    with torch.no_grad():
        for lin in list(m.mlp_feat) + list(m.mlp_rgb):
            lin.bias.copy_(torch.randn(lin.bias.shape, generator=gen).mul_(0.2))
    center, ray, depth = _inputs(R, N)
    g = torch.Generator().manual_seed(9)
    image, mask = torch.rand(1, R, 3, generator=g), (torch.rand(1, R, 1, generator=g) > 0.3).float()

    def run():
        fl = [(l.weight.detach().clone().requires_grad_(), l.bias.detach().clone().requires_grad_()) for l in m.mlp_feat]
        rl = [(l.weight.detach().clone().requires_grad_(), l.bias.detach().clone().requires_grad_()) for l in m.mlp_rgb]
        c, r, d = center, ray, depth
        pts = O.points_from_depth(c, r, d)
        unit = F.normalize(r, dim=-1)[..., None, :].expand_as(pts)
        rgb_s, sig = O.nerf_plain_forward(pts, unit, fl, rl)
        comp = O.composite_plain(r, rgb_s, sig, d)
        img, msk = image, mask
        loss = (msk * (img - comp[0]) ** 2).sum() / (msk.sum() + 1e-5) + 0.1 * comp[1].mean() + 0.05 * comp[2].mean() \
            + 0.01 * sig.mean()
        loss.backward()
        return [t.grad for pair in fl + rl for t in pair]

    return run


def _stl_case(arch, R=256, N=64):
    from texpose_b200.layers.nerf_static_transient_light import NeRF
    opt = adapt_gan_opt()
    for k, v in arch.items():
        opt.arch[k] = v
    torch.manual_seed(0)
    m = NeRF(opt)
    gen = torch.Generator().manual_seed(12)
    with torch.no_grad():
        for lin in list(m.mlp_feat) + list(m.mlp_rgb) + list(m.mlp_trans):
            lin.bias.copy_(torch.randn(lin.bias.shape, generator=gen).mul_(0.2))
    center, ray, depth = _inputs(R, N)
    lt, ll = synth.latents(1)
    g = torch.Generator().manual_seed(9)
    image, mask = torch.rand(1, R, 3, generator=g), (torch.rand(1, R, 1, generator=g) > 0.3).float()
    skip = tuple(opt.arch.skip)

    def run():
        fl = [(l.weight.detach(), l.bias.detach()) for l in m.mlp_feat]
        rl = [(l.weight.detach().clone().requires_grad_(), l.bias.detach().clone().requires_grad_()) for l in m.mlp_rgb]
        tl = [(l.weight.detach().clone().requires_grad_(), l.bias.detach().clone().requires_grad_()) for l in m.mlp_trans]
        lt_o, ll_o = lt.detach().clone().requires_grad_(), ll.detach().clone().requires_grad_()
        c, r, d = center, ray, depth
        pts = O.points_from_depth(c, r, d)
        unit = F.normalize(r, dim=-1)[..., None, :].expand_as(pts)
        rgb, dens, unc = O.nerf_stl_forward(pts, unit, lt_o, ll_o, fl, rl, tl, skip=skip)
        comp = O.composite_stl(r, rgb, dens, d, unc, 0.05)
        img, msk = image, mask
        u = comp[8]
        loss = (msk * ((img - comp[0]) ** 2 / u ** 2)).sum() / (msk.sum() + 1e-5) + (5 + torch.log(u ** 2).mean() / 2) \
            + 0.01 * dens[..., -1].mean()
        loss.backward()
        return [lt_o.grad, ll_o.grad] + [t.grad for pair in rl + tl for t in pair]

    return run


CASES = [
    ("plain 1x256x64", lambda: _plain_case(256, 64)),
    ("plain 1x300x24", lambda: _plain_case(300, 24)),
    ("stl yaml", lambda: _stl_case({})),
    ("stl 6x256 skip 2, rgb 2 hidden", lambda: _stl_case(dict(layers_feat=[None] + [256] * 6, skip=[2],
                                                              layers_rgb=[None, 256, 256, 3], layers_trans=[None, 256, 256, 5]))),
    ("stl 8x256, rgb 1 / trans 4 hidden", lambda: _stl_case(dict(layers_feat=[None] + [256] * 8, skip=[4], layers_rgb=[None, 256, 3],
                                                                 layers_trans=[None, 256, 256, 256, 256, 5]))),
]
FORMATS = ["bf16x2", "bf16x3", "fp16x2s", "fp16x2"]


def main():
    print(f"{'case':36s} {'|grad|max':>10s} " + " ".join(f"{f:>19s}" for f in FORMATS))
    print(f"{'':36s} {'':>10s} " + " ".join(f"{'vs fp32 / vs exact':>19s}" for _ in FORMATS))
    worst = {f: 0.0 for f in FORMATS}
    for name, make in CASES:
        run = make()
        ref32 = run()
        saved = O.F
        try:
            O.F = _FNS
            _Linear.fmt = "exact"
            exact = run()
            cols = []
            for fmt in FORMATS:
                _Linear.fmt = fmt
                got = run()
                e32 = max((a - b).abs().max().item() for a, b in zip(got, ref32))
                e64 = max((a - b).abs().max().item() for a, b in zip(got, exact))
                worst[fmt] = max(worst[fmt], e32)
                cols.append(f"{e32:9.2e}/{e64:9.2e}")
        finally:
            O.F = saved
        mag = max(g.abs().max().item() for g in ref32)
        print(f"{name:36s} {mag:10.3e} " + " ".join(f"{c:>19s}" for c in cols), flush=True)
    print("worst max-abs error against the fp32 autograd: " + ", ".join(f"{f} {w:.2e}" for f, w in worst.items()))


if __name__ == "__main__":
    main()
