"""Test helper (not a test): the plain model's forward and backward in float64 with bf16 rounding where the tensor-core step rounds.

The plain model's bf16 step (texpose_b200/mlp_tc_plain.py) rounds to bf16 at fixed points: the weights of every GEMM, the
inputs the single-pass forward stores as tile images (the encoding, every hidden activation, the trunk feature, the sample
points), and every dz the staged chain stores as a tile image before it feeds the dX and dW GEMMs.  Everything else is exact
here.  Against this reference the kernels' gradients differ only by accumulation order, so their error is held to the bf16
caps.  The distance from this reference to the exact oracle is what bf16 rounding alone costs: 8 trunk layers of it reach 3.7-12 %
of the early trunk layers' gradient norm.  With `rounding=False` this is the exact oracle (tests/test_gradcheck_helper.py)."""
import torch
import torch.nn.functional as F

from oracle import texpose_oracle as O


def _r(x, on):
    """bf16 rounding in the forward, identity in the backward (the backward rounds only where _Linear does)."""
    return x + (x.detach().to(torch.bfloat16).to(x.dtype) - x.detach()) if on else x


class _Linear(torch.autograd.Function):
    """y = x W_r^T + b; backward with dz rounded: dx = dz_r W_r, dW = dz_r^T x, db = sum dz_r (x as handed in)."""

    @staticmethod
    def forward(ctx, x, W, b, on):
        Wr = _r(W, on)
        ctx.save_for_backward(x, Wr)
        ctx.on = on
        return x @ Wr.t() + b

    @staticmethod
    def backward(ctx, g):
        x, Wr = ctx.saved_tensors
        Wr = Wr.detach()
        gr = _r(g, ctx.on)
        flat_g, flat_x = gr.reshape(-1, gr.shape[-1]), x.reshape(-1, x.shape[-1])
        return gr @ Wr, flat_g.t() @ flat_x, flat_g.sum(0), None


def plain_forward(points, ray_unit, feat_layers, rgb_layers, rounding=True, L_3D=10, L_view=4, skip=(4,)):
    """O.nerf_plain_forward with the kernels' bf16 rounding points.  points / ray_unit: float64 copies of the float32 values the
    kernels use; the encodings are the reference's float32 ones."""
    r = lambda x: _r(x, rounding)
    enc = torch.cat([points, O.positional_encoding(points.float(), L_3D).to(points.dtype)], dim=-1)
    h, sigma_raw = r(enc), None
    for li, (W, b) in enumerate(feat_layers):
        if li in skip:
            h = torch.cat([h, r(enc)], dim=-1)
        h = _Linear.apply(h, W, b, rounding)
        if li == len(feat_layers) - 1:
            sigma_raw, h = h[..., 0], h[..., 1:]
        h = r(F.relu(h))
    view = torch.cat([ray_unit, O.positional_encoding(ray_unit.float(), L_view).to(ray_unit.dtype)], dim=-1)
    x = torch.cat([h, view, r(points)], dim=-1)          # the view columns enter as an exact per-ray bias
    for li, (W, b) in enumerate(rgb_layers):
        x = _Linear.apply(x, W, b, rounding)
        if li != len(rgb_layers) - 1:
            x = r(F.relu(x))
    return torch.sigmoid(x), F.softplus(sigma_raw)
