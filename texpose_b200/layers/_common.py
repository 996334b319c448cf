"""Shared host-side pieces of the two NeRF module mirrors."""
from __future__ import annotations

import os

import torch

from .. import ops
from ._mlp import MLPConfig


def layer_dims(layers):
    """util.get_layer_dims (util.py:277-279)."""
    return list(zip(layers[:-1], layers[1:]))


def tf_init_(linear: torch.nn.Linear, out=None):
    """Xavier ("TensorFlow style") init with the same RNG draw order as
    NeRF.tensorflow_init_weights (layers/nerf_static_transient_light.py:63-74), so that
    torch.manual_seed(s); NeRF(opt) reproduces the reference's weights bit for bit."""
    gain = torch.nn.init.calculate_gain("relu")
    if out == "all":
        torch.nn.init.xavier_uniform_(linear.weight)
    elif out == "first":
        torch.nn.init.xavier_uniform_(linear.weight[:1])
        torch.nn.init.xavier_uniform_(linear.weight[1:], gain=gain)
    else:
        torch.nn.init.xavier_uniform_(linear.weight, gain=gain)
    torch.nn.init.zeros_(linear.bias)


def mlp_precision(opt) -> str:
    """'fp32' (SIMT kernels, <=1e-4 parity with the reference), 'bf16' (tcgen05 forward + backward, <=1e-2) or 'auto' = bf16
    whenever the fused kernel implements the architecture (options/nerf_lm_adapt_gan.yaml, frozen trunk, ray-parameterised
    call) and fp32 otherwise.  opt.b200.mlp > $TEXPOSE_B200_MLP > auto."""
    b = opt.get("b200") if hasattr(opt, "get") else None
    p = (b.get("mlp") if b else None) or os.environ.get("TEXPOSE_B200_MLP") or "auto"
    if p not in ("fp32", "bf16", "auto"):
        raise ValueError(f"unknown MLP precision {p!r}")
    return p


def b200_option(opt, name, default=None):
    """opt.b200.<name> (the extension block of the options; absent in the reference yamls)."""
    b = opt.get("b200") if hasattr(opt, "get") else None
    v = b.get(name) if b else None
    return default if v is None else v


def given_keywords(**kw):
    """The optional keywords a caller was given (None = absent), so that a call passes them on only when they were given."""
    return {k: v for k, v in kw.items() if v is not None}


def flat_params(*module_lists):
    out = []
    for ml in module_lists:
        if ml is None:
            continue
        for lin in ml:
            out += [lin.weight, lin.bias]
    return out


def ray_geometry(cfg: MLPConfig, center, ray, depth_samples):
    """Inputs of forward_samples: points are formed inside the encoder kernel, the view direction is encoded
    once per ray (the reference expands it to every sample, nerf_static_transient_light.py:155-157)."""
    ops._need_cuda(center, ray, depth_samples)
    B, R, N = depth_samples.shape[:3]
    c, r, d = ops._f32(center.detach()), ops._f32(ray.detach()), ops._f32(depth_samples.detach())
    memo = {}

    def enc():
        if "enc" not in memo:
            memo["enc"] = ops.points_encode(c, r, d, cfg.L_3D)
        return memo["enc"]

    def view_seg():
        if "view" not in memo:
            memo["view"] = ops.view_encode(r.view(B * R, 3), cfg.L_view, normalize=True)
        return (memo["view"], N, cfg.view_cols)

    return dict(S=B * R * N, per_image=R * N, shape=(B, R, N), mode="rays", center=c, ray=r, depth=d, enc=enc,
                view_seg=view_seg)


def point_geometry(cfg: MLPConfig, points_3D, ray_unit):
    """Inputs of NeRF.forward: explicit points [B,R,N,3] and (already unit) view directions.  An expanded
    per-ray view tensor (stride 0 along N, as forward_samples of the reference builds it) is encoded per ray."""
    ops._need_cuda(points_3D, ray_unit)
    B, R, N, _ = points_3D.shape
    pts = ops._f32(points_3D.detach()).view(B * R * N, 3)
    memo = {}

    def enc():
        if "enc" not in memo:
            memo["enc"] = ops.positional_encode(pts, cfg.L_3D)
        return memo["enc"]

    def view_seg():
        if ray_unit is None:
            return None
        if "view" not in memo:
            ru = ray_unit.detach()
            if ru.dim() == 4 and ru.stride(2) == 0:
                memo["view"] = (ops.view_encode(ops._f32(ru[:, :, 0]).view(B * R, 3), cfg.L_view, False), N)
            elif ru.dim() == 3:
                memo["view"] = (ops.view_encode(ops._f32(ru).view(B * R, 3), cfg.L_view, False), N)
            else:
                memo["view"] = (ops.view_encode(ops._f32(ru).view(B * R * N, 3), cfg.L_view, False), 1)
        t, g = memo["view"]
        return (t, g, cfg.view_cols)

    return dict(S=B * R * N, per_image=R * N, shape=(B, R, N), mode="points", points=pts, enc=enc, view_seg=view_seg)
