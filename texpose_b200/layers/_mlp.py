"""Layer orchestration of the NeRF MLPs over the C-ABI kernels (forward + hand-written backward).

Mirrors the arithmetic of NeRF.forward in layers/nerf_static_transient_light.py:76-145 (static/transient/light
model, trunk under no_grad) and layers/nerf.py:61-99 (plain model, trunk trainable).  torch.cat / expand of the
reference are never materialised: each layer reads a *segmented* input (see tp_linear_forward).

Two arithmetic modes:
  fp32  -- the <=1e-4 parity mode: SIMT FFMA kernels (mlp_simt.cu), forward and backward; calls that record no gradient
           (rendering) run on the tensor cores with split-fp16 operands instead (mlp_tc_split.cu, three MMA passes per K
           step), for any 256-wide static/transient/light architecture (opt.b200.fp32_engine = 'simt' keeps them on SIMT);
           with opt.b200.fp32_engine = 'tc' a gradient-recording ray-mode call trains the heads on the tensor cores too (split
           forward with bf16 hi / lo activation save, split dX chain, dW GEMMs on the hi / lo images: mlp_tc_bwd, split flag);
  bf16  -- fused tcgen05/TMEM forward (mlp_tc.cu) for the static/transient/light model; in training it also saves
           the head activations (bf16 tile images) that the backward consumes.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import torch

from .. import ops

Tensor = torch.Tensor


@dataclass
class MLPConfig:
    L_3D: int
    L_view: int
    skip: Tuple[int, ...]
    view_dep: bool
    n_feat: int                 # number of trunk layers
    n_rgb: int
    n_trans: int                # 0 for the plain model
    n_latent_light: int = 0
    n_latent_trans: int = 0
    precision: str = "fp32"     # "fp32" | "bf16" | "auto" (bf16 when the fused kernel implements the architecture)
    save_for_backward: bool = True
    packed: object = None       # bf16 weight image for the tcgen05 kernel (mlp_tc.pack), or None
    static_only: bool = False   # rendering only: skip the transient head (its outputs come back as zeros), fused kernel only
    fp32_tc: bool = True        # fp32 mode, no gradient wanted: split-bf16 tensor-core kernel (mlp_tc32) instead of SIMT FFMA
    fp32_train_tc: bool = False  # fp32 mode, gradient wanted: split staged kernels instead of SIMT (opt.b200.fp32_engine = 'tc')

    @property
    def stl(self) -> bool:
        return self.n_trans > 0

    @property
    def enc_cols(self) -> int:
        return 3 + 6 * self.L_3D

    @property
    def view_cols(self) -> int:
        return 3 + 6 * self.L_view


def _pairs(params: Sequence[Tensor]) -> List[Tuple[Tensor, Tensor]]:
    return [(params[i], params[i + 1]) for i in range(0, len(params), 2)]


def _c(t: Tensor) -> Tensor:
    return t.detach().contiguous().float()


class _Saved:
    """Activations kept between forward and backward (plain attribute bag; tensors live on the GPU)."""


def mlp_forward_fp32(cfg: MLPConfig, enc: Tensor, view_seg, lat_trans: Optional[Tensor], lat_light: Optional[Tensor],
                     S: int, per_image: int, feat_p, rgb_p, trans_p, sv: Optional[_Saved]):
    dev = enc.device
    ec = cfg.enc_cols
    if cfg.stl:
        rgb = torch.empty(S, 3, 2, device=dev)
        density = torch.empty(S, 2, device=dev)
        uncert = torch.empty(S, device=dev)
    else:
        rgb = torch.empty(S, 3, device=dev)
        density = torch.empty(S, device=dev)
        uncert = None
    # ---- trunk: 8 x (Linear + ReLU), skip concat, row 0 of the last layer = raw density
    h = None
    trunk_in = []
    for li, (W, b) in enumerate(feat_p):
        segs = [(enc, 1, ec)] if li == 0 else [(h, 1, h.shape[1])]
        if li in cfg.skip:
            segs = segs + [(enc, 1, ec)]
        trunk_in.append(segs)
        if li == len(feat_p) - 1:
            Y = torch.empty(S, W.shape[0] - 1, device=dev)
            ops.linear_forward(segs, W, b, S, ops.ACT_TRUNK_LAST_STL if cfg.stl else ops.ACT_TRUNK_LAST_PLAIN, Y,
                               Y.stride(0), aux0=density)
        else:
            Y = torch.empty(S, W.shape[0], device=dev)
            ops.linear_forward(segs, W, b, S, ops.ACT_RELU, Y, Y.stride(0))
        h = Y
    feat = h
    F = feat.shape[1]
    # ---- rgb head: cat([feat, ray_enc, points_3D, latent_light])
    segs = [(feat, 1, F)]
    if cfg.view_dep:
        segs.append(view_seg)
    segs.append((enc, 1, 3))
    if cfg.stl and cfg.n_latent_light:
        segs.append((lat_light, per_image, cfg.n_latent_light))
    rgb_in = []
    h = None
    for li, (W, b) in enumerate(rgb_p):
        cur = segs if li == 0 else [(h, 1, h.shape[1])]
        rgb_in.append(cur)
        if li == len(rgb_p) - 1:
            if cfg.stl:
                ops.linear_forward(cur, W, b, S, ops.ACT_RGB_STATIC, rgb, 6)
            else:
                ops.linear_forward(cur, W, b, S, ops.ACT_SIGMOID, rgb, 3)
        else:
            Y = torch.empty(S, W.shape[0], device=dev)
            ops.linear_forward(cur, W, b, S, ops.ACT_RELU, Y, Y.stride(0))
            h = Y
    # ---- transient head: cat([feat, latent_trans]) -> rgb_t (sigmoid), sigma_t, uncert (softplus)
    trans_in = []
    if cfg.stl:
        segs = [(feat, 1, F)]
        if cfg.n_latent_trans:
            segs.append((lat_trans, per_image, cfg.n_latent_trans))
        h = None
        for li, (W, b) in enumerate(trans_p):
            cur = segs if li == 0 else [(h, 1, h.shape[1])]
            trans_in.append(cur)
            if li == len(trans_p) - 1:
                ops.linear_forward(cur, W, b, S, ops.ACT_TRANS_OUT, rgb, 6, aux0=density, aux1=uncert)
            else:
                Y = torch.empty(S, W.shape[0], device=dev)
                ops.linear_forward(cur, W, b, S, ops.ACT_RELU, Y, Y.stride(0))
                h = Y
    if sv is not None:
        sv.trunk_in, sv.rgb_in, sv.trans_in, sv.feat = trunk_in, rgb_in, trans_in, feat
        sv.rgb, sv.density, sv.uncert = rgb, density, uncert
    return rgb, density, uncert


def _head_backward(dZ: Tensor, layers, inputs, S: int, need: Sequence[bool]):
    """Walks one head from its output layer down to layer 0.  Returns per-layer (dW, db) and dZ of layer 0."""
    grads = [None] * len(layers)
    for li in range(len(layers) - 1, -1, -1):
        W, _ = layers[li]
        if need[li]:
            grads[li] = ops.linear_backward_weight(dZ, inputs[li], S)
        if li > 0:
            h = inputs[li][0][0]            # this layer's input = relu output of layer li-1
            dZ = ops.linear_backward_input(dZ, W, S, h.shape[1], h)
    return grads, dZ


def mlp_backward(cfg: MLPConfig, sv: _Saved, S: int, per_image: int, feat_p, rgb_p, trans_p, g_rgb, g_density, g_uncert,
                 need_feat: Sequence[bool], need_rgb: Sequence[bool], need_trans: Sequence[bool],
                 need_lat_trans: bool, need_lat_light: bool):
    dev = sv.feat.device
    F = sv.feat.shape[1]
    trunk_trainable = any(need_feat)
    dz_rgb = torch.empty(S, 3, device=dev)
    dz_sigma = torch.empty(S, device=dev) if trunk_trainable else None
    if cfg.stl:
        dz_trans = torch.empty(S, 5, device=dev)
        ops._C.call("tp_stl_output_grad", ops._p(sv.rgb), ops._p(sv.density), ops._p(sv.uncert), ops._p(g_rgb),
                    ops._p(g_density), ops._p(g_uncert), S, ops._p(dz_rgb), ops._p(dz_trans), ops._p(dz_sigma),
                    ops._stream())
    else:
        dz_trans = None
        if dz_sigma is None:
            dz_sigma = torch.empty(S, device=dev)
        ops._C.call("tp_plain_output_grad", ops._p(sv.rgb), ops._p(sv.density), ops._p(g_rgb), ops._p(g_density), S,
                    ops._p(dz_rgb), ops._p(dz_sigma), ops._stream())

    g_rgb_layers, dz0_rgb = _head_backward(dz_rgb, rgb_p, sv.rgb_in, S, need_rgb)
    d_feat = None
    if trunk_trainable:
        d_feat = ops.linear_backward_input(dz0_rgb, rgb_p[0][0], S, F, None)
    d_lat_light = None
    if cfg.stl and need_lat_light and cfg.n_latent_light:
        off = sum(int(s[2]) for s in sv.rgb_in[0][:-1])
        col = ops.group_colsum(dz0_rgb, S, per_image)
        d_lat_light = ops.linear_backward_input(col, rgb_p[0][0], col.shape[0], cfg.n_latent_light, None, w_col0=off)

    g_trans_layers, d_lat_trans = [], None
    if cfg.stl:
        g_trans_layers, dz0_trans = _head_backward(dz_trans, trans_p, sv.trans_in, S, need_trans)
        if trunk_trainable:
            d_feat = d_feat + ops.linear_backward_input(dz0_trans, trans_p[0][0], S, F, None)
        if need_lat_trans and cfg.n_latent_trans:
            col = ops.group_colsum(dz0_trans, S, per_image)
            d_lat_trans = ops.linear_backward_input(col, trans_p[0][0], col.shape[0], cfg.n_latent_trans, None,
                                                    w_col0=F)

    g_feat_layers = [None] * len(feat_p)
    if trunk_trainable:
        dZ = torch.empty(S, F + 1, device=dev)
        ops._C.call("tp_trunk_last_grad", ops._p(dz_sigma), ops._p(d_feat), d_feat.stride(0), ops._p(sv.feat),
                    sv.feat.stride(0), S, F, ops._p(dZ), dZ.stride(0), ops._stream())
        for li in range(len(feat_p) - 1, -1, -1):
            W, _ = feat_p[li]
            if need_feat[li]:
                g_feat_layers[li] = ops.linear_backward_weight(dZ, sv.trunk_in[li], S)
            if li > 0:
                h = sv.trunk_in[li][0][0]
                dZ = ops.linear_backward_input(dZ, W, S, h.shape[1], h)
    return g_feat_layers, g_rgb_layers, g_trans_layers, d_lat_trans, d_lat_light


def run_mlp(cfg: MLPConfig, geom, lat_trans, lat_light, *params):
    """NerfMLP.apply, except that an empty sample set (an eval frame whose mask prior selects no pixel, an empty shard)
    returns empty outputs of the reference's shapes without a launch -- as the reference's torch ops do."""
    if geom["S"] == 0:
        shape, dev = geom["shape"], params[0].device
        if cfg.stl:
            return (torch.empty(*shape, 3, 2, device=dev), torch.empty(*shape, 2, device=dev),
                    torch.empty(*shape, 1, device=dev))
        return torch.empty(*shape, 3, device=dev), torch.empty(*shape, device=dev)
    return NerfMLP.apply(cfg, geom, lat_trans, lat_light, *params)


class NerfMLP(torch.autograd.Function):
    """(enc inputs, latents, *weights) -> (rgb, density[, uncert]) per sample, with the fused backward."""

    @staticmethod
    def forward(ctx, cfg: MLPConfig, geom, lat_trans, lat_light, *params):
        n_f, n_r, n_t = 2 * cfg.n_feat, 2 * cfg.n_rgb, 2 * cfg.n_trans
        feat_p = _pairs([_c(p) for p in params[:n_f]])
        rgb_p = _pairs([_c(p) for p in params[n_f:n_f + n_r]])
        trans_p = _pairs([_c(p) for p in params[n_f + n_r:n_f + n_r + n_t]])
        S, per_image = geom["S"], geom["per_image"]
        lt = _c(lat_trans) if lat_trans is not None else None
        ll = _c(lat_light) if lat_light is not None else None
        needs_grad = any(ctx.needs_input_grad)
        sv = _Saved() if (needs_grad and cfg.save_for_backward) else None
        trunk_grad = any(ctx.needs_input_grad[4:4 + n_f])      # frozen in the reference (:34); fp32 path if unfrozen
        use_tc = cfg.precision == "bf16" and cfg.stl and not trunk_grad
        if cfg.precision == "auto" and cfg.stl and not trunk_grad and geom.get("mode") == "rays":
            from .. import mlp_tc
            use_tc = mlp_tc.supported(cfg, feat_p, rgb_p, trans_p)
        use_tc32, single = False, 0
        if sv is None and cfg.stl and geom.get("mode") == "rays":
            from .. import mlp_tc, mlp_tc32
            if cfg.precision == "fp32" or (cfg.precision == "auto" and not use_tc):
                # the <= 1e-4 mode (and 'auto' on an architecture the bf16 kernels below do not cover) without gradients
                use_tc32 = cfg.fp32_tc and mlp_tc32.supported(cfg, feat_p, rgb_p, trans_p)
            if cfg.precision in ("bf16", "auto") and not mlp_tc.supported(cfg, feat_p, rgb_p, trans_p) \
                    and mlp_tc32.supported(cfg, feat_p, rgb_p, trans_p):
                # bf16 on an architecture the lock-step kernel is not specialised for: single-pass launch of the staged kernel
                use_tc32, single, use_tc = True, 1, False
        staged_train = split_train = False
        if sv is not None and cfg.stl and not trunk_grad and cfg.precision in ("bf16", "auto") and geom.get("mode") == "rays":
            from .. import mlp_tc, mlp_tc32, mlp_tc_bwd
            # training on the staged kernels: an architecture the lock-step kernel / fused backward are not specialised for, or
            # images so small that one CTA's tile range of the fused backward would touch more than four of them
            lockstep = mlp_tc.supported(cfg, feat_p, rgb_p, trans_p) and mlp_tc_bwd.fused_supported(S, per_image)
            staged_train = not lockstep and mlp_tc32.supported(cfg, feat_p, rgb_p, trans_p) \
                and (len(rgb_p) - 1) + (len(trans_p) - 1) + 1 <= 16
        if sv is not None and cfg.stl and not trunk_grad and cfg.precision == "fp32" and cfg.fp32_train_tc \
                and geom.get("mode") == "rays":
            from .. import mlp_tc32
            # the <= 1e-4 training step on the tensor cores: the staged kernels in their split form
            staged_train = split_train = mlp_tc32.supported(cfg, feat_p, rgb_p, trans_p) \
                and (len(rgb_p) - 1) + (len(trans_p) - 1) + 1 <= 16
        if staged_train:
            from .. import mlp_tc32
            rgb, density, uncert, (images, n_save) = mlp_tc32.forward(cfg, geom, lt, ll, feat_p, rgb_p, trans_p,
                                                                      precision=0 if split_train else 1, save="heads")
            sv.images, sv.n_save, sv.staged, sv.geom, sv.lat = images, n_save, True, geom, (lt, ll)
            sv.split = split_train
            sv.rgb, sv.density, sv.uncert = rgb, density, uncert
        elif use_tc32:
            from .. import mlp_tc32
            rgb, density, uncert = mlp_tc32.forward(cfg, geom, lt, ll, feat_p, rgb_p, trans_p, static_only=cfg.static_only,
                                                    precision=single)
        elif use_tc:
            from .. import mlp_tc
            if sv is None:
                rgb, density, uncert = mlp_tc.forward(cfg, geom, lt, ll, feat_p, rgb_p, trans_p,
                                                      static_only=cfg.static_only)      # sv is None: no backward will run
            else:
                # training: the kernel also stores the head activations it computed (bf16 tile images); the backward
                # consumes exactly those -- nothing is re-materialised
                rgb, density, uncert, images = mlp_tc.forward(cfg, geom, lt, ll, feat_p, rgb_p, trans_p, save=True)
                sv.images, sv.geom, sv.lat = images, geom, (lt, ll)
                sv.rgb, sv.density, sv.uncert = rgb, density, uncert
        else:
            rgb, density, uncert = mlp_forward_fp32(cfg, geom["enc"](), geom["view_seg"](), lt, ll, S, per_image,
                                                    feat_p, rgb_p, trans_p, sv)
        ctx.cfg, ctx.sv, ctx.S, ctx.per_image = cfg, sv, S, per_image
        ctx.layers = (feat_p, rgb_p, trans_p)
        shape = geom["shape"]       # (B, R, N)
        if cfg.stl:
            return rgb.view(*shape, 3, 2), density.view(*shape, 2), uncert.view(*shape, 1)
        return rgb.view(*shape, 3), density.view(*shape)

    @staticmethod
    def backward(ctx, g_rgb, g_density, g_uncert=None):
        cfg, sv, S = ctx.cfg, ctx.sv, ctx.S
        if sv is None:
            raise RuntimeError("NerfMLP.backward: activations were not saved (cfg.save_for_backward False)")
        feat_p, rgb_p, trans_p = ctx.layers
        n_f, n_r, n_t = 2 * cfg.n_feat, 2 * cfg.n_rgb, 2 * cfg.n_trans
        need = ctx.needs_input_grad[4:]
        g = lambda t: t.contiguous().float() if t is not None else None
        if getattr(sv, "images", None) is not None:
            # tensor-core training: the backward of whichever kernels the forward chose -- the fused backward on the tile images the
            # lock-step forward saved (csrc/mlp_tc_bwd.cu), or the staged kernels (csrc/mlp_tc_chain.cu; split = the fp32 step)
            from .. import mlp_tc_bwd
            if getattr(sv, "staged", False):
                gr, gt, d_lt, d_ll = mlp_tc_bwd.heads_backward_staged(
                    cfg, sv, S, ctx.per_image, rgb_p, trans_p, g(g_rgb), g(g_density), g(g_uncert),
                    bool(ctx.needs_input_grad[2]), bool(ctx.needs_input_grad[3]), split=sv.split)
            else:
                gr, gt, d_lt, d_ll = mlp_tc_bwd.heads_backward(cfg, sv, S, ctx.per_image, rgb_p, trans_p, g(g_rgb), g(g_density),
                                                               g(g_uncert), bool(ctx.needs_input_grad[2]), bool(ctx.needs_input_grad[3]))
            out = [None] * n_f
            for layers in (gr, gt):
                for pair in layers:
                    out += [pair[0], pair[1]]
            out = [o if need[i] else None for i, o in enumerate(out)]
            ctx.sv = None
            return (None, None, d_lt, d_ll, *out)

        def layer_need(off, n):
            return [bool(need[off + 2 * i] or need[off + 2 * i + 1]) for i in range(n)]

        gf, gr, gt, d_lt, d_ll = mlp_backward(
            cfg, sv, S, ctx.per_image, feat_p, rgb_p, trans_p, g(g_rgb), g(g_density), g(g_uncert),
            layer_need(0, cfg.n_feat), layer_need(n_f, cfg.n_rgb), layer_need(n_f + n_r, cfg.n_trans),
            bool(ctx.needs_input_grad[2]), bool(ctx.needs_input_grad[3]))
        out = []
        for layers in (gf, gr, gt):
            for pair in layers:
                out += [pair[0], pair[1]] if pair is not None else [None, None]
        out = [o if need[i] else None for i, o in enumerate(out)]
        ctx.sv = None
        return (None, None, d_lt, d_ll, *out)
