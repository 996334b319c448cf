"""Training step of the plain model (layers/nerf.py:61-99: trunk + rgb head, everything trainable) on the tensor cores.

Forward: the single-pass bf16 launch of csrc/mlp_tc_split.cu with the stage list of the model's architecture; its drain keeps
every hidden activation as a bf16 tile image.  Backward: the staged dX chain (csrc/mlp_tc_chain.cu: rgb output layer -> rgb
hidden layer -> trunk feature -> trunk layers, with the raw-density gradient entering as a thin operand), the weight-gradient
GEMMs on the tile images (tp_tc_dw_gemm, eight 256 x 256 jobs in one launch) and the thin pieces (bias sums, the 63 encoding
columns of trunk layers 0 / skip, the view / xyz columns of the rgb head, the output rows) from the existing helpers.
Tolerance: the bf16 contract (<= 1e-2 on outputs and gradients).

split = True is the same step at the fp32-parity contract (<= 1e-4; opt.b200.mlp = 'fp32' with opt.b200.fp32_engine = 'tc'): the
split-fp16 forward (three passes) saves the activations as bf16 hi + lo image pairs (tp_tc32_forward_split_save), the dX chain
carries dz and the weights as bf16 hi + lo with three passes per K = 16 step (tp_tc_chain_backward_split), and every image helper
runs on the hi and lo images and adds the parts (mlp_tc_bwd, split flag).
"""
from __future__ import annotations

import torch

from . import _C, mlp_tc32, mlp_tc_bwd, ops
from .layers._mlp import MLPConfig

_F = 256


def supported(cfg, feat_p, rgb_p) -> bool:
    """256-wide trunk of 2..8 layers (skip not at the ends), rgb head = one hidden layer (<= 256 wide) + the output layer
    (options/nerf_lm_env.yaml:7: 286 -> 128 -> 3), view-dependent, L_3D = 10."""
    if cfg.stl or not cfg.view_dep or cfg.L_3D != 10 or not (0 <= cfg.L_view <= 4):
        return False
    nf, skip = len(feat_p), set(cfg.skip)
    if not (2 <= nf <= 8) or 0 in skip or nf - 1 in skip or len(rgb_p) != 2:
        return False
    for li, (w, _) in enumerate(feat_p):
        k = cfg.enc_cols if li == 0 else _F + (cfg.enc_cols if li in skip else 0)
        if tuple(w.shape) != ((_F + 1 if li == nf - 1 else _F), k):
            return False
    h = rgb_p[0][0].shape[0]
    return h <= _F and tuple(rgb_p[0][0].shape) == (h, _F + cfg.view_cols + 3) and tuple(rgb_p[1][0].shape) == (3, h)


_PADDED = {}      # persistent padded-head buffers, one set per head (keyed by its parameters' storage): stable addresses, no per-step zero fills
_DUMMY = {}       # the all-zero transient head the staged kernel's stage list carries for the plain model (never executed: static_only)


def _padded_head(rgb_p):
    """rgb hidden layer zero-padded to 256 rows, output layer to 256 columns (exact: the padded units are relu(0) = 0)."""
    (W0, b0), (W1, b1) = rgb_p
    dev = W0.device
    key = (str(dev), W0.data_ptr(), W1.data_ptr(), tuple(W0.shape), tuple(W1.shape))
    buf = _PADDED.get(key)
    if buf is None:
        if len(_PADDED) > 64:
            _PADDED.clear()
        buf = _PADDED[key] = (torch.zeros(_F, W0.shape[1], device=dev), torch.zeros(_F, device=dev), torch.zeros(3, _F, device=dev))
    W0p, b0p, W1p = buf
    W0p[:W0.shape[0]], b0p[:b0.shape[0]] = W0, b0
    W1p[:, :W1.shape[1]] = W1
    return [(W0p, b0p), (W1p, b1.contiguous())]


def _dummy_trans(dev):
    k = str(dev)
    if k not in _DUMMY:
        z = lambda *shape: torch.zeros(*shape, device=dev)
        _DUMMY[k] = ([(z(_F, _F), z(_F)), (z(5, _F), z(5))], z(1, 0))
    return _DUMMY[k]


def _stl_config(cfg, holder, n_feat):
    return MLPConfig(L_3D=cfg.L_3D, L_view=cfg.L_view, skip=cfg.skip, view_dep=True, n_feat=n_feat, n_rgb=2, n_trans=2,
                     n_latent_light=0, n_latent_trans=0, precision="bf16", save_for_backward=False, packed=holder, static_only=True)


class _Holder:
    """Cache slot for the packed images of one forward / backward pair (the padded tensors are rebuilt per call)."""


def forward_train(cfg, geom, feat_p, rgb_p, split=False):
    """-> rgb [S,3], density [S], ctx for `backward`."""
    dev = geom["depth"].device
    B, R, N = geom["shape"]
    rgb_pad = _padded_head(rgb_p)
    trans_dummy, none1 = _dummy_trans(dev)
    holder = _Holder()
    stl = _stl_config(cfg, holder, len(feat_p))
    none = none1.expand(B, 0)
    rgb2, den2, _, (images, n_save) = mlp_tc32.forward(stl, geom, none, none, feat_p, rgb_pad, trans_dummy, static_only=True,
                                                       precision=0 if split else 1, save=True)
    rgb, density = rgb2[:, :, 0].contiguous(), den2[:, 0].contiguous()
    ctx = dict(images=images, n_save=n_save, rgb=rgb, density=density, geom=geom, rgb_pad=rgb_pad, cfg=cfg, split=split)
    return rgb, density, ctx


def _bwd_chunks(cfg, feat_p, rgb_pad, split=False):
    """Transposed weight chunks of the chain, in stage order; returns (desc rows, chain stage rows).  split: the chunks of
    tp_tc_pack_weights_split, one K = 16 step (hi | lo) each, sixteen per layer."""
    nf = len(feat_p)
    rows, stages = [], []
    k = 16 if split else 32             # K rows of W per chunk
    per_layer = _F // k

    def thin_chunk(W, n_rows):          # K = 16 step: chunk element (n, kl) = W[kl][n], kl < n_rows
        rows.append([W.data_ptr(), W.stride(0), 0, _F, 0, n_rows, 256, 0, -1, 1])
        return len(rows) - 1

    def big(W, row0=0):                 # K = 32 (16) chunks: element (n, kl) = W[row0 + k c + kl][n], n < 256
        c0 = len(rows)
        for c in range(0, _F, k):
            rows.append([W.data_ptr(), W.stride(0), 0, _F, row0 + c, k, 256, 0, -1, 1])
        return c0

    slot_h = lambda li: li              # saved slot of trunk activation h_li (output of trunk layer li), li < nf - 1
    slot_feat, slot_rgb_h = nf - 1, nf
    W_out, W_r0 = rgb_pad[1][0], rgb_pad[0][0]
    # stage 0: dz_rgb (thin 0) x W_out -> masked by the rgb hidden activation -> dz slot 0
    stages.append([0, thin_chunk(W_out, 3), 0, 0, slot_rgb_h, 0])
    # stage 1: x W_r0[:, :256] -> masked by the trunk feature -> dz slot 1 (gradient of the feature rows of the last trunk layer)
    stages.append([-1, 0, big(W_r0), per_layer, slot_feat, 1])
    # stage 2: x W_last[1:] + dz_sigma (thin 1) x W_last[0] -> masked by h_{nf-2} -> dz slot 2; then down the trunk
    W_last = feat_p[nf - 1][0]
    tc = thin_chunk(W_last, 1)
    stages.append([1, tc, big(W_last, row0=1), per_layer, slot_h(nf - 2), 2])
    for li in range(nf - 2, 0, -1):     # layer li maps h_{li-1} -> h_li: dz_{li-1} = (dz_li W_li[:, :256]) * [h_{li-1} > 0]
        stages.append([-1, 0, big(feat_p[li][0]), per_layer, slot_h(li - 1), 2 + (nf - 1 - li)])
    return rows, stages


def backward(ctx, g_rgb, g_density, feat_p, rgb_p):
    """-> ([(dW, db)] per trunk layer, [(dW, db)] per rgb layer)."""
    cfg, geom, images, n_save = ctx["cfg"], ctx["geom"], ctx["images"], ctx["n_save"]
    rgb_pad, split = ctx["rgb_pad"], ctx["split"]
    B, R, N = geom["shape"]
    S = geom["S"]
    dev = images.device
    nf = len(feat_p)
    lib = _C.load()
    parts = 2 if split else 1           # tile images per slot (split: hi, lo)
    dz_rgb, dz_sigma = torch.empty(S, 3, device=dev), torch.empty(S, 1, device=dev)
    _C.call("tp_plain_output_grad", ops._p(ctx["rgb"]), ops._p(ctx["density"]), ops._p(ops._f32(g_rgb).reshape(S, 3)),
            ops._p(ops._f32(g_density).reshape(S)), S, ops._p(dz_rgb), ops._p(dz_sigma), ops._stream())
    rows, stages = _bwd_chunks(cfg, feat_p, rgb_pad, split)
    desc = ops.device_table(rows, torch.int64, dev)
    packed = torch.empty(len(rows) * lib.tp_tc_chunk_bytes(), dtype=torch.uint8, device=dev)
    _C.call("tp_tc_pack_weights_split" if split else "tp_tc_pack_weights", ops._p(desc), len(rows), ops._p(packed), ops._stream())
    n_dz = len(stages)
    n_tiles = (S + 127) // 128
    dz = torch.empty(n_tiles * parts * n_dz * 65536, dtype=torch.uint8, device=dev)
    st = torch.tensor(stages, dtype=torch.int32)
    bits = images[n_tiles * parts * n_save * 65536:]          # the ReLU bitmasks the forward wrote behind the tile images
    _C.call("tp_tc_chain_backward_split" if split else "tp_tc_chain_backward", ops._p(dz_rgb), 3, ops._p(dz_sigma), 1, S,
            ops._p(packed), len(rows), ops._p(st), n_dz, ops._p(bits), n_save, ops._p(dz), n_dz, ops._stream())
    # ---- 256 x 256 weight gradients: (dz slot, saved activation slot) per layer; the layers that read the encoding (layer 0, skip
    # layers) add a job against the saved encoding tile, whose column 63 is a constant 1: dz^T of it = [dW encoding columns | db]
    slot_feat, slot_rgb_h, slot_enc = nf - 1, nf, n_save - 1
    dz_slot = lambda li: 2 + (nf - 2 - li) if li < nf - 1 else 1      # dz of trunk layer li's pre-activation (the last layer: its feature rows)
    enc_layers = [0] + sorted(set(cfg.skip))
    pairs = [(0, slot_feat), (1, nf - 2)] + [(dz_slot(li), li - 1) for li in range(nf - 2, 0, -1)] + [(dz_slot(li), slot_enc) for li in enc_layers]
    if split:
        big = mlp_tc_bwd.dw_gemm(dz, n_dz, images, n_save, pairs, S, split=True)
    else:
        big = torch.cat([mlp_tc_bwd.dw_gemm(dz, n_dz, images, n_save, pairs[i:i + 12], S) for i in range(0, len(pairs), 12)], dim=0)      # one launch for <= 12 jobs
    enc_grad = {li: big[nf + j] for j, li in enumerate(enc_layers)}       # [256, 256]: columns 0..62 encoding, 63 bias sum
    # ---- column sums of the dz images whose bias gradient does not come out of an encoding job
    want = [0, 1] + [dz_slot(li) for li in range(nf - 2, 0, -1) if li not in enc_grad]
    sums = mlp_tc_bwd.images_colsum(dz, n_dz, S, want, split=split)
    colsum = lambda slot: sums[want.index(slot)]
    # ---- thin pieces
    h = rgb_p[0][0].shape[0]
    dW_out = mlp_tc_bwd.thin_dw(dz_rgb, images, slot_rgb_h, n_save, S, split=split)[:, :h].contiguous()
    db_out = mlp_tc_bwd.thin_colsum(dz_rgb, S)
    ray_sums0 = mlp_tc_bwd.image_ray_sums(dz, 0, n_dz, S, N, split=split)                    # [B*R,256] of the rgb hidden dz
    view_t, _, vc = geom["view_seg"]()
    dW_view, _ = ops.linear_backward_weight(ray_sums0, [(view_t, 1, vc)], B * R, want_bias=False)          # [256, vc]
    xyz = ops.points_from_depth(geom["center"], geom["ray"], geom["depth"]).view(S, 3)
    dW_xyz = mlp_tc_bwd.thin_dw(xyz, dz, 0, n_dz, S, split=split).t()                                     # [256, 3]
    dW_r0 = torch.cat([big[0], dW_view, dW_xyz], dim=1)[:h].contiguous()
    db_r0 = colsum(0)[:h].contiguous()
    g_rgb_layers = [(dW_r0, db_r0), (dW_out, db_out)]
    # ---- trunk
    ec = cfg.enc_cols
    g_feat = [None] * nf
    dW_sigma = mlp_tc_bwd.thin_dw(dz_sigma, images, nf - 2, n_save, S, split=split)            # [1,256]: row 0 of the last layer
    g_feat[nf - 1] = (torch.cat([dW_sigma, big[1]], dim=0), torch.cat([mlp_tc_bwd.thin_colsum(dz_sigma, S), colsum(1)]))
    for j, li in enumerate(range(nf - 2, 0, -1)):
        if li in enc_grad:
            g_feat[li] = (torch.cat([big[2 + j], enc_grad[li][:, :ec]], dim=1), enc_grad[li][:, 63].contiguous())
        else:
            g_feat[li] = (big[2 + j], colsum(dz_slot(li)))
    g_feat[0] = (enc_grad[0][:, :ec].contiguous(), enc_grad[0][:, 63].contiguous())
    return g_feat, g_rgb_layers


class PlainTC(torch.autograd.Function):
    """(geom, split, *trunk and head parameters) -> (rgb [B,R,N,3], density [B,R,N]) with the tensor-core backward; split = the
    fp32-parity step (<= 1e-4), else bf16 (<= 1e-2)."""

    @staticmethod
    def forward(ctx, cfg, geom, n_feat, split, *params):
        pairs = [(params[i].detach().float().contiguous(), params[i + 1].detach().float().contiguous()) for i in range(0, len(params), 2)]
        feat_p, rgb_p = pairs[:n_feat], pairs[n_feat:]
        rgb, density, saved = forward_train(cfg, geom, feat_p, rgb_p, split)
        ctx.saved, ctx.layers = saved, (feat_p, rgb_p)
        B, R, N = geom["shape"]
        return rgb.view(B, R, N, 3), density.view(B, R, N)

    @staticmethod
    def backward(ctx, g_rgb, g_density):
        feat_p, rgb_p = ctx.layers
        S = ctx.saved["geom"]["S"]
        dev = ctx.saved["images"].device
        g_rgb = g_rgb if g_rgb is not None else torch.zeros(S, 3, device=dev)
        g_density = g_density if g_density is not None else torch.zeros(S, device=dev)
        g_feat, g_rgb_layers = backward(ctx.saved, g_rgb.contiguous(), g_density.contiguous(), feat_p, rgb_p)
        ctx.saved = None
        out = []
        for dW, db in g_feat + g_rgb_layers:
            out += [dW, db]
        need = ctx.needs_input_grad[4:]
        return (None, None, None, None, *[o if need[i] else None for i, o in enumerate(out)])
