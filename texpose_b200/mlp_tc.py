"""Host side of the fused tcgen05 forward (csrc/mlp_tc.cu): weight packing, bias folding, launch.

The packed bf16 weight image is an opaque caller-owned blob cached on the NeRF module and rebuilt when any
parameter's `_version` changes (SURVEY.md 8b: "re-packed when param._version changes").
"""
from __future__ import annotations

import torch

from . import _C, ops

_F = 256
STATIC_ONLY = 1 << 17   # flags bit 17: stop after the rgb head (rendering that uses only the static outputs)
FUSED_N = (32, 64, 128)  # samples per ray the fused render launch takes (a 128-row tile holds whole rays)


def supported(cfg, feat_p, rgb_p, trans_p) -> bool:
    """The fused kernel is specialised for the architecture of options/nerf_lm_adapt_gan.yaml:9-18."""
    if not (cfg.stl and cfg.view_dep and cfg.L_3D == 10 and 0 <= cfg.L_view <= 4 and tuple(cfg.skip) == (4,)):
        return False
    if len(feat_p) != 8 or len(rgb_p) != 4 or len(trans_p) != 4:
        return False
    want_f = [(256, 63)] + [(256, 256)] * 3 + [(256, 319)] + [(256, 256)] * 2 + [(257, 256)]
    if [tuple(w.shape) for w, _ in feat_p] != want_f:
        return False
    k_rgb0 = 256 + cfg.view_cols + 3 + cfg.n_latent_light
    if [tuple(w.shape) for w, _ in rgb_p] != [(256, k_rgb0), (256, 256), (256, 256), (3, 256)]:
        return False
    if [tuple(w.shape) for w, _ in trans_p] != [(256, 256 + cfg.n_latent_trans), (256, 256), (256, 256), (5, 256)]:
        return False
    return True


def _chunk_table(cfg, feat_p, rgb_p, trans_p):
    """Rows {W ptr, ld, row0, rows_valid, col0, cols_valid, n_layout, bias ptr, bias k, 0} in the exact order the kernel
    consumes.  Static biases travel inside the weight image: they multiply the constant-1 column (63) of the encoding
    tile, either in the stage's own last E chunk (trunk 0, 4) or in a dedicated K=16 bias chunk (E columns 48..63)."""
    rows = []

    def big(W, col0, ncols, row0=0, bias=None):      # N=256 x K=32 chunks over source columns [col0, col0+ncols)
        n = len(range(0, ncols, 32))
        for i, c in enumerate(range(0, ncols, 32)):
            last = bias is not None and i == n - 1
            rows.append([W.data_ptr(), W.stride(0), row0, 256, col0 + c, min(32, ncols - c), 256,
                         bias.data_ptr() if last else 0, 31 if last else -1, 0])

    def bias_chunk(b):                                 # N=256 x K=16 chunk on E columns 48..63: only column 63 set
        rows.append([0, 0, 0, 256, 0, 0, 256, b.data_ptr(), 15, 0])

    def small(W, nrows, row0=0):                       # N=16 x K=256 chunk
        rows.append([W.data_ptr(), W.stride(0), row0, nrows, 0, 256, 16, 0, -1, 0])

    f = [w for w, _ in feat_p]
    fb = [b for _, b in feat_p]
    r = [w for w, _ in rgb_p]
    rb = [b for _, b in rgb_p]
    t = [w for w, _ in trans_p]
    tb = [b for _, b in trans_p]
    keep = []
    big(f[0], 0, 63, bias=fb[0])
    for li in (1, 2, 3):
        big(f[li], 0, 256)
        bias_chunk(fb[li])
    big(f[4], 0, 256)
    big(f[4], 256, 63, bias=fb[4])
    for li in (5, 6):
        big(f[li], 0, 256)
        bias_chunk(fb[li])
    small(f[7], 1, row0=0)                 # density row
    big(f[7], 0, 256, row0=1)              # feature rows 1..256
    b7 = fb[7][1:].contiguous()
    keep.append(b7)
    bias_chunk(b7)
    big(r[0], 0, 256)
    big(r[0], 256 + cfg.view_cols, 3)      # raw xyz columns ride on the first K-chunk of the encoding tile
    for li in (1, 2):
        big(r[li], 0, 256)
        bias_chunk(rb[li])
    small(r[3], 3)
    big(t[0], 0, 256)
    for li in (1, 2):
        big(t[li], 0, 256)
        bias_chunk(tb[li])
    small(t[3], 5)
    return rows, keep


_PAD7 = {}


class Packed:
    __slots__ = ("key", "weights", "wview", "biasbuf", "keep", "where")


def _version_key(params):
    return tuple((p.data_ptr(), p._version) for p in params)


def pack(cfg, holder, feat_p, rgb_p, trans_p, params_for_key) -> Packed:
    key = _version_key(params_for_key)
    cached = getattr(holder, "_packed", None)
    if cached is not None and cached.key == key:
        return cached
    lib = _C.load()
    n_chunks, chunk_bytes = lib.tp_tc_num_chunks(), lib.tp_tc_chunk_bytes()
    dev = feat_p[0][0].device
    # the descriptor table holds addresses and strides only: while the parameters stay where they are (an optimizer updates them in
    # place) the table of the previous step is re-used as it is, and only the pack kernel runs again
    where = tuple((w.data_ptr(), w.stride(0), b.data_ptr()) for w, b in feat_p + rgb_p + trans_p)
    if cached is not None and getattr(cached, "where", None) == where:
        desc, keep = cached.keep
    else:
        table, keep = _chunk_table(cfg, feat_p, rgb_p, trans_p)
        assert len(table) == n_chunks, (len(table), n_chunks)
        desc = ops.device_table(table, torch.int64, dev)
    weights = torch.empty(n_chunks * chunk_bytes, dtype=torch.uint8, device=dev)
    _C.call("tp_tc_pack_weights", ops._p(desc), n_chunks, ops._p(weights), ops._stream())
    fb = [b for _, b in feat_p]
    rb = [b for _, b in rgb_p]
    tb = [b for _, b in trans_p]
    pad = _PAD7.get(dev)
    if pad is None:
        pad = _PAD7[dev] = torch.zeros(7, device=dev)
    biasbuf = torch.cat([fb[7][:1].float(), rb[3].float(), tb[3].float(), pad])      # fp32 biases of the three N=16 output stages (one launch)
    out = Packed()
    out.key, out.weights, out.biasbuf = key, weights, biasbuf
    # view-direction columns of mlp_rgb[0] ([unit dir, posenc]: layers/nerf_static_transient_light.py:111-117), transposed to
    # [3+6L, 256] so a warp of the render launch reads one input's 256 weights as two coalesced 512 B rows (a copy, no arithmetic)
    out.wview = rgb_p[0][0][:, 256:256 + cfg.view_cols].t().contiguous()
    out.keep = (desc, keep)
    out.where = where
    if holder is not None:
        holder._packed = out
    return out


_scratch = {}


def _scratch_for(dev):
    k = (dev.type, dev.index)
    if k not in _scratch:
        n = _C.load().tp_tc_scratch_bytes()
        _scratch[k] = torch.empty(n, dtype=torch.uint8, device=dev)
    return _scratch[k]


def image_biases(cfg, B, lat_trans, lat_light, rgb_p, trans_p):
    """Per-image constants folded into the layer-0 biases of the two heads (latents x their weight columns + bias): [B,256] each."""
    dev = rgb_p[0][0].device
    W_r0, b_r0 = rgb_p[0]
    W_t0, b_t0 = trans_p[0]
    if lat_trans.shape[0] != B or lat_light.shape[0] != B:
        raise ValueError(f"latents must have one row per image ({B}); got {tuple(lat_trans.shape)} / {tuple(lat_light.shape)}")
    img = torch.empty(2, B, _F, device=dev)
    _C.call("tp_tc_image_biases", ops._p(W_r0), W_r0.stride(0), 256 + cfg.view_cols + 3, cfg.n_latent_light, ops._p(b_r0),
            ops._p(lat_light), ops._p(W_t0), W_t0.stride(0), 256, cfg.n_latent_trans, ops._p(b_t0), ops._p(lat_trans), B,
            ops._p(img[0]), ops._p(img[1]), ops._stream())
    img_r, img_t = img[0], img[1]
    return img_r, img_t


def forward(cfg, geom, lat_trans, lat_light, feat_p, rgb_p, trans_p, save=False, static_only=False):
    flags = STATIC_ONLY if static_only and not save else 0
    if geom.get("mode") != "rays":
        raise NotImplementedError("the fused bf16 kernel is ray-parameterised (forward_samples)")
    if not supported(cfg, feat_p, rgb_p, trans_p):
        raise NotImplementedError("bf16 tensor-core path implements the nerf_lm_adapt_gan.yaml architecture only; "
                                  "use opt.b200.mlp='fp32' for other layer shapes")
    center, ray, depth = geom["center"], geom["ray"], geom["depth"]
    B, R, N = geom["shape"]
    S, per_image = geom["S"], geom["per_image"]
    dev = depth.device
    flat = [t for pair in (feat_p + rgb_p + trans_p) for t in pair]
    pk = pack(cfg, cfg.packed, feat_p, rgb_p, trans_p, flat)
    W_r0 = rgb_p[0][0]
    img_r, img_t = image_biases(cfg, B, lat_trans, lat_light, rgb_p, trans_p)
    raybias = torch.empty(B * R, _F, device=dev)
    _C.call("tp_tc_ray_bias", ops._p(ray), B * R, R, cfg.L_view, ops._p(W_r0), W_r0.stride(0), 256, ops._p(img_r),
            ops._p(raybias), ops._stream())
    rgb = torch.empty(S, 3, 2, device=dev)
    density = torch.empty(S, 2, device=dev)
    uncert = torch.empty(S, device=dev)
    scratch = _scratch_for(dev)
    images = torch.empty(_C.load().tp_tc_save_bytes(S), dtype=torch.uint8, device=dev) if save else None
    _C.call("tp_tc_nerf_stl_forward", ops._p(center), ops._p(ray), ops._p(depth), S, N, per_image, ops._p(pk.weights),
            ops._p(pk.biasbuf), ops._p(raybias), ops._p(img_t), ops._p(rgb), ops._p(density), ops._p(uncert),
            ops._p(scratch), scratch.numel(), ops._p(images), flags, ops._stream())
    if save:
        return rgb, density, uncert, images
    return rgb, density, uncert


RENDER_KEYS = ("rgb", "rgb_static", "rgb_transient", "depth", "opacity", "opacity_static", "opacity_transient", "uncert",
               "alpha_static", "alpha_transient", "density")


def render_fused(cfg, kinv, pinv, H, W, ray_idx, ray0, R, z_near, z_far, N, lat_trans, lat_light, feat_p, rgb_p, trans_p,
                 min_uncert, rand=None, stratified=True, seed=0, static_only=False, want=RENDER_KEYS, out_ptrs=None):
    """Graph.render after ray selection (model/nerf_adapt_st_gan.py:565-631) as ONE launch: tp_render_fused_forward.

    ray_idx: [B,R] int64 pixel indices, or None for the row block [ray0, ray0+R) of every view.  z_near / z_far: [B,H*W].
    want: which of the reference's eleven outputs are materialised.  out_ptrs: {key: raw device address} overriding the
    destination of an output (e.g. a row block of a frame buffer in a peer GPU's window: the stores then travel over NVLink);
    such outputs are not returned.  Returns the dict of allocated outputs in the reference's shapes."""
    if N not in FUSED_N:
        raise NotImplementedError(f"the fused render launch takes {FUSED_N} samples per ray")
    if not supported(cfg, feat_p, rgb_p, trans_p):
        raise NotImplementedError("bf16 tensor-core path implements the nerf_lm_adapt_gan.yaml architecture only")
    B = kinv.shape[0]
    dev = kinv.device
    flat = [t for pair in (feat_p + rgb_p + trans_p) for t in pair]
    pk = pack(cfg, cfg.packed, feat_p, rgb_p, trans_p, flat)
    img_r, img_t = image_biases(cfg, B, lat_trans, lat_light, rgb_p, trans_p)
    shapes = dict(rgb=(B, R, 3), rgb_static=(B, R, 3), rgb_transient=(B, R, 3), depth=(B, R, 1), opacity=(B, R, 1),
                  opacity_static=(B, R, 1), opacity_transient=(B, R, 1), uncert=(B, R, 1), alpha_static=(B, R, N),
                  alpha_transient=(B, R, N), density=(B, R, N, 2))
    out_ptrs = out_ptrs or {}
    ret = {k: torch.empty(shapes[k], device=dev) for k in want if k not in out_ptrs}
    if B * R == 0:
        return ret
    import ctypes

    def dst(k):
        if k in out_ptrs:
            return ctypes.c_void_p(int(out_ptrs[k]))
        return ops._p(ret[k]) if k in ret else None

    if rand is not None:
        mode, rand_t = 0, ops._f32(rand)
        assert rand_t.numel() == B * R * N
    elif not stratified:
        mode, rand_t = 1, None
    else:
        mode, rand_t = 2, None
    if ray_idx is not None:
        ray_idx = ray_idx.to(torch.int64).contiguous()
        assert ray_idx.shape == (B, R)
    scratch = _scratch_for(dev)
    _C.call("tp_render_fused_forward", ops._p(kinv), ops._p(pinv), B, H, W, 0.5, ops._p(ray_idx), R, int(ray0), ops._p(z_near),
            ops._p(z_far), N, mode, ops._p(rand_t), int(seed), ops._p(pk.weights), ops._p(pk.biasbuf), ops._p(pk.wview),
            cfg.L_view, ops._p(img_r), ops._p(img_t), float(min_uncert), *[dst(k) for k in RENDER_KEYS], ops._p(scratch),
            scratch.numel(), STATIC_ONLY if static_only else 0, ops._stream())
    return ret
