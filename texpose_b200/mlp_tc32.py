"""Host side of the fp32-parity tensor-core forward (csrc/mlp_tc_split.cu): stage list, split weight image, launch.

The kernel takes its stage list as data, so this module derives it from the caller's architecture (trunk depth, skip
positions, head depths: `opt.arch` of the reference yaml files) instead of relying on a table compiled into the kernel.
Every layer is carried as hi + lo fp16 (three MMA passes per K step): <= 1e-4 against the reference where the bf16
kernel (mlp_tc.py) is <= 1e-2.  A training step in the parity mode (opt.b200.fp32_engine = 'tc') uses the split-save launch,
which also keeps the activations as bf16 hi + lo tile images for the split backward (mlp_tc_plain, mlp_tc_bwd).
"""
from __future__ import annotations

import torch

from . import _C, mlp_tc, ops

_F = 256
KIND_HIDDEN, KIND_DENSITY, KIND_RGB_OUT, KIND_TRANS_OUT = 0, 1, 2, 3
BIAS_STATIC, BIAS_RAY, BIAS_IMAGE = 0, 1, 2
F_WAIT_READY, F_RELOAD, F_PARK, F_E_LAST = 1, 2, 4, 8


def supported(cfg, feat_p, rgb_p, trans_p) -> bool:
    """Static / transient / light model with 256-wide hidden layers, any trunk depth >= 2, any skip set (not the first or
    the last trunk layer), any head depth >= 2; L_3D = 10 (the encoding tile has 64 columns)."""
    if not (cfg.stl and cfg.view_dep and cfg.L_3D == 10 and 0 <= cfg.L_view <= 4):
        return False
    nf, nr, nt = len(feat_p), len(rgb_p), len(trans_p)
    if nf < 2 or nr < 2 or nt < 2:
        return False
    skip = set(cfg.skip)
    if 0 in skip or nf - 1 in skip:
        return False
    ec = cfg.enc_cols
    for li, (w, _) in enumerate(feat_p):
        k = ec if li == 0 else _F + (ec if li in skip else 0)
        if tuple(w.shape) != ((_F + 1 if li == nf - 1 else _F), k):
            return False
    k_rgb0 = _F + cfg.view_cols + 3 + cfg.n_latent_light
    want_r = [(_F, k_rgb0)] + [(_F, _F)] * (nr - 2) + [(3, _F)]
    want_t = [(_F, _F + cfg.n_latent_trans)] + [(_F, _F)] * (nt - 2) + [(5, _F)]
    if [tuple(w.shape) for w, _ in rgb_p] != want_r or [tuple(w.shape) for w, _ in trans_p] != want_t:
        return False
    n_stages = (nf + 1) + nr + nt
    return n_stages <= _C.load().tp_tc32_max_stages()


def build_tables(cfg, feat_p, rgb_p, trans_p, static_only=False, save=False):
    """-> (slot descriptor rows, stage rows, bias tensors).  Within a stage the K steps that read the encoding tile come first
    (it is ready long before the previous drain finishes), then the sixteen K steps over the activation tile.  save: every hidden
    stage gets a save slot, numbered in execution order (trunk layers, feature, rgb hidden layers, transient hidden layers)."""
    slots, stages, biases = [], [], []
    off = [0]

    def add_bias(b):
        o = off[0]
        biases.append(b.reshape(-1))
        pad = (-b.numel()) % 4
        if pad:
            biases.append(torch.zeros(pad, device=b.device))
        off[0] += b.numel() + pad
        return o

    def a_slots(W, col0, row0=0):
        for i in range(16):
            slots.append([W.data_ptr(), W.stride(0), row0, _F, col0 + 16 * i, 16, 256, 0])
        return 16

    def e_slots(W, col0, ncols):
        n = (ncols + 15) // 16
        for i in range(n):
            slots.append([W.data_ptr(), W.stride(0), 0, _F, col0 + 16 * i, min(16, ncols - 16 * i), 256, 0])
        return n

    def small(W, row0, nrows):
        slots.append([W.data_ptr(), W.stride(0), row0, nrows, 0, _F, 16, 0])

    ec, skip = cfg.enc_cols, set(cfg.skip)
    nf = len(feat_p)
    for li, (W, b) in enumerate(feat_p[:-1]):
        if li == 0:
            stages.append([0, e_slots(W, 0, ec), KIND_HIDDEN, BIAS_STATIC, add_bias(b), 0])
        else:
            e = e_slots(W, _F, ec) if li in skip else 0
            stages.append([a_slots(W, 0), e, KIND_HIDDEN, BIAS_STATIC, add_bias(b), F_WAIT_READY])
    W, b = feat_p[nf - 1]       # row 0 -> static density, rows 1.. -> the feature both heads read
    small(W, 0, 1)
    stages.append([16, 0, KIND_DENSITY, BIAS_STATIC, add_bias(b[:1]), F_WAIT_READY])
    stages.append([a_slots(W, 0, row0=1), 0, KIND_HIDDEN, BIAS_STATIC, add_bias(b[1:]), 0 if static_only else F_PARK])
    # rgb head: [feature | view encoding + light latent (per-ray bias row) | xyz (first K step of the encoding tile)]
    W, b = rgb_p[0]
    e = e_slots(W, _F + cfg.view_cols, 3)
    stages.append([a_slots(W, 0), e, KIND_HIDDEN, BIAS_RAY, 0, F_WAIT_READY | F_E_LAST])
    for W, b in rgb_p[1:-1]:
        stages.append([a_slots(W, 0), 0, KIND_HIDDEN, BIAS_STATIC, add_bias(b), F_WAIT_READY])
    W, b = rgb_p[-1]
    small(W, 0, 3)
    stages.append([16, 0, KIND_RGB_OUT, BIAS_STATIC, add_bias(b), F_WAIT_READY])
    if not static_only:
        W, b = trans_p[0]      # [feature | transient latent (per-image bias row)]
        stages.append([a_slots(W, 0), 0, KIND_HIDDEN, BIAS_IMAGE, 0, F_RELOAD])
        for W, b in trans_p[1:-1]:
            stages.append([a_slots(W, 0), 0, KIND_HIDDEN, BIAS_STATIC, add_bias(b), F_WAIT_READY])
        W, b = trans_p[-1]
        small(W, 0, 5)
        stages.append([16, 0, KIND_TRANS_OUT, BIAS_STATIC, add_bias(b), F_WAIT_READY])
    # save slots: 'all' / True = every hidden stage in execution order (trunk layers, feature, rgb hidden, transient hidden);
    # 'heads' = from the feature stage on (frozen trunk: layers/nerf_static_transient_light.py:34,87 -- its activations are not needed)
    first = (len(feat_p) - 1) if save == "heads" else 0      # index, among the hidden stages, of the first one that is kept
    n_hidden = 0
    for st in stages:
        hidden = st[2] == KIND_HIDDEN
        st.append(n_hidden - first if (save and hidden and n_hidden >= first) else -1)
        n_hidden += hidden
    return slots, stages, biases


class Packed:
    __slots__ = ("key", "image", "n_slots", "stages", "bias", "keep", "n_save", "wview")


def pack(cfg, holder, feat_p, rgb_p, trans_p, static_only=False, precision=0, save=False) -> Packed:
    """precision 0: split fp16 hi + lo image (three passes, <= 1e-4); 1: bf16 image for the single-pass launch (<= 1e-2)."""
    flat = [t for pair in (feat_p + rgb_p + trans_p) for t in pair]
    key = (mlp_tc._version_key(flat), bool(static_only), int(precision), str(save))
    attr = "_packed32" if precision == 0 else "_packed16"
    cache = getattr(holder, attr, None) if holder is not None else None
    if cache is not None and cache.key == key:
        return cache
    slots, stages, biases = build_tables(cfg, feat_p, rgb_p, trans_p, static_only, save)
    dev = feat_p[0][0].device
    desc = ops.device_table(slots, torch.int64, dev)
    image = torch.empty(len(slots) * _C.load().tp_tc32_slot_bytes(), dtype=torch.uint8, device=dev)
    _C.call("tp_tc32_pack_weights", ops._p(desc), len(slots), int(precision), ops._p(image), ops._stream())
    out = Packed()
    out.key, out.image, out.n_slots = key, image, len(slots)
    out.stages = torch.tensor(stages, dtype=torch.int32)           # host: the launch copies it into the kernel parameters
    out.bias = torch.cat([b.float() for b in biases]).contiguous()
    out.keep = desc
    out.n_save = sum(1 for st in stages if st[6] >= 0) + (1 if save else 0)      # + the encoding tile, in the last slot
    out.wview = None          # the render launch's view-encoding weight columns (render(), built on first use)
    if holder is not None:
        try:
            setattr(holder, attr, out)
        except AttributeError:
            pass
    return out


_scratch = {}


def _scratch_for(dev):
    k = (dev.type, dev.index)
    if k not in _scratch:
        lib = _C.load()      # one buffer for both launches: the render launch's is tp_tc32_forward's plus its view-bias rows
        n = max(lib.tp_tc32_scratch_bytes(), lib.tp_tc32_render_scratch_bytes())
        _scratch[k] = torch.zeros(n, dtype=torch.uint8, device=dev)      # (status word starts at 0)
    return _scratch[k]


def check_range(device=None):
    """Off the hot path (one 4-byte read-back): raises if a split-mode launch on `device` saw a hidden activation outside the fp16
    range (> 6e4, or NaN) since the last check -- its outputs are then not the <= 1e-4 ones; use opt.b200.fp32_engine = 'simt'."""
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    k = (dev.type, dev.index)
    if k not in _scratch:
        return
    off = _C.load().tp_tc32_status_offset()
    word = _scratch[k][off:off + 4]
    bad = int(word.view(torch.int32).item())
    if bad:
        word.zero_()
        raise FloatingPointError("tp_tc32_forward: a hidden activation left the fp16 range of the split-precision mode")


def forward(cfg, geom, lat_trans, lat_light, feat_p, rgb_p, trans_p, static_only=False, precision=0, save=False):
    """NeRF.forward_samples (layers/nerf_static_transient_light.py:147-166) -> rgb [S,3,2], density [S,2], uncert [S]
    (+ (images, n_save) with save: the tile images of every hidden activation -- bf16 for the single-pass launch (precision 1),
    bf16 hi / lo pairs, images 2k and 2k + 1 of save slot k, for the split launch (precision 0, tp_tc32_forward_split_save))."""
    if geom.get("mode") != "rays":
        raise NotImplementedError("the tensor-core kernels are ray-parameterised (forward_samples)")
    if not supported(cfg, feat_p, rgb_p, trans_p):
        raise NotImplementedError("fp32-parity tensor-core path: 256-wide static/transient/light architectures with L_3D = 10")
    center, ray, depth = geom["center"], geom["ray"], geom["depth"]
    B, R, N = geom["shape"]
    S, per_image = geom["S"], geom["per_image"]
    dev = depth.device
    pk = pack(cfg, cfg.packed, feat_p, rgb_p, trans_p, static_only, precision, save)
    W_r0 = rgb_p[0][0]
    img_r, img_t = mlp_tc.image_biases(cfg, B, lat_trans, lat_light, rgb_p, trans_p)
    raybias = torch.empty(B * R, _F, device=dev)
    _C.call("tp_tc_ray_bias", ops._p(ray), B * R, R, cfg.L_view, ops._p(W_r0), W_r0.stride(0), 256, ops._p(img_r),
            ops._p(raybias), ops._stream())
    rgb = torch.empty(S, 3, 2, device=dev)
    density = torch.empty(S, 2, device=dev)
    uncert = torch.empty(S, device=dev)
    scratch = _scratch_for(dev)
    images = None
    if save:
        lib = _C.load()
        nbytes = lib.tp_tc32_save_bytes(S, pk.n_save) if precision else lib.tp_tc32_split_save_bytes(S, pk.n_save)
        images = torch.empty(nbytes, dtype=torch.uint8, device=dev)      # tile images, then ReLU bitmasks
    if save and precision == 0:
        _C.call("tp_tc32_forward_split_save", ops._p(center), ops._p(ray), ops._p(depth), S, N, per_image, ops._p(pk.image),
                pk.n_slots, ops._p(pk.stages), pk.stages.shape[0], ops._p(pk.bias), ops._p(raybias), ops._p(img_t), ops._p(rgb),
                ops._p(density), ops._p(uncert), ops._p(scratch), scratch.numel(), ops._p(images), pk.n_save, pk.n_save - 1,
                ops._stream())
        return rgb, density, uncert, (images, pk.n_save)
    _C.call("tp_tc32_forward", ops._p(center), ops._p(ray), ops._p(depth), S, N, per_image, ops._p(pk.image), pk.n_slots,
            ops._p(pk.stages), pk.stages.shape[0], ops._p(pk.bias), ops._p(raybias), ops._p(img_t), ops._p(rgb),
            ops._p(density), ops._p(uncert), ops._p(scratch), scratch.numel(), int(precision), ops._p(images), pk.n_save if save else 0,
            pk.n_save - 1 if save else -1, ops._stream())
    if save:
        return rgb, density, uncert, (images, pk.n_save)
    return rgb, density, uncert


RENDER_KEYS = ("rgb", "rgb_static", "rgb_transient", "depth", "opacity", "opacity_static", "opacity_transient", "uncert",
               "alpha_static", "alpha_transient", "density")
PLAIN_RENDER_KEYS = ("rgb", "depth", "opacity", "density")      # the plain model (static_only): one compositing chain


def render(cfg, kinv, pinv, H, W, ray_idx, ray0, R, z_near, z_far, N, lat_trans, lat_light, feat_p, rgb_p, trans_p, min_uncert,
           rand=None, stratified=True, seed=0, static_only=False, precision=0, want=None, out_ptrs=None):
    """Graph.render after ray selection as ONE launch of the staged kernel (tp_tc32_render_forward): rays, depths, the per-ray
    bias row and the compositing happen in-kernel.  static_only=True: the plain layers/nerf.py model (its layer list as
    NeRF._tc32_parameters builds it, one compositing chain, outputs PLAIN_RENDER_KEYS, density [B,R,N]); otherwise the static /
    transient / light model (the eleven RENDER_KEYS).  precision 0: split hi + lo (<= 1e-4); 1: single-pass bf16 (<= 1e-2).
    ray_idx / ray0 / R, z_near / z_far, rand / stratified / seed, want and out_ptrs as mlp_tc.render_fused."""
    import ctypes
    if N not in mlp_tc.FUSED_N:
        raise NotImplementedError(f"the staged render launch takes {mlp_tc.FUSED_N} samples per ray")
    if not supported(cfg, feat_p, rgb_p, trans_p):
        raise NotImplementedError("staged render launch: 256-wide static/transient/light layer lists with L_3D = 10")
    keys = PLAIN_RENDER_KEYS if static_only else RENDER_KEYS
    want = tuple(keys if want is None else want)
    out_ptrs = out_ptrs or {}
    bad = [k for k in tuple(want) + tuple(out_ptrs) if k not in keys]
    if bad:
        raise ValueError(f"the {'plain' if static_only else 'static/transient/light'} render has no output {bad}")
    B = kinv.shape[0]
    dev = kinv.device
    pk = pack(cfg, cfg.packed, feat_p, rgb_p, trans_p, static_only, precision)
    if pk.wview is None:
        pk.wview = rgb_p[0][0][:, _F:_F + cfg.view_cols].t().contiguous()
    if cfg.n_latent_light or cfg.n_latent_trans:
        img_r, img_t = mlp_tc.image_biases(cfg, B, lat_trans, lat_light, rgb_p, trans_p)
    else:      # no latents: the per-image rows are the layer-0 biases (tp_tc_image_biases' bits: the bias, no products)
        img_r = rgb_p[0][1].float().expand(B, _F).contiguous()
        img_t = None if static_only else trans_p[0][1].float().expand(B, _F).contiguous()
    shapes = dict(rgb=(B, R, 3), rgb_static=(B, R, 3), rgb_transient=(B, R, 3), depth=(B, R, 1), opacity=(B, R, 1),
                  opacity_static=(B, R, 1), opacity_transient=(B, R, 1), uncert=(B, R, 1), alpha_static=(B, R, N),
                  alpha_transient=(B, R, N), density=(B, R, N) if static_only else (B, R, N, 2))
    ret = {k: torch.empty(shapes[k], device=dev) for k in want if k not in out_ptrs}
    if B * R == 0:
        return ret

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
    _C.call("tp_tc32_render_forward", ops._p(ops._f32(kinv)), ops._p(ops._f32(pinv)), B, H, W, 0.5, ops._p(ray_idx), R, int(ray0),
            ops._p(z_near), ops._p(z_far), N, mode, ops._p(rand_t), int(seed), ops._p(pk.image), pk.n_slots, ops._p(pk.stages),
            pk.stages.shape[0], ops._p(pk.bias), ops._p(pk.wview), cfg.L_view, ops._p(img_r), ops._p(img_t),
            1 if static_only else 3, float(min_uncert), *[dst(k) for k in RENDER_KEYS], ops._p(scratch), scratch.numel(),
            int(precision), ops._stream())
    return ret
