"""Host side of the tensor-core backward of the two heads (bf16 mode): transposed weight image, kernel sequencing.

Two backwards, one per forward: `heads_backward` (csrc/mlp_tc_bwd.cu, tp_tc_heads_backward) after the lock-step forward, and
`heads_backward_staged` (csrc/mlp_tc_chain.cu + the dW GEMM and thin helpers here) after the single-pass staged forward -- or,
with split = True, after the split-save forward of the fp32-parity step.  NerfMLP.forward picks the forward, and with it the
backward.

Gradient sinks are the reference's: mlp_rgb.*, mlp_trans.*, the two latents (model/nerf_adapt_st_gan.py:56-69,108-127);
the trunk is frozen (layers/nerf_static_transient_light.py:34).
"""
from __future__ import annotations

import ctypes
import os

import torch

from . import _C, ops

last_profile_workspace = None       # (workspace tensor, float offset of the counters) of the last instrumented call


def _bwd_table(rgb_p, trans_p):
    rows = []
    for layers in (rgb_p, trans_p):
        W3, W2, W1 = layers[3][0], layers[2][0], layers[1][0]
        rows.append([W3.data_ptr(), W3.stride(0), 0, 256, 0, W3.shape[0], 256, 0, -1, 1])     # K=16 chunk: W3^T
        for W in (W2, W1):
            for c in range(0, 256, 32):
                rows.append([W.data_ptr(), W.stride(0), 0, 256, c, 32, 256, 0, -1, 1])
    return rows


def pack_bwd(holder, rgb_p, trans_p):
    params = [w for w, _ in (rgb_p[1:] + trans_p[1:])]
    key = tuple((p.data_ptr(), p._version) for p in params)
    cached = getattr(holder, "_packed_bwd", None) if holder is not None else None
    if cached is not None and cached[0] == key:
        return cached[1]
    lib = _C.load()
    dev = rgb_p[0][0].device
    where = tuple((p.data_ptr(), p.stride(0)) for p in params)
    if cached is not None and len(cached) > 3 and cached[3] == where:      # same addresses: last step's descriptor table
        desc = cached[2]
    else:
        table = _bwd_table(rgb_p, trans_p)
        assert len(table) == lib.tp_tc_bwd_num_chunks()
        desc = ops.device_table(table, torch.int64, dev)
    n = lib.tp_tc_bwd_num_chunks()
    img = torch.empty(n * lib.tp_tc_chunk_bytes(), dtype=torch.uint8, device=dev)
    _C.call("tp_tc_pack_weights", ops._p(desc), n, ops._p(img), ops._stream())
    if holder is not None:
        holder._packed_bwd = (key, img, desc, where)
    return img


def reduce_partials(partial, splits, count, out=None):
    out = torch.empty(count, device=partial.device) if out is None else out
    _C.call("tp_reduce_partials", ops._p(partial), splits, count, ops._p(out), 0, ops._stream())
    return out


# split = True: the images are the fp32-parity backward's (tp_tc32_forward_split_save, tp_tc_chain_backward_split): every logical
# slot k is the pair of bf16 images 2k (hi) and 2k + 1 (lo), and the helpers below run the bf16 kernels on both and add the parts
# in a fixed order (tp_reduce_partials).  Slot numbers and slot counts passed in are logical.

def dw_gemm(a_images, a_nslots, b_images, b_nslots, pairs, S, split=False):
    """[len(pairs),256,256] fp32: job j = dz[a]^T x[b] over all samples -- one launch per 12 jobs, split over tiles, fixed-order
    reduce.  split: three jobs per pair, (dz_hi, x_hi) + (dz_hi, x_lo) + (dz_lo, x_hi) (the dropped lo x lo term is ~2^-17)."""
    if split:
        n = len(pairs)
        jobs = [(2 * a + i, 2 * b + j) for i, j in ((0, 0), (0, 1), (1, 0)) for a, b in pairs]      # term-major
        parts = torch.cat([dw_gemm(a_images, 2 * a_nslots, b_images, 2 * b_nslots, jobs[k:k + 12], S) for k in range(0, len(jobs), 12)])
        return reduce_partials(parts, 3, n * 65536).view(n, 256, 256)
    n = len(pairs)
    splits = _C.load().tp_tc_dw_splits(S, n)
    partial = torch.empty(splits * n * 65536, device=a_images.device)
    a_s = (ctypes.c_int32 * n)(*[a for a, _ in pairs])
    b_s = (ctypes.c_int32 * n)(*[b for _, b in pairs])
    _C.call("tp_tc_dw_gemm", ops._p(a_images), a_nslots, ops._p(b_images), b_nslots, a_s, b_s, n, S, ops._p(partial),
            partial.numel(), ops._stream())
    return reduce_partials(partial, splits, n * 65536).view(n, 256, 256)


def images_colsum(images, n_slots, S, slots, split=False):
    """[len(slots),256]: column sums over all samples of the selected image slots (bias gradients), one launch + one reduce."""
    lib = _C.load()
    n = len(slots)
    sel_slots = [2 * s for s in slots] + [2 * s + 1 for s in slots] if split else list(slots)
    blocks, n_sel = lib.tp_tc_images_colsum_blocks(), len(sel_slots)
    sel = ops.device_table(sel_slots, torch.int32, images.device)
    partial = torch.empty(blocks * n_sel * 256, device=images.device)
    _C.call("tp_tc_images_colsum", ops._p(images), n_slots * (2 if split else 1), S, ops._p(sel), n_sel, ops._p(partial),
            partial.numel(), ops._stream())
    return reduce_partials(partial, blocks * (n_sel // n), n * 256).view(n, 256)      # [blocks][hi | lo][n][256]


def image_ray_sums(images, slot, n_slots, S, N, split=False):
    rays = (S + N - 1) // N
    if not split:
        out = torch.empty(rays, 256, device=images.device)
        _C.call("tp_tc_image_ray_sums", ops._p(images), slot, n_slots, S, N, ops._p(out), ops._stream())
        return out
    parts = torch.empty(2, rays, 256, device=images.device)
    for i in range(2):
        _C.call("tp_tc_image_ray_sums", ops._p(images), 2 * slot + i, 2 * n_slots, S, N, ops._p(parts[i]), ops._stream())
    return reduce_partials(parts, 2, rays * 256).view(rays, 256)


def thin_colsum(x, S):
    C = x.shape[1]
    ws = torch.empty(2 * 148 * 8 + 64, device=x.device)
    out = torch.empty(C, device=x.device)
    _C.call("tp_thin_colsum", ops._p(x), S, C, ops._p(out), ops._p(ws), ws.numel(), ops._stream())
    return out


def thin_dw(thin, images, slot, n_slots, S, split=False):
    """[M,256] = thin^T x for a thin fp32 operand [S,M] (M in 1,3,5) and an image slot x."""
    M = thin.shape[1]
    max_blocks = 148 * 4 + 8
    parts = 2 if split else 1
    partial = torch.empty(parts * max_blocks * M * 256, device=thin.device)
    used = 0
    for i in range(parts):
        nb = ctypes.c_int(0)
        _C.call("tp_tc_thin_dw", ops._p(thin), M, ops._p(images), parts * slot + i, parts * n_slots, S,
                ops._p(partial[used * M * 256:]), partial.numel() - used * M * 256, ctypes.byref(nb), ops._stream())
        used += nb.value
    return reduce_partials(partial, used, M * 256).view(M, 256)


def fused_supported(S, per_image) -> bool:
    """Whether tp_tc_heads_backward takes a batch: one CTA's contiguous tile range may touch at most four images."""
    return bool(_C.load().tp_tc_heads_backward_supported(S, per_image))


def heads_backward(cfg, sv, S, per_image, rgb_p, trans_p, g_rgb, g_density, g_uncert, need_lat_trans, need_lat_light):
    """Backward of the yaml's 3 x 256 heads on the tile images the lock-step forward saved, in five launches
    (tp_tc_heads_backward).  Returns (rgb layer grads [(dW,db)]*4, trans layer grads, d_lat_trans, d_lat_light).
    The batch must satisfy fused_supported(S, per_image); NerfMLP.forward sends any other batch to the staged kernels."""
    dev = sv.rgb.device
    geom = sv.geom
    lt, ll = sv.lat
    B, R, N = geom["shape"]
    dz_rgb = torch.empty(S, 3, device=dev)
    dz_trans = torch.empty(S, 5, device=dev)
    _C.call("tp_stl_output_grad", ops._p(sv.rgb), ops._p(sv.density), ops._p(sv.uncert), ops._p(g_rgb), ops._p(g_density),
            ops._p(g_uncert), S, ops._p(dz_rgb), ops._p(dz_trans), None, ops._stream())
    packed = pack_bwd(cfg.packed, rgb_p, trans_p)
    lib = _C.load()
    dz = torch.empty(lib.tp_tc_dz_bytes(S), dtype=torch.uint8, device=dev)
    need = lib.tp_tc_heads_backward_workspace(S, B)
    prof = bool(os.environ.get("TEXPOSE_CHAIN_PROF"))       # scripts/chain_prof.py: cycle counters land in the workspace tail
    ws = torch.empty(need + (32 * 160 + 2 if prof else 0), device=dev)
    if prof:
        global last_profile_workspace
        last_profile_workspace = (ws, (need + 1) & ~1)
    grads = []
    for layers in (rgb_p, trans_p):
        for W, b in layers:
            grads += [torch.empty_like(W), torch.empty_like(b)]
    W_r0, W_t0 = rgb_p[0][0], trans_p[0][0]
    d_ll = torch.empty(B, cfg.n_latent_light, device=dev) if need_lat_light else None
    d_lt = torch.empty(B, cfg.n_latent_trans, device=dev) if need_lat_trans else None
    center, ray, depth = geom["center"], geom["ray"], geom["depth"]
    gp = (ctypes.c_void_p * 16)(*[t.data_ptr() for t in grads])
    _C.call("tp_tc_heads_backward", ops._p(dz_rgb), ops._p(dz_trans), S, N, per_image, B, ops._p(center), ops._p(ray),
            ops._p(depth), cfg.L_view, ops._p(packed), ops._p(sv.images), ops._p(dz), ops._p(W_r0), W_r0.stride(0),
            ops._p(W_t0), W_t0.stride(0), ops._p(ll), cfg.n_latent_light, ops._p(lt), cfg.n_latent_trans, gp,
            ops._p(d_ll), ops._p(d_lt), ops._p(ws), ws.numel(), ops._stream())
    pairs = [(grads[2 * i], grads[2 * i + 1]) for i in range(8)]
    return pairs[:4], pairs[4:], d_lt, d_ll


def heads_backward_staged(cfg, sv, S, per_image, rgb_p, trans_p, g_rgb, g_density, g_uncert, need_lat_trans, need_lat_light,
                          split=False):
    """The two heads' backward for ANY head depth (256-wide layers), on the staged kernels: the activations are the tile images /
    ReLU bitmasks the single-pass staged forward saved (slots: feature, rgb hidden 1.., transient hidden 1.., encoding tile), the
    dX chains are two tp_tc_chain_backward launches (one per head: its output layer's dz enters as the thin operand), the
    256 x 256 weight gradients one tp_tc_dw_gemm launch, the thin pieces the helpers above.  Used when tp_tc_heads_backward's
    fixed stage table (the yaml's 3 x 256 heads) does not describe the architecture, or when its images are too small for it
    (fused_supported is false).  split: the fp32-parity step -- the images are the bf16 hi / lo pairs of the split-save forward,
    the chains tp_tc_chain_backward_split launches over K = 16 hi | lo weight slots."""
    from . import mlp_tc32  # noqa: F401  (save layout)
    dev = sv.rgb.device
    geom = sv.geom
    lt, ll = sv.lat
    B, R, N = geom["shape"]
    images, n_save = sv.images, sv.n_save
    nr, nt = len(rgb_p), len(trans_p)
    slot_feat = 0
    slot_r = lambda i: i                  # rgb hidden activation h_i (output of rgb layer i-1), i = 1 .. nr-1
    slot_t = lambda i: (nr - 1) + i       # transient hidden activation, i = 1 .. nt-1
    lib = _C.load()
    parts = 2 if split else 1             # tile images per slot (split: hi, lo)
    k = 16 if split else 32               # K rows of W per packed chunk
    dz_rgb, dz_trans = torch.empty(S, 3, device=dev), torch.empty(S, 5, device=dev)
    _C.call("tp_stl_output_grad", ops._p(sv.rgb), ops._p(sv.density), ops._p(sv.uncert), ops._p(g_rgb), ops._p(g_density),
            ops._p(g_uncert), S, ops._p(dz_rgb), ops._p(dz_trans), None, ops._stream())
    n_tiles = (S + 127) // 128
    n_dz = (nr - 1) + (nt - 1)            # dz of every hidden layer's pre-activation: rgb nr-2 .. 0, then transient nt-2 .. 0
    dz = torch.empty(n_tiles * parts * n_dz * 65536, dtype=torch.uint8, device=dev)
    bits = images[n_tiles * parts * n_save * 65536:]
    rows = []

    def chain(layers, thin, slot_h, dz0):
        """Stage list of one head: out layer (thin) -> hidden layers n-2 .. 1; dz slot dz0 + j holds the dz of layer n-2-j."""
        n = len(layers)
        W_out = layers[n - 1][0]
        rows.append([W_out.data_ptr(), W_out.stride(0), 0, 256, 0, W_out.shape[0], 256, 0, -1, 1])
        stages = [[0, len(rows) - 1, 0, 0, slot_h(n - 1), dz0]]
        for j, li in enumerate(range(n - 2, 0, -1)):
            c0 = len(rows)
            W = layers[li][0]
            for c in range(0, 256, k):
                rows.append([W.data_ptr(), W.stride(0), 0, 256, c, k, 256, 0, -1, 1])
            stages.append([-1, 0, c0, 256 // k, slot_h(li), dz0 + 1 + j])
        return thin, stages

    jobs = [chain(rgb_p, dz_rgb, slot_r, 0), chain(trans_p, dz_trans, slot_t, nr - 1)]
    desc = ops.device_table(rows, torch.int64, dev)
    packed = torch.empty(len(rows) * lib.tp_tc_chunk_bytes(), dtype=torch.uint8, device=dev)
    _C.call("tp_tc_pack_weights_split" if split else "tp_tc_pack_weights", ops._p(desc), len(rows), ops._p(packed), ops._stream())
    for thin, stages in jobs:
        st = torch.tensor(stages, dtype=torch.int32)
        _C.call("tp_tc_chain_backward_split" if split else "tp_tc_chain_backward", ops._p(thin), thin.shape[1], None, 0, S,
                ops._p(packed), len(rows), ops._p(st), len(stages), ops._p(bits), n_save, ops._p(dz), n_dz, ops._stream())
    # dz slot of layer li's pre-activation (li = 0 .. n-2)
    dzr = lambda li: (nr - 2) - li
    dzt = lambda li: (nr - 1) + (nt - 2) - li
    pairs = [(dzr(li), slot_r(li) if li else slot_feat) for li in range(nr - 2, -1, -1)] + \
            [(dzt(li), slot_t(li) if li else slot_feat) for li in range(nt - 2, -1, -1)]
    if split:
        big = dw_gemm(dz, n_dz, images, n_save, pairs, S, split=True)
    else:
        big = torch.cat([dw_gemm(dz, n_dz, images, n_save, pairs[i:i + 12], S) for i in range(0, len(pairs), 12)], dim=0)
    big_r = {li: big[j] for j, li in enumerate(range(nr - 2, -1, -1))}
    big_t = {li: big[(nr - 1) + j] for j, li in enumerate(range(nt - 2, -1, -1))}
    sums = images_colsum(dz, n_dz, S, list(range(n_dz)), split=split)                     # bias gradients of every hidden layer
    grads_r, grads_t = [None] * nr, [None] * nt
    grads_r[nr - 1] = (thin_dw(dz_rgb, images, slot_r(nr - 1), n_save, S, split=split), thin_colsum(dz_rgb, S))
    grads_t[nt - 1] = (thin_dw(dz_trans, images, slot_t(nt - 1), n_save, S, split=split), thin_colsum(dz_trans, S))
    for li in range(1, nr - 1):
        grads_r[li] = (big_r[li], sums[dzr(li)])
    for li in range(1, nt - 1):
        grads_t[li] = (big_t[li], sums[dzt(li)])
    # ---- layer 0 of each head: feature columns from the GEMM, per-ray view / per-sample xyz / per-image latent columns
    W_r0, W_t0 = rgb_p[0][0], trans_p[0][0]
    g_ray = image_ray_sums(dz, dzr(0), n_dz, S, N, split=split)                            # [B*R,256]
    g_img = ops.group_colsum(g_ray, B * R, R)                                              # [B,256]
    g_timg = ops.group_colsum(image_ray_sums(dz, dzt(0), n_dz, S, N, split=split), B * R, R)
    view_t, _, vc = geom["view_seg"]()
    dW_view, _ = ops.linear_backward_weight(g_ray, [(view_t, 1, vc)], B * R, want_bias=False)
    xyz = ops.points_from_depth(geom["center"], geom["ray"], geom["depth"]).view(S, 3)
    dW_xyz = thin_dw(xyz, dz, dzr(0), n_dz, S, split=split).t().contiguous()
    dW_light, _ = ops.linear_backward_weight(g_img, [(ll, 1, cfg.n_latent_light)], B, want_bias=False)
    grads_r[0] = (torch.cat([big_r[0], dW_view, dW_xyz, dW_light], dim=1), sums[dzr(0)])
    d_ll = ops.linear_backward_input(g_img, W_r0, B, cfg.n_latent_light, None, w_col0=256 + vc + 3) if need_lat_light else None
    dW_lt, _ = ops.linear_backward_weight(g_timg, [(lt, 1, cfg.n_latent_trans)], B, want_bias=False)
    grads_t[0] = (torch.cat([big_t[0], dW_lt], dim=1), sums[dzt(0)])
    d_lt = ops.linear_backward_input(g_timg, W_t0, B, cfg.n_latent_trans, None, w_col0=256) if need_lat_trans else None
    return grads_r, grads_t, d_lt, d_ll
