"""Tensor-level wrappers over the C-ABI (`_C.call`): shape checks, output allocation, stream hand-off.

PyTorch is used for device memory, streams and autograd bookkeeping only -- every arithmetic step of the
hot path runs in libtexpose_b200.so.  CPU tensors are rejected (no CPU fallback).
"""
from __future__ import annotations

import collections
import ctypes
from typing import Optional, Sequence, Tuple

import torch

from . import _C

Tensor = torch.Tensor

ACT_NONE, ACT_RELU, ACT_TRUNK_LAST_STL, ACT_TRUNK_LAST_PLAIN, ACT_RGB_STATIC, ACT_TRANS_OUT, ACT_SIGMOID = range(7)


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("texpose_b200 runs on CUDA tensors only (no CPU fallback); got a CPU tensor")


def _f32(t: Optional[Tensor]) -> Optional[Tensor]:
    if t is None:
        return None
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


_EMPTY_ADDR = {}


def _p(t: Optional[Tensor]):
    """Device address for the C-ABI.  NULL means "argument absent" there, and an empty tensor has no storage (data_ptr 0):
    empty tensors are passed as the address of a small per-device dummy buffer, which a zero-sized call never touches."""
    if t is None:
        return None
    if t.numel() == 0:
        buf = _EMPTY_ADDR.get(t.device)
        if buf is None:
            buf = _EMPTY_ADDR[t.device] = torch.zeros(256, dtype=torch.uint8, device=t.device)
        return ctypes.c_void_p(buf.data_ptr())
    return ctypes.c_void_p(t.data_ptr())


def _stream():
    """The caller's stream (torch's current stream on the current device) as a raw cudaStream_t.  The two C calls cost well
    under a microsecond; `torch.cuda.current_stream()` builds a Stream object through several Python layers (~6 us per launch)."""
    return ctypes.c_void_p(torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice()))


_TABLES = collections.OrderedDict()


def device_table(rows, dtype, device) -> Tensor:
    """Small integer table (weight-chunk descriptors, slot lists) as a device tensor, cached by content.  The rows hold pointers and
    strides of parameters, which do not move between training steps, so a step re-uses the table it uploaded before: a fresh
    `torch.tensor(rows, device=...)` is a pageable host-to-device copy, i.e. one stream synchronisation per call and step."""
    flat = tuple(tuple(r) for r in rows) if rows and isinstance(rows[0], (list, tuple)) else tuple(rows)
    key = (str(device), dtype, flat)
    t = _TABLES.get(key)
    if t is None:
        if torch.cuda.is_available() and torch.cuda.is_current_stream_capturing():
            raise RuntimeError("ops.device_table cannot upload a new table while a CUDA graph is being captured: run the same "
                               "call once before the capture (train_graph.GraphedStep's warm-up does)")
        t = _TABLES[key] = torch.tensor(rows, dtype=dtype, device=device)
        if len(_TABLES) > 256:
            _TABLES.popitem(last=False)
    else:
        _TABLES.move_to_end(key)
    return t


# ------------------------------------------------------------------------------------------------- rays


def mask_ray_list(mask: Tensor, N: int) -> Tuple[Tensor, Tensor, Tensor]:
    """Object-pixel ray list of a mask prior (render_by_slices, model/nerf_adapt_st_gan.py:655) for B views, built on the device
    (tp_mask_ray_list): mask [B,...] (object pixel = mask > 0) -> (list int64 [capacity], n_slots int64 [1], counts int64 [B]).
    Entries q = b*HW + pixel, views in order, pixels ascending, each view's run padded to a multiple of 256 / N with ~(b*HW);
    n_slots and counts stay on the device (no read-back)."""
    _need_cuda(mask)
    B = mask.shape[0]
    m = _f32(mask.reshape(B, -1))
    HW = m.shape[1]
    lib = _C.load()
    cap = int(lib.tp_mask_ray_list_capacity(B, HW, N))
    if cap == 0:
        raise ValueError(f"mask_ray_list: B >= 1, H*W >= 1 and N in (32, 64, 128) (got {B}, {HW}, {N})")
    lst = torch.empty(cap, dtype=torch.int64, device=m.device)
    n_slots = torch.empty(1, dtype=torch.int64, device=m.device)
    counts = torch.empty(B, dtype=torch.int64, device=m.device)
    ws = torch.empty(int(lib.tp_mask_ray_list_workspace(B, HW)), dtype=torch.uint8, device=m.device)
    _C.call("tp_mask_ray_list", _p(m), B, HW, N, _p(lst), cap, _p(n_slots), _p(counts), _p(ws), ws.numel(), _stream())
    return lst, n_slots, counts


MASK_DEFAULT_KEYS = ("rgb", "rgb_static", "rgb_transient", "depth", "opacity", "opacity_static", "opacity_transient", "uncert",
                     "alpha_static", "alpha_transient", "density")


def mask_defaults(mask: Tensor, N: int, min_uncert: float, dst: dict, pix0: int = 0, pix1: Optional[int] = None):
    """The defaults of model/nerf_adapt_st_gan.py:657-667 at the background pixels (mask <= 0) of pixels [pix0, pix1) of every
    view (tp_mask_defaults).  dst: {key: frame-layout tensor [B,HW,...] or raw device address}; absent keys are skipped."""
    B = mask.shape[0]
    m = _f32(mask.reshape(B, -1))
    HW = m.shape[1]

    def ptr(k):
        v = dst.get(k)
        return None if v is None else (ctypes.c_void_p(int(v)) if isinstance(v, int) else _p(v))

    _C.call("tp_mask_defaults", _p(m), B, HW, int(pix0), HW if pix1 is None else int(pix1), N, float(min_uncert),
            *[ptr(k) for k in MASK_DEFAULT_KEYS], _stream())


def raygen(kinv: Tensor, pose_inv: Tensor, H: int, W: int, pix_offset: float = 0.5,
           ray_idx: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
    _need_cuda(kinv, pose_inv, ray_idx)
    kinv, pose_inv = _f32(kinv), _f32(pose_inv)
    B = kinv.shape[0]
    if ray_idx is not None:
        ray_idx = ray_idx.to(torch.int64).contiguous()
        assert ray_idx.shape[0] == B
        R = ray_idx.shape[1]
    else:
        R = H * W
    center = torch.empty(B, R, 3, device=kinv.device, dtype=torch.float32)
    ray = torch.empty_like(center)
    _C.call("tp_raygen", _p(kinv), _p(pose_inv), B, H, W, pix_offset, _p(ray_idx), R, _p(center), _p(ray), _stream())
    return center, ray


def patch_rays(kinv: Tensor, pose_inv: Tensor, coords: Tensor, H: int, W: int) -> Tuple[Tensor, Tensor]:
    _need_cuda(kinv, pose_inv, coords)
    kinv, pose_inv, coords = _f32(kinv), _f32(pose_inv), _f32(coords)
    B, h, w, _ = coords.shape
    center = torch.empty(B, h, w, 3, device=coords.device, dtype=torch.float32)
    ray = torch.empty_like(center)
    _C.call("tp_patch_rays", _p(kinv), _p(pose_inv), _p(coords), B, h * w, H, W, _p(center), _p(ray), _stream())
    return center, ray


def grid_sample_bilinear(image: Tensor, coords: Tensor) -> Tensor:
    """F.grid_sample(image[B,C,H,W], coords[B,h,w,2], 'bilinear', align_corners=True) -> [B,C,h,w]."""
    _need_cuda(image, coords)
    image, coords = _f32(image), _f32(coords)
    B, C, H, W = image.shape
    _, h, w, _ = coords.shape
    out = torch.empty(B, C, h, w, device=image.device, dtype=torch.float32)
    _C.call("tp_grid_sample_bilinear", _p(image), _p(coords), B, C, H, W, h * w, _p(out), _stream())
    return out


def gather_rows(src: Tensor, idx: Tensor) -> Tensor:
    _need_cuda(src, idx)
    src = _f32(src)
    idx = idx.to(torch.int64).contiguous()
    B, HW, C = src.shape
    R = idx.shape[1]
    out = torch.empty(B, R, C, device=src.device, dtype=torch.float32)
    if R == 0:
        return out
    _C.call("tp_gather_rows", _p(src), _p(idx), B, HW, C, R, _p(out), _stream())
    return out


def aabb_intersect(aabb_min: Tensor, aabb_max: Tensor, ray_o: Tensor, ray_d: Tensor):
    _need_cuda(aabb_min, aabb_max, ray_o, ray_d)
    ray_o, ray_d = _f32(ray_o), _f32(ray_d)
    B, n, _ = ray_o.shape
    amin, amax = _f32(aabb_min).reshape(-1, 3), _f32(aabb_max).reshape(-1, 3)
    batched = 1 if amin.shape[0] == B and B > 1 else 0
    assert amin.shape[0] in (1, B) and amax.shape[0] == amin.shape[0]
    t_near = torch.empty(B, n, device=ray_o.device, dtype=torch.float32)
    t_far = torch.empty_like(t_near)
    valid = torch.empty(B, n, device=ray_o.device, dtype=torch.uint8)
    _C.call("tp_aabb_intersect", _p(amin), _p(amax), batched, _p(ray_o), _p(ray_d), B, n, _p(t_near), _p(t_far),
            _p(valid), _stream())
    return t_near, t_far, valid.bool()


def sample_depth(z_near: Tensor, z_far: Tensor, N: int, rand: Optional[Tensor] = None, stratified: bool = True,
                 seed: Optional[int] = None) -> Tensor:
    """[B,R] bounds -> [B,R,N,1] depths.  rand: the [B,R,N,1] torch.rand draw (parity mode); with
    stratified and no rand the jitter comes from the in-kernel Philox stream keyed by `seed`."""
    _need_cuda(z_near, z_far, rand)
    z_near, z_far = _f32(z_near), _f32(z_far)
    B, R = z_near.shape
    out = torch.empty(B, R, N, 1, device=z_near.device, dtype=torch.float32)
    if not stratified:
        mode, rand_t = 1, None
    elif rand is not None:
        mode, rand_t = 0, _f32(rand)
        assert rand_t.numel() == B * R * N
    else:
        mode, rand_t = 2, None
    _C.call("tp_sample_depth", _p(z_near), _p(z_far), _p(rand_t), B * R, N, mode, int(seed or 0), _p(out), _stream())
    return out


def box_range(kinv: Tensor, pose_inv: Tensor, H: int, W: int, aabb_min: Tensor, aabb_max: Tensor,
              bg_near: float, bg_far: float, want_valid: bool = False):
    _need_cuda(kinv, pose_inv, aabb_min, aabb_max)
    kinv, pose_inv = _f32(kinv), _f32(pose_inv)
    B = kinv.shape[0]
    amin, amax = _f32(aabb_min).reshape(-1, 3), _f32(aabb_max).reshape(-1, 3)
    batched = 1 if amin.shape[0] == B and B > 1 else 0
    zn = torch.empty(B, H * W, device=kinv.device, dtype=torch.float32)
    zf = torch.empty_like(zn)
    valid = torch.empty(B, H * W, device=kinv.device, dtype=torch.uint8) if want_valid else None
    _C.call("tp_box_range", _p(kinv), _p(pose_inv), B, H, W, _p(amin), _p(amax), batched, bg_near, bg_far, _p(zn),
            _p(zf), _p(valid), _stream())
    return (zn, zf, valid.bool()) if want_valid else (zn, zf)


def depth_guided_range(depth: Tensor, bg_near: float, bg_far: float):
    _need_cuda(depth)
    depth = _f32(depth)
    zn, zf = torch.empty_like(depth), torch.empty_like(depth)
    _C.call("tp_depth_guided_range", _p(depth), depth.numel(), bg_near, bg_far, _p(zn), _p(zf), _stream())
    return zn, zf


def normal_from_depth(kinv: Tensor, pose_inv: Tensor, depth: Tensor) -> Tensor:
    _need_cuda(kinv, pose_inv, depth)
    kinv, pose_inv, depth = _f32(kinv), _f32(pose_inv), _f32(depth)
    B, H, W = depth.shape
    out = torch.empty(B, 3, H, W, device=depth.device, dtype=torch.float32)
    _C.call("tp_normal_from_depth", _p(kinv), _p(pose_inv), _p(depth), B, H, W, _p(out), _stream())
    return out


def points_from_depth(center: Tensor, ray: Tensor, depth: Tensor) -> Tensor:
    """x = c + ray*d for [B,R,N,1] depths (camera.py:317-322): the L=0 case of the point encoder."""
    _need_cuda(center, ray, depth)
    center, ray, depth = _f32(center), _f32(ray), _f32(depth)
    B, R, N = depth.shape[:3]
    out = torch.empty(B, R, N, 3, device=depth.device, dtype=torch.float32)
    _C.call("tp_points_encode", _p(center), _p(ray), _p(depth), B * R * N, N, 0, _p(out), 3, _stream())
    return out


# ------------------------------------------------------------------------------------------------- composite


class CompositeSTL(torch.autograd.Function):
    """NeRF.composite of layers/nerf_static_transient_light.py:168-212 (11 outputs, reference order)."""

    @staticmethod
    def forward(ctx, ray, rgb, density, depth, uncert, min_uncert):
        _need_cuda(ray, rgb, density, depth, uncert)
        ctx.set_materialize_grads(False)      # unused outputs reach the kernel as NULL instead of zero-filled tensors
        ray_c, rgb_c, den_c, dep_c, unc_c = _f32(ray), _f32(rgb), _f32(density), _f32(depth), _f32(uncert)
        B, R, N = den_c.shape[:3]
        dev = ray_c.device
        o3 = [torch.empty(B, R, 3, device=dev) for _ in range(3)]
        o1 = [torch.empty(B, R, 1, device=dev) for _ in range(5)]      # depth, op, op_s, op_t, uncert
        prob = torch.empty(B, R, N, 1, device=dev)
        a_s = torch.empty(B, R, N, device=dev)
        a_t = torch.empty(B, R, N, device=dev)
        _C.call("tp_composite_stl_forward", _p(ray_c), _p(rgb_c), _p(den_c), _p(dep_c), _p(unc_c), B * R, N,
                float(min_uncert), _p(o3[0]), _p(o3[1]), _p(o3[2]), _p(o1[0]), _p(o1[1]), _p(o1[2]), _p(o1[3]),
                _p(prob), _p(o1[4]), _p(a_s), _p(a_t), _stream())
        ctx.save_for_backward(ray_c, rgb_c, den_c, dep_c, unc_c)
        ctx.mark_non_differentiable()
        return (o3[0], o3[1], o3[2], o1[0], o1[1], o1[2], o1[3], prob, o1[4], a_s, a_t)

    @staticmethod
    def backward(ctx, g_rgb, g_rgb_s, g_rgb_t, g_depth, g_op, g_op_s, g_op_t, g_prob, g_unc, g_as, g_at):
        ray, rgb, den, dep, unc = ctx.saved_tensors
        B, R, N = den.shape[:3]
        gs = [_f32(g) for g in (g_rgb, g_rgb_s, g_rgb_t, g_depth, g_op, g_op_s, g_op_t, g_prob, g_unc, g_as, g_at)]
        d_rgb, d_den, d_unc = torch.empty_like(rgb), torch.empty_like(den), torch.empty_like(unc)
        _C.call("tp_composite_stl_backward", _p(ray), _p(rgb), _p(den), _p(dep), _p(unc), B * R, N,
                *[_p(g) for g in gs], _p(d_rgb), _p(d_den), _p(d_unc), _stream())
        return None, d_rgb, d_den, None, d_unc, None


class CompositePlain(torch.autograd.Function):
    """NeRF.composite of layers/nerf.py:117-136."""

    @staticmethod
    def forward(ctx, ray, rgb, density, depth, bgcolor):
        _need_cuda(ray, rgb, density, depth)
        ctx.set_materialize_grads(False)
        ray_c, rgb_c, den_c, dep_c = _f32(ray), _f32(rgb), _f32(density), _f32(depth)
        B, R, N = den_c.shape[:3]
        dev = ray_c.device
        o_rgb = torch.empty(B, R, 3, device=dev)
        o_depth = torch.empty(B, R, 1, device=dev)
        o_op = torch.empty(B, R, 1, device=dev)
        prob = torch.empty(B, R, N, 1, device=dev)
        use_bg = 0 if bgcolor is None else 1
        ctx.bg = (use_bg, float(bgcolor or 0.0))
        _C.call("tp_composite_plain_forward", _p(ray_c), _p(rgb_c), _p(den_c), _p(dep_c), B * R, N, use_bg,
                ctx.bg[1], _p(o_rgb), _p(o_depth), _p(o_op), _p(prob), _stream())
        ctx.save_for_backward(ray_c, rgb_c, den_c, dep_c)
        return o_rgb, o_depth, o_op, prob

    @staticmethod
    def backward(ctx, g_rgb, g_depth, g_op, g_prob):
        ray, rgb, den, dep = ctx.saved_tensors
        B, R, N = den.shape[:3]
        d_rgb, d_den = torch.empty_like(rgb), torch.empty_like(den)
        _C.call("tp_composite_plain_backward", _p(ray), _p(rgb), _p(den), _p(dep), B * R, N, ctx.bg[0], ctx.bg[1],
                _p(_f32(g_rgb)), _p(_f32(g_depth)), _p(_f32(g_op)), _p(_f32(g_prob)), _p(d_rgb), _p(d_den), _stream())
        return None, d_rgb, d_den, None, None


# ------------------------------------------------------------------------------------------------- fused losses


class PatchLoss(torch.autograd.Function):
    """Ray-wise terms of Graph.compute_loss(train_step='nerf') + Model.summarize_loss (model/nerf_adapt_st_gan.py:712-763,
    model/base.py:145-157): patch gather of image / mask, the three loss terms, `all`, and the backward seeds, in two
    launches (csrc/loss.cu).  weights: log10 loss weights (render, uncert, trans_reg); None switches a term off.
    Returns (losses[4] = render, uncert, trans_reg, all; image_sample [B,3,h,w]; mask_sample [B,1,h,w])."""

    @staticmethod
    def forward(ctx, rgb, uncert, density, image, obj_mask, coords, weights):
        _need_cuda(rgb, uncert, image, obj_mask, coords)
        B, h, w, _ = coords.shape
        R = h * w
        H, W = image.shape[-2:]
        rgb_c, unc_c = _f32(rgb.detach()), _f32(uncert.detach())
        den_c = _f32(density.detach()) if density is not None else None
        N = den_c.shape[2] if den_c is not None else 0
        dev = rgb_c.device
        terms, lin = 0, []
        for i, wgt in enumerate(weights):
            terms |= (1 << i) if wgt is not None else 0
            lin.append(10 ** float(wgt) if wgt is not None else 0.0)
        if den_c is None:
            terms &= ~4
        img_s = torch.empty(B, 3, h, w, device=dev)
        mask_s = torch.empty(B, 1, h, w, device=dev)
        losses = torch.empty(4, device=dev)
        ws = torch.empty(_C.load().tp_patch_loss_workspace(), device=dev)
        _C.call("tp_patch_loss", _p(_f32(image)), _p(_f32(obj_mask)), _p(_f32(coords)), B, R, H, W, _p(rgb_c), _p(unc_c),
                _p(den_c), N, lin[0], lin[1], lin[2], terms, _p(img_s), _p(mask_s), _p(losses), None, None, None, _p(ws),
                ws.numel(), _stream())
        ctx.saved = (rgb_c, unc_c, img_s, mask_s, ws)
        ctx.meta = (B, R, N, lin, terms, den_c is not None and density.requires_grad, den_c.shape if den_c is not None else None)
        ctx.mark_non_differentiable(img_s, mask_s)
        return losses, img_s, mask_s

    @staticmethod
    def backward(ctx, g_losses, _gi, _gm):
        """All four scalars are differentiable: the seeds are formed on the device from the upstream gradient vector, so
        `losses[3].backward()`, the reference's `summarize_loss(...).all.backward()` and any re-weighting of the individual
        terms give the right gradients (no host sync)."""
        rgb_c, unc_c, img_s, mask_s, ws = ctx.saved
        ctx.saved = None
        B, R, N, lin, terms, want_den, den_shape = ctx.meta
        g = _f32(g_losses)
        g_rgb, g_unc = torch.empty_like(rgb_c), torch.empty_like(unc_c)
        g_den = torch.empty(den_shape, device=rgb_c.device) if want_den else None
        _C.call("tp_patch_loss_backward", _p(g), _p(img_s), _p(mask_s), B, R, _p(rgb_c), _p(unc_c), N, lin[0], lin[1], lin[2],
                terms, _p(g_rgb), _p(g_unc), _p(g_den), _p(ws), ws.numel(), _stream())
        return g_rgb, g_unc, g_den, None, None, None, None


class LatentRows(torch.autograd.Function):
    """(latent_vars_trans.weight[idx], latent_vars_light.weight[idx]) of model/nerf_adapt_st_gan.py:589-603 in one launch, with
    the dense table gradients formed by one deterministic kernel (torch's index backward: ~14 launches per table)."""

    @staticmethod
    def forward(ctx, table_a, table_b, idx):
        _need_cuda(table_a, table_b, idx)
        ta, tb = _f32(table_a.detach()), _f32(table_b.detach())
        idx_c = idx.detach().to(torch.int64).reshape(-1).contiguous()
        B = idx_c.numel()
        oa = torch.empty(B, ta.shape[1], device=ta.device)
        ob = torch.empty(B, tb.shape[1], device=tb.device)
        _C.call("tp_latent_rows", _p(ta), ta.shape[1], _p(tb), tb.shape[1], _p(idx_c), B, _p(oa), _p(ob), _stream())
        ctx.idx, ctx.shapes = idx_c, (ta.shape, tb.shape)
        return oa, ob

    @staticmethod
    def backward(ctx, ga, gb):
        (ra, ca), (rb, cb) = ctx.shapes
        dev = ctx.idx.device
        B = ctx.idx.numel()
        ga = _f32(ga) if ga is not None else torch.zeros(B, ca, device=dev)
        gb = _f32(gb) if gb is not None else torch.zeros(B, cb, device=dev)
        da, db = torch.empty(ra, ca, device=dev), torch.empty(rb, cb, device=dev)
        _C.call("tp_latent_rows_backward", _p(ga), ca, ra, _p(gb), cb, rb, _p(ctx.idx), B, _p(da), _p(db), _stream())
        return da, db, None


# ------------------------------------------------------------------------------------------------- fp32 MLP layers

Seg = Tuple[Tensor, int, int]   # (tensor [rows, ld], group, cols)


def _seg_arrays(segs: Sequence[Seg]):
    n = len(segs)
    ptrs = (ctypes.c_void_p * n)(*[s[0].data_ptr() for s in segs])
    lds = (ctypes.c_int64 * n)(*[s[0].stride(0) for s in segs])
    groups = (ctypes.c_int64 * n)(*[int(s[1]) for s in segs])
    cols = (ctypes.c_int32 * n)(*[int(s[2]) for s in segs])
    return ptrs, lds, groups, cols, n


def linear_forward(segs: Sequence[Seg], W: Tensor, bias: Optional[Tensor], S: int, act: int, Y: Tensor, ldy: int,
                   aux0: Optional[Tensor] = None, aux1: Optional[Tensor] = None, w_row0: int = 0,
                   n_out: Optional[int] = None):
    ptrs, lds, groups, cols, n = _seg_arrays(segs)
    n_out = W.shape[0] - w_row0 if n_out is None else n_out
    Wp = ctypes.c_void_p(W.data_ptr() + 4 * w_row0 * W.stride(0))
    bp = ctypes.c_void_p(bias.data_ptr() + 4 * w_row0) if bias is not None else None
    _C.call("tp_linear_forward", ptrs, lds, groups, cols, n, Wp, W.stride(0), bp, S, n_out, act, _p(Y), ldy,
            _p(aux0), _p(aux1), _stream())


def linear_backward_input(dY: Tensor, W: Tensor, S: int, K1: int, xact: Optional[Tensor], w_col0: int = 0) -> Tensor:
    dX = torch.empty(S, K1, device=dY.device, dtype=torch.float32)
    Wp = ctypes.c_void_p(W.data_ptr() + 4 * w_col0)
    _C.call("tp_linear_backward_input", _p(dY), dY.stride(0), Wp, W.stride(0), S, dY.shape[1], K1, _p(xact),
            xact.stride(0) if xact is not None else 0, _p(dX), K1, _stream())
    return dX


def linear_backward_weight(dY: Tensor, segs: Sequence[Seg], S: int, want_bias: bool = True):
    ptrs, lds, groups, cols, n = _seg_arrays(segs)
    Nout = dY.shape[1]
    K = sum(int(s[2]) for s in segs)
    lib = _C.load()
    ws_n = lib.tp_linear_backward_weight_workspace(S, Nout, K)
    ws = torch.empty(ws_n, device=dY.device, dtype=torch.float32)
    dW = torch.empty(Nout, K, device=dY.device, dtype=torch.float32)
    db = torch.empty(Nout, device=dY.device, dtype=torch.float32) if want_bias else None
    _C.call("tp_linear_backward_weight", _p(dY), dY.stride(0), ptrs, lds, groups, cols, n, S, Nout, _p(dW), _p(db), 0,
            _p(ws), ws_n, _stream())
    return dW, db


def group_colsum(dY: Tensor, S: int, group: int) -> Tensor:
    Nout = dY.shape[1]
    G = (S + group - 1) // group
    slices = min(256, (group + 511) // 512)
    ws = torch.empty(slices * G * Nout, device=dY.device, dtype=torch.float32)
    out = torch.empty(G, Nout, device=dY.device, dtype=torch.float32)
    _C.call("tp_group_colsum", _p(dY), dY.stride(0), S, group, Nout, _p(out), _p(ws), ws.numel(), _stream())
    return out


def points_encode(center: Tensor, ray: Tensor, depth: Tensor, L: int) -> Tensor:
    S = depth.numel()
    N = depth.shape[2]
    width = 3 + 6 * L
    enc = torch.empty(S, width + (width & 1), device=depth.device, dtype=torch.float32)
    _C.call("tp_points_encode", _p(center), _p(ray), _p(depth), S, N, L, _p(enc), enc.stride(0), _stream())
    return enc


def positional_encode(x: Tensor, L: int) -> Tensor:
    """[S,3] -> [S, 3+6L(+pad)] rows [x, enc(x)]."""
    S = x.shape[0]
    width = 3 + 6 * L
    enc = torch.empty(S, width + (width & 1), device=x.device, dtype=torch.float32)
    _C.call("tp_positional_encode", _p(x), S, L, _p(enc), enc.stride(0), _stream())
    return enc


def view_encode(ray: Tensor, L: int, normalize: bool) -> Tensor:
    R = ray.shape[0]
    width = 3 + 6 * L
    enc = torch.empty(R, width + (width & 1), device=ray.device, dtype=torch.float32)
    _C.call("tp_view_encode", _p(ray), R, L, 1 if normalize else 0, _p(enc), enc.stride(0), _stream())
    return enc
