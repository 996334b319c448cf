"""Drop-in for the ray utilities of camera.py (reference lines cited per function).

Per-image 3x3 / 3x4 algebra (K^-1, pose inversion/composition) stays on the host side as the same torch calls
the reference makes, so the 21 floats per view handed to the kernels carry the reference's bits (SURVEY 8a, a1);
everything per-pixel / per-ray runs in the CUDA library.
"""
from __future__ import annotations

import torch

from . import ops


class Pose:
    """camera.Pose (camera.py:13-61): [...,3,4] poses [R|t]."""

    def __call__(self, R=None, t=None):
        assert R is not None or t is not None
        if R is None:
            t = t if isinstance(t, torch.Tensor) else torch.tensor(t)
            R = torch.eye(3, device=t.device).repeat(*t.shape[:-1], 1, 1)
        elif t is None:
            R = R if isinstance(R, torch.Tensor) else torch.tensor(R)
            t = torch.zeros(R.shape[:-1], device=R.device)
        else:
            R = R if isinstance(R, torch.Tensor) else torch.tensor(R)
            t = t if isinstance(t, torch.Tensor) else torch.tensor(t)
        assert R.shape[:-1] == t.shape and R.shape[-2:] == (3, 3)
        pose = torch.cat([R.float(), t.float()[..., None]], dim=-1)
        assert pose.shape[-2:] == (3, 4)
        return pose

    def invert(self, pose, use_inverse=False):
        R, t = pose[..., :3], pose[..., 3:]
        R_inv = R.inverse() if use_inverse else R.transpose(-1, -2)
        return self(R=R_inv, t=(-R_inv @ t)[..., 0])

    def compose(self, pose_list):
        out = pose_list[0]
        for nxt in pose_list[1:]:
            out = self.compose_pair(out, nxt)
        return out

    def compose_pair(self, pose_a, pose_b):
        R_a, t_a = pose_a[..., :3], pose_a[..., 3:]
        R_b, t_b = pose_b[..., :3], pose_b[..., 3:]
        return self(R=R_b @ R_a, t=(R_b @ t_a + t_b)[..., 0])


pose = Pose()


def to_hom(X):
    return torch.cat([X, torch.ones_like(X[..., :1])], dim=-1)       # camera.py:250-253


def world2cam(X, pose_):
    return to_hom(X) @ pose_.transpose(-1, -2)                         # camera.py:257-259


def cam2img(X, cam_intr):
    return X @ cam_intr.transpose(-1, -2)                              # camera.py:262-263


def img2cam(X, cam_intr):
    return X @ cam_intr.inverse().transpose(-1, -2)                    # camera.py:266-267


def cam2world(X, pose_):
    return to_hom(X) @ Pose().invert(pose_).transpose(-1, -2)          # camera.py:270-277


HOST_MATRICES = False   # True: invert K / the pose on the CPU (LAPACK bits == the CPU reference), costs one sync


def view_matrices(pose_, intr, one_launch=False):
    """(K^-1 [B,3,3], pose^-1 [B,3,4]) -- the per-view constants every ray kernel takes (camera.py:267,270-277).
    By default they are computed where `pose_` lives with the torch calls the reference makes (no host sync; same bits as the
    reference on the same device).  With HOST_MATRICES the two tiny inverses run on the CPU exactly as the CPU reference does,
    which makes generated rays bit-identical to it.  one_launch: tp_view_matrices instead of torch's ~20 tiny launches
    (~1.3 ms per call): K^-1 then differs from torch's LU result in the last bits, so only the bf16 path (1e-2 contract) uses it."""
    if one_launch and pose_.is_cuda and not HOST_MATRICES:
        B = pose_.shape[0]
        intr_c, pose_c = ops._f32(intr.detach()).reshape(B, 9), ops._f32(pose_.detach()).reshape(B, 12)
        kinv = torch.empty(B, 3, 3, device=pose_.device)
        pinv = torch.empty(B, 3, 4, device=pose_.device)
        ops._C.call("tp_view_matrices", ops._p(intr_c), ops._p(pose_c), B, ops._p(kinv), ops._p(pinv), ops._stream())
        return kinv, pinv
    if HOST_MATRICES and pose_.is_cuda:
        from .train_graph import refuse_capture
        refuse_capture("camera.HOST_MATRICES", "the CPU inversion synchronises; compute the matrices eagerly with "
                       "view_matrices() and pass them to Graph.render as a static `view=(kinv, pinv)`")
        dev = pose_.device
        return (intr.detach().cpu().float().inverse().contiguous().to(dev),
                Pose().invert(pose_.detach().cpu().float()).contiguous().to(dev))
    # inv_ex == inverse() bit for bit, minus its error check: that check reads `info` back and would stall the launch
    # queue once per frame (the calibration matrix is never singular; a singular one yields inf/nan rays as before)
    return torch.linalg.inv_ex(intr.float())[0].contiguous(), Pose().invert(pose_.float()).contiguous()


def one_launch_matrices(opt) -> bool:
    """opt.b200.view_matrices: 'kernel' (tp_view_matrices, one launch) | 'torch' (the reference's calls, its bits).  Default:
    'torch' in the fp32 parity mode, 'kernel' wherever the MLP may take the bf16 tensor-core path (1e-2 contract)."""
    from .layers import _common
    v = _common.b200_option(opt, "view_matrices")
    if v is None:
        return _common.mlp_precision(opt) != "fp32"
    if v not in ("kernel", "torch"):
        raise ValueError(f"unknown opt.b200.view_matrices {v!r}")
    return v == "kernel"


def view_or_matrices(opt, pose_, intr, view=None):
    """`view` = (K^-1 [B,3,3], pose^-1 [B,3,4]) computed by the caller (view_matrices, e.g. eagerly outside a captured CUDA graph)
    or None: view_matrices(pose_, intr) as opt selects."""
    if view is not None:
        kinv, pinv = view
        B = pose_.shape[0]
        if tuple(kinv.shape) != (B, 3, 3) or tuple(pinv.shape) != (B, 3, 4):
            raise ValueError(f"view matrices must be [{B},3,3] and [{B},3,4]; got {tuple(kinv.shape)} and {tuple(pinv.shape)}")
        return kinv, pinv
    return view_matrices(pose_, intr, one_launch=one_launch_matrices(opt))


def get_center_and_ray(opt, pose_, intr=None, H=None, W=None, ray_idx=None, view=None):
    """camera.get_center_and_ray (camera.py:292-314).  Extra `ray_idx` [B,R] fuses Graph.ray_batch_sample
    (model/nerf_adapt_st_gan.py:702-710) so only the requested pixels are ever generated; extra `view` = precomputed
    (K^-1, pose^-1), see view_or_matrices."""
    assert opt.camera.model == "perspective"
    if H is None and W is None:
        H, W = opt.H, opt.W
    kinv, pinv = view_or_matrices(opt, pose_, intr, view)
    return ops.raygen(kinv, pinv, H, W, 0.5, ray_idx)


def get_3D_points_from_depth(opt, center, ray, depth, multi_samples=False):
    """camera.py:317-322."""
    if multi_samples:
        return ops.points_from_depth(center, ray, depth)
    B, R = center.shape[:2]
    return ops.points_from_depth(center, ray, depth.reshape(B, R, 1, 1)).view(B, R, 3)


def aabb_ray_intersection(aabb_min, aabb_max, ray_o, ray_d):
    """camera.py:415-433 -> t_near [B,HW], t_far [B,HW], valid [B,HW] bool (bit-exact)."""
    return ops.aabb_intersect(aabb_min, aabb_max, ray_o, ray_d)


def enlarge_diagonal(aabb_min, aabb_max, alpha=0.25):
    """camera.py:436-440 (6 floats; host)."""
    d = aabb_max - aabb_min
    return aabb_min - d * alpha / 2, aabb_max + d * alpha / 2
