"""Drop-in for tools/ray_sampler.py (RaySampler.get_rays / get_bounds / get_image)."""
from __future__ import annotations

import torch

from .. import camera, ops


class RaySampler(object):
    def __init__(self, opt, intrinsics=None):
        self.intrinsics = intrinsics

    @staticmethod
    def _hw(opt, H, W):
        return (opt.H, opt.W) if (H is None and W is None) else (H, W)

    @staticmethod
    def get_image(opt, coords, image, H=None, W=None):
        """tools/ray_sampler.py:12-21: bilinear, align_corners=True."""
        with torch.no_grad():
            return ops.grid_sample_bilinear(image, coords)

    @staticmethod
    def get_bounds(opt, coords, z_near, z_far, H=None, W=None):
        """tools/ray_sampler.py:23-37 -> ([B,h,w], [B,h,w]); one launch per plane straight from the caller's maps (a stacked copy
        plus two strided views cost four launches)."""
        H, W = RaySampler._hw(opt, H, W)
        with torch.no_grad():
            B = coords.shape[0]
            zn = ops.grid_sample_bilinear(z_near.reshape(B, 1, H, W), coords)
            zf = ops.grid_sample_bilinear(z_far.reshape(B, 1, H, W), coords)
        return zn[:, 0], zf[:, 0]

    @staticmethod
    def get_rays(opt, intrinsics, coords, pose, H=None, W=None, view=None):
        """tools/ray_sampler.py:39-69 -> center, ray [B,h,w,3].  view: precomputed (K^-1, pose^-1), camera.view_or_matrices."""
        H, W = RaySampler._hw(opt, H, W)
        with torch.no_grad():
            kinv, pinv = camera.view_or_matrices(opt, pose, intrinsics, view)
            return ops.patch_rays(kinv, pinv, coords, H, W)
