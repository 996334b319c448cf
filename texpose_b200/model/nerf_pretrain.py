"""Drop-in for the render path of model/nerf_pretrain.py `Graph` (reference :449-466, :497-527, :588-660, :707-728).

SURVEY.md 8 keeps the pre-training engine out of scope but asks for its `Graph.render` to keep working: it is the
same hot path (rays -> stratified depths -> plain `layers/nerf.py` MLP -> single-chain compositing) and lands on the
same kernels.  Mirrored here: forward / render / render_by_slices / sample_depth / ray_batch_sample / get_ray_idx and
the three pre-training losses (:529-586; small reductions over [B,R,.], plain torch ops -- not kernels of the path).

Deliberate differences, results identical:
  * only the requested rays are generated (the reference builds the full H*W frame and gathers, :596-604), and a
    contiguous slice is passed to the kernels as a range instead of an index tensor;
  * render_by_slices takes as many rays per launch as the MLP path has room for (`Graph._slice_rays`), not
    opt.nerf.rand_rays, so a 480x640 evaluation frame is one launch of the tcgen05 kernel instead of 150 chunks;
  * the host-syncing NaN retry (:598) runs only under opt.b200.nan_guard; tensors follow `opt.device`;
  * opt.nerf.fine_sampling (a second NeRF, never rendered by the reference's own render()) builds `nerf_fine` so that
    checkpoints load, and is otherwise unused -- as in the reference.
"""
from __future__ import annotations

import torch

from .. import camera, ops
from ..config import AttrDict
from ..layers.nerf import NeRF
from ..layers._common import given_keywords as _given
from ..train_graph import refuse_capture


class Graph(torch.nn.Module):
    RENDER_KEYS = ("rgb", "depth", "opacity", "density")      # what _render_fused can produce

    def __init__(self, opt):
        super().__init__()
        self.nerf = NeRF(opt)
        if opt.nerf.get("fine_sampling"):
            self.nerf_fine = NeRF(opt)

    @staticmethod
    def _b200(opt, key, default=None):
        b = opt.get("b200") if hasattr(opt, "get") else None
        return b.get(key, default) if b else default

    @staticmethod
    def ray_batch_sample(ray_identity, ray_idx):
        """model/nerf_pretrain.py:457-465: rows `ray_idx[b]` of every batch entry."""
        assert ray_identity.shape[0] == ray_idx.shape[0]
        return ops.gather_rows(ray_identity, ray_idx)

    @staticmethod
    def get_ray_idx(opt, var):
        """model/nerf_pretrain.py:497-503: one random subset of the frame, shared by every view of the batch."""
        batch_size = len(var.idx)
        per_view = opt.nerf.rand_rays // batch_size
        var.ray_idx = torch.randperm(opt.H * opt.W, device=opt.device)[:per_view].repeat(batch_size, 1)
        return var

    @staticmethod
    def get_pose(opt, var, mode=None):
        source = dict(gt=var.pose, predicted=var.pose_init if "pose_init" in var else var.pose)
        return source[opt.data.pose_source] if mode == "train" else source["gt"]

    def forward(self, opt, var, mode=None):
        """model/nerf_pretrain.py:513-536."""
        pose = self.get_pose(opt, var, mode=mode)
        depth_range = (var.z_near[:, :, None], var.z_far[:, :, None])       # [B,HW,1] each
        if opt.nerf.rand_rays and mode in ("train", "test-optim"):
            var = self.get_ray_idx(opt, var)
            ret = self.render(opt, pose, intr=var.intr, ray_idx=var.ray_idx, depth_range=depth_range, mode=mode)
        else:
            ret = self.render_by_slices(opt, pose, intr=var.intr, depth_range=depth_range,
                                        object_mask=var.get("obj_mask"), mode=mode)
        var.update(ret)
        return var

    # ---------------------------------------------------------------- the hot path
    def render(self, opt, pose, intr=None, ray_idx=None, depth_range=None, mode=None, view=None):
        """model/nerf_pretrain.py:588-627 -> rgb [B,R,3], depth [B,R,1], opacity [B,R,1].  view: (K^-1, pose^-1) computed by the
        caller (camera.view_matrices), e.g. eagerly outside a captured training step; None computes them here."""
        if opt.camera.ndc:
            raise NotImplementedError("camera.ndc is false in every reference yaml; not implemented")
        B = len(pose)
        if ray_idx is None:         # the novel-view caller (:421-422) passes no ray list: the whole frame
            ray_idx = range(0, opt.H * opt.W)
        if isinstance(ray_idx, range):
            ray_idx = torch.arange(ray_idx.start, ray_idx.stop, device=pose.device)[None].expand(B, -1)
        center, ray = camera.get_center_and_ray(opt, pose, intr=intr, ray_idx=ray_idx, **_given(view=view))
        if self._b200(opt, "nan_guard", False):
            refuse_capture("opt.b200.nan_guard", "the NaN check reads the rays back to the host")
            if bool(ray.isnan().any()):
                raise FloatingPointError("NaN in generated rays")
        depth_min, depth_max = depth_range
        zn = self.ray_batch_sample(depth_min, ray_idx).squeeze(-1)
        zf = self.ray_batch_sample(depth_max, ray_idx).squeeze(-1)
        depth_samples = self.sample_depth(opt, B, (zn, zf), num_rays=ray.shape[1])       # [B,R,N,1]
        rgb_samples, density_samples = self.nerf.forward_samples(opt, center, ray, depth_samples, mode=mode)
        rgb, depth, opacity, _prob = self.nerf.composite(opt, ray, rgb_samples, density_samples, depth_samples)
        return AttrDict(rgb=rgb, depth=depth, opacity=opacity)

    def _render_fused(self, opt, pose, intr, ray_idx, depth_range, sample_idx=None, mode=None, want=None, out_ptrs=None):
        """render() as ONE launch of the staged kernel (NeRF.render_rays): rays, depths and compositing in-kernel.  Same signature
        as the adaptation Graph's, so that parallel.FrameGather renders either engine's frame; sample_idx is unused (no latents).
        ray_idx: [B,R] tensor, or a `range` = contiguous row block.  The view matrices and the jitter draw are render()'s, so a
        seeded call makes the same rays and depths."""
        B = len(pose)
        HW = opt.H * opt.W
        kinv, pinv = camera.view_matrices(pose, intr, one_launch=camera.one_launch_matrices(opt))
        zn, zf = depth_range[0].reshape(B, HW), depth_range[1].reshape(B, HW)
        if isinstance(ray_idx, range):
            assert ray_idx.step == 1
            idx_t, ray0, R = None, ray_idx.start, len(ray_idx)
        else:
            idx_t, ray0, R = ray_idx, 0, ray_idx.shape[1]
        rand, seed = None, 0
        if opt.nerf.sample_stratified:
            if self._b200(opt, "rng", "torch") == "philox":
                refuse_capture("opt.b200.rng = 'philox'", "its seed is drawn on the host; use rng = 'torch'")
                seed = int(torch.randint(0, 2 ** 62, (1,)).item())
            else:
                rand = torch.rand(B, R, opt.nerf.sample_intvs, 1, device=pose.device)      # sample_depth's draw (:707-728)
        ret = self.nerf.render_rays(opt, kinv, pinv, idx_t, ray0, R, zn, zf, mode=mode, rand=rand, seed=seed, want=want,
                                    out_ptrs=out_ptrs)
        return AttrDict(ret)

    def _slice_rays(self, opt):
        """Rays per launch: the tensor-core kernels keep activations on chip, the fp32 SIMT path is bounded by its
        [S,256] activation buffers."""
        user = self._b200(opt, "slice_rays")
        if user:
            return int(user)
        on_tc = self.nerf.uses_tensor_cores(opt) or self.nerf.uses_split_tensor_cores(opt)
        budget = (1 << 26) if on_tc else (1 << 21)
        return max(int(opt.nerf.rand_rays or 2048), budget // opt.nerf.sample_intvs)

    def render_by_slices(self, opt, pose, intr=None, depth_range=None, object_mask=None, mode=None):
        """model/nerf_pretrain.py:629-660: every pixel of the frame (the reference computes the object-pixel list and
        never uses it; `object_mask` is accepted for the same call signature)."""
        HW = opt.H * opt.W
        step = self._slice_rays(opt)
        parts = dict(rgb=[], depth=[], opacity=[])
        for c in range(0, HW, step):
            ret = self.render(opt, pose, intr=intr, ray_idx=range(c, min(c + step, HW)), depth_range=depth_range,
                              mode=mode)
            for k in parts:
                parts[k].append(ret[k])
        return AttrDict({k: (v[0] if len(v) == 1 else torch.cat(v, dim=1)) for k, v in parts.items()})

    def sample_depth(self, opt, batch_size, depth_range, num_rays=None):
        """model/nerf_pretrain.py:707-728.  Same torch.rand draw as the reference, so seeded runs agree."""
        zn, zf = depth_range
        num_rays = num_rays or opt.H * opt.W
        zn, zf = zn.reshape(batch_size, num_rays), zf.reshape(batch_size, num_rays)
        if opt.nerf.depth.param != "metric":
            raise NotImplementedError("nerf.depth.param is 'metric' in every reference yaml")
        N = opt.nerf.sample_intvs
        if not opt.nerf.sample_stratified:
            return ops.sample_depth(zn, zf, N, stratified=False)
        rand = torch.rand(batch_size, num_rays, N, 1, device=zn.device)
        return ops.sample_depth(zn, zf, N, rand=rand)

    # ---------------------------------------------------------------- pre-training losses (host-side torch reductions)
    @staticmethod
    def MSE_loss(pred, label=0):
        return ((pred.contiguous() - label) ** 2).mean()

    @staticmethod
    def scale_invariant_depth_loss(depth_pred, depth_target, mask=None):
        """model/base.py:223-231: 1 - min / (max + 1e-5), averaged over the mask."""
        lo, hi = torch.minimum(depth_pred, depth_target), torch.maximum(depth_pred, depth_target)
        loss = 1 - lo / (hi + 1e-5)
        if mask is not None:
            mask = mask.float()
            loss = (loss * mask).sum() / (mask.sum() + 1e-5)
        return loss

    def compute_loss(self, opt, var, mode=None):
        """model/nerf_pretrain.py:538-586: mask / depth / render terms on the sampled rays."""
        loss = AttrDict()
        B, HW = len(var.idx), opt.H * opt.W
        sampled = bool(opt.nerf.rand_rays) and mode in ("train", "test-optim")

        def per_ray(t, gather):
            t = t.reshape(B, HW, -1)
            return self.ray_batch_sample(t, var.ray_idx) if gather else t

        image = per_ray(var.image.view(B, 3, HW).permute(0, 2, 1).contiguous(), sampled)
        obj = var.erode_mask if opt.data.get("erode_mask_loss") else var.obj_mask
        if opt.loss_weight.mask is not None:
            loss.mask = self.MSE_loss(per_ray(var.obj_mask.float(), sampled), var.opacity)
        if opt.loss_weight.depth is not None:
            in_train = mode == "train"
            loss.depth = self.scale_invariant_depth_loss(var.depth, per_ray(var.depth_gt, in_train),
                                                         per_ray(obj, in_train))
        if opt.loss_weight.render is not None:
            if opt.nerf.get("mask_obj"):
                m = per_ray(obj, mode == "train").float()
                loss.render = (m * (image - var.rgb) ** 2).sum() / (m.sum() + 1e-5)
            else:
                loss.render = self.MSE_loss(var.rgb, image)
        return loss
