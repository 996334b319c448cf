"""Drop-in for the render path of model/nerf_adapt_st_gan.py `Graph` (reference lines :464-514, :547-710).

Only the hot path is mirrored: nerf_forward / render / render_by_slices / sample_depth / ray_batch_sample.
The engine around it (Model, discriminator, perceptual losses, visualisation) is out of scope (SURVEY.md 8)
and keeps calling these methods unchanged -- see INTEGRATION.md for the patch point.

Differences that are deliberate (B200-first, results identical):
  * eval/val modes generate only the requested rays (the reference rebuilds the full frame for every
    2048-ray chunk, :568) and render a whole frame per launch instead of ~150 Python chunks;
  * the host-syncing NaN retry loop (:554,:569) is dropped (opt.b200.nan_guard restores it);
  * no hard-coded .cuda(): tensors follow `opt.device`.
"""
from __future__ import annotations

import torch

from .. import camera, ops
from ..config import AttrDict
from ..layers.nerf_static_transient_light import NeRF
from ..tools.ray_sampler import RaySampler
from ..tools.patch_sampler import FlexPatchSampler
from ..layers._common import given_keywords as _given
from ..train_graph import refuse_capture


_PHILOX = ("opt.b200.rng = 'philox'", "its seed is drawn on the host; use rng = 'torch'")


def rotation_distance(R1, R2, eps=1e-7):
    """camera.rotation_distance (camera.py:345-350): geodesic angle, used once per eval frame (host logic)."""
    R_diff = R1 @ R2.transpose(-2, -1)
    trace = R_diff[..., 0, 0] + R_diff[..., 1, 1] + R_diff[..., 2, 2]
    return ((trace - 1) / 2).clamp(-1 + eps, 1 - eps).acos_()


class Graph(torch.nn.Module):
    RENDER_KEYS = ("rgb", "rgb_static", "rgb_transient", "depth", "opacity", "opacity_static", "opacity_transient", "uncert",
                   "alpha_static", "alpha_transient", "density")      # what _render_fused can produce

    def __init__(self, opt, n_train_images=None):
        super().__init__()
        self.nerf = NeRF(opt)
        self.ray_sampler = RaySampler(opt)
        # :424 builds FlexPatchSampler(opt, scale_anneal=0.0002) (`opt` lands in random_shift: truthy); the engine keeps
        # `patch_sampler.iterations = self.it` up to date (:185), so min_scale anneals 0.8 -> 0.25 as exp(-it * 2e-4)
        self.patch_sampler = FlexPatchSampler(random_shift=True, random_scale=True, min_scale=0.25, max_scale=1.0,
                                              scale_anneal=0.0002)
        if n_train_images is not None:      # the reference attaches these in Model.build_networks (:56-59)
            self.latent_vars_trans = torch.nn.Embedding(n_train_images, opt.nerf.N_latent_trans)
            torch.nn.init.normal_(self.latent_vars_trans.weight)
            self.latent_vars_light = torch.nn.Embedding(n_train_images, opt.nerf.N_latent_light)
            torch.nn.init.normal_(self.latent_vars_light.weight)

    # ---------------------------------------------------------------- small host-side helpers
    @staticmethod
    def get_pose(opt, var, mode=None):
        source = dict(gt=var.pose, predicted=var.pose_init if "pose_init" in var else var.pose)
        return source[opt.data.pose_source] if mode == "train" else source["gt"]

    @staticmethod
    def _b200(opt, key, default=None):
        b = opt.get("b200") if hasattr(opt, "get") else None
        return b.get(key, default) if b else default

    def get_ray_idx(self, opt, var):
        """model/nerf_adapt_st_gan.py:430-434."""
        coords, scales = self.patch_sampler(nbatch=opt.batch_size, patch_size=opt.patch_size, device=opt.device)
        var.ray_idx = coords
        var.ray_scales = scales
        return var

    def compute_loss(self, opt, var, mode=None, train_step="nerf"):
        """Ray-wise terms of model/nerf_adapt_st_gan.py:712-763 (render / uncert / trans_reg) fused with the patch gather
        (csrc/loss.cu).  Returns the reference's dict -- one differentiable scalar per enabled term and NO `all` key, so an
        unmodified Model.summarize_loss (model/base.py:145-157, which asserts "all" not in loss) accepts it; the backward forms
        the seeds on the device from whatever upstream gradients arrive.  The weighted sum the same pass already computed is
        left in `var.loss_all_fused` for texpose_b200.model.base.summarize_loss (no extra launches, no host sync).  The
        VGG / Lab / GAN terms need the engine's pretrained nets and stay with it (they read var.image_sample /
        var.mask_sample, which are filled here as in the reference)."""
        if train_step != "nerf":
            raise NotImplementedError("discriminator losses stay with the engine (out of the hot path, SURVEY.md 8)")
        lw = opt.loss_weight
        for k in ("mask", "feat", "lab", "gan_nerf", "depth"):
            if lw.get(k) is not None:
                raise NotImplementedError(f"loss_weight.{k}: term is outside the hot path (SURVEY.md 8, out of scope)")
        if not opt.nerf.mask_obj:
            raise NotImplementedError("nerf.mask_obj=False (plain MSE) is not enabled in any yaml of the path")
        if not (opt.nerf.rand_rays and mode in ("train", "test-optim")):
            raise NotImplementedError("full-frame loss (no patch gather) is not on the training path")
        B = len(var.idx)
        image = var.image.contiguous()
        obj_mask = var.obj_mask.contiguous().view(B, opt.H, opt.W)
        weights = (lw.get("render"), lw.get("uncert"), lw.get("trans_reg"))
        losses, img_s, mask_s = ops.PatchLoss.apply(var.rgb, var.uncert, var.density, image, obj_mask, var.ray_idx, weights)
        var.image_sample, var.mask_sample = img_s, mask_s
        if "image_syn" in var and "mask_syn" in var:     # consumed only by the engine's VGG / Lab terms (:719-731)
            F = torch.nn.functional
            var.image_syn_sample = F.grid_sample(var.image_syn.contiguous(), var.ray_idx, mode="bilinear", align_corners=True)
            var.mask_syn_sample = F.grid_sample((var.mask_syn > 0).float().view(B, 1, opt.H, opt.W), var.ray_idx, mode="nearest",
                                                align_corners=False)
        else:
            var.image_syn_sample, var.mask_syn_sample = img_s, mask_s
        loss = AttrDict()
        for i, k in enumerate(("render", "uncert", "trans_reg")):
            if weights[i] is not None:
                loss[k] = losses[i]
        var.loss_all_fused = losses[3]
        return loss

    # ---------------------------------------------------------------- reference interface
    def forward(self, opt, var, mode=None):
        return self.nerf_forward(opt, var, mode=mode)

    def nerf_forward(self, opt, var, mode=None):
        """model/nerf_adapt_st_gan.py:464-514 (the discriminator call of train mode stays with the engine)."""
        pose = self.get_pose(opt, var, mode=mode)
        depth_range = (var.z_near[:, :, None], var.z_far[:, :, None])
        if opt.nerf.rand_rays and mode == "train":
            ret = self.render(opt, pose, intr=var.intr, ray_idx=var.ray_idx, depth_range=depth_range,
                              sample_idx=var.idx, mode=mode)
        elif mode == "val":
            ret = self.render_by_slices(opt, pose, intr=var.intr, depth_range=depth_range, object_mask=var.obj_mask,
                                        sample_idx=None, mode=mode)
        else:
            # latent pick (:489-494): the light latent of one of the N_candidate nearest training poses, chosen by ONE
            # randperm draw as in the reference; evaluated per view so a batch of B > 1 frames works, and left on the device
            R_dist = rotation_distance(var.pose[:, None, :3, :3], var.pose_anchor[None, :, :3, :3])        # [B, N_train]
            k = int(opt.render.N_candidate)
            cand = torch.topk(R_dist, k=k, dim=1, largest=False, sorted=True)[1]                           # [B, k]
            latent_light_idx = cand[:, int(torch.randperm(k)[0])]                                          # [B]
            if len(var.pose) == 1:
                latent_light_idx = latent_light_idx[0]
            ret = self.render_by_slices(opt, pose, intr=var.intr, depth_range=depth_range, object_mask=var.obj_mask,
                                        sample_idx=latent_light_idx, mode=mode)
        var.update(ret)
        return var

    def _latents(self, opt, B, sample_idx, mode, dev):
        """Latent rows of model/nerf_adapt_st_gan.py:589-603, one row per view (a single row is broadcast as the
        reference's `.expand(B, ...)` does, layers/nerf_static_transient_light.py:113,127)."""
        if mode == "train":
            if self.latent_vars_trans.weight.is_cuda and sample_idx.dim() == 1:
                lat_trans, lat_light = ops.LatentRows.apply(self.latent_vars_trans.weight, self.latent_vars_light.weight, sample_idx)
            else:
                lat_trans = self.latent_vars_trans.weight[sample_idx]
                lat_light = self.latent_vars_light.weight[sample_idx]
        elif mode == "val":
            lat_trans = self.latent_vars_trans.weight[0][None]
            lat_light = self.latent_vars_light.weight[0][None]
        else:
            if opt.render.transient == "zero":
                lat_trans = torch.zeros(B, opt.nerf.N_latent_trans, device=dev)
            elif opt.render.transient == "sample":
                lat_trans = self.latent_vars_trans.weight[sample_idx].reshape(-1, opt.nerf.N_latent_trans)
            else:
                raise NotImplementedError
            lat_light = self.latent_vars_light.weight[sample_idx].reshape(-1, opt.nerf.N_latent_light)
        if lat_trans.shape[0] != B or lat_light.shape[0] != B:
            if lat_trans.shape[0] not in (1, B) or lat_light.shape[0] not in (1, B):
                raise ValueError(f"latents must have 1 or {B} rows, got {lat_trans.shape[0]} / {lat_light.shape[0]}")
            lat_trans = lat_trans.expand(B, -1).contiguous()
            lat_light = lat_light.expand(B, -1).contiguous()
        return lat_trans, lat_light

    def _render_fused(self, opt, pose, intr, ray_idx, depth_range, sample_idx, mode, want=None, out_ptrs=None, view=None):
        """model/nerf_adapt_st_gan.py:565-631 as one launch (csrc/mlp_tc.cu, render mode): rays, depths, view-direction bias
        and compositing happen inside the fused kernel.  ray_idx: [B,R] tensor, or a `range` = contiguous row block."""
        B = len(pose)
        HW = opt.H * opt.W
        kinv, pinv = camera.view_or_matrices(opt, pose, intr, view)
        zn, zf = depth_range[0].reshape(B, HW), depth_range[1].reshape(B, HW)
        if isinstance(ray_idx, range):
            assert ray_idx.step == 1
            idx_t, ray0, R = None, ray_idx.start, len(ray_idx)
        else:
            idx_t, ray0, R = ray_idx, 0, ray_idx.shape[1]
        lat_trans, lat_light = self._latents(opt, B, sample_idx, mode, pose.device)
        rand, seed = None, 0
        if opt.nerf.sample_stratified:
            if self._b200(opt, "rng", "torch") == "philox":
                refuse_capture(*_PHILOX)
                seed = int(torch.randint(0, 2 ** 62, (1,)).item())
            else:
                rand = torch.rand(B, R, opt.nerf.sample_intvs, 1, device=pose.device)      # the reference's draw (:690)
        ret = self.nerf.render_rays(opt, kinv, pinv, idx_t, ray0, R, zn, zf, lat_trans, lat_light, mode=mode, rand=rand,
                                    seed=seed, want=want, out_ptrs=out_ptrs)
        return AttrDict(ret)

    def render(self, opt, pose, intr=None, ray_idx=None, depth_range=None, sample_idx=None, mode=None, view=None):
        """model/nerf_adapt_st_gan.py:547-631 -> dict of 11 tensors.  view: (K^-1, pose^-1) computed by the caller
        (camera.view_matrices), e.g. eagerly outside a captured training step; None computes them here."""
        depth_min, depth_max = depth_range
        if opt.camera.ndc:
            raise NotImplementedError("camera.ndc is false in every reference yaml; not implemented")
        if mode != "train" and not self._b200(opt, "nan_guard", False) and self.nerf.fused_render_applies(opt, mode):
            return self._render_fused(opt, pose, intr, ray_idx, depth_range, sample_idx, mode, view=view)
        if isinstance(ray_idx, range):
            ray_idx = torch.arange(ray_idx.start, ray_idx.stop, device=pose.device)[None].expand(len(pose), -1)
        if mode == "train":
            B, h, w, _ = ray_idx.shape
            center, ray = self.ray_sampler.get_rays(opt, intrinsics=intr, coords=ray_idx, pose=pose, **_given(view=view))
            zn, zf = self.ray_sampler.get_bounds(opt, coords=ray_idx, z_near=depth_min, z_far=depth_max)
            center, ray = center.view(B, h * w, 3), ray.view(B, h * w, 3)
            zn, zf = zn.reshape(B, h * w), zf.reshape(B, h * w)
        else:
            B = len(pose)
            center, ray = camera.get_center_and_ray(opt, pose, intr=intr, ray_idx=ray_idx, **_given(view=view))
            zn = self.ray_batch_sample(depth_min, ray_idx).squeeze(-1)
            zf = self.ray_batch_sample(depth_max, ray_idx).squeeze(-1)
        if self._b200(opt, "nan_guard", False):
            refuse_capture("opt.b200.nan_guard", "the NaN check reads the rays back to the host")
            if bool(ray.isnan().any()):
                raise FloatingPointError("NaN in generated rays")
        depth_samples = self.sample_depth(opt, B, (zn, zf), num_rays=ray.shape[1])       # [B,R,N,1]

        lat_trans, lat_light = self._latents(opt, B, sample_idx, mode, ray.device)

        rgb_samples, density_samples, uncert_samples = self.nerf.forward_samples(
            opt, center=center, ray=ray, depth_samples=depth_samples, latent_variable_trans=lat_trans,
            latent_variable_light=lat_light, mode=mode)
        (rgb, rgb_static, rgb_transient, depth, opacity, opacity_static, opacity_transient, prob, uncert,
         alpha_static, alpha_transient) = self.nerf.composite(opt, ray, rgb_samples, density_samples, depth_samples,
                                                              uncert_samples)
        return AttrDict(rgb=rgb, rgb_static=rgb_static, rgb_transient=rgb_transient, opacity=opacity,
                        opacity_static=opacity_static, opacity_transient=opacity_transient, uncert=uncert, depth=depth,
                        alpha_static=alpha_static, alpha_transient=alpha_transient, density=density_samples)

    def _slice_rays(self, opt):
        """Rays per launch.  The fused bf16 kernel keeps activations on chip, so a whole 480x640 frame is one
        launch; the fp32 layer-by-layer path is bounded by its [S,256] activation buffers."""
        user = self._b200(opt, "slice_rays")
        if user:
            return int(user)
        n = opt.nerf.sample_intvs
        budget = (1 << 26) if self.nerf.uses_tensor_cores(opt) else (1 << 21)
        return max(int(opt.nerf.rand_rays or 2048), budget // n)

    def render_by_slices(self, opt, pose, intr=None, depth_range=None, object_mask=None, sample_idx=None, mode=None):
        """model/nerf_adapt_st_gan.py:633-680."""
        HW = opt.H * opt.W
        dev = pose.device
        step = self._slice_rays(opt)
        keys = ["rgb", "rgb_static", "rgb_transient", "opacity", "opacity_static", "opacity_transient", "depth",
                "uncert", "alpha_static", "alpha_transient", "density"]
        if mode == "val":
            parts = {k: [] for k in keys}
            B = len(pose)
            for c in range(0, HW, step):
                ray_idx = range(c, min(c + step, HW))       # contiguous block: no index tensor (the fused launch takes ray0 + r)
                ret = self.render(opt, pose, intr=intr, ray_idx=ray_idx, depth_range=depth_range,
                                  sample_idx=sample_idx, mode=mode)
                for k in keys:
                    parts[k].append(ret[k])
            return AttrDict({k: (v[0] if len(v) == 1 else torch.cat(v, dim=1)) for k, v in parts.items()})

        # mask prior: only object pixels are rendered, the rest keeps the defaults of :657-667.  The reference is B = 1 only
        # (its defaults are [1,HW,.] tensors); here every view of the batch gets its own ray list.
        B = len(pose)
        N = opt.nerf.sample_intvs
        ret_all = AttrDict()
        for k in keys:
            if k == "uncert":
                ret_all[k] = torch.full((B, HW, 1), float(opt.nerf.min_uncert), device=dev)
            elif k == "density":
                ret_all[k] = torch.ones(B, HW, N, 2, device=dev)
            elif "rgb" in k:
                ret_all[k] = torch.zeros(B, HW, 3, device=dev)
            elif "alpha" in k:
                ret_all[k] = torch.ones(B, HW, N, device=dev)
            else:
                ret_all[k] = torch.zeros(B, HW, 1, device=dev)
        masks = object_mask.reshape(B, HW)
        for b in range(B):
            ray_idx_obj = (masks[b] > 0).nonzero(as_tuple=True)[0]
            sl = slice(b, b + 1)
            idx_b = sample_idx if (sample_idx is None or torch.as_tensor(sample_idx).dim() == 0) else sample_idx[b]
            for c in range(0, len(ray_idx_obj), step):
                ray_idx = ray_idx_obj[c:c + step][None]
                ret = self.render(opt, pose[sl], intr=intr[sl] if intr is not None else None,
                                  depth_range=tuple(d[sl] for d in depth_range), ray_idx=ray_idx, sample_idx=idx_b, mode=mode)
                for k in keys:
                    ret_all[k][b, ray_idx[0]] = ret[k][0]
        return ret_all

    def render_masked(self, opt, pose, intr, depth_range, object_mask, sample_idx=None, mode="eval", want=None, out_ptrs=None,
                      shard=None):
        """The mask-prior branch of render_by_slices (model/nerf_adapt_st_gan.py:647-680) for B views as one render launch (the
        lock-step bf16 launch where it applies, otherwise the staged kernel's, as NeRF.render_rays chooses): the
        object pixels (object_mask > 0) of every view are rendered from a ray list built on the device (ops.mask_ray_list), every
        other pixel holds the defaults of :657-667.  No host synchronisation: the call can be captured in a CUDA graph.
        Returns render_by_slices' eleven keys ([B,HW,C]; `want` restricts them).  Sample keys are those of a full-frame launch, so
        with rng 'torch' the jitter is a frame-sized torch.rand(B, HW, N, 1): a seeded call equals the seeded full-frame
        `_render_fused(range(0, HW))` call at the object pixels (the seeded stream of render_by_slices' per-view draws differs).
        out_ptrs: {key: device address of a [B*HW,C] frame buffer}, as for _render_fused.  shard = (rank, world): render this
        rank's share of the list and the defaults of the row block parallel.shard_rays(HW, rank, world, align=W) only.

        Where it runs: wherever a render launch renders the model -- the lock-step launch where `fused_render_applies` (bf16 / auto and
        the yaml's architecture), otherwise the staged launch (opt.b200.mlp = 'fp32', and bf16 for other 256-wide architectures), as
        FrameGather's 'val' frames do.  There render_by_slices takes the multi-kernel path instead, whose compositing sums in another
        order: the two agree to <= 1e-4 in the fp32 mode, not bit for bit.  Raises NotImplementedError in training, with a gradient
        recorded, with opt.b200.fused_render = False, and (from NeRF.render_rays) for what neither render launch takes."""
        if opt.camera.ndc:
            raise NotImplementedError("camera.ndc is false in every reference yaml; not implemented")
        if mode == "train" or torch.is_grad_enabled() or not self._b200(opt, "fused_render", True):
            raise NotImplementedError("render_masked runs on a render launch: inference only (torch.no_grad(), not mode 'train')")
        # (NeRF.render_rays raises NotImplementedError for whatever else neither render launch takes: N, precision, architecture)
        from ..parallel import shard_rays
        B, HW, N = len(pose), opt.H * opt.W, opt.nerf.sample_intvs
        dev = pose.device
        kinv, pinv = camera.view_matrices(pose, intr, one_launch=camera.one_launch_matrices(opt))
        zn, zf = depth_range[0].reshape(B, HW), depth_range[1].reshape(B, HW)
        lat_trans, lat_light = self._latents(opt, B, sample_idx, mode, dev)
        mask = ops._f32(object_mask.reshape(B, HW))
        ray_list, n_slots, _ = ops.mask_ray_list(mask, N)
        rand, seed = None, 0
        if opt.nerf.sample_stratified:
            if self._b200(opt, "rng", "torch") == "philox":
                refuse_capture(*_PHILOX)
                seed = int(torch.randint(0, 2 ** 62, (1,)).item())      # (a host generator: no device read-back)
            else:
                rand = torch.rand(B, HW, N, 1, device=dev)
        rank, world = shard if shard is not None else (0, 1)
        keys = tuple(want) if want is not None else self.RENDER_KEYS
        ret = self.nerf.render_rays(opt, kinv, pinv, None, 0, HW, zn, zf, lat_trans, lat_light, mode=mode, rand=rand, seed=seed,
                                    want=keys, out_ptrs=out_ptrs, ray_list=(ray_list, n_slots), shard=(rank, world))
        dst = dict(ret)
        dst.update({k: int(v) for k, v in (out_ptrs or {}).items()})
        pix0, pix1 = shard_rays(HW, rank, world, align=opt.W)
        ops.mask_defaults(mask, N, float(opt.nerf.min_uncert), {k: dst[k] for k in keys}, pix0, pix1)
        return AttrDict(ret)

    def evaluate_frame(self, opt, var):
        """Per-frame numbers of Model.evaluate_full (model/nerf_adapt_st_gan.py:341-362) for every view of the batch, without a
        host sync: rgb_map [B,3,H,W] (from rgb_static), depth_map [B,1,H,W] in metres, image * mask, per-view MSE / PSNR on
        the device (csrc/loss.cu, tp_eval_epilogue).  SSIM / LPIPS need third-party nets and stay with the engine."""
        B, H, W = len(var.pose), opt.H, opt.W
        dev = var.rgb_static.device
        rgb_map = torch.empty(B, 3, H, W, device=dev)
        depth_map = torch.empty(B, 1, H, W, device=dev)
        image_masked = torch.empty(B, 3, H, W, device=dev)
        mse, psnr = torch.empty(B, device=dev), torch.empty(B, device=dev)
        lib = ops._C.load()
        ws = torch.empty(lib.tp_eval_epilogue_workspace(B), device=dev)
        f = ops._f32
        ops._C.call("tp_eval_epilogue", ops._p(f(var.rgb_static)), ops._p(f(var.depth)), ops._p(f(var.image)),
                    ops._p(f(var.obj_mask)), B, H * W, float(opt.nerf.depth.scale), ops._p(rgb_map), ops._p(depth_map),
                    ops._p(image_masked), ops._p(mse), ops._p(psnr), ops._p(ws), ws.numel(), ops._stream())
        return AttrDict(rgb_map=rgb_map, depth_map=depth_map, image_masked=image_masked, mse=mse, psnr=psnr)

    def sample_depth(self, opt, batch_size, depth_range, num_rays=None):
        """model/nerf_adapt_st_gan.py:682-700.  The jitter is the same torch.rand draw as the reference (parity);
        opt.b200.rng = 'philox' switches to the in-kernel stream."""
        zn, zf = depth_range
        num_rays = num_rays or opt.H * opt.W
        zn, zf = zn.reshape(batch_size, num_rays), zf.reshape(batch_size, num_rays)
        if opt.nerf.depth.param != "metric":
            raise NotImplementedError("nerf.depth.param is 'metric' in every reference yaml")
        N = opt.nerf.sample_intvs
        if not opt.nerf.sample_stratified:
            return ops.sample_depth(zn, zf, N, stratified=False)
        if self._b200(opt, "rng", "torch") == "philox":
            refuse_capture(*_PHILOX)
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())
            return ops.sample_depth(zn, zf, N, seed=seed)
        rand = torch.rand(batch_size, num_rays, N, 1, device=zn.device)
        return ops.sample_depth(zn, zf, N, rand=rand)

    @staticmethod
    def ray_batch_sample(ray_identity, ray_idx):
        """model/nerf_adapt_st_gan.py:702-710."""
        assert ray_identity.shape[0] == ray_idx.shape[0]
        return ops.gather_rows(ray_identity, ray_idx)
