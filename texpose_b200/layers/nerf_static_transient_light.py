"""Drop-in for layers/nerf_static_transient_light.py: the static / transient / light NeRF of the texture learner.

Same constructor, parameter containers (`mlp_feat`, `mlp_rgb`, `mlp_trans` ModuleLists of nn.Linear, `progress`)
and method signatures as the reference class, so checkpoints (state-dict keys `nerf.mlp_feat.{i}.weight` ...)
load unchanged; the arithmetic runs in the sm_100a kernels behind the C-ABI.
"""
from __future__ import annotations

import torch

from .. import ops
from . import _common
from ._mlp import MLPConfig, run_mlp


class NeRF(torch.nn.Module):

    def __init__(self, opt):
        super().__init__()
        # layer shapes: layers/nerf_static_transient_light.py:15-61
        d3 = 3 + 6 * opt.arch.posenc.L_3D if opt.arch.posenc else 3
        dview = (3 + 6 * opt.arch.posenc.L_view if opt.arch.posenc.L_view else 3) if opt.nerf.view_dep else 0
        tf = opt.arch.tf_init
        self.mlp_feat = torch.nn.ModuleList()
        dims = _common.layer_dims(opt.arch.layers_feat)
        for li, (k_in, k_out) in enumerate(dims):
            k_in = d3 if li == 0 else k_in
            k_in = k_in + d3 if li in opt.arch.skip else k_in
            last = li == len(dims) - 1
            lin = torch.nn.Linear(k_in, k_out + 1 if last else k_out)
            if tf:
                _common.tf_init_(lin, out="first" if last else None)
            self.mlp_feat.append(lin)
        for p in self.mlp_feat.parameters():      # static scene is frozen (:34, :236-239)
            p.requires_grad = False

        feat_dim = opt.arch.layers_feat[-1]
        self.mlp_rgb = torch.nn.ModuleList()
        dims = _common.layer_dims(opt.arch.layers_rgb)
        for li, (k_in, k_out) in enumerate(dims):
            if li == 0:
                k_in = feat_dim + dview + 3 + opt.nerf.N_latent_light
            lin = torch.nn.Linear(k_in, k_out)
            if tf:
                _common.tf_init_(lin, out="all" if li == len(dims) - 1 else None)
            self.mlp_rgb.append(lin)

        if opt.arch.layers_trans:
            self.mlp_trans = torch.nn.ModuleList()
            dims = _common.layer_dims(opt.arch.layers_trans)
            for li, (k_in, k_out) in enumerate(dims):
                if li == 0:
                    k_in = feat_dim + opt.nerf.N_latent_trans
                lin = torch.nn.Linear(k_in, k_out)
                if tf:
                    _common.tf_init_(lin, out="all" if li == len(dims) - 1 else None)
                self.mlp_trans.append(lin)
        if opt.c2f is not None:
            self.progress = torch.nn.Parameter(torch.tensor(0.))
        self._packed = None     # (version key, packed bf16 weight image) for the tcgen05 kernel

    # ------------------------------------------------------------------ helpers
    def _config(self, opt, mode) -> MLPConfig:
        if opt.arch.density_activ != "softplus":
            raise NotImplementedError("texpose_b200 implements density_activ: softplus (the reference yaml setting)")
        if opt.nerf.density_noise_reg and mode == "train":
            raise NotImplementedError("density_noise_reg is null in every reference yaml; not implemented")
        if opt.c2f is not None and opt.c2f.range is not None:
            raise NotImplementedError("coarse-to-fine windowing (c2f.range) is off in the reference yaml; not implemented")
        if not opt.arch.layers_trans:
            raise NotImplementedError("static/transient NeRF requires arch.layers_trans")
        return MLPConfig(L_3D=opt.arch.posenc.L_3D, L_view=opt.arch.posenc.L_view or 0, skip=tuple(opt.arch.skip),
                         view_dep=bool(opt.nerf.view_dep), n_feat=len(self.mlp_feat), n_rgb=len(self.mlp_rgb),
                         n_trans=len(self.mlp_trans), n_latent_light=opt.nerf.N_latent_light,
                         n_latent_trans=opt.nerf.N_latent_trans, precision=_common.mlp_precision(opt),
                         save_for_backward=torch.is_grad_enabled(), packed=self,
                         static_only=bool(mode == "eval" and _common.b200_option(opt, "static_only", False)),
                         fp32_tc=_common.b200_option(opt, "fp32_engine", "auto") != "simt",
                         fp32_train_tc=_common.b200_option(opt, "fp32_engine", "auto") == "tc")

    def uses_tensor_cores(self, opt, mode="val") -> bool:
        """True when forward_samples of this module will take the fused tcgen05 path under `opt` (opt.b200.mlp)."""
        cfg = self._config(opt, mode)
        if cfg.precision == "fp32":
            return False
        from .. import mlp_tc
        pairs = lambda ml: [(l.weight, l.bias) for l in ml]
        return mlp_tc.supported(cfg, pairs(self.mlp_feat), pairs(self.mlp_rgb), pairs(self.mlp_trans))

    def _run(self, cfg, geom, latent_variable_trans, latent_variable_light):
        # The reference runs the trunk and the static density under torch.no_grad() (:87-101): the static scene never
        # receives a gradient, whatever requires_grad says -- its engine calls toggle_grad(nerf, True) before every
        # nerf_trainstep (model/nerf_adapt_st_gan.py:110).  The trunk parameters therefore enter the autograd function
        # detached: no trunk gradient is computed, none is returned, and the fused bf16 path stays selected.
        trunk = [p.detach() for p in _common.flat_params(self.mlp_feat)]
        params = trunk + _common.flat_params(self.mlp_rgb, self.mlp_trans)
        return run_mlp(cfg, geom, latent_variable_trans, latent_variable_light, *params)

    # ------------------------------------------------------------------ reference interface
    def forward(self, opt, points_3D, ray_unit=None, latent_variable_trans=None, latent_variable_light=None, mode=None):
        """layers/nerf_static_transient_light.py:76-145 -> rgb [B,HW,N,3,2], density [B,HW,N,2], uncert [B,HW,N,1]."""
        assert points_3D.dim() == 4, "points_3D must be [B,HW,N,3] (reference :78)"
        cfg = self._config(opt, mode)
        if cfg.view_dep:
            assert ray_unit is not None
        cfg.precision = "fp32"      # explicit-points entry: the fused bf16 kernel is ray-parameterised
        geom = _common.point_geometry(cfg, points_3D, ray_unit)
        return self._run(cfg, geom, latent_variable_trans, latent_variable_light)

    def forward_samples(self, opt, center, ray, depth_samples, latent_variable_trans=None, latent_variable_light=None,
                        mode=None):
        """layers/nerf_static_transient_light.py:147-166."""
        cfg = self._config(opt, mode)
        geom = _common.ray_geometry(cfg, center, ray, depth_samples)
        return self._run(cfg, geom, latent_variable_trans, latent_variable_light)

    def fused_render_applies(self, opt, mode) -> bool:
        """True when Graph.render may run as ONE launch (tp_render_fused_forward): inference (no gradient recorded), the fused
        kernel's architecture and precision, 32 / 64 / 128 samples per ray.  opt.b200.fused_render = False switches it off."""
        from .. import mlp_tc
        if mode == "train" or torch.is_grad_enabled() or not _common.b200_option(opt, "fused_render", True):
            return False
        if opt.nerf.sample_intvs not in mlp_tc.FUSED_N or opt.nerf.depth.param != "metric" or opt.camera.ndc:
            return False
        return self.uses_tensor_cores(opt, mode)

    def render_rays(self, opt, kinv, pinv, ray_idx, ray0, R, z_near, z_far, latent_variable_trans, latent_variable_light,
                    mode=None, rand=None, seed=0, want=None, out_ptrs=None, ray_list=None, shard=(0, 1)):
        """get_center_and_ray + ray_batch_sample + sample_depth + forward_samples + composite (model/nerf_adapt_st_gan.py:565-631)
        in one launch; returns the dict of the eleven outputs of Graph.render.  The lock-step bf16 render launch
        (tp_render_fused_forward) where it implements the precision and architecture; otherwise the staged kernel's render launch
        (tp_tc32_render_forward, render_precision).  List form: ray_list = (list, n_slots) of ops.mask_ray_list with ray_idx None,
        ray0 0, R = H*W -- the object pixels of a mask prior, frame-sized outputs (mlp_tc.render_fused)."""
        from .. import mlp_tc
        cfg = self._config(opt, mode)
        pairs = lambda ml: [(l.weight.detach(), l.bias.detach()) for l in ml]
        lt = ops._f32(latent_variable_trans.detach())
        ll = ops._f32(latent_variable_light.detach())
        if not self._lockstep_render_applies(opt, cfg):
            from .. import mlp_tc32
            precision = self.render_precision(opt, cfg)
            return mlp_tc32.render(cfg, kinv, pinv, opt.H, opt.W, ray_idx, ray0, R, ops._f32(z_near), ops._f32(z_far),
                                   opt.nerf.sample_intvs, lt, ll, pairs(self.mlp_feat), pairs(self.mlp_rgb), pairs(self.mlp_trans),
                                   float(opt.nerf.min_uncert), rand=rand, stratified=bool(opt.nerf.sample_stratified), seed=seed,
                                   precision=precision, want=want, out_ptrs=out_ptrs, ray_list=ray_list, shard=shard)
        return mlp_tc.render_fused(cfg, kinv, pinv, opt.H, opt.W, ray_idx, ray0, R, ops._f32(z_near), ops._f32(z_far),
                                   opt.nerf.sample_intvs, lt, ll, pairs(self.mlp_feat), pairs(self.mlp_rgb), pairs(self.mlp_trans),
                                   float(opt.nerf.min_uncert), rand=rand, stratified=bool(opt.nerf.sample_stratified), seed=seed,
                                   static_only=cfg.static_only, want=want or mlp_tc.RENDER_KEYS, out_ptrs=out_ptrs,
                                   ray_list=ray_list, shard=shard)

    def _lockstep_render_applies(self, opt, cfg) -> bool:
        """render_rays takes tp_render_fused_forward: bf16 / auto precision and the architecture the lock-step kernel implements."""
        from .. import mlp_tc
        if cfg.precision == "fp32":
            return False
        pairs = lambda ml: [(l.weight, l.bias) for l in ml]
        return mlp_tc.supported(cfg, pairs(self.mlp_feat), pairs(self.mlp_rgb), pairs(self.mlp_trans))

    def render_precision(self, opt, cfg=None) -> int:
        """Arithmetic of the staged render launch: 0 = split hi + lo (<= 1e-4) for opt.b200.mlp 'fp32', 1 = single-pass bf16
        (<= 1e-2) for 'bf16' / 'auto' -- what forward_samples computes for an architecture the lock-step kernel does not implement.
        Raises NotImplementedError when the staged launch cannot render this model under `opt`."""
        from .. import mlp_tc, mlp_tc32
        cfg = cfg or self._config(opt, None)
        if torch.is_grad_enabled():
            raise NotImplementedError("render_rays is inference: call it under torch.no_grad()")
        if opt.camera.ndc:
            raise NotImplementedError("camera.ndc is false in every reference yaml; not implemented")
        if opt.nerf.depth.param != "metric":
            raise NotImplementedError("nerf.depth.param is 'metric' in every reference yaml")
        if opt.nerf.sample_intvs not in mlp_tc.FUSED_N:
            raise NotImplementedError(f"the render launch takes {mlp_tc.FUSED_N} samples per ray, not {opt.nerf.sample_intvs}")
        if cfg.static_only:
            raise NotImplementedError("static-only rendering (opt.b200.static_only) runs on the lock-step bf16 render launch only")
        if cfg.precision == "fp32" and not cfg.fp32_tc:
            raise NotImplementedError("opt.b200.fp32_engine = 'simt' keeps the fp32 mode off the tensor cores")
        pairs = lambda ml: [(l.weight, l.bias) for l in ml]
        if not mlp_tc32.supported(cfg, pairs(self.mlp_feat), pairs(self.mlp_rgb), pairs(self.mlp_trans)):
            raise NotImplementedError("the staged render launch takes 256-wide static/transient/light layer lists with L_3D = 10")
        return 0 if cfg.precision == "fp32" else 1

    @staticmethod
    def composite(opt, ray, rgb_samples, density_samples, depth_samples, uncert_samples=None):
        """layers/nerf_static_transient_light.py:168-212; returns the reference's 11-tuple."""
        return ops.CompositeSTL.apply(ray, rgb_samples, density_samples, depth_samples, uncert_samples,
                                      float(opt.nerf.min_uncert))

    def positional_encoding(self, opt, x, L, c2f=False):
        """layers/nerf_static_transient_light.py:217-234 for [...,3] inputs (c2f window off)."""
        if opt.c2f is not None and opt.c2f.range is not None and c2f:
            raise NotImplementedError("c2f windowing is off in the reference yaml; not implemented")
        if x.shape[-1] != 3:
            raise NotImplementedError("positional_encoding kernel handles 3-vectors (points / view directions)")
        flat = ops._f32(x.detach()).reshape(-1, 3)
        enc = ops.positional_encode(flat, L)
        return enc[:, 3:3 + 6 * L].reshape(*x.shape[:-1], 6 * L)
