"""Drop-in for layers/nerf.py: the plain NeRF (trainable trunk + rgb head, single-chain compositing)."""
from __future__ import annotations

import torch

from .. import ops
from . import _common
from ._mlp import MLPConfig, run_mlp


class NeRF(torch.nn.Module):

    def __init__(self, opt):
        super().__init__()
        # layers/nerf.py:15-48
        d3 = 3 + 6 * opt.arch.posenc.L_3D if opt.arch.posenc else 3
        dview = (3 + 6 * opt.arch.posenc.L_view if opt.arch.posenc else 3) if opt.nerf.view_dep else 0
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
        self.mlp_rgb = torch.nn.ModuleList()
        dims = _common.layer_dims(opt.arch.layers_rgb)
        feat_dim = opt.arch.layers_feat[-1]
        for li, (k_in, k_out) in enumerate(dims):
            if li == 0:
                k_in = feat_dim + dview + 3
            lin = torch.nn.Linear(k_in, k_out)
            if tf:
                _common.tf_init_(lin, out="all" if li == len(dims) - 1 else None)
            self.mlp_rgb.append(lin)
        if opt.c2f is not None:
            self.progress = torch.nn.Parameter(torch.tensor(0.))
        self._packed = None     # (version key, packed bf16 weight image) for the tcgen05 kernel
        self._tc_image = None
        self._tc32_image = None   # (version key, padded head parameters), see _tc_parameters

    def _config(self, opt, mode) -> MLPConfig:
        if opt.arch.density_activ != "softplus":
            raise NotImplementedError("texpose_b200 implements density_activ: softplus (the reference yaml setting)")
        if opt.nerf.density_noise_reg and mode == "train":
            raise NotImplementedError("density_noise_reg is null in every reference yaml; not implemented")
        if opt.c2f is not None:
            raise NotImplementedError("coarse-to-fine windowing is off (c2f null) in nerf_lm_env.yaml; not implemented")
        return MLPConfig(L_3D=opt.arch.posenc.L_3D, L_view=opt.arch.posenc.L_view, skip=tuple(opt.arch.skip),
                         view_dep=bool(opt.nerf.view_dep), n_feat=len(self.mlp_feat), n_rgb=len(self.mlp_rgb), n_trans=0,
                         precision="fp32", save_for_backward=torch.is_grad_enabled())

    def forward(self, opt, points_3D, ray_unit=None, mode=None):
        """layers/nerf.py:61-99 -> rgb [B,HW,N,3], density [B,HW,N]."""
        cfg = self._config(opt, mode)
        geom = _common.point_geometry(cfg, points_3D, ray_unit)
        return run_mlp(cfg, geom, None, None, *_common.flat_params(self.mlp_feat, self.mlp_rgb))

    def forward_samples(self, opt, center, ray, depth_samples, mode=None):
        """layers/nerf.py:101-115.  Rendering (no gradient needed) with opt.b200.mlp 'bf16' / 'auto' runs on the fused
        tcgen05 kernel, with 'fp32' on the split-fp16 kernel; training runs on the tensor cores with 'bf16' / 'auto', and with
        'fp32' when opt.b200.fp32_engine = 'tc' (trains_on_tensor_cores); otherwise on the fp32 SIMT kernels."""
        cfg = self._config(opt, mode)
        geom = _common.ray_geometry(cfg, center, ray, depth_samples)
        if geom["S"] > 0 and self.uses_tensor_cores(opt):
            return self._forward_tc(cfg, geom)
        if geom["S"] > 0 and self.uses_split_tensor_cores(opt):
            return self._forward_tc32(cfg, geom)
        if geom["S"] > 0 and self.trains_on_tensor_cores(opt, cfg):
            from .. import mlp_tc_plain
            split = _common.mlp_precision(opt) == "fp32"
            return mlp_tc_plain.PlainTC.apply(cfg, geom, len(self.mlp_feat), split, *_common.flat_params(self.mlp_feat, self.mlp_rgb))
        return run_mlp(cfg, geom, None, None, *_common.flat_params(self.mlp_feat, self.mlp_rgb))

    # ------------------------------------------------------------------ tensor-core rendering path
    def uses_tensor_cores(self, opt) -> bool:
        """True when forward_samples will take the fused tcgen05 kernel: precision bf16 / auto, no gradient wanted, and
        the architecture is the 8 x 256 trunk (skip 4, L = 10 / <= 4) with an rgb head of 1-3 hidden layers <= 256 wide."""
        if _common.mlp_precision(opt) == "fp32":
            return False
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            return False
        if not (opt.nerf.view_dep and opt.arch.posenc and opt.arch.posenc.L_3D == 10 and 0 <= opt.arch.posenc.L_view <= 4
                and tuple(opt.arch.skip) == (4,)):
            return False
        want_f = [(256, 63)] + [(256, 256)] * 3 + [(256, 319)] + [(256, 256)] * 2 + [(257, 256)]
        if [tuple(l.weight.shape) for l in self.mlp_feat] != want_f:
            return False
        n = len(self.mlp_rgb)
        widths = [l.weight.shape[0] for l in self.mlp_rgb]
        return 2 <= n <= 4 and all(w <= 256 for w in widths[:-1]) and widths[-1] == 3

    def _tc_parameters(self):
        """The plain model expressed in the layer layout the fused kernel streams (static / transient / light model of
        options/nerf_lm_adapt_gan.yaml): hidden layers zero-padded to 256 x 256, missing hidden layers replaced by the
        identity (exact: their input is a ReLU output already rounded to bf16), no latents; the launch is static-only
        (flags bit 17), so the (all-zero) transient head of the image is never streamed.  Rebuilt when a parameter changes."""
        params = [p for l in list(self.mlp_feat) + list(self.mlp_rgb) for p in (l.weight, l.bias)]
        key = tuple((p.data_ptr(), p._version) for p in params)
        if self._tc_image is not None and self._tc_image[0] == key:
            return self._tc_image[1]
        dev = self.mlp_feat[0].weight.device
        z = lambda *shape: torch.zeros(*shape, device=dev)
        feat_p = [(l.weight.detach().float().contiguous(), l.bias.detach().float().contiguous()) for l in self.mlp_feat]
        layers = [(l.weight.detach().float(), l.bias.detach().float()) for l in self.mlp_rgb]
        k0 = layers[0][0].shape[1]
        rgb_p = []
        for li in range(3):
            W, b = z(256, k0 if li == 0 else 256), z(256)
            if li < len(layers) - 1:
                w_src, b_src = layers[li]
                W[:w_src.shape[0], :w_src.shape[1]] = w_src
                b[:b_src.shape[0]] = b_src
            else:
                W += torch.eye(256, device=dev)      # pass-through layer
            rgb_p.append((W, b))
        w_out, b_out = layers[-1]
        W = z(3, 256)
        W[:, :w_out.shape[1]] = w_out
        rgb_p.append((W, b_out.contiguous()))
        trans_p = [(z(256, 256), z(256)), (z(256, 256), z(256)), (z(256, 256), z(256)), (z(5, 256), z(5))]
        self._tc_image = (key, (feat_p, rgb_p, trans_p))
        return self._tc_image[1]

    def _forward_tc(self, cfg, geom):
        from .. import mlp_tc
        feat_p, rgb_p, trans_p = self._tc_parameters()
        B, R, N = geom["shape"]
        dev = geom["depth"].device
        stl = MLPConfig(L_3D=cfg.L_3D, L_view=cfg.L_view, skip=cfg.skip, view_dep=True, n_feat=8, n_rgb=4, n_trans=4,
                        n_latent_light=0, n_latent_trans=0, precision="bf16", save_for_backward=False, packed=self,
                        static_only=True)
        none = torch.zeros(B, 0, device=dev)
        rgb, density, _ = mlp_tc.forward(stl, geom, none, none, feat_p, rgb_p, trans_p, static_only=True)
        return rgb.view(B, R, N, 3, 2)[..., 0].contiguous(), density.view(B, R, N, 2)[..., 0].contiguous()

    def trains_on_tensor_cores(self, opt, cfg=None) -> bool:
        """True when a gradient-recording forward_samples takes the tensor-core training path (mlp_tc_plain: single-pass bf16
        forward with saved activations, staged dX chain, dW GEMMs): opt.b200.mlp 'bf16' / 'auto', or 'fp32' with
        opt.b200.fp32_engine = 'tc' (the split kernels, <= 1e-4), and a supported architecture."""
        if not torch.is_grad_enabled():
            return False
        if _common.mlp_precision(opt) == "fp32" and _common.b200_option(opt, "fp32_engine", "auto") != "tc":
            return False
        from .. import mlp_tc_plain
        cfg = cfg or self._config(opt, None)
        pairs = [(l.weight, l.bias) for l in list(self.mlp_feat) + list(self.mlp_rgb)]
        return mlp_tc_plain.supported(cfg, pairs[:len(self.mlp_feat)], pairs[len(self.mlp_feat):])

    # ------------------------------------------------------------------ fp32-parity rendering on the tensor cores
    def uses_split_tensor_cores(self, opt) -> bool:
        """True when forward_samples will take the split-fp16 kernel (csrc/mlp_tc_split.cu, <= 1e-4): no gradient wanted, the
        bf16 kernel not selected (opt.b200.mlp = 'fp32', or an architecture it does not implement), 256-wide trunk of any depth /
        skip set, rgb head of any depth <= 256 wide, L_3D = 10.  opt.b200.fp32_engine = 'simt' keeps the SIMT kernels."""
        if _common.b200_option(opt, "fp32_engine", "auto") == "simt":
            return False
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            return False
        return self._staged_architecture(opt)

    def _staged_architecture(self, opt) -> bool:
        """The layer shapes the staged kernel (mlp_tc32) takes for this model."""
        if not (opt.nerf.view_dep and opt.arch.posenc and opt.arch.posenc.L_3D == 10 and 0 <= (opt.arch.posenc.L_view or 0) <= 4):
            return False
        nf, skip = len(self.mlp_feat), set(opt.arch.skip)
        if nf < 2 or 0 in skip or nf - 1 in skip or len(self.mlp_rgb) < 2:
            return False
        for li, l in enumerate(self.mlp_feat):
            k = 63 if li == 0 else 256 + (63 if li in skip else 0)
            if tuple(l.weight.shape) != ((257 if li == nf - 1 else 256), k):
                return False
        widths = [l.weight.shape[0] for l in self.mlp_rgb]
        return all(w <= 256 for w in widths[:-1]) and widths[-1] == 3 and nf + 1 + len(widths) <= 24

    def _tc32_parameters(self):
        """The plain model as the layer list mlp_tc32 builds its stages from: rgb hidden layers zero-padded to 256 wide (exact),
        no latents, a dummy transient head that the static-only stage list never streams."""
        params = [p for l in list(self.mlp_feat) + list(self.mlp_rgb) for p in (l.weight, l.bias)]
        key = tuple((p.data_ptr(), p._version) for p in params)
        if self._tc32_image is not None and self._tc32_image[0] == key:
            return self._tc32_image[1]
        dev = self.mlp_feat[0].weight.device
        z = lambda *shape: torch.zeros(*shape, device=dev)
        feat_p = [(l.weight.detach().float().contiguous(), l.bias.detach().float().contiguous()) for l in self.mlp_feat]
        layers = [(l.weight.detach().float(), l.bias.detach().float()) for l in self.mlp_rgb]
        rgb_p = []
        for li, (w_src, b_src) in enumerate(layers):
            last = li == len(layers) - 1
            W, b = z(3 if last else 256, w_src.shape[1] if li == 0 else 256), z(3 if last else 256)
            W[:w_src.shape[0], :w_src.shape[1]] = w_src
            b[:b_src.shape[0]] = b_src
            rgb_p.append((W, b))
        trans_p = [(z(256, 256), z(256)), (z(5, 256), z(5))]
        self._tc32_image = (key, (feat_p, rgb_p, trans_p))
        return self._tc32_image[1]

    def _forward_tc32(self, cfg, geom):
        from .. import mlp_tc32
        feat_p, rgb_p, trans_p = self._tc32_parameters()
        B, R, N = geom["shape"]
        dev = geom["depth"].device
        stl = MLPConfig(L_3D=cfg.L_3D, L_view=cfg.L_view, skip=cfg.skip, view_dep=True, n_feat=len(feat_p), n_rgb=len(rgb_p),
                        n_trans=2, n_latent_light=0, n_latent_trans=0, precision="fp32", save_for_backward=False, packed=self,
                        static_only=True)
        none = torch.zeros(B, 0, device=dev)
        rgb, density, _ = mlp_tc32.forward(stl, geom, none, none, feat_p, rgb_p, trans_p, static_only=True)
        return rgb.view(B, R, N, 3, 2)[..., 0].contiguous(), density.view(B, R, N, 2)[..., 0].contiguous()

    # ------------------------------------------------------------------ one-launch rendering (staged kernel, render mode)
    def render_precision(self, opt) -> int:
        """Arithmetic of render_rays: 0 = split hi + lo (<= 1e-4) for opt.b200.mlp 'fp32' and for 'auto' where the bf16 kernel does
        not implement the architecture (what forward_samples computes then); 1 = single-pass bf16 (<= 1e-2) otherwise.  Raises
        NotImplementedError when the staged launch cannot render this model under `opt`."""
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            raise NotImplementedError("render_rays is inference: call it under torch.no_grad()")
        if opt.nerf.get("setbg_opaque"):
            raise NotImplementedError("render_rays composites without a background colour (opt.nerf.setbg_opaque)")
        if opt.camera.ndc:
            raise NotImplementedError("camera.ndc is false in every reference yaml; not implemented")
        if opt.nerf.depth.param != "metric":
            raise NotImplementedError("nerf.depth.param is 'metric' in every reference yaml")
        from .. import mlp_tc
        if opt.nerf.sample_intvs not in mlp_tc.FUSED_N:
            raise NotImplementedError(f"the render launch takes {mlp_tc.FUSED_N} samples per ray, not {opt.nerf.sample_intvs}")
        prec = _common.mlp_precision(opt)
        if prec == "fp32" and _common.b200_option(opt, "fp32_engine", "auto") == "simt":
            raise NotImplementedError("opt.b200.fp32_engine = 'simt' keeps the fp32 mode off the tensor cores")
        if not self._staged_architecture(opt):
            raise NotImplementedError("the staged render launch takes 256-wide trunks with L_3D = 10 and rgb heads <= 256 wide")
        if prec == "auto":
            return 1 if self.uses_tensor_cores(opt) else 0
        return 0 if prec == "fp32" else 1

    def render_rays(self, opt, kinv, pinv, ray_idx, ray0, R, z_near, z_far, mode=None, rand=None, seed=0, want=None,
                    out_ptrs=None):
        """camera.get_center_and_ray + ray_batch_sample + sample_depth + forward_samples + composite (model/nerf_pretrain.py:588-627)
        as ONE launch of the staged kernel (tp_tc32_render_forward) in render_precision(opt); returns {rgb [B,R,3], depth
        [B,R,1], opacity [B,R,1], density [B,R,N]} (the `want` subset; outputs in out_ptrs are written there instead)."""
        from .. import mlp_tc32
        precision = self.render_precision(opt)
        cfg = self._config(opt, mode)
        feat_p, rgb_p, trans_p = self._tc32_parameters()
        stl = MLPConfig(L_3D=cfg.L_3D, L_view=cfg.L_view, skip=cfg.skip, view_dep=True, n_feat=len(feat_p), n_rgb=len(rgb_p),
                        n_trans=2, n_latent_light=0, n_latent_trans=0, precision="fp32" if precision == 0 else "bf16",
                        save_for_backward=False, packed=self, static_only=True)
        none = torch.zeros(len(kinv), 0, device=kinv.device)
        return mlp_tc32.render(stl, kinv, pinv, opt.H, opt.W, ray_idx, ray0, R, ops._f32(z_near), ops._f32(z_far),
                               opt.nerf.sample_intvs, none, none, feat_p, rgb_p, trans_p, 0.0, rand=rand,
                               stratified=bool(opt.nerf.sample_stratified), seed=seed, static_only=True, precision=precision,
                               want=want, out_ptrs=out_ptrs)

    @staticmethod
    def composite(opt, ray, rgb_samples, density_samples, depth_samples):
        """layers/nerf.py:117-136 -> rgb, depth, opacity, prob."""
        bg = opt.data.bgcolor if opt.nerf.get("setbg_opaque") else None
        return ops.CompositePlain.apply(ray, rgb_samples, density_samples, depth_samples, bg)

    def positional_encoding(self, opt, x, L, c2f=False):
        if opt.c2f is not None and c2f:
            raise NotImplementedError("c2f windowing not implemented")
        flat = ops._f32(x.detach()).reshape(-1, 3)
        enc = ops.positional_encode(flat, L)
        return enc[:, 3:3 + 6 * L].reshape(*x.shape[:-1], 6 * L)
