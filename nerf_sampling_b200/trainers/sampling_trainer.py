"""Mirror of ``nerf_sampling/trainers/sampling_trainer.py`` (DepthNetTrainer)."""

from __future__ import annotations

import os
from typing import Optional

import torch

from .. import ops
from ..depth_nets.depth_net import DepthNet
from ..nerf_pytorch import utils
from ..nerf_pytorch.nerf_utils import create_nerf
from ..nerf_pytorch.run_nerf_helpers import NeRF
from ..nerf_pytorch.trainers import Blender


class DepthNetTrainer(Blender.BlenderTrainer):
    """Config bag + model factory + the two operators the render driver calls back into
    (sampling_trainer.py:16-230).  Select it from YAML with
    ``module: nerf_sampling_b200.trainers.DepthNetTrainer``."""

    def __init__(self, distance=None, sampling_mode=None, n_depth_samples=None, depth_net_path: Optional[str] = None,
                 n_layers: int = 6, layer_width: int = 256, sphere_radius: float = 2.0, **kwargs):
        self.n_layers = n_layers
        self.layer_width = layer_width
        self.depth_net_path = depth_net_path
        self.sphere_radius = sphere_radius
        self.distance = distance
        self.n_depth_samples = n_depth_samples
        self.sampling_mode = sampling_mode
        super().__init__(**kwargs)

    def create_nerf_model(self):
        """NeRF coarse(+fine), DepthNet, both optimizers, checkpoints (sampling_trainer.py:54-122)."""
        render_kwargs_train, render_kwargs_test, _start, grad_vars, optimizer = create_nerf(self, NeRF)
        bds = {"near": self.near, "far": self.far}
        render_kwargs_train.update(bds)
        render_kwargs_test.update(bds)
        depth_network = DepthNet(hidden_sizes=[self.layer_width] * self.n_layers,
                                 cat_hidden_sizes=[self.layer_width] * self.n_layers,
                                 sphere_radius=self.sphere_radius).to(self.device)
        from .. import training

        # torch.optim.Adam semantics and state_dict keys, on the library's fused kernel
        sampling_optimizer = training.Adam(params=list(depth_network.parameters()), lr=self.depth_net_lr)
        if self.depth_net_path is not None and self.depth_net_path != "None":
            ckpts = [self.depth_net_path]
        else:
            d = os.path.join(self.basedir, self.expname)
            ckpts = [os.path.join(d, f) for f in sorted(os.listdir(d)) if "tar" in f] if os.path.isdir(d) else []
        start = None
        if len(ckpts) > 0 and not self.no_reload:
            ckpt = torch.load(ckpts[-1], map_location=self.device, weights_only=False)
            start = ckpt["global_step"]
            utils.load_depth_network(depth_network, sampling_optimizer, ckpt)
        self.global_step = self.start = start if start is not None else 0
        for kw, mode in ((render_kwargs_train, "train"), (render_kwargs_test, "test")):
            kw["depth_network"] = depth_network
            kw["model_mode"] = mode
        return optimizer, sampling_optimizer, render_kwargs_train, render_kwargs_test

    def raw2outputs(self, raw, z_vals, rays_d, raw_noise_std=0, white_bkgd=True, pytest=False, **kwargs):
        """(rgb_map, disp_map, acc_map, depth_map, density, alphas, weights) -- sampling_trainer.py:153-230.

        Unknown keyword arguments are swallowed exactly like the reference's ``**kwargs`` (its DepthNet call sites pass
        misspelled ``raw_noise=`` / ``white_bkdg=``, which is why that path always composites noise-free on white).

        When grad is enabled and ``raw`` or ``z_vals`` requires it, the maps are differentiable w.r.t. both
        (training.CompositeFn; at S == 1 training.CompositeSingleFn, whose only dependence is rgb on raw)."""
        noise = None
        if raw_noise_std > 0.0:
            noise = torch.randn(raw[..., 3].shape, device=raw.device) * raw_noise_std
        if torch.is_grad_enabled() and (raw.requires_grad or z_vals.requires_grad):
            from .. import training

            if z_vals.shape[-1] >= 2:
                rgb, disp, acc, depth, weights, alphas = training.CompositeFn.apply(raw, z_vals, rays_d, noise, white_bkgd)
            else:
                rgb, disp = training.CompositeSingleFn.apply(raw, z_vals, rays_d)
                _, _, acc, depth, weights, alphas = ops.composite(raw.detach(), z_vals.detach(), rays_d, white_bkgd, noise)
            return rgb, disp, acc, depth, raw[..., 3], alphas, weights
        rgb, disp, acc, depth, weights, alphas = ops.composite(raw, z_vals, rays_d, white_bkgd, noise)
        return rgb, disp, acc, depth, raw[..., 3], alphas, weights
