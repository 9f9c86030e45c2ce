"""Mirror of ``nerf_sampling/depth_nets/depth_net.py``: same constructor, parameters and state_dict keys."""

from __future__ import annotations

import torch
from torch import nn

from .. import ops, packing
from ..packing import PREC_SPLIT, PackedDepthNet


class DepthNet(nn.Module):
    """Per-ray depth predictor (depth_nets/depth_net.py:10-169).

    Parameters are created in the reference's order (so a seeded init reproduces its weights) and registered under
    the reference's names.  Under ``torch.no_grad()`` ``forward`` runs the fused tcgen05 kernel (the activation-free
    branch stacks are folded into the first dense layer when the packed image is built, see packing.fold_depthnet);
    with gradients enabled it runs the literal per-layer fp32 form whose backward yields every parameter gradient."""

    def __init__(self, hidden_sizes=[128 for _ in range(6)], cat_hidden_sizes=[128, 128, 128, 128, 256],
                 origin_channels: int = 3, direction_channels: int = 3, multires: int = 10, sphere_radius: float = 2.0,
                 near: int = 2, far: int = 6):
        super().__init__()
        if origin_channels != 3 or direction_channels != 3:
            raise NotImplementedError("the B200 DepthNet kernel implements 3-channel rays")
        if multires not in packing.MULTIRES_RANGE:
            raise ValueError(f"multires={multires} out of range: the B200 DepthNet kernels serve multires 1..10")
        self.sphere_radius = torch.tensor([sphere_radius])
        self.near, self.far = near, far
        d3, d6 = 3 * (1 + 2 * multires), 6 * (1 + 2 * multires)
        self.origin_dims = self.direction_dims = d3
        self.intersection_points_dim = d6
        origin = [nn.Linear(2 * d3, hidden_sizes[0])]
        direction = [nn.Linear(2 * d3, hidden_sizes[0])]
        inter = [nn.Linear(2 * d6, hidden_sizes[0])]
        for i, size in enumerate(hidden_sizes[:-1]):
            for layers in (origin, direction):
                layers.append(nn.Linear(size + d3, hidden_sizes[i + 1]))
        for i, size in enumerate(hidden_sizes[:-1]):
            inter.append(nn.Linear(size + d6, hidden_sizes[i + 1]))
        cat = [nn.Linear(hidden_sizes[-1] * 3 + d3 + d3 + d6, cat_hidden_sizes[0]), nn.LeakyReLU()]
        for i, size in enumerate(cat_hidden_sizes[:-1]):
            cat += [nn.Linear(size, cat_hidden_sizes[i + 1]), nn.LeakyReLU()]
        self.origin_layers = nn.Sequential(*origin)
        self.direction_layers = nn.Sequential(*direction)
        self.intersection_layers = nn.Sequential(*inter)
        self.cat_layers = nn.Sequential(*cat)
        self.to_depth = nn.Sequential(nn.Linear(cat_hidden_sizes[-1], 1), nn.Sigmoid())
        self.precision = PREC_SPLIT
        self._packed = None
        self._packed_key = None

    def packed(self) -> PackedDepthNet:
        params = list(self.parameters())
        key = (self.precision, packing.generation()) + tuple((p.data_ptr(), p._version) for p in params)
        if self._packed is None or key != self._packed_key:
            self._packed = PackedDepthNet(self.state_dict(), params[0].device, self.precision)
            self._packed_key = key
        return self._packed

    def calculate_intersection_points(self, rays_o, rays_d):
        from ..nerf_pytorch.utils import find_intersection_points_with_sphere

        return find_intersection_points_with_sphere(rays_o, rays_d, self.sphere_radius)[1]

    def forward(self, rays_o: torch.Tensor, rays_d: torch.Tensor) -> torch.Tensor:
        """[N,1] depth in [near, far] per ray."""
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            # training: literal per-layer fp32 form with saved activations (csrc/train.cu), differentiable
            from .. import training

            return training.DepthNetTrainFn.apply(rays_o.contiguous().float(), rays_d.contiguous().float(),
                                                  (*training.depthnet_arch(self), training.depthnet_multires(self)),
                                                  float(self.sphere_radius), float(self.near),
                                                  float(self.far), *training.depthnet_params(self))
        return ops.depthnet_forward(self.packed(), rays_o, rays_d, float(self.sphere_radius), float(self.near),
                                    float(self.far))
