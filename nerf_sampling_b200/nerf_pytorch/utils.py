"""Mirror of ``nerf_sampling/nerf_pytorch/utils.py``: checkpoint layout, config plugin hook, geometry helpers."""

from __future__ import annotations

import importlib
from typing import Literal, Optional, Union

import torch

from .. import ops


def load_obj_from_config(cfg: dict):
    """``{"module": "pkg.mod.Class", "kwargs": {...}}`` -> Class(**kwargs) (utils.py:12-21).

    This is the reference's plugin hook: pointing ``module`` at
    ``nerf_sampling_b200.trainers.DepthNetTrainer`` swaps in this implementation."""
    module_name, class_name = cfg["module"].rsplit(".", maxsplit=1)
    return getattr(importlib.import_module(module_name), class_name)(**cfg["kwargs"])


def freeze_model(model):
    for p in model.parameters():
        p.requires_grad = False


def unfreeze_model(model):
    for p in model.parameters():
        p.requires_grad = True


def save_state(global_step: int, network_fn, network_fine, optimizer, depth_network, sampling_optimizer, path: str) -> None:
    """One ``torch.save``d dict with the reference's keys (utils.py:59-89)."""
    data = {
        "global_step": global_step,
        "network_fn_state_dict": network_fn.state_dict(),
        "optimizer_state_dict": optimizer.state_dict(),
        "sampling_optimizer_state_dict": sampling_optimizer.state_dict(),
        "depth_network": depth_network.state_dict(),
    }
    if network_fine is not None:
        data["network_fine_state_dict"] = network_fine.state_dict()
    torch.save(data, path)
    print("Saved checkpoints at", path)


def load_nerf(network_fn, network_fine, optimizer, ckpt) -> None:
    """utils.py:92-108."""
    optimizer.load_state_dict(ckpt["optimizer_state_dict"])
    network_fn.load_state_dict(ckpt["network_fn_state_dict"])
    if network_fine is not None:
        network_fine.load_state_dict(ckpt["network_fine_state_dict"])


def load_depth_network(depth_network, sampling_optimizer, ckpt) -> None:
    """utils.py:111-122."""
    sampling_optimizer.load_state_dict(ckpt["sampling_optimizer_state_dict"])
    depth_network.load_state_dict(ckpt["depth_network"])


def override_config(config, update) -> None:
    """Only existing keys may be overridden (utils.py:125-140)."""
    for key, value in update.items():
        if key not in config:
            raise KeyError(f"Key {key} does not exist in config")
        config[key] = value


def set_global_device(device: Union[Literal["cuda"], Literal["cpu"]]):
    """utils.py:143-149."""
    if device == "cuda":
        if torch.cuda.is_available():
            torch.set_default_device(device="cuda")
    elif device == "cpu":
        torch.set_default_device(device="cpu")


def check_grad(model) -> bool:
    return any(bool(torch.flatten(p.grad).any()) for p in model.parameters())


def solve_quadratic_equation(a: torch.Tensor, b: torch.Tensor, c: torch.Tensor) -> torch.Tensor:
    """Roots stacked as [(-b - sqrt(D)) / 2a, (-b + sqrt(D)) / 2a]; NaN where D < 0 (utils.py:159-179).
    Helper kept for API parity (the DepthNet kernel solves the quadratic in registers)."""
    root = torch.sqrt(b * b - 4 * a * c)
    return torch.stack([(-b - root) / (2 * a), (-b + root) / (2 * a)])


def find_intersection_points_with_sphere(origin, direction, sphere_radius):
    """t [n,2] and hit points [n,2,3] of lines with the origin-centred sphere (utils.py:182-217)."""
    b = 2 * (direction * origin).sum(dim=1)
    c = torch.norm(origin, dim=1) ** 2 - sphere_radius.to(origin.device).reshape(-1)[0] ** 2
    a = (direction * direction).sum(dim=1)
    t = solve_quadratic_equation(a, b, c).T
    return t, origin.unsqueeze(1) + t.unsqueeze(2) * direction.unsqueeze(1)


def sample_points_around_mean(rays_o, rays_d, mean, n_samples=32, mode="gaussian", std=0.1, noise: Optional[torch.Tensor] = None):
    """(pts [N,S,3], z_vals [N,S]) around the predicted depth (utils.py:220-244).

    ``noise`` ([N, n_samples-1] standard normal) makes gaussian mode reproducible; by default it is drawn with
    ``torch.randn`` like the reference.  When grad is enabled and ``mean`` requires it, z and pts are differentiable
    w.r.t. ``mean`` (training.PlaceFn / training.PointsFn; the rays get no gradient)."""
    if torch.is_grad_enabled() and isinstance(mean, torch.Tensor) and mean.requires_grad:
        from .. import training

        z = training.PlaceFn.apply(mean, n_samples, mode, std, noise)
        return training.PointsFn.apply(rays_o, rays_d, z), z
    z = ops.place_samples(mean, n_samples, mode, std, noise)
    return ops.points(rays_o, rays_d, z), z
