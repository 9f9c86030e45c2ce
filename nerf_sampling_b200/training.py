"""Autograd plumbing of the training render (config #5): torch.autograd.Function shells around the C-ABI training
entry points of ``csrc/train.cu``.  No arithmetic happens here; tensors are marshalled, workspaces allocated.

Reference: ``Trainer.core_optimization_loop`` (nerf_pytorch/trainers/Trainer.py:506-544) back-propagates
``mse(z_dn, max_z)`` and ``mse(rgb, target)`` into DepthNet only: the NeRFs are frozen, so the colour loss reaches
DepthNet through ``rgb = sigmoid(raw_rgb(o + d * z_dn))`` (one sample per ray, nerf_utils.py:692-715).
"""

from __future__ import annotations

import ctypes as C
from typing import List

import torch

from . import _lib, packing


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptrs(tensors: List[torch.Tensor]):
    return (C.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])


def _ints(vals: List[int]):
    return (C.c_int * len(vals))(*vals)


def depthnet_arch(module):
    """(branch widths, cat widths) of a DepthNet shell, from its Linear layers."""
    hidden = [m.out_features for m in module.origin_layers]
    cat = [m.out_features for m in module.cat_layers if isinstance(m, torch.nn.Linear)]
    return hidden, cat


def depthnet_multires(module) -> int:
    """The positional-encoding size ``multires`` of a DepthNet shell, from the width of its first origin layer."""
    return packing.depthnet_multires(module.origin_layers[0].in_features)


def depthnet_params(module) -> List[torch.nn.Parameter]:
    """Parameters in the order ``b200nerf_depthnet_train_fwd`` expects (= state_dict order)."""
    out = []
    for seq in (module.origin_layers, module.direction_layers, module.intersection_layers, module.cat_layers, module.to_depth):
        for m in seq:
            if isinstance(m, torch.nn.Linear):
                out += [m.weight, m.bias]
    return out


class DepthNetTrainFn(torch.autograd.Function):
    """z [N,1] = DepthNet(rays_o, rays_d) in literal per-layer fp32 form, differentiable w.r.t. the parameters.
    ``arch`` = (branch widths, cat widths, multires)."""

    @staticmethod
    def forward(ctx, rays_o, rays_d, arch, radius, near, far, *params):
        hidden, cat, multires = arch
        L = _lib.lib()
        n = rays_o.shape[0]
        dev = rays_o.device
        for p in params:
            if p.dtype != torch.float32 or not p.is_cuda or not p.is_contiguous():
                raise _lib.B200NerfError("DepthNet parameters must be contiguous fp32 CUDA tensors")
        ws = torch.empty(L.b200nerf_depthnet_train_ws_floats_multires(n, len(hidden), _ints(hidden), len(cat), _ints(cat), multires),
                         device=dev)
        z = torch.empty(n, 1, device=dev)
        with torch.cuda.device(dev):
            _lib.check(L.b200nerf_depthnet_train_fwd_multires(_ptrs(list(params)), len(hidden), _ints(hidden), len(cat), _ints(cat),
                                                              multires, rays_o.data_ptr(), rays_d.data_ptr(), n, float(radius),
                                                              float(near), float(far), ws.data_ptr(), z.data_ptr(), _stream()))
        ctx.ws, ctx.arch, ctx.nf, ctx.n = ws, arch, (float(near), float(far)), n
        ctx.save_for_backward(*params)
        return z

    @staticmethod
    def backward(ctx, dz):
        params = ctx.saved_tensors
        hidden, cat, multires = ctx.arch
        L = _lib.lib()
        dz = dz.contiguous().float()
        # one flat buffer, parameter order: the C side zeroes it with a single memset (its split-K weight gradients and bias
        # gradients are atomic sums) and parallel.allreduce_gradients reduces it in place without a cat / copy-back
        flat = torch.empty(sum(p.numel() for p in params), device=dz.device)
        grads, off = [], 0
        for p in params:
            grads.append(flat[off:off + p.numel()].view_as(p))
            off += p.numel()
        with torch.cuda.device(dz.device):
            _lib.check(L.b200nerf_depthnet_train_bwd_multires(_ptrs(list(params)), len(hidden), _ints(hidden), len(cat), _ints(cat),
                                                              multires, ctx.n, ctx.nf[0], ctx.nf[1], ctx.ws.data_ptr(), dz.data_ptr(),
                                                              _ptrs(grads), _stream()))
        # the activations in ctx.ws stay valid: the reference back-propagates twice (retain_graph=True, Trainer.py:537-538)
        return (None, None, None, None, None, None) + tuple(grads)


# raw and d raw / d z of the frozen NeRF at one sample per ray: "split" = two launches of the fused split-precision tensor-core MLP
# kernel over the model's packed weights (primal + ReLU masks, then the tangent pass; the precision of PREC_SPLIT inference:
# bf16 hi + lo operands, fp32 accumulate), "fp32" = ~13 grouped 3xTF32 products over the fp32 tensors (b200nerf_nerf_point_jvp).
JVP_MODE = __import__("os").environ.get("B200NERF_TRAIN_JVP", "split")


def nerf_point_jvp(packed, params, rays_o, rays_d, viewdirs, z_flat, raw, draw, stream, S=1):
    """Fills raw [n*S,...,4] and draw [n*S,4] at the sample depths z_flat (n*S values, ray-major: sample r belongs to ray r // S);
    ``packed`` (a packing.PackedNeRF with a split-precision stream) selects the packed route.  Returns the workspace tensor, which
    must stay alive until the launches have run."""
    L = _lib.lib()
    n, dev = z_flat.shape[0] // S, z_flat.device
    if packed is not None and packed.wpack is not None and JVP_MODE == "split":
        ws = torch.empty(L.b200nerf_nerf_samples_jvp_packed_ws_bytes(n, S), dtype=torch.uint8, device=dev)
        _lib.check(L.b200nerf_nerf_samples_jvp_packed(packed.wpack.data_ptr(), packed.aux.data_ptr(), rays_o.data_ptr(),
                                                      rays_d.data_ptr(), viewdirs.data_ptr(), z_flat.data_ptr(), n, S, ws.data_ptr(),
                                                      raw.data_ptr(), draw.data_ptr(), stream))
        return ws
    # the packed route reads the encodings' sizes from its aux block; this one takes them from the tensors' shapes
    mr = packing.nerf_multires(dict(zip(packing.NERF_KEYS, params)))
    ws = torch.empty(L.b200nerf_nerf_samples_ws_floats_multires(n, S, *mr), device=dev)
    _lib.check(L.b200nerf_nerf_samples_jvp_multires(_ptrs(list(params)), *mr, rays_o.data_ptr(), rays_d.data_ptr(), viewdirs.data_ptr(),
                                                    z_flat.data_ptr(), n, S, ws.data_ptr(), raw.data_ptr(), draw.data_ptr(), stream))
    return ws


class NerfPointFn(torch.autograd.Function):
    """raw [N,S,4] of the frozen NeRF at p = o + d z for z [N,S] (or [N]: one sample per ray), differentiable w.r.t. z through
    the forward-mode d raw / d z.  ``packed``: the model's packing.PackedNeRF (split-precision route, see JVP_MODE) or None
    (fp32 route over ``params``)."""

    @staticmethod
    def forward(ctx, z, rays_o, rays_d, viewdirs, packed, *params):
        n = z.shape[0]
        S = z.shape[1] if z.dim() > 1 else 1
        dev = z.device
        raw = torch.empty(n, S, 4, device=dev)
        draw = torch.empty(n * S, 4, device=dev)
        zz = z.detach().reshape(-1).contiguous().float()
        with torch.cuda.device(dev):
            nerf_point_jvp(packed, params, rays_o, rays_d, viewdirs, zz, raw, draw, _stream(), S=S)
        ctx.save_for_backward(draw)
        ctx.zshape = z.shape
        return raw

    @staticmethod
    def backward(ctx, g_raw):
        (draw,) = ctx.saved_tensors
        gz = (g_raw.reshape(-1, 4) * draw).sum(-1).reshape(ctx.zshape)  # chain rule over the four outputs
        return (gz, None, None, None, None) + (None,) * 24


class NerfPtsFn(torch.autograd.Function):
    """raw [N,S,4] of the frozen NeRF at explicit points pts [N,S,3] (Trainer.run_network), differentiable w.r.t. pts through the
    Jacobian d raw / d pts [N*S,3,4] of the split-precision kernel (b200nerf_nerf_pts_jvp_packed)."""

    @staticmethod
    def forward(ctx, pts, viewdirs, packed):
        if packed.wpack is None:
            raise _lib.B200NerfError(
                f"gradients w.r.t. sample points need the split-precision weight image; this NeRF is packed at precision "
                f"{packed.prec} (PREC_FP16 = {packing.PREC_FP16} has none): use PREC_SPLIT or PREC_FAST")
        from . import ops

        L = _lib.lib()
        n, S = pts.shape[0], pts.shape[1]
        p, viewdirs = ops._dev(pts.detach(), "pts"), ops._dev(viewdirs, "viewdirs")
        dev = p.device
        raw = torch.empty(n, S, 4, device=dev)
        jac = torch.empty(n * S, 3, 4, device=dev)
        ws = torch.empty(L.b200nerf_nerf_samples_jvp_packed_ws_bytes(n, S), dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            _lib.check(L.b200nerf_nerf_pts_jvp_packed(packed.wpack.data_ptr(), packed.aux.data_ptr(), p.data_ptr(), viewdirs.data_ptr(),
                                                      n, S, ws.data_ptr(), raw.data_ptr(), jac.data_ptr(), _stream()))
        ctx.save_for_backward(jac)
        ctx.pshape = pts.shape
        return raw

    @staticmethod
    def backward(ctx, g_raw):
        (jac,) = ctx.saved_tensors
        g = (g_raw.reshape(-1, 1, 4) * jac).sum(-1)   # sum over the four outputs of d raw_c / d pts_k
        return g.reshape(ctx.pshape), None, None


class CompositeSingleFn(torch.autograd.Function):
    """raw2outputs with S == 1 (the reference's empty-interval quirk, sampling_trainer.py:178-180,220-221):
    rgb = sigmoid(raw rgb), disp = 1e10, differentiable w.r.t. raw."""

    @staticmethod
    def forward(ctx, raw, z, rays_d):
        from . import ops

        rgb, disp, *_ = ops.composite(raw.detach(), z.detach(), rays_d, white_bkgd=True)
        ctx.save_for_backward(rgb)
        return rgb, disp

    @staticmethod
    def backward(ctx, g_rgb, g_disp):
        (rgb,) = ctx.saved_tensors
        g = torch.zeros(rgb.shape[0], 1, 4, device=rgb.device)
        g[:, 0, :3] = g_rgb * rgb * (1.0 - rgb)
        return g, None, None


class CompositeFn(torch.autograd.Function):
    """raw2outputs for S >= 2 (trainers/sampling_trainer.py:153-230) -> (rgb, disp, acc, depth, weights, alphas), differentiable
    w.r.t. raw and z through b200nerf_composite_bwd.  ``noise`` [N,S] (already scaled) or None is the draw the forward used."""

    @staticmethod
    def forward(ctx, raw, z, rays_d, noise, white_bkgd):
        from . import ops

        ctx.set_materialize_grads(False)
        outs = ops.composite(raw.detach(), z.detach(), rays_d, white_bkgd, noise)
        ctx.save_for_backward(raw, z, rays_d, noise)
        ctx.white = bool(white_bkgd)
        return outs

    @staticmethod
    def backward(ctx, g_rgb, g_disp, g_acc, g_depth, g_weights, g_alphas):
        raw, z, rays_d, noise = ctx.saved_tensors
        L = _lib.lib()
        n, S = z.shape
        dev = raw.device
        f = lambda t: None if t is None else t.detach().contiguous().float()  # noqa: E731
        raw_c, z_c, rd, nz = f(raw), f(z), f(rays_d), f(noise)
        gs = [f(g) for g in (g_rgb, g_disp, g_acc, g_depth, g_weights, g_alphas)]
        g_raw = torch.empty(n, S, 4, device=dev)
        g_z = torch.empty(n, S, device=dev)
        p = lambda t: None if t is None else t.data_ptr()  # noqa: E731
        with torch.cuda.device(dev):
            _lib.check(L.b200nerf_composite_bwd(raw_c.data_ptr(), z_c.data_ptr(), rd.data_ptr(), p(nz), n, S, int(ctx.white),
                                                *[p(g) for g in gs], g_raw.data_ptr(), g_z.data_ptr(), _stream()))
        return (g_raw.reshape(raw.shape) if ctx.needs_input_grad[0] else None,
                g_z if ctx.needs_input_grad[1] else None, None, None, None)


class PlaceFn(torch.autograd.Function):
    """z [N,S] of sample_points_around_mean (ops.place_samples), differentiable w.r.t. ``mean`` (b200nerf_place_samples_bwd)."""

    @staticmethod
    def forward(ctx, mean, n_samples, mode, std, noise):
        from . import ops

        z = ops.place_samples(mean.detach(), n_samples, mode, std, noise)
        ctx.save_for_backward(mean)
        ctx.cfg = (z.shape[1], mode, float(std))
        return z

    @staticmethod
    def backward(ctx, g_z):
        from . import ops

        (mean,) = ctx.saved_tensors
        S, mode, std = ctx.cfg
        m = mean.detach().reshape(-1).contiguous().float()
        n = m.shape[0]
        grid = ops.uniform_grid(std, S, m.device) if (mode == "uniform" and S > 1) else None
        g = g_z.contiguous().float()
        g_mean = torch.empty(n, device=m.device)
        with torch.cuda.device(m.device):
            _lib.check(_lib.lib().b200nerf_place_samples_bwd(m.data_ptr(), None if grid is None else grid.data_ptr(), n, S,
                                                             ops.PLACE_MODES[mode], 2.0, 6.0, g.data_ptr(), g_mean.data_ptr(),
                                                             _stream()))
        return g_mean.reshape(mean.shape), None, None, None, None


class PointsFn(torch.autograd.Function):
    """pts [N,S,3] = o + d z (ops.points), differentiable w.r.t. z (b200nerf_points_bwd); rays get no gradient."""

    @staticmethod
    def forward(ctx, rays_o, rays_d, z):
        from . import ops

        rd = rays_d.detach().contiguous().float()
        ctx.save_for_backward(rd)
        return ops.points(rays_o.detach(), rd, z.detach())

    @staticmethod
    def backward(ctx, g_pts):
        (rd,) = ctx.saved_tensors
        n, S = g_pts.shape[0], g_pts.shape[1]
        g = g_pts.contiguous().float()
        g_z = torch.empty(n, S, device=g.device)
        with torch.cuda.device(g.device):
            _lib.check(_lib.lib().b200nerf_points_bwd(rd.data_ptr(), g.data_ptr(), n, S, g_z.data_ptr(), _stream()))
        return None, None, g_z


def nerf_params(module) -> List[torch.nn.Parameter]:
    """The 24 NeRF tensors in the order of ``b200nerf_nerf_pack``."""
    from .packing import NERF_KEYS

    sd = dict(module.named_parameters())
    return [sd[k] for k in NERF_KEYS]


# Persistent-grid cap (in SMs) of the frozen target render while the DepthNet / JVP chain of the same step runs on a side stream;
# 0 runs the step on one stream; 148 = every SM of a B200, i.e. no cap but still two streams (the best setting since the side chain
# is four fused-kernel launches; it was 128 while the chain was ~25 grouped GEMMs).  B200NERF_TARGET_SMS overrides (measurement).
TARGET_SM_LIMIT = int(__import__("os").environ.get("B200NERF_TARGET_SMS", "148"))
# The backward split at the losses (b200nerf_depthnet_train_jac / _bwd_jac): the sequential input-gradient chain runs with a unit
# upstream gradient in front of the losses -- on a third stream beside d raw / d z (THIRD_STREAM) -- and the weight-only branch
# chain beside the weight gradients after them (FORK_BRANCH_CHAIN).  Measured per graphed step, one-pass -> split:
# 512 rays 0.858 -> 0.759 ms, 1024 0.984 -> 0.831, 2048 1.202 -> 1.065, 4096 1.672 -> 1.600.  B200NERF_SPLIT_BACKWARD=0 keeps the
# one-pass backward (A/B runs); the autograd route (DepthNetTrainFn) always uses it.
SPLIT_BACKWARD = __import__("os").environ.get("B200NERF_SPLIT_BACKWARD", "1") != "0"
THIRD_STREAM = __import__("os").environ.get("B200NERF_THIRD_STREAM", "1") != "0"
FORK_BRANCH_CHAIN = __import__("os").environ.get("B200NERF_FORK_BRANCH_CHAIN", "1") != "0"
_SIDE_STREAMS = {}


def _side_stream(dev, which=0):
    s = _SIDE_STREAMS.get((dev, which))
    if s is None:
        s = _SIDE_STREAMS[(dev, which)] = torch.cuda.Stream(device=dev)
    return s


def fused_render_and_backward(trainer, optimizer, render_kwargs, batch_rays, target_s):
    """The DepthNet training render and both backward passes of ``Trainer.core_optimization_loop`` (Trainer.py:515-538) as a
    handful of C calls on three streams and no autograd graph: hierarchical arg-max target on the frozen NeRFs (tensor-core
    kernels; main stream), DepthNet forward with saved activations and the frozen fine NeRF at one sample per ray with its
    forward-mode d raw / d z (side stream), the backward's input-gradient chain with a unit upstream gradient (third stream:
    it needs neither the losses nor the colour path), then -- after the join -- both losses and the gradient they send into z in
    one kernel (``b200nerf_train_loss``) and DepthNet's weight gradients into ONE flat gradient buffer whose address never
    changes (so the optimizer's pointer table and ``parallel.allreduce_gradients`` see the same tensors every step).

    Returns ``(loss, depth_net_loss, psnr)`` as 0-dim tensors, or ``None`` when the configuration is not the standard one
    (foreign DepthNet / NeRF modules, optimizer over other parameters): the caller then takes the autograd route, which
    computes the same thing through ``DepthNetTrainFn`` / ``NerfPointFn`` / ``CompositeSingleFn``."""
    from . import ops
    from .depth_nets.depth_net import DepthNet

    dn = render_kwargs.get("depth_network")
    net = render_kwargs.get("network_fine") if render_kwargs.get("network_fine") is not None else render_kwargs.get("network_fn")
    if not isinstance(dn, DepthNet) or not hasattr(net, "query") or not render_kwargs.get("use_viewdirs", False):
        return None
    params = depthnet_params(dn)
    opt_params = [p for g in optimizer.param_groups for p in g["params"]]
    if len(opt_params) != len(params) or any(a is not b for a, b in zip(opt_params, params)):
        return None
    if any((not p.requires_grad) or p.dtype != torch.float32 or not p.is_cuda or not p.is_contiguous() for p in params):
        return None
    L = _lib.lib()
    rays_o, rays_d = batch_rays[0].contiguous().float(), batch_rays[1].contiguous().float()
    n, dev = rays_o.shape[0], rays_o.device
    target = target_s.contiguous().float()
    hidden, cat = depthnet_arch(dn)
    arch = (len(hidden), _ints(hidden), len(cat), _ints(cat), depthnet_multires(dn))
    cache = dn.__dict__.get("_b200_train_cache")
    if cache is None or cache["dev"] != dev or cache["ptrs"] != [p.data_ptr() for p in params]:
        flat = torch.zeros(sum(p.numel() for p in params), device=dev)
        grads, off = [], 0
        for p in params:
            grads.append(flat[off:off + p.numel()].view_as(p))
            off += p.numel()
        cache = dn.__dict__["_b200_train_cache"] = dict(dev=dev, ptrs=[p.data_ptr() for p in params], flat=flat, grads=grads, bounds={})
    bounds = cache["bounds"].get((n, float(render_kwargs["near"]), float(render_kwargs["far"])))
    if bounds is None:
        bounds = cache["bounds"][(n, float(render_kwargs["near"]), float(render_kwargs["far"]))] = (
            torch.full((n, 1), float(render_kwargs["near"]), device=dev), torch.full((n, 1), float(render_kwargs["far"]), device=dev))
    with torch.no_grad(), torch.cuda.device(dev):
        viewdirs = ops.normalize_dirs(rays_d)
        kw = render_kwargs
        hier = dict(near=bounds[0], far=bounds[1])
        p_arr = _ptrs(params)
        nf = (float(dn.near), float(dn.far))
        main = torch.cuda.current_stream()
        # Two independent halves until the losses: the frozen hierarchical target (throughput-bound persistent kernels) and the
        # DepthNet forward + NeRF point JVP (a latency-bound chain of ~10 launches).  The chain runs on a side stream beside the
        # target, whose persistent grids can be capped so that it finds free SMs (TARGET_SM_LIMIT; 0 = one stream).
        side = _side_stream(dev) if TARGET_SM_LIMIT > 0 else None
        # every buffer is allocated on the main stream (the side stream only runs kernels between the two wait_stream calls), so the
        # caching allocator never sees a cross-stream hand-off
        ws = torch.empty(L.b200nerf_depthnet_train_ws_floats_multires(n, *arch), device=dev)
        z = torch.empty(n, 1, device=dev)
        net_packed = net.packed() if hasattr(net, "packed") else None   # before the fork: a repack allocates and copies on the main stream
        net_params = nerf_params(net)
        raw = torch.empty(n, 1, 4, device=dev)
        draw = torch.empty(n, 4, device=dev)
        if side is not None:
            side.wait_stream(main)
        st = side.cuda_stream if side is not None else main.cuda_stream
        _lib.check(L.b200nerf_depthnet_train_fwd_multires(p_arr, *arch, rays_o.data_ptr(), rays_d.data_ptr(), n, float(dn.sphere_radius),
                                                          nf[0], nf[1], ws.data_ptr(), z.data_ptr(), st))
        g_arr = _ptrs(cache["grads"])
        split_bwd = SPLIT_BACKWARD
        side2 = _side_stream(dev, 1) if (side is not None and split_bwd and THIRD_STREAM) else None
        if side2 is not None:
            side2.wait_stream(side)
        ws_n = nerf_point_jvp(net_packed, net_params, rays_o, rays_d, viewdirs, z.reshape(-1), raw, draw, st)   # noqa: F841 (kept alive)
        if split_bwd:
            # the backward's sequential half (input-gradient chain with a unit upstream gradient) needs neither the losses nor the
            # colour path: it runs beside d raw / d z on a third stream
            _lib.check(L.b200nerf_depthnet_train_jac_multires(p_arr, *arch, n, nf[0], nf[1], ws.data_ptr(), g_arr,
                                                              side2.cuda_stream if side2 is not None else st))
        prev_limit = L.b200nerf_set_sm_limit(TARGET_SM_LIMIT) if side is not None else 0
        try:
            c = trainer.sample_coarse_points(near=hier["near"], far=hier["far"], perturb=kw["perturb"], N_rays=n, N_samples=kw["N_samples"],
                                             viewdirs=viewdirs, network_fn=kw["network_fn"], network_query_fn=kw["network_query_fn"],
                                             rays_o=rays_o, rays_d=rays_d, raw_noise_std=kw["raw_noise_std"], white_bkgd=kw["white_bkgd"],
                                             pytest=False, lindisp=kw.get("lindisp", False))
            f = trainer.sample_fine_points(z_vals=c[5], weights=c[6], perturb=kw["perturb"], pytest=False, rays_d=rays_d, rays_o=rays_o,
                                           rgb_map=c[0], disp_map=c[1], acc_map=c[2], network_fn=kw["network_fn"],
                                           network_fine=kw["network_fine"], network_query_fn=kw["network_query_fn"], viewdirs=viewdirs,
                                           raw_noise_std=kw["raw_noise_std"], white_bkgd=kw["white_bkgd"])
            _, max_z, _, _ = ops.argmax_gather(f[11], f[7])
        finally:
            if side is not None:
                L.b200nerf_set_sm_limit(prev_limit)
        if side is not None:
            main.wait_stream(side)
        if side2 is not None:
            main.wait_stream(side2)
        st = main.cuda_stream
        losses = torch.empty(3, device=dev)
        dz = torch.empty(n, device=dev)
        ws2 = torch.empty(2, device=dev)
        _lib.check(L.b200nerf_train_loss(raw.data_ptr(), draw.data_ptr(), z.data_ptr(), max_z.data_ptr(), target.data_ptr(), n,
                                         ws2.data_ptr(), losses.data_ptr(), dz.data_ptr(), st))
        if split_bwd:
            aux = side.cuda_stream if (side is not None and FORK_BRANCH_CHAIN) else None   # idle after the join above
            _lib.check(L.b200nerf_depthnet_train_bwd_jac_multires(p_arr, *arch, n, nf[0], nf[1], ws.data_ptr(), dz.data_ptr(), g_arr,
                                                                  st, aux))
        else:
            _lib.check(L.b200nerf_depthnet_train_bwd_multires(p_arr, *arch, n, nf[0], nf[1], ws.data_ptr(), dz.data_ptr(), g_arr, st))
    for p, g in zip(params, cache["grads"]):
        if p.grad is not g:
            p.grad = g
    return losses[0], losses[1], losses[2]


class Adam(torch.optim.Optimizer):
    """torch.optim.Adam semantics (no weight decay, no amsgrad) on the library's fused kernel: ONE launch updates every
    tensor of a parameter group.  ``grad_scale`` multiplies every gradient first (1 / world_size after a sum all-reduce).

    The step counter and the hyper-parameters live in device memory (like ``torch.optim.Adam(capturable=True)``), so
    ``step()`` can be captured in a CUDA graph: the graph re-reads ``lr`` / ``grad_scale`` from a pinned host buffer on every
    replay.  ``state[p]["step"]`` is a 0-dim device tensor shared by the tensors of a group."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8):
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps))

    def _group_buffers(self, gi: int, group, dev):
        bufs = self.__dict__.setdefault("_b200_bufs", {})
        buf = bufs.get(gi)
        if buf is None:
            n = len(group["params"])
            buf = dict(step=torch.zeros((), dtype=torch.int32, device=dev), hyper=torch.zeros(5, device=dev),
                       # eager steps rotate through pinned blocks, each guarded by an event recorded after its upload: the
                       # CPU never rewrites a block whose host->device copy may still be pending
                       hyper_ring=[[torch.zeros(5).pin_memory(), None] for _ in range(4)], hyper_slot=0,
                       # the block a captured graph's memcpy node re-reads on every replay (set_hyper rewrites it)
                       hyper_host=torch.zeros(5).pin_memory(),
                       ptrs=None, table=None, table_host=None,
                       # used only while a CUDA graph is being captured (no page-locked allocation may happen then, and the
                       # graph's memcpy node re-reads this buffer on every replay, so eager steps must never touch it)
                       graph_table_host=torch.zeros(n, 5, dtype=torch.int64).pin_memory(),
                       graph_table=torch.zeros(n, 5, dtype=torch.int64, device=dev))
            bufs[gi] = buf
        return buf

    def _rows(self, group):
        rows, dev = [], None
        for p in group["params"]:
            if p.grad is None:
                continue
            dev = p.device
            st = self.state[p]
            if "exp_avg" not in st:
                st["exp_avg"] = torch.zeros_like(p)
                st["exp_avg_sq"] = torch.zeros_like(p)
            g = p.grad if p.grad.is_contiguous() else p.grad.contiguous()
            rows.append((p, g, st))
        return rows, dev

    @staticmethod
    def _table_ptrs(rows):
        return [x for p, g, st in rows for x in (p.data_ptr(), g.data_ptr(), st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr(), p.numel())]

    @torch.no_grad()
    def stage_for_capture(self, grad_scale: float = 1.0):
        """While a CUDA graph is being captured: put the uploads ``step`` needs -- the pointer table and the hyper-parameter block
        the graph re-reads from pinned memory on every replay -- on a forked stream at the START of the step.  Two memcpy nodes
        in front of the Adam launch cost ~20 us of the step's critical path; here they run under the render.  ``step`` joins the
        fork.  Gradients must already exist at their final addresses (they do after a warm-up step of the fused route)."""
        if not torch.cuda.is_current_stream_capturing():
            return
        cur = torch.cuda.current_stream()
        fork = self.__dict__.get("_b200_stage_stream")
        if fork is None or fork.device != cur.device:
            fork = self.__dict__["_b200_stage_stream"] = torch.cuda.Stream(device=cur.device)
        fork.wait_stream(cur)
        staged = {}
        with torch.cuda.stream(fork):
            for gi, group in enumerate(self.param_groups):
                rows, dev = self._rows(group)
                if not rows:
                    continue
                buf = self._group_buffers(gi, group, dev)
                ptrs = self._table_ptrs(rows)
                host = buf["graph_table_host"][: len(rows)]
                host.view(-1).numpy()[:] = ptrs
                table = buf["graph_table"][: len(rows)]
                table.copy_(host, non_blocking=True)
                b1, b2 = group["betas"]
                buf["hyper_host"].numpy()[:] = [float(group["lr"]), float(b1), float(b2), float(group["eps"]), float(grad_scale)]
                buf["hyper"].copy_(buf["hyper_host"], non_blocking=True)   # a memcpy node that re-reads the host values on every replay
                staged[gi] = ptrs
        self.__dict__["_b200_staged"] = (fork, staged)

    @torch.no_grad()
    def step(self, closure=None, grad_scale: float = 1.0):
        L = _lib.lib()
        capturing = torch.cuda.is_current_stream_capturing()
        fork, staged = self.__dict__.pop("_b200_staged", (None, {})) if capturing else (None, {})
        if fork is not None:
            torch.cuda.current_stream().wait_stream(fork)
        for gi, group in enumerate(self.param_groups):
            b1, b2 = group["betas"]
            rows, dev = self._rows(group)
            if not rows:
                continue
            buf = self._group_buffers(gi, group, dev)
            for p, g, st in rows:
                prev = st.get("step")
                if prev is not buf["step"]:
                    if prev is not None and int(prev) > int(buf["step"]):   # state loaded from a torch checkpoint
                        buf["step"].fill_(int(prev))
                    st["step"] = buf["step"]
            with torch.cuda.device(dev):
                ptrs = self._table_ptrs(rows)
                vals = [float(group["lr"]), float(b1), float(b2), float(group["eps"]), float(grad_scale)]
                if capturing and staged.get(gi) == ptrs:
                    # uploads already captured by stage_for_capture; the host block is plain memory: keep it current
                    table = buf["graph_table"][: len(rows)]
                    buf["hyper_host"].numpy()[:] = vals
                elif capturing:
                    host = buf["graph_table_host"][: len(rows)]
                    host.view(-1).numpy()[:] = ptrs
                    table = buf["graph_table"][: len(rows)]
                    table.copy_(host, non_blocking=True)
                    hh = buf["hyper_host"]
                    hh.numpy()[:] = vals
                    buf["hyper"].copy_(hh, non_blocking=True)   # a memcpy node that re-reads the host values on every replay
                else:
                    if ptrs != buf["ptrs"]:
                        # gradients are new tensors after an eager backward: refresh the pointer table (a fresh pinned buffer
                        # per refresh: the previous upload may still be in flight)
                        host = torch.tensor(ptrs, dtype=torch.int64).reshape(len(rows), 5).pin_memory()
                        buf["table_host"], buf["ptrs"] = host, ptrs
                        buf["table"] = host.to(dev, non_blocking=True)
                        buf["keep"] = [g for _, g, _ in rows]
                    table = buf["table"]
                    slot = buf["hyper_ring"][buf["hyper_slot"]]
                    buf["hyper_slot"] = (buf["hyper_slot"] + 1) % len(buf["hyper_ring"])
                    if slot[1] is not None:
                        slot[1].synchronize()
                    slot[0].numpy()[:] = vals
                    buf["hyper"].copy_(slot[0], non_blocking=True)
                    slot[1] = torch.cuda.Event()
                    slot[1].record()
                _lib.check(L.b200nerf_adam_step_multi_dev(table.data_ptr(), len(rows), buf["hyper"].data_ptr(),
                                                          buf["step"].data_ptr(), _stream()))
            # the kernel wrote the parameters through raw pointers: invalidate the packed inference images
            packing.mark_updated([p for p, _, _ in rows])
        return None

    def params(self):
        return [p for g in self.param_groups for p in g["params"]]

    @torch.no_grad()
    def init_state(self):
        """Create the moment buffers and resolve a checkpoint-loaded step count now (both would otherwise happen lazily inside
        ``step``, which must not allocate pinned memory or synchronise while a CUDA graph is being captured)."""
        for gi, group in enumerate(self.param_groups):
            ps = [p for p in group["params"] if p.requires_grad]
            if not ps:
                continue
            buf = self._group_buffers(gi, group, ps[0].device)
            for p in ps:
                st = self.state[p]
                if "exp_avg" not in st:
                    st["exp_avg"] = torch.zeros_like(p)
                    st["exp_avg_sq"] = torch.zeros_like(p)
                prev = st.get("step")
                if prev is not buf["step"]:
                    if prev is not None and int(prev) > int(buf["step"]):
                        buf["step"].fill_(int(prev))
                    st["step"] = buf["step"]

    def set_hyper(self, grad_scale: float = None):
        """Refresh the pinned hyper-parameter block before replaying a captured step (lr may have been changed on the group);
        ``grad_scale=None`` keeps the value the capture recorded."""
        for gi, group in enumerate(self.param_groups):
            buf = self.__dict__.get("_b200_bufs", {}).get(gi)
            if buf is not None:
                b1, b2 = group["betas"]
                hh = buf["hyper_host"]
                vals = [float(group["lr"]), float(b1), float(b2), float(group["eps"]), float(hh[4]) if grad_scale is None else float(grad_scale)]
                if hh.tolist() != [float(torch.tensor(v, dtype=torch.float32)) for v in vals]:
                    # a replay still in flight may be about to read the block: drain it before the (rare) rewrite
                    torch.cuda.current_stream().synchronize()
                    hh.numpy()[:] = vals


class GraphedTrainStep:
    """``Trainer.core_optimization_loop`` as ONE CUDA graph: training render, zero_grad, both backward passes, the flat NCCL
    gradient all-reduce and the fused Adam step (~90 launches, launch-bound from Python at 512 rays per GPU).

        step = GraphedTrainStep(trainer, sampling_optimizer, render_kwargs_train, n_rays)
        loss, depth_net_loss, psnr = step(batch_rays, target_s)      # fresh 0-dim tensors (no host sync)

    Adam's step counter and hyper-parameters live in device memory and the graph re-reads ``lr`` / ``grad_scale`` from a pinned
    block on every replay, so learning-rate schedules keep working.  NCCL collectives are capturable; set
    ``capture_step=False`` (or ``B200NERF_GRAPH_COLLECTIVE=0``) to keep the all-reduce and Adam eager after the replay.
    Batch shape is fixed at construction; ``perturb`` must be 0 (random draws would be frozen into the graph)."""

    def __init__(self, trainer, optimizer, render_kwargs_train, n_rays: int, warmup: int = 3, capture_step=None):
        import os

        dev = next(p for g in optimizer.param_groups for p in g["params"]).device
        self.trainer, self.opt, self.kw = trainer, optimizer, render_kwargs_train
        self.rays = torch.zeros(2, n_rays, 3, device=dev)
        self.rays[0, :, 2] = 4.0    # placeholder rays for the warm-up steps: straight at the unit sphere
        self.rays[1, :, 2] = -1.0
        self.target = torch.zeros(n_rays, 3, device=dev)
        self.graph = None
        self.warmup = warmup
        self.out = None
        if capture_step is None:
            capture_step = os.environ.get("B200NERF_GRAPH_COLLECTIVE", "1") != "0"
        self.capture_step = bool(capture_step) and isinstance(optimizer, Adam)
        self.params = [p for g in optimizer.param_groups for p in g["params"]]

    def _capture(self):
        import torch.distributed as dist

        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for i in range(self.warmup):   # lazy initialisation (function attributes, cached grids) must not be captured
                self.trainer.render_and_backward(self.opt, self.kw, (self.rays[0], self.rays[1]), i, self.target)
            if self.capture_step:
                self.opt.init_state()      # moment buffers and a possibly checkpoint-loaded step count, outside the capture
                if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
                    dist.all_reduce(torch.zeros(1, device=self.rays.device))   # the communicator must exist before capture
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, capture_error_mode="thread_local"):
            if self.capture_step:
                world = dist.get_world_size() if (dist.is_available() and dist.is_initialized()) else 1
                self.opt.stage_for_capture(grad_scale=1.0 / world)   # Adam's uploads, forked to the start of the step
            loss, dn_loss, psnr, _ = self.trainer.render_and_backward(self.opt, self.kw, (self.rays[0], self.rays[1]), 100, self.target)
            if self.capture_step:
                self.trainer.reduce_and_step(self.opt)
            self.out = torch.stack([loss.detach(), dn_loss.detach(), psnr.detach()])

    def __call__(self, batch_rays, target_s):
        if self.graph is None:
            self._capture()
        self.rays[0].copy_(batch_rays[0])
        self.rays[1].copy_(batch_rays[1])
        self.target.copy_(target_s)
        if self.capture_step:
            self.opt.set_hyper()                  # lr may have been changed on the param group since the last replay
        self.graph.replay()                       # gradients land in the tensors the capture allocated (static addresses)
        if self.capture_step:
            packing.mark_updated(self.params)     # the replayed Adam wrote the weights behind torch's back
        else:
            self.trainer.reduce_and_step(self.opt)    # flat NCCL all-reduce + fused Adam, eager
        out = self.out.clone()                    # the graph's output buffer is overwritten by the next replay
        return out[0], out[1], out[2]
