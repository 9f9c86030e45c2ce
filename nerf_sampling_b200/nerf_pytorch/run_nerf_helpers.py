"""Mirror of ``nerf_sampling/nerf_pytorch/run_nerf_helpers.py`` for the hot path.

``NeRF`` keeps the reference's constructor, attribute names and ``state_dict`` keys (so ``200000.tar`` loads
verbatim) but owns no arithmetic: the positional encoding and all twelve linear layers run inside the fused
tcgen05 kernels (``b200nerf_nerf_query``), fed from a packed weight image cached on the module.
"""

from __future__ import annotations

import numpy as np
import torch
import torch.nn as nn

from .. import ops, packing
from ..packing import PREC_FAST, PackedNeRF

img2mse = lambda x, y: torch.mean((x - y) ** 2)  # noqa: E731  (run_nerf_helpers.py:9)
# run_nerf_helpers.py:10 divides by torch.log(torch.Tensor([10.])) created on the fly: on a GPU that is a pageable
# host->device copy, i.e. a stream synchronisation in the middle of every training step.  Same value, no copy:
_LOG10 = float(torch.log(torch.tensor([10.0])))
mse2psnr = lambda x: -10.0 * torch.log(x) / _LOG10  # noqa: E731
to8b = lambda x: (255 * np.clip(x, 0, 1)).astype(np.uint8)  # noqa: E731


class Embedder:
    """Descriptor of a positional encoding (run_nerf_helpers.py:15-45).

    The kernels fuse the encoding; this object only carries (multires, input_dims, out_dim) to the call sites
    that the reference wires through ``embed_fn`` / ``embeddirs_fn``.  Calling it materialises the encoding with
    torch ops for inspection -- it is not on the render path."""

    def __init__(self, multires: int, input_dims: int):
        self.multires = multires
        self.input_dims = input_dims
        self.out_dim = input_dims * (1 + 2 * multires)

    def __call__(self, x: torch.Tensor) -> torch.Tensor:
        out = [x]
        for j in range(self.multires):
            out += [torch.sin(x * float(2**j)), torch.cos(x * float(2**j))]
        return torch.cat(out, -1)

    embed = __call__


def get_embedder(multires, i=0, input_dims=4):
    """(embed_fn, out_dim), signature of run_nerf_helpers.py:48-63."""
    if i == -1:
        return nn.Identity(), 3
    e = Embedder(multires, input_dims)
    return e, e.out_dim


_INPUT_CH = {3 * (1 + 2 * m) for m in packing.NERF_MULTIRES_RANGE}
_INPUT_CH_VIEWS = {3 * (1 + 2 * m) for m in packing.NERF_MULTIRES_VIEWS_RANGE}


class NeRF(nn.Module):
    """Parameter shell of the 8x256 skip@4 view-dependent NeRF MLP (run_nerf_helpers.py:67-134)."""

    def __init__(self, D=8, W=256, input_ch=3, input_ch_views=3, output_ch=4, skips=[4], use_viewdirs=False):
        super().__init__()
        self.D, self.W = D, W
        self.input_ch, self.input_ch_views = input_ch, input_ch_views
        self.skips, self.use_viewdirs = skips, use_viewdirs
        self.pts_linears = nn.ModuleList(
            [nn.Linear(input_ch, W)]
            + [nn.Linear(W, W) if i not in self.skips else nn.Linear(W + input_ch, W) for i in range(D - 1)]
        )
        self.views_linears = nn.ModuleList([nn.Linear(input_ch_views + W, W // 2)])
        if use_viewdirs:
            self.feature_linear = nn.Linear(W, W)
            self.alpha_linear = nn.Linear(W, 1)
            self.rgb_linear = nn.Linear(W // 2, 3)
        else:
            self.output_linear = nn.Linear(W, output_ch)
        self.precision = PREC_FAST  # fp16 single pass + split-precision guard band; PREC_SPLIT = split everywhere
        self._packed = None
        self._packed_key = None

    def multires(self):
        """(multires, multires_views) of this net's encodings: input_ch = 3 (1 + 2 multires), input_ch_views likewise."""
        self._check_supported()
        return (self.input_ch - 3) // 6, (self.input_ch_views - 3) // 6

    def _check_supported(self):
        if not (self.D == 8 and self.W == 256 and self.input_ch in _INPUT_CH and self.input_ch_views in _INPUT_CH_VIEWS
                and list(self.skips) == [4] and self.use_viewdirs):
            raise NotImplementedError(
                "the B200 kernel implements NeRF(D=8, W=256, input_ch=3*(1+2*multires), input_ch_views=3*(1+2*multires_views), "
                "skips=[4], use_viewdirs=True) with multires in 1..10 and multires_views in 1..4 (the positional encodings of "
                f"experiments/run.py and render.py); got D={self.D}, W={self.W}, input_ch={self.input_ch}, "
                f"input_ch_views={self.input_ch_views}, skips={list(self.skips)}, use_viewdirs={self.use_viewdirs}")

    def packed(self) -> PackedNeRF:
        """Packed weight image for the current parameter values (rebuilt when a parameter changes)."""
        self._check_supported()
        params = list(self.parameters())
        key = (self.precision, packing.generation()) + tuple((p.data_ptr(), p._version) for p in params)
        if self._packed is None or key != self._packed_key:
            self._packed = PackedNeRF(self.state_dict(), params[0].device, self.precision)
            self._packed_key = key
        return self._packed

    def query(self, viewdirs, *, rays_o=None, rays_d=None, z=None, pts=None):
        """raw [N,S,4] for sample positions o + d*z (or explicit pts) with fused encodings.  When ``z`` or ``pts``
        carries a gradient (the training render through the frozen NeRF, nerf_utils.py:692-715, or a user objective
        through the S-sample render) the forward-mode route evaluates raw at split precision together with d raw / d z
        (training.NerfPointFn) or d raw / d pts (training.NerfPtsFn).  The NeRF's own parameters get no gradient."""
        if torch.is_grad_enabled():
            from .. import training

            if z is not None and z.requires_grad:
                return training.NerfPointFn.apply(z, rays_o.contiguous().float(), rays_d.contiguous().float(),
                                                  viewdirs.contiguous().float(), self.packed(), *training.nerf_params(self))
            if z is None and pts is not None and pts.requires_grad:
                return training.NerfPtsFn.apply(pts, viewdirs, self.packed())
        return ops.nerf_mlp(self.packed(), viewdirs, rays_o=rays_o, rays_d=rays_d, z=z, pts=pts)

    def forward(self, x):
        raise NotImplementedError(
            "NeRF.forward on pre-encoded [P,90] inputs is not part of the B200 path: the encoding is fused into the "
            "MLP kernel.  Call Trainer.run_network(pts, viewdirs, model, ...) or NeRF.query(...) instead.")


def get_rays(H, W, K, c2w):
    """rays_o, rays_d [H,W,3] (run_nerf_helpers.py:187-202), generated on the device."""
    dev = c2w.device if isinstance(c2w, torch.Tensor) and c2w.is_cuda else "cuda"
    ro, rd, _ = ops.get_rays(H, W, K, c2w, dev)
    return ro.reshape(H, W, 3), rd.reshape(H, W, 3)


def sample_pdf(bins, weights, N_samples, det=False, pytest=False):
    """Inverse-CDF sampling, signature of run_nerf_helpers.py:250-293 (``pytest`` is unusable in the reference --
    it promotes to float64 and crashes -- and is ignored here)."""
    u = None if det else torch.rand(list(bins.shape[:-1]) + [N_samples], device=bins.device)
    return ops.sample_pdf(bins, weights, N_samples, u)
