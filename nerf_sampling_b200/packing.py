"""Checkpoint tensors -> the packed weight images the tensor-core kernels stream.

``PackedNeRF`` / ``PackedDepthNet`` take reference-layout ``state_dict``s (the ``200000.tar`` keys,
nerf_pytorch/utils.py:59-122) and hold the device-side slab stream + fp32 bias/head block.  Packing itself is
done by the C ABI (``b200nerf_nerf_pack_multires`` / ``b200nerf_depthnet_pack_multires``); the only arithmetic here is the fp64
folding of DepthNet's activation-free branches into its first dense layer.
"""

from __future__ import annotations

import ctypes as C
from typing import Dict, List

import torch

from . import _lib

PREC_SPLIT = 1  # bf16 hi+lo operands, 3 MMAs per K16 block (exact mode, ~16 mantissa bits)
PREC_FP16 = 2   # fp16 operands, 1 MMA per K16 block, throughput kernel, no guard band (PSNR-level parity)
PREC_FAST = 3   # PREC_FP16 + split-precision re-evaluation of the guard band: meets the 1e-3 max-abs contract
GUARD_KAPPA = 1.0 / 32.0  # |sigma_last| < kappa * sum|h7 * w_alpha| is re-evaluated in split precision

NERF_KEYS = (
    [f"pts_linears.{i}.{w}" for i in range(8) for w in ("weight", "bias")]
    + [f"{n}.{w}" for n in ("views_linears.0", "feature_linear", "alpha_linear", "rgb_linear") for w in ("weight", "bias")]
)
NERF_MULTIRES_RANGE = range(1, 11)        # gamma(pts) is 3 (1 + 2 multires) <= 64 columns: its operand block
NERF_MULTIRES_VIEWS_RANGE = range(1, 5)   # gamma(viewdir) is 3 (1 + 2 multires_views) <= 32 columns


def nerf_shapes(multires: int = 10, multires_views: int = 4) -> Dict[str, tuple]:
    """The weight shapes of NeRF(D=8, W=256, input_ch=3(1+2 multires), input_ch_views=3(1+2 multires_views), skips=[4])."""
    d, dv = 3 * (1 + 2 * multires), 3 * (1 + 2 * multires_views)
    return {"pts_linears.0.weight": (256, d), "pts_linears.5.weight": (256, 256 + d), "views_linears.0.weight": (128, 256 + dv),
            "feature_linear.weight": (256, 256), "alpha_linear.weight": (1, 256), "rgb_linear.weight": (3, 128)}


def _octaves(width: int, what: str, name: str, rng: range) -> int:
    m, rest = divmod(width - 3, 6)
    if rest or m not in rng:
        raise ValueError(f"{what} is {width} wide, which is no encoding the NeRF kernels serve: 3 * (1 + 2 * {name}) with {name} "
                         f"in {rng.start}..{rng.stop - 1}")
    return m


def nerf_multires(state_dict: Dict[str, torch.Tensor]):
    """(multires, multires_views) of a NeRF state_dict, from pts_linears.0 (input_ch = 3 (1 + 2 multires)) and views_linears.0
    (256 + input_ch_views); pts_linears.5 must agree (256 + input_ch), as must every other shape."""
    m = _octaves(state_dict["pts_linears.0.weight"].shape[-1], "gamma(pts) (pts_linears.0 in_features)", "multires",
                 NERF_MULTIRES_RANGE)
    mv = _octaves(state_dict["views_linears.0.weight"].shape[-1] - 256, "gamma(viewdir) (views_linears.0 in_features - 256)",
                  "multires_views", NERF_MULTIRES_VIEWS_RANGE)
    for k, shp in nerf_shapes(m, mv).items():
        if tuple(state_dict[k].shape) != shp:
            raise ValueError(f"{k} has shape {tuple(state_dict[k].shape)}, expected {shp} (multires {m}, multires_views {mv})")
    return m, mv


_GENERATION = 0


def mark_updated(params) -> None:
    """Tell the pack caches that ``params`` were rewritten through raw device pointers.

    ``NeRF.packed()`` / ``DepthNet.packed()`` key their packed images on ``(data_ptr, _version)`` of every parameter.
    torch bumps ``_version`` on its own in-place ops, but the library's fused Adam (``b200nerf_adam_step_multi_dev``) and
    CUDA-graph replays write behind torch's back; every such writer calls this, which bumps the version counters (one
    batched call) or, if this torch build lacks the hook, a global generation that is part of every cache key."""
    global _GENERATION
    params = [p for p in params if isinstance(p, torch.Tensor)]
    try:
        torch._C._autograd._unsafe_set_version_counter(params, [p._version + 1 for p in params])
    except Exception:
        _GENERATION += 1


def generation() -> int:
    return _GENERATION


def _host_f32(t: torch.Tensor) -> torch.Tensor:
    return t.detach().to(device="cpu", dtype=torch.float32).contiguous()


def _ptr_array(tensors: List[torch.Tensor]):
    arr = (C.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])
    return arr


class PackedNeRF:
    """Device image of NeRF(D=8, W=256, input_ch=3(1+2m), input_ch_views=3(1+2mv), skips=[4], use_viewdirs=True), m = multires in
    1..10 and mv = multires_views in 1..4 (from the weight shapes, see nerf_multires); the aux block records both for the kernels."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], device, prec: int = PREC_SPLIT):
        L = _lib.lib()
        for k in NERF_KEYS:
            if k not in state_dict:
                raise KeyError(f"NeRF state_dict lacks {k!r}: only the 8x256 skip@4 view-dependent model is supported")
        self.multires, self.multires_views = nerf_multires(state_dict)
        mr = (self.multires, self.multires_views)
        host = [_host_f32(state_dict[k]) for k in NERF_KEYS]
        arr = C.cast(_ptr_array(host), C.c_void_p)
        aux = torch.empty(L.b200nerf_nerf_aux_floats(), dtype=torch.float32)
        self.prec = prec
        self.wpack = None       # split-precision stream of the exact kernel (mlp_exact.cuh): PREC_SPLIT and the guard band of PREC_FAST
        self.wpack_fast = None  # single-pass fp16 stream of the throughput kernel (mlp_fast.cuh)
        wpack = torch.empty(L.b200nerf_nerf_wpack_bytes(PREC_SPLIT), dtype=torch.uint8)
        _lib.check(L.b200nerf_nerf_pack_multires(arr, *mr, PREC_SPLIT, wpack.data_ptr(), aux.data_ptr()))   # also the fp32 bias / head block
        if prec != PREC_FP16:
            self.wpack = wpack.to(device)
        if prec in (PREC_FP16, PREC_FAST):
            wf = torch.empty(L.b200nerf_nerf_fast_wpack_bytes(), dtype=torch.uint8)
            _lib.check(L.b200nerf_nerf_pack_fast_multires(arr, *mr, PREC_FP16, wf.data_ptr()))
            self.wpack_fast = wf.to(device)
        self.aux = aux.to(device)
        self.guard_kappa = GUARD_KAPPA

    def c_model(self) -> "_lib.NerfModel":
        """The ``b200nerf_nerf_model`` descriptor of this image (pass with ctypes.byref)."""
        return _lib.NerfModel(
            None if self.wpack is None else self.wpack.data_ptr(),
            None if self.wpack_fast is None else self.wpack_fast.data_ptr(),
            self.aux.data_ptr(), int(self.prec), float(self.guard_kappa))


MULTIRES_RANGE = range(1, 11)   # positional-encoding sizes DepthNet's kernels serve: enc(o) is at most 63 <= 64 columns wide


def depthnet_multires(origin_in_features: int) -> int:
    """The ``multires`` m of a DepthNet whose ``origin_layers.0`` takes ``origin_in_features`` = 2 d3 inputs, d3 = 3 (1 + 2m)."""
    m, rest = divmod(origin_in_features - 6, 12)
    if rest or m not in MULTIRES_RANGE:
        raise ValueError(f"origin_layers.0 has {origin_in_features} in_features, which is no DepthNet with multires in 1..10 "
                         f"(2 * 3 * (1 + 2 * multires))")
    return m


def fold_depthnet(sd: Dict[str, torch.Tensor]):
    """Fold origin/direction/intersection branches and cat_layers[0] into one affine map (fp64).

    depth_nets/depth_net.py:136-163: every branch layer is ``x = Linear(cat([x, e]))`` with NO activation, so the
    branch output is affine in its encoding e; cat_layers[0] then sees an affine function of (e_o, e_d, e_i).
    Returns (w0 [256,256], b0 [256], hidden [(W [256,256], b [256])...], head_w [256], head_b [1]) over the
    kernel's column layout enc(o) | enc(d) | enc(hit_near) | enc(hit_far), 64 columns each, of which the first
    d3 = 3 (1 + 2 multires) are used (multires from ``origin_layers.0.weight``, see depthnet_multires) and the rest zero."""
    d = {k: v.detach().to("cpu", torch.float64) for k, v in sd.items()}
    m = depthnet_multires(d["origin_layers.0.weight"].shape[1])
    d3 = 3 * (1 + 2 * m)

    def branch(name: str, dim: int):
        w, b = d[f"{name}.0.weight"], d[f"{name}.0.bias"]
        if w.shape[1] != 2 * dim:
            raise ValueError(f"{name}.0.weight: unexpected in_features {w.shape[1]} (multires {m}: {2 * dim})")
        a, c = w[:, :dim] + w[:, dim:], b.clone()
        i = 1
        while f"{name}.{i}.weight" in d:
            w, b = d[f"{name}.{i}.weight"], d[f"{name}.{i}.bias"]
            h = w.shape[1] - dim
            if h != a.shape[0]:
                raise ValueError(f"{name}.{i}.weight: unexpected in_features {w.shape[1]} (multires {m}: {a.shape[0] + dim})")
            a, c = w[:, :h] @ a + w[:, h:], w[:, :h] @ c + b
            i += 1
        return a, c

    a_o, c_o = branch("origin_layers", d3)
    a_d, c_d = branch("direction_layers", d3)
    a_i, c_i = branch("intersection_layers", 2 * d3)
    wc, bc = d["cat_layers.0.weight"], d["cat_layers.0.bias"]
    h = a_o.shape[0]
    if wc.shape[1] != 3 * h + 4 * d3 or wc.shape[0] > 256:
        raise ValueError(f"cat_layers.0 shape {tuple(wc.shape)} not supported (multires {m}: in_features {3 * h + 4 * d3}, width <= 256)")
    e0 = 3 * h
    m_o = wc[:, 0:h] @ a_o + wc[:, e0 : e0 + d3]
    m_d = wc[:, h : 2 * h] @ a_d + wc[:, e0 + d3 : e0 + 2 * d3]
    m_i = wc[:, 2 * h : 3 * h] @ a_i + wc[:, e0 + 2 * d3 : e0 + 4 * d3]
    bias0 = bc + wc[:, 0:h] @ c_o + wc[:, h : 2 * h] @ c_d + wc[:, 2 * h : 3 * h] @ c_i
    n0 = wc.shape[0]
    w0 = torch.zeros(256, 256, dtype=torch.float64)
    w0[:n0, 0:d3] = m_o
    w0[:n0, 64 : 64 + d3] = m_d
    # 6-wide encoding block q holds [near xyz, far xyz]; regroup per hit point
    m_i = m_i.reshape(n0, 1 + 2 * m, 2, 3)
    w0[:n0, 128 : 128 + d3] = m_i[:, :, 0, :].reshape(n0, d3)
    w0[:n0, 192 : 192 + d3] = m_i[:, :, 1, :].reshape(n0, d3)
    b0 = torch.zeros(256, dtype=torch.float64)
    b0[:n0] = bias0

    hidden = []
    prev, i = n0, 2
    while f"cat_layers.{i}.weight" in d:
        w, b = d[f"cat_layers.{i}.weight"], d[f"cat_layers.{i}.bias"]
        if w.shape[0] > 256 or w.shape[1] != prev:
            raise ValueError(f"cat_layers.{i} shape {tuple(w.shape)} not supported")
        wp = torch.zeros(256, 256, dtype=torch.float64)
        wp[: w.shape[0], : w.shape[1]] = w
        bp = torch.zeros(256, dtype=torch.float64)
        bp[: w.shape[0]] = b
        hidden.append((wp, bp))
        prev = w.shape[0]
        i += 2
    hw = torch.zeros(256, dtype=torch.float64)
    hw[:prev] = d["to_depth.0.weight"][0]
    hb = d["to_depth.0.bias"].clone()
    f32 = lambda t: t.to(torch.float32).contiguous()  # noqa: E731
    return f32(w0), f32(b0), [(f32(w), f32(b)) for w, b in hidden], f32(hw), f32(hb)


class PackedDepthNet:
    """Device image of DepthNet for inference (branches folded, see fold_depthnet); the image records its multires."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], device, prec: int = PREC_SPLIT):
        L = _lib.lib()
        w0, b0, hidden, hw, hb = fold_depthnet(state_dict)
        multires = depthnet_multires(state_dict["origin_layers.0.weight"].shape[1])
        flat = [t for pair in hidden for t in pair]
        n_hidden = len(hidden)
        wpack = torch.empty(L.b200nerf_depthnet_wpack_bytes(n_hidden, prec), dtype=torch.uint8)
        aux = torch.empty(L.b200nerf_depthnet_aux_floats(n_hidden), dtype=torch.float32)
        arr = _ptr_array(flat) if flat else None
        _lib.check(
            L.b200nerf_depthnet_pack_multires(w0.data_ptr(), b0.data_ptr(), C.cast(arr, C.c_void_p) if flat else None, n_hidden,
                                              hw.data_ptr(), hb.data_ptr(), multires, prec, wpack.data_ptr(), aux.data_ptr())
        )
        self.prec = prec
        self.multires = multires
        self.n_hidden = n_hidden
        self.wpack = wpack.to(device)
        self.aux = aux.to(device)
        self.folded = (w0, b0, hidden, hw, hb)  # kept for tests / debugging
