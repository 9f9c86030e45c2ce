"""The differentiable S-sample DepthNet render (DESIGN.md §7b): raw2outputs, sample placement and NeRF queries under autograd.

The reference composes a DepthNet objective from plain torch operators -- DepthNet(rays) -> sample_points_around_mean ->
Trainer.run_network (or NeRF.query on depths) -> DepthNetTrainer.raw2outputs -> a loss -- so autograd reaches DepthNet's
parameters through every one of them.  Each operator here is held against torch autograd on ``oracle.nerf_oracle`` in fp64:

  * the composite backward (b200nerf_composite_bwd, training.CompositeFn) at S in {2, 3, 32, 64, 128, 192}, white background on
    and off, noise on and off, each upstream gradient alone and all six together, with rays whose alphas saturate so that the
    transmittance underflows in fp32; bound 1e-4 of each output tensor's largest entry, rays with |sigma_last| < 1e-5 excluded and
    counted (the knife edge of DESIGN.md §2: there d alpha / d sigma = 1e10 |d|);
  * d raw / d z at S samples per ray on both routes (the packed split-precision kernel, the fp32 products), d raw / d pts on the
    packed kernel, with the per-channel 1e-3 bound and the ReLU-kink accounting of test_gpu_parity.test_nerf_point_jvp_vs_torch;
  * the placement backward in all three modes against torch autograd on oracle.place_samples, including samples clipped onto 2
    and 6;
  * the whole reference composition, on the 10x256 DepthNet with the seeded NeRF and on a multires-5 NeRF + DepthNet: every
    DepthNet gradient against fp64 on rays free of LeakyReLU kinks (the screen of test_depthnet_architectures.py), through
    the pts route and the z route.
"""

import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from oracle import nerf_oracle as O

DEV = "cuda"
TAU_COMP = 1e-4    # composite backward: per output tensor, of its largest entry
KNIFE = 1e-5       # |sigma_last| below this: the last interval's 1e10 makes d alpha / d sigma ill-conditioned
TAU_JVP = 1e-3     # d raw / d z, d raw / d pts: per channel, of its largest derivative (test_gpu_parity)
TAU = 1e-4         # DepthNet kink screen: |pre-activation| > TAU * rms(layer) on every cat layer (test_depthnet_architectures)
TAU_G = 3e-3       # whole path: DepthNet gradients, per tensor, of its largest entry.  Not 1e-4: every ray's d loss / d mean
                   # carries the split-precision NeRF derivative's error (up to ~1e-3 of a channel's largest, the d raw / d z tests),
                   # and tensors whose gradient nearly cancels over the rays (the direction branch: largest entry ~1e-9) see it
                   # amplified.  Measured on a B200 (1000 W power limit), worst tensor of the reference models: 1.04e-3, on a
                   # direction-branch tensor whose largest entry is 1e-9; the multires-5 models: 3.6e-5.


def d_of(m):
    return 3 * (1 + 2 * m)


# --------------------------------------------------------------------------------------------- CPU: C ABI, workspaces, dispatch
def test_c_abi_refusals(lib):
    from nerf_sampling_b200 import _lib

    def err():
        return lib.b200nerf_last_error().decode()

    x = torch.zeros(64)
    p = x.data_ptr()
    assert lib.b200nerf_composite_bwd(p, p, p, None, 4, 1, 1, None, None, None, None, None, None, p, p, None) != 0
    assert "S >= 2" in err() and "S=1" in err()
    assert lib.b200nerf_composite_bwd(p, p, p, None, -1, 4, 1, None, None, None, None, None, None, p, p, None) != 0
    assert "bad sizes" in err()
    assert lib.b200nerf_composite_bwd(p, None, p, None, 4, 4, 1, None, None, None, None, None, None, p, p, None) != 0
    assert "null argument" in err()
    assert lib.b200nerf_composite_bwd(p, p, p, None, 4, 4, 1, None, None, None, None, None, None, p, None, None) != 0
    assert "null argument" in err()
    assert lib.b200nerf_composite_bwd(None, None, None, None, 0, 4, 1, None, None, None, None, None, None, None, None, None) == 0

    assert lib.b200nerf_place_samples_bwd(p, p, 4, 4, 7, 2.0, 6.0, p, p, None) != 0 and "unknown mode 7" in err()
    assert lib.b200nerf_place_samples_bwd(p, p, 4, 4, 0, 2.0, 6.0, p, p, None) != 0 and "depth_only needs S == 1" in err()
    assert lib.b200nerf_place_samples_bwd(p, None, 4, 4, 1, 2.0, 6.0, p, p, None) != 0 and "offsets is null" in err()
    assert lib.b200nerf_place_samples_bwd(p, p, 4, 4, 2, 2.0, 6.0, None, p, None) != 0 and "null argument" in err()
    assert lib.b200nerf_place_samples_bwd(p, p, 4, 0, 2, 2.0, 6.0, p, p, None) != 0 and "bad sizes" in err()
    assert lib.b200nerf_points_bwd(p, None, 4, 4, p, None) != 0 and "null argument" in err()
    assert lib.b200nerf_points_bwd(p, p, 4, 0, p, None) != 0 and "bad sizes" in err()

    assert lib.b200nerf_nerf_samples_jvp_packed(p, p, p, p, p, None, 4, 4, p, p, p, None) != 0 and "null argument" in err()
    assert lib.b200nerf_nerf_samples_jvp_packed(p, p, p, p, p, p, 4, 0, p, p, p, None) != 0 and "bad sizes" in err()
    assert lib.b200nerf_nerf_pts_jvp_packed(p, p, None, p, 4, 4, p, p, p, None) != 0 and "null argument" in err()
    arr = C.cast((C.c_void_p * 24)(*([p] * 24)), C.c_void_p)
    assert lib.b200nerf_nerf_samples_jvp_multires(arr, 10, 4, p, p, p, p, 4, 0, p, p, p, None) != 0 and "S >= 1" in err()
    assert lib.b200nerf_nerf_samples_jvp_multires(arr, 11, 4, p, p, p, p, 4, 2, p, p, p, None) != 0 and "out of range" in err()
    assert lib.b200nerf_nerf_samples_jvp_multires(arr, 10, 4, p, p, p, None, 4, 2, p, p, p, None) != 0 and "null argument" in err()
    with pytest.raises(_lib.B200NerfError, match="S >= 2"):
        _lib.check(lib.b200nerf_composite_bwd(p, p, p, None, 4, 1, 1, None, None, None, None, None, None, p, p, None))


@pytest.mark.parametrize("n", [1, 7, 4096])
@pytest.mark.parametrize("S", [1, 2, 32, 192])
def test_workspace_sizes(lib, n, S):
    assert lib.b200nerf_nerf_samples_jvp_packed_ws_bytes(n, S) == 12 * n * S * 4 * 8
    assert lib.b200nerf_nerf_samples_jvp_packed_ws_bytes(n, S) == lib.b200nerf_nerf_point_jvp_packed_ws_bytes(n * S)
    for m, mv in ((10, 4), (5, 2), (1, 1)):
        assert lib.b200nerf_nerf_samples_ws_floats_multires(n, S, m, mv) == lib.b200nerf_nerf_point_ws_floats_multires(n * S, m, mv)
    if S == 1:
        assert lib.b200nerf_nerf_samples_jvp_packed_ws_bytes(n, 1) == lib.b200nerf_nerf_point_jvp_packed_ws_bytes(n)
        assert lib.b200nerf_nerf_samples_ws_floats_multires(n, 1, 10, 4) == lib.b200nerf_nerf_point_ws_floats(n)
    assert lib.b200nerf_nerf_samples_ws_floats_multires(n, S, 11, 4) == 0
    assert lib.b200nerf_nerf_samples_ws_floats_multires(n, 0, 10, 4) == 0


def _boom(*a, **k):
    raise AssertionError("the differentiable route was taken")


def test_no_grad_takes_the_old_path(monkeypatch):
    """Under no_grad, or when nothing requires grad, the three entry points call the operators they called before (the ops are
    replaced by recorders here, the autograd functions by tripwires)."""
    from nerf_sampling_b200 import ops, training
    from nerf_sampling_b200.nerf_pytorch import utils
    from nerf_sampling_b200.nerf_pytorch.run_nerf_helpers import NeRF
    from nerf_sampling_b200.trainers.sampling_trainer import DepthNetTrainer

    for name in ("CompositeFn", "CompositeSingleFn", "PlaceFn", "PointsFn", "NerfPtsFn", "NerfPointFn"):
        monkeypatch.setattr(getattr(training, name), "apply", _boom)
    calls = []
    monkeypatch.setattr(ops, "composite", lambda *a, **k: calls.append("composite") or (None,) * 6)
    monkeypatch.setattr(ops, "place_samples", lambda *a, **k: calls.append("place") or torch.zeros(2, 3))
    monkeypatch.setattr(ops, "points", lambda *a, **k: calls.append("points") or torch.zeros(2, 3, 3))
    monkeypatch.setattr(ops, "nerf_mlp", lambda *a, **k: calls.append("nerf_mlp") or torch.zeros(2, 3, 4))
    monkeypatch.setattr(NeRF, "packed", lambda self: None)
    tr = DepthNetTrainer.__new__(DepthNetTrainer)
    net = NeRF(input_ch=63, input_ch_views=27, output_ch=5, use_viewdirs=True)
    for S in (1, 3):
        raw = torch.zeros(2, S, 4, requires_grad=True)
        z = torch.zeros(2, S, requires_grad=True)
        mean = torch.zeros(2, 1, requires_grad=True)
        pts = torch.zeros(2, S, 3, requires_grad=True)
        with torch.no_grad():
            tr.raw2outputs(raw, z, torch.zeros(2, 3))
            utils.sample_points_around_mean(torch.zeros(2, 3), torch.zeros(2, 3), mean, n_samples=S, mode="uniform")
            net.query(torch.zeros(2, 3), pts=pts)
            net.query(torch.zeros(2, 3), rays_o=torch.zeros(2, 3), rays_d=torch.zeros(2, 3), z=z)
        # grad enabled, nothing requires it
        tr.raw2outputs(raw.detach(), z.detach(), torch.zeros(2, 3))
        utils.sample_points_around_mean(torch.zeros(2, 3), torch.zeros(2, 3), mean.detach(), n_samples=S, mode="uniform")
        net.query(torch.zeros(2, 3), pts=pts.detach())
    assert calls == ["composite", "place", "points", "nerf_mlp", "nerf_mlp", "composite", "place", "points", "nerf_mlp"] * 2


def test_grad_takes_the_new_path(monkeypatch):
    """... and with grad enabled and an input that requires it, the autograd functions (here: tripwires)."""
    from nerf_sampling_b200 import training
    from nerf_sampling_b200.nerf_pytorch import utils
    from nerf_sampling_b200.nerf_pytorch.run_nerf_helpers import NeRF
    from nerf_sampling_b200.trainers.sampling_trainer import DepthNetTrainer

    tr = DepthNetTrainer.__new__(DepthNetTrainer)
    for name in ("CompositeFn", "CompositeSingleFn", "PlaceFn", "NerfPtsFn", "NerfPointFn"):
        monkeypatch.setattr(getattr(training, name), "apply", lambda *a, _n=name, **k: (_ for _ in ()).throw(KeyError(_n)))
    monkeypatch.setattr(NeRF, "packed", lambda self: None)
    net = NeRF(input_ch=63, input_ch_views=27, output_ch=5, use_viewdirs=True)
    with pytest.raises(KeyError, match="CompositeFn"):
        tr.raw2outputs(torch.zeros(2, 3, 4, requires_grad=True), torch.zeros(2, 3), torch.zeros(2, 3))
    with pytest.raises(KeyError, match="CompositeFn"):
        tr.raw2outputs(torch.zeros(2, 3, 4), torch.zeros(2, 3, requires_grad=True), torch.zeros(2, 3))
    with pytest.raises(KeyError, match="CompositeSingleFn"):
        tr.raw2outputs(torch.zeros(2, 1, 4, requires_grad=True), torch.zeros(2, 1), torch.zeros(2, 3))
    with pytest.raises(KeyError, match="PlaceFn"):
        utils.sample_points_around_mean(torch.zeros(2, 3), torch.zeros(2, 3), torch.zeros(2, 1, requires_grad=True), 4, "uniform")
    with pytest.raises(KeyError, match="NerfPtsFn"):
        net.query(torch.zeros(2, 3), pts=torch.zeros(2, 4, 3, requires_grad=True))
    with pytest.raises(KeyError, match="NerfPointFn"):
        net.query(torch.zeros(2, 3), rays_o=torch.zeros(2, 3), rays_d=torch.zeros(2, 3), z=torch.zeros(2, 4, requires_grad=True))


def test_pts_route_refuses_a_model_without_split_image():
    from nerf_sampling_b200 import _lib, training
    from nerf_sampling_b200.packing import PREC_FP16

    class NoSplit:
        wpack = None
        prec = PREC_FP16

    with pytest.raises(_lib.B200NerfError, match=f"precision {PREC_FP16}"):
        training.NerfPtsFn.apply(torch.zeros(2, 3, 3, requires_grad=True), torch.zeros(2, 3), NoSplit())


# --------------------------------------------------------------------------------------------- GPU: composite backward
def _composite_inputs(n, S, seed):
    """raw / z / rays_d / noise with three kinds of rays: ordinary (sigma ~ 3 N(0,1), half of the samples empty), saturating
    (sigma ~ 200: alpha rounds to 1 in fp32 and T underflows after a few samples), and sparse (a few dense samples)."""
    g = torch.Generator().manual_seed(seed)
    raw = torch.randn(n, S, 4, generator=g) * 2.0
    raw[..., 3] = torch.randn(n, S, generator=g) * 3.0
    sat = torch.arange(n) % 3 == 1
    raw[sat, :, 3] = 200.0 + torch.randn(int(sat.sum()), S, generator=g)
    sparse = torch.arange(n) % 3 == 2
    raw[sparse, :, 3] = torch.where(torch.rand(int(sparse.sum()), S, generator=g) < 0.1, 30.0, -1.0)
    z = torch.sort(2.0 + 4.0 * torch.rand(n, S, generator=g), -1).values
    rd = torch.randn(n, 3, generator=g)
    rd = rd / rd.norm(dim=-1, keepdim=True) * (0.5 + 1.5 * torch.rand(n, 1, generator=g))   # |d| in [0.5, 2]: not unit rays
    noise = torch.randn(n, S, generator=g) * 0.5
    return raw.to(DEV), z.to(DEV), rd.to(DEV), noise.to(DEV)


UPSTREAM = ["rgb", "disp", "acc", "depth", "weights", "alphas"]


@pytest.mark.gpu
@pytest.mark.parametrize("use_noise", [False, True])
@pytest.mark.parametrize("white", [True, False])
@pytest.mark.parametrize("S", [2, 3, 32, 64, 128, 192])
def test_composite_backward_vs_fp64(lib, S, white, use_noise):
    from nerf_sampling_b200 import ops
    from nerf_sampling_b200.trainers.sampling_trainer import DepthNetTrainer

    n = 301
    raw, z, rd, noise = _composite_inputs(n, S, 7 * S + 2 * white + use_noise)
    nz = noise if use_noise else None
    tr = DepthNetTrainer.__new__(DepthNetTrainer)
    g = torch.Generator().manual_seed(S)
    up = {"rgb": torch.randn(n, 3, generator=g), "disp": torch.randn(n, generator=g) * 1e-2, "acc": torch.randn(n, generator=g),
          "depth": torch.randn(n, generator=g), "weights": torch.randn(n, S, generator=g), "alphas": torch.randn(n, S, generator=g)}
    up = {k: v.to(DEV) for k, v in up.items()}
    sg_last = raw[:, -1, 3] + (noise[:, -1] if use_noise else 0.0)
    keep = sg_last.abs() >= KNIFE
    n_knife = int((~keep).sum())

    with torch.no_grad():
        ref = ops.composite(raw, z, rd, white, nz)
    r32 = raw.clone().requires_grad_(True)
    z32 = z.clone().requires_grad_(True)
    if use_noise:
        # DepthNetTrainer.raw2outputs draws the noise itself: feed the same draw through the autograd function
        from nerf_sampling_b200 import training

        outs = training.CompositeFn.apply(r32, z32, rd, nz, white)
    else:
        rgb, disp, acc, depth, _, alphas, weights = tr.raw2outputs(r32, z32, rd, 0, white)
        outs = (rgb, disp, acc, depth, weights, alphas)
    for a, b in zip(outs, ref):   # forward values with grad enabled: bitwise the no_grad values
        assert torch.equal(a.detach(), b)
    o = dict(zip(["rgb", "disp", "acc", "depth", "weights", "alphas"], outs))

    r64 = raw.double().requires_grad_(True)
    z64 = z.double().requires_grad_(True)
    rgb, disp, acc, depth, _, alphas, weights = O.raw2outputs(r64, z64, rd.double(), 1.0 if use_noise else 0.0, white,
                                                              noise=noise.double() if use_noise else None)
    w = dict(rgb=rgb, disp=disp, acc=acc, depth=depth, weights=weights, alphas=alphas)
    worst = {}
    for combo in [[k] for k in UPSTREAM] + [UPSTREAM]:
        gr, gz = torch.autograd.grad([o[k] for k in combo], [r32, z32], [up[k] for k in combo], retain_graph=True, allow_unused=True)
        wr, wz = torch.autograd.grad([w[k] for k in combo], [r64, z64], [up[k].double() for k in combo], retain_graph=True,
                                     allow_unused=True)
        for name, got, want in (("raw", gr, wr), ("z", gz, wz)):
            want = torch.zeros_like(r64 if name == "raw" else z64) if want is None else want
            got = torch.zeros_like(want) if got is None else got.double()
            assert bool(torch.isfinite(got[keep]).all()), (combo, name)
            top = float(want[keep].abs().max())
            err = float((got[keep] - want[keep]).abs().max())
            rel = err / top if top > 0 else err
            worst["+".join(combo) + ":" + name] = rel
            assert rel <= TAU_COMP, (combo, name, err, top)
    k = max(worst, key=worst.get)
    print(f"composite backward S={S} white={white} noise={use_noise}: worst {k} {worst[k]:.2e} of its largest entry; "
          f"{n_knife} of {n} rays on the |sigma_last| < {KNIFE} knife edge excluded")


@pytest.mark.gpu
def test_composite_backward_keeps_the_gradient_where_t_underflows(lib):
    """A ray whose second sample is opaque (alpha = 1 in fp32, t = 1e-10) and whose samples behind it are too: T underflows in
    fp32 past the third sample, while d loss / d alpha_0 = T_0 (g_w0 - R_0) stays O(1) -- a division by t would give 0 / 0."""
    from nerf_sampling_b200 import training

    S = 8
    raw = torch.zeros(1, S, 4, device=DEV)
    raw[0, :, 3] = torch.tensor([0.5] + [500.0] * (S - 1))
    z = torch.linspace(2.0, 5.0, S, device=DEV).reshape(1, S)
    rd = torch.tensor([[0.0, 0.0, -1.0]], device=DEV)
    r32 = raw.clone().requires_grad_(True)
    rgb, disp, acc, depth, weights, alphas = training.CompositeFn.apply(r32, z, rd, None, True)
    (gr,) = torch.autograd.grad(depth.sum(), r32)
    r64 = raw.double().requires_grad_(True)
    out = O.raw2outputs(r64, z.double(), rd.double(), 0.0, True)
    (wr,) = torch.autograd.grad(out[3].sum(), r64)
    assert float(weights.detach()[0, 6:].abs().max()) == 0.0   # T underflowed in fp32 (1e-10 per opaque sample)
    assert float(wr[0, 0, 3]) != 0.0 and abs(float(gr[0, 0, 3]) - float(wr[0, 0, 3])) <= 1e-4 * abs(float(wr[0, 0, 3]))


# --------------------------------------------------------------------------------------------- GPU: d raw / d z, d raw / d pts
def _view_rays(side, seed=0):
    packed, *_ = O.prepare_rays(side, side, O.intrinsics(side, side), c2w=O.pose_spherical(30.0 + seed, -30.0, 4.0)[:3, :4])
    return tuple(packed[:, a:b].contiguous().to(DEV) for a, b in ((0, 3), (3, 6), (8, 11)))


def _run_network64(pts, viewdirs, p):
    """O.run_network with the octave counts of the weight shapes, in fp64."""
    m, mv = (p["pts_linears.0.weight"].shape[1] - 3) // 6, (p["views_linears.0.weight"].shape[1] - 259) // 6
    flat = pts.reshape(-1, 3)
    dirs = viewdirs[:, None].expand(pts.shape).reshape(-1, 3)
    emb = torch.cat([O.embed(flat, m), O.embed(dirs, mv)], -1)
    return O.nerf_forward(p, emb, input_ch=d_of(m), input_ch_views=d_of(mv)).reshape(list(pts.shape[:-1]) + [4])


def _nerf(p, prec=None):
    from nerf_sampling_b200.nerf_pytorch.run_nerf_helpers import NeRF

    m, mv = (p["pts_linears.0.weight"].shape[1] - 3) // 6, (p["views_linears.0.weight"].shape[1] - 259) // 6
    net = NeRF(D=8, W=256, input_ch=d_of(m), input_ch_views=d_of(mv), output_ch=5, skips=[4], use_viewdirs=True)
    net.load_state_dict(p)
    if prec is not None:
        net.precision = prec
    return net.to(DEV)


def _jvp_errors(got_cols, want_cols):
    """Per-channel error / the channel's largest fp64 derivative, per sample point (max over its columns); returns (worst on the
    kink-free points, kink mask [n, S]): a point is counted as crossing a ReLU kink when any of its errors exceeds TAU_JVP."""
    errs = [(gg.double() - gw).abs() / float(gw.abs().max()) for gg, gw in zip(got_cols, want_cols)]
    kink = torch.zeros_like(errs[0], dtype=torch.bool)
    for e in errs:
        kink |= e > TAU_JVP
    worst = max(float(e[~kink].max()) for e in errs) if not bool(kink.all()) else 0.0
    return worst, kink


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["split", "fp32"])
@pytest.mark.parametrize("S", [1, 2, 32, 64])
def test_samples_jvp_vs_fp64(lib, oracle_models, route, S):
    """raw and d raw / d z at S samples per ray (NerfPointFn / NeRF.query(z=...)) against fp64 autograd."""
    from nerf_sampling_b200 import training
    from nerf_sampling_b200.packing import PREC_SPLIT

    _, fine, _ = oracle_models
    net = _nerf(fine, PREC_SPLIT)
    ro, rd, vd = _view_rays(23 if S > 2 else 37)
    n = ro.shape[0]
    z = torch.sort(2.5 + 3.0 * torch.rand(n, S, generator=torch.Generator().manual_seed(S)), -1).values.to(DEV).requires_grad_(True)
    raw = training.NerfPointFn.apply(z, ro, rd, vd, net.packed() if route == "split" else None, *training.nerf_params(net))
    assert raw.shape == (n, S, 4)
    p64 = O.params_to({k: v.double() for k, v in fine.items()}, DEV)
    z2 = z.detach().double().clone().requires_grad_(True)
    want = _run_network64(ro.double()[:, None, :] + rd.double()[:, None, :] * z2[:, :, None], vd.double(), p64)
    rerr = float((raw.double() - want).abs().max())
    assert rerr <= (1e-5 if route == "fp32" else 1e-4)
    got_cols, want_cols = [], []
    for c in range(4):   # d raw_c / d z_s: each sample's raw depends on its own depth only, so the column sum separates them
        want_cols.append(torch.autograd.grad(want[..., c].sum(), z2, retain_graph=True)[0])
        got_cols.append(torch.autograd.grad(raw[..., c].sum(), z, retain_graph=True)[0])
    worst, kink = _jvp_errors(got_cols, want_cols)
    n_kink = int(kink.sum())
    print(f"d raw / d z, route {route}, S={S}, {n} rays: max-abs raw error {rerr:.2e}, worst derivative error {worst:.2e} of the "
          f"channel's largest, sample points across a ReLU kink: {n_kink} of {n * S}")
    assert n_kink <= max(1, n * S // 200)

    L = lib
    st = torch.cuda.current_stream().cuda_stream
    zf = z.detach().reshape(-1).contiguous()
    if S == 1:
        # bitwise the one-sample entry points
        raw1, d1 = torch.empty(n, 4, device=DEV), torch.empty(n, 4, device=DEV)
        if route == "split":
            pk = net.packed()
            ws = torch.empty(L.b200nerf_nerf_point_jvp_packed_ws_bytes(n), dtype=torch.uint8, device=DEV)
            assert L.b200nerf_nerf_point_jvp_packed(pk.wpack.data_ptr(), pk.aux.data_ptr(), ro.data_ptr(), rd.data_ptr(), vd.data_ptr(),
                                                    zf.data_ptr(), n, ws.data_ptr(), raw1.data_ptr(), d1.data_ptr(), st) == 0
        else:
            params = training.nerf_params(net)
            ws = torch.empty(L.b200nerf_nerf_point_ws_floats(n), device=DEV)
            assert L.b200nerf_nerf_point_jvp(training._ptrs(params), ro.data_ptr(), rd.data_ptr(), vd.data_ptr(), zf.data_ptr(), n,
                                             ws.data_ptr(), raw1.data_ptr(), d1.data_ptr(), st) == 0
        assert torch.equal(raw1, raw.detach().reshape(n, 4))
        assert torch.equal(d1, torch.stack(got_cols, -1).reshape(n, 4))
    elif route == "split":
        # the packed route at S is itself run as n * S rays of one sample each, bitwise
        rep = lambda t: t.repeat_interleave(S, 0).contiguous()  # noqa: E731
        raw1 = torch.empty(n * S, 1, 4, device=DEV)
        d1 = torch.empty(n * S, 4, device=DEV)
        ws = training.nerf_point_jvp(net.packed(), None, rep(ro), rep(rd), rep(vd), zf, raw1, d1, st)   # noqa: F841
        assert torch.equal(raw1.reshape(n, S, 4), raw.detach())
        assert torch.equal(d1.reshape(n, S, 4), torch.stack(got_cols, -1))


@pytest.mark.gpu
@pytest.mark.parametrize("S", [1, 2, 32, 64])
def test_pts_jvp_vs_fp64_and_z_route(lib, oracle_models, S):
    """raw and d raw / d pts at explicit points (NeRF.query(pts=...) / Trainer.run_network) against fp64 autograd, and J d equal to
    the z route's d raw / d z within rounding."""
    from nerf_sampling_b200 import training
    from nerf_sampling_b200.packing import PREC_SPLIT

    _, fine, _ = oracle_models
    net = _nerf(fine, PREC_SPLIT)
    ro, rd, vd = _view_rays(23 if S > 2 else 37, seed=1)
    n = ro.shape[0]
    z = torch.sort(2.5 + 3.0 * torch.rand(n, S, generator=torch.Generator().manual_seed(S + 1)), -1).values.to(DEV)
    pts = (ro[:, None, :] + rd[:, None, :] * z[:, :, None]).contiguous().requires_grad_(True)
    raw = net.query(vd, pts=pts)
    with torch.no_grad():
        assert torch.equal(raw.detach(), net.query(vd, pts=pts))   # PREC_SPLIT: the primal pass is split-precision inference
    p64 = O.params_to({k: v.double() for k, v in fine.items()}, DEV)
    p2 = pts.detach().double().clone().requires_grad_(True)
    want = _run_network64(p2, vd.double(), p64)
    rerr = float((raw.double() - want).abs().max())
    assert rerr <= 1e-4
    # J[:, :, k, c] = d raw_c / d pts_k
    got_cols, want_cols, jac = [], [], torch.zeros(n, S, 3, 4, device=DEV)
    for c in range(4):
        gg = torch.autograd.grad(raw[..., c].sum(), pts, retain_graph=True)[0]
        gw = torch.autograd.grad(want[..., c].sum(), p2, retain_graph=True)[0]
        jac[..., c] = gg
        for k in range(3):
            got_cols.append(gg[..., k])
            want_cols.append(gw[..., k])
    worst, kink = _jvp_errors(got_cols, want_cols)
    n_kink = int(kink.sum())
    # the chain rule through the pts route: d raw / d z = J d, against the z route's tangent pass along d
    zz = z.clone().requires_grad_(True)
    raw_z = net.query(vd, rays_o=ro, rays_d=rd, z=zz)
    assert torch.equal(raw_z.detach(), raw.detach()) or float((raw_z.detach() - raw.detach()).abs().max()) <= 1e-5
    jd = (jac * rd[:, None, :, None]).sum(2)
    chain = []
    for c in range(4):
        dz = torch.autograd.grad(raw_z[..., c].sum(), zz, retain_graph=True)[0]
        chain.append((jd[..., c] - dz).abs() / float(dz.abs().max()))
    chain_err = max(float(e[~kink].max()) for e in chain)
    print(f"d raw / d pts, S={S}, {n} rays: max-abs raw error {rerr:.2e}, worst derivative error {worst:.2e} of the channel's "
          f"largest, sample points across a ReLU kink: {n_kink} of {n * S}; |J d - d raw / d z| {chain_err:.2e} of the channel's "
          f"largest")
    assert n_kink <= max(1, n * S // 200)
    assert chain_err <= TAU_JVP / 10   # two split-precision evaluations of one derivative: the tangent along d, and J d


# --------------------------------------------------------------------------------------------- GPU: placement
@pytest.mark.gpu
@pytest.mark.parametrize("mode,S", [("uniform", 32), ("uniform", 7), ("uniform", 2), ("gaussian", 32), ("gaussian", 5),
                                    ("depth_only", 1)])
def test_placement_backward_vs_torch(lib, mode, S):
    """sample_points_around_mean under autograd (PlaceFn + PointsFn) against torch autograd on oracle.place_samples; uniform means
    within `distance` of 2 and of 6, so that samples clip (a sample clipped onto a bound gets no gradient)."""
    from nerf_sampling_b200.nerf_pytorch import utils

    n, std = 4099, 0.1
    g = torch.Generator().manual_seed(S)
    mean = 2.0 + 4.0 * torch.rand(n, 1, generator=g)
    mean[: n // 3] = 2.0 + (torch.rand(n // 3, 1, generator=g) - 0.5) * 2.4 * std     # near 2 (some below it)
    mean[n // 3: 2 * n // 3] = 6.0 + (torch.rand(n // 3, 1, generator=g) - 0.5) * 2.4 * std
    mean[:4] = torch.tensor([[2.0], [6.0], [2.0 - std], [6.0 + std]])                  # samples exactly on the bounds
    ro, rd = torch.randn(n, 3, generator=g), torch.randn(n, 3, generator=g) * 1.7
    noise = torch.randn(n, max(S - 1, 1), generator=g)
    gz_up, gp_up = torch.randn(n, S, generator=g), torch.randn(n, S, 3, generator=g)
    ro, rd, mean, noise, gz_up, gp_up = (t.to(DEV) for t in (ro, rd, mean, noise, gz_up, gp_up))

    with torch.no_grad():
        pts0, z0 = utils.sample_points_around_mean(ro, rd, mean, n_samples=S, mode=mode, std=std, noise=noise)
    m32 = mean.clone().requires_grad_(True)
    pts, z = utils.sample_points_around_mean(ro, rd, m32, n_samples=S, mode=mode, std=std, noise=noise)
    assert torch.equal(pts.detach(), pts0) and torch.equal(z.detach(), z0)   # forward with grad: bitwise the no_grad values
    (gz,) = torch.autograd.grad(z, m32, gz_up, retain_graph=True)
    (gp,) = torch.autograd.grad(pts, m32, gp_up, retain_graph=True)

    # the oracle in fp32 on the CPU: the same linspace and the same unclipped fp32 values, so the clip masks must agree exactly
    mc = mean.cpu().requires_grad_(True)
    pc, zc = O.place_samples(ro.cpu(), rd.cpu(), mc, n_samples=S, mode=mode, std=std, noise=noise.cpu() if mode == "gaussian" else None)
    assert torch.equal(zc, z0.cpu())
    (wz,) = torch.autograd.grad(zc, mc, gz_up.cpu(), retain_graph=True)
    (wp,) = torch.autograd.grad(pc, mc, gp_up.cpu(), retain_graph=True)
    wz, wp = wz.double().to(DEV), wp.double().to(DEV)
    if mode == "uniform":
        n_clip = 0
        for s in range(S):
            onehot = torch.zeros(n, S, device=DEV)
            onehot[:, s] = 1.0
            (gs,) = torch.autograd.grad(z, m32, onehot, retain_graph=True)
            (ws,) = torch.autograd.grad(zc, mc, onehot.cpu(), retain_graph=True)
            assert torch.equal(gs.reshape(-1).cpu() != 0, ws.reshape(-1) != 0), f"clip mask of sample {s}"
            n_clip += int((ws == 0).sum())
        assert 0 < n_clip < n * S, "the batch must clip some samples and not all"
    bound = lambda w, t: 4 * S * 6e-8 * float(t.abs().max()) * max(1.0, float(w.abs().max()))  # noqa: E731  (an S-term fp32 sum)
    ez = float((gz.double() - wz).abs().max())
    ep = float((gp.double() - wp).abs().max())
    print(f"placement backward {mode} S={S}: |g_mean - torch| {ez:.2e} (from z), {ep:.2e} (from pts)")
    assert ez <= bound(wz, gz_up) and ep <= bound(wp, gp_up * rd.abs().max())


# --------------------------------------------------------------------------------------------- GPU: the whole composition
def _dn_encoding(m, ro, rd, multires):
    """The ray encoding DepthNet's training kernels compute ([n, 4 d3] at the start of the workspace; see
    test_depthnet_architectures._rays for why the fp64 reference runs on it)."""
    from nerf_sampling_b200 import _lib, training

    params = training.depthnet_params(m)
    hidden, cat = training.depthnet_arch(m)
    L = _lib.lib()
    n = ro.shape[0]
    ints = lambda v: (C.c_int * len(v))(*v)  # noqa: E731
    ws = torch.empty(L.b200nerf_depthnet_train_ws_floats_multires(n, len(hidden), ints(hidden), len(cat), ints(cat), multires), device=DEV)
    z = torch.empty(n, 1, device=DEV)
    _lib.check(L.b200nerf_depthnet_train_fwd_multires(training._ptrs(params), len(hidden), ints(hidden), len(cat), ints(cat), multires,
                                                      ro.data_ptr(), rd.data_ptr(), n, 2.0, 2.0, 6.0, ws.data_ptr(), z.data_ptr(),
                                                      torch.cuda.current_stream().cuda_stream))
    w = 4 * d_of(multires)
    return ws[: n * w].reshape(n, w).clone()


def _dn64(p, enc, multires, near=2.0, far=6.0):
    """DepthNet (oracle.depthnet_forward's layers) on the encoding enc, and every cat layer's pre-activation."""
    d3 = d_of(multires)
    enc = enc.double()
    e_o, e_d, e_i = enc[:, :d3], enc[:, d3:2 * d3], enc[:, 2 * d3:]

    def branch(name, e):
        x, i = e, 0
        while f"{name}.{i}.weight" in p:
            x = F.linear(torch.cat([x, e], -1), p[f"{name}.{i}.weight"], p[f"{name}.{i}.bias"])
            i += 1
        return x

    x = torch.cat([branch("origin_layers", e_o), branch("direction_layers", e_d), branch("intersection_layers", e_i), e_o, e_d, e_i], -1)
    pre, j = [], 0
    while f"cat_layers.{j}.weight" in p:
        y = F.linear(x, p[f"cat_layers.{j}.weight"], p[f"cat_layers.{j}.bias"])
        pre.append(y)
        x = F.leaky_relu(y, 0.01)
        j += 2
    s = torch.sigmoid(F.linear(x, p["to_depth.0.weight"], p["to_depth.0.bias"]))
    return near * (1 - s) + far * s, pre


def _whole_models(which, oracle_models):
    from nerf_sampling_b200.depth_nets import DepthNet

    if which == "reference":
        _, fine, dn = oracle_models
        multires = 10
    else:
        torch.manual_seed(55)
        fine = O.init_nerf(input_ch=d_of(5), input_ch_views=d_of(2))
        # this seed's density head is negative everywhere around the depths (an empty scene: every gradient would be 0); shifted,
        # about half of the samples carry density, like the reference seed's
        fine["alpha_linear.bias"] = fine["alpha_linear.bias"] + 0.07
        torch.manual_seed(56)
        dn = O.init_depthnet([256] * 10, [256] * 10, multires=5)
        multires = 5
    d = DepthNet(hidden_sizes=[256] * 10, cat_hidden_sizes=[256] * 10, sphere_radius=2.0, multires=multires)
    d.load_state_dict(dn)
    return _nerf(fine), d.to(DEV), fine, dn, multires


def _chain64(mean, fine, ro, rd, vd, S, mode, std, noise, target, z_target):
    """fp64 loss of the reference composition from the depths `mean` on: place_samples -> run_network -> raw2outputs -> losses."""
    pts, z = O.place_samples(ro.double(), rd.double(), mean, n_samples=S, mode=mode, std=std,
                             noise=None if noise is None else noise.double())
    raw = _run_network64(pts, vd.double(), {k: v.to(DEV, torch.float64) for k, v in fine.items()})
    rgb, _, _, depth, _, _, _ = O.raw2outputs(raw, z, rd.double(), 0.0, True)
    return F.mse_loss(rgb, target.double()) + F.mse_loss(depth, z_target.double()), raw.detach()


def _chain(route, mean, net, tr, ro, rd, vd, S, mode, std, noise, target, z_target):
    """The same composition through the product: sample_points_around_mean -> Trainer.run_network (route "pts") or
    NeRF.query(z=...) (route "z") -> DepthNetTrainer.raw2outputs -> losses."""
    from nerf_sampling_b200.nerf_pytorch import utils
    from nerf_sampling_b200.nerf_pytorch.run_nerf_helpers import get_embedder
    from nerf_sampling_b200.nerf_pytorch.trainers.Trainer import Trainer

    pts, z = utils.sample_points_around_mean(ro, rd, mean, n_samples=S, mode=mode, std=std, noise=noise)
    if route == "pts":
        m, mv = net.multires()
        raw = Trainer.run_network(tr, pts, vd, net, get_embedder(m, 0, 3)[0], get_embedder(mv, 0, 3)[0])
    else:
        raw = net.query(vd, rays_o=ro, rays_d=rd, z=z)
    rgb, _, _, depth, _, _, _ = tr.raw2outputs(raw, z, rd, 0, True)
    return F.mse_loss(rgb, target) + F.mse_loss(depth, z_target), raw.detach()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["uniform", "gaussian"])
@pytest.mark.parametrize("which", ["reference", "multires5"])
def test_whole_composition_gradients_vs_fp64(lib, oracle_models, which, mode):
    """DepthNet(rays) -> sample_points_around_mean(S=32) -> Trainer.run_network -> DepthNetTrainer.raw2outputs ->
    mse(rgb, target) + mse(depth, z_target) -> backward, and the same with NeRF.query(z=...) in place of run_network: every
    DepthNet gradient against fp64 autograd, and the two routes against each other.  The fp64 reference differentiates DepthNet on
    the kernels' ray encoding and the rest of the composition at the depths the product's DepthNet computed.

    Two kinds of rays are screened out first.  LeakyReLU kinks of DepthNet: the screen of test_depthnet_architectures (fp64
    pre-activations on the kernels' encoding).  ReLU kinks of the NeRF: a sample point whose hidden value lies within rounding
    distance of zero may take the other derivative than fp64 (as in the d raw / d z tests), which moves that ray's d loss / d mean
    by O(1) of the sample's share; such rays are found by comparing d loss / d mean per ray with fp64 (1e-3 of its largest entry,
    both routes), counted and bounded like the kink points of the d raw / d z tests."""
    from nerf_sampling_b200.trainers.sampling_trainer import DepthNetTrainer

    S, std, n = 32, 0.1, 512
    net, dnet, fine, dn, multires = _whole_models(which, oracle_models)
    tr = DepthNetTrainer.__new__(DepthNetTrainer)
    ro, rd, vd = _view_rays(64)
    enc = _dn_encoding(dnet, ro, rd, multires)
    p64 = {k: v.to(DEV, torch.float64) for k, v in dn.items()}
    with torch.no_grad():
        _, pre = _dn64(p64, enc, multires)
    ok = torch.ones(ro.shape[0], dtype=torch.bool, device=DEV)
    for y in pre:
        ok &= y.abs().min(-1).values > TAU * float(y.pow(2).mean().sqrt())
    pool = ok.nonzero().reshape(-1)
    n_dn_kink = ro.shape[0] - pool.numel()
    sel = pool[torch.randperm(pool.numel(), generator=torch.Generator().manual_seed(3)).to(DEV)[: 2 * n]]
    ro, rd, vd, enc = ro[sel].contiguous(), rd[sel].contiguous(), vd[sel].contiguous(), enc[sel]
    g = torch.Generator().manual_seed(4)
    noise = torch.randn(ro.shape[0], S - 1, generator=g).to(DEV) if mode == "gaussian" else None
    target = torch.rand(ro.shape[0], 3, generator=g).to(DEV)
    z_target = (2.0 + 4.0 * torch.rand(ro.shape[0], generator=g)).to(DEV)

    # screen: d loss / d mean per ray, product (both routes) against fp64 at the same depths
    m32 = dnet(ro, rd).detach().requires_grad_(True)
    m64 = m32.detach().double().requires_grad_(True)
    loss64, raw64 = _chain64(m64, fine, ro, rd, vd, S, mode, std, noise, target, z_target)
    (gm64,) = torch.autograd.grad(loss64, m64)
    bad = (raw64[:, -1, 3].abs() < KNIFE).reshape(-1)
    n_knife = int(bad.sum())
    for route in ("pts", "z"):
        (gm,) = torch.autograd.grad(_chain(route, m32, net, tr, ro, rd, vd, S, mode, std, noise, target, z_target)[0], m32)
        bad |= ((gm.double() - gm64).abs() / float(gm64.abs().max())).reshape(-1) > TAU_JVP
    n_nerf_kink = int(bad.sum()) - n_knife
    assert n_nerf_kink <= max(1, 2 * n * S // 200)
    clean = (~bad).nonzero().reshape(-1)[:n]
    assert clean.numel() == n
    ro, rd, vd, enc, target, z_target = (t[clean].contiguous() for t in (ro, rd, vd, enc, target, z_target))
    noise = None if noise is None else noise[clean].contiguous()

    # the fp64 reference: DepthNet on the kernels' encoding (test_depthnet_architectures), the rest of the composition at the depths
    # the product's DepthNet gives -- 1e-6 between fp32 and fp64 depths would move d loss / d mean by ~5e-4 through the NeRF's 2^9
    # octave, which is the DepthNet forward's rounding, not a derivative
    with torch.no_grad():
        m_at = dnet(ro, rd).double()
        assert float((m_at - _dn64(p64, enc, multires)[0]).abs().max()) <= 1e-5
    m_at.requires_grad_(True)
    loss_ref, raw_ref = _chain64(m_at, fine, ro, rd, vd, S, mode, std, noise, target, z_target)
    (gm_ref,) = torch.autograd.grad(loss_ref, m_at)
    p_dn = {k: v.to(DEV, torch.float64).requires_grad_(True) for k, v in dn.items()}
    (_dn64(p_dn, enc, multires)[0] * gm_ref).sum().backward()
    want = {k: v.grad for k, v in p_dn.items()}
    out, worst = {}, {}
    for route in ("pts", "z"):
        dnet.zero_grad(set_to_none=True)
        loss, raw = _chain(route, dnet(ro, rd), net, tr, ro, rd, vd, S, mode, std, noise, target, z_target)
        loss.backward()
        out[route] = {k: p.grad.detach().clone() for k, p in dnet.named_parameters()}
        worst[route] = ("", 0.0)
        for k, gk in out[route].items():
            assert bool(torch.isfinite(gk).all()), (route, k)
            top = float(want[k].abs().max())
            rel = float((gk.double() - want[k]).abs().max()) / max(top, 1e-30)
            worst[route] = max(worst[route], (k, rel), key=lambda t: t[1])
        print(f"whole path {which} {mode} S={S}, route {route}, {n} rays ({n_dn_kink} of {64 * 64} view rays screened for DepthNet "
              f"kinks, {n_nerf_kink} of {2 * n} for NeRF kinks, {n_knife} knife-edge): loss {float(loss):.7f} (fp64 "
              f"{float(loss_ref):.7f}), max-abs raw error {float((raw.double() - raw_ref).abs().max()):.2e}, worst DepthNet gradient "
              f"{worst[route][0]} {worst[route][1]:.2e} of its largest (smallest largest entry "
              f"{min(float(v.abs().max()) for v in want.values()):.2e})")
    agree = max(float((out["pts"][k] - out["z"][k]).abs().max()) / max(float(out["z"][k].abs().max()), 1e-30) for k in out["z"])
    print(f"whole path {which} {mode}: pts route vs z route, worst {agree:.2e} of the largest entry")
    assert worst["pts"][1] <= TAU_G and worst["z"][1] <= TAU_G, worst
    assert agree <= TAU_G


@pytest.mark.gpu
def test_forward_values_with_grad_equal_no_grad(lib, oracle_models):
    """raw2outputs, sample_points_around_mean, Trainer.run_network and NeRF.query(z=...) at S = 32 return, with grad enabled, the
    values they return under no_grad (NeRF at PREC_SPLIT: the precision whose Jacobian the training kernels take)."""
    from nerf_sampling_b200.nerf_pytorch import utils
    from nerf_sampling_b200.nerf_pytorch.run_nerf_helpers import get_embedder
    from nerf_sampling_b200.nerf_pytorch.trainers.Trainer import Trainer
    from nerf_sampling_b200.packing import PREC_SPLIT
    from nerf_sampling_b200.trainers.sampling_trainer import DepthNetTrainer

    _, fine, _ = oracle_models
    net = _nerf(fine, PREC_SPLIT)
    tr = DepthNetTrainer.__new__(DepthNetTrainer)
    embed_fn, _ = get_embedder(10, 0, 3)
    embeddirs_fn, _ = get_embedder(4, 0, 3)
    ro, rd, vd = _view_rays(32)
    n, S = ro.shape[0], 32
    mean = (3.0 + torch.rand(n, 1, generator=torch.Generator().manual_seed(9))).to(DEV)
    for mode in ("uniform", "gaussian"):
        noise = torch.randn(n, S - 1, generator=torch.Generator().manual_seed(10)).to(DEV)
        with torch.no_grad():
            pts0, z0 = utils.sample_points_around_mean(ro, rd, mean, S, mode, 0.1, noise)
            raw_p0 = Trainer.run_network(tr, pts0, vd, net, embed_fn, embeddirs_fn)
            raw_z0 = net.query(vd, rays_o=ro, rays_d=rd, z=z0)
            maps0 = tr.raw2outputs(raw_p0, z0, rd, 0, True)
        m = mean.clone().requires_grad_(True)
        pts, z = utils.sample_points_around_mean(ro, rd, m, S, mode, 0.1, noise)
        raw_p = Trainer.run_network(tr, pts, vd, net, embed_fn, embeddirs_fn)
        raw_z = net.query(vd, rays_o=ro, rays_d=rd, z=z)
        maps = tr.raw2outputs(raw_p, z, rd, 0, True)
        assert raw_p.grad_fn is not None and raw_z.grad_fn is not None and maps[0].grad_fn is not None
        for a, b in [(pts, pts0), (z, z0), (raw_p, raw_p0), (raw_z, raw_z0)] + list(zip(maps, maps0)):
            assert torch.equal(a.detach(), b)
