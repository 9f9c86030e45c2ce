"""The NeRF MLP at every positional-encoding size: multires 1..10 and multires_views 1..4, in inference and training.

``NeRF(input_ch=d, input_ch_views=dv)`` with d = 3 (1 + 2 multires), dv = 3 (1 + 2 multires_views) is what the reference's
``create_nerf`` builds for ``--multires`` / ``--multires_views``.  The kernels place gamma(pts) in the first d of the 64 columns of its
operand block and gamma(viewdir) in the first dv of its 32, with zero weights in the rest, and read both sizes from the aux block of
the packed image.  So a net at (m, mv) packs byte for byte like the 10 / 4 net whose weights are zero-embedded at the kernel's
column positions (``pad``), and computes bit for bit what that net computes.  The fp64 references here derive the octave counts
from the weight shapes (``run_network``), like ``O.run_network`` does at 10 / 4.
"""

import ctypes as C

import pytest
import torch

from oracle import nerf_oracle as O

DEV = "cuda"
RAW_TOL = {1: 1e-4, 2: 5e-4, 3: 5e-4}   # test_gpu_parity.RAW_TOL: split precision / fp16 single pass (FP16 and FAST)
RGB_TOL = 1e-3
SIGMA_GUARD = 1e-5
NERF_BA = 2688                          # aux offset of the alpha-head bias; the octave counts follow it
# 5 and 6 straddle the fast encoder's second accurate octave; (2, 4) has more view octaves than position octaves
GPU_CASES = [(1, 1), (4, 2), (5, 4), (6, 3), (7, 1), (10, 1), (10, 4), (2, 4)]


def d_of(m):
    return 3 * (1 + 2 * m)


def init_nerf(m, mv, seed):
    torch.manual_seed(seed)
    return O.init_nerf(input_ch=d_of(m), input_ch_views=d_of(mv))


def multires_of(p):
    return (p["pts_linears.0.weight"].shape[1] - 3) // 6, (p["views_linears.0.weight"].shape[1] - 259) // 6


def pad(p):
    """The 10 / 4 net whose encoding columns hold the (m, mv) net's weights at the kernel's positions and zeros elsewhere."""
    m, mv = multires_of(p)
    d, dv = d_of(m), d_of(mv)
    q = dict(p)
    w0 = torch.zeros(256, 63, dtype=p["pts_linears.0.weight"].dtype)
    w0[:, :d] = p["pts_linears.0.weight"]
    w5 = torch.zeros(256, 319, dtype=w0.dtype)
    w5[:, :d], w5[:, 63:] = p["pts_linears.5.weight"][:, :d], p["pts_linears.5.weight"][:, d:]
    wv = torch.zeros(128, 283, dtype=w0.dtype)
    wv[:, : 256 + dv] = p["views_linears.0.weight"]
    q.update({"pts_linears.0.weight": w0, "pts_linears.5.weight": w5, "views_linears.0.weight": wv})
    return q


def run_network(pts, viewdirs, p):
    """O.run_network with the octave counts of the weight shapes (trainers/Trainer.py:789-806), in the precision of p."""
    m, mv = multires_of(p)
    dt = p["pts_linears.0.weight"].dtype
    flat = pts.reshape(-1, 3).to(dt)
    dirs = viewdirs[:, None].expand(pts.shape).reshape(-1, 3).to(dt)
    emb = torch.cat([O.embed(flat, m), O.embed(dirs, mv)], -1)
    out = O.nerf_forward(p, emb, input_ch=d_of(m), input_ch_views=d_of(mv))
    return out.reshape(list(pts.shape[:-1]) + [4])


def _module(p, prec=None):
    from nerf_sampling_b200.nerf_pytorch.run_nerf_helpers import NeRF

    m, mv = multires_of(p)
    net = NeRF(D=8, W=256, input_ch=d_of(m), input_ch_views=d_of(mv), output_ch=5, skips=[4], use_viewdirs=True)
    net.load_state_dict(p)
    if prec is not None:
        net.precision = prec
    return net.to(DEV)


def _arr(p):
    from nerf_sampling_b200.packing import NERF_KEYS

    host = [p[k].float().contiguous() for k in NERF_KEYS]
    return host, C.cast((C.c_void_p * len(host))(*[t.data_ptr() for t in host]), C.c_void_p)


def _pack(L, p, mr=None):
    """(split image, aux, fast image) by b200nerf_nerf_pack{,_fast}_multires at mr, or by the entry points without sizes."""
    from nerf_sampling_b200 import _lib

    host, arr = _arr(p)
    wpack = torch.full((L.b200nerf_nerf_wpack_bytes(1),), 0xAB, dtype=torch.uint8)
    aux = torch.full((L.b200nerf_nerf_aux_floats(),), float("nan"))
    wf = torch.full((L.b200nerf_nerf_fast_wpack_bytes(),), 0xAB, dtype=torch.uint8)
    if mr is None:
        _lib.check(L.b200nerf_nerf_pack(arr, 1, wpack.data_ptr(), aux.data_ptr()))
        _lib.check(L.b200nerf_nerf_pack_fast(arr, 2, wf.data_ptr()))
    else:
        _lib.check(L.b200nerf_nerf_pack_multires(arr, *mr, 1, wpack.data_ptr(), aux.data_ptr()))
        _lib.check(L.b200nerf_nerf_pack_fast_multires(arr, *mr, 2, wf.data_ptr()))
    return wpack, aux, wf


ALL = [(m, mv) for m in range(1, 11) for mv in range(1, 5)]


# --------------------------------------------------------------------------------------------- CPU: shapes, refusals, layout
@pytest.mark.parametrize("m,mv", ALL)
def test_constructor_matches_oracle_init(m, mv):
    """NeRF(input_ch=3(1+2m), input_ch_views=3(1+2mv), use_viewdirs=True) draws the reference's seeded weights and is served."""
    from nerf_sampling_b200.nerf_pytorch.run_nerf_helpers import NeRF

    torch.manual_seed(100 + 4 * m + mv)
    net = NeRF(D=8, W=256, input_ch=d_of(m), input_ch_views=d_of(mv), output_ch=5, skips=[4], use_viewdirs=True)
    want = init_nerf(m, mv, 100 + 4 * m + mv)
    sd = net.state_dict()
    assert set(sd) == set(want)
    for k in want:
        assert torch.equal(sd[k], want[k]), k
    assert net.multires() == (m, mv)


def test_out_of_range_and_inconsistent_shapes_are_refused(lib):
    """PackedNeRF, NeRF, both C packers and the fp32 colour route name the ranges; PackedNeRF refuses shapes that disagree."""
    from nerf_sampling_b200.nerf_pytorch.run_nerf_helpers import NeRF
    from nerf_sampling_b200.packing import PackedNeRF

    for m, mv, rng in ((0, 4, r"1\.\.10"), (11, 4, r"1\.\.10"), (10, 0, r"1\.\.4"), (10, 5, r"1\.\.4")):
        torch.manual_seed(0)
        p = O.init_nerf(input_ch=d_of(m), input_ch_views=d_of(mv))
        with pytest.raises(ValueError, match=rng):
            PackedNeRF(p, "cpu")
        net = NeRF(D=8, W=256, input_ch=d_of(m), input_ch_views=d_of(mv), output_ch=5, skips=[4], use_viewdirs=True)
        with pytest.raises(NotImplementedError, match=r"1\.\.10 and multires_views in 1\.\.4"):
            net.packed()
        # the C packers take the sizes as arguments
        _, arr = _arr(init_nerf(10, 4, 0))
        buf = torch.empty(lib.b200nerf_nerf_wpack_bytes(1), dtype=torch.uint8)
        aux = torch.empty(lib.b200nerf_nerf_aux_floats())
        assert lib.b200nerf_nerf_pack_multires(arr, m, mv, 1, buf.data_ptr(), aux.data_ptr()) != 0
        assert "multires 1..10 and multires_views 1..4" in lib.b200nerf_last_error().decode()
        wf = torch.empty(lib.b200nerf_nerf_fast_wpack_bytes(), dtype=torch.uint8)
        assert lib.b200nerf_nerf_pack_fast_multires(arr, m, mv, 2, wf.data_ptr()) != 0
        assert "multires 1..10 and multires_views 1..4" in lib.b200nerf_last_error().decode()
        assert lib.b200nerf_nerf_point_ws_floats_multires(100, m, mv) == 0
        assert lib.b200nerf_nerf_point_jvp_multires(None, m, mv, None, None, None, None, 100, None, None, None, None) != 0
        assert "multires_views 1..4" in lib.b200nerf_last_error().decode()
    p = init_nerf(5, 2, 1)
    for k, other in (("pts_linears.5.weight", (4, 2)), ("pts_linears.0.weight", (6, 2))):
        with pytest.raises(ValueError, match=r"expected \(256, \d+\) \(multires \d, multires_views 2\)"):
            PackedNeRF(dict(p, **{k: init_nerf(*other, 1)[k]}), "cpu")
    with pytest.raises(ValueError, match=r"gamma\(viewdir\) .* is 20 wide"):
        PackedNeRF(dict(p, **{"views_linears.0.weight": torch.zeros(128, 276)}), "cpu")
    for bad in (dict(D=7), dict(W=128), dict(use_viewdirs=False)):
        kw = dict(D=8, W=256, input_ch=33, input_ch_views=15, output_ch=5, skips=[4], use_viewdirs=True)
        kw.update(bad)
        with pytest.raises(NotImplementedError, match=r"multires in 1\.\.10"):
            NeRF(**kw).packed()


def test_run_network_checks_the_embedders_against_the_net():
    """Trainer.run_network: an embedder that states its octave count must agree with the network's shapes."""
    from nerf_sampling_b200.nerf_pytorch.run_nerf_helpers import get_embedder
    from nerf_sampling_b200.nerf_pytorch.trainers.Trainer import Trainer
    from nerf_sampling_b200.nerf_pytorch.run_nerf_helpers import NeRF

    net = NeRF(D=8, W=256, input_ch=33, input_ch_views=15, output_ch=5, skips=[4], use_viewdirs=True)
    pts, vd = torch.zeros(2, 3, 3), torch.zeros(2, 3)
    for e, ed, name in ((get_embedder(10, 0, 3)[0], get_embedder(2, 0, 3)[0], "embed_fn"),
                        (get_embedder(5, 0, 3)[0], get_embedder(4, 0, 3)[0], "embeddirs_fn")):
        with pytest.raises(ValueError, match=f"{name} encodes .*multires 5, multires_views 2"):
            Trainer.run_network(None, pts, vd, net, e, ed)


@pytest.mark.parametrize("m,mv", ALL)
def test_pack_layout_equals_padded_10_4_net(lib, m, mv):
    """b200nerf_nerf_pack{,_fast}_multires at (m, mv) write the bytes the 10 / 4 packers write for pad(W); the aux blocks differ only
    in the two recorded sizes.  At 10 / 4 the _multires packers equal the entry points without sizes, aux included."""
    from nerf_sampling_b200.packing import PackedNeRF

    p = init_nerf(m, mv, 7 * m + mv)
    w_new, a_new, f_new = _pack(lib, p, (m, mv))
    w_pad, a_pad, f_pad = _pack(lib, pad(p))
    assert torch.equal(w_new, w_pad)
    assert torch.equal(f_new, f_pad)
    assert float(a_pad[NERF_BA + 1]) == 0.0 and float(a_pad[NERF_BA + 2]) == 0.0
    assert float(a_new[NERF_BA + 1]) == (0.0 if m == 10 else m) and float(a_new[NERF_BA + 2]) == (0.0 if mv == 4 else mv)
    a_new[NERF_BA + 1 : NERF_BA + 3] = 0.0
    assert torch.equal(a_new.view(torch.int32), a_pad.view(torch.int32))
    if (m, mv) == (10, 4):
        w_old, a_old, f_old = _pack(lib, p)
        assert torch.equal(w_new, w_old) and torch.equal(f_new, f_old)
        assert torch.equal(_pack(lib, p, (10, 4))[1].view(torch.int32), a_old.view(torch.int32))
    pk = PackedNeRF(p, "cpu", prec=3)
    assert (pk.multires, pk.multires_views) == (m, mv)
    assert torch.equal(pk.wpack, w_new) and torch.equal(pk.wpack_fast, f_new)


# --------------------------------------------------------------------------------------------- GPU: inference
def _inputs(n, S, seed, nan=False):
    g = torch.Generator().manual_seed(seed)
    ro = (torch.rand(n, 3, generator=g) - 0.5).to(DEV)
    rd = torch.nn.functional.normalize(torch.randn(n, 3, generator=g), dim=-1).to(DEV)
    z = (2.0 + 4.0 * torch.rand(n, S, generator=g)).to(DEV)
    vd = torch.nn.functional.normalize(torch.randn(n, 3, generator=g), dim=-1).to(DEV)
    pts = (torch.rand(n, S, 3, generator=g) * 8 - 4).to(DEV)
    if nan:
        pts[n // 2, S - 1, 1] = float("nan")
        z[n // 3, 0] = float("nan")
    return ro, rd, z, vd, pts


SHAPES = [(1, 1), (3, 5), (130, 1), (77, 13), (1031, 7)]


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [1, 2, 3])
@pytest.mark.parametrize("m,mv", GPU_CASES)
def test_raw_vs_fp64(lib, m, mv, prec):
    """raw at PREC_SPLIT / PREC_FP16 / PREC_FAST on ragged (n, S), z and pts forms, against fp64 of the net at (m, mv); a NaN
    sample poisons only its own row."""
    from nerf_sampling_b200 import ops
    from nerf_sampling_b200.packing import PackedNeRF

    p = init_nerf(m, mv, 11 * m + mv)
    p64 = {k: v.to(DEV, torch.float64) for k, v in p.items()}
    pk = PackedNeRF(p, DEV, prec)
    worst = 0.0
    for n, S in SHAPES + [(300, 4)]:
        ro, rd, z, vd, pts = _inputs(n, S, n + S, nan=(n == 300))
        zpts = ro[:, None, :] + rd[:, None, :] * z[..., None]   # the kernels' rounding: product, then sum
        for got, at in ((ops.nerf_mlp(pk, vd, rays_o=ro, rays_d=rd, z=z), zpts), (ops.nerf_mlp(pk, vd, pts=pts), pts)):
            with torch.no_grad():
                want = run_network(at, vd, p64)
            assert got.shape == (n, S, 4)
            bad = torch.isnan(got).any(-1)
            assert torch.equal(bad, torch.isnan(at).any(-1))
            if n == 300:
                assert int(bad.sum()) == 1
            err = float((got[~bad].double() - want[~bad]).abs().max())
            worst = max(worst, err)
            assert err <= RAW_TOL[prec], (n, S, err)
    print(f"raw (m, mv) = ({m}, {mv}) prec {prec}: max |err| vs fp64 {worst:.2e}")


def _padded_pair(m, mv, seed):
    p = init_nerf(m, mv, seed)
    return p, pad(p)


@pytest.mark.gpu
@pytest.mark.parametrize("m,mv", GPU_CASES)
def test_bitwise_equal_to_padded_net(lib, m, mv):
    """raw at every precision, and raw / d raw / dz of the packed colour path, equal those of the 10 / 4 net built from pad(W), bit
    for bit: the operands differ only in columns that meet zero weights, and octaves j < m are computed as at 10 / 4."""
    from nerf_sampling_b200 import _lib, ops
    from nerf_sampling_b200.packing import PackedNeRF

    p, q = _padded_pair(m, mv, 13 * m + mv)
    ro, rd, z, vd, pts = _inputs(4099, 16, 5)
    for prec in (1, 2, 3):
        a, b = PackedNeRF(p, DEV, prec), PackedNeRF(q, DEV, prec)
        assert torch.equal(ops.nerf_mlp(a, vd, rays_o=ro, rays_d=rd, z=z), ops.nerf_mlp(b, vd, rays_o=ro, rays_d=rd, z=z)), prec
        assert torch.equal(ops.nerf_mlp(a, vd, pts=pts), ops.nerf_mlp(b, vd, pts=pts)), prec
    n = ro.shape[0]
    outs = []
    for pk in (PackedNeRF(p, DEV, 1), PackedNeRF(q, DEV, 1)):
        raw, draw = torch.empty(n, 4, device=DEV), torch.empty(n, 4, device=DEV)
        ws = torch.empty(lib.b200nerf_nerf_point_jvp_packed_ws_bytes(n), dtype=torch.uint8, device=DEV)
        _lib.check(lib.b200nerf_nerf_point_jvp_packed(pk.wpack.data_ptr(), pk.aux.data_ptr(), ro.data_ptr(), rd.data_ptr(), vd.data_ptr(),
                                                      z[:, :1].contiguous().data_ptr(), n, ws.data_ptr(), raw.data_ptr(), draw.data_ptr(),
                                                      torch.cuda.current_stream().cuda_stream))
        outs.append((raw, draw))
    torch.cuda.synchronize()
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


def truncate(p, m, mv):
    """The (m, mv) net that keeps the weights of the first 3 (1 + 2m) / 3 (1 + 2mv) encoding columns of a 10 / 4 net."""
    d, dv = d_of(m), d_of(mv)
    w5 = p["pts_linears.5.weight"]
    return dict(p, **{"pts_linears.0.weight": p["pts_linears.0.weight"][:, :d].contiguous(),
                      "pts_linears.5.weight": torch.cat([w5[:, :d], w5[:, 63:]], 1),
                      "views_linears.0.weight": p["views_linears.0.weight"][:, : 256 + dv].contiguous()})


@pytest.mark.gpu
def test_fast_kernel_guard_band_vs_split_multires_5_2(lib, oracle_models):
    """The guard-band invariants of test_gpu_parity.test_fast_kernel_guard_band_vs_split for a net at (5, 2): the index-list
    re-evaluation reads the sizes from the same aux block.  The net is the oracle's fine net cut to (5, 2), its alpha bias shifted so
    that the last samples of the view straddle sigma = 0 (the band is not empty)."""
    from nerf_sampling_b200 import ops
    from nerf_sampling_b200.packing import PREC_FAST, PREC_FP16, PREC_SPLIT, PackedDepthNet, PackedNeRF

    _, fine, dn = oracle_models
    fine = truncate(fine, 5, 2)
    packed, *_ = O.prepare_rays(200, 200, O.intrinsics(200, 200), c2w=O.pose_spherical(30.0, -30.0, 4.0)[:3, :4])
    ro, rd, vd = (packed[:, a:b].contiguous().to(DEV) for a, b in ((0, 3), (3, 6), (8, 11)))
    z = ops.place_samples(ops.depthnet_forward(PackedDepthNet(dn, DEV, PREC_SPLIT), ro, rd), 32, "uniform", 0.1)
    raw_s = ops.nerf_mlp(PackedNeRF(fine, DEV, PREC_SPLIT), vd, rays_o=ro, rays_d=rd, z=z)
    fine["alpha_linear.bias"] = fine["alpha_linear.bias"] - raw_s[:, -1, 3].nanmedian().cpu()
    raw_s = ops.nerf_mlp(PackedNeRF(fine, DEV, PREC_SPLIT), vd, rays_o=ro, rays_d=rd, z=z)
    raw_h = ops.nerf_mlp(PackedNeRF(fine, DEV, PREC_FP16), vd, rays_o=ro, rays_d=rd, z=z)
    raw_f = ops.nerf_mlp(PackedNeRF(fine, DEV, PREC_FAST), vd, rays_o=ro, rays_d=rd, z=z)
    ws = ops.nerf_mlp.last_guard_ws
    cnt = int(ws[0])
    assert 0 < cnt < ro.shape[0]   # a band, not every ray
    assert float((raw_h - raw_s).abs().max()) <= RAW_TOL[3]
    sign = lambda r: r[:, -1, 3] > 0   # noqa: E731
    flips_h = sign(raw_h) != sign(raw_s)
    assert int((sign(raw_f) != sign(raw_s)).sum()) == 0
    lst = ws[4 : 4 + cnt].long()
    assert bool(((lst % 32) == 31).all())
    flagged = torch.zeros(ro.shape[0], dtype=torch.bool, device=DEV)
    flagged[lst // 32] = True
    assert bool(flagged[flips_h].all())
    assert torch.equal(raw_f.reshape(-1, 4)[lst], raw_s.reshape(-1, 4)[lst])
    rest = torch.ones(raw_f.numel() // 4, dtype=torch.bool, device=DEV)
    rest[lst] = False
    assert torch.equal(raw_f.reshape(-1, 4)[rest], raw_h.reshape(-1, 4)[rest])
    print(f"guard band at (5, 2): {cnt} samples re-evaluated, {int(flips_h.sum())} fp16 sign flips inside it")


# --------------------------------------------------------------------------------------------- GPU: the colour path of training
@pytest.mark.gpu
@pytest.mark.parametrize("route,side", [("split", 37), ("fp32", 37), ("fp32", 5)])
@pytest.mark.parametrize("m,mv", GPU_CASES)
def test_colour_path_vs_fp64_autograd(lib, m, mv, route, side):
    """raw and d raw / d z at one sample per ray (NerfPointFn: the packed split-precision route, or the fp32 route on its tensor-core
    path and, below 32 rays, its CUDA-core path) against fp64 autograd, with the bounds and kink accounting of
    test_gpu_parity.test_nerf_point_jvp_vs_torch."""
    from nerf_sampling_b200 import training

    p = init_nerf(m, mv, 17 * m + mv)
    net = _module(p)
    packed, *_ = O.prepare_rays(side, side, O.intrinsics(side, side), c2w=O.pose_spherical(30.0, -30.0, 4.0)[:3, :4])
    ro, rd, vd = (packed[:, a:b].contiguous().to(DEV) for a, b in ((0, 3), (3, 6), (8, 11)))
    z = (3.0 + torch.rand(ro.shape[0], 1, generator=torch.Generator().manual_seed(2))).to(DEV).requires_grad_(True)
    raw = training.NerfPointFn.apply(z, ro, rd, vd, net.packed() if route == "split" else None, *training.nerf_params(net))
    p64 = {k: v.to(DEV, torch.float64) for k, v in p.items()}
    z2 = z.detach().double().clone().requires_grad_(True)
    pts = ro.double()[:, None, :] + rd.double()[:, None, :] * z2[:, :, None]
    want = run_network(pts, vd.double(), p64)
    rerr = float((raw.double() - want).abs().max())
    assert rerr <= (1e-5 if route == "fp32" else 1e-4)
    worst, kink, errs = 0.0, torch.zeros(ro.shape[0], dtype=torch.bool, device=DEV), []
    for c in range(4):
        gw, = torch.autograd.grad(want[..., c].sum(), z2, retain_graph=True)
        gg, = torch.autograd.grad(raw[..., c].sum(), z, retain_graph=True)
        err = ((gg.double() - gw).abs() / float(gw.abs().max())).reshape(-1)
        errs.append(err)
        kink |= err > 1e-3
    n_kink = int(kink.sum())
    for err in errs:
        if n_kink < ro.shape[0]:
            worst = max(worst, float(err[~kink].max()))
    print(f"d raw / d z at ({m}, {mv}), route {route}, {side * side} rays: max-abs raw error {rerr:.2e}, worst derivative error "
          f"{worst:.2e} of the channel's largest, rays across a ReLU kink: {n_kink}")
    assert n_kink <= max(1, ro.shape[0] // 200)


# --------------------------------------------------------------------------------------------- GPU: the whole path at (5, 2)
def _nerfs_5_2():
    from nerf_sampling_b200.packing import PREC_FAST

    coarse, fine = init_nerf(5, 2, 520), init_nerf(5, 2, 521)
    return (coarse, fine), (_module(coarse, PREC_FAST), _module(fine, PREC_FAST))


def _depthnet(oracle_models):
    from nerf_sampling_b200.depth_nets import DepthNet

    dn = DepthNet(hidden_sizes=[256] * 10, cat_hidden_sizes=[256] * 10, sphere_radius=2.0)
    dn.load_state_dict(oracle_models[2])
    return dn.to(DEV)


def _render(models, H, W, S, **flags):
    from nerf_sampling_b200.nerf_pytorch import nerf_utils
    from nerf_sampling_b200.trainers import DepthNetTrainer

    coarse, fine, dn = models
    tr = DepthNetTrainer(dataset_type="blender", basedir="/tmp", expname="x", no_batching=True, datadir="x", half_res=True, white_bkgd=True,
                         device=DEV, n_layers=10, layer_width=256, N_importance=128, N_samples=64, input_dims_embed=3, distance=0.1,
                         sampling_mode="uniform", n_depth_samples=S, multires=5, multires_views=2, **flags)
    kw = dict(network_fn=coarse, network_fine=fine, depth_network=dn, network_query_fn=None, N_samples=64, N_importance=128, trainer=tr,
              white_bkgd=True, raw_noise_std=0.0, perturb=False, lindisp=True, ndc=False, near=2.0, far=6.0, use_viewdirs=True,
              model_mode="test")
    with torch.no_grad():
        return nerf_utils.render_test(H, W, O.intrinsics(H, W), chunk=H * W, c2w=O.pose_spherical(30.0, -30.0, 4.0)[:3, :4], **kw)


@pytest.mark.gpu
def test_render_test_multires_5_2_vs_oracle(lib, oracle_models, monkeypatch, tmp_path):
    """render_test with NeRFs at (5, 2), DepthNet mode and use_full_nerf, against the oracle's arithmetic on the device (its
    run_network at the weights' octave counts), with the knife-edge rules of test_gpu_parity; then save_state -> load_nerf into fresh
    NeRFs at (5, 2) renders the same image bit for bit."""
    from nerf_sampling_b200.nerf_pytorch import utils

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    monkeypatch.setattr(O, "run_network", lambda pts, vd, p, netchunk=None: run_network(pts, vd, p))
    (c_sd, f_sd), (coarse, fine) = _nerfs_5_2()
    dn = _depthnet(oracle_models)
    pc, pf, pd = (O.params_to(p, DEV) for p in (c_sd, f_sd, oracle_models[2]))
    c2w = O.pose_spherical(30.0, -30.0, 4.0).to(DEV)[:3, :4]
    H = W = 200
    rgb, _, ex = _render((coarse, fine, dn), H, W, 32)
    with torch.no_grad():
        o = O.render_view(H, W, O.intrinsics(H, W), c2w, pc, pf, pd, chunk=32768, n_depth_samples=32, sampling_mode="uniform",
                          distance=0.1)
    assert float((ex["depth_net_z_vals"] - o["depth_net_z_vals"]).abs().max()) <= 5e-5
    err = (rgb - o["depth_net_rgb_map"]).abs().max(-1).values
    knife = o["raw"][..., -1, 3].abs() < SIGMA_GUARD
    print(f"render_test (5, 2): knife-edge rays {int(knife.sum())} of {H * W}; max rgb err elsewhere {float(err[~knife].max()):.2e}")
    assert float(knife.float().mean()) < 0.002
    assert float(err[~knife].max()) <= RGB_TOL
    # use_full_nerf: the vanilla 64 + 128 hierarchical render through both nets
    Hf = Wf = 32
    rgb_f, _, ex_f = _render((coarse, fine, dn), Hf, Wf, 32, use_full_nerf=True)
    with torch.no_grad():
        of = O.render_view(Hf, Wf, O.intrinsics(Hf, Wf), c2w, pc, pf, pd, chunk=32768, mode="full_nerf")
    assert float((ex_f["depth_net_z_vals"] - of["depth_net_z_vals"]).abs().max()) <= 1e-4
    assert float((rgb_f - of["depth_net_rgb_map"]).abs().max()) <= RGB_TOL
    # checkpoint round trip
    path = str(tmp_path / "000005.tar")
    utils.save_state(5, coarse, fine, torch.optim.Adam(list(coarse.parameters()) + list(fine.parameters())), dn,
                     torch.optim.Adam(dn.parameters(), lr=1e-4), path)
    (_, _), (c2, f2) = _nerfs_5_2()
    with torch.no_grad():
        for t in list(c2.parameters()) + list(f2.parameters()):
            t.zero_()
    utils.load_nerf(c2, f2, torch.optim.Adam(list(c2.parameters()) + list(f2.parameters())), torch.load(path, weights_only=False))
    assert (c2.packed().multires, c2.packed().multires_views) == (5, 2)
    rgb2, _, _ = _render((c2, f2, dn), H, W, 32)
    assert torch.equal(rgb, rgb2)


@pytest.mark.gpu
def test_fused_training_step_multires_5_2_equals_autograd_route(lib, oracle_models):
    """The fused training step with NeRFs at (5, 2) (hierarchical target and the packed colour path) against the autograd route on
    the same batch: same losses, same gradients."""
    from nerf_sampling_b200 import training
    from nerf_sampling_b200.depth_nets import DepthNet
    from nerf_sampling_b200.nerf_pytorch import nerf_utils
    from nerf_sampling_b200.trainers import DepthNetTrainer

    import torch.nn.functional as F

    _, (coarse, fine) = _nerfs_5_2()
    dn = DepthNet(hidden_sizes=[256] * 6, cat_hidden_sizes=[256] * 6, sphere_radius=2.0)
    torch.manual_seed(56)
    dn.load_state_dict(O.init_depthnet([256] * 6, [256] * 6))
    dn.to(DEV)
    tr = DepthNetTrainer(dataset_type="blender", basedir="/tmp", expname="x", no_batching=True, datadir="x", half_res=True, white_bkgd=True,
                         device=DEV, n_layers=6, layer_width=256, N_importance=128, N_samples=64, input_dims_embed=3, distance=0.1,
                         sampling_mode="uniform", n_depth_samples=64, perturb=0.0, multires=5, multires_views=2)
    kw = dict(network_fn=coarse, network_fine=fine, depth_network=dn, network_query_fn=None, N_samples=64, N_importance=128, trainer=tr,
              white_bkgd=True, raw_noise_std=0.0, perturb=0.0, lindisp=True, ndc=False, near=2.0, far=6.0, use_viewdirs=True,
              model_mode="train")
    H = W = 800
    tr.H, tr.W, tr.K, tr.chunk = H, W, O.intrinsics(H, W), 32768
    packed, *_ = O.prepare_rays(H, W, O.intrinsics(H, W), c2w=O.pose_spherical(30.0, -30.0, 4.0)[:3, :4])
    sel = torch.randperm(H * W, generator=torch.Generator().manual_seed(3))[:777]
    ro, rd = packed[sel, 0:3].contiguous().to(DEV), packed[sel, 3:6].contiguous().to(DEV)
    target = torch.rand(777, 3, generator=torch.Generator().manual_seed(4)).to(DEV)
    params = list(dn.parameters())
    opt = training.Adam(params, lr=1e-4)
    out = training.fused_render_and_backward(tr, opt, kw, (ro, rd), target)
    assert out is not None
    fused = [p.grad.detach().clone() for p in params]
    for p in params:
        p.grad = None
    rgb, _, ex = nerf_utils.render(H, W, tr.K, rays=(ro, rd), retraw=True, **kw)
    img_loss = torch.mean((rgb - target) ** 2)
    dn_loss = F.mse_loss(ex["depth_net_z_vals"], ex["max_z_vals"])
    torch.autograd.backward([dn_loss, img_loss])
    assert abs(float(out[0]) - float(img_loss)) <= 1e-6 * max(1.0, float(img_loss))
    assert abs(float(out[1]) - float(dn_loss)) <= 1e-6 * max(1.0, float(dn_loss))
    worst = 0.0
    for p, g in zip(params, fused):
        worst = max(worst, float((p.grad - g).abs().max()) / (float(g.abs().max()) + 1e-30))
        assert float((p.grad - g).abs().max()) <= 1e-4 * float(g.abs().max()) + 1e-12
    print(f"fused step with NeRFs at (5, 2): worst gradient {worst:.2e}")
    for p in params:
        p.grad = None
