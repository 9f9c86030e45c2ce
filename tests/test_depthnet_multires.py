"""DepthNet at every positional-encoding size ``multires`` from 1 to 10, in inference and training, against fp64.

``DepthNet(multires=m)`` encodes o and d into d3 = 3 (1 + 2m) columns each and the two sphere hits into 2 d3 (the reference's
``get_embedder(multires, input_dims=3 / 6)``).  Inference folds the branches into a 256-wide first layer whose four 64-column blocks
hold the encodings (the first d3 columns of each, the rest zero) and records m in the packed image; training takes m through the
``_multires`` entry points of csrc/train.cu.  Every check here uses the fp64 reference, kink screening and bounds of
test_depthnet_architectures.py, on networks of m in {1, 4, 5, 10} and the kernels' own fp32 encoding of the rays at that m.
Observed worst values (B200): see DESIGN.md section 5.
"""

import ctypes as C

import pytest
import torch
import torch.nn.functional as F

import test_depthnet_architectures as A
from oracle import nerf_oracle as O

DEV = "cuda"
GPU_MULTIRES = [1, 4, 5, 10]
GPU_ARCHS = {"A": 1000, "C": 1000, "G": 777}   # 10x256, the constructor's default, mixed widths: batch per architecture
RGB_TOL = 1e-3
SIGMA_GUARD = 1e-5


def d3_of(m):
    return 3 * (1 + 2 * m)


def _param_shapes(hidden, cat, m):
    """Parameter shapes in state_dict order at multires m."""
    d3 = d3_of(m)
    shapes = []
    for d in (d3, d3, 2 * d3):
        prev = d
        for h in hidden:
            shapes += [(h, prev + d), (h,)]
            prev = h
    prev = 3 * hidden[-1] + 4 * d3
    for c in cat:
        shapes += [(c, prev), (c,)]
        prev = c
    return shapes + [(1, prev), (1,)]


# --------------------------------------------------------------------------------------------- CPU: constructor
@pytest.mark.parametrize("m", range(1, 11))
def test_constructor_shapes(m):
    """The reference's shapes (depth_net.py:37-108, encoders get_embedder(multires, 3 / 6)) and its seeded weights at every m."""
    from nerf_sampling_b200.depth_nets import DepthNet

    d3, d6 = d3_of(m), 2 * d3_of(m)
    for hidden, cat in (([128] * 6, [128, 128, 128, 128, 256]), ([200, 136, 256], [256, 64])):
        torch.manual_seed(11)
        dn = DepthNet(hidden_sizes=hidden, cat_hidden_sizes=cat, multires=m)
        assert (dn.origin_dims, dn.direction_dims, dn.intersection_points_dim) == (d3, d3, d6)
        assert dn.origin_layers[0].in_features == dn.direction_layers[0].in_features == 2 * d3
        assert dn.intersection_layers[0].in_features == 2 * d6
        for i in range(1, len(hidden)):
            assert dn.origin_layers[i].in_features == dn.direction_layers[i].in_features == hidden[i - 1] + d3
            assert dn.intersection_layers[i].in_features == hidden[i - 1] + d6
        assert dn.cat_layers[0].in_features == 3 * hidden[-1] + d3 + d3 + d6
        torch.manual_seed(11)
        want = O.init_depthnet(hidden, cat, multires=m)
        sd = dn.state_dict()
        assert set(sd) == set(want)
        for k in want:
            assert torch.equal(sd[k], want[k]), k
    if m == 5:   # the reference's TestBaselineSampler numbers
        dn = DepthNet(multires=5)
        assert dn.cat_layers[0].in_features == 3 * 128 + 33 + 33 + 66
        assert dn.to_depth[0].out_features == 1


@pytest.mark.parametrize("m", [0, 11])
def test_out_of_range_multires_is_refused(lib, m):
    """The constructor, the packer (Python and C) and the training entry points name the range."""
    from nerf_sampling_b200 import _lib
    from nerf_sampling_b200.depth_nets import DepthNet
    from nerf_sampling_b200.packing import PackedDepthNet

    with pytest.raises(ValueError, match=r"1\.\.10"):
        DepthNet(multires=m)
    with pytest.raises(ValueError, match=r"1\.\.10"):
        PackedDepthNet(O.init_depthnet([32, 32], [32, 32], multires=m), "cpu")
    hidden, cat = [64, 64], [64, 64]
    sd = O.init_depthnet(hidden, cat, multires=10)
    w = torch.zeros(256, 256)
    b = torch.zeros(256)
    L = _lib.lib()
    wpack = torch.empty(L.b200nerf_depthnet_wpack_bytes(0, 1), dtype=torch.uint8)
    aux = torch.empty(L.b200nerf_depthnet_aux_floats(0))
    assert L.b200nerf_depthnet_pack_multires(w.data_ptr(), b.data_ptr(), None, 0, b.data_ptr(), b.data_ptr(), m, 1, wpack.data_ptr(),
                                             aux.data_ptr()) != 0
    assert "1..10" in L.b200nerf_last_error().decode()
    assert L.b200nerf_depthnet_train_ws_floats_multires(100, 2, A._ints(hidden), 2, A._ints(cat), m) == 0
    assert "1..10" in L.b200nerf_last_error().decode()
    ptrs = (C.c_void_p * len(sd))(*[0x7F0000000000 + 1024 * i for i in range(len(sd))])
    assert L.b200nerf_debug_depthnet_train_route_multires(ptrs, 2, A._ints(hidden), 2, A._ints(cat), m, 100) < 0


# --------------------------------------------------------------------------------------------- CPU: folding and packing
def kernel_input_layout(rays_o, rays_d, m, radius=2.0):
    """The inference kernel's 256-wide input at multires m: four 64-column blocks, the first d3 columns of each used."""
    _, hits = O.sphere_intersections(rays_o, rays_d, torch.tensor([radius], dtype=rays_o.dtype))
    z = torch.zeros(rays_o.shape[0], 64 - d3_of(m), dtype=rays_o.dtype)
    parts = []
    for x in (rays_o, rays_d, hits[:, 0], hits[:, 1]):
        parts += [O.embed(x, m), z]
    return torch.cat(parts, -1)


@pytest.mark.parametrize("m", [1, 5, 10])
@pytest.mark.parametrize("widths", [([256] * 10, [256] * 10), ([200, 136, 256], [256, 256])])
def test_fold_depthnet_matches_literal_network(m, widths):
    """The fold at multires m against the literal fp64 network (O.depthnet_forward) on doubles."""
    from nerf_sampling_b200.packing import fold_depthnet

    torch.manual_seed(3 + m)
    dn = O.init_depthnet(*widths, multires=m)
    H = W = 12
    ro, rd = O.get_rays(H, W, O.intrinsics(H, W), O.pose_spherical(10.0, -40.0, 4.0)[:3, :4])
    ro, rd = ro.reshape(-1, 3).double().contiguous(), rd.reshape(-1, 3).double().contiguous()
    rd[0] = torch.tensor([0.0, 1.0, 0.0], dtype=torch.float64)   # misses the sphere -> NaN depth in both
    p64 = {k: v.double() for k, v in dn.items()}
    want = O.depthnet_forward(p64, ro, rd, multires=m)
    w0, b0, hidden, hw, hb = fold_depthnet(dn)
    for blk in range(4):
        assert float(w0[:, blk * 64 + d3_of(m) : (blk + 1) * 64].abs().max()) == 0.0
    h = F.leaky_relu(kernel_input_layout(ro, rd, m) @ w0.double().T + b0.double(), 0.01)
    for w, b in hidden:
        h = F.leaky_relu(h @ w.double().T + b.double(), 0.01)
    s = torch.sigmoid(h @ hw.double() + hb.double())
    got = (2 * (1 - s) + 6 * s).reshape(-1, 1)
    assert torch.isnan(want[0]) and torch.isnan(got[0])
    assert float((want[1:] - got[1:]).abs().max()) < 2e-5   # the fold's fp32 rounding of w0 / b0
    assert len(hidden) == len(widths[1]) - 1


def test_fold_rejects_inconsistent_shapes():
    from nerf_sampling_b200.packing import fold_depthnet

    sd = O.init_depthnet([64, 64], [64, 64], multires=5)
    bad = dict(sd, **{"intersection_layers.0.weight": O.init_depthnet([64, 64], [64, 64], multires=4)["intersection_layers.0.weight"]})
    with pytest.raises(ValueError, match="multires 5"):
        fold_depthnet(bad)
    bad = dict(sd, **{"cat_layers.0.weight": O.init_depthnet([64, 64], [64, 64], multires=6)["cat_layers.0.weight"]})
    with pytest.raises(ValueError, match="multires 5"):
        fold_depthnet(bad)


def _pack(L, entry, w0, b0, hidden, hw, hb, *mid):
    flat = [t for pair in hidden for t in pair]
    arr = (C.c_void_p * len(flat))(*[t.data_ptr() for t in flat]) if flat else None
    wpack = torch.empty(L.b200nerf_depthnet_wpack_bytes(len(hidden), 1), dtype=torch.uint8)
    aux = torch.full((L.b200nerf_depthnet_aux_floats(len(hidden)),), float("nan"))
    from nerf_sampling_b200 import _lib

    _lib.check(entry(w0.data_ptr(), b0.data_ptr(), C.cast(arr, C.c_void_p) if flat else None, len(hidden), hw.data_ptr(), hb.data_ptr(),
                     *mid, 1, wpack.data_ptr(), aux.data_ptr()))
    return wpack, aux


def test_pack_multires_entry_point(lib):
    """At multires 10 the new pack entry point writes the bytes b200nerf_depthnet_pack writes; below 10 it records m in the aux slot
    after the head bias, and the PackedDepthNet image carries it."""
    from nerf_sampling_b200.packing import PackedDepthNet, fold_depthnet

    for m in (10, 5, 1):
        torch.manual_seed(m)
        sd = O.init_depthnet([256] * 3, [256] * 4, multires=m)
        folded = fold_depthnet(sd)
        w_old, a_old = _pack(lib, lib.b200nerf_depthnet_pack, *folded)
        w_new, a_new = _pack(lib, lib.b200nerf_depthnet_pack_multires, *folded, m)
        assert torch.equal(w_old, w_new)
        slot = 256 * (len(folded[2]) + 2) + 1
        if m == 10:
            assert torch.equal(a_old.view(torch.int32), a_new.view(torch.int32))
        else:
            assert float(a_old[slot]) == 0.0 and float(a_new[slot]) == m
            a_new[slot] = 0.0
            assert torch.equal(a_old.view(torch.int32), a_new.view(torch.int32))
        pk = PackedDepthNet(sd, "cpu")
        assert pk.multires == m and torch.equal(pk.wpack, w_new)
        assert float(pk.aux[slot]) == (0.0 if m == 10 else m)


def test_route_table_at_multires_5(lib):
    """The route query at multires 5 (row strides h + 33 / h + 66, cat_layers.0 K = 3h + 132), at the thresholds 31 / 32 / 2048 /
    2049: the predicates depend on the widths, the batch and the parameters' alignment, so the table is the one of multires 10."""
    for arch in ("A", "C", "G", "I", "L"):
        hidden, cat, mis = A.ARCHS[arch]
        offs, _ = A._flat_offsets(_param_shapes(hidden, cat, 5), mis)
        ptrs = (C.c_void_p * len(offs))(*[0x7F0000000000 + 4 * o for o in offs])
        for n in (31, 32, 2048, 2049):
            got = lib.b200nerf_debug_depthnet_train_route_multires(ptrs, len(hidden), A._ints(hidden), len(cat), A._ints(cat), 5, n)
            assert got == A.expected_route(arch, n), (arch, n, A.route_name(got), A.route_name(A.expected_route(arch, n)))
        assert lib.b200nerf_debug_depthnet_train_route_multires(ptrs, len(hidden), A._ints(hidden), len(cat), A._ints(cat), 10, 1000) == \
            lib.b200nerf_debug_depthnet_train_route(ptrs, len(hidden), A._ints(hidden), len(cat), A._ints(cat), 1000)


# --------------------------------------------------------------------------------------------- fp64 reference at multires m
def encode(ro, rd, m, radius=2.0):
    """[gamma(o) d3 | gamma(d) d3 | gamma([hit_near, hit_far]) 2 d3] in the precision of the rays."""
    _, hits = O.sphere_intersections(ro, rd, torch.tensor([radius], dtype=ro.dtype, device=ro.device))
    return torch.cat([O.embed(ro, m), O.embed(rd, m), O.embed(torch.flatten(hits, start_dim=1), m)], -1)


def fp64_forward(p, enc, m, near=2.0, far=6.0):
    """z and every cat layer's pre-activation of DepthNet on the encoding enc [n, 4 d3], in the precision of p."""
    d3 = d3_of(m)
    enc = enc.to(next(iter(p.values())).dtype)
    e_o, e_d, e_i = enc[:, :d3], enc[:, d3 : 2 * d3], enc[:, 2 * d3 :]

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


_STATE = {}


def _weights(arch, m):
    if ("w", arch, m) not in _STATE:
        hidden, cat, _ = A.ARCHS[arch]
        torch.manual_seed(2000 + 16 * sorted(A.ARCHS).index(arch) + m)
        _STATE[("w", arch, m)] = O.init_depthnet(hidden, cat, multires=m)
    return _STATE[("w", arch, m)]


def _module(arch, m):
    from nerf_sampling_b200.depth_nets import DepthNet

    hidden, cat, _ = A.ARCHS[arch]
    dn = DepthNet(hidden_sizes=hidden, cat_hidden_sizes=cat, multires=m, sphere_radius=2.0)
    dn.load_state_dict(_weights(arch, m))
    return dn.to(DEV)


def _ptrs(ts):
    return (C.c_void_p * len(ts))(*[t.data_ptr() for t in ts])


def _rays(m):
    """The 128 x 128 sphere-hitting rays of test_depthnet_architectures and the encoding the training kernels compute for them at
    multires m (left at the start of the workspace, [n, 4 d3])."""
    if ("rays", m) not in _STATE:
        from nerf_sampling_b200 import _lib, training

        ro, rd, _, _ = A._rays()
        dn = _module("I", m)
        hidden, cat = training.depthnet_arch(dn)
        L = _lib.lib()
        n = ro.shape[0]
        ws = torch.empty(L.b200nerf_depthnet_train_ws_floats_multires(n, len(hidden), A._ints(hidden), len(cat), A._ints(cat), m), device=DEV)
        z = torch.empty(n, 1, device=DEV)
        _lib.check(L.b200nerf_depthnet_train_fwd_multires(_ptrs(training.depthnet_params(dn)), len(hidden), A._ints(hidden), len(cat),
                                                          A._ints(cat), m, ro.data_ptr(), rd.data_ptr(), n, 2.0, 2.0, 6.0, ws.data_ptr(),
                                                          z.data_ptr(), torch.cuda.current_stream().cuda_stream))
        ew = 4 * d3_of(m)
        enc = ws[: n * ew].reshape(n, ew).clone()
        enc64 = encode(ro.double(), rd.double(), m)
        assert float((enc[:, : 2 * d3_of(m)].double() - enc64[:, : 2 * d3_of(m)]).abs().max()) <= 1e-6
        _STATE[("rays", m)] = (ro, rd, enc)
    return _STATE[("rays", m)]


def _pool(arch, m):
    """Kink-free rays of the pool (fp64 pre-activations on the kernel's encoding farther than TAU x rms from zero)."""
    if ("pool", arch, m) not in _STATE:
        ro, rd, enc = _rays(m)
        p64 = {k: v.to(DEV, torch.float64) for k, v in _weights(arch, m).items()}
        with torch.no_grad():
            z, _ = fp64_forward(p64, encode(ro.double(), rd.double(), m), m)
            want = O.depthnet_forward(p64, ro.double(), rd.double(), multires=m)
            assert float((z - want).abs().max()) <= 1e-12, "the fp64 forward of this file drifted from the oracle"
            z, pre = fp64_forward(p64, enc, m)
        assert not bool(torch.isnan(z).any())
        ok = torch.ones(ro.shape[0], dtype=torch.bool, device=DEV)
        for y in pre:
            ok &= y.abs().min(-1).values > A.TAU * float(y.pow(2).mean().sqrt())
        _STATE[("pool", arch, m)] = ok.nonzero().reshape(-1)
    return _STATE[("pool", arch, m)]


def _batch(arch, m, n):
    ro, rd, enc = _rays(m)
    kink_free = _pool(arch, m)
    assert kink_free.numel() >= n
    sel = kink_free[torch.randperm(kink_free.numel(), generator=torch.Generator().manual_seed(n)).to(DEV)[:n]]
    return ro[sel].contiguous(), rd[sel].contiguous(), enc[sel]


def _fp64_grads(arch, m, enc, upstream):
    p64 = {k: v.to(DEV, torch.float64).requires_grad_(True) for k, v in _weights(arch, m).items()}
    z, _ = fp64_forward(p64, enc, m)
    (z * upstream.double().reshape(z.shape)).sum().backward()
    return z.detach(), {k: v.grad for k, v in p64.items()}


CASES = [(a, m) for a in GPU_ARCHS for m in GPU_MULTIRES]


# --------------------------------------------------------------------------------------------- GPU: inference and training
@pytest.mark.gpu
@pytest.mark.parametrize("arch,m", CASES)
def test_inference_vs_fp64(lib, arch, m):
    """DepthNet(multires=m).forward under no_grad (folded branches, mlp_exact_kernel<IN_DEPTHNET> encoding at the image's m) on
    sphere-hitting rays and one miss."""
    dn = _module(arch, m)
    n = GPU_ARCHS[arch]
    ro, rd, enc = _rays(m)
    ro = torch.cat([ro[:n], ro[:1]]).contiguous()
    rd = torch.cat([rd[:n], torch.tensor([[0.0, 1.0, 0.0]], device=DEV)]).contiguous()
    p64 = {k: v.to(DEV, torch.float64) for k, v in _weights(arch, m).items()}
    with torch.no_grad():
        want, _ = fp64_forward(p64, enc[:n], m)
        got = dn(ro, rd)
    assert dn.packed().multires == m
    assert got.shape == (n + 1, 1)
    assert bool(torch.isnan(got[n])), "the ray that misses the sphere must give NaN"
    err = float((got[:n].double() - want).abs().max())
    print(f"inference {arch} multires={m} n={n}: max |dz| {err:.2e}")
    assert err <= A.Z_INFER_TOL


@pytest.mark.gpu
@pytest.mark.parametrize("arch,m", CASES)
def test_training_forward_and_one_pass_backward_vs_fp64(lib, arch, m):
    """DepthNet(multires=m).forward with gradients (b200nerf_depthnet_train_fwd_multires / _bwd_multires) against fp64 autograd."""
    from nerf_sampling_b200 import training

    dn = _module(arch, m)
    n = GPU_ARCHS[arch]
    hidden, cat = training.depthnet_arch(dn)
    route = lib.b200nerf_debug_depthnet_train_route_multires(_ptrs(training.depthnet_params(dn)), len(hidden), A._ints(hidden), len(cat),
                                                             A._ints(cat), m, n)
    assert route == A.expected_route(arch, n), A.route_name(route)
    ro, rd, enc = _batch(arch, m, n)
    w = torch.linspace(0.5, 1.5, n, device=DEV).reshape(n, 1)
    z = dn(ro, rd)
    (z * w).sum().backward()
    z64, want = _fp64_grads(arch, m, enc, w)
    zerr = float((z.detach().double() - z64).abs().max())
    worst = A._worst(((k, p.grad) for k, p in dn.named_parameters()), want)
    print(f"training {arch} multires={m} n={n} [{A.route_name(route)}]: max |dz| {zerr:.2e}; one-pass backward worst {worst[0]} "
          f"{worst[1]:.2e}")
    assert zerr <= A.Z_TRAIN_TOL
    assert worst[1] <= A.TAU_G, worst


@pytest.mark.gpu
@pytest.mark.parametrize("arch,m", CASES)
def test_split_backward_vs_fp64(lib, arch, m):
    """b200nerf_depthnet_train_jac_multires + _bwd_jac_multires with a random-sign dz, with and without the second stream, into
    NaN-filled gradient buffers."""
    from nerf_sampling_b200 import _lib, training

    dn = _module(arch, m)
    n = GPU_ARCHS[arch]
    params = training.depthnet_params(dn)
    names = [k for k, _ in dn.named_parameters()]
    hidden, cat = training.depthnet_arch(dn)
    ro, rd, enc = _batch(arch, m, n)
    L = _lib.lib()
    arch_args = (len(hidden), A._ints(hidden), len(cat), A._ints(cat), m)
    ws = torch.empty(L.b200nerf_depthnet_train_ws_floats_multires(n, *arch_args), device=DEV)
    z = torch.empty(n, 1, device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    _lib.check(L.b200nerf_depthnet_train_fwd_multires(_ptrs(params), *arch_args, ro.data_ptr(), rd.data_ptr(), n, 2.0, 2.0, 6.0,
                                                      ws.data_ptr(), z.data_ptr(), st))
    dz = (torch.randn(n, generator=torch.Generator().manual_seed(7 + n)) / n).to(DEV)
    _, want = _fp64_grads(arch, m, enc, dz)
    args = arch_args + (n, 2.0, 6.0, ws.data_ptr())
    report = []
    for fork in (False, True):
        grads = [torch.full_like(p, float("nan")) for p in params]
        aux = torch.cuda.Stream() if fork else None
        _lib.check(L.b200nerf_depthnet_train_jac_multires(_ptrs(params), *args, _ptrs(grads), st))
        _lib.check(L.b200nerf_depthnet_train_bwd_jac_multires(_ptrs(params), *args, dz.data_ptr(), _ptrs(grads), st,
                                                              aux.cuda_stream if aux else None))
        torch.cuda.synchronize()
        worst = A._worst(zip(names, grads), want)
        report.append(f"{'forked' if fork else 'one stream'} {worst[0]} {worst[1]:.2e}")
        assert worst[1] <= A.TAU_G, (fork, worst)
    print(f"split backward {arch} multires={m} n={n}: worst " + "; ".join(report))


@pytest.mark.gpu
def test_multires_10_entry_points_are_bitwise_unchanged(lib):
    """At multires 10 the _multires training forward and the image of b200nerf_depthnet_pack_multires give the z of the entry
    points without the argument, bit for bit."""
    from nerf_sampling_b200 import _lib, ops, training
    from nerf_sampling_b200.packing import PackedDepthNet, fold_depthnet

    dn = _module("A", 10)
    ro, rd, _ = _rays(10)
    n = 4096
    ro, rd = ro[:n].contiguous(), rd[:n].contiguous()
    hidden, cat = training.depthnet_arch(dn)
    params = _ptrs(training.depthnet_params(dn))
    st = torch.cuda.current_stream().cuda_stream
    ws = torch.empty(lib.b200nerf_depthnet_train_ws_floats(n, len(hidden), A._ints(hidden), len(cat), A._ints(cat)), device=DEV)
    assert ws.numel() == lib.b200nerf_depthnet_train_ws_floats_multires(n, len(hidden), A._ints(hidden), len(cat), A._ints(cat), 10)
    z_old, z_new = torch.empty(n, device=DEV), torch.empty(n, device=DEV)
    _lib.check(lib.b200nerf_depthnet_train_fwd(params, len(hidden), A._ints(hidden), len(cat), A._ints(cat), ro.data_ptr(), rd.data_ptr(),
                                               n, 2.0, 2.0, 6.0, ws.data_ptr(), z_old.data_ptr(), st))
    _lib.check(lib.b200nerf_depthnet_train_fwd_multires(params, len(hidden), A._ints(hidden), len(cat), A._ints(cat), 10, ro.data_ptr(),
                                                        rd.data_ptr(), n, 2.0, 2.0, 6.0, ws.data_ptr(), z_new.data_ptr(), st))
    assert torch.equal(z_old, z_new)
    pk = PackedDepthNet(dn.state_dict(), DEV)
    w_old, a_old = _pack(lib, lib.b200nerf_depthnet_pack, *fold_depthnet(dn.state_dict()))
    pk_old = PackedDepthNet(dn.state_dict(), DEV)
    pk_old.wpack, pk_old.aux = w_old.to(DEV), a_old.to(DEV)
    with torch.no_grad():
        assert torch.equal(ops.depthnet_forward(pk, ro, rd, 2.0, 2.0, 6.0), ops.depthnet_forward(pk_old, ro, rd, 2.0, 2.0, 6.0))


# --------------------------------------------------------------------------------------------- GPU: the whole path at multires 5
def _render(models, H, W, S):
    from nerf_sampling_b200.nerf_pytorch import nerf_utils
    from nerf_sampling_b200.trainers import DepthNetTrainer

    coarse, fine, dn = models
    tr = DepthNetTrainer(dataset_type="blender", basedir="/tmp", expname="x", no_batching=True, datadir="x", half_res=True, white_bkgd=True,
                         device=DEV, n_layers=6, layer_width=128, N_importance=128, N_samples=64, input_dims_embed=3, distance=0.1,
                         sampling_mode="uniform", n_depth_samples=S)
    kw = dict(network_fn=coarse, network_fine=fine, depth_network=dn, network_query_fn=None, N_samples=64, N_importance=128, trainer=tr,
              white_bkgd=True, raw_noise_std=0.0, perturb=False, lindisp=True, ndc=False, near=2.0, far=6.0, use_viewdirs=True,
              model_mode="test")
    with torch.no_grad():
        return nerf_utils.render_test(H, W, O.intrinsics(H, W), chunk=H * W, c2w=O.pose_spherical(30.0, -30.0, 4.0)[:3, :4], **kw)


def _nerfs(oracle_models):
    from nerf_sampling_b200.nerf_pytorch.run_nerf_helpers import NeRF
    from nerf_sampling_b200.packing import PREC_FAST

    out = []
    for sd in oracle_models[:2]:
        net = NeRF(D=8, W=256, input_ch=63, input_ch_views=27, output_ch=5, skips=[4], use_viewdirs=True)
        net.load_state_dict(sd)
        net.precision = PREC_FAST
        out.append(net.to(DEV))
    return out


@pytest.mark.gpu
def test_render_test_multires_5_vs_oracle(lib, oracle_models, tmp_path):
    """render_test with DepthNet(multires=5) (the constructor's default widths) against the oracle's arithmetic at multires 5 on the
    device: rgb within 1e-3 off the knife edge; then save_state -> load_depth_network into a fresh DepthNet(multires=5) renders the
    same image bit for bit."""
    from nerf_sampling_b200.depth_nets import DepthNet
    from nerf_sampling_b200.nerf_pytorch import utils

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    coarse, fine = _nerfs(oracle_models)
    torch.manual_seed(5)
    dn = DepthNet(multires=5, sphere_radius=2.0).to(DEV)
    H = W = 200
    S = 32
    rgb, _, ex = _render((coarse, fine, dn), H, W, S)
    p_dn = {k: v.detach() for k, v in dn.state_dict().items()}
    p_fine = O.params_to(oracle_models[1], DEV)
    c2w = O.pose_spherical(30.0, -30.0, 4.0).to(DEV)
    with torch.no_grad():
        packed, *_ = O.prepare_rays(H, W, O.intrinsics(H, W), c2w=c2w[:3, :4])
        ro, rd, vd = packed[:, 0:3], packed[:, 3:6], packed[:, -3:]
        z_mean = O.depthnet_forward(p_dn, ro, rd, multires=5)
        pts, z = O.place_samples(ro, rd, z_mean, S, "uniform", 0.1)
        raw = O.run_network(pts, vd, p_fine)
        want, *_ = O.raw2outputs(raw, z, rd, 0.0, True)
    zerr = float((ex["depth_net_z_vals"].reshape(-1, S) - z).abs().max())
    err = (rgb.reshape(-1, 3) - want).abs().max(-1).values
    knife = raw[:, -1, 3].abs() < SIGMA_GUARD
    print(f"render_test multires=5: max |dz| {zerr:.2e}; knife-edge rays {int(knife.sum())} of {H * W}; max rgb err elsewhere "
          f"{float(err[~knife].max()):.2e}")
    assert float(knife.float().mean()) < 0.002
    assert zerr <= 5e-5
    assert float(err[~knife].max()) <= RGB_TOL
    path = str(tmp_path / "000005.tar")
    utils.save_state(5, coarse, fine, torch.optim.Adam(list(coarse.parameters()) + list(fine.parameters())), dn,
                     torch.optim.Adam(dn.parameters(), lr=1e-4), path)
    dn2 = DepthNet(multires=5, sphere_radius=2.0).to(DEV)
    utils.load_depth_network(dn2, torch.optim.Adam(dn2.parameters(), lr=1e-4), torch.load(path, weights_only=False))
    rgb2, _, _ = _render((coarse, fine, dn2), H, W, S)
    assert torch.equal(rgb, rgb2)


@pytest.mark.gpu
def test_fused_training_step_multires_5_equals_autograd_route(lib, oracle_models):
    """A DepthNetTrainer(n_layers=6, layer_width=256) whose depth network is swapped for a DepthNet(multires=5): the fused step
    (fused chain, split-K cat_layers.0 at K = 3 x 256 + 132) against the autograd route on the same batch."""
    from nerf_sampling_b200 import training
    from nerf_sampling_b200.depth_nets import DepthNet
    from nerf_sampling_b200.nerf_pytorch import nerf_utils

    coarse, fine = _nerfs(oracle_models)
    dn = DepthNet(hidden_sizes=[256] * 6, cat_hidden_sizes=[256] * 6, multires=5, sphere_radius=2.0)
    torch.manual_seed(55)
    dn.load_state_dict(O.init_depthnet([256] * 6, [256] * 6, multires=5))
    dn.to(DEV)
    tr, kw = A._trainer_kw((coarse, fine, dn), 6, 256)
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
    print(f"fused step, DepthNet(multires=5) 6x256: worst gradient {worst:.2e}")
    for p in params:
        p.grad = None
