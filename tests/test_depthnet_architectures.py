"""DepthNet at every architecture route of the training passes (csrc/train.cu) and of inference, against fp64.

The architecture, the batch size and the alignment of the parameters pick the kernels of a training step: collapsed branches
(weight-only recurrences on 2-CTA clusters) or literal per-layer branches, the fused split-precision cat chain or per-layer 3xTF32
products, split-K ``cat_layers.0``, the split backward or the one-pass one, the tensor-core or the CUDA-core one-pass backward.  Each
case below takes a different set of those routes (``b200nerf_debug_depthnet_train_route`` reports which; the CPU test pins the
table, the GPU tests assert that the route they ran is the one the table names) and is held against an fp64 evaluation of the same
network, differentiated by torch autograd.  That evaluation (``fp64_forward``) is pinned to ``oracle.nerf_oracle.depthnet_forward``
on doubles to 1e-12 and is run on the ray encoding the kernels compute (the reference's fp32 sphere hits: see ``_rays``).

Gradients are compared on kink-free rays only.  The derivative of a LeakyReLU network jumps where a pre-activation changes sign, so
a ray with a hidden value within rounding distance of zero may legitimately take the other slope than fp64 (DESIGN.md §7b).  A ray
is kept when every cat-layer pre-activation lies farther than TAU x rms(layer) from zero in fp64; TAU is well above the kernels'
pre-activation error (fused chain: ~2^-17 per link), so every route is held to one tight bound, TAU_G of each tensor's largest
entry.  Observed worst tensor on kink-free rays (B200, 1000 W power limit), one-pass / split backward: CUDA-core path below 32 rays
1.7e-6 / 2.0e-5; collapsed + fused chain 2.6e-5 / 3.5e-5; collapsed + per-layer chain 3.1e-5 / 2.7e-5; literal branches 3.2e-5 /
3.1e-5; misaligned parameters (L) 4.4e-5 / 4.2e-5.  Depths: training 1.6e-6, inference 2.4e-6.  The kernels' fp32 encoding differs
from an fp64 one by up to 1.2e-3 (2^9 octave of the sphere hits), which is why the reference takes the kernel's encoding.
"""

import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from oracle import nerf_oracle as O

DEV = "cuda"
COLLAPSED, FUSED_CHAIN, SPLIT_CAT0, SPLIT_BACKWARD, TENSOR_PATH = 1, 2, 4, 8, 16   # b200nerf.h B200NERF_ROUTE_*
TAU = 1e-4      # kink screen: |pre-activation| > TAU * rms(layer) on every cat layer
TAU_G = 1e-4    # gradient bound, per tensor, of its largest entry (2x the worst observed, module docstring)
Z_TRAIN_TOL = 1e-5
Z_INFER_TOL = 2e-5

# id: (branch widths, cat widths, misaligned parameters)
ARCHS = {
    "A": ([256] * 10, [256] * 10, False),                 # the reference's experiments (run.py: n_layers=10, layer_width=256)
    "B": ([256] * 6, [256] * 6, False),                   # DepthNetTrainer's default n_layers=6
    "C": ([128] * 6, [128, 128, 128, 128, 256], False),   # DepthNet()'s constructor default
    "D": ([256] * 11, [256] * 11, False),                 # no aux room for the fused chain; 17 dz-scaled problems
    "E": ([256] * 12, [256] * 12, False),                 # CH_MAXL branch layers; inference has one hidden layer too many
    "F": ([256] * 13, [256] * 2, False),                  # more branch layers than the chain kernels hold
    "G": ([200, 136, 256], [256, 256], False),            # mixed widths: partial 32-row blocks of the branch chain
    "H": ([70] * 3, [96], False),                         # width not a multiple of 4, one cat layer
    "I": ([64] * 2, [64, 32], False),                     # tiny widths
    "J": ([512] * 2, [256] * 3, False),                   # branches wider than 256
    "K": ([256] * 3, [512, 256], False),                  # a cat layer wider than 256
    "L": ([256] * 10, [256] * 10, True),                  # A with every parameter at a 4-byte offset
}
ALL = COLLAPSED | FUSED_CHAIN | SPLIT_CAT0 | SPLIT_BACKWARD | TENSOR_PATH
# route at 32 <= n <= 2048 and at n > 2048; every architecture takes route 0 below 32 rays
ROUTES = {
    "A": (ALL, ALL & ~SPLIT_CAT0),
    "B": (ALL, ALL & ~SPLIT_CAT0),
    "C": (COLLAPSED | SPLIT_BACKWARD | TENSOR_PATH,) * 2,
    "D": (COLLAPSED | SPLIT_BACKWARD | TENSOR_PATH,) * 2,
    "E": (COLLAPSED | SPLIT_BACKWARD | TENSOR_PATH,) * 2,
    "F": (TENSOR_PATH,) * 2,
    "G": (ALL, ALL & ~SPLIT_CAT0),
    "H": (TENSOR_PATH,) * 2,
    "I": (COLLAPSED | SPLIT_BACKWARD | TENSOR_PATH,) * 2,
    "J": (TENSOR_PATH,) * 2,
    "K": (COLLAPSED | SPLIT_BACKWARD | TENSOR_PATH,) * 2,
    "L": (TENSOR_PATH,) * 2,
}
RAYS = {"A": [1, 7, 8, 31, 32, 33, 129, 2048, 2049, 4096], "B": [1000], "C": [1000], "D": [1000], "E": [300], "F": [300], "G": [777],
        "H": [333], "I": [100], "J": [300], "K": [300], "L": [1000]}
CASES = [(a, n) for a in ARCHS for n in RAYS[a]]
INFER_CASES = [(a, n) for a in ARCHS if a not in ("E", "K") for n in RAYS[a]] + [("A", n) for n in (127, 128)]
REJECTED = {"E": "n_hidden=11 out of range", "K": "not supported"}


def expected_route(arch, n):
    if n < 32:
        return 0
    return ROUTES[arch][0] if n <= 2048 else ROUTES[arch][1]


def route_name(mask):
    names = ("collapsed", "fused-chain", "split-cat0", "split-backward", "tensor-path")
    return "+".join(s for i, s in enumerate(names) if mask >> i & 1) or "literal+per-layer+CUDA-core"


def _ints(v):
    return (C.c_int * len(v))(*v)


def _param_shapes(hidden, cat):
    """Parameter shapes in state_dict order (the order of the training entry points)."""
    shapes = []
    for d in (63, 63, 126):
        prev = d
        for h in hidden:
            shapes += [(h, prev + d), (h,)]
            prev = h
    prev = 3 * hidden[-1] + 252
    for c in cat:
        shapes += [(c, prev), (c,)]
        prev = c
    return shapes + [(1, prev), (1,)]


def _flat_offsets(shapes, misaligned):
    """Float offsets of the parameters packed back to back in one buffer; misaligned: the buffer starts one float in."""
    offs, o = [], 1 if misaligned else 0
    for s in shapes:
        offs.append(o)
        n = 1
        for x in s:
            n *= x
        o += n if misaligned else (n + 3) // 4 * 4
    return offs, o


def _route(lib, ptrs, hidden, cat, n):
    arr = (C.c_void_p * len(ptrs))(*ptrs)
    return lib.b200nerf_debug_depthnet_train_route(arr, len(hidden), _ints(hidden), len(cat), _ints(cat), n)


# --------------------------------------------------------------------------------------------- CPU: the route table
def test_route_table(lib):
    """Every row of the table at its own batch and at the thresholds 31 / 32 / 2048 / 2049, on fake pointer values laid out as
    the GPU tests lay out their parameters (16-byte aligned tensors, or all of them at a 4-byte offset for L)."""
    for arch, (hidden, cat, mis) in ARCHS.items():
        offs, _ = _flat_offsets(_param_shapes(hidden, cat), mis)
        ptrs = [0x7F0000000000 + 4 * o for o in offs]
        for n in sorted(set(RAYS[arch] + [31, 32, 2048, 2049])):
            got = _route(lib, ptrs, hidden, cat, n)
            assert got == expected_route(arch, n), (arch, n, route_name(got), route_name(expected_route(arch, n)))
    # one misaligned tensor is enough to leave the collapsed / fused routes
    hidden, cat, _ = ARCHS["A"]
    offs, _ = _flat_offsets(_param_shapes(hidden, cat), False)
    for k in (2 * 10 + 4, 2 * 30 + 2):   # a branch weight, a cat weight
        ptrs = [0x7F0000000000 + 4 * o for o in offs]
        ptrs[k] += 4
        want = TENSOR_PATH if k < 60 else COLLAPSED | SPLIT_BACKWARD | TENSOR_PATH
        assert _route(lib, ptrs, hidden, cat, 1000) == want, k
    ptrs = [0x7F0000000000 + 4 * o for o in offs]
    assert _route(lib, ptrs, hidden, cat, -1) < 0
    assert _route(lib, ptrs, hidden, [], 100) < 0
    assert lib.b200nerf_debug_depthnet_train_route(None, 10, _ints(hidden), 10, _ints(cat), 100) < 0
    assert _route(lib, ptrs, [256] * 9 + [0], cat, 100) < 0


@pytest.mark.parametrize("arch", sorted(REJECTED))
def test_inference_rejects_unservable_architectures(arch):
    """E: eleven folded hidden layers, one more than the inference kernel's bias block holds; K: a cat layer wider than its 256-wide
    tile.  Packing must refuse them with a message instead of returning numbers."""
    from nerf_sampling_b200 import _lib
    from nerf_sampling_b200.packing import PackedDepthNet

    hidden, cat, _ = ARCHS[arch]
    torch.manual_seed(5)
    sd = O.init_depthnet(hidden, cat)
    with pytest.raises((_lib.B200NerfError, ValueError), match=REJECTED[arch]):
        PackedDepthNet(sd, "cpu")


# --------------------------------------------------------------------------------------------- fp64 reference
def encode(ro, rd, radius=2.0):
    """[gamma(o) 63 | gamma(d) 63 | gamma([hit_near, hit_far]) 126] in the precision of the rays (oracle.depthnet_forward's op order)."""
    _, hits = O.sphere_intersections(ro, rd, torch.tensor([radius], dtype=ro.dtype, device=ro.device))
    return torch.cat([O.embed(ro, 10), O.embed(rd, 10), O.embed(torch.flatten(hits, start_dim=1), 10)], -1)


def fp64_forward(p, enc, near=2.0, far=6.0):
    """z and every cat layer's pre-activation of DepthNet on the encoding enc [n, 252], in the precision of p."""
    enc = enc.to(next(iter(p.values())).dtype)
    e_o, e_d, e_i = enc[:, :63], enc[:, 63:126], enc[:, 126:]

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


def _weights(arch):
    """Seeded fp32 weights of the architecture (reference construction order)."""
    if ("w", arch) not in _STATE:
        hidden, cat, _ = ARCHS[arch]
        torch.manual_seed(1000 + sorted(ARCHS).index(arch))
        _STATE[("w", arch)] = O.init_depthnet(hidden, cat)
    return _STATE[("w", arch)]


def _rays():
    """128 x 128 rays of a view in which every ray hits the sphere, and the encoding the training kernels compute for them.

    The encoding is the reference's fp32 arithmetic (sphere hits in its op order, then up to the 2^9 octave), so a one-ulp
    difference in a hit point moves an encoding entry by ~1e-4: the fp64 reference evaluates the network on the kernel's own
    encoding, which b200nerf_depthnet_train_fwd leaves at the start of its workspace ([n, 252]).  The encoding itself is pinned
    against the reference elsewhere (the DepthNet depths of test_gpu_parity); here it is compared with fp64 for the record."""
    if "rays" not in _STATE:
        from nerf_sampling_b200 import _lib, training

        c2w = O.pose_spherical(30.0, -30.0, 4.0)[:3, :4]
        packed, *_ = O.prepare_rays(128, 128, O.intrinsics(128, 128), c2w=c2w)
        ro, rd = packed[:, 0:3].contiguous().to(DEV), packed[:, 3:6].contiguous().to(DEV)
        m = _module("I")
        params = training.depthnet_params(m)
        hidden, cat = training.depthnet_arch(m)
        L = _lib.lib()
        n = ro.shape[0]
        ws = torch.empty(L.b200nerf_depthnet_train_ws_floats(n, len(hidden), _ints(hidden), len(cat), _ints(cat)), device=DEV)
        z = torch.empty(n, 1, device=DEV)
        arr = (C.c_void_p * len(params))(*[t.data_ptr() for t in params])
        _lib.check(L.b200nerf_depthnet_train_fwd(arr, len(hidden), _ints(hidden), len(cat), _ints(cat), ro.data_ptr(), rd.data_ptr(), n,
                                                 2.0, 2.0, 6.0, ws.data_ptr(), z.data_ptr(), torch.cuda.current_stream().cuda_stream))
        enc = ws[: n * 252].reshape(n, 252).clone()
        enc64 = encode(ro.double(), rd.double())
        assert float((enc[:, :126].double() - enc64[:, :126]).abs().max()) <= 1e-6   # o and d: no hit point in front of the octaves
        _STATE["rays"] = (ro, rd, enc, float((enc.double() - enc64).abs().max()))
    return _STATE["rays"]


def _pool(arch):
    """The kink-free rays of the pool for this architecture's weights (fp64 pre-activations on the kernel's encoding)."""
    if ("pool", arch) not in _STATE:
        ro, rd, enc, _ = _rays()
        p64 = {k: v.to(DEV, torch.float64) for k, v in _weights(arch).items()}
        with torch.no_grad():
            z, _ = fp64_forward(p64, encode(ro.double(), rd.double()))
            want = O.depthnet_forward(p64, ro.double(), rd.double())
            assert float((z - want).abs().max()) <= 1e-12, "the fp64 forward of this file drifted from the oracle"
            z, pre = fp64_forward(p64, enc)
        assert not bool(torch.isnan(z).any())
        ok = torch.ones(ro.shape[0], dtype=torch.bool, device=DEV)
        for y in pre:
            rms = float(y.pow(2).mean().sqrt())
            ok &= y.abs().min(-1).values > TAU * rms
        _STATE[("pool", arch)] = ok.nonzero().reshape(-1)
    return _STATE[("pool", arch)]


def _batch(arch, n):
    """n kink-free rays drawn from the pool: rays_o, rays_d, the kernel's encoding of them, and how many pool rays were screened out."""
    ro, rd, enc, _ = _rays()
    kink_free = _pool(arch)
    assert kink_free.numel() >= n, f"{arch}: only {kink_free.numel()} kink-free rays for a batch of {n}"
    sel = kink_free[torch.randperm(kink_free.numel(), generator=torch.Generator().manual_seed(n)).to(DEV)[:n]]
    return ro[sel].contiguous(), rd[sel].contiguous(), enc[sel], ro.shape[0] - kink_free.numel()


def _module(arch):
    """The mirror DepthNet on the device with the seeded weights; L: every parameter a view at a 4-byte offset into one buffer."""
    from nerf_sampling_b200.depth_nets import DepthNet
    from nerf_sampling_b200 import training

    hidden, cat, mis = ARCHS[arch]
    m = DepthNet(hidden_sizes=hidden, cat_hidden_sizes=cat, sphere_radius=2.0)
    m.load_state_dict(_weights(arch))
    m.to(DEV)
    if mis:
        params = training.depthnet_params(m)
        offs, total = _flat_offsets([tuple(p.shape) for p in params], True)
        flat = torch.zeros(total, device=DEV)
        views = {}
        for p, o in zip(params, offs):
            v = flat[o:o + p.numel()].view_as(p)
            v.copy_(p.detach())
            views[id(p)] = torch.nn.Parameter(v)
        for mod in m.modules():
            if isinstance(mod, torch.nn.Linear):
                mod.weight, mod.bias = views[id(mod.weight)], views[id(mod.bias)]
        assert all(p.data_ptr() % 16 == 4 for p in training.depthnet_params(m))
        m.__dict__["_flat"] = flat
    return m


def _route_of(lib, m, n):
    from nerf_sampling_b200 import training

    hidden, cat = training.depthnet_arch(m)
    return _route(lib, [p.data_ptr() for p in training.depthnet_params(m)], hidden, cat, n)


def _fp64_grads(arch, enc, upstream):
    """fp64 z on the encoding enc and the gradients of sum(z * upstream) for every parameter, by name."""
    p64 = {k: v.to(DEV, torch.float64).requires_grad_(True) for k, v in _weights(arch).items()}
    z, _ = fp64_forward(p64, enc)
    (z * upstream.double().reshape(z.shape)).sum().backward()
    return z.detach(), {k: v.grad for k, v in p64.items()}


def _worst(named_got, want):
    """(name, error / largest entry) of the worst tensor."""
    worst = ("", 0.0)
    for k, g in named_got:
        assert g is not None and bool(torch.isfinite(g).all()), k
        rel = float((g.double() - want[k]).abs().max()) / float(want[k].abs().max())
        worst = max(worst, (k, rel), key=lambda t: t[1])
    return worst


# --------------------------------------------------------------------------------------------- GPU: inference
@pytest.mark.gpu
@pytest.mark.parametrize("arch,n", INFER_CASES)
def test_inference_vs_fp64(lib, arch, n):
    """DepthNet.forward under no_grad (folded branches, mlp_exact_kernel<IN_DEPTHNET>) on n sphere-hitting rays and one miss."""
    m = _module(arch)
    ro, rd, enc, enc_err = _rays()
    ro = torch.cat([ro[:n], ro[:1]]).contiguous()
    rd = torch.cat([rd[:n], torch.tensor([[0.0, 1.0, 0.0]], device=DEV)]).contiguous()
    p64 = {k: v.to(DEV, torch.float64) for k, v in _weights(arch).items()}
    with torch.no_grad():
        want, _ = fp64_forward(p64, enc[:n])
        full = O.depthnet_forward(p64, ro.double(), rd.double())
        got = m(ro, rd)
    assert got.shape == (n + 1, 1)
    assert bool(torch.isnan(full[n])) and bool(torch.isnan(got[n])), "the ray that misses the sphere must give NaN"
    err = float((got[:n].double() - want).abs().max())
    print(f"inference {arch} n={n}: n_hidden {m.packed().n_hidden}, max |dz| {err:.2e} (against fp64 from the rays: "
          f"{float((got[:n].double() - full[:n]).abs().max()):.2e}; fp32 encoding vs fp64 {enc_err:.1e})")
    assert err <= Z_INFER_TOL


@pytest.mark.gpu
@pytest.mark.parametrize("arch", sorted(REJECTED))
def test_inference_rejects_unservable_architectures_on_device(lib, arch):
    from nerf_sampling_b200 import _lib

    m = _module(arch)
    ro, rd, _, _ = _rays()
    with torch.no_grad(), pytest.raises((_lib.B200NerfError, ValueError), match=REJECTED[arch]):
        m(ro[:64], rd[:64])


# --------------------------------------------------------------------------------------------- GPU: training
@pytest.mark.gpu
@pytest.mark.parametrize("arch,n", CASES)
def test_training_forward_and_one_pass_backward_vs_fp64(lib, arch, n):
    """DepthNetTrainFn (DepthNet.forward with gradients): z, then autograd's backward (b200nerf_depthnet_train_bwd) with one-sign
    upstream weights, every parameter tensor against fp64 autograd of the same network on the same encoding."""
    m = _module(arch)
    route = _route_of(lib, m, n)
    assert route == expected_route(arch, n), (route_name(route), route_name(expected_route(arch, n)))
    ro, rd, enc, screened = _batch(arch, n)
    w = torch.linspace(0.5, 1.5, n, device=DEV).reshape(n, 1)   # one sign: no cancellation in the bias sums
    z = m(ro, rd)
    (z * w).sum().backward()
    z64, want = _fp64_grads(arch, enc, w)
    zerr = float((z.detach().double() - z64).abs().max())
    worst = _worst(((k, p.grad) for k, p in m.named_parameters()), want)
    print(f"training {arch} n={n} [{route_name(route)}]: {screened} of {128 * 128} pool rays screened out; max |dz| {zerr:.2e}; "
          f"one-pass backward worst {worst[0]} {worst[1]:.2e}")
    assert zerr <= Z_TRAIN_TOL
    assert worst[1] <= TAU_G, worst


@pytest.mark.gpu
@pytest.mark.parametrize("arch,n", CASES)
def test_split_backward_vs_fp64(lib, arch, n):
    """b200nerf_depthnet_train_jac + _bwd_jac with a random-sign dz, with the branch chain forked onto a second stream and without,
    into gradient buffers prefilled with NaN (they must be written, not accumulated).  Where the split backward does not apply,
    _bwd_jac runs the one-pass backward: that fallback is checked too."""
    from nerf_sampling_b200 import _lib, training

    m = _module(arch)
    params = training.depthnet_params(m)
    names = [k for k, _ in m.named_parameters()]
    hidden, cat = training.depthnet_arch(m)
    route = _route_of(lib, m, n)
    assert route == expected_route(arch, n)
    ro, rd, enc, _ = _batch(arch, n)
    L = _lib.lib()
    ptrs = lambda ts: (C.c_void_p * len(ts))(*[t.data_ptr() for t in ts])  # noqa: E731
    ws = torch.empty(L.b200nerf_depthnet_train_ws_floats(n, len(hidden), _ints(hidden), len(cat), _ints(cat)), device=DEV)
    z = torch.empty(n, 1, device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    _lib.check(L.b200nerf_depthnet_train_fwd(ptrs(params), len(hidden), _ints(hidden), len(cat), _ints(cat), ro.data_ptr(), rd.data_ptr(),
                                             n, 2.0, 2.0, 6.0, ws.data_ptr(), z.data_ptr(), st))
    dz = (torch.randn(n, generator=torch.Generator().manual_seed(7 + n)) / n).to(DEV)
    _, want = _fp64_grads(arch, enc, dz)
    args = (len(hidden), _ints(hidden), len(cat), _ints(cat), n, 2.0, 6.0, ws.data_ptr())
    report = []
    for fork in (False, True):
        grads = [torch.full_like(p, float("nan")) for p in params]
        aux = torch.cuda.Stream() if fork else None
        _lib.check(L.b200nerf_depthnet_train_jac(ptrs(params), *args, ptrs(grads), st))
        _lib.check(L.b200nerf_depthnet_train_bwd_jac(ptrs(params), *args, dz.data_ptr(), ptrs(grads), st, aux.cuda_stream if aux else None))
        torch.cuda.synchronize()
        worst = _worst(zip(names, grads), want)
        report.append(f"{'forked' if fork else 'one stream'} {worst[0]} {worst[1]:.2e}")
        assert worst[1] <= TAU_G, (fork, worst)
    print(f"split backward {arch} n={n} [{route_name(route)}]: worst " + "; ".join(report))


def _trainer_kw(models, n_layers, width):
    from nerf_sampling_b200.trainers import DepthNetTrainer

    b_coarse, b_fine, b_dn = models
    tr = DepthNetTrainer(dataset_type="blender", basedir="/tmp", expname="x", no_batching=True, datadir="x", half_res=True, white_bkgd=True,
                         device=DEV, n_layers=n_layers, layer_width=width, N_importance=128, N_samples=64, input_dims_embed=3, distance=0.1,
                         sampling_mode="uniform", n_depth_samples=64, perturb=0.0)
    kw = dict(network_fn=b_coarse, network_fine=b_fine, depth_network=b_dn, network_query_fn=None, N_samples=64, N_importance=128,
              trainer=tr, white_bkgd=True, raw_noise_std=0.0, perturb=0.0, lindisp=True, ndc=False, near=2.0, far=6.0,
              use_viewdirs=True, model_mode="train")
    return tr, kw


@pytest.mark.gpu
@pytest.mark.parametrize("width", [256, 128])
def test_fused_training_step_equals_autograd_route_trainer_default(lib, oracle_models, width):
    """training.fused_render_and_backward for the DepthNet that DepthNetTrainer(n_layers=6, layer_width=256 / 128) builds
    (256: fused chain + split-K cat_layers.0; 128: per-layer chain, non-fused Jacobian pass), against the autograd route on the
    same batch: same losses, same gradients."""
    from nerf_sampling_b200 import training
    from nerf_sampling_b200.depth_nets import DepthNet
    from nerf_sampling_b200.nerf_pytorch import nerf_utils
    from nerf_sampling_b200.nerf_pytorch.run_nerf_helpers import NeRF
    from nerf_sampling_b200.packing import PREC_FAST

    coarse, fine, _ = oracle_models

    def nerf(sd):
        net = NeRF(D=8, W=256, input_ch=63, input_ch_views=27, output_ch=5, skips=[4], use_viewdirs=True)
        net.load_state_dict(sd)
        net.precision = PREC_FAST
        return net.to(DEV)

    dn = DepthNet(hidden_sizes=[width] * 6, cat_hidden_sizes=[width] * 6, sphere_radius=2.0)   # as create_nerf_model builds it
    torch.manual_seed(77)
    dn.load_state_dict(O.init_depthnet([width] * 6, [width] * 6))
    dn.to(DEV)
    models = (nerf(coarse), nerf(fine), dn)
    tr, kw = _trainer_kw(models, 6, width)
    assert dn.origin_layers[-1].out_features == tr.layer_width and len(dn.origin_layers) == tr.n_layers
    H = W = 800
    tr.H, tr.W, tr.K, tr.chunk = H, W, O.intrinsics(H, W), 32768
    packed, *_ = O.prepare_rays(H, W, O.intrinsics(H, W), c2w=O.pose_spherical(30.0, -30.0, 4.0)[:3, :4])
    sel = torch.randperm(H * W, generator=torch.Generator().manual_seed(3))[:777]
    ro, rd = packed[sel, 0:3].contiguous().to(DEV), packed[sel, 3:6].contiguous().to(DEV)
    target = torch.rand(777, 3, generator=torch.Generator().manual_seed(4)).to(DEV)
    route = _route_of(lib, dn, 777)
    assert route == (ALL if width == 256 else COLLAPSED | SPLIT_BACKWARD | TENSOR_PATH), route_name(route)
    params = list(dn.parameters())
    opt = training.Adam(params, lr=1e-4)
    out = training.fused_render_and_backward(tr, opt, kw, (ro, rd), target)
    assert out is not None
    fused = [p.grad.detach().clone() for p in params]
    for p in params:
        p.grad = None
    rgb, _, ex = nerf_utils.render(H, W, tr.K, rays=(ro, rd), retraw=True, **kw)
    img_loss = torch.mean((rgb - target) ** 2)
    dn_loss = torch.nn.functional.mse_loss(ex["depth_net_z_vals"], ex["max_z_vals"])
    torch.autograd.backward([dn_loss, img_loss])
    assert abs(float(out[0]) - float(img_loss)) <= 1e-6 * max(1.0, float(img_loss))
    assert abs(float(out[1]) - float(dn_loss)) <= 1e-6 * max(1.0, float(dn_loss))
    worst = 0.0
    for p, g in zip(params, fused):
        rel = float((p.grad - g).abs().max()) / (float(g.abs().max()) + 1e-30)
        worst = max(worst, rel)
        assert float((p.grad - g).abs().max()) <= 1e-4 * float(g.abs().max()) + 1e-12
    print(f"fused step, DepthNetTrainer(n_layers=6, layer_width={width}) [{route_name(route)}]: worst gradient {worst:.2e}")
    for p in params:
        p.grad = None
