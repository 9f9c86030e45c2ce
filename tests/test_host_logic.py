"""CPU-only tests: C ABI surface, weight packing layout, DepthNet folding, reference known-answer tests."""

import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import nerf_oracle as O


# --------------------------------------------------------------------------------------------- ABI surface
def test_library_exports_every_declared_symbol(lib):
    header = open(os.path.join(ROOT, "include", "b200nerf.h")).read()
    names = set(re.findall(r"\b(b200nerf_[a-z0-9_]+)\s*\(", header))
    assert len(names) >= 18
    for n in names:
        assert hasattr(lib, n), f"libb200nerf.so does not export {n}"
    from nerf_sampling_b200 import _lib

    assert names == set(_lib.SIGNATURES), "ctypes signature table out of sync with include/b200nerf.h"
    assert lib.b200nerf_version() == 100


def test_no_cpu_fallback():
    from nerf_sampling_b200 import _lib, ops

    with pytest.raises(_lib.B200NerfError):
        ops.composite(torch.zeros(2, 4, 4), torch.zeros(2, 4), torch.zeros(2, 3))


# --------------------------------------------------------------------------------------------- packing
def bf16_split(w):
    hi = w.to(torch.bfloat16)
    lo = (w - hi.float()).to(torch.bfloat16)
    return hi, lo


def _piece(buf, n_rows):
    """[2 k chunks][n_rows/8 groups][8 rows][8 k] 16-bit piece -> [n_rows, 16]."""
    return buf.view(2, n_rows // 8, 8, 8).permute(1, 2, 0, 3).reshape(n_rows, 16)


def test_nerf_pack_layout_pipelined_exact(lib, oracle_models):
    """b200nerf_nerf_pack(PREC_SPLIT): [rank][layer][A first, B first, A second, B second][K16 block][hi piece | lo piece],
    one piece = the rank's 64 rows of a 128-row output half (csrc/mlp_exact.cuh)."""
    from nerf_sampling_b200.packing import NERF_KEYS

    _, fine, _ = oracle_models
    host = [fine[k].contiguous() for k in NERF_KEYS]
    arr = (C.c_void_p * 24)(*[t.data_ptr() for t in host])
    wpack = torch.zeros(lib.b200nerf_nerf_wpack_bytes(1), dtype=torch.uint8)
    aux = torch.zeros(lib.b200nerf_nerf_aux_floats(), dtype=torch.float32)
    assert lib.b200nerf_nerf_pack(C.cast(arr, C.c_void_p), 1, wpack.data_ptr(), aux.data_ptr()) == 0
    u = wpack.view(torch.bfloat16)
    w5, wv = fine["pts_linears.5.weight"], fine["views_linears.0.weight"]
    # (weight as [n_out, K] over the operand blocks, operand block -> column block) per layer
    def layer(n_out, first, second, cols):
        return dict(n_out=n_out, first=first, second=second, cols=cols)

    def pad(w, k):
        out = torch.zeros(w.shape[0], k)
        out[:, : w.shape[1]] = w
        return out

    enc, view = list(range(16, 20)), [20, 21]
    layers = [layer(256, enc, [], {16: pad(fine["pts_linears.0.weight"], 64)})]
    for i in (1, 2, 3, 4):
        layers.append(layer(256, list(range(8)), list(range(8, 16)), {0: fine[f"pts_linears.{i}.weight"]}))
    layers.append(layer(256, list(range(8)) + enc, list(range(8, 16)), {0: w5[:, 63:], 16: pad(w5[:, :63], 64)}))
    for name in ("pts_linears.6.weight", "pts_linears.7.weight"):
        layers.append(layer(256, list(range(8)), list(range(8, 16)), {0: fine[name]}))
    # feature_linear (no activation) is folded into the view layer: W' = Wv[:, :256] Wf, bias b' = Wv[:, :256] bf + bv
    wfold = (wv[:, :256].double() @ fine["feature_linear.weight"].double()).float()
    layers.append(layer(128, list(range(8)) + view, list(range(8, 16)), {0: wfold, 20: pad(wv[:, 256:], 32)}))
    per_rank = wpack.numel() // 2 // 2   # bf16 elements per rank
    for r in range(2):
        off = r * per_rank
        for L in layers:
            halves = L["n_out"] // 128
            for rng in (L["first"], L["second"]):
                for half in range(halves):
                    for kb in rng:
                        base = max(b for b in L["cols"] if b <= kb)
                        w = L["cols"][base][half * 128 + r * 64 : half * 128 + r * 64 + 64, (kb - base) * 16 : (kb - base) * 16 + 16]
                        rh, rl = bf16_split(w.contiguous())
                        if L is layers[-1] and base == 0:   # folded block: the fp64 sums may differ in the last bit before the split
                            got = _piece(u[off : off + 1024], 64).float() + _piece(u[off + 1024 : off + 2048], 64).float()
                            assert float((got - w).abs().max()) <= 2.0 ** -15 * float(w.abs().max()), (r, kb, half)
                        else:
                            assert torch.equal(_piece(u[off : off + 1024], 64), rh), (r, kb, half)
                            assert torch.equal(_piece(u[off + 1024 : off + 2048], 64), rl), (r, kb, half)
                        off += 2048
        assert off == (r + 1) * per_rank
    assert torch.equal(aux[2432:2688], fine["alpha_linear.weight"][0])
    want_b = (wv[:, :256].double() @ fine["feature_linear.bias"].double() + fine["views_linears.0.bias"].double()).float()
    assert float((aux[2304:2432] - want_b).abs().max()) <= 1e-6   # NERF_BV holds the folded bias


def test_nerf_pack_fast_layout(lib, oracle_models):
    """b200nerf_nerf_pack_fast: [step][rank][K16 block][piece], piece = the rank's half of the output rows, fp16."""
    from nerf_sampling_b200.packing import NERF_KEYS

    _, fine, _ = oracle_models
    host = [fine[k].contiguous() for k in NERF_KEYS]
    arr = (C.c_void_p * 24)(*[t.data_ptr() for t in host])
    wpack = torch.zeros(lib.b200nerf_nerf_fast_wpack_bytes(), dtype=torch.uint8)
    assert lib.b200nerf_nerf_pack_fast(C.cast(arr, C.c_void_p), 2, wpack.data_ptr()) == 0
    u = wpack.view(torch.float16)
    w5, wv = fine["pts_linears.5.weight"], fine["views_linears.0.weight"]

    def pad(w, k):
        out = torch.zeros(w.shape[0], k)
        out[:, : w.shape[1]] = w
        return out

    steps = [pad(fine["pts_linears.0.weight"], 64)] + [fine[f"pts_linears.{i}.weight"] for i in (1, 2, 3, 4)]
    # feature_linear (no activation) is folded into the view layer: W' = Wv[:, :256] Wf, b' = Wv[:, :256] bf + bv
    wfold = (wv[:, :256].double() @ fine["feature_linear.weight"].double()).float()
    steps += [torch.cat([w5[:, 63:], pad(w5[:, :63], 64)], 1), fine["pts_linears.6.weight"], fine["pts_linears.7.weight"],
              torch.cat([wfold, pad(wv[:, 256:], 32), torch.zeros(128, 32)], 1)]
    off = 0
    for si, w in enumerate(steps):
        half = w.shape[0] // 2
        for r in range(2):
            for kb in range(w.shape[1] // 16):
                want = w[r * half : (r + 1) * half, kb * 16 : kb * 16 + 16].to(torch.float16)
                got = _piece(u[off : off + half * 16], half)
                if si == len(steps) - 1 and kb < 16:   # folded block: fp64 sums may differ in the last bit before rounding
                    assert float((got.float() - want.float()).abs().max()) <= 2.0 ** -10 * float(want.float().abs().max())
                else:
                    assert torch.equal(got, want)
                off += half * 16
    bias = wpack[off * 2 : off * 2 + 512].view(torch.float32)
    want_b = (wv[:, :256].double() @ fine["feature_linear.bias"].double() + fine["views_linears.0.bias"].double()).float()
    assert float((bias - want_b).abs().max()) <= 1e-6
    assert off * 2 + 512 == wpack.numel()


def kernel_input_layout(rays_o, rays_d, radius=2.0):
    """[enc(o)|0|enc(d)|0|enc(hit_near)|0|enc(hit_far)|0] -- the DepthNet kernel's 256-wide input."""
    _, hits = O.sphere_intersections(rays_o, rays_d, torch.tensor([radius]))
    z = torch.zeros(rays_o.shape[0], 1)
    return torch.cat([O.embed(rays_o, 10), z, O.embed(rays_d, 10), z, O.embed(hits[:, 0], 10), z, O.embed(hits[:, 1], 10), z], -1)


@pytest.mark.parametrize("widths", [([256] * 10, [256] * 10), ([128] * 6, [128, 128, 128, 128, 256]), ([64] * 2, [96]),
                                    ([200, 136, 256], [256, 256]), ([512] * 2, [256] * 3)])
def test_fold_depthnet_matches_literal_network(widths):
    """Folding the activation-free branches into the first dense layer is exact up to fp32 round-off."""
    from nerf_sampling_b200.packing import fold_depthnet

    torch.manual_seed(3)
    dn = O.init_depthnet(*widths)
    H = W = 12
    c2w = O.pose_spherical(10.0, -40.0, 4.0)[:3, :4]
    ro, rd = O.get_rays(H, W, O.intrinsics(H, W), c2w)
    ro, rd = ro.reshape(-1, 3).contiguous(), rd.reshape(-1, 3).contiguous()
    rd[0] = torch.tensor([0.0, 1.0, 0.0])  # misses the sphere -> NaN depth in both
    want = O.depthnet_forward(dn, ro, rd).double()
    w0, b0, hidden, hw, hb = fold_depthnet(dn)
    x = kernel_input_layout(ro, rd).double()
    h = torch.nn.functional.leaky_relu(x @ w0.double().T + b0.double(), 0.01)
    for w, b in hidden:
        h = torch.nn.functional.leaky_relu(h @ w.double().T + b.double(), 0.01)
    s = torch.sigmoid(h @ hw.double() + hb.double())
    got = (2 * (1 - s) + 6 * s).reshape(-1, 1)
    assert torch.isnan(want[0]) and torch.isnan(got[0])
    assert float((want[1:] - got[1:]).abs().max()) < 2e-5
    assert len(hidden) == len(widths[1]) - 1


def test_depthnet_pack_roundtrip(lib):
    from nerf_sampling_b200.packing import PackedDepthNet

    torch.manual_seed(0)
    dn = O.init_depthnet([256] * 3, [256] * 3)
    pk = PackedDepthNet(dn, "cpu", prec=1)
    assert pk.n_hidden == 2
    # pipelined exact layout: 3 layers x 32 stages x 8 KB per rank, two ranks
    assert pk.wpack.numel() == 2 * 3 * 16 * 8192   # two ranks x 3 layers x 16 ring stages of 8 KB
    u = pk.wpack.view(torch.bfloat16)
    w0 = pk.folded[0]
    per_rank = u.numel() // 2
    for r in range(2):
        off = r * per_rank   # layer 0: A first (blocks 0..7), B first, A second (8..15), B second
        for rng in (range(0, 8), range(8, 16)):
            for half in range(2):
                for kb in rng:
                    w = w0[half * 128 + r * 64 : half * 128 + r * 64 + 64, kb * 16 : kb * 16 + 16].contiguous()
                    assert torch.equal(_piece(u[off : off + 1024], 64), bf16_split(w)[0])
                    assert torch.equal(_piece(u[off + 1024 : off + 2048], 64), bf16_split(w)[1])
                    off += 2048
    assert torch.equal(pk.aux[768:1024], pk.folded[3])  # head weights after 3 bias rows
    # only split precision exists: the predicted depth feeds the 2^9 octave of the NeRF encoding
    assert lib.b200nerf_depthnet_wpack_bytes(2, 0) == 0 and lib.b200nerf_nerf_wpack_bytes(0) == 0
    # the kernel stages a fixed 3080-float aux block whatever the depth: shallower nets must not get a shorter one (round 1 did,
    # and a 10-layer DepthNet read 1 KB past its block), and the tail is zero
    assert all(lib.b200nerf_depthnet_aux_floats(n) >= 3080 for n in range(0, 11))
    assert pk.aux.numel() >= 3080 and float(pk.aux[3 * 256 + 256 + 4:].abs().max()) == 0.0


# --------------------------------------------------------------------------------------------- module shells
def test_state_dict_keys_match_reference_layout(oracle_models):
    from nerf_sampling_b200.depth_nets import DepthNet
    from nerf_sampling_b200.nerf_pytorch.run_nerf_helpers import NeRF

    coarse, fine, dn = oracle_models
    torch.manual_seed(42)
    a = NeRF(D=8, W=256, input_ch=63, input_ch_views=27, output_ch=5, skips=[4], use_viewdirs=True)
    b = NeRF(D=8, W=256, input_ch=63, input_ch_views=27, output_ch=5, skips=[4], use_viewdirs=True)
    d = DepthNet(hidden_sizes=[256] * 10, cat_hidden_sizes=[256] * 10, sphere_radius=2.0)
    # same construction order => the seeded init reproduces the reference's weights bit for bit
    for mod, sd in ((a, coarse), (b, fine), (d, dn)):
        msd = mod.state_dict()
        assert set(msd) == set(sd)
        for k in sd:
            assert torch.equal(msd[k], sd[k]), k
    assert len(d.state_dict()) == 82 and sum(p.numel() for p in d.parameters()) == 3340545
    assert sum(p.numel() for p in a.parameters()) == 595844


def test_checkpoint_roundtrip(tmp_path):
    """save_state / load_nerf / load_depth_network keep the 200000.tar key layout (reference tests/tests.py:29-77)."""
    from nerf_sampling_b200.depth_nets import DepthNet
    from nerf_sampling_b200.nerf_pytorch import utils
    from nerf_sampling_b200.nerf_pytorch.run_nerf_helpers import NeRF

    mk = lambda: NeRF(D=8, W=256, input_ch=63, input_ch_views=27, skips=[4], use_viewdirs=True)  # noqa: E731
    fn, fine, dn = mk(), mk(), DepthNet([32, 32], [32, 32])
    opt = torch.optim.Adam(list(fn.parameters()) + list(fine.parameters()), lr=1e-3)
    sopt = torch.optim.Adam(dn.parameters(), lr=1e-4)
    path = str(tmp_path / "000123.tar")
    utils.save_state(123, fn, fine, opt, dn, sopt, path)
    ck = torch.load(path, weights_only=False)
    assert set(ck) == {"global_step", "network_fn_state_dict", "network_fine_state_dict", "optimizer_state_dict",
                       "sampling_optimizer_state_dict", "depth_network"}
    fn2, fine2, dn2 = mk(), mk(), DepthNet([32, 32], [32, 32])
    utils.load_nerf(fn2, fine2, torch.optim.Adam(list(fn2.parameters()) + list(fine2.parameters())), ck)
    utils.load_depth_network(dn2, torch.optim.Adam(dn2.parameters()), ck)
    for a, b in ((fn, fn2), (fine, fine2), (dn, dn2)):
        for (k, v), (_, v2) in zip(a.state_dict().items(), b.state_dict().items()):
            assert torch.equal(v, v2), k


def test_depthnet_layer_shapes():
    """reference tests/tests.py:114-194."""
    from nerf_sampling_b200.depth_nets import DepthNet

    hidden, cat = [32, 64, 16], [24, 48]
    d = DepthNet(hidden, cat)
    assert d.origin_layers[0].in_features == 2 * 63 and d.intersection_layers[0].in_features == 2 * 126
    for k in (1, 2):
        assert d.origin_layers[k].in_features == hidden[k - 1] + 63
        assert d.direction_layers[k].in_features == hidden[k - 1] + 63
        assert d.intersection_layers[k].in_features == hidden[k - 1] + 126
    assert d.cat_layers[0].in_features == 3 * hidden[-1] + 63 + 63 + 126
    assert len(d.cat_layers) == 2 * len(cat)
    assert isinstance(d.to_depth[0], torch.nn.Linear) and d.to_depth[0].out_features == 1
    assert isinstance(d.to_depth[1], torch.nn.Sigmoid)


def test_override_config_contract():
    from nerf_sampling_b200.nerf_pytorch.utils import override_config

    cfg = {"a": 1, "b": None}
    override_config(cfg, {"b": 2})
    assert cfg == {"a": 1, "b": 2}
    with pytest.raises(KeyError):
        override_config(cfg, {"c": 3})


def test_plugin_hook_builds_trainer(tmp_path):
    from nerf_sampling_b200.nerf_pytorch.utils import load_obj_from_config

    tr = load_obj_from_config({"module": "nerf_sampling_b200.trainers.DepthNetTrainer",
                               "kwargs": dict(dataset_type="blender", basedir=str(tmp_path), expname="e", no_batching=True,
                                              datadir="x", half_res=True, white_bkgd=True, n_layers=10, layer_width=256,
                                              N_importance=128, input_dims_embed=3)})
    assert tr.lindisp is True and tr.near == 2.0 and tr.far == 6.0 and tr.chunk == 32768 and tr.netchunk == 65536


def test_plugin_subclasses_reference_trainer_and_routes_its_entry_points(tmp_path):
    """nerf_sampling_b200.plugin.B200DepthNetTrainer derives from the REFERENCE's DepthNetTrainer (when baseline/_ref is
    installed), keeps its train()/log()/load_data(), overrides the hot-path operators, and while train() runs the reference's
    nerf_utils render entry points are this repo's (restored afterwards)."""
    import importlib

    from oracle import refpkg

    if not refpkg.import_reference():
        pytest.skip("baseline/_ref (the installed reference) is not present")
    import nerf_sampling.nerf_pytorch.nerf_utils as ref_nu
    from nerf_sampling.nerf_pytorch.trainers.Trainer import Trainer as RefTrainer
    from nerf_sampling.nerf_pytorch.utils import load_obj_from_config
    from nerf_sampling.trainers import DepthNetTrainer as RefDepthNetTrainer

    import nerf_sampling_b200.plugin as plugin
    from nerf_sampling_b200.nerf_pytorch import nerf_utils as nu

    if not plugin.HAVE_REFERENCE:
        plugin = importlib.reload(plugin)
    os.makedirs(tmp_path / "e", exist_ok=True)
    tr = load_obj_from_config({"module": "nerf_sampling_b200.plugin.B200DepthNetTrainer",
                               "kwargs": dict(dataset_type="blender", basedir=str(tmp_path), expname="e", no_batching=True,
                                              datadir="x", half_res=True, white_bkgd=True, n_layers=10, layer_width=256,
                                              N_importance=128, input_dims_embed=3, device="cuda")})
    cls = type(tr)
    assert issubclass(cls, RefDepthNetTrainer) and cls.log is RefTrainer.log and cls.update_learning_rate is RefTrainer.update_learning_rate
    for name in ("create_nerf_model", "render", "core_optimization_loop", "sample_random_ray_batch", "run_network", "raw2outputs",
                 "sample_coarse_points", "sample_fine_points", "_sample_points"):
        assert getattr(cls, name) is not getattr(RefDepthNetTrainer, name), name
    original = ref_nu.render_path
    seen = {}

    def fake_load_data():
        seen["render_path"] = ref_nu.render_path
        seen["render"] = ref_nu.render
        raise KeyboardInterrupt   # leave train() before anything needs a GPU

    tr.load_data = fake_load_data
    with pytest.raises(KeyboardInterrupt):
        tr.train(N_iters=2)
    assert seen["render_path"] is nu.render_path and seen["render"] is nu.render
    assert ref_nu.render_path is original


def test_mirror_trainer_has_the_drivers():
    """The stand-alone mirror offers train / render / log with the reference's signatures (Trainer.py:181, 263, 712)."""
    import inspect

    from nerf_sampling_b200.trainers import DepthNetTrainer

    assert list(inspect.signature(DepthNetTrainer.train).parameters) == ["self", "N_iters"]
    assert list(inspect.signature(DepthNetTrainer.render).parameters) == ["self", "render_test", "save_scene_data", "images", "i_test",
                                                                        "render_poses", "hwf", "render_kwargs_test"]
    assert "sampling_optimizer" in inspect.signature(DepthNetTrainer.log).parameters


# --------------------------------------------------------------------------------------------- reference KATs
def nan_equal(a, b):
    return torch.allclose(a[~torch.isnan(a)], b[~torch.isnan(b)], equal_nan=True) and torch.equal(torch.isnan(a), torch.isnan(b))


@pytest.mark.parametrize("impl", ["oracle", "product"])
def test_quadratic_known_answers(impl):
    """reference tests/tests.py:197-233."""
    if impl == "oracle":
        solve = O.solve_quadratic
    else:
        from nerf_sampling_b200.nerf_pytorch.utils import solve_quadratic_equation as solve
    T = torch.Tensor
    assert nan_equal(solve(T([1]), T([2]), T([1])), T([[-1], [-1]]))
    got = solve(T([1, 4, 5, 1, 4, 5]), T([1, 4, 6, 1, 4, 6]), T([1, 1, 1, 1, 1, 1]))
    nan = float("nan")
    assert nan_equal(got, T([[nan, -0.5, -1, nan, -0.5, -1], [nan, -0.5, -0.2, nan, -0.5, -0.2]]))


SPHERE_KATS = [  # (origin, direction, radius, expected hit points) -- reference tests/tests.py:236-331
    ([-3.0, 0, 0], [1.0, 0, 0], 1.0, [[-1.0, 0, 0], [1.0, 0, 0]]),
    ([-3.0, 0, 0], [0.0, 2.0, 0], 1.0, [[float("nan")] * 3] * 2),
    ([-3.0, 0, 0], [-1.0, 0, 0], 1.0, [[1.0, 0, 0], [-1.0, 0, 0]]),
    ([-3.0, 1.0, 0], [1.0, 0, 0], 1.0, [[0.0, 1.0, 0], [0.0, 1.0, 0]]),
    ([1.0, 0, 0], [0.0, 1.0, 0], 1.0, [[1.0, 0, 0], [1.0, 0, 0]]),
    ([0.0, 0, 0], [-1.0, 0, 0], 1.0, [[1.0, 0, 0], [-1.0, 0, 0]]),
    ([1.0, 0, 0], [-1.0, 0, 0], 1.0, [[1.0, 0, 0], [-1.0, 0, 0]]),
]


@pytest.mark.parametrize("impl", ["oracle", "product"])
@pytest.mark.parametrize("o,d,r,want", SPHERE_KATS)
def test_sphere_intersection_known_answers(impl, o, d, r, want):
    if impl == "oracle":
        fn = O.sphere_intersections
    else:
        from nerf_sampling_b200.nerf_pytorch.utils import find_intersection_points_with_sphere as fn
    t, pts = fn(torch.tensor([o]), torch.tensor([d]), torch.tensor([r]))
    assert pts.shape == (1, 2, 3) and t.shape == (1, 2)
    assert nan_equal(pts[0], torch.tensor(want))


def test_png_writer_roundtrip(tmp_path):
    """The stdlib PNG encoder of render_path: decode the IDAT stream by hand and compare pixels."""
    import struct
    import zlib

    import numpy as np

    from nerf_sampling_b200.nerf_pytorch.nerf_utils import _write_png

    rng = np.random.default_rng(0)
    img = rng.integers(0, 256, size=(13, 7, 3), dtype=np.uint8)
    path = str(tmp_path / "x.png")
    _write_png(path, img)
    data = open(path, "rb").read()
    assert data[:8] == b"\x89PNG\r\n\x1a\n"
    pos, idat, ihdr = 8, b"", None
    while pos < len(data):
        ln, tag = struct.unpack(">I", data[pos : pos + 4])[0], data[pos + 4 : pos + 8]
        body = data[pos + 8 : pos + 8 + ln]
        assert struct.unpack(">I", data[pos + 8 + ln : pos + 12 + ln])[0] == zlib.crc32(tag + body) & 0xFFFFFFFF
        if tag == b"IHDR":
            ihdr = struct.unpack(">IIBBBBB", body)
        if tag == b"IDAT":
            idat += body
        pos += 12 + ln
    assert ihdr == (7, 13, 8, 2, 0, 0, 0)
    rows = np.frombuffer(zlib.decompress(idat), np.uint8).reshape(13, 1 + 7 * 3)
    assert (rows[:, 0] == 0).all() and np.array_equal(rows[:, 1:].reshape(13, 7, 3), img)
