"""Forward + backward of the differentiable S-sample DepthNet render, split into its stages.

    python tools/bench_render_grad.py [--rays 4096] [--samples 1 8 32 64] [--iters 20]

The composition is the reference's: DepthNet(rays) -> sample_points_around_mean (uniform, +-0.1) -> Trainer.run_network (the "pts"
route: d raw / d pts, one primal and three tangent passes) or NeRF.query(z=...) (the "z" route: one primal and one tangent pass)
-> DepthNetTrainer.raw2outputs -> mse(rgb, target) + mse(depth, z_target) -> backward into DepthNet, with the seeded 10x256
DepthNet and NeRF of the oracle on the rays of a 64 x 64 view.  Every time is a mean over --iters repetitions between CUDA events
after two warm-up repetitions:
  * whole_ms: forward + backward of the composition;
  * depthnet_ms: DepthNet forward (DepthNetTrainFn) + its backward with a given upstream gradient;
  * jvp_ms: the NeRF query with its forward-mode derivative (NerfPointFn / NerfPtsFn forward) on the placed samples;
  * composite_fwd_ms / composite_bwd_ms: raw2outputs forward, and its backward alone (b200nerf_composite_bwd; at S = 1 the torch
    arithmetic of CompositeSingleFn).
One JSON line per (S, route) and a last line with the card's name and power limit, read in the same run."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = (s.strip() for s in q.stdout.strip().splitlines()[0].split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def timed(fn, iters):
    import torch

    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rays", type=int, default=4096)
    ap.add_argument("--samples", type=int, nargs="+", default=[1, 8, 32, 64])
    ap.add_argument("--iters", type=int, default=20)
    a = ap.parse_args()

    import torch
    import torch.nn.functional as F

    import nerf_sampling_b200 as pkg

    pkg.build()
    from nerf_sampling_b200.depth_nets import DepthNet
    from nerf_sampling_b200.nerf_pytorch import utils
    from nerf_sampling_b200.nerf_pytorch.run_nerf_helpers import NeRF, get_embedder
    from nerf_sampling_b200.nerf_pytorch.trainers.Trainer import Trainer
    from nerf_sampling_b200.trainers.sampling_trainer import DepthNetTrainer
    from oracle import nerf_oracle as O

    if not torch.cuda.is_available():
        sys.exit("no CUDA device: this benchmark measures the GPU and has nothing to report without one")
    dev = torch.device("cuda", 0)
    _, fine, dn = O.init_models(42)
    net = NeRF(D=8, W=256, input_ch=63, input_ch_views=27, output_ch=5, skips=[4], use_viewdirs=True)
    net.load_state_dict(fine)
    net.to(dev)
    dnet = DepthNet(hidden_sizes=[256] * 10, cat_hidden_sizes=[256] * 10, sphere_radius=2.0)
    dnet.load_state_dict(dn)
    dnet.to(dev)
    side = 1
    while side * side < a.rays:
        side *= 2
    packed, *_ = O.prepare_rays(side, side, O.intrinsics(side, side), c2w=O.pose_spherical(30.0, -30.0, 4.0)[:3, :4])
    ro, rd, vd = (packed[: a.rays, i:j].contiguous().to(dev) for i, j in ((0, 3), (3, 6), (8, 11)))
    n = ro.shape[0]
    g = torch.Generator().manual_seed(0)
    target = torch.rand(n, 3, generator=g).to(dev)
    z_target = (2.0 + 4.0 * torch.rand(n, generator=g)).to(dev)
    tr = DepthNetTrainer.__new__(DepthNetTrainer)
    embed_fn, _ = get_embedder(10, 0, 3)
    embeddirs_fn, _ = get_embedder(4, 0, 3)
    dz_up = torch.randn(n, 1, generator=g).to(dev)

    def depthnet():
        dnet.zero_grad(set_to_none=True)
        dnet(ro, rd).backward(dz_up)

    t_dn = timed(depthnet, a.iters)
    with torch.no_grad():
        mean = dnet(ro, rd)
    for S in a.samples:
        for route in ("z", "pts"):
            m = mean.clone().requires_grad_(True)

            def query(pts, z):
                if route == "pts":
                    return Trainer.run_network(tr, pts, vd, net, embed_fn, embeddirs_fn)
                return net.query(vd, rays_o=ro, rays_d=rd, z=z)

            def whole():
                dnet.zero_grad(set_to_none=True)
                pts, z = utils.sample_points_around_mean(ro, rd, dnet(ro, rd), n_samples=S, mode="uniform", std=0.1)
                rgb, _, _, depth, _, _, _ = tr.raw2outputs(query(pts, z), z, rd, 0, True)
                (F.mse_loss(rgb, target) + F.mse_loss(depth, z_target)).backward()

            pts, z = utils.sample_points_around_mean(ro, rd, m, n_samples=S, mode="uniform", std=0.1)
            t_jvp = timed(lambda: query(pts, z), a.iters)
            raw = query(pts, z).detach().requires_grad_(True)
            zz = z.detach().requires_grad_(True)
            t_cf = timed(lambda: tr.raw2outputs(raw, zz, rd, 0, True), a.iters)
            rgb, _, _, depth, _, _, _ = tr.raw2outputs(raw, zz, rd, 0, True)
            outs = [rgb, depth] if S > 1 else [rgb]   # S == 1: depth is the constant 0 of the empty-interval quirk
            ups = [torch.randn_like(o) for o in outs]
            t_cb = timed(lambda: torch.autograd.grad(outs, [raw, zz], ups, retain_graph=True, allow_unused=True), a.iters)
            t_whole = timed(whole, a.iters)
            print(json.dumps({"rays": n, "S": S, "route": route, "whole_ms": t_whole, "depthnet_ms": t_dn, "jvp_ms": t_jvp,
                              "composite_fwd_ms": t_cf, "composite_bwd_ms": t_cb}), flush=True)
    print(json.dumps(card()), flush=True)


if __name__ == "__main__":
    main()
