"""DepthNet inference and the graphed training step at several positional-encoding sizes, optionally against another checkout.

    python tools/bench_depthnet_multires.py [--multires 10 5] [--rounds 5] [--baseline-tree DIR]

Each measurement is one worker process (``--worker``) that imports the package of its tree and times, with CUDA events:
  * inference: ``DepthNet.forward`` under no_grad on 640,000 rays (the 800 x 800 view of bench.py) -- mlp_exact_kernel<IN_DEPTHNET>
    with the encoder of the image's multires;
  * training: one ``training.GraphedTrainStep`` replay of 4096 rays (config #5: 64 + 128 hierarchical target, DepthNet forward and
    both backward passes, Adam), 10x256 DepthNet.
``--baseline-tree`` names a checkout of another commit with its library built (multires 10 only, the only size it may serve).  The
workers run in alternating order, round by round, so both trees see the same drift of the shared machine; the spread over the rounds
is printed beside the medians.  One JSON line per worker and a summary line; the card name and power limit go into the summary."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def worker(multires: int, iters: int, steps: int) -> dict:
    import torch

    sys.path.insert(0, os.getcwd())
    import bench
    from nerf_sampling_b200 import ops, training
    from nerf_sampling_b200.depth_nets import DepthNet
    from nerf_sampling_b200.packing import PREC_FAST, PREC_SPLIT

    dev = torch.device("cuda", 0)
    coarse, fine, dn = bench.build_models(dev, PREC_FAST)
    if multires != 10:
        torch.manual_seed(43)
        dn = DepthNet(hidden_sizes=[256] * 10, cat_hidden_sizes=[256] * 10, multires=multires, sphere_radius=2.0).to(dev)
    dn.precision = PREC_SPLIT
    ro, rd, _ = ops.get_rays(bench.H, bench.W, bench.intrinsics(), bench.pose_for_step(0), dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.no_grad():
        for _ in range(3):
            z = dn(ro, rd)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(iters):
            z = dn(ro, rd)
        e1.record()
        torch.cuda.synchronize()
    infer_ms = e0.elapsed_time(e1) / iters
    z_sum = float(torch.nan_to_num(z, nan=0.0).double().sum())

    tr, kw = bench.make_trainer((coarse, fine, dn), dev)
    kw = dict(kw, model_mode="train")
    n = 4096
    sel = torch.randperm(ro.shape[0], generator=torch.Generator().manual_seed(0))[:n].to(dev)
    rays = (ro[sel].contiguous(), rd[sel].contiguous())
    target = torch.rand(n, 3, generator=torch.Generator().manual_seed(1)).to(dev)
    step = training.GraphedTrainStep(tr, training.Adam(list(dn.parameters()), lr=1e-4), kw, n)
    for _ in range(3):
        out = step(rays, target)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        out = step(rays, target)
    e1.record()
    torch.cuda.synchronize()
    return {"multires": multires, "infer_ms_640k": infer_ms, "train_step_ms_4096": e0.elapsed_time(e1) / steps,
            "z_checksum": z_sum, "loss": float(out[0])}


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = (s.strip() for s in q.stdout.strip().splitlines()[0].split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--multires", type=int, nargs="+", default=[10, 5])
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20, help="timed inference calls per worker")
    ap.add_argument("--steps", type=int, default=50, help="timed training steps per worker")
    ap.add_argument("--baseline-tree", default=None)
    ap.add_argument("--worker", action="store_true")
    a = ap.parse_args()
    if a.worker:
        print(json.dumps(worker(a.multires[0], a.iters, a.steps)), flush=True)
        return
    runs = [("this", ROOT, m) for m in a.multires]
    if a.baseline_tree:
        runs.insert(0, ("baseline", os.path.abspath(a.baseline_tree), 10))
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    res = {}
    for r in range(a.rounds):
        order = runs if r % 2 == 0 else runs[::-1]
        for tag, tree, m in order:
            cmd = [sys.executable, os.path.join(ROOT, "tools", "bench_depthnet_multires.py"), "--worker", "--multires", str(m),
                   "--iters", str(a.iters), "--steps", str(a.steps)]
            p = subprocess.run(cmd, cwd=tree, env=dict(env, PYTHONPATH=tree), capture_output=True, text=True)
            if p.returncode != 0:
                sys.exit(f"worker {tag} multires={m} failed:\n{p.stdout}\n{p.stderr}")
            line = json.loads(p.stdout.strip().splitlines()[-1])
            line.update(tree=tag, round=r)
            print(json.dumps(line), flush=True)
            res.setdefault((tag, m), []).append(line)
    summary = dict(card())
    for (tag, m), lines in res.items():
        for key in ("infer_ms_640k", "train_step_ms_4096"):
            v = [x[key] for x in lines]
            summary[f"{tag}_m{m}_{key}"] = {"median": statistics.median(v), "min": min(v), "max": max(v)}
        summary[f"{tag}_m{m}_z_checksum"] = sorted({x["z_checksum"] for x in lines})
    print(json.dumps(summary), flush=True)


if __name__ == "__main__":
    main()
