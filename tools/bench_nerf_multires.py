"""The NeRF MLP and the graphed training step at several positional-encoding sizes, optionally against another checkout.

    python tools/bench_nerf_multires.py [--sizes 10,4 5,2 1,1] [--rounds 5] [--baseline-tree DIR]

Each measurement is one worker process (``--worker``) that imports the package of its tree and times, with CUDA events:
  * query: ``b200nerf_nerf_query`` (ops.nerf_mlp) at PREC_FAST (fp16 single pass + split-precision guard band) and PREC_SPLIT on the
    800 x 800 x 64 view of bench.py (40,960,000 sample points, z uniform in [2, 6]) -- nerf_fast_kernel / mlp_exact_kernel<IN_NERF>
    with the encoders of the image's (multires, multires_views);
  * training: one ``training.GraphedTrainStep`` replay of 4096 rays (config #5: 64 + 128 hierarchical target through both NeRFs,
    10x256 DepthNet forward and both backward passes with the packed colour path, Adam), coarse and fine NeRF at that size.
``--baseline-tree`` names a checkout of another commit with its library built (10 / 4 only, the only size it may serve).  The workers
run in alternating order, round by round, so both trees see the same drift of the shared machine; the spread over the rounds is
printed beside the medians.  One JSON line per worker and a summary line; the card name and power limit go into the summary."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def worker(m: int, mv: int, iters: int, steps: int) -> dict:
    import torch

    sys.path.insert(0, os.getcwd())
    import bench
    from nerf_sampling_b200 import ops, training
    from nerf_sampling_b200.nerf_pytorch.run_nerf_helpers import NeRF
    from nerf_sampling_b200.packing import PREC_FAST, PREC_SPLIT, PackedNeRF

    dev = torch.device("cuda", 0)
    coarse, fine, dn = bench.build_models(dev, PREC_FAST)
    if (m, mv) != (10, 4):
        torch.manual_seed(42)
        mk = lambda: NeRF(D=8, W=256, input_ch=3 * (1 + 2 * m), input_ch_views=3 * (1 + 2 * mv), output_ch=5,  # noqa: E731
                          skips=[4], use_viewdirs=True).to(dev)
        coarse, fine = mk(), mk()
    ro, rd, vd = ops.get_rays(bench.H, bench.W, bench.intrinsics(), bench.pose_for_step(0), dev)
    z = 2.0 + 4.0 * torch.rand(ro.shape[0], 64, generator=torch.Generator().manual_seed(0)).to(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    res = {"multires": m, "multires_views": mv}
    for name, prec in (("fast", PREC_FAST), ("split", PREC_SPLIT)):
        pk = PackedNeRF(fine.state_dict(), dev, prec)
        with torch.no_grad():
            for _ in range(2):
                raw = ops.nerf_mlp(pk, vd, rays_o=ro, rays_d=rd, z=z)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(iters):
                raw = ops.nerf_mlp(pk, vd, rays_o=ro, rays_d=rd, z=z)
            e1.record()
            torch.cuda.synchronize()
        res[f"query_{name}_ms_41M"] = e0.elapsed_time(e1) / iters
        res[f"raw_{name}_checksum"] = float(torch.nan_to_num(raw, nan=0.0).double().sum())
        del raw, pk

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
    res.update(train_step_ms_4096=e0.elapsed_time(e1) / steps, loss=float(out[0]))
    return res


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = (s.strip() for s in q.stdout.strip().splitlines()[0].split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", nargs="+", default=["10,4", "5,2", "1,1"], help="multires,multires_views pairs")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=10, help="timed query calls per worker and precision")
    ap.add_argument("--steps", type=int, default=50, help="timed training steps per worker")
    ap.add_argument("--baseline-tree", default=None)
    ap.add_argument("--worker", action="store_true")
    a = ap.parse_args()
    sizes = [tuple(int(x) for x in s.split(",")) for s in a.sizes]
    if a.worker:
        print(json.dumps(worker(*sizes[0], a.iters, a.steps)), flush=True)
        return
    runs = [("this", ROOT, s) for s in sizes]
    if a.baseline_tree:
        runs.insert(0, ("baseline", os.path.abspath(a.baseline_tree), (10, 4)))
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    res = {}
    for r in range(a.rounds):
        order = runs if r % 2 == 0 else runs[::-1]
        for tag, tree, (m, mv) in order:
            cmd = [sys.executable, os.path.join(ROOT, "tools", "bench_nerf_multires.py"), "--worker", "--sizes", f"{m},{mv}",
                   "--iters", str(a.iters), "--steps", str(a.steps)]
            p = subprocess.run(cmd, cwd=tree, env=dict(env, PYTHONPATH=tree), capture_output=True, text=True)
            if p.returncode != 0:
                sys.exit(f"worker {tag} ({m}, {mv}) failed:\n{p.stdout}\n{p.stderr}")
            line = json.loads(p.stdout.strip().splitlines()[-1])
            line.update(tree=tag, round=r)
            print(json.dumps(line), flush=True)
            res.setdefault((tag, m, mv), []).append(line)
    summary = dict(card())
    for (tag, m, mv), lines in res.items():
        for key in ("query_fast_ms_41M", "query_split_ms_41M", "train_step_ms_4096"):
            v = [x[key] for x in lines]
            summary[f"{tag}_{m}_{mv}_{key}"] = {"median": statistics.median(v), "min": min(v), "max": max(v)}
        summary[f"{tag}_{m}_{mv}_raw_checksums"] = sorted({(x["raw_fast_checksum"], x["raw_split_checksum"]) for x in lines})
    print(json.dumps(summary), flush=True)


if __name__ == "__main__":
    main()
