#!/usr/bin/env python
"""Headline benchmark of the render_rays hot path: rays/sec for 800x800 DepthNet renders (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # ours (CUDA, sm_100a)
    python bench.py --impl reference --gpus N --steps K ...   # the reference itself (baseline/_ref) on the host CPU

One step = one 800x800 synthetic Blender-style view per GPU (640,000 rays): DepthNet -> 64 uniform samples around the
predicted depth -> positional encoding + 8x256 skip@4 NeRF MLP -> raw2outputs, random-init weights (seed 42), default
precision (fp16 single pass + split-precision guard band: meets the 1e-3 max-abs contract; --prec selects the others).
With N > 1 every rank renders its own view of an N-view batch (weak scaling, BASELINE config #3) and the rgb|disp image
tiles are all-gathered with NCCL on a side stream, double-buffered, inside the timed region.  Prints ONE JSON line:

  value        device-timed whole-job throughput, inputs resident in HBM (CUDA events, max over ranks)
  e2e          the same metric through host buffers: pinned host rays in, host images out (at N > 1 including the gather)
  e2e_api      ... through the reference-facing Python API ``nerf_utils.render_path`` (poses in, numpy images out)
  roofline     NeRF MLP against the measured bf16 tensor peak; roofline_composite against the measured HBM copy peak
  cpu_baseline the reference (kind "reference", from baseline/_ref) or the oracle port on the host cores, one 32,768-ray chunk
  gpu_eager_baseline  the oracle's plain-torch fp32 arithmetic on the same GPU (TF32 off), one 32,768-ray chunk, extrapolated
  shard_parity (N > 1) one view ray-sharded N ways == rank 0's unsharded render bit for bit; sharded training gradients
  strong       (N > 1) ONE 800x800 view split N ways (strong scaling), gather included
  extra        config4 (vanilla hierarchical 64 + 128, 800x800) and config5 (4096-ray DepthNet training step), at 1 and N GPUs

--dump-outputs DIR saves what the last timed step computed (rank 0's view) as float32 .npy files, so that two builds can be
compared output for output: the inputs depend only on the arguments.  Nothing is written into the source tree, which may be
read-only: a library older than its sources is recompiled into a temporary directory.
"""

from __future__ import annotations

import argparse
import atexit
import glob
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import torch

sys.dont_write_bytecode = True   # no __pycache__ in the tree
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H = W = 800
S = 64
DISTANCE = 0.1
NERF_FLOP_PER_POINT = 1_186_816          # SURVEY.md 8(d): 2 * 593,408 MAC, literal network
NERF_FLOP_EXECUTED = 1_056_768           # feature_linear folded into views_linears.0 at pack time (DESIGN.md 4.1)
DEPTHNET_FLOP_PER_RAY = 6_660_608        # literal network (the folded inference form executes 1,309,184)
COMPOSITE_BYTES_PER_RAY = 24 * S + 36    # SURVEY.md 8(d)
REF_CHUNK = 32768                        # one reference chunk (nerf_utils.py:88, BASELINE.md 3)
DUMP_RAYS = 16384                        # rays whose per-sample arrays --dump-outputs keeps (1.5 KB each; all 640,000 are 0.98 GB)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm=float(p["hbm_gbs"]), tf_sustained=float(p["bf16_tflops_sustained"]), tf_burst=float(p["bf16_tflops"]),
                    src="measured (MEASURED_PEAKS.json)")
    except Exception:
        return dict(hbm=6650.0, tf_sustained=1400.0, tf_burst=1590.0, src="fallback (B200_PROFILING.md)")


def ncu_traffic(prec: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the NeRF MLP kernel(s), from the NEWEST committed ncu
    --set full capture (profiles/*ncu_traffic.json, written by tools/ncu_summary.py next to the summary it came from).
    None when no capture of this precision mode is committed: the number is evidence, never a constant in this file."""
    best = None
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "*ncu_traffic.json"))):
        try:
            with open(path) as f:
                d = json.load(f)
            if prec in d:
                best = (float(d[prec]["bytes"]), os.path.basename(path))
        except Exception:
            continue
    return best


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def pose_spherical(theta: float, phi: float, radius: float) -> torch.Tensor:
    """Camera-to-world matrix of the Blender test orbit (the reference's load_blender.py:8-43): translate along z,
    rotate by phi about x, by theta about y, then the Blender axis flip."""
    import numpy as np

    ph, th = phi / 180.0 * np.pi, theta / 180.0 * np.pi
    t = np.array([[1, 0, 0, 0], [0, 1, 0, 0], [0, 0, 1, radius], [0, 0, 0, 1]], dtype=np.float32)
    rp = np.array([[1, 0, 0, 0], [0, np.cos(ph), -np.sin(ph), 0], [0, np.sin(ph), np.cos(ph), 0], [0, 0, 0, 1]], dtype=np.float32)
    rt = np.array([[np.cos(th), 0, -np.sin(th), 0], [0, 1, 0, 0], [np.sin(th), 0, np.cos(th), 0], [0, 0, 0, 1]], dtype=np.float32)
    flip = np.array([[-1, 0, 0, 0], [0, 0, 1, 0], [0, 1, 0, 0], [0, 0, 0, 1]], dtype=np.float32)
    return torch.from_numpy(flip @ (rt @ (rp @ t)))


def pose_for_step(i: int):
    """Pose i of the 200-view test orbit (theta = -180 + 1.8 i, phi = -30, r = 4.031), 3x4."""
    return pose_spherical(-180.0 + 1.8 * (i % 200), -30.0, 4.031)[:3, :4].contiguous()


def intrinsics():
    import numpy as np

    focal = 0.5 * W / np.tan(0.5 * 0.6911112070083618)
    return np.array([[focal, 0, 0.5 * W], [0, focal, 0.5 * H], [0, 0, 1]])


def workload_config(world: int):
    """The part of `config` that names the workload: identical on both arms (ours and --impl reference)."""
    return {"workload": f"800x800 lego-shaped view per GPU, DepthNet + {S} uniform samples/ray, 8x256 skip@4 NeRF "
                        "(BASELINE config #2; #3 for N>1: one view of the batch per rank, tiles all-gathered)",
            "rays_per_step_per_gpu": H * W, "samples_per_ray": S, "weights": "random-init seed 42"}


def build_models(device, prec):
    """Random-init weights, seed 42, in the reference's construction order (coarse NeRF, fine NeRF, DepthNet)."""
    from nerf_sampling_b200.depth_nets import DepthNet
    from nerf_sampling_b200.nerf_pytorch.run_nerf_helpers import NeRF

    torch.manual_seed(42)
    mk = lambda: NeRF(D=8, W=256, input_ch=63, input_ch_views=27, output_ch=5, skips=[4], use_viewdirs=True)  # noqa: E731
    coarse, fine, dn = mk(), mk(), None
    dn = DepthNet(hidden_sizes=[256] * 10, cat_hidden_sizes=[256] * 10, sphere_radius=2.0)
    for m in (coarse, fine, dn):
        m.precision = prec
        m.to(device)
    return coarse, fine, dn


def make_trainer(models, dev, **flags):
    """The mirror trainer + render kwargs around already-built models (what create_nerf_model returns)."""
    from nerf_sampling_b200.trainers import DepthNetTrainer

    coarse, fine, dn = models
    base = dict(dataset_type="blender", basedir="/tmp", expname="x", no_batching=True, datadir="x", half_res=False, white_bkgd=True,
                device=str(dev), n_layers=10, layer_width=256, N_importance=128, N_samples=64, input_dims_embed=3,
                distance=DISTANCE, sampling_mode="uniform", n_depth_samples=S, perturb=0.0)
    base.update(flags)
    tr = DepthNetTrainer(**base)
    tr.H, tr.W, tr.K, tr.chunk = H, W, intrinsics(), REF_CHUNK
    kw = dict(network_fn=coarse, network_fine=fine, depth_network=dn, network_query_fn=None, N_samples=64, N_importance=128,
              trainer=tr, white_bkgd=True, raw_noise_std=0.0, perturb=0.0, lindisp=True, ndc=False, near=2.0, far=6.0,
              use_viewdirs=True, model_mode="test")
    return tr, kw


# ------------------------------------------------------------------------------------------------- CPU arms
class CpuRenderer:
    """One 32,768-ray chunk of config #2 on the host CPU: the reference itself when baseline/_ref is installed
    (``nerf_utils.render_test`` of the unmodified package, random-init weights built the way experiments/run.py builds
    them), else the oracle port (pinned bit-exactly to the reference by tests/golden/make_golden.py)."""

    def __init__(self):
        import contextlib

        from oracle import refpkg

        torch.set_num_threads(os.cpu_count() or 1)
        self.K = intrinsics()
        self.kind = "port"
        if refpkg.import_reference():
            try:
                self.tmp = tempfile.mkdtemp(prefix="b200ref_")
                with contextlib.redirect_stdout(sys.stderr):   # the reference prints its configuration; stdout carries ONE JSON line
                    self.tr, _, self.rk_test = refpkg.build_reference_trainer(self.tmp, device="cpu", n_depth_samples=S,
                                                                              distance=DISTANCE, sampling_mode="uniform")
                from nerf_sampling.nerf_pytorch import nerf_utils, run_nerf_helpers

                self.ref_nu, self.ref_h = nerf_utils, run_nerf_helpers
                self.kind = "reference"
            except Exception as e:   # fall back to the port, say why
                print(f"[bench] reference import failed ({type(e).__name__}: {e}); timing the oracle port", file=sys.stderr)
        if self.kind == "port":
            from oracle import nerf_oracle as O

            self.O = O
            self.models = O.init_models(42)

    def rays(self, i: int, n: int):
        """n contiguous rays from the image centre of pose i."""
        base = (H // 2) * W
        if self.kind == "reference":
            ro, rd = self.ref_h.get_rays(H, W, self.K, pose_for_step(i))
            return ro.reshape(-1, 3)[base : base + n], rd.reshape(-1, 3)[base : base + n]
        packed, *_ = self.O.prepare_rays(H, W, self.K, c2w=pose_for_step(i))
        return packed[base : base + n]

    def render(self, rays):
        import contextlib

        with torch.no_grad(), contextlib.redirect_stdout(sys.stderr):
            if self.kind == "reference":
                return self.ref_nu.render_test(H, W, self.K, chunk=REF_CHUNK, rays=rays, **self.rk_test)[0]
            c, f, d = self.models
            return self.O.render_rays_test(rays, c, f, d, n_depth_samples=S, sampling_mode="uniform", distance=DISTANCE)["depth_net_rgb_map"]


def run_reference(args, rank, world):
    """`--impl reference`: the reference's own CPU implementation of the path on the box's host cores, rank 0 only."""
    if rank != 0:
        return
    cpu = CpuRenderer()
    n = args.ref_rays
    times = []
    for i in range(args.warmup + args.steps):
        rays = cpu.rays(i, n)
        t0 = time.perf_counter()
        cpu.render(rays)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            times.append(dt)
    total = sum(times)
    val = n * len(times) / total
    cores = torch.get_num_threads()
    line = {
        "impl": "reference", "metric": "rays_per_sec", "value": val, "unit": "rays/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(workload_config(args.gpus), precision="fp32 (the reference's own torch CPU path)",
                       sample_rays_per_step=n,
                       note="each step is a bounded sample of the workload: one 32,768-ray chunk of the view (the reference's own "
                            "chunk size, nerf_utils.py:88), contiguous rays from the image centre; rays/s does not depend on how "
                            "many chunks are rendered"),
        "cpu_baseline": {"value": val, "unit": "rays/s", "cores": cores, "kind": cpu.kind,
                         "sample": f"{n} rays x {S} samples per step, {len(times)} steps"},
        "e2e": {"value": val, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_sample():
    cpu = CpuRenderer()
    cpu.render(cpu.rays(0, 1024))   # warm-up (thread pool, allocator)
    rays = cpu.rays(1, REF_CHUNK)
    t0 = time.perf_counter()
    cpu.render(rays)
    dt = time.perf_counter() - t0
    return {"value": REF_CHUNK / dt, "unit": "rays/s", "cores": torch.get_num_threads(), "kind": cpu.kind,
            "sample": f"one {REF_CHUNK}-ray chunk of the 800x800 view x {S} samples after a 1024-ray warm-up ({dt:.1f} s)"}


def gpu_eager_baseline(dev):
    """The 'same box, same framework' comparator of BASELINE.md 3: the reference's arithmetic as eager fp32 torch ops on the
    B200 (cuBLAS SGEMM, TF32 off) for one 32,768-ray chunk of config #2, CUDA-event timed; rays/s extrapolates linearly."""
    from oracle import nerf_oracle as O

    tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        coarse, fine, dn = (O.params_to(p, dev) for p in O.init_models(42))
        packed, *_ = O.prepare_rays(H, W, intrinsics(), c2w=pose_for_step(0).to(dev))
        chunk = packed[(H // 2) * W : (H // 2) * W + REF_CHUNK]
        run = lambda: O.render_rays_test(chunk, coarse, fine, dn, n_depth_samples=S, sampling_mode="uniform", distance=DISTANCE)  # noqa: E731
        with torch.no_grad():
            run()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                run()
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 3
    finally:
        torch.backends.cuda.matmul.allow_tf32 = tf32
    return {"value": REF_CHUNK / ms * 1e3, "unit": "rays/s", "ms_per_chunk": ms, "kind": "oracle port, eager torch fp32 on cuda (TF32 off)",
            "sample": f"one {REF_CHUNK}-ray chunk x {S} samples, mean of 3 after a warm-up; a view is 19.5 such chunks (extrapolation)"}


# ------------------------------------------------------------------------------------------------- extra configs
def bench_config4(models, dev, world, rank, steps=4):
    """BASELINE config #4: vanilla hierarchical 64 + 128 (192 re-evaluated), 800x800, one view per rank, gather included."""
    import torch.distributed as dist

    from nerf_sampling_b200.nerf_pytorch import nerf_utils

    tr, kw = make_trainer(models, dev, use_full_nerf=True)
    K = intrinsics()
    tile = torch.empty(H * W, 4, device=dev)
    gathered = torch.empty(world * H * W, 4, device=dev) if world > 1 else None

    def one(i):
        rgb, disp, _ = nerf_utils.render_test(H, W, K, chunk=H * W, c2w=pose_for_step(i * world + rank), **kw)
        if world > 1:
            tile[:, :3] = rgb.reshape(-1, 3)
            tile[:, 3] = disp.reshape(-1)
            dist.all_gather_into_tensor(gathered, tile)

    with torch.no_grad():
        for i in range(2):
            one(i)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            one(2 + i)
        e1.record()
        torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1) / steps], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms)
    flop = 256 * NERF_FLOP_PER_POINT * H * W
    return {"metric": "rays_per_sec", "value": world * H * W / ms * 1e3, "ms_per_view": ms, "n_gpus": world, "steps": steps,
            "frac_of_tensor_peak": flop / ms / 1e9 / peaks()["tf_sustained"],
            "workload": "vanilla hierarchical: 64 coarse + 128 fine (all 192 re-evaluated), sample_pdf + merge, 800x800 per GPU, "
                        "through render_test(use_full_nerf) in one pass"}


def bench_config5(models, dev, world, rank, steps=20):
    """BASELINE config #5: DepthNet training step, 4096 rays per batch, data parallel; eager and as one CUDA graph."""
    import torch.distributed as dist

    from nerf_sampling_b200 import ops, training

    out = {}
    n_total = 4096
    per = n_total // world
    ro, rd, _ = ops.get_rays(H, W, intrinsics(), pose_for_step(0), dev)
    sel = torch.randperm(ro.shape[0], generator=torch.Generator().manual_seed(0))[:n_total][rank * per : (rank + 1) * per].to(dev)
    rays = (ro[sel].contiguous(), rd[sel].contiguous())
    target = torch.rand(n_total, 3, generator=torch.Generator().manual_seed(1))[rank * per : (rank + 1) * per].to(dev)
    saved = [p.detach().clone() for p in models[2].parameters()]
    for mode in ("eager", "graph"):
        tr, kw = make_trainer(models, dev)
        kw["model_mode"] = "train"
        opt = training.Adam(list(models[2].parameters()), lr=1e-4)
        if mode == "graph":
            graphed = training.GraphedTrainStep(tr, opt, kw, per)
            run = lambda i: graphed(rays, target)  # noqa: E731
        else:
            run = lambda i: tr.core_optimization_loop(opt, kw, rays, i, target)  # noqa: E731
        for i in range(3):
            res = run(i)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for i in range(steps):
            res = run(3 + i)
        e1.record()
        host_ms = (time.perf_counter() - t0) * 1e3 / steps
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) / steps], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        out[mode] = {"ms_per_step": float(ms), "rays_per_sec": n_total * 1e3 / float(ms), "host_enqueue_ms": host_ms,
                     "loss": float(res[0]), "depth_net_loss": float(res[1])}
        del res, run, opt
        with torch.no_grad():   # both modes start from the same weights
            for p, s0 in zip(models[2].parameters(), saved):
                p.copy_(s0)
    out.update({"n_gpus": world, "rays_per_step": n_total, "steps": steps,
                "workload": "core_optimization_loop: 64 + 192 hierarchical target on the frozen NeRFs, DepthNet fwd/bwd (cat layers and their "
                            "Jacobian chain as single launches of the split-precision tensor-core MLP kernel, the other products 3xTF32 on "
                            "tcgen05), colour gradient through the frozen fine NeRF (two launches of the same kernel), flat NCCL "
                            "all-reduce, fused Adam; 'graph' = the whole step (collective and Adam included) replayed as one CUDA graph"})
    return out


def shard_parity(models, dev, world, rank):
    """Outside every timed region: (1) ONE 800x800 view rendered ray-sharded `world` ways through render_path(shard="rays")
    must equal rank 0's unsharded render bit for bit; (2) one data-parallel training step's all-reduced, averaged DepthNet
    gradient must equal the single-process gradient over the same 4096 rays within fp32 reduction-order noise."""
    import torch.distributed as dist

    from nerf_sampling_b200 import ops, parallel
    from nerf_sampling_b200.nerf_pytorch import nerf_utils

    tr, kw = make_trainer(models, dev)
    K = intrinsics()
    poses = pose_for_step(7)[None]
    with torch.no_grad():
        rgbs_s, disps_s, _ = nerf_utils.render_path(poses, [H, W, float(K[0][0])], K, REF_CHUNK, kw, shard="rays")
        rgbs_1, disps_1, _ = nerf_utils.render_path(poses, [H, W, float(K[0][0])], K, REF_CHUNK, kw)
    import numpy as np

    render_equal = bool(np.array_equal(rgbs_s, rgbs_1) and np.array_equal(disps_s, disps_1))
    # training gradients: every rank computes the full-batch gradient locally, then its shard's, all-reduces, compares
    n_total = 4096
    per = n_total // world
    ro, rd, _ = ops.get_rays(H, W, K, pose_for_step(0), dev)
    sel = torch.randperm(ro.shape[0], generator=torch.Generator().manual_seed(0))[:n_total].to(dev)
    target = torch.rand(n_total, 3, generator=torch.Generator().manual_seed(1)).to(dev)
    kw["model_mode"] = "train"
    params = list(models[2].parameters())

    def grads(idx):
        for p in params:
            p.grad = None
        tr.render_and_backward(torch.optim.SGD(params, lr=0.0), kw, (ro[sel[idx]].contiguous(), rd[sel[idx]].contiguous()), 100, target[idx])
        return params

    full = torch.cat([p.grad.reshape(-1) for p in grads(slice(0, n_total))]).clone()
    grads(slice(rank * per, (rank + 1) * per))
    scale = parallel.allreduce_gradients(params)
    red = torch.cat([p.grad.reshape(-1) for p in params]) * scale
    rel = float((red - full).abs().max() / full.abs().max())
    for p in params:
        p.grad = None
    flags = torch.tensor([1.0 if render_equal else 0.0, rel], device=dev)
    worst = flags.clone()
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    dist.all_reduce(worst, op=dist.ReduceOp.MAX)
    res = {"render_equal": bool(flags[0] > 0.5), "train_grad_rel_err": float(worst[1]), "train_grad_tol": 1e-5}
    res["ok"] = res["render_equal"] and res["train_grad_rel_err"] <= res["train_grad_tol"]
    res["what"] = ("one 800x800 view ray-sharded N ways via render_path(shard='rays') vs unsharded (np.array_equal on every rank); "
                   "4096-ray training step: mean of the N shards' DepthNet gradients after the flat all-reduce vs the single-process "
                   "gradient (max-abs / max|g|; split-K atomics and the reduction order differ, the arithmetic does not)")
    return res


def dump_outputs(out_dir, tile, mean, z, raw, acc, depth, weights):
    """The arrays ops.render_depthnet(tile=True) would return for the last timed step, under its names, as float32 .npy: the
    per-ray maps of the whole view, and z / weights / raw for a fixed, seeded sample of DUMP_RAYS rays (43 MB in all)."""
    import numpy as np

    sel = torch.randperm(z.shape[0], generator=torch.Generator().manual_seed(0))[:DUMP_RAYS].sort().values.to(z.device)
    arrays = {"rgb": tile[:, :3], "disp": tile[:, 3], "acc": acc, "depth": depth, "z_mean": mean, "z": z[sel], "weights": weights[sel],
              "raw": raw[sel]}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy().astype(np.float32))


# ------------------------------------------------------------------------------------------------- our arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--prec", default="fast", choices=["fast", "fp16", "split"],
                    help="NeRF MLP precision: fast = fp16 single-pass + split-precision guard band (meets the 1e-3 contract), "
                         "fp16 = single-pass only, split = bf16 hi+lo everywhere")
    ap.add_argument("--ref-rays", type=int, default=REF_CHUNK, help="rays per step of the CPU reference arm (one reference chunk)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip config4 / config5 / strong / eager-GPU baseline")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import ctypes as C

    import torch.distributed as dist

    from nerf_sampling_b200 import _build, _lib, ops
    from nerf_sampling_b200.nerf_pytorch import nerf_utils
    from nerf_sampling_b200.packing import PREC_FAST, PREC_FP16, PREC_SPLIT

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    if _build.is_stale():
        tmp = tempfile.mkdtemp(prefix="b200nerf_")
        atexit.register(shutil.rmtree, tmp, True)
        _build.LIB_PATH = _build.build(out_path=os.path.join(tmp, "libb200nerf.so"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    prec = {"fast": PREC_FAST, "fp16": PREC_FP16, "split": PREC_SPLIT}[args.prec]
    L = _lib.lib()
    models = build_models(dev, prec)
    coarse, fine, dn = models
    dn.precision = PREC_SPLIT   # z feeds the 2^9 octave: DepthNet always runs split
    pk_dn, pk_nerf = dn.packed(), fine.packed()
    model = pk_nerf.c_model()
    K = intrinsics()
    n_rays = H * W
    total_steps = args.warmup + args.steps

    # inputs resident in HBM before the timed region: this rank's view of every step's batch
    rays = [ops.get_rays(H, W, K, pose_for_step(i * world + rank), dev) for i in range(total_steps)]
    grid = ops.uniform_grid(DISTANCE, S, dev)
    mean = torch.empty(n_rays, 1, device=dev)
    z = torch.empty(n_rays, S, device=dev)
    raw = torch.empty(n_rays, S, 4, device=dev)
    acc = torch.empty(n_rays, device=dev)
    depth = torch.empty(n_rays, device=dev)
    weights = torch.empty(n_rays, S, device=dev)
    guard = torch.zeros(n_rays + 4, dtype=torch.int32, device=dev)
    tiles = [torch.empty(n_rays, 4, device=dev) for _ in range(2)]              # rgb|disp pixels, written by the composite kernel
    gathered = [torch.empty(world * n_rays, 4, device=dev) for _ in range(2)] if world > 1 else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    main_stream = torch.cuda.current_stream()
    side = torch.cuda.Stream(device=dev)
    st = main_stream.cuda_stream
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    marks = []
    slot_free = [None, None]

    def step(i, timed):
        ro, rd, vd = rays[i]
        b = i & 1
        if slot_free[b] is not None:
            main_stream.wait_event(slot_free[b])   # the gather that read this tile two steps ago
        e = [ev() for _ in range(5)] if timed else None
        if timed:
            e[0].record()
        _lib.check(L.b200nerf_depthnet_fwd(pk_dn.wpack.data_ptr(), pk_dn.aux.data_ptr(), pk_dn.n_hidden, PREC_SPLIT, ro.data_ptr(), rd.data_ptr(),
                                           n_rays, 2.0, 2.0, 6.0, mean.data_ptr(), st))
        if timed:
            e[1].record()
        _lib.check(L.b200nerf_place_samples(mean.data_ptr(), grid.data_ptr(), n_rays, S, 1, 2.0, 6.0, z.data_ptr(), st))
        if timed:
            e[2].record()
        _lib.check(L.b200nerf_nerf_query(C.byref(model), ro.data_ptr(), rd.data_ptr(), vd.data_ptr(), z.data_ptr(), None, n_rays, S,
                                         guard.data_ptr(), raw.data_ptr(), st))
        if timed:
            e[3].record()
        _lib.check(L.b200nerf_composite_tile_fwd(raw.data_ptr(), z.data_ptr(), rd.data_ptr(), None, n_rays, S, 1, tiles[b].data_ptr(),
                                                 acc.data_ptr(), depth.data_ptr(), weights.data_ptr(), None, st))
        if timed:
            e[4].record()
            marks.append(e)
        if world > 1:  # image tiles to every rank over NVLink, on the side stream, under the next view's compute
            ready = torch.cuda.Event()
            ready.record(main_stream)
            with torch.cuda.stream(side):
                side.wait_event(ready)
                dist.all_gather_into_tensor(gathered[b], tiles[b])
                slot_free[b] = torch.cuda.Event()
                slot_free[b].record(side)
        flush.zero_()  # evict L2 between iterations (0.04 ms, inside the timed loop, stated in config)

    def drain():
        main_stream.wait_stream(side)

    for i in range(args.warmup):
        step(i, False)
    drain()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = _lib.launch_count()
    t_start, t_end = ev(), ev()
    t_start.record()
    for i in range(args.warmup, total_steps):
        step(i, True)
    drain()           # the last gather belongs to the timed region
    t_end.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    launches = _lib.launch_count() - l0
    ms = torch.tensor([t_start.elapsed_time(t_end)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms)
    value = world * n_rays * args.steps / (ms_total * 1e-3)
    if args.dump_outputs and rank == 0:   # before the e2e passes below reuse the buffers
        dump_outputs(args.dump_outputs, tiles[(total_steps - 1) & 1], mean, z, raw, acc, depth, weights)

    k_ms = [statistics.mean(m[j].elapsed_time(m[j + 1]) for m in marks) for j in range(4)]  # depthnet, place, mlp, composite
    pk = peaks()
    mlp_tflops = NERF_FLOP_PER_POINT * n_rays * S / (k_ms[2] * 1e-3) / 1e12
    comp_gbs = COMPOSITE_BYTES_PER_RAY * n_rays / (k_ms[3] * 1e-3) / 1e9
    guard_points = int(guard[0]) if prec == PREC_FAST else None

    # ---- end to end through host buffers: a DIFFERENT view's rays every iteration (pinned), images back on the host --------------
    n_e2e = max(3, min(args.steps, 10))
    n_sets = min(4, n_e2e)
    h_rays = []
    for j in range(n_sets):
        ro, rd, _ = rays[j % len(rays)]
        h_rays.append((ro.cpu().pin_memory(), rd.cpu().pin_memory()))
    if world == 1:
        h_rgb = torch.empty(n_rays, 3).pin_memory()
        h_disp = torch.empty(n_rays).pin_memory()
        ws = torch.empty(L.b200nerf_render_host_ws_bytes(n_rays, S), dtype=torch.uint8, device=dev)

        def e2e_step(j):
            hro, hrd = h_rays[j % n_sets]
            _lib.check(L.b200nerf_render_depthnet_host(pk_dn.wpack.data_ptr(), pk_dn.aux.data_ptr(), pk_dn.n_hidden, PREC_SPLIT, C.byref(model),
                                                       hro.data_ptr(), hrd.data_ptr(), n_rays, S, 1, grid.data_ptr(), 2.0, 2.0, 6.0,
                                                       ws.data_ptr(), h_rgb.data_ptr(), h_disp.data_ptr(), st))
            flush.zero_()

        e2e_api_name = "b200nerf_render_depthnet_host (pinned host rays -> host rgb + disp)"
        d2h = n_rays * 16
    else:
        d_ro, d_rd, d_vd = (torch.empty(n_rays, 3, device=dev) for _ in range(3))
        h_out = torch.empty(world * n_rays, 4).pin_memory()

        def e2e_step(j):
            hro, hrd = h_rays[j % n_sets]
            d_ro.copy_(hro, non_blocking=True)
            d_rd.copy_(hrd, non_blocking=True)
            _lib.check(L.b200nerf_normalize_dirs(d_rd.data_ptr(), n_rays, d_vd.data_ptr(), st))
            _lib.check(L.b200nerf_render_depthnet_tile(pk_dn.wpack.data_ptr(), pk_dn.aux.data_ptr(), pk_dn.n_hidden, PREC_SPLIT, C.byref(model),
                                                       d_ro.data_ptr(), d_rd.data_ptr(), d_vd.data_ptr(), n_rays, S, 1, grid.data_ptr(),
                                                       2.0, 2.0, 6.0, mean.data_ptr(), z.data_ptr(), raw.data_ptr(), guard.data_ptr(),
                                                       tiles[0].data_ptr(), acc.data_ptr(), depth.data_ptr(), None, st))
            dist.all_gather_into_tensor(gathered[0], tiles[0])
            if rank == 0:
                h_out.copy_(gathered[0], non_blocking=True)       # the driver rank receives all N images ...
            else:
                h_out[:n_rays].copy_(tiles[0], non_blocking=True)  # ... every other rank its own
            flush.zero_()
            main_stream.synchronize()   # the gathered host images are valid on return, like the single-GPU host call

        e2e_api_name = ("pinned host rays -> H2D -> b200nerf_render_depthnet_tile -> NCCL all_gather of the rgb|disp tiles -> D2H of "
                        "all N images on rank 0 (own image on the other ranks)")
        d2h = world * n_rays * 16

    e2e_step(0)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for j in range(n_e2e):
        e2e_step(1 + j)
    torch.cuda.synchronize()
    e2e_s = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_val = world * n_rays * n_e2e / float(e2e_s)

    # ---- end to end through the reference-facing Python API: poses in, numpy images out -----------------------------------------
    tr, kw = make_trainer(models, dev)
    n_api = 10 * world
    api_poses = torch.stack([pose_for_step(40 + i) for i in range(n_api)])
    hwf = [H, W, float(K[0][0])]
    shard = "views" if world > 1 else None
    with torch.no_grad():
        nerf_utils.render_path(api_poses[: 2 * world], hwf, K, REF_CHUNK, kw, shard=shard, dst=0)   # warms the pinned ring and NCCL
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        api_rgbs, _, _ = nerf_utils.render_path(api_poses, hwf, K, REF_CHUNK, kw, shard=shard, dst=0)
        api_s = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(api_s, op=dist.ReduceOp.MAX)
    e2e_api = {"value": n_api * n_rays / float(api_s), "unit": "rays/s", "ms_per_view": 1e3 * float(api_s) / n_api * world, "views": n_api,
               "api": "nerf_utils.render_path(poses, chunk=32768" + (", shard='views', dst=0)" if world > 1 else ")") + " -> numpy rgbs/disps",
               "h2d_bytes_per_step": 48, "d2h_bytes_per_step": (world if world > 1 else 1) * n_rays * 16,
               "note": "rays are generated from the 3x4 pose on the device (get_rays is row a1 of the path); the image stack is "
                       "returned on rank 0"}

    extra, strong, parity, eager = {}, None, None, None
    if not args.no_extra:
        if world > 1:
            parity = shard_parity(models, dev, world, rank)
            # strong scaling: ONE view split N ways, gather included (render_path(shard='rays') schedule, device-timed)
            with torch.no_grad():
                sp = torch.stack([pose_for_step(80 + i) for i in range(8)])
                nerf_utils.render_path(sp[:2], hwf, K, REF_CHUNK, kw, shard="rays", dst=0)
                torch.cuda.synchronize()
                dist.barrier()
                t0 = time.perf_counter()
                nerf_utils.render_path(sp, hwf, K, REF_CHUNK, kw, shard="rays", dst=0)
                s_s = torch.tensor([time.perf_counter() - t0], device=dev)
            dist.all_reduce(s_s, op=dist.ReduceOp.MAX)
            strong = {"value": 8 * n_rays / float(s_s), "unit": "rays/s", "ms_per_view": 1e3 * float(s_s) / 8, "rays_per_gpu_per_view": n_rays // world,
                      "scaling": "strong", "api": "nerf_utils.render_path(shard='rays', dst=0) -> numpy on rank 0, 8 views, wall clock",
                      "limiter": "per view each rank runs the same four launches on 1/N of the rays: the fixed per-launch cost (persistent-"
                                 "kernel prologue/tail, 74 CTA pairs x 4 tiles of 128 points = 592 rays per wave of the MLP kernel, DepthNet's "
                                 "one-tile-ahead staging) and the D2H + host unload of the full image on rank 0 do not shrink with N"}
        extra["config4"] = bench_config4(models, dev, world, rank)
        extra["config5"] = bench_config5(models, dev, world, rank)
        if rank == 0 and world == 1:
            eager = gpu_eager_baseline(dev)

    if rank == 0:
        cpu = None if args.no_cpu_baseline or world > 1 else cpu_baseline_sample()
        traffic = ncu_traffic(args.prec)
        line = {
            "metric": "rays_per_sec", "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {PREC_FAST: "fp16 operands, fp32 accumulate (+ bf16 hi/lo split re-evaluation of the guard band)",
                      PREC_FP16: "fp16", PREC_SPLIT: "bf16x2-split (bf16 hi+lo operands, fp32 accumulate)"}[prec],
            "data": "synthetic",
            "config": dict(workload_config(world), precision=args.prec,
                           l2="256 MiB flush between iterations + per-step working set 840 MB > 126 MB L2",
                           parallelism=(f"one view per rank x{world}; rgb|disp tiles written by the composite kernel, all_gather on a "
                                        "side stream under the next view (double-buffered)") if world > 1 else "single GPU"),
            "e2e": {"value": e2e_val, "unit": "rays/s", "h2d_bytes_per_step": 2 * n_rays * 12, "d2h_bytes_per_step": d2h,
                    "api": e2e_api_name, "steps": n_e2e, "views_rotated": n_sets},
            "e2e_api": e2e_api,
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "tensor",
                         "kernel": ("fast::nerf_fast_kernel<fp16> (+ exact::mlp_exact_kernel over the guard band) via b200nerf_nerf_query"
                                    if prec in (PREC_FAST, PREC_FP16) else "exact::mlp_exact_kernel<NERF> via b200nerf_nerf_query"),
                         "achieved": mlp_tflops, "peak": pk["tf_sustained"], "unit": "TFLOP/s", "frac": mlp_tflops / pk["tf_sustained"],
                         "frac_executed": mlp_tflops * NERF_FLOP_EXECUTED / NERF_FLOP_PER_POINT / pk["tf_sustained"],
                         "traffic": traffic[0] if traffic else None, "traffic_source": traffic[1] if traffic else None,
                         "peak_source": pk["src"] + ", sustained bf16", "ms_per_launch": k_ms[2],
                         "algorithmic_flop_per_point": NERF_FLOP_PER_POINT,
                         "executed_mma_tflops": mlp_tflops * (3 if prec == PREC_SPLIT else 1) * NERF_FLOP_EXECUTED / NERF_FLOP_PER_POINT,
                         "guard_band_points_last_step": guard_points,
                         "note": "achieved counts the reference network's 1,186,816 FLOP/point; the kernels fold the activation-free "
                                 "feature_linear into views_linears.0 when packing (1,056,768 FLOP/point executed), so frac can exceed 1 -- "
                                 "frac_executed = executed_mma_tflops / peak is the tensor-pipe load"},
            "roofline_composite": {"bound": "hbm", "kernel": "comp::composite_tma_kernel<16> (TMA-staged, persistent)", "achieved": comp_gbs,
                                   "peak": pk["hbm"], "unit": "GB/s", "frac": comp_gbs / pk["hbm"], "ms_per_launch": k_ms[3],
                                   "bytes_per_ray": COMPOSITE_BYTES_PER_RAY},
            "kernel_ms": {"depthnet": k_ms[0], "place": k_ms[1], "nerf_mlp": k_ms[2], "composite": k_ms[3]},
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if eager is not None:
            line["gpu_eager_baseline"] = eager
        if parity is not None:
            line["shard_parity"] = parity
        if strong is not None:
            line["strong"] = strong
        if extra:
            line["extra"] = extra
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
