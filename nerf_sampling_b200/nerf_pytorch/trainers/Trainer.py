"""Mirror of ``nerf_pytorch/trainers/Trainer.py`` restricted to what the render_rays path reads:
the constructor's config bag (:18-130), intrinsics (:136-146), ``core_optimization_loop`` (:506-544),
``run_network`` (:789-806) and the coarse / fine samplers (:553-710).  Data loading and logging are caller context."""

from __future__ import annotations

import os
from typing import Optional

import numpy as np
import torch

from ... import ops
from .. import nerf_utils


class Trainer:
    def __init__(self, dataset_type, basedir, expname, no_batching, datadir, device="cpu", render_test=False,
                 config_path=None, N_rand=32 * 32 * 4, render_only=False, chunk=1024 * 32, render_factor=0, multires=10,
                 i_embed=0, multires_views=4, netchunk=1024 * 64, lrate=5e-4, lrate_decay=250, use_viewdirs=True,
                 N_importance=0, netdepth=8, netwidth=256, netdepth_fine=8, netwidth_fine=256, ft_path=None, perturb=1.0,
                 raw_noise_std=0.0, N_samples=64, lindisp=True, precrop_iters=0, precrop_frac=0.5, i_weights=10000,
                 i_testset=100, i_video=5000, i_print=100, input_dims_embed: int = 1, save_train_set_render: bool = True,
                 depth_net_lr: float = 0.0001, train_depth_net_only: bool = False, trial=None, single_image=False,
                 single_ray=False, save_scene_data=False, compare_nerf=False, use_nerf_max_pts=False, use_full_nerf=False):
        loc = dict(locals())
        loc.pop("self")
        for k, v in loc.items():
            setattr(self, k, v)
        self.start = None
        self.use_batching = not self.no_batching
        self.no_reload = False
        self.K = self.global_step = self.W = self.H = self.c2w = None

    def load_data(self):
        """-> (hwf, poses, i_test, i_val, i_train, images, render_poses).  Dataset readers are the host application's
        (SURVEY.md §2: out of scope): ``nerf_sampling_b200.plugin.B200DepthNetTrainer`` inherits the reference's Blender
        loader; a standalone user overrides this method."""
        raise NotImplementedError("dataset loading is outside the B200 hot path: use nerf_sampling_b200.plugin."
                                  "B200DepthNetTrainer (inherits the reference's loaders) or override load_data()")

    def create_log_dir_and_copy_the_config_file(self):
        """args.txt / config.txt next to the checkpoints (Trainer.py:148-160)."""
        d = os.path.join(self.basedir, self.expname)
        os.makedirs(d, exist_ok=True)
        with open(os.path.join(d, "args.txt"), "w") as f:
            for k, v in self.__dict__.items():
                if not k.startswith("_b200"):
                    f.write("{} = {}\n".format(k, v))
        if self.config_path is not None:
            with open(os.path.join(d, "config.txt"), "w") as f, open(self.config_path) as src:
                f.write(src.read())

    # ------------------------------------------------------------------ drivers (Trainer.py:181-230, 263-398, 712-787)
    def render(self, render_test, save_scene_data, images, i_test, render_poses, hwf, render_kwargs_test):
        """Render ``render_poses`` to ``<basedir>/<expname>/renderonly_*`` and return the mean PSNR against the test images
        (Trainer.py:181-230); PNG frames always, ``video.mp4`` when an encoder is installed."""
        with torch.no_grad():
            gt = images[i_test] if render_test else None
            savedir = os.path.join(self.basedir, self.expname,
                                   "renderonly_{}_{:06d}".format("test" if render_test else "path", self.global_step))
            os.makedirs(savedir, exist_ok=True)
            rgbs, _, avg_test_psnr = nerf_utils.render_path(render_poses, hwf, self.K, self.chunk, render_kwargs_test,
                                                            step=self.global_step, save_scene_data=save_scene_data, gt_imgs=gt,
                                                            savedir=savedir, render_factor=self.render_factor)
            nerf_utils.write_video(os.path.join(savedir, "video.mp4"), rgbs)
        return avg_test_psnr

    def log(self, i, render_poses, hwf, poses, i_test, i_train, images, loss, depth_net_loss, psnr, render_kwargs_train,
            render_kwargs_test, optimizer, sampling_optimizer):
        """Periodic test-set render, checkpoint and progress line (the wandb / optuna reporting of Trainer.py:263-398 belongs
        to the host application and is not mirrored)."""
        if i % self.i_testset == 0 and i > 0:
            savedir = os.path.join(self.basedir, self.expname, "testset_{:06d}".format(i))
            with torch.no_grad():
                nerf_utils.render_path(self._host_poses(poses)[i_test], hwf, self.K, self.chunk, render_kwargs_test,
                                       step=self.global_step, save_scene_data=self.save_scene_data, gt_imgs=images[i_test],
                                       savedir=savedir)
        if i % self.i_weights == 0:
            from .. import utils

            utils.save_state(global_step=self.global_step, network_fn=render_kwargs_train["network_fn"],
                             network_fine=render_kwargs_train["network_fine"], optimizer=optimizer,
                             depth_network=render_kwargs_train["depth_network"], sampling_optimizer=sampling_optimizer,
                             path=os.path.join(self.basedir, self.expname, "{:06d}.tar".format(i)))
        if i % self.i_print == 0:
            info = f"Iter: {i} Loss: {loss.item()}, Depth Net Loss: {depth_net_loss.item()}, PSNR: {psnr.item():.5f}"
            print(info)
            with open(os.path.join(self.basedir, self.expname, "psnr.txt"), "a") as f:
                f.write(info + "\n")

    def train(self, N_iters=200000 + 1):
        """load_data -> models -> (render only | optimisation loop), the control flow of Trainer.py:712-787."""
        from .. import utils

        hwf, poses, i_test, i_val, i_train, images, render_poses = self.load_data()
        if self.render_test:
            render_poses = torch.as_tensor(np.array(self._host_poses(poses)[i_test]))
        hwf = self.cast_intrinsics_to_right_types(hwf=hwf)
        self.create_log_dir_and_copy_the_config_file()
        optimizer, sampling_optimizer, render_kwargs_train, render_kwargs_test = self.create_nerf_model()
        if self.train_depth_net_only:
            for key in ("network_fn", "network_fine"):
                if render_kwargs_train[key] is not None:
                    utils.freeze_model(render_kwargs_train[key])
        if self.render_only:
            return self.render(self.render_test, self.save_scene_data, images, i_test, render_poses, hwf, render_kwargs_test)
        if self.use_batching:
            raise NotImplementedError("pre-shuffled ray batching (no_batching=False) needs the host application's "
                                      "prepare_raybatch_tensor_if_batching_random_rays; the lego configuration uses no_batching")
        psnr = None
        for i in range(self.start + 1, N_iters):
            _, _, batch_rays, target_s = self.sample_random_ray_batch(None, None, i_train, images, poses, i)
            loss, depth_net_loss, psnr, _ = self.core_optimization_loop(sampling_optimizer, render_kwargs_train, batch_rays, i, target_s)
            self.update_learning_rate(optimizer)
            self.log(i=i, render_poses=render_poses, hwf=hwf, poses=poses, i_test=i_test, i_train=i_train, images=images,
                     loss=loss, depth_net_loss=depth_net_loss, psnr=psnr, render_kwargs_train=render_kwargs_train,
                     render_kwargs_test=render_kwargs_test, optimizer=optimizer, sampling_optimizer=sampling_optimizer)
            self.global_step += 1
        return psnr

    def cast_intrinsics_to_right_types(self, hwf):
        H, W, focal = hwf
        H, W = int(H), int(W)
        if self.K is None:
            self.K = np.array([[focal, 0, 0.5 * W], [0, focal, 0.5 * H], [0, 0, 1]])
        self.H, self.W = H, W
        return [H, W, focal]

    # ------------------------------------------------------------------ training batches
    def sample_random_ray_batch(self, rays_rgb, i_batch, i_train, images, poses, i):
        """(rays_rgb, i_batch, batch_rays [2,N_rand,3], target_s [N_rand,3]) -- Trainer.py:400-475.

        no_batching (the reference's lego configuration): pick a training image, pick N_rand pixels (centre crop while
        ``i < precrop_iters``), and generate ONLY those rays on the device; the reference builds all H*W rays with
        ``get_rays`` and draws the pixels with ``np.random.choice`` on the host (set ``self.reference_rng = True`` to draw
        them the same way and consume the same NumPy random stream).  ``images`` may be a device tensor [n,H,W,3+]."""
        if self.use_batching:
            batch = torch.transpose(rays_rgb[i_batch : i_batch + self.N_rand], 0, 1)
            batch_rays, target_s = batch[:2], batch[2]
            i_batch += self.N_rand
            if i_batch >= rays_rgb.shape[0]:
                rays_rgb = rays_rgb[torch.randperm(rays_rgb.shape[0], device=rays_rgb.device)]
                i_batch = 0
            return rays_rgb, i_batch, batch_rays, target_s
        img_i = 42 if self.single_image else int(np.random.choice(i_train))
        dev = torch.device(self.device if str(self.device) != "cpu" else "cuda")
        target = self._device_image(images, img_i, dev)
        self.c2w = self._host_poses(poses)[img_i, :3, :4].clone()
        if i < self.precrop_iters:
            dH, dW = int(self.H // 2 * self.precrop_frac), int(self.W // 2 * self.precrop_frac)
            h0, w0, hh, ww = self.H // 2 - dH, self.W // 2 - dW, 2 * dH, 2 * dW
        else:
            h0, w0, hh, ww = 0, 0, self.H, self.W
        n_pix = hh * ww
        if self.single_ray:
            sel = torch.tensor([91], device=dev)
        elif getattr(self, "reference_rng", False):
            sel = torch.from_numpy(np.random.choice(n_pix, size=[self.N_rand], replace=False)).to(dev)
        else:
            sel = torch.randperm(n_pix, device=dev)[: self.N_rand]
        pix = (h0 + sel // ww) * self.W + (w0 + sel % ww)   # flat index into the full image
        rays_o, rays_d, _ = ops.get_rays_at(self.H, self.W, self.K, self.c2w, pix)
        target_s = ops.gather_pixels(target[..., :3].contiguous(), pix)
        return rays_rgb, i_batch, torch.stack([rays_o, rays_d], 0), target_s

    def _device_image(self, images, img_i: int, dev) -> torch.Tensor:
        """Training image ``img_i`` as a device tensor, uploaded once (the reference re-wraps the host array every step,
        Trainer.py:421-422: 7.7 MB of pageable H2D per step at 800x800)."""
        cache = self.__dict__.get("_b200_images")
        if cache is None or cache["owner"] is not images:
            cache = self.__dict__["_b200_images"] = {"owner": images, "dev": {}}
        t = cache["dev"].get(img_i)
        if t is None:
            t = cache["dev"][img_i] = torch.as_tensor(images[img_i], dtype=torch.float32).to(dev).contiguous()
        return t

    def _host_poses(self, poses) -> torch.Tensor:
        """Camera poses on the host (the kernels take the 3x4 matrix by value): one D2H for the whole run, not one per step."""
        cache = self.__dict__.get("_b200_poses")
        if cache is None or cache[0] is not poses:
            cache = self.__dict__["_b200_poses"] = (poses, torch.as_tensor(poses).detach().to("cpu", torch.float32))
        return cache[1]

    # ------------------------------------------------------------------ one optimisation step (config #5)
    def core_optimization_loop(self, sampling_optimizer, render_kwargs_train, batch_rays, i, target_s):
        """Render a ray batch and back-propagate into DepthNet (Trainer.py:506-544): ``mse(z_dn, max_z)`` with
        ``retain_graph`` first, then the colour loss; under ``torch.distributed`` the DepthNet gradients are
        sum-all-reduced as one flat buffer and averaged by the optimizer (equal ray shards per rank reproduce the
        single-process gradient)."""
        loss, depth_net_loss, psnr, psnr0 = self.render_and_backward(sampling_optimizer, render_kwargs_train, batch_rays, i, target_s)
        self.reduce_and_step(sampling_optimizer)
        return loss, depth_net_loss, psnr, psnr0

    def render_and_backward(self, sampling_optimizer, render_kwargs_train, batch_rays, i, target_s):
        """First half of core_optimization_loop: render, zero_grad, both backward passes (Trainer.py:515-538).  Pure device
        work on the current stream -- this is the part ``training.GraphedTrainStep`` captures in a CUDA graph."""
        import torch.nn.functional as F

        from ... import training

        fused = training.fused_render_and_backward(self, sampling_optimizer, render_kwargs_train, batch_rays, target_s)
        if fused is not None:   # the standard configuration: a handful of C calls on three streams, no autograd graph
            return fused[0], fused[1], fused[2], None
        depth_net_rgb, depth_net_disp, extras = nerf_utils.render(self.H, self.W, self.K, chunk=self.chunk, rays=batch_rays,
                                                                  verbose=i < 10, retraw=True, **render_kwargs_train)
        sampling_optimizer.zero_grad()
        img_loss = nerf_utils.run_nerf_helpers.img2mse(depth_net_rgb, target_s)
        loss = img_loss
        psnr = nerf_utils.run_nerf_helpers.mse2psnr(img_loss)
        depth_net_loss = F.mse_loss(extras["depth_net_z_vals"], extras["max_z_vals"])
        # The reference calls depth_net_loss.backward(retain_graph=True) and then loss.backward() (Trainer.py:537-538): the
        # parameter gradients are the sum of the two.  One backward over both roots gives the same sum with ONE pass through
        # DepthNet's backward (autograd adds the two d/dz contributions before it reaches DepthNetTrainFn).
        torch.autograd.backward([depth_net_loss, loss])
        # detached: a caller that keeps the losses (the reference's loop keeps `psnr`) must not keep the autograd graph -- and
        # with it the parameters' AccumulateGrad nodes, which are bound to the stream they were created on -- alive
        return loss.detach(), depth_net_loss.detach(), psnr.detach(), None

    def reduce_and_step(self, sampling_optimizer):
        """Second half: data-parallel gradient all-reduce (one flat buffer) and the optimizer step (Trainer.py:542)."""
        from ... import parallel, training

        params = [p for g in sampling_optimizer.param_groups for p in g["params"]]
        scale = parallel.allreduce_gradients(params)
        if isinstance(sampling_optimizer, training.Adam):
            sampling_optimizer.step(grad_scale=scale)
        else:
            if scale != 1.0:
                for p in params:
                    if p.grad is not None:
                        p.grad.mul_(scale)
            sampling_optimizer.step()

    def update_learning_rate(self, optimizer):
        """Exponential decay of Trainer.py:546-551."""
        new_lrate = self.lrate * (0.1 ** (self.global_step / (self.lrate_decay * 1000)))
        for param_group in optimizer.param_groups:
            param_group["lr"] = new_lrate

    # ------------------------------------------------------------------ operators on the hot path
    def run_network(self, inputs, viewdirs, fn, embed_fn, embeddirs_fn, netchunk=1024 * 64):
        """raw [N,S,4] for sample positions ``inputs`` [N,S,3] (Trainer.py:789-806).

        The encodings described by ``embed_fn`` / ``embeddirs_fn`` are fused into the MLP kernel and the whole batch
        is one launch, so ``netchunk`` has nothing left to bound."""
        if viewdirs is None:
            raise NotImplementedError("the fused kernel implements the NeRF with view directions (use_viewdirs=True)")
        # the network's shapes fix the encodings; an embedder that states its size must agree with them
        m, mv = fn.multires()
        for name, e, want in (("embed_fn", embed_fn, m), ("embeddirs_fn", embeddirs_fn, mv)):
            got = getattr(e, "multires", None)
            if got is not None and got != want:
                raise ValueError(f"{name} encodes {got} octaves but the network was built for {want} "
                                 f"(multires {m}, multires_views {mv})")
        lead = list(inputs.shape[:-1])
        pts = inputs.reshape(viewdirs.shape[0], -1, 3)
        raw = fn.query(viewdirs, pts=pts)
        return raw.reshape(lead + [4])

    def raw2outputs(self, raw, z_vals, rays_d, raw_noise_std=0, white_bkgd=False, pytest=False):
        raise NotImplementedError

    def _sample_points(self, z_vals_mid, weights, perturb, pytest, rays_d, rays_o, n_importance=None):
        """Inverse-CDF samples + their positions (Trainer.py:553-577)."""
        if n_importance is None:
            n_importance = self.N_importance
        z_samples = nerf_utils.run_nerf_helpers.sample_pdf(z_vals_mid, weights[..., 1:-1], n_importance,
                                                           det=(perturb == 0.0), pytest=pytest)
        return z_samples, ops.points(rays_o, rays_d, z_samples)

    def sample_coarse_points(self, near, far, perturb, N_rays, N_samples, viewdirs, network_fn, network_query_fn, rays_o,
                             rays_d, raw_noise_std, white_bkgd, pytest, lindisp, **kwargs):
        """Stratified coarse pass (Trainer.py:579-649); 9-tuple with ``weights`` at slots 3 and 6."""
        if N_samples <= 0:
            return (None,) * 9
        t_rand = torch.rand(N_rays, N_samples, device=rays_o.device) if perturb > 0.0 else None
        z = ops.coarse_z(near, far, N_rays, N_samples, lindisp, t_rand)
        raw = network_fn.query(viewdirs, rays_o=rays_o, rays_d=rays_d, z=z)
        rgb, disp, acc, depth, density, alphas, weights = self.raw2outputs(raw, z, rays_d, raw_noise_std, white_bkgd, pytest=pytest)
        return rgb, disp, acc, weights, depth, z, weights, raw, None

    def sample_fine_points(self, z_vals, weights, perturb, pytest, rays_d, rays_o, rgb_map, disp_map, acc_map, network_fn,
                           network_fine, network_query_fn, viewdirs, raw_noise_std, white_bkgd):
        """Importance pass: sample_pdf, merge with the coarse depths, re-evaluate all (Trainer.py:651-710)."""
        if self.N_importance <= 0:
            return (None,) * 12
        u = None if perturb == 0.0 else torch.rand(z_vals.shape[0], self.N_importance, device=z_vals.device)
        z_samples, z_all, _ = ops.sample_pdf_merge(z_vals, weights, self.N_importance, u)
        run_fn = network_fn if network_fine is None else network_fine
        raw = run_fn.query(viewdirs, rays_o=rays_o, rays_d=rays_d, z=z_all)
        rgb, disp, acc, depth, density, alphas, w = self.raw2outputs(raw, z_all, rays_d, raw_noise_std, white_bkgd, pytest=pytest)
        pts = ops.points(rays_o, rays_d, z_all) if getattr(self, "save_scene_data", False) else None
        return rgb_map, disp_map, acc_map, rgb, disp, acc, raw, z_all, pts, density, alphas, w
