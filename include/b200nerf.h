/*
 * b200nerf.h -- C ABI of libb200nerf.so: the B200 (sm_100a) render_rays hot path of nerf-sampling.
 *
 * The reference (MarcinKadziolka/nerf-sampling) is pure Python/PyTorch and has no FFI of its own; the
 * boundary a maintainer binds is therefore "one entry point per reference operator", called with raw device
 * pointers (tensor.data_ptr()), element counts and a cudaStream_t.  Each declaration cites the reference
 * function (path relative to nerf_sampling/) whose ATen op sequence it replaces.  See INTEGRATION.md for the
 * ctypes stubs the reference side would add.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on error; b200nerf_last_error() gives the message
 *   - no allocation, no host synchronisation inside device entry points; all work is enqueued on `stream`
 *   - device pointers unless the parameter name starts with `h_`
 *   - fp32 tensors, row-major, contiguous
 */
#ifndef B200NERF_H
#define B200NERF_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200NERF_VERSION 100

/* precision of the tensor-core MLPs */
#define B200NERF_PREC_SPLIT 1 /* bf16 hi+lo operands, 3 MMAs / K16 block, ~16 mantissa bits (parity mode) */
#define B200NERF_PREC_FP16 2  /* plain fp16 operands, 1 MMA / K16 block, throughput kernel (PSNR-level parity)  */
#define B200NERF_PREC_FAST 3  /* PREC_FP16 + split-precision re-evaluation of the guard band
                                 (b200nerf_nerf_mlp_guarded_fwd): meets the 1e-3 max-abs contract          */

/* A packed NeRF on the device, as the fused render entry points take it. */
typedef struct b200nerf_nerf_model {
  const void* wpack;      /* slab stream of b200nerf_nerf_pack (PREC_SPLIT); NULL for PREC_FP16             */
  const void* wpack_fast; /* slab stream of b200nerf_nerf_pack_fast; NULL for SPLIT / BF16                   */
  const float* aux;       /* fp32 bias / head block                                                          */
  int prec;               /* B200NERF_PREC_*                                                                 */
  float guard_kappa;      /* PREC_FAST: guard-band width (relative to sum |h7 * w_alpha|)                    */
} b200nerf_nerf_model;

/* sample placement modes (nerf_pytorch/utils.py:220-244) */
#define B200NERF_PLACE_DEPTH_ONLY 0
#define B200NERF_PLACE_UNIFORM 1
#define B200NERF_PLACE_GAUSSIAN 2

int b200nerf_version(void);
const char* b200nerf_last_error(void);

/* ---- weight packing (host side, run once per checkpoint load / optimizer step) ------------------------- */

/* NeRF(D=8, W=256, input_ch=d, input_ch_views=dv, skips=[4], use_viewdirs=True)
 * (nerf_pytorch/run_nerf_helpers.py:67-107), d = 3 (1 + 2 multires), dv = 3 (1 + 2 multires_views).
 * `h_tensors` = 24 host fp32 pointers in this order:
 * pts_linears.0.weight, pts_linears.0.bias, ..., pts_linears.7.{weight,bias}, views_linears.0.{weight,bias},
 * feature_linear.{weight,bias}, alpha_linear.{weight,bias}, rgb_linear.{weight,bias}.
 * Produces the weight-slab stream (`h_wpack`, b200nerf_nerf_wpack_bytes(prec) bytes) and the fp32 bias/head
 * block (`h_aux`, b200nerf_nerf_aux_floats() floats); copy both to the device.
 * b200nerf_nerf_pack_multires serves multires 1..10 and multires_views 1..4: gamma(pts) fills the first d of the 64 columns of
 * its operand block, gamma(viewdir) the first dv of its 32, and the weights of the other columns are zero, so the image has the
 * size of every other multires.  It records both counts in the aux block, so every NeRF entry point that takes `aux` (render,
 * query, guard band, b200nerf_nerf_point_jvp_packed) encodes at the image's own sizes.  b200nerf_nerf_pack is the same with
 * 10 / 4. */
size_t b200nerf_nerf_wpack_bytes(int prec);
size_t b200nerf_nerf_aux_floats(void);
int b200nerf_nerf_pack(const float* const* h_tensors, int prec, void* h_wpack, float* h_aux);
int b200nerf_nerf_pack_multires(const float* const* h_tensors, int multires, int multires_views, int prec, void* h_wpack,
                                float* h_aux);

/* DepthNet (depth_nets/depth_net.py:10-169) in inference form.  Its three branches apply no activation
 * (depth_net.py:140,148,156 are no-ops), so branches + cat_layers[0] are one affine map of the encodings.
 * The host folds them (fp64) into `h_w0` [256,256] / `h_b0` [256] over the kernel's input layout, four 64-column blocks
 *   cols   0.. 63 enc(o) | 64..127 enc(d) | 128..191 enc(hit_near) | 192..255 enc(hit_far)
 * of which the first d3 = 3 (1 + 2 multires) columns hold the encoding and the rest are zero (multires 10: 63 of 64).
 * `h_hidden` = n_hidden pairs (weight [256,256], bias [256]) of the remaining cat_layers (LeakyReLU 0.01),
 * `h_head_w` [256] / `h_head_b` [1] = to_depth.  Narrower layers are zero-padded to 256 by the caller.
 * b200nerf_depthnet_pack_multires serves multires 1..10 and records it in the aux block, so b200nerf_depthnet_fwd and the
 * render entry points encode the rays at the image's own multires; b200nerf_depthnet_pack is the same with multires 10. */
size_t b200nerf_depthnet_wpack_bytes(int n_hidden, int prec);
size_t b200nerf_depthnet_aux_floats(int n_hidden);
int b200nerf_depthnet_pack(const float* h_w0, const float* h_b0, const float* const* h_hidden, int n_hidden,
                           const float* h_head_w, const float* h_head_b, int prec, void* h_wpack, float* h_aux);
int b200nerf_depthnet_pack_multires(const float* h_w0, const float* h_b0, const float* const* h_hidden, int n_hidden,
                                    const float* h_head_w, const float* h_head_b, int multires, int prec, void* h_wpack,
                                    float* h_aux);

/* ---- operators ------------------------------------------------------------------------------------------ */

/* get_rays + view-direction normalisation for one pinhole view
 * (run_nerf_helpers.py:187-202, nerf_utils.py:156-188).  h_c2w = 12 floats (3x4 row-major).
 * Outputs [H*W,3] each; any may be NULL. */
int b200nerf_get_rays(int H, int W, float fx, float fy, float cx, float cy, const float* h_c2w, float* rays_o,
                      float* rays_d, float* viewdirs, void* stream);

/* The same rays for selected pixels only (flat row-major indices, int64): training batches
 * (Trainer.sample_random_ray_batch, nerf_pytorch/trainers/Trainer.py:400-475) without materialising all H*W rays. */
int b200nerf_get_rays_at(int H, int W, float fx, float fy, float cx, float cy, const float* h_c2w, const long long* pix, int n,
                         float* rays_o, float* rays_d, float* viewdirs, void* stream);
/* out[t, :] = image[pix[t], :] -- the target colours of those pixels; image [H*W, channels] on the device. */
int b200nerf_gather_pixels(const float* image, const long long* pix, int n, int channels, float* out, void* stream);

/* viewdirs = rays_d / ||rays_d||  (nerf_utils.py:173) */
int b200nerf_normalize_dirs(const float* rays_d, int n_rays, float* viewdirs, void* stream);

/* DepthNet.forward: one depth in [near, far] per ray (depth_nets/depth_net.py:117-169).  out_z [n_rays].
 * The split-precision kernel encodes the rays one tile ahead into a library-owned staging buffer (~19 MB per device,
 * allocated by the first call on that device -- call once before capturing a CUDA graph); launches of this entry point
 * on the same device must therefore be stream-ordered with respect to each other. */
int b200nerf_depthnet_fwd(const void* wpack, const float* aux, int n_hidden, int prec, const float* rays_o,
                          const float* rays_d, int n_rays, float radius, float near_, float far_, float* out_z,
                          void* stream);

/* sample_points_around_mean (nerf_pytorch/utils.py:220-244) without materialising pts.
 * mean [n_rays]; uniform: `offsets` = the S-1 grid values linspace(-std, std, S-1) (shared by all rays) and the
 * result is clipped to [clip_lo, clip_hi]; gaussian: `offsets` = [n_rays, S-1] already scaled noise (std*randn),
 * no clip; depth_only: S must be 1.  out_z [n_rays, S], ascending per ray. */
int b200nerf_place_samples(const float* mean, const float* offsets, int n_rays, int S, int mode, float clip_lo,
                           float clip_hi, float* out_z, void* stream);

/* pts = rays_o + rays_d * z  ([n_rays,S,3]; the reference materialises it, we only do on request) */
int b200nerf_points(const float* rays_o, const float* rays_d, const float* z, int n_rays, int S, float* out_pts,
                    void* stream);

/* Backward of sample_points_around_mean (nerf_pytorch/utils.py:220-244) w.r.t. `mean`: every placed depth is mean + a constant,
 * so out_g_mean [n_rays] = sum_s g_z[ray, s], except that uniform mode drops the samples torch.clip(z, clip_lo, clip_hi) cut:
 * the mask is clip_lo <= mean + offset <= clip_hi (inclusive, on the UNclipped value; a sample clipped onto a bound gets no
 * gradient).  Gaussian mode has no mask (offsets may be NULL); depth_only (S == 1) is the identity.  Arguments as in
 * b200nerf_place_samples; g_z [n_rays, S]. */
int b200nerf_place_samples_bwd(const float* mean, const float* offsets, int n_rays, int S, int mode, float clip_lo, float clip_hi,
                               const float* g_z, float* out_g_mean, void* stream);

/* Backward of b200nerf_points w.r.t. z: out_g_z [n_rays,S] = sum_k g_pts[ray,s,k] rays_d[ray,k]. */
int b200nerf_points_bwd(const float* rays_d, const float* g_pts, int n_rays, int S, float* out_g_z, void* stream);

/* Trainer.run_network + NeRF.forward (nerf_pytorch/trainers/Trainer.py:789-806,
 * run_nerf_helpers.py:109-134): positional encoding of the sample positions (d wide, 63 at multires 10) and view directions
 * (dv wide, 27 at multires_views 4; both sizes from `aux`) fused into the 8x256 skip@4 MLP.  Sample positions are either o + d*z (`z` [n_rays,S], `pts` NULL) or explicit
 * (`pts` [n_rays,S,3]).  out_raw [n_rays,S,4] = (r,g,b,sigma) pre-activation. */
int b200nerf_nerf_mlp_fwd(const void* wpack, const float* aux, int prec, const float* rays_o, const float* rays_d,
                          const float* viewdirs, const float* z, const float* pts, int n_rays, int S, float* out_raw,
                          void* stream);

/* Single-pass 16-bit image of the same 24 NeRF tensors for the fast kernel (prec = FP16 or BF16):
 * b200nerf_nerf_fast_wpack_bytes() bytes; the fp32 bias/head block is the `h_aux` of b200nerf_nerf_pack.  The _multires form
 * takes the sizes of b200nerf_nerf_pack_multires; its aux block (packed at the same sizes) carries them to the kernel. */
size_t b200nerf_nerf_fast_wpack_bytes(void);
int b200nerf_nerf_pack_fast(const float* const* h_tensors, int prec, void* h_wpack);
int b200nerf_nerf_pack_fast_multires(const float* const* h_tensors, int multires, int multires_views, int prec, void* h_wpack);

/* Same operator as b200nerf_nerf_mlp_fwd on the throughput kernel: two 128-row tiles per SM ping-pong between the
 * tensor core and the epilogue warps, SMs paired as 2-CTA clusters (tcgen05 cta_group::2), one MMA per K16 block.
 * Guard band (optional, guard_count != NULL): every LAST sample of a ray whose |sigma| < guard_kappa * sum|h7*w_alpha|
 * is appended to guard_list (int point indices, at most guard_cap) and counted in guard_count[0] (zeroed by the
 * caller) -- those are the samples whose sign raw2outputs turns into a step function (dist = 1e10,
 * trainers/sampling_trainer.py:178-180). */
int b200nerf_nerf_mlp_fast_fwd(const void* wpack_fast, const float* aux, int prec, const float* rays_o,
                               const float* rays_d, const float* viewdirs, const float* z, const float* pts, int n_rays,
                               int S, float* out_raw, int* guard_count, int* guard_list, int guard_cap, float guard_kappa,
                               void* stream);

/* Fast pass + split-precision re-evaluation of the guard band, in place: the result meets the reference within
 * 1e-3 max-abs like PREC_SPLIT at ~1/3 of the tensor work.  ws_guard: n_rays + 4 ints of device workspace. */
int b200nerf_nerf_mlp_guarded_fwd(const void* wpack_fast, const void* wpack_split, const float* aux, int prec,
                                  const float* rays_o, const float* rays_d, const float* viewdirs, const float* z,
                                  const float* pts, int n_rays, int S, float guard_kappa, int* ws_guard, float* out_raw,
                                  void* stream);

/* Tuning knob: cap the persistent grids of the MLP kernels (b200nerf_nerf_* / b200nerf_depthnet_fwd launched by the calling host
 * thread) at n_sms CTAs so that work on another stream finds free SMs beside them; 0 removes the cap.  Returns the previous value.
 * Results do not depend on it (tiles are distributed grid-stride). */
int b200nerf_set_sm_limit(int n_sms);

/* Precision dispatch over the three entry points above.  ws_guard (n_rays + 4 ints) is needed for PREC_FAST only. */
int b200nerf_nerf_query(const b200nerf_nerf_model* nerf, const float* rays_o, const float* rays_d, const float* viewdirs,
                        const float* z, const float* pts, int n_rays, int S, int* ws_guard, float* out_raw, void* stream);

/* DepthNetTrainer.raw2outputs (trainers/sampling_trainer.py:153-230, raw2alpha nerf_utils.py:27-42).
 * raw [n_rays,S,4], z [n_rays,S], rays_d [n_rays,3], noise [n_rays,S] or NULL (already scaled by raw_noise_std).
 * Outputs: rgb [n_rays,3], disp/acc/depth [n_rays], weights/alphas [n_rays,S] (each may be NULL).
 * S == 1 reproduces the reference's empty-interval quirk: rgb = sigmoid(raw rgb), acc = depth = 0, disp = 1e10. */
int b200nerf_composite_fwd(const float* raw, const float* z, const float* rays_d, const float* noise, int n_rays,
                           int S, int white_bkgd, float* out_rgb, float* out_disp, float* out_acc, float* out_depth,
                           float* out_weights, float* out_alphas, void* stream);

/* Reverse-mode derivative of DepthNetTrainer.raw2outputs (trainers/sampling_trainer.py:153-230) for S >= 2 (S == 1 has no
 * intervals; its colour is sigmoid(raw rgb)).  Inputs as in b200nerf_composite_fwd; upstream gradients g_rgb [n_rays,3],
 * g_disp / g_acc / g_depth [n_rays], g_weights / g_alphas [n_rays,S] -- each may be NULL, meaning zero.  Writes out_g_raw
 * [n_rays,S,4] (sigmoid' on the colour channels; relu'(sigma + noise) times d alpha / d relu on sigma, relu'(0) = 0) and out_g_z
 * [n_rays,S] (through dists = (z_{i+1} - z_i) |rays_d| and depth = sum w z; the 1e10 last interval does not depend on z).  The
 * transmittance term is a reverse scan in double, R_i = g_{i+1} alpha_{i+1} + t_{i+1} R_{i+1}, g_alpha_i = T_i (g_w_i - R_i), with
 * no division by t = 1 - alpha + 1e-10, so the gradient survives where T underflows in fp32.  disp = 1 / max(1e-10, q) sends
 * the gradient to q = depth / (acc + 1e-10) where q > 1e-10 (half of it on a tie), like torch.max. */
int b200nerf_composite_bwd(const float* raw, const float* z, const float* rays_d, const float* noise, int n_rays, int S,
                           int white_bkgd, const float* g_rgb, const float* g_disp, const float* g_acc, const float* g_depth,
                           const float* g_weights, const float* g_alphas, float* out_g_raw, float* out_g_z, void* stream);

/* Same arithmetic, image-tile output: out_rgbd [n_rays,4] = (r, g, b, disp) per ray -- the layout the multi-GPU render
 * all-gathers (one 16-byte pixel per ray, SURVEY.md 8(e)), written by the kernel itself instead of two copy launches. */
int b200nerf_composite_tile_fwd(const float* raw, const float* z, const float* rays_d, const float* noise, int n_rays,
                                int S, int white_bkgd, float* out_rgbd, float* out_acc, float* out_depth,
                                float* out_weights, float* out_alphas, void* stream);

/* render_rays_test, DepthNet mode (nerf_utils.py:736-876): depthnet -> place -> encode+MLP -> composite for
 * n_rays rays already on the device.  ws_z [n_rays,S] and ws_raw [n_rays,S,4] are caller-provided workspaces
 * that double as the `depth_net_z_vals` / `raw` extras; ws_guard = n_rays + 4 ints (PREC_FAST only, else may be
 * NULL); out_weights may be NULL.  dn_prec is the DepthNet's precision (SPLIT or BF16). */
int b200nerf_render_depthnet(const void* dn_wpack, const float* dn_aux, int dn_hidden, int dn_prec,
                             const b200nerf_nerf_model* nerf, const float* rays_o, const float* rays_d,
                             const float* viewdirs, int n_rays, int S, int mode, const float* offsets, float radius,
                             float near_, float far_, float* ws_mean, float* ws_z, float* ws_raw, int* ws_guard,
                             float* out_rgb, float* out_disp, float* out_acc, float* out_depth, float* out_weights,
                             void* stream);

/* b200nerf_render_depthnet with the image-tile output of b200nerf_composite_tile_fwd (out_rgbd [n_rays,4]). */
int b200nerf_render_depthnet_tile(const void* dn_wpack, const float* dn_aux, int dn_hidden, int dn_prec,
                                  const b200nerf_nerf_model* nerf, const float* rays_o, const float* rays_d,
                                  const float* viewdirs, int n_rays, int S, int mode, const float* offsets, float radius,
                                  float near_, float far_, float* ws_mean, float* ws_z, float* ws_raw, int* ws_guard,
                                  float* out_rgbd, float* out_acc, float* out_depth, float* out_weights, void* stream);

/* Same, through host memory: copies h_rays_o / h_rays_d ([n_rays,3] each, ideally pinned) to the device
 * workspace, renders, copies rgb [n_rays,3] and disp [n_rays] back and synchronises `stream`.
 * d_ws must hold b200nerf_render_host_ws_bytes(n_rays, S) bytes. */
size_t b200nerf_render_host_ws_bytes(int n_rays, int S);
int b200nerf_render_depthnet_host(const void* dn_wpack, const float* dn_aux, int dn_hidden, int dn_prec,
                                  const b200nerf_nerf_model* nerf, const float* h_rays_o, const float* h_rays_d,
                                  int n_rays, int S, int mode, const float* offsets, float radius, float near_,
                                  float far_, void* d_ws, float* h_rgb, float* h_disp, void* stream);

/* ---- vanilla hierarchical sampling (config #4 and the training target) ---------------------------------- */

/* Stratified coarse depths of Trainer.sample_coarse_points (nerf_pytorch/trainers/Trainer.py:603-627).
 * near_/far_ [n_rays], t [S] = linspace(0,1,S); lindisp != 0 samples linearly in disparity (the reference
 * default); t_rand [n_rays,S] in [0,1) enables the stratified jitter (perturb > 0), NULL disables it. */
int b200nerf_coarse_depths(const float* near_, const float* far_, const float* t, int n_rays, int S, int lindisp,
                           const float* t_rand, float* out_z, void* stream);

/* sample_pdf (nerf_pytorch/run_nerf_helpers.py:250-293): bins [n_rays,n_bins], weights [n_rays,n_bins-1],
 * u = [n_samples] shared by all rays (u_per_ray == 0, the det=True linspace) or [n_rays,n_samples].
 * out_samples [n_rays,n_samples]; out_inds (may be NULL) = the searchsorted(cdf, u, right=True) indices, int64. */
int b200nerf_sample_pdf(const float* bins, const float* weights, const float* u, int u_per_ray, int n_rays, int n_bins,
                        int n_samples, float* out_samples, long long* out_inds, void* stream);

/* Trainer.sample_fine_points up to the network query (Trainer.py:668-686): mid-point bins of the coarse depths,
 * inner coarse weights, inverse-CDF samples, then sort(cat([z_coarse, z_samples])) -> out_z_all
 * [n_rays, n_coarse+n_importance].  out_samples / out_inds may be NULL. */
int b200nerf_sample_pdf_merge(const float* z_coarse, const float* weights, const float* u, int u_per_ray, int n_rays,
                              int n_coarse, int n_importance, float* out_samples, long long* out_inds, float* out_z_all,
                              void* stream);

/* top = weights.argmax(1) (first maximum) and the gathers that follow it (nerf_utils.py:689-690, :806-812):
 * out_idx int64 [n_rays], out_z / out_w [n_rays], out_rgb [n_rays,3] = sigmoid(raw rgb at top) (raw may be NULL). */
int b200nerf_argmax_gather(const float* weights, const float* z, const float* raw, int n_rays, int S, long long* out_idx,
                           float* out_z, float* out_w, float* out_rgb, void* stream);

/* ---- training (config #5: Trainer.core_optimization_loop, trainers/Trainer.py:506-544) --------------------------- */

/* DepthNet's training forward with saved activations (depth_nets/depth_net.py:117-169): the activation-free branches collapsed to
 * weight-only recurrences (fp32), the branch product and cat_layers.0 as error-compensated 3xTF32 products, the 256-wide activated
 * cat layers behind it + the head as ONE launch of the split-precision tensor-core MLP kernel (bf16 hi + lo operands, fp32
 * accumulate; B200NERF_TRAIN_CHAIN=gemm: per-layer 3xTF32 products; B200NERF_TRAIN_GEMM=fp32: CUDA-core fp32 everywhere).
 * `params` = device pointers of the state_dict tensors in order: origin_layers.{i}.{weight,bias} (n_branch layers of
 * widths hidden[]), direction_layers..., intersection_layers..., cat_layers.{2j}.{weight,bias} (n_cat layers of widths
 * cat_hidden[]), to_depth.0.{weight,bias}: b200nerf_depthnet_n_params() pointers.  `ws` holds
 * b200nerf_depthnet_train_ws_floats() floats and carries the activations from fwd to bwd.  out_z [n_rays].
 * The functions without a `multires` argument serve DepthNet(multires=10); their _multires forms take the positional-encoding
 * size (1..10: gamma(o), gamma(d) are d3 = 3 (1 + 2 multires) wide, gamma(hits) 2 d3), which must be the same in every call of a step. */
size_t b200nerf_depthnet_train_ws_floats(int n_rays, int n_branch, const int* hidden, int n_cat, const int* cat_hidden);
size_t b200nerf_depthnet_train_ws_floats_multires(int n_rays, int n_branch, const int* hidden, int n_cat, const int* cat_hidden,
                                                 int multires);
int b200nerf_depthnet_n_params(int n_branch, int n_cat);
int b200nerf_depthnet_train_fwd(const float* const* params, int n_branch, const int* hidden, int n_cat, const int* cat_hidden,
                                const float* rays_o, const float* rays_d, int n_rays, float radius, float near_, float far_,
                                float* ws, float* out_z, void* stream);
int b200nerf_depthnet_train_fwd_multires(const float* const* params, int n_branch, const int* hidden, int n_cat, const int* cat_hidden,
                                         int multires, const float* rays_o, const float* rays_d, int n_rays, float radius, float near_,
                                         float far_, float* ws, float* out_z, void* stream);
/* Backward of the above: dz [n_rays] -> gradients of every parameter, written (not accumulated) to `grads` (same order
 * and shapes as `params`).  Consumes the activations in `ws`. */
int b200nerf_depthnet_train_bwd(const float* const* params, int n_branch, const int* hidden, int n_cat, const int* cat_hidden,
                                int n_rays, float near_, float far_, float* ws, const float* dz, float* const* grads,
                                void* stream);
int b200nerf_depthnet_train_bwd_multires(const float* const* params, int n_branch, const int* hidden, int n_cat, const int* cat_hidden,
                                         int multires, int n_rays, float near_, float far_, float* ws, const float* dz,
                                         float* const* grads, void* stream);

/* The same backward split at the losses (Trainer.py:525-538: both losses reach DepthNet through ONE scalar per ray, dz, and the
 * backward is linear in it).  b200nerf_depthnet_train_jac runs BEFORE the losses exist: it zeroes `grads` and walks the sequential
 * input-gradient chain with a unit upstream gradient, leaving J_j = d z / d(pre-activation of cat layer j) in `ws`.
 * b200nerf_depthnet_train_bwd_jac then forms every gradient from dz and the J_j as independent products (one grouped launch) plus
 * the weight-only branch chain.  Same results as b200nerf_depthnet_train_bwd up to rounding; where the split does not apply
 * (CUDA-core GEMM path, literal branches, fewer than 32 rays) _jac does nothing and _bwd_jac IS b200nerf_depthnet_train_bwd.
 * One _bwd_jac per _jac: the gradients and the branches' ray reduction are accumulated into what _jac zeroed.
 * stream_aux (optional, another stream of the same device): the weight-only branch chain runs there beside the cat layers' weight
 * gradients; `stream` waits for it before the call's work is complete (event fork / join, capturable in a CUDA graph). */
int b200nerf_depthnet_train_jac(const float* const* params, int n_branch, const int* hidden, int n_cat, const int* cat_hidden,
                                int n_rays, float near_, float far_, float* ws, float* const* grads, void* stream);
int b200nerf_depthnet_train_bwd_jac(const float* const* params, int n_branch, const int* hidden, int n_cat, const int* cat_hidden,
                                    int n_rays, float near_, float far_, float* ws, const float* dz, float* const* grads,
                                    void* stream, void* stream_aux);
int b200nerf_depthnet_train_jac_multires(const float* const* params, int n_branch, const int* hidden, int n_cat, const int* cat_hidden,
                                         int multires, int n_rays, float near_, float far_, float* ws, float* const* grads, void* stream);
int b200nerf_depthnet_train_bwd_jac_multires(const float* const* params, int n_branch, const int* hidden, int n_cat,
                                             const int* cat_hidden, int multires, int n_rays, float near_, float far_, float* ws,
                                             const float* dz, float* const* grads, void* stream, void* stream_aux);

/* The frozen NeRF at ONE sample per ray, p = o + d z (nerf_utils.py:693-715), in fp32, together with d raw / d z
 * (forward-mode derivative along the ray: what loss.backward() propagates from the colour into DepthNet's depth).
 * `params` = the 24 fp32 device tensors in the order of b200nerf_nerf_pack; ws: b200nerf_nerf_point_ws_floats() floats;
 * out_raw [n_rays,4], out_draw_dz [n_rays,4]. */
size_t b200nerf_nerf_point_ws_floats(int n_rays);
int b200nerf_nerf_point_jvp(const float* const* params, const float* rays_o, const float* rays_d, const float* viewdirs,
                            const float* z, int n_rays, float* ws, float* out_raw, float* out_draw_dz, void* stream);
/* The same at multires 1..10 / multires_views 1..4 (the tensors' shapes: pts_linears.0 [256, d], pts_linears.5 [256, d + 256],
 * views_linears.0 [128, 256 + dv]); the functions above are these with 10 / 4.  The workspace size returns 0 out of range. */
size_t b200nerf_nerf_point_ws_floats_multires(int n_rays, int multires, int multires_views);
int b200nerf_nerf_point_jvp_multires(const float* const* params, int multires, int multires_views, const float* rays_o,
                                     const float* rays_d, const float* viewdirs, const float* z, int n_rays, float* ws,
                                     float* out_raw, float* out_draw_dz, void* stream);
/* The same at S samples per ray (Trainer.run_network on o + d z, run_nerf_helpers.py:109-134, differentiated along z):
 * z [n_rays,S], out_raw / out_draw_dz [n_rays*S,4]; the sample points are the rows and row r uses ray r / S.  The functions above
 * are these with S = 1.  ws: b200nerf_nerf_samples_ws_floats_multires(n_rays, S, ...) floats (0 on bad arguments). */
size_t b200nerf_nerf_samples_ws_floats_multires(int n_rays, int S, int multires, int multires_views);
int b200nerf_nerf_samples_jvp_multires(const float* const* params, int multires, int multires_views, const float* rays_o,
                                       const float* rays_d, const float* viewdirs, const float* z, int n_rays, int S, float* ws,
                                       float* out_raw, float* out_draw_dz, void* stream);

/* The same two outputs from the PACKED split-precision model (b200nerf_nerf_pack: bf16 hi + lo operands, three MMAs per block,
 * fp32 accumulate -- the precision of B200NERF_PREC_SPLIT inference) in two launches of the fused tensor-core MLP kernel instead
 * of ~13 grouped products: a primal pass that also records the ReLU masks, and a tangent pass t_k = mask_k * (W_k t_{k-1}).
 * ws: b200nerf_nerf_point_jvp_packed_ws_bytes() bytes (the masks). */
size_t b200nerf_nerf_point_jvp_packed_ws_bytes(int n_rays);
int b200nerf_nerf_point_jvp_packed(const void* wpack, const float* aux, const float* rays_o, const float* rays_d,
                                   const float* viewdirs, const float* z, int n_rays, void* ws, float* out_raw,
                                   float* out_draw_dz, void* stream);
/* The same at S samples per ray: z [n_rays,S], out_raw / out_draw_dz [n_rays*S,4]; the masks are MAX_STEPS x n_rays*S x 4
 * words (b200nerf_nerf_samples_jvp_packed_ws_bytes(n_rays, S) bytes).  The two functions above are these with S = 1. */
size_t b200nerf_nerf_samples_jvp_packed_ws_bytes(int n_rays, int S);
int b200nerf_nerf_samples_jvp_packed(const void* wpack, const float* aux, const float* rays_o, const float* rays_d,
                                     const float* viewdirs, const float* z, int n_rays, int S, void* ws, float* out_raw,
                                     float* out_draw_dz, void* stream);
/* raw and its Jacobian w.r.t. EXPLICIT sample points (Trainer.run_network(pts, ...), Trainer.py:789-806): pts [n_rays,S,3],
 * viewdirs [n_rays,3]; one primal pass with masks, then three tangent passes along the unit axes.  out_raw [n_rays*S,4],
 * out_draw_dpts [n_rays*S,3,4] (d raw / d x, y, z); ws as for b200nerf_nerf_samples_jvp_packed. */
int b200nerf_nerf_pts_jvp_packed(const void* wpack, const float* aux, const float* pts, const float* viewdirs, int n_rays, int S,
                                 void* ws, float* out_raw, float* out_draw_dpts, void* stream);

/* torch.optim.Adam (no weight decay, no amsgrad) on one tensor; the gradient is multiplied by grad_scale first
 * (1/world_size after a sum all-reduce).  step counts from 1. */
int b200nerf_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, size_t n, float lr, float beta1,
                       float beta2, float eps, int step, float grad_scale, void* stream);

/* The same update over a list of tensors in one launch.  d_table: DEVICE array of n_tensors records
 * {float* param; const float* grad; float* exp_avg; float* exp_avg_sq; uint64 numel} (40 bytes each); all tensors share
 * lr / betas / eps / step. */
int b200nerf_adam_step_multi(const void* d_table, int n_tensors, float lr, float beta1, float beta2, float eps, int step,
                             float grad_scale, void* stream);

/* Losses of Trainer.core_optimization_loop on the DepthNet path (nerf_pytorch/trainers/Trainer.py:525-538) and the gradient they send
 * into the predicted depth, in one pass: raw [n,1,4] and draw_dz [n,4] from b200nerf_nerf_point_jvp, z_dn / max_z [n], target [n,3].
 * out_losses = {img_loss = mean((sigmoid(raw rgb) - target)^2), depth_net_loss = mean((z_dn - max_z)^2), psnr = -10 log10(img_loss)};
 * out_dz [n] = d(depth_net_loss + img_loss)/d z_dn (what the reference's two backward() calls accumulate);  ws2: 2 floats of scratch. */
int b200nerf_train_loss(const float* raw, const float* draw_dz, const float* z_dn, const float* max_z, const float* target,
                        int n_rays, float* ws2, float* out_losses, float* out_dz, void* stream);

/* CUDA-graph friendly form: the step counter (*d_step, incremented by the call) and {lr, beta1, beta2, eps, grad_scale}
 * (d_hyper, 5 floats) live in device memory, so a captured launch stays valid while they change. */
int b200nerf_adam_step_multi_dev(const void* d_table, int n_tensors, const float* d_hyper, int* d_step, void* stream);

/* ---- diagnostics ------------------------------------------------------------------------------------------ */

/* D[128,N] = A[128,K] * B[N,K]^T with bf16 inputs (raw uint16), through the same shared-memory operand layout,
 * UMMA descriptors and TMEM read-back as the MLP kernels.  K % 16 == 0, K <= 128, N % 16 == 0, N <= 256. */
int b200nerf_umma_selftest(const uint16_t* A, const uint16_t* B, float* D, int K, int N, void* stream);

/* The strided fp32 GEMM of the training slice, C[M,N] = (beta ? C : 0) + sum_k A[m*sAm + k*sAk] * B[k*sBk + n*sBn] (+ bias[n])
 * (then LeakyReLU(slope) if act): covers X*W^T (Linear forward, depth_net.py:117-169), dY*W and dY^T*X (its backward) without
 * transposes.  Runs as an error-compensated 3xTF32 product on the tcgen05 tensor cores (csrc/tgemm.cuh) unless
 * force_fp32 != 0 or B200NERF_TRAIN_GEMM=fp32 (CUDA-core fp32 kernel).  Exposed for the parity tests. */
int b200nerf_debug_sgemm(int M, int N, int K, const float* A, long sAm, long sAk, const float* B, long sBk, long sBn, float* C,
                         int ldc, int beta, const float* bias, int act, float slope, int force_fp32, void* stream);

/* Diagnostics: the kernels b200nerf_depthnet_train_fwd / _bwd / _jac / _bwd_jac pick for this architecture, batch and parameter
 * alignment, as a bitmask of the predicates they call.  Host code only (reads the pointer values of params, launches nothing);
 * a negative value on bad arguments.
 *   COLLAPSED       the branches run as weight-only recurrences (chain_fwd / chain_bwd / chain_du, 2-CTA clusters), else per layer
 *   FUSED_CHAIN     cat_layers.1 .. n_cat-1 + head in one launch of the split-precision MLP kernel, else per-layer 3xTF32 products
 *   SPLIT_CAT0      cat_layers.0 as four split-K problems (its bias and LeakyReLU move into the fused chain's loader)
 *   SPLIT_BACKWARD  _jac / _bwd_jac run the split backward, else _bwd_jac runs the one-pass backward
 *   TENSOR_PATH     the one-pass backward runs on the tensor-core products, else on the CUDA-core head kernels and mixed products */
#define B200NERF_ROUTE_COLLAPSED 1
#define B200NERF_ROUTE_FUSED_CHAIN 2
#define B200NERF_ROUTE_SPLIT_CAT0 4
#define B200NERF_ROUTE_SPLIT_BACKWARD 8
#define B200NERF_ROUTE_TENSOR_PATH 16
int b200nerf_debug_depthnet_train_route(const float* const* params, int n_branch, const int* hidden, int n_cat, const int* cat_hidden,
                                        int n_rays);
int b200nerf_debug_depthnet_train_route_multires(const float* const* params, int n_branch, const int* hidden, int n_cat,
                                                 const int* cat_hidden, int multires, int n_rays);

/* Diagnostics: CTA 0 of every grouped-GEMM launch writes %globaltimer stamps (ns) of its phases into dev_buf (16 int64):
 * [0] entry, [1] barriers + TMEM ready, [2] last MMA retired, [3] epilogue stored, [4+c] chunk c handed to the MMA warp. */
void b200nerf_debug_set_tgemm_timeline(long long* dev_buf);

/* Diagnostics: the per-step device-side re-pack of DepthNet's 256 x 256 cat layers for the fused training chain (bf16 hi / lo
 * images of W_j for the forward launch and of W_{n-1-j}^T for the Jacobian launch, fp32 bias / head block), exposed so that a
 * test can compare it byte for byte with the host packer of the inference path.  d_W / d_b: host arrays of n_layers DEVICE
 * pointers ([256,256] / [256]); images: b200nerf_debug_catchain_img_bytes() bytes each; d_aux: b200nerf_nerf_aux_floats() floats. */
size_t b200nerf_debug_catchain_img_bytes(int n_layers);
int b200nerf_debug_catchain_pack(const float* const* d_W, const float* const* d_b, const float* d_head_w, const float* d_head_b,
                                 int n_layers, void* d_img_fwd, void* d_img_jac, float* d_aux, void* stream);

/* number of kernels this library has launched since load (bench.py reports it as gpu_launches) */
unsigned long long b200nerf_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* B200NERF_H */
