// Vanilla hierarchical-sampling kernels (config #4 and the training target): stratified coarse depths,
// inverse-CDF importance sampling fused with the coarse/fine merge, and arg-max extraction.
#include <cstdint>

#include "../../include/b200nerf.h"
#include "host_common.h"

#define fail b200_fail

// ------------------------------------------------------------------------------------------- coarse depths
// Trainer.sample_coarse_points (nerf_pytorch/trainers/Trainer.py:603-627): z over t = linspace(0,1,S), linear in
// depth or in disparity, optionally jittered inside the stratified bins.
__device__ __forceinline__ float coarse_depth(float nr, float fr, float t, int lindisp) {
  const float omt = __fadd_rn(1.0f, -t);
  if (lindisp) {
    const float a = __fmul_rn(__fdiv_rn(1.0f, nr), omt);
    const float b = __fmul_rn(__fdiv_rn(1.0f, fr), t);
    return __fdiv_rn(1.0f, __fadd_rn(a, b));
  }
  return __fadd_rn(__fmul_rn(nr, omt), __fmul_rn(fr, t));
}

__global__ void coarse_depths_kernel(const float* __restrict__ near_, const float* __restrict__ far_,
                                     const float* __restrict__ t, int n_rays, int S, int lindisp,
                                     const float* __restrict__ t_rand, float* __restrict__ z) {
  const size_t idx = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<size_t>(n_rays) * S) return;
  const int s = static_cast<int>(idx % S);
  const size_t ray = idx / S;
  const float nr = near_[ray], fr = far_[ray];
  const float zc = coarse_depth(nr, fr, t[s], lindisp);
  if (t_rand == nullptr) {
    z[idx] = zc;
    return;
  }
  const float zl = s > 0 ? coarse_depth(nr, fr, t[s - 1], lindisp) : zc;
  const float zu = s + 1 < S ? coarse_depth(nr, fr, t[s + 1], lindisp) : zc;
  const float lower = s > 0 ? __fmul_rn(0.5f, __fadd_rn(zc, zl)) : zc;
  const float upper = s + 1 < S ? __fmul_rn(0.5f, __fadd_rn(zu, zc)) : zc;
  z[idx] = __fadd_rn(lower, __fmul_rn(__fadd_rn(upper, -lower), t_rand[idx]));
}

extern "C" int b200nerf_coarse_depths(const float* near_, const float* far_, const float* t, int n_rays, int S, int lindisp,
                                      const float* t_rand, float* out_z, void* stream) {
  if (n_rays < 0 || S < 1) return fail("b200nerf_coarse_depths: bad sizes");
  if (n_rays == 0) return 0;
  if (!near_ || !far_ || !t || !out_z) return fail("b200nerf_coarse_depths: null argument");
  const size_t total = static_cast<size_t>(n_rays) * S;
  coarse_depths_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      near_, far_, t, n_rays, S, lindisp, t_rand, out_z);
  LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------- sample_pdf (+ merge)
// sample_pdf (run_nerf_helpers.py:250-293) for one ray per warp.  The CDF lives in shared memory; the running
// sums are carried in double and rounded to float per knot, which is what torch's CPU cumsum does, so on
// identical inputs the searchsorted indices agree with the reference except for u within an ulp of a knot.
// With z_all != nullptr the importance samples are merged with the coarse depths (Trainer.py:675-686):
// a bitonic sort of the padded row, which is also correct for unsorted (random-u) samples.
template <bool FROM_COARSE>
__global__ void sample_pdf_kernel(const float* __restrict__ bins_or_z, const float* __restrict__ weights,
                                  const float* __restrict__ u, int u_per_ray, int n_rays, int B /*knots*/, int Sf, int P,
                                  float* __restrict__ o_samples, long long* __restrict__ o_inds, float* __restrict__ o_all) {
  extern __shared__ float sm[];
  const int wpb = blockDim.x >> 5, wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ray = blockIdx.x * wpb + wib;
  if (ray >= n_rays) return;  // whole warp leaves together
  // per-warp carve-up: bins[B], cdf[B], row[P], merged[B + 1 + Sf]
  float* bins = sm + static_cast<size_t>(wib) * (2 * B + P + B + 1 + Sf);
  float* cdf = bins + B;
  float* row = cdf + B;
  const int Sc = B + 1;  // coarse samples when FROM_COARSE
  const float* zsrc = bins_or_z + static_cast<size_t>(ray) * (FROM_COARSE ? Sc : B);
  // weights: FROM_COARSE -> coarse weights [Sc], inner ones 1..Sc-2 are used; else [B-1]
  const float* wsrc = weights + static_cast<size_t>(ray) * (FROM_COARSE ? Sc : B - 1) + (FROM_COARSE ? 1 : 0);
  const int nw = B - 1;

  for (int i = lane; i < B; i += 32)
    bins[i] = FROM_COARSE ? __fmul_rn(0.5f, __fadd_rn(zsrc[i + 1], zsrc[i])) : zsrc[i];
  // sum of (w + 1e-5)
  double part = 0.0;
  for (int i = lane; i < nw; i += 32) part += static_cast<double>(__fadd_rn(wsrc[i], 1e-5f));
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) part += __shfl_xor_sync(0xffffffffu, part, off);
  const float total = static_cast<float>(part);
  // cdf[0] = 0, cdf[i+1] = float(sum_{j<=i} pdf_j), pdf_j = (w_j + 1e-5) / total
  double carry = 0.0;
  if (lane == 0) cdf[0] = 0.f;
  for (int i0 = 0; i0 < nw; i0 += 32) {
    const int i = i0 + lane;
    double v = i < nw ? static_cast<double>(__fdiv_rn(__fadd_rn(wsrc[i], 1e-5f), total)) : 0.0;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const double t = __shfl_up_sync(0xffffffffu, v, off);
      if (lane >= off) v += t;
    }
    if (i < nw) cdf[i + 1] = static_cast<float>(carry + v);
    carry += __shfl_sync(0xffffffffu, v, 31);
  }
  __syncwarp();

  for (int k = lane; k < Sf; k += 32) {
    const float uu = u[u_per_ray ? static_cast<size_t>(ray) * Sf + k : k];
    // searchsorted(cdf, u, right=True): number of knots <= u
    int lo = 0, hi = B;
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (cdf[mid] <= uu) lo = mid + 1;
      else hi = mid;
    }
    const int below = lo - 1 > 0 ? lo - 1 : 0;
    const int above = lo < B - 1 ? lo : B - 1;
    float denom = __fadd_rn(cdf[above], -cdf[below]);
    if (denom < 1e-5f) denom = 1.0f;
    const float tt = __fdiv_rn(__fadd_rn(uu, -cdf[below]), denom);
    const float smp = __fadd_rn(bins[below], __fmul_rn(tt, __fadd_rn(bins[above], -bins[below])));
    if (o_samples) o_samples[static_cast<size_t>(ray) * Sf + k] = smp;
    if (o_inds) o_inds[static_cast<size_t>(ray) * Sf + k] = lo;
    if (o_all) row[Sc + k] = smp;
  }
  if (o_all == nullptr) return;
  for (int i = lane; i < Sc; i += 32) row[i] = zsrc[i];
  __syncwarp();
  // Deterministic sampling (u = linspace, Trainer.py:651-672 with perturb == 0) gives non-decreasing samples, and the coarse
  // depths are monotone: sort(cat(z_coarse, z_samples)) is then a MERGE of two sorted runs -- every element finds its rank
  // with one binary search over the other run (coarse before equal samples).  ~500 instructions per ray instead of the
  // ~3,500 of the bitonic network below, which remains for random u, unsorted inputs and NaNs (any failed <= sends us there).
  {
    bool sorted = true;
    for (int i = lane; i + 1 < Sc; i += 32) sorted = sorted && (row[i] <= row[i + 1]);
    for (int k = lane; k + 1 < Sf; k += 32) sorted = sorted && (row[Sc + k] <= row[Sc + k + 1]);
    if (__all_sync(0xffffffffu, sorted)) {
      float* out = row + P;
      const float* smp = row + Sc;
      for (int i = lane; i < Sc; i += 32) {
        const float v = row[i];
        int lo = 0, hi = Sf;   // number of samples < v
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (smp[mid] < v) lo = mid + 1;
          else hi = mid;
        }
        out[i + lo] = v;
      }
      for (int k = lane; k < Sf; k += 32) {
        const float v = smp[k];
        int lo = 0, hi = Sc;   // number of coarse depths <= v
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (row[mid] <= v) lo = mid + 1;
          else hi = mid;
        }
        out[k + lo] = v;
      }
      __syncwarp();
      for (int i = lane; i < Sc + Sf; i += 32) o_all[static_cast<size_t>(ray) * (Sc + Sf) + i] = out[i];
      return;
    }
  }
  for (int i = Sc + Sf + lane; i < P; i += 32) row[i] = __int_as_float(0x7f800000);
  __syncwarp();
  for (int k = 2; k <= P; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = lane; i < P; i += 32) {
        const int l = i ^ j;
        if (l > i) {
          const float a = row[i], b = row[l];
          const bool up = (i & k) == 0;
          const bool a_gt_b = (a != a) ? !(b != b) : (!(b != b) && a > b);  // NaN sorts last, like torch.sort
          if (a_gt_b == up) {
            row[i] = b;
            row[l] = a;
          }
        }
      }
      __syncwarp();
    }
  for (int i = lane; i < Sc + Sf; i += 32) o_all[static_cast<size_t>(ray) * (Sc + Sf) + i] = row[i];
}

static int launch_sample_pdf(bool from_coarse, const float* a, const float* w, const float* u, int u_per_ray, int n_rays, int B,
                             int Sf, float* o_samples, long long* o_inds, float* o_all, cudaStream_t st) {
  int P = 1;
  while (P < B + 1 + Sf) P <<= 1;
  const int wpb = 4;
  const size_t smem = static_cast<size_t>(wpb) * (2 * B + P + B + 1 + Sf) * sizeof(float);
  if (smem > 48 * 1024) return fail("sample_pdf: row too long (B=%d, Sf=%d)", B, Sf);
  const unsigned grid = (n_rays + wpb - 1) / wpb;
  if (from_coarse)
    sample_pdf_kernel<true><<<grid, wpb * 32, smem, st>>>(a, w, u, u_per_ray, n_rays, B, Sf, P, o_samples, o_inds, o_all);
  else
    sample_pdf_kernel<false><<<grid, wpb * 32, smem, st>>>(a, w, u, u_per_ray, n_rays, B, Sf, P, o_samples, o_inds, o_all);
  LAUNCH_CHECK();
  return 0;
}

extern "C" int b200nerf_sample_pdf(const float* bins, const float* weights, const float* u, int u_per_ray, int n_rays, int n_bins,
                                   int n_samples, float* out_samples, long long* out_inds, void* stream) {
  if (n_rays < 0 || n_bins < 2 || n_samples < 1) return fail("b200nerf_sample_pdf: bad sizes");
  if (n_rays == 0) return 0;
  if (!bins || !weights || !u || !out_samples) return fail("b200nerf_sample_pdf: null argument");
  return launch_sample_pdf(false, bins, weights, u, u_per_ray, n_rays, n_bins, n_samples, out_samples, out_inds, nullptr,
                           static_cast<cudaStream_t>(stream));
}

extern "C" int b200nerf_sample_pdf_merge(const float* z_coarse, const float* weights, const float* u, int u_per_ray, int n_rays,
                                         int n_coarse, int n_importance, float* out_samples, long long* out_inds, float* out_z_all,
                                         void* stream) {
  if (n_rays < 0 || n_coarse < 3 || n_importance < 1) return fail("b200nerf_sample_pdf_merge: bad sizes");
  if (n_rays == 0) return 0;
  if (!z_coarse || !weights || !u || !out_z_all) return fail("b200nerf_sample_pdf_merge: null argument");
  return launch_sample_pdf(true, z_coarse, weights, u, u_per_ray, n_rays, n_coarse - 1, n_importance, out_samples, out_inds,
                           out_z_all, static_cast<cudaStream_t>(stream));
}

// ------------------------------------------------------------------------------------------- arg-max extraction
// top = weights.argmax(1) (first maximum), then gather z / weight / sigmoid(rgb) -- nerf_utils.py:689-690, :806-812.
__global__ void argmax_gather_kernel(const float* __restrict__ w, const float* __restrict__ z, const float* __restrict__ raw,
                                     int n_rays, int S, long long* __restrict__ o_idx, float* __restrict__ o_z,
                                     float* __restrict__ o_w, float* __restrict__ o_rgb) {
  const int ray = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (ray >= n_rays) return;
  const float* wr = w + static_cast<size_t>(ray) * S;
  float best = -__int_as_float(0x7f800000);
  int bi = 0x7fffffff;
  bool best_nan = false;
  for (int i = lane; i < S; i += 32) {
    const float v = wr[i];
    const bool vn = v != v;  // torch.argmax treats NaN as the maximum
    if ((vn && !best_nan) || (!best_nan && (v > best || (bi == 0x7fffffff)))) {
      best = v;
      bi = i;
      best_nan = vn;
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, off);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
    const bool on = ov != ov;
    const bool take = oi != 0x7fffffff &&
                      (bi == 0x7fffffff || (on && !best_nan) || (on == best_nan && (on ? oi < bi : (ov > best || (ov == best && oi < bi)))));
    if (take) {
      best = ov;
      bi = oi;
      best_nan = on;
    }
  }
  if (lane == 0) {
    const size_t p = static_cast<size_t>(ray) * S + bi;
    if (o_idx) o_idx[ray] = bi;
    if (o_z) o_z[ray] = z[p];
    if (o_w) o_w[ray] = best;
    if (o_rgb && raw) {
      const float4 r = reinterpret_cast<const float4*>(raw)[p];
      o_rgb[ray * 3] = 1.0f / (1.0f + expf(-r.x));
      o_rgb[ray * 3 + 1] = 1.0f / (1.0f + expf(-r.y));
      o_rgb[ray * 3 + 2] = 1.0f / (1.0f + expf(-r.z));
    }
  }
}

extern "C" int b200nerf_argmax_gather(const float* weights, const float* z, const float* raw, int n_rays, int S, long long* out_idx,
                                      float* out_z, float* out_w, float* out_rgb, void* stream) {
  if (n_rays < 0 || S < 1) return fail("b200nerf_argmax_gather: bad sizes");
  if (n_rays == 0) return 0;
  if (!weights || !z) return fail("b200nerf_argmax_gather: null argument");
  const int wpb = 8;
  argmax_gather_kernel<<<(n_rays + wpb - 1) / wpb, wpb * 32, 0, static_cast<cudaStream_t>(stream)>>>(weights, z, raw, n_rays, S,
                                                                                               out_idx, out_z, out_w, out_rgb);
  LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------- placement / points backward
// sample_points_around_mean (nerf_pytorch/utils.py:220-244) under autograd.  Every placed depth is mean + a constant (the sort only
// permutes them), so d/d mean is the sum of the S upstream gradients.  Uniform mode clips: torch.clamp passes the gradient where
// lo <= x <= hi (inclusive) for the UNclipped value x = mean + offset, which is rebuilt here with the forward's rule and rounding
// (place_uniform_kernel, b200nerf.cu).  One warp per ray.
__global__ void place_bwd_kernel(const float* __restrict__ mean, const float* __restrict__ grid, int n_rays, int S, int clip, float lo,
                                 float hi, const float* __restrict__ g_z, float* __restrict__ g_mean) {
  const int ray = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (ray >= n_rays) return;
  const float m = clip ? __ldg(mean + ray) : 0.f;
  float acc = 0.f;
  for (int s = lane; s < S; s += 32) {
    const float g = __ldg(g_z + static_cast<size_t>(ray) * S + s);
    if (clip) {
      float x = m;
      if (s <= S - 2 && __ldg(grid + s) < 0.f) x = __fadd_rn(m, __ldg(grid + s));
      else if (s >= 1 && !(__ldg(grid + s - 1) < 0.f)) x = __fadd_rn(m, __ldg(grid + s - 1));
      if (!(x >= lo && x <= hi)) continue;
    }
    acc += g;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
  if (lane == 0) g_mean[ray] = acc;
}

extern "C" int b200nerf_place_samples_bwd(const float* mean, const float* offsets, int n_rays, int S, int mode, float clip_lo,
                                          float clip_hi, const float* g_z, float* out_g_mean, void* stream) {
  if (n_rays < 0 || S < 1) return b200_fail("b200nerf_place_samples_bwd: bad sizes n_rays=%d S=%d", n_rays, S);
  if (mode != B200NERF_PLACE_DEPTH_ONLY && mode != B200NERF_PLACE_UNIFORM && mode != B200NERF_PLACE_GAUSSIAN)
    return b200_fail("b200nerf_place_samples_bwd: unknown mode %d", mode);
  if (mode == B200NERF_PLACE_DEPTH_ONLY && S != 1) return b200_fail("b200nerf_place_samples_bwd: depth_only needs S == 1");
  if (n_rays == 0) return 0;
  if (!mean || !g_z || !out_g_mean) return b200_fail("b200nerf_place_samples_bwd: null argument");
  const bool clip = mode == B200NERF_PLACE_UNIFORM;
  if (clip && S > 1 && !offsets) return b200_fail("b200nerf_place_samples_bwd: offsets is null (uniform mode needs the grid)");
  const int wpb = 8;
  place_bwd_kernel<<<(n_rays + wpb - 1) / wpb, wpb * 32, 0, static_cast<cudaStream_t>(stream)>>>(mean, offsets, n_rays, S, clip ? 1 : 0,
                                                                                             clip_lo, clip_hi, g_z, out_g_mean);
  LAUNCH_CHECK();
  return 0;
}

// pts = rays_o + rays_d z (b200nerf_points) backward: g_z = sum_k g_pts[k] rays_d[k]
__global__ void points_bwd_kernel(const float* __restrict__ rd, const float* __restrict__ g_pts, size_t total, int S,
                                  float* __restrict__ g_z) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const size_t ray = i / S;
  const float* g = g_pts + i * 3;
  g_z[i] = __fadd_rn(__fadd_rn(__fmul_rn(__ldg(g), __ldg(rd + ray * 3)), __fmul_rn(__ldg(g + 1), __ldg(rd + ray * 3 + 1))),
                     __fmul_rn(__ldg(g + 2), __ldg(rd + ray * 3 + 2)));
}

extern "C" int b200nerf_points_bwd(const float* rays_d, const float* g_pts, int n_rays, int S, float* out_g_z, void* stream) {
  if (n_rays < 0 || S < 1) return b200_fail("b200nerf_points_bwd: bad sizes n_rays=%d S=%d", n_rays, S);
  const size_t total = static_cast<size_t>(n_rays) * S;
  if (total == 0) return 0;
  if (!rays_d || !g_pts || !out_g_z) return b200_fail("b200nerf_points_bwd: null argument");
  points_bwd_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(rays_d, g_pts, total, S,
                                                                                                          out_g_z);
  LAUNCH_CHECK();
  return 0;
}
