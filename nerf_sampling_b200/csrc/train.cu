// Differentiable slice of the training render (config #5: Trainer.core_optimization_loop, trainers/Trainer.py:506-544
// over nerf_utils.render_rays, nerf_pytorch/nerf_utils.py:614-733), in fp32:
//
//   * DepthNet in its literal per-layer form (depth_nets/depth_net.py:117-169) with saved activations, and its
//     backward (input gradient chain + all 82 weight/bias gradients);
//   * the frozen fine NeRF evaluated at ONE sample per ray together with its directional derivative d raw / d z
//     (forward-mode: z is a scalar per ray, so a tangent row next to every primal row replaces a backward pass);
//   * Adam on a list of tensors.
//
// The frozen hierarchical target (257 network evaluations per ray) stays on the tensor-core kernels; this part is
// 512 rays per GPU and two evaluations per ray, i.e. latency- not throughput-bound, and fp32 CUDA-core GEMMs keep the
// gradients at the reference's own precision.  Host loops over layers live here, behind one C call per pass.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../include/b200nerf.h"
#include "host_common.h"
#include "tgemm.cuh"
#include "tgemm_reg.cuh"

// ------------------------------------------------------------------------------------------- strided SGEMM
// C[M,N] (row-major, ldc) = (beta ? C : 0) + sum_k A(m,k) * B(k,n) [+ bias[n]] [then LeakyReLU(slope) if act]
// A(m,k) = A[m*sAm + k*sAk], B(k,n) = B[k*sBk + n*sBn]: covers X*W^T (forward), dY*W (input gradient) and dY^T*X
// (weight gradient) without transposes.  64x64x16 tiles, 256 threads, 4x4 outputs per thread.  gridDim.z > 1 splits
// the K range (the weight gradients reduce over thousands of rays into a 256 x ~300 output: without the split only
// ~20 CTAs would run); the partial sums are then added atomically into a zeroed C.
constexpr int GM = 64, GN = 64, GK = 16;

__global__ void __launch_bounds__(256) sgemm_kernel(int M, int N, int K, const float* __restrict__ A, long sAm, long sAk,
                                                    const float* __restrict__ B, long sBk, long sBn, float* __restrict__ C,
                                                    int ldc, int beta, const float* __restrict__ bias, int act, float slope) {
  __shared__ float As[GK][GM + 4];
  __shared__ float Bs[GK][GN + 4];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.y * GM, n0 = blockIdx.x * GN;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  // element (r, c) of a 64 x 16 tile per thread and pass: walk the contiguous dimension with consecutive threads
  const bool a_kfast = sAk == 1, b_nfast = sBn == 1;
  const int k_per = ((K + gridDim.z - 1) / gridDim.z + GK - 1) / GK * GK;
  const int k_begin = blockIdx.z * k_per;
  const int k_end = min(K, k_begin + k_per);
  const bool split = gridDim.z > 1;
  for (int k0 = k_begin; k0 < k_end; k0 += GK) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int idx = tid + e * 256;
      int m, k;
      if (a_kfast) { m = idx >> 4; k = idx & 15; } else { m = idx & 63; k = idx >> 6; }
      const int gm = m0 + m, gk = k0 + k;
      As[k][m] = (gm < M && gk < k_end) ? __ldg(A + gm * sAm + gk * sAk) : 0.f;
      int n, kb;
      if (b_nfast) { n = idx & 63; kb = idx >> 6; } else { n = idx >> 4; kb = idx & 15; }
      const int gn = n0 + n, gkb = k0 + kb;
      Bs[kb][n] = (gn < N && gkb < k_end) ? __ldg(B + gkb * sBk + gn * sBn) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < GK; ++k) {
      const float4 a4 = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 b4 = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int gm = m0 + ty * 4 + i;
    if (gm >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gn = n0 + tx * 4 + j;
      if (gn >= N) continue;
      float v = acc[i][j];
      float* c = C + static_cast<size_t>(gm) * ldc + gn;
      if (split) {
        if (bias && blockIdx.z == 0) v += __ldg(bias + gn);
        atomicAdd(c, v);
        continue;
      }
      if (beta) v += *c;
      if (bias) v += __ldg(bias + gn);
      if (act) v = v > 0.f ? v : v * slope;
      *c = v;
    }
  }
}

// The tensor-core path (tgemm.cuh: 3xTF32 on tcgen05).  B200NERF_TRAIN_GEMM=fp32 keeps every product on the CUDA-core
// kernel above (A/B measurements, and the reference point of the precision tests).
static bool tgemm_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("B200NERF_TRAIN_GEMM");
    v = (e && strcmp(e, "fp32") == 0) ? 0 : 1;
  }
  return v == 1;
}
// ---- grouped / K-segmented problems for tgemm_kernel ----------------------------------------------------------
struct GemmSeg {
  const float* A; long sAm, sAk;
  const float* B; long sBk, sBn;
  int K;
};
struct GemmProb {
  int M = 0, N = 0, nseg = 0;
  GemmSeg seg[b200::tg::MAX_SEG];
  float* C = nullptr;
  int ldc = 0, beta = 0;
  const float* bias = nullptr;
  int act = 0;
  float slope = 0.f;
  float* colsum = nullptr;       // += column sums of A^T, i.e. sum_k A(m,k) (bias gradient); target pre-zeroed
  const float* dact = nullptr;   // epilogue *= LeakyReLU'(dact)
  int ld_dact = 0;
  const float* kscale = nullptr; // A(m,k) *= kscale[k]: the per-ray factor dz_r of a weight gradient built from a unit-upstream Jacobian
  bool c_zeroed = false;         // C is known to be zero: a split-K launch needs no memset
  int force_splits = 0;          // > 0: this many K slices, partial sums added atomically (no bias / activation then)
  void add(const float* A, long sAm, long sAk, const float* B, long sBk, long sBn, int K) {
    seg[nseg++] = GemmSeg{A, sAm, sAk, B, sBk, sBn, K};
  }
};
// Y[n, M] = sum of X_s[n, K_s] * W[:, off_s : off_s+K_s]^T segments (+ bias) (+ LeakyReLU)
static GemmProb prob_fwd(int n, int M, float* Y, int ldy, const float* bias, int act, float slope) {
  GemmProb q;
  q.M = n; q.N = M; q.C = Y; q.ldc = ldy; q.bias = bias; q.act = act; q.slope = slope;
  return q;
}
static void seg_fwd(GemmProb& q, const float* X, int ldx, const float* W, int ldw, int off, int K) { q.add(X, ldx, 1, W + off, 1, ldw, K); }
// dX[n, K] = dY[n, M] * W[:, off:off+K]   (optionally * LeakyReLU'(post))
static GemmProb prob_dgrad(int n, int M, int K, const float* dY, int ldy, const float* W, int ldw, int off, float* dX, int ldx,
                           const float* post = nullptr, int ld_post = 0, float slope = 0.f) {
  GemmProb q;
  q.M = n; q.N = K; q.C = dX; q.ldc = ldx; q.dact = post; q.ld_dact = ld_post; q.slope = slope;
  q.add(dY, ldy, 1, W + off, ldw, 1, M);
  return q;
}
// dW[:, off:off+K] = dY[n, M]^T * X[n, K]   (+ db[m] = sum_n dY[n, m] when db != nullptr)
static GemmProb prob_wgrad(int n, int M, int K, const float* dY, int ldy, const float* X, int ldx, float* dW, int ldw, int off,
                           float* db, bool zeroed) {
  GemmProb q;
  q.M = M; q.N = K; q.C = dW + off; q.ldc = ldw; q.colsum = db; q.c_zeroed = zeroed;
  q.add(dY, 1, ldy, X, ldx, 1, n);
  return q;
}

static long long* g_tgemm_dbg = nullptr;
/* diagnostics: device buffer of 16 int64; CTA 0 of every grouped-GEMM launch writes its phase time stamps (ns) there */
extern "C" void b200nerf_debug_set_tgemm_timeline(long long* dev_buf) { g_tgemm_dbg = dev_buf; }
static int tgemm_group(cudaStream_t st, const GemmProb* probs, int nprob) {
  namespace tg = b200::tg;
  static int sm_counts[B200_MAX_DEVICES] = {0};
  const int dev = b200_device();
  if (dev < 0) return b200_fail("tgemm_group: no usable CUDA device");
  if (sm_counts[dev] == 0) {
    CUDA_TRY(cudaFuncSetAttribute(tg::tgemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tg::SMEM_BYTES));
    CUDA_TRY(cudaFuncSetAttribute(b200::tgr::tgemm_reg_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, b200::tgr::SMEM_BYTES));
    CUDA_TRY(cudaDeviceGetAttribute(&sm_counts[dev], cudaDevAttrMultiProcessorCount, dev));
  }
  const int g_sm_count = sm_counts[dev];
  if (nprob < 1 || nprob > tg::MAX_PROB) return b200_fail("tgemm_group: %d problems", nprob);
  tg::Group g;
  memset(&g, 0, sizeof(g));
  g.nprob = nprob;
  g.dbg = g_tgemm_dbg;
  for (int i = 0; i < nprob; ++i) {
    const GemmProb& q = probs[i];
    if (q.nseg < 1 || q.nseg > tg::MAX_SEG || q.M < 1 || q.N < 1) return b200_fail("tgemm_group: bad problem %d", i);
  }
  int cta = 0;
  for (int i = 0; i < nprob; ++i) {
    const GemmProb& q = probs[i];
    tg::Prob& P = g.prob[i];
    for (int s = 0; s < q.nseg; ++s) {
      const GemmSeg& a = q.seg[s];
      tg::Seg& S = P.seg[s];
      S.A = a.A; S.B = a.B; S.sAm = a.sAm; S.sAk = a.sAk; S.sBk = a.sBk; S.sBn = a.sBn; S.K = a.K;
      S.vecA = a.sAk == 1 && (a.sAm & 3) == 0 && (reinterpret_cast<uintptr_t>(a.A) & 15) == 0;
      S.vecB = a.sBk == 1 && (a.sBn & 3) == 0 && (reinterpret_cast<uintptr_t>(a.B) & 15) == 0;
    }
    if (q.colsum && q.seg[0].sAk == 1) return b200_fail("tgemm_group: colsum needs a k-strided A");
    P.C = q.C; P.bias = q.bias; P.colsum = q.colsum; P.dact = q.dact; P.kscale = q.kscale;
    if (q.kscale && q.nseg != 1) return b200_fail("tgemm_group: kscale needs a single K segment");
    P.M = q.M; P.N = q.N; P.nseg = q.nseg; P.ldc = q.ldc; P.beta = q.beta; P.act = q.act; P.ld_dact = q.ld_dact; P.slope = q.slope;
    P.tiles_x = (q.N + tg::BN - 1) / tg::BN;
    P.tiles_y = (q.M + tg::BM - 1) / tg::BM;
    int splits = 1;
    const int K0 = q.seg[0].K;
    if (q.force_splits > 0) {
      if (q.nseg != 1 || q.act || q.dact || q.bias) return b200_fail("tgemm_group: force_splits needs one K segment and a plain epilogue");
      splits = q.force_splits;
    } else if (q.nseg == 1 && !q.act && !q.dact && K0 >= 512) {
      // a long reduction into a small output: ~8 chunks per CTA like the CTAs of the other problems of the group -- a CTA that walks
      // the whole reduction would be the launch's tail.  (Measured for the split backward's group of 16 weight gradients, 136 tiles
      // of 128 chunks: ONE wave of unsplit CTAs with plain stores is no faster than 2,176 CTAs of 8 chunks with atomics, 1.651 vs
      // 1.644 ms per 4096-ray step -- the launch is bound by the strided operand reads, not by the per-CTA fixed cost.)
      splits = K0 / 256;
      const int own_tiles = P.tiles_x * P.tiles_y;
      while (splits > 1 && own_tiles * splits > 4 * g_sm_count) splits >>= 1;
    }
    int k_per = (K0 + splits - 1) / splits;
    k_per = (k_per + tg::KC - 1) / tg::KC * tg::KC;
    splits = (K0 + k_per - 1) / k_per;
    P.splits = splits;
    P.k_per = k_per;
    P.cta_begin = cta;
    cta += P.tiles_x * P.tiles_y * splits;
    if (splits > 1 && !q.beta && !q.c_zeroed)
      CUDA_TRY(cudaMemset2DAsync(q.C, static_cast<size_t>(q.ldc) * sizeof(float), 0, static_cast<size_t>(q.N) * sizeof(float), q.M, st));
  }
  {
    // programmatic stream serialization: this launch may start its prologue while the previous kernel of the stream drains
    // (tgemm_kernel executes griddepcontrol.wait before it reads global memory); B200NERF_PDL=0 turns it off for A/B runs
    static int pdl = -1;
    if (pdl < 0) {
      const char* e = getenv("B200NERF_PDL");
      pdl = (e && e[0] == '0') ? 0 : 1;
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    // single-wave launches: the staged kernel (one CTA per SM, operands three chunks ahead); launches of many waves: the register
    // form, two CTAs per SM (tgemm_reg.cuh).  B200NERF_TGEMM=staged / reg forces one of them (A/B measurements).
    static int form = -1;
    if (form < 0) {
      const char* e = getenv("B200NERF_TGEMM");
      form = (e && strcmp(e, "staged") == 0) ? 1 : ((e && strcmp(e, "reg") == 0) ? 2 : 0);
    }
    const bool reg_form = form == 2 || (form == 0 && cta > 2 * g_sm_count);
    cfg.gridDim = dim3(cta);
    cfg.blockDim = dim3(tg::CTA_THREADS);
    cfg.dynamicSmemBytes = reg_form ? b200::tgr::SMEM_BYTES : tg::SMEM_BYTES;
    cfg.stream = st;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    if (reg_form) CUDA_TRY(cudaLaunchKernelEx(&cfg, b200::tgr::tgemm_reg_kernel, g));
    else CUDA_TRY(cudaLaunchKernelEx(&cfg, tg::tgemm_kernel, g));
  }
  LAUNCH_CHECK();
  return 0;
}
static int tgemm(cudaStream_t st, int M, int N, int K, const float* A, long sAm, long sAk, const float* B, long sBk, long sBn,
                 float* C, int ldc, int beta, const float* bias, int act, float slope) {
  GemmProb q;
  q.M = M; q.N = N; q.C = C; q.ldc = ldc; q.beta = beta; q.bias = bias; q.act = act; q.slope = slope;
  q.add(A, sAm, sAk, B, sBk, sBn, K);
  return tgemm_group(st, &q, 1);
}

static int sgemm(cudaStream_t st, int M, int N, int K, const float* A, long sAm, long sAk, const float* B, long sBk, long sBn,
                 float* C, int ldc, int beta, const float* bias = nullptr, int act = 0, float slope = 0.f) {
  if (M <= 0 || N <= 0) return 0;
  if (tgemm_enabled() && M >= 32 && N >= 8 && K >= 8) return tgemm(st, M, N, K, A, sAm, sAk, B, sBk, sBn, C, ldc, beta, bias, act, slope);
  dim3 grid((N + GN - 1) / GN, (M + GM - 1) / GM);
  const int blocks = static_cast<int>(grid.x * grid.y);
  if (!act && blocks < 120 && K >= 512) {
    int splits = (296 + blocks - 1) / blocks;
    const int max_splits = K / 128;
    if (splits > max_splits) splits = max_splits;
    if (splits > 1) {
      grid.z = splits;
      if (!beta) CUDA_TRY(cudaMemset2DAsync(C, static_cast<size_t>(ldc) * sizeof(float), 0, static_cast<size_t>(N) * sizeof(float), M, st));
    }
  }
  sgemm_kernel<<<grid, 256, 0, st>>>(M, N, K, A, sAm, sAk, B, sBk, sBn, C, ldc, beta, bias, act, slope);
  LAUNCH_CHECK();
  return 0;
}
// Y[n, M] (+)= X[n, K] * W[:, off:off+K]^T (+ bias) (+ LeakyReLU)       W is [M, ldw] row-major
static int lin_fwd(cudaStream_t st, int n, int M, int K, const float* X, int ldx, const float* W, int ldw, int off, float* Y,
                   int ldy, int beta, const float* bias, int act, float slope) {
  return sgemm(st, n, M, K, X, ldx, 1, W + off, 1, ldw, Y, ldy, beta, bias, act, slope);
}
// dX[n, K] (+)= dY[n, M] * W[:, off:off+K]
static int lin_dgrad(cudaStream_t st, int n, int M, int K, const float* dY, int ldy, const float* W, int ldw, int off, float* dX,
                     int ldx, int beta) {
  return sgemm(st, n, K, M, dY, ldy, 1, W + off, ldw, 1, dX, ldx, beta);
}
// dW[:, off:off+K] = dY[n, M]^T * X[n, K]
static int lin_wgrad(cudaStream_t st, int n, int M, int K, const float* dY, int ldy, const float* X, int ldx, float* dW, int ldw,
                     int off) {
  return sgemm(st, M, K, n, dY, 1, ldy, X, ldx, 1, dW + off, ldw, 0);
}

// db[m] = sum_n dY[n, m]: 32 columns x 256 rows per block, partial sums added atomically into a zeroed db
__global__ void colsum_kernel(const float* __restrict__ dY, int n, int M, int ldy, float* __restrict__ db) {
  const int m = blockIdx.x * 32 + (threadIdx.x & 31);
  const int part = threadIdx.x >> 5;  // 8 row groups
  __shared__ float red[8][33];
  const int r0 = blockIdx.y * 256, r1 = min(n, r0 + 256);
  float s = 0.f;
  if (m < M)
    for (int r = r0 + part; r < r1; r += 8) s += dY[static_cast<size_t>(r) * ldy + m];
  red[part][threadIdx.x & 31] = s;
  __syncthreads();
  if (part == 0 && m < M) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += red[i][threadIdx.x];
    atomicAdd(db + m, t);
  }
}
static int colsum(cudaStream_t st, const float* dY, int n, int M, int ldy, float* db) {
  CUDA_TRY(cudaMemsetAsync(db, 0, static_cast<size_t>(M) * sizeof(float), st));
  colsum_kernel<<<dim3((M + 31) / 32, (n + 255) / 256), 256, 0, st>>>(dY, n, M, ldy, db);
  LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------- encodings
// gamma(x) of a C-vector: [x, sin(2^0 x), cos(2^0 x), ...] (run_nerf_helpers.py:15-63), C*(1+2F) wide, F = multires
// E[n, 4 d3] = [gamma(o) d3 | gamma(d) d3 | gamma([hit_near, hit_far]) 2 d3], d3 = 3 (1 + 2F); sphere hits in the reference's op order
// (nerf_pytorch/utils.py:159-217), NaN when the ray misses.  Twelve threads per ray -- (vector o / d / hit_near / hit_far) x channel --
// so that a thread runs F accurate sincosf instead of 12 F in a row (the kernel is latency-, not throughput-bound: 4096 rays).
__global__ void depthnet_encode_kernel(const float* __restrict__ ro, const float* __restrict__ rd, int n, float radius, int nf,
                                       float* __restrict__ E) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = t / 12, part = (t % 12) / 3, c = t % 3;
  if (i >= n) return;
  float o[3], d[3];
  for (int k = 0; k < 3; ++k) {
    o[k] = ro[i * 3 + k];
    d[k] = rd[i * 3 + k];
  }
  float x;
  if (part == 0) {
    x = o[c];
  } else if (part == 1) {
    x = d[c];
  } else {
    const float dot_do = __fadd_rn(__fadd_rn(__fmul_rn(d[0], o[0]), __fmul_rn(d[1], o[1])), __fmul_rn(d[2], o[2]));
    const float b = __fmul_rn(2.f, dot_do);
    const float on = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(o[0], o[0]), __fmul_rn(o[1], o[1])), __fmul_rn(o[2], o[2])));
    const float cc = __fadd_rn(__fmul_rn(on, on), -__fmul_rn(radius, radius));
    const float a = __fadd_rn(__fadd_rn(__fmul_rn(d[0], d[0]), __fmul_rn(d[1], d[1])), __fmul_rn(d[2], d[2]));
    const float delta = __fadd_rn(__fmul_rn(b, b), -__fmul_rn(__fmul_rn(4.f, a), cc));
    const float sq = __fsqrt_rn(delta);
    const float two_a = __fmul_rn(2.f, a);
    const float tt = part == 2 ? __fdiv_rn(__fadd_rn(-b, -sq), two_a) : __fdiv_rn(__fadd_rn(-b, sq), two_a);
    x = __fadd_rn(o[c], __fmul_rn(tt, d[c]));
  }
  // gamma of a C-vector is [x (C), sin(2^0 x) (C), cos(2^0 x) (C), ...]: o and d are 3-vectors, the two hit points one 6-vector
  const int C = part < 2 ? 3 : 6;
  const int ch = part < 2 ? c : (part - 2) * 3 + c;
  const int d3 = 3 * (1 + 2 * nf);
  float* e = E + static_cast<size_t>(i) * (4 * d3) + (part == 0 ? 0 : (part == 1 ? d3 : 2 * d3));
  e[ch] = x;
  for (int j = 0; j < nf; ++j) {
    float sn, cs;
    sincosf(x * static_cast<float>(1 << j), &sn, &cs);
    e[C + j * 2 * C + ch] = sn;
    e[C + j * 2 * C + C + ch] = cs;
  }
}

// z = near*(1-s) + far*s, s = sigmoid(t)   (depth_net.py:165-168)
__global__ void depth_head_kernel(const float* __restrict__ t, int n, float near_, float far_, float* __restrict__ s_out,
                                  float* __restrict__ z) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float s = 1.0f / (1.0f + expf(-t[i]));
  s_out[i] = s;
  z[i] = __fadd_rn(__fmul_rn(near_, __fadd_rn(1.0f, -s)), __fmul_rn(far_, s));
}
// dt = dz * (far - near) * s * (1 - s)
__global__ void depth_head_bwd_kernel(const float* __restrict__ dz, const float* __restrict__ s, int n, float near_, float far_,
                                      float* __restrict__ dt) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  dt[i] = dz[i] * (far_ - near_) * s[i] * (1.0f - s[i]);
}
// Fused head (tensor-core path): t = a_last . w + b, s = sigmoid(t), z = near (1 - s) + far s; one warp per ray
__global__ void depth_head_fused_kernel(const float* __restrict__ a, int n, int cl, const float* __restrict__ w, const float* __restrict__ b,
                                        float near_, float far_, float* __restrict__ s_out, float* __restrict__ z) {
  const int ray = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (ray >= n) return;
  const float* row = a + static_cast<size_t>(ray) * cl;
  float acc = 0.f;
  for (int c = lane; c < cl; c += 32) acc = fmaf(row[c], __ldg(w + c), acc);
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
  if (lane == 0) {
    const float s = 1.0f / (1.0f + expf(-(acc + __ldg(b))));
    s_out[ray] = s;
    z[ray] = __fadd_rn(__fmul_rn(near_, __fadd_rn(1.0f, -s)), __fmul_rn(far_, s));
  }
}
// Its backward in one pass over a_last: dt = dz (far - near) s (1 - s);  g[r, c] = dt w[c] LeakyReLU'(a_last[r, c]) (the gradient of
// the last cat layer's pre-activation);  dw[c] += sum_r dt a_last[r, c];  db += sum_r dt  (dw / db pre-zeroed).  dz == nullptr: unit
// upstream gradient (the Jacobian pass); g / dw / db == nullptr: that output is skipped.
constexpr int HEAD_ROWS = 32;
__global__ void __launch_bounds__(256) depth_head_bwd_fused_kernel(const float* __restrict__ dz, const float* __restrict__ s,
                                                                   const float* __restrict__ a, const float* __restrict__ w, int n, int cl,
                                                                   float near_, float far_, float slope, float* __restrict__ g,
                                                                   float* __restrict__ dw, float* __restrict__ db) {
  __shared__ float dts[HEAD_ROWS];
  const int r0 = blockIdx.x * HEAD_ROWS;
  if (threadIdx.x < HEAD_ROWS) {
    const int r = r0 + threadIdx.x;
    dts[threadIdx.x] = r < n ? (dz ? dz[r] : 1.0f) * (far_ - near_) * s[r] * (1.0f - s[r]) : 0.f;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < cl; c += blockDim.x) {
    const float wc = __ldg(w + c);
    float acc = 0.f;
#pragma unroll 8
    for (int q = 0; q < HEAD_ROWS; ++q) {
      const int r = r0 + q;
      if (r >= n) break;
      const float av = a[static_cast<size_t>(r) * cl + c];
      if (g) g[static_cast<size_t>(r) * cl + c] = dts[q] * wc * (av > 0.f ? 1.0f : slope);
      acc = fmaf(dts[q], av, acc);
    }
    if (dw) atomicAdd(dw + c, acc);
  }
  if (threadIdx.x == 0 && db) {
    float t = 0.f;
    for (int q = 0; q < HEAD_ROWS; ++q) t += dts[q];
    atomicAdd(db, t);
  }
}

// dpre = dpost * (post > 0 ? 1 : slope), in place
__global__ void leaky_bwd_kernel(float* __restrict__ d, const float* __restrict__ post, size_t total, float slope) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= total) return;
  if (!(post[i] > 0.f)) d[i] *= slope;
}

// ------------------------------------------------------------------------------------------- DepthNet branches, collapsed
// The origin / direction / intersection branches have NO activation (depth_net.py:140,148,156 construct a LeakyReLU module
// and drop it): x_i = W_i [x_{i-1}; e] + b_i = U_i x_{i-1} + V_i e + b_i is affine in the ray's encoding e, x_i = A_i e + c_i with
//   A_0 = U_0 + V_0, c_0 = b_0,   A_i = U_i A_{i-1} + V_i,   c_i = U_i c_{i-1} + b_i                    (weights only, no ray dimension).
// Forward per ray: ONE product x_last = e A_last^T + c_last instead of L.  Backward, with D = dLoss/dx_last [n, h] per ray:
//   dLoss/dx_i = D Q_i, Q_i = U_{L-1} ... U_{i+1};   G = D^T e [h, d], g = D^T 1 [h]      (ONE reduction over the rays)
//   R_i = Q_i^T [G | g] (R_{L-1} = [G | g], R_{i-1} = U_i^T R_i):   dV_i = R_i[:, :d],  db_i = R_i[:, d],
//   dU_i = dx_i^T x_{i-1} = R_i[:, :d] A_{i-1}^T + R_i[:, d] c_{i-1}^T = R_i [A_{i-1} | c_{i-1}]^T        (dU_0 = R_0[:, :d]).
// 30 per-ray layers of forward and 60 per-ray products of backward (72 % of DepthNet's training FLOPs) become two per-ray
// products, two weight-only recurrences and 27 small [h, d+1] x [d+1, h] products.  The recurrences run in plain fp32 FMA
// (they are tiny and 10 deep: fp32-grade gradients need fp32-grade chain products); their COLUMNS are independent, so a
// CTA owns CH_CW columns of [A_i | c_i] (or R_i) through the whole chain and never talks to another CTA.
constexpr int CH_CW = 4;        // columns per CTA
constexpr int CH_MAXL = 12;     // layers per branch
constexpr int CH_LD = 128;      // row stride of the [h, d+1] chain matrices (d + 1 <= 127)
constexpr int CH_MAXH = 256;    // widths up to 256: one thread per row
struct ChainBranch {
  const float* W[CH_MAXL];
  const float* b[CH_MAXL];
  float* gW[CH_MAXL];
  float* gb[CH_MAXL];
  int h[CH_MAXL];
  int d;              // encoding width (d3 / d3 / 2 d3: 63 / 63 / 126 at multires 10)
  int cta_begin;      // first CTA of this branch in the launch
  float* Aaug;        // [L][CH_MAXH][CH_LD]: [A_i | c_i]
  float* Raug;        // [L][CH_MAXH][CH_LD]: R_i
  float* c_last;      // [h_last]
  const float* G;     // [h_last][CH_LD]: D^T e (columns 0..d-1)
  const float* g;     // [h_last]: D^T 1
};
struct ChainParams {
  ChainBranch br[3];
  int L;
};

__device__ __forceinline__ const ChainBranch& chain_branch(const ChainParams& p, int cta, int* local) {
  const int b = cta >= p.br[2].cta_begin ? 2 : (cta >= p.br[1].cta_begin ? 1 : 0);
  *local = cta - p.br[b].cta_begin;
  return p.br[b];
}

// Both recurrences read the whole W_i = [U_i | V_i] (h x (pw + d) fp32, ~330-390 KB) per layer and CTA.  The rows are 319 / 382
// floats apart, so no vector load is aligned -- but a block of 32 rows is one contiguous, 16-byte aligned span, i.e. one 1-D bulk
// copy (cp.async.bulk, SASS UBLKCP).  A CTA streams the blocks of ALL its layers through a 4-stage ring (the weights do not
// depend on the recurrence, so the ring never drains at a layer boundary) and computes from shared memory; what bounds a layer is
// the bulk-copy bandwidth of one SM, not 4-byte load latency (the first version: 194 / 890 us for the two kernels).
constexpr int CH_THREADS = 1024;
constexpr int CH_STAGES = 4;
constexpr int CH_ROWS = 32;                        // rows of W_i per ring stage
constexpr int CH_STAGE_BYTES = 49152;              // >= 32 x (256 + 126) x 4
constexpr int CH_PART_BYTES = 4 * CH_MAXH * CH_CW * 4;   // bwd: partial sums of the four row groups
// The rows of every layer are split over a cluster of CH_R CTAs (same columns): a CTA streams and multiplies only its CH_RPR rows of
// U_i and the slices meet in distributed shared memory once per layer -- the kernels were instruction-bound on ONE CTA per
// column group (136 / 87 us whatever the batch: the head of the forward chain and the tail of the backward of every step).
constexpr int CH_R = 2;
constexpr int CH_RPR = CH_MAXH / CH_R;
constexpr int CH_SLOT_BYTES = 2 * CH_MAXH * CH_CW * 4;          // bwd: the peer's partial sums, double-buffered by layer parity
constexpr int CH_SMEM_BYTES = CH_STAGES * CH_STAGE_BYTES + CH_PART_BYTES + CH_SLOT_BYTES + 128;
static_assert(CH_R == 2, "the kernels exchange with ONE peer");
static_assert(CH_SMEM_BYTES + 8448 <= 232448, "dynamic + static shared memory of the chain kernels");

__device__ __forceinline__ void st_cluster_f32(uint32_t cluster_addr, float v) {
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(cluster_addr), "f"(v) : "memory");
}
__device__ __forceinline__ void st_cluster_v4(uint32_t cluster_addr, float4 v) {
  asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(cluster_addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
// rows of a layer of width h that rank `rank` owns: [rank * CH_RPR, rank * CH_RPR + own)
__device__ __forceinline__ int chain_own_rows(int h, int rank) {
  const int left = h - rank * CH_RPR;
  return left < 0 ? 0 : (left < CH_RPR ? left : CH_RPR);
}

// the producer side of the ring, run by thread 0: blocks are numbered q = 0, 1, ... over the layers in visiting order
struct ChainFeed {
  int layer, block, issued;
};
template <bool FWD>
__device__ __forceinline__ void chain_feed(const ChainBranch& B, int L, int rank, ChainFeed& f, uint8_t* ring, uint64_t* full,
                                           uint64_t* empty) {
  // layers in which this rank owns no row (widths <= CH_RPR) contribute no block
  while ((FWD ? f.layer < L : f.layer >= 1) && chain_own_rows(B.h[f.layer], rank) == 0) f.layer += FWD ? 1 : -1;
  if (FWD ? f.layer >= L : f.layer < 1) return;
  const int own = chain_own_rows(B.h[f.layer], rank), ldw = B.h[f.layer - 1] + B.d;
  const int s = f.issued % CH_STAGES, use = f.issued / CH_STAGES;
  if (use > 0) b200::mbar_wait(&empty[s], static_cast<uint32_t>(use - 1) & 1u);   // every warp has read the stage's previous block
  const int r0 = f.block * CH_ROWS;
  const int rows = own - r0 < CH_ROWS ? own - r0 : CH_ROWS;
  const uint32_t bytes = static_cast<uint32_t>(rows) * ldw * 4u;
  b200::mbar_arrive_expect_tx(&full[s], bytes);
  // four 8-row copies per block: the latency of one bulk copy (~2 us for 40 KB) bounds the stream unless enough are in flight
  for (int sub = 0; sub < rows; sub += CH_ROWS / 4) {
    const int nr = rows - sub < CH_ROWS / 4 ? rows - sub : CH_ROWS / 4;
    b200::tma_load_1d(ring + static_cast<size_t>(s) * CH_STAGE_BYTES + static_cast<size_t>(sub) * ldw * 4,
                      B.W[f.layer] + static_cast<size_t>(rank * CH_RPR + r0 + sub) * ldw, static_cast<uint32_t>(nr) * ldw * 4u, &full[s]);
  }
  ++f.issued;
  if (++f.block * CH_ROWS >= own) {
    f.block = 0;
    f.layer += FWD ? 1 : -1;
  }
}

// [A_i | c_i][m, c] = sum_k U_i[m, k] [A_{i-1} | c_{i-1}][k, c] + [V_i | b_i][m, c].  Warp w owns row w of every 32-row block; its
// lanes stride over k, the four column sums are reduced with a value-splitting butterfly (6 shuffles).
__global__ void __launch_bounds__(CH_THREADS, 1) chain_fwd_kernel(const __grid_constant__ ChainParams p) {
  extern __shared__ uint8_t ch_smem_[];
  __shared__ __align__(16) float buf[2][CH_MAXH][CH_CW];
  __shared__ uint64_t full[CH_STAGES], empty[CH_STAGES];
  uint8_t* ring = ch_smem_ + ((128u - (b200::smem_u32(ch_smem_) & 127u)) & 127u);
  const int rank = static_cast<int>(b200::cluster_ctarank());
  int local;
  const ChainBranch& B = chain_branch(p, blockIdx.x / CH_R, &local);
  const int d = B.d, c0 = local * CH_CW, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) {
    for (int s = 0; s < CH_STAGES; ++s) {
      b200::mbar_init(&full[s], 1);
      b200::mbar_init(&empty[s], CH_THREADS / 32);
    }
    b200::fence_mbar_init();
  }
  if (tid < CH_MAXH) {   // layer 0 needs no product: every rank fills its own copy, the owner of a row writes it out
    const int m = tid, h = B.h[0], ldw = 2 * d;
    const float* W0 = B.W[0];
#pragma unroll
    for (int j = 0; j < CH_CW; ++j) {
      const int c = c0 + j;
      float v = 0.f;
      if (m < h && c <= d) v = c < d ? W0[static_cast<size_t>(m) * ldw + c] + W0[static_cast<size_t>(m) * ldw + d + c] : B.b[0][m];
      buf[0][m][j] = v;
      if (m < h && c <= d && m / CH_RPR == rank) B.Aaug[static_cast<size_t>(m) * CH_LD + c] = v;
    }
  }
  __syncthreads();
  b200::cluster_sync_all();   // the peer's shared memory exists and is initialised before anyone writes into it
  ChainFeed feed{1, 0, 0};
  if (tid == 0)
    for (int k = 0; k < CH_STAGES - 1; ++k) chain_feed<true>(B, p.L, rank, feed, ring, full, empty);
  static_assert(CH_CW == 4, "the forward recurrence keeps a 4-column slice of [A | c] in registers");
  const bool b4 = (lane & 16) != 0, b3 = (lane & 8) != 0;
  const int my_col = c0 + (b4 ? 2 : 0) + (b3 ? 1 : 0);   // the column whose sum this lane ends up with
  const uint32_t peer_buf = b200::mapa_u32(b200::smem_u32(&buf[0][0][0]), static_cast<uint32_t>(rank ^ 1));
  int q = 0;
  for (int i = 1; i < p.L; ++i) {
    const int h = B.h[i], pw = B.h[i - 1], ldw = pw + d, own = chain_own_rows(h, rank), row_base = rank * CH_RPR;
    float(*dst)[CH_CW] = buf[i & 1];
    const float* bias = B.b[i];
    // this lane's rows k = lane + 32 j of [A_{i-1} | c_{i-1}] stay in registers for the whole layer: every warp multiplies them
    // with one row of U_i per block, and re-reading them from shared memory per row made the kernel shared-memory bound
    float4 a[CH_MAXH / 32];
#pragma unroll
    for (int j = 0; j < CH_MAXH / 32; ++j) {
      const int k = lane + 32 * j;
      a[j] = k < pw ? *reinterpret_cast<const float4*>(buf[(i - 1) & 1][k]) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    for (int r0 = 0; r0 < own; r0 += CH_ROWS, ++q) {
      if (tid == 0) chain_feed<true>(B, p.L, rank, feed, ring, full, empty);
      const int s = q % CH_STAGES;
      b200::mbar_wait(&full[s], static_cast<uint32_t>(q / CH_STAGES) & 1u);
      const float* Us = reinterpret_cast<const float*>(ring + static_cast<size_t>(s) * CH_STAGE_BYTES) + warp * ldw;
      const int m = row_base + r0 + warp;
      const bool live = r0 + warp < own;
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
      if (live) {
#pragma unroll
        for (int j = 0; j < CH_MAXH / 32; ++j) {
          const int k = lane + 32 * j;
          const float u = k < pw ? Us[k] : 0.f;
          a0 = fmaf(u, a[j].x, a0);
          a1 = fmaf(u, a[j].y, a1);
          a2 = fmaf(u, a[j].z, a2);
          a3 = fmaf(u, a[j].w, a3);
        }
      }
      // value-splitting butterfly: every step keeps half of the sums and ships the other half (2 + 1 + 3 shuffles)
      float x0 = b4 ? a2 : a0, x1 = b4 ? a3 : a1;
      x0 += __shfl_xor_sync(0xffffffffu, b4 ? a0 : a2, 16);
      x1 += __shfl_xor_sync(0xffffffffu, b4 ? a1 : a3, 16);
      float y = b3 ? x1 : x0;
      y += __shfl_xor_sync(0xffffffffu, b3 ? x0 : x1, 8);
      y += __shfl_xor_sync(0xffffffffu, y, 4);
      y += __shfl_xor_sync(0xffffffffu, y, 2);
      y += __shfl_xor_sync(0xffffffffu, y, 1);
      if ((lane & 7) == 0 && live) {
        float v = 0.f;
        if (my_col <= d) {
          v = y + (my_col < d ? Us[pw + my_col] : bias[m]);
          B.Aaug[(static_cast<size_t>(i) * CH_MAXH + m) * CH_LD + my_col] = v;
        }
        dst[m][my_col - c0] = v;
        // the peer multiplies the next layer with the whole slice: its copy of this row
        st_cluster_f32(peer_buf + static_cast<uint32_t>((((i & 1) * CH_MAXH + m) * CH_CW + (my_col - c0)) * 4), v);
      }
      __syncwarp();
      if (lane == 0) b200::mbar_arrive(&empty[s]);
    }
    b200::cluster_sync_all();   // both halves of [A_i | c_i] are in both CTAs (release / acquire at cluster scope)
  }
  const int hl = B.h[p.L - 1];
  if (rank == 0 && d >= c0 && d < c0 + CH_CW && tid < hl) B.c_last[tid] = buf[(p.L - 1) & 1][tid][d - c0];
}

// R_{i-1}[k, c] = sum_m U_i[m, k] R_i[m, c]: thread (g, k) sums rows 8 g .. 8 g + 7 of every 32-row block (consecutive threads read
// consecutive shared-memory words), the four partial sums per element are added through shared memory at the end of the layer.
__global__ void __launch_bounds__(CH_THREADS, 1) chain_bwd_kernel(const __grid_constant__ ChainParams p) {
  extern __shared__ uint8_t ch_smem_[];
  __shared__ __align__(16) float buf[2][CH_MAXH][CH_CW];
  __shared__ uint64_t full[CH_STAGES], empty[CH_STAGES];
  uint8_t* ring = ch_smem_ + ((128u - (b200::smem_u32(ch_smem_) & 127u)) & 127u);
  float(*part)[CH_MAXH][CH_CW] = reinterpret_cast<float(*)[CH_MAXH][CH_CW]>(ring + CH_STAGES * CH_STAGE_BYTES);
  // slot[parity][k][c]: the PEER's partial sums over its rows of U_i (it writes them here through distributed shared memory)
  float(*slot)[CH_MAXH][CH_CW] = reinterpret_cast<float(*)[CH_MAXH][CH_CW]>(ring + CH_STAGES * CH_STAGE_BYTES + CH_PART_BYTES);
  const int rank = static_cast<int>(b200::cluster_ctarank());
  int local;
  const ChainBranch& B = chain_branch(p, blockIdx.x / CH_R, &local);
  const int d = B.d, c0 = local * CH_CW, tid = threadIdx.x, lane = tid & 31, k = tid & (CH_MAXH - 1), g = tid >> 8;
  if (tid == 0) {
    for (int s = 0; s < CH_STAGES; ++s) {
      b200::mbar_init(&full[s], 1);
      b200::mbar_init(&empty[s], CH_THREADS / 32);
    }
    b200::fence_mbar_init();
  }
  if (tid < CH_MAXH) {
    const int h = B.h[p.L - 1];
#pragma unroll
    for (int j = 0; j < CH_CW; ++j) {
      const int c = c0 + j;
      float v = 0.f;
      if (tid < h && c <= d) v = c < d ? B.G[static_cast<size_t>(tid) * CH_LD + c] : B.g[tid];
      buf[(p.L - 1) & 1][tid][j] = v;
    }
  }
  __syncthreads();
  b200::cluster_sync_all();   // the peer's shared memory exists before anyone writes into it
  const uint32_t peer_slot = b200::mapa_u32(b200::smem_u32(&slot[0][0][0]), static_cast<uint32_t>(rank ^ 1));
  ChainFeed feed{p.L - 1, 0, 0};
  if (tid == 0)
    for (int n = 0; n < CH_STAGES - 1; ++n) chain_feed<false>(B, p.L, rank, feed, ring, full, empty);
  int q = 0;
  for (int i = p.L - 1; i >= 0; --i) {
    const int h = B.h[i], pw = i ? B.h[i - 1] : d, ldw = pw + d;
    const float(*src)[CH_CW] = buf[i & 1];
    if (tid < h && tid / CH_RPR == rank) {   // gradients of layer i that are columns of R_i: the owner of a row writes it
      float* gw = B.gW[i] + static_cast<size_t>(tid) * ldw;
#pragma unroll
      for (int j = 0; j < CH_CW; ++j) {
        const int c = c0 + j;
        const float r = src[tid][j];
        if (c < d) {
          gw[pw + c] = r;
          if (i == 0) gw[c] = r;
        } else if (c == d) {
          B.gb[i][tid] = r;
        }
        if (c <= d) B.Raug[(static_cast<size_t>(i) * CH_MAXH + tid) * CH_LD + c] = r;
      }
    }
    if (i == 0) break;
    const int own = chain_own_rows(h, rank), row_base = rank * CH_RPR;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    for (int r0 = 0; r0 < own; r0 += CH_ROWS, ++q) {
      if (tid == 0) chain_feed<false>(B, p.L, rank, feed, ring, full, empty);
      const int s = q % CH_STAGES;
      b200::mbar_wait(&full[s], static_cast<uint32_t>(q / CH_STAGES) & 1u);
      const float* Us = reinterpret_cast<const float*>(ring + static_cast<size_t>(s) * CH_STAGE_BYTES) + k;
      if (k < pw) {
#pragma unroll
        for (int r = 0; r < CH_ROWS / 4; ++r) {
          const int rr = g * (CH_ROWS / 4) + r;
          if (r0 + rr < own) {
            const float u = Us[rr * ldw];
            const float4 a = *reinterpret_cast<const float4*>(src[row_base + r0 + rr]);
            a0 = fmaf(u, a.x, a0);
            a1 = fmaf(u, a.y, a1);
            a2 = fmaf(u, a.z, a2);
            a3 = fmaf(u, a.w, a3);
          }
        }
      }
      __syncwarp();
      if (lane == 0) b200::mbar_arrive(&empty[s]);
    }
    *reinterpret_cast<float4*>(part[g][k]) = make_float4(a0, a1, a2, a3);
    __syncthreads();
    const int par = i & 1;
    float4 mine = make_float4(0.f, 0.f, 0.f, 0.f);
    if (tid < CH_MAXH) {   // this rank's partial sums of row tid of R_{i-1}: kept here, sent to the peer
      if (tid < pw) {
        const float4 p0 = *reinterpret_cast<const float4*>(part[0][tid]), p1 = *reinterpret_cast<const float4*>(part[1][tid]);
        const float4 p2 = *reinterpret_cast<const float4*>(part[2][tid]), p3 = *reinterpret_cast<const float4*>(part[3][tid]);
        mine = make_float4((p0.x + p1.x) + (p2.x + p3.x), (p0.y + p1.y) + (p2.y + p3.y), (p0.z + p1.z) + (p2.z + p3.z),
                           (p0.w + p1.w) + (p2.w + p3.w));
      }
      st_cluster_v4(peer_slot + static_cast<uint32_t>(((par * CH_MAXH + tid) * CH_CW) * 4), mine);
    }
    b200::cluster_sync_all();   // the peer's partial sums have arrived; the parity keeps the next layer's writes apart
    if (tid < CH_MAXH) {
      const float4 o = *reinterpret_cast<const float4*>(slot[par][tid]);
      // a + b == b + a bit for bit: both CTAs continue with the same R_{i-1}
      *reinterpret_cast<float4*>(buf[(i - 1) & 1][tid]) = make_float4(mine.x + o.x, mine.y + o.y, mine.z + o.z, mine.w + o.w);
    }
    __syncthreads();
  }
}

// dU_i[m, k] = sum_c R_i[m, c] [A_{i-1} | c_{i-1}][k, c]: up to 3 x (CH_MAXL - 1) independent small products, one launch
struct DuProb {
  const float* R;   // [h, CH_LD]
  const float* A;   // [pw, CH_LD]
  float* C;         // grads of W_i, row stride ldw
  int h, pw, K, ldw;
};
struct DuBatch {
  DuProb p[3 * (CH_MAXL - 1)];
};
__global__ void __launch_bounds__(256) chain_du_kernel(const __grid_constant__ DuBatch batch) {
  const DuProb q = batch.p[blockIdx.z];
  const int m0 = blockIdx.y * GM, n0 = blockIdx.x * GN;
  if (m0 >= q.h || n0 >= q.pw) return;
  __shared__ float Rs[GK][GM + 4];
  __shared__ float As[GK][GN + 4];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int k0 = 0; k0 < q.K; k0 += GK) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int idx = tid + e * 256;
      const int r = idx >> 4, k = idx & 15;   // both operands are k-contiguous
      Rs[k][r] = (m0 + r < q.h && k0 + k < q.K) ? __ldg(q.R + static_cast<size_t>(m0 + r) * CH_LD + k0 + k) : 0.f;
      As[k][r] = (n0 + r < q.pw && k0 + k < q.K) ? __ldg(q.A + static_cast<size_t>(n0 + r) * CH_LD + k0 + k) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < GK; ++k) {
      const float4 a4 = *reinterpret_cast<const float4*>(&Rs[k][ty * 4]);
      const float4 b4 = *reinterpret_cast<const float4*>(&As[k][tx * 4]);
      const float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int gm = m0 + ty * 4 + i;
    if (gm >= q.h) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gn = n0 + tx * 4 + j;
      if (gn < q.pw) q.C[static_cast<size_t>(gm) * q.ldw + gn] = acc[i][j];
    }
  }
}

// B200NERF_TRAIN_BRANCHES=literal keeps the per-layer, per-ray form of the branches (A/B measurements, reference point in tests)
static bool branches_collapsed() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("B200NERF_TRAIN_BRANCHES");
    v = (e && strcmp(e, "literal") == 0) ? 0 : 1;
  }
  return v == 1;
}

// ------------------------------------------------------------------------------------------- DepthNet, literal form
struct DnArch {
  int nb;                 // layers per branch
  int nc;                 // cat layers
  std::vector<int> h;     // branch widths [nb]
  std::vector<int> c;     // cat widths [nc]
  int m;                  // multires: gamma(o) / gamma(d) are d3 = 3 (1 + 2 m) wide, gamma(hits) 2 d3
  int d3, ew;             // d3 and the row width of the encoding E, ew = 4 d3 (= the K of cat_layers.0's encoding segment)
  int ed(int b) const { return b == 2 ? 2 * d3 : d3; }   // encoding width of branch b (origin / direction / intersection)
  int eo(int b) const { return b * d3; }                 // its column offset in E
};
struct DnWs {             // float offsets into the workspace
  size_t E, s, t, total;
  std::vector<size_t> xb[3];   // branch outputs
  std::vector<size_t> a;       // cat layer outputs (post activation)
  size_t g0, g1, g2;           // gradient scratch, [n, maxw] each
  size_t gx[6];                // per-branch ping/pong scratch of the grouped backward
  std::vector<size_t> jac;     // J_j = d z / d(pre-activation of cat layer j) per ray (the split backward)
  size_t img_fwd, img_jac, aux, mask;   // fused cat chain: bf16 hi / lo weight images (W_j, W_j^T), fp32 bias / head block, sign masks
  size_t Aaug[3], Raug[3], G[3], gv[3], c_last[3];   // collapsed-branch chain matrices (weights only, no ray dimension)
};
static DnWs dn_layout(const DnArch& ar, size_t n) {
  DnWs w;
  size_t o = 0;
  auto take = [&](size_t f) { size_t r = o; o += (f + 63) & ~static_cast<size_t>(63); return r; };
  w.E = take(n * ar.ew);
  for (int b = 0; b < 3; ++b)
    for (int i = 0; i < ar.nb; ++i) w.xb[b].push_back(take(n * ar.h[i]));
  for (int j = 0; j < ar.nc; ++j) w.a.push_back(take(n * ar.c[j]));
  w.t = take(n);
  w.s = take(n);
  int maxw = 1;
  for (int v : ar.h) maxw = v > maxw ? v : maxw;
  for (int v : ar.c) maxw = v > maxw ? v : maxw;
  w.g0 = take(n * maxw);
  w.g1 = take(n * maxw);
  w.g2 = take(n * maxw);
  for (int i = 0; i < 6; ++i) w.gx[i] = take(n * maxw);
  for (int j = 0; j < ar.nc; ++j) w.jac.push_back(take(n * ar.c[j]));
  {
    const int nl = ar.nc > 1 ? ar.nc - 1 : 1;
    w.img_fwd = take(b200_catchain_img_bytes(nl) / 4);
    w.img_jac = take(b200_catchain_img_bytes(nl) / 4);
    w.aux = take(b200_catchain_aux_floats());
    w.mask = take(2 * b200_catchain_mask_words(nl, static_cast<int>(n)));
  }
  for (int b = 0; b < 3; ++b) {
    w.Aaug[b] = take(static_cast<size_t>(ar.nb) * CH_MAXH * CH_LD);
    w.Raug[b] = take(static_cast<size_t>(ar.nb) * CH_MAXH * CH_LD);
    w.c_last[b] = take(CH_MAXH);
  }
  for (int b = 0; b < 3; ++b) w.G[b] = take(static_cast<size_t>(CH_MAXH) * CH_LD);   // G and gv back to back: one memset
  for (int b = 0; b < 3; ++b) w.gv[b] = take(CH_MAXH);
  w.total = o;
  return w;
}
static int dn_arch(int nb, const int* h, int nc, const int* c, int multires, DnArch* ar) {
  if (nb < 1 || nc < 1 || !h || !c) return b200_fail("DepthNet architecture: bad arguments");
  // multires 10 is the widest encoding the collapsed-branch chain matrices hold: 2 d3 + 1 = 127 columns of CH_LD
  if (multires < 1 || multires > 10) return b200_fail("DepthNet architecture: multires=%d out of range (1..10)", multires);
  ar->nb = nb;
  ar->nc = nc;
  ar->h.assign(h, h + nb);
  ar->c.assign(c, c + nc);
  ar->m = multires;
  ar->d3 = 3 * (1 + 2 * multires);
  ar->ew = 4 * ar->d3;
  return 0;
}
// parameter order = state_dict order: origin_layers.{i}.{w,b}, direction_layers..., intersection_layers...,
// cat_layers.{2j}.{w,b}, to_depth.0.{w,b}
static inline int pidx_branch(const DnArch& ar, int b, int i) { return (b * ar.nb + i) * 2; }
static inline int pidx_cat(const DnArch& ar, int j) { return (3 * ar.nb + j) * 2; }
static inline int pidx_head(const DnArch& ar) { return (3 * ar.nb + ar.nc) * 2; }

// widths up to 256 and multiples of 4 (every 32-row block of W_i is then a 16-byte multiple), 16-byte aligned weight tensors
static bool can_collapse(const DnArch& ar, int n, const float* const* params) {
  if (!tgemm_enabled() || n < 32 || !branches_collapsed() || ar.nb > CH_MAXL) return false;
  for (int v : ar.h)
    if (v > CH_MAXH || (v & 3)) return false;
  for (int b = 0; b < 3; ++b)
    for (int i = 0; i < ar.nb; ++i)
      if (reinterpret_cast<uintptr_t>(params[pidx_branch(ar, b, i)]) & 15) return false;
  return true;
}
// The activated cat layers behind cat_layers.0 as ONE launch of the fused split-precision MLP kernel (forward: with saved activations;
// split backward: the Jacobian chain over the transposed weights) instead of one grouped product per layer.  Needs 256-wide layers;
// B200NERF_TRAIN_CHAIN=gemm keeps the per-layer 3xTF32 products (A/B measurements, and the reference point of the tests).
static bool fused_chain_ok(const DnArch& ar, int n, const float* const* params) {
  const char* e = getenv("B200NERF_TRAIN_CHAIN");   // read per call: the tests run both routes in one process
  if ((e && strcmp(e, "gemm") == 0) || !can_collapse(ar, n, params) || ar.nc < 2 || ar.nc - 1 > B200_CATCHAIN_MAX_LAYERS) return false;
  if (256 * static_cast<size_t>(ar.nc - 1 + 3) > b200_catchain_aux_floats()) return false;   // biases + head + cat_layers.0's bias in the kernel's aux block
  for (int c : ar.c)
    if (c != 256) return false;
  for (int j = 0; j < ar.nc; ++j)
    if (reinterpret_cast<uintptr_t>(params[pidx_cat(ar, j)]) & 15) return false;
  return true;
}
// The split form of cat_layers.0 pays where the step is a latency chain (512 rays: 58 -> 26 us, step 0.60 -> 0.56 ms); at 4096 rays its
// extra CTAs, atomics and memset cost SM time beside the target render (1.365 -> 1.41 ms).  It hands the bias and the LeakyReLU to the
// fused chain's loader, so it needs that chain.
static bool split_cat0(const DnArch& ar, int n, const float* const* params) { return fused_chain_ok(ar, n, params) && n <= 2048; }
// Below 32 rays (or with B200NERF_TRAIN_GEMM=fp32) every pass runs per layer: CUDA-core head kernels and sgemm's product mix.
static bool tensor_path_ok(int n) { return tgemm_enabled() && n >= 32; }
static int chain_configure() {
  static bool configured[B200_MAX_DEVICES] = {false};
  const int dev = b200_device();
  if (dev < 0) return b200_fail("chain kernels: no usable CUDA device");
  if (!configured[dev]) {
    CUDA_TRY(cudaFuncSetAttribute(chain_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, CH_SMEM_BYTES));
    CUDA_TRY(cudaFuncSetAttribute(chain_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, CH_SMEM_BYTES));
    configured[dev] = true;
  }
  return 0;
}
static ChainParams chain_params(const DnArch& ar, const DnWs& w, float* ws, const float* const* params, float* const* grads) {
  ChainParams cp;
  memset(&cp, 0, sizeof(cp));
  const int ed[3] = {ar.ed(0), ar.ed(1), ar.ed(2)};
  cp.L = ar.nb;
  int cta = 0;
  for (int b = 0; b < 3; ++b) {
    ChainBranch& B = cp.br[b];
    for (int i = 0; i < ar.nb; ++i) {
      B.W[i] = params[pidx_branch(ar, b, i)];
      B.b[i] = params[pidx_branch(ar, b, i) + 1];
      if (grads) {
        B.gW[i] = grads[pidx_branch(ar, b, i)];
        B.gb[i] = grads[pidx_branch(ar, b, i) + 1];
      }
      B.h[i] = ar.h[i];
    }
    B.d = ed[b];
    B.cta_begin = cta;
    cta += (ed[b] + 1 + CH_CW - 1) / CH_CW;
    B.Aaug = ws + w.Aaug[b];
    B.Raug = ws + w.Raug[b];
    B.c_last = ws + w.c_last[b];
    B.G = ws + w.G[b];
    B.g = ws + w.gv[b];
  }
  return cp;
}
static int chain_ctas(const ChainParams& cp) { return cp.br[2].cta_begin + (cp.br[2].d + 1 + CH_CW - 1) / CH_CW; }
// one cluster of CH_R CTAs per column group
static int launch_chain(void (*kern)(const ChainParams), const ChainParams& cp, cudaStream_t st) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CH_R;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.gridDim = dim3(CH_R * chain_ctas(cp));
  cfg.blockDim = dim3(CH_THREADS);
  cfg.dynamicSmemBytes = CH_SMEM_BYTES;
  cfg.stream = st;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, cp));
  LAUNCH_CHECK();
  return 0;
}

extern "C" size_t b200nerf_depthnet_train_ws_floats_multires(int n_rays, int n_branch, const int* hidden, int n_cat, const int* cat_hidden,
                                                            int multires) {
  DnArch ar;
  if (dn_arch(n_branch, hidden, n_cat, cat_hidden, multires, &ar)) return 0;
  return dn_layout(ar, static_cast<size_t>(n_rays)).total;
}
extern "C" size_t b200nerf_depthnet_train_ws_floats(int n_rays, int n_branch, const int* hidden, int n_cat, const int* cat_hidden) {
  return b200nerf_depthnet_train_ws_floats_multires(n_rays, n_branch, hidden, n_cat, cat_hidden, 10);
}
extern "C" int b200nerf_depthnet_n_params(int n_branch, int n_cat) { return (3 * n_branch + n_cat + 1) * 2; }

extern "C" int b200nerf_depthnet_train_fwd_multires(const float* const* params, int n_branch, const int* hidden, int n_cat,
                                                    const int* cat_hidden, int multires, const float* rays_o, const float* rays_d, int n_rays,
                                                    float radius, float near_, float far_, float* ws, float* out_z, void* stream) {
  if (n_rays <= 0) return 0;
  if (!params || !rays_o || !rays_d || !ws || !out_z) return b200_fail("b200nerf_depthnet_train_fwd: null argument");
  DnArch ar;
  if (dn_arch(n_branch, hidden, n_cat, cat_hidden, multires, &ar)) return 1;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int n = n_rays;
  const DnWs w = dn_layout(ar, n);
  float* E = ws + w.E;
  depthnet_encode_kernel<<<(12 * n + 191) / 192, 192, 0, st>>>(rays_o, rays_d, n, radius, ar.m, E);
  LAUNCH_CHECK();
  const int ed[3] = {ar.ed(0), ar.ed(1), ar.ed(2)}, eo[3] = {ar.eo(0), ar.eo(1), ar.eo(2)};
  if (tensor_path_ok(n)) {
    const bool collapse = can_collapse(ar, n, params);
    if (collapse) {
      // collapsed branches: [A_i | c_i] recurrences over the weights (one launch), then x_last = e A_last^T + c_last per ray
      const ChainParams cp = chain_params(ar, w, ws, params, nullptr);
      if (chain_configure()) return 1;
      if (launch_chain(chain_fwd_kernel, cp, st)) return 1;
      GemmProb q[3];
      const int hlast = ar.h[ar.nb - 1];
      for (int b = 0; b < 3; ++b) {
        q[b] = prob_fwd(n, hlast, ws + w.xb[b][ar.nb - 1], hlast, ws + w.c_last[b], 0, 0.f);
        seg_fwd(q[b], E + eo[b], ar.ew, ws + w.Aaug[b] + static_cast<size_t>(ar.nb - 1) * CH_MAXH * CH_LD, CH_LD, 0, ed[b]);
      }
      if (tgemm_group(st, q, 3)) return 1;
    }
    // literal branches: they advance together (one grouped launch per layer index), Linear(cat([x, e])) is two
    // K segments of one product, cat_layers.0 is four
    for (int i = 0; i < (collapse ? 0 : ar.nb); ++i) {
      GemmProb q[3];
      for (int b = 0; b < 3; ++b) {
        const float* e = E + eo[b];
        const float* W = params[pidx_branch(ar, b, i)];
        const int prev_w = i == 0 ? ed[b] : ar.h[i - 1];
        const float* prev = i == 0 ? e : ws + w.xb[b][i - 1];
        const int prev_ld = i == 0 ? ar.ew : ar.h[i - 1];
        const int ldw = prev_w + ed[b];
        q[b] = prob_fwd(n, ar.h[i], ws + w.xb[b][i], ar.h[i], params[pidx_branch(ar, b, i) + 1], 0, 0.f);
        seg_fwd(q[b], prev, prev_ld, W, ldw, 0, prev_w);
        seg_fwd(q[b], e, ar.ew, W, ldw, prev_w, ed[b]);
      }
      if (tgemm_group(st, q, 3)) return 1;
    }
    const int hl = ar.h[ar.nb - 1];
    const bool fused = fused_chain_ok(ar, n, params);
    const bool split0 = split_cat0(ar, n, params);
    {
      const float* W = params[pidx_cat(ar, 0)];
      const int ldw = 3 * hl + ar.ew;
      if (split0) {
        // cat_layers.0 as FOUR split-K problems (one per K segment, two K slices each) that add into the zeroed output: K = 1020 in
        // one CTA is 32 chunks and, at 512 rays, the longest launch in front of the fused chain (58 us); the bias and the LeakyReLU
        // move into the chain kernel's loader, which reads these rows anyway and writes the activated rows back for the backward
        CUDA_TRY(cudaMemsetAsync(ws + w.a[0], 0, static_cast<size_t>(n) * ar.c[0] * sizeof(float), st));
        GemmProb q[4];
        for (int b = 0; b < 3; ++b) {
          q[b] = prob_fwd(n, ar.c[0], ws + w.a[0], ar.c[0], nullptr, 0, 0.f);
          seg_fwd(q[b], ws + w.xb[b][ar.nb - 1], hl, W, ldw, b * hl, hl);
        }
        q[3] = prob_fwd(n, ar.c[0], ws + w.a[0], ar.c[0], nullptr, 0, 0.f);
        seg_fwd(q[3], E, ar.ew, W, ldw, 3 * hl, ar.ew);
        for (int i = 0; i < 4; ++i) {
          q[i].force_splits = 2;
          q[i].c_zeroed = true;
        }
        if (tgemm_group(st, q, 4)) return 1;
      } else {
        GemmProb q = prob_fwd(n, ar.c[0], ws + w.a[0], ar.c[0], params[pidx_cat(ar, 0) + 1], 1, 0.01f);
        for (int b = 0; b < 3; ++b) seg_fwd(q, ws + w.xb[b][ar.nb - 1], hl, W, ldw, b * hl, hl);
        seg_fwd(q, E, ar.ew, W, ldw, 3 * hl, ar.ew);
        if (tgemm_group(st, &q, 1)) return 1;
      }
    }
    if (fused) {
      // cat_layers.1 .. nc-1 + head in one launch: this step's weights -> bf16 hi / lo images (W_j for this pass, W_j^T for the
      // Jacobian pass), then the chain with every layer's activations saved for the backward
      const int nl = ar.nc - 1;
      const float* Wl[B200_CATCHAIN_MAX_LAYERS];
      const float* bl[B200_CATCHAIN_MAX_LAYERS];
      float* save[B200_CATCHAIN_MAX_LAYERS];
      for (int j = 1; j < ar.nc; ++j) {
        Wl[j - 1] = params[pidx_cat(ar, j)];
        bl[j - 1] = params[pidx_cat(ar, j) + 1];
        save[j - 1] = ws + w.a[j];
      }
      if (b200_catchain_pack(Wl, bl, params[pidx_head(ar)], params[pidx_head(ar) + 1], split0 ? params[pidx_cat(ar, 0) + 1] : nullptr, nl,
                             ws + w.img_fwd, ws + w.img_jac, ws + w.aux, st))
        return 1;
      return b200_catchain_fwd(ws + w.img_fwd, ws + w.aux, nl, ws + w.a[0], split0, n, near_, far_, save,
                               reinterpret_cast<unsigned long long*>(ws + w.mask), out_z, ws + w.s, st);
    }
    for (int j = 1; j < ar.nc; ++j) {
      GemmProb q = prob_fwd(n, ar.c[j], ws + w.a[j], ar.c[j], params[pidx_cat(ar, j) + 1], 1, 0.01f);
      seg_fwd(q, ws + w.a[j - 1], ar.c[j - 1], params[pidx_cat(ar, j)], ar.c[j - 1], 0, ar.c[j - 1]);
      if (tgemm_group(st, &q, 1)) return 1;
    }
    const int cl = ar.c[ar.nc - 1];
    depth_head_fused_kernel<<<(n + 7) / 8, 256, 0, st>>>(ws + w.a[ar.nc - 1], n, cl, params[pidx_head(ar)], params[pidx_head(ar) + 1], near_,
                                                        far_, ws + w.s, out_z);
    LAUNCH_CHECK();
    return 0;
  }
  for (int b = 0; b < 3; ++b) {
    const float* e = E + eo[b];
    for (int i = 0; i < ar.nb; ++i) {
      const float* W = params[pidx_branch(ar, b, i)];
      const float* bias = params[pidx_branch(ar, b, i) + 1];
      float* y = ws + w.xb[b][i];
      const int prev_w = i == 0 ? ed[b] : ar.h[i - 1];
      const float* prev = i == 0 ? e : ws + w.xb[b][i - 1];
      const int prev_ld = i == 0 ? ar.ew : ar.h[i - 1];
      const int ldw = prev_w + ed[b];
      // x = Linear(cat([x_prev, e])) -- no activation (depth_net.py:140,148,156 construct a module and drop it)
      if (lin_fwd(st, n, ar.h[i], prev_w, prev, prev_ld, W, ldw, 0, y, ar.h[i], 0, nullptr, 0, 0.f)) return 1;
      if (lin_fwd(st, n, ar.h[i], ed[b], e, ar.ew, W, ldw, prev_w, y, ar.h[i], 1, bias, 0, 0.f)) return 1;
    }
  }
  const int hl = ar.h[ar.nb - 1];
  {
    // cat_layers.0 over cat([x_o, x_d, x_i, e_o, e_d, e_i])
    const float* W = params[pidx_cat(ar, 0)];
    const float* bias = params[pidx_cat(ar, 0) + 1];
    const int ldw = 3 * hl + ar.ew;
    float* y = ws + w.a[0];
    for (int b = 0; b < 3; ++b)
      if (lin_fwd(st, n, ar.c[0], hl, ws + w.xb[b][ar.nb - 1], hl, W, ldw, b * hl, y, ar.c[0], b > 0, nullptr, 0, 0.f)) return 1;
    if (lin_fwd(st, n, ar.c[0], ar.ew, E, ar.ew, W, ldw, 3 * hl, y, ar.c[0], 1, bias, 1, 0.01f)) return 1;
  }
  for (int j = 1; j < ar.nc; ++j) {
    if (lin_fwd(st, n, ar.c[j], ar.c[j - 1], ws + w.a[j - 1], ar.c[j - 1], params[pidx_cat(ar, j)], ar.c[j - 1], 0, ws + w.a[j],
                ar.c[j], 0, params[pidx_cat(ar, j) + 1], 1, 0.01f))
      return 1;
  }
  const int cl = ar.c[ar.nc - 1];
  if (lin_fwd(st, n, 1, cl, ws + w.a[ar.nc - 1], cl, params[pidx_head(ar)], cl, 0, ws + w.t, 1, 0, params[pidx_head(ar) + 1], 0, 0.f))
    return 1;
  depth_head_kernel<<<(n + 255) / 256, 256, 0, st>>>(ws + w.t, n, near_, far_, ws + w.s, out_z);
  LAUNCH_CHECK();
  return 0;
}
extern "C" int b200nerf_depthnet_train_fwd(const float* const* params, int n_branch, const int* hidden, int n_cat,
                                           const int* cat_hidden, const float* rays_o, const float* rays_d, int n_rays, float radius,
                                           float near_, float far_, float* ws, float* out_z, void* stream) {
  return b200nerf_depthnet_train_fwd_multires(params, n_branch, hidden, n_cat, cat_hidden, 10, rays_o, rays_d, n_rays, radius, near_, far_,
                                              ws, out_z, stream);
}

// Weight gradients are split-K sums and bias gradients column sums added atomically: the gradient tensors are zeroed first -- one
// memset when the caller laid them out back to back (training.py does), else one each.
static int zero_grads(const DnArch& ar, float* const* grads, cudaStream_t st) {
  std::vector<size_t> numel;
  const int ed[3] = {ar.ed(0), ar.ed(1), ar.ed(2)};
  const int hl = ar.h[ar.nb - 1], cl = ar.c[ar.nc - 1];
  for (int b = 0; b < 3; ++b)
    for (int i = 0; i < ar.nb; ++i) {
      numel.push_back(static_cast<size_t>(ar.h[i]) * ((i == 0 ? ed[b] : ar.h[i - 1]) + ed[b]));
      numel.push_back(ar.h[i]);
    }
  for (int j = 0; j < ar.nc; ++j) {
    numel.push_back(static_cast<size_t>(ar.c[j]) * (j == 0 ? 3 * hl + ar.ew : ar.c[j - 1]));
    numel.push_back(ar.c[j]);
  }
  numel.push_back(cl);   // the head: its gradients are atomic sums of the fused head kernel
  numel.push_back(1);
  const size_t n_body = numel.size();
  bool flat = true;
  size_t total = 0;
  for (size_t k = 0; k < n_body; ++k) {
    if (k + 1 < n_body && grads[k + 1] != grads[k] + numel[k]) flat = false;
    total += numel[k];
  }
  if (flat) {
    CUDA_TRY(cudaMemsetAsync(grads[0], 0, total * sizeof(float), st));
  } else {
    for (size_t k = 0; k < n_body; ++k) CUDA_TRY(cudaMemsetAsync(grads[k], 0, numel[k] * sizeof(float), st));
  }
  return 0;
}
// The collapsed branches' backward behind the ray reduction (G = D^T e, g = D^T 1 already in the workspace): the R recurrence over the
// weights (writes dV_i, db_i, dU_0), then the 3 (L-1) small dU_i products in one launch.
static int chain_backward(const DnArch& ar, const DnWs& w, float* ws, const float* const* params, float* const* grads, cudaStream_t st) {
  const int ed[3] = {ar.ed(0), ar.ed(1), ar.ed(2)};
  const ChainParams cp = chain_params(ar, w, ws, params, grads);
  if (chain_configure()) return 1;
  if (launch_chain(chain_bwd_kernel, cp, st)) return 1;
  if (ar.nb > 1) {
    DuBatch batch;
    memset(&batch, 0, sizeof(batch));
    int np = 0, maxh = 0, maxpw = 0;
    for (int b = 0; b < 3; ++b)
      for (int i = 1; i < ar.nb; ++i) {
        DuProb& d = batch.p[np++];
        d.R = ws + w.Raug[b] + static_cast<size_t>(i) * CH_MAXH * CH_LD;
        d.A = ws + w.Aaug[b] + static_cast<size_t>(i - 1) * CH_MAXH * CH_LD;
        d.C = grads[pidx_branch(ar, b, i)];
        d.h = ar.h[i];
        d.pw = ar.h[i - 1];
        d.K = ed[b] + 1;
        d.ldw = ar.h[i - 1] + ed[b];
        maxh = d.h > maxh ? d.h : maxh;
        maxpw = d.pw > maxpw ? d.pw : maxpw;
      }
    chain_du_kernel<<<dim3((maxpw + GN - 1) / GN, (maxh + GM - 1) / GM, np), 256, 0, st>>>(batch);
    LAUNCH_CHECK();
  }
  return 0;
}

extern "C" int b200nerf_depthnet_train_bwd_multires(const float* const* params, int n_branch, const int* hidden, int n_cat,
                                                    const int* cat_hidden, int multires, int n_rays, float near_, float far_, float* ws,
                                                    const float* dz, float* const* grads, void* stream) {
  if (n_rays <= 0) return 0;
  if (!params || !ws || !dz || !grads) return b200_fail("b200nerf_depthnet_train_bwd: null argument");
  DnArch ar;
  if (dn_arch(n_branch, hidden, n_cat, cat_hidden, multires, &ar)) return 1;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int n = n_rays;
  const DnWs w = dn_layout(ar, n);
  const float* E = ws + w.E;
  float* g = ws + w.g0;
  float* g2 = ws + w.g1;
  const int cl = ar.c[ar.nc - 1], hl = ar.h[ar.nb - 1];
  // head: t = a_last . w + b, s = sigmoid(t), z = near + (far - near) s
  float* dt = ws + w.t;  // t itself is no longer needed
  const int ph = pidx_head(ar);
  const bool tensor_path = tensor_path_ok(n);
  if (!tensor_path) {
    depth_head_bwd_kernel<<<(n + 255) / 256, 256, 0, st>>>(dz, ws + w.s, n, near_, far_, dt);
    LAUNCH_CHECK();
    if (lin_wgrad(st, n, 1, cl, dt, 1, ws + w.a[ar.nc - 1], cl, grads[ph], cl, 0)) return 1;
    if (colsum(st, dt, n, 1, 1, grads[ph + 1])) return 1;
    if (lin_dgrad(st, n, 1, cl, dt, 1, params[ph], cl, 0, g, cl, 0)) return 1;
  }
  if (tensor_path) {
    if (zero_grads(ar, grads, st)) return 1;
    // head backward + LeakyReLU' of the last cat layer, one pass: g = d(pre-activation of the last cat layer)
    depth_head_bwd_fused_kernel<<<(n + HEAD_ROWS - 1) / HEAD_ROWS, 256, 0, st>>>(dz, ws + w.s, ws + w.a[ar.nc - 1], params[ph], n, cl, near_,
                                                                              far_, 0.01f, g, grads[ph], grads[ph + 1]);
    LAUNCH_CHECK();
    // cat layers: g = d(pre-activation of layer j).  One launch per layer: weight gradient (+ bias gradient from the same
    // loads) and the input gradient, whose epilogue applies LeakyReLU' of the layer below.
    for (int j = ar.nc - 1; j >= 1; --j) {
      const int pc = pidx_cat(ar, j);
      GemmProb q[2];
      q[0] = prob_wgrad(n, ar.c[j], ar.c[j - 1], g, ar.c[j], ws + w.a[j - 1], ar.c[j - 1], grads[pc], ar.c[j - 1], 0, grads[pc + 1], true);
      q[1] = prob_dgrad(n, ar.c[j], ar.c[j - 1], g, ar.c[j], params[pc], ar.c[j - 1], 0, g2, ar.c[j - 1], ws + w.a[j - 1], ar.c[j - 1], 0.01f);
      if (tgemm_group(st, q, 2)) return 1;
      float* tmp = g;
      g = g2;
      g2 = tmp;
    }
    const int ed[3] = {ar.ed(0), ar.ed(1), ar.ed(2)}, eo[3] = {ar.eo(0), ar.eo(1), ar.eo(2)};
    const int pc0 = pidx_cat(ar, 0);
    const int ldw0 = 3 * hl + ar.ew;
    float* cur[3];
    float* alt[3];
    for (int b = 0; b < 3; ++b) {
      cur[b] = ws + w.gx[2 * b];
      alt[b] = ws + w.gx[2 * b + 1];
    }
    {
      GemmProb q[7];
      for (int b = 0; b < 3; ++b)
        q[b] = prob_wgrad(n, ar.c[0], hl, g, ar.c[0], ws + w.xb[b][ar.nb - 1], hl, grads[pc0], ldw0, b * hl, b == 0 ? grads[pc0 + 1] : nullptr, true);
      q[3] = prob_wgrad(n, ar.c[0], ar.ew, g, ar.c[0], E, ar.ew, grads[pc0], ldw0, 3 * hl, nullptr, true);
      for (int b = 0; b < 3; ++b) q[4 + b] = prob_dgrad(n, ar.c[0], hl, g, ar.c[0], params[pc0], ldw0, b * hl, cur[b], hl);
      if (tgemm_group(st, q, 7)) return 1;
    }
    if (can_collapse(ar, n, params)) {
      // cur[b] = D_b = dLoss/dx_{b,last}.  One reduction over the rays per branch (G = D^T e, g = D^T 1), the R recurrence over
      // the weights (writes dV_i, db_i, dU_0), then the 3 (L-1) small dU_i products in one launch.
      CUDA_TRY(cudaMemsetAsync(ws + w.G[0], 0, (w.gv[2] + CH_MAXH - w.G[0]) * sizeof(float), st));
      GemmProb q[3];
      for (int b = 0; b < 3; ++b)
        q[b] = prob_wgrad(n, hl, ed[b], cur[b], hl, E + eo[b], ar.ew, ws + w.G[b], CH_LD, 0, ws + w.gv[b], true);
      if (tgemm_group(st, q, 3)) return 1;
      if (chain_backward(ar, w, ws, params, grads, st)) return 1;
      return 0;
    }
    for (int i = ar.nb - 1; i >= 0; --i) {
      GemmProb q[9];
      int nq = 0;
      for (int b = 0; b < 3; ++b) {
        const float* e = E + eo[b];
        const int pb = pidx_branch(ar, b, i);
        const int prev_w = i == 0 ? ed[b] : ar.h[i - 1];
        const float* prev = i == 0 ? e : ws + w.xb[b][i - 1];
        const int prev_ld = i == 0 ? ar.ew : ar.h[i - 1];
        const int ldw = prev_w + ed[b];
        q[nq++] = prob_wgrad(n, ar.h[i], prev_w, cur[b], ar.h[i], prev, prev_ld, grads[pb], ldw, 0, grads[pb + 1], true);
        q[nq++] = prob_wgrad(n, ar.h[i], ed[b], cur[b], ar.h[i], e, ar.ew, grads[pb], ldw, prev_w, nullptr, true);
        if (i > 0) q[nq++] = prob_dgrad(n, ar.h[i], ar.h[i - 1], cur[b], ar.h[i], params[pb], ldw, 0, alt[b], ar.h[i - 1]);
      }
      if (tgemm_group(st, q, nq)) return 1;
      for (int b = 0; b < 3; ++b) {
        float* t = cur[b];
        cur[b] = alt[b];
        alt[b] = t;
      }
    }
    return 0;
  }
  // cat layers, last to first: g holds d(post-activation output of layer j)
  for (int j = ar.nc - 1; j >= 0; --j) {
    const size_t tot = static_cast<size_t>(n) * ar.c[j];
    leaky_bwd_kernel<<<static_cast<unsigned>((tot + 255) / 256), 256, 0, st>>>(g, ws + w.a[j], tot, 0.01f);
    LAUNCH_CHECK();
    const int pc = pidx_cat(ar, j);
    if (colsum(st, g, n, ar.c[j], ar.c[j], grads[pc + 1])) return 1;
    if (j > 0) {
      if (lin_wgrad(st, n, ar.c[j], ar.c[j - 1], g, ar.c[j], ws + w.a[j - 1], ar.c[j - 1], grads[pc], ar.c[j - 1], 0)) return 1;
      if (lin_dgrad(st, n, ar.c[j], ar.c[j - 1], g, ar.c[j], params[pc], ar.c[j - 1], 0, g2, ar.c[j - 1], 0)) return 1;
      float* tmp = g;
      g = g2;
      g2 = tmp;
    } else {
      const int ldw = 3 * hl + ar.ew;
      for (int b = 0; b < 3; ++b)
        if (lin_wgrad(st, n, ar.c[0], hl, g, ar.c[0], ws + w.xb[b][ar.nb - 1], hl, grads[pc], ldw, b * hl)) return 1;
      if (lin_wgrad(st, n, ar.c[0], ar.ew, g, ar.c[0], E, ar.ew, grads[pc], ldw, 3 * hl)) return 1;
    }
  }
  // g = d(pre-activation of cat_layers.0) [n, c0]; branches
  const float* gc0 = g;
  float* gb = g2;                       // gradient of the current branch layer's output ...
  float* gb_alt = ws + w.g2;            // ... and of the layer below it
  const int ed[3] = {ar.ed(0), ar.ed(1), ar.ed(2)}, eo[3] = {ar.eo(0), ar.eo(1), ar.eo(2)};
  const int pc0 = pidx_cat(ar, 0);
  const int ldw0 = 3 * hl + ar.ew;
  for (int b = 0; b < 3; ++b) {
    const float* e = E + eo[b];
    // d x_b,last = gc0 * W_cat0[:, b*hl : (b+1)*hl]
    if (lin_dgrad(st, n, ar.c[0], hl, gc0, ar.c[0], params[pc0], ldw0, b * hl, gb, hl, 0)) return 1;
    float* cur = gb;
    for (int i = ar.nb - 1; i >= 0; --i) {
      const int pb = pidx_branch(ar, b, i);
      const int prev_w = i == 0 ? ed[b] : ar.h[i - 1];
      const float* prev = i == 0 ? e : ws + w.xb[b][i - 1];
      const int prev_ld = i == 0 ? ar.ew : ar.h[i - 1];
      const int ldw = prev_w + ed[b];
      if (colsum(st, cur, n, ar.h[i], ar.h[i], grads[pb + 1])) return 1;
      if (lin_wgrad(st, n, ar.h[i], prev_w, cur, ar.h[i], prev, prev_ld, grads[pb], ldw, 0)) return 1;
      if (lin_wgrad(st, n, ar.h[i], ed[b], cur, ar.h[i], e, ar.ew, grads[pb], ldw, prev_w)) return 1;
      if (i > 0) {
        float* nxt = cur == gb ? gb_alt : gb;
        if (lin_dgrad(st, n, ar.h[i], ar.h[i - 1], cur, ar.h[i], params[pb], ldw, 0, nxt, ar.h[i - 1], 0)) return 1;
        cur = nxt;
      }
    }
  }
  return 0;
}
extern "C" int b200nerf_depthnet_train_bwd(const float* const* params, int n_branch, const int* hidden, int n_cat,
                                           const int* cat_hidden, int n_rays, float near_, float far_, float* ws, const float* dz,
                                           float* const* grads, void* stream) {
  return b200nerf_depthnet_train_bwd_multires(params, n_branch, hidden, n_cat, cat_hidden, 10, n_rays, near_, far_, ws, dz, grads, stream);
}

// ---- the same backward, split at the losses ----------------------------------------------------------------------------------
// Both losses reach DepthNet through ONE scalar per ray (dz = dLoss/dz_r), and the backward is linear in it:
//   dLoss/d(pre_j)[r, :] = dz_r J_j[r, :],   J_j = d z / d(pre-activation of cat layer j)   (dz-independent).
// The layer-by-layer input-gradient chain -- the sequential part -- therefore runs with a unit upstream gradient BEFORE the losses
// are known (b200nerf_depthnet_train_jac: beside the frozen target render, off the step's critical path), and what remains after
// the losses are INDEPENDENT products,  dW_j = sum_r (dz_r J_j[r, :])^T x_{j-1}[r, :],  db_j = sum_r dz_r J_j[r, :],  one grouped
// launch with dz applied to the k (ray) index of the A operand in the loader (tgemm `kscale`), then the weight-only branch chain.
static bool split_backward_ok(const DnArch& ar, int n, const float* const* params) {
  return tensor_path_ok(n) && can_collapse(ar, n, params);
}
extern "C" int b200nerf_depthnet_train_jac_multires(const float* const* params, int n_branch, const int* hidden, int n_cat,
                                                    const int* cat_hidden, int multires, int n_rays, float near_, float far_, float* ws,
                                                    float* const* grads, void* stream) {
  if (n_rays <= 0) return 0;
  if (!params || !ws || !grads) return b200_fail("b200nerf_depthnet_train_jac: null argument");
  DnArch ar;
  if (dn_arch(n_branch, hidden, n_cat, cat_hidden, multires, &ar)) return 1;
  if (!split_backward_ok(ar, n_rays, params)) return 0;   // b200nerf_depthnet_train_bwd_jac then runs the one-pass backward
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int n = n_rays;
  const DnWs w = dn_layout(ar, n);
  const int cl = ar.c[ar.nc - 1], hl = ar.h[ar.nb - 1];
  const int ph = pidx_head(ar);
  if (zero_grads(ar, grads, st)) return 1;
  CUDA_TRY(cudaMemsetAsync(ws + w.G[0], 0, (w.gv[2] + CH_MAXH - w.G[0]) * sizeof(float), st));
  if (fused_chain_ok(ar, n, params)) {
    // the whole chain in one launch over the transposed images the forward pass packed; step t turns J_{nc-1-t} into J_{nc-2-t}
    const int nl = ar.nc - 1;
    float* save[B200_CATCHAIN_MAX_LAYERS];
    for (int t = 0; t < nl; ++t) save[t] = ws + w.jac[ar.nc - 2 - t];
    if (b200_catchain_jac(ws + w.img_jac, ws + w.aux, nl, ws + w.s, n, near_, far_, ws + w.jac[ar.nc - 1], save,
                          reinterpret_cast<const unsigned long long*>(ws + w.mask), st))
      return 1;
  } else {
    depth_head_bwd_fused_kernel<<<(n + HEAD_ROWS - 1) / HEAD_ROWS, 256, 0, st>>>(nullptr, ws + w.s, ws + w.a[ar.nc - 1], params[ph], n, cl, near_,
                                                                              far_, 0.01f, ws + w.jac[ar.nc - 1], nullptr, nullptr);
    LAUNCH_CHECK();
    for (int j = ar.nc - 1; j >= 1; --j) {
      const int pc = pidx_cat(ar, j);
      GemmProb q = prob_dgrad(n, ar.c[j], ar.c[j - 1], ws + w.jac[j], ar.c[j], params[pc], ar.c[j - 1], 0, ws + w.jac[j - 1], ar.c[j - 1],
                              ws + w.a[j - 1], ar.c[j - 1], 0.01f);
      if (tgemm_group(st, &q, 1)) return 1;
    }
  }
  const int pc0 = pidx_cat(ar, 0), ldw0 = 3 * hl + ar.ew;
  GemmProb q[3];
  for (int b = 0; b < 3; ++b) q[b] = prob_dgrad(n, ar.c[0], hl, ws + w.jac[0], ar.c[0], params[pc0], ldw0, b * hl, ws + w.gx[2 * b], hl);
  return tgemm_group(st, q, 3);
}
extern "C" int b200nerf_depthnet_train_jac(const float* const* params, int n_branch, const int* hidden, int n_cat, const int* cat_hidden,
                                           int n_rays, float near_, float far_, float* ws, float* const* grads, void* stream) {
  return b200nerf_depthnet_train_jac_multires(params, n_branch, hidden, n_cat, cat_hidden, 10, n_rays, near_, far_, ws, grads, stream);
}
// fork / join events of the split backward's second stream, one pair per device and host thread
static int fork_events(cudaEvent_t* fork, cudaEvent_t* join) {
  static thread_local cudaEvent_t ev[B200_MAX_DEVICES][2] = {};
  const int dev = b200_device();
  if (dev < 0) return b200_fail("split backward: no usable CUDA device");
  for (int i = 0; i < 2; ++i)
    if (!ev[dev][i]) CUDA_TRY(cudaEventCreateWithFlags(&ev[dev][i], cudaEventDisableTiming));
  *fork = ev[dev][0];
  *join = ev[dev][1];
  return 0;
}
extern "C" int b200nerf_depthnet_train_bwd_jac_multires(const float* const* params, int n_branch, const int* hidden, int n_cat,
                                                        const int* cat_hidden, int multires, int n_rays, float near_, float far_, float* ws,
                                                        const float* dz, float* const* grads, void* stream, void* stream_aux) {
  if (n_rays <= 0) return 0;
  if (!params || !ws || !dz || !grads) return b200_fail("b200nerf_depthnet_train_bwd_jac: null argument");
  DnArch ar;
  if (dn_arch(n_branch, hidden, n_cat, cat_hidden, multires, &ar)) return 1;
  if (!split_backward_ok(ar, n_rays, params))
    return b200nerf_depthnet_train_bwd_multires(params, n_branch, hidden, n_cat, cat_hidden, multires, n_rays, near_, far_, ws, dz, grads,
                                                stream);
  cudaStream_t st = static_cast<cudaStream_t>(stream), sa = static_cast<cudaStream_t>(stream_aux);
  const bool fork = sa != nullptr && sa != st;
  const int n = n_rays;
  const DnWs w = dn_layout(ar, n);
  const float* E = ws + w.E;
  const int cl = ar.c[ar.nc - 1], hl = ar.h[ar.nb - 1];
  const int ph = pidx_head(ar);
  const int ed[3] = {ar.ed(0), ar.ed(1), ar.ed(2)}, eo[3] = {ar.eo(0), ar.eo(1), ar.eo(2)};
  auto launch_all = [&](std::vector<GemmProb>& q) -> int {
    for (GemmProb& p : q) p.kscale = dz;
    for (size_t i = 0; i < q.size(); i += b200::tg::MAX_PROB) {
      const int cnt = static_cast<int>(q.size() - i < static_cast<size_t>(b200::tg::MAX_PROB) ? q.size() - i : b200::tg::MAX_PROB);
      if (tgemm_group(st, q.data() + i, cnt)) return 1;
    }
    return 0;
  };
  // the branches' one reduction over the rays: G_b = D_b^T e_b, g_b = D_b^T 1 with D_b = dz * (J_0 W_cat0[:, b]) (pre-zeroed by _jac)
  std::vector<GemmProb> qg, q;
  for (int b = 0; b < 3; ++b)
    qg.push_back(prob_wgrad(n, hl, ed[b], ws + w.gx[2 * b], hl, E + eo[b], ar.ew, ws + w.G[b], CH_LD, 0, ws + w.gv[b], true));
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  if (fork) {
    // The weight-only branch chain (chain_bwd + chain_du: ~100 us on 64 SMs, whatever the batch) needs only G: it runs on the second
    // stream beside the cat layers' weight gradients instead of after them.
    if (fork_events(&ev_fork, &ev_join)) return 1;
    if (launch_all(qg)) return 1;
    CUDA_TRY(cudaEventRecord(ev_fork, st));
    CUDA_TRY(cudaStreamWaitEvent(sa, ev_fork, 0));
    if (chain_backward(ar, w, ws, params, grads, sa)) return 1;
    CUDA_TRY(cudaEventRecord(ev_join, sa));
  }
  depth_head_bwd_fused_kernel<<<(n + HEAD_ROWS - 1) / HEAD_ROWS, 256, 0, st>>>(dz, ws + w.s, ws + w.a[ar.nc - 1], params[ph], n, cl, near_,
                                                                            far_, 0.01f, nullptr, grads[ph], grads[ph + 1]);
  LAUNCH_CHECK();
  for (int j = ar.nc - 1; j >= 1; --j) {
    const int pc = pidx_cat(ar, j);
    q.push_back(prob_wgrad(n, ar.c[j], ar.c[j - 1], ws + w.jac[j], ar.c[j], ws + w.a[j - 1], ar.c[j - 1], grads[pc], ar.c[j - 1], 0, grads[pc + 1], true));
  }
  const int pc0 = pidx_cat(ar, 0), ldw0 = 3 * hl + ar.ew;
  for (int b = 0; b < 3; ++b)
    q.push_back(prob_wgrad(n, ar.c[0], hl, ws + w.jac[0], ar.c[0], ws + w.xb[b][ar.nb - 1], hl, grads[pc0], ldw0, b * hl,
                           b == 0 ? grads[pc0 + 1] : nullptr, true));
  q.push_back(prob_wgrad(n, ar.c[0], ar.ew, ws + w.jac[0], ar.c[0], E, ar.ew, grads[pc0], ldw0, 3 * hl, nullptr, true));
  if (!fork) q.insert(q.end(), qg.begin(), qg.end());
  if (launch_all(q)) return 1;
  if (fork) {
    CUDA_TRY(cudaStreamWaitEvent(st, ev_join, 0));
    return 0;
  }
  return chain_backward(ar, w, ws, params, grads, st);
}
extern "C" int b200nerf_depthnet_train_bwd_jac(const float* const* params, int n_branch, const int* hidden, int n_cat,
                                               const int* cat_hidden, int n_rays, float near_, float far_, float* ws, const float* dz,
                                               float* const* grads, void* stream, void* stream_aux) {
  return b200nerf_depthnet_train_bwd_jac_multires(params, n_branch, hidden, n_cat, cat_hidden, 10, n_rays, near_, far_, ws, dz, grads, stream,
                                                  stream_aux);
}

// ------------------------------------------------------------------------------------------- NeRF at S samples per ray + d/dz
// rows 0..n-1 = primal gamma(p), rows n..2n-1 = tangent d gamma(p) / dz, p = o + d z, row width d = 3 (1 + 2 nf); view encoding
// [n, dv], dv = 3 (1 + 2 nv).  n = n_rays * S rows; row i belongs to ray i / S.  Six threads per row: three position channels
// (nf sincosf each) and three view-direction channels (nv).
__global__ void nerf_point_encode_kernel(const float* __restrict__ ro, const float* __restrict__ rd, const float* __restrict__ vd,
                                         const float* __restrict__ z, int n, int S, int nf, int nv, float* __restrict__ enc,
                                         float* __restrict__ venc) {
  const long long t = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int i = static_cast<int>(t / 6), c = static_cast<int>(t % 3);
  if (i >= n) return;
  const size_t ray = static_cast<size_t>(i / S);
  if (t % 6 < 3) {
    const int d3 = 3 * (1 + 2 * nf);
    const float d = rd[ray * 3 + c];
    const float x = __fadd_rn(ro[ray * 3 + c], __fmul_rn(d, z[i]));
    float* p = enc + static_cast<size_t>(i) * d3;
    float* tg = enc + static_cast<size_t>(n + i) * d3;
    p[c] = x;
    tg[c] = d;
    for (int j = 0; j < nf; ++j) {
      const float f = static_cast<float>(1 << j);
      float s, co;
      sincosf(x * f, &s, &co);
      p[3 + j * 6 + c] = s;
      p[3 + j * 6 + 3 + c] = co;
      tg[3 + j * 6 + c] = f * co * d;
      tg[3 + j * 6 + 3 + c] = -f * s * d;
    }
  } else {
    const float v = vd[ray * 3 + c];
    float* e = venc + static_cast<size_t>(i) * (3 * (1 + 2 * nv));
    e[c] = v;
    for (int j = 0; j < nv; ++j) {
      float s, co;
      sincosf(v * static_cast<float>(1 << j), &s, &co);
      e[3 + j * 6 + c] = s;
      e[3 + j * 6 + 3 + c] = co;
    }
  }
}
// primal rows: h = relu(y + b); tangent rows: t = (y_primal + b > 0) ? y_tangent : 0        (in place, Y is [2n, M])
__global__ void relu_jvp_kernel(float* __restrict__ Y, const float* __restrict__ bias, int n, int M, int relu) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<size_t>(n) * M) return;
  const int m = static_cast<int>(i % M);
  const float yp = Y[i] + bias[m];
  const size_t it = i + static_cast<size_t>(n) * M;
  if (relu) {
    Y[i] = fmaxf(yp, 0.f);
    if (!(yp > 0.f)) Y[it] = 0.f;
  } else {
    Y[i] = yp;
  }
}
// raw = [rgb(3), alpha] primal + bias; draw = tangents
__global__ void nerf_point_out_kernel(const float* __restrict__ rgb2, const float* __restrict__ al2, const float* __restrict__ b_rgb,
                                      const float* __restrict__ b_al, int n, float* __restrict__ raw, float* __restrict__ draw) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  for (int c = 0; c < 3; ++c) {
    raw[i * 4 + c] = rgb2[i * 3 + c] + b_rgb[c];
    draw[i * 4 + c] = rgb2[(n + i) * 3 + c];
  }
  raw[i * 4 + 3] = al2[i] + b_al[0];
  draw[i * 4 + 3] = al2[n + i];
}

// raw = [rgb_linear(hv) + b (3), alpha_linear(h7) + b], draw = the same heads applied to the tangents (no bias)
__global__ void nerf_point_heads_kernel(const float* __restrict__ h7, const float* __restrict__ t7, const float* __restrict__ hv,
                                        const float* __restrict__ hvt, const float* __restrict__ wa, const float* __restrict__ ba,
                                        const float* __restrict__ wr, const float* __restrict__ br, int n, float* __restrict__ raw,
                                        float* __restrict__ draw) {
  const int ray = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (ray >= n) return;
  float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // rgb (3), alpha, d rgb (3), d alpha
  const float* a = h7 + static_cast<size_t>(ray) * 256;
  const float* at = t7 + static_cast<size_t>(ray) * 256;
  for (int c = lane; c < 256; c += 32) {
    const float w = __ldg(wa + c);
    v[3] = fmaf(a[c], w, v[3]);
    v[7] = fmaf(at[c], w, v[7]);
  }
  const float* b = hv + static_cast<size_t>(ray) * 128;
  const float* bt = hvt + static_cast<size_t>(ray) * 128;
  for (int c = lane; c < 128; c += 32) {
    const float x = b[c], xt = bt[c];
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
      const float w = __ldg(wr + ch * 128 + c);
      v[ch] = fmaf(x, w, v[ch]);
      v[4 + ch] = fmaf(xt, w, v[4 + ch]);
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) v[i] += __shfl_xor_sync(0xffffffffu, v[i], off);
  if (lane == 0) {
    *reinterpret_cast<float4*>(raw + static_cast<size_t>(ray) * 4) = make_float4(v[0] + __ldg(br), v[1] + __ldg(br + 1), v[2] + __ldg(br + 2), v[3] + __ldg(ba));
    *reinterpret_cast<float4*>(draw + static_cast<size_t>(ray) * 4) = make_float4(v[4], v[5], v[6], v[7]);
  }
}

static bool nerf_point_multires_ok(int multires, int multires_views) {
  return multires >= 1 && multires <= 10 && multires_views >= 1 && multires_views <= 4;
}
// the layout holds the widest encodings (d <= 64, dv <= 32), so the size does not depend on multires / multires_views
extern "C" size_t b200nerf_nerf_samples_ws_floats_multires(int n_rays, int S, int multires, int multires_views) {
  if (!nerf_point_multires_ok(multires, multires_views)) {
    b200_fail("b200nerf_nerf_point_ws_floats: multires=%d / multires_views=%d out of range (multires 1..10, multires_views 1..4)",
              multires, multires_views);
    return 0;
  }
  if (n_rays < 0 || S < 1) {
    b200_fail("b200nerf_nerf_samples_ws_floats: bad sizes n_rays=%d S=%d", n_rays, S);
    return 0;
  }
  const size_t n = static_cast<size_t>(n_rays) * static_cast<size_t>(S);
  return 2 * n * 64 + n * 32 + 3 * (2 * n * 256) + 2 * n * 4 + 2 * n + 256;
}
extern "C" size_t b200nerf_nerf_point_ws_floats_multires(int n_rays, int multires, int multires_views) {
  return b200nerf_nerf_samples_ws_floats_multires(n_rays, 1, multires, multires_views);
}
extern "C" size_t b200nerf_nerf_point_ws_floats(int n_rays) { return b200nerf_nerf_point_ws_floats_multires(n_rays, 10, 4); }

// params: the 24 fp32 device tensors of NeRF in state_dict order (see b200nerf_nerf_pack) at multires / multires_views:
// pts_linears.0 is [256, d], pts_linears.5 [256, d + 256], views_linears.0 [128, 256 + dv]
// S samples per ray: z [n_rays, S], out_raw / out_draw_dz [n_rays * S, 4]; every product runs over the n_rays * S rows
extern "C" int b200nerf_nerf_samples_jvp_multires(const float* const* t, int multires, int multires_views, const float* rays_o,
                                                  const float* rays_d, const float* viewdirs, const float* z, int n_rays, int S,
                                                  float* ws, float* out_raw, float* out_draw_dz, void* stream) {
  if (!nerf_point_multires_ok(multires, multires_views))
    return b200_fail("b200nerf_nerf_point_jvp: multires=%d / multires_views=%d out of range (multires 1..10, multires_views 1..4)",
                     multires, multires_views);
  if (S < 1) return b200_fail("b200nerf_nerf_samples_jvp: S=%d; S >= 1 is required", S);
  if (n_rays <= 0) return 0;
  if (static_cast<long long>(n_rays) * S > (1ll << 26))   // 2^26 rows need ~460 GB of workspace; the row indices stay in int
    return b200_fail("b200nerf_nerf_samples_jvp: n_rays * S = %lld rows exceed 2^26", static_cast<long long>(n_rays) * S);
  if (!t || !rays_o || !rays_d || !viewdirs || !z || !ws || !out_raw || !out_draw_dz) return b200_fail("b200nerf_nerf_point_jvp: null argument");
  const int d = 3 * (1 + 2 * multires), dv = 3 * (1 + 2 * multires_views), ld5 = 256 + d, ldv = 256 + dv;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int n = n_rays * S, n2 = 2 * n;
  float* enc = ws;                                   // [2n, d]
  float* venc = enc + static_cast<size_t>(n2) * 64;  // [n, dv]
  float* h0 = venc + static_cast<size_t>(n) * 32;    // [2n, 256]
  float* h1 = h0 + static_cast<size_t>(n2) * 256;
  float* h2 = h1 + static_cast<size_t>(n2) * 256;
  float* rgb2 = h2 + static_cast<size_t>(n2) * 256;  // [2n, 3]
  float* al2 = rgb2 + static_cast<size_t>(n2) * 4;   // [2n]
  nerf_point_encode_kernel<<<static_cast<unsigned>((6ll * n + 191) / 192), 192, 0, st>>>(rays_o, rays_d, viewdirs, z, n, S, multires,
                                                                                         multires_views, enc, venc);
  LAUNCH_CHECK();
  auto act = [&](float* Y, const float* bias, int M, int relu) -> int {
    const size_t tot = static_cast<size_t>(n) * M;
    relu_jvp_kernel<<<static_cast<unsigned>((tot + 255) / 256), 256, 0, st>>>(Y, bias, n, M, relu);
    LAUNCH_CHECK();
    return 0;
  };
  if (tgemm_enabled() && n >= 32) {
    // Tensor-core path, every epilogue fused: the primal row block runs Linear + bias + ReLU as one problem, the tangent row block
    // W t_{k-1} masked by the primal's post-activation (the `dact` epilogue with slope 0 IS relu_jvp's mask).  The tangent of layer
    // k-1 needs the primal of layer k-1, so launch k carries {primal layer k, tangent layer k-1}: 11 grouped launches instead of
    // 13 products + 11 activation launches.
    const size_t blk = static_cast<size_t>(n) * 256;
    float* hp[2] = {h0, h0 + blk};          // primal ping-pong
    float* ht[2] = {h1, h1 + blk};          // tangent ping-pong
    float* feat = h2;                       // feature_linear(h7) primal, then its tangent next to it
    float* feat_t = h2 + blk;
    const float* enc_t = enc + static_cast<size_t>(n) * d;
    auto primal = [&](int layer, const float* x, float* y) {
      GemmProb q = prob_fwd(n, 256, y, 256, t[2 * layer + 1], 1, 0.f);
      if (layer == 0) {
        seg_fwd(q, enc, d, t[0], d, 0, d);
      } else if (layer == 5) {
        seg_fwd(q, enc, d, t[10], ld5, 0, d);
        seg_fwd(q, x, 256, t[10], ld5, d, 256);
      } else {
        seg_fwd(q, x, 256, t[2 * layer], 256, 0, 256);
      }
      return q;
    };
    auto tangent = [&](int layer, const float* xt, const float* mask, float* yt) {
      GemmProb q = prob_fwd(n, 256, yt, 256, nullptr, 0, 0.f);
      q.dact = mask;
      q.ld_dact = 256;
      q.slope = 0.f;
      if (layer == 0) {
        seg_fwd(q, enc_t, d, t[0], d, 0, d);
      } else if (layer == 5) {
        seg_fwd(q, enc_t, d, t[10], ld5, 0, d);
        seg_fwd(q, xt, 256, t[10], ld5, d, 256);
      } else {
        seg_fwd(q, xt, 256, t[2 * layer], 256, 0, 256);
      }
      return q;
    };
    {
      GemmProb q = primal(0, nullptr, hp[0]);
      if (tgemm_group(st, &q, 1)) return 1;
    }
    for (int k = 1; k <= 7; ++k) {   // h_k in hp[k & 1], t_k in ht[k & 1]
      GemmProb q[2] = {primal(k, hp[(k - 1) & 1], hp[k & 1]), tangent(k - 1, ht[k & 1], hp[(k - 1) & 1], ht[(k - 1) & 1])};
      if (tgemm_group(st, q, 2)) return 1;
    }
    {
      // feature_linear(h7) (bias, no activation) + tangent of layer 7; h7 = hp[1], t6 = ht[0] -> t7 = ht[1]
      GemmProb q[2];
      q[0] = prob_fwd(n, 256, feat, 256, t[19], 0, 0.f);
      seg_fwd(q[0], hp[1], 256, t[18], 256, 0, 256);
      q[1] = tangent(7, ht[0], hp[1], ht[1]);
      if (tgemm_group(st, q, 2)) return 1;
    }
    float* hv = hp[0];        // [n, 128] view-layer activations (h6 is dead)
    float* hv_t = ht[0];      // [n, 128]
    {
      // views_linears.0 on cat([feature, gamma(viewdir)]) + ReLU; feature tangent = W_f t7 (no mask)
      GemmProb q[2];
      q[0] = prob_fwd(n, 128, hv, 128, t[17], 1, 0.f);
      seg_fwd(q[0], feat, 256, t[16], ldv, 0, 256);
      seg_fwd(q[0], venc, dv, t[16], ldv, 256, dv);
      q[1] = prob_fwd(n, 256, feat_t, 256, nullptr, 0, 0.f);
      seg_fwd(q[1], ht[1], 256, t[18], 256, 0, 256);
      if (tgemm_group(st, q, 2)) return 1;
    }
    {
      GemmProb q = prob_fwd(n, 128, hv_t, 128, nullptr, 0, 0.f);   // the view encoding has no tangent
      q.dact = hv;
      q.ld_dact = 128;
      q.slope = 0.f;
      seg_fwd(q, feat_t, 256, t[16], ldv, 0, 256);
      if (tgemm_group(st, &q, 1)) return 1;
    }
    // alpha_linear(h7) / rgb_linear(hv) and their tangents: eight dot products per ray, one warp per ray
    nerf_point_heads_kernel<<<(n + 7) / 8, 256, 0, st>>>(hp[1], ht[1], hv, hv_t, t[20], t[21], t[22], t[23], n, out_raw, out_draw_dz);
    LAUNCH_CHECK();
    return 0;
  }
  float* cur = h0;
  float* nxt = h1;
  // run_nerf_helpers.py:109-134: h = relu(L_i(h)); after layer 4, h = cat([input_pts, h])
  if (lin_fwd(st, n2, 256, d, enc, d, t[0], d, 0, cur, 256, 0, nullptr, 0, 0.f)) return 1;
  if (act(cur, t[1], 256, 1)) return 1;
  for (int i = 1; i < 8; ++i) {
    if (i == 5) {
      if (lin_fwd(st, n2, 256, d, enc, d, t[10], ld5, 0, nxt, 256, 0, nullptr, 0, 0.f)) return 1;
      if (lin_fwd(st, n2, 256, 256, cur, 256, t[10], ld5, d, nxt, 256, 1, nullptr, 0, 0.f)) return 1;
    } else {
      if (lin_fwd(st, n2, 256, 256, cur, 256, t[2 * i], 256, 0, nxt, 256, 0, nullptr, 0, 0.f)) return 1;
    }
    if (act(nxt, t[2 * i + 1], 256, 1)) return 1;
    float* tmp = cur;
    cur = nxt;
    nxt = tmp;
  }
  // alpha_linear and feature_linear on h7 (no activation)
  if (lin_fwd(st, n2, 1, 256, cur, 256, t[20], 256, 0, al2, 1, 0, nullptr, 0, 0.f)) return 1;
  if (lin_fwd(st, n2, 256, 256, cur, 256, t[18], 256, 0, nxt, 256, 0, nullptr, 0, 0.f)) return 1;
  if (act(nxt, t[19], 256, 0)) return 1;
  // views_linears.0 on cat([feature, gamma(viewdir)]): the view part has no tangent
  if (lin_fwd(st, n2, 128, 256, nxt, 256, t[16], ldv, 0, h2, 128, 0, nullptr, 0, 0.f)) return 1;
  if (lin_fwd(st, n, 128, dv, venc, dv, t[16], ldv, 256, h2, 128, 1, nullptr, 0, 0.f)) return 1;
  if (act(h2, t[17], 128, 1)) return 1;
  if (lin_fwd(st, n2, 3, 128, h2, 128, t[22], 128, 0, rgb2, 3, 0, nullptr, 0, 0.f)) return 1;
  nerf_point_out_kernel<<<(n + 255) / 256, 256, 0, st>>>(rgb2, al2, t[23], t[21], n, out_raw, out_draw_dz);
  LAUNCH_CHECK();
  return 0;
}

extern "C" int b200nerf_nerf_point_jvp_multires(const float* const* t, int multires, int multires_views, const float* rays_o,
                                                const float* rays_d, const float* viewdirs, const float* z, int n_rays, float* ws,
                                                float* out_raw, float* out_draw_dz, void* stream) {
  return b200nerf_nerf_samples_jvp_multires(t, multires, multires_views, rays_o, rays_d, viewdirs, z, n_rays, 1, ws, out_raw,
                                            out_draw_dz, stream);
}

extern "C" int b200nerf_nerf_point_jvp(const float* const* t, const float* rays_o, const float* rays_d, const float* viewdirs,
                                       const float* z, int n_rays, float* ws, float* out_raw, float* out_draw_dz, void* stream) {
  return b200nerf_nerf_point_jvp_multires(t, 10, 4, rays_o, rays_d, viewdirs, z, n_rays, ws, out_raw, out_draw_dz, stream);
}

// ------------------------------------------------------------------------------------------- Adam
// torch.optim.Adam (no weight decay, no amsgrad) on one tensor:
//   m = b1 m + (1-b1) g;  v = b2 v + (1-b2) g^2;  p -= lr/(1-b1^t) * m / (sqrt(v)/sqrt(1-b2^t) + eps)
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                            size_t n, float lr, float b1, float b2, float eps, float bc1, float bc2_sqrt, float gscale) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float gi = g[i] * gscale;
  const float mi = b1 * m[i] + (1.f - b1) * gi;
  const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
  m[i] = mi;
  v[i] = vi;
  const float denom = sqrtf(vi) / bc2_sqrt + eps;
  p[i] -= (lr / bc1) * (mi / denom);
}
// The same update over a list of tensors in ONE launch: blockIdx.y walks the tensors of the table.
struct AdamEntry {
  float* p;
  const float* g;
  float* m;
  float* v;
  unsigned long long n;
};
__global__ void adam_multi_kernel(const AdamEntry* __restrict__ table, float lr, float b1, float b2, float eps, float bc1,
                                  float bc2_sqrt, float gscale) {
  const AdamEntry e = table[blockIdx.y];
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < e.n; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float gi = e.g[i] * gscale;
    const float mi = b1 * e.m[i] + (1.f - b1) * gi;
    const float vi = b2 * e.v[i] + (1.f - b2) * gi * gi;
    e.m[i] = mi;
    e.v[i] = vi;
    e.p[i] -= (lr / bc1) * (mi / (sqrtf(vi) / bc2_sqrt + eps));
  }
}
/* d_table: device array of n_tensors {param, grad, exp_avg, exp_avg_sq, numel} records (5 x 8 bytes each) */
extern "C" int b200nerf_adam_step_multi(const void* d_table, int n_tensors, float lr, float beta1, float beta2, float eps, int step,
                                        float grad_scale, void* stream) {
  if (n_tensors <= 0) return 0;
  if (!d_table || step < 1) return b200_fail("b200nerf_adam_step_multi: bad arguments");
  const float bc1 = 1.f - powf(beta1, static_cast<float>(step));
  const float bc2 = 1.f - powf(beta2, static_cast<float>(step));
  adam_multi_kernel<<<dim3(64, n_tensors), 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const AdamEntry*>(d_table), lr, beta1,
                                                                                      beta2, eps, bc1, sqrtf(bc2), grad_scale);
  LAUNCH_CHECK();
  return 0;
}

// CUDA-graph friendly variant: the step counter lives on the device and the hyper-parameters are read from device memory
// (d_hyper = {lr, beta1, beta2, eps, grad_scale}), so a captured launch stays valid while lr / step change.
__global__ void adam_tick_kernel(int* step) { *step += 1; }
__device__ __forceinline__ void adam_update(float& p, float g, float& m, float& v, float lr_bc1, float b1, float b2, float eps,
                                            float bc2_sqrt, float gscale) {
  const float gi = g * gscale;
  const float mi = b1 * m + (1.f - b1) * gi;
  const float vi = b2 * v + (1.f - b2) * gi * gi;
  m = mi;
  v = vi;
  p -= lr_bc1 * (mi / (sqrtf(vi) / bc2_sqrt + eps));
}
// 16-byte accesses where the four arrays of a tensor allow it (they do for every DepthNet tensor: 13.4 MB of parameters, 94 MB of
// traffic per step), scalar tail / scalar path otherwise
__global__ void adam_multi_dev_kernel(const AdamEntry* __restrict__ table, const float* __restrict__ hyper, const int* __restrict__ step) {
  const AdamEntry e = table[blockIdx.y];
  const float lr = hyper[0], b1 = hyper[1], b2 = hyper[2], eps = hyper[3], gscale = hyper[4];
  const float t = static_cast<float>(*step);
  const float bc1 = 1.f - powf(b1, t), bc2_sqrt = sqrtf(1.f - powf(b2, t));
  const float lr_bc1 = lr / bc1;
  const size_t tid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x, nthr = static_cast<size_t>(gridDim.x) * blockDim.x;
  const bool vec = ((reinterpret_cast<uintptr_t>(e.p) | reinterpret_cast<uintptr_t>(e.g) | reinterpret_cast<uintptr_t>(e.m) |
                     reinterpret_cast<uintptr_t>(e.v)) & 15) == 0;
  const size_t n4 = vec ? e.n / 4 : 0;
  for (size_t i = tid; i < n4; i += nthr) {
    float4 p4 = reinterpret_cast<float4*>(e.p)[i], m4 = reinterpret_cast<float4*>(e.m)[i], v4 = reinterpret_cast<float4*>(e.v)[i];
    const float4 g4 = reinterpret_cast<const float4*>(e.g)[i];
    adam_update(p4.x, g4.x, m4.x, v4.x, lr_bc1, b1, b2, eps, bc2_sqrt, gscale);
    adam_update(p4.y, g4.y, m4.y, v4.y, lr_bc1, b1, b2, eps, bc2_sqrt, gscale);
    adam_update(p4.z, g4.z, m4.z, v4.z, lr_bc1, b1, b2, eps, bc2_sqrt, gscale);
    adam_update(p4.w, g4.w, m4.w, v4.w, lr_bc1, b1, b2, eps, bc2_sqrt, gscale);
    reinterpret_cast<float4*>(e.p)[i] = p4;
    reinterpret_cast<float4*>(e.m)[i] = m4;
    reinterpret_cast<float4*>(e.v)[i] = v4;
  }
  for (size_t i = n4 * 4 + tid; i < e.n; i += nthr) adam_update(e.p[i], e.g[i], e.m[i], e.v[i], lr_bc1, b1, b2, eps, bc2_sqrt, gscale);
}
extern "C" int b200nerf_adam_step_multi_dev(const void* d_table, int n_tensors, const float* d_hyper, int* d_step, void* stream) {
  if (n_tensors <= 0) return 0;
  if (!d_table || !d_hyper || !d_step) return b200_fail("b200nerf_adam_step_multi_dev: null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  adam_tick_kernel<<<1, 1, 0, st>>>(d_step);
  LAUNCH_CHECK();
  adam_multi_dev_kernel<<<dim3(64, n_tensors), 256, 0, st>>>(static_cast<const AdamEntry*>(d_table), d_hyper, d_step);
  LAUNCH_CHECK();
  return 0;
}

extern "C" int b200nerf_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, size_t n, float lr, float beta1,
                                  float beta2, float eps, int step, float grad_scale, void* stream) {
  if (n == 0) return 0;
  if (!param || !grad || !exp_avg || !exp_avg_sq || step < 1) return b200_fail("b200nerf_adam_step: bad arguments");
  const float bc1 = 1.f - powf(beta1, static_cast<float>(step));
  const float bc2 = 1.f - powf(beta2, static_cast<float>(step));
  adam_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, bc1, sqrtf(bc2), grad_scale);
  LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------- training losses
// Trainer.core_optimization_loop (Trainer.py:525-538) for the DepthNet path: img_loss = mean((rgb - target)^2) with
// rgb = sigmoid(raw rgb) (one sample per ray: the S == 1 quirk of raw2outputs), depth_net_loss = mean((z_dn - max_z)^2),
// psnr = -10 log10(img_loss), and the gradient both losses send into z_dn -- d(depth loss)/dz + d(img loss)/d rgb * rgb(1-rgb) *
// d raw / dz (the forward-mode tangent of b200nerf_nerf_point_jvp) -- in one pass instead of ~20 elementwise autograd launches.
__global__ void __launch_bounds__(256) train_loss_kernel(const float* __restrict__ raw, const float* __restrict__ draw,
                                                         const float* __restrict__ z, const float* __restrict__ max_z,
                                                         const float* __restrict__ target, int n, float* __restrict__ acc,
                                                         float* __restrict__ dz) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  float img = 0.f, dn = 0.f;
  if (i < n) {
    const float4 r = __ldg(reinterpret_cast<const float4*>(raw) + i), dr = __ldg(reinterpret_cast<const float4*>(draw) + i);
    const float rr[3] = {r.x, r.y, r.z}, dd[3] = {dr.x, dr.y, dr.z};
    const float dzv = z[i] - max_z[i];
    dn = dzv * dzv;
    float gz = 2.0f * dzv / static_cast<float>(n);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float rgb = 1.0f / (1.0f + expf(-rr[c]));
      const float diff = rgb - target[i * 3 + c];
      img = fmaf(diff, diff, img);
      gz = fmaf(2.0f * diff / (3.0f * static_cast<float>(n)) * rgb * (1.0f - rgb), dd[c], gz);
    }
    dz[i] = gz;
  }
  __shared__ float red[2][8];
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    img += __shfl_xor_sync(0xffffffffu, img, off);
    dn += __shfl_xor_sync(0xffffffffu, dn, off);
  }
  if ((threadIdx.x & 31) == 0) {
    red[0][threadIdx.x >> 5] = img;
    red[1][threadIdx.x >> 5] = dn;
  }
  __syncthreads();
  if (threadIdx.x < 2) {
    float t = 0.f;
    for (int k = 0; k < 8; ++k) t += red[threadIdx.x][k];
    atomicAdd(acc + threadIdx.x, t);
  }
}
__global__ void train_loss_finish_kernel(const float* __restrict__ acc, int n, float* __restrict__ out) {
  const float img = acc[0] / (3.0f * static_cast<float>(n));
  out[0] = img;
  out[1] = acc[1] / static_cast<float>(n);
  out[2] = -10.0f * logf(img) / logf(10.0f);
}
extern "C" int b200nerf_train_loss(const float* raw, const float* draw_dz, const float* z_dn, const float* max_z, const float* target,
                                   int n_rays, float* ws2, float* out_losses, float* out_dz, void* stream) {
  if (n_rays <= 0) return b200_fail("b200nerf_train_loss: empty batch");
  if (!raw || !draw_dz || !z_dn || !max_z || !target || !ws2 || !out_losses || !out_dz) return b200_fail("b200nerf_train_loss: null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUDA_TRY(cudaMemsetAsync(ws2, 0, 2 * sizeof(float), st));
  train_loss_kernel<<<(n_rays + 255) / 256, 256, 0, st>>>(raw, draw_dz, z_dn, max_z, target, n_rays, ws2, out_dz);
  LAUNCH_CHECK();
  train_loss_finish_kernel<<<1, 1, 0, st>>>(ws2, n_rays, out_losses);
  LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------- diagnostics
/* The strided GEMM of the training slice (tensor-core 3xTF32 path unless B200NERF_TRAIN_GEMM=fp32, or force_fp32 != 0),
   exposed so that a GPU test can pin it against torch on every operand layout the training passes use. */
extern "C" int b200nerf_debug_sgemm(int M, int N, int K, const float* A, long sAm, long sAk, const float* B, long sBk, long sBn, float* C,
                                    int ldc, int beta, const float* bias, int act, float slope, int force_fp32, void* stream) {
  if (!A || !B || !C || M < 0 || N < 0 || K < 0) return b200_fail("b200nerf_debug_sgemm: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!force_fp32) return sgemm(st, M, N, K, A, sAm, sAk, B, sBk, sBn, C, ldc, beta, bias, act, slope);
  if (M <= 0 || N <= 0) return 0;
  dim3 grid((N + GN - 1) / GN, (M + GM - 1) / GM);
  sgemm_kernel<<<grid, 256, 0, st>>>(M, N, K, A, sAm, sAk, B, sBk, sBn, C, ldc, beta, bias, act, slope);
  LAUNCH_CHECK();
  return 0;
}

/* Which kernels the DepthNet training passes pick for this architecture, batch and parameter alignment, from the same predicates the
   passes call (pure host code: only the pointer VALUES are read, nothing is launched). */
extern "C" int b200nerf_debug_depthnet_train_route_multires(const float* const* params, int n_branch, const int* hidden, int n_cat,
                                                            const int* cat_hidden, int multires, int n_rays) {
  if (!params || n_rays < 0) return -b200_fail("b200nerf_debug_depthnet_train_route: bad arguments");
  DnArch ar;
  if (dn_arch(n_branch, hidden, n_cat, cat_hidden, multires, &ar)) return -1;
  for (int v : ar.h)
    if (v < 1) return -b200_fail("b200nerf_debug_depthnet_train_route: branch width %d", v);
  for (int v : ar.c)
    if (v < 1) return -b200_fail("b200nerf_debug_depthnet_train_route: cat width %d", v);
  const int n = n_rays;
  return (can_collapse(ar, n, params) ? B200NERF_ROUTE_COLLAPSED : 0) | (fused_chain_ok(ar, n, params) ? B200NERF_ROUTE_FUSED_CHAIN : 0) |
         (split_cat0(ar, n, params) ? B200NERF_ROUTE_SPLIT_CAT0 : 0) | (split_backward_ok(ar, n, params) ? B200NERF_ROUTE_SPLIT_BACKWARD : 0) |
         (tensor_path_ok(n) ? B200NERF_ROUTE_TENSOR_PATH : 0);
}
extern "C" int b200nerf_debug_depthnet_train_route(const float* const* params, int n_branch, const int* hidden, int n_cat,
                                                   const int* cat_hidden, int n_rays) {
  return b200nerf_debug_depthnet_train_route_multires(params, n_branch, hidden, n_cat, cat_hidden, 10, n_rays);
}
