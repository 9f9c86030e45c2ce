// libb200nerf.so -- C ABI + the bandwidth-bound kernels of the render_rays hot path (see include/b200nerf.h).
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <utility>
#include <vector>

#include "../../include/b200nerf.h"
#include "host_common.h"
#include "umma_selftest.cuh"
#include "mlp_exact.cuh"
#include "mlp_fast.cuh"
#include "composite_tma.cuh"
#include <cuda.h>
#include <cuda_bf16.h>

using namespace b200;

// ------------------------------------------------------------------------------------------- error plumbing
static thread_local char g_err[512] = "";
std::atomic<unsigned long long> g_b200_launches{0};

int b200_fail(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return 1;
}
#define fail b200_fail

extern "C" int b200nerf_version(void) { return B200NERF_VERSION; }
extern "C" const char* b200nerf_last_error(void) { return g_err; }
extern "C" unsigned long long b200nerf_launch_count(void) { return g_b200_launches.load(); }

// Cap of the persistent MLP grids (0 = all SMs).  A persistent kernel that owns every SM serialises anything launched on another
// stream behind it; the training step caps the frozen target render so that the latency-bound DepthNet / JVP launch chain of the
// same step runs beside it (training.fused_render_and_backward).  Per host thread, like the current device.
static thread_local int g_sm_limit = 0;
extern "C" int b200nerf_set_sm_limit(int n_sms) {
  const int prev = g_sm_limit;
  g_sm_limit = n_sms > 0 ? n_sms : 0;
  return prev;
}

static int sm_count() {
  static int n[B200_MAX_DEVICES] = {0};
  const int dev = b200_device();
  if (dev < 0) return 0;
  if (n[dev] == 0 && cudaDeviceGetAttribute(&n[dev], cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) n[dev] = 0;
  return n[dev];
}

// ------------------------------------------------------------------------------------------- host packing
static inline uint16_t f2bf(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return static_cast<uint16_t>((u >> 16) | 0x40);  // quiet NaN
  u += 0x7fffu + ((u >> 16) & 1u);
  return static_cast<uint16_t>(u >> 16);
}
static inline float bf2f(uint16_t h) {
  uint32_t u = static_cast<uint32_t>(h) << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}


// NeRF aux block (float offsets)
enum : uint32_t {
  NERF_B0 = 0, NERF_BF = 2048, NERF_BV = 2304, NERF_WA = 2432, NERF_BA = 2688, NERF_WR = 2692, NERF_BR = 3076,
  NERF_AUX_FLOATS = 3080
};

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(sym);
  }
  return fn;
}



// ------------------------------------------------------------------------------------------- pipelined exact kernel (mlp_exact.cuh)
// A program = the layer steps the kernel walks + where each operand K16 block finds its weights.  The same description
// drives packing and launching, so the stream order cannot diverge from the issue order.
struct XSeg {            // operand blocks [kb, kb+nblk) multiply W[:, col0 : col0+K] (zero beyond K)
  int kb, nblk;
  const float* W;
  int ldw, col0, K;
};
struct XLayer {
  exact::XStep st;
  int n_out;             // 256 or 128
  XSeg segs[2];
  int n_segs;
};
struct XProgram {
  std::vector<XLayer> layers;
  int stages_per_tile() const {
    int n = 0;
    for (const XLayer& l : layers) n += l.st.halves * (l.st.n1a + l.st.n1b + l.st.n2) / 2;
    return n;
  }
  size_t pack_bytes() const { return static_cast<size_t>(stages_per_tile()) * 2 * exact::STAGE_BYTES; }
};

static exact::XStep xstep(int n1a, int kb1a, int n1b, int kb1b, int n2, int kb2, int halves, int epi, int act, uint32_t bias_off) {
  exact::XStep s;
  memset(&s, 0, sizeof(s));
  s.n1a = n1a; s.kb1a = kb1a; s.n1b = n1b; s.kb1b = kb1b; s.n2 = n2; s.kb2 = kb2;
  s.halves = halves; s.epi = epi; s.act = act; s.bias_off = static_cast<uint16_t>(bias_off);
  return s;
}

// views_linears.0 with the activation-free feature_linear folded in: returns W'' [128, 256 + dv] = [W_view[:, :256] * W_feature |
// W_view[:, 256:]] (valid until the next call on this thread) and, if asked, b' = W_view[:, :256] * b_feature + b_view.
// dv = 3 (1 + 2 multires_views) is the width of gamma(viewdir) (27 at multires_views 4).
static const float* nerf_fold_view(const float* const* t, int dv, float* bias128) {
  static thread_local std::vector<float> wfold;
  const float *Wv = t[16], *bv = t[17], *Wf = t[18], *bf = t[19];
  const int ld = 256 + dv;
  wfold.resize(static_cast<size_t>(128) * ld);
  for (int r = 0; r < 128; ++r) {
    const float* wr = Wv + static_cast<size_t>(r) * ld;
    for (int k = 0; k < 256; ++k) {
      double a = 0.0;
      for (int j = 0; j < 256; ++j) a += static_cast<double>(wr[j]) * static_cast<double>(Wf[static_cast<size_t>(j) * 256 + k]);
      wfold[static_cast<size_t>(r) * ld + k] = static_cast<float>(a);
    }
    for (int k = 256; k < ld; ++k) wfold[static_cast<size_t>(r) * ld + k] = wr[k];
    if (bias128) {
      double b = static_cast<double>(bv[r]);
      for (int j = 0; j < 256; ++j) b += static_cast<double>(wr[j]) * static_cast<double>(bf[j]);
      bias128[r] = static_cast<float>(b);
    }
  }
  return wfold.data();
}

// NeRF (run_nerf_helpers.py:109-134); t = the 24 tensors in state_dict order (may be null when only the steps are needed).
// d = 3 (1 + 2 multires) and dv = 3 (1 + 2 multires_views) are the widths of gamma(pts) and gamma(viewdir): layer 0 is [256, d],
// the skip layer [256, d + 256] over cat([gamma(pts), h]), views_linears.0 [128, 256 + dv].  The encodings sit in the first d / dv
// columns of their 64 / 32-column operand blocks, so the steps (and the pack size) are those of every other multires.
static XProgram nerf_xprogram(const float* const* t, int d = 63, int dv = 27) {
  auto T = [&](int i) { return t ? t[i] : nullptr; };
  XProgram pg;
  auto add = [&](exact::XStep st, int n_out, XSeg a, XSeg b, int n_segs) {
    XLayer l;
    l.st = st; l.n_out = n_out; l.segs[0] = a; l.segs[1] = b; l.n_segs = n_segs;
    pg.layers.push_back(l);
  };
  const XSeg none = {0, 0, nullptr, 0, 0, 0};
  {
    exact::XStep s0 = xstep(4, exact::ENC_KB, 0, 0, 0, 0, 2, exact::EPI_STORE, exact::ACT_RELU, NERF_B0);
    s0.wait_p = 1;
    add(s0, 256, XSeg{exact::ENC_KB, 4, T(0), d, 0, d}, none, 1);
  }
  for (int i = 1; i <= 7; ++i) {
    if (i == 5) {
      exact::XStep s5 = xstep(8, 0, 4, exact::ENC_KB, 8, 8, 2, exact::EPI_STORE, exact::ACT_RELU, NERF_B0 + 256 * 5);
      s5.sig_p = 1;   // gamma(pts) is not read after the first range of the skip layer
      add(s5, 256, XSeg{0, 16, T(10), 256 + d, d, 256}, XSeg{exact::ENC_KB, 4, T(10), 256 + d, 0, d}, 2);
    } else {
      add(xstep(8, 0, 0, 0, 8, 8, 2, i == 7 ? exact::EPI_STORE_ALPHA : exact::EPI_STORE, exact::ACT_RELU, NERF_B0 + 256 * i), 256,
          XSeg{0, 16, T(2 * i), 256, 0, 256}, none, 1);
    }
  }
  {
    // feature_linear has no activation (run_nerf_helpers.py:116-121), so it is folded into views_linears.0 here exactly as in
    // the throughput kernel's pack: W' = W_view[:, :256] * W_feature (fp64 sums; nerf_fold_view), aux[NERF_BV] = folded bias
    exact::XStep s8 = xstep(8, 0, 2, exact::VIEW_KB, 8, 8, 1, exact::EPI_NERF_OUT, exact::ACT_RELU, NERF_BV);
    s8.wait_v = 1;
    s8.sig_v = 1;
    const float* wfold = t ? nerf_fold_view(t, dv, nullptr) : nullptr;
    add(s8, 128, XSeg{0, 16, wfold, 256 + dv, 0, 256}, XSeg{exact::VIEW_KB, 2, wfold, 256 + dv, 256, dv}, 2);
  }
  return pg;
}

// folded DepthNet: n_hidden + 1 LeakyReLU layers of 256x256 (see b200nerf_depthnet_pack)
static XProgram depthnet_xprogram(const float* w0, const float* const* hidden, int n_hidden) {
  XProgram pg;
  const XSeg none = {0, 0, nullptr, 0, 0, 0};
  for (int i = 0; i <= n_hidden; ++i) {
    XLayer l;
    l.st = xstep(8, 0, 0, 0, 8, 8, 2, i == n_hidden ? exact::EPI_DEPTH_OUT : exact::EPI_STORE, exact::ACT_LEAKY, 256u * i);
    if (i == 0) {
      l.st.wait_p = 1;   // enc(o) | enc(d) in columns 0..127
      l.st.wait_v = 2;   // enc(hits) in columns 128..255
    }
    if (i == n_hidden) {
      l.st.sig_p = 1;
      l.st.sig_v = 2;
    }
    l.n_out = 256;
    l.segs[0] = XSeg{0, 16, i == 0 ? w0 : (hidden ? hidden[2 * (i - 1)] : nullptr), 256, 0, 256};
    l.segs[1] = none;
    l.n_segs = 1;
    pg.layers.push_back(l);
  }
  return pg;
}

// pack layout [rank][stage][8 KB]; stage = two K16 blocks of one (layer, output half, K range) in issue order, each block =
// hi piece | lo piece, one piece = this rank's 64 rows of the 128-row half as [2 k chunks][8 row groups][8 rows][8 k] bf16
static int pack_xprogram(const XProgram& pg, uint8_t* out) {
  const size_t per_rank = pg.pack_bytes() / 2;
  for (int r = 0; r < 2; ++r) {
    uint8_t* o = out + r * per_rank;
    for (const XLayer& l : pg.layers) {
      auto emit_block = [&](int half, int kb) {
        const XSeg* sg = nullptr;
        for (int i = 0; i < l.n_segs; ++i)
          if (kb >= l.segs[i].kb && kb < l.segs[i].kb + l.segs[i].nblk) sg = &l.segs[i];
        uint16_t* hi = reinterpret_cast<uint16_t*>(o);
        uint16_t* lo = reinterpret_cast<uint16_t*>(o + 2048);
        for (int kc = 0; kc < 2; ++kc)
          for (int n = 0; n < 64; ++n)
            for (int e = 0; e < 8; ++e) {
              const int k = (kb - (sg ? sg->kb : 0)) * 16 + kc * 8 + e;
              const int row = half * 128 + r * 64 + n;
              float w = 0.f;
              if (sg && sg->W && k < sg->K && row < l.n_out) w = sg->W[static_cast<size_t>(row) * sg->ldw + sg->col0 + k];
              const size_t idx = static_cast<size_t>(kc) * 64 * 8 + static_cast<size_t>(n >> 3) * 64 + (n & 7) * 8 + e;
              const uint16_t h = f2bf(w);
              hi[idx] = h;
              lo[idx] = f2bf(w - bf2f(h));
            }
        o += 4096;
      };
      auto emit_range = [&](int half, int kb, int nblk) {
        for (int k = 0; k < nblk; ++k) emit_block(half, kb + k);
      };
      for (int half = 0; half < l.st.halves; ++half) {
        emit_range(half, l.st.kb1a, l.st.n1a);
        emit_range(half, l.st.kb1b, l.st.n1b);
      }
      for (int half = 0; half < l.st.halves; ++half) emit_range(half, l.st.kb2, l.st.n2);
    }
    if (static_cast<size_t>(o - (out + r * per_rank)) != per_rank) return fail("exact pack: internal size mismatch");
  }
  return 0;
}

static int make_exact_tmap(const void* wpack, size_t bytes, exact::TMap* out) {
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) return fail("cuTensorMapEncodeTiled is not available from the driver");
  const cuuint64_t gdim[2] = {256, bytes / 512};
  const cuuint64_t gstride[1] = {512};
  const cuuint32_t box[2] = {256, 16};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(reinterpret_cast<CUtensorMap*>(out), CU_TENSOR_MAP_DATA_TYPE_UINT16, 2, const_cast<void*>(wpack), gdim,
                         gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled failed (%d)", static_cast<int>(r));
  return 0;
}

template <int INPUT>
static int launch_exact(exact::ExactParams& p, const XProgram& pg, const void* wpack, cudaStream_t st) {
  static int grid_caps[B200_MAX_DEVICES] = {0};
  const int dev = b200_device();
  if (dev < 0) return fail("mlp_exact_kernel: no usable CUDA device");
  int& grid_cap = grid_caps[dev];
  constexpr int smem = exact::smem_bytes();
  auto kern = exact::mlp_exact_kernel<INPUT>;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = exact::NCTA;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.blockDim = dim3(exact::THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (grid_cap == 0) {
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const int sms = sm_count();
    if (sms <= 0) return fail("no CUDA device");
    int cap = (sms / exact::NCTA) * exact::NCTA;
    cfg.gridDim = dim3(cap);
    int n_clusters = 0;
    CUDA_TRY(cudaOccupancyMaxActiveClusters(&n_clusters, kern, &cfg));
    if (n_clusters <= 0) return fail("mlp_exact_kernel: no resident cluster fits");
    if (n_clusters * exact::NCTA < cap) cap = n_clusters * exact::NCTA;
    grid_cap = cap;
  }
  if (static_cast<int>(pg.layers.size()) > exact::MAX_STEPS) return fail("mlp_exact_kernel: too many layers");
  if (INPUT == exact::IN_DEPTHNET) {
    // per-CTA staging image of the next tile's encoded rays (128 KB per CTA, ~19 MB): library-owned, one per (device, stream) --
    // launches on different streams of a device may overlap and must not share it
    static std::mutex mu;
    static std::map<std::pair<int, cudaStream_t>, uint8_t*> scratch;
    {
      std::lock_guard<std::mutex> lock(mu);
      uint8_t*& buf = scratch[std::make_pair(dev, st)];
      if (!buf) CUDA_TRY(cudaMalloc(&buf, static_cast<size_t>(grid_cap) * 2 * 32 * exact::KC_STRIDE));
      p.scratch = buf;
    }
  }
  p.n_steps = static_cast<int>(pg.layers.size());
  for (int i = 0; i < p.n_steps; ++i) p.steps[i] = pg.layers[i].st;
  p.stages_per_tile = pg.stages_per_tile();
  const int tiles = (p.n_rows + exact::TILE_M - 1) / exact::TILE_M;
  int grid = ((tiles + exact::NCTA - 1) / exact::NCTA) * exact::NCTA;
  if (grid > grid_cap) grid = grid_cap;
  if (g_sm_limit >= exact::NCTA && grid > g_sm_limit) grid = (g_sm_limit / exact::NCTA) * exact::NCTA;
  cfg.gridDim = dim3(grid);
  exact::TMap tm;
  const int rc = make_exact_tmap(wpack, pg.pack_bytes(), &tm);
  if (rc) return rc;
  if (b200_sync_check()) {
    const cudaError_t e0 = cudaDeviceSynchronize();
    if (e0 != cudaSuccess) return fail("a kernel launched BEFORE mlp_exact_kernel (not by this library's checked launches) failed: %s", cudaGetErrorString(e0));
    // debugging aid: every pointer the kernel dereferences must lie inside a live device allocation that covers the bytes it needs
    struct Need { const char* name; const void* ptr; size_t bytes; };
    const size_t n = static_cast<size_t>(p.n_rows);
    const Need needs[] = {
        {"wpack", wpack, pg.pack_bytes()}, {"aux", p.aux, exact::AUX_FLOATS * sizeof(float)},
        {"rays_o", p.rays_o, INPUT == exact::IN_DEPTHNET ? n * 12 : 0}, {"rays_d", p.rays_d, INPUT == exact::IN_DEPTHNET ? n * 12 : 0},
        {"out", p.out, INPUT == exact::IN_DEPTHNET ? n * 4 : 0}, {"scratch", p.scratch, INPUT == exact::IN_DEPTHNET ? static_cast<size_t>(grid) * 2 * 32 * exact::KC_STRIDE : 0}};
    for (const Need& nd : needs) {
      if (!nd.bytes) continue;
      CUdeviceptr base = 0;
      size_t size = 0;
      typedef CUresult (*RangeFn)(CUdeviceptr*, size_t*, CUdeviceptr);
      static RangeFn range_fn = nullptr;
      if (!range_fn) {
        void* sym = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &sym, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
          range_fn = reinterpret_cast<RangeFn>(sym);
      }
      if (!range_fn) break;
      const CUresult r = range_fn(&base, &size, reinterpret_cast<CUdeviceptr>(nd.ptr));
      if (r != CUDA_SUCCESS) return fail("mlp_exact_kernel: %s = %p is not inside a device allocation (cuMemGetAddressRange %d)", nd.name, nd.ptr, static_cast<int>(r));
      const size_t off = reinterpret_cast<CUdeviceptr>(nd.ptr) - base;
      if (off + nd.bytes > size)
        return fail("mlp_exact_kernel: %s needs %zu bytes at offset %zu of an allocation of %zu bytes", nd.name, nd.bytes, off, size);
    }
  }
  {
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, p, tm);
    if (e != cudaSuccess)
      return fail("mlp_exact_kernel<%s> launch failed: %s (rows %d, grid %d, index list %d)",
                  INPUT == exact::IN_DEPTHNET ? "DEPTHNET" : (INPUT == exact::IN_NERF ? "NERF" : (INPUT == exact::IN_NERF_MASK ? "NERF+masks" : (INPUT == exact::IN_NERF_TAN ? "NERF tangent" : (INPUT == exact::IN_ACT ? "cat chain" : "cat chain Jacobian")))),
                  cudaGetErrorString(e), p.n_rows, grid, p.row_index != nullptr);
  }
  LAUNCH_CHECK();
  return 0;
}


// Split precision (bf16 hi + lo operands, 3 MMAs per K16 block) is the only mode of the exact kernel (mlp_exact.cuh).
extern "C" size_t b200nerf_nerf_wpack_bytes(int prec) {
  if (prec != B200NERF_PREC_SPLIT) return 0;
  return nerf_xprogram(nullptr).pack_bytes();
}
extern "C" size_t b200nerf_nerf_aux_floats(void) { return NERF_AUX_FLOATS; }

// gamma(pts) fills at most the 64 columns of its operand block (3 (1 + 2 multires) <= 64), gamma(viewdir) at most its 32
static int nerf_multires_check(const char* who, int multires, int multires_views) {
  if (multires < 1 || multires > 10 || multires_views < 1 || multires_views > 4)
    return fail("%s: multires=%d / multires_views=%d out of range: the NeRF kernels serve multires 1..10 and multires_views 1..4", who,
                multires, multires_views);
  return 0;
}

extern "C" int b200nerf_nerf_pack_multires(const float* const* t, int multires, int multires_views, int prec, void* h_wpack,
                                           float* h_aux) {
  if (nerf_multires_check("b200nerf_nerf_pack", multires, multires_views)) return 1;
  if (!t || !h_wpack || !h_aux) return fail("b200nerf_nerf_pack: null argument");
  if (prec != B200NERF_PREC_SPLIT) return fail("b200nerf_nerf_pack: prec must be B200NERF_PREC_SPLIT");
  const int d = 3 * (1 + 2 * multires), dv = 3 * (1 + 2 * multires_views);
  uint8_t* o = static_cast<uint8_t*>(h_wpack);
  const float* B[8];
  for (int i = 0; i < 8; ++i) B[i] = t[2 * i + 1];
  const float *Bf = t[19], *Wa = t[20], *Ba = t[21], *Wr = t[22], *Br = t[23];
  const int rc = pack_xprogram(nerf_xprogram(t, d, dv), o);
  if (rc) return rc;
  memset(h_aux, 0, NERF_AUX_FLOATS * sizeof(float));
  for (int i = 0; i < 8; ++i) memcpy(h_aux + NERF_B0 + 256 * i, B[i], 256 * sizeof(float));
  memcpy(h_aux + NERF_BF, Bf, 256 * sizeof(float));
  nerf_fold_view(t, dv, h_aux + NERF_BV);   // the program runs the view layer with feature_linear folded in
  memcpy(h_aux + NERF_WA, Wa, 256 * sizeof(float));
  h_aux[NERF_BA] = Ba[0];
  // the encoders' octave counts, read by both kernels; 0 means 10 / 4 (images packed before these slots were used)
  h_aux[NERF_BA + 1] = multires == 10 ? 0.f : static_cast<float>(multires);
  h_aux[NERF_BA + 2] = multires_views == 4 ? 0.f : static_cast<float>(multires_views);
  memcpy(h_aux + NERF_WR, Wr, 384 * sizeof(float));
  memcpy(h_aux + NERF_BR, Br, 3 * sizeof(float));
  return 0;
}
extern "C" int b200nerf_nerf_pack(const float* const* t, int prec, void* h_wpack, float* h_aux) {
  return b200nerf_nerf_pack_multires(t, 10, 4, prec, h_wpack, h_aux);
}


// ---- single-pass 16-bit image for nerf_fast_kernel (mlp_fast.cuh) ------------------------------------------
static inline uint16_t f2h(float f) {  // fp32 -> fp16, round to nearest even, subnormals and overflow handled
  uint32_t u;
  memcpy(&u, &f, 4);
  const uint32_t sign = (u >> 16) & 0x8000u;
  u &= 0x7fffffffu;
  if (u > 0x7f800000u) return static_cast<uint16_t>(sign | 0x7e00u);   // NaN
  if (u >= 0x477ff000u) return static_cast<uint16_t>(sign | 0x7c00u);  // rounds to >= 65520 -> inf
  if (u < 0x33000001u) return static_cast<uint16_t>(sign);             // < 2^-25 -> 0
  int e = static_cast<int>(u >> 23) - 127;
  uint32_t m = (u & 0x7fffffu) | 0x800000u;
  int shift = 13;
  if (e < -14) {
    shift += -14 - e;
    e = -15;
  }
  uint32_t r = m >> shift;
  const uint32_t rem = m & ((1u << shift) - 1u), half = 1u << (shift - 1);
  if (rem > half || (rem == half && (r & 1u))) ++r;
  // r carries the implicit bit for normals (bit 10); adding the biased exponent absorbs mantissa carries
  return static_cast<uint16_t>(sign | (static_cast<uint32_t>(e + 15) << 10) + (e == -15 ? r : r - 0x400u));
}

// One step of the layer program: K = the concatenation of up to two column segments of W [N, ldw], each zero-padded
// to a multiple of 16.  Layout [rank 0..1][K16 block][piece]: rank r holds output rows r*N/2 .. (r+1)*N/2-1 (the half
// its CTA of the pair streams), one piece = [2 k chunks][N/16 row groups][8 rows][8 k] 16-bit.
struct FastSeg {
  const float* W;
  int K, ldw, col0, Kpad;
};
static uint8_t* pack_step_fast(int N, const FastSeg* segs, int n_segs, bool fp16, uint8_t* out) {
  const int half = N / 2;
  for (int r = 0; r < 2; ++r)
    for (int sg = 0; sg < n_segs; ++sg) {
      const FastSeg& g = segs[sg];
      for (int k16 = 0; k16 < g.Kpad / 16; ++k16) {
        uint16_t* dst = reinterpret_cast<uint16_t*>(out);
        for (int kc = 0; kc < 2; ++kc)
          for (int n = 0; n < half; ++n)
            for (int e = 0; e < 8; ++e) {
              const int k = k16 * 16 + kc * 8 + e;
              const float w = k < g.K ? g.W[static_cast<size_t>(r * half + n) * g.ldw + g.col0 + k] : 0.f;
              dst[static_cast<size_t>(kc) * half * 8 + static_cast<size_t>(n >> 3) * 64 + (n & 7) * 8 + e] = fp16 ? f2h(w) : f2bf(w);
            }
        out += static_cast<size_t>(half) * 32;
      }
    }
  return out;
}

extern "C" size_t b200nerf_nerf_fast_wpack_bytes(void) { return fast::WPACK_BYTES; }

// The image does not record the octave counts: the kernel reads them from the aux block of b200nerf_nerf_pack_multires, which must
// be packed from the same tensors at the same multires / multires_views.
extern "C" int b200nerf_nerf_pack_fast_multires(const float* const* t, int multires, int multires_views, int prec, void* h_wpack) {
  if (nerf_multires_check("b200nerf_nerf_pack_fast", multires, multires_views)) return 1;
  if (!t || !h_wpack) return fail("b200nerf_nerf_pack_fast: null argument");
  if (prec != B200NERF_PREC_FP16) return fail("b200nerf_nerf_pack_fast: prec must be B200NERF_PREC_FP16");
  const bool fp16 = true;
  const int d = 3 * (1 + 2 * multires), dv = 3 * (1 + 2 * multires_views);
  uint8_t* o = static_cast<uint8_t*>(h_wpack);
  const float* W[8];
  for (int i = 0; i < 8; ++i) W[i] = t[2 * i];
  {
    const FastSeg sg[1] = {{W[0], d, d, 0, 64}};                                    // step 0: pts_linears.0 over gamma(pts)
    o = pack_step_fast(256, sg, 1, fp16, o);
  }
  for (int i = 1; i <= 4; ++i) {
    const FastSeg sg[1] = {{W[i], 256, 256, 0, 256}};
    o = pack_step_fast(256, sg, 1, fp16, o);
  }
  {
    const FastSeg sg[2] = {{W[5], 256, 256 + d, d, 256}, {W[5], d, 256 + d, 0, 64}};   // step 5: hidden columns, then gamma(pts)
    o = pack_step_fast(256, sg, 2, fp16, o);
  }
  for (int i = 6; i <= 7; ++i) {
    const FastSeg sg[1] = {{W[i], 256, 256, 0, 256}};
    o = pack_step_fast(256, sg, 1, fp16, o);
  }
  {
    // step 8: views_linears.0 with feature_linear folded in (no activation between them, run_nerf_helpers.py:116-121):
    //   W' = W_view[:, :256] * W_feature,  b' = W_view[:, :256] * b_feature + b_view   (fp64 sums)
    // K = [h7 (256) | gamma(viewdir) (dv -> 32) | two all-zero K16 blocks that fill the last ring stage]
    float bfold[128];
    const float* wfold = nerf_fold_view(t, dv, bfold);
    const FastSeg sg[3] = {{wfold, 256, 256 + dv, 0, 256}, {wfold, dv, 256 + dv, 256, 32}, {wfold, 0, 256 + dv, 0, 32}};
    o = pack_step_fast(128, sg, 3, fp16, o);
    memcpy(o, bfold, 128 * sizeof(float));   // fast::FOLD_BIAS_OFF
    o += 128 * sizeof(float);
  }
  if (static_cast<size_t>(o - static_cast<uint8_t*>(h_wpack)) != fast::WPACK_BYTES)
    return fail("b200nerf_nerf_pack_fast: internal size mismatch");
  return 0;
}
extern "C" int b200nerf_nerf_pack_fast(const float* const* t, int prec, void* h_wpack) {
  return b200nerf_nerf_pack_fast_multires(t, 10, 4, prec, h_wpack);
}

// the exact kernel keeps all biases + the head in its 3080-float shared-memory block: up to 10 hidden layers (the reference's
// experiments build 10: run.py:104-109)
constexpr int DEPTHNET_MAX_HIDDEN = 10;
static int depthnet_check(const char* who, int n_hidden, int prec) {
  if (prec != B200NERF_PREC_SPLIT) return fail("%s: prec must be B200NERF_PREC_SPLIT (the depth feeds the 2^9 octave of the encoding)", who);
  if (n_hidden < 0 || n_hidden > DEPTHNET_MAX_HIDDEN)
    return fail("%s: n_hidden=%d out of range (0..%d): inference serves DepthNets of 1 to %d cat layers", who, n_hidden, DEPTHNET_MAX_HIDDEN,
                DEPTHNET_MAX_HIDDEN + 1);
  return 0;
}
extern "C" size_t b200nerf_depthnet_wpack_bytes(int n_hidden, int prec) {
  if (prec != B200NERF_PREC_SPLIT || n_hidden < 0 || n_hidden > DEPTHNET_MAX_HIDDEN) return 0;
  return depthnet_xprogram(nullptr, nullptr, n_hidden).pack_bytes();
}
// The kernel stages a fixed-size aux block (exact::AUX_FLOATS = 3080 floats: eleven bias rows + head + 4) into shared memory whatever
// the depth, so the block is always that big (the tail is zero).  Round 1 sized it by n_hidden, and a 9-hidden-layer net read
// 1 KB past its 2,820 floats -- an illegal address whenever the block happened to end a mapped segment.
extern "C" size_t b200nerf_depthnet_aux_floats(int n_hidden) {
  const size_t need = static_cast<size_t>(n_hidden + 1) * 256 + 256 + 4;
  return need > static_cast<size_t>(exact::AUX_FLOATS) ? need : static_cast<size_t>(exact::AUX_FLOATS);
}

extern "C" int b200nerf_depthnet_pack_multires(const float* h_w0, const float* h_b0, const float* const* h_hidden, int n_hidden,
                                               const float* h_head_w, const float* h_head_b, int multires, int prec, void* h_wpack,
                                               float* h_aux) {
  // the architecture first: b200nerf_depthnet_wpack_bytes() is 0 for one it cannot serve, and a caller's empty buffer has no address
  if (depthnet_check("b200nerf_depthnet_pack", n_hidden, prec)) return 1;
  // enc(o) at multires 10 is 63 wide: every encoding fills at most the 64 columns of its block of the layer-0 operand
  if (multires < 1 || multires > 10) return fail("b200nerf_depthnet_pack: multires=%d out of range (1..10)", multires);
  if (!h_w0 || !h_b0 || !h_head_w || !h_head_b || !h_wpack || !h_aux || (n_hidden > 0 && !h_hidden))
    return fail("b200nerf_depthnet_pack: null argument");
  const int rc = pack_xprogram(depthnet_xprogram(h_w0, h_hidden, n_hidden), static_cast<uint8_t*>(h_wpack));
  if (rc) return rc;
  memset(h_aux, 0, b200nerf_depthnet_aux_floats(n_hidden) * sizeof(float));
  memcpy(h_aux, h_b0, 256 * sizeof(float));
  for (int i = 0; i < n_hidden; ++i) memcpy(h_aux + 256 * (i + 1), h_hidden[2 * i + 1], 256 * sizeof(float));
  memcpy(h_aux + 256 * (n_hidden + 1), h_head_w, 256 * sizeof(float));
  float* hb = h_aux + 256 * (n_hidden + 2);
  hb[0] = h_head_b[0];
  hb[1] = multires == 10 ? 0.f : static_cast<float>(multires);   // the encoder's multires; 0 means 10 (images packed before it was stored)
  hb[2] = hb[3] = 0.f;
  return 0;
}
extern "C" int b200nerf_depthnet_pack(const float* h_w0, const float* h_b0, const float* const* h_hidden, int n_hidden,
                                      const float* h_head_w, const float* h_head_b, int prec, void* h_wpack, float* h_aux) {
  return b200nerf_depthnet_pack_multires(h_w0, h_b0, h_hidden, n_hidden, h_head_w, h_head_b, 10, prec, h_wpack, h_aux);
}

// ------------------------------------------------------------------------------------------- ray generation
// get_rays (run_nerf_helpers.py:187-202) + viewdirs (nerf_utils.py:173); pixel centres without +0.5.
struct Cam {
  float r[12];
};
__global__ void get_rays_kernel(int H, int W, float fx, float fy, float cx, float cy, Cam cam, float* __restrict__ ro,
                                float* __restrict__ rd, float* __restrict__ vd) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= H * W) return;
  const float i = static_cast<float>(idx % W), j = static_cast<float>(idx / W);
  const float d0 = __fdiv_rn(__fadd_rn(i, -cx), fx);
  const float d1 = -__fdiv_rn(__fadd_rn(j, -cy), fy);
  const float d2 = -1.f;
  float d[3];
#pragma unroll
  for (int a = 0; a < 3; ++a)
    d[a] = __fadd_rn(__fadd_rn(__fmul_rn(d0, cam.r[4 * a + 0]), __fmul_rn(d1, cam.r[4 * a + 1])), __fmul_rn(d2, cam.r[4 * a + 2]));
  const float nrm = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(d[0], d[0]), __fmul_rn(d[1], d[1])), __fmul_rn(d[2], d[2])));
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    if (ro) ro[idx * 3 + a] = cam.r[4 * a + 3];
    if (rd) rd[idx * 3 + a] = d[a];
    if (vd) vd[idx * 3 + a] = __fdiv_rn(d[a], nrm);
  }
}

extern "C" int b200nerf_get_rays(int H, int W, float fx, float fy, float cx, float cy, const float* h_c2w, float* rays_o,
                                 float* rays_d, float* viewdirs, void* stream) {
  if (H <= 0 || W <= 0 || !h_c2w) return fail("b200nerf_get_rays: bad arguments");
  Cam cam;
  memcpy(cam.r, h_c2w, sizeof(cam.r));
  const int n = H * W;
  get_rays_kernel<<<(n + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(H, W, fx, fy, cx, cy, cam, rays_o, rays_d, viewdirs);
  LAUNCH_CHECK();
  return 0;
}

// Rays of selected pixels only (training batches: Trainer.sample_random_ray_batch, trainers/Trainer.py:400-475, builds
// all H*W rays and then indexes N_rand of them).  pix = flat row-major pixel indices.
__global__ void get_rays_at_kernel(int W, float fx, float fy, float cx, float cy, Cam cam, const long long* __restrict__ pix, int n,
                                   float* __restrict__ ro, float* __restrict__ rd, float* __restrict__ vd) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const long long idx = pix[t];
  const float i = static_cast<float>(idx % W), j = static_cast<float>(idx / W);
  const float d0 = __fdiv_rn(__fadd_rn(i, -cx), fx);
  const float d1 = -__fdiv_rn(__fadd_rn(j, -cy), fy);
  const float d2 = -1.f;
  float d[3];
#pragma unroll
  for (int a = 0; a < 3; ++a)
    d[a] = __fadd_rn(__fadd_rn(__fmul_rn(d0, cam.r[4 * a + 0]), __fmul_rn(d1, cam.r[4 * a + 1])), __fmul_rn(d2, cam.r[4 * a + 2]));
  const float nrm = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(d[0], d[0]), __fmul_rn(d[1], d[1])), __fmul_rn(d[2], d[2])));
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    if (ro) ro[t * 3 + a] = cam.r[4 * a + 3];
    if (rd) rd[t * 3 + a] = d[a];
    if (vd) vd[t * 3 + a] = __fdiv_rn(d[a], nrm);
  }
}
// out[t, :] = image[pix[t], :]   (target colours of the selected pixels)
__global__ void gather_pixels_kernel(const float* __restrict__ image, const long long* __restrict__ pix, int n, int C,
                                     float* __restrict__ out) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * C) return;
  out[t] = image[pix[t / C] * C + t % C];
}

extern "C" int b200nerf_get_rays_at(int H, int W, float fx, float fy, float cx, float cy, const float* h_c2w, const long long* pix,
                                    int n, float* rays_o, float* rays_d, float* viewdirs, void* stream) {
  if (H <= 0 || W <= 0 || !h_c2w || n < 0 || (n && !pix)) return fail("b200nerf_get_rays_at: bad arguments");
  if (n == 0) return 0;
  Cam cam;
  memcpy(cam.r, h_c2w, sizeof(cam.r));
  get_rays_at_kernel<<<(n + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(W, fx, fy, cx, cy, cam, pix, n, rays_o, rays_d, viewdirs);
  LAUNCH_CHECK();
  return 0;
}
extern "C" int b200nerf_gather_pixels(const float* image, const long long* pix, int n, int channels, float* out, void* stream) {
  if (n < 0 || channels <= 0 || (n && (!image || !pix || !out))) return fail("b200nerf_gather_pixels: bad arguments");
  if (n == 0) return 0;
  gather_pixels_kernel<<<(n * channels + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(image, pix, n, channels, out);
  LAUNCH_CHECK();
  return 0;
}

__global__ void normalize_dirs_kernel(const float* __restrict__ rd, int n, float* __restrict__ vd) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float x = rd[i * 3], y = rd[i * 3 + 1], z = rd[i * 3 + 2];
  const float nrm = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)), __fmul_rn(z, z)));
  vd[i * 3] = __fdiv_rn(x, nrm);
  vd[i * 3 + 1] = __fdiv_rn(y, nrm);
  vd[i * 3 + 2] = __fdiv_rn(z, nrm);
}
extern "C" int b200nerf_normalize_dirs(const float* rays_d, int n_rays, float* viewdirs, void* stream) {
  if (n_rays < 0 || (n_rays && (!rays_d || !viewdirs))) return fail("b200nerf_normalize_dirs: bad arguments");
  if (n_rays == 0) return 0;
  normalize_dirs_kernel<<<(n_rays + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(rays_d, n_rays, viewdirs);
  LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------- sample placement
// sample_points_around_mean (nerf_pytorch/utils.py:220-244).  Uniform mode needs no sort: the grid is
// monotone, so sort(cat([mean+grid, mean])) = the grid values below zero, then the mean, then the rest.
__global__ void place_uniform_kernel(const float* __restrict__ mean, const float* __restrict__ grid, int n_rays, int S,
                                     float lo, float hi, float* __restrict__ z) {
  const size_t idx = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<size_t>(n_rays) * S) return;
  const int s = static_cast<int>(idx % S);
  const float m = mean[idx / S];
  float v = m;  // slot n_neg (first slot whose grid value is not negative) holds the mean itself
  if (s <= S - 2 && __ldg(grid + s) < 0.f) v = __fadd_rn(m, __ldg(grid + s));
  else if (s >= 1 && !(__ldg(grid + s - 1) < 0.f)) v = __fadd_rn(m, __ldg(grid + s - 1));
  v = v < lo ? lo : (v > hi ? hi : v);  // NaN (ray missed the sphere) stays NaN, like torch.clip
  z[idx] = v;
}

// The same for S % 4 == 0: one thread writes four consecutive samples as a float4 (32-bit index arithmetic, a quarter of
// the threads); the one-element kernel above ran at ~1 TB/s of the 4*S + 4 B per ray it moves.
__global__ void __launch_bounds__(256) place_uniform_vec4_kernel(const float* __restrict__ mean, const float* __restrict__ grid,
                                                                 int n_rays, int S, float lo, float hi, float* __restrict__ z) {
  const unsigned q = blockIdx.x * blockDim.x + threadIdx.x;   // float4 index
  const unsigned qpr = static_cast<unsigned>(S) >> 2;         // float4s per ray
  const unsigned ray = q / qpr;
  if (ray >= static_cast<unsigned>(n_rays)) return;
  const int s0 = static_cast<int>(q - ray * qpr) * 4;
  const float m = __ldg(mean + ray);
  float v[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int s = s0 + i;
    float x = m;
    if (s <= S - 2 && __ldg(grid + s) < 0.f) x = __fadd_rn(m, __ldg(grid + s));
    else if (s >= 1 && !(__ldg(grid + s - 1) < 0.f)) x = __fadd_rn(m, __ldg(grid + s - 1));
    v[i] = x < lo ? lo : (x > hi ? hi : x);
  }
  reinterpret_cast<float4*>(z)[q] = make_float4(v[0], v[1], v[2], v[3]);
}

// Gaussian mode: one warp sorts one ray's S values (bitonic network over a power-of-two padded row in smem).
__global__ void place_sorted_kernel(const float* __restrict__ mean, const float* __restrict__ offs, int n_rays, int S,
                                    int P /*pow2 >= S*/, float* __restrict__ z) {
  extern __shared__ float srow[];
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ray = blockIdx.x * (blockDim.x >> 5) + wib;
  float* row = srow + wib * P;
  if (ray < n_rays) {
    const float m = mean[ray];
    for (int i = lane; i < P; i += 32)
      row[i] = i < S - 1 ? __fadd_rn(m, offs[static_cast<size_t>(ray) * (S - 1) + i]) : (i == S - 1 ? m : __int_as_float(0x7f800000));
  }
  __syncwarp();
  for (int k = 2; k <= P; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      if (ray < n_rays)
        for (int i = lane; i < P; i += 32) {
          const int l = i ^ j;
          if (l > i) {
            const float a = row[i], b = row[l];
            const bool up = (i & k) == 0;
            // NaN sorts last (as torch.sort does): treat NaN as +inf-and-beyond
            const bool a_gt_b = (a != a) ? !(b != b) : (!(b != b) && a > b);
            if (a_gt_b == up) {
              row[i] = b;
              row[l] = a;
            }
          }
        }
      __syncwarp();
    }
  if (ray < n_rays)
    for (int i = lane; i < S; i += 32) z[static_cast<size_t>(ray) * S + i] = row[i];
}

extern "C" int b200nerf_place_samples(const float* mean, const float* offsets, int n_rays, int S, int mode, float clip_lo,
                                      float clip_hi, float* out_z, void* stream) {
  if (n_rays < 0 || S < 1 || !out_z || !mean) return fail("b200nerf_place_samples: bad arguments");
  if (n_rays == 0) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t total = static_cast<size_t>(n_rays) * S;
  if (mode == B200NERF_PLACE_DEPTH_ONLY) {
    if (S != 1) return fail("b200nerf_place_samples: depth_only needs S == 1");
    CUDA_TRY(cudaMemcpyAsync(out_z, mean, total * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return 0;
  }
  if (S > 1 && !offsets) return fail("b200nerf_place_samples: offsets is null");
  if (mode == B200NERF_PLACE_UNIFORM) {
    if ((S & 3) == 0 && (reinterpret_cast<uintptr_t>(out_z) & 15) == 0 && total / 4 < 0x7fffff00ull)
      place_uniform_vec4_kernel<<<static_cast<unsigned>((total / 4 + 255) / 256), 256, 0, st>>>(mean, offsets, n_rays, S, clip_lo, clip_hi, out_z);
    else
      place_uniform_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, st>>>(mean, offsets, n_rays, S, clip_lo, clip_hi, out_z);
    LAUNCH_CHECK();
    return 0;
  }
  if (mode == B200NERF_PLACE_GAUSSIAN) {
    int P = 1;
    while (P < S) P <<= 1;
    if (P > 4096) return fail("b200nerf_place_samples: S=%d too large for gaussian mode", S);
    const int wpb = 4;
    place_sorted_kernel<<<(n_rays + wpb - 1) / wpb, wpb * 32, wpb * P * sizeof(float), st>>>(mean, offsets, n_rays, S, P, out_z);
    LAUNCH_CHECK();
    return 0;
  }
  return fail("b200nerf_place_samples: unknown mode %d", mode);
}

__global__ void points_kernel(const float* __restrict__ ro, const float* __restrict__ rd, const float* __restrict__ z,
                              size_t total, int S, float* __restrict__ pts) {
  const size_t idx = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total * 3) return;
  const size_t pt = idx / 3;
  const int a = static_cast<int>(idx % 3);
  const size_t ray = pt / S;
  pts[idx] = __fadd_rn(ro[ray * 3 + a], __fmul_rn(rd[ray * 3 + a], z[pt]));
}
extern "C" int b200nerf_points(const float* rays_o, const float* rays_d, const float* z, int n_rays, int S, float* out_pts,
                               void* stream) {
  if (n_rays < 0 || S < 1) return fail("b200nerf_points: bad arguments");
  const size_t total = static_cast<size_t>(n_rays) * S;
  if (total == 0) return 0;
  points_kernel<<<static_cast<unsigned>((total * 3 + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(rays_o, rays_d, z, total, S, out_pts);
  LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------- compositing
// raw2outputs (trainers/sampling_trainer.py:153-230).  LPR lanes cooperate on one ray and every lane owns FOUR
// consecutive samples per pass (four float4 loads of raw, one float4 of z, one float4 store of the weights, all
// coalesced).  The exclusive transmittance product is a local 4-term product followed by a segmented warp scan over
// the LPR lanes, carried in double and rounded per element exactly like the CPU reference's cumprod; the three maps
// are reduced in registers.  One scan step serves four samples, which keeps the kernel bandwidth-bound.
// FULL: S == 4 * LPR (one pass, every lane in range, rows 16-byte aligned) -- no bounds checks in the hot loop.
template <int LPR, bool FULL>
__global__ void __launch_bounds__(256, 4) composite_kernel(const float* __restrict__ raw, const float* __restrict__ z,
                                                        const float* __restrict__ rays_d, const float* __restrict__ noise,
                                                        int n_rays, int S, int white, float* __restrict__ o_rgb,
                                                        float* __restrict__ o_disp, float* __restrict__ o_acc,
                                                        float* __restrict__ o_depth, float* __restrict__ o_w,
                                                        float* __restrict__ o_alpha, int rgb_stride, int disp_stride) {
  const int gtid = blockIdx.x * blockDim.x + threadIdx.x;
  const int lig = threadIdx.x & (LPR - 1);
  int ray = gtid / LPR;
  const bool live = ray < n_rays;
  if (!live) ray = n_rays - 1;
  const size_t base = static_cast<size_t>(ray) * S;
  const float dx = __ldg(rays_d + ray * 3), dy = __ldg(rays_d + ray * 3 + 1), dz = __ldg(rays_d + ray * 3 + 2);
  const float nrm = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz)));
  const bool vec = FULL || (S & 3) == 0;   // rows of z / weights are 16-byte aligned

  double carry = 1.0;
  float s_r = 0.f, s_g = 0.f, s_b = 0.f, s_d = 0.f, s_a = 0.f;
  for (int s0 = 0; s0 < S; s0 += 4 * LPR) {
    const int sb = s0 + lig * 4;
    float zz[5];
    float4 rw[4];
    float nz[4] = {0.f, 0.f, 0.f, 0.f};
    if (vec && (FULL || sb < S)) {
      const float4 z4 = __ldg(reinterpret_cast<const float4*>(z + base + sb));
      zz[0] = z4.x; zz[1] = z4.y; zz[2] = z4.z; zz[3] = z4.w;
      if (FULL) zz[4] = __shfl_down_sync(0xffffffffu, z4.x, 1, LPR);   // the next lane's first depth (unused on the last lane)
      else zz[4] = sb + 4 < S ? __ldg(z + base + sb + 4) : 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) rw[i] = __ldg(reinterpret_cast<const float4*>(raw) + base + sb + i);
      if (noise) {
        const float4 n4 = __ldg(reinterpret_cast<const float4*>(noise + base + sb));
        nz[0] = n4.x; nz[1] = n4.y; nz[2] = n4.z; nz[3] = n4.w;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 5; ++i) zz[i] = sb + i < S ? __ldg(z + base + sb + i) : 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        rw[i] = sb + i < S ? __ldg(reinterpret_cast<const float4*>(raw) + base + sb + i) : make_float4(0.f, 0.f, 0.f, 0.f);
        if (noise && sb + i < S) nz[i] = __ldg(noise + base + sb + i);
      }
    }
    float alpha[4];
    double ex[4];          // exclusive product inside this lane's four samples
    double run = 1.0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int sidx = sb + i;
      ex[i] = run;
      if (FULL || sidx < S) {
        const bool last = FULL ? (i == 3 && lig == LPR - 1) : !(sidx + 1 < S);
        const float dist = __fmul_rn(last ? 1e10f : __fadd_rn(zz[i + 1], -zz[i]), nrm);
        const float sg = noise ? __fadd_rn(rw[i].w, nz[i]) : rw[i].w;
        alpha[i] = __fadd_rn(1.0f, -expf(__fmul_rn(-fmaxf(sg, 0.f), dist)));
        run *= static_cast<double>(__fadd_rn(__fadd_rn(1.0f, -alpha[i]), 1e-10f));
      } else {
        alpha[i] = 0.f;
      }
    }
    double incl = run;
#pragma unroll
    for (int off = 1; off < LPR; off <<= 1) {
      const double t = __shfl_up_sync(0xffffffffu, incl, off, LPR);
      if (lig >= off) incl *= t;
    }
    double excl = __shfl_up_sync(0xffffffffu, incl, 1, LPR);
    if (lig == 0) excl = 1.0;
    excl *= carry;
    carry *= __shfl_sync(0xffffffffu, incl, LPR - 1, LPR);
    float w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float T = static_cast<float>(excl * ex[i]);
      w[i] = (FULL || sb + i < S) ? __fmul_rn(alpha[i], T) : 0.f;
      if (FULL || sb + i < S) {
        // colours: fast exp / reciprocal (<= 3e-7 on a sigmoid); the alpha path above keeps the accurate expf because
        // the weights also feed arg-max and inverse-CDF indices
        s_r = fmaf(w[i], __fdividef(1.0f, 1.0f + __expf(-rw[i].x)), s_r);
        s_g = fmaf(w[i], __fdividef(1.0f, 1.0f + __expf(-rw[i].y)), s_g);
        s_b = fmaf(w[i], __fdividef(1.0f, 1.0f + __expf(-rw[i].z)), s_b);
        s_d = fmaf(w[i], zz[i], s_d);
        s_a += w[i];
      }
    }
    if (live && (FULL || sb < S)) {
      if (vec) {
        if (o_w) *reinterpret_cast<float4*>(o_w + base + sb) = make_float4(w[0], w[1], w[2], w[3]);
        if (o_alpha) *reinterpret_cast<float4*>(o_alpha + base + sb) = make_float4(alpha[0], alpha[1], alpha[2], alpha[3]);
      } else {
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (sb + i < S) {
            if (o_w) o_w[base + sb + i] = w[i];
            if (o_alpha) o_alpha[base + sb + i] = alpha[i];
          }
      }
    }
  }
#pragma unroll
  for (int off = LPR >> 1; off > 0; off >>= 1) {
    s_r += __shfl_xor_sync(0xffffffffu, s_r, off, LPR);
    s_g += __shfl_xor_sync(0xffffffffu, s_g, off, LPR);
    s_b += __shfl_xor_sync(0xffffffffu, s_b, off, LPR);
    s_d += __shfl_xor_sync(0xffffffffu, s_d, off, LPR);
    s_a += __shfl_xor_sync(0xffffffffu, s_a, off, LPR);
  }
  if (live && lig == 0) {
    if (white) {
      const float bg = __fadd_rn(1.0f, -s_a);
      s_r += bg;
      s_g += bg;
      s_b += bg;
    }
    if (o_rgb) {
      o_rgb[ray * rgb_stride] = s_r;
      o_rgb[ray * rgb_stride + 1] = s_g;
      o_rgb[ray * rgb_stride + 2] = s_b;
    }
    if (o_disp) o_disp[ray * disp_stride] = __fdiv_rn(1.0f, fmaxf(1e-10f, __fdiv_rn(s_d, __fadd_rn(s_a, 1e-10f))));
    if (o_acc) o_acc[ray] = s_a;
    if (o_depth) o_depth[ray] = s_d;
  }
}

// S == 1: the reference pads the interval list from an EMPTY slice, so every per-sample tensor is [N,0]
// and the colour is sigmoid(raw rgb) (sampling_trainer.py:178-180, :220-221).
__global__ void composite_single_kernel(const float* __restrict__ raw, int n_rays, float* __restrict__ o_rgb,
                                        float* __restrict__ o_disp, float* __restrict__ o_acc, float* __restrict__ o_depth,
                                        int rgb_stride, int disp_stride) {
  const int ray = blockIdx.x * blockDim.x + threadIdx.x;
  if (ray >= n_rays) return;
  const float4 rw = __ldg(reinterpret_cast<const float4*>(raw) + ray);
  if (o_rgb) {
    o_rgb[ray * rgb_stride] = 1.0f / (1.0f + expf(-rw.x));
    o_rgb[ray * rgb_stride + 1] = 1.0f / (1.0f + expf(-rw.y));
    o_rgb[ray * rgb_stride + 2] = 1.0f / (1.0f + expf(-rw.z));
  }
  if (o_disp) o_disp[ray * disp_stride] = __fdiv_rn(1.0f, fmaxf(1e-10f, __fdiv_rn(0.f, 1e-10f)));
  if (o_acc) o_acc[ray] = 0.f;
  if (o_depth) o_depth[ray] = 0.f;
}

template <int LPR>
static void launch_composite(const float* raw, const float* z, const float* rays_d, const float* noise, int n_rays, int S,
                             int white, float* o_rgb, float* o_disp, float* o_acc, float* o_depth, float* o_w,
                             float* o_alpha, int rs, int ds, cudaStream_t st) {
  const long long threads = static_cast<long long>(n_rays) * LPR;
  const unsigned grid = static_cast<unsigned>((threads + 255) / 256);
  if (S == 4 * LPR) composite_kernel<LPR, true><<<grid, 256, 0, st>>>(raw, z, rays_d, noise, n_rays, S, white, o_rgb, o_disp, o_acc, o_depth, o_w, o_alpha, rs, ds);
  else composite_kernel<LPR, false><<<grid, 256, 0, st>>>(raw, z, rays_d, noise, n_rays, S, white, o_rgb, o_disp, o_acc, o_depth, o_w, o_alpha, rs, ds);
}

// S = 32 / 64 / 128 without a noise input: the TMA-staged persistent kernel (composite_tma.cuh).  raw viewed as
// [n_rays*S/8 rows, 128 B]; one box = 256 rows = one 2048-sample tile, 128-byte swizzle.
template <int LPR>
static int launch_composite_tma(const float* raw, const float* z, const float* rays_d, int n_rays, int white, float* o_rgb,
                                float* o_disp, float* o_acc, float* o_depth, float* o_w, float* o_alpha, int rs, int ds,
                                cudaStream_t st) {
  static bool configured[B200_MAX_DEVICES] = {false};
  auto kern = comp::composite_tma_kernel<LPR>;
  const int dev = b200_device();
  if (dev < 0) return fail("composite_tma_kernel: no usable CUDA device");
  if (!configured[dev]) {
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, comp::SMEM_BYTES));
    configured[dev] = true;
  }
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) return fail("cuTensorMapEncodeTiled is not available from the driver");
  static_assert(sizeof(CUtensorMap) == sizeof(comp::TMap), "tensor map size");
  const long long total = static_cast<long long>(n_rays) * (4 * LPR);
  comp::TMap tm;
  const cuuint64_t gdim[2] = {32, static_cast<cuuint64_t>(total / 8)};
  const cuuint64_t gstride[1] = {128};
  const cuuint32_t box[2] = {32, comp::RAW_BYTES / 128};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(reinterpret_cast<CUtensorMap*>(&tm), CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(raw), gdim, gstride,
                         box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled(raw) failed (%d)", static_cast<int>(r));
  const long long tiles = (total + comp::TILE_SAMPLES - 1) / comp::TILE_SAMPLES;
  const int sms = sm_count();
  if (sms <= 0) return fail("no CUDA device");
  const int grid = static_cast<int>(tiles < 2LL * sms ? tiles : 2LL * sms);
  kern<<<grid, comp::THREADS, comp::SMEM_BYTES, st>>>(tm, z, rays_d, n_rays, white, o_rgb, o_disp, o_acc, o_depth, o_w, o_alpha, rs, ds);
  LAUNCH_CHECK();
  return 0;
}

static bool composite_force_ldg() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("B200NERF_COMPOSITE_LDG");   // A/B switch for measurements: 1 = register-staged kernel everywhere
    v = (e && e[0] == '1') ? 1 : 0;
  }
  return v == 1;
}
static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// rs / ds: element strides of the rgb and disp outputs (3 / 1 for separate maps, 4 / 4 for one [n,4] rgb|disp image tile)
static int composite_impl(const float* raw, const float* z, const float* rays_d, const float* noise, int n_rays, int S,
                          int white_bkgd, float* out_rgb, float* out_disp, float* out_acc, float* out_depth, float* out_weights,
                          float* out_alphas, int rs, int ds, void* stream) {
  if (n_rays < 0 || S < 1) return fail("b200nerf_composite_fwd: bad sizes n_rays=%d S=%d", n_rays, S);
  if (n_rays == 0) return 0;
  if (!raw || !z || !rays_d) return fail("b200nerf_composite_fwd: null input");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (S == 1) {
    composite_single_kernel<<<(n_rays + 255) / 256, 256, 0, st>>>(raw, n_rays, out_rgb, out_disp, out_acc, out_depth, rs, ds);
    LAUNCH_CHECK();
    return 0;
  }
  if ((S == 32 || S == 64 || S == 128) && !noise && static_cast<long long>(n_rays) * S >= comp::TILE_SAMPLES && aligned16(raw) &&
      aligned16(z) && aligned16(out_weights) && aligned16(out_alphas) && !composite_force_ldg()) {
    if (S == 32) return launch_composite_tma<8>(raw, z, rays_d, n_rays, white_bkgd, out_rgb, out_disp, out_acc, out_depth, out_weights, out_alphas, rs, ds, st);
    if (S == 64) return launch_composite_tma<16>(raw, z, rays_d, n_rays, white_bkgd, out_rgb, out_disp, out_acc, out_depth, out_weights, out_alphas, rs, ds, st);
    return launch_composite_tma<32>(raw, z, rays_d, n_rays, white_bkgd, out_rgb, out_disp, out_acc, out_depth, out_weights, out_alphas, rs, ds, st);
  }
  // lanes per ray: four samples per lane and pass
  if (S <= 4) launch_composite<1>(raw, z, rays_d, noise, n_rays, S, white_bkgd, out_rgb, out_disp, out_acc, out_depth, out_weights, out_alphas, rs, ds, st);
  else if (S <= 8) launch_composite<2>(raw, z, rays_d, noise, n_rays, S, white_bkgd, out_rgb, out_disp, out_acc, out_depth, out_weights, out_alphas, rs, ds, st);
  else if (S <= 16) launch_composite<4>(raw, z, rays_d, noise, n_rays, S, white_bkgd, out_rgb, out_disp, out_acc, out_depth, out_weights, out_alphas, rs, ds, st);
  else if (S <= 32) launch_composite<8>(raw, z, rays_d, noise, n_rays, S, white_bkgd, out_rgb, out_disp, out_acc, out_depth, out_weights, out_alphas, rs, ds, st);
  else if (S <= 64) launch_composite<16>(raw, z, rays_d, noise, n_rays, S, white_bkgd, out_rgb, out_disp, out_acc, out_depth, out_weights, out_alphas, rs, ds, st);
  else launch_composite<32>(raw, z, rays_d, noise, n_rays, S, white_bkgd, out_rgb, out_disp, out_acc, out_depth, out_weights, out_alphas, rs, ds, st);
  LAUNCH_CHECK();
  return 0;
}

extern "C" int b200nerf_composite_fwd(const float* raw, const float* z, const float* rays_d, const float* noise, int n_rays,
                                      int S, int white_bkgd, float* out_rgb, float* out_disp, float* out_acc,
                                      float* out_depth, float* out_weights, float* out_alphas, void* stream) {
  return composite_impl(raw, z, rays_d, noise, n_rays, S, white_bkgd, out_rgb, out_disp, out_acc, out_depth, out_weights,
                        out_alphas, 3, 1, stream);
}

extern "C" int b200nerf_composite_tile_fwd(const float* raw, const float* z, const float* rays_d, const float* noise, int n_rays,
                                           int S, int white_bkgd, float* out_rgbd, float* out_acc, float* out_depth,
                                           float* out_weights, float* out_alphas, void* stream) {
  if (!out_rgbd) return fail("b200nerf_composite_tile_fwd: null tile");
  return composite_impl(raw, z, rays_d, noise, n_rays, S, white_bkgd, out_rgbd, out_rgbd + 3, out_acc, out_depth, out_weights,
                        out_alphas, 4, 4, stream);
}

// ------------------------------------------------------------------------------------------- compositing backward
// The reverse-mode derivative of raw2outputs (trainers/sampling_trainer.py:153-230) for S >= 2, one warp per ray, sample
// i0 + lane in pass i0.  The forward's per-sample arithmetic is recomputed bit for bit (alpha, t = 1 - alpha + 1e-10, the 1e10 last
// interval).  With gw_i the total gradient reaching w_i and R_i = sum_{j>i} gw_j alpha_j prod_{i<l<j} t_l,
//   g_alpha_i = g_alphas_i + T_i (gw_i - R_i),   R_i = gw_{i+1} alpha_{i+1} + t_{i+1} R_{i+1},   R_{S-1} = 0,
// a reverse scan (in double, like the forward's cumprod) that never divides by t, so it keeps the gradient where T underflows.
// Pass 1 (ascending) forms T_i as the forward does and parks it in out_g_z; pass 2 (descending) reads it back, runs the scan and
// overwrites out_g_z with d/dz.  dist_j = (z_{j+1} - z_j) |rays_d| feeds z_{j+1} and z_j; lane 0's z-gradient waits for the
// term of the pass below it (`pend`).
__device__ __forceinline__ float comp_alpha(float sg, float dist, float* e) {
  *e = expf(__fmul_rn(-fmaxf(sg, 0.f), dist));
  return __fadd_rn(1.0f, -*e);
}

__global__ void __launch_bounds__(256) composite_bwd_kernel(
    const float* __restrict__ raw, const float* __restrict__ z, const float* __restrict__ rays_d, const float* __restrict__ noise,
    int n_rays, int S, int white, const float* __restrict__ g_rgb, const float* __restrict__ g_disp, const float* __restrict__ g_acc,
    const float* __restrict__ g_depth, const float* __restrict__ g_weights, const float* __restrict__ g_alphas,
    float* __restrict__ out_g_raw, float* __restrict__ out_g_z) {
  const int ray = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (ray >= n_rays) return;   // whole warp leaves together
  const size_t base = static_cast<size_t>(ray) * S;
  const float dx = __ldg(rays_d + ray * 3), dy = __ldg(rays_d + ray * 3 + 1), dz = __ldg(rays_d + ray * 3 + 2);
  const float nrm = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz)));
  auto sample = [&](int i, float4& rw, float& zi, float& alpha, float& e, float& dist, float& sg) {
    rw = __ldg(reinterpret_cast<const float4*>(raw) + base + i);
    zi = __ldg(z + base + i);
    dist = __fmul_rn(i + 1 < S ? __fadd_rn(__ldg(z + base + i + 1), -zi) : 1e10f, nrm);
    sg = noise ? __fadd_rn(rw.w, __ldg(noise + base + i)) : rw.w;
    alpha = comp_alpha(sg, dist, &e);
  };

  // pass 1: T_i (exclusive cumprod of t, double), acc and depth for the disparity's derivative
  double carry = 1.0, acc = 0.0, depth = 0.0;
  for (int i0 = 0; i0 < S; i0 += 32) {
    const int i = i0 + lane;
    float4 rw;
    float zi = 0.f, alpha = 0.f, e, dist, sg;
    double incl = 1.0;
    if (i < S) {
      sample(i, rw, zi, alpha, e, dist, sg);
      incl = static_cast<double>(__fadd_rn(__fadd_rn(1.0f, -alpha), 1e-10f));
    }
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const double v = __shfl_up_sync(0xffffffffu, incl, off);
      if (lane >= off) incl *= v;
    }
    double excl = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane == 0) excl = 1.0;
    const float T = static_cast<float>(carry * excl);
    carry *= __shfl_sync(0xffffffffu, incl, 31);
    if (i < S) {
      const float w = __fmul_rn(alpha, T);
      out_g_z[base + i] = T;
      acc += w;
      depth += static_cast<double>(w) * zi;
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    acc += __shfl_xor_sync(0xffffffffu, acc, off);
    depth += __shfl_xor_sync(0xffffffffu, depth, off);
  }

  // upstream gradients folded into one coefficient per output: rgb_k = sum w c_k + white (1 - acc), disp = 1 / max(1e-10, q),
  // q = depth / (acc + 1e-10) (torch.max sends the gradient to the larger argument, half of it on a tie)
  float gr[3] = {0.f, 0.f, 0.f};
  if (g_rgb)
#pragma unroll
    for (int k = 0; k < 3; ++k) gr[k] = __ldg(g_rgb + ray * 3 + k);
  double gacc = g_acc ? static_cast<double>(__ldg(g_acc + ray)) : 0.0;
  double gdep = g_depth ? static_cast<double>(__ldg(g_depth + ray)) : 0.0;
  if (white) gacc -= static_cast<double>(gr[0]) + gr[1] + gr[2];
  if (g_disp) {
    const double den = acc + 1e-10;
    const double q = depth / den;
    const double m = static_cast<double>(fmaxf(1e-10f, static_cast<float>(q)));
    const double share = q > 1e-10 ? 1.0 : (q == 1e-10 ? 0.5 : 0.0);
    const double gq = -static_cast<double>(__ldg(g_disp + ray)) / (m * m) * share;
    gdep += gq / den;
    gacc -= gq * depth / (den * den);
  }

  // pass 2: reverse scan of R, from the last pass down
  double R_in = 0.0;   // R of the last sample of the pass being processed (R_{S-1} = 0)
  float pend = 0.f;    // z-gradient of the previous pass's first sample, short of the dist term of the sample in front of it
  const int last0 = ((S - 1) >> 5) << 5;
  for (int i0 = last0; i0 >= 0; i0 -= 32) {
    const int i = i0 + lane;
    const bool in = i < S;
    float4 rw = make_float4(0.f, 0.f, 0.f, 0.f);
    float zi = 0.f, alpha = 0.f, e = 1.f, dist = 0.f, sg = 0.f, T = 0.f;
    double t = 1.0, a = 0.0;   // f_i(R) = a_i + t_i R maps R_i onto R_{i-1}
    float gw = 0.f, c[3] = {0.f, 0.f, 0.f};
    if (in) {
      sample(i, rw, zi, alpha, e, dist, sg);
      T = out_g_z[base + i];
      t = static_cast<double>(__fadd_rn(__fadd_rn(1.0f, -alpha), 1e-10f));
      c[0] = 1.0f / (1.0f + expf(-rw.x));
      c[1] = 1.0f / (1.0f + expf(-rw.y));
      c[2] = 1.0f / (1.0f + expf(-rw.z));
      double g = gacc + gdep * zi + static_cast<double>(gr[0]) * c[0] + static_cast<double>(gr[1]) * c[1] +
                 static_cast<double>(gr[2]) * c[2];
      if (g_weights) g += __ldg(g_weights + base + i);
      gw = static_cast<float>(g);
      a = static_cast<double>(gw) * alpha;
    }
    // suffix composition F_l = f_l o f_{l+1} o ... o f_31 as (M, B): F(R) = B + M R
    double M = t, B = a;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const double Mo = __shfl_down_sync(0xffffffffu, M, off), Bo = __shfl_down_sync(0xffffffffu, B, off);
      if (lane + off < 32) {
        B = B + M * Bo;
        M = M * Mo;
      }
    }
    double Mx = __shfl_down_sync(0xffffffffu, M, 1), Bx = __shfl_down_sync(0xffffffffu, B, 1);
    if (lane == 31) {
      Mx = 1.0;
      Bx = 0.0;
    }
    const double Ri = Bx + Mx * R_in;                               // R_i
    const double R_next = __shfl_sync(0xffffffffu, B + M * R_in, 0);   // R_{i0-1}

    float gdist = 0.f, gzi = 0.f;
    if (in) {
      float ga = static_cast<float>(static_cast<double>(T) * (static_cast<double>(gw) - Ri));
      if (g_alphas) ga += __ldg(g_alphas + base + i);
      // alpha = 1 - e, e = exp(-relu(sg) dist): d alpha / d relu = e dist, d alpha / d dist = e relu; relu'(0) = 0
      const float ge = __fmul_rn(ga, e);
      const float gs = sg > 0.f ? __fmul_rn(ge, dist) : 0.f;
      gdist = i + 1 < S ? __fmul_rn(ge, fmaxf(sg, 0.f)) : 0.f;
      const float w = __fmul_rn(alpha, T);
      float4 o;
      o.x = gr[0] * w * c[0] * (1.0f - c[0]);
      o.y = gr[1] * w * c[1] * (1.0f - c[1]);
      o.z = gr[2] * w * c[2] * (1.0f - c[2]);
      o.w = gs;
      reinterpret_cast<float4*>(out_g_raw)[base + i] = o;
      gzi = static_cast<float>(gdep * w) - gdist * nrm;
    }
    // + dist_{i-1}'s term: from the lane below, or (lane 0) from the next pass down
    const float from_below = __shfl_up_sync(0xffffffffu, gdist, 1);
    if (lane > 0 && in) gzi += from_below * nrm;
    const float top = __shfl_sync(0xffffffffu, gdist, 31);   // dist_{i0+31} feeds z_{i0+32}: the previous pass's first sample
    if (lane == 0 && i0 != last0) out_g_z[base + i0 + 32] = pend + top * nrm;
    pend = __shfl_sync(0xffffffffu, gzi, 0);
    if (lane > 0 && in) out_g_z[base + i] = gzi;
    R_in = R_next;
  }
  if (lane == 0) out_g_z[base] = pend;
}

extern "C" int b200nerf_composite_bwd(const float* raw, const float* z, const float* rays_d, const float* noise, int n_rays, int S,
                                      int white_bkgd, const float* g_rgb, const float* g_disp, const float* g_acc, const float* g_depth,
                                      const float* g_weights, const float* g_alphas, float* out_g_raw, float* out_g_z, void* stream) {
  if (n_rays < 0) return fail("b200nerf_composite_bwd: bad sizes n_rays=%d", n_rays);
  if (S < 2) return fail("b200nerf_composite_bwd: S=%d; S >= 2 is required (S == 1 has no intervals: its colour is sigmoid(raw rgb))", S);
  if (n_rays == 0) return 0;
  if (!raw || !z || !rays_d || !out_g_raw || !out_g_z) return fail("b200nerf_composite_bwd: null argument");
  const int wpb = 8;
  composite_bwd_kernel<<<(n_rays + wpb - 1) / wpb, wpb * 32, 0, static_cast<cudaStream_t>(stream)>>>(
      raw, z, rays_d, noise, n_rays, S, white_bkgd, g_rgb, g_disp, g_acc, g_depth, g_weights, g_alphas, out_g_raw, out_g_z);
  LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------------------- MLP launches
// row_index / n_rows_dev != nullptr: evaluate only the listed sample points (at most list_cap of them), in place
static int nerf_exact_launch(const void* wpack, const float* aux, const float* rays_o, const float* rays_d, const float* viewdirs,
                             const float* z, const float* pts, int n_rays, int S, float* out_raw, const int* row_index,
                             const int* n_rows_dev, int list_cap, cudaStream_t st) {
  exact::ExactParams xp;
  memset(&xp, 0, sizeof(xp));
  xp.aux = aux;
  xp.n_rows = row_index ? list_cap : n_rays * S;
  xp.S = S;
  xp.rays_o = rays_o;
  xp.rays_d = rays_d;
  xp.viewdirs = viewdirs;
  xp.z = z;
  xp.pts = pts;
  xp.out = out_raw;
  xp.row_index = row_index;
  xp.n_rows_dev = n_rows_dev;
  xp.head_w_off = NERF_WA;
  xp.head_b_off = NERF_BA;
  xp.rgb_w_off = NERF_WR;
  xp.rgb_b_off = NERF_BR;
  return launch_exact<exact::IN_NERF>(xp, nerf_xprogram(nullptr), wpack, st);
}

// raw and d raw / d z at S samples per ray on the split-precision kernel: a primal pass that also records the ReLU masks, then
// the tangent pass t_k = mask_k * (W_k t_{k-1}) over the same packed weights (mlp_exact.cuh, IN_NERF_MASK / IN_NERF_TAN).
// Rows are the n_rays * S sample points; row r belongs to ray r / S.
static size_t jvp_rows(int n_rays, int S) {
  return n_rays > 0 && S > 0 ? static_cast<size_t>(n_rays) * static_cast<size_t>(S) : 0;
}
extern "C" size_t b200nerf_nerf_samples_jvp_packed_ws_bytes(int n_rays, int S) {
  return static_cast<size_t>(exact::MAX_STEPS) * jvp_rows(n_rays, S) * 4 * sizeof(unsigned long long);
}
extern "C" size_t b200nerf_nerf_point_jvp_packed_ws_bytes(int n_rays) { return b200nerf_nerf_samples_jvp_packed_ws_bytes(n_rays, 1); }

// tan_axis < 0: one tangent pass along rays_d (d / dz); 0..2: the pass for unit direction e_axis at explicit pts (d / d pts)
static int nerf_jvp_packed(const char* who, const void* wpack, const float* aux, const float* rays_o, const float* rays_d,
                           const float* viewdirs, const float* z, const float* pts, int n_rays, int S, void* ws, float* out_raw,
                           float* out_tan, cudaStream_t st) {
  if (n_rays < 0 || S < 1) return fail("%s: bad sizes n_rays=%d S=%d", who, n_rays, S);
  if (n_rays == 0) return 0;
  if (jvp_rows(n_rays, S) > 0x7fffffffull) return fail("%s: n_rays * S = %lld sample points exceed 2^31 - 1", who,
                                                       static_cast<long long>(n_rays) * S);
  exact::ExactParams xp;
  memset(&xp, 0, sizeof(xp));
  xp.aux = aux;
  xp.n_rows = n_rays * S;
  xp.S = S;
  xp.rays_o = rays_o;
  xp.rays_d = rays_d;
  xp.viewdirs = viewdirs;
  xp.z = z;
  xp.pts = pts;
  xp.mask = static_cast<unsigned long long*>(ws);
  xp.head_w_off = NERF_WA;
  xp.head_b_off = NERF_BA;
  xp.rgb_w_off = NERF_WR;
  xp.rgb_b_off = NERF_BR;
  xp.tan_axis = -1;
  const XProgram pg = nerf_xprogram(nullptr);
  xp.out = out_raw;
  if (launch_exact<exact::IN_NERF_MASK>(xp, pg, wpack, st)) return 1;
  if (pts == nullptr) {
    xp.out = out_tan;
    return launch_exact<exact::IN_NERF_TAN>(xp, pg, wpack, st);
  }
  for (int axis = 0; axis < 3; ++axis) {   // out_tan [rows, 3, 4]: the pass for axis k writes slot k of every row
    xp.tan_axis = axis;
    xp.out = out_tan + 4 * axis;
    if (launch_exact<exact::IN_NERF_TAN>(xp, pg, wpack, st)) return 1;
  }
  return 0;
}

extern "C" int b200nerf_nerf_samples_jvp_packed(const void* wpack, const float* aux, const float* rays_o, const float* rays_d,
                                                const float* viewdirs, const float* z, int n_rays, int S, void* ws, float* out_raw,
                                                float* out_draw_dz, void* stream) {
  if (n_rays > 0 && (!wpack || !aux || !rays_o || !rays_d || !viewdirs || !z || !ws || !out_raw || !out_draw_dz))
    return fail("b200nerf_nerf_samples_jvp_packed: null argument");
  return nerf_jvp_packed("b200nerf_nerf_samples_jvp_packed", wpack, aux, rays_o, rays_d, viewdirs, z, nullptr, n_rays, S, ws,
                         out_raw, out_draw_dz, static_cast<cudaStream_t>(stream));
}

extern "C" int b200nerf_nerf_point_jvp_packed(const void* wpack, const float* aux, const float* rays_o, const float* rays_d,
                                              const float* viewdirs, const float* z, int n_rays, void* ws, float* out_raw,
                                              float* out_draw_dz, void* stream) {
  if (n_rays <= 0) return 0;
  if (!wpack || !aux || !rays_o || !rays_d || !viewdirs || !z || !ws || !out_raw || !out_draw_dz)
    return fail("b200nerf_nerf_point_jvp_packed: null argument");
  return nerf_jvp_packed("b200nerf_nerf_point_jvp_packed", wpack, aux, rays_o, rays_d, viewdirs, z, nullptr, n_rays, 1, ws, out_raw,
                         out_draw_dz, static_cast<cudaStream_t>(stream));
}

extern "C" int b200nerf_nerf_pts_jvp_packed(const void* wpack, const float* aux, const float* pts, const float* viewdirs, int n_rays,
                                            int S, void* ws, float* out_raw, float* out_draw_dpts, void* stream) {
  if (n_rays > 0 && (!wpack || !aux || !pts || !viewdirs || !ws || !out_raw || !out_draw_dpts))
    return fail("b200nerf_nerf_pts_jvp_packed: null argument");
  return nerf_jvp_packed("b200nerf_nerf_pts_jvp_packed", wpack, aux, nullptr, nullptr, viewdirs, nullptr, pts, n_rays, S, ws, out_raw,
                         out_draw_dpts, static_cast<cudaStream_t>(stream));
}

// ------------------------------------------------------------------------------------------- cat-layer chain of the training step
// (declarations and the reference lines in host_common.h / mlp_exact.cuh: IN_ACT, IN_JAC)
static XProgram catchain_xprogram(int n_layers, bool forward) {
  XProgram pg;
  const XSeg none = {0, 0, nullptr, 0, 0, 0};
  for (int i = 0; i < n_layers; ++i) {
    XLayer l;
    const bool last = i == n_layers - 1;
    l.st = xstep(8, 0, 0, 0, 8, 8, 2, (forward && last) ? exact::EPI_DEPTH_OUT : exact::EPI_STORE, exact::ACT_LEAKY, 256u * i);
    if (i == 0) {
      l.st.wait_p = 1;   // input columns 0..127
      l.st.wait_v = 2;   // input columns 128..255
    }
    if (last) {
      l.st.sig_p = 1;
      l.st.sig_v = 2;
    }
    l.n_out = 256;
    l.segs[0] = XSeg{0, 16, nullptr, 256, 0, 256};
    l.segs[1] = none;
    l.n_segs = 1;
    pg.layers.push_back(l);
  }
  return pg;
}
size_t b200_catchain_img_bytes(int n_layers) { return catchain_xprogram(n_layers, true).pack_bytes(); }
size_t b200_catchain_aux_floats() { return exact::AUX_FLOATS; }
size_t b200_catchain_mask_words(int n_layers, int n_rows) { return static_cast<size_t>(n_layers + 1) * static_cast<size_t>(n_rows) * 4; }

struct ChainPackArgs {
  const float* W[B200_CATCHAIN_MAX_LAYERS];    // forward image: layer l streams W[l]; transposed image: W[n_layers - 1 - l]^T
  const float* b[B200_CATCHAIN_MAX_LAYERS];
  const float* head_w;
  const float* head_b;
  const float* in_bias;
  int n_layers;
};
// The layout of pack_xprogram for 256 x 256 layers (per rank: layer -> [half 0: K blocks 0..7][half 1: 0..7][half 0: 8..15][half 1:
// 8..15]; a block = hi piece | lo piece of this rank's 64 rows x 16 k), one element per thread.  blockIdx.y: 0 = W, 1 = W^T, 2 = aux.
__global__ void __launch_bounds__(256) catchain_pack_kernel(const __grid_constant__ ChainPackArgs a, uint8_t* __restrict__ img_fwd,
                                                            uint8_t* __restrict__ img_jac, float* __restrict__ aux) {
  const int t = blockIdx.x * 256 + threadIdx.x;
  if (blockIdx.y == 2) {
    if (t < exact::AUX_FLOATS) {
      float v = 0.f;
      const int l = t >> 8, c = t & 255;
      if (l < a.n_layers) v = a.b[l][c];
      else if (l == a.n_layers) v = a.head_w[c];
      else if (l == a.n_layers + 1 && c == 0) v = a.head_b[0];
      else if (l == a.n_layers + 2 && a.in_bias != nullptr) v = a.in_bias[c];
      aux[t] = v;
    }
    return;
  }
  const int per_layer = 32 * 1024, per_rank = a.n_layers * per_layer;   // elements (one hi + one lo bf16 each)
  if (t >= 2 * per_rank) return;
  const int r = t / per_rank, rem0 = t % per_rank;
  const int l = rem0 / per_layer, rem1 = rem0 % per_layer;
  const int bi = rem1 >> 10, idx = rem1 & 1023;
  const int range = bi >> 4, half = (bi >> 3) & 1, kb = range * 8 + (bi & 7);
  const int kc = idx >> 9, rem = idx & 511;
  const int n = (rem >> 6) * 8 + ((rem >> 3) & 7), e = rem & 7;
  const int k = kb * 16 + kc * 8 + e, row = half * 128 + r * 64 + n;
  const float w = blockIdx.y == 0 ? a.W[l][row * 256 + k] : a.W[a.n_layers - 1 - l][k * 256 + row];
  const __nv_bfloat16 h = __float2bfloat16_rn(w);
  const __nv_bfloat16 lo = __float2bfloat16_rn(w - __bfloat162float(h));
  uint8_t* img = blockIdx.y == 0 ? img_fwd : img_jac;
  uint8_t* blk = img + (static_cast<size_t>(r) * per_rank + static_cast<size_t>(l) * per_layer + static_cast<size_t>(bi) * 1024) * 4;
  reinterpret_cast<__nv_bfloat16*>(blk)[idx] = h;
  reinterpret_cast<__nv_bfloat16*>(blk + 2048)[idx] = lo;
}
int b200_catchain_pack(const float* const* W, const float* const* b, const float* head_w, const float* head_b, const float* in_bias,
                       int n_layers, void* img_fwd, void* img_jac, float* aux, cudaStream_t st) {
  if (n_layers < 1 || n_layers > B200_CATCHAIN_MAX_LAYERS || n_layers > exact::MAX_STEPS) return fail("catchain pack: %d layers", n_layers);
  if (in_bias != nullptr && 256 * (n_layers + 3) > exact::AUX_FLOATS) return fail("catchain pack: no room for the input bias with %d layers", n_layers);
  ChainPackArgs a;
  memset(&a, 0, sizeof(a));
  for (int i = 0; i < n_layers; ++i) {
    a.W[i] = W[i];
    a.b[i] = b[i];
  }
  a.head_w = head_w;
  a.head_b = head_b;
  a.in_bias = in_bias;
  a.n_layers = n_layers;
  const int elems = 2 * n_layers * 32 * 1024;
  catchain_pack_kernel<<<dim3((elems + 255) / 256, 3), 256, 0, st>>>(a, static_cast<uint8_t*>(img_fwd), static_cast<uint8_t*>(img_jac), aux);
  LAUNCH_CHECK();
  return 0;
}
/* diagnostics: the device-side re-pack alone, so that a test can compare it byte for byte with the host packer of the inference
   path (b200nerf_depthnet_pack over the same matrices produces the same program: n_layers steps of 256 x 256) */
extern "C" int b200nerf_debug_catchain_pack(const float* const* d_W, const float* const* d_b, const float* d_head_w, const float* d_head_b,
                                            int n_layers, void* d_img_fwd, void* d_img_jac, float* d_aux, void* stream) {
  if (!d_W || !d_b || !d_head_w || !d_head_b || !d_img_fwd || !d_img_jac || !d_aux) return fail("b200nerf_debug_catchain_pack: null argument");
  return b200_catchain_pack(d_W, d_b, d_head_w, d_head_b, nullptr, n_layers, d_img_fwd, d_img_jac, d_aux, static_cast<cudaStream_t>(stream));
}
extern "C" size_t b200nerf_debug_catchain_img_bytes(int n_layers) { return b200_catchain_img_bytes(n_layers); }

static void catchain_params(exact::ExactParams& xp, const float* aux, int n_layers, int n_rows, float near_, float far_) {
  memset(&xp, 0, sizeof(xp));
  xp.aux = aux;
  xp.n_rows = n_rows;
  xp.S = 1;
  xp.head_w_off = 256 * n_layers;
  xp.head_b_off = 256 * (n_layers + 1);
  xp.near = near_;
  xp.far = far_;
  xp.mask_slope = 0.01f;
}
int b200_catchain_fwd(const void* img_fwd, const float* aux, int n_layers, float* in_act, bool in_is_preact, int n_rows, float near_,
                      float far_, float* const* save, unsigned long long* mask, float* out_z, float* out_s, cudaStream_t st) {
  exact::ExactParams xp;
  catchain_params(xp, aux, n_layers, n_rows, near_, far_);
  xp.in_act = in_act;
  xp.in_bias_off = in_is_preact ? 256 * (n_layers + 2) : -1;
  xp.mask = mask;
  xp.out = out_z;
  xp.out2 = out_s;
  for (int i = 0; i < n_layers; ++i) xp.save[i] = save[i];
  return launch_exact<exact::IN_ACT>(xp, catchain_xprogram(n_layers, true), img_fwd, st);
}
int b200_catchain_jac(const void* img_jac, const float* aux, int n_layers, const float* s, int n_rows, float near_, float far_,
                      float* j_last, float* const* save, const unsigned long long* mask, cudaStream_t st) {
  exact::ExactParams xp;
  catchain_params(xp, aux, n_layers, n_rows, near_, far_);
  xp.sgm = s;
  xp.in_bias_off = -1;
  xp.mask = const_cast<unsigned long long*>(mask);
  xp.out2 = j_last;
  for (int i = 0; i < n_layers; ++i) xp.save[i] = save[i];
  return launch_exact<exact::IN_JAC>(xp, catchain_xprogram(n_layers, false), img_jac, st);
}

extern "C" int b200nerf_nerf_mlp_fwd(const void* wpack, const float* aux, int prec, const float* rays_o, const float* rays_d,
                                     const float* viewdirs, const float* z, const float* pts, int n_rays, int S, float* out_raw,
                                     void* stream) {
  if (n_rays < 0 || S < 1) return fail("b200nerf_nerf_mlp_fwd: bad sizes n_rays=%d S=%d", n_rays, S);
  if (n_rays == 0) return 0;
  if (!wpack || !aux || !viewdirs || !out_raw) return fail("b200nerf_nerf_mlp_fwd: null argument");
  if (!pts && (!z || !rays_o || !rays_d)) return fail("b200nerf_nerf_mlp_fwd: need pts or (rays_o, rays_d, z)");
  if (prec != B200NERF_PREC_SPLIT) return fail("b200nerf_nerf_mlp_fwd: prec must be B200NERF_PREC_SPLIT");
  if (static_cast<long long>(n_rays) * S > 0x7fffff00LL) return fail("b200nerf_nerf_mlp_fwd: too many points for one call");
  return nerf_exact_launch(wpack, aux, rays_o, rays_d, viewdirs, z, pts, n_rays, S, out_raw, nullptr, nullptr, 0,
                           static_cast<cudaStream_t>(stream));
}

extern "C" int b200nerf_depthnet_fwd(const void* wpack, const float* aux, int n_hidden, int prec, const float* rays_o,
                                     const float* rays_d, int n_rays, float radius, float near_, float far_, float* out_z,
                                     void* stream) {
  if (n_rays < 0) return fail("b200nerf_depthnet_fwd: bad n_rays");
  if (n_rays == 0) return 0;
  if (!wpack || !aux || !rays_o || !rays_d || !out_z) return fail("b200nerf_depthnet_fwd: null argument");
  if (depthnet_check("b200nerf_depthnet_fwd", n_hidden, prec)) return 1;
  exact::ExactParams xp;
  memset(&xp, 0, sizeof(xp));
  xp.aux = aux;
  xp.n_rows = n_rays;
  xp.S = 1;
  xp.rays_o = rays_o;
  xp.rays_d = rays_d;
  xp.out = out_z;
  xp.head_w_off = 256 * (n_hidden + 1);
  xp.head_b_off = 256 * (n_hidden + 2);
  xp.radius = radius;
  xp.near = near_;
  xp.far = far_;
  return launch_exact<exact::IN_DEPTHNET>(xp, depthnet_xprogram(nullptr, nullptr, n_hidden), wpack, static_cast<cudaStream_t>(stream));
}


// ------------------------------------------------------------------------------------------- fast NeRF MLP
// The weight pack viewed as [bytes/512, 256] 16-bit elements; a box of `rows` rows is a contiguous rows*512-byte piece.
static int make_piece_tmap(const void* wpack, int rows, fast::TMap* out) {
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) return fail("cuTensorMapEncodeTiled is not available from the driver");
  static_assert(sizeof(CUtensorMap) == sizeof(fast::TMap), "tensor map size");
  const cuuint64_t gdim[2] = {256, fast::WPACK_BYTES / 512};
  const cuuint64_t gstride[1] = {512};
  const cuuint32_t box[2] = {256, static_cast<cuuint32_t>(rows)};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(reinterpret_cast<CUtensorMap*>(out), CU_TENSOR_MAP_DATA_TYPE_UINT16, 2, const_cast<void*>(wpack), gdim,
                         gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled failed (%d)", static_cast<int>(r));
  return 0;
}

template <bool FP16>
static int launch_fast(const fast::FastParams& p, cudaStream_t st) {
  static int grid_caps[B200_MAX_DEVICES] = {0};
  const int dev = b200_device();
  if (dev < 0) return fail("nerf_fast_kernel: no usable CUDA device");
  int& grid_cap = grid_caps[dev];
  constexpr int smem = fast::smem_bytes();
  constexpr int NCTA = fast::NCTA;
  auto kern = fast::nerf_fast_kernel<FP16>;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = NCTA;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.blockDim = dim3(fast::THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (grid_cap == 0) {
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const int sms = sm_count();
    if (sms <= 0) return fail("no CUDA device");
    int cap = (sms / NCTA) * NCTA;
    // a persistent grid must be co-resident: ask how many CTA pairs fit
    cfg.gridDim = dim3(cap);
    int n_clusters = 0;
    CUDA_TRY(cudaOccupancyMaxActiveClusters(&n_clusters, kern, &cfg));
    if (n_clusters <= 0) return fail("nerf_fast_kernel: no resident cluster fits");
    if (n_clusters * NCTA < cap) cap = n_clusters * NCTA;
    grid_cap = cap;
  }
  const int tiles = (p.n_rows + fast::TILE_M - 1) / fast::TILE_M;
  const int units = (tiles + 2 * NCTA - 1) / (2 * NCTA);
  int grid = units * NCTA;
  if (grid > grid_cap) grid = grid_cap;
  if (g_sm_limit >= NCTA && grid > g_sm_limit) grid = (g_sm_limit / NCTA) * NCTA;
  cfg.gridDim = dim3(grid);
  fast::TMap tm_full;
  const int rc = make_piece_tmap(p.wpack, 16, &tm_full);   // one ring stage: 8 KB of this CTA's weight pieces
  if (rc) return rc;
  CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, p, tm_full));
  LAUNCH_CHECK();
  return 0;
}

static long long* g_timeline = nullptr;
/* debug hook (only effective in -DB200NERF_TIMELINE builds): device buffer of 3*80*4 int64 clock stamps */
extern "C" void b200nerf_debug_set_timeline(long long* dev_buf) { g_timeline = dev_buf; }

extern "C" int b200nerf_nerf_mlp_fast_fwd(const void* wpack_fast, const float* aux, int prec, const float* rays_o,
                                          const float* rays_d, const float* viewdirs, const float* z, const float* pts,
                                          int n_rays, int S, float* out_raw, int* guard_count, int* guard_list, int guard_cap,
                                          float guard_kappa, void* stream) {
  if (n_rays < 0 || S < 1) return fail("b200nerf_nerf_mlp_fast_fwd: bad sizes n_rays=%d S=%d", n_rays, S);
  if (n_rays == 0) return 0;
  if (!wpack_fast || !aux || !viewdirs || !out_raw) return fail("b200nerf_nerf_mlp_fast_fwd: null argument");
  if (!pts && (!z || !rays_o || !rays_d)) return fail("b200nerf_nerf_mlp_fast_fwd: need pts or (rays_o, rays_d, z)");
  if (prec != B200NERF_PREC_FP16) return fail("b200nerf_nerf_mlp_fast_fwd: prec must be B200NERF_PREC_FP16");
  if (static_cast<long long>(n_rays) * S > 0x7ffff000LL) return fail("b200nerf_nerf_mlp_fast_fwd: too many points for one call");
  if (guard_count && (!guard_list || guard_cap <= 0)) return fail("b200nerf_nerf_mlp_fast_fwd: guard list missing");
  fast::FastParams p;
  memset(&p, 0, sizeof(p));
  p.wpack = static_cast<const uint8_t*>(wpack_fast);
  p.aux = aux;
  p.n_rows = n_rays * S;
  p.S = S;
  p.rays_o = rays_o;
  p.rays_d = rays_d;
  p.viewdirs = viewdirs;
  p.z = z;
  p.pts = pts;
  p.out = out_raw;
  p.guard_count = guard_count;
  p.guard_list = guard_list;
  p.guard_cap = guard_cap;
  p.guard_kappa = guard_kappa;
  p.timeline = g_timeline;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return launch_fast<true>(p, st);
}

extern "C" int b200nerf_nerf_mlp_guarded_fwd(const void* wpack_fast, const void* wpack_split, const float* aux, int prec,
                                             const float* rays_o, const float* rays_d, const float* viewdirs, const float* z,
                                             const float* pts, int n_rays, int S, float guard_kappa, int* ws_guard,
                                             float* out_raw, void* stream) {
  if (n_rays == 0) return 0;
  if (!ws_guard || !wpack_split) return fail("b200nerf_nerf_mlp_guarded_fwd: null argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // ws_guard[0] = number of flagged points, ws_guard[4 .. 4+n_rays) = their indices (at most one per ray)
  CUDA_TRY(cudaMemsetAsync(ws_guard, 0, 4 * sizeof(int), st));
  int rc = b200nerf_nerf_mlp_fast_fwd(wpack_fast, aux, prec, rays_o, rays_d, viewdirs, z, pts, n_rays, S, out_raw, ws_guard,
                                      ws_guard + 4, n_rays, guard_kappa, stream);
  if (rc) return rc;
  // re-evaluate the flagged points in split precision, in place
  return nerf_exact_launch(wpack_split, aux, rays_o, rays_d, viewdirs, z, pts, n_rays, S, out_raw, ws_guard + 4, ws_guard, n_rays, st);
}

// ------------------------------------------------------------------------------------------- fused render
extern "C" int b200nerf_nerf_query(const b200nerf_nerf_model* nerf, const float* rays_o, const float* rays_d,
                                   const float* viewdirs, const float* z, const float* pts, int n_rays, int S, int* ws_guard,
                                   float* out_raw, void* stream) {
  if (!nerf) return fail("b200nerf_nerf_query: null model");
  switch (nerf->prec) {
    case B200NERF_PREC_SPLIT:
      return b200nerf_nerf_mlp_fwd(nerf->wpack, nerf->aux, nerf->prec, rays_o, rays_d, viewdirs, z, pts, n_rays, S, out_raw, stream);
    case B200NERF_PREC_FP16:
      return b200nerf_nerf_mlp_fast_fwd(nerf->wpack_fast, nerf->aux, B200NERF_PREC_FP16, rays_o, rays_d, viewdirs, z, pts, n_rays, S,
                                        out_raw, nullptr, nullptr, 0, 0.f, stream);
    case B200NERF_PREC_FAST:
      return b200nerf_nerf_mlp_guarded_fwd(nerf->wpack_fast, nerf->wpack, nerf->aux, B200NERF_PREC_FP16, rays_o, rays_d, viewdirs, z,
                                           pts, n_rays, S, nerf->guard_kappa, ws_guard, out_raw, stream);
    default:
      return fail("b200nerf_nerf_query: unknown precision %d", nerf->prec);
  }
}

static int render_depthnet_impl(const void* dn_wpack, const float* dn_aux, int dn_hidden, int dn_prec,
                                const b200nerf_nerf_model* nerf, const float* rays_o, const float* rays_d, const float* viewdirs,
                                int n_rays, int S, int mode, const float* offsets, float radius, float near_, float far_,
                                float* ws_mean, float* ws_z, float* ws_raw, int* ws_guard, float* out_rgb, float* out_disp,
                                float* out_acc, float* out_depth, float* out_weights, int rs, int ds, void* stream) {
  if (n_rays == 0) return 0;
  if (!ws_mean || !ws_z || !ws_raw || !nerf) return fail("b200nerf_render_depthnet: null workspace or model");
  int rc = b200nerf_depthnet_fwd(dn_wpack, dn_aux, dn_hidden, dn_prec, rays_o, rays_d, n_rays, radius, near_, far_, ws_mean, stream);
  if (rc) return rc;
  // the reference clips uniform placements to the literal [2, 6] (nerf_pytorch/utils.py:241)
  rc = b200nerf_place_samples(ws_mean, offsets, n_rays, S, mode, 2.0f, 6.0f, ws_z, stream);
  if (rc) return rc;
  rc = b200nerf_nerf_query(nerf, rays_o, rays_d, viewdirs, ws_z, nullptr, n_rays, S, ws_guard, ws_raw, stream);
  if (rc) return rc;
  // DepthNet path: noise 0 and white background regardless of the caller's flags (misspelled kwargs,
  // nerf_utils.py:858-865)
  return composite_impl(ws_raw, ws_z, rays_d, nullptr, n_rays, S, 1, out_rgb, out_disp, out_acc, out_depth, out_weights, nullptr,
                        rs, ds, stream);
}

extern "C" int b200nerf_render_depthnet(const void* dn_wpack, const float* dn_aux, int dn_hidden, int dn_prec,
                                        const b200nerf_nerf_model* nerf, const float* rays_o, const float* rays_d,
                                        const float* viewdirs, int n_rays, int S, int mode, const float* offsets, float radius,
                                        float near_, float far_, float* ws_mean, float* ws_z, float* ws_raw, int* ws_guard,
                                        float* out_rgb, float* out_disp, float* out_acc, float* out_depth, float* out_weights,
                                        void* stream) {
  return render_depthnet_impl(dn_wpack, dn_aux, dn_hidden, dn_prec, nerf, rays_o, rays_d, viewdirs, n_rays, S, mode, offsets, radius,
                              near_, far_, ws_mean, ws_z, ws_raw, ws_guard, out_rgb, out_disp, out_acc, out_depth, out_weights, 3, 1,
                              stream);
}

extern "C" int b200nerf_render_depthnet_tile(const void* dn_wpack, const float* dn_aux, int dn_hidden, int dn_prec,
                                             const b200nerf_nerf_model* nerf, const float* rays_o, const float* rays_d,
                                             const float* viewdirs, int n_rays, int S, int mode, const float* offsets,
                                             float radius, float near_, float far_, float* ws_mean, float* ws_z, float* ws_raw,
                                             int* ws_guard, float* out_rgbd, float* out_acc, float* out_depth, float* out_weights,
                                             void* stream) {
  if (!out_rgbd) return fail("b200nerf_render_depthnet_tile: null tile");
  return render_depthnet_impl(dn_wpack, dn_aux, dn_hidden, dn_prec, nerf, rays_o, rays_d, viewdirs, n_rays, S, mode, offsets, radius,
                              near_, far_, ws_mean, ws_z, ws_raw, ws_guard, out_rgbd, out_rgbd + 3, out_acc, out_depth, out_weights, 4,
                              4, stream);
}

static size_t align256(size_t x) { return (x + 255) & ~static_cast<size_t>(255); }

extern "C" size_t b200nerf_render_host_ws_bytes(int n_rays, int S) {
  const size_t n = static_cast<size_t>(n_rays);
  return 3 * align256(n * 3 * 4) + align256(n * 4) /*mean*/ + align256(n * S * 4) /*z*/ + align256(n * S * 16) /*raw*/ +
         align256(n * 3 * 4) /*rgb*/ + align256(n * 4) /*disp*/ + align256((n + 4) * 4) /*guard list*/;
}

extern "C" int b200nerf_render_depthnet_host(const void* dn_wpack, const float* dn_aux, int dn_hidden, int dn_prec,
                                             const b200nerf_nerf_model* nerf, const float* h_rays_o, const float* h_rays_d,
                                             int n_rays, int S, int mode, const float* offsets, float radius, float near_,
                                             float far_, void* d_ws, float* h_rgb, float* h_disp, void* stream) {
  if (n_rays <= 0 || !d_ws || !h_rays_o || !h_rays_d || !h_rgb || !h_disp) return fail("b200nerf_render_depthnet_host: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t n = static_cast<size_t>(n_rays);
  uint8_t* w = static_cast<uint8_t*>(d_ws);
  float* ro = reinterpret_cast<float*>(w); w += align256(n * 12);
  float* rd = reinterpret_cast<float*>(w); w += align256(n * 12);
  float* vd = reinterpret_cast<float*>(w); w += align256(n * 12);
  float* mean = reinterpret_cast<float*>(w); w += align256(n * 4);
  float* zb = reinterpret_cast<float*>(w); w += align256(n * S * 4);
  float* rawb = reinterpret_cast<float*>(w); w += align256(n * S * 16);
  float* rgb = reinterpret_cast<float*>(w); w += align256(n * 12);
  float* disp = reinterpret_cast<float*>(w); w += align256(n * 4);
  int* guard = reinterpret_cast<int*>(w);
  CUDA_TRY(cudaMemcpyAsync(ro, h_rays_o, n * 12, cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(rd, h_rays_d, n * 12, cudaMemcpyHostToDevice, st));
  int rc = b200nerf_normalize_dirs(rd, n_rays, vd, stream);
  if (rc) return rc;
  rc = b200nerf_render_depthnet(dn_wpack, dn_aux, dn_hidden, dn_prec, nerf, ro, rd, vd, n_rays, S, mode, offsets, radius, near_,
                                far_, mean, zb, rawb, guard, rgb, disp, nullptr, nullptr, nullptr, stream);
  if (rc) return rc;
  CUDA_TRY(cudaMemcpyAsync(h_rgb, rgb, n * 12, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(h_disp, disp, n * 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return 0;
}

// ------------------------------------------------------------------------------------------- diagnostics
extern "C" int b200nerf_umma_selftest(const uint16_t* A, const uint16_t* B, float* D, int K, int N, void* stream) {
  if (!A || !B || !D || K % 16 || K <= 0 || K > 128 || N % 16 || N <= 0 || N > 256) return fail("b200nerf_umma_selftest: bad arguments");
  const int smem = (K / 8) * ACT_KC_STRIDE + (K / 8) * N * 16;
  CUDA_TRY(cudaFuncSetAttribute(umma_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  umma_selftest_kernel<<<1, 128, smem, static_cast<cudaStream_t>(stream)>>>(A, B, D, K, N);
  LAUNCH_CHECK();
  return 0;
}
