// Fused NeRF MLP, single-pass 16-bit operands (fp16 or bf16, fp32 accumulate) on tcgen05 tensor cores (sm_100a).
//
// Reference semantics: Trainer.run_network (nerf_pytorch/trainers/Trainer.py:789-806) + NeRF.forward
// (nerf_pytorch/run_nerf_helpers.py:109-134): gamma(pts) 3 (1 + 2 multires) wide (63 at multires 10, up to 64), gamma(viewdirs)
// 3 (1 + 2 multires_views) wide (27 at 4, up to 32), 8x256 ReLU trunk
// with the input re-concatenated at layer 5, alpha head, feature layer, 128-wide view layer, rgb head.
//
// Throughput design (one persistent CTA per SM, SMs paired as 2-CTA clusters):
//   * two 128-row tiles ("slots") are resident per CTA and ping-pong: while the tensor core runs layer L of
//     slot 0 the epilogue warps turn the finished accumulator of slot 1 into its next operand, so the tensor
//     pipe never waits for an epilogue that is shorter than one layer of MMAs
//   * the pair issues tcgen05.mma.cta_group::2 (M = 256 over both CTAs); each CTA streams only its half of
//     every weight slab (TMA, cta_group::2 completion on the leader's barrier), which halves L2->SM weight
//     traffic and B-operand shared-memory reads per SM
//   * operands: per slot one K-major no-swizzle buffer of 44 K chunks: [h 0..255 | gamma(pts) 256..319 |
//     gamma(viewdir) 320..351]; every epilogue rewrites h in place (its readers have retired: acc_full)
//   * TMEM: slot 0 accumulates in columns 0..255, slot 1 in 256..511
//   * warp roles: 0 = weight producer (TMA), 1 = MMA issuer, 2 = TMEM allocator, 4-11 = epilogue
//     (tcgen05.ld, + bias, ReLU, 16-bit pack, st.shared; fp32 alpha / rgb heads), 12-15 = encoders
//     (o + d*z, sin/cos octaves) which run one tile ahead of the tensor core
//
// Guard band (optional): raw2outputs turns sigma of the LAST sample of a ray into a step function
// (dist = 1e10, trainers/sampling_trainer.py:178-180), so a rounding error that flips the sign of a tiny sigma
// flips the pixel.  The final epilogue therefore appends every last-of-ray sample with
// |sigma| < kappa * sum_i |h7_i * w_alpha_i| to a list; the caller re-evaluates those points with the
// split-precision kernel (mlp_exact.cuh) and overwrites them.
#pragma once
#include <type_traits>

#include "ptx.cuh"

namespace b200 {
namespace fast {

constexpr int TILE_M = 128;
constexpr int KC_STRIDE = 2048;                       // bytes between 8-element K chunks: 16 row groups x 128 B
constexpr int ENC_KB = 16;                            // K16 block of gamma(pts)      (K chunks 32..39)
constexpr int VIEW_KB = 20;                           // K16 block of gamma(viewdir)  (K chunks 40..43)
constexpr int TILE_KC = 44;
constexpr int TILE_ACT_BYTES = TILE_KC * KC_STRIDE;   // 90,112 B per slot
constexpr int RING_BYTES = 32768;
constexpr int AUX_FLOATS = 3080;                      // the fp32 aux block in global memory (shared with the exact kernel)
constexpr int SF32_FLOATS = 1032;                     // its part kept in shared memory as fp32: alpha layer, view layer, heads
constexpr int SBIAS16 = 7 * 256;                      // 16-bit bias table of the seven plain layers (steps 0-6)
constexpr int THREADS = 512;
constexpr int NSTEPS = 9;
constexpr int EPI_WARP0 = 4, EPI_WARPS = 8, PRO_WARP0 = 12, PRO_WARPS = 4;
constexpr size_t FOLD_BIAS_OFF = 65 * 16384;              // after the 65 ring stages: the folded view-layer bias, 128 fp32
constexpr size_t WPACK_BYTES = FOLD_BIAS_OFF + 512;       // 1,065,472 B

// aux block (float offsets) -- same layout as the split-precision kernel's NeRF aux
enum : uint32_t { AUX_B0 = 0, AUX_BF = 2048, AUX_BV = 2304, AUX_WA = 2432, AUX_BA = 2688, AUX_WR = 2692, AUX_BR = 3076 };
// shared-memory fp32 block (float offsets)
enum : uint32_t { SF_B7 = 0, SF_BV = 256, SF_WA = 384, SF_BA = 640, SF_WR = 644, SF_BR = 1028 };

// The layer program.  Step s reads K16 blocks [kb1, kb1+nk1) then [kb2, kb2+nk2) of the slot's operand buffer.
//   s: 0 = pts_linears.0 (gamma(pts) only), 1-4, 5 = skip layer [h | gamma(pts)], 6, 7 (+ alpha head),
//      8 = views_linears.0 on [h7 | gamma(viewdir)] (N = 128, + rgb head).
// feature_linear has NO activation (run_nerf_helpers.py:116-121: `feature = self.feature_linear(h)` goes straight into
// `views_linears[0](cat([feature, input_views]))`), so it is folded into the view layer when the weights are packed:
//   W' = W_view[:, :256] * W_feature (fp64),  b' = W_view[:, :256] * b_feature + b_view.
// One 256x256 layer (11 % of the network's MACs), its epilogue and one 16-bit rounding of the activations disappear; the
// result is the same function of the same parameters (roofline numbers still count the reference's 1,186,816 FLOP/point).
__host__ __device__ constexpr int step_nk1(int s) { return s == 0 ? 4 : 16; }
__host__ __device__ constexpr int step_kb1(int s) { return s == 0 ? ENC_KB : 0; }
__host__ __device__ constexpr int step_nk2(int s) { return s == 5 ? 4 : (s == NSTEPS - 1 ? 2 : 0); }
__host__ __device__ constexpr int step_kb2(int s) { return s == 5 ? ENC_KB : VIEW_KB; }
__host__ __device__ constexpr int step_n(int s) { return s == NSTEPS - 1 ? 128 : 256; }
__host__ __device__ constexpr int step_nk(int s) { return step_nk1(s) + step_nk2(s); }
// ring stages of a step: one stage = 8 KB per CTA = two K16 blocks at N = 256, four at N = 128 (the view layer,
// whose 18 blocks are padded to 20 with zero weights)
__host__ __device__ constexpr int step_stages(int s) { return s == NSTEPS - 1 ? 5 : step_nk(s) / 2; }
__host__ __device__ constexpr uint32_t step_woff(int s) {  // byte offset of the step's first stage in the pack
  uint32_t o = 0;
  for (int i = 0; i < s; ++i) o += static_cast<uint32_t>(step_stages(i)) * 16384u;
  return o;
}

struct alignas(64) TMap {
  uint8_t bytes[128];
};

struct FastParams {
  const uint8_t* wpack;   // weight slabs in streaming order (fp16 or bf16)
  const float* aux;       // biases + head weights (device)
  int n_rows;             // sample points
  int S;                  // samples per ray
  const float* rays_o;    // [rays,3]
  const float* rays_d;    // [rays,3]
  const float* viewdirs;  // [rays,3]
  const float* z;         // [rays,S] or nullptr
  const float* pts;       // [rows,3] or nullptr
  float* out;             // raw [rows,4]
  int* guard_count;       // nullptr: no guard band
  int* guard_list;        // [guard_cap] point indices to re-evaluate
  int guard_cap;
  float guard_kappa;
  long long* timeline;    // debug builds (-DB200NERF_TIMELINE): clock64 stamps of cluster 0's first units
};

#ifdef B200NERF_TIMELINE
#define TL_STAMP(role, idx, j)                                                                         \
  do {                                                                                                 \
    if (p.timeline != nullptr && blockIdx.x == 0 && (idx) < 80) p.timeline[((role) * 80 + (idx)) * 4 + (j)] = clock64(); \
  } while (0)
#else
#define TL_STAMP(role, idx, j) \
  do {                         \
  } while (0)
#endif

constexpr int NSTAGE = 4;                             // ring stages; one stage = this CTA's half of two K16 slabs
constexpr int STAGE_BYTES = RING_BYTES / NSTAGE;      // 8 KB
constexpr int NCTA = 2;                               // CTAs per cluster (tcgen05 cta_group::2 pair)
#ifndef B200NERF_FAST_STAGGER
#define B200NERF_FAST_STAGGER 5
#endif
constexpr int STAGGER = B200NERF_FAST_STAGGER;                            // slot 1 runs this many steps behind slot 0, so that one slot's
                                                      // epilogue-heavy tile boundary (steps 9, 0) meets the other's MMA-heavy steps

struct __align__(16) Tail {
  uint64_t full[NSTAGE];
  uint64_t empty[NSTAGE];
  uint64_t acc_full[2];
  uint64_t a_ready[2];
  uint64_t enc_ready[2];
  uint64_t view_ready[2];
  uint64_t pts_free[2];
  uint64_t view_free[2];
  uint32_t tmem_base;
  uint32_t pad[3];
  float alpha_part[2][TILE_M];  // column half 1's part of the sigma head, per slot
  float eabs_part[2][TILE_M];   // ... and of sum |h7 * w_alpha|
  float rgb_part[2][3][TILE_M]; // column half 1's part of the rgb head
};

__host__ __device__ constexpr int smem_bytes() {
  return 2 * TILE_ACT_BYTES + RING_BYTES + SF32_FLOATS * 4 + SBIAS16 * 2 + static_cast<int>(sizeof(Tail));
}

// ---------------------------------------------------------------------------------------------
// encoders
// ---------------------------------------------------------------------------------------------
template <bool FP16>
__device__ __forceinline__ void store8(uint8_t* dst, const float (&v)[8]) {
  *reinterpret_cast<uint4*>(dst) = make_uint4(pack_half2<FP16, false>(v[0], v[1]), pack_half2<FP16, false>(v[2], v[3]),
                                              pack_half2<FP16, false>(v[4], v[5]), pack_half2<FP16, false>(v[6], v[7]));
}

// [x, sin(2^0 x), cos(2^0 x), ..., sin(2^(NF-1) x), cos(2^(NF-1) x)] zero-padded to NCHUNK*8 columns
// (run_nerf_helpers.py:15-63).  Octaves 0 and 5 are evaluated with accurate sincosf, the others by exact-angle
// doubling from them (<= 4 doublings: error ~1e-6, far below the 16-bit operand rounding).
template <bool FP16, int NF, int NCHUNK>
__device__ __forceinline__ void encode_store(const float (&x)[3], uint8_t* dst /* first K chunk + row offset */) {
  float sn[NF][3], cs[NF][3];
#pragma unroll
  for (int t = 0; t < 3; ++t) {
    sincosf(x[t], &sn[0][t], &cs[0][t]);
    if (NF > 5) sincosf(x[t] * 32.0f, &sn[5][t], &cs[5][t]);
#pragma unroll
    for (int j = 1; j < NF; ++j) {
      if (j == 5) continue;
      const float s = sn[j - 1][t], c = cs[j - 1][t];
      sn[j][t] = 2.0f * s * c;
      cs[j][t] = (c - s) * (c + s);
    }
  }
  constexpr int NCOL = 3 + 6 * NF;
#pragma unroll
  for (int ch = 0; ch < NCHUNK; ++ch) {
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int cc = ch * 8 + i;
      if (cc < 3) v[i] = x[cc];
      else if (cc < NCOL) v[i] = ((cc - 3) % 6) < 3 ? sn[(cc - 3) / 6][(cc - 3) % 6] : cs[(cc - 3) / 6][(cc - 3) % 6 - 3];
      else v[i] = 0.f;
    }
    store8<FP16>(dst + ch * KC_STRIDE, v);
  }
}

// multires 1..9 / multires_views 1..3, out of line: their encoders stay out of the kernel's hot code.  For j < NF the octave
// values are computed exactly as at NF = 10 / 4 (octave 5 accurate when NF > 5).
template <bool FP16>
__device__ __noinline__ void encode_pts_lt10(int nf, float x0, float x1, float x2, uint8_t* dst) {
  const float x[3] = {x0, x1, x2};   // by value: the call keeps the caller's registers off the stack
  switch (nf) {
    case 1: encode_store<FP16, 1, 8>(x, dst); break;
    case 2: encode_store<FP16, 2, 8>(x, dst); break;
    case 3: encode_store<FP16, 3, 8>(x, dst); break;
    case 4: encode_store<FP16, 4, 8>(x, dst); break;
    case 5: encode_store<FP16, 5, 8>(x, dst); break;
    case 6: encode_store<FP16, 6, 8>(x, dst); break;
    case 7: encode_store<FP16, 7, 8>(x, dst); break;
    case 8: encode_store<FP16, 8, 8>(x, dst); break;
    default: encode_store<FP16, 9, 8>(x, dst); break;
  }
}
template <bool FP16>
__device__ __noinline__ void encode_view_lt4(int nv, float v0, float v1, float v2, uint8_t* dst) {
  const float v[3] = {v0, v1, v2};
  switch (nv) {
    case 1: encode_store<FP16, 1, 4>(v, dst); break;
    case 2: encode_store<FP16, 2, 4>(v, dst); break;
    default: encode_store<FP16, 3, 4>(v, dst); break;
  }
}

// ---------------------------------------------------------------------------------------------
// epilogues (one thread = one accumulator row x one column half)
// ---------------------------------------------------------------------------------------------
// 32 accumulator columns: + bias, activation, pack, 4 x 16-byte operand stores (K chunks kc .. kc+3).
// MODE 0: ReLU   1: ReLU + alpha-head partial sums (+ sum of magnitudes)   3: the same without the magnitudes   2: no activation
template <int MODE, bool FP16>
__device__ __forceinline__ void epi_store32(const uint32_t (&v)[32], const float* bias, const float* hw, uint8_t* dst,
                                            float& hsum, float& habs) {
#pragma unroll
  for (int j = 0; j < 32; j += 8) {
    const float4 b0 = *reinterpret_cast<const float4*>(bias + j);
    const float4 b1 = *reinterpret_cast<const float4*>(bias + j + 4);
    float x[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
    for (int i = 0; i < 8; ++i) x[i] += __uint_as_float(v[j + i]);
    uint32_t h[4];
    if (MODE == 1 || MODE == 3) {
      const float4 w0 = *reinterpret_cast<const float4*>(hw + j);
      const float4 w1 = *reinterpret_cast<const float4*>(hw + j + 4);
      const float w[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        x[i] = fmaxf(x[i], 0.f);
        hsum = fmaf(x[i], w[i], hsum);
        if (MODE == 1) habs = fmaf(x[i], fabsf(w[i]), habs);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) h[i] = pack_half2<FP16, false>(x[2 * i], x[2 * i + 1]);
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) h[i] = pack_half2<FP16, MODE == 0>(x[2 * i], x[2 * i + 1]);
    }
    *reinterpret_cast<uint4*>(dst + (j >> 3) * KC_STRIDE) = make_uint4(h[0], h[1], h[2], h[3]);
  }
}

// relu(x + b) (or x + b) on a packed 16-bit pair in one instruction
template <bool FP16, bool RELU>
__device__ __forceinline__ uint32_t bias_act2(uint32_t x2, uint32_t b2) {
  uint32_t r;
  if (FP16) {
    if (RELU) asm("fma.rn.relu.f16x2 %0, %1, %2, %3;" : "=r"(r) : "r"(x2), "r"(0x3C003C00u), "r"(b2));
    else asm("add.rn.f16x2 %0, %1, %2;" : "=r"(r) : "r"(x2), "r"(b2));
  } else {
    if (RELU) asm("fma.rn.relu.bf16x2 %0, %1, %2, %3;" : "=r"(r) : "r"(x2), "r"(0x3F803F80u), "r"(b2));
    else asm("fma.rn.bf16x2 %0, %1, %2, %3;" : "=r"(r) : "r"(x2), "r"(0x3F803F80u), "r"(b2));
  }
  return r;
}

// Plain layer (no head): the accumulator is rounded to the operand format first, bias and ReLU are applied to the packed
// pairs -- 1.25 instructions per column instead of 1.9 (the epilogue is issue-bound).  Costs one extra 16-bit rounding.
template <bool RELU, bool FP16>
__device__ __forceinline__ void epi_store32_packed(const uint32_t (&v)[32], const uint16_t* bias16, uint8_t* dst) {
#pragma unroll
  for (int j = 0; j < 32; j += 8) {
    const uint4 bb = *reinterpret_cast<const uint4*>(bias16 + j);
    const uint32_t b2[4] = {bb.x, bb.y, bb.z, bb.w};
    uint32_t h[4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
      h[i] = bias_act2<FP16, RELU>(pack_half2<FP16, false>(__uint_as_float(v[j + 2 * i]), __uint_as_float(v[j + 2 * i + 1])), b2[i]);
    *reinterpret_cast<uint4*>(dst + (j >> 3) * KC_STRIDE) = make_uint4(h[0], h[1], h[2], h[3]);
  }
}

template <bool RELU, bool FP16>
__device__ __forceinline__ void epilogue_store_packed(uint32_t tacc, const uint16_t* bias16, uint8_t* dst) {
  uint32_t va[32], vb[32];
  tmem_ld_32x32b_x32(tacc, va);
  tmem_ld_wait();
  tmem_ld_32x32b_x32(tacc + 32, vb);
  epi_store32_packed<RELU, FP16>(va, bias16, dst);
  tmem_ld_wait();
  tmem_ld_32x32b_x32(tacc + 64, va);
  epi_store32_packed<RELU, FP16>(vb, bias16 + 32, dst + 4 * KC_STRIDE);
  tmem_ld_wait();
  tmem_ld_32x32b_x32(tacc + 96, vb);
  epi_store32_packed<RELU, FP16>(va, bias16 + 64, dst + 8 * KC_STRIDE);
  tmem_ld_wait();
  epi_store32_packed<RELU, FP16>(vb, bias16 + 96, dst + 12 * KC_STRIDE);
}

template <int MODE, bool FP16>
__device__ __forceinline__ void epilogue_store(uint32_t tacc, const float* bias, const float* hw, uint8_t* dst,
                                               float& hsum, float& habs) {
  uint32_t va[32], vb[32];
  tmem_ld_32x32b_x32(tacc, va);
  tmem_ld_wait();
  tmem_ld_32x32b_x32(tacc + 32, vb);
  epi_store32<MODE, FP16>(va, bias, hw, dst, hsum, habs);
  tmem_ld_wait();
  tmem_ld_32x32b_x32(tacc + 64, va);
  epi_store32<MODE, FP16>(vb, bias + 32, hw + 32, dst + 4 * KC_STRIDE, hsum, habs);
  tmem_ld_wait();
  tmem_ld_32x32b_x32(tacc + 96, vb);
  epi_store32<MODE, FP16>(va, bias + 64, hw + 64, dst + 8 * KC_STRIDE, hsum, habs);
  tmem_ld_wait();
  epi_store32<MODE, FP16>(vb, bias + 96, hw + 96, dst + 12 * KC_STRIDE, hsum, habs);
}

// view layer: 32 columns of relu(acc + bias) folded into the three rgb dot products
__device__ __forceinline__ void epi_rgb32(const uint32_t (&v)[32], const float* bias, const float* wr, float& r, float& g,
                                          float& b) {
#pragma unroll
  for (int j = 0; j < 32; j += 4) {
    const float4 bb = *reinterpret_cast<const float4*>(bias + j);
    const float4 w0 = *reinterpret_cast<const float4*>(wr + j);
    const float4 w1 = *reinterpret_cast<const float4*>(wr + 128 + j);
    const float4 w2 = *reinterpret_cast<const float4*>(wr + 256 + j);
    const float x0 = fmaxf(__uint_as_float(v[j]) + bb.x, 0.f), x1 = fmaxf(__uint_as_float(v[j + 1]) + bb.y, 0.f);
    const float x2 = fmaxf(__uint_as_float(v[j + 2]) + bb.z, 0.f), x3 = fmaxf(__uint_as_float(v[j + 3]) + bb.w, 0.f);
    r = fmaf(x0, w0.x, r); r = fmaf(x1, w0.y, r); r = fmaf(x2, w0.z, r); r = fmaf(x3, w0.w, r);
    g = fmaf(x0, w1.x, g); g = fmaf(x1, w1.y, g); g = fmaf(x2, w1.z, g); g = fmaf(x3, w1.w, g);
    b = fmaf(x0, w2.x, b); b = fmaf(x1, w2.y, b); b = fmaf(x2, w2.z, b); b = fmaf(x3, w2.w, b);
  }
}

// true when the sample position and view direction of point `grow` are finite (sum of magnitudes < inf)
__device__ __forceinline__ bool input_is_finite(const FastParams& p, int grow) {
  const int ray = grow / p.S;
  float m = 0.f;
  if (p.pts != nullptr) {
#pragma unroll
    for (int t = 0; t < 3; ++t) m += fabsf(__ldg(p.pts + static_cast<size_t>(grow) * 3 + t));
  } else {
    const float zz = __ldg(p.z + grow);
#pragma unroll
    for (int t = 0; t < 3; ++t) m += fabsf(__fadd_rn(__ldg(p.rays_o + ray * 3 + t), __fmul_rn(__ldg(p.rays_d + ray * 3 + t), zz)));
  }
#pragma unroll
  for (int t = 0; t < 3; ++t) m += fabsf(__ldg(p.viewdirs + ray * 3 + t));
  return m < __int_as_float(0x7f800000);
}

// ---------------------------------------------------------------------------------------------
// the kernel
// ---------------------------------------------------------------------------------------------
template <bool FP16>
__global__ void __launch_bounds__(THREADS, 1)
nerf_fast_kernel(const __grid_constant__ FastParams p, const __grid_constant__ TMap tm_full) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* act = smem;
  uint8_t* ring = smem + 2 * TILE_ACT_BYTES;
  float* sf32 = reinterpret_cast<float*>(ring + RING_BYTES);
  uint16_t* sb16 = reinterpret_cast<uint16_t*>(ring + RING_BYTES + SF32_FLOATS * 4);
  Tail* tail = reinterpret_cast<Tail*>(ring + RING_BYTES + SF32_FLOATS * 4 + SBIAS16 * 2);

  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);   // warp-uniform for the compiler
  const int lane = threadIdx.x & 31;
  const uint32_t rank = __shfl_sync(0xffffffffu, cluster_ctarank(), 0);
  const bool leader = rank == 0;
  const int cluster_id = blockIdx.x / NCTA;
  const int n_clusters = gridDim.x / NCTA;
  const int num_tiles = (p.n_rows + TILE_M - 1) / TILE_M;
  const int n_units = (num_tiles + 2 * NCTA - 1) / (2 * NCTA);   // one unit = 2 slots x NCTA tiles
  // units this cluster works through; every role walks the same schedule: tick i runs step (i % 10) of slot 0 and
  // step ((i - STAGGER) % 10) of slot 1
  const int my_units = cluster_id < n_units ? (n_units - cluster_id + n_clusters - 1) / n_clusters : 0;
  const int n_ticks = my_units > 0 ? my_units * NSTEPS + STAGGER : 0;

  if (threadIdx.x == 0) {
    for (int i = 0; i < NSTAGE; ++i) {
      mbar_init(&tail->full[i], 1);
      mbar_init(&tail->empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tail->acc_full[i], 1);
      mbar_init(&tail->a_ready[i], EPI_WARPS * NCTA);
      mbar_init(&tail->enc_ready[i], PRO_WARPS * NCTA);
      mbar_init(&tail->view_ready[i], PRO_WARPS * NCTA);
      mbar_init(&tail->pts_free[i], 1);
      mbar_init(&tail->view_free[i], 1);
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc_cg2(&tail->tmem_base, 512);
    tmem_relinquish_cg2();
  }
  for (int i = threadIdx.x; i < SF32_FLOATS; i += THREADS) {
    // B7 | folded view bias | WA | BA.. | WR | BR..: from the global aux block, the folded bias from the tail of the pack
    if (i >= 256 && i < 384) {
      sf32[i] = reinterpret_cast<const float*>(p.wpack + FOLD_BIAS_OFF)[i - 256];
    } else {
      const uint32_t src = i < 256 ? AUX_B0 + 7 * 256 + i : i < 640 ? AUX_WA + (i - 384)
                         : i < 644 ? AUX_BA + (i - 640) : i < 1028 ? AUX_WR + (i - 644) : AUX_BR + (i - 1028);
      sf32[i] = p.aux[src];
    }
  }
  for (int i = threadIdx.x; i < SBIAS16; i += THREADS) {
    // biases of steps 0..6 in the operand's 16-bit format: the plain-layer epilogue adds them with one packed fma.relu
    // per two columns
    sb16[i] = static_cast<uint16_t>(pack_half2<FP16, false>(p.aux[AUX_B0 + i], 0.f) & 0xffffu);
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, tail->tmem_base, 0);
  const uint32_t tail_addr = smem_u32(tail);
  const uint32_t full_addr = tail_addr + offsetof(Tail, full), empty_addr = tail_addr + offsetof(Tail, empty);

  if (warp == 0) {
    // ===================================================================== weight producer (whole warp, one lane issues)
    if (lane == 0) tma_prefetch_desc(&tm_full);
    const uint32_t ring_addr = smem_u32(ring);
    const uint32_t lead_full = mapa_u32(full_addr, 0);   // both halves complete_tx on the leader's barrier
    uint32_t stage = 0, phase = 0;
    for (int i = 0; i < n_ticks; ++i) {
      for (int slot = 0; slot < 2; ++slot) {
        const int j = i - slot * STAGGER;
        if (j < 0 || j >= my_units * NSTEPS) continue;
        const int s = j % NSTEPS;
        const int n2 = step_stages(s);
        // this CTA's stages of the step are contiguous in the pack: [step][rank][stage][8 KB]
        const int row0 = static_cast<int>((step_woff(s) + rank * static_cast<uint32_t>(n2) * STAGE_BYTES) / 512u);
        for (int k2 = 0; k2 < n2; ++k2) {
          mbar_wait_sleepy(empty_addr + stage * 8u, phase ^ 1u, 100);
          if (elect_one()) {
            if (leader) mbar_arrive_expect_tx_addr(full_addr + stage * 8u, 2u * STAGE_BYTES);
            tma_load_2d_cg2(ring_addr + stage * STAGE_BYTES, &tm_full, 0, row0 + k2 * (STAGE_BYTES / 512), lead_full + stage * 8u);
          }
          __syncwarp();
          if (++stage == NSTAGE) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================================================================== MMA issuer (pair leader; whole warp, one lane issues)
    if (leader) {
      const uint32_t act_addr = smem_u32(act);
      const uint32_t ring_addr = smem_u32(ring);
      const uint32_t acc_full_addr = tail_addr + offsetof(Tail, acc_full);
      const uint32_t a_ready_addr = tail_addr + offsetof(Tail, a_ready);
      const uint32_t enc_ready_addr = tail_addr + offsetof(Tail, enc_ready);
      const uint32_t view_ready_addr = tail_addr + offsetof(Tail, view_ready);
      const uint32_t pts_free_addr = tail_addr + offsetof(Tail, pts_free);
      const uint32_t view_free_addr = tail_addr + offsetof(Tail, view_free);
      constexpr uint32_t A_STEP = (2 * KC_STRIDE) >> 4;   // descriptor increment of one K16 block of the operand
      // descriptors: the high word (SBO, version) is constant, the low word is (address >> 4) | LBO field
      constexpr uint32_t DESC_HI = static_cast<uint32_t>(((128ull >> 4) << 32 | (1ull << 46)) >> 32);
      constexpr uint32_t A_LBO = (KC_STRIDE >> 4) << 16;
      uint32_t stage = 0, phase = 0, ca[2] = {0, 0}, ce[2] = {0, 0}, cv[2] = {0, 0};

      // one ring stage = two K16 blocks: wait for the weights, issue two MMAs, release the stage
      auto issue_stage = [&](auto acc_first, uint32_t d_tmem, uint32_t a_lo, uint32_t b_lbo, uint32_t piece16, uint32_t idesc) {
        mbar_wait_lean(full_addr + stage * 8u, phase);
        tc_fence_after();
        const uint32_t b_lo = b_lbo | ((ring_addr + stage * STAGE_BYTES) >> 4);
        if (elect_one()) {
          const uint64_t a0 = (static_cast<uint64_t>(DESC_HI) << 32) | a_lo;
          const uint64_t b0 = (static_cast<uint64_t>(DESC_HI) << 32) | b_lo;
          tc_mma_f16_cg2_imm<decltype(acc_first)::value>(d_tmem, a0, b0, idesc);
          tc_mma_f16_cg2_imm<true>(d_tmem, a0 + A_STEP, b0 + piece16, idesc);
          tc_commit_cg2_addr(empty_addr + stage * 8u, 3);
        }
        stage = (stage + 1) & (NSTAGE - 1);
        phase ^= (stage == 0);
      };

      // view layer (N = 128): one stage = four K16 blocks; a_lo2 is the operand block of MMAs 2 and 3
      auto issue_stage4 = [&](auto acc_first, auto two_only, uint32_t d_tmem, uint32_t a_lo, uint32_t a_lo2, uint32_t idesc) {
        constexpr uint32_t B_LBO = ((128u * 8u) >> 4) << 16, PIECE16 = 128;
        mbar_wait_lean(full_addr + stage * 8u, phase);
        tc_fence_after();
        const uint32_t b_lo = B_LBO | ((ring_addr + stage * STAGE_BYTES) >> 4);
        if (elect_one()) {
          const uint64_t a0 = (static_cast<uint64_t>(DESC_HI) << 32) | a_lo;
          const uint64_t a2 = (static_cast<uint64_t>(DESC_HI) << 32) | a_lo2;
          const uint64_t b0 = (static_cast<uint64_t>(DESC_HI) << 32) | b_lo;
          tc_mma_f16_cg2_imm<decltype(acc_first)::value>(d_tmem, a0, b0, idesc);
          tc_mma_f16_cg2_imm<true>(d_tmem, a0 + A_STEP, b0 + PIECE16, idesc);
          if (!decltype(two_only)::value) {   // the last stage of the view layer holds two real blocks and two all-zero ones
            tc_mma_f16_cg2_imm<true>(d_tmem, a2, b0 + 2 * PIECE16, idesc);
            tc_mma_f16_cg2_imm<true>(d_tmem, a2 + A_STEP, b0 + 3 * PIECE16, idesc);
          }
          tc_commit_cg2_addr(empty_addr + stage * 8u, 3);
        }
        stage = (stage + 1) & (NSTAGE - 1);
        phase ^= (stage == 0);
      };

#pragma unroll 1
      for (int i = 0; i < n_ticks; ++i) {
#pragma unroll
        for (int slot = 0; slot < 2; ++slot) {
          const int j = i - slot * STAGGER;
          if (j < 0 || j >= my_units * NSTEPS) continue;
          const int s = j % NSTEPS;
          const bool first = j < NSTEPS;
          const int n1 = step_nk1(s) / 2, n2 = step_nk(s) / 2;
          const uint32_t n = static_cast<uint32_t>(step_n(s));
          const uint32_t piece16 = n;                        // (n * 16 bytes) >> 4
          const uint32_t idesc = umma_idesc_f16(FP16 ? 0u : 1u, 256, n);
          const uint32_t b_lbo = ((n * 8u) >> 4) << 16;      // LBO = bytes between the two K chunks of a piece
          const uint32_t kb1 = step_kb1(s), kb2 = step_kb2(s);
          [[maybe_unused]] const int tl_idx = j * 2 + slot;
          if (lane == 0) TL_STAMP(0, tl_idx, 0);
          if (s == 0) {
            mbar_wait_lean(enc_ready_addr + slot * 8u, ce[slot]++ & 1u);
            if (!first) mbar_wait_lean(a_ready_addr + slot * 8u, ca[slot]++ & 1u);
          } else {
            mbar_wait_lean(a_ready_addr + slot * 8u, ca[slot]++ & 1u);
          }
          if (s == NSTEPS - 1) mbar_wait_lean(view_ready_addr + slot * 8u, cv[slot]++ & 1u);
          if (lane == 0) TL_STAMP(0, tl_idx, 1);
          const uint32_t d_tmem = tmem_base + slot * 256u;
          const uint32_t a_base = A_LBO | ((act_addr + slot * TILE_ACT_BYTES) >> 4);
          uint32_t a_lo = a_base + kb1 * A_STEP;
          if (s == NSTEPS - 1) {
            // [feature 0..15 | gamma(viewdir) 20,21 | the same two blocks again under zero weights]
            issue_stage4(std::false_type{}, std::false_type{}, d_tmem, a_lo, a_lo + 2 * A_STEP, idesc);
#pragma unroll 1
            for (int k4 = 1; k4 < 4; ++k4) {
              a_lo += 4 * A_STEP;
              issue_stage4(std::true_type{}, std::false_type{}, d_tmem, a_lo, a_lo + 2 * A_STEP, idesc);
            }
            a_lo = a_base + VIEW_KB * A_STEP;
            issue_stage4(std::true_type{}, std::true_type{}, d_tmem, a_lo, a_lo, idesc);   // gamma(viewdir): blocks 20, 21 only
          } else {
            issue_stage(std::false_type{}, d_tmem, a_lo, b_lbo, piece16, idesc);
            for (int k2 = 1; k2 < n1; ++k2) {
              a_lo += 2 * A_STEP;
              issue_stage(std::true_type{}, d_tmem, a_lo, b_lbo, piece16, idesc);
            }
            a_lo = a_base + kb2 * A_STEP;
            for (int k2 = n1; k2 < n2; ++k2) {
              issue_stage(std::true_type{}, d_tmem, a_lo, b_lbo, piece16, idesc);
              a_lo += 2 * A_STEP;
            }
          }
          if (elect_one()) {
            tc_commit_cg2_addr(acc_full_addr + slot * 8u, 3);
            if (s == 5) tc_commit_cg2_addr(pts_free_addr + slot * 8u, 3);
            if (s == NSTEPS - 1) tc_commit_cg2_addr(view_free_addr + slot * 8u, 3);
          }
          if (lane == 0) TL_STAMP(0, tl_idx, 2);
        }
      }
    }
  } else if (warp >= PRO_WARP0) {
    // ===================================================================== encoders (one tile ahead of the tensor core)
    const int row = (warp - PRO_WARP0) * 32 + lane;
    const int row_off = (row >> 3) * 128 + (row & 7) * 16;
    const uint32_t pts_free_addr = tail_addr + offsetof(Tail, pts_free);
    const uint32_t view_free_addr = tail_addr + offsetof(Tail, view_free);
    const uint32_t enc_bar = mapa_u32(tail_addr + offsetof(Tail, enc_ready), 0);
    const uint32_t view_bar = mapa_u32(tail_addr + offsetof(Tail, view_ready), 0);
    // the image's octave counts sit in the aux slots after the alpha-head bias (0 = 10 / 4, images packed before the slots were
    // used); uniform over the kernel: 10 / 4 run the inline encoders, the smaller sizes the out-of-line ones
    const int nf = static_cast<int>(sf32[SF_BA + 1]), nv = static_cast<int>(sf32[SF_BA + 2]);
    const bool nf_full = nf == 0 || nf == 10, nv_full = nv == 0 || nv == 4;
    uint32_t cp[2] = {0, 0}, cw[2] = {0, 0};
    bool first = true;
    for (int u = cluster_id; u < n_units; u += n_clusters) {
#pragma unroll
      for (int slot = 0; slot < 2; ++slot) {
        const int grow = ((u * NCTA + static_cast<int>(rank)) * 2 + slot) * TILE_M + row;
        float x[3] = {0.f, 0.f, 0.f};
        if (grow < p.n_rows) {
          if (p.pts != nullptr) {
#pragma unroll
            for (int t = 0; t < 3; ++t) x[t] = __ldg(p.pts + static_cast<size_t>(grow) * 3 + t);
          } else {
            const int ray = grow / p.S;
            const float zz = __ldg(p.z + grow);
#pragma unroll
            for (int t = 0; t < 3; ++t)  // o + d*z, product and sum rounded separately like torch
              x[t] = __fadd_rn(__ldg(p.rays_o + ray * 3 + t), __fmul_rn(__ldg(p.rays_d + ray * 3 + t), zz));
          }
        }
        if (!first) {
          mbar_wait_sleepy(pts_free_addr + slot * 8u, cp[slot]++ & 1u, 500);   // the previous tile's skip layer has retired
          tc_fence_after();
        }
        uint8_t* enc_dst = act + slot * TILE_ACT_BYTES + ENC_KB * 2 * KC_STRIDE + row_off;
        if (nf_full) encode_store<FP16, 10, 8>(x, enc_dst);
        else encode_pts_lt10<FP16>(nf, x[0], x[1], x[2], enc_dst);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote(enc_bar + slot * 8u);
        // view encoding of the same tile (its region is released by the previous tile's last step; with the slots
        // staggered the four waits of a unit complete in exactly this order)
        float v[3] = {0.f, 0.f, 0.f};
        if (grow < p.n_rows) {
          const int ray = grow / p.S;
#pragma unroll
          for (int t = 0; t < 3; ++t) v[t] = __ldg(p.viewdirs + ray * 3 + t);
        }
        if (!first) {
          mbar_wait_sleepy(view_free_addr + slot * 8u, cw[slot]++ & 1u, 500);  // the previous tile's view layer has retired
          tc_fence_after();
        }
        uint8_t* view_dst = act + slot * TILE_ACT_BYTES + VIEW_KB * 2 * KC_STRIDE + row_off;
        if (nv_full) encode_store<FP16, 4, 4>(v, view_dst);
        else encode_view_lt4<FP16>(nv, v[0], v[1], v[2], view_dst);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote(view_bar + slot * 8u);
      }
      first = false;
    }
  } else if (warp >= EPI_WARP0) {
    // ===================================================================== epilogue warps
    const int q = warp & 3;                  // TMEM lane quarter this warp may read
    const int hf = (warp - EPI_WARP0) >> 2;  // column half
    const int row = q * 32 + lane;
    const int row_off = (row >> 3) * 128 + (row & 7) * 16;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const uint32_t acc_full_addr = tail_addr + offsetof(Tail, acc_full);
    const uint32_t rdy_bar = mapa_u32(tail_addr + offsetof(Tail, a_ready), 0);
    uint32_t cf[2] = {0, 0};
    float alpha_keep[2] = {0.f, 0.f}, eabs_keep[2] = {0.f, 0.f};

#pragma unroll 1
    for (int i = 0; i < n_ticks; ++i) {
      {
#pragma unroll
        for (int slot = 0; slot < 2; ++slot) {
          const int j = i - slot * STAGGER;
          if (j < 0 || j >= my_units * NSTEPS) continue;
          const int s = j % NSTEPS;
          const int u = cluster_id + (j / NSTEPS) * n_clusters;
          [[maybe_unused]] const int tl_idx = j * 2 + slot;
          if (lane == 0 && q == 0) TL_STAMP(1 + hf, tl_idx, 0);
          mbar_wait_lean(acc_full_addr + slot * 8u, cf[slot]++ & 1u);
          tc_fence_after();
          if (lane == 0 && q == 0) TL_STAMP(1 + hf, tl_idx, 1);
          const uint32_t tacc = t_lane + slot * 256u;
          uint8_t* a_tile = act + slot * TILE_ACT_BYTES;
          if (s < NSTEPS - 1) {
            uint8_t* dst = a_tile + hf * 16 * KC_STRIDE + row_off;
            if (s == 7) {
              float hs = 0.f, ha = 0.f;
              // sum |h7 * w_alpha| feeds the guard-band test, which only looks at the LAST sample of a ray: the 32 rows of this
              // warp need it only when one of them is such a row and a guard list was asked for (warp-uniform)
              const int grow0 = ((u * NCTA + static_cast<int>(rank)) * 2 + slot) * TILE_M + (row & ~31);
              const bool need_abs = p.guard_count != nullptr && (p.S - 1 - grow0 % p.S) < 32;
              if (need_abs) epilogue_store<1, FP16>(tacc + hf * 128, sf32 + SF_B7 + hf * 128, sf32 + SF_WA + hf * 128, dst, hs, ha);
              else epilogue_store<3, FP16>(tacc + hf * 128, sf32 + SF_B7 + hf * 128, sf32 + SF_WA + hf * 128, dst, hs, ha);
              if (hf == 1) {
                tail->alpha_part[slot][row] = hs;
                tail->eabs_part[slot][row] = ha;
              } else {
                alpha_keep[slot] = hs;
                eabs_keep[slot] = ha;
              }
            } else {
              epilogue_store_packed<true, FP16>(tacc + hf * 128, sb16 + s * 256 + hf * 128, dst);
            }
          } else {
            // view layer (128 columns, 64 per column half) + rgb head; sigma = alpha head of layer 7
            float r = 0.f, g = 0.f, b = 0.f;
            uint32_t va[32], vb[32];
            tmem_ld_32x32b_x32(tacc + hf * 64, va);
            tmem_ld_wait();
            tmem_ld_32x32b_x32(tacc + hf * 64 + 32, vb);
            epi_rgb32(va, sf32 + SF_BV + hf * 64, sf32 + SF_WR + hf * 64, r, g, b);
            tmem_ld_wait();
            epi_rgb32(vb, sf32 + SF_BV + hf * 64 + 32, sf32 + SF_WR + hf * 64 + 32, r, g, b);
            if (hf == 1) {
              tail->rgb_part[slot][0][row] = r;
              tail->rgb_part[slot][1][row] = g;
              tail->rgb_part[slot][2][row] = b;
            }
            named_bar_sync(2 + q, 64);   // the two warps of this lane quarter
            if (hf == 0) {
              r += tail->rgb_part[slot][0][row];
              g += tail->rgb_part[slot][1][row];
              b += tail->rgb_part[slot][2][row];
              const int grow = ((u * NCTA + static_cast<int>(rank)) * 2 + slot) * TILE_M + row;
              const bool valid = grow < p.n_rows;
              float sigma = alpha_keep[slot] + tail->alpha_part[slot][row] + sf32[SF_BA];
              if (valid) {
                // The hardware ReLU (cvt.relu / fmaxf) maps NaN to 0, torch.relu keeps it: a sample whose position or
                // view direction is not finite (a ray that missed the sphere has a NaN depth) yields NaN like the reference.
                if (!input_is_finite(p, grow)) r = g = b = sigma = __int_as_float(0x7fc00000);
                reinterpret_cast<float4*>(p.out)[grow] =
                    make_float4(r + sf32[SF_BR], g + sf32[SF_BR + 1], b + sf32[SF_BR + 2], sigma);
              }
              if (p.guard_count != nullptr) {
                const float eabs = eabs_keep[slot] + tail->eabs_part[slot][row] + fabsf(sf32[SF_BA]);
                const bool flag = valid && (grow % p.S) == p.S - 1 && !(fabsf(sigma) >= p.guard_kappa * eabs);
                const uint32_t m = __ballot_sync(0xffffffffu, flag);
                if (m != 0) {
                  int base = 0;
                  if (lane == 0) base = atomicAdd(p.guard_count, __popc(m));
                  base = __shfl_sync(0xffffffffu, base, 0);
                  const int idx = base + __popc(m & ((1u << lane) - 1u));
                  if (flag && idx < p.guard_cap) p.guard_list[idx] = grow;
                }
              }
            }
          }
          // (layer 7's alpha partials, written by the column-half-1 warp of a lane quarter, are read by its half-0 partner after
          // the pair barrier of the last step)
          if (s < NSTEPS - 1) fence_proxy_async_smem();    // operand stores -> visible to the tensor core
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_remote(rdy_bar + slot * 8u);
          if (lane == 0 && q == 0) TL_STAMP(1 + hf, tl_idx, 2);
        }
      }
    }
  }

  __syncwarp();
  tc_fence_before();
  cluster_sync_all();
  if (warp == 2) tmem_dealloc_cg2(tmem_base, 512);
}

}  // namespace fast
}  // namespace b200
