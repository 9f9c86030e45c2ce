// Fused MLP chain in SPLIT precision (bf16 hi + bf16 lo operands, three MMAs per K16 block, fp32 accumulate: ~16 mantissa
// bits) on tcgen05 tensor cores, pipelined inside ONE 128-row tile per CTA, SMs paired as 2-CTA clusters.
//
// Used where the single 16-bit pass of mlp_fast.cuh is not enough: DepthNet.forward (its depth feeds the 2^9 octave of the
// NeRF encoding), the guard band of the fast NeRF pass, and PREC_SPLIT.  Reference semantics:
// (run_nerf_helpers.py:109-134, trainers/Trainer.py:789-806, depth_nets/depth_net.py:117-169).
//
// Two operand planes (hi, lo) of one tile already fill shared memory, so there is no second tile to ping-pong with.
// Instead every layer is cut into two 128-column output HALVES (A, B: separate TMEM accumulators) and two K RANGES:
//
//     P0: A += x[K first]   P1: B += x[K first]   P2: A += x[K second]   P3: B += x[K second]
//
// "K first" = operand columns 0..127 (+ the resident encoding blocks), "K second" = columns 128..255.  Half A is complete
// after P2, so its epilogue (tcgen05.ld, + bias, activation, hi/lo split, st.shared) runs under P3 and rewrites operand
// columns 0..127 IN PLACE -- P3 only reads columns 128..255.  Half B's epilogue runs under the next layer's P0/P1, which
// only read columns 0..127, and rewrites columns 128..255 before the next P2 needs them.  The tensor pipe therefore never
// waits for an epilogue in steady state, with a single tile resident.
//
// The CTA pair issues tcgen05.mma.cta_group::2 (M = 256 over both CTAs, N = 128); each CTA streams only its 64 rows of
// every 128-row weight half (2-D TMA, cta_group::2 completion on the leader's barrier).
#pragma once
#include <type_traits>

#include "ptx.cuh"

namespace b200 {
namespace exact {

constexpr int TILE_M = 128;
constexpr int KC_STRIDE = 2048;
constexpr int ENC_KB = 16;                            // K16 block of gamma(pts)      (K chunks 32..39)
constexpr int VIEW_KB = 20;                           // K16 block of gamma(viewdir)  (K chunks 40..43)
constexpr int TILE_KC = 44;
constexpr int PLANE_BYTES = TILE_KC * KC_STRIDE;      // 90,112 B per plane (hi, lo)
constexpr int RING_BYTES = 32768;
constexpr int NSTAGE = 4;
constexpr int STAGE_BYTES = RING_BYTES / NSTAGE;      // 8 KB = two K16 blocks x (hi piece 2 KB + lo piece 2 KB)
constexpr int AUX_FLOATS = 3080;
constexpr int THREADS = 512;
constexpr int NCTA = 2;
constexpr int MAX_STEPS = 12;
constexpr int EPI_WARP0 = 4, EPI_WARPS = 8, PRO_WARP0 = 12, PRO_WARPS = 4;

// IN_NERF_MASK / IN_NERF_TAN: the training render's forward-mode derivative d raw / d z at one sample per ray (nerf_utils.py:693-715
// under Trainer.core_optimization_loop) as two passes over the SAME packed weights.  The primal pass is IN_NERF plus one 64-bit
// word per (layer, row, 64 columns) of ReLU masks; the tangent pass feeds d gamma(o + d z) / dz through the layers without biases,
// t_k = mask_k * (W_k t_{k-1}), and writes the heads applied to the tangents.
//
// IN_ACT / IN_JAC: DepthNet's activated cat layers in the TRAINING step (depth_nets/depth_net.py:158-169 under
// Trainer.core_optimization_loop), weights re-packed on the device every step.  IN_ACT: rows of fp32 activations in (the output of
// cat_layers.0), the remaining LeakyReLU layers + head, every layer's activations saved in fp32 for the backward, one mask word
// per (layer, row, 64 columns).  IN_JAC: the backward's input-gradient chain with a unit upstream gradient over the TRANSPOSED
// weights, J_{j-1} = (J_j W_j) * LeakyReLU'(a_{j-1}), every J_j saved.  One launch each instead of ten grouped products.
enum : int { IN_NERF = 0, IN_DEPTHNET = 1, IN_NERF_MASK = 2, IN_NERF_TAN = 3, IN_ACT = 4, IN_JAC = 5 };
enum : uint8_t { ACT_NONE = 0, ACT_RELU = 1, ACT_LEAKY = 2, ACT_MASK = 3 };
enum : uint8_t {
  EPI_STORE = 0,        // bias + activation -> next layer's operand (hi/lo planes)
  EPI_STORE_ALPHA = 1,  // as EPI_STORE (ReLU) + this thread's part of the sigma head (N = 1), fp32
  EPI_NERF_OUT = 2,     // N = 128 view layer: bias + ReLU, rgb head (N = 3), write raw [r,g,b,sigma]
  EPI_DEPTH_OUT = 3,    // last DepthNet layer: bias + LeakyReLU, depth head (N = 1), sigmoid, near/far scaling
};

// One layer.  Operand K16 blocks: first range = [kb1a, kb1a+n1a) then [kb1b, kb1b+n1b); second range = [kb2, kb2+n2).
struct XStep {
  uint8_t n1a, kb1a, n1b, kb1b, n2, kb2;
  uint8_t halves;       // 2: N = 256, 1: N = 128 (half A only)
  uint8_t epi, act;
  uint8_t wait_p;       // wait ready_p (encoder part 1) before the first range
  uint8_t wait_v;       // wait ready_v (encoder part 2): 1 = before the first range, 2 = before the second range
  uint8_t sig_p;        // commit free_p after the first range of this step (part-1 region no longer read)
  uint8_t sig_v;        // commit free_v: 1 = after the first range, 2 = after the whole step
  uint8_t pad;
  uint16_t bias_off;    // float offset of the layer's bias in aux
};

struct alignas(64) TMap {
  uint8_t bytes[128];
};

struct ExactParams {
  const float* aux;
  XStep steps[MAX_STEPS];
  int n_steps;
  int stages_per_tile;    // ring stages one tile consumes (pack size / 2 ranks / 8 KB)
  int n_rows;             // points (NeRF) or rays (DepthNet); upper bound when n_rows_dev is set
  int S;
  const float* rays_o;
  const float* rays_d;
  const float* viewdirs;
  const float* z;
  const float* pts;
  float* out;             // raw [rows,4] (NeRF) or z [rows] (DepthNet)
  const int* row_index;   // NeRF, optional: row i evaluates sample point row_index[i] and writes it in place
  const int* n_rows_dev;  // optional: actual row count on the device
  uint8_t* scratch;       // DepthNet: per-CTA staging image of the next tile's encoded input (2 planes x 64 KB)
  unsigned long long* mask;   // IN_NERF_MASK writes / IN_NERF_TAN reads: [step][row][4] words, bit c = output column 64 g + c is > 0
                              // IN_ACT writes [layer 0 .. n_steps][row][4] (layer 0 = the input rows), IN_JAC reads them
  float* save[MAX_STEPS];     // IN_ACT / IN_JAC: fp32 copy of step s's output rows [rows, 256] (null: not saved)
  float* in_act;              // IN_ACT: input rows [rows, 256] fp32
  int in_bias_off;            // IN_ACT, >= 0: the rows are PRE-activations (split-K sums of the layer in front): the loader adds
                              // aux[in_bias_off + c], applies LeakyReLU and writes the activated rows back for the backward
  const float* sgm;           // IN_JAC: s = sigmoid(head) per row (the head's derivative)
  float* out2;                // IN_ACT: s per row;  IN_JAC: the loader's own rows, J of the last layer's pre-activation [rows, 256]
  float mask_slope;           // ACT_MASK: factor of the columns whose bit is clear (0: ReLU, 0.01: LeakyReLU)
  uint32_t head_w_off, head_b_off;   // sigma head (NeRF) / depth head (DepthNet): 256 weights + bias
  uint32_t rgb_w_off, rgb_b_off;     // rgb head [3,128] + bias
  float radius, near, far;
  int tan_axis;               // IN_NERF_TAN: < 0 = tangent along rays_d[ray] (d / dz), 0..2 = along the unit axis (d / d pts[axis]);
                              // an axis pass writes out[row * 3] (the caller offsets out by 4 * axis): out is [rows, 3, 4]
};

struct __align__(16) Tail {
  uint64_t full[NSTAGE];
  uint64_t empty[NSTAGE];
  uint64_t acc_full[2];     // per output half
  uint64_t a_ready[2];      // epilogue of a half finished (operand columns rewritten, accumulator drained)
  uint64_t tmem_free_b;     // half B's accumulator has been read (its stores may still be in flight)
  uint64_t ready_p, ready_v;
  uint64_t free_p, free_v;
  uint64_t in_full[2];      // DepthNet: the staged input halves have landed in the operand planes (TMA bytes)
  uint32_t tmem_base;
  uint32_t pad[3];
  float head_part[4][TILE_M];     // N = 1 head: partial sums per (half, column quarter)
  float rgb_part[3][TILE_M];      // rgb head: column quarter 1's partial sums
};

__host__ __device__ constexpr int smem_bytes() {
  return 2 * PLANE_BYTES + RING_BYTES + AUX_FLOATS * 4 + static_cast<int>(sizeof(Tail));
}

// ---------------------------------------------------------------------------------------------
// operand writes: hi = bf16_rn(x), lo = bf16_rn(x - hi)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void store_split8(uint8_t* dst_hi, const float (&x)[8]) {
  uint32_t h[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    h[i] = pack_bf16x2(x[2 * i], x[2 * i + 1]);
    const float r0 = x[2 * i] - __uint_as_float(h[i] << 16);
    const float r1 = x[2 * i + 1] - __uint_as_float(h[i] & 0xffff0000u);
    l[i] = pack_bf16x2(r0, r1);
  }
  *reinterpret_cast<uint4*>(dst_hi) = make_uint4(h[0], h[1], h[2], h[3]);
  *reinterpret_cast<uint4*>(dst_hi + PLANE_BYTES) = make_uint4(l[0], l[1], l[2], l[3]);
}

// [x, sin(2^0 x), cos(2^0 x), ...] zero-padded to NCHUNK*8 columns, accurate sincosf (run_nerf_helpers.py:15-63)
template <int NF, int NCHUNK>
__device__ __forceinline__ void encode_store(const float (&x)[3], uint8_t* dst) {
  constexpr int NCOL = 3 + 6 * NF;
  float sn[NF][3], cs[NF][3];
#pragma unroll
  for (int j = 0; j < NF; ++j) {
    const float f = static_cast<float>(1 << j);
#pragma unroll
    for (int t = 0; t < 3; ++t) sincosf(x[t] * f, &sn[j][t], &cs[j][t]);
  }
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
    store_split8(dst + ch * KC_STRIDE, v);
  }
}

// d/dz of that encoding at x = o + d z: [d, f cos(f x) d, -f sin(f x) d, ...]
template <int NF, int NCHUNK>
__device__ __forceinline__ void encode_tangent_store(const float (&x)[3], const float (&d)[3], uint8_t* dst) {
  constexpr int NCOL = 3 + 6 * NF;
  float sn[NF][3], cs[NF][3];
#pragma unroll
  for (int j = 0; j < NF; ++j) {
    const float f = static_cast<float>(1 << j);
#pragma unroll
    for (int t = 0; t < 3; ++t) {
      float s_, c_;
      sincosf(x[t] * f, &s_, &c_);
      sn[j][t] = -f * s_ * d[t];   // tangent of the cos column
      cs[j][t] = f * c_ * d[t];    // tangent of the sin column
    }
  }
#pragma unroll
  for (int ch = 0; ch < NCHUNK; ++ch) {
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int cc = ch * 8 + i;
      if (cc < 3) v[i] = d[cc];
      else if (cc < NCOL) v[i] = ((cc - 3) % 6) < 3 ? cs[(cc - 3) / 6][(cc - 3) % 6] : sn[(cc - 3) / 6][(cc - 3) % 6 - 3];
      else v[i] = 0.f;
    }
    store_split8(dst + ch * KC_STRIDE, v);
  }
}

// the same encoding written to a staging image whose lo plane sits `lo_off` bytes after the hi plane
template <int NF, int NCHUNK>
__device__ __forceinline__ void encode_store_img(const float (&x)[3], uint8_t* dst, int lo_off) {
  constexpr int NCOL = 3 + 6 * NF;
  float sn[NF][3], cs[NF][3];
#pragma unroll
  for (int j = 0; j < NF; ++j) {
    const float f = static_cast<float>(1 << j);
#pragma unroll
    for (int t = 0; t < 3; ++t) sincosf(x[t] * f, &sn[j][t], &cs[j][t]);
  }
#pragma unroll
  for (int ch = 0; ch < NCHUNK; ++ch) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float v[2];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int cc = ch * 8 + 2 * i + e;
        if (cc < 3) v[e] = x[cc];
        else if (cc < NCOL) v[e] = ((cc - 3) % 6) < 3 ? sn[(cc - 3) / 6][(cc - 3) % 6] : cs[(cc - 3) / 6][(cc - 3) % 6 - 3];
        else v[e] = 0.f;
      }
      h[i] = pack_bf16x2(v[0], v[1]);
      l[i] = pack_bf16x2(v[0] - __uint_as_float(h[i] << 16), v[1] - __uint_as_float(h[i] & 0xffff0000u));
    }
    *reinterpret_cast<uint4*>(dst + ch * KC_STRIDE) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(dst + ch * KC_STRIDE + lo_off) = make_uint4(l[0], l[1], l[2], l[3]);
  }
}

// DepthNet's input tile in the staging image: enc(o) | enc(d) | enc(hit_near) | enc(hit_far), 64 columns each (NF = multires;
// columns 3 + 6 NF .. 63 of each block are zero)
template <int NF>
__device__ __forceinline__ void depthnet_encode_img(const float (&o)[3], const float (&d)[3], const float (&p0)[3], const float (&p1)[3],
                                                    uint8_t* img) {
  encode_store_img<NF, 8>(o, img, 32 * KC_STRIDE);
  encode_store_img<NF, 8>(d, img + 8 * KC_STRIDE, 32 * KC_STRIDE);
  encode_store_img<NF, 8>(p0, img + 16 * KC_STRIDE, 32 * KC_STRIDE);
  encode_store_img<NF, 8>(p1, img + 24 * KC_STRIDE, 32 * KC_STRIDE);
}

// multires 1..9, out of line: their encoders stay out of the kernel's hot code
__device__ __noinline__ void depthnet_encode_img_lt10(int nf, const float (&o)[3], const float (&d)[3], const float (&p0)[3],
                                                      const float (&p1)[3], uint8_t* img) {
  switch (nf) {
    case 1: depthnet_encode_img<1>(o, d, p0, p1, img); break;
    case 2: depthnet_encode_img<2>(o, d, p0, p1, img); break;
    case 3: depthnet_encode_img<3>(o, d, p0, p1, img); break;
    case 4: depthnet_encode_img<4>(o, d, p0, p1, img); break;
    case 5: depthnet_encode_img<5>(o, d, p0, p1, img); break;
    case 6: depthnet_encode_img<6>(o, d, p0, p1, img); break;
    case 7: depthnet_encode_img<7>(o, d, p0, p1, img); break;
    case 8: depthnet_encode_img<8>(o, d, p0, p1, img); break;
    default: depthnet_encode_img<9>(o, d, p0, p1, img); break;
  }
}

// NeRF at multires 1..9 / multires_views 1..3, out of line like depthnet_encode_img_lt10 (octaves j < NF as at NF = 10 / 4)
__device__ __noinline__ void nerf_encode_pts_lt10(int nf, float x0, float x1, float x2, uint8_t* dst) {
  const float x[3] = {x0, x1, x2};   // by value: the call keeps the caller's registers off the stack
  switch (nf) {
    case 1: encode_store<1, 8>(x, dst); break;
    case 2: encode_store<2, 8>(x, dst); break;
    case 3: encode_store<3, 8>(x, dst); break;
    case 4: encode_store<4, 8>(x, dst); break;
    case 5: encode_store<5, 8>(x, dst); break;
    case 6: encode_store<6, 8>(x, dst); break;
    case 7: encode_store<7, 8>(x, dst); break;
    case 8: encode_store<8, 8>(x, dst); break;
    default: encode_store<9, 8>(x, dst); break;
  }
}
__device__ __noinline__ void nerf_encode_tangent_lt10(int nf, float x0, float x1, float x2, float d0, float d1, float d2,
                                                      uint8_t* dst) {
  const float x[3] = {x0, x1, x2}, d[3] = {d0, d1, d2};
  switch (nf) {
    case 1: encode_tangent_store<1, 8>(x, d, dst); break;
    case 2: encode_tangent_store<2, 8>(x, d, dst); break;
    case 3: encode_tangent_store<3, 8>(x, d, dst); break;
    case 4: encode_tangent_store<4, 8>(x, d, dst); break;
    case 5: encode_tangent_store<5, 8>(x, d, dst); break;
    case 6: encode_tangent_store<6, 8>(x, d, dst); break;
    case 7: encode_tangent_store<7, 8>(x, d, dst); break;
    case 8: encode_tangent_store<8, 8>(x, d, dst); break;
    default: encode_tangent_store<9, 8>(x, d, dst); break;
  }
}
__device__ __noinline__ void nerf_encode_view_lt4(int nv, float v0, float v1, float v2, uint8_t* dst) {
  const float v[3] = {v0, v1, v2};
  switch (nv) {
    case 1: encode_store<1, 4>(v, dst); break;
    case 2: encode_store<2, 4>(v, dst); break;
    default: encode_store<3, 4>(v, dst); break;
  }
}

// eight consecutive floats as ONE 256-bit store (STG.E.256: a full 32-byte sector per lane and instruction; the rows of a tile are
// 1 KB apart, so the lanes of a warp can never share a sector)
__device__ __forceinline__ void st_global_v8(float* p, const float (&x)[8]) {
  asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(x[0]), "f"(x[1]), "f"(x[2]), "f"(x[3]), "f"(x[4]),
               "f"(x[5]), "f"(x[6]), "f"(x[7])
               : "memory");
}

template <int ACT>
__device__ __forceinline__ float act_apply(float x) {
  if (ACT == ACT_RELU) return fmaxf(x, 0.f);
  if (ACT == ACT_LEAKY) return x >= 0.f ? x : x * 0.01f;
  return x;
}

// 64 accumulator columns of one row: + bias, activation, optional heads, optional hi/lo operand store
// WM: collect the ReLU mask of the 64 columns into `mask`; ACT_MASK: no bias, column c passes iff bit c of `mask` is set
// SAVE: fp32 copy of the 64 outputs to gsave
template <int EPI, int ACT, bool WM = false, bool SAVE = false>
__device__ __forceinline__ void epi_cols64(const uint32_t (&va)[32], const uint32_t (&vb)[32], const float* bias, const float* hw,
                                           const float* wr, uint8_t* dst, float& hsum, float& rs, float& gs, float& bs,
                                           unsigned long long& mask, float mslope = 0.f, float* gsave = nullptr) {
  constexpr bool STORE = EPI == EPI_STORE || EPI == EPI_STORE_ALPHA;
  constexpr bool HEAD1 = EPI == EPI_STORE_ALPHA || EPI == EPI_DEPTH_OUT;
#pragma unroll
  for (int cc = 0; cc < 2; ++cc) {
#pragma unroll
    for (int j = 0; j < 32; j += 8) {
      const int c = cc * 32 + j;
      const float4 b0 = *reinterpret_cast<const float4*>(bias + c), b1 = *reinterpret_cast<const float4*>(bias + c + 4);
      float x[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
      if (ACT == ACT_MASK) {
        const uint32_t m8 = static_cast<uint32_t>(mask >> c) & 0xffu;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float a = __uint_as_float(cc == 0 ? va[j + i] : vb[j + i]);
          x[i] = (m8 >> i) & 1u ? a : a * mslope;
        }
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) x[i] = act_apply<ACT>(__uint_as_float(cc == 0 ? va[j + i] : vb[j + i]) + x[i]);
      }
      if (WM) {
        uint32_t m8 = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) m8 |= (x[i] > 0.f ? 1u : 0u) << i;
        mask |= static_cast<unsigned long long>(m8) << c;
      }
      if (SAVE) st_global_v8(gsave + c, x);
      if (HEAD1) {
        const float4 w0 = *reinterpret_cast<const float4*>(hw + c), w1 = *reinterpret_cast<const float4*>(hw + c + 4);
        const float w[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
        for (int i = 0; i < 8; ++i) hsum = fmaf(x[i], w[i], hsum);
      }
      if (EPI == EPI_NERF_OUT) {
#pragma unroll
        for (int i = 0; i < 8; i += 4) {
          const float4 w0 = *reinterpret_cast<const float4*>(wr + c + i);
          const float4 w1 = *reinterpret_cast<const float4*>(wr + 128 + c + i);
          const float4 w2 = *reinterpret_cast<const float4*>(wr + 256 + c + i);
          rs = fmaf(x[i], w0.x, rs); rs = fmaf(x[i + 1], w0.y, rs); rs = fmaf(x[i + 2], w0.z, rs); rs = fmaf(x[i + 3], w0.w, rs);
          gs = fmaf(x[i], w1.x, gs); gs = fmaf(x[i + 1], w1.y, gs); gs = fmaf(x[i + 2], w1.z, gs); gs = fmaf(x[i + 3], w1.w, gs);
          bs = fmaf(x[i], w2.x, bs); bs = fmaf(x[i + 1], w2.y, bs); bs = fmaf(x[i + 2], w2.z, bs); bs = fmaf(x[i + 3], w2.w, bs);
        }
      }
      if (STORE) store_split8(dst + (c >> 3) * KC_STRIDE, x);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// the kernel
// ---------------------------------------------------------------------------------------------
template <int INPUT>
__global__ void __launch_bounds__(THREADS, 1) mlp_exact_kernel(const __grid_constant__ ExactParams p, const __grid_constant__ TMap tm) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* act = smem;   // hi plane, lo plane at + PLANE_BYTES
  uint8_t* ring = smem + 2 * PLANE_BYTES;
  float* saux = reinterpret_cast<float*>(ring + RING_BYTES);
  Tail* tail = reinterpret_cast<Tail*>(ring + RING_BYTES + AUX_FLOATS * 4);

  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const uint32_t rank = __shfl_sync(0xffffffffu, cluster_ctarank(), 0);
  const bool leader = rank == 0;
  const int cluster_id = blockIdx.x / NCTA;
  const int n_clusters = gridDim.x / NCTA;
  int n_rows = p.n_rows;
  if (p.n_rows_dev != nullptr) n_rows = min(__ldg(p.n_rows_dev), p.n_rows);
  const int num_tiles = (n_rows + TILE_M - 1) / TILE_M;
  const int n_units = (num_tiles + NCTA - 1) / NCTA;   // one unit = one tile per CTA of the pair
  const int my_units = cluster_id < n_units ? (n_units - cluster_id + n_clusters - 1) / n_clusters : 0;

  if (threadIdx.x == 0) {
    for (int i = 0; i < NSTAGE; ++i) {
      mbar_init(&tail->full[i], 1);
      mbar_init(&tail->empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tail->acc_full[i], 1);
      mbar_init(&tail->a_ready[i], EPI_WARPS * NCTA);
    }
    mbar_init(&tail->tmem_free_b, EPI_WARPS * NCTA);
    mbar_init(&tail->ready_p, (INPUT == IN_DEPTHNET ? 1 : PRO_WARPS) * NCTA);
    mbar_init(&tail->ready_v, (INPUT == IN_DEPTHNET ? 1 : PRO_WARPS) * NCTA);
    static_assert(INPUT >= IN_NERF && INPUT <= IN_JAC, "input mode");
    mbar_init(&tail->in_full[0], 1);
    mbar_init(&tail->in_full[1], 1);
    mbar_init(&tail->free_p, 1);
    mbar_init(&tail->free_v, 1);
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc_cg2(&tail->tmem_base, 256);
    tmem_relinquish_cg2();
  }
  for (int i = threadIdx.x; i < AUX_FLOATS; i += THREADS) saux[i] = p.aux[i];
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, tail->tmem_base, 0);
  const uint32_t tail_addr = smem_u32(tail);
  const uint32_t full_addr = tail_addr + offsetof(Tail, full), empty_addr = tail_addr + offsetof(Tail, empty);

  if (warp == 0) {
    // ===================================================================== weight producer
    if (lane == 0) tma_prefetch_desc(&tm);
    const uint32_t ring_addr = smem_u32(ring);
    const uint32_t lead_full = mapa_u32(full_addr, 0);
    uint32_t stage = 0, phase = 0;
    // this CTA's stages of a tile are contiguous in the pack: [rank][stage][8 KB], consumed in order
    const int row0 = static_cast<int>(rank) * p.stages_per_tile * (STAGE_BYTES / 512);
    for (int u = 0; u < my_units; ++u) {
      for (int k = 0; k < p.stages_per_tile; ++k) {
        mbar_wait_lean(empty_addr + stage * 8u, phase ^ 1u);
        if (elect_one()) {
          if (leader) mbar_arrive_expect_tx_addr(full_addr + stage * 8u, 2u * STAGE_BYTES);
          tma_load_2d_cg2(ring_addr + stage * STAGE_BYTES, &tm, 0, row0 + k * (STAGE_BYTES / 512), lead_full + stage * 8u);
        }
        __syncwarp();
        if (++stage == NSTAGE) {
          stage = 0;
          phase ^= 1u;
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
      const uint32_t tmem_free_addr = tail_addr + offsetof(Tail, tmem_free_b);
      const uint32_t ready_p_addr = tail_addr + offsetof(Tail, ready_p), ready_v_addr = tail_addr + offsetof(Tail, ready_v);
      const uint32_t free_p_addr = tail_addr + offsetof(Tail, free_p), free_v_addr = tail_addr + offsetof(Tail, free_v);
      constexpr uint32_t A_STEP = (2 * KC_STRIDE) >> 4;
      constexpr uint32_t DESC_HI = static_cast<uint32_t>(((128ull >> 4) << 32 | (1ull << 46)) >> 32);
      constexpr uint32_t A_LBO = (KC_STRIDE >> 4) << 16;
      constexpr uint32_t B_LBO = (1024u >> 4) << 16;      // 64 rows x 16 B between the two K chunks of a piece
      constexpr uint32_t PIECE16 = 2048u >> 4;
      constexpr uint32_t LO16 = PLANE_BYTES >> 4;          // hi plane -> lo plane, in descriptor units
      constexpr uint32_t idesc = umma_idesc_f16(1u, 256, 128);
      const uint32_t a_base = A_LBO | (act_addr >> 4);
      uint32_t stage = 0, phase = 0;
      uint32_t c_ra = 0, c_rb = 0, c_tf = 0, c_p = 0, c_v = 0;   // completed-wait counters (parity) per barrier
      int pend_a = 0, pend_b = 0, pend_tf = 0;                   // arrivals not yet consumed

      // one ring stage = two K16 blocks of one output half: hi*Whi + hi*Wlo + lo*Whi per block
      auto issue_stage = [&](bool fresh, uint32_t d_tmem, uint32_t a_lo) {
        mbar_wait_lean(full_addr + stage * 8u, phase);
        tc_fence_after();
        const uint32_t b_lo = B_LBO | ((ring_addr + stage * STAGE_BYTES) >> 4);
        if (elect_one()) {
          const uint64_t a0 = (static_cast<uint64_t>(DESC_HI) << 32) | a_lo;
          const uint64_t b0 = (static_cast<uint64_t>(DESC_HI) << 32) | b_lo;
          tc_mma_f16_cg2(d_tmem, a0, b0, idesc, fresh ? 0u : 1u);            // block 0: hi * Whi
          tc_mma_f16_cg2_imm<true>(d_tmem, a0, b0 + PIECE16, idesc);         //          hi * Wlo
          tc_mma_f16_cg2_imm<true>(d_tmem, a0 + LO16, b0, idesc);            //          lo * Whi
          tc_mma_f16_cg2_imm<true>(d_tmem, a0 + A_STEP, b0 + 2 * PIECE16, idesc);          // block 1
          tc_mma_f16_cg2_imm<true>(d_tmem, a0 + A_STEP, b0 + 3 * PIECE16, idesc);
          tc_mma_f16_cg2_imm<true>(d_tmem, a0 + A_STEP + LO16, b0 + 2 * PIECE16, idesc);
          tc_commit_cg2_addr(empty_addr + stage * 8u, 3);
        }
        stage = (stage + 1) & (NSTAGE - 1);
        phase ^= (stage == 0);
      };
      auto issue_range = [&](bool fresh, uint32_t d_tmem, int kb, int nblk) {
        uint32_t a_lo = a_base + static_cast<uint32_t>(kb) * A_STEP;
        for (int k = 0; k < nblk; k += 2) {
          issue_stage(fresh && k == 0, d_tmem, a_lo);
          a_lo += 2 * A_STEP;
        }
      };
      auto commit = [&](uint32_t addr) {
        if (elect_one()) tc_commit_cg2_addr(addr, 3);
      };

      for (int u = 0; u < my_units; ++u) {
#pragma unroll 1
        for (int s = 0; s < p.n_steps; ++s) {
          const XStep st = p.steps[s];
          // ---- first K range
          if (st.wait_p) mbar_wait_lean(ready_p_addr, c_p++ & 1u);
          if (st.wait_v == 1) mbar_wait_lean(ready_v_addr, c_v++ & 1u);
          if (pend_a) {   // previous half-A epilogue: operand columns 0..127 rewritten, accumulator A drained
            mbar_wait_lean(a_ready_addr, c_ra++ & 1u);
            --pend_a;
          }
          tc_fence_after();
          issue_range(true, tmem_base, st.kb1a, st.n1a);
          if (st.n1b) issue_range(st.n1a == 0, tmem_base, st.kb1b, st.n1b);
          if (st.n2 == 0) commit(acc_full_addr);
          if (st.halves == 2) {
            if (pend_tf) {   // previous half-B epilogue has read accumulator B
              mbar_wait_lean(tmem_free_addr, c_tf++ & 1u);
              --pend_tf;
            }
            tc_fence_after();
            issue_range(true, tmem_base + 128u, st.kb1a, st.n1a);
            if (st.n1b) issue_range(st.n1a == 0, tmem_base + 128u, st.kb1b, st.n1b);
            if (st.n2 == 0) commit(acc_full_addr + 8u);
          }
          if (st.sig_p) commit(free_p_addr);
          if (st.sig_v == 1) commit(free_v_addr);
          // ---- second K range (operand columns 128..255)
          if (st.n2) {
            if (st.wait_v == 2) mbar_wait_lean(ready_v_addr, c_v++ & 1u);
            if (pend_b) {   // previous half-B epilogue: operand columns 128..255 rewritten
              mbar_wait_lean(a_ready_addr + 8u, c_rb++ & 1u);
              --pend_b;
            }
            tc_fence_after();
            issue_range(false, tmem_base, st.kb2, st.n2);
            commit(acc_full_addr);
            if (st.halves == 2) {
              issue_range(false, tmem_base + 128u, st.kb2, st.n2);
              commit(acc_full_addr + 8u);
            }
          }
          if (st.sig_v == 2) commit(free_v_addr);
          ++pend_a;
          if (st.halves == 2) {
            ++pend_b;
            ++pend_tf;
          }
        }
      }
    }
  } else if (warp >= PRO_WARP0) {
    // ===================================================================== encoders (next tile's network input)
    const int row = (warp - PRO_WARP0) * 32 + lane;
    const int row_off = (row >> 3) * 128 + (row & 7) * 16;
    const uint32_t free_p_addr = tail_addr + offsetof(Tail, free_p), free_v_addr = tail_addr + offsetof(Tail, free_v);
    const uint32_t rp_bar = mapa_u32(tail_addr + offsetof(Tail, ready_p), 0);
    const uint32_t rv_bar = mapa_u32(tail_addr + offsetof(Tail, ready_v), 0);
    for (int u = 0; u < my_units; ++u) {
      const int tile = (cluster_id + u * n_clusters) * NCTA + static_cast<int>(rank);
      const int lrow = tile * TILE_M + row;
      const bool valid = lrow < n_rows;
      if (INPUT == IN_ACT || INPUT == IN_JAC) {
        // one thread per row: 256 fp32 values -> hi / lo operand planes, columns 0..127 then 128..255 (each half as soon as the
        // previous tile has released it).  IN_ACT reads the rows; IN_JAC builds them: J = dt w_head LeakyReLU'(a_last), dt = (far - near) s (1 - s).
        float dt = 0.f;
        if (INPUT == IN_JAC && valid) {
          const float sg = __ldg(p.sgm + lrow);
          dt = (p.far - p.near) * sg * (1.0f - sg);
        }
#pragma unroll 1
        for (int part = 0; part < 2; ++part) {
          if (u > 0) {
            mbar_wait_lean(part == 0 ? free_p_addr : free_v_addr, (u - 1) & 1u);
            tc_fence_after();
          }
#pragma unroll 1
          for (int g = 0; g < 2; ++g) {
            const int col0 = part * 128 + g * 64;
            unsigned long long mbits = 0ull;
            const size_t mi = ((static_cast<size_t>(INPUT == IN_JAC ? p.n_steps : 0) * p.n_rows + static_cast<size_t>(lrow)) << 2) + (col0 >> 6);
            if (INPUT == IN_JAC && valid) mbits = __ldg(p.mask + mi);
#pragma unroll 2
            for (int ch = 0; ch < 8; ++ch) {
              const int c = col0 + ch * 8;
              float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
              if (valid) {
                if (INPUT == IN_ACT) {
                  float* src = p.in_act + static_cast<size_t>(lrow) * 256 + c;
                  const float4 q0 = *reinterpret_cast<const float4*>(src), q1 = *reinterpret_cast<const float4*>(src + 4);
                  v[0] = q0.x; v[1] = q0.y; v[2] = q0.z; v[3] = q0.w; v[4] = q1.x; v[5] = q1.y; v[6] = q1.z; v[7] = q1.w;
                  if (p.in_bias_off >= 0) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[i] = act_apply<ACT_LEAKY>(v[i] + saux[p.in_bias_off + c + i]);
                    st_global_v8(src, v);
                  }
                  uint32_t m8 = 0;
#pragma unroll
                  for (int i = 0; i < 8; ++i) m8 |= (v[i] > 0.f ? 1u : 0u) << i;
                  mbits |= static_cast<unsigned long long>(m8) << (ch * 8);
                } else {
                  const uint32_t m8 = static_cast<uint32_t>(mbits >> (ch * 8)) & 0xffu;
#pragma unroll
                  for (int i = 0; i < 8; ++i) v[i] = dt * saux[p.head_w_off + c + i] * ((m8 >> i) & 1u ? 1.0f : p.mask_slope);
                  st_global_v8(p.out2 + static_cast<size_t>(lrow) * 256 + c, v);
                }
              }
              store_split8(act + (c >> 3) * KC_STRIDE + row_off, v);
            }
            if (INPUT == IN_ACT && valid) p.mask[mi] = mbits;
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive_remote(part == 0 ? rp_bar : rv_bar);
        }
      } else if (INPUT != IN_DEPTHNET) {
        const int grow = valid ? (p.row_index != nullptr ? __ldg(p.row_index + lrow) : lrow) : 0;
        const int ray = grow / p.S;
        float x[3] = {0.f, 0.f, 0.f}, v[3] = {0.f, 0.f, 0.f}, dir[3] = {0.f, 0.f, 0.f};
        if (valid) {
          if (INPUT == IN_NERF_TAN) {
#pragma unroll
            for (int t = 0; t < 3; ++t) dir[t] = p.tan_axis < 0 ? __ldg(p.rays_d + ray * 3 + t) : (t == p.tan_axis ? 1.f : 0.f);
          }
          if (p.pts != nullptr) {
#pragma unroll
            for (int t = 0; t < 3; ++t) x[t] = __ldg(p.pts + static_cast<size_t>(grow) * 3 + t);
          } else {
            const float zz = __ldg(p.z + grow);
#pragma unroll
            for (int t = 0; t < 3; ++t)
              x[t] = __fadd_rn(__ldg(p.rays_o + ray * 3 + t), __fmul_rn(__ldg(p.rays_d + ray * 3 + t), zz));
          }
#pragma unroll
          for (int t = 0; t < 3; ++t) v[t] = __ldg(p.viewdirs + ray * 3 + t);
        }
        if (u > 0) {
          mbar_wait_lean(free_p_addr, (u - 1) & 1u);    // the previous tile's skip layer no longer reads gamma(pts)
          tc_fence_after();
        }
        // the image's octave counts sit in the aux slots after the alpha-head bias (0 = 10 / 4, images packed before the slots were
        // used); uniform over the kernel: 10 / 4 run the inline encoders, the smaller sizes the out-of-line ones
        const int nf = static_cast<int>(saux[p.head_b_off + 1]), nv = static_cast<int>(saux[p.head_b_off + 2]);
        uint8_t* enc_dst = act + ENC_KB * 2 * KC_STRIDE + row_off;
        if (nf == 0 || nf == 10) {
          if (INPUT == IN_NERF_TAN) encode_tangent_store<10, 8>(x, dir, enc_dst);
          else encode_store<10, 8>(x, enc_dst);
        } else {
          if (INPUT == IN_NERF_TAN) nerf_encode_tangent_lt10(nf, x[0], x[1], x[2], dir[0], dir[1], dir[2], enc_dst);
          else nerf_encode_pts_lt10(nf, x[0], x[1], x[2], enc_dst);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote(rp_bar);
        if (u > 0) {
          mbar_wait_lean(free_v_addr, (u - 1) & 1u);    // ... nor its view layer gamma(viewdir)
          tc_fence_after();
        }
        if (INPUT == IN_NERF_TAN) {   // the view direction does not depend on z: a zero block
          const float zero8[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int ch = 0; ch < 4; ++ch) store_split8(act + VIEW_KB * 2 * KC_STRIDE + row_off + ch * KC_STRIDE, zero8);
        } else if (nv == 0 || nv == 4) {
          encode_store<4, 4>(v, act + VIEW_KB * 2 * KC_STRIDE + row_off);
        } else {
          nerf_encode_view_lt4(nv, v[0], v[1], v[2], act + VIEW_KB * 2 * KC_STRIDE + row_off);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive_remote(rv_bar);
      } else {
        // DepthNet: 12 multires (120) accurate sincosf per ray are far too slow to sit between two tiles, so the encoders work one
        // tile AHEAD into a per-CTA staging image in global memory (L2-resident, already in the operand layout); when the
        // previous tile releases the operand columns, one lane pulls the image in with two bulk TMA copies per half.
        //   part 1 = enc(o) | enc(d) -> K chunks 0..15, part 2 = enc(hit_near) | enc(hit_far) -> K chunks 16..31
        uint8_t* stage_img = p.scratch + static_cast<size_t>(blockIdx.x) * (2 * 32 * KC_STRIDE);   // hi 64 KB | lo 64 KB
        float o[3] = {0.f, 0.f, 0.f}, d[3] = {0.f, 0.f, 0.f};
        if (valid) {
#pragma unroll
          for (int t = 0; t < 3; ++t) {
            o[t] = __ldg(p.rays_o + static_cast<size_t>(lrow) * 3 + t);
            d[t] = __ldg(p.rays_d + static_cast<size_t>(lrow) * 3 + t);
          }
        }
        // ray / sphere(0, radius) intersection, op order of nerf_pytorch/utils.py:159-217 (NaN when the ray misses)
        const float dot_do = __fadd_rn(__fadd_rn(__fmul_rn(d[0], o[0]), __fmul_rn(d[1], o[1])), __fmul_rn(d[2], o[2]));
        const float b = __fmul_rn(2.f, dot_do);
        const float on = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(o[0], o[0]), __fmul_rn(o[1], o[1])), __fmul_rn(o[2], o[2])));
        const float cc = __fadd_rn(__fmul_rn(on, on), -__fmul_rn(p.radius, p.radius));
        const float a = __fadd_rn(__fadd_rn(__fmul_rn(d[0], d[0]), __fmul_rn(d[1], d[1])), __fmul_rn(d[2], d[2]));
        const float delta = __fadd_rn(__fmul_rn(b, b), -__fmul_rn(__fmul_rn(4.f, a), cc));
        const float sq = __fsqrt_rn(delta);
        const float two_a = __fmul_rn(2.f, a);
        const float t0 = __fdiv_rn(__fadd_rn(-b, -sq), two_a), t1 = __fdiv_rn(__fadd_rn(-b, sq), two_a);
        float p0[3], p1[3];
#pragma unroll
        for (int t = 0; t < 3; ++t) {
          p0[t] = __fadd_rn(o[t], __fmul_rn(t0, d[t]));
          p1[t] = __fadd_rn(o[t], __fmul_rn(t1, d[t]));
        }
        // the image's multires sits in the aux slot after the head bias (0 = 10, the images packed before the slot was used);
        // uniform over the CTA; multires 10 runs the fixed-10 encoder inline, the smaller sizes sit out of line
        const int nf = static_cast<int>(saux[p.head_b_off + 1]);
        if (nf == 0 || nf == 10) depthnet_encode_img<10>(o, d, p0, p1, stage_img + row_off);
        else depthnet_encode_img_lt10(nf, o, d, p0, p1, stage_img + row_off);
        __threadfence();
        fence_proxy_async_all();                       // generic-proxy global writes -> visible to the bulk copy engine
        named_bar_sync(6, PRO_WARPS * 32);
        if (warp == PRO_WARP0 && lane == 0) {
          const uint32_t in_full_addr = tail_addr + offsetof(Tail, in_full);
          constexpr uint32_t HALF = 16 * KC_STRIDE;     // 32 KB: K chunks 0..15 (or 16..31) of one plane
          if (u > 0) mbar_wait_lean(free_p_addr, (u - 1) & 1u);    // the previous tile's last layer has read columns 0..127
          mbar_arrive_expect_tx(&tail->in_full[0], 2 * HALF);
          tma_load_1d(act, stage_img, HALF, &tail->in_full[0]);
          tma_load_1d(act + PLANE_BYTES, stage_img + 32 * KC_STRIDE, HALF, &tail->in_full[0]);
          mbar_wait_lean(in_full_addr, u & 1u);
          mbar_arrive_remote(rp_bar);
          if (u > 0) mbar_wait_lean(free_v_addr, (u - 1) & 1u);    // ... and columns 128..255
          mbar_arrive_expect_tx(&tail->in_full[1], 2 * HALF);
          tma_load_1d(act + HALF, stage_img + HALF, HALF, &tail->in_full[1]);
          tma_load_1d(act + PLANE_BYTES + HALF, stage_img + 32 * KC_STRIDE + HALF, HALF, &tail->in_full[1]);
          mbar_wait_lean(in_full_addr + 8u, u & 1u);
          mbar_arrive_remote(rv_bar);
        }
        named_bar_sync(6, PRO_WARPS * 32);               // the image is free again
      }
    }
  } else if (warp >= EPI_WARP0) {
    // ===================================================================== epilogue warps
    const int q = warp & 3;                   // TMEM lane quarter
    const int sub = (warp - EPI_WARP0) >> 2;  // 64-column quarter inside the 128-column half
    const int row = q * 32 + lane;
    const int row_off = (row >> 3) * 128 + (row & 7) * 16;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const uint32_t acc_full_addr = tail_addr + offsetof(Tail, acc_full);
    const uint32_t rdy_bar = mapa_u32(tail_addr + offsetof(Tail, a_ready), 0);
    const uint32_t tf_bar = mapa_u32(tail_addr + offsetof(Tail, tmem_free_b), 0);
    uint32_t cf[2] = {0, 0};

    for (int u = 0; u < my_units; ++u) {
      const int tile = (cluster_id + u * n_clusters) * NCTA + static_cast<int>(rank);
      const int lrow = tile * TILE_M + row;
      const bool valid = lrow < n_rows;
      const int grow = (INPUT != IN_DEPTHNET && p.row_index != nullptr) ? (valid ? __ldg(p.row_index + lrow) : 0) : lrow;
      constexpr bool TAN = INPUT == IN_NERF_TAN, WM = INPUT == IN_NERF_MASK;
#pragma unroll 1
      for (int s = 0; s < p.n_steps; ++s) {
        const XStep st = p.steps[s];
#pragma unroll 1
        for (int half = 0; half < st.halves; ++half) {
          mbar_wait_lean(acc_full_addr + half * 8u, cf[half]++ & 1u);
          tc_fence_after();
          const int col0 = half * 128 + sub * 64;           // first accumulator / layer-output column of this thread
          const float* bias = saux + st.bias_off + col0;
          unsigned long long mbits = 0ull;
          // mask layer of this step's output: the step itself (NeRF), s + 1 (IN_ACT: layer 0 is the input), n_steps - 1 - s (IN_JAC:
          // step s produces the gradient of layer n_steps - 1 - s's pre-activation)
          const int mlayer = INPUT == IN_ACT ? s + 1 : (INPUT == IN_JAC ? p.n_steps - 1 - s : s);
          const size_t midx = ((static_cast<size_t>(mlayer) * p.n_rows + static_cast<size_t>(lrow)) << 2) + (col0 >> 6);
          if ((TAN || INPUT == IN_JAC) && valid) mbits = __ldg(p.mask + midx);
          // out-of-range rows of the last tile save into a row that exists (their values are zeros or garbage nobody reads): row 0
          float* gsave = (INPUT == IN_ACT || INPUT == IN_JAC) && p.save[s] != nullptr
                             ? p.save[s] + static_cast<size_t>(valid ? lrow : 0) * 256 + col0 : nullptr;
          uint32_t va[32], vb[32];
          tmem_ld_32x32b_x32(t_lane + col0, va);
          tmem_ld_32x32b_x32(t_lane + col0 + 32, vb);
          tmem_ld_wait();
          if (half == 1) {
            // accumulator B is in registers: the next layer's P1 may overwrite it
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_remote(tf_bar);
          }
          const bool store = st.epi == EPI_STORE || st.epi == EPI_STORE_ALPHA;
          const bool head1 = st.epi == EPI_STORE_ALPHA || st.epi == EPI_DEPTH_OUT;
          const float* hw = saux + p.head_w_off + col0;
          const float* wr = saux + p.rgb_w_off + col0;
          uint8_t* dst = act + (col0 >> 3) * KC_STRIDE + row_off;
          float hsum = 0.f, rs = 0.f, gs = 0.f, bs = 0.f;
          if (INPUT == IN_ACT) {
            if (!valid) gsave = nullptr;
            if (st.epi == EPI_STORE) {
              if (gsave) epi_cols64<EPI_STORE, ACT_LEAKY, true, true>(va, vb, bias, hw, wr, dst, hsum, rs, gs, bs, mbits, 0.f, gsave);
              else epi_cols64<EPI_STORE, ACT_LEAKY, true, false>(va, vb, bias, hw, wr, dst, hsum, rs, gs, bs, mbits);
            } else {
              if (gsave) epi_cols64<EPI_DEPTH_OUT, ACT_LEAKY, true, true>(va, vb, bias, hw, wr, dst, hsum, rs, gs, bs, mbits, 0.f, gsave);
              else epi_cols64<EPI_DEPTH_OUT, ACT_LEAKY, true, false>(va, vb, bias, hw, wr, dst, hsum, rs, gs, bs, mbits);
            }
            if (valid) p.mask[midx] = mbits;
          } else if (INPUT == IN_JAC) {
            if (!valid) gsave = nullptr;
            if (gsave) epi_cols64<EPI_STORE, ACT_MASK, false, true>(va, vb, bias, hw, wr, dst, hsum, rs, gs, bs, mbits, p.mask_slope, gsave);
            else epi_cols64<EPI_STORE, ACT_MASK, false, false>(va, vb, bias, hw, wr, dst, hsum, rs, gs, bs, mbits, p.mask_slope);
          } else if (TAN) {
            if (st.epi == EPI_STORE) epi_cols64<EPI_STORE, ACT_MASK>(va, vb, bias, hw, wr, dst, hsum, rs, gs, bs, mbits);
            else if (st.epi == EPI_STORE_ALPHA) epi_cols64<EPI_STORE_ALPHA, ACT_MASK>(va, vb, bias, hw, wr, dst, hsum, rs, gs, bs, mbits);
            else epi_cols64<EPI_NERF_OUT, ACT_MASK>(va, vb, bias, hw, wr, dst, hsum, rs, gs, bs, mbits);
          } else if (st.epi == EPI_STORE) {
            if (st.act == ACT_RELU) epi_cols64<EPI_STORE, ACT_RELU, WM>(va, vb, bias, hw, wr, dst, hsum, rs, gs, bs, mbits);
            else if (st.act == ACT_LEAKY) epi_cols64<EPI_STORE, ACT_LEAKY>(va, vb, bias, hw, wr, dst, hsum, rs, gs, bs, mbits);
            else epi_cols64<EPI_STORE, ACT_NONE>(va, vb, bias, hw, wr, dst, hsum, rs, gs, bs, mbits);
          } else if (st.epi == EPI_STORE_ALPHA) {
            epi_cols64<EPI_STORE_ALPHA, ACT_RELU, WM>(va, vb, bias, hw, wr, dst, hsum, rs, gs, bs, mbits);
          } else if (st.epi == EPI_NERF_OUT) {
            epi_cols64<EPI_NERF_OUT, ACT_RELU, WM>(va, vb, bias, hw, wr, dst, hsum, rs, gs, bs, mbits);
          } else {
            epi_cols64<EPI_DEPTH_OUT, ACT_LEAKY>(va, vb, bias, hw, wr, dst, hsum, rs, gs, bs, mbits);
          }
          if (WM && valid) p.mask[midx] = mbits;
          if (head1) tail->head_part[half * 2 + sub][row] = hsum;
          if (st.epi == EPI_NERF_OUT) {
            if (sub == 1) {
              tail->rgb_part[0][row] = rs;
              tail->rgb_part[1][row] = gs;
              tail->rgb_part[2][row] = bs;
            }
            named_bar_sync(2 + q, 64);   // the two warps of this lane quarter
            if (TAN) {
              if (sub == 0 && valid)
                reinterpret_cast<float4*>(p.out)[static_cast<size_t>(grow) * (p.tan_axis < 0 ? 1 : 3)] =
                    make_float4(rs + tail->rgb_part[0][row], gs + tail->rgb_part[1][row], bs + tail->rgb_part[2][row],
                                tail->head_part[0][row] + tail->head_part[1][row] + tail->head_part[2][row] + tail->head_part[3][row]);
            } else if (sub == 0 && valid) {
              float4 o4;
              o4.x = rs + tail->rgb_part[0][row] + saux[p.rgb_b_off];
              o4.y = gs + tail->rgb_part[1][row] + saux[p.rgb_b_off + 1];
              o4.z = bs + tail->rgb_part[2][row] + saux[p.rgb_b_off + 2];
              o4.w = tail->head_part[0][row] + tail->head_part[1][row] + tail->head_part[2][row] + tail->head_part[3][row] +
                     saux[p.head_b_off];
              // fmaxf(NaN, 0) = 0 but torch.relu(NaN) = NaN: non-finite inputs yield NaN rows like the reference
              const int ry = grow / p.S;
              float m = 0.f;
              if (p.pts != nullptr) {
#pragma unroll
                for (int t = 0; t < 3; ++t) m += fabsf(__ldg(p.pts + static_cast<size_t>(grow) * 3 + t));
              } else {
                const float zz = __ldg(p.z + grow);
#pragma unroll
                for (int t = 0; t < 3; ++t)
                  m += fabsf(__fadd_rn(__ldg(p.rays_o + ry * 3 + t), __fmul_rn(__ldg(p.rays_d + ry * 3 + t), zz)));
              }
#pragma unroll
              for (int t = 0; t < 3; ++t) m += fabsf(__ldg(p.viewdirs + ry * 3 + t));
              if (!(m < __int_as_float(0x7f800000))) o4.x = o4.y = o4.z = o4.w = __int_as_float(0x7fc00000);
              reinterpret_cast<float4*>(p.out)[grow] = o4;
            }
          }
          if (st.epi == EPI_DEPTH_OUT && half == 1) {
            named_bar_sync(1, EPI_WARPS * 32);   // all four partial sums of every row are in shared memory
            if (sub == 0 && valid) {
              const float t = tail->head_part[0][row] + tail->head_part[1][row] + tail->head_part[2][row] + tail->head_part[3][row] +
                              saux[p.head_b_off];
              const float sg = 1.0f / (1.0f + expf(-t));
              // near*(1-s) + far*s with every product / sum rounded separately (depth_net.py:168)
              p.out[grow] = __fadd_rn(__fmul_rn(p.near, __fadd_rn(1.0f, -sg)), __fmul_rn(p.far, sg));
              if (INPUT == IN_ACT) p.out2[grow] = sg;
            }
            named_bar_sync(1, EPI_WARPS * 32);   // head_part may be rewritten by the next tile
          }
          if (st.epi == EPI_STORE_ALPHA && half == 1) named_bar_sync(1, EPI_WARPS * 32);   // sigma partials visible to the output epilogue
          if (store) fence_proxy_async_smem();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_remote(rdy_bar + half * 8u);
        }
      }
    }
  }

  __syncwarp();
  tc_fence_before();
  cluster_sync_all();
  if (warp == 2) tmem_dealloc_cg2(tmem_base, 256);
}

}  // namespace exact
}  // namespace b200
