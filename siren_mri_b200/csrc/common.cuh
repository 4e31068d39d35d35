// Shared definitions for the siren_b200 kernels: HBM plane layout, parameter blocks,
// bf16 hi/lo split helpers and the sine/cosine used by every epilogue.
//
// HBM layout ("planes").  All hidden-width tensors are row-major [rows, H] with H = 256 and
// rows = R = tasks * n_pad (n_pad = coordinates per task rounded up to 128, pad rows are zero
// coordinates on the way in and carry zero adjoints on the way back).  A layer keeps
//   act  : S planes  [S][R][H] bf16 (+ a second "lo" copy in split mode)   h, J_k, D_k
//   c    : 1 plane   [R][H]    stash type (bf16, or fp32 in split mode)     cos(w0 z)
//   jz   : S-1 planes          stash type                                   Jz_k, Dz_k (pre-activation jets)
//   adj  : S planes  bf16 (+lo)                                             zbar, Jzbar_k, Dzbar_k
// with S = 1 + order * d streams (value, d first derivatives, d second derivatives).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <cstdint>

namespace siren {

constexpr int H = 256;        // hidden width served by the tensor-core kernels
constexpr int TILE_M = 128;   // rows per tile (UMMA M)
constexpr int KCHUNK = 64;    // bf16 elements per 128-byte swizzle row

typedef __nv_bfloat16 bf16;

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float bf16_lo_f(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16_hi_f(uint32_t u) { return __uint_as_float(u & 0xFFFF0000u); }
__device__ __forceinline__ float bf16_round_f(float a) { return __bfloat162float(__float2bfloat16_rn(a)); }

// ---- the stash of the fused bf16 path: the "signed sine" ----
// A hidden sine layer leaves ONE plane behind: h = sin(theta) as fp16 whose LOWEST MANTISSA BIT carries the sign of
// cos(theta).  It is the very tile the next layer's MMA multiplies with (the stolen bit is a relative 2^-11, four
// times finer than the bf16 rounding this mode used to have), so stashing costs no staging, no conversion and no
// extra plane: the forward TMA-stores its operand tile as it is.  The backward kernels read
//   sin(theta) = h                                   (weight-gradient operand, converted to bf16 on chip: no SFU)
//   cos(theta) = +-sqrt(1 - h^2), sign from the bit  (dgrad chain; one MUFU, like the cosine of a stored phase)
// The sign: theta = k pi + r with k = rint(theta / pi), r in [-pi/2, pi/2], so cos(theta) = (-1)^k cos(r) and the
// bit is the parity of k -- the low bit of the pattern of kf = fma(theta, 1/pi, 1.5 * 2^23).
constexpr float SGN_MAGIC = 12582912.0f;          // 1.5 * 2^23
constexpr float SGN_INV_PI = 0.3183098861837907f;
__device__ __forceinline__ uint32_t pack_f16(float a, float b) {
  __half2 v = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float sgn_kf(float theta) { return fmaf(theta, SGN_INV_PI, SGN_MAGIC); }
__device__ __forceinline__ uint32_t pack_sgnsine(float s0, float s1, float kf0, float kf1) {
  const uint32_t h = pack_f16(s0, s1);
  const uint32_t b = __byte_perm(__float_as_uint(kf0), __float_as_uint(kf1), 0x4440);   // byte 0 <- kf0, byte 2 <- kf1
  uint32_t r;      // (h & ~m) | (b & m) as ONE lop3 (the compiler emits two)
  asm("lop3.b32 %0, %1, %2, 0x00010001, 0xD8;" : "=r"(r) : "r"(h), "r"(b));
  return r;
}
// the two sines of a word and |cos| of each; the signs are applied to the packed bf16 PRODUCT (sgnsine_flip)
__device__ __forceinline__ void sgnsine_unpack(uint32_t w, float& h0, float& h1, float& c0, float& c1) {
  const float2 h = __half22float2(*reinterpret_cast<const __half2*>(&w));
  h0 = h.x; h1 = h.y;
  // an h of exactly 1 with the bit set reads as 1 + 2^-10: |.| keeps the root real (cos ~ 0 there anyway)
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(c0) : "f"(fabsf(fmaf(-h.x, h.x, 1.f))));
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(c1) : "f"(fabsf(fmaf(-h.y, h.y, 1.f))));
}
// packed bf16 pair (lo, hi) = (x0 |cos0|, x1 |cos1|) -> with the cosine signs of word w
__device__ __forceinline__ uint32_t sgnsine_flip(uint32_t packed_bf16, uint32_t w) {
  return packed_bf16 ^ ((w << 15) & 0x80008000u);
}
__device__ __forceinline__ float sgnsine_sign(float c_abs, uint32_t w, int hi) {       // scalar form
  return __uint_as_float(__float_as_uint(c_abs) | ((hi ? (w << 15) : (w << 31)) & 0x80000000u));
}

// ---- k-space data consistency applied where the network output is completed (data_consistency.py:7-20, 32-47) ----
//   y <- (1 - m pull) y + m pull k0:  pull = 1 is the noiseless (1 - m) y + m k0, pull = v / (1 + v) the noisy form;
//   the adjoint reaching y is scaled by keep = 1 - m pull.
struct DcSpec {
  const float* k0;     // sampled k-space values, or null: no data consistency
  const float* mask;   // sampling mask (1 where sampled)
  float pull;
  int cf;              // 1: k0 / mask are [tasks][o][n] (channel first: the datasets' [B, 2, nx, ny]); 0: [tasks][n][o]
};
__device__ __forceinline__ size_t dc_index(int cf, int task, int row, int c, int n, int o) {
  return cf ? (size_t(task) * o + c) * size_t(n) + row : (size_t(task) * n + row) * size_t(o) + c;
}

// ---- Gaussian Fourier features built on chip (features.py:31-41: x @ B, times 2 pi, sin | cos) ----
//   feat[i] = sin(2 pi u_i),  feat[F + i] = cos(2 pi u_i),  u_i = sum_r x_r B[r][i]          (B: [raw][F], fp32)
// |u| reaches ~100 turns (B ~ N(0, scale^2), scale = 21 in the MRI scripts), where fp32 u alone carries ~2e-5 rad of
// argument error -- the reference's own rounding noise on this op.  Here the FRACTION of u is formed exactly: every
// product p = x_r B_ri is split into whole turns rint(p) (dropped), p - rint(p) (exact) and its fma error term.
struct FourierSpec {
  const float* B;      // [raw][F] device pointer, or null: the coordinates are used as they are
  int F, raw;
};
__device__ __forceinline__ float fourier_frac(const float (&x)[3], int raw, const float* __restrict__ B, int F, int fi) {
  float f = 0.f;
#pragma unroll
  for (int r = 0; r < 3; ++r)
    if (r < raw) {
      const float b = __ldg(B + r * F + fi);
      const float p = x[r] * b;
      const float e = fmaf(x[r], b, -p);
      f += (p - rintf(p)) + e;
    }
  return f - rintf(f);      // in [-0.5, 0.5] turns
}
template <bool ACCURATE>
__device__ __forceinline__ float fourier_value(float f, bool is_cos) {
  if constexpr (ACCURATE) return is_cos ? cospif(2.f * f) : sinpif(2.f * f);
  const float a = 6.283185307179586f * f;      // reduced argument: the SFU's ~5e-7 absolute error
  return is_cos ? __cosf(a) : __sinf(a);
}

// sin/cos of w0*z.
//   accurate=true : CUDA libm sincosf (<= 2 ulp, full range reduction) -- fp32-parity mode.
//   accurate=false: exact fp32 reduction to one revolution, then the SFU on the reduced
//                   argument (abs err ~5e-7, far below the bf16 operand rounding of that mode).
//                   The caller passes t = z * (w0 / 2pi) in revolutions.
__device__ __forceinline__ void sincos_rev(float t, float* s, float* c) {
  const float magic = 12582912.0f;            // 1.5 * 2^23: round-to-nearest-integer by add/sub
  float k = (t + magic) - magic;
  float f = t - k;                            // exact, f in [-0.5, 0.5]
  float r = f * 6.283185307179586f;
  *s = __sinf(r);
  *c = __cosf(r);
}

// sine only (inference: nothing reads the cosine)
__device__ __forceinline__ float sin_rev(float t) {
  const float magic = 12582912.0f;
  const float k = (t + magic) - magic;
  return __sinf((t - k) * 6.283185307179586f);
}

template <bool ACCURATE>
__device__ __forceinline__ void sincos_w0(float z, float w0, float w0_rev, float* s, float* c) {
  if constexpr (ACCURATE) {
    sincosf(w0 * z, s, c);
  } else {
    sincos_rev(z * w0_rev, s, c);
  }
}

// ---- chunk stores / loads used by the epilogues (per thread: CW consecutive columns of one row)
template <int CW>
__device__ __forceinline__ void store_bf16_chunk(bf16* dst, const float* v) {
  uint4* d4 = reinterpret_cast<uint4*>(dst);
#pragma unroll
  for (int i = 0; i < CW / 8; ++i) {
    uint4 u;
    u.x = pack_bf16(v[8 * i + 0], v[8 * i + 1]);
    u.y = pack_bf16(v[8 * i + 2], v[8 * i + 3]);
    u.z = pack_bf16(v[8 * i + 4], v[8 * i + 5]);
    u.w = pack_bf16(v[8 * i + 6], v[8 * i + 7]);
    d4[i] = u;
  }
}
// value = hi + lo with hi = bf16(v), lo = bf16(v - hi)
template <int CW, bool SPLIT>
__device__ __forceinline__ void store_operand_chunk(bf16* hi, bf16* lo, size_t off, const float* v) {
  store_bf16_chunk<CW>(hi + off, v);
  if constexpr (SPLIT) {
    float r[CW];
#pragma unroll
    for (int i = 0; i < CW; ++i) r[i] = v[i] - bf16_round_f(v[i]);
    store_bf16_chunk<CW>(lo + off, r);
  }
}
template <int CW>
__device__ __forceinline__ void load_bf16_chunk(const bf16* src, float* v) {
  const uint4* s4 = reinterpret_cast<const uint4*>(src);
#pragma unroll
  for (int i = 0; i < CW / 8; ++i) {
    uint4 u = __ldg(s4 + i);
    v[8 * i + 0] = bf16_lo_f(u.x); v[8 * i + 1] = bf16_hi_f(u.x);
    v[8 * i + 2] = bf16_lo_f(u.y); v[8 * i + 3] = bf16_hi_f(u.y);
    v[8 * i + 4] = bf16_lo_f(u.z); v[8 * i + 5] = bf16_hi_f(u.z);
    v[8 * i + 6] = bf16_lo_f(u.w); v[8 * i + 7] = bf16_hi_f(u.w);
  }
}
template <int CW, bool SPLIT>
__device__ __forceinline__ void load_operand_chunk(const bf16* hi, const bf16* lo, size_t off, float* v) {
  load_bf16_chunk<CW>(hi + off, v);
  if constexpr (SPLIT) {
    float r[CW];
    load_bf16_chunk<CW>(lo + off, r);
#pragma unroll
    for (int i = 0; i < CW; ++i) v[i] += r[i];
  }
}
// stash planes: fp32 in split mode, bf16 otherwise
template <int CW, bool F32>
__device__ __forceinline__ void store_stash_chunk(void* base, size_t off, const float* v) {
  if constexpr (F32) {
    float4* d = reinterpret_cast<float4*>(reinterpret_cast<float*>(base) + off);
#pragma unroll
    for (int i = 0; i < CW / 4; ++i) d[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
  } else {
    store_bf16_chunk<CW>(reinterpret_cast<bf16*>(base) + off, v);
  }
}
template <int CW, bool F32>
__device__ __forceinline__ void load_stash_chunk(const void* base, size_t off, float* v) {
  if constexpr (F32) {
    const float4* s = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(base) + off);
#pragma unroll
    for (int i = 0; i < CW / 4; ++i) {
      float4 f = __ldg(s + i);
      v[4 * i] = f.x; v[4 * i + 1] = f.y; v[4 * i + 2] = f.z; v[4 * i + 3] = f.w;
    }
  } else {
    load_bf16_chunk<CW>(reinterpret_cast<const bf16*>(base) + off, v);
  }
}

// ---- parameter block of the row-GEMM kernels (forward hidden layer / backward dgrad) ----
struct alignas(64) RowsGemmParams {
  CUtensorMap tmA_hi, tmA_lo;   // A operand planes, 2D [S*R, H], box 64 x 128
  CUtensorMap tmB_hi, tmB_lo;   // weights [tasks*H, H] (K contiguous), box 64 x BN
  // epilogue stores (box CW columns x 32 rows, one per epilogue warp and chunk):
  CUtensorMap tmO_hi, tmO_lo;   // forward: act planes of this layer; backward: adjoint planes of the layer below
  CUtensorMap tmC, tmJ;         // forward: cosine stash [R, H] and jet stash [(S-1)*R, H] (bf16, or fp32 in split mode)
  // backward epilogue loads from the layer below (box CW columns x 32 rows):
  CUtensorMap tmCin, tmJin;     // its cosine and jet stash
  CUtensorMap tmSin_hi, tmSin_lo;   // its sine (act plane 0)
  int R;                        // rows per plane
  int rows_per_task;            // n_pad
  int per_task;                 // weights (and bias) carry a leading task axis
  float w0;
  const float* bias;            // forward: [tasks?][H]
  const float* w_first;         // backward: layer-0 weights [tasks?][H][d] (Jz_k = W0[:, k]) when the layer below is layer 0
  int below_is_first;
  // debug
  float* raw_out;               // [R][H] fp32 raw accumulator of stream 0
};

// ---- parameter block of the weight-gradient kernel ----
// Whole-MLP fused forward (mlp_fused_fwd.cu): bf16 mode, value stream, d_in <= 4.
constexpr int MAX_FUSED_HIDDEN = 8;
constexpr int MAX_FUSED_HIDDEN_SMEM = 8;   // the fused kernel keeps the biases of at most this many hidden layers on chip
struct alignas(64) MlpFwdParams {
  CUtensorMap tmW[MAX_FUSED_HIDDEN];        // K-major fp16 weights of hidden layer l+1 as [tasks?*H, H], box 64 x 128
  CUtensorMap tmW0;                         // l0_mma: first layer as a split-bf16 operand [tasks?*H, 64] (simt.cu prep_first_kernel)
  CUtensorMap tmAct[MAX_FUSED_HIDDEN + 1];  // stash planes: the signed sine (fp16) of layer l as [R, H], box 64 x 32 (a warp's slice)
  const float* bias[MAX_FUSED_HIDDEN];      // fp32 bias of hidden layer l+1 [tasks?][H]
  const float *x, *W0, *b0;                 // coordinates [tasks][n][d], first layer [tasks?][H][d], [tasks?][H]
  FourierSpec ff;                           // ff.B != null (l0_mma only): x holds RAW coordinates [tasks][n][ff.raw] and
                                            // the d = 2 ff.F inputs of the first layer are their Fourier features
  const float *WL, *bL;                     // outermost linear [tasks?][o][H], [tasks?][o]   (fuse_last)
  float* y;                                 // [tasks][n][o]                                    (fuse_last)
  // fuse_last && gt != null: the loss is image_mse (loss_functions.py:66-96) and the thread that completes a row's
  // y also writes its gradient gy = 2 w (y - gt) and sums w (y - gt)^2 into *loss_acc (one atomic per CTA)
  const float* gt;                          // [tasks][n][o]
  float* gy;                                // [tasks][n][o]
  float loss_weight;
  float* loss_acc;
  DcSpec dc;                                // fuse_last && dc.k0 != null: y leaves the kernel data-consistent (and gt / gy /
                                            // the loss refer to that y: gy = 2 w (y_dc - gt) keep)
  int n_hidden, rows_per_task, per_task, tasks, n, d, o, fuse_last;
  int nkc0;                                 // l0_mma: 64-wide K chunks of the first layer (ceil(d / 64); 1 for d <= 16)
  CUtensorMap tmFeat;                       // d > 16, stash: the first layer's INPUT tile (bf16) as [R, H], box 64 x 32 -- the
                                            // weight-gradient kernel's operand for dW_0 (the features are not rebuilt there)
  int l0_mma;                               // d > 4: the first layer runs on the tensor core as well
                                            // (d <= 4: layer 0 leaves NO phase plane; the backward kernels recompute
                                            //  w0 (x W0^T + b0) from the coordinates, bit for bit the same fp32 value)
  float w0;
  long long* dbg;                           // optional clock64 trace of CTA 0 (SIREN_FUSED_DBG)
};

// Fused input-gradient chain (mlp_fused_bwd.cu): adjoint of the top sine layer in, adjoints of the sine
// layers below out (weight-gradient operands), bias gradients and the first layer's weight gradient.
struct alignas(64) MlpBwdParams {
  CUtensorMap tmWt[MAX_FUSED_HIDDEN];       // transposed bf16 weights of hidden layer l+1 as [tasks?*H, H], box 64 x 128
  CUtensorMap tmTop;                        // adjoint plane of the top sine layer [R, H], box 64 x 128 (load)
  CUtensorMap tmC[MAX_FUSED_HIDDEN];        // stash plane (signed sine, fp16) of sine layer l, l < n_hidden, box 64 x 128 (load)
  CUtensorMap tmAdj[MAX_FUSED_HIDDEN + 1];  // adjoint plane of sine layer l, box 64 x 128 (store)
  float* db[MAX_FUSED_HIDDEN + 1];          // bias gradient of sine layer l: [tasks?][H]
  float* dW0;                               // [tasks?][H][d]
  const float* x;                           // coordinates [tasks][n][d]
  const float *W0, *b0;                     // first layer [tasks?][H][d], [tasks?][H]   (l0_from_x)
  int n_hidden, rows_per_task, per_task, tasks, n, d;
  int store_adj0;                           // the caller still needs the layer-0 adjoint (coordinate gradients)
  float w0;
  // db_l for l >= 1 always comes from the weight-gradient kernel (column sums of the adjoint blocks it stages):
  // only db_0 is formed here.  The transposed weights arrive PRE-SCALED by w0 (prep_weights, scale_t), so a hidden
  // step is acc * cos(theta) and nothing else.
  int skip_bottom_sums;                     // d > 4: db_0 and dW_0 come from first_bwd (the layer-0 adjoint is stored for it)
  int l0_from_x;                            // d <= 4: there is no phase plane of layer 0; the bottom step recomputes
                                            // cos(w0 (x W0^T + b0)) from the coordinates in its column pass
  long long* dbg;                           // optional clock64 trace of CTA 0 (SIREN_FUSED_DBG)
  // fuse_top: the chain starts at the loss gradient instead of at the top adjoint plane (no last_bwd launch):
  //   zbar_L = (gy WL) * w0 cos(phase_L),  db_L = colsum,  dWL = gy^T sin(phase_L),  dbL = sum gy
  // tmTop then maps the top layer's PHASE plane, tmAdj[n_hidden] / db[n_hidden] take zbar_L and its column sums
  int fuse_top, o;
  const uint32_t* phase_top;                // fuse_top: the top layer's stash plane [R][128] as fp16 pairs (signed sine) -- the
                                            // top step reads it straight from global memory (column layout: a warp's row
                                            // is one 128-byte line), tmTop only serves the L2 prefetch
  const float* gy;                          // [tasks][n][o]
  DcSpec dc;                                // fuse_top && dc.mask != null: gy is the adjoint of the data-consistent output;
                                            // the step scales it by keep = 1 - mask pull as it picks it up
  const float* WL;                          // [tasks?][o][H]
  float* dWL;                               // [tasks?][o][H]
  float* dbL;                               // [tasks?][o]
};

// The whole bf16 training step in one kernel (mlp_fused_step.cu): the forward's and the chain's parameter blocks side by
// side (image_mse, d_in <= 4, d_out <= 2, fuse_last / fuse_top, l0_from_x, no coordinate gradient).  The top stash
// plane (f.tmAct[n_hidden], b.tmTop, b.phase_top) is not used; f.gy may be null.
constexpr int MAX_FUSED_STEP_HIDDEN = 4;   // its biases of at most this many hidden layers fit next to the chain's sums
struct alignas(64) MlpStepParams {
  MlpFwdParams f;
  MlpBwdParams b;
};

constexpr int MAX_WG_LAYERS = 4;      // hidden layers per weight-gradient launch (kernel-parameter budget)
struct alignas(64) WgradParams {
  CUtensorMap tmA_hi[MAX_WG_LAYERS], tmA_lo[MAX_WG_LAYERS];   // adjoint planes of hidden layer l as [S*R, H], box 64 x KC
  CUtensorMap tmB_hi[MAX_WG_LAYERS], tmB_lo[MAX_WG_LAYERS];   // act planes of layer l-1
  float* dW[MAX_WG_LAYERS];           // [tasks?][H][H] fp32, accumulated with red.add
  float* db[MAX_WG_LAYERS];           // phase_b only, optional: bias gradient [tasks?][H] = column sums of the adjoint
  int n_layers;                       // hidden (H x H) layers
  int S;                              // streams
  int R;
  int rows_per_task;
  int per_task;
  int tasks;
  int slices;                         // split-K slices per (layer, task-group)
  int slices0;                        // ... of item kind 0 when it is the slower kind (l0_from_x: its operand is built
                                      // on chip, one MUFU per element); 0 = the same as the others
  int db_plain;                       // per-layer paths (!phase_b): db[] given, the flush warps take the column sums of the
                                      // staged adjoint blocks of the value stream (hi + lo in split mode)
  int phase_b;                        // the B planes are the fused forward's stash: the layer input's signed sine in
                                      // fp16; the kernel turns each staged block into bf16 in shared memory
  // l0_from_x (phase_b, d <= 4): layer index 0 of this launch is the first hidden layer and its B operand
  // sin(w0 (x W0^T + b0)) has no plane at all: the flush warps build each block from the coordinates
  int l0_from_x, d, n;
  float w0;
  const float *x, *W0, *b0;           // [tasks][n][d], [tasks?][H][d], [tasks?][H]
  // first_wide (phase_b, 4 < d <= 16): one more item kind, index n_layers -- the FIRST layer's own gradients
  //   dW_0 = zbar_0^T x (N = 2 d columns: the inputs as bf16 hi | lo terms, built on chip; with ff.B from the raw
  //   coordinates as Fourier features),  db_0 = column sums of zbar_0
  long long* dbg;                     // optional (SIREN_WGRAD_DBG): per CTA {layer of its first item, start ns, end ns}
  int first_wide;
  CUtensorMap tmA0;                   // layer-0 adjoint plane [R, H], box 64 x KC
  CUtensorMap tmB0;                   // d > 16: the first layer's input plane (bf16, written by the fused forward)
  int nkc0;                           // d > 16: 64-wide feature blocks of that plane in use (N = 64 nkc0)
  float *dW0, *db0;                   // [tasks?][H][d], [tasks?][H]
  FourierSpec ff;
};

}  // namespace siren
