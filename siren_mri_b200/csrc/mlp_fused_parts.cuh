// Pieces shared by the whole-MLP kernels on CTA pairs (mlp_fused_pair.cu forward, mlp_fused_bwd.cu input-gradient
// chain, mlp_fused_step.cu both in one): the common tile geometry, the forward's sine piece and narrow first layer,
// and the chain's bottom pass.  Each kernel file includes it inside its own anonymous namespace.
#pragma once
#include "common.cuh"
#include "ptx.cuh"

namespace siren {
namespace {

constexpr int NSUB = 4;                         // epilogue warps per TMEM lane quadrant (= K chunks of a tile)
constexpr int kThreads = 128 + NSUB * 128;      // 4 control warps + 16 epilogue warps
constexpr int EPI_WARPS = 4 * NSUB;
constexpr int PW = 16;                          // columns per piece
constexpr int NPIECE = 64 / PW;
constexpr int A_CHUNK = TILE_M * 128;           // 16 KB: [128 rows][128 B], one K chunk of an A tile
constexpr int A_TILE = 4 * A_CHUNK;             // 64 KB: [4 k-chunks][128 rows][128 B]
constexpr int B_SLOT = 128 * 128;               // 16 KB: this CTA's [128 out rows][64 k] of one K chunk
constexpr int NKC = 4;                          // K chunks per layer = weight slots

struct EpiOut {
  uint32_t a_row;      // shared address of this thread's 128-byte row inside its A slice (tile 0)
  int row7;            // swizzle term of this thread's row
  int lane;
};

// sine of 16 arguments -> A slice (fp16, in place).  STASH: the low mantissa bit of every element takes the sign of
// the cosine (common.cuh, "signed sine"): the slice is the next layer's operand AND the stash plane.
template <bool STASH>
__device__ __forceinline__ void piece_out(const EpiOut& eo, int tl, int pc, const float* t, float* s, bool write_a) {
#pragma unroll
  for (int j = 0; j < PW; ++j) s[j] = __sinf(t[j]);
  if (write_a) {
    uint32_t w[PW / 2];
#pragma unroll
    for (int j = 0; j < PW / 2; ++j)
      w[j] = STASH ? pack_sgnsine(s[2 * j], s[2 * j + 1], sgn_kf(t[2 * j]), sgn_kf(t[2 * j + 1]))
                   : pack_f16(s[2 * j], s[2 * j + 1]);
    const uint32_t arow = eo.a_row + uint32_t(tl) * A_TILE;
#pragma unroll
    for (int h = 0; h < 2; ++h)
      ptx::st_shared_v4(arow + (uint32_t((2 * pc + h) ^ eo.row7) << 4), w[4 * h], w[4 * h + 1], w[4 * h + 2], w[4 * h + 3]);
  }
}

// Narrow first layer (D = d_in <= 4) of one tile, 32 rows x 64 columns per warp.  Lane j keeps the weights of
// columns 2j, 2j + 1 of the warp's slice in registers and walks the rows, whose coordinates sit in lane r (one
// shuffle per coordinate and row): a row leaves the warp as ONE conflict-free 128-byte store into the A slice.
// (With a thread per row, every element needs its column's weights from shared memory: a broadcast LDS.128 per
// element, 4 LSU cycles each -- the layer cost 7.0k cycles per tile against 4.2k for a hidden layer.)
// The tile is fp16 like every hidden operand.  Nothing is stashed, training or not: theta_0 = fma(x_{D-1}, w_{D-1}, ... fma(x_0, w_0, b)) on w0-scaled fp32
// weights is two to four FMAs per element, and the backward kernels repeat exactly this chain instead of
// reading a 512 B / coordinate phase plane (three plane transfers less per step).
template <int D>
__device__ __forceinline__ void first_rows(const EpiOut& eo, uint32_t a_slice, const float* cx, const float4 wa,
                                           const float4 wb, float ba, float bb) {
  const int lane = eo.lane;
  const uint32_t col4 = uint32_t(lane & 3) << 2, ch = uint32_t(lane >> 2);
#pragma unroll 1
  for (int rb = 0; rb < 4; ++rb) {
    uint32_t hs[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = rb * 8 + i;
      const float x0 = __shfl_sync(0xffffffffu, cx[0], r);
      float za = fmaf(x0, wa.x, ba), zb = fmaf(x0, wb.x, bb);
      if (D > 1) {
        const float x1 = __shfl_sync(0xffffffffu, cx[1], r);
        za = fmaf(x1, wa.y, za); zb = fmaf(x1, wb.y, zb);
      }
      if (D > 2) {
        const float x2 = __shfl_sync(0xffffffffu, cx[2], r);
        za = fmaf(x2, wa.z, za); zb = fmaf(x2, wb.z, zb);
      }
      if (D > 3) {
        const float x3 = __shfl_sync(0xffffffffu, cx[3], r);
        za = fmaf(x3, wa.w, za); zb = fmaf(x3, wb.w, zb);
      }
      hs[i] = pack_f16(__sinf(za), __sinf(zb));
    }
#pragma unroll
    for (int i = 0; i < 8; ++i)                     // row & 7 == i: the slice and the row blocks start at multiples of 8
      ptx::st_shared_u32(a_slice + uint32_t(rb) * 1024u + uint32_t(i) * 128u + ((ch ^ uint32_t(i)) << 4) + col4, hs[i]);
  }
}

// Bottom layer of a narrow input (d <= 4).  The warp's [32 rows x 64 columns] slice holds
// hbar_0 = zbar_1 (w0 W_1) in bf16 (128-byte rows, 128-byte swizzle), just written by this warp in row layout.
// This pass walks it in COLUMN layout -- the lane owns columns 2 lane, 2 lane + 1 -- and forms, per row,
//   zbar_0 = hbar_0 * cos(theta_0),  theta_0 = w0 (x W0^T + b0)
// with theta_0 recomputed from the row's coordinates by the SAME fp32 FMA chain as the forward's first layer
// (mlp_fused_pair.cu, first_rows): layer 0 leaves no phase plane.  db_0 = sum_r zbar_0, dW_0[:, k] = sum_r zbar_0 x_k.
// A row's coordinates sit in the registers of lane r (one shuffle per row and coordinate).  wa / wb = w0 W0 rows
// of the lane's two columns, ba / bb = w0 b0.  STORE: zbar_0 goes back into the slice for the loader's TMA store.
// acc2 -> this lane's float2 in row 0 of the warp's partial sums.
template <int D, bool STORE>
__device__ __forceinline__ void bottom_pass(uint32_t slice, int lane, float x0, float x1, float x2, float x3,
                                            const float4 wa, const float4 wb, float ba, float bb, float2* acc2,
                                            int row_dw0) {
  float sb0 = 0.f, sb1 = 0.f, sw0[D], sw1[D];
#pragma unroll
  for (int k = 0; k < D; ++k) sw0[k] = sw1[k] = 0.f;
  const uint32_t lane_off = uint32_t(lane & 3) * 4u;
  const uint32_t unit = uint32_t(lane >> 2);
#pragma unroll 1
  for (int rb = 0; rb < 32; rb += 8) {
    uint32_t u[8];
    float xr[D][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)      // row & 7 == i: the slice and the row blocks start at multiples of 8
      u[i] = ptx::ld_shared_u32(slice + uint32_t(rb + i) * 128u + ((unit ^ uint32_t(i)) << 4) + lane_off);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      xr[0][i] = __shfl_sync(0xffffffffu, x0, rb + i);
      if constexpr (D > 1) xr[1][i] = __shfl_sync(0xffffffffu, x1, rb + i);
      if constexpr (D > 2) xr[2][i] = __shfl_sync(0xffffffffu, x2, rb + i);
      if constexpr (D > 3) xr[3][i] = __shfl_sync(0xffffffffu, x3, rb + i);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float ta = fmaf(xr[0][i], wa.x, ba), tb = fmaf(xr[0][i], wb.x, bb);
      if constexpr (D > 1) { ta = fmaf(xr[1][i], wa.y, ta); tb = fmaf(xr[1][i], wb.y, tb); }
      if constexpr (D > 2) { ta = fmaf(xr[2][i], wa.z, ta); tb = fmaf(xr[2][i], wb.z, tb); }
      if constexpr (D > 3) { ta = fmaf(xr[3][i], wa.w, ta); tb = fmaf(xr[3][i], wb.w, tb); }
      const float z0 = bf16_lo_f(u[i]) * __cosf(ta), z1 = bf16_hi_f(u[i]) * __cosf(tb);
      sb0 += z0;
      sb1 += z1;
#pragma unroll
      for (int k = 0; k < D; ++k) {
        sw0[k] = fmaf(z0, xr[k][i], sw0[k]);
        sw1[k] = fmaf(z1, xr[k][i], sw1[k]);
      }
      if constexpr (STORE)
        ptx::st_shared_u32(slice + uint32_t(rb + i) * 128u + ((unit ^ uint32_t(i)) << 4) + lane_off, pack_bf16(z0, z1));
    }
  }
  float2 t = acc2[0];
  t.x += sb0; t.y += sb1;
  acc2[0] = t;
#pragma unroll
  for (int k = 0; k < D; ++k) {
    float2 w = acc2[(row_dw0 + k) * 32];
    w.x += sw0[k]; w.y += sw1[k];
    acc2[(row_dw0 + k) * 32] = w;
  }
}

}  // namespace
}  // namespace siren
