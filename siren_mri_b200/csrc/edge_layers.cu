// CUDA-core kernels for the skinny ends of the MLP and the bias gradients.
//   first layer (K = d_in <= 16) forward / backward      modules.py:25-26,38 with in_features = d
//   last layer  (N = d_out <= 8) forward / backward      modules.py:25-26 (outermost linear)
//   column sums of an adjoint plane (db_0 of a wide first layer in fp32-parity mode)
// These are HBM-streaming kernels: one warp per coordinate row, each lane owning 8 consecutive
// feature columns (16-byte bf16 vectors), weights of the current task staged in shared memory,
// per-thread partial sums reduced once per block.  grid = (blocks per task, tasks) so a block
// never straddles two tasks.
#include <cstdlib>

#include "common.cuh"
#include "ptx.cuh"
#include "simt.h"

namespace siren {

namespace {

constexpr int MAXD = 16;
constexpr int kWarps = 8;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// sum the per-thread column partials of all 8 warps and add them into dst[col * stride]
__device__ __forceinline__ void block_cols_atomic(const float (&v)[8], float* red /*[8][256]*/, float* dst,
                                                  int stride) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
#pragma unroll
  for (int j = 0; j < 8; ++j) red[warp * H + lane * 8 + j] = v[j];
  __syncthreads();
  float s = 0.f;
#pragma unroll
  for (int w = 0; w < kWarps; ++w) s += red[w * H + threadIdx.x];
  if (s != 0.f) atomicAdd(dst + size_t(threadIdx.x) * stride, s);
}

struct RowRange {
  int n0, n1;
};
__device__ __forceinline__ RowRange block_rows(int n_pad) {
  const int per = (n_pad + gridDim.x - 1) / gridDim.x;
  int n0 = blockIdx.x * per;
  int n1 = n0 + per;
  if (n1 > n_pad) n1 = n_pad;
  return {n0, n1};
}

// -------------------------------------------------------------------------------------------
// first layer forward
// -------------------------------------------------------------------------------------------
template <bool SPLIT>
__global__ void __launch_bounds__(256) first_fwd_kernel(FirstParams p) {
  __shared__ __align__(16) float sWt[MAXD * H];   // [i][col]
  __shared__ __align__(16) float sB[H];
  const int task = blockIdx.y;
  const int wt = p.per_task ? task : 0;
  const int d = p.d;
  for (int idx = threadIdx.x; idx < H * d; idx += blockDim.x) {
    const int col = idx / d, i = idx - col * d;
    sWt[i * H + col] = p.W[size_t(wt) * H * d + idx];
  }
  sB[threadIdx.x] = p.b[size_t(wt) * H + threadIdx.x];
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int col0 = lane * 8;
  const size_t plane = size_t(p.R) * H;
  const float w0 = p.w0, w0_rev = p.w0 * 0.15915494309189535f;
  const RowRange rr = block_rows(p.n_pad);
  float b[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) b[j] = sB[col0 + j];

  for (int n = rr.n0 + warp; n < rr.n1; n += kWarps) {
    float z[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) z[j] = b[j];
    if (n < p.n) {
      const float* x = p.x + (size_t(task) * p.n + n) * d;
      for (int i = 0; i < d; ++i) {
        const float xi = __ldg(x + i);
        const float4 wa = *reinterpret_cast<const float4*>(&sWt[i * H + col0]);
        const float4 wb = *reinterpret_cast<const float4*>(&sWt[i * H + col0 + 4]);
        z[0] = fmaf(xi, wa.x, z[0]); z[1] = fmaf(xi, wa.y, z[1]); z[2] = fmaf(xi, wa.z, z[2]); z[3] = fmaf(xi, wa.w, z[3]);
        z[4] = fmaf(xi, wb.x, z[4]); z[5] = fmaf(xi, wb.y, z[5]); z[6] = fmaf(xi, wb.z, z[6]); z[7] = fmaf(xi, wb.w, z[7]);
      }
    }
    float s[8], c[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) sincos_w0<SPLIT>(z[j], w0, w0_rev, &s[j], &c[j]);
    const size_t off = (size_t(task) * p.n_pad + n) * H + col0;
    store_operand_chunk<8, SPLIT>(p.act_hi, p.act_lo, off, s);
    if (p.c) store_stash_chunk<8, SPLIT>(p.c, off, c);
    if (p.order >= 1) {
      for (int k = 0; k < d; ++k) {
        float o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = w0 * c[j] * sWt[k * H + col0 + j];
        store_operand_chunk<8, SPLIT>(p.act_hi, p.act_lo, size_t(1 + k) * plane + off, o);
        if (p.order == 2) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float w = sWt[k * H + col0 + j];
            o[j] = -(w0 * w0) * s[j] * w * w;
          }
          store_operand_chunk<8, SPLIT>(p.act_hi, p.act_lo, size_t(1 + d + k) * plane + off, o);
        }
      }
    }
  }
}

// -------------------------------------------------------------------------------------------
// last layer forward: out[s][n, o] = plane_s[n, :] . W_L[o, :]
// -------------------------------------------------------------------------------------------
template <bool SPLIT>
__global__ void __launch_bounds__(256) last_fwd_kernel(LastParams p) {
  __shared__ __align__(16) float sW[8 * H];
  const int task = blockIdx.y;
  const int wt = p.per_task ? task : 0;
  const int o = p.o, d = p.d;
  for (int idx = threadIdx.x; idx < o * H; idx += blockDim.x) sW[idx] = p.W[size_t(wt) * o * H + idx];
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int col0 = lane * 8;
  const size_t plane = size_t(p.R) * H;
  const int S = 1 + p.order * d;
  RowRange rr = block_rows(p.n_pad);
  if (rr.n1 > p.n) rr.n1 = p.n;
  constexpr int UN = 4;   // rows in flight per warp
  for (int nb = rr.n0 + warp * UN; nb < rr.n1; nb += kWarps * UN) {
    // next iteration's rows of every stream into L2 (the stream loop below keeps only UN loads per lane in flight).
    // The fused path (p.phase) skips it, but keep it: without this block ptxas gives the bf16 instantiation 128
    // registers instead of 64, and the fused path's outermost linear for d_out > 2 then takes 79 us instead of 62
    // (262,144 rows, d_out = 3, NVIDIA B200).
    if (!SPLIT && nb + kWarps * UN < rr.n1 && !p.phase)
      for (int s = 0; s < S; ++s)
#pragma unroll
        for (int u = 0; u < UN; ++u) {
          const int n = nb + kWarps * UN + u < rr.n1 ? nb + kWarps * UN + u : rr.n1 - 1;
          const size_t offp = size_t(s) * plane + (size_t(task) * p.n_pad + n) * H + col0;
          ptx::prefetch_l2(p.act_hi + offp);
          if (SPLIT) ptx::prefetch_l2(p.act_lo + offp);
        }
    for (int s = 0; s < S; ++s) {
      float h[UN][8];
#pragma unroll
      for (int u = 0; u < UN; ++u) {
        const int n = nb + u < rr.n1 ? nb + u : rr.n1 - 1;
        if (!SPLIT && p.phase) {      // fused-forward stash: the top layer's signed sine (fp16; the stolen bit is noise)
          const uint4 v = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const __half*>(p.phase) +
                                                               (size_t(task) * p.n_pad + n) * H + col0));
          const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[j]));
            h[u][2 * j] = f.x; h[u][2 * j + 1] = f.y;
          }
        } else
        load_operand_chunk<8, SPLIT>(p.act_hi, p.act_lo,
                                     size_t(s) * plane + (size_t(task) * p.n_pad + n) * H + col0, h[u]);
      }
      for (int oi = 0; oi < o; ++oi) {
        const float4 wa = *reinterpret_cast<const float4*>(&sW[oi * H + col0]);
        const float4 wb = *reinterpret_cast<const float4*>(&sW[oi * H + col0 + 4]);
#pragma unroll
        for (int u = 0; u < UN; ++u) {
          float acc = h[u][0] * wa.x + h[u][1] * wa.y + h[u][2] * wa.z + h[u][3] * wa.w + h[u][4] * wb.x +
                      h[u][5] * wb.y + h[u][6] * wb.z + h[u][7] * wb.w;
          acc = warp_sum(acc);
          const int n = nb + u;
          if (lane == 0 && n < rr.n1) {
            const size_t orow = size_t(task) * p.n + n;
            if (s == 0) p.y[orow * o + oi] = acc + p.b[size_t(wt) * o + oi];
            else if (s <= d) p.J[(orow * o + oi) * d + (s - 1)] = acc;
            else p.Dd[(orow * o + oi) * d + (s - 1 - d)] = acc;
          }
        }
      }
    }
  }
}

// -------------------------------------------------------------------------------------------
// last layer backward: adjoints of the top sine layer from (gy, gJ, gD) -> its sine reverse ->
// adjoint planes; dW_L and db_L.
// -------------------------------------------------------------------------------------------
template <bool SPLIT, int OMAX, bool JETS>
__global__ void __launch_bounds__(256) last_bwd_kernel(LastParams p) {
  __shared__ __align__(16) float sW[OMAX * H];
  __shared__ float red[kWarps * H];
  const int task = blockIdx.y;
  const int wt = p.per_task ? task : 0;
  const int o = p.o, d = p.d, order = p.order;
  for (int idx = threadIdx.x; idx < o * H; idx += blockDim.x) sW[idx] = p.W[size_t(wt) * o * H + idx];
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int col0 = lane * 8;
  const size_t plane = size_t(p.R) * H;
  const float w0 = p.w0;
  const RowRange rr = block_rows(p.n_pad);

  float dw[OMAX][8];
  float dbias[OMAX];
#pragma unroll
  for (int i = 0; i < OMAX; ++i) {
    dbias[i] = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) dw[i][j] = 0.f;
  }

  for (int n = rr.n0 + warp; n < rr.n1; n += kWarps) {
    const size_t off = (size_t(task) * p.n_pad + n) * H + col0;
    float zb[8];
    if (n < p.n) {
      const size_t orow = size_t(task) * p.n + n;
      float s[8], c[8];
      if (!SPLIT && p.phase) {
        // fused-forward stash: one plane, the signed sine (common.cuh): sin as it is, cos = +-sqrt(1 - sin^2)
        const uint4 u = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const __half*>(p.phase) + off));
        const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float c0, c1;
          sgnsine_unpack(w[j], s[2 * j], s[2 * j + 1], c0, c1);
          c[2 * j] = sgnsine_sign(c0, w[j], 0);
          c[2 * j + 1] = sgnsine_sign(c1, w[j], 1);
        }
      } else {
        load_operand_chunk<8, SPLIT>(p.act_hi, p.act_lo, off, s);
        load_stash_chunk<8, SPLIT>(p.c, off, c);
      }
      float ab[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) ab[j] = 0.f;
#pragma unroll
      for (int i = 0; i < OMAX; ++i)
        if (i < o) {
          const float g = __ldg(p.gy + orow * o + i);
          if (lane == 0) dbias[i] += g;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            ab[j] = fmaf(g, sW[i * H + col0 + j], ab[j]);
            dw[i][j] = fmaf(g, s[j], dw[i][j]);
          }
        }
#pragma unroll
      for (int j = 0; j < 8; ++j) zb[j] = w0 * c[j] * ab[j];
      if constexpr (JETS) {
        for (int k = 0; k < d; ++k) {
          float jact[8], dact[8], jb[8], db[8], jz[8], dz[8], jzb[8];
          load_operand_chunk<8, SPLIT>(p.act_hi, p.act_lo, size_t(1 + k) * plane + off, jact);
          if (order == 2) load_operand_chunk<8, SPLIT>(p.act_hi, p.act_lo, size_t(1 + d + k) * plane + off, dact);
#pragma unroll
          for (int j = 0; j < 8; ++j) { jb[j] = 0.f; db[j] = 0.f; }
#pragma unroll
          for (int i = 0; i < OMAX; ++i)
            if (i < o) {
              const float gj = p.gJ ? __ldg(p.gJ + (orow * o + i) * d + k) : 0.f;
              const float gd = (order == 2 && p.gD) ? __ldg(p.gD + (orow * o + i) * d + k) : 0.f;
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const float w = sW[i * H + col0 + j];
                jb[j] = fmaf(gj, w, jb[j]);
                dw[i][j] = fmaf(gj, jact[j], dw[i][j]);
                if (order == 2) {
                  db[j] = fmaf(gd, w, db[j]);
                  dw[i][j] = fmaf(gd, dact[j], dw[i][j]);
                }
              }
            }
          load_stash_chunk<8, SPLIT>(p.jz, size_t(k) * plane + off, jz);
          if (order == 2) load_stash_chunk<8, SPLIT>(p.jz, size_t(d + k) * plane + off, dz);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            zb[j] -= (w0 * w0) * s[j] * jz[j] * jb[j];
            jzb[j] = w0 * c[j] * jb[j];
          }
          if (order == 2) {
            float dzb[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              zb[j] -= (w0 * w0) * s[j] * dz[j] * db[j] + (w0 * w0 * w0) * c[j] * jz[j] * jz[j] * db[j];
              jzb[j] -= 2.f * (w0 * w0) * s[j] * jz[j] * db[j];
              dzb[j] = w0 * c[j] * db[j];
            }
            store_operand_chunk<8, SPLIT>(p.adj_hi, p.adj_lo, size_t(1 + d + k) * plane + off, dzb);
          }
          store_operand_chunk<8, SPLIT>(p.adj_hi, p.adj_lo, size_t(1 + k) * plane + off, jzb);
        }
      }
      store_operand_chunk<8, SPLIT>(p.adj_hi, p.adj_lo, off, zb);
    } else {
      // pad rows carry zero adjoints (they must not reach dW through the weight-gradient GEMM)
#pragma unroll
      for (int j = 0; j < 8; ++j) zb[j] = 0.f;
      const int S = 1 + order * d;
      for (int s = 0; s < S; ++s) store_operand_chunk<8, SPLIT>(p.adj_hi, p.adj_lo, size_t(s) * plane + off, zb);
    }
  }
  // reductions
#pragma unroll
  for (int i = 0; i < OMAX; ++i)
    if (i < o) {
      block_cols_atomic(dw[i], red, p.dW + (size_t(wt) * o + i) * H, 1);
      if (lane == 0 && dbias[i] != 0.f) atomicAdd(p.db + size_t(wt) * o + i, dbias[i]);
    }
}

// -------------------------------------------------------------------------------------------
// last layer backward of the jet paths on bf16 planes, STAGED: the kernel above reads up to ten planes per row with one
// dependent load -> compute -> store chain per warp and two blocks per SM, i.e. too few bytes in flight (0.55 of the
// copy bandwidth at cfg3).  Here the rows arrive by bulk copies (cp.async.bulk, one 4 KB copy per plane and block of
// eight rows, mbarrier transaction counts) into a three-deep ring of shared-memory stages, so 64-80 KB per block are
// in flight whatever the register budget, and a warp reads its row of every plane from shared memory.  Same
// arithmetic, in the same order, as last_bwd_kernel<false, OMAX, true>.
// -------------------------------------------------------------------------------------------
constexpr int ST_ROWS = kWarps;       // rows per stage: one per warp
constexpr int ST_STAGES = 3;
constexpr int ST_ROW_BYTES = H * 2;   // one bf16 row of a plane

__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               :: "r"(ptx::smem_u32(dst)), "l"(src), "r"(bytes), "r"(ptx::smem_u32(bar)) : "memory");
}
// a wait that cannot hang the GPU: a pipeline bug traps instead
__device__ __forceinline__ void mbar_wait_bounded(uint64_t* bar, uint32_t parity) {
  for (uint32_t tries = 0; !ptx::mbar_try_wait(bar, parity); ++tries)
    if (tries > (1u << 26)) __trap();
}
__device__ __forceinline__ void lds_bf16x8(const uint8_t* row, int lane, float* v) {
  uint4 u;
  ptx::ld_shared_v4(ptx::smem_u32(row) + uint32_t(lane) * 16u, u.x, u.y, u.z, u.w);
  v[0] = bf16_lo_f(u.x); v[1] = bf16_hi_f(u.x);
  v[2] = bf16_lo_f(u.y); v[3] = bf16_hi_f(u.y);
  v[4] = bf16_lo_f(u.z); v[5] = bf16_hi_f(u.z);
  v[6] = bf16_lo_f(u.w); v[7] = bf16_hi_f(u.w);
}

template <int OMAX>
__global__ void __launch_bounds__(256) last_bwd_jets_staged_kernel(LastParams p, int n_stages) {
  extern __shared__ __align__(128) uint8_t st_smem[];
  __shared__ __align__(16) float sW[OMAX * H];
  __shared__ float red[kWarps * H];
  __shared__ __align__(8) uint64_t full[ST_STAGES];      // n_stages <= ST_STAGES of them in use
  const int task = blockIdx.y;
  const int wt = p.per_task ? task : 0;
  const int o = p.o, d = p.d, order = p.order;
  const int nj = order * d;                // jet streams: J_k (k < d), then D_k
  const int npl = 2 + 2 * nj;              // planes per row: sine, cosine, act[1 .. nj], jz[0 .. nj - 1]
  const uint32_t stage_bytes = uint32_t(npl) * ST_ROWS * ST_ROW_BYTES;
  for (int idx = threadIdx.x; idx < o * H; idx += blockDim.x) sW[idx] = p.W[size_t(wt) * o * H + idx];
  if (threadIdx.x == 0) {
    for (int i = 0; i < ST_STAGES; ++i) ptx::mbar_init(&full[i], 1);
    ptx::fence_barrier_init();
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int col0 = lane * 8;
  const size_t plane = size_t(p.R) * H;
  const float w0 = p.w0;
  const RowRange rr = block_rows(p.n_pad);
  const int n_iter = (rr.n1 - rr.n0 + ST_ROWS - 1) / ST_ROWS;
  const bf16* cpl = reinterpret_cast<const bf16*>(p.c);
  const bf16* jzpl = reinterpret_cast<const bf16*>(p.jz);

  auto issue = [&](int it) {               // one thread: the copies of iteration `it` into its stage
    const int stage = it % n_stages;
    const int r0 = rr.n0 + it * ST_ROWS;
    const int rows = rr.n1 - r0 < ST_ROWS ? rr.n1 - r0 : ST_ROWS;
    const uint32_t bytes = uint32_t(rows) * ST_ROW_BYTES;
    uint8_t* dst = st_smem + size_t(stage) * stage_bytes;
    const size_t off = (size_t(task) * p.n_pad + r0) * H;
    ptx::mbar_arrive_expect_tx(&full[stage], bytes * uint32_t(npl));
    bulk_g2s(dst, p.act_hi + off, bytes, &full[stage]);
    bulk_g2s(dst + ST_ROWS * ST_ROW_BYTES, cpl + off, bytes, &full[stage]);
    for (int k = 0; k < nj; ++k) {
      bulk_g2s(dst + size_t(2 + k) * ST_ROWS * ST_ROW_BYTES, p.act_hi + size_t(1 + k) * plane + off, bytes, &full[stage]);
      bulk_g2s(dst + size_t(2 + nj + k) * ST_ROWS * ST_ROW_BYTES, jzpl + size_t(k) * plane + off, bytes, &full[stage]);
    }
  };
  if (threadIdx.x == 0)
    for (int it = 0; it < n_stages && it < n_iter; ++it) issue(it);

  float dw[OMAX][8];
  float dbias[OMAX];
#pragma unroll
  for (int i = 0; i < OMAX; ++i) {
    dbias[i] = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) dw[i][j] = 0.f;
  }

  for (int it = 0; it < n_iter; ++it) {
    const int stage = it % n_stages;
    mbar_wait_bounded(&full[stage], uint32_t(it / n_stages) & 1u);
    const int n = rr.n0 + it * ST_ROWS + warp;
    if (n < rr.n1) {
      const size_t off = (size_t(task) * p.n_pad + n) * H + col0;
      const uint8_t* st = st_smem + size_t(stage) * stage_bytes + size_t(warp) * ST_ROW_BYTES;
      float zb[8];
      if (n < p.n) {
        const size_t orow = size_t(task) * p.n + n;
        float s[8], c[8];
        lds_bf16x8(st, lane, s);
        lds_bf16x8(st + ST_ROWS * ST_ROW_BYTES, lane, c);
        float ab[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) ab[j] = 0.f;
#pragma unroll
        for (int i = 0; i < OMAX; ++i)
          if (i < o) {
            const float g = __ldg(p.gy + orow * o + i);
            if (lane == 0) dbias[i] += g;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              ab[j] = fmaf(g, sW[i * H + col0 + j], ab[j]);
              dw[i][j] = fmaf(g, s[j], dw[i][j]);
            }
          }
#pragma unroll
        for (int j = 0; j < 8; ++j) zb[j] = w0 * c[j] * ab[j];
        for (int k = 0; k < d; ++k) {
          float jact[8], dact[8], jb[8], db[8], jz[8], dz[8], jzb[8];
          lds_bf16x8(st + size_t(2 + k) * ST_ROWS * ST_ROW_BYTES, lane, jact);
          lds_bf16x8(st + size_t(2 + nj + k) * ST_ROWS * ST_ROW_BYTES, lane, jz);
          if (order == 2) {
            lds_bf16x8(st + size_t(2 + d + k) * ST_ROWS * ST_ROW_BYTES, lane, dact);
            lds_bf16x8(st + size_t(2 + nj + d + k) * ST_ROWS * ST_ROW_BYTES, lane, dz);
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) { jb[j] = 0.f; db[j] = 0.f; }
#pragma unroll
          for (int i = 0; i < OMAX; ++i)
            if (i < o) {
              const float gj = p.gJ ? __ldg(p.gJ + (orow * o + i) * d + k) : 0.f;
              const float gd = (order == 2 && p.gD) ? __ldg(p.gD + (orow * o + i) * d + k) : 0.f;
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const float w = sW[i * H + col0 + j];
                jb[j] = fmaf(gj, w, jb[j]);
                dw[i][j] = fmaf(gj, jact[j], dw[i][j]);
                if (order == 2) {
                  db[j] = fmaf(gd, w, db[j]);
                  dw[i][j] = fmaf(gd, dact[j], dw[i][j]);
                }
              }
            }
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            zb[j] -= (w0 * w0) * s[j] * jz[j] * jb[j];
            jzb[j] = w0 * c[j] * jb[j];
          }
          if (order == 2) {
            float dzb[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              zb[j] -= (w0 * w0) * s[j] * dz[j] * db[j] + (w0 * w0 * w0) * c[j] * jz[j] * jz[j] * db[j];
              jzb[j] -= 2.f * (w0 * w0) * s[j] * jz[j] * db[j];
              dzb[j] = w0 * c[j] * db[j];
            }
            store_operand_chunk<8, false>(p.adj_hi, p.adj_lo, size_t(1 + d + k) * plane + off, dzb);
          }
          store_operand_chunk<8, false>(p.adj_hi, p.adj_lo, size_t(1 + k) * plane + off, jzb);
        }
        store_operand_chunk<8, false>(p.adj_hi, p.adj_lo, off, zb);
      } else {
        // pad rows carry zero adjoints (they must not reach dW through the weight-gradient GEMM)
#pragma unroll
        for (int j = 0; j < 8; ++j) zb[j] = 0.f;
        for (int sidx = 0; sidx <= nj; ++sidx) store_operand_chunk<8, false>(p.adj_hi, p.adj_lo, size_t(sidx) * plane + off, zb);
      }
    }
    __syncthreads();                       // every warp has read its row of this stage: it may be refilled
    if (threadIdx.x == 0 && it + n_stages < n_iter) {
      ptx::fence_proxy_async();            // the reads above (generic proxy) before the bulk copies' writes (async proxy)
      issue(it + n_stages);
    }
  }
#pragma unroll
  for (int i = 0; i < OMAX; ++i)
    if (i < o) {
      block_cols_atomic(dw[i], red, p.dW + (size_t(wt) * o + i) * H, 1);
      if (lane == 0 && dbias[i] != 0.f) atomicAdd(p.db + size_t(wt) * o + i, dbias[i]);
    }
}

// -------------------------------------------------------------------------------------------
// first layer backward: dW0[col, i] = sum_n zbar0[n, col] x[n, i] (+ sum_n Jzbar_i[n, col]),
// db0[col] = sum_n zbar0[n, col].  Input features are processed in chunks of 4.
// -------------------------------------------------------------------------------------------
template <bool SPLIT, int DCH, bool JETS>
__global__ void __launch_bounds__(256) first_bwd_kernel(FirstParams p) {
  __shared__ float red[kWarps * H];
  const int task = blockIdx.y;
  const int wt = p.per_task ? task : 0;
  const int d = p.d;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int col0 = lane * 8;
  const size_t plane = size_t(p.R) * H;
  RowRange rr = block_rows(p.n_pad);
  if (rr.n1 > p.n) rr.n1 = p.n;
  for (int i0 = 0; i0 < d; i0 += DCH) {
    float dw[DCH][8], db[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      db[j] = 0.f;
#pragma unroll
      for (int i = 0; i < DCH; ++i) dw[i][j] = 0.f;
    }
    for (int n = rr.n0 + warp; n < rr.n1; n += kWarps) {
      const size_t off = (size_t(task) * p.n_pad + n) * H + col0;
      float zb[8];
      load_operand_chunk<8, SPLIT>(p.adj_hi, p.adj_lo, off, zb);
      const float* x = p.x + (size_t(task) * p.n + n) * d + i0;
#pragma unroll
      for (int i = 0; i < DCH; ++i)
        if (i0 + i < d) {
          const float xi = __ldg(x + i);
#pragma unroll
          for (int j = 0; j < 8; ++j) dw[i][j] = fmaf(zb[j], xi, dw[i][j]);
          if constexpr (JETS) {   // d <= 3 here, so this is the only chunk
            float jzb[8];
            load_operand_chunk<8, SPLIT>(p.adj_hi, p.adj_lo, size_t(1 + i0 + i) * plane + off, jzb);
#pragma unroll
            for (int j = 0; j < 8; ++j) dw[i][j] += jzb[j];
          }
        }
      if (i0 == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) db[j] += zb[j];
      }
    }
#pragma unroll
    for (int i = 0; i < DCH; ++i)
      if (i0 + i < d) block_cols_atomic(dw[i], red, p.dW + size_t(wt) * H * d + (i0 + i), d);
    if (i0 == 0) block_cols_atomic(db, red, p.db + size_t(wt) * H, 1);
  }
}

// -------------------------------------------------------------------------------------------
// The other two streaming passes of the jet paths on bf16 planes, staged the same way (sixteen rows per stage: two
// per warp): first_bwd reads 1 + d adjoint planes per row, last_fwd S = 1 + order d activation planes.
// -------------------------------------------------------------------------------------------
constexpr int ST2_ROWS = 2 * kWarps;

template <int D>
__global__ void __launch_bounds__(256) first_bwd_jets_staged_kernel(FirstParams p) {
  extern __shared__ __align__(128) uint8_t st_smem[];
  __shared__ float red[kWarps * H];
  __shared__ __align__(8) uint64_t full[ST_STAGES];
  const int task = blockIdx.y;
  const int wt = p.per_task ? task : 0;
  constexpr int npl = 1 + D;               // zbar_0 and the d first-order jet adjoints
  constexpr uint32_t stage_bytes = npl * ST2_ROWS * ST_ROW_BYTES;
  if (threadIdx.x == 0) {
    for (int i = 0; i < ST_STAGES; ++i) ptx::mbar_init(&full[i], 1);
    ptx::fence_barrier_init();
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t plane = size_t(p.R) * H;
  RowRange rr = block_rows(p.n_pad);
  if (rr.n1 > p.n) rr.n1 = p.n;
  const int n_iter = (rr.n1 - rr.n0 + ST2_ROWS - 1) / ST2_ROWS;
  auto issue = [&](int it) {
    const int stage = it % ST_STAGES;
    const int r0 = rr.n0 + it * ST2_ROWS;
    const int rows = rr.n1 - r0 < ST2_ROWS ? rr.n1 - r0 : ST2_ROWS;
    const uint32_t bytes = uint32_t(rows) * ST_ROW_BYTES;
    uint8_t* dst = st_smem + size_t(stage) * stage_bytes;
    const size_t off = (size_t(task) * p.n_pad + r0) * H;
    ptx::mbar_arrive_expect_tx(&full[stage], bytes * uint32_t(npl));
#pragma unroll
    for (int k = 0; k < npl; ++k)
      bulk_g2s(dst + size_t(k) * ST2_ROWS * ST_ROW_BYTES, p.adj_hi + size_t(k) * plane + off, bytes, &full[stage]);
  };
  if (threadIdx.x == 0)
    for (int it = 0; it < ST_STAGES && it < n_iter; ++it) issue(it);
  float dw[D][8], db[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    db[j] = 0.f;
#pragma unroll
    for (int i = 0; i < D; ++i) dw[i][j] = 0.f;
  }
  for (int it = 0; it < n_iter; ++it) {
    const int stage = it % ST_STAGES;
    mbar_wait_bounded(&full[stage], uint32_t(it / ST_STAGES) & 1u);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int rloc = warp + h * kWarps;
      const int n = rr.n0 + it * ST2_ROWS + rloc;
      if (n < rr.n1) {
        const uint8_t* st = st_smem + size_t(stage) * stage_bytes + size_t(rloc) * ST_ROW_BYTES;
        float zb[8];
        lds_bf16x8(st, lane, zb);
        const float* x = p.x + (size_t(task) * p.n + n) * D;
#pragma unroll
        for (int i = 0; i < D; ++i) {
          const float xi = __ldg(x + i);
          float jzb[8];
          lds_bf16x8(st + size_t(1 + i) * ST2_ROWS * ST_ROW_BYTES, lane, jzb);
#pragma unroll
          for (int j = 0; j < 8; ++j) dw[i][j] = fmaf(zb[j], xi, dw[i][j]) + jzb[j];
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) db[j] += zb[j];
      }
    }
    __syncthreads();
    if (threadIdx.x == 0 && it + ST_STAGES < n_iter) {
      ptx::fence_proxy_async();
      issue(it + ST_STAGES);
    }
  }
#pragma unroll
  for (int i = 0; i < D; ++i) block_cols_atomic(dw[i], red, p.dW + size_t(wt) * H * D + i, D);
  block_cols_atomic(db, red, p.db + size_t(wt) * H, 1);
}

__global__ void __launch_bounds__(256) last_fwd_staged_kernel(LastParams p, int n_stages) {
  extern __shared__ __align__(128) uint8_t st_smem[];
  __shared__ __align__(16) float sW[8 * H];
  __shared__ __align__(8) uint64_t full[ST_STAGES];
  const int task = blockIdx.y;
  const int wt = p.per_task ? task : 0;
  const int o = p.o, d = p.d;
  const int S = 1 + p.order * d;
  const uint32_t stage_bytes = uint32_t(S) * ST2_ROWS * ST_ROW_BYTES;
  for (int idx = threadIdx.x; idx < o * H; idx += blockDim.x) sW[idx] = p.W[size_t(wt) * o * H + idx];
  if (threadIdx.x == 0) {
    for (int i = 0; i < ST_STAGES; ++i) ptx::mbar_init(&full[i], 1);
    ptx::fence_barrier_init();
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int col0 = lane * 8;
  const size_t plane = size_t(p.R) * H;
  RowRange rr = block_rows(p.n_pad);
  if (rr.n1 > p.n) rr.n1 = p.n;
  const int n_iter = (rr.n1 - rr.n0 + ST2_ROWS - 1) / ST2_ROWS;
  auto issue = [&](int it) {
    const int stage = it % n_stages;
    const int r0 = rr.n0 + it * ST2_ROWS;
    const int rows = rr.n1 - r0 < ST2_ROWS ? rr.n1 - r0 : ST2_ROWS;
    const uint32_t bytes = uint32_t(rows) * ST_ROW_BYTES;
    uint8_t* dst = st_smem + size_t(stage) * stage_bytes;
    const size_t off = (size_t(task) * p.n_pad + r0) * H;
    ptx::mbar_arrive_expect_tx(&full[stage], bytes * uint32_t(S));
    for (int k = 0; k < S; ++k)
      bulk_g2s(dst + size_t(k) * ST2_ROWS * ST_ROW_BYTES, p.act_hi + size_t(k) * plane + off, bytes, &full[stage]);
  };
  if (threadIdx.x == 0)
    for (int it = 0; it < n_stages && it < n_iter; ++it) issue(it);
  for (int it = 0; it < n_iter; ++it) {
    const int stage = it % n_stages;
    mbar_wait_bounded(&full[stage], uint32_t(it / n_stages) & 1u);
    for (int sidx = 0; sidx < S; ++sidx) {
      float h[2][8];
#pragma unroll
      for (int u = 0; u < 2; ++u)
        lds_bf16x8(st_smem + size_t(stage) * stage_bytes + (size_t(sidx) * ST2_ROWS + warp + u * kWarps) * ST_ROW_BYTES, lane, h[u]);
      for (int oi = 0; oi < o; ++oi) {
        const float4 wa = *reinterpret_cast<const float4*>(&sW[oi * H + col0]);
        const float4 wb = *reinterpret_cast<const float4*>(&sW[oi * H + col0 + 4]);
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          float acc = h[u][0] * wa.x + h[u][1] * wa.y + h[u][2] * wa.z + h[u][3] * wa.w + h[u][4] * wb.x +
                      h[u][5] * wb.y + h[u][6] * wb.z + h[u][7] * wb.w;
          acc = warp_sum(acc);
          const int n = rr.n0 + it * ST2_ROWS + warp + u * kWarps;
          if (lane == 0 && n < rr.n1) {
            const size_t orow = size_t(task) * p.n + n;
            if (sidx == 0) p.y[orow * o + oi] = acc + p.b[size_t(wt) * o + oi];
            else if (sidx <= d) p.J[(orow * o + oi) * d + (sidx - 1)] = acc;
            else p.Dd[(orow * o + oi) * d + (sidx - 1 - d)] = acc;
          }
        }
      }
    }
    __syncthreads();
    if (threadIdx.x == 0 && it + n_stages < n_iter) {
      ptx::fence_proxy_async();
      issue(it + n_stages);
    }
  }
}

// -------------------------------------------------------------------------------------------
// first layer, wide input (5 <= d <= 16, e.g. the 16 Fourier features of the MRI configs):
// each thread keeps the weights of TWO feature columns in registers (2 x 16 floats) and walks the
// rows; the coordinate row is a warp-uniform (broadcast) load.  128 threads cover one row, a block
// handles two rows at a time.  (The narrow kernel above would re-read W from shared memory for
// every FMA and is shared-memory-bandwidth bound at d = 16.)
// -------------------------------------------------------------------------------------------
constexpr int WCH = 32;   // rows per block-cooperative chunk in the wide first-layer kernels

// stage rows [n0, n0 + WCH) of the task's coordinates in shared memory as [WCH][MAXD] (zero padded)
__device__ __forceinline__ void stage_x_chunk(const FirstParams& p, int task, int n0, float* sx) {
  for (int idx = threadIdx.x; idx < WCH * MAXD; idx += blockDim.x) {
    const int r = idx / MAXD, i = idx - r * MAXD;
    const int n = n0 + r;
    float v = 0.f;
    if (i < p.d && n < p.n) {
      if (p.ff.B) {      // Fourier-feature prologue: the row's raw coordinates -> feature i (features.py:31-41)
        const float* xr = p.x + (size_t(task) * p.n + n) * p.ff.raw;
        float x[3] = {__ldg(xr), p.ff.raw > 1 ? __ldg(xr + 1) : 0.f, p.ff.raw > 2 ? __ldg(xr + 2) : 0.f};
        const bool is_cos = i >= p.ff.F;
        v = fourier_value<true>(fourier_frac(x, p.ff.raw, p.ff.B, p.ff.F, is_cos ? i - p.ff.F : i), is_cos);
      } else {
        v = __ldg(p.x + (size_t(task) * p.n + n) * p.d + i);
      }
    }
    sx[idx] = v;
  }
}

template <bool SPLIT>
__global__ void __launch_bounds__(256) first_fwd_wide_kernel(FirstParams p) {
  __shared__ __align__(16) float sx[WCH * MAXD];
  const int task = blockIdx.y;
  const int wt = p.per_task ? task : 0;
  const int d = p.d;
  const int cp = threadIdx.x & 127, rsub = threadIdx.x >> 7;
  const int col = cp * 2;
  float w[2][MAXD], b[2];
#pragma unroll
  for (int c = 0; c < 2; ++c) {
    b[c] = p.b[size_t(wt) * H + col + c];
#pragma unroll
    for (int i = 0; i < MAXD; ++i) w[c][i] = (i < d) ? p.W[(size_t(wt) * H + col + c) * d + i] : 0.f;
  }
  const float w0 = p.w0, w0_rev = p.w0 * 0.15915494309189535f;
  const RowRange rr = block_rows(p.n_pad);
  for (int n0 = rr.n0; n0 < rr.n1; n0 += WCH) {
    __syncthreads();
    stage_x_chunk(p, task, n0, sx);
    __syncthreads();
#pragma unroll 2
    for (int r = rsub; r < WCH; r += 2) {
      const int n = n0 + r;
      if (n >= rr.n1) break;
      float z0 = b[0], z1 = b[1];
#pragma unroll
      for (int i4 = 0; i4 < MAXD / 4; ++i4) {
        const float4 xv = *reinterpret_cast<const float4*>(&sx[r * MAXD + 4 * i4]);   // warp-uniform: broadcast
        z0 = fmaf(xv.x, w[0][4 * i4], z0); z0 = fmaf(xv.y, w[0][4 * i4 + 1], z0);
        z0 = fmaf(xv.z, w[0][4 * i4 + 2], z0); z0 = fmaf(xv.w, w[0][4 * i4 + 3], z0);
        z1 = fmaf(xv.x, w[1][4 * i4], z1); z1 = fmaf(xv.y, w[1][4 * i4 + 1], z1);
        z1 = fmaf(xv.z, w[1][4 * i4 + 2], z1); z1 = fmaf(xv.w, w[1][4 * i4 + 3], z1);
      }
      float s0, c0, s1, c1;
      sincos_w0<SPLIT>(z0, w0, w0_rev, &s0, &c0);
      sincos_w0<SPLIT>(z1, w0, w0_rev, &s1, &c1);
      const size_t off = (size_t(task) * p.n_pad + n) * H + col;
      *reinterpret_cast<uint32_t*>(p.act_hi + off) = pack_bf16(s0, s1);
      if (SPLIT) {
        *reinterpret_cast<uint32_t*>(p.act_lo + off) = pack_bf16(s0 - bf16_round_f(s0), s1 - bf16_round_f(s1));
        if (p.c) *reinterpret_cast<float2*>(reinterpret_cast<float*>(p.c) + off) = make_float2(c0, c1);
      } else {
        if (p.c) *reinterpret_cast<uint32_t*>(reinterpret_cast<bf16*>(p.c) + off) = pack_bf16(c0, c1);
      }
    }
  }
}

template <bool SPLIT>
__global__ void __launch_bounds__(256) first_bwd_wide_kernel(FirstParams p) {
  // chunk of WCH rows: coordinates [WCH][MAXD] fp32 and the adjoint rows [WCH][256] bf16 (hi, lo);
  // the same buffer is reused for the final cross-phase reduction
  __shared__ __align__(16) float sx[WCH * MAXD];
  constexpr int SZ_WORDS = (SPLIT ? 2 : 1) * WCH * (H / 2);
  constexpr int RED_WORDS = 128 * 2 * (MAXD + 1);
  __shared__ __align__(16) uint32_t sz[SZ_WORDS > RED_WORDS ? SZ_WORDS : RED_WORDS];
  const int task = blockIdx.y;
  const int wt = p.per_task ? task : 0;
  const int d = p.d;
  const int cp = threadIdx.x & 127, rsub = threadIdx.x >> 7;
  const int col = cp * 2;
  float dw[2][MAXD], db[2] = {0.f, 0.f};
#pragma unroll
  for (int c = 0; c < 2; ++c)
#pragma unroll
    for (int i = 0; i < MAXD; ++i) dw[c][i] = 0.f;
  RowRange rr = block_rows(p.n_pad);
  if (rr.n1 > p.n) rr.n1 = p.n;
  for (int n0 = rr.n0; n0 < rr.n1; n0 += WCH) {
    __syncthreads();
    stage_x_chunk(p, task, n0, sx);
    // adjoint rows: WCH x 512 B = 1024 uint4 per plane, 4 per thread, fully coalesced
    for (int idx = threadIdx.x; idx < WCH * (H / 8); idx += blockDim.x) {
      const int r = idx / (H / 8), c8 = idx - r * (H / 8);
      const int n = n0 + r;
      uint4 v = make_uint4(0u, 0u, 0u, 0u), vl = v;
      if (n < rr.n1) {
        const size_t off = (size_t(task) * p.n_pad + n) * H + c8 * 8;
        v = __ldg(reinterpret_cast<const uint4*>(p.adj_hi + off));
        if (SPLIT) vl = __ldg(reinterpret_cast<const uint4*>(p.adj_lo + off));
      }
      reinterpret_cast<uint4*>(sz)[idx] = v;
      if (SPLIT) reinterpret_cast<uint4*>(sz + WCH * (H / 2))[idx] = vl;
    }
    __syncthreads();
#pragma unroll 2
    for (int r = rsub; r < WCH; r += 2) {
      uint32_t u = sz[r * (H / 2) + cp];
      float z0 = bf16_lo_f(u), z1 = bf16_hi_f(u);
      if (SPLIT) {
        u = sz[WCH * (H / 2) + r * (H / 2) + cp];
        z0 += bf16_lo_f(u);
        z1 += bf16_hi_f(u);
      }
      db[0] += z0;
      db[1] += z1;
#pragma unroll
      for (int i4 = 0; i4 < MAXD / 4; ++i4) {
        const float4 xv = *reinterpret_cast<const float4*>(&sx[r * MAXD + 4 * i4]);
        dw[0][4 * i4] = fmaf(z0, xv.x, dw[0][4 * i4]); dw[0][4 * i4 + 1] = fmaf(z0, xv.y, dw[0][4 * i4 + 1]);
        dw[0][4 * i4 + 2] = fmaf(z0, xv.z, dw[0][4 * i4 + 2]); dw[0][4 * i4 + 3] = fmaf(z0, xv.w, dw[0][4 * i4 + 3]);
        dw[1][4 * i4] = fmaf(z1, xv.x, dw[1][4 * i4]); dw[1][4 * i4 + 1] = fmaf(z1, xv.y, dw[1][4 * i4 + 1]);
        dw[1][4 * i4 + 2] = fmaf(z1, xv.z, dw[1][4 * i4 + 2]); dw[1][4 * i4 + 3] = fmaf(z1, xv.w, dw[1][4 * i4 + 3]);
      }
    }
  }
  // combine the two row phases of the block, then one atomic per element and block
  __syncthreads();
  float* red = reinterpret_cast<float*>(sz);          // RED_WORDS floats
  float* mine = red + (cp * 2) * (MAXD + 1);
  if (rsub == 1) {
#pragma unroll
    for (int c = 0; c < 2; ++c) {
#pragma unroll
      for (int i = 0; i < MAXD; ++i) mine[c * (MAXD + 1) + i] = dw[c][i];
      mine[c * (MAXD + 1) + MAXD] = db[c];
    }
  }
  __syncthreads();
  if (rsub == 0) {
#pragma unroll
    for (int c = 0; c < 2; ++c) {
#pragma unroll
      for (int i = 0; i < MAXD; ++i)
        if (i < d) atomicAdd(p.dW + (size_t(wt) * H + col + c) * d + i, dw[c][i] + mine[c * (MAXD + 1) + i]);
      atomicAdd(p.db + size_t(wt) * H + col + c, db[c] + mine[c * (MAXD + 1) + MAXD]);
    }
  }
}

// gradient reaching the coordinates through z0:  gx[n, i] = sum_col zbar0[n, col] W0[col, i]
template <bool SPLIT>
__global__ void __launch_bounds__(256) coords_grad_kernel(FirstParams p) {
  const int task = blockIdx.y;
  const int wt = p.per_task ? task : 0;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  RowRange rr = block_rows(p.n_pad);
  if (rr.n1 > p.n) rr.n1 = p.n;
  const float* W = p.W + size_t(wt) * H * p.d;
  for (int n = rr.n0 + warp; n < rr.n1; n += kWarps) {
    float zb[8];
    load_operand_chunk<8, SPLIT>(p.adj_hi, p.adj_lo, (size_t(task) * p.n_pad + n) * H + lane * 8, zb);
    for (int i = 0; i < p.d; ++i) {
      float acc = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) acc = fmaf(zb[j], __ldg(W + size_t(lane * 8 + j) * p.d + i), acc);
      acc = warp_sum(acc);
      if (lane == 0) p.gx[(size_t(task) * p.n + n) * p.d + i] = acc;
    }
  }
}

// -------------------------------------------------------------------------------------------
// bias gradient of a wide first layer in fp32-parity mode: column sums of its adjoint plane
// -------------------------------------------------------------------------------------------
template <bool SPLIT>
__global__ void __launch_bounds__(256) colsum_kernel(const bf16* __restrict__ hi, const bf16* __restrict__ lo,
                                                     float* __restrict__ db, int n_pad, int per_task) {
  __shared__ float red[kWarps * H];
  const int task = blockIdx.y;
  const int wt = per_task ? task : 0;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const RowRange rr = block_rows(n_pad);
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  constexpr int UN = 4;
  for (int nb = rr.n0 + warp * UN; nb < rr.n1; nb += kWarps * UN) {
    float v[UN][8];
#pragma unroll
    for (int u = 0; u < UN; ++u) {
      const int n = nb + u < rr.n1 ? nb + u : rr.n1 - 1;
      load_operand_chunk<8, SPLIT>(hi, lo, (size_t(task) * n_pad + n) * H + lane * 8, v[u]);
    }
#pragma unroll
    for (int u = 0; u < UN; ++u)
      if (nb + u < rr.n1) {
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] += v[u][j];
      }
  }
  block_cols_atomic(acc, red, db + size_t(wt) * H, 1);
}

// -------------------------------------------------------------------------------------------
// Wide first layer on the per-layer path (16 < d <= 256, fp32-parity mode): the layer runs as ONE MORE hidden layer
// of the tensor-core kernels on an input plane padded to 256 columns.
//   featurize   rows of inputs (the coordinates themselves, or -- ff.B -- the Fourier features of the raw coordinates,
//               features.py:31-41, accurate sinpi / cospi on the exact fraction) -> bf16 hi + lo planes [R, 256]
//   pad_w0      W_0 [tasks?][256][d] fp32 -> bf16 hi + lo [tasks? * 256][256], zero behind d
//   unpad_dw0   dW_0[.., i] += padded dW_0[.., i] for i < d
// -------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) featurize_kernel(FirstParams p) {
  const int task = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int col0 = lane * 8, d = p.d;
  const RowRange rr = block_rows(p.n_pad);
  for (int n = rr.n0 + warp; n < rr.n1; n += kWarps) {
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = 0.f;
    if (n < p.n && col0 < d) {
      if (p.ff.B) {
        const float* xr = p.x + (size_t(task) * p.n + n) * p.ff.raw;
        const float x[3] = {__ldg(xr), p.ff.raw > 1 ? __ldg(xr + 1) : 0.f, p.ff.raw > 2 ? __ldg(xr + 2) : 0.f};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int i = col0 + j;
          if (i < d) {
            const bool is_cos = i >= p.ff.F;
            v[j] = fourier_value<true>(fourier_frac(x, p.ff.raw, p.ff.B, p.ff.F, is_cos ? i - p.ff.F : i), is_cos);
          }
        }
      } else {
        const float* xp = p.x + (size_t(task) * p.n + n) * d;
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (col0 + j < d) v[j] = __ldg(xp + col0 + j);
      }
    }
    store_operand_chunk<8, true>(p.act_hi, p.act_lo, (size_t(task) * p.n_pad + n) * H + col0, v);
  }
}

__global__ void pad_w0_kernel(const float* __restrict__ W0, bf16* __restrict__ hi, bf16* __restrict__ lo, int d, long rows) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < rows * H; i += (long)gridDim.x * blockDim.x) {
    const long r = i / H;
    const int k = int(i - r * H);
    const float v = k < d ? W0[r * d + k] : 0.f;
    const bf16 h = __float2bfloat16_rn(v);
    hi[i] = h;
    lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
  }
}

__global__ void unpad_dw0_kernel(const float* __restrict__ pad, float* __restrict__ dW0, int d, long rows) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < rows * d; i += (long)gridDim.x * blockDim.x) {
    const long r = i / d;
    const int k = int(i - r * d);
    dW0[i] += pad[r * H + k];
  }
}

// the jet paths' streaming kernels on bf16 planes run staged (bulk copies into a shared-memory ring);
// SIREN_EDGE_STAGED=0 keeps the register-only loops for A/B runs.  Read on every call so a test can flip it within one
// process.  Both arms read and write the same workspace planes, so a forward and its backward may even disagree on it.
bool edge_staged() {
  const char* e = getenv("SIREN_EDGE_STAGED");
  return !(e && e[0] == '0');
}

dim3 edge_grid(int n_pad, int tasks, int num_sms, int min_rows, int blocks_per_sm = 8) {
  // enough blocks to fill the machine, each with at least `min_rows` rows.  Kernels that end in a
  // block-level atomic flush use fewer, longer blocks: same-address atomics serialise in L2.
  int want = (num_sms * blocks_per_sm + tasks - 1) / tasks;
  int maxb = (n_pad + min_rows - 1) / min_rows;
  if (want > maxb) want = maxb;
  if (want < 1) want = 1;
  return dim3(want, tasks);
}

}  // namespace

cudaError_t launch_first_fwd(FirstParams p, bool split, int num_sms, cudaStream_t stream) {
  const int tasks = p.R / p.n_pad;
  const dim3 grid = edge_grid(p.n_pad, tasks, num_sms, 32);
  if (p.d > 4 && p.order == 0) {      // fp32-parity only: the bf16 value path runs this layer in mlp_fused_pair.cu
    if (!split) return cudaErrorNotSupported;
    first_fwd_wide_kernel<true><<<grid, 256, 0, stream>>>(p);
    return cudaGetLastError();
  }
  if (split) first_fwd_kernel<true><<<grid, 256, 0, stream>>>(p);
  else first_fwd_kernel<false><<<grid, 256, 0, stream>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_first_bwd(FirstParams p, bool split, int num_sms, cudaStream_t stream) {
  const int tasks = p.R / p.n_pad;
  const dim3 grid = edge_grid(p.n_pad, tasks, num_sms, 64);
  const bool jets = p.order >= 1;
  if (p.only_gx) {
    if (!p.gx) return cudaSuccess;
    if (split) coords_grad_kernel<true><<<grid, 256, 0, stream>>>(p);
    else coords_grad_kernel<false><<<grid, 256, 0, stream>>>(p);
    return cudaGetLastError();
  }
  // bf16 planes come here for the jet paths only: the value path's dW_0 / db_0 come out of the fused kernels
  if (!split && !jets) return cudaErrorNotSupported;
  if (p.d > 4 && !jets) {
    const dim3 gw = edge_grid(p.n_pad, tasks, num_sms, 64, 6);   // 3 resident blocks / SM, 2 waves
    first_bwd_wide_kernel<true><<<gw, 256, 0, stream>>>(p);
    cudaError_t ew = cudaGetLastError();
    if (ew != cudaSuccess || !p.gx) return ew;
    coords_grad_kernel<true><<<grid, 256, 0, stream>>>(p);
    return cudaGetLastError();
  }
  if (jets && !split && p.d <= 3 && edge_staged()) {      // bf16 jet planes: the staged kernel
    const int smem = ST_STAGES * (1 + p.d) * ST2_ROWS * ST_ROW_BYTES;
    if (p.d == 1) { SIREN_ENSURE_SMEM(first_bwd_jets_staged_kernel<1>, ST_STAGES * 2 * ST2_ROWS * ST_ROW_BYTES); first_bwd_jets_staged_kernel<1><<<grid, 256, smem, stream>>>(p); }
    else if (p.d == 2) { SIREN_ENSURE_SMEM(first_bwd_jets_staged_kernel<2>, ST_STAGES * 3 * ST2_ROWS * ST_ROW_BYTES); first_bwd_jets_staged_kernel<2><<<grid, 256, smem, stream>>>(p); }
    else { SIREN_ENSURE_SMEM(first_bwd_jets_staged_kernel<3>, ST_STAGES * 4 * ST2_ROWS * ST_ROW_BYTES); first_bwd_jets_staged_kernel<3><<<grid, 256, smem, stream>>>(p); }
    cudaError_t es = cudaGetLastError();
    if (es != cudaSuccess || !p.gx) return es;
    coords_grad_kernel<false><<<grid, 256, 0, stream>>>(p);
    return cudaGetLastError();
  }
#define FB(SP, DC, JT) first_bwd_kernel<SP, DC, JT><<<grid, 256, 0, stream>>>(p)
  if (split) {
    if (jets) { if (p.d == 1) FB(true, 1, true); else if (p.d == 2) FB(true, 2, true); else FB(true, 3, true); }
    else { if (p.d == 1) FB(true, 1, false); else if (p.d == 2) FB(true, 2, false); else if (p.d == 3) FB(true, 3, false); else FB(true, 4, false); }
  } else {
    if (p.d == 1) FB(false, 1, true); else if (p.d == 2) FB(false, 2, true); else FB(false, 3, true);
  }
#undef FB
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  if (p.gx) {
    if (split) coords_grad_kernel<true><<<grid, 256, 0, stream>>>(p);
    else coords_grad_kernel<false><<<grid, 256, 0, stream>>>(p);
    e = cudaGetLastError();
  }
  return e;
}

cudaError_t launch_last_fwd(LastParams p, bool split, int num_sms, cudaStream_t stream) {
  const int tasks = p.R / p.n_pad;
  const dim3 grid = edge_grid(p.n_pad, tasks, num_sms, 32);
  if (p.order >= 1 && !split && !p.phase && p.d <= 3 && edge_staged()) {      // bf16 jet planes: the staged kernel
    const int S = 1 + p.order * p.d;
    const int n_stages = S <= 4 ? ST_STAGES : 2;      // <= 96 KB of stages per block up to five planes: two blocks per SM
    const int smem = n_stages * S * ST2_ROWS * ST_ROW_BYTES;
    SIREN_ENSURE_SMEM(last_fwd_staged_kernel, ST_STAGES * 7 * ST2_ROWS * ST_ROW_BYTES);
    last_fwd_staged_kernel<<<grid, 256, smem, stream>>>(p, n_stages);
    return cudaGetLastError();
  }
  if (split) last_fwd_kernel<true><<<grid, 256, 0, stream>>>(p);
  else last_fwd_kernel<false><<<grid, 256, 0, stream>>>(p);
  return cudaGetLastError();
}

template <bool SPLIT, bool JETS>
static cudaError_t launch_last_bwd_t(const LastParams& p, dim3 grid, cudaStream_t stream) {
  if (p.o <= 1) last_bwd_kernel<SPLIT, 1, JETS><<<grid, 256, 0, stream>>>(p);
  else if (p.o <= 2) last_bwd_kernel<SPLIT, 2, JETS><<<grid, 256, 0, stream>>>(p);
  else if (p.o <= 4) last_bwd_kernel<SPLIT, 4, JETS><<<grid, 256, 0, stream>>>(p);
  else last_bwd_kernel<SPLIT, 8, JETS><<<grid, 256, 0, stream>>>(p);
  return cudaGetLastError();
}

template <int OMAX>
static cudaError_t launch_last_bwd_staged(const LastParams& p, dim3 grid, cudaStream_t stream) {
  const int npl = 2 + 2 * p.order * p.d;
  const int n_stages = npl <= 8 ? ST_STAGES : 2;      // two blocks per SM either way (<= 96 KB of stages each)
  const int smem = n_stages * npl * ST_ROWS * ST_ROW_BYTES;
  SIREN_ENSURE_SMEM(last_bwd_jets_staged_kernel<OMAX>, ST_STAGES * 14 * ST_ROWS * ST_ROW_BYTES);
  last_bwd_jets_staged_kernel<OMAX><<<grid, 256, smem, stream>>>(p, n_stages);
  return cudaGetLastError();
}

cudaError_t launch_last_bwd(LastParams p, bool split, int num_sms, cudaStream_t stream) {
  const int tasks = p.R / p.n_pad;
  const dim3 grid = edge_grid(p.n_pad, tasks, num_sms, 64);
  // jets on bf16 planes: the staged kernel (bulk copies into a shared-memory ring); SIREN_EDGE_STAGED=0 keeps the
  // register-only loop for A/B runs.
  if (edge_staged() && p.order >= 1 && !split && !p.phase && p.d <= 3) {
    if (p.o <= 1) return launch_last_bwd_staged<1>(p, grid, stream);
    if (p.o <= 2) return launch_last_bwd_staged<2>(p, grid, stream);
    if (p.o <= 4) return launch_last_bwd_staged<4>(p, grid, stream);
    return launch_last_bwd_staged<8>(p, grid, stream);
  }
  if (p.order >= 1)
    return split ? launch_last_bwd_t<true, true>(p, grid, stream) : launch_last_bwd_t<false, true>(p, grid, stream);
  return split ? launch_last_bwd_t<true, false>(p, grid, stream) : launch_last_bwd_t<false, false>(p, grid, stream);
}

cudaError_t launch_featurize(FirstParams p, int num_sms, cudaStream_t stream) {
  const int tasks = p.R / p.n_pad;
  featurize_kernel<<<edge_grid(p.n_pad, tasks, num_sms, 64), 256, 0, stream>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_pad_w0(const float* W0, bf16* hi, bf16* lo, int d, long rows, int num_sms, cudaStream_t stream) {
  pad_w0_kernel<<<num_sms * 2, 256, 0, stream>>>(W0, hi, lo, d, rows);
  return cudaGetLastError();
}

cudaError_t launch_unpad_dw0(const float* pad, float* dW0, int d, long rows, int num_sms, cudaStream_t stream) {
  unpad_dw0_kernel<<<num_sms * 2, 256, 0, stream>>>(pad, dW0, d, rows);
  return cudaGetLastError();
}

cudaError_t launch_colsum(const bf16* hi, const bf16* lo, float* db, int R, int n_pad, int per_task, int num_sms,
                          cudaStream_t stream) {
  const int tasks = R / n_pad;
  const dim3 grid = edge_grid(n_pad, tasks, num_sms, 64);
  colsum_kernel<true><<<grid, 256, 0, stream>>>(hi, lo, db, n_pad, per_task);
  return cudaGetLastError();
}

}  // namespace siren
