// Weight-gradient kernel on tcgen05:  dW_l[out, in] = sum over coordinates (and jet streams) of
// adj_l[n, out] * act_{l-1}[n, in]   -- the dW = dz^T h term of the autograd backward that
// training.py:91 triggers through modules.py:25 (SURVEY.md section 8a row a10, appendix A).
//
// The contraction runs over coordinates, so both operands are "MN-major" for the tensor core:
// TMA drops [KC coordinates x 64 features] boxes (128-byte swizzle) straight from the row-major
// planes and the UMMA descriptors read them transposed; no transposed copies exist in HBM.
// One CTA owns a whole 256x256 fp32 accumulator (2 x 256 TMEM columns) for a slice of the
// coordinates and flushes it once with vector red.add.
#include "common.cuh"
#include "ptx.cuh"
#include "simt.h"

namespace siren {

namespace {

constexpr int kThreads = 384;
constexpr int kEpiWarp0 = 4;
constexpr int kEpiWarps = 8;
constexpr int kStages = 3;

template <bool SPLIT>
struct WgCfg {
  static constexpr int KC = SPLIT ? 32 : 64;            // coordinates per pipeline stage
  static constexpr int OPER = KC * H * 2;               // bytes of one operand block (all 256 features)
  static constexpr int STAGE = OPER * (SPLIT ? 4 : 2);  // 64 KB either way
  static constexpr int SMEM = kStages * STAGE + 1024 + 1024;
};

__device__ __forceinline__ void red_add_v4(float* dst, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(a), "f"(b), "f"(c), "f"(d)
               : "memory");
}

struct Item {
  int layer, row0, row1, task;
};

__device__ __host__ __forceinline__ int wgrad_items(const WgradParams& p) {
  const int groups = p.per_task ? p.tasks : 1;
  const int kinds = p.n_layers + (p.first_wide ? 1 : 0);
  return p.slices0 > 0 ? groups * (p.slices0 + (kinds - 1) * p.slices) : kinds * groups * p.slices;
}

__device__ __forceinline__ Item decode_item(const WgradParams& p, int idx) {
  Item it;
  const int kinds = p.n_layers + (p.first_wide ? 1 : 0);      // index n_layers: the wide first layer's own item
  const int groups = p.per_task ? p.tasks : 1;
  int slices = p.slices, rest;
  if (p.slices0 > 0) {
    // kind 0 is cut into more (shorter) slices than the other kinds; its items come first
    const int n0 = groups * p.slices0;
    if (idx < n0) {
      it.layer = 0;
      rest = idx;
      slices = p.slices0;
    } else {
      idx -= n0;
      it.layer = 1 + idx % (kinds - 1);
      rest = idx / (kinds - 1);
    }
  } else {
    // (the kind rotates with the slice index: a CTA that takes several items -- items = CTAs + a remainder, stride =
    //  grid size, often a multiple of the number of kinds -- then gets DIFFERENT kinds, not the slowest one twice)
    rest = idx / kinds;
    it.layer = (idx % kinds + rest) % kinds;
  }
  const int grp = rest / slices;
  const int sl = rest % slices;
  const int rows_group = p.per_task ? p.rows_per_task : p.R;
  const int tiles = rows_group / TILE_M;
  const int base = tiles / slices, rem = tiles % slices;
  const int t0 = sl * base + (sl < rem ? sl : rem);
  const int n = base + (sl < rem ? 1 : 0);
  it.row0 = grp * rows_group + t0 * TILE_M;
  it.row1 = it.row0 + n * TILE_M;
  it.task = p.per_task ? grp : 0;
  return it;
}

// RAGGED (scenes of different sizes, simt.h ragged_tables): the items of the launch's n_layers kinds over the scenes'
// slices, kinds rotating with the slice index as above; scene t's slices split its own plane rows
__device__ __forceinline__ int wgrad_items_ragged(const WgradParams& p) {
  return p.n_layers * __ldg(p.rag + RAG_SLICE * (p.tasks + 1) + p.tasks);
}

__device__ __forceinline__ Item decode_item_ragged(const WgradParams& p, int idx) {
  Item it;
  const int kinds = p.n_layers, S = p.tasks + 1;
  const int rest = idx / kinds;
  it.layer = (idx % kinds + rest) % kinds;
  const int* sl0 = p.rag + RAG_SLICE * S;
  int lo = 0, hi = p.tasks - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(sl0 + mid) <= rest) lo = mid;
    else hi = mid - 1;
  }
  const int first = __ldg(sl0 + lo), slices = __ldg(sl0 + lo + 1) - first, sl = rest - first;
  const int p0 = __ldg(p.rag + RAG_PROW * S + lo);
  const int tiles = (__ldg(p.rag + RAG_PROW * S + lo + 1) - p0) / TILE_M;
  const int base = tiles / slices, rem = tiles % slices;
  const int t0 = sl * base + (sl < rem ? sl : rem);
  const int n = base + (sl < rem ? 1 : 0);
  it.row0 = p0 + t0 * TILE_M;
  it.row1 = it.row0 + n * TILE_M;
  it.task = lo;
  return it;
}

template <bool RAGGED>
__device__ __forceinline__ Item decode(const WgradParams& p, int idx) {
  if constexpr (RAGGED) return decode_item_ragged(p, idx);
  else return decode_item(p, idx);
}

// Column sums of one staged adjoint block ([4 feature blocks][KC coordinates][64 features] bf16, 128-byte swizzle):
// thread = one pair of adjacent columns (word db_off / unit db_unit) and one half of the rows.
template <int KC>
__device__ __forceinline__ void adj_colsum(uint32_t ablk, int rhalf, uint32_t db_unit, float& bs0, float& bs1) {
#pragma unroll
  for (int rb = 0; rb < KC / 2; rb += 8) {       // eight loads in flight before the first is consumed
    uint32_t u[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int row = rhalf * (KC / 2) + rb + i;
      u[i] = ptx::ld_shared_u32(ablk + uint32_t(row) * 128u + ((db_unit ^ uint32_t(row & 7)) << 4));
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      bs0 += bf16_lo_f(u[i]);
      bs1 += bf16_hi_f(u[i]);
    }
  }
}

// Items of the FIRST hidden layer when its B operand has no plane (l0_from_x, narrow inputs): the flush warps build
// sin(w0 (x W0^T + b0)) for every stage from the coordinates, as the block TMA would have dropped from a sine plane
// -- [4 feature blocks][KC coordinates][64 features] bf16, 128-byte swizzle.  The 256 flush threads split a block as
// (16-byte unit lu of a row, feature block fb, group rg of eight rows); the eight rows of a warp are the same for all
// its lanes, lane i < 8 fetches row i's coordinates (one stage AHEAD, so the load is never waited for) and hands
// them round by shuffle.  The B half of a stage is free as soon as the MMA that last read the stage has committed
// (the producer waits on the same barrier phase), so building runs in parallel with the adjoint block's TMA load.
// theta_0 is the forward's own FMA chain (mlp_fused_pair.cu first_rows): the operand is bit for bit the activation
// the forward multiplied with.
template <int D, int KC, int STAGE_BYTES, int OPER_BYTES, bool RAGGED>
__device__ __forceinline__ void first_layer_item(const WgradParams& p, const Item& it, uint8_t* smem, uint64_t* full,
                                                 uint64_t* empty, uint64_t* ready, int& stage, uint32_t& phase, int tid,
                                                 int lane, bool has_db, uint32_t db_off, int rhalf, uint32_t db_unit,
                                                 float& bs0, float& bs1) {
  constexpr uint32_t LBO = KC * 128;
  const int lu = tid & 7, fb = (tid >> 3) & 3, rg = tid >> 5;
  const int f0 = fb * 64 + lu * 8;
  float w[8][D], b[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
#pragma unroll
    for (int k = 0; k < D; ++k) w[j][k] = p.w0 * __ldg(p.W0 + (size_t(it.task) * H + f0 + j) * D + k);
    b[j] = p.w0 * __ldg(p.b0 + size_t(it.task) * H + f0 + j);
  }
  int p0 = 0, x0 = 0, n_t = 0;      // RAGGED: the item's scene (its rows are all this scene's)
  if constexpr (RAGGED) {
    const int S = p.tasks + 1;
    p0 = __ldg(p.rag + RAG_PROW * S + it.task);
    x0 = __ldg(p.rag + RAG_XROW * S + it.task);
    n_t = __ldg(p.rag + RAG_XROW * S + it.task + 1) - x0;
  }
  auto fetch = [&](int r, float* cx) {      // coordinates of plane row r + rg * 8 + (lane & 7); zero behind the task's n
    const int rp = r + rg * 8 + (lane & 7);
    if constexpr (RAGGED) {
      const int nl = rp - p0;
#pragma unroll
      for (int k = 0; k < D; ++k) cx[k] = (r < it.row1 && nl < n_t) ? __ldg(p.x + (size_t(x0) + nl) * D + k) : 0.f;
    } else {
      const int task = rp / p.rows_per_task, nl = rp - task * p.rows_per_task;
#pragma unroll
      for (int k = 0; k < D; ++k) cx[k] = (r < it.row1 && nl < p.n) ? __ldg(p.x + (size_t(task) * p.n + nl) * D + k) : 0.f;
    }
  };
  float cx[D], cn[D];
  fetch(it.row0, cx);
  for (int r = it.row0; r < it.row1; r += KC) {
    fetch(r + KC, cn);
    ptx::mbar_wait(&empty[stage], phase ^ 1u);
    const uint32_t blk = ptx::smem_u32(smem + stage * STAGE_BYTES + OPER_BYTES);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float xr[D];
#pragma unroll
      for (int k = 0; k < D; ++k) xr[k] = __shfl_sync(0xffffffffu, cx[k], i);
      uint32_t o[4];
#pragma unroll
      for (int j2 = 0; j2 < 4; ++j2) {
        float ta = fmaf(xr[0], w[2 * j2][0], b[2 * j2]), tb = fmaf(xr[0], w[2 * j2 + 1][0], b[2 * j2 + 1]);
#pragma unroll
        for (int k = 1; k < D; ++k) {
          ta = fmaf(xr[k], w[2 * j2][k], ta);
          tb = fmaf(xr[k], w[2 * j2 + 1][k], tb);
        }
        o[j2] = pack_bf16(__sinf(ta), __sinf(tb));
      }
      // row (rg * 8 + i) & 7 == i
      ptx::st_shared_v4(blk + uint32_t(fb) * LBO + uint32_t(rg * 8 + i) * 128u + (uint32_t(lu ^ i) << 4), o[0], o[1], o[2], o[3]);
    }
    ptx::mbar_wait(&full[stage], phase);                    // the adjoint block has landed
    if (has_db) adj_colsum<KC>(ptx::smem_u32(smem + stage * STAGE_BYTES) + db_off, rhalf, db_unit, bs0, bs1);
    ptx::fence_proxy_async();
    __syncwarp();
    if (lane == 0) ptx::mbar_arrive(&ready[stage]);
    if (++stage == kStages) { stage = 0; phase ^= 1u; }
#pragma unroll
    for (int k = 0; k < D; ++k) cx[k] = cn[k];
  }
}

// Items of a WIDE first layer (4 < d <= 16, first_wide): dW_0 = zbar_0^T x on the tensor core.  The B block of a stage is
// [KC coordinates][64 columns] bf16 (one feature block, 128-byte swizzle) of which the MMA reads N = 32 columns: the
// row's inputs as bf16 hi terms (columns 0..15) and lo terms (16..31), so the product carries x to ~2^-17.  The flush
// warps build it: thread = (row tid >> 2 of the stage, inputs 4 c .. 4 c + 3); the inputs are the coordinates
// themselves or, with ff.B, the Fourier features of the raw coordinates (features.py:31-41) -- fetched one stage
// ahead.  db_0 comes from the staged adjoint block like every other layer's.
template <int KC, int STAGE_BYTES, int OPER_BYTES>
__device__ __forceinline__ void wide_first_item(const WgradParams& p, const Item& it, uint8_t* smem, uint64_t* full,
                                                uint64_t* empty, uint64_t* ready, int& stage, uint32_t& phase, int tid,
                                                int lane, bool has_db, uint32_t db_off, int rhalf, uint32_t db_unit,
                                                float& bs0, float& bs1) {
  const int r_in = tid >> 2, c = tid & 3, d = p.d;
  const bool ffm = p.ff.B != nullptr;
  auto fetch = [&](int r, float* raw4, bool& live) {      // this thread's row of the stage starting at plane row r
    const int rp = r + r_in;
    const int task = rp / p.rows_per_task, nl = rp - task * p.rows_per_task;
    live = rp < it.row1 && nl < p.n;
    raw4[0] = raw4[1] = raw4[2] = raw4[3] = 0.f;
    if (!live) return;
    if (ffm) {
      const float* xr = p.x + (size_t(task) * p.n + nl) * p.ff.raw;
      raw4[0] = __ldg(xr);
      if (p.ff.raw > 1) raw4[1] = __ldg(xr + 1);
      if (p.ff.raw > 2) raw4[2] = __ldg(xr + 2);
    } else {
      const float* xp = p.x + (size_t(task) * p.n + nl) * d + 4 * c;
#pragma unroll
      for (int j = 0; j < 4; ++j) raw4[j] = (4 * c + j < d) ? __ldg(xp + j) : 0.f;
    }
  };
  float cur[4], nxt[4];
  bool live, live_n;
  fetch(it.row0, cur, live);
  const uint32_t unit_hi = uint32_t(c >> 1), unit_lo = 2u + uint32_t(c >> 1), off8 = uint32_t(c & 1) * 8u;
  for (int r = it.row0; r < it.row1; r += KC) {
    fetch(r + KC, nxt, live_n);
    // materialised inputs: this thread's four consecutive inputs 4 c .. 4 c + 3.  Fourier features: projections c and
    // c + 4 of the row (F <= 8), sine AND cosine of each from one exact fraction (this kernel only runs in the bf16
    // mode: the SFU on the reduced argument, ~5e-7 absolute, is far below the operand rounding)
    float v[4];
    int col[4];
    if (!ffm) {
#pragma unroll
      for (int j = 0; j < 4; ++j) { v[j] = cur[j]; col[j] = 4 * c + j; }
    } else {
      const float xr[3] = {cur[0], cur[1], cur[2]};
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const int pj = c + 4 * k;
        float sv = 0.f, cv = 0.f;
        if (live && pj < p.ff.F) {
          const float a = 6.283185307179586f * fourier_frac(xr, p.ff.raw, p.ff.B, p.ff.F, pj);
          sv = __sinf(a);
          cv = __cosf(a);
        }
        v[2 * k] = sv; col[2 * k] = pj < p.ff.F ? pj : 99;                   // (99: a projection the layer does not
        v[2 * k + 1] = cv; col[2 * k + 1] = pj < p.ff.F ? p.ff.F + pj : 99;     //  have -- nothing is written for it)
      }
    }
    ptx::mbar_wait(&empty[stage], phase ^ 1u);      // the MMA that last read this stage's B half has committed
    const uint32_t row = ptx::smem_u32(smem + stage * STAGE_BYTES + OPER_BYTES) + uint32_t(r_in) * 128u;
    const uint32_t sw = uint32_t(r_in & 7);
    if (!ffm) {
      float h[4], l[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        h[j] = bf16_round_f(v[j]);
        l[j] = bf16_round_f(v[j] - h[j]);
      }
      asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(row + ((unit_hi ^ sw) << 4) + off8), "r"(pack_bf16(h[0], h[1])),
                   "r"(pack_bf16(h[2], h[3])) : "memory");
      asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(row + ((unit_lo ^ sw) << 4) + off8), "r"(pack_bf16(l[0], l[1])),
                   "r"(pack_bf16(l[2], l[3])) : "memory");
    } else {
      if (2 * p.ff.F < 16 && c == 0) {      // columns 2 F .. 15 (hi and lo) are read by the MMA: keep them zero
        for (int z = 2 * p.ff.F; z < 16; ++z)
#pragma unroll
          for (int part = 0; part < 2; ++part) {
            const uint32_t byte = uint32_t(z + 16 * part) * 2u;
            asm volatile("st.shared.u16 [%0], %1;" ::"r"(row + (((byte >> 4) ^ sw) << 4) + (byte & 15u)), "h"((unsigned short)0) : "memory");
          }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (col[j] >= 2 * p.ff.F) continue;
        const float h = bf16_round_f(v[j]), l = bf16_round_f(v[j] - h);
        const __nv_bfloat16 hb = __float2bfloat16_rn(h), lb = __float2bfloat16_rn(l);
        const uint32_t bh = uint32_t(col[j]) * 2u, bl = bh + 32u;
        asm volatile("st.shared.u16 [%0], %1;" ::"r"(row + (((bh >> 4) ^ sw) << 4) + (bh & 15u)),
                     "h"(*reinterpret_cast<const unsigned short*>(&hb)) : "memory");
        asm volatile("st.shared.u16 [%0], %1;" ::"r"(row + (((bl >> 4) ^ sw) << 4) + (bl & 15u)),
                     "h"(*reinterpret_cast<const unsigned short*>(&lb)) : "memory");
      }
    }
    ptx::mbar_wait(&full[stage], phase);            // the adjoint block has landed
    if (has_db) adj_colsum<KC>(ptx::smem_u32(smem + stage * STAGE_BYTES) + db_off, rhalf, db_unit, bs0, bs1);
    ptx::fence_proxy_async();
    __syncwarp();
    if (lane == 0) ptx::mbar_arrive(&ready[stage]);
    if (++stage == kStages) { stage = 0; phase ^= 1u; }
#pragma unroll
    for (int j = 0; j < 4; ++j) cur[j] = nxt[j];
    live = live_n;
  }
}

template <bool SPLIT, bool RAGGED>
__global__ void __launch_bounds__(kThreads, 1) wgrad_kernel(const __grid_constant__ WgradParams p) {
  using Cfg = WgCfg<SPLIT>;
  constexpr int KC = Cfg::KC;
  constexpr uint32_t IDESC = ptx::umma_idesc_bf16(TILE_M, 256, 1, 1);
  constexpr uint32_t IDESC_W0 = ptx::umma_idesc_bf16(TILE_M, 32, 1, 1);      // wide first layer: N = hi | lo inputs
  constexpr uint32_t LBO = KC * 128;     // bytes between 64-feature blocks
  constexpr uint32_t SBO = 1024;         // bytes between groups of 8 coordinates

  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kStages * Cfg::STAGE);
  uint64_t* full = bars;
  uint64_t* empty = bars + kStages;
  uint64_t* acc_full = bars + 2 * kStages;
  uint64_t* acc_empty = bars + 2 * kStages + 1;
  uint64_t* ready = bars + 2 * kStages + 2;         // [kStages] phase_b: the B block has been turned into sines
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * kStages + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int n_items = RAGGED ? wgrad_items_ragged(p) : wgrad_items(p);
  if (p.dbg && threadIdx.x == 0) {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    p.dbg[3 * blockIdx.x + 0] = int(blockIdx.x) < n_items ? decode<RAGGED>(p, blockIdx.x).layer : -1;
    p.dbg[3 * blockIdx.x + 1] = t;
  }

  if (warp == 1 && lane == 0) {
    for (int i = 0; i < kStages; ++i) {
      ptx::mbar_init(&full[i], 1);
      ptx::mbar_init(&empty[i], 1);
      ptx::mbar_init(&ready[i], kEpiWarps);
    }
    ptx::mbar_init(acc_full, 1);
    ptx::mbar_init(acc_empty, kEpiWarps);
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(tmem_slot, 512);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int idx = blockIdx.x; idx < n_items; idx += gridDim.x) {
        const Item it = decode<RAGGED>(p, idx);
        const bool wide0 = !SPLIT && p.first_wide && it.layer == p.n_layers;
        const int li = wide0 ? 0 : it.layer;
        const CUtensorMap* mA_hi = wide0 ? &p.tmA0 : &p.tmA_hi[li];
        const CUtensorMap* mB_hi = &p.tmB_hi[li];      // (plane0 items: redirected below)
        const CUtensorMap* mA_lo = &p.tmA_lo[li];
        const CUtensorMap* mB_lo = &p.tmB_lo[li];
        const bool plane0 = wide0 && p.d > 16;      // d > 16: the forward left the first layer's input plane
        const bool gen = (wide0 && !plane0) || (!SPLIT && p.l0_from_x && it.layer == 0);      // B is built on chip
        if (plane0) mB_hi = &p.tmB0;
        const int nfb = plane0 ? p.nkc0 : 4;        // feature blocks of the B operand that are loaded
        for (int r = it.row0; r < it.row1; r += KC)
          for (int s = 0; s < p.S; ++s) {
            ptx::mbar_wait(&empty[stage], phase ^ 1u);
            ptx::mbar_arrive_expect_tx(&full[stage], gen ? Cfg::OPER : plane0 ? Cfg::OPER + nfb * int(LBO) : Cfg::STAGE);
            uint8_t* st = smem + stage * Cfg::STAGE;
            const int y = s * p.R + r;
#pragma unroll
            for (int fb = 0; fb < 4; ++fb) {
              ptx::tma_load_2d(st + fb * LBO, mA_hi, &full[stage], fb * 64, y);
              if (!gen && fb < nfb) ptx::tma_load_2d(st + Cfg::OPER + fb * LBO, mB_hi, &full[stage], fb * 64, y);
              if (SPLIT) {
                ptx::tma_load_2d(st + 2 * Cfg::OPER + fb * LBO, mA_lo, &full[stage], fb * 64, y);
                ptx::tma_load_2d(st + 3 * Cfg::OPER + fb * LBO, mB_lo, &full[stage], fb * 64, y);
              }
            }
            if (++stage == kStages) { stage = 0; phase ^= 1u; }
          }
      }
    }
  } else if (warp == 1) {
    int stage = 0;
    uint32_t phase = 0;
    int local = 0;
    for (int idx = blockIdx.x; idx < n_items; idx += gridDim.x, ++local) {
      const Item it = decode<RAGGED>(p, idx);
      ptx::mbar_wait(acc_empty, (uint32_t(local) & 1u) ^ 1u);
      ptx::tc_fence_after();
      const uint32_t idesc = !(!SPLIT && p.first_wide && it.layer == p.n_layers) ? IDESC
                             : p.d > 16 ? ptx::umma_idesc_bf16(TILE_M, 64 * p.nkc0, 1, 1)      // the input plane's blocks
                             : IDESC_W0;
      bool first = true;
      for (int r = it.row0; r < it.row1; r += KC)
        for (int s = 0; s < p.S; ++s) {
          ptx::mbar_wait((p.phase_b || p.db_plain) ? &ready[stage] : &full[stage], phase);
          ptx::tc_fence_after();
          if (lane == 0) {
            const uint32_t base = ptx::smem_u32(smem + stage * Cfg::STAGE);
#pragma unroll
            for (int mh = 0; mh < 2; ++mh) {
              const uint32_t d_tmem = tmem_base + uint32_t(mh * 256);
#pragma unroll
              for (int ks = 0; ks < KC / 16; ++ks) {
                const uint32_t a_hi = base + 2 * mh * LBO + ks * 2048;
                const uint32_t b_hi = base + Cfg::OPER + ks * 2048;
                const uint32_t acc0 = (first && ks == 0) ? 0u : 1u;
                ptx::umma_bf16(d_tmem, ptx::umma_smem_desc(a_hi, LBO, SBO), ptx::umma_smem_desc(b_hi, LBO, SBO),
                               idesc, acc0);
                if (SPLIT) {
                  const uint32_t a_lo = base + 2 * Cfg::OPER + 2 * mh * LBO + ks * 2048;
                  const uint32_t b_lo = base + 3 * Cfg::OPER + ks * 2048;
                  ptx::umma_bf16(d_tmem, ptx::umma_smem_desc(a_hi, LBO, SBO),
                                 ptx::umma_smem_desc(b_lo, LBO, SBO), IDESC, 1u);
                  ptx::umma_bf16(d_tmem, ptx::umma_smem_desc(a_lo, LBO, SBO),
                                 ptx::umma_smem_desc(b_hi, LBO, SBO), IDESC, 1u);
                }
              }
            }
            ptx::umma_commit(&empty[stage]);
          }
          __syncwarp();
          first = false;
          if (++stage == kStages) { stage = 0; phase ^= 1u; }
        }
      if (lane == 0) ptx::umma_commit(acc_full);
      __syncwarp();
    }
  } else if (warp >= kEpiWarp0) {
    const int e = warp - kEpiWarp0;
    const int q = warp & 3;
    const int chalf = e >> 2;
    int local = 0;
    int stage = 0;
    uint32_t phase = 0;
    for (int idx = blockIdx.x; idx < n_items; idx += gridDim.x, ++local) {
      const Item it = decode<RAGGED>(p, idx);
      if (p.db_plain) {
        // Per-layer paths (bf16 x 3 operands, jets): the planes are ready-made operands, nothing to convert -- but the
        // bias gradient db_l = sum over coordinates of zbar_l (value stream; hi + lo in split mode) is the column sum of
        // the adjoint blocks that pass through the stages anyway, so the eight warps take it here instead of a separate
        // pass over the planes (colsum: 2 x 51 us of the 1.7 ms fp32-parity step at cfg2).
        const int tid = e * 32 + lane;
        float* dbp = p.db[it.layer];
        const int cp = tid & 127, rhalf = tid >> 7;
        const uint32_t db_off = uint32_t(cp >> 5) * LBO + (uint32_t(cp & 3) << 2);
        const uint32_t db_unit = uint32_t((cp & 31) >> 2);
        float bs0 = 0.f, bs1 = 0.f;
        for (int r = it.row0; r < it.row1; r += KC)
          for (int sidx = 0; sidx < p.S; ++sidx) {
            ptx::mbar_wait(&full[stage], phase);
            if (dbp && sidx == 0) {
              adj_colsum<KC>(ptx::smem_u32(smem + stage * Cfg::STAGE) + db_off, rhalf, db_unit, bs0, bs1);
              if (SPLIT) adj_colsum<KC>(ptx::smem_u32(smem + stage * Cfg::STAGE + 2 * Cfg::OPER) + db_off, rhalf, db_unit, bs0, bs1);
            }
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&ready[stage]);
            if (++stage == kStages) { stage = 0; phase ^= 1u; }
          }
        if (dbp && it.row1 > it.row0) {
          float* dst = dbp + size_t(it.task) * H + 2 * cp;
          atomicAdd(dst, bs0);
          atomicAdd(dst + 1, bs1);
        }
      }
      if (!SPLIT && p.phase_b) {
        // The B planes carry the layer input as the forward stashed it: the signed sine, fp16 (common.cuh).  The
        // adjoints need bf16's exponent range and kind::f16 takes ONE format pair per instruction (a bf16 x fp16
        // descriptor raises an illegal-instruction fault), so the eight warps turn each staged 32 KB block into bf16
        // in place (flat, 16 bytes per thread and step: two conversions per pair, no SFU) and hand the stage to the
        // MMA warp.
        const int tid = e * 32 + lane;
        // While a stage is in their hands the same warps also take the column sums of its adjoint block (the A
        // operand, [4 feature blocks][64 coordinates][64 features], 128-byte swizzle): the bias gradient
        // db_l = sum over coordinates of zbar_l.  Thread = one pair of adjacent columns and one half of the rows.
        const bool wide0 = p.first_wide && it.layer == p.n_layers;
        float* dbp = wide0 ? p.db0 : p.db[it.layer];
        const int cp = tid & 127, rhalf = tid >> 7;               // column pair 0..127, row half 0..1
        const uint32_t db_off = uint32_t(cp >> 5) * LBO + (uint32_t(cp & 3) << 2);   // feature block, word in its unit
        const uint32_t db_unit = uint32_t((cp & 31) >> 2);        // 16-byte unit inside the 128-byte row
        float bs0 = 0.f, bs1 = 0.f;
        if (wide0 && p.d > 16) {
          // the B operand is the first layer's input plane as the forward stored it (bf16): nothing to build or convert
          for (int r = it.row0; r < it.row1; r += KC) {
            ptx::mbar_wait(&full[stage], phase);
            if (dbp) adj_colsum<KC>(ptx::smem_u32(smem + stage * Cfg::STAGE) + db_off, rhalf, db_unit, bs0, bs1);
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&ready[stage]);
            if (++stage == kStages) { stage = 0; phase ^= 1u; }
          }
        } else if (wide0) {
          wide_first_item<KC, Cfg::STAGE, Cfg::OPER>(p, it, smem, full, empty, ready, stage, phase, tid, lane, dbp != nullptr,
                                                     db_off, rhalf, db_unit, bs0, bs1);
        } else if (p.l0_from_x && it.layer == 0) {
          switch (p.d) {
            case 1: first_layer_item<1, KC, Cfg::STAGE, Cfg::OPER, RAGGED>(p, it, smem, full, empty, ready, stage, phase, tid, lane, dbp != nullptr, db_off, rhalf, db_unit, bs0, bs1); break;
            case 2: first_layer_item<2, KC, Cfg::STAGE, Cfg::OPER, RAGGED>(p, it, smem, full, empty, ready, stage, phase, tid, lane, dbp != nullptr, db_off, rhalf, db_unit, bs0, bs1); break;
            case 3: first_layer_item<3, KC, Cfg::STAGE, Cfg::OPER, RAGGED>(p, it, smem, full, empty, ready, stage, phase, tid, lane, dbp != nullptr, db_off, rhalf, db_unit, bs0, bs1); break;
            default: first_layer_item<4, KC, Cfg::STAGE, Cfg::OPER, RAGGED>(p, it, smem, full, empty, ready, stage, phase, tid, lane, dbp != nullptr, db_off, rhalf, db_unit, bs0, bs1); break;
          }
        } else
        for (int r = it.row0; r < it.row1; r += KC) {
          ptx::mbar_wait(&full[stage], phase);
          const uint32_t blk = ptx::smem_u32(smem + stage * Cfg::STAGE + Cfg::OPER);
          if (dbp) adj_colsum<KC>(ptx::smem_u32(smem + stage * Cfg::STAGE) + db_off, rhalf, db_unit, bs0, bs1);
#pragma unroll
          for (int i = 0; i < Cfg::OPER / (kEpiWarps * 32 * 16); ++i) {
            const uint32_t a = blk + uint32_t(i * kEpiWarps * 32 + tid) * 16u;
            uint32_t w[4];
            ptx::ld_shared_v4(a, w[0], w[1], w[2], w[3]);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float2 h = __half22float2(*reinterpret_cast<const __half2*>(&w[j]));
              w[j] = pack_bf16(h.x, h.y);
            }
            ptx::st_shared_v4(a, w[0], w[1], w[2], w[3]);
          }
          ptx::fence_proxy_async();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&ready[stage]);
          if (++stage == kStages) { stage = 0; phase ^= 1u; }
        }
        if (dbp && it.row1 > it.row0) {
          float* dst = dbp + size_t(it.task) * H + 2 * cp;
          atomicAdd(dst, bs0);
          atomicAdd(dst + 1, bs1);
        }
      }
      ptx::mbar_wait(acc_full, uint32_t(local) & 1u);
      ptx::tc_fence_after();
      const bool has_rows = it.row1 > it.row0;
      if (!SPLIT && p.first_wide && it.layer == p.n_layers) {
        if (p.d > 16) {      // N = 64 nkc0 columns of which d are real: the regular block walk, row stride d
#pragma unroll
          for (int mh = 0; mh < 2; ++mh) {
            const int orow = mh * 128 + q * 32 + lane;
#pragma unroll 1
            for (int cc = 0; cc < 4; ++cc) {
              const int col = chalf * 128 + cc * 32;
              if (col >= p.d) break;
              float v[32];
              ptx::tmem_ld32(tmem_base + (uint32_t(q * 32) << 16) + uint32_t(mh * 256 + col), reinterpret_cast<uint32_t*>(v));
              ptx::tmem_wait_ld();
              if (has_rows) {
                float* dst = p.dW0 + (size_t(it.task) * H + orow) * p.d + col;
#pragma unroll
                for (int i = 0; i < 32; ++i)
                  if (col + i < p.d) atomicAdd(dst + i, v[i]);
              }
            }
          }
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(acc_empty);
          continue;
        }
        // dW_0[row, i] = acc[row, i] (hi terms) + acc[row, 16 + i] (lo terms); the four chalf == 0 warps cover the lanes
        if (chalf == 0) {
#pragma unroll
          for (int mh = 0; mh < 2; ++mh) {
            const int orow = mh * 128 + q * 32 + lane;
            float v[32];
            ptx::tmem_ld32(tmem_base + (uint32_t(q * 32) << 16) + uint32_t(mh * 256), reinterpret_cast<uint32_t*>(v));
            ptx::tmem_wait_ld();
            if (has_rows) {
              float* dst = p.dW0 + (size_t(it.task) * H + orow) * p.d;
              if (p.d == 16) {
#pragma unroll
                for (int i = 0; i < 4; ++i)
                  red_add_v4(dst + 4 * i, v[4 * i] + v[16 + 4 * i], v[4 * i + 1] + v[17 + 4 * i], v[4 * i + 2] + v[18 + 4 * i],
                             v[4 * i + 3] + v[19 + 4 * i]);
              } else {
#pragma unroll
                for (int i = 0; i < 16; ++i)
                  if (i < p.d) atomicAdd(dst + i, v[i] + v[16 + i]);
              }
            }
          }
        }
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(acc_empty);
        continue;
      }
      float* dW = p.dW[it.layer] + size_t(it.task) * H * H;
      // every CTA flushes the same 256 KB at about the same time: each starts at a different block of it, so the
      // red.adds of the split-K slices spread over the L2 slices instead of queueing on the same lines
      const int rot = blockIdx.x;
#pragma unroll
      for (int mh_ = 0; mh_ < 2; ++mh_) {
        const int mh = (mh_ + (rot >> 2)) & 1;
        const int orow = mh * 128 + q * 32 + lane;
#pragma unroll
        for (int cc_ = 0; cc_ < 4; ++cc_) {
          const int cc = (cc_ + rot) & 3;
          const int col = chalf * 128 + cc * 32;
          float v[32];
          ptx::tmem_ld32(tmem_base + (uint32_t(q * 32) << 16) + uint32_t(mh * 256 + col),
                         reinterpret_cast<uint32_t*>(v));
          ptx::tmem_wait_ld();
          if (has_rows) {
            float* dst = dW + size_t(orow) * H + col;
#pragma unroll
            for (int i = 0; i < 8; ++i) red_add_v4(dst + 4 * i, v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
          }
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(acc_empty);
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (p.dbg && threadIdx.x == 0) {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    p.dbg[3 * blockIdx.x + 2] = t;
  }
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, 512);
  }
}

}  // namespace

int wgrad_kc(bool split) { return split ? 32 : 64; }

cudaError_t launch_wgrad(const WgradParams& p, bool split, int num_sms, cudaStream_t stream) {
  const int n_items = wgrad_items(p);
  int grid = n_items < num_sms ? n_items : num_sms;
  if (grid < 1) return cudaSuccess;
  if (split) {
    SIREN_ENSURE_SMEM((wgrad_kernel<true, false>), WgCfg<true>::SMEM);
    wgrad_kernel<true, false><<<grid, kThreads, WgCfg<true>::SMEM, stream>>>(p);
  } else {
    SIREN_ENSURE_SMEM((wgrad_kernel<false, false>), WgCfg<false>::SMEM);
    wgrad_kernel<false, false><<<grid, kThreads, WgCfg<false>::SMEM, stream>>>(p);
  }
  return cudaGetLastError();
}

// bf16 only; grid: at most the item count (the items are counted on the device, from the tables)
cudaError_t launch_wgrad_ragged(const WgradParams& p, int grid, cudaStream_t stream) {
  if (grid < 1) return cudaSuccess;
  SIREN_ENSURE_SMEM((wgrad_kernel<false, true>), WgCfg<false>::SMEM);
  wgrad_kernel<false, true><<<grid, kThreads, WgCfg<false>::SMEM, stream>>>(p);
  return cudaGetLastError();
}

}  // namespace siren
