// The forward, MSE gradient and input-gradient chain of a bf16 training step in ONE kernel on CTA pairs (cluster of 2,
// tcgen05 cta_group::2): image_mse, value stream, d_in <= 4, d_out <= 2, <= 4 hidden layers.  It runs, per unit of
// its pair's range, what mlp_fused_pair.cu (forward, STASH) and mlp_fused_bwd.cu (fuse_top, l0_from_x) run in two
// launches, with the same arithmetic in the same order:
//
//   forward        layer 0 from the coordinates, hidden layers 1..L on the tensor core (fp16 W_l), y, the loss sum and
//                  gy = 2 w (y - gt) where a row's y is completed.  Stash planes 1..L-1 are TMA-stored for the weight
//                  gradients; the top layer's signed sine stays in the A tile and is never stored
//   top step       zbar_L = (gy WL) * w0 cos(theta_L), dWL, dbL in column layout, reading h_L from the tile the forward
//                  has just written and gy from shared memory (the quadrant's sub == 0 warp leaves it there)
//   chain          zbar_l = (zbar_{l+1} w0 W_{l+1}) * cos(theta_l), l = L-1..1, on the tensor core (bf16 w0 W_l^T): the
//                  stash tile is TMA-loaded into the drained A tile, read back from L2 (this pair wrote it a few
//                  microseconds earlier); the bottom pass forms db_0 / dW_0 from theta_0 recomputed from x
//
// Compared with the two launches this removes the top stash plane, the launch boundary with its second prologue, the
// gy round trip through HBM and the critical-path wait on HBM for stash loads that fell out of L2.
//
// Roles: warp 0 streams 2 L weight layers per unit through the 4-slot ring (W_1..W_L, then w0 W_L^T..W_1^T), warp 1
// issues the MMAs of both halves (leader CTA), warp 2 owns TMEM, warp 3 owns the bulk copies of the backward half
// (stash loads, adjoint stores), warps 4..19 are the epilogue of both halves.  X and Y stay skewed by half a step
// throughout: the forward's top layer and the top step run tile by tile, so Y's forward epilogue overlaps X's first
// backward MMA.
#include "common.cuh"
#include "ptx.cuh"
#include "simt.h"
#include "mlp_fused_parts.cuh"

#include <type_traits>

namespace siren {

namespace {

constexpr int MAXL = MAX_FUSED_STEP_HIDDEN;
// per row of the tile in flight: [0..2] the partial last-layer dots of the sub 1..3 warps, [3] gy (two outputs each).
// One tile's worth is enough: the quadrant barrier behind gy orders its reuse for the other tile
constexpr int Y_BYTES = TILE_M * NSUB * 2 * 4;            // 4 KB
constexpr int BIAS_BYTES = MAXL * H * 4;                  // w0 * b_l of hidden layers 1..L
constexpr int WL_BYTES = 2 * H * 4;                       // outermost linear rows (d_out <= 2)
constexpr int NSUM = 1 + 4;                               // partial-sum rows per warp: db_0, dW0[:, k]; dWL reuses rows 0, 1
constexpr int SUM_BYTES = EPI_WARPS * NSUM * 64 * 4;      // 20 KB
constexpr int MISC = 1024;
constexpr int SMEM_STEP = 2 * A_TILE + NKC * B_SLOT + Y_BYTES + BIAS_BYTES + WL_BYTES + SUM_BYTES + MISC + 1024;
static_assert(SMEM_STEP <= 232448, "shared memory budget");

struct UnitInfo {
  int task, ntile;
  int row0[2];
  bool valid[2];
};
__device__ __forceinline__ UnitInfo unit_info(const MlpFwdParams& p, int unit, int rank) {
  const int tiles_task = (p.rows_per_task + 255) / 256;
  const int units_task = (tiles_task + 1) / 2;
  UnitInfo u;
  u.task = unit / units_task;
  const int lu = unit - u.task * units_task;
  u.ntile = (2 * lu + 1 < tiles_task) ? 2 : 1;
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    const int r = (2 * lu + t) * 256 + rank * TILE_M;
    u.valid[t] = r < p.rows_per_task;
    u.row0[t] = u.task * p.rows_per_task + r;
  }
  return u;
}

// w0 W0 and w0 b0 of columns c, c + 1 (the values the forward kernel stages in shared memory and the chain's bottom
// pass forms): unused coordinates are zero
__device__ __forceinline__ void first_weights(const MlpFwdParams& p, int wt, int c, float4& wa, float4& wb, float& ba,
                                              float& bb) {
  const float w0 = p.w0;
  const float* wr = p.W0 + (size_t(wt) * H + c) * p.d;
  wa = make_float4(w0 * __ldg(wr), 0.f, 0.f, 0.f);
  wb = make_float4(w0 * __ldg(wr + p.d), 0.f, 0.f, 0.f);
  if (p.d > 1) { wa.y = w0 * __ldg(wr + 1); wb.y = w0 * __ldg(wr + p.d + 1); }
  if (p.d > 2) { wa.z = w0 * __ldg(wr + 2); wb.z = w0 * __ldg(wr + p.d + 2); }
  if (p.d > 3) { wa.w = w0 * __ldg(wr + 3); wb.w = w0 * __ldg(wr + p.d + 3); }
  ba = w0 * __ldg(p.b0 + size_t(wt) * H + c);
  bb = w0 * __ldg(p.b0 + size_t(wt) * H + c + 1);
}

__device__ __forceinline__ void row_coords(const MlpFwdParams& p, const UnitInfo& ui, int t, int row_t, float* x) {
  x[0] = x[1] = x[2] = x[3] = 0.f;
  const int nr = ui.row0[t] + row_t - ui.task * p.rows_per_task;
  if (t < ui.ntile && ui.valid[t] && nr < p.n) {
    const float* xp = p.x + (size_t(ui.task) * p.n + nr) * p.d;
    x[0] = __ldg(xp);
    if (p.d > 1) x[1] = __ldg(xp + 1);
    if (p.d > 2) x[2] = __ldg(xp + 2);
    if (p.d > 3) x[3] = __ldg(xp + 3);
  }
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
    mlp_fused_step_kernel(const __grid_constant__ MlpStepParams sp) {
  const MlpFwdParams& p = sp.f;
  const MlpBwdParams& pb = sp.b;
  constexpr uint32_t IDESC_F = ptx::umma_idesc_f16(256, 256, 0, 0, ptx::FMT_F16, ptx::FMT_F16);   // forward
  constexpr uint32_t IDESC_B = ptx::umma_idesc_bf16(256, 256, 0, 0);                              // chain
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;                                             // [2 tiles][4 chunks][128][128 B]
  uint8_t* sB = sA + 2 * A_TILE;                                  // [4 k-chunks][128][128 B]
  float* sY = reinterpret_cast<float*>(sB + NKC * B_SLOT);        // [128][NSUB][2]
  float* sBias = sY + Y_BYTES / 4;                                // [MAXL][256], times w0
  float* sWL = sBias + MAXL * H;                                  // [2][256]
  float* sSum = sWL + 2 * H;                                      // [16 warps][NSUM][64]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sSum + EPI_WARPS * NSUM * 64);
  uint64_t* b_full = bars;                // [NKC]  leader's: both halves of a weight chunk landed
  uint64_t* b_empty = bars + NKC;         // [NKC]  multicast commit: the slot's last MMA is done
  uint64_t* acc_full = bars + 2 * NKC;    // [2]    multicast commit: accumulator ready, A tile drained
  uint64_t* a_ready = acc_full + 2;       // [2]    leader's: 16 warps x 2 CTAs wrote the A tile
  uint64_t* c_full = a_ready + 2;         // [2][4] local: chunk kc of the A tile holds the stash tile (chain), or may be
                                          //        rewritten (the next unit's layer 0, the bottom pass)
  uint64_t* written = c_full + 8;         // [2]    local: the 16 epilogue warps wrote an adjoint into the A tile
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(written + 2);
  float* sDbL = reinterpret_cast<float*>(tmem_slot + 4);          // [4 quadrants][2]
  float* sLoss = sDbL + 8;                                        // [4 quadrants]

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int NH = p.n_hidden;
  const int rank = int(ptx::cluster_ctarank());
  const bool leader = rank == 0;
  const int n_cl = gridDim.x >> 1, cl = blockIdx.x >> 1;
  const int tiles_task = (p.rows_per_task + 255) / 256;
  const int n_units = ((tiles_task + 1) / 2) * p.tasks;
  const int base = n_units / n_cl, rem = n_units % n_cl;
  const int u0 = cl * base + (cl < rem ? cl : rem);
  const int u1 = u0 + base + (cl < rem ? 1 : 0);

  if (warp == 0 && lane == 0) {
    for (int l = 0; l < NH; ++l) {
      ptx::prefetch_tmap(&p.tmW[l]);
      ptx::prefetch_tmap(&pb.tmWt[l]);
      if (l > 0) {
        ptx::prefetch_tmap(&p.tmAct[l]);
        ptx::prefetch_tmap(&pb.tmC[l]);
      }
      ptx::prefetch_tmap(&pb.tmAdj[l + 1]);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < NKC; ++i) {
      ptx::mbar_init(&b_full[i], 1);
      ptx::mbar_init(&b_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&acc_full[i], 1);
      ptx::mbar_init(&a_ready[i], 2 * EPI_WARPS);
      for (int kc = 0; kc < 4; ++kc) ptx::mbar_init(&c_full[i * 4 + kc], 1);
      ptx::mbar_init(&written[i], EPI_WARPS);
    }
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc_pair(tmem_slot, 512);
    ptx::tmem_relinquish_pair();
  }
  for (int i = threadIdx.x; i < EPI_WARPS * NSUM * 64; i += kThreads) sSum[i] = 0.f;
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();           // both CTAs' barriers are initialised before any remote arrive / multicast commit
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // register split as in the two kernels: 128 x 56 + 512 x 104 inside the 640 x 96 of the launch
  if (warp < 4) {
  ptx::setmaxnreg_dec<56>();
  if (warp == 0) {
    // ===================== weight producer (both CTAs: each loads its half of the output features) ==========
    if (lane == 0) {
      uint32_t n = 0;            // layers streamed so far: slot kc holds K chunk kc of every layer, once per layer
      for (int un = u0; un < u1; ++un) {
        const UnitInfo ui = unit_info(p, un, rank);
        const int wrow = (p.per_task ? ui.task : 0) * H + rank * 128;
        for (int s = 0; s < 2 * NH; ++s, ++n) {
          const CUtensorMap* tm = s < NH ? &p.tmW[s] : &pb.tmWt[2 * NH - 1 - s];
          for (int kc = 0; kc < NKC; ++kc) {
            ptx::mbar_wait(&b_empty[kc], (n & 1u) ^ 1u);      // Y of the previous layer is done with the slot
            if (leader) ptx::mbar_arrive_expect_tx(&b_full[kc], 2 * B_SLOT);
            ptx::tma_load_2d_pair(sB + kc * B_SLOT, tm, &b_full[kc], kc * KCHUNK, wrow);
          }
        }
      }
      // the last multicast commits have landed in this CTA before it may exit
      for (int kc = 0; kc < NKC; ++kc) ptx::mbar_wait(&b_empty[kc], (n & 1u) ^ 1u);
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (leader) {
      uint32_t n = 0;                // layers so far (phases of b_full)
      uint32_t rnd = 0u;             // bit tl: phase of a_ready[tl]
      for (int un = u0; un < u1; ++un) {
        const UnitInfo ui = unit_info(p, un, rank);
        for (int s = 0; s < 2 * NH; ++s, ++n) {
          for (int tl = 0; tl < ui.ntile; ++tl) {
            ptx::mbar_wait_cluster(&a_ready[tl], (rnd >> tl) & 1u);   // both CTAs: A tile written, accumulator drained
            rnd ^= 1u << tl;
            for (int kc = 0; kc < NKC; ++kc) {
              if (tl == 0) ptx::mbar_wait(&b_full[kc], n & 1u);
              ptx::tc_fence_after();
              if (lane == 0) {
                const uint32_t a_addr = ptx::smem_u32(sA + tl * A_TILE + kc * A_CHUNK);
                const uint32_t b_addr = ptx::smem_u32(sB + kc * B_SLOT);
#pragma unroll
                for (int ks = 0; ks < 4; ++ks)
                  ptx::umma_bf16_pair(tmem_base + uint32_t(tl * 256), ptx::umma_smem_desc(a_addr + ks * 32, 16, 1024),
                                      ptx::umma_smem_desc(b_addr + ks * 32, 16, 1024), s < NH ? IDESC_F : IDESC_B,
                                      (kc | ks) ? 1u : 0u);
                if (tl == ui.ntile - 1) ptx::umma_commit_pair(&b_empty[kc], 3);
              }
              __syncwarp();
            }
            if (lane == 0) ptx::umma_commit_pair(&acc_full[tl], 3);
            __syncwarp();
          }
        }
      }
    }
  } else if (warp == 3) {
    // ===================== tile loader (both CTAs): the bulk copies of the backward half =====================
    // As in mlp_fused_bwd.cu: in the order the epilogue walks the chain's tiles, load the stash tile of step k once
    // MMA(k) has drained the A tile, then retire step k-1 (store its adjoint).  A tile's bottom step frees it for the
    // next unit's forward (c_full), after the stores that left from it have been read.
    if (lane == 0) {
      uint32_t accph = 0u, wrph = 0u;
      auto tile_free = [&](int tl) {
        for (int kc = 0; kc < 4; ++kc) ptx::mbar_arrive(&c_full[tl * 4 + kc]);
      };
      struct Pending {
        int un, l, tl, row0;
        bool valid;
      } pd = {-1, 0, 0, 0, false};
      auto retire = [&]() {
        if (pd.un < 0) return;
        ptx::mbar_wait(&written[pd.tl], (wrph >> pd.tl) & 1u);
        wrph ^= 1u << pd.tl;
        if (pd.l == NH)
          // the top step follows the epilogue warps' wait for their stash stores to complete: the stash tiles this
          // thread loads next are read from global memory by the async proxy
          ptx::fence_proxy_async_global();
        if (pd.valid && pd.l > 0) {
          for (int kc = 0; kc < 4; ++kc)
            ptx::tma_store_2d(&pb.tmAdj[pd.l], sA + pd.tl * A_TILE + kc * A_CHUNK, kc * KCHUNK, pd.row0);
          ptx::bulk_commit();
        }
        if (pd.l == 0 && pd.un + 1 < u1) {         // bottom step (nothing stored): the tile is free for the next unit
          const UnitInfo nx = unit_info(p, pd.un + 1, rank);
          if (pd.tl < nx.ntile) tile_free(pd.tl);
        }
        pd.un = -1;
      };
      if (u0 < u1) {
        const UnitInfo ui = unit_info(p, u0, rank);
        for (int tl = 0; tl < ui.ntile; ++tl) tile_free(tl);
      }
      for (int un = u0; un < u1; ++un) {
        const UnitInfo ui = unit_info(p, un, rank);
        if (un > u0) {               // a tile the previous (single-tile) unit did not use: nobody freed it
          const UnitInfo pv = unit_info(p, un - 1, rank);
          for (int tl = pv.ntile; tl < ui.ntile; ++tl) {
            ptx::bulk_wait_read<0>();
            tile_free(tl);
          }
        }
        // the forward's NH accumulator phases of each tile are the epilogue's; this thread waits on the chain's only.
        // (It is never more than one phase behind: it reaches a tile's first chain wait after the top step of that
        // tile, i.e. after the forward consumed its phases.)
        for (int tl = 0; tl < ui.ntile; ++tl) accph ^= uint32_t(NH & 1) << tl;
        for (int tl = 0; tl < ui.ntile; ++tl) {    // top step: the epilogue turns the A tile into zbar_L
          retire();
          pd.un = un; pd.l = NH; pd.tl = tl; pd.row0 = ui.row0[tl]; pd.valid = ui.valid[tl];
        }
        for (int l = NH - 1; l >= 0; --l)
          for (int tl = 0; tl < ui.ntile; ++tl) {
            if (pd.un >= 0 && pd.tl == tl) retire();                // single-tile unit: same buffer, store it first
            ptx::mbar_wait(&acc_full[tl], (accph >> tl) & 1u);      // the MMA has read the A tile (both CTAs')
            accph ^= 1u << tl;
            ptx::bulk_wait_read<0>();                               // ... and so has the last store issued from it
            if (l == 0) {
              // narrow first layer: no stash plane -- the epilogue only needs to know that the tile may be rewritten
              tile_free(tl);
            } else {
              for (int kc = 0; kc < 4; ++kc) {
                ptx::mbar_arrive_expect_tx(&c_full[tl * 4 + kc], A_CHUNK);
                ptx::tma_load_2d(sA + tl * A_TILE + kc * A_CHUNK, &pb.tmC[l], &c_full[tl * 4 + kc], kc * KCHUNK, ui.row0[tl]);
              }
            }
            retire();
            pd.un = un; pd.l = l; pd.tl = tl; pd.row0 = ui.row0[tl]; pd.valid = ui.valid[tl];
          }
      }
      retire();
      ptx::bulk_wait_all();
    }
  }
  } else {
    ptx::setmaxnreg_inc<104>();
    // ===================== epilogue warps (both CTAs) =====================
    const int e = warp - 4;
    const int q = warp & 3;                 // TMEM lane quadrant this warp may read
    const int sub = e >> 2;                 // K chunk (64 columns) this warp owns
    const int tid_e = threadIdx.x - 128;
    const int row_t = q * 32 + lane;
    const float w0 = p.w0;
    const int colw = sub * 64;
    EpiOut eo;
    eo.a_row = ptx::smem_u32(sA) + uint32_t(sub) * A_CHUNK + uint32_t(row_t) * 128u;
    eo.row7 = row_t & 7;
    eo.lane = lane;
    const uint32_t lane_off = uint32_t(lane & 3) * 4u, unit16 = uint32_t(lane >> 2);
    // This warp's stash stores leave from its A slices (forward).  A slice may be rewritten once the store that last
    // left from it has been read out; the stores alternate between the tiles, so one younger group may stay in flight
    // when the latest store was the other tile's.
    int last_store_tl = -1;
    auto slice_free = [&](int tl) {
      if (lane == 0) {
        if (last_store_tl == tl) ptx::bulk_wait_read<0>();
        else ptx::bulk_wait_read<1>();
      }
      __syncwarp();
    };
    uint32_t accph = 0u, cph = 0u;          // bit tl: phases of acc_full[tl], c_full[tl * 4 + sub]
    int cur_task = -1;
    float lsum = 0.f;                       // sum of (y - gt)^2 over the rows this thread completes
    const uint32_t wl_addr = ptx::smem_u32(sWL + colw);
    float* my_sum = sSum + e * (NSUM * 64);
    const int n_dw0 = p.d;
    float dbl0 = 0.f, dbl1 = 0.f;           // sum of gy over this warp's rows (sub == 0 warps)
    float dwl00 = 0.f, dwl01 = 0.f, dwl10 = 0.f, dwl11 = 0.f;      // dWL[i, colw + 2 lane + {0, 1}]
    float w00 = 0.f, w01 = 0.f, w10 = 0.f, w11 = 0.f;              // w0 WL[i, colw + 2 lane + {0, 1}]

    // partial sums -> global, as in mlp_fused_bwd.cu: the four quadrant warps of a column chunk are combined, then ONE
    // atomic per element and CTA
    auto flush = [&](int wt) {
      ptx::named_bar_sync(15, EPI_WARPS * 32);
      for (int i = tid_e; i < (1 + n_dw0) * H; i += EPI_WARPS * 32) {
        const int r = i / H, col = i - r * H;
        float* s = sSum + ((col >> 6) * 4) * (NSUM * 64) + r * 64 + (col & 63);
        const float tot = s[0] + s[NSUM * 64] + s[2 * NSUM * 64] + s[3 * NSUM * 64];
        s[0] = s[NSUM * 64] = s[2 * NSUM * 64] = s[3 * NSUM * 64] = 0.f;
        if (r < 1) atomicAdd(pb.db[0] + size_t(wt) * H + col, tot);
        else atomicAdd(pb.dW0 + (size_t(wt) * H + col) * p.d + (r - 1), tot);
      }
      ptx::named_bar_sync(15, EPI_WARPS * 32);
      float2* d0 = reinterpret_cast<float2*>(my_sum) + lane;
      d0[0] = make_float2(dwl00, dwl01);
      if (p.o > 1) d0[32] = make_float2(dwl10, dwl11);
      if (sub == 0 && lane == 0) {
        sDbL[q * 2 + 0] = dbl0;
        sDbL[q * 2 + 1] = dbl1;
      }
      dwl00 = dwl01 = dwl10 = dwl11 = 0.f;
      dbl0 = dbl1 = 0.f;
      ptx::named_bar_sync(15, EPI_WARPS * 32);
      for (int i = tid_e; i < p.o * H; i += EPI_WARPS * 32) {
        const int r = i / H, col = i - r * H;
        float* s = sSum + ((col >> 6) * 4) * (NSUM * 64) + r * 64 + (col & 63);
        const float tot = s[0] + s[NSUM * 64] + s[2 * NSUM * 64] + s[3 * NSUM * 64];
        s[0] = s[NSUM * 64] = s[2 * NSUM * 64] = s[3 * NSUM * 64] = 0.f;
        atomicAdd(pb.dWL + (size_t(wt) * p.o + r) * H + col, tot);
      }
      if (tid_e < p.o)
        atomicAdd(pb.dbL + size_t(wt) * p.o + tid_e, sDbL[tid_e] + sDbL[2 + tid_e] + sDbL[4 + tid_e] + sDbL[6 + tid_e]);
      ptx::named_bar_sync(15, EPI_WARPS * 32);
    };

    for (int un = u0; un < u1; ++un) {
      const UnitInfo ui = unit_info(p, un, rank);
      const int wt = p.per_task ? ui.task : 0;
      if (wt != cur_task) {                  // (re)load the biases and outermost weights of this task
        if (cur_task >= 0) flush(cur_task);
        ptx::named_bar_sync(15, EPI_WARPS * 32);
        for (int col = tid_e; col < H; col += EPI_WARPS * 32) {
          for (int l = 0; l < NH; ++l) sBias[l * H + col] = w0 * __ldg(p.bias[l] + size_t(wt) * H + col);
          sWL[col] = __ldg(p.WL + (size_t(wt) * p.o) * H + col);
          sWL[H + col] = p.o > 1 ? __ldg(p.WL + (size_t(wt) * p.o + 1) * H + col) : 0.f;
        }
        ptx::named_bar_sync(15, EPI_WARPS * 32);
        cur_task = wt;
        const float2 wl0 = __ldg(reinterpret_cast<const float2*>(p.WL + (size_t(wt) * p.o) * H + colw) + lane);
        w00 = w0 * wl0.x; w01 = w0 * wl0.y;
        if (p.o > 1) {
          const float2 wl1 = __ldg(reinterpret_cast<const float2*>(p.WL + (size_t(wt) * p.o + 1) * H + colw) + lane);
          w10 = w0 * wl1.x; w11 = w0 * wl1.y;
        }
      }
      // ---------------- forward, layer 0 (d <= 4): SIMT, straight into the A tiles ----------------
      float cx[2][4];
      row_coords(p, ui, 0, row_t, cx[0]);
      row_coords(p, ui, 1, row_t, cx[1]);
      for (int tl = 0; tl < ui.ntile; ++tl) {
        float4 wa, wb;
        float ba, bb;
        first_weights(p, wt, colw + 2 * lane, wa, wb, ba, bb);
        const uint32_t a_slice = ptx::smem_u32(sA) + uint32_t(tl) * A_TILE + uint32_t(sub) * A_CHUNK +
                                 uint32_t(q) * (32u * 128u);
        const float cxt[4] = {tl ? cx[1][0] : cx[0][0], tl ? cx[1][1] : cx[0][1], tl ? cx[1][2] : cx[0][2],
                              tl ? cx[1][3] : cx[0][3]};
        slice_free(tl);
        ptx::mbar_wait(&c_full[tl * 4 + sub], (cph >> tl) & 1u);    // the previous unit's chain is done with the tile
        cph ^= 1u << tl;
        switch (p.d) {
          case 1: first_rows<1>(eo, a_slice, cxt, wa, wb, ba, bb); break;
          case 2: first_rows<2>(eo, a_slice, cxt, wa, wb, ba, bb); break;
          case 3: first_rows<3>(eo, a_slice, cxt, wa, wb, ba, bb); break;
          default: first_rows<4>(eo, a_slice, cxt, wa, wb, ba, bb); break;
        }
        ptx::fence_proxy_async();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive_leader(&a_ready[tl]);
      }
      // ---------------- forward, hidden layers 1..L; the top one ends in y, the loss and the top step ----------------
      for (int l = 1; l <= NH; ++l) {
        const bool top = (l == NH);
        if (top && sub == 0 && un + 1 < u1) {      // pull the next unit's coordinates towards L2 while this one finishes
          const UnitInfo nx = unit_info(p, un + 1, rank);
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            const int nr = nx.row0[t] + row_t - nx.task * p.rows_per_task;
            if (t < nx.ntile && nx.valid[t] && nr < p.n) ptx::prefetch_l2(p.x + (size_t(nx.task) * p.n + nr) * p.d);
          }
        }
        const uint32_t bias_addr = ptx::smem_u32(sBias + (l - 1) * H + colw);
        for (int tl = 0; tl < ui.ntile; ++tl) {
          const int row0 = ui.row0[tl];
          const bool valid = ui.valid[tl];
          const int n_row = row0 + row_t - ui.task * p.rows_per_task;
          const uint32_t taddr = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(tl * 256 + colw);
          float ydot0 = 0.f, ydot1 = 0.f;
          float gt0 = 0.f, gt1 = 0.f;       // this row's target, fetched now, used when the row's y is complete
          if (top && sub == 0 && valid && n_row < p.n) {
            const float* gp = p.gt + (size_t(ui.task) * p.n + n_row) * p.o;
            gt0 = __ldg(gp);
            if (p.o > 1) gt1 = __ldg(gp + 1);
          }
          float va[PW], vb[PW];
          ptx::mbar_wait(&acc_full[tl], (accph >> tl) & 1u);
          accph ^= 1u << tl;
          ptx::tc_fence_after();
          ptx::tmem_ld<PW>(taddr, reinterpret_cast<uint32_t*>(va));
          slice_free(tl);                   // the store that last left from this slice (one layer ago) has been read
#pragma unroll
          for (int pc = 0; pc < NPIECE; ++pc) {
            float* v = (pc & 1) ? vb : va;
            ptx::tmem_wait_ld();
            if (pc + 1 < NPIECE)
              ptx::tmem_ld<PW>(taddr + uint32_t((pc + 1) * PW), reinterpret_cast<uint32_t*>((pc & 1) ? va : vb));
            float t[PW], s[PW];
#pragma unroll
            for (int j4 = 0; j4 < PW / 4; ++j4) {
              const float4 bb = ptx::ld_shared_f4(bias_addr + uint32_t(pc * (PW / 4) + j4) * 16u);
              t[4 * j4 + 0] = fmaf(v[4 * j4 + 0], w0, bb.x);
              t[4 * j4 + 1] = fmaf(v[4 * j4 + 1], w0, bb.y);
              t[4 * j4 + 2] = fmaf(v[4 * j4 + 2], w0, bb.z);
              t[4 * j4 + 3] = fmaf(v[4 * j4 + 3], w0, bb.w);
            }
            piece_out<true>(eo, tl, pc, t, s, true);
            if (top) {
#pragma unroll
              for (int j4 = 0; j4 < PW / 4; ++j4) {
                const float4 ww = ptx::ld_shared_f4(wl_addr + uint32_t(pc * (PW / 4) + j4) * 16u);
                ydot0 = fmaf(s[4 * j4 + 0], ww.x, ydot0); ydot0 = fmaf(s[4 * j4 + 1], ww.y, ydot0);
                ydot0 = fmaf(s[4 * j4 + 2], ww.z, ydot0); ydot0 = fmaf(s[4 * j4 + 3], ww.w, ydot0);
              }
              if (p.o > 1) {
#pragma unroll
                for (int j4 = 0; j4 < PW / 4; ++j4) {
                  const float4 ww = ptx::ld_shared_f4(wl_addr + uint32_t(H * 4) + uint32_t(pc * (PW / 4) + j4) * 16u);
                  ydot1 = fmaf(s[4 * j4 + 0], ww.x, ydot1); ydot1 = fmaf(s[4 * j4 + 1], ww.y, ydot1);
                  ydot1 = fmaf(s[4 * j4 + 2], ww.z, ydot1); ydot1 = fmaf(s[4 * j4 + 3], ww.w, ydot1);
                }
              }
            }
          }
          ptx::tc_fence_before();
          if (!top) {
            ptx::fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
              if (valid) {      // the slice as it stands is the layer's stash plane (signed sine)
                ptx::tma_store_2d(&p.tmAct[l], sA + tl * A_TILE + sub * A_CHUNK + q * (32 * 128), colw, row0 + q * 32);
                ptx::bulk_commit();
              }
              ptx::mbar_arrive_leader(&a_ready[tl]);
            }
            if (valid) last_store_tl = tl;
            continue;
          }
          // ---- y, loss and gy of the rows of this quadrant ----
          float* sy = sY + row_t * (NSUB * 2);
          if (sub != 0) {
            sy[(sub - 1) * 2 + 0] = ydot0;
            sy[(sub - 1) * 2 + 1] = ydot1;
          }
          ptx::named_bar_sync(1 + q, NSUB * 32);
          if (sub == 0) {
            float g0 = 0.f, g1 = 0.f;      // zero on pad / invalid rows
            if (valid && n_row < p.n) {
#pragma unroll
              for (int u = 0; u < NSUB - 1; ++u) {
                ydot0 += sy[u * 2 + 0];
                ydot1 += sy[u * 2 + 1];
              }
              const size_t yi = (size_t(ui.task) * p.n + n_row) * p.o;
              const float y0 = ydot0 + __ldg(p.bL + size_t(wt) * p.o);
              const float y1 = p.o > 1 ? ydot1 + __ldg(p.bL + size_t(wt) * p.o + 1) : 0.f;
              p.y[yi] = y0;
              if (p.o > 1) p.y[yi + 1] = y1;
              const float d0 = y0 - gt0;
              g0 = 2.f * p.loss_weight * d0;
              lsum = fmaf(d0, d0, lsum);
              if (p.o > 1) {
                const float d1 = y1 - gt1;
                g1 = 2.f * p.loss_weight * d1;
                lsum = fmaf(d1, d1, lsum);
              }
              if (p.gy) {
                p.gy[yi] = g0;
                if (p.o > 1) p.gy[yi + 1] = g1;
              }
            }
            sy[(NSUB - 1) * 2 + 0] = g0;
            sy[(NSUB - 1) * 2 + 1] = g1;
          }
          ptx::named_bar_sync(1 + q, NSUB * 32);
          const float g0 = sy[(NSUB - 1) * 2 + 0], g1 = sy[(NSUB - 1) * 2 + 1];
          // ---- top step (mlp_fused_bwd.cu, fuse_top) on the tile the forward has just written ----
          //   zbar_L = (sum_i gy_i WL_i) * w0 cos(theta_L),  dWL_i = sum_rows gy_i sin(theta_L),  dbL_i = sum_rows gy_i
          // in COLUMN layout: the lane owns columns 2 lane, 2 lane + 1 of the warp's slice, gy of row r sits in lane r
          if (sub == 0) {
            float r0 = g0, r1 = g1;
#pragma unroll
            for (int m = 16; m >= 1; m >>= 1) {
              r0 += __shfl_xor_sync(0xffffffffu, r0, m);
              r1 += __shfl_xor_sync(0xffffffffu, r1, m);
            }
            dbl0 += r0;
            dbl1 += r1;
          }
          const uint32_t slice = ptx::smem_u32(sA) + uint32_t(tl) * A_TILE + uint32_t(sub) * A_CHUNK + uint32_t(q) * (32 * 128);
          uint32_t u[32];
#pragma unroll
          for (int r = 0; r < 32; ++r)       // row & 7 == r & 7: the slice starts at a multiple of 8
            u[r] = valid ? ptx::ld_shared_u32(slice + uint32_t(r) * 128u + ((unit16 ^ uint32_t(r & 7)) << 4) + lane_off) : 0u;
          auto top_rows = [&](auto o_tag) {
            constexpr int O = decltype(o_tag)::value;
#pragma unroll
            for (int rb = 0; rb < 32; rb += 8) {
              float ga[8], gb[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                ga[i] = __shfl_sync(0xffffffffu, g0, rb + i);
                gb[i] = O > 1 ? __shfl_sync(0xffffffffu, g1, rb + i) : 0.f;
              }
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                float s0, s1, c0, c1;
                sgnsine_unpack(u[rb + i], s0, s1, c0, c1);
                float z0 = ga[i] * w00, z1 = ga[i] * w01;
                if (O > 1) { z0 = fmaf(gb[i], w10, z0); z1 = fmaf(gb[i], w11, z1); }
                z0 *= c0;
                z1 *= c1;
                dwl00 = fmaf(ga[i], s0, dwl00);
                dwl01 = fmaf(ga[i], s1, dwl01);
                if (O > 1) {
                  dwl10 = fmaf(gb[i], s0, dwl10);
                  dwl11 = fmaf(gb[i], s1, dwl11);
                }
                ptx::st_shared_u32(slice + uint32_t(rb + i) * 128u + ((unit16 ^ uint32_t(i)) << 4) + lane_off,
                                   sgnsine_flip(pack_bf16(z0, z1), u[rb + i]));
              }
            }
          };
          if (p.o > 1) top_rows(std::integral_constant<int, 2>());
          else top_rows(std::integral_constant<int, 1>());
          ptx::fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            ptx::mbar_arrive_leader(&a_ready[tl]);
            // the loader TMA-loads this unit's stash tiles back from global memory: every store of this warp has
            // landed there before it hears that the top step is done
            ptx::bulk_wait_all();
            ptx::mbar_arrive(&written[tl]);
          }
        }
      }
      // ---------------- chain steps L-1..1 and the bottom pass (mlp_fused_bwd.cu) ----------------
      for (int l = NH - 1; l >= 0; --l) {
        const bool bottom = (l == 0);
        for (int tl = 0; tl < ui.ntile; ++tl) {
          const bool valid = ui.valid[tl];
          const uint32_t a_row = eo.a_row + uint32_t(tl) * A_TILE;
          const uint32_t taddr = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(tl * 256 + colw);
          // bottom: this row's coordinates (L2: the forward read them) and the lane's first-layer weights, loaded
          // before the waits
          float xr[4] = {0.f, 0.f, 0.f, 0.f};
          float4 wa = make_float4(0.f, 0.f, 0.f, 0.f), wb = wa;
          float ba = 0.f, bb = 0.f;
          if (bottom) {
            row_coords(p, ui, tl, row_t, xr);
            first_weights(p, wt, colw + 2 * lane, wa, wb, ba, bb);
          }
          float va[PW], vb[PW];
          ptx::mbar_wait(&acc_full[tl], (accph >> tl) & 1u);
          accph ^= 1u << tl;
          ptx::tc_fence_after();
          ptx::tmem_ld<PW>(taddr, reinterpret_cast<uint32_t*>(va));
          // this warp's chunk of the stash tile is in the A tile (bottom: the tile may be rewritten)
          ptx::mbar_wait(&c_full[tl * 4 + sub], (cph >> tl) & 1u);
          cph ^= 1u << tl;
#pragma unroll
          for (int pc = 0; pc < NPIECE; ++pc) {
            float* v = (pc & 1) ? vb : va;
            ptx::tmem_wait_ld();
            if (pc + 1 < NPIECE)
              ptx::tmem_ld<PW>(taddr + uint32_t((pc + 1) * PW), reinterpret_cast<uint32_t*>((pc & 1) ? va : vb));
            const uint32_t s0 = a_row + (uint32_t((2 * pc) ^ eo.row7) << 4), s1 = a_row + (uint32_t((2 * pc + 1) ^ eo.row7) << 4);
            uint32_t pk[8];
            if (!bottom) {
              uint32_t cw[8];
              ptx::ld_shared_v4(s0, cw[0], cw[1], cw[2], cw[3]);
              ptx::ld_shared_v4(s1, cw[4], cw[5], cw[6], cw[7]);
#pragma unroll
              for (int j = 0; j < 8; ++j) {     // the tile holds the layer's signed sine: cos = +-sqrt(1 - sin^2)
                float h0, h1, c0, c1;
                sgnsine_unpack(cw[j], h0, h1, c0, c1);
                pk[j] = sgnsine_flip(pack_bf16(v[2 * j] * c0, v[2 * j + 1] * c1), cw[j]);
              }
            } else {
#pragma unroll
              for (int j = 0; j < 8; ++j) pk[j] = pack_bf16(v[2 * j], v[2 * j + 1]);
            }
            ptx::st_shared_v4(s0, pk[0], pk[1], pk[2], pk[3]);
            ptx::st_shared_v4(s1, pk[4], pk[5], pk[6], pk[7]);
          }
          ptx::tc_fence_before();
          if (bottom) {
            // column pass over this warp's slice (hbar_0 in bf16, just written): times cos(theta_0) from the
            // coordinates, db_0 and dW_0 sums; rows behind the task's padded extent contribute nothing
            __syncwarp();
            if (valid) {
              const uint32_t slice = ptx::smem_u32(sA) + uint32_t(tl) * A_TILE + uint32_t(sub) * A_CHUNK + uint32_t(q) * (32 * 128);
              float2* acc2 = reinterpret_cast<float2*>(my_sum) + lane;
              if (p.d == 1) bottom_pass<1, false>(slice, lane, xr[0], xr[1], xr[2], xr[3], wa, wb, ba, bb, acc2, 1);
              else if (p.d == 2) bottom_pass<2, false>(slice, lane, xr[0], xr[1], xr[2], xr[3], wa, wb, ba, bb, acc2, 1);
              else if (p.d == 3) bottom_pass<3, false>(slice, lane, xr[0], xr[1], xr[2], xr[3], wa, wb, ba, bb, acc2, 1);
              else bottom_pass<4, false>(slice, lane, xr[0], xr[1], xr[2], xr[3], wa, wb, ba, bb, acc2, 1);
            }
          } else {
            ptx::fence_proxy_async();         // the tile is read by the next MMA and by the loader's TMA store
          }
          __syncwarp();
          if (lane == 0) {
            ptx::mbar_arrive(&written[tl]);   // loader: store the adjoint / free the tile
            if (!bottom) ptx::mbar_arrive_leader(&a_ready[tl]);
          }
        }
      }
    }
    if (cur_task >= 0) flush(cur_task);
    if (p.loss_acc) {                        // one atomic per CTA: w * sum over its rows of (y - gt)^2
      if (sub == 0) {
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) lsum += __shfl_xor_sync(0xffffffffu, lsum, m);
        if (lane == 0) sLoss[q] = lsum;
      }
      ptx::named_bar_sync(15, EPI_WARPS * 32);
      if (tid_e == 0) atomicAdd(p.loss_acc, p.loss_weight * (sLoss[0] + sLoss[1] + sLoss[2] + sLoss[3]));
    }
    if (lane == 0) ptx::bulk_wait_all();
  }

  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();           // neither CTA leaves (or frees TMEM) while the other may still touch it
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc_pair(tmem_base, 512);
  }
}

}  // namespace

cudaError_t launch_mlp_fused_step(const MlpStepParams& p, int num_sms, cudaStream_t stream) {
  const int tiles_task = (p.f.rows_per_task + 255) / 256;
  const int n_units = ((tiles_task + 1) / 2) * p.f.tasks;
  int n_cl = num_sms / 2;
  if (n_cl > n_units) n_cl = n_units;
  if (n_cl < 1) n_cl = 1;
  SIREN_ENSURE_SMEM(mlp_fused_step_kernel, SMEM_STEP);
  mlp_fused_step_kernel<<<2 * n_cl, kThreads, SMEM_STEP, stream>>>(p);
  return cudaGetLastError();
}

}  // namespace siren
