// Fused input-gradient chain of the hidden sine layers on CTA PAIRS (cluster of 2, tcgen05 cta_group::2);
// bf16 mode, value stream, <= 8 hidden layers (d_in > 4: dW_0 / db_0 are items of the weight-gradient kernel).  Backward counterpart of mlp_fused_pair.cu.
//
//   in    gy                loss gradient w.r.t. the network output (fuse_top), or
//         zbar_L            adjoint of the top sine layer as written by last_bwd             [R, 256] bf16
//         h_l               stash of the fused forward: the signed sine of layer l (common.cuh) [R, 256] fp16
//                           (l >= 1; l = 0 only for d_in > 4 -- for narrow inputs theta_0 is recomputed from x)
//         w0 W_l^T          transposed hidden weights, pre-scaled by w0 (prep_weights)       bf16
//   out   zbar_L = (gy WL) * w0 cos(theta_L),  dWL = gy^T sin(theta_L),  dbL                 (fuse_top)
//         zbar_l = (zbar_{l+1} w0 W_{l+1}) * cos(theta_l)   for l = L-1 .. 1  (wgrad operands; l = 0 on request)
//         db_0   = column sums of zbar_0,  dW_0 = zbar_0^T x                                 (d_in <= 4)
//         (db_l, l >= 1, are column sums the weight-gradient kernel takes from the adjoint blocks it stages)
//   (autograd of FCBlock's [BatchLinear, Sine] chain + outermost linear, modules.py:92-97 / training.py:91)
//
// A pair of SMs carries two 256-row tiles (X, Y) down the layers; each CTA owns 128 rows of each tile.
// The adjoint tile is the MMA's A operand and lives in shared memory; between layers it never travels
// through HBM as an operand (the per-layer kernels re-read it: one plane per layer saved).  Per layer:
//   MMA      D = zbar_{l+1} W_{l+1}   (cta_group::2, M = 256, B = this CTA's half of W^T, resident per layer)
//   loader   one thread owns every bulk copy on the A tiles: once the MMA has drained a tile it TMA-loads the
//            layer's phase tile INTO it (prefetched to L2 a step earlier); once the epilogue has rewritten the
//            tile it TMA-stores the adjoint for the weight-gradient kernel
//   epilogue zbar_l = D * cos(theta_l), written back in place over theta_l (each thread overwrites exactly
//            what it read).  The two MMA-less ends of the chain run in COLUMN layout (the lane owns two adjacent
//            columns of the warp's 32 x 64 slice and walks its rows): the top step turns the phase tile into
//            zbar_L and keeps the dWL sums in registers (no cross-lane reduction at all); the bottom step of a
//            narrow first layer multiplies by cos(theta_0) recomputed from the coordinates and sums db_0 / dW_0
// X and Y are skewed by half a step so the tensor core and the loads hide behind the epilogue.
#include "common.cuh"
#include "ptx.cuh"
#include "simt.h"
#include "mlp_fused_parts.cuh"

#include <type_traits>

namespace siren {

namespace {

constexpr int MAXL = MAX_FUSED_HIDDEN_SMEM;
constexpr int NSLOT = 4;                        // weight chunk slots (ring)
constexpr int NSUM = 1 + 4;                     // partial-sum rows per warp: db_0, dW0[:, k] (<= 4); dWL[i, :] reuses rows 0, 1
constexpr int SUM_BYTES = EPI_WARPS * NSUM * 64 * 4;   // 20 KB: [16 warps][NSUM][64 columns]
// per-row inputs of a unit, staged one unit ahead by cp.async (double-buffered by unit parity):
//   coordinates [2 parities][2 tiles][128 rows][4 floats], loss gradient [2][2][128][2 floats]
constexpr int XIN_BYTES = 2 * 2 * TILE_M * 4 * 4;      // 8 KB
constexpr int GIN_BYTES = 2 * 2 * TILE_M * 2 * 4;      // 4 KB
constexpr int MISC = 1024;
constexpr int SMEM_BWD = 2 * A_TILE + NSLOT * B_SLOT + SUM_BYTES + XIN_BYTES + GIN_BYTES + MISC + 1024;
static_assert(SMEM_BWD <= 232448, "shared memory budget");

struct UnitInfo {
  int task, ntile;
  int row0[2];
  bool valid[2];
};
// `step` counts this pair's units in the order it walks them: DESCENDING through its range [u0, u1).  The forward
// walked the same range ascending, so the phase tiles of the units the chain starts with are the ones the forward
// wrote last -- still in L2.
__device__ __forceinline__ UnitInfo unit_info(const MlpBwdParams& p, int step, int rank, int u0, int u1) {
  const int unit = u0 + u1 - 1 - step;
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

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
    mlp_fused_bwd_kernel(const __grid_constant__ MlpBwdParams p) {
  constexpr uint32_t IDESC = ptx::umma_idesc_bf16(256, 256, 0, 0);
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;                               // [2 tiles][4 chunks][128][128 B]
  uint8_t* sB = sA + 2 * A_TILE;                    // [NSLOT][128][128 B]
  float* sSum = reinterpret_cast<float*>(sB + NSLOT * B_SLOT);   // [16 warps][NSUM][64]
  float* sXin = sSum + EPI_WARPS * NSUM * 64;                    // [2][2][128][4]
  float* sGin = sXin + XIN_BYTES / 4;                            // [2][2][128][2]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sGin + GIN_BYTES / 4);
  uint64_t* b_full = bars;                          // [NKC]  leader's: both halves of a weight chunk landed
  uint64_t* b_empty = bars + NSLOT;                 // [NKC]  multicast commit
  uint64_t* acc_full = bars + 2 * NSLOT;            // [2]    multicast commit: accumulator ready, A tile drained
  uint64_t* a_ready = acc_full + 2;                 // [2]    leader's: 16 warps x 2 CTAs wrote zbar_l into the A tile
  uint64_t* a_load = a_ready + 2;                   // [2]    leader's: both halves of the top adjoint tile landed
  uint64_t* c_full = a_load + 2;                    // [2][4] local: K chunk kc of the phase tile landed in the A tile
                                                    //        (a warp waits for ITS chunk only: load and epilogue overlap)
  uint64_t* written = c_full + 8;                   // [2]    local: the 16 epilogue warps are done with the A tile
  uint64_t* in_full = written + 2;                  // [2]    local: the unit's row inputs (parity slot) have landed
  uint64_t* in_empty = in_full + 2;                 // [2]    local: the 16 epilogue warps are done with the slot
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(in_empty + 2);
  float* sDbL = reinterpret_cast<float*>(tmem_slot + 4);      // [4 quadrants][2]  sum of gy, per sub == 0 warp

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
      ptx::prefetch_tmap(&p.tmWt[l]);
      ptx::prefetch_tmap(&p.tmC[l]);
    }
    ptx::prefetch_tmap(&p.tmTop);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < NSLOT; ++i) {
      ptx::mbar_init(&b_full[i], 1);
      ptx::mbar_init(&b_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&acc_full[i], 1);
      ptx::mbar_init(&a_ready[i], 2 * EPI_WARPS);
      ptx::mbar_init(&a_load[i], 1);
      for (int kc = 0; kc < 4; ++kc) ptx::mbar_init(&c_full[i * 4 + kc], 1);
      ptx::mbar_init(&written[i], EPI_WARPS);
      ptx::mbar_init(&in_full[i], 32);
      ptx::mbar_init(&in_empty[i], EPI_WARPS);
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
  ptx::cluster_sync();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const bool trace = p.dbg != nullptr && blockIdx.x == 0;
#define TRACE(u_, l_, k_) do { if (trace && lane == 0 && (u_) - u0 < 3) p.dbg[(((u_) - u0) * 8 + (l_)) * 8 + (k_)] = clock64(); } while (0)
  if (trace && threadIdx.x == 0) p.dbg[0] = clock64();
  if (p.dbg != nullptr && threadIdx.x == 0) {      // per-CTA start (and, at the end, finish) time: spread across the grid
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    p.dbg[2048 + 2 * blockIdx.x] = t;
  }

  // Register reallocation between the warp groups: the four control warps give back 40 registers each,
  // the epilogue warps get 104 (128 x 56 + 512 x 104 stays inside the 640 x 96 the CTA was launched with)
  if (warp < 4) {
  ptx::setmaxnreg_dec<56>();
  if (warp == 0) {
    // ===================== weight producer (both CTAs: each loads its half of W^T's rows) =====================
    if (lane == 0) {
      // ring of NSLOT chunk slots, one more than a layer has chunks: the first chunk of the next layer is
      // already on chip when X gets there, the others follow as Y releases the current layer's
      uint32_t seq = 0;
      for (int un = u0; un < u1; ++un) {
        const UnitInfo ui = unit_info(p, un, rank, u0, u1);
        const int wrow = (p.per_task ? ui.task : 0) * H + rank * 128;
        for (int l = NH; l >= 1; --l)
          for (int kc = 0; kc < NKC; ++kc, ++seq) {
            const uint32_t sl = seq % NSLOT, ph = (seq / NSLOT) & 1u;
            ptx::mbar_wait(&b_empty[sl], ph ^ 1u);
            if (leader) ptx::mbar_arrive_expect_tx(&b_full[sl], 2 * B_SLOT);
            ptx::tma_load_2d_pair(sB + sl * B_SLOT, &p.tmWt[l - 1], &b_full[sl], kc * KCHUNK, wrow);
          }
      }
      // the last multicast commits have landed in this CTA before it may exit
      for (int i = 0; i < NSLOT; ++i, ++seq) ptx::mbar_wait(&b_empty[seq % NSLOT], ((seq / NSLOT) & 1u) ^ 1u);
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (leader) {
      uint32_t seq0 = 0;             // ring position of the layer's first chunk
      uint32_t rnd = 0u;             // bit tl: phase of a_ready[tl]
      uint32_t lph = 0u;             // bit tl: phase of a_load[tl]
      for (int un = u0; un < u1; ++un) {
        const UnitInfo ui = unit_info(p, un, rank, u0, u1);
        for (int l = NH; l >= 1; --l, seq0 += NKC) {
          for (int tl = 0; tl < ui.ntile; ++tl) {
            if (l == NH && !p.fuse_top) {      // first layer of the unit: the A tile comes from HBM as it is
              ptx::mbar_wait(&a_load[tl], (lph >> tl) & 1u);
              lph ^= 1u << tl;
            } else {
              ptx::mbar_wait_cluster(&a_ready[tl], (rnd >> tl) & 1u);
              rnd ^= 1u << tl;
            }
            TRACE(un, l, 512 + tl * 2 + 0);
            for (int kc = 0; kc < NKC; ++kc) {
              const uint32_t sl = (seq0 + kc) % NSLOT;
              if (tl == 0) ptx::mbar_wait(&b_full[sl], ((seq0 + kc) / NSLOT) & 1u);
              ptx::tc_fence_after();
              if (lane == 0) {
                const uint32_t a_addr = ptx::smem_u32(sA + tl * A_TILE + kc * A_CHUNK);
                const uint32_t b_addr = ptx::smem_u32(sB + sl * B_SLOT);
#pragma unroll
                for (int ks = 0; ks < 4; ++ks)
                  ptx::umma_bf16_pair(tmem_base + uint32_t(tl * 256), ptx::umma_smem_desc(a_addr + ks * 32, 16, 1024),
                                      ptx::umma_smem_desc(b_addr + ks * 32, 16, 1024), IDESC, (kc | ks) ? 1u : 0u);
                if (tl == ui.ntile - 1) ptx::umma_commit_pair(&b_empty[sl], 3);
              }
              __syncwarp();
            }
            if (lane == 0) ptx::umma_commit_pair(&acc_full[tl], 3);
            __syncwarp();
            TRACE(un, l, 512 + tl * 2 + 1);
          }
        }
      }
    }
  } else if (warp == 2) {
    // ===================== row-input loader (both CTAs): gy and coordinates of this CTA's rows, one unit ahead =====
    // A global load issued by an epilogue warp where the value is consumed costs the loaded-HBM latency (3-9k cycles
    // in the clock64 trace, four times per unit), and fetching a unit ahead into registers does not survive the
    // register allocator (the values are spilled at once, which waits for them).  So this otherwise idle warp copies
    // them with cp.async into a parity slot of shared memory and the epilogue reads them from there.
    const uint32_t xin = ptx::smem_u32(sXin), gin = ptx::smem_u32(sGin);
    uint32_t k = 0;
    for (int un = u0; un < u1; ++un, ++k) {
      const uint32_t par = k & 1u;
      ptx::mbar_wait(&in_empty[par], ((k >> 1) & 1u) ^ 1u);
      const UnitInfo u = unit_info(p, un, rank, u0, u1);
      for (int i = lane; i < 2 * TILE_M; i += 32) {
        const int t = i >> 7, r = i & (TILE_M - 1);
        const int n_row = u.row0[t] + r - u.task * p.rows_per_task;
        const bool live = t < u.ntile && u.valid[t] && n_row < p.n;
        const size_t ri = size_t(u.task) * p.n + (live ? n_row : 0);
        const uint32_t xd = xin + ((par * 2 + t) * TILE_M + r) * 16u, gd = gin + ((par * 2 + t) * TILE_M + r) * 8u;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const bool on = live && p.l0_from_x && c < p.d;
          ptx::cp_async_4(xd + 4u * c, p.x + ri * p.d + (on ? c : 0), on ? 4u : 0u);
        }
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          const bool on = live && p.fuse_top && c < p.o;
          ptx::cp_async_4(gd + 4u * c, on ? static_cast<const void*>(p.gy + ri * p.o + c) : static_cast<const void*>(p.x), on ? 4u : 0u);
        }
      }
      ptx::cp_async_mbar_arrive_noinc(&in_full[par]);
    }
  } else if (warp == 3) {
    // ===================== tile loader (both CTAs): top adjoint / phase tiles, then a phase tile per layer ==========
    if (lane == 0) {
      // This thread owns every bulk copy that touches the A tiles, so it alone knows when a tile may be
      // refilled.  In the order the epilogue walks the tiles, k = 0, 1, 2, ...:
      //   load c(k)     as soon as MMA(k) has read the tile (acc_full) and the store of the tile's previous
      //                 contents has drained
      //   retire(k-1)   once the epilogue has written tile k-1 (written): store the adjoint it holds; if it was
      //                 a bottom-layer tile, start the next unit's top adjoint load into it
      // Retiring k-1 only AFTER the load for k is under way keeps the phase-tile loads off the critical path.
      uint32_t accph = 0u, wrph = 0u;
      auto top_load = [&](const UnitInfo& ui, int tl) {
        if (p.fuse_top) {
          // the epilogue warps read the top layer's phase themselves (global memory, coalesced in their column
          // layout): nothing is loaded into the tile, they only need to know that it may be rewritten
          for (int kc = 0; kc < 4; ++kc) ptx::mbar_arrive(&c_full[tl * 4 + kc]);
        } else {                     // the top adjoint tile, straight for the pair's MMA
          if (leader) ptx::mbar_arrive_expect_tx(&a_load[tl], 2 * A_TILE);
          for (int kc = 0; kc < 4; ++kc)
            ptx::tma_load_2d_pair(sA + tl * A_TILE + kc * A_CHUNK, &p.tmTop, &a_load[tl], kc * KCHUNK, ui.row0[tl]);
        }
        if (NH - 1 > 0 || !p.l0_from_x)
          for (int kc = 0; kc < 4; ++kc) ptx::tma_prefetch_2d(&p.tmC[NH - 1], kc * KCHUNK, ui.row0[tl]);
      };
      struct Pending {
        int un, l, tl, row0;
        bool valid;
      } pd = {-1, 0, 0, 0, false};
      auto retire = [&]() {
        if (pd.un < 0) return;
        ptx::mbar_wait(&written[pd.tl], (wrph >> pd.tl) & 1u);
        wrph ^= 1u << pd.tl;
        const bool stores = pd.valid && (pd.l > 0 || p.store_adj0);
        if (stores) {
          for (int kc = 0; kc < 4; ++kc)
            ptx::tma_store_2d(&p.tmAdj[pd.l], sA + pd.tl * A_TILE + kc * A_CHUNK, kc * KCHUNK, pd.row0);
          ptx::bulk_commit();
        }
        if (pd.l == 0 && pd.un + 1 < u1) {         // bottom layer: the tile is free for the next unit
          const UnitInfo nx = unit_info(p, pd.un + 1, rank, u0, u1);
          if (pd.tl < nx.ntile) {
            if (stores) ptx::bulk_wait_read<0>();
            top_load(nx, pd.tl);
          }
        }
        pd.un = -1;
      };
      if (u0 < u1) {
        const UnitInfo ui = unit_info(p, u0, rank, u0, u1);
        for (int tl = 0; tl < ui.ntile; ++tl) top_load(ui, tl);
      }
      for (int un = u0; un < u1; ++un) {
        const UnitInfo ui = unit_info(p, un, rank, u0, u1);
        if (un > u0) {               // a tile the previous (single-tile) unit did not use: nobody retires it
          const UnitInfo pv = unit_info(p, un - 1, rank, u0, u1);
          for (int tl = pv.ntile; tl < ui.ntile; ++tl) {
            ptx::bulk_wait_read<0>();
            top_load(ui, tl);
          }
        }
        if (p.fuse_top)              // top step: the epilogue turns the phase tile into the top adjoint, no load here
          for (int tl = 0; tl < ui.ntile; ++tl) {
            retire();
            pd.un = un; pd.l = NH; pd.tl = tl; pd.row0 = ui.row0[tl]; pd.valid = ui.valid[tl];
          }
        for (int l = NH - 1; l >= 0; --l)
          for (int tl = 0; tl < ui.ntile; ++tl) {
            if (pd.un >= 0 && pd.tl == tl) retire();                // single-tile unit: same buffer, store it first
            ptx::mbar_wait(&acc_full[tl], (accph >> tl) & 1u);      // the MMA has read the A tile (both CTAs')
            accph ^= 1u << tl;
            TRACE(un, l + 1, 1024 + tl * 2 + 0);
            ptx::bulk_wait_read<0>();                               // ... and so has the last store issued from it
            TRACE(un, l + 1, 1024 + tl * 2 + 1);
            if (l == 0 && p.l0_from_x) {
              // narrow first layer: no phase plane -- the epilogue only needs to know that the tile may be rewritten
              for (int kc = 0; kc < 4; ++kc) ptx::mbar_arrive(&c_full[tl * 4 + kc]);
            } else {
              for (int kc = 0; kc < 4; ++kc) {
                ptx::mbar_arrive_expect_tx(&c_full[tl * 4 + kc], A_CHUNK);
                ptx::tma_load_2d(sA + tl * A_TILE + kc * A_CHUNK, &p.tmC[l], &c_full[tl * 4 + kc], kc * KCHUNK, ui.row0[tl]);
              }
            }
            // what this tile needs next goes to L2 now: the phase tile one layer down, or the next unit's top tile
            if (l > 1 || (l == 1 && !p.l0_from_x)) {
              for (int kc = 0; kc < 4; ++kc) ptx::tma_prefetch_2d(&p.tmC[l - 1], kc * KCHUNK, ui.row0[tl]);
            } else if (l > 0) {
              // layer 0 comes from the coordinates: nothing to pull
            } else if (un + 1 < u1) {
              const UnitInfo nx = unit_info(p, un + 1, rank, u0, u1);
              if (tl < nx.ntile)
                for (int kc = 0; kc < 4; ++kc) ptx::tma_prefetch_2d(&p.tmTop, kc * KCHUNK, nx.row0[tl]);
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
    const int q = warp & 3;
    const int sub = e >> 2;
    const int tid_e = threadIdx.x - 128;
    const int row_t = q * 32 + lane;
    const int row7 = row_t & 7;
    const float w0 = p.w0;
    const int colw = sub * 64;
    const uint32_t a_row0 = ptx::smem_u32(sA) + uint32_t(sub) * A_CHUNK + uint32_t(row_t) * 128u;
    // this warp's private partial sums [NSUM][64] over the warp's 64 columns: row 0 = db_0, rows 1 .. d = dW0[:, k]
    // (narrow first layer only); the dWL[i, :] sums live in registers and pass through rows 0, 1 when flushed.
    // Private means plain read-modify-write (shared fp32 atomics are CAS loops).
    float* my_sum = sSum + e * (NSUM * 64);
    uint32_t accph = 0u, cph = 0u;
    int cur_wt = -1;
    const int n_db = p.l0_from_x ? 1 : 0;
    const int n_dw0 = p.l0_from_x ? p.d : 0;
    const int row_dw0 = n_db;
    const int n_dwl = p.fuse_top ? p.o : 0;
    float dbl0 = 0.f, dbl1 = 0.f;           // sum of gy over this warp's rows (sub == 0 warps, every lane the same)
    // dWL[i, colw + 2 lane + {0, 1}] summed over this warp's rows, all tiles and units of the current weight set:
    // the top step runs in column layout, so these sums never cross lanes
    float2 dwl0 = make_float2(0.f, 0.f), dwl1 = dwl0;
    const uint32_t lane_off = uint32_t(lane & 3) * 4u, unit16 = uint32_t(lane >> 2);

    // partial sums -> global: the four quadrant warps of a column chunk are combined here, then ONE atomic
    // per element and CTA (same-address atomics serialise in L2)
    auto flush = [&](int wt) {
      ptx::named_bar_sync(15, EPI_WARPS * 32);
      for (int i = tid_e; i < (n_db + n_dw0) * H; i += EPI_WARPS * 32) {
        const int r = i / H, col = i - r * H;
        float* s = sSum + ((col >> 6) * 4) * (NSUM * 64) + r * 64 + (col & 63);
        const float tot = s[0] + s[NSUM * 64] + s[2 * NSUM * 64] + s[3 * NSUM * 64];
        s[0] = s[NSUM * 64] = s[2 * NSUM * 64] = s[3 * NSUM * 64] = 0.f;
        if (r < n_db) atomicAdd(p.db[0] + size_t(wt) * H + col, tot);
        else atomicAdd(p.dW0 + (size_t(wt) * H + col) * p.d + (r - n_db), tot);
      }
      if (p.fuse_top) {
        // second pass through the same rows: the dWL sums the warps kept in registers
        ptx::named_bar_sync(15, EPI_WARPS * 32);
        float2* d0 = reinterpret_cast<float2*>(my_sum) + lane;
        d0[0] = dwl0;
        if (p.o > 1) d0[32] = dwl1;
        if (sub == 0 && lane == 0) {
          sDbL[q * 2 + 0] = dbl0;
          sDbL[q * 2 + 1] = dbl1;
        }
        dwl0 = dwl1 = make_float2(0.f, 0.f);
        dbl0 = dbl1 = 0.f;
        ptx::named_bar_sync(15, EPI_WARPS * 32);
        for (int i = tid_e; i < n_dwl * H; i += EPI_WARPS * 32) {
          const int r = i / H, col = i - r * H;
          float* s = sSum + ((col >> 6) * 4) * (NSUM * 64) + r * 64 + (col & 63);
          const float tot = s[0] + s[NSUM * 64] + s[2 * NSUM * 64] + s[3 * NSUM * 64];
          s[0] = s[NSUM * 64] = s[2 * NSUM * 64] = s[3 * NSUM * 64] = 0.f;
          atomicAdd(p.dWL + (size_t(wt) * p.o + r) * H + col, tot);
        }
        if (tid_e < p.o)
          atomicAdd(p.dbL + size_t(wt) * p.o + tid_e, sDbL[tid_e] + sDbL[2 + tid_e] + sDbL[4 + tid_e] + sDbL[6 + tid_e]);
      }
      ptx::named_bar_sync(15, EPI_WARPS * 32);
    };

    // Per-row inputs of this thread's row in tiles X / Y -- the loss gradient (top step) and the coordinates (bottom
    // step) -- come from the parity slot the row-input loader (warp 2) filled one unit ahead.
    const uint32_t xin_row = ptx::smem_u32(sXin) + uint32_t(row_t) * 16u, gin_row = ptx::smem_u32(sGin) + uint32_t(row_t) * 8u;
    uint32_t kin = 0;                          // units this warp has started (parity slot and phase of in_full)
    float2 wl0 = make_float2(0.f, 0.f), wl1 = wl0;         // w0 WL[i, colw + 2 lane + {0, 1}] of the current weight set

    for (int un = u0; un < u1; ++un) {
      const UnitInfo ui = unit_info(p, un, rank, u0, u1);
      const int wt = p.per_task ? ui.task : 0;
      const uint32_t par = kin & 1u;
      ptx::mbar_wait(&in_full[par], (kin >> 1) & 1u);      // this unit's gy / coordinates are in shared memory
      ++kin;
      if (wt != cur_wt) {
        if (cur_wt >= 0) flush(cur_wt);
        cur_wt = wt;
        if (p.fuse_top) {
          const float2 wr0 = __ldg(reinterpret_cast<const float2*>(p.WL + (size_t(wt) * p.o) * H + colw) + lane);
          wl0 = make_float2(w0 * wr0.x, w0 * wr0.y);
          if (p.o > 1) {
            const float2 wr1 = __ldg(reinterpret_cast<const float2*>(p.WL + (size_t(wt) * p.o + 1) * H + colw) + lane);
            wl1 = make_float2(w0 * wr1.x, w0 * wr1.y);
          }
        }
      }
      // ---------------- top step (fuse_top): loss gradient -> adjoint of the top sine layer ----------------
      //   zbar_L = (sum_i gy_i WL_i) * w0 cos(phase),  dWL_i = sum_rows gy_i sin(phase),  dbL_i = sum_rows gy_i
      // No accumulator is involved, so the warp walks its [32 rows x 64 columns] slice of the phase tile in COLUMN
      // layout: the lane owns columns 2 lane, 2 lane + 1 (one 32-bit word per row, conflict-free), gy of row r
      // sits in lane r (one shuffle per row and output), w0 WL of the two columns in registers.
      if (p.fuse_top)
        for (int tl = 0; tl < ui.ntile; ++tl) {
          const int row0 = ui.row0[tl];
          const bool valid = ui.valid[tl];
          float g0, g1;                     // zero on pad / invalid rows
          asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(g0), "=f"(g1) : "r"(gin_row + (par * 2u + uint32_t(tl)) * (TILE_M * 8u)));
          if (p.dc.mask) {       // gy is the adjoint of the data-consistent output: this row's share keep = 1 - mask pull
            const int n_row = row0 + row_t - ui.task * p.rows_per_task;
            if (valid && n_row < p.n) {
              g0 *= 1.f - p.dc.pull * __ldg(p.dc.mask + dc_index(p.dc.cf, ui.task, n_row, 0, p.n, p.o));
              if (p.o > 1) g1 *= 1.f - p.dc.pull * __ldg(p.dc.mask + dc_index(p.dc.cf, ui.task, n_row, 1, p.n, p.o));
            }
          }
          if (sub == 0) {              // dbL = sum over rows of gy (each row counted once)
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
          // The top layer's phase, this lane's two columns of the warp's 32 rows, straight from the plane: in column
          // layout a row of the warp is ONE 128-byte line, so the loads are fully coalesced (the row layout of the MMA
          // steps is what forces those through TMA).  All 32 go out before the tile is even free, so the step does not
          // start with a TMA load into the tile that could only be issued once the previous unit had left it.
          uint32_t u[32];
          {
            const uint32_t* gph = p.phase_top + (size_t(row0) + size_t(q * 32)) * (H / 2) + (colw >> 1) + lane;
#pragma unroll
            for (int r = 0; r < 32; ++r) u[r] = valid ? __ldg(gph + size_t(r) * (H / 2)) : 0u;
          }
          ptx::mbar_wait(&c_full[tl * 4 + sub], (cph >> tl) & 1u);   // the tile may be rewritten (its last store has drained)
          cph ^= 1u << tl;
          if (e == 0) TRACE(un, NH + 1, tl * 4 + 1);
          // (one code copy per output count: with a single output the second gy shuffle and its three FMAs per
          //  row and column pair are not there at all)
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
              for (int i = 0; i < 8; ++i) {      // row & 7 == i
                float s0, s1, c0, c1;      // the top layer's signed sine: sin as it is, |cos| = sqrt(1 - sin^2)
                sgnsine_unpack(u[rb + i], s0, s1, c0, c1);
                const float2 s = make_float2(s0, s1), ga2 = make_float2(ga[i], ga[i]);
                float2 z = ptx::mul2(wl0, ga2);
                if (O > 1) z = ptx::fma2(wl1, make_float2(gb[i], gb[i]), z);
                z = ptx::mul2(z, make_float2(c0, c1));
                dwl0 = ptx::fma2(s, ga2, dwl0);
                if (O > 1) dwl1 = ptx::fma2(s, make_float2(gb[i], gb[i]), dwl1);
                ptx::st_shared_u32(slice + uint32_t(rb + i) * 128u + ((unit16 ^ uint32_t(i)) << 4) + lane_off,
                                   sgnsine_flip(pack_bf16(z.x, z.y), u[rb + i]));      // the cosine signs go onto the product
              }
            }
          };
          if (p.o > 1) top_rows(std::integral_constant<int, 2>());
          else top_rows(std::integral_constant<int, 1>());
          ptx::fence_proxy_async();
          __syncwarp();
          if (e == 0) TRACE(un, NH + 1, tl * 4 + 2);
          if (lane == 0) {
            ptx::mbar_arrive(&written[tl]);
            ptx::mbar_arrive_leader(&a_ready[tl]);
          }
        }
      for (int l = NH - 1; l >= 0; --l) {
        const bool bottom = (l == 0);
        const bool from_x = bottom && p.l0_from_x;      // no phase tile: cos(theta_0) from the coordinates, in the column pass
        const bool store = !bottom || p.store_adj0;
        for (int tl = 0; tl < ui.ntile; ++tl) {
          const int row0 = ui.row0[tl];
          const bool valid = ui.valid[tl];
          const uint32_t a_row = a_row0 + uint32_t(tl) * A_TILE;
          const uint32_t taddr = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(tl * 256 + colw);
          float x0 = 0.f, x1 = 0.f, x2 = 0.f, x3 = 0.f;
          if (from_x) {
            const float4 xv = ptx::ld_shared_f4(xin_row + (par * 2u + uint32_t(tl)) * (TILE_M * 16u));
            x0 = xv.x; x1 = xv.y; x2 = xv.z; x3 = xv.w;
          }
          // first-layer weights of this lane's two columns (bottom step): the loads go out before the waits, so the
          // column pass does not start with an exposed L1 / L2 round trip (9 % of the kernel's stall samples)
          float2 w2[4], b2 = make_float2(0.f, 0.f);       // (column 2 lane, column 2 lane + 1) of each coordinate
          for (int k = 0; k < 4; ++k) w2[k] = b2;
          if (from_x) {
            const float* wr = p.W0 + (size_t(wt) * H + colw + 2 * lane) * p.d;
            for (int k = 0; k < 4; ++k)
              if (k < p.d) w2[k] = make_float2(__ldg(wr + k), __ldg(wr + p.d + k));
            b2 = make_float2(__ldg(p.b0 + size_t(wt) * H + colw + 2 * lane), __ldg(p.b0 + size_t(wt) * H + colw + 2 * lane + 1));
          }
          float va[PW], vb[PW];
          ptx::mbar_wait(&acc_full[tl], (accph >> tl) & 1u);
          accph ^= 1u << tl;
          ptx::tc_fence_after();
          if (e == 0) TRACE(un, l + 1, tl * 4 + 0);
          ptx::tmem_ld<PW>(taddr, reinterpret_cast<uint32_t*>(va));
          // this warp's chunk of the phase tile is in the A tile (from_x: the tile may be rewritten, nothing was loaded)
          ptx::mbar_wait(&c_full[tl * 4 + sub], (cph >> tl) & 1u);
          cph ^= 1u << tl;
          if (e == 0) TRACE(un, l + 1, tl * 4 + 1);
#pragma unroll
          for (int pc = 0; pc < NPIECE; ++pc) {
            float* v = (pc & 1) ? vb : va;
            ptx::tmem_wait_ld();
            if (pc + 1 < NPIECE)
              ptx::tmem_ld<PW>(taddr + uint32_t((pc + 1) * PW), reinterpret_cast<uint32_t*>((pc & 1) ? va : vb));
            const uint32_t s0 = a_row + (uint32_t((2 * pc) ^ row7) << 4), s1 = a_row + (uint32_t((2 * pc + 1) ^ row7) << 4);
            uint32_t pk[8];
            if (!from_x) {
              uint32_t cw[8];
              ptx::ld_shared_v4(s0, cw[0], cw[1], cw[2], cw[3]);
              ptx::ld_shared_v4(s1, cw[4], cw[5], cw[6], cw[7]);
#pragma unroll
              for (int j = 0; j < 8; ++j) {     // the tile holds the layer's signed sine: cos = +-sqrt(1 - sin^2), one MUFU
                float h0, h1, c0, c1;           // (the accumulator already carries w0: the weights were pre-scaled)
                sgnsine_unpack(cw[j], h0, h1, c0, c1);
                const float2 z = ptx::mul2(make_float2(v[2 * j], v[2 * j + 1]), make_float2(c0, c1));
                pk[j] = sgnsine_flip(pack_bf16(z.x, z.y), cw[j]);
              }
            } else {
#pragma unroll
              for (int j = 0; j < 8; ++j) pk[j] = pack_bf16(v[2 * j], v[2 * j + 1]);
            }
            if (store || bottom) {
              ptx::st_shared_v4(s0, pk[0], pk[1], pk[2], pk[3]);
              ptx::st_shared_v4(s1, pk[4], pk[5], pk[6], pk[7]);
            }
          }
          ptx::tc_fence_before();
          if (from_x) {
            // Column pass over this warp's own [32 rows x 64 columns] slice (hbar_0 in bf16, just written): times
            // cos(theta_0) from the coordinates, db_0 and dW_0 sums; rows behind the task's padded extent (the
            // other CTA's half of an odd last tile) hold another task's numbers and contribute nothing.
            __syncwarp();
            if (e == 0) TRACE(un, l + 1, tl * 4 + 1);
            if (valid) {
              // w0-scaled, exactly as the forward forms them (w0 * W0 and w0 * b0 in fp32)
              for (int k = 0; k < 4; ++k) w2[k] = make_float2(w2[k].x * w0, w2[k].y * w0);
              b2 = make_float2(b2.x * w0, b2.y * w0);
              const uint32_t slice = ptx::smem_u32(sA) + uint32_t(tl) * A_TILE + uint32_t(sub) * A_CHUNK + uint32_t(q) * (32 * 128);
              float2* acc2 = reinterpret_cast<float2*>(my_sum) + lane;      // columns 2 lane, 2 lane + 1 of row 0
              if (p.store_adj0) {
                if (p.d == 1) bottom_pass<1, true>(slice, lane, x0, x1, x2, x3, w2, b2, acc2, row_dw0);
                else if (p.d == 2) bottom_pass<2, true>(slice, lane, x0, x1, x2, x3, w2, b2, acc2, row_dw0);
                else if (p.d == 3) bottom_pass<3, true>(slice, lane, x0, x1, x2, x3, w2, b2, acc2, row_dw0);
                else bottom_pass<4, true>(slice, lane, x0, x1, x2, x3, w2, b2, acc2, row_dw0);
              } else {
                if (p.d == 1) bottom_pass<1, false>(slice, lane, x0, x1, x2, x3, w2, b2, acc2, row_dw0);
                else if (p.d == 2) bottom_pass<2, false>(slice, lane, x0, x1, x2, x3, w2, b2, acc2, row_dw0);
                else if (p.d == 3) bottom_pass<3, false>(slice, lane, x0, x1, x2, x3, w2, b2, acc2, row_dw0);
                else bottom_pass<4, false>(slice, lane, x0, x1, x2, x3, w2, b2, acc2, row_dw0);
              }
            }
          }
          if (e == 0) TRACE(un, l + 1, tl * 4 + 3);
          if (store) ptx::fence_proxy_async();      // the tile is read by the next MMA and by the loader's TMA store
          __syncwarp();
          if (e == 0) TRACE(un, l + 1, tl * 4 + 2);
          if (lane == 0) {
            ptx::mbar_arrive(&written[tl]);           // loader: store the adjoint / reuse the tile
            if (!bottom) ptx::mbar_arrive_leader(&a_ready[tl]);
          }
        }
      }
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&in_empty[par]);      // the slot may take the unit after next
    }
    if (cur_wt >= 0) flush(cur_wt);
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (p.dbg != nullptr && threadIdx.x == 0) {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    p.dbg[2048 + 2 * blockIdx.x + 1] = t;
  }
  ptx::cluster_sync();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc_pair(tmem_base, 512);
  }
}

}  // namespace

cudaError_t launch_mlp_fused_bwd(const MlpBwdParams& p, int num_sms, cudaStream_t stream) {
  const int tiles_task = (p.rows_per_task + 255) / 256;
  const int n_units = ((tiles_task + 1) / 2) * p.tasks;
  int n_cl = num_sms / 2;
  if (n_cl > n_units) n_cl = n_units;
  if (n_cl < 1) n_cl = 1;
  SIREN_ENSURE_SMEM(mlp_fused_bwd_kernel, SMEM_BWD);
  mlp_fused_bwd_kernel<<<2 * n_cl, kThreads, SMEM_BWD, stream>>>(p);
  return cudaGetLastError();
}

}  // namespace siren
