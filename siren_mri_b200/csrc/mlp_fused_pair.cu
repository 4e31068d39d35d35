// Whole-MLP fused forward on CTA PAIRS (cluster of 2, tcgen05 cta_group::2); bf16 mode, value stream,
// d_in <= 256, <= 8 hidden layers.  A pair of SMs carries two 256-row tiles (X, Y) through every layer
// without the activations leaving the chip; each CTA owns 128 rows of each tile.
//
//   layer 0        d_in <= 4: sin(w0 (x W0^T + b0)) computed by the epilogue warps straight into the A-operand
//                  tiles in shared memory (K-major, 128-byte swizzle); wider inputs: one more MMA round on
//                  split-bf16 operands (l0_mma)
//   layers 1..NH   tcgen05.mma.cta_group::2, M = 256: each CTA supplies its 128 rows of A and HALF of the
//                  layer's weight matrix (128 of the 256 output features, 64 KB) -- so a whole layer's B
//                  operand stays resident while first X, then Y run through it, and the next layer's
//                  chunks stream in behind Y.  Accumulators in TMEM (2 x 256 columns per CTA).  The
//                  epilogue writes sin() back IN PLACE as the next layer's A operand.
//   last layer     the outermost linear (d_out <= 2) is a dot product in the top layer's epilogue
//
// X and Y are skewed by half a step: while the epilogue warps work on X(l) the tensor core runs Y(l),
// while they work on Y(l) it runs X(l+1).  The MMA time is hidden behind the sine epilogue, which is
// what bounds this kernel (one MUFU per element plus ~8 issue slots; with the stash also the stores).
//
// Epilogue work split: warp (q, sub) owns TMEM lanes / tile rows [32q, 32q+32) and the 64 columns of
// K-chunk `sub`, i.e. one contiguous 4 KB slice of the A tile -- no warp waits for another one inside
// a layer.  Columns are processed in pieces of 16 with the next TMEM load in flight.
//
// Operands of the hidden layers are fp16 (sines live in [-1, 1], the weights are ~1e-2: 11 mantissa bits instead of
// bf16's 8 at the same tensor-core rate); only the wide first layer's split operands are bf16.
//
// STASH = true (training): each hidden sine layer leaves ONE plane behind, and it is the operand tile itself -- the
// "signed sine" (common.cuh): fp16 sin(theta) whose lowest mantissa bit carries the sign of cos(theta).  Once a warp
// has rewritten its 4 KB slice of the A tile it TMA-stores the slice as it is (one bulk store per warp and layer, no
// staging buffer, no per-piece hand-shake); the backward kernels take sin(theta) from the plane as it is and
// cos(theta) = +-sqrt(1 - h^2).  STASH = false (inference): nothing but y is written.
//
// The sine argument is theta = fma(acc, w0, w0*b), handed to the SFU as it is: its own 1/(2 pi) scaling keeps the
// absolute error below |theta| * 2^-23, far under the fp16 rounding of the result (tests/test_gpu_fused.py holds it
// to 360 rad; the fp32-parity mode reduces the argument exactly and uses sincosf).  The sign bit of the stash comes
// from kf = fma(theta, 1/pi, 1.5 * 2^23): one more FMA per element.
//
// Reference semantics: modules.py:25-26 (BatchLinear), :38 (Sine), :92-97 (FCBlock chain).
#include "common.cuh"
#include "ptx.cuh"
#include "simt.h"
#include "mlp_fused_parts.cuh"

namespace siren {

namespace {

constexpr int MAX_FUSED_LAYERS = MAX_FUSED_HIDDEN_SMEM;
constexpr int Y_BYTES = 2 * TILE_M * (NSUB - 1) * 2 * 4;   // partial last-layer dots [2 tiles][128][3][2]
constexpr int W0_BYTES = H * 4 * 4;             // (w0 * W0 | w0 * b0) as one float4 per column (d <= 3) ...
constexpr int B0_BYTES = H * 4;                 // ... and w0 * b0 separately for d == 4
constexpr int BIAS_BYTES = MAX_FUSED_LAYERS * H * 4;
constexpr int WL_BYTES = 2 * H * 4;             // outermost linear rows (d_out <= 2)
constexpr int MISC = 1024;
constexpr int SMEM_PAIR = 2 * A_TILE + NKC * B_SLOT + Y_BYTES + W0_BYTES + B0_BYTES + BIAS_BYTES + WL_BYTES + MISC + 1024;
static_assert(SMEM_PAIR <= 232448, "shared memory budget");

struct UnitInfo {
  int task;
  int ntile;           // 256-row tiles in this unit (1 or 2)
  int row0[2];         // first row (in the [R, 256] planes) of THIS CTA's 128 rows of tile X / Y
  bool valid[2];       // false: the rows fall behind the task's padded extent (odd number of 128-row tiles)
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

template <bool STASH>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
    mlp_fused_pair_kernel(const __grid_constant__ MlpFwdParams p) {
  constexpr uint32_t IDESC = ptx::umma_idesc_f16(256, 256, 0, 0, ptx::FMT_F16, ptx::FMT_F16);       // hidden layers
  constexpr uint32_t IDESC_L0 = ptx::umma_idesc_bf16(256, 256, 0, 0);                               // split first layer
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;                               // [2 tiles][4 chunks][128][128 B]
  uint8_t* sB = sA + 2 * A_TILE;                    // [4 k-chunks][128][128 B]
  float* sY = reinterpret_cast<float*>(sB + NKC * B_SLOT); // [2][128][NSUB-1][2]
  // [128 column pairs][4 coordinates][2 columns]: a lane's first_rows weight pairs are two LDS.128
  float4* sW0 = reinterpret_cast<float4*>(reinterpret_cast<uint8_t*>(sY) + Y_BYTES);
  float* sB0 = reinterpret_cast<float*>(sW0 + H);   // [256]
  float* sBias = sB0 + H;                           // [MAX_FUSED_LAYERS][256], times w0
  float* sWL = sBias + MAX_FUSED_LAYERS * H;        // [2][256]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sWL + 2 * H);
  uint64_t* b_full = bars;                          // [NKC]  (leader's are used)
  uint64_t* b_empty = bars + NKC;                   // [NKC]  (multicast commit: both CTAs)
  uint64_t* acc_full = bars + 2 * NKC;              // [2]    (multicast commit: both CTAs)
  uint64_t* a_ready = bars + 2 * NKC + 2;           // [2]    (leader's: 16 warps x 2 CTAs arrive)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * NKC + 4);
  float* sLoss = reinterpret_cast<float*>(tmem_slot + 4);      // [4 quadrants] fused MSE: sum of (y - gt)^2

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int NH = p.n_hidden;
  const int rank = int(ptx::cluster_ctarank());
  const bool leader = rank == 0;
  // contiguous range of units (two 256-row tiles each) for this CTA pair
  const int n_cl = gridDim.x >> 1, cl = blockIdx.x >> 1;
  const int tiles_task = (p.rows_per_task + 255) / 256;
  const int n_units = ((tiles_task + 1) / 2) * p.tasks;
  const int base = n_units / n_cl, rem = n_units % n_cl;
  const int u0 = cl * base + (cl < rem ? cl : rem);
  const int u1 = u0 + base + (cl < rem ? 1 : 0);

  if (warp == 0 && lane == 0) {
    for (int l = 0; l < NH; ++l) ptx::prefetch_tmap(&p.tmW[l]);
    if (p.l0_mma) ptx::prefetch_tmap(&p.tmW0);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < NKC; ++i) {
      ptx::mbar_init(&b_full[i], 1);
      ptx::mbar_init(&b_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&acc_full[i], 1);
      ptx::mbar_init(&a_ready[i], 2 * EPI_WARPS);
    }
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc_pair(tmem_slot, 512);
    ptx::tmem_relinquish_pair();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();           // both CTAs' barriers are initialised before any remote arrive / multicast commit
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

  // Register reallocation between the warp groups: the four control warps give back 40 registers each, the
  // epilogue warps get 104 (128 x 56 + 512 x 104 stays inside the 640 x 96 the CTA was launched with) -- at 96 the
  // epilogue re-derives its shared-memory addresses from the thread index in every piece
  if (warp < 4) {
  ptx::setmaxnreg_dec<56>();
  if (warp == 0) {
    // ===================== weight producer (both CTAs: each loads its half of the output features) ==========
    if (lane == 0) {
      // slot kc holds K chunk kc of the layer in flight.  With l0_mma the first nkc0 slots also take the first layer's
      // chunks, so they are used once more per unit than the others: a slot's use count (its barrier phases) is the
      // number of full rounds so far plus, for kc < nkc0, the number of first-layer rounds
      uint32_t n_full = 0u, n_l0 = 0u;
      const int nkc0 = p.l0_mma ? p.nkc0 : 0;
      auto uses = [&](int kc) { return n_full + (kc < nkc0 ? n_l0 : 0u); };
      const int l_first = p.l0_mma ? -1 : 0;
      for (int un = u0; un < u1; ++un) {
        const UnitInfo ui = unit_info(p, un, rank);
        const int wrow = (p.per_task ? ui.task : 0) * H + rank * 128;
        for (int l = l_first; l < NH; ++l) {
          for (int kc = 0; kc < (l < 0 ? nkc0 : NKC); ++kc) {
            ptx::mbar_wait(&b_empty[kc], (uses(kc) & 1u) ^ 1u);       // Y of the previous round is done with the slot
            if (leader) ptx::mbar_arrive_expect_tx(&b_full[kc], 2 * B_SLOT);
            ptx::tma_load_2d_pair(sB + kc * B_SLOT, l < 0 ? &p.tmW0 : &p.tmW[l], &b_full[kc], kc * KCHUNK, wrow);
          }
          if (l < 0) ++n_l0;
          else ++n_full;
        }
      }
      // the last multicast commits have landed in this CTA before it may exit
      for (int kc = 0; kc < NKC; ++kc) ptx::mbar_wait(&b_empty[kc], (uses(kc) & 1u) ^ 1u);
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (leader) {
      uint32_t n_full = 0u, n_l0 = 0u;      // rounds so far: a slot's use count as in the producer (phases of b_full)
      const int nkc0 = p.l0_mma ? p.nkc0 : 0;
      auto uses = [&](int kc) { return n_full + (kc < nkc0 ? n_l0 : 0u); };
      uint32_t rnd = 0u;             // bit tl: phase of a_ready[tl]
      const int l_first = p.l0_mma ? -1 : 0;
      for (int un = u0; un < u1; ++un) {
        const UnitInfo ui = unit_info(p, un, rank);
        for (int l = l_first; l < NH; ++l) {      // l = -1: the first layer, nkc0 K chunks of bf16 operands
          const int nkc = l < 0 ? nkc0 : NKC;
          for (int tl = 0; tl < ui.ntile; ++tl) {
            if (tl == 0) TRACE(un, l + 1, 0);
            ptx::mbar_wait_cluster(&a_ready[tl], (rnd >> tl) & 1u);   // both CTAs: A tile written, accumulator drained
            rnd ^= 1u << tl;
            TRACE(un, l + 1, 1 + tl);
            for (int kc = 0; kc < nkc; ++kc) {
              if (tl == 0) ptx::mbar_wait(&b_full[kc], uses(kc) & 1u);
              ptx::tc_fence_after();
              if (lane == 0) {
                const uint32_t a_addr = ptx::smem_u32(sA + tl * A_TILE + kc * (TILE_M * 128));
                const uint32_t b_addr = ptx::smem_u32(sB + kc * B_SLOT);
#pragma unroll
                for (int ks = 0; ks < 4; ++ks)
                  ptx::umma_bf16_pair(tmem_base + uint32_t(tl * 256), ptx::umma_smem_desc(a_addr + ks * 32, 16, 1024),
                                      ptx::umma_smem_desc(b_addr + ks * 32, 16, 1024), l < 0 ? IDESC_L0 : IDESC,
                                      (kc | ks) ? 1u : 0u);
                if (tl == ui.ntile - 1) ptx::umma_commit_pair(&b_empty[kc], 3);
              }
              __syncwarp();
            }
            if (lane == 0) ptx::umma_commit_pair(&acc_full[tl], 3);
            __syncwarp();
          }
          if (l < 0) ++n_l0;
          else ++n_full;
          TRACE(un, l + 1, 3);
        }
      }
    }
  }
  } else {
    ptx::setmaxnreg_inc<104>();
    // ===================== epilogue / layer-0 warps (both CTAs) =====================
    const int e = warp - 4;
    const int q = warp & 3;                 // TMEM lane quadrant this warp may read
    const int sub = e >> 2;                 // K chunk (64 columns) this warp owns
    const int tid_e = threadIdx.x - 128;
    const int row_t = q * 32 + lane;
    const float w0 = p.w0;
    EpiOut eo;
    eo.a_row = ptx::smem_u32(sA) + uint32_t(sub) * (TILE_M * 128) + uint32_t(row_t) * 128u;
    eo.row7 = row_t & 7;
    eo.lane = lane;
    // STASH: this warp's bulk stores leave from its A slices.  A slice may be rewritten once the store that last
    // left from it has been read out; the warp's stores alternate between the tiles, so one younger group may stay
    // in flight when the latest store was the other tile's.
    int last_store_tl = -1;
    auto slice_free = [&](int tl) {
      if (STASH) {
        if (lane == 0) {
          if (last_store_tl == tl) ptx::bulk_wait_read<0>();
          else ptx::bulk_wait_read<1>();
        }
        __syncwarp();
      }
    };
    uint32_t accph = 0u;                    // bit tl: phase of acc_full[tl]
    int cur_task = -1;
    float lsum = 0.f;                       // fused MSE: sum of (y - gt)^2 over the rows this thread completes
    const int colw = sub * 64;              // first column of this warp
    const uint32_t w0_addr = ptx::smem_u32(sW0 + colw), b0_addr = ptx::smem_u32(sB0 + colw);
    const uint32_t wl_addr = ptx::smem_u32(sWL + colw);

    for (int un = u0; un < u1; ++un) {
      const UnitInfo ui = unit_info(p, un, rank);
      const int wt = p.per_task ? ui.task : 0;
      if (wt != cur_task) {                  // (re)load the first-layer weights and the biases of this task
        ptx::named_bar_sync(15, EPI_WARPS * 32);
        for (int col = tid_e; col < H; col += EPI_WARPS * 32) {
          const float* wr = p.W0 + (size_t(wt) * H + col) * p.d;
          const float bb = w0 * __ldg(p.b0 + size_t(wt) * H + col);
          if (!p.l0_mma) {
            float4 w;
            w.x = w0 * __ldg(wr);
            w.y = p.d > 1 ? w0 * __ldg(wr + 1) : 0.f;
            w.z = p.d > 2 ? w0 * __ldg(wr + 2) : 0.f;
            w.w = p.d > 3 ? w0 * __ldg(wr + 3) : 0.f;
            float* f = reinterpret_cast<float*>(sW0) + (col >> 1) * 8 + (col & 1);
            f[0] = w.x; f[2] = w.y; f[4] = w.z; f[6] = w.w;
          }
          sB0[col] = bb;
          for (int l = 0; l < NH; ++l) sBias[l * H + col] = w0 * __ldg(p.bias[l] + size_t(wt) * H + col);
          if (p.fuse_last) {
            sWL[col] = __ldg(p.WL + (size_t(wt) * p.o) * H + col);
            sWL[H + col] = p.o > 1 ? __ldg(p.WL + (size_t(wt) * p.o + 1) * H + col) : 0.f;
          }
        }
        ptx::named_bar_sync(15, EPI_WARPS * 32);
        cur_task = wt;
      }
      // ---------------- wide first layer (4 < d <= 16): its A operand for the tensor core ----------------
      // x W0^T to near-fp32 accuracy as one 64-wide K chunk of split-bf16 operands (layout: simt.cu,
      // prep_first_kernel).  Thread (row, sub) writes the two 16-byte units 2 sub, 2 sub + 1 of its row in K chunk 0
      // of the tile: elements k = 16 sub .. 16 sub + 15, group g = k / d of coordinate i = k % d.
      if (p.l0_mma)
        for (int tl = 0; tl < ui.ntile; ++tl) {
          if (p.d > 16) {
            // 16 < d <= 256: nkc0 K chunks of plain bf16 inputs (this precision mode's operand rounding).  Warp (q, sub) writes ITS OWN slice -- inputs
            // 64 sub .. 64 sub + 63 of its 32 rows -- and (training) stores it as the layer's INPUT plane: dW_0 is a
            // regular item of the weight-gradient kernel on that plane (64 Fourier features per thread and stage would
            // make the rebuild there the slowest item by far).  Warps behind the last chunk only announce the tile.
            const int nr = ui.row0[tl] + row_t - ui.task * p.rows_per_task;
            const bool live = ui.valid[tl] && nr < p.n;
            const bool mine = sub < p.nkc0;
            slice_free(tl);
            if (mine) {
              const float* xp = p.x + (size_t(ui.task) * p.n + (live ? nr : 0)) * (p.ff.B ? p.ff.raw : p.d);
              float xr[3] = {0.f, 0.f, 0.f};
              if (p.ff.B) {
                xr[0] = __ldg(xp);
                if (p.ff.raw > 1) xr[1] = __ldg(xp + 1);
                if (p.ff.raw > 2) xr[2] = __ldg(xp + 2);
              }
              const uint32_t arow = eo.a_row + uint32_t(tl) * A_TILE;
#pragma unroll 1
              for (int g = 0; g < 4; ++g) {
                uint32_t w[8];
#pragma unroll
                for (int j2 = 0; j2 < 8; ++j2) {
                  float v2[2];
#pragma unroll
                  for (int h2 = 0; h2 < 2; ++h2) {
                    const int i = 64 * sub + 16 * g + 2 * j2 + h2;
                    float v = 0.f;
                    if (live && i < p.d) {
                      if (p.ff.B) {
                        const bool is_cos = i >= p.ff.F;
                        v = fourier_value<false>(fourier_frac(xr, p.ff.raw, p.ff.B, p.ff.F, is_cos ? i - p.ff.F : i), is_cos);
                      } else {
                        v = __ldg(xp + i);
                      }
                    }
                    v2[h2] = v;
                  }
                  w[j2] = pack_bf16(v2[0], v2[1]);
                }
                ptx::st_shared_v4(arow + (uint32_t((2 * g) ^ eo.row7) << 4), w[0], w[1], w[2], w[3]);
                ptx::st_shared_v4(arow + (uint32_t((2 * g + 1) ^ eo.row7) << 4), w[4], w[5], w[6], w[7]);
              }
            }
            ptx::fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
              if (STASH && mine && ui.valid[tl]) {
                ptx::tma_store_2d(&p.tmFeat, sA + tl * A_TILE + sub * (TILE_M * 128) + q * (32 * 128), colw, ui.row0[tl] + q * 32);
                ptx::bulk_commit();
              }
              ptx::mbar_arrive_leader(&a_ready[tl]);
            }
            if (STASH && mine && ui.valid[tl]) last_store_tl = tl;
            continue;
          }
          if (STASH) {
            // K chunk 0 of the tile is the slice of the sub == 0 warps, and every warp of the quadrant writes into
            // it here: the previous unit's top-layer stores of all four must have left shared memory
            slice_free(tl);
            ptx::named_bar_sync(1 + q, NSUB * 32);
          }
          const int nr = ui.row0[tl] + row_t - ui.task * p.rows_per_task;
          const bool live = ui.valid[tl] && nr < p.n;
          const float* xp = p.x + (size_t(ui.task) * p.n + (live ? nr : 0)) * (p.ff.B ? p.ff.raw : p.d);
          const int groups = 64 / p.d < 6 ? 64 / p.d : 6;
          float a0[16];
          if (p.ff.B) {
            // Fourier-feature prologue (features.py:31-41): the layer's inputs are built from the row's raw coordinates
            float xr[3] = {0.f, 0.f, 0.f};
            xr[0] = __ldg(xp);
            if (p.ff.raw > 1) xr[1] = __ldg(xp + 1);
            if (p.ff.raw > 2) xr[2] = __ldg(xp + 2);
            if (p.d == 16) {
              // F = 8 (the reference's configuration): k = 16 sub + j is group g = sub of feature j -- the warp holds
              // the hi terms (sub 0, 1) or the lo terms (sub 2, 3) of all sixteen features; one code path, no division
              const bool lo_role = sub >= 2;
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const float a = 6.283185307179586f * fourier_frac(xr, p.ff.raw, p.ff.B, 8, i);
                const float sv = live ? __sinf(a) : 0.f, cv = live ? __cosf(a) : 0.f;
                const float hs = bf16_round_f(sv), hc = bf16_round_f(cv);
                a0[i] = lo_role ? bf16_round_f(sv - hs) : hs;
                a0[8 + i] = lo_role ? bf16_round_f(cv - hc) : hc;
              }
            } else {
#pragma unroll
              for (int jj = 0; jj < 16; ++jj) a0[jj] = 0.f;
#pragma unroll 1
              for (int j = 0; j < 16; ++j) {
                const int k = 16 * sub + j, g = k / p.d, i = k - g * p.d;
                float v = 0.f;
                if (live && g < groups) {
                  const bool is_cos = i >= p.ff.F;
                  const float x = fourier_value<false>(fourier_frac(xr, p.ff.raw, p.ff.B, p.ff.F, is_cos ? i - p.ff.F : i), is_cos);
                  const float h = bf16_round_f(x), l = bf16_round_f(x - h);
                  v = g < 2 || g == 4 ? h : g < 4 ? l : bf16_round_f(x - h - l);
                }
                // (a0 is indexed by the loop counter of a rolled loop: pick the register by a chain of selects)
#pragma unroll
                for (int jj = 0; jj < 16; ++jj) a0[jj] = (jj == j) ? v : a0[jj];
              }
            }
          } else if (p.d == 16) {
            // d = 16: group g = sub of input j, no division; the row is four 16-byte loads
            const bool lo_role = sub >= 2;
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4) {
              const float4 xv = live ? __ldg(reinterpret_cast<const float4*>(xp) + j4) : make_float4(0.f, 0.f, 0.f, 0.f);
              const float xs[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
              for (int c = 0; c < 4; ++c) {
                const float h = bf16_round_f(xs[c]);
                a0[4 * j4 + c] = lo_role ? bf16_round_f(xs[c] - h) : h;
              }
            }
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const int k = 16 * sub + j, g = k / p.d, i = k - g * p.d;
              float v = 0.f;
              if (live && g < groups) {
                const float x = __ldg(xp + i);
                const float h = bf16_round_f(x), l = bf16_round_f(x - h);
                v = g < 2 || g == 4 ? h : g < 4 ? l : bf16_round_f(x - h - l);
              }
              a0[j] = v;
            }
          }
          const uint32_t arow0 = ptx::smem_u32(sA) + uint32_t(tl) * A_TILE + uint32_t(row_t) * 128u;
#pragma unroll
          for (int h = 0; h < 2; ++h)
            ptx::st_shared_v4(arow0 + (uint32_t((2 * sub + h) ^ eo.row7) << 4), pack_bf16(a0[8 * h], a0[8 * h + 1]),
                              pack_bf16(a0[8 * h + 2], a0[8 * h + 3]), pack_bf16(a0[8 * h + 4], a0[8 * h + 5]),
                              pack_bf16(a0[8 * h + 6], a0[8 * h + 7]));
          ptx::fence_proxy_async();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive_leader(&a_ready[tl]);
        }
      // ---------------- narrow first layer (d <= 4): SIMT, straight into the A tiles ----------------
      // this thread's row of both tiles: fetch the coordinates up front so that Y's are in flight during X
      float cx[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        const int nr = ui.row0[t] + row_t - ui.task * p.rows_per_task;
        if (!p.l0_mma && t < ui.ntile && ui.valid[t] && nr < p.n) {
          const float* xp = p.x + (size_t(ui.task) * p.n + nr) * p.d;
          cx[t][0] = __ldg(xp);
          if (p.d > 1) cx[t][1] = __ldg(xp + 1);
          if (p.d > 2) cx[t][2] = __ldg(xp + 2);
          if (p.d > 3) cx[t][3] = __ldg(xp + 3);
        }
      }
      for (int tl = 0; tl < (p.l0_mma ? 0 : ui.ntile); ++tl) {
        if (e == 0) TRACE(un, 0, 4 + 2 * tl);
        // columns colw + 2 lane, + 1 of this warp's slice (.w of a packed column is W0[.][3] only for d = 4)
        const float4 wa = ptx::ld_shared_f4(w0_addr + uint32_t(lane) * 32u);
        const float4 wb = ptx::ld_shared_f4(w0_addr + uint32_t(lane) * 32u + 16u);
        const float2 w2[4] = {make_float2(wa.x, wa.y), make_float2(wa.z, wa.w), make_float2(wb.x, wb.y),
                              make_float2(wb.z, wb.w)};
        const float2 b2 = make_float2(ptx::ld_shared_f32(b0_addr + uint32_t(lane) * 8u),
                                      ptx::ld_shared_f32(b0_addr + uint32_t(lane) * 8u + 4u));
        const uint32_t a_slice = ptx::smem_u32(sA) + uint32_t(tl) * A_TILE + uint32_t(sub) * (TILE_M * 128) +
                                 uint32_t(q) * (32u * 128u);
        const float cxt[4] = {tl ? cx[1][0] : cx[0][0], tl ? cx[1][1] : cx[0][1], tl ? cx[1][2] : cx[0][2],
                              tl ? cx[1][3] : cx[0][3]};
        slice_free(tl);        // the previous unit's top-layer store of this slice has left shared memory
        // no stash for this layer even when training: the backward kernels recompute w0 (x W0^T + b0) from the
        // coordinates with the same FMA chain (mlp_fused_bwd.cu bottom_pass, wgrad.cu build_first_sines)
        switch (p.d) {
          case 1: first_rows<1>(eo, a_slice, cxt, w2, b2); break;
          case 2: first_rows<2>(eo, a_slice, cxt, w2, b2); break;
          case 3: first_rows<3>(eo, a_slice, cxt, w2, b2); break;
          default: first_rows<4>(eo, a_slice, cxt, w2, b2); break;
        }
        ptx::fence_proxy_async();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive_leader(&a_ready[tl]);
        if (e == 0) TRACE(un, 0, 5 + 2 * tl);
      }
      // ---------------- hidden layers ----------------
      for (int l = p.l0_mma ? 0 : 1; l <= NH; ++l) {
        const bool top = (l == NH);
        if (top && sub == 0 && un + 1 < u1) {      // pull the next unit's coordinates towards L2 while this one finishes
          const UnitInfo nx = unit_info(p, un + 1, rank);
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            const int nr = nx.row0[t] + row_t - nx.task * p.rows_per_task;
            if (t < nx.ntile && nx.valid[t] && nr < p.n)
              ptx::prefetch_l2(p.x + (size_t(nx.task) * p.n + nr) * (p.ff.B ? p.ff.raw : p.d));
          }
        }
        const uint32_t bias_addr = l == 0 ? ptx::smem_u32(sB0 + colw) : ptx::smem_u32(sBias + (l - 1) * H + colw);
        for (int tl = 0; tl < ui.ntile; ++tl) {
          const int row0 = ui.row0[tl];
          const bool valid = ui.valid[tl];
          const int n_row = row0 + row_t - ui.task * p.rows_per_task;
          // the sine slice is the next layer's operand and (training) the layer's stash plane; the top layer of an
          // inference run needs neither
          const bool write_a = !top || STASH;
          const uint32_t taddr = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(tl * 256 + colw);
          float ydot0 = 0.f, ydot1 = 0.f;
          float gt0 = 0.f, gt1 = 0.f;       // fused MSE: this row's target, fetched now, used when the row's y is complete
          if (top && p.fuse_last && p.gt && sub == 0 && valid && n_row < p.n) {
            const float* gp = p.gt + (size_t(ui.task) * p.n + n_row) * p.o;
            gt0 = __ldg(gp);
            if (p.o > 1) gt1 = __ldg(gp + 1);
          }
          // data consistency (data_consistency.py:7-20): this row's mask and sampled values, fetched with the target
          float dm0 = 0.f, dm1 = 0.f, dk0 = 0.f, dk1 = 0.f;
          if (top && p.fuse_last && p.dc.k0 && sub == 0 && valid && n_row < p.n) {
            const size_t i0 = dc_index(p.dc.cf, ui.task, n_row, 0, p.n, p.o);
            dm0 = __ldg(p.dc.mask + i0) * p.dc.pull;
            dk0 = __ldg(p.dc.k0 + i0);
            if (p.o > 1) {
              const size_t i1 = dc_index(p.dc.cf, ui.task, n_row, 1, p.n, p.o);
              dm1 = __ldg(p.dc.mask + i1) * p.dc.pull;
              dk1 = __ldg(p.dc.k0 + i1);
            }
          }
          float va[PW], vb[PW];
          ptx::mbar_wait(&acc_full[tl], (accph >> tl) & 1u);
          accph ^= 1u << tl;
          ptx::tc_fence_after();
          if (e == 0) TRACE(un, l, 4 + 2 * tl);
          ptx::tmem_ld<PW>(taddr, reinterpret_cast<uint32_t*>(va));
          if (write_a) slice_free(tl);      // the store that last left from this slice (one layer ago) has been read
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
              const float2 t01 = ptx::fma2(make_float2(v[4 * j4 + 0], v[4 * j4 + 1]), make_float2(w0, w0), make_float2(bb.x, bb.y));
              const float2 t23 = ptx::fma2(make_float2(v[4 * j4 + 2], v[4 * j4 + 3]), make_float2(w0, w0), make_float2(bb.z, bb.w));
              t[4 * j4 + 0] = t01.x; t[4 * j4 + 1] = t01.y;
              t[4 * j4 + 2] = t23.x; t[4 * j4 + 3] = t23.y;
            }
            piece_out<STASH>(eo, tl, pc, t, s, write_a);
            if (top && p.fuse_last) {
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
          if (write_a) {
            ptx::fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
              if (STASH && valid) {      // the slice as it stands is the layer's stash plane (signed sine)
                ptx::tma_store_2d(&p.tmAct[l], sA + tl * A_TILE + sub * (TILE_M * 128) + q * (32 * 128), colw, row0 + q * 32);
                ptx::bulk_commit();
              }
              if (!top) ptx::mbar_arrive_leader(&a_ready[tl]);
            }
            if (STASH && valid) last_store_tl = tl;
          }
          if (e == 0) TRACE(un, l, 5 + 2 * tl);
          if (top && p.fuse_last) {
            float* sy = sY + tl * (TILE_M * (NSUB - 1) * 2);
            if (sub != 0) {
              sy[(row_t * (NSUB - 1) + sub - 1) * 2 + 0] = ydot0;
              sy[(row_t * (NSUB - 1) + sub - 1) * 2 + 1] = ydot1;
            }
            ptx::named_bar_sync(1 + q, NSUB * 32);
            if (sub == 0 && valid && n_row < p.n) {
#pragma unroll
              for (int u = 0; u < NSUB - 1; ++u) {
                ydot0 += sy[(row_t * (NSUB - 1) + u) * 2 + 0];
                ydot1 += sy[(row_t * (NSUB - 1) + u) * 2 + 1];
              }
              const size_t yi = (size_t(ui.task) * p.n + n_row) * p.o;
              float y0 = ydot0 + __ldg(p.bL + size_t(wt) * p.o);
              float y1 = p.o > 1 ? ydot1 + __ldg(p.bL + size_t(wt) * p.o + 1) : 0.f;
              y0 = fmaf(dm0, dk0, (1.f - dm0) * y0);      // (1 - m pull) y + m pull k0: a sampled entry (m pull = 1) is
              y1 = fmaf(dm1, dk1, (1.f - dm1) * y1);      // k0 to the bit; dm = 0 without data consistency
              p.y[yi] = y0;
              if (p.o > 1) p.y[yi + 1] = y1;
              if (p.gt) {
                const float d0 = y0 - gt0;
                p.gy[yi] = 2.f * p.loss_weight * d0 * (1.f - dm0);
                lsum = fmaf(d0, d0, lsum);
                if (p.o > 1) {
                  const float d1 = y1 - gt1;
                  p.gy[yi + 1] = 2.f * p.loss_weight * d1 * (1.f - dm1);
                  lsum = fmaf(d1, d1, lsum);
                }
              }
            }
          }
        }
      }
    }
    if (p.gt && p.loss_acc) {               // one atomic per CTA: w * sum over its rows of (y - gt)^2
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
#undef TRACE

  ptx::tc_fence_before();
  __syncthreads();
  if (p.dbg != nullptr && threadIdx.x == 0) {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    p.dbg[2048 + 2 * blockIdx.x + 1] = t;
  }
  ptx::cluster_sync();           // neither CTA leaves (or frees TMEM) while the other may still touch it
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc_pair(tmem_base, 512);
  }
}

}  // namespace

cudaError_t launch_mlp_fused_pair(const MlpFwdParams& p, bool stash, int num_sms, cudaStream_t stream) {
  const int tiles_task = (p.rows_per_task + 255) / 256;
  const int n_units = ((tiles_task + 1) / 2) * p.tasks;
  int n_cl = num_sms / 2;
  if (n_cl > n_units) n_cl = n_units;
  if (n_cl < 1) n_cl = 1;
  const int G = 2 * n_cl;
  if (stash) {
    SIREN_ENSURE_SMEM(mlp_fused_pair_kernel<true>, SMEM_PAIR);
    mlp_fused_pair_kernel<true><<<G, kThreads, SMEM_PAIR, stream>>>(p);
  } else {
    SIREN_ENSURE_SMEM(mlp_fused_pair_kernel<false>, SMEM_PAIR);
    mlp_fused_pair_kernel<false><<<G, kThreads, SMEM_PAIR, stream>>>(p);
  }
  return cudaGetLastError();
}

}  // namespace siren
