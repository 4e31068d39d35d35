// Row-tile GEMM kernels on tcgen05: a 128-row tile of S coordinate-jet streams times one
// resident 256-wide weight block, accumulators in TMEM, with the sine (forward) or the
// sine-reverse (backward dgrad) fused into the epilogue.
//
//   forward  hidden layer l :  z = h W^T + b ; h' = sin(w0 z), c = cos(w0 z)
//                              Jz_k = J_k W^T ; J'_k = w0 c Jz_k
//                              Dz_k = D_k W^T ; D'_k = w0 c Dz_k - w0^2 s Jz_k^2
//       (reference: modules.py:25-26 BatchLinear.forward + modules.py:38 Sine.forward; the jet
//        streams replace the double backward of diff_operators.py:27-43)
//   backward hidden layer l :  (hbar, Jbar_k, Dbar_k) = (zbar, Jzbar_k, Dzbar_k) W_l, then the
//                              reverse of the sine of layer l-1 (SURVEY.md appendix A)
//
// Warp roles (384 threads): warp 0 TMA producer, warp 1 MMA issuer, warp 2 TMEM allocator,
// warps 4..11 epilogue (two warps per TMEM lane quadrant, each taking half of the columns).
#include "common.cuh"
#include "ptx.cuh"
#include "simt.h"

namespace siren {

namespace {

constexpr int kEpiWarp0 = 4;

template <int ORDER, int D, bool SPLIT, int MODE>
struct RowsCfg {
  static constexpr int S = 1 + ORDER * D;
  // weight block width.  Three or four streams: 64 columns leave room for TWO accumulator sets (MMA under the
  // epilogue) -- measured at cfg3: dgrad 1140 -> 911 us (bf16), 2449 -> 2084 us (fp32-parity), fp32-parity forward
  // 2493 -> 2317 us; the bf16 forward alone is faster with 128 (909 against 1015 us: its epilogue is short and the A
  // tile is read half as often)
  static constexpr int BN = (S == 1) ? (SPLIT ? 128 : 256) : (S <= 2 ? 128 : (S <= 4 && MODE == 0 && !SPLIT) ? 128 : 64);
  // columns per thread and pass.  The jet epilogues walk the streams one (J_k, D_k) pair at a
  // time, so only a handful of chunks are live at once whatever S is: 32 columns forward,
  // 16 backward (the reverse of the sine keeps more of them alive).
  static constexpr int CW = (S == 1) ? (SPLIT ? 16 : 32) : (MODE == 1 ? 16 : 32);
  static constexpr int NACC = (2 * S * BN <= 512) ? 2 : 1;
  static constexpr int NSPLIT = SPLIT ? 2 : 1;
  static constexpr int B_BYTES = NSPLIT * 4 * BN * 128;
  static constexpr bool BIG_B = B_BYTES >= 128 * 1024;     // a 128 KB weight block leaves little shared memory
  // epilogue warps per TMEM lane quadrant.  The epilogue is latency-bound, so the light
  // single-stream configurations run 4 warps per quadrant; the jet epilogues need > 96 registers
  // per thread (640 threads x 96 registers fill the file) and stay at 2.
  static constexpr int NQW = (S == 1 && !(MODE == 1 && BIG_B)) ? 4 : 2;
  static constexpr int EPI_WARPS = 4 * NQW;
  static constexpr int THREADS = 128 + NQW * 128;
  static constexpr int A_STAGE = TILE_M * 128;   // 16 KB
  // warp-private staging of the epilogue's TMA stores: [32 rows][CW columns] per buffer
  static constexpr int OUT_ELEM = (MODE == 0 && SPLIT) ? 4 : 2;          // widest element stored (fp32 stash forward)
  static constexpr int NBUF = BIG_B ? 1 : 2;
  static constexpr int OUT_BUF = 32 * CW * OUT_ELEM;
  static constexpr int OUT_BYTES = (MODE == 2) ? 0 : EPI_WARPS * NBUF * OUT_BUF;
  // warp-private ring of TMA-loaded stash chunks for the backward epilogue
  static constexpr int NLB = (S == 1 || BIG_B) ? 2 : 4;
  static constexpr int IN_BUF = 32 * CW * (SPLIT ? 4 : 2);
  static constexpr int IN_BYTES = (MODE == 1) ? EPI_WARPS * NLB * IN_BUF : 0;
  static constexpr int NST_MAX = (225 * 1024 - 2048 - B_BYTES - OUT_BYTES - IN_BYTES) / A_STAGE;
  static constexpr int NST = NST_MAX > 6 ? 6 : NST_MAX;
  static constexpr int SMEM = B_BYTES + NST * A_STAGE + OUT_BYTES + IN_BYTES + 1024 /*barriers*/ + 1024 /*align slack*/;
  static_assert(S * BN * NACC <= 512, "TMEM columns");
  static_assert(NST >= 2, "pipeline depth");
};

struct TileRange {
  int t0, t1;
};
__device__ __forceinline__ TileRange cta_tiles(int tiles_m, int g, int G) {
  int base = tiles_m / G, rem = tiles_m % G;
  int t0 = g * base + (g < rem ? g : rem);
  int n = base + (g < rem ? 1 : 0);
  return {t0, t0 + n};
}

// -------------------------------------------------------------------------------------------
// epilogues.  acc[s][j]: stream s, column col0 + j of this thread's row.
// -------------------------------------------------------------------------------------------
// Warp-private staged output: each epilogue warp owns NBUF shared-memory buffers of
// [32 rows][CW columns]; a chunk of CW values per lane (= row) is written there with the TMA
// swizzle of its row width and leaves as ONE bulk tensor store (box CW x 32).  This replaces
// row-strided global stores, which cost 32 L1 tag cycles per warp instruction.
template <int CW, int NBUF>
struct WarpOut {
  uint32_t base;      // shared address of this warp's first buffer
  uint32_t buf_bytes;
  int cur;
  int lane;
  int y;              // global row of lane 0 inside a plane (tile row0 + 32 * quadrant)
  int x;              // first column of the chunk

  template <int ELEM>   // bytes per element: 2 (bf16) or 4 (fp32)
  __device__ __forceinline__ uint32_t slot(int chunk16) const {
    constexpr int RB = CW * ELEM;                       // row bytes: 32, 64 or 128
    const int r = lane;
    const int swz = (RB == 128) ? (r & 7) : (RB == 64) ? ((r >> 1) & 3) : (RB == 32) ? ((r >> 2) & 1) : 0;
    return base + cur * buf_bytes + uint32_t(r * RB) + (uint32_t(chunk16 ^ swz) << 4);
  }
  __device__ __forceinline__ void begin() {
    if (lane == 0) ptx::bulk_wait_read<NBUF - 1>();     // the buffer we are about to overwrite has been read
    __syncwarp();
  }
  __device__ __forceinline__ void finish(const CUtensorMap* m, int plane_row) {
    ptx::fence_proxy_async();
    __syncwarp();
    if (lane == 0) {
      ptx::tma_store_2d(m, reinterpret_cast<const void*>(__cvta_shared_to_generic(base + cur * buf_bytes)), x,
                        plane_row + y);
      ptx::bulk_commit();
    }
    cur = (cur + 1 == NBUF) ? 0 : cur + 1;
  }
  // bf16 plane (plane_row = first row of the plane inside the mapped tensor)
  __device__ __forceinline__ void put_bf16(const CUtensorMap* m, int plane_row, const float* v) {
    begin();
#pragma unroll
    for (int i = 0; i < CW / 8; ++i)
      ptx::st_shared_v4(slot<2>(i), pack_bf16(v[8 * i], v[8 * i + 1]), pack_bf16(v[8 * i + 2], v[8 * i + 3]),
                        pack_bf16(v[8 * i + 4], v[8 * i + 5]), pack_bf16(v[8 * i + 6], v[8 * i + 7]));
    finish(m, plane_row);
  }
  __device__ __forceinline__ void put_f32(const CUtensorMap* m, int plane_row, const float* v) {
    begin();
#pragma unroll
    for (int i = 0; i < CW / 4; ++i)
      ptx::st_shared_v4(slot<4>(i), __float_as_uint(v[4 * i]), __float_as_uint(v[4 * i + 1]),
                        __float_as_uint(v[4 * i + 2]), __float_as_uint(v[4 * i + 3]));
    finish(m, plane_row);
  }
  // MMA operand plane: bf16 hi (+ bf16 lo = bf16(v - hi) in split mode)
  template <bool SPLIT>
  __device__ __forceinline__ void put_operand(const CUtensorMap* hi, const CUtensorMap* lo, int plane_row,
                                              const float* v) {
    put_bf16(hi, plane_row, v);
    if constexpr (SPLIT) {
      float r[CW];
#pragma unroll
      for (int i = 0; i < CW; ++i) r[i] = v[i] - bf16_round_f(v[i]);
      put_bf16(lo, plane_row, r);
    }
  }
  // stash plane: fp32 in split mode, bf16 otherwise
  template <bool SPLIT>
  __device__ __forceinline__ void put_stash(const CUtensorMap* m, int plane_row, const float* v) {
    if constexpr (SPLIT) put_f32(m, plane_row, v);
    else put_bf16(m, plane_row, v);
  }
};

// Warp-private in-order stream of TMA-loaded stash chunks ([32 rows][CW columns] each) for the
// backward epilogue.  The order in which chunks are consumed is fixed (see BwdLoadSeq), so lane 0
// keeps up to NLB loads in flight and every take() refills the slot it just drained.
struct LoadDesc {
  int which;               // 0: cosine stash, 1: sine hi, 2: sine lo, 3: jet stash
  int x, y;
  uint32_t bytes;
};

template <int ORDER, int D, bool SPLIT, int CW, int NCH>
struct BwdLoadSeq {
  int below_is_first, R;
  int t, t1, cc, pi;       // tile, chunk inside the warp's column slice, plane index inside the chunk
  int q, colbase;          // lane quadrant, first column of the warp's slice
  __device__ __forceinline__ int planes() const {
    // c [, s_hi [, s_lo], then per k: jz_k [, dz_k]  (jz/dz come from W0 when the layer below is layer 0)
    if (ORDER == 0) return 1;
    const int per_k = below_is_first ? 0 : (ORDER == 2 ? 2 : 1);
    return 1 + (SPLIT ? 2 : 1) + D * per_k;
  }
  __device__ __forceinline__ bool done() const { return t >= t1; }
  __device__ __forceinline__ LoadDesc current() const {
    LoadDesc d;
    d.x = colbase + cc * CW;
    d.y = t * TILE_M + q * 32;
    const int ns = SPLIT ? 2 : 1;
    if (pi == 0) {
      d.which = 0;
      d.bytes = 32 * CW * (SPLIT ? 4 : 2);
    } else if (pi <= ns) {
      d.which = pi;                                   // 1: hi, 2: lo
      d.bytes = 32 * CW * 2;
    } else {
      const int j = pi - 1 - ns;                       // 0 .. D*per_k-1 in consumption order
      const int per_k = (ORDER == 2) ? 2 : 1;
      const int k = j / per_k, which = j - k * per_k;  // which: 0 = jz_k, 1 = dz_k
      d.which = 3;
      d.y += (which * D + k) * R;
      d.bytes = 32 * CW * (SPLIT ? 4 : 2);
    }
    return d;
  }
  __device__ __forceinline__ void advance() {
    if (++pi == planes()) {
      pi = 0;
      if (++cc == NCH) {
        cc = 0;
        ++t;
      }
    }
  }
};

template <int CW, int NLB, class Seq>
struct WarpIn {
  uint32_t base, buf_bytes;
  uint64_t* bars;          // [NLB]
  int lane;
  uint32_t issued, taken;
  Seq seq;

  __device__ __forceinline__ void issue_one(const RowsGemmParams& p) {
    if (seq.done()) return;
    if (lane == 0) {
      const LoadDesc d = seq.current();
      const uint32_t b = issued % NLB;
      ptx::mbar_arrive_expect_tx(&bars[b], d.bytes);
      void* dst = reinterpret_cast<void*>(__cvta_shared_to_generic(base + b * buf_bytes));
      // one call site per tensor map: the maps live in kernel-parameter space and are named statically
      if (d.which == 0) ptx::tma_load_2d(dst, &p.tmCin, &bars[b], d.x, d.y);
      else if (d.which == 1) ptx::tma_load_2d(dst, &p.tmSin_hi, &bars[b], d.x, d.y);
      else if (d.which == 2) ptx::tma_load_2d(dst, &p.tmSin_lo, &bars[b], d.x, d.y);
      else ptx::tma_load_2d(dst, &p.tmJin, &bars[b], d.x, d.y);
    }
    seq.advance();
    ++issued;
  }
  __device__ __forceinline__ void prime(const RowsGemmParams& p) {
#pragma unroll
    for (int i = 0; i < NLB; ++i) issue_one(p);
  }
  template <int ELEM>
  __device__ __forceinline__ uint32_t slot(uint32_t b, int chunk16) const {
    constexpr int RB = CW * ELEM;
    const int r = lane;
    const int swz = (RB == 128) ? (r & 7) : (RB == 64) ? ((r >> 1) & 3) : (RB == 32) ? ((r >> 2) & 1) : 0;
    return base + b * buf_bytes + uint32_t(r * RB) + (uint32_t(chunk16 ^ swz) << 4);
  }
  __device__ __forceinline__ uint32_t wait_front() {
    const uint32_t b = taken % NLB;
    ptx::mbar_wait(&bars[b], (taken / NLB) & 1u);
    return b;
  }
  __device__ __forceinline__ void pop(const RowsGemmParams& p) {
    ++taken;
    __syncwarp();            // every lane has read the slot before lane 0 refills it
    issue_one(p);
  }
  template <bool ACC>
  __device__ __forceinline__ void take_bf16_t(const RowsGemmParams& p, float* v) {
    const uint32_t b = wait_front();
#pragma unroll
    for (int i = 0; i < CW / 8; ++i) {
      uint32_t a0, a1, a2, a3;
      ptx::ld_shared_v4(slot<2>(b, i), a0, a1, a2, a3);
      if constexpr (ACC) {
        v[8 * i + 0] += bf16_lo_f(a0); v[8 * i + 1] += bf16_hi_f(a0); v[8 * i + 2] += bf16_lo_f(a1); v[8 * i + 3] += bf16_hi_f(a1);
        v[8 * i + 4] += bf16_lo_f(a2); v[8 * i + 5] += bf16_hi_f(a2); v[8 * i + 6] += bf16_lo_f(a3); v[8 * i + 7] += bf16_hi_f(a3);
      } else {
        v[8 * i + 0] = bf16_lo_f(a0); v[8 * i + 1] = bf16_hi_f(a0); v[8 * i + 2] = bf16_lo_f(a1); v[8 * i + 3] = bf16_hi_f(a1);
        v[8 * i + 4] = bf16_lo_f(a2); v[8 * i + 5] = bf16_hi_f(a2); v[8 * i + 6] = bf16_lo_f(a3); v[8 * i + 7] = bf16_hi_f(a3);
      }
    }
    pop(p);
  }
  __device__ __forceinline__ void take_f32(const RowsGemmParams& p, float* v) {
    const uint32_t b = wait_front();
#pragma unroll
    for (int i = 0; i < CW / 4; ++i) {
      uint32_t a0, a1, a2, a3;
      ptx::ld_shared_v4(slot<4>(b, i), a0, a1, a2, a3);
      v[4 * i] = __uint_as_float(a0); v[4 * i + 1] = __uint_as_float(a1);
      v[4 * i + 2] = __uint_as_float(a2); v[4 * i + 3] = __uint_as_float(a3);
    }
    pop(p);
  }
  template <bool SPLIT>
  __device__ __forceinline__ void take_stash(const RowsGemmParams& p, float* v) {
    if constexpr (SPLIT) take_f32(p, v);
    else take_bf16_t<false>(p, v);
  }
  template <bool SPLIT>
  __device__ __forceinline__ void take_operand(const RowsGemmParams& p, float* v) {      // hi (+ lo)
    take_bf16_t<false>(p, v);
    if constexpr (SPLIT) take_bf16_t<true>(p, v);
  }
};

// taddr: TMEM address of stream 0 at this thread's lane quadrant and first column; stream s lives
// BN columns further.  The value stream is read first; the jet streams follow one k at a time.
template <int ORDER, int D, bool SPLIT, int CW, int BN, int NBUF>
__device__ __forceinline__ void epilogue_forward(const RowsGemmParams& p, WarpOut<CW, NBUF>& io, uint32_t taddr,
                                                 int col0, int task) {
  const float w0 = p.w0;
  const float w0_rev = w0 * 0.15915494309189535f;
  const float* bias = p.bias + (p.per_task ? task * H : 0) + col0;
  const int R = p.R;
  float s[CW], c[CW];
  {
    float z[CW];
    ptx::tmem_ld<CW>(taddr, reinterpret_cast<uint32_t*>(z));
    ptx::tmem_wait_ld();
#pragma unroll
    for (int j = 0; j < CW; ++j) sincos_w0<SPLIT>(z[j] + __ldg(bias + j), w0, w0_rev, &s[j], &c[j]);
  }
  io.template put_operand<SPLIT>(&p.tmO_hi, &p.tmO_lo, 0, s);
  io.template put_stash<SPLIT>(&p.tmC, 0, c);
  if constexpr (ORDER >= 1) {
#pragma unroll
    for (int k = 0; k < D; ++k) {
      float jz[CW], o[CW];
      ptx::tmem_ld<CW>(taddr + uint32_t((1 + k) * BN), reinterpret_cast<uint32_t*>(jz));
      ptx::tmem_wait_ld();
      io.template put_stash<SPLIT>(&p.tmJ, k * R, jz);
      if constexpr (ORDER == 2) {
        float dz[CW];
        ptx::tmem_ld<CW>(taddr + uint32_t((1 + D + k) * BN), reinterpret_cast<uint32_t*>(dz));
        ptx::tmem_wait_ld();
        io.template put_stash<SPLIT>(&p.tmJ, (D + k) * R, dz);
#pragma unroll
        for (int j = 0; j < CW; ++j) o[j] = w0 * c[j] * dz[j] - (w0 * w0) * s[j] * jz[j] * jz[j];
        io.template put_operand<SPLIT>(&p.tmO_hi, &p.tmO_lo, (1 + D + k) * R, o);
      }
#pragma unroll
      for (int j = 0; j < CW; ++j) o[j] = w0 * c[j] * jz[j];
      io.template put_operand<SPLIT>(&p.tmO_hi, &p.tmO_lo, (1 + k) * R, o);
    }
  }
}

template <int ORDER, int D, bool SPLIT, int CW, int BN, int NBUF, class In>
__device__ __forceinline__ void epilogue_backward(const RowsGemmParams& p, WarpOut<CW, NBUF>& io, In& in,
                                                  uint32_t taddr, int col0, int task) {
  const int R = p.R;
  const float w0 = p.w0;
  float c[CW], zb[CW];
  in.template take_stash<SPLIT>(p, c);
  {
    float hb[CW];
    ptx::tmem_ld<CW>(taddr, reinterpret_cast<uint32_t*>(hb));
    ptx::tmem_wait_ld();
#pragma unroll
    for (int j = 0; j < CW; ++j) zb[j] = w0 * c[j] * hb[j];
  }
  if constexpr (ORDER >= 1) {
    float s[CW];
    in.template take_operand<SPLIT>(p, s);
#pragma unroll
    for (int k = 0; k < D; ++k) {
      float jz[CW], jb[CW], o[CW];
      ptx::tmem_ld<CW>(taddr + uint32_t((1 + k) * BN), reinterpret_cast<uint32_t*>(jb));
      if (p.below_is_first) {
        const float* w = p.w_first + (size_t(p.per_task ? task : 0) * H + col0) * D + k;
#pragma unroll
        for (int j = 0; j < CW; ++j) jz[j] = __ldg(w + j * D);
      } else {
        in.template take_stash<SPLIT>(p, jz);
      }
      ptx::tmem_wait_ld();
#pragma unroll
      for (int j = 0; j < CW; ++j) {
        zb[j] -= (w0 * w0) * s[j] * jz[j] * jb[j];
        o[j] = w0 * c[j] * jb[j];
      }
      if constexpr (ORDER == 2) {
        float dz[CW], db[CW];
        ptx::tmem_ld<CW>(taddr + uint32_t((1 + D + k) * BN), reinterpret_cast<uint32_t*>(db));
        if (p.below_is_first) {
#pragma unroll
          for (int j = 0; j < CW; ++j) dz[j] = 0.f;
        } else {
          in.template take_stash<SPLIT>(p, dz);
        }
        ptx::tmem_wait_ld();
#pragma unroll
        for (int j = 0; j < CW; ++j) {
          zb[j] -= (w0 * w0) * s[j] * dz[j] * db[j] + (w0 * w0 * w0) * c[j] * jz[j] * jz[j] * db[j];
          o[j] -= 2.f * (w0 * w0) * s[j] * jz[j] * db[j];
          dz[j] = w0 * c[j] * db[j];                      // Dzbar_k
        }
        io.template put_operand<SPLIT>(&p.tmO_hi, &p.tmO_lo, (1 + D + k) * R, dz);
      }
      io.template put_operand<SPLIT>(&p.tmO_hi, &p.tmO_lo, (1 + k) * R, o);
    }
  }
  io.template put_operand<SPLIT>(&p.tmO_hi, &p.tmO_lo, 0, zb);
}

// -------------------------------------------------------------------------------------------
// MODE 0: forward sine epilogue, 1: backward sine-reverse epilogue, 2: raw fp32 accumulator
// -------------------------------------------------------------------------------------------
template <int ORDER, int D, bool SPLIT, int MODE>
__global__ void __launch_bounds__(RowsCfg<ORDER, D, SPLIT, MODE>::THREADS, 1)
rows_gemm_kernel(const __grid_constant__ RowsGemmParams p) {
  using Cfg = RowsCfg<ORDER, D, SPLIT, MODE>;
  constexpr int S = Cfg::S, BN = Cfg::BN, CW = Cfg::CW, NACC = Cfg::NACC, NST = Cfg::NST;
  constexpr int NB = H / BN;
  constexpr uint32_t IDESC = ptx::umma_idesc_bf16(TILE_M, BN, 0, 0);

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sB = smem;                             // [NSPLIT][4 chunks][BN rows][128 B]
  uint8_t* sA = smem + Cfg::B_BYTES;              // [NST][128 rows][128 B]
  uint8_t* sStg = sA + NST * Cfg::A_STAGE;        // [epilogue warps][NBUF][32 rows][CW cols]   staged stores
  uint8_t* sIn = sStg + Cfg::OUT_BYTES;           // [epilogue warps][NLB][32 rows][CW cols]    staged stash loads
  uint64_t* bars = reinterpret_cast<uint64_t*>(sIn + Cfg::IN_BYTES);
  uint64_t* full = bars;                          // [NST]
  uint64_t* empty = bars + NST;                   // [NST]
  uint64_t* b_full = bars + 2 * NST;
  uint64_t* b_empty = bars + 2 * NST + 1;
  uint64_t* acc_full = bars + 2 * NST + 2;        // [NACC]
  uint64_t* acc_empty = bars + 2 * NST + 2 + NACC;
  uint64_t* in_bars = bars + 2 * NST + 2 + 2 * NACC;     // [epilogue warps][NLB]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(in_bars + Cfg::EPI_WARPS * Cfg::NLB);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int nb = blockIdx.x % NB;
  const int G = gridDim.x / NB;
  const int g = blockIdx.x / NB;
  const int tiles_m = p.R / TILE_M;
  const TileRange tr = cta_tiles(tiles_m, g, G);

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&p.tmA_hi);
    ptx::prefetch_tmap(&p.tmB_hi);
    if (SPLIT) {
      ptx::prefetch_tmap(&p.tmA_lo);
      ptx::prefetch_tmap(&p.tmB_lo);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < NST; ++i) {
      ptx::mbar_init(&full[i], 1);
      ptx::mbar_init(&empty[i], 1);
    }
    ptx::mbar_init(b_full, 1);
    ptx::mbar_init(b_empty, 1);
    for (int i = 0; i < NACC; ++i) {
      ptx::mbar_init(&acc_full[i], 1);
      ptx::mbar_init(&acc_empty[i], 4 * Cfg::NQW);
    }
    if (MODE == 1)
      for (int i = 0; i < Cfg::EPI_WARPS * Cfg::NLB; ++i) ptx::mbar_init(&in_bars[i], 1);
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
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int cur_task = -1;
      uint32_t b_gen = 0;   // weight blocks loaded so far
      for (int t = tr.t0; t < tr.t1; ++t) {
        const int row0 = t * TILE_M;
        const int task = p.per_task ? row0 / p.rows_per_task : 0;
        if (task != cur_task) {
          // b_empty completes one phase per finished run of same-task tiles (see the MMA warp)
          if (b_gen > 0) ptx::mbar_wait(b_empty, (b_gen - 1) & 1u);
          ++b_gen;
          ptx::mbar_arrive_expect_tx(b_full, Cfg::B_BYTES);
#pragma unroll
          for (int part = 0; part < Cfg::NSPLIT; ++part)
#pragma unroll
            for (int kc = 0; kc < 4; ++kc)
              ptx::tma_load_2d(sB + (part * 4 + kc) * BN * 128, part ? &p.tmB_lo : &p.tmB_hi, b_full, kc * KCHUNK,
                               task * H + nb * BN);
          cur_task = task;
        }
        for (int s = 0; s < S; ++s)
          for (int part = 0; part < Cfg::NSPLIT; ++part)
            for (int kc = 0; kc < 4; ++kc) {
              ptx::mbar_wait(&empty[stage], phase ^ 1u);
              ptx::mbar_arrive_expect_tx(&full[stage], Cfg::A_STAGE);
              ptx::tma_load_2d(sA + stage * Cfg::A_STAGE, part ? &p.tmA_lo : &p.tmA_hi, &full[stage], kc * KCHUNK,
                               s * p.R + row0);
              if (++stage == NST) { stage = 0; phase ^= 1u; }
            }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    int stage = 0;
    uint32_t phase = 0;
    int cur_task = -1;
    uint32_t b_loads = 0;
    int local = 0;
    for (int t = tr.t0; t < tr.t1; ++t, ++local) {
      const int row0 = t * TILE_M;
      const int task = p.per_task ? row0 / p.rows_per_task : 0;
      const int a = local % NACC;
      ptx::mbar_wait(&acc_empty[a], ((uint32_t(local / NACC)) & 1u) ^ 1u);
      if (task != cur_task) {
        ptx::mbar_wait(b_full, b_loads & 1u);
        ++b_loads;
        cur_task = task;
      }
      ptx::tc_fence_after();
      for (int s = 0; s < S; ++s) {
        const uint32_t d_tmem = tmem_base + uint32_t(a * S * BN + s * BN);
        for (int part = 0; part < Cfg::NSPLIT; ++part)
          for (int kc = 0; kc < 4; ++kc) {
            ptx::mbar_wait(&full[stage], phase);
            ptx::tc_fence_after();
            if (lane == 0) {
              const uint32_t a_addr = ptx::smem_u32(sA + stage * Cfg::A_STAGE);
              const uint32_t bh_addr = ptx::smem_u32(sB + kc * BN * 128);
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) {
                const uint64_t adesc = ptx::umma_smem_desc(a_addr + ks * 32, 16, 1024);
                const uint64_t bdesc = ptx::umma_smem_desc(bh_addr + ks * 32, 16, 1024);
                ptx::umma_bf16(d_tmem, adesc, bdesc, IDESC, (part | kc | ks) ? 1u : 0u);
                if (SPLIT && part == 0) {   // a_hi * b_lo
                  const uint64_t bl = ptx::umma_smem_desc(bh_addr + 4 * BN * 128 + ks * 32, 16, 1024);
                  ptx::umma_bf16(d_tmem, adesc, bl, IDESC, 1u);
                }
              }
              ptx::umma_commit(&empty[stage]);
            }
            __syncwarp();
            if (++stage == NST) { stage = 0; phase ^= 1u; }
          }
      }
      const int next_task = (t + 1 < tr.t1) ? (p.per_task ? (row0 + TILE_M) / p.rows_per_task : 0) : -1;
      if (lane == 0) {
        ptx::umma_commit(&acc_full[a]);
        if (next_task != task) ptx::umma_commit(b_empty);   // weight block may be overwritten
      }
      __syncwarp();
    }
  } else if (warp >= kEpiWarp0) {
    // ===================== epilogue =====================
    const int e = warp - kEpiWarp0;
    const int q = warp & 3;                 // TMEM lane quadrant this warp may touch
    const int chalf = e >> 2;               // which slice of the BN columns
    constexpr int COLS_PER_WARP = BN / Cfg::NQW;
    constexpr int NCH = COLS_PER_WARP / CW;
    WarpOut<CW, Cfg::NBUF> io;
    io.base = ptx::smem_u32(sStg + e * Cfg::NBUF * Cfg::OUT_BUF);
    io.buf_bytes = Cfg::OUT_BUF;
    io.cur = 0;
    io.lane = lane;
    using Seq = BwdLoadSeq<ORDER, D, SPLIT, CW, NCH>;
    WarpIn<CW, Cfg::NLB, Seq> in;
    if constexpr (MODE == 1) {
      in.base = ptx::smem_u32(sIn + e * Cfg::NLB * Cfg::IN_BUF);
      in.buf_bytes = Cfg::IN_BUF;
      in.bars = in_bars + e * Cfg::NLB;
      in.lane = lane;
      in.issued = in.taken = 0;
      in.seq.below_is_first = p.below_is_first;
      in.seq.R = p.R;
      in.seq.t = tr.t0;
      in.seq.t1 = tr.t1;
      in.seq.cc = 0;
      in.seq.pi = 0;
      in.seq.q = q;
      in.seq.colbase = nb * BN + chalf * COLS_PER_WARP;
      in.prime(p);
    }
    int local = 0;
    for (int t = tr.t0; t < tr.t1; ++t, ++local) {
      const int row0 = t * TILE_M;
      const int task = p.per_task ? row0 / p.rows_per_task : 0;
      const int a = local % NACC;
      ptx::mbar_wait(&acc_full[a], (uint32_t(local / NACC)) & 1u);
      ptx::tc_fence_after();
      const int row = row0 + q * 32 + lane;
      for (int cc = 0; cc < NCH; ++cc) {
        const int ctile = chalf * COLS_PER_WARP + cc * CW;      // column inside the BN block
        const uint32_t taddr = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(a * S * BN + ctile);
        const int col0 = nb * BN + ctile;
        io.x = col0;
        io.y = row0 + q * 32;
        if constexpr (MODE == 0) epilogue_forward<ORDER, D, SPLIT, CW, BN, Cfg::NBUF>(p, io, taddr, col0, task);
        if constexpr (MODE == 1) epilogue_backward<ORDER, D, SPLIT, CW, BN, Cfg::NBUF>(p, io, in, taddr, col0, task);
        if constexpr (MODE == 2) {
          float acc[CW];
          ptx::tmem_ld<CW>(taddr, reinterpret_cast<uint32_t*>(acc));
          ptx::tmem_wait_ld();
          float4* d = reinterpret_cast<float4*>(p.raw_out + size_t(row) * H + col0);
#pragma unroll
          for (int i = 0; i < CW / 4; ++i) d[i] = make_float4(acc[4 * i], acc[4 * i + 1], acc[4 * i + 2], acc[4 * i + 3]);
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&acc_empty[a]);
    }
    if (MODE != 2 && lane == 0) ptx::bulk_wait_all();   // this warp's staged stores have left shared memory
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, 512);
  }
}

template <int ORDER, int D, bool SPLIT, int MODE>
cudaError_t launch_one(const RowsGemmParams& p, int num_sms, cudaStream_t stream) {
  using Cfg = RowsCfg<ORDER, D, SPLIT, MODE>;
  constexpr int NB = H / Cfg::BN;
  auto kern = rows_gemm_kernel<ORDER, D, SPLIT, MODE>;
  SIREN_ENSURE_SMEM(kern, Cfg::SMEM);
  const int tiles_m = p.R / TILE_M;
  int G = num_sms / NB;
  if (G > tiles_m) G = tiles_m;
  if (G < 1) G = 1;
  kern<<<G * NB, Cfg::THREADS, Cfg::SMEM, stream>>>(p);
  return cudaGetLastError();
}

template <bool SPLIT, int MODE>
cudaError_t dispatch_order(const RowsGemmParams& p, int order, int d, int num_sms, cudaStream_t stream) {
  // bf16 value layers run inside the fused kernels (mlp_fused_pair.cu / mlp_fused_bwd.cu): on bf16 planes order 0
  // is the raw product of siren_b200_debug_linear only
  if constexpr (SPLIT || MODE == 2)
    if (order == 0) return launch_one<0, 0, SPLIT, MODE>(p, num_sms, stream);
  if constexpr (MODE != 2) {
    if (order == 1 && d == 1) return launch_one<1, 1, SPLIT, MODE>(p, num_sms, stream);
    if (order == 1 && d == 2) return launch_one<1, 2, SPLIT, MODE>(p, num_sms, stream);
    if (order == 1 && d == 3) return launch_one<1, 3, SPLIT, MODE>(p, num_sms, stream);
    if (order == 2 && d == 1) return launch_one<2, 1, SPLIT, MODE>(p, num_sms, stream);
    if (order == 2 && d == 2) return launch_one<2, 2, SPLIT, MODE>(p, num_sms, stream);
    if (order == 2 && d == 3) return launch_one<2, 3, SPLIT, MODE>(p, num_sms, stream);
  }
  return cudaErrorInvalidValue;
}

}  // namespace

// mode: 0 forward, 1 backward, 2 raw
cudaError_t launch_rows_gemm(const RowsGemmParams& p, int mode, int order, int d, bool split, int num_sms,
                             cudaStream_t stream) {
  if (mode == 0) return split ? dispatch_order<true, 0>(p, order, d, num_sms, stream)
                              : dispatch_order<false, 0>(p, order, d, num_sms, stream);
  if (mode == 1) return split ? dispatch_order<true, 1>(p, order, d, num_sms, stream)
                              : dispatch_order<false, 1>(p, order, d, num_sms, stream);
  if (mode == 2) return split ? dispatch_order<true, 2>(p, 0, 0, num_sms, stream)
                              : dispatch_order<false, 2>(p, 0, 0, num_sms, stream);
  return cudaErrorInvalidValue;
}

// columns per staged epilogue store (the host builds the store tensor maps with it)
int rows_gemm_cw(int order, int d, bool split, int mode) {
  const int S = 1 + order * d;
  if (S == 1) return split ? 16 : 32;
  return mode == 1 ? 16 : 32;
}

// box rows of the weight tensor map for a given configuration (the host builds tmB with it)
int rows_gemm_bn(int order, int d, bool split, int mode) {
  const int S = 1 + order * d;
  return (S == 1) ? (split ? 128 : 256) : (S <= 2 ? 128 : (S <= 4 && mode == 0 && !split) ? 128 : 64);
}

}  // namespace siren
