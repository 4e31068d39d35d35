// C ABI of libsiren_b200.so (declared in include/siren_b200.h): argument checks, the HBM
// workspace layout, TMA tensor maps and the launch sequence of one forward / backward.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <unordered_map>
#include <utility>

#include "../../include/siren_b200.h"
#include "simt.h"

using namespace siren;

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
#define CUDA_TRY(expr)                                                                         \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) return fail(SIREN_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(_e)); \
  } while (0)

constexpr int MAX_HIDDEN = 8;

// ---- optional per-kernel timing (siren_b200_profile_begin/end): CUDA events around every launch
struct ProfRec {
  const char* name;
  cudaEvent_t a, b;
};
constexpr int PROF_MAX = 8192;
// process-wide (autograd runs the backward on its own thread); guarded by g_prof_mu
bool g_prof_on = false;
int g_prof_n = 0;
ProfRec g_prof[PROF_MAX];
std::mutex g_prof_mu;

struct ProfScope {
  cudaStream_t s;
  int idx;
  ProfScope(const char* name, cudaStream_t stream) : s(stream), idx(-1) {
    if (!g_prof_on) return;
    std::lock_guard<std::mutex> lk(g_prof_mu);
    if (g_prof_n < PROF_MAX) {
      idx = g_prof_n++;
      g_prof[idx].name = name;
      cudaEventCreate(&g_prof[idx].a);
      cudaEventCreate(&g_prof[idx].b);
      cudaEventRecord(g_prof[idx].a, s);
    }
  }
  ~ProfScope() {
    if (idx >= 0) cudaEventRecord(g_prof[idx].b, s);
  }
};
#define LAUNCH_N(name, expr)        \
  do {                              \
    ProfScope _ps(name, stream);    \
    CUDA_TRY(expr);                 \
  } while (0)

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

// Tensor maps are pure functions of (base address, element size, rows, box): a step re-encodes the same ~15 maps on
// every call (cuTensorMapEncodeTiled costs 1-2 us each on the host), so they are kept in a small process-wide cache.
// An address that is freed and reused with the same shape yields the same map, so entries never go stale.
struct MapKey {
  const void* base;
  uint64_t rows;
  uint32_t box_cols, box_rows, elem, promo;
  bool operator==(const MapKey& o) const {
    return base == o.base && rows == o.rows && box_cols == o.box_cols && box_rows == o.box_rows && elem == o.elem &&
           promo == o.promo;
  }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    size_t h = reinterpret_cast<size_t>(k.base) * 0x9E3779B97F4A7C15ull;
    h ^= (k.rows + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2));
    h ^= (size_t(k.box_cols) << 40) ^ (size_t(k.box_rows) << 20) ^ (size_t(k.elem) << 8) ^ k.promo;
    return h;
  }
};
std::unordered_map<MapKey, CUtensorMap, MapKeyHash> g_maps;
std::mutex g_maps_mu;
constexpr size_t MAP_CACHE_MAX = 4096;      // cleared wholesale when full (workspaces come and go with batch shapes)

int encode_cached(CUtensorMap* m, const void* base, int elem, uint64_t rows, uint32_t box_cols, uint32_t box_rows,
                  CUtensorMapSwizzle sw, CUtensorMapL2promotion promo) {
  const MapKey key{base, rows, box_cols, box_rows, uint32_t(elem), uint32_t(promo)};
  {
    std::lock_guard<std::mutex> lk(g_maps_mu);
    auto it = g_maps.find(key);
    if (it != g_maps.end()) {
      *m = it->second;
      return SIREN_OK;
    }
  }
  EncodeTiledFn fn = encode_fn();
  if (!fn) return fail(SIREN_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {uint64_t(H), rows};
  cuuint64_t strides[1] = {uint64_t(H) * uint64_t(elem)};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, elem == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                  const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, promo,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(SIREN_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", int(r));
  std::lock_guard<std::mutex> lk(g_maps_mu);
  if (g_maps.size() >= MAP_CACHE_MAX) g_maps.clear();
  g_maps.emplace(key, *m);
  return SIREN_OK;
}

// bf16 matrix [rows, 256] row-major; box = 64 columns x box_rows rows, 128-byte swizzle
int make_map(CUtensorMap* m, const void* base, uint64_t rows, uint32_t box_rows) {
  return encode_cached(m, base, 2, rows, 64, box_rows, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
}

// [rows, 256] plane of bf16 (elem = 2) or fp32 (elem = 4); box = box_cols x box_rows with the swizzle
// that matches the box's row width (32 / 64 / 128 bytes) -- the epilogue staging uses the same pattern
int make_map_ex(CUtensorMap* m, const void* base, int elem, uint64_t rows, uint32_t box_cols, uint32_t box_rows) {
  const uint32_t row_bytes = box_cols * uint32_t(elem);
  CUtensorMapSwizzle sw = CU_TENSOR_MAP_SWIZZLE_NONE;
  if (row_bytes == 128) sw = CU_TENSOR_MAP_SWIZZLE_128B;
  else if (row_bytes == 64) sw = CU_TENSOR_MAP_SWIZZLE_64B;
  else if (row_bytes == 32) sw = CU_TENSOR_MAP_SWIZZLE_32B;
  else return fail(SIREN_ERR_INVALID, "unsupported staged row width %u", row_bytes);
  return encode_cached(m, base, elem, rows, box_cols, box_rows, sw, CU_TENSOR_MAP_L2_PROMOTION_NONE);
}

int num_sms() {
  static int cached[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct Layout {
  int S, Ls, Tw, R, n_pad;
  bool split;
  size_t plane_op, plane_st;
  size_t wk_hi[MAX_HIDDEN], wk_lo[MAX_HIDDEN], wt_hi[MAX_HIDDEN], wt_lo[MAX_HIDDEN];
  size_t act_hi[MAX_HIDDEN + 1], act_lo[MAX_HIDDEN + 1], c[MAX_HIDDEN + 1], jz[MAX_HIDDEN + 1];
  size_t adj_hi[MAX_HIDDEN + 1], adj_lo[MAX_HIDDEN + 1];
  size_t w0k;      // first-layer weights as a bf16 MMA operand [Tw*256][64 * nkc0] (fused forward, d > 4)
  size_t feat;     // d > 16: the first layer's input plane (bf16), written by the fused forward for the dW_0 items
  // d > 16 on the per-layer fp32-parity path: the first layer runs as one more hidden layer on padded operands
  size_t feat_lo, w0p_hi, w0p_lo, dw0pad;
  size_t rag;      // scenes of different sizes: the prefix tables (simt.h ragged_tables)
  size_t gyscr;    // [tasks][n][d_out] floats: the masked output adjoint of a data-consistency backward off the fused path
  int nkc0;        // 64-wide K chunks of the first layer (fused forward, d > 4)
  size_t total;             // bytes without the optional layer-0 adjoint plane of the fused path
  size_t total_with_adj0;   // ... with it (a backward that is asked for gcoords needs it)
};

// bf16 mode without coordinate jets: the whole-MLP kernels on CTA pairs (mlp_fused_pair.cu / mlp_fused_bwd.cu, one
// fp16 phase plane per hidden layer), at every depth check_desc accepts
static_assert(MAX_FUSED_HIDDEN_SMEM >= MAX_HIDDEN, "the fused kernels must take every n_hidden the library accepts");
bool fused_path(const siren_desc_t* d) { return d->precision == SIREN_PREC_BF16 && d->deriv_order == 0; }

int check_desc(const siren_desc_t* d) {
  if (!d) return fail(SIREN_ERR_INVALID, "null descriptor");
  if (d->hidden != H) return fail(SIREN_ERR_UNSUPPORTED, "hidden_features=%d (native kernels serve 256)", d->hidden);
  if (d->n_hidden < 1 || d->n_hidden > MAX_HIDDEN)
    return fail(SIREN_ERR_UNSUPPORTED, "num_hidden_layers=%d outside 1..%d", d->n_hidden, MAX_HIDDEN);
  if (d->d_in < 1 || d->d_in > 256) return fail(SIREN_ERR_UNSUPPORTED, "in_features=%d outside 1..256", d->d_in);
  if (d->d_in > 16 && !(fused_path(d) || (d->precision == SIREN_PREC_FP32_PARITY && d->deriv_order == 0)))
    return fail(SIREN_ERR_UNSUPPORTED, "in_features=%d: 17..256 inputs are served by the bf16 and the fp32-parity "
                "value paths (deriv_order 0)", d->d_in);
  if (d->d_out < 1 || d->d_out > 8) return fail(SIREN_ERR_UNSUPPORTED, "out_features=%d outside 1..8", d->d_out);
  if (d->deriv_order < 0 || d->deriv_order > 2) return fail(SIREN_ERR_INVALID, "deriv_order=%d", d->deriv_order);
  if (d->deriv_order > 0 && d->d_in > 3)
    return fail(SIREN_ERR_UNSUPPORTED, "coordinate derivatives need in_features <= 3 (got %d)", d->d_in);
  if (d->tasks < 1 || d->n_coords < 1) return fail(SIREN_ERR_INVALID, "empty batch");
  if (d->precision != SIREN_PREC_FP32_PARITY && d->precision != SIREN_PREC_BF16)
    return fail(SIREN_ERR_INVALID, "precision=%d", d->precision);
  const long n_pad = (d->n_coords + TILE_M - 1) / TILE_M * TILE_M;
  const long S = 1 + d->deriv_order * d->d_in;
  if (n_pad * d->tasks * S >= (1L << 31)) return fail(SIREN_ERR_UNSUPPORTED, "batch too large for 32-bit rows");
  return SIREN_OK;
}

// Planes are laid out per PATH.  The per-layer kernels (fp32-parity mode, jets) keep
// act / c / jz / adj for every layer.  The fused bf16 path keeps only what crosses a kernel boundary: one stash plane
// c[l] (the layer's signed sine, fp16: common.cuh) and one adjoint plane adj[l] per HIDDEN sine layer l >= 1 (layer 0
// too for a wide first layer, d > 4, whose dW / db come from first_bwd) and -- LAST, counted only on request -- the
// layer-0 adjoint a backward call with gcoords stores (narrow first layer).  Planes a path never touches alias
// c[NH], so a tensor map built on them is harmless.
// rag_rows > 0: scenes of different sizes, whose planes have rag_rows rows in all (each scene's padded to 128)
void make_layout(const siren_desc_t* d, Layout* L, long rag_rows = 0) {
  L->split = d->precision == SIREN_PREC_FP32_PARITY;
  L->S = 1 + d->deriv_order * d->d_in;
  L->Ls = d->n_hidden + 1;
  L->Tw = d->per_task ? d->tasks : 1;
  L->n_pad = int((d->n_coords + TILE_M - 1) / TILE_M * TILE_M);
  L->R = rag_rows > 0 ? int(rag_rows) : L->n_pad * d->tasks;
  L->plane_op = size_t(L->R) * H * 2;
  L->plane_st = size_t(L->R) * H * (L->split ? 4 : 2);
  size_t off = 0;
  auto take = [&](size_t bytes) {
    size_t o = off;
    off = align_up(off + bytes, 1024);
    return o;
  };
  const size_t wbytes = size_t(L->Tw) * H * H * 2;
  for (int l = 0; l < d->n_hidden; ++l) {
    L->wk_hi[l] = take(wbytes);
    L->wk_lo[l] = L->split ? take(wbytes) : L->wk_hi[l];
    L->wt_hi[l] = take(wbytes);
    L->wt_lo[l] = L->split ? take(wbytes) : L->wt_hi[l];
  }
  L->nkc0 = d->d_in > 16 ? (d->d_in + 63) / 64 : 1;
  L->w0k = take(size_t(L->Tw) * H * 64 * L->nkc0 * 2);
  const bool fusedp = fused_path(d);
  const int NH = d->n_hidden;
  const bool wide = d->d_in > 4;
  const size_t shared_c = fusedp ? take(L->plane_st) : 0;      // = c[NH]; also the alias of every untouched plane
  for (int l = 0; l < L->Ls; ++l) {
    const bool need_act = !fusedp;
    const bool need_c = !fusedp || l >= 1 || wide;
    const bool need_adj = !fusedp || l >= 1 || wide;
    L->act_hi[l] = need_act ? take(L->S * L->plane_op) : shared_c;
    L->act_lo[l] = need_act && L->split ? take(L->S * L->plane_op) : L->act_hi[l];
    L->c[l] = (fusedp && l == NH) ? shared_c : need_c ? take(L->plane_st) : shared_c;
    L->jz[l] = (L->S > 1 && l >= 1) ? take((L->S - 1) * L->plane_st) : L->c[l];
    L->adj_hi[l] = need_adj ? take(L->S * L->plane_op) : shared_c;
    L->adj_lo[l] = need_adj && L->split ? take(L->S * L->plane_op) : L->adj_hi[l];
  }
  L->feat = (fusedp && d->d_in > 16) ? take(L->plane_op) : 0;
  L->feat_lo = L->w0p_hi = L->w0p_lo = L->dw0pad = 0;
  if (!fusedp && d->d_in > 16) {
    L->feat = take(L->plane_op);
    L->feat_lo = take(L->plane_op);
    L->w0p_hi = take(wbytes);
    L->w0p_lo = take(wbytes);
    L->dw0pad = take(size_t(L->Tw) * H * H * 4);
  }
  L->rag = rag_rows > 0 ? take(size_t(ragged_table_ints(d->tasks)) * 4) : 0;
  L->gyscr = rag_rows > 0 ? 0 : take(size_t(d->tasks) * d->n_coords * d->d_out * 4);      // (no two-launch ragged step)
  L->total = off;
  L->total_with_adj0 = off;
  if (fusedp && !wide) {      // the optional layer-0 adjoint plane: behind everything else
    L->adj_hi[0] = L->adj_lo[0] = take(L->plane_op);
    L->total_with_adj0 = off;
  }
}

// siren_b200_forward_backward_mse as ONE kernel (mlp_fused_step.cu): the fused path's shapes the trainer takes, with an
// outermost linear the forward fuses (d_out <= 2) and a first layer without a phase plane (d_in <= 4).
// SIREN_FUSED_STEP=0 runs the same entry as the two launches of forward_mse and backward, for A/B.
bool fused_step(const siren_desc_t* d) {
  const char* e = getenv("SIREN_FUSED_STEP");
  return fused_path(d) && !(e && e[0] == '0') && d->n_hidden <= MAX_FUSED_STEP_HIDDEN && d->d_in <= 4 &&
         d->d_out <= 2;
}

template <typename T>
T* at(const void* ws, size_t off) {
  return reinterpret_cast<T*>(const_cast<char*>(reinterpret_cast<const char*>(ws)) + off);
}

}  // namespace

extern "C" {

int siren_b200_version(void) { return SIREN_B200_VERSION; }
const char* siren_b200_last_error(void) { return g_err; }

int siren_b200_device_ok(void) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return fail(SIREN_ERR_CUDA, "no CUDA device");
  int major = 0;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (major != 10) return fail(SIREN_ERR_UNSUPPORTED, "compute capability %d.x: this library is sm_100a only", major);
  return SIREN_OK;
}

size_t siren_b200_workspace_bytes_ex(const siren_desc_t* desc, int want_gcoords) {
  if (check_desc(desc) != SIREN_OK) return 0;
  Layout L;
  make_layout(desc, &L);
  return want_gcoords ? L.total_with_adj0 : L.total;
}

size_t siren_b200_workspace_bytes(const siren_desc_t* desc) { return siren_b200_workspace_bytes_ex(desc, 1); }

// bf16 (hi, lo) copies of the hidden weights, as stored and transposed, into the workspace
static int prep_impl(const siren_desc_t* desc, const Layout& L, const float* const* W, void* ws, cudaStream_t stream) {
  PrepParams pp;
  memset(&pp, 0, sizeof(pp));
  for (int l = 0; l < desc->n_hidden; ++l) {
    pp.W[l] = W[l + 1];
    pp.k_hi[l] = at<bf16>(ws, L.wk_hi[l]); pp.k_lo[l] = at<bf16>(ws, L.wk_lo[l]);
    pp.t_hi[l] = at<bf16>(ws, L.wt_hi[l]); pp.t_lo[l] = at<bf16>(ws, L.wt_lo[l]);
  }
  pp.n_layers = desc->n_hidden; pp.tasks = L.Tw; pp.split = L.split ? 1 : 0;
  // fused bf16 path: the dgrad chain reads w0 W^T, so that its accumulator times cos(theta) is the adjoint
  pp.scale_t = fused_path(desc) ? desc->w0 : 1.f;
  pp.k_f16 = fused_path(desc) ? 1 : 0;      // ... and its forward multiplies fp16 operands
  LAUNCH_N("prep_weights", launch_prep_weights(pp, stream));
  return SIREN_OK;
}

// Fourier-feature prologue (siren_b200_forward_ff / _backward_ff): the first layer's inputs are built on chip
static int check_fourier(const siren_desc_t* d, const siren_fourier_t* ff) {
  if (!ff) return SIREN_OK;
  if (!ff->B) return fail(SIREN_ERR_INVALID, "fourier: null B");
  if (ff->raw_dim < 1 || ff->raw_dim > 3) return fail(SIREN_ERR_UNSUPPORTED, "fourier: raw_dim=%d outside 1..3", ff->raw_dim);
  if (ff->n_features < 3 || ff->n_features > 128)
    return fail(SIREN_ERR_UNSUPPORTED, "fourier: n_features=%d outside 3..128 (in_features = 2 F must be 6..256)", ff->n_features);
  if (d->d_in != 2 * ff->n_features)
    return fail(SIREN_ERR_INVALID, "fourier: in_features=%d but 2 * n_features=%d", d->d_in, 2 * ff->n_features);
  if (d->deriv_order != 0) return fail(SIREN_ERR_UNSUPPORTED, "fourier: value path only (deriv_order 0)");
  return SIREN_OK;
}
// k-space data consistency behind the outermost linear (siren_b200_forward_dc / _backward_dc)
static int check_dc(const siren_desc_t* d, const siren_dc_t* dc, bool need_k0) {
  if (!dc) return SIREN_OK;
  if (!dc->mask || (need_k0 && !dc->k0)) return fail(SIREN_ERR_INVALID, "data consistency: null k0 / mask");
  if (d->deriv_order != 0) return fail(SIREN_ERR_UNSUPPORTED, "data consistency: value path only (deriv_order 0)");
  if (!(dc->noise_lvl >= 0.f)) return fail(SIREN_ERR_INVALID, "data consistency: noise_lvl=%g", double(dc->noise_lvl));
  return SIREN_OK;
}
static DcSpec dc_spec(const siren_dc_t* dc) {
  DcSpec s;
  s.k0 = dc ? dc->k0 : nullptr;
  s.mask = dc ? dc->mask : nullptr;
  s.pull = dc ? (dc->noise_lvl > 0.f ? dc->noise_lvl / (1.f + dc->noise_lvl) : 1.f) : 0.f;
  s.cf = dc ? (dc->channels_first ? 1 : 0) : 0;
  return s;
}
static FourierSpec fourier_spec(const siren_fourier_t* ff) {
  FourierSpec f;
  f.B = ff ? ff->B : nullptr;
  f.F = ff ? ff->n_features : 0;
  f.raw = ff ? ff->raw_dim : 0;
  return f;
}

// SIREN_FUSED_DBG: spread of the CTAs' run times (globaltimer) of a fused kernel
static void print_cta_spread(const char* what, const long long* host) {
  long long t0 = 0, emin = 0, emax = 0, dsum = 0;
  int n = 0;
  for (int i = 0; i < 512; ++i)
    if (host[2048 + 2 * i] && (!t0 || host[2048 + 2 * i] < t0)) t0 = host[2048 + 2 * i];
  for (int i = 0; i < 512; ++i) {
    if (!host[2048 + 2 * i]) continue;
    const long long en = host[2048 + 2 * i + 1] - t0;
    if (!n || en < emin) emin = en;
    if (!n || en > emax) emax = en;
    dsum += en;
    ++n;
  }
  if (n) fprintf(stderr, "[%s dbg] %d CTAs end %lld..%lld ns after the first start (mean %lld)\n", what, n, emin, emax, dsum / n);
}

// The step of scenes of different sizes (siren_b200_forward_backward_mse_ragged): plane rows in all, units of the
// one-kernel step, and the per-scene loss sums
struct Ragged {
  long rows;
  int units;
  float* task_loss;
};

// mse_gt != null: the loss is image_mse; gy = 2 w (y - gt) and w sum (y - gt)^2 (into loss4[1]) come out of the forward
// itself -- inside the fused kernel when it also forms y, by one mse_grad launch behind the forward otherwise.
static int forward_impl(const siren_desc_t* desc, const float* coords, const float* const* W, const float* const* b,
                        float* y, float* J, float* D, void* ws, void* stream_, bool stash, bool weights_ready = false,
                        const float* mse_gt = nullptr, float mse_w = 0.f, float* mse_gy = nullptr, float* loss4 = nullptr,
                        const siren_fourier_t* ff = nullptr, const siren_dc_t* dc = nullptr,
                        const void* const* ext_wk = nullptr, MlpFwdParams* step_fwd = nullptr,
                        const Ragged* rg = nullptr) {
  int rc = check_desc(desc);
  if (rc) return rc;
  if ((rc = check_fourier(desc, ff))) return rc;
  if ((rc = check_dc(desc, dc, true))) return rc;
  if (!coords || !W || !b || !y || !ws) return fail(SIREN_ERR_INVALID, "null pointer argument");
  if (desc->deriv_order >= 1 && !J) return fail(SIREN_ERR_INVALID, "J required for deriv_order >= 1");
  if (desc->deriv_order >= 2 && !D) return fail(SIREN_ERR_INVALID, "D required for deriv_order == 2");
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  Layout L;
  make_layout(desc, &L, rg ? rg->rows : 0);
  const int sms = num_sms();
  const bool split = L.split;
  const int order = desc->deriv_order, d = desc->d_in;

  // ext_wk: the hidden weights arrive as ready-made operands (siren_b200_hyper_head wrote them): nothing to convert
  if (ext_wk && !fused_path(desc))
    return fail(SIREN_ERR_UNSUPPORTED, "prepared weight operands are taken by the fused bf16 path only");
  if (ext_wk)
    for (int l = 0; l < desc->n_hidden; ++l)
      if (!ext_wk[l]) return fail(SIREN_ERR_INVALID, "prepared weight operand %d is null", l);
  if (!weights_ready && !ext_wk)
    if ((rc = prep_impl(desc, L, W, ws, stream))) return rc;

  if (fused_path(desc)) {
    // whole-MLP kernel: activations stay in shared memory / TMEM from the coordinates to y.  (When the outermost
    // linear is too wide to fuse, d_out > 2, inference also leaves the planes: last_fwd reads the top one.)
    const bool fuse_last = desc->d_out <= 2;
    stash = stash || !fuse_last;
    MlpFwdParams m;
    memset(&m, 0, sizeof(m));
    for (int l = 0; l < desc->n_hidden; ++l) {
      if ((rc = make_map(&m.tmW[l], ext_wk ? ext_wk[l] : at<void>(ws, L.wk_hi[l]), uint64_t(L.Tw) * H, 128))) return rc;
      m.bias[l] = b[l + 1];
    }
    if (stash) {
      // the stash of this path: ONE fp16 plane per hidden sine layer, its signed sine (common.cuh), which is the next
      // layer's operand tile stored as it stands (box 64 columns x 32 rows: a warp's slice), kept where the
      // per-layer path keeps the cosine (c[l]).  A narrow first layer, d <= 4, leaves no plane: the backward
      // recomputes its phase from the coordinates.
      for (int l = d <= 4 ? 1 : 0; l <= desc->n_hidden; ++l)
        if ((rc = make_map(&m.tmAct[l], at<void>(ws, L.c[l]), L.R, 32))) return rc;
    }
    m.x = coords; m.W0 = W[0]; m.b0 = b[0];
    m.ff = fourier_spec(ff);
    if (d > 4) {
      // wide first layer: on the tensor core as well, from a split-bf16 copy of W0 (one 64-wide K chunk)
      m.l0_mma = 1;
      LAUNCH_N("prep_first", launch_prep_first(W[0], at<bf16>(ws, L.w0k), L.Tw, d, stream));
      EncodeTiledFn fn = encode_fn();
      if (!fn) return fail(SIREN_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
      m.nkc0 = L.nkc0;
      if (d > 16 && stash)
        if ((rc = make_map(&m.tmFeat, at<void>(ws, L.feat), L.R, 32))) return rc;
      cuuint64_t dims[2] = {uint64_t(64 * L.nkc0), uint64_t(L.Tw) * H};
      cuuint64_t strides[1] = {uint64_t(64 * L.nkc0) * 2};
      cuuint32_t box[2] = {64, 128};
      cuuint32_t estr[2] = {1, 1};
      CUresult r = fn(&m.tmW0, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, at<void>(ws, L.w0k), dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) return fail(SIREN_ERR_CUDA, "cuTensorMapEncodeTiled (first layer) failed (%d)", int(r));
    }
    m.n_hidden = desc->n_hidden; m.rows_per_task = L.n_pad; m.per_task = desc->per_task; m.tasks = L.R / L.n_pad;
    m.n = int(desc->n_coords); m.d = d; m.o = desc->d_out; m.w0 = desc->w0;
    if (fuse_last) {
      m.fuse_last = 1;
      m.WL = W[desc->n_hidden + 1]; m.bL = b[desc->n_hidden + 1]; m.y = y;
      if (mse_gt) {
        m.gt = mse_gt; m.gy = mse_gy; m.loss_weight = mse_w; m.loss_acc = loss4 ? loss4 + 1 : nullptr;
        mse_gt = nullptr;      // done in the kernel
      }
      if (dc) {
        m.dc = dc_spec(dc);
        dc = nullptr;          // done in the kernel
      }
    }
    if (step_fwd) {            // the training step's single kernel takes it from here (backward_impl)
      *step_fwd = m;
      return SIREN_OK;
    }
    // developer aid: SIREN_FUSED_DBG=1 dumps a clock64 trace of the first CTA pair (tools/fused_trace.py)
    static long long* dbg_buf = nullptr;
    const bool dbg = getenv("SIREN_FUSED_DBG") != nullptr;
    if (dbg) {
      if (!dbg_buf) cudaMalloc(&dbg_buf, 4096 * sizeof(long long));
      cudaMemsetAsync(dbg_buf, 0, 4096 * sizeof(long long), stream);
      m.dbg = dbg_buf;
    }
    LAUNCH_N("mlp_fused_fwd", launch_mlp_fused_pair(m, stash, sms, stream));
    if (dbg) {
      static long long host[4096];
      cudaStreamSynchronize(stream);
      cudaMemcpy(host, dbg_buf, sizeof(host), cudaMemcpyDeviceToHost);
      const long long t0 = host[0];
      print_cta_spread("fused fwd", host);
      for (int pr = 0; pr < 3; ++pr)
        for (int l = 0; l <= desc->n_hidden; ++l) {
          fprintf(stderr, "[fused dbg] pair %d layer %d:", pr, l);
          for (int k = 0; k < 8; ++k) fprintf(stderr, " %lld", host[(pr * 8 + l) * 8 + k] ? host[(pr * 8 + l) * 8 + k] - t0 : -1);
          fprintf(stderr, "\n");
        }
    }
    if (!fuse_last) {
      LastParams lp;
      memset(&lp, 0, sizeof(lp));
      lp.W = W[desc->n_hidden + 1]; lp.b = b[desc->n_hidden + 1];
      lp.phase = at<void>(ws, L.c[desc->n_hidden]);      // the top layer's signed sine
      lp.y = y;
      lp.R = L.R; lp.n_pad = L.n_pad; lp.n = int(desc->n_coords); lp.d = d; lp.o = desc->d_out; lp.order = 0;
      lp.per_task = desc->per_task; lp.w0 = desc->w0;
      LAUNCH_N("last_fwd", launch_last_fwd(lp, split, sms, stream));
    }
    if (dc) LAUNCH_N("dc_blend", launch_dc_blend(y, dc_spec(dc), desc->tasks, int(desc->n_coords), desc->d_out, sms, stream));
    if (mse_gt)
      LAUNCH_N("mse_grad", launch_mse_grad(y, mse_gt, mse_gy, long(desc->tasks) * desc->n_coords * desc->d_out, mse_w,
                                           loss4 ? loss4 + 1 : nullptr, sms, stream));
    if (mse_gt && dc)
      LAUNCH_N("dc_grad", launch_dc_grad(mse_gy, mse_gy, dc_spec(dc), desc->tasks, int(desc->n_coords), desc->d_out, sms, stream));
    return SIREN_OK;
  }
  // the per-layer kernels: fp32-parity mode and the jet paths
  FirstParams fp;
  memset(&fp, 0, sizeof(fp));
  fp.x = coords; fp.W = W[0]; fp.b = b[0];
  fp.act_hi = at<bf16>(ws, L.act_hi[0]); fp.act_lo = at<bf16>(ws, L.act_lo[0]);
  fp.c = at<void>(ws, L.c[0]);
  fp.R = L.R; fp.n_pad = L.n_pad; fp.n = int(desc->n_coords); fp.d = d; fp.order = order;
  fp.per_task = desc->per_task; fp.w0 = desc->w0;
  fp.ff = fourier_spec(ff);
  const int bn = rows_gemm_bn(order, order ? d : 0, split, 0);
  if (d > 16) {
    // wide first layer, fp32-parity mode: the inputs (or their Fourier features) as padded hi + lo planes, W_0 padded
    // to 256 columns, and the layer itself through the hidden-layer kernel
    FirstParams fz = fp;
    fz.act_hi = at<bf16>(ws, L.feat); fz.act_lo = at<bf16>(ws, L.feat_lo);
    LAUNCH_N("featurize", launch_featurize(fz, sms, stream));
    LAUNCH_N("pad_w0", launch_pad_w0(W[0], at<bf16>(ws, L.w0p_hi), at<bf16>(ws, L.w0p_lo), d, long(L.Tw) * H, sms, stream));
    RowsGemmParams p;
    memset(&p, 0, sizeof(p));
    if ((rc = make_map(&p.tmA_hi, at<void>(ws, L.feat), L.R, TILE_M))) return rc;
    if ((rc = make_map(&p.tmA_lo, at<void>(ws, L.feat_lo), L.R, TILE_M))) return rc;
    if ((rc = make_map(&p.tmB_hi, at<void>(ws, L.w0p_hi), uint64_t(L.Tw) * H, bn))) return rc;
    if ((rc = make_map(&p.tmB_lo, at<void>(ws, L.w0p_lo), uint64_t(L.Tw) * H, bn))) return rc;
    p.R = L.R; p.rows_per_task = L.n_pad; p.per_task = desc->per_task; p.w0 = desc->w0;
    p.bias = b[0];
    const int cw = rows_gemm_cw(0, 0, split, 0);
    if ((rc = make_map_ex(&p.tmO_hi, at<void>(ws, L.act_hi[0]), 2, L.R, cw, 32))) return rc;
    if ((rc = make_map_ex(&p.tmO_lo, at<void>(ws, L.act_lo[0]), 2, L.R, cw, 32))) return rc;
    if ((rc = make_map_ex(&p.tmC, at<void>(ws, L.c[0]), 4, L.R, cw, 32))) return rc;
    if ((rc = make_map_ex(&p.tmJ, at<void>(ws, L.jz[0]), 4, L.R, cw, 32))) return rc;
    LAUNCH_N("hidden_fwd", launch_rows_gemm(p, 0, 0, 0, split, sms, stream));
  } else {
    LAUNCH_N("first_fwd", launch_first_fwd(fp, split, sms, stream));
  }

  for (int l = 1; l <= desc->n_hidden; ++l) {
    RowsGemmParams p;
    memset(&p, 0, sizeof(p));
    if ((rc = make_map(&p.tmA_hi, at<void>(ws, L.act_hi[l - 1]), uint64_t(L.S) * L.R, TILE_M))) return rc;
    if ((rc = make_map(&p.tmA_lo, at<void>(ws, L.act_lo[l - 1]), uint64_t(L.S) * L.R, TILE_M))) return rc;
    if ((rc = make_map(&p.tmB_hi, at<void>(ws, L.wk_hi[l - 1]), uint64_t(L.Tw) * H, bn))) return rc;
    if ((rc = make_map(&p.tmB_lo, at<void>(ws, L.wk_lo[l - 1]), uint64_t(L.Tw) * H, bn))) return rc;
    p.R = L.R; p.rows_per_task = L.n_pad; p.per_task = desc->per_task; p.w0 = desc->w0;
    p.bias = b[l];
    {
      const int cw = rows_gemm_cw(order, order ? d : 0, split, 0);
      const int se = split ? 4 : 2;      // stash element size
      if ((rc = make_map_ex(&p.tmO_hi, at<void>(ws, L.act_hi[l]), 2, uint64_t(L.S) * L.R, cw, 32))) return rc;
      if ((rc = make_map_ex(&p.tmO_lo, at<void>(ws, L.act_lo[l]), 2, uint64_t(L.S) * L.R, cw, 32))) return rc;
      if ((rc = make_map_ex(&p.tmC, at<void>(ws, L.c[l]), se, L.R, cw, 32))) return rc;
      if ((rc = make_map_ex(&p.tmJ, at<void>(ws, L.jz[l]), se, uint64_t(L.S > 1 ? L.S - 1 : 1) * L.R, cw, 32))) return rc;
    }
    LAUNCH_N("hidden_fwd", launch_rows_gemm(p, 0, order, order ? d : 0, split, sms, stream));
  }

  LastParams lp;
  memset(&lp, 0, sizeof(lp));
  const int top = desc->n_hidden;
  lp.W = W[desc->n_hidden + 1]; lp.b = b[desc->n_hidden + 1];
  lp.act_hi = at<bf16>(ws, L.act_hi[top]); lp.act_lo = at<bf16>(ws, L.act_lo[top]);
  lp.y = y; lp.J = J; lp.Dd = D;
  lp.R = L.R; lp.n_pad = L.n_pad; lp.n = int(desc->n_coords); lp.d = d; lp.o = desc->d_out; lp.order = order;
  lp.per_task = desc->per_task; lp.w0 = desc->w0;
  LAUNCH_N("last_fwd", launch_last_fwd(lp, split, sms, stream));
  if (dc) LAUNCH_N("dc_blend", launch_dc_blend(y, dc_spec(dc), desc->tasks, int(desc->n_coords), desc->d_out, sms, stream));
  if (mse_gt)
    LAUNCH_N("mse_grad", launch_mse_grad(y, mse_gt, mse_gy, long(desc->tasks) * desc->n_coords * desc->d_out, mse_w,
                                         loss4 ? loss4 + 1 : nullptr, sms, stream));
  if (mse_gt && dc)
    LAUNCH_N("dc_grad", launch_dc_grad(mse_gy, mse_gy, dc_spec(dc), desc->tasks, int(desc->n_coords), desc->d_out, sms, stream));
  return SIREN_OK;
}

int siren_b200_forward(const siren_desc_t* desc, const float* coords, const float* const* W, const float* const* b,
                       float* y, float* J, float* D, void* ws, void* stream_) {
  return forward_impl(desc, coords, W, b, y, J, D, ws, stream_, true);
}

int siren_b200_forward_infer(const siren_desc_t* desc, const float* coords, const float* const* W,
                             const float* const* b, float* y, void* ws, void* stream_) {
  if (desc && desc->deriv_order != 0) return fail(SIREN_ERR_INVALID, "forward_infer is value-only (deriv_order 0)");
  return forward_impl(desc, coords, W, b, y, nullptr, nullptr, ws, stream_, false);
}

static int backward_impl(const siren_desc_t* desc, const float* coords, const float* const* W, const float* const* b,
                         const void* ws, const float* gy, const float* gJ, const float* gD, float* const* dW,
                         float* const* db, float* gcoords, int accumulate, void* stream_, const siren_fourier_t* ff,
                         const siren_dc_t* dc = nullptr, const void* const* ext_wt = nullptr,
                         const MlpFwdParams* step_fwd = nullptr, const Ragged* rg = nullptr) {
  int rc = check_desc(desc);
  if (rc) return rc;
  if ((rc = check_fourier(desc, ff))) return rc;
  if ((rc = check_dc(desc, dc, false))) return rc;
  if (ext_wt && !fused_path(desc))
    return fail(SIREN_ERR_UNSUPPORTED, "prepared weight operands are taken by the fused bf16 path only");
  if (ext_wt)
    for (int l = 0; l < desc->n_hidden; ++l)
      if (!ext_wt[l]) return fail(SIREN_ERR_INVALID, "prepared weight operand %d is null", l);
  if (ff && gcoords) return fail(SIREN_ERR_UNSUPPORTED, "fourier: no gradient w.r.t. the raw coordinates");
  if (desc->d_in > 16 && gcoords) return fail(SIREN_ERR_UNSUPPORTED, "in_features=%d: no coordinate gradient above 16 inputs", desc->d_in);
  if (!coords || !W || !b || !ws || (!gy && !step_fwd) || !dW || !db) return fail(SIREN_ERR_INVALID, "null pointer argument");
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  Layout L;
  make_layout(desc, &L, rg ? rg->rows : 0);
  const int sms = num_sms();
  const bool split = L.split;
  const int order = desc->deriv_order, d = desc->d_in, o = desc->d_out;
  const int nl = desc->n_hidden + 2;

  if (!accumulate) {      // every parameter gradient cleared by one launch (ten memset nodes otherwise)
    float* ptrs[20];
    long counts[20];
    for (int l = 0; l < nl; ++l) {
      const long fin = l == 0 ? d : H, fout = l == nl - 1 ? o : H;
      ptrs[2 * l] = dW[l]; counts[2 * l] = long(L.Tw) * fout * fin;
      ptrs[2 * l + 1] = db[l]; counts[2 * l + 1] = long(L.Tw) * fout;
    }
    LAUNCH_N("zero_grads", launch_zero_many(ptrs, counts, 2 * nl, sms, stream));
  }

  const int top = desc->n_hidden;
  LastParams lp;
  memset(&lp, 0, sizeof(lp));
  lp.W = W[nl - 1]; lp.b = b[nl - 1];
  lp.act_hi = at<bf16>(ws, L.act_hi[top]); lp.act_lo = at<bf16>(ws, L.act_lo[top]);
  lp.c = at<void>(ws, L.c[top]); lp.jz = at<void>(ws, L.jz[top]);
  // the fused forward left ONE plane per layer (its signed sine) instead of sine + cosine planes
  const bool fused = fused_path(desc);
  if (fused) lp.phase = at<void>(ws, L.c[top]);
  lp.gy = gy; lp.gJ = order >= 1 ? gJ : nullptr; lp.gD = order >= 2 ? gD : nullptr;
  lp.adj_hi = at<bf16>(ws, L.adj_hi[top]); lp.adj_lo = at<bf16>(ws, L.adj_lo[top]);
  lp.dW = dW[nl - 1]; lp.db = db[nl - 1];
  lp.R = L.R; lp.n_pad = L.n_pad; lp.n = int(desc->n_coords); lp.d = d; lp.o = o; lp.order = order;
  lp.per_task = desc->per_task; lp.w0 = desc->w0;
  // The fused chain can start at the loss gradient itself (no last_bwd launch) when the outermost linear is narrow
  // enough for its per-warp partial sums (db_0, d columns of dW0, o rows of dWL: eight shared-memory rows).
  const bool fuse_top = fused && o <= 2;
  if (dc && !fuse_top) {      // off the fused top step: the masked adjoint as one elementwise pass into the workspace
    float* scr = at<float>(ws, L.gyscr);
    LAUNCH_N("dc_grad", launch_dc_grad(gy, scr, dc_spec(dc), desc->tasks, int(desc->n_coords), o, sms, stream));
    gy = scr;
    lp.gy = scr;
    dc = nullptr;
  }
  if (!fuse_top) LAUNCH_N("last_bwd", launch_last_bwd(lp, split, sms, stream));

  // whole input-gradient chain in one launch (mlp_fused_bwd.cu)
  const bool fuse_dw0 = fused && d <= 4;
  const bool wide_wg = fused && d > 4;      // wide first layer on the fused path: dW_0 / db_0 are weight-gradient items
  const int bn = rows_gemm_bn(order, order ? d : 0, split, 1);
  if (fused) {
    MlpBwdParams m;
    memset(&m, 0, sizeof(m));
    const int NH = desc->n_hidden;
    if ((rc = make_map(&m.tmTop, at<void>(ws, fuse_top ? L.c[NH] : L.adj_hi[NH]), L.R, 128))) return rc;
    if (fuse_top) {
      if ((rc = make_map(&m.tmAdj[NH], at<void>(ws, L.adj_hi[NH]), L.R, 128))) return rc;
      m.db[NH] = db[NH];
      m.fuse_top = 1; m.o = o; m.gy = gy;
      m.dc = dc_spec(dc);
      m.phase_top = at<uint32_t>(ws, L.c[NH]);
      m.WL = W[nl - 1]; m.dWL = dW[nl - 1]; m.dbL = db[nl - 1];
    }
    for (int l = 0; l < NH; ++l) {
      if ((rc = make_map(&m.tmWt[l], ext_wt ? ext_wt[l] : at<void>(ws, L.wt_hi[l]), uint64_t(L.Tw) * H, 128))) return rc;
      if (l > 0 || d > 4)
        if ((rc = make_map(&m.tmC[l], at<void>(ws, L.c[l]), L.R, 128))) return rc;
      if ((rc = make_map(&m.tmAdj[l], at<void>(ws, L.adj_hi[l]), L.R, 128))) return rc;
      m.db[l] = db[l];
    }
    m.dW0 = dW[0]; m.x = coords; m.W0 = W[0]; m.b0 = b[0];
    if (d > 4) {           // wide first layer: its dW and db come from first_bwd, which reads the stored layer-0 adjoint
      m.store_adj0 = 1;
      m.skip_bottom_sums = 1;
    } else {               // narrow first layer: no phase plane, cos(theta_0) recomputed from the coordinates
      m.l0_from_x = 1;
    }
    m.n_hidden = NH; m.rows_per_task = L.n_pad; m.per_task = desc->per_task; m.tasks = L.R / L.n_pad;
    m.n = int(desc->n_coords); m.d = d; m.store_adj0 = (gcoords || d > 4) ? 1 : 0; m.w0 = desc->w0;
    if (step_fwd) {            // forward, loss gradient and this chain as one kernel (mlp_fused_step.cu)
      MlpStepParams sp;
      sp.f = *step_fwd;
      sp.b = m;
      sp.rag = nullptr; sp.task_loss = nullptr; sp.rag_units = 0;
      if (rg) {
        sp.f.tasks = desc->tasks;
        sp.rag = at<int>(ws, L.rag); sp.task_loss = rg->task_loss; sp.rag_units = rg->units;
        LAUNCH_N("mlp_fused_step_ragged", launch_mlp_fused_step_ragged(sp, sms, stream));
      } else {
        LAUNCH_N("mlp_fused_step", launch_mlp_fused_step(sp, sms, stream));
      }
    }
    static long long* dbg_buf = nullptr;
    const bool dbg = getenv("SIREN_FUSED_DBG") != nullptr;
    if (dbg) {
      if (!dbg_buf) cudaMalloc(&dbg_buf, 4096 * sizeof(long long));
      cudaMemsetAsync(dbg_buf, 0, 4096 * sizeof(long long), stream);
      m.dbg = dbg_buf;
    }
    if (!step_fwd) LAUNCH_N("mlp_fused_bwd", launch_mlp_fused_bwd(m, sms, stream));
    if (dbg) {
      static long long host[4096];
      cudaStreamSynchronize(stream);
      cudaMemcpy(host, dbg_buf, sizeof(host), cudaMemcpyDeviceToHost);
      const long long t0 = host[0];
      print_cta_spread("fused bwd", host);
      for (int pr = 0; pr < 3; ++pr)
        for (int l = 1; l <= NH + (fuse_top ? 1 : 0); ++l) {
          fprintf(stderr, "[fused bwd dbg] unit %d -> layer %d:", pr, l - 1);
          for (int k = 0; k < 8; ++k) fprintf(stderr, " %lld", host[(pr * 8 + l) * 8 + k] ? host[(pr * 8 + l) * 8 + k] - t0 : -1);
          fprintf(stderr, "  | mma");
          for (int k = 0; k < 4; ++k) fprintf(stderr, " %lld", host[(pr * 8 + l) * 8 + 512 + k] ? host[(pr * 8 + l) * 8 + 512 + k] - t0 : -1);
          fprintf(stderr, "  | loader");
          for (int k = 0; k < 4; ++k) fprintf(stderr, " %lld", host[(pr * 8 + l) * 8 + 1024 + k] ? host[(pr * 8 + l) * 8 + 1024 + k] - t0 : -1);
          fprintf(stderr, "\n");
        }
    }
  }
  for (int l = desc->n_hidden; l >= 1 && !fused; --l) {
    RowsGemmParams p;
    memset(&p, 0, sizeof(p));
    if ((rc = make_map(&p.tmA_hi, at<void>(ws, L.adj_hi[l]), uint64_t(L.S) * L.R, TILE_M))) return rc;
    if ((rc = make_map(&p.tmA_lo, at<void>(ws, L.adj_lo[l]), uint64_t(L.S) * L.R, TILE_M))) return rc;
    if ((rc = make_map(&p.tmB_hi, at<void>(ws, L.wt_hi[l - 1]), uint64_t(L.Tw) * H, bn))) return rc;
    if ((rc = make_map(&p.tmB_lo, at<void>(ws, L.wt_lo[l - 1]), uint64_t(L.Tw) * H, bn))) return rc;
    p.R = L.R; p.rows_per_task = L.n_pad; p.per_task = desc->per_task; p.w0 = desc->w0;
    p.w_first = W[0]; p.below_is_first = (l - 1 == 0) ? 1 : 0;
    {
      const int cw = rows_gemm_cw(order, order ? d : 0, split, 1);
      const int se = split ? 4 : 2;      // stash element size
      if ((rc = make_map_ex(&p.tmO_hi, at<void>(ws, L.adj_hi[l - 1]), 2, uint64_t(L.S) * L.R, cw, 32))) return rc;
      if ((rc = make_map_ex(&p.tmO_lo, at<void>(ws, L.adj_lo[l - 1]), 2, uint64_t(L.S) * L.R, cw, 32))) return rc;
      if ((rc = make_map_ex(&p.tmCin, at<void>(ws, L.c[l - 1]), se, L.R, cw, 32))) return rc;
      if ((rc = make_map_ex(&p.tmJin, at<void>(ws, L.jz[l - 1]), se, uint64_t(L.S > 1 ? L.S - 1 : 1) * L.R, cw, 32))) return rc;
      if ((rc = make_map_ex(&p.tmSin_hi, at<void>(ws, L.act_hi[l - 1]), 2, uint64_t(L.S) * L.R, cw, 32))) return rc;
      if ((rc = make_map_ex(&p.tmSin_lo, at<void>(ws, L.act_lo[l - 1]), 2, uint64_t(L.S) * L.R, cw, 32))) return rc;
    }
    LAUNCH_N("hidden_dgrad", launch_rows_gemm(p, 1, order, order ? d : 0, split, sms, stream));
  }

  // weight gradients of the hidden layers (groups of up to MAX_WG_LAYERS per launch)
  const int kc = wgrad_kc(split);
  for (int l0 = 1; l0 <= desc->n_hidden; l0 += MAX_WG_LAYERS) {
    WgradParams wp;
    memset(&wp, 0, sizeof(wp));
    int cnt = 0;
    for (int l = l0; l <= desc->n_hidden && cnt < MAX_WG_LAYERS; ++l, ++cnt) {
      if ((rc = make_map(&wp.tmA_hi[cnt], at<void>(ws, L.adj_hi[l]), uint64_t(L.S) * L.R, kc))) return rc;
      if ((rc = make_map(&wp.tmA_lo[cnt], at<void>(ws, L.adj_lo[l]), uint64_t(L.S) * L.R, kc))) return rc;
      if ((rc = make_map(&wp.tmB_hi[cnt], at<void>(ws, fused ? L.c[l - 1] : L.act_hi[l - 1]), uint64_t(L.S) * L.R, kc))) return rc;
      if ((rc = make_map(&wp.tmB_lo[cnt], at<void>(ws, L.act_lo[l - 1]), uint64_t(L.S) * L.R, kc))) return rc;
      wp.dW[cnt] = dW[l];
      wp.db[cnt] = db[l];      // bias gradient = column sums of the staged adjoint blocks
    }
    wp.n_layers = cnt; wp.S = L.S; wp.R = L.R; wp.rows_per_task = L.n_pad;
    wp.per_task = desc->per_task; wp.tasks = desc->tasks;
    wp.phase_b = fused ? 1 : 0;
    wp.db_plain = fused ? 0 : 1;
    if (fused && d <= 4 && l0 == 1) {      // first hidden layer: sin(theta_0) is built from the coordinates on chip
      wp.l0_from_x = 1; wp.d = d; wp.n = int(desc->n_coords); wp.w0 = desc->w0;
      wp.x = coords; wp.W0 = W[0]; wp.b0 = b[0];
    }
    if (wide_wg && l0 == 1) {      // wide first layer: its own dW_0 / db_0 as one more item kind of this launch
      wp.first_wide = 1;
      if ((rc = make_map(&wp.tmA0, at<void>(ws, L.adj_hi[0]), L.R, kc))) return rc;
      wp.dW0 = dW[0]; wp.db0 = db[0];
      wp.d = d; wp.n = int(desc->n_coords); wp.x = coords;
      wp.ff = fourier_spec(ff);
      if (d > 16) {      // the forward left the layer's input plane: a TMA-fed operand, nkc0 feature blocks wide
        wp.nkc0 = L.nkc0;
        if ((rc = make_map(&wp.tmB0, at<void>(ws, L.feat), L.R, kc))) return rc;
      }
    }
    if (rg) {      // items per (scene, layer, slice) from the tables; the device counts them
      wp.rag = at<int>(ws, L.rag);
      const long most = long(cnt) * (L.R / TILE_M);
      LAUNCH_N("wgrad_ragged", launch_wgrad_ragged(wp, int(most < sms ? most : sms), stream));
      continue;
    }
    const int groups = desc->per_task ? desc->tasks : 1;
    const int tiles_group = (desc->per_task ? L.n_pad : L.R) / TILE_M;
    const int base = (cnt + wp.first_wide) * groups;
    int best = 1;
    double best_eff = 0.0;
    for (int s = 1; s <= 64; ++s) {
      if (s > tiles_group) break;
      const long n = long(base) * s;
      const long waves = (n + sms - 1) / sms;
      const double eff = double(n) / double(waves * sms);
      if (eff > best_eff + 1e-9) { best_eff = eff; best = s; }
      if (eff >= 0.95) break;
    }
    wp.slices = best;
    if (const char* e = getenv("SIREN_WGRAD_SLICES")) {      // developer aid: sweep the split-K factor
      const int v = atoi(e);
      if (v >= 1 && v <= tiles_group) wp.slices = v;
    }
    // The items of the first hidden layer BUILD their operand (one MUFU per element) and end ~17 % later than the
    // TMA-fed ones (tools/probe_wgrad.py: 113-125 us against 98-107 us at cfg2): when every item has a CTA of its own
    // they are cut into more, shorter slices so that all kinds end together.
    if (wp.l0_from_x && cnt >= 2 && base * wp.slices <= sms && !getenv("SIREN_WGRAD_EVEN")) {
      const int others = (cnt + wp.first_wide - 1) * groups;
      int s = int(double(sms) / (groups * (cnt + wp.first_wide - 1 + 1.17)));
      if (s < 1) s = 1;
      int s0 = (sms - others * s) / groups;
      if (s0 > tiles_group) s0 = tiles_group;
      if (s <= tiles_group && s0 > s) {
        wp.slices = s;
        wp.slices0 = s0;
      }
    }
    // developer aid: SIREN_WGRAD_DBG=1 prints, per item kind, when its CTAs started and finished (tools/probe_wgrad.py)
    static long long* wg_dbg = nullptr;
    const bool wdbg = getenv("SIREN_WGRAD_DBG") != nullptr;
    if (wdbg) {
      if (!wg_dbg) cudaMalloc(&wg_dbg, 3 * 256 * sizeof(long long));
      cudaMemsetAsync(wg_dbg, 0, 3 * 256 * sizeof(long long), stream);
      wp.dbg = wg_dbg;
    }
    LAUNCH_N("wgrad", launch_wgrad(wp, split, sms, stream));
    if (wdbg) {
      static long long host[3 * 256];
      cudaStreamSynchronize(stream);
      cudaMemcpy(host, wg_dbg, sizeof(host), cudaMemcpyDeviceToHost);
      long long t0 = 0;
      for (int i = 0; i < 256; ++i) if (host[3 * i + 1] && (!t0 || host[3 * i + 1] < t0)) t0 = host[3 * i + 1];
      for (int kind = 0; kind <= cnt; ++kind) {
        long long smin = 0, smax = 0, emin = 0, emax = 0; int nct = 0;
        for (int i = 0; i < 256; ++i) {
          if (!host[3 * i + 1] || host[3 * i] != kind) continue;
          const long long st = host[3 * i + 1] - t0, en = host[3 * i + 2] - t0;
          if (!nct || st < smin) smin = st;
          if (!nct || st > smax) smax = st;
          if (!nct || en < emin) emin = en;
          if (!nct || en > emax) emax = en;
          ++nct;
        }
        if (nct) fprintf(stderr, "[wgrad dbg] item kind %d: %d CTAs, start %lld..%lld ns, end %lld..%lld ns\n", kind, nct, smin, smax, emin, emax);
      }
    }
  }
  const bool wide_pl = !fused && d > 16;      // wide first layer on the per-layer (fp32-parity) path
  if (wide_pl) {
    // dW_0 = zbar_0^T [inputs] as one more weight-gradient launch on the padded input planes, into a padded scratch
    float* pad = at<float>(ws, L.dw0pad);
    CUDA_TRY(cudaMemsetAsync(pad, 0, size_t(L.Tw) * H * H * sizeof(float), stream));
    WgradParams wp;
    memset(&wp, 0, sizeof(wp));
    if ((rc = make_map(&wp.tmA_hi[0], at<void>(ws, L.adj_hi[0]), L.R, kc))) return rc;
    if ((rc = make_map(&wp.tmA_lo[0], at<void>(ws, L.adj_lo[0]), L.R, kc))) return rc;
    if ((rc = make_map(&wp.tmB_hi[0], at<void>(ws, L.feat), L.R, kc))) return rc;
    if ((rc = make_map(&wp.tmB_lo[0], at<void>(ws, L.feat_lo), L.R, kc))) return rc;
    wp.dW[0] = pad;
    wp.n_layers = 1; wp.S = 1; wp.R = L.R; wp.rows_per_task = L.n_pad;
    wp.per_task = desc->per_task; wp.tasks = desc->tasks;
    const int groups = desc->per_task ? desc->tasks : 1;
    const int tiles_group = (desc->per_task ? L.n_pad : L.R) / TILE_M;
    int sl = sms / groups;
    if (sl < 1) sl = 1;
    if (sl > tiles_group) sl = tiles_group;
    if (sl > 64) sl = 64;
    wp.slices = sl;
    LAUNCH_N("wgrad", launch_wgrad(wp, split, sms, stream));
    LAUNCH_N("unpad_dw0", launch_unpad_dw0(pad, dW[0], d, long(L.Tw) * H, sms, stream));
    LAUNCH_N("colsum", launch_colsum(at<bf16>(ws, L.adj_hi[0]), at<bf16>(ws, L.adj_lo[0]), db[0], L.R, L.n_pad,
                                     desc->per_task, sms, stream));
  }

  FirstParams fp;
  memset(&fp, 0, sizeof(fp));
  fp.x = coords; fp.W = W[0]; fp.b = b[0];
  fp.adj_hi = at<bf16>(ws, L.adj_hi[0]); fp.adj_lo = at<bf16>(ws, L.adj_lo[0]);
  fp.dW = dW[0]; fp.db = db[0]; fp.gx = gcoords;
  fp.R = L.R; fp.n_pad = L.n_pad; fp.n = int(desc->n_coords); fp.d = d; fp.order = order;
  fp.per_task = desc->per_task; fp.w0 = desc->w0;
  fp.ff = fourier_spec(ff);
  fp.only_gx = (fuse_dw0 || wide_wg) ? 1 : 0;          // dW0 / db0 already came out of the dgrad epilogue / wgrad
  if (wide_pl) return SIREN_OK;                        // (no coordinate gradient above 16 inputs: rejected above)
  if (!(fuse_dw0 || wide_wg) || gcoords) LAUNCH_N("first_bwd", launch_first_bwd(fp, split, sms, stream));
  return SIREN_OK;
}

int siren_b200_backward(const siren_desc_t* desc, const float* coords, const float* const* W, const float* const* b,
                        const void* ws, const float* gy, const float* gJ, const float* gD, float* const* dW,
                        float* const* db, float* gcoords, int accumulate, void* stream_) {
  return backward_impl(desc, coords, W, b, ws, gy, gJ, gD, dW, db, gcoords, accumulate, stream_, nullptr);
}

int siren_b200_forward_ff(const siren_desc_t* desc, const siren_fourier_t* ff, const float* raw_coords,
                          const float* const* W, const float* const* b, float* y, void* ws, int inference,
                          void* stream_) {
  if (!ff) return fail(SIREN_ERR_INVALID, "null fourier descriptor");
  return forward_impl(desc, raw_coords, W, b, y, nullptr, nullptr, ws, stream_, inference == 0, false, nullptr, 0.f, nullptr,
                      nullptr, ff);
}

int siren_b200_backward_ff(const siren_desc_t* desc, const siren_fourier_t* ff, const float* raw_coords,
                           const float* const* W, const float* const* b, const void* ws, const float* gy,
                           float* const* dW, float* const* db, int accumulate, void* stream_) {
  if (!ff) return fail(SIREN_ERR_INVALID, "null fourier descriptor");
  return backward_impl(desc, raw_coords, W, b, ws, gy, nullptr, nullptr, dW, db, nullptr, accumulate, stream_, ff);
}

int siren_b200_forward_dc(const siren_desc_t* desc, const siren_fourier_t* ff, const siren_dc_t* dc, const float* coords,
                          const float* const* W, const float* const* b, float* y, void* ws, int inference,
                          void* stream_) {
  if (!dc) return fail(SIREN_ERR_INVALID, "null data-consistency descriptor");
  return forward_impl(desc, coords, W, b, y, nullptr, nullptr, ws, stream_, inference == 0, false, nullptr, 0.f, nullptr,
                      nullptr, ff, dc);
}

int siren_b200_backward_dc(const siren_desc_t* desc, const siren_fourier_t* ff, const siren_dc_t* dc, const float* coords,
                           const float* const* W, const float* const* b, const void* ws, const float* gy,
                           float* const* dW, float* const* db, int accumulate, void* stream_) {
  if (!dc) return fail(SIREN_ERR_INVALID, "null data-consistency descriptor");
  return backward_impl(desc, coords, W, b, ws, gy, nullptr, nullptr, dW, db, nullptr, accumulate, stream_, ff, dc);
}

int siren_b200_forward_call(const siren_desc_t* desc, const siren_call_t* call, const float* coords,
                            const float* const* W, const float* const* b, float* y, void* ws, int inference,
                            void* stream_) {
  if (!call) return fail(SIREN_ERR_INVALID, "null call descriptor");
  if (desc && desc->deriv_order != 0) return fail(SIREN_ERR_INVALID, "forward_call is value-only (deriv_order 0)");
  return forward_impl(desc, coords, W, b, y, nullptr, nullptr, ws, stream_, inference == 0, false, nullptr, 0.f, nullptr,
                      nullptr, call->fourier, call->dc, call->wk16);
}

int siren_b200_backward_call(const siren_desc_t* desc, const siren_call_t* call, const float* coords,
                             const float* const* W, const float* const* b, const void* ws, const float* gy,
                             float* const* dW, float* const* db, int accumulate, void* stream_) {
  if (!call) return fail(SIREN_ERR_INVALID, "null call descriptor");
  return backward_impl(desc, coords, W, b, ws, gy, nullptr, nullptr, dW, db, nullptr, accumulate, stream_, call->fourier,
                       call->dc, call->wt16);
}

int siren_b200_hyper_head(const float* h, const float* Wlast, const float* blast, int tasks, int k_h, float w0,
                          float* W_out, void* wk16, void* wt16, float* sumsq, void* stream_) {
  if (!h || !Wlast || !blast || !W_out) return fail(SIREN_ERR_INVALID, "null pointer argument");
  if (tasks < 1) return fail(SIREN_ERR_INVALID, "empty batch");
  if (k_h < 4 || k_h > 512 || (k_h & 3))
    return fail(SIREN_ERR_UNSUPPORTED, "hyper_hidden_features=%d: the head kernel takes multiples of 4 in 4..512", k_h);
  HyperHeadParams p;
  p.h = h; p.Wlast = Wlast; p.blast = blast; p.W_out = W_out;
  p.wk16 = reinterpret_cast<__half*>(wk16); p.wt16 = reinterpret_cast<bf16*>(wt16);
  p.sumsq = sumsq; p.tasks = tasks; p.k_h = k_h; p.w0 = w0;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  LAUNCH_N("hyper_head", launch_hyper_head(p, stream));
  return SIREN_OK;
}

int siren_b200_forward_dc_mse(const siren_desc_t* desc, const siren_fourier_t* ff, const siren_dc_t* dc,
                              const float* coords, const float* const* W, const float* const* b, float* y,
                              const float* gt, float weight, float* gy, float* loss4, void* ws, void* stream_) {
  if (!dc || !gt || !gy) return fail(SIREN_ERR_INVALID, "null pointer argument");
  return forward_impl(desc, coords, W, b, y, nullptr, nullptr, ws, stream_, true, false, gt, weight, gy, loss4, ff, dc);
}

int siren_b200_prepare_weights(const siren_desc_t* desc, const float* const* W, void* ws, void* stream_) {
  int rc = check_desc(desc);
  if (rc) return rc;
  if (!W || !ws) return fail(SIREN_ERR_INVALID, "null pointer argument");
  Layout L;
  make_layout(desc, &L);
  return prep_impl(desc, L, W, ws, reinterpret_cast<cudaStream_t>(stream_));
}

int siren_b200_forward_prepared(const siren_desc_t* desc, const float* coords, const float* const* W,
                                const float* const* b, float* y, float* J, float* D, void* ws, void* stream_) {
  return forward_impl(desc, coords, W, b, y, J, D, ws, stream_, true, true);
}

int siren_b200_forward_mse(const siren_desc_t* desc, const float* coords, const float* const* W, const float* const* b,
                           float* y, const float* gt, float weight, float* gy, float* loss4, void* ws,
                           int weights_ready, void* stream_) {
  if (!gt || !gy) return fail(SIREN_ERR_INVALID, "null pointer argument");
  if (desc && desc->deriv_order != 0) return fail(SIREN_ERR_INVALID, "forward_mse is value-only (deriv_order 0)");
  return forward_impl(desc, coords, W, b, y, nullptr, nullptr, ws, stream_, true, weights_ready != 0, gt, weight, gy, loss4);
}

int siren_b200_forward_backward_mse(const siren_desc_t* desc, const float* coords, const float* const* W,
                                    const float* const* b, float* y, const float* gt, float weight, float* gy,
                                    float* loss4, void* ws, int weights_ready, float* const* dW, float* const* db,
                                    int accumulate, void* stream_) {
  if (!gt) return fail(SIREN_ERR_INVALID, "null pointer argument");
  if (desc && desc->deriv_order != 0) return fail(SIREN_ERR_INVALID, "forward_backward_mse is value-only (deriv_order 0)");
  int rc = check_desc(desc);
  if (rc) return rc;
  if (!fused_step(desc)) {
    // two launches: gy is their hand-over (the workspace's scratch plane when the caller does not want it)
    if (!gy) {
      if (!ws) return fail(SIREN_ERR_INVALID, "null pointer argument");
      Layout L;
      make_layout(desc, &L);
      gy = at<float>(ws, L.gyscr);
    }
    if ((rc = siren_b200_forward_mse(desc, coords, W, b, y, gt, weight, gy, loss4, ws, weights_ready, stream_))) return rc;
    return siren_b200_backward(desc, coords, W, b, ws, gy, nullptr, nullptr, dW, db, nullptr, accumulate, stream_);
  }
  MlpFwdParams f;
  if ((rc = forward_impl(desc, coords, W, b, y, nullptr, nullptr, ws, stream_, true, weights_ready != 0, gt, weight, gy,
                         loss4, nullptr, nullptr, nullptr, &f)))
    return rc;
  return backward_impl(desc, coords, W, b, ws, gy, nullptr, nullptr, dW, db, nullptr, accumulate, stream_, nullptr,
                       nullptr, nullptr, &f);
}

// ---- scenes of different sizes (siren_b200_*_ragged) ----
// The counts, the envelope (the one-kernel step's) and the plane rows in all; eq = desc with n_coords = the largest count
static int check_ragged(const siren_desc_t* desc, const long* n_host, siren_desc_t* eq, long* rows) {
  if (!desc || !n_host) return fail(SIREN_ERR_INVALID, "null pointer argument");
  if (desc->per_task != 1) return fail(SIREN_ERR_INVALID, "scenes of different sizes need per_task = 1");
  if (desc->tasks < 1) return fail(SIREN_ERR_INVALID, "empty batch");
  if (desc->tasks > MAX_TASKS) return fail(SIREN_ERR_UNSUPPORTED, "tasks=%d above %d", desc->tasks, MAX_TASKS);
  long nmax = 0, r = 0;
  for (int t = 0; t < desc->tasks; ++t) {
    if (n_host[t] < 1) return fail(SIREN_ERR_INVALID, "scene %d has %ld coordinates", t, n_host[t]);
    if (n_host[t] > nmax) nmax = n_host[t];
    r += (n_host[t] + TILE_M - 1) / TILE_M * TILE_M;
    if (r >= (1L << 31)) return fail(SIREN_ERR_UNSUPPORTED, "batch too large for 32-bit rows");
  }
  *eq = *desc;
  eq->n_coords = nmax;
  int rc = check_desc(eq);
  if (rc) return rc;
  if (!fused_path(eq) || eq->n_hidden > MAX_FUSED_STEP_HIDDEN || eq->d_in > 4 || eq->d_out > 2)
    return fail(SIREN_ERR_UNSUPPORTED, "scenes of different sizes train on the one-kernel bf16 step only (value path, "
                "in_features <= 4, out_features <= 2, at most %d hidden layers)", MAX_FUSED_STEP_HIDDEN);
  *rows = r;
  return SIREN_OK;
}

// Weight-gradient slices: scene t is cut into ceil(tiles_t / K) slices of about K 128-row tiles (at least one), so that
// a scene's flushes (256 KB of red.add per item) follow its size.  K is the longest scene's tiles over s, for the
// smallest s = 1..64 at which the estimated time is within 95 % of the ideal (the equal-N rule: items / (waves * SMs),
// here also bounded by the longest item, K tiles, against the total tiles per SM); else the best such estimate.  With
// equal counts this is the equal-N split.
static int ragged_slice_tiles(const long* n, int T, int kinds, int sms) {
  long tmax = 0, total = 0;
  for (int t = 0; t < T; ++t) {
    const long tiles = (n[t] + TILE_M - 1) / TILE_M;
    tmax = tiles > tmax ? tiles : tmax;
    total += tiles;
  }
  long best = tmax, prev = 0;
  double best_eff = 0.0;
  for (long s = 1; s <= 64 && s <= tmax; ++s) {
    const long K = (tmax + s - 1) / s;
    if (K == prev) continue;
    prev = K;
    long items = 0;
    for (int t = 0; t < T; ++t) items += ((n[t] + TILE_M - 1) / TILE_M + K - 1) / K;
    items *= kinds;
    const long waves = (items + sms - 1) / sms;
    // share of the ideal time (the items' tiles spread evenly): waves of items of the average length, and no less
    // than the longest item
    const double fill = double(items) / double(waves * sms), longest = double(kinds) * total / (double(sms) * K);
    const double eff = fill < longest ? fill : longest;
    if (eff > best_eff + 1e-9) { best_eff = eff; best = K; }
    if (eff >= 0.95) break;
  }
  return int(best);
}

size_t siren_b200_workspace_bytes_ragged(const siren_desc_t* desc, const long* n_host) {
  siren_desc_t eq;
  long rows = 0;
  if (check_ragged(desc, n_host, &eq, &rows) != SIREN_OK) return 0;
  Layout L;
  make_layout(&eq, &L, rows);
  return L.total;
}

int siren_b200_ragged_tables(const siren_desc_t* desc, const long* n_host, int sms, int* tables) {
  siren_desc_t eq;
  long rows = 0;
  int rc = check_ragged(desc, n_host, &eq, &rows);
  if (rc) return rc;
  if (!tables) return fail(SIREN_ERR_INVALID, "null pointer argument");
  ragged_tables(n_host, desc->tasks, ragged_slice_tiles(n_host, desc->tasks, desc->n_hidden, sms > 0 ? sms : num_sms()),
                tables);
  return SIREN_OK;
}

int siren_b200_prepare_ragged(const siren_desc_t* desc, const long* n_host, void* ws, void* stream_) {
  siren_desc_t eq;
  long rows = 0;
  int rc = check_ragged(desc, n_host, &eq, &rows);
  if (rc) return rc;
  if (!ws) return fail(SIREN_ERR_INVALID, "null pointer argument");
  Layout L;
  make_layout(&eq, &L, rows);
  RaggedPrepParams pp;
  memset(&pp, 0, sizeof(pp));
  for (int t = 0; t < desc->tasks; ++t) pp.n[t] = n_host[t];
  pp.T = desc->tasks;
  pp.K = ragged_slice_tiles(n_host, desc->tasks, desc->n_hidden, num_sms());
  pp.tab = at<int>(ws, L.rag);
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  LAUNCH_N("prepare_ragged", launch_prepare_ragged(pp, stream));
  return SIREN_OK;
}

int siren_b200_forward_backward_mse_ragged(const siren_desc_t* desc, const long* n_host, const float* coords,
                                           const float* const* W, const float* const* b, float* y, const float* gt,
                                           float weight, float* gy, float* loss4, float* task_loss, void* ws,
                                           int weights_ready, float* const* dW, float* const* db, int accumulate,
                                           void* stream_) {
  siren_desc_t eq;
  long rows = 0;
  int rc = check_ragged(desc, n_host, &eq, &rows);
  if (rc) return rc;
  if (!gt || !task_loss) return fail(SIREN_ERR_INVALID, "null pointer argument");
  Ragged rg;
  rg.rows = rows;
  rg.task_loss = task_loss;
  rg.units = 0;
  for (int t = 0; t < desc->tasks; ++t) rg.units += int(((n_host[t] + TILE_M - 1) / TILE_M + 1) / 2 + 1) / 2;
  MlpFwdParams f;
  if ((rc = forward_impl(&eq, coords, W, b, y, nullptr, nullptr, ws, stream_, true, weights_ready != 0, gt, weight, gy,
                         loss4, nullptr, nullptr, nullptr, &f, &rg)))
    return rc;
  return backward_impl(&eq, coords, W, b, ws, gy, nullptr, nullptr, dW, db, nullptr, accumulate, stream_, nullptr,
                       nullptr, nullptr, &f, &rg);
}

static int adam_step_impl(float* param, float* grad, float* m, float* v, long n, float lr, double beta1, double beta2,
                          float eps, float max_grad_norm, float grad_scale, void* state, int zero_grad, float* loss4,
                          const siren_desc_t* desc, const float* const* W, void* ws, void* stream_,
                          const float* const* peers, int world, float* zero_buf) {
  if (!param || !grad || !m || !v || !state || n <= 0) return fail(SIREN_ERR_INVALID, "bad adam arguments");
  if (world > 1 && (!peers || world > 64)) return fail(SIREN_ERR_INVALID, "bad peer arguments");
  if (zero_buf && (reinterpret_cast<uintptr_t>(zero_buf) & 15)) return fail(SIREN_ERR_INVALID, "zero_buf alignment");
  if ((reinterpret_cast<uintptr_t>(param) | reinterpret_cast<uintptr_t>(grad) | reinterpret_cast<uintptr_t>(m) |
       reinterpret_cast<uintptr_t>(v)) & 15)
    return fail(SIREN_ERR_INVALID, "adam_step needs 16-byte aligned buffers");
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  const int sms = num_sms();
  AdamFusedParams a;
  memset(&a, 0, sizeof(a));
  a.p = param; a.g = grad; a.m = m; a.v = v; a.n = n;
  a.lr = lr; a.eps = eps; a.max_norm = max_grad_norm; a.grad_scale = grad_scale; a.b1 = beta1; a.b2 = beta2;
  a.st = reinterpret_cast<AdamState*>(state);
  a.zero_grad = zero_grad ? 1 : 0;
  a.loss4 = loss4;
  a.peers = peers; a.world = world > 1 ? world : 1; a.zero_buf = zero_buf;
  if (desc && W && ws) {      // keep the workspace's bf16 weight copies in step with the parameters
    int rc = check_desc(desc);
    if (rc) return rc;
    if (desc->per_task) return fail(SIREN_ERR_UNSUPPORTED, "adam_step refreshes shared weights only");
    Layout L;
    make_layout(desc, &L);
    a.n_w = desc->n_hidden;
    a.split = L.split ? 1 : 0;
    a.scale_t = fused_path(desc) ? desc->w0 : 1.f;
    a.k_f16 = fused_path(desc) ? 1 : 0;
    for (int l = 0; l < desc->n_hidden; ++l) {
      const long off = long(W[l + 1] - param);
      if (off < 0 || off + long(H) * H > n)
        return fail(SIREN_ERR_INVALID, "hidden weight %d does not live inside the flat parameter buffer", l + 1);
      a.w_off[l] = off;
      a.k_hi[l] = at<bf16>(ws, L.wk_hi[l]); a.k_lo[l] = at<bf16>(ws, L.wk_lo[l]);
      a.t_hi[l] = at<bf16>(ws, L.wt_hi[l]); a.t_lo[l] = at<bf16>(ws, L.wt_lo[l]);
    }
  }
  // the squared gradient norm accumulates into state->sumsq, which the previous adam_step left at zero
  if (max_grad_norm > 0.f) {
    if (a.world > 1) LAUNCH_N("sumsq", launch_sumsq_peers(peers, a.world, n, &a.st->sumsq, sms, stream));
    else LAUNCH_N("sumsq", launch_sumsq(grad, n, &a.st->sumsq, sms, stream));
  }
  LAUNCH_N("adam_step", launch_adam_fused(a, sms, stream));
  return SIREN_OK;
}

int siren_b200_adam_step(float* param, float* grad, float* m, float* v, long n, float lr, double beta1, double beta2,
                         float eps, float max_grad_norm, float grad_scale, void* state, int zero_grad, float* loss4,
                         const siren_desc_t* desc, const float* const* W, void* ws, void* stream_) {
  return adam_step_impl(param, grad, m, v, n, lr, beta1, beta2, eps, max_grad_norm, grad_scale, state, zero_grad, loss4,
                        desc, W, ws, stream_, nullptr, 1, nullptr);
}

int siren_b200_adam_step_peers(float* param, float* grad, float* m, float* v, long n, float lr, double beta1,
                               double beta2, float eps, float max_grad_norm, float grad_scale, void* state,
                               float* loss4, const siren_desc_t* desc, const float* const* W, void* ws,
                               const float* const* peer_grads, int world, float* zero_buf, void* stream_) {
  return adam_step_impl(param, grad, m, v, n, lr, beta1, beta2, eps, max_grad_norm, grad_scale, state, 1, loss4, desc, W,
                        ws, stream_, peer_grads, world, zero_buf);
}

// The segment table of T networks stacked in one flat buffer of n floats at `base`: parameter W[l] / b[l] is
// [T][out][in] / [T][out] at its offset from base.  The parameters must tile [0, n) exactly, in any order.
static int task_tail(const siren_desc_t* desc, const float* const* W, const float* const* b, const float* base, long n,
                     float max_norm, const float* y, const float* gt, float weight, float* task_sumsq,
                     float* task_loss, float* loss4, TaskTail* tt) {
  int rc = check_desc(desc);
  if (rc) return rc;
  if (!desc->per_task) return fail(SIREN_ERR_INVALID, "the per-task tail needs per_task = 1");
  if (desc->tasks > MAX_TASKS) return fail(SIREN_ERR_UNSUPPORTED, "tasks=%d above %d", desc->tasks, MAX_TASKS);
  if (!W || !b || !base || !task_sumsq || !task_loss || n <= 0 || (!y != !gt))
    return fail(SIREN_ERR_INVALID, "bad per-task tail arguments");
  memset(tt, 0, sizeof(*tt));
  const int L = desc->n_hidden + 2;
  for (int l = 0; l < L; ++l) {
    if (!W[l] || !b[l]) return fail(SIREN_ERR_INVALID, "null parameter pointer (layer %d)", l);
    const int out = l == L - 1 ? desc->d_out : H, in = l == 0 ? desc->d_in : H;
    tt->seg_off[2 * l] = long(W[l] - base);
    tt->seg_per[2 * l] = out * in;
    tt->seg_hidden[2 * l] = (l >= 1 && l <= desc->n_hidden) ? l - 1 : -1;
    tt->seg_off[2 * l + 1] = long(b[l] - base);
    tt->seg_per[2 * l + 1] = out;
    tt->seg_hidden[2 * l + 1] = -1;
  }
  tt->n_seg = 2 * L;
  for (int i = 1; i < tt->n_seg; ++i)      // ascending offsets
    for (int j = i; j > 0 && tt->seg_off[j] < tt->seg_off[j - 1]; --j) {
      std::swap(tt->seg_off[j], tt->seg_off[j - 1]);
      std::swap(tt->seg_per[j], tt->seg_per[j - 1]);
      std::swap(tt->seg_hidden[j], tt->seg_hidden[j - 1]);
    }
  long end = 0;
  for (int s = 0; s < tt->n_seg; ++s) {
    if (tt->seg_off[s] != end)
      return fail(SIREN_ERR_INVALID, "parameters do not tile the flat buffer (a gap or an overlap at float %ld)", end);
    end += long(desc->tasks) * tt->seg_per[s];
    tt->seg_cum[s + 1] = tt->seg_cum[s] + tt->seg_per[s];
  }
  if (end != n) return fail(SIREN_ERR_INVALID, "parameters cover %ld floats of a flat buffer of %ld", end, n);
  tt->tasks = desc->tasks;
  tt->max_norm = max_norm > 0.f ? max_norm : 0.f;
  tt->sumsq = task_sumsq;
  tt->loss = task_loss;
  tt->loss4 = loss4;
  tt->y = y;
  tt->gt = gt;
  tt->rows = desc->n_coords * desc->d_out;
  tt->weight = weight;
  return SIREN_OK;
}

int siren_b200_adam_step_tasks(const siren_desc_t* desc, const float* const* W, const float* const* b, float* param,
                               float* grad, float* m, float* v, long n, float lr, double beta1, double beta2, float eps,
                               float max_grad_norm, void* state, const float* y, const float* gt, float weight,
                               float* task_sumsq, float* task_loss, float* loss4, void* ws, void* stream_) {
  if (!param || !grad || !m || !v || !state) return fail(SIREN_ERR_INVALID, "bad adam arguments");
  if ((reinterpret_cast<uintptr_t>(param) | reinterpret_cast<uintptr_t>(grad) | reinterpret_cast<uintptr_t>(m) |
       reinterpret_cast<uintptr_t>(v)) & 15)
    return fail(SIREN_ERR_INVALID, "adam_step_tasks needs 16-byte aligned buffers");
  TaskTail tt;
  int rc = task_tail(desc, W, b, param, n, max_grad_norm, y, gt, weight, task_sumsq, task_loss, loss4, &tt);
  if (rc) return rc;
  tt.publish = 1;
  AdamFusedParams a;
  memset(&a, 0, sizeof(a));
  a.p = param; a.g = grad; a.m = m; a.v = v; a.n = n;
  a.lr = lr; a.eps = eps; a.b1 = beta1; a.b2 = beta2;
  a.st = reinterpret_cast<AdamState*>(state);
  a.zero_grad = 1;
  a.world = 1;
  if (ws) {      // the workspace's copies of every task's hidden weights, as prep_impl lays them out
    Layout L;
    make_layout(desc, &L);
    a.split = L.split ? 1 : 0;
    a.scale_t = fused_path(desc) ? desc->w0 : 1.f;
    a.k_f16 = fused_path(desc) ? 1 : 0;
    for (int l = 0; l < desc->n_hidden; ++l) {
      a.k_hi[l] = at<bf16>(ws, L.wk_hi[l]); a.k_lo[l] = at<bf16>(ws, L.wk_lo[l]);
      a.t_hi[l] = at<bf16>(ws, L.wt_hi[l]); a.t_lo[l] = at<bf16>(ws, L.wt_lo[l]);
    }
  } else {
    for (int s = 0; s < tt.n_seg; ++s) tt.seg_hidden[s] = -1;
  }
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  const int sms = num_sms();
  if (tt.max_norm > 0.f) {
    // the norms and, in the same pass, the losses; Adam then only publishes them
    TaskTail pre = tt;
    pre.publish = 0;
    LAUNCH_N("task_norms", launch_task_norms(grad, pre, a.st, sms, stream));
    tt.y = tt.gt = nullptr;
  }
  LAUNCH_N("adam_step_tasks", launch_adam_tasks(a, tt, sms, stream));
  return SIREN_OK;
}

int siren_b200_clip_grad_tasks(const siren_desc_t* desc, float* const* dW, float* const* db, float* grad, long n,
                               float max_grad_norm, void* state, const float* y, const float* gt, float weight,
                               float* task_sumsq, float* task_loss, float* loss4, int publish, void* stream_) {
  if (!grad || !state) return fail(SIREN_ERR_INVALID, "bad clip_grad_tasks arguments");
  TaskTail tt;
  int rc = task_tail(desc, dW, db, grad, n,
                     max_grad_norm, y, gt, weight, task_sumsq, task_loss, loss4, &tt);
  if (rc) return rc;
  tt.publish = publish ? 1 : 0;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  const int sms = num_sms();
  AdamState* st = reinterpret_cast<AdamState*>(state);
  if (tt.max_norm > 0.f) {
    TaskTail pre = tt;
    pre.publish = 0;
    LAUNCH_N("task_norms", launch_task_norms(grad, pre, st, sms, stream));
    LAUNCH_N("task_clip", launch_task_clip(grad, n, tt, st, sms, stream));
  } else if (tt.y || tt.publish) {
    LAUNCH_N("task_norms", launch_task_norms(grad, tt, st, sms, stream));
  }
  return SIREN_OK;
}

int siren_b200_allreduce_peers(float* const* peers, int world, int rank, long n, float scale, void* stream_) {
  if (!peers) return fail(SIREN_ERR_INVALID, "null pointer argument");
  if (world < 1 || world > 16 || rank < 0 || rank >= world) return fail(SIREN_ERR_INVALID, "rank %d of %d", rank, world);
  if (n < 0 || (n & 3)) return fail(SIREN_ERR_INVALID, "n=%ld: the buffer length must be a multiple of 4 floats", n);
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  LAUNCH_N("peer_allreduce", launch_peer_allreduce(peers, world, rank, n / 4, scale, num_sms(), stream));
  return SIREN_OK;
}

int siren_b200_allreduce_multicast(float* mc, int world, int rank, long n, float scale, void* stream_) {
  if (!mc) return fail(SIREN_ERR_INVALID, "null pointer argument");
  if (world < 1 || rank < 0 || rank >= world) return fail(SIREN_ERR_INVALID, "rank %d of %d", rank, world);
  if (n < 0 || (n & 3)) return fail(SIREN_ERR_INVALID, "n=%ld: the buffer length must be a multiple of 4 floats", n);
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  LAUNCH_N("peer_allreduce_mc", launch_peer_allreduce_mc(mc, world, rank, n / 4, scale, num_sms(), stream));
  return SIREN_OK;
}

int siren_b200_laplace_mse_grad(const float* D, const float* gt, float* gD, long n, int d, float weight, float* loss4,
                                void* stream_) {
  if (!D || !gt || !gD || n <= 0 || d < 1 || d > 3) return fail(SIREN_ERR_INVALID, "bad laplace_mse arguments");
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  LAUNCH_N("laplace_mse_grad", launch_laplace_mse_grad(D, gt, gD, n, d, weight, loss4 ? loss4 + 1 : nullptr, num_sms(), stream));
  return SIREN_OK;
}

int siren_b200_sdf_grad(const float* y, const float* J, const float* sdf, const float* normals, float* gy, float* gJ,
                        long n, float weight, float* loss4, void* stream_) {
  if (!y || !J || !sdf || !normals || !gy || !gJ || n <= 0) return fail(SIREN_ERR_INVALID, "bad sdf arguments");
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  LAUNCH_N("sdf_grad", launch_sdf_grad(y, J, sdf, normals, gy, gJ, n, weight, loss4 ? loss4 + 1 : nullptr, num_sms(), stream));
  return SIREN_OK;
}

int siren_b200_clip_grad(float* grad, long n, float max_grad_norm, void* state, void* stream_) {
  if (!grad || !state || n <= 0 || !(max_grad_norm > 0.f)) return fail(SIREN_ERR_INVALID, "bad clip_grad arguments");
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  LAUNCH_N("clip_grad", launch_clip_grad(grad, n, max_grad_norm, reinterpret_cast<AdamState*>(state), num_sms(), stream));
  return SIREN_OK;
}

int siren_b200_loss_roll(float* loss4, void* stream_) {
  if (!loss4) return fail(SIREN_ERR_INVALID, "null pointer argument");
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  LAUNCH_N("loss_roll", launch_loss_roll(loss4, stream));
  return SIREN_OK;
}

int siren_b200_adam(float* param, const float* grad, float* m, float* v, long n, float lr, double beta1,
                    double beta2, float eps, float max_grad_norm, float grad_scale, void* state, void* stream_) {
  if (!param || !grad || !m || !v || !state || n <= 0) return fail(SIREN_ERR_INVALID, "bad adam arguments");
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  const int sms = num_sms();
  AdamState* st = reinterpret_cast<AdamState*>(state);
  if (max_grad_norm > 0.f) {
    CUDA_TRY(cudaMemsetAsync(&st->sumsq, 0, sizeof(float), stream));
    LAUNCH_N("sumsq", launch_sumsq(grad, n, &st->sumsq, sms, stream));
  }
  LAUNCH_N("adam", launch_adam(param, grad, m, v, n, lr, beta1, beta2, eps, max_grad_norm, grad_scale, st, sms, stream));
  return SIREN_OK;
}

int siren_b200_mse_grad(const float* y, const float* gt, float* gy, long n, float weight, float* loss,
                        void* stream_) {
  if (!y || !gt || !gy || n <= 0) return fail(SIREN_ERR_INVALID, "bad mse arguments");
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  LAUNCH_N("mse_grad", launch_mse_grad(y, gt, gy, n, weight, loss, num_sms(), stream));
  return SIREN_OK;
}

int siren_b200_publish(const float* src, float* dst_host, int n, void* stream_) {
  if (!src || !dst_host || n <= 0 || n > 1024) return fail(SIREN_ERR_INVALID, "bad publish arguments");
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  LAUNCH_N("publish", launch_publish(src, dst_host, n, stream));
  return SIREN_OK;
}

int siren_b200_profile_begin(void) {
  g_prof_n = 0;
  g_prof_on = true;
  return SIREN_OK;
}

int siren_b200_profile_end(char* buf, size_t buflen) {
  g_prof_on = false;
  if (!buf || buflen < 64) return fail(SIREN_ERR_INVALID, "profile buffer too small");
  struct Agg { const char* name; int count; double ms; };
  Agg agg[64];
  int na = 0;
  for (int i = 0; i < g_prof_n; ++i) {
    float ms = 0.f;
    cudaEventSynchronize(g_prof[i].b);
    cudaEventElapsedTime(&ms, g_prof[i].a, g_prof[i].b);
    cudaEventDestroy(g_prof[i].a);
    cudaEventDestroy(g_prof[i].b);
    int j = 0;
    for (; j < na; ++j)
      if (strcmp(agg[j].name, g_prof[i].name) == 0) break;
    if (j == na) {
      if (na == 64) continue;
      agg[na++] = {g_prof[i].name, 0, 0.0};
    }
    agg[j].count++;
    agg[j].ms += ms;
  }
  g_prof_n = 0;
  size_t off = 0;
  buf[0] = 0;
  for (int j = 0; j < na; ++j) {
    int w = snprintf(buf + off, buflen - off, "%s %d %.6f\n", agg[j].name, agg[j].count, agg[j].ms);
    if (w < 0 || size_t(w) >= buflen - off) break;
    off += size_t(w);
  }
  return SIREN_OK;
}

int siren_b200_debug_linear(const float* A, const float* Wm, float* out, long R, int precision, void* scratch,
                            void* stream_) {
  if (!A || !Wm || !out || !scratch || R <= 0 || R % TILE_M) return fail(SIREN_ERR_INVALID, "bad debug_linear args");
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  const bool split = precision == SIREN_PREC_FP32_PARITY;
  char* s = reinterpret_cast<char*>(scratch);
  const size_t pl = size_t(R) * H * 2, wb = size_t(H) * H * 2;
  bf16 *a_hi = (bf16*)s, *a_lo = (bf16*)(s + pl), *k_hi = (bf16*)(s + 2 * pl), *k_lo = (bf16*)(s + 2 * pl + wb),
       *t_hi = (bf16*)(s + 2 * pl + 2 * wb), *t_lo = (bf16*)(s + 2 * pl + 3 * wb);
  LAUNCH_N("to_planes", launch_to_planes(A, a_hi, a_lo, R * H, split, stream));
  PrepParams pp;
  memset(&pp, 0, sizeof(pp));
  pp.W[0] = Wm; pp.k_hi[0] = k_hi; pp.k_lo[0] = k_lo; pp.t_hi[0] = t_hi; pp.t_lo[0] = t_lo;
  pp.n_layers = 1; pp.tasks = 1; pp.split = split ? 1 : 0;
  LAUNCH_N("prep_weights", launch_prep_weights(pp, stream));
  RowsGemmParams p;
  memset(&p, 0, sizeof(p));
  int rc;
  const int bn = rows_gemm_bn(0, 0, split, 0);
  if ((rc = make_map(&p.tmA_hi, a_hi, R, TILE_M))) return rc;
  if ((rc = make_map(&p.tmA_lo, split ? a_lo : a_hi, R, TILE_M))) return rc;
  if ((rc = make_map(&p.tmB_hi, k_hi, H, bn))) return rc;
  if ((rc = make_map(&p.tmB_lo, split ? k_lo : k_hi, H, bn))) return rc;
  p.R = int(R); p.rows_per_task = int(R); p.per_task = 0; p.w0 = 1.f; p.raw_out = out;
  LAUNCH_N("debug_linear", launch_rows_gemm(p, 2, 0, 0, split, num_sms(), stream));
  return SIREN_OK;
}

int siren_b200_debug_wgrad(const float* A, const float* B, float* dWm, long R, int precision, void* scratch,
                           void* stream_) {
  if (!A || !B || !dWm || !scratch || R <= 0 || R % TILE_M) return fail(SIREN_ERR_INVALID, "bad debug_wgrad args");
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  const bool split = precision == SIREN_PREC_FP32_PARITY;
  char* s = reinterpret_cast<char*>(scratch);
  const size_t pl = size_t(R) * H * 2;
  bf16 *a_hi = (bf16*)s, *a_lo = (bf16*)(s + pl), *b_hi = (bf16*)(s + 2 * pl), *b_lo = (bf16*)(s + 3 * pl);
  LAUNCH_N("to_planes", launch_to_planes(A, a_hi, a_lo, R * H, split, stream));
  LAUNCH_N("to_planes", launch_to_planes(B, b_hi, b_lo, R * H, split, stream));
  CUDA_TRY(cudaMemsetAsync(dWm, 0, size_t(H) * H * sizeof(float), stream));
  WgradParams wp;
  memset(&wp, 0, sizeof(wp));
  int rc;
  const int kc = wgrad_kc(split);
  if ((rc = make_map(&wp.tmA_hi[0], a_hi, R, kc))) return rc;
  if ((rc = make_map(&wp.tmA_lo[0], split ? a_lo : a_hi, R, kc))) return rc;
  if ((rc = make_map(&wp.tmB_hi[0], b_hi, R, kc))) return rc;
  if ((rc = make_map(&wp.tmB_lo[0], split ? b_lo : b_hi, R, kc))) return rc;
  wp.dW[0] = dWm; wp.n_layers = 1; wp.S = 1; wp.R = int(R); wp.rows_per_task = int(R); wp.per_task = 0; wp.tasks = 1;
  const int tiles = int(R / TILE_M);
  wp.slices = tiles < num_sms() ? tiles : num_sms();
  LAUNCH_N("wgrad", launch_wgrad(wp, split, num_sms(), stream));
  return SIREN_OK;
}

}  // extern "C"
