// Host-side declarations of the kernel launchers (internal; the public boundary is
// include/siren_b200.h).
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"

// The dynamic shared-memory limit of a kernel is a PER-DEVICE attribute: one process may drive several GPUs
// (nn.DataParallel threads, cuda:1 after cuda:0), so the "already set" flag is kept per device.  Racing threads
// write the same value.
#define SIREN_ENSURE_SMEM(kern, bytes)                                                                     \
  do {                                                                                                     \
    static bool _set[64];                                                                                  \
    int _dev = 0;                                                                                          \
    if (cudaGetDevice(&_dev) != cudaSuccess) _dev = -1;                                                    \
    if (_dev < 0 || _dev >= 64 || !_set[_dev]) {                                                           \
      cudaError_t _e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);     \
      if (_e != cudaSuccess) return _e;                                                                    \
      if (_dev >= 0 && _dev < 64) _set[_dev] = true;                                                       \
    }                                                                                                      \
  } while (0)

namespace siren {

// device-resident optimizer state (SIREN_ADAM_STATE_BYTES = 64, zero-initialised by the caller)
struct AdamState {
  float sumsq;      // squared global gradient norm of the current step (clip)
  float bc1;        // 1 - beta1^step
  float bc2_sqrt;   // sqrt(1 - beta2^step)
  float pad;
  long step;        // completed steps
  long pad2;        // low word: blocks of the running launch that have finished (adam_step, clip_grad)
  double pow1;      // beta1^step, beta2^step kept as running products (started afresh at step 1; 0 after an underflow
  double pow2;      // stays 0): the bias corrections cost every block of adam_step two multiplications, not two pow()
  double pad3[2];
};
static_assert(sizeof(AdamState) == 64, "AdamState layout");

struct FirstParams {
  const float* x;        // [tasks][n][d]
  const float* W;        // [tasks?][H][d]
  const float* b;        // [tasks?][H]
  bf16 *act_hi, *act_lo; // layer-0 act planes [S][R][H]
  void* c;               // layer-0 cos stash
  bf16 *adj_hi, *adj_lo; // layer-0 adjoint planes (backward)
  float* dW;             // [tasks?][H][d]
  float* db;             // [tasks?][H]
  float* gx;             // [tasks][n][d] or null
  int R, n_pad, n, d, order, per_task;
  float w0;
  int rows_per_block;
  int only_gx;           // skip dW0/db0 (already produced by the fused dgrad epilogue)
  FourierSpec ff;        // ff.B != null (d > 4): x holds RAW coordinates [tasks][n][ff.raw]; the layer's d = 2 ff.F
                         // inputs are their Gaussian Fourier features, built on chip (common.cuh)
};

struct LastParams {
  const float* W;        // [tasks?][o][H]
  const float* b;        // [tasks?][o]
  const bf16 *act_hi, *act_lo;  // top sine layer act planes
  const void* c;         // top sine layer cos stash
  const void* phase;     // or: the fused forward's stash of the layer, the signed sine (fp16, common.cuh): sine as it
                         // is, cosine = +-sqrt(1 - sin^2)
  const void* jz;        // top sine layer Jz/Dz stash
  float *y, *J, *Dd;     // forward outputs [tasks][n][o], [tasks][n][o][d] x2
  const float *gy, *gJ, *gD;
  bf16 *adj_hi, *adj_lo; // adjoint planes of the top sine layer
  float* dW;             // [tasks?][o][H]
  float* db;             // [tasks?][o]
  int R, n_pad, n, d, o, order, per_task;
  float w0;
  int rows_per_block;
};

// fp32 hidden weights -> bf16 (hi, lo), as stored ("k": [out][in]) and transposed ("t": [in][out])
struct PrepParams {
  const float* W[8];
  bf16 *k_hi[8], *k_lo[8], *t_hi[8], *t_lo[8];
  int n_layers, tasks, split;
  float scale_t;     // factor folded into the transposed copies (w0 on the fused bf16 path: the dgrad chain's
                     // accumulator then needs cos(theta) only; 1 otherwise)
  int k_f16;         // fused bf16 path: the as-stored copy (forward operand) is fp16, not bf16 (mlp_fused_pair.cu)
};
cudaError_t launch_prep_weights(const PrepParams& p, cudaStream_t stream);
cudaError_t launch_prep_first(const float* W0, bf16* w0k, int tasks, int d, cudaStream_t stream);
cudaError_t launch_first_fwd(FirstParams p, bool split, int num_sms, cudaStream_t stream);
cudaError_t launch_first_bwd(FirstParams p, bool split, int num_sms, cudaStream_t stream);
cudaError_t launch_last_fwd(LastParams p, bool split, int num_sms, cudaStream_t stream);
cudaError_t launch_last_bwd(LastParams p, bool split, int num_sms, cudaStream_t stream);
cudaError_t launch_featurize(FirstParams p, int num_sms, cudaStream_t stream);
cudaError_t launch_pad_w0(const float* W0, bf16* hi, bf16* lo, int d, long rows, int num_sms, cudaStream_t stream);
cudaError_t launch_unpad_dw0(const float* pad, float* dW0, int d, long rows, int num_sms, cudaStream_t stream);
// column sums of hi + lo adjoint planes: db_0 of a wide first layer (d > 16) in fp32-parity mode
cudaError_t launch_colsum(const bf16* hi, const bf16* lo, float* db, int R, int n_pad, int per_task, int num_sms,
                          cudaStream_t stream);
cudaError_t launch_sumsq(const float* g, long n, float* out, int num_sms, cudaStream_t stream);
cudaError_t launch_sumsq_peers(const float* const* peers, int world, long n, float* out, int num_sms, cudaStream_t stream);
cudaError_t launch_adam(float* p, const float* g, float* m, float* v, long n, float lr, double b1, double b2,
                        float eps, float max_norm, float grad_scale, AdamState* st, int num_sms,
                        cudaStream_t stream);
// clip + Adam + step tick in ONE launch, which also clears the gradient it consumed, refreshes the bf16 copies of
// the hidden weights the tensor-core kernels read, and finalises the step's loss (training step of trainer.py)
struct AdamFusedParams {
  float *p, *g, *m, *v;
  long n;
  float lr, eps, max_norm, grad_scale;
  double b1, b2;
  AdamState* st;
  int zero_grad;
  // world > 1: the gradient is the SUM over the ranks' flat buffers, read straight from peer memory over NVLink (peers =
  // device array of `world` pointers, this rank's own buffer among them, summed in rank order on every rank so the
  // replicas stay bit-identical); `zero_buf` (the buffer the NEXT step accumulates into) is cleared instead of `g`
  const float* const* peers;
  int world;
  float* zero_buf;
  float* loss4;             // [0] loss of the last finished step, [1] running sum of this step; or null
  int n_w;                  // hidden weight matrices inside the flat buffer whose bf16 copies are refreshed
  long w_off[8];            // offset of hidden weight l in the flat buffer ([H][H] floats each)
  bf16 *k_hi[8], *k_lo[8], *t_hi[8], *t_lo[8];
  int split;
  float scale_t;
  int k_f16;                // as PrepParams::k_f16
};
cudaError_t launch_adam_fused(const AdamFusedParams& a, int num_sms, cudaStream_t stream);

// The optimizer tail of T independent networks stacked in one flat buffer (SirenTrainer with several scenes): every
// parameter s holds the tasks' copies one after the other, [T][seg_per[s]] floats at seg_off[s]; the segments tile
// the buffer.  Each task is clipped by its own gradient norm and has its own image_mse loss.
constexpr int MAX_TASK_SEGS = 20;      // W and b of at most 10 layers
constexpr int MAX_TASKS = 1024;
// Scenes of different sizes in one training step (siren_b200_prepare_ragged): scene t has n_t >= 1 coordinates,
// packed [sum n_t][.] without gaps, and ceil(n_t / 128) * 128 rows in the workspace planes.  The prefix tables, int32,
// [T + 1] entries each (entry T is the total):
//   RAG_UNIT   first unit (pair of 256-row tiles of a CTA pair) of the one-kernel step
//   RAG_PROW   first plane row
//   RAG_XROW   first packed row (the scene's count is the difference to the next entry)
//   RAG_SLICE  first weight-gradient slice: scene t is cut into ceil(tiles_t / K) slices of about K 128-row tiles,
//              at least one; the items are (slice, hidden layer) pairs
// followed by K itself.
enum { RAG_UNIT = 0, RAG_PROW = 1, RAG_XROW = 2, RAG_SLICE = 3, RAG_TABLES = 4 };
__host__ __device__ inline int ragged_table_ints(int T) { return RAG_TABLES * (T + 1) + 1; }
__host__ __device__ inline void ragged_tables(const long* n, int T, int K, int* tab) {
  const int S = T + 1;
  int unit = 0, prow = 0, xrow = 0, slice = 0;
  for (int t = 0; t <= T; ++t) {
    tab[RAG_UNIT * S + t] = unit;
    tab[RAG_PROW * S + t] = prow;
    tab[RAG_XROW * S + t] = xrow;
    tab[RAG_SLICE * S + t] = slice;
    if (t == T) break;
    const int tiles = int((n[t] + 127) / 128);
    const int pairs = (tiles + 1) / 2;
    unit += (pairs + 1) / 2;
    prow += tiles * 128;
    xrow += int(n[t]);
    slice += (tiles + K - 1) / K;
  }
  tab[RAG_TABLES * S] = K;
}
struct RaggedPrepParams {
  long n[MAX_TASKS];
  int T, K;
  int* tab;
};
cudaError_t launch_prepare_ragged(const RaggedPrepParams& p, cudaStream_t stream);
cudaError_t launch_mlp_fused_step_ragged(const MlpStepParams& p, int num_sms, cudaStream_t stream);
cudaError_t launch_wgrad_ragged(const WgradParams& p, int grid, cudaStream_t stream);

struct TaskTail {
  int n_seg, tasks;
  long seg_off[MAX_TASK_SEGS];
  int seg_per[MAX_TASK_SEGS];
  int seg_cum[MAX_TASK_SEGS + 1];  // prefix sums of seg_per: one task's parameters as one index range
  int seg_hidden[MAX_TASK_SEGS];   // hidden layer (0-based) whose bf16 / fp16 copies segment s refreshes, or -1
  float max_norm;                  // > 0: clip each task by its own norm
  float* sumsq;                    // [T] squared gradient norm per task (the caller's, cleared by the last launch)
  float* loss;                     // [2T]: [0, T) loss of the last finished micro-batch, [T, 2T) running sum
  float* loss4;                    // or null: loss4[1] -> loss4[0] with the publication (sum over the tasks)
  const float *y, *gt;             // [T][rows] network output and target of the step (null: no loss pass)
  long rows;                       // n_coords * d_out
  float weight;                    // image_mse weight of this micro-batch
  int publish;                     // the launch's last block moves the running losses to the finished ones
};
// squared gradient norm of each task (clip) and / or each task's loss, accumulated into sumsq / loss[T..2T)
cudaError_t launch_task_norms(const float* g, const TaskTail& tt, AdamState* st, int num_sms, cudaStream_t stream);
// g of task t *= min(1, max_norm / (|g_t| + 1e-6)) in place (accumulation micro-batches)
cudaError_t launch_task_clip(float* g, long n, const TaskTail& tt, AdamState* st, int num_sms, cudaStream_t stream);
// adam_fused with per-task clip coefficients, per-task weight copies and, given y / gt, the loss pass folded in
cudaError_t launch_adam_tasks(const AdamFusedParams& a, const TaskTail& tt, int num_sms, cudaStream_t stream);
cudaError_t launch_laplace_mse_grad(const float* D, const float* gt, float* gD, long n, int d, float weight, float* loss,
                                    int num_sms, cudaStream_t stream);
cudaError_t launch_sdf_grad(const float* y, const float* J, const float* sdf, const float* normals, float* gy, float* gJ,
                            long n, float weight, float* loss, int num_sms, cudaStream_t stream);
cudaError_t launch_clip_grad(float* g, long n, float max_norm, AdamState* st, int num_sms, cudaStream_t stream);
cudaError_t launch_loss_roll(float* loss4, cudaStream_t stream);
cudaError_t launch_mse_grad(const float* y, const float* gt, float* gy, long n, float weight, float* loss,
                            int num_sms, cudaStream_t stream);
cudaError_t launch_dc_blend(float* y, const DcSpec& dc, int tasks, int n, int o, int num_sms, cudaStream_t stream);
cudaError_t launch_dc_grad(const float* gy, float* out, const DcSpec& dc, int tasks, int n, int o, int num_sms,
                           cudaStream_t stream);
cudaError_t launch_peer_allreduce(float* const* peers, int world, int rank, long n4, float scale, int num_sms,
                                  cudaStream_t stream);
cudaError_t launch_peer_allreduce_mc(float* mc, int world, int rank, long n4, float scale, int num_sms, cudaStream_t stream);
cudaError_t launch_zero_many(float* const* ptrs, const long* counts, int cnt, int num_sms, cudaStream_t stream);
cudaError_t launch_publish(const float* src, float* dst_host, int n, cudaStream_t stream);
cudaError_t launch_to_planes(const float* src, bf16* hi, bf16* lo, long n, bool split, cudaStream_t stream);

// hypernetwork head in the consumer's layout (hyper_head.cu)
struct HyperHeadParams {
  const float* h;        // [tasks][k_h] last hidden activation of the head
  const float* Wlast;    // [H * H][k_h]
  const float* blast;    // [H * H]
  float* W_out;          // [tasks][H][H] fp32
  __half* wk16;          // [tasks][H][H] fp16 as stored, or null
  bf16* wt16;            // [tasks][H][H] bf16 transposed, times w0, or null
  float* sumsq;          // += sum W_out^2, or null
  int tasks, k_h;
  float w0;
};
cudaError_t launch_hyper_head(const HyperHeadParams& p, cudaStream_t stream);

// tensor-core kernels
cudaError_t launch_rows_gemm(const RowsGemmParams& p, int mode, int order, int d, bool split, int num_sms,
                             cudaStream_t stream);
int rows_gemm_bn(int order, int d, bool split, int mode);
int rows_gemm_cw(int order, int d, bool split, int mode);
cudaError_t launch_mlp_fused_bwd(const MlpBwdParams& p, int num_sms, cudaStream_t stream);
cudaError_t launch_mlp_fused_pair(const MlpFwdParams& p, bool stash, int num_sms, cudaStream_t stream);
cudaError_t launch_mlp_fused_step(const MlpStepParams& p, int num_sms, cudaStream_t stream);
cudaError_t launch_wgrad(const WgradParams& p, bool split, int num_sms, cudaStream_t stream);
int wgrad_kc(bool split);

}  // namespace siren
