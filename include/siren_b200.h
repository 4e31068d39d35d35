/* siren_b200 -- C ABI of the B200-native SIREN hot path.
 *
 * The reference (jonbmartin/siren_mri) is pure Python/PyTorch: it has no FFI for this path.  The
 * boundary it does have is the nn.Module contract of modules.py; the host-side mirror of that
 * contract lives in siren_mri_b200/modules.py and calls the entry points below through ctypes.
 * Each entry point states which reference code it stands in for (paths relative to the reference
 * root).
 *
 * Conventions
 *   - plain C, no libtorch types: raw device pointers, sizes, a cudaStream_t passed as void*.
 *   - every call is asynchronous on the given stream, allocates nothing, never synchronises and
 *     is CUDA-graph capturable.  The caller owns all memory, including the workspace.
 *   - return value 0 = success; non-zero = error code, message via siren_b200_last_error()
 *     (thread-local).  Nothing throws or aborts across the boundary.
 *   - all tensors are contiguous fp32 unless stated otherwise.
 */
#ifndef SIREN_B200_H_
#define SIREN_B200_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SIREN_B200_VERSION 1

/* error codes */
#define SIREN_OK 0
#define SIREN_ERR_UNSUPPORTED 1   /* shape / device outside the native envelope            */
#define SIREN_ERR_INVALID 2       /* bad argument                                          */
#define SIREN_ERR_CUDA 3          /* CUDA runtime / driver error                           */

/* precision of the tensor-core layers */
#define SIREN_PREC_FP32_PARITY 0  /* bf16 hi/lo split operands, 3 MMAs per product, fp32 stash */
#define SIREN_PREC_BF16 1         /* single 16-bit operands (fp16 activations / weights in the forward, bf16      */
                                  /* adjoints in the backward), fp32 accumulate, one fp16 stash plane per layer   */

/* Problem descriptor.  Mirrors the constructor arguments of modules.SingleBVPNet /
 * modules.FCBlock (modules.py:45-46, 125-126) plus the batch geometry of one call. */
typedef struct {
  int d_in;          /* in_features: <= 16; 17..256 with deriv_order 0 and without coordinate  */
                     /* gradient (bf16: the whole-MLP kernels; fp32-parity: per layer)            */
  int hidden;        /* hidden_features; the native kernels serve 256                          */
  int n_hidden;      /* num_hidden_layers (hidden x hidden linears), 1..8                      */
  int d_out;         /* out_features (<= 8)                                                    */
  float w0;          /* Sine.w0 (modules.py:31-38)                                             */
  int tasks;         /* leading batch dimension B of model_input['coords'] ([B, N, d])        */
  int per_task;      /* 1: weights are [B, out, in] / biases [B, out] (hypernetwork output,    */
                     /*    meta_modules.py:50-54); 0: shared [out, in] / [out]                 */
  long n_coords;     /* N, coordinates per task; any positive value (ragged tails are masked)  */
  int precision;     /* SIREN_PREC_*                                                           */
  int deriv_order;   /* 0: value only; 1: + dy/dx_k; 2: + d2y/dx_k^2  (needs d_in <= 3)        */
} siren_desc_t;

int siren_b200_version(void);
const char* siren_b200_last_error(void);

/* 0 when the current CUDA device is an sm_100 part the kernels can run on. */
int siren_b200_device_ok(void);

/* Bytes of workspace a forward(+backward) needs.  The same buffer must be handed to backward
 * unchanged: it holds the activation / cosine / jet stash between the two calls.  0 on error. */
size_t siren_b200_workspace_bytes(const siren_desc_t* desc);
/* The same with the caller's intent: want_gcoords = 0 promises that siren_b200_backward will be called with
 * gcoords == NULL, which saves the layer-0 adjoint plane on the fused bf16 path (512 B per coordinate).
 * siren_b200_workspace_bytes(desc) == siren_b200_workspace_bytes_ex(desc, 1). */
size_t siren_b200_workspace_bytes_ex(const siren_desc_t* desc, int want_gcoords);

/* Forward of the sine MLP.
 * Replaces: SingleBVPNet.forward -> FCBlock.forward -> MetaSequential[BatchLinear, Sine] x (n_hidden+1)
 *           + BatchLinear (modules.py:146-164, 92-97, 16-27, 35-38) and, for deriv_order > 0,
 *           the values diff_operators.gradient / divergence / laplace (diff_operators.py:27-43)
 *           would obtain by double backward.
 *   coords [tasks, n_coords, d_in]
 *   W[l], b[l], l = 0..n_hidden+1: device pointers (host array of n_hidden+2 entries)
 *   y  [tasks, n_coords, d_out]
 *   J  [tasks, n_coords, d_out, d_in]   dy_o/dx_k        (deriv_order >= 1, else NULL)
 *   D  [tasks, n_coords, d_out, d_in]   d2y_o/dx_k^2     (deriv_order == 2, else NULL)
 */
int siren_b200_forward(const siren_desc_t* desc, const float* coords, const float* const* W,
                       const float* const* b, float* y, float* J, float* D, void* workspace, void* stream);

/* Forward for inference (value only, no backward will follow): same result as siren_b200_forward, but the
 * stash the backward would need is not written (bf16 mode: the cosine planes and, with d_out <= 2, the top
 * layer's activation plane stay on chip).  Replaces the torch.no_grad() uses of the same modules
 * (sdf_meshing.py:46-56, utils.py:275-304).  The workspace is still required (layer-to-layer planes).
 * bf16 mode (training forward and this entry alike): the sine argument w0 (z + b) goes to the SFU as it is; the SFU's
 * own 1/(2 pi) scaling keeps the absolute error below |arg| * 2^-23 (checked up to ~360 rad,
 * tests/test_gpu_fused.py::test_large_argument_sine), far under the fp16 rounding of the result.  The fp32-parity mode
 * reduces the argument exactly and uses sincosf. */
int siren_b200_forward_infer(const siren_desc_t* desc, const float* coords, const float* const* W,
                             const float* const* b, float* y, void* workspace, void* stream);

/* Backward (reverse of the forward above, including the reverse of the jet streams).
 * Replaces: the autograd backward training.py:91 triggers through modules.py:25-26,38, i.e.
 *           per layer dz = dh * w0 cos(w0 z), dh_prev = dz W, dW = dz^T h_prev, db = sum dz, and
 *           the second / third order graphs built by diff_operators.py:27-43.
 *   gy [tasks, n, d_out], gJ / gD [tasks, n, d_out, d_in] (NULL = zero)
 *   dW[l], db[l]: outputs shaped like W[l], b[l]; overwritten unless accumulate != 0
 *   gcoords [tasks, n, d_in] or NULL: adjoint reaching the coordinates through the first layer
 */
int siren_b200_backward(const siren_desc_t* desc, const float* coords, const float* const* W,
                        const float* const* b, const void* workspace, const float* gy, const float* gJ,
                        const float* gD, float* const* dW, float* const* db, float* gcoords, int accumulate,
                        void* stream);

/* ---- Fourier-feature prologue (MRI neural-process scripts) ---------------------------------------------------
 * Replaces: features.GaussianFourierFeatureTransform.forward (features.py:31-41: x @ B, times 2 pi, cat[sin, cos])
 *           applied to model_input['coords'] by the training loops (training.py:61-64, training_ddp.py:66-69) before
 *           the model is called.  The [tasks, n, 2 F] feature tensor is never materialised: the first layer's operand
 *           producer (and, in the backward, the kernel that forms dW_0) builds the features of a row from its raw
 *           coordinates.  desc->d_in must equal 2 * n_features, 3 <= n_features <= 128 (see siren_desc_t for the
 *           envelope above 16 inputs), deriv_order 0.
 *   B [raw_dim, n_features] fp32 device pointer (GaussianFourierFeatureTransform._B_spatial), raw_dim <= 3
 *   raw_coords [tasks, n_coords, raw_dim]
 * forward_ff:  siren_b200_forward (inference == 0) / siren_b200_forward_infer (inference != 0) on those features.
 * backward_ff: siren_b200_backward on the same workspace; there is no gradient w.r.t. the raw coordinates. */
typedef struct {
  const float* B;
  int n_features;
  int raw_dim;
} siren_fourier_t;
int siren_b200_forward_ff(const siren_desc_t* desc, const siren_fourier_t* ff, const float* raw_coords,
                          const float* const* W, const float* const* b, float* y, void* workspace, int inference,
                          void* stream);
int siren_b200_backward_ff(const siren_desc_t* desc, const siren_fourier_t* ff, const float* raw_coords,
                           const float* const* W, const float* const* b, const void* workspace, const float* gy,
                           float* const* dW, float* const* db, int accumulate, void* stream);

/* ---- k-space data-consistency epilogue (MRI neural-process models) --------------------------------------------
 * Replaces: data_consistency.DataConsistencyInKspace.forward -> data_consistency() (data_consistency.py:7-20, 32-47),
 *           which meta_modules.py:217-219 applies to model_out right behind the hypo-network:
 *             out = (1 - mask) pred + mask k0                          (noise_lvl == 0)
 *             out = (1 - mask) pred + mask (pred + v k0) / (1 + v)     (noise_lvl = v > 0)
 *           and its autograd backward (the output adjoint scaled by 1 - mask, resp. 1 - mask v / (1 + v)).
 *           On the fused bf16 path (d_out <= 2) the thread that completes a row's y applies the blend before it
 *           stores y, and the input-gradient chain scales gy as it picks it up: no pass over [tasks, n, d_out] is left.
 *           Elsewhere the library runs one elementwise launch on either side.
 *   k0, mask: channels_first != 0: [tasks, d_out, n_coords] -- the datasets' [B, 2, nx, ny] as they are (the permute +
 *             view of data_consistency.py:40-45 is an index map); channels_first == 0: [tasks, n_coords, d_out].
 *   ff: optional Fourier prologue (NULL: coords are the first layer's inputs).
 * forward_dc:     siren_b200_forward / _forward_ff (inference != 0: the no-stash variants) with y data-consistent.
 * backward_dc:    siren_b200_backward / _backward_ff where gy is the adjoint of that data-consistent y.
 * forward_dc_mse: forward_dc that also forms image_mse(y_dc, gt) (loss_functions.py:66-96, high_freq False) into
 *                 loss4[1] and ITS gradient w.r.t. the network output, gy = 2 weight (y_dc - gt) (1 - mask pull):
 *                 follow it with the PLAIN siren_b200_backward / _backward_ff. */
typedef struct {
  const float* k0;
  const float* mask;
  float noise_lvl;       /* 0: noiseless */
  int channels_first;
} siren_dc_t;
int siren_b200_forward_dc(const siren_desc_t* desc, const siren_fourier_t* ff, const siren_dc_t* dc, const float* coords,
                          const float* const* W, const float* const* b, float* y, void* workspace, int inference,
                          void* stream);
int siren_b200_backward_dc(const siren_desc_t* desc, const siren_fourier_t* ff, const siren_dc_t* dc, const float* coords,
                           const float* const* W, const float* const* b, const void* workspace, const float* gy,
                           float* const* dW, float* const* db, int accumulate, void* stream);
int siren_b200_forward_dc_mse(const siren_desc_t* desc, const siren_fourier_t* ff, const siren_dc_t* dc,
                              const float* coords, const float* const* W, const float* const* b, float* y,
                              const float* gt, float weight, float* gy, float* loss4, void* workspace, void* stream);

/* ---- hypernetwork head in the consumer's layout (MRI neural-process models) -----------------------------------
 * hyper_head replaces, for one HIDDEN weight matrix of the hypo-network, three passes of the reference flow:
 *   - the last linear of its HyperNetwork head, meta_modules.py:32-35, 50-54 (FCBlock(..., outermost_linear=True,
 *     'relu').net[-1] = BatchLinear(hyper_hidden -> 256 * 256), reshaped to [B, 256, 256]);
 *   - the conversion of that fp32 tensor into the tensor-core operands every forward call starts with;
 *   - the sum of squares loss_functions.hypo_weight_loss adds up (loss_functions.py:279-287).
 * One pass over Wlast writes  W_out [tasks, 256, 256] fp32 (the hypo_params entry),  wk16 [tasks * 256, 256] fp16 (as
 * stored: the fused forward's operand),  wt16 [tasks * 256, 256] bf16 = w0 * W^T (the dgrad chain's operand) and adds
 * sum W_out^2 to *sumsq (wk16 / wt16 / sumsq may be NULL).
 *   h [tasks, k_h]: the head's last hidden activation;  Wlast [65536, k_h], blast [65536]: its last linear;
 *   k_h a multiple of 4, <= 512.
 * forward_call / backward_call: the general form of the value-path entry points -- optional Fourier prologue, optional
 * data-consistency epilogue, optional READY-MADE weight operands (wk16 / wt16: host arrays of n_hidden device pointers,
 * hidden layer l + 1 at index l, e.g. written by hyper_head); with them the call converts no weights at all.  The
 * operands are taken by the fused bf16 path only (SIREN_ERR_UNSUPPORTED otherwise); forward needs wk16, backward wt16. */
typedef struct {
  const siren_fourier_t* fourier;   /* NULL: coords are the first layer's inputs */
  const siren_dc_t* dc;             /* NULL: no data consistency */
  const void* const* wk16;          /* NULL: the call converts W itself */
  const void* const* wt16;
} siren_call_t;
int siren_b200_hyper_head(const float* h, const float* Wlast, const float* blast, int tasks, int k_h, float w0,
                          float* W_out, void* wk16, void* wt16, float* sumsq, void* stream);
int siren_b200_forward_call(const siren_desc_t* desc, const siren_call_t* call, const float* coords,
                            const float* const* W, const float* const* b, float* y, void* workspace, int inference,
                            void* stream);
int siren_b200_backward_call(const siren_desc_t* desc, const siren_call_t* call, const float* coords,
                             const float* const* W, const float* const* b, const void* workspace, const float* gy,
                             float* const* dW, float* const* db, int accumulate, void* stream);

/* ---- the fast training step (image-MSE fit): three launches per step on the fused bf16 path ---------------
 * forward_backward_mse (= forward_mse -> backward: forward, loss gradient and dgrad chain in one kernel, then the
 * weight gradients) -> [allreduce] -> adam_step.
 * Replaces the loop body training.py:66-103 (model -> loss_functions.image_mse -> backward -> clip -> Adam.step
 * -> zero_grad) for a sine FCBlock whose parameters live in one flat buffer.
 *
 * prepare_weights: the bf16 copies of the hidden weights (as stored and transposed) the tensor-core kernels
 *   read, written into the workspace.  siren_b200_forward does this itself on every call; the training step
 *   does it ONCE (and after any outside change of the weights): adam_step keeps the copies current.
 * forward_prepared: siren_b200_forward without that conversion.
 * forward_mse: the training forward that also forms the loss image_mse(y, gt) (loss_functions.py:66-96, high_freq
 *   False) and its gradient: gy = 2 weight (y - gt) and weight * sum (y - gt)^2 accumulated into loss4[1] -- by the
 *   thread that completes a row's y inside the fused forward kernel (bf16 mode, d_out <= 2), by one mse_grad launch
 *   behind the forward otherwise.  weights_ready != 0 skips the weight conversion (see prepare_weights).
 *   loss4: four device floats, zero-initialised once: [0] = loss of the last step adam_step finished,
 *   [1] = running sum of the step in flight.
 * adam_step: siren_b200_adam in one launch (two with clipping), which additionally clears the gradient it
 *   consumed (zero_grad != 0), moves loss4[1] to loss4[0], and -- when desc / W / workspace are given and the
 *   hidden weights W[1..n_hidden] live inside the flat parameter buffer -- rewrites their bf16 copies in the
 *   workspace from the updated values. */
int siren_b200_prepare_weights(const siren_desc_t* desc, const float* const* W, void* workspace, void* stream);
int siren_b200_forward_prepared(const siren_desc_t* desc, const float* coords, const float* const* W,
                                const float* const* b, float* y, float* J, float* D, void* workspace, void* stream);
int siren_b200_forward_mse(const siren_desc_t* desc, const float* coords, const float* const* W,
                           const float* const* b, float* y, const float* gt, float weight, float* gy, float* loss4,
                           void* workspace, int weights_ready, void* stream);
/* forward_backward_mse: forward_mse followed by backward (gJ = gD = null, no coordinate gradient) on the same arguments.
 *   On the fused bf16 path with d_in <= 4, d_out <= 2 and at most 4 hidden layers it is ONE kernel for the forward,
 *   the loss gradient and the input-gradient chain (gy never leaves the chip, the top layer leaves no stash plane),
 *   plus the weight-gradient launch; elsewhere, and with SIREN_FUSED_STEP=0, the two calls.  gy may be null: the
 *   loss gradient is then not written out. */
int siren_b200_forward_backward_mse(const siren_desc_t* desc, const float* coords, const float* const* W,
                                    const float* const* b, float* y, const float* gt, float weight, float* gy,
                                    float* loss4, void* workspace, int weights_ready, float* const* dW,
                                    float* const* db, int accumulate, void* stream);
/* ---- scenes of different sizes in one step (one SIREN per image of a collection whose images differ in size) ------
 * desc->per_task = 1, desc->tasks = T <= 1024 scenes, scene t with n_host[t] >= 1 coordinates (host array of T longs;
 * desc->n_coords is not read).  Coordinates, gt, y and gy are PACKED: [sum n_t, d] without gaps, scene t from row
 * sum_{s<t} n_s.  The workspace planes hold each scene's rows padded to 128, so memory and work follow sum n_t.
 * Envelope: the one-kernel step of forward_backward_mse (bf16, deriv_order 0, d_in <= 4, d_out <= 2, at most 4 hidden
 * layers); SIREN_ERR_UNSUPPORTED elsewhere, SIREN_ERR_INVALID for a count below 1 or per_task != 1.  There is no
 * two-launch form (SIREN_FUSED_STEP is not read).
 * workspace_bytes_ragged: the workspace of these calls (0 on error).
 * prepare_ragged: writes the scenes' prefix tables (first unit, plane row and packed row of each scene, the weight-gradient
 *   items) into the workspace from the counts, by one small kernel that takes them as launch parameters: no copy, CUDA-graph
 *   capturable.  Once per count vector, before the step.
 * ragged_tables: the same tables on the host, for the device of sms SMs (sms <= 0: the current device's); tables has
 *   4 (T + 1) + 1 ints.  Inspection hook.
 * forward_backward_mse_ragged: forward_backward_mse on the packed buffers.  Each scene's weight * sum (y - gt)^2 is added to
 *   task_loss[T + t] (task_loss as for adam_step_tasks) and their total to loss4[1] (loss4 may be NULL): follow it with
 *   adam_step_tasks / clip_grad_tasks with y = gt = NULL. */
size_t siren_b200_workspace_bytes_ragged(const siren_desc_t* desc, const long* n_host);
int siren_b200_prepare_ragged(const siren_desc_t* desc, const long* n_host, void* workspace, void* stream);
int siren_b200_ragged_tables(const siren_desc_t* desc, const long* n_host, int sms, int* tables);
int siren_b200_forward_backward_mse_ragged(const siren_desc_t* desc, const long* n_host, const float* coords,
                                           const float* const* W, const float* const* b, float* y, const float* gt,
                                           float weight, float* gy, float* loss4, float* task_loss, void* workspace,
                                           int weights_ready, float* const* dW, float* const* db, int accumulate,
                                           void* stream);
int siren_b200_adam_step(float* param, float* grad, float* m, float* v, long n, float lr, double beta1,
                         double beta2, float eps, float max_grad_norm, float grad_scale, void* state, int zero_grad,
                         float* loss4, const siren_desc_t* desc, const float* const* W, void* workspace,
                         void* stream);

/* adam_step with the gradient all-reduce FUSED in: the gradient of element i is the sum over the ranks' flat buffers,
 * read straight from peer memory over NVLink / NVSwitch inside the Adam kernel (peer_grads = DEVICE array of `world`
 * device pointers to the ranks' buffers, this rank's own among them; summed in rank order, so replicas stay
 * bit-identical).  Replaces ncclAllReduce + adam_step, i.e. the DDP Reducer + optimizer step of
 * train_mri_neural_process_ddp.py:238 / training.py:101-103, for the single-scene configurations.
 * Protocol (the caller provides the cross-rank ordering, e.g. one symmetric-memory barrier per step): every rank's
 * backward of step k must be complete before any rank runs this call for step k; gradients are DOUBLE-BUFFERED --
 * step k accumulates into buffer k mod 2 and this call clears `zero_buf`, the buffer step k + 1 accumulates into
 * (no rank reads it any more: all of them passed the barrier of step k after finishing step k - 1), so no second
 * barrier is needed. */
int siren_b200_adam_step_peers(float* param, float* grad, float* m, float* v, long n, float lr, double beta1,
                               double beta2, float eps, float max_grad_norm, float grad_scale, void* state,
                               float* loss4, const siren_desc_t* desc, const float* const* W, void* workspace,
                               const float* const* peer_grads, int world, float* zero_buf, void* stream);

/* ---- the optimizer tail of T independent networks in one step (one SIREN per image / slice / frame) ------------
 * Replaces, for each task t on its own: loss_functions.image_mse on scene t (loss_functions.py:66-96), clip_grad_norm_
 * over models[t].parameters() only and torch.optim.Adam.step / zero_grad on them (training.py:23, 88-103) -- T reference
 * loops that share the step counter, lr, betas and eps.
 * desc->per_task = 1, desc->tasks = T <= 1024.  The parameters live in one flat buffer of n floats: W[l] / b[l] point
 * to [T, out, in] / [T, out] blocks inside it, which must tile the buffer exactly (SIREN_ERR_INVALID otherwise); grad,
 * m and v share that layout.  The caller owns the per-task state, zero-initialised once:
 *   task_sumsq [T]:  each task's squared gradient norm between the launches of one step;
 *   task_loss [2T]:  [0, T) each task's loss of the last finished micro-batch, [T, 2T) the running sums;
 *   loss4 (or NULL): moved [1] -> [0] whenever task_loss is published (forward_backward_mse adds the sum over tasks).
 * y, gt [T, n_coords, d_out] (both or neither): the step's output and target; given, the call adds
 * weight * sum (y - gt)^2 over each task's rows to task_loss[T + t] -- in the norm pass with clipping, in the Adam
 * launch otherwise.
 * adam_step_tasks: siren_b200_adam_step per task: clip by the task's own norm (max_grad_norm > 0), Adam, the
 *   gradient cleared, the running losses published and -- workspace given -- every task's fp16 / bf16 hidden-weight
 *   copies rewritten as prepare_weights would.  One launch, two with clipping.  y = gt = NULL: the losses of this
 *   micro-batch are already in task_loss[T, 2T) (clip_grad_tasks).
 * clip_grad_tasks: a micro-batch that ends without an optimizer step (gradient accumulation, training.py:90-103):
 *   the loss pass and, with max_grad_norm > 0, each task's ACCUMULATED gradient clipped in place by its own norm;
 *   publish != 0 publishes the losses (the step ends here).  dW / db: the gradient's views, as W / b above. */
int siren_b200_adam_step_tasks(const siren_desc_t* desc, const float* const* W, const float* const* b, float* param,
                               float* grad, float* m, float* v, long n, float lr, double beta1, double beta2, float eps,
                               float max_grad_norm, void* state, const float* y, const float* gt, float weight,
                               float* task_sumsq, float* task_loss, float* loss4, void* workspace, void* stream);
int siren_b200_clip_grad_tasks(const siren_desc_t* desc, float* const* dW, float* const* db, float* grad, long n,
                               float max_grad_norm, void* state, const float* y, const float* gt, float weight,
                               float* task_sumsq, float* task_loss, float* loss4, int publish, void* stream);

/* The two derivative losses of the configurations, on the jets the forward returns (scalar output), with their
 * gradients w.r.t. those jets -- what autograd would hand to siren_b200_backward as gy / gJ / gD.  Each adds the loss
 * value to loss4[1] (see forward_mse).
 * laplace_mse_grad: loss_functions.laplace_mse (loss_functions.py:350-355): mean((sum_k D[n, k] - gt[n])^2);
 *   D, gD [n, d] (d <= 3), gt [n].
 * sdf_grad: loss_functions.sdf (loss_functions.py:460-484) summed as the training loop does (training.py:68-76):
 *   3e3 mean|y| on the surface (sdf != -1) + 1e2 mean exp(-1e2 |y|) off it + 1e2 mean(1 - cos(J, normal)) on it
 *   + 5e1 mean| |J| - 1 |;   y, sdf, gy [n], J, normals, gJ [n, 3].
 * weight multiplies loss and gradients (1 / accumulation_steps, or a shard's share n_local / n_global). */
int siren_b200_laplace_mse_grad(const float* D, const float* gt, float* gD, long n, int d, float weight, float* loss4,
                                void* stream);
int siren_b200_sdf_grad(const float* y, const float* J, const float* sdf, const float* normals, float* gy, float* gJ,
                        long n, float weight, float* loss4, void* stream);

/* Gradient accumulation (training.py:90, 93-103): a micro-batch that does not end in an optimizer step still clips
 * the ACCUMULATED gradient in place (clip_grad: g *= min(1, max_norm / (|g| + 1e-6)), as clip_grad_norm_ does after
 * every backward of the reference loop) and publishes its own loss (loss_roll: loss4[1] -> loss4[0]). */
int siren_b200_clip_grad(float* grad, long n, float max_grad_norm, void* state, void* stream);
int siren_b200_loss_roll(float* loss4, void* stream);

/* Fused (optional clip_grad_norm_) + Adam over one flat parameter buffer.
 * Replaces: torch.nn.utils.clip_grad_norm_ + torch.optim.Adam.step (training.py:23, 93-103);
 *           defaults beta = (0.9, 0.999), eps = 1e-8, no weight decay.
 *   state: SIREN_ADAM_STATE_BYTES of device memory, zero-initialised once by the caller; holds the step
 *          counter, the bias corrections (and the running powers of the betas they come from) and the
 *          squared gradient norm, so that the call is CUDA-graph capturable (each call advances the
 *          step by one).
 *   max_grad_norm <= 0 disables clipping.  grad_scale multiplies the gradient first
 *   (1/world for an all-reduced sum). */
#define SIREN_ADAM_STATE_BYTES 64
int siren_b200_adam(float* param, const float* grad, float* m, float* v, long n, float lr, double beta1,
                    double beta2, float eps, float max_grad_norm, float grad_scale, void* state, void* stream);

/* gy = 2 * weight * (y - gt); *loss += weight * sum (y - gt)^2   (loss may be NULL).
 * Replaces: loss_functions.image_mse with high_freq=False (loss_functions.py:66-96,
 *           weight = 1/16384) and its autograd backward; used by the fast training step. */
int siren_b200_mse_grad(const float* y, const float* gt, float* gy, long n, float weight, float* loss,
                        void* stream);

/* n <= 1024 floats from device memory to pinned (page-locked, device-mapped) host memory, written by a kernel.
 * Replaces: the per-step `train_loss.item()` / `writer.add_scalar` reads of the training loop (training.py:77-104,
 *           a blocking copy each): the logged scalars leave the GPU as posted stores at the end of the step's CUDA
 *           graph instead of through the copy engine, whose hand-over costs ~35 us per step on the compute stream.
 *   The values are visible to the host once an event recorded after the call has completed. */
int siren_b200_publish(const float* src, float* dst_host, int n, void* stream);

/* Gradient all-reduce over the GPUs of one box: ONE ncclAllReduce(sum, fp32) on the flat gradient buffer.
 * Replaces: the DDP Reducer path (train_mri_neural_process_ddp.py:238, training_ddp.py:155-164) for the
 *           single-scene configurations.  NCCL is resolved at run time (dlopen of libnccl.so.2, i.e. the copy
 *           PyTorch already loaded).  Rank 0 creates the 128-byte id, the host hands it to the other ranks.
 *   The all-reduce is asynchronous on the given stream and CUDA-graph capturable. */
#define SIREN_COMM_ID_BYTES 128
int siren_b200_comm_unique_id(void* id_out);
int siren_b200_comm_init(int rank, int world, const void* id, void** comm_out);
int siren_b200_allreduce(void* comm, float* buf, long n, void* stream);
int siren_b200_comm_destroy(void* comm);
const char* siren_b200_comm_last_error(void);

/* All-reduce (sum, fp32, in place) of a flat buffer over the GPUs of one box through PEER MEMORY, as one kernel per
 * rank: rank r sums slice r of every rank's buffer (loads over NVLink / NVSwitch, in rank order) and stores the total,
 * times `scale`, into slice r of EVERY rank's buffer (stores over NVLink) -- reduce-scatter and all-gather in one pass,
 * no staging buffer, every replica receives the same bits.
 * Replaces: the DDP Reducer's bucketed ncclAllReduce over the 31.3 M parameters of the neural-process models
 *           (train_mri_neural_process_ddp.py:238) when their gradients live in one flat symmetric-memory buffer
 *           (siren_mri_b200.parallel.PeerGradientReducer).
 *   peers: DEVICE array of `world` device pointers to the ranks' buffers (this rank's own among them), n floats
 *          each, n a multiple of 4, world <= 16.
 * The caller orders the ranks: every rank's buffer is complete before any rank launches this, and every rank's launch
 * is complete before any rank reads its buffer (e.g. one symmetric-memory barrier on either side). */
int siren_b200_allreduce_peers(float* const* peers, int world, int rank, long n, float scale, void* stream);

/* The same all-reduce through the NVSwitch MULTICAST mapping of the buffer (NVLS; `mc` = the multicast address of the
 * symmetric allocation, e.g. torch's _SymmetricMemory.multicast_ptr): rank r reads slice r with multimem.ld_reduce (the
 * switch sums the ranks' copies in fp32) and broadcasts the total, times `scale`, with multimem.st.  A rank moves its
 * slice once per direction instead of world - 1 times.  Same ordering duties as siren_b200_allreduce_peers. */
int siren_b200_allreduce_multicast(float* mc, int world, int rank, long n, float scale, void* stream);

/* Per-kernel timing for bench.py: between begin and end every kernel launched by this thread
 * through the calls above is bracketed by CUDA events on its stream.  end() synchronises on those
 * events and writes one line per kernel, "name launches total_ms\n", into buf. */
int siren_b200_profile_begin(void);
int siren_b200_profile_end(char* buf, size_t buflen);

/* ---- test hooks: the bare tensor-core cores, used by tests/ to localise layout errors ---- */
/* out[R,256] = A[R,256] * W[256,256]^T   (R multiple of 128; scratch >= 8*R*256 + 1 MiB bytes) */
int siren_b200_debug_linear(const float* A, const float* W, float* out, long R, int precision, void* scratch,
                            void* stream);
/* dW[256,256] = A[R,256]^T * B[R,256]    (same scratch rule) */
int siren_b200_debug_wgrad(const float* A, const float* B, float* dW, long R, int precision, void* scratch,
                           void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SIREN_B200_H_ */
