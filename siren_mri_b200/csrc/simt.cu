// Small CUDA-core kernels around the tensor-core layers: weight conversion to bf16 (both
// orientations), fused clip + Adam and the MSE loss gradient used by the fast training step.
// (The first/last layers and the bias gradients live in edge_layers.cu.)
#include "common.cuh"
#include "simt.h"

namespace siren {

namespace {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// -------------------------------------------------------------------------------------------
// fp32 weights [T][256][256] -> bf16 (hi, lo) in both orientations
// -------------------------------------------------------------------------------------------
__global__ void prep_weights_kernel(PrepParams p) {
  __shared__ float tile[32][33];
  const int layer = blockIdx.z / p.tasks, task = blockIdx.z - layer * p.tasks;
  const float* __restrict__ W = p.W[layer];
  bf16* __restrict__ k_hi = p.k_hi[layer];
  bf16* __restrict__ k_lo = p.k_lo[layer];
  bf16* __restrict__ t_hi = p.t_hi[layer];
  bf16* __restrict__ t_lo = p.t_lo[layer];
  const size_t base = size_t(task) * H * H;
  const int bx = blockIdx.x * 32, by = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const float v = W[base + size_t(by + i) * H + bx + threadIdx.x];
    tile[i][threadIdx.x] = v;
    const bf16 h = __float2bfloat16_rn(v);
    if (p.k_f16) reinterpret_cast<__half*>(k_hi)[base + size_t(by + i) * H + bx + threadIdx.x] = __float2half_rn(v);
    else k_hi[base + size_t(by + i) * H + bx + threadIdx.x] = h;
    if (p.split) k_lo[base + size_t(by + i) * H + bx + threadIdx.x] = __float2bfloat16_rn(v - __bfloat162float(h));
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const float v = tile[threadIdx.x][i] * p.scale_t;
    const bf16 h = __float2bfloat16_rn(v);
    t_hi[base + size_t(bx + i) * H + by + threadIdx.x] = h;
    if (p.split) t_lo[base + size_t(bx + i) * H + by + threadIdx.x] = __float2bfloat16_rn(v - __bfloat162float(h));
  }
}

// First-layer weights [T][256][d] (4 < d <= 16) as the K-major bf16 B operand of ONE 64-wide K chunk that reproduces
// the fp32 product x W0^T on the tensor core: every value is split into bf16 terms (hi + lo + lolo) and the
// largest cross products are laid out as G = min(6, 64 / d) groups of d columns,
//   B groups  W_hi  W_lo  W_hi  W_lo  W_lolo  W_hi
//   A groups  x_hi  x_hi  x_lo  x_lo  x_hi    x_lolo      (built by the fused forward, mlp_fused_pair.cu)
// columns G d .. 63 are zero.  With d = 16 the four groups leave a relative error of ~2^-16 in z (the dropped
// terms are hi x lolo), i.e. ~1e-3 rad in w0 z: the order of the fp16 phase stash.
__global__ void prep_first_kernel(const float* __restrict__ W0, bf16* __restrict__ w0k, int d) {
  const int row = blockIdx.x * 4 + (threadIdx.x >> 6);        // task * 256 + feature; one thread per (row, column)
  const int k = threadIdx.x & 63;
  if (d > 16) {      // 16 < d <= 256 (bf16 mode only): the inputs fill the chunk(s) themselves, plain bf16, zero padded
    const int kw = ((d + 63) / 64) * 64;
    for (int kk = k; kk < kw; kk += 64)
      w0k[size_t(row) * kw + kk] = __float2bfloat16_rn(kk < d ? W0[size_t(row) * d + kk] : 0.f);
    return;
  }
  const int groups = 64 / d < 6 ? 64 / d : 6;
  const int g = k / d, i = k - g * d;
  float v = 0.f;
  if (g < groups) {
    const float x = W0[size_t(row) * d + i];
    const float h = bf16_round_f(x), l = bf16_round_f(x - h);
    v = (g == 0 || g == 2 || g == 5) ? h : (g == 1 || g == 3) ? l : bf16_round_f(x - h - l);
  }
  w0k[size_t(row) * 64 + k] = __float2bfloat16_rn(v);
}

// -------------------------------------------------------------------------------------------
// optimizer tail: global grad norm (for clip_grad_norm_) and Adam, over one flat buffer
// -------------------------------------------------------------------------------------------
__global__ void sumsq_kernel(const float* __restrict__ g, long n, float* __restrict__ out) {
  float acc = 0.f;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const float v = g[i];
    acc = fmaf(v, v, acc);
  }
  acc = warp_sum(acc);
  __shared__ float part[32];
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? part[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) atomicAdd(out, v);
  }
}

// squared norm of the SUM of the ranks' gradients, each read from peer memory (clip_grad_norm_ of the reduced gradient)
__global__ void sumsq_peers_kernel(const float* const* __restrict__ peers, int world, long n, float* __restrict__ out) {
  float acc = 0.f;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    float v = 0.f;
    for (int r = 0; r < world; ++r) v += peers[r][i];
    acc = fmaf(v, v, acc);
  }
  acc = warp_sum(acc);
  __shared__ float part[32];
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? part[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) atomicAdd(out, v);
  }
}

// one thread: advance the step counter and refresh the bias corrections (in double, like the
// Python-side arithmetic of torch.optim.Adam).  Keeping the counter on the device makes the
// whole optimizer tail CUDA-graph capturable.
__global__ void adam_tick_kernel(AdamState* st, double b1, double b2) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    const long step = st->step + 1;
    st->step = step;
    const double p1 = pow(b1, (double)step), p2 = pow(b2, (double)step);
    st->pow1 = p1;      // adam_step continues from these
    st->pow2 = p2;
    st->bc1 = (float)(1.0 - p1);
    st->bc2_sqrt = (float)sqrt(1.0 - p2);
  }
}

__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, long n, float lr, float b1, float b2, float eps,
                            float max_norm, float grad_scale, const AdamState* __restrict__ st) {
  float scale = grad_scale;
  if (max_norm > 0.f) {
    const float total = sqrtf(st->sumsq) * grad_scale;
    const float coef = max_norm / (total + 1e-6f);
    scale *= fminf(coef, 1.0f);
  }
  const float step_size = lr / st->bc1;
  const float bc2_sqrt = st->bc2_sqrt;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const float gi = g[i] * scale;
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] = p[i] - step_size * (mi / denom);
  }
}

// The whole optimizer tail of the fast training step in one launch.  Every block derives the bias corrections of
// step + 1 from the counter it reads (double arithmetic, like the Python side of torch.optim.Adam); the LAST block
// to finish publishes the new counter, clears the clip norm and moves the step's loss sum into place, so nothing
// a slower block still reads is overwritten.  Per element: clip scale, Adam update, the gradient cleared for the
// next step's accumulation, and -- for elements of a hidden weight matrix -- the bf16 copies (as stored and
// transposed, the latter times scale_t) that the next forward / dgrad chain will read (what prep_weights_kernel
// would have rebuilt from scratch at the start of the next step).
__global__ void adam_fused_kernel(const AdamFusedParams a) {
  __shared__ float s_bc1, s_bc2;
  __shared__ double s_p1, s_p2;
  const long step = a.st->step + 1;
  if (threadIdx.x == 0) {
    // beta^step as a running product (torch computes 1 - beta ** step in Python doubles: equal to ~1e-16 relative).
    // Only step 1 starts it: for beta <= 0.5 the product underflows to exactly 0.0 (beta = 0.5 after 1075 steps)
    // and must stay there -- the bias correction is then 1, not that of a restarted step 1.
    const double q1 = a.st->pow1, q2 = a.st->pow2;
    s_p1 = (step == 1 ? 1.0 : q1) * a.b1;
    s_p2 = (step == 1 ? 1.0 : q2) * a.b2;
    s_bc1 = (float)(1.0 - s_p1);
    s_bc2 = (float)sqrt(1.0 - s_p2);
  }
  float scale = a.grad_scale;
  if (a.max_norm > 0.f) {
    const float total = sqrtf(a.st->sumsq) * a.grad_scale;
    const float coef = a.max_norm / (total + 1e-6f);
    scale *= fminf(coef, 1.0f);
  }
  __syncthreads();
  const float b1 = (float)a.b1, b2 = (float)a.b2;
  const float step_size = a.lr / s_bc1;
  const float bc2_sqrt = s_bc2;
  auto update = [&](long i, float gi, float mi, float vi, float pi, float& mo, float& vo, float& po) {
    gi *= scale;
    mo = b1 * mi + (1.f - b1) * gi;
    vo = b2 * vi + (1.f - b2) * gi * gi;
    const float denom = sqrtf(vo) / bc2_sqrt + a.eps;
    po = pi - step_size * (mo / denom);
#pragma unroll 1
    for (int l = 0; l < a.n_w; ++l) {
      const long k = i - a.w_off[l];
      if (k >= 0 && k < long(H) * H) {
        const int r = int(k >> 8), c = int(k & 255);
        const bf16 h = __float2bfloat16_rn(po);
        if (a.k_f16) reinterpret_cast<__half*>(a.k_hi[l])[k] = __float2half_rn(po);
        else a.k_hi[l][k] = h;
        const float vt = po * a.scale_t;
        const bf16 ht = __float2bfloat16_rn(vt);
        a.t_hi[l][c * H + r] = ht;
        if (a.split) {
          a.k_lo[l][k] = __float2bfloat16_rn(po - __bfloat162float(h));
          a.t_lo[l][c * H + r] = __float2bfloat16_rn(vt - __bfloat162float(ht));
        }
      }
    }
  };
  // four elements per thread and trip (float4): the 198 k parameters of a 3 x 256 SIREN are one trip of one
  // DRAM round trip for the whole grid, instead of a dependent load -> store chain per element
  const long n4 = a.n / 4, stride = (long)gridDim.x * blockDim.x, t = blockIdx.x * (long)blockDim.x + threadIdx.x;
  float4* p4 = reinterpret_cast<float4*>(a.p);
  float4* g4 = reinterpret_cast<float4*>(a.g);
  float4* m4 = reinterpret_cast<float4*>(a.m);
  float4* v4 = reinterpret_cast<float4*>(a.v);
  float4* z4 = reinterpret_cast<float4*>(a.world > 1 ? a.zero_buf : a.g);
  for (long i = t; i < n4; i += stride) {
    float4 g;
    if (a.world > 1) {
      g = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int r = 0; r < a.world; ++r) {
        const float4 q = reinterpret_cast<const float4*>(a.peers[r])[i];
        g.x += q.x; g.y += q.y; g.z += q.z; g.w += q.w;
      }
    } else {
      g = g4[i];
    }
    const float4 m = m4[i], v = v4[i], pp = p4[i];
    float4 mo, vo, po;
    update(4 * i + 0, g.x, m.x, v.x, pp.x, mo.x, vo.x, po.x);
    update(4 * i + 1, g.y, m.y, v.y, pp.y, mo.y, vo.y, po.y);
    update(4 * i + 2, g.z, m.z, v.z, pp.z, mo.z, vo.z, po.z);
    update(4 * i + 3, g.w, m.w, v.w, pp.w, mo.w, vo.w, po.w);
    m4[i] = mo;
    v4[i] = vo;
    p4[i] = po;
    if (a.zero_grad && z4) z4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  float* zs = a.world > 1 ? a.zero_buf : a.g;
  for (long i = 4 * n4 + t; i < a.n; i += stride) {
    float gi = a.g[i];
    if (a.world > 1) {
      gi = 0.f;
      for (int r = 0; r < a.world; ++r) gi += a.peers[r][i];
    }
    float mo, vo, po;
    update(i, gi, a.m[i], a.v[i], a.p[i], mo, vo, po);
    a.m[i] = mo;
    a.v[i] = vo;
    a.p[i] = po;
    if (a.zero_grad && zs) zs[i] = 0.f;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    unsigned int* done = reinterpret_cast<unsigned int*>(&a.st->pad2);
    if (atomicAdd(done, 1u) == gridDim.x - 1) {
      a.st->step = step;
      a.st->bc1 = s_bc1;
      a.st->bc2_sqrt = s_bc2;
      a.st->pow1 = s_p1;
      a.st->pow2 = s_p2;
      a.st->sumsq = 0.f;
      *done = 0u;
      if (a.loss4) {
        a.loss4[0] = a.loss4[1];
        a.loss4[1] = 0.f;
      }
      __threadfence();
    }
  }
}

// clip_grad_norm_ in place (gradient accumulation: the reference clips the accumulated .grad after every
// micro-batch, training.py:93-97): g *= min(1, max_norm / (sqrt(sumsq) + 1e-6)); the last block clears sumsq
__global__ void clip_scale_kernel(float* __restrict__ g, long n, float max_norm, AdamState* st) {
  const float coef = fminf(max_norm / (sqrtf(st->sumsq) + 1e-6f), 1.0f);
  if (coef < 1.0f)
    for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) g[i] *= coef;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    unsigned int* done = reinterpret_cast<unsigned int*>(&st->pad2);
    if (atomicAdd(done, 1u) == gridDim.x - 1) {
      st->sumsq = 0.f;
      *done = 0u;
      __threadfence();
    }
  }
}

// -------------------------------------------------------------------------------------------
// optimizer tail of T stacked networks (TaskTail, simt.h): per-task clip norms, losses and Adam
// -------------------------------------------------------------------------------------------
// block-wide sum of v, valid in thread 0; may be called again at once (the barrier in front protects part[])
__device__ __forceinline__ float block_sum(float v, float* part) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = v;
  __syncthreads();
  float s = 0.f;
  if (threadIdx.x < 32) s = warp_sum(threadIdx.x < (blockDim.x >> 5) ? part[threadIdx.x] : 0.f);
  return s;
}

// segment of flat element i (the segments ascend and tile the buffer), and the task that owns i inside segment s
__device__ __forceinline__ int task_seg(const TaskTail& tt, long i) {
  int s = 0;
  while (s + 1 < tt.n_seg && i >= tt.seg_off[s + 1]) ++s;
  return s;
}
__device__ __forceinline__ int task_of(const TaskTail& tt, int s, long i) {
  return int(unsigned(i - tt.seg_off[s]) / unsigned(tt.seg_per[s]));
}

// The per-task sums as work items of TASK_ITEM floats of one task: its gradient (all segments as one index range,
// grads only) and its loss rows (y given).  One block reduction and one atomic per item.
constexpr int TASK_ITEM = 4096;
__device__ void task_reduce(const float* __restrict__ g, const TaskTail& tt, bool grads, float* part) {
  const int P = tt.seg_cum[tt.n_seg];
  const int gs = grads ? (P + TASK_ITEM - 1) / TASK_ITEM : 0;
  const int ls = tt.y ? int((tt.rows + TASK_ITEM - 1) / TASK_ITEM) : 0;
  const long g_items = long(tt.tasks) * gs, items = long(tt.tasks) * (gs + ls);
  for (long it = blockIdx.x; it < items; it += gridDim.x) {
    float acc = 0.f;
    if (it < g_items) {
      const int t = int(it / gs), a = int(it - long(t) * gs) * TASK_ITEM, e = min(a + TASK_ITEM, P);
      for (int s = 0; s < tt.n_seg; ++s) {
        const int lo = max(a, tt.seg_cum[s]), hi = min(e, tt.seg_cum[s + 1]);
        const float* src = g + tt.seg_off[s] + long(t) * tt.seg_per[s] - tt.seg_cum[s];
        for (int j = lo + threadIdx.x; j < hi; j += blockDim.x) {
          const float v = src[j];
          acc = fmaf(v, v, acc);
        }
      }
      acc = block_sum(acc, part);
      if (threadIdx.x == 0) atomicAdd(&tt.sumsq[t], acc);
    } else {
      const long k = it - g_items;
      const int t = int(k / ls);
      const long a = (k - long(t) * ls) * TASK_ITEM, e = min(a + TASK_ITEM, tt.rows);
      const float* y = tt.y + long(t) * tt.rows;
      const float* gt = tt.gt + long(t) * tt.rows;
      for (long j = a + threadIdx.x; j < e; j += blockDim.x) {
        const float dlt = y[j] - gt[j];
        acc = fmaf(dlt, dlt, acc);
      }
      acc = block_sum(acc, part);
      if (threadIdx.x == 0) atomicAdd(&tt.loss[tt.tasks + t], acc * tt.weight);
    }
  }
}

// true in every thread of the block that finishes the launch last (completion count in AdamState::pad2, which
// that block resets): everything the other blocks wrote or added is visible to it
__device__ __forceinline__ bool last_block(AdamState* st) {
  __shared__ bool s_last;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    unsigned int* done = reinterpret_cast<unsigned int*>(&st->pad2);
    s_last = atomicAdd(done, 1u) == gridDim.x - 1;
    if (s_last) *done = 0u;
  }
  __syncthreads();
  return s_last;
}

// the end of the tail (last block of its last launch): norms cleared for the next step and, with publish, every
// task's running loss moved to its finished one (and loss4[1] -> loss4[0])
__device__ void task_finish(const TaskTail& tt) {
  for (int t = threadIdx.x; t < tt.tasks; t += blockDim.x) {
    tt.sumsq[t] = 0.f;
    if (tt.publish) tt.loss[t] = atomicExch(&tt.loss[tt.tasks + t], 0.f);
  }
  if (threadIdx.x == 0 && tt.publish && tt.loss4) {
    tt.loss4[0] = tt.loss4[1];
    tt.loss4[1] = 0.f;
  }
  __threadfence();
}

__device__ __forceinline__ void task_coefs(const TaskTail& tt, float* coef) {
  for (int t = threadIdx.x; t < tt.tasks; t += blockDim.x)
    coef[t] = tt.max_norm > 0.f ? fminf(tt.max_norm / (sqrtf(tt.sumsq[t]) + 1e-6f), 1.0f) : 1.0f;
}

__global__ void __launch_bounds__(256) task_norms_kernel(const float* __restrict__ g, const TaskTail tt, AdamState* st) {
  __shared__ float part[32];
  task_reduce(g, tt, tt.max_norm > 0.f, part);
  if (tt.publish && last_block(st)) task_finish(tt);
}

// clip_grad_norm_ of every task in place: g *= min(1, max_norm / (|g_task| + 1e-6))
__global__ void __launch_bounds__(256) task_clip_kernel(float* __restrict__ g, long n, const TaskTail tt, AdamState* st) {
  __shared__ float s_coef[MAX_TASKS];
  task_coefs(tt, s_coef);
  __syncthreads();
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const float c = s_coef[task_of(tt, task_seg(tt, i), i)];
    if (c < 1.0f) g[i] *= c;
  }
  if (last_block(st)) task_finish(tt);
}

// adam_fused_kernel for T stacked networks (one rank): the clip coefficient of an element is its task's, resolved per
// element (the outermost bias holds d_out floats per task, so one float4 can span two tasks); the fp16 / bf16 copies
// of every task's hidden weights are rewritten in place of prep_weights_kernel's; y / gt given, the loss pass runs
// behind the update.  The last block advances the step and ends the tail (task_finish).
__global__ void __launch_bounds__(256) adam_tasks_kernel(const AdamFusedParams a, const TaskTail tt) {
  __shared__ float s_bc1, s_bc2;
  __shared__ double s_p1, s_p2;
  __shared__ float s_coef[MAX_TASKS];
  __shared__ float part[32];
  const long step = a.st->step + 1;
  if (threadIdx.x == 0) {
    const double q1 = a.st->pow1, q2 = a.st->pow2;      // as adam_fused_kernel: only step 1 starts the product
    s_p1 = (step == 1 ? 1.0 : q1) * a.b1;
    s_p2 = (step == 1 ? 1.0 : q2) * a.b2;
    s_bc1 = (float)(1.0 - s_p1);
    s_bc2 = (float)sqrt(1.0 - s_p2);
  }
  task_coefs(tt, s_coef);
  __syncthreads();
  const float b1 = (float)a.b1, b2 = (float)a.b2;
  const float step_size = a.lr / s_bc1;
  const float bc2_sqrt = s_bc2;
  auto update = [&](long i, int s, float gi, float mi, float vi, float pi, float& mo, float& vo, float& po) {
    if (tt.max_norm > 0.f) gi *= s_coef[task_of(tt, s, i)];
    mo = b1 * mi + (1.f - b1) * gi;
    vo = b2 * vi + (1.f - b2) * gi * gi;
    const float denom = sqrtf(vo) / bc2_sqrt + a.eps;
    po = pi - step_size * (mo / denom);
    const int l = tt.seg_hidden[s];
    if (l >= 0) {
      const long k = i - tt.seg_off[s];                 // task * H * H + row * H + column
      const long base = k & ~long(H * H - 1);
      const int r = int(k >> 8) & (H - 1), c = int(k & (H - 1));
      const bf16 h = __float2bfloat16_rn(po);
      if (a.k_f16) reinterpret_cast<__half*>(a.k_hi[l])[k] = __float2half_rn(po);
      else a.k_hi[l][k] = h;
      const float vt = po * a.scale_t;
      const bf16 ht = __float2bfloat16_rn(vt);
      a.t_hi[l][base + c * H + r] = ht;
      if (a.split) {
        a.k_lo[l][k] = __float2bfloat16_rn(po - __bfloat162float(h));
        a.t_lo[l][base + c * H + r] = __float2bfloat16_rn(vt - __bfloat162float(ht));
      }
    }
  };
  const long n4 = a.n / 4, stride = (long)gridDim.x * blockDim.x, t0 = blockIdx.x * (long)blockDim.x + threadIdx.x;
  float4* p4 = reinterpret_cast<float4*>(a.p);
  float4* g4 = reinterpret_cast<float4*>(a.g);
  float4* m4 = reinterpret_cast<float4*>(a.m);
  float4* v4 = reinterpret_cast<float4*>(a.v);
  for (long i = t0; i < n4; i += stride) {
    const long e = 4 * i;
    int s = task_seg(tt, e);
    auto next = [&](long j) {
      if (s + 1 < tt.n_seg && j >= tt.seg_off[s + 1]) ++s;      // every segment holds at least one float
    };
    const float4 g = g4[i], m = m4[i], v = v4[i], pp = p4[i];
    float4 mo, vo, po;
    update(e, s, g.x, m.x, v.x, pp.x, mo.x, vo.x, po.x);
    next(e + 1);
    update(e + 1, s, g.y, m.y, v.y, pp.y, mo.y, vo.y, po.y);
    next(e + 2);
    update(e + 2, s, g.z, m.z, v.z, pp.z, mo.z, vo.z, po.z);
    next(e + 3);
    update(e + 3, s, g.w, m.w, v.w, pp.w, mo.w, vo.w, po.w);
    m4[i] = mo;
    v4[i] = vo;
    p4[i] = po;
    if (a.zero_grad) g4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  for (long i = 4 * n4 + t0; i < a.n; i += stride) {
    float mo, vo, po;
    update(i, task_seg(tt, i), a.g[i], a.m[i], a.v[i], a.p[i], mo, vo, po);
    a.m[i] = mo;
    a.v[i] = vo;
    a.p[i] = po;
    if (a.zero_grad) a.g[i] = 0.f;
  }
  if (tt.y) task_reduce(nullptr, tt, false, part);
  if (last_block(a.st)) {
    if (threadIdx.x == 0) {
      a.st->step = step;
      a.st->bc1 = s_bc1;
      a.st->bc2_sqrt = s_bc2;
      a.st->pow1 = s_p1;
      a.st->pow2 = s_p2;
    }
    task_finish(tt);
  }
}

// loss4[0] = loss4[1]; loss4[1] = 0  (a micro-batch without optimizer step: adam_step does this otherwise)
__global__ void loss_roll_kernel(float* loss4) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    loss4[0] = loss4[1];
    loss4[1] = 0.f;
  }
}

// gy = 2 w (y - gt); loss += w sum (y - gt)^2
__global__ void mse_grad_kernel(const float* __restrict__ y, const float* __restrict__ gt, float* __restrict__ gy,
                                long n, float weight, float* __restrict__ loss) {
  float acc = 0.f;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const float dlt = y[i] - gt[i];
    gy[i] = 2.f * weight * dlt;
    acc = fmaf(dlt, dlt, acc);
  }
  acc = warp_sum(acc);
  __shared__ float part[32];
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? part[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0 && loss) atomicAdd(loss, v * weight);
  }
}

// k-space data consistency for the paths whose y is not completed inside a fused kernel (data_consistency.py:7-20):
//   blend: y[t][r][c] <- (1 - m pull) y + m pull k0   (in place);   grad: out = gy (1 - m pull)
__global__ void dc_blend_kernel(float* __restrict__ y, DcSpec dc, int tasks, int n, int o) {
  const long total = long(tasks) * n * o;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int c = int(i % o);
    const long tr = i / o;
    const size_t j = dc_index(dc.cf, int(tr / n), int(tr % n), c, n, o);
    const float a = dc.mask[j] * dc.pull;
    y[i] = fmaf(a, dc.k0[j], (1.f - a) * y[i]);      // a sampled entry (a = 1) is k0 to the bit
  }
}
__global__ void dc_grad_kernel(const float* __restrict__ gy, float* __restrict__ out, DcSpec dc, int tasks, int n, int o) {
  const long total = long(tasks) * n * o;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int c = int(i % o);
    const long tr = i / o;
    const size_t j = dc_index(dc.cf, int(tr / n), int(tr % n), c, n, o);
    out[i] = gy[i] * (1.f - dc.mask[j] * dc.pull);
  }
}

// Two-shot all-reduce of a flat fp32 buffer over peer memory in ONE kernel: this rank owns slice `rank` of the
// buffer; it sums that slice over every rank's copy (loads over NVLink, rank order: one total per element, so all
// replicas receive the same bits) and stores the total into slice `rank` of EVERY rank's copy (stores over NVLink).
// The caller orders it across ranks: every rank's buffer complete before the launch, every rank's launch complete
// before anyone reads the result (two symmetric-memory barriers).
__global__ void __launch_bounds__(256) peer_allreduce_kernel(float* const* __restrict__ peers, int world, long b4, long e4,
                                                             float scale) {
  float4* bufs[16];
#pragma unroll
  for (int r = 0; r < 16; ++r) bufs[r] = r < world ? reinterpret_cast<float4*>(peers[r]) : nullptr;
  for (long i = b4 + blockIdx.x * (long)blockDim.x + threadIdx.x; i < e4; i += (long)gridDim.x * blockDim.x) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int r = 0; r < 16; ++r)
      if (r < world) {
        const float4 q = bufs[r][i];
        v.x += q.x; v.y += q.y; v.z += q.z; v.w += q.w;
      }
    v.x *= scale; v.y *= scale; v.z *= scale; v.w *= scale;
#pragma unroll
    for (int r = 0; r < 16; ++r)
      if (r < world) bufs[r][i] = v;
  }
}

// The same all-reduce through the NVSwitch MULTICAST mapping of the buffer (NVLS): one multimem.ld_reduce returns an
// element summed over every rank's copy -- the switch pulls the operands and adds them in fp32 -- and one multimem.st
// broadcasts the total to every copy, so a rank moves its slice once in each direction instead of world - 1 times.
__global__ void __launch_bounds__(256) peer_allreduce_mc_kernel(float* __restrict__ mc, long b4, long e4, float scale) {
  float4* m4 = reinterpret_cast<float4*>(mc);
  constexpr int U = 4;      // reductions in flight per thread (a multimem round trip crosses the switch twice)
  const long stride = (long)gridDim.x * blockDim.x;
  for (long i0 = b4 + blockIdx.x * (long)blockDim.x + threadIdx.x; i0 < e4; i0 += U * stride) {
    float4 v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long i = i0 + u * stride;
      if (i < e4)
        asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
                     : "=f"(v[u].x), "=f"(v[u].y), "=f"(v[u].z), "=f"(v[u].w) : "l"(m4 + i) : "memory");
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long i = i0 + u * stride;
      if (i < e4)
        asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};"
                     :: "l"(m4 + i), "f"(v[u].x * scale), "f"(v[u].y * scale), "f"(v[u].z * scale), "f"(v[u].w * scale) : "memory");
    }
  }
  __threadfence_system();
}

// block-wide sum of ``acc`` added to *loss (one atomic per block)
__device__ __forceinline__ void block_add(float acc, float scale, float* loss) {
  acc = warp_sum(acc);
  __shared__ float part[32];
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? part[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0 && loss) atomicAdd(loss, v * scale);
  }
}

// loss_functions.laplace_mse (loss_functions.py:350-355) on the second-order jets of a scalar output and its
// gradient: lap = sum_k D[n, k]; loss = mean((lap - gt)^2); gD[n, k] = 2 (lap - gt) / N for every k
__global__ void laplace_mse_grad_kernel(const float* __restrict__ D, const float* __restrict__ gt, float* __restrict__ gD,
                                        long n, int d, float weight, float* __restrict__ loss) {
  float acc = 0.f;
  const float inv = weight / float(n);
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    float lap = 0.f;
    for (int k = 0; k < d; ++k) lap += D[i * d + k];
    const float dlt = lap - gt[i];
    acc = fmaf(dlt, dlt, acc);
    const float g = 2.f * dlt * inv;
    for (int k = 0; k < d; ++k) gD[i * d + k] = g;
  }
  block_add(acc, inv, loss);
}

// loss_functions.sdf (loss_functions.py:460-484; summed as training.py:68-76 does, each term's .mean() over the N
// points) on the value y and the first-order jets J = dy/dx of a scalar output in 3-D, and its gradients gy, gJ:
//   on-surface points (sdf != -1):   3e3 |y|  +  1e2 (1 - cos(J, normal))
//   off-surface points:              1e2 exp(-1e2 |y|)
//   every point:                     5e1 | |J| - 1 |
__device__ __forceinline__ float sgnf(float v) { return v > 0.f ? 1.f : (v < 0.f ? -1.f : 0.f); }
__global__ void sdf_grad_kernel(const float* __restrict__ y, const float* __restrict__ J, const float* __restrict__ sdf,
                                const float* __restrict__ normals, float* __restrict__ gy, float* __restrict__ gJ,
                                long n, float weight, float* __restrict__ loss) {
  float acc = 0.f;
  const float inv = weight / float(n);
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const float pred = y[i];
    const float g0 = J[3 * i], g1 = J[3 * i + 1], g2 = J[3 * i + 2];
    const bool on = sdf[i] != -1.f;
    const float gn = sqrtf(g0 * g0 + g1 * g1 + g2 * g2);
    float dy, d0 = 0.f, d1 = 0.f, d2 = 0.f;
    if (on) {
      acc += 3e3f * fabsf(pred);
      dy = 3e3f * sgnf(pred);
      const float n0 = normals[3 * i], n1 = normals[3 * i + 1], n2 = normals[3 * i + 2];
      const float nn = sqrtf(n0 * n0 + n1 * n1 + n2 * n2);
      const float gc = fmaxf(gn, 1e-8f), nc = fmaxf(nn, 1e-8f);      // F.cosine_similarity clamps each norm
      const float dot = g0 * n0 + g1 * n1 + g2 * n2;
      acc += 1e2f * (1.f - dot / (gc * nc));
      // d cos / d g = n / (|g| |n|) - (g.n) g / (|g|^3 |n|)   (|g| above the clamp)
      const float a = -1e2f / (gc * nc);
      const float b = gn > 1e-8f ? 1e2f * dot / (gn * gn * gc * nc) : 0.f;
      d0 = fmaf(a, n0, b * g0); d1 = fmaf(a, n1, b * g1); d2 = fmaf(a, n2, b * g2);
    } else {
      const float e = __expf(-1e2f * fabsf(pred));
      acc += 1e2f * e;
      dy = -1e4f * sgnf(pred) * e;
    }
    acc += 5e1f * fabsf(gn - 1.f);
    if (gn > 0.f) {
      const float c = 5e1f * sgnf(gn - 1.f) / gn;
      d0 = fmaf(c, g0, d0); d1 = fmaf(c, g1, d1); d2 = fmaf(c, g2, d2);
    }
    gy[i] = dy * inv;
    gJ[3 * i] = d0 * inv; gJ[3 * i + 1] = d1 * inv; gJ[3 * i + 2] = d2 * inv;
  }
  block_add(acc, inv, loss);
}

// fp32 rows [R,256] -> bf16 (hi, lo) planes (debug entry points)
__global__ void to_planes_kernel(const float* __restrict__ src, bf16* __restrict__ hi, bf16* __restrict__ lo,
                                 long n, int split) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const float v = src[i];
    const bf16 h = __float2bfloat16_rn(v);
    hi[i] = h;
    if (split) lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
  }
}

}  // namespace

cudaError_t launch_prep_weights(const PrepParams& p, cudaStream_t stream) {
  dim3 grid(H / 32, H / 32, p.tasks * p.n_layers), block(32, 8);
  prep_weights_kernel<<<grid, block, 0, stream>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_prep_first(const float* W0, bf16* w0k, int tasks, int d, cudaStream_t stream) {
  prep_first_kernel<<<tasks * H / 4, 256, 0, stream>>>(W0, w0k, d);
  return cudaGetLastError();
}

cudaError_t launch_sumsq(const float* g, long n, float* out, int num_sms, cudaStream_t stream) {
  long blocks = (n + 1023) / 1024;
  if (blocks > num_sms * 4) blocks = num_sms * 4;
  if (blocks < 1) blocks = 1;
  sumsq_kernel<<<(int)blocks, 256, 0, stream>>>(g, n, out);
  return cudaGetLastError();
}

cudaError_t launch_sumsq_peers(const float* const* peers, int world, long n, float* out, int num_sms, cudaStream_t stream) {
  long blocks = (n + 1023) / 1024;
  if (blocks > num_sms * 4) blocks = num_sms * 4;
  if (blocks < 1) blocks = 1;
  sumsq_peers_kernel<<<(int)blocks, 256, 0, stream>>>(peers, world, n, out);
  return cudaGetLastError();
}

cudaError_t launch_adam(float* p, const float* g, float* m, float* v, long n, float lr, double b1, double b2,
                        float eps, float max_norm, float grad_scale, AdamState* st, int num_sms,
                        cudaStream_t stream) {
  adam_tick_kernel<<<1, 32, 0, stream>>>(st, b1, b2);
  long blocks = (n + 255) / 256;
  if (blocks > num_sms * 8) blocks = num_sms * 8;
  if (blocks < 1) blocks = 1;
  adam_kernel<<<(int)blocks, 256, 0, stream>>>(p, g, m, v, n, lr, (float)b1, (float)b2, eps, max_norm,
                                                grad_scale, st);
  return cudaGetLastError();
}

cudaError_t launch_clip_grad(float* g, long n, float max_norm, AdamState* st, int num_sms, cudaStream_t stream) {
  cudaError_t e = launch_sumsq(g, n, &st->sumsq, num_sms, stream);
  if (e != cudaSuccess) return e;
  long blocks = (n + 255) / 256;
  if (blocks > num_sms * 8) blocks = num_sms * 8;
  if (blocks < 1) blocks = 1;
  clip_scale_kernel<<<(int)blocks, 256, 0, stream>>>(g, n, max_norm, st);
  return cudaGetLastError();
}

cudaError_t launch_loss_roll(float* loss4, cudaStream_t stream) {
  loss_roll_kernel<<<1, 32, 0, stream>>>(loss4);
  return cudaGetLastError();
}

cudaError_t launch_dc_blend(float* y, const DcSpec& dc, int tasks, int n, int o, int num_sms, cudaStream_t stream) {
  long blocks = (long(tasks) * n * o + 255) / 256;
  if (blocks > num_sms * 8) blocks = num_sms * 8;
  if (blocks < 1) blocks = 1;
  dc_blend_kernel<<<(int)blocks, 256, 0, stream>>>(y, dc, tasks, n, o);
  return cudaGetLastError();
}

cudaError_t launch_dc_grad(const float* gy, float* out, const DcSpec& dc, int tasks, int n, int o, int num_sms,
                           cudaStream_t stream) {
  long blocks = (long(tasks) * n * o + 255) / 256;
  if (blocks > num_sms * 8) blocks = num_sms * 8;
  if (blocks < 1) blocks = 1;
  dc_grad_kernel<<<(int)blocks, 256, 0, stream>>>(gy, out, dc, tasks, n, o);
  return cudaGetLastError();
}

cudaError_t launch_peer_allreduce(float* const* peers, int world, int rank, long n4, float scale, int num_sms,
                                  cudaStream_t stream) {
  const long per = (n4 + world - 1) / world;
  const long b4 = per * rank, e4 = b4 + per < n4 ? b4 + per : n4;
  if (b4 >= e4) return cudaSuccess;
  long blocks = (e4 - b4 + 255) / 256;
  if (blocks > num_sms * 4) blocks = num_sms * 4;
  peer_allreduce_kernel<<<(int)blocks, 256, 0, stream>>>(peers, world, b4, e4, scale);
  return cudaGetLastError();
}

cudaError_t launch_peer_allreduce_mc(float* mc, int world, int rank, long n4, float scale, int num_sms, cudaStream_t stream) {
  const long per = (n4 + world - 1) / world;
  const long b4 = per * rank, e4 = b4 + per < n4 ? b4 + per : n4;
  if (b4 >= e4) return cudaSuccess;
  long blocks = (e4 - b4 + 4 * 256 - 1) / (4 * 256);
  if (blocks > num_sms * 8) blocks = num_sms * 8;
  if (blocks < 1) blocks = 1;
  peer_allreduce_mc_kernel<<<(int)blocks, 256, 0, stream>>>(mc, b4, e4, scale);
  return cudaGetLastError();
}

cudaError_t launch_laplace_mse_grad(const float* D, const float* gt, float* gD, long n, int d, float weight, float* loss,
                                    int num_sms, cudaStream_t stream) {
  long blocks = (n + 255) / 256;
  if (blocks > num_sms * 8) blocks = num_sms * 8;
  if (blocks < 1) blocks = 1;
  laplace_mse_grad_kernel<<<(int)blocks, 256, 0, stream>>>(D, gt, gD, n, d, weight, loss);
  return cudaGetLastError();
}

cudaError_t launch_sdf_grad(const float* y, const float* J, const float* sdf, const float* normals, float* gy, float* gJ,
                            long n, float weight, float* loss, int num_sms, cudaStream_t stream) {
  long blocks = (n + 255) / 256;
  if (blocks > num_sms * 8) blocks = num_sms * 8;
  if (blocks < 1) blocks = 1;
  sdf_grad_kernel<<<(int)blocks, 256, 0, stream>>>(y, J, sdf, normals, gy, gJ, n, weight, loss);
  return cudaGetLastError();
}

cudaError_t launch_adam_fused(const AdamFusedParams& a, int num_sms, cudaStream_t stream) {
  // two blocks per SM at most: every block pays a fixed prologue (bias corrections in double) and epilogue
  // (fence + completion count), which ~800 one-element-per-thread blocks would pay five waves deep
  long blocks = (a.n + 255) / 256;
  if (blocks > num_sms * 2) blocks = num_sms * 2;
  if (blocks < 1) blocks = 1;
  adam_fused_kernel<<<(int)blocks, 256, 0, stream>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_task_norms(const float* g, const TaskTail& tt, AdamState* st, int num_sms, cudaStream_t stream) {
  const long gs = tt.max_norm > 0.f ? (tt.seg_cum[tt.n_seg] + TASK_ITEM - 1) / TASK_ITEM : 0;
  const long ls = tt.y ? (tt.rows + TASK_ITEM - 1) / TASK_ITEM : 0;
  long blocks = long(tt.tasks) * (gs + ls);
  if (blocks > num_sms * 4) blocks = num_sms * 4;
  if (blocks < 1) blocks = 1;
  task_norms_kernel<<<(int)blocks, 256, 0, stream>>>(g, tt, st);
  return cudaGetLastError();
}

cudaError_t launch_task_clip(float* g, long n, const TaskTail& tt, AdamState* st, int num_sms, cudaStream_t stream) {
  long blocks = (n + 255) / 256;
  if (blocks > num_sms * 8) blocks = num_sms * 8;
  if (blocks < 1) blocks = 1;
  task_clip_kernel<<<(int)blocks, 256, 0, stream>>>(g, n, tt, st);
  return cudaGetLastError();
}

cudaError_t launch_adam_tasks(const AdamFusedParams& a, const TaskTail& tt, int num_sms, cudaStream_t stream) {
  long blocks = (a.n + 255) / 256;      // as launch_adam_fused: at most two blocks per SM
  if (blocks > num_sms * 2) blocks = num_sms * 2;
  if (blocks < 1) blocks = 1;
  adam_tasks_kernel<<<(int)blocks, 256, 0, stream>>>(a, tt);
  return cudaGetLastError();
}

cudaError_t launch_mse_grad(const float* y, const float* gt, float* gy, long n, float weight, float* loss,
                            int num_sms, cudaStream_t stream) {
  long blocks = (n + 1023) / 1024;
  if (blocks > num_sms * 4) blocks = num_sms * 4;
  if (blocks < 1) blocks = 1;
  mse_grad_kernel<<<(int)blocks, 256, 0, stream>>>(y, gt, gy, n, weight, loss);
  return cudaGetLastError();
}

// clear up to 20 fp32 buffers in ONE launch (the parameter gradients of a backward call: ten memsets otherwise)
struct ZeroMany {
  float* p[20];
  long n[20];
};
__global__ void zero_many_kernel(const ZeroMany z) {
  float* p = z.p[blockIdx.y];
  const long n = z.n[blockIdx.y];
  const long stride = long(gridDim.x) * blockDim.x, t = long(blockIdx.x) * blockDim.x + threadIdx.x;
  if ((reinterpret_cast<uintptr_t>(p) & 15) == 0) {
    float4* p4 = reinterpret_cast<float4*>(p);
    for (long i = t; i < n / 4; i += stride) p4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (long i = (n / 4) * 4 + t; i < n; i += stride) p[i] = 0.f;
  } else {
    for (long i = t; i < n; i += stride) p[i] = 0.f;
  }
}

cudaError_t launch_zero_many(float* const* ptrs, const long* counts, int cnt, int num_sms, cudaStream_t stream) {
  if (cnt < 1 || cnt > 20) return cudaErrorInvalidValue;
  ZeroMany z;
  long mx = 0;
  for (int i = 0; i < cnt; ++i) {
    z.p[i] = ptrs[i];
    z.n[i] = counts[i];
    if (counts[i] > mx) mx = counts[i];
  }
  long bx = (mx / 4 + 255) / 256;
  if (bx > 4L * num_sms) bx = 4L * num_sms;
  if (bx < 1) bx = 1;
  zero_many_kernel<<<dim3((unsigned)bx, (unsigned)cnt), 256, 0, stream>>>(z);
  return cudaGetLastError();
}

// n floats from device memory to MAPPED pinned host memory: posted stores from one warp, no copy engine
__global__ void publish_kernel(const float* __restrict__ src, volatile float* dst, int n) {
  for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
  __threadfence_system();
}

cudaError_t launch_publish(const float* src, float* dst_host, int n, cudaStream_t stream) {
  publish_kernel<<<1, 32, 0, stream>>>(src, dst_host, n);
  return cudaGetLastError();
}

cudaError_t launch_to_planes(const float* src, bf16* hi, bf16* lo, long n, bool split, cudaStream_t stream) {
  to_planes_kernel<<<1024, 256, 0, stream>>>(src, hi, lo, n, split ? 1 : 0);
  return cudaGetLastError();
}

}  // namespace siren
