"""Fused (clip_grad_norm_ +) Adam over one flat fp32 buffer.

Mirrors ``torch.optim.Adam(lr=lr, params=model.parameters())`` as constructed at
training.py:23 (betas (0.9, 0.999), eps 1e-8, no weight decay, no amsgrad) and the optional
``torch.nn.utils.clip_grad_norm_`` of training.py:93-97, in two kernel launches instead of a
foreach pass over ten small tensors.
"""
import torch

from . import _lib


def flatten_parameters(params, grad=None):
    """Re-home ``params`` as views of one flat buffer; returns (flat_param, flat_grad).  ``grad``: a preallocated
    (zeroed) flat gradient buffer to use, e.g. one half of a symmetric-memory allocation peers can read."""
    params = list(params)
    n = sum(p.numel() for p in params)
    dev, dt = params[0].device, params[0].dtype
    flat = torch.empty(n, device=dev, dtype=dt)
    if grad is None:
        grad = torch.zeros(n, device=dev, dtype=dt)
    off = 0
    with torch.no_grad():
        for p in params:
            k = p.numel()
            flat[off:off + k].copy_(p.reshape(-1))
            p.data = flat[off:off + k].view_as(p)
            p.grad = grad[off:off + k].view_as(p)
            off += k
    return flat, grad


def stacked_segments(shapes, tasks):
    """Layout of ``tasks`` copies of every parameter in one flat buffer: parameter j is one [tasks, *shapes[j]] block,
    the blocks one after the other.  Returns the segment table [(offset, floats per task)] and the total length --
    the table the per-task optimizer kernels derive from the parameters' addresses (siren_b200_adam_step_tasks)."""
    segs, off = [], 0
    for shape in shapes:
        k = 1
        for s in shape:
            k *= int(s)
        segs.append((off, k))
        off += tasks * k
    return segs, off


def flatten_parameters_stacked(param_lists):
    """Re-home the parameters of T models of one architecture (``param_lists[t]``: model t's parameters, in the same
    order for every model) as views of one flat buffer laid out by ``stacked_segments``: parameter j of model t becomes
    task slice t of the stacked [T, *shape] tensor j, and its ``.grad`` the same slice of the flat gradient.
    Returns (flat_param, flat_grad, stacked params, stacked grads)."""
    param_lists = [list(ps) for ps in param_lists]
    T = len(param_lists)
    shapes = [tuple(p.shape) for p in param_lists[0]]
    for ps in param_lists[1:]:
        if [tuple(p.shape) for p in ps] != shapes:
            raise ValueError("the models' parameters differ in shape")
    segs, n = stacked_segments(shapes, T)
    p0 = param_lists[0][0]
    flat = torch.empty(n, device=p0.device, dtype=p0.dtype)
    grad = torch.zeros(n, device=p0.device, dtype=p0.dtype)
    stacked, stacked_grad = [], []
    with torch.no_grad():
        for j, ((off, k), shape) in enumerate(zip(segs, shapes)):
            w = flat[off:off + T * k].view((T,) + shape)
            g = grad[off:off + T * k].view((T,) + shape)
            for t in range(T):
                p = param_lists[t][j]
                w[t].copy_(p)
                p.data = w[t]
                p.grad = g[t]
            stacked.append(w)
            stacked_grad.append(g)
    return flat, grad, stacked, stacked_grad


class FusedAdam:
    """Adam on a flat buffer.  ``step()`` consumes ``flat_grad`` (optionally clipping its global
    L2 norm to ``max_grad_norm`` and scaling by ``grad_scale`` first)."""

    def __init__(self, flat_param, flat_grad, lr=1e-4, betas=(0.9, 0.999), eps=1e-8, max_grad_norm=0.0):
        if not flat_param.is_cuda:
            raise _lib.NativeError("FusedAdam needs CUDA tensors")
        self.p, self.g = flat_param, flat_grad
        self.m = torch.zeros_like(flat_param)
        self.v = torch.zeros_like(flat_param)
        self.state = torch.zeros(64, device=flat_param.device, dtype=torch.uint8)   # AdamState (csrc/simt.h)
        self.lr, self.betas, self.eps = lr, betas, eps
        self.max_grad_norm = float(max_grad_norm)
        self.steps = 0
        self.task_sumsq = None    # [T] squared gradient norm per task between the launches of a step (step_tasks)

    def step(self, grad_scale=1.0):
        lib = _lib.load()
        self.steps += 1          # host mirror; the authoritative counter lives in self.state
        stream = torch.cuda.current_stream(self.p.device).cuda_stream
        with torch.cuda.device(self.p.device):
            rc = lib.siren_b200_adam(_lib.dptr(self.p), _lib.dptr(self.g), _lib.dptr(self.m), _lib.dptr(self.v),
                                     self.p.numel(), self.lr, self.betas[0], self.betas[1], self.eps,
                                     self.max_grad_norm, float(grad_scale), _lib.dptr(self.state), stream)
        _lib.check(rc, "siren_b200_adam")

    def step_fused(self, grad_scale=1.0, zero_grad=True, loss4=None, desc=None, w_ptrs=None, ws=None, clip=True):
        """The same update in ONE launch (siren_b200_adam_step): step tick, clip, Adam, the consumed gradient cleared,
        ``loss4[1] -> loss4[0]``, and (``desc`` / ``w_ptrs`` / ``ws`` given) the workspace's bf16 weight copies
        refreshed from the updated parameters -- the optimizer tail of SirenTrainer's captured step."""
        lib = _lib.load()
        self.steps += 1
        stream = torch.cuda.current_stream(self.p.device).cuda_stream
        with torch.cuda.device(self.p.device):
            rc = lib.siren_b200_adam_step(_lib.dptr(self.p), _lib.dptr(self.g), _lib.dptr(self.m), _lib.dptr(self.v),
                                          self.p.numel(), self.lr, self.betas[0], self.betas[1], self.eps,
                                          self.max_grad_norm if clip else 0.0, float(grad_scale), _lib.dptr(self.state),
                                          1 if zero_grad else 0, _lib.dptr(loss4), desc, w_ptrs, _lib.dptr(ws), stream)
        _lib.check(rc, "siren_b200_adam_step")

    def step_peers(self, peers_dev, world, zero_buf, grad_scale=1.0, loss4=None, desc=None, w_ptrs=None, ws=None,
                   clip=True):
        """step_fused with the all-reduce fused in (siren_b200_adam_step_peers): the gradient is summed over the ranks'
        buffers read from peer memory; ``zero_buf`` (the buffer the next step accumulates into) is cleared."""
        lib = _lib.load()
        self.steps += 1
        stream = torch.cuda.current_stream(self.p.device).cuda_stream
        with torch.cuda.device(self.p.device):
            rc = lib.siren_b200_adam_step_peers(_lib.dptr(self.p), _lib.dptr(self.g), _lib.dptr(self.m), _lib.dptr(self.v),
                                                self.p.numel(), self.lr, self.betas[0], self.betas[1], self.eps,
                                                self.max_grad_norm if clip else 0.0, float(grad_scale),
                                                _lib.dptr(self.state), _lib.dptr(loss4), desc, w_ptrs, _lib.dptr(ws),
                                                _lib.dptr(peers_dev), int(world), _lib.dptr(zero_buf), stream)
        _lib.check(rc, "siren_b200_adam_step_peers")

    def step_tasks(self, desc, w_ptrs, b_ptrs, task_loss, y=None, gt=None, weight=0.0, loss4=None, ws=None, clip=True):
        """step_fused for ``desc.tasks`` networks stacked in the flat buffer (siren_b200_adam_step_tasks): each task is
        clipped by its own gradient norm and, ``y`` / ``gt`` given, gets its own loss in ``task_loss``."""
        lib = _lib.load()
        self.steps += 1
        P = _lib.dptr
        self._task_state(desc.tasks)
        stream = torch.cuda.current_stream(self.p.device).cuda_stream
        with torch.cuda.device(self.p.device):
            rc = lib.siren_b200_adam_step_tasks(desc, w_ptrs, b_ptrs, P(self.p), P(self.g), P(self.m), P(self.v),
                                                self.p.numel(), self.lr, self.betas[0], self.betas[1], self.eps,
                                                self.max_grad_norm if clip else 0.0, P(self.state), P(y), P(gt),
                                                float(weight), P(self.task_sumsq), P(task_loss), P(loss4), P(ws), stream)
        _lib.check(rc, "siren_b200_adam_step_tasks")

    def clip_tasks(self, desc, dw_ptrs, db_ptrs, task_loss, y=None, gt=None, weight=0.0, loss4=None, clip=True,
                   publish=True):
        """A micro-batch without optimizer step (siren_b200_clip_grad_tasks): its per-task losses and, with clipping,
        each task's accumulated gradient clipped in place by its own norm."""
        lib = _lib.load()
        P = _lib.dptr
        self._task_state(desc.tasks)
        stream = torch.cuda.current_stream(self.p.device).cuda_stream
        with torch.cuda.device(self.p.device):
            rc = lib.siren_b200_clip_grad_tasks(desc, dw_ptrs, db_ptrs, P(self.g), self.g.numel(),
                                                self.max_grad_norm if clip else 0.0, P(self.state), P(y), P(gt),
                                                float(weight), P(self.task_sumsq), P(task_loss), P(loss4),
                                                1 if publish else 0, stream)
        _lib.check(rc, "siren_b200_clip_grad_tasks")

    def _task_state(self, tasks):
        if self.task_sumsq is None or self.task_sumsq.numel() != tasks:
            self.task_sumsq = torch.zeros(tasks, device=self.p.device)

    def zero_grad(self):
        self.g.zero_()
