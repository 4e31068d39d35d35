"""Autograd boundary of the native SIREN path.

``siren_mlp(coords, weights, biases, w0, ...)`` evaluates the sine MLP of the reference
(modules.py:16-27 BatchLinear, modules.py:35-38 Sine, chained as in modules.py:68-85 with an
outermost linear layer) through the C ABI (include/siren_b200.h) and returns a tensor that
behaves under autograd like the reference's output:

* gradients w.r.t. the weights / biases (shared ``[out,in]`` or per-task ``[B,out,in]`` tensors,
  e.g. the output of meta_modules.HyperNetwork) come from the fused backward kernels;
* gradients w.r.t. the coordinates under ``torch.autograd.grad(..., create_graph=True)``, nested
  to second order (diff_operators.py:27-43), come from forward-mode jets the kernels propagate
  next to the activations (``coord_derivs=1|2``), attached to the graph by two tiny Functions
  (SURVEY.md section 8b).  Only the diagonal second derivatives d2y/dx_k^2 are represented,
  which is all gradient / divergence / laplace use; full Hessians need ``coord_derivs=0``, where
  any higher-order query transparently re-runs the composed PyTorch graph.
"""
import ctypes
import math
import threading
import warnings
from collections import OrderedDict

import torch

from . import _lib


# --------------------------------------------------------------------------------------------
# composed PyTorch path (reference semantics; used for CPU tensors, unsupported shapes and
# higher-order queries when no jets were requested)
# --------------------------------------------------------------------------------------------
def composed_mlp(coords, weights, biases, w0):
    h = coords
    last = len(weights) - 1
    for l, (W, b) in enumerate(zip(weights, biases)):
        h = h.matmul(W.transpose(-1, -2)) + b.unsqueeze(-2)
        if l != last:
            h = torch.sin(w0 * h)
    return h


def fourier_features(x, B):
    """features.py:31-41 (GaussianFourierFeatureTransform.forward): ``cat[sin, cos](2 pi x @ B)``."""
    x = x @ B.to(x.device)
    x = 2 * math.pi * x
    return torch.cat([torch.sin(x), torch.cos(x)], dim=-1)


# --------------------------------------------------------------------------------------------
# native kernels
# --------------------------------------------------------------------------------------------
def _wide_inputs_ok(precision, coord_derivs, coords_grad):
    """17..256 first-layer inputs are served by the bf16 and the fp32-parity value paths (check_desc in
    csrc/api.cu)."""
    if coord_derivs or coords_grad:
        return False
    return precision in ("fp32", "bf16")


def native_supported(coords, weights, biases, coord_derivs=0, fourier=None, precision=None, coords_grad=False):
    """True when the C ABI serves this call (see check_desc / check_fourier in csrc/api.cu).  ``fourier`` = the
    ``[raw, F]`` matrix of a Gaussian Fourier-feature prologue: ``coords`` are then the RAW coordinates."""
    if not coords.is_cuda or coords.dtype != torch.float32 or coords.dim() != 3:
        return False
    if fourier is not None:
        f_max = 128 if _wide_inputs_ok(precision, coord_derivs, coords_grad) else 8
        if (coord_derivs or fourier.dim() != 2 or fourier.dtype != torch.float32 or fourier.shape[0] != coords.shape[-1]
                or not 1 <= fourier.shape[0] <= 3 or not 3 <= fourier.shape[1] <= f_max
                or weights[0].shape[-1] != 2 * fourier.shape[1]):
            return False
        coords = coords.new_empty((coords.shape[0], coords.shape[1], 2 * fourier.shape[1]))      # shape checks below
    n_layers = len(weights)
    if n_layers < 3 or n_layers > 10:
        return False
    hid = weights[0].shape[-2]
    if hid != 256 or coords.shape[1] < 1 or coords.shape[0] < 1:
        return False
    per_task = weights[0].dim() == 3
    for l, (W, b) in enumerate(zip(weights, biases)):
        if b is None or W.dtype != torch.float32 or not W.is_cuda or W.dim() != (3 if per_task else 2):
            return False
        fin = coords.shape[-1] if l == 0 else hid
        fout = hid if l < n_layers - 1 else W.shape[-2]
        if tuple(W.shape[-2:]) != (fout, fin) or b.shape[-1] != fout or b.dim() != (2 if per_task else 1):
            return False
        if per_task and (W.shape[0] != coords.shape[0] or b.shape[0] != coords.shape[0]):
            return False
    if weights[-1].shape[-2] > 8 or coords.shape[-1] > 256:
        return False
    if coords.shape[-1] > 16 and not _wide_inputs_ok(precision, coord_derivs, coords_grad):
        return False
    if coord_derivs and coords.shape[-1] > 3:
        return False
    return True


# Workspaces are large (GBs for the MRI configs) and have the same size step after step.  Handing
# them back to torch's caching allocator lets smaller tensors split the block, after which the next
# step pays a cudaMalloc; a tiny per-(device, stream, size) free list avoids that.  Reuse is
# stream-ordered: a workspace only ever returns to the list of the stream it was used on.
_WS_CACHE = OrderedDict()      # (device, stream, nbytes) -> [tensors], least recently used first
_WS_CACHE_MAX = 2               # workspaces kept per key
_WS_CACHE_KEYS = 3              # distinct sizes kept; older ones go back to the allocator
_WS_LOCK = threading.Lock()     # nn.DataParallel replicas call from one thread per GPU; autograd backward threads release


def _ws_acquire(nbytes, dev, stream):
    key = (dev.index, stream, nbytes)
    with _WS_LOCK:
        lst = _WS_CACHE.get(key)
        if lst:
            _WS_CACHE.move_to_end(key)
            return lst.pop()
    return torch.empty(nbytes, dtype=torch.uint8, device=dev)


def _ws_release(ws, dev, stream):
    key = (dev.index, stream, ws.numel())
    with _WS_LOCK:
        lst = _WS_CACHE.setdefault(key, [])
        _WS_CACHE.move_to_end(key)
        if len(lst) < _WS_CACHE_MAX:
            lst.append(ws)
        while len(_WS_CACHE) > _WS_CACHE_KEYS:
            _WS_CACHE.popitem(last=False)


def clear_workspace_cache():
    with _WS_LOCK:
        _WS_CACHE.clear()


class _WsHolder:
    """Owns a workspace for the lifetime of the autograd node; hands it back to the free list
    when the graph is released (so ``retain_graph=True`` keeps the stash valid)."""

    def __init__(self, ws, dev, stream):
        self.ws, self.dev, self.stream = ws, dev, stream

    def __del__(self):
        try:
            if self.ws is not None:
                _ws_release(self.ws, self.dev, self.stream)
        except Exception:      # interpreter shutdown
            pass


def _make_desc(coords, weights, w0, precision, order):
    d = _lib.SirenDesc()
    d.d_in = coords.shape[-1]
    d.hidden = weights[0].shape[-2]
    d.n_hidden = len(weights) - 2
    d.d_out = weights[-1].shape[-2]
    d.w0 = float(w0)
    d.tasks = coords.shape[0]
    d.per_task = 1 if weights[0].dim() == 3 else 0
    d.n_coords = coords.shape[1]
    d.precision = _lib.PRECISIONS[precision]
    d.deriv_order = order
    return d


class _SirenKernelFn(torch.autograd.Function):
    """(coords, W0, b0, ..., WL, bL) -> y [, J [, D]] through libsiren_b200."""

    @staticmethod
    def forward(ctx, w0, precision, order, coords_grad, coords, *params):
        lib = _lib.load()
        coords_c = coords.detach().contiguous()
        ps = [p.detach().contiguous() for p in params]
        weights, biases = ps[0::2], ps[1::2]
        desc = _make_desc(coords_c, weights, w0, precision, order)
        nbytes = lib.siren_b200_workspace_bytes_ex(desc, 1 if coords_grad else 0)
        if nbytes == 0:
            _lib.check(1, "siren_b200_workspace_bytes")
        T, N, d = coords_c.shape
        o = desc.d_out
        dev = coords_c.device
        stream = torch.cuda.current_stream(dev).cuda_stream
        ws = _ws_acquire(nbytes, dev, stream)
        y = torch.empty((T, N, o), dtype=torch.float32, device=dev)
        J = torch.empty((T, N, o, d), dtype=torch.float32, device=dev) if order >= 1 else None
        D = torch.empty((T, N, o, d), dtype=torch.float32, device=dev) if order >= 2 else None
        infer = order == 0 and not any(ctx.needs_input_grad)      # e.g. under torch.no_grad(): no backward follows
        with torch.cuda.device(dev):
            if infer:
                rc = lib.siren_b200_forward_infer(desc, _lib.dptr(coords_c), _lib.ptr_array(weights),
                                                  _lib.ptr_array(biases), _lib.dptr(y), _lib.dptr(ws), stream)
            else:
                rc = lib.siren_b200_forward(desc, _lib.dptr(coords_c), _lib.ptr_array(weights),
                                            _lib.ptr_array(biases), _lib.dptr(y), _lib.dptr(J), _lib.dptr(D),
                                            _lib.dptr(ws), stream)
        _lib.check(rc, "siren_b200_forward")
        holder = _WsHolder(ws, dev, stream)       # released when this node (or this call, for inference) dies
        ctx.desc = desc
        ctx.ws_holder = holder
        ctx.coords_c = coords_c
        ctx.ps = ps
        ctx.w0 = w0
        ctx.coords_grad = coords_grad
        ctx.order = order
        # originals, for the composed re-evaluation when a higher-order graph is requested
        ctx.save_for_backward(coords, *params)
        ctx.set_materialize_grads(False)
        if order == 0:
            return y
        if order == 1:
            return y, J
        return y, J, D

    @staticmethod
    def backward(ctx, gy, gJ=None, gD=None):
        if torch.is_grad_enabled():
            return _SirenKernelFn._composed_backward(ctx, gy, gJ, gD)
        lib = _lib.load()
        desc = ctx.desc
        ps = ctx.ps
        weights, biases = ps[0::2], ps[1::2]
        dev = ctx.coords_c.device
        T, N, d = ctx.coords_c.shape
        if gy is None:
            gy = torch.zeros((T, N, desc.d_out), dtype=torch.float32, device=dev)
        gy = gy.contiguous()
        gJ = gJ.contiguous() if gJ is not None else None
        gD = gD.contiguous() if gD is not None else None
        dWs = [torch.empty_like(w) for w in weights]
        dbs = [torch.empty_like(b) for b in biases]
        gx = torch.empty_like(ctx.coords_c) if (ctx.coords_grad and ctx.needs_input_grad[4]) else None
        stream = torch.cuda.current_stream(dev).cuda_stream
        with torch.cuda.device(dev):
            rc = lib.siren_b200_backward(desc, _lib.dptr(ctx.coords_c), _lib.ptr_array(weights),
                                         _lib.ptr_array(biases), _lib.dptr(ctx.ws_holder.ws), _lib.dptr(gy), _lib.dptr(gJ),
                                         _lib.dptr(gD), _lib.ptr_array(dWs), _lib.ptr_array(dbs), _lib.dptr(gx), 0,
                                         stream)
        _lib.check(rc, "siren_b200_backward")
        grads = []
        for i in range(len(weights)):
            grads.append(dWs[i] if ctx.needs_input_grad[5 + 2 * i] else None)
            grads.append(dbs[i] if ctx.needs_input_grad[6 + 2 * i] else None)
        return (None, None, None, None, gx) + tuple(grads)

    @staticmethod
    def _composed_backward(ctx, gy, gJ, gD):
        """create_graph=True reached the kernel Function itself: answer with the composed
        PyTorch graph so that any higher-order query (including full Hessians) is exact."""
        if ctx.order != 0:
            raise RuntimeError(
                "siren_mri_b200: a differentiable backward through the jet outputs was requested "
                "(derivative order above coord_derivs=%d). Raise coord_derivs or use coord_derivs=0." % ctx.order)
        if not getattr(_SirenKernelFn, "_warned", False):
            warnings.warn("siren_mri_b200: coordinate derivatives requested with coord_derivs=0; using the "
                          "composed PyTorch path for this query. Set coord_derivs=1|2 for the fused jet kernels.")
            _SirenKernelFn._warned = True
        saved = ctx.saved_tensors
        coords, params = saved[0], saved[1:]
        with torch.enable_grad():
            y = composed_mlp(coords, params[0::2], params[1::2], ctx.w0)
            inputs = [t for t in (coords,) + tuple(params) if t.requires_grad]
            got = torch.autograd.grad(y, inputs, gy, create_graph=True, allow_unused=True)
        it = iter(got)
        out = [next(it) if t.requires_grad else None for t in (coords,) + tuple(params)]
        return (None, None, None, None) + tuple(out)


class _SirenFourierFn(torch.autograd.Function):
    """(raw coords, B, W0, b0, ..., WL, bL) -> y with the Gaussian Fourier features of the coordinates as the first
    layer's input, built inside the kernels (siren_b200_forward_ff / _backward_ff): the ``[B, N, 2F]`` tensor that
    features.py:31-41 returns is never written.  No gradient flows to the raw coordinates or to B (nothing in the
    reference's MRI loops asks for one)."""

    @staticmethod
    def forward(ctx, w0, precision, coords, B, *params):
        lib = _lib.load()
        coords_c = coords.detach().contiguous()
        B_c = B.detach().to(coords_c.device).contiguous()
        ps = [p.detach().contiguous() for p in params]
        weights, biases = ps[0::2], ps[1::2]
        T, N, raw = coords_c.shape
        F = B_c.shape[1]
        desc = _make_desc(coords_c, weights, w0, precision, 0)
        desc.d_in = 2 * F
        ff = _lib.SirenFourier()
        ff.B = _lib.dptr(B_c)
        ff.n_features = F
        ff.raw_dim = raw
        nbytes = lib.siren_b200_workspace_bytes_ex(desc, 0)
        if nbytes == 0:
            _lib.check(1, "siren_b200_workspace_bytes")
        dev = coords_c.device
        stream = torch.cuda.current_stream(dev).cuda_stream
        ws = _ws_acquire(nbytes, dev, stream)
        y = torch.empty((T, N, desc.d_out), dtype=torch.float32, device=dev)
        infer = not any(ctx.needs_input_grad)
        with torch.cuda.device(dev):
            rc = lib.siren_b200_forward_ff(desc, ff, _lib.dptr(coords_c), _lib.ptr_array(weights), _lib.ptr_array(biases),
                                           _lib.dptr(y), _lib.dptr(ws), 1 if infer else 0, stream)
        _lib.check(rc, "siren_b200_forward_ff")
        ctx.desc, ctx.ff, ctx.B_c = desc, ff, B_c
        ctx.ws_holder = _WsHolder(ws, dev, stream)
        ctx.coords_c, ctx.ps, ctx.w0 = coords_c, ps, w0
        ctx.save_for_backward(*params)
        ctx.set_materialize_grads(False)
        return y

    @staticmethod
    def backward(ctx, gy):
        weights, biases = ctx.ps[0::2], ctx.ps[1::2]
        dev = ctx.coords_c.device
        if torch.is_grad_enabled():      # create_graph=True: answer with the composed graph (exact to any order)
            params = ctx.saved_tensors
            with torch.enable_grad():
                y = composed_mlp(fourier_features(ctx.coords_c, ctx.B_c), params[0::2], params[1::2], ctx.w0)
                inputs = [t for t in params if t.requires_grad]
                got = iter(torch.autograd.grad(y, inputs, gy, create_graph=True, allow_unused=True))
            return (None, None, None, None) + tuple(next(got) if t.requires_grad else None for t in params)
        lib = _lib.load()
        if gy is None:
            gy = torch.zeros(ctx.coords_c.shape[:2] + (ctx.desc.d_out,), dtype=torch.float32, device=dev)
        gy = gy.contiguous()
        dWs = [torch.empty_like(w) for w in weights]
        dbs = [torch.empty_like(b) for b in biases]
        stream = torch.cuda.current_stream(dev).cuda_stream
        with torch.cuda.device(dev):
            rc = lib.siren_b200_backward_ff(ctx.desc, ctx.ff, _lib.dptr(ctx.coords_c), _lib.ptr_array(weights),
                                            _lib.ptr_array(biases), _lib.dptr(ctx.ws_holder.ws), _lib.dptr(gy),
                                            _lib.ptr_array(dWs), _lib.ptr_array(dbs), 0, stream)
        _lib.check(rc, "siren_b200_backward_ff")
        grads = []
        for i in range(len(weights)):
            grads.append(dWs[i] if ctx.needs_input_grad[4 + 2 * i] else None)
            grads.append(dbs[i] if ctx.needs_input_grad[5 + 2 * i] else None)
        return (None, None, None, None) + tuple(grads)


def data_consistency_blend(pred, k0, mask, noise_lvl=None):
    """data_consistency.py:7-20 as one blend (``k0`` / ``mask`` already in the prediction's ``[B, N, o]`` layout)."""
    a = mask if not noise_lvl else mask * (noise_lvl / (1.0 + noise_lvl))
    return (1.0 - a) * pred + a * k0      # a sampled entry of the noiseless blend is k0 to the bit, as in the reference


def _channels_last(t, o):
    """``[B, o, ...]`` (channel first, as the datasets deliver k-space) -> ``[B, N, o]`` (data_consistency.py:40-45)."""
    return t.reshape(t.shape[0], o, -1).transpose(1, 2)


class _SirenDCFn(torch.autograd.Function):
    """The general value-path call (siren_b200_forward_call / _backward_call):
    (coords, B | None, k0 | None, mask | None, ops | None, W0, b0, ..., WL, bL) -> y, with any of

    * ``B``: the first layer reads the Gaussian Fourier features of the raw coordinates, built on chip;
    * ``k0`` / ``mask``: the k-space data-consistency blend of data_consistency.py:7-20 applied where the kernels
      complete a row's output -- the datasets' channel-first ``[B, o, nx, ny]`` tensors as they are
      (``channels_first``) or ``[B, N, o]``;
    * ``ops = (wk16, wt16)``: the hidden weights as READY-MADE tensor-core operands (lists of fp16 / bf16 tensors
      written by the hypernetwork head, ``_HyperHeadFn``): the call converts no weights.

    k0 / mask / B / coords are data: no gradient flows to them."""

    @staticmethod
    def forward(ctx, w0, precision, noise_lvl, channels_first, coords, B, k0, mask, ops, *params):
        lib = _lib.load()
        coords_c = coords.detach().contiguous()
        B_c = None if B is None else B.detach().to(coords_c.device).contiguous()
        ps = [p.detach().contiguous() for p in params]
        weights, biases = ps[0::2], ps[1::2]
        T, N, _ = coords_c.shape
        desc = _make_desc(coords_c, weights, w0, precision, 0)
        call = _lib.SirenCall()
        keep = [B_c]
        if B_c is not None:
            ff = _lib.SirenFourier()
            ff.B, ff.n_features, ff.raw_dim = _lib.dptr(B_c), B_c.shape[1], coords_c.shape[-1]
            desc.d_in = 2 * B_c.shape[1]
            call.fourier = ctypes.pointer(ff)
            keep.append(ff)
        k0_c = mask_c = None
        if k0 is not None:
            k0_c = k0.detach().to(torch.float32).contiguous()
            mask_c = mask.detach().to(torch.float32).contiguous()
            if k0_c.numel() != T * N * desc.d_out or mask_c.numel() != k0_c.numel():
                raise ValueError("data consistency: k0 / mask hold %d / %d values, the output %d"
                                 % (k0_c.numel(), mask_c.numel(), T * N * desc.d_out))
            dc = _lib.SirenDC()
            dc.k0, dc.mask = _lib.dptr(k0_c), _lib.dptr(mask_c)
            dc.noise_lvl = float(noise_lvl or 0.0)
            dc.channels_first = 1 if channels_first else 0
            call.dc = ctypes.pointer(dc)
            keep += [dc, k0_c, mask_c]
        if ops is not None:
            wk, wt = _lib.ptr_array(ops[0]), _lib.ptr_array(ops[1])
            call.wk16 = ctypes.cast(wk, ctypes.POINTER(ctypes.c_void_p))
            call.wt16 = ctypes.cast(wt, ctypes.POINTER(ctypes.c_void_p))
            keep += [wk, wt, ops]
        nbytes = lib.siren_b200_workspace_bytes_ex(desc, 0)
        if nbytes == 0:
            _lib.check(1, "siren_b200_workspace_bytes")
        dev = coords_c.device
        stream = torch.cuda.current_stream(dev).cuda_stream
        ws = _ws_acquire(nbytes, dev, stream)
        y = torch.empty((T, N, desc.d_out), dtype=torch.float32, device=dev)
        infer = not any(ctx.needs_input_grad)
        with torch.cuda.device(dev):
            rc = lib.siren_b200_forward_call(desc, call, _lib.dptr(coords_c), _lib.ptr_array(weights),
                                             _lib.ptr_array(biases), _lib.dptr(y), _lib.dptr(ws), 1 if infer else 0, stream)
        _lib.check(rc, "siren_b200_forward_call")
        ctx.desc, ctx.call, ctx.keep = desc, call, keep
        ctx.dc_data = (B_c, k0_c, mask_c)
        ctx.noise_lvl, ctx.channels_first = noise_lvl, channels_first
        ctx.ws_holder = _WsHolder(ws, dev, stream)
        ctx.coords_c, ctx.ps, ctx.w0 = coords_c, ps, w0
        ctx.save_for_backward(*params)
        ctx.set_materialize_grads(False)
        return y

    @staticmethod
    def backward(ctx, gy):
        weights, biases = ctx.ps[0::2], ctx.ps[1::2]
        dev = ctx.coords_c.device
        B_c, k0_c, mask_c = ctx.dc_data
        NA = 9      # non-parameter arguments of forward
        if torch.is_grad_enabled():      # create_graph=True: answer with the composed graph (exact to any order)
            params = ctx.saved_tensors
            o = ctx.desc.d_out
            with torch.enable_grad():
                x = ctx.coords_c if B_c is None else fourier_features(ctx.coords_c, B_c)
                y = composed_mlp(x, params[0::2], params[1::2], ctx.w0)
                if k0_c is not None:
                    k0, mask = (k0_c, mask_c) if not ctx.channels_first else (_channels_last(k0_c, o), _channels_last(mask_c, o))
                    y = data_consistency_blend(y, k0.reshape(y.shape), mask.reshape(y.shape), ctx.noise_lvl)
                inputs = [t for t in params if t.requires_grad]
                got = iter(torch.autograd.grad(y, inputs, gy, create_graph=True, allow_unused=True))
            return (None,) * NA + tuple(next(got) if t.requires_grad else None for t in params)
        lib = _lib.load()
        if gy is None:
            gy = torch.zeros(ctx.coords_c.shape[:2] + (ctx.desc.d_out,), dtype=torch.float32, device=dev)
        gy = gy.contiguous()
        dWs = [torch.empty_like(w) for w in weights]
        dbs = [torch.empty_like(b) for b in biases]
        stream = torch.cuda.current_stream(dev).cuda_stream
        with torch.cuda.device(dev):
            rc = lib.siren_b200_backward_call(ctx.desc, ctx.call, _lib.dptr(ctx.coords_c), _lib.ptr_array(weights),
                                              _lib.ptr_array(biases), _lib.dptr(ctx.ws_holder.ws), _lib.dptr(gy),
                                              _lib.ptr_array(dWs), _lib.ptr_array(dbs), 0, stream)
        _lib.check(rc, "siren_b200_backward_call")
        grads = []
        for i in range(len(weights)):
            grads.append(dWs[i] if ctx.needs_input_grad[NA + 2 * i] else None)
            grads.append(dbs[i] if ctx.needs_input_grad[NA + 1 + 2 * i] else None)
        return (None,) * NA + tuple(grads)


class _HyperHeadFn(torch.autograd.Function):
    """Last linear of a HyperNetwork head for a HIDDEN hypo weight (meta_modules.py:32-35, 50-54) through
    siren_b200_hyper_head: ``(h [B, k_h], Wlast [65536, k_h], blast [65536]) -> W [B, 256, 256]`` fp32 plus, from the
    same pass over Wlast, the two tensor-core operands of that weight (fp16 as stored, bf16 ``w0 W^T``) and
    ``sum W^2`` (the term loss_functions.hypo_weight_loss adds up).  The backward is three plain GEMMs (cuBLAS)."""

    @staticmethod
    def forward(ctx, h, Wlast, blast, w0):
        lib = _lib.load()
        h_c, W_c, b_c = h.detach().contiguous(), Wlast.detach().contiguous(), blast.detach().contiguous()
        Bn, K = h_c.shape
        dev = h_c.device
        W = torch.empty((Bn, 256, 256), dtype=torch.float32, device=dev)
        wk = torch.empty((Bn, 256, 256), dtype=torch.float16, device=dev)
        wt = torch.empty((Bn, 256, 256), dtype=torch.bfloat16, device=dev)
        ss = torch.zeros((), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            rc = lib.siren_b200_hyper_head(_lib.dptr(h_c), _lib.dptr(W_c), _lib.dptr(b_c), Bn, K, ctypes.c_float(w0),
                                           _lib.dptr(W), _lib.dptr(wk), _lib.dptr(wt), _lib.dptr(ss),
                                           torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(rc, "siren_b200_hyper_head")
        ctx.save_for_backward(h_c, W_c, W)
        ctx.mark_non_differentiable(wk, wt)
        ctx.set_materialize_grads(False)
        return W, wk, wt, ss

    @staticmethod
    def backward(ctx, gW, _gwk, _gwt, gss):
        h, Wlast, W = ctx.saved_tensors
        g = gW
        if gss is not None:      # d (sum W^2) / dW = 2 W
            g = 2.0 * gss * W if g is None else g + 2.0 * gss * W
        if g is None:
            return None, None, None, None
        gf = g.reshape(g.shape[0], -1)
        dh = gf @ Wlast if ctx.needs_input_grad[0] else None
        dWl = gf.t() @ h if ctx.needs_input_grad[1] else None
        dbl = gf.sum(0) if ctx.needs_input_grad[2] else None
        return dh, dWl, dbl, None


def hyper_head_supported(h, Wlast, blast):
    """True when siren_b200_hyper_head serves this head: a hidden hypo weight (65,536 outputs), fp32 CUDA tensors,
    hyper_hidden_features a multiple of 4 up to 512."""
    return (torch.is_tensor(h) and h.is_cuda and h.dtype == torch.float32 and h.dim() == 2
            and Wlast.is_cuda and Wlast.dtype == torch.float32 and tuple(Wlast.shape) == (256 * 256, h.shape[1])
            and blast is not None and blast.dtype == torch.float32 and blast.numel() == 256 * 256
            and 4 <= h.shape[1] <= 512 and h.shape[1] % 4 == 0)


def attach_ops(W, wk, wt, ss, w0):
    """Tag a hypo weight with its ready-made operands (picked up by siren_mlp) and its sum of squares."""
    W._siren_ops = (wk, wt, float(w0), W._version)
    W._siren_sumsq = ss
    return W


def _prepared_ops(weights, w0, precision, n_tasks):
    """(wk16 list, wt16 list) when EVERY hidden weight carries operands written for this w0 and is unchanged since,
    and the call will take the fused bf16 path; else None."""
    if precision != "bf16":
        return None
    wk, wt = [], []
    for W in weights[1:-1]:
        tag = getattr(W, "_siren_ops", None)
        if tag is None or tag[2] != float(w0) or tag[3] != W._version or W.dim() != 3 or W.shape[0] != n_tasks \
                or tuple(W.shape[1:]) != (256, 256) or not W.is_contiguous():
            return None
        wk.append(tag[0])
        wt.append(tag[1])
    return wk, wt


class _AttachJ(torch.autograd.Function):
    """J' = J as a value; d J'[.., o, k] / d x_k := D[.., o, k]  (diagonal second derivatives)."""

    @staticmethod
    def forward(ctx, x, J, D):
        ctx.save_for_backward(D)
        ctx.has_D = D is not None
        return J.clone()

    @staticmethod
    def backward(ctx, gJ):
        (D,) = ctx.saved_tensors if ctx.has_D else (None,)
        gx = (gJ * D).sum(dim=-2) if D is not None else None
        return gx, gJ, None


class _AttachJNoD(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, J):
        return J.clone()

    @staticmethod
    def backward(ctx, gJ):
        return None, gJ


class _AttachY(torch.autograd.Function):
    """y' = y as a value; d y'[.., o] / d x_k := J[.., o, k]."""

    @staticmethod
    def forward(ctx, x, y, J):
        ctx.save_for_backward(J)
        return y.clone()

    @staticmethod
    def backward(ctx, gy):
        (J,) = ctx.saved_tensors
        gx = (gy.unsqueeze(-1) * J).sum(dim=-2)
        return gx, gy, None


def siren_mlp(coords, weights, biases, w0=30.0, precision="fp32", coord_derivs=0, coords_grad=False, fourier=None,
              dc=None):
    """Native sine MLP.  ``coords`` [B, N, d] fp32 CUDA; returns ``model_out`` [B, N, o].

    The result is differentiable w.r.t. weights/biases and (through the attached jets or the
    composed fallback) w.r.t. ``coords``.  With ``fourier`` = the ``[raw, F]`` matrix of
    features.GaussianFourierFeatureTransform, ``coords`` are the raw ``[B, N, raw]`` coordinates and the first layer
    (in_features = 2 F) reads their Fourier features, built on chip.  With ``dc = (k0, mask, noise_lvl,
    channels_first)`` the output leaves the kernels data-consistent (data_consistency.py:7-20; value path only)."""
    flat = []
    for W, b in zip(weights, biases):
        flat += [W, b]
    ops = None
    if not coord_derivs and not coords_grad:
        ops = _prepared_ops(weights, w0, precision, coords.shape[0])
    if dc is not None or ops is not None:
        if coord_derivs or coords_grad:
            raise ValueError("siren_mlp: the data-consistency epilogue serves the value path (no coordinate derivatives)")
        k0, mask, noise_lvl, channels_first = dc if dc is not None else (None, None, None, False)
        if not torch.is_grad_enabled():
            flat = [t.detach() for t in flat]
        return _SirenDCFn.apply(float(w0), precision, noise_lvl, bool(channels_first), coords.detach(), fourier, k0, mask,
                                ops, *flat)
    if fourier is not None:
        if not torch.is_grad_enabled():
            flat = [t.detach() for t in flat]
        return _SirenFourierFn.apply(float(w0), precision, coords.detach(), fourier, *flat)
    order = int(coord_derivs)
    if not torch.is_grad_enabled():
        # torch.no_grad(): ctx.needs_input_grad still mirrors requires_grad inside Function.forward,
        # so hand the kernel detached tensors -- that is what selects the stash-free inference launch
        coords = coords.detach()
        flat = [t.detach() for t in flat]
    if order == 0 or not coords.requires_grad:
        out = _SirenKernelFn.apply(float(w0), precision, 0, bool(coords_grad), coords, *flat)
        return out
    ws_, bs_ = list(weights), list(biases)
    # the kernel Function sees detached coordinates: the only autograd path from the outputs to
    # ``coords`` is through the attach Functions below
    if order == 1:
        y, J = _SirenKernelFn.apply(float(w0), precision, 1, False, coords.detach(), *flat)
        Jx = _AttachJNoD.apply(coords, J)
    else:
        y, J, D = _SirenKernelFn.apply(float(w0), precision, 2, False, coords.detach(), *flat)
        Jx = _AttachJ.apply(coords, J, D)
    out = _AttachY.apply(coords, y, Jx)
    # The jets carry first derivatives and the DIAGONAL second derivatives only.  Queries that need mixed second
    # derivatives (diff_operators.hessian, jacobian of a gradient) cannot be answered from them: they re-evaluate the
    # composed graph through this hook (see tag_composed / composed_of) instead of silently reading zeros.
    tag_composed(out, lambda: composed_mlp(coords, ws_, bs_, w0), order)
    return out


def tag_composed(out, fn, order):
    """Attach to a jet-path output the closure that re-evaluates it as the composed PyTorch graph on the same
    coordinate leaf (a plain Python attribute: reshaped views must be re-tagged, modules.FCBlock does)."""
    out._siren_composed = fn
    out._siren_jets = order
    return out


def composed_of(y):
    """``y`` itself, or -- when it came from the native jet path -- the same function of the same coordinate leaf
    and parameters as a composed PyTorch graph (exact for derivatives of any order, including mixed ones)."""
    fn = getattr(y, "_siren_composed", None)
    return y if fn is None else fn()
