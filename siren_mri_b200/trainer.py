"""Fast training step: forward, loss + loss gradient, backward, gradient all-reduce, clip + Adam -- one CUDA
graph, no host synchronisation.  Losses: ``image_mse`` (loss_functions.py:66-96, the image fits, cfg1 / cfg2),
``sdf`` (loss_functions.py:460-484, first-order coordinate derivatives, cfg3) and ``laplace_mse``
(loss_functions.py:350-355, second order, cfg4); the derivative losses read the jets the forward kernels return.

It is the sibling of the reference loop body at training.py:66-103
(``model(model_input)`` -> ``image_mse`` -> ``backward`` -> ``clip_grad_norm_`` -> ``Adam.step``)
with identical arithmetic, for callers that do not need the per-step tensorboard scalars
(training.py:77-81 force a device->host sync every step).  The model is an ordinary
``modules.SingleBVPNet`` / ``FCBlock``; its parameters are re-homed into one flat buffer so that
the all-reduce is a single collective and Adam a single kernel (SURVEY.md section 8e).

Multi-GPU: every rank holds the full weights and a contiguous shard of the coordinates; the
loss weight carries the GLOBAL normalisation, gradients are summed with one flat all-reduce
(``torch.distributed``, NCCL over NVLink) and every rank applies the same Adam update, so the
replicas stay bit-identical without a broadcast.

Several scenes: ``SirenTrainer([model_0, ..., model_{T-1}], n)`` fits T independent networks of one architecture in
one step, as T tasks with per-task weights (one SIREN per image, MRI slice or frame).  Each scene has its own
image_mse, its own clip_grad_norm_ and its own Adam moments -- T reference loops (training.py:66-103) sharing the step
counter and the hyper-parameters.  The models' parameters become task slices of per-layer stacked tensors
[T, out, in] / [T, out] inside the one flat buffer; ``loss`` is then the [T] vector of the scenes' losses.

Scenes of different sizes: ``SirenTrainer(models, n_coords=[n_0, ..., n_{T-1}])`` gives scene t its own coordinate
count.  ``coords`` / ``gt`` / ``y`` are then packed, [sum n_t, features] without gaps (``scene(t)`` returns scene t's
views), and memory and work follow sum n_t rather than T * max n_t.  Each scene's image_mse is its own sum of squares /
16384, as in the reference loop.  This runs on the one-kernel bf16 step only (image_mse, in_features <= 4,
out_features <= 2, at most 4 hidden layers; ValueError elsewhere), even with a single scene or equal counts.
"""
import os

import torch

from . import _lib
from .optim import FusedAdam, flatten_parameters, flatten_parameters_stacked


def _fcblock_of(model):
    net = model
    while not hasattr(net, "_n_layers"):
        net = net.net
    return net


# loss name -> (order of the coordinate jets the forward must return, ground-truth tensors as (dict key, features))
LOSSES = {
    "image_mse": (0, None),                              # gt['img'] [1, N, out_features]
    "sdf": (1, (("sdf", 1), ("normals", 3))),            # gt['sdf'] [1, N, 1], gt['normals'] [1, N, 3]
    "laplace_mse": (2, (("laplace", 1),)),               # gt['laplace'] [1, N, 1]
}


class SirenTrainer:
    def __init__(self, model, n_coords, lr=1e-4, loss_weight=None, max_grad_norm=0.0, precision=None,
                 process_group=None, use_graph=True, comm="c_abi", distributed=True, loss="image_mse"):
        if loss not in LOSSES:
            raise ValueError("loss must be one of %s" % sorted(LOSSES))
        self.loss_kind = loss
        models = list(model) if isinstance(model, (list, tuple)) else [model]
        if not models:
            raise ValueError("SirenTrainer needs at least one model")
        self.tasks = len(models)          # scenes trained side by side, each by its own model
        # a list of counts: scenes of different sizes, packed (the ragged step); an int: every scene has n_coords
        self.counts = None
        if isinstance(n_coords, (list, tuple)):
            if len(n_coords) != self.tasks:
                raise ValueError("n_coords has %d counts for %d scenes" % (len(n_coords), self.tasks))
            if any(int(c) != c or int(c) < 1 for c in n_coords):
                raise ValueError("every scene needs a positive integer coordinate count (got %s)" % list(n_coords))
            self.counts = [int(c) for c in n_coords]
        self._stacked = self.tasks > 1 or self.counts is not None      # per-task weights and tail
        blocks = [_fcblock_of(m) for m in models]
        self.block = blocks[0]
        if not self.block._sine:
            raise ValueError("SirenTrainer needs a sine FCBlock")
        if self._stacked:
            self._check_scenes(blocks, loss)
        self.lib = _lib.load()
        params = list(self.block.parameters())
        self.device = params[0].device
        if self.device.type != "cuda":
            raise _lib.NativeError("SirenTrainer needs the model on a CUDA device")
        self.pg = process_group
        self.world = 1
        self.comm = None
        self.p2p = None           # fused all-reduce over peer memory (comm 'p2p' / 'auto'), see _make_p2p
        # distributed=False: a purely local trainer inside a multi-rank job (no gradient all-reduce)
        if distributed and (process_group is not None or
                            (torch.distributed.is_available() and torch.distributed.is_initialized())):
            self.world = torch.distributed.get_world_size(process_group)
        if self._stacked and self.world > 1:
            raise ValueError("several scenes train on one rank: pass distributed=False (one trainer per rank; the "
                             "scenes share no gradients, so no collective is needed)")
        n_flat = sum(p.numel() for p in params)
        grad0 = None
        if self.world > 1 and comm in ("p2p", "auto"):
            self.p2p = self._make_p2p(n_flat)
            if self.p2p is not None:
                grad0 = self.p2p["bufs"][0]
            elif comm == "p2p":
                raise _lib.NativeError("SirenTrainer(comm='p2p'): symmetric memory is not available on this system")
            else:
                comm = "c_abi"
        layers = range(self.block._n_layers)
        if not self._stacked:
            self.flat, self.grad = flatten_parameters(params, grad0)
            self.weights = [self.block.net[l][0].weight for l in layers]
            self.biases = [self.block.net[l][0].bias for l in layers]
            self._wgrads, self._bgrads = [w.grad for w in self.weights], [b.grad for b in self.biases]
        else:
            # W_0, b_0, W_1, ...: per layer one [T, out, in] and one [T, out] block of the flat buffer
            self.flat, self.grad, stacked, stacked_grad = flatten_parameters_stacked(
                [[p for l in layers for p in (b.net[l][0].weight, b.net[l][0].bias)] for b in blocks])
            self.weights, self.biases = stacked[0::2], stacked[1::2]
            self._wgrads, self._bgrads = stacked_grad[0::2], stacked_grad[1::2]
        self.opt = FusedAdam(self.flat, self.grad, lr=lr, max_grad_norm=max_grad_norm)
        if self.world > 1 and comm == "c_abi":
            self.comm = self._make_comm()
        d_in = self.weights[0].shape[-1]
        d_out = self.weights[-1].shape[-2]
        self.n = sum(self.counts) if self.counts else int(n_coords)      # rows of coords / gt / y
        self.precision = precision or self.block._opt("precision")
        desc = _lib.SirenDesc()
        desc.d_in, desc.hidden, desc.n_hidden, desc.d_out = d_in, self.weights[0].shape[-2], self.block._n_layers - 2, d_out
        desc.w0, desc.tasks, desc.per_task, desc.n_coords = self.block._w0, self.tasks, int(self._stacked), self.n
        if self.counts:
            desc.n_coords = max(self.counts)      # (not read by the ragged entries)
        order, gt_spec = LOSSES[loss]
        if order and (d_out != 1 or d_in > 3):
            raise ValueError("loss %r needs a scalar output and in_features <= 3" % loss)
        if loss == "sdf" and d_in != 3:
            raise ValueError("loss 'sdf' needs in_features == 3")
        desc.precision, desc.deriv_order = _lib.PRECISIONS[self.precision], order
        self.desc = desc
        if self.counts:
            self._counts_c = _lib.long_array(self.counts)
            nbytes = self.lib.siren_b200_workspace_bytes_ragged(desc, self._counts_c)
            if nbytes == 0:      # outside the ragged step's envelope, or bad counts
                raise ValueError("scenes of different sizes: %s" % self.lib.siren_b200_last_error().decode())
            starts = [0]
            for c in self.counts:
                starts.append(starts[-1] + c)
            self._starts = starts
        else:
            nbytes = self.lib.siren_b200_workspace_bytes_ex(desc, 0)      # the step never asks for coordinate gradients
        if nbytes == 0:
            _lib.check(1, "siren_b200_workspace_bytes")
        dev = self.device
        self.ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        T = self.tasks
        lead = () if self.counts else (T,)      # packed [sum n_t, .] with counts
        self.coords = torch.zeros(lead + (self.n, d_in), device=dev)
        self.gt_keys = [k for k, _ in gt_spec] if gt_spec else ["img"]
        self.gts = [torch.zeros(lead + (self.n, f), device=dev) for _, f in (gt_spec or (("img", d_out),))]
        self.gt = self.gts[0]
        self.y = torch.empty(lead + (self.n, d_out), device=dev)
        self.gy = torch.zeros_like(self.y)
        self.J = torch.empty((1, self.n, d_out, d_in), device=dev) if order >= 1 else None
        self.D = torch.empty((1, self.n, d_out, d_in), device=dev) if order >= 2 else None
        self.gJ = torch.zeros_like(self.J) if loss == "sdf" else None
        self.gD = torch.zeros_like(self.D) if order >= 2 else None
        # [0] loss of the last finished step, [1] running sum of the step in flight (include/siren_b200.h: loss4)
        self.loss4 = torch.zeros(4, device=dev)
        self.loss = self.loss4[0:1]
        if self._stacked:
            # per scene: [0, T) loss of the last finished step, [T, 2T) running sums (loss4 keeps their total)
            self.task_loss = torch.zeros(2 * T, device=dev)
            self.loss = self.task_loss[:T]
            self.opt._task_state(T)
        # image_mse (loss_functions.py:88): sum of squares / 16384 regardless of the image size; the derivative losses
        # are means over the points: their weight is this shard's share of the batch
        default_w = (1.0 / 16384.0) if loss == "image_mse" else 1.0 / self.world
        self.loss_weight = default_w if loss_weight is None else float(loss_weight)
        self._w_ptrs = _lib.ptr_array(self.weights)
        self._b_ptrs = _lib.ptr_array(self.biases)
        self._dw_ptrs = _lib.ptr_array(self._wgrads)
        self._db_ptrs = _lib.ptr_array(self._bgrads)
        self._parity = 0          # p2p: which of the two gradient buffers the step in flight accumulates into
        if self.p2p is not None:
            # the same views into the second gradient buffer
            base0, base1 = self.p2p["bufs"][0].data_ptr(), self.p2p["bufs"][1].data_ptr()
            ptrs = lambda ts: [_lib.ptr_array([t.grad for t in ts]),      # noqa: E731
                               _lib.ptr_array_raw([t.grad.data_ptr() - base0 + base1 for t in ts])]
            self._dw_ptrs2, self._db_ptrs2 = ptrs(self.weights), ptrs(self.biases)
        self.use_graph = use_graph
        self.graph = None
        self.steps = 0            # completed optimizer steps (host count; the device counter is in opt.state)
        self.micro = 0            # micro-batches accumulated since the last optimizer step (gradient accumulation)
        # kernels of this library launched per step (see csrc/api.cu):
        #   bf16 image_mse (the fused kernels): mlp_fused_fwd, mlp_fused_bwd, one wgrad per group of four hidden
        #   layers, adam_step; mlp_fused_step replaces the first two for <= 4 hidden layers, d_in <= 4 and d_out <= 2
        #   (SIREN_FUSED_STEP=0: not); + sumsq with clipping, + prep_first for d_in > 4, + last_fwd / mse_grad /
        #   last_bwd when the outermost linear is not fused (d_out > 2)
        #   per-layer path: first_fwd, hidden_fwd and hidden_dgrad per hidden layer, mse_grad, last_bwd, wgrad,
        #   adam_step; plus (fp32-parity) colsum per hidden layer below the top, last_fwd, first_bwd
        nh = desc.n_hidden
        clip = 1 if max_grad_norm > 0 else 0
        if self.counts:
            self.kernels_per_step = 3 + clip      # mlp_fused_step_ragged, wgrad_ragged, adam_step (+ its norm pass)
        elif self.precision == "bf16" and order == 0:
            self.kernels_per_step = 3 + (nh + 3) // 4 + clip + (0 if d_out <= 2 else 3) + (0 if d_in <= 4 else 1)
            if nh <= 4 and d_in <= 4 and d_out <= 2 and os.environ.get("SIREN_FUSED_STEP", "1")[:1] != "0":
                self.kernels_per_step -= 1
        else:
            self.kernels_per_step = 2 * nh + 5 + clip
            if self.precision != "bf16":
                self.kernels_per_step += (nh - 1) + 2
        if self.counts:      # the scenes' prefix tables, once per count vector
            with torch.cuda.device(dev):
                _lib.check(self.lib.siren_b200_prepare_ragged(desc, self._counts_c, _lib.dptr(self.ws),
                                                              torch.cuda.current_stream(dev).cuda_stream),
                           "prepare_ragged")
        self.refresh_weights()

    def scene(self, t):
        """Scene t's (coords, gt, y) as views of the packed buffers (scenes of different sizes)."""
        if not self.counts:
            return self.coords[t], self.gt[t], self.y[t]
        a, b = self._starts[t], self._starts[t + 1]
        return self.coords[a:b], self.gt[a:b], self.y[a:b]

    @staticmethod
    def _check_scenes(blocks, loss):
        """Several scenes step as one stacked network: same architecture, w0 and precision, the image loss."""
        if len(blocks) > 1024:
            raise ValueError("at most 1024 scenes per trainer (got %d)" % len(blocks))
        if loss != "image_mse":
            raise ValueError("several scenes train with loss 'image_mse' only (got %r)" % loss)
        ref = blocks[0]
        shapes = [tuple(p.shape) for p in ref.parameters()]
        for b in blocks[1:]:
            if not b._sine or b._n_layers != ref._n_layers or [tuple(p.shape) for p in b.parameters()] != shapes:
                raise ValueError("the scenes' models must share one architecture")
            if b._w0 != ref._w0:
                raise ValueError("the scenes' models must share w0 (%g, %g)" % (ref._w0, b._w0))
            if b._opt("precision") != ref._opt("precision"):
                raise ValueError("the scenes' models must share one precision (%s, %s)"
                                 % (ref._opt("precision"), b._opt("precision")))

    def _make_comm(self):
        """NCCL communicator of the C ABI: rank 0 draws the id, torch.distributed hands it round."""
        import ctypes
        dist = torch.distributed
        rank = dist.get_rank(self.pg)
        idbuf = (ctypes.c_char * 128)()
        if rank == 0:
            _lib.check(self.lib.siren_b200_comm_unique_id(ctypes.cast(idbuf, ctypes.c_void_p)), "comm_unique_id")
        t = torch.frombuffer(bytearray(bytes(idbuf)), dtype=torch.uint8).clone().to(self.device)
        dist.broadcast(t, src=dist.get_global_rank(self.pg, 0) if self.pg is not None else 0, group=self.pg)
        raw = bytes(t.cpu().numpy().tobytes())
        comm = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            rc = self.lib.siren_b200_comm_init(rank, self.world, ctypes.c_char_p(raw), ctypes.byref(comm))
        _lib.check(rc, "comm_init")
        return comm

    def _make_p2p(self, n_flat):
        """Two flat gradient buffers in ONE symmetric-memory allocation every rank of the box can read over NVLink
        (torch.distributed._symmetric_memory), and per buffer the device array of the ranks' pointers the fused
        Adam kernel sums over.  Returns None -- on EVERY rank, the decision is all-reduced -- when that is not
        available, and the trainer falls back to the NCCL all-reduce."""
        dist = torch.distributed
        ok, hdl, buf = 1, None, None
        n_pad = (n_flat + 1023) // 1024 * 1024
        try:
            import torch.distributed._symmetric_memory as symm
            group = self.pg if self.pg is not None else dist.group.WORLD
            buf = symm.empty(2 * n_pad, dtype=torch.float32, device=self.device)
            hdl = symm.rendezvous(buf, group)
            ptrs = [int(p) for p in hdl.buffer_ptrs]
            if len(ptrs) != self.world or any(p == 0 for p in ptrs):
                ok = 0
        except Exception as e:          # pragma: no cover  (no NVLink peer access, old driver, ...)
            ok = 0
            self._p2p_error = repr(e)
        flag = torch.tensor([ok], device=self.device, dtype=torch.int32)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.pg)
        if int(flag.item()) == 0:
            return None
        buf.zero_()
        peers = [torch.tensor([p + par * n_pad * 4 for p in ptrs], dtype=torch.int64, device=self.device)
                 for par in (0, 1)]
        torch.cuda.synchronize(self.device)
        dist.barrier(group=self.pg)      # every rank's buffers are zero before anyone's first step can read them
        return dict(hdl=hdl, buf=buf, bufs=[buf[0:n_flat], buf[n_pad:n_pad + n_flat]], peers=peers)

    def refresh_weights(self):
        """(Re)build the bf16 copies of the hidden weights in the workspace.  The captured step does not convert
        the weights -- its Adam kernel keeps the copies current -- so this runs once here and must be called again
        after any outside change of the parameters (``load_state_dict``, manual edits)."""
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            _lib.check(self.lib.siren_b200_prepare_weights(self.desc, self._w_ptrs, _lib.dptr(self.ws), stream),
                       "prepare_weights")

    def _fwd_bwd(self, coords, gt, weight, stream):
        lib, d, P = self.lib, self.desc, _lib.dptr
        gts = list(gt) if isinstance(gt, (list, tuple)) else [gt]
        dw_ptrs, db_ptrs = self._dw_ptrs, self._db_ptrs
        if self.p2p is not None:      # the gradient buffer of this step's parity
            dw_ptrs, db_ptrs = self._dw_ptrs2[self._parity], self._db_ptrs2[self._parity]
        if self.loss_kind != "image_mse":
            # forward with jets -> loss value and its gradient w.r.t. (y, J, D) -> reverse of the jets
            _lib.check(lib.siren_b200_forward_prepared(d, P(coords), self._w_ptrs, self._b_ptrs, P(self.y), P(self.J),
                                                       P(self.D), P(self.ws), stream), "forward_prepared")
            if self.loss_kind == "sdf":
                _lib.check(lib.siren_b200_sdf_grad(P(self.y), P(self.J), P(gts[0]), P(gts[1]), P(self.gy), P(self.gJ),
                                                   self.n, weight, P(self.loss4), stream), "sdf_grad")
            else:
                _lib.check(lib.siren_b200_laplace_mse_grad(P(self.D), P(gts[0]), P(self.gD), self.n, d.d_in, weight,
                                                           P(self.loss4), stream), "laplace_mse_grad")
            _lib.check(lib.siren_b200_backward(d, P(coords), self._w_ptrs, self._b_ptrs, P(self.ws), P(self.gy),
                                               P(self.gJ), P(self.gD), dw_ptrs, db_ptrs, None, 1, stream),
                       "backward")
            return
        gt = gts[0]
        if self.counts:
            # the ragged step: each scene's loss goes to task_loss[T + t] from inside the step kernel
            _lib.check(lib.siren_b200_forward_backward_mse_ragged(
                d, self._counts_c, P(coords), self._w_ptrs, self._b_ptrs, P(self.y), P(gt), weight, None, P(self.loss4),
                P(self.task_loss), P(self.ws), 1, dw_ptrs, db_ptrs, 1, stream), "forward_backward_mse_ragged")
            return
        # forward + loss + loss gradient + backward: one kernel up to the weight gradients on the fused path (it forms
        # gy and the loss sum as it completes y and keeps gy on chip); every gradient is a view of one flat buffer the
        # previous adam_step left cleared: the kernels accumulate
        _lib.check(lib.siren_b200_forward_backward_mse(d, P(coords), self._w_ptrs, self._b_ptrs, P(self.y), P(gt), weight,
                                                       None, P(self.loss4), P(self.ws), 1, dw_ptrs, db_ptrs, 1, stream),
                   "forward_backward_mse")

    # one step, enqueued on the current stream (batch buffers other than self.coords / self.gt: the pipelined entry)
    def _enqueue(self, coords=None, gt=None, loss_out=None, update=True, accumulation_steps=1):
        lib = self.lib
        coords = self.coords if coords is None else coords
        gt = self.gts if gt is None else gt
        stream = torch.cuda.current_stream(self.device).cuda_stream
        P = _lib.dptr
        self._fwd_bwd(coords, gt, self.loss_weight / accumulation_steps, stream)
        if accumulation_steps > 1 and self.opt.max_grad_norm > 0 and not self._stacked:
            # training.py:93-97 clips the ACCUMULATED gradient in place after every micro-batch
            _lib.check(lib.siren_b200_clip_grad(P(self._cur_grad()), self.grad.numel(), self.opt.max_grad_norm,
                                                P(self.opt.state), stream), "clip_grad")
        if self._stacked:
            self._tasks_tail(gt[0], update, accumulation_steps)
        elif update and self.p2p is not None:
            # all-reduce fused into the Adam kernel: one symmetric-memory barrier (every rank's backward of this step is
            # complete), then every rank sums the ranks' buffers of this parity from peer memory and clears the other
            par = self._parity
            self.p2p["hdl"].barrier(channel=0)
            self.opt.g = self.p2p["bufs"][par]
            self.opt.step_peers(self.p2p["peers"][par], self.world, self.p2p["bufs"][1 - par], loss4=self.loss4,
                                desc=self.desc, w_ptrs=self._w_ptrs, ws=self.ws, clip=accumulation_steps == 1)
            # (the parity flips when the step EXECUTES: _flip, called by step / submit_from_host / _warm_up)
        elif update:
            if self.world > 1:
                if self.comm is not None:
                    _lib.check(lib.siren_b200_allreduce(self.comm, P(self.grad), self.grad.numel(), stream), "allreduce")
                else:
                    torch.distributed.all_reduce(self.grad, group=self.pg)
            self.opt.step_fused(zero_grad=True, loss4=self.loss4, desc=self.desc, w_ptrs=self._w_ptrs, ws=self.ws,
                                clip=accumulation_steps == 1)
        else:
            _lib.check(lib.siren_b200_loss_roll(P(self.loss4), stream), "loss_roll")
        if loss_out is not None:
            # pinned host word, written by a kernel (a copy-engine node here costs ~35 us per step of hand-over)
            _lib.check(lib.siren_b200_publish(P(self.loss), loss_out.data_ptr(), self.tasks, stream), "publish")

    def _tasks_tail(self, gt, update, accumulation_steps):
        """The optimizer tail of several scenes: each scene clipped by its own gradient norm (with accumulation after
        every micro-batch, training.py:93-97), Adam, and each scene's image_mse from self.y and gt -- in the norm pass
        with clipping, in the Adam launch otherwise."""
        opt, w = self.opt, self.loss_weight / accumulation_steps
        clip_each = accumulation_steps > 1 and opt.max_grad_norm > 0
        y = None if self.counts else self.y      # the ragged step has added the losses itself
        gt = None if self.counts else gt
        if clip_each or not update:
            opt.clip_tasks(self.desc, self._dw_ptrs, self._db_ptrs, self.task_loss, y, gt, w, self.loss4,
                           clip=clip_each, publish=not update)
        if update:
            yg = (None, None) if clip_each else (y, gt)      # the losses are in already
            opt.step_tasks(self.desc, self._w_ptrs, self._b_ptrs, self.task_loss, yg[0], yg[1], w, self.loss4, self.ws,
                           clip=accumulation_steps == 1)

    def _cur_grad(self):
        return self.grad if self.p2p is None else self.p2p["bufs"][self._parity]

    def gradients(self):
        """The flat gradient of the loss on ``self.coords`` / ``self.gt`` at the current weights, through exactly the
        launches a step makes (forward_mse, backward) but without the update, and the loss ([T] per scene).
        Test / inspection hook."""
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            self._fwd_bwd(self.coords, self.gts, self.loss_weight, stream)
            g = self._cur_grad().clone()
            loss = self.loss4[1:2].clone()
            if self._stacked:
                if not self.counts:
                    self.opt.clip_tasks(self.desc, self._dw_ptrs, self._db_ptrs, self.task_loss, self.y, self.gt,
                                        self.loss_weight, None, clip=False, publish=False)
                loss = self.task_loss[self.tasks:].clone()
                self.task_loss[self.tasks:].zero_()
            self._cur_grad().zero_()
            self.loss4[1:2].zero_()
        return g, loss

    def _warm_up(self, update=True, accumulation_steps=1):
        """Two steps of the variant about to be captured, outside capture (function attributes, lazily loaded kernels,
        NCCL), with parameters, optimizer state and gradient restored afterwards."""
        key = (bool(update), int(accumulation_steps))
        warm = self.__dict__.setdefault("_warm", set())
        if key in warm:
            return
        tensors = (self.flat, self.opt.m, self.opt.v, self.opt.state, self.loss4,
                   self.grad if self.p2p is None else self.p2p["buf"])
        if self._stacked:
            tensors += (self.task_loss, self.opt.task_sumsq)
        state = [t.clone() for t in tensors]
        s = torch.cuda.Stream(self.device)
        s.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(s):
            for _ in range(2):           # an even number: the gradient-buffer parity ends where it started
                self._enqueue(None, None, None, update, accumulation_steps)
                self._flip(update)
        torch.cuda.current_stream(self.device).wait_stream(s)
        torch.cuda.synchronize(self.device)
        if self.p2p is not None:         # no rank restores (rewrites) its buffers while a peer's warm-up still reads them
            torch.distributed.barrier(group=self.pg)
        for dst, src in zip(tensors, state):
            dst.copy_(src)
        self.refresh_weights()            # the warm-up steps moved the weights (and their bf16 copies): back in step
        torch.cuda.synchronize(self.device)
        warm.add(key)

    def _capture(self, coords=None, gt=None, loss_out=None, update=True, accumulation_steps=1):
        self._warm_up(update, accumulation_steps)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            self._enqueue(coords, gt, loss_out, update, accumulation_steps)
        return graph              # capture does not execute: state is untouched

    def _count(self, update):
        self.micro += 1
        if update:
            self.steps += 1
            self.micro = 0

    def _flip(self, update):
        """An executed optimizer step of the fused-all-reduce path moves on to the other gradient buffer."""
        if update and self.p2p is not None:
            self._parity ^= 1

    def _key(self, update, accumulation_steps):
        return (bool(update), int(accumulation_steps), self._parity)

    def step(self, update=True, accumulation_steps=1):
        """Run one training step on the data currently in ``self.coords`` / ``self.gt``.

        Gradient accumulation as at training.py:90, 99-103: every call adds the gradient of ``loss /
        accumulation_steps`` to the flat buffer (and, with clipping, clips the accumulated gradient in place, as
        the reference does after every micro-batch); the optimizer moves only when ``update`` is true."""
        self._count(update)
        with torch.cuda.device(self.device):
            if not self.use_graph:
                self._enqueue(None, None, None, update, accumulation_steps)
                self._flip(update)
                return
            if self.graph is None:
                self.graph = {}
            key = self._key(update, accumulation_steps)      # one graph per gradient-buffer parity (fused all-reduce)
            if key not in self.graph:
                self.graph[key] = self._capture(None, None, None, update, accumulation_steps)
            self.graph[key].replay()
            self._flip(update)

    def step_from_host(self, coords_host, gt_host, update=True, accumulation_steps=1):
        """Public end-to-end step: pinned host batch in, loss value out.  With scenes of different sizes the batch is
        packed [sum n_t, .] or a list of the T scenes' tensors."""
        self.coords.copy_(self._host_coords(coords_host), non_blocking=True)
        for dst, src in zip(self.gts, self._gt_list(gt_host)):
            dst.copy_(src.view_as(dst), non_blocking=True)
        self.step(update, accumulation_steps)
        if self._stacked:
            return [v * accumulation_steps for v in self.loss.tolist()]
        return float(self.loss.item()) * accumulation_steps

    def _gt_list(self, gt_host):
        """One host tensor per ground-truth tensor of the loss: a tensor, a sequence, or the reference's gt dict."""
        if isinstance(gt_host, dict):
            gt_host = [gt_host[k] for k in self.gt_keys]
            if self.counts:
                gt_host = gt_host[0]
        if self.counts:      # one tensor, packed or as the scenes' list
            return [self._pack(gt_host, self.gt.shape[-1])]
        return list(gt_host) if isinstance(gt_host, (list, tuple)) else [gt_host]

    def _host_coords(self, coords_host):
        if self.counts:
            return self._pack(coords_host, self.coords.shape[-1])
        return coords_host.view_as(self.coords)

    def _pack(self, x, features):
        """A packed [sum n_t, features] tensor from a packed tensor or a list of the T scenes' tensors."""
        if isinstance(x, (list, tuple)):
            if len(x) != self.tasks:
                raise ValueError("expected %d scene tensors, got %d" % (self.tasks, len(x)))
            for t, (xt, n) in enumerate(zip(x, self.counts)):
                if xt.numel() != n * features:
                    raise ValueError("scene %d: %d values, expected %d x %d" % (t, xt.numel(), n, features))
            x = torch.cat([xt.reshape(-1, features) for xt in x])
            return x.pin_memory() if x.device.type == "cpu" else x
        return x.reshape(self.n, features)

    def submit_from_host(self, coords_host, gt_host, update=True, accumulation_steps=1):
        """Pipelined end-to-end step: enqueue (pinned host batch -> device -> step -> loss to pinned host memory)
        and return a handle at once; ``handle.result()`` blocks for that step's loss.  Reading a step's loss
        after submitting the next step lets the upload of step k+1 run under the kernels of step k.

        Four batch slots (device coords + gt, one pinned loss word, one captured graph each) are used in turn: the
        upload goes straight into the slot its graph reads, on a copy stream, and the loss leaves through a kernel
        at the end of the graph that stores it to pinned host memory (siren_b200_publish) -- the compute stream
        carries nothing but graph launches, and no copy-engine hand-over.

        (The training loop of the reference logs the loss every step, training.py:83-104; a loop built on this
        call logs it one step late.)"""
        dev = self.device
        if getattr(self, "_slots", None) is None:
            self._copy_stream = torch.cuda.Stream(dev)
            self._slots = [dict(coords=torch.empty_like(self.coords), gt=[torch.empty_like(g) for g in self.gts],
                                loss=torch.zeros(self.tasks, dtype=torch.float32).pin_memory(), staged=torch.cuda.Event(),
                                done=torch.cuda.Event(), graphs={}) for _ in range(4)]
            self._submitted = 0
        key = self._key(update, accumulation_steps)
        if self.use_graph and key not in self._slots[self._submitted % len(self._slots)]["graphs"]:
            # the graphs of this kind for every slot now: no capture (it synchronises) in later steps.  With the fused
            # all-reduce the gradient-buffer parity alternates from step to step, so slot i + k is captured for the
            # parity it will see if every step is an optimizer step.
            with torch.cuda.device(dev):
                par0 = self._parity
                for k in range(len(self._slots)):
                    sl = self._slots[(self._submitted + k) % len(self._slots)]
                    if self.p2p is not None and update:
                        self._parity = (par0 + k) & 1
                    kk = self._key(update, accumulation_steps)
                    if kk not in sl["graphs"]:
                        sl["graphs"][kk] = self._capture(sl["coords"], sl["gt"], sl["loss"], update, accumulation_steps)
                self._parity = par0
        s = self._slots[self._submitted % len(self._slots)]
        self._submitted += 1
        self._count(update)
        cur = torch.cuda.current_stream(dev)
        cs = self._copy_stream
        cs.wait_event(s["done"])                  # the step that last read this slot has finished (no-op the first time)
        with torch.cuda.stream(cs):
            s["coords"].copy_(self._host_coords(coords_host), non_blocking=True)
            for dst, src in zip(s["gt"], self._gt_list(gt_host)):
                dst.copy_(src.view_as(dst), non_blocking=True)
            s["staged"].record(cs)
        with torch.cuda.device(dev):
            cur.wait_event(s["staged"])
            if self.use_graph:
                s["graphs"][key].replay()
            else:
                self._enqueue(s["coords"], s["gt"], s["loss"], update, accumulation_steps)
            self._flip(update)
        s["done"].record(cur)
        return _LossHandle(s["loss"], s["done"], float(accumulation_steps), self._stacked)


class _LossHandle:
    """Result of ``SirenTrainer.submit_from_host``: the step's loss (a list of the scenes' losses with several scenes)
    once its device-to-host copy has landed.  Valid until three further steps have been submitted (the pinned slots
    are a ring of four)."""

    def __init__(self, slot, event, scale=1.0, per_scene=False):
        self._slot, self._event, self._scale, self._per_scene = slot, event, scale, per_scene

    def result(self):
        self._event.synchronize()
        # the loss as logged: before the division by accumulation_steps
        if self._per_scene:
            return [v * self._scale for v in self._slot.tolist()]
        return float(self._slot[0]) * self._scale
