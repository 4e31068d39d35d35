"""Scenes of different sizes in one training step (siren_b200_forward_backward_mse_ragged and the ragged SirenTrainer):
packed coordinates / gt / y / gy, each scene with its own count, weights, gradients and loss.

Through the C entry against fp64 per scene, against the equal-N entry where the counts are equal, for robustness (NaN
guards behind every output, a 0xFF workspace, accumulate 0 / 1, gy = NULL, run to run, one scene's parameters changed)
and for its refusals; through the trainer, each scene against a single-scene trainer at its own count."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import siren_oracle as so
from tests.helpers import log_errors, oracle_chunked, rel_l2, rel_l2_per_task

pytestmark = pytest.mark.gpu

W_MSE = 1.0 / 16384.0


def _max_rel(a, ref):
    ref = np.asarray(ref, np.float64)
    return float(np.abs(np.asarray(a, np.float64) - ref).max() / max(np.sqrt((ref * ref).mean()), 1e-300))


class _Ragged:
    """The ragged entry through ctypes on device copies of seeded inputs.  Every buffer it writes is a view of a larger
    buffer whose tail holds NaN: a write past the view shows there."""

    def __init__(self, counts, d, nh, o, seed=300, precision="bf16"):
        from siren_mri_b200 import _lib
        self.counts, self.d, self.nh, self.o, self.T = list(counts), d, nh, o, len(counts)
        self.total = sum(counts)
        self.Ws, self.bs = so.make_params(d, 256, nh, o, seed=seed, tasks=self.T)
        rng = np.random.default_rng(seed + 1)
        self.x = rng.uniform(-1, 1, size=(self.total, d)).astype(np.float32)
        self.gt = rng.uniform(-1, 1, size=(self.total, o)).astype(np.float32)
        self.starts = np.concatenate([[0], np.cumsum(counts)]).astype(int)
        self.lib = _lib.load()
        self.Wd = [torch.from_numpy(w).cuda() for w in self.Ws]
        self.bd = [torch.from_numpy(b).cuda() for b in self.bs]
        self.xd = torch.from_numpy(self.x).cuda()
        self.gtd = torch.from_numpy(self.gt).cuda()
        self.desc = self.make_desc(precision)
        self.n_c = _lib.long_array(self.counts)
        self.nbytes = self.lib.siren_b200_workspace_bytes_ragged(self.desc, self.n_c)
        self.loss_init = np.array([3.0, 11.0, 5.0, 7.0], np.float32)
        self.tl_init = np.concatenate([np.arange(1, self.T + 1), np.zeros(self.T)]).astype(np.float32)

    def make_desc(self, precision="bf16"):
        from siren_mri_b200 import _lib
        desc = _lib.SirenDesc()
        desc.d_in, desc.hidden, desc.n_hidden, desc.d_out = self.d, 256, self.nh, self.o
        desc.w0, desc.tasks, desc.per_task, desc.n_coords = 30.0, self.T, 1, max(self.counts)
        desc.precision, desc.deriv_order = _lib.PRECISIONS[precision], 0
        return desc

    def workspace(self, fill=0xFF):
        assert self.nbytes > 0
        ws = torch.empty(self.nbytes, dtype=torch.uint8, device="cuda")
        ws.fill_(fill)
        _lib_check(self.lib.siren_b200_prepare_ragged(self.desc, self.n_c, ws.data_ptr(),
                                                      torch.cuda.current_stream().cuda_stream), "prepare_ragged")
        return ws

    @staticmethod
    def _guarded(shape, start=None):
        full = torch.full((shape[0] + 1,) + tuple(shape[1:]), float("nan"), device="cuda")
        view = full[:shape[0]]
        if start is not None:
            view.copy_(torch.from_numpy(np.asarray(start, np.float32)))
        return view, full[shape[0]:]

    def call(self, ws, gy=True, accumulate=0, grads=None, Wd=None):
        from siren_mri_b200 import _lib
        params = self.Ws + self.bs
        if grads is None:
            grads = [None if not accumulate else np.zeros(a.shape, np.float32) for a in params]
        y, yg = self._guarded((self.total, self.o))
        gyv, gyg = self._guarded((self.total, self.o)) if gy else (None, None)
        gv = [self._guarded(a.shape, s) for a, s in zip(params, grads)]
        # [0, T) is not the entry's (it must stay), [T, 2T) starts at zero: the scenes' losses are ~1e-5 .. 1, an fp32
        # start of order T would round them away
        tl, tlg = self._guarded((2 * self.T,), self.tl_init)
        loss4 = torch.from_numpy(self.loss_init.copy()).cuda()
        nl = len(self.Ws)
        P = _lib.dptr
        torch.cuda.synchronize()
        self.lib.siren_b200_profile_begin()
        rc = self.lib.siren_b200_forward_backward_mse_ragged(
            self.desc, self.n_c, P(self.xd), _lib.ptr_array(Wd or self.Wd), _lib.ptr_array(self.bd), P(y), P(self.gtd),
            W_MSE, P(gyv), P(loss4), P(tl), P(ws), 0, _lib.ptr_array([v for v, _ in gv[:nl]]),
            _lib.ptr_array([v for v, _ in gv[nl:]]), accumulate, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        buf = ctypes.create_string_buffer(1 << 14)
        self.lib.siren_b200_profile_end(buf, len(buf))
        _lib_check(rc, "forward_backward_mse_ragged")
        names = [ln.split()[0] for ln in buf.value.decode().strip().splitlines()]
        assert "mlp_fused_step_ragged" in names and "wgrad_ragged" in names, names
        assert "mlp_fused_step" not in names and "wgrad" not in names, names
        for what, g in [("y", yg), ("gy", gyg), ("task_loss", tlg)] + [("grad %d" % i, g) for i, (_, g) in enumerate(gv)]:
            assert g is None or bool(torch.isnan(g).all()), "write past the end of " + what
        return dict(y=y.cpu().numpy(), gy=None if gyv is None else gyv.cpu().numpy(), loss4=loss4.cpu().numpy(),
                    task_loss=tl.cpu().numpy(), g=[v.cpu().numpy() for v, _ in gv])

    def scene(self, a, t):
        return a[self.starts[t]:self.starts[t + 1]]

    def oracle(self):
        """fp64 y [total, o] and per-scene gradients [T, ...] (one oracle call per scene at its own count)."""
        y = np.empty((self.total, self.o))
        g = [np.zeros(a.shape) for a in self.Ws + self.bs]
        nl = len(self.Ws)
        for t in range(self.T):
            xt = self.scene(self.x, t)[None]
            gtt = self.scene(self.gt, t)[None].astype(np.float64)

            def adj(t0, t1, n0, n1, yc, Jc, Dc):
                return so.image_mse(yc, gtt[:, n0:n1], weight=W_MSE)[1], None, None
            yo, _, _, oW, ob = oracle_chunked(xt, [w[t:t + 1] for w in self.Ws], [b[t:t + 1] for b in self.bs], adj)
            y[self.starts[t]:self.starts[t + 1]] = yo[0]
            for l in range(nl):
                g[l][t] = oW[l][0]
                g[nl + l][t] = ob[l][0]
        return y, g

    def grad_errs(self, got, ref):
        nl = len(self.Ws)
        e = {}
        for l in range(nl):
            e["dW%d" % l] = rel_l2_per_task(got[l], ref[l])
            e["db%d" % l] = rel_l2_per_task(got[nl + l], ref[nl + l])
        return e


def _lib_check(rc, what):
    from siren_mri_b200 import _lib
    _lib.check(rc, what)


FP64_CASES = {
    # name: (counts, d_in, n_hidden, d_out)
    "edges_t11": ([1, 127, 128, 129, 255, 256, 257, 511, 512, 513, 4097], 2, 3, 1),
    "large_first_t3": ([65536, 1, 4097], 3, 2, 2),
    "small_first_t3": ([1, 257, 65536], 4, 4, 2),
    "t1": ([4097], 1, 1, 1),
    "t2": ([513, 128], 2, 4, 1),
    "t7": ([257, 1, 4097, 128, 511, 129, 255], 1, 2, 2),
    "t64": (list(np.random.default_rng(7).integers(1, 3000, size=64)), 2, 3, 1),
}


@pytest.mark.parametrize("case", sorted(FP64_CASES))
def test_ragged_step_against_fp64(case):
    """One call on a 0xFF workspace with NaN gradient buffers and accumulate = 0: y / gy per element, gradients and
    losses per scene against fp64; gy and each scene's loss exactly as the entry defines them from its own y."""
    counts, d, nh, o = FP64_CASES[case]
    e = _Ragged(counts, d, nh, o)
    out = e.call(e.workspace(0xFF))
    yo, gref = e.oracle()
    y, gy = out["y"], out["gy"]
    gyo = 2.0 * W_MSE * (yo - e.gt.astype(np.float64))
    errs = {"y": rel_l2(y, yo), "y_max": _max_rel(y, yo), "gy": rel_l2(gy, gyo), "gy_max": _max_rel(gy, gyo)}
    errs.update(e.grad_errs(out["g"], gref))
    # the outermost bias gradient is the sum of a scene's gy, which can cancel: per scene it is held to the sum of the
    # entry's own gy (see test_gpu_fused_step.py), over all scenes to fp64
    nl = len(e.Ws)
    gy64 = gy.astype(np.float64)
    own = np.stack([e.scene(gy64, t).sum(0) for t in range(e.T)])
    mag = np.stack([np.abs(e.scene(gy64, t)).sum(0) for t in range(e.T)])
    errs["dbL_own"] = float((np.abs(out["g"][-1] - own) / np.maximum(mag, 1e-30)).max())
    errs["db%d" % (nl - 1)] = rel_l2(out["g"][-1], gref[-1])
    # losses: each scene's w sum (y - gt)^2 of the entry's own y, and their total added to loss4[1]
    d2 = (y.astype(np.float64) - e.gt) ** 2
    ls = np.array([W_MSE * e.scene(d2, t).sum() for t in range(e.T)])
    lo = np.array([W_MSE * ((e.scene(yo, t) - e.scene(e.gt, t)) ** 2).sum() for t in range(e.T)])
    got = out["task_loss"][e.T:].astype(np.float64)
    errs["loss_own"] = float(np.max(np.abs(got - ls) / np.maximum(ls, 1e-30)))
    errs["loss_fp64"] = float(np.max(np.abs(got - lo) / np.maximum(lo, 1e-30)))
    log_errors("ragged_fp64/%s" % case, **errs)
    tol = 2e-2
    bad = {k: v for k, v in errs.items()
           if not v < {"y_max": 3e-2, "gy_max": 3e-2, "dbL_own": 1e-5, "loss_own": 1e-5, "loss_fp64": 5e-2}.get(k, tol)}
    assert not bad, (case, errs)
    assert np.array_equal(out["task_loss"][:e.T], e.tl_init[:e.T])
    assert np.array_equal(gy.view(np.uint32), (np.float32(2.0 * W_MSE) * (y - e.gt)).astype(np.float32).view(np.uint32))
    inc = float(out["loss4"][1]) - float(e.loss_init[1])
    assert abs(inc - ls.sum()) <= 1e-5 * ls.sum() + 1e-6, (inc, ls.sum())
    for i in (0, 2, 3):
        assert out["loss4"][i] == e.loss_init[i]


def test_ragged_equal_counts_match_equal_entry():
    """Equal counts: the ragged entry runs the units of forward_backward_mse with per-task weights."""
    from siren_mri_b200 import _lib
    T, n, d, nh, o = 5, 3000, 2, 3, 2
    e = _Ragged([n] * T, d, nh, o, seed=410)
    out = e.call(e.workspace(0))
    desc = e.make_desc()
    desc.n_coords = n
    ws = torch.zeros(e.lib.siren_b200_workspace_bytes_ex(desc, 0), dtype=torch.uint8, device="cuda")
    y = torch.empty(T, n, o, device="cuda")
    gy = torch.empty_like(y)
    loss4 = torch.zeros(4, device="cuda")
    grads = [torch.zeros(a.shape, device="cuda") for a in e.Ws + e.bs]
    nl = len(e.Ws)
    P = _lib.dptr
    _lib.check(e.lib.siren_b200_forward_backward_mse(
        desc, P(e.xd), _lib.ptr_array(e.Wd), _lib.ptr_array(e.bd), P(y), P(e.gtd), W_MSE, P(gy), P(loss4), P(ws), 0,
        _lib.ptr_array(grads[:nl]), _lib.ptr_array(grads[nl:]), 0, torch.cuda.current_stream().cuda_stream),
        "forward_backward_mse")
    torch.cuda.synchronize()
    assert np.array_equal(out["y"].view(np.uint32), y.cpu().numpy().reshape(-1, o).view(np.uint32))
    assert np.array_equal(out["gy"].view(np.uint32), gy.cpu().numpy().reshape(-1, o).view(np.uint32))
    errs = e.grad_errs(out["g"], [g.cpu().numpy() for g in grads])
    assert max(errs.values()) < 1e-5, errs
    scene_losses = out["task_loss"][T:].astype(np.float64)
    assert abs(scene_losses.sum() - float(loss4[1])) <= 1e-5 * float(loss4[1])
    assert abs(float(out["loss4"][1]) - e.loss_init[1] - float(loss4[1])) <= 1e-5 * float(loss4[1])


def test_ragged_robustness():
    """accumulate 0 / 1, gy = NULL, run to run, and a scene whose parameters change moves only its own gradients."""
    counts = [700, 1, 5000, 129]
    e = _Ragged(counts, 2, 2, 1, seed=500)
    ws = e.workspace(0xFF)
    a = e.call(ws)
    b = e.call(ws)                                   # run to run
    assert np.array_equal(a["y"].view(np.uint32), b["y"].view(np.uint32))
    assert max(e.grad_errs(b["g"], a["g"]).values()) < 1e-5
    c = e.call(ws, gy=False)                         # gy = NULL: same y and gradients
    assert np.array_equal(a["y"].view(np.uint32), c["y"].view(np.uint32))
    assert max(e.grad_errs(c["g"], a["g"]).values()) < 1e-5
    acc = e.call(ws, accumulate=1, grads=a["g"])    # adds to what is there
    assert max(e.grad_errs(acc["g"], [2 * g for g in a["g"]]).values()) < 1e-5
    # scene 2's hidden and outermost weights reloaded: its gradients change, the others' do not
    Wd = [w.clone() for w in e.Wd]
    for l in (1, len(Wd) - 1):
        Wd[l][2].mul_(0.5)
    r = e.call(ws, Wd=Wd)
    for i, (x, ref) in enumerate(zip(r["g"], a["g"])):
        for t in range(e.T):
            err = rel_l2(x[t], ref[t])
            assert (t == 2 and (i != 1 or err > 1e-3)) or err < 1e-5, (i, t, err)


@pytest.mark.parametrize("what,rc", [("count0", 2), ("count_neg", 2), ("shared", 2), ("fp32", 1), ("d_in5", 1),
                                     ("d_out3", 1), ("hidden5", 1), ("tasks1025", 1)])
def test_ragged_refusals(what, rc):
    from siren_mri_b200 import _lib
    counts, d, nh, o, prec = [100, 200], 2, 2, 1, "bf16"
    if what == "count0":
        counts = [100, 0]
    if what == "count_neg":
        counts = [-5, 100]
    d = 5 if what == "d_in5" else d
    o = 3 if what == "d_out3" else o
    nh = 5 if what == "hidden5" else nh
    prec = "fp32" if what == "fp32" else prec
    if what == "tasks1025":
        counts = [10] * 1025
    e = _Ragged.__new__(_Ragged)
    e.counts, e.d, e.nh, e.o, e.T = counts, d, nh, o, len(counts)
    desc = e.make_desc(prec)
    if what == "shared":
        desc.per_task = 0
    lib = _lib.load()
    n_c = _lib.long_array(counts)
    assert lib.siren_b200_workspace_bytes_ragged(desc, n_c) == 0
    ws = torch.zeros(1 << 20, dtype=torch.uint8, device="cuda")
    assert lib.siren_b200_prepare_ragged(desc, n_c, ws.data_ptr(), None) == rc
    dummy = torch.zeros(16, device="cuda")
    ptrs = _lib.ptr_array([dummy] * (nh + 2))
    got = lib.siren_b200_forward_backward_mse_ragged(desc, n_c, dummy.data_ptr(), ptrs, ptrs, dummy.data_ptr(),
                                                      dummy.data_ptr(), W_MSE, None, None, dummy.data_ptr(),
                                                      ws.data_ptr(), 0, ptrs, ptrs, 1, None)
    assert got == rc, lib.siren_b200_last_error()


# ---------------- the trainer ----------------

def _models(T, nh, d, o, seed):
    from siren_mri_b200 import modules
    torch.manual_seed(seed)
    return [modules.SingleBVPNet(in_features=d, out_features=o, num_hidden_layers=nh, precision="bf16").cuda()
            for _ in range(T)]


@pytest.mark.parametrize("clip,accum,graph", [(0.0, 1, True), (1e-3, 1, True), (0.0, 2, True), (1e-3, 2, False)])
def test_ragged_trainer_matches_single_scene_trainers(clip, accum, graph):
    from siren_mri_b200.trainer import SirenTrainer
    counts, d, nh, o = [1000, 257, 4096, 1], 2, 3, 1
    T = len(counts)
    models = _models(T, nh, d, o, seed=3)
    states = [{k: v.clone() for k, v in m.state_dict().items()} for m in models]
    rng = np.random.default_rng(4)
    xs = [torch.from_numpy(rng.uniform(-1, 1, (n, d)).astype(np.float32)) for n in counts]
    gts = [torch.from_numpy(rng.uniform(-1, 1, (n, o)).astype(np.float32)) for n in counts]
    tr = SirenTrainer(models, counts, lr=1e-4, max_grad_norm=clip, use_graph=graph)
    assert tr.kernels_per_step == 3 + (1 if clip else 0)
    singles = []
    for t in range(T):
        m = _models(1, nh, d, o, seed=100 + t)[0]
        m.load_state_dict(states[t])
        s = SirenTrainer(m, counts[t], lr=1e-4, max_grad_norm=clip, use_graph=graph)
        s.coords.copy_(xs[t].view(1, -1, d))
        s.gt.copy_(gts[t].view(1, -1, o))
        singles.append(s)
    for t in range(T):
        cx, cg, _ = tr.scene(t)
        cx.copy_(xs[t])
        cg.copy_(gts[t])
    # gradients and losses at the initial weights
    g, loss = tr.gradients()
    for t, s in enumerate(singles):
        gs, ls = s.gradients()
        assert np.array_equal(tr.scene(t)[2].cpu().numpy().view(np.uint32), s.y[0].cpu().numpy().view(np.uint32))
        for stk, prm in zip(tr.weights + tr.biases, s.weights + s.biases):
            off = prm.data_ptr() - s.flat.data_ptr()
            mine = g[(stk[t].data_ptr() - tr.flat.data_ptr()) // 4:][:prm.numel()]
            assert rel_l2(mine.cpu().numpy(), gs[off // 4:off // 4 + prm.numel()].cpu().numpy()) < 1e-5
        assert abs(float(loss[t]) - float(ls)) <= 1e-5 * float(ls)
    # five optimizer steps (each of accum micro-batches): the weights move alike
    for _ in range(5):
        for k in range(accum):
            up = k == accum - 1
            tr.step(update=up, accumulation_steps=accum)
            for s in singles:
                s.step(update=up, accumulation_steps=accum)
    torch.cuda.synchronize()
    # Adam normalises every element's step: where a gradient element is near zero, a summation-order difference in it
    # moves that element by up to lr (as in test_gpu_fused_step.py's training comparison)
    init = [[st[k] for k in sorted(st) if k.endswith("weight")] for st in states]
    for t, s in enumerate(singles):
        for l, (stk, prm) in enumerate(zip(tr.weights, s.weights)):
            mine, ref, w0 = (a.detach().cpu().numpy() for a in (stk[t], prm, init[t][l]))
            assert rel_l2(mine - w0, ref - w0) < 5e-3, (t, l, rel_l2(mine - w0, ref - w0))
            assert rel_l2(mine, ref) < 5e-4, (t, l, rel_l2(mine, ref))
        assert abs(float(tr.loss[t]) - float(s.loss[0])) <= 2e-4 * float(s.loss[0])


def test_ragged_trainer_host_batches():
    """step_from_host / submit_from_host take a packed tensor or the scenes' list; bad lists are refused."""
    from siren_mri_b200.trainer import SirenTrainer
    counts, d, o = [300, 50, 129], 2, 1
    tr = SirenTrainer(_models(3, 3, d, o, seed=5), counts, lr=1e-4)
    assert tr.coords.shape == (sum(counts), d) and tr.y.shape == (sum(counts), o)
    rng = np.random.default_rng(6)
    xs = [torch.from_numpy(rng.uniform(-1, 1, (n, d)).astype(np.float32)) for n in counts]
    gs = [torch.from_numpy(rng.uniform(-1, 1, (n, o)).astype(np.float32)) for n in counts]
    l_list = tr.step_from_host(xs, gs, update=False)
    l_pack = tr.step_from_host(torch.cat(xs), {"img": torch.cat(gs)}, update=False)
    assert len(l_list) == 3 and l_list == l_pack and all(v > 0 for v in l_list)
    assert torch.equal(tr.coords.cpu(), torch.cat(xs))
    h = tr.submit_from_host(xs, gs, update=False)
    assert h.result() == l_list
    with pytest.raises(ValueError):
        tr.step_from_host(xs[:2], gs)
    with pytest.raises(ValueError):
        SirenTrainer(_models(2, 3, 5, o, seed=5), [10, 20])          # d_in 5: outside the ragged step
