"""The one-kernel bf16 training step (forward, loss gradient and input-gradient chain: mlp_fused_step.cu) against the
two-launch step it replaces (SIREN_FUSED_STEP=0: mlp_fused_fwd + mlp_fused_bwd) on the same seeded inputs.

Both run the same arithmetic in the same order, so y and gy are bit-equal; the loss sum, the bias / first-layer /
outermost gradients the chain sums per warp and every weight gradient's atomics differ only in summation order.

The second half drives the C entry siren_b200_forward_backward_mse directly, at the multi-task / per-task shapes the
trainer never reaches, against the fp64 oracle, the two launches, itself (workspace contents, entry arguments, run to
run) and NaN guards behind every output buffer."""
import numpy as np
import pytest
import torch

from oracle import siren_oracle as so
from tests.helpers import log_errors, oracle_chunked, rel_l2, rel_l2_per_task

pytestmark = pytest.mark.gpu


def _trainer(monkeypatch, fused, n, nh, d_in, d_out, seed, **kw):
    from siren_mri_b200 import modules
    from siren_mri_b200.trainer import SirenTrainer
    monkeypatch.setenv("SIREN_FUSED_STEP", "1" if fused else "0")
    Ws, bs = so.make_params(d_in, 256, nh, d_out, seed=seed)
    m = modules.SingleBVPNet(in_features=d_in, out_features=d_out, num_hidden_layers=nh, precision="bf16").cuda()
    with torch.no_grad():
        for l in range(nh + 2):
            m.net.net[l][0].weight.copy_(torch.from_numpy(Ws[l]))
            m.net.net[l][0].bias.copy_(torch.from_numpy(bs[l]))
    tr = SirenTrainer(m, n, lr=1e-4, precision="bf16", **kw)
    x = so.make_coords(1, n, d_in, seed=seed + 1)
    gt = np.random.default_rng(seed + 2).uniform(-1, 1, size=(1, n, d_out)).astype(np.float32)
    tr.coords.copy_(torch.from_numpy(x))
    tr.gt.copy_(torch.from_numpy(gt))
    return tr, m, Ws


def _views(tr, flat):
    out, off = [], 0
    for prm in tr.block.parameters():
        out.append(flat[off:off + prm.numel()].cpu().numpy())
        off += prm.numel()
    return out


@pytest.mark.parametrize("n,nh,d_in,d_out", [
    (262144, 3, 2, 1),            # cfg2: many units per CTA pair
    (1000, 3, 2, 1),              # ragged, one unit per pair
    (131372, 3, 2, 1),            # ragged, the last unit has a single tile
    (5000, 1, 1, 1),
    (5000, 2, 3, 2),
    (70000, 4, 4, 2),
    (70000, 4, 2, 2),
])
def test_fused_step_gradients_match_two_launch(monkeypatch, n, nh, d_in, d_out):
    res = {}
    for fused in (False, True):
        tr, _, _ = _trainer(monkeypatch, fused, n, nh, d_in, d_out, seed=40 + nh, use_graph=False)
        assert tr.kernels_per_step == (3 if fused else 4)
        g, loss = tr.gradients()
        torch.cuda.synchronize()
        res[fused] = (_views(tr, g), float(loss.item()), tr.y.clone())
    (g0, l0, y0), (g1, l1, y1) = res[False], res[True]
    assert torch.equal(y0, y1)
    assert abs(l1 - l0) <= 1e-6 * abs(l0)
    for i, (a, b) in enumerate(zip(g0, g1)):
        assert rel_l2(b, a) < 1e-5, (i, rel_l2(b, a))


def test_fused_step_writes_the_same_gy(monkeypatch):
    """The C entry with gy requested: the loss gradient it writes is the two-launch step's, bit for bit."""
    from siren_mri_b200 import _lib
    n = 3000
    out = {}
    for fused in (False, True):
        tr, _, _ = _trainer(monkeypatch, fused, n, 3, 2, 2, seed=60, use_graph=False)
        gy = torch.full_like(tr.y, float("nan"))
        stream = torch.cuda.current_stream().cuda_stream
        P = _lib.dptr
        _lib.check(tr.lib.siren_b200_forward_backward_mse(
            tr.desc, P(tr.coords), tr._w_ptrs, tr._b_ptrs, P(tr.y), P(tr.gt), tr.loss_weight, P(gy), P(tr.loss4),
            P(tr.ws), 1, tr._dw_ptrs, tr._db_ptrs, 1, stream), "forward_backward_mse")
        torch.cuda.synchronize()
        out[fused] = (gy, tr.grad.clone())
    assert torch.equal(out[False][0], out[True][0])
    assert rel_l2(out[True][1].cpu().numpy(), out[False][1].cpu().numpy()) < 1e-5


@pytest.mark.parametrize("graph,clip,accum", [(False, 0, 1), (True, 0, 1), (True, 1, 1), (True, 0, 2), (False, 1, 2)])
def test_fused_step_training_matches_two_launch(monkeypatch, graph, clip, accum):
    n = 20000
    got = {}
    for fused in (False, True):
        tr, m, Ws = _trainer(monkeypatch, fused, n, 3, 2, 1, seed=80, use_graph=graph, max_grad_norm=0.5 * clip)
        while tr.steps < 10:
            for k in range(accum):
                tr.step(update=k == accum - 1, accumulation_steps=accum)
        torch.cuda.synchronize()
        got[fused] = ([m.net.net[l][0].weight.detach().cpu().numpy() for l in range(5)], float(tr.loss.item()))
    # Adam normalises every element's step: where a gradient element is near zero, a summation-order difference in it
    # moves that element by up to lr (most visible in the 512-element first layer)
    errs = [rel_l2(got[True][0][l] - Ws[l], got[False][0][l] - Ws[l]) for l in range(5)]
    assert max(errs) < 5e-3, errs
    assert abs(got[True][1] - got[False][1]) <= 1e-5 * abs(got[False][1])


@pytest.mark.parametrize("nh,d_in,d_out,clip", [
    (3, 2, 1, 0),                 # cfg2: the one-kernel step
    (5, 2, 1, 0),                 # two launches and two weight-gradient launches
    (8, 2, 1, 1),                 # the deepest net, with clipping
    (5, 16, 3, 0),                # first layer on the tensor core, outermost linear as kernels of its own
])
def test_kernels_per_step_is_what_the_library_launches(monkeypatch, nh, d_in, d_out, clip):
    """SirenTrainer.kernels_per_step against the launches the library's profile records over ten steps, counted as
    bench.py counts them."""
    import ctypes
    tr, _, _ = _trainer(monkeypatch, True, 5000, nh, d_in, d_out, seed=90 + nh, use_graph=False,
                        max_grad_norm=0.5 * clip)
    tr.step()
    torch.cuda.synchronize()
    steps = 10
    tr.lib.siren_b200_profile_begin()
    for _ in range(steps):
        tr.step()
    torch.cuda.synchronize()
    buf = ctypes.create_string_buffer(1 << 16)
    tr.lib.siren_b200_profile_end(buf, len(buf))
    table = {}
    for ln in buf.value.decode().strip().splitlines():
        name, cnt, _ = ln.split()
        table[name] = int(cnt)
    # one entry per launch site; the "adam" and "clip_grad" sites launch two kernels each
    launches = sum(table.values()) + table.get("adam", 0) + table.get("clip_grad", 0)
    assert launches == steps * tr.kernels_per_step, (tr.kernels_per_step, table)


# ---------------------------------------------------------------------------------------------------------------------
# The C entry siren_b200_forward_backward_mse at the shapes only it reaches: several tasks, per-task weights, gy handed
# back or not, accumulate = 0, weights_ready = 0, and a workspace holding someone else's planes.  (SirenTrainer always
# runs one task, shared weights, accumulate = 1, weights_ready = 1 and gy = NULL.)
#
# Bounds against the fp64 oracle (image_mse at the entry's weight 1/16384):
#   y, gy   rel-L2 < 2e-2 and, per element, max|d| / rms(ref) < 3e-2.  A CPU emulation of the fp16 forward gives rel-L2
#           1.0-1.5e-3 and max|d| / rms 5-7e-3 at 20-40k rows; one wrong row scores about 1.
#   dW, db  rel-L2 < 2e-2 up to four hidden layers, 3e-2 above (DESIGN.md section 4); per task with per-task weights.
# Measured on an NVIDIA B200, largest over the cases below (one kernel and two launches give the same numbers):
#   y rel-L2 7.7e-4 (8.6e-4 on the fallback shapes), max|d| / rms 3.2e-3 (3.4e-3); gy 6.5e-5, max|d| / rms 2.8e-4;
#   gradients 1.29e-2 (pertask_8x16384_d4 dW0; five hidden layers: 1.27e-2 against 3e-2).
#   One kernel against two launches: y, gy bit-equal; loss 2.3e-7; gradients per task <= 3.8e-7 (bound 1e-5).
# ---------------------------------------------------------------------------------------------------------------------

W_MSE = 1.0 / 16384           # image_mse's weight (loss_functions.py), the one so.image_mse defaults to

STEP_CASES = {
    # name: d, n_hidden, o, tasks, per_task, n
    # n_pad = 384: each task's second tile is half valid, and its invalid half overlaps the next task's first rows
    "shared_3x300": (2, 3, 1, 3, False, 300),
    # ragged tail per task, two outputs: y / gt / gy indexed per task
    "shared_5x1000_o2": (3, 2, 2, 5, False, 1000),
    # 2.5 pair tiles per task: each task ends in a single-tile unit, the task index moves between the tiles of a pair
    "pertask_3x640": (3, 3, 1, 3, True, 640),
    # the regime case: a pair walks 5-6 units across task boundaries, each task ends in a single half-valid tile
    "pertask_40x4700": (3, 3, 2, 40, True, 4700),
    # deepest and widest step shape, per task
    "pertask_8x16384_d4": (4, 4, 2, 8, True, 16384),
    # every unit is a different task: a flush after every unit, single-tile units only
    "pertask_200x128": (1, 1, 1, 200, True, 128),
    # one valid row per task
    "pertask_2x1": (2, 3, 1, 2, True, 1),
}
# shapes the one kernel does not take: the entry makes its two calls, and with gy = NULL hands gy over through the
# workspace's scratch plane
FALLBACK_CASES = {
    "fallback_d7_pertask": (7, 3, 1, 3, True, 900),       # first layer on the tensor core
    "fallback_nh5_o3": (2, 5, 3, 2, False, 700),          # five hidden layers, outermost linear as its own kernel
}
CASES = dict(STEP_CASES, **FALLBACK_CASES)


def _grad_tol(nh):
    return 2e-2 if nh <= 4 else 3e-2


def _inputs(case, seed):
    d, nh, o, tasks, per_task, n = CASES[case]
    Ws, bs = so.make_params(d, 256, nh, o, seed=seed, tasks=tasks if per_task else 0)
    x = so.make_coords(tasks, n, d, seed=seed + 1)
    gt = np.random.default_rng(seed + 2).uniform(-1, 1, size=(tasks, n, o)).astype(np.float32)
    return Ws, bs, x, gt


class _Entry:
    """siren_b200_forward_backward_mse through ctypes on device copies of one case's inputs.  Every buffer the entry
    writes (y, gy, each dW / db) is the view of a larger buffer whose tail, one task more, holds NaN: a write past the
    view shows there."""

    def __init__(self, monkeypatch, case, seed):
        from siren_mri_b200 import _lib, functional as F
        self.case = case
        self.d, self.nh, self.o, self.T, self.per_task, self.n = CASES[case]
        self.Ws, self.bs, self.x, self.gt = _inputs(case, seed)
        self.monkeypatch = monkeypatch
        self.lib = _lib.load()
        self.xd = torch.from_numpy(self.x).cuda()
        self.gtd = torch.from_numpy(self.gt).cuda()
        self.Wd = [torch.from_numpy(w).cuda() for w in self.Ws]
        self.bd = [torch.from_numpy(b).cuda() for b in self.bs]
        self.desc = F._make_desc(self.xd, self.Wd, 30.0, "bf16", 0)
        assert self.desc.per_task == int(self.per_task) and self.desc.tasks == self.T
        self.nbytes = self.lib.siren_b200_workspace_bytes_ex(self.desc, 0)
        assert self.nbytes > 0
        self.w_ptrs = _lib.ptr_array(self.Wd)
        self.b_ptrs = _lib.ptr_array(self.bd)
        # loss4[1] starts near the expected sum, so that an entry overwriting instead of adding is off by ~100 %
        self.loss_init = np.array([3.0, W_MSE * self.T * self.n * self.o / 3.0, 5.0, 7.0], np.float32)

    def workspace(self, fill):
        ws = torch.empty(self.nbytes, dtype=torch.uint8, device="cuda")
        ws.fill_(fill)            # 0xFF: NaN in fp16, bf16 and fp32
        return ws

    def _guarded(self, shape, tasked, start=None):
        """(view, guard): view has `shape`; the guard behind it is one task's worth of NaN ([tasks, ...] buffers: one
        more task; a shared parameter: one more copy).  start: what the view holds before the call (NaN if None)."""
        if tasked:
            full = torch.full((shape[0] + 1,) + tuple(shape[1:]), float("nan"), device="cuda")
            view, guard = full[:shape[0]], full[shape[0]:]
        else:
            full = torch.full((2,) + tuple(shape), float("nan"), device="cuda")
            view, guard = full[0], full[1]
        if start is not None:
            view.copy_(torch.from_numpy(np.asarray(start, np.float32)))
        return view, guard

    def call(self, ws, fused=True, gy=True, accumulate=1, grads=None, weights_ready=0):
        """One entry call.  grads: the [dW..., db...] the gradient buffers start from; None: NaN with accumulate = 0,
        zero with accumulate = 1.  Returns y, gy, the gradients and loss4 as numpy arrays."""
        import ctypes
        from siren_mri_b200 import _lib
        self.monkeypatch.setenv("SIREN_FUSED_STEP", "1" if fused else "0")
        params = self.Ws + self.bs
        if grads is None:
            grads = [None if not accumulate else np.zeros(a.shape, np.float32) for a in params]
        y, y_guard = self._guarded((self.T, self.n, self.o), True)
        gyv, gy_guard = self._guarded((self.T, self.n, self.o), True) if gy else (None, None)
        gv = [self._guarded(a.shape, self.per_task, s) for a, s in zip(params, grads)]
        loss4 = torch.from_numpy(self.loss_init.copy()).cuda()
        nl = len(self.Ws)
        P = _lib.dptr
        torch.cuda.synchronize()
        self.lib.siren_b200_profile_begin()
        rc = self.lib.siren_b200_forward_backward_mse(
            self.desc, P(self.xd), self.w_ptrs, self.b_ptrs, P(y), P(self.gtd), W_MSE, P(gyv), P(loss4), P(ws),
            weights_ready, _lib.ptr_array([v for v, _ in gv[:nl]]), _lib.ptr_array([v for v, _ in gv[nl:]]),
            accumulate, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        buf = ctypes.create_string_buffer(1 << 14)
        self.lib.siren_b200_profile_end(buf, len(buf))
        _lib.check(rc, "forward_backward_mse")
        # the path the case is meant to test, not a quiet change of fused_step()
        names = [ln.split()[0] for ln in buf.value.decode().strip().splitlines()]
        if fused and self.case in STEP_CASES:
            assert "mlp_fused_step" in names and "mlp_fused_fwd" not in names and "mlp_fused_bwd" not in names, names
        else:
            assert "mlp_fused_step" not in names and "mlp_fused_fwd" in names, names
        # every write stayed inside the caller's views
        for what, guard in [("y", y_guard), ("gy", gy_guard)] + [("grad %d" % i, g) for i, (_, g) in enumerate(gv)]:
            assert guard is None or bool(torch.isnan(guard).all()), "write past the end of " + what
        return dict(y=y.cpu().numpy(), gy=None if gyv is None else gyv.cpu().numpy(), loss4=loss4.cpu().numpy(),
                    g=[v.cpu().numpy() for v, _ in gv])

    def grad_errs(self, got, ref):
        """{dW<l> / db<l>: rel-L2} of two [dW..., db...] lists, per task with per-task weights."""
        err = rel_l2_per_task if self.per_task else rel_l2
        nl = len(self.Ws)
        e = {}
        for l in range(nl):
            e["dW%d" % l] = err(got[l], ref[l])
            e["db%d" % l] = err(got[nl + l], ref[nl + l])
        return e


_ORACLE = {}


def _oracle(e):
    """fp64 y and gradients of a case's image_mse step (one entry: the variants of a case run back to back)."""
    key = (e.case, e.Ws[0].tobytes()[:64])
    if key not in _ORACLE:
        _ORACLE.clear()
        gt = e.gt

        def adj(t0, t1, n0, n1, yc, Jc, Dc):
            return so.image_mse(yc, gt[t0:t1, n0:n1].astype(np.float64), weight=W_MSE)[1], None, None
        yo, _, _, oW, ob = oracle_chunked(e.x, e.Ws, e.bs, adj)
        _ORACLE[key] = (yo, oW + ob)
    return _ORACLE[key]


def _max_rel(a, ref):
    """Largest per-element error over the reference's rms: one wrong row out of 10^5 scores ~1 here."""
    ref = np.asarray(ref, np.float64)
    return float(np.abs(np.asarray(a, np.float64) - ref).max() / max(np.sqrt((ref * ref).mean()), 1e-300))


def _assert_bits(a, b, what):
    assert a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32)), \
        (what, int((a.view(np.uint32) != b.view(np.uint32)).sum()))


def _assert_grads_close(e, got, ref, tol, what):
    errs = e.grad_errs(got, ref)
    bad = {k: v for k, v in errs.items() if not v < tol}
    assert not bad, (what, errs)
    return errs


FP64_RUNS = [(c, "step") for c in STEP_CASES] + [(c, "two_launch") for c in STEP_CASES] + \
            [(c, "entry") for c in FALLBACK_CASES]


@pytest.mark.parametrize("case,path", sorted(FP64_RUNS))
def test_step_against_fp64(monkeypatch, case, path):
    """One call on a workspace of 0xFF bytes with NaN gradient buffers and accumulate = 0, against fp64; gy and the
    loss exactly as the entry defines them from its own y; nothing written outside the caller's buffers."""
    e = _Entry(monkeypatch, case, seed=200)
    out = e.call(e.workspace(0xFF), fused=path != "two_launch", accumulate=0)
    yo, gref = _oracle(e)
    y, gy, gt = out["y"], out["gy"], e.gt
    gyo = 2.0 * W_MSE * (yo - gt.astype(np.float64))
    errs = {"y": rel_l2(y, yo), "y_max": _max_rel(y, yo), "gy": rel_l2(gy, gyo), "gy_max": _max_rel(gy, gyo)}
    errs.update(e.grad_errs(out["g"], gref))
    # The outermost bias gradient is the sum of a task's loss gradient, which can cancel almost to zero: in task 20 of
    # pertask_200x128, sum |gy| / |sum gy| = 1.1e4, and the one kernel, the two launches and fp64 differ there by
    # 2.2e-2 relative.  So it is held to fp64 over all tasks, and per task to the sum of the entry's OWN gy, to
    # summation rounding (1e-5 of sum |gy|): that still catches a sum flushed into the wrong task.
    nl = len(e.Ws)
    axes = 1 if e.per_task else (0, 1)
    gy64 = gy.astype(np.float64)
    errs["dbL_own"] = float((np.abs(out["g"][-1] - gy64.sum(axes)) / np.abs(gy64).sum(axes)).max())
    errs["db%d" % (nl - 1)] = rel_l2(out["g"][-1], gref[-1])
    log_errors("step_fp64/%s/%s" % (case, path), **errs)
    tol = _grad_tol(e.nh)
    bad = {k: v for k, v in errs.items()
           if not v < {"y": 2e-2, "gy": 2e-2, "y_max": 3e-2, "gy_max": 3e-2, "dbL_own": 1e-5}.get(k, tol)}
    assert not bad, (case, path, errs)
    # gy = 2 w (y - gt) in fp32 on the entry's own y, bit for bit (scaling by two is exact)
    _assert_bits(gy, (np.float32(2.0 * W_MSE) * (y - gt)).astype(np.float32), "gy")
    # loss4[1] += w sum (y - gt)^2; the other slots are not the entry's
    lsum = W_MSE * float(((y.astype(np.float64) - gt) ** 2).sum())
    inc = float(out["loss4"][1]) - float(e.loss_init[1])
    assert abs(inc - lsum) <= 1e-5 * lsum, (inc, lsum)
    for i in (0, 2, 3):
        assert out["loss4"][i] == e.loss_init[i], (i, out["loss4"])


@pytest.mark.parametrize("case", sorted(STEP_CASES))
def test_step_matches_two_launch_at_entry(monkeypatch, case):
    """The one kernel against the two launches it replaces, through the same entry on the same inputs: y and gy to
    the bit, the loss and every gradient (per task) to summation order."""
    e = _Entry(monkeypatch, case, seed=300)
    one = e.call(e.workspace(0), fused=True, accumulate=0)
    two = e.call(e.workspace(0), fused=False, accumulate=0)
    _assert_bits(one["y"], two["y"], "y")
    _assert_bits(one["gy"], two["gy"], "gy")
    l1, l2 = float(one["loss4"][1]), float(two["loss4"][1])
    assert abs(l1 - l2) <= 1e-6 * abs(l2), (l1, l2)
    errs = _assert_grads_close(e, one["g"], two["g"], 1e-5, "one kernel vs two launches")
    log_errors("step_vs_two_launch/%s" % case, loss=abs(l1 - l2) / abs(l2), **errs)


@pytest.mark.parametrize("case", sorted(CASES))
def test_step_ignores_workspace_contents(monkeypatch, case):
    """Results do not depend on what the workspace held: 0xFF bytes (NaN in every float format the planes use) or
    the planes of an earlier call on other inputs give what a zeroed workspace gives."""
    e = _Entry(monkeypatch, case, seed=400)
    ws = e.workspace(0xFF)
    a = e.call(ws)
    b = e.call(e.workspace(0))
    _assert_bits(a["y"], b["y"], "y")
    _assert_bits(a["gy"], b["gy"], "gy")
    _assert_grads_close(e, a["g"], b["g"], 1e-5, "0xFF workspace vs zeroed")
    # the same workspace again, now holding the planes of the call above, on new inputs (gy not handed back)
    e2 = _Entry(monkeypatch, case, seed=410)
    c = e2.call(ws, gy=False)
    d = e2.call(e2.workspace(0), gy=False)
    _assert_bits(c["y"], d["y"], "y")
    _assert_grads_close(e2, c["g"], d["g"], 1e-5, "reused workspace vs zeroed")
    assert abs(float(c["loss4"][1]) - float(d["loss4"][1])) <= 1e-6 * abs(float(d["loss4"][1]))


@pytest.mark.parametrize("case", sorted(CASES))
def test_step_entry_arguments(monkeypatch, case):
    """accumulate, a running gradient, weights_ready after prepare_weights and gy = NULL change nothing but what they
    are meant to."""
    e = _Entry(monkeypatch, case, seed=500)
    base = e.call(e.workspace(0), accumulate=1)                  # zeroed gradient buffers
    # accumulate = 0 clears NaN buffers before anything is added
    z = e.call(e.workspace(0), accumulate=0)
    _assert_bits(z["y"], base["y"], "y")
    _assert_grads_close(e, z["g"], base["g"], 1e-5, "accumulate = 0 on NaN vs 1 on zeros")
    # accumulate = 1 adds to what the buffers hold: a random G0 of the gradient's own scale
    rng = np.random.default_rng(7)
    g0 = [(rng.standard_normal(g.shape) * np.sqrt(np.mean(g.astype(np.float64) ** 2))).astype(np.float32)
          for g in base["g"]]
    acc = e.call(e.workspace(0), accumulate=1, grads=g0)
    _assert_grads_close(e, acc["g"], [a.astype(np.float64) + b for a, b in zip(g0, base["g"])], 1e-5, "G0 + grad")
    # weights converted by prepare_weights, then weights_ready = 1
    ws = e.workspace(0)
    stream = torch.cuda.current_stream().cuda_stream
    from siren_mri_b200 import _lib
    _lib.check(e.lib.siren_b200_prepare_weights(e.desc, e.w_ptrs, _lib.dptr(ws), stream), "prepare_weights")
    pre = e.call(ws, weights_ready=1)
    _assert_bits(pre["y"], base["y"], "y")
    _assert_bits(pre["gy"], base["gy"], "gy")
    _assert_grads_close(e, pre["g"], base["g"], 1e-5, "weights_ready = 1 after prepare_weights")
    # gy = NULL: the same y and gradients (off the one kernel, gy goes through the workspace's scratch plane)
    ng = e.call(e.workspace(0), gy=False)
    _assert_bits(ng["y"], base["y"], "y")
    _assert_grads_close(e, ng["g"], base["g"], 1e-5, "gy = NULL")
    assert abs(float(ng["loss4"][1]) - float(base["loss4"][1])) <= 1e-6 * abs(float(base["loss4"][1]))


@pytest.mark.parametrize("case", sorted(CASES))
def test_step_run_to_run(monkeypatch, case):
    """y and gy use no atomics: two calls on the same inputs give the same bits (exactly two calls)."""
    e = _Entry(monkeypatch, case, seed=600)
    ws = e.workspace(0)
    a = e.call(ws)
    b = e.call(ws)
    _assert_bits(a["y"], b["y"], "y")
    _assert_bits(a["gy"], b["gy"], "gy")
