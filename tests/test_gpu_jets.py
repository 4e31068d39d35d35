"""The coordinate-jet paths (deriv_order 1 and 2, d_in <= 3) through siren_b200_forward / siren_b200_backward against
the fp64 oracle, across their envelope: d = 1, 2, 3; one to eight hidden layers (two weight-gradient launches above
four); d_out = 1 to 8 (every OMAX of the staged last_bwd); several tasks with shared and per-task weights; one row;
rows that leave partial stages in the edge kernels.

The backward is checked one adjoint stream at a time (only gy, only gJ, only gD): in a combined call the streams arrive
at very different scales, and a dropped or mis-signed term of one of them can hide under the others' bound.  The fp64
reference is linear in the adjoints, so the combined call is held to the sum of the isolated references.

Also: the staged edge kernels (bulk copies into a shared-memory ring) against the register-only loops they replace
(SIREN_EDGE_STAGED=0), NaN bands behind every output buffer, accumulate, the workspace's stash surviving a backward,
and the refusals of the entries."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import siren_oracle as so
from tests.helpers import log_errors, rel_l2, rel_l2_per_task

pytestmark = pytest.mark.gpu

W0 = 30.0

CASES = {
    # name: d, order, n_hidden, d_out, tasks, per_task, n
    # On a 148-SM B200 (edge_grid): one row, so most edge blocks have an empty range; S = 2
    "d1_j1_n1": (1, 1, 1, 1, 1, False, 1),
    # S = 3 with d = 1, OMAX 2, a one-row partial stage
    "d1_j2_o2": (1, 2, 3, 2, 1, False, 4097),
    # d = 1 per task, OMAX 4, one full weight-gradient group
    "d1_j1_o4_pt": (1, 1, 4, 4, 9, True, 700),
    # shared weights over several tasks
    "d2_j1_o3_t3": (2, 1, 2, 3, 3, False, 1000),
    # S = 5, two-stage rings, two weight-gradient launches
    "d2_j2_deep5": (2, 2, 5, 1, 1, False, 20000),
    # ~111 rows per edge block: partial 15-row and 7-row stages
    "d2_j1_tails": (2, 1, 3, 1, 1, False, 131149),
    # OMAX 8, per-task weights in the staged kernels
    "d3_j1_o8_pt": (3, 1, 3, 8, 7, True, 3000),
    # S = 7, 14 planes per row, OMAX 8
    "d3_j2_o5_pt": (3, 2, 2, 5, 4, True, 2500),
    # the deepest net: two weight-gradient launches with S = 7
    "d3_j2_deep8": (3, 2, 8, 2, 1, False, 5000),
}
RUNS = [(c, p) for c in CASES for p in ("bf16", "fp32")]

# Bounds, per metric: '_l2' is rel-L2 (per task where there are several), '_max' is max|d| / rms(ref) per element (per
# (task, output, k) stream for y, J, D and gcoords; per tensor for dW, db).  fp32-parity: the suite's 1e-4 for rel-L2,
# 1.5e-4 for the hidden-layer dW of the second-order reverse (DESIGN.md section 4), 1e-3 per element.  bf16: about
# 2-3x the largest value measured on a B200 over the cases above, rel-L2 at most 3e-2; nets with more than four hidden
# layers compound the stash rounding further and have their own column (DESIGN.md section 5).
FP32 = {"l2": 1e-4, "max": 1e-3}
FP32_HIDDEN_J2 = 1.5e-4
BF16 = {  # metric: (up to four hidden layers, five to eight)
    "y_l2": (1.5e-2, 1.5e-2), "y_max": (8e-2, 5e-2),
    "J_l2": (2.5e-2, 3e-2), "J_max": (0.1, 0.2),
    "D_l2": (2e-2, 3e-2), "D_max": (8e-2, 0.3),
    "dW_l2": (3e-2, 3e-2), "dW_max": (0.15, 0.25),
    "db_l2": (3e-2, 3e-2), "db_max": (0.1, 0.2),
    "gx_l2": (3e-2, 3e-2), "gx_max": (0.25, 0.3),
}


def _bound(prec, key, order, n_hidden):
    """key: '<stream>:<name>_<kind>' (backward) or '<name>_<kind>' (forward)."""
    name, kind = key.split(":")[-1].rsplit("_", 1)
    if prec == "fp32":
        hidden_dw = name.startswith("dW") and 1 <= int(name[2:]) <= n_hidden
        return FP32_HIDDEN_J2 if (order == 2 and hidden_dw and kind == "l2") else FP32[kind]
    base = "dW" if name.startswith("dW") else "db" if name.startswith("db") else name
    return BF16["%s_%s" % (base, kind)][1 if n_hidden > 4 else 0]


def _max_rel(a, ref, axes=None):
    """Largest |a - ref| over rms(ref); with `axes`, per slice along the other axes (the worst slice counts)."""
    a = np.asarray(a, np.float64)
    ref = np.asarray(ref, np.float64)
    err = np.abs(a - ref)
    if axes is None:
        return float(err.max() / max(np.sqrt((ref * ref).mean()), 1e-300))
    rms = np.sqrt((ref * ref).mean(axis=axes))
    return float((err.max(axis=axes) / np.maximum(rms, 1e-300)).max())


def _bits_equal(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


class _Jets:
    """siren_b200_forward / siren_b200_backward through ctypes on device copies of one case's seeded inputs.  Every
    buffer the entries write is the view of a larger buffer whose tail (one task more; one copy more for a shared
    parameter) holds NaN, and that tail is checked after every call."""

    def __init__(self, case, prec, seed=900):
        from siren_mri_b200 import _lib, functional as F
        self.case, self.prec = case, prec
        self.d, self.order, self.nh, self.o, self.T, self.per_task, self.n = CASES[case]
        self.Ws, self.bs = so.make_params(self.d, 256, self.nh, self.o, seed=seed,
                                          tasks=self.T if self.per_task else 0)
        self.x = so.make_coords(self.T, self.n, self.d, seed=seed + 1)
        rng = np.random.default_rng(seed + 2)
        T, n, o, d = self.T, self.n, self.o, self.d
        # the scales of the configurations' losses: J carries a factor w0, D a factor w0^2 over y
        self.gy = (rng.standard_normal((T, n, o)) / n).astype(np.float32)
        self.gJ = (rng.standard_normal((T, n, o, d)) / (W0 * n)).astype(np.float32)
        self.gD = (rng.standard_normal((T, n, o, d)) / (W0 * W0 * n)).astype(np.float32) if self.order == 2 else None
        self.lib = _lib.load()
        self.xd = torch.from_numpy(self.x).cuda()
        self.Wd = [torch.from_numpy(w).cuda() for w in self.Ws]
        self.bd = [torch.from_numpy(b).cuda() for b in self.bs]
        self.desc = F._make_desc(self.xd, self.Wd, W0, prec, self.order)
        assert self.desc.per_task == int(self.per_task) and self.desc.tasks == T
        self.nbytes = self.lib.siren_b200_workspace_bytes(self.desc)
        assert self.nbytes > 0
        self.w_ptrs = _lib.ptr_array(self.Wd)
        self.b_ptrs = _lib.ptr_array(self.bd)

    def workspace(self):
        ws = torch.empty(self.nbytes, dtype=torch.uint8, device="cuda")
        ws.fill_(0xFF)            # NaN in every float format the planes use
        return ws

    @staticmethod
    def _guarded(shape, tasked, start=None):
        if tasked:
            full = torch.full((shape[0] + 1,) + tuple(shape[1:]), float("nan"), device="cuda")
            view, guard = full[:shape[0]], full[shape[0]:]
        else:
            full = torch.full((2,) + tuple(shape), float("nan"), device="cuda")
            view, guard = full[0], full[1]
        if start is not None:
            view.copy_(torch.from_numpy(np.asarray(start, np.float32)))
        return view, guard

    @staticmethod
    def _check_guards(guards):
        torch.cuda.synchronize()
        for what, g in guards:
            assert g is None or bool(torch.isnan(g).all()), "write past the end of " + what

    def forward(self, ws):
        from siren_mri_b200 import _lib
        T, n, o, d = self.T, self.n, self.o, self.d
        y, yg = self._guarded((T, n, o), True)
        J, Jg = self._guarded((T, n, o, d), True)
        D, Dg = self._guarded((T, n, o, d), True) if self.order == 2 else (None, None)
        P = _lib.dptr
        _lib.check(self.lib.siren_b200_forward(self.desc, P(self.xd), self.w_ptrs, self.b_ptrs, P(y), P(J), P(D),
                                               P(ws), torch.cuda.current_stream().cuda_stream), "forward")
        self._check_guards([("y", yg), ("J", Jg), ("D", Dg)])
        return dict(y=y.cpu().numpy(), J=J.cpu().numpy(), D=None if D is None else D.cpu().numpy())

    def backward(self, ws, gy, gJ=None, gD=None, accumulate=0, grads=None, gcoords=True):
        """One backward call on `ws` (holding a forward's stash).  grads: what the gradient buffers start from (None:
        NaN).  Returns the [dW..., db...] list and gcoords as numpy arrays."""
        from siren_mri_b200 import _lib
        params = self.Ws + self.bs
        if grads is None:
            grads = [None] * len(params)
        gv = [self._guarded(a.shape, self.per_task, s) for a, s in zip(params, grads)]
        gx, gxg = self._guarded((self.T, self.n, self.d), True) if gcoords else (None, None)
        dev = [None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (gy, gJ, gD)]
        nl = len(self.Ws)
        P = _lib.dptr
        _lib.check(self.lib.siren_b200_backward(
            self.desc, P(self.xd), self.w_ptrs, self.b_ptrs, P(ws), P(dev[0]), P(dev[1]), P(dev[2]),
            _lib.ptr_array([v for v, _ in gv[:nl]]), _lib.ptr_array([v for v, _ in gv[nl:]]), P(gx), accumulate,
            torch.cuda.current_stream().cuda_stream), "backward")
        self._check_guards([("gcoords", gxg)] + [("grad %d" % i, g) for i, (_, g) in enumerate(gv)])
        return [v.cpu().numpy() for v, _ in gv], None if gx is None else gx.cpu().numpy()

    def streams(self):
        """The isolated adjoint streams: (name, gy, gJ, gD).  gy cannot be NULL, so it is passed as zeros."""
        zy = np.zeros_like(self.gy)
        out = [("gy", self.gy, None, None), ("gJ", zy, self.gJ, None)]
        if self.order == 2:
            out.append(("gD", zy, None, self.gD))
        return out

    def grad_names(self):
        nl = len(self.Ws)
        return ["dW%d" % l for l in range(nl)] + ["db%d" % l for l in range(nl)]


# ---------------------------------------------------------------------------------------------------------------------
# fp64 oracle: rows are independent, so each task is walked in chunks; the forward of a chunk is shared by the
# backward of every isolated adjoint stream.  One case is kept at a time (the tests of a case run back to back).
# ---------------------------------------------------------------------------------------------------------------------
_ORACLE = {}


def _oracle(e, chunk=16384):
    if e.case in _ORACLE:
        return _ORACLE[e.case]
    _ORACLE.clear()
    T, n, o, d = e.T, e.n, e.o, e.d
    W64 = [np.asarray(w, np.float64) for w in e.Ws]
    b64 = [np.asarray(b, np.float64) for b in e.bs]
    y = np.empty((T, n, o))
    J = np.empty((T, n, o, d))
    D = np.empty((T, n, o, d)) if e.order == 2 else None
    names = [s[0] for s in e.streams()]
    g = {s: [np.zeros_like(a) for a in W64 + b64] for s in names}
    gx = {s: np.empty((T, n, d)) for s in names}
    nl = len(W64)
    for t in range(T):
        Wt = [w[t:t + 1] for w in W64] if e.per_task else W64
        bt = [b[t:t + 1] for b in b64] if e.per_task else b64
        for n0 in range(0, n, chunk):
            n1 = min(n, n0 + chunk)
            yc, Jc, Dc, cache = so.siren_forward(e.x[t:t + 1, n0:n1].astype(np.float64), Wt, bt, W0, e.order)
            y[t, n0:n1], J[t, n0:n1] = yc[0], Jc[0]
            if e.order == 2:
                D[t, n0:n1] = Dc[0]
            for s, gy, gJ, gD in e.streams():
                cut = [None if a is None else a[t:t + 1, n0:n1].astype(np.float64) for a in (gy, gJ, gD)]
                dW, db, gxc = so.siren_backward(cache, Wt, *cut)
                gx[s][t, n0:n1] = gxc[0]
                for l in range(nl):
                    for i, a in ((l, dW[l]), (nl + l, db[l])):
                        if e.per_task:
                            g[s][i][t:t + 1] += a
                        else:
                            g[s][i] += a
    _ORACLE[e.case] = (y, J, D, g, gx)
    return _ORACLE[e.case]


def _grad_errs(e, got, ref, gx, gx_ref, prefix):
    errs = {}
    l2 = rel_l2_per_task if e.per_task else rel_l2
    for name, a, r in zip(e.grad_names(), got, ref):
        if not np.any(r):
            continue          # an exactly-zero reference (the outermost bias without gy) is checked for exact zeros
        errs["%s:%s_l2" % (prefix, name)] = l2(a, r)
        errs["%s:%s_max" % (prefix, name)] = _max_rel(a, r)
    errs["%s:gx_l2" % prefix] = rel_l2_per_task(gx, gx_ref)
    errs["%s:gx_max" % prefix] = _max_rel(gx, gx_ref, axes=1)
    return errs


def _same_grads(e, got, ref, start=None):
    """{name: error} of a kernel result against another kernel result: rel-L2 (per task with per-task weights) for every
    gradient but the outermost bias.  That one is a sum of gy, which cancels (sum |gy| / |sum gy| is about sqrt(n) for
    these adjoints), so it is held per (task, output) to the size of its terms: |d| / (sum |gy| + |start|)."""
    l2 = rel_l2_per_task if e.per_task else rel_l2
    names = e.grad_names()
    errs = {k: l2(a, b) for k, a, b in zip(names[:-1], got[:-1], ref[:-1])}
    terms = np.abs(e.gy.astype(np.float64)).sum(axis=1 if e.per_task else (0, 1))
    if start is not None:
        terms = terms + np.abs(start[-1])
    errs[names[-1]] = float((np.abs(got[-1].astype(np.float64) - ref[-1]) / terms).max())
    return errs


def _same_tol(e, key):
    """Bound of a _same_grads error.  Two results that differ in the order of their atomics: 1e-6 for the hidden layers
    (measured <= 3e-7).  The first and outermost layers' dW and db_0 are sums over every row that end in one atomic per
    block and element, and cancel: two identical calls at 131,149 rows measured 9.7e-7 (dW_L) and 7.1e-7 (db_0), so
    these, and a sum with a running gradient (one more rounding), are held to 1e-5."""
    last = len(e.Ws) - 1
    edge = ("dW0", "db0", "dW%d" % last)
    return 1e-5 if key.startswith("acc:") or key.split(":")[-1] in edge else 1e-6


@pytest.mark.parametrize("case,prec", RUNS)
def test_jets_against_fp64(case, prec):
    """Forward (y, J, D) per element and per task, then the backward one adjoint stream at a time and combined, every
    call into NaN-filled gradient buffers with accumulate = 0 on a workspace of 0xFF bytes."""
    e = _Jets(case, prec)
    ws = e.workspace()
    out = e.forward(ws)
    yo, Jo, Do, gref, gxref = _oracle(e)
    errs = {}
    for name, a, r in (("y", out["y"], yo), ("J", out["J"], Jo), ("D", out["D"], Do)):
        if r is None:
            continue
        assert np.isfinite(a).all(), name
        errs[name + "_l2"] = rel_l2_per_task(a, r)
        errs[name + "_max"] = _max_rel(a, r, axes=1)          # each (task, output, k) stream over its rows
    nl = len(e.Ws)
    for s, gy, gJ, gD in e.streams():
        g, gx = e.backward(ws, gy, gJ, gD)
        assert all(np.isfinite(a).all() for a in g) and np.isfinite(gx).all(), s
        if s != "gy":
            # the outermost bias gradient is the sum of gy alone
            assert not np.any(g[2 * nl - 1]), (s, g[2 * nl - 1])
        errs.update(_grad_errs(e, g, gref[s], gx, gxref[s], s))
    g, gx = e.backward(ws, e.gy, e.gJ, e.gD)
    streams = [s[0] for s in e.streams()]
    gsum = [sum(gref[s][i] for s in streams) for i in range(2 * nl)]
    errs.update(_grad_errs(e, g, gsum, gx, sum(gxref[s] for s in streams), "all"))
    log_errors("jets_fp64/%s/%s" % (case, prec), **errs)
    bad = {k: v for k, v in errs.items() if not v < _bound(prec, k, e.order, e.nh)}
    assert not bad, (case, prec, bad)


def _kernel_names(fn, tmpdir):
    """Names of the CUDA kernels fn() launches, from a torch.profiler trace."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    path = os.path.join(str(tmpdir), "trace.json")
    prof.export_chrome_trace(path)
    with open(path) as f:
        ev = json.load(f)["traceEvents"]
    return res, {x["name"] for x in ev if x.get("cat") == "kernel"}


@pytest.mark.parametrize("case", list(CASES))
def test_staged_matches_register_loops(case, monkeypatch, tmp_path):
    """bf16 jet planes: the staged edge kernels against the register-only loops (SIREN_EDGE_STAGED=0), flipped within
    one process.  Both compute each row's outputs with the same arithmetic, and each thread's partial sums over the
    same rows in the same order, so y, J, D and gcoords are bit-equal; dW_L, db_L, dW_0 and db_0 end in one atomic
    per block and element, so they differ in the order of those atomics only."""
    e = _Jets(case, "bf16")
    omax = 1 if e.o <= 1 else 2 if e.o <= 2 else 4 if e.o <= 4 else 8
    staged = {"last_fwd_staged_kernel", "last_bwd_jets_staged_kernel<%d>" % omax,
              "first_bwd_jets_staged_kernel<%d>" % e.d}
    res = {}
    for arm in ("1", "0"):
        monkeypatch.setenv("SIREN_EDGE_STAGED", arm)
        ws = e.workspace()

        def run():
            f = e.forward(ws)
            g, gx = e.backward(ws, e.gy, e.gJ, e.gD)
            return f, g, gx
        res[arm], names = _kernel_names(run, tmp_path)
        hit = {k for k in staged if any(k in nm for nm in names)}
        if arm == "1":
            assert hit == staged, (sorted(staged - hit), sorted(names))
        else:
            assert not any("_staged_kernel" in nm for nm in names), sorted(names)
            assert any("last_bwd_kernel<" in nm for nm in names), sorted(names)
    (f1, g1, x1), (f0, g0, x0) = res["1"], res["0"]
    for k in ("y", "J", "D"):
        if f1[k] is not None:
            assert _bits_equal(f1[k], f0[k]), (k, int((f1[k].view(np.uint32) != f0[k].view(np.uint32)).sum()))
    assert _bits_equal(x1, x0), int((x1.view(np.uint32) != x0.view(np.uint32)).sum())
    errs = _same_grads(e, g1, g0)
    log_errors("jets_staged_vs_register/%s" % case, **errs)
    bad = {k: v for k, v in errs.items() if not v < _same_tol(e, k)}
    assert not bad, (case, bad)


@pytest.mark.parametrize("case,prec", RUNS)
def test_jets_entry_arguments(case, prec):
    """accumulate = 1 adds onto a running gradient; accumulate = 0 clears NaN buffers; a second backward on the same
    workspace gives the first one's result (the backward leaves the forward's stash intact); gcoords = NULL changes
    nothing else."""
    e = _Jets(case, prec)
    ws = e.workspace()
    e.forward(ws)
    base, gx = e.backward(ws, e.gy, e.gJ, e.gD)
    assert all(np.isfinite(a).all() for a in base) and np.isfinite(gx).all()
    errs = {}
    # the same call again on the same workspace
    again, gx2 = e.backward(ws, e.gy, e.gJ, e.gD)
    assert _bits_equal(gx, gx2)
    errs.update({"again:" + k: v for k, v in _same_grads(e, again, base).items()})
    # accumulate = 1 onto a random running gradient of the gradient's own scale
    rng = np.random.default_rng(11)
    g0 = [(rng.standard_normal(g.shape) * np.sqrt(np.mean(g.astype(np.float64) ** 2))).astype(np.float32)
          for g in base]
    acc, gx3 = e.backward(ws, e.gy, e.gJ, e.gD, accumulate=1, grads=g0)
    assert _bits_equal(gx, gx3)
    errs.update({"acc:" + k: v for k, v in
                 _same_grads(e, acc, [a.astype(np.float64) + b for a, b in zip(g0, base)], start=g0).items()})
    # no coordinate gradient asked for
    nog, _ = e.backward(ws, e.gy, e.gJ, e.gD, gcoords=False)
    errs.update({"nogx:" + k: v for k, v in _same_grads(e, nog, base).items()})
    log_errors("jets_args/%s/%s" % (case, prec), **errs)
    bad = {k: v for k, v in errs.items() if not v < _same_tol(e, k)}
    assert not bad, (case, prec, bad)


@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_jets_refusals(prec):
    """d_in = 4 with jets is outside the envelope (SIREN_ERR_UNSUPPORTED); deriv_order 3, and J = NULL with
    deriv_order >= 1, are bad arguments (SIREN_ERR_INVALID).  Nothing is written."""
    from siren_mri_b200 import _lib
    lib = _lib.load()
    P = _lib.dptr
    stream = torch.cuda.current_stream().cuda_stream
    e = _Jets("d2_j1_o3_t3", prec)
    ws = torch.zeros(e.nbytes, dtype=torch.uint8, device="cuda")
    y = torch.full((e.T, e.n, e.o), float("nan"), device="cuda")
    J = torch.full((e.T, e.n, e.o, 4), float("nan"), device="cuda")
    D = torch.full_like(J, float("nan"))
    gy = torch.zeros_like(y)
    dW = [torch.full_like(w, float("nan")) for w in e.Wd]
    db = [torch.full_like(b, float("nan")) for b in e.bd]

    def fwd(desc, Jp=J, Dp=D):
        return lib.siren_b200_forward(desc, P(e.xd), e.w_ptrs, e.b_ptrs, P(y), P(Jp), P(Dp), P(ws), stream)

    def bwd(desc):
        return lib.siren_b200_backward(desc, P(e.xd), e.w_ptrs, e.b_ptrs, P(ws), P(gy), None, None,
                                       _lib.ptr_array(dW), _lib.ptr_array(db), None, 0, stream)

    def desc_with(**kw):
        dsc = _lib.SirenDesc.from_buffer_copy(e.desc)
        for k, v in kw.items():
            setattr(dsc, k, v)
        return dsc

    # four inputs: coordinate derivatives need d_in <= 3 (the first layer's shape is not read before the refusal)
    for order in (1, 2):
        d4 = desc_with(d_in=4, deriv_order=order)
        assert lib.siren_b200_workspace_bytes(d4) == 0
        assert fwd(d4) == 1 and bwd(d4) == 1, order
    d3 = desc_with(deriv_order=3)
    assert lib.siren_b200_workspace_bytes(d3) == 0
    assert fwd(d3) == 2 and bwd(d3) == 2
    for order in (1, 2):
        assert fwd(desc_with(deriv_order=order), Jp=None) == 2, order
    assert fwd(desc_with(deriv_order=2), Dp=None) == 2
    torch.cuda.synchronize()
    for t in [y, J, D] + dW + db:
        assert bool(torch.isnan(t).all())
