"""The value path (deriv_order 0) through its C entries -- siren_b200_forward, _forward_infer, _forward_prepared,
_backward, the Fourier variants _forward_ff / _backward_ff and the operand variants _forward_call / _backward_call --
against the fp64 oracle, per element and per task, in both precisions.  This is what every SingleBVPNet call under
autograd runs, including the hypo-network of the MRI neural-process models.

Shapes: one row; many units per CTA pair; ragged tails in every task; every unit a different task; first-layer widths
1..4 (CUDA cores), 5..16 with six, five and four operand groups (tensor core), and 17..256 (one to four K chunks of
plain bf16 inputs); one to eight hidden layers; d_out 1..8 (the outermost linear fused into the forward, or last_fwd /
last_bwd of its own); shared and per-task weights; Fourier features built on chip from one to three raw channels.

Also: the coordinate gradient of the value path (gcoords, the layer-0 adjoint plane the fused chain stores only when
asked), a guard band behind the workspace sized exactly by siren_b200_workspace_bytes_ex, NaN bands behind every
output, 0xFF and reused workspaces, accumulate, run to run, ready-made weight operands and the refusals.  Every call
is profiled, and the launches it must make are asserted, so each case runs the path it was written for."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import siren_oracle as so
from tests.helpers import log_errors, oracle_chunked, rel_l2, rel_l2_per_task

pytestmark = pytest.mark.gpu

W0 = 30.0

CASES = {
    # name: d, n_hidden, d_out, tasks, per_task, n
    # one row: most CTAs have nothing to do
    "d1_n1": (1, 1, 1, 1, False, 1),
    # one hidden layer, a 2-row second tile in the only unit
    "d1_n130": (1, 1, 1, 1, False, 130),
    # whole units only
    "d2_whole": (2, 3, 1, 1, False, 4096),
    # many units per CTA pair, ragged last tile
    "d2_units": (2, 3, 1, 1, False, 150001),
    # padded to 384 rows: the second CTA's half of the last tile is empty
    "d2_n300_o2": (2, 3, 2, 1, False, 300),
    # narrow first layer, outermost linear in last_fwd / last_bwd
    "d2_o3": (2, 2, 3, 1, False, 900),
    # six and eight hidden layers with a narrow first layer (two wgrad launches)
    "d2_deep6": (2, 6, 1, 1, False, 5000),
    "d3_deep8": (3, 8, 1, 1, False, 2000),
    # shared weights, a ragged tail in every task
    "d3_t5": (3, 2, 2, 5, False, 1000),
    # widest CUDA-core first layer; 2.5 pair tiles per task
    "d4_pt": (4, 4, 2, 3, True, 640),
    # every unit a different task
    "d2_pt200": (2, 3, 1, 200, True, 128),
    # six operand groups; outermost linear in last_fwd / last_bwd
    "d5_o3": (5, 3, 3, 2, False, 900),
    # six groups, d does not divide 64
    "d7": (7, 2, 1, 1, False, 900),
    # five groups
    "d11_pt": (11, 3, 2, 4, True, 1300),
    # four groups, d does not divide 64; eight outputs
    "d13_o8": (13, 2, 8, 1, False, 2000),
    # five hidden layers per task: the MRI neural-process default
    "d16_deep5_pt": (16, 5, 2, 2, True, 700),
    # deepest net, two wgrad launches
    "d16_deep8": (16, 8, 2, 2, True, 700),
    # one K chunk of plain bf16 inputs
    "d17": (17, 3, 1, 1, False, 4097),
    # three K chunks, ragged last chunk
    "d130_pt": (130, 3, 2, 3, True, 700),
    # four K chunks, five hidden layers
    "d256_deep5": (256, 5, 2, 1, False, 20000),
}
FF_CASES = {
    # name: (F, raw channels), n_hidden, d_out, tasks, per_task, n.  d = 2 F
    "ff3_r1": ((3, 1), 3, 1, 1, False, 3000),        # d = 6: six groups
    "ff6_r3": ((6, 3), 3, 2, 3, True, 700),          # d = 12: five groups
    "ff8_r2": ((8, 2), 3, 2, 2, True, 1300),         # d = 16: the MRI scripts' features, four groups
    "ff9_r2": ((9, 2), 3, 2, 2, False, 900),         # d = 18: the wide first layer, one K chunk
    "ff103_r2": ((103, 2), 3, 2, 3, True, 700),      # d = 206: four K chunks, ragged last chunk
    "ff128_r3": ((128, 3), 5, 2, 1, False, 5000),    # d = 256, five hidden layers
}
RUNS = [(c, p) for c in list(CASES) + list(FF_CASES) for p in ("bf16", "fp32")]

# Bounds, per metric: '_l2' is rel-L2 (per task with several tasks), '_max' is max|d| / rms(ref) per element (per
# (task, output) stream for y, per (task, coordinate) stream for gcoords, per tensor for dW and db).  dbL is the
# outermost bias gradient, a sum of gy that can cancel: |d| / sum|gy| per task and output.  fp32-parity: the suite's
# 1e-4 for rel-L2 and 1e-3 per element.  bf16: 2-3x the largest value measured on a B200 over the cases above (DESIGN.md
# section 5), rel-L2 at most 3e-2.  The wide first layer (d > 16) multiplies its inputs and W_0 as plain bf16: that
# rounding alone, emulated in fp64, gives y 8.4e-3 rel-L2 and 3.9e-2 per element at d = 18 (measured: 8.5e-3, 3.8e-2),
# so y has a column of its own there.
FP32 = {"l2": 1e-4, "max": 1e-3}
BF16 = {  # metric: (d <= 16 with up to four hidden layers, d <= 16 with five to eight, d > 16)
    "y_l2": (5e-3, 5e-3, 2e-2), "y_max": (2e-2, 2e-2, 0.1),
    "yinf_l2": (5e-3, 5e-3, 2e-2), "yinf_max": (2e-2, 2e-2, 0.1),
    # forward_infer against forward (the stolen stash bit, see test_value_path_against_fp64)
    "infer_l2": (5e-3, 5e-3, 5e-3), "infer_max": (2e-2, 2e-2, 2e-2),
    "dW_l2": (3e-2, 3e-2, 3e-2), "dW_max": (0.25, 0.25, 0.25),
    "db_l2": (3e-2, 3e-2, 3e-2), "db_max": (0.2, 0.2, 0.2),
    "gx_l2": (3e-2, 3e-2, None), "gx_max": (0.3, 0.4, None),
}
DBL = 1e-5
SAME = 1e-5          # kernel against kernel: the weight-gradient atomics may sum in another order


def _bound(prec, key, d, n_hidden):
    if key == "dbL":
        return DBL
    name, kind = key.rsplit("_", 1)
    if prec == "fp32":
        return FP32[kind]
    base = "dW" if name.startswith("dW") else "db" if name.startswith("db") else name
    return BF16["%s_%s" % (base, kind)][2 if d > 16 else 1 if n_hidden > 4 else 0]


def _max_rel(a, ref, axes=None):
    """Largest |a - ref| over rms(ref); with `axes`, per slice along the other axes (the worst slice counts)."""
    a = np.asarray(a, np.float64)
    ref = np.asarray(ref, np.float64)
    err = np.abs(a - ref)
    if axes is None:
        return float(err.max() / max(np.sqrt((ref * ref).mean()), 1e-300))
    rms = np.sqrt((ref * ref).mean(axis=axes))
    return float((err.max(axis=axes) / np.maximum(rms, 1e-300)).max())


def _assert_bits(a, b, what):
    assert a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32)), \
        (what, int((a.view(np.uint32) != b.view(np.uint32)).sum()))


def _stream():
    return torch.cuda.current_stream().cuda_stream


class _Value:
    """The value-path entries through ctypes on device copies of one case's seeded inputs.  Every buffer the entries
    write is the view of a larger buffer whose tail (one task more; one copy more for a shared parameter) holds NaN,
    and every workspace is followed by a guard band of one plane (R x 512 bytes) of a fixed byte pattern; both are
    checked after every call, as are the launches the call made."""

    def __init__(self, case, prec, seed=700, cases=None):
        from siren_mri_b200 import _lib, functional as F
        self.case, self.prec = case, prec
        cases = cases or dict(CASES, **FF_CASES)
        spec = cases[case]
        if isinstance(spec[0], tuple):       # Fourier features: (F, raw) in place of d
            (self.F, self.raw), spec = spec[0], (2 * spec[0][0],) + spec[1:]
        else:
            self.F = self.raw = 0
        self.d, self.nh, self.o, self.T, self.per_task, self.n = spec[:6]
        d, T, n, o = self.d, self.T, self.n, self.o
        self.Ws, self.bs = so.make_params(d, 256, self.nh, o, seed=seed, tasks=T if self.per_task else 0)
        rng = np.random.default_rng(seed + 2)
        if self.F:
            self.x = so.make_coords(T, n, self.raw, seed=seed + 1)
            self.B = (21.0 * rng.standard_normal((self.raw, self.F))).astype(np.float32)
        else:
            self.x = so.make_coords(T, n, d, seed=seed + 1)
            self.B = None
        self.gy = (rng.standard_normal((T, n, o)) / n).astype(np.float32)
        self.lib = _lib.load()
        self.xd = torch.from_numpy(self.x).cuda()
        self.gyd = torch.from_numpy(self.gy).cuda()
        self.Wd = [torch.from_numpy(w).cuda() for w in self.Ws]
        self.bd = [torch.from_numpy(b).cuda() for b in self.bs]
        self.desc = F._make_desc(self.xd, self.Wd, W0, prec, 0)
        self.desc.d_in = d
        assert self.desc.per_task == int(self.per_task) and self.desc.tasks == T
        self.ff = None
        if self.F:
            self.Bd = torch.from_numpy(self.B).cuda()
            self.ff = _lib.SirenFourier()
            self.ff.B, self.ff.n_features, self.ff.raw_dim = self.Bd.data_ptr(), self.F, self.raw
        # the coordinate gradient: d <= 16 and no Fourier prologue
        self.gx_ok = d <= 16 and not self.F
        self.nbytes = [self.lib.siren_b200_workspace_bytes_ex(self.desc, w) for w in (0, 1)]
        assert self.nbytes[0] > 0 and self.nbytes[1] == self.lib.siren_b200_workspace_bytes(self.desc)
        self.plane = T * ((n + 127) // 128 * 128) * 512
        self.set_weights(self.Wd)
        self.call = None

    def set_weights(self, Wd):
        from siren_mri_b200 import _lib
        self.Wd = Wd
        self.w_ptrs = _lib.ptr_array(self.Wd)
        self.b_ptrs = _lib.ptr_array(self.bd)

    def set_operands(self, wk, wt):
        """siren_call_t with the Fourier prologue of the case (if any) and ready-made weight operands (or None)."""
        from siren_mri_b200 import _lib
        call = _lib.SirenCall()
        if self.ff is not None:
            call.fourier = ctypes.pointer(self.ff)
        self._ops = []
        for name, ops in (("wk16", wk), ("wt16", wt)):
            if ops is not None:
                arr = _lib.ptr_array_raw([None if t is None else t.data_ptr() for t in ops])
                self._ops.append(arr)
                setattr(call, name, ctypes.cast(arr, ctypes.POINTER(ctypes.c_void_p)))
        self.call = call

    def workspace(self, want, fill=0xFF):
        """(workspace, band): exactly workspace_bytes_ex(desc, want) bytes of `fill` (0xFF: NaN in every float format
        the planes use), then one plane of the pattern 0, 1, .., 250, 0, 1, .."""
        buf = torch.empty(self.nbytes[want] + self.plane, dtype=torch.uint8, device="cuda")
        ws, band = buf[:self.nbytes[want]], buf[self.nbytes[want]:]
        ws.fill_(fill)
        band.copy_(self.pattern())
        return ws, band

    def pattern(self):
        if getattr(self, "_pattern", None) is None:
            tile = torch.arange(251, dtype=torch.uint8, device="cuda")
            self._pattern = tile.repeat(self.plane // 251 + 1)[:self.plane]
        return self._pattern

    def check_band(self, band, what):
        torch.cuda.synchronize()
        bad = int((band != self.pattern()).sum())
        assert bad == 0, "%s wrote %d bytes of the band behind the workspace" % (what, bad)

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

    def _launch(self, fn, what):
        """rc of fn() and {kernel: launches} from the library's profile."""
        from siren_mri_b200 import _lib
        torch.cuda.synchronize()
        self.lib.siren_b200_profile_begin()
        rc = fn()
        torch.cuda.synchronize()
        buf = ctypes.create_string_buffer(1 << 14)
        self.lib.siren_b200_profile_end(buf, len(buf))
        _lib.check(rc, what)
        table = {}
        for ln in buf.value.decode().strip().splitlines():
            name, cnt, _ = ln.split()
            table[name] = int(cnt)
        return table

    def expect_forward(self, kind):
        bf, d, nh = self.prec == "bf16", self.d, self.nh
        e = {} if kind in ("prepared", "call", "call_infer") else {"prep_weights": 1}
        if bf:
            e["mlp_fused_fwd"] = 1
            if d > 4:
                e["prep_first"] = 1
            if self.o > 2:
                e["last_fwd"] = 1
        else:
            e.update(dict(featurize=1, pad_w0=1, hidden_fwd=nh + 1) if d > 16 else dict(first_fwd=1, hidden_fwd=nh))
            e["last_fwd"] = 1
        return e

    def expect_backward(self, gcoords, accumulate):
        bf, d, nh = self.prec == "bf16", self.d, self.nh
        e = {} if accumulate else {"zero_grads": 1}
        wg = (nh + 3) // 4                 # up to four hidden layers per weight-gradient launch
        if bf:
            e.update(mlp_fused_bwd=1, wgrad=wg)
            if self.o > 2:
                e["last_bwd"] = 1
            if gcoords:
                e["first_bwd"] = 1
        else:
            e.update(last_bwd=1, hidden_dgrad=nh)
            e.update(dict(wgrad=wg + 1, unpad_dw0=1, colsum=1) if d > 16 else dict(wgrad=wg, first_bwd=1))
        return e

    def forward(self, ws, kind="forward"):
        """y of one forward call: kind 'forward', 'infer', 'prepared' (after prepare_weights on ws), 'call' or
        'call_infer' (siren_b200_forward_call with the operands of set_operands).  Cases with Fourier features go
        through forward_ff (or forward_call with the prologue)."""
        from siren_mri_b200 import _lib
        P, lib, s = _lib.dptr, self.lib, _stream()
        y, yg = self._guarded((self.T, self.n, self.o), True)
        if kind == "prepared":
            _lib.check(lib.siren_b200_prepare_weights(self.desc, self.w_ptrs, P(ws), s), "prepare_weights")
        x, w, b = P(self.xd), self.w_ptrs, self.b_ptrs
        if kind in ("call", "call_infer"):
            fn = lambda: lib.siren_b200_forward_call(self.desc, self.call, x, w, b, P(y), P(ws),  # noqa: E731
                                                     int(kind == "call_infer"), s)
        elif self.ff is not None:
            assert kind in ("forward", "infer")
            fn = lambda: lib.siren_b200_forward_ff(self.desc, self.ff, x, w, b, P(y), P(ws),  # noqa: E731
                                                   int(kind == "infer"), s)
        elif kind == "forward":
            fn = lambda: lib.siren_b200_forward(self.desc, x, w, b, P(y), None, None, P(ws), s)  # noqa: E731
        elif kind == "infer":
            fn = lambda: lib.siren_b200_forward_infer(self.desc, x, w, b, P(y), P(ws), s)  # noqa: E731
        else:
            fn = lambda: lib.siren_b200_forward_prepared(self.desc, x, w, b, P(y), None, None, P(ws), s)  # noqa: E731
        names = self._launch(fn, "forward (%s)" % kind)
        assert names == self.expect_forward(kind), (kind, names)
        assert bool(torch.isnan(yg).all()), "write past the end of y"
        return y.cpu().numpy()

    def backward(self, ws, gcoords=True, accumulate=0, grads=None, kind="backward"):
        """[dW..., db...] and gcoords (None if not asked for) of one backward call on ws, which holds a forward's
        stash.  grads: what the gradient buffers start from (None: NaN).  kind 'call': siren_b200_backward_call."""
        from siren_mri_b200 import _lib
        P, lib, s = _lib.dptr, self.lib, _stream()
        params = self.Ws + self.bs
        grads = grads if grads is not None else [None] * len(params)
        gv = [self._guarded(a.shape, self.per_task, g0) for a, g0 in zip(params, grads)]
        gx, gxg = self._guarded((self.T, self.n, self.d), True) if gcoords else (None, None)
        nl = len(self.Ws)
        dW = _lib.ptr_array([v for v, _ in gv[:nl]])
        db = _lib.ptr_array([v for v, _ in gv[nl:]])
        x, w, b = P(self.xd), self.w_ptrs, self.b_ptrs
        if kind == "call":
            assert not gcoords
            fn = lambda: lib.siren_b200_backward_call(self.desc, self.call, x, w, b, P(ws), P(self.gyd), dW, db,  # noqa
                                                      accumulate, s)
        elif self.ff is not None:
            assert not gcoords
            fn = lambda: lib.siren_b200_backward_ff(self.desc, self.ff, x, w, b, P(ws), P(self.gyd), dW, db,  # noqa
                                                    accumulate, s)
        else:
            fn = lambda: lib.siren_b200_backward(self.desc, x, w, b, P(ws), P(self.gyd), None, None, dW, db,  # noqa
                                                 P(gx), accumulate, s)
        names = self._launch(fn, "backward (%s)" % kind)
        assert names == self.expect_backward(gcoords, accumulate), (kind, gcoords, accumulate, names)
        for what, g in [("gcoords", gxg)] + [("grad %d" % i, g) for i, (_, g) in enumerate(gv)]:
            assert g is None or bool(torch.isnan(g).all()), "write past the end of " + what
        return [v.cpu().numpy() for v, _ in gv], None if gx is None else gx.cpu().numpy()

    def grad_names(self):
        nl = len(self.Ws)
        return ["dW%d" % l for l in range(nl)] + ["db%d" % l for l in range(nl)]

    def dbl_err(self, got, ref, start=None):
        """The outermost bias gradient: |d| / (sum|gy| + |start|) per task (with per-task weights) and output."""
        terms = np.abs(self.gy.astype(np.float64)).sum(axis=1 if self.per_task else (0, 1))
        if start is not None:
            terms = terms + np.abs(start)
        return float((np.abs(got.astype(np.float64) - ref) / terms).max())

    def same_grads(self, got, ref, start=None):
        """{name: error} of a kernel result against another kernel result (or G0 + one): rel-L2, per task with
        per-task weights, for all but the outermost bias, which is held by dbl_err."""
        l2 = rel_l2_per_task if self.per_task else rel_l2
        names = self.grad_names()
        errs = {k: l2(a, b) for k, a, b in zip(names[:-1], got[:-1], ref[:-1])}
        errs["dbL"] = self.dbl_err(got[-1], ref[-1], None if start is None else start[-1])
        return errs


# ---------------------------------------------------------------------------------------------------------------------
# fp64 oracle of a case (on fp64 features of the fp32 inputs and B for the Fourier cases), kept for the one case whose
# runs are in progress: the two precisions of a case run back to back.
# ---------------------------------------------------------------------------------------------------------------------
_ORACLE = {}


def _oracle(e):
    if e.case not in _ORACLE:
        _ORACLE.clear()
        x = e.x.astype(np.float64)
        if e.F:
            x = so.fourier_features(x, e.B.astype(np.float64))
        gy = e.gy

        def adj(t0, t1, n0, n1, yc, Jc, Dc):
            return gy[t0:t1, n0:n1].astype(np.float64), None, None
        y, _, _, dW, db, gx = oracle_chunked(x, e.Ws, e.bs, adj, w0=W0, chunk=16384, with_gx=True)
        _ORACLE[e.case] = (y, dW + db, gx)
    return _ORACLE[e.case]


@pytest.mark.parametrize("case,prec", RUNS)
def test_value_path_against_fp64(case, prec):
    """forward, forward_infer and forward_prepared (or the _ff entries) each on a workspace of 0xFF bytes, then the
    backward into NaN gradient buffers with accumulate = 0 and, for d <= 16, gcoords -- against fp64 per task and
    per element.  forward_prepared gives forward's y to the bit, and so does forward_infer where the top layer's
    plane is written either way (d_out > 2, or fp32-parity mode)."""
    e = _Value(case, prec)
    want = int(e.gx_ok)
    ws, band = e.workspace(want)
    y = e.forward(ws)
    e.check_band(band, "forward")
    yo, gref, gxo = _oracle(e)
    assert np.isfinite(y).all()
    errs = {"y_l2": rel_l2_per_task(y, yo), "y_max": _max_rel(y, yo, axes=1)}
    ws2, band2 = e.workspace(want)
    y_inf = e.forward(ws2, "infer")
    e.check_band(band2, "forward_infer")
    if prec == "bf16" and e.o <= 2:
        # The training forward multiplies each hidden layer's stash plane as it stands: the signed sine, whose lowest
        # fp16 mantissa bit is the sign of the cosine.  Without a stash the operand is the plain fp16 sine, so y
        # differs by that stolen bit (2^-11 relative per operand).  With d_out > 2 the top plane is written either
        # way (last_fwd reads it) and the two are bit-equal.
        errs.update({"yinf_l2": rel_l2_per_task(y_inf, yo), "yinf_max": _max_rel(y_inf, yo, axes=1),
                     "infer_l2": rel_l2_per_task(y_inf, y), "infer_max": _max_rel(y_inf, y, axes=1)})
    else:
        _assert_bits(y_inf, y, "forward_infer")
    if e.ff is None:
        ws3, band3 = e.workspace(want)
        _assert_bits(e.forward(ws3, "prepared"), y, "forward_prepared")
        e.check_band(band3, "forward_prepared")
    g, gx = e.backward(ws, gcoords=e.gx_ok)
    e.check_band(band, "backward")
    assert all(np.isfinite(a).all() for a in g)
    l2 = rel_l2_per_task if e.per_task else rel_l2
    for name, a, r in zip(e.grad_names()[:-1], g[:-1], gref[:-1]):
        errs[name + "_l2"] = l2(a, r)
        errs[name + "_max"] = _max_rel(a, r)
    # the outermost bias gradient is the fp64 sum of the fp32 gy
    errs["dbL"] = e.dbl_err(g[-1], gref[-1])
    if e.gx_ok:
        assert np.isfinite(gx).all()
        errs["gx_l2"] = rel_l2_per_task(gx, gxo)
        errs["gx_max"] = _max_rel(gx, gxo, axes=1)
    log_errors("value_fp64/%s/%s" % (case, prec), **errs)
    bad = {k: v for k, v in errs.items() if not v < _bound(prec, k, e.d, e.nh)}
    assert not bad, (case, prec, bad)


@pytest.mark.parametrize("case,prec", RUNS)
def test_value_path_workspace(case, prec):
    """The workspace of workspace_bytes_ex(desc, 0) serves a backward without gcoords, the one of (desc, 1) one with
    gcoords: neither call writes past it, and the two give the same y and gradients.  A second backward on the same
    workspace, a zeroed workspace and a workspace holding the planes of other inputs give the same bits."""
    e = _Value(case, prec)
    narrow_bf16 = prec == "bf16" and e.d <= 4
    # the layer-0 adjoint plane of the fused path with a narrow first layer is the only difference
    assert e.nbytes[1] - e.nbytes[0] == (e.plane if narrow_bf16 else 0), (e.nbytes, e.plane)
    top = int(e.gx_ok)
    runs = {}
    for want in sorted({0, top}):
        ws, band = e.workspace(want)
        y = e.forward(ws)
        e.check_band(band, "forward (want_gcoords = %d)" % want)
        g, gx = e.backward(ws, gcoords=bool(want))
        e.check_band(band, "backward (want_gcoords = %d)" % want)
        runs[want] = (y, g, gx, ws, band)
    y1, g1, gx1, ws1, band1 = runs[top]
    errs = {}
    if top:
        y0, g0, _, _, _ = runs[0]
        _assert_bits(y0, y1, "y, want_gcoords 0 vs 1")
        errs.update({"nogx:" + k: v for k, v in e.same_grads(g0, g1).items()})
    # the stash survives a backward
    g2, gx2 = e.backward(ws1, gcoords=bool(top))
    e.check_band(band1, "second backward")
    if top:
        _assert_bits(gx2, gx1, "gcoords, second backward")
    errs.update({"again:" + k: v for k, v in e.same_grads(g2, g1).items()})
    # a zeroed workspace
    wsz, bandz = e.workspace(top, fill=0)
    _assert_bits(e.forward(wsz), y1, "y, zeroed workspace")
    gz, gxz = e.backward(wsz, gcoords=bool(top))
    e.check_band(bandz, "zeroed workspace")
    if top:
        _assert_bits(gxz, gx1, "gcoords, zeroed workspace")
    errs.update({"zero:" + k: v for k, v in e.same_grads(gz, g1).items()})
    # a workspace that holds the planes of other inputs of the same shape
    other = _Value(case, prec, seed=750)
    wsr, bandr = e.workspace(top)
    other.forward(wsr)
    other.backward(wsr, gcoords=bool(top))
    _assert_bits(e.forward(wsr), y1, "y, reused workspace")
    gr, gxr = e.backward(wsr, gcoords=bool(top))
    e.check_band(bandr, "reused workspace")
    if top:
        _assert_bits(gxr, gx1, "gcoords, reused workspace")
    errs.update({"reuse:" + k: v for k, v in e.same_grads(gr, g1).items()})
    log_errors("value_ws/%s/%s" % (case, prec), **errs)
    bad = {k: v for k, v in errs.items() if not v < SAME}
    assert not bad, (case, prec, bad)


@pytest.mark.parametrize("case,prec", RUNS)
def test_value_path_arguments(case, prec):
    """Run to run (exactly two calls): y and gcoords are written without atomics and are bit-equal; the gradients
    agree to the order of their atomics.  accumulate = 1 onto a random G0 of the gradient's own scale gives G0 + grad
    and launches no clearing kernel; accumulate = 0 clears NaN buffers (every call of the first two)."""
    e = _Value(case, prec)
    top = int(e.gx_ok)
    out = []
    for _ in range(2):
        ws, band = e.workspace(top)
        y = e.forward(ws)
        g, gx = e.backward(ws, gcoords=bool(top))
        e.check_band(band, "forward + backward")
        out.append((y, g, gx, ws))
    (ya, ga, gxa, _), (yb, gb, gxb, wsb) = out
    _assert_bits(ya, yb, "y, run to run")
    if top:
        _assert_bits(gxa, gxb, "gcoords, run to run")
    errs = {"run:" + k: v for k, v in e.same_grads(gb, ga).items()}
    rng = np.random.default_rng(17)
    g0 = [(rng.standard_normal(a.shape) * np.sqrt(np.mean(a.astype(np.float64) ** 2))).astype(np.float32) for a in ga]
    gacc, gxacc = e.backward(wsb, gcoords=bool(top), accumulate=1, grads=g0)
    if top:
        _assert_bits(gxacc, gxa, "gcoords, accumulate = 1")
    errs.update({"acc:" + k: v for k, v in
                 e.same_grads(gacc, [a.astype(np.float64) + b for a, b in zip(g0, ga)], start=g0).items()})
    log_errors("value_args/%s/%s" % (case, prec), **errs)
    bad = {k: v for k, v in errs.items() if not v < SAME}
    assert not bad, (case, prec, bad)


# ---------------------------------------------------------------------------------------------------------------------
# Ready-made weight operands (siren_call_t.wk16 / wt16): from siren_b200_hyper_head for per-task weights, W.half() and
# (w0 W)^T.bfloat16() for shared ones.  They are the roundings prepare_weights makes, so forward_call gives forward's y
# to the bit and backward_call forward's gradients to the order of the atomics.
# ---------------------------------------------------------------------------------------------------------------------
OPERAND_CASES = {
    # name: d (or (F, raw)), n_hidden, d_out, tasks, per_task, n
    "hyper_t3": (2, 3, 2, 3, True, 1000),
    "hyper_ff8_t2": ((8, 2), 3, 2, 2, True, 1300),      # the hypo-network of the MRI neural-process models
    "shared_o3": (3, 4, 3, 2, False, 900),
    "shared_d13_deep5": (13, 5, 1, 1, False, 3000),
}


def _hyper_weights(e, k_h=64, seed=31):
    """The hidden weights as the output of hyper heads (h [T, k_h] -> W [T, 256, 256]) at the scale of sine_init, and
    the operands the heads write."""
    from siren_mri_b200 import _lib
    rng = np.random.default_rng(seed)
    std = np.sqrt(6.0 / 256) / W0 / np.sqrt(3.0)
    Wd, wk, wt = list(e.Wd), [], []
    for l in range(1, e.nh + 1):
        h = torch.from_numpy(rng.standard_normal((e.T, k_h)).astype(np.float32)).cuda()
        Wl = torch.from_numpy((rng.standard_normal((65536, k_h)) * std / np.sqrt(k_h)).astype(np.float32)).cuda()
        bl = torch.from_numpy((rng.standard_normal(65536) * std * 0.1).astype(np.float32)).cuda()
        W = torch.empty((e.T, 256, 256), device="cuda")
        k16 = torch.empty((e.T * 256, 256), dtype=torch.float16, device="cuda")
        t16 = torch.empty((e.T * 256, 256), dtype=torch.bfloat16, device="cuda")
        _lib.check(e.lib.siren_b200_hyper_head(_lib.dptr(h), _lib.dptr(Wl), _lib.dptr(bl), e.T, k_h,
                                               ctypes.c_float(W0), _lib.dptr(W), _lib.dptr(k16), _lib.dptr(t16),
                                               None, _stream()), "hyper_head")
        Wd[l] = W
        wk.append(k16)
        wt.append(t16)
    torch.cuda.synchronize()
    return Wd, wk, wt


@pytest.mark.parametrize("case", list(OPERAND_CASES))
def test_operand_entries(case):
    """forward_call with wk16 gives the y of forward (training) and forward_infer / forward_ff (inference) to the bit
    on a workspace whose weight copies were never written; backward_call with wt16 gives backward's gradients to 1e-5.  Neither converts a
    weight (no prep_weights launch)."""
    e = _Value(case, "bf16", cases=OPERAND_CASES)
    if e.per_task:
        Wd, wk, wt = _hyper_weights(e)
        e.set_weights(Wd)
    else:
        wk = [w.half() for w in e.Wd[1:-1]]
        wt = [(w * W0).t().contiguous().bfloat16() for w in e.Wd[1:-1]]
    ws, band = e.workspace(0)
    y = {"call": e.forward(ws)}
    g, _ = e.backward(ws, gcoords=False)
    wsi, _ = e.workspace(0)
    y["call_infer"] = e.forward(wsi, "infer")
    e.set_operands(wk, wt)
    for kind in ("call_infer", "call"):       # the training forward last: its stash feeds backward_call
        wsc, bandc = e.workspace(0)
        _assert_bits(e.forward(wsc, kind), y[kind], "y, forward_call (%s)" % kind)
        e.check_band(bandc, kind)
    gc, _ = e.backward(wsc, gcoords=False, kind="call")
    e.check_band(bandc, "backward_call")
    assert all(np.isfinite(a).all() for a in gc)
    errs = e.same_grads(gc, g)
    log_errors("value_operands/%s" % case, **errs)
    bad = {k: v for k, v in errs.items() if not v < SAME}
    assert not bad, (case, bad)


@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_value_path_refusals(prec):
    """gcoords above 16 inputs: SIREN_ERR_UNSUPPORTED.  forward_infer / forward_call with deriv_order 1:
    SIREN_ERR_INVALID.  Weight operands in fp32-parity mode: SIREN_ERR_UNSUPPORTED; a NULL operand:
    SIREN_ERR_INVALID.  Nothing is written."""
    from siren_mri_b200 import _lib
    P, s = _lib.dptr, _stream()
    e = _Value("d17", prec)
    lib = e.lib
    ws, band = e.workspace(1)
    e.forward(ws)
    dW = [torch.full_like(w, float("nan")) for w in e.Wd]
    db = [torch.full_like(b, float("nan")) for b in e.bd]
    gx = torch.full((e.T, e.n, e.d), float("nan"), device="cuda")
    y = torch.full((e.T, e.n, e.o), float("nan"), device="cuda")
    assert lib.siren_b200_backward(e.desc, P(e.xd), e.w_ptrs, e.b_ptrs, P(ws), P(e.gyd), None, None,
                                   _lib.ptr_array(dW), _lib.ptr_array(db), P(gx), 0, s) == 1
    # deriv_order 1 is not a value-path call, whatever the shape
    e3 = _Value("d3_t5", prec)
    d1 = _lib.SirenDesc.from_buffer_copy(e3.desc)
    d1.deriv_order = 1
    ws3, _ = e3.workspace(1)
    y3 = torch.full((e3.T, e3.n, e3.o), float("nan"), device="cuda")
    assert lib.siren_b200_forward_infer(d1, P(e3.xd), e3.w_ptrs, e3.b_ptrs, P(y3), P(ws3), s) == 2
    e3.set_operands(None, None)
    assert lib.siren_b200_forward_call(d1, e3.call, P(e3.xd), e3.w_ptrs, e3.b_ptrs, P(y3), P(ws3), 0, s) == 2
    assert lib.siren_b200_forward_call(d1, e3.call, P(e3.xd), e3.w_ptrs, e3.b_ptrs, P(y3), P(ws3), 1, s) == 2
    # operands: the fused bf16 path only; every hidden layer's operand given
    op = torch.zeros((256, 256), dtype=torch.float16, device="cuda")
    dW3 = [torch.full_like(w, float("nan")) for w in e3.Wd]
    db3 = [torch.full_like(b, float("nan")) for b in e3.bd]

    def ops(nh, null):        # null: the layer whose operand is NULL (first or last), or None
        return [None if l == {"first": 0, "last": nh - 1}.get(null) else op for l in range(nh)]
    for null, code in [(None, 1)] if prec == "fp32" else [("first", 2), ("last", 2)]:
        e.set_operands(ops(e.nh, null), ops(e.nh, null))
        assert lib.siren_b200_forward_call(e.desc, e.call, P(e.xd), e.w_ptrs, e.b_ptrs, P(y), P(ws), 0, s) == code
        e3.set_operands(ops(e3.nh, null), ops(e3.nh, null))
        assert lib.siren_b200_backward_call(e3.desc, e3.call, P(e3.xd), e3.w_ptrs, e3.b_ptrs, P(ws3), P(e3.gyd),
                                            _lib.ptr_array(dW3), _lib.ptr_array(db3), 0, s) == code
    torch.cuda.synchronize()
    e.check_band(band, "refused calls")
    for t in [y, y3, gx] + dW + db + dW3 + db3:
        assert bool(torch.isnan(t).all())
