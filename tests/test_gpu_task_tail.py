"""The optimizer tail of T stacked networks through its two C entries, siren_b200_adam_step_tasks and
siren_b200_clip_grad_tasks, on synthetic flat buffers, against the float64 restatement in tests/task_tail_ref.py.

No forward pass is needed: param / grad / m / v are filled directly in a flat layout (tests/task_tail_ref.layout), in
the trainer's parameter order and three others, with W / b pointer arrays into them.  The data make the mistakes these
kernels can make large against the tolerances:
  - task t's gradient has norm exactly 2 ** (t / 128) (one task all zero), max_norm sits between two neighbouring
    norms near the median, so about half the tasks clip and no norm is within 0.27 % of max_norm;
  - the elements at task and segment boundaries and at local indices 0 and 4095 mod 4096 (the ends of the kernels'
    work items) are 30x the rest, as are the loss values at 0, 4095, 4096 and the last of each task: one dropped or
    doubled element moves its task's norm or loss by at least 0.1 %;
  - m and v start random and non-zero and the step above 1, so the update depends on the clip coefficient.
Every output buffer has a sentinel band behind it that must come back unchanged."""
import ctypes
import functools
import struct

import numpy as np
import pytest
import torch

from siren_mri_b200 import _lib
from tests import task_tail_ref as ref
from tests.helpers import log_errors

pytestmark = pytest.mark.gpu

H = 256
BAND = 64                 # floats of sentinel behind every buffer
SENT = -1234.5
STATE_FMT = "<ffffqqdd16x"        # AdamState (csrc/simt.h)
LR, EPS = 1e-3, 1e-8
TM_CLIP, TM_FREE = 1e-6, 3e-7     # m / v, relative to the magnitude of the terms forming them (clipped / unclipped task)


@pytest.fixture(autouse=True)
def _peak_memory(request):
    """Every case stays well inside 16 GB of device memory (its peak is logged with the errors).  The peak counts
    from what is allocated when the case starts: tensors that earlier test modules keep alive are not this case's."""
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    yield
    peak = (torch.cuda.max_memory_allocated() - base) / 2 ** 30
    log_errors("peak_memory:" + request.node.name, gib=peak)
    assert peak < 12.0, (request.node.name, peak)


def _P(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _banded(n, fill=None):
    t = torch.full((n + BAND,), SENT, device="cuda")
    if fill is not None:
        t[:n] = fill
    return t


def _state(step=0, pow1=0.0, pow2=0.0):
    raw = struct.pack(STATE_FMT, 0.0, 0.25, 0.5, 0.0, step, 0, pow1, pow2)
    t = torch.full((64 + 4 * BAND,), 0xA5, dtype=torch.uint8, device="cuda")
    t[:64] = torch.frombuffer(bytearray(raw), dtype=torch.uint8).cuda()
    return t


def _read_state(t):
    assert bool((t[64:] == 0xA5).all()), "AdamState band"
    sumsq, bc1, bc2, _, step, pad2, pow1, pow2 = struct.unpack(STATE_FMT, bytes(t[:64].cpu().numpy()))
    return dict(sumsq=sumsq, bc1=bc1, bc2_sqrt=bc2, step=step, done=pad2 & 0xFFFFFFFF, pow1=pow1, pow2=pow2)


def _desc(arch, T, n_coords, precision="bf16", per_task=1, deriv_order=0):
    d_in, nh, d_out = arch
    return _lib.SirenDesc(d_in, H, nh, d_out, 30.0, T, per_task, n_coords, _lib.PRECISIONS[precision], deriv_order)


@functools.lru_cache(maxsize=None)
def _pow(beta, k):
    return ref.running_pow(beta, k)


class Tail:
    """One problem: the flat buffers (sentinel-banded), per-task state and y / gt of T networks of ``arch``."""

    def __init__(self, arch, T, order, n_coords, seed=0, precision="bf16", zero_task=True, deriv_order=0):
        self.arch, self.T, self.n_coords = arch, T, n_coords
        self.segs, self.n = ref.layout(arch, T, order)
        self.desc = _desc(arch, T, n_coords, precision, deriv_order=deriv_order)
        n, dev = self.n, "cuda"
        gen = torch.Generator(device=dev).manual_seed(seed)
        rnd = lambda k: torch.randn(k, generator=gen, device=dev)      # noqa: E731
        g = rnd(n)
        cum = 0
        for s, v in zip(self.segs, ref.views(g, self.segs, T)):
            j = torch.arange(s["per"], device=dev) + cum
            edge = (j % 4096 == 0) | (j % 4096 == 4095) | (j == cum) | (j == cum + s["per"] - 1)
            v.mul_(torch.where(edge, 30.0, 1.0))
            cum += s["per"]
        self.P = cum                       # floats per task
        scale = 2.0 ** (torch.arange(T, device=dev, dtype=torch.float64) / 128)
        if zero_task and T >= 3:
            scale[1] = 0.0
        f = (scale / torch.sqrt(ref.task_sumsq(g, self.segs, T))).float()
        for v in ref.views(g, self.segs, T):
            v.mul_(f[:, None])
        typ = ref.per_element((scale.clamp(min=1.0) / np.sqrt(self.P)).float(), self.segs, T)
        self.init = dict(p=(torch.rand(n, generator=gen, device=dev) - 0.5) * 0.2, g=g,
                         m=rnd(n) * typ * 0.5, v=(torch.rand(n, generator=gen, device=dev) * 1.5 + 0.5) * typ * typ)
        nz = sorted(x for x in torch.sqrt(ref.task_sumsq(g, self.segs, T)).tolist() if x > 0)
        tm = (len(nz) - 1) // 2
        self.max_norm = float(np.sqrt(nz[tm] * nz[tm + 1])) if len(nz) > 1 else 0.5 * nz[0]
        rows = n_coords * arch[2]
        self.rows = rows
        gt = rnd(T * rows).view(T, rows)
        d = rnd(T * rows).view(T, rows) * 0.1
        marks = torch.ones(rows, device=dev)
        for r in (0, 4095, 4096, rows - 1):
            if r < rows:
                marks[r] = 30.0
        d = d * marks * (2.0 ** (torch.arange(T, device=dev) / 128))[:, None]
        self.gt = gt.view(T, n_coords, arch[2]).contiguous()
        self.y = (gt + d).view(T, n_coords, arch[2]).contiguous()
        self.reset()

    def reset(self, step=0, b1=0.9, b2=0.999):
        T, n = self.T, self.n
        self.buf = {k: _banded(n, v) for k, v in self.init.items()}
        self.sumsq = _banded(T, 0.0)
        self.running = torch.arange(T, device="cuda", dtype=torch.float32) * 0.125 + 0.5
        self.loss = _banded(2 * T, torch.cat([torch.full((T,), 7.0, device="cuda"), self.running]))
        self.loss4 = torch.tensor([3.0, 5.0, 11.0, 13.0], device="cuda")
        self.state = _state(step, _pow(b1, step), _pow(b2, step))

    def ptrs(self, flat):
        W, b = [None] * (self.arch[1] + 2), [None] * (self.arch[1] + 2)
        for s in self.segs:
            (W if s["kind"] == "W" else b)[s["layer"]] = flat.data_ptr() + 4 * s["off"]
        return _lib.ptr_array_raw(W), _lib.ptr_array_raw(b)

    def adam(self, max_norm, b1=0.9, b2=0.999, y=True, weight=0.37, ws=None):
        W, b = self.ptrs(self.buf["p"])
        yy, gg = (self.y, self.gt) if y else (None, None)
        return _lib.load().siren_b200_adam_step_tasks(
            self.desc, W, b, _P(self.buf["p"]), _P(self.buf["g"]), _P(self.buf["m"]), _P(self.buf["v"]), self.n, LR,
            b1, b2, EPS, max_norm, _P(self.state), _P(yy), _P(gg), weight, _P(self.sumsq), _P(self.loss),
            _P(self.loss4), _P(ws), _stream())

    def clip(self, max_norm, y=True, weight=0.37, publish=1):
        dW, db = self.ptrs(self.buf["g"])
        yy, gg = (self.y, self.gt) if y else (None, None)
        return _lib.load().siren_b200_clip_grad_tasks(
            self.desc, dW, db, _P(self.buf["g"]), self.n, max_norm, _P(self.state), _P(yy), _P(gg), weight,
            _P(self.sumsq), _P(self.loss), _P(self.loss4), publish, _stream())

    def bands_intact(self):
        for k, t in list(self.buf.items()) + [("sumsq", self.sumsq), ("loss", self.loss)]:
            assert bool((t[-BAND:] == SENT).all()), "sentinel band behind %s overwritten" % k

    def snapshot(self):
        return {k: v[:self.n].clone() for k, v in self.buf.items()}

    def coefs(self, g, max_norm):
        return ref.clip_coefs(g, self.segs, self.T, max_norm)[0]


def _pieces(tl, limit=1 << 22):
    """The flat layout as (segment, first task, end task) pieces of at most ``limit`` floats (or one task row): the
    float64 checks of T = 1024 then stay within a few hundred MB."""
    for k, s in enumerate(tl.segs):
        step = max(1, limit // s["per"])
        for t0 in range(0, tl.T, step):
            yield k, t0, min(tl.T, t0 + step)


def _piece(flat, tl, k, t0, t1):
    s = tl.segs[k]
    return flat[s["off"] + t0 * s["per"]:s["off"] + t1 * s["per"]].view(t1 - t0, s["per"])


def _check_adam(tl, before, coef, step, b1, b2, case, mask=None):
    """p, m, v of one adam_step_tasks call against the float64 reference from ``before``; g cleared.
    m and v to TM_CLIP / TM_FREE of the magnitude of the terms that form them; p to 2 ulp + 1e-5 of its update, plus
    what the allowed error of m moves it by (m can cancel: b1 m0 = -(1 - b1) c g)."""
    mb1, mb2 = ref.moment_beta(b1), ref.moment_beta(b2)
    step_size, bc2 = LR / (1.0 - b1 ** step), 1.0 - b2 ** step
    errs = dict(m_clip=0.0, m_free=0.0, v_clip=0.0, v_free=0.0, p=0.0)
    for k, t0, t1 in _pieces(tl):
        P = lambda f: _piece(f, tl, k, t0, t1)      # noqa: E731
        c = coef[t0:t1, None]
        p0, g0, m0, v0 = (P(before[x]).double() for x in "pgmv")
        p1, m1, v1 = ref.adam(p0, g0, m0, v0, c, step, LR, b1, b2, EPS, mb1, mb2)
        clipped = (c < 1).expand_as(p1)
        tol = TM_FREE + (TM_CLIP - TM_FREE) * clipped.double()
        keep = torch.ones_like(clipped) if mask is None else P(mask)
        gc = g0 * c
        term_m = (mb1 * m0).abs() + ((1 - mb1) * gc).abs()
        for name, want, term in (("m", m1, term_m), ("v", v1, (mb2 * v0).abs() + ((1 - mb2) * gc * gc).abs())):
            r = (P(tl.buf[name]).double() - want).abs() / (term + 1e-300)
            for tag, sel in (("_clip", clipped & keep), ("_free", ~clipped & keep)):
                if bool(sel.any()):
                    errs[name + tag] = max(errs[name + tag], float(r[sel].max()))
            bad = (r > tol) & keep
            assert not bool(bad.any()), (case, name, k, t0, int(bad.sum()), errs)
        denom = torch.sqrt(v1) / np.sqrt(bc2) + EPS
        tol_p = 2 * ref.ulp32(p1) + 1e-5 * (p1 - p0).abs() + step_size * tol * term_m / denom
        r = (P(tl.buf["p"]).double() - p1).abs() / tol_p
        errs["p"] = max(errs["p"], float(r[keep].max()))
        bad = (r > 1) & keep
        assert not bool(bad.any()), (case, "p", k, t0, int(bad.sum()), errs)
    assert bool((tl.buf["g"][:tl.n] == 0).all()), (case, "g not cleared")
    log_errors("task_tail_adam:" + case, **errs)
    return errs


def _check_clipped(tl, before_g, coef, what):
    """The gradient after clip_grad_tasks: a task that does not clip is untouched, the others are g * coef to 1e-6."""
    err = 0.0
    for k, t0, t1 in _pieces(tl):
        g0 = _piece(before_g, tl, k, t0, t1)
        got = _piece(tl.buf["g"], tl, k, t0, t1)
        c = coef[t0:t1]
        free = c == 1.0
        assert torch.equal(got[free], g0[free]), what
        if bool((~free).any()):
            want = g0[~free].double() * c[~free][:, None]
            err = max(err, float(((got[~free].double() - want).abs() / (want.abs() + 1e-300)).max()))
    assert err < 1e-6, (what, err)
    return err


def _check_state(tl, step, b1, b2):
    st = _read_state(tl.state)
    q1, q2 = _pow(b1, step), _pow(b2, step)
    assert st["step"] == step and st["done"] == 0, st
    assert st["pow1"] == q1 and st["pow2"] == q2, (st, q1, q2)
    assert st["bc1"] == np.float32(1.0 - q1) and st["bc2_sqrt"] == np.float32(np.sqrt(1.0 - q2)), st
    assert abs(st["bc1"] - (1.0 - b1 ** step)) <= 6e-8 and abs(st["bc2_sqrt"] - np.sqrt(1.0 - b2 ** step)) <= 6e-8, st
    assert st["sumsq"] == 0.0, st


def _check_losses(tl, want, published, case, rtol=1e-5):
    """task_loss after a call that added ``want`` [T] (float64) to the running sums."""
    T = tl.T
    got = tl.loss[:2 * T].double()
    run = tl.running.double() + want
    if published:
        err = float(((got[:T] - run).abs() / run.abs()).max())
        assert err < rtol, (case, err)
        assert bool((tl.loss[T:2 * T] == 0).all()), case
    else:
        assert bool((tl.loss[:T] == 7.0).all()), case
        err = float(((got[T:] - run).abs() / run.abs()).max())
        assert err < rtol, (case, err)
    return err


# (arch, T, order, n_coords): every architecture in every order; T from 1 to 1024; n * d_out around the 4096-float
# work items of the loss pass (1, 4095, 4096, 4097, > 3 * 4096)
ARCHS = [(1, 1, 1), (2, 3, 1), (3, 2, 3), (4, 4, 2), (16, 8, 8), (60, 3, 2)]
ARCH_N = {(1, 1, 1): 4097, (2, 3, 1): 4096, (3, 2, 3): 1365, (4, 4, 2): 2049, (16, 8, 8): 513, (60, 3, 2): 6145}
CASES = [(a, 7, o, ARCH_N[a]) for a in ARCHS for o in ref.ORDERS] + [
    ((1, 1, 1), 1, "trainer", 4095), ((1, 1, 1), 1, "biases_first", 1), ((2, 3, 1), 2, "random", 1),
    ((2, 3, 1), 2, "biases_first", 12289), ((2, 3, 1), 7, "biases_first", 1), ((2, 3, 1), 7, "reversed", 4097),
    ((2, 3, 1), 64, "trainer", 4096),       # the benchmarked shape
    ((3, 2, 3), 64, "biases_first", 4097), ((16, 8, 8), 64, "random", 100), ((60, 3, 2), 64, "reversed", 2048),
    ((1, 1, 1), 1024, "trainer", 1), ((1, 1, 1), 1024, "biases_first", 4097), ((1, 1, 1), 1023, "random", 4096),
]


def _id(c):
    return "%s-T%d-%s-n%d" % ("x".join(map(str, c[0])), c[1], c[2], c[3])


@pytest.mark.parametrize("clip", [False, True])
@pytest.mark.parametrize("case", CASES, ids=[_id(c) for c in CASES])
def test_adam_step_tasks(case, clip):
    """One adam_step_tasks call from step 4, against float64: p, m, v per element, g cleared, the per-task losses
    published, loss4 rolled, task_sumsq cleared and the AdamState advanced."""
    arch, T, order, n_coords = case
    b1, b2 = 0.9, 0.999
    tl = Tail(arch, T, order, n_coords, seed=T + arch[1])
    tl.reset(step=4)
    before = tl.snapshot()
    max_norm = tl.max_norm if clip else 0.0
    coef = tl.coefs(before["g"], max_norm)
    if clip and T > 1:
        assert float(coef[0]) == 1.0 and float(coef[-1]) < 1.0 and 0 < int((coef < 1).sum()) < T
    assert tl.adam(max_norm, b1, b2) == 0, _lib.load().siren_b200_last_error()
    torch.cuda.synchronize()
    tl.bands_intact()
    _check_adam(tl, before, coef, 5, b1, b2, _id(case) + ("-clip" if clip else ""))
    _check_losses(tl, ref.task_losses(tl.y, tl.gt, 0.37), True, case)
    assert tl.loss4.tolist() == [5.0, 0.0, 11.0, 13.0]
    assert bool((tl.sumsq[:T] == 0).all())
    _check_state(tl, 5, b1, b2)


CLIP_CASES = [((2, 3, 1), 7, "biases_first", 4097), ((3, 2, 3), 64, "random", 1366), ((16, 8, 8), 2, "reversed", 513),
              ((1, 1, 1), 1024, "trainer", 4096), ((60, 3, 2), 7, "trainer", 1)]


@pytest.mark.parametrize("case", CLIP_CASES, ids=[_id(c) for c in CLIP_CASES])
def test_clip_grad_tasks(case):
    """clip_grad_tasks in every combination of publish, y given or not and max_norm > 0 or 0: the clipped gradient
    per element, the losses added to the running sums and published (or not), task_sumsq cleared, the step counter
    untouched."""
    arch, T, order, n_coords = case
    tl = Tail(arch, T, order, n_coords, seed=11)
    for publish in (0, 1):
        for with_y in (False, True):
            for clip in (True, False):
                if T == 1024 and not (clip and with_y):
                    continue
                what = (case, publish, with_y, clip)
                tl.reset(step=9)
                before = tl.snapshot()
                max_norm = tl.max_norm if clip else 0.0
                coef = tl.coefs(before["g"], max_norm)
                assert tl.clip(max_norm, y=with_y, publish=publish) == 0, _lib.load().siren_b200_last_error()
                torch.cuda.synchronize()
                tl.bands_intact()
                err = _check_clipped(tl, before["g"], coef, what)
                for k in "pmv":
                    assert torch.equal(tl.buf[k][:tl.n], before[k]), (what, k)
                added = ref.task_losses(tl.y, tl.gt, 0.37) if with_y else torch.zeros(T, dtype=torch.float64,
                                                                                       device="cuda")
                _check_losses(tl, added, bool(publish), what)
                assert tl.loss4.tolist() == ([5.0, 0.0, 11.0, 13.0] if publish else [3.0, 5.0, 11.0, 13.0]), what
                assert bool((tl.sumsq[:T] == 0).all()), what
                st = _read_state(tl.state)
                assert st["step"] == 9 and st["done"] == 0 and st["pow1"] == _pow(0.9, 9), (what, st)
                log_errors("task_tail_clip:%s-p%d-y%d-c%d" % (_id(case), publish, with_y, clip), g=err)


@pytest.mark.parametrize("case,acc", [(((3, 2, 3), 7, "biases_first", 1366), 3), (((1, 1, 1), 64, "random", 4097), 2),
                                      (((4, 4, 2), 5, "reversed", 2049), 1)], ids=["3x2x3-acc3", "1x1x1-acc2",
                                                                                  "4x4x2-acc1"])
def test_microbatch_sequence(case, acc):
    """Three optimizer steps as the trainer's _tasks_tail makes them: per micro-batch the gradient accumulates and
    clip_grad_tasks clips it and adds the loss (publishing it unless the micro-batch updates), then adam_step_tasks
    without clipping and without y; with acc = 1 one adam_step_tasks with clip and y.  Every call is checked against
    float64 from the kernel's own inputs; the norms and losses must not carry over between calls."""
    arch, T, order, n_coords = case
    b1, b2 = 0.9, 0.999
    tl = Tail(arch, T, order, n_coords, seed=5)
    tl.reset(step=0)
    tl.buf["g"][:tl.n] = 0.0
    w = 0.37 / acc
    step = 0
    for s in range(3):
        for k in range(acc):
            # the micro-batch's gradient, task-scaled like the initial one, accumulates onto the clipped sum
            tl.buf["g"][:tl.n] += tl.init["g"] * ((1.0 + 0.1 * k + 0.2 * s) / acc)
            tl.y.add_(0.01)
            want_loss = ref.task_losses(tl.y, tl.gt, w)
            tl.running = tl.loss[T:2 * T].clone()
            stale = tl.loss[:T].clone()
            before = tl.snapshot()
            update = k == acc - 1
            if acc > 1:
                coef = tl.coefs(before["g"], tl.max_norm)
                assert tl.clip(tl.max_norm, y=True, weight=w, publish=0 if update else 1) == 0
                torch.cuda.synchronize()
                tl.bands_intact()
                _check_clipped(tl, before["g"], coef, (s, k))
                if update:
                    assert torch.equal(tl.loss[:T], stale)
                    run = tl.running.double() + want_loss
                    assert float(((tl.loss[T:2 * T].double() - run).abs() / run).max()) < 1e-5, (s, k)
                else:
                    _check_losses(tl, want_loss, True, (s, k))
                assert bool((tl.sumsq[:T] == 0).all()), (s, k)
            if update:
                before = tl.snapshot()
                tl.running = tl.loss[T:2 * T].clone()
                mn = tl.max_norm if acc == 1 else 0.0
                coef = tl.coefs(before["g"], mn)
                assert tl.adam(mn, b1, b2, y=acc == 1, weight=w) == 0
                torch.cuda.synchronize()
                tl.bands_intact()
                step += 1
                _check_adam(tl, before, coef, step, b1, b2, "seq-%s-acc%d-s%d" % (_id(case), acc, s))
                _check_losses(tl, want_loss if acc == 1 else torch.zeros_like(want_loss), True, (s, k))
                assert bool((tl.sumsq[:T] == 0).all())
                _check_state(tl, step, b1, b2)


# the copy layouts (precision, deriv_order): the fused bf16 value path (fp16 copy as stored, bf16 transposed copy times
# w0), the bf16 jet paths (plain bf16 copies) and the fp32 path (bf16 hi / lo copies)
PATHS = {"fused": ("bf16", 0), "unfused": ("bf16", 1), "fp32": ("fp32", 0)}
WS_CASES = ([(p, (3, h, 1), 3, o) for p in PATHS for h in range(1, 9) for o in ("trainer", "biases_first")] +
            [(p, (1, 1, 1), 1024, "biases_first") for p in PATHS] +
            [("fused", (60, 3, 2), 5, "random"), ("fp32", (60, 3, 2), 5, "random"), ("unfused", (3, 8, 8), 7, "random")])


@pytest.mark.parametrize("path,arch,T,order", WS_CASES,
                         ids=["%s-%s-T%d-%s" % (c[0], "x".join(map(str, c[1])), c[2], c[3]) for c in WS_CASES])
def test_workspace_equals_prepare_weights(path, arch, T, order):
    """prepare_weights(old) + adam_step_tasks leaves the WHOLE workspace byte-equal to prepare_weights(new) on a
    zeroed one: every task's 16-bit copies of every hidden layer in every layout, and no write anywhere else."""
    precision, deriv_order = PATHS[path]
    lib = _lib.load()
    tl = Tail(arch, T, order, 1, seed=3, precision=precision, deriv_order=deriv_order)
    tl.reset(step=2)
    nbytes = lib.siren_b200_workspace_bytes_ex(tl.desc, 0)
    assert nbytes > 0, lib.siren_b200_last_error()
    W, _ = tl.ptrs(tl.buf["p"])
    ws = torch.zeros(nbytes + 1024, dtype=torch.uint8, device="cuda")
    ws[nbytes:] = 0x5A
    _lib.check(lib.siren_b200_prepare_weights(tl.desc, W, _P(ws), _stream()), "prepare_weights")
    assert tl.adam(tl.max_norm, ws=ws) == 0, lib.siren_b200_last_error()
    ws2 = torch.zeros_like(ws)
    ws2[nbytes:] = 0x5A
    _lib.check(lib.siren_b200_prepare_weights(tl.desc, W, _P(ws2), _stream()), "prepare_weights")
    torch.cuda.synchronize()
    tl.bands_intact()
    assert not torch.equal(tl.buf["p"][:tl.n], tl.init["p"])
    diff = (ws != ws2).nonzero()
    assert diff.numel() == 0, (int(diff.numel()), int(diff[0]), nbytes)


def _copies(ws, arch, T, precision):
    """The workspace's weight copies as [n_hidden, planes, T, H * H] 16-bit words (the layout of make_layout in
    csrc/api.cu: per hidden layer the as-stored then the transposed copy, each hi [, lo], one after the other)."""
    planes = 4 if precision == "fp32" else 2
    nh = arch[1]
    return ws[:nh * planes * T * H * H * 2].view(torch.int16).view(nh, planes, T, H * H)


@pytest.mark.parametrize("mode", ["nan", "one_nan", "huge"])
def test_one_scene_cannot_touch_another(mode):
    """Task k's gradient all NaN, one NaN element, or 1e6 times larger; every other task below max_norm (coefficient
    exactly 1).  Every other task's p, m, v, weight copies and loss are bit-equal to a clean run.
    Expected for task k: with one NaN its squared norm is NaN and fminf(NaN, 1) = 1, so the task is NOT clipped: the
    NaN element updates to NaN and the others update unclipped.  torch's clip_grad_norm_ multiplies every gradient
    of the model by the NaN coefficient instead, so there the whole model becomes NaN -- as it does here when every
    element is NaN.  The 1e6 task is clipped to max_norm and stays finite."""
    arch, T, order, k = (2, 3, 1), 7, "biases_first", 3
    lib = _lib.load()
    runs = {}
    for dirty in (False, True):
        tl = Tail(arch, T, order, 200, seed=21)
        tl.reset(step=3)
        gk = [v[k] for v in ref.views(tl.buf["g"], tl.segs, T)]
        if dirty:
            if mode == "nan":
                for v in gk:
                    v.fill_(float("nan"))
            elif mode == "one_nan":
                gk[2][5] = float("nan")
            else:
                for v in gk:
                    v.mul_(1e6)
        norms = torch.sqrt(ref.task_sumsq(tl.init["g"], tl.segs, T))
        max_norm = float(norms.max()) * 10.0
        before = tl.snapshot()
        nbytes = lib.siren_b200_workspace_bytes_ex(tl.desc, 0)
        ws = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
        W, _ = tl.ptrs(tl.buf["p"])
        _lib.check(lib.siren_b200_prepare_weights(tl.desc, W, _P(ws), _stream()), "prepare_weights")
        assert tl.adam(max_norm, ws=ws) == 0
        torch.cuda.synchronize()
        tl.bands_intact()
        runs[dirty] = (tl, ws, before, max_norm)
    (clean, ws0, _, _), (dirty, ws1, before, max_norm) = runs[False], runs[True]
    others = [t for t in range(T) if t != k]
    for name in "pmv":
        for a, b in zip(ref.views(clean.buf[name], clean.segs, T), ref.views(dirty.buf[name], dirty.segs, T)):
            assert torch.equal(a[others], b[others]), (mode, name)
    c0, c1 = _copies(ws0, arch, T, "bf16"), _copies(ws1, arch, T, "bf16")
    assert torch.equal(c0[:, :, others], c1[:, :, others]), mode
    assert torch.equal(ws0[c0.numel() * 2:], ws1[c1.numel() * 2:]), mode
    assert torch.equal(clean.loss[:T], dirty.loss[:T]), mode          # the loss comes from y / gt, not from g
    pk = torch.cat([v[k] for v in ref.views(dirty.buf["p"], dirty.segs, T)])
    if mode == "nan":
        assert bool(torch.isnan(pk).all())
    elif mode == "one_nan":
        assert int(torch.isnan(pk).sum()) == 1
        coef = torch.ones(T, dtype=torch.float64, device="cuda")
        g = before["g"].clone()
        g[torch.isnan(g)] = 0.0
        mask = ~torch.isnan(dirty.buf["p"][:dirty.n])
        _check_adam(dirty, dict(before, g=g), coef, 4, 0.9, 0.999, "one_nan", mask=mask)
        # torch: the whole model NaN
        ps = [torch.nn.Parameter(torch.ones(3, device="cuda")) for _ in range(2)]
        ps[0].grad = torch.tensor([1.0, float("nan"), 1.0], device="cuda")
        ps[1].grad = torch.ones(3, device="cuda")
        torch.nn.utils.clip_grad_norm_(ps, max_norm=1.0)
        assert bool(torch.isnan(ps[1].grad).all())
    else:
        assert bool(torch.isfinite(pk).all())
        coef = ref.clip_coefs(before["g"], dirty.segs, T, max_norm)[0]
        assert float(coef[k]) < 1e-4 and bool((coef[others] == 1).all())
        _check_adam(dirty, before, coef, 4, 0.9, 0.999, "huge")


BETAS = [(0.9, 0.999), (0.5, 0.999), (0.3, 0.5)]
KS = [1, 1074, 1075, 1076, 10 ** 5, 10 ** 6]


@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("betas", BETAS, ids=["0.9-0.999", "0.5-0.999", "0.3-0.5"])
@pytest.mark.parametrize("entry", ["adam_step", "adam_step_tasks"])
def test_bias_correction_long_runs(entry, betas, k):
    """Step k from the AdamState of k - 1 steps (pow1 / pow2 the running products): the step size and the stored
    bc1, bc2_sqrt, pow1, pow2 against 1 - beta ** k.  The running product of beta <= 0.5 underflows to exactly 0.0
    (beta = 0.5 after 1075 steps, 0.3 after 619), which must not read as a fresh state."""
    b1, b2 = betas
    tl = Tail((1, 1, 1), 2, "trainer", 1, seed=4)
    tl.reset(step=k - 1, b1=b1, b2=b2)
    before = tl.snapshot()
    if entry == "adam_step":
        rc = _lib.load().siren_b200_adam_step(_P(tl.buf["p"]), _P(tl.buf["g"]), _P(tl.buf["m"]), _P(tl.buf["v"]), tl.n,
                                              LR, b1, b2, EPS, 0.0, 1.0, _P(tl.state), 1, None, None, None, None,
                                              _stream())
    else:
        rc = tl.adam(0.0, b1, b2, y=False)
    assert rc == 0, _lib.load().siren_b200_last_error()
    torch.cuda.synchronize()
    tl.bands_intact()
    coef = torch.ones(2, dtype=torch.float64, device="cuda")
    p1, _, _ = ref.adam(before["p"], before["g"], before["m"], before["v"], 1.0, k, LR, b1, b2, EPS,
                        ref.moment_beta(b1), ref.moment_beta(b2))
    dp_ref = p1 - before["p"].double()
    dp = tl.buf["p"][:tl.n].double() - before["p"].double()
    big = dp_ref.abs() > 1e3 * ref.ulp32(before["p"].double())
    ratio = float((dp[big] / dp_ref[big]).median())
    log_errors("bias_correction:%s-%s-%s-k%d" % (entry, b1, b2, k), step_ratio=ratio)
    st = _read_state(tl.state)
    assert abs(ratio - 1.0) < 1e-4, (entry, betas, k, ratio, st)
    _check_adam(tl, before, coef, k, b1, b2, "bias-%s-%g-%g-k%d" % (entry, b1, b2, k))
    _check_state(tl, k, b1, b2)


def test_refusals():
    """T = 1025: SIREN_ERR_UNSUPPORTED; per_task = 0, y without gt and an unaligned m: SIREN_ERR_INVALID.  Nothing is
    written."""
    lib = _lib.load()
    tl = Tail((1, 1, 1), 3, "trainer", 16, seed=1)
    tl.reset(step=1)
    before = tl.snapshot()
    W, b = tl.ptrs(tl.buf["p"])
    dW, db = tl.ptrs(tl.buf["g"])
    P, s = _P, _stream()

    def adam(desc, m=tl.buf["m"], y=None, gt=None):
        return lib.siren_b200_adam_step_tasks(desc, W, b, P(tl.buf["p"]), P(tl.buf["g"]), P(m), P(tl.buf["v"]), tl.n,
                                              LR, 0.9, 0.999, EPS, 1.0, P(tl.state), P(y), P(gt), 0.37, P(tl.sumsq),
                                              P(tl.loss), P(tl.loss4), None, s)

    def clip(desc, y=None, gt=None):
        return lib.siren_b200_clip_grad_tasks(desc, dW, db, P(tl.buf["g"]), tl.n, 1.0, P(tl.state), P(y), P(gt), 0.37,
                                              P(tl.sumsq), P(tl.loss), P(tl.loss4), 1, s)

    big = _desc((1, 1, 1), 1025, 16)
    assert adam(big) == 1 and clip(big) == 1
    shared = _desc((1, 1, 1), 3, 16, per_task=0)
    assert adam(shared) == 2 and clip(shared) == 2
    assert adam(tl.desc, y=tl.y) == 2 and adam(tl.desc, gt=tl.gt) == 2 and clip(tl.desc, y=tl.y) == 2
    m_off = tl.buf["m"][1:]
    assert adam(tl.desc, m=m_off) == 2
    torch.cuda.synchronize()
    for k in "pgmv":
        assert torch.equal(tl.buf[k][:tl.n], before[k]), k
    assert _read_state(tl.state)["step"] == 1
    assert tl.loss4.tolist() == [3.0, 5.0, 11.0, 13.0]


def test_trainer_refuses_1025_scenes():
    from siren_mri_b200 import modules
    from siren_mri_b200.trainer import SirenTrainer
    m = modules.SingleBVPNet(in_features=2, out_features=1, num_hidden_layers=1)
    with pytest.raises(ValueError, match="1024"):
        SirenTrainer([m] * 1025, 16)
