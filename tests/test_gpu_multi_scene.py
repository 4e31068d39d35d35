"""SirenTrainer over several scenes at once (T tasks with per-task weights): against T single-scene trainers, the
fp64 oracle and T reference loops with their own clip_grad_norm_ and Adam."""
import copy
import ctypes

import numpy as np
import pytest
import torch

from oracle import siren_oracle as so
from tests.helpers import rel_l2, rel_l2_per_task

pytestmark = pytest.mark.gpu

T = 5


def _scene_params(t):
    return so.make_params(2, 256, 3, 1, seed=101 + t)


def _models(T_, precision, backend="auto"):
    ms = []
    for t in range(T_):
        Ws, bs = _scene_params(t)
        m = _module(precision, backend)
        with torch.no_grad():
            for l in range(5):
                m.net.net[l][0].weight.copy_(torch.from_numpy(Ws[l]))
                m.net.net[l][0].bias.copy_(torch.from_numpy(bs[l]))
        ms.append(m)
    return ms


def _module(precision, backend="auto", layers=3):
    from siren_mri_b200 import modules
    return modules.SingleBVPNet(in_features=2, out_features=1, precision=precision, num_hidden_layers=layers,
                                backend=backend).cuda()


def _data(T_, n, seed=7):
    x = so.make_coords(T_, n, 2, seed=seed)
    gt = np.random.default_rng(seed + 1).uniform(-1, 1, size=(T_, n, 1)).astype(np.float32)
    return x, gt


def _task_grads(tr, flat_grad):
    """[T, per-task floats] from the stacked flat gradient: task t's slice of every parameter, in parameter order."""
    g = flat_grad.view(-1)
    out, off = [], 0
    for w, b in zip(tr.weights, tr.biases):
        for p in (w, b):
            k = p[0].numel()
            out.append(g[off:off + tr.tasks * k].view(tr.tasks, k))
            off += tr.tasks * k
    return torch.cat(out, dim=1).cpu().numpy()


def _oracle_snapshots(Ws, bs, x, gt, steps, lr=1e-4):
    """fp64 reference loop of one scene; weights after every step in ``steps``."""
    W = [w.astype(np.float64) for w in Ws]
    b = [v.astype(np.float64) for v in bs]
    mW = [np.zeros_like(w) for w in W]; vW = [np.zeros_like(w) for w in W]
    mb = [np.zeros_like(v) for v in b]; vb = [np.zeros_like(v) for v in b]
    snaps = {}
    for s in range(1, max(steps) + 1):
        y, _, _, cache = so.siren_forward(x.astype(np.float64), W, b, 30.0, 0)
        loss, gy = so.image_mse(y, gt.astype(np.float64))
        dW, db, _ = so.siren_backward(cache, W, gy)
        for l in range(len(W)):
            W[l], mW[l], vW[l] = so.adam_step(W[l], dW[l], mW[l], vW[l], s, lr=lr)
            b[l], mb[l], vb[l] = so.adam_step(b[l], db[l], mb[l], vb[l], s, lr=lr)
        if s in steps:
            snaps[s] = ([w.copy() for w in W], loss)
    return snaps


@pytest.mark.parametrize("n", [3000, 4700])
@pytest.mark.parametrize("graph", [False, True])
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_matches_separate_trainers(precision, graph, n):
    """One T-scene trainer against T single-scene trainers on the same scenes: y bit-equal, first-step gradients and
    losses to summation order, weights after 1 and 10 steps against the fp64 oracle (fp32) / the single trainers."""
    from siren_mri_b200.trainer import SirenTrainer
    x, gt = _data(T, n)
    models = _models(T, precision)
    singles = [SirenTrainer(copy.deepcopy(m), n, lr=1e-4, use_graph=graph) for m in models]
    tr = SirenTrainer(models, n, lr=1e-4, use_graph=graph)
    assert tr.loss.shape == (T,) and tuple(tr.y.shape) == (T, n, 1)
    tr.coords.copy_(torch.from_numpy(x))
    tr.gt.copy_(torch.from_numpy(gt))
    for t, s in enumerate(singles):
        s.coords.copy_(torch.from_numpy(x[t:t + 1]))
        s.gt.copy_(torch.from_numpy(gt[t:t + 1]))
    g, loss = tr.gradients()
    got = _task_grads(tr, g)
    for t, s in enumerate(singles):
        gs, ls = s.gradients()
        assert torch.equal(tr.y[t], s.y[0]), t          # the same arithmetic per row
        assert rel_l2(got[t], gs.cpu().numpy()) < 1e-5, (t, rel_l2(got[t], gs.cpu().numpy()))
        assert abs(float(loss[t]) - float(ls)) <= 1e-5 * abs(float(ls)), (t, float(loss[t]), float(ls))
    snaps = _oracle_snapshots_all(x, gt, (1, 10)) if precision == "fp32" and n == 3000 else None
    for steps in (1, 10):
        while tr.steps < steps:
            tr.step()
            for s in singles:
                s.step()
        torch.cuda.synchronize()
        single_loss = np.array([float(s.loss.item()) for s in singles])
        assert np.all(np.abs(tr.loss.cpu().numpy() - single_loss) <= 1e-4 * np.abs(single_loss)), (tr.loss, single_loss)
        for l in range(5):
            got_w = tr.weights[l].detach().cpu().numpy()
            sing_w = np.stack([s.weights[l].detach().cpu().numpy() for s in singles])
            W0 = np.stack([_scene_params(t)[0][l] for t in range(T)])
            assert rel_l2_per_task(got_w - W0, sing_w - W0) < 2e-2, (steps, l)
            if snaps is not None:
                ref = np.stack([snaps[t][steps][0][l] for t in range(T)])
                # the UPDATE (w - w0) per task: Adam's first steps are +-lr per element
                assert rel_l2_per_task(got_w - W0, ref - W0) < 2e-2, (steps, l, rel_l2_per_task(got_w - W0, ref - W0))
                assert rel_l2_per_task(got_w, ref) < 1e-4
        if snaps is not None:
            ref_loss = np.array([snaps[t][steps][1] for t in range(T)])
            assert np.all(np.abs(tr.loss.cpu().numpy() - ref_loss) < 1e-4 * np.abs(ref_loss)), (tr.loss, ref_loss)


_ORACLE = {}


def _oracle_snapshots_all(x, gt, steps):
    key = (x.shape, steps)      # the graph on / off cases share the scenes
    if key not in _ORACLE:
        _ORACLE[key] = [_oracle_snapshots(*_scene_params(t), x[t:t + 1], gt[t:t + 1], steps) for t in range(x.shape[0])]
    return _ORACLE[key]


def _clip_norms(x, gt, n):
    """Each scene's first-step gradient norm, through torch autograd on the composed model."""
    norms = []
    for t, m in enumerate(_models(x.shape[0], "fp32", "composed")):
        out = m({"coords": torch.from_numpy(x[t:t + 1]).cuda()})["model_out"]
        (((out - torch.from_numpy(gt[t:t + 1]).cuda()) ** 2).sum() / 16384.0).backward()
        norms.append(float(torch.sqrt(sum((p.grad ** 2).sum() for p in m.parameters()))))
    return norms


@pytest.mark.parametrize("acc,clip", [(1, "between"), (2, 0.0), (2, 0.05)])
def test_clip_and_accumulation_per_scene(acc, clip):
    """training.py:88-103 run for each scene alone (image_mse, backward of loss / acc, clip_grad_norm_ over THAT
    model's parameters after every micro-batch, Adam step every acc micro-batches) against one 3-scene trainer.
    'between': scene 0's targets are scaled so that its gradient norm is far above max_grad_norm, scene 1 stays below
    it -- one global norm would clip scene 1 as well."""
    from siren_mri_b200.trainer import SirenTrainer
    T_, n, batches = 3, 1500, 4
    xs, gts = zip(*[_data(T_, n, seed=40 + 3 * k) for k in range(batches)])
    gts = [g.copy() for g in gts]
    for g in gts:
        g[0] *= 50.0
    if clip == "between":
        norms = _clip_norms(xs[0], gts[0], n)
        clip = float(np.sqrt(norms[0] * norms[1]))
        assert norms[1] < 0.5 * clip and norms[0] > 2.0 * clip, (norms, clip)
    refs = _models(T_, "fp32", "composed")
    ref_losses = np.zeros((batches, T_))
    for t, ref in enumerate(refs):
        opt = torch.optim.Adam(lr=1e-4, params=ref.parameters())
        for k in range(batches):
            out = ref({"coords": torch.from_numpy(xs[k][t:t + 1]).cuda()})["model_out"]
            loss = ((out - torch.from_numpy(gts[k][t:t + 1]).cuda()) ** 2).sum() / 16384.0
            ref_losses[k, t] = float(loss.detach())
            (loss / acc).backward()
            if clip:
                torch.nn.utils.clip_grad_norm_(ref.parameters(), max_norm=clip)
            if (k + 1) % acc == 0:
                opt.step()
                opt.zero_grad()
    models = _models(T_, "fp32")
    tr = SirenTrainer(models, n, lr=1e-4, max_grad_norm=clip, precision="fp32")
    got = np.zeros((batches, T_))
    for k in range(batches):
        tr.coords.copy_(torch.from_numpy(xs[k]))
        tr.gt.copy_(torch.from_numpy(gts[k]))
        tr.step(update=(k + 1) % acc == 0, accumulation_steps=acc)
        got[k] = tr.loss.cpu().numpy() * acc
    torch.cuda.synchronize()
    assert tr.steps == batches // acc
    assert np.all(np.abs(got - ref_losses) < 2e-4 * np.abs(ref_losses)), (ref_losses, got)
    for t, (ref, m) in enumerate(zip(refs, models)):
        for pr, pn in zip(ref.parameters(), m.parameters()):
            du = (pn.detach() - pr.detach()).norm() / pr.detach().norm()
            assert float(du) < 1e-3, (t, float(du))


def _profiled_names(tr):
    from siren_mri_b200 import _lib
    lib = _lib.load()
    torch.cuda.synchronize()
    lib.siren_b200_profile_begin()
    tr.step()
    torch.cuda.synchronize()
    buf = ctypes.create_string_buffer(1 << 14)
    lib.siren_b200_profile_end(buf, len(buf))
    return [ln.split()[0] for ln in buf.value.decode().strip().splitlines()], \
        sum(int(ln.split()[1]) for ln in buf.value.decode().strip().splitlines())


@pytest.mark.parametrize("clip", [0.0, 1.0])
def test_launch_budget(clip):
    """A non-graph 8-scene step on the one-kernel path: mlp_fused_step, wgrad and the per-task Adam (and the per-task
    norm pass with clipping) -- the launches of a single-scene step."""
    from siren_mri_b200.trainer import SirenTrainer
    n = 4096
    single = SirenTrainer(_module("bf16"), n, lr=1e-4, max_grad_norm=clip, use_graph=False)
    tr = SirenTrainer([_module("bf16") for _ in range(8)], n, lr=1e-4, max_grad_norm=clip, use_graph=False)
    x, gt = _data(8, n)
    tr.coords.copy_(torch.from_numpy(x))
    tr.gt.copy_(torch.from_numpy(gt))
    tr.step()
    names, launches = _profiled_names(tr)
    _, single_launches = _profiled_names(single)
    assert "mlp_fused_step" in names and "adam_step_tasks" in names, names
    assert ("task_norms" in names) == (clip > 0), names
    assert launches <= single_launches == (4 if clip else 3), (names, launches, single_launches)


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_weight_copies_match_prepare_weights(precision):
    """After 10 steps the workspace's weight copies, kept current by the per-task Adam, equal what prepare_weights
    writes from the current parameters: a forward on either gives bit-equal y."""
    from siren_mri_b200 import _lib
    from siren_mri_b200.trainer import SirenTrainer
    n = 3000
    x, gt = _data(T, n)
    tr = SirenTrainer(_models(T, precision), n, lr=1e-3)
    tr.coords.copy_(torch.from_numpy(x))
    tr.gt.copy_(torch.from_numpy(gt))
    for _ in range(10):
        tr.step()
    lib, P = tr.lib, _lib.dptr
    stream = torch.cuda.current_stream().cuda_stream
    ws2 = torch.zeros_like(tr.ws)
    _lib.check(lib.siren_b200_prepare_weights(tr.desc, tr._w_ptrs, P(ws2), stream), "prepare_weights")
    ys = []
    for ws in (tr.ws, ws2):
        y = torch.empty_like(tr.y)
        _lib.check(lib.siren_b200_forward_prepared(tr.desc, P(tr.coords), tr._w_ptrs, tr._b_ptrs, P(y), None, None,
                                                   P(ws), stream), "forward_prepared")
        ys.append(y)
    torch.cuda.synchronize()
    assert torch.isfinite(ys[0]).all()
    assert torch.equal(ys[0], ys[1])


def test_models_are_views():
    """Each model stays a usable module on its task's slice: its own forward gives the trainer's y, a
    load_state_dict into it (+ refresh_weights) changes that task's gradient only, and the host entries return the
    same per-scene losses as tr.loss."""
    from siren_mri_b200.trainer import SirenTrainer
    n, T_ = 2048, 3
    x, gt = _data(T_, n)
    models = _models(T_, "bf16")
    tr = SirenTrainer(models, n, lr=1e-4)
    tr.coords.copy_(torch.from_numpy(x))
    tr.gt.copy_(torch.from_numpy(gt))
    for _ in range(5):
        tr.step()
    g0, _ = tr.gradients()
    with torch.no_grad():
        for t, m in enumerate(models):
            y = m({"coords": tr.coords[t:t + 1]})["model_out"]
            assert rel_l2(y.cpu().numpy(), tr.y[t:t + 1].cpu().numpy()) < 1e-2, t
    fresh = _module("bf16")
    models[1].load_state_dict(fresh.state_dict())
    tr.refresh_weights()
    g1, _ = tr.gradients()
    a, b = _task_grads(tr, g0), _task_grads(tr, g1)
    assert rel_l2(b[1], a[1]) > 1e-1
    for t in (0, 2):
        assert rel_l2(b[t], a[t]) < 1e-5, t
    xs, gs = torch.from_numpy(x).pin_memory(), torch.from_numpy(gt).pin_memory()
    losses = tr.step_from_host(xs, gs)
    assert len(losses) == T_ and losses == tr.loss.tolist()
    h = tr.submit_from_host(xs, gs)
    got = h.result()
    torch.cuda.synchronize()
    assert len(got) == T_ and got == tr.loss.tolist()


def test_rejected_inputs(monkeypatch):
    from siren_mri_b200 import _lib
    from siren_mri_b200.trainer import SirenTrainer
    with pytest.raises(ValueError):
        SirenTrainer([_module("bf16"), _module("bf16", layers=2)], 1024)
    with pytest.raises(ValueError):
        SirenTrainer([_module("bf16"), _module("fp32")], 1024)
    with pytest.raises(ValueError):
        SirenTrainer([_module("fp32") for _ in range(2)], 1024, loss="laplace_mse")
    monkeypatch.setattr(torch.distributed, "get_world_size", lambda group=None: 2)
    with pytest.raises(ValueError):
        SirenTrainer([_module("bf16") for _ in range(2)], 1024, process_group=object())
    tr = SirenTrainer([_module("bf16") for _ in range(2)], 1024, process_group=object(), distributed=False)
    monkeypatch.undo()
    # the C entries refuse parameters that do not tile the flat buffer
    lib, P, opt = tr.lib, _lib.dptr, tr.opt
    stream = torch.cuda.current_stream().cuda_stream
    args = lambda w, b, n: (tr.desc, w, b, P(opt.p), P(opt.g), P(opt.m), P(opt.v), n, 1e-4, 0.9, 0.999, 1e-8,  # noqa
                            0.0, P(opt.state), None, None, 0.0, P(opt.task_sumsq), P(tr.task_loss), None, None, stream)
    n = opt.p.numel()
    assert lib.siren_b200_adam_step_tasks(*args(tr._w_ptrs, tr._b_ptrs, n)) == 0
    torch.cuda.synchronize()
    assert lib.siren_b200_adam_step_tasks(*args(tr._w_ptrs, tr._b_ptrs, n + 4)) == 2
    shifted = _lib.ptr_array_raw([b.data_ptr() + (4 if l == 2 else 0) for l, b in enumerate(tr.biases)])
    assert lib.siren_b200_adam_step_tasks(*args(tr._w_ptrs, shifted, n)) == 2
    overlap = _lib.ptr_array_raw([tr.weights[0].data_ptr()] + [w.data_ptr() for w in tr.weights[1:]])
    overlap[3] = tr.weights[2].data_ptr()
    assert lib.siren_b200_adam_step_tasks(*args(overlap, tr._b_ptrs, n)) == 2
    assert lib.siren_b200_clip_grad_tasks(tr.desc, tr._dw_ptrs, tr._db_ptrs, P(opt.g), n - 1, 1.0, P(opt.state), None,
                                          None, 0.0, P(opt.task_sumsq), P(tr.task_loss), None, 0, stream) == 2


def _arch_models(arch, T_, precision, seed=301):
    from siren_mri_b200 import modules
    d_in, nh, d_out = arch
    ms = []
    for t in range(T_):
        Ws, bs = so.make_params(d_in, 256, nh, d_out, seed=seed + t)
        m = modules.SingleBVPNet(in_features=d_in, out_features=d_out, precision=precision,
                                 num_hidden_layers=nh).cuda()
        with torch.no_grad():
            for l in range(nh + 2):
                m.net.net[l][0].weight.copy_(torch.from_numpy(Ws[l]))
                m.net.net[l][0].bias.copy_(torch.from_numpy(bs[l]))
        ms.append(m)
    return ms


# (arch, scenes, n, precision, graph): the benchmarked 64 x 4096 (tools/bench_multi_scene.py); the fused forward with
# an outermost linear it does not fuse (two-launch step); a first layer wider than 4 inputs (prep_first every step);
# the fp32 per-layer path
MORE = {"bench-64x4096": ((2, 3, 1), 64, 4096, "bf16", True), "3x5x3-bf16": ((3, 5, 3), 3, 1500, "bf16", False),
        "16x2x2-bf16": ((16, 2, 2), 3, 1500, "bf16", False), "3x2x3-fp32": ((3, 2, 3), 3, 1500, "fp32", False)}


@pytest.mark.parametrize("case", list(MORE))
def test_matches_separate_trainers_more_shapes(case):
    """test_matches_separate_trainers at the shapes the benchmark and the other kernels reach: y bit-equal to the
    single-scene trainers', per-task gradients and losses to 1e-5, weights after 5 steps."""
    from siren_mri_b200.trainer import SirenTrainer
    from tests.helpers import log_errors
    arch, T_, n, precision, graph = MORE[case]
    x = so.make_coords(T_, n, arch[0], seed=17)
    gt = np.random.default_rng(18).uniform(-1, 1, size=(T_, n, arch[2])).astype(np.float32)
    models = _arch_models(arch, T_, precision)
    W0 = [np.stack([m.net.net[l][0].weight.detach().cpu().numpy() for m in models]) for l in range(arch[1] + 2)]
    singles = [SirenTrainer(copy.deepcopy(m), n, lr=1e-4, use_graph=graph) for m in models]
    tr = SirenTrainer(models, n, lr=1e-4, use_graph=graph)
    tr.coords.copy_(torch.from_numpy(x))
    tr.gt.copy_(torch.from_numpy(gt))
    for t, s in enumerate(singles):
        s.coords.copy_(torch.from_numpy(x[t:t + 1]))
        s.gt.copy_(torch.from_numpy(gt[t:t + 1]))
    g, loss = tr.gradients()
    got = _task_grads(tr, g)
    dy, dg, dl = 0.0, 0.0, 0.0
    for t, s in enumerate(singles):
        gs, ls = s.gradients()
        dy = max(dy, float((tr.y[t] - s.y[0]).abs().max()))
        dg = max(dg, rel_l2(got[t], gs.cpu().numpy()))
        dl = max(dl, abs(float(loss[t]) - float(ls)) / abs(float(ls)))
    log_errors("more_shapes:" + case, y_max_abs=dy, grad_rel_l2=dg, loss_rel=dl)
    assert dy == 0.0, (case, dy)           # the same arithmetic per row
    assert dg < 1e-5 and dl < 1e-5, (case, dg, dl)
    for _ in range(5):
        tr.step()
        for s in singles:
            s.step()
    torch.cuda.synchronize()
    single_loss = np.array([float(s.loss.item()) for s in singles])
    assert np.all(np.abs(tr.loss.cpu().numpy() - single_loss) <= 1e-4 * np.abs(single_loss)), (tr.loss, single_loss)
    for l in range(arch[1] + 2):
        got_w = tr.weights[l].detach().cpu().numpy()
        sing_w = np.stack([s.weights[l].detach().cpu().numpy() for s in singles])
        err = rel_l2_per_task(got_w - W0[l], sing_w - W0[l])
        log_errors("more_shapes_w:%s-l%d" % (case, l), update_rel_l2=err)
        assert err < 2e-2, (case, l, err)
