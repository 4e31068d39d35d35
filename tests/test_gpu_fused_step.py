"""The one-kernel bf16 training step (forward, loss gradient and input-gradient chain: mlp_fused_step.cu) against the
two-launch step it replaces (SIREN_FUSED_STEP=0: mlp_fused_fwd + mlp_fused_bwd) on the same seeded inputs.

Both run the same arithmetic in the same order, so y and gy are bit-equal; the loss sum, the bias / first-layer /
outermost gradients the chain sums per warp and every weight gradient's atomics differ only in summation order."""
import numpy as np
import pytest
import torch

from oracle import siren_oracle as so
from tests.helpers import rel_l2

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
