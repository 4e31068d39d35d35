"""The oracle's coordinate jets and their reverse (so.siren_forward / so.siren_backward) against torch float64 autograd
on CPU, at the shapes the golden fixtures do not pin (those cover d in {2, 3}, d_out in {1, 3} and three hidden layers):
one input with five outputs and one hidden layer, three inputs with eight outputs and five hidden layers, and per-task
weights.  tests/test_gpu_jets.py holds the CUDA kernels to this oracle at these shapes."""
import numpy as np
import pytest
import torch

from oracle import siren_oracle as so
from tests.helpers import rel_l2

W0 = 30.0
TOL = 1e-10

SHAPES = {
    # name: d, n_hidden, d_out, tasks, per_task
    "d1_o5_h1": (1, 1, 5, 1, False),
    "d3_o8_h5": (3, 5, 8, 1, False),
    "d2_o3_h2_shared_t3": (2, 2, 3, 3, False),
    "d3_o2_h3_pertask_t4": (3, 3, 2, 4, True),
    "d1_o4_h4_pertask_t3": (1, 4, 4, 3, True),
}


def _torch_net(x, Ws, bs):
    """The sine MLP in torch float64, shared ([out, in]) or per-task ([T, out, in]) weights."""
    h = x
    for l, (W, b) in enumerate(zip(Ws, bs)):
        z = torch.matmul(h, W.transpose(-1, -2)) + b.unsqueeze(-2)
        h = z if l == len(Ws) - 1 else torch.sin(W0 * z)
    return h


def _torch_jets(x, Ws, bs, order):
    """y, J = dy_o/dx_k and D = d2y_o/dx_k^2 by (double) backward.  Rows are independent, so the gradient of a sum over
    rows is each row's own derivative."""
    y = _torch_net(x, Ws, bs)
    d = x.shape[-1]
    Jl, Dl = [], []
    for i in range(y.shape[-1]):
        gi = torch.autograd.grad(y[..., i].sum(), x, create_graph=True)[0]          # [T, N, d]
        Jl.append(gi)
        if order == 2:
            Dl.append(torch.stack([torch.autograd.grad(gi[..., k].sum(), x, create_graph=True)[0][..., k]
                                   for k in range(d)], -1))
    J = torch.stack(Jl, -2)
    D = torch.stack(Dl, -2) if order == 2 else None
    return y, J, D


def _case(name, order, seed):
    d, nh, o, T, per_task = SHAPES[name]
    Ws, bs = so.make_params(d, 256, nh, o, seed=seed, tasks=T if per_task else 0)
    x = so.make_coords(T, 9, d, seed=seed + 1).astype(np.float64)
    W64 = [w.astype(np.float64) for w in Ws]
    b64 = [b.astype(np.float64) for b in bs]
    rng = np.random.default_rng(seed + 2)
    gy = rng.standard_normal((T, 9, o))
    gJ = rng.standard_normal((T, 9, o, d)) / W0
    gD = rng.standard_normal((T, 9, o, d)) / W0 ** 2 if order == 2 else None
    return x, W64, b64, gy, gJ, gD


def _close(a, b, what):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    e = rel_l2(a, b)
    m = float(np.abs(a - b).max() / max(np.sqrt((b * b).mean()), 1e-300))
    assert e < TOL and m < TOL, (what, e, m)


@pytest.mark.parametrize("order", [1, 2])
@pytest.mark.parametrize("name", sorted(SHAPES))
def test_oracle_jets_match_autograd(name, order):
    x, W64, b64, gy, gJ, gD = _case(name, order, seed=70 + 10 * order)
    yo, Jo, Do, cache = so.siren_forward(x, W64, b64, W0, order)
    xt = torch.from_numpy(x).requires_grad_(True)
    Wt = [torch.from_numpy(w).requires_grad_(True) for w in W64]
    bt = [torch.from_numpy(b).requires_grad_(True) for b in b64]
    y, J, D = _torch_jets(xt, Wt, bt, order)
    _close(yo, y.detach().numpy(), "y")
    _close(Jo, J.detach().numpy(), "J")
    if order == 2:
        _close(Do, D.detach().numpy(), "D")
    # parameter gradients of sum(gy y + gJ J + gD D)
    s = (torch.from_numpy(gy) * y).sum() + (torch.from_numpy(gJ) * J).sum()
    if order == 2:
        s = s + (torch.from_numpy(gD) * D).sum()
    g = torch.autograd.grad(s, Wt + bt)
    dWs, dbs, _ = so.siren_backward(cache, W64, gy, gJ, gD)
    nl = len(W64)
    for l in range(nl):
        _close(dWs[l], g[l].numpy(), "dW%d" % l)
        _close(dbs[l], g[nl + l].numpy(), "db%d" % l)


@pytest.mark.parametrize("name", sorted(SHAPES))
def test_oracle_gx_is_the_value_adjoint(name):
    """The oracle's gx (what siren_b200_backward returns as gcoords) is the adjoint reaching the coordinates through the
    first pre-activation.  With gy alone nothing else reaches them, and it is autograd's coordinate gradient."""
    x, W64, b64, gy, _, _ = _case(name, 1, seed=90)
    _, _, _, cache = so.siren_forward(x, W64, b64, W0, 0)
    _, _, gx = so.siren_backward(cache, W64, gy)
    xt = torch.from_numpy(x).requires_grad_(True)
    y = _torch_net(xt, [torch.from_numpy(w) for w in W64], [torch.from_numpy(b) for b in b64])
    ref = torch.autograd.grad((torch.from_numpy(gy) * y).sum(), xt)[0]
    _close(gx, ref.numpy(), "gx")
    # the same with the jet streams carried (order 1 and 2) but given no adjoint
    for order in (1, 2):
        _, _, _, cache = so.siren_forward(x, W64, b64, W0, order)
        _, _, gx = so.siren_backward(cache, W64, gy)
        _close(gx, ref.numpy(), "gx order %d" % order)
