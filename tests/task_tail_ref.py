"""float64 restatement of the optimizer tail of T stacked networks (siren_b200_adam_step_tasks,
siren_b200_clip_grad_tasks), in torch on any device, and the flat layouts the tests drive it with.

A network of ``(d_in, n_hidden, d_out)`` has L = n_hidden + 2 linear layers; parameter W[l] is [T, out, in] and b[l]
[T, out], each one segment of the flat buffer.  The entries accept the segments in any order."""
import numpy as np
import torch

from siren_mri_b200.optim import stacked_segments

H = 256
ORDERS = ("trainer", "reversed", "biases_first", "random")


def param_shapes(arch):
    """[(kind, layer, shape)] in the trainer's order W0, b0, W1, b1, ..."""
    d_in, n_hidden, d_out = arch
    L = n_hidden + 2
    out = []
    for l in range(L):
        o, i = (d_out if l == L - 1 else H), (d_in if l == 0 else H)
        out += [("W", l, (o, i)), ("b", l, (o,))]
    return out


def layout(arch, T, order):
    """The segments of the flat buffer in the given order: dicts with kind, layer, per (floats per task), off, and
    hidden (the hidden layer whose 16-bit copies the segment feeds, or -1); and the buffer's length."""
    params = param_shapes(arch)
    idx = list(range(len(params)))
    if order == "reversed":
        idx = idx[::-1]
    elif order == "biases_first":
        # the outermost bias (d_out floats per task) first: with d_out * T odd every later segment starts off a
        # multiple of 4, so float4s straddle every boundary, hidden weights included
        biases = [j for j in idx if params[j][0] == "b"]
        idx = [biases[-1]] + biases[:-1] + [j for j in idx if params[j][0] == "W"]
    elif order == "random":
        idx = [int(j) for j in np.random.default_rng(20261021).permutation(len(params))]
    elif order != "trainer":
        raise ValueError(order)
    segs, n = stacked_segments([params[j][2] for j in idx], T)
    n_hidden = arch[1]
    out = []
    for j, (off, per) in zip(idx, segs):
        kind, l, shape = params[j]
        out.append(dict(kind=kind, layer=l, shape=shape, per=per, off=off,
                        hidden=l - 1 if kind == "W" and 1 <= l <= n_hidden else -1))
    return out, n


def views(flat, segs, T):
    """[T, per] view of every segment of ``flat``."""
    return [flat[s["off"]:s["off"] + T * s["per"]].view(T, s["per"]) for s in segs]


def per_element(per_task, segs, T):
    """Expand a [T] vector to the flat layout: element i gets the value of the task that owns it."""
    out = torch.empty(sum(T * s["per"] for s in segs), dtype=per_task.dtype, device=per_task.device)
    for s, v in zip(segs, views(out, segs, T)):
        v.copy_(per_task[:, None].expand(T, s["per"]))
    return out


def task_sumsq(g, segs, T):
    """Each task's squared gradient norm over its slice of every segment (float64)."""
    acc = torch.zeros(T, dtype=torch.float64, device=g.device)
    for v in views(g, segs, T):
        acc += (v.double() ** 2).sum(1)
    return acc


def clip_coefs(g, segs, T, max_norm):
    """clip_grad_norm_ of every task on its own: min(1, max_norm / (|g_t| + 1e-6)); ones without clipping."""
    sq = task_sumsq(g, segs, T)
    if not max_norm > 0:
        return torch.ones(T, dtype=torch.float64, device=g.device), sq
    return torch.clamp(max_norm / (torch.sqrt(sq) + 1e-6), max=1.0), sq


def task_losses(y, gt, weight):
    """image_mse of every task: weight * sum (y - gt)^2 over its n * d_out values."""
    T = y.shape[0]
    d = y.double().reshape(T, -1) - gt.double().reshape(T, -1)
    return (d * d).sum(1) * weight


def moment_beta(beta):
    """The beta the kernels multiply the moments by: the fp32 rounding of the double argument (their bias corrections
    use the double).  torch's fp32 Adam rounds beta and 1 - beta separately; at beta2 = 0.999 the two (1 - beta2)
    differ by 1.3e-5 of the (1 - beta2) g^2 term."""
    return float(np.float32(beta))


def adam(p, g, m, v, coef, step, lr, b1, b2, eps, mb1=None, mb2=None):
    """One Adam step on the clipped gradient coef * g (coef per element), float64; the bias corrections
    1 - beta ** step in double, as torch.optim.Adam computes them.  mb1 / mb2: the moment betas (default b1 / b2).
    Returns (p, m, v)."""
    mb1 = b1 if mb1 is None else mb1
    mb2 = b2 if mb2 is None else mb2
    gc = g.double() * coef
    m1 = mb1 * m.double() + (1.0 - mb1) * gc
    v1 = mb2 * v.double() + (1.0 - mb2) * gc * gc
    bc1 = 1.0 - b1 ** step
    bc2 = 1.0 - b2 ** step
    p1 = p.double() - (lr / bc1) * (m1 / (torch.sqrt(v1) / np.sqrt(bc2) + eps))
    return p1, m1, v1


def running_pow(beta, k):
    """beta ** k as the kernels keep it: a running product in double, one multiplication per step."""
    q = 1.0
    for _ in range(k):
        q *= beta
    return q


def ulp32(x):
    """The spacing of fp32 numbers at |x| (float64 tensor in, float64 out)."""
    _, e = torch.frexp(x.abs().clamp(min=2.0 ** -126))
    return torch.ldexp(torch.ones_like(x), e - 24)
