"""Shared helpers for the parity tests (numpy side)."""
import json
import os

import numpy as np

from oracle import siren_oracle as so

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name, tag="f64"):
    return dict(np.load(os.path.join(GOLDEN, "%s_%s.npz" % (name, tag)), allow_pickle=False))


def rel_l2(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    den = np.sqrt((b * b).sum())
    return float(np.sqrt(((a - b) ** 2).sum()) / max(den, 1e-300))


def rel_l2_per_task(a, b):
    """Largest rel_l2 over the leading (task) axis: one task's gradient wrong by a few percent is a few percent here,
    where over the whole [tasks, ...] tensor it shrinks by about sqrt(tasks)."""
    a = np.asarray(a)
    b = np.asarray(b)
    assert a.shape == b.shape and a.ndim >= 1, (a.shape, b.shape)
    return max(rel_l2(a[t], b[t]) for t in range(a.shape[0]))


def log_errors(case, **vals):
    """Append the measured errors of a case to the JSON-lines file SIREN_TEST_LOG names (if it is set)."""
    path = os.environ.get("SIREN_TEST_LOG")
    if path:
        with open(path, "a") as f:
            f.write(json.dumps(dict(case=case, **{k: float(v) for k, v in vals.items()})) + "\n")


def sample(a, stride=97):
    return np.ascontiguousarray(np.asarray(a).reshape(-1)[::stride])


def check_grads(prefix, g, dWs, dbs, tol):
    """Compare full oracle/CUDA gradients with the sampled golden record."""
    worst = 0.0
    for l in range(len(dWs)):
        key = "%s_dW%d" % (prefix, l)
        if key in g:
            e = rel_l2(dWs[l], g[key])
        else:
            e = rel_l2(sample(dWs[l]), g[key + "_sample"])
            l2 = float(np.sqrt((np.asarray(dWs[l], np.float64) ** 2).sum()))
            e = max(e, abs(l2 - float(g[key + "_l2"])) / max(float(g[key + "_l2"]), 1e-300))
        worst = max(worst, e)
        assert e <= tol, "%s: rel err %.3e > %.1e" % (key, e, tol)
        ref_b = g["%s_db%d" % (prefix, l)]
        if np.abs(ref_b).max() == 0:
            assert np.abs(dbs[l]).max() <= 1e-12 + tol
        else:
            e = rel_l2(dbs[l], ref_b)
            worst = max(worst, e)
            assert e <= tol, "%s_db%d: rel err %.3e > %.1e" % (prefix, l, e, tol)
    return worst


def case_inputs(g, tasks=0):
    d, o, n, seed = int(g["d"]), int(g["o"]), int(g["n"]), int(g["seed"])
    Ws, bs = so.make_params(d, 256, 3, o, seed=seed, tasks=tasks)
    x = so.make_coords(max(tasks, 1), n, d, seed=seed + 100)
    return d, o, n, Ws, bs, x


def loss_adjoints_gradmse(J, gt_grad):
    """dL/dJ for loss_functions.gradients_mse (loss_functions.py:330-335)."""
    g = so.gradient(J)
    T, N = g.shape[:2]
    gg = 2.0 * (g - gt_grad) / (T * N)
    return np.broadcast_to(gg[..., None, :], J.shape).copy()


def loss_adjoints_lapmse(D, gt_lap):
    """dL/dD for loss_functions.laplace_mse (loss_functions.py:350-355)."""
    lap = so.laplace(D)
    gl = 2.0 * (lap - gt_lap) / lap.size
    return np.broadcast_to(gl[..., None], D.shape).copy() * (np.arange(D.shape[-2]) == 0)[:, None]


def oracle_chunked(x, Ws, bs, gy_fn, order=0, w0=30.0, chunk=32768):
    """fp64 oracle at BASELINE sizes without holding every plane at once: rows are independent through the
    forward and the input-gradient chain, and dW / db are sums over rows, so the batch is walked in chunks of
    ``chunk`` coordinates per task.  ``gy_fn(t0, t1, n0, n1, y, J, D) -> (gy, gJ, gD)`` supplies the output
    adjoints of a chunk (tasks t0:t1, coordinates n0:n1).  Returns ``(y, J, D, dWs, dbs)`` like one call of
    so.siren_forward + so.siren_backward would."""
    x = np.asarray(x)
    T, N, d = x.shape
    per_task = Ws[0].ndim == 3
    W64 = [np.asarray(w, np.float64) for w in Ws]
    b64 = [np.asarray(b, np.float64) for b in bs]
    o = W64[-1].shape[-2]
    y = np.empty((T, N, o), np.float64)
    J = np.empty((T, N, o, d), np.float64) if order >= 1 else None
    D = np.empty((T, N, o, d), np.float64) if order >= 2 else None
    dWs = [np.zeros_like(w) for w in W64]
    dbs = [np.zeros_like(b) for b in b64]
    for t in range(T):
        Wt = [w[t:t + 1] for w in W64] if per_task else W64
        bt = [b[t:t + 1] for b in b64] if per_task else b64
        for n0 in range(0, N, chunk):
            n1 = min(N, n0 + chunk)
            yc, Jc, Dc, cache = so.siren_forward(x[t:t + 1, n0:n1].astype(np.float64), Wt, bt, w0, order)
            y[t:t + 1, n0:n1] = yc
            if order >= 1:
                J[t:t + 1, n0:n1] = Jc
            if order >= 2:
                D[t:t + 1, n0:n1] = Dc
            gy, gJ, gD = gy_fn(t, t + 1, n0, n1, yc, Jc, Dc)
            dW, db, _ = so.siren_backward(cache, Wt, gy, gJ, gD)
            for l in range(len(W64)):
                if per_task:
                    dWs[l][t:t + 1] += dW[l]
                    dbs[l][t:t + 1] += db[l]
                else:
                    dWs[l] += dW[l]
                    dbs[l] += db[l]
    return y, J, D, dWs, dbs
