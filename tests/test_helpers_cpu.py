"""The chunked fp64 oracle the BASELINE-size GPU tests use equals one unchunked oracle call."""
import numpy as np
import pytest

from oracle import siren_oracle as so
from tests.helpers import oracle_chunked, rel_l2, rel_l2_per_task


@pytest.mark.parametrize("tasks,per_task,order", [(1, False, 0), (3, True, 0), (2, False, 2), (2, True, 1)])
def test_oracle_chunked_equals_unchunked(tasks, per_task, order):
    d, o, n = 2, 1, 300
    Ws, bs = so.make_params(d, 256, 2, o, seed=1, tasks=tasks if per_task else 0)
    x = so.make_coords(tasks, n, d, seed=2)
    rng = np.random.default_rng(3)
    gy = rng.standard_normal((tasks, n, o))
    gJ = rng.standard_normal((tasks, n, o, d)) if order >= 1 else None
    gD = rng.standard_normal((tasks, n, o, d)) if order >= 2 else None
    W64 = [w.astype(np.float64) for w in Ws]
    b64 = [b.astype(np.float64) for b in bs]
    y, J, D, cache = so.siren_forward(x.astype(np.float64), W64, b64, 30.0, order)
    dW, db, _ = so.siren_backward(cache, W64, gy, gJ, gD)

    def adj(t0, t1, n0, n1, yc, Jc, Dc):
        return (gy[t0:t1, n0:n1], None if gJ is None else gJ[t0:t1, n0:n1], None if gD is None else gD[t0:t1, n0:n1])
    y2, J2, D2, dW2, db2 = oracle_chunked(x, Ws, bs, adj, order=order, chunk=77)
    assert rel_l2(y2, y) < 1e-13
    if order >= 1:
        assert rel_l2(J2, J) < 1e-13
    if order >= 2:
        assert rel_l2(D2, D) < 1e-13
    for l in range(len(Ws)):
        assert rel_l2(dW2[l], dW[l]) < 1e-12
        assert rel_l2(db2[l], db[l]) < 1e-12


@pytest.mark.parametrize("d,tasks,per_task", [(1, 1, False), (3, 4, True), (5, 2, False)])
def test_oracle_chunked_gx_equals_unchunked(d, tasks, per_task):
    """with_gx: the coordinate gradient, dW and db of the chunked walk are those of one unchunked call, and the first
    five results are what the call without with_gx returns."""
    o, n = 2, 203
    Ws, bs = so.make_params(d, 256, 2, o, seed=5, tasks=tasks if per_task else 0)
    x = so.make_coords(tasks, n, d, seed=6)
    gy = np.random.default_rng(7).standard_normal((tasks, n, o)) / n
    W64 = [w.astype(np.float64) for w in Ws]
    b64 = [b.astype(np.float64) for b in bs]
    y, _, _, cache = so.siren_forward(x.astype(np.float64), W64, b64, 30.0, 0)
    dW, db, gx = so.siren_backward(cache, W64, gy)

    def adj(t0, t1, n0, n1, yc, Jc, Dc):
        return gy[t0:t1, n0:n1], None, None
    res = oracle_chunked(x, Ws, bs, adj, chunk=50, with_gx=True)
    assert len(res) == 6
    y2, _, _, dW2, db2, gx2 = res
    assert gx2.shape == (tasks, n, d) and gx2.dtype == np.float64
    assert rel_l2_per_task(gx2, gx) < 1e-13
    assert np.abs(gx2 - gx).max() < 1e-13 * np.abs(gx).max()
    assert rel_l2(y2, y) < 1e-13
    for l in range(len(Ws)):
        assert rel_l2(dW2[l], dW[l]) < 1e-12
        assert rel_l2(db2[l], db[l]) < 1e-12
    plain = oracle_chunked(x, Ws, bs, adj, chunk=50)
    assert len(plain) == 5
    for a, b in zip(plain, res[:5]):
        if a is None:
            assert b is None
        elif isinstance(a, list):
            assert all(np.array_equal(u, v) for u, v in zip(a, b))
        else:
            assert np.array_equal(a, b)


def test_rel_l2_per_task_is_the_worst_task():
    rng = np.random.default_rng(4)
    ref = rng.standard_normal((40, 8, 5))
    got = ref.copy()
    assert rel_l2_per_task(got, ref) == 0.0
    got[17, :2] *= 1.05                 # one task, two of its rows 5 % off
    own = rel_l2(got[17], ref[17])
    assert rel_l2_per_task(got, ref) == own
    assert 5e-3 < own < 5e-2
    assert rel_l2(got, ref) < own / 5   # over the whole tensor the same error looks sqrt(40) times smaller
    with pytest.raises(AssertionError):
        rel_l2_per_task(got[:, :4], ref)
