"""The float64 reference of the per-task optimizer tail (tests/task_tail_ref.py) against the numpy oracle, and its
layouts against the segment table the C entries derive.  Runs without a GPU."""
import numpy as np
import pytest
import torch

from oracle import siren_oracle as so
from tests import task_tail_ref as ref


@pytest.mark.parametrize("order", ref.ORDERS)
@pytest.mark.parametrize("arch,T", [((1, 1, 1), 1), ((3, 2, 3), 7), ((16, 8, 8), 2)])
def test_layout_tiles_the_buffer(arch, T, order):
    segs, n = ref.layout(arch, T, order)
    assert len(segs) == 2 * (arch[1] + 2) <= 20
    ends = sorted((s["off"], s["off"] + T * s["per"]) for s in segs)
    assert ends[0][0] == 0 and ends[-1][1] == n
    assert all(a[1] == b[0] for a, b in zip(ends, ends[1:]))
    assert sorted((s["kind"], s["layer"]) for s in segs) == sorted((k, l) for k, l, _ in ref.param_shapes(arch))
    assert [s["hidden"] for s in segs if s["hidden"] >= 0] == [s["layer"] - 1 for s in segs if s["hidden"] >= 0]
    if order == "biases_first" and arch[2] * T % 2:
        assert all(s["off"] % 4 for s in segs[1:]), [s["off"] for s in segs]


def _grads(arch, T, seed):
    rng = np.random.default_rng(seed)
    return [[rng.standard_normal(shape) * 2.0 ** (t / 128) for _, _, shape in ref.param_shapes(arch)]
            for t in range(T)]


@pytest.mark.parametrize("max_norm", [0.0, "median"])
def test_reference_matches_oracle(max_norm):
    """Per task: clip coefficient = oracle.clip_coef over that task's parameters, Adam = oracle.adam_step, loss =
    oracle.image_mse scaled; in every parameter order."""
    arch, T, step, lr = (3, 1, 2), 5, 4, 1e-3
    b1, b2, eps = 0.9, 0.999, 1e-8
    rng = np.random.default_rng(3)
    per_task = _grads(arch, T, 1)
    p_t = [[rng.uniform(-1, 1, g.shape) for g in gs] for gs in per_task]
    m_t = [[rng.standard_normal(g.shape) * 0.1 for g in gs] for gs in per_task]
    v_t = [[rng.uniform(0.5, 2.0, g.shape) for g in gs] for gs in per_task]
    norms = [so.clip_coef(gs, 1.0)[1] for gs in per_task]
    mn = float(np.median(norms)) if max_norm == "median" else 0.0
    for order in ref.ORDERS:
        segs, n = ref.layout(arch, T, order)
        flat = {k: torch.zeros(n, dtype=torch.float64) for k in "pgmv"}
        shapes = ref.param_shapes(arch)
        for s, vw in zip(segs, ref.views(flat["g"], segs, T)):
            j = shapes.index((s["kind"], s["layer"], s["shape"]))
            for name, src in (("p", p_t), ("g", per_task), ("m", m_t), ("v", v_t)):
                view = ref.views(flat[name], segs, T)[segs.index(s)]
                for t in range(T):
                    view[t] = torch.from_numpy(src[t][j].reshape(-1))
        coef, sq = ref.clip_coefs(flat["g"], segs, T, mn)
        p1, m1, v1 = ref.adam(flat["p"], flat["g"], flat["m"], flat["v"], ref.per_element(coef, segs, T), step, lr,
                              b1, b2, eps)
        for t in range(T):
            c, total = so.clip_coef(per_task[t], mn) if mn > 0 else (1.0, norms[t])
            assert abs(float(coef[t]) - c) <= 1e-15 * c
            assert abs(float(torch.sqrt(sq[t])) - total) <= 1e-12 * total
            for s in segs:
                j = shapes.index((s["kind"], s["layer"], s["shape"]))
                k = segs.index(s)
                po, mo, vo = so.adam_step(p_t[t][j], c * per_task[t][j], m_t[t][j], v_t[t][j], step, lr, b1, b2, eps)
                for got, want in ((p1, po), (m1, mo), (v1, vo)):
                    np.testing.assert_allclose(ref.views(got, segs, T)[k][t].numpy(), want.reshape(-1),
                                               rtol=1e-13, atol=1e-16)
        if mn > 0:
            assert (coef < 1).any() and (coef == 1).any()
    y = torch.from_numpy(rng.standard_normal((T, 37, 2)))
    gt = torch.from_numpy(rng.standard_normal((T, 37, 2)))
    got = ref.task_losses(y, gt, 0.25)
    for t in range(T):
        want, _ = so.image_mse(y[t].numpy(), gt[t].numpy(), weight=0.25)
        assert abs(float(got[t]) - want) <= 1e-13 * want


def test_moment_beta_and_running_pow():
    assert ref.moment_beta(0.5) == 0.5 and ref.moment_beta(0.9) == float(np.float32(0.9))
    assert ref.running_pow(0.9, 3) == 0.9 * 0.9 * 0.9
    # the running product of beta <= 0.5 underflows to exactly 0 (the case the kernels' bias correction must not
    # mistake for a fresh state); above 0.5 it sticks at the smallest subnormal
    assert ref.running_pow(0.5, 1074) == 2.0 ** -1074 and ref.running_pow(0.5, 1075) == 0.0
    assert ref.running_pow(0.3, 618) > 0.0 and ref.running_pow(0.3, 619) == 0.0
    x = torch.tensor([1.0, 0.75, -3.0, 1e-30], dtype=torch.float64)
    want = [float(np.spacing(np.float32(abs(v)))) for v in x.tolist()]
    assert ref.ulp32(x).tolist() == want
