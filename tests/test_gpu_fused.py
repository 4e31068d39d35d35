"""Whole-MLP fused forward (csrc/mlp_fused_pair.cu; bf16 value path) through siren_mlp: deep nets stay on the fused
kernels, and first-layer arguments of a few hundred radians agree with fp64.  The value path's shapes, entries and
gradients are tested against fp64 per element in tests/test_gpu_value_path.py.

Tolerance: the bf16 mode's documented bound (DESIGN.md), rel-L2 <= 2e-2 against the fp64 oracle.
"""
import numpy as np
import pytest
import torch

from oracle import siren_oracle as so
from tests.helpers import rel_l2

pytestmark = pytest.mark.gpu

TOL = 2e-2


def _params(d, n_hidden, o, tasks, per_task, seed):
    Ws, bs = so.make_params(d, 256, n_hidden, o, seed=seed, tasks=tasks if per_task else 0)
    return [w.astype(np.float32) for w in Ws], [b.astype(np.float32) for b in bs]


def _run(x, Ws, bs):
    from siren_mri_b200 import functional as F
    with torch.no_grad():
        return F.siren_mlp(torch.from_numpy(x).cuda(), [torch.from_numpy(w).cuda() for w in Ws],
                           [torch.from_numpy(b).cuda() for b in bs], w0=30.0, precision="bf16").cpu().numpy()


def _oracle(x, Ws, bs):
    return so.siren_forward(x.astype(np.float64), [w.astype(np.float64) for w in Ws],
                            [b.astype(np.float64) for b in bs], 30.0, order=0)[0]


def test_deep_nets_run_on_the_fused_kernels():
    """Five to eight hidden layers (the MRI scripts use 5 and 6) stay on the whole-MLP kernels: one forward launch."""
    import ctypes
    from siren_mri_b200 import _lib
    lib = _lib.load()
    Ws, bs = _params(2, 5, 1, 1, False, seed=21)
    x = so.make_coords(1, 512, 2, seed=2)
    yo = _oracle(x, Ws, bs)
    lib.siren_b200_profile_begin()
    y = _run(x, Ws, bs)
    buf = ctypes.create_string_buffer(1 << 14)
    lib.siren_b200_profile_end(buf, len(buf))
    names = [ln.split()[0] for ln in buf.value.decode().strip().splitlines()]
    assert "mlp_fused_fwd" in names and "hidden_fwd" not in names, names
    assert rel_l2(y, yo) < TOL


def test_large_argument_sine():
    """First-layer arguments of a few hundred radians (wide coordinate range): the fused kernel hands them
    to the SFU without an explicit argument reduction; it must still agree with fp64."""
    Ws, bs = _params(2, 3, 1, 1, False, seed=4)
    x = (so.make_coords(1, 2048, 2, seed=3) * 12.0).astype(np.float32)     # |w0 x W0| up to ~360 rad
    yo = _oracle(x, Ws, bs)
    y_f = _run(x, Ws, bs)
    assert rel_l2(y_f, yo) < TOL, rel_l2(y_f, yo)
