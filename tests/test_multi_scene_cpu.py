"""CPU checks of the multi-scene trainer's host side: the stacked flat layout and the scene checks."""
import pytest
import torch

from siren_mri_b200.optim import flatten_parameters_stacked, stacked_segments


def test_stacked_layout_and_segment_table():
    torch.manual_seed(0)
    shapes = [(8, 2), (8,), (8, 8), (8,), (1, 8), (1,)]
    T = 3
    models = [[torch.nn.Parameter(torch.randn(s)) for s in shapes] for _ in range(T)]
    before = [[p.detach().clone() for p in ps] for ps in models]
    segs, n = stacked_segments(shapes, T)
    # the segments tile the buffer, one [T, *shape] block per parameter, in parameter order
    end = 0
    for (off, k), s in zip(segs, shapes):
        assert off == end and k == torch.Size(s).numel()
        end += T * k
    assert end == n == T * sum(torch.Size(s).numel() for s in shapes)
    flat, grad, stacked, stacked_grad = flatten_parameters_stacked(models)
    assert flat.numel() == grad.numel() == n and not grad.any()
    for j, ((off, k), s) in enumerate(zip(segs, shapes)):
        assert stacked[j].shape == (T,) + s and stacked_grad[j].shape == (T,) + s
        assert stacked[j].data_ptr() == flat.data_ptr() + 4 * off
        for t in range(T):
            p = models[t][j]
            # model t's parameter is task slice t: same values, a view of the flat buffer and of the flat gradient
            assert torch.equal(p.detach(), before[t][j])
            assert p.data_ptr() == flat.data_ptr() + 4 * (off + t * k)
            assert p.grad.data_ptr() == grad.data_ptr() + 4 * (off + t * k)
            assert torch.equal(stacked[j][t], before[t][j])
    with torch.no_grad():
        models[1][2].add_(1.0)
    assert torch.equal(stacked[2][1], before[1][2] + 1.0)
    assert torch.equal(stacked[2][0], before[0][2])


def test_stacked_layout_rejects_other_shapes():
    a = [torch.nn.Parameter(torch.zeros(4, 2)), torch.nn.Parameter(torch.zeros(4))]
    b = [torch.nn.Parameter(torch.zeros(4, 3)), torch.nn.Parameter(torch.zeros(4))]
    with pytest.raises(ValueError):
        flatten_parameters_stacked([a, b])


def test_trainer_rejects_mismatched_scenes():
    """Checked before anything touches the device."""
    from siren_mri_b200 import modules
    from siren_mri_b200.trainer import SirenTrainer
    m = lambda **kw: modules.SingleBVPNet(in_features=2, out_features=1, **kw)  # noqa: E731
    with pytest.raises(ValueError, match="architecture"):
        SirenTrainer([m(), m(num_hidden_layers=2)], 64)
    with pytest.raises(ValueError, match="w0"):
        SirenTrainer([m(), m(w0=20)], 64)
    with pytest.raises(ValueError, match="precision"):
        SirenTrainer([m(precision="bf16"), m(precision="fp32")], 64)
    with pytest.raises(ValueError, match="image_mse"):
        SirenTrainer([m(), m()], 64, loss="sdf")
