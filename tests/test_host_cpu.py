"""CPU tests of the host side: C-ABI library loads and exports every declared symbol, the module
mirror keeps the reference's contracts, and the autograd wiring of the jet outputs (attach
Functions) reproduces the reference's double/triple-backward results."""
import ctypes
import os
import re
from collections import OrderedDict

import numpy as np
import pytest
import torch

from oracle import siren_oracle as so
from tests.helpers import GOLDEN, case_inputs, check_grads, load_golden, rel_l2

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_abi_library_loads_and_exports_every_declared_symbol():
    from siren_mri_b200 import _lib
    header = open(os.path.join(ROOT, "include", "siren_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(siren_b200_[a-z_0-9]+)\s*\(", header)))
    assert declared, "no declarations parsed"
    assert sorted(_lib.SYMBOLS) == declared
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert _lib.load().siren_b200_version() == 1


def test_desc_struct_matches_header_layout():
    from siren_mri_b200 import _lib
    # int,int,int,int,float,int,int,(pad),long,int,int -> 48 bytes on LP64
    assert ctypes.sizeof(_lib.SirenDesc) == 48
    assert _lib.SirenDesc.n_coords.offset == 32


def test_workspace_bytes_rejects_unsupported_shapes_without_gpu():
    from siren_mri_b200 import _lib
    lib = _lib.load()
    d = _lib.SirenDesc(2, 256, 3, 1, 30.0, 1, 0, 1000, 0, 0)
    assert lib.siren_b200_workspace_bytes(d) > 0
    d.hidden = 512
    assert lib.siren_b200_workspace_bytes(d) == 0
    assert b"hidden_features" in lib.siren_b200_last_error()
    d.hidden, d.deriv_order, d.d_in = 256, 2, 16
    assert lib.siren_b200_workspace_bytes(d) == 0


def test_get_subdict_semantics():
    from siren_mri_b200.meta import get_subdict
    d = OrderedDict([("net.0.weight", 1), ("net.0.bias", 2), ("net.10.weight", 3), ("other", 4), ("net.", 5)])
    assert list(get_subdict(d, "net").items()) == [("0.weight", 1), ("0.bias", 2), ("10.weight", 3)]
    assert list(get_subdict(d, "net.0").items()) == [("weight", 1), ("bias", 2)]
    assert get_subdict(None, "x") is None and get_subdict(d, "") is d and get_subdict(d, None) is d


def test_state_dict_keys_and_hypernetwork_contract_match_reference():
    from siren_mri_b200 import meta_modules, modules
    g = np.load(os.path.join(GOLDEN, "hypernet_contract.npz"))
    hypo = modules.SingleBVPNet(out_features=2, type="sine", in_features=16, hidden_features=256,
                                num_hidden_layers=3)
    assert list(hypo.state_dict().keys()) == list(g["state_keys"])
    hyper = meta_modules.HyperNetwork(8, 1, 16, hypo)
    params = hyper(torch.randn(3, 8))
    assert list(params.keys()) == list(g["names"])
    assert [str(tuple(v.shape)) for v in params.values()] == list(g["shapes"])
    assert all(v.requires_grad for v in params.values())
    assert isinstance(hypo.net.net[0][0], torch.nn.Linear)
    assert [n for n, _ in hypo.meta_named_parameters()] == list(hypo.state_dict().keys())


def test_init_distributions_match_reference_ranges():
    from siren_mri_b200 import modules
    torch.manual_seed(0)
    m = modules.SingleBVPNet(in_features=2, out_features=1)
    w0 = m.net.net[0][0].weight
    w1 = m.net.net[1][0].weight
    assert w0.abs().max() <= 0.5 and w0.abs().max() > 0.45
    bound = np.sqrt(6 / 256) / 30
    assert w1.abs().max() <= bound and w1.abs().max() > 0.95 * bound


@pytest.mark.parametrize("name", ["img_d2_o1", "vec_d2_o3"])
def test_composed_cpu_path_matches_reference(name):
    """CPU tensors take the composed PyTorch path (same ops as the reference)."""
    from siren_mri_b200 import diff_operators, modules
    g = load_golden(name, "f64")
    d, o, n, Ws, bs, x = case_inputs(g)
    m = modules.SingleBVPNet(out_features=o, in_features=d).double()
    sd = OrderedDict()
    for l, (W, b) in enumerate(zip(Ws, bs)):
        sd["net.net.%d.0.weight" % l] = torch.from_numpy(W).double()
        sd["net.net.%d.0.bias" % l] = torch.from_numpy(b).double()
    m.load_state_dict(sd)
    out = m({"coords": torch.from_numpy(x).double(), "ignored": 1})
    assert out["model_in"].requires_grad and out["model_in"].is_leaf
    assert rel_l2(out["model_out"].detach().numpy(), g["y"]) < 1e-12
    grad = diff_operators.gradient(out["model_out"], out["model_in"])
    assert rel_l2(grad.detach().numpy(), g["grad"]) < 1e-12
    if o == 1:
        lap = diff_operators.laplace(out["model_out"], out["model_in"])
        assert rel_l2(lap.detach().numpy(), g["lap"]) < 1e-12
    # per-sample params route
    y2 = m({"coords": torch.from_numpy(x).double()}, params=OrderedDict(m.named_parameters()))["model_out"]
    assert torch.equal(y2, out["model_out"])
    acts = m.forward_with_activations({"coords": torch.from_numpy(x).double()})
    assert len(acts["activations"]) == 1 + 2 * 4   # input + (linear, sine) x 4; the last linear is popped as model_out


class _OracleKernelFn(torch.autograd.Function):
    """Stand-in for the CUDA kernel Function with the same signature, backed by the numpy oracle
    (fp64).  Lets the attach-Function wiring be verified on CPU."""

    @staticmethod
    def forward(ctx, w0, precision, order, coords_grad, coords, *params):
        Ws = [p.detach().numpy() for p in params[0::2]]
        bs = [p.detach().numpy() for p in params[1::2]]
        y, J, D, cache = so.siren_forward(coords.detach().numpy(), Ws, bs, w0, order=order)
        ctx.cache, ctx.Ws, ctx.order = cache, Ws, order
        ctx.set_materialize_grads(False)
        outs = [torch.from_numpy(y)]
        if order >= 1:
            outs.append(torch.from_numpy(np.ascontiguousarray(J)))
        if order >= 2:
            outs.append(torch.from_numpy(np.ascontiguousarray(D)))
        return outs[0] if order == 0 else tuple(outs)

    @staticmethod
    def backward(ctx, gy, gJ=None, gD=None):
        assert not torch.is_grad_enabled()
        y_shape = ctx.cache["h"][-1].shape[:-1] + (ctx.Ws[-1].shape[-2],)
        gy = np.zeros(y_shape) if gy is None else gy.numpy()
        dWs, dbs, gx = so.siren_backward(ctx.cache, ctx.Ws, gy, None if gJ is None else gJ.numpy(),
                                         None if gD is None else gD.numpy())
        grads = []
        for dW, db in zip(dWs, dbs):
            grads += [torch.from_numpy(dW), torch.from_numpy(db)]
        return (None, None, None, None, None) + tuple(grads)


@pytest.mark.parametrize("name", ["img_d2_o1", "sdf_d3_o1"])
def test_attach_functions_reproduce_reference_derivative_queries(name, monkeypatch):
    from siren_mri_b200 import diff_operators, functional
    monkeypatch.setattr(functional, "_SirenKernelFn", _OracleKernelFn)
    g = load_golden(name, "f64")
    d, o, n, Ws, bs, x = case_inputs(g)
    weights = [torch.from_numpy(w).double().requires_grad_(True) for w in Ws]
    biases = [torch.from_numpy(b).double().requires_grad_(True) for b in bs]

    def run(order):
        for t in weights + biases:
            t.grad = None
        coords = torch.from_numpy(x).double().requires_grad_(True)
        return coords, functional.siren_mlp(coords, weights, biases, 30.0, "fp32", coord_derivs=order)

    coords, y = run(2)
    grad = diff_operators.gradient(y, coords)
    lap = diff_operators.laplace(y, coords)
    assert rel_l2(grad.detach().numpy(), g["grad"]) < 1e-9
    assert rel_l2(lap.detach().numpy(), g["lap"]) < 1e-9
    loss = torch.mean((lap - torch.from_numpy(g["gt_lap"]).double()) ** 2)
    loss.backward()
    check_grads("lapmse", g, [w.grad.numpy() for w in weights],
                [b.grad.numpy() if b.grad is not None else np.zeros(b.shape) for b in biases], 1e-9)

    coords, y = run(1)
    grad = diff_operators.gradient(y, coords)
    loss = torch.mean((grad - torch.from_numpy(g["gt_grad"]).double()).pow(2).sum(-1))
    loss.backward()
    check_grads("gradmse", g, [w.grad.numpy() for w in weights],
                [b.grad.numpy() if b.grad is not None else np.zeros(b.shape) for b in biases], 1e-9)

    # plain value loss with jets attached: parameter grads unchanged, coords.grad = J-weighted gy
    coords, y = run(1)
    loss = ((y - torch.from_numpy(g["gt"]).double()) ** 2).sum() / 16384.0
    loss.backward()
    check_grads("mse", g, [w.grad.numpy() for w in weights], [b.grad.numpy() for b in biases], 1e-9)
    assert rel_l2(coords.grad.numpy(), g["mse_gx"]) < 1e-9


def test_native_path_fails_loudly_without_library(monkeypatch):
    from siren_mri_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libsiren_b200.so")
    with pytest.raises(_lib.NativeError):
        _lib.load()


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "siren_mri_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("no silent fallback", ""), os.path.join(dirpath, f)


@pytest.mark.parametrize("name", ["img_d2_o1", "vec_d2_o3", "sdf_d3_o1"])
@pytest.mark.parametrize("order", [1, 2])
def test_jacobian_and_hessian_on_jet_outputs(name, order, monkeypatch):
    """diff_operators.jacobian / hessian (reference diff_operators.py:46-59, 5-24) on outputs of the jet path: the
    Jacobian comes from the jets; the Hessian's mixed terms are not in the jets, so hessian() re-evaluates the
    composed graph (functional.composed_of) instead of returning zeroed off-diagonals."""
    from siren_mri_b200 import diff_operators, functional
    monkeypatch.setattr(functional, "_SirenKernelFn", _OracleKernelFn)
    g = load_golden(name, "f64")
    d, o, n, Ws, bs, x = case_inputs(g)
    weights = [torch.from_numpy(w).double().requires_grad_(True) for w in Ws]
    biases = [torch.from_numpy(b).double().requires_grad_(True) for b in bs]
    coords = torch.from_numpy(x).double().requires_grad_(True)
    y = functional.siren_mlp(coords, weights, biases, 30.0, "fp32", coord_derivs=order)
    assert getattr(y, "_siren_jets", 0) == order
    jac, status = diff_operators.jacobian(y, coords)
    assert status == 0 and rel_l2(jac.detach().numpy(), g["jac"]) < 1e-6        # the record is fp32
    hes, status = diff_operators.hessian(y, coords)
    assert status == 0 and rel_l2(hes.detach().numpy(), g["hess"]) < 1e-6
    off = hes.detach().numpy()[..., 0, 1]
    assert np.abs(off).max() > 0                                                 # mixed terms are really there
    # and it is still a differentiable function of the parameters
    hes.pow(2).mean().backward()
    assert weights[1].grad is not None and torch.isfinite(weights[1].grad).all()


def test_siren_alias_matches_notebook_definition():
    """modules.Siren / SineLayer (explore_siren.ipynb cell 3): keys, init ranges, (output, coords) contract, both
    outermost settings and unequal omegas -- against the formula written out."""
    from siren_mri_b200 import modules
    torch.manual_seed(0)
    for outer, w_first in ((True, 30.0), (False, 30.0), (True, 7.0)):
        m = modules.Siren(2, 64, 2, 3, outermost_linear=outer, first_omega_0=w_first, hidden_omega_0=30.0)
        keys = list(m.state_dict().keys())
        assert keys[:2] == ["net.0.linear.weight", "net.0.linear.bias"]
        assert keys[-2:] == (["net.3.weight", "net.3.bias"] if outer else ["net.3.linear.weight", "net.3.linear.bias"])
        assert m.net[0].linear.weight.abs().max() <= 0.5 and m.net[1].linear.weight.abs().max() <= np.sqrt(6 / 64) / 30
        x = torch.rand(50, 2) * 2 - 1
        y, c = m(x)
        assert c.requires_grad and c is not x and y.shape == (50, 3)
        h = x
        for i, layer in enumerate(m.net):
            lin = layer.linear if hasattr(layer, "linear") else layer
            h = h @ lin.weight.t() + lin.bias
            if hasattr(layer, "linear"):
                h = torch.sin((w_first if i == 0 else 30.0) * h)
        assert torch.allclose(y, h, atol=1e-6)
        (g,) = torch.autograd.grad(y.sum(), c)
        assert g.shape == (50, 2)


def test_fourier_feature_mirror_and_lazy_tag_cpu():
    """features.GaussianFourierFeatureTransform mirrors features.py:21-53; the lazy tag is only handed on for CUDA
    tensors, and a tagged tensor that reaches a non-native path is materialised with the reference's ops."""
    import numpy as np
    import torch
    from siren_mri_b200 import data_consistency, features, functional, modules
    from tests.helpers import load_golden, rel_l2
    g = load_golden("fourier_t2_f8_o2", "f64")
    tr = features.GaussianFourierFeatureTransform(num_input_channels=2, mapping_size_spatial=8, scale=21, lazy=True)
    tr.set_B(torch.from_numpy(g["B"]).double())
    assert tuple(tr.get_B().shape) == (2, 8)
    x = torch.from_numpy(g["x"]).double()
    feat = tr(x)                                   # CPU: never lazy
    assert getattr(feat, "_siren_fourier", None) is None
    assert rel_l2(feat.numpy(), g["feat"]) < 1e-12
    # a tagged tensor on a path the kernels do not serve gives the same numbers as the materialised features
    torch.manual_seed(0)
    net = modules.SingleBVPNet(in_features=16, out_features=2).double()
    tagged = x.detach().view_as(x)
    tagged._siren_fourier = tr.get_B()
    out_a = net({"coords": tagged})
    out_b = net({"coords": functional.fourier_features(x, tr.get_B())})
    assert torch.equal(out_a["model_out"], out_b["model_out"])
    assert tuple(out_a["model_in"].shape) == (2, 300, 2)      # lazy: model_in stays the raw coordinates
    # DataConsistencyInKspace mirror (data_consistency.py:32-47)
    dc = data_consistency.DataConsistencyInKspace(noise_lvl=None)
    y_dc = dc(torch.from_numpy(g["y"]), torch.from_numpy(g["k0"]).double(), torch.from_numpy(g["mask"]).double())
    assert rel_l2(y_dc.numpy(), g["y_dc"]) < 1e-12
    assert tuple(features.AsinhTransform()(torch.ones(2, 3)).shape) == (2, 3)


def test_sdf_grid_sampling_matches_the_reference_enumeration():
    """sdf_meshing.sample_sdf_grid: the reference's point enumeration (sdf_meshing.py:25-38, floor divisions) generated
    chunk by chunk, values in place."""
    import torch
    from siren_mri_b200 import modules, sdf_meshing
    N = 7
    idx = torch.arange(N ** 3)
    ref = torch.zeros(N ** 3, 3)
    vs = 2.0 / (N - 1)
    ref[:, 2] = (idx % N) * vs - 1
    ref[:, 1] = ((idx // N) % N) * vs - 1
    ref[:, 0] = ((idx // N // N) % N) * vs - 1
    got = torch.cat([sdf_meshing.grid_coords(h, min(h + 50, N ** 3), N, "cpu") for h in range(0, N ** 3, 50)])
    assert torch.allclose(got, ref, atol=1e-7)
    torch.manual_seed(0)
    net = modules.SingleBVPNet(in_features=3, out_features=1)
    # the net stays on the host; create_mesh samples on the GPU when there is one
    decoder = lambda c: net({"coords": c.cpu()})["model_out"]      # noqa: E731
    vol = sdf_meshing.sample_sdf_grid(decoder, N=N, max_batch=100, device="cpu")
    with torch.no_grad():
        want = net({"coords": ref})["model_out"].reshape(N, N, N)
    assert vol.shape == (N, N, N) and torch.allclose(vol, want, atol=1e-6)
    seen = {}
    sdf_meshing.create_mesh(decoder, "/tmp/unused", N=N, max_batch=64,
                            convert=lambda s, o, v, f, off, sc: seen.update(shape=tuple(s.shape), origin=o, size=v, file=f))
    assert seen["shape"] == (N, N, N) and seen["origin"] == [-1, -1, -1] and seen["file"] == "/tmp/unused.ply"


def test_data_consistency_mirror_matches_the_oracle_and_honours_the_fused_tag():
    """data_consistency.DataConsistencyInKspace (mirror of data_consistency.py:23-47): noiseless and noisy blends equal
    the oracle's restatement of the reference, sampled entries of the noiseless blend are the samples to the bit, and a
    prediction tagged by the fused epilogue is passed on."""
    import numpy as np
    import torch
    from oracle import siren_oracle as so
    from siren_mri_b200 import data_consistency
    rng = np.random.default_rng(0)
    pred = rng.standard_normal((2, 12, 2))
    k0 = rng.standard_normal((2, 2, 3, 4))
    mask = (rng.uniform(size=(2, 2, 3, 4)) < 0.5).astype(np.float64)
    for noise in (None, 0.3):
        dc = data_consistency.DataConsistencyInKspace(noise_lvl=noise)
        got = dc(torch.from_numpy(pred), torch.from_numpy(k0), torch.from_numpy(mask)).numpy()
        assert np.allclose(got, so.data_consistency(pred, k0, mask, noise), rtol=0, atol=1e-14)
    got = data_consistency.DataConsistencyInKspace()(torch.from_numpy(pred), torch.from_numpy(k0), torch.from_numpy(mask)).numpy()
    m_l = np.transpose(mask, (0, 2, 3, 1)).reshape(2, -1, 2) > 0
    assert np.array_equal(got[m_l], np.transpose(k0, (0, 2, 3, 1)).reshape(2, -1, 2)[m_l])
    t = torch.from_numpy(pred).clone()
    t._siren_dc_done = 0.0
    assert data_consistency.DataConsistencyInKspace()(t, torch.from_numpy(k0), torch.from_numpy(mask)) is t


def test_hypernetwork_mirror_off_the_gpu_is_the_reference_flow():
    """meta_modules.HyperNetwork with native_heads left to its default: CPU tensors take the reference's flow
    (net(z).reshape, meta_modules.py:50-54); hypo_weight_loss equals loss_functions.py:279-287."""
    import torch
    from siren_mri_b200 import meta_modules, modules
    torch.manual_seed(0)
    hypo = modules.SingleBVPNet(out_features=2, type="sine", in_features=4, hidden_features=256, num_hidden_layers=1)
    hyper = meta_modules.HyperNetwork(hyper_in_features=8, hyper_hidden_layers=1, hyper_hidden_features=16, hypo_module=hypo)
    z = torch.randn(3, 8)
    hp = hyper(z)
    assert list(hp.keys()) == [n for n, _ in hypo.meta_named_parameters()]
    for (name, p), (n2, ref) in zip(hp.items(), hypo.meta_named_parameters()):
        assert tuple(p.shape) == (3,) + tuple(ref.shape)
        assert getattr(p, "_siren_ops", None) is None
    want = sum(torch.sum(w ** 2) for w in hp.values()) * (1 / sum(w.numel() for w in hp.values()))
    assert torch.allclose(meta_modules.hypo_weight_loss({"hypo_params": hp}), want)


def test_hypernetwork_batched_trunks_equal_the_per_head_flow():
    """HyperNetwork._hidden_batched (all heads' ReLU trunks as one baddbmm per level) against the reference's per-head
    flow (meta_modules.py:50-54), values and every parameter gradient, in fp64."""
    import torch
    from siren_mri_b200 import meta_modules, modules
    torch.manual_seed(1)
    hypo = modules.SingleBVPNet(out_features=2, type="sine", in_features=4, hidden_features=256, num_hidden_layers=1)
    hyper = meta_modules.HyperNetwork(hyper_in_features=8, hyper_hidden_layers=2, hyper_hidden_features=16,
                                      hypo_module=hypo).double()
    z = torch.randn(3, 8, dtype=torch.float64)
    ref = hyper(z)                                                      # CPU: the reference's flow
    loss_ref = sum((v ** 2).sum() for v in ref.values())
    g_ref = torch.autograd.grad(loss_ref, list(hyper.parameters()))
    hid = hyper._hidden_batched(z)
    outs = []
    for p, (name, net) in enumerate(zip(hyper.names, hyper.nets)):
        last = net.net[-1][0]
        outs.append(torch.addmm(last.bias, hid[p], last.weight.t()).reshape(ref[name].shape))
        assert torch.allclose(outs[-1], ref[name], rtol=0, atol=1e-13)
    g_bat = torch.autograd.grad(sum((v ** 2).sum() for v in outs), list(hyper.parameters()))
    for a, b in zip(g_bat, g_ref):
        assert torch.allclose(a, b, rtol=1e-10, atol=1e-13)
