"""Drop-in hook against the UNMODIFIED reference, the original siren_mri project.

What the original computes is stored under tests/golden/ (tests/golden/make_golden.py), and the comparisons with it run
everywhere: here the lazy Fourier tag on the original's Fourier-feature flow, and in test_host_cpu.py the reference
checkpoint keys, values and derivatives, the HyperNetwork contract and the data consistency.  The tests that take the
``ref_modules`` fixture patch or instantiate the original's own classes (integration.patch_reference rebinds them in
place), so they need the live original: a checkout named by the SIREN_MRI_REFERENCE environment variable.  The
repository does not contain it, and without one they skip."""
import os
import sys
import types
from collections import OrderedDict

import numpy as np
import pytest
import torch

from oracle import siren_oracle as so
from tests.helpers import case_inputs, load_golden, rel_l2

REF = os.environ.get("SIREN_MRI_REFERENCE", "")


@pytest.fixture()
def ref_modules():
    if not os.path.isdir(REF):
        pytest.skip("needs a checkout of the original project (set SIREN_MRI_REFERENCE)")
    saved = dict(sys.modules)
    saved_path = list(sys.path)
    sys.path.insert(0, REF)
    pkg = types.ModuleType("torchmeta")
    pkg.__path__ = [os.path.join(REF, "torchmeta")]
    sys.modules["torchmeta"] = pkg
    import modules as ref_mod
    import meta_modules as ref_meta
    from siren_mri_b200 import integration
    integration.patch_reference(ref_mod)
    yield ref_mod, ref_meta
    integration.unpatch_reference(ref_mod)
    sys.path[:] = saved_path
    for k in list(sys.modules):
        if k not in saved:
            del sys.modules[k]


def test_lazy_fourier_tag_reproduces_the_stored_reference_flow():
    """Raw coordinates tagged by the lazy Fourier transform, through the native block with per-task weights, give the
    numbers the original's own flow gave (features.py:31-41 materialised, SingleBVPNet, then
    DataConsistencyInKspace), stored in fourier_t2_f8_o2_f64; model_in is the raw leaf."""
    from siren_mri_b200 import data_consistency, modules
    g = load_golden("fourier_t2_f8_o2", "f64")
    Ws, bs = so.make_params(2 * int(g["F"]), 256, 3, int(g["o"]), seed=int(g["seed"]), tasks=int(g["tasks"]))
    params = OrderedDict()
    for l, (W, b) in enumerate(zip(Ws, bs)):
        params["net.net.%d.0.weight" % l] = torch.from_numpy(W).double()
        params["net.net.%d.0.bias" % l] = torch.from_numpy(b).double()
    net = modules.SingleBVPNet(out_features=int(g["o"]), type="sine", in_features=2 * int(g["F"])).double()
    x = torch.from_numpy(g["x"]).double()
    tagged = x.detach().view_as(x)
    tagged._siren_fourier = torch.from_numpy(g["B"]).double()
    out = net({"coords": tagged}, params=params)
    assert tuple(out["model_in"].shape) == tuple(g["x"].shape)
    assert rel_l2(out["model_out"].detach().numpy(), g["y"]) < 1e-12
    y_dc = data_consistency.DataConsistencyInKspace(noise_lvl=None)(
        out["model_out"], torch.from_numpy(g["k0"]).double(), torch.from_numpy(g["mask"]).double())
    assert rel_l2(y_dc.detach().numpy(), g["y_dc"]) < 1e-12


def test_patched_reference_builds_native_blocks_and_matches_golden(ref_modules):
    ref_mod, ref_meta = ref_modules
    from torchmeta.modules import MetaModule
    g = load_golden("img_d2_o1", "f64")
    d, o, n, Ws, bs, x = case_inputs(g)
    m = ref_mod.SingleBVPNet(out_features=o, type="sine", in_features=d).double()   # the reference class
    assert type(m.net).__module__.startswith("siren_mri_b200")                      # ... with the native FCBlock
    assert isinstance(m.net, MetaModule) and isinstance(m.net.net[0][0], MetaModule)
    sd = OrderedDict()
    for l, (W, b) in enumerate(zip(Ws, bs)):
        sd["net.net.%d.0.weight" % l] = torch.from_numpy(W).double()
        sd["net.net.%d.0.bias" % l] = torch.from_numpy(b).double()
    m.load_state_dict(sd)                                                            # same checkpoint keys
    out = m({"coords": torch.from_numpy(x).double()})
    assert rel_l2(out["model_out"].detach().numpy(), g["y"]) < 1e-12
    import diff_operators as ref_diff                                                # unchanged reference operators
    lap = ref_diff.laplace(out["model_out"], out["model_in"])
    assert rel_l2(lap.detach().numpy(), g["lap"]) < 1e-12


def test_reference_hypernetwork_drives_native_block(ref_modules):
    ref_mod, ref_meta = ref_modules
    hypo = ref_mod.SingleBVPNet(out_features=2, type="sine", in_features=16)
    hyper = ref_meta.HyperNetwork(hyper_in_features=8, hyper_hidden_layers=1, hyper_hidden_features=16,
                                  hypo_module=hypo)
    params = hyper(torch.randn(3, 8))
    assert list(params.keys()) == [k for k, _ in hypo.meta_named_parameters()]
    out = hypo({"coords": torch.rand(3, 50, 16)}, params=params)
    assert out["model_out"].shape == (3, 50, 2)
    out["model_out"].sum().backward()
    assert all(p.grad is not None for p in hyper.parameters())


def test_reference_bvp_net_carries_the_lazy_fourier_tag(ref_modules):
    """The reference's own SingleBVPNet (patched) with raw coordinates tagged by the lazy Fourier transform gives the
    numbers of the reference flow (features.py:31-41 materialised, then the model); model_in is the raw leaf."""
    ref_mod, ref_meta = ref_modules
    import features as ref_features                      # the reference's transform
    torch.manual_seed(0)
    hypo = ref_mod.SingleBVPNet(out_features=2, type="sine", in_features=16).double()
    tr = ref_features.GaussianFourierFeatureTransform(num_input_channels=2, mapping_size_spatial=8, scale=21, device="cpu")
    tr.set_B(tr.get_B().double())
    x = torch.rand(2, 40, 2, dtype=torch.float64)
    ref_out = hypo({"coords": tr(x)})["model_out"]
    tagged = x.detach().view_as(x)
    tagged._siren_fourier = tr.get_B()
    out = hypo({"coords": tagged})
    assert tuple(out["model_in"].shape) == (2, 40, 2)
    assert torch.allclose(out["model_out"], ref_out, rtol=0, atol=1e-12)
    assert getattr(hypo.net, "_siren_pending_fourier", None) is None


def test_patched_data_consistency_passes_a_fused_prediction_on(ref_modules):
    """patch_reference(..., ref_data_consistency=...) wraps the reference's DataConsistencyInKspace.forward
    (data_consistency.py:32-47): an untagged prediction takes the reference's own code, a prediction tagged by the
    kernels' fused epilogue comes back as it is, and a noise-level mismatch is an error; fuse_dc is switched on and
    the patched SingleBVPNet hands img_sparse / dc_mask to its (native) FCBlock for the duration of the call."""
    ref_mod, ref_meta = ref_modules
    import data_consistency as ref_dc
    from siren_mri_b200 import config, integration
    integration.patch_reference(ref_mod, ref_data_consistency=ref_dc)
    try:
        assert config.get_defaults()["fuse_dc"] is True
        dc = ref_dc.DataConsistencyInKspace(noise_lvl=None)
        pred = torch.rand(2, 12, 2, dtype=torch.float64)
        k0 = torch.rand(2, 2, 3, 4, dtype=torch.float64)
        mask = (torch.rand(2, 2, 3, 4) < 0.5).double()
        want = ref_dc.DataConsistencyInKspace._reference_forward(dc, pred, k0, mask)
        assert torch.equal(dc(pred, k0, mask), want)
        tagged = pred.clone()
        tagged._siren_dc_done = 0.0
        assert dc(tagged, k0, mask) is tagged
        with pytest.raises(RuntimeError):
            ref_dc.DataConsistencyInKspace(noise_lvl=0.1)(tagged, k0, mask)
        # CPU tensors are outside the native envelope: the block computes the plain prediction, leaves it untagged and
        # the data consistency runs in the reference's module -- same numbers as the unpatched flow
        torch.manual_seed(0)
        hypo = ref_mod.SingleBVPNet(out_features=2, type="sine", in_features=2).double()
        x = torch.rand(2, 12, 2, dtype=torch.float64)
        seen = []
        orig = type(hypo.net).forward
        type(hypo.net).forward = lambda self, *a, **k: (seen.append(getattr(self, "_siren_pending_dc", None)), orig(self, *a, **k))[1]
        try:
            out = hypo({"coords": x, "img_sparse": k0, "dc_mask": mask})["model_out"]
        finally:
            type(hypo.net).forward = orig
        assert seen and seen[0] is not None and seen[0][0] is k0
        assert getattr(out, "_siren_dc_done", None) is None and hypo.net._siren_pending_dc is None
    finally:
        integration.unpatch_data_consistency(ref_dc)
    assert config.get_defaults()["fuse_dc"] is False


def test_neural_process_model_mirror_matches_the_reference_class(ref_modules, monkeypatch):
    """meta_modules.ConvolutionalNeuralProcessImplicit2DHypernetFourierFeatures (mirror of meta_modules.py:175-232) takes
    the reference model's state_dict as it is and returns the reference's numbers (CPU: every piece on the reference
    flow -- ConvImgEncoder, HyperNetwork heads, per-sample SingleBVPNet, data consistency)."""
    ref_mod, ref_meta = ref_modules
    from siren_mri_b200 import meta_modules
    monkeypatch.setattr(torch.Tensor, "cuda", lambda self, *a, **k: self)      # ImageDownsampling.__init__ (modules.py:202-203)
    torch.manual_seed(0)
    kw = dict(in_features=16, out_features=2, image_resolution=(8, 8), fourier_features_size=16, latent_dim=16,
              num_hidden_layers=1, hyper_hidden_features=16, num_conv_res_blocks=1)
    ref = ref_meta.ConvolutionalNeuralProcessImplicit2DHypernetFourierFeatures(**kw)
    ours = meta_modules.ConvolutionalNeuralProcessImplicit2DHypernetFourierFeatures(**kw)
    missing = ours.load_state_dict(ref.state_dict(), strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    x = {"coords": torch.rand(2, 64, 16), "img_sparse": torch.rand(2, 2, 8, 8), "dc_mask": (torch.rand(2, 2, 8, 8) < 0.5).float()}
    a, b = ref(x), ours(x)
    assert list(a["hypo_params"].keys()) == list(b["hypo_params"].keys())
    assert torch.allclose(a["model_out"], b["model_out"], rtol=0, atol=1e-6)
    assert torch.allclose(a["latent_vec"], b["latent_vec"], rtol=0, atol=1e-6)
    for k in a["hypo_params"]:
        assert torch.allclose(a["hypo_params"][k], b["hypo_params"][k], rtol=0, atol=1e-6)
