"""The host mirror's differentiable inverse (Glow / RealNVPFlow.inverse_autograd) on the CPU: it is the exact inverse of
forward_autograd, it matches the oracle's fp64 component_inverse on every golden and synthetic kind (BatchNorm, ResidualNet,
invconv LU-decomposed and plain, odd D, the toy base) and the reference's own additive-Glow decode, and torch.autograd.gradcheck
passes through it in fp64."""
import numpy as np
import pytest
import torch

from helpers import build_model, golden_model
from oracle import gbnf_oracle as orc
from tests.golden import store

GOLDEN = ["glow_d43", "glow_d43_h128_depth2", "glow_d43_invconv_plain", "glow_d6_additive_relu", "glow_d6_invconv", "realnvp_d5_mixed",
          "realnvp_d5_residual2_bn", "realnvp_d6_bn", "realnvp_d6_residual", "toy_d2"]
SYNTHETIC = {
    "glow_d7_affine_tanh_depth0": dict(kind="glow", D=7, C=2, K=3, h=16, depth=0),
    "glow_d9_additive_relu_depth3": dict(kind="glow", D=9, C=2, K=2, h=12, depth=3, act="relu", coupling="additive"),
    "glow_d8_invconv_plain": dict(kind="glow", D=8, C=2, K=2, h=16, invconv=True),
    "realnvp_d7_mixed_bn": dict(kind="realnvp", D=7, C=2, K=4, h=16, act="mixed", batch_norm=True),
    "realnvp_d5_residual_toy": dict(kind="realnvp", D=5, C=2, K=3, h=16, depth=2, act="residual", toy_base=True),
}


def _model64(md):
    m = build_model(md, "cpu").double()
    return m


def _check_against_oracle(md, z64):
    m64 = orc.cast_model(md, np.float64)
    model = _model64(md)
    for c in range(md["C"]):
        x_ref, ldj_ref = orc.component_inverse(m64, z64, c)
        with torch.no_grad():
            x, ldj = model.flows[c].inverse_autograd(torch.from_numpy(z64))
        np.testing.assert_allclose(x.numpy(), x_ref, rtol=1e-10, atol=1e-10)
        np.testing.assert_allclose(ldj.numpy(), ldj_ref, rtol=1e-10, atol=1e-10)


@pytest.mark.parametrize("name", GOLDEN)
def test_matches_oracle_on_golden_models(name):
    g = store.load(name)
    md = golden_model(g)
    _check_against_oracle(md, g["z64"][0])


@pytest.mark.parametrize("name", list(SYNTHETIC))
def test_matches_oracle_on_synthetic_models(name):
    md = orc.make_synthetic_model(seed=3, init_rows=256, **SYNTHETIC[name])
    z = np.random.default_rng(4).standard_normal((37, md["D"]))
    _check_against_oracle(md, z)


def test_reproduces_the_reference_decode():
    """The reference's own additive-Glow decode (models/glow.py:344-366), in fp64 and in fp32."""
    g = store.load("glow_d6_additive_relu")
    md = golden_model(g)
    model = build_model(md, "cpu")
    model64 = _model64(md)
    for c in range(md["C"]):
        with torch.no_grad():
            x64, _ = model64.flows[c].inverse_autograd(torch.from_numpy(g["z64"][c]))
            x32, _ = model.flows[c].inverse_autograd(torch.from_numpy(g["z32"][c]))
        np.testing.assert_allclose(x64.numpy(), g[f"dec64.c{c}"], rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(x32.numpy(), g[f"dec32.c{c}"], rtol=2e-5, atol=2e-5)


@pytest.mark.parametrize("name", ["glow_d43_invconv_plain", "glow_d6_invconv", "realnvp_d5_residual2_bn", "realnvp_d6_bn", "toy_d2"])
def test_forward_of_inverse_is_identity(name):
    g = store.load(name)
    md = golden_model(g)
    model = _model64(md)
    z = torch.from_numpy(np.random.default_rng(5).standard_normal((29, md["D"])))
    for c in range(md["C"]):
        with torch.no_grad():
            x, ldj_inv = model.flows[c].inverse_autograd(z)
            z2, ldj = model.flows[c].forward_autograd(x)
        assert float((z2 - z).abs().max()) < 1e-10
        assert float((ldj + ldj_inv).abs().max()) < 1e-8       # slogdet of a 43 x 43 invconv weight: ~1e-10 of |ldj|


GRADCHECK = {
    "glow_affine": dict(kind="glow", D=5, C=1, K=2, h=6),
    "glow_additive": dict(kind="glow", D=4, C=1, K=2, h=6, act="relu", coupling="additive"),
    "realnvp_flip0_bn": dict(kind="realnvp", D=5, C=2, K=3, h=6, batch_norm=True),
    "realnvp_mixed": dict(kind="realnvp", D=5, C=2, K=2, h=6, act="mixed", depth=2),
    "glow_invconv": dict(kind="glow", D=4, C=1, K=2, h=6, invconv=True),
}


@pytest.mark.parametrize("name", list(GRADCHECK))
def test_gradcheck(name):
    """gradcheck in fp64 through every parameter and z: component 0 and (RealNVP) component 1, the other flip parity."""
    md = orc.make_synthetic_model(seed=6, init_rows=64, **GRADCHECK[name])
    model = _model64(md)
    z = torch.from_numpy(np.random.default_rng(7).standard_normal((3, md["D"])) * 0.5)
    for c in range(md["C"]):
        flow = model.flows[c]
        names = [n for n, _ in flow.named_parameters()]

        def fn(zz, *ps):
            return torch.func.functional_call(_Inverse(flow), {"f." + n: p for n, p in zip(names, ps)}, (zz,))

        inputs = (z.clone().requires_grad_(True),) + tuple(p.detach().clone().requires_grad_(True) for p in flow.parameters())
        assert torch.autograd.gradcheck(fn, inputs, eps=1e-6, atol=1e-6, rtol=1e-5)


class _Inverse(torch.nn.Module):
    """inverse_autograd as a module's forward, so that torch.func.functional_call can substitute the parameters."""

    def __init__(self, flow):
        super().__init__()
        self.f = flow

    def forward(self, z):
        return self.f.inverse_autograd(z)
