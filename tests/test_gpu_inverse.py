"""Inverse / sampling direction (-m gpu), SURVEY 8(f).3: x = f_c^{-1}(z) through gbnf_component_inverse, pinned by
decode(encode(x)) == x, by the fp64 oracle inverse, and -- where upstream's decode is not broken (1-D Glow with additive
coupling, FlowStep.decode models/glow.py:344-366) -- by the reference's own decode output; per-sample component assignment
for mixture sampling is bit-exact under the inverse-CDF rule (SURVEY 8c)."""
import numpy as np
import pytest
import torch

from conftest import GOLDEN_CASES
from helpers import build_model, golden_model
from oracle import gbnf_oracle as orc
from gbnf_b200._lib import GbnfError

pytestmark = pytest.mark.gpu


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _f16_ok(md):
    return md["h"] % 128 == 0 and md["h"] <= 512 and md["depth"] == 1


@pytest.mark.parametrize("mode", ["fp32", "f16", "f16fast"])
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_inverse_vs_reference_golden_and_round_trip(golden, name, mode):
    g = golden(name); md = golden_model(g)
    model = build_model(md, "cuda", gemm_mode=mode)
    try:
        x = dev(g["x"])
        if mode != "fp32" and not _f16_ok(md):
            with pytest.raises(GbnfError, match="inverse direction"):
                model.component_inverse(x, 0)
            return
        m64 = orc.cast_model(md, np.float64)
        for c in range(md["C"]):
            z, ldj = model.component_forward(x, c)
            xr, ldji = model.component_inverse(z, c)
            # decode(encode(x)) == x: both directions evaluate the coupling networks on the same z1, so even the f16 modes invert
            # their own forward map to fp32 rounding
            np.testing.assert_allclose(xr.cpu().numpy(), g["x"], rtol=2e-4, atol=2e-4)
            np.testing.assert_allclose((ldj + ldji).cpu().numpy(), 0.0, atol=2e-4 * max(1.0, float(ldj.abs().max())))
            # the fp64 oracle inverse on the reference's own z
            xo, ldjo = orc.component_inverse(m64, g["z64"][c], c)
            np.testing.assert_allclose(xo, g["x"], rtol=1e-9, atol=1e-9)                  # oracle inverts the reference's forward
            xk, ldjk = model.component_inverse(dev(g["z32"][c]), c)
            tol = 2e-4 if mode == "fp32" else 2e-2
            np.testing.assert_allclose(xk.cpu().numpy(), xo, rtol=tol, atol=tol)
            np.testing.assert_allclose(ldjk.cpu().numpy(), ldjo, rtol=tol, atol=tol)
            if f"dec32.c{c}" in g:                                                        # the reference's own decode output
                np.testing.assert_allclose(xk.cpu().numpy(), g[f"dec32.c{c}"], rtol=tol, atol=tol)
            # the drop-in call: model(z=z, components=c, reverse=True) -> x
            xd = model(z=dev(g["z32"][c]), components=c, reverse=True)
            assert torch.equal(xd, xk)
    finally:
        model.release()


INV_VARIANTS = {
    "glow_affine_d63_h512": dict(kind="glow", D=63, C=2, K=3, h=512),
    "glow_additive_relu_d7_h128": dict(kind="glow", D=7, C=2, K=3, h=128, coupling="additive", act="relu"),
    "realnvp_bn_d9_h384": dict(kind="realnvp", D=9, C=2, K=3, h=384, batch_norm=True),
    "realnvp_mixed_d5_h256": dict(kind="realnvp", D=5, C=3, K=4, h=256, act="mixed"),
    "realnvp_toy_d2_h128": dict(kind="realnvp", D=2, C=3, K=2, h=128, rho_init="uniform", toy_base=True),
    "glow_depth2_h64_fp32only": dict(kind="glow", D=10, C=2, K=2, h=64, depth=2),
    "glow_depth0_h128_fp32only": dict(kind="glow", D=10, C=2, K=2, h=128, depth=0),
    "realnvp_bn_depth3_h256_fp32only": dict(kind="realnvp", D=9, C=2, K=3, h=256, depth=3, batch_norm=True),
    "glow_additive_depth4_h192_fp32only": dict(kind="glow", D=7, C=2, K=2, h=192, depth=4, coupling="additive"),
    "glow_h1024_fp32only": dict(kind="glow", D=12, C=1, K=2, h=1024),
}


@pytest.mark.parametrize("mode", ["fp32", "f16fast"])
@pytest.mark.parametrize("name", list(INV_VARIANTS))
def test_inverse_variants_vs_oracle(name, mode):
    kw = dict(INV_VARIANTS[name])
    md = orc.make_synthetic_model(kw.pop("kind"), kw.pop("D"), kw.pop("C"), kw.pop("K"), kw.pop("h"), seed=41, **kw)
    if mode != "fp32" and name.endswith("fp32only"):
        pytest.skip("served by the fp32 kernel only")
    B = 517
    x = np.random.default_rng(5).standard_normal((B, md["D"])).astype(np.float32)
    model = build_model(md, "cuda", gemm_mode=mode)
    try:
        m64 = orc.cast_model(md, np.float64)
        for c in range(md["C"]):
            z64, ldj64 = orc.component_forward(m64, x.astype(np.float64), c)
            xk, ldjk = model.component_inverse(dev(z64.astype(np.float32)), c)
            tol = 5e-4 if mode == "fp32" else 3e-2
            np.testing.assert_allclose(xk.cpu().numpy(), x, rtol=tol, atol=tol)
            np.testing.assert_allclose(ldjk.cpu().numpy(), -ldj64, rtol=tol, atol=tol)
            z, ldj = model.component_forward(dev(x), c)
            xr, _ = model.component_inverse(z, c)
            np.testing.assert_allclose(xr.cpu().numpy(), x, rtol=5e-4, atol=5e-4)
        model.check_status()
    finally:
        model.release()


def test_mixture_sampling_assignment_is_bit_exact_and_rows_invert():
    md = orc.make_synthetic_model("glow", 8, 5, 2, 128, seed=9)
    model = build_model(md, "cuda", gemm_mode="fp32")
    try:
        model.component, model.all_trained = 4, True
        n = 4096
        gen = torch.Generator(device="cuda").manual_seed(3)
        u = torch.rand(n, dtype=torch.float64, device="cuda", generator=gen)
        z = torch.randn((n, 8), device="cuda", generator=gen)
        x, comp = model.sample(n, u=u, z=z)
        ref = orc.assign_components(md["rho"], 5, u.cpu().numpy())
        assert np.array_equal(comp.cpu().numpy(), ref)                      # bit-exact assignment for identical uniforms
        assert set(np.unique(ref)) == set(range(5))
        for c in range(5):
            rows = np.nonzero(ref == c)[0]
            xo, _ = orc.component_inverse(orc.cast_model(md, np.float64), z.cpu().numpy()[rows].astype(np.float64), c)
            np.testing.assert_allclose(x.cpu().numpy()[rows], xo, rtol=5e-4, atol=5e-4)
        # the sampled points are where the mixture has mass: log G(x) is finite and close to the component densities
        G = model.mixture_log_density(x, 5)
        assert torch.isfinite(G).all()
        # edge uniforms
        ue = torch.tensor([0.0, 1.0 - 2 ** -53], dtype=torch.float64, device="cuda")
        ce = model.assign_components(ue, n=5).cpu().numpy()
        assert ce[0] == 0 and ce[1] == 4
        # decode with z = None draws sample_size rows from the prior
        xs = model.decode(None, None, 0.7, "c")
        assert xs.shape == (model.flows[4].sample_size, 8) and torch.isfinite(xs).all()
    finally:
        model.release()
