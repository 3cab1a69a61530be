"""Inverse / sampling direction of h = 1024 Glow components in the f16 tensor-core modes (-m gpu): the CTA-pair kernel's
INV = 1 instantiation (coupling_tc3.cuh) behind gbnf_component_inverse, pinned by the fp64 oracle inverse, by
decode(encode(x)) == x, by the fp32 CUDA-core inverse, and by row-independence across tiles, launches and launch slices."""
import numpy as np
import pytest
import torch

from helpers import build_model
from oracle import gbnf_oracle as orc
from gbnf_b200._lib import GbnfError

pytestmark = pytest.mark.gpu

MODES = ["f16", "f16fast"]
H = 1024


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def pair_model(md, mode):
    model = build_model(md, "cuda", gemm_mode=mode)
    assert model.info()["pipelined"] == 2          # the CTA-pair kernel serves this handle
    return model


VARIANTS = {
    "affine_tanh_d63_k3": dict(D=63, C=1, K=3),
    "affine_tanh_d64_k2_c3": dict(D=64, C=3, K=2),
    "affine_tanh_d9": dict(D=9, C=1, K=2),          # one layer-1 k-slab, last layer Np = 16
    "affine_tanh_d2": dict(D=2, C=1, K=3),          # smallest |z1|
    "affine_tanh_d7": dict(D=7, C=1, K=3),          # odd |z1|
    "additive_relu_d21": dict(D=21, C=1, K=3, coupling="additive", act="relu"),
    "additive_tanh_d43": dict(D=43, C=1, K=3, coupling="additive"),
    "cfg5_d63_k10": dict(D=63, C=1, K=10),          # the BSDS300 shape, one component
}


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", list(VARIANTS))
def test_pair_inverse_vs_oracle_and_round_trip(name, mode):
    kw = dict(VARIANTS[name])
    D, C, K = kw.pop("D"), kw.pop("C"), kw.pop("K")
    md = orc.make_synthetic_model("glow", D, C, K, H, seed=43, **kw)
    B = 517
    x = np.random.default_rng(7).standard_normal((B, D)).astype(np.float32)
    rt_tol = 5e-4 if K <= 3 else 2e-3
    model = pair_model(md, mode)
    try:
        m64 = orc.cast_model(md, np.float64)
        for c in range(C):
            z64, ldj64 = orc.component_forward(m64, x.astype(np.float64), c)
            zk = dev(z64.astype(np.float32))
            xk, ldjk = model.component_inverse(zk, c)
            np.testing.assert_allclose(xk.cpu().numpy(), x, rtol=3e-2, atol=3e-2)
            np.testing.assert_allclose(ldjk.cpu().numpy(), -ldj64, rtol=3e-2, atol=3e-2)
            # decode(encode(x)) == x: both directions run the same networks on (nearly) the same z1
            z, ldj = model.component_forward(dev(x), c)
            xr, ldji = model.component_inverse(z, c)
            err = float((xr - dev(x)).abs().max())
            err_ldj = float((ldj + ldji).abs().max())
            print(f"[{name}, {mode}, c = {c}] round trip: max |x - f^-1(f(x))| = {err:.3e}, max |ldj + ldj_inv| = {err_ldj:.3e} "
                  f"(max |ldj| = {float(ldj.abs().max()):.3e})")
            np.testing.assert_allclose(xr.cpu().numpy(), x, rtol=rt_tol, atol=rt_tol)
            np.testing.assert_allclose((ldj + ldji).cpu().numpy(), 0.0, atol=rt_tol * max(1.0, float(ldj.abs().max())))
            # the drop-in call model(z=z, components=c, reverse=True) runs the same launch
            xd = model(z=zk, components=c, reverse=True)
            assert torch.equal(xd, xk)
        model.check_status()
    finally:
        model.release()


@pytest.mark.parametrize("mode", MODES)
def test_pair_inverse_tiles_slices_and_determinism(mode):
    md = orc.make_synthetic_model("glow", 21, 1, 2, H, seed=44)
    N = 20000
    x = torch.randn(N, 21, device="cuda", generator=torch.Generator(device="cuda").manual_seed(5))
    model = pair_model(md, mode)
    try:
        z, _ = model.component_forward(x, 0)
        full, ldj_full = model.component_inverse(z, 0)
        assert model.info()["grid"] % 2 == 0                  # whole CTA pairs
        np.testing.assert_allclose(full.cpu().numpy(), x.cpu().numpy(), rtol=5e-4, atol=5e-4)
        again, ldj_again = model.component_inverse(z, 0)
        assert torch.equal(again, full) and torch.equal(ldj_again, ldj_full)
        for B in (1, 127, 128, 129, 517):
            xb, lb = model.component_inverse(z[:B].contiguous(), 0)
            assert torch.equal(xb, full[:B]) and torch.equal(lb, ldj_full[:B]), B
            assert model.info()["grid"] % 2 == 0
        for r0, r1 in ((5000, 5300), (127, 129)):
            xs, ls = model.component_inverse(z[r0:r1].contiguous(), 0)
            assert torch.equal(xs, full[r0:r1]) and torch.equal(ls, ldj_full[r0:r1]), (r0, r1)
        # against the fp64 oracle on the first 517 rows of the batch
        xo, ldjo = orc.component_inverse(orc.cast_model(md, np.float64), z[:517].cpu().numpy().astype(np.float64), 0)
        np.testing.assert_allclose(full[:517].cpu().numpy(), xo, rtol=3e-2, atol=3e-2)
        np.testing.assert_allclose(ldj_full[:517].cpu().numpy(), ldjo, rtol=3e-2, atol=3e-2)
        model.check_status()
    finally:
        model.release()


@pytest.mark.parametrize("mode", MODES)
def test_pair_inverse_above_the_launch_slice(mode):
    md = orc.make_synthetic_model("glow", 9, 1, 2, H, seed=45)
    B = (1 << 22) + 300
    z = torch.randn(B, 9, device="cuda", generator=torch.Generator(device="cuda").manual_seed(6))
    model = pair_model(md, mode)
    try:
        x, ldj = model.component_inverse(z, 0)
        xt, lt = model.component_inverse(z[-400:].contiguous(), 0)
        assert torch.equal(x[-400:], xt) and torch.equal(ldj[-400:], lt)
        assert torch.isfinite(x).all() and torch.isfinite(ldj).all()
        xo, _ = orc.component_inverse(orc.cast_model(md, np.float64), z[-400:].cpu().numpy().astype(np.float64), 0)
        np.testing.assert_allclose(xt.cpu().numpy(), xo, rtol=3e-2, atol=3e-2)
        model.check_status()
    finally:
        model.release()


@pytest.mark.parametrize("mode", MODES)
def test_pair_inverse_agrees_with_fp32_inverse(mode):
    md = orc.make_synthetic_model("glow", 63, 1, 3, H, seed=46)
    z = torch.randn(517, 63, device="cuda", generator=torch.Generator(device="cuda").manual_seed(7))
    ref = build_model(md, "cuda", gemm_mode="fp32")
    try:
        x32, l32 = ref.component_inverse(z, 0)
    finally:
        ref.release()
    model = pair_model(md, mode)
    try:
        xk, lk = model.component_inverse(z, 0)
        np.testing.assert_allclose(xk.cpu().numpy(), x32.cpu().numpy(), rtol=3e-2, atol=3e-2)
        np.testing.assert_allclose(lk.cpu().numpy(), l32.cpu().numpy(), rtol=3e-2, atol=3e-2)
        model.check_status()
    finally:
        model.release()


@pytest.mark.parametrize("mode", MODES)
def test_pair_inverse_reports_values_outside_fp16(mode):
    md = orc.make_synthetic_model("glow", 21, 1, 2, H, seed=47)
    z = torch.randn(300, 21, device="cuda", generator=torch.Generator(device="cuda").manual_seed(8))
    bad = z.clone()
    bad[150] = 1e6
    model = pair_model(md, mode)
    try:
        model.component_inverse(bad, 0)
        with pytest.raises(GbnfError, match="not finite in fp16"):
            model.check_status()
        x, ldj = model.component_inverse(z, 0)                # the handle stays usable
        model.check_status()
        assert torch.isfinite(x).all() and torch.isfinite(ldj).all()
    finally:
        model.release()


@pytest.mark.parametrize("mode", MODES)
def test_pair_mixture_sampling(mode):
    md = orc.make_synthetic_model("glow", 8, 3, 2, H, seed=48)
    model = pair_model(md, mode)
    try:
        model.component, model.all_trained = 2, True
        n = 4096
        gen = torch.Generator(device="cuda").manual_seed(3)
        u = torch.rand(n, dtype=torch.float64, device="cuda", generator=gen)
        z = torch.randn((n, 8), device="cuda", generator=gen)
        x, comp = model.sample(n, u=u, z=z)
        ref = orc.assign_components(md["rho"], 3, u.cpu().numpy())
        assert np.array_equal(comp.cpu().numpy(), ref)
        assert set(np.unique(ref)) == {0, 1, 2}
        m64 = orc.cast_model(md, np.float64)
        for c in range(3):
            rows = np.nonzero(ref == c)[0]
            xo, _ = orc.component_inverse(m64, z.cpu().numpy()[rows].astype(np.float64), c)
            np.testing.assert_allclose(x.cpu().numpy()[rows], xo, rtol=3e-2, atol=3e-2)
        xs = model.decode(None, None, 0.7, "c")
        assert xs.shape == (model.flows[0].sample_size, 8) and torch.isfinite(xs).all()
        model.check_status()
    finally:
        model.release()
