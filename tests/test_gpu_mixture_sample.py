"""Sampling from the whole mixture in one launch (-m gpu): gbnf_mixture_inverse sorts the rows by component on the device and runs
one inverse launch over all of them.  Every row must carry the bits gbnf_component_inverse gives it (pinned against a per-component
loop written here), sample() must match the fp64 oracle, refusals must leave x untouched, an out-of-range id must be reported by
check_status() without a fault, and sample() must replay from a CUDA graph."""
import ctypes as C

import numpy as np
import pytest
import torch

from helpers import build_model
from oracle import gbnf_oracle as orc
from gbnf_b200 import _lib
from gbnf_b200._lib import GbnfError

pytestmark = pytest.mark.gpu


def per_component(model, z, comp, n):
    """The per-component algorithm sample() used before: gather each component's rows, invert them, scatter back."""
    x = torch.full_like(z, float("nan"))
    ldj = torch.full((z.shape[0],), float("nan"), device=z.device)
    for c in range(n):
        rows = torch.nonzero(comp == c, as_tuple=False).squeeze(1)
        if rows.numel():
            xc, lc = model.component_inverse(z[rows].contiguous(), c)
            x[rows], ldj[rows] = xc, lc
    return x, ldj


def assert_bitwise(model, z, comp, n):
    x, ldj = model.mixture_inverse(z, comp, n)
    xr, lr = per_component(model, z, comp, n)
    assert torch.equal(x, xr) and torch.equal(ldj, lr)
    model.check_status()
    return x, ldj


def inputs(B, D, n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(B, D, device="cuda", generator=g), torch.randint(0, n, (B,), device="cuda", generator=g)


MODELS = {
    # pipelined tensor-core kernel (coupling_tc2.cuh) widths, h = 215 padded
    "glow_h128_d7": dict(kind="glow", D=7, C=3, K=2, h=128),
    "realnvp_h256_d6": dict(kind="realnvp", D=6, C=4, K=2, h=256),
    "glow_h512_d43": dict(kind="glow", D=43, C=3, K=2, h=512),
    "glow_h215_d10": dict(kind="glow", D=10, C=3, K=2, h=215),
    # CTA-pair kernel (coupling_tc3.cuh), h = 630 padded to 1024
    "glow_h1024_d21": dict(kind="glow", D=21, C=3, K=2, h=1024),
    "glow_h630_d9": dict(kind="glow", D=9, C=2, K=2, h=630),
    "realnvp_h1024_d8": dict(kind="realnvp", D=8, C=3, K=2, h=1024),
    "realnvp_h630_d7": dict(kind="realnvp", D=7, C=2, K=2, h=630),
    # BatchNorm with odd D, the toy base
    "realnvp_bn_h256_d9": dict(kind="realnvp", D=9, C=3, K=3, h=256, batch_norm=True),
    "realnvp_toy_h128_d2": dict(kind="realnvp", D=2, C=3, K=2, h=128, rho_init="uniform", toy_base=True),
    # fp32-only models
    "realnvp_residual_fp32only": dict(kind="realnvp", D=6, C=3, K=2, h=64, act="residual"),
    "glow_invconv_fp32only": dict(kind="glow", D=6, C=3, K=2, h=64, invconv=True),
}


def make(name, seed=51):
    kw = dict(MODELS[name])
    return orc.make_synthetic_model(kw.pop("kind"), kw.pop("D"), kw.pop("C"), kw.pop("K"), kw.pop("h"), seed=seed, **kw)


@pytest.mark.parametrize("mode", ["fp32", "f16", "f16fast"])
@pytest.mark.parametrize("name", list(MODELS))
def test_mixture_inverse_is_bitwise_the_per_component_inverse(name, mode):
    if mode != "fp32" and name.endswith("fp32only"):
        pytest.skip("served by the fp32 kernel only")
    md = make(name)
    model = build_model(md, "cuda", gemm_mode=mode)
    try:
        if mode != "fp32":
            assert model.info()["pipelined"] == (2 if md["h"] > 512 else 1)
        z, comp = inputs(1000, md["D"], md["C"], 1)
        x, ldj = assert_bitwise(model, z, comp, md["C"])
        assert torch.isfinite(x).all() and torch.isfinite(ldj).all()
    finally:
        model.release()


EDGE_MODELS = ["glow_h128_d7", "glow_h1024_d21"]


@pytest.mark.parametrize("mode", ["fp32", "f16fast"])
@pytest.mark.parametrize("name", EDGE_MODELS)
def test_assignment_edge_cases(name, mode, monkeypatch):
    md = make(name)
    n, D = md["C"], md["D"]
    model = build_model(md, "cuda", gemm_mode=mode)
    try:
        z, comp = inputs(1000, D, n, 2)
        assert_bitwise(model, z, torch.full_like(comp, 1), n)                      # all rows on one component
        assert_bitwise(model, z, torch.where(comp == 1, 0, comp), n)               # a component without rows
        seg = torch.cat([torch.full((128,), 2), torch.full((129,), 0), torch.full((128,), 1), torch.full((129,), 2)]).cuda()
        assert_bitwise(model, z[:seg.shape[0]].contiguous(), seg, n)               # segments of exactly 128 and 129 rows
        assert_bitwise(model, z[:seg.shape[0]].contiguous(), seg[torch.randperm(seg.shape[0], device="cuda")].contiguous(), n)
        for B in (1, 77):
            assert_bitwise(model, z[:B].contiguous(), comp[:B].contiguous(), n)
        # a "-c" exclusion: ids from the mixture without component 1
        model.component, model.all_trained = 1, True
        u = torch.rand(1000, dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(4))
        ex = model.assign_components(u, n, exclude=1)
        assert not bool((ex == 1).any())
        assert_bitwise(model, z, ex, n)
        # a capped grid: every CTA (pair) walks many units of different components
        ref = model.mixture_inverse(z, comp, n)
        monkeypatch.setenv("GBNF_GRID", "3")
        capped = model.mixture_inverse(z, comp, n)
        assert model.info()["grid"] in (3, 6)
        monkeypatch.delenv("GBNF_GRID")
        assert torch.equal(capped[0], ref[0]) and torch.equal(capped[1], ref[1])
        model.check_status()
    finally:
        model.release()


@pytest.mark.parametrize("mode", ["fp32", "f16fast"])
def test_batch_above_the_launch_slice(mode):
    md = orc.make_synthetic_model("glow", 4, 3, 1, 128, seed=52)
    model = build_model(md, "cuda", gemm_mode=mode)
    try:
        z, comp = inputs((1 << 22) + 300, 4, 3, 3)
        assert_bitwise(model, z, comp, 3)
    finally:
        model.release()


@pytest.mark.parametrize("mode", ["fp32", "f16", "f16fast"])
@pytest.mark.parametrize("name", ["glow_h512_d43", "realnvp_h256_d6", "realnvp_h1024_d8"])
def test_sample_against_the_oracle(name, mode):
    md = make(name)
    n = md["C"]
    model = build_model(md, "cuda", gemm_mode=mode)
    try:
        model.component, model.all_trained = n - 1, True
        g = torch.Generator(device="cuda").manual_seed(5)
        u = torch.rand(4096, dtype=torch.float64, device="cuda", generator=g)
        z = torch.randn((4096, md["D"]), device="cuda", generator=g)
        x, comp = model.sample(4096, u=u, z=z)
        ref = orc.assign_components(md["rho"], n, u.cpu().numpy())
        assert np.array_equal(comp.cpu().numpy(), ref)
        assert set(np.unique(ref)) == set(range(n))
        m64 = orc.cast_model(md, np.float64)
        tol = 5e-4 if mode == "fp32" else 3e-2
        for c in range(n):
            rows = np.nonzero(ref == c)[0]
            xo, _ = orc.component_inverse(m64, z.cpu().numpy()[rows].astype(np.float64), c)
            np.testing.assert_allclose(x.cpu().numpy()[rows], xo, rtol=tol, atol=tol)
        model.check_status()
    finally:
        model.release()


def raw_call(model, z, comp, n, x, ldj):
    return _lib.load().gbnf_mixture_inverse(model.handle(z.device), C.c_void_p(z.data_ptr()), z.shape[0],
                                            C.c_void_p(comp.data_ptr()), n, C.c_void_p(x.data_ptr()), C.c_void_p(ldj.data_ptr()),
                                            C.c_void_p(torch.cuda.current_stream().cuda_stream))


def test_serial_kernel_refuses_and_leaves_x_untouched():
    md = orc.make_synthetic_model("glow", 10, 2, 2, 64, seed=53)            # h = 64: the serial tensor-core kernel
    model = build_model(md, "cuda", gemm_mode="f16")
    try:
        z, comp = inputs(300, 10, 2, 6)
        with pytest.raises(GbnfError, match="inverse direction"):
            model.mixture_inverse(z, comp, 2)
        x = torch.full_like(z, 7.0)
        ldj = torch.full((300,), 7.0, device="cuda")
        rc = raw_call(model, z, comp, 2, x, ldj)
        assert rc == -1 and "inverse direction" in _lib.load().gbnf_last_error().decode()
        torch.cuda.synchronize()
        assert bool((x == 7.0).all()) and bool((ldj == 7.0).all())
    finally:
        model.release()


@pytest.mark.parametrize("mode", ["fp32", "f16fast"])
def test_out_of_range_ids_raise_at_check_status(mode):
    md = orc.make_synthetic_model("glow", 7, 3, 2, 128, seed=54)
    model = build_model(md, "cuda", gemm_mode=mode)
    try:
        z, comp = inputs(1000, 7, 3, 7)
        bad = comp.clone()
        bad[5], bad[600] = 3, -1
        x, ldj = model.mixture_inverse(z, bad, 3)
        with pytest.raises(GbnfError, match="outside"):
            model.check_status()
        ok = (bad >= 0) & (bad < 3)
        xr, lr = per_component(model, z, comp, 3)                                # the other rows are computed as usual
        assert torch.equal(x[ok], xr[ok]) and torch.equal(ldj[ok], lr[ok])
        assert_bitwise(model, z, comp, 3)                                        # the handle stays usable
    finally:
        model.release()


def test_unpacked_component_is_a_state_error():
    md = orc.make_synthetic_model("glow", 7, 3, 2, 128, seed=55)
    model = build_model(md, "cuda", gemm_mode="fp32")
    try:
        model.pack_component(0)
        model.pack_component(1)
        z, comp = inputs(100, 7, 3, 8)
        x, ldj = torch.empty_like(z), torch.empty(100, device="cuda")
        assert raw_call(model, z, comp, 3, x, ldj) == -3                         # GBNF_ERR_STATE: component 2 is not packed
        assert "has not been packed" in _lib.load().gbnf_last_error().decode()
    finally:
        model.release()


@pytest.mark.parametrize("mode", ["fp32", "f16fast"])
@pytest.mark.parametrize("name", ["glow_h512_d43", "glow_h1024_d21"])
def test_sample_replays_from_a_cuda_graph(name, mode):
    md = make(name)
    n, D, B = md["C"], md["D"], 4096
    model = build_model(md, "cuda", gemm_mode=mode)
    try:
        model.component, model.all_trained = n - 1, True
        g = torch.Generator(device="cuda").manual_seed(9)
        u_s = torch.rand(B, dtype=torch.float64, device="cuda", generator=g)
        z_s = torch.randn((B, D), device="cuda", generator=g)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            model.sample(B, u=u_s, z=z_s)                                        # warm-up: packs, scratch
        torch.cuda.current_stream().wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            x_g, comp_g = model.sample(B, u=u_s, z=z_s)
        for seed in (10, 11):
            g2 = torch.Generator(device="cuda").manual_seed(seed)
            u_s.copy_(torch.rand(B, dtype=torch.float64, device="cuda", generator=g2))
            z_s.copy_(torch.randn((B, D), device="cuda", generator=g2))
            graph.replay()
            x_e, comp_e = model.sample(B, u=u_s.clone(), z=z_s.clone())
            torch.cuda.synchronize()
            assert torch.equal(comp_g, comp_e) and torch.equal(x_g, x_e)
        model.check_status()
    finally:
        model.release()
