"""GPU parity tests of the two shape-specific alternatives to the pipelined kernel.
The two-chain schedule (csrc/coupling_tc4.cuh): Glow / affine / tanh components of hidden width 512.  It must be BITWISE
identical to the single-chain pipelined kernel (same operands, same accumulation order) and inside the f16 gates against the
fp64 oracle.  GBNF_TC4 is read when the handle is created: 0 = single chain, 2 = prefer two chains.
The interleaved s / t kernel (csrc/coupling_tc5.cuh): RealNVP / tanh, h = 256.  It differs from the serial-network kernel only
in the fp32 summation order of the last layer.  GBNF_TC5=0 keeps the serial-network kernel."""
import os

import numpy as np
import pytest
import torch

from helpers import build_model, golden_model
from oracle import gbnf_oracle as orc

pytestmark = pytest.mark.gpu


def _model(md, mode, tc4):
    old = os.environ.get("GBNF_TC4")
    try:
        if tc4 is None:
            os.environ.pop("GBNF_TC4", None)
        else:
            os.environ["GBNF_TC4"] = str(tc4)
        m = build_model(md, "cuda", gemm_mode=mode)
        m.pack_all()          # creates the handle (the switch is read here)
        return m
    finally:
        if old is None:
            os.environ.pop("GBNF_TC4", None)
        else:
            os.environ["GBNF_TC4"] = old


def _run(md, x, mode, tc4, n_mix=None):
    m = _model(md, mode, tc4)
    try:
        G, lq = m.mixture_log_density(x, md["C"] if n_mix is None else n_mix, return_logq=True)
        m.check_status()
        torch.cuda.synchronize()
        return G.clone(), lq.clone(), m.info()
    finally:
        m.release()


@pytest.mark.parametrize("mode", ["f16fast", "f16"])
def test_bench_shape_bitwise_equal_to_single_chain(mode):
    """cfg3's shape at a ragged 65 536 + 77 rows: 6.9 work units per CTA, chains in different units at unit boundaries."""
    md = orc.make_synthetic_model("glow", 43, 8, 5, 512, seed=1)
    x = torch.from_numpy(np.random.default_rng(5).standard_normal((65536 + 77, 43)).astype(np.float32)).cuda()
    G2, lq2, inf2 = _run(md, x, mode, None)
    G1, lq1, inf1 = _run(md, x, mode, 0)
    assert inf2["two_chain"] == 1 and inf1["two_chain"] == 0 and inf2["pipelined"] == 1
    assert torch.equal(lq2, lq1) and torch.equal(G2, G1)
    ref = orc.all_component_logq(orc.cast_model(md, np.float64), x[:1024].cpu().numpy().astype(np.float64))
    err = np.abs(lq2[:1024].cpu().numpy() - ref) / np.abs(ref)
    assert err.max() < 1e-4, err.max()


@pytest.mark.parametrize("C,K,D,B", [(2, 1, 12, 300), (4, 2, 43, 777), (6, 3, 21, 1000), (8, 2, 32, 129), (4, 1, 5, 1), (4, 2, 63, 200)])
def test_small_shapes_forced_two_chain(C, K, D, B):
    """Few tiles (the cost model would split down to one component per unit): GBNF_TC4=2 forces the two-chain kernel.
    D = 63: two z tiles do not fit next to a three-stage weight ring -> the handle keeps the single-chain kernel."""
    md = orc.make_synthetic_model("glow", D, C, K, 512, seed=10 + C)
    x = torch.from_numpy(np.random.default_rng(C).standard_normal((B, D)).astype(np.float32)).cuda()
    G2, lq2, inf2 = _run(md, x, "f16fast", 2)
    G1, lq1, inf1 = _run(md, x, "f16fast", 0)
    assert inf2["two_chain"] == (1 if D <= 44 else 0) and inf1["two_chain"] == 0
    assert torch.equal(lq2, lq1) and torch.equal(G2, G1)
    ref = orc.all_component_logq(orc.cast_model(md, np.float64), x.cpu().numpy().astype(np.float64))
    np.testing.assert_allclose(lq2.cpu().numpy(), ref, rtol=1e-4, atol=2e-2 if D < 16 else 2e-3)
    Gref = orc.mixture_recursion(ref, md["rho"].astype(np.float64), C)
    np.testing.assert_allclose(G2.cpu().numpy(), Gref, rtol=1e-4, atol=2e-2 if D < 16 else 2e-3)


def test_partial_mixture_and_odd_counts_fall_back():
    """n_mix < C with an even count stays on two chains; an odd count of components runs the single-chain kernel."""
    md = orc.make_synthetic_model("glow", 43, 8, 2, 512, seed=3)
    x = torch.from_numpy(np.random.default_rng(9).standard_normal((4096, 43)).astype(np.float32)).cuda()
    m = _model(md, "f16fast", 2)
    m0 = _model(md, "f16fast", 0)
    try:
        for n_mix, two in ((6, 1), (7, 0), (2, 1), (1, 0)):
            G = m.mixture_log_density(x, n_mix)
            assert m.info()["two_chain"] == two, (n_mix, m.info())
            assert torch.equal(G, m0.mixture_log_density(x, n_mix))
        m.check_status()
    finally:
        m.release(); m0.release()


def test_reference_golden_h512(golden):
    """The reference-made fixture glow_d43_h512 (C = 2, K = 2) through the two-chain kernel."""
    g = golden("glow_d43_h512")
    md = golden_model(g)
    x = torch.from_numpy(g["x"]).cuda()
    G, lq, inf = _run(md, x, "f16fast", 2)
    assert inf["two_chain"] == 1
    ref = g["logq64"]
    assert np.max(np.abs(lq.cpu().numpy() - ref) / np.abs(ref)) < 1e-4


# ---- RealNVP, h = 256: interleaved s / t kernel (csrc/coupling_tc5.cuh) -------------------------------------------------------------
def _run_rnvp(md, x, mode, tc5, n_mix=None):
    """GBNF_TC5 is read when the handle is created: 0 = serial-network kernel."""
    old = os.environ.get("GBNF_TC5")
    try:
        if tc5 is None:
            os.environ.pop("GBNF_TC5", None)
        else:
            os.environ["GBNF_TC5"] = str(tc5)
        m = build_model(md, "cuda", gemm_mode=mode)
        m.pack_all()
    finally:
        if old is None:
            os.environ.pop("GBNF_TC5", None)
        else:
            os.environ["GBNF_TC5"] = old
    try:
        G, lq = m.mixture_log_density(x, md["C"] if n_mix is None else n_mix, return_logq=True)
        inf = m.info()
        z, ldj = m.component_forward(x, md["C"] - 1)
        m.check_status()
        torch.cuda.synchronize()
        return G.clone(), lq.clone(), z.clone(), ldj.clone(), inf
    finally:
        m.release()


RNVP_SHAPES = [(6, 4, 5, 65536 + 33, False, False), (2, 8, 2, 5000, False, True), (5, 4, 4, 777, True, False),
               (21, 2, 3, 300, True, False), (32, 2, 2, 129, False, False), (2, 8, 1, 4096, False, True)]


@pytest.mark.parametrize("mode", ["f16fast", "f16"])
@pytest.mark.parametrize("D,C,K,B,bn,toy", RNVP_SHAPES)
def test_realnvp_interleaved_kernel_vs_serial_network(D, C, K, B, bn, toy, mode):
    """serial-network kernel (tc2) vs interleaved s / t (tc5): same operands, only the last layer's two k-pieces are summed in
    registers instead of in the tensor-core accumulator -> equal to fp32 rounding.
    Odd D (the halves alternate), eval-BatchNorm, the toy base, z_out (single-component launches stay on tc5 / tc2)."""
    md = orc.make_synthetic_model("realnvp", D, C, K, 256, seed=20 + D, batch_norm=bn, toy_base=toy)
    x = torch.from_numpy(np.random.default_rng(D).standard_normal((B, D)).astype(np.float32)).cuda()
    G5, lq5, z5, l5, inf5 = _run_rnvp(md, x, mode, None)     # the default
    G2, lq2, z2, l2, inf2 = _run_rnvp(md, x, mode, 0)
    assert inf5["two_chain"] == 2 and inf2["two_chain"] == 0
    for a_, b_ in ((lq5, lq2), (G5, G2), (z5, z2), (l5, l2)):
        d = (a_ - b_).abs().double()
        # fp32 summation order of the last layer only: 1e-7-level differences on average; on a handful of the 400 k values that
        # last bit flips the fp16 rounding of a later step's activation (2^-11 relative), i.e. the difference between two equally
        # valid fp16 roundings (f16 tolerance class, measured max 3.4e-4)
        rel = d / (b_.abs().double() + 1.0)
        assert float(rel.mean()) < 2e-6 and float(rel.max()) < 2e-3, (float(rel.mean()), float(rel.max()))
    n = min(B, 2048)
    ref = orc.all_component_logq(orc.cast_model(md, np.float64), x[:n].cpu().numpy().astype(np.float64))
    np.testing.assert_allclose(lq5[:n].cpu().numpy(), ref, rtol=1e-4, atol=2e-2)


def test_realnvp_interleaved_partial_mixture_and_rows_independent():
    """The default handle runs the interleaved s / t kernel for every component count and every work-unit split, and the last
    unit of a tile reduces the mixture terms in component order: a row slice is BITWISE equal to the same rows of the full batch."""
    md = orc.make_synthetic_model("realnvp", 6, 4, 5, 256, seed=4)
    x = torch.from_numpy(np.random.default_rng(2).standard_normal((4096 + 5, 6)).astype(np.float32)).cuda()
    m = build_model(md, "cuda", gemm_mode="f16fast")
    try:
        for n_mix in (4, 3):
            G = m.mixture_log_density(x, n_mix)
            assert m.info()["two_chain"] == 2, (n_mix, m.info())
            for a_, b_ in ((0, 1), (7, 140), (1000, 4101)):
                assert torch.equal(m.mixture_log_density(x[a_:b_].contiguous(), n_mix), G[a_:b_]), (n_mix, a_, b_)
                assert m.info()["two_chain"] == 2
        m.check_status()
    finally:
        m.release()


def test_odd_component_counts_use_two_chain_for_the_even_part():
    """n = 3, 5, 7 components: two-chain kernel on the first n - 1 (mixture terms only), single-chain kernel on the last one, whose
    reduce covers all terms -> bitwise equal to the single-chain kernel on all n; also the log q matrix and a large ragged batch."""
    md = orc.make_synthetic_model("glow", 43, 8, 3, 512, seed=6)
    x = torch.from_numpy(np.random.default_rng(11).standard_normal((20000 + 3, 43)).astype(np.float32)).cuda()
    m = _model(md, "f16fast", None)
    m0 = _model(md, "f16fast", 0)
    try:
        for n_mix in (3, 5, 7):
            l0 = m.info()["launches"]
            G, lq = m.mixture_log_density(x, n_mix, return_logq=True)
            assert m.info()["launches"] - l0 == 2, "even part + last component"
            G0, lq0 = m0.mixture_log_density(x, n_mix, return_logq=True)
            assert torch.equal(G, G0) and torch.equal(lq, lq0)
        assert torch.equal(m.component_log_density(x, 1, 6), m0.component_log_density(x, 1, 6))      # 5 components, log q only
        m.check_status()
    finally:
        m.release(); m0.release()
