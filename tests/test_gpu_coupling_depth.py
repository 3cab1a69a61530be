"""Every coupling-network depth the library accepts (-m gpu), against the fp64 oracle.

The f16 modes run a shape on the serial tensor-core kernel (coupling_tc.cuh) when the pipelined kernels do not serve it:
coupling_network_depth 0, 2, 3 or 4 at any h <= 512 (padded to the next multiple of 64), and depth 1 at h = 64, 192, 320 or
448.  The exact fp32 kernel (coupling_fp32.cuh) runs the same models, and is the only kernel for depth > 1 with h > 512.  Each
case asserts the kernel it ran on (model.info()), so that a routing change cannot move it to another kernel unnoticed.

Tolerances are those of tests/test_gpu_parity.py: 1e-4 relative on log q and G_ll in the f16 modes, plus an absolute 2e-2
for RealNVP and for D < 16; 1e-5 relative in fp32; 2e-2 on z / ldj in every mode.

Measured on an NVIDIA B200 (1000 W power limit), largest f16 / f16fast error on log q against the oracle per depth.  Glow with
D >= 16, relative: 1.9e-5 at depth 3, 2.0e-5 at 2, 3.5e-5 at 1, 4.0e-5 at 0 (RealNVP D = 64 at depth 4: 1.3e-5).  RealNVP and
D < 16, absolute: 1.3e-3 at depth 4, 7.1e-5 at 3, 3.2e-3 at 2, 5.7e-3 at 1, 2.3e-2 at 0.  The depth-0 value (realnvp_bn_d6_h128_depth0, on a row with
|log q| = 37, inside its bound of 2.4e-2) is the fp16 rounding of the GEMM operands: the oracle with its matrix-product operands
rounded to fp16 gives the same 2.32e-2.  fp32: at most 4.6e-7 relative at every depth."""
import numpy as np
import pytest
import torch

from gbnf_b200._lib import GbnfError
from helpers import build_model
from oracle import gbnf_oracle as orc

pytestmark = pytest.mark.gpu

F16_MODES = ["f16", "f16fast"]
ALL_MODES = ["f16", "f16fast", "fp32"]
TOL = {"fp32": 1e-5, "f16": 1e-4, "f16fast": 1e-4}
F16_ATOL = {"glow": 0.0, "realnvp": 2e-2}

# (kind, D, C, K, h, extra model args).  Together: depth 0 .. 4, h = 64 .. 512 in steps of 64 (300 pads to 320), D = 2 .. 64,
# Glow affine / additive, RealNVP tanh / relu / mixed, BatchNorm, the toy base.  realnvp_bn_d64_h512_depth4 is the largest
# shared-memory layout the serial kernel's plan accepts (194 048 B before the weight ring: two 16 KB ring stages).
SERIAL_CASES = {
    "glow_d43_h192_depth1": ("glow", 43, 3, 2, 192, {}),
    "glow_additive_relu_d21_h320_depth1": ("glow", 21, 2, 3, 320, dict(coupling="additive", act="relu")),
    "realnvp_mixed_bn_d9_h448_depth1": ("realnvp", 9, 2, 3, 448, dict(act="mixed", batch_norm=True)),
    "glow_d43_h256_depth0": ("glow", 43, 2, 2, 256, dict(depth=0)),
    "realnvp_bn_d6_h128_depth0": ("realnvp", 6, 2, 3, 128, dict(depth=0, batch_norm=True)),
    "glow_d64_h512_depth2": ("glow", 64, 2, 2, 512, dict(depth=2)),
    "realnvp_mixed_d6_h256_depth2": ("realnvp", 6, 4, 5, 256, dict(depth=2, act="mixed")),
    "glow_d43_h300_depth2": ("glow", 43, 2, 2, 300, dict(depth=2)),
    "glow_relu_d63_h384_depth3": ("glow", 63, 2, 2, 384, dict(depth=3, act="relu")),
    "realnvp_relu_toy_d2_h256_depth3": ("realnvp", 2, 3, 2, 256, dict(depth=3, act="relu", toy_base=True)),
    "glow_additive_d5_h64_depth4": ("glow", 5, 2, 3, 64, dict(depth=4, coupling="additive")),
    "realnvp_bn_d64_h512_depth4": ("realnvp", 64, 2, 2, 512, dict(depth=4, batch_norm=True)),
}
# depth > 1 with h > 512: the f16 modes refuse these (test_gpu_hidden_width.py), the fp32 kernel runs them
FP32_CASES = {
    "glow_d21_h640_depth2": ("glow", 21, 2, 2, 640, dict(depth=2)),
    "realnvp_bn_d6_h1024_depth3": ("realnvp", 6, 2, 2, 1024, dict(depth=3, batch_norm=True)),
}
CASES = {**SERIAL_CASES, **FP32_CASES}


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def synth(name, seed=3):
    kind, D, C, K, h, kw = CASES[name]
    return orc.make_synthetic_model(kind, D, C, K, h, seed=seed, init_rows=1024, **kw)


def family(md):
    return "realnvp" if md["kind"] == "realnvp" or md["D"] < 16 else "glow"


def close(got, ref, mode, md, what=""):
    got = np.asarray(got.cpu() if torch.is_tensor(got) else got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    atol = F16_ATOL[family(md)] if mode != "fp32" else 0.0
    err = np.abs(got - ref)
    bad = err > TOL[mode] * np.abs(ref) + atol + 2e-6 * np.abs(ref)
    rel = float(np.max(err / np.abs(ref)))
    print(f"[{mode} depth {md['depth']} h {md['h']} {what}] max abs err {float(err.max()):.3e}, max rel err {rel:.3e}")
    assert not bad.any(), (what, mode, float(err.max()), rel)


def assert_route(model, mode):
    """The kernel the handle's last launch ran on: the serial tensor-core kernel, or the fp32 kernel."""
    inf = model.info()
    if mode == "fp32":
        assert inf["tmem_cols"] == 0, inf
    else:
        assert inf["pipelined"] == 0 and inf["two_chain"] == 0 and inf["tmem_cols"] == 512, inf
    return inf


def rows(D, B, seed=21):
    return np.random.default_rng(seed).standard_normal((B, D)).astype(np.float32)


# ---- 1. the serial kernel across its envelope, and the fp32 kernel on the same models -----------------------------------------
@pytest.mark.parametrize("name,mode", [(n, m) for n in SERIAL_CASES for m in ALL_MODES] + [(n, "fp32") for n in FP32_CASES])
def test_depth_and_width_vs_oracle(name, mode):
    md = synth(name)
    C = md["C"]
    x = rows(md["D"], 517)                                   # four full 128-row tiles and a ragged one
    xd = dev(x)
    model = build_model(md, "cuda", gemm_mode=mode)
    try:
        G, lq = model.mixture_log_density(xd, C, return_logq=True)
        assert_route(model, mode)
        z, ldj = model.component_forward(xd, C - 1)
        assert_route(model, mode)
        model.check_status()
        m64 = orc.cast_model(md, np.float64)
        ref = orc.all_component_logq(m64, x.astype(np.float64))
        close(lq, ref, mode, md, "log q")
        close(G, orc.mixture_recursion(ref, md["rho"].astype(np.float64), C), mode, md, "G_ll")
        zr, ldjr = orc.component_forward(m64, x.astype(np.float64), C - 1)
        np.testing.assert_allclose(z.cpu().numpy(), zr, rtol=2e-2, atol=2e-2)
        np.testing.assert_allclose(ldj.cpu().numpy(), ldjr, rtol=2e-2, atol=2e-2)
        # the unfused call and a component sub-range give the fused call's bits
        assert torch.equal(model.component_log_density(xd), lq)
        assert torch.equal(model.component_log_density(xd, 1, C), lq[:, 1:])
        # ragged batches around the 128-row tile give the rows of the full batch
        for B in (1, 127, 129):
            Gb, lqb = model.mixture_log_density(dev(x[:B]), C, return_logq=True)
            assert torch.equal(Gb, G[:B]) and torch.equal(lqb, lq[:B]), B
        model.check_status()
    finally:
        model.release()


# ---- 2. persistent CTAs walking several tiles ----------------------------------------------------------------------------------
# Each tile is computed independently, so a CTA that walks several tiles (its weight ring, mbarrier phases, per-tile logsumexp
# and z tile carried from one tile to the next) must give the bits of one CTA per tile.  GBNF_GRID caps the grid at every launch.
GRID_CASES = ["glow_d43_h192_depth1", "realnvp_mixed_d6_h256_depth2", "realnvp_bn_d64_h512_depth4"]


@pytest.mark.parametrize("mode", ALL_MODES)
@pytest.mark.parametrize("name", GRID_CASES)
def test_capped_grid_is_bitwise_equal(name, mode, monkeypatch):
    md = synth(name)
    C = md["C"]
    xd = dev(rows(md["D"], 517))
    model = build_model(md, "cuda", gemm_mode=mode)
    try:
        def run():
            G, lq = model.mixture_log_density(xd, C, return_logq=True)
            z, ldj = model.component_forward(xd, C - 1)
            return (G, lq, z, ldj), assert_route(model, mode)

        base, inf = run()
        assert inf["grid"] == -(-517 // inf["rows_per_cta"]), inf      # one tile per CTA
        for grid in (1, 2):
            monkeypatch.setenv("GBNF_GRID", str(grid))
            got, inf = run()
            assert inf["grid"] == grid, inf
            for k, a, b in zip(("G_ll", "log q", "z", "ldj"), base, got):
                assert torch.equal(a, b), (grid, k)
        model.check_status()
    finally:
        model.release()


_BIG_REF = {}


@pytest.mark.parametrize("mode", ALL_MODES)
def test_every_cta_walks_at_least_two_tiles_vs_oracle(mode):
    md = synth("glow_d43_h192_depth1")
    C = md["C"]
    model = build_model(md, "cuda", gemm_mode=mode)
    try:
        sms = model.info()["num_sms"]
        B = 2 * sms * 128 + 77                              # 2 sms + 1 tiles of 128 rows, the last one ragged
        x = rows(md["D"], B, seed=22)
        G, lq = model.mixture_log_density(dev(x), C, return_logq=True)
        inf = assert_route(model, mode)
        assert inf["grid"] == sms and -(-B // inf["rows_per_cta"]) > 2 * sms, inf
        model.check_status()
        if B not in _BIG_REF:                               # about a second of host time, shared by the three modes
            _BIG_REF[B] = orc.all_component_logq(orc.cast_model(md, np.float64), x.astype(np.float64))
        ref = _BIG_REF[B]
        close(lq, ref, mode, md, "log q")
        close(G, orc.mixture_recursion(ref, md["rho"].astype(np.float64), C), mode, md, "G_ll")
    finally:
        model.release()


# ---- 3. the serial kernel's own mixture reduction (in-kernel online logsumexp) ---------------------------------------------------
MIX_CASES = {
    "realnvp_mixed_d6_h256_depth2": CASES["realnvp_mixed_d6_h256_depth2"],      # C = 4
    "glow_d21_c6_h128_depth3": ("glow", 21, 6, 2, 128, dict(depth=3)),
    "glow_d8_c20_h64": ("glow", 8, 20, 1, 64, {}),                              # more terms than the 16 kept in registers elsewhere
}


@pytest.mark.parametrize("mode", ALL_MODES)
@pytest.mark.parametrize("name", list(MIX_CASES))
def test_fused_mixture_settings_vs_oracle(name, mode):
    kind, D, C, K, h, kw = MIX_CASES[name]
    md = orc.make_synthetic_model(kind, D, C, K, h, seed=4, init_rows=1024, **kw)
    x = rows(D, 517, seed=23)
    xd = dev(x)
    model = build_model(md, "cuda", gemm_mode=mode)
    try:
        _, lq = model.mixture_log_density(xd, C, return_logq=True)
        assert_route(model, mode)
        ref = orc.all_component_logq(orc.cast_model(md, np.float64), x.astype(np.float64))
        close(lq, ref, mode, md, "log q")
        rho = md["rho"].astype(np.float64)
        for n in sorted({1, 2, C - 1, C}):
            for skip_c in (-1, 1, C - 1):
                for raw in (False, True):
                    G = model.mixture_log_density(xd, n, skip_c=skip_c, raw_rho=raw)
                    close(G, orc.mixture_recursion(ref, rho, n, skip_c, normalized=not raw), mode, md,
                          f"G_ll n {n} skip_c {skip_c} raw_rho {raw}")
                    # the standalone mixture kernel on the kernel's own log q: the same value up to logsumexp reassociation
                    Gu = model.mixture_from_logq(lq, n, skip_c=skip_c, raw_rho=raw)
                    np.testing.assert_allclose(Gu.cpu().numpy(), G.cpu().numpy(), rtol=2e-6, atol=2e-6)
        model.check_status()
    finally:
        model.release()


# ---- 4. range reporting and refusals specific to deep networks -------------------------------------------------------------------
@pytest.mark.parametrize("mode", F16_MODES)
def test_relu_overflow_in_a_later_hidden_layer_is_reported(mode):
    # additive coupling keeps the fp32 density finite (an affine step's sigmoid would underflow to a log-density of -inf)
    md = orc.make_synthetic_model("glow", 8, 1, 2, 128, seed=5, depth=3, act="relu", coupling="additive")
    x = torch.randn(300, 8, device="cuda", generator=torch.Generator(device="cuda").manual_seed(9))
    model = build_model(md, "cuda", gemm_mode=mode)
    ref = build_model(md, "cuda", gemm_mode="fp32")
    try:
        model.mixture_log_density(x, 1)
        assert_route(model, mode)
        model.check_status()                                 # in range before the edit
        for m in (model, ref):
            with torch.no_grad():                            # network[4]: hidden layer 2, the second hidden-to-hidden Linear
                m.flows[0].flow.layers[0].block.network[4].bias.fill_(7.0e4)
        model.mixture_log_density(x, 1)
        with pytest.raises(GbnfError, match="not finite in fp16") as e:
            model.check_status()
        assert e.value.code == -4
        G = ref.mixture_log_density(x, 1)
        ref.check_status()
        assert torch.isfinite(G).all()
    finally:
        model.release()
        ref.release()


@pytest.mark.parametrize("mode", F16_MODES)
@pytest.mark.parametrize("h,depth", [(128, 2), (192, 1)])
def test_serial_kernel_refuses_the_inverse(h, depth, mode):
    md = orc.make_synthetic_model("glow", 10, 2, 2, h, seed=7, depth=depth)
    model = build_model(md, "cuda", gemm_mode=mode)
    try:
        x = torch.randn(64, 10, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
        z, _ = model.component_forward(x, 1)
        assert_route(model, mode)
        with pytest.raises(GbnfError, match="serial tensor-core kernel"):
            model.component_inverse(z, 1)
        with pytest.raises(GbnfError, match="serial tensor-core kernel"):
            model(z=z, components=0, reverse=True)
        model.component, model.all_trained = 1, True
        with pytest.raises(GbnfError, match="serial tensor-core kernel"):
            model.sample(100, generator=torch.Generator(device="cuda").manual_seed(4))
        model.check_status()
    finally:
        model.release()
