"""Hidden widths the f16 tensor-core kernels do not run natively (-m gpu): zero padding of the hidden width in the handle's plan,
and RealNVP components with 512 < h <= 1024 on the CTA-pair kernel (coupling_tc3.cuh, RNVP = 1).

A padded hidden unit has zero weights and a zero bias: it computes act(0) = 0 exactly and meets zero weights in the next layer.
So a handle at the true width h gives the same bits as a handle at the padded width hp whose extra rows, columns and bias entries
are explicit zeros.  Against the fp64 oracle the tolerances are those of tests/test_gpu_parity.py: 1e-4 relative on log q, plus
an absolute 2e-2 for RealNVP and for low-dimensional data."""
import argparse
import copy

import numpy as np
import pytest
import torch

import gbnf_b200
from gbnf_b200._lib import GbnfError
from helpers import args_for, build_model, load_into
from oracle import gbnf_oracle as orc

pytestmark = pytest.mark.gpu

MODES = ["f16", "f16fast"]
TOL = 1e-4
F16_ATOL = {"glow": 0.0, "realnvp": 2e-2}


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def close(got, ref, fam, scale=1.0):
    got = np.asarray(got, dtype=np.float64); ref = np.asarray(ref, dtype=np.float64)
    bound = scale * (TOL * np.abs(ref) + F16_ATOL[fam]) + 2e-6 * np.abs(ref)
    bad = np.abs(got - ref) > bound
    assert not bad.any(), (fam, float(np.max(np.abs(got - ref))), float(np.max(np.abs(got - ref) / np.maximum(np.abs(ref), 1e-30))))


def family(md):
    return "realnvp" if md["kind"] == "realnvp" or md["D"] < 16 else "glow"


def synth(kind, D, C, K, h, seed=3, **kw):
    return orc.make_synthetic_model(kind, D, C, K, h, seed=seed, init_rows=1024, **kw)


def pad_model(md, hp):
    """The same model at hidden width hp: every hidden layer gains hp - h zero units (zero weight rows, bias entries and
    the matching zero weight columns of the next layer)."""
    out = copy.deepcopy(md)
    out["h"] = hp
    for comp in out["components"]:
        for st in comp["steps"]:
            for key in (("net",) if md["kind"] == "glow" else ("t", "s")):
                layers = st[key]
                n = len(layers)
                for i, (W, b) in enumerate(layers):
                    rows = hp - W.shape[0] if i < n - 1 else 0
                    cols = hp - W.shape[1] if i > 0 else 0
                    layers[i] = (np.pad(W, ((0, rows), (0, cols))), np.pad(b, (0, rows)))
    return out


def outputs(model, x, C, inverse):
    """log q of every component, the fused G_ll, z / ldj and the inverse (x, ldj) of the last component, and the handle's
    info() after the fused evaluation (which kernel it took)."""
    r = {"lq": model.component_log_density(x)}
    r["G"], r["lq_fused"] = model.mixture_log_density(x, C, return_logq=True)
    inf = model.info()
    r["z"], r["ldj"] = model.component_forward(x, C - 1)
    if inverse:
        r["xi"], r["ldji"] = model.component_inverse(r["z"], C - 1)
    torch.cuda.synchronize()
    return r, inf


# one case per route: (kind, D, C, K, h, extra model args, kernel {pipelined: 0 serial / 1 pipelined / 2 pair}, alternative)
PAD_CASES = {
    "glow_h1": ("glow", 7, 2, 2, 1, {}, 1, 0),
    "realnvp_relu_h17": ("realnvp", 6, 2, 2, 17, dict(act="relu", batch_norm=True), 1, 0),
    "glow_additive_h60": ("glow", 21, 2, 2, 60, dict(coupling="additive"), 1, 0),
    "realnvp_mixed_h100": ("realnvp", 5, 2, 3, 100, dict(act="mixed", toy_base=True), 1, 0),
    "realnvp_tanh_h200_interleaved": ("realnvp", 6, 2, 2, 200, {}, 1, 2),
    "glow_h215_single_chain": ("glow", 43, 2, 2, 215, {}, 1, 0),
    "glow_h430_two_chain": ("glow", 43, 2, 2, 430, {}, 1, 1),
    "glow_depth2_h100_serial": ("glow", 10, 2, 2, 100, dict(depth=2), 0, 0),
    "glow_h600_pair": ("glow", 21, 2, 2, 600, {}, 2, 0),
    "glow_h630_pair": ("glow", 63, 2, 2, 630, {}, 2, 0),
    "realnvp_h600_pair": ("realnvp", 21, 2, 2, 600, dict(batch_norm=True), 2, 0),
}


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", list(PAD_CASES))
def test_padding_is_bitwise_exact(name, mode, monkeypatch):
    kind, D, C, K, h, kw, kernel, alt = PAD_CASES[name]
    if alt == 1:
        monkeypatch.setenv("GBNF_TC4", "2")     # few tiles: prefer the two-chain kernel over one component per work unit
    md = synth(kind, D, C, K, h, **kw)
    hp = {0: -(-h // 64) * 64, 1: -(-h // 128) * 128, 2: 1024}[kernel]
    x = dev(np.random.default_rng(11).standard_normal((517, D)).astype(np.float32))
    res = []
    for m in (md, pad_model(md, hp)):
        model = build_model(m, "cuda", gemm_mode=mode)
        try:
            r, inf = outputs(model, x, C, inverse=kernel > 0)
            assert inf["pipelined"] == kernel and inf["two_chain"] == alt, inf
            model.check_status()
            res.append(r)
        finally:
            model.release()
    for k in res[0]:
        assert torch.equal(res[0][k], res[1][k]), (name, k)
    assert all(torch.isfinite(v).all() for v in res[0].values())


ORACLE_CASES = {
    "glow_affine_d2_h215": ("glow", 2, 2, 2, 215, {}),
    "glow_additive_d5_h100": ("glow", 5, 2, 2, 100, dict(coupling="additive")),
    "glow_affine_d43_h430": ("glow", 43, 2, 2, 430, {}),
    "glow_affine_relu_d63_h630": ("glow", 63, 2, 2, 630, dict(act="relu")),
    "glow_additive_d43_h700": ("glow", 43, 3, 2, 700, dict(coupling="additive")),
    "realnvp_tanh_bn_d5_h60": ("realnvp", 5, 2, 3, 60, dict(batch_norm=True)),
    "realnvp_mixed_toy_d2_h17": ("realnvp", 2, 2, 2, 17, dict(act="mixed", toy_base=True)),
    "realnvp_tanh_d63_h200": ("realnvp", 63, 2, 2, 200, {}),
    "realnvp_relu_bn_d43_h600": ("realnvp", 43, 2, 2, 600, dict(act="relu", batch_norm=True)),
    "realnvp_mixed_toy_d63_h1000": ("realnvp", 63, 3, 2, 1000, dict(act="mixed", toy_base=True)),
    "realnvp_tanh_d2_h1024": ("realnvp", 2, 2, 2, 1024, {}),
}


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", list(ORACLE_CASES))
def test_padded_and_pair_shapes_vs_oracle(name, mode):
    kind, D, C, K, h, kw = ORACLE_CASES[name]
    md = synth(kind, D, C, K, h, **kw)
    x = np.random.default_rng(21).standard_normal((517, D)).astype(np.float32)
    model = build_model(md, "cuda", gemm_mode=mode)
    try:
        m64 = orc.cast_model(md, np.float64)
        ref = orc.all_component_logq(m64, x.astype(np.float64))
        G, lq = model.mixture_log_density(dev(x), C, return_logq=True)
        model.check_status()
        close(lq.cpu().numpy(), ref, family(md))
        close(G.cpu().numpy(), orc.mixture_recursion(ref, md["rho"].astype(np.float64), C), family(md))
        z, ldj = model.component_forward(dev(x), C - 1)
        zr, ldjr = orc.component_forward(m64, x.astype(np.float64), C - 1)
        np.testing.assert_allclose(z.cpu().numpy(), zr, rtol=2e-2, atol=2e-2)
        np.testing.assert_allclose(ldj.cpu().numpy(), ldjr, rtol=2e-2, atol=2e-2)
        # ragged batches across the 128-row tiles give the rows of the full batch
        for B in (1, 127, 129, 300):
            assert torch.equal(model.mixture_log_density(dev(x[:B]), C), G[:B]), B
    finally:
        model.release()


# ---- RealNVP on the CTA-pair kernel -----------------------------------------------------------------------------------------
def rnvp_pair(D, C, K, mode, seed=5, **kw):
    md = synth("realnvp", D, C, K, 1024, seed=seed, **kw)
    model = build_model(md, "cuda", gemm_mode=mode)
    assert model.info()["pipelined"] == 2
    return md, model


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("K", [1, 3])
def test_realnvp_pair_vs_oracle_and_round_trip(K, mode):
    # C = 3 (odd): components 0 and 2 start unflipped, component 1 flipped; D = 63 (odd) gives |z1| != |z2| both ways
    md, model = rnvp_pair(63, 3, K, mode, batch_norm=True)
    x = np.random.default_rng(31).standard_normal((517, 63)).astype(np.float32)
    try:
        m64 = orc.cast_model(md, np.float64)
        ref = orc.all_component_logq(m64, x.astype(np.float64))
        G, lq = model.mixture_log_density(dev(x), 3, return_logq=True)
        close(lq.cpu().numpy(), ref, "realnvp")
        close(G.cpu().numpy(), orc.mixture_recursion(ref, md["rho"].astype(np.float64), 3), "realnvp")
        for c in range(3):
            z64, ldj64 = orc.component_forward(m64, x.astype(np.float64), c)
            xk, ldjk = model.component_inverse(dev(z64.astype(np.float32)), c)
            xo, ldjo = orc.component_inverse(m64, z64, c)
            np.testing.assert_allclose(xk.cpu().numpy(), xo, rtol=3e-2, atol=3e-2)
            np.testing.assert_allclose(ldjk.cpu().numpy(), ldjo, rtol=3e-2, atol=3e-2)
            z, ldj = model.component_forward(dev(x), c)
            xr, ldji = model.component_inverse(z, c)
            err, err_ldj = float((xr - dev(x)).abs().max()), float((ldj + ldji).abs().max())
            print(f"[K = {K}, {mode}, c = {c}] round trip: max |x - f^-1(f(x))| = {err:.3e}, max |ldj + ldj_inv| = {err_ldj:.3e}")
            # fp32 resolution of the largest value the round trip passes through (z2 = BN(z2) e^s + t) bounds it
            scale = max(1.0, float(z.abs().max()), float(np.abs(x).max()))
            assert err < 2e-4 * scale and err_ldj < 2e-4 * max(1.0, float(ldj.abs().max())), (c, err, err_ldj, scale)
        model.check_status()
    finally:
        model.release()


@pytest.mark.parametrize("mode", MODES)
def test_realnvp_pair_slices_determinism_and_fp32(mode):
    md, model = rnvp_pair(21, 2, 2, mode, act="mixed")
    N = 20000
    x = torch.randn(N, 21, device="cuda", generator=torch.Generator(device="cuda").manual_seed(5))
    try:
        G = model.mixture_log_density(x, 2)
        z, ldj = model.component_forward(x, 1)
        xi, ldji = model.component_inverse(z, 1)
        assert torch.equal(model.mixture_log_density(x, 2), G)
        z2, ldj2 = model.component_forward(x, 1)
        assert torch.equal(z2, z) and torch.equal(ldj2, ldj)
        xi2, ldji2 = model.component_inverse(z, 1)
        assert torch.equal(xi2, xi) and torch.equal(ldji2, ldji)
        for r0, r1 in ((0, 1), (0, 129), (5000, 5300), (127, 129)):
            assert torch.equal(model.mixture_log_density(x[r0:r1].contiguous(), 2), G[r0:r1]), (r0, r1)
            xs, ls = model.component_inverse(z[r0:r1].contiguous(), 1)
            assert torch.equal(xs, xi[r0:r1]) and torch.equal(ls, ldji[r0:r1]), (r0, r1)
        model.check_status()
    finally:
        model.release()
    ref = build_model(md, "cuda", gemm_mode="fp32")
    try:
        G32 = ref.mixture_log_density(x[:517], 2)
        x32, l32 = ref.component_inverse(z[:517], 1)
    finally:
        ref.release()
    close(G[:517].cpu().numpy(), G32.cpu().numpy(), "realnvp")
    np.testing.assert_allclose(xi[:517].cpu().numpy(), x32.cpu().numpy(), rtol=3e-2, atol=3e-2)
    np.testing.assert_allclose(ldji[:517].cpu().numpy(), l32.cpu().numpy(), rtol=3e-2, atol=3e-2)


@pytest.mark.parametrize("mode", MODES)
def test_realnvp_pair_reports_values_outside_fp16(mode):
    md, model = rnvp_pair(10, 1, 2, mode)
    x = torch.randn(300, 10, device="cuda", generator=torch.Generator(device="cuda").manual_seed(8))
    bad = x.clone()
    bad[150] = 1e6
    try:
        model.component_log_density(bad)
        with pytest.raises(GbnfError, match="not finite in fp16"):
            model.check_status()
        model.component_inverse(bad, 0)
        with pytest.raises(GbnfError, match="not finite in fp16"):
            model.check_status()
        lq = model.component_log_density(x)              # the handle stays usable
        model.check_status()
        assert torch.isfinite(lq).all()
    finally:
        model.release()


@pytest.mark.parametrize("mode", MODES)
def test_realnvp_pair_above_the_launch_slice(mode):
    md, model = rnvp_pair(9, 1, 1, mode)
    B = (1 << 22) + 300
    x = torch.randn(B, 9, device="cuda", generator=torch.Generator(device="cuda").manual_seed(6))
    try:
        lq = model.component_log_density(x)
        assert torch.equal(model.component_log_density(x[-400:].contiguous()), lq[-400:])
        xi, ldji = model.component_inverse(x, 0)
        xt, lt = model.component_inverse(x[-400:].contiguous(), 0)
        assert torch.equal(xi[-400:], xt) and torch.equal(ldji[-400:], lt)
        m64 = orc.cast_model(md, np.float64)
        close(lq[-400:].cpu().numpy(), orc.all_component_logq(m64, x[-400:].cpu().numpy().astype(np.float64)), "realnvp")
        xo, _ = orc.component_inverse(m64, x[-400:].cpu().numpy().astype(np.float64), 0)
        np.testing.assert_allclose(xt.cpu().numpy(), xo, rtol=3e-2, atol=3e-2)
        model.check_status()
    finally:
        model.release()


# ---- upstream's getting-started density shape: Glow, D = 43, h = h_size_factor 5 x 43 = 215, default gemm_mode ----------------
def _reference_grads(model, c, x, dz, dldj):
    """fp64 autograd gradients of component c's parameters (module order) for upstream (dz, dldj)."""
    flow = copy.deepcopy(model.flows[c]).to(torch.float64)
    for s_src, s_dst in zip(model.flows[c].steps(), flow.steps()):
        s_dst.permutation.set_indices(s_src.permutation.indices)
        s_dst.actnorm.inited = True
    params = list(flow.parameters())
    for p in params:
        p.requires_grad_(True)
    z, ldj = flow.forward_autograd(x.double())
    return torch.autograd.grad((z, ldj), params, grad_outputs=(dz.double(), dldj.double()))


def test_getting_started_shape_end_to_end():
    md = synth("glow", 43, 2, 2, 215, seed=9)
    model = gbnf_b200.BoostedFlow(args_for(md, "cuda"))
    load_into(model, md)
    model = model.to("cuda").eval()
    ref = build_model(md, "cuda", gemm_mode="fp32")
    try:
        assert model.gemm_mode == "f16"
        gen = torch.Generator(device="cuda").manual_seed(3)
        x = torch.randn(1000, 43, device="cuda", generator=gen)
        with torch.no_grad():
            out = model(x=x, components="c")
        assert len(out) == 5 and out[0].shape == (1000, 43) and out[3].shape == (1000,)
        assert model.info()["pipelined"] == 1
        args = argparse.Namespace(flow="boosted", boosted=True, device=torch.device("cuda"))
        for m in (model, ref):
            m.component, m.all_trained = 1, False
        with torch.no_grad():
            l16 = gbnf_b200.compute_kl_pq_loss(model, x, args, generator=torch.Generator(device="cuda").manual_seed(4))
            l32 = gbnf_b200.compute_kl_pq_loss(ref, x, args, generator=torch.Generator(device="cuda").manual_seed(4))
        close(l16["G_nll"].item(), l32["G_nll"].item(), "glow")
        for m in (model, ref):
            m.component = 0
        with torch.no_grad():
            close(gbnf_b200.compute_kl_pq_loss(model, x, args)["nll"].item(), gbnf_b200.compute_kl_pq_loss(ref, x, args)["nll"].item(),
                  "glow")
        for m in (model, ref):
            m.component = 1
        loader = [(x[:500], None), (x[500:], None)]
        e16, e32 = gbnf_b200.evaluate(model, loader, args), gbnf_b200.evaluate(ref, loader, args)
        for k in ("nll", "g_nll"):
            close(e16[k], e32[k], "glow")
        xs, comp = model.sample(777, generator=torch.Generator(device="cuda").manual_seed(5))
        assert xs.shape == (777, 43) and torch.isfinite(xs).all() and set(comp.unique().tolist()) <= {0, 1}
        # training the new component: forward and backward through the library, against fp64 autograd
        for i, f in enumerate(model.flows):
            for p in f.parameters():
                p.requires_grad_(i == 1)
        g = torch.Generator(device="cuda").manual_seed(6)
        dz = torch.randn(1000, 43, device="cuda", generator=g) / 1000
        dldj = (torch.rand(1000, device="cuda", generator=g) * 2 - 1) / 1000
        z, _, _, ldj, _ = model(x=x, components="c")
        assert type(z.grad_fn).__name__.startswith("_FusedComponentFlow")
        ((z * dz).sum() + (ldj * dldj).sum()).backward()
        for p, r in zip(model.flows[1].parameters(), _reference_grads(model, 1, x, dz, dldj)):
            err, scale = float((p.grad.double() - r).abs().max()), float(r.abs().max())
            assert err <= 1e-4 * scale + 1e-7, (tuple(r.shape), err, scale)
        model.check_status()
    finally:
        model.release()
        ref.release()


# ---- shapes that stay refused in the f16 modes ---------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("kind,h,depth", [("realnvp", 600, 2), ("realnvp", 1100, 1), ("glow", 1100, 1), ("glow", 800, 2)])
def test_widths_beyond_the_tensor_core_kernels_are_refused(kind, h, depth, mode):
    md = synth(kind, 10, 1, 1, h, depth=depth)
    model = build_model(md, "cuda", gemm_mode=mode)
    try:
        with pytest.raises(GbnfError, match="<= 512, or <= 1024 with coupling_network_depth 1"):
            model.component_log_density(torch.randn(8, 10, device="cuda"))
    finally:
        model.release()
