"""Sampling with gradients (-m gpu): the fused backward of the inverse map (gbnf_component_inverse_backward /
gbnf_mixture_inverse_backward) and BoostedFlow.rsample, against fp64 autograd through the host mirror's inverse_autograd.

Every gradient tensor, dL/dz included, is held to max|g - g_ref| <= 1e-4 max|g_ref| + 1e-7.  The backward computes in fp32 on
CUDA cores whatever the handle's GEMM mode, so fp32, f16 and f16fast handles are all held to that bound.
"""
import copy
import ctypes
import math

import numpy as np
import pytest
import torch

import gbnf_b200
from gbnf_b200 import _lib
from gbnf_b200 import boosted_flow as bf
from helpers import build_model
from oracle import gbnf_oracle as orc

pytestmark = pytest.mark.gpu

TOL = 1e-4


def _model(kind, D, h, K, C=2, depth=1, act="tanh", coupling="affine", mode="fp32", seed=5, fused_backward=True, **kw):
    md = orc.make_synthetic_model(kind, D, C, K, h, seed=seed, depth=depth, act=act, coupling=coupling, init_rows=512, **kw)
    return build_model(md, "cuda", gemm_mode=mode, fused_backward=fused_backward)


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _upstream(B, D, seed, which="both"):
    g = _gen(seed)
    dx = torch.randn(B, D, device="cuda", generator=g) / B
    dldj = (torch.rand(B, device="cuda", generator=g) * 2 - 1) / B
    if which == "dx":
        dldj.zero_()
    elif which == "dldj":
        dx.zero_()
    return dx, dldj


def _flow64(model, c):
    flow = copy.deepcopy(model.flows[c]).to(torch.float64)
    if model.component_type == "glow":
        for s_src, s_dst in zip(model.flows[c].steps(), flow.steps()):
            if s_src.permutation is not None:
                s_dst.permutation.set_indices(s_src.permutation.indices)
            s_dst.actnorm.inited = True
    return flow


def _reference(model, z, comp, dx, dldj, n_comp):
    """fp64 autograd through inverse_autograd: ({c: [grads in module order]}, dL/dz)."""
    z64 = z.detach().double().requires_grad_(True)
    grads, loss = {}, 0
    flows = {}
    for c in range(n_comp):
        rows = (comp == c).nonzero().flatten()
        flows[c] = _flow64(model, c)
        for p in flows[c].parameters():
            p.requires_grad_(True)
        if len(rows):
            x, ldj = flows[c].inverse_autograd(z64[rows])
            loss = loss + (x * dx[rows].double()).sum() + (ldj * dldj[rows].double()).sum()
    out = torch.autograd.grad(loss, [z64] + [p for c in range(n_comp) for p in flows[c].parameters()], allow_unused=True)
    i = 1
    for c in range(n_comp):
        ps = list(flows[c].parameters())
        grads[c] = [g if g is not None else torch.zeros_like(p) for g, p in zip(out[i:i + len(ps)], ps)]
        i += len(ps)
    return grads, out[0]


def _close(got, ref, what, tol=TOL):
    assert got is not None, what
    assert tuple(got.shape) == tuple(ref.shape), (what, tuple(got.shape), tuple(ref.shape))
    scale = float(ref.abs().max())
    err = float((got.double() - ref).abs().max())
    assert err <= tol * scale + 1e-7, (what, err, scale)


def _component_call(model, c, z, dx, dldj, fill=None):
    """gbnf_component_inverse_backward through ctypes.  Returns (rc, error text, [grads in module order], dz); with `fill` every
    output buffer starts at that value."""
    dev = z.device
    model.pack_component(c)
    keep, out = [], {}
    cp, garr = model._backward_arrays(c, dev, keep, out)
    params = list(model.flows[c].parameters())
    grads = [out.get(id(p)) for p in params]
    dz = torch.empty_like(z)
    for t in [g for g in grads if g is not None] + [dz]:
        t.fill_(float("nan") if fill is None else fill)
    rc = _lib.load().gbnf_component_inverse_backward(model.handle(dev), c, ctypes.byref(cp), ctypes.c_void_p(z.data_ptr()), z.shape[0],
                                                     ctypes.c_void_p(dx.data_ptr()), ctypes.c_void_p(dldj.data_ptr()),
                                                     ctypes.cast(garr, ctypes.POINTER(_lib.StepGrads)), ctypes.c_void_p(dz.data_ptr()),
                                                     ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    torch.cuda.synchronize()
    return rc, _lib.load().gbnf_last_error().decode(), grads, dz


def _check_component(model, c, z, dx, dldj):
    rc, err, grads, dz = _component_call(model, c, z, dx, dldj)
    assert rc == 0, err
    comp = torch.full((z.shape[0],), c, device="cuda", dtype=torch.int64)
    ref, ref_dz = _reference(model, z, comp, dx, dldj, c + 1)
    for i, (g, r) in enumerate(zip(grads, ref[c])):
        _close(g, r, ("param", c, i))
    _close(dz, ref_dz, "dz")


KINDS = {   # (kind, coupling, act, D, h, K)
    "glow_affine_tanh_d43_h512": ("glow", "affine", "tanh", 43, 512, 3),
    "glow_additive_relu": ("glow", "additive", "relu", 7, 64, 3),
    "realnvp_tanh": ("realnvp", "affine", "tanh", 7, 64, 3),
    "realnvp_relu": ("realnvp", "affine", "relu", 7, 128, 3),
    "realnvp_mixed": ("realnvp", "affine", "mixed", 7, 64, 3),
}


@pytest.mark.parametrize("mode", ["fp32", "f16", "f16fast"])
@pytest.mark.parametrize("name", list(KINDS))
def test_envelope_kinds(name, mode):
    """Both Glow couplings, RealNVP with every activation at odd D; components 0 and 1 see both flip parities."""
    kind, coupling, act, D, h, K = KINDS[name]
    model = _model(kind, D, h, K, act=act, coupling=coupling, mode=mode)
    try:
        for c in (0, 1):
            z = torch.randn(300, D, device="cuda", generator=_gen(10 + c))
            dx, dldj = _upstream(300, D, 20 + c)
            _check_component(model, c, z, dx, dldj)
        model.check_status()
    finally:
        model.release()


SHAPES = {   # (kind, act, D, h, K, depth, mode)
    "glow_depth0": ("glow", "tanh", 9, 64, 3, 0, "f16fast"),
    "glow_depth2": ("glow", "relu", 9, 128, 2, 2, "f16"),
    "glow_depth4": ("glow", "tanh", 9, 64, 2, 4, "fp32"),
    "realnvp_depth0": ("realnvp", "mixed", 9, 64, 3, 0, "fp32"),
    "realnvp_depth4": ("realnvp", "tanh", 9, 64, 2, 4, "f16fast"),
    "glow_h100": ("glow", "tanh", 21, 100, 2, 1, "fp32"),
    "realnvp_h215": ("realnvp", "relu", 21, 215, 2, 2, "fp32"),
    "glow_d2": ("glow", "tanh", 2, 64, 3, 1, "f16fast"),
    "realnvp_d2": ("realnvp", "tanh", 2, 64, 3, 1, "fp32"),
    "glow_d64": ("glow", "tanh", 64, 128, 2, 1, "f16fast"),
    "realnvp_d64": ("realnvp", "mixed", 64, 128, 2, 2, "fp32"),
}


@pytest.mark.parametrize("name", list(SHAPES))
def test_depths_widths_and_feature_counts(name):
    kind, act, D, h, K, depth, mode = SHAPES[name]
    model = _model(kind, D, h, K, depth=depth, act=act, mode=mode)
    try:
        for c in (0, 1):
            z = torch.randn(100, D, device="cuda", generator=_gen(30 + c))
            dx, dldj = _upstream(100, D, 40 + c)
            _check_component(model, c, z, dx, dldj)
    finally:
        model.release()


@pytest.mark.parametrize("B", [1, 15, 16, 17, 129, 65536])
def test_batch_sizes(B):
    model = _model("glow", 21, 128, 2, mode="f16fast")
    try:
        z = torch.randn(B, 21, device="cuda", generator=_gen(50))
        dx, dldj = _upstream(B, 21, 51)
        _check_component(model, 1, z, dx, dldj)
    finally:
        model.release()


@pytest.mark.parametrize("which", ["both", "dx", "dldj"])
@pytest.mark.parametrize("kind", ["glow", "realnvp"])
def test_each_upstream_gradient_alone(kind, which):
    model = _model(kind, 11, 64, 3)
    try:
        z = torch.randn(70, 11, device="cuda", generator=_gen(60))
        dx, dldj = _upstream(70, 11, 61, which)
        _check_component(model, 1, z, dx, dldj)
    finally:
        model.release()


@pytest.mark.parametrize("group", [("glow", 43, 512), ("realnvp", 21, 256)], ids=lambda t: "_".join(map(str, t)))
def test_deepest_component_and_one_more(group):
    """The largest K fused_backward_smem_bytes admits is served; K + 1 is refused with every buffer untouched, and rsample
    differentiates it through autograd."""
    kind, D, h = group
    K = 1
    while bf.fused_backward_smem_bytes(kind, D, h, K + 1) <= bf.FUSED_BACKWARD_MAX_SMEM:
        K += 1
    for k, served in ((K, True), (K + 1, False)):
        model = _model(kind, D, h, k, mode="f16fast")
        try:
            z = torch.randn(33, D, device="cuda", generator=_gen(70))
            dx, dldj = _upstream(33, D, 71)
            if served:
                _check_component(model, 1, z, dx, dldj)
            else:
                rc, err, grads, dz = _component_call(model, 1, z, dx, dldj, fill=-3.0)
                assert rc == -1 and "shared-memory" in err, (rc, err)
                assert all(bool((t == -3.0).all()) for t in grads + [dz])
                _check_public(model, 33, seed=72, expect_fused=False)
        finally:
            model.release()


REFUSED = {   # configurations outside the envelope: (kind, D, h, K, depth, extra model args, mode)
    "realnvp_batch_norm": ("realnvp", 6, 64, 3, 1, dict(batch_norm=True), "fp32"),
    "realnvp_residual": ("realnvp", 6, 64, 2, 1, dict(act="residual"), "fp32"),
    "glow_invconv": ("glow", 6, 64, 2, 1, dict(invconv=True), "fp32"),
    "glow_h640": ("glow", 21, 640, 2, 1, {}, "f16fast"),
    "glow_d65": ("glow", 65, 64, 2, 1, {}, "fp32"),
}


@pytest.mark.parametrize("name", list(REFUSED))
def test_refusals_leave_buffers_untouched(name):
    """The library refuses them before writing anything; rsample differentiates them through inverse_autograd instead."""
    kind, D, h, K, depth, kw, mode = REFUSED[name]
    model = _model(kind, D, h, K, depth=depth, mode=mode, **kw)
    try:
        z = torch.randn(40, D, device="cuda", generator=_gen(80))
        dx, dldj = _upstream(40, D, 81)
        if name == "glow_invconv":
            # invconv components carry no permutation to pass: the configuration check refuses before it reads the steps
            cp, garr, dz = _lib.ComponentParams(), (_lib.StepGrads * K)(), torch.full_like(z, 7.0)
            rc = _lib.load().gbnf_component_inverse_backward(model.handle(), 1, ctypes.byref(cp), ctypes.c_void_p(z.data_ptr()), 40,
                                                             ctypes.c_void_p(dx.data_ptr()), ctypes.c_void_p(dldj.data_ptr()),
                                                             ctypes.cast(garr, ctypes.POINTER(_lib.StepGrads)),
                                                             ctypes.c_void_p(dz.data_ptr()), None)
            torch.cuda.synchronize()
            assert rc == -1 and bool((dz == 7.0).all())
        else:
            rc, err, grads, dz = _component_call(model, 1, z, dx, dldj, fill=7.0)
            assert rc == -1, (rc, err)
            assert all(t is None or bool((t == 7.0).all()) for t in grads + [dz])
        _check_public(model, 40, seed=82, expect_fused=False)
    finally:
        model.release()


def test_unpacked_component_is_refused():
    model = _model("glow", 9, 64, 2, C=3)
    try:
        z = torch.randn(20, 9, device="cuda", generator=_gen(85))
        dx, dldj = _upstream(20, 9, 86)
        keep, out = [], {}
        cp, garr = model._backward_arrays(2, z.device, keep, out)
        bufs = list(out.values())
        for t in bufs:
            t.fill_(5.0)
        dz = torch.full_like(z, 5.0)
        rc = _lib.load().gbnf_component_inverse_backward(model.handle(), 2, ctypes.byref(cp), ctypes.c_void_p(z.data_ptr()), 20,
                                                         ctypes.c_void_p(dx.data_ptr()), ctypes.c_void_p(dldj.data_ptr()),
                                                         ctypes.cast(garr, ctypes.POINTER(_lib.StepGrads)), ctypes.c_void_p(dz.data_ptr()),
                                                         None)
        torch.cuda.synchronize()
        assert rc == -3 and "packed" in _lib.load().gbnf_last_error().decode()
        assert all(bool((t == 5.0).all()) for t in bufs + [dz])
    finally:
        model.release()


# ---------------------------------------------------------------------------------------------------------------- mixture
def _mixture_call(model, z, comp, n, dx, dldj, trained):
    grads, dz = model._mixture_inverse_backward(z, comp, n, dx, dldj, trained, with_dz=True)
    torch.cuda.synchronize()
    return {c: [grads[id(p)] for p in model.flows[c].parameters()] for c in trained}, dz


@pytest.mark.parametrize("kind", ["glow", "realnvp"])
def test_mixture_matches_per_component_calls(kind):
    """C = 8, rows in random component order; components 3 and 6 draw no rows, components 1 and 5 need no gradient.  Each
    trained component's W and b equal a component call on its rows alone bit for bit, its ActNorm gradients to 1e-6; dz is
    bitwise the component call's per row; the gradients match fp64 autograd; two identical calls agree bit for bit."""
    D = 11
    model = _model(kind, D, 128, 3, C=8, act="tanh" if kind == "glow" else "mixed", mode="f16")
    try:
        model.pack_all()
        B = 700
        pool = torch.tensor([0, 1, 2, 4, 5, 7], device="cuda")
        comp = pool[torch.randint(0, len(pool), (B,), device="cuda", generator=_gen(90))].contiguous()
        z = torch.randn(B, D, device="cuda", generator=_gen(91))
        dx, dldj = _upstream(B, D, 92)
        trained = {0, 2, 3, 4, 6, 7}
        g1, dz1 = _mixture_call(model, z, comp, 8, dx, dldj, trained)
        g2, dz2 = _mixture_call(model, z, comp, 8, dx, dldj, trained)
        names = {c: [n for n, _ in model.flows[c].named_parameters()] for c in trained}
        assert torch.equal(dz1, dz2)
        ref, ref_dz = _reference(model, z, comp, dx, dldj, 8)
        _close(dz1, ref_dz, "dz")
        for c in trained:
            for i, (g, r) in enumerate(zip(g1[c], ref[c])):
                _close(g, r, ("param", c, i))
            rows = (comp == c).nonzero().flatten()
            if len(rows) == 0:
                assert all(bool((g == 0).all()) for g in g1[c]), c
                continue
            rc, err, gc, dzc = _component_call(model, c, z[rows].contiguous(), dx[rows].contiguous(), dldj[rows].contiguous())
            assert rc == 0, err
            assert torch.equal(dzc, dz1[rows]), c
            for n_, a, b, a2 in zip(names[c], g1[c], gc, g2[c]):
                if "actnorm" in n_:
                    assert float((a - b).abs().max()) <= 1e-6 * float(b.abs().max()) + 1e-12, (c, n_)
                    assert float((a - a2).abs().max()) <= 1e-6 * float(a.abs().max()) + 1e-12, (c, n_)
                else:
                    assert torch.equal(a, b), (c, n_)
                    assert torch.equal(a, a2), (c, n_)
        model.check_status()
    finally:
        model.release()


def test_out_of_range_id_raises_at_check_status():
    model = _model("glow", 9, 64, 2, C=3)
    try:
        model.pack_all()
        comp = torch.tensor([0, 1, 7, 2, 1], device="cuda", dtype=torch.int64)
        z = torch.randn(5, 9, device="cuda", generator=_gen(95))
        dx, dldj = _upstream(5, 9, 96)
        model._mixture_inverse_backward(z, comp, 3, dx, dldj, {0, 1, 2}, with_dz=True)
        with pytest.raises(_lib.GbnfError, match="outside"):
            model.check_status()
        model.check_status()          # reported once; the handle stays usable
    finally:
        model.release()


# ---------------------------------------------------------------------------------------------------------------- public path
def _check_public(model, n, seed, expect_fused=True, n_comp=None):
    """rsample + backward() with every component's parameters and z requiring grad, against fp64 autograd."""
    if n_comp is not None:
        model.component, model.all_trained = n_comp - 1, False
    nc = model.num_components if model.all_trained else model.component + 1
    for p in model.parameters():
        p.grad = None
        p.requires_grad_(True)
    z = torch.randn(n, model.z_size, device="cuda", generator=_gen(seed)).requires_grad_(True)
    u = torch.rand(n, dtype=torch.float64, device="cuda", generator=_gen(seed + 1))
    x, ldj, comp = model.rsample(n, u=u, z=z)
    assert (type(x.grad_fn).__name__ == "_FusedMixtureInverseBackward") == expect_fused, type(x.grad_fn).__name__
    if expect_fused:
        xm, lm = model.mixture_inverse(z.detach(), comp, nc)
        assert torch.equal(x.detach(), xm) and torch.equal(ldj.detach(), lm)
    dx, dldj = _upstream(n, model.z_size, seed + 2)
    ((x * dx).sum() + (ldj * dldj).sum()).backward()
    ref, ref_dz = _reference(model, z, comp, dx, dldj, nc)
    _close(z.grad, ref_dz, "z.grad")
    for c in range(nc):
        for i, (p, r) in enumerate(zip(model.flows[c].parameters(), ref[c])):
            _close(p.grad if p.grad is not None else torch.zeros_like(p), r, ("param", c, i))


@pytest.mark.parametrize("mode", ["fp32", "f16fast"])
@pytest.mark.parametrize("kind", ["glow", "realnvp"])
def test_rsample_fused(kind, mode):
    model = _model(kind, 13, 128, 3, C=4, mode=mode)
    try:
        model.all_trained = True
        _check_public(model, 500, seed=100)
        model.check_status()
    finally:
        model.release()


FALLBACK = {   # (kind, D, h, K, extra model args, mode)
    "realnvp_batch_norm": ("realnvp", 7, 64, 3, dict(batch_norm=True), "fp32"),
    "realnvp_residual": ("realnvp", 7, 64, 2, dict(act="residual"), "fp32"),
    "glow_invconv": ("glow", 6, 64, 2, dict(invconv=True), "fp32"),
    "glow_h1024_pair": ("glow", 12, 1024, 2, {}, "f16fast"),
    "glow_fused_backward_off": ("glow", 13, 128, 3, dict(fused_backward=False), "f16fast"),
}


@pytest.mark.parametrize("name", list(FALLBACK))
def test_rsample_fallback(name):
    kind, D, h, K, kw, mode = FALLBACK[name]
    model = _model(kind, D, h, K, C=3, mode=mode, **kw)
    try:
        model.all_trained = True
        _check_public(model, 200, seed=110, expect_fused=False)
    finally:
        model.release()


def test_two_rsamples_then_backward_on_the_first():
    """The backward redoes the sort from the saved ids: another draw in between does not disturb it."""
    model = _model("glow", 13, 128, 3, C=4, mode="f16fast")
    try:
        model.all_trained = True
        for p in model.parameters():
            p.requires_grad_(True)
        z = torch.randn(400, 13, device="cuda", generator=_gen(120)).requires_grad_(True)
        u = torch.rand(400, dtype=torch.float64, device="cuda", generator=_gen(121))
        x, ldj, comp = model.rsample(400, u=u, z=z)
        model.rsample(900, generator=_gen(122))
        dx, dldj = _upstream(400, 13, 123)
        ((x * dx).sum() + (ldj * dldj).sum()).backward()
        ref, ref_dz = _reference(model, z, comp, dx, dldj, 4)
        _close(z.grad, ref_dz, "z.grad")
        for c in range(4):
            for i, (p, r) in enumerate(zip(model.flows[c].parameters(), ref[c])):
                _close(p.grad, r, ("param", c, i))
    finally:
        model.release()


def test_sample_keeps_its_no_grad_contract():
    model = _model("glow", 13, 128, 3, C=4, mode="f16fast")
    try:
        model.all_trained = True
        for p in model.parameters():
            p.requires_grad_(True)
        x, comp = model.sample(100, generator=_gen(130))
        assert not x.requires_grad
        xr, ldjr, compr = model.rsample(100, generator=_gen(130))
        assert xr.requires_grad and torch.equal(compr, comp) and torch.equal(xr.detach(), x)
    finally:
        model.release()


def test_reverse_kl_training_loop():
    """Fit the newest component by reverse KL to a diagonal Gaussian with an analytic log p: 30 Adam steps through rsample and
    the fused inverse backward lower KL(q || p) = E_q[log q(x) - log p(x)] by at least 20 % (mean of the last five steps against
    the first five)."""
    D = 6
    model = _model("glow", D, 128, 3, C=2, mode="f16fast", seed=7)
    fused = []
    apply = bf._FusedMixtureInverse.apply
    bf._FusedMixtureInverse.apply = lambda *a: fused.append(1) or apply(*a)
    try:
        model.component, model.all_trained = 0, False
        params = list(model.flows[0].parameters())
        opt = torch.optim.Adam(params, lr=1e-2)
        mu = torch.linspace(-2, 2, D, device="cuda")
        sd = torch.linspace(0.5, 2.0, D, device="cuda")
        gen = _gen(140)
        losses = []
        for _ in range(30):
            opt.zero_grad()
            z = torch.randn(512, D, device="cuda", generator=gen)
            x, ldj, _ = model.rsample(512, z=z, comp=torch.zeros(512, dtype=torch.int64, device="cuda"))
            log_q = -0.5 * (z ** 2).sum(1) - 0.5 * D * math.log(2 * math.pi) - ldj
            log_p = (-0.5 * ((x - mu) / sd) ** 2 - torch.log(sd) - 0.5 * math.log(2 * math.pi)).sum(1)
            loss = (log_q - log_p).mean()
            loss.backward()
            opt.step()
            losses.append(float(loss))
        assert len(fused) == 30
        assert all(math.isfinite(v) for v in losses)
        assert np.mean(losses[-5:]) < 0.8 * np.mean(losses[:5]), losses
        model.check_status()
    finally:
        bf._FusedMixtureInverse.apply = apply
        model.release()
