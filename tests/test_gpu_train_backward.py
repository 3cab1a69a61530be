"""The fused training backward (gbnf_component_backward, csrc/train_bwd.cuh) against torch autograd in fp64 (-m gpu).

The reference differentiates the host mirror's forward (forward_autograd, pinned to the reference's outputs by
tests/test_host_modules.py) in float64 on the GPU with torch.autograd.grad((z, ldj), params + [x], (dz, dldj)).  Upstream
gradients are random per row and unrelated to z, so a kernel that reads dL/dldj or dL/dz from the wrong row cannot pass.

The backward recomputes and differentiates in fp32 CUDA-core arithmetic whatever the handle's GEMM mode (it packs its own
fp32 weight copies), so every mode is held to max|g - g_ref| <= 1e-4 max|g_ref| + 1e-7 per tensor.  Shapes cover both
phases' tile edges (phase A: 16-row tiles; phase B: 64 x 64 output tiles, 32-row chunks), odd D (|z1| != |z2|, RealNVP's
flipped steps both ways through the parity of c), the zero padding of h = 100 / 200 and the deepest component the
shared-memory history holds.  D = 1 is not a shape of this library: gbnf_create refuses D < 2, because Glow's split of a
1-D input leaves its coupling network no input (|z1| = D // 2 = 0).
"""
import copy
import ctypes

import numpy as np
import pytest
import torch

from gbnf_b200 import _lib
from gbnf_b200 import boosted_flow as bf
from helpers import build_model
from oracle import gbnf_oracle as orc

pytestmark = pytest.mark.gpu

TOL = 1e-4


def _model(kind, D, h, K, coupling="affine", act="tanh", mode="fp32", seed=5):
    md = orc.make_synthetic_model(kind, D, 2, K, h, seed=seed, act=act, coupling=coupling, init_rows=512)
    return build_model(md, "cuda", gemm_mode=mode)


def _rows(B, D, seed):
    return torch.randn(B, D, device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed))


def _upstream(B, D, seed, which="both"):
    """dL/dz ~ N(0, 1) / B and dL/dldj ~ U(-1, 1) / B, drawn per row; `which` keeps one of them ("dz" / "dldj")."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    dz = torch.randn(B, D, device="cuda", generator=g) / B
    dldj = (torch.rand(B, device="cuda", generator=g) * 2 - 1) / B
    if which == "dz":
        dldj.zero_()
    elif which == "dldj":
        dz.zero_()
    return dz, dldj


def _reference(model, c, x, dz, dldj):
    """fp64 autograd gradients of component c's parameters (module order) and of x for upstream (dz, dldj)."""
    flow = copy.deepcopy(model.flows[c]).to(torch.float64)
    if model.component_type == "glow":
        for s_src, s_dst in zip(model.flows[c].steps(), flow.steps()):
            s_dst.permutation.set_indices(s_src.permutation.indices)
            s_dst.actnorm.inited = True
    params = list(flow.parameters())
    for p in params:
        p.requires_grad_(True)
    x64 = x.detach().double().requires_grad_(True)
    z, ldj = flow.forward_autograd(x64)
    g = torch.autograd.grad((z, ldj), params + [x64], grad_outputs=(dz.double(), dldj.double()))
    return list(g[:-1]), g[-1]


def _close(got, ref, what, tol=TOL):
    """max|got - ref| <= tol max|ref| + 1e-7; returns the error relative to max|ref|."""
    assert got is not None, what
    assert tuple(got.shape) == tuple(ref.shape), (what, tuple(got.shape), tuple(ref.shape))
    scale = float(ref.abs().max())
    err = float((got.double() - ref).abs().max())
    assert err <= tol * scale + 1e-7, (what, err, scale)
    return err / max(scale, 1e-30)


def _check_abi(model, c, x, dz, dldj, tol=TOL):
    """model._component_backward (the ABI call, dL/dx requested) against the fp64 reference."""
    ref, ref_dx = _reference(model, c, x, dz, dldj)
    grads, dx = model._component_backward(c, x, dz, dldj, with_dx=True)
    errs = [_close(grads[id(p)], r, ("param", i), tol) for i, (p, r) in enumerate(zip(model.flows[c].parameters(), ref))]
    errs.append(_close(dx, ref_dx, "dx", tol))
    return max(errs)


def _public_loss(z, ldj, dz, dldj, which):
    # a loss whose upstream gradients are exactly (dz, dldj); "dz" / "dldj" leave the other output out of the graph
    if which == "dz":
        return (z * dz).sum()
    if which == "dldj":
        return (ldj * dldj).sum()
    return (z * dz).sum() + (ldj * dldj).sum()


def _check_public(model, c, x, dz, dldj, which="both", expect_fused=True, tol=TOL):
    """model(x=x, components="c") + backward(), x requiring grad, against the fp64 reference."""
    ref, ref_dx = _reference(model, c, x, dz, dldj)
    model.component = c
    for p in model.parameters():
        p.grad = None
    xg = x.clone().requires_grad_(True)
    z, _, _, ldj, _ = model(x=xg, components="c")
    assert type(z.grad_fn).__name__.startswith("_FusedComponentFlow") == expect_fused
    _public_loss(z, ldj, dz, dldj, which).backward()
    for i, (p, r) in enumerate(zip(model.flows[c].parameters(), ref)):
        _close(p.grad, r, ("param", i), tol)
    _close(xg.grad, ref_dx, "x.grad", tol)


def _abi_backward(model, c, x, dz, dldj, fill):
    """gbnf_component_backward straight through ctypes into gradient buffers (and dL/dx) the test owns, pre-filled with
    `fill`.  Returns the status code and the buffers after a device synchronise."""
    dev = x.device
    steps = model._component_tensors(c)
    parr, garr = (_lib.StepParams * len(steps))(), (_lib.StepGrads * len(steps))()
    keep, bufs = [], []

    def dv(t, dtype=torch.float32):
        t = t.detach().to(device=dev, dtype=dtype).contiguous()
        keep.append(t)
        return t.data_ptr()

    def gb(p):
        g = torch.full(tuple(p.shape), fill, device=dev)
        bufs.append(g)
        return g.data_ptr()

    for k, (d, step) in enumerate(zip(steps, model.flows[c].steps())):
        sp, sg = parr[k], garr[k]
        if "an_bias" in d:
            sp.an_bias, sp.an_logs, sp.perm = dv(d["an_bias"].reshape(-1)), dv(d["an_logs"].reshape(-1)), dv(d["perm"], torch.int64)
            sg.an_bias, sg.an_logs = gb(step.actnorm.bias), gb(step.actnorm.logs)
        for n, lins in enumerate(d["nets"]):
            for l, lin in enumerate(lins):
                sp.W[n][l], sp.b[n][l] = dv(lin.weight), dv(lin.bias)
                sg.W[n][l], sg.b[n][l] = gb(lin.weight), gb(lin.bias)
    cp = _lib.ComponentParams()
    cp.flip_init, cp.n_steps = getattr(model.flows[c], "flip_init", 0), len(steps)
    cp.steps = ctypes.cast(parr, ctypes.POINTER(_lib.StepParams))
    dx = torch.full_like(x, fill)
    bufs.append(dx)
    rc = _lib.load().gbnf_component_backward(model.handle(dev), c, ctypes.byref(cp), ctypes.c_void_p(x.data_ptr()), x.shape[0],
                                             ctypes.c_void_p(dz.data_ptr()), ctypes.c_void_p(dldj.data_ptr()),
                                             ctypes.cast(garr, ctypes.POINTER(_lib.StepGrads)), ctypes.c_void_p(dx.data_ptr()),
                                             ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    torch.cuda.synchronize()
    return rc, bufs


# (kind, coupling, act, D, h, K)
KINDS = {
    "glow_affine_tanh": ("glow", "affine", "tanh", 7, 64, 3),
    "glow_affine_relu": ("glow", "affine", "relu", 7, 128, 3),
    "glow_additive_relu": ("glow", "additive", "relu", 7, 64, 3),
    "realnvp_tanh": ("realnvp", "affine", "tanh", 7, 64, 3),
    "realnvp_relu": ("realnvp", "affine", "relu", 7, 128, 3),
    "realnvp_mixed": ("realnvp", "affine", "mixed", 7, 64, 3),
}
SHAPES = {}
for _D in (2, 3, 31, 32, 33, 63, 64):            # odd D: |z1| != |z2|; Glow affine at 63 / 64 fills the 64-wide output rows
    SHAPES[f"glow_affine_tanh_d{_D}"] = ("glow", "affine", "tanh", _D, 64, 2)
    SHAPES[f"realnvp_tanh_d{_D}"] = ("realnvp", "affine", "tanh", _D, 64, 2)
SHAPES["glow_additive_relu_d63"] = ("glow", "additive", "relu", 63, 64, 2)
for _h in (100, 200, 384, 512):                  # 100 / 200: the zero padding to 128 / 256 (fp32 handles: the f16 modes need h % 64 == 0)
    SHAPES[f"glow_affine_relu_d33_h{_h}"] = ("glow", "affine", "relu", 33, _h, 2)
    SHAPES[f"realnvp_mixed_d33_h{_h}"] = ("realnvp", "affine", "mixed", 33, _h, 2)
SHAPES["glow_affine_tanh_k1"] = ("glow", "affine", "tanh", 5, 64, 1)
SHAPES["realnvp_relu_k1"] = ("realnvp", "affine", "relu", 5, 64, 1)


@pytest.mark.parametrize("mode", ["fp32", "f16", "f16fast"])
@pytest.mark.parametrize("name", list(KINDS))
def test_kinds_and_couplings_match_fp64(name, mode):
    kind, coupling, act, D, h, K = KINDS[name]
    model = _model(kind, D, h, K, coupling, act, mode)
    try:
        for c in (0, 1):
            x = _rows(300, D, 10 + c)
            dz, dldj = _upstream(300, D, 20 + c)
            _check_abi(model, c, x, dz, dldj)
            _check_public(model, c, x, dz, dldj)
        model.check_status()
    finally:
        model.release()


@pytest.mark.parametrize("which", ["dz", "dldj"])
@pytest.mark.parametrize("name", list(KINDS))
def test_one_upstream_gradient_zero(name, which):
    """dz = 0 alone and dldj = 0 alone; on the public path the loss leaves the other output out, so the autograd Function
    receives zeros for it."""
    kind, coupling, act, D, h, K = KINDS[name]
    model = _model(kind, D, h, K, coupling, act, "f16fast")
    try:
        c = 1
        x = _rows(77, D, 3)
        dz, dldj = _upstream(77, D, 4, which)
        _check_abi(model, c, x, dz, dldj)
        _check_public(model, c, x, dz, dldj, which)
    finally:
        model.release()


@pytest.mark.parametrize("name", list(SHAPES))
def test_widths_depths_and_padding_match_fp64(name):
    kind, coupling, act, D, h, K = SHAPES[name]
    model = _model(kind, D, h, K, coupling, act, "fp32" if h % 64 else "f16fast")
    try:
        for c in (0, 1):
            x = _rows(300, D, 30 + c)
            dz, dldj = _upstream(300, D, 40 + c)
            _check_abi(model, c, x, dz, dldj)
            _check_public(model, c, x, dz, dldj)
    finally:
        model.release()


@pytest.mark.parametrize("B", [1, 15, 16, 17, 31, 33, 300, 512])
@pytest.mark.parametrize("name", ["realnvp_mixed_d5_h64", "glow_affine_d63_h100"])
def test_batch_sizes_around_the_tiles(name, B):
    """Phase A's 16-row tiles and phase B's 32-row chunks: a partial last tile, exactly one tile, one row."""
    kind, coupling, act, D, h, K = {"realnvp_mixed_d5_h64": ("realnvp", "affine", "mixed", 5, 64, 3),
                                    "glow_affine_d63_h100": ("glow", "affine", "tanh", 63, 100, 2)}[name]
    model = _model(kind, D, h, K, coupling, act, "fp32")
    try:
        for c in (0, 1):
            x = _rows(B, D, 50 + c)
            dz, dldj = _upstream(B, D, 60 + c)
            _check_abi(model, c, x, dz, dldj)
            _check_public(model, c, x, dz, dldj)
    finally:
        model.release()


def test_large_batch_cfg4_shape():
    """B = 65 536 at cfg4's component shape (Glow D = 21, h = 512, K = 10): phase B sums every row of the batch sequentially in
    fp32.  Measured on an NVIDIA B200 (1000 W power limit): the worst error of any gradient tensor, dL/dx included, was
    1.26e-5 of its max |g_ref|, so the tolerance of every other case holds here too."""
    B, D = 65536, 21
    model = _model("glow", D, 512, 10, mode="f16fast")
    try:
        x = _rows(B, D, 70)
        dz, dldj = _upstream(B, D, 71)
        err = _check_abi(model, 1, x, dz, dldj, tol=TOL)
        print(f"large batch: worst relative gradient error {err:.3e}")
    finally:
        model.release()


def test_deterministic_and_independent_of_the_gemm_mode():
    """Weight / bias gradients and dL/dx are bitwise equal across calls and across fp32 / f16 / f16fast handles (no atomics;
    the backward never reads the handle's fp16 weights); the ActNorm gradients (atomics) agree to 1e-6."""
    runs = []
    x = _rows(1000, 33, 80)
    dz, dldj = _upstream(1000, 33, 81)
    for mode in ("fp32", "f16", "f16fast"):
        model = _model("glow", 33, 128, 3, mode=mode)
        try:
            params = list(model.flows[1].parameters())
            actnorm = [i for i, (n, _) in enumerate(model.flows[1].named_parameters()) if "actnorm" in n]
            for _ in range(2):
                grads, dx = model._component_backward(1, x, dz, dldj, with_dx=True)
                runs.append([grads[id(p)] for p in params] + [dx])
        finally:
            model.release()
    assert actnorm
    for other in runs[1:]:
        for i, (a, b) in enumerate(zip(runs[0], other)):
            if i in actnorm:
                assert float((a - b).abs().max()) <= 1e-6 * float(a.abs().max()), i
            else:
                assert torch.equal(a, b), i


def test_rows_are_independent():
    """dL/dx of a row slice is bitwise the same rows of the full batch's dL/dx; the parameter gradients of the full batch are
    the sum of two disjoint halves (within fp32 rounding)."""
    model = _model("realnvp", 9, 200, 3, act="mixed")
    try:
        B = 300
        x = _rows(B, 9, 90)
        dz, dldj = _upstream(B, 9, 91)
        params = list(model.flows[1].parameters())
        full, dx = model._component_backward(1, x, dz, dldj, with_dx=True)
        full = [full[id(p)].clone() for p in params]
        dx = dx.clone()
        _, dx_slice = model._component_backward(1, x[17:].contiguous(), dz[17:].contiguous(), dldj[17:].contiguous(), with_dx=True)
        assert torch.equal(dx_slice, dx[17:])
        halves = []
        for sl in (slice(0, 150), slice(150, B)):
            g, _ = model._component_backward(1, x[sl].contiguous(), dz[sl].contiguous(), dldj[sl].contiguous())
            halves.append([g[id(p)].clone() for p in params])
        for i, (f, a, b) in enumerate(zip(full, *halves)):
            _close(f, (a.double() + b.double()), ("param", i))
    finally:
        model.release()


def test_scratch_reuse_across_batches_and_components():
    """One handle: large B, small B, large B, a larger B, alternating the component (and with it which RealNVP steps are
    flipped at odd D); every call matches the reference, so a regrown or reused scratch never serves stale rows."""
    model = _model("realnvp", 5, 200, 3, act="mixed")
    try:
        for i, (B, c) in enumerate([(2000, 1), (37, 0), (2000, 1), (4100, 0), (1, 1)]):
            x = _rows(B, 5, 100 + i)
            dz, dldj = _upstream(B, 5, 110 + i)
            _check_abi(model, c, x, dz, dldj)
    finally:
        model.release()


def test_partial_freezing_and_accumulation():
    """Frozen parameters get no gradient; two backward() calls without zero_grad accumulate to twice the reference."""
    model = _model("glow", 11, 64, 3, mode="f16fast")
    try:
        c = 1
        model.component = c
        params = list(model.flows[c].parameters())
        for i, p in enumerate(params):
            p.requires_grad_(i % 3 != 1)
        x = _rows(200, 11, 120)
        dz, dldj = _upstream(200, 11, 121)
        ref, _ = _reference(model, c, x, dz, dldj)
        for _ in range(2):
            z, _, _, ldj, _ = model(x=x, components="c")
            assert type(z.grad_fn).__name__.startswith("_FusedComponentFlow")
            _public_loss(z, ldj, dz, dldj, "both").backward()
        for i, (p, r) in enumerate(zip(params, ref)):
            if i % 3 == 1:
                assert p.grad is None, i
            else:
                _close(p.grad, 2 * r, ("param", i))
    finally:
        model.release()


@pytest.mark.parametrize("kind", ["glow", "realnvp"])
def test_dx_through_the_abi_and_the_public_path(kind):
    """dL/dx through d_dx_opt, and x.grad on the public path (x.requires_grad_(True)) with the component's parameters
    trainable and with all of them frozen."""
    model = _model(kind, 13, 128, 3, mode="f16fast")
    try:
        c = 1
        x = _rows(150, 13, 130)
        dz, dldj = _upstream(150, 13, 131)
        _check_abi(model, c, x, dz, dldj)
        _check_public(model, c, x, dz, dldj)
        _, ref_dx = _reference(model, c, x, dz, dldj)
        for p in model.flows[c].parameters():
            p.requires_grad_(False)
            p.grad = None
        xg = x.clone().requires_grad_(True)
        z, _, _, ldj, _ = model(x=xg, components="c")
        assert type(z.grad_fn).__name__.startswith("_FusedComponentFlow")
        _public_loss(z, ldj, dz, dldj, "both").backward()
        _close(xg.grad, ref_dx, "x.grad, parameters frozen")
        assert all(p.grad is None for p in model.flows[c].parameters())
    finally:
        model.release()


# (kind, coupling, act, D, h, K, served by the fused backward): both sides of the shared-memory bound
ENVELOPE = [
    ("glow", "affine", "tanh", 43, 512, 10, True),    # cfg3's width at cfg4's depth (refused mid-backward before oh shrank)
    ("glow", "affine", "tanh", 21, 512, 10, True),    # cfg4
    ("glow", "affine", "tanh", 43, 512, 15, True),
    ("glow", "affine", "tanh", 43, 512, 16, False),
    ("glow", "additive", "relu", 64, 512, 12, True),
    ("glow", "additive", "relu", 64, 512, 13, False),
    ("glow", "affine", "relu", 2, 64, 47, True),
    ("glow", "affine", "relu", 2, 64, 48, False),
    ("realnvp", "affine", "tanh", 43, 512, 9, True),
    ("realnvp", "affine", "tanh", 43, 512, 10, False),
    ("realnvp", "affine", "mixed", 2, 64, 24, True),
    ("realnvp", "affine", "mixed", 2, 64, 25, False),
    ("realnvp", "affine", "relu", 63, 200, 12, True),  # h = 200: 256-wide activation rows leave room for more steps
    ("realnvp", "affine", "relu", 63, 200, 13, False),
]


@pytest.mark.parametrize("case", ENVELOPE, ids=lambda t: "_".join(map(str, t)))
def test_envelope_agrees_with_the_library(case):
    """Where BoostedFlow routes a component to the fused backward, the library serves it and matches the reference; where it
    does not, training runs through autograd and the library refuses the shape before writing anything.  No GbnfError ever
    leaves backward()."""
    kind, coupling, act, D, h, K, served = case
    model = _model(kind, D, h, K, coupling, act, "fp32" if h % 64 else "f16fast")
    try:
        c, B = 1, 40
        x = _rows(B, D, 140)
        dz, dldj = _upstream(B, D, 141)
        assert model._fused_backward_ok(x) == served
        _check_public(model, c, x, dz, dldj, expect_fused=served)
        if served:
            _check_abi(model, c, x, dz, dldj)
        else:
            rc, bufs = _abi_backward(model, c, x, dz, dldj, fill=7.0)
            assert rc == -1, rc                               # GBNF_ERR_INVALID
            assert "shared-memory" in _lib.load().gbnf_last_error().decode()
            assert all(bool((b == 7.0).all()) for b in bufs)  # nothing written, ActNorm gradients not zeroed
        model.check_status()
    finally:
        model.release()


@pytest.mark.parametrize("group", [("glow", 43, 512), ("glow", 2, 64), ("realnvp", 21, 384), ("realnvp", 64, 100)],
                         ids=lambda t: "_".join(map(str, t)))
def test_deepest_component_the_library_serves(group):
    """fused_backward_smem_bytes is the library's own count: the largest K it admits runs and matches the reference, K + 1 is
    refused with every caller buffer untouched."""
    kind, D, h = group
    K = 1
    while bf.fused_backward_smem_bytes(kind, D, h, K + 1) <= bf.FUSED_BACKWARD_MAX_SMEM:
        K += 1
    for k, served in ((K, True), (K + 1, False)):
        model = _model(kind, D, h, k, mode="fp32")
        try:
            x = _rows(33, D, 150)
            dz, dldj = _upstream(33, D, 151)
            assert model._fused_backward_ok(x) == served
            rc, bufs = _abi_backward(model, 1, x, dz, dldj, fill=-3.0)
            if served:
                assert rc == 0, _lib.load().gbnf_last_error()
                ref, ref_dx = _reference(model, 1, x, dz, dldj)
                for i, (g, r) in enumerate(zip(bufs, ref + [ref_dx])):
                    _close(g, r.reshape(g.shape), ("buffer", i))
            else:
                assert rc == -1 and all(bool((b == -3.0).all()) for b in bufs)
        finally:
            model.release()


def test_one_dimensional_data_is_refused_at_create():
    """D = 1 has no fused backward to test: gbnf_create refuses it (see the module docstring)."""
    cfg = _lib.Config()
    cfg.kind, cfg.D, cfg.h, cfg.K, cfg.C, cfg.depth = _lib.KIND["glow"], 1, 64, 1, 1, 1
    cfg.act, cfg.coupling, cfg.base, cfg.gemm_mode, cfg.device = _lib.ACT["tanh"], 0, 0, _lib.GEMM["fp32"], 0
    h = ctypes.c_void_p()
    assert _lib.load().gbnf_create(ctypes.byref(h), ctypes.byref(cfg)) == -1 and not h.value
