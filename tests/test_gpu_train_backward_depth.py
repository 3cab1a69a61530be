"""The fused training backward (gbnf_component_backward) at every coupling-network depth other than 1 (-m gpu), against torch
autograd in fp64.

tests/test_gpu_train_backward.py covers depth 1; this file runs the same rule at depth 0 (Linear(in, h), activation,
Linear(h, out): no hidden-to-hidden layer) and at depths 2, 3 and 4 (depth x Linear(h, h) between them): every gradient
tensor, dL/dx included, within max|g - g_ref| <= 1e-4 max|g_ref| + 1e-7 of fp64 autograd through forward_autograd.  The
backward computes in fp32 whatever the handle's GEMM mode, so fp32, f16 and f16fast handles are all held to that bound.  The
shared-memory history does not grow with the depth (the hidden layers ping-pong between two activation rows), so the
deepest component served at each depth is the one fused_backward_smem_bytes admits at depth 1.

Measured on an NVIDIA B200 (1000 W power limit), the worst error of any gradient tensor relative to its max |g_ref|, over
every served case of this file: 2.9e-6 at depth 0, 1.5e-5 at depth 2, 3.2e-6 at depth 3, 2.7e-6 at depth 4 (printed at the end
of the module's run).
"""
import argparse
import ctypes
import math

import pytest
import torch

import gbnf_b200
from gbnf_b200 import _lib
from gbnf_b200 import boosted_flow as bf
from helpers import build_model
from oracle import gbnf_oracle as orc
from tests.test_gpu_train_backward import _close, _reference, _upstream

pytestmark = pytest.mark.gpu

TOL = 1e-4
DEPTHS = [0, 2, 3, 4]
WORST = {}        # depth -> worst relative gradient error of the served cases run so far


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    yield
    for d in sorted(WORST):
        print(f"depth {d}: worst relative gradient error {WORST[d]:.3e}")


def _model(kind, D, h, K, depth, coupling="affine", act="tanh", mode="fp32", seed=5, **kw):
    md = orc.make_synthetic_model(kind, D, 2, K, h, seed=seed, depth=depth, act=act, coupling=coupling, init_rows=512, **kw)
    return build_model(md, "cuda", gemm_mode=mode)


def _rows(B, D, seed):
    return torch.randn(B, D, device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed))


def _note(model, err):
    d = model.args.coupling_network_depth
    WORST[d] = max(WORST.get(d, 0.0), err)


def _check_abi(model, c, x, dz, dldj):
    """model._component_backward (the ABI call, dL/dx requested) against the fp64 reference."""
    ref, ref_dx = _reference(model, c, x, dz, dldj)
    grads, dx = model._component_backward(c, x, dz, dldj, with_dx=True)
    errs = [_close(grads[id(p)], r, ("param", i), TOL) for i, (p, r) in enumerate(zip(model.flows[c].parameters(), ref))]
    errs.append(_close(dx, ref_dx, "dx", TOL))
    _note(model, max(errs))


def _check_public(model, c, x, dz, dldj, expect_fused=True):
    """model(x=x, components="c") + backward() with x requiring grad, against the fp64 reference; the component is trained
    through _FusedComponentFlow exactly when expect_fused."""
    ref, ref_dx = _reference(model, c, x, dz, dldj)
    model.component = c
    for p in model.parameters():
        p.grad = None
    xg = x.clone().requires_grad_(True)
    z, _, _, ldj, _ = model(x=xg, components="c")
    assert type(z.grad_fn).__name__.startswith("_FusedComponentFlow") == expect_fused
    ((z * dz).sum() + (ldj * dldj).sum()).backward()
    errs = [_close(p.grad, r, ("param", i), TOL) for i, (p, r) in enumerate(zip(model.flows[c].parameters(), ref))]
    errs.append(_close(xg.grad, ref_dx, "x.grad", TOL))
    if expect_fused:
        _note(model, max(errs))


def _abi_call(model, c, x, dz, dldj, fill):
    """gbnf_component_backward through ctypes into gradient buffers (and dL/dx) the test owns, pre-filled with `fill`, passing
    every tensor the component has (BatchNorm included, so that the library sees it).  Returns the status code, the error
    text and the buffers after a device synchronise."""
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
        if "bn" in d:
            sp.bn_log_gamma, sp.bn_beta, sp.bn_mean, sp.bn_var = [dv(t) for t in d["bn"]]
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
    return rc, _lib.load().gbnf_last_error().decode(), bufs


# (kind, coupling, act, D, h, K): both Glow couplings, RealNVP with every activation; odd D, so that RealNVP's flipped steps
# have |z1| != |z2| and components 0 and 1 see both parities
KINDS = {
    "glow_affine_tanh": ("glow", "affine", "tanh", 7, 64, 3),
    "glow_additive_relu": ("glow", "additive", "relu", 7, 64, 3),
    "realnvp_tanh": ("realnvp", "affine", "tanh", 7, 64, 3),
    "realnvp_relu": ("realnvp", "affine", "relu", 7, 128, 3),
    "realnvp_mixed": ("realnvp", "affine", "mixed", 7, 64, 3),
}


@pytest.mark.parametrize("mode", ["fp32", "f16", "f16fast"])
@pytest.mark.parametrize("depth", DEPTHS)
@pytest.mark.parametrize("name", list(KINDS))
def test_kinds_at_every_depth(name, depth, mode):
    kind, coupling, act, D, h, K = KINDS[name]
    model = _model(kind, D, h, K, depth, coupling, act, mode)
    try:
        for c in (0, 1):
            x = _rows(300, D, 10 + c)
            dz, dldj = _upstream(300, D, 20 + c)
            _check_abi(model, c, x, dz, dldj)
            _check_public(model, c, x, dz, dldj)
        model.check_status()
    finally:
        model.release()


@pytest.mark.parametrize("depth", [2, 3])
@pytest.mark.parametrize("h", [64, 100, 300, 448, 512])
@pytest.mark.parametrize("kind", ["glow", "realnvp"])
def test_hidden_widths(kind, h, depth):
    """h = 100 / 300: the zero padding of every hidden layer to 128 / 320 (fp32 handles: the f16 modes need h % 64 == 0).
    RealNVP runs tanh networks here.  With ReLU, one of the 2 x 4 x 448 x 300 ReLU inputs of realnvp mixed at h = 448, depth 3
    lies 2.7e-8 from zero: the fp32 kernel and the fp64 reference take different branches there, and that row's share of the
    first layer's weight gradient (3.5e-3 of its max) differs entirely.  Flipping that one ReLU in the reference brings every
    gradient within 1.1e-6, so the miss is the kink, not the backward; the mixed networks are covered by the other tests."""
    act = "relu" if kind == "glow" else "tanh"
    model = _model(kind, 33, h, 2, depth, act=act, mode="fp32" if h % 64 else "f16fast")
    try:
        for c in (0, 1):
            x = _rows(300, 33, 30 + c)
            dz, dldj = _upstream(300, 33, 40 + c)
            _check_abi(model, c, x, dz, dldj)
            _check_public(model, c, x, dz, dldj)
    finally:
        model.release()


@pytest.mark.parametrize("depth", [2, 3])
@pytest.mark.parametrize("D", [2, 3, 33, 63, 64])
@pytest.mark.parametrize("kind", ["glow", "realnvp"])
def test_feature_counts(kind, D, depth):
    """D = 2 / 3: one-column networks inputs; 63 / 64: Glow affine fills the 64-wide output rows."""
    model = _model(kind, D, 64, 2, depth, mode="f16fast")
    try:
        for c in (0, 1):
            x = _rows(300, D, 50 + c)
            dz, dldj = _upstream(300, D, 60 + c)
            _check_abi(model, c, x, dz, dldj)
            _check_public(model, c, x, dz, dldj)
    finally:
        model.release()


@pytest.mark.parametrize("B", [1, 15, 16, 17, 33, 300])
@pytest.mark.parametrize("depth", [0, 4])
@pytest.mark.parametrize("name", ["realnvp_mixed_d5_h64", "glow_affine_d63_h100"])
def test_batch_sizes_around_the_tiles(name, depth, B):
    """Phase A's 16-row tiles and phase B's 32-row chunks at the shallowest and the deepest network."""
    kind, act, D, h, K = {"realnvp_mixed_d5_h64": ("realnvp", "mixed", 5, 64, 3),
                          "glow_affine_d63_h100": ("glow", "tanh", 63, 100, 2)}[name]
    model = _model(kind, D, h, K, depth, act=act)
    try:
        for c in (0, 1):
            x = _rows(B, D, 70 + c)
            dz, dldj = _upstream(B, D, 80 + c)
            _check_abi(model, c, x, dz, dldj)
            _check_public(model, c, x, dz, dldj)
    finally:
        model.release()


def test_large_batch_cfg4_shape_at_depth_2():
    """B = 65 536 at cfg4's component shape (Glow D = 21, h = 512, K = 10) with two hidden-to-hidden layers: phase B sums every
    row of the batch sequentially in fp32, and the scratch holds 3 hidden activations and 4 d pre-activations per step."""
    B, D = 65536, 21
    model = _model("glow", D, 512, 10, 2, mode="f16fast")
    try:
        x = _rows(B, D, 90)
        dz, dldj = _upstream(B, D, 91)
        _check_abi(model, 1, x, dz, dldj)
    finally:
        model.release()


@pytest.mark.parametrize("depth", [0, 2, 4])
@pytest.mark.parametrize("group", [("glow", 43, 512), ("glow", 2, 64), ("realnvp", 21, 384), ("realnvp", 64, 100)],
                         ids=lambda t: "_".join(map(str, t)))
def test_deepest_component_at_every_depth(group, depth):
    """The largest K fused_backward_smem_bytes admits is served at every depth and matches the reference; K + 1 trains through
    autograd on the public path (no GbnfError reaches backward()) and the library refuses it with every caller buffer
    untouched."""
    kind, D, h = group
    K = 1
    while bf.fused_backward_smem_bytes(kind, D, h, K + 1) <= bf.FUSED_BACKWARD_MAX_SMEM:
        K += 1
    for k, served in ((K, True), (K + 1, False)):
        model = _model(kind, D, h, k, depth)
        try:
            c = 1
            x = _rows(33, D, 100)
            dz, dldj = _upstream(33, D, 101)
            assert model._fused_backward_ok(x) == served
            _check_public(model, c, x, dz, dldj, expect_fused=served)
            if served:
                _check_abi(model, c, x, dz, dldj)
            else:
                rc, err, bufs = _abi_call(model, c, x, dz, dldj, fill=-3.0)
                assert rc == -1 and "shared-memory" in err, (rc, err)
                assert all(bool((b == -3.0).all()) for b in bufs)
            model.check_status()
        finally:
            model.release()


# configurations the fused backward does not serve at any depth: (kind, D, h, K, depth, extra model args)
REFUSED = {
    "realnvp_batch_norm_depth0": ("realnvp", 6, 64, 3, 0, dict(batch_norm=True)),
    "realnvp_batch_norm_depth2": ("realnvp", 6, 64, 3, 2, dict(batch_norm=True)),
    "realnvp_residual_depth2": ("realnvp", 6, 64, 2, 2, dict(act="residual")),
    "glow_h640_depth2": ("glow", 21, 640, 2, 2, {}),
}


@pytest.mark.parametrize("name", list(REFUSED))
def test_still_refused_at_other_depths(name):
    """RealNVP with BatchNorm, ResidualNet and h > 512 train through autograd at every depth, and the library refuses them
    before it writes anything."""
    kind, D, h, K, depth, kw = REFUSED[name]
    model = _model(kind, D, h, K, depth, **kw)
    try:
        c = 1
        x = _rows(40, D, 110)
        dz, dldj = _upstream(40, D, 111)
        assert not model._fused_backward_ok(x)
        _check_public(model, c, x, dz, dldj, expect_fused=False)
        rc, err, bufs = _abi_call(model, c, x, dz, dldj, fill=7.0)
        assert rc == -1, (rc, err)
        assert all(bool((b == 7.0).all()) for b in bufs)
    finally:
        model.release()


@pytest.mark.parametrize("depth", [0, 2, 4])
@pytest.mark.parametrize("kind", ["glow", "realnvp"])
def test_deterministic(kind, depth):
    """Weight / bias gradients and dL/dx are bitwise equal across calls (no atomics); the ActNorm gradients (atomics) agree
    to 1e-6."""
    model = _model(kind, 33, 128, 3, depth, act="tanh" if kind == "glow" else "mixed", mode="f16")
    try:
        x = _rows(1000, 33, 120)
        dz, dldj = _upstream(1000, 33, 121)
        named = list(model.flows[1].named_parameters())
        runs = []
        for _ in range(2):
            grads, dx = model._component_backward(1, x, dz, dldj, with_dx=True)
            runs.append([grads[id(p)].clone() for _, p in named] + [dx.clone()])
        for i, (a, b) in enumerate(zip(*runs)):
            if i < len(named) and "actnorm" in named[i][0]:
                assert float((a - b).abs().max()) <= 1e-6 * float(a.abs().max()), i
            else:
                assert torch.equal(a, b), i
    finally:
        model.release()


def test_training_loop_at_depth_2(monkeypatch):
    """compute_kl_pq_loss(...)['nll'].backward() + clip + Adam (density_experiment.py:359-374) on an f16 handle with
    coupling_network_depth 2: every step trains the new component through the fused backward, and the loss goes down."""
    fused = []
    apply = bf._FusedComponentFlow.apply
    monkeypatch.setattr(bf._FusedComponentFlow, "apply", lambda *a: fused.append(1) or apply(*a))
    md = orc.make_synthetic_model("glow", 10, 3, 3, 128, seed=2, depth=2)
    model = build_model(md, "cuda", gemm_mode="f16")
    try:
        model.component, model.all_trained = 2, False
        for i, f in enumerate(model.flows):
            for p in f.parameters():
                p.requires_grad_(i == 2)
        model.train()
        opt = torch.optim.Adam(list(model.flows[2].parameters()), lr=2e-3)
        x = torch.randn(512, 10, device="cuda", generator=torch.Generator(device="cuda").manual_seed(7)) * 0.5 + 0.3
        args = argparse.Namespace(flow="boosted")
        gen = torch.Generator(device="cuda").manual_seed(11)
        first = last = None
        for _ in range(30):
            opt.zero_grad()
            losses = gbnf_b200.compute_kl_pq_loss(model, x, args, generator=gen)
            losses["nll"].backward()
            torch.nn.utils.clip_grad_norm_(model.flows[2].parameters(), 5.0)
            opt.step()
            last = float(losses["g_nll"].detach())
            first = last if first is None else first
        assert len(fused) == 30
        assert math.isfinite(last) and last < first - 0.05, (first, last)
        model.check_status()
    finally:
        model.release()
