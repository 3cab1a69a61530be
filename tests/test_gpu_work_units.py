"""The production tensor-core kernels' work units (-m gpu), against the fp64 oracle and against their own larger batches.

The pipelined kernels -- the single chain (coupling_tc2.cuh), the two-chain kernel (coupling_tc4.cuh), the interleaved s / t
kernel (coupling_tc5.cuh) and the CTA pair (coupling_tc3.cuh) -- split each 128-row tile's components over `split` work units.
Every unit leaves its mixture terms coef_c + log q_c in scratch on the handle; the last unit of a tile to arrive (an atomic ticket
it resets) reduces them in component order.  Each CTA, or CTA pair, walks units u, u + grid, ...  These tests pin what that
machinery promises: G_ll and log q do not depend on the split, the batch, the grid or what ran before on the handle.

The split is read off model.info()["grid"]: while the unit count is below the number of workers (SMs, or resident CTA pairs),
grid = tiles * split (twice that for the pair).  The batches are chosen to land on the splits named in SPLITS; a change to the
cost model that moves them fails the coverage assertion rather than silently testing something else.  GBNF_TC4 is read when a
handle is created, GBNF_GRID at every launch.

Tolerances are those of tests/test_gpu_parity.py: 1e-4 relative on log q and G_ll, plus an absolute 2e-2 for RealNVP and for
D < 16.

Measured on an NVIDIA B200 (1000 W power limit), largest error against the oracle over log q and G_ll in both f16 modes.  Glow
with D >= 16, relative: single chain 2.9e-5 (D = 43, h = 256), two-chain 3.0e-5 (D = 43, h = 512; 4.3e-5 on the cfg3 shape's odd
counts), CTA pair 2.4e-5 (D = 21).  RealNVP and D < 16, absolute: single chain 9.1e-3 (RealNVP ReLU with BatchNorm, D = 5) and
8.6e-4 (Glow D = 4, C = 256), two-chain 8.2e-4 (Glow D = 8, C = 34), interleaved 7.3e-4, CTA pair 3.1e-3 (RealNVP D = 9).  The
module runs in about 20 s there."""
import ctypes as C

import numpy as np
import pytest
import torch

from gbnf_b200 import _lib
from helpers import build_model
from oracle import gbnf_oracle as orc

pytestmark = pytest.mark.gpu

MODES = ["f16", "f16fast"]
NAN = float("nan")

# name -> (kind, D, C, K, h, extra model args, GBNF_TC4 at handle creation, route)
MODELS = {
    "single_glow_d43_h256_c5": ("glow", 43, 5, 2, 256, {}, None, "single"),
    "single_glow_d43_h256_c7": ("glow", 43, 7, 2, 256, {}, None, "single"),
    "single_realnvp_relu_bn_d5_h128_c6": ("realnvp", 5, 6, 2, 128, dict(act="relu", batch_norm=True), None, "single"),
    "two_glow_d43_h512_c6": ("glow", 43, 6, 2, 512, {}, None, "two"),
    "two_glow_d43_h512_c6_forced": ("glow", 43, 6, 2, 512, {}, "2", "two"),
    "two_glow_d43_h512_c8": ("glow", 43, 8, 2, 512, {}, None, "two"),
    "two_glow_d43_h512_c8_forced": ("glow", 43, 8, 2, 512, {}, "2", "two"),
    "interleaved_realnvp_toy_d6_h256_c6": ("realnvp", 6, 6, 2, 256, dict(toy_base=True), None, "interleaved"),
    "pair_glow_d21_h1024_c6": ("glow", 21, 6, 1, 1024, {}, None, "pair"),
    "pair_realnvp_d9_h1024_c4": ("realnvp", 9, 4, 1, 1024, {}, None, "pair"),
    "many_single_glow_d4_h128_c256": ("glow", 4, 256, 1, 128, {}, None, "single"),
    "many_two_glow_d8_h512_c34": ("glow", 8, 34, 1, 512, {}, None, "two"),
}
# splits test_split_and_batch_independence must see (where the grid shows them): split 1, a split at or near C (a unit per
# component or per pair of components), and a ragged final unit (C = 5 over 3 units of 2, C = 7 over 4 units of 2)
SPLITS = {
    "single_glow_d43_h256_c5": {1, 3},
    "single_glow_d43_h256_c7": {1, 4},
    "single_realnvp_relu_bn_d5_h128_c6": {1, 3},
    "two_glow_d43_h512_c6": {1, 3},
    "two_glow_d43_h512_c6_forced": {1, 3},
    "two_glow_d43_h512_c8": {1, 2, 8},
    "two_glow_d43_h512_c8_forced": {1, 2, 4},
    "interleaved_realnvp_toy_d6_h256_c6": {1, 3},
    "pair_glow_d21_h1024_c6": {1, 3},
    "pair_realnvp_d9_h1024_c4": {1, 4},
    "many_single_glow_d4_h128_c256": {64, 128},
    "many_two_glow_d8_h512_c34": {1, 17},
}
ROWS = 65536 + 77          # the largest batch: a ragged multi-wave batch on every kernel
_MD = {}


def synth(name):
    if name not in _MD:
        kind, D, C_, K, h, kw, _, _ = MODELS[name]
        _MD[name] = orc.make_synthetic_model(kind, D, C_, K, h, seed=31 + C_, init_rows=1024, **kw)
    return _MD[name]


def make(name, mode, monkeypatch):
    """A model whose handle was created with the case's GBNF_TC4 (the switch is read when pack_all creates the handle)."""
    tc4 = MODELS[name][6]
    if tc4 is None:
        monkeypatch.delenv("GBNF_TC4", raising=False)
    else:
        monkeypatch.setenv("GBNF_TC4", tc4)
    monkeypatch.delenv("GBNF_GRID", raising=False)
    m = build_model(synth(name), "cuda", gemm_mode=mode)
    m.pack_all()
    return m


def assert_route(model, name, n):
    """The kernel the handle's last launch of n components ran on; returns info().  A two-chain handle runs the single chain
    where the cost model prefers it (two_chain 0) unless GBNF_TC4=2 forces two chains, which it can for an even n only (an odd
    n ends with the single chain's launch on the last component)."""
    inf = model.info()
    route, forced = MODELS[name][7], MODELS[name][6] == "2"
    if route == "single":
        assert inf["pipelined"] == 1 and inf["two_chain"] == 0, inf
    elif route == "two":
        assert inf["pipelined"] == 1 and inf["two_chain"] in ((1,) if forced and n % 2 == 0 else (0, 1)), inf
    elif route == "interleaved":
        assert inf["pipelined"] == 1 and inf["two_chain"] == 2, inf
    else:
        assert inf["pipelined"] == 2 and inf["two_chain"] == 0, inf
    return inf


def workers_of(inf, name):
    """CTAs, or CTA pairs, of the last launch's grid."""
    return inf["grid"] // 2 if MODELS[name][7] == "pair" else inf["grid"]


def rows(D, B, seed=41):
    return np.random.default_rng(seed).standard_normal((B, D)).astype(np.float32)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def atol_of(md):
    return 2e-2 if md["kind"] == "realnvp" or md["D"] < 16 else 0.0


def close(got, ref, md, what):
    got = np.asarray(got.cpu() if torch.is_tensor(got) else got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    err = np.abs(got - ref)
    bad = err > (1e-4 + 2e-6) * np.abs(ref) + atol_of(md)
    print(f"[{what}] max abs err {float(err.max()):.3e}, max rel err {float(np.max(err / np.abs(ref))):.3e}")
    assert not bad.any(), (what, float(err.max()), float(np.max(err / np.abs(ref))))


def fused(model, x, n, skip_c=-1, raw=False):
    """gbnf_fused_eval with G_ll and log q pre-filled with NaN: a row or column no unit wrote cannot pass."""
    B = x.shape[0]
    G = torch.full((B,), NAN, device=x.device)
    lq = torch.full((B, n), NAN, device=x.device)
    rho = model.rho.detach().to(x.device, torch.float32).contiguous()
    _lib.check(_lib.load().gbnf_fused_eval(model.handle(x.device), x.data_ptr(), B, n, rho.data_ptr(), skip_c,
                                           _lib.MIX_RAW_RHO if raw else _lib.MIX_SIMPLEX, G.data_ptr(), lq.data_ptr(),
                                           C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return G, lq


# ---- 1. the fused mixture options against the oracle ------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", list(MODELS))
def test_mixture_options_vs_oracle(name, mode, monkeypatch):
    md = synth(name)
    C_ = md["C"]
    x = rows(md["D"], 517)                  # four full tiles and a ragged one: split > 1 on every kernel
    xd = dev(x)
    model = make(name, mode, monkeypatch)
    try:
        _, lq = fused(model, xd, C_)
        assert_route(model, name, C_)
        ref = orc.all_component_logq(orc.cast_model(md, np.float64), x.astype(np.float64))
        close(lq, ref, md, f"{name} {mode} log q")
        rho = md["rho"].astype(np.float64)
        for n in sorted({1, 2, 3, C_ - 1, C_} & set(range(1, C_ + 1))):
            for skip_c in sorted({-1} | {s for s in (1, n - 1) if 1 <= s < n}):
                for raw in (False, True):
                    G, lqn = fused(model, xd, n, skip_c, raw)
                    assert_route(model, name, n)
                    close(G, orc.mixture_recursion(ref, rho, n, skip_c, normalized=not raw), md,
                          f"{name} {mode} G_ll n {n} skip_c {skip_c} raw_rho {raw}")
                    assert torch.equal(lqn, lq[:, :n]), (n, skip_c, raw)
                    # the standalone mixture kernel on the kernel's own log q: the same value up to logsumexp reassociation
                    Gu = model.mixture_from_logq(lqn, n, skip_c=skip_c, raw_rho=raw)
                    np.testing.assert_allclose(Gu.cpu().numpy(), G.cpu().numpy(), rtol=2e-6, atol=2e-6)
        model.check_status()
    finally:
        model.release()


# ---- 2. the split and the batch do not change a row's bits ---------------------------------------------------------------------------
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", list(MODELS))
def test_split_and_batch_independence(name, mode, monkeypatch):
    md = synth(name)
    C_ = md["C"]
    x = rows(md["D"], ROWS, seed=42)
    xd = dev(x)
    model = make(name, mode, monkeypatch)
    try:
        G_all, lq_all = fused(model, xd, C_)
        inf = assert_route(model, name, C_)
        workers = workers_of(inf, name)     # 513 tiles: more units than workers, so the grid is every worker
        routes, splits = {inf["two_chain"]}, set()
        sms = inf["num_sms"]
        # one tile, a few tiles, 60 and 140 tiles (below a wave of pairs / of CTAs), the wave edge and one row past it
        for B in (1, 77, 128, 129, 517, 60 * 128 - 23, 140 * 128 - 23, sms * 128, sms * 128 + 1):
            G, lq = fused(model, xd[:B], C_)
            inf = assert_route(model, name, C_)
            routes.add(inf["two_chain"])
            assert torch.equal(G, G_all[:B]), (B, "G_ll")
            assert torch.equal(lq, lq_all[:B]), (B, "log q")
            tiles, w = -(-B // 128), workers_of(inf, name)
            if w < workers:
                assert w % tiles == 0, (B, inf)
                splits.add(w // tiles)
        assert SPLITS[name] <= splits, (sorted(splits), "the batches no longer land on the splits this test is meant to cover")
        if MODELS[name][7] == "two":
            assert 1 in routes, routes
        model.check_status()
        # a subset against the oracle: the first tile and the ragged last one of the largest batch
        idx = np.r_[0:128, ROWS - 77:ROWS]
        ref = orc.all_component_logq(orc.cast_model(md, np.float64), x[idx].astype(np.float64))
        close(lq_all.cpu().numpy()[idx], ref, md, f"{name} {mode} log q")
        close(G_all.cpu().numpy()[idx], orc.mixture_recursion(ref, md["rho"].astype(np.float64), C_), md, f"{name} {mode} G_ll")
    finally:
        model.release()


# ---- 3. capped grids: every CTA (pair) walks several units -----------------------------------------------------------------------
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", list(MODELS))
def test_capped_grid_is_bitwise_equal(name, mode, monkeypatch):
    md = synth(name)
    C_, B = md["C"], 517
    xd = dev(rows(md["D"], B, seed=43))
    pair = MODELS[name][7] == "pair"
    model = make(name, mode, monkeypatch)
    try:
        def run():
            G, lq = fused(model, xd, C_)
            infs = [assert_route(model, name, C_)]
            z, ldj = model.component_forward(xd, C_ - 1)
            infs.append(model.info())
            xi, ldji = model.component_inverse(z, C_ - 1)
            infs.append(model.info())
            return (G, lq, z, ldj, xi, ldji), infs

        base, infs = run()
        tiles = -(-B // 128)
        assert workers_of(infs[0], name) > tiles, ("the fused launch must split the tiles' components", infs[0])
        for grid in (1, 2, 3):
            monkeypatch.setenv("GBNF_GRID", str(grid))
            got, infs = run()
            for inf in infs:
                assert inf["grid"] == (2 * grid if pair else grid), (grid, inf)
            for k, a, b in zip(("G_ll", "log q", "z", "ldj", "inverse x", "inverse ldj"), base, got):
                assert torch.equal(a, b), (grid, k)
        model.check_status()
    finally:
        model.release()


# ---- 4. the tile tickets and the mixture-term scratch carried from launch to launch on one handle ---------------------------------
# Each step's result must be the bits of the same call on a freshly created handle.  tile_ctr is zeroed only when it is
# allocated (room for at least 1024 tiles); in between, every last arriver must have reset its ticket.
REUSE_MODELS = ["two_glow_d43_h512_c8", "many_single_glow_d4_h128_c256"]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", REUSE_MODELS)
def test_ticket_and_scratch_reuse(name, mode, monkeypatch):
    md = synth(name)
    x = dev(rows(md["D"], 131073 + 77, seed=44))        # 1025 tiles: past the first tile_ctr allocation
    steps = [("fused", 517, 8, -1), ("fused", 131073 + 77, 8, -1), ("fused", 517, 8, -1), ("fused", 20003, 8, -1),
             ("fused", 20003, 3, -1), ("fused", 20003, 8, -1), ("fused", 517, 3, -1), ("fused", 517, 8, 1),
             ("fused", 517, 8, -1), ("fused", 517, 8, 7), ("logq", 517, 8, -1), ("fused", 517, 8, -1),
             ("forward", 20003, 5, -1), ("fused", 20003, 8, -1), ("fused", 65536, 7, -1), ("fused", 512, 7, 6),
             ("fused", 65536, 3, 1), ("fused", 20003, 5, -1), ("fused", 517, 8, -1)]
    model = make(name, mode, monkeypatch)
    fresh = make(name, mode, monkeypatch)
    try:
        for i, (what, B, n, skip_c) in enumerate(steps):
            outs = []
            for m in (model, fresh):
                if m is fresh:
                    m.release()
                    m.pack_all()                          # a new handle: tile_ctr and the scratch start from nothing
                xb = x[:B]
                if what == "fused":
                    G, lq = fused(m, xb, n, skip_c)
                    assert torch.isfinite(G).all() and torch.isfinite(lq).all(), (i, what, B, n, skip_c)
                    outs.append((G, lq))
                elif what == "logq":
                    outs.append((m.component_log_density(xb, 0, n),))
                else:
                    outs.append(m.component_forward(xb, n))
                assert_route(m, name, n)
            for a, b in zip(*outs):
                assert torch.equal(a, b), (i, what, B, n, skip_c)
        model.check_status()
        fresh.check_status()
    finally:
        model.release()
        fresh.release()


# ---- 5. odd component counts on the cfg3 shape (Glow D = 43, C = 8, K = 5, h = 512) -------------------------------------------------
# An odd n >= 3 runs as two launches -- the two-chain kernel on the first n - 1 (mixture terms only), the single chain on the last
# component -- exactly when the cost model puts n - 1 components on the two-chain kernel; otherwise as one single-chain launch.
_CFG3 = {}


@pytest.fixture(scope="module")
def cfg3_models():
    yield _CFG3
    for m in _CFG3.values():
        m.release()
    _CFG3.clear()


def cfg3_model(mode, tc4):
    if (mode, tc4) not in _CFG3:
        if "cfg3" not in _MD:
            _MD["cfg3"] = orc.make_synthetic_model("glow", 43, 8, 5, 512, seed=8, init_rows=1024)
        with pytest.MonkeyPatch.context() as mp:
            mp.delenv("GBNF_GRID", raising=False)
            if tc4 is None:
                mp.delenv("GBNF_TC4", raising=False)
            else:
                mp.setenv("GBNF_TC4", tc4)
            m = build_model(_MD["cfg3"], "cuda", gemm_mode=mode)
            m.pack_all()
        _CFG3[(mode, tc4)] = m
    return _CFG3[(mode, tc4)]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("B", [512, 20003, 65536])
@pytest.mark.parametrize("n", [3, 5, 7])
def test_odd_counts(n, B, mode, cfg3_models, monkeypatch):
    monkeypatch.delenv("GBNF_GRID", raising=False)
    m, m0 = cfg3_model(mode, None), cfg3_model(mode, "0")
    md = _MD["cfg3"]
    x = rows(43, B, seed=45)
    xd = dev(x)
    m.mixture_log_density(xd, n - 1)
    even_two = m.info()["two_chain"] == 1
    l0 = m.info()["launches"]
    G, lq = fused(m, xd, n)
    assert m.info()["launches"] - l0 == (2 if even_two else 1), (n, B, even_two)
    assert m.info()["pipelined"] == 1 and m.info()["two_chain"] == 0, m.info()    # the last launch is the single chain
    G0, lq0 = fused(m0, xd, n)
    assert torch.equal(G, G0) and torch.equal(lq, lq0)
    idx = np.r_[0:128, B - 64:B]                       # the first tile and the end of the last one
    ref = orc.all_component_logq(orc.cast_model(md, np.float64), x[idx].astype(np.float64), n)
    close(lq.cpu().numpy()[idx], ref, md, f"odd n {n} B {B} {mode} log q")
    rho = md["rho"].astype(np.float64)
    for skip_c in (1, n - 1):                          # n - 1: masks the component the second launch computes
        for raw in (False, True):
            Gs, lqs = fused(m, xd, n, skip_c, raw)
            assert torch.equal(lqs, lq)
            Gs0, _ = fused(m0, xd, n, skip_c, raw)
            assert torch.equal(Gs, Gs0), (skip_c, raw)
            close(Gs.cpu().numpy()[idx], orc.mixture_recursion(ref, rho, n, skip_c, normalized=not raw), md,
                  f"odd n {n} B {B} {mode} G_ll skip_c {skip_c} raw_rho {raw}")
    m.check_status()
    m0.check_status()
