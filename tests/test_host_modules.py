"""Host-side mirror of the reference API (no GPU): constructors, state_dict keys, RNG order, autograd forward."""
import numpy as np
import pytest
import torch

import gbnf_b200
from conftest import ALL_CASES as GOLDEN_CASES
from helpers import args_for, build_model, golden_model, load_into
from tests.golden.configs import CONFIGS


def _fresh(name, g):
    kw, seed, B, toy = CONFIGS[name]
    md = golden_model(g)
    perm = kw.get("flow_permutation", "shuffle")
    bn = kw.get("batch_norm", False)
    a = args_for(md, "cpu", flow_permutation=perm, batch_norm=bn, rho_init=kw.get("rho_init", "decreasing"),
                 LU_decomposed=kw.get("LU_decomposed", True))
    assert a.coupling_network == kw.get("coupling_network", "tanh")
    torch.manual_seed(seed)
    return gbnf_b200.BoostedFlow(a), md


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_same_seed_same_initial_state_as_reference(golden, name):
    """Same torch seed => bit-identical state_dict keys, shapes and values as the reference constructor."""
    g = golden(name)
    model, md = _fresh(name, g)
    ref = {k[len("state0."):]: v for k, v in g.items() if k.startswith("state0.")}
    mine = {k: v.numpy() for k, v in model.state_dict().items()}
    sha = {k[len("state0sha."):]: v for k, v in g.items() if k.startswith("state0sha.")}    # large fixtures: digests only
    assert sorted(ref) == sorted(mine) or sorted(sha) == sorted(mine)
    for k in ref:
        assert ref[k].shape == mine[k].shape, k
        np.testing.assert_array_equal(ref[k], mine[k], err_msg=k)
    for k in sha:
        import hashlib
        assert hashlib.sha1(np.ascontiguousarray(mine[k]).tobytes()).digest() == sha[k].tobytes(), k
    if md["kind"] == "glow" and CONFIGS[name][0].get("flow_permutation") != "invconv":   # permutation indices are not in the state_dict; they must match too
        for c in range(md["C"]):
            for k, st in enumerate(model.flows[c].steps()):
                np.testing.assert_array_equal(st.permutation.indices.numpy(), md["components"][c]["steps"][k]["perm"])


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_autograd_forward_matches_reference(golden, name):
    """The caller-side torch forward used for the component under training equals the reference's fp32 output."""
    g = golden(name); md = golden_model(g)
    model = build_model(md, "cpu")
    x = torch.from_numpy(g["x"])
    for c in range(md["C"]):
        z, ldj = model.flows[c].forward_autograd(x)
        np.testing.assert_allclose(z.detach().numpy(), g["z32"][c], rtol=2e-5, atol=2e-5)
        np.testing.assert_allclose(ldj.detach().numpy(), g["ldj32"][c], rtol=2e-5, atol=2e-5)
    # gradients flow to the component's parameters
    for p in model.flows[0].parameters():
        p.requires_grad_(True)
    model.component = 0
    z, _, _, ldj, _ = model(x=x, components="c")
    (z.pow(2).sum() + ldj.sum()).backward()
    assert all(p.grad is not None for p in model.flows[0].parameters() if p.requires_grad)


def test_extract_roundtrip(golden):
    g = golden("realnvp_d6_bn"); md = golden_model(g)
    model = build_model(md, "cpu")
    md2 = gbnf_b200.extract_model(model)
    for c in range(md["C"]):
        for k in range(md["K"]):
            a, b = md["components"][c]["steps"][k], md2["components"][c]["steps"][k]
            for (W1, b1), (W2, b2) in zip(a["t"] + a["s"], b["t"] + b["s"]):
                np.testing.assert_array_equal(W1, W2); np.testing.assert_array_equal(b1, b2)
            assert (a["bn"] is None) == (b["bn"] is None)


def test_component_state_machine_and_sampling_strings(golden):
    g = golden("glow_d43"); md = golden_model(g)
    m = build_model(md, "cpu")
    C = md["C"]
    assert m.component == 0 and not m.all_trained
    for i in range(1, C):
        m.increment_component(); assert m.component == i and not m.all_trained
    m.increment_component(); assert m.component == 0 and m.all_trained          # models/boosted_flow.py:52-59
    m.component, m.all_trained = 1, False
    assert m._sample_component("c") == 1
    torch.manual_seed(0)
    assert m._sample_component("1:c-1") == 0                                     # only component 0 is fixed
    assert m._sample_component("1:c") in (0, 1)
    m.all_trained = True
    assert m._sample_component("-c") != 1
    with pytest.raises(ValueError):
        m._sample_component("all")
    with pytest.raises(NotImplementedError):
        a = args_for(md); a.component_type = "maf"; gbnf_b200.BoostedFlow(a)
    assert isinstance(m.base_dist, torch.distributions.Normal)
    np.testing.assert_allclose(m.rho.numpy(), np.maximum(1 / 2.0 ** np.arange(C), 0.05).astype(np.float32))


def test_no_cpu_fallback(golden):
    """Product path must fail loudly without CUDA: no oracle, no torch fallback for fixed components."""
    g = golden("glow_d43"); md = golden_model(g)
    m = build_model(md, "cpu")
    x = torch.from_numpy(g["x"])
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    with torch.no_grad():
        with pytest.raises((RuntimeError, AssertionError)):
            m(x=x, components=0)
    with pytest.raises((RuntimeError, AssertionError)):
        m.mixture_log_density(x, 2)
    import inspect
    import gbnf_b200.boosted_flow as bf, gbnf_b200.losses as ls, gbnf_b200.dist as ds, gbnf_b200._lib as lb
    for mod in (bf, ls, ds, lb):
        assert "oracle" not in inspect.getsource(mod).replace("the oracle", "").replace("CPU oracle", "")


def test_actnorm_uninitialised_raises_in_eval(golden):
    g = golden("glow_d43"); md = golden_model(g)
    a = args_for(md)
    torch.manual_seed(0)
    m = gbnf_b200.BoostedFlow(a)
    m.eval()
    with pytest.raises(ValueError):                                              # models/layers.py:474-475
        m(x=torch.from_numpy(g["x"]), components=0)
    m.train()
    m(x=torch.from_numpy(g["x"]), components=0)                                  # data-dependent init on first train batch
    st = m.flows[0].steps()[0]
    assert st.actnorm.inited
    y = (torch.from_numpy(g["x"]) + st.actnorm.bias) * torch.exp(st.actnorm.logs)
    np.testing.assert_allclose(y.mean(0).detach().numpy(), 0, atol=1e-5)
    np.testing.assert_allclose((y ** 2).mean(0).detach().numpy(), 1, atol=1e-3)


def test_fused_backward_depth_bound():
    """The shared-memory count that decides which components train through the fused backward: the deepest component served
    at a few shapes (the table in include/gbnf.h).  tests/test_gpu_train_backward.py pins the count to the library's own."""
    from gbnf_b200.boosted_flow import FUSED_BACKWARD_MAX_SMEM, fused_backward_smem_bytes

    def deepest(kind, D, h):
        K = 0
        while fused_backward_smem_bytes(kind, D, h, K + 1) <= FUSED_BACKWARD_MAX_SMEM:
            K += 1
        return K
    assert [deepest("glow", D, 512) for D in (2, 21, 43, 64)] == [27, 20, 15, 12]
    assert [deepest("realnvp", D, 512) for D in (2, 21, 43, 64)] == [14, 11, 9, 8]
    assert [deepest("glow", D, 64) for D in (2, 21, 43, 64)] == [47, 36, 28, 23]
    assert [deepest("realnvp", D, 64) for D in (2, 21, 43, 64)] == [24, 20, 17, 15]
    # cfg3 / cfg4 (Glow, h = 512): one 16 x 64 output block per step, not two
    assert fused_backward_smem_bytes("glow", 43, 512, 5) == 178432 - 5 * 16 * 64 * 4
    assert fused_backward_smem_bytes("glow", 21, 512, 10) == 214848 - 10 * 16 * 64 * 4
