"""Fixture configurations shared by make_golden.py (needs the reference) and the tests (do not)."""
import argparse

CONFIGS = {
    # name: (args kwargs, seed, B, toy_base)
    "glow_d43": (dict(kind="glow", D=43, C=3, K=2, h=64), 1, 192, False),
    "glow_d6_additive_relu": (dict(kind="glow", D=6, C=2, K=3, h=64, flow_coupling="additive", coupling_network="relu",
                                   flow_permutation="reverse"), 2, 160, False),
    "realnvp_d6_bn": (dict(kind="realnvp", D=6, C=4, K=5, h=64, batch_norm=True), 3, 200, False),
    "realnvp_d5_mixed": (dict(kind="realnvp", D=5, C=3, K=4, h=64, coupling_network="mixed"), 4, 130, False),
    # wide enough (h % 128 == 0) for the pipelined tensor-core kernel: pins it against the reference itself
    "glow_d43_h256": (dict(kind="glow", D=43, C=2, K=2, h=256), 6, 160, False),
    "realnvp_d6_h128_bn": (dict(kind="realnvp", D=6, C=2, K=3, h=128, batch_norm=True), 7, 150, False),
    "toy_d2": (dict(kind="realnvp", D=2, C=8, K=1, h=64, rho_init="uniform"), 5, 100, True),
    # the HEADLINE instantiation of the pipelined kernel (h = 512: tight TMEM geometry, 128 / 64-column layer-2 chunks) and a
    # depth-2 coupling network (serial tensor-core kernel), both pinned against the reference itself
    "glow_d43_h512": (dict(kind="glow", D=43, C=2, K=2, h=512), 8, 160, False),
    "glow_d43_h128_depth2": (dict(kind="glow", D=43, C=2, K=2, h=128, coupling_network_depth=2), 9, 150, False),
    # ResidualNet s / t networks (models/layers.py:246-301): one and two pre-activation blocks
    "realnvp_d6_residual": (dict(kind="realnvp", D=6, C=2, K=3, h=64, coupling_network="residual"), 10, 140, False),
    "realnvp_d5_residual2_bn": (dict(kind="realnvp", D=5, C=2, K=2, h=64, coupling_network="residual", coupling_network_depth=2,
                                     batch_norm=True), 11, 120, False),
    # Glow with the invertible 1x1 convolution as the permutation (models/glow.py:275-278, models/layers.py:722-796; LU-decomposed
    # and plain).  (Glow + ResidualNet cannot be built upstream: models/glow.py:294 names ResidualNet without importing it.)  Upstream's InvertibleConv1x1.forward unpacks a
    # 4-D shape and crashes on feature vectors: make_golden.py feeds it [B, D, 1, 1] views (the fixture script only).
    "glow_d6_invconv": (dict(kind="glow", D=6, C=2, K=3, h=64, flow_permutation="invconv"), 13, 150, False),
    "glow_d43_invconv_plain": (dict(kind="glow", D=43, C=2, K=2, h=64, flow_permutation="invconv", LU_decomposed=False), 14, 140, False),
}
# fixtures whose initial state_dict is stored as per-tensor SHA-1 digests instead of values (file size: every fixture stays under 1 MB)
STATE0_DIGEST_ONLY = {"glow_d43_h512", "glow_d43_h256", "glow_d43_h128_depth2", "realnvp_d6_bn", "realnvp_d6_h128_bn",
                      "realnvp_d5_residual2_bn"}
# fixtures whose coupling-network weights and biases are not stored at all: they are the seeded initial values (nothing before the
# fixture is taken changes them), rebuilt by store.load() from the seed.  Subset of STATE0_DIGEST_ONLY: the digests vouch for them.
SEEDED_WEIGHTS = {"glow_d43_h512", "glow_d43_h256"}


def make_args(kind, D, C, K, h, **kw):
    """The reference's argument namespace for a fixture (density_experiment.py defaults, CPU)."""
    import torch
    a = argparse.Namespace(
        flow="boosted", boosted=True, density_evaluation=True, device=torch.device("cpu"), cuda=False,
        component_type=kind, num_components=C, num_flows=K, z_size=D, input_size=[D], h_size=h,
        rho_init="decreasing", coupling_network="tanh", coupling_network_depth=1, batch_norm=False,
        flow_permutation="shuffle", flow_coupling="affine", actnorm_scale=1.0, LU_decomposed=True, num_blocks=1,
        num_dequant_blocks=0, learn_top=False, y_classes=1, y_condition=False, sample_size=16, save_results=False,
        num_components_=C, batch_size=64, rho_iters=0)
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def fixture_args(name):
    kw = dict(CONFIGS[name][0])
    return make_args(kw.pop("kind"), kw.pop("D"), kw.pop("C"), kw.pop("K"), kw.pop("h"), **kw)
