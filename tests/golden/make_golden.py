"""Generates tests/golden/*.npz by running the UNMODIFIED reference (imported from /root/reference, CPU).

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py

The reference has no tests or golden vectors of its own (SURVEY 4), so these fixtures ARE the pin for the oracle:
each file stores a small seeded reference model (all parameters + the permutation indices that are not in the
state_dict), inputs, and the reference's outputs for every function on the hot path, in fp32 (reference numerics)
and from a .double() copy (ground truth).  The script cannot run on the GPU box (no /root/reference there); the
fixtures travel instead.
"""
import copy
import os
import sys
import types

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference"
sys.path.insert(0, ROOT)
sys.path.insert(0, REF)

import numpy as np  # noqa: E402
import torch  # noqa: E402

# logging / IO-only modules the reference drivers import but the hot path never touches
sys.modules.setdefault("tensorboardX", types.SimpleNamespace(SummaryWriter=object))
sys.modules.setdefault("h5py", types.ModuleType("h5py"))
for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.cm", "matplotlib.colors"):
    if name not in sys.modules:
        m = types.ModuleType(name)
        m.use = lambda *a, **k: None
        sys.modules[name] = m

from models.boosted_flow import BoostedFlow as RefBoostedFlow  # noqa: E402
import models.layers as ref_layers  # noqa: E402

# Upstream's InvertibleConv1x1 is written for images: get_weight unpacks `b, c, h, w = sample.shape` (models/layers.py:751) and
# F.conv2d needs 4-D input, so flow_permutation='invconv' crashes on the tabular path.  In THIS SCRIPT ONLY a feature vector is
# handed to the unmodified module as the 1 x 1 image it is; parameters, weight formula and log-det are upstream's own.
_ref_invconv_forward = ref_layers.InvertibleConv1x1.forward


def _invconv_forward_1d(self, sample, logdet=None, reverse=False):
    if sample.dim() == 2:
        if self.LU_decomposed and self.l_mask.dtype != sample.dtype:     # plain attributes: .double() does not convert them, and
            self.l_mask, self.eye = self.l_mask.to(sample.dtype), self.eye.to(sample.dtype)   # get_weight's in-place `u +=` needs one dtype
        z, ld = _ref_invconv_forward(self, sample[:, :, None, None], logdet, reverse)
        return z[:, :, 0, 0], ld
    return _ref_invconv_forward(self, sample, logdet, reverse)


ref_layers.InvertibleConv1x1.forward = _invconv_forward_1d
import density_experiment as ref_density  # noqa: E402
from utils.distributions import log_normal_standard  # noqa: E402

from gbnf_b200.extract import extract_model  # noqa: E402
from oracle import gbnf_oracle as orc  # noqa: E402


from tests.golden.configs import CONFIGS, fixture_args  # noqa: E402
from tests.golden.store import compact  # noqa: E402


def eight_gaussians(n, rng):
    """utils/load_data.py:248-254 shape: 8 modes on a circle of radius ~2.8, sigma ~0.35 (values are only inputs)."""
    centers = np.array([(1, 0), (-1, 0), (0, 1), (0, -1), (0.7071, 0.7071), (0.7071, -0.7071), (-0.7071, 0.7071),
                        (-0.7071, -0.7071)], dtype=np.float32) * 4.0
    pts = rng.standard_normal((n, 2)).astype(np.float32) * 0.5 + centers[rng.integers(0, 8, n)]
    return (pts / 1.414).astype(np.float32)


def ref_forward_all(model, x, toy_base):
    """Per-component z, ldj, logq from the reference model."""
    zs, ldjs, lqs = [], [], []
    for c in range(model.num_components):
        z, _, _, ldj, _ = model(x=x, components=c)
        if toy_base:
            lq = model.base_dist.log_prob(z).sum(1) + ldj
        else:
            lq = log_normal_standard(z, reduce=True, dim=-1, device=torch.device("cpu")) + ldj
        zs.append(z); ldjs.append(ldj); lqs.append(lq)
    return torch.stack(zs, 0), torch.stack(ldjs, 0), torch.stack(lqs, 1)


def build_case(name, out_dir=None):
    """out_dir: where to write (default: next to this script); tests/test_golden_regeneration.py regenerates into a temp dir."""
    _, seed, B, toy_base = CONFIGS[name]
    args = fixture_args(name)
    torch.manual_seed(seed)
    model = RefBoostedFlow(args)
    state0 = {k: v.clone() for k, v in model.state_dict().items()}   # initial state, pins our constructors' RNG order
    rng = np.random.default_rng(1000 + seed)
    D = args.z_size
    if toy_base:
        x_np = eight_gaussians(B, rng)
        x_init = eight_gaussians(512, rng)
    else:
        x_np = rng.standard_normal((B, D)).astype(np.float32)
        x_init = rng.standard_normal((512, D)).astype(np.float32)
    x, xi = torch.from_numpy(x_np), torch.from_numpy(x_init)
    # data-dependent ActNorm init / BatchNorm running statistics: a few train-mode forwards, as the driver does
    # (density_experiment.py:346-356); then perturb BN affine parameters so they are not at their trivial init
    model.train()
    with torch.no_grad():
        for _ in range(3):
            for c in range(model.num_components):
                model(x=xi, components=c)
        for n_, p in model.named_parameters():
            if n_.endswith("log_gamma") or n_.endswith("beta"):
                p.add_(0.1 * torch.randn_like(p))
    model.eval()
    with torch.no_grad():
        z32, ldj32, lq32 = ref_forward_all(model, x, toy_base)
    m64 = copy.deepcopy(model).double()
    for c in range(model.num_components):          # plain attributes deepcopy keeps; make the intent explicit
        if args.component_type == "glow":
            for k in range(args.num_flows):
                src = model.flows[c].flow.layers[k]
                dst = m64.flows[c].flow.layers[k]
                dst.actnorm.inited = True
                if hasattr(src, "invconv"):
                    # FlowStep.flow_permutation is a lambda closing over the ORIGINAL step (models/glow.py:277-278); deepcopy keeps
                    # the function object, so the copy would run the fp32 convolution: rebind it to the copy's own module
                    dst.flow_permutation = lambda z, logdet, rev, _s=dst: _s.invconv(z, logdet, rev)
                    continue
                psrc = src.shuffle if hasattr(src, "shuffle") else src.reverse
                pdst = dst.shuffle if hasattr(dst, "shuffle") else dst.reverse
                pdst.indices = psrc.indices.clone()
    with torch.no_grad():
        z64, ldj64, lq64 = ref_forward_all(m64, x.double(), toy_base)

    out = {"x": x_np, "x_init": x_init, "z32": z32.numpy(), "ldj32": ldj32.numpy(), "logq32": lq32.numpy(),
           "z64": z64.numpy(), "ldj64": ldj64.numpy(), "logq64": lq64.numpy()}
    for k, v in state0.items():
        out["state0." + k] = v.numpy()
    out["seed"] = np.array(seed)
    # inverse direction: the reference's own decode where it is not broken upstream (1-D Glow with ADDITIVE coupling:
    # FlowStep.decode glow.py:344-366; the affine branch raises on 2-D tensors, RealNVP's decode is not an inverse -- SURVEY 7)
    if args.component_type == "glow" and args.flow_coupling == "additive":
        with torch.no_grad():
            for c in range(model.num_components):
                xr = model.flows[c](z=z32[c], y_onehot=None, temperature=None, reverse=True)
                out[f"dec32.c{c}"] = xr.numpy()
                out[f"dec64.c{c}"] = m64.flows[c](z=z64[c], y_onehot=None, temperature=None, reverse=True).numpy()
    md = extract_model(model, toy_base=toy_base)
    for k, v in orc.flatten_model(md).items():
        out["model." + k] = v

    # ---- mixture / weights / resampling / objective through the reference driver functions ----------------
    C = args.num_components
    if not toy_base:
        for comp, all_tr in [(c, False) for c in range(1, C)] + [(1 if C > 2 else 0, True)]:
            model.component, model.all_trained = comp, all_tr
            tag = f"kl.c{comp}.a{int(all_tr)}."
            torch.manual_seed(77 + comp)
            with torch.no_grad():
                losses = ref_density.compute_kl_pq_loss(model, x, args)
            # replay the intermediate quantities exactly as density_experiment.py:612-644 computes them
            with torch.no_grad():
                G_ll = torch.zeros(x.size(0))
                for c in range(model.component):
                    if c == 0:
                        G_ll = lq32[:, 0]
                    else:
                        rs = model.rho[0:(c + 1)] / torch.sum(model.rho[0:(c + 1)])
                        G_ll = torch.logsumexp(torch.stack([torch.log(1 - rs[c]) + G_ll, torch.log(rs[c]) + lq32[:, c]], 1), 1)
                w = ref_density.softmax(-G_ll)
                clamped = bool(w.max() > 0.1)
                if clamped:
                    w = torch.max(torch.min(w, torch.tensor([0.1])), torch.tensor([0.01]))
                if w.sum() != 1.0:
                    w = w / torch.sum(w)
                torch.manual_seed(77 + comp)
                idx = torch.multinomial(w, x.size(0), replacement=True)
                torch.manual_seed(77 + comp)
                u = torch.rand(x.size(0), dtype=torch.float64)
            out[tag + "G_ll"] = G_ll.numpy(); out[tag + "w"] = w.numpy(); out[tag + "clamped"] = np.array(clamped)
            out[tag + "idx"] = idx.numpy(); out[tag + "u"] = u.numpy()
            for k in ("nll", "G_nll", "g_nll"):
                out[tag + k] = np.array(float(losses[k]))
            # the oracle's resampling contract must reproduce torch.multinomial on these very weights
            assert np.array_equal(orc.resample_indices(w.numpy(), u.numpy()), idx.numpy()), "multinomial replay mismatch"
            # the unclamped branch: flatten G_ll so that no weight exceeds 0.1
            with torch.no_grad():
                G_flat = G_ll * (0.02 / max(1e-6, float(G_ll.std()))) if model.component > 0 else G_ll
                w2 = ref_density.softmax(-G_flat)
                assert not bool(w2.max() > 0.1)
                if w2.sum() != 1.0:
                    w2 = w2 / torch.sum(w2)
            out[tag + "G_flat"] = G_flat.numpy(); out[tag + "w_flat"] = w2.numpy()
        # evaluate(): density_experiment.py:544-603
        for comp, all_tr in [(0, False), (C - 1, False), (1 if C > 2 else 0, True)]:
            model.component, model.all_trained = comp, all_tr
            loader = [(x[:B // 2], None), (x[B // 2:], None)]
            with torch.no_grad():
                ev = ref_density.evaluate(model, loader, args)
            for k, v in ev.items():
                out[f"eval.c{comp}.a{int(all_tr)}.{k}"] = np.array(v)
        # update_rho loop (models/boosted_flow.py:141-207).  Upstream formats two undefined names into a LOG message at :185
        # (NameError whenever rho_iters > 0 and component > 0); they are defined here, in the fixture script only, so that the
        # reference's own loop runs: the arithmetic (decayed-step SGD on rho[component], clamp to [0.01, 100]) is untouched.
        import models.boosted_flow as ref_bf_module
        ref_bf_module.g_nll = torch.zeros(2); ref_bf_module.G_nll = torch.zeros(2)
        rho0 = model.rho.clone()
        model.component, model.all_trained = C - 1, False
        args.rho_iters, args.rho_lr, args.snap_dir = 14, 0.05, "/tmp"
        model.args.rho_iters, model.args.rho_lr, model.args.snap_dir = 14, 0.05, "/tmp"
        model.update_rho([(x[:B // 2], None), (x[B // 2:], None)])
        out["urho.rho_final"] = model.rho.detach().numpy().copy()
        out["urho.iters"] = np.array(14); out["urho.lr"] = np.array(0.05)
        with torch.no_grad():
            model.rho.copy_(rho0)
        model.args.rho_iters = args.rho_iters = 0
        # _rho_gradients raw-rho recursion (models/boosted_flow.py:119-139)
        model.component, model.all_trained = C - 1, False
        new_ll, fixed_ll, full_ll = model._rho_gradients(x)
        out["rhograd.new"], out["rhograd.fixed"], out["rhograd.full"] = new_ll.numpy(), fixed_ll.numpy(), full_ll.numpy()
    else:
        import toy_experiment as ref_toy
        args.snap_dir = "/tmp"
        for comp, all_tr in [(3, False), (2, True)]:
            model.component, model.all_trained = comp, all_tr
            tag = f"toykl.c{comp}.a{int(all_tr)}."
            np.random.seed(0)   # np.random.rand() > 0.9 gate of the debug dump (toy_experiment.py:464): 0.5488 -> skipped
            torch.manual_seed(91 + comp)
            with torch.no_grad():
                losses = ref_toy.compute_kl_pq_loss(model, x, 1.0, args)
            with torch.no_grad():
                G_ll = torch.zeros(x.size(0))
                n = C if all_tr else comp
                for c in range(n):
                    if all_tr and c == comp:
                        continue
                    rs = model.rho[0:c + 1] / torch.sum(model.rho[0:c + 1])
                    if c == 0:
                        G_ll = lq32[:, 0]
                    else:
                        G_ll = torch.logsumexp(torch.stack([torch.log(1.0 - rs[c]) + G_ll, torch.log(rs[c]) + lq32[:, c]], 1), 1)
                w = ref_toy.softmax(-G_ll)
                w = w / torch.sum(w)
                clamped = bool(w.max() > 0.1)
                if clamped:
                    w = torch.max(torch.min(w, torch.tensor([0.1])), torch.tensor([0.1 / args.batch_size]))
                    w = w / torch.sum(w)
                torch.manual_seed(91 + comp)
                idx = torch.multinomial(w, x.size(0), replacement=True)
                torch.manual_seed(91 + comp)
                u = torch.rand(x.size(0), dtype=torch.float64)
            assert np.array_equal(orc.resample_indices(w.numpy(), u.numpy()), idx.numpy()), "multinomial replay mismatch"
            out[tag + "G_ll"] = G_ll.numpy(); out[tag + "w"] = w.numpy(); out[tag + "clamped"] = np.array(clamped)
            out[tag + "idx"] = idx.numpy(); out[tag + "u"] = u.numpy()
            out[tag + "batch_size"] = np.array(args.batch_size)
            for k in ("nll", "G_nll", "g_nll"):
                out[tag + k] = np.array(float(losses[k]))
        # grid density of the boosted model, geometric mixture (utils/density_plotting.py:185-226), through the reference's
        # own plotting function with recording axes (matplotlib is stubbed: only the numbers are kept)
        from utils import density_plotting as ref_plot
        ref_plot.plt.cm = types.SimpleNamespace(viridis=lambda *a, **k: None)

        class _Ax:
            def __init__(self):
                self.grids = []

            def pcolormesh(self, xx, yy, prob, cmap=None):
                self.grids.append(prob.clone())

            def set_facecolor(self, *a, **k):
                pass

            def set_title(self, *a, **k):
                pass

        class _Axs(dict):
            def __missing__(self, key):
                self[key] = _Ax()
                return self[key]

        n_pts = 12
        args.num_components = C
        model.component, model.all_trained = C - 1, False
        grid = ref_plot.setup_grid(4, n_pts, args)
        axs = _Axs()
        with torch.no_grad():
            total = ref_plot.plot_boosted_fwd_flow_density(model, axs, grid, n_pts, 50, args)
        plt_width = max(2, int(np.ceil(np.sqrt(C))))
        out["grid.n_pts"] = np.array(n_pts)
        out["grid.zz"] = grid[2].numpy()
        out["grid.total_prob"] = total.numpy()
        for c in range(C):
            out[f"grid.prob.c{c}"] = axs[(int(1 + np.floor(c / plt_width)), int(c % plt_width))].grids[0].numpy()
    path = os.path.join(out_dir or HERE, name + ".npz")
    np.savez_compressed(path, **compact(name, out))
    print(f"{name}: wrote {path} ({os.path.getsize(path) / 1024:.0f} KiB), |logq32-logq64|max = "
          f"{np.abs(lq32.numpy() - lq64.numpy()).max():.3e}")


if __name__ == "__main__":
    if not os.path.isdir(REF):
        raise SystemExit("the reference tree /root/reference is required to regenerate the fixtures")
    for n in (sys.argv[1:] or CONFIGS):
        build_case(n)
