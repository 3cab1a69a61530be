"""Host-side parameter containers for the coupling-flow components (1-D / tabular only).

These modules own the parameters under the SAME state_dict keys as the reference so checkpoints and the optimizer's
name-based parameter groups (optimization/optimizers.py:29-35) carry over:

    Glow    component c, step k : flows.{c}.flow.layers.{k}.actnorm.{bias,logs}
                                  flows.{c}.flow.layers.{k}.block.network.{0,2,4}.{weight,bias}
                                  flows.{c}.{prior_h,bounds}
    RealNVP component c, step k : flows.{c}.flow_param.{k}.{0|1}.network.{0,2,4}.{weight,bias}   (0 = t_net, 1 = s_net)
                                  flows.{c}.flow_param.{k}.2.{log_gamma,beta,running_mean,running_var,batch_mean,batch_var}
                                  flows.{c}.{base_dist_mean,base_dist_var,prior_h}

and they consume the torch RNG in the same order as the reference constructors (models/realnvp.py:18-78,
models/glow.py:13-60,230-241,265-308, models/generative_flow.py:14-35), so a model built under the same
torch.manual_seed has bit-identical initial parameters and permutations (tests/golden pins this).

Evaluation of FIXED components never runs through these modules' torch code: BoostedFlow routes it to the CUDA
library.  `forward_autograd` below exists only for the component that is currently being trained, whose loss needs
autograd (SURVEY 8 a12 / 8(f).1: its fused backward is the next row of the scope table).  `inverse_autograd` is its sampling
counterpart: x = f^{-1}(z) and the log-det of the inverse map, differentiable in the parameters and in z.  It is the fp64
reference of the library's fused inverse backward and the path BoostedFlow.rsample takes where that backward does not serve.
"""
import math

import torch
import torch.nn as nn

_ACTS = {"tanh": nn.Tanh, "relu": nn.ReLU}


class CouplingMLP(nn.Module):
    """in -> h -> (h ->)*depth -> out with one activation type; `network.{0,2,4,...}` are the Linear layers
    (reference: TanhNet / ReLUNet, models/layers.py:208-243)."""

    def __init__(self, in_dim, out_dim, hidden_dim, depth, act):
        super().__init__()
        self.act = act
        mods = [nn.Linear(in_dim, hidden_dim)]
        for _ in range(depth):
            mods += [_ACTS[act](), nn.Linear(hidden_dim, hidden_dim)]
        mods += [_ACTS[act](), nn.Linear(hidden_dim, out_dim)]
        self.network = nn.Sequential(*mods)

    def linears(self):
        return [m for m in self.network if isinstance(m, nn.Linear)]

    def forward(self, x):
        return self.network(x)


class ResidualBlock(nn.Module):
    """Pre-activation ReLU block with a skip (models/layers.py:246-274): same attribute names, same RNG draws at construction
    (two default-initialised Linears, then the second one re-drawn uniform(-1e-3, 1e-3))."""

    def __init__(self, hidden_dim):
        super().__init__()
        self.activation = nn.ReLU()
        self.linear_layers = nn.ModuleList([nn.Linear(hidden_dim, hidden_dim) for _ in range(2)])
        nn.init.uniform_(self.linear_layers[-1].weight, -1e-3, 1e-3)
        nn.init.uniform_(self.linear_layers[-1].bias, -1e-3, 1e-3)

    def forward(self, inputs):
        t = self.linear_layers[0](self.activation(inputs))
        t = self.linear_layers[1](self.activation(t))
        return inputs + t


class ResidualNet(nn.Module):
    """initial Linear -> `num_layers` residual blocks -> final Linear (models/layers.py:277-301; the s / t networks of a RealNVP
    component with args.coupling_network == 'residual', models/realnvp.py:59-60)."""

    act = "residual"

    def __init__(self, in_dim, out_dim, hidden_dim, num_layers=2):
        super().__init__()
        self.hidden_dim = hidden_dim
        self.initial_layer = nn.Linear(in_dim, hidden_dim)
        self.blocks = nn.ModuleList([ResidualBlock(hidden_dim) for _ in range(num_layers)])
        self.final_layer = nn.Linear(hidden_dim, out_dim)

    def linears(self):
        out = [self.initial_layer]
        for b in self.blocks:
            out += list(b.linear_layers)
        return out + [self.final_layer]

    def forward(self, inputs):
        t = self.initial_layer(inputs)
        for b in self.blocks:
            t = b(t)
        return self.final_layer(t)


class ActNorm1d(nn.Module):
    """Per-feature affine with data-dependent initialisation (models/layers.py:453-545)."""

    def __init__(self, num_features, scale=1.0):
        super().__init__()
        self.bias = nn.Parameter(torch.zeros(1, num_features))
        self.logs = nn.Parameter(torch.zeros(1, num_features))
        self.num_features = num_features
        self.scale = scale
        self.inited = False   # plain attribute, NOT in the state_dict (as upstream)

    @torch.no_grad()
    def initialize_parameters(self, sample):
        if not self.training:
            raise ValueError("In Eval mode, but ActNorm not initiated")
        if sample.is_cuda and sample.dtype == torch.float32 and sample.dim() == 2 and sample.shape[1] <= 256:
            # two fused column reductions in the C-ABI library (gbnf_actnorm_init)
            from . import _lib
            x = sample.detach().contiguous()
            bias = torch.empty(x.shape[1], device=x.device, dtype=torch.float32)
            logs = torch.empty_like(bias)
            with torch.cuda.device(x.device):
                _lib.check(_lib.load().gbnf_actnorm_init(x.data_ptr(), x.shape[0], x.shape[1], float(self.scale), bias.data_ptr(),
                                                         logs.data_ptr(), torch.cuda.current_stream(x.device).cuda_stream))
            self.bias.copy_(bias.view(1, -1))       # in-place under no_grad: bumps the version counter the pack cache keys on
            self.logs.copy_(logs.view(1, -1))
        else:   # CPU tensors (host-side tests): the reference's own formula
            shift = -sample.mean(dim=0, keepdim=True)
            second = ((sample + shift) ** 2).mean(dim=0, keepdim=True)
            self.bias.copy_(shift)
            self.logs.copy_(torch.log(self.scale / (second.sqrt() + 1e-6)))
        self.inited = True

    def forward(self, x, logdet):
        if not self.inited:
            self.initialize_parameters(x)
        return (x + self.bias) * torch.exp(self.logs), logdet + self.logs.sum()

    def inverse(self, y, logdet):
        """Reverse: scale then centre (models/layers.py:505-518)."""
        if not self.inited:
            raise ValueError("In Eval mode, but ActNorm not initiated")
        return y * torch.exp(-self.logs) - self.bias, logdet - self.logs.sum()


class Permute1d(nn.Module):
    """Fixed feature permutation: reversed arange, optionally shuffled (models/layers.py:633-668)."""

    def __init__(self, num_dim, shuffle):
        super().__init__()
        self.num_dim = num_dim
        self.indices = torch.arange(num_dim - 1, -1, -1, dtype=torch.long)
        if shuffle:
            self.indices = self.indices[torch.randperm(num_dim)]
        self._refresh_inverse()

    def _refresh_inverse(self):
        self.indices_inverse = torch.empty_like(self.indices)
        self.indices_inverse[self.indices] = torch.arange(self.num_dim, dtype=torch.long)

    def set_indices(self, indices):
        self.indices = indices.detach().to("cpu", torch.long).clone()
        self._refresh_inverse()

    def forward(self, x):
        return x[:, self.indices.to(x.device)]


class InvertibleConv1x1(nn.Module):
    """Glow's invertible 1x1 convolution (models/layers.py:722-796) on FEATURE VECTORS: same parameters / buffers and the same RNG
    draws as upstream's constructor (torch.qr of a random matrix, then its LU factors), same weight formula; upstream's forward
    unpacks a 4-D shape (:751) and therefore crashes on the tabular path -- here a [B, D] input is the h = w = 1 case of it:
    z = x W^T, logdet += sum(log_s) (or slogdet(weight))."""

    def __init__(self, num_dim, LU_decomposed):
        super().__init__()
        w_shape = [num_dim, num_dim]
        w_init = torch.qr(torch.randn(*w_shape))[0]
        if not LU_decomposed:
            self.weight = nn.Parameter(torch.Tensor(w_init))
        else:
            p, lower, upper = torch.lu_unpack(*torch.lu(w_init))
            s = torch.diag(upper)
            self.register_buffer("p", p)
            self.register_buffer("sign_s", torch.sign(s))
            self.lower = nn.Parameter(lower)
            self.log_s = nn.Parameter(torch.log(torch.abs(s)))
            self.upper = nn.Parameter(torch.triu(upper, 1))
            self.l_mask = torch.tril(torch.ones(w_shape), -1)
            self.eye = torch.eye(*w_shape)
        self.w_shape = w_shape
        self.LU_decomposed = LU_decomposed

    def get_weight(self):
        """(W [D, D], dlogdet) of the forward direction (models/layers.py:751-779 with h * w == 1)."""
        if not self.LU_decomposed:
            return self.weight, torch.slogdet(self.weight)[1]
        l_mask, eye = self.l_mask.to(self.lower.device), self.eye.to(self.lower.device)
        lower = self.lower * l_mask + eye
        u = self.upper * l_mask.transpose(0, 1).contiguous()
        u = u + torch.diag(self.sign_s * torch.exp(self.log_s))
        return torch.matmul(self.p, torch.matmul(lower, u)), torch.sum(self.log_s)

    def forward(self, x, logdet):
        w, dlogdet = self.get_weight()
        return x @ w.t(), logdet + dlogdet


class GlowStep(nn.Module):
    """ActNorm1d -> Permute1d | InvertibleConv1x1 -> affine/additive coupling (models/glow.py:261-342, 1-D branch)."""

    def __init__(self, dim, hidden_dim, actnorm_scale, flow_permutation, flow_coupling, coupling_network, depth, LU_decomposed=True):
        super().__init__()
        if flow_permutation not in ("shuffle", "reverse", "invconv"):
            raise NotImplementedError("flow_permutation must be 'shuffle', 'reverse' or 'invconv'")
        if coupling_network not in _ACTS:
            # upstream: 'residual' raises NameError for Glow (models/glow.py:294 uses ResidualNet without importing it), 'random' draws
            # the network type from numpy's global RNG
            raise NotImplementedError("1-D Glow coupling_network must be 'tanh' or 'relu'")
        self.flow_coupling = flow_coupling
        self.actnorm = ActNorm1d(dim, actnorm_scale)
        if flow_permutation == "invconv":
            self.invconv = InvertibleConv1x1(dim, LU_decomposed=LU_decomposed)
        elif flow_permutation == "shuffle":
            self.shuffle = Permute1d(dim, shuffle=True)
        else:
            self.reverse = Permute1d(dim, shuffle=False)
        d_in = dim // 2
        d_out = dim - d_in
        self.block = CouplingMLP(d_in, d_out * (2 if flow_coupling == "affine" else 1), hidden_dim, depth, coupling_network)

    @property
    def permutation(self):
        if hasattr(self, "invconv"):
            return None
        return self.shuffle if hasattr(self, "shuffle") else self.reverse

    def forward_autograd(self, x, logdet):
        y, logdet = self.actnorm(x, logdet)
        if hasattr(self, "invconv"):
            y, logdet = self.invconv(y, logdet)
        else:
            y = self.permutation(y)
        d_in = y.shape[1] // 2
        y1, y2 = y[:, :d_in], y[:, d_in:]
        out = self.block(y1)
        if self.flow_coupling == "additive":
            y2 = y2 + out
        else:
            gate = torch.sigmoid(out[:, 1::2] + 2.0)
            y2 = (y2 + out[:, 0::2]) * gate
            logdet = logdet + torch.log(gate).sum(dim=1)
        return torch.cat((y1, y2), dim=1), logdet

    def inverse_autograd(self, y, logdet):
        """Coupling^-1, then permutation^-1 / 1x1 convolution^-1, then ActNorm^-1 (models/glow.py:344-366)."""
        d_in = y.shape[1] // 2
        y1, y2 = y[:, :d_in], y[:, d_in:]
        out = self.block(y1)
        if self.flow_coupling == "additive":
            y2 = y2 - out
        else:
            gate = torch.sigmoid(out[:, 1::2] + 2.0)
            y2 = y2 / gate - out[:, 0::2]
            logdet = logdet - torch.log(gate).sum(dim=1)
        z = torch.cat((y1, y2), dim=1)
        if hasattr(self, "invconv"):
            w, dlogdet = self.invconv.get_weight()
            z = z @ torch.linalg.inv(w).t()
            logdet = logdet - dlogdet
        else:
            z = z[:, self.permutation.indices_inverse.to(z.device)]
        return self.actnorm.inverse(z, logdet)


class GlowNet(nn.Module):
    def __init__(self, dim, hidden_dim, K, **kw):
        super().__init__()
        self.layers = nn.ModuleList([GlowStep(dim, hidden_dim, **kw) for _ in range(K)])


class Glow(nn.Module):
    """One Glow component on feature vectors (models/glow.py:12-110, non-image branch)."""

    kind = "glow"

    def __init__(self, args):
        super().__init__()
        if len(args.input_size) != 1:
            raise NotImplementedError("only 1-D (tabular) Glow components are on this path")
        self.sample_size = args.sample_size
        self.z_size = args.z_size
        self.flow = GlowNet(args.input_size[0], args.h_size, args.num_flows, actnorm_scale=args.actnorm_scale,
                            flow_permutation=args.flow_permutation, flow_coupling=args.flow_coupling,
                            coupling_network=args.coupling_network, depth=args.coupling_network_depth,
                            LU_decomposed=getattr(args, "LU_decomposed", True))
        self.register_buffer("prior_h", torch.zeros([1, args.z_size * 2]))
        self.register_buffer("bounds", torch.tensor([0.9], dtype=torch.float32))

    def steps(self):
        return list(self.flow.layers)

    def actnorm_ready(self):
        return all(s.actnorm.inited for s in self.flow.layers)

    def set_actnorm_init(self):
        for s in self.flow.layers:
            s.actnorm.inited = True

    def forward_autograd(self, x):
        logdet = torch.zeros(x.size(0), device=x.device)
        z = x
        for s in self.flow.layers:
            z, logdet = s.forward_autograd(z, logdet)
        return z, logdet

    def inverse_autograd(self, z):
        """(x, log-det of the inverse map) = f^{-1}(z), differentiable: the steps from the last to the first."""
        logdet = torch.zeros(z.size(0), device=z.device, dtype=z.dtype)
        x = z
        for s in reversed(self.flow.layers):
            x, logdet = s.inverse_autograd(x, logdet)
        return x, logdet


class BatchNorm(nn.Module):
    """RealNVP batch norm with log-det (models/layers.py:320-372).  Kernels implement the eval-mode branch."""

    def __init__(self, input_size, momentum=0.9, eps=1e-5):
        super().__init__()
        self.momentum, self.eps = momentum, eps
        self.log_gamma = nn.Parameter(torch.zeros(input_size))
        self.beta = nn.Parameter(torch.zeros(input_size))
        self.register_buffer("running_mean", torch.zeros(input_size))
        self.register_buffer("running_var", torch.ones(input_size))
        self.register_buffer("batch_mean", torch.zeros(input_size))
        self.register_buffer("batch_var", torch.zeros(input_size))

    def forward(self, x):
        if self.training:
            self.batch_mean = x.mean(0)
            self.batch_var = x.var(0)
            self.running_mean.mul_(self.momentum).add_(self.batch_mean.data * (1 - self.momentum))
            self.running_var.mul_(self.momentum).add_(self.batch_var.data * (1 - self.momentum))
            mean, var = self.batch_mean, self.batch_var
        else:
            mean, var = self.running_mean, self.running_var
        y = self.log_gamma.exp() * ((x - mean) / torch.sqrt(var + self.eps)) + self.beta
        ladj = self.log_gamma - 0.5 * torch.log(var + self.eps)
        return y, ladj.expand_as(x).sum(dim=1)

    def inverse_eval(self, y):
        """Inverse of the eval-mode branch (running statistics, as every inverse kernel uses): (x, its log-det)."""
        sd = torch.sqrt(self.running_var + self.eps)
        x = (y - self.beta) * torch.exp(-self.log_gamma) * sd + self.running_mean
        ladj = -(self.log_gamma - 0.5 * torch.log(self.running_var + self.eps))
        return x, ladj.expand_as(x).sum(dim=1)


class RealNVPFlow(nn.Module):
    """One RealNVP component (models/realnvp.py:14-133): K steps, step k flipped iff (k + flip_init) is odd."""

    kind = "realnvp"

    def __init__(self, args, flip_init=0):
        super().__init__()
        D = args.z_size
        self.z_size, self.num_flows, self.flip_init, self.sample_size = D, args.num_flows, flip_init, args.sample_size
        # same two RNG draws as GenerativeFlow.__init__ (models/generative_flow.py:22-23)
        self.register_buffer("base_dist_mean", torch.randn(D, device=args.device).normal_(0, 0.1))
        self.register_buffer("base_dist_var", 3.0 * torch.ones(D, device=args.device))
        if args.coupling_network == "mixed":
            acts = ("relu", "tanh")                     # t_net ReLU, s_net Tanh (models/realnvp.py:47-51)
        elif args.coupling_network in _ACTS or args.coupling_network == "residual":
            acts = (args.coupling_network,) * 2
        else:
            raise NotImplementedError("coupling_network must be 'tanh', 'relu', 'residual' or 'mixed' on this path ('random' draws the "
                                      "network type from numpy's global RNG upstream)")
        self.flow_param = nn.ModuleList()
        for k in range(self.num_flows):
            flipped = ((k + flip_init) % 2) > 0
            d_in, d_out = (D - D // 2, D // 2) if flipped else (D // 2, D - D // 2)
            nets = [ResidualNet(d_in, d_out, args.h_size, args.coupling_network_depth) if a == "residual"
                    else CouplingMLP(d_in, d_out, args.h_size, args.coupling_network_depth, a) for a in acts]
            bn = BatchNorm(D) if (args.batch_norm and k < self.num_flows - 1) else None
            self.flow_param.append(nn.ModuleList(nets + [bn]))
        self.register_buffer("prior_h", torch.zeros([1, 2 * D]))

    def steps(self):
        return list(self.flow_param)

    def actnorm_ready(self):
        return True

    def forward_autograd(self, x):
        logdet = torch.zeros(x.size(0), device=x.device)
        z = x
        h0 = self.z_size // 2
        for k, (t_net, s_net, bn) in enumerate(self.flow_param):
            if bn is not None:
                z, l_bn = bn(z)
                logdet = logdet + l_bn
            if ((k + self.flip_init) % 2) > 0:
                z_b, z_a = z[:, :h0], z[:, h0:]
            else:
                z_a, z_b = z[:, :h0], z[:, h0:]
            log_s = s_net(z_a)
            z_b = t_net(z_a) + z_b * torch.exp(log_s)
            z = torch.cat([z_a, z_b], dim=1)
            logdet = logdet + log_s.sum(dim=1)
        return z, logdet

    def inverse_autograd(self, z):
        """(x, log-det of the inverse map) = f^{-1}(z), differentiable: per step from the last, coupling^-1 (the forward's
        output is [z1, z2'] for both flips) then eval-mode BatchNorm^-1."""
        logdet = torch.zeros(z.size(0), device=z.device, dtype=z.dtype)
        x = z
        h0 = self.z_size // 2
        for k in range(self.num_flows - 1, -1, -1):
            t_net, s_net, bn = self.flow_param[k]
            flipped = ((k + self.flip_init) % 2) > 0
            n1 = self.z_size - h0 if flipped else h0
            z1, z2 = x[:, :n1], x[:, n1:]
            log_s = s_net(z1)
            z2 = (z2 - t_net(z1)) * torch.exp(-log_s)
            x = torch.cat([z2, z1], dim=1) if flipped else torch.cat([z1, z2], dim=1)
            logdet = logdet - log_s.sum(dim=1)
            if bn is not None:
                x, l_bn = bn.inverse_eval(x)
                logdet = logdet + l_bn
        return x, logdet


def rho_initial(num_components, rho_init, device):
    """models/boosted_flow.py:32-39."""
    if rho_init == "decreasing":
        return torch.clamp(1.0 / torch.pow(2.0, torch.arange(num_components * 1.0, device=device)), min=0.05)
    return torch.full((num_components,), 1.0 / num_components, device=device)


LOG_2PI = math.log(2.0 * math.pi)
