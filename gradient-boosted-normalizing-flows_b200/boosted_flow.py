"""BoostedFlow: the reference's mixture-of-flows container (models/boosted_flow.py:17-228) with the evaluation of
fixed components, the mixture, the boosting weights and the resampling served by libgbnf_b200.so.

Drop-in surface kept (SURVEY 8b): constructor `BoostedFlow(args)`, call signature
`model(x=, y_onehot=, z=, temperature=, components=int|"c"|"1:c"|"1:c-1"|"-c", reverse=False)` returning the
5-tuple `(z, z_mu, z_var, log_det_j, y_logits)`, attributes `rho / component / all_trained / num_components /
flows / args / base_dist`, methods `increment_component / update_rho / _sample_component`, state_dict keys.

New, kernel-backed entry points used by losses.py: `component_log_density`, `mixture_log_density`,
`boosting_weights`, `resample`.
"""
import ctypes as C

import torch
import torch.nn as nn
import torch.distributions as TD

from . import _lib
from .flow_modules import Glow, RealNVPFlow, rho_initial


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(None)


def _stream(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


# the fused backward's per-row kernel (train_bwd.cuh: train_bwd_rows_kernel) and the shared memory one block may use
FUSED_BACKWARD_ROWS = 16
FUSED_BACKWARD_MAX_SMEM = 227 * 1024


def fused_backward_smem_bytes(kind, D, h, K):
    """Dynamic shared memory of the fused backward's per-row kernel for a component of K steps, counted as
    train_bwd_smem_bytes (train_bwd.cuh) counts it; gbnf_component_backward refuses a component above FUSED_BACKWARD_MAX_SMEM.
    Layout: step inputs zh[K + 1][R][D] | network outputs oh[K][nets][R][64] | 3 activation rows [R][ld] | weight tiles
    [2][32][64] | 2 x [R][D], with ld = round_up(h, 64) + 4 (the |z1| <= 32 input columns of D <= 64 never widen it)."""
    R, nnets = FUSED_BACKWARD_ROWS, 1 if kind == "glow" else 2
    ld = -(-h // 64) * 64 + 4
    r4 = lambda n: (n + 3) & ~3
    return 4 * (r4((K + 1) * R * D) + K * nnets * R * 64 + 3 * R * ld + 2 * 32 * 64 + 2 * r4(R * D))


def _f32c(t):
    assert t.dtype == torch.float32 and t.is_cuda and t.is_contiguous(), "expected a contiguous CUDA float32 tensor"
    return t


class _FusedComponentFlow(torch.autograd.Function):
    """(z, log_det_j) = flows[c](x) for the component that is being TRAINED, both directions served by the library: the forward
    is the fixed-component kernel (nothing saved), the backward recomputes in-kernel and returns the gradients of every
    parameter of the component (gbnf_component_backward), and dL/dx when x requires grad.  density_experiment.py:647-661 +
    loss.backward() :361."""

    @staticmethod
    def forward(ctx, model, c, x, *params):
        with torch.no_grad():
            z, ldj = model.component_forward(x, c)
        ctx.model, ctx.c, ctx.params = model, c, params
        ctx.save_for_backward(x)
        return z, ldj

    @staticmethod
    def backward(ctx, dz, dldj):
        (x,) = ctx.saved_tensors
        dz = torch.zeros_like(x) if dz is None else dz.contiguous().float()
        dldj = torch.zeros(x.shape[0], device=x.device) if dldj is None else dldj.contiguous().float()
        grads, dx = ctx.model._component_backward(ctx.c, x, dz, dldj, with_dx=ctx.needs_input_grad[2])
        return (None, None, dx) + tuple(grads[id(p)] if p.requires_grad else None for p in ctx.params)


class _FusedMixtureInverse(torch.autograd.Function):
    """(x, ldj_inv) with x[i] = flows[comp[i]]^{-1}(z[i]): the reparameterised sample of BoostedFlow.rsample, both directions
    served by the library -- the forward is gbnf_mixture_inverse (nothing saved but z and the ids), the backward recomputes
    in-kernel (gbnf_mixture_inverse_backward) and returns the gradients of every drawn component's parameters that require grad,
    and dL/dz when z requires grad.  The inverse counterpart of _FusedComponentFlow."""

    @staticmethod
    def forward(ctx, model, n_comp, z, comp, *params):
        with torch.no_grad():
            x, ldj = model.mixture_inverse(z, comp, n_comp)
        ctx.model, ctx.n_comp, ctx.params = model, n_comp, params
        ctx.save_for_backward(z, comp)
        return x, ldj

    @staticmethod
    def backward(ctx, dx, dldj):
        z, comp = ctx.saved_tensors
        model, n = ctx.model, ctx.n_comp
        dx = torch.zeros_like(z) if dx is None else dx.contiguous().float()
        dldj = torch.zeros(z.shape[0], device=z.device) if dldj is None else dldj.contiguous().float()
        trained = {c for c in range(n) if any(p.requires_grad for p in model.flows[c].parameters())}
        grads, dz = model._mixture_inverse_backward(z, comp, n, dx, dldj, trained, with_dz=ctx.needs_input_grad[2])
        return (None, None, dz, None) + tuple(grads.get(id(p)) if p.requires_grad else None for p in ctx.params)


# the inverse backward's largest batch (gbnf_mixture_inverse_backward); rsample differentiates larger ones through autograd
FUSED_INVERSE_MAX_ROWS = 1 << 22


class BoostedFlow(nn.Module):
    def __init__(self, args, gemm_mode=None):
        super().__init__()
        self.args = args
        self.num_flows = args.num_flows
        self.z_size = args.z_size
        self.density_evaluation = args.density_evaluation
        # same RNG consumption as GenerativeFlow.__init__ (models/generative_flow.py:22-23)
        self.register_buffer("base_dist_mean", torch.randn(self.z_size, device=args.device).normal_(0, 0.1))
        self.register_buffer("base_dist_var", 3.0 * torch.ones(self.z_size, device=args.device))
        self.amortized = not args.density_evaluation
        self.all_trained = False
        self.component_type = args.component_type
        self.num_components = args.num_components
        self.component = 0
        self.register_buffer("rho", rho_initial(self.num_components, args.rho_init, args.device).to(args.device))
        self.flows = nn.ModuleList()
        for c in range(self.num_components):
            if args.component_type == "realnvp":
                self.flows.append(RealNVPFlow(args, flip_init=c))
            elif args.component_type == "glow":
                self.flows.append(Glow(args))
            else:
                raise NotImplementedError("Only glow and realnvp components are currently implemented")
        # ---- kernel-side state (created lazily on first use on a CUDA device) ----
        self.gemm_mode = gemm_mode or getattr(args, "gemm_mode", "f16")
        self.toy_base = bool(getattr(args, "toy_base", False))   # toy_experiment.py uses model.base_dist
        self.fused_backward = bool(getattr(args, "fused_backward", True))   # train the new component through the library
        self._handle = None
        self._handle_device = None
        self._handle_cfg = None
        self._base_sig = None
        self._pack_sig = {}
        self._keepalive = {}

    # ------------------------------------------------------------------ reference API
    @property
    def base_dist(self):
        return TD.Normal(self.base_dist_mean, self.base_dist_var)   # models/generative_flow.py:38-42

    def increment_component(self):                                   # models/boosted_flow.py:52-59
        if self.component == self.num_components - 1:
            self.component = 0
            self.all_trained = True
        else:
            self.component = min(self.component + 1, self.num_components - 1)

    def _sample_component(self, sampling_components, u=None):
        """models/boosted_flow.py:61-96.  With `u` (a uniform in [0,1)) the draw follows the inverse-CDF contract of
        SURVEY 8c through gbnf_sample_component; without it the reference's torch.multinomial(p, 1) is used."""
        if sampling_components == "c":
            return min(self.component, self.num_components - 1)
        if sampling_components in ("1:c", "1:c-1"):
            if sampling_components == "1:c-1":
                n = self.component
            else:
                n = self.num_components if self.all_trained else self.component + 1
            n = min(max(n, 1), self.num_components)
            exclude = -1
        elif sampling_components == "-c":
            n, exclude = self.num_components, self.component
        else:
            raise ValueError("z_k can only be sampled from ['c', '1:c-1', '1:c', '-c'] (corresponding to 'new', "
                             "'fixed', or new+fixed components)")
        if u is not None:
            rho = self.rho.detach().float().cpu().contiguous()
            arr = (C.c_float * n)(*rho[:n].tolist())
            j = C.c_int32(0)
            _lib.check(_lib.load().gbnf_sample_component(arr, n, float(u), exclude, C.byref(j)))
            return int(j.value)
        p = self.rho[:n].clone().detach()
        if exclude >= 0:
            p[exclude] = 0.0
        return torch.multinomial(p / p.sum(), 1, replacement=True).item()

    def encode(self, x, y_onehot, components):
        c = self._sample_component(components) if isinstance(components, str) else components
        flow = self.flows[c]
        needs_grad = torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in flow.parameters()))
        if not flow.actnorm_ready():
            z, ldj = flow.forward_autograd(x)     # first training batch: data-dependent ActNorm initialisation (layers.py:473-486)
        elif needs_grad and self._fused_backward_ok(x):
            # component under training: forward AND backward through the library (recompute-in-kernel backward)
            z, ldj = _FusedComponentFlow.apply(self, c, x.contiguous(), *list(flow.parameters()))
        elif needs_grad:
            z, ldj = flow.forward_autograd(x)     # configurations the fused backward does not cover: the caller's autograd
        else:
            z, ldj = self.component_forward(x, c)
        zeros = x.new_zeros((x.shape[0], self.z_size))
        return z, zeros, zeros.clone(), ldj, None

    @torch.no_grad()
    def _fused_backward_ok(self, x):
        """Whether gbnf_component_backward serves this configuration.  Besides the architecture (tanh / relu networks of any
        coupling_network_depth gbnf_create accepts, h <= 512, D <= 64, no invconv, no BatchNorm), the per-row kernel keeps every
        step's input and network outputs in shared memory, so num_flows x (z_size + 64 x networks per step) must fit beside the
        h-wide activation rows: see fused_backward_smem_bytes, which does not depend on the depth.  The deepest component served
        at D = 2 / 21 / 43 / 64 is, at h = 512, K = 27 / 20 / 15 / 12 for Glow and K = 14 / 11 / 9 / 8 for RealNVP; at h = 64,
        K = 47 / 36 / 28 / 23 and 24 / 20 / 17 / 15.  Everything else trains through the caller's autograd."""
        a = self.args
        if not (self.fused_backward and x.is_cuda and x.dtype == torch.float32 and a.h_size <= 512 and self.z_size <= 64):
            return False
        if fused_backward_smem_bytes(self.component_type, self.z_size, a.h_size, a.num_flows) > FUSED_BACKWARD_MAX_SMEM:
            return False
        if self.component_type == "glow":
            return a.coupling_network in ("tanh", "relu") and getattr(a, "flow_permutation", "shuffle") != "invconv"
        # RealNVP: train-mode BatchNorm couples the rows of a batch -> those configurations stay on the caller's autograd
        return a.coupling_network in ("tanh", "relu", "mixed") and not getattr(a, "batch_norm", False)

    def _component_backward(self, c, x, dz, dldj, with_dx=False):
        """Gradients of component c's parameters for upstream (dz, dldj) through gbnf_component_backward:
        ({id(param): grad}, dL/dx if with_dx else None).  Every Linear layer of every coupling network is passed, depth + 2 per
        network at any coupling_network_depth."""
        device = x.device
        h = self.handle(device)
        keep, out = [], {}
        cp, garr = self._backward_arrays(c, device, keep, out)
        dx = torch.empty_like(x, dtype=torch.float32) if with_dx else None
        _lib.check(_lib.load().gbnf_component_backward(h, c, C.byref(cp), _ptr(x), x.shape[0], _ptr(dz), _ptr(dldj),
                                                       C.cast(garr, C.POINTER(_lib.StepGrads)), _ptr(dx), _stream(device)))
        self._keepalive[("bwd", c)] = keep
        return out, dx

    def _backward_arrays(self, c, device, keep, out, with_grads=True):
        """(gbnf_component_params, gbnf_step_grads array or None) of component c for the fused backward calls: the raw parameters
        (device copies appended to `keep`) and, with_grads, fresh gradient buffers registered in out[id(param)]."""
        steps = self._component_tensors(c)
        parr = (_lib.StepParams * len(steps))()
        garr = (_lib.StepGrads * len(steps))() if with_grads else None

        def dev(t, dtype=torch.float32):
            t = t.detach().to(device=device, dtype=dtype).contiguous()
            keep.append(t)
            return t.data_ptr()

        def grad_of(pm):
            g = torch.empty_like(pm, dtype=torch.float32, device=device).contiguous()
            out[id(pm)] = g
            return g.data_ptr()

        for k, (d, step) in enumerate(zip(steps, self.flows[c].steps())):
            sp = parr[k]
            if "an_bias" in d:
                sp.an_bias, sp.an_logs = dev(d["an_bias"].reshape(-1)), dev(d["an_logs"].reshape(-1))
                sp.perm = dev(d["perm"], torch.int64)
                if with_grads:
                    garr[k].an_bias, garr[k].an_logs = grad_of(step.actnorm.bias), grad_of(step.actnorm.logs)
            if "bn" in d:                                  # passed so that the library refuses these steps
                sp.bn_log_gamma, sp.bn_beta, sp.bn_mean, sp.bn_var = [dev(t) for t in d["bn"]]
            for n, lins in enumerate(d["nets"]):          # Glow: the block; RealNVP: t_net, s_net
                for l, lin in enumerate(lins):
                    sp.W[n][l], sp.b[n][l] = dev(lin.weight), dev(lin.bias)
                    if with_grads:
                        garr[k].W[n][l], garr[k].b[n][l] = grad_of(lin.weight), grad_of(lin.bias)
        cp = _lib.ComponentParams()
        cp.flip_init, cp.n_steps = getattr(self.flows[c], "flip_init", 0), len(steps)
        cp.steps = C.cast(parr, C.POINTER(_lib.StepParams))
        keep.append(parr)
        return cp, garr

    def _mixture_inverse_backward(self, z, comp, n_comp, dx, dldj, trained, with_dz=False):
        """Gradients through x[i] = flows[comp[i]]^{-1}(z[i]) for upstream (dx, dldj) through gbnf_mixture_inverse_backward:
        ({id(param): grad} for the components in `trained`, dL/dz if with_dz else None)."""
        device = z.device
        h = self.handle(device)
        keep, out = [], {}
        parr = (_lib.ComponentParams * n_comp)()
        gptrs = (C.POINTER(_lib.StepGrads) * n_comp)()
        for c in range(n_comp):
            parr[c], garr = self._backward_arrays(c, device, keep, out, with_grads=c in trained)
            if garr is not None:
                keep.append(garr)
                gptrs[c] = C.cast(garr, C.POINTER(_lib.StepGrads))
        dz = torch.empty_like(z) if with_dz else None
        _lib.check(_lib.load().gbnf_mixture_inverse_backward(h, parr, _ptr(z), z.shape[0], _ptr(comp), n_comp, _ptr(dx), _ptr(dldj),
                                                             gptrs, _ptr(dz), _stream(device)))
        self._keepalive["inv_bwd"] = keep
        return out, dz

    def decode(self, z, y_onehot, temperature, components):
        """x = flows[c]^{-1}(z) for ONE component c (models/boosted_flow.py:209-218; upstream's `y_onhot` keyword typo is not
        reproduced).  z = None draws sample_size rows from the prior N(0, (exp(0) * temperature)^2) as Glow.decode /
        RealNVPFlow.decode do (models/glow.py:114-116, models/realnvp.py:99-101)."""
        c = self._sample_component(components) if isinstance(components, str) else components
        if z is None:
            t = 1.0 if temperature is None else float(temperature)
            z = torch.normal(torch.zeros(self.flows[c].sample_size, self.z_size, device=self.rho.device),
                             torch.ones(self.flows[c].sample_size, self.z_size, device=self.rho.device) * t)
        return self.component_inverse(z, c)[0]

    @torch.no_grad()
    def component_inverse(self, z, c):
        """(x, log-det of the inverse map) of component c through gbnf_component_inverse."""
        z = _f32c(z)
        self.pack_component(c)
        x = torch.empty_like(z)
        ldj = torch.empty(z.shape[0], device=z.device, dtype=torch.float32)
        _lib.check(_lib.load().gbnf_component_inverse(self.handle(z.device), _ptr(z), z.shape[0], c, _ptr(x), _ptr(ldj),
                                                      _stream(z.device)))
        return x, ldj

    @torch.no_grad()
    def assign_components(self, u, n=None, exclude=-1):
        """Per-sample component ids for mixture sampling: j_i = #{k : cum_k < u_i}, cum = cumsum_fp64(rho[:n]) / sum -- the
        inverse-CDF contract of SURVEY 8c, bit-exact for given float64 uniforms (same kernel as the batch resampling)."""
        n = (self.num_components if self.all_trained else self.component + 1) if n is None else n
        p = self.rho[:n].detach().to(u.device, torch.float32).clone()
        if exclude >= 0:
            p[exclude] = 0.0
        return self.resample(p.contiguous(), u)

    @torch.no_grad()
    def sample(self, n, u=None, z=None, temperature=1.0, generator=None):
        """n draws from the boosted mixture G = sum_c rho_c q_c: every sample gets its OWN component (upstream's TODO at
        models/boosted_flow.py:210-213), z ~ N(0, temperature^2), x = f_c^{-1}(z).  Returns (x, component ids)."""
        dev = self.rho.device
        if u is None:
            u = torch.rand(n, dtype=torch.float64, device=dev, generator=generator)
        if z is None:
            z = torch.randn((n, self.z_size), device=dev, generator=generator) * float(temperature)
        n_comp = self.num_components if self.all_trained else self.component + 1
        comp = self.assign_components(u, n_comp)
        return self.mixture_inverse(z.contiguous(), comp, n_comp)[0], comp

    def rsample(self, n, u=None, z=None, temperature=1.0, generator=None, comp=None):
        """Reparameterised draws from the boosted mixture: (x, ldj_inv, comp) with x[i] = flows[comp[i]]^{-1}(z[i]) and the log-det
        of the inverse map, so that log q_c(x) = log N(z) - ldj_inv (reverse-KL / density-matching losses).  Draws u, z and the
        component ids as sample() does (comp, when given, is used instead of u).  Differentiable: gradients reach the parameters of
        every drawn component that requires grad, and z (or the temperature) when it requires grad.  Inside the fused backward's
        envelope (_fused_backward_ok) x and ldj are bitwise those of mixture_inverse and the backward runs in the library
        (gbnf_mixture_inverse_backward); elsewhere, or with args.fused_backward = False, each component's rows go through its
        inverse_autograd (the parameters' dtype, one host synchronisation for the row counts)."""
        dev = self.rho.device
        n_comp = self.num_components if self.all_trained else self.component + 1
        if comp is None:
            if u is None:
                u = torch.rand(n, dtype=torch.float64, device=dev, generator=generator)
            comp = self.assign_components(u, n_comp)
        if z is None:
            z = torch.randn((n, self.z_size), device=dev, generator=generator) * temperature
        if self._fused_backward_ok(z) and z.shape[0] <= FUSED_INVERSE_MAX_ROWS:
            params = [p for c in range(n_comp) for p in self.flows[c].parameters()]
            x, ldj = _FusedMixtureInverse.apply(self, n_comp, z.contiguous(), comp, *params)
            return x, ldj, comp
        if bool(((comp < 0) | (comp >= n_comp)).any()):
            raise ValueError(f"rsample: component ids must lie in [0, {n_comp})")
        order = torch.argsort(comp, stable=True)
        counts = torch.bincount(comp, minlength=n_comp).tolist()
        xs, ls = [], []
        for c, rows in zip(range(n_comp), torch.split(order, counts)):
            if len(rows):
                xc, lc = self.flows[c].inverse_autograd(z[rows])
                xs.append(xc)
                ls.append(lc)
        back = torch.argsort(order)
        return torch.cat(xs)[back], torch.cat(ls)[back], comp

    @torch.no_grad()
    def mixture_inverse(self, z, comp, n=None):
        """(x, log-det of the inverse map) with x[i] = flows[comp[i]]^{-1}(z[i]) through gbnf_mixture_inverse: one coupling launch
        over every component's rows, no host synchronisation (after a first call at this batch size the call allocates nothing in
        the library, so it can be captured in a CUDA graph).  comp: int64 ids in [0, n) (n defaults to every component); an id
        outside it raises at the next check_status()."""
        z = _f32c(z)
        n = self.num_components if n is None else n
        assert comp.dtype == torch.int64 and comp.is_cuda and comp.is_contiguous() and comp.shape == (z.shape[0],)
        for c in range(n):
            self.pack_component(c)
        x = torch.empty_like(z)
        ldj = torch.empty(z.shape[0], device=z.device, dtype=torch.float32)
        _lib.check(_lib.load().gbnf_mixture_inverse(self.handle(z.device), _ptr(z), z.shape[0], _ptr(comp), n, _ptr(x), _ptr(ldj),
                                                    _stream(z.device)))
        return x, ldj

    def forward(self, x=None, y_onehot=None, z=None, temperature=None, components=None, reverse=False):
        if reverse:
            return self.decode(z, y_onehot, temperature, components)
        return self.encode(x, y_onehot, components)

    # ------------------------------------------------------------------ kernel plumbing
    def _config(self, device):
        a = self.args
        cfg = _lib.Config()
        cfg.kind = _lib.KIND[self.component_type]
        cfg.D, cfg.h, cfg.K, cfg.C = self.z_size, a.h_size, a.num_flows, self.num_components
        cfg.depth = a.coupling_network_depth
        cfg.act = _lib.ACT[a.coupling_network]
        cfg.coupling = _lib.COUPLING[getattr(a, "flow_coupling", "affine")] if self.component_type == "glow" else 0
        cfg.base = _lib.BASE_DIAG_NORMAL if self.toy_base else _lib.BASE_STD_NORMAL
        cfg.gemm_mode = _lib.GEMM[self.gemm_mode]
        cfg.device = device.index if device.index is not None else torch.cuda.current_device()
        cfg.glow_invconv = 1 if (self.component_type == "glow" and getattr(a, "flow_permutation", "shuffle") == "invconv") else 0
        return cfg

    def _config_key(self):
        a = self.args
        return (self.component_type, self.z_size, a.h_size, a.num_flows, self.num_components, a.coupling_network_depth,
                a.coupling_network, getattr(a, "flow_coupling", "affine"), getattr(a, "flow_permutation", "shuffle"), self.toy_base,
                self.gemm_mode)

    def handle(self, device=None):
        device = torch.device(device) if device is not None else self.rho.device
        if device.type != "cuda":
            raise RuntimeError("the GBNF density path runs on CUDA only (there is no CPU fallback); move the model "
                               "and data to a B200")
        if self._handle is not None and self._handle_device == device and self._handle_cfg == self._config_key():
            return self._handle
        self.release()
        lib = _lib.load()
        h = C.c_void_p()
        cfg = self._config(device)
        _lib.check(lib.gbnf_create(C.byref(h), C.byref(cfg)))
        self._handle, self._handle_device = h, device
        self._handle_cfg = self._config_key()
        self._pack_sig = {}
        if self.toy_base:   # copied by the library (stream-ordered): nothing to keep alive
            m = self.base_dist_mean.detach().to(device, torch.float32).contiguous()
            s = self.base_dist_var.detach().to(device, torch.float32).contiguous()
            _lib.check(lib.gbnf_set_base(h, _ptr(m), _ptr(s), _stream(device)))
            self._base_sig = self._base_signature()
        return h

    def _base_signature(self):
        return tuple((t.data_ptr(), t._version) for t in (self.base_dist_mean, self.base_dist_var))

    def invalidate(self):
        """Forget every packed component (call after writes the version counters cannot see: `.data` edits, load())."""
        self._pack_sig = {}
        self._base_sig = None

    def check_status(self):
        """Synchronise and raise GbnfError if a kernel reported a numeric problem (a value not finite in fp16) or a
        watchdog timeout since the last check (gbnf_check_status)."""
        if self._handle is not None:
            _lib.check(_lib.load().gbnf_check_status(self._handle, _stream(self._handle_device)))

    def release(self):
        if self._handle is not None:
            _lib.load().gbnf_destroy(self._handle)
            self._handle = None
            self._pack_sig = {}

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass

    def _component_tensors(self, c):
        """Raw tensors of component c in the order gbnf_step_params wants them (+ the permutation indices that are
        NOT in the state_dict, models/layers.py:637)."""
        flow = self.flows[c]
        out = []
        for step in flow.steps():
            d = {}
            if self.component_type == "glow":
                if not step.actnorm.inited:
                    raise ValueError("In Eval mode, but ActNorm not initiated")   # models/layers.py:474-475
                d["an_bias"], d["an_logs"] = step.actnorm.bias, step.actnorm.logs
                if hasattr(step, "invconv"):
                    # the dense weight, its inverse (fp64 inversion) and dlogdet, formed from the module's factors at pack time
                    # (tiny D x D host-side algebra, off the hot path; models/layers.py:751-779)
                    with torch.no_grad():
                        w, dl = step.invconv.get_weight()
                        d["invconv"] = (w.detach().float().contiguous(),
                                        torch.linalg.inv(w.detach().double()).float().contiguous(),
                                        dl.detach().float().reshape(1).contiguous())
                else:
                    d["perm"] = step.permutation.indices
                d["nets"] = [step.block.linears()]
            else:
                t_net, s_net, bn = step[0], step[1], step[2]
                d["nets"] = [t_net.linears(), s_net.linears()]
                if bn is not None:
                    d["bn"] = (bn.log_gamma, bn.beta, bn.running_mean, bn.running_var)
            out.append(d)
        return out

    def _signature(self, c):
        sig = []
        for t in list(self.flows[c].parameters()) + list(self.flows[c].buffers()):
            sig.append((t.data_ptr(), t._version))
        if self.component_type == "glow":
            for s in self.flows[c].steps():
                if s.permutation is not None:
                    idx = s.permutation.indices
                    sig.append((id(idx), idx._version))
        return tuple(sig)

    def pack_component(self, c, force=False):
        """(Re)tile component c's parameters into the library's packed blob when they changed since the last pack."""
        device = self.rho.device
        h = self.handle(device)
        if self.toy_base and getattr(self, "_base_sig", None) != self._base_signature():
            # the toy base density lives in every component's pack: re-send it, which un-packs all components
            m = self.base_dist_mean.detach().to(device, torch.float32).contiguous()
            s = self.base_dist_var.detach().to(device, torch.float32).contiguous()
            _lib.check(_lib.load().gbnf_set_base(h, _ptr(m), _ptr(s), _stream(device)))
            self._base_sig = self._base_signature()
            self._pack_sig = {}
        sig = self._signature(c)
        if not force and self._pack_sig.get(c) == sig:
            return
        lib = _lib.load()
        steps = self._component_tensors(c)
        arr = (_lib.StepParams * len(steps))()
        keep = []

        def dev(t, dtype=torch.float32):
            t = t.detach().to(device=device, dtype=dtype).contiguous()
            keep.append(t)
            return t.data_ptr()

        for k, d in enumerate(steps):
            sp = arr[k]
            if "an_bias" in d:
                sp.an_bias, sp.an_logs = dev(d["an_bias"].reshape(-1)), dev(d["an_logs"].reshape(-1))
                if "invconv" in d:
                    sp.invconv_w, sp.invconv_winv, sp.invconv_logdet = [dev(t) for t in d["invconv"]]
                else:
                    sp.perm = dev(d["perm"], torch.int64)
            if "bn" in d:
                sp.bn_log_gamma, sp.bn_beta, sp.bn_mean, sp.bn_var = [dev(t) for t in d["bn"]]
            for n, lins in enumerate(d["nets"]):
                for l, lin in enumerate(lins):
                    sp.W[n][l] = dev(lin.weight)
                    sp.b[n][l] = dev(lin.bias)
        cp = _lib.ComponentParams()
        cp.flip_init = getattr(self.flows[c], "flip_init", 0)
        cp.n_steps = len(steps)
        cp.steps = C.cast(arr, C.POINTER(_lib.StepParams))
        _lib.check(lib.gbnf_pack_component(h, c, C.byref(cp), _stream(device)))
        self._keepalive[("pack", c)] = keep   # borrowed until the pack kernels ran (stream-ordered)
        self._pack_sig[c] = sig

    def pack_all(self, n=None, force=False):
        for c in range(self.num_components if n is None else n):
            self.pack_component(c, force)

    # ------------------------------------------------------------------ kernel-backed hot path
    @torch.no_grad()
    def component_forward(self, x, c):
        """(z, log_det_j) of component c: `flows[c](x)` (models/boosted_flow.py:220-222)."""
        x = _f32c(x)
        self.pack_component(c)
        B = x.shape[0]
        z = torch.empty_like(x)
        ldj = torch.empty(B, device=x.device, dtype=torch.float32)
        _lib.check(_lib.load().gbnf_component_logq(self.handle(x.device), _ptr(x), B, c, c + 1, None, _ptr(z), _ptr(ldj),
                                                   _stream(x.device)))
        return z, ldj

    @torch.no_grad()
    def component_log_density(self, x, c0=0, c1=None):
        """log q_c(x) for c in [c0, c1) -> [B, c1-c0]   (density_experiment.py:613-616 per component)."""
        x = _f32c(x)
        c1 = self.num_components if c1 is None else c1
        for c in range(c0, c1):
            self.pack_component(c)
        out = torch.empty((x.shape[0], c1 - c0), device=x.device, dtype=torch.float32)
        _lib.check(_lib.load().gbnf_component_logq(self.handle(x.device), _ptr(x), x.shape[0], c0, c1, _ptr(out), None, None,
                                                   _stream(x.device)))
        return out

    @torch.no_grad()
    def mixture_from_logq(self, logq, n_comp, skip_c=-1, raw_rho=False, geometric=False):
        """Mixture log-density from materialised log q_c: the logsumexp recursion (default / raw_rho), or the rho-weighted
        mean of log q_c that utils/density_plotting.py:199-226 plots for the whole model (geometric=True)."""
        logq = _f32c(logq)
        G = torch.empty(logq.shape[0], device=logq.device, dtype=torch.float32)
        rho = self.rho.detach().to(logq.device, torch.float32).contiguous()
        _lib.check(_lib.load().gbnf_mixture_logdensity(self.handle(logq.device), _ptr(logq), logq.shape[0], logq.shape[1],
                                                       n_comp, _ptr(rho), skip_c,
                                                       _lib.MIX_GEOMETRIC if geometric else
                                                       _lib.MIX_RAW_RHO if raw_rho else _lib.MIX_SIMPLEX, _ptr(G),
                                                       _stream(logq.device)))
        return G

    @torch.no_grad()
    def mixture_log_density(self, x, n_comp, skip_c=-1, raw_rho=False, return_logq=False):
        """G_ll = log sum_c rho-weights * q_c(x) over the first n_comp components in ONE fused launch
        (density_experiment.py:612-622 / :561-571; toy_experiment.py:413-432 with skip_c)."""
        x = _f32c(x)
        for c in range(n_comp):
            self.pack_component(c)
        B = x.shape[0]
        G = torch.empty(B, device=x.device, dtype=torch.float32)
        logq = torch.empty((B, n_comp), device=x.device, dtype=torch.float32) if return_logq else None
        rho = self.rho.detach().to(x.device, torch.float32).contiguous()
        _lib.check(_lib.load().gbnf_fused_eval(self.handle(x.device), _ptr(x), B, n_comp, _ptr(rho), skip_c,
                                               _lib.MIX_RAW_RHO if raw_rho else _lib.MIX_SIMPLEX, _ptr(G), _ptr(logq),
                                               _stream(x.device)))
        return (G, logq) if return_logq else G

    @torch.no_grad()
    def boosting_weights(self, G_ll, mode="density", batch_size=None, return_stats=False):
        """density_experiment.py:627-641 / toy_experiment.py:440,453-459."""
        G_ll = _f32c(G_ll)
        B = G_ll.shape[0]
        w = torch.empty_like(G_ll)
        stats = torch.zeros(4, device=G_ll.device, dtype=torch.float32)
        lo = 0.01 if mode == "density" else 0.1 / float(batch_size if batch_size is not None else B)
        _lib.check(_lib.load().gbnf_boost_weights(self.handle(G_ll.device), _ptr(G_ll), B, lo, 0.1, _lib.WEIGHTS[mode],
                                                  _ptr(w), _ptr(stats), _stream(G_ll.device)))
        return (w, stats) if return_stats else w

    @torch.no_grad()
    def resample(self, weights, u):
        """Inverse-CDF indices for float64 uniforms `u` (the contract pinning torch.multinomial, SURVEY 8c)."""
        weights = _f32c(weights)
        assert u.dtype == torch.float64 and u.is_cuda and u.is_contiguous()
        idx = torch.empty(u.shape[0], device=weights.device, dtype=torch.int64)
        _lib.check(_lib.load().gbnf_resample(self.handle(weights.device), _ptr(weights), weights.shape[0], _ptr(u),
                                             u.shape[0], _ptr(idx), _stream(weights.device)))
        return idx

    @torch.no_grad()
    def gather_rows(self, x, idx):
        x = _f32c(x)
        out = torch.empty((idx.shape[0], x.shape[1]), device=x.device, dtype=torch.float32)
        _lib.check(_lib.load().gbnf_gather_rows(self.handle(x.device), _ptr(x), x.shape[1], _ptr(idx), idx.shape[0],
                                                _ptr(out), _stream(x.device)))
        return out

    def info(self):
        inf = _lib.Info()
        _lib.check(_lib.load().gbnf_get_info(self.handle(), C.byref(inf)))
        return {n: getattr(inf, n) for n, _ in _lib.Info._fields_}

    def profile(self):
        buf = (C.c_int64 * 32)()
        _lib.check(_lib.load().gbnf_get_profile(self.handle(), buf))
        return list(buf)

    def trace(self):
        buf = (C.c_int64 * 256)()
        _lib.check(_lib.load().gbnf_get_trace(self.handle(), buf))
        return list(buf)

    # ------------------------------------------------------------------ rho update (models/boosted_flow.py:119-207)
    @torch.no_grad()
    def _rho_gradients(self, x):
        """new_ll, fixed_ll, full_ll with the RAW-rho recursion of models/boosted_flow.py:124-137."""
        n = self.component + 1
        logq = self.component_log_density(x, 0, n)
        full = self.mixture_from_logq(logq, n, raw_rho=True)
        fixed = self.mixture_from_logq(logq, n - 1, raw_rho=True) if n > 1 else torch.zeros_like(full)
        new = logq[:, n - 1].contiguous() if n > 1 else torch.zeros_like(full)
        return new, fixed, full

    def update_rho(self, data_loader):
        """Decayed-step SGD on rho[component] (models/boosted_flow.py:141-207; the upstream NameError at :185 on its
        log message is not reproduced)."""
        if self.component == 0 and not self.all_trained:
            return
        if self.args.rho_iters == 0:
            return
        self.eval()
        prev = self.rho[self.component].item()
        it = iter(data_loader)
        for batch_id in range(self.args.rho_iters):
            try:
                x, _ = next(it)
            except StopIteration:
                it = iter(data_loader)
                x, _ = next(it)
            x = x.detach().to(self.args.device)
            g_ll, G_ll, _ = self._rho_gradients(x)
            gradient = torch.mean((-g_ll) - (-G_ll)).item()
            step = self.args.rho_lr / (0.05 * batch_id + 1)
            rho = min(max(prev - step * gradient, 0.01), 100.0)
            self.rho[self.component] = rho
            dif, prev = abs(prev - rho), rho
            if batch_id > 10 and (batch_id > self.args.rho_iters or dif < 0.001):
                break
