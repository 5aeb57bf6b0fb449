"""Multi-fidelity deep GP with the reference's interface (dgp_dace/models/MF_DGP.py: `DGP_Base.make_mf_dgp`, `propagate`,
`predict_f`, `E_log_p_Y`, `ELBO`, `predict_y`; `MultiFidelityDeepGP.predict / objective / optimize_adam`): fidelity l's layer sees
`[x, f_{l-1}(x)]`, its kernel is `k_corr (k_prev + Linear) + k_in (+ White)` with `active_dims`, and its inducing inputs are
`Z = [Z_left, Z_right]` with `Z_right` re-sampled through the earlier layers (and differentiated through) at every ELBO evaluation
(MF_DGP.py:32-44,199-207).

Kernel matrices, their adjoints, the layer conditionals / KL and their adjoints are library calls (`composite.py`); torch.autograd
chains them. The reference needs a locally patched GPflow `InducingPoints(layers=…, Z=…)` that is not in its repository; assumed
semantics (from the call sites utils/layers.py:208-213, MF_DGP.py:204-207,375-377): `Z_left` is the trainable parameter, `Z_right`
/ `Z` are plain tensors the model overwrites.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from .. import _lib
from ..composite import (EVAL_CACHE, RBF, CompositeKernelEval, LinearKernel, PrepCache, SVGPFromK, White, stash_budget_bytes,
                         svgp_from_k_full_cov)
from ..gpflow_shim import DEFAULT_JITTER, Gaussian, Parameter, _Module, set_trainable


class _Feature(_Module):
    pass


class MFLayer(_Module):
    """SVGP_Layer(kern, Z, num_outputs, Zero(), augmented=…, layers=…) of utils/layers.py:180-224 for composite kernels."""

    def __init__(self, kern, Z, num_outputs, mean_function=None, augmented=False, layers=None, draw=None, layers_red=None,
                 Z_right=None):
        Z = np.asarray(Z.numpy() if hasattr(Z, "numpy") else Z, dtype=np.float64)
        self.kern = kern
        self.num_outputs = int(num_outputs)
        self.num_inducing = Z.shape[0]
        self.augmented = bool(augmented)
        self.white = False
        self.feature = _Feature()
        self.q_mu = Parameter(np.zeros((self.num_inducing, self.num_outputs)), name="q_mu")
        if not augmented:
            self.feature.Z = Parameter(Z, name="Z")
            Zfull = self.feature.Z.value
        else:
            self.feature.Z_left = Parameter(Z, name="Z_left")
            with torch.no_grad():      # utils/layers.py:210-213: 100 propagated samples of Z_left through the earlier layers
                if Z_right is not None:      # supplied by the caller (MO_DGP.py: the multi-objective chain samples it its own way)
                    self.feature.Z_right = Z_right
                elif layers_red is None:
                    self.feature.Z_right = sample_Z_right_array_all_layers(layers, self.feature.Z_left.value, 100, draw)
                else:      # embedded mapping: Z_left lives in this fidelity's input space (utils/layers_red.py:110-129)
                    from .MF_DGP_EM import sample_Z_right as _szr_em
                    self.feature.Z_right = _szr_em(layers, layers_red, self.feature.Z_left.value, None, draw, 100)
            self.feature.Z = torch.cat([self.feature.Z_left.value, self.feature.Z_right], 1)
            Zfull = self.feature.Z
        self.D = Zfull.shape[1]
        self.eval = CompositeKernelEval(kern, self.D)
        with torch.no_grad():          # q(u) initialised to the prior (:219-223)
            Ku = self.eval.K(Zfull) + DEFAULT_JITTER * torch.eye(self.num_inducing, dtype=torch.float64, device=Zfull.device)
            Lu = _chol(Ku)
        self.q_sqrt = Parameter(Lu[None].repeat(self.num_outputs, 1, 1), transform="triangular", name="q_sqrt")

    @property
    def device(self):
        return self.q_mu.value.device

    def Zfull(self, values):
        if not self.augmented:
            return values.get(self.feature.Z, self.feature.Z.value)
        return self.feature.Z

    def conditional_ND(self, X, values=None):
        """(mean, var [P, D_out], kl) -- utils/layers.py:237-278 + :280-308, white = False, Zero mean function. Extra input columns
        beyond the kernel's are ignored, as GPflow's active_dims slicing does (MF_DGP.py:42-43 feeds layer 0 augmented inputs)."""
        values = values or {}
        if X.shape[1] < self.D:
            raise ValueError(f"the layer's kernel addresses {self.D} input columns, got {X.shape[1]}")
        X = X[:, :self.D]
        Z = self.Zfull(values)
        M = self.num_inducing
        # one ELBO evaluation applies a layer several times with the same inducing inputs and q(u): Kuu + jitter I (one autograd node
        # whose adjoint collects every use) and the library's factorisation / M^3 products / KL are then shared (PrepCache)
        shared = values.get(EVAL_CACHE)
        ent = None if shared is None else shared.get((id(self), id(Z)))
        if ent is None:
            Ku = self.eval.K(Z, None, values) + DEFAULT_JITTER * torch.eye(M, dtype=torch.float64, device=X.device)
            ent = {"Z": Z, "Ku": Ku, "prep": None if shared is None else PrepCache(M, self.num_outputs, X.device)}
            if shared is not None:
                shared[(id(self), id(Z))] = ent       # holds Z: its id stays unique while the entry lives
                ent["prep"].budget = shared.setdefault("_stash_budget", [stash_budget_bytes()])
        Kuf = self.eval.K(Z, X.contiguous(), values)
        Kdiag = self.eval.K_diag(X.contiguous(), values)
        return SVGPFromK.apply(ent["Ku"], Kuf, Kdiag, values.get(self.q_mu, self.q_mu.value), values.get(self.q_sqrt, self.q_sqrt.value),
                               ent["prep"])

    def sample_from_conditional(self, X, z=None, values=None, draw=None, full_cov=False, shared_input=False):
        """utils/layers.py:87-130: X [S, N, D] -> samples, mean [S, N, D_out], var [S, N, D_out] (full_cov=True: [S, N, N, D_out]).
        shared_input: every sample's input is X[0] (the first application of a chain), so K(X_s, X_s) is one shared block."""
        if full_cov:
            return self._sample_full_cov(X, z, values, draw, shared_input)
        S, N, D = X.shape
        mean, var, _ = self.conditional_ND(X.reshape(S * N, D), values)
        mean, var = mean.reshape(S, N, self.num_outputs), var.reshape(S, N, self.num_outputs)
        if z is None:
            z = (draw or _default_draw(self.device))((S, N, self.num_outputs))
        return mean + z * torch.sqrt(var + DEFAULT_JITTER), mean, var

    def _sample_full_cov(self, X, z, values, draw, shared_input):
        """conditional_SND(full_cov=True) + reparameterize(full_cov=True) (utils/layers.py:76-80,264-268,276; utils/utils.py:43-52):
        per sample the N x N covariance and a correlated draw, one dgp_svgp_from_k_full_cov call. Forward only. The draws are one
        `draw((S, N, D_out))`, as on the diagonal path, so seeds and recorded draws line up across the two modes."""
        values = values or {}
        S, N, D = X.shape
        if D < self.D:
            raise ValueError(f"the layer's kernel addresses {self.D} input columns, got {D}")
        Xk = X[:, :, :self.D]
        Z = self.Zfull(values)
        Ku = self.eval.K(Z, None, values) + DEFAULT_JITTER * torch.eye(self.num_inducing, dtype=torch.float64, device=X.device)
        Kuf = self.eval.K(Z, Xk.reshape(S * N, self.D).contiguous(), values)
        Kff = self.eval.K_blocks(Xk[:1] if shared_input else Xk, values)
        if z is None:
            z = (draw or _default_draw(self.device))((S, N, self.num_outputs))
        z = z.expand(S, N, self.num_outputs)
        return svgp_from_k_full_cov(Ku, Kuf, Kff, values.get(self.q_mu, self.q_mu.value), values.get(self.q_sqrt, self.q_sqrt.value), z,
                                    DEFAULT_JITTER)

    def KL(self, values=None):
        """utils/layers.py:280-308 (one dummy point: the KL needs Ku and q only)."""
        values = values or {}
        Z = self.Zfull(values)
        return self.conditional_ND(Z[:1].detach(), values)[2]


def check_full_cov_inputs(X, values):
    """The full_cov=True path has no adjoint: refuse inputs that ask for one rather than return a silently detached result."""
    leaves = [X] + [v for v in (values or {}).values() if isinstance(v, torch.Tensor)]
    if any(isinstance(t, torch.Tensor) and t.requires_grad for t in leaves):
        raise NotImplementedError("full_cov=True has no adjoint: X and the tensors in `values` must not require grad")


def _chol(K):
    """Cholesky through the library (dgp_svgp_from_k's factorisation is internal; this is constructor-time only)."""
    return torch.linalg.cholesky(K)


class _PhiloxDraws:
    """Default source of N(0, 1) draws: the library's Philox stream (dgp_philox_normal), one stream index per call."""

    def __init__(self, device, seed=0):
        self.device, self.seed, self.calls = device, seed, 0

    def __call__(self, shape):
        S, N, D = shape
        z = torch.empty(shape, dtype=torch.float64, device=self.device)
        _lib.get_context(self.device).call("dgp_philox_normal", int(self.seed), int(self.calls), S, N, D, 0, _lib.ptr(z))
        self.calls += 1
        return z


_draws = {}


def _default_draw(device):
    if device not in _draws:
        _draws[device] = _PhiloxDraws(device)
    return _draws[device]


def sample(layer, Z, num_samples=50, values=None, draw=None):
    """MF_DGP.py:33-35."""
    Zs = Z[None].expand(num_samples, -1, -1)
    return layer.sample_from_conditional(Zs, values=values, draw=draw)[0].mean(0)


def sample_Z_right(layers, Z, values=None, draw=None):
    """MF_DGP.py:38-44, as written: the first layer is applied twice (the second time on the augmented input, whose extra column its
    kernel ignores), every later layer once on [Z, Z_right]."""
    for i, layer in enumerate(layers):
        if i == 0:
            Z_right = sample(layer, Z, 50, values, draw)
        Z_aug = torch.cat([Z, Z_right], 1)
        Z_right = sample(layer, Z_aug, 50, values, draw)
    return Z_right


def sample_Z_right_array_all_layers(layers, Z, S, draw=None):
    """utils/layers.py:170-177 (constructor-time initial Z_right)."""
    for i, layer in enumerate(layers):
        Z_right = sample(layer, Z if i == 0 else torch.cat([Z, Z_right], 1), S, None, draw)
    return Z_right


def init_layers_mf(Z, kernels, num_outputs=None, Layer=MFLayer, draw=None):
    """MF_DGP.py:46-64."""
    num_outputs = num_outputs or 1
    layers = [Layer(kernels[0], Z[0], num_outputs, None, draw=draw)]
    for i in range(1, len(Z)):
        layers.append(Layer(kernels[i], Z[i], num_outputs, None, augmented=True, layers=layers[:i], draw=draw))
    return layers


class DGP_Base(_Module):
    """MF_DGP.py:67-304."""

    def __init__(self, likelihood, layers, minibatch_size=None, num_samples=1, draw=None, **kwargs):
        self.name = kwargs.get("name", "mf_dgp_base")
        self.minibatch_size = minibatch_size
        self.num_samples = num_samples
        self._train_upto_fidelity = -1
        self.num_layers = len(layers)
        self.layers = layers
        self.likelihood = _Lik(likelihood)
        self.draw = draw

    @property
    def device(self):
        return self.layers[0].device

    def propagate(self, X, full_cov=False, S=1, zs=None, values=None):
        """MF_DGP.py:98-132: layer l >= 1 sees the input augmented with the previous layer's sample. full_cov=True: Fvars[l] is
        [S, N, N, D_l] and the samples are correlated over the N points (forward only, N <= 768)."""
        if full_cov:
            check_full_cov_inputs(X, values)
        X = _lib.as_device(X, self.device)
        sX = X[None].expand(S, -1, -1)
        Fs, Fmeans, Fvars = [], [], []
        F = sX
        zs = zs or [None] * len(self.layers)
        for i, (layer, z) in enumerate(zip(self.layers, zs)):
            inp = F if i == 0 else torch.cat([sX, F], 2)
            z = None if z is None else _lib.as_device(z, self.device)
            F, Fmean, Fvar = layer.sample_from_conditional(inp, z=z, values=values, draw=self.draw, full_cov=full_cov, shared_input=i == 0)
            Fs.append(F); Fmeans.append(Fmean); Fvars.append(Fvar)
        return Fs, Fmeans, Fvars

    def predict_f(self, X, full_cov=False, S=1, fidelity=None, values=None):
        """MF_DGP.py:134-149 (full_cov=True: the variance is [S, N, N, D])."""
        _, Fmeans, Fvars = self.propagate(X, full_cov=full_cov, S=S, values=values)
        f = -1 if fidelity is None else fidelity
        return Fmeans[f], Fvars[f]

    def _likelihood_at_fidelity(self, Fmu, Fvar, Y, variance):
        """MF_DGP.py:151-162."""
        return -0.5 * np.log(2 * np.pi) - 0.5 * torch.log(variance) - 0.5 * ((Y - Fmu) ** 2 + Fvar) / variance

    def E_log_p_Y(self, X_f, Y_f, fidelity=None, values=None):
        """MF_DGP.py:164-197: the last fidelity uses the model's Gaussian likelihood, the others the White variance of their kernel."""
        values = values or {}
        Fmean, Fvar = self.predict_f(X_f, S=self.num_samples, fidelity=fidelity, values=values)
        Y = _lib.as_device(Y_f, self.device)[None]
        if fidelity == self.num_layers - 1:
            p = self.likelihood.likelihood.variance
        else:
            p = self.layers[fidelity].kern.kernels[-1].variance
        return self._likelihood_at_fidelity(Fmean, Fvar, Y, values.get(p, p.value)).mean(0)

    def refresh_Z_right(self, values=None):
        """MF_DGP.py:204-207: Z_right of every augmented layer re-sampled through the earlier layers; Z = [Z_left, Z_right]."""
        values = values or {}
        for i in range(1, len(self.layers)):
            f = self.layers[i].feature
            zl = values.get(f.Z_left, f.Z_left.value)
            f.Z_right = sample_Z_right(self.layers[0:i], zl, values, self.draw)
            f.Z = torch.cat([zl, f.Z_right], 1)

    def ELBO(self, data, tf_sample_Z_right=True, values=None):
        """MF_DGP.py:199-226 -> 0-d tensor (differentiable w.r.t. the leaves in `values`)."""
        if tf_sample_Z_right:
            self.refresh_Z_right(values)
        X, Y = data
        L = 0.0
        KL = 0.0
        for fidelity in range(self.num_layers):
            if self._train_upto_fidelity != -1 and fidelity > self._train_upto_fidelity:
                continue
            L = L + self.E_log_p_Y(X[fidelity], Y[fidelity], fidelity, values).sum()     # scale is identically 1 (:219-220)
            KL = KL + self.layers[fidelity].KL(values)
        self.L, self.KL = L, KL
        return L - KL

    ELBO_closure = ELBO

    def ELBO_and_grads(self, data, params=None):
        """ELBO and its constrained-space gradients w.r.t. `params` (default: the trainable parameters): {Parameter: tensor}."""
        params = self.trainable_parameters if params is None else params
        values = {p: p.value.detach().clone().requires_grad_(True) for p in params}
        values[EVAL_CACHE] = {}
        elbo = self.ELBO(data, values=values)
        grads = torch.autograd.grad(elbo, [values[p] for p in params], allow_unused=True)
        self._detach_features()
        return elbo.detach(), {p: (torch.zeros_like(p.value) if g is None else g) for p, g in zip(params, grads)}

    def _detach_features(self):
        for layer in self.layers[1:]:
            layer.feature.Z_right = layer.feature.Z_right.detach()
            layer.feature.Z = layer.feature.Z.detach()

    def predict_all_layers(self, Xnew, num_samples):
        with torch.no_grad():
            return self.propagate(Xnew, S=num_samples)

    def predict_y(self, Xnew, num_samples, full_cov=False):
        """MF_DGP.py:238-240. `full_cov` is accepted and not passed on: this returns the diagonal moments whatever it is (whether
        the reference passes it on is not pinned by a test of the reference's own code)."""
        with torch.no_grad():
            Fmean, Fvar = self.predict_f(Xnew, S=num_samples)
            return Fmean, Fvar + self.likelihood.likelihood.variance.value

    @classmethod
    def make_mf_dgp(cls, Z, add_linear=True, minibatch_size=None, draw=None):
        """MF_DGP.py:249-297."""
        n_fidelities = len(Z)
        Din, Dout = Z[0].shape[1], 1
        kernels = [RBF(active_dims=list(range(Din)), variance=1.0, lengthscales=[1.0] * Din)]
        for l in range(1, n_fidelities):
            D_range = list(range(Din + Dout))
            k_corr = RBF(active_dims=D_range[:Din], variance=1.0)
            k_prev = RBF(active_dims=D_range[Din:], variance=1.0)
            k_in = RBF(active_dims=D_range[:Din], variance=1.0)
            k_l = k_corr * (k_prev + LinearKernel(active_dims=D_range[Din:], variance=1.0)) + k_in if add_linear else k_corr * k_prev + k_in
            kernels.append(k_l)
        for i in range(len(kernels) - 1):
            kernels[i] = kernels[i] + White(variance=1e-6)
        layers = init_layers_mf(Z, kernels, num_outputs=Dout, draw=draw)
        return cls(Gaussian(), layers, num_samples=10, minibatch_size=minibatch_size, draw=draw)

    def fix_inducing_point_locations(self):
        for layer in self.layers:
            set_trainable(layer.feature.Z_left if layer.augmented else layer.feature.Z, False)


class _Lik(_Module):
    def __init__(self, likelihood):
        self.likelihood = likelihood


class MultiFidelityDeepGP(_Module):
    """MF_DGP.py:306-537."""

    def __init__(self, X, Y, Z=None, n_iter=5000, fix_inducing=True, minibatch_size=None, draw=None):
        self.name = "mf_dgp"
        self._X = [np.asarray(x, dtype=np.float64) for x in X]
        self._Y = [np.asarray(y, dtype=np.float64) for y in Y]
        self.minibatch_size = minibatch_size
        self.Z = [x.copy() for x in self._X] if Z is None else Z          # :521-537
        self.model = DGP_Base.make_mf_dgp(self.Z, minibatch_size=minibatch_size, draw=draw)
        self.n_fidelities = len(X)
        self.n_iter = n_iter
        self.fix_inducing = fix_inducing

    def predict(self, X_test, full_cov=False):
        """MF_DGP.py:336-341: 250 samples; mean of the means, mean of the variances + variance of the means."""
        y_m, y_v = self.model.predict_y(X_test, 250, full_cov=full_cov)
        y_m, y_v = y_m.cpu().numpy(), y_v.cpu().numpy()
        return np.mean(y_m, axis=0).flatten()[:, None], (np.mean(y_v, axis=0).flatten() + np.var(y_m, axis=0).flatten())[:, None]

    def objective(self):
        with torch.no_grad():
            return self.model.ELBO((self._X, self._Y))

    def _adam_phase(self, params, state, t0, iterations, lr, beta_1, beta_2, epsilon, messages):
        """One phase of the reference's loops (:381-388): ELBO + gradients through the library calls, then the library's fused Adam
        launch (dgp_adam_step with the GPflow bijectors) on a flat gradient buffer."""
        m = self.model
        for it in range(iterations):
            elbo, grads = m.ELBO_and_grads((self._X, self._Y), params)
            flat = torch.cat([grads[p].reshape(-1) for p in params]) if params else torch.zeros(1, dtype=torch.float64, device=m.device)
            if params:
                _adam_step(m.device, params, flat, state, t0 + it, lr, beta_1, beta_2, epsilon)
            if it % messages == 0:
                print(f"ELBO: {float(elbo)}")
        return t0 + iterations

    def optimize_adam(self, lr=0.01, iterations1=2000, iterations2=5000, iterations3=7500, beta_1=0.9, beta_2=0.999, epsilon=1e-07,
                      messages=500):
        """MF_DGP.py:345-424: three phases (kernel parameters; + inducing inputs; + variational parameters and likelihood variance)."""
        m = self.model
        for i, layer in enumerate(m.layers[:-1]):
            layer.q_mu.assign(self._Y[i]); set_trainable(layer.q_mu, False)
            layer.q_sqrt.assign(layer.q_sqrt.value * 1e-2 * self._Y[i].var()); set_trainable(layer.q_sqrt, False)
        m.layers[-1].q_sqrt.assign(m.layers[-1].q_sqrt.value * self._Y[-1].var() * 1e-2)
        set_trainable(m.layers[-1].q_sqrt, False); set_trainable(m.layers[-1].q_mu, False)
        m.layers[-1].q_mu.assign(self._Y[-1])
        m.likelihood.likelihood.variance.assign(self._Y[-1].var() * 1e-2)
        set_trainable(m.likelihood.likelihood.variance, False)
        set_trainable(m.layers[0].feature.Z, False)
        for layer in m.layers[1:]:
            set_trainable(layer.feature.Z_left, False)
        state = {}        # per-parameter (m, v) of tf.optimizers.Adam: ONE optimiser serves the three phases (:360)
        print('Training part 1')
        t = self._adam_phase(m.trainable_parameters, state, 1, iterations1, lr, beta_1, beta_2, epsilon, messages)
        set_trainable(m.layers[0].feature.Z, True)
        for layer in m.layers[1:]:
            set_trainable(layer.feature.Z_left, True)
        print('Training part 2')
        t = self._adam_phase(m.trainable_parameters, state, t, iterations2, lr, beta_1, beta_2, epsilon, messages)
        set_trainable(m.likelihood.likelihood.variance, True)
        for layer in m.layers:
            set_trainable(layer.q_mu, True); set_trainable(layer.q_sqrt, True)
        print('Training part 3')
        self._adam_phase(m.trainable_parameters, state, t, iterations3, lr, beta_1, beta_2, epsilon, messages)
        with torch.no_grad():
            m.refresh_Z_right()


    def optimize_nat_adam(self, lr_adam=0.01, lr_gamma=0.01, iterations1=2000, iterations2=5000, iterations3=7500, beta_1=0.9, beta_2=0.999,
                          epsilon=1e-07, messages=500):
        """MF_DGP.py:426-512: Adam on the kernel parameters; + inducing inputs; then per iteration an Adam step on those and the
        likelihood variance plus a natural-gradient step on every layer's (q_mu, q_sqrt) (two ELBO evaluations per iteration)."""
        m = self.model
        data = (self._X, self._Y)
        for i, layer in enumerate(m.layers[:-1]):
            layer.q_mu.assign(self._Y[i]); set_trainable(layer.q_mu, False)
            layer.q_sqrt.assign(layer.q_sqrt.value * 1e-2 * self._Y[i].var()); set_trainable(layer.q_sqrt, False)
        m.layers[-1].q_sqrt.assign(m.layers[-1].q_sqrt.value * self._Y[-1].var() * 1e-2)
        set_trainable(m.layers[-1].q_sqrt, False); set_trainable(m.layers[-1].q_mu, False)
        m.layers[-1].q_mu.assign(self._Y[-1])
        m.likelihood.likelihood.variance.assign(self._Y[-1].var() * 1e-2)
        set_trainable(m.likelihood.likelihood.variance, False)
        set_trainable(m.layers[0].feature.Z, False)
        for layer in m.layers[1:]:
            set_trainable(layer.feature.Z_left, False)
        state = {}
        t = self._adam_phase(m.trainable_parameters, state, 1, iterations1, lr_adam, beta_1, beta_2, epsilon, messages)
        set_trainable(m.layers[0].feature.Z, True)
        for layer in m.layers[1:]:
            set_trainable(layer.feature.Z_left, True)
        t = self._adam_phase(m.trainable_parameters, state, t, iterations2, lr_adam, beta_1, beta_2, epsilon, messages)
        with torch.no_grad():
            m.refresh_Z_right()
        set_trainable(m.likelihood.likelihood.variance, True)
        nat_adam_phase(m, data, state, t, iterations3, lr_adam, beta_1, beta_2, epsilon, lr_gamma, list(m.layers), messages)
        with torch.no_grad():
            m.refresh_Z_right()
        _lib.get_context(m.device).check()


def natgrad_pairs(model, data, gamma, layers):
    """GPflow `NaturalGradient(gamma).minimize(lambda: -ELBO(data), var_list=[(q_mu, q_sqrt) of layers])` (MF_DGP.py:501-507,
    MF_DGP_EM.py, MO_DGP.py:480-487): a FRESH ELBO evaluation (new draws, Z_right re-sampled) differentiated w.r.t. the variational
    parameters through the library's layer adjoints, then one dgp_natgrad_pairs call (XiNat step, batched over layers and outputs,
    in place). Returns that evaluation's ELBO."""
    params = [p for l in layers for p in (l.q_mu, l.q_sqrt)]
    elbo, grads = model.ELBO_and_grads(data, params)
    arr = (_lib.NatPair * len(layers))()
    keep = []
    for i, l in enumerate(layers):
        gm, gs = grads[l.q_mu].contiguous(), grads[l.q_sqrt].contiguous()
        keep += [gm, gs]
        arr[i].q_mu, arr[i].q_sqrt = l.q_mu.value.data_ptr(), l.q_sqrt.value.data_ptr()
        arr[i].g_mu, arr[i].g_sqrt = gm.data_ptr(), gs.data_ptr()
        arr[i].M, arr[i].D_out = int(l.q_mu.value.shape[0]), int(l.q_mu.value.shape[1])
    _lib.get_context(model.device).call("dgp_natgrad_pairs", arr, len(layers), float(gamma))
    return elbo


def nat_adam_phase(model, data, state, t0, iterations, lr, beta_1, beta_2, epsilon, gamma, layers, messages):
    """Part 3 of the reference's optimize_nat_adam loops (MF_DGP.py:499-509): per iteration one Adam step on the trainable
    (non-variational) parameters and one natural-gradient step on `layers`, each with its own ELBO evaluation."""
    for it in range(iterations):
        params = model.trainable_parameters
        elbo, grads = model.ELBO_and_grads(data, params)
        if params:
            _adam_step(model.device, params, torch.cat([grads[p].reshape(-1) for p in params]), state, t0 + it, lr, beta_1, beta_2, epsilon)
        natgrad_pairs(model, data, gamma, layers)
        if it % messages == 0:
            print(f"ELBO: {float(elbo)}")
    return t0 + iterations


def _adam_step(device, params, flat, state, t, lr, beta_1, beta_2, epsilon):
    """dgp_adam_step (one launch, GPflow bijectors inside) on `params`, gradients concatenated in `flat` in the same order. `state`
    maps a Parameter to its (m, v) slots, so the phases of the reference's loop -- whose trainable sets differ -- share one
    optimiser state like tf's Adam does; the slots of the active parameters are gathered into the flat layout the launch expects."""
    code = {None: 0, "positive": 1, "positive_shift": 2, "triangular": 3}
    arr = (_lib.AdamParam * len(params))()
    off = 0
    for i, p in enumerate(params):
        v = p.value
        if p not in state:
            state[p] = (torch.zeros_like(v).reshape(-1), torch.zeros_like(v).reshape(-1))
        arr[i].value, arr[i].count = v.data_ptr(), v.numel()
        arr[i].grad_offset, arr[i].grad_count = off, v.numel()
        arr[i].transform, arr[i].M = code[p.transform], (v.shape[-1] if p.transform == "triangular" else 0)
        off += v.numel()
    ms = torch.cat([state[p][0] for p in params])
    vs = torch.cat([state[p][1] for p in params])
    _lib.get_context(device).call("dgp_adam_step", arr, len(params), _lib.ptr(flat), _lib.ptr(ms), _lib.ptr(vs), int(t), float(lr),
                                  float(beta_1), float(beta_2), float(epsilon))
    off = 0
    for p in params:
        n = p.value.numel()
        state[p][0].copy_(ms[off:off + n]); state[p][1].copy_(vs[off:off + n])
        off += n
