"""Multi-fidelity deep GP with embedded mapping — fidelities with DIFFERENT input spaces (dgp_dace/models/MF_DGP_EM.py,
utils/layers_red.py; BASELINE config 4, Notebooks_dgp/nb_mfdgpem.ipynb): projection layers `layers_red` map a higher fidelity's input
space into the next lower one (multi-output SVGP layers with ARD RBF kernels, trained against the nominal mappings `X_red` through a
second Gaussian likelihood), the fidelity layers see `[H_k, f_{l-1}]` with `H_k` the input projected into their own space.
Same machinery as models/MF_DGP.py: kernels, layer conditionals / KL and all adjoints are library calls chained by torch.autograd."""
from __future__ import annotations

import functools

import numpy as np
import torch

from .. import _lib
from ..composite import EVAL_CACHE, RBF, LinearKernel, White
from ..gpflow_shim import Gaussian, _Module, set_trainable
from .MF_DGP import MFLayer, _Lik, _adam_step, _weighted_kl, check_full_cov_inputs, sample


def sample_Z_right(layers, layers_red, Z, values=None, draw=None, num_samples=50):
    """MF_DGP_EM.py:38-58: project Z through the given projection layers, then through the fidelity layers (layer i >= 1 on
    [H of its own space, Z_right])."""
    H = Z
    Hs = [H]
    for layer_red in layers_red:
        H = sample(layer_red, H, num_samples, values, draw)
        Hs.append(H)
    for i, layer in enumerate(layers):
        if i == 0:
            Z_right = sample(layer, Hs[-1], num_samples, values, draw)
        else:
            Z_right = sample(layer, torch.cat([Hs[-(i + 1)], Z_right], 1), num_samples, values, draw)
    return Z_right


def projection_scale(counts, fidelity):
    """Weight n(X[l+1]) / n(X[l]) of fidelity l's projection term (MF_DGP_EM.py:283), from the point counts of the whole batch."""
    return float(counts[fidelity + 1]) / float(counts[fidelity])


def init_layers_mf(X, Z, W, kernels, kernels_red, num_outputs=None, draw=None):
    """MF_DGP_EM.py:60-85."""
    num_outputs = num_outputs or 1
    layers_red = [MFLayer(kernels_red[i - 1], W[i - 1], X[-(1 + i)].shape[1], None, draw=draw) for i in range(1, len(X))]
    L = len(layers_red)
    layers = [MFLayer(kernels[0], Z[0], num_outputs, None, draw=draw)]
    for i in range(1, len(Z)):
        layers.append(MFLayer(kernels[i], Z[i], num_outputs, None, augmented=True, layers=layers[:i], draw=draw,
                              layers_red=layers_red[L - i:]))
    return layers, layers_red


class DGP_Base(_Module):
    """MF_DGP_EM.py:88-380."""

    def __init__(self, likelihood, layers, layers_red, minibatch_size=None, num_samples=1, draw=None, **kwargs):
        self.name = kwargs.get("name", "mf_dgp_em_base")
        self.minibatch_size = minibatch_size
        self.num_samples = num_samples
        self._train_upto_fidelity = -1
        self.num_layers = len(layers)
        self.layers = layers
        self.layers_red = layers_red
        self.likelihood = _Lik(likelihood)
        self.likelihood_projection = _Lik(Gaussian())
        self.draw = draw

    @property
    def device(self):
        return self.layers[0].device

    def propagate(self, X, full_cov=False, S=1, zs=None, ws=None, fidelity_dim=None, project=False, values=None, n_offset=0):
        """MF_DGP_EM.py:120-168: X lives in the input space of fidelity `fidelity_dim` (default: the highest). full_cov=True: the
        variances (Hvars with project=True) are [S, N, N, D] and the samples are correlated over the N points (forward only,
        N <= 768). n_offset: global index of X's first point (a data-parallel shard)."""
        if full_cov:
            check_full_cov_inputs(X, values)
        X = _lib.as_device(X, self.device)
        sX = X[None].expand(S, -1, -1)
        L = len(self.layers_red)
        fidelity_dim = L if fidelity_dim is None else fidelity_dim
        zs = zs or [None] * (L + 1)
        ws = ws or [None] * L
        dev = lambda z: None if z is None else _lib.as_device(z, self.device)
        H, Hs, Hmeans, Hvars = sX, [sX], [], []
        # the first application of the chain sees X itself for every sample: the first projection layer, or layer 0 without one
        for j, (layer_red, w) in enumerate(zip(self.layers_red[L - fidelity_dim:], ws[L - fidelity_dim:])):
            H, Hmean, Hvar = layer_red.sample_from_conditional(H, z=dev(w), values=values, draw=self.draw, full_cov=full_cov,
                                                               shared_input=j == 0, n_offset=n_offset)
            Hs.append(H); Hmeans.append(Hmean); Hvars.append(Hvar)
        if project:
            return Hs, Hmeans, Hvars
        Fs, Fmeans, Fvars = [], [], []
        for i, (layer, z) in enumerate(zip(self.layers[:fidelity_dim + 1], zs[:fidelity_dim + 1])):
            inp = Hs[-1] if i == 0 else torch.cat([Hs[-(i + 1)], F], 2)
            F, Fmean, Fvar = layer.sample_from_conditional(inp, z=dev(z), values=values, draw=self.draw, full_cov=full_cov,
                                                           shared_input=i == 0 and len(Hs) == 1, n_offset=n_offset)
            Fs.append(F); Fmeans.append(Fmean); Fvars.append(Fvar)
        return Fs, Fmeans, Fvars

    def predict_f(self, X, full_cov=False, S=1, fidelity=None, fidelity_dim=None, values=None, n_offset=0):
        """`full_cov` is accepted and not passed on (so is `project`'s): both return the diagonal moments whatever it is. Whether the
        reference passes it on is not pinned by a test of the reference's own code; propagate(full_cov=True) gives the covariances."""
        _, Fmeans, Fvars = self.propagate(X, S=S, fidelity_dim=fidelity_dim, values=values, n_offset=n_offset)
        f = -1 if fidelity is None else fidelity
        return Fmeans[f], Fvars[f]

    def project(self, X, full_cov=False, S=1, fidelity=None, fidelity_dim=None, values=None, n_offset=0):
        _, Hmeans, Hvars = self.propagate(X, S=S, fidelity_dim=fidelity_dim, project=True, values=values, n_offset=n_offset)
        f = -1 if fidelity is None else fidelity
        return Hmeans[f], Hvars[f]

    @staticmethod
    def _gauss(Fmu, Fvar, Y, variance):
        return -0.5 * np.log(2 * np.pi) - 0.5 * torch.log(variance) - 0.5 * ((Y - Fmu) ** 2 + Fvar) / variance

    def E_log_p_Y(self, X_f, Y_f, fidelity=None, fidelity_dim=None, project=False, values=None, n_offset=0):
        """MF_DGP_EM.py:217-255."""
        values = values or {}
        Y = _lib.as_device(Y_f, self.device)[None]
        if project:
            Hmean, Hvar = self.project(X_f, S=self.num_samples, fidelity=fidelity, fidelity_dim=fidelity_dim, values=values,
                                       n_offset=n_offset)
            p = self.likelihood_projection.likelihood.variance
            return self._gauss(Hmean, Hvar, Y, values.get(p, p.value)).mean(0)
        Fmean, Fvar = self.predict_f(X_f, S=self.num_samples, fidelity=fidelity, fidelity_dim=fidelity_dim, values=values,
                                     n_offset=n_offset)
        p = self.likelihood.likelihood.variance if fidelity == self.num_layers - 1 else self.layers[fidelity].kern.kernels[-1].variance
        return self._gauss(Fmean, Fvar, Y, values.get(p, p.value)).mean(0)

    def refresh_Z_right(self, values=None):
        values = values or {}
        L = len(self.layers_red)
        for i in range(1, len(self.layers)):
            f = self.layers[i].feature
            zl = values.get(f.Z_left, f.Z_left.value)
            f.Z_right = sample_Z_right(self.layers[0:i], self.layers_red[L - i:], zl, values, self.draw)
            f.Z = torch.cat([zl, f.Z_right], 1)

    def ELBO(self, data, values=None, shard=None):
        """MF_DGP_EM.py:257-297, as written: the projection term of fidelity l is scaled by n(X[l+1]) / n(X[l]). shard
        (distributed.CompositeShard): `data` is one rank's part of the points (X_red[l] split as X[l+1]); data terms are partial
        sums, the projection scale uses the global point counts and every KL term is weighted by shard.kl_weight."""
        X, Y, X_red = data
        self.refresh_Z_right(values)
        Lf = KL = L_red = KL_red = 0.0
        counts = [np.shape(x)[0] for x in X] if shard is None else shard.counts
        off = [0] * len(X) if shard is None else shard.offsets
        for fidelity in range(self.num_layers):
            if self._train_upto_fidelity != -1 and fidelity > self._train_upto_fidelity:
                continue
            Lf = Lf + self.E_log_p_Y(X[fidelity], Y[fidelity], fidelity, fidelity_dim=fidelity, values=values, n_offset=off[fidelity]).sum()
            KL = KL + _weighted_kl(self.layers[fidelity], values, shard)
            if fidelity < self.num_layers - 1:
                scale = projection_scale(counts, fidelity)
                L_red = L_red + self.E_log_p_Y(X[fidelity + 1], X_red[fidelity], fidelity, fidelity_dim=fidelity + 1, project=True,
                                               values=values, n_offset=off[fidelity + 1]).sum() * scale
                KL_red = KL_red + _weighted_kl(self.layers_red[fidelity], values, shard)
        self.L, self.KL, self.L_red, self.KL_red = Lf, KL, L_red, KL_red
        return Lf + L_red - KL - KL_red

    ELBO_closure = ELBO

    def ELBO_and_grads(self, data, params=None, shard=None):
        params = self.trainable_parameters if params is None else params
        values = {p: p.value.detach().clone().requires_grad_(True) for p in params}
        values[EVAL_CACHE] = {}
        elbo = self.ELBO(data, values=values, shard=shard)
        grads = torch.autograd.grad(elbo, [values[p] for p in params], allow_unused=True)
        for layer in self.layers[1:]:
            layer.feature.Z_right = layer.feature.Z_right.detach()
            layer.feature.Z = layer.feature.Z.detach()
        return elbo.detach(), {p: (torch.zeros_like(p.value) if g is None else g) for p, g in zip(params, grads)}

    def predict_y(self, Xnew, num_samples, full_cov=False):
        with torch.no_grad():
            Fmean, Fvar = self.predict_f(Xnew, S=num_samples)
            return Fmean, Fvar + self.likelihood.likelihood.variance.value

    @classmethod
    def make_mf_dgp(cls, X, Z, W, add_linear=True, minibatch_size=None, draw=None):
        """MF_DGP_EM.py:318-365."""
        n_fidelities = len(Z)
        Din, Dout = X[0].shape[1], 1
        kernels = [RBF(active_dims=list(range(Din)), variance=1.0, lengthscales=[1.0] * Din)]
        for l in range(1, n_fidelities):
            Din = X[l].shape[1]
            D_range = list(range(Din + Dout))
            k_corr = RBF(active_dims=D_range[:Din], variance=1.0)
            k_prev = RBF(active_dims=D_range[Din:], variance=1.0)
            k_in = RBF(active_dims=D_range[:Din], variance=1.0)
            kernels.append(k_corr * (k_prev + LinearKernel(active_dims=D_range[Din:], variance=1.0)) + k_in if add_linear
                           else k_corr * k_prev + k_in)
        kernels_red = [RBF(variance=1.0, lengthscales=[1.0] * X[-(l + 1)].shape[1]) for l in range(n_fidelities - 1)]
        for i in range(len(kernels) - 1):
            kernels[i] = kernels[i] + White(variance=1e-6)
        layers, layers_red = init_layers_mf(X, Z, W, kernels, kernels_red, num_outputs=Dout, draw=draw)
        return cls(Gaussian(), layers, layers_red, num_samples=100, minibatch_size=minibatch_size, draw=draw)


class MultiFidelityDeepGP_EM(_Module):
    """MF_DGP_EM.py:376-596 (Adam schedule)."""

    def __init__(self, X, Y, X_red, Z=None, W=None, n_iter=5000, fix_inducing=True, minibatch_size=None, draw=None):
        self.name = "mf_dgp_EM"
        f64 = lambda a: np.asarray(a, dtype=np.float64)
        self._X, self._Y, self._X_red = [f64(x) for x in X], [f64(y) for y in Y], [f64(x) for x in X_red]
        self.Z = [x.copy() for x in self._X] if Z is None else Z
        self.W = ([self._X[-1].copy()] + [self._X[-(1 + i)] for i in range(1, len(X) - 1)]) if W is None else W      # :392-397
        self.model = DGP_Base.make_mf_dgp(self._X, self.Z, self.W, minibatch_size=minibatch_size, draw=draw)
        self.n_fidelities = len(X)

    def predict(self, X_test, full_cov=False):
        y_m, y_v = self.model.predict_y(X_test, 250, full_cov=full_cov)
        y_m, y_v = y_m.cpu().numpy(), y_v.cpu().numpy()
        return np.mean(y_m, axis=0).flatten()[:, None], (np.mean(y_v, axis=0).flatten() + np.var(y_m, axis=0).flatten())[:, None]

    def objective(self):
        with torch.no_grad():
            return self.model.ELBO((self._X, self._Y, self._X_red))

    def _phase(self, state, t0, iterations, lr, beta_1, beta_2, epsilon, messages, evaluate=None):
        m = self.model
        params = m.trainable_parameters
        evaluate = evaluate or functools.partial(m.ELBO_and_grads, (self._X, self._Y, self._X_red))
        for it in range(iterations):
            elbo, grads = evaluate(params)
            if params:
                _adam_step(m.device, params, torch.cat([grads[p].reshape(-1) for p in params]), state, t0 + it, lr, beta_1, beta_2, epsilon)
            if it % messages == 0:
                print(f"ELBO: {float(elbo)}")
        return t0 + iterations

    def optimize_adam(self, lr=0.01, iterations1=2000, iterations2=5000, iterations3=7500, beta_1=0.9, beta_2=0.999, epsilon=1e-07,
                      messages=500, evaluate=None):
        """MF_DGP_EM.py:417-480. evaluate: callable `params -> (elbo, grads)` used instead of `model.ELBO_and_grads` on this object's
        data (the data-parallel evaluation of distributed.ShardedComposite)."""
        m = self.model
        for i, layer in enumerate(m.layers[:-1]):
            layer.q_mu.assign(self._Y[i]); set_trainable(layer.q_mu, False)
            layer.q_sqrt.assign(layer.q_sqrt.value * 1e-2 * self._Y[i].var()); set_trainable(layer.q_sqrt, False)
        m.layers[-1].q_sqrt.assign(m.layers[-1].q_sqrt.value * self._Y[-1].var() * 1e-2)
        set_trainable(m.layers[-1].q_sqrt, False); set_trainable(m.layers[-1].q_mu, False)
        m.layers[-1].q_mu.assign(self._Y[-1])
        for i, layer in enumerate(m.layers_red):
            layer.q_sqrt.assign(layer.q_sqrt.value * 1e-2); set_trainable(layer.q_sqrt, False)
            layer.q_mu.assign(self._X_red[-(i + 1)]); set_trainable(layer.q_mu, False)
        m.likelihood.likelihood.variance.assign(self._Y[-1].var() * 1e-2)
        set_trainable(m.likelihood.likelihood.variance, False)
        set_trainable(m.layers[0].feature.Z, False)
        for layer in m.layers[1:]:
            set_trainable(layer.feature.Z_left, False)
        state = {}
        t = self._phase(state, 1, iterations1, lr, beta_1, beta_2, epsilon, messages, evaluate)
        set_trainable(m.layers[0].feature.Z, True)
        for layer in m.layers[1:]:
            set_trainable(layer.feature.Z_left, True)
        t = self._phase(state, t, iterations2, lr, beta_1, beta_2, epsilon, messages, evaluate)
        set_trainable(m.likelihood.likelihood.variance, True)
        for layer in m.layers:
            set_trainable(layer.q_mu, True); set_trainable(layer.q_sqrt, True)
        self._phase(state, t, iterations3, lr, beta_1, beta_2, epsilon, messages, evaluate)
        with torch.no_grad():
            m.refresh_Z_right()

    def optimize_nat_adam(self, lr_adam=0.01, lr_gamma=0.01, iterations1=2000, iterations2=5000, iterations3=7500, beta_1=0.9, beta_2=0.999,
                          epsilon=1e-07, messages=500, evaluate=None):
        """MF_DGP_EM.py:501-582, as written: start scalings 1e-3 / 1e-5, the likelihood variances stay frozen in part 3 (:563), the
        natural-gradient step covers the fidelity layers and the projection layers (:564-565). evaluate: as in optimize_adam."""
        from .MF_DGP import nat_adam_phase
        m = self.model
        data = (self._X, self._Y, self._X_red)
        for i, layer in enumerate(m.layers[:-1]):
            layer.q_mu.assign(self._Y[i]); set_trainable(layer.q_mu, False)
            layer.q_sqrt.assign(layer.q_sqrt.value * 1e-3 * self._Y[i].var()); set_trainable(layer.q_sqrt, False)
        m.layers[-1].q_sqrt.assign(m.layers[-1].q_sqrt.value * self._Y[-1].var() * 1e-3)
        set_trainable(m.layers[-1].q_sqrt, False); set_trainable(m.layers[-1].q_mu, False)
        m.layers[-1].q_mu.assign(self._Y[-1])
        for i, layer in enumerate(m.layers_red):
            layer.q_sqrt.assign(layer.q_sqrt.value * 1e-5); set_trainable(layer.q_sqrt, False)
            layer.q_mu.assign(self._X_red[-(i + 1)]); set_trainable(layer.q_mu, False)
        m.likelihood_projection.likelihood.variance.assign(self._X_red[-1].var() * 1e-3)
        set_trainable(m.likelihood_projection.likelihood.variance, False)
        m.likelihood.likelihood.variance.assign(self._Y[-1].var() * 1e-3)
        set_trainable(m.likelihood.likelihood.variance, False)
        set_trainable(m.layers[0].feature.Z, False)
        for layer in m.layers[1:]:
            set_trainable(layer.feature.Z_left, False)
        state = {}
        t = self._phase(state, 1, iterations1, lr_adam, beta_1, beta_2, epsilon, messages, evaluate)
        set_trainable(m.layers[0].feature.Z, True)
        for layer in m.layers[1:]:
            set_trainable(layer.feature.Z_left, True)
        t = self._phase(state, t, iterations2, lr_adam, beta_1, beta_2, epsilon, messages, evaluate)
        with torch.no_grad():
            m.refresh_Z_right()
        nat_adam_phase(m, data, state, t, iterations3, lr_adam, beta_1, beta_2, epsilon, lr_gamma, list(m.layers) + list(m.layers_red), messages,
                       evaluate)
        with torch.no_grad():
            m.refresh_Z_right()
        _lib.get_context(m.device).check()
