"""Multi-objective deep GP with the reference's interface (dgp_dace/models/MO_DGP.py: `DGP_Base.propagate / predict_f / E_log_p_Y /
ELBO / predict_y / make_mf_dgp`, `MultiObjDeepGP.predict / objective / optimize_adam`): two SVGP layers, one per objective, each on
`[x, f_other(x)]` with the composite kernel `k_corr (k_prev + Linear) + k_in (+ White)`; a prediction starts from an N(0,1) column
and cycles objective 0 -> 1 -> 0 ... `loop` times before the two outputs are read (MO_DGP.py:88-122).

Kernel matrices, layer conditionals, KL and all their adjoints are the library calls of the multi-fidelity path (`composite.py`,
`MF_DGP.MFLayer`); torch.autograd chains them.

Parity: `DGP_Base.propagate / predict_f / E_log_p_Y / ELBO(tf_sample_Z_right=False)` and `EHVI`'s `mo_dgp` branch are pinned to the
reference's own code executed under tests/ref_shim (tests/golden/mo_dgp.npz, tests/golden/make_golden_mo.py). Two places of the
reference cannot execute as written, and are implemented here with the smallest change that makes them run -- both marked
DEVIATION below and unpinned:
  * `make_mf_dgp` reads `Din = Z[0].shape[1]` (MO_DGP.py:257), but `Z[0]` is layer 0's inducing input `[x, y_1]` with one column more
    than the objectives' input space (`_make_inducing_points`, :507-510), so its kernels address a column neither `Z[0]` nor the
    propagated `[x, f]` has. Here `Din = Z[-1].shape[1]` (the augmented layer's `Z_left`, which lives in the input space).
  * `sample_Z_right` (:29-35, taken over from the multi-fidelity file) gives layer 0 the bare `Z_left` although layer 0 expects
    `[x, f_1]`. Here the missing column is an N(0,1) draw, which is how `propagate` starts the same chain (:104-106).
"""
from __future__ import annotations

import functools

import numpy as np
import torch

from .. import _lib
from ..composite import RBF, LinearKernel, White
from ..gpflow_shim import Gaussian, _Module, set_trainable
from . import MF_DGP as _MF
from .MF_DGP import MFLayer, _adam_step, _weighted_kl, draw_normal, sample


def _start_column(n, device, draw, n_offset=0):
    """tf.random.normal([n, 1]) of MO_DGP.py:104: one draw per call, shared by all S samples (n_offset: as in draw_normal)."""
    return draw_normal(draw, device, (1, n, 1), n_offset).reshape(n, 1)


def sample_Z_right(layers, Z, values=None, draw=None, num_samples=50):
    """MO_DGP.py:29-35. DEVIATION (module docstring): the first application of layer 0 sees [Z, eps], eps ~ N(0, 1), instead of the
    bare Z the reference passes (which its kernel cannot evaluate); the rest is as written -- every layer of `layers` is then applied
    once to [Z, Z_right]."""
    for i, layer in enumerate(layers):
        if i == 0:
            Z_right = sample(layer, torch.cat([Z, _start_column(Z.shape[0], Z.device, draw)], 1), num_samples, values, draw)
        Z_aug = torch.cat([Z, Z_right], 1)
        Z_right = sample(layer, Z_aug, num_samples, values, draw)
    return Z_right


def init_layers_mf(Z, kernels, num_outputs=None, Layer=MFLayer, draw=None):
    """MO_DGP.py:37-56: layer 0 on the full inducing inputs Z[0], the later layers augmented (Z = [Z_left, Z_right]); the initial
    Z_right comes from 100 samples of the chain (utils/layers.py:170-177,210-213 with the DEVIATION of sample_Z_right)."""
    num_outputs = num_outputs or 1
    layers = [Layer(kernels[0], Z[0], num_outputs, None, draw=draw)]
    for i in range(1, len(Z)):
        with torch.no_grad():
            zl = _lib.as_device(np.asarray(Z[i], dtype=np.float64), layers[0].device)
            zr = sample_Z_right(layers[:i], zl, None, draw, 100)
        layers.append(Layer(kernels[i], Z[i], num_outputs, None, augmented=True, layers=layers[:i], draw=draw, Z_right=zr))
    return layers


class DGP_Base(_MF.DGP_Base):
    """MO_DGP.py:59-304."""

    def __init__(self, likelihood, layers, minibatch_size=None, num_samples=1, loop=2, draw=None, **kwargs):
        super().__init__(likelihood, layers, minibatch_size=minibatch_size, num_samples=num_samples, draw=draw, **kwargs)
        self.name = kwargs.get("name", "mo_dgp_base")
        self._train_upto_objective = -1
        self.loop = loop

    def propagate(self, X, full_cov=False, S=1, zs=None, values=None, n_offset=0):
        """MO_DGP.py:88-122 -> (Fs, Fmeans, Fvars), two entries each (objective 0, objective 1), [S, N, 1]. The chain starts from one
        N(0,1) column per point (shared by the S samples), runs layer 0, then alternates layers 1, 0, 1, 0 ... (2 loop applications;
        loop = 0: layer 1 once), reads objective 0 from the last application and objective 1 from one more application of layer 1.
        `zs[k]`, when given, is reused by every application of layer k, as in the reference. full_cov=True: Fvars are [S, N, N, 1]
        and the samples are correlated over the N points (forward only, N <= 768). n_offset: global index of X's first point (a
        data-parallel shard)."""
        if full_cov:
            _MF.check_full_cov_inputs(X, values)
        if not (isinstance(X, torch.Tensor) and X.requires_grad):      # a leaf the caller differentiates w.r.t. (EHVI_with_grad)
            X = _lib.as_device(X, self.device)
        sX = X[None].expand(S, -1, -1)
        zs = [None if z is None else _lib.as_device(z, self.device) for z in (zs or [None] * len(self.layers))]

        def apply(k, F, shared=False):
            return self.layers[k].sample_from_conditional(torch.cat([sX, F], 2), z=zs[k], values=values, draw=self.draw,
                                                          full_cov=full_cov, shared_input=shared, n_offset=n_offset)

        F = _start_column(X.shape[0], self.device, self.draw, n_offset)[None].expand(S, -1, -1)
        F, Fmean, Fvar = apply(0, F, shared=True)      # [x, start column] is the same for every sample
        if self.loop == 0:
            F, Fmean, Fvar = apply(1, F)
        else:
            for j in range(2 * self.loop):
                F, Fmean, Fvar = apply((j + 1) % 2, F)
        Fs, Fmeans, Fvars = [F], [Fmean], [Fvar]
        F, Fmean, Fvar = apply(1, F)
        Fs.append(F); Fmeans.append(Fmean); Fvars.append(Fvar)
        return Fs, Fmeans, Fvars

    def predict_f(self, X, full_cov=False, S=1, objective=None, values=None, fidelity=None, n_offset=0):
        """MO_DGP.py:124-138 (full_cov=True: the variance is [S, N, N, 1])."""
        objective = fidelity if objective is None else objective
        _, Fmeans, Fvars = self.propagate(X, full_cov=full_cov, S=S, values=values, n_offset=n_offset)
        o = -1 if objective is None else objective
        return Fmeans[o], Fvars[o]

    _likelihood_at_objective = _MF.DGP_Base._likelihood_at_fidelity      # MO_DGP.py:140-151

    def E_log_p_Y(self, X_o, Y_o, objective=None, values=None, n_offset=0):
        """MO_DGP.py:153-185: objective 1 (the last layer) uses the model's Gaussian likelihood, objective 0 the White variance of
        its kernel."""
        return super().E_log_p_Y(X_o, Y_o, objective, values, n_offset)

    def refresh_Z_right(self, values=None):
        """MO_DGP.py:192-195 (with the DEVIATION of sample_Z_right)."""
        values = values or {}
        for i in range(1, len(self.layers)):
            f = self.layers[i].feature
            if not self.layers[i].augmented:
                continue
            zl = values.get(f.Z_left, f.Z_left.value)
            f.Z_right = sample_Z_right(self.layers[0:i], zl, values, self.draw)
            f.Z = torch.cat([zl, f.Z_right], 1)

    def ELBO(self, data, tf_sample_Z_right=True, values=None, shard=None):
        """MO_DGP.py:187-216: every objective's term runs its own chain (`predict_f(objective)`); scale is identically 1 (:207-208).
        shard: as in MF_DGP.DGP_Base.ELBO (one rank's part of every objective's points)."""
        if tf_sample_Z_right:
            self.refresh_Z_right(values)
        X, Y = data
        L = 0.0
        KL = 0.0
        for objective in range(self.num_layers):
            off = 0 if shard is None else shard.offsets[objective]
            L = L + self.E_log_p_Y(X[objective], Y[objective], objective, values, n_offset=off).sum()
            KL = KL + _weighted_kl(self.layers[objective], values, shard)
        self.L, self.KL = L, KL
        return L - KL

    ELBO_closure = ELBO

    def ELBO_and_grads(self, data, params=None, tf_sample_Z_right=True, shard=None):
        """ELBO and its constrained-space gradients w.r.t. `params` (default: the trainable parameters): {Parameter: tensor}."""
        params = self.trainable_parameters if params is None else params
        values = {p: p.value.detach().clone().requires_grad_(True) for p in params}
        values[_MF.EVAL_CACHE] = {}
        elbo = self.ELBO(data, tf_sample_Z_right=tf_sample_Z_right, values=values, shard=shard)
        grads = torch.autograd.grad(elbo, [values[p] for p in params], allow_unused=True)
        self._detach_features()
        return elbo.detach(), {p: (torch.zeros_like(p.value) if g is None else g) for p, g in zip(params, grads)}

    def _detach_features(self):
        for layer in self.layers[1:]:
            if layer.augmented:
                layer.feature.Z_right = layer.feature.Z_right.detach()
                layer.feature.Z = layer.feature.Z.detach()

    def mixture_moments(self, X, S):
        """Moment-matched (mean, var) [N] of both objectives from ONE chain: EHVI.py:124-130 (`mo_dgp` branch; predict_f moments).
        The reduction over the S samples is the library's dgp_mixture_moments."""
        with torch.no_grad():
            _, Fmeans, Fvars = self.propagate(X, S=S)
        ctx = _lib.get_context(self.device)
        out = []
        for o in (-2, -1):
            fm, fv = Fmeans[o].contiguous(), Fvars[o].contiguous()
            nd = fm.shape[1] * fm.shape[2]
            mean = torch.empty(nd, dtype=torch.float64, device=self.device)
            var = torch.empty(nd, dtype=torch.float64, device=self.device)
            if nd:
                ctx.call("dgp_mixture_moments", _lib.ptr(fm), _lib.ptr(fv), int(S), int(nd), None, _lib.ptr(mean), _lib.ptr(var))
            out.append((mean, var))
        return out

    @classmethod
    def make_mf_dgp(cls, Z, loop=2, add_linear=True, minibatch_size=None, draw=None):
        """MO_DGP.py:244-292: every layer (layer 0 too) gets k_corr (k_prev + Linear) + k_in, all but the last a White(1e-6).
        DEVIATION (module docstring): Din = Z[-1].shape[1]."""
        n_objectives = len(Z)
        Din, Dout = Z[-1].shape[1], 1
        if Z[0].shape[1] != Din + Dout:
            raise ValueError(f"Z[0] must hold [x, y_other] ({Din + Dout} columns), got {Z[0].shape[1]}")
        kernels = []
        for l in range(n_objectives):
            D_range = list(range(Din + Dout))
            k_corr = RBF(active_dims=D_range[:Din], variance=1.0)
            k_prev = RBF(active_dims=D_range[Din:], variance=1.0)
            k_in = RBF(active_dims=D_range[:Din], variance=1.0)
            kernels.append(k_corr * (k_prev + LinearKernel(active_dims=D_range[Din:], variance=1.0)) + k_in if add_linear
                           else k_corr * k_prev + k_in)
        for i in range(len(kernels) - 1):
            kernels[i] = kernels[i] + White(variance=1e-6)
        layers = init_layers_mf(Z, kernels, num_outputs=Dout, draw=draw)
        return cls(Gaussian(), layers, loop=loop, num_samples=10, minibatch_size=minibatch_size, draw=draw)


class MultiObjDeepGP(_Module):
    """MO_DGP.py:306-512 (two objectives observed on the same design X[0] == X[1] rows when Z is defaulted, :507-510)."""

    def __init__(self, X, Y, Z=None, n_iter=5000, loop=2, fix_inducing=True, training=True, minibatch_size=None, draw=None):
        self.name = "mo_dgp"
        self._X = [np.asarray(x, dtype=np.float64) for x in X]
        self._Y = [np.asarray(y, dtype=np.float64) for y in Y]
        self.minibatch_size = minibatch_size
        self.loop = loop
        self.Z = self._make_inducing_points(self._X, self._Y) if Z is None else Z
        self.model = DGP_Base.make_mf_dgp(self.Z, loop=loop, minibatch_size=minibatch_size, draw=draw)
        self.n_fidelities = len(X)
        self.n_iter = n_iter
        self.fix_inducing = fix_inducing

    @staticmethod
    def _make_inducing_points(X, Y):
        """MO_DGP.py:496-512: layer 0's inducing inputs are [X[0], Y[1]], the other layers' Z_left their own inputs."""
        return [np.concatenate((X[0].copy(), Y[1].copy()), axis=1)] + [x.copy() for x in X[1:]]

    def predict(self, X_test, full_cov=False):
        """MO_DGP.py:335-340: the LAST objective, 250 samples; mean of the means, mean of the variances + variance of the means."""
        y_m, y_v = self.model.predict_y(X_test, 250, full_cov=full_cov)
        y_m, y_v = y_m.cpu().numpy(), y_v.cpu().numpy()
        return np.mean(y_m, axis=0).flatten()[:, None], (np.mean(y_v, axis=0).flatten() + np.var(y_m, axis=0).flatten())[:, None]

    def objective(self):
        with torch.no_grad():
            return self.model.ELBO((self._X, self._Y))

    def _adam_phase(self, params, state, t0, iterations, lr, epsilon, messages, tf_sample_Z_right=True, evaluate=None):
        m = self.model
        evaluate = evaluate or functools.partial(m.ELBO_and_grads, (self._X, self._Y))
        for it in range(iterations):
            elbo, grads = evaluate(params, tf_sample_Z_right=tf_sample_Z_right)
            if params:
                flat = torch.cat([grads[p].reshape(-1) for p in params])
                _adam_step(m.device, params, flat, state, t0 + it, lr, 0.9, 0.999, epsilon)
            if it % messages == 0:
                print(f"ELBO: {float(elbo)}")
        return t0 + iterations

    def optimize_adam(self, lr=0.01, iterations1=2000, iterations2=5000, iterations3=7500, messages=500, evaluate=None):
        """MO_DGP.py:344-417, as written: tf.optimizers.Adam(lr, epsilon=1e-8) shared by three phases (kernel parameters -- and, as
        written, layer 0's q_sqrt, which the reference never freezes; + inducing inputs; + variational parameters and the likelihood
        variance), Z_right re-sampled at every ELBO evaluation and once more after each phase. evaluate: callable
        `params, tf_sample_Z_right=True -> (elbo, grads)` used instead of `model.ELBO_and_grads` on this object's data (the
        data-parallel evaluation of distributed.ShardedComposite)."""
        m = self.model
        m.layers[0].q_mu.assign(self._Y[0]); set_trainable(m.layers[0].q_mu, False)
        for i, layer in enumerate(m.layers[1:]):
            layer.q_mu.assign(self._Y[i + 1]); set_trainable(layer.q_mu, False)
            layer.q_sqrt.assign(layer.q_sqrt.value * 1e-5 * self._Y[i].var()); set_trainable(layer.q_sqrt, False)
        m.layers[-1].q_sqrt.assign(m.layers[-1].q_sqrt.value * self._Y[-1].var()); set_trainable(m.layers[-1].q_sqrt, False)
        m.likelihood.likelihood.variance.assign(self._Y[-1].var() * 1e-2)
        set_trainable(m.likelihood.likelihood.variance, False)
        set_trainable(m.layers[0].feature.Z, False)
        for layer in m.layers[1:]:
            set_trainable(layer.feature.Z_left, False)
        state = {}
        print('Training part 1')
        t = self._adam_phase(m.trainable_parameters, state, 1, iterations1, lr, 1e-8, messages, evaluate=evaluate)
        set_trainable(m.layers[0].feature.Z, True)
        for layer in m.layers[1:]:
            set_trainable(layer.feature.Z_left, True)
        with torch.no_grad():
            m.refresh_Z_right()
        print('Training part 2')
        t = self._adam_phase(m.trainable_parameters, state, t, iterations2, lr, 1e-8, messages, evaluate=evaluate)
        with torch.no_grad():
            m.refresh_Z_right()
        set_trainable(m.likelihood.likelihood.variance, True)
        for layer in m.layers:
            set_trainable(layer.q_mu, True); set_trainable(layer.q_sqrt, True)
        print('Training part 3')
        self._adam_phase(m.trainable_parameters, state, t, iterations3, lr, 1e-8, messages, evaluate=evaluate)
        with torch.no_grad():
            m.refresh_Z_right()
        _lib.get_context(m.device).check()

    def optimize_nat_adam(self, lr_adam=0.01, lr_gamma=0.01, iterations1=2000, iterations2=5000, iterations3=7500, messages=500,
                          evaluate=None):
        """MO_DGP.py:418-494, as written: part 1 without re-sampling Z_right (:462), start scalings 1e-2, then Adam + a natural-gradient
        step on both layers per iteration. evaluate: as in optimize_adam."""
        from .MF_DGP import nat_adam_phase
        m = self.model
        m.layers[0].q_mu.assign(self._Y[0]); set_trainable(m.layers[0].q_mu, False)
        for i, layer in enumerate(m.layers[1:]):
            layer.q_mu.assign(self._Y[i + 1]); set_trainable(layer.q_mu, False)
            layer.q_sqrt.assign(layer.q_sqrt.value * 1e-2 * self._Y[i].var()); set_trainable(layer.q_sqrt, False)
        m.layers[-1].q_sqrt.assign(m.layers[-1].q_sqrt.value * self._Y[-1].var() * 1e-2); set_trainable(m.layers[-1].q_sqrt, False)
        m.likelihood.likelihood.variance.assign(self._Y[-1].var() * 1e-2)
        set_trainable(m.likelihood.likelihood.variance, False)
        set_trainable(m.layers[0].feature.Z, False)
        for layer in m.layers[1:]:
            set_trainable(layer.feature.Z_left, False)
        state = {}
        print('Training part 1')
        t = self._adam_phase(m.trainable_parameters, state, 1, iterations1, lr_adam, 1e-8, messages, tf_sample_Z_right=False,
                             evaluate=evaluate)
        set_trainable(m.layers[0].feature.Z, True)
        for layer in m.layers[1:]:
            set_trainable(layer.feature.Z_left, True)
        print('Training part 2')
        t = self._adam_phase(m.trainable_parameters, state, t, iterations2, lr_adam, 1e-8, messages, evaluate=evaluate)
        with torch.no_grad():
            m.refresh_Z_right()
        set_trainable(m.likelihood.likelihood.variance, True)
        print('Training part 3')
        nat_adam_phase(m, (self._X, self._Y), state, t, iterations3, lr_adam, 0.9, 0.999, 1e-8, lr_gamma, list(m.layers), messages, evaluate)
        with torch.no_grad():
            m.refresh_Z_right()
        _lib.get_context(m.device).check()
