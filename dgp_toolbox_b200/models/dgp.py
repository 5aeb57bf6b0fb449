"""DGP_Base / DGP with the reference's interface (dgp_dace/models/dgp.py:21-130,221-254,348-366).

propagate / predict / ELBO and the ELBO gradient run in libdgp_b200 (hand-written sm_100a CUDA behind the C ABI of
include/dgp_b200.h). The optimiser loops keep the reference's structure (dgp.py:255-345): a Python `for` around one
ELBO+gradient evaluation per step, Adam on the *unconstrained* variables exactly as tf.GradientTape sees them.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from .. import _lib
from .. import gpflow_shim as gpflow
from ..gpflow_shim import _Module
from ..utils.layer_initializations import init_layers_linear
from ..utils.utils import BroadcastingLikelihood


class DGP_Base(_Module):
    """dgp_dace/models/dgp.py:21-130."""

    def __init__(self, likelihood, layers, num_samples=1, seed=0, **kwargs):
        self.name = "dgp"
        self.num_samples = num_samples
        self.likelihood = BroadcastingLikelihood(likelihood)
        self.layers = layers
        self.seed = int(seed)        # Philox key of the in-kernel draws (replaces tf.random.normal, utils/layers.py:113)
        self._draw = 0               # advanced once per stochastic evaluation so successive steps use fresh draws

    # ------------------------------------------------------------------ plumbing
    @property
    def device(self):
        return self.layers[0].feature.Z.value.device

    @property
    def parameters(self):
        out, seen = [], set()
        for p in [q for l in self.layers for q in l.parameters] + list(self.likelihood.likelihood.parameters):
            if id(p) not in seen:          # one entry per Parameter object even when a kernel is shared between layers (GPflow semantics)
                seen.add(id(p))
                out.append(p)
        return out

    @property
    def trainable_variables(self):
        return self.trainable_parameters

    def _model_desc(self):
        keep = []
        arr = (_lib.LayerDesc * len(self.layers))()
        for i, l in enumerate(self.layers):
            d, k = l._desc()
            arr[i] = d
            keep.append(k)
        lv = self.likelihood.likelihood.variance.value.reshape(1)
        keep.append(lv)
        m = _lib.ModelDesc(len(self.layers), arr, lv.data_ptr())
        keep.append(arr)
        return m, keep

    def _check_X(self, X):
        D0 = self.layers[0].feature.Z.shape[1]
        if X.dim() != 2 or X.shape[1] != D0:
            raise ValueError(f"X has shape {tuple(X.shape)}, the first layer expects [N, {D0}]")
        return X

    def _check_XY(self, X, Y):
        self._check_X(X)
        DL = self.layers[-1].num_outputs
        if Y.dim() != 2 or tuple(Y.shape) != (X.shape[0], DL):
            raise ValueError(f"Y has shape {tuple(Y.shape)}, expected [{X.shape[0]}, {DL}]")

    def _next_seed(self, seed):
        if seed is not None:
            return int(seed)
        s = (self.seed + 0x9E3779B97F4A7C15 * self._draw) & 0xFFFFFFFFFFFFFFFF
        self._draw += 1
        return s

    def _zs(self, zs, S, N):
        if zs is None:
            return None, None
        ts = [None if z is None else _lib.as_device(z, self.device).reshape(S, N, l.num_outputs)
              for z, l in zip(zs, self.layers)]
        return ts, _lib.ptr_array(ts)

    # ------------------------------------------------------------------ a7: propagate
    def propagate(self, X, full_cov=False, S=1, zs=None, seed=None, n_offset=0, group_size=None):
        """dgp.py:34-63 -> (Fs, Fmeans, Fvars), lists of [S,N,D_l] tensors; full_cov=True draws samples correlated over the inputs
        (Fvars then [S,N,N,D_l]: utils/layers.py:76-80,264-268; utils/utils.py:43-52). With full_cov=True and group_size=q the
        N points are N/q independent groups of q consecutive points: samples are correlated within a group only, group g is what
        propagate(X[g q:(g+1) q], full_cov=True, n_offset=n_offset + g q) gives with the same seed, and Fvars[l] is
        [S, N/q, q, q, D_l] (dgp_propagate_grouped_cov: 1 <= q <= 32, no limit on N)."""
        if group_size is not None and not full_cov:
            raise ValueError("group_size needs full_cov=True")
        X = self._check_X(_lib.as_device(X, self.device))
        N = X.shape[0]
        mk = lambda: [torch.empty((S, N, l.num_outputs), dtype=torch.float64, device=X.device) for l in self.layers]
        Fs, Fmeans = mk(), mk()
        if group_size is not None:
            q = int(group_size)
            qs = max(q, 0)
            G = N // q if q > 0 else 0
            Fvars = [torch.empty((S, G, qs, qs, l.num_outputs), dtype=torch.float64, device=X.device) for l in self.layers]
        elif full_cov:
            Fvars = [torch.empty((S, N, N, l.num_outputs), dtype=torch.float64, device=X.device) for l in self.layers]
        else:
            Fvars = mk()
        if N == 0 or S == 0:
            return Fs, Fmeans, Fvars
        m, keep = self._model_desc()
        zt, zp = self._zs(zs, S, N)
        ctx = _lib.get_context(X.device)
        if group_size is not None:
            ctx.call("dgp_propagate_grouped_cov", C.byref(m), _lib.ptr(X), N, S, q, zp, self._next_seed(seed), int(n_offset),
                     _lib.ptr_array(Fs), _lib.ptr_array(Fmeans), _lib.ptr_array(Fvars))
            return Fs, Fmeans, Fvars
        ctx.call("dgp_propagate_full_cov" if full_cov else "dgp_propagate", C.byref(m), _lib.ptr(X), N, S, zp,
                 self._next_seed(seed), int(n_offset), _lib.ptr_array(Fs), _lib.ptr_array(Fmeans), _lib.ptr_array(Fvars))
        return Fs, Fmeans, Fvars

    def predict_f(self, X, full_cov=False, S=1, zs=None, seed=None, group_size=None):
        """dgp.py:66-77: last layer's mean [S,N,D_L] and variance [S,N,D_L] (full_cov=True: covariance [S,N,N,D_L]; with
        group_size=q, the [S,N/q,q,q,D_L] blocks of propagate(group_size=q))."""
        if group_size is not None and not full_cov:
            raise ValueError("group_size needs full_cov=True")
        if full_cov:
            _, Fmeans, Fvars = self.propagate(X, full_cov=True, S=S, zs=zs, seed=seed, group_size=group_size)
            return Fmeans[-1], Fvars[-1]
        X = self._check_X(_lib.as_device(X, self.device))
        N, L = X.shape[0], len(self.layers)
        D = self.layers[-1].num_outputs
        Fmean = torch.empty((S, N, D), dtype=torch.float64, device=X.device)
        Fvar = torch.empty_like(Fmean)
        if N == 0 or S == 0:
            return Fmean, Fvar
        m, keep = self._model_desc()
        zt, zp = self._zs(zs, S, N)
        _lib.get_context(X.device).call("dgp_propagate", C.byref(m), _lib.ptr(X), N, S, zp, self._next_seed(seed), 0, None,
                                        _lib.ptr_array([None] * (L - 1) + [Fmean]), _lib.ptr_array([None] * (L - 1) + [Fvar]))
        return Fmean, Fvar

    # ------------------------------------------------------------------ a8-a10: ELBO and its gradient
    def E_log_p_Y(self, X, Y, zs=None, seed=None):
        """dgp.py:79-87 -> [N, D]: one dgp_e_log_p_y call (chain + Gaussian variational expectations + mean over S in-library)."""
        X = _lib.as_device(X, self.device)
        Y = _lib.as_device(Y, self.device)
        self._check_XY(X, Y)
        N, S = X.shape[0], self.num_samples
        out = torch.empty((N, self.layers[-1].num_outputs), dtype=torch.float64, device=X.device)
        if N == 0:
            return out
        m, keep = self._model_desc()
        zt, zp = self._zs(zs, S, N)
        _lib.get_context(X.device).call("dgp_e_log_p_y", C.byref(m), _lib.ptr(X), _lib.ptr(Y), N, S, zp, self._next_seed(seed), 0,
                                        _lib.ptr(out))
        return out

    def grad_layout(self):
        m, keep = self._model_desc()
        offs = (_lib.GradOffsets * len(self.layers))()
        _lib.lib.dgp_grad_layout(C.byref(m), offs)
        return int(_lib.lib.dgp_grad_size(C.byref(m))), offs

    def elbo_flat(self, data, want_grad=True, scale=1.0, kl_weight=1.0, zs=None, seed=None, n_offset=0, out=None):
        """One dgp_elbo_grad call. Returns the flat device buffer
        [data term, kl_weight*sum KL, d/d lik_var, per layer dZ, dlengthscales, dvariance, dq_mu, dq_sqrt] (constrained space)."""
        X, Y = data
        X = _lib.as_device(X, self.device)
        Y = _lib.as_device(Y, self.device)
        self._check_XY(X, Y)
        N, S = X.shape[0], self.num_samples
        if N == 0:
            raise ValueError("empty minibatch")
        m, keep = self._model_desc()
        n = int(_lib.lib.dgp_grad_size(C.byref(m))) if want_grad else 3
        if out is None:
            out = torch.empty(n, dtype=torch.float64, device=X.device)
        zt, zp = self._zs(zs, S, N)
        _lib.get_context(X.device).call("dgp_elbo_grad", C.byref(m), _lib.ptr(X), _lib.ptr(Y), N, S, float(scale), float(kl_weight),
                                        zp, self._next_seed(seed), int(n_offset), 1 if want_grad else 0, _lib.ptr(out))
        return out

    def elbo_flat_host(self, X_host: np.ndarray, Y_host: np.ndarray, want_grad=True, scale=1.0, kl_weight=1.0, seed=None,
                       n_offset=0, out_host=None):
        """dgp_elbo_grad_host: HOST numpy in, HOST numpy out; the host<->device copies are part of the call."""
        X_host = np.ascontiguousarray(X_host, dtype=np.float64)
        Y_host = np.ascontiguousarray(Y_host, dtype=np.float64)
        self._check_XY(torch.from_numpy(X_host), torch.from_numpy(Y_host))
        m, keep = self._model_desc()
        n = int(_lib.lib.dgp_grad_size(C.byref(m))) if want_grad else 3
        if out_host is None:
            out_host = np.empty(n, dtype=np.float64)
        _lib.get_context(self.device).call("dgp_elbo_grad_host", C.byref(m), X_host.ctypes.data_as(C.c_void_p),
                                           Y_host.ctypes.data_as(C.c_void_p), X_host.shape[0], self.num_samples, float(scale),
                                           float(kl_weight), self._next_seed(seed), int(n_offset), 1 if want_grad else 0,
                                           out_host.ctypes.data_as(C.c_void_p))
        return out_host

    def ELBO(self, data, zs=None, seed=None):
        """dgp.py:89-100 -> 0-d tensor. The reference's minibatch scale is identically 1 (dgp.py:95-99)."""
        flat = self.elbo_flat(data, want_grad=False, zs=zs, seed=seed)
        _lib.get_context(self.device).check()   # the value path reports a failed Cholesky; the training loop stays asynchronous
        return flat[0] - flat[1]

    def ELBO_closure(self, data, zs=None, seed=None):
        """dgp.py:102-109 (the reference wraps ELBO in tf.function; here it is already one C-ABI call)."""
        return self.ELBO(data, zs=zs, seed=seed)

    def unpack_grads(self, flat):
        """flat buffer -> {Parameter: constrained-space gradient tensor} (views into `flat`)."""
        _, offs = self.grad_layout()
        out = {}
        for l, o in zip(self.layers, offs):
            M, D_in = l.feature.Z.shape
            D_out = l.num_outputs
            out[l.feature.Z] = flat[o.dZ:o.dZ + M * D_in].reshape(M, D_in)
            gl = flat[o.dlengthscales:o.dlengthscales + D_in]
            out[l.kern.lengthscales] = gl if l.kern.lengthscales.value.numel() == D_in and l.kern.lengthscales.value.dim() > 0 \
                else gl.sum().reshape(l.kern.lengthscales.value.shape)
            out[l.kern.variance] = flat[o.dvariance:o.dvariance + 1].reshape(())
            out[l.q_mu] = flat[o.dq_mu:o.dq_mu + M * D_out].reshape(M, D_out)
            out[l.q_sqrt] = flat[o.dq_sqrt:o.dq_sqrt + D_out * M * M].reshape(D_out, M, M)
        out[self.likelihood.likelihood.variance] = flat[2].reshape(())
        return out

    def ELBO_and_grads(self, data, zs=None, seed=None, scale=1.0):
        """ELBO and constrained-space gradients as a dict keyed like the oracle (`layers.i.Z`, ..., `lik_var`)."""
        flat = self.elbo_flat(data, want_grad=True, zs=zs, seed=seed, scale=scale)
        g = self.unpack_grads(flat)
        named = {}
        for i, l in enumerate(self.layers):
            named[f"layers.{i}.Z"] = g[l.feature.Z]
            named[f"layers.{i}.lengthscales"] = g[l.kern.lengthscales]
            named[f"layers.{i}.variance"] = g[l.kern.variance]
            named[f"layers.{i}.q_mu"] = g[l.q_mu]
            named[f"layers.{i}.q_sqrt"] = g[l.q_sqrt]
        named["lik_var"] = g[self.likelihood.likelihood.variance]
        return flat[0] - flat[1], named

    # ------------------------------------------------------------------ a11: prediction
    def predict_y(self, Xnew, num_samples, zs=None, seed=None):
        """dgp.py:113-124: (mu, var + sigma_n^2), both [S,N,D_L]."""
        Fmean, Fvar = self.predict_f(Xnew, S=num_samples, zs=zs, seed=seed)
        return self.likelihood.predict_mean_and_var(Fmean, Fvar)

    def predict_density(self, Xnew, Ynew, num_samples):
        raise NotImplementedError("broken in the reference (tf.log, dgp.py:129); not on the accelerated path")

    def predict_moments(self, Xnew, num_samples, add_lik_var=True, zs=None, seed=None, out=None):
        """Mixture moments over the S samples reduced on the device (dgp.py:362-366; Infill_criteria.py:39-41). `out=(mean, var)`
        writes into caller-owned [N, D] buffers: the search loops pass the same pair every call so that graph replay
        (dgp_set_graph) sees addresses that never move, whatever the caching allocator does."""
        X = self._check_X(_lib.as_device(Xnew, self.device))
        N, D = X.shape[0], self.layers[-1].num_outputs
        if out is not None:
            mean, var = out
            for t in (mean, var):
                if tuple(t.shape) != (N, D) or t.dtype != torch.float64 or t.device != X.device or not t.is_contiguous():
                    raise ValueError("out= must be two contiguous float64 [N, D] tensors on the model's device")
        else:
            mean = torch.empty((N, D), dtype=torch.float64, device=X.device)
            var = torch.empty_like(mean)
        if N == 0:
            return mean, var
        m, keep = self._model_desc()
        zt, zp = self._zs(zs, num_samples, N)
        _lib.get_context(X.device).call("dgp_predict_moments", C.byref(m), _lib.ptr(X), N, num_samples, zp, self._next_seed(seed), 0,
                                        1 if add_lik_var else 0, _lib.ptr(mean), _lib.ptr(var))
        return mean, var

    def predict(self, Xnew, num_samples, zs=None, seed=None):
        """dgp.py:362-366 (DGP.predict: mixture moments of predict_y), reduced on the device. Raises on a non-positive-definite
        Kuu instead of returning NaN (the search loops call predict_moments directly and check once at their end)."""
        out = self.predict_moments(Xnew, num_samples, add_lik_var=True, zs=zs, seed=seed)
        _lib.get_context(self.device).check()
        return out

    # ------------------------------------------------------------------ optimisers (callers of the hot path, SURVEY §8 f1)
    _TRANSFORM_CODE = {None: 0, "positive": 1, "positive_shift": 2, "triangular": 3}

    def _adam_params(self, params):
        """Parameter list -> (dgp_adam_param array, keep-alive list): where each trainable Parameter lives, where its gradient sits
        in the dgp_elbo_grad buffer and which GPflow bijector maps it to the variable tf.optimizers.Adam updates."""
        _, offs = self.grad_layout()
        where = {}
        kerns = [id(l.kern) for l in self.layers]
        if len(set(kerns)) != len(kerns):
            raise NotImplementedError("one kernel object shared by several layers: its gradient would be the sum over those layers, "
                                      "which the fused Adam launch does not form -- give every layer its own kernel object")
        for l, o in zip(self.layers, offs):
            M, D_in = l.feature.Z.shape
            where[id(l.feature.Z)] = (o.dZ, M * D_in, None, 0)
            ls = l.kern.lengthscales
            if ls.value.numel() == D_in and ls.value.dim() > 0:
                where[id(ls)] = (o.dlengthscales, D_in, None, 0)
            else:   # one lengthscale shared by all inputs: gradient summed, value re-broadcast into the [D_in] vector of the ABI
                where[id(ls)] = (o.dlengthscales, D_in, l.kern.lengthscales_vector(D_in), 0)
            where[id(l.kern.variance)] = (o.dvariance, 1, None, 0)
            where[id(l.q_mu)] = (o.dq_mu, M * l.num_outputs, None, 0)
            where[id(l.q_sqrt)] = (o.dq_sqrt, l.num_outputs * M * M, None, M)
        where[id(self.likelihood.likelihood.variance)] = (2, 1, None, 0)
        if len(params) > 48:     # kAdamMaxParams (csrc/small.cuh): the table travels as a kernel argument
            raise ValueError(f"{len(params)} trainable parameters: one fused Adam launch holds at most 48 (9 layers x 5 + likelihood); "
                             "fix some with set_trainable(p, False) or train in two groups")
        arr = (_lib.AdamParam * len(params))()
        keep = []
        for i, p in enumerate(params):
            if id(p) not in where:
                raise NotImplementedError(f"{p!r} has no gradient on the accelerated path (SURVEY §8 f2): set_trainable(p, False)")
            off, gcount, mirror, M = where[id(p)]
            v = p.value
            if not v.is_contiguous():
                raise ValueError(f"{p!r} must be contiguous")
            arr[i].value, arr[i].count = v.data_ptr(), v.numel()
            arr[i].grad_offset, arr[i].grad_count = off, gcount
            arr[i].transform, arr[i].M = self._TRANSFORM_CODE[p.transform], M
            if mirror is not None:
                arr[i].mirror, arr[i].mirror_count = mirror.data_ptr(), mirror.numel()
                keep.append(mirror)
            keep.append(v)
        return arr, keep

    def _adam_state(self, params):
        """(m, v) of tf.optimizers.Adam, flat in `params` order."""
        n = sum(p.value.numel() for p in params)
        return (torch.zeros(n, dtype=torch.float64, device=self.device), torch.zeros(n, dtype=torch.float64, device=self.device))

    def _adam_step(self, params, flat, state, t, lr, beta_1, beta_2, epsilon):
        """One dgp_adam_step: Keras/TF Adam on the unconstrained variables from the constrained-space gradients in `flat`."""
        arr, keep = self._adam_params(params)
        _lib.get_context(self.device).call("dgp_adam_step", arr, len(params), _lib.ptr(flat), _lib.ptr(state[0]), _lib.ptr(state[1]),
                                           int(t), float(lr), float(beta_1), float(beta_2), float(epsilon))

    def _train_adam(self, data, params, state, t0, steps, lr, beta_1, beta_2, epsilon, scale=1.0, kl_weight=1.0):
        """`steps` iterations of (ELBO gradient, Adam update) in one dgp_train_adam call; returns the per-step ELBO estimates
        (device tensor [steps]). Seeds continue the model's draw sequence exactly like `steps` elbo_flat calls would."""
        X, Y = data
        X = _lib.as_device(X, self.device)
        Y = _lib.as_device(Y, self.device)
        self._check_XY(X, Y)
        if X.shape[0] == 0:
            raise ValueError("empty minibatch")
        if steps <= 0:
            return torch.empty(0, dtype=torch.float64, device=X.device)
        m, keep = self._model_desc()
        arr, keep2 = self._adam_params(params)
        n = int(_lib.lib.dgp_grad_size(C.byref(m)))
        if getattr(self, "_train_flat", None) is None or self._train_flat.numel() != n or self._train_flat.device != X.device:
            self._train_flat = torch.empty(n, dtype=torch.float64, device=X.device)   # one address across calls: graph replay
        trace = torch.empty(max(steps, 1), dtype=torch.float64, device=X.device)
        seed0 = self._next_seed(None)
        self._draw += steps - 1
        _lib.get_context(X.device).call("dgp_train_adam", C.byref(m), _lib.ptr(X), _lib.ptr(Y), X.shape[0], self.num_samples,
                                        float(scale), float(kl_weight), seed0, 0x9E3779B97F4A7C15, 0, arr, len(params),
                                        _lib.ptr(state[0]), _lib.ptr(state[1]), int(t0), int(steps), float(lr), float(beta_1),
                                        float(beta_2), float(epsilon), _lib.ptr(self._train_flat), _lib.ptr(trace))
        return trace[:steps]

    def _adam_loop(self, data, params, state, t0, iterations, lr, beta_1, beta_2, epsilon, messages):
        """The reference's loop (dgp.py:146-154) in blocks that end on the steps it prints at (step % messages == 0)."""
        ctx = _lib.get_context(self.device)
        X = _lib.as_device(data[0], self.device)
        data = (X, _lib.as_device(data[1], self.device))   # one device copy for the whole loop: stable addresses
        # launch-bound problems (the library's own threshold for its sub-wave paths): replay the step as a CUDA graph
        auto_graph = not ctx.graph and X.shape[0] * self.num_samples <= 32768
        if auto_graph:
            ctx.set_graph(True)
        try:
            step = 0
            while step < iterations:
                n = 1 if step == 0 else min(messages, iterations - step)
                trace = self._train_adam(data, params, state, t0 + step, n, lr, beta_1, beta_2, epsilon)
                step += n
                if (step - 1) % messages == 0:
                    print(f"ELBO: {trace[-1].item()}")
                    ctx.check()   # .item() has synchronised already: a failed Cholesky is raised at the block it happened in,
                    #               with the parameters frozen at their last good values (adam_kernel skips flagged steps)
            ctx.check()
        finally:
            if auto_graph:
                ctx.set_graph(False)

    def optimize_adam(self, data, iterations=5000, lr=0.01, beta_1=0.9, beta_2=0.999, epsilon=1e-07, messages=100):
        """dgp.py:132-154. The whole loop runs in the library (dgp_train_adam); the host only prints."""
        params = self.trainable_parameters
        state = self._adam_state(params)
        self._adam_loop(data, params, state, 1, iterations, lr, beta_1, beta_2, epsilon, messages)

    def natgrad_step(self, data, gamma, variational_params, scale=1.0, seed=None, zs=None, out=None):
        """One GPflow NaturalGradient(gamma).minimize(-ELBO, var_list=[(q_mu, q_sqrt), ...]) step with the default XiNat
        parameterisation (dgp.py:188,218,312,343; SURVEY §2): theta <- theta - gamma * d(-ELBO)/d eta with natural parameters
        theta = (S^-1 mu, -S^-1/2) and expectation parameters eta = (mu, S + mu mu^T), S = R R^T, R = q_sqrt, per output column.
        With G_mu, G_R the loss gradients, dS = R^-T P R^-1 (Cholesky adjoint, P = sym(Phi(R^T G_R))) and d_eta = (G_mu - 2 dS mu,
        dS), the update collapses to
            S_new^-1 = S^-1 + 2 gamma dS = R^-T (I + 2 gamma P) R^-1,      mu_new = mu - gamma S_new G_mu,
        so with the reverse Cholesky I + 2 gamma P = U U^T (U upper) the new factor is q_sqrt_new = R U^-T (lower times lower, positive
        diagonal: the Cholesky factor of S_new) and mu_new = mu - gamma q_sqrt_new q_sqrt_new^T G_mu -- one triangular product, one
        M x M Cholesky and one triangular inverse per output, no explicit inverse of S. The ELBO gradient comes from one dgp_elbo_grad
        call and the update from one dgp_natgrad_step call (batched over layers and outputs in the library's own kernels; no
        torch.linalg). Checked against the oracle, which takes d/d eta by autograd through the expectation parameters."""
        flat = self.elbo_flat(data, want_grad=True, scale=scale, seed=seed, zs=zs, out=out)
        m, keep = self._model_desc()
        ids = self._nat_layer_ids(variational_params)
        _lib.get_context(self.device).call("dgp_natgrad_step", C.byref(m), ids, len(ids), float(gamma), _lib.ptr(flat))
        return flat[0] - flat[1]

    def _nat_layer_ids(self, variational_params):
        """[(q_mu, q_sqrt), ...] (the reference's var_list) -> C int array of layer indices."""
        idx = []
        for pair in variational_params:
            q_mu, q_sqrt = pair[0], pair[1]
            hit = [i for i, l in enumerate(self.layers) if l.q_mu is q_mu and l.q_sqrt is q_sqrt]
            if not hit:
                raise ValueError("natural-gradient pairs must be the (q_mu, q_sqrt) of this model's layers")
            idx.append(hit[0])
        return (C.c_int * len(idx))(*idx)

    def _train_nat_adam(self, data, params, state, t0, steps, lr, beta_1, beta_2, epsilon, variational_params, gamma, scale=1.0,
                        kl_weight=1.0):
        """`steps` iterations of part 2 of optimize_nat_adam in one dgp_train_nat_adam call; returns the per-iteration ELBO estimates."""
        X, Y = data
        X = _lib.as_device(X, self.device)
        Y = _lib.as_device(Y, self.device)
        self._check_XY(X, Y)
        if steps <= 0:
            return torch.empty(0, dtype=torch.float64, device=X.device)
        m, keep = self._model_desc()
        arr, keep2 = self._adam_params(params) if params else (None, [])
        n = int(_lib.lib.dgp_grad_size(C.byref(m)))
        if getattr(self, "_train_flat", None) is None or self._train_flat.numel() != n or self._train_flat.device != X.device:
            self._train_flat = torch.empty(n, dtype=torch.float64, device=X.device)
        trace = torch.empty(steps, dtype=torch.float64, device=X.device)
        ids = self._nat_layer_ids(variational_params)
        seed0 = self._next_seed(None)
        self._draw += 2 * steps - 1
        _lib.get_context(X.device).call("dgp_train_nat_adam", C.byref(m), _lib.ptr(X), _lib.ptr(Y), X.shape[0], self.num_samples,
                                        float(scale), float(kl_weight), seed0, 0x9E3779B97F4A7C15, 0, arr, len(params),
                                        _lib.ptr(state[0]), _lib.ptr(state[1]), int(t0), int(steps), float(lr), float(beta_1),
                                        float(beta_2), float(epsilon), ids, len(ids), float(gamma), _lib.ptr(self._train_flat),
                                        _lib.ptr(trace))
        return trace

    def optimize_nat_adam(self, data, iterations1=100, iterations2=5000, lr_adam=0.01, lr_gamma=0.01, beta_1=0.9, beta_2=0.999,
                          epsilon=1e-07, ng_all=True, messages=100):
        """dgp.py:155-220: part 1 Adam on the kernel / inducing-input / likelihood parameters with q fixed; part 2 alternates
        one Adam step with one natural-gradient step on the (q_mu, q_sqrt) pairs (all layers, or the last one only)."""
        nat_layers = self.layers if ng_all else self.layers[-1:]
        for layer in nat_layers:
            gpflow.set_trainable(layer.q_mu, False)
            gpflow.set_trainable(layer.q_sqrt, False)
        variational_params = [(layer.q_mu, layer.q_sqrt) for layer in nat_layers]
        params = self.trainable_parameters
        state = self._adam_state(params)
        self._adam_loop(data, params, state, 1, iterations1, lr_adam, beta_1, beta_2, epsilon, messages)
        ctx = _lib.get_context(self.device)
        X = _lib.as_device(data[0], self.device)
        data = (X, _lib.as_device(data[1], self.device))      # one device copy: stable addresses for graph replay
        auto_graph = not ctx.graph and X.shape[0] * self.num_samples <= 32768
        if auto_graph:
            ctx.set_graph(True)
        try:
            # part 2 in blocks that end on the iterations the reference prints at (step % messages == 0); the whole block
            # (two ELBO+gradient evaluations, Adam and natural-gradient launches per iteration) runs in the library
            step = 0
            while step < iterations2:
                n = 1 if step == 0 else min(messages, iterations2 - step)
                trace = self._train_nat_adam(data, params, state, iterations1 + 1 + step, n, lr_adam, beta_1, beta_2, epsilon,
                                             variational_params, lr_gamma)
                step += n
                if (step - 1) % messages == 0:
                    print(f"ELBO: {trace[-1].item()}")
                    ctx.check()
            ctx.check()
        finally:
            if auto_graph:
                ctx.set_graph(False)

    def number_parameters(self, trainable=True):
        """dgp.py:348-360."""
        ps = self.trainable_parameters if trainable else self.parameters
        return int(sum(int(np.prod(p.shape)) if len(p.shape) else 1 for p in ps))


class DGP(DGP_Base):
    """dgp_dace/models/dgp.py:221-366: doubly-stochastic DGP with linear/identity mean functions."""

    def __init__(self, X, Y, Z, kernels, num_units, likelihood, num_outputs=None, mean_function=None, white=False, **kwargs):
        layers = init_layers_linear(X, Y, Z, kernels, num_units, num_outputs=num_outputs,
                                    mean_function=mean_function, white=white)
        DGP_Base.__init__(self, likelihood, layers, **kwargs)
        self.data = (_lib.as_device(X, self.device), _lib.as_device(Y, self.device))

    def optimize_adam(self, iterations=5000, lr=0.01, beta_1=0.9, beta_2=0.999, epsilon=1e-07, messages=100):
        """dgp.py:255-279: hidden layers' q_sqrt *= 1e-3 first (:268-269), then Adam."""
        for layer in self.layers[:-1]:
            layer.q_sqrt.assign(layer.q_sqrt.value * 1e-3)
        DGP_Base.optimize_adam(self, self.data, iterations, lr, beta_1, beta_2, epsilon, messages)

    def optimize_nat_adam(self, iterations1=100, iterations2=5000, lr_adam=0.01, lr_gamma=0.01, beta_1=0.9, beta_2=0.999,
                          epsilon=1e-07, ng_all=True, messages=100):
        """dgp.py:281-345: as DGP_Base.optimize_nat_adam on self.data after the hidden layers' q_sqrt *= 1e-3 (:323-324)."""
        for layer in self.layers[:-1]:
            layer.q_sqrt.assign(layer.q_sqrt.value * 1e-3)
        DGP_Base.optimize_nat_adam(self, self.data, iterations1, iterations2, lr_adam, lr_gamma, beta_1, beta_2, epsilon,
                                   ng_all, messages)

