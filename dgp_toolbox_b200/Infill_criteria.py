"""The reference's infill criteria with their interface (dgp_dace/Infill_criteria.py): evaluation on the accelerated path
(dgp_ei, dgp_ei_grad, dgp_predict_moments + dgp_acq_moments) and the `optimize` searches (differential evolution, then Adam on
the sigmoid-reparameterised x; Infill_criteria.py:61-87,142-168,207-233) with the search state on the device (search.py,
SURVEY §8 f3)."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib, search


class Infill_criteria(object):
    def __init__(self):
        self.name = 'Infill criteria'

    def run(self, x):
        raise NotImplementedError("method not implemented")

    def optimize(self):
        raise NotImplementedError("method not implemented")


class EI(Infill_criteria):
    """Infill_criteria.py:20-52."""

    def __init__(self, y_min, d):
        self.name = 'Expected Improvement'
        self.y_min = y_min
        self.d = d
        self.IC_optimized = None
        self.x_opt = None

    def run(self, model, x, analytic=True, num_samples=1000, zs=None, seed=None, out=None):
        """Returns -EI [N, D_L]. analytic: moment-match predict_f over the S samples (:39-41) then the closed form
        (:43-47); otherwise mean_s max(y_min - F, 0) on propagated samples (:49-51). One C-ABI call (dgp_ei).
        `out`: result buffer to reuse (search loops keep every address fixed so that the call replays as a graph)."""
        if getattr(model, "name", None) != 'dgp':
            raise NotImplementedError("only model.name == 'dgp' is on the accelerated path")
        X = model._check_X(_lib.as_device(x, model.device))
        N, D = X.shape[0], model.layers[-1].num_outputs
        own_out = out is None
        if out is None:
            out = torch.empty((N, D), dtype=torch.float64, device=X.device)
        if N == 0:
            return out
        m, keep = model._model_desc()
        zt, zp = model._zs(zs, num_samples, N)
        y_min = float(self.y_min.item() if hasattr(self.y_min, "item") else self.y_min)
        ctx = _lib.get_context(X.device)
        ctx.call("dgp_ei", C.byref(m), _lib.ptr(X), N, num_samples, zp, model._next_seed(seed), 0,
                 y_min, 1 if analytic else 0, _lib.ptr(out))
        if own_out:
            ctx.check()   # a user call: raise on a non-positive-definite Kuu instead of returning NaN (search loops pass `out`)
        return out

    def run_with_grad(self, model, x, num_samples=1000, zs=None, seed=None, out=None, dx=None):
        """(-EI [N, D_L], d sum(-EI) / dx [N, d]): the value and the gradient the reference's Adam-on-x loop takes with
        tape.gradient(loss, x) (Infill_criteria.py:79-84), analytic EI. One C-ABI call (dgp_ei_grad)."""
        if getattr(model, "name", None) != 'dgp':
            raise NotImplementedError("only model.name == 'dgp' is on the accelerated path")
        X = model._check_X(_lib.as_device(x, model.device))
        N, D = X.shape[0], model.layers[-1].num_outputs
        if out is None:
            out = torch.empty((N, D), dtype=torch.float64, device=X.device)
        if dx is None:
            dx = torch.zeros_like(X)
        if N == 0:
            return out, dx
        m, keep = model._model_desc()
        zt, zp = model._zs(zs, num_samples, N)
        y_min = float(self.y_min.item() if hasattr(self.y_min, "item") else self.y_min)
        _lib.get_context(X.device).call("dgp_ei_grad", C.byref(m), _lib.ptr(X), N, num_samples, zp, model._next_seed(seed), 0,
                                        y_min, _lib.ptr(out), _lib.ptr(dx))
        return out, dx

    def loss(self, model, x, analytic):
        """Infill_criteria.py:53-60."""
        return self.run(model, x, analytic)

    def optimize(self, model, bounds, popsize_DE=300, popstd_DE=1.5, iterations_DE=400, init_adam=None, iterations_adam=1000,
                 method='DE', analytic=True, num_samples=1000, seed=None, adam_starts=1):
        """Infill_criteria.py:61-87: minimise -EI over the box `bounds = (lw, up)`; 'DE' (differential evolution, population
        popsize_DE around u = 0 with spread popstd_DE, iterations_DE generations, one dgp_ei call per generation), 'Adam'
        (iterations_adam steps of lr 0.01 on u from init_adam, one dgp_ei_grad call per step) or 'DE+Adam'. Sets and returns
        x_opt [d, 1] (numpy, like the reference); IC_optimized is the criterion there. Every evaluation draws fresh samples,
        as the reference's tf.random.normal does. adam_starts > 1 (an extension; the reference refines one point) starts the
        Adam stage of 'DE+Adam' from the best `adam_starts` members of the final population side by side -- the same number
        of launches, one dgp_ei_grad call over adam_starts candidates per step -- and keeps the best end point."""
        lw = np.broadcast_to(np.asarray(bounds[0], dtype=np.float64).reshape(-1), (self.d,)).copy()
        up = np.broadcast_to(np.asarray(bounds[1], dtype=np.float64).reshape(-1), (self.d,)).copy()
        if method not in ('DE', 'Adam', 'DE+Adam'):
            raise ValueError(f"unknown method {method!r}")
        de_seed = model._next_seed(seed)
        with search.GraphScope(model.device):
            if method in ('DE', 'DE+Adam'):
                res = search.de_minimize(lambda X, out: self.run(model, X, analytic, num_samples, out=out), lw, up, self.d,
                                         model.device, popsize_DE, popstd_DE, iterations_DE, seed=de_seed)
                self.x_opt = res["x"].cpu().numpy().reshape(self.d, 1)
                starts_u = res["population_u"][torch.argsort(res["values"])[:max(1, int(adam_starts))]].contiguous()
                self.de_iterations = res["iterations"]      # < iterations_DE when the population collapsed (TFP position_tolerance)
                self.IC_optimized = self.run(model, self.x_opt.reshape(1, self.d), analytic, num_samples)
            if method in ('Adam', 'DE+Adam'):
                if not analytic:
                    raise NotImplementedError("the input gradient exists for the analytic EI only")
                if init_adam is None:
                    init_adam = np.zeros(self.d) if self.x_opt is None else self.x_opt
                init_adam = np.asarray(init_adam, dtype=np.float64).reshape(self.d)
                u0 = _lib.as_device(np.log((up - init_adam + 1e-3) / (init_adam - lw + 1e-3)).reshape(1, self.d), model.device)
                if method == 'DE+Adam' and int(adam_starts) > 1:
                    u0 = starts_u            # the population is already in u-space
                n = u0.shape[0]
                out = torch.empty((n, model.layers[-1].num_outputs), dtype=torch.float64, device=u0.device)
                dx = torch.zeros_like(u0)
                u, X, val = search.adam_box_minimize(
                    lambda X: self.run_with_grad(model, X, num_samples, out=out, dx=dx), lw, up, u0, iterations_adam, lr=0.01)
                best = int(torch.argmin(val.sum(dim=1))) if n > 1 else 0
                self.x_opt = X[best].cpu().numpy().reshape(self.d, 1)
                self.IC_optimized = val[best:best + 1].clone()
        return self.x_opt


class qEI(Infill_criteria):
    """Batch expected improvement of q points: EI.run(analytic=False)'s mean_s max(y_min - F, 0) (Infill_criteria.py:49-51) with
    F replaced by the minimum over a batch of q points sampled jointly (propagate(full_cov=True) on the q points)."""

    def __init__(self, y_min, d, q):
        self.name = 'q-point Expected Improvement'
        self.y_min = y_min
        self.d = d
        self.q = int(q)
        self.IC_optimized = None
        self.x_opt = None

    def run(self, model, x, num_samples=1000, zs=None, seed=None, out=None):
        """Returns -q-EI [G, D_L] of the G batches in x ([G q, d], batch g = rows g q .. g q + q - 1, or [G, q, d]). Batches are
        independent of each other. One C-ABI call (dgp_qei); `out` is a result buffer to reuse, as in EI.run."""
        if getattr(model, "name", None) != 'dgp':
            raise NotImplementedError("only model.name == 'dgp' is on the accelerated path")
        X = _lib.as_device(x, model.device)
        if X.dim() == 3:
            if X.shape[1] != self.q:
                raise ValueError(f"x has shape {tuple(X.shape)}, expected [G, {self.q}, d]")
            X = X.reshape(-1, X.shape[2])
        X = model._check_X(X)
        N, D = X.shape[0], model.layers[-1].num_outputs
        own_out = out is None
        if out is None:
            out = torch.empty((N // self.q if self.q > 0 else 0, D), dtype=torch.float64, device=X.device)
        if N == 0:
            return out
        m, keep = model._model_desc()
        zt, zp = model._zs(zs, num_samples, N)
        ctx = _lib.get_context(X.device)
        ctx.call("dgp_qei", C.byref(m), _lib.ptr(X), N, num_samples, self.q, zp, model._next_seed(seed), 0, _scalar(self.y_min),
                 _lib.ptr(out))
        if own_out:
            ctx.check()
        return out

    def optimize(self, model, bounds, popsize_DE=300, popstd_DE=1.5, iterations_DE=400, method='DE', num_samples=1000, seed=None):
        """Minimise -q-EI over batches of q points in the box `bounds = (lw, up)`: differential evolution in q d dimensions (the box
        tiled q times; member k decodes to the batch x[k].reshape(q, d)), one dgp_qei call per generation with fresh draws. Sets
        and returns x_opt [q, d] (numpy); IC_optimized [1, D_L] is the criterion there. The full-covariance path has no adjoint,
        so there is no Adam stage."""
        if method in ('Adam', 'DE+Adam'):
            raise NotImplementedError("q-EI has no input gradient (the full-covariance path has no adjoint): use method='DE'")
        if method != 'DE':
            raise ValueError(f"unknown method {method!r}")
        if getattr(model, "name", None) != 'dgp':
            raise NotImplementedError("only model.name == 'dgp' is on the accelerated path")
        lw = np.broadcast_to(np.asarray(bounds[0], dtype=np.float64).reshape(-1), (self.d,))
        up = np.broadcast_to(np.asarray(bounds[1], dtype=np.float64).reshape(-1), (self.d,))
        qd = self.q * self.d
        res = search.de_minimize(lambda X, out: self.run(model, X.reshape(-1, self.d), num_samples, out=out), np.tile(lw, self.q),
                                 np.tile(up, self.q), qd, model.device, popsize_DE, popstd_DE, iterations_DE, seed=model._next_seed(seed))
        self.x_opt = res["x"].cpu().numpy().reshape(self.q, self.d)
        self.de_iterations = res["iterations"]
        self.IC_optimized = self.run(model, self.x_opt, num_samples)
        return self.x_opt


def _scalar(v):
    return float(v.item() if hasattr(v, "item") else v)


def _moment_scratch(model, N, D):
    """One (mean, var) pair per model and population size, reused by every criterion evaluation of a search: temporaries whose
    addresses stay put so a captured graph can be replayed."""
    cache = model.__dict__.setdefault("_moment_bufs", {})
    key = (N, D, str(model.device))
    if key not in cache:
        if len(cache) >= 4:
            cache.clear()
        cache[key] = (torch.empty((N, D), dtype=torch.float64, device=model.device),
                      torch.empty((N, D), dtype=torch.float64, device=model.device))
    return cache[key]


def _moment_criterion(kind, model, x, y, num_samples, zs, seed, with_x=False, out=None):
    """predict_y mixture moments over `num_samples` propagated samples (the reference hard-codes 500), then one
    dgp_acq_moments launch. `out` ([N, 1], or [N, d] with `with_x`) receives the values when given."""
    if getattr(model, "name", None) != 'dgp':
        raise NotImplementedError("only model.name == 'dgp' is on the accelerated path")
    X = model._check_X(_lib.as_device(x, model.device))
    N, d = X.shape
    D = model.layers[-1].num_outputs
    if D != 1:
        raise ValueError("the criterion expects a single-output model")
    m, v = model.predict_moments(X, num_samples, add_lik_var=True, zs=zs, seed=seed, out=_moment_scratch(model, N, D))
    if out is None:
        out = torch.empty((N, d if with_x else 1), dtype=torch.float64, device=X.device)
    elif tuple(out.shape) != (N, d if with_x else 1):
        raise ValueError(f"out= must be [{N}, {d if with_x else 1}]")
    if N:
        _lib.get_context(X.device).call("dgp_acq_moments", kind, _lib.ptr(m), _lib.ptr(v), N, _scalar(y),
                                        _lib.ptr(X) if with_x else None, d if with_x else 0, _lib.ptr(out))
    return out


def _moment_criterion_grad(kind, model, x, y, num_samples, zs, seed, out=None, dx=None):
    """(criterion [N, 1], d sum(criterion) / dx [N, d]) for kind 1 (WB2) / 2 (EV) / 3 (WB2S: criterion [N, d]) on predict_y mixture
    moments: one dgp_acq_grad call (criterion adjoints, then the data path of the adjoint chain)."""
    if getattr(model, "name", None) != 'dgp':
        raise NotImplementedError("only model.name == 'dgp' is on the accelerated path")
    X = model._check_X(_lib.as_device(x, model.device))
    N, D = X.shape[0], model.layers[-1].num_outputs
    if D != 1:
        raise ValueError("the criterion expects a single-output model")
    if out is None:
        out = torch.empty((N, X.shape[1] if kind == 3 else D), dtype=torch.float64, device=X.device)
    if dx is None:
        dx = torch.zeros_like(X)
    if N == 0:
        return out, dx
    m, keep = model._model_desc()
    zt, zp = model._zs(zs, num_samples, N)
    _lib.get_context(X.device).call("dgp_acq_grad", C.byref(m), kind, _lib.ptr(X), N, num_samples, zp, model._next_seed(seed), 0,
                                    _scalar(y), _lib.ptr(out), _lib.ptr(dx))
    return out, dx


def _optimize_de(crit, run, model, bounds, popsize_DE, popstd_DE, iterations_DE, method, seed):
    """The DE stage of the reference's `optimize` for the moment-based criteria (Infill_criteria.py:142-168,207-233)."""
    if method != 'DE':
        raise NotImplementedError("method 'Adam' / 'DE+Adam' needs the input gradient, which WB2S does not have on this path")
    lw = np.broadcast_to(np.asarray(bounds[0], dtype=np.float64).reshape(-1), (crit.d,)).copy()
    up = np.broadcast_to(np.asarray(bounds[1], dtype=np.float64).reshape(-1), (crit.d,)).copy()
    with search.GraphScope(model.device):
        res = search.de_minimize(run, lw, up, crit.d, model.device, popsize_DE, popstd_DE, iterations_DE,
                                 seed=model._next_seed(seed))
        crit.x_opt = res["x"].cpu().numpy().reshape(crit.d, 1)
        crit.de_iterations = res["iterations"]
        crit.IC_optimized = run(crit.x_opt.reshape(1, crit.d), None)
    return crit.x_opt


class WB2(Infill_criteria):
    """Infill_criteria.py:106-141: -(EI - mean) on predict_y moments."""

    def __init__(self, y_min, d):
        self.name = 'WB2 criterion'
        self.y_min = y_min
        self.d = d
        self.IC_optimized = None
        self.x_opt = None

    def run(self, model, x, num_samples=500, zs=None, seed=None, out=None):
        return _moment_criterion(1, model, x, self.y_min, num_samples, zs, seed, out=out)

    def loss(self, model, x):
        return self.run(model, x)

    def run_with_grad(self, model, x, num_samples=500, zs=None, seed=None, out=None, dx=None):
        """(WB2 [N, 1], d sum(WB2) / dx [N, d]) -- what tape.gradient(loss, x) gives the reference's Adam stage (:160-165)."""
        return _moment_criterion_grad(1, model, x, self.y_min, num_samples, zs, seed, out, dx)

    @staticmethod
    def ncol(d):
        return 1

    def optimize(self, model, bounds, popsize_DE=300, popstd_DE=1.5, iterations_DE=400, init_adam=None, iterations_adam=1000,
                 method='DE', seed=None):
        """Infill_criteria.py:142-168: 'DE', 'Adam' or 'DE+Adam' like EI.optimize."""
        return _optimize_de_adam(self, model, bounds, popsize_DE, popstd_DE, iterations_DE, init_adam, iterations_adam, method, seed)


def _optimize_de_adam(crit, model, bounds, popsize_DE, popstd_DE, iterations_DE, init_adam, iterations_adam, method, seed):
    """The two stages of the reference's `optimize` for a moment-based criterion with `run` and `run_with_grad` (WB2, WB2S)."""
    if method not in ('DE', 'Adam', 'DE+Adam'):
        raise ValueError(f"unknown method {method!r}")
    d = crit.d
    lw = np.broadcast_to(np.asarray(bounds[0], dtype=np.float64).reshape(-1), (d,)).copy()
    up = np.broadcast_to(np.asarray(bounds[1], dtype=np.float64).reshape(-1), (d,)).copy()
    if method in ('DE', 'DE+Adam'):
        _optimize_de(crit, lambda X, out: crit.run(model, X, out=out), model, bounds, popsize_DE, popstd_DE, iterations_DE, 'DE', seed)
    if method in ('Adam', 'DE+Adam'):
        with search.GraphScope(model.device):
            if init_adam is None:
                init_adam = np.zeros(d) if crit.x_opt is None else crit.x_opt
            init_adam = np.asarray(init_adam, dtype=np.float64).reshape(d)
            u0 = _lib.as_device(np.log((up - init_adam + 1e-3) / (init_adam - lw + 1e-3)).reshape(1, d), model.device)
            out = torch.empty((1, crit.ncol(d)), dtype=torch.float64, device=u0.device)
            dx = torch.zeros_like(u0)
            u, X, val = search.adam_box_minimize(lambda X: crit.run_with_grad(model, X, out=out, dx=dx), lw, up, u0,
                                                 iterations_adam, lr=0.01)
            crit.x_opt = X.cpu().numpy().reshape(d, 1)
            crit.IC_optimized = val.clone()
    return crit.x_opt


class WB2S(Infill_criteria):
    """Infill_criteria.py:169-206: -(S * EI - mean) with S = 1 / (1 + 1/exp(x)) elementwise in x -> [N, d]."""

    def __init__(self, y_min, d):
        self.name = 'WB2S criterion'
        self.y_min = y_min
        self.d = d
        self.IC_optimized = None
        self.x_opt = None

    def run(self, model, x, num_samples=500, zs=None, seed=None, out=None):
        return _moment_criterion(3, model, x, self.y_min, num_samples, zs, seed, with_x=True, out=out)

    def loss(self, model, x):
        return self.run(model, x)

    def run_with_grad(self, model, x, num_samples=500, zs=None, seed=None, out=None, dx=None):
        """(WB2S [N, d], d sum(WB2S) / dx [N, d]): the chain's input gradient plus the explicit -sig'(x) EI term (:187,198,225-230)."""
        return _moment_criterion_grad(3, model, x, self.y_min, num_samples, zs, seed, out, dx)

    @staticmethod
    def ncol(d):
        return d

    def optimize(self, model, bounds, popsize_DE=300, popstd_DE=1.5, iterations_DE=400, init_adam=None, iterations_adam=1000,
                 method='DE', seed=None):
        """Infill_criteria.py:207-233: 'DE', 'Adam' or 'DE+Adam' (the [N, d] criterion is summed over its columns per candidate)."""
        return _optimize_de_adam(self, model, bounds, popsize_DE, popstd_DE, iterations_DE, init_adam, iterations_adam, method, seed)


class EV_one_constraint(Infill_criteria):
    """Infill_criteria.py:235-262: expected violation of one constraint model, analytic (moment-matched) or Monte-Carlo."""

    def __init__(self, zero_c, d):
        self.name = 'Expected Violation'
        self.zero_c = zero_c
        self.d = d
        self.IC_optimized = None

    def run_with_grad(self, model, x, num_samples=500, zs=None, seed=None, out=None, dx=None):
        """(EV [N, 1], d sum(EV) / dx [N, d]) for the analytic expected violation (constrained searches differentiate it)."""
        return _moment_criterion_grad(2, model, x, self.zero_c, num_samples, zs, seed, out, dx)

    def run(self, model, x, analytic=True, num_samples=100, zs=None, seed=None, out=None):
        if analytic:
            return _moment_criterion(2, model, x, self.zero_c, 500 if zs is None else num_samples, zs, seed, out=out)
        if getattr(model, "name", None) != 'dgp':
            raise NotImplementedError("only model.name == 'dgp' is on the accelerated path")
        F = model.propagate(x, S=num_samples, zs=zs, seed=seed)[0][-1]            # [S, N, D_L]
        S, N, D = F.shape
        if out is None:
            out = torch.empty((N, D), dtype=torch.float64, device=F.device)
        if N:
            _lib.get_context(F.device).call("dgp_ev_mc", _lib.ptr(F), S, N * D, _scalar(self.zero_c), _lib.ptr(out))
        return out


class EV(Infill_criteria):
    """Infill_criteria.py:264-288: expected violations of a list of constraint models side by side, and the constrained
    criterion `where(max_j EV_j > threshold, sum_j EV_j + 10000, IC)` (the reference loops tf.cond per candidate, :284-288;
    here it is one vectorised select on the device, same values)."""

    def __init__(self, zero_c, d):
        self.name = 'Expected Violation'
        self.zero_c = zero_c
        self.d = d
        self.IC_optimized = None

    def run(self, model_C, x, analytic=True, num_samples=100, zs=None, seed=None):
        cols = [EV_one_constraint(self.zero_c[i], self.d).run(model_C[i], x, analytic=analytic, num_samples=num_samples,
                                                              zs=None if zs is None else zs[i], seed=seed)
                for i in range(len(model_C))]
        return torch.cat(cols, 1)

    def run_with_IC(self, IC, model_Y, model_C, x, threshold=0.1, analytic=True, num_samples=100, seed=None):
        ev = self.run(model_C, x, analytic=analytic, num_samples=num_samples, seed=seed)
        ic = IC.run(model_Y, x, seed=seed)
        return torch.where(ev.max(dim=1, keepdim=True).values > threshold, ev.sum(dim=1, keepdim=True) + 10000.0, ic)


def _ev_optimize_with_IC(self, IC, model_Y, model_C, bounds, threshold=0.1, analytic=True, num_samples=100, popsize_DE=300,
                         popstd_DE=1.5, iterations_DE=400, init_adam=None, iterations_adam=1000, method='DE', seed=None):
    """Infill_criteria.py:290-316: minimise `run_with_IC` (the criterion where every constraint's expected violation is below
    `threshold`, sum of violations + 10000 elsewhere) over the box. 'DE' evaluates the whole population per generation; the
    'Adam' stage differentiates the branch tf.cond takes at the current point: sum_j dEV_j/dx where a violation exceeds the
    threshold, dIC/dx otherwise (analytic EV; IC needs run_with_grad: EI or WB2). The reference passes the literal 0.1 to the
    objective regardless of `threshold` (:292); the argument is honoured here."""
    if method not in ('DE', 'Adam', 'DE+Adam'):
        raise ValueError(f"unknown method {method!r}")
    d = self.d
    lw = np.broadcast_to(np.asarray(bounds[0], dtype=np.float64).reshape(-1), (d,)).copy()
    up = np.broadcast_to(np.asarray(bounds[1], dtype=np.float64).reshape(-1), (d,)).copy()
    dev = model_Y.device
    if getattr(self, "x_opt", None) is None:
        self.x_opt = None
    with search.GraphScope(dev):
        if method in ('DE', 'DE+Adam'):
            def objective(X, out):
                v = self.run_with_IC(IC, model_Y, model_C, X, threshold, analytic, num_samples)
                if out is None:
                    return v.contiguous()
                out.copy_(v)
                return out
            res = search.de_minimize(objective, lw, up, d, dev, popsize_DE, popstd_DE, iterations_DE, seed=model_Y._next_seed(seed))
            self.x_opt = res["x"].cpu().numpy().reshape(d, 1)
            self.de_iterations = res["iterations"]
            self.IC_optimized = self.run_with_IC(IC, model_Y, model_C, self.x_opt.reshape(1, d), threshold, analytic, num_samples)
        if method in ('Adam', 'DE+Adam'):
            if not analytic or not hasattr(IC, "run_with_grad"):
                raise NotImplementedError("the Adam stage needs the analytic EV and a criterion with run_with_grad (EI, WB2)")
            if init_adam is None:
                init_adam = np.zeros(d) if self.x_opt is None else self.x_opt
            init_adam = np.asarray(init_adam, dtype=np.float64).reshape(d)
            u0 = _lib.as_device(np.log((up - init_adam + 1e-3) / (init_adam - lw + 1e-3)).reshape(1, d), dev)
            ones = [EV_one_constraint(self.zero_c[i], d) for i in range(len(model_C))]

            def value_and_grad(X):
                evs = [c.run_with_grad(m, X) for c, m in zip(ones, model_C)]
                ev = torch.cat([v for v, _ in evs], 1)
                ic, dic = IC.run_with_grad(model_Y, X)
                bad = ev.max(dim=1, keepdim=True).values > threshold
                val = torch.where(bad, ev.sum(dim=1, keepdim=True) + 10000.0, ic.sum(dim=1, keepdim=True))
                dx = torch.where(bad, sum(g for _, g in evs), dic)
                return val, dx.contiguous()

            u, X, val = search.adam_box_minimize(value_and_grad, lw, up, u0, iterations_adam, lr=0.01)
            self.x_opt = X.cpu().numpy().reshape(d, 1)
            self.IC_optimized = val.clone()
    return self.x_opt


EV.optimize_with_IC = _ev_optimize_with_IC


class PoF(Infill_criteria):
    """Infill_criteria.py:318-354, repaired. The reference's `run` computes EI-style terms t1, t2 and returns nothing (:325-341),
    `run_with_IC` multiplies by the CLASS name (`-1*EI*PoF`, :345) and drops the box bounds when mapping x_opt back (:353). What the
    name and the use say: PoF(x) = P[c(x) <= zero_c] = Phi((zero_c - mean) / sigma) on the predict_y mixture moments of the
    constraint model (500 samples like the other criteria), and the constrained criterion to MINIMISE is IC(x) * PoF(x) with
    IC.run = -EI (so -EI * PoF)."""

    def __init__(self, zero_c, d):
        self.name = 'Probability of feasability'
        self.zero_c = zero_c
        self.d = d
        self.IC_optimized = None
        self.x_opt = None

    def run(self, model_C, x, num_samples=500, zs=None, seed=None, out=None):
        """P[constraint <= zero_c] per candidate -> [N, 1]."""
        return _moment_criterion(4, model_C, x, self.zero_c, num_samples, zs, seed, out=out)

    def run_with_IC(self, IC, model_Y, model_C, x, seed=None):
        return IC.run(model_Y, x, seed=seed) * self.run(model_C, x, seed=seed)

    def optimize_with_IC(self, IC, model_Y, model_C, bounds, popsize_DE=300, popstd_DE=1.5, iterations_DE=400, seed=None):
        """:346-354: differential evolution (TFP defaults of the reference: population 300 around u = 0, spread 1.5, 400 generations)
        on x = lw + (up - lw) / (1 + exp(u)); x_opt is mapped back into the box (the reference forgets lw / up there)."""
        d = self.d
        lw = np.broadcast_to(np.asarray(bounds[0], dtype=np.float64).reshape(-1), (d,)).copy()
        up = np.broadcast_to(np.asarray(bounds[1], dtype=np.float64).reshape(-1), (d,)).copy()
        with search.GraphScope(model_Y.device):
            def objective(X, out):
                v = self.run_with_IC(IC, model_Y, model_C, X)
                if out is None:
                    return v.contiguous()
                out.copy_(v)
                return out
            res = search.de_minimize(objective, lw, up, d, model_Y.device, popsize_DE, popstd_DE, iterations_DE,
                                     seed=model_Y._next_seed(seed))
            self.x_opt = res["x"].cpu().numpy().reshape(d, 1)
            self.IC_optimized = self.run_with_IC(IC, model_Y, model_C, self.x_opt.reshape(1, d))
        return self.x_opt
