"""2-objective expected hypervolume improvement with the reference's interface (dgp_dace/EHVI.py:90-157, exact
uncorrelated branch for a list of two DGPs). The moment matching and the strip sum run in libdgp_b200."""
from __future__ import annotations

import numpy as np
import torch

from . import _lib


def Y_ND(Y, ND, nadir, ideal=[0, 0]):
    """EHVI.py:90-100: the non-dominated front padded with nadir/ideal (host numpy, tens of points)."""
    Y0 = np.asarray(Y[0])[ND]
    Y1 = np.asarray(Y[1])[ND]
    Y_ = [np.zeros((len(ND) + 2, 1)), np.zeros((len(ND) + 2, 1))]
    Y_[0][1:-1] = Y0.reshape(-1, 1)
    Y_[1][1:-1] = Y1.reshape(-1, 1)
    Y_[0][0] = nadir[0]
    Y_[0][-1] = ideal[0]
    Y_[1][0] = ideal[1]
    Y_[1][-1] = nadir[1]
    return Y_


def NDC(Y, C, obj1_ascending=True):
    """EHVI.py:38-81: indices of the feasible (every constraint value <= 0), non-dominated points of the two-objective
    DoE `Y = [y0 [n,1], y1 [n,1]]`, ordered by objective 0 (ascending, ties in DoE order; descending when
    `obj1_ascending=False`). Host numpy over the DoE (tens of points): one pairwise dominance table instead of the
    reference's double loop and bubble sort."""
    y = np.concatenate((np.asarray(Y[0], dtype=np.float64).reshape(-1, 1), np.asarray(Y[1], dtype=np.float64).reshape(-1, 1)), axis=1)
    C = np.asarray(C, dtype=np.float64).reshape(len(y), -1)
    feasible = np.flatnonzero(C.max(axis=1) <= 0)
    if feasible.size == 0:
        return []
    f = y[feasible]
    le = (f[:, None, :] <= f[None, :, :]).all(-1)          # le[j, i]: point j is no worse than point i in both objectives
    lt = (f[:, None, :] < f[None, :, :]).any(-1)           # ... and strictly better in at least one
    dominated = (le & lt).any(axis=0)
    front = feasible[~dominated]
    front = front[np.argsort(y[front, 0], kind="stable")]
    nd = [int(i) for i in front]
    return nd if obj1_ascending else nd[::-1]


def HV_calcul(ND, Y, bounds):
    """EHVI.py:8-36: hypervolume (minimisation) of the front `ND` (sorted by objective 0 ascending) w.r.t. the reference
    point (U1, U2); strips are added front point by front point exactly as the reference does, including its treatment
    of points beyond the reference point."""
    _, _, U1, U2 = bounds
    if len(ND) == 0:
        return 0
    y1 = np.asarray(Y[0], dtype=np.float64).reshape(-1)[list(ND)]
    y2 = np.asarray(Y[1], dtype=np.float64).reshape(-1)[list(ND)]
    if np.any((y1 > U1) & (y2 > U2)):
        return 0
    hv = max((U1 - y1[0]) * (U2 - y2[0]), 0.0)
    nxt1, nxt2, prev2 = y1[1:], y2[1:], y2[:-1]
    outside = (nxt1 > U1) | (nxt2 > U2)
    first_inside = (nxt2 <= U2) & (prev2 > U2)
    height = np.where(first_inside, U2 - nxt2, prev2 - nxt2)
    return float(hv + np.sum(np.where(outside, 0.0, height * (U1 - nxt1))))


def psi(a, b, mu, sigma):
    """EHVI.py:102-104 on tensors (helper for callers; the EHVI kernel evaluates it in-kernel)."""
    u = (b - mu) / sigma
    pdf = torch.exp(-0.5 * u * u) / np.sqrt(2 * np.pi)
    cdf = 0.5 * torch.erfc(-u / np.sqrt(2.0))
    return sigma * pdf + (a - mu) * cdf


def _is_mo(model_Y):
    return not isinstance(model_Y, list) and getattr(model_Y, "name", None) == 'mo_dgp'


def _mo_ehvi_with_grad(model_Y, Xcand, YND, S):
    """EHVI_with_grad for the multi-objective object: the chain is differentiated by torch.autograd through the library's layer /
    kernel adjoints (models/MO_DGP.py), the criterion's partial derivatives w.r.t. the four moments come from dgp_ehvi2d_grad."""
    m = model_Y.model
    dev = m.device
    X = _lib.as_device(Xcand, dev).detach().clone().requires_grad_(True)
    N = X.shape[0]
    _, Fmeans, Fvars = m.propagate(X, S=S)
    mom = []
    for o in (-2, -1):     # EHVI.py:126-130, with the centred variance of dgp_mixture_moments (no cancellation at large |mean|)
        mu = Fmeans[o].mean(0)
        mom += [mu.reshape(-1), (Fvars[o].mean(0) + ((Fmeans[o] - mu) ** 2).mean(0)).reshape(-1)]
    val = torch.empty((N, 1), dtype=torch.float64, device=dev)
    g = torch.empty((N, 4), dtype=torch.float64, device=dev)
    y0 = _lib.as_device(np.asarray(YND[0], dtype=np.float64).reshape(-1), dev)
    y1 = _lib.as_device(np.asarray(YND[1], dtype=np.float64).reshape(-1), dev)
    d = [t.detach().contiguous() for t in mom]
    _lib.get_context(dev).call("dgp_ehvi2d_grad", _lib.ptr(d[0]), _lib.ptr(d[1]), _lib.ptr(d[2]), _lib.ptr(d[3]), N, _lib.ptr(y0),
                               _lib.ptr(y1), int(y0.numel()), _lib.ptr(val), _lib.ptr(g))
    dx, = torch.autograd.grad(mom, X, grad_outputs=[-g[:, k].contiguous() for k in range(4)])
    return -val, dx


def EHVI(model_Y, Xcand, YND, corr=False, approximation='None', S=1000, zs=None, seed=None):
    """EHVI.py:107-157, approximation='None', corr=False -> [N, 1], for `model_Y` = [dgp0, dgp1] (:110-119) or a multi-objective
    DGP object (`name == 'mo_dgp'`, :124-130: both objectives' moments from ONE chain of `model_Y.model`)."""
    if approximation != 'None' or corr:
        raise NotImplementedError("only the exact uncorrelated EHVI is on the accelerated path")
    if _is_mo(model_Y):
        (m0, v0), (m1, v1) = model_Y.model.mixture_moments(Xcand, S)
    else:
        if not isinstance(model_Y, list) or len(model_Y) != 2 or any(getattr(m, "name", None) != 'dgp' for m in model_Y):
            raise NotImplementedError("a list of two DGP models or a MultiObjDeepGP is expected (SURVEY §8 a12)")
        zs = zs or [None, None]
        seeds = seed if isinstance(seed, (list, tuple)) else [seed, seed]
        # moment matching over the S propagated samples (EHVI.py:112-119), predict_f moments (no likelihood variance)
        m0, v0 = model_Y[0].predict_moments(Xcand, S, add_lik_var=False, zs=zs[0], seed=seeds[0])
        m1, v1 = model_Y[1].predict_moments(Xcand, S, add_lik_var=False, zs=zs[1], seed=seeds[1])
        if m0.shape[1] != 1 or m1.shape[1] != 1:
            raise ValueError("each objective model must have one output")
    N = m0.shape[0]
    dev = m0.device
    y0 = _lib.as_device(np.asarray(YND[0], dtype=np.float64).reshape(-1), dev)
    y1 = _lib.as_device(np.asarray(YND[1], dtype=np.float64).reshape(-1), dev)
    out = torch.empty((N, 1), dtype=torch.float64, device=dev)
    if N == 0:
        return out
    _lib.get_context(dev).call("dgp_ehvi2d", _lib.ptr(m0), _lib.ptr(v0), _lib.ptr(m1), _lib.ptr(v1), N, _lib.ptr(y0),
                               _lib.ptr(y1), int(y0.numel()), _lib.ptr(out))
    return out


def EHVI_with_grad(model_Y, Xcand, YND, S=1000, zs=None, seed=None):
    """(-EHVI [N, 1], d sum(-EHVI) / dX [N, d]) for `model_Y` = [dgp0, dgp1]: the value and gradient the Adam stage of optimize_EHVI
    (EHVI.py:218-234) takes with tf.GradientTape. One propagation per model for the moments, dgp_ehvi2d_grad for the criterion and its
    partial derivatives w.r.t. the four moments, then one adjoint chain per model (dgp_acq_grad kind 4) with the SAME draws."""
    import ctypes as C
    if _is_mo(model_Y):
        return _mo_ehvi_with_grad(model_Y, Xcand, YND, S)
    if not isinstance(model_Y, list) or len(model_Y) != 2 or any(getattr(m, "name", None) != 'dgp' for m in model_Y):
        raise NotImplementedError("a list of two DGP models is expected")
    dev = model_Y[0].device
    X = model_Y[0]._check_X(_lib.as_device(Xcand, dev))
    N = X.shape[0]
    zs = zs or [None, None]
    seeds = list(seed) if isinstance(seed, (list, tuple)) else [seed, seed]
    seeds = [model_Y[k]._next_seed(seeds[k]) for k in range(2)]     # fixed here: the adjoint chain must see the draws of the forward
    mom = [model_Y[k].predict_moments(X, S, add_lik_var=False, zs=zs[k], seed=seeds[k]) for k in range(2)]
    if any(m.shape[1] != 1 for m, _ in mom):
        raise ValueError("each objective model must have one output")
    val = torch.empty((N, 1), dtype=torch.float64, device=dev)
    dx = torch.zeros_like(X)
    if N == 0:
        return val, dx
    y0 = _lib.as_device(np.asarray(YND[0], dtype=np.float64).reshape(-1), dev)
    y1 = _lib.as_device(np.asarray(YND[1], dtype=np.float64).reshape(-1), dev)
    g = torch.empty((N, 4), dtype=torch.float64, device=dev)
    ctx = _lib.get_context(dev)
    ctx.call("dgp_ehvi2d_grad", _lib.ptr(mom[0][0]), _lib.ptr(mom[0][1]), _lib.ptr(mom[1][0]), _lib.ptr(mom[1][1]), N, _lib.ptr(y0),
             _lib.ptr(y1), int(y0.numel()), _lib.ptr(val), _lib.ptr(g))
    for k in range(2):
        ext = (-g[:, 2 * k:2 * k + 2]).contiguous()                 # adjoints of -EHVI w.r.t. (mean, var) of objective k
        dxk = torch.empty_like(X)
        m, keep = model_Y[k]._model_desc()
        zt, zp = model_Y[k]._zs(zs[k], S, N)
        ctx.call("dgp_acq_grad", C.byref(m), 4, _lib.ptr(X), N, S, zp, seeds[k], 0, 0.0, _lib.ptr(ext), _lib.ptr(dxk))
        dx += dxk
    return -val, dx


def EI_and_EHVI(model_Y, Xcand, YND, y_min, S=1000, zs=None, seed=None):
    """-EI of objective 0 (EI.run analytic, Infill_criteria.py:36-47) and the exact EHVI of both objectives (EHVI.py:107-157) for the
    same candidates from ONE propagation per model: both criteria moment-match the same predict_f samples of model 0, so a
    4 M-candidate sweep that wants both (BASELINE config 5) does two chains per chunk instead of three. Returns ([N,1], [N,1])."""
    if not isinstance(model_Y, list) or len(model_Y) != 2 or any(getattr(m, "name", None) != 'dgp' for m in model_Y):
        raise NotImplementedError("a list of two DGP models is expected")
    zs = zs or [None, None]
    seeds = seed if isinstance(seed, (list, tuple)) else [seed, seed]
    m0, v0 = model_Y[0].predict_moments(Xcand, S, add_lik_var=False, zs=zs[0], seed=seeds[0])
    m1, v1 = model_Y[1].predict_moments(Xcand, S, add_lik_var=False, zs=zs[1], seed=seeds[1])
    N, dev = m0.shape[0], m0.device
    ei = torch.empty((N, 1), dtype=torch.float64, device=dev)
    out = torch.empty((N, 1), dtype=torch.float64, device=dev)
    if N == 0:
        return ei, out
    y0 = _lib.as_device(np.asarray(YND[0], dtype=np.float64).reshape(-1), dev)
    y1 = _lib.as_device(np.asarray(YND[1], dtype=np.float64).reshape(-1), dev)
    ctx = _lib.get_context(dev)
    ctx.call("dgp_acq_moments", 0, _lib.ptr(m0), _lib.ptr(v0), N, float(y_min), None, 0, _lib.ptr(ei))
    ctx.call("dgp_ehvi2d", _lib.ptr(m0), _lib.ptr(v0), _lib.ptr(m1), _lib.ptr(v1), N, _lib.ptr(y0), _lib.ptr(y1), int(y0.numel()),
             _lib.ptr(out))
    return ei, out


def optimize_EHVI(model, YND, popsize_DE=300, popstd_DE=1.5, iterations_DE=400, init_adam=None, lr_adam=0.01, iterations_adam=1000,
                  method='DE', corr=False, approximation='None', S=1000, seed=None, bounds=(0.0, 1.0)):
    """EHVI.py:208-235 for `model` = [dgp0, dgp1] (the two-DGP list path of EHVI()): search the box for the candidate with the
    largest expected hypervolume improvement. As written the reference (i) passes population_size / population_stddev swapped
    (:217-218), (ii) MINIMISES the positive EHVI (:212), (iii) reads the input dimension from the MO-DGP object (`model._X`, :210) and
    (iv) discards the DE result before the Adam stage (`x_opt = np.array([[0]])`, :221). Implemented here is the evident intent:
    differential evolution (rand/1/bin, TFP defaults) on u with x = lw + (up - lw) / (1 + exp(u)) minimising -EHVI, every
    generation one EHVI evaluation of the whole population on the device; then (method 'Adam' / 'DE+Adam') Keras Adam on u started
    from the DE result (or `init_adam`, or zeros as in the reference), with the gradient of -EHVI w.r.t. the candidate from EHVI_with_grad
    (fresh draws every step, like the reference's loss). `model` may also be the multi-objective object (`MultiObjDeepGP`, the case
    the reference's `model._X` was written for). Returns x_opt [d, 1] like the reference."""
    from . import search
    mo = _is_mo(model)
    if not mo and (not isinstance(model, list) or len(model) != 2):
        raise NotImplementedError("optimize_EHVI expects a list of two DGP models or a MultiObjDeepGP")
    if method not in ('DE', 'Adam', 'DE+Adam'):
        raise ValueError(f"unknown method {method!r}")
    if corr or approximation != 'None':
        raise NotImplementedError("only the exact uncorrelated EHVI is on the accelerated path")
    d = model._X[0].shape[1] if mo else model[0].layers[0].feature.Z.shape[1]     # EHVI.py:210
    lw = np.broadcast_to(np.asarray(bounds[0], dtype=np.float64).reshape(-1), (d,)).copy()
    up = np.broadcast_to(np.asarray(bounds[1], dtype=np.float64).reshape(-1), (d,)).copy()
    dev = model.model.device if mo else model[0].device
    first = model.model if mo else model[0]
    x_opt = None
    if method in ('DE', 'DE+Adam'):
        import contextlib
        with (contextlib.nullcontext() if mo else search.GraphScope(dev)):     # the MO chain is host-chained library calls: no replay
            def objective(X, out):
                v = -EHVI(model, X, YND, corr=corr, approximation=approximation, S=S)
                if out is None:
                    return v.contiguous()
                out.copy_(v)
                return out
            res = search.de_minimize(objective, lw, up, d, dev, popsize_DE, popstd_DE, iterations_DE,
                                     seed=(0 if seed is None else int(seed)) if mo else first._next_seed(seed))
        x_opt = res["x"].cpu().numpy().reshape(d)
    if method in ('Adam', 'DE+Adam'):
        if init_adam is None:
            init_adam = np.zeros(d) if x_opt is None else x_opt     # the reference's default start ([0.] * d, EHVI.py:222)
        init_adam = np.asarray(init_adam, dtype=np.float64).reshape(d)
        u0 = _lib.as_device(np.log((up - init_adam + 1e-3) / (init_adam - lw + 1e-3)).reshape(1, d), dev)
        _, X, _ = search.adam_box_minimize(lambda X: EHVI_with_grad(model, X, YND, S=S), lw, up, u0, iterations_adam, lr=lr_adam)
        x_opt = X.cpu().numpy().reshape(d)
    _lib.get_context(dev).check()
    return x_opt.reshape(d, 1)
