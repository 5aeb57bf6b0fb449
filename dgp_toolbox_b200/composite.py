"""Composite kernels with `active_dims` and SVGP layers on supplied kernel matrices (SURVEY §8 f2) — what the reference's
multi-fidelity model is built from (dgp_dace/models/MF_DGP.py:262-290):

    k_l = k_corr * (k_prev + Linear) + k_in  (+ White)       k_corr, k_in on the input columns, k_prev / Linear on the previous fidelity's output

GPflow-style kernel algebra (`RBF(active_dims=…) * (RBF(…) + Linear(…)) + RBF(…) + White(…)`) is recognised and lowered to ONE
library descriptor (`dgp_comp_kernel`); K, K_diag and their adjoints are the library's CUDA kernels (`csrc/compkern.cuh`), the
layer's conditional / KL and their adjoints run on the supplied matrices in the library's DMMA GEMM pipeline (`dgp_svgp_from_k`,
`dgp_svgp_from_k_grad`). torch.autograd only chains these calls (concatenations, means over samples, sums): plumbing.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from .gpflow_shim import Parameter, SquaredExponential, _Module

THETA = 7   # in_var, corr_var, corr_ls, prev_var, prev_ls, lin_var, white_var, then in_ls[...]


class CompKernelDesc(C.Structure):
    _fields_ = [("D", C.c_int32), ("Da", C.c_int32), ("has_prod", C.c_int32), ("has_linear", C.c_int32), ("in_ard", C.c_int32),
                ("in_variance", C.c_void_p), ("in_lengthscales", C.c_void_p), ("corr_variance", C.c_void_p),
                ("corr_lengthscale", C.c_void_p), ("prev_variance", C.c_void_p), ("prev_lengthscale", C.c_void_p),
                ("lin_variance", C.c_void_p), ("white_variance", C.c_void_p)]


# ---------------------------------------------------------------------------------------------- kernel algebra (gpflow.kernels)
class _KernelOps:
    def __add__(self, other):
        return Sum([self, other])

    def __mul__(self, other):
        return Product([self, other])


class RBF(SquaredExponential, _KernelOps):
    """gpflow.kernels.RBF with `active_dims` (a list of input columns)."""

    def __init__(self, variance=1.0, lengthscales=1.0, active_dims=None, name=None):
        SquaredExponential.__init__(self, variance, lengthscales, None, name)
        self.active_dims = None if active_dims is None else [int(i) for i in active_dims]


class LinearKernel(_Module, _KernelOps):
    """gpflow.kernels.Linear: variance * <x, y> on `active_dims`."""

    def __init__(self, variance=1.0, active_dims=None, name=None):
        self.variance = Parameter(np.asarray(variance, dtype=np.float64).reshape(()), transform="positive", name="variance")
        self.active_dims = None if active_dims is None else [int(i) for i in active_dims]


class White(_Module, _KernelOps):
    """gpflow.kernels.White: variance * I for K(X) and K_diag, zero for K(X, X2)."""

    def __init__(self, variance=1.0, active_dims=None, name=None):
        self.variance = Parameter(np.asarray(variance, dtype=np.float64).reshape(()), transform="positive", name="variance")
        self.active_dims = None


class _Combination(_Module, _KernelOps):
    def __init__(self, kernels):
        flat = []
        for k in kernels:
            flat.extend(k.kernels if isinstance(k, type(self)) else [k])      # GPflow flattens nested combinations of one type
        self.kernels = flat


class Sum(_Combination):
    pass


class Product(_Combination):
    pass


Linear = LinearKernel


def lower(kern, D):
    """GPflow kernel tree -> dict of the roles of the library's composite kernel, or NotImplementedError.
    Accepted shapes (MF_DGP.py:266-290): RBF_a [+ White]  and  RBF_a * (RBF_b [+ Linear_b]) + RBF_a [+ White]."""
    terms = kern.kernels if isinstance(kern, Sum) else [kern]
    white = [t for t in terms if isinstance(t, White)]
    rbfs = [t for t in terms if isinstance(t, SquaredExponential)]
    prods = [t for t in terms if isinstance(t, Product)]
    if len(white) > 1 or len(rbfs) != 1 or len(prods) > 1 or len(white) + len(rbfs) + len(prods) != len(terms):
        raise NotImplementedError("composite kernel: expected RBF [+ RBF * (RBF [+ Linear])] [+ White]")
    k_in = rbfs[0]
    a = list(range(D)) if getattr(k_in, "active_dims", None) is None else list(k_in.active_dims)
    if a != list(range(len(a))):
        raise NotImplementedError("composite kernel: k_in must act on the leading input columns")
    roles = dict(D=D, Da=len(a), k_in=k_in, white=white[0] if white else None, k_corr=None, k_prev=None, lin=None)
    if prods:
        fac = prods[0].kernels
        if len(fac) != 2 or not isinstance(fac[0], SquaredExponential):
            raise NotImplementedError("composite kernel: the product must be RBF * (RBF [+ Linear])")
        inner = fac[1].kernels if isinstance(fac[1], Sum) else [fac[1]]
        prev = [t for t in inner if isinstance(t, SquaredExponential)]
        lin = [t for t in inner if isinstance(t, LinearKernel)]
        b = list(range(len(a), D))
        if len(prev) != 1 or len(lin) > 1 or len(prev) + len(lin) != len(inner) or list(getattr(fac[0], "active_dims", None) or []) != a \
                or list(getattr(prev[0], "active_dims", None) or []) != b or (lin and list(lin[0].active_dims or []) != b):
            raise NotImplementedError("composite kernel: k_corr on the input columns, k_prev / Linear on the remaining ones")
        for kk in (fac[0], prev[0]):
            if kk.lengthscales.value.numel() != 1:
                raise NotImplementedError("composite kernel: k_corr and k_prev are isotropic (one lengthscale), as the reference builds them")
        roles.update(k_corr=fac[0], k_prev=prev[0], lin=lin[0] if lin else None)
    elif len(a) != D:
        raise NotImplementedError("composite kernel: without a product part k_in must cover every column")
    return roles


ROLE_PARAMS = ("in_var", "in_ls", "corr_var", "corr_ls", "prev_var", "prev_ls", "lin_var", "white_var")


def role_parameters(roles):
    """The Parameter objects behind the eight descriptor slots (None where the role is absent)."""
    k_in, kc, kp, lin, w = roles["k_in"], roles["k_corr"], roles["k_prev"], roles["lin"], roles["white"]
    return dict(in_var=k_in.variance, in_ls=k_in.lengthscales, corr_var=kc.variance if kc else None, corr_ls=kc.lengthscales if kc else None,
                prev_var=kp.variance if kp else None, prev_ls=kp.lengthscales if kp else None, lin_var=lin.variance if lin else None,
                white_var=w.variance if w else None)


def _desc(roles, th):
    """th: dict role -> contiguous float64 CUDA tensor (or None)."""
    d = CompKernelDesc()
    d.D, d.Da = roles["D"], roles["Da"]
    d.has_prod = 1 if roles["k_corr"] is not None else 0
    d.has_linear = 1 if roles["lin"] is not None else 0
    d.in_ard = 1 if th["in_ls"].numel() > 1 else 0
    if d.in_ard and th["in_ls"].numel() != d.Da:
        raise ValueError("k_in: one lengthscale per active column expected")
    p = lambda t: None if t is None else t.data_ptr()
    d.in_variance, d.in_lengthscales = p(th["in_var"]), p(th["in_ls"])
    d.corr_variance, d.corr_lengthscale = p(th["corr_var"]), p(th["corr_ls"])
    d.prev_variance, d.prev_lengthscale = p(th["prev_var"]), p(th["prev_ls"])
    d.lin_variance, d.white_variance = p(th["lin_var"]), p(th["white_var"])
    return d


def _theta_grads(roles, th, dtheta):
    """dtheta (library layout) -> gradient per role tensor, shaped like it."""
    slot = dict(in_var=0, corr_var=1, corr_ls=2, prev_var=3, prev_ls=4, lin_var=5, white_var=6)
    out = []
    for r in ROLE_PARAMS:
        t = th[r]
        if t is None:
            out.append(None)
        elif r == "in_ls":
            out.append(dtheta[THETA:THETA + t.numel()].reshape(t.shape).clone())
        else:
            out.append(dtheta[slot[r]].reshape(t.shape).clone())
    return out


class CompK(torch.autograd.Function):
    """kern.K(X, X2) through dgp_comp_K / dgp_comp_K_grad."""

    @staticmethod
    def forward(ctx, roles, X, X2, *theta):
        th = {r: (None if t is None else t.detach().contiguous()) for r, t in zip(ROLE_PARAMS, theta)}
        X = X.detach().contiguous()
        X2c = None if X2 is None else X2.detach().contiguous()
        out = torch.empty((X.shape[0], (X if X2c is None else X2c).shape[0]), dtype=torch.float64, device=X.device)
        d = _desc(roles, th)
        _lib.get_context(X.device).call("dgp_comp_K", C.byref(d), _lib.ptr(X), X.shape[0], None if X2c is None else _lib.ptr(X2c),
                                        0 if X2c is None else X2c.shape[0], _lib.ptr(out))
        ctx.roles, ctx.th, ctx.X, ctx.X2 = roles, th, X, X2c
        return out

    @staticmethod
    def backward(ctx, Kbar):
        roles, th, X, X2 = ctx.roles, ctx.th, ctx.X, ctx.X2
        Kbar = Kbar.contiguous()
        dX = torch.empty_like(X)
        dX2 = None if X2 is None else torch.empty_like(X2)
        nt = THETA + th["in_ls"].numel()
        dth = torch.empty(nt, dtype=torch.float64, device=X.device)
        d = _desc(roles, th)
        _lib.get_context(X.device).call("dgp_comp_K_grad", C.byref(d), _lib.ptr(X), X.shape[0], None if X2 is None else _lib.ptr(X2),
                                        0 if X2 is None else X2.shape[0], _lib.ptr(Kbar), _lib.ptr(dX), None if X2 is None else _lib.ptr(dX2),
                                        _lib.ptr(dth))
        return (None, dX, dX2) + tuple(_theta_grads(roles, th, dth))


class CompKdiag(torch.autograd.Function):
    """kern.K_diag(X) through dgp_comp_Kdiag / dgp_comp_Kdiag_grad."""

    @staticmethod
    def forward(ctx, roles, X, *theta):
        th = {r: (None if t is None else t.detach().contiguous()) for r, t in zip(ROLE_PARAMS, theta)}
        X = X.detach().contiguous()
        out = torch.empty(X.shape[0], dtype=torch.float64, device=X.device)
        d = _desc(roles, th)
        _lib.get_context(X.device).call("dgp_comp_Kdiag", C.byref(d), _lib.ptr(X), X.shape[0], _lib.ptr(out))
        ctx.roles, ctx.th, ctx.X = roles, th, X
        return out

    @staticmethod
    def backward(ctx, g):
        roles, th, X = ctx.roles, ctx.th, ctx.X
        g = g.contiguous()
        dX = torch.empty_like(X)
        dth = torch.empty(THETA + th["in_ls"].numel(), dtype=torch.float64, device=X.device)
        d = _desc(roles, th)
        _lib.get_context(X.device).call("dgp_comp_Kdiag_grad", C.byref(d), _lib.ptr(X), X.shape[0], _lib.ptr(g), _lib.ptr(dX), _lib.ptr(dth))
        grads = _theta_grads(roles, th, dth)
        grads[1] = None if th["in_ls"] is None else torch.zeros_like(th["in_ls"])      # K_diag does not depend on the lengthscales
        return (None, dX) + tuple(grads)


class PrepCache:
    """Device buffer for the replicated per-evaluation work of one layer (dgp_svgp_from_k_cached): valid while Ku, q_mu and q_sqrt
    keep their values, i.e. for all applications of a layer inside ONE ELBO evaluation and their adjoints."""

    def __init__(self, M, D_out, device):
        ctx = _lib.get_context(device)
        self.nbytes = int(_lib.lib.dgp_svgp_prep_cache_bytes(ctx.h, int(M), int(D_out)))
        if self.nbytes <= 0:
            raise _lib.DGPError(f"dgp_svgp_prep_cache_bytes({M}, {D_out}) failed: {_lib.lib.dgp_last_error(ctx.h).decode()}")
        self.buf = torch.empty((self.nbytes + 7) // 8, dtype=torch.float64, device=device)
        self.filled = False
        self.budget = None       # [bytes left] for the forward-plane stashes of this ELBO evaluation, shared by all its layers


def stash_budget_bytes():
    """Device memory one ELBO evaluation may spend on keeping the A / T_d planes of its layer applications for their adjoints
    (env DGP_B200_STASH_GB, default 48): applications beyond it recompute the planes in the adjoint call, as the uncached path does."""
    import os
    return int(float(os.environ.get("DGP_B200_STASH_GB", "48")) * (1 << 30))


EVAL_CACHE = "_eval_cache"      # key of the per-evaluation cache dict inside a `values` dict (models/MF_DGP.py: MFLayer.conditional_ND)


class SVGPFromK(torch.autograd.Function):
    """(mean [P, D], var [P, D], kl) of SVGP_Layer.conditional_ND + KL (utils/layers.py:237-308) on supplied Ku = Kuu + jitter I,
    Kuf, Kdiag: dgp_svgp_from_k / dgp_svgp_from_k_grad, or their `_cached` forms when the caller supplies a PrepCache."""

    @staticmethod
    def forward(ctx, Ku, Kuf, Kdiag, q_mu, q_sqrt, cache=None):
        Ku, Kuf, Kdiag, q_mu, q_sqrt = [t.detach().contiguous() for t in (Ku, Kuf, Kdiag, q_mu, q_sqrt)]
        M, P, D = Ku.shape[0], Kuf.shape[1], q_mu.shape[1]
        mean = torch.empty((P, D), dtype=torch.float64, device=Ku.device)
        var = torch.empty_like(mean)
        kl = torch.empty(1, dtype=torch.float64, device=Ku.device)
        if cache is None:
            _lib.get_context(Ku.device).call("dgp_svgp_from_k", M, D, P, _lib.ptr(Ku), _lib.ptr(Kuf), _lib.ptr(Kdiag), _lib.ptr(q_mu),
                                             _lib.ptr(q_sqrt), _lib.ptr(mean), _lib.ptr(var), _lib.ptr(kl))
        else:
            stash = None
            if cache.budget is not None and any(ctx.needs_input_grad):
                nb = int(_lib.lib.dgp_svgp_stash_bytes(M, D, P))
                if 0 < nb <= cache.budget[0]:
                    cache.budget[0] -= nb
                    stash = torch.empty(nb // 8, dtype=torch.float64, device=Ku.device)
            _lib.get_context(Ku.device).call("dgp_svgp_from_k_cached", M, D, P, _lib.ptr(Ku), _lib.ptr(Kuf), _lib.ptr(Kdiag),
                                             _lib.ptr(q_mu), _lib.ptr(q_sqrt), _lib.ptr(mean), _lib.ptr(var), _lib.ptr(kl),
                                             _lib.ptr(cache.buf), cache.nbytes, 1 if cache.filled else 0, _lib.ptr(stash))
            cache.filled = True
            ctx.stash = stash
        ctx.cache = cache
        ctx.save_for_backward(Ku, Kuf, Kdiag, q_mu, q_sqrt)
        return mean, var, kl.reshape(())

    @staticmethod
    def backward(ctx, gmean, gvar, gkl):
        Ku, Kuf, Kdiag, q_mu, q_sqrt = ctx.saved_tensors
        cache = ctx.cache
        M, P, D = Ku.shape[0], Kuf.shape[1], q_mu.shape[1]
        gmean = torch.zeros((P, D), dtype=torch.float64, device=Ku.device) if gmean is None else gmean.contiguous()
        gvar = torch.zeros((P, D), dtype=torch.float64, device=Ku.device) if gvar is None else gvar.contiguous()
        dKu, dKuf, dKdiag = torch.empty_like(Ku), torch.empty_like(Kuf), torch.empty_like(Kdiag)
        dq_mu, dq_sqrt = torch.empty_like(q_mu), torch.empty_like(q_sqrt)
        args = (M, D, P, _lib.ptr(Ku), _lib.ptr(Kuf), _lib.ptr(Kdiag), _lib.ptr(q_mu), _lib.ptr(q_sqrt), _lib.ptr(gmean), _lib.ptr(gvar),
                float(gkl) if gkl is not None else 0.0, _lib.ptr(dKu), _lib.ptr(dKuf), _lib.ptr(dKdiag), _lib.ptr(dq_mu), _lib.ptr(dq_sqrt))
        if cache is None:
            _lib.get_context(Ku.device).call("dgp_svgp_from_k_grad", *args)
        else:
            _lib.get_context(Ku.device).call("dgp_svgp_from_k_grad_cached", *args, _lib.ptr(cache.buf), cache.nbytes, _lib.ptr(ctx.stash))
            ctx.stash = None
        return dKu, dKuf, dKdiag, dq_mu, dq_sqrt, None


def _no_adjoint(name, tensors):
    if torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors):
        raise NotImplementedError(f"{name}: the full_cov=True path has no adjoint; call it on tensors that do not require grad")


def comp_K_blocks(roles, X, *theta):
    """kern.K(X_b, X_b) [B, N, N] for X [B, N, D] (White on each block's diagonal) through dgp_comp_K_blocks: one launch for all
    blocks. Forward only."""
    _no_adjoint("comp_K_blocks", (X,) + theta)
    th = {r: (None if t is None else t.detach().contiguous()) for r, t in zip(ROLE_PARAMS, theta)}
    X = X.detach().contiguous()
    B, N = X.shape[0], X.shape[1]
    out = torch.empty((B, N, N), dtype=torch.float64, device=X.device)
    d = _desc(roles, th)
    _lib.get_context(X.device).call("dgp_comp_K_blocks", C.byref(d), _lib.ptr(X), B, N, _lib.ptr(out))
    return out


def svgp_from_k_full_cov(Ku, Kuf, Kff, q_mu, q_sqrt, z, jitter):
    """SVGP_Layer.conditional_ND(full_cov=True) per sample + reparameterize(full_cov=True) (utils/layers.py:76-80,264-268,276;
    utils/utils.py:43-52) on supplied Ku = Kuu + jitter I [M, M], Kuf [M, S*N] (column s*N + n), Kff [1 or S, N, N], draws z
    [S, N, D_out] through dgp_svgp_from_k_full_cov -> (F [S, N, D_out], mean [S, N, D_out], cov [S, N, N, D_out]). Forward only:
    raises NotImplementedError when an input requires grad."""
    _no_adjoint("svgp_from_k_full_cov", (Ku, Kuf, Kff, q_mu, q_sqrt, z))
    Ku, Kuf, Kff, q_mu, q_sqrt, z = [t.detach().contiguous() for t in (Ku, Kuf, Kff, q_mu, q_sqrt, z)]
    S, N, D = z.shape
    M = Ku.shape[0]
    if Kuf.shape != (M, S * N) or Kff.shape[1:] != (N, N) or q_mu.shape != (M, D):
        raise ValueError(f"svgp_from_k_full_cov: shapes Ku {tuple(Ku.shape)}, Kuf {tuple(Kuf.shape)}, Kff {tuple(Kff.shape)}, "
                         f"q_mu {tuple(q_mu.shape)}, z {tuple(z.shape)} do not fit together")
    mean = torch.empty((S, N, D), dtype=torch.float64, device=Ku.device)
    cov = torch.empty((S, N, N, D), dtype=torch.float64, device=Ku.device)
    F = torch.empty_like(mean)
    _lib.get_context(Ku.device).call("dgp_svgp_from_k_full_cov", M, D, N, S, _lib.ptr(Ku), _lib.ptr(Kuf), _lib.ptr(Kff), Kff.shape[0],
                                     _lib.ptr(q_mu), _lib.ptr(q_sqrt), _lib.ptr(z), float(jitter), _lib.ptr(mean), _lib.ptr(cov),
                                     _lib.ptr(F))
    return F, mean, cov


class CompositeKernelEval:
    """K / K_diag of a lowered kernel on leaf tensors `th` (dict role -> tensor): differentiable through the library's adjoints."""

    def __init__(self, kern, D):
        self.roles = lower(kern, D)
        self.params = role_parameters(self.roles)

    def leaves(self, values):
        """values: dict Parameter -> tensor to use for it (e.g. autograd leaves); defaults to the parameter's own value."""
        return [None if p is None else values.get(p, p.value) for p in (self.params[r] for r in ROLE_PARAMS)]

    def K(self, X, X2=None, values=None):
        return CompK.apply(self.roles, X, X2, *self.leaves(values or {}))

    def K_diag(self, X, values=None):
        return CompKdiag.apply(self.roles, X, *self.leaves(values or {}))

    def K_blocks(self, X, values=None):
        """K(X_b, X_b) [B, N, N] for X [B, N, D]; forward only (the full_cov=True path)."""
        return comp_K_blocks(self.roles, X, *self.leaves(values or {}))
