"""Float64 CPU reference for the composite-kernel layer path (TEST INFRASTRUCTURE, NOT PRODUCT).

Two library operations, written directly in torch so that autograd supplies every adjoint:
  * comp_K / comp_Kdiag: the multi-fidelity kernel of the reference's MF / MO models (MF_DGP.py:262-290)
        k(x, y) = k_corr(x_a, y_a) * (k_prev(x_b, y_b) + s_l^2 <x_b, y_b>) + k_in(x_a, y_a)      (+ s_w^2 I for K(X) / K_diag)
    a = the first Da columns, b = the rest; k_corr, k_prev isotropic RBF, k_in RBF (ARD or isotropic). The library's kernels are
    dgp_comp_K / dgp_comp_Kdiag and their adjoints (csrc/compkern.cuh).
  * svgp_from_k: the SVGP layer's conditional and KL on supplied Ku = Kuu + jitter I, Kuf, K_diag, in the op order of
    dgp_oracle.conditional_ND (utils/layers.py:237-278) and dgp_oracle.layer_KL (:280-308). The library's calls are
    dgp_svgp_from_k / dgp_svgp_from_k_grad (csrc/extk.cuh and svgp_from_k_run).

Kernel parameters are a dict keyed by the library's role names (ROLES); a role that is absent is None or missing:
has_prod <=> corr_var is given, has_linear <=> lin_var is given, in_ard <=> in_ls has more than one entry, White <=> white_var.

The *_vjp functions are the chunked adjoints for large P (they build their own autograd graphs, so they also work with grad
mode off, e.g. inside the backward of an autograd.Function). Per-column results (K, mean, var, dKuf, dKdiag, dX2) are computed chunk
by chunk; the sums over columns (dKu, dq_mu, dq_sqrt, dX, d theta) are accumulated chunk by chunk, as
dgp_oracle.elbo_and_grads_chunked does, so no whole-P autograd graph is ever held.
"""
from __future__ import annotations

import torch

DTYPE = torch.float64
ROLES = ("in_var", "in_ls", "corr_var", "corr_ls", "prev_var", "prev_ls", "lin_var", "white_var")


def _sqdist(A, B):
    """sum_k (A_ik - B_jk)^2 in difference form (no cancellation for close points)."""
    return ((A[:, None, :] - B[None, :, :]) ** 2).sum(-1)


def _get(th, r):
    return th.get(r) if th is not None else None


# ------------------------------------------------------------------------------------------------------------------ composite kernel
def comp_K(X, X2, Da, th):
    """K(X, X2) [P, P2]; X2 None: K(X, X) with the White variance on the diagonal."""
    Y = X if X2 is None else X2
    a, ya = X[:, :Da], Y[:, :Da]
    K = th["in_var"] * torch.exp(-0.5 * _sqdist(a / th["in_ls"], ya / th["in_ls"]))
    if _get(th, "corr_var") is not None:
        b, yb = X[:, Da:], Y[:, Da:]
        kc = th["corr_var"] * torch.exp(-0.5 * _sqdist(a, ya) / th["corr_ls"] ** 2)
        inner = th["prev_var"] * torch.exp(-0.5 * _sqdist(b, yb) / th["prev_ls"] ** 2)
        if _get(th, "lin_var") is not None:
            inner = inner + th["lin_var"] * (b @ yb.T)
        K = kc * inner + K
    if X2 is None and _get(th, "white_var") is not None:
        K = K + th["white_var"] * torch.eye(X.shape[0], dtype=DTYPE)
    return K


def comp_Kdiag(X, Da, th):
    """K_diag(X) [P]: k(x, x) + White."""
    v = th["in_var"] * torch.ones(X.shape[0], dtype=DTYPE)
    if _get(th, "corr_var") is not None:
        inner = th["prev_var"] * torch.ones(X.shape[0], dtype=DTYPE)
        if _get(th, "lin_var") is not None:
            b = X[:, Da:]
            inner = inner + th["lin_var"] * (b * b).sum(-1)
        v = v + th["corr_var"] * inner
    if _get(th, "white_var") is not None:
        v = v + th["white_var"]
    return v


def _leaves(th):
    return {r: th[r].detach().clone().requires_grad_(True) for r in ROLES if _get(th, r) is not None}


def _acc(dst, names, grads):
    for r, g in zip(names, grads):
        if g is not None:
            dst[r] += g


@torch.enable_grad()
def comp_K_vjp(X, X2, Da, th, Kbar, chunk=2048):
    """(K, dX, dX2, dtheta) for the upstream gradient Kbar: dX = d<Kbar, K>/dX etc.; dtheta has one zero-filled entry per given role
    (roles K does not depend on, e.g. White for K(X, X2), get exact zeros). X2 None: one autograd pass (K(Z) is M x M)."""
    lv = _leaves(th)
    names = list(lv)
    dth = {r: torch.zeros_like(t) for r, t in lv.items()}
    Xl = X.detach().clone().requires_grad_(True)
    if X2 is None:
        K = comp_K(Xl, None, Da, lv)
        g = torch.autograd.grad(K, [Xl] + [lv[r] for r in names], Kbar, allow_unused=True)
        _acc(dth, names, g[1:])
        return K.detach(), g[0], None, dth
    dX = torch.zeros_like(X)
    Ks, dX2s = [], []
    for lo in range(0, X2.shape[0], chunk):
        X2c = X2[lo:lo + chunk].detach().clone().requires_grad_(True)
        Kc = comp_K(Xl, X2c, Da, lv)
        g = torch.autograd.grad(Kc, [Xl, X2c] + [lv[r] for r in names], Kbar[:, lo:lo + chunk], allow_unused=True)
        dX += g[0]
        dX2s.append(g[1])
        _acc(dth, names, g[2:])
        Ks.append(Kc.detach())
    return torch.cat(Ks, 1), dX, torch.cat(dX2s, 0), dth


@torch.enable_grad()
def comp_Kdiag_vjp(X, Da, th, g, chunk=1 << 16):
    """(K_diag, dX, dtheta) for the upstream gradient g [P]."""
    lv = _leaves(th)
    names = list(lv)
    dth = {r: torch.zeros_like(t) for r, t in lv.items()}
    outs, dXs = [], []
    for lo in range(0, X.shape[0], chunk):
        Xc = X[lo:lo + chunk].detach().clone().requires_grad_(True)
        v = comp_Kdiag(Xc, Da, lv)
        gr = torch.autograd.grad(v, [Xc] + [lv[r] for r in names], g[lo:lo + chunk], allow_unused=True)
        dXs.append(torch.zeros_like(Xc) if gr[0] is None else gr[0])
        _acc(dth, names, gr[1:])
        outs.append(v.detach())
    return torch.cat(outs), torch.cat(dXs, 0), dth


# ------------------------------------------------------------------------------------------------ SVGP layer on supplied matrices
def _moments(Ku, Kuf, Kdiag, q_mu, q_sqrt):
    """dgp_oracle.conditional_ND lines 176-190 with Ku (already + jitter I), Kuf and K_diag supplied."""
    D_out = q_mu.shape[1]
    Lu = torch.linalg.cholesky(Ku)
    A = torch.linalg.solve_triangular(Lu, Kuf, upper=False)
    A = torch.linalg.solve_triangular(Lu.T, A, upper=True)
    mean = A.T @ q_mu
    A_tiled = A[None].expand(D_out, -1, -1)
    SK = -Ku[None].expand(D_out, -1, -1) + q_sqrt @ q_sqrt.transpose(1, 2)
    B = SK @ A_tiled
    delta = (A_tiled * B).sum(1)
    var = (Kdiag[None] + delta).T
    return mean, var


def svgp_kl(Ku, q_mu, q_sqrt):
    """dgp_oracle.layer_KL (non-white branch) with Ku supplied."""
    M, D_out = q_mu.shape
    Lu = torch.linalg.cholesky(Ku)
    KL = torch.tensor(-0.5 * D_out * M, dtype=DTYPE)
    KL = KL - 0.5 * torch.log(torch.diagonal(q_sqrt, dim1=1, dim2=2) ** 2).sum()
    KL = KL + torch.log(torch.diagonal(Lu)).sum() * D_out
    LinvR = torch.linalg.solve_triangular(Lu[None].expand(D_out, -1, -1), q_sqrt, upper=False)
    KL = KL + 0.5 * (LinvR ** 2).sum()
    KL = KL + 0.5 * (q_mu * torch.cholesky_solve(q_mu, Lu)).sum()
    return KL


def svgp_from_k(Ku, Kuf, Kdiag, q_mu, q_sqrt, chunk=None):
    """(mean [P, D_out], var [P, D_out], kl). Differentiable (autograd) when chunk is None; otherwise computed chunk by chunk."""
    kl = svgp_kl(Ku, q_mu, q_sqrt)
    if chunk is None:
        return _moments(Ku, Kuf, Kdiag, q_mu, q_sqrt) + (kl,)
    ms, vs = [], []
    with torch.no_grad():
        for lo in range(0, Kuf.shape[1], chunk):
            m, v = _moments(Ku, Kuf[:, lo:lo + chunk], Kdiag[lo:lo + chunk], q_mu, q_sqrt)
            ms.append(m)
            vs.append(v)
    return torch.cat(ms), torch.cat(vs), kl.detach()


@torch.enable_grad()
def svgp_from_k_vjp(Ku, Kuf, Kdiag, q_mu, q_sqrt, Gm, Gv, gkl, chunk=1 << 15):
    """(mean, var, kl, dKu, dKuf, dKdiag, dq_mu, dq_sqrt) of the loss <Gm, mean> + <Gv, var> + gkl kl, by autograd chunk by chunk.
    dq_sqrt is the full gradient of the (lower-triangular) q_sqrt input; the library returns its lower triangle. dKu is symmetric
    (the Cholesky adjoint symmetrises); only the symmetric part of a gradient w.r.t. the symmetric Ku is defined.
    The *_vjp functions build their own autograd graphs, also when called with grad mode off (inside an autograd backward)."""
    Kul, qml, qsl = [t.detach().clone().requires_grad_(True) for t in (Ku, q_mu, q_sqrt)]
    kl = svgp_kl(Kul, qml, qsl)
    dKu, dqm, dqs = torch.autograd.grad(kl, [Kul, qml, qsl], torch.tensor(float(gkl), dtype=DTYPE))
    ms, vs, dKufs, dKds = [], [], [], []
    for lo in range(0, Kuf.shape[1], chunk):
        Kfc = Kuf[:, lo:lo + chunk].detach().clone().requires_grad_(True)
        Kdc = Kdiag[lo:lo + chunk].detach().clone().requires_grad_(True)
        m, v = _moments(Kul, Kfc, Kdc, qml, qsl)
        g = torch.autograd.grad([m, v], [Kul, Kfc, Kdc, qml, qsl], [Gm[lo:lo + chunk], Gv[lo:lo + chunk]])
        dKu, dqm, dqs = dKu + g[0], dqm + g[3], dqs + g[4]
        dKufs.append(g[1])
        dKds.append(g[2])
        ms.append(m.detach())
        vs.append(v.detach())
    return torch.cat(ms), torch.cat(vs), kl.detach(), dKu, torch.cat(dKufs, 1), torch.cat(dKds), dqm, dqs
