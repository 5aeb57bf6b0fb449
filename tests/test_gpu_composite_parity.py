"""The composite-kernel layer path (csrc/compkern.cuh, csrc/extk.cuh, svgp_from_k_run) against the float64 CPU reference of
oracle/composite_oracle.py at the shapes the multi-fidelity / multi-objective models run at: every adjoint instantiation
(compk_grad_rows_kernel<8>, <16>, <32>), the column-split adjoint of Kuf up to 32 splits with an uneven last chunk, the
supplied-matrix pipeline at padded M, several outputs, D_out = 32 and up to 524 288 columns, the prep cache, the forward-plane
stash and the workspace limit; then whole MF-DGP-EM / MO-DGP ELBO evaluations with the library swapped for the reference.

The CPU tests at the top tie the reference to what is already trusted (dgp_oracle.conditional_ND / layer_KL, the numpy GPflow
expression) and run without a GPU. Inputs are seeded; every Ku has cond <= 2e3 (asserted), so 1e-9 relative parity (rel_err,
relative to the un-cancelled scale) is above the conditioning noise floor of the float64 reference."""
import os

import numpy as np
import pytest
import torch

from oracle import composite_oracle as CO
from oracle import dgp_oracle as O
from tests.helpers import rel_err

DT = torch.float64
COND_MAX = 2e3
DEV = torch.device("cuda", 0)
SLOT = dict(in_var=0, corr_var=1, corr_ls=2, prev_var=3, prev_ls=4, lin_var=5, white_var=6)


# ---------------------------------------------------------------------------------------------------------------- input builders
def _theta(D, Da, prod, lin, white, ard, seed):
    """Kernel parameters (dict role -> CPU tensor, None where the role is absent), scaled so that every term of k is O(0.1 .. 1)
    on inputs in [0, 1]^D."""
    g = torch.Generator().manual_seed(seed)
    u = lambda *s: torch.rand(*s, generator=g, dtype=DT)
    sa, sb = max(Da, 1) ** 0.5, max(D - Da, 1) ** 0.5
    th = dict.fromkeys(CO.ROLES)
    th["in_var"] = 0.5 + u(())
    th["in_ls"] = 0.4 * sa * (0.7 + 0.6 * u(Da)) if ard else 0.4 * sa * (0.7 + 0.6 * u(()))
    if prod:
        th["corr_var"], th["corr_ls"] = 0.5 + u(()), 0.5 * sa * (0.8 + 0.4 * u(()))
        th["prev_var"], th["prev_ls"] = 0.5 + u(()), 0.5 * sb * (0.8 + 0.4 * u(()))
        if lin:
            th["lin_var"] = 0.3 + 0.5 * u(())
    if white:
        th["white_var"] = 0.01 + 0.02 * u(())
    return th


def _rbf_inputs(M, P, d, seed, variance=1.3):
    """Ku = RBF(Z) + 1e-6 I with cond(Ku) <= COND_MAX (the lengthscale shrinks until it holds, as tests.helpers._condition does),
    Kuf = RBF(Z, X), Kdiag = variance: the matrices a layer of the model hands the library."""
    rng = np.random.default_rng(seed)
    Z = torch.as_tensor(rng.uniform(0, 1, (M, d)))
    X = torch.as_tensor(rng.uniform(0, 1, (P, d)))
    ls, var = torch.full((d,), 0.6, dtype=DT), torch.tensor(variance, dtype=DT)
    for _ in range(80):
        Ku = O.kernel_K(Z, None, ls, var) + 1e-6 * torch.eye(M, dtype=DT)
        cond = float(torch.linalg.cond(Ku))
        if cond <= COND_MAX:
            break
        ls = ls * 0.85
    assert cond <= COND_MAX, cond
    Kuf = torch.cat([O.kernel_K(Z, X[lo:lo + 65536], ls, var) for lo in range(0, P, 65536)], 1)
    return Ku, Kuf, torch.full((P,), variance, dtype=DT)


def _q(M, D_out, seed):
    rng = np.random.default_rng(seed)
    q_mu = torch.as_tensor(0.5 * rng.standard_normal((M, D_out)))
    q_sqrt = torch.as_tensor(np.tril(0.6 * np.eye(M)[None] + (0.3 / M ** 0.5) * rng.standard_normal((D_out, M, M))))
    return q_mu, q_sqrt


# ------------------------------------------------------------------------------------------------ CPU: the reference is the oracle
@pytest.mark.parametrize("M,D_out,P", [(1, 1, 1), (9, 2, 14), (40, 3, 200)])
def test_svgp_from_k_reference_equals_oracle_conditional_and_kl(M, D_out, P):
    """On RBF matrices built by dgp_oracle.kernel_K, svgp_from_k is dgp_oracle.conditional_ND + layer_KL."""
    rng = np.random.default_rng(M)
    Z, X = rng.uniform(0, 1, (M, 2)), rng.uniform(0, 1, (P, 2))
    q_mu, q_sqrt = _q(M, D_out, M + 1)
    layer = O.make_layer(Z, np.array([0.4, 0.5]), 1.3, D_out, q_mu=q_mu, q_sqrt=q_sqrt)
    Ku, _ = O.kuu_chol(layer)
    Kuf = O.kernel_K(layer.Z, torch.as_tensor(X), layer.lengthscales, layer.variance)
    mean, var, kl = CO.svgp_from_k(Ku, Kuf, O.rbf_K_diag(torch.as_tensor(X), layer.variance), layer.q_mu, layer.q_sqrt)
    m_o, v_o = O.conditional_ND(layer, torch.as_tensor(X))
    assert rel_err(mean, m_o) < 1e-13 and rel_err(var, v_o, 1.3) < 1e-13
    assert abs(float(kl) - float(O.layer_KL(layer))) <= 1e-12 * max(1.0, abs(float(kl)))


def test_comp_K_reference_equals_the_gpflow_expression():
    """comp_K / comp_Kdiag against the numpy GPflow expression of test_gpu_mf.test_composite_kernel_matches_gpflow_semantics."""
    rng = np.random.default_rng(1)
    X, X2 = rng.standard_normal((7, 3)), rng.standard_normal((5, 3))
    th = dict(in_var=torch.tensor(0.5, dtype=DT), in_ls=torch.tensor(1.4, dtype=DT), corr_var=torch.tensor(0.7, dtype=DT),
              corr_ls=torch.tensor(0.9, dtype=DT), prev_var=torch.tensor(1.3, dtype=DT), prev_ls=torch.tensor(1.1, dtype=DT),
              lin_var=torch.tensor(0.8, dtype=DT), white_var=torch.tensor(0.03, dtype=DT))
    se = lambda A, B, v, l: v * np.exp(-0.5 * ((A[:, None, :] - B[None, :, :]) ** 2).sum(-1) / l ** 2)
    ref = lambda A, B: se(A[:, :2], B[:, :2], 0.7, 0.9) * (se(A[:, 2:], B[:, 2:], 1.3, 1.1) + 0.8 * A[:, 2:] @ B[:, 2:].T) + se(A[:, :2], B[:, :2], 0.5, 1.4)
    Xt, X2t = torch.as_tensor(X), torch.as_tensor(X2)
    assert rel_err(CO.comp_K(Xt, X2t, 2, th), ref(X, X2)) < 1e-14
    assert rel_err(CO.comp_K(Xt, None, 2, th), ref(X, X) + 0.03 * np.eye(7)) < 1e-14
    assert rel_err(CO.comp_Kdiag(Xt, 2, th), np.diag(ref(X, X)) + 0.03) < 1e-14
    # ARD k_in without the product part (the first fidelity / projection layers)
    ls = np.array([0.6, 0.9, 1.7])
    th1 = dict(in_var=torch.tensor(0.5, dtype=DT), in_ls=torch.as_tensor(ls))
    ref1 = 0.5 * np.exp(-0.5 * (((X[:, None, :] - X2[None, :, :]) / ls) ** 2).sum(-1))
    assert rel_err(CO.comp_K(Xt, X2t, 3, th1), ref1) < 1e-14
    assert rel_err(CO.comp_Kdiag(Xt, 3, th1), np.full(7, 0.5)) == 0.0


def test_comp_K_reference_gradients_match_finite_differences():
    """The autograd adjoint of comp_K (symmetric and cross) on a few directional central differences."""
    D, Da = 5, 3
    th = _theta(D, Da, True, True, True, True, 3)
    g = torch.Generator().manual_seed(4)
    X, X2 = torch.rand(6, D, generator=g, dtype=DT), torch.rand(4, D, generator=g, dtype=DT)
    for Y in (X2, None):
        Kbar = torch.randn(6, 6 if Y is None else 4, generator=g, dtype=DT)
        _, dX, _, dth = CO.comp_K_vjp(X, Y, Da, th, Kbar)
        V = torch.randn(6, D, generator=g, dtype=DT)
        f = lambda e: float((Kbar * CO.comp_K(X + e * V, None if Y is None else Y, Da, th)).sum())
        h = 1e-6
        assert abs((f(h) - f(-h)) / (2 * h) - float((dX * V).sum())) < 1e-7
        for r in ("in_ls", "corr_ls", "prev_var", "lin_var", "white_var"):
            th2 = dict(th)
            f2 = lambda e: float((Kbar * CO.comp_K(X, Y, Da, dict(th2, **{r: th[r] + e}))).sum())
            fd = ((f2(h) - f2(-h)) / (2 * h))
            assert abs(fd - float(dth[r].sum())) < 1e-7 * max(1.0, abs(fd)), r


def test_chunked_reference_equals_unchunked():
    """The chunked adjoints (the form used at large P) against one whole-P autograd pass, to rounding."""
    M, D_out, P = 24, 3, 301
    Ku, Kuf, Kdiag = _rbf_inputs(M, P, 2, 5)
    q_mu, q_sqrt = _q(M, D_out, 6)
    g = torch.Generator().manual_seed(7)
    Gm, Gv = torch.randn(P, D_out, generator=g, dtype=DT), torch.randn(P, D_out, generator=g, dtype=DT)
    leaves = [t.clone().requires_grad_(True) for t in (Ku, Kuf, Kdiag, q_mu, q_sqrt)]
    mean, var, kl = CO.svgp_from_k(*leaves)
    whole = torch.autograd.grad([mean, var, kl], leaves, [Gm, Gv, torch.tensor(0.7, dtype=DT)])
    ch = CO.svgp_from_k_vjp(Ku, Kuf, Kdiag, q_mu, q_sqrt, Gm, Gv, 0.7, chunk=64)
    m2, v2, kl2 = CO.svgp_from_k(Ku, Kuf, Kdiag, q_mu, q_sqrt, chunk=50)
    for a, b in zip((ch[0], ch[1], m2, v2), (mean, var, mean, var)):
        assert rel_err(a, b) < 1e-14
    assert abs(float(ch[2]) - float(kl.detach())) < 1e-13 * abs(float(kl.detach())) and float(kl2) == float(ch[2])
    for a, b in zip(ch[3:], whole):
        assert rel_err(a, b) < 1e-13
    D, Da = 9, 8
    th = _theta(D, Da, True, True, True, False, 8)
    X, X2 = torch.rand(5, D, generator=g, dtype=DT), torch.rand(700, D, generator=g, dtype=DT)
    Kbar = torch.randn(5, 700, generator=g, dtype=DT)
    a = CO.comp_K_vjp(X, X2, Da, th, Kbar, chunk=128)
    b = CO.comp_K_vjp(X, X2, Da, th, Kbar, chunk=700)
    for u, v in zip(a[:3], b[:3]):
        assert rel_err(u, v) < 1e-14
    assert all(rel_err(a[3][r], b[3][r]) < 1e-13 for r in a[3])
    gk = torch.randn(700, generator=g, dtype=DT)
    a, b = CO.comp_Kdiag_vjp(X2, Da, th, gk, chunk=128), CO.comp_Kdiag_vjp(X2, Da, th, gk, chunk=700)
    assert rel_err(a[0], b[0]) == 0.0 and rel_err(a[1], b[1]) == 0.0 and all(rel_err(a[2][r], b[2][r]) < 1e-13 for r in a[2])


# ---------------------------------------------------------------------------------------------------------------- GPU helpers
def _roles(D, Da, th):
    return dict(D=D, Da=Da, k_corr=True if th["corr_var"] is not None else None, lin=True if th["lin_var"] is not None else None)


def _dev(th):
    return {r: None if t is None else t.cuda() for r, t in th.items()}


def _raw_dtheta(name, roles, thg, *args):
    """The library's raw d theta vector (7 + Da slots, NaN-filled first, so every slot must be written)."""
    from dgp_toolbox_b200 import _lib
    from dgp_toolbox_b200.composite import THETA, _desc
    nt = THETA + thg["in_ls"].numel()
    dth = torch.full((nt,), float("nan"), dtype=DT, device="cuda")
    _lib.get_context(0).call(name, C_byref(_desc(roles, thg)), *args, _lib.ptr(dth))
    torch.cuda.synchronize()
    return dth.cpu()


def C_byref(d):
    import ctypes
    return ctypes.byref(d)


def _check_dtheta(raw, dth_ref, th, ard, tol, where):
    """Every slot of the library's d theta against the reference; slots of absent roles (and White in K(X, X2)) exactly 0."""
    for r, s in SLOT.items():
        if th[r] is None:
            assert float(raw[s]) == 0.0, (where, r, float(raw[s]))
        else:
            ref = dth_ref[r].reshape(())
            assert rel_err(raw[s], ref) < tol, (where, r, rel_err(raw[s], ref))
    ls = raw[7:]
    assert ls.numel() == (th["in_ls"].numel() if ard else 1)
    assert rel_err(ls, dth_ref["in_ls"].reshape(-1)) < tol, (where, "in_ls", rel_err(ls, dth_ref["in_ls"].reshape(-1)))


# ------------------------------------------------------------------------------- (a) composite kernel and its adjoint, at size
COMPK_CASES = [
    # (D, Da, prod, lin, white, ard, P, P2): P2 None = K(X, X)
    (3, 2, True, True, True, False, 7, 9),            # fixture-sized
    (5, 5, False, False, False, True, 256, 20001),    # k_in alone, ARD (EM projection layer): <8>, 16 splits, uneven last chunk
    (8, 7, True, True, True, False, 256, 20001),      # last <8> width
    (9, 8, True, True, True, False, 256, 20001),      # first <16> width (the MO benchmark's D = 9)
    (16, 15, True, False, False, True, 64, 40001),    # last <16> width, 32 splits
    (17, 16, True, False, False, True, 64, 40001),    # first <32> width, 32 splits
    (32, 31, True, True, False, False, 70, 2048),     # <32> at kCompMaxD, nsplit 1 -> 2 threshold
    (32, 31, True, True, False, False, 70, 2047),     # ... just below it
    (9, 8, True, True, True, False, 256, None),       # K(Z): symmetric path, White gradient on the diagonal
    (9, 8, True, True, True, True, 300, None),
    (1, 1, False, False, False, False, 1, 1),         # degenerate
    (1, 1, False, False, True, False, 1, None),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", COMPK_CASES, ids=lambda c: f"D{c[0]}-Da{c[1]}-{c[6]}x{c[7] or 'sym'}")
def test_comp_K_and_adjoint_match_reference(case):
    from dgp_toolbox_b200 import _lib
    from dgp_toolbox_b200.composite import ROLE_PARAMS, CompK
    D, Da, prod, lin, white, ard, P, P2 = case
    seed = D * 1000 + P
    th = _theta(D, Da, prod, lin, white, ard, seed)
    g = torch.Generator().manual_seed(seed + 1)
    X = torch.rand(P, D, generator=g, dtype=DT)
    X2 = None if P2 is None else torch.rand(P2, D, generator=g, dtype=DT)
    Kbar = torch.randn(P, P if P2 is None else P2, generator=g, dtype=DT)     # dense and, for K(X, X), not symmetric
    K_ref, dX_ref, dX2_ref, dth_ref = CO.comp_K_vjp(X, X2, Da, th, Kbar)
    roles, thg = _roles(D, Da, th), _dev(th)
    leaves = [None if thg[r] is None else thg[r].clone().requires_grad_(True) for r in ROLE_PARAMS]
    Xg = X.cuda().requires_grad_(True)
    X2g = None if X2 is None else X2.cuda().requires_grad_(True)
    K = CompK.apply(roles, Xg, X2g, *leaves)
    assert rel_err(K, K_ref) < 1e-13
    K.backward(Kbar.cuda())
    assert rel_err(Xg.grad, dX_ref) < 1e-9, rel_err(Xg.grad, dX_ref)
    if X2 is not None:
        assert rel_err(X2g.grad, dX2_ref) < 1e-9, rel_err(X2g.grad, dX2_ref)
    for r, t in zip(ROLE_PARAMS, leaves):
        if t is not None:
            assert rel_err(t.grad, dth_ref[r]) < 1e-9, (r, rel_err(t.grad, dth_ref[r]))
    Xc, X2c, Kbc = X.cuda(), None if X2 is None else X2.cuda(), Kbar.cuda()      # named: alive until the call has run
    dX = torch.empty_like(Xc)
    dX2 = None if X2c is None else torch.empty_like(X2c)
    raw = _raw_dtheta("dgp_comp_K_grad", roles, thg, _lib.ptr(Xc), P, _lib.ptr(X2c), 0 if X2c is None else P2, _lib.ptr(Kbc),
                      _lib.ptr(dX), _lib.ptr(dX2))
    _check_dtheta(raw, dth_ref, th, ard, 1e-9, case)


@pytest.mark.gpu
@pytest.mark.parametrize("P", [129, 524289])
def test_comp_Kdiag_and_adjoint_match_reference(P):
    """K_diag and its adjoint; at P = 524 289 many partial blocks go through reduce_partials_kernel."""
    from dgp_toolbox_b200 import _lib
    from dgp_toolbox_b200.composite import ROLE_PARAMS, CompKdiag
    D, Da = 9, 8
    for prod, lin, white, ard in ((True, True, True, True), (False, False, False, False)):
        th = _theta(D if prod else Da, Da, prod, lin, white, ard, P)
        Dx = D if prod else Da
        g = torch.Generator().manual_seed(P)
        X, gk = torch.rand(P, Dx, generator=g, dtype=DT), torch.randn(P, generator=g, dtype=DT)
        v_ref, dX_ref, dth_ref = CO.comp_Kdiag_vjp(X, Da, th, gk)
        roles, thg = _roles(Dx, Da, th), _dev(th)
        leaves = [None if thg[r] is None else thg[r].clone().requires_grad_(True) for r in ROLE_PARAMS]
        Xg = X.cuda().requires_grad_(True)
        v = CompKdiag.apply(roles, Xg, *leaves)
        assert rel_err(v, v_ref) < 1e-14
        v.backward(gk.cuda())
        assert rel_err(Xg.grad, dX_ref) < 1e-12 if prod and lin else float(Xg.grad.abs().max()) == 0.0
        for r, t in zip(ROLE_PARAMS, leaves):
            if t is not None:
                assert rel_err(t.grad, dth_ref[r]) < 1e-9, (r, rel_err(t.grad, dth_ref[r]))
        Xc, gkc = X.cuda(), gk.cuda()
        dXc = torch.empty_like(Xc)
        raw = _raw_dtheta("dgp_comp_Kdiag_grad", roles, thg, _lib.ptr(Xc), P, _lib.ptr(gkc), _lib.ptr(dXc))
        for r, s in SLOT.items():
            assert (float(raw[s]) == 0.0) if th[r] is None else rel_err(raw[s], dth_ref[r].reshape(())) < 1e-9, (r, P)
        assert float(raw[7:].abs().max()) == 0.0        # K_diag does not depend on the lengthscales


@pytest.mark.gpu
def test_comp_kernel_argument_errors_raise_and_launch_nothing():
    """D = 33, a product part with Da = D, a missing parameter pointer: every entry point raises DGPError before any launch."""
    from dgp_toolbox_b200 import _lib
    from dgp_toolbox_b200.composite import THETA, _desc
    ctx = _lib.get_context(0)
    bad = []
    th = _dev(_theta(33, 33, False, False, False, False, 1))
    bad.append((33, dict(D=33, Da=33, k_corr=None, lin=None), th))
    th = _dev(_theta(3, 2, True, True, False, False, 2))
    bad.append((3, dict(D=3, Da=3, k_corr=True, lin=True), th))
    th = _dev(_theta(3, 2, True, True, False, False, 3))
    th["prev_ls"] = None
    bad.append((3, dict(D=3, Da=2, k_corr=True, lin=True), th))
    for D, roles, thg in bad:
        d = _desc(roles, thg)
        X = torch.rand(5, D, dtype=DT, device="cuda")
        X2 = torch.rand(4, D, dtype=DT, device="cuda")
        out = torch.full((5, 4), float("nan"), dtype=DT, device="cuda")
        dX, dX2 = torch.full_like(X, float("nan")), torch.full_like(X2, float("nan"))
        dth = torch.full((THETA + thg["in_ls"].numel(),), float("nan"), dtype=DT, device="cuda")
        Kbar = torch.ones(5, 4, dtype=DT, device="cuda")
        p = _lib.ptr
        calls = [("dgp_comp_K", p(X), 5, p(X2), 4, p(out)), ("dgp_comp_Kdiag", p(X), 5, p(out)),
                 ("dgp_comp_K_grad", p(X), 5, p(X2), 4, p(Kbar), p(dX), p(dX2), p(dth)),
                 ("dgp_comp_Kdiag_grad", p(X), 5, p(Kbar), p(dX), p(dth))]
        for name, *args in calls:
            n0 = ctx.launch_count()
            with pytest.raises(_lib.DGPError, match="composite kernel"):
                ctx.call(name, C_byref(d), *args)
            assert ctx.launch_count() == n0, name
        torch.cuda.synchronize()
        assert bool(out.isnan().all() and dX.isnan().all() and dX2.isnan().all() and dth.isnan().all())


# ------------------------------------------------------------------------------ (b) the SVGP layer on supplied matrices, at size
SVGP_CASES = [
    # (M, D_out, P, gkl)
    (1, 1, 1, 0.7),
    (7, 1, 9, 0.0),
    (64, 1, 128, 0.7),
    (70, 3, 129, 0.0),          # padded M, the Pp tile boundary
    (250, 4, 3001, 0.7),
    (320, 32, 1000, 0.0),       # D_out at kMaxD: the 32-wide qmuP / GmPad layouts are full
    (256, 1, 327680, 0.7),      # one config-4 layer application (32 768 points x S = 10)
    (256, 1, 524288, 0.0),      # one config-5 application (16 384 candidates x S = 32)
]


def _svgp_gpu(Ku, Kuf, Kdiag, q_mu, q_sqrt, Gm, Gv, gkl, cache):
    from dgp_toolbox_b200.composite import SVGPFromK
    leaves = [t.detach().clone().requires_grad_(True) for t in (Ku, Kuf, Kdiag, q_mu, q_sqrt)]
    mean, var, kl = SVGPFromK.apply(*leaves, cache)
    grads = torch.autograd.grad([mean, var, kl], leaves, [Gm, Gv, torch.tensor(gkl, dtype=DT, device="cuda")])
    return [mean.detach(), var.detach(), kl.detach()] + list(grads)


NAMES = ("mean", "var", "kl", "dKu", "dKuf", "dKdiag", "dq_mu", "dq_sqrt")


def _sym(t):
    """Ku is symmetric, so only the symmetric part of d/dKu is defined: the reference's is symmetric, the library's is not
    symmetrised (its callers feed it to the K(Z) adjoint, which reads both triangles)."""
    return 0.5 * (t + t.T)


def _check_svgp(out, ref, Kdiag, where, tol=1e-9):
    worst = {}
    for name, a, b in zip(NAMES, out, ref):
        if name == "dq_sqrt":
            a, b = torch.tril(a), torch.tril(b)
        elif name == "dKu":
            a, b = _sym(a), _sym(b)
        worst[name] = rel_err(a, b, float(Kdiag.max()) if name == "var" else None)
        assert worst[name] < tol, (where, name, worst[name])
    return worst


@pytest.mark.gpu
@pytest.mark.parametrize("case", SVGP_CASES, ids=lambda c: f"M{c[0]}-D{c[1]}-P{c[2]}")
def test_svgp_from_k_matches_reference(case):
    """Plain, with a PrepCache (store, then load) and with a PrepCache plus a stash budget: all against the same reference."""
    from dgp_toolbox_b200.composite import PrepCache
    M, D_out, P, gkl = case
    Ku, Kuf, Kdiag = _rbf_inputs(M, P, 4, M * 7 + P)
    q_mu, q_sqrt = _q(M, D_out, M + P)
    g = torch.Generator().manual_seed(P)
    Gm, Gv = torch.randn(P, D_out, generator=g, dtype=DT), torch.randn(P, D_out, generator=g, dtype=DT)
    ref = CO.svgp_from_k_vjp(Ku, Kuf, Kdiag, q_mu, q_sqrt, Gm, Gv, gkl)
    dev = [t.cuda() for t in (Ku, Kuf, Kdiag, q_mu, q_sqrt, Gm, Gv)]
    cache = PrepCache(M, D_out, DEV)
    stashing = PrepCache(M, D_out, DEV)
    stashing.budget = [1 << 40]
    for way, c in (("plain", None), ("store", cache), ("load", cache), ("stash", stashing)):
        assert way != "load" or cache.filled
        _check_svgp(_svgp_gpu(*dev, gkl, c), ref, Kdiag, (case, way))
    assert stashing.budget[0] < (1 << 40)


# ------------------------------------------------------------------------------------------ (c) cache, stash and workspace edges
@pytest.mark.gpu
def test_prep_cache_survives_an_arena_reallocation(monkeypatch):
    """A PrepCache stored by a small call, then a large call that makes ensure_ws free and reallocate the arena, then loads at both
    sizes: all against the reference. A fresh context guarantees that the arena grows."""
    from dgp_toolbox_b200 import _lib
    from dgp_toolbox_b200.composite import PrepCache
    fresh = _lib.Context(0)
    monkeypatch.setitem(_lib._ctxs, 0, fresh)
    M, D_out = 70, 2
    q_mu, q_sqrt = _q(M, D_out, 11)
    Ku, Kuf_l, Kd_l = _rbf_inputs(M, 40000, 3, 12)
    Kuf_s, Kd_s = Kuf_l[:, :129].contiguous(), Kd_l[:129].contiguous()
    g = torch.Generator().manual_seed(13)
    Gm_l, Gv_l = torch.randn(40000, D_out, generator=g, dtype=DT), torch.randn(40000, D_out, generator=g, dtype=DT)
    Gm_s, Gv_s = Gm_l[:129].contiguous(), Gv_l[:129].contiguous()
    ref_s = CO.svgp_from_k_vjp(Ku, Kuf_s, Kd_s, q_mu, q_sqrt, Gm_s, Gv_s, 0.7)
    ref_l = CO.svgp_from_k_vjp(Ku, Kuf_l, Kd_l, q_mu, q_sqrt, Gm_l, Gv_l, 0.7)
    d = lambda *ts: [t.cuda() for t in ts]
    small = d(Ku, Kuf_s, Kd_s, q_mu, q_sqrt, Gm_s, Gv_s)
    large = d(Ku, Kuf_l, Kd_l, q_mu, q_sqrt, Gm_l, Gv_l)
    cache = PrepCache(M, D_out, DEV)
    _check_svgp(_svgp_gpu(*small, 0.7, cache), ref_s, Kd_s, "store")
    ws0 = fresh.workspace_bytes()
    _check_svgp(_svgp_gpu(*large, 0.7, None), ref_l, Kd_l, "large, uncached")
    assert fresh.workspace_bytes() > ws0
    _check_svgp(_svgp_gpu(*small, 0.7, cache), ref_s, Kd_s, "load, small")
    _check_svgp(_svgp_gpu(*large, 0.7, cache), ref_l, Kd_l, "load, large")
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_stash_budget_running_out_midway_is_bitwise_and_matches_reference():
    """Four applications of one layer in one evaluation; the budget holds the stashes of the first two only, so two adjoints read
    stashes and two recompute the forward planes. Bitwise equal to budget 0, and equal to the reference."""
    from dgp_toolbox_b200 import _lib
    from dgp_toolbox_b200.composite import PrepCache, SVGPFromK
    M, D_out, Ps = 64, 2, (300, 500, 700, 900)
    q_mu, q_sqrt = _q(M, D_out, 21)
    Ku, Kuf_all, Kd_all = _rbf_inputs(M, sum(Ps), 3, 22)
    offs = np.cumsum((0,) + Ps)
    Kufs = [Kuf_all[:, a:b].contiguous() for a, b in zip(offs[:-1], offs[1:])]
    Kds = [Kd_all[a:b].contiguous() for a, b in zip(offs[:-1], offs[1:])]
    g = torch.Generator().manual_seed(23)
    Gms = [torch.randn(P, D_out, generator=g, dtype=DT) for P in Ps]
    Gvs = [torch.randn(P, D_out, generator=g, dtype=DT) for P in Ps]
    nb = [int(_lib.lib.dgp_svgp_stash_bytes(M, D_out, P)) for P in Ps]
    # reference: the per-application adjoints, with the shared leaves summed
    refs = [CO.svgp_from_k_vjp(Ku, Kf, Kd, q_mu, q_sqrt, Gm, Gv, 0.7) for Kf, Kd, Gm, Gv in zip(Kufs, Kds, Gms, Gvs)]

    def run(budget):
        cache = PrepCache(M, D_out, DEV)
        cache.budget = [budget]
        Kul, qml, qsl = [t.cuda().requires_grad_(True) for t in (Ku, q_mu, q_sqrt)]
        Kfl = [t.cuda().requires_grad_(True) for t in Kufs]
        Kdl = [t.cuda().requires_grad_(True) for t in Kds]
        loss = 0.0
        outs = []
        for Kf, Kd, Gm, Gv in zip(Kfl, Kdl, Gms, Gvs):
            mean, var, kl = SVGPFromK.apply(Kul, Kf, Kd, qml, qsl, cache)
            loss = loss + (mean * Gm.cuda()).sum() + (var * Gv.cuda()).sum() + 0.7 * kl
            outs += [mean.detach(), var.detach(), kl.detach()]
        left = cache.budget[0]
        grads = torch.autograd.grad(loss, [Kul, qml, qsl] + Kfl + Kdl)
        return outs, list(grads), left

    o0, g0, _ = run(0)
    o1, g1, left = run(nb[0] + nb[1] + 1)
    assert left == 1                                   # applications 0 and 1 stashed, 2 and 3 recomputed
    for a, b in zip(o0 + g0, o1 + g1):
        assert torch.equal(a, b)
    for i, r in enumerate(refs):
        assert rel_err(o1[3 * i], r[0]) < 1e-9 and rel_err(o1[3 * i + 1], r[1], float(Kds[i].max())) < 1e-9
        assert abs(float(o1[3 * i + 2]) - float(r[2])) <= 1e-9 * abs(float(r[2]))
        assert rel_err(g1[3 + i], r[4]) < 1e-9 and rel_err(g1[7 + i], r[5]) < 1e-9
    dKu, dqm, dqs = sum(r[3] for r in refs), sum(r[6] for r in refs), sum(r[7] for r in refs)
    assert rel_err(_sym(g1[0]), _sym(dKu)) < 1e-9 and rel_err(g1[1], dqm) < 1e-9 and rel_err(torch.tril(g1[2]), torch.tril(dqs)) < 1e-9


@pytest.mark.gpu
def test_workspace_limit_raises_cleanly_and_context_recovers():
    """With the workspace limit below what one call needs the call raises ("split the points"); the same context then gives the
    right answer once the limit is restored."""
    from dgp_toolbox_b200 import _lib
    M, D_out, P = 64, 1, 200000
    q_mu, q_sqrt = _q(M, D_out, 31)
    Ku, Kuf, Kdiag = _rbf_inputs(M, P, 3, 32)
    g = torch.Generator().manual_seed(33)
    Gm, Gv = torch.randn(P, D_out, generator=g, dtype=DT), torch.randn(P, D_out, generator=g, dtype=DT)
    dev = [t.cuda() for t in (Ku, Kuf, Kdiag, q_mu, q_sqrt, Gm, Gv)]
    ctx = _lib.get_context(0)
    ctx.set_workspace_limit(64 << 20)                  # one [64 x 200 064] plane is 102 MB
    try:
        with pytest.raises(_lib.DGPError, match="split the points"):
            _svgp_gpu(*dev, 0.7, None)
    finally:
        ctx.set_workspace_limit(int(float(os.environ.get("DGP_B200_WS_GB", "24")) * (1 << 30)))
    ref = CO.svgp_from_k_vjp(Ku, Kuf, Kdiag, q_mu, q_sqrt, Gm, Gv, 0.7)
    _check_svgp(_svgp_gpu(*dev, 0.7, None), ref, Kdiag, "after the limit is restored")


# ------------------------------------------------------------------------- (d) model level: the product's wiring on the reference
class _RefCompK(torch.autograd.Function):
    """composite.CompK with the CPU reference in place of dgp_comp_K / dgp_comp_K_grad."""

    @staticmethod
    def forward(ctx, roles, X, X2, *theta):
        from dgp_toolbox_b200.composite import ROLE_PARAMS
        th = {r: None if t is None else t.detach().cpu() for r, t in zip(ROLE_PARAMS, theta)}
        Xc, X2c = X.detach().cpu(), None if X2 is None else X2.detach().cpu()
        ctx.saved = (roles, th, Xc, X2c, X.device)
        if X2c is None:
            return CO.comp_K(Xc, None, roles["Da"], th).to(X.device)
        return torch.cat([CO.comp_K(Xc, X2c[lo:lo + 4096], roles["Da"], th) for lo in range(0, X2c.shape[0], 4096)], 1).to(X.device)

    @staticmethod
    def backward(ctx, Kbar):
        from dgp_toolbox_b200.composite import ROLE_PARAMS
        roles, th, Xc, X2c, dev = ctx.saved
        _, dX, dX2, dth = CO.comp_K_vjp(Xc, X2c, roles["Da"], th, Kbar.cpu())
        return (None, dX.to(dev), None if dX2 is None else dX2.to(dev)) + tuple(None if th[r] is None else dth[r].to(dev) for r in ROLE_PARAMS)


class _RefCompKdiag(torch.autograd.Function):
    @staticmethod
    def forward(ctx, roles, X, *theta):
        from dgp_toolbox_b200.composite import ROLE_PARAMS
        th = {r: None if t is None else t.detach().cpu() for r, t in zip(ROLE_PARAMS, theta)}
        ctx.saved = (roles, th, X.detach().cpu(), X.device)
        return CO.comp_Kdiag(ctx.saved[2], roles["Da"], th).to(X.device)

    @staticmethod
    def backward(ctx, g):
        from dgp_toolbox_b200.composite import ROLE_PARAMS
        roles, th, Xc, dev = ctx.saved
        _, dX, dth = CO.comp_Kdiag_vjp(Xc, roles["Da"], th, g.cpu())
        return (None, dX.to(dev)) + tuple(None if th[r] is None else dth[r].to(dev) for r in ROLE_PARAMS)


class _RefSVGPFromK(torch.autograd.Function):
    """composite.SVGPFromK with the CPU reference in place of dgp_svgp_from_k / dgp_svgp_from_k_grad (the cache is unused)."""

    @staticmethod
    def forward(ctx, Ku, Kuf, Kdiag, q_mu, q_sqrt, cache=None):
        ins = [t.detach().cpu() for t in (Ku, Kuf, Kdiag, q_mu, q_sqrt)]
        ctx.saved, ctx.dev = ins, Ku.device
        mean, var, kl = CO.svgp_from_k(*ins, chunk=1 << 15)
        return mean.to(Ku.device), var.to(Ku.device), kl.reshape(()).to(Ku.device)

    @staticmethod
    def backward(ctx, gmean, gvar, gkl):
        ins = ctx.saved
        P, D = ins[1].shape[1], ins[3].shape[1]
        z = torch.zeros(P, D, dtype=DT)
        Gm = z if gmean is None else gmean.cpu()
        Gv = z if gvar is None else gvar.cpu()
        out = CO.svgp_from_k_vjp(*ins, Gm, Gv, 0.0 if gkl is None else float(gkl))
        return tuple(t.to(ctx.dev) for t in out[3:]) + (None,)


def _use_reference(monkeypatch):
    from dgp_toolbox_b200 import composite
    from dgp_toolbox_b200.models import MF_DGP
    monkeypatch.setattr(composite, "CompK", _RefCompK)
    monkeypatch.setattr(composite, "CompKdiag", _RefCompKdiag)
    monkeypatch.setattr(MF_DGP, "SVGPFromK", _RefSVGPFromK)


class _Draws:
    """Seeded N(0, 1) draws, recorded on the first pass and replayed on the next (the models call `draw(shape)`)."""

    def __init__(self, seed):
        self.rng, self.log, self.i = np.random.default_rng(seed), [], None

    def replay(self):
        self.i = 0
        return self

    def __call__(self, shape):
        if self.i is None:
            self.log.append(torch.as_tensor(self.rng.standard_normal(shape), device=DEV))
            return self.log[-1]
        z = self.log[self.i]
        self.i += 1
        assert tuple(z.shape) == tuple(shape), (z.shape, shape, self.i)
        return z


def _layer_cond(layer):
    from dgp_toolbox_b200.composite import role_parameters
    params = role_parameters(layer.eval.roles)
    th = {r: None if p is None else p.value.detach().cpu() for r, p in params.items()}
    Z = layer.Zfull({}).detach().cpu()
    return float(torch.linalg.cond(CO.comp_K(Z, None, layer.eval.roles["Da"], th) + 1e-6 * torch.eye(Z.shape[0], dtype=DT)))


def _condition_layers(layers, white=0.05):
    """cond(Kuu) <= COND_MAX at the layers' inducing inputs: White (where the model has one) at `white`, then the lengthscales of
    k_in and k_corr shrink until the bound holds (k_corr (k_prev + Linear) is a Schur product of PSD kernels: it cannot lower the
    smallest eigenvalue). q(u) gets a nonzero mean and a scaled-down q_sqrt."""
    from dgp_toolbox_b200.composite import role_parameters
    rng = np.random.default_rng(99)
    for layer in layers:
        params = role_parameters(layer.eval.roles)
        if params["white_var"] is not None:
            params["white_var"].assign(white)
        for _ in range(80):
            if _layer_cond(layer) <= COND_MAX:
                break
            for r in ("in_ls", "corr_ls"):
                if params[r] is not None:
                    params[r].assign(params[r].value * 0.85)
        assert _layer_cond(layer) <= COND_MAX
        layer.q_mu.assign(0.3 * rng.standard_normal(tuple(layer.q_mu.value.shape)))
        layer.q_sqrt.assign(0.5 * layer.q_sqrt.value)


def _compare_runs(model, data, params, monkeypatch, layers, **kw):
    draws = _Draws(5)
    model.draw = draws
    elbo, grads = model.ELBO_and_grads(data, params, **kw)
    with monkeypatch.context() as mp:
        _use_reference(mp)
        model.draw = draws.replay()
        elbo_r, grads_r = model.ELBO_and_grads(data, params, **kw)
    assert draws.i == len(draws.log)
    for layer in layers:                                 # at the inducing inputs the evaluation re-sampled
        assert _layer_cond(layer) <= COND_MAX
    assert abs(float(elbo) - float(elbo_r)) <= 1e-9 * abs(float(elbo_r)), (float(elbo), float(elbo_r))
    worst = 0.0
    for i, p in enumerate(params):
        a, b = grads[p], grads_r[p]
        if a.dim() == 3:
            a, b = torch.tril(a), torch.tril(b)
        e = rel_err(a, b)
        worst = max(worst, e)
        assert e < 1e-8, (i, tuple(p.value.shape), e)
    return worst


@pytest.mark.gpu
def test_mf_dgp_em_at_config4_shapes_matches_the_reference_wiring(monkeypatch):
    """MF-DGP-EM as in config 4 with smaller minibatches: 3 fidelities with 2/3/4-D inputs, M = 256, S = 10, N = 1024 / 256 / 64
    (10 240 point-samples in the first fidelity: 8 column splits of the Kuf adjoint)."""
    from scipy.stats import qmc
    from dgp_toolbox_b200.models import MF_DGP_EM
    rng = np.random.default_rng(0)
    dims, ns = [2, 3, 4], [1024, 256, 64]
    f4 = lambda x: np.sin(3 * x[:, :1]) + 0.5 * x[:, 1:2]
    X = [rng.uniform(0, 1, (n, d)) for n, d in zip(ns, dims)]
    Y = [f4(X[0]), 1.2 * f4(X[1]) + 0.3 * X[1][:, :1] ** 2, 1.5 * f4(X[2]) - 0.2 * X[2][:, 1:2]]
    sob = lambda d, s: qmc.Sobol(d, scramble=True, seed=s).random(256)
    ctor = np.random.default_rng(1)
    em = MF_DGP_EM.DGP_Base.make_mf_dgp(X, [sob(d, 10 + d) for d in dims], [sob(4, 20), sob(3, 21)],
                                        draw=lambda shape: torch.as_tensor(ctor.standard_normal(shape), device=DEV))
    em.num_samples = 10
    _condition_layers(list(em.layers) + list(em.layers_red))
    data = (X, Y, [X[1][:, :2].copy(), X[2][:, :2].copy()])
    _compare_runs(em, data, em.trainable_parameters, monkeypatch, list(em.layers) + list(em.layers_red))


@pytest.mark.gpu
def test_mo_dgp_at_config5_shapes_matches_the_reference_wiring(monkeypatch):
    """MO-DGP as in config 5 (D_in = 8, M = 256, loop = 2) with S = 8, N = 512; then EHVI on the `mo_dgp` object (2 048 candidates,
    S = 32, the 32-point front) against O.ehvi_exact on the moments of the reference run (dgp_mixture_moments at size)."""
    import types
    import dgp_toolbox_b200 as D
    from dgp_toolbox_b200.models import MO_DGP
    rng = np.random.default_rng(0)
    g0 = lambda x: np.sin(3 * x[:, :1]) + 0.5 * x[:, 1:2]
    g1 = lambda x: np.cos(2 * x[:, :1]) * x[:, 1:2] - 0.3
    Zx = rng.uniform(0, 1, (256, 8))
    ctor = np.random.default_rng(1)
    mo = MO_DGP.DGP_Base.make_mf_dgp([np.concatenate([Zx, g1(Zx)], 1), Zx.copy()], loop=2,
                                     draw=lambda shape: torch.as_tensor(ctor.standard_normal(shape), device=DEV))
    mo.num_samples = 8
    _condition_layers(mo.layers)
    X = [rng.uniform(0, 1, (512, 8)) for _ in range(2)]
    Y = [g0(X[0]), g1(X[1])]
    _compare_runs(mo, (X, Y), mo.trainable_parameters, monkeypatch, mo.layers)

    y0 = np.linspace(0.05, 0.95, 32)
    y1 = 1.0 - np.sqrt(y0)
    order = np.argsort(-y0)
    ynd0, ynd1 = O.Y_ND(y0[order], y1[order], (1.1, 1.1), (-0.1, -0.1))
    xc = torch.as_tensor(rng.uniform(0, 1, (2048, 8)), device=DEV)
    obj = types.SimpleNamespace(name="mo_dgp", model=mo, _X=[Zx, Zx])
    draws = _Draws(6)
    mo.draw = draws
    ehvi = D.EHVI(obj, xc, [ynd0[:, None], ynd1[:, None]], S=32)
    with monkeypatch.context() as mp, torch.no_grad():
        _use_reference(mp)
        mo.draw = draws.replay()
        _, Fm, Fv = mo.propagate(xc, S=32)
    assert draws.i == len(draws.log)
    mom = []
    for o in (-2, -1):
        m, v = O.mixture_moments(Fm[o].cpu(), Fv[o].cpu())
        mom += [m.reshape(-1), v.reshape(-1)]
    ehvi_o = O.ehvi_exact(*mom, ynd0, ynd1)
    assert rel_err(ehvi.reshape(-1), ehvi_o.reshape(-1)) < 1e-8, rel_err(ehvi.reshape(-1), ehvi_o.reshape(-1))
