"""full_cov=True on supplied kernel matrices (dgp_svgp_from_k_full_cov, dgp_comp_K_blocks) and the MF-DGP, MF-DGP-EM and MO-DGP
propagate(full_cov=True) built on them, against a float64 CPU reference.

The reference of one full-covariance layer application is `svgp_from_k_full` below, written in the op order of
dgp_oracle.conditional_ND_full (utils/layers.py:237-278 with full_cov=True); samples are dgp_oracle.reparameterize_full. The CPU
test ties it to conditional_ND_full and to composite_oracle.svgp_from_k. Inputs are seeded and every Ku has cond <= 2e3
(asserted), as in test_gpu_composite_parity.py, whose reference stand-ins for the library calls are reused at model level."""
import os

import numpy as np
import pytest
import torch

from oracle import composite_oracle as CO
from oracle import dgp_oracle as O
from tests.helpers import rel_err
from tests.test_gpu_composite_parity import COND_MAX, _condition_layers, _Draws, _q, _theta, _use_reference

DT = torch.float64
DEV = torch.device("cuda", 0)


# ------------------------------------------------------------------------------------------------------------------ reference
def svgp_from_k_full(Ku, Kuf, Kff, q_mu, q_sqrt):
    """One sample's conditional with full_cov=True on supplied Ku = Kuu + jitter I [M, M], Kuf [M, N], Kff [N, N]: mean [N, D_out],
    cov [N, N, D_out], in the op order of dgp_oracle.conditional_ND_full (white = False, zero mean function)."""
    Lu = torch.linalg.cholesky(Ku)
    A = torch.linalg.solve_triangular(Lu, Kuf, upper=False)
    A = torch.linalg.solve_triangular(Lu.T, A, upper=True)
    mean = A.T @ q_mu
    SK = -Ku[None] + q_sqrt @ q_sqrt.transpose(1, 2)
    delta = A.T[None] @ (SK @ A[None])
    return mean, (Kff[None] + delta).permute(2, 1, 0)


def full_ref(Ku, Kuf, Kff, q_mu, q_sqrt, z):
    """S samples (column s * N + n of Kuf, block s or 0 of Kff) -> F, mean [S, N, D], cov [S, N, N, D]."""
    S, N, _ = z.shape
    mv = [svgp_from_k_full(Ku, Kuf[:, s * N:(s + 1) * N], Kff[s if Kff.shape[0] > 1 else 0], q_mu, q_sqrt) for s in range(S)]
    mean, cov = torch.stack([m for m, _ in mv]), torch.stack([c for _, c in mv])
    return O.reparameterize_full(mean, cov, z), mean, cov


def _rbf_problem(M, N, S, Kff_batch, d, seed):
    """Ku = RBF(Z) + 1e-6 I with cond <= COND_MAX, X [S, N, d] (the same rows for every sample when Kff_batch = 1), Kuf = RBF(Z, X)
    over the S * N columns, Kff = RBF(X_s, X_s) [Kff_batch, N, N]."""
    rng = np.random.default_rng(seed)
    Z = torch.as_tensor(rng.uniform(0, 1, (M, d)))
    X = torch.as_tensor(rng.uniform(0, 1, (1 if Kff_batch == 1 else S, N, d))).expand(S, N, d).contiguous()
    ls, var = torch.full((d,), 0.6, dtype=DT), torch.tensor(1.3, dtype=DT)
    for _ in range(80):
        Ku = O.kernel_K(Z, None, ls, var) + 1e-6 * torch.eye(M, dtype=DT)
        cond = float(torch.linalg.cond(Ku))
        if cond <= COND_MAX:
            break
        ls = ls * 0.85
    assert cond <= COND_MAX, cond
    Kuf = O.kernel_K(Z, X.reshape(S * N, d), ls, var)
    Kff = torch.stack([O.kernel_K(X[s], None, ls, var) for s in range(Kff_batch)])
    return Ku, Kuf, Kff, (Z, X, ls, var)


# ------------------------------------------------------------------------------------------------ CPU: the reference is the oracle
@pytest.mark.parametrize("M,D_out,N", [(1, 1, 1), (9, 2, 14), (40, 3, 60)])
def test_full_reference_equals_oracle_conditional_full_and_diagonal_reference(M, D_out, N):
    rng = np.random.default_rng(M + N)
    Z, X = rng.uniform(0, 1, (M, 2)), torch.as_tensor(rng.uniform(0, 1, (N, 2)))
    q_mu, q_sqrt = _q(M, D_out, M + 1)
    layer = O.make_layer(Z, np.array([0.4, 0.5]), 1.3, D_out, q_mu=q_mu, q_sqrt=q_sqrt)
    Ku, _ = O.kuu_chol(layer)
    Kuf = O.kernel_K(layer.Z, X, layer.lengthscales, layer.variance)
    Kff = O.kernel_K(X, None, layer.lengthscales, layer.variance)
    mean, cov = svgp_from_k_full(Ku, Kuf, Kff, layer.q_mu, layer.q_sqrt)
    m_o, c_o = O.conditional_ND_full(layer, X)
    assert rel_err(mean, m_o) < 1e-12 and rel_err(cov, c_o, 1.3) < 1e-12
    m_d, v_d, _ = CO.svgp_from_k(Ku, Kuf, torch.diagonal(Kff), layer.q_mu, layer.q_sqrt)
    assert rel_err(mean, m_d) < 1e-12
    assert rel_err(torch.diagonal(cov, dim1=0, dim2=1).T, v_d, 1.3) < 1e-12


# ------------------------------------------------------------------------------------------------------------ GPU helpers
def _call_full(ctx, Ku, Kuf, Kff, q_mu, q_sqrt, z, N, S, mean, cov, F, Kff_batch=None, jitter=O.JITTER):
    from dgp_toolbox_b200 import _lib
    p = _lib.ptr
    M, D = q_mu.shape
    ctx.call("dgp_svgp_from_k_full_cov", M, D, N, S, p(Ku), p(Kuf), p(Kff), Kff.shape[0] if Kff_batch is None else Kff_batch,
             p(q_mu), p(q_sqrt), p(z), float(jitter), p(mean), p(cov), p(F))


def _outs(S, N, D):
    nan = lambda *s: torch.full(s, float("nan"), dtype=DT, device=DEV)
    return nan(S, N, D), nan(S, N, N, D), nan(S, N, D)


# ------------------------------------------------------------------------------------------------ (a) blocked composite K(X, X)
DESCS = [
    # (D, Da, prod, lin, white, ard)
    (3, 2, True, True, True, False),      # the models' layer >= 1 kernel, with White
    (9, 8, True, False, False, True),     # product without Linear, ARD k_in, no White
    (4, 4, False, False, True, True),     # k_in alone (first fidelity / projection layers), ARD, White
]


@pytest.mark.gpu
@pytest.mark.parametrize("desc", DESCS, ids=lambda c: f"D{c[0]}-Da{c[1]}-prod{int(c[2])}-lin{int(c[3])}-white{int(c[4])}")
@pytest.mark.parametrize("B,N", [(1, 1), (3, 63), (3, 64), (3, 65), (1, 768), (250, 65), (250, 768)])
def test_comp_K_blocks_equals_comp_K_per_block(desc, B, N):
    from dgp_toolbox_b200.composite import ROLE_PARAMS, CompK, comp_K_blocks
    D, Da, prod, lin, white, ard = desc
    th = _theta(D, Da, prod, lin, white, ard, 7 * D + N)
    roles = dict(D=D, Da=Da, k_corr=True if prod else None, lin=True if lin else None)
    theta = [None if th[r] is None else th[r].cuda() for r in ROLE_PARAMS]
    X = torch.rand(B, N, D, generator=torch.Generator().manual_seed(B * N), dtype=DT).cuda()
    K = comp_K_blocks(roles, X, *theta)
    assert tuple(K.shape) == (B, N, N)
    for b in range(B):
        Kb = CompK.apply(roles, X[b].contiguous(), None, *theta)
        assert rel_err(K[b], Kb) < 1e-12, (b, rel_err(K[b], Kb))
    if B <= 3 and N <= 65:                           # White on each block's diagonal only
        assert rel_err(K[-1], CO.comp_K(X[-1].cpu(), None, Da, th)) < 1e-13


@pytest.mark.gpu
def test_comp_K_blocks_argument_errors_raise_and_launch_nothing():
    import ctypes
    from dgp_toolbox_b200 import _lib
    from dgp_toolbox_b200.composite import _desc
    ctx = _lib.get_context(0)
    good = dict(D=3, Da=2, k_corr=True, lin=True)
    thg = {r: None if t is None else t.cuda() for r, t in _theta(3, 2, True, True, True, False, 1).items()}
    bad_th = dict(thg, prev_ls=None)
    X = torch.rand(2, 5, 3, dtype=DT, device=DEV)
    out = torch.full((2, 5, 5), float("nan"), dtype=DT, device=DEV)
    cases = [(good, thg, 0, 5), (good, thg, 2, 0), (dict(D=3, Da=3, k_corr=True, lin=True), thg, 2, 5), (good, bad_th, 2, 5)]
    for roles, th, B, N in cases:
        n0 = ctx.launch_count()
        with pytest.raises(_lib.DGPError):
            ctx.call("dgp_comp_K_blocks", ctypes.byref(_desc(roles, th)), _lib.ptr(X), B, N, _lib.ptr(out))
        assert ctx.launch_count() == n0, (roles, B, N)
    torch.cuda.synchronize()
    assert bool(out.isnan().all())


# ------------------------------------------------------------------------------------ (b) the full-covariance layer call
FULL_CASES = [
    # (M, D_out, N, S, Kff_batch)
    (1, 1, 1, 1, 1),
    (9, 2, 5, 3, 3),
    (64, 1, 64, 4, 1),
    (256, 1, 768, 2, 2),
    (256, 4, 700, 3, 3),
    (320, 32, 40, 2, 2),
    (768, 1, 65, 2, 1),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", FULL_CASES, ids=lambda c: "M{}-D{}-N{}-S{}-K{}".format(*c))
def test_svgp_from_k_full_cov_matches_reference(case):
    from dgp_toolbox_b200 import _lib
    from dgp_toolbox_b200.composite import SVGPFromK, svgp_from_k_full_cov
    M, D_out, N, S, Kb = case
    Ku, Kuf, Kff, _ = _rbf_problem(M, N, S, Kb, 4, M + N + S)
    q_mu, q_sqrt = _q(M, D_out, M * 3 + N)
    z = torch.as_tensor(np.random.default_rng(N).standard_normal((S, N, D_out)))
    F_r, m_r, c_r = full_ref(Ku, Kuf, Kff, q_mu, q_sqrt, z)
    g = [t.cuda() for t in (Ku, Kuf, Kff, q_mu, q_sqrt, z)]
    F, mean, cov = svgp_from_k_full_cov(*g, O.JITTER)
    scale = float(torch.diagonal(c_r, dim1=1, dim2=2).abs().max())
    assert rel_err(mean, m_r) < 1e-9, rel_err(mean, m_r)
    assert rel_err(cov, c_r, scale) < 1e-9, rel_err(cov, c_r, scale)
    assert rel_err(F, F_r) < 1e-8, rel_err(F, F_r)
    # the mean is dgp_svgp_from_k's, bit for bit; the diagonal of cov is its variance
    Kdiag = torch.diagonal(g[2], dim1=1, dim2=2).expand(S, N).reshape(S * N).contiguous()
    with torch.no_grad():
        m_d, v_d, _ = SVGPFromK.apply(g[0], g[1], Kdiag, g[3], g[4])
    assert torch.equal(mean.reshape(S * N, D_out), m_d)
    assert rel_err(torch.diagonal(cov, dim1=1, dim2=2).permute(0, 2, 1).reshape(S * N, D_out), v_d, scale) < 1e-12
    ctx = _lib.get_context(0)
    m0, c0, F0 = _outs(S, N, D_out)                  # z = 0: F is the mean
    _call_full(ctx, *g[:5], torch.zeros_like(g[5]), N, S, m0, c0, F0)
    assert torch.equal(F0, m0) and torch.equal(m0, mean) and torch.equal(c0, cov)
    m1, c1, _ = _outs(S, N, D_out)                   # cov / F NULL: the other outputs do not change
    _call_full(ctx, *g[:5], None, N, S, m1, None, None)
    _call_full(ctx, *g[:5], None, N, S, m0, c1, None)
    assert torch.equal(m1, mean) and torch.equal(m0, mean) and torch.equal(c1, cov)
    m2, _, F2 = _outs(S, N, D_out)
    _call_full(ctx, *g[:5], g[5], N, S, m2, None, F2)
    assert torch.equal(m2, mean) and torch.equal(F2, F)


@pytest.mark.gpu
def test_rbf_composite_layer_equals_the_rbf_full_cov_path():
    """A composite layer that is RBF-ARD alone against dgp_propagate_full_cov on the equivalent one-layer DGP (same Z, lengthscales,
    variance, q and draws)."""
    import dgp_toolbox_b200 as D
    from dgp_toolbox_b200.composite import RBF, CompositeKernelEval, svgp_from_k_full_cov
    M, D_in, D_out, N, S = 64, 3, 2, 100, 3
    rng = np.random.default_rng(41)
    Z, X = rng.uniform(0, 1, (M, D_in)), rng.uniform(0, 1, (N, D_in))
    ls, var = np.array([0.5, 0.7, 0.6]), 1.2
    for _ in range(80):
        Ku = O.kernel_K(torch.as_tensor(Z), None, torch.as_tensor(ls), torch.tensor(var)) + 1e-6 * torch.eye(M, dtype=DT)
        if float(torch.linalg.cond(Ku)) <= COND_MAX:
            break
        ls = ls * 0.85
    assert float(torch.linalg.cond(Ku)) <= COND_MAX
    q_mu, q_sqrt = _q(M, D_out, 42)
    z = torch.as_tensor(rng.standard_normal((S, N, D_out)))
    layer = D.SVGP_Layer(D.SquaredExponential(variance=var, lengthscales=ls), Z, D_out, D.Zero())
    layer.q_mu.assign(q_mu.numpy())
    layer.q_sqrt.assign(q_sqrt.numpy())
    model = D.DGP_Base(D.Gaussian(0.1), [layer], num_samples=S)
    Fs, Fm, Fv = model.propagate(X, full_cov=True, S=S, zs=[z])
    ev = CompositeKernelEval(RBF(variance=var, lengthscales=list(ls)), D_in)
    Zg, Xg = torch.as_tensor(Z, device=DEV), torch.as_tensor(X, device=DEV)
    Kug = ev.K(Zg) + O.JITTER * torch.eye(M, dtype=DT, device=DEV)
    Kuf = ev.K(Zg, Xg[None].expand(S, N, D_in).reshape(S * N, D_in).contiguous())
    F, mean, cov = svgp_from_k_full_cov(Kug, Kuf, ev.K_blocks(Xg[None]), q_mu.cuda(), q_sqrt.cuda(), z.cuda(), O.JITTER)
    assert rel_err(mean, Fm[0]) < 1e-9 and rel_err(cov, Fv[0], var) < 1e-9 and rel_err(F, Fs[0]) < 1e-9, \
        (rel_err(mean, Fm[0]), rel_err(cov, Fv[0], var), rel_err(F, Fs[0]))


@pytest.mark.gpu
def test_refusals_launch_nothing_and_the_next_call_is_right():
    from dgp_toolbox_b200 import _lib
    ctx = _lib.get_context(0)
    M, D_out, N, S = 64, 1, 65, 2
    Ku, Kuf, Kff, _ = _rbf_problem(M, N, S, S, 3, 5)
    q_mu, q_sqrt = _q(M, D_out, 6)
    z = torch.as_tensor(np.random.default_rng(7).standard_normal((S, N, D_out)))
    g = [t.cuda() for t in (Ku, Kuf, Kff, q_mu, q_sqrt, z)]
    F_r, m_r, c_r = full_ref(Ku, Kuf, Kff, q_mu, q_sqrt, z)

    def right():
        m, c, F = _outs(S, N, D_out)
        _call_full(ctx, *g, N, S, m, c, F)
        assert rel_err(m, m_r) < 1e-9 and rel_err(c, c_r, 1.3) < 1e-9 and rel_err(F, F_r) < 1e-8

    def refused(match, *args, **kw):
        n0 = ctx.launch_count()
        with pytest.raises(_lib.DGPError, match=match):
            _call_full(ctx, *args, **kw)
        assert ctx.launch_count() == n0, match
        right()

    big = torch.zeros(769 * 769, dtype=DT, device=DEV).reshape(1, 769, 769)
    m, c, F = _outs(1, 769, D_out)
    refused("N > 768", g[0], torch.zeros(M, 769, dtype=DT, device=DEV), big, g[3], g[4],
            torch.zeros(1, 769, D_out, dtype=DT, device=DEV), 769, 1, m, c, F)
    m, c, F = _outs(S, N, D_out)
    refused("Kff_batch", *g, N, S, m, c, F, Kff_batch=3)
    refused("needs the draws", *g[:5], None, N, S, m, c, F)
    Sb, Nb = 16, 768
    Ku2, Kuf2, Kff2, _ = _rbf_problem(M, Nb, Sb, 1, 3, 8)
    zb = torch.zeros(Sb, Nb, D_out, dtype=DT, device=DEV)
    mb, cb, Fb = _outs(Sb, Nb, D_out)
    ctx.set_workspace_limit(64 << 20)              # the 2 x 16 factor blocks of 768 x 768 alone are 151 MB
    try:
        refused("workspace limit", Ku2.cuda(), Kuf2.cuda(), Kff2.cuda(), g[3], g[4], zb, Nb, Sb, mb, cb, Fb)
    finally:
        ctx.set_workspace_limit(int(float(os.environ.get("DGP_B200_WS_GB", "24")) * (1 << 30)))
    right()
    negI = -torch.eye(N, dtype=DT, device=DEV)[None].expand(S, N, N).contiguous()
    with pytest.raises(_lib.DGPError, match=r"\(-4\): .*not positive definite"):      # DGP_ERR_NUMERIC
        _call_full(ctx, g[0], g[1], negI, g[3], g[4], g[5], N, S, m, c, F)
    right()


# --------------------------------------------------------------------------------------------- (c) model level and wiring
def _ref_comp_K_blocks(roles, X, *theta):
    from dgp_toolbox_b200.composite import ROLE_PARAMS
    th = {r: None if t is None else t.detach().cpu() for r, t in zip(ROLE_PARAMS, theta)}
    Xc = X.detach().cpu()
    return torch.stack([CO.comp_K(Xc[b], None, roles["Da"], th) for b in range(Xc.shape[0])]).to(X.device)


def _ref_svgp_full(Ku, Kuf, Kff, q_mu, q_sqrt, z, jitter):
    assert jitter == O.JITTER
    S, N, D = z.shape
    F, mean, cov = full_ref(*[t.detach().cpu() for t in (Ku, Kuf, Kff, q_mu, q_sqrt)], z.detach().cpu().expand(S, N, D))
    return F.to(Ku.device), mean.to(Ku.device), cov.to(Ku.device)


def _use_full_reference(mp):
    from dgp_toolbox_b200 import composite
    from dgp_toolbox_b200.models import MF_DGP
    _use_reference(mp)
    mp.setattr(composite, "comp_K_blocks", _ref_comp_K_blocks)
    mp.setattr(MF_DGP, "svgp_from_k_full_cov", _ref_svgp_full)


def _ctor_draw(seed):
    rng = np.random.default_rng(seed)
    return lambda shape: torch.as_tensor(rng.standard_normal(shape), device=DEV)


def _mf_model(M=256, dims=(2, 2, 2)):
    from dgp_toolbox_b200.models import MF_DGP
    rng = np.random.default_rng(3)
    Z = [rng.uniform(0, 1, (M, d)) for d in dims]
    m = MF_DGP.DGP_Base.make_mf_dgp(Z, draw=_ctor_draw(1))
    _condition_layers(m.layers)
    return m, [m.layers]


def _em_model(M=64):
    from scipy.stats import qmc
    from dgp_toolbox_b200.models import MF_DGP_EM
    dims = [2, 3, 4]
    X = [np.random.default_rng(d).uniform(0, 1, (M, d)) for d in dims]
    sob = lambda d, s: qmc.Sobol(d, scramble=True, seed=s).random(M)
    em = MF_DGP_EM.DGP_Base.make_mf_dgp(X, [sob(d, 10 + d) for d in dims], [sob(4, 20), sob(3, 21)], draw=_ctor_draw(1))
    _condition_layers(list(em.layers) + list(em.layers_red))
    return em


def _mo_model(loop, M=64, d=3):
    from dgp_toolbox_b200.models import MO_DGP
    Zx = np.random.default_rng(0).uniform(0, 1, (M, d))
    mo = MO_DGP.DGP_Base.make_mf_dgp([np.concatenate([Zx, np.sin(3 * Zx[:, :1])], 1), Zx.copy()], loop=loop, draw=_ctor_draw(1))
    _condition_layers(mo.layers)
    return mo


def _compare_full(model, X, S, monkeypatch, **kw):
    draws = _Draws(11)
    model.draw = draws
    with torch.no_grad():
        out = model.propagate(X, full_cov=True, S=S, **kw)
    with monkeypatch.context() as mp, torch.no_grad():
        _use_full_reference(mp)
        model.draw = draws.replay()
        ref = model.propagate(X, full_cov=True, S=S, **kw)
    assert draws.i == len(draws.log)
    N = X.shape[0]
    for l, (F, m, v, Fr, mr, vr) in enumerate(zip(*out, *ref)):
        assert tuple(v.shape) == (S, N, N, m.shape[2])
        scale = float(torch.diagonal(vr, dim1=1, dim2=2).abs().max())
        e = (rel_err(m, mr), rel_err(v, vr, scale), rel_err(F, Fr))
        assert e[0] < 1e-9 and e[1] < 1e-9 and e[2] < 1e-8, (l, e)
    return out, ref


@pytest.mark.gpu
def test_mf_dgp_full_cov_matches_the_reference_wiring(monkeypatch):
    """MultiFidelityDeepGP's DGP_Base: 3 fidelities, M = 256, N = 512, S = 8; predict_f returns the last / selected entry."""
    model, _ = _mf_model()
    X = np.random.default_rng(5).uniform(0, 1, (512, 2))
    out, _ = _compare_full(model, X, 8, monkeypatch)
    draws = _Draws(11)
    model.draw = draws
    with torch.no_grad():
        m, v = model.predict_f(X, full_cov=True, S=8)
        model.draw = draws.replay()
        m0, v0 = model.predict_f(X, full_cov=True, S=8, fidelity=0)
    assert tuple(v.shape) == (8, 512, 512, 1) and tuple(v0.shape) == (8, 512, 512, 1)
    assert rel_err(m, out[1][-1]) < 1e-9 and rel_err(v0, out[2][0], float(v0.abs().max())) < 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize("fidelity_dim,project", [(None, False), (1, False), (0, False), (None, True)])
def test_mf_dgp_em_full_cov_matches_the_reference_wiring(monkeypatch, fidelity_dim, project):
    """MF-DGP-EM with 2/3/4-D inputs: through both projection layers, one, none (layer 0 on X itself), and the projection chain."""
    em = _em_model()
    dim = 4 if fidelity_dim is None else [2, 3, 4][fidelity_dim]
    X = np.random.default_rng(6).uniform(0, 1, (96, dim))
    _compare_full(em, X, 4, monkeypatch, fidelity_dim=fidelity_dim, project=project)


@pytest.mark.gpu
@pytest.mark.parametrize("loop", [0, 1, 2])
def test_mo_dgp_full_cov_matches_the_reference_wiring(monkeypatch, loop):
    mo = _mo_model(loop)
    X = np.random.default_rng(7).uniform(0, 1, (96, 3))
    out, _ = _compare_full(mo, X, 4, monkeypatch)
    draws = _Draws(11)
    mo.draw = draws
    with torch.no_grad():
        m, v = mo.predict_f(X, full_cov=True, S=4, objective=0)
    assert tuple(v.shape) == (4, 96, 96, 1) and rel_err(m, out[1][0]) < 1e-9


class _Zeros:
    def __call__(self, shape):
        return torch.zeros(shape, dtype=DT, device=DEV)


def _wiring_models():
    em = _em_model()
    return [("mf", _mf_model(M=64)[0], 2), ("em", em, 4), ("mo", _mo_model(2), 3)]


@pytest.mark.gpu
def test_zero_draws_give_the_diagonal_path_moments():
    """With every draw zero both modes feed the means forward: propagate(full_cov=True) has the full_cov=False means and, on the
    diagonal of its covariances, the full_cov=False variances (the diagonal path is pinned to the reference's own code)."""
    for name, model, d in _wiring_models():
        X = np.random.default_rng(8).uniform(0, 1, (80, d))
        model.draw = _Zeros()
        with torch.no_grad():
            Fs, Fm, Fv = model.propagate(X, full_cov=True, S=3)
            Fs0, Fm0, Fv0 = model.propagate(X, full_cov=False, S=3)
        assert len(Fm) == len(Fm0)
        for l in range(len(Fm)):
            dv = torch.diagonal(Fv[l], dim1=1, dim2=2).permute(0, 2, 1)
            assert rel_err(Fm[l], Fm0[l]) < 1e-12 and rel_err(dv, Fv0[l]) < 1e-12, (name, l, rel_err(Fm[l], Fm0[l]), rel_err(dv, Fv0[l]))
            assert rel_err(Fs[l], Fm[l]) == 0.0


@pytest.mark.gpu
def test_samples_are_mean_plus_cholesky_times_draws():
    """With nonzero draws, F = mean + chol(cov + jitter I) z for the first application of each chain (MF layer 0, EM's first
    projection layer; MO's first application is not returned, so its last one) and for the last application of every chain."""
    for name, model, d in _wiring_models():
        X = np.random.default_rng(9).uniform(0, 1, (80, d))
        draws = _Draws(12)
        model.draw = draws
        with torch.no_grad():
            Fs, Fm, Fv = model.propagate(X, full_cov=True, S=3, **({"project": True} if name == "em" else {}))
        if name == "em":
            Fs, Fm, Fv = Fs[1:], Fm, Fv                 # Hs[0] is X itself
        checks = [(-1, -1)] + ([(0, 0)] if name != "mo" else [])
        for l, k in checks:
            z = draws.log[k].cpu()
            F_r = O.reparameterize_full(Fm[l].cpu(), Fv[l].cpu(), z)
            assert rel_err(Fs[l], F_r) < 1e-8, (name, l, rel_err(Fs[l], F_r))


@pytest.mark.gpu
def test_gradient_request_under_full_cov_raises():
    model, _ = _mf_model(M=64)
    X = torch.rand(10, 2, dtype=DT, device=DEV, requires_grad=True)
    with pytest.raises(NotImplementedError, match="no adjoint"):
        model.propagate(X, full_cov=True, S=2)
    p = model.layers[0].q_mu
    with pytest.raises(NotImplementedError, match="no adjoint"):
        model.propagate(X.detach(), full_cov=True, S=2, values={p: p.value.clone().requires_grad_(True)})
    mo = _mo_model(1)
    with pytest.raises(NotImplementedError, match="no adjoint"):
        mo.propagate(torch.rand(10, 3, dtype=DT, device=DEV, requires_grad=True), full_cov=True, S=2)
    em = _em_model()
    with pytest.raises(NotImplementedError, match="no adjoint"):
        em.propagate(torch.rand(10, 4, dtype=DT, device=DEV, requires_grad=True), full_cov=True, S=2)


@pytest.mark.gpu
def test_one_layer_application_at_s250_launches_the_blocked_kernel_once():
    from torch.profiler import ProfilerActivity, profile
    model, _ = _mf_model(M=64)
    layer = model.layers[1]
    N, S = 40, 250
    X = torch.rand(S, N, layer.D, dtype=DT, device=DEV)
    layer.sample_from_conditional(X, full_cov=True, draw=_Zeros())       # warm up
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof, torch.no_grad():
        F, mean, cov = layer.sample_from_conditional(X, full_cov=True, draw=_Zeros())
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert sum("compk_K_blocks_kernel" in n for n in names) == 1, [n for n in names if "compk" in n]
    assert sum("fullcov_ext_kernel" in n for n in names) == 1
    assert tuple(cov.shape) == (S, N, N, 1)
