"""The acquisition epilogues of csrc/acq.cuh against arbitrary-precision (mpmath) references at their numerical edges.

These kernels turn the chain's per-sample moments into the numbers a BO search ranks: mixture_moments_kernel (dgp_mixture_moments,
dgp_predict_moments, EI.run), ei_analytic_kernel, ei_upstream_kernel (dgp_acq_grad), acq_moments_kernel (dgp_acq_moments) and the
exact 2-D EHVI kernels. The float64 oracle restates the same formulas and only meets them at benign moments, so it cannot show
where they are inaccurate; the references here are computed from the exact double inputs at DPS decimal digits, and every bound
is stated in units of the machine epsilon EPS of float64:
  - mixture moments: |d mean| <= 2 S EPS mean_s |m_s|, |d var| <= 4 S EPS var (the centred two-pass form; the one-pass
    mean_s (v + m^2) - mean^2 cancels when |mean| is large next to the spread, see test_one_pass_replay_violates_the_moment_bound);
  - EI-type criteria on (mean, var): 8 (1 + u^4) EPS scale on the cancelling side of EI = (y - m) Phi(u) + s phi(u), where the
    formula loses accuracy as u^4 (the reference's formula, kept as it is), 8 (1 + u^2) EPS scale elsewhere, plus a floor of a few
    subnormal ulps where the terms leave the normal range; exactly 0 where EI underflows;
  - EHVI strip sums and their partials: 16 EPS T + 2 n EPS A (ehvi_bound), with T what an error of eps times its rounding scale in
    either factor of each strip moves the sum by, and A = sum_i |strip_i| for the rounding of the n-term sum (mp_ehvi_scales).
The CPU self-tests at the end (not marked gpu) check the references against scipy and numpy, replay the kernels' formulas in numpy
to show the bounds hold with margin, and show that the one-pass reduction violates the moment bound on the offset cases."""
import ctypes as C
import types

import numpy as np
import pytest
import torch
from mpmath import mp

from oracle import dgp_oracle as O
from tests.helpers import _condition, product_model_from_problem

EPS = float(np.finfo(np.float64).eps)
TINY = 2.0 ** -1074                       # the smallest subnormal
DBL_MIN = float(np.finfo(np.float64).tiny)  # the smallest normal
DPS = 40
GPU = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------------------------------
# mpmath references
# ---------------------------------------------------------------------------------------------------------------------------
def mp_moments(Fm, Fv, add=0.0):
    """Exact mixture moments of the columns of Fm, Fv [S, K] (doubles taken exactly): [(mean, var, mean_s |m_s|)] per column,
    var = mean_s (v_s + add) + mean_s (m_s - mean)^2."""
    S, K = Fm.shape
    out = []
    with mp.workdps(DPS):
        a = mp.mpf(float(add))
        for k in range(K):
            ms = [mp.mpf(float(x)) for x in Fm[:, k]]
            mu = mp.fsum(ms) / S
            var = (mp.fsum(mp.mpf(float(x)) for x in Fv[:, k]) + S * a + mp.fsum((m - mu) ** 2 for m in ms)) / S
            out.append((mu, var, mp.fsum(abs(m) for m in ms) / S))
    return out


def mp_criterion(kind, m, v, y, x=()):
    """dgp_acq_moments kinds 0-4 on exact (m, v): -EI, -(EI - m), EV, [-(sig(x_j) EI - m)], Phi((y - m) / s). Also returns the
    criterion's argument (u, or t for EV) and its adjoints (dc/dm, dc/dv) as dgp_acq_grad defines them (kind 3: of sum_j)."""
    with mp.workdps(DPS):
        m, v, y = mp.mpf(m), mp.mpf(v), mp.mpf(y)
        s = mp.sqrt(v)
        if kind == 4:
            u = (y - m) / s
            return mp.ncdf(u), u, None
        if kind == 2:
            t = (m - y) / s
            return (m - y) * mp.ncdf(t) + s * mp.npdf(t), t, (mp.ncdf(t), mp.npdf(t) / (2 * s))
        u = (y - m) / s
        ei = (y - m) * mp.ncdf(u) + s * mp.npdf(u)
        dm, dv = mp.ncdf(u), -mp.npdf(u) / (2 * s)
        if kind == 0:
            return -ei, u, (dm, dv)
        if kind == 1:
            return -(ei - m), u, (dm + 1, dv)
        sig = [1 / (1 + mp.exp(-mp.mpf(float(xj)))) for xj in x]
        return [-(sg * ei - m) for sg in sig], u, (dm * mp.fsum(sig) + len(sig), dv * mp.fsum(sig), ei, sig)


def criterion_bound(kind, value, u, m, v, ei=0.0):
    """Allowed |computed - exact| of a criterion value (see the module docstring). `value` is the exact criterion, u its argument.
    WB2S (kind 3, pass its EI): sig(x) = 1 / (1 + 1 / exp(x)) is 0 below x ~ -709.8, where the exact sigmoid is subnormal.
    A Phi(u) below the normal range may come out as 0 (erfc need not return subnormals): that term's whole size is allowed."""
    with mp.workdps(DPS):
        cdf = float(mp.ncdf(u))
    flushed = cdf if cdf < DBL_MIN else 0.0
    u, value, m, v = float(u), abs(float(value)), abs(float(m)), float(v)
    if kind == 4:
        return 8 * (1 + u * u) * EPS * value + 8 * (1 + u * u) * TINY + 2 * flushed
    scale = value + (m if kind in (1, 3) else 0.0)
    fac = 1 + u ** 4 if u < 0 else 1 + u * u
    floor = 8 * (1 + abs(u)) * max(1.0, v) * TINY + 2 * abs(u) * np.sqrt(v) * flushed
    return 8 * fac * EPS * scale + floor + 2 * abs(float(ei)) * DBL_MIN


def _psi(a, b, mu, s):
    u = (b - mu) / s
    return s * mp.npdf(u) + (a - mu) * mp.ncdf(u)


def mp_ehvi(m0, v0, m1, v1, y0, y1):
    """The strip sum of EHVI.py:154-157 on the padded front (y0, y1)."""
    s0, s1 = mp.sqrt(v0), mp.sqrt(v1)
    n = len(y0)
    cl = mp.ncdf((y0[-1] - m0) / s0)
    terms = []
    for i in range(1, n):
        d1 = _psi(y1[i], y1[i], m1, s1) - _psi(y1[i], y1[0], m1, s1)
        f = _psi(y0[i - 1], y0[i - 1], m0, s0) - _psi(y0[i - 1], y0[i], m0, s0)
        if i < n - 1:
            f += (y0[i - 1] - y0[i]) * (mp.ncdf((y0[i] - m0) / s0) - cl)
        terms.append(f * d1)
    return mp.fsum(terms)


def _psi_mags(a, b, mu, s):
    """Rounding scales of psi(a, b, mu, s) = s phi(u) + (a - mu) Phi(u), u = (b - mu) / s, and of its derivatives w.r.t. mu and
    v = s^2 as a kernel computes them: every piece in absolute value; a relative error eps of u costs a phi(u) piece u^2 eps (through
    exp) and a Phi(u) piece |u| phi(u) eps, so the phi-bearing pieces carry (1 + u^2) and the Phi pieces add |u| phi."""
    u = (b - mu) / s
    pdf, cdf, am, g = mp.npdf(u), mp.ncdf(u), abs(a - mu), 1 + u * u
    val = s * pdf * g + am * (cdf + abs(u) * pdf)
    dmu = abs(u) * pdf * g + cdf + abs(u) * pdf + am * pdf * g / s            # u phi - Phi - (a - mu) phi / s
    dv = (pdf * g * g + am * abs(u) * pdf * g / s) / (2 * s)                   # (phi (1 + u^2) - (a - mu) phi u / s) / (2 s)
    return val, dmu, dv


def _cdf_mags(b, mu, s):
    """The same for Phi(u) and its derivatives -phi / s and -u phi / (2 s^2)."""
    u = (b - mu) / s
    pdf, g = mp.npdf(u), 1 + u * u
    return mp.ncdf(u) + abs(u) * pdf, pdf * g / s, abs(u) * pdf * g / (2 * s * s)


def _strip_f(i, m0, v0, y0):
    """The objective-0 factor of strip i (exact)."""
    s0 = mp.sqrt(v0)
    f = _psi(y0[i - 1], y0[i - 1], m0, s0) - _psi(y0[i - 1], y0[i], m0, s0)
    if i < len(y0) - 1:
        f += (y0[i - 1] - y0[i]) * (mp.ncdf((y0[i] - m0) / s0) - mp.ncdf((y0[-1] - m0) / s0))
    return f


def _strip_d1(i, m1, v1, y1):
    """The objective-1 factor of strip i (exact)."""
    s1 = mp.sqrt(v1)
    return _psi(y1[i], y1[i], m1, s1) - _psi(y1[i], y1[0], m1, s1)


def mp_ehvi_scales(m0, v0, m1, v1, y0, y1):
    """How far the rounding of a strip sum can move it: [T, T_m0, T_v0, T_m1, T_v1] and [A, A_m0, A_v0, A_m1, A_v1]. Strip i is f_i d1_i; an error of each factor
    within eps times its rounding scale M (built from _psi_mags / _cdf_mags) moves the strip by eps (|f| M(d1) + M(f) |d1|), and the
    partial derivative (f d1)' = f' d1 + f d1' by eps (M(f') |d1| + |f'| M(d1) + M(f) |d1'| + |f| M(d1')). The exact factors and
    their derivatives come from mpmath (mp.diff). A = sum_i |f_i d1_i| (and sum_i |(f_i d1_i)'|) is what the rounding of the
    n-term sum scales with. T >= A; it is larger where a factor is itself a cancelled difference (sigma large next to the front),
    and so is the error a kernel makes there."""
    s0, s1 = mp.sqrt(v0), mp.sqrt(v1)
    n = len(y0)
    cl = _cdf_mags(y0[-1], m0, s0)
    T, A = [mp.mpf(0)] * 5, [mp.mpf(0)] * 5
    for i in range(1, n):
        pa, pb = _psi_mags(y1[i], y1[i], m1, s1), _psi_mags(y1[i], y1[0], m1, s1)
        Md1 = [pa[k] + pb[k] for k in range(3)]
        qa, qb = _psi_mags(y0[i - 1], y0[i - 1], m0, s0), _psi_mags(y0[i - 1], y0[i], m0, s0)
        Mf = [qa[k] + qb[k] for k in range(3)]
        if i < n - 1:
            w, ci = abs(y0[i - 1] - y0[i]), _cdf_mags(y0[i], m0, s0)
            Mf = [Mf[k] + w * (ci[k] + cl[k]) for k in range(3)]
        f, d1 = abs(_strip_f(i, m0, v0, y0)), abs(_strip_d1(i, m1, v1, y1))
        fm = abs(mp.diff(lambda t: _strip_f(i, t, v0, y0), m0, h=s0 * mp.mpf("1e-20")))
        fv = abs(mp.diff(lambda t: _strip_f(i, m0, t, y0), v0, h=v0 * mp.mpf("1e-20")))
        dm = abs(mp.diff(lambda t: _strip_d1(i, t, v1, y1), m1, h=s1 * mp.mpf("1e-20")))
        dv = abs(mp.diff(lambda t: _strip_d1(i, m1, t, y1), v1, h=v1 * mp.mpf("1e-20")))
        T[0] += f * Md1[0] + Mf[0] * d1
        T[1] += Mf[1] * d1 + fm * Md1[0]
        T[2] += Mf[2] * d1 + fv * Md1[0]
        T[3] += Mf[0] * dm + f * Md1[1]
        T[4] += Mf[0] * dv + f * Md1[2]
        for k, t in enumerate((f * d1, fm * d1, fv * d1, f * dm, f * dv)):
            A[k] += t
    return T, A


def ehvi_bound(n, T, A, k):
    """|computed - exact| allowed for the value (k = 0) or partial k - 1 of an n-entry strip sum: 16 EPS per strip's rounding scale,
    2 n EPS for the sequential sum, and 16 n subnormal ulps."""
    return 16 * EPS * float(T[k]) + 2 * n * EPS * float(A[k]) + 16 * n * TINY


def mp_ehvi_partials(m0, v0, m1, v1, y0, y1):
    """(dE/dm0, dE/dv0, dE/dm1, dE/dv1) by mp.diff (central differences at raised precision), independent of psi_grad."""
    s0, s1 = mp.sqrt(v0), mp.sqrt(v1)
    return [mp.diff(lambda t: mp_ehvi(t, v0, m1, v1, y0, y1), m0, h=s0 * mp.mpf("1e-20")),
            mp.diff(lambda t: mp_ehvi(m0, t, m1, v1, y0, y1), v0, h=v0 * mp.mpf("1e-20")),
            mp.diff(lambda t: mp_ehvi(m0, v0, t, v1, y0, y1), m1, h=s1 * mp.mpf("1e-20")),
            mp.diff(lambda t: mp_ehvi(m0, v0, m1, t, y0, y1), v1, h=v1 * mp.mpf("1e-20"))]


# ---------------------------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------------------------
OFFSETS = (0.0, 1.0, -50.0, 300.0, 1e3)
SPREADS = (0.0, 1e-4, 1e-2, 1.0)
VARS = (0.0, 1e-12, 1e-9, 1e-8, 0.1)
GRID = [(o, sp, v) for o in OFFSETS for sp in SPREADS for v in VARS]      # 100 columns
LIK = 1e-9


def grid_samples(S, ND, seed):
    """Fm, Fv [S, ND]: column j is GRID[j % 100]: m_s = offset + spread z_s, v_s = v w_s with w_s in [0.5, 1.5)."""
    rng = np.random.default_rng(seed)
    cols = np.array([GRID[j % len(GRID)] for j in range(ND)])
    Fm = cols[:, 0] + cols[:, 1] * rng.standard_normal((S, ND))
    Fv = cols[:, 2] * rng.uniform(0.5, 1.5, (S, ND))
    return Fm, Fv


def one_pass(Fm, Fv, add=0.0):
    """numpy replay of the parent's mixture_moments_kernel: sequential sums, var = sq / S - mean^2."""
    sm, sq = np.zeros(Fm.shape[1]), np.zeros(Fm.shape[1])
    for s in range(Fm.shape[0]):
        sm = sm + Fm[s]
        sq = sq + ((Fv[s] + add) + Fm[s] * Fm[s])
    mu = sm / Fm.shape[0]
    return mu, sq / Fm.shape[0] - mu * mu


def centred(Fm, Fv, add=0.0):
    """numpy replay of the centred two-pass mixture_moments_kernel."""
    sm = np.zeros(Fm.shape[1])
    for s in range(Fm.shape[0]):
        sm = sm + Fm[s]
    mu = sm / Fm.shape[0]
    acc = np.zeros(Fm.shape[1])
    for s in range(Fm.shape[0]):
        d = Fm[s] - mu
        acc = acc + ((Fv[s] + add) + d * d)
    return mu, acc / Fm.shape[0]


def moment_violations(mean, var, ref, S, cols):
    """Columns (with ratios) where (mean, var) break the mixture-moment bounds against the mpmath reference `ref` of `cols`."""
    bad = []
    for k, (mu, vx, mabs) in zip(cols, ref):
        dm = abs(mp.mpf(float(mean[k])) - mu)
        dv = abs(mp.mpf(float(var[k])) - vx)
        if dm > 2 * S * EPS * mabs or dv > 4 * S * EPS * vx or (vx == 0 and var[k] != 0.0):
            bad.append((k, float(dm), float(dv), float(vx)))
    return bad


def u_grid():
    return np.unique(np.concatenate([np.linspace(-40.0, 40.0, 81), [-38.5, 38.5, -38.6, -38.65, -37.5, -0.5, 0.5, -1e-3, 1e-3]]))


SIGMAS = (1e-6, 1e-2, 1.0, 1e3)
ACQ_OFFSETS = (0.0, 1.5, -50.0, 1e3)
XS = (0.3, -2.0, 710.0, -720.0, 800.0, -709.5)


def acq_inputs():
    """(mean, var, y, u) over the u grid x sigma x offset: y = m + u s for every kind but EV, for which y = m - u s (so that its
    argument t = (m - y) / s runs over the grid too); mean and y are doubles and the references take them as they are."""
    rows = [(o, s, u) for o in ACQ_OFFSETS for s in SIGMAS for u in u_grid()]
    m = np.array([r[0] for r in rows])
    s = np.array([r[1] for r in rows])
    u = np.array([r[2] for r in rows])
    return m, s * s, s, u


# ---------------------------------------------------------------------------------------------------------------------------
# device helpers
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.fixture
def ctx():
    """The device context, with every flag this file touches restored afterwards."""
    import dgp_toolbox_b200 as D
    c = D._lib.get_context(0)
    try:
        yield c
    finally:
        c.set_fused(True)
        c.set_vform(True, True)


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def _p(t):
    import dgp_toolbox_b200 as D
    return D._lib.ptr(t)


def device_moments(ctx, Fm, Fv, lik):
    S, ND = Fm.shape
    fm, fv = _dev(Fm), _dev(Fv)
    lk = _dev(np.array([lik])) if lik else None
    mean, var = torch.empty(ND, dtype=torch.float64, device="cuda"), torch.empty(ND, dtype=torch.float64, device="cuda")
    ctx.call("dgp_mixture_moments", _p(fm), _p(fv), S, ND, _p(lk) if lik else None, _p(mean), _p(var))
    torch.cuda.synchronize()
    return mean.cpu().numpy(), var.cpu().numpy()


def acq_grad(ctx, pm, kind, X, S, zs, y, value=None):
    """dgp_acq_grad on the host array X with the draws zs: (value, d_value_dX) as numpy. kind 4 takes `value` [N, 1, 2] as input."""
    N, d0 = X.shape
    Xd = _dev(X)
    m, keep = pm._model_desc()
    zt, zp = pm._zs(zs, S, N)
    if value is None:
        val = torch.empty((N, d0 if kind == 3 else 1), dtype=torch.float64, device="cuda")
    else:
        val = _dev(value)
    dx = torch.zeros((N, d0), dtype=torch.float64, device="cuda")
    ctx.call("dgp_acq_grad", C.byref(m), kind, _p(Xd), N, S, zp, 0, 0, float(y), _p(val), _p(dx))
    torch.cuda.synchronize()
    return val.cpu().numpy(), dx.cpu().numpy()


# ---------------------------------------------------------------------------------------------------------------------------
# 1a. dgp_mixture_moments called directly
# ---------------------------------------------------------------------------------------------------------------------------
@GPU
@pytest.mark.parametrize("S", [1, 2, 33, 1000, 4096])
def test_mixture_moments_grid(ctx, S):
    """The (offset, spread, v) grid across the columns of one call, with and without a likelihood variance."""
    Fm, Fv = grid_samples(S, len(GRID), S)
    ref0 = mp_moments(Fm, Fv)
    cols = list(range(len(GRID)))
    for lik in (0.0, LIK):
        ref = ref0 if not lik else [(mu, vx + mp.mpf(lik), ma) for mu, vx, ma in ref0]
        mean, var = device_moments(ctx, Fm, Fv, lik)
        assert np.isfinite(var).all() and (var >= 0).all(), (S, lik)
        bad = moment_violations(mean, var, ref, S, cols)
        assert not bad, (S, lik, [(GRID[k], r) for k, *r in bad[:5]])
        worst = max(float(abs(mp.mpf(float(var[k])) - vx) / (4 * S * EPS * vx)) if vx else 0.0 for k, (mu, vx, _) in enumerate(ref))
        print(f"mixture moments S={S} lik={lik}: largest var error / bound {worst:.3g}")


@GPU
@pytest.mark.parametrize("ND", [1, 255, 257, 70001])
@pytest.mark.parametrize("S", [1, 2])
def test_mixture_moments_partial_blocks(ctx, S, ND):
    """Partial blocks and the grid tail: every column finite and non-negative, a sample including the first and last columns
    against the reference."""
    Fm, Fv = grid_samples(S, ND, 7 * ND + S)
    cols = sorted(set([0, ND - 1] + list(range(0, ND, max(1, ND // 150)))))
    for lik in (0.0, LIK):
        mean, var = device_moments(ctx, Fm, Fv, lik)
        assert np.isfinite(mean).all() and np.isfinite(var).all() and (var >= 0).all(), (S, ND, lik)
        ref = mp_moments(Fm[:, cols], Fv[:, cols], lik)
        bad = moment_violations(mean, var, ref, S, cols)
        assert not bad, (S, ND, lik, bad[:5])


# ---------------------------------------------------------------------------------------------------------------------------
# 1b / 1c. the same reduction inside the chain's epilogues
# ---------------------------------------------------------------------------------------------------------------------------
def offset_model(units, S, offset=1e3):
    """D0 = 2, M = 30, last layer with a Linear mean (W = 0.05, b = offset), q_sqrt = 1e-4 I and a likelihood variance of 1e-8.
    X = the first layer's inducing inputs (tiny per-sample variance there), ten other points and two with |x| > 709."""
    prob = O.synthetic_problem(2, units, 30, 10, lik_var=1e-8)
    last = prob["layers"][-1]
    last["mean_kind"], last["mf_W"], last["mf_b"] = "linear", np.full((last["Z"].shape[1], 1), 0.05), np.array([offset])
    for layer in prob["layers"]:
        layer["q_sqrt"] = 1e-4 * np.repeat(np.eye(30)[None], layer["q_mu"].shape[1], 0)
    prob = _condition(prob)
    pm = product_model_from_problem(prob, S)
    X = np.concatenate([prob["layers"][0]["Z"], prob["X"], [[710.0, 0.2], [-720.0, -0.1]]])
    return pm, X


def benign_model(S):
    """The synthetic problem as it is (zero-mean last layer, q_sqrt = 0.5 I + noise): |mean| ~ 1, |u| <= 10."""
    prob = _condition(O.synthetic_problem(2, [2], 30, 40))
    return product_model_from_problem(prob, S), prob["X"]


def _draws(pm, S, N, seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(S, N, l.num_outputs, dtype=torch.float64, generator=g) for l in pm.layers]


_CASES = {}


def model_case(name, S):
    """(pm, X, zs, Fm, Fv, ref_f, ref_y, lik, sigma2): the last layer's per-sample moments from propagate with the draws zs and
    their exact mixture moments (predict_f and predict_y), cached per module."""
    key = (name, S)
    if key not in _CASES:
        pm, X = {"one-layer": lambda: offset_model([], S), "two-layer": lambda: offset_model([2], S),
                 "benign": lambda: benign_model(S)}[name]()
        zs = _draws(pm, S, X.shape[0], 11 + S)
        _, Fms, Fvs = pm.propagate(X, S=S, zs=zs)
        torch.cuda.synchronize()
        Fm, Fv = Fms[-1][:, :, 0].cpu().numpy(), Fvs[-1][:, :, 0].cpu().numpy()
        lik = float(pm.likelihood.likelihood.variance.value.reshape(-1)[0])
        ref_f = mp_moments(Fm, Fv)
        ref_y = [(mu, vx + mp.mpf(lik), ma) for mu, vx, ma in ref_f]
        sigma2 = float(pm.layers[-1].kern.variance.value.reshape(-1)[0])
        _CASES[key] = (pm, X, zs, Fm, Fv, ref_f, ref_y, lik, sigma2)
    return _CASES[key]


def moment_tols(ref, S, sigma2):
    """The 1a bounds plus 1e-12 sigma^2 of the last layer for the chain's own rounding."""
    return ([2 * S * EPS * float(ma) + 1e-12 * np.sqrt(sigma2) for _, _, ma in ref],
            [4 * S * EPS * float(vx) + 1e-12 * sigma2 for _, vx, _ in ref])


def _y_for(ref, p=0, shift=0.5):
    """A threshold at shift sigma from the exact mean of point p (a moderate u there)."""
    mu, vx, _ = ref[p]
    return float(mu + shift * mp.sqrt(vx))


def check_values(kind, got, ref, y, tm, tv, what):
    """got [N] against the criterion on the exact moments, with the moment tolerances carried through the adjoints."""
    worst = 0.0
    for k, (mu, vx, _) in enumerate(ref):
        c, u, (dm, dv) = mp_criterion(kind, mu, vx, y)[:3]
        tol = abs(float(dm)) * tm[k] + abs(float(dv)) * tv[k] + criterion_bound(kind, c, u, mu, vx)
        err = abs(float(mp.mpf(float(got[k])) - c))
        worst = max(worst, err / tol)
        assert err <= tol, (what, kind, k, float(c), float(got[k]), err, tol)
    return worst


@GPU
@pytest.mark.parametrize("S", [1, 1000])
@pytest.mark.parametrize("name", ["one-layer", "two-layer"])
def test_chain_epilogues_match_exact_mixture_moments(ctx, name, S):
    """predict_moments, EI.run(analytic=True) and the values of dgp_acq_grad kinds 0-2 against the mpmath reduction of the
    per-sample moments propagate gives with the same draws, on a model whose last-layer mean sits at 1e3 with a per-sample
    variance of ~1e-6 at the inducing inputs. The one-pass reduction misses here by ~1e-10 absolute in var at S = 1000."""
    import dgp_toolbox_b200 as D
    pm, X, zs, Fm, Fv, ref_f, ref_y, lik, sigma2 = model_case(name, S)
    for add, ref in ((False, ref_f), (True, ref_y)):
        tm, tv = moment_tols(ref, S, sigma2)
        mean, var = pm.predict_moments(X, S, add_lik_var=add, zs=zs)
        mean, var = mean.cpu().numpy().reshape(-1), var.cpu().numpy().reshape(-1)
        assert (var > 0).all()
        for k, (mu, vx, _) in enumerate(ref):
            assert abs(float(mp.mpf(float(mean[k])) - mu)) <= tm[k], (name, S, add, "mean", k)
            assert abs(float(mp.mpf(float(var[k])) - vx)) <= tv[k], (name, S, add, "var", k, float(var[k]), float(vx))
    tm_f, tv_f = moment_tols(ref_f, S, sigma2)
    tm_y, tv_y = moment_tols(ref_y, S, sigma2)
    worst = 0.0
    for shift in (0.5, -3.0):
        y = _y_for(ref_f, 0, shift)
        neg_ei = D.EI(y, 2).run(pm, X, analytic=True, num_samples=S, zs=zs).cpu().numpy().reshape(-1)
        worst = max(worst, check_values(0, neg_ei, ref_f, y, tm_f, tv_f, "dgp_ei"))
        val, _ = acq_grad(ctx, pm, 0, X, S, zs, y)
        worst = max(worst, check_values(0, val.reshape(-1), ref_f, y, tm_f, tv_f, "acq_grad"))
        yy = _y_for(ref_y, 0, shift)
        for kind in (1, 2):
            val, _ = acq_grad(ctx, pm, kind, X, S, zs, yy)
            worst = max(worst, check_values(kind, val.reshape(-1), ref_y, yy, tm_y, tv_y, "acq_grad"))
    print(f"chain epilogues {name} S={S}: largest error / bound {worst:.3g}")


def _spread(kind, mu, vx, y, xk, tm, tv, c, a):
    """The largest change of the criterion values and of (dc/dm, dc/dv, EI) over the corners (mu +- tm, vx +- tv): what the
    kernel's legitimately rounded moments may move them by."""
    dc, da = [0.0] * (len(c) if kind == 3 else 1), [0.0, 0.0, 0.0]
    for sm in (-1, 1):
        for sv in (-1, 1):
            cc, _, aa = mp_criterion(kind, mu + sm * tm, max(vx + sv * tv, vx / 2), y, xk)
            cs, c0 = (cc, c) if kind == 3 else ([cc], [c])
            dc = [max(dc[j], abs(float(cs[j] - c0[j]))) for j in range(len(dc))]
            da = [max(da[i], abs(float(aa[i] - a[i]))) for i in range(3 if kind == 3 else 2)] + ([] if kind == 3 else [0.0])
    return dc, da


@GPU
@pytest.mark.parametrize("S", [1, 1000])
@pytest.mark.parametrize("name", ["benign", "one-layer", "two-layer"])
def test_acq_grad_adjoints_match_exact_criterion_adjoints(ctx, name, S):
    """d_value_dX of dgp_acq_grad kinds 0-2 against a kind-4 call on the same model, draws and X fed the adjoints (dc/dmean,
    dc/dvar) mpmath computes from the exact mixture moments: both run the same adjoint chain, so a difference comes from the
    criterion's adjoints inside ei_upstream_kernel. Kind 3 (WB2S): value and input gradient (chain + explicit -sig'(x) EI term)
    against mpmath, including inputs with |x| > 709 where the sigmoid saturates.
    Tolerance per point: 1e-10 max |d_value_dX| plus what the 1a rounding of the moments may move the adjoints by, carried
    through the chain (kind-4 calls with unit adjoints give each point's d/d(dc/dm) and d/d(dc/dv)). The mean's own rounding
    matters where sigma is small next to |mean|: at mean 1e3, sigma 1e-3 and S = 1000 it moves u by up to ~4e-7."""
    pm, X, zs, Fm, Fv, ref_f, ref_y, lik, sigma2 = model_case(name, S)
    N = X.shape[0]
    worst = 0.0
    for kind in (0, 1, 2, 3):
        ref = ref_f if kind == 0 else ref_y
        tm, tv = moment_tols(ref, S, sigma2)
        y4 = 0.0 if kind == 0 else 1.0                 # kind 4: y != 0 selects predict_y moments
        _, Jm = acq_grad(ctx, pm, 4, X, S, zs, y4, value=np.tile([1.0, 0.0], (N, 1, 1)))
        _, Jv = acq_grad(ctx, pm, 4, X, S, zs, y4, value=np.tile([0.0, 1.0], (N, 1, 1)))
        for shift in (0.5, -2.0):
            y = _y_for(ref, 0, shift) if name != "benign" else float(np.median([float(r[0]) for r in ref])) + shift * 0.1
            val, dx = acq_grad(ctx, pm, kind, X, S, zs, y)
            adj = np.zeros((N, 1, 2))
            direct, slack = np.zeros_like(X), np.zeros_like(X)
            for k, (mu, vx, _) in enumerate(ref):
                xk = X[k] if kind == 3 else ()
                c, u, a = mp_criterion(kind, mu, vx, y, xk)
                dc, da = _spread(kind, mu, vx, y, xk, tm[k], tv[k], c, a)
                adj[k, 0] = [float(a[0]), float(a[1])]
                slack[k] = da[0] * np.abs(Jm[k]) + da[1] * np.abs(Jv[k])
                if kind == 3:
                    ei, sig = a[2], a[3]
                    direct[k] = [float(-sg * (1 - sg) * ei) for sg in sig]
                    slack[k] += [float(sg * (1 - sg)) * da[2] for sg in sig]
                    for j in range(X.shape[1]):
                        err = abs(float(mp.mpf(float(val[k, j])) - c[j]))
                        assert err <= criterion_bound(3, c[j], u, mu, vx, ei) + dc[j], (name, S, k, j, float(c[j]), float(val[k, j]))
            _, dx4 = acq_grad(ctx, pm, 4, X, S, zs, y4, value=adj)
            want = dx4 + direct
            tol = 1e-10 * max(float(np.abs(want).max()), 1e-300) + slack
            ratio = float((np.abs(dx - want) / tol).max())
            worst = max(worst, ratio)
            assert ratio <= 1.0, (name, S, kind, shift, ratio, float(np.abs(dx - want).max()))
    print(f"acq_grad adjoints {name} S={S}: largest error / tolerance {worst:.3g}")


# ---------------------------------------------------------------------------------------------------------------------------
# 1d. dgp_acq_moments on supplied (mean, var)
# ---------------------------------------------------------------------------------------------------------------------------
_ACQ_REF = {}


def acq_reference(kind):
    if kind not in _ACQ_REF:
        m, v, s, u = acq_inputs()
        y = m - u * s if kind == 2 else m + u * s
        x = np.array([[XS[i % len(XS)], XS[(i + 1) % len(XS)]] for i in range(len(m))])
        refs = [mp_criterion(kind, m[i], v[i], y[i], x[i] if kind == 3 else ()) for i in range(len(m))]
        _ACQ_REF[kind] = (m, v, y, x, refs)
    return _ACQ_REF[kind]


def acq_violations(kind, got, m, v, refs):
    """(largest error / bound, list of violations) of the device values `got` [n] or [n, d] against the references."""
    worst, bad = 0.0, []
    for i, (c, u, a) in enumerate(refs):
        cs = c if kind == 3 else [c]
        ei = a[2] if kind == 3 else 0.0
        gs = got[i] if kind == 3 else [got[i]]
        for cj, gj in zip(cs, gs):
            if not np.isfinite(gj):
                bad.append((i, "nan", float(u)))
                continue
            b = criterion_bound(kind, cj, u, m[i], v[i], ei)
            err = abs(float(mp.mpf(float(gj)) - cj))
            worst = max(worst, err / b)
            if err > b:
                bad.append((i, float(u), float(m[i]), float(v[i]), float(cj), float(gj), err / b))
    return worst, bad


@GPU
@pytest.mark.parametrize("kind", [0, 1, 2, 3, 4])
def test_acq_moments_criteria_at_their_edges(ctx, kind):
    """-EI, WB2, EV, WB2S and PoF on u (t for EV) from -40 to 40 including +-38.5 and the underflow boundary, sigma from 1e-6 to
    1e3 and offsets up to 1e3, against mpmath; where EI underflows (u <= -38.65) the criterion is exactly 0 (EI, EV) or exactly
    the mean (WB2, WB2S)."""
    m, v, y, x, refs = acq_reference(kind)
    n, d = len(m), x.shape[1]
    got = np.empty((n, d) if kind == 3 else (n,))
    for yv in np.unique(y):            # one call per threshold: y is a scalar argument
        idx = np.flatnonzero(y == yv)
        mi, vi, xi = _dev(m[idx]), _dev(v[idx]), _dev(x[idx])
        oi = torch.empty((len(idx), d) if kind == 3 else (len(idx),), dtype=torch.float64, device="cuda")
        ctx.call("dgp_acq_moments", kind, _p(mi), _p(vi), len(idx), float(yv), _p(xi) if kind == 3 else None, d if kind == 3 else 0,
                 _p(oi))
        torch.cuda.synchronize()
        got[idx] = oi.cpu().numpy()
    worst, bad = acq_violations(kind, got, m, v, refs)
    assert not bad, (kind, len(bad), bad[:5])
    u = np.array([float(r[1]) for r in refs])
    under = u <= -38.65
    if kind in (0, 2):
        assert (got[under] == 0.0).all()
    elif kind == 1:
        assert (got[under] == m[under]).all()
    elif kind == 3:
        assert (got[under] == m[under][:, None]).all()
    print(f"dgp_acq_moments kind {kind}: largest error / bound {worst:.3g} over {n} points")


# ---------------------------------------------------------------------------------------------------------------------------
# 1e. dgp_ehvi2d and dgp_ehvi2d_grad
# ---------------------------------------------------------------------------------------------------------------------------
def padded_front(n):
    """oracle.Y_ND on n - 2 points of y1 = 1 - sqrt(y0), objective 0 descending, nadir (1.1, 1.1), ideal (-0.1, -0.1)."""
    y0 = np.linspace(0.95, 0.05, n - 2)
    return O.Y_ND(y0, 1.0 - np.sqrt(y0), nadir=(1.1, 1.1), ideal=(-0.1, -0.1))


def ehvi_candidates(n):
    """(m0, m1, sigma) rows: dominating the whole front, dominated by it, exactly on a front point (u = 0), within a sigma of that
    point (u = -0.7 and 0.4), far beyond the nadir; sigma in {1e-8, 1, 1e3} for n <= 33, three of them at the largest front (the
    reference costs ~n special functions per term)."""
    a, b = padded_front(n)
    k = (n - 1) // 2
    on = (float(a[k]), float(b[k]))
    if n > 64:
        return [(on[0], on[1], 1.0), (0.0, 0.0, 1e-8), (0.97, 0.9, 1e3)]
    return [row for s in (1e-8, 1.0, 1e3)
            for row in ((0.0, 0.0, s), (0.97, 0.9, s), (on[0], on[1], s), (on[0] + 0.7 * s, on[1] - 0.4 * s, s), (50.0, 60.0, s))]


_EHVI_REF = {}


def ehvi_reference(n):
    if n not in _EHVI_REF:
        a, b = padded_front(n)
        rows = []
        with mp.workdps(DPS):
            y0, y1 = [mp.mpf(float(t)) for t in a], [mp.mpf(float(t)) for t in b]
            for m0, m1, s in ehvi_candidates(n):
                v = s * s
                args = (mp.mpf(m0), mp.mpf(v), mp.mpf(m1), mp.mpf(v))
                rows.append((mp_ehvi(*args, y0, y1), mp_ehvi_partials(*args, y0, y1), mp_ehvi_scales(*args, y0, y1)))
        _EHVI_REF[n] = (a, b, rows)
    return _EHVI_REF[n]


@GPU
@pytest.mark.parametrize("n", [2, 3, 33, 2048])
def test_ehvi2d_value_and_partials_match_mpmath(ctx, n):
    """Value and the four partial derivatives (mp.diff at DPS digits, not a restatement of psi_grad) within ehvi_bound; the values
    of dgp_ehvi2d and dgp_ehvi2d_grad agree within the same bound."""
    a, b, rows = ehvi_reference(n)
    cand = ehvi_candidates(n)
    N = len(cand)
    m0, m1 = _dev([c[0] for c in cand]), _dev([c[1] for c in cand])
    v = _dev([c[2] * c[2] for c in cand])
    y0, y1 = _dev(a), _dev(b)
    out, out2 = torch.empty(N, dtype=torch.float64, device="cuda"), torch.empty(N, dtype=torch.float64, device="cuda")
    g = torch.empty((N, 4), dtype=torch.float64, device="cuda")
    ctx.call("dgp_ehvi2d", _p(m0), _p(v), _p(m1), _p(v), N, _p(y0), _p(y1), n, _p(out))
    ctx.call("dgp_ehvi2d_grad", _p(m0), _p(v), _p(m1), _p(v), N, _p(y0), _p(y1), n, _p(out2), _p(g))
    torch.cuda.synchronize()
    out, out2, g = out.cpu().numpy(), out2.cpu().numpy(), g.cpu().numpy()
    worst = 0.0
    for c, (e, parts, (T, A)) in enumerate(rows):
        bound = ehvi_bound(n, T, A, 0)
        for got, what in ((out[c], "ehvi2d"), (out2[c], "ehvi2d_grad value")):
            err = abs(float(mp.mpf(float(got)) - e))
            worst = max(worst, err / bound)
            assert err <= bound, (n, cand[c], what, float(e), float(got), err, bound)
        assert abs(out[c] - out2[c]) <= bound, (n, cand[c])
        for k in range(4):
            bk = ehvi_bound(n, T, A, k + 1)
            err = abs(float(mp.mpf(float(g[c, k])) - parts[k]))
            worst = max(worst, err / bk)
            assert err <= bk, (n, cand[c], k, float(parts[k]), float(g[c, k]), err, bk)
    print(f"ehvi2d n={n}: largest error / bound {worst:.3g}")


@GPU
@pytest.mark.parametrize("n", [1, 2049])
def test_ehvi2d_refuses_front_sizes_outside_2_to_2048(ctx, n):
    import dgp_toolbox_b200 as D
    m, y = _dev(np.zeros(4)), _dev(np.zeros(max(n, 1)))
    out, g = torch.empty(4, dtype=torch.float64, device="cuda"), torch.empty((4, 4), dtype=torch.float64, device="cuda")
    for name, extra in (("dgp_ehvi2d", ()), ("dgp_ehvi2d_grad", (_p(g),))):
        torch.cuda.synchronize()
        n0 = ctx.launch_count()
        with pytest.raises(D._lib.DGPError):
            ctx.call(name, _p(m), _p(m), _p(m), _p(m), 4, _p(y), _p(y), n, _p(out), *extra)
        assert ctx.launch_count() == n0, (name, "a refused call launched kernels")


@GPU
def test_mo_ehvi_with_grad_hands_over_centred_moments(monkeypatch):
    """EHVI_with_grad on a multi-objective object reduces the chain's per-sample moments in torch before dgp_ehvi2d_grad. With
    propagate replaced by offset moments (means at 1e3 and 300 with small spreads and variances), the moments it hands over match
    the mpmath mixture moments within the 1a bounds."""
    import dgp_toolbox_b200 as D
    S, N = 1000, 6
    rng = np.random.default_rng(5)
    Z = [torch.from_numpy(rng.standard_normal((S, N, 1))).cuda() for _ in range(2)]
    seen = {}

    class Offset:
        device = torch.device("cuda", 0)

        def propagate(self, X, S=1):
            base = X.sum(1).reshape(1, -1, 1)
            Fm = [1e3 + 1e-4 * Z[0] + 1e-3 * base, 300.0 + 1e-2 * Z[1] - 1e-3 * base]
            Fv = [(1e-9 * (1 + X[:, :1] ** 2)).reshape(1, -1, 1).expand(S, -1, -1), torch.full((S, N, 1), 1e-8, device="cuda") + 0 * base]
            seen["F"] = [t.detach().cpu().numpy()[:, :, 0] for t in Fm + Fv]
            return None, Fm, Fv

    by_ptr, handed = {}, []
    real_ptr, real_call = D._lib.ptr, D._lib.Context.call

    def ptr(t):
        if t is not None:
            by_ptr[t.data_ptr()] = t
        return real_ptr(t)

    def call(self, name, *args):
        if name == "dgp_ehvi2d_grad":          # (m0, v0, m1, v1) as the library receives them, before it runs
            handed.append([by_ptr[a.value].detach().cpu().numpy().copy() for a in args[:4]])
        return real_call(self, name, *args)

    monkeypatch.setattr(D._lib, "ptr", ptr)
    monkeypatch.setattr(D._lib.Context, "call", call)
    obj = types.SimpleNamespace(name="mo_dgp", model=Offset())
    a, b = padded_front(5)
    val, dx = D.EHVI_with_grad(obj, rng.uniform(0, 1, (N, 2)), [a, b], S=S)
    torch.cuda.synchronize()
    monkeypatch.undo()
    assert np.isfinite(val.cpu().numpy()).all() and np.isfinite(dx.cpu().numpy()).all()
    assert len(handed) == 1
    handed = handed[0]
    Fm0, Fm1, Fv0, Fv1 = seen["F"]
    for (mean, var), (Fm, Fv) in zip(((handed[0], handed[1]), (handed[2], handed[3])), ((Fm0, Fv0), (Fm1, Fv1))):
        ref = mp_moments(Fm, Fv)
        bad = moment_violations(mean, var, ref, S, range(N))
        assert not bad, bad


# ---------------------------------------------------------------------------------------------------------------------------
# 1f. CPU self-tests: the references, the bounds' margin and the teeth of the moment checks
# ---------------------------------------------------------------------------------------------------------------------------
def _np_criterion(kind, m, v, y, x=None):
    """numpy replay of acq_moments_kernel (Phi through erfc, as the kernel does)."""
    from scipy.special import erfc
    cdf = lambda t: 0.5 * erfc(-t * 0.70710678118654752440)
    pdf = lambda t: 0.39894228040143267794 * np.exp(-0.5 * t * t)
    s = np.sqrt(v)
    if kind == 4:
        return cdf((y - m) / s)
    if kind == 2:
        t = (m - y) / s
        return (m - y) * cdf(t) + v * (pdf(t) / s)
    u = (y - m) / s
    ei = (y - m) * cdf(u) + v * (pdf(u) / s)
    if kind == 0:
        return -ei
    if kind == 1:
        return -(ei - m)
    with np.errstate(over="ignore", divide="ignore"):
        sg = 1.0 / (1.0 + 1.0 / np.exp(x))
    return -(sg * ei[:, None] - m[:, None])


def test_mp_references_match_scipy_and_numpy_at_benign_points():
    from scipy.special import ndtr
    u = np.linspace(-3.0, 3.0, 13)
    with mp.workdps(DPS):
        assert max(abs(float(mp.ncdf(t)) - ndtr(t)) / ndtr(t) for t in u) < 1e-14
    m, v = np.full(13, 0.3), np.full(13, 0.04)
    y = m + 0.2 * u
    x = np.tile([0.3, -1.2], (13, 1))
    for kind in range(5):
        want = _np_criterion(kind, m, v, y, x)
        got = np.array([[float(c) for c in mp_criterion(kind, m[i], v[i], y[i], x[i] if kind == 3 else ())[0]] if kind == 3
                        else float(mp_criterion(kind, m[i], v[i], y[i])[0]) for i in range(13)])
        assert np.max(np.abs(got - want)) <= 1e-14 * np.max(np.abs(want)), kind
    Fm = 0.3 + 0.1 * np.random.default_rng(0).standard_normal((8, 5))
    Fv = np.full((8, 5), 0.05)
    ref = mp_moments(Fm, Fv, 0.1)
    om, ov = O.mixture_moments(torch.as_tensor(Fm), torch.as_tensor(Fv + 0.1))
    assert np.allclose([float(r[0]) for r in ref], om.numpy(), rtol=1e-15, atol=0)
    assert np.allclose([float(r[1]) for r in ref], ov.numpy(), rtol=1e-14, atol=0)


def test_mp_ehvi_reference_matches_the_oracle_at_benign_points():
    """The mpmath strip sum and its mp.diff partials against torch autograd through oracle.ehvi_exact (float64)."""
    a, b = padded_front(7)
    m = [torch.tensor([v], dtype=torch.float64, requires_grad=True) for v in (0.4, 0.09, 0.5, 0.16)]
    e = O.ehvi_exact(*m, torch.as_tensor(a), torch.as_tensor(b))
    e.sum().backward()
    with mp.workdps(DPS):
        y0, y1 = [mp.mpf(float(t)) for t in a], [mp.mpf(float(t)) for t in b]
        args = [mp.mpf(float(t.detach())) for t in m]
        assert abs(float(mp_ehvi(*args, y0, y1)) - float(e.detach())) <= 1e-14 * abs(float(e.detach()))
        parts = mp_ehvi_partials(*args, y0, y1)
        T, A = mp_ehvi_scales(*args, y0, y1)
    assert float(T[0]) >= float(A[0]) >= (1 - 1e-12) * abs(float(e.detach()))
    for k in range(4):
        assert abs(float(parts[k]) - float(m[k].grad)) <= 1e-12 * float(A[k + 1]), k


def _np_ehvi_grad(m0, v0, m1, v1, y0, y1, middle=1.0):
    """Scalar replay of ehvi2d_grad_kernel in float64 (Phi through math.erfc): (value, [dE/dm0, dE/dv0, dE/dm1, dE/dv1]). `middle`
    scales the w (Phi(u_i) - Phi_last) term of the objective-0 factor: 0 drops it, -1 flips its sign (mutants for the bound's teeth)."""
    import math
    cdf = lambda t: 0.5 * math.erfc(-t * 0.70710678118654752440)
    pdf = lambda t: 0.39894228040143267794 * math.exp(-0.5 * t * t)

    def pg(a, b, mu, s):
        u = (b - mu) / s
        p, c = pdf(u), cdf(u)
        q = (a - mu) * p / s
        return s * p + (a - mu) * c, u * p - c - q, p * (1.0 + u * u) - q * u

    n = len(y0)
    s0, s1 = math.sqrt(v0), math.sqrt(v1)
    ul = (y0[n - 1] - m0) / s0
    cl, pl = cdf(ul), pdf(ul)
    e = gm0 = gs0 = gm1 = gs1 = 0.0
    for i in range(1, n):
        pa, pam, pas = pg(y1[i], y1[i], m1, s1)
        pb, pbm, pbs = pg(y1[i], y1[0], m1, s1)
        d1, d1m, d1s = pa - pb, pam - pbm, pas - pbs
        f = fm = fs = 0.0
        if i < n - 1:
            w, u = y0[i - 1] - y0[i], (y0[i] - m0) / s0
            p = pdf(u)
            f += middle * w * (cdf(u) - cl)
            fm += middle * w * (-p + pl) / s0
            fs += middle * w * (-u * p + ul * pl) / s0
        pa, pam, pas = pg(y0[i - 1], y0[i - 1], m0, s0)
        pb, pbm, pbs = pg(y0[i - 1], y0[i], m0, s0)
        f += pa - pb
        fm += pam - pbm
        fs += pas - pbs
        e += f * d1
        gm0 += fm * d1
        gs0 += fs * d1
        gm1 += f * d1m
        gs1 += f * d1s
    return e, [gm0, gs0 / (2.0 * s0), gm1, gs1 / (2.0 * s1)]


def _ehvi_ratios(n, middle=1.0):
    """Per candidate of ehvi_candidates(n): (sigma, [error / bound of the value and of the four partials]) of the numpy replay."""
    a, b, rows = ehvi_reference(n)
    out = []
    for (m0, m1, s), (e, parts, (T, A)) in zip(ehvi_candidates(n), rows):
        val, grads = _np_ehvi_grad(m0, s * s, m1, s * s, [float(t) for t in a], [float(t) for t in b], middle)
        got, want = [val] + grads, [e] + list(parts)
        out.append((s, [abs(float(mp.mpf(g) - w)) / ehvi_bound(n, T, A, k) for k, (g, w) in enumerate(zip(got, want))]))
    return out


@pytest.mark.parametrize("n", [2, 3, 33])
def test_ehvi_bound_holds_with_margin_for_the_numpy_replay(n):
    """The ehvi_bound of test_ehvi2d_value_and_partials_match_mpmath, checked on the CPU: the kernel's arithmetic replayed in
    float64 stays within half of it for the value and the four partials of every candidate."""
    worst = max(max(r) for _, r in _ehvi_ratios(n))
    print(f"numpy replay ehvi2d n={n}: largest error / bound {worst:.3g}")
    assert worst <= 0.5, worst


@pytest.mark.parametrize("middle", [0.0, -1.0], ids=["dropped", "flipped"])
@pytest.mark.parametrize("n", [3, 33])
def test_ehvi_bound_catches_a_wrong_middle_strip_term(n, middle):
    """The bound has teeth at every sigma: a strip sum without the w (Phi(u_i) - Phi_last) term, or with its sign flipped, breaks it
    for the value and for each of the four partials at sigma = 1e-8, 1 and 1e3 (for some candidate at that sigma)."""
    caught = {}
    for s, r in _ehvi_ratios(n, middle):
        caught[s] = [c or x > 1.0 for c, x in zip(caught.get(s, [False] * 5), r)]
    assert set(caught) == {1e-8, 1.0, 1e3}
    assert all(all(v) for v in caught.values()), caught


def test_criterion_bound_holds_with_margin_for_the_numpy_replay():
    """The c = 8 of the criterion bounds, checked on the CPU: the kernel's formula replayed in numpy (scipy's erfc, numpy's exp)
    stays within half the bound over the whole grid of test_acq_moments_criteria_at_their_edges."""
    for kind in range(5):
        m, v, y, x, refs = acq_reference(kind)
        worst, bad = acq_violations(kind, _np_criterion(kind, m, v, y, x), m, v, refs)
        assert not bad and worst <= 0.5, (kind, worst, bad[:3])
        print(f"numpy replay kind {kind}: largest error / bound {worst:.3g}")


@pytest.mark.parametrize("S,offset,spread,v", [(1, 1e3, 0.0, 1e-9), (1000, 1e3, 0.0, 1e-9), (1000, 300.0, 1e-4, 1e-8),
                                               (4096, -50.0, 1e-2, 1e-12)])
def test_one_pass_replay_violates_the_moment_bound(S, offset, spread, v):
    """The parent's one-pass reduction, replayed in numpy, breaks |d var| <= 4 S EPS var on these offset columns (or returns a
    variance of zero or below); the centred two-pass reduction meets the bound on the same inputs."""
    rng = np.random.default_rng(S)
    K = 8
    Fm = offset + spread * rng.standard_normal((S, K))
    Fv = v * rng.uniform(0.5, 1.5, (S, K))
    ref = mp_moments(Fm, Fv)
    mean, var = one_pass(Fm, Fv)
    assert moment_violations(mean, var, ref, S, range(K)), "the one-pass replay met the bound"
    mean, var = centred(Fm, Fv)
    assert not moment_violations(mean, var, ref, S, range(K))
