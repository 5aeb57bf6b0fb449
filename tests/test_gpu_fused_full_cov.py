"""full_cov=True of the RBF / Matérn SVGP layers on the library's own kernel path: the covariance tiles build K(X_s, X_s) from the
inputs (fullcov_kernel, upper-triangular tiles mirrored), on the V-form planes of the fused conditional kernel or, for layers the
fused kernel does not take, on the A-form planes of the unfused pipeline. Per-sample inputs X [S, N, D_in] are one library call
(dgp_propagate_full_cov_snd).

Checked against a float64 reference written from the formula cov_d = Kff - A^T (P - q_sqrt_d q_sqrt_d^T) A (A = Ku^-1 Kuf, P = Ku;
whitened: A = Lu^-1 Kuf, P = I) and against the supplied-matrix path (dgp_svgp_from_k_full_cov) on matrices built in torch."""
from collections import Counter

import numpy as np
import pytest
import torch
from torch.profiler import ProfilerActivity, profile

from oracle import dgp_oracle as O
from tests.helpers import _condition, both_models, oracle_zs, product_model_from_problem, rel_err

pytestmark = pytest.mark.gpu

TOL = 1e-9


@pytest.fixture(scope="module")
def ctx():
    import dgp_toolbox_b200 as D
    c = D._lib.get_context(0)
    c.set_fused(True)
    yield c
    c.set_fused(True)


def layer_case(kernel, white, M, N, D_in=3, D_out=2):
    """(oracle layer, product layer, X [N, D_in]) of one D_in -> D_out layer with cond(Ku) <= 2e3, a non-trivial q(u) and a
    Linear mean function."""
    prob = O.synthetic_problem(D_in, [], M, N)
    rng = np.random.default_rng(7)
    prob["layers"][0].update(kernel=kernel, white=white, q_mu=0.1 * rng.standard_normal((M, D_out)),
                             q_sqrt=0.5 * np.eye(M)[None] + 0.05 * np.tril(rng.standard_normal((D_out, M, M))),
                             mean_kind="linear", mf_W=0.3 * rng.standard_normal((D_in, D_out)), mf_b=0.1 * rng.standard_normal(D_out))
    prob = _condition(prob)
    ol = O.model_from_problem(prob, 1).layers[0]
    pl = product_model_from_problem(prob, 1).layers[0]
    return ol, pl, torch.as_tensor(prob["X"])


def per_sample_inputs(X, S):
    return torch.stack([X * (1.0 - 0.07 * s) + 0.05 * s for s in range(S)])


def reference(ol, Xs):
    """float64 CPU: mean [S, N, D_out] (with the mean function), cov [S, N, N, D_out] from the formula."""
    Ku = O.kernel_K(ol.Z, None, ol.lengthscales, ol.variance, ol.kernel_kind) + O.JITTER * torch.eye(ol.M, dtype=torch.float64)
    means, covs = [], []
    for X in Xs:
        Kuf = O.kernel_K(ol.Z, X, ol.lengthscales, ol.variance, ol.kernel_kind)
        Kff = O.kernel_K(X, None, ol.lengthscales, ol.variance, ol.kernel_kind)
        if ol.white:
            A, P = torch.linalg.solve_triangular(torch.linalg.cholesky(Ku), Kuf, upper=False), torch.eye(ol.M, dtype=torch.float64)
        else:
            A, P = torch.linalg.solve(Ku, Kuf), Ku
        means.append(A.T @ ol.q_mu + O.mean_function(ol, X))
        covs.append(torch.stack([Kff - A.T @ (P - L @ L.T) @ A for L in ol.q_sqrt], -1))
    return torch.stack(means), torch.stack(covs)


def launched(fn):
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, Counter(e.name.replace(" ", "") for e in prof.events())


def ran(names, kernel):
    return any(kernel + "(" in n or n.endswith(kernel) for n in names)


def check_against_reference(pl, ol, Xs):
    (mean, cov), names = launched(lambda: pl.conditional_SND(Xs.numpy(), full_cov=True))
    S, N = Xs.shape[0], Xs.shape[1]
    assert tuple(mean.shape) == (S, N, ol.D_out) and tuple(cov.shape) == (S, N, N, ol.D_out)
    assert mean.dtype == cov.dtype == torch.float64
    m_r, c_r = reference(ol, Xs)
    assert rel_err(mean, m_r) < TOL
    assert rel_err(cov, c_r, scale=float(ol.variance)) < TOL
    assert torch.equal(cov, cov.transpose(1, 2)), "the mirrored tiles must equal the computed ones bit for bit"
    md, vd = pl.conditional_SND(Xs.numpy())
    assert rel_err(torch.diagonal(cov, dim1=1, dim2=2).permute(0, 2, 1), vd, scale=float(ol.variance)) < TOL
    assert rel_err(mean, md) < TOL
    return names


# The four forward configurations of the fused conditional kernel: 128-row blocks (Mp % 128 == 0) or 64-row blocks, each with
# 64-point tiles or the halved 32-point tiles of calls with at most 74 tiles (S * N <= 4 736). N and M off the tile multiples.
FUSED_CASES = {
    "cfg0": (128, 600, 8, "fused_forward_kernel<128,64,4,2>"),
    "cfg1": (128, 77, 3, "fused_forward_kernel<128,32,4,2>"),
    "cfg2": (50, 600, 8, "fused_forward_kernel<64,64,2,4>"),
    "cfg3": (64, 45, 2, "fused_forward_kernel<64,32,2,4>"),
}


@pytest.mark.parametrize("white", [False, True], ids=["plain", "white"])
@pytest.mark.parametrize("kernel", ["rbf", "matern32", "matern52"])
@pytest.mark.parametrize("case", list(FUSED_CASES))
def test_fused_full_cov_matches_the_formula(ctx, case, kernel, white):
    M, N, S, fused = FUSED_CASES[case]
    ol, pl, X = layer_case(kernel, white, M, N)
    names = check_against_reference(pl, ol, per_sample_inputs(X, S))
    assert ran(names, fused) and ran(names, "fullcov_kernel") and not ran(names, "kuf_kernel"), sorted(names)


@pytest.mark.parametrize("kernel", ["rbf", "matern32", "matern52"])
@pytest.mark.parametrize("dims", [(50, 45, 3), (64, 1, 4), (130, 200, 2)], ids=["m50-n45", "n1", "m130-n200"])
def test_unfused_full_cov_matches_the_formula(ctx, kernel, dims):
    M, N, S = dims
    ol, pl, X = layer_case(kernel, False, M, N)
    ctx.set_fused(False)
    try:
        names = check_against_reference(pl, ol, per_sample_inputs(X, S))
    finally:
        ctx.set_fused(True)
    assert ran(names, "kuf_kernel") and ran(names, "fullcov_kernel") and not any("fused_forward_kernel" in n for n in names)


def test_full_cov_on_a_shape_without_a_fused_configuration(ctx):
    """M = 640 with 16 -> 32 has no fused configuration; full_cov=True used to be refused there and now runs the unfused pipeline."""
    ol, pl, X = layer_case("matern52", False, 640, 40, D_in=16, D_out=32)
    names = check_against_reference(pl, ol, per_sample_inputs(X, 2))
    assert ran(names, "kuf_kernel") and not any("fused_forward_kernel" in n for n in names)


@pytest.mark.parametrize("kernel", ["rbf", "matern32"])
def test_fused_agrees_with_the_supplied_matrix_path(ctx, kernel):
    """The same layer through dgp_svgp_from_k_full_cov on Kuu + jitter I, Kuf and Kff built in torch (float64, on the GPU)."""
    from dgp_toolbox_b200 import composite
    S, N = 3, 70
    ol, pl, X = layer_case(kernel, False, 96, N)
    Xs = per_sample_inputs(X, S)
    z = torch.randn(S, N, ol.D_out, dtype=torch.float64, generator=torch.Generator().manual_seed(7))
    F, mean, cov = pl.sample_from_conditional(Xs.numpy(), z=z, full_cov=True)
    dev = mean.device
    Z, ls, var = ol.Z.to(dev), ol.lengthscales.to(dev), ol.variance.to(dev)
    Xd = Xs.to(dev)
    Ku = O.kernel_K(Z, None, ls, var, kernel) + O.JITTER * torch.eye(ol.M, dtype=torch.float64, device=dev)
    Kuf = O.kernel_K(Z, Xd.reshape(S * N, -1), ls, var, kernel)
    Kff = torch.stack([O.kernel_K(x, None, ls, var, kernel) for x in Xd])
    F_k, mean_k, cov_k = composite.svgp_from_k_full_cov(Ku, Kuf, Kff, ol.q_mu.to(dev), ol.q_sqrt.to(dev), z.to(dev), O.JITTER)
    mf = O.mean_function(ol, Xs.reshape(S * N, -1)).reshape(S, N, -1).to(dev)
    assert rel_err(mean - mf, mean_k) < TOL
    assert rel_err(cov, cov_k, scale=float(ol.variance)) < TOL
    assert rel_err(F - mf, F_k) < 1e-8


def test_per_sample_call_matches_one_call_per_sample(ctx):
    """conditional_SND / sample_from_conditional(full_cov=True) are one call for all S samples; each sample agrees with the
    shared-input call on that sample's rows, and without z sample s still draws the stream of seed + s."""
    S, N = 4, 33
    ol, pl, X = layer_case("matern32", True, 64, N)
    Xs = per_sample_inputs(X, S)
    mean, cov = pl.conditional_SND(Xs.numpy(), full_cov=True)
    F, fm, fv = pl.sample_from_conditional(Xs.numpy(), full_cov=True, seed=11)
    for s in range(S):
        Fs, ms, vs = pl._propagate_full(Xs[s].to(mean.device).contiguous(), 1, None, 11 + s)
        assert rel_err(mean[s], ms[0]) < 1e-12 and rel_err(cov[s], vs[0], scale=1.0) < 1e-12
        assert rel_err(F[s], Fs[0]) < 1e-10
    assert torch.equal(fm, mean) and torch.equal(fv, cov)


@pytest.mark.parametrize("white", [[False, False], [True, False]], ids=["plain", "white-first"])
def test_model_propagate_full_cov_on_both_pipelines(ctx, white):
    """DGP_Base.propagate(full_cov=True) layer to layer against the oracle, fused and (non-white stacks) unfused."""
    S, N = 3, 37
    prob, om, pm = both_models(3, [2], 50, N, S, kernels=["matern52", "rbf"], white=white)
    zs = oracle_zs(om, N, S, 5)
    with torch.no_grad():
        Fs_o, Fm_o, Fv_o = O.propagate_full_cov(om.layers, torch.as_tensor(prob["X"]), S, zs)
    for fused in ([True] if white[0] else [True, False]):
        ctx.set_fused(fused)
        try:
            Fs, Fm, Fv = pm.propagate(prob["X"], full_cov=True, S=S, zs=zs)
        finally:
            ctx.set_fused(True)
        for l, ol in enumerate(om.layers):
            assert rel_err(Fm[l], Fm_o[l]) < TOL and rel_err(Fv[l], Fv_o[l], scale=float(ol.variance)) < TOL
            assert rel_err(Fs[l], Fs_o[l]) < 1e-8


def test_refusals_launch_nothing(ctx):
    import dgp_toolbox_b200 as D
    ol, pl, X = layer_case("rbf", False, 64, 769)
    Xs = per_sample_inputs(X, 2)
    _, wl, Xw = layer_case("rbf", True, 64, 20)
    torch.cuda.synchronize()
    n0 = ctx.launch_count()
    with pytest.raises(D._lib.DGPError, match="N > 768"):
        pl.conditional_SND(Xs.numpy(), full_cov=True)
    ctx.set_fused(False)
    try:
        with pytest.raises(D._lib.DGPError, match="white=True layers run on the fused conditional kernel only"):
            wl.conditional_SND(per_sample_inputs(Xw, 2).numpy(), full_cov=True)
    finally:
        ctx.set_fused(True)
    assert ctx.launch_count() == n0, "a refused call launched kernels"
    ol, pl, X = layer_case("rbf", False, 64, 20)
    check_against_reference(pl, ol, per_sample_inputs(X, 2))

