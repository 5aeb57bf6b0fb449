"""Grouped full_cov=True (dgp_propagate_grouped_cov) and batch expected improvement (dgp_qei, qEI): the N = G q points of a call are
G independent groups of q consecutive points, and group g is what propagate(full_cov=True) gives for its q points alone with
n_offset = g q. Checked group by group against that standalone call, against the float64 oracle, and for q-EI against a torch
reduction of the same call's samples."""
import re
from collections import Counter

import numpy as np
import pytest
import torch
from torch.profiler import ProfilerActivity, profile

from oracle import dgp_oracle as O
from tests.helpers import _condition, product_model_from_problem, rel_err

pytestmark = pytest.mark.gpu

TOL = 1e-9


@pytest.fixture(scope="module")
def ctx():
    import dgp_toolbox_b200 as D
    c = D._lib.get_context(0)
    c.set_fused(True)
    yield c
    c.set_fused(True)
    c.set_workspace_limit(24 << 30)


def launched(fn):
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, Counter(e.name.replace(" ", "") for e in prof.events())


def count(names, kernel):
    """Launches of `kernel` (any template instance) among the profiled names, e.g. "voiddgp::grouped_cov_kernel<4>(...)"."""
    pat = re.compile(r"(?:^|:|void)" + kernel + r"[<(]")
    return sum(v for n, v in names.items() if pat.search(n))


def model(kernels, white, units, N, S, M=40, D0=2, seed_shift=0, D_L=1):
    prob = O.synthetic_problem(D0, units, M, N, seed_shift=seed_shift)
    for l, k, w in zip(prob["layers"], kernels, white):
        l["kernel"], l["white"] = k, w
    if D_L > 1:   # a multi-output last layer
        rng = np.random.default_rng(5)
        last = prob["layers"][-1]
        last["q_mu"] = 0.1 * rng.standard_normal((M, D_L))
        last["q_sqrt"] = 0.5 * np.eye(M)[None] + 0.05 * np.tril(rng.standard_normal((D_L, M, M)))
    prob = _condition(prob)
    return prob, O.model_from_problem(prob, S), product_model_from_problem(prob, S)


def standalone(pm, X, g, q, S, seed=None, zs=None):
    Xg = X[g * q:(g + 1) * q]
    zg = None if zs is None else [z[:, g * q:(g + 1) * q] for z in zs]
    return pm.propagate(Xg, full_cov=True, S=S, seed=seed, zs=zg, n_offset=g * q)


def group_blocks(Fv, g):
    return Fv[:, g]   # [S, q, q, D]


def rows(F, g, q):
    return F[:, g * q:(g + 1) * q]


# (kernels, white, hidden units, fused, q, G, S): RBF / Matérn32 / Matérn52, plain, white and mixed stacks, the fused pipeline and
# dgp_set_fused(0) (plain stacks: white layers need the fused kernel), hidden layers with D_out > 1, and every q size class.
EQUIV_CASES = {
    "rbf-plain-q1": (["rbf", "rbf"], [False, False], [3], True, 1, 3, 7),
    "m32-mixed-q2": (["matern32", "rbf"], [True, False], [2], True, 2, 3, 64),
    "m52-white-q5": (["matern52", "matern52"], [True, True], [3], True, 5, 3, 1),
    "rbf-unfused-q8": (["rbf", "matern32"], [False, False], [3], False, 8, 3, 7),
    "m52-unfused-q17": (["matern52", "rbf", "rbf"], [False, False, False], [2, 3], False, 17, 3, 7),
    "m32-white-q32": (["matern32", "matern52"], [True, False], [3], True, 32, 1, 7),
    "rbf-mixed-G150": (["rbf", "matern52"], [False, True], [2], True, 8, 150, 1),
    "m52-plain-q32-S64": (["matern52", "rbf"], [False, False], [2], True, 32, 3, 64),
}


@pytest.mark.parametrize("case", list(EQUIV_CASES))
def test_each_group_is_the_standalone_full_cov_call(ctx, case):
    kernels, white, units, fused, q, G, S = EQUIV_CASES[case]
    N = G * q
    prob, om, pm = model(kernels, white, units, N, S)
    X = torch.as_tensor(prob["X"]).cuda()
    ctx.set_fused(fused)
    try:
        Fs, Fm, Fv = pm.propagate(X, full_cov=True, S=S, seed=123, group_size=q)
        for l, ol in enumerate(om.layers):
            assert tuple(Fv[l].shape) == (S, G, q, q, ol.D_out) and tuple(Fs[l].shape) == (S, N, ol.D_out)
        bitwise_means = True
        for g in range(G):
            Ss, Sm, Sv = standalone(pm, X, g, q, S, seed=123)
            for l, ol in enumerate(om.layers):
                assert rel_err(rows(Fm[l], g, q), Sm[l]) < TOL
                bitwise_means &= torch.equal(rows(Fm[l], g, q), Sm[l])
                assert rel_err(group_blocks(Fv[l], g), Sv[l], scale=float(ol.variance)) < TOL
                assert rel_err(rows(Fs[l], g, q), Ss[l]) < 1e-8
        # supplied draws: group g uses columns g q .. of zs
        zs = [torch.randn(S, N, ol.D_out, dtype=torch.float64, generator=torch.Generator().manual_seed(3 + l)).cuda()
              for l, ol in enumerate(om.layers)]
        Fs, Fm, Fv = pm.propagate(X, full_cov=True, S=S, zs=zs, group_size=q)
        for g in range(G):
            Ss, Sm, Sv = standalone(pm, X, g, q, S, zs=zs)
            for l, ol in enumerate(om.layers):
                assert rel_err(group_blocks(Fv[l], g), Sv[l], scale=float(ol.variance)) < TOL
                assert rel_err(rows(Fs[l], g, q), Ss[l]) < 1e-8
    finally:
        ctx.set_fused(True)
    print(f"[{case}] means bitwise equal to the standalone calls: {bitwise_means}")


@pytest.mark.parametrize("stack", [(["rbf", "matern32"], [False, False], [3], 4, 5, 6),
                                   (["matern52", "rbf", "rbf"], [True, False, False], [2, 2], 7, 3, 4)], ids=["plain", "white-3layer"])
def test_grouped_call_matches_the_float64_oracle(ctx, stack):
    kernels, white, units, q, G, S = stack
    N = G * q
    prob, om, pm = model(kernels, white, units, N, S)
    zs = [torch.randn(S, N, ol.D_out, dtype=torch.float64, generator=torch.Generator().manual_seed(9 + l)) for l, ol in enumerate(om.layers)]
    Fs, Fm, Fv = pm.propagate(prob["X"], full_cov=True, S=S, zs=zs, group_size=q)
    X = torch.as_tensor(prob["X"])
    for g in range(G):
        with torch.no_grad():
            Fs_o, Fm_o, Fv_o = O.propagate_full_cov(om.layers, X[g * q:(g + 1) * q], S, [z[:, g * q:(g + 1) * q] for z in zs])
        for l, ol in enumerate(om.layers):
            assert rel_err(rows(Fm[l], g, q), Fm_o[l]) < TOL
            assert rel_err(group_blocks(Fv[l], g), Fv_o[l], scale=float(ol.variance)) < TOL
            assert rel_err(rows(Fs[l], g, q), Fs_o[l]) < 1e-8


def test_blocks_are_symmetric_and_their_diagonal_is_the_marginal_variance(ctx):
    q, G, S = 6, 9, 5
    prob, om, pm = model(["matern32", "rbf"], [False, False], [3], G * q, S)
    zs = [torch.randn(S, G * q, ol.D_out, dtype=torch.float64, generator=torch.Generator().manual_seed(l)) for l, ol in enumerate(om.layers)]
    Fs, Fm, Fv = pm.propagate(prob["X"], full_cov=True, S=S, zs=zs, group_size=q)
    for l in range(len(om.layers)):
        assert torch.equal(Fv[l], Fv[l].transpose(2, 3)), "blocks must be symmetric bit for bit"
    _, _, Vd = pm.propagate(prob["X"], S=S, zs=zs)   # the first layer's input is X in both calls
    diag = torch.diagonal(Fv[0], dim1=2, dim2=3).permute(0, 1, 3, 2).reshape(S, G * q, -1)
    assert rel_err(diag, Vd[0], scale=float(om.layers[0].variance)) < TOL


def test_chunked_call_is_bitwise_equal_to_one_chunk_and_launches(ctx):
    """A workspace limit that splits the 31 groups (a prime count: every split is uneven) into at least three chunks gives the same
    bits as one chunk; one grouped_cov_kernel per layer and chunk, and none of the dense full-covariance kernels."""
    q, G, S = 4, 31, 1000   # ~270 MB of chunk buffers against limits from 64 MiB (the smallest dgp_set_workspace_limit takes)
    prob, om, pm = model(["rbf", "matern52"], [False, False], [3], G * q, S, M=64)
    X = torch.as_tensor(prob["X"]).cuda()
    L = len(om.layers)
    run = lambda: pm.propagate(X, full_cov=True, S=S, seed=7, group_size=q)
    ref, names = launched(run)
    assert count(names, "grouped_cov_kernel") == L
    assert count(names, "fullcov_kernel") == 0 and count(names, "fullcov_sample_kernel") == 0
    assert count(names, "chol_inv_kernel") == 1   # the prep's Kuu factorisation of all layers, not a covariance block
    chunks = 0
    try:
        for mib in (64, 80, 96, 128, 160):
            ctx.set_workspace_limit(mib << 20)
            out, names = launched(run)
            chunks = count(names, "grouped_cov_kernel") // L
            if 3 <= chunks < G:
                break
        assert 3 <= chunks < G, chunks
        assert count(names, "grouped_cov_kernel") == L * chunks and count(names, "fullcov_kernel") == 0
        for a, b in zip(out, ref):
            for x, y in zip(a, b):
                assert torch.equal(x, y)
    finally:
        ctx.set_workspace_limit(24 << 30)


def test_above_the_dense_limit(ctx):
    """G = 300, q = 4: N = 1 200 points, above the N <= 768 of the dense full_cov call."""
    q, G, S = 4, 300, 8
    prob, om, pm = model(["rbf", "rbf"], [False, False], [2], G * q, S)
    X = torch.as_tensor(prob["X"]).cuda()
    Fs, Fm, Fv = pm.propagate(X, full_cov=True, S=S, seed=5, group_size=q)
    for g in (0, 151, 299):
        Ss, Sm, Sv = standalone(pm, X, g, q, S, seed=5)
        for l, ol in enumerate(om.layers):
            assert rel_err(group_blocks(Fv[l], g), Sv[l], scale=float(ol.variance)) < TOL
            assert rel_err(rows(Fs[l], g, q), Ss[l]) < 1e-8


def torch_neg_qei(F, q, y_min):
    S, N, D = F.shape
    m = F.reshape(S, N // q, q, D).amin(dim=2)
    return -torch.clamp(y_min - m, min=0.0).mean(dim=0)


@pytest.mark.parametrize("D_L", [1, 2])
def test_qei_values(ctx, D_L):
    import dgp_toolbox_b200 as D
    q, G, S = 3, 20, 64
    prob, om, pm = model(["matern32", "rbf"], [False, False], [2], G * q, S, D_L=D_L)
    y_min = float(np.min(prob["Y"]))
    crit = D.qEI(y_min, 2, q)
    X = torch.as_tensor(prob["X"]).cuda()
    val = crit.run(pm, X, num_samples=S, seed=31)
    assert tuple(val.shape) == (G, D_L)
    Fs, _, _ = pm.propagate(X, full_cov=True, S=S, seed=31, group_size=q)
    assert rel_err(val, torch_neg_qei(Fs[-1], q, y_min)) < 1e-12
    assert torch.equal(crit.run(pm, X.reshape(G, q, 2), num_samples=S, seed=31), val)   # [G, q, d] input
    # float64 reference chain on the same Philox draws (group g: n_offset = g q), plus the reduction
    Xc = torch.as_tensor(prob["X"])
    ref = []
    for g in range(G):
        zs = [torch.as_tensor(O.philox_normal(31, l, S, q, ol.D_out, g * q)) for l, ol in enumerate(om.layers)]
        with torch.no_grad():
            Fs_o, _, _ = O.propagate_full_cov(om.layers, Xc[g * q:(g + 1) * q], S, zs)
        ref.append(torch_neg_qei(Fs_o[-1], q, y_min)[0])
    assert rel_err(val, torch.stack(ref)) < 1e-8


def test_refusals_launch_nothing_and_the_next_call_is_right(ctx):
    import dgp_toolbox_b200 as D
    prob, om, pm = model(["rbf", "rbf"], [False, False], [2], 12, 3)
    X = torch.as_tensor(prob["X"]).cuda()
    crit = D.qEI(0.0, 2, 5)
    torch.cuda.synchronize()
    n0 = ctx.launch_count()
    for q, what in ((0, "1 .. 32"), (33, "1 .. 32"), (5, "multiple of the group size")):
        with pytest.raises(D._lib.DGPError, match=what):
            pm.propagate(X, full_cov=True, S=3, seed=1, group_size=q)
    with pytest.raises(D._lib.DGPError, match="multiple of the group size"):
        crit.run(pm, X, num_samples=3, seed=1)
    assert ctx.launch_count() == n0, "a refused call launched kernels"
    with pytest.raises(ValueError, match="full_cov"):
        pm.propagate(X, S=3, group_size=4)
    with pytest.raises(ValueError, match="full_cov"):
        pm.predict_f(X, S=3, group_size=4)
    Fs, Fm, Fv = pm.propagate(X, full_cov=True, S=3, seed=1, group_size=4)
    Ss, Sm, Sv = standalone(pm, X, 2, 4, 3, seed=1)
    assert rel_err(group_blocks(Fv[-1], 2), Sv[-1], scale=1.0) < TOL and rel_err(rows(Fs[-1], 2, 4), Ss[-1]) < 1e-8
    m, v = pm.predict_f(X, full_cov=True, S=3, seed=1, group_size=4)
    assert tuple(v.shape) == (3, 3, 4, 4, 1) and torch.equal(v, Fv[-1]) and torch.equal(m, Fm[-1])
    with pytest.raises(NotImplementedError):
        D.qEI(0.0, 2, 4).optimize(pm, (np.zeros(2), np.ones(2)), method='DE+Adam')
    with pytest.raises(NotImplementedError):
        D.qEI(0.0, 2, 4).optimize(pm, (np.zeros(2), np.ones(2)), method='Adam')


def test_a_non_positive_pivot_in_a_group_block_is_reported(ctx, monkeypatch):
    """Well-separated Z, q_sqrt ~ 0, inputs at the inducing points and jitter = -sigma^2 / 2: Kuu + jitter I ~ sigma^2 / 2 I stays
    positive definite while each q x q block is ~ sigma^2 I - 2 sigma^2 I - sigma^2 / 2 I."""
    import dgp_toolbox_b200 as D
    from dgp_toolbox_b200 import gpflow_shim
    M = 8
    Z = np.stack([np.arange(M) * 10.0, np.zeros(M)], 1)
    layer = D.SVGP_Layer(D.SquaredExponential(variance=1.0, lengthscales=[1.0, 1.0]), Z, 1, D.Zero())
    layer.q_mu.assign(np.zeros((M, 1)))
    layer.q_sqrt.assign(1e-6 * np.eye(M)[None])
    pm = D.DGP_Base(D.Gaussian(0.1), [layer], num_samples=2)
    crit = D.qEI(0.0, 2, 4)
    out = torch.empty((2, 1), dtype=torch.float64, device="cuda")
    monkeypatch.setattr(gpflow_shim, "DEFAULT_JITTER", -0.5)
    crit.run(pm, Z, num_samples=2, seed=1, out=out)
    with pytest.raises(D._lib.DGPError, match="not positive definite"):
        ctx.check()
    monkeypatch.setattr(gpflow_shim, "DEFAULT_JITTER", 1e-6)
    crit.run(pm, Z + 0.3, num_samples=2, seed=1, out=out)
    ctx.check()


def test_qei_optimize_on_a_1d_dgp(ctx):
    """qEI(q = 2).optimize returns a pair inside the box whose -q-EI (fresh draws, S = 256) is within Monte-Carlo noise of the
    best pair of a 64 x 64 grid scored in one call; the same seed and draw state give the same pair."""
    import dgp_toolbox_b200 as D
    rng = np.random.default_rng(3)
    X = np.linspace(-1.0, 1.0, 14)[:, None]
    Y = np.sin(4.0 * X) + 0.3 * X + 0.02 * rng.standard_normal(X.shape)
    mdl = D.DGP(X, Y, X.copy(), [D.RBF(lengthscales=[0.4], variance=1.0) for _ in range(2)], [1], D.Gaussian(0.01),
                num_samples=8, seed=5)
    D.DGP_Base.optimize_adam(mdl, mdl.data, iterations=300, lr=0.02, messages=10 ** 9)
    crit = D.qEI(float(Y.min()), 1, 2)
    box = (np.array([-1.0]), np.array([1.0]))
    draw0 = mdl._draw
    x_opt = crit.optimize(mdl, box, popsize_DE=32, iterations_DE=40, num_samples=64, seed=11)
    assert x_opt.shape == (2, 1) and np.all((-1.0 <= x_opt) & (x_opt <= 1.0))
    assert tuple(crit.IC_optimized.shape) == (1, 1)
    g1 = np.linspace(-1.0, 1.0, 64)
    pairs = np.stack(np.meshgrid(g1, g1, indexing="ij"), -1).reshape(-1, 2, 1)
    g = crit.run(mdl, pairs, num_samples=256, seed=77).cpu().numpy().reshape(-1)
    best = pairs[np.argmin(g)]
    # both pairs re-scored on the same fresh draws (one batch each, seed 78): the grid minimum itself is biased low by its selection
    at_opt = float(crit.run(mdl, x_opt, num_samples=256, seed=78))
    at_best = float(crit.run(mdl, best, num_samples=256, seed=78))
    assert at_opt <= at_best + 0.10 * abs(at_best) + 1e-6, (at_opt, at_best, g.min(), x_opt.ravel(), best.ravel())
    mdl._draw = draw0
    x_again = crit.optimize(mdl, box, popsize_DE=32, iterations_DE=40, num_samples=64, seed=11)
    assert np.array_equal(x_again, x_opt)
