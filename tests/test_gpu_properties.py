"""GPU tests that do not need the oracle at full size: size-independent properties of the path at BASELINE config-2
dimensions (M=256, D=8, S=32, 16384 points), edge cases and error behaviour of the drop-in classes."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _c2_model(S=32, seed=1234):
    from dgp_toolbox_b200 import synthetic
    cfg = synthetic.CONFIGS["c2"]
    prob = synthetic.synthetic_problem(cfg["D0"], cfg["num_units"], cfg["M"], 8)
    return synthetic.model_from_problem(prob, S, seed=seed), cfg


def test_full_size_prior_gives_kdiag_zero_kl_and_closed_form_elbo():
    """q(u) = p(u) (q_mu = 0, q_sqrt = chol(Kuu + jitter I)) => var = K_diag, mean = mean function, KL = 0 in every layer;
    the last layer (Zero mean) then gives ELBO = sum_n -0.5 log 2pi - 0.5 log s_n^2 - 0.5 (Y_n^2 + s2) / s_n^2 for ANY draws
    (the identity behind the reference notebooks' first printed ELBO, SURVEY §8c KAT-1) -- at config-2 size."""
    from dgp_toolbox_b200 import synthetic
    model, cfg = _c2_model()
    for layer in model.layers:
        layer.q_mu.assign(np.zeros(layer.q_mu.shape))
        layer.build_cholesky_if_needed()
        layer.q_sqrt.assign(layer.Lu[None].repeat(layer.num_outputs, 1, 1))
    N = 16384
    X, Y = synthetic.minibatch(cfg["D0"], N, 0)
    for layer in model.layers:
        assert abs(float(layer.KL())) < 1e-7
    Fs, Fm, Fv = model.propagate(X, S=4, seed=3)
    for l, layer in enumerate(model.layers):
        assert float((Fv[l] - 1.0).abs().max()) < 1e-8                      # K_diag = variance = 1
    assert float(Fm[-1].abs().max()) < 1e-8                                 # Zero mean function
    assert float((Fm[0] - torch.as_tensor(X, device="cuda")[None]).abs().max()) < 1e-8   # Identity mean function
    sn2 = 0.1
    expected = float(np.sum(-0.5 * math.log(2 * math.pi) - 0.5 * math.log(sn2) - 0.5 * (Y ** 2 + 1.0) / sn2))
    got = float(model.ELBO((X, Y), seed=11))
    assert abs(got - expected) <= 1e-9 * abs(expected), (got, expected)


def test_full_size_sharded_sum_equals_full_batch_and_is_deterministic():
    """Two 'ranks' run one after the other on one GPU: shards of the points with kl_weight = 1/2 and global-index Philox
    counters (n_offset) must add up to the full-batch buffer; the same call twice is bitwise identical."""
    from dgp_toolbox_b200 import synthetic
    from dgp_toolbox_b200.distributed import shard_bounds
    model, cfg = _c2_model()
    N = 4096
    X, Y = synthetic.minibatch(cfg["D0"], N, 1)
    full = model.elbo_flat((X, Y), want_grad=True, seed=77).clone()
    again = model.elbo_flat((X, Y), want_grad=True, seed=77).clone()
    assert torch.equal(full, again)
    acc = torch.zeros_like(full)
    for r in range(2):
        lo, hi = shard_bounds(N, r, 2)
        acc += model.elbo_flat((X[lo:hi], Y[lo:hi]), want_grad=True, seed=77, kl_weight=0.5, n_offset=lo)
    scale = float(full.abs().max())
    assert float((acc - full).abs().max()) <= 1e-11 * scale


def test_full_size_fused_and_unfused_conditionals_agree():
    import dgp_toolbox_b200 as D
    from dgp_toolbox_b200 import synthetic
    model, cfg = _c2_model()
    X, Y = synthetic.minibatch(cfg["D0"], 2048, 2)
    ctx = D._lib.get_context(0)
    a = model.elbo_flat((X, Y), want_grad=True, seed=5).clone()
    ctx.set_fused(False)
    try:
        b = model.elbo_flat((X, Y), want_grad=True, seed=5).clone()
    finally:
        ctx.set_fused(True)
    assert float((a - b).abs().max()) <= 1e-10 * float(a.abs().max())


def test_predict_moments_equal_reduction_of_predict_y():
    model, cfg = _c2_model(S=8)
    from dgp_toolbox_b200 import synthetic
    X, _ = synthetic.minibatch(cfg["D0"], 1000, 3)
    ym, yv = model.predict_y(X, 8, seed=9)
    m, v = model.predict(X, 8, seed=9)
    m2 = ym.mean(0)
    v2 = (yv + ym ** 2).mean(0) - m2 ** 2
    assert float((m - m2).abs().max()) < 1e-12 and float((v - v2).abs().max()) < 1e-12


@pytest.mark.parametrize("N,S,M,D0,units", [(1, 1, 1, 1, [1]), (1, 3, 64, 2, [2]), (3, 1, 65, 3, [2]), (130, 2, 7, 2, [3, 1])])
def test_edge_shapes_match_oracle(N, S, M, D0, units):
    from oracle import dgp_oracle as O
    from tests.helpers import both_models, oracle_zs, rel_err
    prob, om, pm = both_models(D0, units, M, N, S)
    zs = oracle_zs(om, N, S, 2)
    X, Y = torch.as_tensor(prob["X"]), torch.as_tensor(prob["Y"])
    val_o, g_o = O.elbo_and_grads(om, X, Y, zs)
    val, g = pm.ELBO_and_grads((prob["X"], prob["Y"]), zs=zs)
    assert abs(float(val) - float(val_o)) <= 1e-9 * max(abs(float(val_o)), 1.0)
    for k, go in g_o.items():
        assert rel_err(g[k].reshape(go.shape), go, scale=1e-6) < 1e-8, k


def test_empty_inputs_and_error_behaviour():
    import dgp_toolbox_b200 as D
    model, cfg = _c2_model(S=2)
    Fs, Fm, Fv = model.propagate(np.zeros((0, 8)), S=2)
    assert Fs[-1].shape == (2, 0, 1) and Fm[0].shape == (2, 0, 8)
    m, v = model.predict(np.zeros((0, 8)), 2)
    assert m.shape == (0, 1)
    assert model.layers[0].conditional_ND(np.zeros((0, 8)))[0].shape == (0, 8)
    assert model.propagate(np.zeros((4, 8)), full_cov=True, S=2)[2][0].shape == (2, 4, 4, 8)
    with pytest.raises(D._lib.DGPError, match="N > 768"):
        model.propagate(np.zeros((800, 8)), full_cov=True, S=1)
    with pytest.raises(NotImplementedError):
        D.SVGP_Layer(D.RBF(lengthscales=[1.0]), np.zeros((4, 1)), 1, D.Zero(), augmented=True)
    with pytest.raises(ValueError):           # Y width does not match the last layer
        model.elbo_flat((np.zeros((4, 8)), np.zeros((4, 3))))
    with pytest.raises(ValueError):           # X width does not match the first layer
        model.propagate(np.zeros((4, 5)))
    bad = D.SVGP_Layer(D.RBF(lengthscales=[1.0], variance=1.0), np.linspace(0, 1, 5)[:, None], 1, D.Zero())
    bad.kern.variance.assign(-1.0)            # Kuu + jitter I is no longer positive definite
    with pytest.raises(D._lib.DGPError):
        bad.build_cholesky_if_needed()
    # the asynchronous ELBO path reports the same failure through dgp_check on the value path
    bad_model = D.DGP_Base(D.Gaussian(0.1), [bad], num_samples=2)
    with pytest.raises(D._lib.DGPError):
        bad_model.ELBO((np.linspace(0, 1, 7)[:, None], np.zeros((7, 1))))
    model.ELBO((np.zeros((4, 8)), np.zeros((4, 1))))   # the flag does not stick to later calls


def test_optimize_adam_increases_elbo():
    import dgp_toolbox_b200 as D
    rng = np.random.default_rng(0)
    X = rng.uniform(-1, 1, (200, 2))
    Y = np.sin(3 * X[:, :1]) * np.cos(2 * X[:, 1:]) + 0.05 * rng.standard_normal((200, 1))
    Z = X[:20].copy()
    kernels = [D.RBF(lengthscales=[0.7, 0.7], variance=1.0) for _ in range(2)]
    model = D.DGP(X, Y, Z, kernels, [2], D.Gaussian(0.1), num_samples=4, seed=1)
    before = float(model.ELBO((X, Y), seed=123))
    D.DGP_Base.optimize_adam(model, model.data, iterations=150, lr=0.01, messages=10 ** 9)   # no q_sqrt rescaling (dgp.py:268)
    after = float(model.ELBO((X, Y), seed=123))
    assert after > before + 50.0, (before, after)


def _bo_model(seed=1):
    import dgp_toolbox_b200 as D
    rng = np.random.default_rng(0)
    X = rng.uniform(-1, 1, (60, 2))
    Y = np.sin(3 * X[:, :1]) * np.cos(2 * X[:, 1:]) + 0.05 * rng.standard_normal((60, 1))
    kernels = [D.RBF(lengthscales=[0.7, 0.7], variance=1.0) for _ in range(3)]
    return D.DGP(X, Y, X[:20].copy(), kernels, [2, 2], D.Gaussian(0.1), num_samples=5, seed=seed), X, Y


def test_graph_replay_is_bit_exact():
    """dgp_set_graph(1) replays the captured launch sequence with the seed read from device memory: ELBO + gradients, mixture
    moments and EI must equal the directly launched calls bit for bit, for every seed, after in-place parameter updates
    (same buffers -> same graph) and for a second call signature held in the cache at the same time."""
    import dgp_toolbox_b200 as D
    model, X, Y = _bo_model()
    ctx = D._lib.get_context(0)
    Xd, Yd = model.data
    Xs = Xd[:25].contiguous()
    out_a = torch.empty(model.grad_layout()[0], dtype=torch.float64, device="cuda")
    out_b = torch.empty_like(out_a)
    try:
        for rnd in range(2):
            for seed in (3, 4, 2 ** 63 + 11):
                ctx.set_graph(False)
                ref = model.elbo_flat((Xd, Yd), seed=seed, out=out_a).clone()
                ref_small = model.elbo_flat((Xs, Yd[:25].contiguous()), seed=seed).clone()
                pm_ref = [t.clone() for t in model.predict_moments(Xd, 5, seed=seed)]
                ctx.set_graph(True)
                n0 = ctx.launch_count(reset=True)
                got = model.elbo_flat((Xd, Yd), seed=seed, out=out_b)
                assert torch.equal(got, ref)
                got2 = model.elbo_flat((Xd, Yd), seed=seed, out=out_b)      # replay of the entry captured above
                assert torch.equal(got2, ref)
                assert ctx.launch_count() > 20                               # replays count the launches of the captured step
                Ys = Yd[:25].contiguous()
                assert torch.equal(model.elbo_flat((Xs, Ys), seed=seed), ref_small)   # fresh buffers: a new signature (LRU cache)
                pm_got = model.predict_moments(Xd, 5, seed=seed)
                assert all(torch.equal(a, b) for a, b in zip(pm_got, pm_ref))
            # move the parameters in place: the cached graphs must see the new values
            model.layers[0].kern.lengthscales.assign(model.layers[0].kern.lengthscales.value * 1.1)
            model.layers[-1].q_mu.assign(model.layers[-1].q_mu.value + 0.05)
    finally:
        ctx.set_graph(False)


def test_sharded_training_step_equals_the_unsharded_one():
    """ShardedELBO.train_adam_step on the two halves of a minibatch in turn (what two ranks do before their allreduce), summed
    by hand, followed by dgp_adam_step == one unsharded training iteration: same parameters to rounding of the sum order."""
    import dgp_toolbox_b200 as D
    from dgp_toolbox_b200.distributed import ShardedELBO, shard_bounds
    ma, X, Y = _bo_model(seed=3)
    mb, _, _ = _bo_model(seed=3)
    Xd, Yd = ma.data
    pa, pb = ma.trainable_parameters, mb.trainable_parameters
    sa, sb = ma._adam_state(pa), mb._adam_state(pb)
    for t in range(1, 4):
        flat = ma.elbo_flat((Xd, Yd), seed=100 + t)
        ma._adam_step(pa, flat, sa, t, 0.02, 0.9, 0.999, 1e-7)
        parts = []
        for r in range(2):
            lo, hi = shard_bounds(Xd.shape[0], r, 2)
            parts.append(mb.elbo_flat((Xd[lo:hi].contiguous(), Yd[lo:hi].contiguous()), kl_weight=0.5, seed=100 + t, n_offset=lo))
        mb._adam_step(pb, parts[0] + parts[1], sb, t, 0.02, 0.9, 0.999, 1e-7)
    for a, b in zip(pa, pb):
        assert float((a.value - b.value).abs().max()) <= 1e-9 * max(1.0, float(a.value.abs().max()))
    one = ShardedELBO(mb)                      # world 1: the wrapper is the plain step + dgp_adam_step
    before = [p.value.clone() for p in pb]
    one.train_adam_step(Xd, Yd, 0, pb, sb, 4, lr=0.02, seed=7)
    assert any(not torch.equal(p.value, q) for p, q in zip(pb, before))


def test_train_adam_equals_stepwise_calls_and_graph_replay():
    """dgp_train_adam (loop in the library) == elbo_flat + dgp_adam_step called step by step with the model's seed sequence,
    bit for bit, with and without graph replay."""
    import dgp_toolbox_b200 as D
    ctx = D._lib.get_context(0)
    results = []
    for mode in ("stepwise", "library", "library+graph"):
        model, X, Y = _bo_model(seed=7)
        params = model.trainable_parameters
        state = model._adam_state(params)
        try:
            ctx.set_graph(mode == "library+graph")
            if mode == "stepwise":
                trace = []
                for t in range(1, 13):
                    flat = model.elbo_flat(model.data)
                    trace.append((flat[0] - flat[1]).reshape(1))
                    model._adam_step(params, flat, state, t, 0.02, 0.9, 0.999, 1e-7)
                trace = torch.cat(trace)
            else:
                trace = torch.cat([model._train_adam(model.data, params, state, 1, 5, 0.02, 0.9, 0.999, 1e-7),
                                   model._train_adam(model.data, params, state, 6, 7, 0.02, 0.9, 0.999, 1e-7)])
        finally:
            ctx.set_graph(False)
        results.append((trace.clone(), [p.value.clone() for p in params], model._draw))
    for trace, values, draw in results[1:]:
        assert draw == results[0][2]
        assert torch.equal(trace, results[0][0])
        assert all(torch.equal(a, b) for a, b in zip(values, results[0][1]))


@pytest.mark.parametrize("fused", [True, False])
def test_first_layer_sharing_equals_per_sample_evaluation(fused):
    """The first layer is evaluated once per point and expanded over the S samples; switching that off evaluates every
    point-sample like the reference. Values, gradients and propagated samples must agree to summation order."""
    import dgp_toolbox_b200 as D
    from dgp_toolbox_b200 import synthetic
    model, cfg = _c2_model(S=8)
    X, Y = synthetic.minibatch(cfg["D0"], 700, 4)
    ctx = D._lib.get_context(0)
    ctx.set_fused(fused)
    try:
        a = model.elbo_flat((X, Y), want_grad=True, seed=21).clone()
        Fa = [t.clone() for t in sum(model.propagate(X, S=8, seed=22), [])]
        ctx.set_share_first_layer(False)
        b = model.elbo_flat((X, Y), want_grad=True, seed=21).clone()
        Fb = [t.clone() for t in sum(model.propagate(X, S=8, seed=22), [])]
    finally:
        ctx.set_share_first_layer(True)
        ctx.set_fused(True)
    assert float((a - b).abs().max()) <= 1e-10 * float(b.abs().max())
    for x, y in zip(Fa, Fb):
        assert float((x - y).abs().max()) <= 1e-11 * max(float(y.abs().max()), 1.0)


def test_notebook_regression_schedule_learns_the_step():
    """Notebooks_dgp/nb_DGP_regression.ipynb cells 10-26 on the drop-in classes with a shortened schedule: the ELBO starts at
    the notebook's printed -85.988 (KAT-1), drops to -406.376 after the hidden q_sqrt rescaling (KAT-1b) and must climb well
    above that under optimize_nat_adam; the full schedule reaches 106.3 +- 1.6 (profiles/r01h_notebook_regression.log; notebook: 104-109)."""
    import dgp_toolbox_b200 as D
    np.random.seed(0)
    X = np.random.uniform(0, 1, 50)[:, None]
    Z = np.random.uniform(0, 1, 25)[:, None]
    Y = (X >= 0.5).astype(np.float64) + 1e-2 * np.random.randn(50, 1)
    model = D.DGP(X, Y, Z, [D.RBF(lengthscales=[1.0], variance=1.0) for _ in range(3)], [1, 1], D.Gaussian(), num_samples=10, seed=0)
    assert abs(float(model.ELBO((X, Y))) - (-85.98812279560475)) < 1e-7
    model.optimize_nat_adam(iterations1=200, iterations2=800, lr_adam=0.01, beta_1=0.8, beta_2=0.9, lr_gamma=0.01, ng_all=False,
                            messages=10 ** 9)
    elbo = np.mean([float(model.ELBO((X, Y), seed=500 + i)) for i in range(10)])
    assert elbo > -60.0, elbo
    m, _ = model.predict(np.array([[0.1], [0.9]]), 50, seed=3)
    assert float(m[0]) < 0.3 and float(m[1]) > 0.7


def test_vform_forward_equals_reference_operation_order():
    """Forward-only calls fold C_d = q_sqrt_d^T Lu^-T and beta = Lu^-1 q_mu once and skip the A = Lu^-T V pass; switching
    that off keeps the reference's operation order. Same values to rounding."""
    import dgp_toolbox_b200 as D
    from dgp_toolbox_b200 import synthetic
    model, cfg = _c2_model(S=4)
    X, _ = synthetic.minibatch(cfg["D0"], 300, 6)
    ctx = D._lib.get_context(0)
    a = [t.clone() for t in sum(model.propagate(X, S=4, seed=5), [])]
    ma, va = model.predict(X, 4, seed=6)
    Y = np.sin(X.sum(1, keepdims=True))
    ctx.set_vform(True, "always")
    ga = model.elbo_flat((X, Y), want_grad=True, seed=7).clone()
    ctx.set_vform(False, False)
    try:
        b = [t.clone() for t in sum(model.propagate(X, S=4, seed=5), [])]
        mb, vb = model.predict(X, 4, seed=6)
        gb = model.elbo_flat((X, Y), want_grad=True, seed=7).clone()
    finally:
        ctx.set_vform(True, True)
    for x, y in zip(a + [ma, va], b + [mb, vb]):
        assert float((x - y).abs().max()) <= 1e-10 * max(float(y.abs().max()), 1.0)
    # gradients: same adjoint through two different parameterisations (V-form maps back through the Cholesky adjoint)
    _, offs = model.grad_layout()
    bounds = [0, 3] + [o.dZ for o in offs[1:]] + [ga.numel()]
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        assert float((ga[lo:hi] - gb[lo:hi]).abs().max()) <= 1e-8 * max(float(gb[lo:hi].abs().max()), 1e-12)


def test_failed_cholesky_is_raised_at_the_failing_block_and_freezes_the_parameters(capsys):
    """A non-positive-definite Kuu (here: a negative kernel variance written behind the bijector's back) must not destroy
    the model: the flag is sticky until reported, the fused Adam launch skips flagged steps, and the training loop raises at
    the message block the failure happened in (the reference raises at the failing step, models/dgp.py:142-146)."""
    import dgp_toolbox_b200 as D
    from oracle import dgp_oracle as O
    from tests.helpers import product_model_from_problem
    prob = O.synthetic_problem(3, [3], 16, 40)
    pm = product_model_from_problem(prob, 4)
    data = (prob["X"], prob["Y"])
    pm.optimize_adam(data, iterations=2, messages=1)          # healthy steps first
    before = [p.value.clone() for p in pm.trainable_parameters]
    good_var = pm.layers[1].kern.variance.value.clone()
    pm.layers[1].kern.variance.value.fill_(-1.0)
    before[[id(p) for p in pm.trainable_parameters].index(id(pm.layers[1].kern.variance))].fill_(-1.0)
    with pytest.raises(D._lib.DGPError, match="positive definite"):
        pm.optimize_adam(data, iterations=5, messages=1)
    for p, b in zip(pm.trainable_parameters, before):
        assert torch.equal(p.value, b), p                      # nothing was overwritten with NaN
    with pytest.raises(D._lib.DGPError, match="positive definite"):
        pm.predict(prob["X"], 4)
    pm.layers[1].kern.variance.value.copy_(good_var)
    m, v = pm.predict(prob["X"], 4)                            # reported once: the next call starts clean
    assert bool(torch.isfinite(m).all()) and bool(torch.isfinite(v).all())
    capsys.readouterr()


def test_foreign_dlpack_producers_enter_through_as_device():
    """north_star: tensors are exchanged via DLPack. TensorFlow is absent from the image, so the producer here is a minimal foreign
    object exposing only `__dlpack__` / `__dlpack_device__` (what an eager tf.Tensor offers), on the host and on the device; both
    must give the same results as a numpy input through the public API."""
    import dgp_toolbox_b200 as D

    class Foreign:
        def __init__(self, backing):
            self._b = backing

        def __dlpack__(self, *args, **kwargs):
            return self._b.__dlpack__(*args, **kwargs)

        def __dlpack_device__(self):
            return self._b.__dlpack_device__()

    model, cfg = _c2_model(S=4)
    X = np.random.default_rng(0).standard_normal((33, cfg["D0"]))
    ref_m, ref_v = model.predict(X, 4, seed=9)
    host = Foreign(X.copy())                                     # kDLCPU capsule
    dev = Foreign(torch.as_tensor(X).cuda())                     # kDLCUDA capsule: zero-copy path
    for obj in (host, dev):
        t = D._lib.as_device(obj)
        assert t.is_cuda and t.dtype == torch.float64 and torch.equal(t.cpu(), torch.as_tensor(X))
        m, v = model.predict(obj, 4, seed=9)
        assert torch.equal(m, ref_m) and torch.equal(v, ref_v)
    assert D._lib.as_device(dev).data_ptr() == dev._b.data_ptr()  # no copy for a float64 CUDA producer


def test_kernel_exponential_is_accurate_to_ulps():
    """The kernel functions use a branch-free exp for non-positive arguments (csrc/common.cuh exp_nonpos) so that independent
    evaluations interleave; it must stay within 2 ulp of the correctly rounded value over the whole argument range, give exp(0) = 1
    exactly (unit diagonal of Kuu / variance) and clamp below -700 (true value < 1e-304)."""
    import dgp_toolbox_b200 as D
    G = D.gpflow_shim
    x = np.concatenate([np.linspace(0.0, 37.0, 20001), np.random.default_rng(0).uniform(0.0, 37.0, 20000)])[:, None]
    k = G.SquaredExponential(variance=1.0, lengthscales=1.0)
    K = k.K(x, np.zeros((1, 1))).cpu().numpy()[:, 0]
    ref = np.exp(-0.5 * x[:, 0] ** 2)
    assert K[0] == 1.0
    rel = np.abs(K - ref) / ref
    assert rel.max() < 2 * np.finfo(np.float64).eps, rel.max()
    far = k.K(np.array([[40.0], [1e3]]), np.zeros((1, 1))).cpu().numpy()[:, 0]
    assert np.all(far >= 0.0) and np.all(far < 1e-300)
    for cls, f in ((G.Matern32, lambda r: (1 + np.sqrt(3) * r) * np.exp(-np.sqrt(3) * r)),
                   (G.Matern52, lambda r: (1 + np.sqrt(5) * r + 5.0 / 3.0 * r * r) * np.exp(-np.sqrt(5) * r))):
        Km = cls(variance=1.0, lengthscales=1.0).K(x[1:], np.zeros((1, 1))).cpu().numpy()[:, 0]
        refm = f(x[1:, 0])
        assert (np.abs(Km - refm) / refm).max() < 1e-14


def test_bench_dump_outputs_are_the_last_timed_step(tmp_path):
    """bench.py --dump-outputs writes the ELBO terms and the gradients of its last timed step: the same arrays come out of
    one direct elbo_flat call on that step's inputs (bench.step_inputs: minibatch, Philox seed, point offset and scale)."""
    import json
    import os
    import subprocess
    import sys
    import bench
    from dgp_toolbox_b200 import synthetic
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    steps, nb = bench.N_POOL + 2, 512      # the last step reuses a pool minibatch with its own seed and point offset
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
                          "--nb", str(nb), "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    model, cfg = _c2_model()
    s = bench.step_inputs(steps - 1, nb)
    X, Y = synthetic.minibatch(cfg["D0"], nb, s["batch"])
    flat = model.elbo_flat((X, Y), scale=s["scale"], seed=s["seed"], n_offset=s["n_offset"])
    ref = bench.step_outputs(model, flat)
    assert sorted(os.listdir(tmp_path)) == sorted(k + ".npy" for k in ref)
    for k, v in ref.items():
        got = np.load(os.path.join(tmp_path, k + ".npy"))
        assert got.dtype == np.float64 and got.shape == v.shape, k
        assert np.max(np.abs(got - v), initial=0.0) <= 1e-11 * max(np.max(np.abs(v), initial=0.0), 1e-300), k
    assert abs(float(np.load(os.path.join(tmp_path, "elbo.npy"))) - line["elbo_last_step"]) <= 1e-12 * abs(line["elbo_last_step"])
