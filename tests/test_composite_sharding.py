"""Host logic of the data-parallel composite-kernel models (distributed.composite_shard / ShardedComposite): the per-fidelity
shard layout with X_red aligned to X[l+1], the projection scale from global counts, the 1/world KL weight, the refusals, and the
packing / reduction of ShardedComposite over gloo with a CPU stand-in model. No GPU needed."""
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _em_data(ns=(25, 11, 6), dims=(2, 3, 4)):
    rng = np.random.default_rng(0)
    X = [rng.uniform(0, 1, (n, d)) for n, d in zip(ns, dims)]
    Y = [x[:, :1] ** 2 for x in X]
    X_red = [X[l + 1][:, :dims[l]].copy() for l in range(len(X) - 1)]
    return X, Y, X_red


@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_shard_layout_per_fidelity_and_x_red_alignment(world):
    from dgp_toolbox_b200.distributed import composite_shard, shard_bounds
    X, Y, X_red = _em_data()
    parts = [composite_shard((X, Y, X_red), r, world) for r in range(world)]
    for l, x in enumerate(X):
        assert all(p.counts[l] == x.shape[0] for p in parts)
        for r, p in enumerate(parts):
            lo, hi = shard_bounds(x.shape[0], r, world)
            assert p.offsets[l] == lo
            assert np.array_equal(p.data[0][l], x[lo:hi]) and np.array_equal(p.data[1][l], Y[l][lo:hi])
        assert np.array_equal(np.concatenate([p.data[0][l] for p in parts]), x)
    for p in parts:        # X_red[l] takes the bounds of X[l+1]: the pairs stay row for row
        for l, xr in enumerate(p.data[2]):
            assert np.array_equal(xr, p.data[0][l + 1][:, :xr.shape[1]])
    if world == 1:
        assert parts[0].offsets == (0, 0, 0) and parts[0].kl_weight == 1.0


def test_shard_layout_of_two_set_data_and_torch_tensors():
    from dgp_toolbox_b200.distributed import composite_shard
    X = [torch.arange(10.0).reshape(5, 2), torch.arange(6.0).reshape(3, 2)]
    Y = [torch.ones(5, 1), torch.zeros(3, 1)]
    p = composite_shard((X, Y), 1, 2)
    assert len(p.data) == 2 and p.offsets == (3, 2) and p.counts == (5, 3)
    assert torch.equal(p.data[0][0], X[0][3:]) and torch.equal(p.data[0][1], X[1][2:])


def test_projection_scale_uses_global_counts():
    from dgp_toolbox_b200.distributed import composite_shard
    from dgp_toolbox_b200.models.MF_DGP_EM import projection_scale
    X, Y, X_red = _em_data((25, 11, 6))
    full = [float(X[l + 1].shape[0]) / float(X[l].shape[0]) for l in range(2)]
    assert [projection_scale([x.shape[0] for x in X], l) for l in range(2)] == full
    for world in (2, 3, 4):
        for r in range(world):
            p = composite_shard((X, Y, X_red), r, world)
            assert [projection_scale(p.counts, l) for l in range(2)] == full
    p = composite_shard((X, Y, X_red), 3, 4)           # shard sizes 6, 2, 1: the local ratio would differ
    local = [float(p.data[0][l + 1].shape[0]) / float(p.data[0][l].shape[0]) for l in range(2)]
    assert local != full


@pytest.mark.parametrize("world", [1, 2, 3, 5, 8])
def test_kl_weight_sums_to_one_over_the_ranks(world):
    from dgp_toolbox_b200.distributed import composite_shard
    X, Y, X_red = _em_data((25, 11, 9))
    w = [composite_shard((X, Y, X_red), r, world).kl_weight for r in range(world)]
    assert all(v == 1.0 / world for v in w)
    assert math.isclose(math.fsum(w), 1.0, rel_tol=0, abs_tol=1e-15)


def test_refusals():
    from dgp_toolbox_b200.distributed import composite_shard
    X, Y, X_red = _em_data((25, 11, 3))
    with pytest.raises(ValueError, match="fewer than the 4 ranks"):
        composite_shard((X, Y, X_red), 0, 4)
    with pytest.raises(ValueError, match="row for row"):
        composite_shard((X, Y, [X_red[0], X_red[1][:-1]]), 0, 2)
    with pytest.raises(ValueError, match="row for row"):
        composite_shard((X, Y, X_red[:1]), 0, 2)
    with pytest.raises(ValueError, match="outputs"):
        composite_shard((X, [Y[0], Y[1][:-1], Y[2]], X_red), 0, 2)
    with pytest.raises(ValueError, match="output sets"):
        composite_shard((X, Y[:2]), 0, 2)
    with pytest.raises(ValueError, match="fewer than the 2 ranks"):     # MO-DGP / MF-DGP data: every objective counts
        composite_shard(([np.zeros((4, 2)), np.zeros((1, 2))], [np.zeros((4, 1)), np.zeros((1, 1))]), 1, 2)


class _P:
    def __init__(self, v):
        self.value = torch.as_tensor(v, dtype=torch.float64)


class _ToyModel:
    """CPU stand-in with the interface ShardedComposite drives: ELBO = sum_n a . x_n - |b|^2 (+ the EM projection terms), the
    data terms local partial sums and the KL terms weighted by shard.kl_weight, as the composite models do."""

    def __init__(self, em):
        self.a, self.b = _P([0.5, -1.0]), _P([[0.3, 0.2], [0.1, -0.4]])
        self.device = torch.device("cpu")
        self.em = em

    @property
    def trainable_parameters(self):
        return [self.a, self.b]

    def ELBO_and_grads(self, data, params=None, shard=None):
        vals = {p: p.value.clone().requires_grad_(True) for p in params}
        a, b = vals[self.a], vals[self.b]
        w = 1.0 if shard is None else shard.kl_weight
        self.L = sum((torch.as_tensor(x) @ a).sum() for x in data[0])
        self.KL = (b ** 2).sum() * w
        if self.em:
            self.L_red = sum((torch.as_tensor(x).sum(1) * a[0]).sum() for x in data[2])
            self.KL_red = (b[0] ** 2).sum() * w
        elbo = self.L + getattr(self, "L_red", 0.0) - self.KL - getattr(self, "KL_red", 0.0)
        g = torch.autograd.grad(elbo, [vals[p] for p in params])
        return elbo.detach(), dict(zip(params, g))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gloo_worker(rank, world, port, q):
    import types
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(1)
    from dgp_toolbox_b200.distributed import ShardedComposite
    rng = np.random.default_rng(1)
    X = [rng.standard_normal((7, 2)), rng.standard_normal((5, 2))]
    Y = [np.zeros((7, 1)), np.zeros((5, 1))]
    out = []
    for em in (False, True):
        data = (X, Y, [X[1][:, :1].copy()]) if em else (X, Y)
        m = _ToyModel(em)
        sc = ShardedComposite(types.SimpleNamespace(model=m))
        elbo, g = sc.ELBO_and_grads(sc.local_data(data))
        ref = _ToyModel(em)
        full, gf = ref.ELBO_and_grads(data, ref.trainable_parameters)
        ok = abs(float(elbo - full)) <= 1e-12 * abs(float(full))
        ok = ok and all(torch.allclose(g[p], gf[pr], rtol=1e-12, atol=1e-13) and g[p].shape == p.value.shape
                        for p, pr in zip(m.trainable_parameters, ref.trainable_parameters))
        out.append(bool(ok))
    q.put((rank, out))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_composite_reduces_to_the_full_batch_gloo_world2():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    try:
        res = dict(q.get(timeout=120) for _ in procs)
    finally:
        for p in procs:
            p.join(timeout=60)
            if p.is_alive():
                p.terminate()
    assert all(p.exitcode == 0 for p in procs)
    assert res == {0: [True, True], 1: [True, True]}
