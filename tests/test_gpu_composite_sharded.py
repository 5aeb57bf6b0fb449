"""Data-parallel MF-DGP, MF-DGP-EM and MO-DGP (distributed.ShardedComposite): draws indexed by the global point, the world-1
path, the shards of one GPU summed against the full batch, and -- with two GPUs -- the library allreduce and the sharded
training schedules against the one-GPU run."""
import contextlib
import io
import os
import socket
import traceback

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _rel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.max(np.abs(a - b))) / max(float(np.max(np.abs(b))), 1e-300)


def _make(name, dev):
    """The shapes of test_gpu_mf.py / test_gpu_mo.py with odd point counts, so that two shards are uneven. Constructor draws
    from a fixed Philox stream: every process builds the same model."""
    import dgp_toolbox_b200 as D
    from dgp_toolbox_b200.models.MF_DGP import _PhiloxDraws
    draw = _PhiloxDraws(dev, 1)
    if name == "mf":
        rng = np.random.default_rng(3)
        f_lo = lambda x: np.sin(6 * x)
        X = [rng.uniform(0, 1, (31, 1)), rng.uniform(0, 1, (13, 1))]
        obj = D.MultiFidelityDeepGP(X, [f_lo(X[0]), 1.5 * f_lo(X[1]) + 0.3 * X[1]], draw=draw)
        obj.model.num_samples = 4
        return obj, (obj._X, obj._Y)
    if name == "em":
        rng = np.random.default_rng(5)
        X = [rng.uniform(0, 1, (25, 2)), rng.uniform(0, 1, (11, 3))]
        f = lambda x: np.sin(4 * x[:, :1]) + x[:, 1:2]
        obj = D.MultiFidelityDeepGP_EM(X, [f(X[0]), 1.3 * f(X[1]) + 0.2 * X[1][:, 2:3]], [X[1][:, :2].copy()], draw=draw)
        obj.model.num_samples = 3
        obj.model.layers[0].kern.kernels[-1].variance.assign(1e-2)
        return obj, (obj._X, obj._Y, obj._X_red)
    rng = np.random.default_rng(11)
    X = rng.uniform(0, 1, (17, 2))
    Y = [np.sin(3 * X[:, :1]) + 0.5 * X[:, 1:2], np.cos(2 * X[:, :1]) * X[:, 1:2] - 0.3]
    obj = D.MultiObjDeepGP([X, X.copy()], Y, loop=1, draw=draw)
    obj.model.num_samples = 3
    obj.model.layers[0].kern.kernels[-1].variance.assign(1e-1)
    return obj, (obj._X, obj._Y)


MODELS = ["mf", "em", "mo"]
DEV = torch.device("cuda", 0)


class _Recording:
    def __init__(self, dev, seed):
        from dgp_toolbox_b200.models.MF_DGP import _PhiloxDraws
        self.d, self.log = _PhiloxDraws(dev, seed), []

    def __call__(self, shape, n_offset=0):
        z = self.d(shape, n_offset=n_offset)
        self.log.append((n_offset, z))
        return z


def test_philox_draw_with_offset_is_the_slice_of_the_full_draw():
    from dgp_toolbox_b200.models.MF_DGP import _PhiloxDraws
    full = _PhiloxDraws(DEV, 5)((3, 37, 2))
    for lo, hi in [(0, 19), (19, 37), (7, 8), (36, 37)]:
        assert torch.equal(_PhiloxDraws(DEV, 5)((3, hi - lo, 2), n_offset=lo), full[:, lo:hi])


@pytest.mark.parametrize("name", MODELS)
def test_shard_draws_are_slices_of_the_full_batch_draws(name):
    """Every draw of a shard's evaluation (data-term chains, MO-DGP's start column, the replicated Z_right refresh) equals the
    full-batch evaluation's draw of the same call, restricted to the shard's global points, bit for bit."""
    from dgp_toolbox_b200.distributed import composite_shard
    obj, data = _make(name, DEV)
    m = obj.model
    m.draw = full = _Recording(DEV, 7)
    m.ELBO_and_grads(data)
    for r in range(2):
        local = composite_shard(data, r, 2)
        m.draw = part = _Recording(DEV, 7)
        m.ELBO_and_grads(local.data, shard=local)
        assert len(part.log) == len(full.log)
        for (off, z), (off_f, zf) in zip(part.log, full.log):
            assert off_f == 0 and torch.equal(z, zf[:, off:off + z.shape[1]])
        assert (max(off for off, _ in part.log) > 0) == (r == 1)


@pytest.mark.parametrize("name", MODELS)
def test_world_one_is_the_single_gpu_path(name, capsys):
    from dgp_toolbox_b200.distributed import ShardedComposite
    from dgp_toolbox_b200.models.MF_DGP import _PhiloxDraws
    obj, data = _make(name, DEV)
    m = obj.model
    sc = ShardedComposite(obj)
    assert sc.world == 1
    m.draw = _PhiloxDraws(DEV, 7)
    e0, g0 = m.ELBO_and_grads(data)
    m.draw = _PhiloxDraws(DEV, 7)
    e1, g1 = sc.ELBO_and_grads(sc.local_data(data))
    assert torch.equal(e0, e1) and all(torch.equal(g0[p], g1[p]) for p in g0)
    runs = []
    for wrap in (lambda o: o, ShardedComposite):
        o, _ = _make(name, DEV)
        o.model.draw = _PhiloxDraws(DEV, 9)
        wrap(o).optimize_adam(lr=0.01, iterations1=1, iterations2=1, iterations3=1, messages=1)
        runs.append([p.value.clone() for p in o.model.parameters])
    assert all(torch.equal(a, b) for a, b in zip(*runs))
    capsys.readouterr()


@pytest.mark.parametrize("name", MODELS)
def test_two_uneven_shards_sum_to_the_full_batch(name):
    """What two ranks compute before their allreduce, evaluated in turn on one GPU: local data terms, KL weighted 1/2, the same
    Z_right refresh. Their sum is the full-batch ELBO (1e-9) and every gradient (1e-8)."""
    from dgp_toolbox_b200.distributed import composite_shard
    from dgp_toolbox_b200.models.MF_DGP import _PhiloxDraws
    obj, data = _make(name, DEV)
    m = obj.model
    params = m.trainable_parameters
    m.draw = _PhiloxDraws(DEV, 7)
    elbo, grads = m.ELBO_and_grads(data, params)
    tot, gtot = 0.0, [torch.zeros_like(p.value) for p in params]
    for r in range(2):
        local = composite_shard(data, r, 2)
        assert local.data[0][0].shape[0] == data[0][0].shape[0] // 2 + (1 - r)      # uneven
        m.draw = _PhiloxDraws(DEV, 7)
        e, g = m.ELBO_and_grads(local.data, params, shard=local)
        tot = tot + float(e)
        gtot = [a + g[p] for a, p in zip(gtot, params)]
    assert abs(tot - float(elbo)) <= 1e-9 * abs(float(elbo)), (tot, float(elbo))
    for p, g in zip(params, gtot):
        assert _rel(g.cpu().numpy(), grads[p].cpu().numpy()) < 1e-8, (p, _rel(g.cpu().numpy(), grads[p].cpu().numpy()))


# ---- two GPUs: the library communicator ----

TRAIN = [("optimize_adam", dict(lr=0.01, iterations1=2, iterations2=2, iterations3=2, messages=1)),
         ("optimize_nat_adam", dict(lr_adam=0.01, lr_gamma=1e-4, iterations1=1, iterations2=1, iterations3=2, messages=1))]


def _flat(elbo, grads, params):
    return np.concatenate([np.asarray([float(elbo)])] + [grads[p].reshape(-1).cpu().numpy() for p in params])


def _worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from dgp_toolbox_b200.distributed import ShardedComposite
    from dgp_toolbox_b200.models.MF_DGP import _PhiloxDraws
    out = {}
    sc = None
    try:
        for name in MODELS:
            obj, data = _make(name, dev)
            m = obj.model
            params = m.trainable_parameters
            sc = ShardedComposite(obj)
            m.draw = _PhiloxDraws(dev, 7)
            out[(name, "reduced")] = _flat(*sc.ELBO_and_grads(sc.local_data(data), params), params)
            if rank == 0:
                m.draw = _PhiloxDraws(dev, 7)
                out[(name, "full")] = _flat(*m.ELBO_and_grads(data, params), params)
            sc.close()
            sc = None
            for method, kw in TRAIN:
                obj, _ = _make(name, dev)
                obj.model.draw = _PhiloxDraws(dev, 11)
                sc = ShardedComposite(obj)
                buf = io.StringIO()
                with contextlib.redirect_stdout(buf):
                    getattr(sc, method)(**kw)
                sc.close()
                sc = None
                out[(name, method, "printed")] = "ELBO:" in buf.getvalue()
                out[(name, method, "sharded")] = [p.value.cpu().numpy() for p in obj.model.parameters]
                if rank == 0:
                    obj, _ = _make(name, dev)
                    obj.model.draw = _PhiloxDraws(dev, 11)
                    with contextlib.redirect_stdout(io.StringIO()):
                        getattr(obj, method)(**kw)
                    out[(name, method, "one_gpu")] = [p.value.cpu().numpy() for p in obj.model.parameters]
        q.put((rank, out))
    except Exception:
        q.put((rank, traceback.format_exc()))
    finally:
        if sc is not None:
            sc.close()
        dist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpus_match_the_one_gpu_full_batch_and_training():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    try:
        res = dict(q.get(timeout=900) for _ in procs)
    finally:
        for p in procs:
            p.join(timeout=120)
            if p.is_alive():
                p.terminate()
                p.join()
    for r in (0, 1):
        assert isinstance(res[r], dict), res[r]
    assert all(p.exitcode == 0 for p in procs)
    r0, r1 = res[0], res[1]
    for name in MODELS:
        red, full = r0[(name, "reduced")], r0[(name, "full")]
        assert np.array_equal(red, r1[(name, "reduced")])                  # the reduced buffer is the same on both ranks
        assert abs(red[0] - full[0]) <= 1e-9 * abs(full[0]), (name, red[0], full[0])
        assert _rel(red[1:], full[1:]) < 1e-8, (name, _rel(red[1:], full[1:]))
        for method, _ in TRAIN:
            a, b, one = r0[(name, method, "sharded")], r1[(name, method, "sharded")], r0[(name, method, "one_gpu")]
            assert r0[(name, method, "printed")] and not r1[(name, method, "printed")]
            assert all(np.array_equal(x, y) for x, y in zip(a, b)), (name, method)     # lockstep without a broadcast
            worst = max(_rel(x, y) for x, y in zip(a, one))
            assert worst < 1e-7, (name, method, worst)
