"""CPU-side checks: the C-ABI library loads and exports every symbol include/dgp_b200.h declares (no compute calls),
the product-side synthetic generator equals the oracle's, host-side parameter transforms, and the sharding arithmetic of
the multi-GPU path on a world_size-2 gloo group (with the oracle standing in for the per-rank compute)."""
import os
import re
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import dgp_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_header_symbol():
    import ctypes
    import __graft_entry__ as G
    G.build()
    lib = ctypes.CDLL(os.path.join(ROOT, "dgp_toolbox_b200", "libdgp_b200.so"))
    hdr = open(os.path.join(ROOT, "include", "dgp_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = set(re.findall(r"\b(dgp_[A-Za-z0-9_]+)\s*\(", hdr))
    assert len(names) >= 20
    for n in sorted(names):
        assert hasattr(lib, n), f"{n} declared in include/dgp_b200.h but not exported"
    from dgp_toolbox_b200 import _lib
    assert set(_lib.EXPORTED_SYMBOLS) <= names
    assert lib.dgp_version() == 100


def test_grad_layout_sizes():
    import ctypes as C
    from dgp_toolbox_b200 import _lib
    arr = (_lib.LayerDesc * 2)()
    arr[0].D_in, arr[0].D_out, arr[0].M = 3, 4, 10
    arr[1].D_in, arr[1].D_out, arr[1].M = 4, 1, 10
    m = _lib.ModelDesc(2, arr, None)
    n = _lib.lib.dgp_grad_size(C.byref(m))
    offs = (_lib.GradOffsets * 2)()
    assert _lib.lib.dgp_grad_layout(C.byref(m), offs) == 0
    assert offs[0].dZ == 3 and offs[0].dlengthscales == 33 and offs[0].dvariance == 36 and offs[0].dq_mu == 37
    assert offs[0].dq_sqrt == 77 and offs[1].dZ == 477
    assert n == 3 + (30 + 3 + 1 + 40 + 400) + (40 + 4 + 1 + 10 + 100)


def test_product_synthetic_generator_equals_oracle_generator():
    from dgp_toolbox_b200 import synthetic
    for args in [(8, [8, 8], 32, 20), (5, [3, 6], 16, 30)]:
        a = synthetic.synthetic_problem(*args)
        b = O.synthetic_problem(*args)
        assert np.array_equal(a["X"], b["X"]) and np.array_equal(a["Y"], b["Y"])
        for la, lb in zip(a["layers"], b["layers"]):
            for k in ("Z", "lengthscales", "q_mu", "q_sqrt"):
                assert np.array_equal(la[k], lb[k])
            assert la["mean_kind"] == lb["mean_kind"]
            assert (la["mf_W"] is None) == (lb["mf_W"] is None)
            if la["mf_W"] is not None:
                assert np.array_equal(la["mf_W"], lb["mf_W"])
    f_fwd, f_step = synthetic.flops_per_point_sample(8, [8, 8, 8], 256)
    assert f_fwd == 3 * (10 * 65536 + 4096 + 8704) + (3 * 65536 + 4096 + 1536) and f_step == 3 * f_fwd   # SURVEY §8d: 2.207 MFLOP
    fl = synthetic.flops_per_layer(8, [8, 8, 8], 256, vform=True)
    assert fl[0] == 9 * 65536 + 4096 + 8704 and fl[-1] == 2 * 65536 + 4096 + 1536
    f_v, _ = synthetic.flops_per_point_sample(8, [8, 8, 8], 256, S=32)
    assert abs(f_v - (fl[0] / 32 + sum(fl[1:]))) < 1e-9


def test_shard_bounds_cover_and_are_contiguous():
    from dgp_toolbox_b200.distributed import shard_bounds
    for N in (1, 7, 16, 1000):
        for world in (1, 2, 3, 8):
            cuts = [shard_bounds(N, r, world) for r in range(world)]
            assert cuts[0][0] == 0 and cuts[-1][1] == N
            assert all(cuts[i][1] == cuts[i + 1][0] for i in range(world - 1))
            sizes = [b - a for a, b in cuts]
            assert max(sizes) - min(sizes) <= 1


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gloo_worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(1)
    from dgp_toolbox_b200.distributed import shard_bounds
    N, S, seed = 24, 3, 77
    prob = O.synthetic_problem(3, [3], 12, N)
    om = O.model_from_problem(prob, S)
    X, Y = torch.as_tensor(prob["X"]), torch.as_tensor(prob["Y"])
    # full-batch draws indexed by the GLOBAL point index (placement-invariant Philox counters)
    zs_full = [torch.as_tensor(O.philox_normal(seed, l, S, N, layer.D_out)) for l, layer in enumerate(om.layers)]
    lo, hi = shard_bounds(N, rank, world)
    zs_loc = [torch.as_tensor(O.philox_normal(seed, l, S, hi - lo, layer.D_out, n_offset=lo)) for l, layer in enumerate(om.layers)]
    for zf, zl in zip(zs_full, zs_loc):
        assert torch.equal(zf[:, lo:hi], zl)
    # per-rank: data term on the shard, KL weighted 1/world  ==  what dgp_elbo_grad(kl_weight=1/world) returns
    params = om.named_params()
    leaves = {k: v.detach().clone().requires_grad_(True) for k, v in params.items()}
    layers = [O.OLayer(Z=leaves[f"layers.{i}.Z"], lengthscales=leaves[f"layers.{i}.lengthscales"], variance=leaves[f"layers.{i}.variance"],
                       q_mu=leaves[f"layers.{i}.q_mu"], q_sqrt=leaves[f"layers.{i}.q_sqrt"], mean_kind=l.mean_kind, mf_W=l.mf_W,
                       mf_b=l.mf_b) for i, l in enumerate(om.layers)]
    m2 = O.OModel(layers=layers, lik_var=leaves["lik_var"], num_samples=S)
    data = O.E_log_p_Y(m2, X[lo:hi], Y[lo:hi], zs_loc).sum()
    kl = sum(O.layer_KL(l) for l in layers) / world
    (data - kl).backward()
    flat = torch.cat([data.detach().reshape(1), kl.detach().reshape(1)] + [leaves[k].grad.reshape(-1) for k in sorted(leaves)])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM)
    if rank == 0:
        val, g = O.elbo_and_grads(om, X, Y, zs_full)
        full = torch.cat([g[k].reshape(-1) if "q_sqrt" not in k else torch.zeros(0) for k in sorted(g)])
        red = torch.cat([leaves[k].grad.reshape(-1) * 0 + flat[2 + off: 2 + off + leaves[k].numel()] if "q_sqrt" not in k else torch.zeros(0)
                         for k, off in zip(sorted(leaves), np.cumsum([0] + [leaves[k].numel() for k in sorted(leaves)])[:-1])])
        ok = abs(float(flat[0] - flat[1]) - float(val)) <= 1e-11 * abs(float(val)) and float((full - red).abs().max()) <= 1e-10 * float(full.abs().max())
        q.put(bool(ok))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_sum_equals_full_batch_gloo_world2():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    ok = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert ok


def test_parameter_transforms_round_trip():
    # softplus / FillTriangular helpers used by the optimiser shim (SURVEY §9)
    x = np.arange(1.0, 7.0)
    L = O.fill_triangular(x)
    assert np.array_equal(L, np.array([[4.0, 0, 0], [6.0, 5.0, 0], [3.0, 2.0, 1.0]]))
    assert np.array_equal(O.fill_triangular_inverse(L), x)
    th = np.array([1e-3, 0.5, 3.0, 40.0])
    assert np.allclose(O.softplus(O.softplus_inv(th)), th, rtol=1e-12)


def test_bench_reference_arm_prints_one_json_line():
    """bench.py --impl reference runs on host cores only (no GPU, no /root/reference) and prints the contract's JSON line."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--nb-cpu", "32"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-500:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "point-samples/s" and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["e2e"]["h2d_bytes_per_step"] == 0 and d["value"] > 0


def test_bench_dump_outputs_keep_to_the_size_limit(tmp_path):
    """bench.py --dump-outputs: float64 arrays under the size limit are written whole; above it, the large arrays become the
    same seeded sample of their entries on every run."""
    import bench
    arrays = {"small": np.arange(10.0), "large": np.random.default_rng(1).standard_normal((3, 100, 100))}
    bench.dump_outputs(str(tmp_path / "whole"), arrays)
    for k, v in arrays.items():
        assert np.array_equal(np.load(tmp_path / "whole" / (k + ".npy")), v)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays, limit=1 << 12)
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= (1 << 12) + 2 * 128   # + the .npy headers
    small, large = np.load(tmp_path / "a" / "small.npy"), np.load(tmp_path / "a" / "large.npy")
    assert np.array_equal(small, arrays["small"]) and large.dtype == np.float64 and large.shape == ((1 << 12) // 16,)
    assert np.all(np.isin(large, arrays["large"])) and np.array_equal(large, np.load(tmp_path / "b" / "large.npy"))


def test_chunked_oracle_equals_single_pass():
    """oracle.elbo_and_grads_chunked (used by the full-size GPU parity tests) == oracle.elbo_and_grads on the same Philox draws."""
    import torch
    from oracle import dgp_oracle as O
    prob = O.synthetic_problem(3, [3], 16, 50)
    om = O.model_from_problem(prob, 4)
    X, Y = torch.as_tensor(prob["X"]), torch.as_tensor(prob["Y"])
    zs = [torch.as_tensor(O.philox_normal(9, l, 4, 50, layer.D_out)) for l, layer in enumerate(om.layers)]
    v, g = O.elbo_and_grads(om, X, Y, zs, scale=2.0)
    v2, g2 = O.elbo_and_grads_chunked(om, X, Y, 9, chunk=16, scale=2.0)
    assert abs(float(v) - v2) <= 1e-12 * abs(v2)
    for k in g:
        assert float((g[k] - g2[k]).abs().max()) <= 1e-10 * float(g[k].abs().max() + 1e-300), k
