"""Data-parallel ELBO + gradient of the composite-kernel models (distributed.ShardedComposite) on 1..8 GPUs. Prints one JSON line.

   python tools/bench_composite_sharded.py                                     # world 1 (+ the replicated share of a step)
   python -m torch.distributed.run --nproc-per-node N tools/bench_composite_sharded.py

Workloads (BASELINE config 4 and the MO-DGP training step of tools/bench_mo.py):
  * MF-DGP-EM, 3 fidelities with 2/3/4-D inputs, M = 256, S = 10. Weak scaling: 32 768 / 8 192 / 2 048 points per fidelity and GPU;
    strong scaling: that minibatch split over the GPUs.
  * MO-DGP, D_in = 8, M = 256, S = 32, loop = 2. Weak scaling: 16 384 points per objective and GPU; strong: 16 384 in all.
Per run: median ms per step (CUDA events around each step, which ends in a synchronise; the slowest rank's median), point-samples/s,
and the bytes of the one allreduce per step ([data terms, KL terms, gradients] in float64, from the parameter shapes). With world 1
also the replicated part of a step: the same step on 8 points per fidelity, i.e. the Z_right refresh, the per-layer prep (Kuu and
its factorisation), the KL terms and the launches of the data chains, which every rank repeats whatever its share of the points.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=10)
ap.add_argument("--warmup", type=int, default=2)
args = ap.parse_args()

if "RANK" in os.environ:
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local_rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
rank = dist.get_rank() if dist.is_initialized() else 0
world = dist.get_world_size() if dist.is_initialized() else 1
dev = torch.device("cuda", torch.cuda.current_device())

import dgp_toolbox_b200 as D
from dgp_toolbox_b200.distributed import ShardedComposite

D._lib.get_context(dev).set_workspace_limit(64 << 30)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(dev.index)],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(dev)


def timed(fn):
    for _ in range(args.warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(args.steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    med = float(np.median(ms))
    if world > 1:
        meds = [None] * world
        dist.all_gather_object(meds, med)
        med = max(meds)
    return med


def em_problem(n):
    """Config 4 (bench.py's c4_mf_dgp_em) with n[l] points of fidelity l; the same inducing inputs on every rank."""
    rng = np.random.default_rng(0)
    dims = [2, 3, 4]
    f4 = lambda x: np.sin(3 * x[:, :1]) + 0.5 * x[:, 1:2]
    X = [rng.uniform(0, 1, (k, d)) for k, d in zip(n, dims)]
    Y = [f4(X[0]), 1.2 * f4(X[1]) + 0.3 * X[1][:, :1] ** 2, 1.5 * f4(X[2]) - 0.2 * X[2][:, 1:2]]
    X_red = [X[1][:, :2].copy(), X[2][:, :2].copy()]      # as bench.py c4_mf_dgp_em
    obj = D.MultiFidelityDeepGP_EM(X, Y, X_red, Z=[rng.uniform(0, 1, (256, d)) for d in dims],
                                   W=[rng.uniform(0, 1, (256, 4)), rng.uniform(0, 1, (256, 3))])
    obj.model.num_samples = 10
    return obj, (X, Y, X_red)


def mo_problem(n):
    rng = np.random.default_rng(0)
    f0 = lambda x: np.sin(3 * x[:, :1]) + 0.5 * x[:, 1:2]
    f1 = lambda x: np.cos(2 * x[:, :1]) * x[:, 1:2] - 0.3
    Zx = rng.uniform(0, 1, (256, 8))
    X = rng.uniform(0, 1, (n, 8))
    obj = D.MultiObjDeepGP([X, X.copy()], [f0(X), f1(X)], Z=[np.concatenate([Zx, f1(Zx)], 1), Zx.copy()], loop=2)
    obj.model.layers[0].kern.kernels[-1].variance.assign(1e-2)
    for k, layer in enumerate(obj.model.layers):
        layer.q_mu.assign((f0, f1)[k](Zx) + 0.05 * rng.standard_normal((256, 1)))
        layer.q_sqrt.assign(0.1 * layer.q_sqrt.value)
    obj.model.num_samples = 32
    return obj, ([X, X.copy()], [f0(X), f1(X)])


def on_device(data):
    return tuple([torch.as_tensor(a, device=dev) for a in part] for part in data)


def run(make, n_global):
    obj, data = make(n_global)
    sc = ShardedComposite(obj)
    local = sc.local_data(on_device(data))
    params = obj.model.trainable_parameters
    ms = timed(lambda: sc.ELBO_and_grads(local, params))
    sc.close()
    S = obj.model.num_samples
    point_samples = sum(np.shape(x)[0] for x in data[0]) * S
    res = {"ms_per_step": ms, "point_samples_per_step": point_samples, "point_samples_per_s": point_samples / (ms * 1e-3),
           "allreduce_bytes": 8 * (2 + sum(p.value.numel() for p in params)) if world > 1 else 0}
    del obj, sc, local
    torch.cuda.empty_cache()
    return res


EM_PER_GPU, MO_PER_GPU = [32768, 8192, 2048], 16384
out = {"world": world, "card": card(), "steps": args.steps, "warmup": args.warmup,
       "mf_dgp_em": {"weak": run(em_problem, [k * world for k in EM_PER_GPU]), "strong": run(em_problem, EM_PER_GPU)},
       "mo_dgp": {"weak": run(mo_problem, MO_PER_GPU * world), "strong": run(mo_problem, MO_PER_GPU)}}
if world == 1:
    for key, make, tiny in (("mf_dgp_em", em_problem, [8, 8, 8]), ("mo_dgp", mo_problem, 8)):
        rep = run(make, tiny)["ms_per_step"]
        full = out[key]["strong"]["ms_per_step"]
        out[key]["replicated"] = {"ms_per_step": rep, "share_of_step": rep / full,
                                  "strong_scaling_cap_8": full / (rep + (full - rep) / 8)}
D._lib.get_context(dev).check()
if rank == 0:
    print(json.dumps(out))
if dist.is_initialized():
    dist.destroy_process_group()
