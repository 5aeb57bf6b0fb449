"""full_cov=True of one RBF SVGP layer on per-sample inputs X [S, N, D_in] with draws z, at the config-4 / config-5 layer shapes
(M = 256, D_out = 1; config 4: D_in = 4, S = 10, N = 768; config 5: D_in = 8, S = 8, N = 512). Three ways to get the same
(F, mean, cov):
  fused        SVGP_Layer.sample_from_conditional(full_cov=True): one dgp_propagate_full_cov_snd call (fused conditional, covariance
               tiles with K(X_s, X_s) built in the tile, Cholesky, samples).
  torch_k      Kuu + jitter I, Kuf and the S blocks K(X_s, X_s) built in PyTorch (float64 on the GPU, the oracle's formulas), then
               composite.svgp_from_k_full_cov (the supplied-matrix path).
  per_sample   one shared-input dgp_propagate_full_cov call per sample (how sample_from_conditional ran before it took all S
               samples in one call).
Each arm is warmed up, then timed with CUDA events over --iters calls per repetition; repetitions alternate the arms. Prints one
JSON line per shape: median, min and max ms per call over the repetitions, the largest relative difference of torch_k and
per_sample from fused, and the GPU's name and power limit. The working set (S * D_out blocks of N x N, a few MB) sits in L2.
Needs a GPU.
   python tools/bench_fused_full_cov.py [--reps 7] [--iters 10]"""
import argparse, json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import dgp_toolbox_b200 as D
from dgp_toolbox_b200 import composite
from oracle import dgp_oracle as O

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=7)
ap.add_argument("--iters", type=int, default=10)
ap.add_argument("--arms", default="fused,torch_k,per_sample")
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("bench_fused_full_cov.py needs a CUDA device")
SHAPES = {"c4": dict(din=4, M=256, S=10, N=768), "c5": dict(din=8, M=256, S=8, N=512)}
dev = torch.device("cuda:0")


def make(din, M, S, N):
    rng = np.random.default_rng(0)
    Z = rng.uniform(0, 1, (M, din))
    kern = D.SquaredExponential(variance=1.0, lengthscales=np.full(din, 0.5))
    layer = D.SVGP_Layer(kern, Z, 1, D.Zero())
    layer.q_mu.assign(0.1 * rng.standard_normal((M, 1)))
    layer.q_sqrt.assign(0.5 * np.eye(M)[None] + 0.01 * np.tril(rng.standard_normal((1, M, M))))
    X = torch.as_tensor(rng.uniform(0, 1, (S, N, din)), device=dev)
    z = torch.as_tensor(rng.standard_normal((S, N, 1)), device=dev)
    return layer, X, z


def arms(layer, X, z):
    S, N, din = X.shape
    Zd = layer.feature.Z.value
    ls, var = layer.kern.lengthscales_vector(din), layer.kern.variance.value.reshape(())
    eye = torch.eye(Zd.shape[0], dtype=torch.float64, device=dev)

    def fused():
        return layer.sample_from_conditional(X, z=z, full_cov=True)

    def torch_k():
        Ku = O.kernel_K(Zd, None, ls, var) + O.JITTER * eye
        Kuf = O.kernel_K(Zd, X.reshape(S * N, din), ls, var)
        Kff = torch.stack([O.kernel_K(x, None, ls, var) for x in X])
        return composite.svgp_from_k_full_cov(Ku, Kuf, Kff, layer.q_mu.value, layer.q_sqrt.value, z, O.JITTER)

    def per_sample():
        outs = [layer._propagate_full(X[s].contiguous(), 1, [z[s:s + 1].contiguous()], 0) for s in range(S)]
        return tuple(torch.cat([o[k] for o in outs]) for k in range(3))

    return {"fused": fused, "torch_k": torch_k, "per_sample": per_sample}


def rel(a, b):
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-300))


try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                         text=True, timeout=30).stdout.strip()
except Exception:
    smi = torch.cuda.get_device_name(0)
names = args.arms.split(",")
for key, shp in SHAPES.items():
    layer, X, z = make(shp["din"], shp["M"], shp["S"], shp["N"])
    fns = {k: v for k, v in arms(layer, X, z).items() if k in names}
    with torch.no_grad():
        outs = {k: f() for k, f in fns.items()}
        for _ in range(2):
            for f in fns.values():
                f()
        torch.cuda.synchronize()
        times = {k: [] for k in fns}
        for _ in range(args.reps):
            for k, f in fns.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.iters):
                    f()
                e1.record()
                torch.cuda.synchronize()
                times[k].append(e0.elapsed_time(e1) / args.iters)
    ref = outs[names[0]]
    diff = {k: {"F": rel(o[0], ref[0]), "mean": rel(o[1], ref[1]), "cov": rel(o[2], ref[2])} for k, o in outs.items() if k != names[0]}
    print(json.dumps({"metric": f"{key}: one-layer full_cov=True ms per call", "unit": "ms", "gpu": smi,
                      "ms": {k: {"median": float(np.median(t)), "min": min(t), "max": max(t)} for k, t in times.items()},
                      "rel_diff_from_" + names[0]: diff,
                      "config": {"workload": f"RBF SVGP layer, D_in={shp['din']}, M={shp['M']}, D_out=1, S={shp['S']}, N={shp['N']}, "
                                             f"per-sample inputs, float64", "reps": args.reps, "iters": args.iters}}), flush=True)
