"""Batch expected improvement (q-EI) of G candidate batches of q points each, at two shapes:
  bo   a BO-sized DGP: D = 2, M = 50, 2 layers (2 -> 2 -> 1), G = 300, q = 4, S = 1000 (the reference's num_samples default)
  c2   a config-2-like stack: D = 8, M = 256, 3 layers (8 -> 8 -> 8 -> 1), G = 300, q = 8, S = 64
Arms (each one call of the criterion over all G batches, or what it takes without it):
  qei      qEI.run: one dgp_qei call (conditional per layer + one grouped_cov_kernel per layer + the q-EI reduction)
  loop     G propagate(full_cov=True) calls on q points each (n_offset = g q) plus a torch reduction: the way to get the same
           values without the grouped call
  dense    one propagate(full_cov=True) on G = 96 batches at once (N = 768, the dense path's limit): one (N x N) block per sample
           and output, which also correlates batches that should be independent (timing only)
plus one full qEI.optimize (popsize 300, 400 generations: 300 x 401 batch evaluations) at the bo shape.
Times are CUDA events around each arm, median / min / max over --reps repetitions, arms alternating; the GPU's name and power limit
are read in the same run. A separate profiled pass (torch.profiler, CUDA activity) of one qEI.run per shape splits the device time
into the conditional (fused / unfused conditional kernels and GEMMs), grouped_cov_kernel, and the rest. One JSON line per result.
Needs a GPU; --dry builds the inputs and stops before the first library call.
   python tools/bench_qei.py [--reps 5] [--shapes bo,c2] [--arms qei,loop,dense] [--no-optimize] [--dry]"""
import argparse, json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from oracle import dgp_oracle as O

SHAPES = {"bo": dict(D0=2, units=[2], M=50, G=300, q=4, S=1000), "c2": dict(D0=8, units=[8, 8], M=256, G=300, q=8, S=64)}
DENSE_G = 96

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--shapes", default="bo,c2")
ap.add_argument("--arms", default="qei,loop,dense")
ap.add_argument("--no-optimize", action="store_true")
ap.add_argument("--dry", action="store_true", help="build the inputs, then stop before the first library call")
args = ap.parse_args()
shapes = {k: SHAPES[k] for k in args.shapes.split(",")}
arm_names = args.arms.split(",")
for a in arm_names:
    if a not in ("qei", "loop", "dense"):
        sys.exit(f"unknown arm {a!r}")


def problem(D0, units, M, G, q, S):
    """Inputs of one shape (numpy): the synthetic problem's layers and G q candidate points in [-1, 1]^D0."""
    prob = O.synthetic_problem(D0, units, M, 64)
    X = np.random.default_rng(1).uniform(-1.0, 1.0, (G * q, D0))
    return prob, X, float(prob["Y"].min())


inputs = {k: problem(**s) for k, s in shapes.items()}
if args.dry:
    for k, (prob, X, y_min) in inputs.items():
        print(json.dumps({"shape": k, "X": list(X.shape), "layers": [l["Z"].shape[1] for l in prob["layers"]] + [1], "y_min": y_min,
                          **{n: shapes[k][n] for n in ("M", "G", "q", "S")}}))
    sys.exit(0)
if not torch.cuda.is_available():
    sys.exit("bench_qei.py needs a CUDA device")

import dgp_toolbox_b200 as D  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

dev = torch.device("cuda:0")


def build_model(prob, S):
    layers = []
    for l in prob["layers"]:
        mf = D.Zero() if l["mean_kind"] == "zero" else (D.Identity() if l["mean_kind"] == "identity" else D.Linear(l["mf_W"], l["mf_b"]))
        layer = D.SVGP_Layer(D.SquaredExponential(variance=l["variance"], lengthscales=l["lengthscales"]), l["Z"], l["q_mu"].shape[1], mf)
        layer.q_mu.assign(l["q_mu"])
        layer.q_sqrt.assign(l["q_sqrt"])
        layers.append(layer)
    return D.DGP_Base(D.Gaussian(prob["lik_var"]), layers, num_samples=S, seed=1)


def timed(fn, reps):
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1))
    return out


def stats(t):
    return {"median": float(np.median(t)), "min": float(min(t)), "max": float(max(t))}


try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                         text=True, timeout=30).stdout.strip()
except Exception:
    smi = torch.cuda.get_device_name(0)
ctx = D._lib.get_context(0)

for key, shp in shapes.items():
    prob, Xn, y_min = inputs[key]
    G, q, S = shp["G"], shp["q"], shp["S"]
    model = build_model(prob, S)
    X = torch.as_tensor(Xn, device=dev)
    crit = D.qEI(y_min, shp["D0"], q)
    out = torch.empty((G, 1), dtype=torch.float64, device=dev)

    def qei():
        return crit.run(model, X, num_samples=S, seed=3, out=out)

    def loop():
        vals = []
        for g in range(G):
            Fs, _, _ = model.propagate(X[g * q:(g + 1) * q], full_cov=True, S=S, seed=3, n_offset=g * q)
            vals.append(-torch.clamp(y_min - Fs[-1].amin(dim=1), min=0.0).mean(dim=0))
        return torch.stack(vals)

    Xd = X[:DENSE_G * q].contiguous()

    def dense():
        return model.propagate(Xd, full_cov=True, S=S, seed=3)

    fns = {"qei": qei, "loop": loop, "dense": dense}
    fns = {k: fns[k] for k in arm_names}
    with torch.no_grad():
        for f in fns.values():   # warm-up: module loads, arena growth
            f()
        torch.cuda.synchronize()
        ctx.check()
        agree = None
        if "loop" in fns:
            agree = float((qei() - loop()).abs().max() / loop().abs().max().clamp_min(1e-300))
        times = {k: [] for k in fns}
        for _ in range(args.reps):
            for k, f in fns.items():
                times[k] += timed(f, 1)
    print(json.dumps({"metric": f"{key}: ms per evaluation of {G} batches", "unit": "ms", "gpu": smi,
                      "ms": {k: stats(t) for k, t in times.items()}, "qei_vs_loop_rel_diff": agree,
                      "config": {"workload": f"DGP D={shp['D0']} layers={[shp['D0']] + shp['units'] + [1]} M={shp['M']} G={G} q={q} S={S}, "
                                             f"dense arm G={DENSE_G}", "reps": args.reps}}), flush=True)

    # profiled pass (separate from the timed ones): where one qEI.run spends its device time
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        qei()
        torch.cuda.synchronize()
    split = {"conditional": 0.0, "grouped_cov": 0.0, "other": 0.0}
    for e in prof.key_averages():
        us = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
        name = e.key
        if "grouped_cov_kernel" in name:
            split["grouped_cov"] += us / 1e3
        elif any(t in name for t in ("fused_forward_kernel", "kuf_kernel", "moments_kernel", "gemm")):
            split["conditional"] += us / 1e3
        else:
            split["other"] += us / 1e3
    total = sum(split.values())
    print(json.dumps({"metric": f"{key}: device-time split of one qEI.run (profiled pass)", "unit": "ms", "gpu": smi,
                      "ms": split, "grouped_cov_share": split["grouped_cov"] / total if total else None}), flush=True)

    if key == "bo" and not args.no_optimize:
        box = (np.full(shp["D0"], -1.0), np.full(shp["D0"], 1.0))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        x_opt = crit.optimize(model, box, popsize_DE=300, popstd_DE=1.5, iterations_DE=400, num_samples=S, seed=5)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        print(json.dumps({"metric": "bo: one qEI.optimize (popsize 300, 400 generations)", "unit": "s", "gpu": smi, "s": dt,
                          "generations": crit.de_iterations, "IC_optimized": float(crit.IC_optimized.sum()),
                          "x_opt": x_opt.tolist()}), flush=True)
