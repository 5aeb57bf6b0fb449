"""MultiFidelityDeepGP's predict_f(full_cov=True): 3 fidelities, M = 256 inducing points per layer, N = 768 test points (the
largest N the full-covariance path factorises), S = 250 samples (the model's `predict`). Every layer application is one
dgp_comp_K_blocks call for K(X_s, X_s), the dgp_comp_K calls for Kuu and Kuf, and one dgp_svgp_from_k_full_cov call. Prints one
JSON line: the time per predict_f call (CUDA events, profiling off) and, from a separate profiled call, the library's per-category
device time split (dgp_get_profile). Needs a GPU.
   python tools/bench_full_cov.py [--n 768] [--samples 250] [--m 256] [--din 4] [--reps 3]"""
import argparse, json, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import dgp_toolbox_b200 as D
from dgp_toolbox_b200.models import MF_DGP

ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, default=768)
ap.add_argument("--samples", type=int, default=250)
ap.add_argument("--m", type=int, default=256)
ap.add_argument("--din", type=int, default=4)
ap.add_argument("--reps", type=int, default=3)
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("bench_full_cov.py needs a CUDA device")
rng = np.random.default_rng(0)
Z = [rng.uniform(0, 1, (args.m, args.din)) for _ in range(3)]
model = MF_DGP.DGP_Base.make_mf_dgp(Z)
X = torch.as_tensor(rng.uniform(0, 1, (args.n, args.din))).cuda()
ctx = D._lib.get_context(0)


def run():
    with torch.no_grad():
        return model.predict_f(X, full_cov=True, S=args.samples)


run()                                   # warm-up: module load, arena growth
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(args.reps):
    m, v = run()
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / args.reps
ctx.get_profile(reset=True)
ctx.set_profiling(True)
run()
prof = ctx.get_profile(reset=True)
ctx.set_profiling(False)
try:
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                         text=True, timeout=30).stdout.strip()
except Exception:
    smi = torch.cuda.get_device_name(0)
print(json.dumps({"metric": "MF-DGP predict_f(full_cov=True) ms per call", "value": ms, "unit": "ms", "gpu": smi,
                  "profile_ms_launches": {k: [round(t, 3), n] for k, (t, n) in prof.items() if n},
                  "var_shape": list(v.shape), "finite": bool(torch.isfinite(v).all() and torch.isfinite(m).all()),
                  "config": {"workload": f"MF_DGP.DGP_Base.make_mf_dgp, 3 fidelities, D_in={args.din}, M={args.m}, N={args.n}, "
                                         f"S={args.samples}, full_cov=True, float64", "reps": args.reps}}))
