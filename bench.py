#!/usr/bin/env python
"""Benchmark of the DGP hot path: ELBO + gradient point-samples/s on BASELINE.json's config 2
(3-layer DGP = 4 SVGP layers, ARD-RBF, D=8, M=256 inducing points, S=32 Monte-Carlo samples, float64).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA through the C ABI)
    python bench.py --impl reference --gpus N --steps K ...  # reference arm: the reference's CPU algorithm on host cores
    python bench.py --gpus 1 --steps K --dump-outputs DIR    # also write the last timed step's result to DIR/*.npy

One step = one ELBO+gradient evaluation over one minibatch of N_b points per GPU (weak scaling: every rank owns N_b
points x S samples) followed, for N > 1, by ONE NCCL sum-allreduce of the flat [ELBO terms, gradients] buffer.
`value` times device-resident inputs; `e2e` times the host-buffer entry point (H2D of the minibatch, D2H of the result).
Prints ONE JSON line on rank 0.

The inputs (parameters, minibatches, Philox seeds) depend only on the arguments, so two builds run with the same arguments
can be compared output for output through --dump-outputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "DGP ELBO+grad point-samples/s"
UNIT = "point-samples/s"
FP64_PEAK_FALLBACK_TFLOPS = 37.07   # profiles/r0*_fp64_peaks.json (DMMA.8x8x4 register-resident loop, this pool's B200)
DUMP_LIMIT_BYTES = 64 << 20
N_POOL = 4   # distinct minibatches cycled through (fresh X, Y every step)


def step_inputs(i, nb, world=1, rank=0):
    """Inputs of timed step i on `rank` besides the model: the synthetic.minibatch index of its nb points (pool entry
    i % N_POOL), the global index of its first point (Philox counters), the ELBO scale (N = 1M points behind the
    minibatch, BASELINE config 2) and the Philox seed."""
    return {"batch": (i % N_POOL) * world + rank, "n_offset": (i * world + rank) * nb, "scale": 1.0e6 / (nb * world),
            "seed": 1234 + i}


def step_outputs(model, flat):
    """The flat [data term, KL, gradients] buffer of one step as named float64 arrays, gradients named like
    DGP_Base.ELBO_and_grads."""
    flat = flat.detach().cpu()
    names = {model.likelihood.likelihood.variance: "grad_lik_var"}
    for i, l in enumerate(model.layers):
        for key, p in (("Z", l.feature.Z), ("lengthscales", l.kern.lengthscales), ("variance", l.kern.variance),
                       ("q_mu", l.q_mu), ("q_sqrt", l.q_sqrt)):
            names[p] = f"grad_layers.{i}.{key}"
    out = {"data_term": flat[0], "kl": flat[1], "elbo": flat[0] - flat[1]}
    out.update({names[p]: g for p, g in model.unpack_grads(flat).items()})
    return {k: v.numpy().astype("float64") for k, v in out.items()}


def dump_outputs(directory, arrays, limit=DUMP_LIMIT_BYTES):
    """Writes every array as directory/<name>.npy in float64. When they add up to more than `limit` bytes, an array larger
    than an equal share of the limit is replaced by a fixed, seeded sample of its flattened entries (sorted positions), the
    same positions for the same shapes on every run."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    cap = None if sum(a.size for a in arrays.values()) * 8 <= limit else limit // 8 // len(arrays)
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64)
        if cap is not None and a.size > cap:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))]
        np.save(os.path.join(directory, name + ".npy"), a)


def load_synthetic(package):
    """The numpy-only module with the benchmark configurations and flop counts. Our arm imports it as part of the package;
    the reference arm must not import `dgp_toolbox_b200` (its __init__ maps libdgp_b200.so into the process), so there the
    file is loaded by path under another name."""
    if package:
        from dgp_toolbox_b200 import synthetic
        return synthetic
    import importlib.util
    spec = importlib.util.spec_from_file_location("_bench_synthetic", os.path.join(ROOT, "dgp_toolbox_b200", "synthetic.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def load_traffic():
    """Measured DRAM bytes per launch of the dominant kernels (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum),
    read from the profile summary committed with this build (profiles/r02_traffic.json, taken from the summaries tools/ncu_round.sh
    writes for the SAME bench command; its header names the commit). No file -> traffic stays null: never a pasted literal."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def fp64_peak():
    """MEASURED_PEAKS.json has no FP64 figure (bf16 + HBM only), so the denominator is this repo's own calibration
    (tools/fp64_peaks.cu run on this pool's B200, committed as profiles/r01_fp64_peaks.json)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_fp64_peaks.json")) as f:
            return float(json.load(f)["summary"]["fp64_dmma_tflops"]), ("profiles/r02_fp64_peaks.json (own DMMA calibration, tools/fp64_peaks.cu; "
                                                                        "MEASURED_PEAKS.json has no FP64 entry; DMMA and DFMA share the pipe, so this is the ceiling)")
    except Exception:
        return FP64_PEAK_FALLBACK_TFLOPS, "fallback constant (own r01 DMMA calibration)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def cpu_reference_throughput(cfg, nb_cpu, steps, warmup):
    """The reference's CPU algorithm for the path: TensorFlow/GPflow are not installable here (no network, absent from the
    image), so this is the op-for-op float64 restatement in oracle/ (kind = "port"), run on all host cores."""
    import torch
    from oracle import dgp_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    prob = O.synthetic_problem(cfg["D0"], cfg["num_units"], cfg["M"], nb_cpu)
    om = O.model_from_problem(prob, cfg["S"])
    g = torch.Generator().manual_seed(0)
    zs = [torch.randn(cfg["S"], nb_cpu, l.D_out, dtype=torch.float64, generator=g) for l in om.layers]
    X, Y = torch.as_tensor(prob["X"]), torch.as_tensor(prob["Y"])
    for _ in range(warmup):
        O.elbo_and_grads(om, X, Y, zs)
    t0 = time.perf_counter()
    for _ in range(steps):
        O.elbo_and_grads(om, X, Y, zs)
    dt = (time.perf_counter() - t0) / steps
    return nb_cpu * cfg["S"] / dt, dt, cores


def cpu_forward_baseline(kind, cfg, n_cpu, reps=3):
    """CPU leg of the forward-only configurations (oracle port on all host cores, bounded sample): kind "predict" = DGP.predict
    (models/dgp.py:362-366); kind "acq" = EI.run analytic + exact EHVI over two DGPs (Infill_criteria.py:36-52, EHVI.py:107-157)."""
    import numpy as np
    import torch
    from oracle import dgp_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    S = cfg["S"]
    probs = [O.synthetic_problem(cfg["D0"], cfg["num_units"], cfg["M"], n_cpu, seed_shift=k) for k in ((0,) if kind == "predict" else (0, 100))]
    oms = [O.model_from_problem(p, S) for p in probs]
    X = torch.as_tensor(probs[0]["X"])
    g = torch.Generator().manual_seed(0)
    zss = [[torch.randn(S, n_cpu, l.D_out, dtype=torch.float64, generator=g) for l in om.layers] for om in oms]
    y0 = np.linspace(0.95, 0.05, 32)
    ynd = O.Y_ND(y0, 1.0 - np.sqrt(y0), (1.1, 1.1), (-0.1, -0.1))

    def once():
        with torch.no_grad():
            if kind == "predict":
                O.predict(oms[0], X, S, zss[0])
            else:
                mom = []
                for om, zs in zip(oms, zss):
                    _, Fm, Fv = O.propagate(om.layers, X, S, zs)
                    mom += list(O.mixture_moments(Fm[-1], Fv[-1]))
                    if om is oms[0]:
                        O.ei_analytic(Fm[-1], Fv[-1], 0.0)
                O.ehvi_exact(*mom, ynd[0], ynd[1])
    once()
    t0 = time.perf_counter()
    for _ in range(reps):
        once()
    return (time.perf_counter() - t0) / reps, cores


def forward_extras(D, synthetic, torch, steps, peak, with_cpu):
    """BASELINE configs 3 and 5 (forward-only paths; one GPU): device-resident rate, the same through HOST buffers (H2D of the
    candidates and D2H of the results inside the timed region), the useful FP64 rate against the peak, and the CPU port on a bounded
    sample. These ride in `extra.configs` of the JSON line; the headline metric stays config 2."""
    import numpy as np
    out = {}

    def timed(fn, k, w=2):
        for i in range(w):
            fn(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(k):
            fn(w + i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / k

    # ---- config 3: 5-layer DGP (6 SVGP layers), D = 20, M = 512, S = 64: predict (predict_y mixture moments), chunks of 8192 points ----
    cfg = synthetic.CONFIGS["c3"]
    nb3 = 8192
    model = synthetic.model_from_problem(synthetic.synthetic_problem(cfg["D0"], cfg["num_units"], cfg["M"], 8), cfg["S"])
    host = [torch.from_numpy(synthetic.minibatch(cfg["D0"], nb3, 40 + i)[0]).pin_memory() for i in range(3)]
    dev = [h.cuda() for h in host]
    res_host = [torch.empty((nb3, 1), dtype=torch.float64).pin_memory() for _ in range(2)]
    ms = timed(lambda i: model.predict_moments(dev[i % 3], cfg["S"], seed=100 + i), steps)

    def predict_host(i):
        x = host[i % 3].to("cuda", non_blocking=True)
        m, v = model.predict_moments(x, cfg["S"], seed=100 + i)
        res_host[0].copy_(m, non_blocking=True); res_host[1].copy_(v, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    ms_h = timed(predict_host, steps)
    D._lib.get_context(0).check()
    f_fwd, _ = synthetic.flops_per_point_sample(cfg["D0"], cfg["num_units"], cfg["M"], S=cfg["S"])
    ps = nb3 * cfg["S"]
    ach = f_fwd * ps / (ms * 1e-3) / 1e12
    out["c3_predict"] = {
        "metric": "DGP predict point-samples/s", "value": ps / (ms * 1e-3), "unit": "point-samples/s", "ms_per_step": ms,
        "config": {"workload": "5-layer DGP (6 SVGP layers), D=20, M=512, S=64, predict (predict_y mixture moments), float64; one step = one "
                               "8192-point chunk of the N = 10 M sweep", "points_per_step": nb3, "samples": cfg["S"]},
        "roofline": {"bound": "tensor", "kernel": "dgp::fused_forward_kernel", "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                     "frac": ach / peak, "algorithmic_flops_per_point_sample": f_fwd, "traffic": None},
        "e2e": {"value": ps / (ms_h * 1e-3), "unit": "point-samples/s", "ms_per_step": ms_h, "h2d_bytes_per_step": nb3 * cfg["D0"] * 8,
                "d2h_bytes_per_step": nb3 * 2 * 8}}
    if with_cpu:
        dt, cores = cpu_forward_baseline("predict", cfg, 64)
        out["c3_predict"]["cpu_baseline"] = {"value": 64 * cfg["S"] / dt, "unit": "point-samples/s", "cores": cores, "kind": "port",
                                             "sample": f"64 points x S={cfg['S']} samples per pass ({dt:.2f} s/pass)"}
    del model, dev
    torch.cuda.empty_cache()

    # ---- config 5: EI (analytic) + exact 2-objective EHVI, two 3-layer DGPs (D = 8, M = 256), S = 32, chunks of 16384 candidates ----
    cfg = synthetic.CONFIGS["c2"]
    nb5 = 16384
    m0 = synthetic.model_from_problem(synthetic.synthetic_problem(cfg["D0"], cfg["num_units"], cfg["M"], 8), cfg["S"])
    m1 = synthetic.model_from_problem(synthetic.synthetic_problem(cfg["D0"], cfg["num_units"], cfg["M"], 8, seed_shift=100), cfg["S"])
    host = [torch.from_numpy(synthetic.minibatch(cfg["D0"], nb5, 60 + i)[0]).pin_memory() for i in range(3)]
    dev = [h.cuda() for h in host]
    y0 = np.linspace(0.95, 0.05, 32)
    ynd = D.Y_ND([y0, 1.0 - np.sqrt(y0)], np.arange(32), nadir=(1.1, 1.1), ideal=(-0.1, -0.1))
    ms = timed(lambda i: D.EI_and_EHVI([m0, m1], dev[i % 3], ynd, 0.0, S=cfg["S"], seed=[i, 1000 + i]), steps)
    res_host = [torch.empty((nb5, 1), dtype=torch.float64).pin_memory() for _ in range(2)]

    def acq_host(i):
        x = host[i % 3].to("cuda", non_blocking=True)
        ei, eh = D.EI_and_EHVI([m0, m1], x, ynd, 0.0, S=cfg["S"], seed=[i, 1000 + i])
        res_host[0].copy_(ei, non_blocking=True); res_host[1].copy_(eh, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    ms_h = timed(acq_host, steps)
    D._lib.get_context(0).check()
    f_fwd, _ = synthetic.flops_per_point_sample(cfg["D0"], cfg["num_units"], cfg["M"], S=cfg["S"])
    flops = 2 * f_fwd * nb5 * cfg["S"]     # one propagation per model and candidate (model 0's moments serve EI and EHVI)
    ach = flops / (ms * 1e-3) / 1e12
    out["c5_ei_ehvi"] = {
        "metric": "DGP EI+EHVI candidates/s", "value": nb5 / (ms * 1e-3), "unit": "candidates/s", "ms_per_step": ms,
        "config": {"workload": "EI (analytic) + exact 2-objective EHVI, two 3-layer DGPs (D=8, M=256), S=32, 32-point Pareto front, float64; "
                               "one step = one 16384-candidate chunk of the 4 M sweep; model 0 is propagated once for both criteria",
                   "candidates_per_step": nb5, "samples": cfg["S"]},
        "roofline": {"bound": "tensor", "kernel": "dgp::fused_forward_kernel", "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                     "frac": ach / peak, "traffic": None},
        "e2e": {"value": nb5 / (ms_h * 1e-3), "unit": "candidates/s", "ms_per_step": ms_h, "h2d_bytes_per_step": nb5 * cfg["D0"] * 8,
                "d2h_bytes_per_step": nb5 * 2 * 8}}
    if with_cpu:
        dt, cores = cpu_forward_baseline("acq", cfg, 128)
        out["c5_ei_ehvi"]["cpu_baseline"] = {"value": 128 / dt, "unit": "candidates/s", "cores": cores, "kind": "port",
                                             "sample": f"128 candidates x S={cfg['S']} samples, two models, per pass ({dt:.2f} s/pass)"}
    del m0, m1, dev
    torch.cuda.empty_cache()

    # ---- config 4: multi-fidelity DGP with embedded mapping (MF_DGP_EM.py), 3 fidelities (input spaces of 2, 3, 4 dimensions), M = 256,
    # ELBO + every gradient on one minibatch of the N = 500 k data set (the full data set in one evaluation would need the [S, N] planes
    # of 50 M point-samples; the reference has no minibatching either) ----
    from dgp_toolbox_b200.models import MF_DGP_EM
    rng = np.random.default_rng(0)
    dims, n4, S4 = [2, 3, 4], [32768, 8192, 2048], 10
    f4 = lambda x: np.sin(3 * x[:, :1]) + 0.5 * x[:, 1:2]
    X = [rng.uniform(0, 1, (n, d)) for n, d in zip(n4, dims)]
    Y = [f4(X[0]), 1.2 * f4(X[1]) + 0.3 * X[1][:, :1] ** 2, 1.5 * f4(X[2]) - 0.2 * X[2][:, 1:2]]
    em = MF_DGP_EM.DGP_Base.make_mf_dgp(X, [rng.uniform(0, 1, (256, d)) for d in dims], [rng.uniform(0, 1, (256, 4)), rng.uniform(0, 1, (256, 3))])
    em.num_samples = S4
    Xh = [torch.from_numpy(x).pin_memory() for x in X + Y + [X[1][:, :2].copy(), X[2][:, :2].copy()]]
    to_dev = lambda: [h.to("cuda", non_blocking=True) for h in Xh]
    d4 = to_dev()
    params = em.trainable_parameters
    ms = timed(lambda i: em.ELBO_and_grads((d4[0:3], d4[3:6], d4[6:8]), params), steps, w=1)

    def em_host(i):
        d = to_dev()
        elbo, grads = em.ELBO_and_grads((d[0:3], d[3:6], d[6:8]), params)
        torch.cat([elbo.reshape(1)] + [grads[p].reshape(-1) for p in params]).cpu()
    ms_h = timed(em_host, steps, w=1)
    ps4 = sum(n4) * S4
    out["c4_mf_dgp_em"] = {
        "metric": "MF-DGP-EM ELBO+grad point-samples/s", "value": ps4 / (ms * 1e-3), "unit": "point-samples/s", "ms_per_step": ms,
        "config": {"workload": "multi-fidelity DGP with embedded mapping (MF_DGP_EM.py), 3 fidelities with 2/3/4-D inputs, M=256, S=10, one "
                               "minibatch of 32768 / 8192 / 2048 points per fidelity, ELBO + every gradient, float64", "point_samples_per_step": ps4},
        "roofline": None,
        "e2e": {"value": ps4 / (ms_h * 1e-3), "unit": "point-samples/s", "ms_per_step": ms_h,
                "h2d_bytes_per_step": int(sum(h.numel() for h in Xh) * 8), "d2h_bytes_per_step": int(sum(p.value.numel() for p in params) * 8 + 8)},
        "cpu_baseline": None,
        "note": "composite-kernel layers run the unfused GEMM pipeline on supplied kernel matrices (DESIGN.md §6); no CPU port of this model "
                "exists in oracle/ (parity is against the reference's own MF_DGP_EM.py executed under tests/ref_shim, tests/golden/mf_dgp_em.npz)"}
    del em, d4
    torch.cuda.empty_cache()

    # ---- config 5 through the multi-objective DGP object (MO_DGP.py; EHVI.py:124-130 `mo_dgp` branch): two composite-kernel layers,
    # loop = 2 (6 layer applications per chain), both objectives' moments from ONE chain, exact EHVI; chunks of 16384 candidates ----
    import types
    from dgp_toolbox_b200.models import MO_DGP
    rng = np.random.default_rng(0)
    g0 = lambda x: np.sin(3 * x[:, :1]) + 0.5 * x[:, 1:2]
    g1 = lambda x: np.cos(2 * x[:, :1]) * x[:, 1:2] - 0.3
    Zx = rng.uniform(0, 1, (256, 8))
    mo = MO_DGP.DGP_Base.make_mf_dgp([np.concatenate([Zx, g1(Zx)], 1), Zx.copy()], loop=2)
    mo.layers[0].kern.kernels[-1].variance.assign(1e-2)
    for k5, layer in enumerate(mo.layers):
        layer.q_mu.assign((g0, g1)[k5](Zx) + 0.05 * rng.standard_normal((256, 1)))
        layer.q_sqrt.assign(0.1 * layer.q_sqrt.value)
    obj = types.SimpleNamespace(name="mo_dgp", model=mo, _X=[Zx, Zx])
    host = [torch.from_numpy(rng.uniform(0, 1, (nb5, 8))).pin_memory() for i in range(3)]
    dev = [h.cuda() for h in host]
    ms = timed(lambda i: D.EHVI(obj, dev[i % 3], ynd, S=32), steps)
    res_mo = torch.empty((nb5, 1), dtype=torch.float64).pin_memory()

    def mo_host(i):
        x = host[i % 3].to("cuda", non_blocking=True)
        res_mo.copy_(D.EHVI(obj, x, ynd, S=32), non_blocking=True)
        torch.cuda.current_stream().synchronize()
    ms_h = timed(mo_host, steps)
    D._lib.get_context(0).check()
    out["c5_mo_dgp_ehvi"] = {
        "metric": "MO-DGP EHVI candidates/s", "value": nb5 / (ms * 1e-3), "unit": "candidates/s", "ms_per_step": ms,
        "config": {"workload": "exact 2-objective EHVI through the multi-objective DGP object (MO_DGP.py: 2 composite-kernel layers, D=8, M=256, "
                               "loop=2 = 6 layer applications per chain), S=32, 32-point Pareto front, float64; one step = one 16384-candidate chunk",
                   "candidates_per_step": nb5, "samples": 32},
        "roofline": None,
        "e2e": {"value": nb5 / (ms_h * 1e-3), "unit": "candidates/s", "ms_per_step": ms_h, "h2d_bytes_per_step": nb5 * 8 * 8,
                "d2h_bytes_per_step": nb5 * 8},
        "cpu_baseline": None,
        "note": "composite-kernel layers run the unfused GEMM pipeline on supplied kernel matrices (DESIGN.md §6); parity is against the "
                "reference's own MO_DGP.py / EHVI.py executed under tests/ref_shim (tests/golden/mo_dgp.npz)"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2")
    ap.add_argument("--nb", type=int, default=16384, help="minibatch points per GPU per step")
    ap.add_argument("--nb-cpu", type=int, default=512, help="points of the bounded CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip extra.configs (configs 3 and 5) and extra.strong_scaling")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the ELBO terms and gradients of the last timed step (rank 0) "
                    "as DIR/<name>.npy, float64, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)

    synthetic = load_synthetic(package=args.impl == "ours")
    cfg = synthetic.CONFIGS[args.config]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    f_fwd_ref, f_step_ref = synthetic.flops_per_point_sample(cfg["D0"], cfg["num_units"], cfg["M"])            # reference formulation
    f_fwd, f_step = synthetic.flops_per_point_sample(cfg["D0"], cfg["num_units"], cfg["M"], S=cfg["S"])      # V-form + first-layer sharing
    workload = (f"{len(cfg['num_units'])}-layer DGP ({len(cfg['num_units']) + 1} SVGP layers), ARD-RBF, D={cfg['D0']}, "
                f"M={cfg['M']}, S={cfg['S']}, minibatch ELBO+grad, float64")

    if args.impl == "reference":
        if rank != 0:
            return
        val, dt, cores = cpu_reference_throughput(cfg, args.nb_cpu, args.steps, warmup)
        sample = f"N_b={args.nb_cpu} points x S={cfg['S']} samples per step (reference formulation materialises [D_out,M,S*N] twice)"
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload, "points_per_step": args.nb_cpu, "samples": cfg["S"]},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "TensorFlow/GPflow absent from the image: oracle/ float64 torch-CPU restatement of the reference op sequence",
        }))
        assert "dgp_toolbox_b200" not in sys.modules, "the reference arm must not load the product library"
        return

    import torch
    import torch.distributed as dist
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"   # keep NCCL's version banner off stdout: rank 0 prints exactly one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    import dgp_toolbox_b200 as D
    from dgp_toolbox_b200.distributed import ShardedELBO

    ctx = D._lib.get_context(local_rank)
    ctx.set_workspace_limit(64 << 30)
    prob = synthetic.synthetic_problem(cfg["D0"], cfg["num_units"], cfg["M"], 8)
    model = synthetic.model_from_problem(prob, cfg["S"])
    sharded = ShardedELBO(model)
    nb, S = args.nb, cfg["S"]
    pool_host = []
    for i in range(N_POOL):
        X, Y = synthetic.minibatch(cfg["D0"], nb, step_inputs(i, nb, world, rank)["batch"])
        pool_host.append((torch.from_numpy(X).pin_memory(), torch.from_numpy(Y).pin_memory()))
    pool_dev = [(x.cuda(), y.cuda()) for x, y in pool_host]

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def step_dev(i):
        X, Y = pool_dev[i % N_POOL]
        s = step_inputs(i, nb, world, rank)
        return sharded.step(X, Y, n_offset=s["n_offset"], scale=s["scale"], seed=s["seed"])

    def step_host(i):
        X, Y = pool_host[i % N_POOL]
        s = step_inputs(i, nb, world, rank)
        return sharded.step_host(X, Y, n_offset=s["n_offset"], scale=s["scale"], seed=s["seed"])

    def timed(fn, k):
        import gc
        gc.collect()
        gc.disable()       # a collector pause between launches shows up as GPU idle time in a region of only k steps
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(k):
            out = fn(i)
        e1.record()
        sync_all()
        gc.enable()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    for i in range(warmup):
        step_dev(i)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ctx.launch_count(reset=True)
    ms_total, out = timed(step_dev, args.steps)
    launches = ctx.launch_count(reset=True)
    clocks = sampler.stop() if rank == 0 else None
    elbo = float((out[0] - out[1]).item())
    # Kernel durations for the roofline: the same K steps once more with a CUDA-event pair around every launch. The library
    # keeps all launches on one stream while it profiles (in the timed region above the parameter contractions of a layer run
    # side by side and overlap the next layer's data path, so an event pair there would time the sharing of the SMs, not the
    # kernel); `ms_per_step` / `value` come from the unprofiled region.
    ctx.get_profile(reset=True)
    ctx.set_profiling(True)
    ms_profiled, _ = timed(step_dev, args.steps)
    prof = ctx.get_profile(reset=True)
    ctx.set_profiling(False)

    for i in range(warmup):
        step_host(i)
    ms_e2e, _ = timed(step_host, args.steps)

    # ---- strong scaling: the SAME 16384-point minibatch split over the ranks (north_star: "minibatch points x samples shard across
    # the GPUs"); at N = 1 this is the headline measurement itself ----
    strong = None
    if world > 1 and not args.no_extras:
        from dgp_toolbox_b200.distributed import shard_bounds
        lo, hi = shard_bounds(nb, rank, world)
        sscale = 1.0e6 / nb

        def step_strong(i):
            X, Y = pool_dev[i % N_POOL]
            return sharded.step(X[lo:hi], Y[lo:hi], n_offset=i * nb + lo, scale=sscale, seed=1234 + i)
        for i in range(warmup):
            step_strong(i)
        ms_strong, _ = timed(step_strong, args.steps)
        strong = {"points_per_step_total": nb, "points_per_gpu": hi - lo, "ms_per_step": ms_strong / args.steps,
                  "value": nb * S / (ms_strong / args.steps * 1e-3), "unit": UNIT,
                  "note": "efficiency = (ms_per_step of the N = 1 run) / (N x this ms_per_step); replicated per-step work "
                          "(Kuu, Cholesky, operator packing, KL and its adjoint) and the allreduce do not shrink with N"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, step_outputs(model, out))

    ps_per_step = nb * S * world
    ms_step = ms_total / args.steps
    value = ps_per_step / (ms_step * 1e-3)
    e2e_value = ps_per_step / (ms_e2e / args.steps * 1e-3)
    # Two kernels carry the step: the fused conditional kernel (forward, F_fwd flops per point-sample) and the DMMA GEMM
    # engine (adjoint contractions, 2 F_fwd). `roofline` describes the one with the larger share of the timed region,
    # `roofline.other_kernels` the other; both from CUDA-event pairs recorded on the launching stream during the profiled pass.
    peak, peak_src = fp64_peak()
    all_ms = sum(v[0] for v in prof.values())
    n_grad, _ = model.grad_layout()

    def kernel_entry(name, cats, flops_per_ps, traffic=None):
        ms = sum(prof[k][0] for k in cats)
        n = sum(prof[k][1] for k in cats)
        ach = flops_per_ps * nb * S * args.steps / (ms * 1e-3) / 1e12 if ms > 0 else 0.0
        return {"kernel": name, "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                "traffic": traffic, "algorithmic_flops_per_point_sample": flops_per_ps, "launches_in_region": n,
                "kernel_ms_per_step": ms / args.steps, "share_of_step": ms / all_ms if all_ms > 0 else None}

    fwd_cats = [k for k in ("fused_fwd", "gemm_fwd") if prof[k][0] > 0]
    traffic = load_traffic()
    k_fwd = kernel_entry("dgp::fused_forward_kernel (Kuf tile -> V = Lu^-1 Kuf -> T_d = (q_sqrt_d^T Lu^-T) V -> moments/sample, FP64 DMMA, "
                         "bulk-copy (UBLKCP) operand ring)" if prof["fused_fwd"][0] > 0 else "dgp::gemm_kernel (forward contractions)",
                         fwd_cats, f_fwd, traffic=traffic.get("fused_forward_kernel"))
    # adjoint = data path (fused_backward_kernel, or the unfused GEMMs + rbf_bwd when DGP_B200_FUSED_BWD=0) + parameter contractions;
    # algorithmic flops: F_fwd each (SURVEY §9: the adjoint is exactly twice the forward)
    data_cats = [k for k in ("fused_bwd", "gemm_bwd_data", "rbf_bwd") if prof[k][0] > 0]
    k_data = kernel_entry("dgp::fused_backward_kernel (dV = sum_d C_d^T (2Gv_d o T_d) + ..., K-bar = Lu^-T dV, kernel adjoint on resident "
                          "tiles; panels + T_d slabs through one bulk-copy ring, FP64 DMMA)" if prof["fused_bwd"][0] > 0
                          else "dgp::gemm_kernel + rbf_bwd_kernel (unfused data adjoint)", data_cats, f_fwd,
                          traffic=traffic.get("fused_backward_kernel"))
    f_param = synthetic.param_flops_per_point_sample(cfg["D0"], cfg["num_units"], cfg["M"], cfg["S"])
    f_step = 2 * f_fwd + f_param   # forward + data adjoint + parameter contractions (W-form: D_out instead of 1 + D_out products)
    k_param = kernel_entry("dgp::gemm_kernel (FP64 DMMA contractions over the point-samples: tril(V diag(2Gv_d) V^T) per output, "
                           "V Gm, Gbar [X,1])", ["gemm_bwd_param"], f_param, traffic=traffic.get("gemm_kernel_param"))
    kernels = sorted([k_fwd, k_data, k_param], key=lambda k: -k["kernel_ms_per_step"])
    main, others = kernels[0], kernels[1:]
    flops_rank_step = f_step * nb * S
    roofline = dict(main)
    roofline.update({
        "peak_source": peak_src,
        "whole_step_frac": flops_rank_step / (ms_step * 1e-3) / 1e12 / peak,
        "reference_formulation": {
            "flops_per_point_sample": f_step_ref,
            "note": "the reference tiles X over the S samples, evaluates the first layer S times per point (models/dgp.py:49) and forms "
                    "A = Ku^-1 Kuf explicitly (utils/layers.py:245-247); this implementation evaluates the first layer once per point "
                    "and folds q_sqrt_d^T Lu^-T once per step (V-form, no A pass) - identical results - so the kernels need "
                    f"{f_step:.0f} flops per point-sample instead of {f_step_ref}. `achieved`/`frac` use the smaller figure "
                    "(work the kernels actually have to do); this entry says what rate the reference's formulation would need "
                    "for the same throughput.",
            "equivalent_tflops": f_step_ref * nb * S / (ms_step * 1e-3) / 1e12},
        "other_kernels": others,
        "traffic_source": traffic.get("source"),
        "categories_ms_per_step": {k: v[0] / args.steps for k, v in prof.items()},
        "profiled_pass_ms_per_step": ms_profiled / args.steps,
        "note": "achieved = algorithmic (triangular-aware, useful) FP64 flops of SURVEY.md §8d / CUDA-event time of the kernel's launches, "
                "taken in a second pass over the same steps with every launch on one stream (profiled_pass_ms_per_step; the timed "
                "region overlaps kernels across streams, so its step time is shorter than the sum of the kernel times); "
                "ncu pipe utilisation (executed work) is in profiles/",
    })
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": workload, "points_per_gpu_per_step": nb, "samples": S, "point_samples_per_step": ps_per_step,
                   "parallelism": f"dp{world} (points sharded, parameters replicated, one allreduce of {n_grad} doubles)",
                   "l2": "per-step working set (stashed A/T tiles, >30 GB) far exceeds the 126 MB L2; a different minibatch every step"},
        "roofline": roofline,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": world * nb * (cfg["D0"] + 1) * 8,
                "d2h_bytes_per_step": n_grad * 8, "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches,
        "clocks": clocks,
        "elbo_last_step": elbo,
    }
    if world == 1 and not args.no_cpu_baseline:
        val, dt, cores = cpu_reference_throughput(cfg, args.nb_cpu, 10, 2)
        line["cpu_baseline"] = {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"N_b={args.nb_cpu} points x S={S} samples, 10 steps after 2 warm-ups ({dt:.2f} s/step)"}
    extra = {}
    if strong is not None:
        strong["efficiency_vs_weak_step"] = ms_step / (world * strong["ms_per_step"])
        extra["strong_scaling"] = strong
    if world == 1 and not args.no_extras:
        del pool_dev, sharded, model
        torch.cuda.empty_cache()
        extra["configs"] = forward_extras(D, synthetic, torch, args.steps, peak, not args.no_cpu_baseline)
        extra["fp64_pipe"] = {"dmma_dfma_co_issue": False, "source": "profiles/r02_fp64_peaks.json (tools/fp64_peaks.cu: DMMA-only 37.1, "
                              "DFMA-only 36.5, both in one warp 35.8, warp-specialised 36.4 TFLOP/s: one shared FP64 pipe, so the DMMA "
                              "peak is the ceiling of the kernels' mixed DMMA + DFMA instruction stream)"}
    if extra:
        line["extra"] = extra
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
