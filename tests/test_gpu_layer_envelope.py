"""The SVGP-DGP layer path across its whole supported envelope, against the float64 oracle (oracle/dgp_oracle.py).

Which kernel instantiation runs is decided at run time: pick_fused_cfg / pick_fused_bwd_cfg choose from shared-memory formulas,
forward_layer halves the point tile when a launch has few tiles (Pp / 64 <= num_sms / 2), layers with no fused configuration
run the unfused pipeline, and the adjoint takes the A-form or the V-form by point-sample count. Every case here runs under
torch.profiler and asserts the instantiations it exists to cover, so a change to those formulas cannot silently move a shape
onto a path nobody compares. Layers >= 1 run N * S = 10 000 point-samples (157 tiles of 64: above the halving threshold and
more than one persistent wave of 148 CTAs); the shared first layer runs N of them.

Tolerances keep the meaning of test_gpu_parity.py: 1e-9 relative to the un-cancelled scale for values, variances (relative to
sigma^2) and gradients; 1e-8 for samples through an N x N Cholesky, the EI input gradient and the natural-gradient step. Every
Kuu + jitter I has cond <= 2e3 (asserted), so 1e-9 sits above the conditioning noise floor of the float64 oracle."""
import itertools
import os
import subprocess
import sys
from collections import Counter

import numpy as np
import pytest
import torch
from torch.profiler import ProfilerActivity, profile

from oracle import dgp_oracle as O
from tests.helpers import _condition, oracle_zs, product_model_from_problem, rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-9
COND_MAX = 2e3
KINDS = ("rbf", "matern32", "matern52")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---------------------------------------------------------------------------------------------------------------------------
# builders and the profiler helper
# ---------------------------------------------------------------------------------------------------------------------------
def make_problem(dims, M, N, kernels, white, seed_shift=0):
    """dims = [D0, D1, ..., D_L]: one SVGP layer per consecutive pair. synthetic_problem's inputs and mean functions; a last
    width above 1 gets its own q_mu / q_sqrt and Y columns. Kuu of every layer is conditioned to cond <= COND_MAX (asserted)."""
    prob = O.synthetic_problem(dims[0], dims[1:-1], M, N, seed_shift=seed_shift)
    DL = dims[-1]
    if DL != 1:
        rng = np.random.default_rng(40 + seed_shift)
        last = prob["layers"][-1]
        last["q_mu"] = 0.1 * rng.standard_normal((M, DL))
        last["q_sqrt"] = 0.5 * np.eye(M)[None] + 0.05 * np.tril(rng.standard_normal((DL, M, M)))
        cols = np.arange(1, DL + 1) / DL
        prob["Y"] = np.sin(prob["X"].sum(1, keepdims=True) * cols) + 0.1 * rng.standard_normal((N, DL))
    for l, layer in enumerate(prob["layers"]):
        layer["kernel"] = kernels[l]
        layer["white"] = bool(white[l])
    prob = _condition(prob, COND_MAX)
    for layer in prob["layers"]:
        Ku = O.kernel_K(torch.as_tensor(layer["Z"]), None, torch.as_tensor(layer["lengthscales"]),
                        torch.tensor(float(layer["variance"])), layer["kernel"])
        assert float(torch.linalg.cond(Ku + O.JITTER * torch.eye(M, dtype=torch.float64))) <= COND_MAX
    return prob


def models(prob, S):
    return O.model_from_problem(prob, S), product_model_from_problem(prob, S)


def _norm(name):
    return name.replace(" ", "")


def launched(fn):
    """(fn(), Counter of the launched kernel names with spaces removed, e.g. 'voiddgp::fused_forward_kernel<64,64,2,4>(...)').
    CUPTI sees the library's own launches on every stream; the library's profiling mode is left off (it serialises the side
    streams and so changes the path)."""
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, Counter(_norm(e.name) for e in prof.events())


def count(names, kernel):
    k = _norm(kernel)
    return sum(n for name, n in names.items() if k + "(" in name or name.endswith(k))


def assert_ran(names, kernels, what=""):
    for k in kernels:
        assert count(names, k) > 0, (what, k, sorted(n for n in names if "kernel" in n))


def assert_not_ran(names, kernels, what=""):
    for k in kernels:
        assert count(names, k) == 0, (what, k)


def compare_propagate(om, pm, X, S, zs):
    Fs_o, Fm_o, Fv_o = O.propagate(om.layers, torch.as_tensor(X), S, zs)
    (Fs, Fm, Fv), names = launched(lambda: pm.propagate(X, S=S, zs=zs))
    for l in range(len(om.layers)):
        s2 = float(om.layers[l].variance)
        assert rel_err(Fm[l], Fm_o[l]) < TOL, ("mean", l)
        assert rel_err(Fv[l], Fv_o[l], scale=s2) < TOL, ("var", l)
        assert rel_err(Fs[l], Fs_o[l]) < TOL, ("sample", l)
    return names


def compare_grads(pm, prob, zs, ref, what):
    val_o, g_o = ref
    (val, g), names = launched(lambda: pm.ELBO_and_grads((prob["X"], prob["Y"]), zs=zs))
    assert abs(float(val) - float(val_o)) <= TOL * abs(float(val_o)), what
    for k, go in g_o.items():
        assert rel_err(g[k].reshape(go.shape), go) < TOL, (what, k)
    return names


def compare_ei_grad(om, pm, prob, S, zs):
    import dgp_toolbox_b200 as D
    Xg = torch.as_tensor(prob["X"]).clone().requires_grad_(True)
    _, Fm, Fv = O.propagate(om.layers, Xg, S, zs)
    y_min = float(prob["Y"].min())
    neg_ei_o = O.ei_analytic(Fm[-1], Fv[-1], y_min)
    neg_ei_o.sum().backward()
    (neg_ei, dx), names = launched(lambda: D.EI(y_min, prob["X"].shape[1]).run_with_grad(pm, prob["X"], num_samples=S, zs=zs))
    assert rel_err(neg_ei, neg_ei_o.detach()) < 1e-8
    assert rel_err(dx, Xg.grad) < 1e-8
    return names


@pytest.fixture
def ctx():
    """The device context, with every flag this file touches restored afterwards."""
    import dgp_toolbox_b200 as D
    c = D._lib.get_context(0)
    try:
        yield c
    finally:
        c.set_fused(True)
        c.set_vform(True, True)
        c.set_workspace_limit(24 << 30)


# ---------------------------------------------------------------------------------------------------------------------------
# 1. natural selection: each row is a layer shape and the instantiations pick_fused_cfg / pick_fused_bwd_cfg / forward_layer
#    choose for it (computed from the smem_bytes formulas of fused.cuh / fused_bwd.cuh for 227 KB of shared memory)
# ---------------------------------------------------------------------------------------------------------------------------
F0, F1, F2, F3 = ("fused_forward_kernel<128,64,4,2>", "fused_forward_kernel<128,32,4,2>", "fused_forward_kernel<64,64,2,4>",
                  "fused_forward_kernel<64,32,2,4>")


def FB(bm, dmax):
    return f"fused_backward_kernel<{bm},64,{4 if bm == 128 else 2},{2 if bm == 128 else 4},{dmax}>"


# id: (dims, M, N, S, white admitted, forward kernels, V-form adjoint kernels, A-form adjoint kernels)
ROWS = {
    # config 1's training shape: Mp = 64 -> config 2; the shared first layer (1 000 point-samples) runs it halved (config 3)
    "cfg1-shape-mp64": ([2, 2, 1], 50, 1000, 10, True, [F2, F3], [FB(64, 8)], ["rbf_bwd2d_kernel<2,false>"]),
    # Mp = 128 with D_in = 9..16: config 0 (halved to 1 on the first layer), BM 128 adjoint with DMAX 16
    "mp128-din16": ([12, 16, 9, 1], 120, 1000, 10, True, [F0, F1], [FB(128, 16)], ["rbf_bwd2d_kernel<16,false>"]),
    # Mp = 192: three 64-row blocks, config 2 / 3, BM 64 adjoint with DMAX 8
    "mp192": ([5, 3, 1], 130, 1000, 10, True, [F2, F3], [FB(64, 8)], ["rbf_bwd2d_kernel<8,false>"]),
    # Mp = 384: config 1 (BM 128, PT 32), three row blocks; no fused adjoint fits: GEMM + rbf_bwd
    "mp384": ([6, 6, 1], 384, 1000, 10, True, [F1], ["rbf_bwd2d_kernel<8,true>"], ["rbf_bwd2d_kernel<8,false>"]),
    # Mp = 448 / 576 / 640: config 3 chosen directly (7 / 9 / 10 row blocks), GEMM adjoint
    "mp448": ([4, 4, 1], 448, 1000, 10, True, [F3], ["rbf_bwd2d_kernel<4,true>"], ["rbf_bwd2d_kernel<4,false>"]),
    "mp576": ([3, 3, 1], 576, 1000, 10, True, [F3], ["rbf_bwd2d_kernel<4,true>"], ["rbf_bwd2d_kernel<4,false>"]),
    "mp640": ([2, 2, 1], 640, 1000, 10, True, [F3], ["rbf_bwd2d_kernel<2,true>"], ["rbf_bwd2d_kernel<2,false>"]),
    # Mp = 256 with D_out = 16: config 1 on 16 -> 16, config 0 on 16 -> 1; fused adjoint config 1 (BM 64) with DMAX 16
    "mp256-16to16": ([16, 16, 1], 256, 1000, 10, True, [F1, F0], [FB(64, 16)], ["rbf_bwd2d_kernel<16,false>"]),
    # Mp = 256, 31 -> 32 (a single layer with 32 outputs): config 1 forward, GEMM adjoint with rbf_bwd at DMAX 32
    "mp256-31to32": ([31, 32], 256, 300, 4, True, [F1], ["rbf_bwd2d_kernel<32,true>"], ["rbf_bwd2d_kernel<32,false>"]),
    # 40 000 point-samples: the V-form adjoint is the default and rbf_bwd takes its 128-column variant
    "mp256-31to1-bigP": ([31, 1], 256, 20000, 2, True, [F0], ["rbf_bwd_kernel<32,true>"], None),
    # Mp = 640, 16 -> 32: no fused configuration fits -> the unfused pipeline is the default path; white is refused (see below)
    "mp640-unfused": ([16, 32], 640, 150, 2, False, ["kuf_kernel", "moments_kernel<32>"], None, ["rbf_bwd2d_kernel<16,false>"]),
}

# kernel / white combinations: layer l gets KINDS[(l + shift) % 3], so over the three combinations every layer position meets
# every kernel, and white / non-white
COMBOS = {"plain": (0, "none"), "white": (1, "all"), "mixed": (2, "alt")}


def _cases():
    for rid, row in ROWS.items():
        for cid in COMBOS:
            if cid != "plain" and not row[4]:
                continue
            if rid == "mp640-unfused" and cid == "plain":
                for k in ("rbf", "matern32"):
                    yield pytest.param(rid, cid, k, id=f"{rid}-{cid}-{k}")
                continue
            yield pytest.param(rid, cid, None, id=f"{rid}-{cid}")


def _layout(nl, cid, kernel):
    shift, wmode = COMBOS[cid]
    kernels = [kernel] * nl if kernel else [KINDS[(l + shift) % 3] for l in range(nl)]
    white = [wmode == "all" or (wmode == "alt" and l % 2 == 1) for l in range(nl)]
    if wmode == "alt" and nl == 1:
        white = [True]
    return kernels, white


@pytest.mark.parametrize("rid,cid,kernel", list(_cases()))
def test_natural_selection_matches_oracle(rid, cid, kernel, ctx):
    dims, M, N, S, _, fwd, bwd_v, bwd_a = ROWS[rid]
    nl = len(dims) - 1
    kernels, white = _layout(nl, cid, kernel)
    prob = make_problem(dims, M, N, kernels, white)
    om, pm = models(prob, S)
    zs = oracle_zs(om, N, S, 7)
    X, Y = torch.as_tensor(prob["X"]), torch.as_tensor(prob["Y"])

    names = compare_propagate(om, pm, prob["X"], S, zs)
    assert_ran(names, fwd, "propagate")
    if rid == "cfg1-shape-mp64":                      # un-halved on the 10 000-sample layer, halved on the 1 000-point layer
        assert count(names, F2) == 1 and count(names, F3) == 1

    ref = O.elbo_and_grads(om, X, Y, zs)
    names = compare_grads(pm, prob, zs, ref, "default")
    assert_ran(names, fwd, "ELBO")
    all_white, any_white = all(white), any(white)
    default_vform = N * S >= 32768
    if all_white or default_vform:
        assert_ran(names, bwd_v, "V-form adjoint")
    elif bwd_a is not None and not any_white:
        assert_ran(names, bwd_a, "A-form adjoint")
    if not all_white and not default_vform and bwd_v is not None:
        ctx.set_vform(True, "always")
        try:
            names = compare_grads(pm, prob, zs, ref, "vform-always")
        finally:
            ctx.set_vform(True, True)
        assert_ran(names, bwd_v, "V-form adjoint (always)")

    if cid == "plain" and dims[-1] == 1:
        names = compare_ei_grad(om, pm, prob, S, zs)
        assert_ran(names, fwd, "EI")

    if cid == "plain" and bwd_v is not None:         # the reference's operation order, then the unfused GEMM pipeline
        ctx.set_vform(False, False)
        try:
            compare_propagate(om, pm, prob["X"], S, zs)
            compare_grads(pm, prob, zs, ref, "fused-aform")
        finally:
            ctx.set_vform(True, True)
        if M * max(dims[1:]) * 8 <= 160 * 1024:
            ctx.set_fused(False)
            try:
                names = compare_propagate(om, pm, prob["X"], S, zs)
                assert_ran(names, ["kuf_kernel"], "unfused")
                assert_not_ran(names, [F0, F1, F2, F3], "unfused")
                compare_grads(pm, prob, zs, ref, "unfused")
            finally:
                ctx.set_fused(True)


def test_workspace_chunks_match_oracle(ctx):
    """A workspace limit that splits the 1 000-point minibatch into several chunks (every forward kernel then launches once
    per chunk): the same oracle values, white and Matern layers at Mp = 192 included."""
    prob = make_problem([5, 3, 1], 130, 1000, ["matern52", "rbf"], [False, True])
    om, pm = models(prob, 10)
    zs = oracle_zs(om, 1000, 10, 3)
    ref = O.elbo_and_grads(om, torch.as_tensor(prob["X"]), torch.as_tensor(prob["Y"]), zs)
    ctx.set_workspace_limit(128 << 20)
    names = compare_grads(pm, prob, zs, ref, "chunked")
    assert count(names, F2) + count(names, F3) >= 4, names      # two layers, two chunks at least
    ctx.set_vform(True, "always")
    names = compare_grads(pm, prob, zs, ref, "chunked vform-always")
    assert count(names, FB(64, 8)) >= 4


# ---------------------------------------------------------------------------------------------------------------------------
# 2. forced configurations: DGP_B200_FUSED_CFG / DGP_B200_FUSED_BWD_CFG are read once per process, so one child per setting
# ---------------------------------------------------------------------------------------------------------------------------
FORCED_DIMS, FORCED_M, FORCED_N, FORCED_S = [8, 8, 8, 1], 256, 5000, 2      # first layer 5 000, later layers 10 000 samples
FORCED_KERNELS, FORCED_WHITE = ["rbf", "matern52", "matern32"], [False, True, False]
# between two forced configurations only the tiling of the same float64 products changes: the largest relative difference
# measured on a B200 (1000 W power limit) was 2.0e-14
FORCED_CROSS_TOL = 1e-13


def _forced_problem():
    return make_problem(FORCED_DIMS, FORCED_M, FORCED_N, FORCED_KERNELS, FORCED_WHITE)


def forced_child(out_path):
    """Runs in a child process whose environment forces the configurations: propagate and ELBO_and_grads (V-form adjoint)."""
    import dgp_toolbox_b200 as D
    prob = _forced_problem()
    om, pm = models(prob, FORCED_S)
    ctx = D._lib.get_context(0)
    ctx.set_vform(True, "always")
    zs = oracle_zs(om, FORCED_N, FORCED_S, 5)
    (Fs, Fm, Fv), n1 = launched(lambda: pm.propagate(prob["X"], S=FORCED_S, zs=zs))
    (val, g), n2 = launched(lambda: pm.ELBO_and_grads((prob["X"], prob["Y"]), zs=zs))
    torch.save({"Fs": [t.cpu() for t in Fs], "Fm": [t.cpu() for t in Fm], "Fv": [t.cpu() for t in Fv], "val": float(val),
                "g": {k: v.cpu() for k, v in g.items()}, "names": dict(n1 + n2)}, out_path)


FORCED = [(0, 0), (1, 1), (2, 0), (3, 1)]       # (forward config, adjoint config): each of the 4 + 2 reached


def test_forced_configurations_match_oracle_and_each_other(tmp_path):
    outs = {}
    for fcfg, bcfg in FORCED:
        path = tmp_path / f"forced_{fcfg}_{bcfg}.pt"
        env = dict(os.environ, DGP_B200_FUSED_CFG=str(fcfg), DGP_B200_FUSED_BWD_CFG=str(bcfg),
                   PYTHONPATH=os.pathsep.join([ROOT] + [p for p in os.environ.get("PYTHONPATH", "").split(os.pathsep) if p]))
        flags = ["-s"] if sys.flags.no_user_site else []
        r = subprocess.run([sys.executable, *flags, "-c", "import sys; from tests.test_gpu_layer_envelope import forced_child; "
                            "forced_child(sys.argv[1])", str(path)], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-4000:]
        outs[(fcfg, bcfg)] = torch.load(path)
        names = Counter(outs[(fcfg, bcfg)]["names"])
        assert_ran(names, [(F0, F1, F2, F3)[fcfg], FB((128, 64)[bcfg], 8)], (fcfg, bcfg))
        assert_not_ran(names, [k for i, k in enumerate((F0, F1, F2, F3)) if i != fcfg] + [FB((64, 128)[bcfg], 8)], (fcfg, bcfg))

    prob = _forced_problem()
    om, _ = models(prob, FORCED_S)
    zs = oracle_zs(om, FORCED_N, FORCED_S, 5)
    X, Y = torch.as_tensor(prob["X"]), torch.as_tensor(prob["Y"])
    Fs_o, Fm_o, Fv_o = O.propagate(om.layers, X, FORCED_S, zs)
    val_o, g_o = O.elbo_and_grads(om, X, Y, zs)
    for key, o in outs.items():
        for l in range(len(om.layers)):
            assert rel_err(o["Fm"][l], Fm_o[l]) < TOL and rel_err(o["Fs"][l], Fs_o[l]) < TOL, (key, l)
            assert rel_err(o["Fv"][l], Fv_o[l], scale=float(om.layers[l].variance)) < TOL, (key, l)
        assert abs(o["val"] - float(val_o)) <= TOL * abs(float(val_o)), key
        for k, go in g_o.items():
            assert rel_err(o["g"][k].reshape(go.shape), go) < TOL, (key, k)
    worst = 0.0
    for a, b in itertools.combinations(outs.values(), 2):
        for k in ("Fs", "Fm", "Fv"):
            worst = max(worst, max(rel_err(x, y) for x, y in zip(a[k], b[k])))
        worst = max(worst, abs(a["val"] - b["val"]) / abs(b["val"]), max(rel_err(a["g"][k], b["g"][k]) for k in a["g"]))
    print(f"largest relative difference between forced configurations: {worst:.3e}")
    assert worst < FORCED_CROSS_TOL, worst


# ---------------------------------------------------------------------------------------------------------------------------
# 3. the envelope's edges: what must still run, and what must be refused before any launch
# ---------------------------------------------------------------------------------------------------------------------------
EDGE_RUNS = {
    # q_mu of the unfused moments kernel staged at exactly 640 * 32 * 8 B = 160 KiB
    # (its kernel adjoint's Z tile and row-group partial sums need 217.5 KiB: the one-thread-per-column kernel takes it)
    "m640-matern52-31to32": ([31, 32], 640, 150, 2, ["matern52"], [False], ["kuf_kernel", "moments_kernel<32>"],
                             ["rbf_bwd_kernel<32,false>"]),
    # the largest M, with the widest D_out the unfused moments kernel stages (768 * 26 * 8 B <= 160 KiB)
    "m768-matern32-26to26": ([26, 26], 768, 150, 2, ["matern32"], [False], ["kuf_kernel", "moments_kernel<32>"],
                             ["rbf_bwd_kernel<32,false>"]),
    # 63 padding rows at the top Mp
    "m705-stack": ([3, 2, 1], 705, 300, 3, ["rbf", "matern52"], [False, False], ["kuf_kernel", "moments_kernel<2>",
                                                                                     "moments_kernel<1>"], ["rbf_bwd2d_kernel<4,false>"]),
}


@pytest.mark.parametrize("eid", list(EDGE_RUNS))
def test_envelope_edge_runs_match_oracle(eid, ctx):
    dims, M, N, S, kernels, white, kern, adj = EDGE_RUNS[eid]
    prob = make_problem(dims, M, N, kernels, white)
    om, pm = models(prob, S)
    zs = oracle_zs(om, N, S, 2)
    names = compare_propagate(om, pm, prob["X"], S, zs)
    assert_ran(names, kern, eid)
    assert_not_ran(names, [F0, F1, F2, F3], eid)
    ref = O.elbo_and_grads(om, torch.as_tensor(prob["X"]), torch.as_tensor(prob["Y"]), zs)
    names = compare_grads(pm, prob, zs, ref, eid)
    assert_ran(names, adj, eid)


@pytest.mark.parametrize("N", [768, 700])
def test_full_cov_at_the_largest_n_matches_oracle(N):
    prob = make_problem([4, 3, 1], 256, N, ["matern52", "matern32"], [True, False])
    om, pm = models(prob, 2)
    zs = oracle_zs(om, N, 2, 3)
    with torch.no_grad():
        Fs_o, Fm_o, Fv_o = O.propagate_full_cov(om.layers, torch.as_tensor(prob["X"]), 2, zs)
    Fs, Fm, Fv = pm.propagate(prob["X"], full_cov=True, S=2, zs=zs)
    for l in range(len(om.layers)):
        assert tuple(Fv[l].shape) == (2, N, N, om.layers[l].D_out)
        assert rel_err(Fm[l], Fm_o[l]) < TOL and rel_err(Fv[l], Fv_o[l], scale=float(om.layers[l].variance)) < TOL
        assert rel_err(Fs[l], Fs_o[l]) < 1e-8


@pytest.mark.parametrize("M,white", [(768, False), (576, True)])
def test_natural_gradient_step_at_large_m_matches_oracle(M, white):
    prob = make_problem([2, 2, 1], M, 200, ["rbf", "matern52"], [white, white])
    om, pm = models(prob, 2)
    zs = oracle_zs(om, 200, 2, 9)
    new = O.natgrad_step(om, torch.as_tensor(prob["X"]), torch.as_tensor(prob["Y"]), zs, 1e-3, [0, 1])
    pm.natgrad_step((prob["X"], prob["Y"]), 1e-3, [(l.q_mu, l.q_sqrt) for l in pm.layers], zs=zs)
    for (mu_o, R_o), layer in zip(new, pm.layers):
        assert rel_err(layer.q_mu.value, mu_o) < 1e-8
        assert rel_err(layer.q_sqrt.value, R_o) < 1e-8


# (dims, M, white, fused, message); each is built at a shape the library refuses. M = 769 is refused by the first library
# call, the layer constructor's Cholesky.
EDGE_ERRORS = {
    "m769": ([2, 2, 1], 769, [False, False], True, "M > 768 is not supported"),
    "white-mp704": ([2, 1], 704, [True], True, "white=True layers run on the fused conditional kernel only"),
    "white-mp768": ([2, 1], 768, [True], True, "white=True layers run on the fused conditional kernel only"),
    "white-m640-16to32": ([16, 32], 640, [True], True, "white=True layers run on the fused conditional kernel only"),
    "white-unfused": ([2, 2, 1], 64, [True, False], False, "white=True layers run on the fused conditional kernel only"),
    "m641-dout32-unfused": ([16, 32], 641, [False], True, "160 KiB"),
}


@pytest.fixture(scope="module")
def valid_case():
    """A small valid model and its oracle ELBO: the call after each refused one must still be right."""
    prob = make_problem([3, 3, 1], 100, 200, ["matern32", "rbf"], [True, False])
    om, pm = models(prob, 4)
    zs = oracle_zs(om, 200, 4, 1)
    return prob, pm, zs, O.elbo_and_grads(om, torch.as_tensor(prob["X"]), torch.as_tensor(prob["Y"]), zs)


def _refused(ctx, call, message):
    import dgp_toolbox_b200 as D
    torch.cuda.synchronize()
    n0 = ctx.launch_count()
    with pytest.raises(D._lib.DGPError, match=message):
        call()
    assert ctx.launch_count() == n0, "a refused call launched kernels"


@pytest.mark.parametrize("eid", list(EDGE_ERRORS))
def test_envelope_edge_refusals_launch_nothing(eid, ctx, valid_case):
    dims, M, white, fused, message = EDGE_ERRORS[eid]
    prob = O.synthetic_problem(dims[0], dims[1:-1], M, 40)        # shape only: values do not matter for a refusal
    if dims[-1] != 1:
        prob["layers"][-1]["q_mu"] = np.zeros((M, dims[-1]))
        prob["layers"][-1]["q_sqrt"] = np.eye(M)[None].repeat(dims[-1], 0)
        prob["Y"] = np.zeros((40, dims[-1]))
    for layer, w in zip(prob["layers"], white):
        layer["white"] = w
    ctx.set_fused(fused)
    try:
        if M > 768:
            _refused(ctx, lambda: product_model_from_problem(prob, 2), message)
        else:
            pm = product_model_from_problem(prob, 2)
            _refused(ctx, lambda: pm.ELBO_and_grads((prob["X"], prob["Y"]), seed=3), message)
            _refused(ctx, lambda: pm.propagate(prob["X"], S=2, seed=3), message)
    finally:
        ctx.set_fused(True)
    vprob, vpm, zs, ref = valid_case
    compare_grads(vpm, vprob, zs, ref, "after " + eid)


def test_full_cov_refuses_n_above_768(ctx, valid_case):
    prob = make_problem([2, 2, 1], 40, 769, ["rbf", "matern52"], [False, True])
    _, pm = models(prob, 1)
    _refused(ctx, lambda: pm.propagate(prob["X"], full_cov=True, S=1, seed=1), "N > 768")
    vprob, vpm, zs, ref = valid_case
    compare_grads(vpm, vprob, zs, ref, "after full_cov N = 769")
