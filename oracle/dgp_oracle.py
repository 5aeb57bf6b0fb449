"""CPU oracle for the doubly-stochastic DGP hot path (TEST INFRASTRUCTURE, NOT PRODUCT).

This is a float64 torch-CPU restatement, op for op, of the reference path
(/root/reference, cited as file:line below). Only ``tests/``, ``__graft_entry__.smoke()``
and the ``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may import it; the product
package ``dgp_toolbox_b200`` never does.

PARITY STATUS: the reference's arithmetic lives in GPflow 2.0.x / TensorFlow 2.x / TFP, none of which
is installed here and none of which is pinned by the reference (README.md:5 says "GPflow 2.0").  The
restatement is pinned to reference-produced numbers only through the notebook known answers
(KAT-1 -85.98812279560475, KAT-2 -73.6722504558447, KAT-3 2032 parameters; tests/test_oracle_kat.py).
Everything else is "parity unpinned": validated by finite differences and algebraic identities.

Third-party semantics restated (published GPflow 2.0 algorithms):
  * SquaredExponential.K: sigma^2 exp(-0.5 r2), r2 = |x/l|^2 + |x'/l|^2 - 2 (x/l).(x'/l)  (expanded, unclamped)
  * covariances.Kuu = K(Z) + jitter I (jitter = default_jitter() = 1e-6); Kuf = K(Z, X)
  * Gaussian.variational_expectations / predict_mean_and_var
  * mean functions Zero / Identity / Linear
  * positive() = softplus, likelihood variance softplus + 1e-6 shift; triangular() = tfp FillTriangular
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np
import torch

DTYPE = torch.float64
JITTER = 1e-6  # gpflow.default_jitter()


def _t(x):
    if isinstance(x, torch.Tensor):
        return x.to(DTYPE)
    return torch.as_tensor(np.asarray(x, dtype=np.float64))


# --------------------------------------------------------------------------------------
# kernel (GPflow SquaredExponential; call sites utils/layers.py:221,230,243,272)
# --------------------------------------------------------------------------------------
def rbf_K(X, X2, lengthscales, variance):
    """GPflow SquaredExponential.K with the expanded-square distance (gpflow/utilities/ops.py
    square_distance): -2 X X2^T + |X|^2 + |X2|^2 on inputs pre-divided by the lengthscales."""
    Xs = X / lengthscales
    if X2 is None:
        sq = (Xs * Xs).sum(-1, keepdim=True)
        dist = -2.0 * Xs @ Xs.T
        dist = dist + (sq + sq.T)
    else:
        X2s = X2 / lengthscales
        a = (Xs * Xs).sum(-1)
        b = (X2s * X2s).sum(-1)
        dist = -2.0 * Xs @ X2s.T
        dist = dist + (a[:, None] + b[None, :])
    return variance * torch.exp(-0.5 * dist)


def _scaled_sqdist(X, X2, lengthscales):
    """gpflow/utilities/ops.py square_distance on inputs divided by the lengthscales (expanded form, unclamped)."""
    Xs = X / lengthscales
    if X2 is None:
        sq = (Xs * Xs).sum(-1, keepdim=True)
        return -2.0 * Xs @ Xs.T + (sq + sq.T)
    X2s = X2 / lengthscales
    return -2.0 * Xs @ X2s.T + ((Xs * Xs).sum(-1)[:, None] + (X2s * X2s).sum(-1)[None, :])


def kernel_K(X, X2, lengthscales, variance, kind="rbf"):
    """GPflow stationary kernels: SquaredExponential (K_r2), Matern32 / Matern52 (K_r with r = sqrt(max(r2, 1e-36)),
    gpflow/kernels/stationaries.py) — the three kernels BO/SO_BO.py:190-197,237-244 offers."""
    if kind == "rbf":
        return rbf_K(X, X2, lengthscales, variance)
    r = torch.sqrt(torch.clamp(_scaled_sqdist(X, X2, lengthscales), min=1e-36))
    if kind == "matern32":
        a = math.sqrt(3.0)
        return variance * (1.0 + a * r) * torch.exp(-a * r)
    if kind == "matern52":
        a = math.sqrt(5.0)
        return variance * (1.0 + a * r + 5.0 / 3.0 * r * r) * torch.exp(-a * r)
    raise ValueError(kind)


def rbf_K_diag(X, variance):
    return variance * torch.ones(X.shape[0], dtype=DTYPE)


# --------------------------------------------------------------------------------------
# layer parameters
# --------------------------------------------------------------------------------------
@dataclass
class OLayer:
    """State of one reference SVGP_Layer (utils/layers.py:180-224)."""
    Z: torch.Tensor            # [M, D_in]
    lengthscales: torch.Tensor  # [D_in] (ARD) or [] / [1] (isotropic)
    variance: torch.Tensor      # []
    q_mu: torch.Tensor          # [M, D_out]
    q_sqrt: torch.Tensor        # [D_out, M, M] lower triangular
    mean_kind: str = "zero"     # zero | identity | linear
    mf_W: Optional[torch.Tensor] = None  # [D_in, D_out]
    mf_b: Optional[torch.Tensor] = None  # [D_out]
    white: bool = False
    kernel_kind: str = "rbf"    # rbf | matern32 | matern52

    @property
    def M(self):
        return self.Z.shape[0]

    @property
    def D_out(self):
        return self.q_mu.shape[1]

    @property
    def D_in(self):
        return self.Z.shape[1]

    def params(self):
        return {"Z": self.Z, "lengthscales": self.lengthscales, "variance": self.variance,
                "q_mu": self.q_mu, "q_sqrt": self.q_sqrt}


def make_layer(Z, lengthscales, variance, D_out, mean_kind="zero", mf_W=None, mf_b=None, white=False,
               q_mu=None, q_sqrt=None, kernel_kind="rbf") -> OLayer:
    """SVGP_Layer.__init__ (utils/layers.py:181-224): q_mu = 0; q_sqrt = I, or chol(K(Z)+jitter I) when not white."""
    Z = _t(Z).clone()
    ls = _t(lengthscales).clone()
    var = _t(variance).clone().reshape(())
    M = Z.shape[0]
    if q_mu is None:
        q_mu = torch.zeros(M, D_out, dtype=DTYPE)
    if q_sqrt is None:
        if white:
            q_sqrt = torch.eye(M, dtype=DTYPE)[None].repeat(D_out, 1, 1)
        else:
            Ku = kernel_K(Z, None, ls, var, kernel_kind)  # utils/layers.py:221
            Lu = torch.linalg.cholesky(Ku + torch.eye(M, dtype=DTYPE) * JITTER)  # :222
            q_sqrt = Lu[None].repeat(D_out, 1, 1)  # :223
    return OLayer(Z=Z, lengthscales=ls, variance=var, q_mu=_t(q_mu).clone(), q_sqrt=_t(q_sqrt).clone(),
                  mean_kind=mean_kind, mf_W=None if mf_W is None else _t(mf_W).clone(),
                  mf_b=None if mf_b is None else _t(mf_b).clone(), white=white, kernel_kind=kernel_kind)


def mean_function(layer: OLayer, X):
    """GPflow mean_functions Zero / Identity / Linear (utils/layer_initializations.py:27,42,52)."""
    if layer.mean_kind == "zero":
        return torch.zeros(X.shape[0], 1, dtype=DTYPE)  # broadcasts against [P, D_out]
    if layer.mean_kind == "identity":
        return X
    if layer.mean_kind == "linear":
        out = X @ layer.mf_W
        if layer.mf_b is not None:
            out = out + layer.mf_b
        return out
    raise ValueError(layer.mean_kind)


# --------------------------------------------------------------------------------------
# a1-a4: SVGP_Layer.build_cholesky_if_needed / conditional_ND  (utils/layers.py:227-278)
# --------------------------------------------------------------------------------------
def kuu_chol(layer: OLayer):
    """utils/layers.py:227-234."""
    M = layer.M
    Ku = kernel_K(layer.Z, None, layer.lengthscales, layer.variance, layer.kernel_kind) + JITTER * torch.eye(M, dtype=DTYPE)
    Lu = torch.linalg.cholesky(Ku)
    return Ku, Lu


def conditional_ND(layer: OLayer, X):
    """utils/layers.py:237-278, diagonal (full_cov=False) branch, same op order:
    Kuf -> triangular_solve(Lu) -> triangular_solve(Lu^T) -> A^T q_mu -> SK = q_sqrt q_sqrt^T - Ku
    -> B = SK A_tiled -> sum(A_tiled * B, 1) -> K_diag + delta -> transpose -> + mean_function."""
    Ku, Lu = kuu_chol(layer)
    D_out = layer.D_out
    M = layer.M
    Kuf = kernel_K(layer.Z, X, layer.lengthscales, layer.variance, layer.kernel_kind)   # :243  [M, P]
    A = torch.linalg.solve_triangular(Lu, Kuf, upper=False)                        # :245
    if not layer.white:
        A = torch.linalg.solve_triangular(Lu.T, A, upper=True)                     # :247
    mean = A.T @ layer.q_mu                                                        # :249
    A_tiled = A[None].expand(D_out, -1, -1)                                        # :251
    if layer.white:
        SK = -torch.eye(M, dtype=DTYPE)[None].expand(D_out, -1, -1)                # :255
    else:
        SK = -Ku[None].expand(D_out, -1, -1)                                       # :257
    SK = SK + layer.q_sqrt @ layer.q_sqrt.transpose(1, 2)                          # :260
    B = SK @ A_tiled                                                               # :263
    delta = (A_tiled * B).sum(1)                                                   # :271  [D_out, P]
    Kff = rbf_K_diag(X, layer.variance)                                            # :272
    var = (Kff[None] + delta).T                                                    # :275-276
    return mean + mean_function(layer, X), var                                     # :278


def layer_KL(layer: OLayer):
    """utils/layers.py:280-308."""
    Ku, Lu = kuu_chol(layer)
    D_out, M = layer.D_out, layer.M
    KL = torch.tensor(-0.5 * D_out * M, dtype=DTYPE)
    diag = torch.diagonal(layer.q_sqrt, dim1=1, dim2=2)
    KL = KL - 0.5 * torch.log(diag ** 2).sum()
    if not layer.white:
        KL = KL + torch.log(torch.diagonal(Lu)).sum() * D_out
        LinvR = torch.linalg.solve_triangular(Lu[None].expand(D_out, -1, -1), layer.q_sqrt, upper=False)
        KL = KL + 0.5 * (LinvR ** 2).sum()
        Kinv_m = torch.cholesky_solve(layer.q_mu, Lu)
        KL = KL + 0.5 * (layer.q_mu * Kinv_m).sum()
    else:
        KL = KL + 0.5 * (layer.q_sqrt ** 2).sum()
        KL = KL + 0.5 * (layer.q_mu ** 2).sum()
    return KL


# --------------------------------------------------------------------------------------
# a5-a7: conditional_SND, sample_from_conditional, reparameterize, propagate
# --------------------------------------------------------------------------------------
def conditional_SND(layer: OLayer, X):
    """utils/layers.py:63-85 (full_cov=False): [S,N,D] -> [S*N,D] -> conditional_ND -> [S,N,D_out]."""
    S, N, D = X.shape
    mean, var = conditional_ND(layer, X.reshape(S * N, D))
    return mean.reshape(S, N, layer.D_out), var.reshape(S, N, layer.D_out)


def reparameterize(mean, var, z):
    """utils/utils.py:40-41 (diagonal branch): mean + z * (var + jitter) ** 0.5."""
    if var is None:
        return mean
    return mean + z * (var + JITTER) ** 0.5


def sample_from_conditional(layer: OLayer, X, z):
    """utils/layers.py:87-130 without input propagation (input_prop_dim is never set by any constructor)."""
    mean, var = conditional_SND(layer, X)
    samples = reparameterize(mean, var, z)
    return samples, mean, var


def propagate(layers: Sequence[OLayer], X, S: int, zs: Sequence[torch.Tensor]):
    """models/dgp.py:34-63 with explicit zs (the reference's `zs=` hook)."""
    F = X[None].expand(S, -1, -1)
    Fs, Fmeans, Fvars = [], [], []
    for layer, z in zip(layers, zs):
        F, Fmean, Fvar = sample_from_conditional(layer, F, z)
        Fs.append(F)
        Fmeans.append(Fmean)
        Fvars.append(Fvar)
    return Fs, Fmeans, Fvars


# ---- full_cov=True branches (SURVEY §8 f4; not on the accelerated path yet: the oracle states them for the next round) ----
def conditional_ND_full(layer: OLayer, X):
    """utils/layers.py:237-278 with full_cov=True: mean [N, D_out], cov [N, N, D_out] = transpose(K(X, X)[None] + A^T SK_d A)."""
    Ku, Lu = kuu_chol(layer)
    M = layer.M
    Kuf = kernel_K(layer.Z, X, layer.lengthscales, layer.variance, layer.kernel_kind)
    A = torch.linalg.solve_triangular(Lu, Kuf, upper=False)
    if not layer.white:
        A = torch.linalg.solve_triangular(Lu.T, A, upper=True)
    mean = A.T @ layer.q_mu
    SK = -(torch.eye(M, dtype=DTYPE) if layer.white else Ku)[None] + layer.q_sqrt @ layer.q_sqrt.transpose(1, 2)
    delta = A.T[None] @ (SK @ A[None])                                            # :265  [D_out, N, N]
    Kff = kernel_K(X, None, layer.lengthscales, layer.variance, layer.kernel_kind)   # :266
    return mean + mean_function(layer, X), (Kff[None] + delta).permute(2, 1, 0)       # tf.transpose reverses the axes (:276)


def reparameterize_full(mean, var, z):
    """utils/utils.py:43-52: mean [S,N,D], var [S,N,N,D], z [S,N,D] -> mean + chol(var_sd + jitter I) z_sd per sample and output."""
    S, N, D = mean.shape
    v = var.permute(0, 3, 1, 2) + JITTER * torch.eye(N, dtype=DTYPE)
    f = mean.permute(0, 2, 1) + (torch.linalg.cholesky(v) @ z.permute(0, 2, 1)[..., None])[..., 0]
    return f.permute(0, 2, 1)


def propagate_full_cov(layers: Sequence[OLayer], X, S: int, zs: Sequence[torch.Tensor]):
    """models/dgp.py:34-63 with full_cov=True: every layer's conditional is evaluated per sample (conditional_SND's map_fn,
    utils/layers.py:76-79) and sampled with the full N x N covariance. Returns Fs, Fmeans [S,N,D_l], Fvars [S,N,N,D_l]."""
    F = X[None].expand(S, -1, -1)
    Fs, Fmeans, Fvars = [], [], []
    for layer, z in zip(layers, zs):
        mv = [conditional_ND_full(layer, F[s]) for s in range(S)]
        mean, var = torch.stack([m for m, _ in mv]), torch.stack([v for _, v in mv])
        F = reparameterize_full(mean, var, z)
        Fs.append(F)
        Fmeans.append(mean)
        Fvars.append(var)
    return Fs, Fmeans, Fvars


# --------------------------------------------------------------------------------------
# a8-a11: Gaussian likelihood, ELBO, predict
# --------------------------------------------------------------------------------------
def gaussian_variational_expectations(Fmu, Fvar, Y, lik_var):
    """GPflow Gaussian.variational_expectations via utils/utils.py:89-93 (Y broadcast on a new leading axis)."""
    return (-0.5 * math.log(2 * math.pi) - 0.5 * torch.log(lik_var)
            - 0.5 * ((Y[None] - Fmu) ** 2 + Fvar) / lik_var)


@dataclass
class OModel:
    layers: List[OLayer]
    lik_var: torch.Tensor
    num_samples: int = 1

    def named_params(self):
        out = {}
        for i, l in enumerate(self.layers):
            for k, v in l.params().items():
                out[f"layers.{i}.{k}"] = v
        out["lik_var"] = self.lik_var
        return out


def E_log_p_Y(model: OModel, X, Y, zs):
    """models/dgp.py:79-87."""
    _, Fmeans, Fvars = propagate(model.layers, X, model.num_samples, zs)
    ve = gaussian_variational_expectations(Fmeans[-1], Fvars[-1], Y, model.lik_var)
    return ve.mean(0)


def elbo(model: OModel, X, Y, zs, scale: float = 1.0):
    """models/dgp.py:89-100 (the reference's scale is identically 1, dgp.py:95-99; exposed for minibatching)."""
    L = E_log_p_Y(model, X, Y, zs).sum()
    KL = sum(layer_KL(l) for l in model.layers)
    return L * scale - KL


def elbo_and_grads(model: OModel, X, Y, zs, scale: float = 1.0, wrt_X: bool = False):
    """ELBO value and constrained-space gradients by autograd (the gradient oracle; reference uses
    tf.GradientTape over the same ops, models/dgp.py:272-275)."""
    params = model.named_params()
    leaves = {k: v.detach().clone().requires_grad_(True) for k, v in params.items()}
    layers = []
    for i, l in enumerate(model.layers):
        layers.append(OLayer(Z=leaves[f"layers.{i}.Z"], lengthscales=leaves[f"layers.{i}.lengthscales"],
                             variance=leaves[f"layers.{i}.variance"], q_mu=leaves[f"layers.{i}.q_mu"],
                             q_sqrt=leaves[f"layers.{i}.q_sqrt"], mean_kind=l.mean_kind, mf_W=l.mf_W, mf_b=l.mf_b,
                             white=l.white, kernel_kind=l.kernel_kind))
    m2 = OModel(layers=layers, lik_var=leaves["lik_var"], num_samples=model.num_samples)
    Xl = X.detach().clone().requires_grad_(wrt_X)
    val = elbo(m2, Xl, Y, zs, scale)
    val.backward()
    grads = {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in leaves.items()}
    for i in range(len(layers)):  # q_sqrt gradient lives on the lower triangle only (FillTriangular)
        grads[f"layers.{i}.q_sqrt"] = torch.tril(grads[f"layers.{i}.q_sqrt"])
    if wrt_X:
        grads["X"] = Xl.grad
    return val.detach(), grads


def elbo_and_grads_chunked(model: OModel, X, Y, seed: int, chunk: int = 256, scale: float = 1.0, n_offset: int = 0):
    """ELBO and constrained-space gradients of a LARGE minibatch, accumulated over chunks of points: the data term
    sum_n E_log_p_Y (models/dgp.py:96) is additive over points and the KL terms (:97) are added once, so the reference's value
    and gradient on the whole minibatch equal the sums below. Draws are the Philox stream of `seed` at the GLOBAL point index
    (what the CUDA kernels draw for the same seed), so no [S, N, D] array of the whole minibatch is ever materialised."""
    params = model.named_params()
    total = {k: torch.zeros_like(v) for k, v in params.items()}
    value = 0.0
    N = X.shape[0]
    for lo in range(0, N, chunk):
        hi = min(N, lo + chunk)
        zs = [torch.as_tensor(philox_normal(seed, l, model.num_samples, hi - lo, layer.D_out, n_offset=n_offset + lo))
              for l, layer in enumerate(model.layers)]
        leaves = {k: v.detach().clone().requires_grad_(True) for k, v in params.items()}
        layers = [OLayer(Z=leaves[f"layers.{i}.Z"], lengthscales=leaves[f"layers.{i}.lengthscales"], variance=leaves[f"layers.{i}.variance"],
                         q_mu=leaves[f"layers.{i}.q_mu"], q_sqrt=leaves[f"layers.{i}.q_sqrt"], mean_kind=l.mean_kind, mf_W=l.mf_W,
                         mf_b=l.mf_b, white=l.white, kernel_kind=l.kernel_kind) for i, l in enumerate(model.layers)]
        m2 = OModel(layers=layers, lik_var=leaves["lik_var"], num_samples=model.num_samples)
        term = E_log_p_Y(m2, X[lo:hi], Y[lo:hi], zs).sum() * scale
        if lo == 0:
            term = term - sum(layer_KL(l) for l in layers)
        term.backward()
        value += float(term.detach())
        for k, v in leaves.items():
            if v.grad is not None:
                total[k] += v.grad
    for i in range(len(model.layers)):
        total[f"layers.{i}.q_sqrt"] = torch.tril(total[f"layers.{i}.q_sqrt"])
    return value, total


def predict_f(model: OModel, X, S, zs):
    """models/dgp.py:66-77."""
    _, Fmeans, Fvars = propagate(model.layers, X, S, zs)
    return Fmeans[-1], Fvars[-1]


def predict_y(model: OModel, X, S, zs):
    """models/dgp.py:113-124 + Gaussian.predict_mean_and_var: (mu, var + sigma_n^2)."""
    m, v = predict_f(model, X, S, zs)
    return m, v + model.lik_var


def predict(model: OModel, X, S, zs):
    """models/dgp.py:362-366: mixture moments over the S samples."""
    ym, yv = predict_y(model, X, S, zs)
    mean = ym.mean(0)
    var = (yv + ym ** 2).mean(0) - mean ** 2
    return mean, var


# --------------------------------------------------------------------------------------
# layer construction: init_layers_linear (utils/layer_initializations.py:24-68) and DGP (models/dgp.py:245-254)
# --------------------------------------------------------------------------------------
def init_layers_linear(X, Y, Z, kernels, num_units, num_outputs=None, final_mean="zero", white=False):
    """kernels: list of (lengthscales, variance) pairs, one per SVGP layer (len(num_units)+1)."""
    X = np.asarray(X, dtype=np.float64)
    Z = np.asarray(Z, dtype=np.float64)
    num_outputs = num_outputs or Y.shape[1]
    layers = []
    dims = [X.shape[1]] + list(num_units)
    X_running, Z_running = X.copy(), Z.copy()
    for dim_in, dim_out, (ls, var) in zip(dims[:-1], dims[1:], kernels[:-1]):
        W = None
        if dim_in == dim_out:
            kind = "identity"                                                  # :41-42
        else:
            if dim_in > dim_out:                                               # :45-47 PCA projection
                _, _, V = np.linalg.svd(X_running, full_matrices=False)
                W = V[:dim_out, :].T
            else:                                                              # :49-50 identity + zero padding
                W = np.concatenate([np.eye(dim_in), np.zeros((dim_in, dim_out - dim_in))], 1)
            kind = "linear"
        layers.append(make_layer(Z_running, ls, var, dim_out, kind, mf_W=W,
                                 mf_b=None if W is None else np.zeros(dim_out), white=white))
        if dim_in != dim_out:                                                  # :59-61
            Z_running = Z_running.dot(W)
            X_running = X_running.dot(W)
    ls, var = kernels[-1]
    layers.append(make_layer(Z_running, ls, var, num_outputs, final_mean, white=white))   # :67
    return layers


def make_dgp(X, Y, Z, kernels, num_units, lik_var=1.0, num_samples=1, white=False) -> OModel:
    layers = init_layers_linear(X, Y, Z, kernels, num_units, white=white)
    return OModel(layers=layers, lik_var=_t(lik_var).reshape(()), num_samples=num_samples)


def number_parameters(model: OModel) -> int:
    """models/dgp.py:348-360 with trainable=False: every GPflow Parameter, i.e. per layer q_mu, q_sqrt (full
    [D_out,M,M] array as .numpy() returns it), Z, kernel variance, kernel lengthscales, Linear mean-function A and b
    (present but non-trainable), plus the likelihood variance."""
    n = 1
    for l in model.layers:
        n += l.q_mu.numel() + l.q_sqrt.numel() + l.Z.numel() + 1 + l.lengthscales.numel()
        if l.mean_kind == "linear":
            n += l.mf_W.numel() + (l.mf_b.numel() if l.mf_b is not None else 0)
    return n


# --------------------------------------------------------------------------------------
# a12: acquisition (Infill_criteria.py:28-52, EHVI.py:90-104,110-119,154-157)
# --------------------------------------------------------------------------------------
def _Phi(x):
    return 0.5 * (1.0 + torch.erf(x / math.sqrt(2.0)))


def _phi(x):
    return torch.exp(-0.5 * x * x) / math.sqrt(2 * math.pi)


def mixture_moments(Fmean, Fvar):
    """Infill_criteria.py:40-41 / EHVI.py:114-115."""
    m = Fmean.mean(0)
    v = (Fvar + Fmean ** 2).mean(0) - m ** 2
    return m, v


def ei_analytic(Fmean, Fvar, y_min):
    """Infill_criteria.py:39-47,52: Normal(mean, sqrt(var)); t1 = (y_min-mean) cdf(y_min);
    t2 = var * pdf(y_min) (= sigma*phi(u)); returns -EI."""
    m, v = mixture_moments(Fmean, Fvar)
    s = torch.sqrt(v)
    u = (y_min - m) / s
    t1 = (y_min - m) * _Phi(u)
    t2 = v * (_phi(u) / s)
    return -(t1 + t2)


def ei_mc(F_last, y_min):
    """Infill_criteria.py:49-52: mean_s where(F - y_min < 0, y_min - F, 0); returns -EI."""
    imp = torch.where((F_last - y_min) < 0, y_min - F_last, torch.zeros_like(F_last))
    return -imp.mean(0)


def _ei_from_moments(m, v, y):
    s = torch.sqrt(v)
    u = (y - m) / s
    return (y - m) * _Phi(u) + v * (_phi(u) / s)


def wb2(Ymean, Yvar, y_min):
    """Infill_criteria.py:124-133: -(EI - mean) on predict_y mixture moments."""
    m, v = mixture_moments(Ymean, Yvar)
    return -(_ei_from_moments(m, v, y_min) - m)


def wb2s(Ymean, Yvar, y_min, x):
    """Infill_criteria.py:187-198: -(S * EI - mean), S = 1 / (1 + 1 / exp(x))."""
    m, v = mixture_moments(Ymean, Yvar)
    S = 1.0 / (1.0 + 1.0 / torch.exp(x))
    return -(S * _ei_from_moments(m, v, y_min) - m)


def pof(Ymean, Yvar, zero_c):
    """Probability of feasibility P[c <= zero_c] = Phi((zero_c - mean) / sigma) on predict_y mixture moments: the quantity
    Infill_criteria.py:318-345 (PoF) needs but never returns (its `run` has no return statement)."""
    m, v = mixture_moments(Ymean, Yvar)
    return _Phi((zero_c - m) / torch.sqrt(v))


def ev_analytic(Ymean, Yvar, zero_c):
    """Infill_criteria.py:249-257: Normal(-mean, sqrt(var)); t1 = (-c + mean) cdf(-c); t2 = var * pdf(-c)."""
    m, v = mixture_moments(Ymean, Yvar)
    s = torch.sqrt(v)
    u = (m - zero_c) / s
    return (m - zero_c) * _Phi(u) + v * (_phi(u) / s)


def ev_mc(F_last, zero_c):
    """Infill_criteria.py:259-262."""
    return torch.where((F_last - zero_c) < 0, torch.zeros_like(F_last), F_last - zero_c).mean(0)


def Y_ND(Y0, Y1, nadir, ideal=(0.0, 0.0)):
    """EHVI.py:90-100: pad the sorted Pareto front with nadir/ideal."""
    n = len(Y0)
    a = np.zeros(n + 2)
    b = np.zeros(n + 2)
    a[1:-1] = Y0
    b[1:-1] = Y1
    a[0], a[-1] = nadir[0], ideal[0]
    b[0], b[-1] = ideal[1], nadir[1]
    return a, b


def psi(a, b, mu, sigma):
    """EHVI.py:102-104."""
    u = (b - mu) / sigma
    return sigma * _phi(u) + (a - mu) * _Phi(u)


def ehvi_exact(m0, v0, m1, v1, ynd0, ynd1):
    """EHVI.py:154-157 (uncorrelated exact 2-objective EHVI strip sum); ynd* are the padded fronts."""
    s0, s1 = torch.sqrt(v0), torch.sqrt(v1)
    n = len(ynd0)
    t1 = torch.zeros_like(m0)
    for i in range(1, n - 1):
        t1 = t1 + ((ynd0[i - 1] - ynd0[i])
                   * (_Phi((ynd0[i] - m0) / s0) - _Phi((ynd0[-1] - m0) / s0))
                   * (psi(ynd1[i], ynd1[i], m1, s1) - psi(ynd1[i], ynd1[0], m1, s1)))
    t2 = torch.zeros_like(m0)
    for i in range(1, n):
        t2 = t2 + ((psi(ynd0[i - 1], ynd0[i - 1], m0, s0) - psi(ynd0[i - 1], ynd0[i], m0, s0))
                   * (psi(ynd1[i], ynd1[i], m1, s1) - psi(ynd1[i], ynd1[0], m1, s1)))
    return t1 + t2


# --------------------------------------------------------------------------------------
# GPflow NaturalGradient (XiNat) step on (q_mu, q_sqrt) pairs — models/dgp.py:188,218,312,343
# --------------------------------------------------------------------------------------
def natgrad_step(model: OModel, X, Y, zs, gamma: float, layer_indices: Sequence[int], scale: float = 1.0):
    """theta <- theta - gamma * d(-ELBO)/d eta, theta = (S^-1 mu, -S^-1/2), eta = (mu, S + mu mu^T), S = q_sqrt q_sqrt^T
    (GPflow 2.0 optimizers/natgrad.py, default XiNat). The gradient w.r.t. the expectation parameters is taken by autograd
    through eta -> (mu, chol(eta2 - mu mu^T)), i.e. by a different route than the product's closed-form Cholesky adjoint.
    Returns the new [(q_mu, q_sqrt)] for the given layers (the model is not modified)."""
    etas = []
    layers = []
    for i, l in enumerate(model.layers):
        if i in layer_indices:
            mu = l.q_mu.detach().T.unsqueeze(-1)                                   # [D, M, 1]
            S = l.q_sqrt.detach() @ l.q_sqrt.detach().transpose(1, 2)
            e1 = mu.clone().requires_grad_(True)
            e2 = (S + mu @ mu.transpose(1, 2)).clone().requires_grad_(True)
            etas.append((i, e1, e2))
            Sfrom = e2 - e1 @ e1.transpose(1, 2)
            layers.append(OLayer(Z=l.Z, lengthscales=l.lengthscales, variance=l.variance, q_mu=e1.squeeze(-1).T,
                                 q_sqrt=torch.linalg.cholesky(Sfrom), mean_kind=l.mean_kind, mf_W=l.mf_W, mf_b=l.mf_b, white=l.white,
                                 kernel_kind=l.kernel_kind))
        else:
            layers.append(l)
    loss = -elbo(OModel(layers=layers, lik_var=model.lik_var, num_samples=model.num_samples), X, Y, zs, scale)
    loss.backward()
    out = []
    for i, e1, e2 in etas:
        l = model.layers[i]
        mu = l.q_mu.detach().T.unsqueeze(-1)
        Sinv = torch.cholesky_inverse(l.q_sqrt.detach())
        g2 = 0.5 * (e2.grad + e2.grad.transpose(1, 2))
        theta1 = Sinv @ mu - gamma * e1.grad
        theta2 = -0.5 * Sinv - gamma * g2
        # one matrix at a time: with the MKL build of torch 2.11, a batched float64 torch.linalg.inv of 256 x 256 or larger after
        # any torch.set_num_threads call stops in MKL ("Parameter 6 was incorrect on entry to DLASWP") and never returns
        S_new = torch.stack([torch.linalg.inv(m) for m in -2.0 * theta2])
        S_new = 0.5 * (S_new + S_new.transpose(1, 2))
        out.append(((S_new @ theta1).squeeze(-1).T.contiguous(), torch.linalg.cholesky(S_new)))
    return out


class AdamOracle:
    """tf.optimizers.Adam(lr, beta_1, beta_2, epsilon) on the GPflow variables of a model, minimising -ELBO (reference
    models/dgp.py:132-154: optimizer.apply_gradients(zip(tape.gradient(-ELBO, trainable_variables), trainable_variables))).
    GPflow stores UNCONSTRAINED variables: softplus^-1(value) for kernel lengthscales / variance (positive()),
    softplus^-1(value - 1e-6) for the Gaussian likelihood variance, the lower-triangle entries of q_sqrt (FillTriangular; kept
    here as a full matrix whose upper triangle never receives gradient), identity for Z and q_mu. The variables persist across
    steps, constrained values are rebuilt from them, and the gradient w.r.t. the variables is taken by autograd THROUGH the
    bijectors -- the product instead inverts the bijector every step and applies the chain rule in closed form.
    Keras Adam: lr_t = lr sqrt(1 - b2^t) / (1 - b1^t); m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2; u -= lr_t m / (sqrt(v) + eps)."""

    BIJECTOR = {"Z": "identity", "lengthscales": "positive", "variance": "positive", "q_mu": "identity", "q_sqrt": "triangular",
                "lik_var": "positive_shift"}

    def __init__(self, model: OModel, lr=0.01, beta_1=0.9, beta_2=0.999, epsilon=1e-7, names: Optional[Sequence[str]] = None):
        self.lr, self.b1, self.b2, self.eps, self.t = lr, beta_1, beta_2, epsilon, 0
        params = model.named_params()
        self.names = list(params) if names is None else list(names)
        self.u = {k: self._inverse(k, params[k].detach().clone()) for k in self.names}
        self.m = {k: torch.zeros_like(v) for k, v in self.u.items()}
        self.v = {k: torch.zeros_like(v) for k, v in self.u.items()}

    @classmethod
    def _kind(cls, name):
        return cls.BIJECTOR[name.split(".")[-1]]

    @classmethod
    def _inverse(cls, name, value):
        kind = cls._kind(name)
        if kind in ("positive", "positive_shift"):
            y = value - (1e-6 if kind == "positive_shift" else 0.0)
            return y + torch.log(-torch.expm1(-y))
        return value

    @classmethod
    def _forward(cls, name, u):
        kind = cls._kind(name)
        if kind in ("positive", "positive_shift"):
            return torch.logaddexp(u, torch.zeros_like(u)) + (1e-6 if kind == "positive_shift" else 0.0)
        if kind == "triangular":
            return torch.tril(u)
        return u

    def step(self, model: OModel, X, Y, zs, scale: float = 1.0):
        """One apply_gradients; returns (the step's ELBO, a new OModel holding the updated constrained values)."""
        params = model.named_params()
        leaves = {k: self.u[k].detach().clone().requires_grad_(True) for k in self.names}
        val = {k: (self._forward(k, leaves[k]) if k in leaves else params[k].detach()) for k in params}
        layers = [OLayer(Z=val[f"layers.{i}.Z"], lengthscales=val[f"layers.{i}.lengthscales"], variance=val[f"layers.{i}.variance"],
                         q_mu=val[f"layers.{i}.q_mu"], q_sqrt=val[f"layers.{i}.q_sqrt"], mean_kind=l.mean_kind, mf_W=l.mf_W,
                         mf_b=l.mf_b, white=l.white, kernel_kind=l.kernel_kind) for i, l in enumerate(model.layers)]
        value = elbo(OModel(layers=layers, lik_var=val["lik_var"], num_samples=model.num_samples), X, Y, zs, scale)
        (-value).backward()
        self.t += 1
        lr_t = self.lr * np.sqrt(1.0 - self.b2 ** self.t) / (1.0 - self.b1 ** self.t)
        for k in self.names:
            g = leaves[k].grad
            self.m[k] = self.b1 * self.m[k] + (1.0 - self.b1) * g
            self.v[k] = self.b2 * self.v[k] + (1.0 - self.b2) * g * g
            self.u[k] = self.u[k] - lr_t * self.m[k] / (torch.sqrt(self.v[k]) + self.eps)
        new = {k: (self._forward(k, self.u[k]).detach() if k in self.u else params[k].detach()) for k in params}
        out = OModel(layers=[OLayer(Z=new[f"layers.{i}.Z"], lengthscales=new[f"layers.{i}.lengthscales"],
                                    variance=new[f"layers.{i}.variance"], q_mu=new[f"layers.{i}.q_mu"],
                                    q_sqrt=new[f"layers.{i}.q_sqrt"], mean_kind=l.mean_kind, mf_W=l.mf_W, mf_b=l.mf_b,
                                    white=l.white, kernel_kind=l.kernel_kind) for i, l in enumerate(model.layers)],
                     lik_var=new["lik_var"], num_samples=model.num_samples)
        return value.detach(), out


# --------------------------------------------------------------------------------------
# parameter transforms kept host-side (SURVEY §9)
# --------------------------------------------------------------------------------------
def softplus(u):
    return np.logaddexp(0.0, u)


def softplus_inv(theta):
    return theta + np.log(-np.expm1(-theta))


def softplus_grad_from_constrained(theta):
    """d theta / d u for theta = softplus(u): 1 - exp(-theta)."""
    return -np.expm1(-theta)


def fill_triangular(x: np.ndarray) -> np.ndarray:
    """tfp.bijectors.FillTriangular (lower): x has length n(n+1)/2; concat([x[n:], reverse(x)]) -> [n,n] -> lower band."""
    m = x.shape[-1]
    n = int(round((math.sqrt(8 * m + 1) - 1) / 2))
    assert n * (n + 1) // 2 == m
    y = np.concatenate([x[..., n:], x[..., ::-1]], axis=-1).reshape(x.shape[:-1] + (n, n))
    return np.tril(y)


def fill_triangular_inverse(L: np.ndarray) -> np.ndarray:
    """Inverse of fill_triangular (tfp FillTriangular.inverse)."""
    n = L.shape[-1]
    m = n * (n + 1) // 2
    idx = fill_triangular(np.arange(1, m + 1, dtype=np.float64))  # 1-based positions, 0 above the diagonal
    out = np.zeros(L.shape[:-2] + (m,), dtype=L.dtype)
    ii, jj = np.nonzero(idx)
    out[..., (idx[ii, jj] - 1).astype(int)] = L[..., ii, jj]
    return out


# --------------------------------------------------------------------------------------
# Philox-4x32-10 + Box-Muller: the draw layout the CUDA kernels use (bit-exact integer plumbing)
# --------------------------------------------------------------------------------------
_PH_M0, _PH_M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_PH_W0, _PH_W1 = np.uint32(0x9E3779B9), np.uint32(0xBB67AE85)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Vectorised Philox-4x32-10 (Salmon et al. 2011). All inputs uint32 arrays (broadcastable); returns 4 uint32 arrays."""
    c0, c1, c2, c3 = [np.asarray(c, dtype=np.uint32) for c in (c0, c1, c2, c3)]
    c0, c1, c2, c3 = np.broadcast_arrays(c0, c1, c2, c3)
    k0 = np.uint32(k0)
    k1 = np.uint32(k1)
    with np.errstate(over="ignore"):
        for _ in range(10):
            p0 = c0.astype(np.uint64) * _PH_M0
            p1 = c2.astype(np.uint64) * _PH_M1
            hi0 = (p0 >> np.uint64(32)).astype(np.uint32)
            lo0 = p0.astype(np.uint32)
            hi1 = (p1 >> np.uint64(32)).astype(np.uint32)
            lo1 = p1.astype(np.uint32)
            c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
            k0 = np.uint32(k0 + _PH_W0)
            k1 = np.uint32(k1 + _PH_W1)
    return c0, c1, c2, c3


def philox_uint32(seed: int, layer: int, S: int, N: int, D: int, n_offset: int = 0):
    """Raw Philox words for element (layer, s, n, d): key = (seed_lo, seed_hi), counter = (n_global, s, d, layer).
    Returns uint32 array [S, N, D, 4]. n_offset shifts n to the global point index (multi-GPU shards)."""
    s = np.arange(S, dtype=np.uint32)[:, None, None]
    n = (np.arange(N, dtype=np.uint64) + np.uint64(n_offset)).astype(np.uint32)[None, :, None]
    d = np.arange(D, dtype=np.uint32)[None, None, :]
    r = philox4x32_10(n, s, d, np.uint32(layer), seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    return np.stack(r, axis=-1)


def philox_normal(seed: int, layer: int, S: int, N: int, D: int, n_offset: int = 0) -> np.ndarray:
    """z[s,n,d] = sqrt(-2 ln u1) cos(2 pi u2), u = ((hi >> 5) * 2^26 + (lo >> 6) + 0.5) / 2^53 from words (0,1) and (2,3)."""
    r = philox_uint32(seed, layer, S, N, D, n_offset).astype(np.uint64)
    u1 = ((r[..., 0] >> np.uint64(5)) * np.uint64(67108864) + (r[..., 1] >> np.uint64(6))).astype(np.float64)
    u2 = ((r[..., 2] >> np.uint64(5)) * np.uint64(67108864) + (r[..., 3] >> np.uint64(6))).astype(np.float64)
    u1 = (u1 + 0.5) / 9007199254740992.0
    u2 = (u2 + 0.5) / 9007199254740992.0
    return np.sqrt(-2.0 * np.log(u1)) * np.cos(2.0 * np.pi * u2)


# --------------------------------------------------------------------------------------
# acquisition search (reference Infill_criteria.py:61-87): differential evolution, then Adam, on u with
# x = lw + (up - lw) / (1 + exp(u))
# --------------------------------------------------------------------------------------
def box_from_u(u, lw, up):
    return lw + (up - lw) / (1.0 + np.exp(u))


def de_choices(seed: int, generation: int, pop: int, d: int):
    """Random choices of one generation, the word layout of csrc/acq.cuh: Philox key = seed, counter = (member, generation,
    slot, 0xDE). Slot 0 -> partners a, b, c (distinct, != member: w_k mod (pop-1-k), then skipping the excluded indices in
    ascending order) and the forced dimension w3 mod d; slot 1 + j // 4, word j % 4 -> uniform (w + 0.5) / 2^32 of dimension j.
    Returns (a, b, c, forced) int arrays [pop] and uniforms [pop, d]."""
    i = np.arange(pop, dtype=np.uint32)
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    w = philox4x32_10(i, np.uint32(generation), np.uint32(0), np.uint32(0xDE), k0, k1)

    def skip(v, excl):
        v = v.copy()
        for e in excl:            # ascending per member
            v = v + (v >= e)
        return v

    ii = np.arange(pop)
    a = skip((w[0] % np.uint32(pop - 1)).astype(np.int64), [ii])
    lo, hi = np.minimum(ii, a), np.maximum(ii, a)
    b = skip((w[1] % np.uint32(pop - 2)).astype(np.int64), [lo, hi])
    e = np.sort(np.stack([ii, a, b], 1), axis=1)
    c = skip((w[2] % np.uint32(pop - 3)).astype(np.int64), [e[:, 0], e[:, 1], e[:, 2]])
    forced = (w[3] % np.uint32(d)).astype(np.int64)
    uni = np.empty((pop, d))
    for j in range(d):
        r = philox4x32_10(i, np.uint32(generation), np.uint32(1 + j // 4), np.uint32(0xDE), k0, k1)
        uni[:, j] = (r[j % 4].astype(np.float64) + 0.5) / 4294967296.0
    return a, b, c, forced, uni


def de_minimize(objective, lw, up, pop_u0, iterations: int, seed: int, weight: float = 0.5, crossover: float = 0.9):
    """tfp.optimizer.differential_evolution_minimize restated ("rand/1/bin", TFP defaults weight 0.5 / crossover 0.9; TFP itself
    is not in this image -- published algorithm: Storn & Price 1997, TFP API docs): every generation builds one candidate per
    member, pop[a] + weight (pop[b] - pop[c]) on the crossed-over dimensions, evaluates the whole candidate population at once and
    keeps the strictly better of (member, candidate). objective(x [pop, d], generation) -> [pop] values; generation 0 is the
    evaluation of the initial population. Returns (population_u, values)."""
    lw, up = np.asarray(lw, dtype=np.float64), np.asarray(up, dtype=np.float64)
    pop_u = np.array(pop_u0, dtype=np.float64)
    pop, d = pop_u.shape
    vals = np.asarray(objective(box_from_u(pop_u, lw, up), 0), dtype=np.float64).reshape(pop)
    for g in range(1, iterations + 1):
        a, b, c, forced, uni = de_choices(seed, g, pop, d)
        mutant = pop_u[a] + weight * (pop_u[b] - pop_u[c])
        take = uni < crossover
        take[np.arange(pop), forced] = True
        cand = np.where(take, mutant, pop_u)
        cv = np.asarray(objective(box_from_u(cand, lw, up), g), dtype=np.float64).reshape(pop)
        better = cv < vals
        pop_u[better] = cand[better]
        vals[better] = cv[better]
    return pop_u, vals


def adam_box_minimize(value_and_grad, lw, up, u0, iterations: int, lr=0.01, beta_1=0.9, beta_2=0.999, epsilon=1e-7):
    """tf.optimizers.Adam on u (Infill_criteria.py:72-86); value_and_grad(u, step) -> (value, d value / d u) with the gradient
    taken by autograd through x = lw + (up - lw) / (1 + exp(u)). Returns (u, last value)."""
    u = np.array(u0, dtype=np.float64)
    m, v = np.zeros_like(u), np.zeros_like(u)
    val = None
    for t in range(1, iterations + 1):
        val, g = value_and_grad(u, t - 1)
        m = beta_1 * m + (1.0 - beta_1) * g
        v = beta_2 * v + (1.0 - beta_2) * g * g
        u = u - lr * np.sqrt(1.0 - beta_2 ** t) / (1.0 - beta_1 ** t) * m / (np.sqrt(v) + epsilon)
    return u, val


# --------------------------------------------------------------------------------------
# synthetic benchmark inputs (SURVEY §8d) shared by tests and bench.py's cpu_baseline leg
# --------------------------------------------------------------------------------------
def synthetic_problem(D0, num_units, M, N, seed_shift=0, lik_var=0.1, ls_scale=1.0):
    """X ~ N(0,I), Y = sin(sum x / sqrt(D0)) + 0.1 eps, Z_l ~ N(0,I), l = sqrt(D_in), sigma^2 = 1,
    q_mu = 0.1 N(0,1), q_sqrt = 0.5 I + 0.05 tril(N(0,1)). ls_scale shrinks the lengthscales for low-dimensional
    problems, where l = sqrt(D_in) would make cond(Ku) jitter-limited (~1e7) and 1e-9 parity meaningless. Returns numpy dict."""
    rng = np.random.default_rng(0 + seed_shift)
    X = rng.standard_normal((N, D0))
    Y = np.sin(X.sum(1, keepdims=True) / math.sqrt(D0)) + 0.1 * np.random.default_rng(1 + seed_shift).standard_normal((N, 1))
    dims = [D0] + list(num_units) + [1]
    layers = []
    for l, (din, dout) in enumerate(zip(dims[:-1], dims[1:])):
        Z = np.random.default_rng(10 + l + seed_shift).standard_normal((M, din))
        q_mu = 0.1 * np.random.default_rng(20 + l + seed_shift).standard_normal((M, dout))
        R = np.random.default_rng(30 + l + seed_shift).standard_normal((dout, M, M))
        q_sqrt = 0.5 * np.eye(M)[None] + 0.05 * np.tril(R)
        last = l == len(dims) - 2
        if last:
            kind, W = "zero", None
        elif din == dout:
            kind, W = "identity", None
        elif din > dout:
            _, _, V = np.linalg.svd(X if l == 0 else rng.standard_normal((max(N, din), din)), full_matrices=False)
            kind, W = "linear", V[:dout, :].T
        else:
            kind, W = "linear", np.concatenate([np.eye(din), np.zeros((din, dout - din))], 1)
        layers.append(dict(Z=Z, lengthscales=np.full(din, ls_scale * math.sqrt(din)), variance=1.0, q_mu=q_mu, q_sqrt=q_sqrt,
                           mean_kind=kind, mf_W=W, mf_b=None if W is None else np.zeros(dout)))
    return dict(X=X, Y=Y, layers=layers, lik_var=lik_var)


def model_from_problem(prob, num_samples) -> OModel:
    layers = [make_layer(l["Z"], l["lengthscales"], l["variance"], l["q_mu"].shape[1], l["mean_kind"], l["mf_W"],
                         l["mf_b"], bool(l.get("white", False)), l["q_mu"], l["q_sqrt"], l.get("kernel", "rbf")) for l in prob["layers"]]
    return OModel(layers=layers, lik_var=_t(prob["lik_var"]).reshape(()), num_samples=num_samples)
