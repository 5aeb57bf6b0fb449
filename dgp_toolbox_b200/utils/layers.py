"""Layer / SVGP_Layer with the reference's interface (dgp_dace/utils/layers.py:47-130,180-308); the arithmetic of
every method runs in libdgp_b200 (CUDA, sm_100a) through the C ABI — there is no torch/numpy fallback."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from .. import _lib
from .. import gpflow_shim as gpflow
from ..gpflow_shim import Parameter, _Module


class Layer(_Module):
    """dgp_dace/utils/layers.py:47-130."""

    def __init__(self, input_prop_dim=None, **kwargs):
        if input_prop_dim:
            raise NotImplementedError("input_prop_dim is never enabled by the reference constructors (SURVEY §8 a6)")
        self.input_prop_dim = input_prop_dim

    def conditional_ND(self, X, full_cov=False):
        raise NotImplementedError

    def _desc(self):
        raise NotImplementedError

    def KL(self):
        return torch.zeros((), dtype=torch.float64)

    def conditional_SND(self, X, full_cov=False):
        """:63-85. [S,N,D_in] -> flatten (p = s*N + n) -> conditional_ND -> [S,N,D_out]; full_cov=True maps conditional_ND over the
        samples (:76-80) -> mean [S,N,D_out], var [S,N,N,D_out]. Host inputs go to the device the layer's parameters live on."""
        X = _lib.as_device(X, self.feature.Z.value.device)
        S, N, D = X.shape
        if full_cov:
            _, mean, var = self._propagate_full(X.contiguous(), S, None, 0, want_sample=False)
            return [mean, var]
        mean, var = self.conditional_ND(X.reshape(S * N, D))
        return [m.reshape(S, N, self.num_outputs) for m in (mean, var)]

    def sample_from_conditional(self, X, z=None, full_cov=False, seed=0, layer_index=0):
        """:87-130. z=None draws from the library's Philox-4x32-10 stream (counter = (n, s, d, layer_index))."""
        X = _lib.as_device(X, self.feature.Z.value.device)
        S, N, _ = X.shape
        D = self.num_outputs
        ctx = _lib.get_context(X.device)
        if full_cov:
            # per sample: full N x N covariance per output and the Cholesky reparameterisation (utils/utils.py:43-52), all S
            # samples in one call. Without z, sample s draws the stream of seed + s (counter (n, 0, d, 0)), as one call per sample did.
            if z is None:
                z = torch.empty((S, N, D), dtype=torch.float64, device=X.device)
                for s in range(S if N else 0):
                    ctx.call("dgp_philox_normal", int(seed) + s, 0, 1, N, D, 0, _lib.ptr(z[s]))
            else:
                z = _lib.as_device(z, X.device).reshape(S, N, D).contiguous()
            return self._propagate_full(X.contiguous(), S, [z], 0)
        if z is None:
            z = torch.empty((S, N, D), dtype=torch.float64, device=X.device)
            ctx.call("dgp_philox_normal", int(seed), int(layer_index), S, N, D, 0, _lib.ptr(z))
        else:
            z = _lib.as_device(z, X.device).reshape(S, N, D)
        # one-layer chain over the S*N flattened rows (p = s*N + n) with the draws supplied explicitly:
        # conditional + reparameterisation (utils/utils.py:40-41) run fused in the library
        samples = torch.empty((S, N, D), dtype=torch.float64, device=X.device)
        mean, var = torch.empty_like(samples), torch.empty_like(samples)
        d, keep = self._desc()
        m = _lib.ModelDesc(1, C.pointer(d), None)
        ctx.call("dgp_propagate", C.byref(m), _lib.ptr(X), S * N, 1, _lib.ptr_array([z]), 0, 0,
                 _lib.ptr_array([samples]), _lib.ptr_array([mean]), _lib.ptr_array([var]))
        return samples, mean, var


class SVGP_Layer(Layer):
    """dgp_dace/utils/layers.py:180-308 (augmented=False). white=True is the whitened representation q(v) = N(q_mu, q_sqrt q_sqrt^T),
    u = Lu v (:246,254-255,296-303); the reference default is white=False."""

    def __init__(self, kern, Z, num_outputs, mean_function, augmented=False, layers=None, white=False,
                 input_prop_dim=None, **kwargs):
        Layer.__init__(self, input_prop_dim)
        if augmented:
            raise NotImplementedError("augmented inducing inputs belong to the MF/MO models (SURVEY §8 f2)")
        Z = np.asarray(Z.detach().cpu().numpy() if hasattr(Z, "detach") else Z, dtype=np.float64)
        self.num_inducing = Z.shape[0]
        self.num_outputs = int(num_outputs)
        self.white = white
        self.kern = kern
        self.mean_function = mean_function
        self.feature = InducingPoints(Z)
        self.q_mu = Parameter(np.zeros((self.num_inducing, self.num_outputs)), name="q_mu")
        if white:      # q(v) = N(0, I)   (:203-206)
            self.q_sqrt = Parameter(np.tile(np.eye(self.num_inducing)[None], (self.num_outputs, 1, 1)), transform="triangular",
                                    name="q_sqrt")
        else:          # q(u) initialised to the prior, q_sqrt = chol(K(Z) + jitter I)   (:219-223)
            _, Lu = self._kuu_chol()
            self.q_sqrt = Parameter(Lu[None].repeat(self.num_outputs, 1, 1), transform="triangular", name="q_sqrt")
        self.needs_build_cholesky = True

    # ---- descriptor handed to the C ABI (pointers into the Parameter tensors) ----
    def _desc(self, need_q=True):
        Z = self.feature.Z.value
        M, D_in = Z.shape
        keep = [Z]
        ls = self.kern.lengthscales_vector(D_in)
        var = self.kern.variance.value.reshape(1)
        keep += [ls, var]
        d = _lib.LayerDesc()
        d.D_in, d.D_out, d.M = D_in, self.num_outputs, M
        d.white = 1 if self.white else 0
        d.mean_kind = self.mean_function.mean_kind
        d.kernel_kind = self.kern.kernel_kind
        d.Z, d.lengthscales, d.variance = Z.data_ptr(), ls.data_ptr(), var.data_ptr()
        if need_q:
            d.q_mu, d.q_sqrt = self.q_mu.value.data_ptr(), self.q_sqrt.value.data_ptr()
        else:  # constructor: q not built yet; any valid buffer satisfies the null check
            dummy = torch.zeros(max(M * M, M) * self.num_outputs, dtype=torch.float64, device=Z.device)
            keep.append(dummy)
            d.q_mu, d.q_sqrt = dummy.data_ptr(), dummy.data_ptr()
        if d.mean_kind == 2:
            W = self.mean_function.A.value.contiguous()
            b = self.mean_function.b.value.contiguous()
            if tuple(W.shape) != (D_in, self.num_outputs):
                raise ValueError(f"Linear mean function A has shape {tuple(W.shape)}, expected {(D_in, self.num_outputs)}")
            keep += [W, b]
            d.mf_W, d.mf_b = W.data_ptr(), b.data_ptr()
        d.jitter = gpflow.default_jitter()
        return d, keep

    def _kuu_chol(self):
        Z = self.feature.Z.value
        M = Z.shape[0]
        Ku = torch.empty((M, M), dtype=torch.float64, device=Z.device)
        Lu = torch.empty_like(Ku)
        d, keep = self._desc(need_q=hasattr(self, "q_sqrt"))
        _lib.get_context(Z.device).call("dgp_kuu_chol", C.byref(d), _lib.ptr(Ku), _lib.ptr(Lu))
        return Ku, Lu

    def build_cholesky_if_needed(self):
        """:227-234. Ku = Kuu + jitter I, Lu = chol(Ku) (recomputed on every call, like the reference)."""
        self.Ku, self.Lu = self._kuu_chol()
        self.Ku_tiled = self.Ku[None].expand(self.num_outputs, -1, -1)
        self.Lu_tiled = self.Lu[None].expand(self.num_outputs, -1, -1)
        self.needs_build_cholesky = False

    def conditional_ND(self, X, full_cov=False):
        """:237-278: X [P, D_in] -> mean [P, D_out] (includes the mean function) and var [P, D_out], or with full_cov=True the
        covariance [P, P, D_out] (:264-268,276)."""
        X = _lib.as_device(X, self.feature.Z.value.device)
        P = X.shape[0]
        if full_cov:
            _, mean, var = self._propagate_full(X, 1, None, 0, want_sample=False)
            return mean[0], var[0]
        mean = torch.empty((P, self.num_outputs), dtype=torch.float64, device=X.device)
        var = torch.empty_like(mean)
        if P == 0:
            return mean, var
        d, keep = self._desc()
        _lib.get_context(X.device).call("dgp_conditional_nd", C.byref(d), _lib.ptr(X), P, _lib.ptr(mean), _lib.ptr(var))
        return mean, var

    def _propagate_full(self, X, S, zs, seed, want_sample=True):
        """One-layer full_cov call: X [N, D_in] shared by the S samples (dgp_propagate_full_cov) or X [S, N, D_in] per sample
        (dgp_propagate_full_cov_snd) -> (F, mean [S,N,D], var [S,N,N,D])."""
        N, D = X.shape[-2], self.num_outputs
        mean = torch.empty((S, N, D), dtype=torch.float64, device=X.device)
        var = torch.empty((S, N, N, D), dtype=torch.float64, device=X.device)
        F = torch.empty((S, N, D), dtype=torch.float64, device=X.device) if want_sample else None
        if N == 0:
            return F, mean, var
        d, keep = self._desc()
        m = _lib.ModelDesc(1, C.pointer(d), None)
        zp = _lib.ptr_array(zs) if zs is not None else None
        fn = "dgp_propagate_full_cov_snd" if X.dim() == 3 else "dgp_propagate_full_cov"
        _lib.get_context(X.device).call(fn, C.byref(m), _lib.ptr(X), N, S, zp, int(seed), 0,
                                        _lib.ptr_array([F]), _lib.ptr_array([mean]), _lib.ptr_array([var]))
        return F, mean, var

    def KL(self):
        """:280-308 -> 0-d tensor."""
        out = torch.empty(1, dtype=torch.float64, device=self.feature.Z.value.device)
        d, keep = self._desc()
        _lib.get_context(out.device).call("dgp_kl", C.byref(d), _lib.ptr(out))
        return out.reshape(())


class InducingPoints(_Module):
    """gpflow.inducing_variables.InducingPoints: holds Z [M, D_in]."""

    def __init__(self, Z):
        self.Z = Parameter(Z, name="Z")

    def __len__(self):
        return self.Z.shape[0]
