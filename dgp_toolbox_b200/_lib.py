"""ctypes binding of libdgp_b200.so (C ABI in include/dgp_b200.h).

The product path has no CPU fallback: importing this module without the built library, or creating a
context without an sm_100 GPU, raises. Device memory, streams and DLPack exchange are torch's job
(plumbing); every flop of the DGP hot path runs inside the library's CUDA kernels.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DGP_B200_LIB") or os.path.join(_HERE, "libdgp_b200.so")   # env override: A/B builds

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(nvcc -gencode arch=compute_100a,code=sm_100a). dgp_toolbox_b200 has no CPU fallback.")

lib = C.CDLL(LIB_PATH)

c_double_p = C.POINTER(C.c_double)


class LayerDesc(C.Structure):
    _fields_ = [("D_in", C.c_int32), ("D_out", C.c_int32), ("M", C.c_int32), ("white", C.c_int32),
                ("mean_kind", C.c_int32), ("kernel_kind", C.c_int32),
                ("Z", C.c_void_p), ("lengthscales", C.c_void_p), ("variance", C.c_void_p),
                ("q_mu", C.c_void_p), ("q_sqrt", C.c_void_p), ("mf_W", C.c_void_p), ("mf_b", C.c_void_p),
                ("jitter", C.c_double)]


class ModelDesc(C.Structure):
    _fields_ = [("num_layers", C.c_int32), ("layers", C.POINTER(LayerDesc)), ("lik_variance", C.c_void_p)]


class GradOffsets(C.Structure):
    _fields_ = [("dZ", C.c_int64), ("dlengthscales", C.c_int64), ("dvariance", C.c_int64),
                ("dq_mu", C.c_int64), ("dq_sqrt", C.c_int64)]


class AdamParam(C.Structure):
    _fields_ = [("value", C.c_void_p), ("count", C.c_int64), ("grad_offset", C.c_int64), ("grad_count", C.c_int64),
                ("transform", C.c_int32), ("M", C.c_int32), ("mirror", C.c_void_p), ("mirror_count", C.c_int64)]


class NatPair(C.Structure):       # dgp_nat_pair
    _fields_ = [("q_mu", C.c_void_p), ("q_sqrt", C.c_void_p), ("g_mu", C.c_void_p), ("g_sqrt", C.c_void_p), ("M", C.c_int32),
                ("D_out", C.c_int32)]


_vp, _i, _i64, _u64, _d = C.c_void_p, C.c_int, C.c_int64, C.c_uint64, C.c_double
_SIG = {
    "dgp_version": (C.c_int, []),
    "dgp_ctx_create": (C.c_int, [_i, _vp, C.POINTER(_vp)]),
    "dgp_ctx_destroy": (None, [_vp]),
    "dgp_last_error": (C.c_char_p, [_vp]),
    "dgp_set_stream": (C.c_int, [_vp, _vp]),
    "dgp_check": (C.c_int, [_vp]),
    "dgp_workspace_bytes": (_i64, [_vp]),
    "dgp_set_workspace_limit": (C.c_int, [_vp, _i64]),
    "dgp_launch_count": (_i64, [_vp, _i]),
    "dgp_set_profiling": (C.c_int, [_vp, _i]),
    "dgp_set_fused": (C.c_int, [_vp, _i]),
    "dgp_set_graph": (C.c_int, [_vp, _i]),
    "dgp_set_share_first_layer": (C.c_int, [_vp, _i]),
    "dgp_set_vform": (C.c_int, [_vp, _i, _i]),
    "dgp_set_parallel_layers": (C.c_int, [_vp, _i]),
    "dgp_get_profile": (C.c_int, [_vp, _vp, _vp, _i]),
    "dgp_philox_normal": (C.c_int, [_vp, _u64, _i, _i64, _i64, _i, _i64, _vp]),
    "dgp_philox_raw": (C.c_int, [_vp, _u64, _i, _i64, _i64, _i, _i64, _vp]),
    "dgp_kernel_K": (C.c_int, [_vp, _i, _i, _vp, _vp, _vp, _i64, _vp, _i64, _vp]),
    "dgp_kuu_chol": (C.c_int, [_vp, C.POINTER(LayerDesc), _vp, _vp]),
    "dgp_conditional_nd": (C.c_int, [_vp, C.POINTER(LayerDesc), _vp, _i64, _vp, _vp]),
    "dgp_kl": (C.c_int, [_vp, C.POINTER(LayerDesc), _vp]),
    "dgp_propagate": (C.c_int, [_vp, C.POINTER(ModelDesc), _vp, _i64, _i64, C.POINTER(_vp), _u64, _i64,
                                C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)]),
    "dgp_grad_size": (_i64, [C.POINTER(ModelDesc)]),
    "dgp_grad_layout": (C.c_int, [C.POINTER(ModelDesc), C.POINTER(GradOffsets)]),
    "dgp_elbo_grad": (C.c_int, [_vp, C.POINTER(ModelDesc), _vp, _vp, _i64, _i64, _d, _d, C.POINTER(_vp), _u64, _i64,
                                _i, _vp]),
    "dgp_elbo_grad_host": (C.c_int, [_vp, C.POINTER(ModelDesc), _vp, _vp, _i64, _i64, _d, _d, _u64, _i64, _i, _vp]),
    "dgp_adam_step": (C.c_int, [_vp, C.POINTER(AdamParam), _i, _vp, _vp, _vp, _i64, _d, _d, _d, _d]),
    "dgp_train_adam": (C.c_int, [_vp, C.POINTER(ModelDesc), _vp, _vp, _i64, _i64, _d, _d, _u64, _u64, _i64, C.POINTER(AdamParam), _i,
                                 _vp, _vp, _i64, _i64, _d, _d, _d, _d, _vp, _vp]),
    "dgp_comp_K": (C.c_int, [_vp, _vp, _vp, _i64, _vp, _i64, _vp]),
    "dgp_comp_Kdiag": (C.c_int, [_vp, _vp, _vp, _i64, _vp]),
    "dgp_comp_K_blocks": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _vp]),
    "dgp_comp_K_grad": (C.c_int, [_vp, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp]),
    "dgp_comp_Kdiag_grad": (C.c_int, [_vp, _vp, _vp, _i64, _vp, _vp, _vp]),
    "dgp_svgp_from_k": (C.c_int, [_vp, _i, _i, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "dgp_svgp_from_k_grad": (C.c_int, [_vp, _i, _i, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _d, _vp, _vp, _vp, _vp, _vp]),
    "dgp_svgp_prep_cache_bytes": (_i64, [_vp, _i, _i]),
    "dgp_svgp_stash_bytes": (_i64, [_i, _i, _i64]),
    "dgp_svgp_from_k_cached": (C.c_int, [_vp, _i, _i, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i, _vp]),
    "dgp_svgp_from_k_grad_cached": (C.c_int, [_vp, _i, _i, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _d, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "dgp_svgp_from_k_full_cov": (C.c_int, [_vp, _i, _i, _i64, _i64, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _d, _vp, _vp, _vp]),
    "dgp_comm_unique_id": (C.c_int, [_vp]),
    "dgp_comm_init": (C.c_int, [_vp, _i, _i, _vp]),
    "dgp_allreduce_grads": (C.c_int, [_vp, _vp, _i64]),
    "dgp_comm_destroy": (C.c_int, [_vp]),
    "dgp_elbo_grad_sharded": (C.c_int, [_vp, C.POINTER(ModelDesc), _vp, _vp, _i64, _i64, _d, _u64, _i64, _i, _vp]),
    "dgp_natgrad_step": (C.c_int, [_vp, C.POINTER(ModelDesc), C.POINTER(C.c_int), _i, _d, _vp]),
    "dgp_natgrad_pairs": (C.c_int, [_vp, C.POINTER(NatPair), _i, _d]),
    "dgp_train_nat_adam": (C.c_int, [_vp, C.POINTER(ModelDesc), _vp, _vp, _i64, _i64, _d, _d, _u64, _u64, _i64, C.POINTER(AdamParam), _i,
                                     _vp, _vp, _i64, _i64, _d, _d, _d, _d, C.POINTER(C.c_int), _i, _d, _vp, _vp]),
    "dgp_propagate_full_cov": (C.c_int, [_vp, C.POINTER(ModelDesc), _vp, _i64, _i64, C.POINTER(_vp), _u64, _i64, C.POINTER(_vp),
                                         C.POINTER(_vp), C.POINTER(_vp)]),
    "dgp_propagate_full_cov_snd": (C.c_int, [_vp, C.POINTER(ModelDesc), _vp, _i64, _i64, C.POINTER(_vp), _u64, _i64, C.POINTER(_vp),
                                             C.POINTER(_vp), C.POINTER(_vp)]),
    "dgp_propagate_grouped_cov": (C.c_int, [_vp, C.POINTER(ModelDesc), _vp, _i64, _i64, _i, C.POINTER(_vp), _u64, _i64,
                                            C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)]),
    "dgp_qei": (C.c_int, [_vp, C.POINTER(ModelDesc), _vp, _i64, _i64, _i, C.POINTER(_vp), _u64, _i64, _d, _vp]),
    "dgp_e_log_p_y": (C.c_int, [_vp, C.POINTER(ModelDesc), _vp, _vp, _i64, _i64, C.POINTER(_vp), _u64, _i64, _vp]),
    "dgp_predict_moments": (C.c_int, [_vp, C.POINTER(ModelDesc), _vp, _i64, _i64, C.POINTER(_vp), _u64, _i64, _i,
                                      _vp, _vp]),
    "dgp_ei": (C.c_int, [_vp, C.POINTER(ModelDesc), _vp, _i64, _i64, C.POINTER(_vp), _u64, _i64, _d, _i, _vp]),
    "dgp_ei_grad": (C.c_int, [_vp, C.POINTER(ModelDesc), _vp, _i64, _i64, C.POINTER(_vp), _u64, _i64, _d, _vp, _vp]),
    "dgp_acq_grad": (C.c_int, [_vp, C.POINTER(ModelDesc), _i, _vp, _i64, _i64, C.POINTER(_vp), _u64, _i64, _d, _vp, _vp]),
    "dgp_acq_moments": (C.c_int, [_vp, _i, _vp, _vp, _i64, _d, _vp, _i, _vp]),
    "dgp_de_propose": (C.c_int, [_vp, _vp, _i64, _i, _vp, _vp, _u64, _i64, _d, _d, _vp, _vp]),
    "dgp_de_select": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _i]),
    "dgp_box_from_u": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i, _vp]),
    "dgp_adam_box_step": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i, _i64, _d, _d, _d, _d, _vp]),
    "dgp_ev_mc": (C.c_int, [_vp, _vp, _i64, _i64, _d, _vp]),
    "dgp_mixture_moments": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp]),
    "dgp_ehvi2d": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _i, _vp]),
    "dgp_ehvi2d_grad": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _i, _vp, _vp]),
    "dgp_debug_gemm": (C.c_int, [_vp, _i, _i, _i, _i, _d, _vp, _vp, _d, _vp, _i, _i, _i, _i, _vp]),
}
for _name, (_res, _args) in _SIG.items():
    _f = getattr(lib, _name)
    _f.restype = _res
    _f.argtypes = _args

EXPORTED_SYMBOLS = tuple(_SIG)


class DGPError(RuntimeError):
    pass


class Context:
    """One dgp_ctx per (process, device). Not thread-safe; calls are asynchronous on torch's current stream."""

    def __init__(self, device: int):
        if not torch.cuda.is_available():
            raise DGPError("dgp_toolbox_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.device = device
        h = _vp()
        with torch.cuda.device(device):
            torch.cuda.current_stream()  # make sure the primary context exists
            rc = lib.dgp_ctx_create(device, _vp(torch.cuda.current_stream(device).cuda_stream), C.byref(h))
        if rc != 0:
            raise DGPError(f"dgp_ctx_create(device={device}) failed with code {rc} "
                           "(-3: device is not sm_100; -1: CUDA error)")
        self.h = h
        self.graph = False

    def call(self, name, *args):
        lib.dgp_set_stream(self.h, _vp(torch.cuda.current_stream(self.device).cuda_stream))
        rc = getattr(lib, name)(self.h, *args)
        if rc != 0:
            raise DGPError(f"{name} failed ({rc}): {lib.dgp_last_error(self.h).decode()}")

    def check(self):
        """Synchronise and raise if an asynchronous call hit a non-positive-definite Kuu."""
        rc = lib.dgp_check(self.h)
        if rc != 0:
            raise DGPError(f"dgp_check ({rc}): {lib.dgp_last_error(self.h).decode()}")

    def launch_count(self, reset=False) -> int:
        return int(lib.dgp_launch_count(self.h, 1 if reset else 0))

    PROFILE_CATEGORIES = ("prep", "kuf", "gemm_fwd", "moments", "gemm_bwd_data", "rbf_bwd", "gemm_bwd_param", "other", "fused_fwd", "fused_bwd")

    def set_profiling(self, on: bool):
        lib.dgp_set_profiling(self.h, 1 if on else 0)

    def get_profile(self, reset=True):
        """{category: (device ms, launches)} accumulated since the last reset (synchronises the stream)."""
        n = len(self.PROFILE_CATEGORIES)
        ms = (C.c_double * n)()
        cnt = (C.c_int64 * n)()
        lib.dgp_get_profile(self.h, C.cast(ms, _vp), C.cast(cnt, _vp), 1 if reset else 0)
        return {k: (float(ms[i]), int(cnt[i])) for i, k in enumerate(self.PROFILE_CATEGORIES)}

    def set_share_first_layer(self, on: bool):
        lib.dgp_set_share_first_layer(self.h, 1 if on else 0)

    def set_vform(self, forward: bool = True, grad=True):
        """grad: False (A-form adjoint), True (V-form adjoint for calls with >= 32768 point-samples), "always"."""
        lib.dgp_set_vform(self.h, 1 if forward else 0, 2 if grad == "always" else (1 if grad else 0))

    def set_parallel_layers(self, on: bool):
        lib.dgp_set_parallel_layers(self.h, 1 if on else 0)

    def set_fused(self, on: bool):
        lib.dgp_set_fused(self.h, 1 if on else 0)

    def set_graph(self, on: bool):
        """CUDA-graph replay of the model-level calls (dgp_set_graph): for launch-bound, BO-sized problems whose buffers stay
        in place from call to call. Turning it off drops the cached graphs."""
        rc = lib.dgp_set_graph(self.h, 1 if on else 0)
        if rc != 0:
            raise DGPError(f"dgp_set_graph ({rc}): {lib.dgp_last_error(self.h).decode()}")
        self.graph = bool(on)

    def set_workspace_limit(self, nbytes: int):
        rc = lib.dgp_set_workspace_limit(self.h, int(nbytes))
        if rc != 0:
            raise DGPError("dgp_set_workspace_limit: invalid size")

    def workspace_bytes(self) -> int:
        return int(lib.dgp_workspace_bytes(self.h))

    def __del__(self):
        try:
            if getattr(self, "h", None):
                lib.dgp_ctx_destroy(self.h)
                self.h = None
        except Exception:
            pass


_ctx_lock = threading.Lock()
_ctxs = {}


def get_context(device=None) -> Context:
    if device is None:
        device = torch.cuda.current_device() if torch.cuda.is_available() else 0
    if isinstance(device, torch.device):
        device = device.index if device.index is not None else torch.cuda.current_device()
    with _ctx_lock:
        ctx = _ctxs.get(device)
        if ctx is None:
            ctx = _ctxs[device] = Context(device)
        return ctx


def as_device(x, device=None) -> torch.Tensor:
    """numpy / torch / any DLPack exporter (e.g. an eager tf.Tensor) -> contiguous float64 CUDA tensor."""
    if device is None:
        device = torch.cuda.current_device()
    dev = torch.device("cuda", device) if not isinstance(device, torch.device) else device
    if isinstance(x, torch.Tensor):
        t = x
    elif isinstance(x, np.ndarray) or np.isscalar(x) or isinstance(x, (list, tuple)):
        t = torch.from_numpy(np.ascontiguousarray(np.asarray(x, dtype=np.float64)))
    elif hasattr(x, "__dlpack__"):
        t = torch.from_dlpack(x)
    elif hasattr(x, "numpy"):
        t = torch.from_numpy(np.ascontiguousarray(np.asarray(x.numpy(), dtype=np.float64)))
    else:
        t = torch.as_tensor(np.asarray(x, dtype=np.float64))
    return t.detach().to(device=dev, dtype=torch.float64).contiguous()


def ptr(t) -> _vp:
    return _vp(0) if t is None else _vp(t.data_ptr())


def ptr_array(tensors):
    """HOST array of device pointers (None entries -> NULL); returns None when `tensors` is None."""
    if tensors is None:
        return None
    arr = (_vp * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = None if t is None else t.data_ptr()
    return arr
