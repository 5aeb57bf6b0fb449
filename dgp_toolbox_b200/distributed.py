"""Data-parallel ELBO+gradient over the GPUs of one box (SURVEY §8e): the minibatch's points are split contiguously over
the ranks (each rank keeps all S samples of its points; Philox counters use the global point index so the draws do not
depend on the placement), parameters — hence Kuu, its Cholesky and the KL term — are replicated, and ONE sum-allreduce of
the flat [data term, KL, gradients] buffer per step restores the full-batch result (KL pre-weighted by 1/world).
ShardedELBO does this for the RBF / Matérn DGP, ShardedComposite for the composite-kernel models (MF-DGP, MF-DGP-EM, MO-DGP)."""
from __future__ import annotations

import contextlib
import io
from dataclasses import dataclass

import numpy as np
import torch
import torch.distributed as dist


def shard_bounds(N, rank, world):
    """Contiguous split of N points: rank r owns [lo, hi)."""
    base, rem = divmod(N, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class ShardedELBO:
    def __init__(self, model, group=None, library_comm=True):
        """library_comm: the allreduce runs inside libdgp_b200 (dgp_comm_init / dgp_allreduce_grads: the library's own NCCL
        communicator on the ctx's stream, SURVEY §8b) -- torch.distributed only carries the 128-byte ncclUniqueId to the ranks.
        False, or a CPU model (gloo tests of the host logic): torch.distributed.all_reduce."""
        self.model = model
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self._pinned_out = None
        self._ctx = None
        if library_comm and self.world > 1 and torch.cuda.is_available() and model.device.type == "cuda":
            from . import _lib
            import ctypes as C
            uid = torch.zeros(128, dtype=torch.uint8)
            if self.rank == 0:
                rc = _lib.lib.dgp_comm_unique_id(C.c_void_p(uid.data_ptr()))
                if rc != 0:
                    raise _lib.DGPError(f"dgp_comm_unique_id failed ({rc}): libnccl.so.2 could not be loaded")
            uid_dev = uid.to(model.device)
            dist.broadcast(uid_dev, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
            uid = uid_dev.cpu()
            self._ctx = _lib.get_context(model.device)
            self._ctx.call("dgp_comm_init", self.rank, self.world, C.c_void_p(uid.data_ptr()))

    def step(self, X_local, Y_local, n_offset, scale=1.0, want_grad=True, seed=None, zs=None):
        """Device-resident shard in, reduced flat device buffer out."""
        flat = self.model.elbo_flat((X_local, Y_local), want_grad=want_grad, scale=scale, kl_weight=1.0 / self.world,
                                    seed=seed, n_offset=n_offset, zs=zs)
        if self.world > 1:
            if self._ctx is not None:
                from . import _lib
                self._ctx.call("dgp_allreduce_grads", _lib.ptr(flat), flat.numel())
            else:
                dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group)
        return flat

    def train_adam_step(self, X_local, Y_local, n_offset, params, state, t, lr=0.01, beta_1=0.9, beta_2=0.999, epsilon=1e-7,
                        scale=1.0, seed=None):
        """One data-parallel training iteration: sharded ELBO gradient, the allreduce, then the same dgp_adam_step on every
        rank (the reduced buffer is bit-identical across ranks, so the replicated parameters stay in lockstep without a
        broadcast). `params` / `state` as in DGP_Base._adam_state; t counts from 1. Returns the reduced flat buffer."""
        flat = self.step(X_local, Y_local, n_offset, scale=scale, want_grad=True, seed=seed)
        self.model._adam_step(params, flat, state, t, lr, beta_1, beta_2, epsilon)
        return flat

    def step_host(self, X_host: torch.Tensor, Y_host: torch.Tensor, n_offset, scale=1.0, want_grad=True, seed=None):
        """Pinned HOST shard in, HOST result out: H2D copies, the step, the allreduce and the D2H copy of the result."""
        dev = self.model.device
        if self.world == 1:
            if self._pinned_out is None:
                n, _ = self.model.grad_layout()
                self._pinned_out = torch.empty(n, dtype=torch.float64).pin_memory()
            out = self._pinned_out.numpy()
            self.model.elbo_flat_host(X_host.numpy(), Y_host.numpy(), want_grad=want_grad, scale=scale, kl_weight=1.0,
                                      seed=seed, n_offset=n_offset, out_host=out)
            return self._pinned_out
        X = X_host.to(dev, non_blocking=True)
        Y = Y_host.to(dev, non_blocking=True)
        flat = self.step(X, Y, n_offset, scale, want_grad, seed)
        if self._pinned_out is None or self._pinned_out.numel() != flat.numel():
            self._pinned_out = torch.empty(flat.numel(), dtype=torch.float64).pin_memory()
        self._pinned_out.copy_(flat, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()
        return self._pinned_out


@dataclass(frozen=True)
class CompositeShard:
    """One rank's part of a composite-kernel model's minibatch (MF-DGP / MO-DGP `(X, Y)`, MF-DGP-EM `(X, Y, X_red)`).
    data: the local slices, in the model's data format; offsets[l]: global index of the first local point of fidelity (objective)
    l, which indexes the Philox draws; counts[l]: that fidelity's point count over all ranks; kl_weight: 1 / world, the weight of
    every KL term, so that the sum over the ranks of the local ELBOs and gradients is the full-batch one."""
    data: tuple
    offsets: tuple
    counts: tuple
    kl_weight: float


def composite_shard(data, rank, world):
    """Split a composite-kernel model's data contiguously (shard_bounds per fidelity / objective); X_red[l] pairs row for row with
    X[l+1] and takes its bounds. Raises ValueError when a fidelity has fewer points than ranks or the pairings do not line up."""
    X, Y = data[0], data[1]
    if len(X) != len(Y):
        raise ValueError(f"{len(X)} input sets but {len(Y)} output sets")
    counts = tuple(int(np.shape(x)[0]) for x in X)
    for l, (x, y) in enumerate(zip(X, Y)):
        if np.shape(y)[0] != counts[l]:
            raise ValueError(f"fidelity {l}: {counts[l]} inputs but {np.shape(y)[0]} outputs")
        if counts[l] < world:
            raise ValueError(f"fidelity {l} has {counts[l]} points, fewer than the {world} ranks")
    bounds = [shard_bounds(n, rank, world) for n in counts]
    local = ([x[lo:hi] for x, (lo, hi) in zip(X, bounds)], [y[lo:hi] for y, (lo, hi) in zip(Y, bounds)])
    if len(data) == 3:
        X_red = data[2]
        if len(X_red) != len(X) - 1 or any(np.shape(xr)[0] != counts[l + 1] for l, xr in enumerate(X_red)):
            raise ValueError(f"X_red[l] must pair row for row with X[l+1]: got {[np.shape(xr)[0] for xr in X_red]} rows for "
                             f"{list(counts[1:])} points")
        local += ([xr[lo:hi] for xr, (lo, hi) in zip(X_red, bounds[1:])],)
    return CompositeShard(local, tuple(lo for lo, _ in bounds), counts, 1.0 / world)


class ShardedComposite:
    def __init__(self, model, group=None):
        """Data-parallel ELBO, gradients and training of a MultiFidelityDeepGP, MultiFidelityDeepGP_EM or MultiObjDeepGP over the
        ranks of `group` (one GPU each, every rank holding the same model and data). Each fidelity's (objective's) points are split
        contiguously; parameters, the Z_right refresh (same draws on every rank) and the KL terms (weighted 1 / world) are
        replicated. One evaluation is the model's own library calls on the local points and ONE sum-allreduce of the flat
        [data terms, KL terms, gradients] buffer inside the library (dgp_allreduce_grads on its NCCL communicator; torch.distributed
        only carries the 128-byte unique id, or, for a CPU model, does the reduction). The model's draw must accept `n_offset`
        (the default Philox draw does). With world 1 every call is the single-GPU path. Call close() when done."""
        self.obj, self.model = model, model.model
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self._ctx = None
        if self.world > 1 and self.model.device.type == "cuda":
            from . import _lib
            import ctypes as C
            uid = torch.zeros(128, dtype=torch.uint8)
            if self.rank == 0:
                rc = _lib.lib.dgp_comm_unique_id(C.c_void_p(uid.data_ptr()))
                if rc != 0:
                    raise _lib.DGPError(f"dgp_comm_unique_id failed ({rc}): libnccl.so.2 could not be loaded")
            uid_dev = uid.to(self.model.device)
            dist.broadcast(uid_dev, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
            uid = uid_dev.cpu()
            self._ctx = _lib.get_context(self.model.device)
            self._ctx.call("dgp_comm_init", self.rank, self.world, C.c_void_p(uid.data_ptr()))

    def close(self):
        """Release the library's communicator (dgp_comm_destroy)."""
        if self._ctx is not None:
            from . import _lib
            _lib.lib.dgp_comm_destroy(self._ctx.h)
            self._ctx = None

    def local_data(self, data):
        """This rank's CompositeShard of the full data `(X, Y)` or `(X, Y, X_red)` (refusals as in composite_shard)."""
        return composite_shard(data, self.rank, self.world)

    def ELBO_and_grads(self, local, params=None, **kwargs):
        """(ELBO, {Parameter: gradient}) of the whole batch, identical on every rank. `local`: local_data(...); kwargs go to the
        model's ELBO_and_grads (MO-DGP: tf_sample_Z_right)."""
        m = self.model
        if self.world == 1:
            return m.ELBO_and_grads(local.data, params, **kwargs)
        params = m.trainable_parameters if params is None else params
        _, grads = m.ELBO_and_grads(local.data, params, shard=local, **kwargs)
        terms = (m.L + getattr(m, "L_red", 0.0), m.KL + getattr(m, "KL_red", 0.0))     # MF-DGP-EM: + projection terms
        flat = torch.cat([torch.stack([torch.as_tensor(t, dtype=torch.float64, device=m.device) for t in terms]).detach()]
                         + [grads[p].reshape(-1) for p in params])
        if self._ctx is not None:
            from . import _lib
            self._ctx.call("dgp_allreduce_grads", _lib.ptr(flat), flat.numel())
        else:
            dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group)
        out, off = {}, 2
        for p in params:
            out[p] = flat[off:off + p.value.numel()].view_as(p.value)
            off += p.value.numel()
        return flat[0] - flat[1], out

    def optimize_adam(self, *args, **kwargs):
        """The object's own optimize_adam (same arguments and three-phase schedule) on the sharded, reduced evaluation: every
        rank takes the same Adam steps on identical gradients, so the parameters stay equal without a broadcast. Only rank 0
        prints."""
        return self._train(self.obj.optimize_adam, args, kwargs)

    def optimize_nat_adam(self, *args, **kwargs):
        """The object's own optimize_nat_adam; both evaluations of a natural-gradient iteration are sharded (as optimize_adam)."""
        return self._train(self.obj.optimize_nat_adam, args, kwargs)

    def _train(self, fn, args, kwargs):
        o = self.obj
        local = self.local_data((o._X, o._Y, o._X_red) if hasattr(o, "_X_red") else (o._X, o._Y))
        quiet = contextlib.redirect_stdout(io.StringIO()) if self.rank else contextlib.nullcontext()
        with quiet:
            return fn(*args, evaluate=lambda params, **kw: self.ELBO_and_grads(local, params, **kw), **kwargs)
