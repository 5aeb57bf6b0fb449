"""Runs the reference's OWN source (the `dgp_dace` package of a reference checkout whose root DGP_REFERENCE_ROOT names,
imported unmodified) on the stand-in tensorflow / gpflow / tensorflow_probability modules of tests/ref_shim (torch-CPU
float64). Test infrastructure: used by tests/test_reference_exec.py and the tests/golden/make_golden*.py scripts. The
repository does not contain the reference; without a checkout the tests compare with the reference outputs stored under
tests/golden/."""
import importlib
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
SHIM = os.path.join(HERE, "ref_shim")
REFERENCE = os.environ.get("DGP_REFERENCE_ROOT", "")


def available():
    return bool(REFERENCE) and os.path.isdir(os.path.join(REFERENCE, "dgp_dace"))


_mods = None


def load():
    """→ namespace with tf, gpflow, tfp and the reference modules layers, utils, layer_initializations, dgp, Infill_criteria, EHVI."""
    global _mods
    if _mods is not None:
        return _mods
    if not available():
        raise RuntimeError("no reference checkout: set DGP_REFERENCE_ROOT to the directory that holds dgp_dace/")
    for p in (REFERENCE, SHIM):
        if p not in sys.path:
            sys.path.insert(0, p)
    import tensorflow as tf
    assert os.path.dirname(os.path.dirname(tf.__file__)) == SHIM, "a real tensorflow shadows the stand-in: " + tf.__file__
    import gpflow
    import tensorflow_probability as tfp
    ns = types.SimpleNamespace(tf=tf, gpflow=gpflow, tfp=tfp)
    for name, mod in (("layers", "dgp_dace.utils.layers"), ("utils", "dgp_dace.utils.utils"),
                      ("layer_initializations", "dgp_dace.utils.layer_initializations"), ("dgp", "dgp_dace.models.dgp"),
                      ("Infill_criteria", "dgp_dace.Infill_criteria"), ("EHVI", "dgp_dace.EHVI")):
        m = importlib.import_module(mod)
        assert m.__file__.startswith(REFERENCE), m.__file__
        setattr(ns, name, m)
    _mods = ns
    return ns


def _kernel(ns, l):
    cls = {"rbf": ns.gpflow.kernels.SquaredExponential, "matern32": ns.gpflow.kernels.Matern32,
           "matern52": ns.gpflow.kernels.Matern52}[l.get("kernel", "rbf")]
    return cls(variance=float(l["variance"]), lengthscales=np.asarray(l["lengthscales"], dtype=np.float64))


def _mean_function(ns, l):
    mf = ns.gpflow.mean_functions
    if l["mean_kind"] == "zero":
        return mf.Zero()
    if l["mean_kind"] == "identity":
        return mf.Identity()
    m = mf.Linear(l["mf_W"], l["mf_b"])
    ns.gpflow.set_trainable(m, False)
    return m


def reference_model(prob, num_samples):
    """The reference's `DGP_Base` (models/dgp.py:21-32) over the reference's `SVGP_Layer`s (utils/layers.py:180-224) holding
    the parameters of an `oracle.synthetic_problem` dict."""
    ns = load()
    layers = []
    for l in prob["layers"]:
        layer = ns.layers.SVGP_Layer(_kernel(ns, l), np.asarray(l["Z"]), l["q_mu"].shape[1], _mean_function(ns, l),
                                     white=bool(l.get("white", False)))
        layer.q_mu.assign(l["q_mu"])
        layer.q_sqrt.assign(l["q_sqrt"])
        layers.append(layer)
    return ns.dgp.DGP_Base(ns.gpflow.likelihoods.Gaussian(float(prob["lik_var"])), layers, num_samples=num_samples)


class fixed_draws:
    """with fixed_draws(zs): every tf.random.normal call inside returns the next array of `zs` (a missing draw raises) —
    the reference's `z=None` code path (utils/layers.py:112-113) fed with the oracle's draws."""

    def __init__(self, zs):
        self.zs = [np.asarray(z) for z in zs]
        self.i = 0

    def __enter__(self):
        ns = load()
        self._prev = ns.tf.random.source
        ns.tf.random.source = self._next
        return self

    def _next(self, shape):
        z = self.zs[self.i]
        self.i += 1
        assert tuple(z.shape) == tuple(shape), (z.shape, shape)
        return z

    def __exit__(self, *exc):
        load().tf.random.source = self._prev
        return False


def constrained_grads(model, grads_by_variable):
    """Reference gradients are w.r.t. GPflow's unconstrained variables (`tape.gradient(objective, trainable_variables)`,
    models/dgp.py:145); this maps them to constrained-space gradients named like `oracle.OModel.named_params()`:
    softplus θ = log(1+eᵘ): ∂u = ∂θ·(1−e^{−θ}) (likelihood: θ−1e-6); FillTriangular is a permutation."""
    out = {}

    def conv(p):
        g = grads_by_variable.get(id(p.unconstrained_variable))
        if g is None:
            return None
        g = g.as_subclass(torch.Tensor)
        tname = type(p.transform).__name__
        if tname == "Identity":
            return g
        if tname == "FillTriangular":
            return p.transform.forward(g).as_subclass(torch.Tensor)
        theta = p.value().detach().as_subclass(torch.Tensor)
        if tname == "Chain":
            theta = theta - p.transform.bijectors[0].shift
        return g / (1.0 - torch.exp(-theta))

    for i, layer in enumerate(model.layers):
        for name, p in (("Z", layer.feature.Z), ("lengthscales", layer.kern.lengthscales), ("variance", layer.kern.variance),
                        ("q_mu", layer.q_mu), ("q_sqrt", layer.q_sqrt)):
            g = conv(p)
            if g is not None:
                out[f"layers.{i}.{name}"] = g
    g = conv(model.likelihood.likelihood.variance)
    if g is not None:
        out["lik_var"] = g
    return out


def elbo_and_grads(model, X, Y, zs):
    """ELBO through the reference's training-step code path (`ELBO_closure` under a GradientTape, models/dgp.py:142-145),
    with the draws of `zs` served to the reference's own tf.random.normal calls."""
    ns = load()
    tvars = list(model.trainable_variables)
    with fixed_draws(zs):
        with ns.tf.GradientTape(watch_accessed_variables=False) as tape:
            tape.watch(tvars)
            objective = -model.ELBO_closure((ns.tf.constant(X), ns.tf.constant(Y)))
            gradients = tape.gradient(objective, tvars)
    by_var = {id(v): (None if g is None else -g) for v, g in zip(tvars, gradients)}
    return float(-objective.numpy()), constrained_grads(model, by_var)
