"""Binding of the native kernels into UNMODIFIED reference Pyro (the stub a maintainer would add).

``import pyro`` must already work (the reference tree on ``sys.path``; in this repository's tests that is
``oracle/_ref`` + the ``opt_einsum`` stand-in, see :func:`add_reference_to_path`).  Nothing in Pyro is
patched; every object below plugs into a seam the reference already exposes (SURVEY.md 8b):

=====================  ==========================================================================
seam (reference)        what is handed over
=====================  ==========================================================================
``SVI(loss=...)``       :func:`Trace_ELBO` / :func:`TraceMeanField_ELBO` -- subclasses of the
(pyro/infer/svi.py      reference classes.  Pyro's own poutine builds the traces (trace, replay,
:76-90)                 plate, broadcast); scoring + backward of every site is one fused kernel
                        (``b2_site_score`` / ``b2_event_score`` / ``b2_glm_bernoulli_logits``),
                        replacing ``Trace.compute_log_prob`` (pyro/poutine/trace_struct.py:248-288)
                        and the autograd backward (pyro/infer/trace_elbo.py:130-159).
``SVI(optim=...)``      :func:`ClippedAdam` / :func:`AdagradRMSProp` -- ``pyro.optim.PyroOptim``
(pyro/optim/optim.py    objects whose ``__call__`` is one multi-tensor launch
:72-155)                (``b2_clipped_adam``); ``get_state/set_state/save/load`` keep the reference's
                        per-parameter ``torch.optim`` state_dict schema.
whole step              :func:`SVI` -- ``pyro.infer.SVI`` subclass whose ``step`` replays the captured
                        CUDA graph of (guide, model, fused scoring, backward, fused optimiser).
``NUTS(potential_fn)``  :func:`potential_fn` -- a differentiable ``z dict -> U`` callable backed by
(pyro/infer/mcmc/hmc.py ``b2_potential_grad`` for the reference's own Python tree builder, and
:96-118)                :func:`NUTS` -- an ``MCMCKernel`` whose ``sample`` advances ALL chains on the
                        device (whole transitions in ``b2_nuts_small`` / the lockstep tree).
=====================  ==========================================================================

Distribution objects stay the reference's (``pyro.distributions.*``, i.e. ``torch.distributions``
subclasses): :func:`to_b2` reads their parameters at scoring time, so ``biject_to(support)``,
``kl_divergence`` and user ``isinstance`` checks keep working.
"""
import os
import sys

import torch

from . import distributions as b2d
from . import _native as N  # noqa: F401  (fails loudly if the library is missing)

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def add_reference_to_path():
    """Make ``import pyro`` resolve to the vendored, unmodified reference (``oracle/_ref``, installed by
    ``__graft_entry__.build()`` from the reference source tree, oracle/reference_pyro.py) plus the ~30-line
    stand-in for its absent ``opt_einsum`` dependency.  Returns True if both are present."""
    ref = os.path.join(_ROOT, "oracle", "_ref")
    shim = os.path.join(_ROOT, "tests", "golden", "opt_einsum_standin")
    if not os.path.isdir(os.path.join(ref, "pyro")):
        return False
    for p in (ref, shim):
        if p not in sys.path:
            sys.path.insert(0, p)
    return True


# ---------------------------------------------------------------------------------------------------------
# reference distribution object -> kernel-backed equivalent (parameters are shared, not copied)
# ---------------------------------------------------------------------------------------------------------
def _bern(fn):
    if "logits" in fn.__dict__:
        return b2d.Bernoulli(logits=fn.__dict__["logits"])
    return b2d.Bernoulli(probs=fn.probs)


def _cat(fn):
    if "logits" in fn.__dict__:
        return b2d.Categorical(logits=fn.__dict__["logits"])
    return b2d.Categorical(probs=fn.probs)


_SIMPLE = {
    "Normal": lambda fn: b2d.Normal(fn.loc, fn.scale),
    "Cauchy": lambda fn: b2d.Cauchy(fn.loc, fn.scale),
    "HalfCauchy": lambda fn: b2d.HalfCauchy(fn.scale),
    "HalfNormal": lambda fn: b2d.HalfNormal(fn.scale),
    "LogNormal": lambda fn: b2d.LogNormal(fn.loc, fn.scale),
    "Exponential": lambda fn: b2d.Exponential(fn.rate),
    "Uniform": lambda fn: b2d.Uniform(fn.low, fn.high),
    "Gamma": lambda fn: b2d.Gamma(fn.concentration, fn.rate),
    "Beta": lambda fn: b2d.Beta(fn.concentration1, fn.concentration0),
    "Poisson": lambda fn: b2d.Poisson(fn.rate),
    "Bernoulli": _bern,
    "Dirichlet": lambda fn: b2d.Dirichlet(fn.concentration),
    "Categorical": _cat,
    "MultivariateNormal": lambda fn: b2d.MultivariateNormal(fn.loc, scale_tril=fn._unbroadcasted_scale_tril),
}


def to_b2(fn):
    """Kernel-backed equivalent of a reference distribution object, or None (the caller then scores the
    site with the reference's own ``log_prob`` + autograd, which is always correct)."""
    if isinstance(fn, b2d.Distribution):
        return fn
    name = type(fn).__name__
    try:
        if name == "Independent":
            base = to_b2(fn.base_dist)
            return None if base is None else base.to_event(fn.reinterpreted_batch_ndims)
        if name == "MaskedDistribution":
            base = to_b2(fn.base_dist)
            return None if base is None else base.mask(fn._mask)
        if name == "ExpandedDistribution":
            base = to_b2(fn.base_dist)
            return None if base is None else base.expand(fn.batch_shape)
        make = _SIMPLE.get(name)
        if make is None:
            return None
        out = make(fn)
        if tuple(out.batch_shape) != tuple(fn.batch_shape):
            out = out.expand(fn.batch_shape)
        return out
    except Exception:  # noqa: BLE001 -- an unsupported parameterisation falls back to the reference path
        return None


def _convert_sites(*traces):
    for trace in traces:
        for site in trace.nodes.values():
            if site["type"] == "sample":
                conv = to_b2(site["fn"])
                if conv is not None:
                    site["_ref_fn"] = site["fn"]
                    site["fn"] = conv


_CACHE = {}


def _load():
    """Build the subclasses against the importable ``pyro`` (once)."""
    if _CACHE:
        return _CACHE
    import pyro
    import pyro.poutine as poutine
    from pyro.infer import SVI as RefSVI
    from pyro.infer import Trace_ELBO as RefTrace_ELBO
    from pyro.infer import TraceMeanField_ELBO as RefTraceMeanField_ELBO
    from pyro.infer.mcmc.mcmc_kernel import MCMCKernel
    from pyro.infer.util import is_validation_enabled
    from pyro.optim import PyroOptim as RefPyroOptim
    from pyro.poutine.util import prune_subsample_sites
    from pyro.util import check_model_guide_match, warn_if_nan

    from . import infer as own_infer
    from . import optim as own_optim
    from .infer import svi as own_svi
    from .infer.mcmc import potential as own_pot
    from .infer.mcmc.compile import recognise
    from .lazy import unwrap_site_values, wrap_site_values

    def unscored_traces(self, model, guide, args, kwargs):
        """pyro/infer/enum.py:45-85 without the two scoring calls: the guide runs, the model is replayed
        against it by the reference's own poutine, subsample sites are pruned."""
        guide_trace = poutine.trace(guide, graph_type="flat").get_trace(*args, **kwargs)
        wrap_site_values(guide_trace)
        try:
            model_trace = poutine.trace(poutine.replay(model, trace=guide_trace),
                                        graph_type="flat").get_trace(*args, **kwargs)
        finally:
            unwrap_site_values(guide_trace)
        unwrap_site_values(model_trace)
        if is_validation_enabled():
            check_model_guide_match(model_trace, guide_trace, self.max_plate_nesting)
        guide_trace = prune_subsample_sites(guide_trace)
        model_trace = prune_subsample_sites(model_trace)
        _convert_sites(model_trace, guide_trace)
        return model_trace, guide_trace

    def make_elbo(ref_cls, engine_cls, label):
        class _B2ELBO(ref_cls):
            __doc__ = "``pyro.infer.%s`` with sites scored by the fused sm_100a kernels." % label
            capture_graph = False

            def __init__(self, *args, **kwargs):
                super().__init__(*args, **kwargs)
                # the scoring engine shares this object's particle / plate configuration
                self._engine = engine_cls(num_particles=self.num_particles,
                                          max_plate_nesting=float("inf"),
                                          vectorize_particles=self.vectorize_particles,
                                          retain_graph=self.retain_graph)
                self._fused_traces = False

            def _get_trace(self, model, guide, args, kwargs):
                if self._fused_traces:
                    return unscored_traces(self, model, guide, args, kwargs)
                return super()._get_trace(model, guide, args, kwargs)

            def loss_and_grads_tensor(self, model, guide, *args, **kwargs):
                eng = self._engine
                eng.num_particles = self.num_particles
                loss = None
                self._fused_traces = True
                try:
                    traces = list(self._get_traces(model, guide, args, kwargs))
                finally:
                    self._fused_traces = False
                for model_trace, guide_trace in traces:
                    part = eng._score_and_backward(model_trace, guide_trace)
                    if part is None:
                        # a site without a reparameterised sampler: the reference algorithm, unchanged
                        return torch.as_tensor(ref_cls.loss_and_grads(self, model, guide, *args, **kwargs))
                    loss = part if loss is None else loss + part
                return loss if loss is not None else torch.zeros(())

            def loss_and_grads(self, model, guide, *args, **kwargs):
                loss = self.loss_and_grads_tensor(model, guide, *args, **kwargs)
                loss = loss.item() if isinstance(loss, torch.Tensor) else float(loss)
                warn_if_nan(loss, "loss")
                return loss

        _B2ELBO.__name__ = _B2ELBO.__qualname__ = label
        return _B2ELBO

    Trace_ELBO = make_elbo(RefTrace_ELBO, own_infer.Trace_ELBO, "Trace_ELBO")
    TraceMeanField_ELBO = make_elbo(RefTraceMeanField_ELBO, own_infer.TraceMeanField_ELBO,
                                    "TraceMeanField_ELBO")

    class JitTrace_ELBO(Trace_ELBO):
        """Marks the loss as capturable: :class:`SVI` below captures the whole step into a CUDA graph
        (the role ``torch.jit.trace`` plays in pyro/infer/trace_elbo.py:162-257)."""
        capture_graph = True

    # ---- optimisers: real PyroOptim objects, fused multi-tensor update -----------------------------------
    def make_optim(own_cls, label):
        class _B2Optim(RefPyroOptim):
            __doc__ = "``pyro.optim.%s`` as one fused launch per step (b2 kernels)." % label

            def __init__(self, optim_args, clip_args=None):
                # the constructor argument keeps PyroOptim's checks and `optim_args` bookkeeping happy;
                # the update itself never instantiates per-parameter torch optimisers
                super().__init__(torch.optim.SGD, optim_args, clip_args)
                self._b2 = own_cls(optim_args, clip_args)
                self._b2._store = pyro.get_param_store

            def __call__(self, params, *args, **kwargs):
                self._b2(list(params), *args, **kwargs)

            def flush_pending(self):
                self._b2.flush_pending()

            def get_state(self):
                return self._b2.get_state()

            def set_state(self, state_dict):
                self._b2.set_state(state_dict)

        _B2Optim.__name__ = _B2Optim.__qualname__ = label
        return _B2Optim

    ClippedAdam = make_optim(own_optim.ClippedAdam, "ClippedAdam")
    AdagradRMSProp = make_optim(own_optim.AdagradRMSProp, "AdagradRMSProp")

    # ---- whole-step capture ----------------------------------------------------------------------------
    class SVI(RefSVI, own_svi.SVI):
        """``pyro.infer.SVI`` (same constructor); with a ``JitTrace_ELBO`` loss the second ``step`` captures
        guide + model + fused scoring + backward + fused optimiser into one CUDA graph."""
        _poutine = poutine

        def __init__(self, model, guide, optim, loss, loss_and_grads=None, num_samples=0, num_steps=0, **kw):
            RefSVI.__init__(self, model, guide, optim, loss, loss_and_grads, num_samples, num_steps, **kw)
            self._loss_obj = loss
            self._loss_and_grads_tensor = getattr(loss, "loss_and_grads_tensor", None)
            self._capture = bool(getattr(loss, "capture_graph", False))
            self._graph = None
            self._graph_state = None
            self._steps_done = 0

        def step(self, *args, **kwargs):
            return own_svi.SVI.step(self, *args, **kwargs)

        def _capture_graph(self, args, private=False):
            # torch.distributions' argument validation reads `valid.all()` back to the host, which a
            # capturing stream forbids.  The first (eager) step ran with the user's validation setting;
            # the captured step is recorded without it (pyro.validation_enabled is the reference's own
            # switch, pyro/__init__.py) -- the analogue of JitTrace_ELBO's ignore_jit_warnings.
            with pyro.validation_enabled(False):
                return own_svi.SVI._capture_graph(self, args, private=private)

    # ---- MCMC --------------------------------------------------------------------------------------------
    class _PotentialFn(torch.autograd.Function):
        @staticmethod
        def forward(ctx, pot, z):
            U, g = pot.value_and_grad(z.detach().reshape(1, -1))
            ctx.save_for_backward(g.reshape(z.shape))
            return U.reshape(())

        @staticmethod
        def backward(ctx, gout):
            (g,) = ctx.saved_tensors
            return None, g * gout

    def potential_fn(native, site="z"):
        """``potential_fn`` for the reference ``HMC/NUTS(potential_fn=...)``: a single latent site ``site``
        holding the unconstrained vector of a native model class; value and gradient come from ONE
        ``b2_potential_grad`` launch instead of a model re-trace + autograd."""
        def fn(params):
            return _PotentialFn.apply(native, params[site])
        fn.native = native
        return fn

    class NUTS(MCMCKernel):
        """``MCMCKernel`` (pyro/infer/mcmc/mcmc_kernel.py:8-80) for the reference ``pyro.infer.MCMC``:
        ``num_chains`` chains advance together on the device per ``sample`` call; the returned site
        values carry the chain dimension first.  Constructor arguments follow ``pyro.infer.NUTS``."""

        def __init__(self, model=None, potential_fn=None, num_chains=1, seed=0, **kwargs):
            self._kernel = own_infer.NUTS(model=None if model is None else model,
                                          potential_fn=potential_fn, **kwargs) \
                if model is None else None
            self._model = model
            self.model = None         # pyro/infer/mcmc/api.py:377 reads these two attributes
            self.transforms = {}      # sample() already returns constrained values
            self._kwargs = kwargs
            self._num_chains = num_chains
            self._seed = seed
            self._initial = None

        def setup(self, warmup_steps, *args, **kwargs):
            if self._kernel is None:
                native = recognise(self._model, args, kwargs, poutine=poutine)
                if native is None:
                    raise NotImplementedError(
                        "pyro_b200.bind.NUTS: this model is not one of the compiled model classes; use "
                        "pyro.infer.NUTS(model) (reference tree, per-site kernels through bind.Trace_ELBO "
                        "are not involved) or pass potential_fn=")
                self._kernel = own_infer.NUTS(potential_fn=native, **self._kwargs)
            self._kernel.setup(warmup_steps, self._num_chains, seed=self._seed)
            self._t = 0

        @property
        def initial_params(self):
            k = self._kernel
            return {name: v for name, v in k.potential.unpack(k._z).items()}

        @initial_params.setter
        def initial_params(self, params):
            self._initial = params

        def sample(self, params):
            k = self._kernel
            z = k.sample()
            return k.potential.unpack(z)

        def logging(self):
            k = self._kernel
            return {"step size": "{:.2e}".format(float(k._adapter.step_size.mean())),
                    "acc. prob": "{:.3f}".format(float(k._mean_accept.mean()))}

        def diagnostics(self):
            return self._kernel.diagnostics()

        def cleanup(self):
            pass

    _CACHE.update(dict(Trace_ELBO=Trace_ELBO, TraceMeanField_ELBO=TraceMeanField_ELBO,
                       JitTrace_ELBO=JitTrace_ELBO, ClippedAdam=ClippedAdam, AdagradRMSProp=AdagradRMSProp,
                       SVI=SVI, NUTS=NUTS, potential_fn=potential_fn, recognise=recognise,
                       HierNormalPotential=own_pot.HierNormalPotential,
                       LogisticPotential=own_pot.LogisticPotential))
    return _CACHE


def __getattr__(name):
    if name in ("Trace_ELBO", "TraceMeanField_ELBO", "JitTrace_ELBO", "ClippedAdam", "AdagradRMSProp",
                "SVI", "NUTS", "potential_fn", "recognise", "HierNormalPotential", "LogisticPotential"):
        return _load()[name]
    raise AttributeError(name)
