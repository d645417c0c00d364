"""The binding of INTEGRATION.md executed against UNMODIFIED reference Pyro (pyro 1.9.1 from
``oracle/_ref``, copied by ``__graft_entry__.build()`` from the reference source tree,
oracle/reference_pyro.py; without it these tests skip): models and guides are written with ``import pyro``;
``pyro.infer.SVI`` / ``pyro.infer.MCMC`` drive them; the kernels enter through the seams of SURVEY.md 8b
(``loss=``, ``optim=``, ``potential_fn=``, ``kernel=``).

Every scenario runs twice: in the CPU tier with the native seams replaced by the oracle-backed stand-ins
(host logic only) and in the ``-m gpu`` tier through the real kernels.  Reference numbers are the
goldens recorded from the same unmodified Pyro (tests/golden/make_golden.py)."""
import numpy as np
import pytest
import torch
from torch.distributions import constraints

from conftest import EMULATE, load_npz


def _import_pyro():
    from pyro_b200 import bind
    if not bind.add_reference_to_path():
        pytest.skip("reference Pyro is not vendored (oracle/_ref missing; see oracle/reference_pyro.py)")
    import pyro
    assert pyro.__version__.startswith("1.9"), pyro.__version__
    assert "pyro_b200" not in (pyro.__file__ or "")
    return pyro, bind


def _models(pyro):
    import pyro.distributions as dist
    from pyro.poutine.messenger import Messenger

    def logistic_model(X, y):                         # tests/infer/mcmc/test_hmc.py:189-198, vectorised
        D = X.shape[-1]
        w = pyro.sample("w", dist.Normal(X.new_zeros(D), X.new_ones(D)).to_event(1))
        b = pyro.sample("b", dist.Normal(X.new_zeros(()), X.new_full((), 10.0)))
        with pyro.plate("data", X.shape[0]):
            logits = w.squeeze(-2) @ X.T + b if w.dim() > 1 else X @ w + b
            pyro.sample("y", dist.Bernoulli(logits=logits), obs=y)

    def logistic_guide(X, y):
        D = X.shape[-1]
        w_loc = pyro.param("w_loc", lambda: X.new_zeros(D))
        w_scale = pyro.param("w_scale", lambda: X.new_full((D,), 0.1), constraint=constraints.positive)
        b_loc = pyro.param("b_loc", lambda: X.new_zeros(()))
        b_scale = pyro.param("b_scale", lambda: X.new_full((), 0.1), constraint=constraints.positive)
        pyro.sample("w", dist.Normal(w_loc, w_scale).to_event(1))
        pyro.sample("b", dist.Normal(b_loc, b_scale))

    class InjectNoise(Messenger):                    # the replay technique of tests/infer/test_gradient.py:77-91
        def __init__(self, eps):
            super().__init__()
            self.eps = eps

        def _pyro_sample(self, msg):
            if msg["name"] in self.eps and not msg["is_observed"]:
                base = msg["fn"]
                while hasattr(base, "base_dist"):
                    base = base.base_dist
                e = self.eps[msg["name"]]
                # value only (not "done"): the plate's BroadcastMessenger still expands the site's fn, and
                # pyro/poutine/runtime.py:341 keeps a pre-set value instead of sampling
                msg["value"] = base.loc + e.to(base.loc.dtype) * base.scale

    def eight_schools(sigma, y=None):                # examples/eight_schools/mcmc.py:27-34
        J = sigma.shape[0]
        eta = pyro.sample("eta", dist.Normal(sigma.new_zeros(J), sigma.new_ones(J)))
        mu = pyro.sample("mu", dist.Normal(sigma.new_zeros(1), 10 * sigma.new_ones(1)))
        tau = pyro.sample("tau", dist.HalfCauchy(scale=25 * sigma.new_ones(1)))
        theta = mu + tau * eta
        return pyro.sample("obs", dist.Normal(theta, sigma), obs=y)

    return logistic_model, logistic_guide, InjectNoise, eight_schools


def _svi_trajectory(dev, dtype, tag, tol, svi_cls=None, elbo="Trace_ELBO", steps=None, then=None):
    pyro, bind = _import_pyro()
    logistic_model, logistic_guide, InjectNoise, _ = _models(pyro)
    g = load_npz("svi_logistic.npz")
    pyro.clear_param_store()
    torch.set_default_dtype(dtype)
    try:
        X, y = torch.as_tensor(g["X"]).to(dev, dtype), torch.as_tensor(g["y"]).to(dev, dtype)
        eps_w, eps_b = torch.as_tensor(g["eps_w"]).to(dev, dtype), torch.as_tensor(g["eps_b"]).to(dev, dtype)
        P = int(g["P"])
        # fixed noise buffers refilled before every step: the same code serves the eager and the
        # CUDA-graph captured runs (a captured graph bakes in the buffer addresses, not the values)
        bw, bb = torch.empty_like(eps_w[0]), torch.empty_like(eps_b[0])

        def guide(X, y):
            with InjectNoise({"w": bw, "b": bb}):
                logistic_guide(X, y)

        SVI = pyro.infer.SVI if svi_cls is None else getattr(bind, svi_cls)
        loss_obj = getattr(bind, elbo)(num_particles=P, vectorize_particles=True, max_plate_nesting=1)
        assert isinstance(loss_obj, pyro.infer.Trace_ELBO)      # a subclass of the reference class
        optim = bind.ClippedAdam({"lr": 0.01})
        assert isinstance(optim, pyro.optim.PyroOptim)
        svi = SVI(logistic_model, guide, optim, loss_obj)
        for i in range(eps_w.shape[0] if steps is None else steps):
            bw.copy_(eps_w[i])
            bb.copy_(eps_b[i])
            loss = svi.step(X, y)
            assert abs(loss - g["losses_" + tag][i]) <= 10 * tol * abs(g["losses_" + tag][i]), (i, loss)
            store = pyro.get_param_store()
            flat = torch.cat([store[k].detach().reshape(-1).double().cpu()
                              for k in ("w_loc", "w_scale", "b_loc", "b_scale")])
            assert torch.allclose(flat, torch.as_tensor(g["params_" + tag][i]), atol=10 * tol, rtol=10 * tol), i
        if then is not None:
            then(pyro, bind, optim)
        return optim
    finally:
        pyro.clear_param_store()
        torch.set_default_dtype(torch.float32)


def _lazy_site_reaches_glm(dev):
    """The unchanged ``w.squeeze(-2) @ X.T + b`` of a reference model arrives at the likelihood site as a
    lazy linear predictor: the converted site is the fused-GLM Bernoulli, and no [P, N] logits exist."""
    pyro, bind = _import_pyro()
    import pyro.poutine as poutine
    from pyro_b200 import distributions as b2d
    from pyro_b200.lazy import LinearPredictorTensor, unwrap_site_values, wrap_site_values
    logistic_model, logistic_guide, _, _ = _models(pyro)
    pyro.clear_param_store()
    X = torch.randn(64, 32, device=dev)
    y = (torch.rand(64, device=dev) < 0.5).float()
    P = 4
    elbo = bind.Trace_ELBO(num_particles=P, vectorize_particles=True, max_plate_nesting=1)
    guide_trace = poutine.trace(elbo._vectorized_num_particles(logistic_guide)).get_trace(X, y)
    wrap_site_values(guide_trace)
    model_trace = poutine.trace(poutine.replay(elbo._vectorized_num_particles(logistic_model),
                                               trace=guide_trace)).get_trace(X, y)
    unwrap_site_values(guide_trace, model_trace)
    fn = model_trace.nodes["y"]["fn"]
    while hasattr(fn, "base_dist"):
        fn = fn.base_dist
    assert isinstance(fn.__dict__["logits"], LinearPredictorTensor)
    assert tuple(fn.batch_shape) == (P, 64)
    conv = bind.to_b2(model_trace.nodes["y"]["fn"])
    assert isinstance(conv, b2d._BernoulliLinear)
    pyro.clear_param_store()


def _nuts_eight_schools(dev, kernel_kind):
    pyro, bind = _import_pyro()
    from pyro.infer import MCMC
    _, _, _, eight_schools = _models(pyro)
    g = load_npz("mcmc.npz")
    y = torch.tensor([28.0, 8.0, -3.0, 7.0, -1.0, 1.0, 18.0, 12.0], device=dev, dtype=torch.float64)
    sigma = torch.tensor([15.0, 10.0, 16.0, 11.0, 9.0, 11.0, 10.0, 18.0], device=dev, dtype=torch.float64)
    pyro.set_rng_seed(0)
    if kernel_kind == "kernel":
        # bind.NUTS: an MCMCKernel for the reference MCMC driver; the model is recognised as the
        # hierarchical-Normal class and 32 chains advance per sample() call
        on_gpu = str(dev) == "cuda"
        extra = {} if on_gpu else {"native_small": False}   # no CPU stand-in of b2_nuts_small
        kernel = bind.NUTS(eight_schools, num_chains=32 if on_gpu else 8, seed=3, **extra)
        n = 150 if on_gpu else 50
        mcmc = MCMC(kernel, num_samples=n, warmup_steps=n, num_chains=1, disable_progbar=True)
        mcmc.run(sigma, y)
        s = mcmc.get_samples()
        mu = s["mu"].double().reshape(-1)
        tau = s["tau"].double().reshape(-1)
    else:
        # reference NUTS (python tree) on the native potential through potential_fn=
        native = bind.recognise(eight_schools, (sigma, y), {}, poutine=pyro.poutine)
        assert native is not None and type(native).__name__ == "HierNormalPotential"
        pf = bind.potential_fn(native)
        kernel = pyro.infer.NUTS(potential_fn=pf, max_tree_depth=6)
        init = {"z": torch.zeros(native.dim, device=dev, dtype=torch.float64)}
        mcmc = MCMC(kernel, num_samples=120, warmup_steps=120, initial_params=init, disable_progbar=True)
        mcmc.run()
        z = mcmc.get_samples()["z"]
        vals = native.unpack(z)
        mu, tau = vals["mu"].double().reshape(-1), vals["tau"].double().reshape(-1)
    # the reference's own long runs (tests/golden/mcmc.npz): posterior mean of mu ~ 4.4, tau ~ 3.6
    tol = 1.5 if str(dev) == "cuda" else 2.5
    assert abs(float(mu.mean()) - float(g["es.long.mu.mean"])) < tol, float(mu.mean())
    assert abs(float(tau.mean()) - float(g["es.long.tau.mean"])) < tol, float(tau.mean())


# ---- CPU tier: host logic of the binding on the oracle-backed stand-ins ------------------------------------
@pytest.fixture
def emu():
    import cpu_emulation
    with cpu_emulation.enabled():
        yield


def test_bind_svi_trajectory_reference_pyro_cpu(emu):
    _svi_trajectory("cpu", torch.float64, "f64", 1e-9)


def test_bind_lazy_linear_predictor_cpu(emu):
    _lazy_site_reaches_glm("cpu")


def test_bind_optimizer_state_roundtrip_cpu(emu, tmp_path):
    """``save`` / ``load`` of the fused optimiser inside reference Pyro keeps the reference's state_dict
    schema (pyro/optim/optim.py:157-198; tests/optim/test_optim.py:372-437)."""
    def check(pyro, bind, optim):
        state = optim.get_state()
        assert set(state) == {"w_loc", "w_scale", "b_loc", "b_scale"}
        one = state["w_loc"]
        assert set(one) == {"state", "param_groups"} and one["state"][0]["step"] == 2
        assert {"exp_avg", "exp_avg_sq", "step"} <= set(one["state"][0])
        f = str(tmp_path / "opt.pt")
        optim.save(f)
        other = bind.ClippedAdam({"lr": 0.01})
        other.load(f)
        assert set(other._b2._state_waiting_to_be_consumed) == set(state)
        # a state dict written by the REFERENCE optimiser loads as well (same schema)
        ref_optim = pyro.optim.ClippedAdam({"lr": 0.01})
        store = pyro.get_param_store()
        params = [store[k].unconstrained() for k in ("w_loc", "w_scale", "b_loc", "b_scale")]
        for p in params:
            p.grad = torch.ones_like(p)
        ref_optim(params)
        f2 = str(tmp_path / "ref.pt")
        ref_optim.save(f2)
        third = bind.ClippedAdam({"lr": 0.01})
        third.load(f2)
        for p in params:
            p.grad = torch.ones_like(p)
        third(params)
        st = third.get_state()["w_loc"]["state"][0]
        assert st["step"] == 2 and torch.isfinite(st["exp_avg"]).all()

    _svi_trajectory("cpu", torch.float64, "f64", 1e-9, steps=2, then=check)


def test_bind_nuts_kernel_in_reference_mcmc_cpu(emu):
    _nuts_eight_schools("cpu", "kernel")


# ---- GPU tier: the same scenarios through the real kernels ---------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("tag,dtype,tol", [("f64", torch.float64, 1e-9), ("f32", torch.float32, 3e-4)])
def test_bind_svi_trajectory_reference_pyro_gpu(tag, dtype, tol):
    if EMULATE:
        pytest.skip("covered by the cpu test")
    _svi_trajectory("cuda", dtype, tag, tol)


@pytest.mark.gpu
def test_bind_captured_svi_reference_pyro_gpu():
    """bind.SVI + JitTrace_ELBO: the whole reference-Pyro step captured in a CUDA graph; with injected
    noise the captured steps reproduce the reference trajectory (fp32 tolerance)."""
    if EMULATE:
        pytest.skip("needs CUDA graphs")
    _svi_trajectory("cuda", torch.float32, "f32", 3e-4, svi_cls="SVI", elbo="JitTrace_ELBO")


@pytest.mark.gpu
def test_bind_lazy_linear_predictor_gpu():
    if EMULATE:
        pytest.skip("covered by the cpu test")
    _lazy_site_reaches_glm("cuda")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["kernel", "potential_fn"])
def test_bind_nuts_reference_mcmc_gpu(kind):
    if EMULATE:
        pytest.skip("covered by the cpu test")
    _nuts_eight_schools("cuda", kind)
