"""GPU-tier parity tests added in round 2 (VERDICT r1 "close the GPU-tier test holes"): the scenarios that
round 1 only exercised on the CPU stand-ins now run through the real kernels on device tensors --
score-function ELBO (a10), HMC.sample (b3), warm-up adaptation pieces (b6), r_hat / ESS (b7), optimiser
checkpoints (f3) -- plus the exactness of the CUDA-graph step, the safety of its input buffers, and
the unchanged logistic model reaching the tcgen05 GLM kernel (checked against the oracle at D = 32 and at
the full BASELINE size)."""
import math

import numpy as np
import pytest
import torch
from torch.distributions import constraints

import models
import pyro_b200 as pyro
import pyro_b200.distributions as dist
from conftest import EMULATE, device, load_npz
from oracle import dists as od
from oracle import mcmc as omcmc
from oracle import svi as osvi
from pyro_b200 import poutine
from pyro_b200.infer import HMC, MCMC, SVI, JitTrace_ELBO, Trace_ELBO
from pyro_b200.infer.mcmc import LogisticPotential
from pyro_b200.optim import ClippedAdam

pytestmark = pytest.mark.gpu
DEV = device()


# ---- a10: non-reparameterised guide site -> log_r / score-function surrogate -----------------------------
def test_score_function_path_matches_reference_kat_gpu():
    """tests/infer/test_gradient.py:50-127 style: Bernoulli guide site (no rsample), Rao-Blackwellised
    log_r through MultiFrameTensor; loss and gradient against an independent autograd computation."""
    torch.set_default_dtype(torch.float64)
    data = torch.tensor([1.0, 0.0, 1.0, 1.0], device=DEV)
    zs = torch.tensor([[1.0], [0.0], [1.0]], device=DEV)  # 3 particles

    def model():
        p = pyro.sample("z", dist.Bernoulli(probs=torch.tensor(0.4, device=DEV)))
        with pyro.plate("d", 4):
            pyro.sample("x", dist.Bernoulli(probs=0.2 + 0.6 * p), obs=data)

    class Inject(poutine.Messenger):
        def _pyro_sample(self, msg):
            if msg["name"] == "z":
                msg["value"] = zs
                msg["done"] = True

    def guide():
        q = pyro.param("q", torch.tensor(0.3, device=DEV), constraint=constraints.unit_interval)
        with Inject():
            pyro.sample("z", dist.Bernoulli(probs=q))

    elbo = Trace_ELBO(num_particles=3, vectorize_particles=True, max_plate_nesting=1)
    with poutine.trace(param_only=True) as cap:
        loss = elbo.loss_and_grads(model, guide)
    got = cap.trace.nodes["q"]["value"]._pyro_unconstrained_param.grad.cpu()
    u = torch.tensor(0.3).logit().clone().requires_grad_(True)
    q = torch.sigmoid(u)
    B = torch.distributions.Bernoulli
    zc, dc = zs.cpu(), data.cpu()
    lq = B(probs=q).log_prob(zc)
    lpz = B(probs=torch.tensor(0.4)).log_prob(zc)
    lpx = B(probs=0.2 + 0.6 * zc).log_prob(dc)
    log_r = (lpz - lq).detach() + lpx.sum(-1, keepdim=True).detach()
    (-((log_r * lq).sum()) / 3).backward()
    assert torch.allclose(got, u.grad, atol=1e-10)
    assert abs(loss + float((lpz + lpx.sum(-1, keepdim=True) - lq).sum() / 3)) < 1e-10


# ---- b3: HMC.sample on the device ------------------------------------------------------------------------
def test_hmc_sample_recovers_posterior_logistic_gpu():
    """pyro/infer/mcmc/hmc.py:371-438 (momentum draw, fixed-length trajectory on the leapfrog kernels,
    Metropolis correction, step-size / mass adaptation) against the oracle's recursive NUTS."""
    torch.set_default_dtype(torch.float64)
    g = load_npz("mcmc.npz")
    X, y = torch.as_tensor(g["lr.X"]).to(DEV), torch.as_tensor(g["lr.y"]).to(DEV)
    kernel = HMC(potential_fn=LogisticPotential(X, y, 1.0), step_size=0.1, trajectory_length=1.0)
    mc = MCMC(kernel, num_samples=200, warmup_steps=100, num_chains=16, seed=4)
    mc.run()
    s = mc.get_samples()["beta"].cpu()
    chain = omcmc.NUTSChain(omcmc.logistic_potential(X.cpu(), y.cpu(), 1.0), 3, seed=2)
    ref, _ = chain.run(torch.zeros(3, dtype=torch.float64), 150, 600)
    assert torch.allclose(s.mean(0), ref.mean(0), atol=0.12)
    assert torch.allclose(s.std(0), ref.std(0), atol=0.08)
    assert float(torch.as_tensor(mc.diagnostics()["acceptance rate"]).min()) > 0.5
    assert float(mc.diagnostics()["beta"]["r_hat"].max()) < 1.1


# ---- b6: adaptation pieces on device tensors ---------------------------------------------------------------
def test_adaptation_pieces_on_device_match_reference():
    """Dual averaging (pyro/ops/dual_averaging.py:55-72), Welford + Stan shrinkage
    (pyro/ops/welford.py:27-51) and the window schedule (pyro/infer/mcmc/adaptation.py:98-132) with their
    state on the GPU, against the sequences recorded from the reference."""
    from pyro_b200.infer.mcmc.adaptation import DualAveraging, WelfordDiag, build_adaptation_schedule
    g = load_npz("mcmc.npz")
    for w in (5, 19, 100, 150, 200, 500, 1000):
        assert [[a.start, a.end] for a in build_adaptation_schedule(w)] == g["sched.%d" % w].tolist()
    dev = torch.device(DEV)
    da = DualAveraging(2, dev, prox_center=math.log(10 * 0.3))
    for gg, ref in zip(g["da.g"], g["da.x"]):
        da.step(torch.full((2,), float(gg), dtype=torch.float64, device=dev))
        xt, xavg = da.get_state()
        assert xt.device.type == dev.type
        assert abs(float(xt[1]) - ref[0]) < 1e-12 and abs(float(xavg[0]) - ref[1]) < 1e-12
    wf = WelfordDiag()
    for s in torch.as_tensor(g["wf.samples"]).to(dev):
        wf.update(s.expand(3, -1))
    assert torch.allclose(wf.get_covariance(True)[2].cpu(), torch.as_tensor(g["wf.cov_reg"]), atol=1e-12)


# ---- b7: diagnostics on device tensors --------------------------------------------------------------------
def test_stats_on_device_match_reference():
    from pyro_b200.infer.mcmc.stats import effective_sample_size, split_gelman_rubin
    g = load_npz("mcmc.npz")
    x = torch.as_tensor(g["stats.x"]).to(DEV)
    r, n = split_gelman_rubin(x), effective_sample_size(x)
    assert r.device.type == torch.device(DEV).type
    assert torch.allclose(r.cpu(), torch.as_tensor(g["stats.rhat"]), atol=1e-10)
    assert torch.allclose(n.cpu(), torch.as_tensor(g["stats.neff"]), rtol=1e-8)


# ---- f3: optimiser checkpoints on the device ---------------------------------------------------------------
def _noise_guide(eps_w, eps_b, box):
    def guide(X, y):
        with models.InjectNoise({"w": eps_w[box["i"]], "b": eps_b[box["i"]]}):
            models.logistic_guide(X, y)
    return guide


def test_optimizer_checkpoint_roundtrip_gpu(tmp_path):
    """tests/optim/test_optim.py:372-437: save -> clear -> load -> identical trajectory, fused kernels."""
    torch.set_default_dtype(torch.float64)
    g = load_npz("svi_logistic.npz")
    X, y = torch.as_tensor(g["X"]).to(DEV), torch.as_tensor(g["y"]).to(DEV)
    eps_w, eps_b = torch.as_tensor(g["eps_w"]).to(DEV), torch.as_tensor(g["eps_b"]).to(DEV)
    box = {"i": 0}
    guide = _noise_guide(eps_w, eps_b, box)

    def make():
        return SVI(models.logistic_model, guide, ClippedAdam({"lr": 0.01, "lrd": 0.9}),
                   Trace_ELBO(num_particles=8, vectorize_particles=True, max_plate_nesting=1))
    svi = make()
    for i in range(2):
        box["i"] = i
        svi.step(X, y)
    svi.optim.save(str(tmp_path / "opt.pt"))
    pyro.get_param_store().save(str(tmp_path / "params.pt"))
    state = svi.optim.get_state()
    assert state["w_loc"]["state"][0]["step"] == 2
    assert abs(state["w_loc"]["param_groups"][0]["lr"] - 0.01 * 0.9 ** 2) < 1e-15
    ref = []
    for i in range(2, 5):
        box["i"] = i
        ref.append(svi.step(X, y))
    pyro.clear_param_store()
    pyro.get_param_store().load(str(tmp_path / "params.pt"), map_location=DEV)
    svi2 = make()
    svi2.optim.load(str(tmp_path / "opt.pt"), map_location=DEV)
    got = []
    for i in range(2, 5):
        box["i"] = i
        got.append(svi2.step(X, y))
    assert np.allclose(ref, got, rtol=1e-12)


# ---- the CUDA-graph step: exact, one update per call, never writes the caller's tensors --------------------
def _graph_run(elbo_cls, dtype, tag, steps, tol):
    """Noise is injected through fixed device buffers refilled before every step, so the eager and the
    captured runs consume identical draws and can be compared exactly -- and with the reference goldens."""
    g = load_npz("svi_logistic.npz")
    torch.set_default_dtype(dtype)
    pyro.clear_param_store()
    X, y = torch.as_tensor(g["X"]).to(DEV, dtype), torch.as_tensor(g["y"]).to(DEV, dtype)
    eps_w, eps_b = torch.as_tensor(g["eps_w"]).to(DEV, dtype), torch.as_tensor(g["eps_b"]).to(DEV, dtype)
    bw, bb = torch.empty_like(eps_w[0]), torch.empty_like(eps_b[0])

    def guide(X, y):
        with models.InjectNoise({"w": bw, "b": bb}):
            models.logistic_guide(X, y)

    svi = SVI(models.logistic_model, guide, ClippedAdam({"lr": 0.01}),
              elbo_cls(num_particles=int(g["P"]), vectorize_particles=True, max_plate_nesting=1))
    losses, traj = [], []
    for i in range(steps):
        bw.copy_(eps_w[i])
        bb.copy_(eps_b[i])
        losses.append(svi.step(X, y))
        store = pyro.get_param_store()
        traj.append(torch.cat([store[k].detach().reshape(-1).double().cpu()
                               for k in ("w_loc", "w_scale", "b_loc", "b_scale")]))
        assert abs(losses[-1] - g["losses_" + tag][i]) <= 10 * tol * abs(g["losses_" + tag][i]), (i, losses[-1])
        assert torch.allclose(traj[-1], torch.as_tensor(g["params_" + tag][i]), atol=10 * tol, rtol=10 * tol), i
    steps_done = svi.optim.get_state()["w_loc"]["state"][0]["step"]
    return losses, traj, steps_done


@pytest.mark.parametrize("tag,dtype,tol", [("f64", torch.float64, 1e-9), ("f32", torch.float32, 3e-4)])
def test_captured_graph_step_is_exact_and_counts_one_update_per_call(tag, dtype, tol):
    if EMULATE:
        pytest.skip("graph capture needs a GPU")
    l_e, p_e, n_e = _graph_run(Trace_ELBO, dtype, tag, 5, tol)
    l_g, p_g, n_g = _graph_run(JitTrace_ELBO, dtype, tag, 5, tol)
    assert n_e == 5 and n_g == 5          # the capturing call performs exactly ONE update
    exact = 1e-12 if dtype == torch.float64 else 2e-6
    for a, b in zip(l_e, l_g):
        assert abs(a - b) <= exact * abs(a)
    for a, b in zip(p_e, p_g):
        assert torch.allclose(a, b, atol=exact, rtol=exact)


def test_captured_step_never_writes_caller_tensors():
    """A resident data set stepped through minibatch VIEWS: the graph first reads the caller's tensor in
    place; when another view arrives it re-captures with private buffers instead of copying into the
    first view (ADVICE r1, svi.py:180)."""
    if EMULATE:
        pytest.skip("graph capture needs a GPU")
    torch.manual_seed(0)
    N_, D, B = 4096, 8, 1024
    X = torch.randn(N_, D, device=DEV)
    y = (torch.rand(N_, device=DEV) < torch.sigmoid(X[:, 0])).float()
    X0, y0 = X.clone(), y.clone()
    pyro.clear_param_store()
    svi = SVI(models.logistic_model, models.logistic_guide, ClippedAdam({"lr": 0.01}),
              JitTrace_ELBO(num_particles=8, vectorize_particles=True, max_plate_nesting=1))
    for k in range(12):
        i = (k * B) % N_
        loss = svi.step(X[i:i + B], y[i:i + B])
        assert loss == loss
    assert torch.equal(X, X0) and torch.equal(y, y0)
    assert svi.optim.get_state()["w_loc"]["state"][0]["step"] == 12


# ---- the unchanged model reaches the tcgen05 GLM kernel; parity against the oracle --------------------------
def test_unchanged_logistic_model_d32_matches_oracle_trajectory():
    """models.logistic_model is the reference model verbatim (`w.squeeze(-2) @ X.T + b`); at D = 32 its
    likelihood site is scored by the tcgen05 kernel (lazy linear predictor).  Three SVI steps with
    injected noise against oracle/svi.py (itself pinned to reference Pyro's trajectory)."""
    torch.manual_seed(0)
    N_, D, P = 70000, 32, 16          # >= 64 Ki rows: the default (W-split) precision mode
    X = torch.randn(N_, D)
    y = (torch.rand(N_) < torch.sigmoid(X[:, 0] - 0.5 * X[:, 1] + 0.25)).float()
    eps_w, eps_b = torch.randn(3, P, 1, D), torch.randn(3, P, 1)
    ref = osvi.LogisticSVIMatmul(D, P, lr=0.01)
    ref_losses = [ref.step(X, y, eps_w[i], eps_b[i]) for i in range(3)]
    pyro.clear_param_store()
    Xd, yd = X.to(DEV), y.to(DEV)
    box = {"i": 0}
    seen = []

    def guide(X_, y_):
        with models.InjectNoise({"w": eps_w[box["i"]].to(DEV), "b": eps_b[box["i"]].to(DEV)}):
            models.logistic_guide(X_, y_)

    real = dist._BernoulliLinear._fused_sum

    def spy(self, *a, **k):
        seen.append(type(self).__name__)
        return real(self, *a, **k)
    dist._BernoulliLinear._fused_sum = spy
    try:
        svi = SVI(models.logistic_model, guide, ClippedAdam({"lr": 0.01}),
                  Trace_ELBO(num_particles=P, vectorize_particles=True, max_plate_nesting=1))
        for i in range(3):
            box["i"] = i
            loss = svi.step(Xd, yd)
            assert abs(loss - ref_losses[i]) <= 2e-5 * abs(ref_losses[i]), (i, loss, ref_losses[i])
    finally:
        dist._BernoulliLinear._fused_sum = real
    assert len(seen) == 3                      # every step took the fused GLM site
    got = pyro.get_param_store()
    cons = ref.constrained()
    for k in ("w_loc", "w_scale", "b_loc", "b_scale"):
        assert torch.allclose(got[k].detach().cpu().reshape(-1), cons[k].reshape(-1), atol=2e-4), k


@pytest.mark.parametrize("flag_name,tol_sum,tol_g", [("default", 2e-5, 2e-4), ("B2_FLAG_GLM_3XTF32", 2e-5, 2e-4)])
def test_glm_kernel_full_size_against_oracle(flag_name, tol_sum, tol_g):
    """BASELINE size (N = 1e6, D = 32, P = 64): per-particle sums, dW and db of the tcgen05 kernel against
    the oracle's fp64 Bernoulli log-density (oracle/dists.py) differentiated by autograd on the CPU.
    Default path: fp32 tolerances (2e-5 on sums, 2e-4 x scale on gradients)."""
    if EMULATE:
        pytest.skip("kernel test")
    import ctypes  # noqa: F401
    from pyro_b200 import _native as N
    torch.manual_seed(1)
    n, D, P = 1_000_000, 32, 64
    X = torch.randn(n, D)
    wt = torch.randn(D) / D ** 0.5
    y = (torch.rand(n) < torch.sigmoid(X @ wt + 0.5)).float()
    W = (0.3 * torch.randn(P, D) + wt)
    b = 0.5 + 0.2 * torch.randn(P)
    Wd = W.double().requires_grad_(True)
    bd = b.double().requires_grad_(True)
    lp = od.bernoulli_logits(y.double(), Wd @ X.double().t() + bd[:, None])
    s_ref = lp.sum(1)
    gW, gb = torch.autograd.grad(s_ref.sum(), [Wd, bd])
    Xg, yg, Wg, bg = X.to(DEV), y.to(DEV), W.to(DEV).contiguous(), b.to(DEV).contiguous()
    sum_p = torch.empty(P, device=DEV)
    total = torch.empty((), device=DEV)
    dW = torch.empty(P, D, device=DEV)
    db = torch.empty(P, device=DEV)
    ws = N.workspace(torch.device(DEV), int(N.lib().b2_glm_workspace(n, D, P)), tag="glm_full")
    flags = 0 if flag_name == "default" else getattr(N, flag_name)
    N.check(N.lib().b2_glm_bernoulli_logits(Xg.data_ptr(), yg.data_ptr(), Wg.data_ptr(), bg.data_ptr(), n, D, P,
                                            1.0, 1.0, 1.0, flags, sum_p.data_ptr(), total.data_ptr(),
                                            dW.data_ptr(), db.data_ptr(), ws.data_ptr(), ws.numel(),
                                            N.stream_ptr(torch.device(DEV))), "b2_glm_bernoulli_logits")
    torch.cuda.synchronize()
    assert float(((sum_p.double().cpu() - s_ref).abs() / s_ref.abs()).max()) <= tol_sum
    assert abs(float(total) - float(s_ref.sum())) <= tol_sum * abs(float(s_ref.sum()))
    assert float((dW.double().cpu() - gW).abs().max()) <= tol_g * float(gW.abs().max())
    assert float((db.double().cpu() - gb).abs().max()) <= tol_g * float(gb.abs().max())
    # size-independent property: the launch is deterministic (fixed-order reductions, no float atomics)
    sum2 = torch.empty(P, device=DEV)
    N.check(N.lib().b2_glm_bernoulli_logits(Xg.data_ptr(), yg.data_ptr(), Wg.data_ptr(), bg.data_ptr(), n, D, P,
                                            1.0, 1.0, 1.0, flags, sum2.data_ptr(), total.data_ptr(),
                                            dW.data_ptr(), db.data_ptr(), ws.data_ptr(), ws.numel(),
                                            N.stream_ptr(torch.device(DEV))), "b2_glm_bernoulli_logits")
    torch.cuda.synchronize()
    assert torch.equal(sum_p, sum2)


@pytest.mark.parametrize("n,P,bias,flag,y_offset", [
    (1, 1, True, "B2_FLAG_GLM_3XTF32", 0), (127, 3, False, "B2_FLAG_GLM_3XTF32", 0),
    (128, 64, True, "B2_FLAG_GLM_3XTF32", 0), (129, 65, True, "B2_FLAG_GLM_3XTF32", 0),
    (1, 1, True, None, 0), (5000, 130, False, None, 0),
    (8192, 64, True, None, 0), (70001, 64, True, None, 0), (65535, 130, False, None, 0),
    (20000, 64, True, None, 4)])
def test_glm_tc_kernel_ragged_shapes_against_oracle(n, P, bias, flag, y_offset):
    """Edge cases of the tiled kernel: a single row, one row short of / one past a 128-row tile, ragged
    particle slabs (65, 130), no bias.  With an explicit tensor-core flag the tcgen05 kernel runs at any
    size and its gradient contraction is single-pass TF32 on round-to-nearest operands: the tolerance is
    2^-11 of the LARGEST TERM budget (5e-4 x scale) for tiny N, where nothing averages; the default
    dispatch (flag None: exact fp32 SIMT below 8 Ki rows, tcgen05 above) must meet the fp32 tolerances.
    y_offset: y starts that many bytes past a 16-byte boundary, which TMA cannot load; such a y takes the
    fp32 SIMT kernel at any size."""
    if EMULATE:
        pytest.skip("kernel test")
    from pyro_b200 import _native as N
    torch.manual_seed(n + P)
    D = 32
    X = torch.randn(n, D)
    y = (torch.rand(n) < 0.4).float()
    W = 0.3 * torch.randn(P, D)
    b = torch.randn(P) if bias else None
    logits = W.double() @ X.double().t() + (b.double()[:, None] if bias else 0.0)
    s_ref = od.bernoulli_logits(y.double(), logits).sum(1)
    g = y.double() - torch.sigmoid(logits)
    gW, gb = g @ X.double(), g.sum(1)
    Xg, Wg = X.to(DEV), W.to(DEV)
    yg = torch.cat([torch.zeros(y_offset // 4), y]).to(DEV)[y_offset // 4:]
    assert yg.data_ptr() % 16 == y_offset
    bg = b.to(DEV) if bias else None
    sum_p = torch.empty(P, device=DEV)
    dW = torch.empty(P, D, device=DEV)
    db = torch.empty(P, device=DEV)
    ws = N.workspace(torch.device(DEV), int(N.lib().b2_glm_workspace(n, D, P)), tag="glm_ragged")
    N.check(N.lib().b2_glm_bernoulli_logits(Xg.data_ptr(), yg.data_ptr(), Wg.data_ptr(),
                                            bg.data_ptr() if bias else None, n, D, P, 1.0, 1.0, 1.0,
                                            getattr(N, flag) if flag else 0,
                                            sum_p.data_ptr(), None, dW.data_ptr(), db.data_ptr(), ws.data_ptr(),
                                            ws.numel(), N.stream_ptr(torch.device(DEV))), "b2_glm_bernoulli_logits")
    torch.cuda.synchronize()
    tol_g = 5e-4 if flag else 2e-4
    assert float((sum_p.double().cpu() - s_ref).abs().max()) <= 2e-5 * max(1.0, float(s_ref.abs().max()))
    assert float((dW.double().cpu() - gW).abs().max()) <= tol_g * max(1.0, float(gW.abs().max()))
    assert float((db.double().cpu() - gb).abs().max()) <= tol_g * max(1.0, float(gb.abs().max()))


def test_full_mass_nuts_correlated_posterior_gpu():
    """``NUTS(full_mass=True)`` (dense mass matrix via whitened coordinates) on the device."""
    from test_host_logic_cpu import _full_mass_case
    _full_mass_case(DEV)


def test_slice_sampling_nuts_posterior_gpu():
    from test_host_logic_cpu import _slice_nuts_case
    _slice_nuts_case(DEV)


def test_config4_potential_and_integrator_at_baseline_size():
    """BASELINE config 4 at its stated size (J = 1 000 000 groups, D = J + 2): the native hierarchical-Normal
    potential and gradient against the fp64 oracle (oracle/mcmc.py, chain 0 and chain 3 of 4), and two
    size-independent properties of the C-ABI leapfrog at that size -- time reversibility (n steps forward,
    momentum flipped, n steps back returns to the start) and second-order convergence of the energy error."""
    if EMULATE:
        pytest.skip("needs the device kernels")
    from pyro_b200.infer.mcmc import HierNormalPotential
    torch.manual_seed(4)
    J, C = 1_000_000, 4
    sig = 5 + 15 * torch.rand(J, device=DEV)
    yy = 5 + 3 * torch.randn(J, device=DEV) + sig * torch.randn(J, device=DEV)
    pot = HierNormalPotential(yy, sig)
    z = torch.cat([torch.randn(C, 2, device=DEV) * 0.1, torch.randn(C, J, device=DEV)], 1).contiguous()
    U, G = pot.value_and_grad(z)
    ref_U = omcmc.eight_schools_potential(yy.double().cpu(), sig.double().cpu())
    for c in (0, 3):
        g_ref, u_ref = omcmc.potential_grad(ref_U, z[c].double().cpu())
        assert abs(float(U[c]) - float(u_ref)) <= 2e-6 * abs(float(u_ref))
        assert float((G[c].double().cpu() - g_ref).abs().max()) <= 1e-3 * max(1.0, float(g_ref.abs().max()))
    k = HMC(potential_fn=pot, adapt_step_size=False, adapt_mass_matrix=False)
    k.setup(0, C, initial_params=z.clone())
    minv = torch.ones(C, J + 2, device=DEV)
    r0 = torch.randn(C, J + 2, device=DEV)
    e0 = U + 0.5 * (r0 * r0).sum(1)

    def run(step, n):
        eps = torch.full((C,), step, device=DEV)
        zc, rc, gc = z.clone(), r0.clone(), G.clone()
        for _ in range(n):
            zc, rc, gc, Uc, ke = k._leapfrog(zc, rc, gc, eps, minv)
        return zc, rc, gc, (Uc + ke - e0), eps

    # second order: the same trajectory length with half the step has ~1/4 of the energy error (errors of a few
    # hundred / tens on a total energy of 6e6 -- O(eps^2 D) -- well above the fp32 noise of the sums)
    _, _, _, err_coarse, _ = run(2e-3, 4)
    zc, rc, gc, err_fine, eps = run(1e-3, 8)
    assert float((err_fine.abs() / e0.abs()).max()) < 1e-4
    ratio = (err_coarse / err_fine).cpu()
    assert bool(((ratio > 2.5) & (ratio < 6.5)).all()), ratio
    # time reversibility: flip the momentum, integrate back
    rb = (-rc).contiguous()
    zb, gb = zc, gc
    for _ in range(8):
        zb, rb, gb, _, _ = k._leapfrog(zb, rb, gb, eps, minv)
    assert float((zb - z).abs().max()) < 5e-5
    assert float((rb + r0).abs().max()) < 5e-4
