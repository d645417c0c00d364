"""End-to-end parity of the two hot paths on the GPU: SVI steps (eager, fused GLM, CUDA-graph
captured) against the reference's recorded trajectory; optimisers; leapfrog / potentials / NUTS
against goldens and the oracle.  See test_gpu_kernels.py for the tolerance policy."""
import math

import numpy as np
import pytest
import torch
from torch.distributions import constraints

import models
import pyro_b200 as pyro
import pyro_b200.distributions as dist
from conftest import device, load_npz, EMULATE
from oracle import mcmc as omcmc
from oracle import svi as osvi
from pyro_b200 import poutine
from pyro_b200.infer import MCMC, NUTS, HMC, SVI, JitTrace_ELBO, Trace_ELBO, TraceMeanField_ELBO
from pyro_b200.infer.mcmc import HierNormalPotential, LogisticPotential, TracePotential
from pyro_b200.optim import AdagradRMSProp, ClippedAdam

pytestmark = pytest.mark.gpu
DEV = device()


def _svi_trajectory(model, elbo_cls, dtype, tag, tol, steps=None, fused_draw=False):
    g = load_npz("svi_logistic.npz")
    torch.set_default_dtype(dtype)
    X, y = torch.as_tensor(g["X"]).to(DEV, dtype), torch.as_tensor(g["y"]).to(DEV, dtype)
    eps_w, eps_b = torch.as_tensor(g["eps_w"]).to(DEV, dtype), torch.as_tensor(g["eps_b"]).to(DEV, dtype)
    P = int(g["P"])
    box = {"i": 0}

    def guide(X, y):
        with models.InjectNoise({"w": eps_w[box["i"]], "b": eps_b[box["i"]]}, fused_draw=fused_draw):
            models.logistic_guide(X, y)

    svi = SVI(model, guide, ClippedAdam({"lr": 0.01}),
              elbo_cls(num_particles=P, vectorize_particles=True, max_plate_nesting=1))
    for i in range(eps_w.shape[0] if steps is None else steps):
        box["i"] = i
        loss = svi.step(X, y)
        assert abs(loss - g["losses_" + tag][i]) <= 10 * tol * abs(g["losses_" + tag][i]), (i, loss)
        store = pyro.get_param_store()
        flat = torch.cat([store[k].detach().reshape(-1).double().cpu() for k in ("w_loc", "w_scale", "b_loc", "b_scale")])
        assert torch.allclose(flat, torch.as_tensor(g["params_" + tag][i]), atol=10 * tol, rtol=10 * tol), i


@pytest.mark.parametrize("tag,dtype,tol", [("f64", torch.float64, 1e-9), ("f32", torch.float32, 3e-4)])
@pytest.mark.parametrize("fused_draw", [False, True])
def test_svi_logistic_matches_reference_trajectory(tag, dtype, tol, fused_draw):
    """fused_draw: the guide draws and their log densities come from the fused rsample kernel
    (b2 family 14) and the ELBO claims them; otherwise every site is scored by b2_site_score."""
    _svi_trajectory(models.logistic_model, Trace_ELBO, dtype, tag, tol, fused_draw=fused_draw)


def test_svi_logistic_fused_glm_matches_reference_trajectory():
    """fp32 SIMT GLM kernel (D = 4 here, so the tensor-core path is not taken): ELBO within 5e-4
    relative, parameters within 5e-3 absolute of the reference after 5 steps."""
    _svi_trajectory(models.logistic_model_fused, Trace_ELBO, torch.float32, "f32", 5e-4)


def test_tf32_glm_elbo_close_to_fp32_at_scale():
    """Stated tolerance of the tensor-core likelihood at BASELINE size (N = 1e6, D = 32, P = 64):
    ELBO term within 1e-5 relative of the fp32 kernel, gradients within 1e-3 of their scale."""
    if EMULATE:
        pytest.skip("needs the device kernels")
    torch.manual_seed(0)
    n, D, P = 1_000_000, 32, 64
    X = torch.randn(n, D, device=DEV)
    y = (torch.rand(n, device=DEV) < torch.sigmoid(X[:, 0])).float()
    w = (0.1 * torch.randn(P, 1, D, device=DEV)).requires_grad_(True)
    b = torch.zeros(P, 1, device=DEV, requires_grad=True)
    res = []
    for tc in (False, True):
        out = dist.Bernoulli(logits=dist.linear_predictor(X, w, b, tensor_cores=tc))._fused_sum(y, None, 1.0, -1.0 / P, 1.0, True)
        gw, gb = torch.autograd.grad(out, [w, b])
        res.append((float(out), gw, gb))
    assert abs(res[0][0] - res[1][0]) <= 1e-5 * abs(res[0][0])
    assert float((res[0][1] - res[1][1]).abs().max()) <= 1e-3 * float(res[0][1].abs().max())
    assert float((res[0][2] - res[1][2]).abs().max()) <= 1e-3 * max(1.0, float(res[0][2].abs().max()))


@pytest.mark.parametrize("tensor_cores", [False, True])
def test_glm_kernel_against_oracle(tensor_cores):
    """X, y read once; sum / dW / db vs float64 autograd of the oracle, ragged N, several D and P:
    sum within 2e-5 relative, gradients 2e-4.  Every size here is below 8 Ki rows, so tensor_cores=True
    (no B2_FLAG_GLM_FP32) also takes the exact fp32 SIMT kernel and is held to the same tolerances."""
    torch.manual_seed(0)
    for (n, D, P) in [(1, 4, 1), (63, 8, 3), (64, 16, 64), (1000, 32, 7), (4097, 32, 64), (130, 4, 130),
                      (1, 32, 1), (65, 32, 33), (200, 32, 130)]:
        X = torch.randn(n, D, device=DEV)
        y = (torch.rand(n, device=DEV) < 0.4).float()
        w = (0.5 * torch.randn(P, 1, D, device=DEV)).requires_grad_(True)
        b = torch.randn(P, 1, device=DEV).requires_grad_(True)
        d = dist.Bernoulli(logits=dist.linear_predictor(X, w, b, tensor_cores=tensor_cores))
        out = d._fused_sum(y, None, 1.5, -0.25, 1.0, True)
        gw, gb = torch.autograd.grad(out, [w, b])
        wo = w.detach().double().cpu().requires_grad_(True)
        bo = b.detach().double().cpu().requires_grad_(True)
        logits = wo.squeeze(-2) @ X.double().cpu().t() + bo
        from oracle import dists as od
        tot = (od.bernoulli_logits(y.double().cpu(), logits) * 1.5).sum()
        tol_sum = 2e-5 * max(1.0, abs(float(tot)))
        assert abs(float(out) - float(tot)) <= tol_sum, (n, D, P, float(out), float(tot))
        ow, ob = torch.autograd.grad(-0.25 * tot, [wo, bo])
        gt = 2e-4
        sc = max(1.0, float(ow.abs().max()))
        assert float((gw.double().cpu() - ow).abs().max()) <= gt * sc, (n, D, P)
        assert float((gb.double().cpu() - ob).abs().max()) <= gt * max(1.0, float(ob.abs().max())), (n, D, P)


def test_captured_graph_step_equals_eager():
    """JitTrace_ELBO analogue: the CUDA-graph replayed step must follow the same trajectory as eager
    steps when the guide noise comes from the same generator state."""
    if EMULATE:
        pytest.skip("graph capture needs a GPU")
    torch.manual_seed(0)
    N_, D, P = 4096, 8, 16
    X = torch.randn(N_, D, device=DEV)
    y = (torch.rand(N_, device=DEV) < torch.sigmoid(X[:, 0])).float()

    def run(elbo_cls, nsteps):
        pyro.clear_param_store()
        torch.manual_seed(1)
        torch.cuda.manual_seed(1)
        svi = SVI(models.logistic_model, models.logistic_guide, ClippedAdam({"lr": 0.05}),
                  elbo_cls(num_particles=P, vectorize_particles=True, max_plate_nesting=1))
        losses = [svi.step(X, y) for _ in range(nsteps)]
        store = pyro.get_param_store()
        return losses, {k: store[k].detach().clone() for k in store.keys()}

    l_e, p_e = run(Trace_ELBO, 40)
    l_g, p_g = run(JitTrace_ELBO, 40)
    # different RNG consumption under capture -> compare statistically: both must have learned
    assert l_g[-1] < l_g[0] and l_e[-1] < l_e[0]
    assert abs(np.mean(l_g[-10:]) - np.mean(l_e[-10:])) < 0.05 * abs(np.mean(l_e[-10:]))
    for k in p_e:
        assert torch.allclose(p_e[k], p_g[k], atol=0.15), k


@pytest.mark.parametrize("cls,tag", [(Trace_ELBO, "trace"), (TraceMeanField_ELBO, "meanfield")])
def test_elbo_grads_gamma_poisson_mask_subsample(cls, tag):
    g = load_npz("elbo_grad.npz")
    torch.set_default_dtype(torch.float64)
    data, counts = torch.as_tensor(g["data"]).to(DEV), torch.as_tensor(g["counts"]).to(DEV)
    mask = torch.as_tensor(g["mask"]).to(DEV)
    eps, ueps = torch.as_tensor(g["eps"]).to(DEV), torch.as_tensor(g["ueps"]).to(DEV)
    n = data.shape[0]
    T = lambda v: torch.tensor(v, device=DEV)  # noqa: E731

    def model():
        z = pyro.sample("z", dist.Normal(T(0.0), T(2.0)))
        rate = pyro.sample("rate", dist.Gamma(T(2.0), T(0.5)))
        with pyro.plate("data", 2 * n, subsample_size=n, dim=-1):
            with poutine.mask(mask=mask):
                pyro.sample("x", dist.Normal(z, T(1.3)), obs=data)
            pyro.sample("c", dist.Poisson(rate), obs=counts)

    class Inject(poutine.Messenger):
        def __init__(self, vals):
            self.vals = vals

        def _pyro_sample(self, msg):
            if msg["name"] in self.vals:
                msg["value"] = self.vals[msg["name"]]
                msg["done"] = True

    def guide():
        loc = pyro.param("loc", T(0.3))
        scale = pyro.param("scale", T(0.7), constraint=constraints.positive)
        conc = pyro.param("conc", T(3.0), constraint=constraints.positive)
        grate = pyro.param("grate", T(1.2), constraint=constraints.positive)
        with Inject({"z": loc + eps * scale, "rate": conc / grate * (0.5 + ueps)}):
            pyro.sample("z", dist.Normal(loc, scale))
            pyro.sample("rate", dist.Gamma(conc, grate))

    elbo = cls(num_particles=6, vectorize_particles=True, max_plate_nesting=1)
    with poutine.trace(param_only=True) as cap:
        loss = elbo.loss_and_grads(model, guide)
    assert abs(loss - float(g[tag + ".loss"])) < 1e-8 * abs(float(g[tag + ".loss"]))
    for name, site in cap.trace.nodes.items():
        ref = torch.as_tensor(g["%s.grad.%s" % (tag, name)])
        got = site["value"]._pyro_unconstrained_param.grad.cpu()
        assert torch.allclose(got, ref, atol=1e-7, rtol=1e-7), name


@pytest.mark.parametrize("tag,dtype,tol", [("f64", torch.float64, 1e-12), ("f32", torch.float32, 2e-6)])
@pytest.mark.parametrize("q_shape", [(5, 3), (70, 100)])
def test_fused_optimisers_match_reference(tag, dtype, tol, q_shape):
    """q_shape (5, 3): every tensor fits one CTA, ClippedAdam's advance + update is ONE launch;
    (70, 100) exceeds that bound and takes the advance kernel + multi-CTA update kernel."""
    g = load_npz("optim.npz")
    for name, mk in (
        ("clipped_adam", lambda: ClippedAdam({"lr": 0.05, "betas": (0.9, 0.99), "clip_norm": 2.0, "lrd": 0.97, "weight_decay": 0.01})),
        ("clipped_adam_default", lambda: ClippedAdam({"lr": 0.01})),
        ("adagrad_rmsprop", lambda: AdagradRMSProp({"eta": 4.5, "t": 0.1})),
    ):
        p = torch.as_tensor(g["p0_" + tag]).to(DEV).clone().requires_grad_(True)
        q = torch.zeros(q_shape, device=DEV, dtype=dtype).requires_grad_(True)  # a second tensor in the same launch
        pyro.get_param_store()._param_to_name[p] = "p"
        pyro.get_param_store()._param_to_name[q] = "q"
        opt = mk()
        p.grad = torch.zeros_like(p)
        q.grad = torch.zeros_like(q)
        for i, gr in enumerate(torch.as_tensor(g["grads_" + tag]).to(DEV)):
            p.grad.copy_(gr)
            q.grad.fill_(0.1)
            opt([p, q])
            ref = torch.as_tensor(g["%s_%s" % (name, tag)][i])
            assert torch.allclose(p.detach().cpu(), ref, atol=tol, rtol=tol), (name, i)
            assert float(p.grad.abs().max()) == 0.0  # zeroed in the same pass
        st = opt.get_state()["p"]["state"][0]
        assert st["step"] == 12


def test_native_potentials_and_leapfrog_match_reference():
    g = load_npz("mcmc.npz")
    dt = torch.float64
    y, sigma = torch.as_tensor(g["es.y"]).to(DEV), torch.as_tensor(g["es.sigma"]).to(DEV)
    Z = torch.as_tensor(g["es.Z"]).to(DEV)
    pot = HierNormalPotential(y, sigma, 10.0, 25.0)
    U, G = pot.value_and_grad(Z)
    assert torch.allclose(U.cpu(), torch.as_tensor(g["es.U"]), atol=1e-9, rtol=1e-10)
    assert torch.allclose(G.cpu(), torch.as_tensor(g["es.G"]), atol=1e-9, rtol=1e-10)
    lp = LogisticPotential(torch.as_tensor(g["lr.X"]).to(DEV), torch.as_tensor(g["lr.y"]).to(DEV), 1.0)
    U, G = lp.value_and_grad(torch.as_tensor(g["lr.B"]).to(DEV))
    assert torch.allclose(U.cpu(), torch.as_tensor(g["lr.U"]), atol=1e-9, rtol=1e-10)
    assert torch.allclose(G.cpu(), torch.as_tensor(g["lr.G"]), atol=1e-9, rtol=1e-10)
    # 7 leapfrog steps of the C-ABI integrator == reference velocity_verlet (integrator.py:14-65)
    k = HMC(potential_fn=pot, adapt_step_size=False, adapt_mass_matrix=False)
    k.setup(0, 1, initial_params=Z[:1].clone())
    z = Z[:1].clone().contiguous()
    r = torch.as_tensor(g["es.vv.r0"]).to(DEV)[None].contiguous()
    minv = torch.as_tensor(g["es.vv.minv"]).to(DEV)[None].contiguous()
    eps = torch.full((1,), 0.05, dtype=dt, device=DEV)
    _, gcur = pot.value_and_grad(z)
    for _ in range(7):
        z, r, gcur, Ucur, ke = k._leapfrog(z, r, gcur, eps, minv)
    assert torch.allclose(z[0].cpu(), torch.as_tensor(g["es.vv.z"]), atol=1e-9)
    assert torch.allclose(r[0].cpu(), torch.as_tensor(g["es.vv.r"]), atol=1e-9)
    assert abs(float(Ucur) - float(g["es.vv.U"])) < 1e-8
    assert abs(float(ke) - 0.5 * float((minv * r * r).sum())) < 1e-9
    # fp32, large J, many chains: property test (energy error of a short trajectory is O(eps^2))
    torch.manual_seed(0)
    J, C = 200_000, 8
    sig = (5 + 15 * torch.rand(J, device=DEV))
    yy = 5 + 3 * torch.randn(J, device=DEV) + sig * torch.randn(J, device=DEV)
    big = HierNormalPotential(yy, sig)
    z = torch.cat([torch.randn(C, 2, device=DEV) * 0.1, torch.randn(C, J, device=DEV)], 1).contiguous()
    U1, G1 = big.value_and_grad(z)
    ref_U = omcmc.eight_schools_potential(yy.double().cpu(), sig.double().cpu())
    g_ref, u_ref = omcmc.potential_grad(ref_U, z[0].double().cpu())
    assert abs(float(U1[0]) - float(u_ref)) <= 2e-6 * abs(float(u_ref))
    assert float((G1[0].double().cpu() - g_ref).abs().max()) <= 1e-3 * max(1.0, float(g_ref.abs().max()))


def test_trace_potential_matches_reference():
    torch.set_default_dtype(torch.float64)
    g = load_npz("mcmc.npz")
    y, sigma = torch.as_tensor(g["es.y"]).to(DEV), torch.as_tensor(g["es.sigma"]).to(DEV)
    Z = torch.as_tensor(g["es.Z"]).to(DEV)
    pot = TracePotential(models.eight_schools, (sigma, y), {}, num_chains=Z.shape[0])
    order = list(pot.sites)
    cols = {"mu": Z[:, 0:1], "tau": Z[:, 1:2], "eta": Z[:, 2:]}
    U, G = pot.value_and_grad(torch.cat([cols[n] for n in order], dim=1))
    assert torch.allclose(U.cpu(), torch.as_tensor(g["es.U"]), atol=1e-9, rtol=1e-9)
    Gr = torch.as_tensor(g["es.G"])
    ref_cols = {"mu": Gr[:, 0:1], "tau": Gr[:, 1:2], "eta": Gr[:, 2:]}
    assert torch.allclose(G.cpu(), torch.cat([ref_cols[n] for n in order], dim=1), atol=1e-9, rtol=1e-9)


def test_native_nuts_eight_schools_posterior():
    """BASELINE config 1 through the whole-transition kernel: posterior moments vs the reference's
    long run (golden es.long.*); tolerances in the spirit of tests/infer/mcmc/test_nuts.py."""
    if EMULATE:
        pytest.skip("needs the device kernel")
    g = load_npz("mcmc.npz")
    y, sigma = torch.as_tensor(g["es.y"]).to(DEV), torch.as_tensor(g["es.sigma"]).to(DEV)
    kernel = NUTS(potential_fn=HierNormalPotential(y, sigma, 10.0, 25.0))
    mc = MCMC(kernel, num_samples=1000, warmup_steps=300, num_chains=16, seed=0)
    mc.run()
    s = mc.get_samples()
    assert abs(float(s["mu"].mean()) - float(g["es.long.mu.mean"][0])) < 0.4
    assert abs(float(s["tau"].mean()) - float(g["es.long.tau.mean"][0])) < 0.6
    assert float((s["eta"].mean(0).cpu() - torch.as_tensor(g["es.long.eta.mean"])).abs().max()) < 0.1
    assert abs(float(s["mu"].std()) - float(g["es.long.mu.std"][0])) < 0.5
    d = mc.diagnostics()
    assert float(d["mu"]["r_hat"].max()) < 1.05
    assert kernel.leapfrog_count() > 16 * 1300


@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-10), (torch.float32, 2e-4)])
def test_fused_leaf_kernel_equals_generic_leaf(dtype, tol):
    """b2_nuts_leaf_hier (leapfrog with recomputed local gradients + tree vectors + scalar logic in
    two launches) against the generic leaf built from b2_leapfrog_half_kick_drift, b2_potential_grad,
    b2_leapfrog_half_kick and b2_nuts_leaf_vector, over leaves 0..7 of one subtree from the same
    start: positions, momenta, potential, global gradients, momentum sums, checkpoints, subtree
    weights and U-turn decisions."""
    torch.manual_seed(0)
    C, J = 5, 3000
    D = J + 2
    sig = (5 + 15 * torch.rand(J)).to(DEV, dtype)
    yy = (5 + 3 * torch.randn(J)).to(DEV, dtype) + sig * torch.randn(J).to(DEV, dtype)
    pot = HierNormalPotential(yy, sig, 10.0, 25.0)
    k = NUTS(potential_fn=pot, native_small=False, max_tree_depth=4)
    k.setup(10, C, seed=0)
    assert k._use_fused_hier
    z0 = (0.3 * torch.randn(C, D)).to(DEV, dtype)
    U0, g0 = pot.value_and_grad(z0.clone())
    minv = (0.5 + torch.rand(C, D)).to(DEV, dtype)
    r0 = torch.randn(C, D).to(DEV, dtype)
    eps = (torch.tensor([1e-3, -1e-3, 2e-3, -5e-4, 1e-3])).to(DEV, dtype)
    energy0 = U0 + 0.5 * (minv * r0 * r0).sum(-1)
    u8 = dict(dtype=torch.uint8, device=DEV)
    # chains 0, 2, 4 grow the right end (eps > 0), chains 1, 3 the left end
    dirv = (eps > 0).to(torch.uint8)
    t = {"minv": minv, "energy0": energy0, "zL": z0.clone(), "rL": r0.clone(), "zR": z0.clone(), "rR": r0.clone(),
         "gscL": g0[:, :2].contiguous().clone(), "gscR": g0[:, :2].contiguous().clone(), "dir": dirv,
         "eps": eps, "rsub": torch.full((C, D), 7.0, device=DEV, dtype=dtype),   # stale: leaf 0 must overwrite
         "rck": torch.zeros(5, C, D, device=DEV, dtype=dtype), "sck": torch.zeros(5, C, D, device=DEV, dtype=dtype),
         "sum_accept": torch.zeros(C, device=DEV, dtype=dtype), "num_prop": torch.zeros(C, device=DEV, dtype=dtype),
         "done": torch.zeros(C, **u8), "diverged": torch.zeros(C, **u8), "take": torch.zeros(C, **u8),
         "num_leapfrogs": torch.zeros(C, dtype=torch.int32, device=DEV), "rng_counter": k._rng_counter,
         "gsc_s": torch.zeros(C, 2, device=DEV, dtype=dtype), "U": torch.zeros(C, device=DEV, dtype=dtype),
         "Us": torch.zeros(C, device=DEV, dtype=dtype), "zs": torch.zeros(C, D, device=DEV, dtype=dtype),
         "logw_sub": torch.full((C,), float("-inf"), device=DEV, dtype=dtype)}
    st = {"c": k._lockstep_struct(t), "t": t}
    rm = dirv.bool()[:, None]
    # generic twin
    z, r, g = z0.clone(), r0.clone(), g0.clone()
    rsub = torch.zeros(C, D, device=DEV, dtype=dtype)
    rck, sck = torch.zeros(5, C, D, device=DEV, dtype=dtype), torch.zeros(5, C, D, device=DEV, dtype=dtype)
    zs, gs = z.clone(), g.clone()
    act8 = torch.ones(C, **u8)
    logw = torch.full((C,), float("-inf"), device=DEV, dtype=dtype)
    for leaf in range(8):
        k._leaf_hier(st, leaf)
        z, r, g, U, ke = k._leapfrog(z, r, g, eps, minv, act8)
        take8 = torch.zeros(C, **u8)
        turn = k._leaf_vector(z, r, g, minv, act8, take8, rsub, zs, gs, rck, sck, leaf)
        sc = lambda a: a.abs().max().clamp(min=1.0)  # noqa: E731
        zf, rf = torch.where(rm, t["zR"], t["zL"]), torch.where(rm, t["rR"], t["rL"])
        gf = torch.where(rm, t["gscR"], t["gscL"])
        # the end that does not grow is untouched
        assert torch.equal(torch.where(rm, t["zL"], t["zR"]), z0) and torch.equal(torch.where(rm, t["rL"], t["rR"]), r0)
        assert float((zf - z).abs().max()) <= tol * float(sc(z)), leaf
        assert float((rf - r).abs().max()) <= tol * float(sc(r)) * 10, leaf
        assert torch.allclose(t["U"], U, rtol=tol, atol=tol * float(sc(U))), leaf
        assert torch.allclose(gf, g[:, :2], rtol=50 * tol, atol=50 * tol * float(sc(g[:, :2]))), leaf
        assert float((t["rsub"] - rsub).abs().max()) <= 20 * tol * float(sc(rsub)), leaf
        if leaf % 2 == 0:
            i = bin(leaf >> 1).count("1")
            assert float((t["rck"][i] - rck[i]).abs().max()) <= 20 * tol * float(sc(rck[i])), leaf
            assert float((t["sck"][i] - sck[i]).abs().max()) <= 20 * tol * float(sc(sck[i])), leaf
        w_leaf = -((U + ke) - energy0)
        logw = w_leaf if leaf == 0 else torch.logaddexp(logw, w_leaf)
        assert torch.allclose(t["logw_sub"], logw, rtol=0, atol=200 * tol * float(sc(energy0))), leaf
        # 8 tiny steps from a random momentum: no U-turn, no divergence, in either implementation
        assert not bool(turn.any()) and not bool(t["done"].any()) and not bool(t["diverged"].any()), leaf
    assert int(t["num_leapfrogs"].sum()) == 8 * C
    assert torch.allclose(t["num_prop"], torch.full_like(t["num_prop"], 8.0))
    # root merge: rsum += rsub and the whole-tree U-turn products, against plain torch
    rsum0 = torch.randn(C, D, device=DEV, dtype=dtype)
    t["done"][1] = 1
    rsum = rsum0.clone()
    dots = k._tree_merge(t, rsum)
    sq = minv.sqrt()
    ul, ur = t["rL"] * sq, t["rR"] * sq
    ref_sum = rsum0 + t["rsub"]
    rho = ref_sum - 0.5 * (ul + ur)
    ref = torch.stack([(ul * rho).sum(-1), (ur * rho).sum(-1)], -1)
    live = torch.tensor([0, 2, 3, 4], device=DEV)
    assert torch.allclose(rsum[live], ref_sum[live], rtol=tol, atol=tol)
    assert torch.equal(rsum[1], rsum0[1])
    assert torch.allclose(dots[live], ref[live], rtol=100 * tol, atol=100 * tol * float(ref.abs().max()))
    # masked row copy
    dst = torch.zeros(C, D, device=DEV, dtype=dtype)
    mask = torch.tensor([1, 0, 0, 1, 0], device=DEV, dtype=torch.bool)
    k._rows_copy(dst, z0, mask)
    assert torch.equal(dst[mask], z0[mask]) and float(dst[~mask].abs().max()) == 0.0


def test_fused_leaf_nuts_eight_schools_posterior():
    """BASELINE config 1's model through the lockstep driver on the fused leaf kernel (the path
    config 4 takes at J = 1e6), fp32, 16 chains: posterior moments vs the reference's long run."""
    torch.set_default_dtype(torch.float32)
    g = load_npz("mcmc.npz")
    y, sigma = torch.as_tensor(g["es.y"]).to(DEV, torch.float32), torch.as_tensor(g["es.sigma"]).to(DEV, torch.float32)
    kernel = NUTS(potential_fn=HierNormalPotential(y, sigma, 10.0, 25.0), native_small=False)
    n_s, n_w, C = (500, 200, 16) if not EMULATE else (60, 60, 4)
    mc = MCMC(kernel, num_samples=n_s, warmup_steps=n_w, num_chains=C, seed=0)
    mc.run()
    assert kernel._use_fused_hier
    s = mc.get_samples()
    tol = 1.0 if not EMULATE else 3.0
    assert abs(float(s["mu"].mean()) - float(g["es.long.mu.mean"][0])) < 0.6 * tol
    assert abs(float(s["tau"].mean()) - float(g["es.long.tau.mean"][0])) < 0.8 * tol
    assert float((s["eta"].mean(0).cpu() - torch.as_tensor(g["es.long.eta.mean"])).abs().max()) < 0.15 * tol
    assert kernel.leapfrog_count() > C * (n_s + n_w)


def test_lockstep_nuts_logistic_posterior():
    torch.set_default_dtype(torch.float64)
    g = load_npz("mcmc.npz")
    X, y = torch.as_tensor(g["lr.X"]).to(DEV), torch.as_tensor(g["lr.y"]).to(DEV)
    kernel = NUTS(potential_fn=LogisticPotential(X, y, 1.0), native_small=False)
    mc = MCMC(kernel, num_samples=200, warmup_steps=150, num_chains=8, seed=1)
    mc.run()
    s = mc.get_samples()["beta"].cpu()
    chain = omcmc.NUTSChain(omcmc.logistic_potential(X.cpu(), y.cpu(), 1.0), 3, seed=2)
    ref, _ = chain.run(torch.zeros(3, dtype=torch.float64), 150, 600)
    assert torch.allclose(s.mean(0), ref.mean(0), atol=0.12)
    assert torch.allclose(s.std(0), ref.std(0), atol=0.08)


def test_generic_model_nuts_runs_and_agrees():
    """An unchanged Pyro-style model through TracePotential + lockstep NUTS."""
    torch.set_default_dtype(torch.float64)
    g = load_npz("mcmc.npz")
    X, y = torch.as_tensor(g["lr.X"]).to(DEV), torch.as_tensor(g["lr.y"]).to(DEV)
    mc = MCMC(NUTS(models.logreg_mcmc_model), num_samples=120, warmup_steps=100, num_chains=6, seed=3)
    mc.run(X, y)
    s = mc.get_samples()["beta"].cpu()
    chain = omcmc.NUTSChain(omcmc.logistic_potential(X.cpu(), y.cpu(), 1.0), 3, seed=5)
    ref, _ = chain.run(torch.zeros(3, dtype=torch.float64), 150, 500)
    assert torch.allclose(s.mean(0), ref.mean(0), atol=0.15)


def test_nuts_leaf_vector_kernel_matches_torch_restatement():
    """b2_nuts_leaf_vector (fused per-leaf bookkeeping of the lockstep tree) against the plain
    torch restatement used by the CPU tier, on even (checkpoint store) and odd (U-turn dots) leaves."""
    if EMULATE:
        pytest.skip("needs the device kernel")
    import cpu_emulation
    from pyro_b200.infer.mcmc.nuts import NUTS as K
    torch.manual_seed(0)
    C, D, slots = 5, 1037, 6
    for dtype in (torch.float64, torch.float32):
        mk = lambda *s: torch.randn(*s, device=DEV, dtype=dtype)  # noqa: E731
        z, r, g = mk(C, D), mk(C, D), mk(C, D)
        minv = torch.rand(C, D, device=DEV, dtype=dtype) + 0.5
        active = torch.tensor([1, 0, 1, 1, 1], device=DEV, dtype=torch.uint8)
        take = torch.tensor([1, 1, 0, 1, 0], device=DEV, dtype=torch.uint8)
        state = [mk(C, D), mk(C, D), mk(C, D), mk(slots, C, D), mk(slots, C, D)]
        for leaf in (0, 2, 6, 1, 3, 7, 11):
            a = [t.clone() for t in state]
            b = [t.cpu().clone() for t in state]
            kern = K.__new__(K)
            turn_k = K._leaf_vector(kern, z, r, g, minv, active, take, *a, leaf)
            turn_t = cpu_emulation._leaf_vector(None, z.cpu(), r.cpu(), g.cpu(), minv.cpu(), active.cpu(),
                                                take.cpu(), *b, leaf)
            tol = 1e-12 if dtype == torch.float64 else 1e-5
            for x, y in zip(a, b):
                assert torch.allclose(x.cpu(), y, atol=tol, rtol=tol), leaf
            act = active.bool().cpu()
            assert torch.equal(turn_k.cpu()[act], turn_t[act]), leaf


def test_sparse_gamma_def_meanfield_matches_reference():
    """BASELINE config 5 structure through the CUDA kernels (fused Gamma||Gamma KL, Poisson site,
    fused AdagradRMSProp): the reference's 6-step loss trajectory and final parameters (fp64, 1e-9)."""
    from test_host_logic_cpu import _def_meanfield
    _def_meanfield(DEV)
