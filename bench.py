#!/usr/bin/env python
"""bench.py -- the hot path of BASELINE.json measured on B200.

Workload (config 2 of BASELINE.json, the one the metric is quoted on):
  Bayesian logistic regression, synthetic X[1e6, 32] fp32, 64 vectorised particles, Trace_ELBO,
  ClippedAdam(lr 0.01), through the public API ``SVI.step``.  One "step" = one full SVI step
  (guide sampling, model, fused scoring, backward, fused optimiser, loss read-back).

    python bench.py --gpus N --steps K --warmup W          # our arm  (torchrun for N > 1)
    python bench.py --impl reference ...                   # reference arm: UNMODIFIED Pyro (oracle/_ref) on the host cores

One JSON line on stdout (rank 0).  Keys follow the driver contract; extra keys:
  roofline      dominant kernel of the measured path: algorithmic bytes per launch / its average
                duration (CUDA events on the launching stream) vs MEASURED_PEAKS.json
  cpu_baseline  the oracle port of the reference's CPU path timed on this box's host cores
  variants      the other execution paths of the same workload (generic per-site kernels / fused
                GLM kernel, eager / CUDA-graph) with their own step time and kernel roofline
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
# run from a tree that build() has completed (the build() call below then finds everything current), the
# benchmark writes nothing into it, so that the tree may be read-only: no bytecode caches either
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

N_ROWS, D_FEAT, PARTICLES = 1_000_000, 32, 64
NUTS_W, NUTS_S = 10, 10     # warm-up / sampling transitions of the config-4 section (bounded sample)
METRIC = "svi_steps_per_sec"
UNIT = "steps/s"
WORKLOAD = "bayesian_logistic_regression_svi N=1e6 D=32 Trace_ELBO P=64 ClippedAdam"


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def make_data(device, dtype=torch.float32, n=N_ROWS, seed=0):
    g = torch.Generator().manual_seed(seed)
    X = torch.randn(n, D_FEAT, generator=g, dtype=dtype)
    w_true = torch.randn(D_FEAT, generator=g, dtype=dtype) / D_FEAT ** 0.5
    y = torch.bernoulli(torch.sigmoid(X @ w_true + 0.5), generator=g)
    return X.to(device), y.to(device)


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i] == "Active"})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def bind_near_gpu(index):
    """Pin this process to the CPUs local to GPU ``index`` (sysfs local_cpulist) so that pinned host
    buffers are first-touched on the GPU's NUMA node; a remote node costs host->device bandwidth."""
    try:
        p = torch.cuda.get_device_properties(index)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        with open("/sys/bus/pci/devices/%s/local_cpulist" % bdf) as f:
            text = f.read().strip()
        cpus = set()
        for part in text.split(","):
            if "-" in part:
                lo, hi = part.split("-")
                cpus.update(range(int(lo), int(hi) + 1))
            elif part:
                cpus.add(int(part))
        allowed = os.sched_getaffinity(0)
        use = cpus & allowed
        if use and use != allowed:
            os.sched_setaffinity(0, use)
        return {"gpu": bdf, "local_cpus": len(cpus), "bound_to": len(use) if use else len(allowed)}
    except Exception as e:  # noqa: BLE001 -- diagnostic only
        return {"error": repr(e)[:120]}


def build_svi(path, particles, lr=0.01, sharded=False):
    """Every path runs the SAME, unchanged model (tests/models.py::logistic_model is the reference's
    tests/infer/mcmc/test_hmc.py:189-198 with `w.squeeze(-2) @ X.T + b`).  "glm": latent values reach the
    model as lazy-aware tensors, so the likelihood site is scored by the fused tcgen05 kernel
    (pyro_b200/lazy.py); "site": that mechanism is switched off and the [P, N] logits are materialised
    (cuBLAS) and scored by the per-site kernel."""
    import models
    import pyro_b200 as pyro
    from pyro_b200.infer import SVI, JitTrace_ELBO, Trace_ELBO
    from pyro_b200.infer import elbo as elbo_mod
    from pyro_b200.optim import ClippedAdam
    pyro.clear_param_store()
    elbo_mod.LAZY_LINEAR = "glm" in path
    model = models.logistic_model
    guide = models.logistic_guide
    if sharded:
        model, guide = models.logistic_model_sharded, models.logistic_guide_sharded
    elbo_cls = JitTrace_ELBO if "graph" in path else Trace_ELBO
    return SVI(model, guide, ClippedAdam({"lr": lr}),
               elbo_cls(num_particles=particles, vectorize_particles=True, max_plate_nesting=1))


def particle_weak_section(dev, rank, world, flush, a):
    """SURVEY.md 8(e), the particle axis: every rank scores its OWN 64 particles (different seed) on the full
    data set, loss and gradients averaged by the one packed all-reduce per step -- weak scaling (64 * world
    particles per step at the per-rank work of the 1-GPU line)."""
    import torch.distributed as dist
    import pyro_b200 as pyro
    X, y = make_data(dev)
    torch.manual_seed(1234 + 7919 * rank)
    pyro.set_rng_seed(1234 + 7919 * rank)
    svi = build_svi("glm+graph", PARTICLES, sharded=False)
    steps = max(10, a.steps // 2)
    dist.barrier()
    ms, loss = time_steps(svi, (X, y), steps, 5, dev, flush)
    torch.cuda.synchronize(dev)
    tot = torch.tensor([sum(ms)], device=dev, dtype=torch.float64)
    dist.all_reduce(tot, op=dist.ReduceOp.MAX)
    tot = float(tot)
    del svi, X, y
    torch.cuda.empty_cache()
    return {"ms_per_step": round(tot / steps, 4), "steps_per_sec": round(steps / (tot * 1e-3), 2),
            "global_particles": PARTICLES * world,
            "particle_steps_per_sec": round(PARTICLES * world * steps / (tot * 1e-3), 1),
            "scaling": "weak: %d particles per rank, full data on every rank, 1 all-reduce of [loss, grads] per step"
                       % PARTICLES, "final_loss": round(float(loss), 3)}


def time_steps(svi, args, steps, warmup, device, flush, sync_each=True):
    """Per-step CUDA-event timing on the current stream; the L2 is flushed (256 MB write) between
    steps, outside the timed interval.  The timed call is ``SVI.step_async`` -- the same step, its loss left
    on the device as a 0-d tensor -- and the host does not wait inside the loop, so an interval is the step's
    device time and contains no host round trip (the per-step read-back of the loss is part of `e2e`, not of
    `value`); the last loss is read once at the end.  Returns (list of ms per step, last loss)."""
    step = getattr(svi, "step_async", None) or svi.step
    for _ in range(warmup):
        loss = step(*args)
    torch.cuda.synchronize(device)
    events = []
    for _ in range(steps):
        if flush is not None:
            flush.zero_()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        loss = step(*args)
        e1.record()
        events.append((e0, e1))
    torch.cuda.synchronize(device)
    ms = [e0.elapsed_time(e1) for e0, e1 in events]
    if isinstance(loss, torch.Tensor):
        loss = float(loss)
    return ms, loss


def dump_outputs(out_dir, loss):
    """What a caller of the timed path holds after its last step: the loss it returned and every parameter
    of the store (constrained values), as ``<out_dir>/<name>.npy`` in float32 / float64."""
    import numpy as np
    import pyro_b200 as pyro
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), np.asarray(loss, dtype=np.float64))
    store = pyro.get_param_store()
    for name in sorted(store.keys()):
        t = store[name].detach().cpu()
        np.save(os.path.join(out_dir, "param_%s.npy" % name),
                t.numpy() if t.dtype == torch.float64 else t.float().numpy())


def kernel_time_ms(fn, iters, flush):
    """Average device time of one launch sequence ``fn``: CUDA events on the launching stream
    around a replay of the sequence captured in a CUDA graph (so the Python wrapper cost of the
    call is not inside the interval); L2 flushed between replays, outside the interval."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        fn()
    tot = 0.0
    for _ in range(iters):
        if flush is not None:
            flush.zero_()
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        graph.replay()
        e1.record()
        e1.synchronize()
        tot += e0.elapsed_time(e1)
    return tot / iters


def roofline_for(path, X, y, particles, flush):
    """Dominant kernel of the path, timed alone on its own inputs."""
    import pyro_b200.distributions as dist
    peak, how = peaks()
    dev = X.device
    P, n = particles, X.shape[0]
    if "glm" in path:
        w = (0.1 * torch.randn(P, 1, D_FEAT, device=dev)).requires_grad_(True)
        b = torch.zeros(P, 1, device=dev, requires_grad=True)

        def fn():
            dist.Bernoulli(logits=dist.linear_predictor(X, w, b))._fused_sum(y, None, 1.0, -1.0 / P, 1.0, True)
        ms = kernel_time_ms(fn, 20, flush)
        alg = n * D_FEAT * 4 + n * 4  # X and y once, for value AND gradient (SURVEY 8d)
        name = "glm_bernoulli_tc_kernel + glm_finish_kernel"
    else:
        logits = torch.randn(P, n, device=dev).requires_grad_(True)

        def fn():
            dist.Bernoulli(logits=logits)._fused_sum(y, None, 1.0, -1.0 / P, 1.0, True)
        ms = kernel_time_ms(fn, 20, flush)
        alg = P * n * 4 + n * 4 + P * n * 4  # read logits + y, write d/dlogits (full shape)
        name = "site_vec_kernel<BernoulliLogits,float,GRAD>"
    ach = alg / (ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")  # dram read+write per launch, from ncu --set full
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f).get(name.split(" ")[0].split("<")[0])
    out = {"bound": "hbm", "kernel": name, "achieved": round(ach, 1), "peak": peak, "unit": "GB/s",
           "frac": round(ach / peak, 4), "traffic": traffic, "ms_per_launch": round(ms, 4),
           "algorithmic_bytes": alg, "peak_source": how}
    if "glm" in path:
        # this kernel is not HBM-bound: 3 SFU ops per (row, particle) at 16/clk/SM, and the K = 8 TF32
        # tcgen05 instructions are bound by their shared-memory operand fetch (profiles/glm_tc_r2.md)
        sfu_us = 3.0 * n * P / (148 * 16 * 1.965e9) * 1e6
        out["note"] = ("tcgen05/TMA kernel, shared-memory/tensor-pipe bound (ncu: tensor pipe active 89 %%): "
                       "MUFU floor %.0f us, HBM floor %.0f us, measured %.0f us incl. the finish kernel; "
                       "4*N*D*P = %.1f GFLOP nominal (x2 for the W hi+lo split) = %.0f TFLOP/s nominal"
                       % (sfu_us, alg / peak / 1e3, ms * 1e3, 4.0 * n * D_FEAT * P / 1e9,
                          4.0 * n * D_FEAT * P / (ms * 1e-3) / 1e12))
    return out


class _RefPyroSVI:
    """UNMODIFIED reference Pyro (pyro 1.9.1, copied into oracle/_ref by __graft_entry__.build(),
    plus the stand-in for its absent opt_einsum dependency) running the same
    workload through its own public API on CPU tensors: pyro.infer.SVI / Trace_ELBO(num_particles=64,
    vectorize_particles=True) / pyro.optim.ClippedAdam.  None of this repo's kernels is involved."""

    def __init__(self):
        from pyro_b200 import bind
        if not bind.add_reference_to_path():
            raise RuntimeError("oracle/_ref is missing")
        import pyro
        import pyro.distributions as dist
        from torch.distributions import constraints
        assert os.path.join("oracle", "_ref") in pyro.__file__ and pyro.__version__.startswith("1.9")
        pyro.clear_param_store()

        def model(X, y):
            D = X.shape[-1]
            w = pyro.sample("w", dist.Normal(X.new_zeros(D), X.new_ones(D)).to_event(1))
            b = pyro.sample("b", dist.Normal(X.new_zeros(()), X.new_full((), 10.0)))
            with pyro.plate("data", X.shape[0]):
                logits = w.squeeze(-2) @ X.T + b if w.dim() > 1 else X @ w + b
                pyro.sample("y", dist.Bernoulli(logits=logits), obs=y)

        def guide(X, y):
            D = X.shape[-1]
            w_loc = pyro.param("w_loc", lambda: X.new_zeros(D))
            w_scale = pyro.param("w_scale", lambda: X.new_full((D,), 0.1), constraint=constraints.positive)
            b_loc = pyro.param("b_loc", lambda: X.new_zeros(()))
            b_scale = pyro.param("b_scale", lambda: X.new_full((), 0.1), constraint=constraints.positive)
            pyro.sample("w", dist.Normal(w_loc, w_scale).to_event(1))
            pyro.sample("b", dist.Normal(b_loc, b_scale))

        self.svi = pyro.infer.SVI(model, guide, pyro.optim.ClippedAdam({"lr": 0.01}),
                                  pyro.infer.Trace_ELBO(num_particles=PARTICLES, vectorize_particles=True,
                                                        max_plate_nesting=1))
        self.version = pyro.__version__

    def step(self, X, y):
        return self.svi.step(X, y)


def _ref_pyro_nuts(y, sigma, warmup=100, samples=100):
    """eight_schools through UNMODIFIED reference Pyro (oracle/_ref): pyro.infer.MCMC(pyro.infer.NUTS(model)),
    one chain on the host; leapfrogs counted at pyro.ops.integrator.potential_grad (one call per leapfrog,
    pyro/ops/integrator.py:45-65).  None when the reference is not importable."""
    try:
        from pyro_b200 import bind
        if not bind.add_reference_to_path():
            return None
        import pyro
        import pyro.distributions as dist
        import pyro.ops.integrator as integ
        assert os.path.join("oracle", "_ref") in pyro.__file__
    except Exception:  # noqa: BLE001
        return None

    def model(y, sigma):
        eta = pyro.sample("eta", dist.Normal(torch.zeros(8, dtype=y.dtype), torch.ones(8, dtype=y.dtype)))
        mu = pyro.sample("mu", dist.Normal(torch.zeros(1, dtype=y.dtype), 10 * torch.ones(1, dtype=y.dtype)))
        tau = pyro.sample("tau", dist.HalfCauchy(25 * torch.ones(1, dtype=y.dtype)))
        pyro.sample("obs", dist.Normal(mu + tau * eta, sigma), obs=y)

    calls = [0]
    orig = integ.potential_grad

    def counted(potential_fn, z):
        calls[0] += 1
        return orig(potential_fn, z)

    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    integ.potential_grad = counted
    try:
        pyro.set_rng_seed(0)
        pyro.clear_param_store()
        mcmc = pyro.infer.MCMC(pyro.infer.NUTS(model), num_samples=samples, warmup_steps=warmup,
                               disable_progbar=True)
        t0 = time.perf_counter()
        mcmc.run(y, sigma)
        dt = time.perf_counter() - t0
    except Exception:  # noqa: BLE001
        return None
    finally:
        integ.potential_grad = orig
        torch.set_num_threads(threads)
    return {"leapfrog_per_sec": round(calls[0] / dt, 1), "cores": 1, "kind": "reference",
            "sample": "eight_schools (examples/eight_schools/mcmc.py model), 1 chain, %d warm-up + %d samples, "
                      "pyro %s pyro.infer.MCMC(NUTS(model)) on the host, fp64, %d potential_grad calls in %.1f s"
                      % (warmup, samples, pyro.__version__, calls[0], dt)}


def cpu_reference(steps, warmup, threads=None, n=N_ROWS):
    """The reference's CPU path for this workload, all host threads: unmodified Pyro when it is vendored
    (kind "reference"), else the oracle port (oracle/svi.py, pinned against reference Pyro's own trajectory
    in tests/test_oracle_golden.py; kind "port").  Returns (steps/s, ms/step, threads, loss, kind)."""
    X, y = make_data("cpu", n=n)
    try:
        m = _RefPyroSVI()
        cpu_reference.kind = "reference"
    except Exception as e:  # noqa: BLE001
        from oracle import svi as osvi
        m = osvi.LogisticSVIMatmul(D_FEAT, PARTICLES, lr=0.01)
        cpu_reference.kind = "port (reference Pyro unavailable: %s)" % repr(e)[:80]
    if threads is None:
        # be fair to the reference: torch CPU kernels often run slower with every hardware thread
        # than with a subset, so take the thread count that is fastest on this box
        ncpu = os.cpu_count() or 1
        best = None
        for cand in sorted({ncpu, max(1, ncpu // 2), min(ncpu, 32), min(ncpu, 16)}, reverse=True):
            torch.set_num_threads(cand)
            m.step(X, y)
            t0 = time.perf_counter()
            m.step(X, y)
            dt = time.perf_counter() - t0
            if best is None or dt < best[0]:
                best = (dt, cand)
        threads = best[1]
    torch.set_num_threads(threads)
    for _ in range(warmup):
        m.step(X, y)
    t0 = time.perf_counter()
    for _ in range(steps):
        loss = m.step(X, y)
    dt = time.perf_counter() - t0
    return steps / dt, dt / steps * 1e3, threads, loss


def nuts_section(dev, quick=False):
    """NUTS leapfrog-steps/s (second half of BASELINE.json's metric), reported as extra keys:
    config 1 (eight_schools, 4 chains, 200+200) and the same model with 1024 vectorised chains
    through the whole-transition kernel; config 4's model (hierarchical Normal, J=1e6) through the
    lockstep tree driver with the fused potential; and the oracle's CPU restatement of the
    reference sampler for config 1 as the CPU baseline."""
    import numpy as np
    from oracle import mcmc as omcmc
    from pyro_b200.infer import MCMC, NUTS
    from pyro_b200.infer.mcmc import HierNormalPotential
    out = {}
    y = torch.tensor([28.0, 8.0, -3.0, 7.0, -1.0, 1.0, 18.0, 12.0], device=dev)
    sigma = torch.tensor([15.0, 10.0, 16.0, 11.0, 9.0, 11.0, 10.0, 18.0], device=dev)
    for chains in (4, 1024):
        k = NUTS(potential_fn=HierNormalPotential(y, sigma, 10.0, 25.0))
        mc = MCMC(k, num_samples=200, warmup_steps=200, num_chains=chains, seed=0)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        mc.run()
        e1.record()
        e1.synchronize()
        n = k.leapfrog_count()
        s = mc.get_samples()
        out["eight_schools_%dchains" % chains] = {
            "leapfrogs": n, "seconds": round(e0.elapsed_time(e1) * 1e-3, 4),
            "leapfrog_per_sec": round(n / (e0.elapsed_time(e1) * 1e-3), 1),
            "mu_mean": round(float(s["mu"].mean()), 3), "tau_mean": round(float(s["tau"].mean()), 3),
            "path": "b2_nuts_small: whole transitions on device, 1 thread per chain; warm-up adaptation between launches"}
    # config 4 model at J = 1e6: sampling-phase throughput (warm-up, with its allocations and step-size
    # search, is timed separately)
    # BASELINE config 4 at its stated per-GPU size: 128 chains per GPU, J = 1e6 groups, max_tree_depth 10,
    # save_params = [mu, tau]; the MODEL is handed over unchanged (tests/models.py::eight_schools) and is
    # recognised as the hierarchical-Normal class (pyro_b200/infer/mcmc/compile.py).  The 200 + 200
    # transitions of the config are bounded to W + S here so that the default bench stays within minutes.
    import models
    J, C = 1_000_000, (8 if quick else 128)
    g = torch.Generator().manual_seed(0)
    sig = (5 + 15 * torch.rand(J, generator=g)).to(dev)
    yy = (5 + 3 * torch.randn(J, generator=g)).to(dev) + sig * torch.randn(J, generator=g).to(dev)
    k = NUTS(models.eight_schools, max_tree_depth=10)
    W, S = NUTS_W, NUTS_S
    marks = {}

    def hook(kernel, z, stage, t):
        if stage == "Warmup" and t == W - 1:
            torch.cuda.synchronize(dev)
            marks["t"], marks["n"] = time.perf_counter(), kernel.leapfrog_count()

    # config 4 keeps only mu and tau; every site's running mean / variance is streamed on the device
    mc = MCMC(k, num_samples=S, warmup_steps=W, num_chains=C, seed=0, hook_fn=hook, save_params=["mu", "tau"])
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    mc.run(sig, yy)
    torch.cuda.synchronize(dev)
    assert type(k.potential).__name__ == "HierNormalPotential", "model class not recognised"
    t1 = time.perf_counter()
    n = k.leapfrog_count()
    ns, ts = n - marks["n"], t1 - marks["t"]
    out["hier_normal_J1e6_%dchains" % C] = {
        "leapfrogs": ns, "seconds": round(ts, 3), "leapfrog_per_sec": round(ns / ts, 1),
        "algorithmic_GBps": round(ns * 16e6 / ts / 1e9, 1),
        "frac_of_16B_roofline": round(ns * 16e6 / ts / 1e9 / peaks()[0], 3),
        "incl_warmup": {"leapfrogs": n, "seconds": round(t1 - t0, 3), "leapfrog_per_sec": round(n / (t1 - t0), 1)},
        "path": "lockstep iterative tree, every leaf = b2_nuts_leaf_hier (fused leapfrog with recomputed local "
                "gradients + tree vectors + scalar logic, 2 launches, ~40 B moved per chain-element); root merge "
                "and proposal hand-over = b2_nuts_tree_merge / b2_rows_copy_masked; save_params=[mu, tau] + streamed "
                "per-chain mean/variance of every site; NUTS(model=eight_schools) recognised as the native class; "
                "%d chains, max_tree_depth 10, %d sampling transitions timed after %d warm-up "
                "(config 4 asks for 200 + 200: bounded sample)" % (C, S, W)}
    # CPU baseline: unmodified reference Pyro (config 1, one chain), else the oracle restatement of its sampler
    ref = _ref_pyro_nuts(y.double().cpu(), sigma.double().cpu())
    if ref is not None:
        out["cpu_baseline"] = ref
        return out
    torch.set_num_threads(1)
    U = omcmc.eight_schools_potential(y.double().cpu(), sigma.double().cpu())
    chain = omcmc.NUTSChain(U, 10, seed=0)
    t0 = time.perf_counter()
    chain.run(torch.zeros(10, dtype=torch.float64), 100, 100)
    dt = time.perf_counter() - t0
    out["cpu_baseline"] = {"leapfrog_per_sec": round(chain.num_leapfrogs / dt, 1), "cores": 1, "kind": "port",
                           "sample": "eight_schools, 1 chain, 100 warm-up + 100 samples, oracle/mcmc.py NUTSChain "
                                     "(reference Pyro itself measured 522-541 leapfrog/s in the build container, "
                                     "tests/golden/make_golden.py)"}
    torch.set_num_threads(os.cpu_count())
    return out


def nuts_multirank(dev, rank, world):
    """Chain-sharded NUTS at N > 1 (SURVEY.md 8(e): rank r owns chains [r*C/W, (r+1)*C/W), no
    collective during warm-up or sampling).  Times are CUDA-event times, max over ranks; leapfrog
    counts are summed over ranks."""
    import torch.distributed as dist
    from pyro_b200.infer import MCMC, NUTS
    from pyro_b200.infer.mcmc import HierNormalPotential
    out = {}
    y = torch.tensor([28.0, 8.0, -3.0, 7.0, -1.0, 1.0, 18.0, 12.0], device=dev)
    sigma = torch.tensor([15.0, 10.0, 16.0, 11.0, 9.0, 11.0, 10.0, 18.0], device=dev)

    def timed(label, make, note):
        k, mc = make()
        dist.barrier()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        mc.run()
        e1.record()
        e1.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) * 1e-3], device=dev, dtype=torch.float64)
        n = torch.tensor([float(k.leapfrog_count())], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(n, op=dist.ReduceOp.SUM)
        out[label] = {"leapfrogs": int(n), "seconds": round(float(t), 4),
                      "leapfrog_per_sec": round(float(n) / float(t), 1), "scaling": note}

    for total, note in ((1024, "strong: 1024 chains total, %d per rank" % (1024 // world)),
                        (1024 * world, "weak: 1024 chains per rank")):
        def make(total=total):
            k = NUTS(potential_fn=HierNormalPotential(y, sigma, 10.0, 25.0))
            return k, MCMC(k, num_samples=200, warmup_steps=200, num_chains=total, seed=0)
        timed("eight_schools_%dchains" % total, make, note)
    J, C = 1_000_000, 128
    g = torch.Generator().manual_seed(0)
    sig = (5 + 15 * torch.rand(J, generator=g)).to(dev)
    yy = (5 + 3 * torch.randn(J, generator=g)).to(dev) + sig * torch.randn(J, generator=g).to(dev)

    def make4():
        k = NUTS(potential_fn=HierNormalPotential(yy, sig, 10.0, 25.0), native_small=False, max_tree_depth=10)
        return k, MCMC(k, num_samples=NUTS_S, warmup_steps=NUTS_W, num_chains=C * world, seed=0,
                       save_params=["mu", "tau"])
    timed("hier_normal_J1e6_%dchains" % (C * world), make4,
          "weak: %d chains per rank (config 4: 1024 over 8 GPUs), %d + %d transitions, max_tree_depth 10"
          % (C, NUTS_W, NUTS_S))
    out["hier_normal_J1e6_%dchains" % (C * world)]["algorithmic_GBps"] = round(
        out["hier_normal_J1e6_%dchains" % (C * world)]["leapfrog_per_sec"] * 16e6 / 1e9, 1)
    return out


def config3_section(dev):
    """BASELINE config 3: GaussianHMM SVI step, H = 512, O = 4, T = 10 000, one B200 (structure of
    profiler/gaussianhmm.py:12-56): learnable parameters for the five parts, empty guide, Trace_ELBO,
    ClippedAdam.  The contraction runs on library GEMMs (cuBLAS / cuSOLVER through torch) -- see DESIGN.md."""
    from torch.distributions import constraints
    import pyro_b200 as pyro
    import pyro_b200.distributions as dist
    from pyro_b200.infer import SVI, Trace_ELBO
    from pyro_b200.optim import ClippedAdam
    T, H, O = 10000, 512, 4
    gen = torch.Generator().manual_seed(0)
    data = torch.randn(T, O, generator=gen).to(dev)
    F0 = (0.5 * torch.randn(H, H, generator=gen) / H ** 0.5).to(dev)
    H0 = torch.randn(H, O, generator=gen).to(dev)
    t0s = (torch.randn(H, generator=gen) * 0.1).exp().to(dev)
    o0s = (torch.randn(O, generator=gen) * 0.1).exp().to(dev)

    def model(x):
        F = pyro.param("trans_matrix", lambda: F0.clone())
        Hm = pyro.param("obs_matrix", lambda: H0.clone())
        tsc = pyro.param("trans_scale", lambda: t0s.clone(), constraint=constraints.positive)
        osc = pyro.param("obs_scale", lambda: o0s.clone(), constraint=constraints.positive)
        isc = pyro.param("init_scale", lambda: torch.ones(H, device=dev), constraint=constraints.positive)
        z = torch.zeros(H, device=dev)
        hmm = dist.GaussianHMM(dist.Normal(z, isc).to_event(1), F, dist.Normal(z, tsc).to_event(1), Hm,
                               dist.Normal(torch.zeros(O, device=dev), osc).to_event(1), duration=x.shape[0])
        pyro.sample("obs", hmm, obs=x)

    pyro.clear_param_store()
    svi = SVI(model, lambda x: None, ClippedAdam({"lr": 1e-3}), Trace_ELBO())
    for _ in range(2):
        loss = svi.step(data)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        loss = svi.step(data)
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1) / 5
    pyro.clear_param_store()
    general_flops = (T - 1) * (H ** 3 / 3 + 2 * H ** 3 + 8 * H ** 3)     # SURVEY.md 8d, forward
    return {"workload": "GaussianHMM SVI step H=512 O=4 T=10000 fp32 (BASELINE config 3)",
            "ms_per_step": round(ms, 2), "steps_per_sec": round(1e3 / ms, 2), "loss": round(float(loss), 2),
            "path": "innovation-form Kalman recursion; time-invariant parameters: covariance steps until "
                    "convergence, then a blocked linear scan of the means; GEMMs / Choleskys are LIBRARY calls "
                    "(cuBLAS, cuSOLVER via torch), not hand-written kernels",
            "flops_general_formulation_fwd": general_flops,
            "note": "the H^3 FLOPs of the covariance steps skipped after convergence are neither performed nor "
                    "counted as achieved; no tensor-pipe figure is claimed for this row"}


def config5_section(dev, rank, world):
    """BASELINE config 5: sparse-gamma DEF (examples/sparse_gamma_def.py:43-165), x [320, 4096] synthetic
    Poisson counts, widths 100/40/15, TraceMeanField_ELBO with 256 vectorised particles, AdagradRMSProp;
    particles are sharded over the ranks (256 / world each, different seeds), loss + gradients averaged by
    the ONE all-reduce of SVI._allreduce."""
    import models
    import pyro_b200 as pyro
    from pyro_b200.infer import SVI, TraceMeanField_ELBO
    from pyro_b200.optim import AdagradRMSProp
    N, PX, P = 320, 4096, 256 // world
    gen = torch.Generator().manual_seed(0)
    rate = torch.distributions.Gamma(0.5, 0.5).sample((N, PX)) * 2.0
    x = torch.poisson(rate, generator=gen).to(dev)
    torch.manual_seed(100 + rank)
    pyro.clear_param_store()
    m = models.SparseGammaDEF(PX, (100, 40, 15), device=dev, dtype=torch.float32)
    elbo = TraceMeanField_ELBO(num_particles=P, vectorize_particles=True, max_plate_nesting=1)
    elbo.capture_graph = True
    svi = SVI(m.model, m.guide, AdagradRMSProp({"eta": 4.5, "t": 0.1}), elbo)
    for _ in range(4):
        loss = svi.step(x)
    torch.cuda.synchronize(dev)
    steps = 20
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = svi.step(x)
    e1.record()
    e1.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / steps], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t)
    pyro.clear_param_store()
    return {"workload": "sparse_gamma_def N=320x4096 widths 100/40/15 TraceMeanField_ELBO P=256 (BASELINE config 5)",
            "particles_per_rank": P, "ms_per_step": round(ms, 3), "steps_per_sec": round(1e3 / ms, 2),
            "poisson_terms_per_sec": round(256 * N * PX / (ms * 1e-3), 1), "loss": round(float(loss), 1),
            "scaling": "strong: 256 particles total, %d per rank" % P}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--path", default="glm+graph",
                    help="ours: site | site+graph | glm | glm+graph (default)")
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--cpu-steps", type=int, default=4)
    ap.add_argument("--no-nuts", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the config 3 / config 5 sections")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the loss and parameters of the last step as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    a.warmup = max(a.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if a.impl == "reference":
        if rank != 0:
            return
        steps = a.steps
        v, ms, threads, loss = cpu_reference(steps, min(a.warmup, 2))
        kind = cpu_reference.kind
        what = ("pyro.infer.SVI.step of unmodified Pyro (oracle/_ref)" if kind == "reference"
                else "oracle/svi.py LogisticSVIMatmul")
        out = {"impl": "reference", "metric": METRIC, "value": round(v, 4), "unit": UNIT, "n_gpus": a.gpus,
               "steps": steps, "warmup": min(a.warmup, 2), "ms_per_step": round(ms, 3),
               "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
               "data": "synthetic", "config": {"workload": WORKLOAD, "global_particles": PARTICLES},
               "cpu_baseline": {"value": round(v, 4), "unit": UNIT, "cores": threads, "kind": kind,
                                "sample": "%d full-size steps (N=1e6, P=64) of %s" % (steps, what)},
               "e2e": {"value": round(v, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(out))
        return

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        import torch.distributed as dist
        # keep stdout for the ONE JSON line: NCCL's version / debug banner goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    from pyro_b200 import _native
    import __graft_entry__
    if rank == 0:
        __graft_entry__.build()
    if world > 1:
        dist.barrier()
    _native.lib()
    # every rank draws the SAME guide samples (same seed): the data plate, not the particle plate,
    # is sharded, so ranks differ only in the rows they score
    torch.manual_seed(1234)
    P_local = PARTICLES
    X, y = make_data(dev)
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)  # 256 MB > 126 MB L2
    path = a.path
    sharded = world > 1
    step_args = (X, y)
    if sharded:
        lo, hi = rank * N_ROWS // world, (rank + 1) * N_ROWS // world
        X, y = X[lo:hi].contiguous(), y[lo:hi].contiguous()
        step_args = (X, y, torch.arange(lo, hi, device=dev), N_ROWS)

    # launches per step, counted on an eager twin of the path (a graph replay re-issues exactly the
    # launches captured from one eager step)
    probe = build_svi(path.replace("+graph", ""), P_local, sharded=sharded)
    probe.step(*step_args)
    n0 = _native.launch_count()
    probe.step(*step_args)
    per_step_launches = _native.launch_count() - n0
    del probe
    svi = build_svi(path, P_local, sharded=sharded)

    sampler = ClockSampler(local_rank)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    if rank == 0:
        sampler.start()
        time.sleep(0.15)
    ms, loss = time_steps(svi, step_args, a.steps, a.warmup + 2, dev, flush)
    torch.cuda.synchronize(dev)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, loss)
    if world > 1:
        dist.barrier()
    total_ms = torch.tensor([sum(ms)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms)
    value = a.steps / (total_ms * 1e-3)

    # ---- e2e: host (pinned) inputs copied every step through the same public call --------------------
    # Every step's X and y travel host -> device inside the timed region (K copies for K steps) and
    # the loss comes back to the host every step.  The copy of step k+1 is issued on a second stream
    # before step k's loss is read, so the transfer overlaps the previous step's kernels (what a
    # prefetching data loader does); the step itself is the unmodified public SVI.step call.
    torch.ones(1 << 22).sum()            # intra-op thread pool exists (full affinity) before binding
    all_cpus = os.sched_getaffinity(0)
    numa = bind_near_gpu(local_rank)     # pinned pages are first-touched on the GPU's NUMA node ...
    Xh = torch.empty(X.shape, dtype=X.dtype).pin_memory()
    yh = torch.empty(y.shape, dtype=y.dtype).pin_memory()
    Xh.copy_(X)
    yh.copy_(y)
    os.sched_setaffinity(0, all_cpus)    # ... and the CPU baseline below gets every core back
    copy_stream = torch.cuda.Stream(dev)
    bufs = [(torch.empty_like(X), torch.empty_like(y)) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]

    def prefetch(k):
        b = k % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[b])
            bufs[b][0].copy_(Xh, non_blocking=True)
            bufs[b][1].copy_(yh, non_blocking=True)
            ready[b].record(copy_stream)

    def e2e_run(n):
        for ev in consumed:
            ev.record()
        prefetch(0)
        for k in range(n):
            b = k % 2
            torch.cuda.current_stream(dev).wait_event(ready[b])
            if k + 1 < n:
                prefetch(k + 1)
            svi.step(bufs[b][0], bufs[b][1], *step_args[2:])
            consumed[b].record()

    e2e_run(3)
    torch.cuda.synchronize(dev)
    # pure transfer rate of this box (diagnostic: the e2e number is PCIe-bound)
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for _ in range(4):
        bufs[0][0].copy_(Xh, non_blocking=True)
        bufs[0][1].copy_(yh, non_blocking=True)
    c1.record()
    c1.synchronize()
    h2d = Xh.numel() * 4 + yh.numel() * 4
    h2d_gbps = 4 * h2d / (c0.elapsed_time(c1) * 1e-3) / 1e9
    e2e_n = max(5, min(a.steps, 20))
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    e2e_run(e2e_n)
    e1.record()
    e1.synchronize()
    e2e_ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_val = e2e_n / (float(e2e_ms) * 1e-3)
    clocks = sampler.stop() if rank == 0 else None
    weak = None
    if world > 1 and not a.no_variants:
        try:
            weak = particle_weak_section(dev, rank, world, flush, a)
        except Exception as e:  # pragma: no cover
            weak = {"error": repr(e)[:300]}
    nuts_mr = None
    if world > 1 and not a.no_nuts:
        try:
            nuts_mr = nuts_multirank(dev, rank, world)
        except Exception as e:  # pragma: no cover
            nuts_mr = {"error": repr(e)[:300]}

    cfg5 = None
    if not a.no_configs:
        try:
            cfg5 = config5_section(dev, rank, world)
        except Exception as e:  # pragma: no cover
            cfg5 = {"error": repr(e)[:300]}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    out = {"metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": a.steps,
           "warmup": a.warmup + 2, "ms_per_step": round(total_ms / a.steps, 4), "higher_is_better": True,
           "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": WORKLOAD, "global_particles": PARTICLES,
                      "model": "tests/models.py::logistic_model -- the reference model unchanged "
                               "(w.squeeze(-2) @ X.T + b -> Bernoulli(logits)); no repo-specific API in the model",
                      "precision": "fp32 storage and accumulation; the two contractions run on tcgen05 tensor cores "
                                   "with TF32 operands, W split hi+lo (removes the row-coherent rounding error): "
                                   "sum / dW / db within 2e-5 / 2e-4 of fp64 (tests/test_gpu_tier2.py, N=1e6)",
                      "parallelism": ("data plate (rows) sharded over %d ranks, same particles on every rank, "
                                      "1 all-reduce of [loss, grads] (67 floats) per step between two "
                                      "CUDA graphs" % world) if world > 1 else "single GPU",
                      "path": path, "l2": "256 MB flush write between timed steps (outside the timed interval); "
                                          "inputs 132 MB > 126 MB L2",
                      "timing": "per-step CUDA events on the launching stream around SVI.step_async (loss stays on the device; "
                                "no host wait inside the loop), summed; max over ranks"},
           "final_loss": round(float(loss), 3),
           "e2e": {"value": round(e2e_val, 2), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                   "h2d_GBps_this_box": round(h2d_gbps, 1), "numa": numa,
                   "note": "SVI.step on pinned host X,y: every step's inputs are copied host->device inside the "
                           "timed region (double-buffered on a copy stream so the transfer of step k+1 overlaps "
                           "step k), loss read back every step; PCIe-bound"},
           "gpu_launches": int(per_step_launches * a.steps), "gpu_launches_per_step": int(per_step_launches),
           "clocks": clocks}
    if world == 1:
        out["roofline"] = roofline_for(path, X, y, P_local, flush)
        if not a.no_variants:
            variants = {}
            for vp in ("site", "site+graph", "glm", "glm+graph"):
                if vp == path:
                    continue
                try:
                    s2 = build_svi(vp, P_local)
                    vms, _ = time_steps(s2, (X, y), max(10, a.steps // 3), 5, dev, flush)
                    variants[vp] = {"ms_per_step": round(sum(vms) / len(vms), 4),
                                    "steps_per_sec": round(len(vms) / (sum(vms) * 1e-3), 2)}
                except Exception as e:  # pragma: no cover
                    variants[vp] = {"error": repr(e)[:200]}
            for vp in ("site", "glm"):
                if vp in variants and "error" not in variants[vp]:
                    variants[vp]["roofline"] = roofline_for(vp, X, y, P_local, flush)
            # the per-family fused log_prob table (SURVEY.md 8d "micro log_prob"): HBM GB/s on the
            # algorithmic bytes vs the measured copy peak, re-measured by the driver every round
            try:
                sys.path.insert(0, os.path.join(ROOT, "profiles"))
                import micro_logprob
                variants["micro"] = micro_logprob.run(verbose=False)
                torch.cuda.empty_cache()
            except Exception as e:  # pragma: no cover
                variants["micro"] = {"error": repr(e)[:200]}
            out["variants"] = variants
        v, cms, threads, _ = cpu_reference(a.cpu_steps, 1)
        out["cpu_baseline"] = {"value": round(v, 4), "unit": UNIT, "cores": threads, "kind": cpu_reference.kind,
                               "sample": "%d full-size steps (N=1e6, P=64) of %s, torch CPU ops, the fastest of "
                                         "several host thread counts" % (
                                             a.cpu_steps, "pyro.infer.SVI.step of unmodified Pyro (oracle/_ref)"
                                             if cpu_reference.kind == "reference" else "oracle/svi.py LogisticSVIMatmul"),
                               "ms_per_step": round(cms, 2)}
        if not a.no_nuts:
            try:
                out["nuts"] = nuts_section(dev)
            except Exception as e:  # pragma: no cover
                out["nuts"] = {"error": repr(e)[:300]}
    if weak is not None:
        out["variants"] = {"particle_sharded_weak": weak}
    if nuts_mr is not None:
        out["nuts"] = nuts_mr
    if not a.no_configs:
        out["configs"] = {"config5": cfg5}
        if world == 1:
            try:
                out["configs"]["config3"] = config3_section(dev)
            except Exception as e:  # pragma: no cover
                out["configs"]["config3"] = {"error": repr(e)[:300]}
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
