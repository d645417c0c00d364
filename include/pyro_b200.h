/*
 * pyro_b200.h -- C ABI of the B200-native numerics library behind Pyro's two hot paths
 * (Trace_ELBO SVI step, NUTS/HMC leapfrog).
 *
 * Every entry point replaces one piece of arithmetic that reference Pyro (pyro-ppl/pyro 1.9.1)
 * executes as a chain of ATen launches.  The reference-side binding is a ctypes stub
 * (see INTEGRATION.md); there are no torch types in any signature.
 *
 * Conventions
 *   - All data pointers are DEVICE pointers owned by the caller.  The library never allocates,
 *     frees or retains them beyond the call.  `stream` is a cudaStream_t passed as void*.
 *   - Every function returns B2_OK (0) or a negative B2_ERR_* code; nothing throws or aborts.
 *     Numerical failures are data (NaN / -inf in outputs), exactly like the reference, where a
 *     NaN energy means "reject" (pyro/infer/mcmc/nuts.py:209-214).
 *   - Functions are re-entrant and stream ordered, do not synchronise, and are CUDA-graph
 *     capturable.  Reductions use a fixed order (no floating-point atomics): results are
 *     bit-stable from run to run for a given shape.
 *   - Tensors are described by b2_tensor: a common broadcast shape and per-operand element
 *     strides (0 = broadcast along that dim), so Pyro's ExpandedDistribution / MaskedDistribution /
 *     Independent views (pyro/distributions/torch_distribution.py:163-232,302-374,399-488)
 *     never need a copy.
 */
#ifndef PYRO_B200_H_
#define PYRO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2_MAX_DIMS 8

/* ---- error codes ------------------------------------------------------------------------ */
#define B2_OK 0
#define B2_ERR_BAD_DTYPE (-1)
#define B2_ERR_BAD_SHAPE (-2)
#define B2_ERR_BAD_FAMILY (-3)
#define B2_ERR_NULL (-4)
#define B2_ERR_WORKSPACE (-5)
#define B2_ERR_UNSUPPORTED_REDUCTION (-6) /* gradient output broadcast pattern not fused; caller
                                             asks for a full-shape gradient and reduces it */
#define B2_ERR_LAUNCH (-7)                /* cudaGetLastError() != cudaSuccess after launch */
#define B2_ERR_TOO_LARGE (-8)
#define B2_ERR_NO_DEVICE (-9)

/* ---- dtypes ------------------------------------------------------------------------------ */
#define B2_F32 0
#define B2_F64 1
#define B2_I64 2
#define B2_U8 3 /* torch.bool / uint8 masks */

/* ---- distribution families ---------------------------------------------------------------
 * Elementwise families (event_dim 0).  Parameter order is fixed, as listed.
 * Formulas restate torch.distributions (the third-party arithmetic the reference delegates to,
 * pyro/distributions/torch.py:23-257), see SURVEY.md Appendix A. */
#define B2_NORMAL 0            /* (loc, scale)            torch/distributions/normal.py:87-102    */
#define B2_BERNOULLI_LOGITS 1  /* (logits)                torch/distributions/bernoulli.py:121-125 */
#define B2_GAMMA 2             /* (concentration, rate)   torch/distributions/gamma.py:89-98      */
#define B2_BETA 3              /* (concentration1, concentration0)  beta.py:87-91                 */
#define B2_POISSON 4           /* (rate)                  torch/distributions/poisson.py:75-79    */
#define B2_CAUCHY 5            /* (loc, scale)            torch/distributions/cauchy.py:81-88     */
#define B2_HALFCAUCHY 6        /* (scale)                 torch/distributions/half_cauchy.py:73-81 */
#define B2_EXPONENTIAL 7       /* (rate)                  torch/distributions/exponential.py      */
#define B2_LOGNORMAL 8         /* (loc, scale)            log_normal.py (Normal o Exp transform)  */
#define B2_HALFNORMAL 9        /* (scale)                 torch/distributions/half_normal.py      */
#define B2_BERNOULLI_PROBS 10  /* (probs)                 bernoulli.py (probs parametrisation)    */
#define B2_UNIFORM 11          /* (low, high)             torch/distributions/uniform.py          */
#define B2_KL_NORMAL_NORMAL 12 /* value unused; (loc_p, scale_p, loc_q, scale_q) kl.py:468-471    */
#define B2_KL_GAMMA_GAMMA 13   /* value unused; (conc_p, rate_p, conc_q, rate_q) kl.py:301-306    */
/* Reparameterised Normal draw fused with its own score (SURVEY.md 8(f) row 1; replaces
 * rsample torch/distributions/normal.py:82-85 + the guide site's log_prob + its backward).
 * Both are launched with scale = weight = 1.
 *   B2_NORMAL_RSAMPLE:      value = eps ~ N(0,1), params (loc, scale);
 *                           out_dvalue (full shape) receives z = loc + eps*scale,
 *                           out_sum receives sum_coeff * SUM Normal(loc, scale).log_prob(z)
 *   B2_NORMAL_RSAMPLE_BWD:  value = dL/dz, params (eps, scale, c);
 *                           out_dparams[0] = dL/dloc   = SUM dL/dz
 *                           out_dparams[1] = dL/dscale = SUM (dL/dz * eps - c/scale)
 *                           (c = coefficient of SUM log q(z) in L; both reduced to the stored
 *                           shapes of loc / scale)                                              */
#define B2_NORMAL_RSAMPLE 14
#define B2_NORMAL_RSAMPLE_BWD 15
#define B2_NUM_ELEMENTWISE_FAMILIES 16
/* Event families (event_dim >= 1), scored by b2_event_score. */
#define B2_DIRICHLET 32   /* (concentration[...,K])           torch/distributions/dirichlet.py:90-97 */
#define B2_CATEGORICAL 33 /* (logits[...,K]), int64 value      categorical.py:78,151-157             */
#define B2_MVN_TRIL 34    /* (loc[...,n], scale_tril[...,n,n]) multivariate_normal.py:256-264        */

#define B2_MAX_PARAMS 4
#define B2_SITE_SMALL_N 8192 /* sites up to this many elements: single-CTA kernel, fused reductions */

typedef struct {
  void* ptr;
  int32_t dtype;
  int32_t ndim;
  int64_t shape[B2_MAX_DIMS];
  int64_t stride[B2_MAX_DIMS]; /* in elements; 0 = broadcast */
} b2_tensor;

/* flags for b2_site_score */
#define B2_FLAG_ACCUMULATE_SUM 1 /* out_sum += coeff*sum instead of out_sum = coeff*sum */
#define B2_FLAG_SITE_LARGE 4     /* b2_site_score: take the multi-CTA kernels even for a site of at
                                    most B2_SITE_SMALL_N elements (tests cover both paths on the
                                    reference's small fixtures) */
#define B2_FLAG_GLM_FP32 2       /* b2_glm_bernoulli_logits: fp32 SIMT contractions instead of the
                                    tensor-core path */
#define B2_FLAG_GLM_3XTF32 32    /* b2_glm_bernoulli_logits: split X as well as W (every logit exact to
                                    ~1e-6; the default splits W only, see below) */
/* bits 8, 16 and 64 are retired (they selected removed GLM kernel variants); b2_glm_bernoulli_logits
   rejects them with B2_ERR_BAD_SHAPE */

/*
 * b2_site_score -- fused log_prob + score of one sample site for an elementwise family.
 *
 * Replaces, in one pass over the operands:
 *   site["fn"].log_prob(value)                      pyro/poutine/trace_struct.py:225,264,304
 *   scale_and_mask(log_p, scale, mask)              pyro/distributions/util.py:311-328
 *   log_p.sum()                                     pyro/poutine/trace_struct.py:240,278
 *   and the autograd backward of those ATen chains  (pyro/infer/trace_elbo.py:153-157)
 *
 * All tensors are expressed on ONE common broadcast shape (value->shape); params[i], mask,
 * upstream and the outputs carry their own strides (0 where broadcast).
 *
 *   lp_i      = family log density at element i
 *   m_i       = mask ? mask_i : 1
 *   out_logprob_i = m_i ? scale*lp_i : 0            (if out_logprob != NULL)
 *   out_sum   (=|+=) sum_coeff * SUM_i m_i*scale*lp_i  (if out_sum != NULL; dtype of value)
 *   u_i       = upstream ? upstream_i : 1
 *   grad of operand o at i:  weight * u_i * m_i * scale * d lp_i / d o
 * Gradient outputs (out_dvalue, out_dparams[k]; ptr may be NULL = not wanted) are written to a
 * tensor that is either full shape (no zero stride on a dim of size > 1) or a scalar (all strides
 * zero: the gradient is summed over every element).  A mixed pattern (zero stride on some dims:
 * the operand's stored shape, e.g. loc[D] scored against value[P, D]) is reduced in the same
 * launch for sites of at most B2_SITE_SMALL_N elements -- those run as ONE CTA, one launch --
 * and returns B2_ERR_UNSUPPORTED_REDUCTION without launching for larger ones (the caller then
 * asks for a full-shape gradient and sums it with b2_reduce_to).
 *
 * workspace: b2_site_score_workspace() bytes, zero-initialised ONCE by the caller; the library
 * leaves it zeroed.  Must not be shared by kernels running concurrently on different streams.
 */
int b2_site_score(int family, const b2_tensor* value, const b2_tensor* params, int n_params,
                  const b2_tensor* mask, double scale, const b2_tensor* upstream, double weight,
                  double sum_coeff, int flags, b2_tensor* out_logprob, void* out_sum,
                  b2_tensor* out_dvalue, b2_tensor* out_dparams, void* workspace,
                  size_t workspace_bytes, void* stream);

size_t b2_site_score_workspace(void);

/*
 * b2_event_score -- fused log_prob (+ gradients) for families with an event dimension.
 * `batch` describes the common batch shape; the event dims are the trailing dims of each
 * operand and must be contiguous.
 *   DIRICHLET:   params[0]=concentration[batch,K], value[batch,K]
 *   CATEGORICAL: params[0]=logits[batch,K] (un-normalised; normalised inside exactly like the
 *                constructor's logits - logsumexp), value int64 [batch]
 *   MVN_TRIL:    params[0]=loc[batch,n], params[1]=scale_tril[batch,n,n], value[batch,n]
 * out_logprob is [batch] (scaled/masked like b2_site_score); gradients, when requested, are full
 * shape [batch, event...] or, for a batch-broadcast operand (all batch strides zero), reduced
 * over the batch.
 */
int b2_event_score(int family, const b2_tensor* value, const b2_tensor* params, int n_params,
                   int event_size, const b2_tensor* mask, double scale, const b2_tensor* upstream,
                   double weight, double sum_coeff, int flags, b2_tensor* out_logprob,
                   void* out_sum, b2_tensor* out_dvalue, b2_tensor* out_dparams, void* workspace,
                   size_t workspace_bytes, void* stream);

/*
 * b2_normal_rsample -- reparameterised Normal draw with the noise generated in the kernel (Philox4x32-10),
 * fused with the site's own log density: z = loc + eps*scale, eps ~ N(0,1), *out_sum = SUM log Normal(z).
 * Replaces torch.randn + addcmul (torch/distributions/normal.py:82-85) and the guide site's
 * log_prob + sum (pyro/poutine/trace_struct.py:264-278) -- SURVEY.md 8(f) row 1.
 * loc, scale: broadcast views over `shape` (element strides, 0 = broadcast); z, eps: contiguous outputs
 * of prod(shape) <= B2_RSAMPLE_MAX_N elements (one CTA); out_sum: 0-d, same dtype.
 * rng_state: device array of two uint64 {seed, launch counter}; the kernel increments the counter, so a
 * replayed CUDA graph draws fresh noise with no host-side RNG bookkeeping.
 */
#define B2_RSAMPLE_MAX_N 65536
int b2_normal_rsample(const b2_tensor* loc, const b2_tensor* scale, int ndim, const int64_t* shape, void* z,
                      void* eps, void* out_sum, void* rng_state, void* stream);

/*
 * b2_gamma_rsample -- reparameterised Gamma(concentration, rate) draws (Marsaglia-Tsang on the in-kernel Philox
 * stream) together with d z / d concentration by implicit reparameterisation: replaces _standard_gamma +
 * division + clamp (torch/distributions/gamma.py:79-87) and the ATen backward _standard_gamma_grad --
 * SURVEY.md 8(f) row 1.  conc, rate: broadcast views over `shape`; z, dz_dconc (nullable): contiguous outputs
 * of prod(shape) elements; rng_state as for b2_normal_rsample.  d z / d rate = -z / rate is left to the caller.
 */
int b2_gamma_rsample(const b2_tensor* conc, const b2_tensor* rate, int ndim, const int64_t* shape, void* z,
                     void* dz_dconc, void* rng_state, void* stream);

/*
 * The "latent sites" block of an SVI step (pyro_b200/csrc/latent.cu): a reparameterised Normal guide site
 * z ~ Normal(loc, scale) -- scale possibly given as log(scale), the unconstrained storage of a positive
 * parameter (pyro/params/param_store.py:125-156) -- together with a Normal prior on the same z whose
 * parameters need no gradient.  Replaces, per site and step, the reference's exp / randn / addcmul
 * (torch/distributions/normal.py:82-85), both log_prob + sum chains (pyro/poutine/trace_struct.py:264-278) and
 * their autograd backward, including the accumulation of the two gradients that reach z.
 * A job is one site (<= B2_RSAMPLE_MAX_N elements); one CTA per job, so the sites of a step share a launch.
 *   b2_latent_normal_draw      z, eps [shape] contiguous out; out0 = 0-d SUM log Normal(z | loc, scale);
 *                              noise from Philox(seed, stream = job << 32 | element, launch counter)
 *   b2_latent_normal_prior     out0 = 0-d SUM log Normal(z | prior_loc, prior_scale), value only
 *   b2_latent_normal_backward  g = gz + prior_weight * d log p(z)/dz;  out0 = d/dloc = g,
 *                              out1 = d/dscale = g*eps - c/scale  (or d/dlog_scale = g*eps*scale - c), each summed
 *                              over the dims where the operand's stride is 0 (its stored shape, contiguous)
 * loc_stride .. prior_scale_stride: element strides of the broadcast views over shape (0 = broadcast).
 */
#define B2_LATENT_MAX_JOBS 8
#define B2_LATENT_LOG_SCALE 1   /* `scale` holds log(scale) */
#define B2_LATENT_ACC_OUT0 2    /* backward: out0 += d/dloc (accumulate into an existing .grad) instead of = */
#define B2_LATENT_ACC_OUT1 4    /* backward: out1 += d/dscale | d/dlog_scale */
typedef struct {
  int32_t dtype, ndim, flags, pad_;
  int64_t shape[B2_MAX_DIMS];
  int64_t loc_stride[B2_MAX_DIMS], scale_stride[B2_MAX_DIMS];
  int64_t prior_loc_stride[B2_MAX_DIMS], prior_scale_stride[B2_MAX_DIMS];
  const void* loc;
  const void* scale;
  const void* prior_loc;   /* may be NULL (draw, backward without prior) */
  const void* prior_scale;
  void* z;
  void* eps;
  const void* gz;          /* backward only; NULL = zero */
  void* out0;
  void* out1;
  double c;                /* backward: coefficient of SUM log q in the loss */
  double prior_weight;     /* backward: coefficient of SUM log p in the loss */
} b2_latent_job;
int b2_latent_normal_draw(const b2_latent_job* jobs, int n_jobs, void* rng_state, void* stream);
int b2_latent_normal_prior(const b2_latent_job* jobs, int n_jobs, void* stream);
int b2_latent_normal_backward(const b2_latent_job* jobs, int n_jobs, void* stream);
/* The prior sums of all jobs AND the assembly of the step's loss in one one-CTA launch (replaces
 * b2_latent_normal_prior + b2_elbo_combine when the sites are small):
 *   *out = SUM_j job_coeffs[j] * SUM log Normal(z_j | prior_j)  +  SUM_t term_coeffs[t] * *terms[t]
 * terms: 0-d device scalars of the jobs' dtype (the other per-site sums of the ELBO); jobs[j].out0 (optional)
 * receives the j-th prior sum.  pyro/infer/trace_elbo.py:82-112,147-152. */
#define B2_LATENT_MAX_TERMS 24
int b2_latent_normal_prior_combine(const b2_latent_job* jobs, int n_jobs, const double* job_coeffs,
                                   const void* const* terms, const double* term_coeffs, int n_terms, void* out,
                                   void* stream);

/*
 * b2_reduce_to -- sum a strided full-shape tensor down to an output whose zero strides mark the
 * reduced dims (the "sum_to_size" the fused kernels do not cover in-kernel).
 */
int b2_reduce_to(const b2_tensor* src, b2_tensor* dst, void* workspace, size_t workspace_bytes,
                 void* stream);

/*
 * b2_elbo_combine -- out = SUM_i coeffs[i] * (*terms[i]) over n <= 32 zero-dimensional DEVICE
 * scalars of `dtype` (`terms` and `coeffs` are HOST arrays, passed to the kernel by value; added
 * in index order).  Assembles the loss from the per-site sums in one launch; replaces the chain
 * of python-level `elbo_particle = elbo_particle + site["log_prob_sum"]` additions, the
 * `/ num_particles` and the negation of pyro/infer/trace_elbo.py:82-112,147-152.
 */
int b2_elbo_combine(const void* const* terms, const double* coeffs, int n, int dtype, void* out,
                    void* stream);

/*
 * b2_glm_bernoulli_logits -- fused Bayesian-logistic-regression likelihood term (BASELINE
 * config 2): for P particles, logits[p,n] = <X[n,:], W[p,:]> + b[p];
 *   sum_p[p]  = SUM_n ( y[n]*logits - softplus(logits) )               (Bernoulli log_prob)
 *   dW[p,:]   = weight * SUM_n (y[n] - sigmoid(logits[p,n])) * X[n,:]
 *   db[p]     = weight * SUM_n (y[n] - sigmoid(logits[p,n]))
 * X and y are read from HBM exactly once for value AND gradient.  Replaces the chain
 * matmul -> Bernoulli(logits).log_prob -> sum -> backward (pyro/poutine/trace_struct.py:264-278
 * applied to the model of tests/infer/mcmc/test_hmc.py:189-198).
 * X: [N,D] row-major fp32 (16-byte aligned), D in {4, 8, 16, 32}; W: [P,D]; b: [P] (nullable);
 * y: [N] fp32.
 * out_total (nullable): scalar, (=|+=) sum_coeff * scale * SUM_p sum_p[p].
 * flags: B2_FLAG_ACCUMULATE_SUM, B2_FLAG_GLM_FP32, B2_FLAG_GLM_3XTF32; any other bit -> B2_ERR_BAD_SHAPE.
 * Kernel choice:
 *   - the exact fp32 SIMT kernel when B2_FLAG_GLM_FP32 is set, D != 32, y is not 16-byte aligned,
 *     N >= 2^31, or N < 8192 without B2_FLAG_GLM_3XTF32;
 *   - otherwise the tcgen05 tensor-core kernel, which runs both contractions out of TMA-staged tiles with
 *     TMEM accumulators (glm_tc.cu).  W is split hi + lo (two TF32 MMAs per k-step), which removes the
 *     only error that is COHERENT over rows (a rounded W shifts every row's logit the same way and
 *     survives the N-term sums); g = y - sigmoid is rounded to nearest TF32.  X is split hi + lo as well
 *     (every logit fp32-exact) when B2_FLAG_GLM_3XTF32 is set or N < 65536; above that it is rounded to
 *     nearest TF32 (incoherent, averages as 1/sqrt(N)): sum_p, dW, db agree with an fp64 evaluation to
 *     ~1e-6 / ~1e-5 relative at N = 1e6.
 * workspace: b2_glm_workspace() bytes, zero-initialised ONCE by the caller (its first 256 bytes
 * hold a ticket counter that the library leaves zeroed).  Two launches: the streaming kernel
 * and a finish kernel that sums the CTA partials in a fixed order (deterministic).
 */
int b2_glm_bernoulli_logits(const float* X, const float* y, const float* W, const float* b,
                            int64_t N, int D, int P, double scale, double weight, double sum_coeff,
                            int flags, float* out_sum_p, float* out_total, float* out_dW,
                            float* out_db, void* workspace, size_t workspace_bytes, void* stream);
size_t b2_glm_workspace(int64_t N, int D, int P);

/* ---- optimisers --------------------------------------------------------------------------
 * Multi-tensor fused updates replacing PyroOptim's per-parameter Python loop
 * (pyro/optim/optim.py:117-155).  Per-tensor scalar state lives in DEVICE arrays so a captured
 * CUDA graph can be replayed: `steps` (int32) and `lrs` (double) are advanced on device. */

/*
 * b2_clipped_adam -- pyro/optim/clipped_adam.py:62-98 for n tensors in one launch sequence:
 *   lr <- lr*lrd;  g <- clamp(g, -clip, clip);  t += 1;  g += wd*p (if wd != 0)
 *   m <- b1*m + (1-b1)*g;  v <- b2*v + (1-b2)*g*g
 *   p <- p - lr*sqrt(1-b2^t)/(1-b1^t) * m/(sqrt(v)+eps)
 * ptr tables (device arrays of n device pointers): p, g, m, v; numel: device int64[n].
 * hyper: device double[n*8] rows (beta1, beta2, eps, weight_decay, clip_norm, lrd, -, -); slot 6
 * receives the bias-corrected step size computed on device.
 * lrs: device double[n] (current lr, updated in place); steps: device int32[n] (updated).
 * zero_grad != 0 also zeroes g (pyro/infer/util.py:85-91 fused in).  dtype: B2_F32 or B2_F64.
 * total_numel/max_numel are host-side hints for grid sizing.
 */
int b2_clipped_adam(int n, void* const* p, void* const* g, void* const* m, void* const* v,
                    const int64_t* numel, double* hyper, double* lrs, int32_t* steps, int dtype,
                    int zero_grad, int64_t max_numel, void* stream);

/*
 * b2_adagrad_rmsprop -- pyro/optim/adagrad_rmsprop.py:54-87:
 *   s = g*g (first step) else s <- (1-t)*s + t*g*g;  lr = eta*step^(-0.5+delta)
 *   p <- p - lr*g/(1+sqrt(s))
 * hyper: device double[n*4] rows (eta, delta, t, -); slot 3 receives the step's lr.
 */
int b2_adagrad_rmsprop(int n, void* const* p, void* const* g, void* const* s,
                       const int64_t* numel, double* hyper, int32_t* steps, int dtype,
                       int zero_grad, int64_t max_numel, void* stream);

/* ---- HMC / NUTS --------------------------------------------------------------------------
 * State layout: chains are the leading dim, [C, D] row-major ("one row per chain"). */

/*
 * b2_leapfrog_half_kick_drift / b2_leapfrog_half_kick -- the two elementwise halves of
 * pyro/ops/integrator.py:45-65 (_single_step_verlet) over [C,D] with per-chain step size and
 * diagonal inverse mass (pyro/infer/mcmc/adaptation.py:328-347 kinetic_grad):
 *   kick_drift:  r <- r - (eps/2)*g ;  z <- z + eps * minv * r
 *   kick:        r <- r - (eps/2)*g ;  ke[c] = 0.5 * SUM_d minv*r*r   (optional)
 * eps: [C] (signed: direction folded in); minv: [C,D] or [D] (minv_chain_stride 0);
 * active (nullable uint8 [C]): chains with active==0 are left untouched.
 * workspace for the kinetic-energy reduction and the potentials: b2_mcmc_workspace(C) bytes.
 */
size_t b2_mcmc_workspace(int64_t C);
int b2_leapfrog_half_kick_drift(void* z, void* r, const void* g, const void* eps,
                                const void* minv, int64_t minv_chain_stride,
                                const uint8_t* active, int64_t C, int64_t D, int dtype,
                                void* stream);
int b2_leapfrog_half_kick(void* r, const void* g, const void* eps, const void* minv,
                          int64_t minv_chain_stride, const uint8_t* active, void* ke, int64_t C,
                          int64_t D, int dtype, void* workspace, size_t workspace_bytes,
                          void* stream);

/* Native potentials ("compiled model classes").  U is the potential energy in UNCONSTRAINED
 * space including the log|det J| of the constraining transforms, exactly as
 * pyro/infer/mcmc/util.py:275-286 builds it. */
#define B2_MODEL_HIER_NORMAL 0 /* eight_schools family, examples/eight_schools/mcmc.py:27-34:
                                  z = [mu, log_tau, eta[J]];  mu~N(0,s_mu), tau~HalfCauchy(s_tau),
                                  eta~N(0,1), y~N(mu+tau*eta, sigma).  data = (y[J], sigma[J]),
                                  hyper = (s_mu, s_tau) */
#define B2_MODEL_LOGISTIC 1    /* tests/infer/mcmc/test_hmc.py:189-198 family:
                                  z = beta[D];  beta ~ Normal(0, s) i.i.d.,
                                  y ~ Bernoulli(logits = X beta).  data = (X[J,D], y[J]),
                                  hyper = (s) */

typedef struct {
  int32_t model;  /* B2_MODEL_* */
  int32_t dtype;  /* B2_F32 / B2_F64 for state and data */
  int64_t J;      /* data size */
  int64_t D;      /* latent dimension of one chain */
  const void* data0; /* y      | X[J, D]  */
  const void* data1; /* sigma  | y[J]     */
  double hyper[4];
} b2_model;

/*
 * b2_potential_grad -- U[c] and dU/dz[c,:] for C chains in one launch
 * (pyro/ops/integrator.py:68-94 potential_grad + pyro/infer/mcmc/util.py:275-286).
 */
int b2_potential_grad(const b2_model* model, const void* z, void* U, void* grad, int64_t C,
                      const uint8_t* active, void* workspace, size_t workspace_bytes,
                      void* stream);
size_t b2_potential_workspace(const b2_model* model, int64_t C);

/*
 * b2_nuts_small -- whole NUTS transitions on device for a native model with small D
 * (D <= B2_NUTS_SMALL_MAX_D): one warp per chain keeps (z, r, grad) and the tree
 * bookkeeping in registers/shared memory; iterative tree doubling, multinomial sampling,
 * U-turn checks and Philox draws happen without returning to the host
 * (pyro/infer/mcmc/nuts.py:197-522).  Runs `num_transitions` transitions per chain.
 *   z [C,D] in/out; U [C], grad [C,D] in/out (cached, nuts.py:480-494);
 *   step_size [C]; minv [C,D] (diag inverse mass);
 *   seed + chain offset feed a counter-based Philox stream (rng_counter [C] uint64 in/out);
 *   samples_out (nullable) [num_transitions, C, D]; accept_prob_out [num_transitions, C];
 *   depth_out / diverging_out / num_steps_out [num_transitions, C] int32.
 */
#define B2_NUTS_SMALL_MAX_D 64
int b2_nuts_small(const b2_model* model, void* z, void* U, void* grad, const void* step_size,
                  const void* minv, int64_t C, int num_transitions, int max_tree_depth,
                  double max_delta_energy, uint64_t seed, uint64_t* rng_counter,
                  void* samples_out, void* accept_prob_out, int32_t* depth_out,
                  int32_t* diverging_out, int32_t* num_steps_out, void* stream);

/*
 * b2_nuts_leaf_vector -- lockstep iterative NUTS (large latent dimension): everything a new leaf
 * needs over the [C, D] state in ONE pass (pyro/infer/mcmc/nuts.py:197-248,285-342 restated
 * iteratively): whitened momentum ru = r*sqrt(minv); rsub += ru; proposal copy zs,gs <- z,g where
 * take[c]; on an even leaf the checkpoint store rck/sck[store_slot] (store_slot >= 0), on an odd
 * leaf (store_slot < 0) the 2*nblk U-turn dot products of the blocks ending at this leaf
 * (checkpoint slots idx_max, idx_max-1, ...), written to dots[c*2*nblk + 2j + {0,1}].
 * rck/sck: [slots, C, D].  Chains with active[c]==0 are untouched.
 */
int b2_nuts_leaf_vector(const void* z, const void* r, const void* g, const void* minv,
                        int64_t minv_chain_stride, const uint8_t* active, const uint8_t* take,
                        void* rsub, void* zs, void* gs, void* rck, void* sck, int store_slot,
                        int idx_max, int nblk, void* dots, int64_t C, int64_t D, int dtype,
                        void* workspace, size_t workspace_bytes, void* stream);

/*
 * b2_nuts_leaf_hier -- lockstep iterative NUTS, one new leaf for every still-active chain, for the
 * B2_MODEL_HIER_NORMAL model class (BASELINE configs 1 / 4) at any J: TWO launches replace the
 * five launches + ~20 [C]-sized tensor ops of the generic leaf (b2_leapfrog_half_kick_drift,
 * b2_potential_grad, b2_leapfrog_half_kick, b2_nuts_leaf_vector and the scalar glue):
 *   pass 1, over [C, D]: the whole velocity-Verlet step (pyro/ops/integrator.py:45-65) with the
 *     local gradients recomputed from the global coordinates instead of stored; whitened momentum,
 *     running subtree sum, checkpoint store (store_slot >= 0, even leaf) or the 2*nblk U-turn dot
 *     products (odd leaf; checkpoint slots idx_max, idx_max-1, ...); proposal copy zs <- z for
 *     chains whose PREVIOUS leaf was drawn (take[c], written by the previous call);
 *   pass 2, one warp per chain: potential energy and global gradients at the new point, second
 *     half kick of the global coordinates, then the scalar tree logic of pyro/infer/mcmc/nuts.py:
 *     197-248 for one leaf: energy (NaN -> inf), divergence (delta > max_delta_energy), accept-prob
 *     sum, progressive multinomial draw (Philox stream (seed, chain), counter rng_counter[c]),
 *     U-turn flags -> done[c].
 * State is advanced IN PLACE.  After the last leaf of a subtree the caller copies z -> zs for
 * chains with take[c] still set.  Chains with done[c] != 0 are untouched.
 */
typedef struct {
  void *zL, *rL, *zR, *rR; /* [C, D] position / momentum at the two ends of the trajectory, D = J + 2;
                              the end picked by dir[c] is advanced IN PLACE (a doubling always extends
                              the trajectory; a chain cut short is `done` and its ends are dead) */
  const uint8_t* dir; /* [C] 1 = the right end grows (with eps[c] > 0), 0 = the left end */
  void *gscL, *gscR;  /* [C, 2] dU/d(mu, log tau) at the two ends */
  const void* minv;   /* diagonal inverse mass, chain stride minv_chain_stride (0 = shared) */
  int64_t minv_chain_stride;
  void *rsub;         /* [C, D] whitened momentum sum of the subtree under construction (leaf 0
                         overwrites it: no zero-fill needed between subtrees) */
  void *zs;           /* [C, D] proposal of the subtree */
  void *rck, *sck;    /* [slots, C, D] checkpoints: first-leaf momentum / running sum */
  const void* eps;    /* [C] signed step size */
  void *gsc_s;        /* [C, 2] dU/d(mu, log tau) at the proposal */
  void *U, *Us;       /* [C] potential at the growing end / at the proposal */
  const void* energy0; /* [C] initial energy of the transition */
  void *logw_sub, *sum_accept, *num_prop; /* [C] */
  uint8_t *done, *diverged, *take;        /* [C] */
  int32_t* num_leapfrogs;                 /* [C] nullable: += 1 per active chain */
  uint64_t* rng_counter;                  /* [C] */
  uint64_t seed;
  double max_delta_energy;
  int64_t C;
} b2_nuts_lockstep;

int b2_nuts_leaf_hier(const b2_model* model, const b2_nuts_lockstep* st, int leaf, int store_slot,
                      int idx_max, int nblk, void* workspace, size_t workspace_bytes, void* stream);
size_t b2_nuts_leaf_hier_workspace(int64_t C, int64_t J);

/*
 * b2_nuts_tree_merge -- root of the doubling loop (pyro/infer/mcmc/nuts.py:285-342, 404-440) after
 * a subtree is finished, for every chain with done[c] == 0:  rsum += rsub;  rho = rsum -
 * (ruL + ruR)/2 with ru = r * sqrt(minv) at the two trajectory ends;  dots[c] = (<ruL, rho>,
 * <ruR, rho>) -- the generalised U-turn test of the whole tree.  One pass over [C, D].
 * workspace: C * 64 * 2 doubles (the b2_mcmc_workspace() size suffices).
 */
int b2_nuts_tree_merge(const void* rL, const void* rR, const void* minv, int64_t minv_chain_stride,
                       void* rsum, const void* rsub, const uint8_t* done, void* dots, int64_t C,
                       int64_t D, int dtype, void* workspace, size_t workspace_bytes, void* stream);

/* b2_rows_copy_masked -- dst[c, :] = src[c, :] for chains with mask[c] != 0 ([C, D] row-major):
 * the proposal hand-over `torch.where(accepted, new, old)` of nuts.py:303-320 moving only the
 * accepted rows. */
int b2_rows_copy_masked(void* dst, const void* src, const uint8_t* mask, int64_t C, int64_t D,
                        int dtype, void* stream);

/* ---- misc -------------------------------------------------------------------------------- */
const char* b2_last_error(int code);
int b2_version(void);
/* number of kernel launches issued by this library in this process (for bench.py's
 * gpu_launches claim). */
int64_t b2_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* PYRO_B200_H_ */
