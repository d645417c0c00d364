// glm.cu -- fused Bayesian-logistic-regression likelihood term for P particles (BASELINE config 2).
//
// One pass over X[N,D] and y[N] yields, for every particle p:
//   sum_p = SUM_n  y_n * l_pn - softplus(l_pn),      l_pn = <X[n,:], W[p,:]> + b[p]
//   dW[p,:] = weight * SUM_n (y_n - sigmoid(l_pn)) X[n,:],   db[p] = weight * SUM_n (y_n - sigmoid(l_pn))
// so X and y are read from HBM exactly once for the value AND the gradient (132 MB at
// N=1e6, D=32), instead of materialising the [P,N] logits / log_prob / grad tensors that the
// reference chain (matmul -> Bernoulli.log_prob -> sum -> backward) writes and re-reads.
//
// SIMT formulation (first version): CTA = 256 threads = 4 row groups x 64 particles.  Each thread
// keeps W[p,:] and its dW[p,:] accumulator in registers; X tiles are staged through shared memory
// with cp.async double buffering and read back as warp-wide broadcasts (every lane of a warp has a
// different particle but the same row, so an LDS.128 serves 4 FMAs x 2 uses for all 32 lanes).
// FLOPs = 4*N*D*P; at P=64, D=32 the FMA pipe, not HBM, bounds this version (see DESIGN.md).
#include <cuda_pipeline.h>

#include "b2_common.cuh"
#include "b2_math.cuh"

namespace b2 {

constexpr int kGlmTileRows = 64;     // rows per shared-memory tile
constexpr int kGlmParticles = 64;    // particles per CTA (blockIdx.y slabs of 64)
constexpr int kGlmRowGroups = 4;     // 256 / 64

template <int D>
__global__ void __launch_bounds__(256) glm_bernoulli_kernel(const float* __restrict__ X,
                                                            const float* __restrict__ y,
                                                            const float* __restrict__ W,
                                                            const float* __restrict__ b, int64_t N,
                                                            int P, float* __restrict__ partials) {
  // partials layout: [gridDim.x][P][D + 2]  (dW..., db, sum)
  __shared__ __align__(16) float xs[2][kGlmTileRows * D];
  __shared__ float ys[2][kGlmTileRows];
  const int tid = threadIdx.x;
  const int pl = tid & (kGlmParticles - 1);
  const int rg = tid >> 6;
  const int p = blockIdx.y * kGlmParticles + pl;
  const bool pon = p < P;

  float w[D], dw[D];
#pragma unroll
  for (int d = 0; d < D; ++d) {
    w[d] = pon ? W[(int64_t)p * D + d] : 0.f;
    dw[d] = 0.f;
  }
  const float bias = (pon && b) ? b[p] : 0.f;
  float db = 0.f, sum = 0.f;

  const int64_t ntiles = (N + kGlmTileRows - 1) / kGlmTileRows;
  constexpr int kVecPerTile = kGlmTileRows * D / 4;

  auto stage = [&](int buf, int64_t tile) {
    const int64_t row0 = tile * kGlmTileRows;
    const int64_t rows = (N - row0 < kGlmTileRows) ? (N - row0) : kGlmTileRows;
    const float4* src = reinterpret_cast<const float4*>(X + row0 * D);
    float4* dst = reinterpret_cast<float4*>(xs[buf]);
    const int nvec = (int)(rows * D / 4);
    for (int i = tid; i < kVecPerTile; i += 256) {
      if (i < nvec) __pipeline_memcpy_async(dst + i, src + i, 16);
      else dst[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if (tid < kGlmTileRows) {
      if (tid < rows) __pipeline_memcpy_async(&ys[buf][tid], y + row0 + tid, 4);
      else ys[buf][tid] = 0.f;
    }
    __pipeline_commit();
  };

  int64_t tile = blockIdx.x;
  int buf = 0;
  if (tile < ntiles) stage(0, tile);
  for (; tile < ntiles; tile += gridDim.x) {
    const int64_t next = tile + gridDim.x;
    if (next < ntiles) stage(buf ^ 1, next);
    else __pipeline_commit();
    __pipeline_wait_prior(1);
    __syncthreads();
    const int64_t row0 = tile * kGlmTileRows;
    const int rows = (int)((N - row0 < kGlmTileRows) ? (N - row0) : kGlmTileRows);
    const float* xt = xs[buf];
#pragma unroll 2
    for (int r = rg; r < rows; r += kGlmRowGroups) {
      const float4* xr = reinterpret_cast<const float4*>(xt + r * D);
      float xv[D];
#pragma unroll
      for (int q = 0; q < D / 4; ++q) {
        const float4 v = xr[q];
        xv[4 * q + 0] = v.x; xv[4 * q + 1] = v.y; xv[4 * q + 2] = v.z; xv[4 * q + 3] = v.w;
      }
      // four independent partial dot products: a single accumulator is a chain of D dependent
      // FMAs (4 cycles each), which 4 resident warps per scheduler cannot hide
      float l0 = bias, l1 = 0.f, l2 = 0.f, l3 = 0.f;
#pragma unroll
      for (int d = 0; d < D; d += 4) {
        l0 = fmaf(xv[d + 0], w[d + 0], l0);
        l1 = fmaf(xv[d + 1], w[d + 1], l1);
        l2 = fmaf(xv[d + 2], w[d + 2], l2);
        l3 = fmaf(xv[d + 3], w[d + 3], l3);
      }
      const float l = (l0 + l1) + (l2 + l3);
      const float yn = ys[buf][r];
      // softplus / sigmoid sharing one exp (fast intrinsics: ex2.approx / lg2.approx / rcp)
      const float e = __expf(-fabsf(l));
      const float inv = __frcp_rn(1.f + e);
      const float sp = fmaxf(l, 0.f) + __logf(1.f + e);
      const float sg = (l >= 0.f) ? inv : e * inv;
      sum += yn * l - sp;
      const float g = yn - sg;
      db += g;
#pragma unroll
      for (int d = 0; d < D; ++d) dw[d] = fmaf(g, xv[d], dw[d]);
    }
    __syncthreads();
    buf ^= 1;
  }
  __pipeline_wait_prior(0);

  // reduce the 4 row groups through shared memory (reuse xs[0]: 64*D floats >= 3*64*(D+2)? no: use a loop)
  __syncthreads();
  float* red = xs[0];  // capacity kGlmTileRows*D = 64*D floats; we need 64 floats per pass
  float* out = partials + ((int64_t)blockIdx.x * P + p) * (D + 2);
#pragma unroll
  for (int d = 0; d < D + 2; ++d) {
    const float v = (d < D) ? dw[d < D ? d : 0] : (d == D ? db : sum);
    // stage groups 1..3, group 0 adds them in a fixed order
    if (rg > 0) red[(rg - 1) * kGlmParticles + pl] = v;
    __syncthreads();
    if (rg == 0 && pon) {
      out[d] = ((v + red[pl]) + red[kGlmParticles + pl]) + red[2 * kGlmParticles + pl];
    }
    __syncthreads();
  }
}

// second stage: fixed-order sum over the CTAs' partials; applies weight / scale.
// One WARP per entry of the [P, D+2] table: lanes stride over the CTAs (L2-resident partials),
// then a shuffle tree -- a thread-per-entry loop over ~300 dependent loads took 35 us.
__global__ void __launch_bounds__(256) glm_finish_kernel(const float* __restrict__ partials,
                                                         int nblocks, int P, int D, double scale,
                                                         double weight, float* __restrict__ sum_p,
                                                         float* __restrict__ out_dW,
                                                         float* __restrict__ out_db,
                                                         double sum_coeff, int flags,
                                                         float* __restrict__ out_total,
                                                         unsigned int* __restrict__ ticket) {
  pdl_enter();
  const int total = P * (D + 2);
  const int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (e >= total) return;
  double s = 0.0;
  for (int bl = lane; bl < nblocks; bl += 32) s += (double)partials[(int64_t)bl * total + e];
  s = warp_sum(s);
  const int p = e / (D + 2), d = e - p * (D + 2);
  if (d < D) {
    if (lane == 0 && out_dW) out_dW[(int64_t)p * D + d] = (float)(weight * scale * s);
    return;
  }
  if (d == D) {
    if (lane == 0 && out_db) out_db[p] = (float)(weight * scale * s);
    return;
  }
  // per-particle sum; the LAST of the P warps to get here also totals them (fixed order), with
  // the ELBO coefficient -- a ticket instead of a third launch
  unsigned int t = 0;
  if (lane == 0) {
    sum_p[p] = (float)(scale * s);
    if (out_total) {
      __threadfence();
      t = atomicAdd(ticket, 1u);
    }
  }
  if (!out_total) return;
  t = __shfl_sync(0xffffffffu, t, 0);
  if (t != (unsigned)(P - 1)) return;
  __threadfence();
  double acc = 0.0;
  for (int q = lane; q < P; q += 32) acc += (double)__ldcg(sum_p + q);
  acc = warp_sum(acc);
  if (lane == 0) {
    const double v = sum_coeff * acc;
    *out_total = (flags & B2_FLAG_ACCUMULATE_SUM) ? (float)((double)*out_total + v) : (float)v;
    *ticket = 0u;
  }
}

// tcgen05 + TMA variant (glm_tc.cu)
int glm_tc_grid_x(int64_t N);
int launch_glm_tc(const float* X, const float* y, const float* W, const float* b, int64_t N, int P,
                  float* partials, int gx, bool split_x, cudaStream_t s);

inline int glm_grid_x(int64_t N) {
  const int64_t ntiles = (N + kGlmTileRows - 1) / kGlmTileRows;
  int64_t gx = (int64_t)kNumSMs * 2;  // two 256-thread CTAs per SM (register-limited)
  if (gx > ntiles) gx = ntiles;
  if (gx < 1) gx = 1;
  return (int)gx;
}

}  // namespace b2

using namespace b2;

extern "C" size_t b2_glm_workspace(int64_t N, int D, int P) {
  // [ticket, 256 B] + CTA partials + one [P] row for the per-particle sums
  return 256 + ((size_t)glm_grid_x(N) * (size_t)P * (size_t)(D + 2) + (size_t)P) * sizeof(float);
}

extern "C" int b2_glm_bernoulli_logits(const float* X, const float* y, const float* W,
                                       const float* b, int64_t N, int D, int P, double scale,
                                       double weight, double sum_coeff, int flags,
                                       float* out_sum_p, float* out_total, float* out_dW,
                                       float* out_db, void* workspace, size_t workspace_bytes,
                                       void* stream) {
  if (!X || !y || !W) return B2_ERR_NULL;
  if (N <= 0 || P <= 0) return B2_ERR_BAD_SHAPE;
  // an unknown bit is refused, not ignored: a caller asking for a kernel variant must not silently get another
  if (flags & ~(B2_FLAG_ACCUMULATE_SUM | B2_FLAG_GLM_FP32 | B2_FLAG_GLM_3XTF32)) return B2_ERR_BAD_SHAPE;
  if (reinterpret_cast<uintptr_t>(X) % 16 != 0) return B2_ERR_BAD_SHAPE;
  if (!workspace || workspace_bytes < b2_glm_workspace(N, D, P)) return B2_ERR_WORKSPACE;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  // below 8 Ki rows the single-pass TF32 gradient contraction has not averaged its operand rounding
  // (2^-12 relative per term) below the fp32 tolerance yet: those sizes take the exact fp32 SIMT kernel
  // unless B2_FLAG_GLM_3XTF32 asks for the tensor cores explicitly; the TMA loads need a 16-byte aligned y
  // and 32-bit row coordinates
  const bool use_tc = (D == 32) && !(flags & B2_FLAG_GLM_FP32) && (N >= 8192 || (flags & B2_FLAG_GLM_3XTF32)) &&
                      reinterpret_cast<uintptr_t>(y) % 16 == 0 && N < ((int64_t)1 << 31);
  const int gx = use_tc ? glm_tc_grid_x(N) : glm_grid_x(N);
  dim3 grid((unsigned)gx, (unsigned)((P + kGlmParticles - 1) / kGlmParticles), 1);
  unsigned int* ticket = reinterpret_cast<unsigned int*>(workspace);
  float* partials = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + 256);
  if (use_tc) {
    // W split by default; below 64 Ki rows the incoherent X rounding has not averaged out yet -> X split too
    const bool split_x = (flags & B2_FLAG_GLM_3XTF32) || N < 65536;
    const int rc = launch_glm_tc(X, y, W, b, N, P, partials, gx, split_x, s);
    if (rc != 0) return rc;
  } else
  switch (D) {
    case 4: glm_bernoulli_kernel<4><<<grid, 256, 0, s>>>(X, y, W, b, N, P, partials); break;
    case 8: glm_bernoulli_kernel<8><<<grid, 256, 0, s>>>(X, y, W, b, N, P, partials); break;
    case 16: glm_bernoulli_kernel<16><<<grid, 256, 0, s>>>(X, y, W, b, N, P, partials); break;
    case 32: glm_bernoulli_kernel<32><<<grid, 256, 0, s>>>(X, y, W, b, N, P, partials); break;
    default: return B2_ERR_BAD_SHAPE;
  }
  float* sum_p = out_sum_p ? out_sum_p : partials + (size_t)gx * P * (D + 2);
  const int total = P * (D + 2);
  launch_pdl(glm_finish_kernel, dim3((total + 7) / 8), dim3(256), 0, s,
             partials, gx, P, D, scale, weight, sum_p, out_dW, out_db, sum_coeff, flags, out_total, ticket);
  const int nl = 2;
  count_launch(nl);
  return check_launch();
}
