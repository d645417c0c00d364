// glm_tc.cu -- Blackwell-native fused logistic-regression likelihood kernel (BASELINE config 2):
// TMA tile loads, tcgen05.mma with TMEM accumulators, warp-specialised persistent CTAs.
//
// Same contract as glm_bernoulli_kernel (glm.cu): ONE pass over X[N,32] and y[N] gives, for up to 64
// weight vectors (particles) per CTA slab, sum_n log Bernoulli(y_n | logits = x_n.w_p + b_p), dW and
// db.  It replaces (reference, per SVI step): the user model's `w @ X.T + b`, then
// torch/distributions/bernoulli.py:121-125 (log_prob), pyro/poutine/trace_struct.py:264-278 (.sum())
// and the autograd backward of all three.
//
// Per 128-row tile (one persistent CTA per SM, tiles round-robin over CTAs):
//
//   GEMM 1   D1[n, p] = sum_d X[n, d] W[p, d] + b[p]      M = 128 rows, N = 64 particles, K = 32
//            W split hi + lo, two TF32 MMAs per k-step -- the rounding of W is the only error of a TF32
//            GEMM 1 that is COHERENT over rows (it shifts all N logits of a particle the same way and
//            survives the N-term sums); X is rounded to nearest in place (incoherent, averages as
//            1/sqrt(N)).  SPLIT_X splits X as well (every logit exact to ~1e-6).  fp32 accumulation in
//            TMEM; the bias enters through one more MMA (A = ones, B = [b_hi, b_lo, 0...]).
//   epilogue sixteen warps tcgen05.ld the 128 x 64 logits (thread = row, 16 particles each), evaluate
//            lp = y*l - softplus(l), g = y - sigmoid(l) (3 MUFU + ~12 FMA-pipe ops per element, in
//            batches of 8 so the MUFU latency is covered inside the warp), keep the per-particle lp sums
//            in registers and store g^T (rounded to nearest TF32) into shared memory as the K-major A
//            operand of GEMM 2.
//   GEMM 2   [dW | db][p, :] += sum_n g[n, p] [X | 1][n, :]   M = 64, N = 40 (32 columns of X^T and 8 rows
//            of ones), K = 128: single-pass TF32 on round-to-nearest operands (unbiased;
//            |err| <= 2^-11 sum|g x|, measured 4e-6 relative at N = 1e6); one accumulator per 32-row
//            k-block, summed once at the end of the kernel.
//
// TF32 MN-major operands only exist in the 32-byte-atom swizzle, so instead of re-reading the X tile
// in a second layout, four "split" warps transform each TMA tile once: RN-rounded X in place (plus X_lo
// with SPLIT_X) for GEMM 1 and the transposed X^T[d, n] for GEMM 2.  All operand tiles are K-major
// SWIZZLE_128B, the layout TMA writes natively.
//
// Warp roles (704 threads): warp 0 TMA producer, warp 1 MMA issuer + TMEM owner (the whole warp walks
// the loop, one elected lane issues; the issue order of a batch is static so consecutive MMAs are 1-3
// instructions apart), warps 2-17 epilogue (TMEM sub-partition = warp % 4), warps 18-21 split pass.
// Pipelines (all mbarriers): TMA ring of 4 X stages, X^T/y ring of 3 stages, D1 double-buffered in TMEM
// with GEMM 1 running TWO tiles ahead (it is issued interleaved with GEMM 2 of tile j as soon as the
// epilogue of tile j is done), g^T double-buffered in shared memory.
//
// What bounds it (B200, N = 1e6, P = 64; profiles/glm_tc_r2.md): 89 us.  An isolated tcgen05.mma of these
// shapes costs (A bytes + B bytes) / 128 B per clock -- 51 cycles for 128x64x8, 28 for 64x40x8
// (profiles/umma_bench.cu) -- i.e. the K = 8 TF32 instruction is bound by the shared-memory operand
// fetch, and that same 128 B/clk port also carries the split pass, the g^T stores and the TMA writes:
// ~200 KB of shared-memory traffic per 16 KB tile, >= 1600 cycles, against 1536 cycles of MUFU work.
// ncu: tensor pipe active 89 %, issue slots 65 %, XU pipe 56 %, DRAM 1.0x the algorithmic bytes.
//
// Determinism: every CTA writes its partials once; glm_finish_kernel adds them in a fixed order.
#include <cuda.h>
#include <cuda/std/type_traits>

#include "b2_common.cuh"

namespace b2 {
namespace tc {

constexpr int kRows = 128;
constexpr int kD = 32;
constexpr int kP = 64;
constexpr int kMaxStagesT = 3;
constexpr int kEpiWarp0 = 2, kEpiWarps = 16;       // 4 per SM sub-partition: latency hiding for the MUFU chains
constexpr int kEpiCols = kP * 4 / kEpiWarps;        // particles (TMEM columns) per epilogue thread
constexpr int kSplitWarp0 = kEpiWarp0 + kEpiWarps, kSplitWarps = 4;
constexpr int kThreads = (kSplitWarp0 + kSplitWarps) * 32;
constexpr int kMaxStagesX = 4;

constexpr uint32_t kTile = kRows * kD * 4;                    // 16 KB
constexpr uint32_t kXStage = kTile + 512;                     // bytes per TMA transaction: X tile + 128 y values
constexpr uint32_t kGBuf = 4 * kP * 128;                      // g^T: [kb 4][p 64][32 n] fp32 = 32 KB
constexpr uint32_t kXtBlock = (kD + 8) * 128;                 // X^T k-block: 32 rows of d + 8 rows of ones
constexpr uint32_t kXtStage = 4 * kXtBlock;                   // 20 KB

// Precision of GEMM 1 (the logits).  Default (SPLIT_X = false): W split hi/lo -- the rounding error of W
// is the only COHERENT error of a TF32 GEMM 1 (it is the same for all rows, so it does not average out
// over the N-term sums); X is rounded to nearest in place (incoherent, averages as 1/sqrt(N)).
// SPLIT_X: full 3xTF32 (X split as well): every logit exact to ~1e-6, at the price of a shallower TMA
// ring (the X_lo tiles take the shared memory of two X stages).  Taken below 64 Ki rows, where the
// incoherent X rounding has not averaged out yet.
template <bool SPLIT_X>
struct Layout {
  static constexpr int kStagesX = SPLIT_X ? 2 : 4;                 // TMA ring: X tile (hi in place) + y
  static constexpr int kStagesL = SPLIT_X ? 2 : 0;                 // X_lo ring
  static constexpr int kStagesT = 3;                               // GEMM 2 B-operand (+ y) ring: split pass -> GEMM 2
                                                                   // (>= 3: GEMM 1 runs two tiles ahead)
  static constexpr uint32_t OFF_X = 0;
  static constexpr uint32_t OFF_XLO = OFF_X + kStagesX * kTile;
  static constexpr uint32_t OFF_XT = OFF_XLO + kStagesL * kTile;   // [stage][kb 4][d 32 + 8 ones][32 n] fp32
  static constexpr uint32_t OFF_G = OFF_XT + kStagesT * kXtStage;
  // the g buffers double as the [128][65] fp32 scratch of the final reduction (33 280 bytes)
  static_assert(2 * kGBuf >= 128 * 65 * 4, "reduction scratch");
  static constexpr uint32_t OFF_WHI = OFF_G + 2 * kGBuf;           // [p 64][32 d] SW128, 8 KB
  static constexpr uint32_t OFF_WLO = OFF_WHI + 8192;
  static constexpr uint32_t OFF_WB = OFF_WLO + 8192;               // bias tile (k = 0: b_hi, k = 1: b_lo)
  static constexpr uint32_t OFF_ONES = OFF_WB + 8192;              // 4 KB of 1.0f (no-swizzle operand)
  static constexpr uint32_t OFF_Y = OFF_ONES + 4096;               // [stage T][128] fp32 (epilogue reads)
  static constexpr uint32_t OFF_YX = OFF_Y + kStagesT * 512;       // [stage X][128] fp32 (TMA target)
  static constexpr uint32_t OFF_BAR = OFF_YX + kStagesX * 512;
  static constexpr uint32_t kSmemBytes = OFF_BAR + 256 + 1024;     // + slack for the 1024-byte alignment
};
static_assert(Layout<false>::kSmemBytes <= 232448 && Layout<true>::kSmemBytes <= 232448, "shared memory budget");

// barrier slots (8 bytes each)
enum : int {
  BAR_XFULL = 0,                         // [kMaxStagesX] TMA landed
  BAR_XREADY = BAR_XFULL + kMaxStagesX,  // [kMaxStagesX] split pass done
  BAR_XEMPTY = BAR_XREADY + kMaxStagesX, // [kMaxStagesX] GEMM 1 finished reading the X tile
  BAR_LEMPTY = BAR_XEMPTY + kMaxStagesX, // [2] GEMM 1 finished reading X_lo (SPLIT_X)
  BAR_TEMPTY = BAR_LEMPTY + 2,           // [kStagesT] GEMM 2 finished reading X^T
  BAR_D1FULL = BAR_TEMPTY + kMaxStagesT, // [2]
  BAR_D1EMPTY = BAR_D1FULL + 2,          // [2]
  BAR_GFULL = BAR_D1EMPTY + 2,           // [2]
  BAR_GEMPTY = BAR_GFULL + 2,            // [2]
  BAR_DONE = BAR_GEMPTY + 2,
  BAR_COUNT
};
static_assert(BAR_COUNT * 8 + 8 <= 256, "barrier block overflow");

constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kColD1 = 0, kColD2 = 128;   // D2[kb]: 40 columns each (32 of dW + 8 equal columns of db), kb = 0..3

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0, spins = 0;
  for (;;) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    if (ok) return;
    if (++spins > (1u << 26)) __trap();   // a protocol bug must not hang the device
  }
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void tma_load_1d(uint32_t dst, const CUtensorMap* map, int c0, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.1d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2}], [%3];"
      ::"r"(dst), "l"(map), "r"(c0), "r"(bar)
      : "memory");
}

// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout): start address >> 4 in
// [0,14), leading byte offset >> 4 in [16,30), stride byte offset >> 4 in [32,46), version 1 in
// [46,48), layout type in [61,64) (0 = no swizzle, 2 = SWIZZLE_128B).
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo, uint32_t layout) {
  return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) | (1ull << 46) | ((uint64_t)layout << 61);
}
// K-major SWIZZLE_128B tile of 128-byte rows: 8-row groups are 1024 bytes apart
__device__ __forceinline__ uint64_t desc_sw128(uint32_t saddr) { return make_desc(saddr, 0, 1024, 2); }

// instruction descriptor, kind::tf32, fp32 accumulate, both operands K-major
__host__ __device__ constexpr uint32_t idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void mma_tf32(uint32_t d_tmem, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a), "l"(b), "r"(idesc), "r"(acc)
      : "memory");
}

// one lane of a converged warp (the pattern the compiler needs to emit warp-uniform tcgen05 issue code
// without a per-instruction election loop)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred)
      :
      : "memory");
  return pred != 0;
}

__device__ __forceinline__ float ex2f(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float lg2f(float x) {
  float r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float rcpf(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float tf32_trunc(float x) { return __uint_as_float(__float_as_uint(x) & 0xffffe000u); }
__device__ __forceinline__ float tf32_rn(float x) {
  return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
}

// B elements at once, stage by stage: the MUFU results are consumed a whole stage (>= B instructions)
// after they were issued, so their latency is covered inside the warp instead of by warp switching.
template <bool MASK, int B>
__device__ __forceinline__ void epi_batch(const uint32_t* lr, float y, float vw, float* acc, float* g) {
  float e[B], den[B], inv[B], lg[B];
#pragma unroll
  for (int j = 0; j < B; ++j) e[j] = ex2f(-1.4426950408889634f * fabsf(__uint_as_float(lr[j])));
#pragma unroll
  for (int j = 0; j < B; ++j) den[j] = 1.f + e[j];
#pragma unroll
  for (int j = 0; j < B; ++j) inv[j] = rcpf(den[j]);
#pragma unroll
  for (int j = 0; j < B; ++j) lg[j] = lg2f(den[j]);
#pragma unroll
  for (int j = 0; j < B; ++j) {
    const float l = __uint_as_float(lr[j]);
    if (MASK) {
      acc[j] = fmaf(vw, fmaf(y, l, -fmaxf(l, 0.f)), acc[j]);
    } else {
      acc[j] = fmaf(y, l, acc[j]);
      acc[j] -= fmaxf(l, 0.f);
    }
  }
#pragma unroll
  for (int j = 0; j < B; ++j) {
    const float l = __uint_as_float(lr[j]);
    const float sg = (l >= 0.f) ? inv[j] : e[j] * inv[j];
    float gg = y - sg;
    if (MASK) {
      gg *= vw;
      acc[j] = fmaf(vw * lg[j], -0.6931471805599453f, acc[j]);
    } else {
      acc[j] = fmaf(lg[j], -0.6931471805599453f, acc[j]);
    }
    g[j] = tf32_rn(gg);
  }
}

template <bool SPLIT_X>
__global__ void __launch_bounds__(kThreads, 1)
glm_bernoulli_tc_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_y,
                        const float* __restrict__ W, const float* __restrict__ bvec, int64_t N, int P,
                        float* __restrict__ partials) {
  pdl_enter();   // lets glm_finish_kernel be resident (blocked in its griddepcontrol.wait) before this kernel ends
  using L = Layout<SPLIT_X>;
  constexpr int SX = L::kStagesX;
  constexpr int kStagesT = L::kStagesT;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* sm = smem_raw + (base - raw);
  const uint32_t bar0 = base + L::OFF_BAR;
  auto bar = [&](int i) { return bar0 + 8u * (uint32_t)i; };
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(sm + L::OFF_BAR + 8 * BAR_COUNT);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int slab = blockIdx.y;
  const int64_t ntiles = (N + kRows - 1) / kRows;
  // tiles handled by this CTA: blockIdx.x, blockIdx.x + gridDim.x, ...
  const int nt = (int)((ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x);

  // ---- one-time setup --------------------------------------------------------------------------------
  if (tid == 0) {
    for (int i = 0; i < kMaxStagesX; ++i) {
      mbar_init(bar(BAR_XFULL + i), 1);
      mbar_init(bar(BAR_XREADY + i), kSplitWarps * 32);
      mbar_init(bar(BAR_XEMPTY + i), 1);
    }
    for (int i = 0; i < 2; ++i) mbar_init(bar(BAR_LEMPTY + i), 1);
    for (int i = 0; i < kMaxStagesT; ++i) mbar_init(bar(BAR_TEMPTY + i), 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar(BAR_D1FULL + i), 1);
      mbar_init(bar(BAR_D1EMPTY + i), kEpiWarps * 32);
      mbar_init(bar(BAR_GFULL + i), kEpiWarps * 32);
      mbar_init(bar(BAR_GEMPTY + i), 1);
    }
    mbar_init(bar(BAR_DONE), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     base + L::OFF_BAR + 8 * BAR_COUNT),
                 "r"(kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  // weight / bias / ones tiles (generic-proxy writes, made visible to the MMA unit below)
  {
    float* whi = reinterpret_cast<float*>(sm + L::OFF_WHI);
    float* wlo = reinterpret_cast<float*>(sm + L::OFF_WLO);
    float* wb = reinterpret_cast<float*>(sm + L::OFF_WB);
    for (int e = tid; e < kP * kD; e += kThreads) {
      const int p = e >> 5, d = e & 31;
      const int gp = slab * kP + p;
      const float w = (gp < P) ? W[(int64_t)gp * kD + d] : 0.f;
      const float hi = tf32_trunc(w);
      const int off = p * 32 + ((((d >> 2) ^ (p & 7)) << 2) | (d & 3));   // float index, 128B swizzle
      whi[off] = hi;
      wlo[off] = w - hi;
      float bv = 0.f;
      if (d < 2 && bvec != nullptr && gp < P) {
        const float bb = bvec[gp];
        const float bh = tf32_trunc(bb);
        bv = (d == 0) ? bh : (bb - bh);
      }
      wb[off] = bv;
    }
    float* ones = reinterpret_cast<float*>(sm + L::OFF_ONES);
    for (int e = tid; e < 1024; e += kThreads) ones[e] = 1.f;
    // rows 32..39 of every X^T k-block are ones: GEMM 2 then yields db in columns 32..39 of D2
    for (int e = tid; e < kStagesT * 4 * 256; e += kThreads) {
      const int blk = e >> 8, w = e & 255;
      reinterpret_cast<float*>(sm + L::OFF_XT + blk * kXtBlock + kD * 128)[w] = 1.f;
    }
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    // =========================== TMA producer ===========================================================
    if (lane == 0) {
      for (int it = 0; it < nt; ++it) {
        const int sx = it % SX, ux = it / SX;
        const int64_t tile = blockIdx.x + (int64_t)it * gridDim.x;
        mbar_wait(bar(BAR_XEMPTY + sx), (ux & 1) ^ 1);
        mbar_expect_tx(bar(BAR_XFULL + sx), kXStage);
        tma_load_2d(base + L::OFF_X + sx * kTile, &map_x, 0, (int)(tile * kRows), bar(BAR_XFULL + sx));
        tma_load_1d(base + L::OFF_YX + sx * 512, &map_y, (int)(tile * kRows), bar(BAR_XFULL + sx));
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer =============================================================
    // The whole warp walks the loop (waits included); one elected lane issues the tcgen05 instructions.
    // Back-to-back MMAs into the SAME accumulator serialise on the tensor pipe's accumulate latency
    // (~100 cycles measured, far above the 20-35 cycle issue cost of these small shapes), so the issue
    // order interleaves five independent chains: GEMM 2 of tile j keeps one accumulator per 32-row
    // k-block (D2[0..3], summed once at the end of the kernel) and GEMM 1 of tile j+2 is threaded
    // through them.
    constexpr uint32_t id1 = idesc_tf32(128, 64);
    constexpr uint32_t id2 = idesc_tf32(64, 40);
    const uint64_t d_whi = desc_sw128(base + L::OFF_WHI);
    const uint64_t d_wlo = desc_sw128(base + L::OFF_WLO);
    const uint64_t d_wb = desc_sw128(base + L::OFF_WB);
    const uint64_t d_ones = make_desc(base + L::OFF_ONES, 128, 256, 0);
    const uint64_t d_x0 = desc_sw128(base + L::OFF_X);
    const uint64_t d_xl0 = desc_sw128(base + L::OFF_XLO);
    const uint64_t d_g0 = desc_sw128(base + L::OFF_G);
    const uint64_t d_xt0 = desc_sw128(base + L::OFF_XT);
    constexpr int kG1 = SPLIT_X ? 12 : 8;                        // data MMAs of GEMM 1
    constexpr int n_g1 = kG1 + 1;                                 // + the bias MMA (a zero tile without bias)

    // i-th MMA of GEMM 1 (i is a compile-time constant after unrolling); d1 / ax / al: accumulator and
    // operand descriptors of the tile
    auto g1_mma = [&](int i, uint32_t d1, uint64_t ax, uint64_t al) {
      if (i == kG1) {
        mma_tf32(d1, d_ones, d_wb, id1, 1u);
        return;
      }
      constexpr int per_k = kG1 / 4;
      const int k = i / per_k, part = i % per_k;
      if (part == 0) mma_tf32(d1, ax + (uint64_t)(k * 2), d_whi + (uint64_t)(k * 2), id1, k > 0 ? 1u : 0u);
      else if (part == 1) mma_tf32(d1, ax + (uint64_t)(k * 2), d_wlo + (uint64_t)(k * 2), id1, 1u);
      else mma_tf32(d1, al + (uint64_t)(k * 2), d_whi + (uint64_t)(k * 2), id1, 1u);
    };
    auto g1_commit = [&](int it) {
      tc_commit(bar(BAR_D1FULL + (it & 1)));
      tc_commit(bar(BAR_XEMPTY + it % SX));
      if (SPLIT_X) tc_commit(bar(BAR_LEMPTY + (it & 1)));
    };
    auto g1_wait = [&](int it) {
      mbar_wait(bar(BAR_XREADY + it % SX), (it / SX) & 1);
      mbar_wait(bar(BAR_D1EMPTY + (it & 1)), ((it >> 1) & 1) ^ 1);
    };
    // GEMM 2 of tile j, with GEMM 1 of tile j+2 threaded through when WITH_G1 (static issue order)
    auto batch = [&](int j, auto with_g1_tag) {
      constexpr bool WITH_G1 = decltype(with_g1_tag)::value;
      const int st = j % kStagesT, bj = j & 1;
      const int it = j + 2;
      const uint32_t d1 = tmem + kColD1 + (uint32_t)(it & 1) * 64u;
      const uint64_t ax = d_x0 + (uint64_t)((uint32_t)(it % SX) * (kTile >> 4));
      const uint64_t al = d_xl0 + (uint64_t)((uint32_t)(it & 1) * (kTile >> 4));
      // descriptor start addresses advance in 16-byte units: +2 per k-step of 8 floats inside a 32-float
      // k-block, + one block (kP*128 resp. kXtBlock bytes) per k-block
      const uint64_t da0 = d_g0 + (uint64_t)((uint32_t)bj * (kGBuf >> 4));
      const uint64_t db0 = d_xt0 + (uint64_t)((uint32_t)st * (kXtStage >> 4));
      const uint32_t acc0 = j > 0 ? 1u : 0u;
      int gi = 0;
#pragma unroll
      for (int sstep = 0; sstep < 4; ++sstep) {
#pragma unroll
        for (int kb = 0; kb < 4; ++kb) {
          const uint64_t da = da0 + (uint64_t)(kb * ((kP * 128) >> 4) + sstep * 2);
          const uint64_t db = db0 + (uint64_t)(kb * (kXtBlock >> 4) + sstep * 2);
          mma_tf32(tmem + kColD2 + (uint32_t)kb * 40u, da, db, id2, sstep > 0 ? 1u : acc0);
          if (WITH_G1) {
            const int upto = ((sstep * 4 + kb + 1) * n_g1 + 15) >> 4;   // spread evenly over the 16 slots
#pragma unroll
            for (int q = 0; q < 2; ++q)
              if (gi < upto) {
                g1_mma(gi, d1, ax, al);
                ++gi;
              }
          }
        }
      }
      if (WITH_G1) g1_commit(it);
      tc_commit(bar(BAR_TEMPTY + st));
      tc_commit(bar(BAR_GEMPTY + bj));
    };
    // prologue: GEMM 1 of the first two tiles
    for (int it = 0; it < 2 && it < nt; ++it) {
      g1_wait(it);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t d1 = tmem + kColD1 + (uint32_t)(it & 1) * 64u;
        const uint64_t ax = d_x0 + (uint64_t)((uint32_t)(it % SX) * (kTile >> 4));
        const uint64_t al = d_xl0 + (uint64_t)((uint32_t)(it & 1) * (kTile >> 4));
#pragma unroll
        for (int i = 0; i < n_g1; ++i) g1_mma(i, d1, ax, al);
        g1_commit(it);
      }
      __syncwarp();
    }
    for (int j = 0; j < nt; ++j) {
      const bool has_g1 = (j + 2 < nt);
      if (has_g1) g1_wait(j + 2);                      // long satisfied: split pass / epilogue of older tiles
      mbar_wait(bar(BAR_GFULL + (j & 1)), (j >> 1) & 1);   // epilogue of tile j has written g^T
      tc_fence_after();
      if (elect_one()) {
        if (has_g1) batch(j, cuda::std::true_type{});
        else batch(j, cuda::std::false_type{});
      }
      __syncwarp();
    }
    if (elect_one()) tc_commit(bar(BAR_DONE));
    __syncwarp();
  } else if (warp >= kSplitWarp0) {
    // =========================== split / transposition warps ===========================================
    const int r = tid - kSplitWarp0 * 32;           // row of the tile owned by this thread
    const int kb = r >> 5;                          // 32-row k-block of the transposed tile
    for (int it = 0; it < nt; ++it) {
      const int sx = it % SX, ux = it / SX;
      const int st = it % kStagesT, ut = it / kStagesT;
      mbar_wait(bar(BAR_XFULL + sx), ux & 1);
      mbar_wait(bar(BAR_TEMPTY + st), (ut & 1) ^ 1);           // GEMM 2 of tile it-3 released X^T[st]
      if (SPLIT_X) mbar_wait(bar(BAR_LEMPTY + (it & 1)), ((it >> 1) & 1) ^ 1);
      float4* xhi = reinterpret_cast<float4*>(sm + L::OFF_X + sx * kTile);
      float4* xlo = reinterpret_cast<float4*>(sm + L::OFF_XLO + (it & 1) * kTile);
      float* xt = reinterpret_cast<float*>(sm + L::OFF_XT + st * kXtStage + kb * kXtBlock);
      // y travels with the X^T stage (the epilogue reads it after the X stage may have been refilled)
      reinterpret_cast<float*>(sm + L::OFF_Y + st * 512)[r] =
          reinterpret_cast<const float*>(sm + L::OFF_YX + sx * 512)[r];
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const int idx = r * 8 + (c ^ (r & 7));      // 16-byte chunk holding d = 4c .. 4c+3 of row r
        const float4 v = xhi[idx];
        float x[4] = {v.x, v.y, v.z, v.w};
        if (SPLIT_X) {
          float4 h, l;
          h.x = tf32_trunc(v.x); h.y = tf32_trunc(v.y); h.z = tf32_trunc(v.z); h.w = tf32_trunc(v.w);
          l.x = v.x - h.x; l.y = v.y - h.y; l.z = v.z - h.z; l.w = v.w - h.w;
          xhi[idx] = h;
          xlo[idx] = l;
#pragma unroll
          for (int q = 0; q < 4; ++q) x[q] = tf32_rn(x[q]);
        } else {
#pragma unroll
          for (int q = 0; q < 4; ++q) x[q] = tf32_rn(x[q]);
          xhi[idx] = make_float4(x[0], x[1], x[2], x[3]);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int d = c * 4 + q;
          // X^T[d][n = r]: row d of k-block kb, 16-byte chunk (lane >> 2) ^ (d & 7), element lane & 3
          xt[d * 32 + (((((r & 31) >> 2) ^ (d & 7)) << 2) | (r & 3))] = x[q];
        }
      }
      fence_proxy_async();
      mbar_arrive(bar(BAR_XREADY + sx));
    }
  } else {
    // =========================== epilogue warps ========================================================
    const int ew = warp - kEpiWarp0;
    const int sub = warp & 3;                       // TMEM sub-partition this warp may access
    const int part = ew >> 2;                       // particles [kEpiCols*part, kEpiCols*(part+1))
    const int r = sub * 32 + lane;                  // row of the tile
    float acc[kEpiCols];
#pragma unroll
    for (int j = 0; j < kEpiCols; ++j) acc[j] = 0.f;
    // g^T[p][n = r]: k-block = sub, chunk (lane >> 2) ^ (p & 7); p & 7 == j & 7 because kEpiCols % 8 == 0
    uint32_t gofs[8];
#pragma unroll
    for (int j = 0; j < 8; ++j)
      gofs[j] = (uint32_t)sub * (kP * 128) + (uint32_t)part * (kEpiCols * 128) +
                ((((uint32_t)(lane >> 2) ^ (uint32_t)j) << 4) | ((uint32_t)(lane & 3) << 2));
    for (int it = 0; it < nt; ++it) {
      const int st = it % kStagesT;
      const int b = it & 1, v = it >> 1;
      const int64_t row0 = (blockIdx.x + (int64_t)it * gridDim.x) * kRows;
      // GEMM 2 of tile it-2 (long finished) has released g^T[b]
      mbar_wait(bar(BAR_GEMPTY + b), (v & 1) ^ 1);
      // d1_full implies the split pass of this tile ran (x_ready -> GEMM 1 -> d1_full): y[st] is in place
      mbar_wait(bar(BAR_D1FULL + b), v & 1);
      tc_fence_after();
      uint32_t lr[kEpiCols];
      const uint32_t taddr = tmem + ((uint32_t)(sub * 32) << 16) + kColD1 + (uint32_t)b * 64u +
                             (uint32_t)part * kEpiCols;
      static_assert(kEpiCols == 16, "the TMEM load below is the .x16 form");
      asm volatile(
          "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
          "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
          : "=r"(lr[0]), "=r"(lr[1]), "=r"(lr[2]), "=r"(lr[3]), "=r"(lr[4]), "=r"(lr[5]), "=r"(lr[6]),
            "=r"(lr[7]), "=r"(lr[8]), "=r"(lr[9]), "=r"(lr[10]), "=r"(lr[11]), "=r"(lr[12]), "=r"(lr[13]),
            "=r"(lr[14]), "=r"(lr[15])
          : "r"(taddr)
          : "memory");
      const float y = reinterpret_cast<const float*>(sm + L::OFF_Y + st * 512)[r];
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      tc_fence_before();
      mbar_arrive(bar(BAR_D1EMPTY + b));            // D1[b] is in registers now
      uint8_t* gt = sm + L::OFF_G + b * kGBuf;
      if (row0 + kRows <= N) {
#pragma unroll
        for (int j0 = 0; j0 < kEpiCols; j0 += 8) {
          float g[8];
          epi_batch<false, 8>(lr + j0, y, 1.f, acc + j0, g);
#pragma unroll
          for (int j = 0; j < 8; ++j) *reinterpret_cast<float*>(gt + gofs[j] + (j0 + j) * 128) = g[j];
        }
      } else {
        const float vw = (row0 + r < N) ? 1.f : 0.f;
#pragma unroll
        for (int j0 = 0; j0 < kEpiCols; j0 += 8) {
          float g[8];
          epi_batch<true, 8>(lr + j0, y, vw, acc + j0, g);
#pragma unroll
          for (int j = 0; j < 8; ++j) *reinterpret_cast<float*>(gt + gofs[j] + (j0 + j) * 128) = g[j];
        }
      }
      fence_proxy_async();
      mbar_arrive(bar(BAR_GFULL + b));
    }
    // ---- CTA results: dW, db from TMEM; lp sums through shared memory (fixed order) ---------------------
    mbar_wait(bar(BAR_DONE), 0);
    tc_fence_after();
    float* scratch = reinterpret_cast<float*>(sm + L::OFF_G);    // [128 rows][65]; GEMM 2 is finished with g^T
#pragma unroll
    for (int j = 0; j < kEpiCols; ++j) scratch[r * 65 + part * kEpiCols + j] = acc[j];
    asm volatile("bar.sync 1, %0;" ::"n"(kEpiWarps * 32) : "memory");
    float* out = partials + ((int64_t)blockIdx.x * P) * (kD + 2);
    if (ew < 4) {
      // M = 64 accumulators: row p lives in lane (p % 16) of sub-partition p / 16
      float dwf[32], dbf = 0.f;
#pragma unroll
      for (int d = 0; d < 32; ++d) dwf[d] = 0.f;
      const uint32_t t2 = tmem + ((uint32_t)(sub * 32) << 16);
#pragma unroll
      for (int kb = 0; kb < 4; ++kb) {
        uint32_t dw[32], dbv[8];
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
            "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
            : "=r"(dw[0]), "=r"(dw[1]), "=r"(dw[2]), "=r"(dw[3]), "=r"(dw[4]), "=r"(dw[5]), "=r"(dw[6]),
              "=r"(dw[7]), "=r"(dw[8]), "=r"(dw[9]), "=r"(dw[10]), "=r"(dw[11]), "=r"(dw[12]), "=r"(dw[13]),
              "=r"(dw[14]), "=r"(dw[15]), "=r"(dw[16]), "=r"(dw[17]), "=r"(dw[18]), "=r"(dw[19]), "=r"(dw[20]),
              "=r"(dw[21]), "=r"(dw[22]), "=r"(dw[23]), "=r"(dw[24]), "=r"(dw[25]), "=r"(dw[26]), "=r"(dw[27]),
              "=r"(dw[28]), "=r"(dw[29]), "=r"(dw[30]), "=r"(dw[31])
            : "r"(t2 + kColD2 + (uint32_t)kb * 40u)
            : "memory");
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                     : "=r"(dbv[0]), "=r"(dbv[1]), "=r"(dbv[2]), "=r"(dbv[3]), "=r"(dbv[4]), "=r"(dbv[5]),
                       "=r"(dbv[6]), "=r"(dbv[7])
                     : "r"(t2 + kColD2 + (uint32_t)kb * 40u + 32u)
                     : "memory");
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int d = 0; d < 32; ++d) dwf[d] += __uint_as_float(dw[d]);
        dbf += __uint_as_float(dbv[0]);
      }
      const int pl = sub * 16 + lane;               // valid for lane < 16
      const int gp = slab * kP + pl;
      if (lane < 16 && gp < P) {
        float s = 0.f;
        for (int n = 0; n < kRows; ++n) s += scratch[n * 65 + pl];
        float* o = out + (int64_t)gp * (kD + 2);
#pragma unroll
        for (int d = 0; d < kD; ++d) o[d] = dwf[d];
        o[kD] = dbf;
        o[kD + 1] = s;
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTmemCols) : "memory");
  }
}

// ---- host side -------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

}  // namespace tc

int glm_tc_grid_x(int64_t N) {
  const int64_t ntiles = (N + tc::kRows - 1) / tc::kRows;
  int64_t gx = kNumSMs;
  if (gx > ntiles) gx = ntiles;
  if (gx < 1) gx = 1;
  return (int)gx;
}

// returns 0 on success, a negative B2_ERR code when the TMA path cannot be used for these operands
int launch_glm_tc(const float* X, const float* y, const float* W, const float* b, int64_t N, int P,
                  float* partials, int gx, bool split_x, cudaStream_t s) {
  using namespace tc;
  EncodeTiledFn enc = encode_fn();
  if (enc == nullptr) return B2_ERR_LAUNCH;
  if (reinterpret_cast<uintptr_t>(X) % 16 != 0 || reinterpret_cast<uintptr_t>(y) % 16 != 0) return B2_ERR_BAD_SHAPE;
  if (N >= (int64_t)1 << 31) return B2_ERR_TOO_LARGE;
  CUtensorMap mx, my;
  {
    const cuuint64_t dims[2] = {(cuuint64_t)kD, (cuuint64_t)N};
    const cuuint64_t strides[1] = {(cuuint64_t)kD * 4};
    const cuuint32_t box[2] = {(cuuint32_t)kD, (cuuint32_t)kRows};
    const cuuint32_t estr[2] = {1, 1};
    if (enc(&mx, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(X), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return B2_ERR_LAUNCH;
  }
  {
    const cuuint64_t dims[1] = {(cuuint64_t)N};
    const cuuint64_t strides[1] = {0};
    const cuuint32_t box[1] = {(cuuint32_t)kRows};
    const cuuint32_t estr[1] = {1};
    if (enc(&my, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 1, const_cast<float*>(y), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
      return B2_ERR_LAUNCH;
  }
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(glm_bernoulli_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         (int)Layout<false>::kSmemBytes);
    cudaFuncSetAttribute(glm_bernoulli_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         (int)Layout<true>::kSmemBytes);
    attr_set = true;
  }
  dim3 grid((unsigned)gx, (unsigned)((P + kP - 1) / kP), 1);
  if (split_x)
    launch_pdl(glm_bernoulli_tc_kernel<true>, grid, dim3(kThreads), (size_t)Layout<true>::kSmemBytes, s, mx, my, W, b, N, P, partials);
  else
    launch_pdl(glm_bernoulli_tc_kernel<false>, grid, dim3(kThreads), (size_t)Layout<false>::kSmemBytes, s, mx, my, W, b, N, P, partials);
  return 0;
}

}  // namespace b2
