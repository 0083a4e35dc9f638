// amwg_kernels.cu -- libamwg_b200.so: the AMWG hot path of bayes.js as sm_100a CUDA + the C ABI of include/amwg.h.
//
// Reference path replaced (all under /root/reference/):
//   Sampler.sample / burn / step                     mcmc.js:985-1039
//   AmwgStepper.step (in-place substepper shuffle)    mcmc.js:886-892
//   MultidimComponentMetropolisStepper.step           mcmc.js:685-688  (nested_array_random_apply :244-263)
//   OnedimMetropolisStepper.step (+ batch adaptation) mcmc.js:517-553
//   BinaryStepper.step                                mcmc.js:753-767
//   rnorm / shuffle_array                             mcmc.js:43-54, 228-236
//   user log_post -> ld.*                             distributions.js (per opcode, amwg_ld.cuh)
//
// One thread per chain.  Per-chain state is SoA in HBM ([component][chain], coalesced); data[] is staged into
// shared memory once per CTA by 1-D bulk TMA (cp.async.bulk + mbarrier) and read as warp broadcasts.
// The current log-density is cached per chain: log_post is a pure function of the state, so the reference's
// first evaluation of every step (mcmc.js:524) returns exactly the value cached here (DESIGN.md "one eval per step").
// Compiled with --fmad=false; fma() is written out only inside the factorised plates.
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <cmath>
#include <string>
#include <vector>
#include <algorithm>
#include <sys/stat.h>
#include <unistd.h>
#include <cuda_runtime.h>
#include <math_constants.h>

#include "../../include/amwg.h"
#include "amwg_math.cuh"
#include "amwg_ld.cuh"
#include "amwg_tma.cuh"

namespace amwg {

constexpr int kMaxColumns = 32;
constexpr int kMaxParams = 255;      // substepper order: packed 4 bits per named parameter up to 16, a byte per entry in global memory beyond
constexpr int kMaxDim0 = 65535;      // top-level visit order of a multi-dim parameter: local bytes up to 256, 16-bit rows in global memory beyond
constexpr int kMaxDerived = 32;
constexpr int kStack = 32;          // operand stack of the interpreter; validate_model rejects programs that need more
#ifndef AMWG_THREADS
#define AMWG_THREADS 128
#endif
constexpr int kThreads = AMWG_THREADS;
#ifndef AMWG_SYNC_THREADS
#define AMWG_SYNC_THREADS 128
#endif
constexpr int kSyncThreads = AMWG_SYNC_THREADS;   // CTA size of the phase-synchronised sweep kernel
constexpr int kAdaptChunk = 64;
constexpr long long kHostChunkSweeps = 10;       // sample() to a host buffer: sweeps per launch, so copies overlap compute at this granularity
constexpr unsigned kSmemBudget = 200u * 1024u;   // bytes of dynamic shared memory we are willing to fill with data
constexpr unsigned kRingStageBytes = 16u * 1024u;   // TMA tile ring for columns that do not fit: 2 stages of 16 KB (six CTAs per SM beside it)
constexpr int kRingStages = 2;

// ---- model image as the kernels see it (passed by value) ------------------------------------------------------
struct ModelDev {
  const unsigned char* image;      // global: [code | consts | plates | params] packed, 16B aligned sections
  unsigned image_bytes;            // multiple of 16
  unsigned off_code, off_consts, off_plates, off_params;
  unsigned off_comp_prog, off_touch_off, off_touch_terms;   // dependency-aware evaluation tables (amwg_model.comp_prog ...), valid when n_terms > 0
  int n_terms;                     // > 0: per-chain term cache in use
  int n_block_params;              // multi-dim parameters stepped with one evaluation (amwg_model.block_params)
  int block_params[AMWG_MAX_BLOCK_PARAMS];
  unsigned off_tbc;                // image offset of term_block_comp [n_block_params][n_terms]
  int stat_prog;                   // >= 0: sweeps run with pre-evaluated plate statistics (amwg_model.stat_prog), by amwg_stat_sweep_kernel
  int stat_barriers;               // CTA barriers between the phases of a statistics sweep (instruction-cache locality)
  int scratch_smem_off;            // >= 0: byte offset in dynamic smem of the CTA's per-chain working set (amwg_stat_sweep_kernel), -1: global rows
  const double* col_global[kMaxColumns];
  unsigned col_bytes[kMaxColumns];     // padded to 16
  int col_smem_off[kMaxColumns];       // byte offset in dynamic smem, or -1: read from global/L2
  int n_columns, n_plates, n_params, D, n_derived;
  int logpost_prog, derived_prog;
  const unsigned char* adapting;   // [D] global, host-maintained (start/stop_adaptation)
  int phase_sync;                  // 1: every chain takes the same number of steps per sweep -> CTA-wide phase barriers are legal
  int ring_smem_off;               // byte offset of the 2-stage TMA tile ring in dynamic smem, -1: every column is resident
  int has_pois;                    // the model has a POIS_LOGLIN plate: stage_model fills ctx.exp_tab
  int n_variant_comps;             // binary components whose value selects the program (amwg_model.variant_*), 0 = single program
  int variant_comps[AMWG_MAX_VARIANT_COMPS];
  int variant_logpost[1 << AMWG_MAX_VARIANT_COMPS];
  int variant_derived[1 << AMWG_MAX_VARIANT_COMPS];
};

struct Ctx {                       // lives in shared memory
  const int* code;
  const double* consts;
  const amwg_plate* plates;
  const amwg_param* params;
  const int* comp_prog;            // per-component programs / touched-term lists (n_terms > 0)
  const int* touch_off;
  const int* touch_terms;
  const int* tbc;                  // term_block_comp
  const double* col[kMaxColumns];  // generic pointers (shared or global)
  unsigned col_saddr[kMaxColumns]; // 32-bit shared-window address, 0 when the column is served from global/L2
  double norm_c0;                  // -0.5 * Math.log(2 * Math.PI), evaluated once per CTA with the device's js_log
  unsigned ring_saddr;             // shared address of the TMA tile ring (0: none, or this kernel does not run CTA-uniformly)
  unsigned ring_uses[kRingStages]; // fills of each stage so far (mbarrier phase parity = fills & 1)
  unsigned long long ring_bar[kRingStages];
  double exp_tab[256];             // 2^(j/256) for the Poisson plate's exponential (filled only when the model has such a plate)
};

struct EvalStateBase {
  const double* st;   // state base + chain
  unsigned long long stride;
  int moved;          // component carrying the proposal, or -1
  double val;
  __device__ __forceinline__ EvalStateBase(const double* st_, unsigned long long stride_, int moved_, double val_)
      : st(st_), stride(stride_), moved(moved_), val(val_) {}
  __device__ __forceinline__ double comp(int c) const { return c == moved ? val : st[(unsigned long long)c * stride]; }
};
// CACHE = false: the model evaluates the full program at every step (no term cache; the hot configuration of the headline
// benchmark) -- the cache plumbing compiles away. CACHE = true: dependency-aware evaluation (amwg_model.comp_prog).
template <bool CACHE>
struct EvalStateT : EvalStateBase {
  using EvalStateBase::EvalStateBase;
  __device__ __forceinline__ void store(int, double) const {}
  __device__ __forceinline__ double cached(int) const { return 0.0; }
  __device__ __forceinline__ double cand(int) const { return 0.0; }
};
template <>
struct EvalStateT<true> : EvalStateBase {
  using EvalStateBase::EvalStateBase;
  double* tval = nullptr;     // term cache of this chain (base + chain), stride tstride; nullptr: not in use
  double* tcand = nullptr;
  unsigned long long tstride = 0;
  bool direct = false;        // STORE writes the cache itself (initial full evaluation) instead of the candidate slots
  const double* bprop = nullptr;   // block step: components [blk_lo, blk_hi) are read from the chain's proposal array
  int blk_lo = 0, blk_hi = 0;
  __device__ __forceinline__ double comp(int c) const {
    if (c >= blk_lo && c < blk_hi) return bprop[(unsigned long long)c * tstride];
    return c == moved ? val : st[(unsigned long long)c * stride];
  }
  __device__ __forceinline__ void store(int t, double v) const { if (tval) (direct ? tval : tcand)[(unsigned long long)t * tstride] = v; }
  __device__ __forceinline__ double cached(int t) const { return tval[(unsigned long long)t * tstride]; }
  __device__ __forceinline__ double cand(int t) const { return tcand[(unsigned long long)t * tstride]; }
};
using EvalState = EvalStateT<true>;

// Stage the model image and every data column that fits into shared memory; fill ctx. All threads call this.
__device__ __forceinline__ void stage_model(const ModelDev& m, unsigned char* smem, Ctx& ctx, unsigned long long* bar) {
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    for (int k = 0; k < kRingStages; ++k) { mbar_init(&ctx.ring_bar[k], 1); ctx.ring_uses[k] = 0; }
    // the ring needs every thread of the CTA to walk the same plates in the same order: uniform steps and a single program
    ctx.ring_saddr = (m.ring_smem_off >= 0 && m.phase_sync && m.n_variant_comps == 0) ? smem_u32(smem + m.ring_smem_off) : 0u;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned total = m.image_bytes;
    for (int k = 0; k < m.n_columns; ++k)
      if (m.col_smem_off[k] >= 0) total += m.col_bytes[k];
    mbar_expect_tx(bar, total);
    tma_bulk_g2s(smem, m.image, m.image_bytes, bar);
    for (int k = 0; k < m.n_columns; ++k)
      if (m.col_smem_off[k] >= 0) tma_bulk_g2s(smem + m.col_smem_off[k], m.col_global[k], m.col_bytes[k], bar);
    ctx.code = reinterpret_cast<const int*>(smem + m.off_code);
    ctx.consts = reinterpret_cast<const double*>(smem + m.off_consts);
    ctx.plates = reinterpret_cast<const amwg_plate*>(smem + m.off_plates);
    ctx.params = reinterpret_cast<const amwg_param*>(smem + m.off_params);
    ctx.comp_prog = reinterpret_cast<const int*>(smem + m.off_comp_prog);
    ctx.touch_off = reinterpret_cast<const int*>(smem + m.off_touch_off);
    ctx.touch_terms = reinterpret_cast<const int*>(smem + m.off_touch_terms);
    ctx.tbc = reinterpret_cast<const int*>(smem + m.off_tbc);
    for (int k = 0; k < m.n_columns; ++k) {
      bool in_smem = m.col_smem_off[k] >= 0;
      ctx.col[k] = in_smem ? reinterpret_cast<const double*>(smem + m.col_smem_off[k]) : m.col_global[k];
      ctx.col_saddr[k] = in_smem ? smem_u32(smem + m.col_smem_off[k]) : 0u;
    }
    ctx.norm_c0 = -0.5 * js_log(2 * AMWG_JS_PI);
  }
  if (m.has_pois) for (int j = threadIdx.x; j < 256; j += blockDim.x) ctx.exp_tab[j] = exp2((double)j * (1.0 / 256.0));
  __syncthreads();
  mbar_wait(bar, 0);
}

// ---- TMA tile ring: plates over a column that does not fit in shared memory ------------------------------------------------
// Legal only when the whole CTA walks the plate together (ModelDev.phase_sync: every chain takes the same steps per sweep and
// evaluates every step). Thread 0 is the producer: it arms a stage's mbarrier with the tile's byte count and issues the bulk
// copy (cp.async.bulk); all threads wait on the stage, accumulate their own chain from it (warp-broadcast LDS, same inner loop
// as the resident case), and a CTA barrier hands the stage back to the producer, which refills it with the tile after next.
__device__ __forceinline__ void ring_issue(Ctx& ctx, int stage, const void* src, unsigned bytes) {
  mbar_expect_tx(&ctx.ring_bar[stage], bytes);
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(ctx.ring_saddr + (unsigned)stage * kRingStageBytes),
               "l"(src), "r"(bytes), "r"(smem_u32(&ctx.ring_bar[stage]))
               : "memory");
}

__device__ __noinline__ double sum_sq_stream(Ctx& ctx, const double* __restrict__ gx, int n, double mean) {
  const int tile = (int)(kRingStageBytes >> 3);                       // doubles per stage
  const int ntiles = (n + tile - 1) / tile;
  __syncthreads();                                                    // earlier users of the ring are done; ring_uses is stable
  const unsigned u0 = ctx.ring_uses[0], u1 = ctx.ring_uses[1];
  if (threadIdx.x == 0) {
    for (int t = 0; t < 2 && t < ntiles; ++t) {
      int cnt = min(tile, n - t * tile);
      ring_issue(ctx, t, gx + (size_t)t * tile, (unsigned)((cnt * 8 + 15) & ~15));
    }
  }
  double S = 0.0;
  for (int t = 0; t < ntiles; ++t) {
    const int s = t & 1;
    mbar_wait(&ctx.ring_bar[s], ((s ? u1 : u0) + (unsigned)(t >> 1)) & 1u);
    const int cnt = min(tile, n - t * tile);
    const unsigned sa = ctx.ring_saddr + (unsigned)s * kRingStageBytes;
    const double* sp = reinterpret_cast<const double*>(__cvta_shared_to_generic((size_t)sa));
    S = S + sum_sq_dev(sp, sa, cnt, mean);
    __syncthreads();                                                  // every warp has consumed stage s
    if (threadIdx.x == 0 && t + 2 < ntiles) {
      int c2 = min(tile, n - (t + 2) * tile);
      ring_issue(ctx, s, gx + (size_t)(t + 2) * tile, (unsigned)((c2 * 8 + 15) & ~15));
    }
  }
  if (threadIdx.x == 0) { ctx.ring_uses[0] = u0 + (unsigned)((ntiles + 1) >> 1); ctx.ring_uses[1] = u1 + (unsigned)(ntiles >> 1); }
  return S;
}

__device__ __forceinline__ double norm_factorised(const Ctx& ctx, double n, double S, double sd) {
  return n * (ctx.norm_c0 - js_log(sd)) - S / (2 * sd * sd);
}

// S = sum_i (x_i - mean)^2 of a NORM_IID plate: the O(N) part
__device__ __forceinline__ double plate_sum_sq(const Ctx& ctx, int q, double mean) {
  const amwg_plate& pl = ctx.plates[q];
  int c = pl.col[0], off = pl.iparam[2];
  unsigned sa = ctx.col_saddr[c] ? ctx.col_saddr[c] + 8u * (unsigned)off : 0u;
  const double* gx = ctx.col[c] + off;
  if (sa == 0u && ctx.ring_saddr && (reinterpret_cast<unsigned long long>(gx) & 15ull) == 0)
    return sum_sq_stream(const_cast<Ctx&>(ctx), gx, pl.n, mean);       // column lives in HBM/L2: TMA tile ring
  return sum_sq_dev(gx, sa, pl.n, mean);
}

__device__ __noinline__ double plate_norm_iid(const Ctx& ctx, int q, double mean, double sd) {
  const double S = plate_sum_sq(ctx, q, mean);
  return norm_factorised(ctx, (double)ctx.plates[q].n, S, sd);
}
__device__ __noinline__ double plate_sum_sq_call(const Ctx& ctx, int q, double mean) { return plate_sum_sq(ctx, q, mean); }

// sum_i ld.bern(y_i, p): sequential, bit-faithful to distributions.js:228-230 (x*prob + (1-x)*(1-prob) is exact for x in {0,1}).
__device__ __noinline__ double plate_bern_iid(const Ctx& ctx, int q, double p, double lp) {
  const amwg_plate& pl = ctx.plates[q];
  double l1 = js_log(1.0 * p + (1 - 1.0) * (1 - p));
  double l0 = js_log(0.0 * p + (1 - 0.0) * (1 - p));
  const double* __restrict__ y = ctx.col[pl.col[0]] + pl.iparam[2];
  for (int i = 0; i < pl.n; ++i) {
    double yi = y[i];
    lp = lp + (yi == 1.0 ? l1 : (yi == 0.0 ? l0 : -CUDART_INF));
  }
  return lp;
}

// sum_i ld.norm(y_i, mu[g_i], sd) with points sorted by group; group j occupies [start[j], start[j+1]).
__device__ __noinline__ double plate_norm_grouped(const Ctx& ctx, int q, const EvalStateBase& es, double sd) {
  const amwg_plate& pl = ctx.plates[q];
  int c = pl.col[0], off = pl.iparam[2];
  const double* __restrict__ start = ctx.col[pl.col[1]];
  int J = pl.iparam[1], base = pl.iparam[0];
  double S = 0.0;
  for (int j = 0; j < J; ++j) {
    int a = (int)start[j] + off, b = (int)start[j + 1] + off;
    unsigned sa = ctx.col_saddr[c] ? ctx.col_saddr[c] + 8u * (unsigned)a : 0u;
    S = S + sum_sq_dev(ctx.col[c] + a, sa, b - a, es.comp(base + j));
  }
  return norm_factorised(ctx, (double)pl.n, S, sd);
}

// sum_i ld.pois(y_i, exp(eta_i)), eta_i = sum_k X_ik beta_k (k ascending, as the JS loop). With log(exp(eta)) -> eta the sum is
//     sum_i y_i eta_i  -  sum_i exp(eta_i)  -  sum_i lfactorial(y_i)
// whose first part is linear in beta, beta . (X^T y), and whose last part is a constant: the host precomputes X^T y and the
// lfactorial total (plate column [2], amwg.h), and the O(N) work per evaluation is the dot product and the exponential of every
// row -- the part that depends on beta non-linearly. (KS-level parity; real parameters only; `faithful` handles use the JS loop.)
// Rows are consumed from shared memory: a resident X directly, a larger one through the TMA tile ring.
//
// exp(): table-driven, 2^(j/256) (256 entries in shared memory, filled once per CTA) times a degree-4 polynomial on
// |r| <= ln2/512 (truncation 4e-17 relative): 9 fp64-pipe instructions including the accumulation, against ~25 for exp().
__device__ __noinline__ double exp_acc_slow(double x, double s) { return s + exp(x); }
// the constants whose low words are not zero come from the constant bank (an operand of DFMA, no instruction): as literals each
// costs two moves per use at the sweep kernels' register cap
__constant__ double kExpC[5] = {369.3299304675746 /* 256/ln2 */, -0.0027076061742263846 /* -HI */, 1.6409824502660487e-13 /* LO: ln2/256 = HI - LO */,
                                1.0 / 24.0, 1.0 / 6.0};
// |x| < 690, tested on the high word (integer pipe: the fp64 pipe is the bound); huge, infinite and NaN arguments fail
__device__ __forceinline__ bool exp_in_range(double x) { return ((unsigned)__double2hiint(x) & 0x7fffffffu) < 0x40859000u; }
__device__ __forceinline__ double exp_acc_fast(double x, unsigned tab_sa, double s) {   // s + exp(x) for x in range
  const double tm = fma(x, kExpC[0], 6755399441055744.0);          // x * 256/ln2 + 1.5*2^52: the integer lands in the low word
  const int ki = __double2loint(tm);
  const double kf = tm - 6755399441055744.0;
  double r = fma(kf, kExpC[1], x);                                 // Cody-Waite: ln2/256 = HI (32 bits) + LO
  r = fma(kf, kExpC[2], r);
  double p = fma(r, kExpC[3], kExpC[4]);
  p = fma(p, r, 0.5);
  p = fma(p, r, 1.0);
  p = fma(p, r, 1.0);
  const double T = lds_f64_sa(tab_sa + 8u * (unsigned)(ki & 255));
  const double Ts = __hiloint2double(__double2hiint(T) + ((ki >> 8) << 20), __double2loint(T));      // * 2^(ki >> 8)
  return fma(Ts, p, s);
}
__device__ __forceinline__ double exp_acc(double x, unsigned tab_sa, double s) {        // s + exp(x)
  if (!exp_in_range(x)) return exp_acc_slow(x, s);                 // the library function, out of line
  return exp_acc_fast(x, tab_sa, s);
}

template <int K>
__device__ __forceinline__ void pois_rows(unsigned xsa, int rows, const double (&beta)[K], unsigned tab_sa, double& s0, double& s1) {
  // four rows per iteration: four independent dependency chains per thread (a row is K dependent FMAs, then ~10 dependent
  // operations of the exponential; with three to six warps per scheduler that latency has to be covered inside the thread)
  int i = 0;
  if constexpr (K <= 8) {
    for (; i + 4 <= rows; i += 4, xsa += 32u * K) {
      double e0 = 0.0, e1 = 0.0, e2 = 0.0, e3 = 0.0;
      if constexpr ((K & 1) == 0) {
#pragma unroll
        for (int k = 0; k < K; k += 2) {
          const double2 a = lds_f64x2(xsa + 8u * k), b = lds_f64x2(xsa + 8u * (K + k)), c = lds_f64x2(xsa + 8u * (2 * K + k)), d = lds_f64x2(xsa + 8u * (3 * K + k));
          e0 = fma(a.x, beta[k], e0); e1 = fma(b.x, beta[k], e1); e2 = fma(c.x, beta[k], e2); e3 = fma(d.x, beta[k], e3);
          e0 = fma(a.y, beta[k + 1], e0); e1 = fma(b.y, beta[k + 1], e1); e2 = fma(c.y, beta[k + 1], e2); e3 = fma(d.y, beta[k + 1], e3);
        }
      } else {
#pragma unroll
        for (int k = 0; k < K; ++k) {
          e0 = fma(lds_f64_sa(xsa + 8u * k), beta[k], e0); e1 = fma(lds_f64_sa(xsa + 8u * (K + k)), beta[k], e1);
          e2 = fma(lds_f64_sa(xsa + 8u * (2 * K + k)), beta[k], e2); e3 = fma(lds_f64_sa(xsa + 8u * (3 * K + k)), beta[k], e3);
        }
      }
      s0 = exp_acc(e0, tab_sa, s0);
      s1 = exp_acc(e1, tab_sa, s1);
      s0 = exp_acc(e2, tab_sa, s0);
      s1 = exp_acc(e3, tab_sa, s1);
    }
  }
  for (; i + 2 <= rows; i += 2, xsa += 16u * K) {
    double e0 = 0.0, e1 = 0.0;
    if constexpr ((K & 1) == 0) {
#pragma unroll
      for (int k = 0; k < K; k += 2) {
        const double2 a = lds_f64x2(xsa + 8u * k), b = lds_f64x2(xsa + 8u * (K + k));
        e0 = fma(a.x, beta[k], e0); e1 = fma(b.x, beta[k], e1);
        e0 = fma(a.y, beta[k + 1], e0); e1 = fma(b.y, beta[k + 1], e1);
      }
    } else {
#pragma unroll
      for (int k = 0; k < K; ++k) { e0 = fma(lds_f64_sa(xsa + 8u * k), beta[k], e0); e1 = fma(lds_f64_sa(xsa + 8u * (K + k)), beta[k], e1); }
    }
    s0 = exp_acc(e0, tab_sa, s0);
    s1 = exp_acc(e1, tab_sa, s1);
  }
  if (i < rows) {
    double e0 = 0.0;
#pragma unroll
    for (int k = 0; k < K; ++k) e0 = fma(lds_f64_sa(xsa + 8u * k), beta[k], e0);
    s0 = exp_acc(e0, tab_sa, s0);
  }
}

// ---- the same rows on the fp64 tensor core (K = 8, a full warp) ------------------------------------------------------------------
// eta[row, chain] = sum_k X[row, k] beta[chain, k] is a GEMM: DMMA.8x8x4 (mma.sync m8n8k4 f64) forms it for 8 rows x 8 chains per
// instruction, so a warp's 32 chains take 8 DMMAs per 8 rows instead of 64 DFMAs per thread -- and, what matters more, ONE
// conflict-free LDS.128 per 8 rows instead of 32 broadcast LDS.128 (measured on this part, scripts/microbench/fp64_pipes.cu: a
// broadcast LDS.128 costs 2.5 cycles of the SM's shared-memory pipe and overlaps poorly with the fp64 pipe; the per-thread form
// spends as long on its loads as on its arithmetic. DMMA runs on the same fp64 pipe as DFMA at the same flop rate, 16 cycles each).
// Fragment layout (PTX ISA, m8n8k4 .f64): lane = 4 * g + j. A: row g, one k per step; B: column (chain) g of the tile, one k per
// step; C: row g, chains 2j and 2j + 1 of the tile. Lane j takes k = 2j (step 0) and k = 2j + 1 (step 1), adjacent in the row.
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
struct PoisMma {
  double bf[4][2];        // B fragments: tile t (chains 8t..8t+7 of the warp), k step s
  double acc[8];          // sum of exp(eta) over the rows this lane saw: tile t, chain 2j + e -> acc[2t + e]
  __device__ __forceinline__ void init(const double (&beta)[8]) {
    const unsigned lane = threadIdx.x & 31u, j = lane & 3u;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      bf[t][0] = bf[t][1] = 0.0;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const double w = __shfl_sync(0xffffffffu, beta[k], 8 * t + (int)(lane >> 2));
        if (k == (int)(2u * j)) bf[t][0] = w;
        if (k == (int)(2u * j + 1u)) bf[t][1] = w;
      }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.0;
  }
  // `rows` rows (row-major, 8 doubles per row) starting at shared address xsa, in groups of 8; in a last, partial group the lanes
  // of the missing rows compute on whatever follows in the tile and drop the result (a row of D depends on its own row of A only)
  __device__ __forceinline__ void rows8(unsigned xsa, int rows, unsigned tab_sa) {
    const unsigned lane = threadIdx.x & 31u;
    unsigned addr = xsa + (lane >> 2) * 64u + (lane & 3u) * 16u;
    int left = rows - (int)(lane >> 2);                         // this lane's row of the group exists while left > 0
    const int groups = (rows + 7) >> 3;
#pragma unroll 1
    for (int g = 0; g < groups; ++g, left -= 8, addr += 512u) {
      const double2 a = lds_f64x2(addr);
      const bool mine = left > 0;
#pragma unroll
      for (int t = 0; t < 4; t += 2) {
        double c00 = 0.0, c01 = 0.0, c10 = 0.0, c11 = 0.0;
        dmma884(c00, c01, a.x, bf[t][0]); dmma884(c10, c11, a.x, bf[t + 1][0]);
        dmma884(c00, c01, a.y, bf[t][1]); dmma884(c10, c11, a.y, bf[t + 1][1]);
        if (mine) {
          // one range test for the four values: no branches between their dependency chains, which then interleave
          if (exp_in_range(c00) && exp_in_range(c01) && exp_in_range(c10) && exp_in_range(c11)) {
            acc[2 * t] = exp_acc_fast(c00, tab_sa, acc[2 * t]); acc[2 * t + 1] = exp_acc_fast(c01, tab_sa, acc[2 * t + 1]);
            acc[2 * t + 2] = exp_acc_fast(c10, tab_sa, acc[2 * t + 2]); acc[2 * t + 3] = exp_acc_fast(c11, tab_sa, acc[2 * t + 3]);
          } else {
            acc[2 * t] = exp_acc(c00, tab_sa, acc[2 * t]); acc[2 * t + 1] = exp_acc(c01, tab_sa, acc[2 * t + 1]);
            acc[2 * t + 2] = exp_acc(c10, tab_sa, acc[2 * t + 2]); acc[2 * t + 3] = exp_acc(c11, tab_sa, acc[2 * t + 3]);
          }
        }
      }
    }
  }
  // this lane's chain: the eight row classes added up, then the total moved to the lane that owns the chain
  __device__ __forceinline__ double total() {
    const unsigned lane = threadIdx.x & 31u;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], 4);
      acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], 8);
      acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], 16);
    }
    double S = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const double w = __shfl_sync(0xffffffffu, acc[i], (int)((lane & 7u) >> 1));
      if (i == (int)(2u * (lane >> 3) + (lane & 1u))) S = w;
    }
    return S;
  }
};

// rows from global / L2 when neither residency nor the ring applies (models whose chains take different steps per sweep)
template <int K>
__device__ __forceinline__ void pois_rows_global(const double* __restrict__ X, int rows, const double (&beta)[K], unsigned tab_sa, double& s0, double& s1) {
  for (int i = 0; i < rows; ++i) {
    double e = 0.0;
#pragma unroll
    for (int k = 0; k < K; ++k) e = fma(X[(size_t)i * K + k], beta[k], e);
    if (i & 1) s1 = exp_acc(e, tab_sa, s1); else s0 = exp_acc(e, tab_sa, s0);
  }
}

template <int K>
__device__ __forceinline__ double pois_plate_k(Ctx& ctx, const amwg_plate& pl, const EvalStateBase& es) {
  const double* __restrict__ X = ctx.col[pl.col[1]];
  const double* __restrict__ stats = ctx.col[pl.col[2]];          // [X^T y (K) | sum lfactorial(y)]
  const int base = pl.iparam[0], n = pl.n;
  double beta[K];
  double lin = 0.0;
#pragma unroll
  for (int k = 0; k < K; ++k) { beta[k] = es.comp(base + k); lin = fma(stats[k], beta[k], lin); }
  const unsigned tab_sa = smem_u32(ctx.exp_tab);
  double s0 = 0.0, s1 = 0.0;
  const unsigned xres = ctx.col_saddr[pl.col[1]];
  if (xres) {
    pois_rows<K>(xres, n, beta, tab_sa, s0, s1);
  } else if (!ctx.ring_saddr || (reinterpret_cast<unsigned long long>(X) & 15ull)) {
    pois_rows_global<K>(X, n, beta, tab_sa, s0, s1);
  } else {
    const int R = (int)((kRingStageBytes / (unsigned)(K * 8)) & ~1u);          // rows per stage (even: every tile is a multiple of 16 B)
    const int ntiles = (n + R - 1) / R;
    __syncthreads();
    const unsigned u0 = ctx.ring_uses[0], u1 = ctx.ring_uses[1];
    if (threadIdx.x == 0)
      for (int t = 0; t < 2 && t < ntiles; ++t) {
        const int rows = min(R, n - t * R);
        ring_issue(ctx, t, X + (size_t)t * R * K, (unsigned)((rows * K * 8 + 15) & ~15));
      }
    // K = 8: the dot products on the tensor core (every thread of the CTA is here: whole warps)
    [[maybe_unused]] PoisMma mm;
    if constexpr (K == 8) mm.init(beta);
    for (int t = 0; t < ntiles; ++t) {
      const int st = t & 1;
      mbar_wait(&ctx.ring_bar[st], ((st ? u1 : u0) + (unsigned)(t >> 1)) & 1u);
      const unsigned tile_sa = ctx.ring_saddr + (unsigned)st * kRingStageBytes;
      const int rows = min(R, n - t * R);
      if constexpr (K == 8) {
        mm.rows8(tile_sa, rows, tab_sa);
      } else {
        pois_rows<K>(tile_sa, rows, beta, tab_sa, s0, s1);
      }
      __syncthreads();
      if (threadIdx.x == 0 && t + 2 < ntiles) {
        const int rows = min(R, n - (t + 2) * R);
        ring_issue(ctx, st, X + (size_t)(t + 2) * R * K, (unsigned)((rows * K * 8 + 15) & ~15));
      }
    }
    if (threadIdx.x == 0) { ctx.ring_uses[0] = u0 + (unsigned)((ntiles + 1) >> 1); ctx.ring_uses[1] = u1 + (unsigned)(ntiles >> 1); }
    if constexpr (K == 8) s0 = s0 + mm.total();
  }
  return (lin - (s0 + s1)) - stats[K];
}

__device__ __noinline__ double plate_pois_loglin(const Ctx& ctx_in, int q, const EvalStateBase& es) {
  Ctx& ctx = const_cast<Ctx&>(ctx_in);
  const amwg_plate& pl = ctx.plates[q];
  switch (pl.iparam[1]) {                                          // the coefficients live in registers: one instance per K
    case 1: return pois_plate_k<1>(ctx, pl, es);
    case 2: return pois_plate_k<2>(ctx, pl, es);
    case 3: return pois_plate_k<3>(ctx, pl, es);
    case 4: return pois_plate_k<4>(ctx, pl, es);
    case 5: return pois_plate_k<5>(ctx, pl, es);
    case 6: return pois_plate_k<6>(ctx, pl, es);
    case 7: return pois_plate_k<7>(ctx, pl, es);
    case 8: return pois_plate_k<8>(ctx, pl, es);
    case 10: return pois_plate_k<10>(ctx, pl, es);
    case 12: return pois_plate_k<12>(ctx, pl, es);
    case 16: return pois_plate_k<16>(ctx, pl, es);
    default: return CUDART_NAN;                                    // the host only emits the plate for these K (tracer._loglinear)
  }
}

// ---- the interpreter: ONE instance of the opcode switch in the whole library ---------------------------------------------
// Runs the program at `pc` to its END (encoding: include/amwg.h).  log_post programs accumulate into lp (ACC flag / PLATE /
// LOOP_END) and return it; expression programs (constant folding, ld.* evaluation) return the top of stack; derived programs
// STORE into der[].  The program and the constants are read through 32-bit shared-memory addresses; the top of the stack
// lives in a register, the rest in local memory (rarely touched: leaf operands are encoded inline).
__device__ __forceinline__ unsigned lds_u32(unsigned saddr) { unsigned v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(saddr)); return v; }
__device__ __forceinline__ double lds_f64(unsigned saddr) { double v; asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(saddr)); return v; }

// Rare opcodes (the ld.* that are not expanded into primitives by the host, lgamma & co, general pow) live out of line so
// that the interpreter's hot loop stays a few hundred instructions.
__device__ __noinline__ double cold_op(int op, double x, double y, double z, double t) {
  switch (op) {
    case AMWG_OP_POW: return pow(x, y);
    case AMWG_OP_LGAMMA: return ld_lgamma(x);
    case AMWG_OP_LFACTORIAL: return ld_lfactorial(x);
    case AMWG_OP_LCHOOSE: return ld_lchoose(x, y);
    case AMWG_OP_LBETA: return ld_lbeta(x, y);
    case AMWG_OP_LD_NORM: return ld_norm(x, y, z);
    case AMWG_OP_LD_UNIF: return ld_unif(x, y, z);
    case AMWG_OP_LD_BETA: return ld_beta(x, y, z);
    case AMWG_OP_LD_BERN: return ld_bern(x, y);
    case AMWG_OP_LD_POIS: return ld_pois(x, y);
    case AMWG_OP_LD_CAUCHY: return ld_cauchy(x, y, z);
    case AMWG_OP_LD_LAPLACE: return ld_laplace(x, y, z);
    case AMWG_OP_LD_GAMMA: return ld_gamma(x, y, z);
    case AMWG_OP_LD_INVGAMMA: return ld_invgamma(x, y, z);
    case AMWG_OP_LD_LNORM: return ld_lnorm(x, y, z);
    case AMWG_OP_LD_PARETO: return ld_pareto(x, y, z);
    case AMWG_OP_LD_T: return ld_t(x, y, z, t);
    case AMWG_OP_LD_WEIBULL: return ld_weibull(x, y, z);
    case AMWG_OP_LD_LOGIS: return ld_logis(x, y, z);
    case AMWG_OP_LD_EXP: return ld_exp(x, y);
    case AMWG_OP_LD_BINOM: return ld_binom(x, y, z);
    case AMWG_OP_LD_NBINOM: return ld_nbinom(x, y, z);
    case AMWG_OP_LD_HYPER: return ld_hyper(x, y, z, t);
    default: return CUDART_NAN;
  }
}

template <bool CACHE>
__device__ __noinline__ double run_program_t(unsigned code_sa, unsigned consts_sa, const Ctx& ctx, const EvalStateT<CACHE>& es, int pc,
                                             double* der, bool want_top) {
  double stk[kStack];
  double tos = 0.0;
  int sp = 0;
  double lp = 0.0;
  int loop_i = 0, loop_n = 0;
#define AMWG_NEXT() ((int)lds_u32(code_sa + 4u * (unsigned)(pc++)))
#define AMWG_POP(dst) do { dst = tos; --sp; tos = stk[sp]; } while (0)
#define AMWG_OPND(dst, mode)                                                               \
  do {                                                                                     \
    if ((mode) == AMWG_MODE_STACK) { AMWG_POP(dst); }                                      \
    else { int _ix = AMWG_NEXT(); dst = ((mode) == AMWG_MODE_CONST) ? lds_f64(consts_sa + 8u * (unsigned)_ix) : es.comp(_ix); } \
  } while (0)
  for (;;) {
    const unsigned w = (unsigned)AMWG_NEXT();
    const int op = w & 0xff;
    const bool acc = (w >> 16) & 1;
    const bool store = (w & AMWG_STORE_FLAG) != 0;
    const int a = (int)(w >> 18);
    // operands, last one first (the order inline words are laid out and stack operands are popped)
    double x = 0.0, y = 0.0, z = 0.0, t = 0.0;
    if (op != AMWG_OP_PLATE) {                          // plates fetch their own operands
      const int mD = (w >> 14) & 3, mC = (w >> 12) & 3, mB = (w >> 10) & 3, mA = (w >> 8) & 3;
      if (mD != AMWG_MODE_NONE) AMWG_OPND(t, mD);
      if (mC != AMWG_MODE_NONE) AMWG_OPND(z, mC);
      if (mB != AMWG_MODE_NONE) AMWG_OPND(y, mB);
      if (mA != AMWG_MODE_NONE) AMWG_OPND(x, mA);
    }
    double r = 0.0;
    bool has_r = true;
    switch (op) {
      case AMWG_OP_CONST: r = lds_f64(consts_sa + 8u * (unsigned)a); break;
      case AMWG_OP_COMP: r = es.comp(a); break;
      case AMWG_OP_DATA: r = ctx.col[a][AMWG_NEXT()]; break;
      case AMWG_OP_DATA_I: { int off = AMWG_NEXT(); int stride = AMWG_NEXT(); r = ctx.col[a][off + stride * loop_i]; break; }
      case AMWG_OP_COMP_I: {
        int off = AMWG_NEXT(); int stride = AMWG_NEXT(); int base = AMWG_NEXT();
        r = es.comp(base + (int)ctx.col[a][off + stride * loop_i]);
        break;
      }
      case AMWG_OP_ADD: r = x + y; break;
      case AMWG_OP_SUB: r = x - y; break;
      case AMWG_OP_MUL: r = x * y; break;
      case AMWG_OP_DIV: r = x / y; break;
      case AMWG_OP_NEG: r = -x; break;
      case AMWG_OP_LOG: r = js_log(x); break;
      case AMWG_OP_EXP: r = js_exp(x); break;
      case AMWG_OP_SQRT: r = sqrt(x); break;
      case AMWG_OP_ABS: r = fabs(x); break;
      case AMWG_OP_POW: r = (y == 2.0) ? x * x : cold_op(op, x, y, z, t); break;
      case AMWG_OP_LT: r = x < y ? 1.0 : 0.0; break;
      case AMWG_OP_LE: r = x <= y ? 1.0 : 0.0; break;
      case AMWG_OP_GT: r = x > y ? 1.0 : 0.0; break;
      case AMWG_OP_GE: r = x >= y ? 1.0 : 0.0; break;
      case AMWG_OP_EQ: r = x == y ? 1.0 : 0.0; break;
      case AMWG_OP_NE: r = x != y ? 1.0 : 0.0; break;
      case AMWG_OP_AND: r = (x != 0.0 && y != 0.0) ? 1.0 : 0.0; break;
      case AMWG_OP_OR: r = (x != 0.0 || y != 0.0) ? 1.0 : 0.0; break;
      case AMWG_OP_NOT: r = x != 0.0 ? 0.0 : 1.0; break;
      case AMWG_OP_SELECT: r = x != 0.0 ? y : z; break;
      case AMWG_OP_NORM_K: { double d = x - y; r = z - (d * d) / t; break; }
      case AMWG_OP_UNIF_K: r = (x < y || x > z) ? -CUDART_INF : t; break;
      case AMWG_OP_BETA_K: r = (x > 1 || x < 0) ? -CUDART_INF : (y * js_log(x) + z * js_log(1 - x)) - t; break;
      case AMWG_OP_PLATE_SS: {               // the plate's statistic at `mean`; also kept in its cache slot (amwg.h stat_prog)
        const int slot = AMWG_NEXT();
        r = plate_sum_sq_call(ctx, a, x);
        es.store(slot, r);
        break;
      }
      case AMWG_OP_NORM_SS: r = norm_factorised(ctx, (double)ctx.plates[a].n, x, y); break;
      case AMWG_OP_CACHED: r = es.cached(a); break;
      case AMWG_OP_CAND: r = es.cand(a); break;
      case AMWG_OP_ACC: { double v; AMWG_POP(v); lp = lp + v; has_r = false; break; }
      case AMWG_OP_ACC_RANGE: {              // terms that do not read the moved component: their cached values, one by one, in order
        const int cnt = AMWG_NEXT();
        int k = 0;
        for (; k + 8 <= cnt; k += 8) {       // the loads first (independent, eight in flight), then the adds in order
          const double v0 = es.cached(a + k), v1 = es.cached(a + k + 1), v2 = es.cached(a + k + 2), v3 = es.cached(a + k + 3);
          const double v4 = es.cached(a + k + 4), v5 = es.cached(a + k + 5), v6 = es.cached(a + k + 6), v7 = es.cached(a + k + 7);
          lp = lp + v0; lp = lp + v1; lp = lp + v2; lp = lp + v3; lp = lp + v4; lp = lp + v5; lp = lp + v6; lp = lp + v7;
        }
        for (; k < cnt; ++k) lp = lp + es.cached(a + k);
        has_r = false;
        break;
      }
      case AMWG_OP_PLATE: {
        has_r = false;
        const int kind = ctx.plates[a].kind;
        double v = 0.0;
        if (kind == AMWG_PLATE_NORM_IID) {
          double mean, sd; AMWG_OPND(sd, (w >> 10) & 3); AMWG_OPND(mean, (w >> 8) & 3);
          v = plate_norm_iid(ctx, a, mean, sd);
          lp = lp + v;
        } else if (kind == AMWG_PLATE_BERN_IID) {
          double p; AMWG_OPND(p, (w >> 8) & 3);
          lp = plate_bern_iid(ctx, a, p, lp);
        } else if (kind == AMWG_PLATE_NORM_GROUPED) {
          double sd; AMWG_OPND(sd, (w >> 8) & 3);
          v = plate_norm_grouped(ctx, a, es, sd);
          lp = lp + v;
        } else if (kind == AMWG_PLATE_POIS_LOGLIN) {
          v = plate_pois_loglin(ctx, a, es);
          lp = lp + v;
        }
        if (store) { const int t = AMWG_NEXT(); es.store(t, v); }
        break;
      }
      case AMWG_OP_LOOP_BEGIN: {
        int skip_to = AMWG_NEXT();
        loop_i = 0; loop_n = ctx.plates[a].n;
        if (loop_n <= 0) pc = skip_to;
        has_r = false;
        break;
      }
      case AMWG_OP_LOOP_END: {
        int body = AMWG_NEXT();
        double v; AMWG_POP(v);
        lp = lp + v;
        if (++loop_i < loop_n) pc = body; else loop_i = 0;
        has_r = false;
        break;
      }
      case AMWG_OP_STORE: { double v; AMWG_POP(v); der[a] = v; has_r = false; break; }
      case AMWG_OP_END: return (want_top && sp > 0) ? tos : lp;
      default: r = cold_op(op, x, y, z, t); break;
    }
    if (has_r) {
      if (acc) {
        lp = lp + r;
        if (store) { const int t = AMWG_NEXT(); es.store(t, r); }
      } else { stk[sp] = tos; ++sp; tos = r; }
    }
  }
#undef AMWG_NEXT
#undef AMWG_POP
#undef AMWG_OPND
}

// which recorded configuration of the binary components applies to this evaluation state (0 when the model has one program)
__device__ __forceinline__ double run_program(unsigned code_sa, unsigned consts_sa, const Ctx& ctx, const EvalState& es, int pc, double* der, bool want_top) {
  return run_program_t<true>(code_sa, consts_sa, ctx, es, pc, der, want_top);
}
__device__ __forceinline__ int variant_of(const ModelDev& m, const EvalStateBase& es) {
  int v = 0;
  for (int k = 0; k < m.n_variant_comps; ++k) v |= (es.comp(m.variant_comps[k]) != 0.0) ? (1 << k) : 0;
  return v;
}
__device__ __forceinline__ int logpost_pc(const ModelDev& m, const EvalStateBase& es) {
  return m.n_variant_comps ? m.variant_logpost[variant_of(m, es)] : m.logpost_prog;
}
__device__ __forceinline__ int derived_pc(const ModelDev& m, const EvalStateBase& es) {
  return m.n_variant_comps ? m.variant_derived[variant_of(m, es)] : m.derived_prog;
}
template <bool CACHE>
__device__ __forceinline__ double eval_logpost(const Ctx& ctx, const EvalStateT<CACHE>& es, int pc) {
  return run_program_t<CACHE>(smem_u32(ctx.code), smem_u32(ctx.consts), ctx, es, pc, nullptr, false);
}
__device__ __forceinline__ double run_ctx(const Ctx& ctx, const EvalState& es, int pc, double* der, bool want_top) {
  return run_program(smem_u32(ctx.code), smem_u32(ctx.consts), ctx, es, pc, der, want_top);
}

// ---- K0: constant folding (amwg_model.fold_*), then place every chain at init and evaluate log_post once (mcmc.js:954-963) ---
__global__ void amwg_fold_kernel(ModelDev m, int n_fold, const int* __restrict__ fold_prog, const int* __restrict__ fold_dst) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ Ctx ctx;
  __shared__ __align__(8) unsigned long long bar;
  stage_model(m, smem, ctx, &bar);
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  double* consts_global = reinterpret_cast<double*>(const_cast<unsigned char*>(m.image) + m.off_consts);
  double* consts_smem = const_cast<double*>(ctx.consts);
  EvalState es{nullptr, 0, -1, 0.0};
  for (int k = 0; k < n_fold; ++k) {          // in order: later folds may use earlier ones
    double v = run_ctx(ctx, es, fold_prog[k], nullptr, true);
    consts_global[fold_dst[k]] = v;
    consts_smem[fold_dst[k]] = v;
  }
}

__global__ void __launch_bounds__(kThreads) amwg_init_kernel(ModelDev m, ChainArrays a, const double* __restrict__ init,
                                                            const double* __restrict__ pls0) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ Ctx ctx;
  __shared__ __align__(8) unsigned long long bar;
  stage_model(m, smem, ctx, &bar);
  const unsigned long long tid = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = tid < a.C;
  if (!valid && !ctx.ring_saddr) return;
  const unsigned long long chain = valid ? tid : a.C - 1;              // shadow threads keep a streamed plate CTA-uniform
  if (valid) {
    for (int c = 0; c < m.D; ++c) {
      a.state[(unsigned long long)c * a.C + chain] = init[c];
      a.pls[(unsigned long long)c * a.C + chain] = pls0[c];
      a.psd[(unsigned long long)c * a.C + chain] = js_exp(pls0[c]);
      a.acc[(unsigned long long)c * a.C + chain] = 0;
    }
    unsigned long long perm = 0;
    if (a.perm_ext) for (int p = 0; p < m.n_params; ++p) a.perm_ext[(unsigned long long)p * a.C + chain] = (unsigned char)p;
    else for (int p = 0; p < m.n_params; ++p) perm |= (unsigned long long)p << (4 * p);
    a.perm[chain] = perm;
    a.rng_n[chain] = 0;
  }
  // every chain starts from the same `init`: evaluate from it directly (a shadow thread must not race with the owner's writes)
  EvalState es{init, 1, -1, 0.0};
  if (m.n_terms > 0 && valid) { es.tval = a.tval + chain; es.tcand = a.tcand + chain; es.tstride = a.C; es.direct = true; }
  double lp0 = eval_logpost(ctx, es, logpost_pc(m, es));
  if (valid) a.curr_lp[chain] = lp0;
}

// log_post at the chains' CURRENT state, evaluated afresh with the full program (nothing is stored): what sampler.log_post()
// returns for handles whose sweep kernel does not carry the value along (the run-time specialised sweep works on differences).
__global__ void __launch_bounds__(kThreads) amwg_relp_kernel(ModelDev m, ChainArrays a) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ Ctx ctx;
  __shared__ __align__(8) unsigned long long bar;
  stage_model(m, smem, ctx, &bar);
  const unsigned long long tid = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = tid < a.C;
  if (!valid && !ctx.ring_saddr) return;
  const unsigned long long chain = valid ? tid : a.C - 1;              // shadow threads keep a streamed plate CTA-uniform
  EvalState es{a.state + chain, a.C, -1, 0.0};
  const double lp = eval_logpost(ctx, es, logpost_pc(m, es));
  if (valid) a.curr_lp[chain] = lp;
}

// ---- K1: n_sweeps Sampler.step()s per chain, samples recorded before each kept sweep --------------------------------
// Phase synchronisation: when every chain takes the same number of steps per sweep (all parameters scalar, or a single
// parameter), the CTA runs propose / evaluate / accept in lock step (__syncthreads between phases). Warps that share a
// scheduler then execute the same few hundred instructions together (instruction-cache hits instead of every warp streaming
// the whole sweep body past the others), while the CTAs resident on one SM drift apart and overlap their fp64 loops with each
// other's bookkeeping. Threads past the last chain shadow chain C-1 and write nothing, so they can take part in the barriers.
#ifndef AMWG_MINBLOCKS
#define AMWG_MINBLOCKS 7
#endif
template <bool CACHE>
__global__ void __launch_bounds__(kSyncThreads, AMWG_MINBLOCKS) amwg_sweep_kernel(ModelDev m, ChainArrays a, SweepArgs sa) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ Ctx ctx;
  __shared__ __align__(8) unsigned long long bar;
  stage_model(m, smem, ctx, &bar);

  const unsigned long long C = a.C;
  const unsigned long long tid = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = tid < C;
  const bool sync = m.phase_sync != 0;
  if (!valid && !sync) return;
  const unsigned long long chain = valid ? tid : C - 1;
  double* st = a.state + chain;
  const unsigned long long gchain = a.first_chain + chain;      // global chain id: the Philox counter's upper words

  RandomStream g;
  g.init(a.rng_n[chain]);
  unsigned long long perm = a.perm[chain];
  double curr = a.curr_lp[chain];
  const int P = m.n_params;
  unsigned char order[kLocalOrder];

  // `i % thin === 0` (mcmc.js:1021) without a 64-bit division per sweep: position inside the thinning interval and next row
  long long rec_phase = sa.record ? sa.sample_i0 % sa.thin : 0;
  long long row = sa.record ? (sa.sample_i0 + sa.thin - 1) / sa.thin : 0;
  for (long long s = 0; s < sa.n_sweeps; ++s) {
    // -- Sampler.sample: record the state BEFORE stepping (mcmc.js:1021-1027)
    if (sa.record) {
      const bool rec_now = rec_phase == 0;
      if (++rec_phase == sa.thin) rec_phase = 0;
      if (rec_now && valid) {
        double der[kMaxDerived];
        bool have_der = false;
        for (int j = 0; j < sa.n_monitor; ++j) {
          int e = sa.monitor[j];
          double v;
          if (e < m.D) {
            v = st[(unsigned long long)e * C];
          } else {
            if (!have_der) { EvalState es{st, C, -1, 0.0}; run_ctx(ctx, es, derived_pc(m, es), der, false); have_der = true; }
            v = der[e - m.D];
          }
          sa.out[((unsigned long long)row * sa.n_monitor + j) * C + chain] = v;
        }
      }
      if (rec_now) ++row;
    }
    // -- AmwgStepper.step: shuffle_array(this.substeppers), in place (mcmc.js:887, 228-236)
    for (int i = P - 1; i > 0; --i) {
      int j = (int)floor(g.next(a.seed, gchain) * (i + 1));
      perm_swap(a, perm, chain, i, j, valid);
    }
    for (int slot = 0; slot < P; ++slot) {
      const amwg_param& pa = ctx.params[perm_get(a, perm, chain, slot)];   // read from shared memory where needed: not kept in registers
      const int n_rounds = pa.n_comp;
      const int inner = pa.n_comp / pa.dim0;
      if (pa.n_comp > 1) {
        // nested_array_random_apply: fresh identity, shuffled, top level only (mcmc.js:246-252)
        for (int i = 0; i < pa.dim0; ++i) ord_set(a, order, chain, pa.dim0, i, i, valid);
        for (int i = pa.dim0 - 1; i > 0; --i) {
          int j = (int)floor(g.next(a.seed, gchain) * (i + 1));
          const int t = ord_get(a, order, chain, pa.dim0, i);
          ord_set(a, order, chain, pa.dim0, i, ord_get(a, order, chain, pa.dim0, j), valid);
          ord_set(a, order, chain, pa.dim0, j, t, valid);
        }
      }
      int block_slot = -1;
      if constexpr (CACHE) {
        const int pidx = perm_get(a, perm, chain, slot);
        for (int k = 0; k < m.n_block_params; ++k) if (m.block_params[k] == pidx) block_slot = k;
      }
      // A block-stepped parameter (amwg.h block_params) takes ONE round for all its components; otherwise one round per component.
      // Propose / evaluate / accept share their barrier points and the evaluation call site between the two kinds of round, so
      // that lanes of one warp that drew different parameters for this slot still execute the same barriers (bar.sync is aligned)
      // and, with the tile ring, walk the plates of the full program together.
      const bool is_block = CACHE && block_slot >= 0;
      const int rounds = is_block ? 1 : n_rounds;
      for (int r = 0; r < rounds; ++r) {
        // ---- phase 1: propose
        if (sync) __syncthreads();
        int c = pa.comp_offset;
        if (!is_block && pa.n_comp > 1) c += ord_get(a, order, chain, pa.dim0, r / inner) * inner + (r % inner);
        const unsigned long long ci = (unsigned long long)c * C;
        double cur = 0.0, prop = 0.0;
        bool need;
        if (is_block) {
          // proposals and accept uniforms of every component, in the chain's visiting order: the Math.random() calls of
          // mcmc.js:519-528 in their original order (a uniform is only drawn for an in-bounds proposal)
          for (int q = 0; q < n_rounds; ++q) {
            const int cq = pa.comp_offset + ord_get(a, order, chain, pa.dim0, q / inner) * inner + (q % inner);
            const unsigned long long cqi = (unsigned long long)cq * C + chain;
            const double curq = a.state[cqi];
            double pq = js_rnorm(g, a.seed, gchain, curq, a.psd[cqi]);
            if (pa.type == AMWG_INT) pq = js_round(pq);
            const bool inb = !(pq < pa.lower || pq > pa.upper);
            const double coin = inb ? g.next(a.seed, gchain) : -1.0;
            if (valid) { a.bprop[cqi] = inb ? pq : curq; a.bcoin[cqi] = coin; }
          }
          need = true;
        } else {
          cur = st[ci];
          if (pa.type == AMWG_BINARY) {
            prop = (cur == 0.0) ? 1.0 : 0.0;               // the state value whose log_post is not cached
            need = true;
          } else {
            // generate_proposal (mcmc.js:519, 577-579 / 596-598) and the bounds check (:520)
            prop = js_rnorm(g, a.seed, gchain, cur, a.psd[ci + chain]);
            if (pa.type == AMWG_INT) prop = js_round(prop);
            need = !(prop < pa.lower || prop > pa.upper);
          }
        }
        // ---- phase 2: evaluate log_post at the proposal (the O(N) likelihood sum)
        if (sync) __syncthreads(); else __syncwarp(__activemask());
        double lp_new = 0.0;
        if (need || ctx.ring_saddr) {                     // with the tile ring the plate is a CTA-wide collective: nobody may skip it
          EvalStateT<CACHE> es{st, C, is_block ? -1 : c, need ? prop : cur};
          int pc;
          if constexpr (CACHE) {
            es.tval = a.tval + chain; es.tcand = a.tcand + chain; es.tstride = C;
            if (is_block) {                               // the whole block at its proposals: every term's candidate value -> tcand
              es.bprop = a.bprop + chain; es.blk_lo = pa.comp_offset; es.blk_hi = pa.comp_offset + pa.n_comp;
              pc = m.logpost_prog;
            } else {
              // dependency-aware: only the terms that read component c are recomputed; with the tile ring every lane must walk
              // the same plates in the same order, so everybody runs the full program
              pc = ctx.ring_saddr ? m.logpost_prog : ctx.comp_prog[c];
            }
          } else {
            pc = logpost_pc(m, es);
          }
          lp_new = eval_logpost<CACHE>(ctx, es, pc);
        }
        // ---- phase 3: accept / reject
        if (sync) __syncthreads();
        if (is_block) {
          // one component at a time, in visiting order: log_post of "component c at its proposal" is the in-order sum of the cached
          // terms with c's terms taken from the candidates -- exactly what the per-component program adds
          const int* tbc = ctx.tbc + block_slot * m.n_terms;
          for (int q = 0; q < n_rounds; ++q) {
            const int cq = pa.comp_offset + ord_get(a, order, chain, pa.dim0, q / inner) * inner + (q % inner);
            const unsigned long long cqi = (unsigned long long)cq * C + chain;
            const double coin = a.bcoin[cqi];
            if (coin < 0.0) continue;                        // out of bounds: rejected without evaluation (mcmc.js:520-522)
            double lpq = 0.0;
            int t = 0;
            for (; t + 4 <= m.n_terms; t += 4) {             // loads first (four in flight), adds in order
              double v[4];
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                const unsigned long long ti = (unsigned long long)(t + u) * C + chain;
                v[u] = (tbc[t + u] == cq ? a.tcand : a.tval)[ti];
              }
              lpq = lpq + v[0]; lpq = lpq + v[1]; lpq = lpq + v[2]; lpq = lpq + v[3];
            }
            for (; t < m.n_terms; ++t) {
              const unsigned long long ti = (unsigned long long)t * C + chain;
              lpq = lpq + (tbc[t] == cq ? a.tcand[ti] : a.tval[ti]);
            }
            const double accept_prob = js_exp(lpq - curr);
            if (accept_prob > coin) {
              curr = lpq;
              if (valid) {
                a.state[cqi] = a.bprop[cqi];
                if (m.adapting[cq]) a.acc[cqi] += 1;
                for (int k = ctx.touch_off[cq]; k < ctx.touch_off[cq + 1]; ++k) {
                  const unsigned long long ti = (unsigned long long)ctx.touch_terms[k] * C + chain;
                  a.tval[ti] = a.tcand[ti];
                }
              }
            }
          }
        } else if (pa.type == AMWG_BINARY) {
          // BinaryStepper.step (mcmc.js:753-767); log_post of the current value is the cached one
          double z0raw = (cur == 0.0) ? curr : lp_new, z1raw = (cur == 0.0) ? lp_new : curr;
          double mx = js_max(z0raw, z1raw);
          double z0 = z0raw - mx, z1 = z1raw - mx;
          double zero_prob = js_exp(z0 - js_log(js_exp(z0) + js_exp(z1)));
          bool zero = g.next(a.seed, gchain) < zero_prob;
          const bool changed = zero != (cur == 0.0);
          if (valid) st[ci] = zero ? 0.0 : 1.0;
          curr = zero ? z0raw : z1raw;
          if (CACHE && changed && valid)
            for (int k = ctx.touch_off[c]; k < ctx.touch_off[c + 1]; ++k) {
              const unsigned long long ti = (unsigned long long)ctx.touch_terms[k] * C + chain;
              a.tval[ti] = a.tcand[ti];
            }
        } else if (need) {
          // Metropolis accept (mcmc.js:527-534): strict >, NaN rejects
          double accept_prob = js_exp(lp_new - curr);
          if (accept_prob > g.next(a.seed, gchain)) {
            curr = lp_new;
            if (valid) {
              st[ci] = prop;
              if (m.adapting[c]) a.acc[ci + chain] += 1;
              if (CACHE)                                  // commit the recomputed terms to the chain's term cache
                for (int k = ctx.touch_off[c]; k < ctx.touch_off[c + 1]; ++k) {
                  const unsigned long long ti = (unsigned long long)ctx.touch_terms[k] * C + chain;
                  a.tval[ti] = a.tcand[ti];
                }
            }
          }
        }
      }
    }
  }
  if (valid) {
    a.rng_n[chain] = g.n;
    a.perm[chain] = perm;
    a.curr_lp[chain] = curr;
  }
}

// ---- K1s: sweeps with pre-evaluated plate statistics (amwg_model.stat_prog) ---------------------------------------------
// Per sweep: (a) every step's proposal and accept uniform, drawn in the chain's visiting order -- the Math.random() calls of
// mcmc.js:887/246-252 (shuffles) and :519-528 (rnorm trials, one uniform per in-bounds proposal) in their original order, none of
// which depends on a log_post value; (b) ONE pass over the data: stat_prog evaluates every plate's S at the proposals (all
// threads of the CTA together: resident columns by broadcast LDS, larger ones through the TMA tile ring); (c) the steps in
// visiting order, each an O(1) evaluation of comp_prog[c] from cached terms and statistics, accept/reject and commit as
// mcmc.js:527-534. Same values, sums and uniforms as stepping with the full program -> the same draws, bit for bit.
//
// Per-chain working set: rows [tval n_terms | tcand n_terms | bprop D | bcoin D | state D] of doubles + vseq D of u16. When it
// fits beside the model and the data (scratch_smem_off >= 0: small models, e.g. the headline one) it lives in SHARED memory for
// the whole launch, one column per thread (row stride = CTA size, conflict-free): state and term cache are read from HBM once
// per launch and written back once, the per-sweep temporaries never leave the SM. Otherwise the rows are the global arrays
// (row stride = C), which amwg_create lays out back to back in the same order.
__global__ void __launch_bounds__(kSyncThreads, AMWG_MINBLOCKS) amwg_stat_sweep_kernel(ModelDev m, ChainArrays a, SweepArgs sa) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ Ctx ctx;
  __shared__ __align__(8) unsigned long long bar;
  stage_model(m, smem, ctx, &bar);

  const unsigned long long C = a.C;
  const unsigned long long tid = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = tid < C;                                   // threads past the last chain shadow chain C-1 and write nothing:
  const unsigned long long chain = valid ? tid : C - 1;         // they take part in the CTA-wide data pass and the barriers
  const unsigned long long gchain = a.first_chain + chain;
  const int P = m.n_params, D = m.D, NT = m.n_terms;
  const bool in_smem = m.scratch_smem_off >= 0;
  // rows of the working set: wk[row * ws]; state rows: sp[c * ss]
  double* wk = in_smem ? reinterpret_cast<double*>(smem + m.scratch_smem_off) + threadIdx.x : a.tval + chain;
  const unsigned long long ws = in_smem ? (unsigned long long)kSyncThreads : C;
  double* sp = in_smem ? wk + (unsigned long long)(2 * NT + 2 * D) * ws : a.state + chain;
  unsigned short* vq = in_smem ? reinterpret_cast<unsigned short*>(smem + m.scratch_smem_off + (size_t)(2 * NT + 3 * D) * kSyncThreads * sizeof(double)) + threadIdx.x
                               : a.vseq + chain;
  const int rTC = NT, rBP = 2 * NT, rBC = 2 * NT + D;           // first rows of tcand, bprop, bcoin
  if (in_smem) {
    for (int t = 0; t < NT; ++t) wk[(unsigned long long)t * ws] = a.tval[(unsigned long long)t * C + chain];
    for (int c = 0; c < D; ++c) sp[(unsigned long long)c * ws] = a.state[(unsigned long long)c * C + chain];
  }
  const bool wr = valid || in_smem;                             // may this thread write its working set? (a shadow's shared column is its own)

  RandomStream g;
  g.init(a.rng_n[chain]);
  unsigned long long perm = a.perm[chain];
  double curr = a.curr_lp[chain];
  unsigned char order[kLocalOrder];

  long long rec_phase = sa.record ? sa.sample_i0 % sa.thin : 0;
  long long row = sa.record ? (sa.sample_i0 + sa.thin - 1) / sa.thin : 0;
  for (long long s = 0; s < sa.n_sweeps; ++s) {
    if (sa.record) {                                            // Sampler.sample: the state BEFORE stepping (mcmc.js:1021-1027)
      const bool rec_now = rec_phase == 0;
      if (++rec_phase == sa.thin) rec_phase = 0;
      if (rec_now && valid) {
        double der[kMaxDerived];
        bool have_der = false;
        for (int j = 0; j < sa.n_monitor; ++j) {
          int e = sa.monitor[j];
          double v;
          if (e < D) {
            v = sp[(unsigned long long)e * ws];
          } else {
            if (!have_der) { EvalState es{sp, ws, -1, 0.0}; run_ctx(ctx, es, derived_pc(m, es), der, false); have_der = true; }
            v = der[e - D];
          }
          sa.out[((unsigned long long)row * sa.n_monitor + j) * C + chain] = v;
        }
      }
      if (rec_now) ++row;
    }
    // ---- (a) this sweep's random numbers, in the reference's order
    if (m.stat_barriers) __syncthreads();
    for (int i = P - 1; i > 0; --i) {                           // shuffle_array(this.substeppers), in place (mcmc.js:887, 228-236)
      int j = (int)floor(g.next(a.seed, gchain) * (i + 1));
      perm_swap(a, perm, chain, i, j, valid);
    }
    int pos = 0;
    for (int slot = 0; slot < P; ++slot) {
      const amwg_param& pa = ctx.params[perm_get(a, perm, chain, slot)];
      const int inner = pa.n_comp / pa.dim0;
      if (pa.n_comp > 1) {                                      // nested_array_random_apply: top level only (mcmc.js:246-252)
        for (int i = 0; i < pa.dim0; ++i) ord_set(a, order, chain, pa.dim0, i, i, valid);
        for (int i = pa.dim0 - 1; i > 0; --i) {
          int j = (int)floor(g.next(a.seed, gchain) * (i + 1));
          const int t = ord_get(a, order, chain, pa.dim0, i);
          ord_set(a, order, chain, pa.dim0, i, ord_get(a, order, chain, pa.dim0, j), valid);
          ord_set(a, order, chain, pa.dim0, j, t, valid);
        }
      }
      for (int r = 0; r < pa.n_comp; ++r, ++pos) {
        int c = pa.comp_offset;
        if (pa.n_comp > 1) c += ord_get(a, order, chain, pa.dim0, r / inner) * inner + (r % inner);
        const double cur = sp[(unsigned long long)c * ws];
        double prop = js_rnorm(g, a.seed, gchain, cur, a.psd[(unsigned long long)c * C + chain]);   // generate_proposal (mcmc.js:519, 577-579 / 596-598)
        if (pa.type == AMWG_INT) prop = js_round(prop);
        const bool inb = !(prop < pa.lower || prop > pa.upper);              // bounds check (:520): no uniform when it fails
        const double coin = inb ? g.next(a.seed, gchain) : -1.0;
        if (wr) {
          wk[(unsigned long long)(rBP + c) * ws] = inb ? prop : cur;
          wk[(unsigned long long)(rBC + c) * ws] = coin;
          vq[(unsigned long long)pos * ws] = (unsigned short)c;
        }
      }
    }
    // ---- (b) one pass over the data: every plate statistic at the proposals -> candidate slots
    if (m.stat_barriers) __syncthreads();
    {
      EvalState es{sp, ws, -1, 0.0};
      es.tval = wr ? wk : nullptr;                              // a shadow of a global column computes along (barriers) and stores nothing
      es.tcand = wk + (unsigned long long)rTC * ws; es.tstride = ws;
      es.bprop = wk + (unsigned long long)rBP * ws; es.blk_lo = 0; es.blk_hi = D;
      eval_logpost<true>(ctx, es, m.stat_prog);
    }
    // ---- (c) the steps, in visiting order: O(1) each
    int c_next = (int)vq[0];
    double coin_next = wk[(unsigned long long)(rBC + c_next) * ws], prop_next = wk[(unsigned long long)(rBP + c_next) * ws];
    for (int i = 0; i < D; ++i) {
      if (m.stat_barriers && D <= 8) __syncthreads();           // few steps: keep the CTA's warps in the same code (instruction cache)
      const int c = c_next;
      const double coin = coin_next, prop = prop_next;
      if (i + 1 < D) {                                          // the next step's operands are on their way while this one is evaluated
        c_next = (int)vq[(unsigned long long)(i + 1) * ws];
        coin_next = wk[(unsigned long long)(rBC + c_next) * ws]; prop_next = wk[(unsigned long long)(rBP + c_next) * ws];
      }
      if (!wr || coin < 0.0) continue;                          // out of bounds: rejected without evaluation (mcmc.js:520-522)
      const bool adapting = m.adapting[c] != 0;
      EvalState es{sp, ws, c, prop};
      es.tval = wk; es.tcand = wk + (unsigned long long)rTC * ws; es.tstride = ws;
      const double lp_new = eval_logpost<true>(ctx, es, ctx.comp_prog[c]);
      const double accept_prob = js_exp(lp_new - curr);         // Metropolis accept (mcmc.js:527-534): strict >, NaN rejects
      if (accept_prob > coin) {
        curr = lp_new;
        sp[(unsigned long long)c * ws] = prop;
        if (adapting && valid) atomicAdd(&a.acc[(unsigned long long)c * C + chain], 1);      // result unused: a fire-and-forget RED
        for (int k = ctx.touch_off[c]; k < ctx.touch_off[c + 1]; ++k) {
          const unsigned long long t = (unsigned long long)ctx.touch_terms[k];
          wk[t * ws] = wk[(t + rTC) * ws];
        }
      }
    }
  }
  if (valid) {
    a.rng_n[chain] = g.n;
    a.perm[chain] = perm;
    a.curr_lp[chain] = curr;
    if (in_smem) {
      for (int t = 0; t < NT; ++t) a.tval[(unsigned long long)t * C + chain] = wk[(unsigned long long)t * ws];
      for (int c = 0; c < D; ++c) a.state[(unsigned long long)c * C + chain] = sp[(unsigned long long)c * ws];
    }
  }
}

// ---- K2: Roberts-Rosenthal batch update of prop_log_scale (mcmc.js:538-550), a follow-on kernel -----------------------
struct AdaptArgs {
  int c0, n;
  double delta[kAdaptChunk];        // min(max_adaptation, initial_adaptation / sqrt(batch_count))
  double batch_size[kAdaptChunk];
  double target[kAdaptChunk];
  unsigned char apply[kAdaptChunk];
};

__global__ void __launch_bounds__(256) amwg_adapt_kernel(ChainArrays a, AdaptArgs ad) {
  unsigned long long chain = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (chain >= a.C) return;
  for (int k = 0; k < ad.n; ++k) {
    if (!ad.apply[k]) continue;
    unsigned long long idx = (unsigned long long)(ad.c0 + k) * a.C + chain;
    double rate = (double)a.acc[idx] / ad.batch_size[k];
    double ls = a.pls[idx];
    ls = (rate > ad.target[k]) ? ls + ad.delta[k] : ls - ad.delta[k];
    a.pls[idx] = ls;
    a.psd[idx] = js_exp(ls);          // the proposal sd of the next batch: Math.exp(prop_log_scale), mcmc.js:578
    a.acc[idx] = 0;
  }
}

// ---- derived quantities for amwg_get_state ------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) amwg_derived_kernel(ModelDev m, ChainArrays a, double* out /*[n_derived][C]*/) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ Ctx ctx;
  __shared__ __align__(8) unsigned long long bar;
  stage_model(m, smem, ctx, &bar);
  unsigned long long chain = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (chain >= a.C) return;
  double der[kMaxDerived];
  EvalState es{a.state + chain, a.C, -1, 0.0};
  run_ctx(ctx, es, derived_pc(m, es), der, false);
  for (int d = 0; d < m.n_derived; ++d) out[(unsigned long long)d * a.C + chain] = der[d];
}

// ---- primitives for the parity tests / the `ld` host module ---------------------------------------------------------------
// one row of arguments -> one ld.* value, through the same interpreter: program `<op A=const0 B=const1 ..> END`, the
// row's arguments are the thread's private constants (staged in shared memory like a model's).
__global__ void __launch_bounds__(128) amwg_ld_kernel(int word, int arity, const double* __restrict__ args, long long n, double* __restrict__ out) {
  __shared__ int code[8];
  __shared__ double consts[128 * 4];
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (threadIdx.x == 0) {
    int nc = 0;
    code[nc++] = word;
    for (int k = arity - 1; k >= 0; --k) code[nc++] = k;      // inline operand words: last operand first
    code[nc++] = AMWG_WORD(AMWG_OP_END, AMWG_MODE_NONE, AMWG_MODE_NONE, AMWG_MODE_NONE, AMWG_MODE_NONE, 0, 0);
  }
  if (i < n) for (int k = 0; k < arity; ++k) consts[threadIdx.x * 4 + k] = args[i * arity + k];
  __syncthreads();
  if (i >= n) return;
  Ctx ctx{};
  EvalState es{nullptr, 0, -1, 0.0};
  out[i] = run_program(smem_u32(code), smem_u32(consts + threadIdx.x * 4), ctx, es, 0, nullptr, true);
}

__global__ void amwg_primitive_kernel(int kind, const double* __restrict__ x, long long n, unsigned long long seed,
                                      unsigned long long chain, double* __restrict__ out) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  __shared__ double tab[256];
  if (kind == 5) {                       // the Poisson plate's table-driven exponential (exp_acc), for its accuracy test
    for (int j = threadIdx.x; j < 256; j += blockDim.x) tab[j] = exp2((double)j * (1.0 / 256.0));
    __syncthreads();
    if (i < n) out[i] = exp_acc(x[i], smem_u32(tab), 0.0);
    return;
  }
  if (i >= n) return;
  if (kind == 0) out[i] = js_log(x[i]);
  else if (kind == 1) out[i] = js_exp(x[i]);
  else if (kind == 2) { RandomStream g; g.init((unsigned long long)i); out[i] = g.next(seed, chain); }
  else if (kind == 3) {   // sequential rnorm(x[0], x[1]) draws of one chain: thread 0 only
    if (i == 0) { RandomStream g; g.init(0); for (long long k = 0; k < n; ++k) out[k] = js_rnorm(g, seed, chain, x[0], x[1]); }
  } else if (kind == 4) out[i] = js_round(x[i]);
}

}  // namespace amwg

// ===================================================================================================================
// Host side: the C ABI
// ===================================================================================================================
using namespace amwg;

static thread_local std::string g_last_error;
static int fail(const std::string& msg) { g_last_error = msg; return -1; }
#define CUDA_TRY(expr)                                                                                 \
  do {                                                                                                 \
    cudaError_t _e = (expr);                                                                           \
    if (_e != cudaSuccess) return fail(std::string(#expr) + ": " + cudaGetErrorString(_e));           \
  } while (0)

struct amwg_sampler {
  int device = 0;
  cudaStream_t stream = nullptr, copy_stream = nullptr;
  ModelDev m{};
  ChainArrays a{};
  unsigned smem_bytes = 0;
  int D = 0, P = 0, n_derived = 0;
  std::vector<amwg_param> params;
  std::vector<amwg_comp_options> opts;
  std::vector<int> comp_type;                 // per component: AMWG_REAL/INT/BINARY
  std::vector<unsigned char> is_adapting;     // per component (host mirror of m.adapting)
  std::vector<double> iter_since, batch_count;   // chain-invariant counters (mcmc.js:510-511)
  std::vector<void*> dev_allocs;
  unsigned char* d_adapting = nullptr;
  double* d_out = nullptr; size_t d_out_bytes = 0;
  int* d_monitor = nullptr; int d_monitor_cap = 0;
  long long launches = 0;
  double last_sweep_ms = 0.0;
  // run-time specialised sweep (amwg_jit.cuh): active when jit_kernel != nullptr
  cudaKernel_t jit_kernel = nullptr;
  unsigned jit_smem = 0;
  int jit_threads = 0;
  std::string jit_note = "not attempted";
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev_pool;
};

template <typename T>
static int dev_upload(amwg_sampler* s, const T* host, size_t n, T** out, size_t pad_to = 16) {
  size_t bytes = std::max<size_t>(((n * sizeof(T) + pad_to - 1) / pad_to) * pad_to, pad_to);
  void* p = nullptr;
  CUDA_TRY(cudaMalloc(&p, bytes));
  s->dev_allocs.push_back(p);
  CUDA_TRY(cudaMemsetAsync(p, 0, bytes, s->stream));
  if (n) CUDA_TRY(cudaMemcpyAsync(p, host, n * sizeof(T), cudaMemcpyHostToDevice, s->stream));
  *out = reinterpret_cast<T*>(p);
  return 0;
}
template <typename T>
static int dev_alloc(amwg_sampler* s, size_t n, T** out) {
  void* p = nullptr;
  CUDA_TRY(cudaMalloc(&p, std::max<size_t>(n * sizeof(T), 16)));
  s->dev_allocs.push_back(p);
  *out = reinterpret_cast<T*>(p);
  return 0;
}

static unsigned pad16(size_t b) { return (unsigned)((b + 15) / 16 * 16); }

#include "amwg_jit.cuh"

// arguments of the run-time specialised sweep (amwg_jit_kernel.cuh: struct JitArgs, same layout)
struct JitArgsHost {
  ChainArrays a;
  SweepArgs sa;
  const double* col[kMaxColumns];
  const unsigned char* adapting;
};

static int validate_model(const amwg_model* md) {
  if (!md) return fail("amwg_create: model is NULL");
  if (md->abi_version != AMWG_ABI_VERSION) return fail("amwg_create: ABI version mismatch");
  if (md->n_params < 1 || md->n_params > kMaxParams) return fail("amwg_create: between 1 and 255 named parameters are supported");
  if (md->n_columns > kMaxColumns) return fail("amwg_create: at most 32 data columns are supported");
  if (md->n_derived > kMaxDerived) return fail("amwg_create: at most 32 derived quantities are supported");
  int D = 0;
  for (int p = 0; p < md->n_params; ++p) {
    const amwg_param& pa = md->params[p];
    if (pa.lower > pa.upper) return fail("Can not initialize parameter where lower bound > upper bound");   // mcmc.js:314-316
    if (pa.type < 0 || pa.type > 2) return fail("AmwgStepper can't handle parameter with this type");        // mcmc.js:867
    if (pa.n_comp < 1 || pa.dim0 < 1 || pa.n_comp % pa.dim0) return fail("amwg_create: bad parameter dimensions");
    if (pa.dim0 > kMaxDim0) return fail("amwg_create: dim[0] > 65535 is not supported");
    if (pa.comp_offset != D) return fail("amwg_create: comp_offset must be the running component count");
    if (pa.type == AMWG_BINARY)
      for (int c = 0; c < pa.n_comp; ++c)
        if (md->init[D + c] != 0.0 && md->init[D + c] != 1.0) return fail("amwg_create: binary parameters must start at 0 or 1");
    D += pa.n_comp;
  }
  if (D != md->n_comp) return fail("amwg_create: n_comp does not match the parameter list");
  if (md->logpost_prog < 0 || md->logpost_prog >= md->n_code) return fail("amwg_create: logpost_prog out of range");
  if (md->n_variant_comps < 0 || md->n_variant_comps > AMWG_MAX_VARIANT_COMPS) return fail("amwg_create: at most 4 program-selecting binary components are supported");
  for (int k = 0; k < md->n_variant_comps; ++k)
    if (md->variant_comps[k] < 0 || md->variant_comps[k] >= D) return fail("amwg_create: variant component out of range");
  for (int v = 0; v < (md->n_variant_comps ? (1 << md->n_variant_comps) : 0); ++v)
    if (md->variant_logpost[v] < 0 || md->variant_logpost[v] >= md->n_code) return fail("amwg_create: variant program out of range");
  if (md->n_derived > 0 && (md->derived_prog < 0 || md->derived_prog >= md->n_code)) return fail("amwg_create: derived_prog out of range");
  if (md->n_block_params < 0 || md->n_block_params > AMWG_MAX_BLOCK_PARAMS) return fail("amwg_create: at most 4 block-stepped parameters are supported");
  for (int k = 0; k < md->n_block_params; ++k)
    if (md->block_params[k] < 0 || md->block_params[k] >= md->n_params) return fail("amwg_create: block_params out of range");
  if (md->comp_prog && md->n_terms > 0) {
    if (!md->touch_off || !md->touch_terms) return fail("amwg_create: comp_prog without touch lists");
    if (md->n_variant_comps > 0) return fail("amwg_create: comp_prog cannot be combined with variant programs");
    for (int c = 0; c < md->n_comp; ++c) {
      if (md->comp_prog[c] < 0 || md->comp_prog[c] >= md->n_code) return fail("amwg_create: comp_prog out of range");
      if (md->touch_off[c] > md->touch_off[c + 1]) return fail("amwg_create: touch_off must be non-decreasing");
    }
    for (int k = 0; k < md->touch_off[md->n_comp]; ++k)
      if (md->touch_terms[k] < 0 || md->touch_terms[k] >= md->n_terms) return fail("amwg_create: touch_terms out of range");
  }
  for (int k = 0; k < md->n_fold; ++k)
    if (md->fold_prog[k] < 0 || md->fold_prog[k] >= md->n_code || md->fold_dst[k] < 0 || md->fold_dst[k] >= md->n_consts)
      return fail("amwg_create: constant-folding table out of range");
  // every program: well-formed words, operand stack within the interpreter's, every index inside its table
  std::vector<int> progs;
  progs.push_back(md->logpost_prog);
  if (md->n_derived > 0) progs.push_back(md->derived_prog);
  for (int v = 0; v < (md->n_variant_comps ? (1 << md->n_variant_comps) : 0); ++v) {
    progs.push_back(md->variant_logpost[v]);
    if (md->variant_derived && md->variant_derived[v] >= 0) progs.push_back(md->variant_derived[v]);
  }
  if (md->comp_prog && md->n_terms > 0) for (int c = 0; c < md->n_comp; ++c) progs.push_back(md->comp_prog[c]);
  if (md->comp_prog && md->n_terms > 0 && md->stat_prog >= 0) progs.push_back(md->stat_prog);
  for (int k = 0; k < md->n_fold; ++k) progs.push_back(md->fold_prog[k]);
  const int n_slots = (md->comp_prog && md->n_terms > 0) ? md->n_terms : 0;
  for (int pc : progs) {
    std::vector<jit::Insn> ins;
    std::string err;
    int depth = 0;
    if (!jit::decode_program(md, pc, ins, &depth, err)) return fail("amwg_create: malformed program: " + err);
    if (depth > kStack)
      return fail("log_post nests expressions " + std::to_string(depth) + " deep; the device's operand stack holds " + std::to_string(kStack));
    int loop_n = 0;
    for (const jit::Insn& in : ins) {
      for (int k = 0; k < 4; ++k) {
        if (in.mode[k] == AMWG_MODE_CONST && (in.inl[k] < 0 || in.inl[k] >= md->n_consts)) return fail("amwg_create: constant index out of range");
        if (in.mode[k] == AMWG_MODE_COMP && (in.inl[k] < 0 || in.inl[k] >= D)) return fail("amwg_create: component index out of range");
      }
      switch (in.op) {
        case AMWG_OP_CONST: if (in.a >= md->n_consts) return fail("amwg_create: constant index out of range"); break;
        case AMWG_OP_COMP: if (in.a >= D) return fail("amwg_create: component index out of range"); break;
        case AMWG_OP_DATA:
          if (in.a >= md->n_columns || in.extra[0] < 0 || in.extra[0] >= md->columns[in.a].n) return fail("amwg_create: data index out of range");
          break;
        case AMWG_OP_LOOP_BEGIN:
          if (in.a >= md->n_plates) return fail("amwg_create: plate index out of range");
          loop_n = md->plates[in.a].n;
          break;
        case AMWG_OP_DATA_I: case AMWG_OP_COMP_I: {
          if (in.a >= md->n_columns) return fail("amwg_create: data column out of range");
          const long long off = in.extra[0], stride = in.extra[1], last = off + stride * (long long)std::max(loop_n - 1, 0);
          if (off < 0 || off >= md->columns[in.a].n || last < 0 || last >= md->columns[in.a].n) return fail("amwg_create: plate walks past the end of a data column");
          if (in.op == AMWG_OP_COMP_I)           // state[base + data[i]]: JS would read `undefined` outside the array; refuse instead of reading past the state
            for (int i = 0; i < loop_n; ++i) {
              const double v = md->columns[in.a].values[off + stride * i];
              if (!(v == std::floor(v)) || in.extra[2] + v < 0 || in.extra[2] + v >= D) return fail("log_post indexes a parameter array with a data value outside its bounds");
            }
          break;
        }
        case AMWG_OP_PLATE: case AMWG_OP_PLATE_SS: case AMWG_OP_NORM_SS: {
          if (in.a >= md->n_plates) return fail("amwg_create: plate index out of range");
          const amwg_plate& pl = md->plates[in.a];
          for (int j = 0; j < 3; ++j) if (pl.col[j] >= md->n_columns) return fail("amwg_create: plate column out of range");
          if (in.op != AMWG_OP_NORM_SS && pl.kind != AMWG_PLATE_GENERIC) {
            if (pl.col[0] < 0 || pl.iparam[2] < 0 || (long long)pl.iparam[2] + pl.n > md->columns[pl.col[0]].n) return fail("amwg_create: plate runs past its data column");
            if ((pl.kind == AMWG_PLATE_NORM_GROUPED || pl.kind == AMWG_PLATE_POIS_LOGLIN) && (pl.iparam[0] < 0 || pl.iparam[1] < 0 || pl.iparam[0] + pl.iparam[1] > D))
              return fail("amwg_create: plate parameter range out of bounds");
          }
          if (in.op == AMWG_OP_PLATE_SS && (in.extra[0] < 0 || in.extra[0] >= n_slots)) return fail("amwg_create: statistic slot out of range");
          break;
        }
        case AMWG_OP_CACHED: case AMWG_OP_CAND: if (in.a >= n_slots) return fail("amwg_create: cache slot out of range"); break;
        case AMWG_OP_ACC_RANGE: if (in.extra[0] < 0 || in.a + in.extra[0] > n_slots) return fail("amwg_create: ACC_RANGE out of range"); break;
        case AMWG_OP_STORE: if (in.a >= std::max(md->n_derived, 1)) return fail("amwg_create: derived index out of range"); break;
        default: break;
      }
      if (in.term >= 0 && n_slots > 0 && in.term >= n_slots) return fail("amwg_create: term id out of range");
    }
  }
  return 0;
}

extern "C" int amwg_abi_version(void) { return AMWG_ABI_VERSION; }
extern "C" const char* amwg_last_error(void) { return g_last_error.c_str(); }
extern "C" int64_t amwg_kernel_launches(const amwg_sampler* s) { return s ? s->launches : 0; }
extern "C" double amwg_last_sweep_kernel_ms(const amwg_sampler* s) { return s ? s->last_sweep_ms : 0.0; }
extern "C" uint64_t amwg_n_chains(const amwg_sampler* s) { return s ? s->a.C : 0; }

extern "C" void amwg_destroy(amwg_sampler* s) {
  if (!s) return;
  cudaSetDevice(s->device);
  if (s->stream) cudaStreamSynchronize(s->stream);
  if (s->copy_stream) cudaStreamSynchronize(s->copy_stream);
  for (void* p : s->dev_allocs) cudaFree(p);
  if (s->d_out) cudaFree(s->d_out);
  if (s->d_monitor) cudaFree(s->d_monitor);
  for (auto& e : s->ev_pool) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
  if (s->stream) cudaStreamDestroy(s->stream);
  if (s->copy_stream) cudaStreamDestroy(s->copy_stream);
  delete s;
}

static unsigned grid_for(unsigned long long C, int threads) { return (unsigned)((C + threads - 1) / threads); }

// -0.5 * Math.log(2 * Math.PI) with the DEVICE's log (the value every kernel uses for the factorised Normal plates)
static int device_norm_c0(int device, double* out) {
  const double two_pi = 2 * AMWG_JS_PI;
  double lg = 0.0;
  if (amwg_primitive_eval(0, &two_pi, 1, 0, 0, &lg, device)) return -1;
  *out = -0.5 * lg;
  return 0;
}

// Try to replace the interpreter sweep of this handle by a kernel specialised for its model (amwg_jit.cuh). Never fatal: on any
// failure the handle keeps the interpreter kernels and s->jit_note says why.
static void try_jit(amwg_sampler* s, const amwg_model* md) {
  s->jit_note = "off";
  int want = -1;                                        // -1: when it pays (many chains), 0: never, 1: whenever the model is eligible
  if (const char* e = getenv("AMWG_JIT")) want = atoi(e);
  if (want == 0) { s->jit_note = "disabled (AMWG_JIT=0)"; return; }
  const bool stat_model = s->m.stat_prog >= 0;
  if (!stat_model && s->m.n_terms > 0) { s->jit_note = "the model steps with a term cache (interpreter kernels)"; return; }
  if (want < 0 && s->a.C < 4096) { s->jit_note = "fewer than 4096 chains: the interpreter kernels start faster than a compilation"; return; }
  std::vector<double> consts((size_t)std::max(md->n_consts, 1), 0.0);
  if (md->n_consts > 0 &&
      cudaMemcpy(consts.data(), s->m.image + s->m.off_consts, sizeof(double) * (size_t)md->n_consts, cudaMemcpyDeviceToHost) != cudaSuccess) {
    s->jit_note = "could not read the folded constants back"; cudaGetLastError(); return;
  }
  double c0 = 0.0;
  if (device_norm_c0(s->device, &c0)) { s->jit_note = "could not evaluate the Normal constant on the device"; return; }
  cudaDeviceProp prop{};
  if (cudaGetDeviceProperties(&prop, s->device) != cudaSuccess) { s->jit_note = "cudaGetDeviceProperties failed"; cudaGetLastError(); return; }
  jit::Source src;
  std::string why = stat_model ? jit::build_source(md, consts, s->a.C, prop.multiProcessorCount, c0, src)
                               : jit::build_source_full(md, consts, s->a.C, prop.multiProcessorCount, c0, src);
  if (!why.empty()) { s->jit_note = "not specialised: " + why; return; }
  if (src.plan.smem_bytes > (unsigned)prop.sharedMemPerBlockOptin) { s->jit_note = "not specialised: shared-memory plan does not fit"; return; }
  const unsigned long long key = jit::fnv1a(src.generated, jit::fnv1a(src.prelude));
  jit::Loaded ld;
  {
    std::lock_guard<std::mutex> lock(jit::g_cache_mu);
    auto it = jit::g_cache.find({s->device, key});
    if (it != jit::g_cache.end()) ld = it->second;
  }
  bool disk = false;
  if (!ld.kernel) {
    std::vector<char> cubin;
    std::string log;
    std::string e = jit::get_cubin(src, cubin, log, &disk);
    if (!e.empty()) { s->jit_note = "compilation failed: " + e + (log.empty() ? "" : "\n" + log); return; }
    if (cudaLibraryLoadData(&ld.lib, cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0) != cudaSuccess ||
        cudaLibraryGetKernel(&ld.kernel, ld.lib, "amwg_jit_sweep") != cudaSuccess) {
      s->jit_note = std::string("loading the compiled kernel failed: ") + cudaGetErrorString(cudaGetLastError());
      return;
    }
    std::lock_guard<std::mutex> lock(jit::g_cache_mu);
    jit::g_cache[{s->device, key}] = ld;
  }
  if (cudaFuncSetAttribute((const void*)ld.kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)src.plan.smem_bytes) != cudaSuccess) {
    s->jit_note = std::string("cudaFuncSetAttribute on the compiled kernel failed: ") + cudaGetErrorString(cudaGetLastError());
    return;
  }
  s->jit_kernel = ld.kernel;
  s->jit_smem = src.plan.smem_bytes;
  s->jit_threads = src.plan.threads;
  char note[256];
  snprintf(note, sizeof note, "specialised %s: %d threads x %d CTAs/SM, %u B shared memory, %d resident column(s)%s%s%s", src.full ? "full-program sweep" : "sweep", src.plan.threads, src.plan.minblocks,
           src.plan.smem_bytes, src.plan.n_res, src.plan.stream_col >= 0 ? ", one streamed column" : "", src.plan.ws_smem ? ", working set in shared memory" : "",
           disk ? " (cubin from the disk cache)" : "");
  s->jit_note = note;
}

extern "C" int amwg_create(const amwg_model* md, uint64_t n_chains, uint64_t first_chain, uint64_t seed, int device,
                           amwg_sampler** out) {
  if (!out) return fail("amwg_create: out is NULL");
  *out = nullptr;
  if (validate_model(md)) return -1;
  if (n_chains == 0) return fail("amwg_create: n_chains must be > 0");
  int ndev = 0;
  CUDA_TRY(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail("amwg_create: no such CUDA device (this library has no CPU fallback)");
  CUDA_TRY(cudaSetDevice(device));
  amwg_sampler* s = new amwg_sampler();
  s->device = device;
  auto bail = [&](int rc) { amwg_destroy(s); return rc; };
  if (cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking) != cudaSuccess) return bail(fail("cudaStreamCreate failed"));
  if (cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking) != cudaSuccess) return bail(fail("cudaStreamCreate failed"));

  s->D = md->n_comp; s->P = md->n_params; s->n_derived = md->n_derived;
  s->params.assign(md->params, md->params + md->n_params);
  s->opts.assign(md->comp_options, md->comp_options + md->n_comp);
  s->comp_type.resize(s->D);
  for (const auto& pa : s->params) for (int c = 0; c < pa.n_comp; ++c) s->comp_type[pa.comp_offset + c] = pa.type;
  s->is_adapting.resize(s->D);
  for (int c = 0; c < s->D; ++c) s->is_adapting[c] = (s->comp_type[c] != AMWG_BINARY && s->opts[c].is_adapting) ? 1 : 0;
  s->iter_since.assign(s->D, 0.0);
  s->batch_count.assign(s->D, 0.0);

  // model image: [code | consts | plates | params], 16B-aligned sections, one bulk-TMA transfer per CTA
  ModelDev& m = s->m;
  std::vector<unsigned char> image;
  auto append = [&](const void* p, size_t bytes) { unsigned off = (unsigned)image.size(); image.resize(off + pad16(std::max<size_t>(bytes, 1)), 0); if (bytes) memcpy(image.data() + off, p, bytes); return off; };
  m.off_code = append(md->code, sizeof(int32_t) * (size_t)md->n_code);
  m.off_consts = append(md->consts, sizeof(double) * (size_t)md->n_consts);
  m.off_plates = append(md->plates, sizeof(amwg_plate) * (size_t)md->n_plates);
  m.off_params = append(md->params, sizeof(amwg_param) * (size_t)md->n_params);
  m.n_terms = (md->comp_prog && md->n_terms > 0) ? md->n_terms : 0;
  if (const char* e = getenv("AMWG_TERM_CACHE")) { if (atoi(e) == 0) m.n_terms = 0; }
  m.off_comp_prog = append(md->comp_prog, m.n_terms ? sizeof(int32_t) * (size_t)md->n_comp : 0);
  m.off_touch_off = append(md->touch_off, m.n_terms ? sizeof(int32_t) * (size_t)(md->n_comp + 1) : 0);
  m.off_touch_terms = append(md->touch_terms, m.n_terms ? sizeof(int32_t) * (size_t)md->touch_off[md->n_comp] : 0);
  m.n_block_params = (m.n_terms && md->block_params && md->term_block_comp) ? md->n_block_params : 0;
  if (const char* e = getenv("AMWG_BLOCK_STEPS")) { if (atoi(e) == 0) m.n_block_params = 0; }
  for (int k = 0; k < m.n_block_params; ++k) m.block_params[k] = md->block_params[k];
  m.off_tbc = append(md->term_block_comp, m.n_block_params ? sizeof(int32_t) * (size_t)m.n_block_params * (size_t)m.n_terms : 0);
  // pre-evaluated statistics: comp_prog then reads candidate slots that only amwg_stat_sweep_kernel fills, so switching the
  // sweep off (AMWG_STAT_SWEEP=0, for A/B runs) also drops the term cache: every step evaluates the full program
  m.stat_prog = (m.n_terms && md->stat_prog >= 0) ? md->stat_prog : -1;
  if (md->stat_prog >= 0) {
    bool off = md->n_variant_comps > 0 || md->n_comp > 65535;
    if (const char* e = getenv("AMWG_STAT_SWEEP")) off = off || atoi(e) == 0;
    if (off) { m.stat_prog = -1; m.n_terms = 0; m.n_block_params = 0; }
  }
  m.stat_barriers = 1;
  if (const char* e = getenv("AMWG_STAT_BARRIERS")) m.stat_barriers = atoi(e) != 0;
  m.image_bytes = (unsigned)image.size();
  unsigned char* d_image = nullptr;
  if (dev_upload(s, image.data(), image.size(), &d_image)) return bail(-1);
  m.image = d_image;
  m.n_columns = md->n_columns; m.n_plates = md->n_plates; m.n_params = md->n_params; m.D = md->n_comp;
  m.n_derived = md->n_derived; m.logpost_prog = md->logpost_prog; m.derived_prog = md->derived_prog;
  m.n_variant_comps = md->n_variant_comps;
  m.has_pois = 0;
  for (int q = 0; q < md->n_plates; ++q) m.has_pois |= md->plates[q].kind == AMWG_PLATE_POIS_LOGLIN;
  for (int k = 0; k < md->n_variant_comps; ++k) m.variant_comps[k] = md->variant_comps[k];
  for (int v = 0; v < (md->n_variant_comps ? (1 << md->n_variant_comps) : 0); ++v) {
    m.variant_logpost[v] = md->variant_logpost[v];
    m.variant_derived[v] = md->variant_derived ? md->variant_derived[v] : -1;
  }
  {
    bool all_scalar = true;                       // "scalar" = one evaluation per sweep slot: scalar parameters and block-stepped ones
    for (int p = 0; p < md->n_params; ++p) {
      bool block = false;
      for (int k = 0; k < m.n_block_params; ++k) block = block || m.block_params[k] == p;
      all_scalar = all_scalar && (md->params[p].n_comp == 1 || block);
    }
    m.phase_sync = (all_scalar || md->n_params == 1) ? 1 : 0;
    if (const char* e = getenv("AMWG_PHASE_SYNC")) m.phase_sync = m.phase_sync && atoi(e) != 0;
    if (m.stat_prog >= 0) m.phase_sync = 1;        // the data pass is CTA-uniform by construction
  }

  unsigned smem_used = m.image_bytes;
  {   // if the columns do not all fit, reserve the TMA tile ring first, then keep resident whatever still fits
    size_t all = m.image_bytes;
    for (int k = 0; k < md->n_columns; ++k) all += pad16(std::max<size_t>(sizeof(double) * (size_t)md->columns[k].n, 16));
    m.ring_smem_off = -1;
    // the ring is only usable by CTA-uniform models (see stage_model): do not spend shared memory (= resident CTAs) on it otherwise
    if (all > kSmemBudget && m.phase_sync && m.n_variant_comps == 0) { m.ring_smem_off = (int)smem_used; smem_used += kRingStages * kRingStageBytes; }
  }
  const unsigned resident_budget = m.ring_smem_off >= 0 ? 36u * 1024u : kSmemBudget;    // with the ring: keep six CTAs per SM
  for (int k = 0; k < md->n_columns; ++k) {
    double* d_col = nullptr;
    if (dev_upload(s, md->columns[k].values, (size_t)md->columns[k].n, &d_col)) return bail(-1);
    m.col_global[k] = d_col;
    m.col_bytes[k] = pad16(std::max<size_t>(sizeof(double) * (size_t)md->columns[k].n, 16));
    if (smem_used + m.col_bytes[k] <= resident_budget) { m.col_smem_off[k] = (int)smem_used; smem_used += m.col_bytes[k]; }
    else m.col_smem_off[k] = -1;       // too large for shared memory: served from L2 (streamed tiles: DESIGN.md "next")
  }
  // working set of a statistics sweep in shared memory, when 7 CTAs per SM still fit (the register cap's occupancy)
  m.scratch_smem_off = -1;
  if (m.stat_prog >= 0) {
    const size_t per_thread = sizeof(double) * (size_t)(2 * m.n_terms + 3 * md->n_comp) + sizeof(unsigned short) * (size_t)md->n_comp;
    const size_t need = pad16(per_thread * kSyncThreads);
    bool use = pad16(smem_used) + need <= (227u * 1024u) / 7u - 1024u;
    if (const char* e = getenv("AMWG_STAT_SMEM")) use = use && atoi(e) != 0;
    if (use) { m.scratch_smem_off = (int)pad16(smem_used); smem_used = (unsigned)(pad16(smem_used) + need); }
  }
  s->smem_bytes = smem_used;
  if (cudaFuncSetAttribute(amwg_sweep_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBudget) != cudaSuccess ||
      cudaFuncSetAttribute(amwg_sweep_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBudget) != cudaSuccess ||
      cudaFuncSetAttribute(amwg_stat_sweep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBudget) != cudaSuccess ||
      cudaFuncSetAttribute(amwg_init_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBudget) != cudaSuccess ||
      cudaFuncSetAttribute(amwg_relp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBudget) != cudaSuccess ||
      cudaFuncSetAttribute(amwg_fold_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBudget) != cudaSuccess ||
      cudaFuncSetAttribute(amwg_derived_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBudget) != cudaSuccess)
    return bail(fail("cudaFuncSetAttribute(MaxDynamicSharedMemorySize) failed"));

  if (dev_upload(s, s->is_adapting.data(), (size_t)s->D, &s->d_adapting)) return bail(-1);
  m.adapting = s->d_adapting;

  ChainArrays& a = s->a;
  a.C = n_chains; a.first_chain = first_chain; a.seed = seed;
  size_t DC = (size_t)s->D * (size_t)n_chains;
  if (dev_alloc(s, DC, &a.state) || dev_alloc(s, DC, &a.pls) || dev_alloc(s, DC, &a.psd) || dev_alloc(s, DC, &a.acc) || dev_alloc(s, (size_t)n_chains, &a.curr_lp) ||
      dev_alloc(s, (size_t)n_chains, &a.perm) || dev_alloc(s, (size_t)n_chains, &a.rng_n))
    return bail(-1);
  a.tval = a.tcand = a.bprop = a.bcoin = nullptr;
  a.vseq = nullptr;
  a.perm_ext = nullptr;
  a.order_ext = nullptr;
  {
    int max_dim0 = 1;
    for (const auto& pa : s->params) if (pa.n_comp > 1) max_dim0 = std::max(max_dim0, pa.dim0);
    if (s->P > 16 && dev_alloc(s, (size_t)s->P * (size_t)n_chains, &a.perm_ext)) return bail(-1);
    if (max_dim0 > kLocalOrder && dev_alloc(s, (size_t)max_dim0 * (size_t)n_chains, &a.order_ext)) return bail(-1);
  }
  if (m.n_terms > 0) {
    // one allocation, rows [tval n_terms | tcand n_terms | bprop D | bcoin D] x C: amwg_stat_sweep_kernel addresses them as one block
    const size_t TC = (size_t)m.n_terms * (size_t)n_chains;
    if (dev_alloc(s, 2 * TC + 2 * DC, &a.tval)) return bail(-1);
    a.tcand = a.tval + TC; a.bprop = a.tcand + TC; a.bcoin = a.bprop + DC;
    if (m.stat_prog >= 0 && dev_alloc(s, DC, &a.vseq)) return bail(-1);
  }

  double* d_init = nullptr; double* d_pls0 = nullptr;
  std::vector<double> pls0(s->D);
  for (int c = 0; c < s->D; ++c) pls0[c] = s->opts[c].prop_log_scale;
  if (dev_upload(s, md->init, (size_t)s->D, &d_init) || dev_upload(s, pls0.data(), (size_t)s->D, &d_pls0)) return bail(-1);

  if (md->n_fold > 0) {
    int *d_fp = nullptr, *d_fd = nullptr;
    if (dev_upload(s, md->fold_prog, (size_t)md->n_fold, &d_fp) || dev_upload(s, md->fold_dst, (size_t)md->n_fold, &d_fd)) return bail(-1);
    amwg_fold_kernel<<<1, 32, s->smem_bytes, s->stream>>>(m, md->n_fold, d_fp, d_fd);
    s->launches++;
  }
  amwg_init_kernel<<<grid_for(n_chains, kThreads), kThreads, s->smem_bytes, s->stream>>>(m, a, d_init, d_pls0);
  s->launches++;
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaStreamSynchronize(s->stream);
  if (e != cudaSuccess) return bail(fail(std::string("amwg_init_kernel: ") + cudaGetErrorString(e)));
  try_jit(s, md);
  *out = s;
  return 0;
}

// Run n Sampler.step()s. Between sweep launches the host advances the chain-invariant adaptation counters and, when a
// component reaches its batch boundary (mcmc.js:538), launches the adaptation kernel. A launch never crosses a boundary.
static int run_sweeps(amwg_sampler* s, long long n, int record, long long thin, const int* d_monitor, int n_monitor, double* d_out,
                      double* host_out) {
  const unsigned long long C = s->a.C;
  long long i0 = 0;
  size_t n_events = 0;
  long long rows_copied = 0;
  while (i0 < n) {
    long long L = n - i0;
    for (int c = 0; c < s->D; ++c) {
      if (!s->is_adapting[c]) continue;
      double need = std::ceil(s->opts[c].batch_size - s->iter_since[c]);
      if (!(need >= 1.0)) need = 1.0;
      if (need < (double)L) L = (long long)need;
    }
    if (record && host_out && L > kHostChunkSweeps) L = kHostChunkSweeps;   // finer launches: the D2H of finished rows trails the sweeps closely
    // ... and the last launches taper off (.., 10, 5, 3, 2), because the copy of the final launch's rows is the one that nothing hides
    if (record && host_out && n - i0 <= kHostChunkSweeps && L > 2) L = std::min(L, std::max<long long>(2, (n - i0 + 1) / 2));
    SweepArgs sa{L, i0, thin, record, n_monitor, d_monitor, d_out};
    if (n_events >= s->ev_pool.size()) {
      cudaEvent_t e0, e1;
      CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
      s->ev_pool.emplace_back(e0, e1);
    }
    CUDA_TRY(cudaEventRecord(s->ev_pool[n_events].first, s->stream));
    if (s->jit_kernel) {
      JitArgsHost ja{};
      ja.a = s->a; ja.sa = sa; ja.adapting = s->d_adapting;
      for (int k = 0; k < kMaxColumns; ++k) ja.col[k] = k < s->m.n_columns ? s->m.col_global[k] : nullptr;
      void* kargs[] = {&ja};
      CUDA_TRY(cudaLaunchKernel((const void*)s->jit_kernel, dim3(grid_for(C, s->jit_threads)), dim3((unsigned)s->jit_threads), kargs, s->jit_smem, s->stream));
    } else {
      const int threads = s->m.phase_sync ? kSyncThreads : kThreads;
      if (s->m.stat_prog >= 0) amwg_stat_sweep_kernel<<<grid_for(C, kSyncThreads), kSyncThreads, s->smem_bytes, s->stream>>>(s->m, s->a, sa);
      else if (s->m.n_terms > 0) amwg_sweep_kernel<true><<<grid_for(C, threads), threads, s->smem_bytes, s->stream>>>(s->m, s->a, sa);
      else amwg_sweep_kernel<false><<<grid_for(C, threads), threads, s->smem_bytes, s->stream>>>(s->m, s->a, sa);
    }
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(s->ev_pool[n_events].second, s->stream));
    n_events++;
    s->launches++;

    // chain-invariant bookkeeping of OnedimMetropolisStepper (mcmc.js:536-551)
    bool any = false;
    std::vector<unsigned char> apply(s->D, 0);
    std::vector<double> delta(s->D, 0.0);
    for (int c = 0; c < s->D; ++c) {
      if (!s->is_adapting[c]) continue;
      s->iter_since[c] += (double)L;
      if (s->iter_since[c] >= s->opts[c].batch_size) {
        s->batch_count[c] += 1.0;
        double adj = s->opts[c].initial_adaptation / std::sqrt(s->batch_count[c]);
        double mx = s->opts[c].max_adaptation;
        delta[c] = (adj != adj || mx != mx) ? NAN : std::min(mx, adj);
        apply[c] = 1; any = true;
        s->iter_since[c] = 0.0;
      }
    }
    if (any) {
      for (int c0 = 0; c0 < s->D; c0 += kAdaptChunk) {
        AdaptArgs ad{};
        ad.c0 = c0; ad.n = std::min(kAdaptChunk, s->D - c0);
        bool chunk_any = false;
        for (int k = 0; k < ad.n; ++k) {
          ad.apply[k] = apply[c0 + k]; ad.delta[k] = delta[c0 + k];
          ad.batch_size[k] = s->opts[c0 + k].batch_size; ad.target[k] = s->opts[c0 + k].target_accept_rate;
          chunk_any |= (apply[c0 + k] != 0);
        }
        if (!chunk_any) continue;
        amwg_adapt_kernel<<<grid_for(C, 256), 256, 0, s->stream>>>(s->a, ad);
        CUDA_TRY(cudaGetLastError());
        s->launches++;
      }
    }
    i0 += L;
    // rows [rows_copied, rows_done) are final: overlap their D2H with the next sweeps
    if (record && host_out) {
      long long rows_done = (i0 + thin - 1) / thin;
      if (rows_done > rows_copied) {
        cudaEvent_t done = s->ev_pool[n_events - 1].second;
        CUDA_TRY(cudaStreamWaitEvent(s->copy_stream, done, 0));
        size_t row_elems = (size_t)n_monitor * (size_t)C;
        CUDA_TRY(cudaMemcpyAsync(host_out + (size_t)rows_copied * row_elems, d_out + (size_t)rows_copied * row_elems,
                                 (size_t)(rows_done - rows_copied) * row_elems * sizeof(double), cudaMemcpyDeviceToHost, s->copy_stream));
        rows_copied = rows_done;
      }
    }
  }
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  if (record && host_out) CUDA_TRY(cudaStreamSynchronize(s->copy_stream));
  double ms = 0.0;
  for (size_t k = 0; k < n_events; ++k) {
    float t = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&t, s->ev_pool[k].first, s->ev_pool[k].second));
    ms += t;
  }
  s->last_sweep_ms = ms;
  return 0;
}

extern "C" int amwg_burn(amwg_sampler* s, int64_t n) {
  if (!s) return fail("amwg_burn: NULL handle");
  if (n < 0) return fail("amwg_burn: n must be >= 0");
  CUDA_TRY(cudaSetDevice(s->device));
  if (n == 0) { s->last_sweep_ms = 0.0; return 0; }
  return run_sweeps(s, n, 0, 1, nullptr, 0, nullptr, nullptr);
}

static int prepare_monitor(amwg_sampler* s, const int32_t* monitor, int32_t n_monitor) {
  if (n_monitor < 0 || (n_monitor > 0 && !monitor)) return fail("amwg_sample: bad monitor list");
  for (int j = 0; j < n_monitor; ++j)
    if (monitor[j] < 0 || monitor[j] >= s->D + s->n_derived) return fail("amwg_sample: monitor entry out of range");
  if (n_monitor > s->d_monitor_cap) {
    if (s->d_monitor) cudaFree(s->d_monitor);
    s->d_monitor = nullptr; s->d_monitor_cap = 0;
    CUDA_TRY(cudaMalloc(&s->d_monitor, sizeof(int) * (size_t)std::max(n_monitor, 16)));
    s->d_monitor_cap = std::max(n_monitor, 16);
  }
  if (n_monitor) CUDA_TRY(cudaMemcpyAsync(s->d_monitor, monitor, sizeof(int) * (size_t)n_monitor, cudaMemcpyHostToDevice, s->stream));
  return 0;
}

extern "C" int amwg_sample_device(amwg_sampler* s, int64_t n, int64_t thin, const int32_t* monitor, int32_t n_monitor, double* dev_out) {
  if (!s) return fail("amwg_sample: NULL handle");
  if (n < 0 || thin < 1) return fail("amwg_sample: n must be >= 0 and thin >= 1");
  CUDA_TRY(cudaSetDevice(s->device));
  if (prepare_monitor(s, monitor, n_monitor)) return -1;
  if (n == 0) { s->last_sweep_ms = 0.0; return 0; }
  if (n_monitor > 0 && !dev_out) return fail("amwg_sample_device: dev_out is NULL");
  return run_sweeps(s, n, 1, thin, s->d_monitor, n_monitor, dev_out, nullptr);
}

extern "C" int amwg_sample(amwg_sampler* s, int64_t n, int64_t thin, const int32_t* monitor, int32_t n_monitor, double* host_out) {
  if (!s) return fail("amwg_sample: NULL handle");
  if (n < 0 || thin < 1) return fail("amwg_sample: n must be >= 0 and thin >= 1");
  CUDA_TRY(cudaSetDevice(s->device));
  if (prepare_monitor(s, monitor, n_monitor)) return -1;
  if (n == 0) { s->last_sweep_ms = 0.0; return 0; }
  if (n_monitor > 0 && !host_out) return fail("amwg_sample: host_out is NULL");
  size_t rows = (size_t)((n + thin - 1) / thin);
  size_t bytes = rows * (size_t)n_monitor * (size_t)s->a.C * sizeof(double);
  if (bytes > s->d_out_bytes) {
    if (s->d_out) cudaFree(s->d_out);
    s->d_out = nullptr; s->d_out_bytes = 0;
    CUDA_TRY(cudaMalloc(&s->d_out, std::max<size_t>(bytes, 16)));
    s->d_out_bytes = bytes;
  }
  return run_sweeps(s, n, 1, thin, s->d_monitor, n_monitor, s->d_out, host_out);
}

extern "C" int amwg_get_state(amwg_sampler* s, double* host_out) {
  if (!s || !host_out) return fail("amwg_get_state: NULL argument");
  CUDA_TRY(cudaSetDevice(s->device));
  size_t C = (size_t)s->a.C;
  CUDA_TRY(cudaMemcpyAsync(host_out, s->a.state, sizeof(double) * (size_t)s->D * C, cudaMemcpyDeviceToHost, s->stream));
  if (s->n_derived > 0) {
    double* d_der = nullptr;
    CUDA_TRY(cudaMalloc(&d_der, sizeof(double) * (size_t)s->n_derived * C));
    amwg_derived_kernel<<<grid_for(C, kThreads), kThreads, s->smem_bytes, s->stream>>>(s->m, s->a, d_der);
    s->launches++;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(host_out + (size_t)s->D * C, d_der, sizeof(double) * (size_t)s->n_derived * C, cudaMemcpyDeviceToHost, s->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s->stream);
    cudaFree(d_der);
    if (e != cudaSuccess) return fail(std::string("amwg_get_state: ") + cudaGetErrorString(e));
    return 0;
  }
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  return 0;
}

extern "C" int amwg_get_log_post(amwg_sampler* s, double* host_out) {
  if (!s || !host_out) return fail("amwg_get_log_post: NULL argument");
  CUDA_TRY(cudaSetDevice(s->device));
  if (s->jit_kernel) {          // the specialised sweep steps on differences: evaluate log_post at the current state now
    amwg_relp_kernel<<<grid_for(s->a.C, kThreads), kThreads, s->smem_bytes, s->stream>>>(s->m, s->a);
    CUDA_TRY(cudaGetLastError());
    s->launches++;
  }
  CUDA_TRY(cudaMemcpyAsync(host_out, s->a.curr_lp, sizeof(double) * (size_t)s->a.C, cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  return 0;
}

extern "C" int amwg_set_adapting(amwg_sampler* s, int32_t flag) {
  if (!s) return fail("amwg_set_adapting: NULL handle");
  CUDA_TRY(cudaSetDevice(s->device));
  for (int c = 0; c < s->D; ++c) s->is_adapting[c] = (s->comp_type[c] != AMWG_BINARY && flag) ? 1 : 0;
  CUDA_TRY(cudaMemcpyAsync(s->d_adapting, s->is_adapting.data(), (size_t)s->D, cudaMemcpyHostToDevice, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  return 0;
}

extern "C" int amwg_info(amwg_sampler* s, double* scalars, double* prop_log_scale, int32_t* acceptance_count) {
  if (!s) return fail("amwg_info: NULL handle");
  CUDA_TRY(cudaSetDevice(s->device));
  if (scalars)
    for (int c = 0; c < s->D; ++c) {
      scalars[c * 3 + 0] = s->is_adapting[c]; scalars[c * 3 + 1] = s->iter_since[c]; scalars[c * 3 + 2] = s->batch_count[c];
    }
  size_t DC = (size_t)s->D * (size_t)s->a.C;
  if (prop_log_scale) CUDA_TRY(cudaMemcpyAsync(prop_log_scale, s->a.pls, sizeof(double) * DC, cudaMemcpyDeviceToHost, s->stream));
  if (acceptance_count) CUDA_TRY(cudaMemcpyAsync(acceptance_count, s->a.acc, sizeof(int) * DC, cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  return 0;
}

// 1 when the handle runs the run-time specialised sweep, 0 when it runs the interpreter kernels; `note` says what was built or why not
extern "C" int amwg_jit_status(const amwg_sampler* s, char* note, int64_t cap) {
  if (!s) return 0;
  if (note && cap > 0) { snprintf(note, (size_t)cap, "%s", s->jit_note.c_str()); }
  return s->jit_kernel ? 1 : 0;
}

// Generate and compile the specialised sweep of `model` without a GPU (NVRTC targets sm_100a from any host): 0 = compiled,
// 1 = the model is not eligible (reason in `log`), -1 = generation or compilation failed (message in `log`). `src`, when given,
// receives the generated source. Constants that the device would fold at create are left as they are in the model.
extern "C" int amwg_jit_compile_check(const amwg_model* md, uint64_t n_chains, char* log, int64_t log_cap, char* src_out, int64_t src_cap) {
  auto put = [](char* dst, int64_t cap, const std::string& s) { if (dst && cap > 0) snprintf(dst, (size_t)cap, "%s", s.c_str()); };
  if (validate_model(md)) { put(log, log_cap, g_last_error); return -1; }
  std::vector<double> consts(md->consts, md->consts + md->n_consts);
  if (consts.empty()) consts.push_back(0.0);
  jit::Source src;
  const bool stat_model = md->comp_prog && md->n_terms > 0 && md->stat_prog >= 0;
  std::string why = stat_model ? jit::build_source(md, consts, n_chains ? n_chains : 1, 148, -0.9189385332046727, src)
                               : jit::build_source_full(md, consts, n_chains ? n_chains : 1, 148, -0.9189385332046727, src);
  if (!why.empty()) { put(log, log_cap, why); return 1; }
  put(src_out, src_cap, src.prelude + src.generated);
  std::vector<char> cubin;
  std::string clog;
  std::string e = jit::compile(src, cubin, clog);
  if (!e.empty()) { put(log, log_cap, e + "\n" + clog); return -1; }
  char info[160];
  snprintf(info, sizeof info, "ok: cubin %zu bytes, %d threads x %d CTAs/SM, %u B shared memory", cubin.size(), src.plan.threads, src.plan.minblocks, src.plan.smem_bytes);
  put(log, log_cap, std::string(info) + (clog.size() > 1 ? "\n" + clog : ""));
  return 0;
}

extern "C" int amwg_ld_eval(int32_t op, const double* args, int32_t arity, int64_t n, double* out, int device) {
  if (n <= 0) return 0;
  if (op <= AMWG_OP_COMP_I || (op >= AMWG_OP_ACC && op < AMWG_OP_NORM_K) || op >= AMWG_OP__COUNT || arity < 1 || arity > 4)
    return fail("amwg_ld_eval: bad opcode or arity");
  CUDA_TRY(cudaSetDevice(device));
  const int c = AMWG_MODE_CONST;
  const int none = AMWG_MODE_NONE;
  int word = AMWG_WORD(op, c, arity > 1 ? c : none, arity > 2 ? c : none, arity > 3 ? c : none, 0, 0);
  double *d_args = nullptr, *d_out = nullptr;
  CUDA_TRY(cudaMalloc(&d_args, sizeof(double) * (size_t)n * arity));
  if (cudaMalloc(&d_out, sizeof(double) * (size_t)n) != cudaSuccess) { cudaFree(d_args); return fail("amwg_ld_eval: cudaMalloc failed"); }
  cudaError_t e = cudaMemcpy(d_args, args, sizeof(double) * (size_t)n * arity, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    amwg_ld_kernel<<<(unsigned)((n + 127) / 128), 128>>>(word, arity, d_args, n, d_out);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpy(out, d_out, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost);
  cudaFree(d_args); cudaFree(d_out);
  if (e != cudaSuccess) return fail(std::string("amwg_ld_eval: ") + cudaGetErrorString(e));
  return 0;
}

extern "C" int amwg_primitive_eval(int32_t kind, const double* x, int64_t n, uint64_t seed, uint64_t chain, double* out, int device) {
  if (n <= 0) return 0;
  CUDA_TRY(cudaSetDevice(device));
  double *d_x = nullptr, *d_out = nullptr;
  CUDA_TRY(cudaMalloc(&d_x, sizeof(double) * (size_t)n));
  if (cudaMalloc(&d_out, sizeof(double) * (size_t)n) != cudaSuccess) { cudaFree(d_x); return fail("amwg_primitive_eval: cudaMalloc failed"); }
  cudaError_t e = cudaMemcpy(d_x, x, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    amwg_primitive_kernel<<<(unsigned)((n + 127) / 128), 128>>>(kind, d_x, n, seed, chain, d_out);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpy(out, d_out, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost);
  cudaFree(d_x); cudaFree(d_out);
  if (e != cudaSuccess) return fail(std::string("amwg_primitive_eval: ") + cudaGetErrorString(e));
  return 0;
}

#include "amwg_summary.cuh"
#include "amwg_rank.cuh"
#include "amwg_peak.cuh"
