// amwg_jit_kernel.cuh -- the sweep kernel that amwg_jit.cuh specialises per model and compiles with NVRTC for sm_100a.
//
// Reference path (all under /root/reference/): Sampler.sample / burn / step (mcmc.js:985-1039), AmwgStepper.step (:886-892),
// MultidimComponentMetropolisStepper.step (:685-688), OnedimMetropolisStepper.step (:517-553), rnorm / shuffle_array (:43-54,
// :228-236), and the user's log_post -> ld.* (distributions.js) -- the same path as amwg_stat_sweep_kernel, for the same class of
// models (amwg.h stat_prog: every O(N) piece of log_post is a Normal plate whose mean reads exactly one component), with the
// bytecode interpreter replaced by code generated from the model's programs:
//
//   (a) this sweep's random numbers -- substepper shuffle, visiting orders, rnorm trials, accept uniforms -- in the reference's
//       order (none of them depends on a log_post value);
//   (b) ONE pass over the data: every plate's S = sum_i (x_i - mean)^2 at the proposals. Resident columns are read as warp
//       broadcasts from shared memory (staged once per CTA by bulk TMA); a column that does not fit streams through a 4-stage
//       TMA tile ring (one mbarrier per stage, one CTA barrier per tile);
//   (c) the steps in the chain's visiting order, each an O(1) DELTA evaluation: log_post(proposal) - log_post(current) is the sum
//       over the terms that read the moved component of (new value - cached value); the accept test is exp(delta) > u as in
//       mcmc.js:527-528. This is the production ("fast") path: like the factorised plates it equals the reference's arithmetic
//       up to rounding (KS-level parity, as BASELINE.json states for real parameters); `faithful` handles never come here.
//
// The generated part of the translation unit (amwg_jit.cuh) comes first and defines the J* constants, the parameter and plate
// tables and the functions jit_step / jit_stat_extra / jit_derived used below.
#pragma once

namespace amwg {

struct JitArgs {
  ChainArrays a;
  SweepArgs sa;
  const double* col[JMAXCOL];        // the model's data columns in HBM
  const unsigned char* adapting;     // [JD] host-maintained (start/stop_adaptation)
};

// working-set rows of one chain (layout of amwg_create: [tval JNT | tcand JNT | bprop JD | bcoin JD] then state JD)
#define TV(t) wk[(unsigned long long)(t) * ws]
#define TC(t) wk[(unsigned long long)(JNT + (t)) * ws]
#define BP(c) wk[(unsigned long long)(2 * JNT + (c)) * ws]
#define BC(c) wk[(unsigned long long)(2 * JNT + JD + (c)) * ws]
#define ST(c) sp[(unsigned long long)(c) * ss]

// The Metropolis decision js_exp(dl) > coin, taken without the fdlibm exp wherever it is certain (AMWG_JIT_ACCEPT_SCREEN).
// 1 accept, 0 reject, -1 undecided: the caller then evaluates js_exp(dl) > coin itself. A lane that decides here skips the
// out-of-line exp; a warp skips it when all its lanes do. coin is a uniform in [0, 1), and > 0 means >= 2^-53.
//   * dl >= 0: js_exp(dl) >= 1 > coin (fdlibm returns 1 + dl below 2^-27 and is within 1 ulp of exp(dl) >= 1 + 2^-27 above).
//   * dl < -40 (-inf too), coin > 0: js_exp(dl) <= exp(-40) (1 + 2^-52) < 4.3e-18 < 2^-53 <= coin.
//   * -40 <= dl < 0: est = exp2f(t), t = (float)(dl * log2 e), |t| < 57.8. Relative error of est against exp(dl):
//       the double product and the constant log2 e   <= 2^-51      (negligible: < 3e-14 absolute in t)
//       rounding t to float (ulp <= 2^-18 below 64)  <= ln 2 * 2^-19 < 1.33e-6
//       exp2f (CUDA: 2 ulp; glibc: 1 ulp), est >= 2^-58 is a normal float: <= 2^-22 < 2.4e-7
//     so |est / exp(dl) - 1| < 1.6e-6, and js_exp(dl) is within 2^-52 of exp(dl). With the band B = 2^-16 (1.5e-5, nine times the
//     error): est > coin (1 + B) proves exp(dl) > coin; est < coin (1 - B) proves js_exp(dl) <= coin. The products coin (1 +- B)
//     round by 2^-53 relative, far inside the margin. A lane lands in the band with probability < 2 B.
//   * NaN dl, coin == 0 and the band: undecided. (NaN compares false throughout; js_exp(NaN) > coin then rejects.)
__device__ __forceinline__ int jit_accept_screen(const double dl, const double coin) {
  if (dl >= 0.0) return 1;
  if (!(coin > 0.0)) return -1;
  if (dl < -40.0) return 0;
  const double est = (double)exp2f((float)(dl * 1.4426950408889634));
  if (est > coin * (1.0 + 0x1p-16)) return 1;
  if (est < coin * (1.0 - 0x1p-16)) return 0;
  return -1;
}

}  // namespace amwg

#include "amwg_jit_generated.inc"

namespace amwg {

extern "C" __global__ void __launch_bounds__(JTHREADS, JMINB) amwg_jit_sweep(const __grid_constant__ JitArgs A) {
  extern __shared__ __align__(16) unsigned char smem[];
  __shared__ __align__(8) unsigned long long bar_res;
#if JSTREAM
  __shared__ __align__(8) unsigned long long ring_full[JRING_STAGES];
#endif
  const ChainArrays& a = A.a;
  const SweepArgs& sa = A.sa;
  const unsigned long long C = a.C;
  const unsigned long long tid = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = tid < C;                                   // threads past the last chain shadow chain C-1 and write nothing:
  const unsigned long long chain = valid ? tid : C - 1;         // they take part in the CTA-wide data pass and its barriers
  const unsigned long long gchain = a.first_chain + chain;

  // ---- stage the resident columns: one bulk-TMA copy each, one mbarrier for all
  if (threadIdx.x == 0) {
    mbar_init(&bar_res, 1);
#if JSTREAM
    for (int k = 0; k < JRING_STAGES; ++k) mbar_init(&ring_full[k], 1);
#endif
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
#if JN_RES > 0
  if (threadIdx.x == 0) {
    mbar_expect_tx(&bar_res, JRES_TOTAL_BYTES);
#pragma unroll
    for (int k = 0; k < JN_RES; ++k) tma_bulk_g2s(smem + JRES_OFF[k], A.col[JRES_COL[k]], JRES_BYTES[k], &bar_res);
  }
  mbar_wait(&bar_res, 0);
#endif

  // ---- the chain's working set: shared memory for small models (one column per thread, conflict-free), else the global rows
#if JWS_SMEM
  double* wk = reinterpret_cast<double*>(smem + JWS_OFF) + threadIdx.x;
  const unsigned long long ws = JTHREADS, ss = JTHREADS;
  double* sp = wk + (unsigned long long)(2 * JNT + 2 * JD) * ws;
  unsigned short* vq = reinterpret_cast<unsigned short*>(smem + JWS_OFF + (size_t)(2 * JNT + 3 * JD) * JTHREADS * sizeof(double)) + threadIdx.x;
  for (int t = 0; t < JNT; ++t) TV(t) = a.tval[(unsigned long long)t * C + chain];
  for (int c = 0; c < JD; ++c) ST(c) = a.state[(unsigned long long)c * C + chain];
  const bool wr = true;                                         // a shadow's shared column is its own
#else
  double* wk = a.tval + chain;
  const unsigned long long ws = C, ss = C;
  double* sp = a.state + chain;
  unsigned short* vq = a.vseq + chain;
  const bool wr = valid;
#endif

  RandomStream g;
  g.init(a.rng_n[chain]);
  unsigned long long perm = a.perm[chain];
#if JMAX_DIM0 > 1
  unsigned char order[JMAX_DIM0 < kLocalOrder ? JMAX_DIM0 : kLocalOrder];
#endif
#if JSTREAM
  unsigned ring_fills = 0;                                      // tiles streamed so far by this CTA (stage = fills % stages)
#endif

  long long rec_phase = sa.record ? sa.sample_i0 % sa.thin : 0;
  long long row = sa.record ? (sa.sample_i0 + sa.thin - 1) / sa.thin : 0;
  for (long long s = 0; s < sa.n_sweeps; ++s) {
    if (sa.record) {                                            // Sampler.sample: the state BEFORE stepping (mcmc.js:1021-1027)
      const bool rec_now = rec_phase == 0;
      if (++rec_phase == sa.thin) rec_phase = 0;
      if (rec_now && valid) {
#if JN_DERIVED > 0
        double der[JN_DERIVED];
        bool have_der = false;
#endif
        for (int j = 0; j < sa.n_monitor; ++j) {
          const int e = sa.monitor[j];
          double v;
          if (e < JD) {
            v = ST(e);
          } else {
#if JN_DERIVED > 0
            if (!have_der) { jit_derived(sp, ss, der); have_der = true; }
            v = der[e - JD];
#else
            v = CUDART_NAN;
#endif
          }
          sa.out[((unsigned long long)row * sa.n_monitor + j) * C + chain] = v;
        }
      }
      if (rec_now) ++row;
    }
    // ---- (a) this sweep's random numbers, in the reference's order
#if JP > 1
    for (int i = JP - 1; i > 0; --i) {                          // shuffle_array(this.substeppers), in place (mcmc.js:887, 228-236)
      const int j = (int)floor(g.next(a.seed, gchain) * (i + 1));
      perm_swap(a, perm, chain, i, j, valid);
    }
#endif
    int pos = 0;
#pragma unroll 1
    for (int slot = 0; slot < JP; ++slot) {
      const int p = (JP > 1) ? perm_get(a, perm, chain, slot) : 0;
      const int n_comp = jp_ncomp(p), off = jp_off(p), ptype = jp_type(p);
      const double lower = jp_lower(p), upper = jp_upper(p);
#if JMAX_DIM0 > 1
      const int dim0 = jp_dim0(p);
      const int inner = n_comp / dim0;
      if (n_comp > 1) {                                         // nested_array_random_apply: top level only (mcmc.js:246-252)
        for (int i = 0; i < dim0; ++i) ord_set(a, order, chain, dim0, i, i, valid);
        for (int i = dim0 - 1; i > 0; --i) {
          const int j = (int)floor(g.next(a.seed, gchain) * (i + 1));
          const int t = ord_get(a, order, chain, dim0, i);
          ord_set(a, order, chain, dim0, i, ord_get(a, order, chain, dim0, j), valid);
          ord_set(a, order, chain, dim0, j, t, valid);
        }
      }
#endif
#pragma unroll 1
      for (int r = 0; r < n_comp; ++r, ++pos) {
        int c = off;
#if JMAX_DIM0 > 1
        if (n_comp > 1) c += ord_get(a, order, chain, dim0, r / inner) * inner + (r % inner);
#endif
#if JBLOCK >= 0 && JBLOCK_FREE
        if (p == JBLOCK) {
          // an unbounded parameter always draws its accept uniform: the sweep's random numbers do not depend on its value or its
          // proposal scale. Only the ratio v / u of the accepted Leva trial is kept here; the proposal is finished below in index
          // order, where the rows of state and scale are read contiguously instead of one scattered row per lane.
          const double z = js_rnorm_ratio(g, a.seed, gchain);
          const double coin = g.next(a.seed, gchain);
          if (wr) { BP(c) = z; BC(c) = coin; }
          continue;
        }
#endif
        const double cur = ST(c);
        double prop = js_rnorm(g, a.seed, gchain, cur, a.psd[(unsigned long long)c * C + chain]);   // generate_proposal (mcmc.js:519, 577-579 / 596-598)
        if (ptype == AMWG_INT) prop = js_round(prop);
        const bool inb = !(prop < lower || prop > upper);       // bounds check (:520): no uniform when it fails
        const double coin = inb ? g.next(a.seed, gchain) : -1.0;
        if (wr) {
          BP(c) = inb ? prop : cur;
          BC(c) = coin;
          vq[(unsigned long long)pos * ws] = (unsigned short)c;
        }
      }
    }
#if JBLOCK >= 0 && JBLOCK_FREE
    {
      const int n_b = jp_ncomp(JBLOCK), off_b = jp_off(JBLOCK);
      const bool is_int = jp_type(JBLOCK) == AMWG_INT;
#pragma unroll 4
      for (int r = 0; r < n_b; ++r) {                           // (v / u) * sd + mean, the last two operations of rnorm (mcmc.js:53)
        const int c = off_b + r;
        double prop = BP(c) * a.psd[(unsigned long long)c * C + chain] + ST(c);
        if (is_int) prop = js_round(prop);
        if (wr) BP(c) = prop;
      }
    }
#endif
    // ---- (b) one pass over the data: every plate statistic at the proposals -> candidate slots
#if JN_RSTAT > 0
#pragma unroll 1
    for (int k = 0; k < JN_RSTAT; ++k) {                        // plates over resident columns whose mean is a component
      const double mean = BP(JR_COMP[k]);
      const unsigned sa0 = smem_u32(smem) + JR_SOFF[k];
      const double S = sum_sq_dev(reinterpret_cast<const double*>(smem + JR_SOFF[k]), sa0, JR_N[k], mean);
      if (wr) TC(JR_SLOT[k]) = S;
    }
#endif
    jit_stat_extra(smem, wk, ws, sp, ss, wr);                    // plates whose mean is an expression (generated)
#if JSTREAM
    {
      // the streamed column: plates JS_*[0..JN_SSTAT) tile it in order. Tile t+S-1 is issued at the top of iteration t, after the
      // CTA barrier that says everybody is done with tile t-1 (whose stage it reuses).
      const int nt = (JS_TOTAL + JRING_TILE - 1) / JRING_TILE;
      const double* gx = A.col[JS_COL] + JS_BEGIN;
      __syncthreads();                                          // the previous pass has drained: every stage is free
      if (threadIdx.x == 0)
        for (int t = 0; t < JRING_STAGES - 1 && t < nt; ++t) {
          const unsigned st = (ring_fills + (unsigned)t) % JRING_STAGES;
          const int cnt = min(JRING_TILE, JS_TOTAL - t * JRING_TILE);
          const unsigned bytes = (unsigned)((cnt * 8 + 15) & ~15);
          mbar_expect_tx(&ring_full[st], bytes);
          tma_bulk_g2s(smem + JRING_OFF + st * (JRING_TILE * 8), gx + (size_t)t * JRING_TILE, bytes, &ring_full[st]);
        }
      int pk = 0;
      double S = 0.0;
      double mean = BP(JS_COMP[0]);
      int pend = JS_END[0];
#pragma unroll 1
      for (int t = 0; t < nt; ++t) {
        __syncthreads();
        if (threadIdx.x == 0 && t + JRING_STAGES - 1 < nt) {
          const int t2 = t + JRING_STAGES - 1;
          const unsigned st = (ring_fills + (unsigned)t2) % JRING_STAGES;
          const int cnt = min(JRING_TILE, JS_TOTAL - t2 * JRING_TILE);
          const unsigned bytes = (unsigned)((cnt * 8 + 15) & ~15);
          mbar_expect_tx(&ring_full[st], bytes);
          tma_bulk_g2s(smem + JRING_OFF + st * (JRING_TILE * 8), gx + (size_t)t2 * JRING_TILE, bytes, &ring_full[st]);
        }
        const unsigned f = ring_fills + (unsigned)t;
        const unsigned st = f % JRING_STAGES;
        mbar_wait(&ring_full[st], (f / JRING_STAGES) & 1u);
        const int lo = t * JRING_TILE, hi = min(lo + JRING_TILE, JS_TOTAL);
        int p0 = lo;
        while (p0 < hi) {
          const int e = min(pend, hi);
          const unsigned boff = JRING_OFF + st * (JRING_TILE * 8) + 8u * (unsigned)(p0 - lo);
          S = S + sum_sq_dev(reinterpret_cast<const double*>(smem + boff), smem_u32(smem) + boff, e - p0, mean);
          p0 = e;
          if (p0 == pend) {
            if (wr) TC(JS_SLOT[pk]) = S;
            ++pk;
            S = 0.0;
            if (pk < JN_SSTAT) { mean = BP(JS_COMP[pk]); pend = JS_END[pk]; }
          }
        }
      }
      ring_fills += (unsigned)nt;
    }
#endif
    // ---- (c) the steps: O(1) each. Named parameters in the chain's substepper order, the components of a multi-dim parameter in its
    // visiting order -- with one exception. When the components of a (large) multi-dim parameter never share a term (JBLOCK: the
    // group means of a hierarchical model), every one of its decisions depends only on that component's own proposal, uniform and
    // terms: any order gives the same draws. Its steps are then taken in INDEX order by all chains of the warp at once, so that every
    // row access is contiguous (the visiting order is per chain: lanes would read 32 different rows), between the steps of the
    // parameters the chain visits before it and those it visits after it.
#if JBLOCK < 0
    {
      int c_next = (int)vq[0];
      double coin_next = BC(c_next), prop_next = BP(c_next);
#pragma unroll 1
      for (int i = 0; i < JD; ++i) {
        const int c = c_next;
        const double coin = coin_next, prop = prop_next;
        if (i + 1 < JD) {                                       // the next step's operands are on their way while this one is evaluated
          c_next = (int)vq[(unsigned long long)(i + 1) * ws];
          coin_next = BC(c_next); prop_next = BP(c_next);
        }
        if (!wr || coin < 0.0) continue;                        // out of bounds: rejected without evaluation (mcmc.js:520-522)
        if (jit_step(c, prop, coin, wk, ws, sp, ss) && valid && A.adapting[c])
          atomicAdd(&a.acc[(unsigned long long)c * C + chain], 1);        // acceptance_count (mcmc.js:530); result unused: a RED
      }
    }
#else
    {
      int pos_b = 0;
      for (int slot = 0; slot < JP; ++slot) if (((JP > 1) ? perm_get(a, perm, chain, slot) : 0) == JBLOCK) pos_b = slot;
#pragma unroll 1
      for (int part = 0; part < 3; ++part) {
        if (part == 1) {
          const int n_b = jp_ncomp(JBLOCK), off_b = jp_off(JBLOCK);
          double coin_next = BC(off_b), prop_next = BP(off_b);
#pragma unroll 1
          for (int r = 0; r < n_b; ++r) {
            const int c = off_b + r;
            const double coin = coin_next, prop = prop_next;
            if (r + 1 < n_b) { coin_next = BC(c + 1); prop_next = BP(c + 1); }
            if (!wr || coin < 0.0) continue;
            if (jit_step(c, prop, coin, wk, ws, sp, ss) && valid && A.adapting[c]) atomicAdd(&a.acc[(unsigned long long)c * C + chain], 1);
          }
          continue;
        }
        const int lo = part == 0 ? 0 : pos_b + 1, hi = part == 0 ? pos_b : JP;
        int pos0 = 0;
#pragma unroll 1
        for (int slot = 0; slot < JP; ++slot) {
          const int p = (JP > 1) ? perm_get(a, perm, chain, slot) : 0;
          const int n_comp = jp_ncomp(p);
          if (slot >= lo && slot < hi) {
            int c_next = (int)vq[(unsigned long long)pos0 * ws];
            double coin_next = BC(c_next), prop_next = BP(c_next);
#pragma unroll 1
            for (int r = 0; r < n_comp; ++r) {
              const int c = c_next;
              const double coin = coin_next, prop = prop_next;
              if (r + 1 < n_comp) {                             // the next step's operands are on their way while this one is evaluated
                c_next = (int)vq[(unsigned long long)(pos0 + r + 1) * ws];
                coin_next = BC(c_next); prop_next = BP(c_next);
              }
              if (!wr || coin < 0.0) continue;                  // out of bounds: rejected without evaluation (mcmc.js:520-522)
              if (jit_step(c, prop, coin, wk, ws, sp, ss) && valid && A.adapting[c])
                atomicAdd(&a.acc[(unsigned long long)c * C + chain], 1);      // acceptance_count (mcmc.js:530); result unused: a RED
            }
          }
          pos0 += n_comp;
        }
      }
    }
#endif
  }
  if (valid) {
    a.rng_n[chain] = g.n;
    a.perm[chain] = perm;
#if JWS_SMEM
    for (int t = 0; t < JNT; ++t) a.tval[(unsigned long long)t * C + chain] = TV(t);
    for (int c = 0; c < JD; ++c) a.state[(unsigned long long)c * C + chain] = ST(c);
#endif
  }
}

}  // namespace amwg
