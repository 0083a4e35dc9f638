/*
 * amwg.h -- C ABI of the B200-native many-chain AMWG sampler (libamwg_b200.so).
 *
 * The reference (rasmusab/bayes.js) has no FFI: its boundary is the JavaScript object API
 *     new mcmc.AmwgSampler(params, log_post, data, options)   mcmc.js:1090-1092, 940-966
 *     .burn(n) .sample(n) .step() .thin(k) .monitor(names)     mcmc.js:985-1055
 *     .start_adaptation() .stop_adaptation() .info()           mcmc.js:1060-1073, 977-980
 * This header is what the Node N-API addon (js/amwg_napi.cc, see INTEGRATION.md), the Python host (bayes.js_b200/_ffi.py) or any other host
 * binds instead.  Plain pointers and sizes only; every call returns 0 or a negative status and
 * amwg_last_error() gives the message the JS shim re-throws as a bare string (the reference
 * throws strings, mcmc.js:165,299,315,340,445,490,495,636,746,790,867,972).
 *
 * Calls block until the result is usable; a handle is not thread-safe (the reference is
 * single-threaded); all per-chain state stays resident in HBM between calls, so successive
 * burn()/sample() calls continue the same chains (mcmc.js:964-965, 509-511).
 *
 * A handle owns `n_chains` independent chains with global ids [first_chain, first_chain+n_chains).
 * Chain g behaves exactly like one run of the reference with Math.random() replaced by the
 * Philox4x32-10 stream (seed, g) defined in DESIGN.md "RNG contract"; results therefore do not
 * depend on how chains are sharded over handles / GPUs.
 */
#ifndef AMWG_H_
#define AMWG_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AMWG_ABI_VERSION 8
#define AMWG_MAX_BLOCK_PARAMS 4
#if defined(__GNUC__)
#define AMWG_API __attribute__((visibility("default")))
#else
#define AMWG_API
#endif

/* ---- parameters: one entry per key of the completed `params` object (mcmc.js:357-403) ---- */
enum { AMWG_REAL = 0, AMWG_INT = 1, AMWG_BINARY = 2 };

typedef struct {
  int32_t type;          /* AMWG_REAL | AMWG_INT | AMWG_BINARY                      (mcmc.js:844-868) */
  int32_t n_comp;        /* prod(dim): scalar components, flattened row-major                          */
  int32_t dim0;          /* dim[0]: the level visited in random order each sweep   (mcmc.js:244-263)  */
  int32_t comp_offset;   /* index of the first component in the flat state vector                     */
  double lower, upper;   /* bounds, +-inf allowed                                  (mcmc.js:497-498)  */
} amwg_param;

/* per scalar component: the options OnedimMetropolisStepper resolves (mcmc.js:500-505, 658-660) */
typedef struct {
  double prop_log_scale;       /* default 0    */
  double batch_size;           /* default 50   */
  double max_adaptation;       /* default 0.33 */
  double initial_adaptation;   /* default 1.0  */
  double target_accept_rate;   /* default 0.44 */
  int32_t is_adapting;         /* default 1    */
  int32_t _pad;
} amwg_comp_options;

/* ---- data: named fp64 columns (JS numbers); copied to the device at create ---- */
typedef struct {
  const double* values;
  int64_t n;
} amwg_column;

/* ---- log_post as a program --------------------------------------------------------------
 * log_post(state, data) (mcmc.js:958-960) arrives as a postfix program over an fp64 stack.
 * Instruction word (int32):
 *     bits  0-7   opcode
 *     bits  8-9   mode of operand A     0 = popped from the stack, 1 = consts[next word], 2 = state component [next word],
 *                                       3 = the opcode has no such operand
 *     bits 10-11  mode of operand B     (operands are named in source order: op(A, B, C, D))
 *     bits 12-13  mode of operand C
 *     bits 14-15  mode of operand D
 *     bit  16     ACC flag: the result is added to lp (lp = lp + result) instead of being pushed
 *     bit  17     STORE flag (only with ACC, or on PLATE): the value is also written to the chain's term cache; the term id
 *                 follows as the last extra word of the instruction
 *     bits 18-31  immediate `a` (const index, component, column, plate id ...)
 * Inline operand words follow the instruction word in consumption order: last operand first (D, C, B, A), which is
 * also the order stack operands are popped.  Further extra words are noted per opcode.
 * The accumulator `lp` starts at 0 and receives terms strictly in program order, so the sum is formed in the same
 * order as the JS `log_post += ...` statements.  Every arithmetic op is a single IEEE-754 fp64 operation (no FMA
 * contraction); LOG/EXP are the fdlibm algorithms V8's Math.log/Math.exp port; LD_* follow distributions.js operation
 * by operation (cited per opcode in csrc/amwg_ld.cuh).
 */
#define AMWG_MODE_STACK 0
#define AMWG_MODE_CONST 1
#define AMWG_MODE_COMP 2
#define AMWG_MODE_NONE 3
#define AMWG_WORD(op, mA, mB, mC, mD, acc, a) \
  ((int32_t)((uint32_t)(op) | ((uint32_t)(mA) << 8) | ((uint32_t)(mB) << 10) | ((uint32_t)(mC) << 12) | ((uint32_t)(mD) << 14) | \
             ((uint32_t)((acc) ? 1 : 0) << 16) | ((uint32_t)(a) << 18)))
#define AMWG_STORE_FLAG (1u << 17)
#define AMWG_MAX_IMMEDIATE 16383

enum {
  AMWG_OP_END = 0,
  AMWG_OP_CONST,        /* push consts[operand]                                             */
  AMWG_OP_COMP,         /* push state component `operand` (proposal value for the moved one) */
  AMWG_OP_DATA,         /* push columns[operand][next word]                                  */
  AMWG_OP_DATA_I,       /* push columns[operand][off + stride*i], i = plate point; next words: off, stride */
  AMWG_OP_COMP_I,       /* push state component base + (int)columns[operand][off + stride*i]; next words: off, stride, base */
  AMWG_OP_ADD, AMWG_OP_SUB, AMWG_OP_MUL, AMWG_OP_DIV, AMWG_OP_NEG,
  AMWG_OP_LOG, AMWG_OP_EXP, AMWG_OP_SQRT, AMWG_OP_ABS, AMWG_OP_POW,
  AMWG_OP_LT, AMWG_OP_LE, AMWG_OP_GT, AMWG_OP_GE, AMWG_OP_EQ, AMWG_OP_NE,   /* push 1.0 / 0.0 */
  AMWG_OP_AND, AMWG_OP_OR, AMWG_OP_NOT,
  AMWG_OP_SELECT,       /* pops b, a, c ; pushes c != 0 ? a : b                              */
  AMWG_OP_LGAMMA, AMWG_OP_LFACTORIAL, AMWG_OP_LCHOOSE, AMWG_OP_LBETA,   /* distributions.js:63-92 */
  AMWG_OP_LD_NORM, AMWG_OP_LD_UNIF, AMWG_OP_LD_BETA, AMWG_OP_LD_BERN, AMWG_OP_LD_POIS,
  AMWG_OP_LD_CAUCHY, AMWG_OP_LD_LAPLACE, AMWG_OP_LD_GAMMA, AMWG_OP_LD_INVGAMMA, AMWG_OP_LD_LNORM,
  AMWG_OP_LD_PARETO, AMWG_OP_LD_T, AMWG_OP_LD_WEIBULL, AMWG_OP_LD_LOGIS, AMWG_OP_LD_EXP,
  AMWG_OP_LD_BINOM, AMWG_OP_LD_NBINOM, AMWG_OP_LD_HYPER,
  AMWG_OP_ACC,          /* lp = lp + pop                                                     */
  AMWG_OP_PLATE,        /* lp = plate[operand](lp, popped operands): a recognised O(N) likelihood sum */
  AMWG_OP_STORE,        /* derived[operand] = pop   (derived-quantity program only)          */
  AMWG_OP_LOOP_BEGIN,   /* start of a GENERIC plate body: i = 0 (plate[a].n points); next word: offset to continue at when n == 0 */
  AMWG_OP_LOOP_END,     /* lp = lp + pop; if (++i < n) jump to the word offset in the next word (first word of the body) */
  /* ld.* with constant hyper-parameters, partially evaluated by the host: the constant parts are folded once on the device
   * (fold table), the rest is the same operations in the same order as distributions.js -> same bits as the LD_* opcode. */
  AMWG_OP_NORM_K,       /* (x, mean, K1, K2): K1 - pow(x-mean,2)/K2,  K1 = -0.5*log(2pi) - log(sd), K2 = 2*sd*sd   (:119-121) */
  AMWG_OP_UNIF_K,       /* (x, min, max, K):  (x<min || x>max) ? -inf : K,  K = log(1/(max-min))                    (:221-223) */
  AMWG_OP_BETA_K,       /* (x, a1, b1, K):    (x>1 || x<0) ? -inf : a1*log(x) + b1*log(1-x) - K, a1 = shape1-1, b1 = shape2-1, K = lbeta (:104-113) */
  AMWG_OP_ACC_RANGE,    /* lp = lp + cache[a] + cache[a+1] + ... (next word: count), one term at a time, in order: the terms of the
                           sum that do not read the moved component, taken from the chain's term cache (see amwg_model.comp_prog) */
  /* Pre-evaluated plate statistics (see amwg_model.stat_prog). A NORM_IID plate is  f(S, sd) = n*(-0.5*log(2pi) - log(sd)) - S/(2*sd*sd)
   * with S = sum_i (x_i - mean)^2 -- the O(N) part, which only depends on the mean operand. */
  AMWG_OP_PLATE_SS,     /* (mean): push S of plate `a`; next word: the statistic's slot in the term cache, S is stored there too */
  AMWG_OP_NORM_SS,      /* (S, sd): f(S, sd) of plate `a` (same operations as AMWG_PLATE_NORM_IID, given its S)                */
  AMWG_OP_CACHED,       /* push cache[a]      : the committed value of slot a (a statistic of the chain's current state)       */
  AMWG_OP_CAND,         /* push candidate[a]  : the value the last stat_prog evaluation computed for slot a (at the proposals)   */
  AMWG_OP__COUNT
};

/* A plate is a run of N structurally identical likelihood terms, `for (i...) log_post += ld.X(data[i], ...)`.
 * Recognised shapes get a hand-written inner loop (AMWG_OP_PLATE; their index-free operands are evaluated by
 * the program and popped from the stack); anything else is a bytecode loop over its body
 * (AMWG_OP_LOOP_BEGIN ... AMWG_OP_LOOP_END, body uses DATA_I / COMP_I), bit-faithful to the JS loop. */
enum {
  AMWG_PLATE_GENERIC = 0,   /* bytecode loop: lp += body(i), i = 0..n-1, in order                                   */
  AMWG_PLATE_NORM_IID,      /* operands A = mean, B = sd.  sum_i ld.norm(x_i, mean, sd), factorised:
                               N*(-0.5*log(2pi) - log(sd)) - sum_i (x_i-mean)^2 / (2*sd*sd)     (KS-level parity)   */
  AMWG_PLATE_BERN_IID,      /* operand A = p.  sum_i ld.bern(y_i, p), sequential, bit-faithful                       */
  AMWG_PLATE_NORM_GROUPED,  /* operand A = sd.  sum_i ld.norm(y_i, mu[g_i], sd); points sorted by group              */
  AMWG_PLATE_POIS_LOGLIN    /* sum_i ld.pois(y_i, exp(sum_k X_ik * beta_k)) = beta . (X^T y) - sum_i exp(X_i . beta) - sum_i lfactorial(y_i):
                               the linear part and the constant come precomputed (col[2]), the device sums the exponentials.
                               K in {1..8, 10, 12, 16}                                           (KS-level parity)   */
};

typedef struct {
  int32_t kind;          /* AMWG_PLATE_*                                                          */
  int32_t n;             /* number of points                                                       */
  int32_t col[4];        /* data columns: [0] x or y; GROUPED: [1] group start offsets (J+1);
                            POIS_LOGLIN: [1] X row-major n*K, [2] K+1 values filled by the host: X^T y, then sum_i lfactorial(y_i) */
  int32_t iparam[4];     /* GROUPED: [0] first mu component, [1] J;  POIS_LOGLIN: [0] first beta component, [1] K;
                            all specialised kinds: [2] offset of the plate's first point inside col[0]              */
} amwg_plate;

typedef struct {
  int32_t abi_version;                     /* AMWG_ABI_VERSION */
  int32_t n_params;   const amwg_param* params;
  int32_t n_comp;     const double* init;                  /* params[*].init flattened, length n_comp */
  const amwg_comp_options* comp_options;                   /* length n_comp (ignored for binary)      */
  int32_t n_code;     const int32_t* code;                 /* all programs, concatenated              */
  int32_t logpost_prog;                                    /* word offset of the log_post program     */
  int32_t derived_prog;                                    /* word offset of the derived program, -1  */
  int32_t n_derived;                                       /* derived quantities (state keys beyond params, mcmc.js:990) */
  int32_t n_consts;   const double* consts;
  int32_t n_columns;  const amwg_column* columns;
  int32_t n_plates;   const amwg_plate* plates;
  /* Constant sub-expressions (no parameter, no plate index) are evaluated ONCE on the device at create, with the
   * device's own arithmetic, and stored into consts[fold_dst[k]]: fold_prog[k] is the word offset of an
   * END-terminated expression program.  (log(2*pi), log(sd) of a constant sd, ... : same bits, computed once.) */
  int32_t n_fold;     const int32_t* fold_prog;  const int32_t* fold_dst;
  /* Control flow on binary parameters (`if (m === 0) ... else ...`, tests/test_data.js:163-168) cannot be recorded as one
   * expression, so the host records log_post once per configuration of up to AMWG_MAX_VARIANT_COMPS binary components.
   * Configuration v has bit k set when state component variant_comps[k] is non-zero (the proposal counts for the moved one);
   * its programs start at variant_logpost[v] / variant_derived[v]. n_variant_comps == 0: logpost_prog / derived_prog are used. */
  /* Dependency-aware evaluation (optional). log_post is a sum of terms; a step that moves component c only changes the terms
   * that read c. With comp_prog != NULL the sampler keeps every value-term of every chain in a term cache (n_terms doubles per
   * chain) and evaluates a proposal for component c with comp_prog[c]: the terms that read c are recomputed (STORE flag: the new
   * value goes to a candidate slot), the others are added from the cache by ACC_RANGE -- each in its original position, so the
   * sum is formed in the same order with the same values as the full program (bit-identical). On acceptance the candidates of
   * touch_terms[touch_off[c] .. touch_off[c+1]) are committed. logpost_prog is the full program (it stores every value-term). */
  int32_t n_terms;          const int32_t* comp_prog;      /* n_comp word offsets, or NULL */
  const int32_t* touch_off; const int32_t* touch_terms;    /* n_comp + 1 offsets into touch_terms */
  /* Block steps (optional, needs comp_prog). A multi-dim parameter whose components never share a term (every term reads at most
   * one of them: the group means of a hierarchical model) can be stepped with ONE evaluation of the full program: the proposals
   * (and accept uniforms) of all its components are drawn first, in the chain's random visiting order, the program is evaluated
   * with all of them in place (every term's candidate value lands in the term cache), and the accept decisions are then taken one
   * component at a time in visiting order from the cached terms -- the same sums, values and uniforms as stepping them one by
   * one. block_params lists such parameters (indices into params[]); term_block_comp[k * n_terms + t] is the component of
   * block_params[k] that term t reads, or -1. */
  int32_t n_block_params;   const int32_t* block_params;   const int32_t* term_block_comp;
  /* Pre-evaluated statistics (optional, needs comp_prog; no binary parameter, no variants). When every O(N) plate is a NORM_IID
   * plate whose mean reads exactly ONE component, the expensive part of a proposal's evaluation -- S at the proposed value of that
   * component -- does not depend on how the other steps of the sweep turn out, and neither do the sweep's random numbers (a step
   * consumes its rnorm trials and, if the proposal is in bounds, one uniform, whatever log_post says: mcmc.js:519-528). So a sweep
   * is run as: (a) draw every step's proposal and accept uniform, in the chain's visiting order; (b) ONE pass over the data:
   * stat_prog evaluates every statistic at the proposals (candidate slots n_sum_terms .. n_terms-1 of the term cache);
   * (c) the steps, in visiting order, each with comp_prog[c] -- which now contains no O(N) work: a plate term is NORM_SS of
   * CAND(slot) (the moved component is the plate's mean) or CACHED(slot) (it is not). Same values, same sums, same uniforms as
   * stepping with the full program, at one data pass per sweep instead of one per step. The term cache then has n_terms slots of
   * which the first n_sum_terms are terms of the sum (ACC_RANGE only ever covers those); without stat_prog n_sum_terms == n_terms. */
  int32_t stat_prog;        int32_t n_sum_terms;           /* stat_prog: word offset, -1 = not in use */
  int32_t n_variant_comps;  const int32_t* variant_comps;
  const int32_t* variant_logpost;  const int32_t* variant_derived;     /* 1 << n_variant_comps entries each (derived: -1 if none) */
} amwg_model;
#define AMWG_MAX_VARIANT_COMPS 4

typedef struct amwg_sampler amwg_sampler;

/* new mcmc.AmwgSampler(...) for n_chains chains on CUDA device `device` (mcmc.js:1090-1092, 940-966):
 * uploads the model, places every chain at params[*].init and evaluates log_post once. */
AMWG_API int amwg_create(const amwg_model* model, uint64_t n_chains, uint64_t first_chain, uint64_t seed,
                int device, amwg_sampler** out);
AMWG_API void amwg_destroy(amwg_sampler* s);

/* sampler.burn(n) -- mcmc.js:1035-1039 */
AMWG_API int amwg_burn(amwg_sampler* s, int64_t n);

/* sampler.sample(n) with thinning interval `thin` and the monitored entries `monitor[n_monitor]`
 * (index < n_comp: state component; n_comp + d: derived quantity d) -- mcmc.js:1005-1030.
 * Row r is the state BEFORE sweep r*thin (row 0 is the pre-existing state, mcmc.js:1021-1027).
 * Output layout: out[row][monitor][chain], fp64, rows = ceil(n/thin).
 *   amwg_sample        : host buffer (pinned memory recommended); D2H copies overlap the sweeps.
 *   amwg_sample_device : device buffer on the handle's device; no host traffic. */
AMWG_API int amwg_sample(amwg_sampler* s, int64_t n, int64_t thin, const int32_t* monitor, int32_t n_monitor, double* host_out);
AMWG_API int amwg_sample_device(amwg_sampler* s, int64_t n, int64_t thin, const int32_t* monitor, int32_t n_monitor, double* dev_out);

/* live state, as sampler.step() returns it (mcmc.js:985-997): out[entry][chain], entries = n_comp + n_derived */
AMWG_API int amwg_get_state(amwg_sampler* s, double* host_out);

/* sampler.log_post() -- the closure the Sampler ctor stores (mcmc.js:958-960): log_post at the chain's current state, out[chain] */
AMWG_API int amwg_get_log_post(amwg_sampler* s, double* host_out);

/* sampler.start_adaptation() / stop_adaptation() -- mcmc.js:1060-1073 */
AMWG_API int amwg_set_adapting(amwg_sampler* s, int32_t flag);

/* stepper info() (mcmc.js:563-571): per component, chain-invariant counters and per-chain arrays.
 * scalars[c*3 + {0,1,2}] = is_adapting, iterations_since_adaption, batch_count  (host, length 3*n_comp)
 * prop_log_scale[c][chain], acceptance_count[c][chain] (host; either may be NULL) */
AMWG_API int amwg_info(amwg_sampler* s, double* scalars, double* prop_log_scale, int32_t* acceptance_count);

/* instrumentation */
AMWG_API int64_t amwg_kernel_launches(const amwg_sampler* s);   /* kernels this handle has launched so far       */
AMWG_API double amwg_last_sweep_kernel_ms(const amwg_sampler* s); /* CUDA-event time of the sweep kernels of the last burn/sample call */
AMWG_API uint64_t amwg_n_chains(const amwg_sampler* s);

AMWG_API const char* amwg_last_error(void);
AMWG_API int amwg_abi_version(void);

/* ld.* evaluated on the device, one value per input row (used by the `ld` host module and by the
 * parity tests): op is an AMWG_OP_LD_* / AMWG_OP_LGAMMA.. opcode, args is [n][arity] row-major. */
AMWG_API int amwg_ld_eval(int32_t op, const double* args, int32_t arity, int64_t n, double* out, int device);

/* Math.log / Math.exp / the Philox uniform stream on the device, for parity tests of the primitives.
 * kind: 0 log, 1 exp, 2 stream uniform (x[i] reinterpreted: out[i] = uniform #i of chain `chain`), 3 rnorm(x[0], x[1]) draws of
 * one chain, 4 Math.round, 5 the Poisson plate's table-driven exp (KS-level path; accuracy test) */
AMWG_API int amwg_primitive_eval(int32_t kind, const double* x, int64_t n, uint64_t seed, uint64_t chain, double* out, int device);

/* ---- post-path reductions on device (SURVEY 8(f).3) ------------------------------------------------------------------
 * The reference returns raw draws only (mcmc.js:1029; README.md:44-52 leaves the summary to the caller). With millions of
 * chains the summary is formed where the draws are. Both calls read a DEVICE-resident sample block in amwg_sample_device's
 * layout, x[row][entry][chain]; neither needs a sampler handle (they are reductions over the block).
 *
 * amwg_summary_moments: host_stats[entry][4] = { chains, mean of the per-chain means, M2 of the per-chain means
 *   (sum_c (m_c - mean)^2), sum over chains of the within-chain M2 (sum_r (x_rc - m_c)^2) }, merged in a fixed order
 *   (deterministic). Pooled mean / sd and the Gelman-Rubin statistic follow from these; shards (multi-GPU) merge exactly.
 *
 * amwg_summary_digit_hist: one pass (0..7, most significant byte first) of an exact radix select over the order-preserving
 *   64-bit key of the draws: dev_counts[entry][prefix][256] += number of values of `entry` whose key's top 8*pass bits equal
 *   dev_prefix[entry][prefix] and whose next byte is the bin (pass 0 ignores the prefixes). Integer counts: exact and
 *   order-independent; the caller sums them over GPUs, picks the byte holding each wanted order statistic and extends the
 *   prefixes. n_prefix <= 32.
 *
 * amwg_summary_autocov: split-chain autocovariance sums for the effective sample size. Per chain h = rows / 2; the half-chains are
 *   the first and the last h rows (the middle row of an odd `rows` is dropped). y = x, or y = (x <= dev_threshold[entry] ? 1 : 0)
 *   when dev_threshold (DEVICE, [entries]) is not NULL. For each live entry i (host_live[i], or every entry when host_live is
 *   NULL) host_out[i][3 + n_lags] = { half-chains M', mean of the half-chain means, M2 of the half-chain means,
 *   S_t for t = lag0 .. lag0 + n_lags - 1 }, S_t = sum over half-chains of sum_{n=0}^{h-1-t} (y_n - ybar)(y_{n+t} - ybar), ybar the
 *   half-chain's mean (0 when t >= h). Merged in a fixed order (deterministic); a lag's sum has the same bits whatever lag0 and
 *   n_lags. Shards merge like amwg_summary_moments records, with the S_t added. 8 <= rows < 2^31 - 64, 1 <= n_lags <= 16. */
AMWG_API int amwg_summary_moments(int device, const double* dev_samples, int64_t rows, int32_t entries, int64_t chains, double* host_stats);
AMWG_API int amwg_summary_digit_hist(int device, const double* dev_samples, int64_t rows, int32_t entries, int64_t chains, int32_t pass,
                                     const uint64_t* dev_prefix, int32_t n_prefix, uint64_t* dev_counts);
AMWG_API int amwg_summary_autocov(int device, const double* dev_samples, int64_t rows, int32_t entries, int64_t chains,
                                  const double* dev_threshold, const int32_t* host_live, int32_t n_live, int32_t lag0, int32_t n_lags,
                                  double* host_out);

/* ---- rank normalisation (sample_summary(rank=True)) ------------------------------------------------------------------------
 * The exact pooled average rank of every split draw of one entry, and z = Phi^-1((r - 3/8) / (S + 1/4)) (Vehtari et al. 2021),
 * in five steps that the caller chains (and, across GPUs, interleaves with an exchange of the runs: summary.py). All pointers
 * named dev_ are DEVICE memory owned by the caller; keys are the order-preserving 64-bit keys of amwg_summary_digit_hist, with
 * -0 canonicalised to +0 (so -0 and +0 tie). n (keys, draws) must be 1 <= n < 2^32; the library's own scratch is about
 * n / 4 bytes during a sort, released when the call ends (only scratch up to 64 MiB is kept between calls). Every call returns
 * after its work is complete.
 *
 * amwg_summary_rank_keys: the split draws of `entry` (per chain h = rows / 2: the first and the last h rows; the middle row of an
 *   odd `rows` is dropped), S = 2h * chains of them, folded to |x - *host_center| when host_center is not NULL ->
 *   dev_keys[S] and dev_vals[S] = r' * chains + c, the position in a split block [2h][chains] (r' = 0 .. 2h - 1).
 * amwg_summary_rank_sort: stable LSD radix sort of the (key, u32) pairs by the key, 8-bit digits. One read histograms all eight
 *   digits; a pass whose digit is the same for every key is skipped. host_passes[3] = { passes run, passes skipped, 1 when the
 *   sorted pairs are in dev_keys_alt / dev_vals_alt (an odd number of passes ran), else 0 }. 24 bytes per key in all.
 * amwg_summary_rank_runs: run-length encoding of sorted keys: dev_run_id[n] = the run of each position, dev_run_keys[runs] (may
 *   be NULL) the distinct keys, dev_run_counts[runs] their counts, or, when dev_weights is not NULL, the sum over the run of
 *   dev_weights[dev_sorted_vals[i]] (the payloads index the weights; dev_sorted_vals may be NULL otherwise) and dev_weight_scan[n]
 *   is the caller's scratch for their prefix sums (NULL without weights). *host_n_runs = runs.
 * amwg_summary_rank_z: dev_run_z[i] = Phi^-1((r_i - 3/8) / (total + 1/4)) with the average 1-based rank
 *   r_i = offset + (counts of the runs before i) + (count_i + 1) / 2. 0 <= offset, 1 <= total < 2^50. CUDA's normcdfinv.
 *   dev_run_z must not overlap dev_run_counts (the counts are scanned in dev_run_z first).
 * amwg_summary_rank_scatter: dev_out[((p / chains) * entries + entry) * chains + p % chains] = dev_run_z[dev_run_id[i]] with
 *   p = dev_sorted_vals[i]: the z of each draw into a block [2h][entries][chains] (entries = 1, chains = n: dev_out[p]). */
AMWG_API int amwg_summary_rank_keys(int device, const double* dev_samples, int64_t rows, int32_t entries, int64_t chains, int32_t entry,
                                    const double* host_center, uint64_t* dev_keys, uint32_t* dev_vals);
AMWG_API int amwg_summary_rank_sort(int device, uint64_t* dev_keys, uint32_t* dev_vals, int64_t n, uint64_t* dev_keys_alt,
                                    uint32_t* dev_vals_alt, int32_t* host_passes);
AMWG_API int amwg_summary_rank_runs(int device, const uint64_t* dev_sorted_keys, const uint32_t* dev_sorted_vals, const int64_t* dev_weights,
                                    int64_t* dev_weight_scan, int64_t n, uint32_t* dev_run_id, uint64_t* dev_run_keys, int64_t* dev_run_counts,
                                    int64_t* host_n_runs);
AMWG_API int amwg_summary_rank_z(int device, const int64_t* dev_run_counts, int64_t n_runs, int64_t offset, int64_t total, double* dev_run_z);
AMWG_API int amwg_summary_rank_scatter(int device, const uint32_t* dev_sorted_vals, const uint32_t* dev_run_id, int64_t n,
                                       const double* dev_run_z, double* dev_out, int32_t entries, int64_t chains, int32_t entry);

/* ---- run-time specialisation ----------------------------------------------------------------------------------------------
 * For models that run the statistics sweep (stat_prog) amwg_create generates CUDA source from the model's programs, compiles it
 * for sm_100a with NVRTC and steps with that kernel instead of the bytecode interpreter (csrc/amwg_jit.cuh; AMWG_JIT=0 in the
 * environment keeps the interpreter, AMWG_JIT=1 specialises whatever the number of chains). amwg_jit_status: 1 when the handle
 * runs a specialised kernel, with a one-line description (or the reason it does not) in `note`. amwg_jit_compile_check: generate
 * and compile without a GPU (0 compiled, 1 model not eligible, -1 error; message in `log`, generated source in `src`). */
AMWG_API int amwg_jit_status(const amwg_sampler* s, char* note, int64_t cap);
AMWG_API int amwg_jit_compile_check(const amwg_model* model, uint64_t n_chains, char* log, int64_t log_cap, char* src, int64_t src_cap);

/* ---- measurement ---------------------------------------------------------------------------------------------------------
 * The binding roof of this path is the non-tensor fp64 pipe (DADD + DFMA per data point), which MEASURED_PEAKS.json does not
 * hold: amwg_peak_fp64 measures it (TFLOP/s, 2 flop per DFMA; best of `reps` launches of a DFMA-chain kernel that fills every SM,
 * CUDA events on the launching stream). bench.py reports roofline fractions against this number, taken in the same process. */
AMWG_API int amwg_peak_fp64(int device, int reps, double* tflops_out, double* ms_out);

#ifdef __cplusplus
}
#endif
#endif /* AMWG_H_ */
