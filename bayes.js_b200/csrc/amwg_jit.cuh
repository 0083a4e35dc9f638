// amwg_jit.cuh -- run-time specialisation of the statistics sweep (host side). Included into amwg_kernels.cu.
//
// The ABI hands log_post over as bytecode (include/amwg.h). For the interpreter kernels that bytecode is data; here it is
// SOURCE: the programs of a model eligible for pre-evaluated plate statistics (amwg_model.stat_prog) are decoded, turned into
// straight-line CUDA C++ (one function per class of structurally identical component programs, indices that differ between the
// members of a class read from small tables), joined with the kernel skeleton amwg_jit_kernel.cuh and compiled for sm_100a by
// NVRTC (dlopen'ed: the library loads without it; a model that cannot be specialised runs on the interpreter kernels -- there
// is still no CPU path). The cubin is loaded through the runtime's library API (cudaLibraryLoadData), cached per process by
// source hash. What the generated step computes differs from the interpreter's in one respect (DESIGN.md section 2): it forms
// log_post(proposal) - log_post(current) as a sum of per-term differences instead of re-adding every cached term in order.
#pragma once
#include <dlfcn.h>
#include <array>
#include <map>
#include <mutex>
#include <regex>
#include <set>
#include <sstream>

namespace jit {

// ---- bytecode decoder (the encoding of include/amwg.h, as run_program_t consumes it) ---------------------------------------
struct Insn {
  int pc = 0, next = 0;
  int op = 0, a = 0;
  bool acc = false, store = false;
  int mode[4] = {AMWG_MODE_NONE, AMWG_MODE_NONE, AMWG_MODE_NONE, AMWG_MODE_NONE};   // operands A..D as the instruction uses them
  int inl[4] = {-1, -1, -1, -1};       // inline word of operand A..D (const index / component), when its mode is CONST / COMP
  int extra[3] = {0, 0, 0};
  int n_extra = 0;
  int term = -1;                       // term id of the STORE flag
  int pops = 0, pushes = 0;
};

static bool has_result(int op) {
  switch (op) {
    case AMWG_OP_ACC: case AMWG_OP_ACC_RANGE: case AMWG_OP_PLATE: case AMWG_OP_LOOP_BEGIN: case AMWG_OP_LOOP_END:
    case AMWG_OP_STORE: case AMWG_OP_END: return false;
    default: return true;
  }
}

// Decode the instruction at word `pc`. Returns false (with `err`) when the word stream is malformed.
static bool decode(const amwg_model* md, int pc, Insn& in, std::string& err) {
  const int32_t* code = md->code;
  const int n = md->n_code;
  auto need = [&](int k) { if (pc + k > n) { err = "program runs past the end of the code"; return false; } return true; };
  in = Insn();
  in.pc = pc;
  if (!need(1)) return false;
  const unsigned w = (unsigned)code[pc++];
  in.op = (int)(w & 0xff);
  in.acc = (w >> 16) & 1;
  in.store = (w & AMWG_STORE_FLAG) != 0;
  in.a = (int)(w >> 18);
  if (in.op < 0 || in.op >= AMWG_OP__COUNT) { err = "unknown opcode"; return false; }
  int used[4] = {0, 0, 0, 0};                                 // which operand slots this instruction consumes
  if (in.op == AMWG_OP_PLATE) {
    if (in.a >= md->n_plates) { err = "plate index out of range"; return false; }
    const int kind = md->plates[in.a].kind;
    if (kind == AMWG_PLATE_NORM_IID) { used[0] = used[1] = 1; }
    else if (kind == AMWG_PLATE_BERN_IID || kind == AMWG_PLATE_NORM_GROUPED) { used[0] = 1; }
  } else {
    for (int k = 0; k < 4; ++k) used[k] = ((w >> (8 + 2 * k)) & 3) != AMWG_MODE_NONE;
  }
  for (int k = 3; k >= 0; --k) {                              // consumption order: last operand first
    if (!used[k]) continue;
    const int m = (w >> (8 + 2 * k)) & 3;
    in.mode[k] = m;
    if (m == AMWG_MODE_STACK) in.pops++;
    else if (m == AMWG_MODE_NONE) { err = "plate operand without a mode"; return false; }
    else { if (!need(1)) return false; in.inl[k] = code[pc++]; }
  }
  auto take = [&](int k) { if (!need(k)) return false; for (int j = 0; j < k; ++j) in.extra[in.n_extra++] = code[pc++]; return true; };
  switch (in.op) {
    case AMWG_OP_DATA: if (!take(1)) return false; break;
    case AMWG_OP_DATA_I: if (!take(2)) return false; break;
    case AMWG_OP_COMP_I: if (!take(3)) return false; break;
    case AMWG_OP_PLATE_SS: case AMWG_OP_ACC_RANGE: case AMWG_OP_LOOP_BEGIN: if (!take(1)) return false; break;
    case AMWG_OP_LOOP_END: if (!take(1)) return false; in.pops++; break;
    case AMWG_OP_ACC: case AMWG_OP_STORE: in.pops++; break;
    default: break;
  }
  if (has_result(in.op)) {
    if (in.acc) { if (in.store) { if (!need(1)) return false; in.term = code[pc++]; } }
    else in.pushes = 1;
  } else if (in.op == AMWG_OP_PLATE && in.store) {
    if (!need(1)) return false;
    in.term = code[pc++];
  }
  in.next = pc;
  return true;
}

// Decode a whole program (to its END); also reports the deepest operand stack it needs.
static bool decode_program(const amwg_model* md, int pc, std::vector<Insn>& out, int* max_depth, std::string& err) {
  out.clear();
  int depth = 0, deepest = 0;
  if (pc < 0 || pc >= md->n_code) { err = "program offset out of range"; return false; }
  for (int guard = 0; guard < md->n_code + 1; ++guard) {
    Insn in;
    if (!decode(md, pc, in, err)) return false;
    depth -= in.pops;
    if (depth < 0) { err = "operand stack underflow"; return false; }
    depth += in.pushes;
    deepest = std::max(deepest, depth);
    out.push_back(in);
    if (in.op == AMWG_OP_END) { if (max_depth) *max_depth = deepest; return true; }
    pc = in.next;
  }
  err = "program has no END";
  return false;
}

// ---- text helpers --------------------------------------------------------------------------------------------------------------
static std::string lit(double v) {
  if (v != v) return "CUDART_NAN";
  if (v == INFINITY) return "CUDART_INF";
  if (v == -INFINITY) return "(-CUDART_INF)";
  char buf[64];
  snprintf(buf, sizeof buf, "%a", v);                         // hex float: exact
  std::string s(buf);
  if (v < 0 || (v == 0 && std::signbit(v))) s = "(" + s + ")";
  return s;
}
static std::string istr(long long v) { return std::to_string(v); }
static std::string bits(double v) {                            // the value's bit pattern: table initialisers must be constant expressions
  long long b;
  memcpy(&b, &v, 8);
  return std::to_string(b) + "LL";
}

struct Plan {                                                  // shared-memory plan and launch shape of one specialisation
  int threads = 128, minblocks = 7;
  int n_res = 0;                                               // resident columns
  std::vector<int> res_col, res_off, res_bytes;
  std::vector<int> col_smem_off;                               // per model column: byte offset in smem, -1 not resident
  int stream_col = -1;                                         // the one column streamed through the tile ring, -1: none
  int ring_off = 0, ring_stages = 4, ring_tile = 1024;         // tile in doubles
  int ws_smem = 0, ws_off = 0;
  unsigned smem_bytes = 0;
  std::vector<int> bern_mask_off;                              // per plate: byte offset of a BERN_IID plate's bit mask in smem, -1 none (full-program form)
};

struct Source {
  bool full = false;                                           // amwg_jit_full_kernel.cuh instead of amwg_jit_kernel.cuh
  std::string generated;                                       // "amwg_jit_generated.inc"
  std::string prelude;                                         // the #defines and tables that precede the skeleton
  Plan plan;
};

static const int kMaxGeneratedInsns = 6000;                    // beyond this the straight-line code would thrash the instruction cache
static const unsigned kResidentBudget = 64u * 1024u;           // columns staged in shared memory per CTA
static const unsigned kJitWsSmemLimit = 20u * 1024u;           // working set kept in shared memory up to this many bytes per CTA

// One straight-line function body under construction: operand stack of C expressions + text-level common-subexpression reuse
struct Emitter {
  std::ostringstream os;
  std::map<std::string, std::string> cse;
  std::vector<std::string> stk;
  std::vector<std::map<std::string, std::string>> scopes;     // values named inside a generated loop are not visible after it
  int nv = 0;
  std::string tmp(const std::string& rhs) {
    auto it = cse.find(rhs);
    if (it != cse.end()) return it->second;
    std::string name = "v" + std::to_string(nv++);
    os << "    const double " << name << " = " << rhs << ";\n";
    cse[rhs] = name;
    return name;
  }
};

// The instances a piece of generated code stands for: the members of a class of structurally identical component programs
// (index variable `m`), or the iterations of a run of structurally identical terms inside one program (index variable `j`).
// A field that is the same in every instance becomes a literal, one that differs a lookup in a small table `T<k>[ix]`.
struct Inst {
  std::vector<Insn> ins;
  int moved = -1;                                              // the component this instance steps (-1: none, e.g. stat / derived code)
};
struct GenCtx {
  const amwg_model* md = nullptr;
  const Plan* plan = nullptr;                                  // shared-memory offsets of the resident columns (full-program code)
  const std::vector<double>* consts = nullptr;                 // constants with the device-folded values filled in
  std::ostringstream* tables = nullptr;                        // where the integer tables are emitted
  int* table_counter = nullptr;
  std::string field(const std::vector<int>& vals, const std::string& ix, bool* same = nullptr, int* value0 = nullptr) const {
    bool eq = true;
    for (int v : vals) eq = eq && v == vals[0];
    if (same) *same = eq;
    if (value0) *value0 = vals[0];
    if (eq) return std::to_string(vals[0]);
    const int id = (*table_counter)++;
    (*tables) << "__device__ const int T" << id << "[" << vals.size() << "] = {";
    for (size_t i = 0; i < vals.size(); ++i) (*tables) << (i ? "," : "") << vals[i];
    (*tables) << "};\n";
    return "T" + std::to_string(id) + "[" + ix + "]";
  }
  std::string dfield(const std::vector<double>& vals, const std::string& ix) const {     // the same for a derived double (plate sizes)
    bool eq = true;
    for (double v : vals) eq = eq && v == vals[0];
    if (eq) return lit(vals[0]);
    const int id = (*table_counter)++;
    (*tables) << "__device__ const double T" << id << "[" << vals.size() << "] = {";
    for (size_t i = 0; i < vals.size(); ++i) (*tables) << (i ? "," : "") << lit(vals[i]);
    (*tables) << "};\n";
    return "T" + std::to_string(id) + "[" + ix + "]";
  }
};

enum CompContext { CTX_STEP, CTX_STAT, CTX_DERIVED, CTX_FULL };
struct Term { std::string tid, val; };

// the value of state component `idx` as an instance's code sees it
static std::string comp_ref(const std::vector<Inst>& inst, const std::vector<int>& idxs, const std::string& idx, bool same, CompContext cx) {
  if (cx == CTX_STAT) return "BP(" + idx + ")";               // the whole proposal vector (amwg.h stat_prog)
  if (cx == CTX_DERIVED) return "ST(" + idx + ")";
  if (cx == CTX_FULL) return "CM(" + idx + ")";               // full-program evaluation: the moved component is a run-time value
  bool all_moved = true, none_moved = true;
  for (size_t m = 0; m < inst.size(); ++m) { all_moved = all_moved && idxs[m] == inst[m].moved; none_moved = none_moved && idxs[m] != inst[m].moved; }
  if (all_moved) return "prop";
  if (none_moved) return "ST(" + idx + ")";
  (void)same;
  return "((" + idx + ") == c ? prop : ST(" + idx + "))";
}

// Emit instructions [i0, i1) of the instances as straight-line code. `terms` receives every finished term of the sum (its id and
// the name of its new value), `cand_slots` the statistic slots read as candidates. false: something cannot be specialised.
static bool emit_range(const GenCtx& gc, const std::vector<Inst>& inst, size_t i0, size_t i1, const std::string& ix, CompContext cx, Emitter& em,
                       std::vector<Term>& terms, std::vector<std::string>& cand_slots, std::vector<std::pair<int, std::string>>& derived_out,
                       std::string& why) {
  const auto& rep = inst[0].ins;
  const size_t M = inst.size();
  const amwg_model* md = gc.md;
  auto gather = [&](size_t i, auto getter) { std::vector<int> v(M); for (size_t m = 0; m < M; ++m) v[m] = getter(inst[m].ins[i]); return v; };
  for (size_t i = i0; i < i1; ++i) {
    const Insn& in = rep[i];
    std::string opnd[4];
    for (int k = 3; k >= 0; --k) {                             // operands are consumed last one first
      if (in.mode[k] == AMWG_MODE_NONE) continue;
      if (in.mode[k] == AMWG_MODE_STACK) {
        if (em.stk.empty()) { why = "stack underflow in a program"; return false; }
        opnd[k] = em.stk.back(); em.stk.pop_back();
      } else {
        bool same; int v0;
        std::vector<int> vals = gather(i, [k](const Insn& x) { return x.inl[k]; });
        std::string idx = gc.field(vals, ix, &same, &v0);
        if (in.mode[k] == AMWG_MODE_CONST) {
          for (int v : vals) if (v < 0 || v >= md->n_consts) { why = "const index out of range"; return false; }
          opnd[k] = same ? lit((*gc.consts)[v0]) : "KC(" + idx + ")";
        } else {
          for (int v : vals) if (v < 0 || v >= md->n_comp) { why = "component index out of range"; return false; }
          opnd[k] = comp_ref(inst, vals, idx, same, cx);
        }
      }
    }
    const std::string &x = opnd[0], &y = opnd[1], &z = opnd[2], &t = opnd[3];
    std::string r;
    bool has_r = true;
    auto imm_vals = [&]() { return gather(i, [](const Insn& q) { return q.a; }); };
    switch (in.op) {
      case AMWG_OP_CONST: {
        bool s; int v0; std::vector<int> vals = imm_vals(); std::string idx = gc.field(vals, ix, &s, &v0);
        for (int v : vals) if (v < 0 || v >= md->n_consts) { why = "const index out of range"; return false; }
        r = s ? lit((*gc.consts)[v0]) : "KC(" + idx + ")"; break;
      }
      case AMWG_OP_COMP: {
        bool s; int v0; std::vector<int> vals = imm_vals(); std::string idx = gc.field(vals, ix, &s, &v0);
        for (int v : vals) if (v < 0 || v >= md->n_comp) { why = "component index out of range"; return false; }
        r = comp_ref(inst, vals, idx, s, cx);
        break;
      }
      case AMWG_OP_DATA: {
        std::vector<double> dv(M);
        for (size_t m = 0; m < M; ++m) {
          const int c0 = inst[m].ins[i].a, i0d = inst[m].ins[i].extra[0];
          if (c0 >= md->n_columns || i0d < 0 || i0d >= md->columns[c0].n) { why = "data index out of range"; return false; }
          dv[m] = md->columns[c0].values[i0d];
        }
        r = gc.dfield(dv, ix);
        break;
      }
      case AMWG_OP_ADD: r = "(" + x + " + " + y + ")"; break;
      case AMWG_OP_SUB: r = "(" + x + " - " + y + ")"; break;
      case AMWG_OP_MUL: r = "(" + x + " * " + y + ")"; break;
      case AMWG_OP_DIV: r = "(" + x + " / " + y + ")"; break;
      case AMWG_OP_NEG: r = "(-" + x + ")"; break;
      case AMWG_OP_LOG: r = "js_log(" + x + ")"; break;
      case AMWG_OP_EXP: r = "js_exp(" + x + ")"; break;
      case AMWG_OP_SQRT: r = "sqrt(" + x + ")"; break;
      case AMWG_OP_ABS: r = "fabs(" + x + ")"; break;
      case AMWG_OP_POW: r = "js_pow(" + x + ", " + y + ")"; break;
      case AMWG_OP_LT: r = "(" + x + " < " + y + " ? 1.0 : 0.0)"; break;
      case AMWG_OP_LE: r = "(" + x + " <= " + y + " ? 1.0 : 0.0)"; break;
      case AMWG_OP_GT: r = "(" + x + " > " + y + " ? 1.0 : 0.0)"; break;
      case AMWG_OP_GE: r = "(" + x + " >= " + y + " ? 1.0 : 0.0)"; break;
      case AMWG_OP_EQ: r = "(" + x + " == " + y + " ? 1.0 : 0.0)"; break;
      case AMWG_OP_NE: r = "(" + x + " != " + y + " ? 1.0 : 0.0)"; break;
      case AMWG_OP_AND: r = "((" + x + " != 0.0 && " + y + " != 0.0) ? 1.0 : 0.0)"; break;
      case AMWG_OP_OR: r = "((" + x + " != 0.0 || " + y + " != 0.0) ? 1.0 : 0.0)"; break;
      case AMWG_OP_NOT: r = "(" + x + " != 0.0 ? 0.0 : 1.0)"; break;
      case AMWG_OP_SELECT: r = "(" + x + " != 0.0 ? " + y + " : " + z + ")"; break;
      case AMWG_OP_NORM_K: { std::string d = em.tmp("(" + x + " - " + y + ")"); r = "(" + z + " - (" + d + " * " + d + ") / " + t + ")"; break; }
      case AMWG_OP_UNIF_K: r = "((" + x + " < " + y + " || " + x + " > " + z + ") ? -CUDART_INF : " + t + ")"; break;
      case AMWG_OP_BETA_K: {
        std::string l1 = em.tmp("js_log(" + x + ")"), l2 = em.tmp("js_log((1 - " + x + "))");
        r = "((" + x + " > 1 || " + x + " < 0) ? -CUDART_INF : (" + y + " * " + l1 + " + " + z + " * " + l2 + ") - " + t + ")";
        break;
      }
      case AMWG_OP_LGAMMA: r = "ld_lgamma(" + x + ")"; break;
      case AMWG_OP_LFACTORIAL: r = "ld_lfactorial(" + x + ")"; break;
      case AMWG_OP_LCHOOSE: r = "ld_lchoose(" + x + ", " + y + ")"; break;
      case AMWG_OP_LBETA: r = "ld_lbeta(" + x + ", " + y + ")"; break;
      case AMWG_OP_LD_NORM: r = "ld_norm(" + x + ", " + y + ", " + z + ")"; break;
      case AMWG_OP_LD_UNIF: r = "ld_unif(" + x + ", " + y + ", " + z + ")"; break;
      case AMWG_OP_LD_BETA: r = "ld_beta(" + x + ", " + y + ", " + z + ")"; break;
      case AMWG_OP_LD_BERN: r = "ld_bern(" + x + ", " + y + ")"; break;
      case AMWG_OP_LD_POIS: r = "ld_pois(" + x + ", " + y + ")"; break;
      case AMWG_OP_LD_CAUCHY: r = "ld_cauchy(" + x + ", " + y + ", " + z + ")"; break;
      case AMWG_OP_LD_LAPLACE: r = "ld_laplace(" + x + ", " + y + ", " + z + ")"; break;
      case AMWG_OP_LD_GAMMA: r = "ld_gamma(" + x + ", " + y + ", " + z + ")"; break;
      case AMWG_OP_LD_INVGAMMA: r = "ld_invgamma(" + x + ", " + y + ", " + z + ")"; break;
      case AMWG_OP_LD_LNORM: r = "ld_lnorm(" + x + ", " + y + ", " + z + ")"; break;
      case AMWG_OP_LD_PARETO: r = "ld_pareto(" + x + ", " + y + ", " + z + ")"; break;
      case AMWG_OP_LD_T: r = "ld_t(" + x + ", " + y + ", " + z + ", " + t + ")"; break;
      case AMWG_OP_LD_WEIBULL: r = "ld_weibull(" + x + ", " + y + ", " + z + ")"; break;
      case AMWG_OP_LD_LOGIS: r = "ld_logis(" + x + ", " + y + ", " + z + ")"; break;
      case AMWG_OP_LD_EXP: r = "ld_exp(" + x + ", " + y + ")"; break;
      case AMWG_OP_LD_BINOM: r = "ld_binom(" + x + ", " + y + ", " + z + ")"; break;
      case AMWG_OP_LD_NBINOM: r = "ld_nbinom(" + x + ", " + y + ", " + z + ")"; break;
      case AMWG_OP_LD_HYPER: r = "ld_hyper(" + x + ", " + y + ", " + z + ", " + t + ")"; break;
      case AMWG_OP_CACHED: case AMWG_OP_CAND: {
        std::vector<int> vals = imm_vals();
        for (int v : vals) if (v < 0 || v >= md->n_terms) { why = "cache slot out of range"; return false; }
        std::string idx = gc.field(vals, ix);
        if (in.op == AMWG_OP_CACHED) r = "TV(" + idx + ")";
        else { r = "TC(" + idx + ")"; cand_slots.push_back(idx); }
        break;
      }
      case AMWG_OP_NORM_SS: {              // f(S, sd) = n * (c0 - log sd) - S / (2 sd^2), the operations of norm_factorised()
        std::vector<double> nv(M);
        for (size_t m = 0; m < M; ++m) {
          const int q = inst[m].ins[i].a;
          if (q >= md->n_plates) { why = "plate index out of range"; return false; }
          nv[m] = (double)md->plates[q].n;
        }
        std::string nn = gc.dfield(nv, ix);
        std::string lsd = em.tmp("js_log(" + y + ")");
        std::string k2 = em.tmp("(2 * " + y + " * " + y + ")");
        r = "(" + nn + " * (JNORM_C0 - " + lsd + ") - " + x + " / " + k2 + ")";
        break;
      }
      case AMWG_OP_DATA_I: case AMWG_OP_COMP_I: {             // inside a generated loop: columns[a][off + stride * i_]
        if (cx != CTX_FULL || M != 1 || !gc.plan) { why = "plate-indexed data outside a full-program loop"; return false; }
        if (in.a >= md->n_columns || gc.plan->col_smem_off[in.a] < 0) { why = "a looped column is not resident"; return false; }
        std::string at = "LD(" + std::to_string(gc.plan->col_smem_off[in.a] + 8 * in.extra[0]) + "u + " + std::to_string(8 * in.extra[1]) + "u * (unsigned)i_)";
        r = in.op == AMWG_OP_DATA_I ? at : "CM(" + std::to_string(in.extra[2]) + " + (int)" + at + ")";
        break;
      }
      case AMWG_OP_ACC: {
        if (cx != CTX_FULL) { why = "ACC outside a full-program evaluation"; return false; }
        if (em.stk.empty()) { why = "stack underflow"; return false; }
        em.os << "    lp = lp + " << em.stk.back() << ";\n"; em.stk.pop_back();
        has_r = false;
        break;
      }
      case AMWG_OP_LOOP_BEGIN: {
        if (cx != CTX_FULL) { why = "loop outside a full-program evaluation"; return false; }
        if (in.a >= md->n_plates) { why = "plate index out of range"; return false; }
        em.scopes.push_back(em.cse);
        em.os << "    for (int i_ = 0; i_ < " << md->plates[in.a].n << "; ++i_) {\n";
        has_r = false;
        break;
      }
      case AMWG_OP_LOOP_END: {
        if (cx != CTX_FULL || em.scopes.empty() || em.stk.empty()) { why = "malformed loop"; return false; }
        em.os << "    lp = lp + " << em.stk.back() << ";\n    }\n"; em.stk.pop_back();
        em.cse = em.scopes.back(); em.scopes.pop_back();
        has_r = false;
        break;
      }
      case AMWG_OP_PLATE: {
        if (cx != CTX_FULL || !gc.plan) { why = "plate outside a full-program evaluation"; return false; }
        const amwg_plate& pq = md->plates[in.a];
        const int c0 = pq.col[0];
        if (c0 < 0 || c0 >= md->n_columns || gc.plan->col_smem_off[c0] < 0) { why = "a plate's column is not resident"; return false; }
        const std::string boff = std::to_string(gc.plan->col_smem_off[c0] + 8 * pq.iparam[2]);
        if (pq.kind == AMWG_PLATE_NORM_IID) {                   // operands: A = mean, B = sd
          em.os << "    lp = lp + jit_norm_factorised(" << lit((double)pq.n) << ", sum_sq_dev(reinterpret_cast<const double*>(smem + " << boff << "), smem_u32(smem) + "
                << boff << "u, " << pq.n << ", " << x << "), " << y << ");\n";
        } else if (pq.kind == AMWG_PLATE_BERN_IID) {
          const int mo = in.a < (int)gc.plan->bern_mask_off.size() ? gc.plan->bern_mask_off[in.a] : -1;
          if (mo >= 0) em.os << "    lp = jit_plate_bern_mask<" << pq.n << ">(smem, " << boff << "u, " << mo << "u, " << x << ", lp);\n";
          else em.os << "    lp = jit_plate_bern(smem_u32(smem) + " << boff << "u, " << pq.n << ", " << x << ", lp);\n";
        } else if (pq.kind == AMWG_PLATE_NORM_GROUPED) {        // operand A = sd; points sorted by group, starts in col[1]
          const int c1 = pq.col[1];
          if (c1 < 0 || c1 >= md->n_columns || gc.plan->col_smem_off[c1] < 0) { why = "a plate's column is not resident"; return false; }
          const std::string soff = std::to_string(gc.plan->col_smem_off[c1]), coff = std::to_string(gc.plan->col_smem_off[c0]);
          em.os << "    {\n      double S_ = 0.0;\n      for (int j_ = 0; j_ < " << pq.iparam[1] << "; ++j_) {\n"
                << "        const int a_ = (int)LD(" << soff << "u + 8u * (unsigned)j_) + " << pq.iparam[2] << ", b_ = (int)LD(" << soff << "u + 8u * (unsigned)(j_ + 1)) + " << pq.iparam[2] << ";\n"
                << "        S_ = S_ + sum_sq_dev(reinterpret_cast<const double*>(smem + " << coff << " + 8 * a_), smem_u32(smem) + " << coff << "u + 8u * (unsigned)a_, b_ - a_, CM(" << pq.iparam[0] << " + j_));\n"
                << "      }\n      lp = lp + jit_norm_factorised(" << lit((double)pq.n) << ", S_, " << x << ");\n    }\n";
        } else { why = "this plate kind is not specialised"; return false; }
        has_r = false;
        break;
      }
      case AMWG_OP_STORE: {
        if (cx != CTX_DERIVED) { why = "STORE outside a derived-quantity program"; return false; }
        if (em.stk.empty()) { why = "stack underflow"; return false; }
        derived_out.emplace_back(in.a, em.stk.back()); em.stk.pop_back();
        has_r = false;
        break;
      }
      case AMWG_OP_END: has_r = false; break;
      default: why = "opcode " + std::to_string(in.op) + " cannot be specialised"; return false;
    }
    if (!has_r) continue;
    std::string name = em.tmp(r);                               // every value gets a name; identical right-hand sides are shared
    if (in.acc && cx == CTX_FULL) {
      em.os << "    lp = lp + " << name << ";\n";              // the sum is formed in program order, like the JS `log_post += ...`
    } else if (in.acc) {
      if (!in.store) { why = "a term of the sum is not cached"; return false; }
      terms.push_back(Term{gc.field(gather(i, [](const Insn& q) { return q.term; }), ix), name});
    } else {
      em.stk.push_back(name);
    }
  }
  return true;
}

static std::string insn_sig(const Insn& in) {
  char b[64];
  snprintf(b, sizeof b, "%d:%d%d%d%d:%d%d;", in.op, in.mode[0], in.mode[1], in.mode[2], in.mode[3], (int)in.acc, (int)in.store);
  return b;
}

// One class of component programs -> the body of its `case` in jit_step: the per-term differences are summed into `dl`; `commit`
// is what an accepted step writes back. Inside a single program, a run of >= 4 consecutive terms of identical shape (the 64 plate
// terms a shared sd touches in a hierarchical model) becomes a loop over small tables instead of straight-line code.
static bool emit_step_class(const GenCtx& gc, const std::vector<Inst>& members, std::string& body, std::string& commit, int* n_insns, std::string& why) {
  const auto& rep = members[0].ins;
  std::vector<std::pair<size_t, size_t>> chunks;               // [begin, end) instruction ranges, one per term of the sum
  {
    size_t b0 = 0;
    for (size_t i = 0; i < rep.size(); ++i)
      if (rep[i].acc || rep[i].op == AMWG_OP_END) { chunks.emplace_back(b0, i + 1); b0 = i + 1; }
    if (b0 < rep.size()) chunks.emplace_back(b0, rep.size());
  }
  auto chunk_sig = [&](const std::pair<size_t, size_t>& ch) { std::string sg; for (size_t i = ch.first; i < ch.second; ++i) sg += insn_sig(rep[i]); return sg; };
  Emitter em;
  std::ostringstream bd, cm;
  std::vector<std::pair<int, std::string>> der;
  size_t k = 0;
  while (k < chunks.size()) {
    size_t run = 1;
    if (members.size() == 1 && rep[chunks[k].second - 1].acc) {
      const std::string sg = chunk_sig(chunks[k]);
      while (k + run < chunks.size() && chunk_sig(chunks[k + run]) == sg) ++run;
    }
    // the first (or only) chunk: straight line
    {
      std::vector<Term> terms; std::vector<std::string> cands;
      const size_t before = em.os.str().size();
      if (!emit_range(gc, members, chunks[k].first, chunks[k].second, "m", CTX_STEP, em, terms, cands, der, why)) return false;
      if (!em.stk.empty() && rep[chunks[k].second - 1].acc) { why = "a term leaves operands on the stack"; return false; }
      bd << em.os.str().substr(before);
      for (auto& t : terms) { bd << "    dl = dl + (" << t.val << " - TV(" << t.tid << "));\n"; cm << "    TV(" << t.tid << ") = " << t.val << ";\n"; }
      for (auto& sl : cands) cm << "    TV(" << sl << ") = TC(" << sl << ");\n";
      *n_insns += (int)(chunks[k].second - chunks[k].first);
    }
    if (run >= 4) {
      // chunks k+1 .. k+run-1 as a loop: instance j = chunk k+1+j, re-based to instruction 0
      std::vector<Inst> iters;
      for (size_t j = 1; j < run; ++j) {
        Inst it;
        it.ins.assign(rep.begin() + chunks[k + j].first, rep.begin() + chunks[k + j].second);
        it.moved = members[0].moved;
        iters.push_back(it);
      }
      Emitter inner;
      inner.cse = em.cse;                                       // loop-invariant values (log sd, 2 sd^2) were named by the first chunk
      inner.nv = em.nv;
      std::vector<Term> terms; std::vector<std::string> cands;
      if (!emit_range(gc, iters, 0, iters[0].ins.size(), "j", CTX_STEP, inner, terms, cands, der, why)) return false;
      if (!inner.stk.empty()) { why = "a term leaves operands on the stack"; return false; }
      em.nv = inner.nv;
      bd << "    for (int j = 0; j < " << iters.size() << "; ++j) {\n" << inner.os.str();
      for (auto& t : terms) bd << "      dl = dl + (" << t.val << " - TV(" << t.tid << "));\n";
      bd << "    }\n";
      cm << "    for (int j = 0; j < " << iters.size() << "; ++j) {\n" << inner.os.str();
      for (auto& t : terms) cm << "      TV(" << t.tid << ") = " << t.val << ";\n";
      for (auto& sl : cands) cm << "      TV(" << sl << ") = TC(" << sl << ");\n";
      cm << "    }\n";
      *n_insns += (int)iters[0].ins.size();
      k += run;
    } else {
      k += 1;
    }
  }
  body = bd.str();
  commit = cm.str();
  return true;
}

static std::string signature(const std::vector<Insn>& prog) {
  std::string s;
  for (const Insn& in : prog) {
    char b[64];
    snprintf(b, sizeof b, "%d:%d%d%d%d:%d%d;", in.op, in.mode[0], in.mode[1], in.mode[2], in.mode[3], (int)in.acc, (int)in.store);
    s += b;
  }
  return s;
}

// Launch shape: CTA size and resident CTAs per SM such that the chains spread evenly over the SMs; the per-chain working set
// (`per_thread` bytes) goes to shared memory when it is small. `off`: shared memory already planned (columns, ring).
static std::string choose_shape(Plan& pl, unsigned off, size_t per_thread, unsigned long long n_chains, int sm_count) {
  const unsigned base = off;
  int best_t = 0, best_r = 1, best_ws = 0;
  double best_eff = -1.0;
  const int cands[] = {128, 64, 96, 160, 192, 224, 256};
  int forced_t = 0;
  if (const char* e = getenv("AMWG_JIT_THREADS")) { int t = atoi(e); if (t >= 32 && t <= 1024 && t % 32 == 0) forced_t = t; }
  for (int t : cands) {
    if (forced_t) t = forced_t;
    const size_t need = pad16(per_thread * (size_t)t);
    const int ws_smem = need <= kJitWsSmemLimit;
    const unsigned smem = std::max((unsigned)(pad16(base) + (ws_smem ? need : 0)), 16u);
    int r_max = (int)std::min<unsigned>(std::min<unsigned>((227u * 1024u) / (smem + 1024u), 2048u / (unsigned)t), 8u);
    if (r_max < 1) continue;
    const double ctas = std::ceil((double)n_chains / t);
    const double cap = (double)sm_count * r_max;
    double eff; int r_need;
    if (ctas <= cap) { const double per_sm = std::ceil(ctas / sm_count); eff = ((double)n_chains / sm_count) / (per_sm * t); r_need = (int)per_sm; }
    else { eff = ctas / (std::ceil(ctas / cap) * cap) * ((double)n_chains / (ctas * t)); r_need = r_max; }
    // 128-thread CTAs are the default; another size has to fill the SMs a good deal more evenly to win (config 4 at 2^16 chains:
    // 224 x 2 CTAs/SM is 14 % better balanced than 128 x 4 and measured 6 % SLOWER -- more, smaller CTAs overlap their phases)
    if (eff > best_eff + (best_t == 0 ? 0.0 : 0.15)) { best_eff = eff; best_t = t; best_r = r_need; best_ws = ws_smem; }
    if (forced_t) break;
  }
  if (!best_t) return "no launch shape fits";
  pl.threads = best_t;
  if (best_ws) { pl.ws_smem = 1; pl.ws_off = (int)pad16(off); off = (unsigned)(pad16(off) + pad16(per_thread * (size_t)best_t)); }
  pl.smem_bytes = std::max(off, 16u);
  pl.minblocks = std::max(1, best_r);
  if (const char* e = getenv("AMWG_JIT_MINBLOCKS")) { int v = atoi(e); if (v >= 1 && v <= 16) pl.minblocks = v; }
  return "";
}


static void emit_param_tables(std::ostringstream& tables, const amwg_model* md) {
  const int P = md->n_params;
  auto ptab = [&](const char* ty, const char* name, auto get) {
    tables << "__constant__ " << ty << " " << name << "[" << P << "] = {";
    for (int p = 0; p < P; ++p) tables << (p ? "," : "") << get(md->params[p]);
    tables << "};\n";
  };
  ptab("int", "JP_TYPE", [](const amwg_param& p) { return istr(p.type); });
  ptab("int", "JP_NCOMP", [](const amwg_param& p) { return istr(p.n_comp); });
  ptab("int", "JP_DIM0", [](const amwg_param& p) { return istr(p.dim0); });
  ptab("int", "JP_OFF", [](const amwg_param& p) { return istr(p.comp_offset); });
  ptab("long long", "JP_LOWER", [](const amwg_param& p) { return bits(p.lower); });
  ptab("long long", "JP_UPPER", [](const amwg_param& p) { return bits(p.upper); });
  tables << "__device__ __forceinline__ int jp_type(int p) { return JP_TYPE[p]; }\n"
            "__device__ __forceinline__ int jp_ncomp(int p) { return JP_NCOMP[p]; }\n"
            "__device__ __forceinline__ int jp_dim0(int p) { return JP_DIM0[p]; }\n"
            "__device__ __forceinline__ int jp_off(int p) { return JP_OFF[p]; }\n"
            "__device__ __forceinline__ double jp_lower(int p) { return __longlong_as_double(JP_LOWER[p]); }\n"
            "__device__ __forceinline__ double jp_upper(int p) { return __longlong_as_double(JP_UPPER[p]); }\n";
}


// a run-time switch read when the specialisation is built (DESIGN.md section 6b): unset -> `dflt`, else its integer value != 0
static bool env_flag(const char* name, bool dflt) {
  const char* e = getenv(name);
  return e ? atoi(e) != 0 : dflt;
}

struct StepClass { std::string body, commit; bool uses_m; };    // one `case` of jit_step as emit_step_class printed it

// The merged form of jit_step (AMWG_JIT_MERGE_STEPS). The lanes of a warp step components of different classes at the same time
// (each chain shuffles its substeppers), so in the switch form every class body -- with its out-of-line js_log / js_exp calls --
// runs one after another under divergence. Here each class body is split into
//   (A) per class: the operands of its heavy calls (a js_log / js_exp whose argument does not depend on another such call);
//   (B) the heavy calls, once per warp: slot j of a function takes the j-th such call of every class (a class without one skips
//       it behind a branch no lane of that class takes);
//   (C) per class: the rest of the body in its original order -- every `dl = dl + ...` keeps its place, so dl is the same sum;
//   one accept test for all classes; then the per-class commit.
// Every value is computed by the same operations as in the switch form: the draws are bit-identical. Values cross the phases in
// function-scope variables named k<class>_v<n>. false: the body text is not in the form emit_step_class prints.
static bool emit_merged_step(const std::vector<StepClass>& cls, const std::string& accept_test, std::ostringstream& out) {
  static const std::regex def_re("^    const double (v[0-9]+) = (.*);$"), name_re("\\bv[0-9]+\\b");
  static const char* const kHeavy[2] = {"js_log", "js_exp"};
  auto refs_of = [](const std::string& s) {
    std::set<std::string> r;
    for (std::sregex_iterator it(s.begin(), s.end(), name_re), e; it != e; ++it) r.insert(it->str());
    return r;
  };
  auto heavy_of = [](const std::string& rhs, std::string& arg) -> int {     // rhs is exactly one call js_log(...) / js_exp(...)
    for (int f = 0; f < 2; ++f) {
      const std::string head = std::string(kHeavy[f]) + "(";
      if (rhs.compare(0, head.size(), head) != 0 || rhs.back() != ')') continue;
      int depth = 0;
      for (size_t i = head.size() - 1; i < rhs.size(); ++i) {
        depth += rhs[i] == '(' ? 1 : rhs[i] == ')' ? -1 : 0;
        if (depth == 0 && i + 1 != rhs.size()) return -1;
      }
      arg = rhs.substr(head.size(), rhs.size() - head.size() - 1);
      return f;
    }
    return -1;
  };
  struct Stmt { std::string text, name, rhs; bool def = false; int heavy = -1, slot = -1; std::string arg; bool phase_a = false; };
  std::vector<std::vector<Stmt>> body(cls.size());
  int n_slots[2] = {0, 0};
  std::vector<std::array<std::vector<std::string>, 2>> args(cls.size());     // per class and function: the operand of each slot
  bool uses_m = false;
  for (size_t k = 0; k < cls.size(); ++k) {
    uses_m = uses_m || cls[k].uses_m;
    std::istringstream in(cls[k].body);
    std::vector<Stmt>& st = body[k];
    for (std::string ln; std::getline(in, ln);) {
      Stmt s;
      std::smatch mt;
      if (ln.compare(0, 9, "    for (") == 0) {                 // a generated loop: one statement, to its closing brace
        s.text = ln + "\n";
        bool closed = false;
        while (!closed && std::getline(in, ln)) { s.text += ln + "\n"; closed = ln == "    }"; }
        if (!closed) return false;
      } else if (std::regex_match(ln, mt, def_re)) {
        s.def = true; s.name = mt[1]; s.rhs = mt[2];
      } else {
        s.text = ln + "\n";
      }
      st.push_back(s);
    }
    // heavy calls whose operand depends on no heavy result; `tainted`: every value that does
    std::set<std::string> tainted;
    int used[2] = {0, 0};
    for (Stmt& s : st) {
      if (!s.def) continue;
      bool dep = false;
      for (const auto& r : refs_of(s.rhs)) dep = dep || tainted.count(r);
      std::string arg;
      const int f = heavy_of(s.rhs, arg);
      if (f >= 0 && !dep) { s.heavy = f; s.slot = used[f]++; s.arg = arg; args[k][f].push_back(arg); }
      if (f >= 0 || dep) tainted.insert(s.name);
    }
    for (int f = 0; f < 2; ++f) n_slots[f] = std::max(n_slots[f], used[f]);
    // (A) holds only what the operands need, so that little is live across the calls
    std::set<std::string> need;
    for (int f = 0; f < 2; ++f) for (const auto& a : args[k][f]) for (const auto& r : refs_of(a)) need.insert(r);
    for (size_t i = st.size(); i-- > 0;)
      if (st[i].def && st[i].heavy < 0 && need.count(st[i].name) && !tainted.count(st[i].name)) {
        st[i].phase_a = true;
        for (const auto& r : refs_of(st[i].rhs)) need.insert(r);
      }
  }
  auto ren = [&](size_t k, const std::string& s) { return std::regex_replace(s, name_re, "k" + std::to_string(k) + "_$&"); };
  auto slot_var = [](const char* pre, int f, int j) { return std::string(pre) + (f == 0 ? "l" : "e") + std::to_string(j); };
  auto all_have = [&](int f, int j) { for (const auto& a : args) if ((int)a[f].size() <= j) return false; return true; };

  out << "__device__ __forceinline__ bool jit_step(const int c, const double prop, const double coin, double* __restrict__ wk, const unsigned long long ws,\n"
         "                                         double* __restrict__ sp, const unsigned long long ss) {\n";
  if (uses_m) out << "  const int m = JMEM[c];\n";
  for (size_t k = 0; k < cls.size(); ++k) {
    std::string names;
    for (const Stmt& s : body[k]) if (s.def) names += (names.empty() ? "" : ", ") + ren(k, s.name);
    if (!names.empty()) out << "  double " << names << ";\n";
  }
  for (int f = 0; f < 2; ++f)
    for (int j = 0; j < n_slots[f]; ++j) {
      out << "  double " << slot_var("a", f, j) << " = 1.0;\n";
      if (!all_have(f, j)) out << "  bool " << slot_var("u", f, j) << " = false;\n";
    }
  out << "  double dl = 0.0;\n  switch (JCLS[c]) {\n";              // (A)
  for (size_t k = 0; k < cls.size(); ++k) {
    out << "  case " << k << ": {\n";
    for (const Stmt& s : body[k]) if (s.phase_a) out << "    " << ren(k, s.name) << " = " << ren(k, s.rhs) << ";\n";
    for (int f = 0; f < 2; ++f)
      for (int j = 0; j < (int)args[k][f].size(); ++j) {
        out << "    " << slot_var("a", f, j) << " = " << ren(k, args[k][f][j]) << ";\n";
        if (!all_have(f, j)) out << "    " << slot_var("u", f, j) << " = true;\n";
      }
    out << "    break;\n  }\n";
  }
  out << "  }\n";
  for (int f = 0; f < 2; ++f)                                       // (B)
    for (int j = 0; j < n_slots[f]; ++j) {
      const std::string call = std::string(kHeavy[f]) + "(" + slot_var("a", f, j) + ")";
      if (all_have(f, j)) out << "  const double " << slot_var("r", f, j) << " = " << call << ";\n";
      else out << "  double " << slot_var("r", f, j) << " = 0.0;\n  if (" << slot_var("u", f, j) << ") " << slot_var("r", f, j) << " = " << call << ";\n";
    }
  out << "  switch (JCLS[c]) {\n";                                  // (C)
  for (size_t k = 0; k < cls.size(); ++k) {
    out << "  case " << k << ": {\n";
    for (const Stmt& s : body[k]) {
      if (s.phase_a) continue;
      if (!s.def) out << ren(k, s.text);
      else out << "    " << ren(k, s.name) << " = " << (s.heavy >= 0 ? slot_var("r", s.heavy, s.slot) : ren(k, s.rhs)) << ";\n";
    }
    out << "    break;\n  }\n";
  }
  out << "  }\n" << accept_test << "  ST(c) = prop;\n  switch (JCLS[c]) {\n";
  for (size_t k = 0; k < cls.size(); ++k) out << "  case " << k << ": {\n" << ren(k, cls[k].commit) << "    break;\n  }\n";
  out << "  }\n  return true;\n}\n";
  return true;
}

// Build the specialised translation unit for `md`. Returns "" and fills `src` on success, else the reason it does not apply.
static std::string build_source(const amwg_model* md, const std::vector<double>& consts, unsigned long long n_chains, int sm_count,
                                double norm_c0, Source& src) {
  if (!md->comp_prog || md->n_terms <= 0 || md->stat_prog < 0) return "the model has no pre-evaluated statistics";
  if (md->n_variant_comps > 0) return "variant programs";
  const int D = md->n_comp, P = md->n_params, NT = md->n_terms;
  if (D > 65535 || P > 255) return "too many components / parameters";
  int max_dim0 = 1;
  for (int p = 0; p < P; ++p) {
    if (md->params[p].type == AMWG_BINARY) return "binary parameter";
    if (md->params[p].n_comp > 1) max_dim0 = std::max(max_dim0, std::max(md->params[p].dim0, 2));   // >= 2: a [1, n] matrix is multi-component too
  }
  std::string err;

  // ---- the statistics pass: PLATE_SS entries of stat_prog
  std::vector<Insn> stat;
  if (!decode_program(md, md->stat_prog, stat, nullptr, err)) return "stat_prog: " + err;
  struct StatEntry { int q, slot, comp; size_t first, last; bool simple; };      // instructions [first, last] produce the entry
  std::vector<StatEntry> entries;
  {
    size_t start = 0;
    for (size_t i = 0; i < stat.size(); ++i) {
      if (stat[i].op == AMWG_OP_END) break;
      if (stat[i].op != AMWG_OP_PLATE_SS) continue;
      StatEntry e{stat[i].a, stat[i].extra[0], -1, start, i, false};
      if (e.q < 0 || e.q >= md->n_plates || md->plates[e.q].kind != AMWG_PLATE_NORM_IID) return "stat_prog refers to a plate that is not NORM_IID";
      if (e.slot < 0 || e.slot >= NT) return "statistic slot out of range";
      if (i == start && stat[i].mode[0] == AMWG_MODE_COMP) { e.simple = true; e.comp = stat[i].inl[0]; if (e.comp < 0 || e.comp >= D) return "component out of range"; }
      entries.push_back(e);
      start = i + 1;
    }
  }
  if (entries.empty()) return "no plate statistics";

  // ---- shared-memory plan: which columns are resident, which one streams
  Plan& pl = src.plan;
  pl = Plan();
  pl.col_smem_off.assign(md->n_columns, -1);
  std::vector<char> col_used(md->n_columns, 0);
  for (const auto& e : entries) {
    const int c = md->plates[e.q].col[0];
    if (c < 0 || c >= md->n_columns) return "plate column out of range";
    const amwg_plate& p = md->plates[e.q];
    if (p.iparam[2] < 0 || (long long)p.iparam[2] + p.n > md->columns[c].n) return "plate runs past its column";
    col_used[c] = 1;
  }
  unsigned off = 0;
  std::vector<int> big;
  for (int c = 0; c < md->n_columns; ++c) {
    if (!col_used[c]) continue;
    const unsigned bytes = pad16(std::max<size_t>(sizeof(double) * (size_t)md->columns[c].n, 16));
    if (off + bytes <= kResidentBudget) {
      pl.col_smem_off[c] = (int)off; pl.res_col.push_back(c); pl.res_off.push_back((int)off); pl.res_bytes.push_back((int)bytes);
      off += bytes;
    } else big.push_back(c);
  }
  pl.n_res = (int)pl.res_col.size();
  if (big.size() > 1) return "more than one column exceeds shared memory";
  std::vector<StatEntry> r_entries, s_entries, x_entries;      // resident simple / streamed simple / expression means
  for (const auto& e : entries) {
    const int c = md->plates[e.q].col[0];
    const bool resident = pl.col_smem_off[c] >= 0;
    if (e.simple) (resident ? r_entries : s_entries).push_back(e);
    else { if (!resident) return "a plate with an expression mean lies on a streamed column"; x_entries.push_back(e); }
  }
  int s_begin = 0, s_total = 0;
  if (!big.empty()) {
    pl.stream_col = big[0];
    if (s_entries.empty()) return "streamed column without plates";
    std::stable_sort(s_entries.begin(), s_entries.end(), [&](const StatEntry& a, const StatEntry& b) { return md->plates[a.q].iparam[2] < md->plates[b.q].iparam[2]; });
    s_begin = md->plates[s_entries[0].q].iparam[2];
    if (s_begin & 1) return "streamed plates start at an odd offset";
    int cur = s_begin;
    for (const auto& e : s_entries) {
      const amwg_plate& p = md->plates[e.q];
      if (p.iparam[2] != cur || p.n <= 0) return "streamed plates do not tile their column";
      cur += p.n;
    }
    s_total = cur - s_begin;
    pl.ring_off = (int)off;
    off += (unsigned)(pl.ring_stages * pl.ring_tile * 8);
  }
  {
    const size_t per_thread = sizeof(double) * (size_t)(2 * NT + 3 * D) + sizeof(unsigned short) * (size_t)D;
    std::string e = choose_shape(pl, off, per_thread, n_chains, sm_count);
    if (!e.empty()) return e;
  }

  // ---- component programs -> classes
  std::ostringstream tables, funcs;
  int table_counter = 0;
  GenCtx gc;
  gc.md = md; gc.consts = &consts; gc.tables = &tables; gc.table_counter = &table_counter;
  std::vector<std::vector<Insn>> progs(D);
  std::map<std::string, std::vector<int>> classes_by_sig;
  std::vector<std::string> sig_order;
  int total_insns = 0;
  for (int c = 0; c < D; ++c) {
    std::vector<Insn> full;
    if (!decode_program(md, md->comp_prog[c], full, nullptr, err)) return "comp_prog: " + err;
    for (const Insn& in : full) if (in.op != AMWG_OP_ACC_RANGE) progs[c].push_back(in);
    std::string sg = signature(progs[c]);
    if (!classes_by_sig.count(sg)) sig_order.push_back(sg);
    classes_by_sig[sg].push_back(c);
  }
  std::vector<int> cls_of(D, 0), mem_of(D, 0);
  funcs << "namespace amwg {\n";
  const bool screen = env_flag("AMWG_JIT_ACCEPT_SCREEN", true);
  const std::string accept_test = screen ? "    int acc_ = jit_accept_screen(dl, coin);              // certain from dl's sign or an fp32 estimate; -1: undecided\n"
                                           "    if (acc_ < 0) acc_ = js_exp(dl) > coin;            // Metropolis accept (mcmc.js:527-534): strict >, NaN rejects\n"
                                           "    if (!acc_) return false;\n"
                                         : "    if (!(js_exp(dl) > coin)) return false;            // Metropolis accept (mcmc.js:527-534): strict >, NaN rejects\n";
  std::vector<StepClass> step_classes;
  std::ostringstream step;
  step << "__device__ __forceinline__ bool jit_step(const int c, const double prop, const double coin, double* __restrict__ wk, const unsigned long long ws,\n"
          "                                         double* __restrict__ sp, const unsigned long long ss) {\n";
  if (sig_order.size() > 1) step << "  switch (JCLS[c]) {\n";
  bool need_mem = false;
  for (size_t k = 0; k < sig_order.size(); ++k) {
    const std::vector<int>& members = classes_by_sig[sig_order[k]];
    std::vector<Inst> inst;
    for (size_t m = 0; m < members.size(); ++m) {
      Inst it; it.ins = progs[members[m]]; it.moved = members[m];
      inst.push_back(it);
      cls_of[members[m]] = (int)k; mem_of[members[m]] = (int)m;
    }
    std::string body, commit, why;
    if (!emit_step_class(gc, inst, body, commit, &total_insns, why)) return "component program: " + why;
    if (total_insns > kMaxGeneratedInsns) return "the component programs are too long to specialise";
    if (commit.empty()) return "a component touches no term";
    if (sig_order.size() > 1) step << "  case " << k << ": {\n";
    else step << "  {\n";
    if (inst.size() > 1) { step << "    const int m = JMEM[c];\n"; need_mem = true; }
    step << "    double dl = 0.0;\n" << body;
    step << accept_test;
    step << "    ST(c) = prop;\n" << commit;
    step << "    return true;\n  }\n";
    step_classes.push_back(StepClass{body, commit, inst.size() > 1});
  }
  if (sig_order.size() > 1) step << "  }\n  return false;\n";
  step << "}\n";
  if (sig_order.size() > 1 && env_flag("AMWG_JIT_MERGE_STEPS", true)) {
    step.str("");
    if (!emit_merged_step(step_classes, accept_test, step)) return "component program: unexpected generated step code";
  }

  // ---- statistics whose mean is an expression
  std::ostringstream extra;
  extra << "__device__ __forceinline__ void jit_stat_extra(unsigned char* smem, double* __restrict__ wk, const unsigned long long ws,\n"
           "                                               double* __restrict__ sp, const unsigned long long ss, const bool wr) {\n";
  for (const auto& e : x_entries) {
    Inst it;
    it.ins.assign(stat.begin() + e.first, stat.begin() + e.last);                  // the mean's code (without the PLATE_SS itself)
    std::vector<Inst> inst{it};
    const Insn pss = stat[e.last];
    Emitter em;
    std::vector<Term> terms; std::vector<std::string> cands; std::vector<std::pair<int, std::string>> der;
    std::string why;
    if (!emit_range(gc, inst, 0, it.ins.size(), "m", CTX_STAT, em, terms, cands, der, why)) return "stat_prog: " + why;
    std::string mean;
    if (pss.mode[0] == AMWG_MODE_STACK) { if (em.stk.empty()) return "stat_prog: missing mean"; mean = em.stk.back(); }
    else if (pss.mode[0] == AMWG_MODE_CONST) { if (pss.inl[0] < 0 || pss.inl[0] >= md->n_consts) return "stat_prog: const out of range"; mean = lit(consts[pss.inl[0]]); }
    else mean = "BP(" + std::to_string(pss.inl[0]) + ")";
    total_insns += (int)it.ins.size();
    const amwg_plate& p = md->plates[e.q];
    const int so = pl.col_smem_off[p.col[0]] + 8 * p.iparam[2];
    extra << "  {\n" << em.os.str();
    extra << "    const double S = sum_sq_dev(reinterpret_cast<const double*>(smem + " << so << "), smem_u32(smem) + " << so << "u, " << p.n << ", " << mean << ");\n";
    extra << "    if (wr) TC(" << e.slot << ") = S;\n  }\n";
  }
  extra << "  (void)smem; (void)wk; (void)ws; (void)sp; (void)ss; (void)wr;\n}\n";

  // ---- derived quantities
  std::ostringstream dfun;
  if (md->n_derived > 0) {
    Inst it;
    if (!decode_program(md, md->derived_prog, it.ins, nullptr, err)) return "derived_prog: " + err;
    std::vector<Inst> inst{it};
    Emitter em;
    std::vector<Term> terms; std::vector<std::string> cands; std::vector<std::pair<int, std::string>> der;
    std::string why;
    if (!emit_range(gc, inst, 0, it.ins.size(), "m", CTX_DERIVED, em, terms, cands, der, why)) return "derived program: " + why;
    dfun << "__device__ __forceinline__ void jit_derived(const double* __restrict__ sp, const unsigned long long ss, double* der) {\n" << em.os.str();
    for (auto& d : der) { if (d.first < 0 || d.first >= md->n_derived) return "derived index out of range"; dfun << "    der[" << d.first << "] = " << d.second << ";\n"; }
    dfun << "}\n";
  }

  // ---- tables
  auto int_table = [&](const char* qual, const char* name, const std::vector<long long>& v) {
    tables << qual << " " << name << "[" << std::max<size_t>(v.size(), 1) << "] = {";
    for (size_t i = 0; i < v.size(); ++i) tables << (i ? "," : "") << v[i];
    if (v.empty()) tables << "0";
    tables << "};\n";
  };
  {
    std::vector<long long> v;
    if (sig_order.size() > 1) { v.assign(cls_of.begin(), cls_of.end()); int_table("__device__ const unsigned char", "JCLS", v); }
    if (need_mem) { v.assign(mem_of.begin(), mem_of.end()); int_table("__device__ const unsigned short", "JMEM", v); }
    tables << "__device__ const long long KCB[" << std::max(md->n_consts, 1) << "] = {";
    for (int i = 0; i < md->n_consts; ++i) tables << (i ? "," : "") << bits(consts[i]);
    if (md->n_consts == 0) tables << "0LL";
    tables << "};\n#define KC(i) __longlong_as_double(KCB[i])\n";
    emit_param_tables(tables, md);                              // parameters (mcmc.js:357-403 completed)
    // resident columns and the simple statistics over them
    std::vector<long long> a, b, c2, d;
    for (int k = 0; k < pl.n_res; ++k) { a.push_back(pl.res_off[k]); b.push_back(pl.res_col[k]); c2.push_back(pl.res_bytes[k]); }
    int_table("__constant__ unsigned", "JRES_OFF", a); int_table("__constant__ int", "JRES_COL", b); int_table("__constant__ unsigned", "JRES_BYTES", c2);
    a.clear(); b.clear(); c2.clear();
    for (const auto& e : r_entries) {
      const amwg_plate& p = md->plates[e.q];
      a.push_back(e.comp); b.push_back(pl.col_smem_off[p.col[0]] + 8 * p.iparam[2]); c2.push_back(p.n); d.push_back(e.slot);
    }
    int_table("__constant__ int", "JR_COMP", a); int_table("__constant__ unsigned", "JR_SOFF", b); int_table("__constant__ int", "JR_N", c2); int_table("__constant__ int", "JR_SLOT", d);
    a.clear(); b.clear(); d.clear();
    int cur = 0;
    for (const auto& e : s_entries) { cur += md->plates[e.q].n; a.push_back(e.comp); b.push_back(cur); d.push_back(e.slot); }
    int_table("__constant__ int", "JS_COMP", a); int_table("__constant__ int", "JS_END", b); int_table("__constant__ int", "JS_SLOT", d);
  }

  unsigned long long res_total = 0;
  for (int k = 0; k < pl.n_res; ++k) res_total += (unsigned)pl.res_bytes[k];
  // JBLOCK: the largest multi-dim parameter whose components never share a term or a statistic (pairwise disjoint touch lists)
  int jblock = -1;
  for (int p = 0, best = 7; p < P; ++p) {
    const amwg_param& pa = md->params[p];
    if (pa.n_comp <= best) continue;
    bool indep = true;
    std::vector<int> owner((size_t)NT, -1);
    for (int c = pa.comp_offset; c < pa.comp_offset + pa.n_comp && indep; ++c)
      for (int k = md->touch_off[c]; k < md->touch_off[c + 1]; ++k) {
        int& o = owner[(size_t)md->touch_terms[k]];
        if (o >= 0 && o != c) { indep = false; break; }
        o = c;
      }
    if (indep) { jblock = p; best = pa.n_comp; }
  }
  if (const char* e = getenv("AMWG_JIT_BLOCK")) { if (atoi(e) == 0) jblock = -1; }
  const bool jblock_free = jblock >= 0 && md->params[jblock].lower == -INFINITY && md->params[jblock].upper == INFINITY;
  std::ostringstream pre;
  pre << "#define JBLOCK " << jblock << "\n#define JBLOCK_FREE " << (jblock_free ? 1 : 0) << "\n";
  pre << "#define JD " << D << "\n#define JP " << P << "\n#define JNT " << NT << "\n#define JNSUM " << md->n_sum_terms << "\n"
      << "#define JTHREADS " << pl.threads << "\n#define JMINB " << pl.minblocks << "\n#define JWS_SMEM " << pl.ws_smem << "\n#define JWS_OFF " << pl.ws_off << "\n"
      << "#define JN_DERIVED " << md->n_derived << "\n#define JMAX_DIM0 " << max_dim0 << "\n#define JMAXCOL " << kMaxColumns << "\n"
      << "#define JN_RES " << pl.n_res << "\n#define JRES_TOTAL_BYTES " << res_total << "u\n#define JN_RSTAT " << r_entries.size() << "\n"
      << "#define JSTREAM " << (pl.stream_col >= 0 ? 1 : 0) << "\n#define JS_COL " << std::max(pl.stream_col, 0) << "\n#define JS_BEGIN " << s_begin << "\n#define JS_TOTAL " << s_total << "\n"
      << "#define JN_SSTAT " << s_entries.size() << "\n#define JRING_OFF " << pl.ring_off << "u\n#define JRING_STAGES " << pl.ring_stages << "\n#define JRING_TILE " << pl.ring_tile << "\n"
      << "#define JNORM_C0 " << lit(norm_c0) << "\n#define AMWG_REAL 0\n#define AMWG_INT 1\n#define AMWG_BINARY 2\n";
  // accumulators of the plate loop: four (eight measured 5 % slower on config 4 at 3.5 warps per scheduler, profiles/r02_config4_tuning.txt)
  int nacc = 4;
  if (const char* e = getenv("AMWG_JIT_NACC")) { int v = atoi(e); if (v == 4 || v == 8) nacc = v; }
  pre << "#define AMWG_NACC " << nacc << "\n";

  src.prelude = pre.str();
  funcs << tables.str() << step.str() << extra.str() << dfun.str() << "}  // namespace amwg\n";
  src.generated = funcs.str();
  return "";
}


// The specialised form of the full-program sweep (amwg_jit_full_kernel.cuh): for models that evaluate all of log_post at every step
// (no term cache, no statistics): the program -- per configuration of the binary components, if it has variants -- printed as
// straight-line code, bit-identical to what the interpreter computes. Returns "" and fills `src`, else why it does not apply.
static std::string build_source_full(const amwg_model* md, const std::vector<double>& consts, unsigned long long n_chains, int sm_count,
                                     double norm_c0, Source& src) {
  if (md->comp_prog && md->n_terms > 0) return "the model steps with a term cache";
  const int D = md->n_comp, P = md->n_params;
  if (D > 65535 || P > 255) return "too many components / parameters";
  int max_dim0 = 1;
  // JMAX_DIM0 > 1 is what compiles the multi-component stepping in: a [1, n] matrix (dim0 = 1, tests/test_data.js:176) needs it too
  for (int p = 0; p < P; ++p) if (md->params[p].n_comp > 1) max_dim0 = std::max(max_dim0, std::max(md->params[p].dim0, 2));
  std::string err;
  Plan& pl = src.plan;
  pl = Plan();
  pl.col_smem_off.assign(md->n_columns, -1);
  unsigned off = 0;
  for (int c = 0; c < md->n_columns; ++c) {                     // every column resident, or the model stays on the interpreter
    const unsigned bytes = pad16(std::max<size_t>(sizeof(double) * (size_t)md->columns[c].n, 16));
    if (off + bytes > kResidentBudget) return "the data does not fit in shared memory";
    pl.col_smem_off[c] = (int)off; pl.res_col.push_back(c); pl.res_off.push_back((int)off); pl.res_bytes.push_back((int)bytes);
    off += bytes;
  }
  pl.n_res = (int)pl.res_col.size();
  // Bernoulli plates: the 0/1 column as a bit mask (+ one word: "some point is neither 0 nor 1"), built once per launch by the CTA
  pl.bern_mask_off.assign(std::max(md->n_plates, 0), -1);
  std::vector<long long> bm_plate;
  for (int q = 0; q < md->n_plates; ++q) {
    const amwg_plate& pq = md->plates[q];
    if (pq.kind != AMWG_PLATE_BERN_IID || pq.n < 1 || pq.col[0] < 0 || pq.col[0] >= md->n_columns) continue;
    if (pq.iparam[2] < 0 || (long long)pq.iparam[2] + pq.n > md->columns[pq.col[0]].n) return "a plate runs past its column";
    off = (unsigned)pad16(off);
    pl.bern_mask_off[q] = (int)off; bm_plate.push_back(q);
    off += 4u * (unsigned)((pq.n + 31) / 32 + 1);
  }
  { std::string e = choose_shape(pl, off, sizeof(double) * (size_t)D, n_chains, sm_count); if (!e.empty()) return e; }

  std::ostringstream tables, funcs;
  int table_counter = 0, total_insns = 0;
  GenCtx gc;
  gc.md = md; gc.consts = &consts; gc.tables = &tables; gc.table_counter = &table_counter; gc.plan = &pl;
  // the distinct programs: one, or one per configuration of the program-selecting binary components
  const int n_var = md->n_variant_comps ? (1 << md->n_variant_comps) : 1;
  auto emit_program = [&](int pc, const std::string& name, bool derived) -> std::string {
    Inst it;
    if (!decode_program(md, pc, it.ins, nullptr, err)) return "program: " + err;
    total_insns += (int)it.ins.size();
    if (total_insns > kMaxGeneratedInsns) return "the programs are too long to specialise";
    std::vector<Inst> inst{it};
    Emitter em;
    std::vector<Term> terms; std::vector<std::string> cands; std::vector<std::pair<int, std::string>> der;
    std::string why;
    if (!emit_range(gc, inst, 0, it.ins.size(), "m", derived ? CTX_DERIVED : CTX_FULL, em, terms, cands, der, why)) return why;
    if (!em.scopes.empty()) return "unterminated loop";
    if (derived) {
      funcs << "__device__ __forceinline__ void " << name << "(unsigned char* smem, const double* __restrict__ sp, const unsigned long long ss, double* der) {\n" << em.os.str();
      for (auto& d : der) { if (d.first < 0 || d.first >= md->n_derived) return std::string("derived index out of range"); funcs << "    der[" << d.first << "] = " << d.second << ";\n"; }
      funcs << "  (void)smem;\n}\n";
    } else {
      funcs << "__device__ " << (it.ins.size() > 600 ? "__noinline__" : "__forceinline__") << " double " << name
            << "(unsigned char* smem, const double* __restrict__ sp, const unsigned long long ss, const int moved, const double val) {\n    double lp = 0.0;\n"
            << em.os.str() << "    (void)smem;\n    return lp;\n}\n";
    }
    return "";
  };
  for (int v = 0; v < n_var; ++v) {
    const int pc = md->n_variant_comps ? md->variant_logpost[v] : md->logpost_prog;
    std::string e = emit_program(pc, "jit_prog_" + std::to_string(v), false);
    if (!e.empty()) return "log_post: " + e;
  }
  if (md->n_derived > 0)
    for (int v = 0; v < n_var; ++v) {
      const int pc = md->n_variant_comps ? (md->variant_derived ? md->variant_derived[v] : -1) : md->derived_prog;
      if (pc < 0) return "a configuration has no derived program";
      std::string e = emit_program(pc, "jit_der_" + std::to_string(v), true);
      if (!e.empty()) return "derived: " + e;
    }
  // which recorded configuration of the binary components applies (amwg.h variant_*): bit k set when component variant_comps[k] != 0
  auto variant_expr = [&](bool with_moved) {
    std::string e = "0";
    for (int k = 0; k < md->n_variant_comps; ++k) {
      const std::string c = std::to_string(md->variant_comps[k]);
      e += " | ((" + (with_moved ? "CM(" + c + ")" : "ST(" + c + ")") + " != 0.0) ? " + std::to_string(1 << k) + " : 0)";
    }
    return e;
  };
  funcs << "__device__ __forceinline__ double jit_logpost(unsigned char* smem, const double* __restrict__ sp, const unsigned long long ss, const int moved, const double val) {\n";
  if (n_var == 1) funcs << "  return jit_prog_0(smem, sp, ss, moved, val);\n";
  else {
    funcs << "  switch (" << variant_expr(true) << ") {\n";
    for (int v = 0; v < n_var; ++v) funcs << "    case " << v << ": return jit_prog_" << v << "(smem, sp, ss, moved, val);\n";
    funcs << "  }\n  return CUDART_NAN;\n";
  }
  funcs << "}\n";
  if (md->n_derived > 0) {
    funcs << "__device__ __forceinline__ void jit_derived(unsigned char* smem, const double* __restrict__ sp, const unsigned long long ss, double* der) {\n";
    if (n_var == 1) funcs << "  jit_der_0(smem, sp, ss, der);\n";
    else {
      funcs << "  switch (" << variant_expr(false) << ") {\n";
      for (int v = 0; v < n_var; ++v) funcs << "    case " << v << ": jit_der_" << v << "(smem, sp, ss, der); break;\n";
      funcs << "  }\n";
    }
    funcs << "}\n";
  }
  // tables the skeleton reads
  std::ostringstream t2;
  emit_param_tables(t2, md);
  auto int_table = [&](const char* qual, const char* name, const std::vector<long long>& v) {
    t2 << qual << " " << name << "[" << std::max<size_t>(v.size(), 1) << "] = {";
    for (size_t i = 0; i < v.size(); ++i) t2 << (i ? "," : "") << v[i];
    if (v.empty()) t2 << "0";
    t2 << "};\n";
  };
  std::vector<long long> a1, b1, c1;
  for (int k = 0; k < pl.n_res; ++k) { a1.push_back(pl.res_off[k]); b1.push_back(pl.res_col[k]); c1.push_back(pl.res_bytes[k]); }
  int_table("__constant__ unsigned", "JRES_OFF", a1); int_table("__constant__ int", "JRES_COL", b1); int_table("__constant__ unsigned", "JRES_BYTES", c1);
  {
    std::vector<long long> bd, bn, bo;
    for (long long q : bm_plate) {
      const amwg_plate& pq = md->plates[q];
      bd.push_back(pl.col_smem_off[pq.col[0]] + 8 * pq.iparam[2]); bn.push_back(pq.n); bo.push_back(pl.bern_mask_off[q]);
    }
    int_table("__constant__ unsigned", "JBERN_DATA", bd); int_table("__constant__ int", "JBERN_N", bn); int_table("__constant__ unsigned", "JBERN_MASK", bo);
  }
  t2 << "__device__ const long long KCB[" << std::max(md->n_consts, 1) << "] = {";
  for (int i = 0; i < md->n_consts; ++i) t2 << (i ? "," : "") << bits(consts[i]);
  if (md->n_consts == 0) t2 << "0LL";
  t2 << "};\n#define KC(i) __longlong_as_double(KCB[i])\n";
  unsigned long long res_total = 0;
  for (int k = 0; k < pl.n_res; ++k) res_total += (unsigned)pl.res_bytes[k];
  std::ostringstream pre;
  pre << "#define JFULL 1\n#define JD " << D << "\n#define JP " << P << "\n#define JTHREADS " << pl.threads << "\n#define JMINB " << pl.minblocks
      << "\n#define JWS_SMEM " << pl.ws_smem << "\n#define JWS_OFF " << pl.ws_off << "\n#define JN_DERIVED " << md->n_derived << "\n#define JMAX_DIM0 " << max_dim0
      << "\n#define JMAXCOL " << kMaxColumns << "\n#define JN_BERN " << bm_plate.size() << "\n#define JN_RES " << pl.n_res << "\n#define JRES_TOTAL_BYTES " << res_total << "u\n#define JNORM_C0 " << lit(norm_c0)
      << "\n#define AMWG_REAL 0\n#define AMWG_INT 1\n#define AMWG_BINARY 2\n#define AMWG_NACC 4\n";
  src.prelude = pre.str();
  // the generated header: parameter / staging tables and constants, tables the programs index, then the programs and their dispatch
  src.generated = "namespace amwg {\n#define LD(o) lds_f64_sa(smem_u32(smem) + (o))\n" + t2.str() + tables.str() + funcs.str() + "}  // namespace amwg\n";
  src.full = true;
  return "";
}

// ---- NVRTC (loaded at run time) ---------------------------------------------------------------------------------------------------
typedef int nvrtcResult_t;
typedef struct _nvrtcProgram* nvrtcProgram_t;
struct Nvrtc {
  void* h = nullptr;
  nvrtcResult_t (*CreateProgram)(nvrtcProgram_t*, const char*, const char*, int, const char* const*, const char* const*) = nullptr;
  nvrtcResult_t (*DestroyProgram)(nvrtcProgram_t*) = nullptr;
  nvrtcResult_t (*CompileProgram)(nvrtcProgram_t, int, const char* const*) = nullptr;
  nvrtcResult_t (*GetCUBINSize)(nvrtcProgram_t, size_t*) = nullptr;
  nvrtcResult_t (*GetCUBIN)(nvrtcProgram_t, char*) = nullptr;
  nvrtcResult_t (*GetProgramLogSize)(nvrtcProgram_t, size_t*) = nullptr;
  nvrtcResult_t (*GetProgramLog)(nvrtcProgram_t, char*) = nullptr;
  const char* (*GetErrorString)(nvrtcResult_t) = nullptr;
  std::string error;
};

static Nvrtc* nvrtc() {
  static Nvrtc lib;
  static std::once_flag once;
  std::call_once(once, [] {
    const char* names[] = {getenv("AMWG_NVRTC"), "libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so.12", "libnvrtc.so"};
    for (const char* nme : names) {
      if (!nme || !*nme) continue;
      lib.h = dlopen(nme, RTLD_NOW | RTLD_LOCAL);
      if (lib.h) break;
    }
    if (!lib.h) { lib.error = "libnvrtc.so.12 could not be loaded"; return; }
    auto sym = [&](const char* s) { void* p = dlsym(lib.h, s); if (!p) lib.error = std::string("missing NVRTC symbol ") + s; return p; };
    lib.CreateProgram = (decltype(lib.CreateProgram))sym("nvrtcCreateProgram");
    lib.DestroyProgram = (decltype(lib.DestroyProgram))sym("nvrtcDestroyProgram");
    lib.CompileProgram = (decltype(lib.CompileProgram))sym("nvrtcCompileProgram");
    lib.GetCUBINSize = (decltype(lib.GetCUBINSize))sym("nvrtcGetCUBINSize");
    lib.GetCUBIN = (decltype(lib.GetCUBIN))sym("nvrtcGetCUBIN");
    lib.GetProgramLogSize = (decltype(lib.GetProgramLogSize))sym("nvrtcGetProgramLogSize");
    lib.GetProgramLog = (decltype(lib.GetProgramLog))sym("nvrtcGetProgramLog");
    lib.GetErrorString = (decltype(lib.GetErrorString))sym("nvrtcGetErrorString");
  });
  return &lib;
}

// the device headers, embedded at build time (csrc/Makefile: amwg_embedded.inc)
#include "amwg_embedded.inc"

static std::string main_source(const Source& s) {
  return s.prelude + "#include \"amwg_math.cuh\"\n#include \"amwg_ld.cuh\"\n#include \"amwg_tma.cuh\"\n#include \"" +
         (s.full ? "amwg_jit_full_kernel.cuh" : "amwg_jit_kernel.cuh") + "\"\n";
}

// Compile to a cubin for sm_100a. Returns "" on success.
static std::string compile(const Source& s, std::vector<char>& cubin, std::string& log) {
  Nvrtc* nv = nvrtc();
  if (!nv->error.empty()) return nv->error;
  const std::string main_src = main_source(s);
  const char* headers[] = {kSrcMath, kSrcLd, kSrcTma, kSrcJitKernel, kSrcJitFullKernel, s.generated.c_str()};
  const char* names[] = {"amwg_math.cuh", "amwg_ld.cuh", "amwg_tma.cuh", "amwg_jit_kernel.cuh", "amwg_jit_full_kernel.cuh", "amwg_jit_generated.inc"};
  nvrtcProgram_t prog = nullptr;
  nvrtcResult_t rc = nv->CreateProgram(&prog, main_src.c_str(), "amwg_jit_model.cu", 6, headers, names);
  if (rc != 0) return std::string("nvrtcCreateProgram: ") + nv->GetErrorString(rc);
  const char* opts[] = {"--gpu-architecture=sm_100a", "--std=c++17", "--fmad=false", "-lineinfo", "-DAMWG_JIT=1", "--ptxas-options=-v"};
  rc = nv->CompileProgram(prog, 6, opts);
  size_t ln = 0;
  if (nv->GetProgramLogSize(prog, &ln) == 0 && ln > 1) { log.resize(ln); nv->GetProgramLog(prog, &log[0]); }
  if (rc != 0) { std::string e = std::string("nvrtcCompileProgram: ") + nv->GetErrorString(rc); nv->DestroyProgram(&prog); return e; }
  size_t sz = 0;
  rc = nv->GetCUBINSize(prog, &sz);
  if (rc == 0) { cubin.resize(sz); rc = nv->GetCUBIN(prog, cubin.data()); }
  nv->DestroyProgram(&prog);
  if (rc != 0) return std::string("nvrtcGetCUBIN: ") + nv->GetErrorString(rc);
  if (const char* d = getenv("AMWG_JIT_DUMP")) {             // debugging: keep the generated source and the cubin
    std::string base = std::string(d) + "/amwg_jit_" + std::to_string((long long)getpid());
    if (FILE* f = fopen((base + ".cu").c_str(), "w")) { fputs((s.prelude + s.generated).c_str(), f); fclose(f); }
    if (FILE* f = fopen((base + ".cubin").c_str(), "wb")) { fwrite(cubin.data(), 1, cubin.size(), f); fclose(f); }
  }
  return "";
}

static unsigned long long fnv1a(const std::string& s, unsigned long long h = 1469598103934665603ull) {
  for (unsigned char ch : s) { h ^= ch; h *= 1099511628211ull; }
  return h;
}

struct Loaded { cudaLibrary_t lib = nullptr; cudaKernel_t kernel = nullptr; };
static std::mutex g_cache_mu;
static std::map<std::pair<int, unsigned long long>, Loaded> g_cache;      // (device, source hash) -> loaded kernel

// disk cache of cubins (compile once per source): $AMWG_JIT_CACHE or <library dir>/jit_cache
static std::string cache_dir() {
  if (const char* e = getenv("AMWG_JIT_CACHE")) return e;
  Dl_info info;
  if (dladdr((void*)&fnv1a, &info) && info.dli_fname) {
    std::string p(info.dli_fname);
    size_t k = p.find_last_of('/');
    return (k == std::string::npos ? std::string(".") : p.substr(0, k)) + "/jit_cache";
  }
  return "";
}

static bool read_file(const std::string& path, std::vector<char>& out) {
  FILE* f = fopen(path.c_str(), "rb");
  if (!f) return false;
  fseek(f, 0, SEEK_END); long n = ftell(f); fseek(f, 0, SEEK_SET);
  out.resize(n > 0 ? (size_t)n : 0);
  bool ok = n > 0 && fread(out.data(), 1, (size_t)n, f) == (size_t)n;
  fclose(f);
  return ok;
}
static void write_file(const std::string& dir, const std::string& path, const std::vector<char>& data) {
  if (dir.empty()) return;
  std::string cmd_dir = dir;
  mkdir(cmd_dir.c_str(), 0755);
  std::string tmp = path + ".tmp" + std::to_string((long long)getpid());
  FILE* f = fopen(tmp.c_str(), "wb");
  if (!f) return;
  bool ok = fwrite(data.data(), 1, data.size(), f) == data.size();
  fclose(f);
  if (ok) rename(tmp.c_str(), path.c_str()); else remove(tmp.c_str());
}

static std::string get_cubin(const Source& s, std::vector<char>& cubin, std::string& log, bool* from_cache) {
  const unsigned long long h = fnv1a(s.generated, fnv1a(s.prelude, fnv1a(kSrcJitKernel, fnv1a(kSrcJitFullKernel, fnv1a(kSrcTma, fnv1a(kSrcMath, fnv1a(kSrcLd)))))));
  char name[64];
  snprintf(name, sizeof name, "/amwg_%016llx.cubin", h);
  const std::string dir = cache_dir(), path = dir + name;
  if (from_cache) *from_cache = false;
  if (!dir.empty() && !getenv("AMWG_JIT_NO_DISK_CACHE") && read_file(path, cubin)) { if (from_cache) *from_cache = true; return ""; }
  std::string e = compile(s, cubin, log);
  if (e.empty() && !getenv("AMWG_JIT_NO_DISK_CACHE")) write_file(dir, path, cubin);
  return e;
}

}  // namespace jit
