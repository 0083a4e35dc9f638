// amwg_napi.cc -- Node N-API addon: the `amwg_native` module js/mcmc.js and js/distributions.js require.
//
// A thin layer over the C ABI of include/amwg.h (libamwg_b200.so): every AMWG_API export has a binding here, the model
// descriptor js/mcmc.js builds (DeviceModel: plain objects and arrays) is marshalled into an `amwg_model`, results come back as
// typed arrays, and a non-zero status becomes a thrown STRING (the reference throws bare strings, mcmc.js:165,299,315,...).
//
// Build (where Node's headers exist; this image has neither node nor node_api.h, so the repo's tests drive the same C ABI through
// tests/js_host.py, call for call):
//     g++ -std=c++17 -shared -fPIC -I<node headers>/include/node -I../include amwg_napi.cc
//         -L../bayes.js_b200 -lamwg_b200 -Wl,-rpath,'$ORIGIN/../bayes.js_b200' -o amwg_native.node
// The reference has no FFI at all (SURVEY 8(b)): this file is the binding a maintainer adds next to mcmc.js to keep
// `new mcmc.AmwgSampler(params, log_post, data, options)` (mcmc.js:1090-1092) while the stepping moves to the GPU.
#include <node_api.h>

#include <cmath>
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include "../include/amwg.h"

namespace {

// ---- small helpers ----------------------------------------------------------------------------------------------------------
struct Throw { std::string message; };                       // unwound to the binding's entry point, then napi_throw(string)

void check(napi_env env, napi_status st, const char* what) {
  (void)env;
  if (st != napi_ok) throw Throw{std::string("amwg_native: ") + what};
}
void fail_from_library() { throw Throw{amwg_last_error()}; }

napi_value js_undefined(napi_env env) { napi_value v; napi_get_undefined(env, &v); return v; }
napi_value js_number(napi_env env, double x) { napi_value v; check(env, napi_create_double(env, x, &v), "create number"); return v; }
napi_value js_string(napi_env env, const std::string& s) { napi_value v; check(env, napi_create_string_utf8(env, s.c_str(), s.size(), &v), "create string"); return v; }

double to_double(napi_env env, napi_value v) {
  napi_valuetype t;
  check(env, napi_typeof(env, v, &t), "typeof");
  if (t == napi_boolean) { bool b; napi_get_value_bool(env, v, &b); return b ? 1.0 : 0.0; }
  if (t == napi_bigint) { uint64_t u; bool lossless; check(env, napi_get_value_bigint_uint64(env, v, &u, &lossless), "bigint"); return (double)u; }
  double x;
  check(env, napi_get_value_double(env, v, &x), "a number was expected");
  return x;
}
uint64_t to_u64(napi_env env, napi_value v) {                // seeds and chain ids: numbers up to 2^53, or BigInt for the full range
  napi_valuetype t;
  check(env, napi_typeof(env, v, &t), "typeof");
  if (t == napi_bigint) { uint64_t u; bool lossless; check(env, napi_get_value_bigint_uint64(env, v, &u, &lossless), "bigint"); return u; }
  double x = to_double(env, v);
  if (!(x >= 0) || x > 9007199254740992.0 || x != std::floor(x)) throw Throw{"amwg_native: expected a non-negative integer"};
  return (uint64_t)x;
}
bool has(napi_env env, napi_value obj, const char* key) { bool b = false; napi_has_named_property(env, obj, key, &b); return b; }
napi_value prop(napi_env env, napi_value obj, const char* key) {
  napi_value v;
  check(env, napi_get_named_property(env, obj, key, &v), key);
  return v;
}
double num_prop(napi_env env, napi_value obj, const char* key) { return to_double(env, prop(env, obj, key)); }
uint32_t length_of(napi_env env, napi_value arr) {
  bool is_ta = false;
  napi_is_typedarray(env, arr, &is_ta);
  if (is_ta) { size_t n; napi_typedarray_type ty; check(env, napi_get_typedarray_info(env, arr, &ty, &n, nullptr, nullptr, nullptr), "typed array"); return (uint32_t)n; }
  uint32_t n;
  check(env, napi_get_array_length(env, arr, &n), "an array was expected");
  return n;
}
napi_value elem(napi_env env, napi_value arr, uint32_t i) { napi_value v; check(env, napi_get_element(env, arr, i, &v), "array element"); return v; }

// array / typed array of numbers (nested arrays are flattened row-major) -> doubles
void flatten(napi_env env, napi_value v, std::vector<double>& out) {
  bool is_ta = false, is_arr = false;
  napi_is_typedarray(env, v, &is_ta);
  if (is_ta) {
    napi_typedarray_type ty; size_t n; void* data;
    check(env, napi_get_typedarray_info(env, v, &ty, &n, &data, nullptr, nullptr), "typed array");
    if (ty == napi_float64_array) { const double* p = (const double*)data; out.insert(out.end(), p, p + n); return; }
    if (ty == napi_int32_array) { const int32_t* p = (const int32_t*)data; for (size_t i = 0; i < n; ++i) out.push_back(p[i]); return; }
    throw Throw{"amwg_native: Float64Array or Int32Array expected"};
  }
  napi_is_array(env, v, &is_arr);
  if (is_arr) { uint32_t n = length_of(env, v); for (uint32_t i = 0; i < n; ++i) flatten(env, elem(env, v, i), out); return; }
  out.push_back(to_double(env, v));
}
std::vector<double> doubles(napi_env env, napi_value v) { std::vector<double> out; flatten(env, v, out); return out; }
std::vector<int32_t> ints(napi_env env, napi_value v) {
  std::vector<double> d = doubles(env, v);
  std::vector<int32_t> out(d.size());
  for (size_t i = 0; i < d.size(); ++i) out[i] = (int32_t)d[i];
  return out;
}
napi_value f64_array(napi_env env, const double* src, size_t n) {
  void* data = nullptr;
  napi_value buf, ta;
  check(env, napi_create_arraybuffer(env, n * sizeof(double), &data, &buf), "arraybuffer");
  if (n) std::memcpy(data, src, n * sizeof(double));
  check(env, napi_create_typedarray(env, napi_float64_array, n, buf, 0, &ta), "Float64Array");
  return ta;
}
napi_value i32_array(napi_env env, const int32_t* src, size_t n) {
  void* data = nullptr;
  napi_value buf, ta;
  check(env, napi_create_arraybuffer(env, n * sizeof(int32_t), &data, &buf), "arraybuffer");
  if (n) std::memcpy(data, src, n * sizeof(int32_t));
  check(env, napi_create_typedarray(env, napi_int32_array, n, buf, 0, &ta), "Int32Array");
  return ta;
}

// ---- the handle: an external whose finalizer destroys the sampler -------------------------------------------------------------
struct Handle {
  amwg_sampler* s = nullptr;
  int n_comp = 0, n_derived = 0;
  uint64_t n_chains = 0;
};
void finalize_handle(napi_env, void* data, void*) {
  Handle* h = (Handle*)data;
  if (h->s) amwg_destroy(h->s);
  delete h;
}
Handle* handle_of(napi_env env, napi_value v) {
  void* p = nullptr;
  check(env, napi_get_value_external(env, v, &p), "a sampler handle was expected");
  Handle* h = (Handle*)p;
  if (!h || !h->s) throw Throw{"amwg_native: the sampler has been destroyed"};
  return h;
}

// ---- model marshalling: the descriptor of js/mcmc.js (DeviceModel) -> amwg_model ----------------------------------------------
struct Model {
  amwg_model m{};
  std::vector<amwg_param> params;
  std::vector<double> init, consts;
  std::vector<amwg_comp_options> opts;
  std::vector<int32_t> code, fold_prog, fold_dst, comp_prog, touch_off, touch_terms, block_params, term_block_comp, variant_comps, variant_logpost, variant_derived;
  std::vector<std::vector<double>> columns;
  std::vector<amwg_column> column_refs;
  std::vector<amwg_plate> plates;
};

void marshal(napi_env env, napi_value d, Model& M) {
  napi_value a = prop(env, d, "params");
  for (uint32_t i = 0, n = length_of(env, a); i < n; ++i) {
    napi_value p = elem(env, a, i);
    amwg_param q{};
    q.type = (int32_t)num_prop(env, p, "type"); q.n_comp = (int32_t)num_prop(env, p, "n_comp"); q.dim0 = (int32_t)num_prop(env, p, "dim0");
    q.comp_offset = (int32_t)num_prop(env, p, "comp_offset"); q.lower = num_prop(env, p, "lower"); q.upper = num_prop(env, p, "upper");
    M.params.push_back(q);
  }
  M.init = doubles(env, prop(env, d, "init"));
  a = prop(env, d, "comp_options");
  for (uint32_t i = 0, n = length_of(env, a); i < n; ++i) {
    napi_value o = elem(env, a, i);
    amwg_comp_options c{};
    c.prop_log_scale = num_prop(env, o, "prop_log_scale"); c.batch_size = num_prop(env, o, "batch_size"); c.max_adaptation = num_prop(env, o, "max_adaptation");
    c.initial_adaptation = num_prop(env, o, "initial_adaptation"); c.target_accept_rate = num_prop(env, o, "target_accept_rate");
    c.is_adapting = num_prop(env, o, "is_adapting") != 0 ? 1 : 0;
    M.opts.push_back(c);
  }
  if (M.opts.size() != M.init.size()) throw Throw{"amwg_native: comp_options and init differ in length"};
  M.code = ints(env, prop(env, d, "code"));
  M.consts = doubles(env, prop(env, d, "consts"));
  a = prop(env, d, "columns");
  for (uint32_t i = 0, n = length_of(env, a); i < n; ++i) M.columns.push_back(doubles(env, elem(env, a, i)));
  for (auto& c : M.columns) M.column_refs.push_back(amwg_column{c.data(), (int64_t)c.size()});
  a = prop(env, d, "plates");
  for (uint32_t i = 0, n = length_of(env, a); i < n; ++i) {
    napi_value p = elem(env, a, i);
    amwg_plate q{};
    q.kind = (int32_t)num_prop(env, p, "kind"); q.n = (int32_t)num_prop(env, p, "n");
    std::vector<int32_t> col = ints(env, prop(env, p, "col")), ip = ints(env, prop(env, p, "iparam"));
    for (int k = 0; k < 4; ++k) { q.col[k] = k < (int)col.size() ? col[k] : -1; q.iparam[k] = k < (int)ip.size() ? ip[k] : 0; }
    M.plates.push_back(q);
  }
  M.fold_prog = ints(env, prop(env, d, "fold_prog")); M.fold_dst = ints(env, prop(env, d, "fold_dst"));
  M.comp_prog = ints(env, prop(env, d, "comp_prog")); M.touch_off = ints(env, prop(env, d, "touch_off")); M.touch_terms = ints(env, prop(env, d, "touch_terms"));
  M.block_params = ints(env, prop(env, d, "block_params")); M.term_block_comp = ints(env, prop(env, d, "term_block_comp"));
  M.variant_comps = ints(env, prop(env, d, "variant_comps")); M.variant_logpost = ints(env, prop(env, d, "variant_logpost")); M.variant_derived = ints(env, prop(env, d, "variant_derived"));

  amwg_model& m = M.m;
  m.abi_version = AMWG_ABI_VERSION;
  m.n_params = (int32_t)M.params.size(); m.params = M.params.data();
  m.n_comp = (int32_t)M.init.size(); m.init = M.init.data(); m.comp_options = M.opts.data();
  m.n_code = (int32_t)M.code.size(); m.code = M.code.data();
  m.logpost_prog = (int32_t)num_prop(env, d, "logpost_prog"); m.derived_prog = (int32_t)num_prop(env, d, "derived_prog"); m.n_derived = (int32_t)num_prop(env, d, "n_derived");
  m.n_consts = (int32_t)M.consts.size(); m.consts = M.consts.data();
  m.n_columns = (int32_t)M.column_refs.size(); m.columns = M.column_refs.data();
  m.n_plates = (int32_t)M.plates.size(); m.plates = M.plates.data();
  m.n_fold = (int32_t)M.fold_prog.size(); m.fold_prog = M.fold_prog.data(); m.fold_dst = M.fold_dst.data();
  m.n_terms = (int32_t)num_prop(env, d, "n_terms");
  const bool cached = m.n_terms > 0;
  m.comp_prog = cached ? M.comp_prog.data() : nullptr; m.touch_off = cached ? M.touch_off.data() : nullptr; m.touch_terms = cached ? M.touch_terms.data() : nullptr;
  m.n_block_params = (int32_t)M.block_params.size();
  m.block_params = M.block_params.empty() ? nullptr : M.block_params.data(); m.term_block_comp = M.block_params.empty() ? nullptr : M.term_block_comp.data();
  m.stat_prog = (int32_t)num_prop(env, d, "stat_prog"); m.n_sum_terms = (int32_t)num_prop(env, d, "n_sum_terms");
  m.n_variant_comps = (int32_t)M.variant_comps.size();
  if (M.variant_derived.empty()) M.variant_derived.push_back(-1);
  if (M.variant_comps.empty()) M.variant_comps.push_back(0);
  if (M.variant_logpost.empty()) M.variant_logpost.push_back(0);
  m.variant_comps = M.variant_comps.data(); m.variant_logpost = M.variant_logpost.data(); m.variant_derived = M.variant_derived.data();
}

// ---- argument plumbing ------------------------------------------------------------------------------------------------------------
struct Args {
  napi_value v[10];
  size_t n = 10;
  Args(napi_env env, napi_callback_info info) { check(env, napi_get_cb_info(env, info, &n, v, nullptr, nullptr), "arguments"); }
  napi_value at(size_t i) const { if (i >= n) throw Throw{"amwg_native: missing argument"}; return v[i]; }
};
template <typename F>
napi_value guarded(napi_env env, F&& body) {                   // C++ exception -> JS `throw "<string>"`
  try { return body(); }
  catch (const Throw& t) { napi_throw(env, js_string(env, t.message)); }
  catch (const std::exception& e) { napi_throw(env, js_string(env, std::string("amwg_native: ") + e.what())); }
  return nullptr;
}
#define BINDING(name) napi_value name(napi_env env, napi_callback_info info) { return guarded(env, [&]() -> napi_value { Args a(env, info);
#define END_BINDING }); }

// ---- the bindings, one per AMWG_API export -------------------------------------------------------------------------------------------
// create(descriptor, n_chains, first_chain, seed, device) -> handle            amwg_create   (mcmc.js:1090-1092, 940-966)
BINDING(create)
  Model M;
  marshal(env, a.at(0), M);
  Handle* h = new Handle();
  if (amwg_create(&M.m, to_u64(env, a.at(1)), to_u64(env, a.at(2)), to_u64(env, a.at(3)), (int)to_double(env, a.at(4)), &h->s) != 0) { delete h; fail_from_library(); }
  h->n_comp = M.m.n_comp; h->n_derived = M.m.n_derived; h->n_chains = amwg_n_chains(h->s);
  napi_value ext;
  check(env, napi_create_external(env, h, finalize_handle, nullptr, &ext), "external");
  return ext;
END_BINDING
// destroy(handle)                                                               amwg_destroy
BINDING(destroy)
  void* p = nullptr;
  check(env, napi_get_value_external(env, a.at(0), &p), "a sampler handle was expected");
  Handle* h = (Handle*)p;
  if (h && h->s) { amwg_destroy(h->s); h->s = nullptr; }
  return js_undefined(env);
END_BINDING
// burn(handle, n)                                                               amwg_burn     (mcmc.js:1035-1039)
BINDING(burn)
  if (amwg_burn(handle_of(env, a.at(0))->s, (int64_t)to_double(env, a.at(1))) != 0) fail_from_library();
  return js_undefined(env);
END_BINDING
// sample(handle, n, thin, monitor[]) -> Float64Array [rows][monitor][chains]   amwg_sample   (mcmc.js:1005-1030)
BINDING(sample)
  Handle* h = handle_of(env, a.at(0));
  const int64_t n = (int64_t)to_double(env, a.at(1)), thin = (int64_t)to_double(env, a.at(2));
  std::vector<int32_t> mon = ints(env, a.at(3));
  const size_t rows = (n <= 0 || thin < 1) ? 0 : (size_t)((n + thin - 1) / thin), total = rows * mon.size() * (size_t)h->n_chains;
  void* data = nullptr;
  napi_value buf, ta;
  check(env, napi_create_arraybuffer(env, total * sizeof(double), &data, &buf), "arraybuffer");
  if (amwg_sample(h->s, n, thin, mon.data(), (int32_t)mon.size(), (double*)data) != 0) fail_from_library();
  check(env, napi_create_typedarray(env, napi_float64_array, total, buf, 0, &ta), "Float64Array");
  return ta;
END_BINDING
// sample_device(handle, n, thin, monitor[], device_pointer BigInt)             amwg_sample_device (draws stay in HBM)
BINDING(sample_device)
  Handle* h = handle_of(env, a.at(0));
  std::vector<int32_t> mon = ints(env, a.at(3));
  if (amwg_sample_device(h->s, (int64_t)to_double(env, a.at(1)), (int64_t)to_double(env, a.at(2)), mon.data(), (int32_t)mon.size(), (double*)(uintptr_t)to_u64(env, a.at(4))) != 0)
    fail_from_library();
  return js_undefined(env);
END_BINDING
// get_state(handle) -> Float64Array [n_comp + n_derived][chains]               amwg_get_state (mcmc.js:985-997)
BINDING(get_state)
  Handle* h = handle_of(env, a.at(0));
  std::vector<double> out((size_t)(h->n_comp + h->n_derived) * (size_t)h->n_chains);
  if (amwg_get_state(h->s, out.data()) != 0) fail_from_library();
  return f64_array(env, out.data(), out.size());
END_BINDING
// get_log_post(handle) -> Float64Array [chains]                                 amwg_get_log_post (mcmc.js:958-960)
BINDING(get_log_post)
  Handle* h = handle_of(env, a.at(0));
  std::vector<double> out((size_t)h->n_chains);
  if (amwg_get_log_post(h->s, out.data()) != 0) fail_from_library();
  return f64_array(env, out.data(), out.size());
END_BINDING
// set_adapting(handle, flag)                                                    amwg_set_adapting (mcmc.js:1060-1073)
BINDING(set_adapting)
  if (amwg_set_adapting(handle_of(env, a.at(0))->s, to_double(env, a.at(1)) != 0 ? 1 : 0) != 0) fail_from_library();
  return js_undefined(env);
END_BINDING
// info(handle) -> {scalars, prop_log_scale, acceptance_count}                    amwg_info     (mcmc.js:563-571)
BINDING(info)
  Handle* h = handle_of(env, a.at(0));
  const size_t DC = (size_t)h->n_comp * (size_t)h->n_chains;
  std::vector<double> scal((size_t)h->n_comp * 3), pls(DC);
  std::vector<int32_t> acc(DC);
  if (amwg_info(h->s, scal.data(), pls.data(), acc.data()) != 0) fail_from_library();
  napi_value o;
  check(env, napi_create_object(env, &o), "object");
  napi_set_named_property(env, o, "scalars", f64_array(env, scal.data(), scal.size()));
  napi_set_named_property(env, o, "prop_log_scale", f64_array(env, pls.data(), pls.size()));
  napi_set_named_property(env, o, "acceptance_count", i32_array(env, acc.data(), acc.size()));
  return o;
END_BINDING
BINDING(kernel_launches) return js_number(env, (double)amwg_kernel_launches(handle_of(env, a.at(0))->s)); END_BINDING            // amwg_kernel_launches
BINDING(last_sweep_kernel_ms) return js_number(env, amwg_last_sweep_kernel_ms(handle_of(env, a.at(0))->s)); END_BINDING             // amwg_last_sweep_kernel_ms
BINDING(n_chains) return js_number(env, (double)amwg_n_chains(handle_of(env, a.at(0))->s)); END_BINDING                              // amwg_n_chains
BINDING(last_error) (void)a; return js_string(env, amwg_last_error()); END_BINDING                                                   // amwg_last_error
BINDING(abi_version) (void)a; return js_number(env, amwg_abi_version()); END_BINDING                                                 // amwg_abi_version
// ld_eval(opcode, rows[][]) -> Float64Array                                      amwg_ld_eval  (distributions.js:63-284 on the device)
BINDING(ld_eval)
  napi_value rows = a.at(1);
  const uint32_t n = length_of(env, rows);
  std::vector<double> flat;
  uint32_t arity = 0;
  for (uint32_t i = 0; i < n; ++i) {
    std::vector<double> r = doubles(env, elem(env, rows, i));
    if (i == 0) arity = (uint32_t)r.size();
    if (r.size() != arity) throw Throw{"amwg_native: ld_eval rows differ in length"};
    flat.insert(flat.end(), r.begin(), r.end());
  }
  std::vector<double> out(n);
  int device = a.n > 2 ? (int)to_double(env, a.at(2)) : 0;
  if (n && amwg_ld_eval((int32_t)to_double(env, a.at(0)), flat.data(), (int32_t)arity, n, out.data(), device) != 0) fail_from_library();
  return f64_array(env, out.data(), out.size());
END_BINDING
// primitive_eval(kind, x[], seed, chain) -> Float64Array                          amwg_primitive_eval
BINDING(primitive_eval)
  std::vector<double> x = doubles(env, a.at(1)), out(x.size());
  if (!x.empty() && amwg_primitive_eval((int32_t)to_double(env, a.at(0)), x.data(), (int64_t)x.size(), to_u64(env, a.at(2)), to_u64(env, a.at(3)), out.data(), a.n > 4 ? (int)to_double(env, a.at(4)) : 0) != 0)
    fail_from_library();
  return f64_array(env, out.data(), out.size());
END_BINDING
// stream_uniforms(seed, chain, first, count): Math.random() calls #first .. of the Philox stream (seed, chain)   amwg_primitive_eval kind 2
BINDING(stream_uniforms)
  const uint64_t first = to_u64(env, a.at(2)), count = to_u64(env, a.at(3));
  std::vector<double> x((size_t)(first + count), 0.0), out(x.size());
  if (!x.empty() && amwg_primitive_eval(2, x.data(), (int64_t)x.size(), to_u64(env, a.at(0)), to_u64(env, a.at(1)), out.data(), 0) != 0) fail_from_library();
  return f64_array(env, out.data() + first, (size_t)count);
END_BINDING
// device_log(x): Math.log as the device computes it                             amwg_primitive_eval kind 0
BINDING(device_log)
  double x = to_double(env, a.at(0)), out = 0.0;
  if (amwg_primitive_eval(0, &x, 1, 0, 0, &out, 0) != 0) fail_from_library();
  return js_number(env, out);
END_BINDING
// summary_moments(device, device_pointer BigInt, rows, entries, chains) -> Float64Array [entries][4]     amwg_summary_moments
BINDING(summary_moments)
  const int32_t entries = (int32_t)to_double(env, a.at(3));
  std::vector<double> out((size_t)entries * 4);
  if (amwg_summary_moments((int)to_double(env, a.at(0)), (const double*)(uintptr_t)to_u64(env, a.at(1)), (int64_t)to_double(env, a.at(2)), entries, (int64_t)to_double(env, a.at(4)), out.data()) != 0)
    fail_from_library();
  return f64_array(env, out.data(), out.size());
END_BINDING
// summary_digit_hist(device, samples ptr, rows, entries, chains, pass, prefix ptr, n_prefix, counts ptr)    amwg_summary_digit_hist
BINDING(summary_digit_hist)
  if (amwg_summary_digit_hist((int)to_double(env, a.at(0)), (const double*)(uintptr_t)to_u64(env, a.at(1)), (int64_t)to_double(env, a.at(2)), (int32_t)to_double(env, a.at(3)),
                              (int64_t)to_double(env, a.at(4)), (int32_t)to_double(env, a.at(5)), (const uint64_t*)(uintptr_t)to_u64(env, a.at(6)), (int32_t)to_double(env, a.at(7)),
                              (uint64_t*)(uintptr_t)to_u64(env, a.at(8))) != 0)
    fail_from_library();
  return js_undefined(env);
END_BINDING
// summary_autocov(device, samples ptr, rows, entries, chains, threshold ptr (0: none), lag0, n_lags) -> Float64Array [entries][3 + n_lags]
//                                                                                 amwg_summary_autocov (every entry live)
BINDING(summary_autocov)
  const int32_t entries = (int32_t)to_double(env, a.at(3)), n_lags = (int32_t)to_double(env, a.at(7));
  std::vector<double> out((size_t)std::max(entries, 0) * (size_t)(3 + std::max(n_lags, 0)));
  if (amwg_summary_autocov((int)to_double(env, a.at(0)), (const double*)(uintptr_t)to_u64(env, a.at(1)), (int64_t)to_double(env, a.at(2)), entries,
                           (int64_t)to_double(env, a.at(4)), (const double*)(uintptr_t)to_u64(env, a.at(5)), nullptr, 0, (int32_t)to_double(env, a.at(6)),
                           n_lags, out.data()) != 0)
    fail_from_library();
  return f64_array(env, out.data(), out.size());
END_BINDING
// summary_rank_keys(device, samples ptr, rows, entries, chains, entry, center (NaN: no fold), keys ptr, vals ptr)   amwg_summary_rank_keys
BINDING(summary_rank_keys)
  const double center = to_double(env, a.at(6));
  if (amwg_summary_rank_keys((int)to_double(env, a.at(0)), (const double*)(uintptr_t)to_u64(env, a.at(1)), (int64_t)to_double(env, a.at(2)),
                             (int32_t)to_double(env, a.at(3)), (int64_t)to_double(env, a.at(4)), (int32_t)to_double(env, a.at(5)),
                             std::isnan(center) ? nullptr : &center, (uint64_t*)(uintptr_t)to_u64(env, a.at(7)), (uint32_t*)(uintptr_t)to_u64(env, a.at(8))) != 0)
    fail_from_library();
  return js_undefined(env);
END_BINDING
// summary_rank_sort(device, keys ptr, vals ptr, n, keys_alt ptr, vals_alt ptr) -> [passes run, skipped, in alt]   amwg_summary_rank_sort
BINDING(summary_rank_sort)
  int32_t passes[3] = {0, 0, 0};
  if (amwg_summary_rank_sort((int)to_double(env, a.at(0)), (uint64_t*)(uintptr_t)to_u64(env, a.at(1)), (uint32_t*)(uintptr_t)to_u64(env, a.at(2)),
                             (int64_t)to_double(env, a.at(3)), (uint64_t*)(uintptr_t)to_u64(env, a.at(4)), (uint32_t*)(uintptr_t)to_u64(env, a.at(5)), passes) != 0)
    fail_from_library();
  const double p[3] = {(double)passes[0], (double)passes[1], (double)passes[2]};
  return f64_array(env, p, 3);
END_BINDING
// summary_rank_runs(device, sorted keys ptr, sorted vals ptr, weights ptr (0: none), weight scan ptr (0: none), n, run_id ptr,
//                   run_keys ptr (0), run_counts ptr) -> runs                                   amwg_summary_rank_runs
BINDING(summary_rank_runs)
  int64_t runs = 0;
  if (amwg_summary_rank_runs((int)to_double(env, a.at(0)), (const uint64_t*)(uintptr_t)to_u64(env, a.at(1)), (const uint32_t*)(uintptr_t)to_u64(env, a.at(2)),
                             (const int64_t*)(uintptr_t)to_u64(env, a.at(3)), (int64_t*)(uintptr_t)to_u64(env, a.at(4)), (int64_t)to_double(env, a.at(5)),
                             (uint32_t*)(uintptr_t)to_u64(env, a.at(6)), (uint64_t*)(uintptr_t)to_u64(env, a.at(7)), (int64_t*)(uintptr_t)to_u64(env, a.at(8)),
                             &runs) != 0)
    fail_from_library();
  return js_number(env, (double)runs);
END_BINDING
// summary_rank_z(device, run_counts ptr, n_runs, offset, total, run_z ptr)      amwg_summary_rank_z
BINDING(summary_rank_z)
  if (amwg_summary_rank_z((int)to_double(env, a.at(0)), (const int64_t*)(uintptr_t)to_u64(env, a.at(1)), (int64_t)to_double(env, a.at(2)),
                          (int64_t)to_double(env, a.at(3)), (int64_t)to_double(env, a.at(4)), (double*)(uintptr_t)to_u64(env, a.at(5))) != 0)
    fail_from_library();
  return js_undefined(env);
END_BINDING
// summary_rank_scatter(device, sorted vals ptr, run_id ptr, n, run_z ptr, out ptr, entries, chains, entry)   amwg_summary_rank_scatter
BINDING(summary_rank_scatter)
  if (amwg_summary_rank_scatter((int)to_double(env, a.at(0)), (const uint32_t*)(uintptr_t)to_u64(env, a.at(1)), (const uint32_t*)(uintptr_t)to_u64(env, a.at(2)),
                                (int64_t)to_double(env, a.at(3)), (const double*)(uintptr_t)to_u64(env, a.at(4)), (double*)(uintptr_t)to_u64(env, a.at(5)),
                                (int32_t)to_double(env, a.at(6)), (int64_t)to_double(env, a.at(7)), (int32_t)to_double(env, a.at(8))) != 0)
    fail_from_library();
  return js_undefined(env);
END_BINDING
// peak_fp64(device, reps) -> {tflops, ms}                                        amwg_peak_fp64
BINDING(peak_fp64)
  double tf = 0.0, ms = 0.0;
  if (amwg_peak_fp64((int)to_double(env, a.at(0)), a.n > 1 ? (int)to_double(env, a.at(1)) : 3, &tf, &ms) != 0) fail_from_library();
  napi_value o;
  check(env, napi_create_object(env, &o), "object");
  napi_set_named_property(env, o, "tflops", js_number(env, tf));
  napi_set_named_property(env, o, "ms", js_number(env, ms));
  return o;
END_BINDING
// jit_status(handle) -> "specialised: ..." | "interpreter: ..."                  amwg_jit_status
BINDING(jit_status)
  char note[1024];
  note[0] = 0;
  const int on = amwg_jit_status(handle_of(env, a.at(0))->s, note, sizeof note);
  return js_string(env, std::string(on ? "specialised: " : "interpreter: ") + note);
END_BINDING
// jit_compile_check(descriptor, n_chains) -> {rc, log}                           amwg_jit_compile_check
BINDING(jit_compile_check)
  Model M;
  marshal(env, a.at(0), M);
  std::vector<char> log(1 << 16);
  const int rc = amwg_jit_compile_check(&M.m, to_u64(env, a.at(1)), log.data(), (int64_t)log.size(), nullptr, 0);
  napi_value o;
  check(env, napi_create_object(env, &o), "object");
  napi_set_named_property(env, o, "rc", js_number(env, rc));
  napi_set_named_property(env, o, "log", js_string(env, log.data()));
  return o;
END_BINDING

}  // namespace

NAPI_MODULE_INIT() {
  const struct { const char* name; napi_callback fn; } table[] = {
      {"create", create}, {"destroy", destroy}, {"burn", burn}, {"sample", sample}, {"sample_device", sample_device}, {"get_state", get_state},
      {"get_log_post", get_log_post}, {"set_adapting", set_adapting}, {"info", info}, {"kernel_launches", kernel_launches},
      {"last_sweep_kernel_ms", last_sweep_kernel_ms}, {"n_chains", n_chains}, {"last_error", last_error}, {"abi_version", abi_version},
      {"ld_eval", ld_eval}, {"primitive_eval", primitive_eval}, {"stream_uniforms", stream_uniforms}, {"device_log", device_log},
      {"summary_moments", summary_moments}, {"summary_digit_hist", summary_digit_hist}, {"summary_autocov", summary_autocov},
      {"summary_rank_keys", summary_rank_keys}, {"summary_rank_sort", summary_rank_sort}, {"summary_rank_runs", summary_rank_runs},
      {"summary_rank_z", summary_rank_z}, {"summary_rank_scatter", summary_rank_scatter}, {"peak_fp64", peak_fp64}, {"jit_status", jit_status},
      {"jit_compile_check", jit_compile_check}};
  for (const auto& e : table) {
    napi_value fn;
    if (napi_create_function(env, e.name, NAPI_AUTO_LENGTH, e.fn, nullptr, &fn) != napi_ok) return nullptr;
    if (napi_set_named_property(env, exports, e.name, fn) != napi_ok) return nullptr;
  }
  return exports;
}
