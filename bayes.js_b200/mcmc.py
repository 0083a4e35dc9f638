"""``mcmc`` -- host-side mirror of /root/reference/mcmc.js for the one path this package accelerates:

    sampler = mcmc.AmwgSampler(params, log_post, data, options)     # mcmc.js:1090-1092, 940-966
    sampler.burn(1000); samples = sampler.sample(5000)              # mcmc.js:1035-1039, 1005-1030

Same names, argument meaning and error strings as the reference; the stepping itself happens in
libamwg_b200.so (CUDA, sm_100a) for ``options["chains"]`` independent chains at once.  The host
language is Python because no JavaScript engine exists in this image; INTEGRATION.md shows the N-API
binding a Node host would put under the same `mcmc` / `ld` module names.

New, non-reference options (the many-chain setting needs them): ``chains`` (default 1: output is
shaped exactly like the reference's), ``seed``, ``device``, ``distributed``, ``first_chain`` (global id of
the first chain, default 0), ``faithful`` (no factorised likelihood plates: bit-faithful, slower).
"""
from __future__ import annotations

import copy
import ctypes as C
import math
import os
import sys
import time
from typing import Any, Dict, List, Optional

import numpy as np

from . import _ffi
from ._ffi import AmwgColumn, AmwgCompOptions, AmwgModel, AmwgParam, AmwgPlate, BINARY, INT, REAL
from .tracer import JsThrow, Math, Sym, points, trace, where  # noqa: F401  (re-exported)

Infinity = float("inf")
_TYPE_CODE = {"real": REAL, "int": INT, "binary": BINARY}


# ------------------------------------------------------------------------------------------------
# helpers -- mcmc.js:131-303
# ------------------------------------------------------------------------------------------------
def is_number(x) -> bool:
    """mcmc.js:131-133"""
    return isinstance(x, (int, float, np.integer, np.floating)) and not isinstance(x, bool)


def create_array(dim, init):
    """mcmc.js:147-168 -- nested list of shape `dim`; `init` is a value or a zero-arg function."""
    dim = list(dim)
    if len(dim) == 1:
        return [init() if callable(init) else init for _ in range(int(dim[0]))]
    if len(dim) > 1:
        return [create_array(dim[1:], init) for _ in range(int(dim[0]))]
    raise JsThrow("create_array can't create a dimensionless array")


def array_dim(a) -> List[int]:
    """mcmc.js:178-184"""
    if len(a) > 0 and isinstance(a[0], (list, tuple, np.ndarray)):
        return [len(a)] + array_dim(a[0])
    return [len(a)]


def array_equal(a1, a2) -> bool:
    """mcmc.js:191-205"""
    if len(a1) != len(a2):
        return False
    for x, y in zip(a1, a2):
        if isinstance(x, (list, tuple)) and isinstance(y, (list, tuple)):
            if not array_equal(x, y):
                return False
        elif x != y:
            return False
    return True


def _flatten(a) -> List[Any]:
    if isinstance(a, (list, tuple, np.ndarray)):
        out: List[Any] = []
        for v in a:
            out.extend(_flatten(v))
        return out
    return [a]


def _js_truthy(v) -> bool:
    """JS truthiness for the `a || b` option merge (mcmc.js:873-878): undefined/null/0/NaN/false/"" are falsy, arrays are truthy."""
    if v is None or v is False:
        return False
    if isinstance(v, str):
        return v != ""
    if is_number(v):
        return not (v == 0 or v != v)
    return True


def _js_join(a) -> str:
    """Array -> string as JS string concatenation does it ("" + [1,[2,3]] === "1,2,3")."""
    return ",".join(_js_join(v) if isinstance(v, (list, tuple)) else _js_num(v) for v in a)


def _js_num(v) -> str:
    if isinstance(v, float):
        if v == Infinity: return "Infinity"
        if v == -Infinity: return "-Infinity"
        if v != v: return "NaN"
        if v == int(v) and abs(v) < 1e21: return str(int(v))
    return str(v)


def get_option(option_name: str, options: Optional[dict], defaul_value):
    """mcmc.js:280-285 -- undefined and null fall back to the default; 0 / false do not."""
    options = options or {}
    v = options.get(option_name) if option_name in options else None
    return v if v is not None else defaul_value


def get_multidim_option(option_name: str, options: Optional[dict], dim, defaul_value):
    """mcmc.js:293-303"""
    value = get_option(option_name, options, defaul_value)
    if not isinstance(value, (list, tuple)):
        value = create_array(dim, value)
    if not array_equal(array_dim(value), list(dim)):
        raise JsThrow("The option " + option_name + " is of dimension [" + _js_join(array_dim(value)) +
                      "] but should be [" + _js_join(list(dim)) + "].")
    return value


def js_round(x: float) -> float:
    """Math.round: halves toward +infinity."""
    r = math.ceil(x)
    if r - 0.5 > x:
        r -= 1.0
    return float(r)


# ------------------------------------------------------------------------------------------------
# parameter handling -- mcmc.js:313-403
# ------------------------------------------------------------------------------------------------
def param_init_fixed(type, lower, upper):
    """mcmc.js:313-341"""
    if lower > upper:
        raise JsThrow("Can not initialize parameter where lower bound > upper bound")
    if type == "real":
        if lower == -Infinity and upper == Infinity: return 0.5
        if lower == -Infinity: return upper - 0.5
        if upper == Infinity: return lower + 0.5
        if lower <= upper: return (lower + upper) / 2
    elif type == "int":
        if lower == -Infinity and upper == Infinity: return 1
        if lower == -Infinity: return upper - 1
        if upper == Infinity: return lower + 1
        if lower <= upper: return js_round((lower + upper) / 2)
    elif type == "binary":
        return 1
    raise JsThrow("Could not initialize parameter of type " + str(type) + "[" + _js_num(lower) + ", " + _js_num(upper) + "]")


def complete_params(params_to_complete: Dict[str, dict], param_init=param_init_fixed) -> Dict[str, dict]:
    """mcmc.js:357-403 -- returns a completed deep copy; the input is not modified."""
    params = copy.deepcopy(params_to_complete)
    for param_name, param in params.items():
        if "type" not in param:
            param["type"] = "real"
        if "dim" not in param:
            param["dim"] = [1]
        if is_number(param["dim"]):
            param["dim"] = [param["dim"]]
        param["dim"] = list(param["dim"])
        if param["type"] == "binary":
            param["upper"] = 1
            param["lower"] = 0
        if "upper" not in param:
            param["upper"] = Infinity
        if "lower" not in param:
            param["lower"] = -Infinity
        if "init" in param:
            if array_equal(param["dim"], [1]) and callable(param["init"]):
                param["init"] = param["init"]()
            elif not array_equal(param["dim"], [1]) and not isinstance(param["init"], (list, tuple, np.ndarray)):
                param["init"] = create_array(param["dim"], param["init"])
        else:
            if array_equal(param["dim"], [1]):
                param["init"] = param_init(param["type"], param["lower"], param["upper"])
            else:
                param["init"] = create_array(
                    param["dim"], lambda p=param: param_init(p["type"], p["lower"], p["upper"]))
    return params


# ------------------------------------------------------------------------------------------------
# exported RNG helpers -- mcmc.js:31-54 (kept for the export list; the sampler does not use them)
# ------------------------------------------------------------------------------------------------
class _HostStream:
    """`Math.random()` for the exported helpers: the Philox stream definition of the sampler, drawn on the device."""
    seed = 0x6d636d63
    chain = 0xFFFFFFFF
    n = 0
    _block = np.empty(0)
    _block0 = 0

    @classmethod
    def random(cls) -> float:
        k = cls.n - cls._block0
        if not (0 <= k < cls._block.size):
            want = cls.n + 1024
            buf = np.empty(want)
            _ffi.check(_ffi.lib().amwg_primitive_eval(2, np.zeros(want).ctypes.data, want, cls.seed, cls.chain,
                                                      buf.ctypes.data, _default_device()))
            cls._block, cls._block0 = buf[cls.n:], cls.n
            k = 0
        cls.n += 1
        return float(cls._block[k])


def set_random_stream(seed: int, chain: int = 0, position: int = 0):
    """Not in the reference (its helpers use the engine's unseedable Math.random): choose the Philox stream (seed, chain) the
    exported helpers runif / runif_discrete / rnorm draw from, and the position in it."""
    _HostStream.seed, _HostStream.chain, _HostStream.n = int(seed) & 0xFFFFFFFFFFFFFFFF, int(chain) & 0xFFFFFFFFFFFFFFFF, int(position)
    _HostStream._block, _HostStream._block0 = np.empty(0), 0


def _device_log(x: float) -> float:
    """Math.log as the device computes it (fdlibm e_log, csrc/amwg_math.cuh): the helpers agree with the sampler bit for bit."""
    a, out = np.array([float(x)]), np.empty(1)
    _ffi.check(_ffi.lib().amwg_primitive_eval(0, a.ctypes.data, 1, 0, 0, out.ctypes.data, _default_device()))
    return float(out[0])


def runif(min, max):
    """mcmc.js:31-33"""
    return _HostStream.random() * (max - min) + min


def runif_discrete(min, max):
    """mcmc.js:36-38"""
    return math.floor(_HostStream.random() * (max - min + 1)) + min


def rnorm(mean, sd):
    """mcmc.js:43-54"""
    while True:
        u = _HostStream.random()
        v = 1.7156 * (_HostStream.random() - 0.5)
        x = u - 0.449871
        y = abs(v) + 0.386595
        q = x * x + y * (0.19600 * y - 0.25472 * x)
        if not (q > 0.27597 and (q > 0.27846 or v * v > -4 * _device_log(u) * u * u)):
            break
    return (v / u) * sd + mean


def _default_device() -> int:
    return int(os.environ.get("LOCAL_RANK", "0")) if os.environ.get("AMWG_DEVICE") is None else int(os.environ["AMWG_DEVICE"])


# ------------------------------------------------------------------------------------------------
# option resolution -- AmwgStepper ctor (mcmc.js:837-881) + stepper ctors (:500-505, :644-649)
# ------------------------------------------------------------------------------------------------
_STEPPER_OPTIONS = (("prop_log_scale", 0), ("batch_size", 50), ("max_adaptation", 0.33), ("initial_adaptation", 1.0),
                    ("target_accept_rate", 0.44), ("is_adapting", True))


def resolve_stepper_options(params: Dict[str, dict], options: Optional[dict]) -> Dict[str, Dict[str, list]]:
    """Per parameter, per option: the flat list (one entry per component) the reference's steppers end up with.

    Reproduces the `a || b` merge of mcmc.js:871-878, including its quirks: falsy per-parameter and global values
    (0, false) fall through to the next level, and options.params[name] is mutated in place."""
    out: Dict[str, Dict[str, list]] = {}
    for name, param in params.items():
        if param["type"] not in _TYPE_CODE:
            raise JsThrow("AmwgStepper can't handle parameter " + name + " with type " + str(param["type"]))
        options = options or {}
        po = (options.get("params") or {}).get(name) if _js_truthy(options.get("params")) else None
        param_options = po if _js_truthy(po) else {}
        for key, _ in _STEPPER_OPTIONS:
            mine = param_options.get(key)
            param_options[key] = mine if _js_truthy(mine) else options.get(key)
        resolved: Dict[str, list] = {}
        if param["type"] != "binary":
            for key, default in _STEPPER_OPTIONS:
                if array_equal(param["dim"], [1]):
                    resolved[key] = [get_option(key, param_options, default)]
                else:
                    resolved[key] = _flatten(get_multidim_option(key, param_options, param["dim"], default))
        out[name] = resolved
    return out


# ------------------------------------------------------------------------------------------------
# Sampler / AmwgSampler -- mcmc.js:940-1099
# ------------------------------------------------------------------------------------------------
class Sampler:
    """mcmc.js:940-1073.  `create_stepper_ensamble` is the subclass hook, as in the reference."""

    def __init__(self, params, log_post, data=None, options=None):
        self.data = data
        self.param_names = list(params.keys())
        self.param_init_fun = get_option("param_init_fun", options, param_init_fixed)
        thinning_interval = get_option("thin", options, 1)
        params_to_monitor = get_option("monitor", options, None)
        self.thin(thinning_interval)
        self.monitor(params_to_monitor)
        self.options = options
        self.params = complete_params(params, self.param_init_fun)
        self._user_log_post = log_post
        self._handle = None
        self.steppers = self.create_stepper_ensamble(self.params, None, log_post, self.options)

    def create_stepper_ensamble(self, params, state, log_post, options):
        raise JsThrow("Every Sampler needs to implement create_stepper_ensamble()")

    def thin(self, thinning_interval):
        """mcmc.js:1053-1055"""
        self.thinning_interval = thinning_interval

    def monitor(self, params_to_monitor):
        """mcmc.js:1045-1047"""
        self.monitored_params = params_to_monitor


class AmwgSampler(Sampler):
    """mcmc.js:1090-1099 -- the AMWG sampler, `options["chains"]` chains at once on one B200."""

    # -- construction ---------------------------------------------------------------------------
    def _resolve_options(self, params, options):
        """AmwgStepper's per-parameter option merge (mcmc.js:871-878); the stand-alone steppers read `options` directly."""
        return resolve_stepper_options(params, options)

    def create_stepper_ensamble(self, params, state, log_post, options):
        options = options if options is not None else {}
        self.n_chains = int(get_option("chains", options, 1))
        if self.n_chains < 1:
            raise JsThrow("options.chains must be >= 1")
        seed = get_option("seed", options, None)
        self.seed = int.from_bytes(os.urandom(8), "little") if seed is None else int(seed) & 0xFFFFFFFFFFFFFFFF
        self.device = int(get_option("device", options, _default_device()))
        self.distributed = bool(get_option("distributed", options, False))
        self.gather = get_option("gather", options, "all")                # distributed sample(): "all" | "root" | "none"
        if self.gather not in ("all", "root", "none"):
            raise JsThrow("options.gather must be \"all\", \"root\" or \"none\"")
        self.faithful = bool(get_option("faithful", options, False))      # no factorised plates: bit-faithful sums, slower

        # flat component layout: Object.keys(params) order, row-major inside a parameter
        self._offsets: Dict[str, int] = {}
        n_comp = 0
        for name in self.param_names:
            self._offsets[name] = n_comp
            n_comp += int(np.prod(self.params[name]["dim"]))
        self.n_comp = n_comp

        resolved = self._resolve_options(self.params, options)
        self._program, self._derived_names = trace(self._user_log_post, self.params, self._offsets, n_comp, self.data, self.faithful)

        # shard the chains when running one process per GPU (torch.distributed, see parallel.py)
        self.first_chain, self.local_chains = int(get_option("first_chain", options, 0)), self.n_chains
        if self.distributed:
            from .parallel import shard_chains
            self.first_chain, self.local_chains = shard_chains(self.n_chains)

        self._build_model(resolved)
        return ["AmwgStepper"]

    def _build_model(self, resolved):
        P = len(self.param_names)
        prm = (AmwgParam * P)()
        init = np.empty(self.n_comp)
        opts = (AmwgCompOptions * self.n_comp)()
        for k, name in enumerate(self.param_names):
            p = self.params[name]
            ncomp = int(np.prod(p["dim"]))
            off = self._offsets[name]
            prm[k] = AmwgParam(_TYPE_CODE[p["type"]], ncomp, int(p["dim"][0]), off, float(p["lower"]), float(p["upper"]))
            flat = _flatten(p["init"])
            if len(flat) != ncomp:
                raise JsThrow("The init of parameter " + name + " does not match its dim")
            init[off:off + ncomp] = [float(v) for v in flat]
            for c in range(ncomp):
                o = opts[off + c]
                if p["type"] == "binary":
                    o.prop_log_scale, o.batch_size, o.max_adaptation = 0.0, 50.0, 0.33
                    o.initial_adaptation, o.target_accept_rate, o.is_adapting = 1.0, 0.44, 0
                else:
                    r = resolved[name]
                    o.prop_log_scale = float(r["prop_log_scale"][c]); o.batch_size = float(r["batch_size"][c])
                    o.max_adaptation = float(r["max_adaptation"][c]); o.initial_adaptation = float(r["initial_adaptation"][c])
                    o.target_accept_rate = float(r["target_accept_rate"][c]); o.is_adapting = 1 if r["is_adapting"][c] else 0
        prog = self._program
        code = np.asarray(prog.code, dtype=np.int32)
        consts = np.asarray(prog.consts if prog.consts else [0.0], dtype=np.float64)
        cols = (AmwgColumn * max(len(prog.columns), 1))()
        self._col_keepalive = [np.ascontiguousarray(c, dtype=np.float64) for c in prog.columns]
        for k, c in enumerate(self._col_keepalive):
            cols[k] = AmwgColumn(c.ctypes.data_as(C.POINTER(C.c_double)), c.size)
        plates = (AmwgPlate * max(len(prog.plates), 1))()
        for k, pl in enumerate(prog.plates):
            q = AmwgPlate()
            q.kind, q.n = pl["kind"], pl["n"]
            for j in range(4):
                q.col[j] = pl["col"][j]; q.iparam[j] = pl["iparam"][j]
            plates[k] = q
        m = AmwgModel()
        m.abi_version = _ffi.ABI_VERSION
        m.n_params, m.params = P, prm
        m.n_comp, m.init = self.n_comp, init.ctypes.data_as(C.POINTER(C.c_double))
        m.comp_options = opts
        m.n_code, m.code = code.size, code.ctypes.data_as(C.POINTER(C.c_int32))
        m.logpost_prog, m.derived_prog, m.n_derived = prog.logpost_prog, prog.derived_prog, len(self._derived_names)
        m.n_consts, m.consts = consts.size, consts.ctypes.data_as(C.POINTER(C.c_double))
        m.n_columns, m.columns = len(prog.columns), cols
        m.n_plates, m.plates = len(prog.plates), plates
        fold_prog = np.asarray(prog.fold_prog if prog.fold_prog else [0], dtype=np.int32)
        fold_dst = np.asarray(prog.fold_dst if prog.fold_dst else [0], dtype=np.int32)
        m.n_fold = len(prog.fold_prog)
        m.fold_prog = fold_prog.ctypes.data_as(C.POINTER(C.c_int32))
        m.fold_dst = fold_dst.ctypes.data_as(C.POINTER(C.c_int32))
        comp_prog = np.asarray(prog.comp_prog if prog.n_terms else [0], dtype=np.int32)
        touch_off = np.asarray(prog.touch_off if prog.n_terms else [0], dtype=np.int32)
        touch_terms = np.asarray(prog.touch_terms if prog.touch_terms else [0], dtype=np.int32)
        m.n_terms = prog.n_terms
        m.comp_prog = comp_prog.ctypes.data_as(C.POINTER(C.c_int32)) if prog.n_terms else None
        m.touch_off = touch_off.ctypes.data_as(C.POINTER(C.c_int32)) if prog.n_terms else None
        m.touch_terms = touch_terms.ctypes.data_as(C.POINTER(C.c_int32)) if prog.n_terms else None
        block_params = np.asarray(prog.block_params if prog.block_params else [0], dtype=np.int32)
        tbc = np.asarray(prog.term_block_comp if prog.term_block_comp else [0], dtype=np.int32)
        m.n_block_params = len(prog.block_params)
        m.block_params = block_params.ctypes.data_as(C.POINTER(C.c_int32)) if prog.block_params else None
        m.term_block_comp = tbc.ctypes.data_as(C.POINTER(C.c_int32)) if prog.block_params else None
        m.stat_prog = prog.stat_prog
        m.n_sum_terms = prog.n_sum_terms if prog.stat_prog >= 0 else prog.n_terms
        self._cache_keepalive = (comp_prog, touch_off, touch_terms, block_params, tbc)
        vcomps = np.asarray(prog.variant_comps if prog.variant_comps else [0], dtype=np.int32)
        vlp = np.asarray(prog.variant_logpost if prog.variant_logpost else [0], dtype=np.int32)
        vder = np.asarray(prog.variant_derived if prog.variant_derived else [-1], dtype=np.int32)
        m.n_variant_comps = len(prog.variant_comps)
        m.variant_comps = vcomps.ctypes.data_as(C.POINTER(C.c_int32))
        m.variant_logpost = vlp.ctypes.data_as(C.POINTER(C.c_int32))
        m.variant_derived = vder.ctypes.data_as(C.POINTER(C.c_int32))
        self._model_keepalive = (prm, init, opts, code, consts, cols, plates, fold_prog, fold_dst, vcomps, vlp, vder, m)
        L = _ffi.lib()
        if get_option("_model_only", self.options, False):       # tests: lower the model, do not touch a device
            self._model = m
            return
        h = C.c_void_p()
        rc = L.amwg_create(C.byref(m), self.local_chains, self.first_chain, self.seed, self.device, C.byref(h))
        if rc != 0:
            raise JsThrow(L.amwg_last_error().decode())
        self._handle = h

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def close(self):
        if getattr(self, "_handle", None):
            _ffi.lib().amwg_destroy(self._handle)
            self._handle = None

    # -- layout helpers -------------------------------------------------------------------------
    def _state_keys(self) -> List[str]:
        """Object.keys(state): the parameters, then the derived quantities in creation order (mcmc.js:1010)."""
        return self.param_names + self._derived_names

    def _entries(self, name: str) -> List[int]:
        if name in self._offsets:
            n = int(np.prod(self.params[name]["dim"]))
            return list(range(self._offsets[name], self._offsets[name] + n))
        if name in self._derived_names:
            return [self.n_comp + self._derived_names.index(name)]
        return []          # JS: state[name] is undefined -> the column is filled with undefined

    def _shape_out(self, name: str, arr: np.ndarray) -> np.ndarray:
        """arr: [rows, entries, chains] -> reference-shaped array ([rows, *dim] for one chain, else [rows, chains, *dim])."""
        rows, _, chains = arr.shape
        dim = self.params[name]["dim"] if name in self.params else [1]
        a = np.moveaxis(arr, 1, 2)                        # [rows, chains, entries]
        a = a.reshape(rows, chains) if list(dim) == [1] else a.reshape(rows, chains, *dim)
        return a[:, 0] if self.n_chains == 1 else a

    # -- the reference's methods -----------------------------------------------------------------
    def step(self):
        """mcmc.js:985-997 -- one sweep; returns the live state."""
        self.burn(1)
        return self.state

    @property
    def state(self) -> Dict[str, Any]:
        L = _ffi.lib()
        n_entries = self.n_comp + len(self._derived_names)
        buf = np.empty((n_entries, self.local_chains))
        _ffi.check(L.amwg_get_state(self._handle, buf.ctypes.data))
        out = {}
        for name in self._state_keys():
            e = self._entries(name)
            out[name] = self._shape_out(name, buf[e][None, :, :])[0]
        return out

    def log_post(self):
        """mcmc.js:958-960 -- `sampler.log_post()`: log_post at the current state (one number, or one per chain)."""
        buf = np.empty(self.local_chains)
        _ffi.check(_ffi.lib().amwg_get_log_post(self._handle, buf.ctypes.data))
        return float(buf[0]) if self.n_chains == 1 else buf

    def burn(self, n_iterations):
        """mcmc.js:1035-1039"""
        L = _ffi.lib()
        rc = L.amwg_burn(self._handle, int(n_iterations))
        if rc != 0:
            raise JsThrow(L.amwg_last_error().decode())

    def sample(self, n_iterations):
        """mcmc.js:1005-1030 -- {name: draws}; rows = ceil(n/thin); row r is the state before sweep r*thin."""
        monitored = self._state_keys() if self.monitored_params is None else list(self.monitored_params)
        entries: List[int] = []
        spans = {}
        for name in monitored:
            e = self._entries(name)
            spans[name] = (len(entries), len(e))
            entries.extend(e)
        n = int(n_iterations)
        thin = abs(int(self.thinning_interval))                 # `i % thin === 0` (mcmc.js:1021): the sign of thin does not matter ...
        if thin == 0:                                           # ... and i % 0 is NaN: nothing is ever recorded, the chains still step
            self.burn(max(n, 0))
            return {name: np.empty((0,)) for name in monitored}
        rows = 0 if n <= 0 else (n + thin - 1) // thin
        raw = self._sample_raw(n, thin, entries, rows)          # [rows, n_entries, chains]
        out = {}
        for name in monitored:
            s, ln = spans[name]
            if ln == 0:
                out[name] = np.full((rows,), np.nan)
            else:
                out[name] = self._shape_out(name, raw[:, s:s + ln, :])
        return out

    def _sample_raw(self, n: int, thin: int, entries: List[int], rows: int) -> np.ndarray:
        L = _ffi.lib()
        mon = np.asarray(entries, dtype=np.int32)
        if self.distributed:
            from .parallel import sample_and_gather
            return sample_and_gather(self, n, thin, mon, rows)
        buf = _pinned_empty((rows, len(entries), self.local_chains))
        rc = L.amwg_sample(self._handle, n, thin, mon.ctypes.data_as(C.POINTER(C.c_int32)), len(entries), buf.ctypes.data)
        if rc != 0:
            raise JsThrow(L.amwg_last_error().decode())
        return buf

    def sample_summary(self, n_iterations, probs=(0.025, 0.25, 0.5, 0.75, 0.975), ess=False, rank=False):
        """Not in the reference (SURVEY 8(f).3): the same sweeps and the same kept rows as `sample(n)` (thin / monitor apply), but the
        draws stay in HBM and only their summary comes back: {name: {"mean", "sd", "rhat", "quantiles", "n_draws"}}, pooled over
        all chains and kept rows; multi-dim parameters give arrays of their `dim` ("quantiles": [len(probs), *dim], exact order
        statistics with numpy.quantile's linear rule; a long grid such as numpy.linspace(0, 1, 41) gives an equal-mass histogram and
        runs as several radix selects of 16 probabilities each). With options.distributed every rank returns the all-GPU summary
        (two small collectives, summary.py). Advances the chains exactly as sample(n) does.

        ess=True adds, per name and shaped like "mean": "ess", the bulk effective sample size of the mean on split chains without
        rank normalisation (posterior::ess_mean, ArviZ ess(method="mean")); "ess_tail", the smaller ESS of the indicators x <= q05
        and x <= q95 at the exact pooled 5 % / 95 % quantiles (posterior::ess_tail); "mcse", sd / sqrt(ess). NaN with fewer than 8
        kept rows, for a constant entry or indicator, or when a draw is not finite. The autocovariances are reduced on the device
        in tiles of lags, read only for the entries whose Geyer sequence is still positive (summary.summarise_ess). With
        options.distributed every rank returns the same bits; they equal a single GPU's ESS to rounding, not bit for bit, because
        the sums are grouped differently. The other fields are the same bits as with ess=False.

        rank=True (independent of ess) adds, per name and shaped like "mean", the rank-normalised diagnostics of Vehtari et al. (2021):
        "rhat_bulk", the split R-hat of the rank-normalised split draws (ArviZ rhat(method="z_scale")); "rhat_folded", that of the
        draws folded about their median; "rhat_rank", the larger of the two (posterior::rhat, ArviZ rhat(method="rank")); and
        "ess_bulk", the Geyer ESS of the rank-normalised draws (posterior::ess_bulk). The exact pooled ranks come from a radix sort
        on the device, entry by entry (summary.summarise_rank); with options.distributed the draws' runs are exchanged so that every
        rank ranks over all chains, and every rank returns the same bits. NaN as for ess=True and when an entry is constant. The
        other fields are the same bits as with rank=False."""
        import torch
        from .summary import CudaBlockReducer, RankWorkingSetError, summarise_block, summarise_ess, summarise_rank
        monitored = self._state_keys() if self.monitored_params is None else list(self.monitored_params)
        entries: List[int] = []
        spans = {}
        for name in monitored:
            e = self._entries(name)
            spans[name] = (len(entries), len(e))
            entries.extend(e)
        n = int(n_iterations)
        thin = abs(int(self.thinning_interval))
        rows = 0 if (n <= 0 or thin == 0) else (n + thin - 1) // thin
        if rows == 0 or not entries:
            raise JsThrow("sample_summary needs at least one kept iteration and one monitored entry")
        L = _ffi.lib()
        dev = torch.device("cuda", self.device)
        need = rows * len(entries) * self.local_chains * 8
        free, _total = torch.cuda.mem_get_info(dev)
        if need + 2 * len(entries) * self.local_chains * 8 > 0.9 * free:
            raise JsThrow("sample_summary: the sample block (%.1f GB) does not fit in device memory; raise thin() or lower n" % (need / 1e9))
        h = rows // 2
        if rank and h >= 4:
            split = 2 * h * self.local_chains
            if split >= 1 << 32:
                raise JsThrow("sample_summary(rank=True): %d split draws of one entry on one GPU; the rank sort takes fewer than 2^32 "
                              "(raise thin() or lower n)" % split)
            # the z block, and per entry being sorted: keys and payloads double-buffered (24 B) and the sort's tile counts (1/4 B).
            # Across GPUs the runs keep their keys (8 B) and each GPU merges the runs it receives (summary.RECV_BYTES_PER_RUN per
            # run), counted here for as many runs as it sorted itself; the exchange checks the actual count again.
            from .summary import RECV_BYTES_PER_RUN
            per_draw = 24.25 + ((8 + RECV_BYTES_PER_RUN + 8) if self.distributed else 0)
            need_rank = split * len(entries) * 8 + int(split * per_draw)
            if need + need_rank + 2 * len(entries) * self.local_chains * 8 > 0.9 * free:
                raise JsThrow("sample_summary(rank=True): the sample block (%.1f GB) and the rank working set (%.1f GB) do not fit in "
                              "device memory; raise thin() or lower n" % (need / 1e9, need_rank / 1e9))
        timing = os.environ.get("AMWG_SUMMARY_TIMING") == "1"
        t0 = time.perf_counter()
        block = torch.empty((rows, len(entries), self.local_chains), dtype=torch.float64, device=dev)
        mon = np.asarray(entries, dtype=np.int32)
        torch.cuda.current_stream(dev).synchronize()
        t1 = time.perf_counter()
        rc = L.amwg_sample_device(self._handle, n, thin, mon.ctypes.data_as(C.POINTER(C.c_int32)), len(entries), block.data_ptr())
        if rc != 0:
            raise JsThrow(L.amwg_last_error().decode())
        t2 = time.perf_counter()
        reducer = CudaBlockReducer(self.device)
        M = rows * self.n_chains
        middle = [M // 2 - 1, M // 2] if M % 2 == 0 else [M // 2]        # numpy.median's order statistics, for the fold
        if ess:                                                 # the tail ESS thresholds ride along in the same radix selects
            probs = [float(p) for p in probs]
            select = probs + [p for p in (0.05, 0.95) if p not in probs]
            res = summarise_block(reducer, block, rows, self.n_chains, select, self.distributed, middle if rank else ())
            mean, sd, rhat, q = res[:4]
            t3 = time.perf_counter()
            ess_v, tail_v, tiles = summarise_ess(reducer, block, rows, self.n_chains, q[select.index(0.05)], q[select.index(0.95)],
                                                 self.distributed)
            finite = np.isfinite(mean)                          # also covers the middle row of an odd `rows`, which no half-chain holds
            ess_v, tail_v = np.where(finite, ess_v, np.nan), np.where(finite, tail_v, np.nan)
            with np.errstate(invalid="ignore", divide="ignore"):
                mcse = sd / np.sqrt(ess_v)
            q = q[:len(probs)]
        else:
            res = summarise_block(reducer, block, rows, self.n_chains, probs, self.distributed, middle if rank else ())
            mean, sd, rhat, q = res[:4]
        if rank:
            t5 = time.perf_counter()
            ost = res[4]
            med = ost[0] if len(middle) == 1 else (ost[0] + ost[1]) / 2
            rank_stats = {}
            try:
                r_bulk, r_fold, r_rank, ess_bulk = summarise_rank(reducer, block, rows, self.n_chains, med, self.distributed, rank_stats)
            except RankWorkingSetError as e:
                raise JsThrow(str(e)) from None
            finite = np.isfinite(mean)
            r_bulk, r_fold, r_rank, ess_bulk = (np.where(finite, a, np.nan) for a in (r_bulk, r_fold, r_rank, ess_bulk))
            t6 = time.perf_counter()
        del block
        if timing:
            t4 = time.perf_counter()
            print("sample_summary: alloc %.2f ms, sweeps %.2f ms, reductions %.2f ms" %
                  (1e3 * (t1 - t0), 1e3 * (t2 - t1), 1e3 * (t4 - t2)), file=sys.stderr, flush=True)
            if ess:
                print("sample_summary: of which ess %.2f ms, %d lag tiles (mean, q05, q95 indicators; max per entry %d)" %
                      (1e3 * (t5 - t3 if rank else t4 - t3), int(tiles.sum()), int(tiles.max(initial=0))), file=sys.stderr, flush=True)
            if rank:
                print("sample_summary: of which rank %.2f ms, %d sort passes run, %d skipped" %
                      (1e3 * (t6 - t5), rank_stats.get("passes", 0), rank_stats.get("skipped", 0)), file=sys.stderr, flush=True)
        out = {}
        for name in monitored:
            s0, ln = spans[name]
            if ln == 0:
                continue
            dim = list(self.params[name]["dim"]) if name in self.params else [1]
            shape = (lambda a: float(a[0])) if dim == [1] else (lambda a, dim=dim: np.asarray(a).reshape(*dim))
            out[name] = {"mean": shape(mean[s0:s0 + ln]), "sd": shape(sd[s0:s0 + ln]), "rhat": shape(rhat[s0:s0 + ln]),
                         "quantiles": q[:, s0] if dim == [1] else q[:, s0:s0 + ln].reshape(len(q), *dim),
                         "n_draws": rows * self.n_chains}
            if ess:
                out[name].update(ess=shape(ess_v[s0:s0 + ln]), ess_tail=shape(tail_v[s0:s0 + ln]), mcse=shape(mcse[s0:s0 + ln]))
            if rank:
                out[name].update(rhat_bulk=shape(r_bulk[s0:s0 + ln]), rhat_folded=shape(r_fold[s0:s0 + ln]),
                                 rhat_rank=shape(r_rank[s0:s0 + ln]), ess_bulk=shape(ess_bulk[s0:s0 + ln]))
        return out

    def start_adaptation(self):
        """mcmc.js:1060-1064"""
        _ffi.check(_ffi.lib().amwg_set_adapting(self._handle, 1))

    def stop_adaptation(self):
        """mcmc.js:1069-1073"""
        _ffi.check(_ffi.lib().amwg_set_adapting(self._handle, 0))

    def info(self):
        """mcmc.js:977-980 + AmwgStepper.info (:906-912) + OnedimMetropolisStepper.info (:563-571).
        (The reference returns the thin/monitor *methods* under those keys -- a bug; the values are returned here.)"""
        L = _ffi.lib()
        scal = np.empty(self.n_comp * 3)
        pls = np.empty((self.n_comp, self.local_chains))
        acc = np.empty((self.n_comp, self.local_chains), dtype=np.int32)
        _ffi.check(L.amwg_info(self._handle, scal.ctypes.data, pls.ctypes.data, acc.ctypes.data))
        per_param = {}
        for name in self.param_names:
            p = self.params[name]
            if p["type"] == "binary":
                per_param[name] = {}                       # BinaryStepper inherits Stepper.info -> {} (mcmc.js:465-468)
                continue
            e = self._entries(name)
            dim = list(p["dim"])

            def per_chain(a, dim=dim):                     # a: [entries, chains]
                a = a[0] if dim == [1] else a.reshape(*dim, a.shape[-1])
                return a[..., 0] if self.n_chains == 1 else a

            def invariant(vals, dim=dim):
                return vals[0] if dim == [1] else np.asarray(vals).reshape(*dim)

            per_param[name] = {
                "prop_log_scale": per_chain(pls[e]),
                "is_adapting": invariant([bool(scal[c * 3]) for c in e]),
                "acceptance_count": per_chain(acc[e]),
                "iterations_since_adaption": invariant([scal[c * 3 + 1] for c in e]),
                "batch_count": invariant([scal[c * 3 + 2] for c in e]),
            }
        return {"state": self.state, "thin": self.thinning_interval, "monitor": self.monitored_params,
                "steppers": [per_param]}

    # -- instrumentation (not in the reference) -------------------------------------------------------
    def kernel_launches(self) -> int:
        return int(_ffi.lib().amwg_kernel_launches(self._handle))

    def last_sweep_kernel_ms(self) -> float:
        return float(_ffi.lib().amwg_last_sweep_kernel_ms(self._handle))

    def program_summary(self) -> List[str]:
        return list(self._program.summary)

    def jit_status(self):
        """(active, note): does this handle step with a kernel specialised for its model at run time (csrc/amwg_jit.cuh)?"""
        if not getattr(self, "_handle", None):
            return False, "no device handle"
        buf = C.create_string_buffer(4096)
        on = _ffi.lib().amwg_jit_status(self._handle, buf, len(buf))
        return bool(on), buf.value.decode("utf-8", "replace")

    def jit_compile_check(self, n_chains=None):
        """Generate and compile the specialised sweep of this model without running it (works without a GPU).
        -> (rc, message, source): rc 0 compiled, 1 model not eligible, -1 error."""
        log = C.create_string_buffer(1 << 16)
        src = C.create_string_buffer(1 << 20)
        m = self._model_keepalive[-1]
        rc = _ffi.lib().amwg_jit_compile_check(C.byref(m), int(n_chains or self.n_chains), log, len(log), src, len(src))
        return rc, log.value.decode("utf-8", "replace"), src.value.decode("utf-8", "replace")


class _PinnedPool:
    """Page-locked host buffers for sample(): pinning GBs costs more than the copy itself, so buffers are recycled once
    every array handed to the user (all views of the buffer) has been garbage collected."""

    def __init__(self):
        self._free: Dict[tuple, list] = {}

    def get(self, shape) -> np.ndarray:
        shape = tuple(int(v) for v in shape)
        try:
            import torch
            if not torch.cuda.is_available():
                raise RuntimeError
        except Exception:
            return np.empty(shape, dtype=np.float64)
        import weakref
        lst = self._free.get(shape)
        t = lst.pop() if lst else torch.empty(shape, dtype=torch.float64, pin_memory=True)
        a = t.numpy()
        weakref.finalize(a, self._put, shape, t)
        return a

    def _put(self, shape, t):
        lst = self._free.setdefault(shape, [])
        if len(lst) < 2:
            lst.append(t)


_PINNED = _PinnedPool()


def _pinned_empty(shape) -> np.ndarray:
    return _PINNED.get(shape)


# ------------------------------------------------------------------------------------------------
# stand-alone steppers -- mcmc.js:433-912 (the export list of mcmc.js:1103-1117)
# ------------------------------------------------------------------------------------------------
def _resolve_direct(params: Dict[str, dict], options: Optional[dict]) -> Dict[str, Dict[str, list]]:
    """Option handling of the stepper constructors themselves: get_option / get_multidim_option on `options`
    (mcmc.js:500-505, 644-649) -- no AmwgStepper merge."""
    out: Dict[str, Dict[str, list]] = {}
    for name, param in params.items():
        r: Dict[str, list] = {}
        if param["type"] != "binary":
            for key, default in _STEPPER_OPTIONS:
                if array_equal(param["dim"], [1]):
                    r[key] = [get_option(key, options, default)]
                else:
                    r[key] = _flatten(get_multidim_option(key, options, param["dim"], default))
        out[name] = r
    return out


def _set_nested(dst, src):
    """copy a nested array into an existing nested list IN PLACE (the reference's steppers mutate state[name][i]...)"""
    for i, v in enumerate(src):
        if isinstance(v, (list, np.ndarray)) and isinstance(dst[i], list):
            _set_nested(dst[i], v)
        else:
            dst[i] = float(v)


class _SteppedModel(AmwgSampler):
    """The device machinery of AmwgSampler behind a zero-argument `log_post` that closes over the caller's `state` object:
    the closure is recorded by temporarily putting symbolic values into `state`."""

    def __init__(self, params, state, log_post, options, direct_options: bool):
        self._user_state, self._zero_arg_log_post, self._direct = state, log_post, direct_options
        names = list(params.keys())

        def foreign(v, key):
            """numeric entries of `state` that belong to OTHER steppers: marked, so that a log_post that reads them is noticed"""
            if is_number(v):
                return Sym("FOREIGN", (), key)
            if isinstance(v, list):
                return [foreign(x, key) for x in v]
            return v

        def recorded(sym_state, _data):
            others = [k for k in list(state.keys()) if k not in names]
            saved = {n: state[n] for n in names + others}
            try:
                for n in names:
                    state[n] = sym_state[n]
                for k in others:
                    state[k] = foreign(saved[k], k)
                result = log_post()
            finally:
                for n in saved:
                    state[n] = saved[n]
            # The reference's steppers close over the LIVE state object (mcmc.js:433-437): a second stepper's updates are seen by
            # this one's log_post. Here log_post is recorded once, so a value owned by another stepper would be frozen into the
            # device program -- refuse instead of silently sampling the wrong conditional.
            stack, seen = [result] if isinstance(result, Sym) else [], 0
            while stack:
                node = stack.pop()
                if node.op == "FOREIGN":
                    raise JsThrow("log_post reads state." + str(node.val) + ", which this stepper does not step: composing several "
                                  "stand-alone steppers over one state object is not supported on the device; give one "
                                  "AmwgStepper / AmwgSampler all the parameters")
                stack.extend(node.args)
                seen += 1
            return result
        p = copy.deepcopy(params)
        for n in names:
            p[n]["init"] = copy.deepcopy(state[n])          # a stepper starts from the state it is given, not from params.init
        sampler_options = {k: v for k, v in (options or {}).items()}
        Sampler.__init__(self, p, recorded, None, sampler_options)

    def _resolve_options(self, params, options):
        stepper_options = {k: v for k, v in (options or {}).items() if k not in ("chains", "seed", "device", "first_chain", "faithful")}
        return _resolve_direct(params, stepper_options) if self._direct else resolve_stepper_options(params, stepper_options)

    def advance(self):
        """one step; writes the new values into the caller's state object (in place for arrays) and returns them by name"""
        self.burn(1)
        new = self.state
        for n in self.param_names:
            v = new[n]
            if isinstance(self._user_state[n], list):
                _set_nested(self._user_state[n], np.asarray(v).tolist())
            else:
                self._user_state[n] = v.tolist() if isinstance(v, np.ndarray) else float(v)
        return new


class Stepper:
    """mcmc.js:433-468 -- the Stepper "interface"."""

    def __init__(self, params, state, log_post):
        self.params, self.state, self.log_post = params, state, log_post

    def step(self):
        raise JsThrow("Every Stepper need to implement step()")

    def start_adaptation(self):
        pass

    def stop_adaptation(self):
        pass

    def info(self):
        return {}


class _DeviceStepper(Stepper):
    _type: Optional[str] = None        # proposal kind forced by the class (the reference's Real/Int steppers ignore params.type)
    _onedim = True
    _who = "Stepper"

    def __init__(self, params, state, log_post, options=None):
        super().__init__(params, state, log_post)
        names = list(params.keys())
        self._check(names, params)
        self.param_name = names[0] if len(names) == 1 else None
        p = complete_params(copy.deepcopy(params))
        if self._type is not None:
            for n in names:
                p[n]["type"] = self._type
                if self._type == "binary":
                    p[n]["lower"], p[n]["upper"] = 0, 1
        self._model = _SteppedModel(p, state, log_post, options, direct_options=self._who != "AmwgStepper")

    def _check(self, names, params):
        pass

    def step(self):
        new = self._model.advance()
        return self.state[self.param_name] if self.param_name is not None else self.state

    def start_adaptation(self):
        self._model.start_adaptation()

    def stop_adaptation(self):
        self._model.stop_adaptation()

    def _info_of(self, name):
        per = self._model.info()["steppers"][0][name]
        if not per:
            return {}
        dim = list(self._model.params[name]["dim"])
        if dim == [1]:
            return per
        keys = list(per.keys())                          # nested arrays of info objects (mcmc.js:698-702)
        flat = {k: np.asarray(per[k]).reshape(-1) for k in keys}
        objs = [{k: flat[k][c].item() for k in keys} for c in range(int(np.prod(dim)))]

        def nest(lst, d):
            if len(d) == 1:
                return lst
            step = len(lst) // d[0]
            return [nest(lst[i * step:(i + 1) * step], d[1:]) for i in range(d[0])]
        return nest(objs, dim)

    def info(self):
        return self._info_of(self.param_name)


class OnedimMetropolisStepper(_DeviceStepper):
    """mcmc.js:485-571"""
    _who = "OnedimMetropolisStepper"

    def _check(self, names, params):
        if len(names) != 1:
            raise JsThrow("OnedimMetropolisStepper can only handle one parameter.")
        dim = params[names[0]].get("dim", [1])
        if not array_equal([dim] if is_number(dim) else list(dim), [1]):
            raise JsThrow("OnedimMetropolisStepper can only handle one one-dimensional parameter.")


class RealMetropolisStepper(OnedimMetropolisStepper):
    """mcmc.js:586-591"""
    _type = "real"


class IntMetropolisStepper(OnedimMetropolisStepper):
    """mcmc.js:605-610"""
    _type = "int"


class MultidimComponentMetropolisStepper(_DeviceStepper):
    """mcmc.js:631-702"""
    _who = "MultidimComponentMetropolisStepper"

    def _check(self, names, params):
        if len(names) != 1:
            raise JsThrow("MultidimComponentMetropolisStepper can't handle more than one parameter.")


class MultiRealComponentMetropolisStepper(MultidimComponentMetropolisStepper):
    """mcmc.js:709-714"""
    _type = "real"


class MultiIntComponentMetropolisStepper(MultidimComponentMetropolisStepper):
    """mcmc.js:721-726"""
    _type = "int"


class BinaryStepper(_DeviceStepper):
    """mcmc.js:740-767"""
    _type = "binary"
    _who = "BinaryStepper"

    def _check(self, names, params):
        if len(names) != 1:
            raise JsThrow("BinaryStepper can't handle more than one parameter.")


class BinaryComponentStepper(_DeviceStepper):
    """mcmc.js:781-820"""
    _type = "binary"
    _who = "BinaryComponentStepper"

    def _check(self, names, params):
        if len(names) != 1:
            raise JsThrow("BinaryComponentStepper can't handle more than one parameter.")


class AmwgStepper(_DeviceStepper):
    """mcmc.js:837-912 -- any number of parameters; per-parameter option merge as in AmwgSampler."""
    _who = "AmwgStepper"

    def info(self):
        return {n: self._info_of(n) for n in self._model.param_names}
