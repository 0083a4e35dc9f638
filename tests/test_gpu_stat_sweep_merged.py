"""The statistics sweep's step phase in its merged form (AMWG_JIT_MERGE_STEPS: the heavy calls of all component classes taken once
per warp) and with the screened accept test (AMWG_JIT_ACCEPT_SCREEN: js_exp skipped where the decision is certain) changes no
arithmetic: with both switches off and on, the same model, seed and sweeps give the same draws, state, acceptance counts and
proposal scales bit for bit, across adaptation batch boundaries."""
import numpy as np
import pytest

import models
from conftest import config2_data

pytestmark = pytest.mark.gpu

SWITCHES = ("AMWG_JIT_MERGE_STEPS", "AMWG_JIT_ACCEPT_SCREEN")


def _run(pkg, monkeypatch, on, params, log_post, data, chains, seed=7, burn=120, sample=30):
    monkeypatch.setenv("AMWG_JIT", "1")
    for k in SWITCHES:
        monkeypatch.setenv(k, "1" if on else "0")
    s = pkg.mcmc.AmwgSampler(params, log_post, data, {"chains": chains, "seed": seed})
    active, note = s.jit_status()
    assert active, note
    src = s.jit_compile_check()[2]
    assert ("jit_accept_screen(dl, coin)" in src) == on
    s.burn(burn)                                    # batches of 50 sweeps: crosses two adaptation boundaries
    draws = s.sample(sample)
    info = s.info()["steppers"][0]
    later = s.sample(3)                             # continues from each chain's stream position
    out = {"draws": draws, "later": later, "state": s.state, "info": info}
    for k in SWITCHES:
        monkeypatch.delenv(k)
    return out


def _bits(a):
    a = np.ascontiguousarray(np.asarray(a, dtype=np.float64))
    return a.view(np.uint64)


def _assert_identical(off, on):
    for part in ("draws", "later", "state"):
        assert off[part].keys() == on[part].keys()
        for name in off[part]:
            assert np.array_equal(_bits(off[part][name]), _bits(on[part][name])), (part, name)
    for name, st in off["info"].items():
        for key in ("prop_log_scale", "acceptance_count", "batch_count", "iterations_since_adaption"):
            assert np.array_equal(_bits(st[key]), _bits(on["info"][name][key])), (name, key)


def _compare(pkg, monkeypatch, params, log_post, data, chains, **kw):
    off = _run(pkg, monkeypatch, False, params, log_post, data, chains, **kw)
    on = _run(pkg, monkeypatch, True, params, log_post, data, chains, **kw)
    _assert_identical(off, on)
    return on


@pytest.mark.parametrize("chains", [1 << 14, 4099])
def test_headline_model(gpu_pkg, monkeypatch, chains):
    """BASELINE config 2's model and data: two component classes whose steps the lanes of a warp take at the same time"""
    pkg = gpu_pkg
    on = _compare(pkg, monkeypatch, models.PARAMS_NORM, models.norm_post_readme(pkg.ld), config2_data().tolist(), chains)
    mu = np.asarray(on["draws"]["mu"])
    moved = np.mean(mu[1:] != mu[:-1])
    assert 0.05 < moved < 0.95, moved                # both outcomes of the accept test were taken


@pytest.mark.parametrize("J,per", [(8, 256), (16, 1024)])
def test_hierarchical_model_resident_and_streamed(gpu_pkg, monkeypatch, J, per):
    """config 4's shape: a block of group means and a shared sd whose plate terms are a loop; 16 x 1024 points stream"""
    pkg = gpu_pkg
    rng = np.random.default_rng(J * per)
    g = np.repeat(np.arange(J), per)
    y = rng.normal(100, 20, J)[g] + rng.normal(0, 5, J * per)
    params = {"mu": {"type": "real", "dim": [J], "init": 100.0}, "sigma": {"type": "real", "lower": 0, "init": 5.0}}
    _compare(pkg, monkeypatch, params, models.hier_norm_post(pkg.ld), {"y": y, "g": g.astype(float)}, 4096)


def test_bounded_and_int_parameters(gpu_pkg, monkeypatch):
    """proposals of bounded reals and ints fall out of bounds (no accept uniform, no step) and ints are rounded; the two side
    parameters form one class of two members next to mu's and sigma's classes"""
    pkg = gpu_pkg
    ld = pkg.ld
    y = np.random.default_rng(31).normal(5, 2, 300)
    params = {"sigma": {"type": "real", "lower": 0, "init": 2.0}, "mu": {"type": "real", "init": 5.0},
              "n": {"type": "int", "lower": -3, "upper": 4, "init": 0}, "b": {"type": "real", "lower": -1.5, "upper": 2.5, "init": 0}}

    def log_post(state, d):
        lp = ld.gamma(state.sigma, 2, 0.5)
        lp += ld.norm(state.mu, 5, 10)
        lp += ld.norm(state.n, 0.5, 1.2)
        lp += ld.norm(state.b, -0.3, 1.2)
        for i in range(len(d)):
            lp += ld.norm(d[i], state.mu, state.sigma)
        return lp
    on = _compare(pkg, monkeypatch, params, log_post, y.tolist(), 4096 + 64 + 5)
    n = np.asarray(on["draws"]["n"])
    assert np.all(n == np.round(n)) and n.min() >= -3 and n.max() <= 4 and np.unique(n).size > 3
