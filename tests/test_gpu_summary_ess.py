"""Effective sample size in `sample_summary(ess=True)` on the device: amwg_summary_autocov against the numpy direct sums, and
the whole path against the host reference on the raw draws of an identically seeded sampler."""
import numpy as np
import pytest

import models
from conftest import NORM_DATA, config2_data
from summary_ess_ref import NumpyEssReducer

pytestmark = pytest.mark.gpu


def _host_ess(raw, name, rows, n_chains):
    """host reference on the draws sample() returns: summarise_ess over the numpy stand-in, q05 / q95 from numpy.quantile"""
    import torch
    from bayes_js_b200.summary import summarise_ess
    x = raw[name]                                            # [rows, chains, *dim]
    flat = np.moveaxis(x.reshape(x.shape[0], x.shape[1], -1), 2, 1)      # [rows, entries, chains]
    q05, q95 = np.quantile(np.moveaxis(flat, 1, 0).reshape(flat.shape[1], -1), [0.05, 0.95], axis=1)
    ess, tail, _ = summarise_ess(NumpyEssReducer(), torch.from_numpy(np.ascontiguousarray(flat)), rows, n_chains, q05, q95, False)
    sd = np.moveaxis(flat, 1, 0).reshape(flat.shape[1], -1).std(axis=1, ddof=1)
    return ess, tail, sd / np.sqrt(ess)


def _check(summary, raw, name, rows, n_chains, rtol=1e-9):
    ess, tail, mcse = _host_ess(raw, name, rows, n_chains)
    dim = raw[name].shape[2:]
    shape = (lambda a: a.reshape(dim)) if dim else (lambda a: a[0])
    got = summary[name]
    assert np.allclose(got["ess"], shape(ess), rtol=rtol, atol=0, equal_nan=True), (name, got["ess"], ess)
    assert np.allclose(got["ess_tail"], shape(tail), rtol=rtol, atol=0, equal_nan=True), (name, got["ess_tail"], tail)
    assert np.allclose(got["mcse"], shape(mcse), rtol=rtol, atol=0, equal_nan=True), name


def test_c_abi_autocov_on_an_adversarial_block(gpu_pkg):
    """ragged chain counts, odd rows, lag0 > 0, tiles reaching past h (empty sums are exactly 0), indicator mode, a constant
    column; two calls give the same bits"""
    import torch
    from bayes_js_b200.summary import CudaBlockReducer
    red, ref = CudaBlockReducer(0), NumpyEssReducer()
    dev = torch.device("cuda", 0)
    for rows, chains in [(37, 1000), (24, 4097)]:
        rng = np.random.default_rng(rows)
        x = rng.normal(0, 1, (rows, 4, chains)).cumsum(axis=0) * 0.3
        x[:, 1] = np.round(3 * x[:, 1])
        x[:, 2] = 184.5 + 0.01 * x[:, 2]
        x[:, 3] = 7.25
        block = torch.from_numpy(x).to(dev)
        h = rows // 2
        thr = np.quantile(np.moveaxis(x, 1, 0).reshape(4, -1), 0.3, axis=1)
        for thresholds in (None, thr):
            for live in (np.arange(4), np.array([2, 0])):
                for lag0 in (0, 5, h - 3, h + 2):
                    got = red.autocov(block, thresholds, live, lag0, 16)
                    want = ref.autocov(torch.from_numpy(x), thresholds, live, lag0, 16)
                    assert np.array_equal(got[:, 0], want[:, 0])
                    assert np.allclose(got[:, 1:], want[:, 1:], rtol=1e-11, atol=1e-12 * chains), (rows, chains, lag0)
                    past = lag0 + np.arange(16) >= h
                    assert np.all(got[:, 3:][:, past] == 0)
                    again = red.autocov(block, thresholds, live, lag0, 16)
                    assert np.array_equal(got.view(np.uint64), again.view(np.uint64))
            const = red.autocov(block, thresholds, np.array([3]), 0, 16)
            assert const[0, 2] == 0 and np.all(const[0, 3:] == 0)
        # a shorter tile returns the leading lags of the full one, bit for bit
        a = red.autocov(block, None, np.arange(4), 3, 16)
        b = red.autocov(block, None, np.arange(4), 3, 5)
        assert np.array_equal(a[:, :8].view(np.uint64), b.view(np.uint64))


def test_sample_summary_ess_config2_shape(gpu_pkg):
    mcmc, ld = gpu_pkg.mcmc, gpu_pkg.ld
    params = {"mu": {"type": "real"}, "sigma": {"type": "real", "lower": 0}}
    data = config2_data().tolist()
    mk = lambda: mcmc.AmwgSampler(params, models.norm_post_readme(ld), data, {"chains": 4096, "seed": 21})
    a, b, c = mk(), mk(), mk()
    for s in (a, b, c):
        s.burn(2500)
    raw = a.sample(50)
    with_ess = b.sample_summary(50, ess=True)
    plain = c.sample_summary(50)
    for name in ("mu", "sigma"):
        _check(with_ess, raw, name, 50, 4096)
        assert 0 < with_ess[name]["ess"] < 50 * 4096 * np.log10(50 * 4096)
        for k in ("mean", "sd", "rhat", "quantiles", "n_draws"):
            assert np.array_equal(np.asarray(with_ess[name][k]), np.asarray(plain[name][k])), (name, k)
        assert set(with_ess[name]) == set(plain[name]) | {"ess", "ess_tail", "mcse"}
    sb, sc = b.state, c.state
    assert np.array_equal(sb["mu"], sc["mu"]) and np.array_equal(sb["sigma"], sc["sigma"])


def test_sample_summary_ess_thin_multidim_int_and_derived(gpu_pkg):
    mcmc, ld = gpu_pkg.mcmc, gpu_pkg.ld
    pars = {"x": {"type": "int", "dim": [2, 2], "lower": 0, "init": [[1, 10], [100, 1000]]}}
    mk = lambda: mcmc.AmwgSampler(pars, models.multivar_poisson_dens(ld), None, {"chains": 300, "seed": 5, "thin": 3})
    a, b = mk(), mk()
    a.burn(100); b.burn(100)
    raw, summ = a.sample(31), b.sample_summary(31, (0.1, 0.5, 0.9), ess=True)
    assert summ["x"]["ess"].shape == (2, 2) and summ["x"]["quantiles"].shape == (3, 2, 2)
    _check(summ, raw, "x", 11, 300)
    pars = {"mu": {"type": "real"}, "sigma": {"type": "real", "lower": 0}}
    mk = lambda: mcmc.AmwgSampler(pars, models.norm_post_test(ld), NORM_DATA, {"chains": 257, "seed": 6, "monitor": ["var", "mu"]})
    a, b = mk(), mk()
    a.burn(200); b.burn(200)
    raw, summ = a.sample(20), b.sample_summary(20, (0.05, 0.5), ess=True)
    assert set(summ) == {"var", "mu"} and len(summ["mu"]["quantiles"]) == 2
    for name in ("var", "mu"):
        _check(summ, raw, name, 20, 257)
    # fewer than 8 kept rows: NaN, the rest of the summary as usual
    short = b.sample_summary(7, ess=True)
    assert np.isnan(short["mu"]["ess"]) and np.isnan(short["mu"]["ess_tail"]) and np.isnan(short["mu"]["mcse"])
    assert np.isfinite(short["mu"]["mean"])


def test_entries_needing_different_numbers_of_tiles(gpu_pkg):
    """a config-4-shaped model (mu dim [64] + sigma: 65 entries). The group means adapt and mix fast; sigma keeps a tiny proposal
    scale (its adaptation capped at 1e-9 per batch), so its sequence runs to the end of the chain and needs many more tiles."""
    import torch
    from bayes_js_b200.summary import CudaBlockReducer, summarise_ess
    mcmc, ld = gpu_pkg.mcmc, gpu_pkg.ld
    J, per, chains, n = 64, 16, 512, 1000
    g = np.repeat(np.arange(J), per)
    y = np.random.default_rng(64).normal(0, 2, J)[g] + np.random.default_rng(65).normal(0, 5, J * per)
    params = {"mu": {"type": "real", "dim": [J]}, "sigma": {"type": "real", "lower": 0, "init": 5}}
    data = {"y": y, "g": g.astype(np.float64)}
    mk = lambda: mcmc.AmwgSampler(params, models.hier_norm_post(ld), data,
                                  {"chains": chains, "seed": 8, "params": {"sigma": {"prop_log_scale": -5, "max_adaptation": 1e-9}}})
    a, b = mk(), mk()
    a.burn(500); b.burn(500)
    raw, summ = a.sample(n), b.sample_summary(n, ess=True)
    for name in raw:
        _check(summ, raw, name, n, chains)
    # the tile counts differ between entries, and the device path reads only the live ones
    x = np.concatenate([raw[k].reshape(n, chains, -1) for k in ("mu", "sigma")], axis=2)
    block = torch.from_numpy(np.ascontiguousarray(np.moveaxis(x, 2, 1))).to(torch.device("cuda", 0))
    q05, q95 = np.quantile(np.moveaxis(x, 2, 0).reshape(x.shape[2], -1), [0.05, 0.95], axis=1)
    _, _, tiles = summarise_ess(CudaBlockReducer(0), block, n, chains, q05, q95, False)
    assert x.shape[2] == 65 and tiles[0, :64].max() < tiles[0, 64], tiles[0]
