"""Rank normalisation in `sample_summary(rank=True)` on the device: the radix sort against numpy's stable argsort on adversarial
keys, the z block against ndtri of the exact average ranks, and the whole path against the host reference on the raw draws of
an identically seeded sampler."""
import ctypes as C

import numpy as np
import pytest

import models
from conftest import NORM_DATA, config2_data
from summary_rank_ref import NumpyRankReducer, reference_z

pytestmark = pytest.mark.gpu


def _sort(pkg, keys_u64):
    """-> (sorted keys, payloads, passes run, skipped) from amwg_summary_rank_sort on payloads 0 .. n-1"""
    import torch
    dev = torch.device("cuda", 0)
    k = torch.from_numpy(keys_u64.view(np.int64).copy()).to(dev)
    v = torch.arange(k.numel(), dtype=torch.int32, device=dev)
    ka, va = torch.empty_like(k), torch.empty_like(v)
    passes = (C.c_int32 * 3)()
    L = pkg._ffi.lib()
    pkg._ffi.check(L.amwg_summary_rank_sort(0, k.data_ptr(), v.data_ptr(), k.numel(), ka.data_ptr(), va.data_ptr(), passes))
    if passes[2]:
        k, v = ka, va
    return k.cpu().numpy().view(np.uint64), v.cpu().numpy().astype(np.int64), passes[0], passes[1]


def test_radix_sort_against_numpy_argsort(gpu_pkg):
    from bayes_js_b200.summary import double_to_key
    rng = np.random.default_rng(7)
    u = lambda n: rng.integers(0, 1 << 63, n, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, n).astype(np.uint64)
    base = np.uint64(0x4067_1000_0000_0000)
    special = np.array([0.0, -0.0, 5e-324, -5e-324, 2.2e-308, -2.2e-308, np.inf, -np.inf, 1.0, -1.0] * 50)
    cases = {
        "one": (np.array([12345], dtype=np.uint64), 8),
        "ragged": (u(3 * 4096 + 5), 0),
        "top byte": ((rng.integers(0, 256, 9000).astype(np.uint64) << np.uint64(56)) | np.uint64(0x1234), 7),
        "low byte": (base | rng.integers(0, 256, 9000).astype(np.uint64), 7),
        "all bytes": (u(200_003), 0),
        "one value 1e6 times": (np.full(1_000_000, base, dtype=np.uint64), 8),        # every pass skipped: the skip logic only
        # 90 % equal keys with varying low bytes: heavy ties go through the stable scatter passes
        "mostly one value": (np.where(rng.random(300_000) < 0.9, base, base + np.uint64(1) + rng.integers(0, 1000, 300_000).astype(np.uint64)), None),
        "signed zeros, subnormals, infinities": (double_to_key(np.where(special == 0, 0.0, special)), None),
    }
    for name, (keys, skipped) in cases.items():
        got_k, got_v, run, skip = _sort(gpu_pkg, keys)
        order = np.argsort(keys, kind="stable")
        assert np.array_equal(got_k, keys[order]), name
        assert np.array_equal(got_v, order), name                    # stable: equal keys keep their input order
        assert run + skip == 8, name
        if skipped is not None:
            assert skip == skipped, (name, skip)


def test_z_block_against_ndtri_of_exact_ranks(gpu_pkg):
    """within 8 ulp of ndtri (1e-15 absolute near z = 0); adjacent ranks differ by far more, so every rank is exact"""
    import torch
    from bayes_js_b200.summary import CudaBlockReducer, rank_normalise
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(3)
    for rows, chains in [(41, 1000), (24, 4097), (2, 1)]:
        x = np.empty((rows, 4, chains))
        x[:, 0] = 184.5 + 0.01 * rng.normal(size=(rows, chains))
        x[:, 1] = np.round(3 * rng.normal(size=(rows, chains)))
        x[:, 2] = np.where(rng.random((rows, chains)) < 0.5, -0.0, 0.0) + np.where(rng.random((rows, chains)) < 0.1, 5e-324, 0.0)
        x[:, 3] = rng.standard_cauchy(size=(rows, chains))
        block = torch.from_numpy(x).to(dev)
        med = np.median(np.moveaxis(x, 1, 0).reshape(4, -1), axis=1)
        for center in (None, med):
            z, finite = rank_normalise(CudaBlockReducer(0), block, rows, chains, center, False)
            again, _ = rank_normalise(CudaBlockReducer(0), block, rows, chains, center, False)
            got = z.cpu().numpy()
            assert finite.all() and np.array_equal(got.view(np.uint64), again.cpu().numpy().view(np.uint64))
            host, _ = rank_normalise(NumpyRankReducer(), torch.from_numpy(x), rows, chains, center, False)
            for e in range(4):
                want = reference_z(x[:, e], None if center is None else med[e])
                tol = 8 * np.spacing(np.abs(want)) + 1e-15
                assert np.all(np.abs(got[:, e] - want) <= tol), (rows, chains, e, np.abs(got[:, e] - want).max())
                assert np.all(np.abs(got[:, e] - host.numpy()[:, e]) <= tol)


def test_owner_merge_z_and_reply_against_the_numpy_stand_in(gpu_pkg):
    """the device side of the exchange across GPUs, on one GPU: rank_merge (sort with the receive index as payload, weighted
    run-length encoding), rank_z at a rank offset and the 1-d rank_scatter that puts each received pair's z in receive order,
    against the numpy stand-in. Equal keys arrive from several senders out of order, some keys once, and a receive is empty."""
    import torch
    from bayes_js_b200.summary import CudaBlockReducer, double_to_key
    dev = torch.device("cuda", 0)
    red, ref = CudaBlockReducer(0), NumpyRankReducer()
    rng = np.random.default_rng(11)
    values = np.round(rng.normal(size=400), 1)
    cases = []
    for senders in (2, 3, 5):                                   # each sender's runs: sorted distinct keys with counts
        parts = []
        for _ in range(senders):
            v = np.unique(rng.choice(values, 120))
            parts.append((double_to_key(v), rng.integers(1, 1 << 20, len(v))))
        keys = np.concatenate([p[0] for p in parts])
        counts = np.concatenate([p[1] for p in parts])
        cases.append((keys, counts))
    big = double_to_key(np.round(rng.normal(size=300_000), 3))   # many equal keys per run, more than a sort tile
    cases.append((big, rng.integers(1, 100, big.size)))
    cases.append((np.array([12345], dtype=np.uint64), np.array([7])))
    cases.append((np.zeros(0, dtype=np.uint64), np.zeros(0, dtype=np.int64)))
    total = 1 << 40
    for keys, counts in cases:
        k = torch.from_numpy(keys.view(np.int64).copy())
        c = torch.from_numpy(counts.astype(np.int64))
        offset = int(rng.integers(0, 1 << 30))
        want_runs = ref.rank_merge(k.clone(), c)
        want_z = ref.rank_z(want_runs.counts, offset, total)
        want = torch.empty(keys.size, dtype=torch.float64)
        ref.rank_scatter(want_runs, want_z, want, 0)
        got_runs = red.rank_merge(k.clone().to(dev), c.to(dev))
        assert np.array_equal(got_runs.counts.cpu().numpy(), want_runs.counts.numpy())
        got_z = red.rank_z(got_runs.counts, offset, total)
        got = torch.empty(keys.size, dtype=torch.float64, device=dev)
        red.rank_scatter(got_runs, got_z, got, 0)
        w = want.numpy()
        assert np.all(np.abs(got.cpu().numpy() - w) <= 8 * np.spacing(np.abs(w)) + 1e-15), keys.size
        assert len(np.unique(keys)) == got_runs.counts.numel() and int(got_runs.counts.sum()) == int(counts.sum())


def _gloo_worker(rank, world, port, q):
    import os
    import sys
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    sys.path.insert(0, os.path.join(root, "tests"))
    import torch
    import torch.distributed as dist
    import __graft_entry__ as graft
    graft.load_package()
    from bayes_js_b200.parallel import shard_bounds
    from bayes_js_b200.summary import CudaBlockReducer, rank_normalise, summarise_rank
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        dev = torch.device("cuda", 0)
        rng = np.random.default_rng(17)
        rows, chains = 40, 3001
        x = np.empty((rows, 3, chains))
        x[:, 0] = 184.5 + 0.1 * rng.normal(size=(rows, chains)).cumsum(axis=0)
        x[:, 1] = np.round(2 * rng.normal(size=(rows, chains)))
        x[:, 2] = (rng.random((rows, chains)) < 0.1).astype(np.float64)
        first, count = shard_bounds(chains, rank, world)
        mine = torch.from_numpy(np.ascontiguousarray(x[:, :, first:first + count])).to(dev)
        full = torch.from_numpy(x).to(dev)
        med = np.median(np.moveaxis(x, 1, 0).reshape(3, -1), axis=1)
        ok = True
        for center in (None, med):
            z, _ = rank_normalise(CudaBlockReducer(0), mine, rows, chains, center, True)
            z1, _ = rank_normalise(CudaBlockReducer(0), full, rows, chains, center, False)
            ok &= np.array_equal(z.cpu().numpy().view(np.uint64), np.ascontiguousarray(z1.cpu().numpy()[:, :, first:first + count]).view(np.uint64))
        got = np.array(summarise_rank(CudaBlockReducer(0), mine, rows, chains, med, True))
        one = np.array(summarise_rank(CudaBlockReducer(0), full, rows, chains, med, False))
        ok &= np.allclose(got, one, rtol=1e-12, atol=0, equal_nan=True)
        q.put((rank, bool(ok), got.tobytes()))
    finally:
        dist.destroy_process_group()


def test_rank_exchange_of_two_processes_sharing_the_gpu(gpu_pkg):
    """the whole exchange with the device reducer: two processes on GPU 0 (gloo carries the collectives). Each rank's z block is
    the single-GPU slice bit for bit, and both ranks return the same bits, equal to one GPU to rtol 1e-12"""
    import socket
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in procs]
    res = [q.get(timeout=300) for _ in procs]
    [p.join(timeout=60) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    assert all(ok for _, ok, _ in res)
    assert res[0][2] == res[1][2]


def _host_rank(raw, name, rows, n_chains):
    """host reference on the draws sample() returns: summarise_rank over the numpy stand-in, med from numpy.median"""
    import torch
    from bayes_js_b200.summary import summarise_rank
    x = raw[name]                                            # [rows, chains, *dim]
    flat = np.ascontiguousarray(np.moveaxis(x.reshape(x.shape[0], x.shape[1], -1), 2, 1))      # [rows, entries, chains]
    med = np.median(np.moveaxis(flat, 1, 0).reshape(flat.shape[1], -1), axis=1)
    return summarise_rank(NumpyRankReducer(), torch.from_numpy(flat), rows, n_chains, med, False)


def _check(summary, raw, name, rows, n_chains, rtol=1e-9):
    want = _host_rank(raw, name, rows, n_chains)
    dim = raw[name].shape[2:]
    shape = (lambda a: a.reshape(dim)) if dim else (lambda a: a[0])
    got = summary[name]
    for key, w in zip(("rhat_bulk", "rhat_folded", "rhat_rank", "ess_bulk"), want):
        assert np.allclose(got[key], shape(w), rtol=rtol, atol=0, equal_nan=True), (name, key, got[key], w)


def test_sample_summary_rank_config2_shape(gpu_pkg):
    mcmc, ld = gpu_pkg.mcmc, gpu_pkg.ld
    params = {"mu": {"type": "real"}, "sigma": {"type": "real", "lower": 0}}
    data = config2_data().tolist()
    mk = lambda: mcmc.AmwgSampler(params, models.norm_post_readme(ld), data, {"chains": 4096, "seed": 21})
    a, b, c, d = mk(), mk(), mk(), mk()
    for s in (a, b, c, d):
        s.burn(2500)
    raw = a.sample(50)
    with_rank = b.sample_summary(50, rank=True)
    plain = c.sample_summary(50)
    both = d.sample_summary(50, ess=True, rank=True)
    for name in ("mu", "sigma"):
        _check(with_rank, raw, name, 50, 4096)
        assert 0.99 < with_rank[name]["rhat_rank"] < 1.1
        for k in ("mean", "sd", "rhat", "quantiles", "n_draws"):
            assert np.array_equal(np.asarray(with_rank[name][k]), np.asarray(plain[name][k])), (name, k)
            assert np.array_equal(np.asarray(both[name][k]), np.asarray(plain[name][k])), (name, k)
        for k in ("rhat_bulk", "rhat_folded", "rhat_rank", "ess_bulk"):
            assert np.array_equal(np.asarray(both[name][k]), np.asarray(with_rank[name][k])), (name, k)
        assert set(with_rank[name]) == set(plain[name]) | {"rhat_bulk", "rhat_folded", "rhat_rank", "ess_bulk"}
    for s in (b, d):
        assert np.array_equal(s.state["mu"], c.state["mu"]) and np.array_equal(s.state["sigma"], c.state["sigma"])


def test_sample_summary_rank_thin_multidim_int_and_derived(gpu_pkg):
    mcmc, ld = gpu_pkg.mcmc, gpu_pkg.ld
    pars = {"x": {"type": "int", "dim": [2, 2], "lower": 0, "init": [[1, 10], [100, 1000]]}}
    mk = lambda: mcmc.AmwgSampler(pars, models.multivar_poisson_dens(ld), None, {"chains": 300, "seed": 5, "thin": 3})
    a, b, c = mk(), mk(), mk()
    a.burn(100); b.burn(100); c.burn(100)
    raw, summ, plain = a.sample(31), b.sample_summary(31, (0.1, 0.5, 0.9), rank=True), c.sample_summary(31, (0.1, 0.5, 0.9))
    assert summ["x"]["rhat_rank"].shape == (2, 2) and summ["x"]["ess_bulk"].shape == (2, 2)
    _check(summ, raw, "x", 11, 300)
    assert np.array_equal(summ["x"]["quantiles"], plain["x"]["quantiles"])
    pars = {"mu": {"type": "real"}, "sigma": {"type": "real", "lower": 0}}
    mk = lambda: mcmc.AmwgSampler(pars, models.norm_post_test(ld), NORM_DATA, {"chains": 257, "seed": 6, "monitor": ["var", "mu"]})
    a, b = mk(), mk()
    a.burn(200); b.burn(200)
    raw, summ = a.sample(20), b.sample_summary(20, (0.05, 0.5), rank=True)
    assert set(summ) == {"var", "mu"}
    for name in ("var", "mu"):
        _check(summ, raw, name, 20, 257)
    short = b.sample_summary(7, rank=True)                    # fewer than 8 kept rows: NaN, the rest as usual
    assert np.isnan(short["mu"]["rhat_rank"]) and np.isnan(short["mu"]["ess_bulk"]) and np.isfinite(short["mu"]["mean"])


def test_sample_summary_rank_hierarchical_65_entries(gpu_pkg):
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
    raw, summ = a.sample(n), b.sample_summary(n, ess=True, rank=True)
    for name in raw:
        _check(summ, raw, name, n, chains)
