"""Host side of the rank-normalised diagnostics in `sample_summary(rank=True)` (bayes_js_b200.summary.summarise_rank), on CPU
tensors with the numpy stand-in of the amwg_summary_rank_* calls (tests/summary_rank_ref.py): against an independent reference
(rankdata over the pooled split draws, ndtri, reference_ess, a direct split R-hat), on the cases the diagnostics exist for, across
gloo worlds of 2 and 3, and the argument checks of the new exports."""
import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rank(x, distributed=False, total_chains=None):
    import torch
    from bayes_js_b200.summary import summarise_rank
    from summary_rank_ref import NumpyRankReducer
    med = np.median(np.moveaxis(x, 1, 0).reshape(x.shape[1], -1), axis=1)
    return np.array(summarise_rank(NumpyRankReducer(), torch.from_numpy(np.ascontiguousarray(x)), x.shape[0],
                                   total_chains or x.shape[2], med, distributed))


def _block(rows, chains, seed):
    """entries: an autocorrelated real, tied integers, a binary entry, -0.0 next to +0.0, IID normals"""
    rng = np.random.default_rng(seed)
    x = np.empty((rows, 5, chains))
    x[:, 0] = 184.5 + 0.14 * rng.normal(size=(rows, chains)).cumsum(axis=0) / np.sqrt(np.arange(1, rows + 1))[:, None]
    x[:, 1] = np.round(3 * rng.normal(size=(rows, chains)))
    x[:, 2] = (rng.random((rows, chains)) < 0.3).astype(np.float64)
    x[:, 3] = np.where(rng.random((rows, chains)) < 0.5, -0.0, 0.0) + np.round(rng.normal(size=(rows, chains)))
    x[:, 4] = rng.normal(size=(rows, chains))
    return x


@pytest.mark.parametrize("rows,chains", [(40, 33), (41, 17), (9, 64), (200, 5), (8, 3)])
def test_host_rank_matches_the_independent_reference(pkg, rows, chains):
    from summary_rank_ref import reference_rank_block
    x = _block(rows, chains, rows * chains)
    got = _rank(x)
    want = reference_rank_block(x)
    assert np.allclose(got, want, rtol=1e-10, atol=0, equal_nan=True), (got, want)
    assert np.all(np.isfinite(got)), got


def test_signed_zeros_tie(pkg):
    import torch
    from bayes_js_b200.summary import rank_normalise
    from summary_rank_ref import NumpyRankReducer, reference_z
    x = np.zeros((10, 1, 4))
    x[:, 0, :2] = -0.0
    x[3, 0, 1] = 1.0
    z, finite = rank_normalise(NumpyRankReducer(), torch.from_numpy(x), 10, 4, None, False)
    assert finite[0]
    assert np.array_equal(z.numpy()[:, 0], reference_z(x[:, 0]))
    assert len(np.unique(z.numpy())) == 2


def test_z_block_matches_rankdata_and_ndtri(pkg):
    import torch
    from bayes_js_b200.summary import rank_normalise
    from summary_rank_ref import NumpyRankReducer, reference_z
    x = _block(41, 17, 3)
    med = np.median(np.moveaxis(x, 1, 0).reshape(5, -1), axis=1)
    for center in (None, med):
        z, finite = rank_normalise(NumpyRankReducer(), torch.from_numpy(x), 41, 17, center, False)
        assert z.shape == (40, 5, 17) and finite.all()
        for e in range(5):
            want = reference_z(x[:, e], None if center is None else med[e])
            assert np.allclose(z.numpy()[:, e], want, rtol=1e-14, atol=1e-15)


def test_nan_cases(pkg):
    got = _rank(_block(7, 10, 1))                             # fewer than 8 rows
    assert np.all(np.isnan(got))
    x = _block(20, 12, 2)
    x[:, 0] = 3.5                                             # a constant entry: z = 0 everywhere, W = 0
    x[5, 1, 3] = np.inf                                       # a non-finite draw
    x[2, 2, 0] = np.nan
    got = _rank(x)
    assert np.all(np.isnan(got[:, 0])) and np.all(np.isnan(got[:, 1])) and np.all(np.isnan(got[:, 2]))
    assert np.all(np.isfinite(got[:, 3:]))


def test_scale_difference_is_caught_by_the_folded_rhat(pkg):
    """half the chains N(0, 1), half N(0, 3): the means agree, so the classic R-hat misses it; the folded draws do not"""
    from summary_ref import numpy_summary
    for seed in range(2):
        rng = np.random.default_rng(100 + seed)
        x = rng.normal(size=(200, 1, 64)) * np.where(np.arange(64) < 32, 1.0, 3.0)
        _, _, rhat, _ = numpy_summary(x, [])
        bulk, folded, rk, ess = _rank(x)[:, 0]
        assert rhat[0] < 1.01 and folded > 1.1 and rk > 1.1 and rk == max(bulk, folded), (rhat, bulk, folded)


def test_cauchy_chains_have_bulk_ess_near_the_draw_count(pkg):
    for seed in range(2):
        x = np.random.default_rng(200 + seed).standard_cauchy(size=(200, 1, 64))
        bulk, folded, rk, ess = _rank(x)[:, 0]
        S = 200 * 64
        assert abs(ess / S - 1) < 0.1 and rk < 1.01, (ess / S, rk)


# ---- several ranks: gloo worlds of 2 and 3 with ragged shards
def _cases(world):
    """-> [(name, x)]: a value tied across a splitter, each rank's values all below the next rank's, owners that receive nothing"""
    from bayes_js_b200.parallel import shard_bounds
    rng = np.random.default_rng(5)
    tied = np.round(rng.normal(size=(30, 3, 37)))
    tied[:, 1] = 2.0 * (rng.random((30, 37)) < 0.5)         # two values: one of them sits on a splitter
    low = rng.normal(size=(30, 2, 37))
    for r in range(world):
        first, count = shard_bounds(37, r, world)
        low[:, :, first:first + count] += 100.0 * r           # rank 0 lies below everyone, rank 1 below the rest, ..
    few = (rng.random((30, 1, 37)) < 0.1).astype(np.float64)  # 90 % zeros: every sample and so every splitter is 0, and the
    few[4, 0, 5] = -0.25                                       # owners below it receive nothing
    return [("tied", tied), ("low", low), ("few", few)]


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch
    import torch.distributed as dist
    import __graft_entry__ as graft
    graft.load_package()
    from bayes_js_b200.parallel import shard_bounds
    from bayes_js_b200.summary import rank_normalise, summarise_rank
    from summary_rank_ref import NumpyRankReducer
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        out = []
        for name, x in _cases(world):
            rows, entries, chains = x.shape
            first, count = shard_bounds(chains, rank, world)
            mine = torch.from_numpy(np.ascontiguousarray(x[:, :, first:first + count]))
            med = np.median(np.moveaxis(x, 1, 0).reshape(entries, -1), axis=1)
            ok = True
            for center in (None, med):
                z, fin = rank_normalise(NumpyRankReducer(), mine, rows, chains, center, True)
                z1, fin1 = rank_normalise(NumpyRankReducer(), torch.from_numpy(x), rows, chains, center, False)
                ok &= np.array_equal(z.numpy().view(np.uint64), np.ascontiguousarray(z1.numpy()[:, :, first:first + count]).view(np.uint64))
                ok &= np.array_equal(fin, fin1)
            got = np.array(summarise_rank(NumpyRankReducer(), mine, rows, chains, med, True))
            one = np.array(summarise_rank(NumpyRankReducer(), torch.from_numpy(x), rows, chains, med, False))
            ok &= np.allclose(got, one, rtol=1e-12, atol=0, equal_nan=True)
            out.append((name, bool(ok), got.tobytes()))
        q.put((rank, out))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_rank_over_gloo_worlds(world):
    """every rank's z block is the single-shard slice bit for bit; every rank returns the same bits, equal to one shard to rounding"""
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    [p.start() for p in procs]
    res = [q.get(timeout=180) for _ in procs]
    [p.join(timeout=60) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    for _, out in res:
        for name, ok, _ in out:
            assert ok, name
    for i in range(len(res[0][1])):
        assert len({out[i][2] for _, out in res}) == 1


def test_rank_argument_errors_come_back_without_a_gpu(pkg):
    import ctypes as C
    L = pkg._ffi.lib()
    fake = 0x1000                                             # never dereferenced: the checks come before any CUDA call
    passes = (C.c_int32 * 3)()
    runs = C.c_int64(0)
    center = C.c_double(0.0)

    def err(fn, *args):
        assert fn(*args) != 0
        return L.amwg_last_error().decode()

    keys = L.amwg_summary_rank_keys
    assert "empty" in err(keys, 0, fake, 0, 1, 4, 0, None, fake, fake)
    assert "rows" in err(keys, 0, fake, 1, 1, 4, 0, None, fake, fake)
    assert "entry" in err(keys, 0, fake, 8, 2, 4, 2, None, fake, fake)
    assert "2^32" in err(keys, 0, fake, 1 << 20, 1, 1 << 12, 0, C.byref(center), fake, fake)
    assert "null" in err(keys, 0, None, 8, 1, 4, 0, None, fake, fake)
    assert "null" in err(keys, 0, fake, 8, 1, 4, 0, None, fake, None)
    assert "device" in err(keys, 64, fake, 8, 1, 4, 0, None, fake, fake)
    sort = L.amwg_summary_rank_sort
    assert "n must" in err(sort, 0, fake, fake, 0, fake, fake, passes)
    assert "2^32" in err(sort, 0, fake, fake, 1 << 32, fake, fake, passes)
    assert "null" in err(sort, 0, fake, fake, 10, None, fake, passes)
    assert "null" in err(sort, 0, fake, fake, 10, fake, fake, None)
    assert "device" in err(sort, -1, fake, fake, 10, fake, fake, passes)
    rl = L.amwg_summary_rank_runs
    assert "n must" in err(rl, 0, fake, fake, None, None, 0, fake, None, fake, C.byref(runs))
    assert "2^32" in err(rl, 0, fake, fake, None, None, 1 << 32, fake, None, fake, C.byref(runs))
    assert "null" in err(rl, 0, fake, None, fake, fake, 10, fake, None, fake, C.byref(runs))
    assert "scan buffer" in err(rl, 0, fake, fake, fake, None, 10, fake, None, fake, C.byref(runs))
    assert "null" in err(rl, 0, fake, fake, None, None, 10, fake, None, None, C.byref(runs))
    z = L.amwg_summary_rank_z
    assert "n_runs" in err(z, 0, fake, 0, 0, 10, fake)
    assert "total" in err(z, 0, fake, 5, -1, 10, fake)
    assert "total" in err(z, 0, fake, 5, 0, 0, fake)
    assert "total" in err(z, 0, fake, 5, 0, 1 << 50, fake)
    assert "null" in err(z, 0, None, 5, 0, 10, fake)
    sc = L.amwg_summary_rank_scatter
    assert "n must" in err(sc, 0, fake, fake, 0, fake, fake, 1, 4, 0)
    assert "2^32" in err(sc, 0, fake, fake, 1 << 32, fake, fake, 1, 4, 0)
    assert "empty" in err(sc, 0, fake, fake, 10, fake, fake, 0, 4, 0)
    assert "entry" in err(sc, 0, fake, fake, 10, fake, fake, 2, 4, 2)
    assert "null" in err(sc, 0, fake, fake, 10, fake, None, 1, 4, 0)
