"""Host side of the effective sample size in `sample_summary(ess=True)`: Geyer's sequence over tiles of split-chain
autocovariance sums (bayes_js_b200.summary.summarise_ess), on CPU tensors with the numpy stand-in of amwg_summary_autocov
(tests/summary_ess_ref.py), against an independent FFT-based reference and the analytic ESS of AR(1) chains."""
import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ess(x, lag_tile=16):
    import torch
    from bayes_js_b200.summary import summarise_ess
    from summary_ess_ref import NumpyEssReducer
    q05, q95 = np.quantile(np.moveaxis(x, 1, 0).reshape(x.shape[1], -1), [0.05, 0.95], axis=1)
    return summarise_ess(NumpyEssReducer(lag_tile), torch.from_numpy(x), x.shape[0], x.shape[2], q05, q95, False)


def _ar1(phi, rows, chains, seed):
    """stationary AR(1) chains with unit marginal variance, [rows, chains]"""
    rng = np.random.default_rng(seed)
    y = np.empty((rows, chains))
    y[0] = rng.normal(size=chains)
    e = rng.normal(0, np.sqrt(1 - phi * phi), (rows, chains))
    for r in range(1, rows):
        y[r] = phi * y[r - 1] + e[r]
    return y


def _block(rows, chains, seed):
    """entries: an autocorrelated real, an int-valued one with many ties, an IID one"""
    x = np.empty((rows, 3, chains))
    x[:, 0] = 184.5 + 0.14 * _ar1(0.7, rows, chains, seed)
    x[:, 1] = np.round(3 * _ar1(0.4, rows, chains, seed + 1))
    x[:, 2] = np.random.default_rng(seed + 2).normal(size=(rows, chains))
    return x


@pytest.mark.parametrize("rows,chains", [(40, 33), (41, 17), (9, 64), (200, 5)])
def test_host_ess_matches_the_independent_reference(pkg, rows, chains):
    from summary_ess_ref import reference_ess_block
    x = _block(rows, chains, rows + chains)
    ess, tail, tiles = _ess(x)
    ess0, tail0 = reference_ess_block(x)
    assert np.allclose(ess, ess0, rtol=1e-10, atol=0), (ess, ess0)
    assert np.allclose(tail, tail0, rtol=1e-10, atol=0), (tail, tail0)
    assert tiles.shape == (3, 3) and np.all(tiles >= 1)


def test_indicator_thresholds_are_per_entry(pkg):
    import torch
    from bayes_js_b200.summary import _ess_pass
    from summary_ess_ref import NumpyEssReducer, reference_ess, split_chains
    x = _block(30, 21, 4)
    thr = np.array([184.5, 0.0, 1.0])
    got, _ = _ess_pass(NumpyEssReducer(), torch.from_numpy(x), 15, thr, False)
    want = [reference_ess(split_chains((x[:, e] <= thr[e]).astype(float))) for e in range(3)]
    assert np.allclose(got, want, rtol=1e-10, atol=0)


@pytest.mark.parametrize("phi", [0.9, 0.5, -0.3])
def test_ar1_ess_matches_the_analytic_value(pkg, phi):
    # h = 2000 draws per half-chain. The estimator itself (ArviZ / posterior, independent reference included) carries an O(1/h)
    # bias per lag: at 4096 chains x 400 rows it gives ess / S 20 % low at phi = 0.9 and 7 % high at phi = -0.3.
    rows, chains = 4000, 1024
    x = _ar1(phi, rows, chains, int(1000 * (phi + 1)))[:, None, :]
    ess, _, _ = _ess(x)
    S = 2 * chains * (rows // 2)
    want = (1 - phi) / (1 + phi)
    assert abs(ess[0] / S / want - 1) < 0.05, (ess[0] / S, want)
    if phi < 0:
        assert 1 < ess[0] / S < np.log10(S)                   # antithetic: above S, under the 1/log10(S) cap on tau


def test_iid_draws_have_ess_near_the_draw_count(pkg):
    rows, chains = 400, 4096
    x = np.random.default_rng(9).normal(size=(rows, 1, chains))
    ess, tail, _ = _ess(x)
    S = 2 * chains * (rows // 2)
    assert abs(ess[0] / S - 1) < 0.05 and abs(tail[0] / S - 1) < 0.05


def test_nan_cases(pkg):
    # fewer than 8 rows: half-chains shorter than 4 draws
    ess, tail, tiles = _ess(_block(7, 10, 1))
    assert np.all(np.isnan(ess)) and np.all(np.isnan(tail)) and tiles.sum() == 0
    x = _block(20, 12, 2)
    x[:, 0] = 3.5                                           # a constant entry
    x[5, 1, 3] = np.inf                                     # a non-finite draw
    x[:, 2] = np.where(np.arange(12) < 6, 1.0, 2.0)[None, :]      # two values, each chain constant
    ess, tail, _ = _ess(x)
    assert np.isnan(ess[0]) and np.isnan(tail[0])
    assert np.isnan(ess[1]) and np.isnan(tail[1])
    # entry 2 is constant within every chain: var+ > 0 for the mean, but q05 = 1 and q95 = 2 make x <= q95 constant
    assert not np.isnan(ess[2]) and np.isnan(tail[2])


def test_tiling_does_not_change_a_bit(pkg):
    """tile length 2 (a device call per pair of lags, entries dropping out one by one) against one tile covering every lag"""
    x = _block(60, 9, 7)
    x[:, 0] = 184.5 + 0.14 * _ar1(0.95, 60, 9, 7)          # a long sequence: many tiles
    a = _ess(x, lag_tile=2)
    b = _ess(x, lag_tile=64)
    assert a[2][0, 0] > 5 and np.all(b[2] == 1)
    for u, v in zip(a[:2], b[:2]):
        assert np.array_equal(u.view(np.uint64), v.view(np.uint64))


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch
    import torch.distributed as dist
    import __graft_entry__ as graft
    graft.load_package()
    from bayes_js_b200.parallel import shard_bounds
    from bayes_js_b200.summary import summarise_ess
    from summary_ess_ref import NumpyEssReducer
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        x = _block(50, 37, 11)                                 # ragged: 19 + 18 chains
        first, count = shard_bounds(37, rank, world)
        q05, q95 = np.quantile(np.moveaxis(x, 1, 0).reshape(3, -1), [0.05, 0.95], axis=1)
        mine = torch.from_numpy(np.ascontiguousarray(x[:, :, first:first + count]))
        ess, tail, tiles = summarise_ess(NumpyEssReducer(4), mine, 50, 37, q05, q95, True)
        one, one_tail, _ = summarise_ess(NumpyEssReducer(4), torch.from_numpy(x), 50, 37, q05, q95, False)
        ok = np.allclose(ess, one, rtol=1e-12, atol=0) and np.allclose(tail, one_tail, rtol=1e-12, atol=0) and tiles.max() > 1
        q.put((rank, bool(ok), ess.tobytes() + tail.tobytes() + tiles.tobytes()))
    finally:
        dist.destroy_process_group()


def test_ess_over_gloo_world2():
    """every rank reduces its shard; after each tile the sums are all-gathered and merged in rank order, so both ranks take the
    same continuation decisions and return the same bits, equal to the single-shard numbers to rounding"""
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in procs]
    res = [q.get(timeout=120) for _ in procs]
    [p.join(timeout=60) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    assert all(ok for _, ok, _ in res)
    assert res[0][2] == res[1][2]


def test_autocov_argument_errors_come_back_without_a_gpu(pkg):
    L = pkg._ffi.lib()
    out = np.empty(64)
    live = np.zeros(1, dtype=np.int32)
    fake = 0x1000                                              # never dereferenced: the checks come before any CUDA call

    def err(*args):
        assert L.amwg_summary_autocov(*args) != 0
        return L.amwg_last_error().decode()

    assert "rows" in err(0, fake, 7, 1, 4, None, None, 0, 0, 16, out.ctypes.data)
    assert "lag0" in err(0, fake, 8, 1, 4, None, None, 0, -1, 16, out.ctypes.data)
    assert "n_lags" in err(0, fake, 8, 1, 4, None, None, 0, 0, 0, out.ctypes.data)
    assert "n_lags" in err(0, fake, 8, 1, 4, None, None, 0, 0, 17, out.ctypes.data)
    assert "null" in err(0, None, 8, 1, 4, None, None, 0, 0, 16, out.ctypes.data)
    assert "null" in err(0, fake, 8, 1, 4, None, None, 0, 0, 16, None)
    assert "empty" in err(0, fake, 8, 0, 4, None, None, 0, 0, 16, out.ctypes.data)
    live[0] = 3
    assert "out of range" in err(0, fake, 8, 2, 4, None, live.ctypes.data, 1, 0, 16, out.ctypes.data)
    assert "n_live" in err(0, fake, 8, 2, 4, None, live.ctypes.data, 3, 0, 16, out.ctypes.data)
