"""Posterior summaries formed on the device (SURVEY 8(f).3): pooled mean / sd, exact quantiles and the Gelman-Rubin
statistic per monitored entry, over all chains and kept rows of one `sample()` block that never leaves HBM.

The reference returns raw draws (mcmc.js:1029) and its README summarises them on the caller's side (README.md:44-52); at
2^20..2^22 chains the raw block is GBs per call, so `AmwgSampler.sample_summary(n)` keeps it on the GPU and moves a few
hundred bytes instead. Multi-GPU (one process per GPU): every rank reduces its own shard; the shards are combined with two
small collectives -- an all-gather of the per-rank moment records (merged exactly, in rank order) and a sum all-reduce of the
radix-select digit counts (integers) -- so every rank returns the same numbers as a single GPU holding all chains.

With ess=True the summary also carries the effective sample size (`summarise_ess`): split-chain autocovariance sums over lag
tiles, all-gathered and merged in rank order after each tile. With rank=True it carries the rank-normalised split R-hat and bulk
ESS (`summarise_rank`): exact pooled ranks from a device radix sort, the runs of equal values exchanged across GPUs.

Host logic here is plain numpy (tested on CPU); the device work is behind `CudaBlockReducer` (C ABI: amwg_summary_moments,
amwg_summary_digit_hist, amwg_summary_autocov, amwg_summary_rank_*). There is no CPU fallback: without the library or a GPU the
reducer raises.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Sequence, Tuple

import numpy as np

MAX_PREFIXES = 32                      # include/amwg.h: n_prefix <= 32
_SIGN = np.uint64(1 << 63)


# ---------------------------------------------------------------------------------------------------------------------
# moments
def merge_moment_records(records: Sequence[np.ndarray]) -> np.ndarray:
    """Chan merge of per-shard records [entries, 4] = (chains, mean of chain means, M2 of chain means, sum of within-chain M2),
    in the order given (rank order): the same arithmetic as the device tree, so shards combine exactly."""
    acc = np.array(records[0], dtype=np.float64, copy=True)
    for rec in records[1:]:
        b = np.asarray(rec, dtype=np.float64)
        n = acc[:, 0] + b[:, 0]
        d = b[:, 1] - acc[:, 1]
        with np.errstate(invalid="ignore", divide="ignore"):
            mean = np.where(b[:, 0] == 0, acc[:, 1], np.where(acc[:, 0] == 0, b[:, 1], acc[:, 1] + d * (b[:, 0] / n)))
            m2 = np.where(b[:, 0] == 0, acc[:, 2], np.where(acc[:, 0] == 0, b[:, 2], acc[:, 2] + b[:, 2] + d * d * (acc[:, 0] * b[:, 0] / n)))
        acc = np.stack([n, mean, m2, acc[:, 3] + b[:, 3]], axis=1)
    return acc


def finalize_moments(rec: np.ndarray, rows: int) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """(mean, sd, rhat) per entry from the merged record. sd: pooled over all rows*chains draws, ddof=1. rhat: Gelman-Rubin
    potential scale reduction sqrt(((n-1)/n W + B/n) / W) with n = rows, W the mean within-chain variance, B/n the variance of
    the chain means (NaN with fewer than 2 rows or chains, or when W = 0)."""
    G, mean, b2, sw = rec[:, 0], rec[:, 1], rec[:, 2], rec[:, 3]
    M = G * rows
    with np.errstate(invalid="ignore", divide="ignore"):
        sd = np.sqrt((sw + rows * b2) / (M - 1))
        W = sw / (G * (rows - 1))
        varplus = (rows - 1) / rows * W + b2 / (G - 1)
        rhat = np.sqrt(varplus / W)
    return mean, sd, rhat


# ---------------------------------------------------------------------------------------------------------------------
# exact quantiles: MSD radix select on the order-preserving key of an IEEE double
def key_to_double(keys: np.ndarray) -> np.ndarray:
    k = np.asarray(keys, dtype=np.uint64)
    u = np.where((k & _SIGN) != 0, k ^ _SIGN, ~k)
    return u.view(np.float64) if u.ndim else np.array([u], dtype=np.uint64).view(np.float64)[0]


def double_to_key(x: np.ndarray) -> np.ndarray:
    u = np.ascontiguousarray(x, dtype=np.float64).view(np.uint64)
    return np.where((u & _SIGN) != 0, ~u, u | _SIGN)


def quantile_targets(M: int, probs: Sequence[float]):
    """numpy.quantile's default (linear) rule: position p*(M-1) between order statistics lo and lo+1.
    Returns (sorted distinct 0-based ranks, per-prob (index of lo, index of hi, fraction))."""
    ranks: List[int] = []
    plan = []
    for p in probs:
        if not (0.0 <= p <= 1.0):
            raise ValueError("probs must be in [0, 1]")
        pos = p * (M - 1)
        lo = int(np.floor(pos))
        hi = min(lo + 1, M - 1)
        plan.append((lo, hi, pos - lo))
        ranks += [lo, hi]
    uniq = sorted(set(ranks))
    index = {r: i for i, r in enumerate(uniq)}
    return np.asarray(uniq, dtype=np.int64), [(index[lo], index[hi], g) for lo, hi, g in plan]


def _lerp(a, b, t):
    """numpy's _lerp (lib/_function_base_impl.py): a + (b-a)*t, computed from b when t >= 0.5."""
    d = b - a
    return np.where(t >= 0.5, b - d * (1 - t), a + d * t)


class RadixSelect:
    """Host side of the 8-pass select: which prefixes the device should histogram next, and how the summed counts narrow
    each wanted order statistic down by one byte. ranks: sorted 0-based ranks, shared by all entries."""

    def __init__(self, entries: int, ranks: np.ndarray):
        self.E = entries
        self.T = len(ranks)
        self.prefix = np.zeros((entries, self.T), dtype=np.uint64)
        self.rem = np.tile(np.asarray(ranks, dtype=np.int64), (entries, 1))
        self.npass = 0

    def prefixes(self) -> Tuple[np.ndarray, np.ndarray]:
        """([entries, n_prefix] uint64 distinct prefixes padded with repeats, [entries, T] index of each target's prefix)."""
        uniq = [np.unique(self.prefix[e]) for e in range(self.E)]
        n = max(len(u) for u in uniq)
        if n > MAX_PREFIXES:
            raise ValueError("too many quantiles at once: %d distinct order statistics (max %d)" % (n, MAX_PREFIXES))
        table = np.empty((self.E, n), dtype=np.uint64)
        which = np.empty((self.E, self.T), dtype=np.int64)
        for e, u in enumerate(uniq):
            table[e, :len(u)] = u
            table[e, len(u):] = u[0]
            which[e] = np.searchsorted(u, self.prefix[e])
        return table, which

    def advance(self, counts: np.ndarray, which: np.ndarray) -> None:
        """counts [entries, n_prefix, 256] summed over all shards for the prefixes handed out by prefixes()."""
        sel = np.take_along_axis(np.asarray(counts, dtype=np.int64), which[:, :, None], axis=1)      # [E, T, 256]: each target's histogram
        cum = np.cumsum(sel, axis=2)
        d = (cum <= self.rem[:, :, None]).sum(axis=2)                                             # first byte whose cumulative count exceeds the rank
        if np.any(d > 255):
            raise RuntimeError("radix select: rank beyond the counted values (inconsistent histogram)")
        below = np.take_along_axis(cum, np.maximum(d - 1, 0)[:, :, None], axis=2)[:, :, 0]
        self.rem = self.rem - np.where(d > 0, below, 0)
        self.prefix = (self.prefix << np.uint64(8)) | d.astype(np.uint64)
        self.npass += 1

    def values(self) -> np.ndarray:
        assert self.npass == 8
        return key_to_double(self.prefix)


# ---------------------------------------------------------------------------------------------------------------------
class CudaBlockReducer:
    """The device reductions over a torch CUDA tensor block[rows, entries, chains] (fp64, contiguous)."""

    def __init__(self, device: int):
        from . import _ffi
        self.L = _ffi.lib()                       # raises when the extension is missing: no CPU fallback
        self._ffi = _ffi
        self.device = device

    def moments(self, block) -> np.ndarray:
        rows, entries, chains = block.shape
        out = np.empty((entries, 4), dtype=np.float64)
        self._ffi.check(self.L.amwg_summary_moments(self.device, block.data_ptr(), rows, entries, chains, out.ctypes.data))
        return out

    def digit_counts(self, block, npass: int, prefix_table: np.ndarray):
        """-> torch int64 CUDA tensor [entries, n_prefix, 256] (this shard's counts)."""
        import torch
        rows, entries, chains = block.shape
        n_prefix = prefix_table.shape[1]
        dev = block.device
        pre = torch.from_numpy(prefix_table.view(np.int64).copy()).to(dev)
        counts = torch.zeros((entries, n_prefix, 256), dtype=torch.int64, device=dev)
        torch.cuda.current_stream(dev).synchronize()
        self._ffi.check(self.L.amwg_summary_digit_hist(self.device, block.data_ptr(), rows, entries, chains, npass,
                                                       pre.data_ptr(), n_prefix, counts.data_ptr()))
        return counts

    lag_tile = 16                                 # lags per amwg_summary_autocov call (the kernel's compile-time tile)

    def autocov(self, block, thresholds, live, lag0: int, n_lags: int) -> np.ndarray:
        """-> [len(live), 3 + n_lags] (half-chains, mean and M2 of the half-chain means, S_lag0 ..) for this shard (include/amwg.h).
        thresholds: None (y = x) or [entries] (y = x <= thresholds[entry])."""
        import torch
        rows, entries, chains = block.shape
        live = np.ascontiguousarray(live, dtype=np.int32)
        thr = None if thresholds is None else torch.from_numpy(np.ascontiguousarray(thresholds, dtype=np.float64)).to(block.device)
        out = np.empty((len(live), 3 + n_lags), dtype=np.float64)
        torch.cuda.current_stream(block.device).synchronize()
        self._ffi.check(self.L.amwg_summary_autocov(self.device, block.data_ptr(), rows, entries, chains,
                                                    None if thr is None else thr.data_ptr(), live.ctypes.data, len(live),
                                                    int(lag0), int(n_lags), out.ctypes.data))
        return out

    # ---- rank normalisation (include/amwg.h: amwg_summary_rank_*); the returned RankRuns keeps the device buffers alive
    def rank_runs(self, block, entry: int, center, keep_keys: bool) -> "RankRuns":
        """Sort the split draws of `entry` (folded about `center` unless None) and run-length encode them. keep_keys: also the
        distinct keys (int64 view) and the sorted keys, for the exchange across GPUs."""
        import torch
        rows, entries, chains = block.shape
        n = 2 * (rows // 2) * chains
        dev = block.device
        keys = torch.empty(n, dtype=torch.int64, device=dev)
        vals = torch.empty(n, dtype=torch.int32, device=dev)
        keys_alt = torch.empty_like(keys)
        vals_alt = torch.empty_like(vals)
        c = None if center is None else C.byref(C.c_double(float(center)))
        torch.cuda.current_stream(dev).synchronize()
        self._ffi.check(self.L.amwg_summary_rank_keys(self.device, block.data_ptr(), rows, entries, chains, int(entry), c,
                                                      keys.data_ptr(), vals.data_ptr()))
        passes = (C.c_int32 * 3)()
        self._ffi.check(self.L.amwg_summary_rank_sort(self.device, keys.data_ptr(), vals.data_ptr(), n, keys_alt.data_ptr(),
                                                      vals_alt.data_ptr(), passes))
        if passes[2]:
            keys, keys_alt, vals, vals_alt = keys_alt, keys, vals_alt, vals
        # after the sort: vals_alt holds the run of each position, keys_alt the run counts; run keys only when asked for
        runs = self._runs(keys, vals, None, vals_alt, keys_alt, torch.empty(n, dtype=torch.int64, device=dev) if keep_keys else None)
        runs.passes, runs.skipped = int(passes[0]), int(passes[1])
        runs.sorted_keys = keys
        return runs

    def _runs(self, keys, vals, weights, run_id, counts, run_keys) -> "RankRuns":
        import torch
        n = keys.numel()
        n_runs = C.c_int64(0)
        scan = None if weights is None else torch.empty(n, dtype=torch.int64, device=keys.device)
        self._ffi.check(self.L.amwg_summary_rank_runs(self.device, keys.data_ptr(), vals.data_ptr(),
                                                      None if weights is None else weights.data_ptr(),
                                                      None if scan is None else scan.data_ptr(), n, run_id.data_ptr(),
                                                      None if run_keys is None else run_keys.data_ptr(), counts.data_ptr(), C.byref(n_runs)))
        r = n_runs.value
        return RankRuns(vals, run_id, counts[:r], None if run_keys is None else run_keys[:r], n)

    def rank_merge(self, keys, counts) -> "RankRuns":
        """Owner side across GPUs: the received (key, count) pairs sorted by key (payload: the receive index), equal keys'
        counts summed. `keys` (int64 view) is sorted in place: the caller gives up its contents. Device memory while it runs:
        40 B per received pair with `keys` and `counts`; 16 B per pair stay in the result."""
        import torch
        n = keys.numel()
        dev = keys.device
        if n == 0:
            e = torch.empty(0, dtype=torch.int64, device=dev)
            return RankRuns(torch.empty(0, dtype=torch.int32, device=dev), torch.empty(0, dtype=torch.int32, device=dev), e, e, 0)
        k = keys
        v = torch.arange(n, dtype=torch.int32, device=dev)
        k_alt, v_alt = torch.empty_like(k), torch.empty_like(v)
        passes = (C.c_int32 * 3)()
        torch.cuda.current_stream(dev).synchronize()
        self._ffi.check(self.L.amwg_summary_rank_sort(self.device, k.data_ptr(), v.data_ptr(), n, k_alt.data_ptr(), v_alt.data_ptr(), passes))
        if passes[2]:
            k, k_alt, v, v_alt = k_alt, k, v_alt, v
        return self._runs(k, v, counts.contiguous(), v_alt, k_alt, None)

    def rank_z(self, counts, offset: int, total: int, out=None):
        """-> float64 tensor (`out` when given): z per run (include/amwg.h amwg_summary_rank_z)."""
        import torch
        z = torch.empty(counts.numel(), dtype=torch.float64, device=counts.device) if out is None else out
        if counts.numel():
            torch.cuda.current_stream(counts.device).synchronize()
            self._ffi.check(self.L.amwg_summary_rank_z(self.device, counts.data_ptr(), counts.numel(), int(offset), int(total), z.data_ptr()))
        return z

    def rank_scatter(self, runs: "RankRuns", run_z, out, entry: int) -> None:
        """out[2h, entries, chains]: the z of every split draw of `entry`; out 1-d: out[payload] (the owner's reply)."""
        import torch
        if runs.n == 0:
            return
        torch.cuda.current_stream(out.device).synchronize()
        entries, chains = (out.shape[1], out.shape[2]) if out.dim() == 3 else (1, out.numel())
        self._ffi.check(self.L.amwg_summary_rank_scatter(self.device, runs.vals.data_ptr(), runs.run_id.data_ptr(), runs.n,
                                                         run_z.data_ptr(), out.data_ptr(), entries, chains, int(entry)))


def summarise_block(reducer, block, rows: int, total_chains: int, probs: Sequence[float], distributed: bool, order_stats: Sequence[int] = ()):
    """-> (mean, sd, rhat, quantiles[len(probs)]) per entry, over all shards. `reducer` does the per-shard device work;
    the collectives run on the tensors it returns (NCCL for CUDA tensors, gloo for the CPU stand-in used in the tests).
    With order_stats (0-based ranks over all rows * total_chains draws) also -> [len(order_stats), entries] those order
    statistics, selected in the first radix select alongside the quantiles (the quantiles are the same bits either way)."""
    import torch
    entries = block.shape[1]
    rec = reducer.moments(block)
    if distributed:
        import torch.distributed as dist
        ws = dist.get_world_size()
        mine = torch.from_numpy(rec.copy())
        if block.is_cuda:
            mine = mine.to(block.device)
        gathered = torch.empty((ws * entries, 4), dtype=mine.dtype, device=mine.device)     # concatenated on dim 0
        dist.all_gather_into_tensor(gathered, mine)
        rec = merge_moment_records(list(gathered.cpu().numpy().reshape(ws, entries, 4)))
    mean, sd, rhat = finalize_moments(rec, rows)

    probs = [float(p) for p in probs]
    q = np.empty((len(probs), entries))
    extra = np.asarray(order_stats, dtype=np.int64)
    ostat = np.empty((len(extra), entries))
    per_select = MAX_PREFIXES // 2                            # every probability needs at most two order statistics
    chunks, first = [], 0
    while first < len(probs) or (len(extra) and not chunks):  # long probability grids (equal-mass histograms): several selects
        size = per_select - ((len(extra) + 1) // 2 if not chunks else 0)
        chunks.append(first)
        first += size
    for ci, first in enumerate(chunks):
        chunk = probs[first:chunks[ci + 1] if ci + 1 < len(chunks) else len(probs)]
        ranks, plan = quantile_targets(rows * total_chains, chunk)
        if ci == 0 and len(extra):
            union = np.union1d(ranks, extra)
            pos = np.searchsorted(union, ranks)
            plan = [(pos[lo], pos[hi], g) for lo, hi, g in plan]
            ranks = union
        sel = RadixSelect(entries, ranks)
        for npass in range(8):
            table, which = sel.prefixes()
            counts = reducer.digit_counts(block, npass, table)
            if distributed:
                import torch.distributed as dist
                dist.all_reduce(counts)                       # integer sums: exact, independent of the number of GPUs
            sel.advance(counts.cpu().numpy(), which)
        vals = sel.values()                                   # [entries, T]
        for i, (lo, hi, g) in enumerate(plan):
            q[first + i] = _lerp(vals[:, lo], vals[:, hi], g)
        if ci == 0 and len(extra):
            ostat[:] = vals[:, np.searchsorted(ranks, extra)].T
    if len(extra):
        return mean, sd, rhat, q, ostat
    return mean, sd, rhat, q


# ---------------------------------------------------------------------------------------------------------------------
# effective sample size (bulk ESS of the mean and tail ESS) on split chains, without rank normalisation
#
# Per chain h = rows // 2: the half-chains are the first h and the last h kept rows (the middle row of an odd `rows` is dropped);
# M' = 2 x chains over all shards. y = x, or the indicator y = (x <= thr). The device returns, per entry, M', the Chan record
# (mean, M2) of the half-chain means and S_t = sum_halfchains sum_{n=0}^{h-1-t} (y_n - ybar)(y_{n+t} - ybar), ybar the half-chain's
# mean. From these, with S = M' h:
#   W = S_0 / (M'(h-1)),   var+ = S_0 / (M' h) + M2_means / (M'-1),   rho_t = 1 - (W - S_t / (M' h)) / var+
# and Geyer's initial positive sequence with the monotone correction, as ArviZ `_ess` / posterior:::.ess write it (0-based):
#   rho_even = 1, rho_odd = rho_1; t = 1
#   while t < h - 3 and rho_even + rho_odd > 0:            pairs (rho_{t+1}, rho_{t+2}): lags up to h - 2 are read
#       rho_even, rho_odd = rho_{t+1}, rho_{t+2}; kept (else left 0) when rho_even + rho_odd >= 0; t += 2
#   max_t = t - 2; rho_{max_t+1} = rho_even if rho_even > 0           (the "improved estimate" term)
#   for t = 1, 3, .. while t <= max_t - 2: a pair larger than the one before it is set to that pair's mean (monotone pass)
#   tau = max(-1 + 2 sum_{t=0}^{max_t} rho_t + rho_{max_t+1}, 1 / log10(S)),   ess = S / tau
# These are the loop bounds of ArviZ `_ess` and posterior:::.ess (Vehtari et al. 2021, section 3.2; Stan reference manual,
# "Effective sample size"). NaN when h < 4, when a draw of the entry is not finite, or when var+ is 0 (a constant entry or
# indicator). The tail ESS is min(ESS of x <= q05, ESS of x <= q95), as posterior::ess_tail (no rank normalisation).
def geyer_ess(S: np.ndarray, halfchains: float, m2_means: float, h: int):
    """ESS of one entry from its split-chain sums S[0 .. len(S)) (above), or None when Geyer's sequence still needs a lag at or
    beyond len(S). A pure function of the sums it reads: the result does not depend on how the lags were tiled."""
    M = float(halfchains)
    S = np.asarray(S, dtype=np.float64)
    W = S[0] / (M * (h - 1))
    var_plus = S[0] / (M * h) + m2_means / (M - 1)
    if not (np.isfinite(var_plus) and np.isfinite(W) and var_plus > 0):
        return np.nan
    rho = 1.0 - (W - S / (M * h)) / var_plus
    r = [1.0, rho[1]]
    even, odd = 1.0, rho[1]
    t = 1
    while t < h - 3 and even + odd > 0.0:
        if t + 2 >= len(S):
            return None
        even, odd = rho[t + 1], rho[t + 2]
        r += [even, odd] if even + odd >= 0 else [0.0, 0.0]
        t += 2
    max_t = t - 2
    if even > 0:
        r[max_t + 1] = even
    t = 1
    while t <= max_t - 2:
        if r[t + 1] + r[t + 2] > r[t - 1] + r[t]:
            r[t + 1] = (r[t - 1] + r[t]) / 2.0
            r[t + 2] = r[t + 1]
        t += 2
    r = np.asarray(r)
    total = M * h
    tau = -1.0 + 2.0 * np.sum(r[:max_t + 1]) + np.sum(r[max_t + 1:max_t + 2])
    tau = max(tau, 1.0 / np.log10(total))
    return np.nan if np.isnan(r).any() else total / tau


def _gather_autocov(out: np.ndarray, block) -> np.ndarray:
    """All ranks' [live, 3 + n] outputs -> one, merged in rank order: Chan merge of the half-chain-mean records, S_t added."""
    import torch
    import torch.distributed as dist
    ws = dist.get_world_size()
    mine = torch.from_numpy(np.ascontiguousarray(out))
    if block.is_cuda:
        mine = mine.to(block.device)
    gathered = torch.empty((ws * out.shape[0], out.shape[1]), dtype=mine.dtype, device=mine.device)
    dist.all_gather_into_tensor(gathered, mine)
    parts = gathered.cpu().numpy().reshape(ws, *out.shape)
    zero = np.zeros((out.shape[0], 1))
    rec = merge_moment_records([np.concatenate([p[:, :3], zero], axis=1) for p in parts])
    s = parts[0, :, 3:].copy()
    for p in parts[1:]:
        s = s + p[:, 3:]
    return np.concatenate([rec[:, :3], s], axis=1)


def _ess_pass(reducer, block, h: int, thresholds, distributed: bool, want_record: bool = False):
    """-> (ess [entries], lag tiles read per entry). Every entry starts live; after each tile of reducer.lag_tile lags the entries
    whose sequence has ended drop out, and only the live ones are read for the next tile. want_record: also -> the first tile's
    [entries, 4] (half-chains, mean and M2 of the half-chain means, S_0), merged over all shards."""
    entries = block.shape[1]
    L = reducer.lag_tile
    ess = np.full(entries, np.nan)
    tiles = np.zeros(entries, dtype=np.int64)
    S = [np.empty(0)] * entries
    rec = None
    live = np.arange(entries)
    lag0 = 0
    while len(live):
        out = reducer.autocov(block, thresholds, live, lag0, L)
        if distributed:
            out = _gather_autocov(out, block)
        if rec is None:
            rec = out[:, :4].copy()                  # the first tile covers every entry
        nxt = []
        for i, e in enumerate(live):
            S[e] = np.concatenate([S[e], out[i, 3:]])
            tiles[e] += 1
            r = geyer_ess(S[e], rec[e, 0], rec[e, 2], h)
            if r is None:
                nxt.append(e)
            else:
                ess[e] = r
        live = np.asarray(nxt, dtype=np.int64)
        lag0 += L
    if want_record:
        return ess, tiles, rec
    return ess, tiles


def summarise_ess(reducer, block, rows: int, total_chains: int, q05, q95, distributed: bool):
    """-> (ess, ess_tail, tiles[3, entries]) per entry over all shards (definition above). q05 / q95: the pooled 5 % and 95 %
    quantiles per entry; tiles: the lag tiles read for the mean, the q05 and the q95 indicator. Multi-GPU: after each tile the
    per-rank sums are all-gathered and merged in rank order, so every rank takes the same decisions and returns the same bits;
    one GPU and N GPUs agree to rounding, not bit for bit, since the sums are grouped differently."""
    entries = block.shape[1]
    h = rows // 2
    nan = np.full(entries, np.nan)
    if h < 4:
        return nan, nan.copy(), np.zeros((3, entries), dtype=np.int64)
    ess, t0 = _ess_pass(reducer, block, h, None, distributed)
    e05, t1 = _ess_pass(reducer, block, h, np.asarray(q05, dtype=np.float64), distributed)
    e95, t2 = _ess_pass(reducer, block, h, np.asarray(q95, dtype=np.float64), distributed)
    tail = np.where(np.isnan(ess), np.nan, np.minimum(e05, e95))      # a non-finite draw leaves the indicators finite
    return ess, tail, np.stack([t0, t1, t2])


# ---------------------------------------------------------------------------------------------------------------------
# rank-normalised split R-hat and bulk ESS (Vehtari, Gelman, Simpson, Carpenter, Buerkner 2021; posterior::rhat, ess_bulk)
#
# Split: per chain h = rows // 2, the half-chains are the first h and the last h kept rows (the middle row of an odd `rows` is
# dropped, as posterior split_chains / ArviZ _split_chains); S = 2h x total chains split draws per entry.
# Ranks: average ranks (ties get the mean of their positions, scipy.stats.rankdata(method="average")) of the S split draws of the
# entry, pooled over all chains on all GPUs; -0.0 and +0.0 tie. z = Phi^-1((r - 3/8) / (S + 1/4)) (CUDA normcdfinv on the device).
# Fold: zeta = |x - med|, med = numpy.median of all rows x chains draws (the middle row included), (a + b) / 2 of the two middle
# order statistics; zeta goes through the same split, rank and z steps.
# Split R-hat of a z block from the first tile of amwg_summary_autocov (M' half-chains, M2 of the half-chain means, S_0):
#   W = S_0 / (M'(h-1)),   var+ = (h-1)/h W + M2_means / (M'-1),   R-hat = sqrt(var+ / W)
# rhat_bulk is that of z, rhat_folded that of the folded z, rhat_rank = max(rhat_bulk, rhat_folded); ess_bulk is geyer_ess of z
# (the loop bounds above). NaN with fewer than 8 kept rows, when a split draw is not finite, and when W or var+ is 0 (a constant
# entry ties everywhere: z = 0).
#
# Several GPUs: the ranks must be exact over all shards. Every rank sorts its own draws and run-length encodes them into
# (key, count) runs. Regular-sampling splitters: each rank contributes G keys at evenly spaced positions of its sorted draws, they
# are all-gathered and sorted, and every G-th one is a splitter. A run goes to the owner of its key's range (key < splitter), so all
# copies of a value meet at one owner; all_to_all_single moves the runs (keys as an int64 view), the owner merges them (the same
# sort, counts of equal keys summed), its rank offset is the scan of the owners' totals (one all-gather of one integer), and the z
# of every run returns by the reverse all_to_all_single. So every rank's z block is the matching slice of a single GPU's, bit for bit.
class RankRuns:
    """One sorted, run-length encoded key set: vals (payload per sorted position), run_id (run per sorted position), counts (per
    run), keys (per run, int64 view, or None), n (keys sorted)."""

    def __init__(self, vals, run_id, counts, keys, n: int):
        self.vals, self.run_id, self.counts, self.keys, self.n = vals, run_id, counts, keys, n
        self.passes = self.skipped = 0
        self.sorted_keys = None


_KEY_FLIP = -(1 << 63)                 # x ^ _KEY_FLIP on an int64 view: signed order == the keys' unsigned order
RECV_BYTES_PER_RUN = 40 + 16           # the owner's merge (rank_merge with the received keys and counts), then z owned + z sent back


class RankWorkingSetError(MemoryError):
    """The runs one GPU receives in the exchange do not fit in its free device memory (raised on every rank alike)."""


def _device_free(dev) -> int:
    """bytes a new tensor can take: free device memory plus what torch's allocator holds unused"""
    import torch
    free, _ = torch.cuda.mem_get_info(dev)
    return free + torch.cuda.memory_reserved(dev) - torch.cuda.memory_allocated(dev)


def _exchange_z(reducer, runs: RankRuns, total: int):
    """-> float64 tensor [runs]: the z of this rank's runs, ranked over all ranks' draws (above). Before the runs move, every rank
    checks that what it will receive fits (RECV_BYTES_PER_RUN per received run); when one does not, all raise RankWorkingSetError."""
    import torch
    import torch.distributed as dist
    G, me = dist.get_world_size(), dist.get_rank()
    dev = runs.counts.device
    n_runs = runs.counts.numel()
    pos = torch.tensor([(i * runs.n) // G for i in range(G)], dtype=torch.int64, device=dev)
    samples = runs.sorted_keys[pos].contiguous()
    runs.sorted_keys = None                                   # spent: its memory goes to the receive side
    every = torch.empty(G * G, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(every, samples)
    u = np.sort(every.cpu().numpy().view(np.uint64))
    splitters = u[G::G][:G - 1]
    flipped = lambda k: k ^ _KEY_FLIP
    cut = torch.searchsorted(flipped(runs.keys), flipped(torch.from_numpy(splitters.view(np.int64).copy()).to(dev))) if G > 1 else \
        torch.empty(0, dtype=torch.int64, device=dev)
    bounds = [0] + cut.cpu().tolist() + [n_runs]
    send = [bounds[j + 1] - bounds[j] for j in range(G)]
    sizes = torch.tensor(send, dtype=torch.int64, device=dev)
    got = torch.empty_like(sizes)
    dist.all_to_all_single(got, sizes)
    recv = got.cpu().tolist()
    R = sum(recv)
    short = torch.zeros(1, dtype=torch.int64, device=dev)
    need = RECV_BYTES_PER_RUN * R + R // 4 + 8 * n_runs         # + the sort's tile counts, + this rank's z
    if dev.type == "cuda" and need > 0.9 * _device_free(dev):
        short[0] = need
    dist.all_reduce(short, op=dist.ReduceOp.MAX)
    if int(short.item()):
        raise RankWorkingSetError("sample_summary(rank=True): a GPU would receive runs needing %.1f GB in the exchange of ranks, "
                                  "more than its free device memory; raise thin() or lower n" % (int(short.item()) / 1e9))
    keys_in = torch.empty(R, dtype=torch.int64, device=dev)
    counts_in = torch.empty(R, dtype=torch.int64, device=dev)
    dist.all_to_all_single(keys_in, runs.keys.contiguous(), recv, send)
    dist.all_to_all_single(counts_in, runs.counts.contiguous(), recv, send)
    owned = reducer.rank_merge(keys_in, counts_in)              # sorts keys_in in place
    del keys_in
    mine = counts_in.sum().reshape(1).to(torch.int64)
    del counts_in
    totals = torch.empty(G, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(totals, mine)
    offset = int(totals[:me].sum().item())
    z_owned = reducer.rank_z(owned.counts, offset, total)
    z_in = torch.empty(R, dtype=torch.float64, device=dev)
    reducer.rank_scatter(owned, z_owned, z_in, 0)
    del owned, z_owned
    z = torch.empty(n_runs, dtype=torch.float64, device=dev)
    dist.all_to_all_single(z, z_in, send, recv)
    return z


def rank_normalise(reducer, block, rows: int, total_chains: int, center, distributed: bool, out=None, stats=None):
    """-> (z block [2h, entries, chains] (float64, on the block's device; `out` when given), finite [entries] bool): the
    rank-normalised split draws of every entry (definition above), folded about center[entry] unless center is None. Entries go
    through the sort one at a time. finite: every split draw of the entry is finite, over all shards. stats (a dict) collects the
    sort passes run and skipped."""
    import torch
    h = rows // 2
    _, entries, chains = block.shape
    if out is None:
        out = torch.empty((2 * h, entries, chains), dtype=torch.float64, device=block.device)
    total = 2 * h * total_chains
    lo_inf, hi_inf = double_to_key(np.array([-np.inf, np.inf]))
    finite = np.ones(entries, dtype=np.int64)
    for e in range(entries):
        runs = reducer.rank_runs(block, e, None if center is None else float(center[e]), distributed)
        if stats is not None:
            stats["passes"] = stats.get("passes", 0) + runs.passes
            stats["skipped"] = stats.get("skipped", 0) + runs.skipped
        ends = runs.sorted_keys[[0, -1]].cpu().numpy().view(np.uint64)
        if distributed:
            z = _exchange_z(reducer, runs, total)
        else:                                                  # the sorted keys are spent: their buffer takes the z
            z = reducer.rank_z(runs.counts, 0, total, out=runs.sorted_keys.view(torch.float64)[:runs.counts.numel()])
        finite[e] = int(ends[0] > lo_inf and ends[1] < hi_inf)
        reducer.rank_scatter(runs, z, out, e)
        del runs, z
    if distributed:
        import torch.distributed as dist
        f = torch.from_numpy(finite).to(block.device)
        dist.all_reduce(f, op=dist.ReduceOp.MIN)
        finite = f.cpu().numpy()
    return out, finite.astype(bool)


def split_rhat(rec: np.ndarray, h: int) -> np.ndarray:
    """R-hat per entry from [entries, >= 4] (half-chains M', mean and M2 of the half-chain means, S_0) of amwg_summary_autocov."""
    M, m2, S0 = rec[:, 0], rec[:, 2], rec[:, 3]
    with np.errstate(invalid="ignore", divide="ignore"):
        W = S0 / (M * (h - 1))
        var_plus = (h - 1) / h * W + m2 / (M - 1)
        ok = (W > 0) & (var_plus > 0) & np.isfinite(W) & np.isfinite(var_plus)
        return np.where(ok, np.sqrt(np.where(ok, var_plus / W, 1.0)), np.nan)


def summarise_rank(reducer, block, rows: int, total_chains: int, med, distributed: bool, stats=None):
    """-> (rhat_bulk, rhat_folded, rhat_rank, ess_bulk) per entry over all shards (definition above). med: numpy.median of
    every draw of each entry. One z block: the bulk z for ess_bulk and rhat_bulk (the first lag tile's record, merged over the
    shards), then refilled with the folded z for one single-lag autocovariance call. Every rank returns the same bits."""
    entries = block.shape[1]
    h = rows // 2
    nan = np.full(entries, np.nan)
    if h < 4:
        return nan, nan.copy(), nan.copy(), nan.copy()
    z, finite = rank_normalise(reducer, block, rows, total_chains, None, distributed, stats=stats)
    ess, _, rec = _ess_pass(reducer, z, h, None, distributed, want_record=True)
    bulk = split_rhat(rec, h)
    z, finite_f = rank_normalise(reducer, block, rows, total_chains, med, distributed, out=z, stats=stats)
    out = reducer.autocov(z, None, np.arange(entries), 0, 1)
    if distributed:
        out = _gather_autocov(out, z)
    folded = split_rhat(out, h)
    del z
    ok = finite & finite_f
    bulk, folded = np.where(ok, bulk, np.nan), np.where(ok, folded, np.nan)
    return bulk, folded, np.maximum(bulk, folded), np.where(ok, ess, np.nan)
