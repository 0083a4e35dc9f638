"""Posterior summaries formed on the device (SURVEY 8(f).3): pooled mean / sd, exact quantiles and the Gelman-Rubin
statistic per monitored entry, over all chains and kept rows of one `sample()` block that never leaves HBM.

The reference returns raw draws (mcmc.js:1029) and its README summarises them on the caller's side (README.md:44-52); at
2^20..2^22 chains the raw block is GBs per call, so `AmwgSampler.sample_summary(n)` keeps it on the GPU and moves a few
hundred bytes instead. Multi-GPU (one process per GPU): every rank reduces its own shard; the shards are combined with two
small collectives -- an all-gather of the per-rank moment records (merged exactly, in rank order) and a sum all-reduce of the
radix-select digit counts (integers) -- so every rank returns the same numbers as a single GPU holding all chains.

With ess=True the summary also carries the effective sample size (`summarise_ess`): split-chain autocovariance sums over lag
tiles, all-gathered and merged in rank order after each tile.

Host logic here is plain numpy (tested on CPU); the device work is behind `CudaBlockReducer` (C ABI: amwg_summary_moments,
amwg_summary_digit_hist, amwg_summary_autocov). There is no CPU fallback: without the library or a GPU the reducer raises.
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


def summarise_block(reducer, block, rows: int, total_chains: int, probs: Sequence[float], distributed: bool):
    """-> (mean, sd, rhat, quantiles[len(probs)]) per entry, over all shards. `reducer` does the per-shard device work;
    the collectives run on the tensors it returns (NCCL for CUDA tensors, gloo for the CPU stand-in used in the tests)."""
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
    per_select = MAX_PREFIXES // 2                            # every probability needs at most two order statistics
    for first in range(0, len(probs), per_select):            # long probability grids (equal-mass histograms): several selects
        chunk = probs[first:first + per_select]
        ranks, plan = quantile_targets(rows * total_chains, chunk)
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


def _ess_pass(reducer, block, h: int, thresholds, distributed: bool):
    """-> (ess [entries], lag tiles read per entry). Every entry starts live; after each tile of reducer.lag_tile lags the entries
    whose sequence has ended drop out, and only the live ones are read for the next tile."""
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
            rec = out[:, :3].copy()                  # the first tile covers every entry
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
