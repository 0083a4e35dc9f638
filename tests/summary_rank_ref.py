"""Test infrastructure: the numpy stand-in of tests/summary_ess_ref.py with the rank-normalisation calls of
bayes_js_b200.summary.CudaBlockReducer added (amwg_summary_rank_*: np.unique instead of the radix sort, scipy's ndtri instead of
normcdfinv), so that the host logic and the collectives of summarise_rank run on CPU tensors; and an independent reference
(scipy.stats.rankdata over the pooled split draws, ndtri, reference_ess, a direct split R-hat). Never imported by the product."""
import numpy as np
from scipy.special import ndtri
from scipy.stats import rankdata

from summary_ess_ref import NumpyEssReducer, reference_ess, split_chains


def _keys(y):
    from bayes_js_b200.summary import double_to_key
    y = np.where(y == 0.0, 0.0, y)                           # -0 and +0 tie
    return double_to_key(y)


def _z(below, counts, total):
    """the device formula, operation for operation: average rank below + (count + 1) / 2, then Phi^-1"""
    r = below.astype(np.float64) + 0.5 * (counts + 1).astype(np.float64)
    return ndtri((r - 0.375) / (float(total) + 0.25))


class NumpyRankReducer(NumpyEssReducer):
    def rank_runs(self, block, entry, center, keep_keys):
        import torch
        from bayes_js_b200.summary import RankRuns
        x = block.numpy()[:, entry, :]
        rows = x.shape[0]
        h = rows // 2
        y = np.concatenate([x[:h], x[rows - h:]], axis=0)    # [2h, chains]: position r' * chains + c
        if center is not None:
            y = np.abs(y - center)
        k = _keys(y.ravel())
        uniq, inverse, counts = np.unique(k, return_inverse=True, return_counts=True)
        runs = RankRuns(torch.from_numpy(np.arange(k.size)), torch.from_numpy(inverse.astype(np.int64)), torch.from_numpy(counts.astype(np.int64)),
                        torch.from_numpy(uniq.view(np.int64).copy()) if keep_keys else None, k.size)
        runs.sorted_keys = torch.from_numpy(np.sort(k).view(np.int64).copy())
        return runs

    def rank_merge(self, keys, counts):
        import torch
        from bayes_js_b200.summary import RankRuns
        k = keys.numpy().view(np.uint64)
        uniq, inverse = np.unique(k, return_inverse=True)
        summed = np.zeros(len(uniq), dtype=np.int64)
        np.add.at(summed, inverse, counts.numpy())
        return RankRuns(torch.from_numpy(np.arange(k.size)), torch.from_numpy(inverse.astype(np.int64)), torch.from_numpy(summed),
                        None, k.size)

    def rank_z(self, counts, offset, total, out=None):
        import torch
        c = counts.numpy()
        below = offset + np.concatenate([[0], np.cumsum(c)[:-1]]).astype(np.int64) if len(c) else np.zeros(0, dtype=np.int64)
        z = torch.from_numpy(_z(below, c, total))
        if out is not None:
            out.copy_(z)
            return out
        return z

    def rank_scatter(self, runs, run_z, out, entry):
        z = run_z.numpy()[runs.run_id.numpy()]               # per payload position (vals is the identity here)
        o = out.numpy()
        if o.ndim == 3:
            o[:, entry, :] = z.reshape(o.shape[0], o.shape[2])
        else:
            o[runs.vals.numpy()] = z


def reference_z(x, center=None):
    """x [rows, chains] -> the z of the split draws [2h, chains] (scipy.stats.rankdata, ndtri)"""
    rows = x.shape[0]
    h = rows // 2
    y = np.concatenate([x[:h], x[rows - h:]], axis=0)
    if center is not None:
        y = np.abs(y - center)
    r = rankdata(y.ravel(), method="average")
    return ndtri((r - 0.375) / (y.size + 0.25)).reshape(y.shape)


def reference_split_rhat(z):
    """z [2h, chains] -> split R-hat over the 2 x chains half-chains, from numpy's variances"""
    halves = split_chains(z)                                  # [2 chains, h]
    n = halves.shape[1]
    W = halves.var(axis=1, ddof=1).mean()
    B_over_n = halves.mean(axis=1).var(ddof=1)
    with np.errstate(invalid="ignore", divide="ignore"):
        v = (n - 1) / n * W + B_over_n
        return np.sqrt(v / W) if W > 0 and v > 0 else np.nan


def reference_rank_block(x):
    """x [rows, entries, chains] -> (rhat_bulk, rhat_folded, rhat_rank, ess_bulk) per entry, as posterior / ArviZ define them"""
    rows, entries, _ = x.shape
    out = np.full((4, entries), np.nan)
    if rows < 8:
        return out
    for e in range(entries):
        y = x[:, e, :]
        if not np.all(np.isfinite(y)):
            continue
        z = reference_z(y)
        zf = reference_z(y, np.median(y))
        out[0, e] = reference_split_rhat(z)
        out[1, e] = reference_split_rhat(zf)
        out[2, e] = max(out[0, e], out[1, e])
        out[3, e] = reference_ess(split_chains(z)) if not np.isnan(out[0, e]) else np.nan
    return out
