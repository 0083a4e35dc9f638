#!/usr/bin/env python3
"""Cost of the effective sample size in `sample_summary`: `sample_summary(n)` and `sample_summary(n, ess=True)`, alternating,
on one GPU, for bench.py's config 2 (2^20 chains, n = 100 and n = 1000) and config 4 (2^16 chains, n = 200).

    python scripts/bench_summary_ess.py OUTDIR [--rounds 4] [--cases c2n100 c2n1000 c4n200]

Writes OUTDIR/summary_ess.json (nothing into the source tree). Per case: median and spread (min .. max) of each setting's wall time;
the ESS reduction alone on a block of the same shape, with CUDA events around every amwg_summary_autocov call (both kernels and
their small copies); lag tiles per entry; the algorithmic DFMA and HBM bytes of those calls and their share of the bound (the
fp64 peak measured in this process by amwg_peak_fp64, and 7.7 TB/s); n_draws / ess per parameter. The card's name, power limit
and max SM clock are read with nvidia-smi --query-gpu."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
HBM_BYTES_PER_S = 7.7e12                      # HGX B200 data sheet, one GPU
CASES = {"c2n100": (2, 1 << 20, 100), "c2n1000": (2, 1 << 20, 1000), "c4n200": (4, 1 << 16, 200)}


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return "unknown (%s)" % e


def spread(v):
    return {"median": statistics.median(v), "min": min(v), "max": max(v), "runs": v}


def run_case(pkg, bench, k, chains, n, rounds):
    import torch
    from bayes_js_b200.summary import CudaBlockReducer, summarise_block, summarise_ess
    cfg = bench.Config(k, pkg.ld, pkg.mcmc)
    s = pkg.mcmc.AmwgSampler(cfg.params, cfg.log_post, cfg.data, {"chains": chains, "seed": 1, "device": 0})
    s.burn(cfg.burn)
    s.sample_summary(n)                                   # warm-up of every shape the timed runs use
    s.sample_summary(n, ess=True)
    t = {"plain": [], "ess": []}
    last = None
    for r in range(rounds):
        for setting in (("plain", "ess") if r % 2 == 0 else ("ess", "plain")):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = s.sample_summary(n, ess=(setting == "ess"))
            torch.cuda.synchronize()
            t[setting].append(1e3 * (time.perf_counter() - t0))
            if setting == "ess":
                last = out

    # the ESS reduction alone, on a block of the same shape left in HBM by amwg_sample_device
    entries = list(range(cfg.n_entries))
    rows = n
    block = torch.empty((rows, len(entries), chains), dtype=torch.float64, device="cuda:0")
    mon = np.asarray(entries, dtype=np.int32)
    L = pkg._ffi.lib()
    pkg._ffi.check(L.amwg_sample_device(s._handle, n, 1, mon.ctypes.data_as(C.POINTER(C.c_int32)), len(entries), block.data_ptr()))
    calls = []

    class Timed(CudaBlockReducer):
        def autocov(self, block, thresholds, live, lag0, n_lags):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            out = super().autocov(block, thresholds, live, lag0, n_lags)
            b.record()
            b.synchronize()
            calls.append((len(live), lag0, n_lags, a.elapsed_time(b)))
            return out

    red = Timed(0)
    _, _, _, q = summarise_block(red, block, rows, chains, [0.05, 0.95], False)
    summarise_ess(red, block, rows, chains, q[0], q[1], False)           # warm-up
    calls.clear()
    _, _, tiles = summarise_ess(red, block, rows, chains, q[0], q[1], False)
    h = rows // 2
    dfma = sum(nl * 2 * chains * sum(max(h - (lag0 + j), 0) for j in range(nlag)) for nl, lag0, nlag, _ in calls)
    hbm = sum(nl * 2 * (2 * h) * chains * 8 for nl, _, _, _ in calls)  # the means pass reads the halves; the lag pass again
    ms = sum(c[3] for c in calls)
    tf, pk_ms = C.c_double(0), C.c_double(0)
    pkg._ffi.check(L.amwg_peak_fp64(0, 3, C.byref(tf), C.byref(pk_ms)))
    bound_fp64 = 2 * dfma / (tf.value * 1e12) * 1e3
    bound_hbm = hbm / HBM_BYTES_PER_S * 1e3
    del block
    res = {"config": k, "chains": chains, "n": n, "entries": cfg.n_entries, "rounds": rounds,
           "sample_summary_ms": spread(t["plain"]), "sample_summary_ess_ms": spread(t["ess"]),
           "ess_added_fraction": statistics.median(t["ess"]) / statistics.median(t["plain"]) - 1,
           "ess_reduction": {"autocov_calls": len(calls), "autocov_ms_cuda_events": ms,
                             "tiles_per_entry": {"mean": tiles[0].tolist() if cfg.n_entries <= 2 else
                                                 {"min": int(tiles[0].min()), "max": int(tiles[0].max())},
                                                 "q05_indicator": {"min": int(tiles[1].min()), "max": int(tiles[1].max())},
                                                 "q95_indicator": {"min": int(tiles[2].min()), "max": int(tiles[2].max())}},
                             "dfma": dfma, "hbm_bytes": hbm, "fp64_peak_tflops_measured": tf.value,
                             "bound_ms": {"fp64": bound_fp64, "hbm": bound_hbm},
                             "share_of_bound": max(bound_fp64, bound_hbm) / ms if ms > 0 else None,
                             "bound_by": "fp64" if bound_fp64 >= bound_hbm else "hbm"}}
    res["draws_per_ess"] = {name: (np.asarray(v["n_draws"]) / np.asarray(v["ess"])).tolist() for name, v in last.items()} \
        if cfg.n_entries <= 2 else {name: {"min": float(np.min(v["n_draws"] / np.asarray(v["ess"]))),
                                           "max": float(np.max(v["n_draws"] / np.asarray(v["ess"])))} for name, v in last.items()}
    res["ess"] = {name: np.asarray(v["ess"]).tolist() for name, v in last.items()} if cfg.n_entries <= 2 else None
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("outdir")
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--cases", nargs="+", default=list(CASES), choices=list(CASES))
    args = ap.parse_args()
    os.makedirs(args.outdir, exist_ok=True)
    jit_cache = None
    if "AMWG_JIT_CACHE" not in os.environ:            # by default the library caches cubins next to itself, in the source tree
        jit_cache = tempfile.TemporaryDirectory()
        os.environ["AMWG_JIT_CACHE"] = jit_cache.name
    import __graft_entry__ as graft
    import bench
    pkg = graft.load_package()
    out = {"gpu": card(), "note": "wall times: host clock around sample_summary with a device synchronise; rounds alternate the "
                                  "order of the two settings", "cases": {}}
    for name in args.cases:
        k, chains, n = CASES[name]
        out["cases"][name] = run_case(pkg, bench, k, chains, n, args.rounds)
        print(name, json.dumps(out["cases"][name]), flush=True)
    out["gpu_after"] = card()
    with open(os.path.join(args.outdir, "summary_ess.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"gpu": out["gpu"], "added": {k: v["ess_added_fraction"] for k, v in out["cases"].items()}}))


if __name__ == "__main__":
    main()
