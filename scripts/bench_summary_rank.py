#!/usr/bin/env python3
"""Cost of the rank-normalised diagnostics in `sample_summary`: `sample_summary(n)` and `sample_summary(n, rank=True)`,
alternating, for bench.py's config 2 (2^20 chains, n = 100 and n = 1000) and config 4 (2^16 chains, n = 200).

    python scripts/bench_summary_rank.py OUTDIR [--rounds 4] [--cases c2n100 c2n1000 c4n200]
    torchrun --nproc_per_node 2 scripts/bench_summary_rank.py OUTDIR --cases c2n100

Writes OUTDIR/summary_rank.json (OUTDIR/summary_rank_2gpu.json under torchrun; nothing into the source tree). Per case: median and
spread (min .. max) of each setting's wall time; the rank normalisation alone on a block of the same shape, with CUDA events
around every amwg_summary_rank_sort call; the sort passes run and skipped; the bytes those passes move and their time at
7.7 TB/s. The card's name, power limit and max SM clock are read with nvidia-smi --query-gpu. Under torchrun every rank runs the
distributed sampler, and the script asserts that both ranks return identical bits and that they match a single-GPU handle over
the same chains to rtol 1e-12 (with fewer GPUs than ranks, the ranks share the GPUs and the collectives go over gloo)."""
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
RANK_KEYS = ("rhat_bulk", "rhat_folded", "rhat_rank", "ess_bulk")


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return "unknown (%s)" % e


def spread(v):
    return {"median": statistics.median(v), "min": min(v), "max": max(v), "runs": v}


def sort_alone(pkg, s, cfg, chains, n):
    """the rank normalisation (bulk and folded) alone on a block left in HBM by amwg_sample_device, sorts timed with CUDA events"""
    import torch
    from bayes_js_b200.summary import CudaBlockReducer, rank_normalise, summarise_block
    entries = list(range(cfg.n_entries))
    block = torch.empty((n, len(entries), chains), dtype=torch.float64, device="cuda:0")
    mon = np.asarray(entries, dtype=np.int32)
    L = pkg._ffi.lib()
    pkg._ffi.check(L.amwg_sample_device(s._handle, n, 1, mon.ctypes.data_as(C.POINTER(C.c_int32)), len(entries), block.data_ptr()))
    sorts = []
    red = CudaBlockReducer(0)
    real_lib = red.L

    def timed_sort(*args):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        rc = real_lib.amwg_summary_rank_sort(*args)
        b.record()
        b.synchronize()
        sorts.append((int(args[3]), args[6][0], args[6][1], a.elapsed_time(b)))
        return rc

    class Lib:                                                  # the library with the sort timed, every other call as is
        def __getattr__(self, name):
            return timed_sort if name == "amwg_summary_rank_sort" else getattr(real_lib, name)

    red.L = Lib()
    middle = [n * chains // 2 - 1, n * chains // 2] if n * chains % 2 == 0 else [n * chains // 2]
    ost = summarise_block(red, block, n, chains, [], False, middle)[4]
    med = ost[0] if len(middle) == 1 else (ost[0] + ost[1]) / 2
    rank_normalise(red, block, n, chains, None, False)         # warm-up
    sorts.clear()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    z, _ = rank_normalise(red, block, n, chains, None, False)
    rank_normalise(red, block, n, chains, med, False, out=z)
    torch.cuda.synchronize()
    wall = 1e3 * (time.perf_counter() - t0)
    del z, block
    # per pass: the count kernel reads the keys (8 B), the scatter reads and writes key + payload (2 x 12 B); one histogram read
    hbm = sum(k * (8 + run * (8 + 24)) for k, run, _, _ in sorts)
    ms = sum(c[3] for c in sorts)
    return {"sorts": len(sorts), "sort_ms_cuda_events": ms, "passes_run": sum(c[1] for c in sorts), "passes_skipped": sum(c[2] for c in sorts),
            "keys_per_sort": sorts[0][0] if sorts else 0, "sort_hbm_bytes": hbm, "sort_bound_ms_hbm": hbm / HBM_BYTES_PER_S * 1e3,
            "sort_share_of_hbm_bound": (hbm / HBM_BYTES_PER_S * 1e3) / ms if ms > 0 else None,
            "rank_normalise_wall_ms": wall}


def run_case(pkg, bench, k, chains, n, rounds):
    import torch
    cfg = bench.Config(k, pkg.ld, pkg.mcmc)
    s = pkg.mcmc.AmwgSampler(cfg.params, cfg.log_post, cfg.data, {"chains": chains, "seed": 1, "device": 0})
    s.burn(cfg.burn)
    s.sample_summary(n)                                   # warm-up of every shape the timed runs use
    s.sample_summary(n, rank=True)
    t = {"plain": [], "rank": []}
    last = None
    for r in range(rounds):
        for setting in (("plain", "rank") if r % 2 == 0 else ("rank", "plain")):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = s.sample_summary(n, rank=(setting == "rank"))
            torch.cuda.synchronize()
            t[setting].append(1e3 * (time.perf_counter() - t0))
            if setting == "rank":
                last = out
    res = {"config": k, "chains": chains, "n": n, "entries": cfg.n_entries, "rounds": rounds,
           "sample_summary_ms": spread(t["plain"]), "sample_summary_rank_ms": spread(t["rank"]),
           "rank_added_fraction": statistics.median(t["rank"]) / statistics.median(t["plain"]) - 1,
           "rank_alone": sort_alone(pkg, s, cfg, chains, n)}
    if cfg.n_entries <= 2:
        res["values"] = {name: {key: float(v[key]) for key in RANK_KEYS + ("rhat",)} for name, v in last.items()}
    else:
        res["values"] = {name: {key: [float(np.min(v[key])), float(np.max(v[key]))] for key in RANK_KEYS + ("rhat",)} for name, v in last.items()}
    return res


def run_distributed(pkg, bench, k, chains, n):
    """every rank: the distributed summary; rank 0 also a single-GPU handle over all chains. Asserts identical bits across ranks."""
    import torch
    import torch.distributed as dist
    cfg = bench.Config(k, pkg.ld, pkg.mcmc)
    opts = {"chains": chains, "seed": 1, "distributed": True, "device": torch.cuda.current_device()}
    s = pkg.mcmc.AmwgSampler(cfg.params, cfg.log_post, cfg.data, opts)
    s.burn(cfg.burn)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = s.sample_summary(n, rank=True)
    torch.cuda.synchronize()
    wall = 1e3 * (time.perf_counter() - t0)
    mine = np.concatenate([np.ravel(np.asarray(out[name][key], dtype=np.float64)) for name in sorted(out) for key in RANK_KEYS])
    t = torch.from_numpy(mine).cuda()
    every = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(every, t)
    same = all(np.array_equal(e.cpu().numpy().view(np.uint64), mine.view(np.uint64)) for e in every)
    res = {"world": dist.get_world_size(), "backend": dist.get_backend(), "gpus": torch.cuda.device_count(), "config": k, "chains": chains,
           "n": n, "wall_ms": wall, "ranks_bit_identical": same}
    if dist.get_rank() == 0:
        one = pkg.mcmc.AmwgSampler(cfg.params, cfg.log_post, cfg.data, {"chains": chains, "seed": 1, "device": 0})
        one.burn(cfg.burn)
        ref = one.sample_summary(n, rank=True)
        single = np.concatenate([np.ravel(np.asarray(ref[name][key], dtype=np.float64)) for name in sorted(ref) for key in RANK_KEYS])
        res["matches_single_gpu_rtol_1e-12"] = bool(np.allclose(mine, single, rtol=1e-12, atol=0, equal_nan=True))
        res["max_rel_diff_vs_single_gpu"] = float(np.nanmax(np.abs(mine - single) / np.abs(single)))
        assert res["matches_single_gpu_rtol_1e-12"], res
    assert same, res
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
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch
        import torch.distributed as dist
        # one GPU per rank over NCCL; with fewer GPUs than ranks the ranks share them and gloo carries the collectives (NCCL
        # refuses two ranks on one GPU): the same exchange and the same bits, not the same timing
        shared = torch.cuda.device_count() < int(os.environ["WORLD_SIZE"])
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")) % torch.cuda.device_count())
        dist.init_process_group("gloo" if shared else "nccl")
        try:
            out = {"gpu": card(), "cases": {}}
            for name in args.cases:
                k, chains, n = CASES[name]
                out["cases"][name] = run_distributed(pkg, bench, k, chains, n)
            if dist.get_rank() == 0:
                with open(os.path.join(args.outdir, "summary_rank_2gpu.json"), "w") as f:
                    json.dump(out, f, indent=1)
                print(json.dumps(out))
        finally:
            dist.destroy_process_group()
        return
    out = {"gpu": card(), "note": "wall times: host clock around sample_summary with a device synchronise; rounds alternate the "
                                  "order of the two settings", "cases": {}}
    for name in args.cases:
        k, chains, n = CASES[name]
        out["cases"][name] = run_case(pkg, bench, k, chains, n, args.rounds)
        print(name, json.dumps(out["cases"][name]), flush=True)
    out["gpu_after"] = card()
    with open(os.path.join(args.outdir, "summary_rank.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"gpu": out["gpu"], "added": {k: v["rank_added_fraction"] for k, v in out["cases"].items()}}))


if __name__ == "__main__":
    main()
