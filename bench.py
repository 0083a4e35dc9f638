#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric, posterior draws/sec (chains x iters), on the BASELINE configs.

    default   config 2 (the headline): Normal(mu,sigma), N=1024 synthetic data, 2^20 chains per GPU (weak scaling)
    --config  3 | 4 | 5: the other BASELINE configs at their stated per-GPU size (2^20 / 2^16 / 2^19 chains per GPU;
              config 4 is quoted on 4 GPUs, config 5 on 8), same JSON line, same legs
    step      one `sample(ITERS)` call, adaptation running, after a burn-in done in setup; `value` = kernel path with the
              samples left in HBM (amwg_sample_device), `e2e` = the public API call mcmc.AmwgSampler.sample() returning host
              arrays (D2H inside the timed region); at N > 1 also the NCCL gather legs (gather = "all" and "root")
    parity    every run carries an in-run parity probe on the full-size data: chains {0, 1, C-1} stepped by the CPU oracle
              and by a `faithful` device handle, compared bit for bit; and a fast-vs-faithful two-sample KS
    --impl reference   the CPU restatement of mcmc.js (oracle/, Node is absent) on all host cores, one C call per step.
    --dump-outputs DIR   after the timed steps, the draws of the last one as DIR/<name>.npy (see dump_outputs)

One JSON line on stdout (rank 0). Nothing is written into the source tree, which may be read-only: no bytecode, and the
cubins of the run-time specialised sweep are cached in a temporary directory.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
import __graft_entry__ as graft  # noqa: E402

METRIC = "posterior draws/sec (chains x iters) Normal(mu,sigma) N=1024 at 1/2/4/8 B200"
FP64_NOMINAL_TFLOPS = 37.0       # B200 non-tensor fp64 (HGX B200 datasheet: 296 TF / 8 GPUs); only used when the measurement fails
PARAMS = {"mu": {"type": "real"}, "sigma": {"type": "real", "lower": 0}}
N_DATA = 1024
CHAINS_PER_GPU = 1 << 20


def config2_data():
    return np.random.default_rng(1024).normal(184.5, 4.5, N_DATA)


# ---------------------------------------------------------------------------------------------------------------------
# The BASELINE configs (BASELINE.json configs[1..4], SURVEY.md 8(d)): model, synthetic data, sizes, algorithmic work per draw
# ---------------------------------------------------------------------------------------------------------------------
class Config:
    def __init__(self, k, ld, mcmc):
        self.k = k
        if k == 2:
            self.workload = "config 2: Normal(mu,sigma), N=1024 synthetic, 2^20 chains per GPU"
            self.metric = METRIC
            self.params = PARAMS
            x = config2_data()
            self.data, self.oracle_model, self.oracle_data = x.tolist(), "norm_readme", x
            self.chains, self.iters, self.burn, self.gpus_quoted = 1 << 20, 100, 1000, 1

            def log_post(state, data):                    # README.md:26-36
                log_post = 0
                log_post += ld.norm(state.mu, 0, 100)
                log_post += ld.unif(state.sigma, 0, 100)
                for i in range(len(data)):
                    log_post += ld.norm(data[i], state.mu, state.sigma)
                return log_post
            self.log_post = log_post
            # BASELINE.md section 4: 2 components x 1024 points x 3 flop; 16 B sample write + ~1.4 B amortised state/log-SD/counters
            self.flop_per_draw, self.hbm_bytes_per_draw = 6144.0, 17.4
            self.flop_note = "2 components x 1 likelihood evaluation x 1024 points x 3 flop (BASELINE.md section 4)"
            self.cpu_draws, self.probe_sweeps, self.ks_chains, self.ks_sweeps = 2000, 30, 4096, 400
        elif k == 3:
            self.workload = "config 3: Beta-Bernoulli (theta~beta(2,2), y~bern) N=256 + binary indicator m, 2^20 chains per GPU"
            self.metric = "posterior draws/sec (chains x iters) Beta-Bernoulli N=256 + binary indicator"
            self.params = {"theta": {"type": "real", "lower": 0, "upper": 1}, "m": {"type": "binary"}}
            y = (np.random.default_rng(256).random(256) < 0.7).astype(np.float64)
            self.data, self.oracle_model, self.oracle_data = {"x": y.tolist()}, "spike_bern", {"x": y}
            self.chains, self.iters, self.burn, self.gpus_quoted = 1 << 20, 100, 500, 1

            def log_post(state, d):                       # README.md:149-164 + indicator (pattern of tests/test_data.js:154-171)
                lp = 0
                lp += ld.beta(state.theta, 2, 2)
                lp += ld.bern(state.m, 0.5)
                for i in range(len(d.x)):
                    lp += ld.bern(d.x[i], mcmc.where(state.m == 0, 0.5, state.theta))
                return lp
            self.log_post = log_post
            self.flop_per_draw, self.hbm_bytes_per_draw = 512.0, 17.4
            self.flop_note = "2 steps x 256 sequential adds (the bit-faithful Bernoulli sum; SURVEY 8(d) config 3)"
            self.cpu_draws, self.probe_sweeps, self.ks_chains, self.ks_sweeps = 5000, 60, 4096, 300
        elif k == 4:
            J, per = 64, 1024
            self.workload = "config 4: hierarchical Normal, mu dim=[64] + sigma, N=65536 (64 groups x 1024), 2^16 chains per GPU (2^18 on 4 GPUs)"
            self.metric = "posterior draws/sec (chains x iters) hierarchical Normal D=65 N=65536"
            self.params = {"mu": {"type": "real", "dim": [J]}, "sigma": {"type": "real", "lower": 0}}
            g = np.repeat(np.arange(J), per)
            mu_true = np.random.default_rng(64).normal(100, 20, J)
            yy = mu_true[g] + np.random.default_rng(65).normal(0, 5, J * per)
            self.data = {"y": yy, "g": g.astype(np.float64)}
            self.oracle_model, self.oracle_data = "hier_norm", {"y": yy, "g": g}
            self.chains, self.iters, self.burn, self.gpus_quoted = 1 << 16, 10, 100, 4

            def log_post(state, d):                       # SURVEY 8(d).4
                lp = 0
                for j in range(J):
                    lp += ld.norm(state.mu[j], 0, 100)
                lp += ld.unif(state.sigma, 0, 100)
                for i in range(len(d.y)):
                    lp += ld.norm(d.y[i], state.mu[d.g[i]], state.sigma)
                return lp
            self.log_post = log_post
            self.flop_per_draw = 131072.0 * 3
            self.hbm_bytes_per_draw = 65 * 8 + 65 * (16 + 16 + 4) / 50.0
            self.flop_note = "SURVEY 8(d): minimal 64 x 1024 + 65536 = 131072 point-terms x 3 flop (the kernel caches each group's sum of squares: 65536 point-terms per sweep)"
            self.cpu_draws, self.probe_sweeps, self.ks_chains, self.ks_sweeps = 3, 1, 512, 5
        elif k == 5:
            K, n = 8, 1000000
            self.workload = "config 5: Poisson regression, 8 real coefs, N=1e6, 2^19 chains per GPU (2^22 on 8 GPUs)"
            self.metric = "posterior draws/sec (chains x iters) Poisson regression K=8 N=1e6"
            self.params = {"beta": {"type": "real", "dim": [K]}}
            X = np.column_stack([np.ones(n), np.random.default_rng(8).normal(0, 0.5, (n, K - 1))])
            beta_true = np.random.default_rng(9).normal(0, 0.3, K)
            yc = np.random.default_rng(10).poisson(np.exp(X @ beta_true)).astype(np.float64)
            self.data = {"y": yc, "X": X}
            self.oracle_model, self.oracle_data = "pois_reg", {"y": yc, "X": X}
            self.chains, self.iters, self.burn, self.gpus_quoted = 1 << 19, 1, 1, 8

            def log_post(state, d):                       # SURVEY 8(d).5
                lp = 0
                for k_ in range(K):
                    lp += ld.norm(state.beta[k_], 0, 10)
                for i in mcmc.points(len(d.y)):
                    eta = 0
                    for k_ in range(K):
                        eta += d.X[i][k_] * state.beta[k_]
                    lp += ld.pois(d.y[i], mcmc.Math.exp(eta))
                return lp
            self.log_post = log_post
            self.flop_per_draw = 8 * 1e6 * 20.0
            self.hbm_bytes_per_draw = 8 * 8 + 8 * (16 + 16 + 4) / 50.0
            self.flop_note = "SURVEY 8(d): 8 steps x 1e6 points x (8 FMA + exp + 2 FMA ~ 20 flop)"
            self.cpu_draws, self.probe_sweeps, self.ks_chains, self.ks_sweeps = 1, 1, 0, 0
        else:
            raise SystemExit(f"bench.py: no such config {k}")
        self.n_entries = sum(int(np.prod(p.get("dim", [1]))) for p in self.params.values())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region: one `nvidia-smi -lms 100` process started before the region and
    stopped after it (a fresh nvidia-smi per sample takes longer than a whole timed step)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        rows = []
        if self.proc is not None:
            try:
                self.proc.terminate()
                out, _ = self.proc.communicate(timeout=5)
                rows = [[f.strip() for f in ln.split(",")] for ln in out.strip().splitlines() if ln.strip()]
            except Exception:
                try:
                    self.proc.kill()
                except Exception:
                    pass
        if not rows:                                  # the region was shorter than nvidia-smi's start-up: one sample right after it
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=10).stdout.strip()
                rows = [[f.strip() for f in out.split(",")]] if out else []
            except Exception:
                rows = []

        def num(v):
            try:
                return float(v)
            except ValueError:
                return None
        sm = [num(r[0]) for r in rows if r and num(r[0]) is not None]
        mx = [num(r[1]) for r in rows if len(r) > 1 and num(r[1]) is not None]
        pw = [num(r[2]) for r in rows if len(r) > 2 and num(r[2]) is not None]
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(rows)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(cfg_k: int, chains: int):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the dominant kernel, as scripts/ncu_traffic.py wrote it into
    profiles/ from an `ncu --set full` capture of THIS bench command (the build it was taken on is recorded beside it)."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return None, None
    try:
        with open(p) as f:
            d = json.load(f)
        e = d.get(f"config{cfg_k}")
        if e and int(e.get("chains", -1)) == int(chains):
            return e, "profiles/ncu_traffic.json (%s)" % e.get("source", "?")
    except Exception:
        try:                                         # cgroup v1
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
                cores = max(1, min(visible, int(quota + 0.999)))
        except Exception:
            pass
    return None, None


# ---------------------------------------------------------------------------------------------------------------------
def cpu_port_draws_per_sec(orc, cfg: Config, seconds_target: float = 12.0):
    """Oracle (CPU restatement of mcmc.js, 2 evals per step like the reference) on ONE core, bounded sample of the workload."""
    n0 = cfg.cpu_draws
    t = orc.time_model(cfg.oracle_model, cfg.oracle_data, cfg.params, chains=1, burn=0, sample=n0)
    n = int(max(n0, min(100 * n0, n0 * seconds_target / max(t, 1e-6))))
    if n > n0:
        t = orc.time_model(cfg.oracle_model, cfg.oracle_data, cfg.params, chains=1, burn=0, sample=n)
    return n / t, f"1 chain x {n} draws of {cfg.workload.split(',')[0]}, single thread"


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path = the oracle port (Node is absent) on all host cores.
    One step = ONE C call that runs `cores` independent chains on `cores` pthreads (orc_run_chains_mt): no per-step Python."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    orc = graft.load_oracle()
    pkg = graft.load_package()
    cfg = Config(args.config, pkg.ld, pkg.mcmc)
    visible = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    cores, quota = visible, None
    try:                                             # a container may see 128 CPUs and be allowed a fraction of them (cgroup v2 cpu.max)
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = float(q) / float(per)
            cores = max(1, min(visible, int(quota + 0.999)))
    except Exception:
        pass
    # per-thread work sized from a single-core probe so that one step is about 2.5 s
    t1 = orc.time_model(cfg.oracle_model, cfg.oracle_data, cfg.params, chains=1, burn=0, sample=cfg.cpu_draws)
    one_core = cfg.cpu_draws / t1
    per_thread = int(max(1, round(one_core * 2.5)))

    def step():
        return orc.time_model(cfg.oracle_model, cfg.oracle_data, cfg.params, chains=cores, burn=0, sample=per_thread, threads=cores)

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    value = cores * per_thread * args.steps / dt
    sample = f"{cores} pthreads x 1 chain x {per_thread} draws per step (one C call per step)"
    line = {"impl": "reference", "metric": cfg.metric, "value": value, "unit": "draws/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": cfg.workload, "note": "CPU restatement of mcmc.js (Node unavailable); independent chains are the only parallelism the reference admits"},
            "cpu_baseline": {"value": value, "unit": "draws/s", "cores": cores, "kind": "port", "sample": sample,
                             "single_core_draws_per_s": one_core, "parallel_efficiency": value / (one_core * cores),
                             "cpus_visible": visible, "cgroup_cpu_quota": quota},
            "e2e": {"value": value, "unit": "draws/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
def ks_2samp(a, b):
    a, b = np.sort(np.asarray(a, float).ravel()), np.sort(np.asarray(b, float).ravel())
    allv = np.concatenate([a, b])
    return float(np.max(np.abs(np.searchsorted(a, allv, side="right") / a.size - np.searchsorted(b, allv, side="right") / b.size)))


def parity_probe(cfg: Config, mcmc, orc, chains_total: int, device: int, seed: int):
    """In-run parity on the full-size data. (1) bit-exact: chains {0, 1, C-1} for a few sweeps, CPU oracle vs a `faithful` device
    handle (global chain ids select the Philox streams, so a 2-chain handle at first_chain=0 and a 1-chain handle at C-1 are those
    chains of the big run). (2) statistical: the production (fast) lowering vs the faithful one, two-sample KS over `ks_chains`
    chains after `ks_sweeps` sweeps from the common initial state (disjoint chain ids, so the samples are independent)."""
    out = {"sweeps": cfg.probe_sweeps, "chains": [0, 1, chains_total - 1]}
    ok = True
    t0 = time.perf_counter()
    for first, n in ((0, 2), (chains_total - 1, 1)):
        s = mcmc.AmwgSampler(cfg.params, cfg.log_post, cfg.data, {"chains": n, "first_chain": first, "seed": seed, "device": device, "faithful": True})
        got = s.sample(cfg.probe_sweeps + 1)
        s.close()
        ref = orc.run_model(cfg.oracle_model, cfg.oracle_data, cfg.params, chains=n, first_chain=first, seed=seed, sample=cfg.probe_sweeps + 1)
        for name in cfg.params:
            a, b = np.asarray(got[name], dtype=np.float64), np.asarray(ref[name], dtype=np.float64)
            ok = ok and a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))
    out["bit_exact_vs_oracle"] = bool(ok)
    out["bit_exact_seconds"] = round(time.perf_counter() - t0, 2)
    if cfg.ks_chains:
        t0 = time.perf_counter()
        name = next(iter(cfg.params))
        fast = mcmc.AmwgSampler(cfg.params, cfg.log_post, cfg.data, {"chains": cfg.ks_chains, "first_chain": 0, "seed": seed, "device": device})
        fast.burn(cfg.ks_sweeps)
        a = np.asarray(fast.state[name]).reshape(cfg.ks_chains, -1)[:, 0]
        fast.close()
        slow = mcmc.AmwgSampler(cfg.params, cfg.log_post, cfg.data, {"chains": cfg.ks_chains, "first_chain": 1 << 30, "seed": seed, "device": device, "faithful": True})
        slow.burn(cfg.ks_sweeps)
        b = np.asarray(slow.state[name]).reshape(cfg.ks_chains, -1)[:, 0]
        slow.close()
        d = ks_2samp(a, b)
        crit = 1.63 * np.sqrt(2.0 / cfg.ks_chains)             # two-sample KS, alpha = 0.01
        out.update({"ks_fast_vs_faithful": d, "ks_critical_1pct": float(crit), "ks_chains": cfg.ks_chains, "ks_sweeps": cfg.ks_sweeps,
                    "ks_entry": name + "[0]" if a.ndim else name, "ks_ok": bool(d < crit), "ks_seconds": round(time.perf_counter() - t0, 2)})
    return out


DUMP_BYTES = 32 << 20          # --dump-outputs writes at most this many bytes of draws


def dump_outputs(out_dir, sampler, cfg: Config, dev_out):
    """--dump-outputs: what the last timed step returned, dev_out = [iters, entries, chains] float64 draws in HBM, written as
    <name>.npy per parameter in the layout sample() returns ([iters, chains, *dim]). Above DUMP_BYTES a fixed seeded sample of the
    chains is kept (and of the rows, if one chain's rows alone exceed it), so that runs with the same arguments compare file for file."""
    import torch
    rows, E, chains = dev_out.shape
    rng = np.random.default_rng(0)
    budget = DUMP_BYTES // 8
    keep_rows = np.arange(rows) if rows * E <= budget else np.sort(rng.choice(rows, max(1, budget // E), replace=False))
    keep_chains = np.sort(rng.choice(chains, min(chains, budget // (keep_rows.size * E)), replace=False))
    sub = dev_out.index_select(0, torch.as_tensor(keep_rows, device=dev_out.device))
    sub = sub.index_select(2, torch.as_tensor(keep_chains, device=dev_out.device)).cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name in cfg.params:
        np.save(os.path.join(out_dir, name + ".npy"), sampler._shape_out(name, sub[:, sampler._entries(name), :]))


def run_ours(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the sampler has no CPU fallback")
    torch.cuda.set_device(local_rank)
    pkg = graft.load_package()
    mcmc, ld, ffi = pkg.mcmc, pkg.ld, pkg._ffi
    numa = pkg.parallel.bind_to_gpu_numa_node(local_rank) if world > 1 else None     # before any pinned allocation
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    L = ffi.lib()
    cfg = Config(args.config, ld, mcmc)
    chains = args.chains or cfg.chains
    iters = args.iters or cfg.iters
    burn = cfg.burn if args.burn is None else args.burn
    seed = 0

    jit_cache = None
    if "AMWG_JIT_CACHE" not in os.environ:            # by default the library caches cubins next to itself, in the source tree
        jit_cache = tempfile.TemporaryDirectory(prefix="amwg_jit_cache_")
        os.environ["AMWG_JIT_CACHE"] = jit_cache.name

    chains_total = chains * world
    t_create = time.perf_counter()
    sampler = mcmc.AmwgSampler(cfg.params, cfg.log_post, cfg.data,
                               {"chains": chains_total, "seed": seed, "device": local_rank, "distributed": world > 1, "gather": "none"})
    t_create = time.perf_counter() - t_create
    local = sampler.local_chains
    E = cfg.n_entries
    mon = np.arange(E, dtype=np.int32)
    monp = mon.ctypes.data_as(C.POINTER(C.c_int32))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- N > 1: the gathered block holds the right VALUES (not just the right shape): before anything else has advanced the
    # chains, sample a few rows with gather="all" and compare another rank's shard with a fresh 64-chain single handle bit for bit
    gather_check = None
    if world > 1:
        sampler.gather = "all"
        rows_chk = 3
        blk = sampler.sample(rows_chk)
        if rank == 0:
            first_other = pkg.parallel.shard_bounds(chains_total, world - 1, world)[0]
            nchk = min(64, chains)
            lone = mcmc.AmwgSampler(cfg.params, cfg.log_post, cfg.data, {"chains": nchk, "first_chain": first_other, "seed": seed, "device": local_rank})
            ref = lone.sample(rows_chk)
            lone.close()
            okc = True
            for name in cfg.params:
                a = np.asarray(blk[name])[:, first_other:first_other + nchk]
                b = np.asarray(ref[name])
                okc = okc and a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))
            gather_check = {"bit_equal_to_single_handle": bool(okc), "rank_checked": world - 1, "chains_checked": nchk, "rows": rows_chk}
        del blk
        sampler.gather = "none"

    sampler.burn(burn)
    dev_out = torch.empty((iters, E, local), dtype=torch.float64, device=f"cuda:{local_rank}")

    def step_device():
        ffi.check(L.amwg_sample_device(sampler._handle, iters, 1, monp, E, dev_out.data_ptr()))
        return sampler.last_sweep_kernel_ms()

    # ---- value: device-resident --------------------------------------------------------------------------------
    for _ in range(args.warmup):
        step_device()
    clocks = ClockSampler(local_rank) if rank == 0 else None
    if clocks:
        clocks.start()
        time.sleep(0.3)                               # let nvidia-smi come up: its samples then fall inside the timed region
    launches0 = sampler.kernel_launches()
    barrier()
    t0 = time.perf_counter()
    kernel_ms = 0.0
    for _ in range(args.steps):
        kernel_ms += step_device()
    barrier()
    dt = time.perf_counter() - t0
    launches = sampler.kernel_launches() - launches0
    clk = clocks.stop() if clocks else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, sampler, cfg, dev_out)
    del dev_out

    # ---- the measured fp64 roof, same process, same clocks ------------------------------------------------------------
    tf, ms_pk = C.c_double(0.0), C.c_double(0.0)
    fp64_peak, fp64_src = FP64_NOMINAL_TFLOPS, "nominal (measurement failed)"
    if L.amwg_peak_fp64(local_rank, 3, C.byref(tf), C.byref(ms_pk)) == 0 and tf.value > 0:
        fp64_peak, fp64_src = tf.value, "measured in this run (amwg_peak_fp64: DFMA chains on every SM, best of 3, %.1f ms)" % ms_pk.value

    # ---- e2e: public API, host arrays ---------------------------------------------------------------------------
    # N > 1: "none" = every process receives the draws of its own chains in its own host memory (one PCIe link per GPU, the way a
    # one-process-per-GPU job consumes them); "all" = north_star's collective (NCCL all-gather over NVLink, every rank returns all
    # chains); "root" = rank 0 alone ends up with all chains.
    e2e_steps = max(1, min(args.steps, 5))

    def e2e_leg(mode, steps, its):
        sampler.gather = mode
        w1 = sampler.sample(its)               # warm-up: two live results = the two pinned buffers the loop alternates between
        w2 = sampler.sample(its)
        del w1, w2
        barrier()
        t = time.perf_counter()
        for _ in range(steps):
            draws = sampler.sample(its)
        barrier()
        dt_leg = time.perf_counter() - t
        want = chains_total if (mode == "all" or (mode == "root" and rank == 0)) else local
        first = next(iter(cfg.params))
        assert np.asarray(draws[first]).shape[:2] == (its, want), (np.asarray(draws[first]).shape, its, want)
        del draws
        return dt_leg

    dt_e2e = e2e_leg("none", e2e_steps, iters)
    gather_steps = max(1, min(args.steps, 5))
    # the gathered result is chains_total wide on every rank ("all"): bound it to ~2 GB of pinned host memory per buffer
    iters_g = max(1, min(iters, int(2e9 // (E * chains_total * 8))))
    dt_all = e2e_leg("all", gather_steps, iters_g) if world > 1 else 0.0
    dt_root = e2e_leg("root", gather_steps, iters_g) if world > 1 else 0.0
    sampler.gather = "none"

    # ---- e2e with the summary formed on the device (SURVEY 8(f).3): same sweeps, only mean/sd/quantiles/R-hat leave the GPUs
    first_name = next(iter(cfg.params))
    dt_sum, sum_ms, summ = 0.0, [], None
    if args.config != 5:
        summ = sampler.sample_summary(iters)       # warm-up
        barrier()
        t2 = time.perf_counter()
        for _ in range(e2e_steps):
            t3 = time.perf_counter()
            summ = sampler.sample_summary(iters)
            sum_ms.append(round(1e3 * (time.perf_counter() - t3), 2))
        barrier()
        dt_sum = time.perf_counter() - t2

    times = torch.tensor([dt, dt_e2e, kernel_ms, dt_sum, dt_root, dt_all], dtype=torch.float64, device=f"cuda:{local_rank}")
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    dt, dt_e2e, kernel_ms, dt_sum, dt_root, dt_all = [float(v) for v in times.tolist()]
    info = sampler.program_summary() + ["sweep kernel: " + sampler.jit_status()[1]]
    sampler.close()

    if rank == 0:
        draws_per_step = chains_total * iters
        value = draws_per_step * args.steps / dt
        e2e = draws_per_step * e2e_steps / dt_e2e
        # roofline of the dominant kernel, per GPU, from the library's CUDA-event time on its launch stream
        kern_draws_per_s = (local * iters * args.steps) / (kernel_ms * 1e-3)
        hbm_peak, how = measured_peaks()
        ach_gbs = kern_draws_per_s * cfg.hbm_bytes_per_draw / 1e9
        ach_tf = kern_draws_per_s * cfg.flop_per_draw / 1e12
        traffic, traffic_src = ncu_traffic(cfg.k, local)
        sweeps_per_launch = min(iters, 50)
        d2h = int(iters * E * chains_total * 8)
        line = {
            "metric": cfg.metric, "value": value, "unit": "draws/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": cfg.workload, "chains_per_gpu": local, "chains_total": chains_total, "iters_per_step": iters,
                       "burn_in_setup": burn, "adapting": True, "gpus_quoted_in_BASELINE": cfg.gpus_quoted,
                       "parallelism": f"chains sharded x{world}, no data-path collective",
                       "l2": "every step writes its samples (iters*entries*chains*8 B = %.2f GB per GPU) and re-reads per-chain state; "
                             "inputs + outputs exceed the 126 MB L2" % (iters * E * local * 8 / 1e9),
                       "lowering": info[-1] if info else None, "create_seconds": round(t_create, 2)},
            "roofline": {"bound": "hbm", "achieved": ach_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": ach_gbs / hbm_peak,
                         "traffic": (traffic or {}).get("dram_bytes_per_launch"), "traffic_source": traffic_src,
                         "traffic_kernel": (traffic or {}).get("kernel"), "traffic_sweeps_per_launch": (traffic or {}).get("sweeps_per_launch"),
                         "algorithmic_bytes_per_launch": cfg.hbm_bytes_per_draw * sweeps_per_launch * local,
                         "peak_source": how, "algorithmic_bytes_per_draw": cfg.hbm_bytes_per_draw,
                         "note": "north_star names HBM; with the N-point sum fused in-kernel the binding roof is the fp64 pipe, see roofline_fp64"},
            "roofline_fp64": {"bound": "fp64-issue", "achieved": ach_tf, "peak": fp64_peak, "unit": "TFLOP/s",
                              "frac": ach_tf / fp64_peak, "peak_source": fp64_src, "nominal_peak": FP64_NOMINAL_TFLOPS,
                              "algorithmic_flop_per_draw": cfg.flop_per_draw, "flop_note": cfg.flop_note,
                              "kernel_ms_per_step": kernel_ms / args.steps},
            "e2e": {"value": e2e, "unit": "draws/s", "h2d_bytes_per_step": int(mon.nbytes),
                    "d2h_bytes_per_step": d2h, "steps": e2e_steps, "d2h_gbs_aggregate": d2h * e2e_steps / dt_e2e / 1e9,
                    "numa": numa,
                    "note": "mcmc.AmwgSampler.sample(): pinned host buffer, D2H overlapped with the sweeps"
                            + ("; every rank copies the draws of its own chains to its own host memory (gather=\"none\")" if world > 1 else "")},
            "e2e_gather_all": ({"value": chains_total * iters_g * gather_steps / dt_all, "unit": "draws/s", "steps": gather_steps, "iters_per_step": iters_g,
                                "note": "gather=\"all\" (north_star's collective): NCCL all-gather of the shards over NVLink, one collective per "
                                        "chunk, every rank copies ALL chains to its host"} if dt_all > 0 else None),
            "e2e_gather_root": ({"value": chains_total * iters_g * gather_steps / dt_root, "unit": "draws/s", "steps": gather_steps, "iters_per_step": iters_g,
                                 "note": "gather=\"root\": NCCL gather of the shards to rank 0, one host copy of all draws over rank 0's PCIe link"} if dt_root > 0 else None),
            "gather_check": gather_check,
            "gpu_launches": int(launches), "clocks": clk,
        }
        if summ is not None:
            s0 = summ[first_name]
            pick = (lambda v: float(np.asarray(v).reshape(-1)[0]))
            line["e2e_summary"] = {"value": draws_per_step * e2e_steps / dt_sum, "unit": "draws/s", "steps": e2e_steps,
                                   "ms_per_call_rank0": sum_ms,
                                   "median_call_value": draws_per_step / (1e-3 * sorted(sum_ms)[len(sum_ms) // 2]),
                                   first_name: {"mean": pick(s0["mean"]), "sd": pick(s0["sd"]), "rhat": pick(s0["rhat"])},
                                   "note": "mcmc.AmwgSampler.sample_summary(): the draws stay in HBM; pooled mean/sd, exact quantiles (radix "
                                           "select) and R-hat over all chains x iterations come back"
                                           + ("; shards combined by an all-gather of moment records and an all-reduce of digit counts (NCCL)" if world > 1 else "")}
        if not args.no_cpu:
            orc = graft.load_oracle()
            if world == 1:
                v, sample = cpu_port_draws_per_sec(orc, cfg)
                line["cpu_baseline"] = {"value": v, "unit": "draws/s", "cores": 1, "kind": "port", "sample": sample,
                                        "published_reference": "README.md:252: ~4e4 draws/s at N=1000 (author's machine, 2015)"}
            # The probe steps `faithful` handles (the reference's arithmetic, term by term) on the FULL-SIZE data. On config 5 that is
            # 8 x 1e6 interpreted point-terms per sweep for a single warp (minutes): asked for with --probe, recorded in profiles/.
            # At N > 1 the other ranks would idle behind rank 0: the probe belongs to the single-GPU run of the same config.
            want_probe = args.probe or (not args.no_probe and world == 1 and cfg.k != 5)
            if want_probe:
                line["parity_probe"] = parity_probe(cfg, mcmc, orc, chains_total, local_rank, seed)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5], help="BASELINE config (default: 2, the headline metric)")
    ap.add_argument("--chains", type=int, default=0, help="chains per GPU (default: the config's BASELINE size)")
    ap.add_argument("--iters", type=int, default=0, help="sweeps per step (default: per config)")
    ap.add_argument("--burn", type=int, default=None, help="burn-in sweeps done in setup (untimed)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg and the parity probe")
    ap.add_argument("--no-probe", action="store_true", help="skip the in-run parity probe")
    ap.add_argument("--probe", action="store_true", help="force the in-run parity probe (default: single-GPU runs of configs 2-4)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the draws of the last timed step as DIR/<name>.npy (float64; rank 0's chains, a fixed sample above 32 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU sampler (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
