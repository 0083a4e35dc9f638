#!/usr/bin/env python3
"""A/B of the statistics sweep's step-phase switches: bench.py with AMWG_JIT_MERGE_STEPS and AMWG_JIT_ACCEPT_SCREEN all off and
all on, alternating (the order flips every round), for configs 2 and 4 on one GPU.

    python scripts/ab_stat_sweep.py OUTDIR [--rounds 3] [--configs 2 4] [--steps 30] [--warmup 3]

Writes every bench line and a summary to OUTDIR (nothing into the source tree). The draws each run dumps go to a temporary
directory that is deleted once hashed; every .npy file must be byte-identical across all runs of a config. Prints the median and
spread (min .. max) of `value` and `roofline_fp64.kernel_ms_per_step` per setting. Exit code 1 if the draws differ or a run fails."""
import argparse
import hashlib
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SWITCHES = ("AMWG_JIT_MERGE_STEPS", "AMWG_JIT_ACCEPT_SCREEN")


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return "unknown (%s)" % e


def bench(cfg, setting, rnd, args):
    dump = os.path.join(args.tmp, "dump_c%d_%s_%d" % (cfg, setting, rnd))
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    for k in SWITCHES:
        env[k] = "1" if setting == "on" else "0"
    cmd = [sys.executable, "-B", os.path.join(ROOT, "bench.py"), "--gpus", "1", "--config", str(cfg), "--steps", str(args.steps),
           "--warmup", str(args.warmup), "--no-cpu", "--dump-outputs", dump]
    r = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=args.outdir)
    line = None
    for ln in r.stdout.splitlines():
        if ln.startswith("{"):
            try:
                line = json.loads(ln)
            except ValueError:
                pass
    if r.returncode != 0 or line is None:
        sys.stderr.write("config %d %s round %d failed (rc %d):\n%s\n" % (cfg, setting, rnd, r.returncode, r.stderr[-3000:]))
        return None, dump
    with open(os.path.join(args.outdir, "bench_c%d_%s_%d.json" % (cfg, setting, rnd)), "w") as f:
        f.write(json.dumps(line) + "\n")
    return line, dump


def digests(dump):
    out = {}
    for name in sorted(os.listdir(dump)) if os.path.isdir(dump) else []:
        if name.endswith(".npy"):
            with open(os.path.join(dump, name), "rb") as f:
                out[name] = hashlib.sha256(f.read()).hexdigest()
    shutil.rmtree(dump, ignore_errors=True)
    return out


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "n": len(xs)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--configs", type=int, nargs="+", default=[2, 4])
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    args.outdir = os.path.abspath(args.outdir)
    os.makedirs(args.outdir, exist_ok=True)
    args.tmp = tempfile.mkdtemp(prefix="ab_stat_sweep_")
    summary = {"card": card(), "switches": list(SWITCHES), "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds, "configs": {}}
    print("card (name, power limit, max SM clock):", summary["card"], flush=True)
    ok = True
    for cfg in args.configs:
        res = {"off": [], "on": []}
        ref_digest, identical = None, True
        for rnd in range(args.rounds):
            for setting in (("off", "on") if rnd % 2 == 0 else ("on", "off")):
                line, dump = bench(cfg, setting, rnd, args)
                if line is None:
                    ok = False
                    continue
                res[setting].append(line)
                d = digests(dump)
                if not d:
                    identical = False
                elif ref_digest is None:
                    ref_digest = d
                elif d != ref_digest:
                    identical = False
                print("config %d round %d %-3s value %.4e draws/s  kernel %.3f ms/step" %
                      (cfg, rnd, setting, line["value"], line["roofline_fp64"]["kernel_ms_per_step"]), flush=True)
        c = {"draws_identical": identical, "sha256": ref_digest or {}}
        for setting in ("off", "on"):
            if res[setting]:
                c[setting] = {"value": spread([l["value"] for l in res[setting]]),
                              "kernel_ms_per_step": spread([l["roofline_fp64"]["kernel_ms_per_step"] for l in res[setting]])}
        if "off" in c and "on" in c:
            c["speedup_median_value"] = c["on"]["value"]["median"] / c["off"]["value"]["median"]
            c["speedup_median_kernel"] = c["off"]["kernel_ms_per_step"]["median"] / c["on"]["kernel_ms_per_step"]["median"]
            c["spreads_overlap"] = not (c["on"]["value"]["min"] > c["off"]["value"]["max"] or c["off"]["value"]["min"] > c["on"]["value"]["max"])
        ok = ok and identical
        summary["configs"][str(cfg)] = c
        print(json.dumps({"config": cfg, **c}, indent=1), flush=True)
    shutil.rmtree(args.tmp, ignore_errors=True)
    with open(os.path.join(args.outdir, "ab_summary.json"), "w") as f:
        json.dump(summary, f, indent=1)
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
