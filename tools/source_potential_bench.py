"""Throughput of a source potential (CudaPotential) against the built-in plugin it restates.

Workload: banana d = 50, Zig-Zag, grid_size = 10, analytic (JVP) derivative, 4096 chains x 1000 events, Philox draws,
no history (the kernel alone).  The built-in runs with PDMPFLUX_FORCE_GENERIC=1, i.e. on the same generic kernel the
source potential always uses.  The two alternate, 5 timed runs each after one warm-up each.  Also reports the cold
and warm (cached) NVRTC time per instantiation, and the card name and power limit read in the same process.

    python tools/source_potential_bench.py [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import pdmpflux_b200 as p  # noqa: E402
from test_source_potential_cpu import BANANA_SRC  # noqa: E402

D, CHAINS, EVENTS, REPS = 50, 4096, 1000, 5


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"unavailable ({e})"
    return q


def events_per_s(sampler, x0, v0, seed):
    ch = p.DeviceChains(sampler, x0, v0, seed=seed)
    ch.get_state()                      # synchronises: set-up done
    t0 = time.perf_counter()
    ch.advance(EVENTS)
    ch.status()                         # synchronises
    dt = time.perf_counter() - t0
    ch.close()
    return CHAINS * EVENTS / dt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON result to this file")
    args = ap.parse_args()
    count = p.lib().pdmpflux_jit_compile_count
    g = np.random.default_rng(0)
    x0 = g.standard_normal((CHAINS, D))
    v0 = np.where(g.random((CHAINS, D)) < 0.5, -1.0, 1.0)

    # NVRTC: the first sampler compiles the contract check and its kernels, the second finds them cached
    n0, t0 = count(), time.perf_counter()
    src = p.ZigZag(D, p.CudaPotential(BANANA_SRC), grid_size=10, AD_backend="ForwardDiff")
    cold_s, n_cold = time.perf_counter() - t0, count() - n0
    n0, t0 = count(), time.perf_counter()
    src = p.ZigZag(D, p.CudaPotential(BANANA_SRC), grid_size=10, AD_backend="ForwardDiff")
    warm_s, n_warm = time.perf_counter() - t0, count() - n0
    builtin = p.ZigZag(D, p.Banana(), grid_size=10, AD_backend="ForwardDiff")

    os.environ["PDMPFLUX_FORCE_GENERIC"] = "1"
    rates = {"builtin": [], "source": []}
    for s in (builtin, src):            # warm-up: module loads, first launches
        events_per_s(s, x0, v0, 1)
    for r in range(REPS):
        rates["builtin"].append(events_per_s(builtin, x0, v0, 100 + r))
        rates["source"].append(events_per_s(src, x0, v0, 100 + r))
    os.environ.pop("PDMPFLUX_FORCE_GENERIC")

    res = {
        "workload": f"ZigZag banana d={D}, grid_size=10, JVP, generic kernel, {CHAINS} chains x {EVENTS} events, Philox",
        "card": card(),
        "events_per_s": {k: {"runs": v, "median": float(np.median(v)), "min": min(v), "max": max(v)} for k, v in rates.items()},
        "source_over_builtin_median": float(np.median(rates["source"]) / np.median(rates["builtin"])),
        "nvrtc": {"cold_s_per_instantiation": cold_s / max(n_cold, 1), "cold_compiles": n_cold,
                  "warm_s_per_instantiation": warm_s / max(n_cold, 1), "warm_compiles": n_warm},
    }
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
