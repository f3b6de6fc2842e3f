"""Throughput of a source potential that declares its line model, against the built-in it restates and against the same
source without the declaration.

Workload: the C2 shape -- Zig-Zag, banana d = 50, grid_size = 0 (Brent bounds), Philox draws, 1000 events per chain,
no history (the kernel alone) -- at 4096 chains (teams of 8, transposed search) and 65536 chains (a chain per thread,
compressed line model).  Three arms alternate, 5 timed runs each after one warm-up each:
  builtin     p.Banana() on its own fast path
  declared    the restated banana with `affine` / `special = 2` (the same fast-path kernel, compiled at run time)
  undeclared  the same source without them (the generic kernel)
Also reports the cold NVRTC time per instantiation of each arm, and the card name and power limit read in the same
process.

    python tools/source_line_model_bench.py [--out result.json]
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
from test_source_line_model_cpu import BANANA_LM_SRC  # noqa: E402
from test_source_potential_cpu import BANANA_SRC  # noqa: E402

D, EVENTS, REPS = 50, 1000, 5
CHAINS = (4096, 65536)


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
    return x0.shape[0] * EVENTS / dt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON result to this file")
    args = ap.parse_args()
    count = p.lib().pdmpflux_jit_compile_count

    samplers, nvrtc = {"builtin": p.ZigZag(D, p.Banana(), grid_size=0)}, {}
    for arm, src in (("declared", BANANA_LM_SRC), ("undeclared", BANANA_SRC)):
        n0, t0 = count(), time.perf_counter()
        samplers[arm] = p.ZigZag(D, p.CudaPotential(src), grid_size=0)
        dt, n = time.perf_counter() - t0, count() - n0   # the contract check, then teams 8 and 1
        nvrtc[arm] = {"cold_s": dt, "compiles": n, "cold_s_per_compile": dt / max(n, 1)}

    res = {"workload": f"ZigZag banana d={D}, grid_size=0 (Brent), Philox, {EVENTS} events per chain, no history",
           "card": card(), "nvrtc": nvrtc, "events_per_s": {}}
    g = np.random.default_rng(0)
    for n_chains in CHAINS:
        x0 = g.standard_normal((n_chains, D))
        v0 = np.where(g.random((n_chains, D)) < 0.5, -1.0, 1.0)
        rates = {arm: [] for arm in samplers}
        for s in samplers.values():     # warm-up: module loads, first launches
            events_per_s(s, x0, v0, 1)
        for r in range(REPS):
            for arm, s in samplers.items():
                rates[arm].append(events_per_s(s, x0, v0, 100 + r))
        med = {arm: float(np.median(v)) for arm, v in rates.items()}
        res["events_per_s"][str(n_chains)] = {
            "arms": {arm: {"runs": v, "median": med[arm], "min": min(v), "max": max(v)} for arm, v in rates.items()},
            "declared_over_builtin_median": med["declared"] / med["builtin"],
            "declared_over_undeclared_median": med["declared"] / med["undeclared"],
        }
    res["card_after"] = card()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
