"""Where the cycles of one C2 event go: the phase clock of the thinning loop (chain.cuh, PDMPFLUX_PHASE_CLOCK).

Builds a separate copy of the library with -DPDMPFLUX_PHASE_CLOCK into OUT/ (the in-tree build is left alone), runs
the bench workload (Zig-Zag, banana d = 50, Brent bounds, Philox draws, 4096 chains x 1000 events) on it once to warm
up and once counted, and prints the lane cycles per event in each phase:

  func    compute_functionals, line model, classification
  pass    speculative passes of the transposed Brent search (the first one also evaluates the bound's starting point)
  replay  commit of a pass and the one-at-a-time iterations after it (or the broadcast of the final value)
  next    next_event and its exponential draw (after a bound and after a rejection)
  rate    the rate at the proposal and the accept uniform
  flip    flow, flip and record of an accepted event
  idle    waiting while other lanes of the warp run a block this lane skips

The clock reads perturb the schedule a little; compare splits taken with this tool, not with the bench's kernel time.

    python tools/phase_clock.py [--out DIR] [--lib PREBUILT.so] [--json FILE]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PHASES = ("func", "pass", "replay", "next", "rate", "flip", "idle")
D, CHAINS, EVENTS, SEED = 50, 4096, 1000, 2024


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "pdmpflux_phase_clock"), help="build directory")
    ap.add_argument("--lib", help="an already built phase-clock library (skips the build)")
    ap.add_argument("--json", help="also write the split to this file")
    args = ap.parse_args()
    lib_path = args.lib
    if not lib_path:
        out = os.path.abspath(args.out)
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "pdmpflux.jl_b200", "csrc"), "-j8",
                               f"OBJDIR={out}/build", f"LIBDIR={out}/lib", "EXTRA_NVCCFLAGS=-DPDMPFLUX_PHASE_CLOCK"])
        lib_path = os.path.join(out, "lib", "libpdmpflux_cuda.so")
    os.environ["PDMPFLUX_CUDA_LIB"] = os.path.abspath(lib_path)
    sys.path.insert(0, ROOT)
    import numpy as np
    import pdmpflux_b200 as p

    read = p.lib().pdmpflux_phase_clock
    read.argtypes = [ctypes.c_void_p]
    read.restype = ctypes.c_int
    cnt = np.zeros(len(PHASES) + 1, dtype=np.uint64)
    sampler = p.ZigZag(D, p.Banana(), grid_size=0)
    ch = p.DeviceChains(sampler, np.ones((CHAINS, D)), np.ones((CHAINS, D)), seed=SEED)
    ch.advance(EVENTS)                  # warm-up
    ch.status()
    assert read(cnt.ctypes.data) == 0
    ch.advance(EVENTS)
    ch.status()
    assert read(cnt.ctypes.data) == 0
    ch.close()
    lane_events = float(cnt[-1])
    assert lane_events > 0, "no events counted: is this a PDMPFLUX_PHASE_CLOCK build?"
    per_event = {k: float(c) / lane_events for k, c in zip(PHASES, cnt[:-1])}
    total = sum(per_event.values())
    try:
        card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader",
                               "-i", "0"], capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        card = f"unavailable ({e})"
    res = dict(lib=lib_path, card=card, workload=f"C2 {CHAINS} chains x {EVENTS} events", lane_cycles_per_event=total,
               split={k: dict(cycles=round(v), share=round(v / total, 4)) for k, v in per_event.items()})
    print(f"# phase clock, {res['workload']}, {lib_path}\n# card: {card}")
    print(f"{'phase':8s} {'cycles/event':>12s} {'share':>7s}")
    for k, v in per_event.items():
        print(f"{k:8s} {v:12.0f} {100 * v / total:6.1f}%")
    print(f"{'total':8s} {total:12.0f}")
    if args.json:
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
