"""Events per second of GaussDense (a Gaussian with a dense precision matrix) on Zig-Zag and BPS.

Zig-Zag runs the vectorised grid bound (ZigZagAD, grid_size = 10) and the Brent bound (grid_size = 0); BPS the default
grid bound with refresh_rate = 0.1.  P is a random SPD matrix with condition number 100 and chains start in the target.
Each configuration is warmed up, then timed over `--events` events per chain with no history (device clock around work
that ends in a synchronise).  Bytes of P read per event: 8 d per Zig-Zag flip (one row), 8 d^2 per BPS reflection or
refresh (all of P), out of the L2 (P is at most 32 MB).

    python tools/gauss_dense_bench.py [--dims 100 1000] [--chains 4096 16384] [--events 200] [--out FILE]

Prints one JSON line per configuration (and writes them all to --out)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def random_spd(d, cond=100.0, seed=0):
    g = np.random.default_rng([seed, d])
    q, _ = np.linalg.qr(g.standard_normal((d, d)))
    P = (q * np.geomspace(1.0, cond, d)) @ q.T
    return 0.5 * (P + P.T)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dims", type=int, nargs="+", default=[100, 1000])
    ap.add_argument("--chains", type=int, nargs="+", default=[4096, 16384])
    ap.add_argument("--events", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import pdmpflux_b200 as p

    info = gpu_info()
    lines = []
    for d in a.dims:
        P = random_spd(d)
        L = np.linalg.cholesky(np.linalg.inv(P))
        pot = p.GaussDense(P)
        for name, make in (("zigzag_grid10", lambda: p.ZigZagAD(d, pot)), ("zigzag_brent", lambda: p.ZigZag(d, pot, grid_size=0)),
                           ("bps_grid10", lambda: p.BPS(d, pot, refresh_rate=0.1))):
            s = make()
            for n in a.chains:
                g = np.random.default_rng([d, n])
                x0 = g.standard_normal((n, d)) @ L.T
                if name.startswith("zigzag"):
                    v0 = np.where(g.random((n, d)) < 0.5, -1.0, 1.0)
                else:
                    v0 = g.standard_normal((n, d)); v0 /= np.linalg.norm(v0, axis=1, keepdims=True)
                ch = p.DeviceChains(s, x0, v0, seed=1)
                ch.advance(a.warmup)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                ch.advance(a.events)
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                ch.status()
                ch.close()
                rec = dict(config=name, d=d, chains=n, events_per_chain=a.events, seconds=dt,
                           events_per_s=n * a.events / dt, gpu=info)
                print(json.dumps(rec), flush=True)
                lines.append(rec)
    if a.out:
        with open(a.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
