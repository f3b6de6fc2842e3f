#!/usr/bin/env python
"""Device-resident throughput of the BASELINE configurations (kernel time by CUDA events; not a bench line).

usage: tools/perf_probe.py SPEC [SPEC ...]     SPEC = config[:chains[:events[:team]]]   e.g.  c2:4096:1000:8  c5f
Each spec runs in a fresh subprocess-free loop: warm-up launch, then best of 3 timed launches; full PDMPHistory stored.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402
import pdmpflux_b200 as p  # noqa: E402


def run(name, nch, n_ev, team, reps=3):
    if team:
        os.environ["PDMPFLUX_TEAM"] = str(team)
    else:
        os.environ.pop("PDMPFLUX_TEAM", None)
    cfgd = bench.CONFIGS[name]
    d = cfgd["d"]
    s = bench.make_sampler(p, name)
    dev = torch.device("cuda")
    f64 = torch.float64
    x0 = torch.full((nch, d), cfgd["x0"], dtype=f64, device=dev)
    v0 = torch.ones((nch, d), dtype=f64, device=dev) / (d ** 0.5 if cfgd["unit_v"] else 1.0)
    ch = p.DeviceChains(s, x0, v0, seed=2024)
    bufs = dict(X=torch.empty((nch, n_ev, d), dtype=f64, device=dev), V=torch.empty((nch, n_ev, d), dtype=f64, device=dev),
                t=torch.empty((nch, n_ev), dtype=f64, device=dev), horizon=torch.empty((nch, n_ev), dtype=f64, device=dev),
                ar=torch.empty((nch, n_ev), dtype=f64, device=dev),
                error_value_ar=torch.empty((nch, n_ev, 5), dtype=f64, device=dev),
                errored_bound=torch.empty((nch, n_ev), dtype=torch.int32, device=dev),
                rejected=torch.empty((nch, n_ev), dtype=torch.int32, device=dev),
                hitting_horizon=torch.empty((nch, n_ev), dtype=torch.int32, device=dev))
    view = p.device_history_view(n_ev, **bufs)
    st = torch.cuda.current_stream().cuda_stream
    ch.advance(n_ev, view, 0, st)
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(reps):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); ch.advance(n_ev, view, 0, st); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) * 1e-3)
    _, _, cnt = ch.status()
    ev = nch * n_ev
    bpe = bench.bytes_per_event(d)
    print(f"{name:4s} team={team or 'auto':>4} chains={nch:6d} n_ev={n_ev:5d} {best*1e3:9.2f} ms  {ev/best/1e6:9.2f} Mev/s "
          f"{ev*bpe/best/1e9:8.1f} GB/s ({100*ev*bpe/best/1e9/6548.5:5.1f}% HBM)  builds/ev={cnt[:,0].sum()/(ev*(reps+1)):.2f} "
          f"rates/ev={cnt[:,1].sum()/(ev*(reps+1)):.2f}", flush=True)
    ch.close()


for spec in sys.argv[1:]:
    parts = spec.split(":")
    name = parts[0]
    nch = int(parts[1]) if len(parts) > 1 and parts[1] else bench.DEFAULT_CHAINS[name]
    n_ev = int(parts[2]) if len(parts) > 2 and parts[2] else bench.DEFAULT_EVENTS[name]
    team = int(parts[3]) if len(parts) > 3 and parts[3] else 0
    try:
        run(name, nch, n_ev, team)
    except Exception as e:  # keep going: one failing variant must not hide the others
        print(f"{spec}: FAILED {type(e).__name__}: {e}", flush=True)
