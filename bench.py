#!/usr/bin/env python
"""bench.py -- skeleton events/s (+ ESS/s) of the grid-based Poisson-thinning hot path on B200.

Workload (BASELINE.json configs[1], "C2"): ZigZag, banana potential d=50 with the manual gradient,
grid_size=0 (constant bound via Brent), 4096 chains per GPU, Philox draws, full PDMPHistory columns stored.
One "step" = every chain advanced by --events accepted events (one launch of the skeleton kernel), followed
by the closed-form moment kernel, pdmpflux_moments_reduce and (N > 1) pdmpflux_moments_allreduce (NCCL, in the library).

  value  events/s, whole job, state and outputs resident in HBM (CUDA events, max over ranks)
  e2e    events/s through pdmpflux_sample_skeleton with HOST (pinned) buffers: H2D of the initial states and
         D2H of the full history inside the timed region (median, mean and max of individually timed calls)
  e2e_moments_only  the same metric end to end with fused in-kernel moments and no stored skeleton (only the
         initial states and 4 x d moment sums cross PCIe)
  roofline  the governing roofline north_star names: algorithmic bytes (16 d + 76 per event: X, V, t, horizon, ar,
         error_value_ar, 3 int32 counters) / skeleton-kernel time vs the measured HBM copy bandwidth
         (MEASURED_PEAKS.json); for --config c4 algorithmic FP64 flops vs the DMMA peak measured in this run
         (tools/fp64_peaks.cu, reported under roofline_fp64).  roofline.issue: fraction of the instruction-issue ceiling
         (what actually bounds the HBM-named kernels), from the ncu instruction count of this build (profiles/traffic.json,
         refused when its source stamp does not match the sources)
  strong_scaling  BASELINE config 5 (FECMC / Boomerang d = 1000): 65536 chains in total sharded over the N ranks
  cpu_baseline  the C restatement of the reference (oracle/, OpenMP, one chain per thread) on the host cores
`--impl reference` times that CPU restatement alone (Julia, hence the reference itself, is not installed).
`--dump-outputs DIR` writes the last timed step's history and moment sums (a seeded sample of chains, < 64 MB) as .npy.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
ALL_CPUS = os.sched_getaffinity(0)
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: (description, sampler ctor, d, vinit unit-norm?, x0 value, oracle (sampler, potential, params, kwargs))
    "c1": dict(desc="ZigZagAD std Gaussian d=10, grid_size=10 (README example)", d=10, unit_v=False, x0=0.0,
               oracle=(0, 0, None, dict())),
    "c2": dict(desc="ZigZag banana d=50, manual gradient, grid_size=0 (Brent constant bounds)", d=50, unit_v=False,
               x0=1.0, oracle=(0, 3, None, dict(grid_size=0))),
    "c3": dict(desc="BPS slanted (equicorrelated rho=0.9) Gaussian d=100, grid_size=10, refresh 0.1", d=100,
               unit_v=True, x0=0.0, oracle=(1, 2, [0.9], dict(tmax=1.0, refresh_rate=0.1))),
    "c4": dict(desc="ZigZag Bayesian logistic regression d=100, n=1e5 synthetic rows, grid_size=10 (FP64 DMMA gradient)",
               d=100, unit_v=False, x0=0.0, oracle=(0, 5, "logreg:100000", dict())),
    "c5f": dict(desc="ForwardECMC std Gaussian d=1000, grid_size=10", d=1000, unit_v=True, x0=0.0,
                oracle=(2, 0, None, dict())),
    "c5b": dict(desc="Boomerang std Gaussian d=1000, grid_size=10, refresh 0.1", d=1000, unit_v=False, x0=0.0,
                oracle=(3, 0, None, dict(tmax=1.0, refresh_rate=0.1, deriv_mode=1))),
}
DEFAULT_CHAINS = {"c1": 65536, "c2": 4096, "c3": 16384, "c4": 4096, "c5f": 8192, "c5b": 8192}
DEFAULT_EVENTS = {"c1": 500, "c2": 1000, "c3": 300, "c4": 8, "c5f": 40, "c5b": 40}


def logreg_data(n, d, seed=2024, sigma0=10.0):
    """Synthetic design of SURVEY.md 8d (C4): rows ~ N(0, I/d), theta* ~ N(0, I), y ~ Bernoulli(sigma(x.theta*))."""
    import numpy as np
    g = np.random.default_rng([seed, n, d])
    X = g.standard_normal((n, d)) / np.sqrt(d)
    theta = g.standard_normal(d)
    y = (g.random(n) < 1.0 / (1.0 + np.exp(-X @ theta))).astype(np.float64)
    return X, y, sigma0


def make_sampler(p, name):
    if name == "c1":
        return p.ZigZagAD(10, p.GaussStd())
    if name == "c2":
        return p.ZigZag(50, p.Banana(), grid_size=0)
    if name == "c3":
        return p.BPS(100, p.GaussEquicorr(0.9), refresh_rate=0.1)
    if name == "c4":
        X, y, s0 = logreg_data(100000, 100)
        return p.ZigZagAD(100, p.LogReg(X, y, s0))
    if name == "c5f":
        return p.ForwardECMC(1000, p.GaussStd())
    if name == "c5b":
        return p.Boomerang(1000, p.GaussStd())
    raise SystemExit(f"unknown config {name}")


FP64_PEAK_FALLBACK = 37.0  # TFLOP/s DMMA, earlier measurement on this pool (profiles/r2_fp64_peaks.json); used only when
                           # tools/fp64_peaks cannot run


def source_stamp():
    """sha256 over the kernel sources: ncu-derived numbers in profiles/traffic.json are only quoted for the build they
    were measured on."""
    import hashlib
    h = hashlib.sha256()
    csrc = os.path.join(ROOT, "pdmpflux.jl_b200", "csrc")
    for f in sorted(os.listdir(csrc)):
        if f.endswith((".cu", ".cuh")):
            h.update(open(os.path.join(csrc, f), "rb").read())
    return h.hexdigest()[:16]


def measured_profile(name):
    """(dram traffic per launch, warp instructions per event) from the committed ncu capture of THIS build, else Nones."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except (OSError, ValueError):
        return None, None, "profiles/traffic.json missing"
    if t.get("_source_stamp") != source_stamp():
        return None, None, "profiles/traffic.json was measured on another build (stamp %s != %s): not quoted" % (
            t.get("_source_stamp"), source_stamp())
    e = t.get(name) or {}
    return e.get("dram_bytes_per_launch"), e.get("warp_inst_per_event"), "ncu --set full capture of this build (profiles/)"


def fp64_peaks():
    """FP64 tensor (DMMA) and vector (DFMA) throughput of this GPU, measured now by tools/fp64_peaks (a few 10 ms)."""
    exe = os.path.join(ROOT, "tools", "fp64_peaks")
    try:
        out = subprocess.run([exe], capture_output=True, text=True, timeout=120).stdout.strip().splitlines()[-1]
        r = json.loads(out)
        if "dmma_tflops" in r:
            r["source"] = "measured in this run (tools/fp64_peaks.cu)"
            return r
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        pass
    return {"dmma_tflops": FP64_PEAK_FALLBACK, "dfma_tflops": 33.4, "source": "fallback: earlier measurement on this pool"}


def pin_to_gpu_numa_node(index):
    """Run (and allocate pinned host memory) on the CPUs local to the GPU's PCIe root: host buffers on the remote
    NUMA node make the D2H leg of the end-to-end number vary by 2-3x from run to run."""
    try:
        bdf = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(index)],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if bdf.startswith("00000000:"):
            bdf = bdf[4:]
        cpus = open(f"/sys/bus/pci/devices/{bdf}/local_cpulist").read().strip()
        ids = set()
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids.update(range(int(a), int(b or a) + 1))
        ids &= os.sched_getaffinity(0)
        if ids:
            os.sched_setaffinity(0, ids)
            return cpus
    except (OSError, ValueError, subprocess.SubprocessError):
        pass
    return None


def bytes_per_event(d):
    return 16 * d + 76


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for ts, r in self.rows if t0 <= ts <= t1 + 0.2] or [r for _, r in self.rows[-3:]]
        sm, mx, reasons = [], None, set()
        for r in rows:
            try:
                sm.append(float(r[1])); mx = float(r[2])
            except (ValueError, IndexError):
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_baseline(name, target_seconds=12.0, threads=None):
    """C restatement of the reference (oracle/) on the host cores, one chain per OpenMP thread, Philox draws:
    a bounded sample of the same workload."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import oracle_c as oc
    cfgd = CONFIGS[name]
    sampler, pot, pp, kw = cfgd["oracle"]
    d = cfgd["d"]
    threads = threads or os.cpu_count() or 1
    if isinstance(pp, str) and pp.startswith("logreg:"):
        import numpy as np
        X, y, s0 = logreg_data(int(pp.split(":")[1]), d)
        pp = np.concatenate([[float(X.shape[0]), s0], X.ravel(), y])
    cfg = oc.make_cfg(sampler, pot, d, pp, **kw)
    nch = threads * 4
    x0 = np.full((nch, d), cfgd["x0"]); v0 = np.ones((nch, d)) / (d ** 0.5 if cfgd["unit_v"] else 1.0)
    n_ev = 50 if name != "c4" else 1
    if name == "c4":
        nch = threads
        x0, v0 = x0[:nch], v0[:nch]
    t0 = time.perf_counter()
    oc.sample_skeleton(cfg, n_ev + 1, x0, v0, seed=2024, nthreads=threads)
    dt = time.perf_counter() - t0
    want = n_ev * target_seconds / max(dt, 1e-4)          # events per chain for the target time at nch chains
    n_ev = int(max(50 if name != "c4" else 1, min(20000, want)))   # cap the stored history (16 d bytes per event per chain)
    if want > n_ev:
        nch = int(min(threads * 64, max(nch, threads * round(nch * want / n_ev / threads))))
        x0 = np.full((nch, d), cfgd["x0"]); v0 = np.ones((nch, d)) / (d ** 0.5 if cfgd["unit_v"] else 1.0)
    t0 = time.perf_counter()
    r = oc.sample_skeleton(cfg, n_ev + 1, x0, v0, seed=2024, nthreads=threads)
    dt = time.perf_counter() - t0
    assert (r.status == 0).all()
    return {"value": nch * n_ev / dt, "unit": "events/s", "cores": threads, "kind": "port",
            "sample": f"{nch} chains x {n_ev} events, {dt:.1f} s, C restatement of the reference (oracle/pdmp_oracle.c) "
                      f"with OpenMP; Julia (the reference runtime) is not installed"}, dt, nch * n_ev


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name = args.config
    vals = []
    for _ in range(args.warmup):
        cpu_baseline(name, target_seconds=2.0)
    total_t, total_ev = 0.0, 0
    for _ in range(args.steps):
        cb, dt, ev = cpu_baseline(name, target_seconds=max(2.0, 60.0 / max(args.steps, 1)))
        vals.append(cb); total_t += dt; total_ev += ev
    v = total_ev / total_t
    cb = dict(vals[-1]); cb["value"] = v
    line = {"metric": "skeleton events/sec", "value": v, "unit": "events/s", "impl": "reference", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_t / max(args.steps, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{name}: {CONFIGS[name]['desc']}, CPU port of the reference, one chain per thread"},
            "cpu_baseline": cb,
            "e2e": {"value": v, "unit": "events/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def alloc_history(torch, dev, nch, n_ev, d):
    f64 = torch.float64
    return dict(X=torch.empty((nch, n_ev, d), dtype=f64, device=dev), V=torch.empty((nch, n_ev, d), dtype=f64, device=dev),
                t=torch.empty((nch, n_ev), dtype=f64, device=dev), horizon=torch.empty((nch, n_ev), dtype=f64, device=dev),
                ar=torch.empty((nch, n_ev), dtype=f64, device=dev),
                error_value_ar=torch.empty((nch, n_ev, 5), dtype=f64, device=dev),
                errored_bound=torch.empty((nch, n_ev), dtype=torch.int32, device=dev),
                rejected=torch.empty((nch, n_ev), dtype=torch.int32, device=dev),
                hitting_horizon=torch.empty((nch, n_ev), dtype=torch.int32, device=dev))


def init_states(torch, dev, name, nch):
    cfgd = CONFIGS[name]; d = cfgd["d"]
    x0 = torch.full((nch, d), cfgd["x0"], dtype=torch.float64, device=dev)
    v0 = torch.ones((nch, d), dtype=torch.float64, device=dev) / (d ** 0.5 if cfgd["unit_v"] else 1.0)
    return x0, v0


DUMP_BYTES = 60 * 10 ** 6   # array data of --dump-outputs; with the .npy headers the directory stays below 64 MB


def dump_outputs(out_dir, bufs, m1, m2, T, sums, seed=0):
    """Write what the last timed step handed back as out_dir/<name>.npy in float64: the 4 x d moment sums whole, and
    for a fixed, seeded sample of chains (as many as fit in DUMP_BYTES, in chain order) every history column and the
    chain's moments.  Same arguments give the same inputs, so two builds can be compared output for output."""
    import numpy as np
    import torch
    per_chain = dict(bufs, chain_m1=m1, chain_m2=m2, chain_T=T)
    nch = T.shape[0]
    chain_bytes = sum(a[0].numel() for a in per_chain.values()) * 8
    k = min(nch, max(1, (DUMP_BYTES - sums.numel() * 8) // chain_bytes))
    idx = np.sort(np.random.default_rng(seed).choice(nch, size=k, replace=False))
    sel = torch.from_numpy(idx).to(T.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "moment_sums.npy"), sums.cpu().numpy())
    for name, a in per_chain.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.index_select(0, sel).cpu().numpy().astype(np.float64))


C4_ROWS, C4_GRID = 100000, 10


def c4_flops(d, builds, rates, n_chain_launches):
    """FP64 work of the logistic-regression kernel.  algorithmic: 2nd(2 + 2G) per bound build (z = Xx, w = Xv and the
    d x 2G product), 2nd(2 + 1) per rate evaluation.  executed: the same minus the z / w products the (z, w) cache
    skips (a chain recomputes them on its first request of a launch and on every 64th request)."""
    nd2 = 2.0 * C4_ROWS * d
    alg = nd2 * ((2 + 2 * C4_GRID) * builds + 3 * rates)
    zw_done = n_chain_launches + (builds + rates) / 64.0
    exe = nd2 * (2 * C4_GRID * builds + rates) + 2 * nd2 * zw_done
    return alg, exe


def roofline_block(name, nch, n_ev, kern_s, builds, rates, n_chain_launches, hbm_peak, peak_src, fp64, clock_mhz, prof_key=None):
    """The governing roofline north_star names for the workload (HBM skeleton writes; FP64 DMMA for C4), from the
    kernel's CUDA-event time in THIS run, plus what actually limits it (instruction issue) where that is not the roofline."""
    d = CONFIGS[name]["d"]
    traffic, inst_per_event, prof_note = measured_profile(prof_key or name)
    events = nch * n_ev
    if traffic is not None:   # the capture was taken at the bench's launch shape; scale if this run's differs
        try:
            ev_prof = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[prof_key or name]["events_in_launch"]
            traffic = traffic * events / ev_prof
        except (OSError, ValueError, KeyError):
            pass
    if name == "c4":
        alg, exe = c4_flops(d, builds, rates, n_chain_launches)
        peak = float(fp64["dmma_tflops"])
        return {"bound": "fp64", "achieved": alg / kern_s / 1e12, "peak": peak, "unit": "TFLOP/s", "frac": alg / kern_s / 1e12 / peak,
                "executed": exe / kern_s / 1e12, "executed_frac": exe / kern_s / 1e12 / peak, "traffic": traffic,
                "kernel": "logreg_zigzag_kernel", "kernel_ms": kern_s * 1e3, "flop_per_event": alg / events,
                "peak_source": "FP64 DMMA (mma.sync.m8n8k4.f64), " + fp64["source"], "dfma_peak_tflops": fp64.get("dfma_tflops"),
                "note": "achieved counts the algorithmic flops (incl. the z/w products the (z, w) cache skips); executed "
                        "counts the DMMA work actually issued", "profile": prof_note}
    achieved = events * bytes_per_event(d) / kern_s / 1e9
    r = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic,
         "kernel": "skeleton_kernel", "kernel_ms": kern_s * 1e3, "bytes_per_event": bytes_per_event(d), "peak_source": peak_src,
         "profile": prof_note}
    if inst_per_event and clock_mhz:
        # every instruction of these kernels (FP64 arithmetic, selects, moves) issues at one per two cycles per scheduler
        # (tools/lat_probe.cu): the issue ceiling is 4 schedulers x 148 SMs x clock / 2 warp instructions per second
        ceiling = 4 * 148 * clock_mhz * 1e6 / 2.0
        r["issue"] = {"warp_inst_per_event": inst_per_event, "warp_inst_per_s": inst_per_event * events / kern_s,
                      "ceiling_warp_inst_per_s": ceiling, "frac": inst_per_event * events / kern_s / ceiling,
                      "note": "the kernel is bound by FP64 / ALU instruction issue, not by HBM: fraction of the measured "
                              "issue ceiling (one warp instruction per 2 cycles per scheduler)"}
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--chains", type=int, default=0, help="chains per GPU (default: the BASELINE config's)")
    ap.add_argument("--events", type=int, default=0, help="events per chain per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the short runs of the other BASELINE configs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    import pdmpflux_b200 as p

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    numa_cpus = pin_to_gpu_numa_node(local)
    torch.cuda.set_device(local)
    p.lib().pdmpflux_set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    comm = p.dist.Comm(dev)          # the library's own NCCL communicator (unique id carried by torch.distributed)

    name = args.config
    cfgd = CONFIGS[name]
    d = cfgd["d"]
    nch = args.chains or DEFAULT_CHAINS[name]
    n_ev = args.events or DEFAULT_EVENTS[name]
    sampler = make_sampler(p, name)
    f64 = torch.float64
    x0, v0 = init_states(torch, dev, name, nch)
    chain_offset, _ = p.dist.shard(nch * world, rank, world)      # weak scaling: nch chains on every rank
    chains = p.DeviceChains(sampler, x0, v0, seed=2024, chain_offset=chain_offset)
    bufs = alloc_history(torch, dev, nch, n_ev, d)
    view = p.device_history_view(n_ev, **bufs)
    m1 = torch.empty((nch, d), dtype=f64, device=dev); m2 = torch.empty((nch, d), dtype=f64, device=dev)
    Tl = torch.empty((nch,), dtype=f64, device=dev)
    sums = torch.empty((4, d), dtype=f64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    lib = p.lib()
    from pdmpflux_b200 import _lib as L

    kern_ms = []

    def step(timed):
        k0 = torch.cuda.Event(enable_timing=True); k1 = torch.cuda.Event(enable_timing=True)
        k0.record()
        chains.advance(n_ev, view, 0, stream)                       # skeleton kernel: n_ev events per chain
        k1.record()
        L.check(lib.pdmpflux_skeleton_moments(sampler.flow_kind, d, n_ev, nch, 0, bufs["X"].data_ptr(),
                                              bufs["V"].data_ptr(), bufs["t"].data_ptr(), m1.data_ptr(), m2.data_ptr(),
                                              Tl.data_ptr(), 1, stream))
        p.dist.moment_sums_device(m1, m2, Tl, sums, stream)         # pdmpflux_moments_reduce: 4 x d sufficient statistics
        comm.all_reduce(sums, stream)                               # pdmpflux_moments_allreduce: the only collective
        if timed:
            kern_ms.append((k0, k1))
        return sums

    for _ in range(max(args.warmup, 3)):
        step(False)
    torch.cuda.synchronize()
    _, _, cnt0 = chains.status()
    if world > 1:
        dist.barrier()
    launches0 = lib.pdmpflux_launch_count()
    clocks = ClockSampler(local); clocks.start()
    time.sleep(0.25)
    torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    w0 = time.time()
    e0.record()
    for _ in range(args.steps):
        step(True)
    e1.record()
    torch.cuda.synchronize()
    w1 = time.time()
    if world > 1:
        dist.barrier()
    clk = clocks.stop(w0, w1)
    launches = lib.pdmpflux_launch_count() - launches0
    elapsed = torch.tensor([e0.elapsed_time(e1) * 1e-3], dtype=f64, device=dev)
    kern = torch.tensor([sum(a.elapsed_time(b) for a, b in kern_ms) * 1e-3 / len(kern_ms)], dtype=f64, device=dev)
    per_rank_kernel_ms = [float(kern) * 1e3]
    if world > 1:
        gathered = [torch.empty_like(kern) for _ in range(world)]
        dist.all_gather(gathered, kern)
        per_rank_kernel_ms = [float(g) * 1e3 for g in gathered]
        dist.all_reduce(elapsed, op=dist.ReduceOp.MAX)
        dist.all_reduce(kern, op=dist.ReduceOp.MAX)
    elapsed = float(elapsed); kern = float(kern)
    _, _, cnt1 = chains.status()  # raises if any chain stopped
    builds = float((cnt1[:, 0] - cnt0[:, 0]).sum()) / args.steps
    rates = float((cnt1[:, 1] - cnt0[:, 1]).sum()) / args.steps
    total_chains = nch * world
    events_per_step = total_chains * n_ev
    value = events_per_step * args.steps / elapsed

    # ESS/s from the last step's cross-chain moment sums (definition: SURVEY.md 8d / sample.ess_from_chain_means)
    stats = p.dist.ess_from_sums(sums)
    ess_per_s = float(stats["ess"].min() / (elapsed / args.steps))

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (measured copy)" if peaks else "fallback 6.65 TB/s"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, bufs, m1, m2, Tl, sums)
    chains.close()
    del bufs, view
    torch.cuda.empty_cache()
    fp64 = fp64_peaks() if (rank == 0) else {"dmma_tflops": FP64_PEAK_FALLBACK, "source": "fallback"}
    roofline = roofline_block(name, nch, n_ev, kern, builds, rates, nch, hbm_peak, peak_src, fp64, clk.get("sm_mhz"))

    line = {"metric": "skeleton events/sec", "value": value, "unit": "events/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": 1e3 * elapsed / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{name}: {cfgd['desc']}", "chains_per_gpu": nch, "events_per_chain_per_step": n_ev,
                       "draws": "philox4x32-10 keyed (seed=2024, chain, event)", "stored": "full PDMPHistory row",
                       "l2": ("outputs per step (%.2f GB) exceed the 126 MB L2" % (nch * n_ev * bytes_per_event(d) / 1e9)) if name != "c4"
                             else "the (z, w) cache streamed per step (1.6 MB per chain, 6.6 GB) exceeds the 126 MB L2; X (80 MB) is meant to stay in it",
                       "parity": "unpinned against Julia (no Julia in the image): parity is against the CPU restatement in oracle/"},
            "ess_per_s": ess_per_s, "ess_definition": "min over coordinates of C * Var_pi(x_i) / Var_c(chain time-average of x_i), per step window",
            "gpu_launches": int(launches), "clocks": clk, "roofline": roofline, "roofline_fp64": fp64, "host_cpus": numa_cpus,
            "per_rank_kernel_ms": per_rank_kernel_ms, "source_stamp": source_stamp()}

    # strong scaling (BASELINE.json config 5): 65536 chains in total, sharded over the ranks of this job
    line["strong_scaling"] = strong_scaling(p, torch, dist, rank, world, dev)

    if not args.no_e2e:
        # every rank runs its shard through the host-buffer call at the same time (they share the host's memory
        # system and CPUs); the slowest rank's time counts
        if world > 1:
            # CPUs this rank may use for rebuilding the V rows: an equal share of the CPUs local to its GPU
            local_cpus = sorted(os.sched_getaffinity(0))
            sharing = [None] * world
            dist.all_gather_object(sharing, local_cpus)
            peers = sum(1 for other in sharing if other == local_cpus)
            os.environ["PDMPFLUX_HOST_THREADS"] = str(max(1, min(16, len(local_cpus) // max(peers, 1))))
            # (one rank alone needs >= 12 threads to beat the plain copy of the V rows -- the library's own default -- but
            # with several ranks the host's ingest bandwidth saturates (plain copy: 75 ms per step at 1 rank, 97 at 2,
            # 211 at 4), so moving half the bytes wins even with few threads per rank)
            os.environ["PDMPFLUX_VBITS"] = "1"
            dist.barrier()
        res = e2e(p, sampler, name, nch, n_ev, world, dev)
        if world > 1:
            dist.barrier()    # the two modes are measured one after the other on ALL ranks (they share the host)
        mom = e2e_moments(p, sampler, name, nch, n_ev, dev)
        if world > 1:
            worst = torch.tensor([res["ms_per_step"], mom["ms_per_step"] or 0.0], dtype=f64, device=dev)
            dist.all_reduce(worst, op=dist.ReduceOp.MAX)
            res["ms_per_step"] = float(worst[0])
            res["value"] = world * nch * n_ev / (float(worst[0]) * 1e-3)
            if mom["value"] is not None:
                mom["ms_per_step"] = float(worst[1])
                mom["value"] = world * nch * n_ev / (float(worst[1]) * 1e-3)
            for r_ in (res, mom):
                r_["h2d_bytes_per_step"] *= world; r_["d2h_bytes_per_step"] *= world
                r_["timing"] += "; all %d ranks concurrently, max over ranks" % world
            res["history_bytes_per_step"] *= world
        gbs = res["d2h_bytes_per_step"] / (res["ms_per_step"] * 1e-3) / 1e9
        res["d2h_gbs"] = gbs
        res["limiter"] = ("host ingest of the full history: %.1f GB/s device-to-host into one host's DRAM (all ranks together)" % gbs
                          if gbs > 15.0 else "the kernel (the history is small next to the compute)")
        line["e2e"] = res
        line["e2e_moments_only"] = mom
    if rank == 0 and world == 1 and not args.no_extra:
        line["extra_workloads"] = extra_workloads(p, name, hbm_peak, peak_src, fp64, clk.get("sm_mhz"))
    if world > 1:
        dist.barrier()
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        os.sched_setaffinity(0, ALL_CPUS)  # the CPU baseline uses every host core
        line["cpu_baseline"] = cpu_baseline(name)[0]
    if rank == 0:
        print(json.dumps(line))
    comm.close()
    if world > 1:
        dist.destroy_process_group()


def timed_launches(p, torch, name, nch, n_ev, dev, chain_offset=0, reps=3):
    """Kernel time (CUDA events, best of `reps` after a warm-up launch) of one advance() of n_ev events per chain with the
    full history stored; returns (seconds, builds, rates) with the counters of one launch."""
    d = CONFIGS[name]["d"]
    s = make_sampler(p, name)
    x0, v0 = init_states(torch, dev, name, nch)
    ch = p.DeviceChains(s, x0, v0, seed=2024, chain_offset=chain_offset)
    bufs = alloc_history(torch, dev, nch, n_ev, d)
    view = p.device_history_view(n_ev, **bufs)
    st = torch.cuda.current_stream().cuda_stream
    ch.advance(n_ev, view, 0, st)
    torch.cuda.synchronize()
    _, _, c0 = ch.status()
    best = float("inf")
    for _ in range(reps):
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        a.record(); ch.advance(n_ev, view, 0, st); b.record(); torch.cuda.synchronize()
        best = min(best, a.elapsed_time(b) * 1e-3)
    _, _, c1 = ch.status(); ch.close()
    del bufs, view, ch
    torch.cuda.empty_cache()
    return best, float((c1[:, 0] - c0[:, 0]).sum()) / reps, float((c1[:, 1] - c0[:, 1]).sum()) / reps


def strong_scaling(p, torch, dist, rank, world, dev):
    """BASELINE.json config 5: ForwardECMC / Boomerang, Gaussian d = 1000, 65536 chains IN TOTAL sharded over the ranks
    (fixed total work: strong scaling).  Device-timed kernel, slowest rank counts; the driver's N = 1, 2, 4, 8 runs give
    the curve."""
    out = {"scaling": "strong", "chains_total": 65536, "events_per_chain": 20}
    for name in ("c5f", "c5b"):
        off, cnt = p.dist.shard(65536, rank, world)
        sec, _, _ = timed_launches(p, torch, name, cnt, 20, dev, chain_offset=off, reps=2)
        t = torch.tensor([sec], dtype=torch.float64, device=dev)
        per_rank = [sec * 1e3]
        if world > 1:
            g = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(g, t)
            per_rank = [float(x) * 1e3 for x in g]
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sec = float(t)
        out[name] = {"workload": CONFIGS[name]["desc"], "events_per_s": 65536 * 20 / sec, "ms": sec * 1e3,
                     "per_rank_kernel_ms": per_rank, "chains_per_rank": cnt,
                     "hbm_gbs_per_gpu": cnt * 20 * bytes_per_event(1000) / sec / 1e9}
    return out


def extra_workloads(p, main, hbm_peak, peak_src, fp64, clock_mhz):
    """Short device-resident runs (kernel time by CUDA events, best of 3 after a warm-up launch) of the other
    BASELINE.json configurations and of the headline config at 65536 chains; same roofline accounting as the main line."""
    import torch
    out = {}
    todo = [(n, DEFAULT_CHAINS[n], DEFAULT_EVENTS[n]) for n in ("c1", "c2", "c3", "c4", "c5f", "c5b") if n != main]
    todo.append((main, 65536, 100 if main != "c4" else 2))
    dev = torch.device("cuda")
    for name, nch, n_ev in todo:
        if name == "c4" and nch > 8192:
            continue
        best, builds, rates = timed_launches(p, torch, name, nch, n_ev, dev)
        rl = roofline_block(name, nch, n_ev, best, builds, rates, nch, hbm_peak, peak_src, fp64, clock_mhz,
                            prof_key=(f"{name}@{nch}" if nch != DEFAULT_CHAINS[name] else None))
        e = {"workload": CONFIGS[name]["desc"], "chains": nch, "events_per_chain": n_ev, "events_per_s": nch * n_ev / best,
             "ms": best * 1e3, "roofline": rl}
        if rl["bound"] == "hbm":
            e.update({"hbm_gbs": rl["achieved"], "hbm_frac": rl["frac"], "bytes_per_event": rl["bytes_per_event"]})
        else:
            e.update({"fp64_tflops": rl["achieved"], "fp64_frac": rl["frac"], "fp64_executed_frac": rl["executed_frac"],
                      "fp64_peak_tflops": rl["peak"]})
        out[f"{name}@{nch}"] = e
    return out


def _pinned(lib, L, shape, dtype):
    import ctypes as C
    import numpy as np
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    ptr = C.c_void_p()
    L.check(lib.pdmpflux_host_alloc(C.byref(ptr), n))
    buf = (C.c_char * n).from_address(ptr.value)
    return np.frombuffer(buf, dtype=dtype).reshape(shape), ptr


def e2e(p, sampler, name, nch, n_ev, world, dev):
    """Same metric through the public C-ABI call with HOST buffers (pinned): every step copies the initial states
    host->device and the full history device->host inside the timed region.  Returns this rank's shard; the caller
    runs it on all ranks at once and takes the slowest."""
    import ctypes as C
    import numpy as np
    from pdmpflux_b200 import _lib as L
    lib = p.lib()
    cfgd = CONFIGS[name]
    d = cfgd["d"]
    n_sk = n_ev + 1
    arrs, ptrs = {}, []
    for f, shape, dt in (("X", (nch, n_sk, d), np.float64), ("V", (nch, n_sk, d), np.float64), ("t", (nch, n_sk), np.float64),
                         ("horizon", (nch, n_sk), np.float64), ("ar", (nch, n_sk), np.float64),
                         ("error_value_ar", (nch, n_sk, 5), np.float64), ("errored_bound", (nch, n_sk), np.int32),
                         ("rejected", (nch, n_sk), np.int32), ("hitting_horizon", (nch, n_sk), np.int32),
                         ("x0", (nch, d), np.float64), ("v0", (nch, d), np.float64)):
        arrs[f], ptr = _pinned(lib, L, shape, dt)
        ptrs.append(ptr)
    arrs["x0"][:] = cfgd["x0"]
    arrs["v0"][:] = 1.0 / (d ** 0.5 if cfgd["unit_v"] else 1.0)
    status = np.zeros(nch, dtype=np.int32)
    view = L.History(*(arrs[f].ctypes.data for f in ("X", "V", "t", "horizon", "ar", "error_value_ar", "errored_bound",
                                                     "rejected", "hitting_horizon")),
                     status.ctypes.data, None, None, n_sk, 0)

    def call(seed):
        L.check(lib.pdmpflux_sample_skeleton(sampler._handle, nch, n_sk, arrs["x0"].ctypes.data, arrs["v0"].ctypes.data,
                                             C.c_uint64(seed), 0, None, C.byref(view), None), status)

    import torch
    for w in range(4):  # warm-up calls: slab allocation, lazy module loading, PCIe / copy-engine ramp
        call(100 + w)
    torch.cuda.synchronize()
    # Each call is timed on its own; the median is the headline (on these shared hosts the PCIe / host-memory leg is
    # occasionally 10-20x slower for a single call), mean and max are reported beside it.
    reps, times = 7, []
    for i in range(reps):
        t0 = time.perf_counter()
        call(2 + i)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    times.sort()
    dt = times[len(times) // 2]
    ok = bool(np.isfinite(arrs["t"][:, -1]).all())
    arrs.clear()                             # views of the pinned buffers freed next
    for ptr in ptrs:
        lib.pdmpflux_host_free(ptr)
    lib.pdmpflux_sampler_release_workspace(sampler._handle)
    h2d, d2h = C.c_int64(0), C.c_int64(0)
    lib.pdmpflux_last_transfer_bytes(C.byref(h2d), C.byref(d2h))   # counted by the library from the copies it issued
    return {"value": nch * n_ev / dt, "unit": "events/s", "h2d_bytes_per_step": int(h2d.value),
            "d2h_bytes_per_step": int(d2h.value), "history_bytes_per_step": nch * n_sk * bytes_per_event(d),
            "ms_per_step": dt * 1e3, "ms_mean": 1e3 * sum(times) / reps, "ms_min": times[0] * 1e3, "ms_max": times[-1] * 1e3,
            "finite": ok, "timing": "median of %d individually timed calls" % reps,
            "call": "pdmpflux_sample_skeleton (host buffers, pinned): the reference's sample_skeleton with the full PDMPHistory returned to the host"}


def e2e_moments(p, sampler, name, nch, n_ev, dev):
    """End to end in moments-only mode: initial states from pinned host memory, the chains advance with fused in-kernel
    moments and NO stored skeleton (pdmpflux_chains_enable_moments, NULL history), the 4 x d sufficient statistics are
    reduced on the device and read back.  Nothing else crosses PCIe: this is the path that scales with the GPUs."""
    import ctypes as C
    import numpy as np
    import torch
    from pdmpflux_b200 import _lib as L
    lib = p.lib()
    cfgd = CONFIGS[name]; d = cfgd["d"]
    if name == "c4":
        return {"value": None, "unit": "events/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "ms_per_step": None,
                "timing": "", "call": "fused moments are not available for the logistic-regression kernel"}
    x0, px = _pinned(lib, L, (nch, d), np.float64); v0, pv = _pinned(lib, L, (nch, d), np.float64)
    sums_h, ps = _pinned(lib, L, (4, d), np.float64)
    x0[:] = cfgd["x0"]; v0[:] = 1.0 / (d ** 0.5 if cfgd["unit_v"] else 1.0)
    f64 = torch.float64
    m1 = torch.empty((nch, d), dtype=f64, device=dev); m2 = torch.empty_like(m1)
    T = torch.empty((nch,), dtype=f64, device=dev); sums = torch.empty((4, d), dtype=f64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def call(seed):
        ch = p.DeviceChains(sampler, x0, v0, seed=seed)            # H2D of the initial states
        ch.enable_moments()
        ch.advance(n_ev, None, 0, stream)
        L.check(lib.pdmpflux_chains_get_moments(ch._h, m1.data_ptr(), m2.data_ptr(), 1))
        L.check(lib.pdmpflux_chains_get_state(ch._h, None, None, T.data_ptr(), None, 1))
        p.dist.moment_sums_device(m1, m2, T, sums, stream)         # pdmpflux_moments_reduce
        torch.cuda.synchronize()
        sums_h[:] = sums.cpu().numpy()                              # D2H of the result
        ch.status(); ch.close()

    for w in range(2):
        call(50 + w)
    reps, times = 5, []
    for i in range(reps):
        t0 = time.perf_counter(); call(7 + i); times.append(time.perf_counter() - t0)
    times.sort()
    dt = times[len(times) // 2]
    finite = bool(np.isfinite(sums_h).all())
    del sums_h, x0, v0                       # views of the pinned buffers freed next
    for ptr in (px, pv, ps):
        lib.pdmpflux_host_free(ptr)
    return {"value": nch * n_ev / dt, "unit": "events/s", "h2d_bytes_per_step": 2 * 8 * d * nch, "d2h_bytes_per_step": 4 * 8 * d,
            "ms_per_step": dt * 1e3, "ms_mean": 1e3 * sum(times) / reps, "ms_max": times[-1] * 1e3,
            "finite": finite, "timing": "median of %d individually timed calls" % reps,
            "call": "pdmpflux_chains_create + enable_moments + chains_advance(NULL history) + moments_reduce, host (pinned) initial states in, 4 x d moment sums out"}


if __name__ == "__main__":
    main()
