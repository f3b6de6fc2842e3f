#!/usr/bin/env python
"""Tiny run of every kernel family through the public API: odd dimensions, chain counts that do not fill a block and
every team width exercise the ragged paths.  Asserts finite output only; the write-bounds check of the same shapes is
tests/test_gpu_guard_bands.py (canary bands around every history column) and the values are checked by the parity tests."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

import pdmpflux_b200 as p  # noqa: E402

g = np.random.default_rng(0)


def run(name, mk, d, nch, n_sk, team=None, unit=False, **env):
    for k, v in env.items():
        os.environ[k] = str(v)
    if team:
        os.environ["PDMPFLUX_TEAM"] = str(team)
    try:
        x0 = g.standard_normal((nch, d))
        v0 = g.standard_normal((nch, d)) if unit else np.where(g.random((nch, d)) < 0.5, -1.0, 1.0)
        if unit:
            v0 /= np.linalg.norm(v0, axis=1, keepdims=True)
        s = mk()
        h = p.sample_skeleton(s, n_sk, x0, v0, seed=3)
        assert np.isfinite(h.X).all(), name
        out = p.sample_from_skeleton(s, 17, h)
        assert np.isfinite(out).all(), name
        print("ok", name, flush=True)
    finally:
        os.environ.pop("PDMPFLUX_TEAM", None)
        for k in env:
            os.environ.pop(k, None)


for team in (1, 8, 32):
    run(f"zz_brent_banana_t{team}", lambda: p.ZigZag(50, p.Banana(), grid_size=0), 50, 37, 9, team)
run("zz_brent_thread_per_chain_auto", lambda: p.ZigZag(33, p.GaussDiag(np.linspace(0.5, 2, 33)), grid_size=0), 33, 10300, 4)
run("zz_grid_t1", lambda: p.ZigZagAD(10, p.GaussStd()), 10, 70, 11, 1)
run("zz_grid_t8_equi", lambda: p.ZigZagAD(33, p.GaussEquicorr(0.5)), 33, 13, 9, 8)
run("zz_generic_fd", lambda: p.ZigZag(6, p.Banana(), grid_size=8), 6, 5, 6)  # finite differences: generic path
run("bps_t8", lambda: p.BPS(100, p.GaussEquicorr(0.9)), 100, 19, 9, 8, unit=True)
run("bps_t1", lambda: p.BPS(7, p.GaussStd(), refresh_rate=0.5), 7, 33, 9, 1, unit=True)
run("fecmc_t32", lambda: p.ForwardECMC(1000, p.GaussStd()), 1000, 5, 5, 32, unit=True)
run("fecmc_t8_global_scratch", lambda: p.ForwardECMC(200, p.GaussStd()), 200, 21, 5, 8, unit=True)
run("fecmc_small_smem_scratch", lambda: p.ForwardECMC(6, p.Banana(), ran_p=True, mix_p=0.7), 6, 9, 9, unit=True)
run("boom_fd_t32", lambda: p.Boomerang(1000, p.GaussStd()), 1000, 3, 5, 32, unit=True)
run("boom_t8", lambda: p.Boomerang(20, p.GaussDiag(np.linspace(0.5, 2, 20)), AD_backend="ForwardDiff"), 20, 7, 9, 8, unit=True)
run("sticky_t8", lambda: p.StickyZigZagAD(7, p.GaussStd(), np.full(7, 0.7)), 7, 9, 40, 8)
run("sticky_t1", lambda: p.StickyZigZagAD(3, p.GaussStd(), np.full(3, 1.5)), 3, 5, 40, 1)
run("speedup_t8", lambda: p.SpeedUpZigZagAD(9, p.GaussDiag(np.linspace(0.5, 2, 9))), 9, 6, 12, 8)
X = g.standard_normal((70, 5)) / np.sqrt(5); y = (g.random(70) < 0.5).astype(float)
run("logreg", lambda: p.ZigZagAD(5, p.LogReg(X, y, 10.0), grid_size=6), 5, 9, 6)
run("zz_host_path_many_slices", lambda: p.ZigZagAD(9, p.GaussStd()), 9, 11, 70, PDMPFLUX_SLAB_BYTES=1 << 14, PDMPFLUX_VBITS=1)
s = p.ZigZagAD(5, p.GaussStd())
hs = p.sample_skeleton(s, 2.5, g.standard_normal((6, 5)), np.ones((6, 5)), seed=1, batch=True)
print("ok until", [len(h) for h in hs], flush=True)
hb = p.sample_skeleton(s, 30, g.standard_normal((6, 5)), np.ones((6, 5)), seed=1)
m1, m2, T = p.skeleton_moments(s, hb)
from pdmpflux_b200 import _lib  # noqa: E402
sums = np.empty((4, 5))
_lib.check(p.lib().pdmpflux_moments_reduce(5, 6, m1.ctypes.data, m2.ctypes.data, None, sums.ctypes.data, 0, None))
print("ok reduce", p.RV_diagnostic(hb.chain(0), p.GaussStd(), B=5) >= 0, flush=True)
