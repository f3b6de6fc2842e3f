"""Host model of the first pass of the speculative Brent search (chain.cuh: build_bound_brent, NW = -1), which also
evaluates the bound's starting point, against the oracle's one-at-a-time recurrence (oracle/pdmp_oracle_np.py:
brent_minimum).

In the first pass of a bound, slot 0 (lane 0, block 0) holds the starting point x = golden * h itself: its rate comes
out of the pass's batch like every other and no iteration, stopping rule or check runs there.  Slot k + 1 holds
iteration k, so f(x) of the initial state reaches iteration 0 through the same rotation as any other value, and the
pass covers the initial point plus 39 iterations.  Later passes start from a committed state whose f(x) is known and
map slot k to iteration k.  This file restates that map on top of the tol-step exit of
tests/test_brent_tol_step_model.py and checks it returns the serial recurrence's minimum after the same number of
iterations -- on increasing, decreasing and non-monotone rates, with the latest stop a first pass sees, and with
bounds that need more passes."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
import pdmp_oracle_np as o  # noqa: E402
from test_brent_speculation_model import G, N, TEAM, golden, parabola, serial, serial_step  # noqa: E402
from test_brent_tol_step_model import stops  # noqa: E402


def speculative_first_slot(f, h, stats):
    """the speculative search whose first pass evaluates the starting point in slot 0; (minimum, iterations)"""
    x0 = 0.0 + G * (h - 0.0)
    st = (0.0, h, x0, x0, x0, None, None, None, 0.0, 0.0)   # f(x0) is not known before the first pass
    it, done, first_pass = 0, False, True
    while it < 1000 and not done:
        sh = 1 if first_pass else 0                          # slot of iteration 0
        lo, hi, x, w, v, fx, fw, fv, stp, old = st
        right = x < (hi + lo) / 2
        E = hi if right else lo
        Xi = [x]
        for _ in range(N):
            Xi.append(Xi[-1] + G * (E - Xi[-1]))
        Wi = [w] + Xi[:-1]
        Vi = [v, w] + Xi[:-2]
        X = [x] * sh + Xi[:N - sh]                           # slot p: the state at the start of iteration p - sh
        W = [w] * sh + Wi[:N - sh]
        V = [v] * sh + Vi[:N - sh]
        F, TOL, U = [0.0] * N, [0.0] * N, [0.0] * N
        stop, asok, small, stop2 = [False] * N, [False] * N, [False] * N, [False] * N
        for p in range(N):
            start = p < sh
            moving = (lo if right else hi) if p == sh else W[p]
            lo_, hi_ = (moving, hi) if right else (lo, moving)
            U[p], TOL[p], mid, og, gstp = golden(lo_, hi_, X[p])
            if start:
                U[p] = x
            stop[p] = not start and abs(X[p] - mid) <= 2 * TOL[p] - (hi_ - lo_) / 2
            direction = (X[p] < mid) == right
            asok[p] = direction and abs(gstp) >= TOL[p]
            small[p] = not start and direction and abs(gstp) < TOL[p] and (U[p] < X[p]) != right
            lo2, hi2 = (X[p], hi_) if right else (lo_, X[p])
            stop2[p] = stops(lo2, hi2, U[p])
            F[p] = f(U[p])
        best, fin, good = [False] * N, [False] * N, [False] * N
        for p in range(N):
            if first_pass:                                   # f(x0) = fw = fv of the initial state sit in slot 0
                fxk, fwk, fvk = F[max(p - 1, 0)], F[max(p - 2, 0)], F[max(p - 3, 0)]
            else:
                fxk = F[p - 1] if p >= 1 else fx
                fwk = F[p - 2] if p >= 2 else (fx if p == 1 else fw)
                fvk = F[p - 3] if p >= 3 else (fx if p == 2 else (fw if p == 1 else fv))
            start = p < sh
            moving = (lo if right else hi) if p == sh else W[p]
            lo_, hi_ = (moving, hi) if right else (lo, moving)
            oldk = old if p == sh else E - W[p]
            para, _, _ = parabola((lo_, hi_, X[p], W[p], V[p], fxk, fwk, fvk, 0.0, oldk), TOL[p])
            best[p] = (not para) and F[p] < fxk
            fin[p] = best[p] and small[p] and stop2[p] and p < N - 1
            if fin[p]:
                stop[p + 1] = True
            good[p] = (best[p] and asok[p]) or fin[p] or start
        nterm = next((p for p in range(N) if stop[p]), N)
        nbad = next((p for p in range(N) if not good[p]), N)
        nc = min(nterm, nbad)
        it += nc - sh
        stats["passes"] += 1
        if nterm <= nbad and nterm < N:
            if first_pass:
                stats["last_stop_slot"] = max(stats["last_stop_slot"], nterm)
            if nterm >= 1:
                fx = F[nterm - 1]
            st, done = (lo, hi, x, w, v, fx, fw, fv, stp, old), True
        else:
            if first_pass:
                fx = fw = fv = F[0]
                st = (lo, hi, x, w, v, fx, fw, fv, stp, old)
            if nc > sh:
                xn = X[nc] if nc < N else U[N - 1]
                wn = X[nc - 1]
                vn = X[nc - 2] if nc >= 2 else w
                f1 = F[nc - 1]
                f2 = F[nc - 2] if nc >= 2 else fx
                f3 = F[nc - 3] if nc >= 3 else (fx if nc == 2 else fw)
                lo2, hi2 = (wn, hi) if right else (lo, wn)
                o2 = E - wn
                st = (lo2, hi2, xn, wn, vn, f1, f2, f3, G * o2, o2)
            if nc < N:
                for _ in range(TEAM):
                    st, stopped = serial_step(st, f)
                    if stopped:
                        done = True
                        break
                    it += 1
                    stats["replayed"] += 1
        first_pass = False
    return st[5], it


def new_stats():
    return dict(passes=0, replayed=0, last_stop_slot=0)


def check(f, h, stats):
    a, na = speculative_first_slot(f, h, stats)
    assert a == o.brent_minimum(f, 0.0, h) and na == serial(f, h)[1], (h, a, na)
    return na


@pytest.mark.parametrize("name", ["banana50", "gauss_increasing", "negative_curvature", "saddle"])
def test_first_slot_search_equals_serial_recurrence(name):
    d = {"banana50": 50, "gauss_increasing": 33, "negative_curvature": 20, "saddle": 20}[name]
    pot = {"banana50": lambda: o.Banana(), "gauss_increasing": lambda: o.GaussDiag(np.linspace(0.5, 2.0, d)),
           "negative_curvature": lambda: o.GaussDiag(-np.linspace(0.5, 2.0, d)),
           "saddle": lambda: o.GaussDiag(np.where(np.arange(d) % 2 == 0, 1.0, -1.0) * np.linspace(0.5, 2.0, d))}[name]()
    s = o.Sampler(d, pot, o.Config(sampler=o.ZIGZAG, grid_size=0))
    g = np.random.default_rng(7)
    stats = new_stats()
    n_bounds = 60
    for _ in range(n_bounds):
        x0, v0, h = g.standard_normal(d), np.where(g.random(d) < 0.5, -1.0, 1.0), float(g.uniform(0.05, 2.0))
        check(lambda t: -s.rate(x0, v0, t), h, stats)
    if name in ("banana50", "gauss_increasing"):   # increasing rates: the initial point and the whole search, one pass
        assert stats["passes"] == n_bounds and stats["replayed"] == 0, stats
    else:                                          # later passes and replays are exercised
        assert stats["passes"] > n_bounds and stats["replayed"] > n_bounds, stats


def test_latest_stop_of_the_first_pass():
    # A first pass that walks right on golden steps stops after 34 .. 36 iterations whatever h is (the stopping rule
    # only sees the bracket, and tol is relative there), so its latest stop is iteration 36 in slot 37: the initial
    # point and the whole search fit the 40 slots with two to spare.  A walk to the left turns back at iteration 0 and
    # continues in later passes (test_bounds_that_need_more_passes).
    stats = new_stats()
    for h in np.geomspace(1e-3, 1e6, 3000):
        check(lambda t: -t, float(h), stats)
    assert stats["passes"] == 3000 and stats["last_stop_slot"] == 37, stats


def test_bounds_that_need_more_passes():
    # decreasing and non-monotone rates: 60 .. 90 iterations, so the first pass commits and later passes follow
    stats = new_stats()
    for h in np.geomspace(1e-6, 1e6, 400):
        check(lambda t: t, float(h), stats)
        check(lambda t: 1.0 - np.sqrt(t), float(h), stats)
        check(lambda t: (t - 0.3 * h) ** 2, float(h), stats)
    assert stats["passes"] > 3 * 400 and stats["replayed"] > 0, stats
