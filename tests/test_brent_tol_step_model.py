"""Host model of the tol-step exit of the speculative Brent search (chain.cuh: build_bound_brent, NW = -1) against the
oracle's one-at-a-time recurrence (oracle/pdmp_oracle_np.py: brent_minimum).

A tol step is an iteration whose golden step is shorter than the tolerance, so the recurrence moves x by +-tol instead
of by the predicted golden step.  Every check of the pass holds for it except |gstp| >= tol; on increasing rates (the
C2 bound) it is the last step before the stopping rule.  The lane that owns it knows the state it leaves (x = u, the
bracket end on u's side unchanged, the other end the old x) and evaluates the stopping rule of the next iteration from
that state.  When the tol step is a new best in the assumed direction, is not the pass's last iteration and that rule
fires, the search ends on the tol step's value; anything else takes the commit-and-replay path of
tests/test_brent_speculation_model.py.  This file restates that logic in plain Python floats and checks it returns the
serial recurrence's minimum after the same number of iterations, and which exit each case takes."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
import pdmp_oracle_np as o  # noqa: E402
from test_brent_speculation_model import EPS, G, N, SQRT_EPS, TEAM, golden, parabola, serial, serial_step, start  # noqa: E402,E501


def stops(lo, hi, x):
    _, tol, mid, _, _ = golden(lo, hi, x)
    return abs(x - mid) <= 2 * tol - (hi - lo) / 2


def speculative_tol(f, h, stats):
    """the speculative search with the tol-step exit; stats counts the exits and the tol steps that fall back"""
    st, it, done = start(f, h), 0, False
    while it < 1000 and not done:
        lo, hi, x, w, v, fx, fw, fv, stp, old = st
        right = x < (hi + lo) / 2
        E = hi if right else lo
        X = [x]
        for _ in range(N):
            X.append(X[-1] + G * (E - X[-1]))
        W = [w] + X[:-1]
        V = [v, w] + X[:-2]
        F, TOL, U = [0.0] * N, [0.0] * N, [0.0] * N
        stop, asok, small, stop2 = [False] * N, [False] * N, [False] * N, [False] * N
        for k in range(N):
            moving = (lo if right else hi) if k == 0 else W[k]
            lo_, hi_ = (moving, hi) if right else (lo, moving)
            U[k], TOL[k], mid, og, gstp = golden(lo_, hi_, X[k])
            stop[k] = abs(X[k] - mid) <= 2 * TOL[k] - (hi_ - lo_) / 2
            direction = (X[k] < mid) == right
            asok[k] = direction and abs(gstp) >= TOL[k]
            small[k] = direction and abs(gstp) < TOL[k] and (U[k] < X[k]) != right
            lo2, hi2 = (X[k], hi_) if right else (lo_, X[k])   # the state a tol step that is a new best leaves
            stop2[k] = stops(lo2, hi2, U[k])
            F[k] = f(U[k])
        best, fin = [False] * N, [False] * N
        for k in range(N):
            fxk = F[k - 1] if k >= 1 else fx
            fwk = F[k - 2] if k >= 2 else (fx if k == 1 else fw)
            fvk = F[k - 3] if k >= 3 else (fx if k == 2 else (fw if k == 1 else fv))
            moving = (lo if right else hi) if k == 0 else W[k]
            lo_, hi_ = (moving, hi) if right else (lo, moving)
            oldk = old if k == 0 else E - W[k]
            para, _, _ = parabola((lo_, hi_, X[k], W[k], V[k], fxk, fwk, fvk, 0.0, oldk), TOL[k])
            best[k] = (not para) and F[k] < fxk
            fin[k] = best[k] and small[k] and stop2[k] and k < N - 1
            if fin[k]:
                stop[k + 1] = True                      # the lane of the tol step sets its successor's stop bit
        good = [(best[k] and asok[k]) or fin[k] for k in range(N)]
        nterm = next((k for k in range(N) if stop[k]), N)
        nbad = next((k for k in range(N) if not good[k]), N)
        nc = min(nterm, nbad)
        it += nc
        stats["passes"] += 1
        if nterm <= nbad and nterm < N:
            if nterm >= 1:
                fx = F[nterm - 1]
                stats["tol_exit"] += fin[nterm - 1]      # without it, nbad = nterm - 1: a replay
            st, done = (lo, hi, x, w, v, fx, fw, fv, stp, old), True
        else:
            if nbad < N and small[nbad]:                # a tol step that takes the replay path, and why
                why = "tol_last" if nbad == N - 1 else ("tol_not_best" if not best[nbad] else "tol_no_stop")
                stats[why] += 1
            if nc >= 1:
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
    return st[5], it


def new_stats():
    return dict(passes=0, replayed=0, tol_exit=0, tol_last=0, tol_not_best=0, tol_no_stop=0)


def check(f, h, stats):
    a, na = speculative_tol(f, h, stats)
    assert a == o.brent_minimum(f, 0.0, h) and na == serial(f, h)[1], (h, a, na)


@pytest.mark.parametrize("name", ["banana50", "gauss_increasing", "negative_curvature", "saddle"])
def test_tol_step_exit_equals_serial_recurrence(name):
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
    if name in ("banana50", "gauss_increasing"):   # increasing rates: one pass per bound, ended by the tol step
        assert stats["passes"] == n_bounds and stats["replayed"] == 0 and stats["tol_exit"] == n_bounds, stats
    else:                                          # the replay branches are still exercised
        assert stats["replayed"] > n_bounds, stats


def test_tol_step_at_the_last_iteration_of_a_pass_is_replayed():
    # decreasing rates: the search walks left towards 0, where tol shrinks to eps (60 .. 90 iterations, with replays
    # in between); over a wide range of h the tol step lands on every position of a pass, the last one included
    stats = new_stats()
    for h in np.geomspace(1e-6, 1e6, 1500):
        check(lambda t: t, float(h), stats)
        check(lambda t: 1.0 - np.sqrt(t), float(h), stats)
    assert stats["tol_last"] > 0 and stats["tol_exit"] > 0, stats


def test_tol_step_that_is_not_a_new_best_is_replayed():
    # -rate has its minimum at c just below h: the tol step jumps over it onto a worse value
    g = np.random.default_rng(3)
    stats = new_stats()
    for _ in range(400):
        h = float(g.uniform(0.5, 2.0))
        c = h * (1.0 - float(g.uniform(0.0, 4.0)) * o.SQRT_EPS)
        check(lambda t, c=c: -t if t < c else 3.0 * (t - c) - c, h, stats)
    assert stats["tol_not_best"] > 0, stats


def test_successor_of_a_tol_step_always_stops():
    # A tol step in the assumed direction leaves the bracket [x, E] (or [E, x]) of length |E - x| < tol / golden
    # < 2.62 tol, with x moved by tol; the stopping rule |x' - mid| <= 2 tol' - L / 2 then holds (L <= 3 tol).  So the
    # fallback for "tol step whose successor does not stop" is kept for exactness only: check the bound on random
    # brackets and that no search above or here reached that fallback.
    g = np.random.default_rng(11)
    stats = new_stats()
    for _ in range(20000):
        x = float(g.uniform(0.0, 10.0)) * 10.0 ** float(g.uniform(-12, 1))
        tol = SQRT_EPS * abs(x) + EPS
        right = bool(g.random() < 0.5)
        L = float(g.uniform(0.0, 1.0)) * tol / G
        far = x + L if right else x - L
        other = x - float(g.uniform(0.0, 1.0)) * L if right else x + float(g.uniform(0.0, 1.0)) * L
        lo, hi = (other, far) if right else (far, other)
        u, tol_, mid, _, gstp = golden(lo, hi, x)
        if (x < mid) != right or abs(gstp) >= tol_:
            continue
        lo2, hi2 = (x, hi) if right else (lo, x)
        assert stops(lo2, hi2, u), (lo, hi, x)
    for h in np.geomspace(0.05, 20.0, 200):
        speculative_tol(lambda t: t, float(h), stats)
        speculative_tol(lambda t: -t, float(h), stats)
    assert stats["tol_no_stop"] == 0, stats
