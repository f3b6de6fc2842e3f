"""GPU parity tests: libpdmpflux_cuda.so (through the C ABI / pdmpflux_b200) against the CPU oracle.

Parity tiers (DESIGN.md "Parity"):
  * one-step (teacher-forced): every event k of every case is regenerated on the GPU from the oracle's state
    k-1 and tape cursor; JVP/grid bounds must match to 1e-10 relative (north_star tolerance), Brent and
    finite-difference modes to 1e-6 (they amplify last-bit summation-order differences by 1/sqrt(eps)).
    Velocity signs, rejected / hitting_horizon / errored_bound counters and draw consumption are exact.
  * free-running: same init + tape for the whole skeleton; held to 1e-10 over 10^4 events for the
    non-chaotic configurations (ZigZag on Gaussians, the README config C1).
"""
import os

import numpy as np
import pytest

import oracle_c as oc
from conftest import record_parity_error
from oracle_cases import CASES, case_inputs, pot_params, tier_tolerance

pytestmark = pytest.mark.gpu


def _potential(p, kind, pp):
    def logreg():
        n = int(pp[0])
        d = (len(pp) - 2 - n) // n
        return p.LogReg(pp[2:2 + n * d].reshape(n, d), pp[2 + n * d:], pp[1])
    return {0: lambda: p.GaussStd(), 1: lambda: p.GaussDiag(pp), 2: lambda: p.GaussEquicorr(pp[0]),
            3: lambda: p.Banana(), 4: lambda: p.BananaReadmeScalar(), 5: logreg}[kind]()


def make_sampler(p, sampler, pk, pp, d, kw):
    kw = dict(kw)
    ad = "ForwardDiff" if kw.pop("deriv_mode", 0) == 0 else "FiniteDiff"
    pot = _potential(p, pk, pp)
    if sampler == 0:
        return p.ZigZag(d, pot, AD_backend=ad, **kw)
    if sampler == 1:
        if "gaussian_velocity" in kw:
            kw["Gaussian_velocity"] = kw.pop("gaussian_velocity")
        return p.BPS(d, pot, AD_backend=ad, **kw)
    if sampler == 2:
        return p.ForwardECMC(d, pot, AD_backend=ad, **kw)
    return p.Boomerang(d, pot, AD_backend=ad, **kw)


def relerr(a, b):
    scale = max(np.max(np.abs(a)), np.max(np.abs(b)), 1e-300)
    return float(np.max(np.abs(a - b)) / scale)


@pytest.fixture(scope="module")
def p():
    import pdmpflux_b200
    n = __import__("ctypes").c_int(0)
    pdmpflux_b200.lib().pdmpflux_device_count(__import__("ctypes").byref(n))
    assert n.value > 0, "GPU tests need a CUDA device"
    return pdmpflux_b200


def set_team(team):
    if team:
        os.environ["PDMPFLUX_TEAM"] = str(team)
    else:
        os.environ.pop("PDMPFLUX_TEAM", None)


@pytest.mark.parametrize("generic", [0, 1], ids=["auto", "generic"])
@pytest.mark.parametrize("team", [1, 8, 32])
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_one_step_parity(p, case, team, generic):
    """`auto` runs the path the library picks (affine fast paths where they exist); `generic` forces the
    per-node generic kernel on the same case, so both implementations are held to the oracle.  Zig-Zag x Brent on
    teams of 8 runs the transposed search for d <= 64 and the register-resident line model for 64 < d <= 128."""
    name, sampler, pk, pp, d, kw, n_sk = case
    zz_brent_affine = sampler == 0 and kw.get("grid_size", 10) == 0 and pk in (0, 1, 2, 3) and not generic
    if generic and team != 8:
        pytest.skip("generic path is exercised at one team width")
    if team == 1 and d > 100:
        pytest.skip("thread-per-chain is for small d")
    if team == 1 and zz_brent_affine and d > 64:
        pytest.skip("thread-per-chain Zig-Zag x Brent is built for d <= 64 (the library ignores PDMPFLUX_TEAM=1 there)")
    if pk == 5 and (team != 8 or generic):
        pytest.skip("logistic regression has its own CTA-per-chain kernel (team width does not apply)")
    pp = pot_params(pp, d)
    x0, v0, (E, U, N) = case_inputs(name, sampler, d, n_sk)
    r = oc.sample_skeleton(oc.make_cfg(sampler, pk, d, pp, **kw), n_sk, x0, v0, tape=(E, U, N))
    assert r.status[0] == oc.ST_OK
    n = n_sk - 1
    pos = r.tape_pos[0]                       # cursor after event k
    use = np.diff(pos, axis=0)                # draws consumed by event k+1
    wE, wU, wN = (int(use[:, i].max()) + 1 for i in range(3))
    idx = lambda start, w: start[:, None] + np.arange(w)[None, :]
    pad = lambda a, w: np.concatenate([a, np.ones(w)])
    tE = pad(E[0], wE)[idx(pos[:-1, 0], wE)]
    tU = pad(U[0], wU)[idx(pos[:-1, 1], wU)]
    tN = pad(N[0], wN)[idx(pos[:-1, 2], wN)]
    s = make_sampler(p, sampler, pk, pp, d, kw)
    set_team(team)
    os.environ["PDMPFLUX_FORCE_GENERIC"] = str(generic)
    try:
        h = p.sample_skeleton(s, 2, r.X[0, :-1], r.V[0, :-1], tape=(tE, tU, tN), t0=r.t[0, :-1],
                              horizon0=r.horizon[0, :-1], batch=True)
    finally:
        set_team(None)
        os.environ.pop("PDMPFLUX_FORCE_GENERIC")
    tol = tier_tolerance(kw)
    assert np.array_equal(h.X[:, 0], r.X[0, :-1]) and np.array_equal(h.t[:, 0], r.t[0, :-1])
    scale_x = np.maximum(np.abs(r.X[0, 1:]).max(axis=1), 1e-300)
    ex = (np.abs(h.X[:, 1] - r.X[0, 1:]).max(axis=1) / scale_x).max()
    scale_v = np.abs(r.V[0, 1:]).max(axis=1)
    ev = (np.abs(h.V[:, 1] - r.V[0, 1:]).max(axis=1) / scale_v).max()
    dt_o = r.t[0, 1:] - r.t[0, :-1]
    et = (np.abs((h.t[:, 1] - h.t[:, 0]) - dt_o) / dt_o).max()
    eh = (np.abs(h.horizon[:, 1] - r.horizon[0, 1:]) / r.horizon[0, 1:]).max()
    ea = np.abs(h.ar[:, 1] - r.ar[0, 1:]).max()
    record_parity_error(f"one_step/{name}/team{team}/{'generic' if generic else 'auto'}", x=ex, v=ev, t=et, horizon=eh,
                        ar=ea, tol=tol)
    assert max(ex, ev, et, eh, ea) < tol, dict(x=ex, v=ev, t=et, horizon=eh, ar=ea)
    assert np.array_equal(np.sign(h.V[:, 1]), np.sign(r.V[0, 1:]))
    assert np.array_equal(h.rejected[:, 1], r.rejected[0, 1:])
    assert np.array_equal(h.hitting_horizon[:, 1], r.hitting_horizon[0, 1:])
    assert np.array_equal(h.errored_bound[:, 1], r.errored_bound[0, 1:])
    assert np.allclose(h.error_value_ar[:, 1], r.error_value_ar[0, 1:], rtol=tol, atol=0)
    assert np.array_equal(h.tape_pos, use)
    assert h.counters[:, 0].sum() == r.counters[0, 0] and h.counters[:, 1].sum() == r.counters[0, 1]


FREE_RUNNING = [
    # name, sampler, pot, pp, d, kw, n_sk, teams
    ("C1_zigzagAD_gauss10_1e4", 0, 0, None, 10, dict(), 10001),
    ("zz_gauss10_unsigned", 0, 0, None, 10, dict(signed_bound=False), 3001),
    ("zz_diag70", 0, 1, "linspace", 70, dict(), 3001),
    ("zz_equicorr33_nonadaptive", 0, 2, [0.5], 33, dict(grid_size=5, adaptive=False, tmax=0.3), 3001),
    # BASELINE.json config 3 at full size: BPS on the slanted Gaussian d = 100 (reflections + refreshes; the two CPU
    # restatements stay within 5e-15 of each other over 1200 events, so the dynamics do not amplify rounding)
    ("C3_bps_equi100_free", 1, 2, [0.9], 100, dict(tmax=1.0, refresh_rate=0.1), 3001),
]


@pytest.mark.parametrize("team", [1, 8, 32])
@pytest.mark.parametrize("case", FREE_RUNNING, ids=[c[0] for c in FREE_RUNNING])
def test_free_running_parity(p, case, team):
    """north_star: with injected draws, event times / positions / velocities match the Float64 reference path to
    1e-10 relative for the first 10^4 events, velocity signs bit-exact."""
    name, sampler, pk, pp, d, kw, n_sk = case
    if team == 1 and d > 70:
        pytest.skip("thread-per-chain is for small d")
    pp = pot_params(pp, d)
    nch = 3
    x0, v0, (E, U, N) = case_inputs(name, sampler, d, n_sk, n_chains=nch)
    r = oc.sample_skeleton(oc.make_cfg(sampler, pk, d, pp, **kw), n_sk, x0, v0, tape=(E, U, N))
    assert (r.status == 0).all()
    s = make_sampler(p, sampler, pk, pp, d, kw)
    set_team(team)
    try:
        h = p.sample_skeleton(s, n_sk, x0, v0, tape=(E, U, N))
    finally:
        set_team(None)
    worst = 0.0
    for c in range(nch):
        e = max(relerr(h.X[c], r.X[c]), relerr(h.t[c], r.t[c]), relerr(h.horizon[c], r.horizon[c]), relerr(h.ar[c], r.ar[c]))
        if sampler == 0:
            assert np.array_equal(h.V[c], r.V[c])  # ZigZag velocities are +-1: bit-exact
        else:
            e = max(e, relerr(h.V[c], r.V[c]))
            assert np.array_equal(np.sign(h.V[c]), np.sign(r.V[c]))
        worst = max(worst, e)
    record_parity_error(f"free_running/{name}/team{team}", max_rel=worst, events=n_sk - 1, tol=1e-10)
    assert worst < 1e-10, worst
    assert np.array_equal(h.rejected, r.rejected) and np.array_equal(h.hitting_horizon, r.hitting_horizon)
    assert np.array_equal(h.errored_bound, r.errored_bound) and np.array_equal(h.tape_pos, r.tape_used)
    assert np.array_equal(h.counters, r.counters)


def test_philox_mode_matches_oracle_draw_spec(p):
    """Without a tape both sides draw from Philox4x32-10(seed, chain, event): the GPU run must track the CPU
    oracle (differences only from device libm ulps in log/sincos)."""
    d, n_sk, nch = 10, 2001, 5
    x0 = np.zeros((nch, d)); v0 = np.ones((nch, d))
    r = oc.sample_skeleton(oc.make_cfg(0, 0, d), n_sk, x0, v0, seed=2024, chain_offset=7)
    s = p.ZigZagAD(d, p.GaussStd())
    h = p.sample_skeleton(s, n_sk, x0, v0, seed=2024, chain_offset=7)
    assert relerr(h.X, r.X) < 1e-9 and relerr(h.t, r.t) < 1e-9 and np.array_equal(h.V, r.V)
    # chain streams are keyed by the global chain id: shard [2:4] of the same run is reproduced exactly
    h2 = p.sample_skeleton(s, n_sk, x0[2:4], v0[2:4], seed=2024, chain_offset=9)
    assert np.array_equal(h2.X, h.X[2:4]) and np.array_equal(h2.t, h.t[2:4])
    # BPS refresh (normals) and FECMC switch (2d normals) also follow the spec
    for sampler, kw, mk in ((1, dict(tmax=1.0, refresh_rate=0.5), lambda: p.BPS(d, p.GaussStd(), refresh_rate=0.5)),
                            (2, dict(), lambda: p.ForwardECMC(d, p.GaussStd()))):
        v1 = v0 / np.sqrt(d)
        r = oc.sample_skeleton(oc.make_cfg(sampler, 0, d, **kw), 60, x0, v1, seed=11)
        h = p.sample_skeleton(mk(), 60, x0, v1, seed=11)
        assert relerr(h.X[:, :40], r.X[:, :40]) < 1e-7 and relerr(h.t[:, :40], r.t[:, :40]) < 1e-7


def test_resume_and_host_slicing_are_bit_identical(p):
    d, n_sk, nch = 6, 401, 9
    g = np.random.default_rng(3)
    x0 = g.standard_normal((nch, d)); v0 = g.standard_normal((nch, d)); v0 /= np.linalg.norm(v0, axis=1, keepdims=True)
    # Banana: the literal passes after an event; the Gaussians: the accept that accumulates the functionals and the line
    # model of the new state along with its own passes -- which must be exactly what a fresh launch computes from (x, v)
    for s in (p.BPS(d, p.Banana(), refresh_rate=0.3), p.BPS(d, p.GaussEquicorr(0.6), refresh_rate=0.3),
              p.BPS(d, p.GaussDiag(np.linspace(0.5, 2, d)), refresh_rate=0.1), p.ForwardECMC(d, p.GaussEquicorr(0.4))):
        h = p.sample_skeleton(s, n_sk, x0, v0, seed=5)
        os.environ["PDMPFLUX_SLAB_BYTES"] = str(1 << 20 >> 4)  # force many small device slabs
        try:
            hs = p.sample_skeleton(s, n_sk, x0, v0, seed=5)
        finally:
            os.environ.pop("PDMPFLUX_SLAB_BYTES")
        for f in ("X", "V", "t", "horizon", "ar", "error_value_ar", "errored_bound", "rejected", "hitting_horizon"):
            assert np.array_equal(getattr(h, f), getattr(hs, f)), f
        k = 150  # checkpoint = column k of the first run
        h2 = p.sample_skeleton(s, n_sk - k, h.X[:, k], h.V[:, k], seed=5, t0=h.t[:, k], horizon0=h.horizon[:, k], event0=k)
        assert np.array_equal(h2.X[:, 1:], h.X[:, k + 1:]) and np.array_equal(h2.t[:, 1:], h.t[:, k + 1:])
        assert np.array_equal(h2.V[:, 1:], h.V[:, k + 1:])


def test_sample_from_skeleton_and_moments(p):
    d, n_sk = 5, 3000
    for mk, fk, kw in ((lambda: p.ZigZagAD(d, p.GaussStd()), 0, dict()),
                       (lambda: p.Boomerang(d, p.GaussDiag(np.linspace(0.5, 2, d)), refresh_rate=0.4), 1, dict())):
        s = mk()
        hb = p.sample_skeleton(s, n_sk, np.zeros((3, d)), np.ones((3, d)), seed=1)
        N = 4567
        out = p.sample_from_skeleton(s, N, hb)
        full = p.sample_from_skeleton(s, N, hb, discard_vt=False)
        for c in range(3):
            ref = oc.sample_from_skeleton(fk, hb.X[c], hb.V[c], hb.t[c], N)
            assert relerr(out[c], ref) < 1e-13
            reff = oc.sample_from_skeleton(fk, hb.X[c], hb.V[c], hb.t[c], N, discard_vt=False)
            assert relerr(full[c], reff) < 1e-13
        # single-chain, reference-shaped API: (d, N) matrix
        h1 = hb.chain(1)
        o1 = p.sample_from_skeleton(s, N, h1)
        assert o1.shape == (d, N) and np.array_equal(o1, out[1].T)
        # closed-form moments agree with dense sampling of the same path
        m1, m2, T = p.skeleton_moments(s, hb)
        dense = p.sample_from_skeleton(s, 400000, hb)
        assert np.allclose(m1, dense.mean(axis=1), atol=5e-3) and np.allclose(m2, (dense**2).mean(axis=1), atol=1e-2)
        assert np.allclose(T, hb.t[:, -1])


def test_statistical_envelopes_of_reference_tests(p):
    """Philox-seeded runs against the envelopes the reference's own tests assert (test_property_based.jl:87-100,
    test_samplers.jl:51-54, test_comprehensive.jl:147,172-180) and posterior moments within Monte Carlo error."""
    s = p.ZigZagAD(1, p.GaussStd(), grid_size=0)
    h = p.sample_skeleton(s, 5000, 0.0, 1.0, seed=42)
    x = p.sample_from_skeleton(s, 5000, h)
    assert x.shape == (1, 5000) and abs(x.mean()) < 0.2 and 0.8 < x.var() < 1.2
    assert np.all(np.diff(h.t) > 0) and np.all(np.abs(h.V) == 1.0) and h.X.shape == (1, 5000)
    # many chains: pooled moments of N(0, I) to MC accuracy, all four samplers' stationary laws for the three
    # that target it (Boomerang's code path does not, see test_oracle_kat)
    d, nch, n_sk = 8, 512, 600
    for mk in (lambda: p.ZigZagAD(d, p.GaussStd()), lambda: p.BPS(d, p.GaussStd(), refresh_rate=0.5),
               lambda: p.ForwardECMC(d, p.GaussStd())):
        s = mk()
        g = np.random.default_rng(0)
        x0 = g.standard_normal((nch, d))
        v0 = np.ones((nch, d)) if isinstance(s, p.ZigZag) else np.ones((nch, d)) / np.sqrt(d)
        hb = p.sample_skeleton(s, n_sk, x0, v0, seed=9)
        m1, m2, T = p.skeleton_moments(s, hb, burn_in_cols=100)
        assert np.all(np.abs(m1.mean(axis=0)) < 0.05), m1.mean(axis=0)
        assert np.all(np.abs(m2.mean(axis=0) - 1.0) < 0.08), m2.mean(axis=0)


def test_error_behaviour_matches_reference(p):
    with pytest.raises(p.ArgumentError):
        p.ZigZag(0, p.GaussStd())
    with pytest.raises(p.ArgumentError):
        p.ZigZag(2, p.GaussStd(), grid_size=-1)
    with pytest.raises(p.ArgumentError):
        p.ForwardECMC(1, p.GaussStd())
    with pytest.raises(p.UnsupportedError):
        p.ZigZag(2, lambda x: x)
    s = p.ZigZag(3, p.GaussStd())
    with pytest.raises(p.ArgumentError):
        p.sample_skeleton(s, 0, np.zeros(3), np.ones(3))
    with pytest.raises(p.DimensionMismatch):
        p.sample_skeleton(s, 10, np.zeros(2), np.ones(2))
    h = p.sample_skeleton(s, 10, np.zeros(3), np.ones(3), seed=1)
    with pytest.raises(p.ArgumentError):
        p.sample_from_skeleton(s, 0, h)
    # Categorical(p) with sum(lambda) == 0 throws upstream: x = 0, grid_size=0 never leaves the origin's zero rate?
    # (a chain that cannot produce an event is reported, not hung)
    with pytest.raises(p.ChainError) as ei:
        p.sample_skeleton(p.ZigZag(2, p.GaussStd(), max_steps=50), 5, np.zeros(2), np.ones(2),
                          tape=(np.ones((1, 2)), np.full((1, 2), 0.5), np.zeros((1, 1))))
    assert ei.value.status[0] == 1  # tape exhausted


@pytest.mark.parametrize("d,team,n_sk,nch", [(10, 1, 37, 70), (3, 1, 50, 33), (7, 1, 41, 5), (50, 8, 29, 13),
                                             (33, 8, 30, 9), (64, 32, 21, 6), (1000, 32, 7, 3)])
def test_vector_and_bulk_store_paths_match_scalar_stores(p, d, team, n_sk, nch):
    """The 256-bit / TMA-bulk / zero-fill write path must produce exactly the bytes of the plain scalar-store path,
    for aligned and misaligned rows, heads and tails (odd d, odd n_sk, chain slabs starting mid-sector)."""
    g = np.random.default_rng(d)
    x0 = g.standard_normal((nch, d)); v0 = np.where(g.random((nch, d)) < 0.5, -1.0, 1.0)
    s = p.ZigZagAD(d, p.GaussStd())
    outs = []
    for nobulk in ("0", "1"):
        os.environ["PDMPFLUX_NO_BULK"] = nobulk
        set_team(team)
        try:
            outs.append(p.sample_skeleton(s, n_sk, x0, v0, seed=77))
        finally:
            set_team(None)
            os.environ.pop("PDMPFLUX_NO_BULK")
    a, b = outs
    for f in ("X", "V", "t", "horizon", "ar", "error_value_ar", "errored_bound", "rejected", "hitting_horizon"):
        assert np.array_equal(getattr(a, f), getattr(b, f)), f
    assert np.isfinite(a.X).all() and np.isfinite(a.t).all()


def test_logreg_free_running_and_posterior(p):
    """Config C4 in miniature: Zig-Zag on a logistic-regression posterior (four-chains-per-CTA DMMA kernel).  Free-running
    parity with injected draws, Philox determinism across sharding, and a posterior sanity check against a Laplace
    approximation."""
    from oracle_cases import logreg_data
    n, d, n_sk, nch = 200, 8, 400, 6
    X, y, s0 = logreg_data(n, d)
    pp = np.concatenate([[float(n), s0], X.ravel(), y])
    x0, v0, (E, U, N) = case_inputs("logreg_free", 0, d, n_sk, n_chains=nch)
    r = oc.sample_skeleton(oc.make_cfg(0, 5, d, pp, grid_size=8), n_sk, x0, v0, tape=(E, U, N))
    assert (r.status == 0).all()
    s = p.ZigZagAD(d, p.LogReg(X, y, s0), grid_size=8)
    h = p.sample_skeleton(s, n_sk, x0, v0, tape=(E, U, N))
    assert relerr(h.X, r.X) < 1e-9 and relerr(h.t, r.t) < 1e-9 and np.array_equal(h.V, r.V)
    assert np.array_equal(h.rejected, r.rejected) and np.array_equal(h.hitting_horizon, r.hitting_horizon)
    assert np.array_equal(h.tape_pos[:, :2], r.tape_used[:, :2])
    # smallest / largest grid (a pass carries 64 residual columns: with G = 12 only two bound requests fit, the
    # others wait a round) and a chain count that leaves the last CTA partly empty
    for G in (2, 12):
        xg, vg, tape_g = case_inputs("logreg_grid%d" % G, 0, d, 80, n_chains=9)
        rg = oc.sample_skeleton(oc.make_cfg(0, 5, d, pp, grid_size=G), 80, xg, vg, tape=tape_g)
        hg = p.sample_skeleton(p.ZigZagAD(d, p.LogReg(X, y, s0), grid_size=G), 80, xg, vg, tape=tape_g)
        assert (rg.status == 0).all() and relerr(hg.X, rg.X) < 1e-9 and relerr(hg.t, rg.t) < 1e-9
        assert np.array_equal(hg.V, rg.V) and np.array_equal(hg.rejected, rg.rejected)
    # Philox mode: shards reproduce the big run
    hp = p.sample_skeleton(s, 60, x0, v0, seed=3)
    hp2 = p.sample_skeleton(s, 60, x0[2:5], v0[2:5], seed=3, chain_offset=2)
    assert np.array_equal(hp.X[2:5], hp2.X) and np.array_equal(hp.t[2:5], hp2.t)
    # posterior mean ~ MAP (Laplace) within a few posterior standard deviations, pooled over chains
    nch2 = 64
    hb = p.sample_skeleton(s, 1500, np.zeros((nch2, d)), np.where(np.arange(nch2 * d).reshape(nch2, d) % 2, 1.0, -1.0), seed=11)
    m1, m2, T = p.skeleton_moments(s, hb, burn_in_cols=300)
    theta = np.zeros(d)
    for _ in range(50):  # Newton iterations for the MAP
        sg = 1 / (1 + np.exp(-X @ theta))
        g = X.T @ (sg - y) + theta / s0**2
        Hm = X.T @ (X * (sg * (1 - sg))[:, None]) + np.eye(d) / s0**2
        theta -= np.linalg.solve(Hm, g)
    sd = np.sqrt(np.diag(np.linalg.inv(Hm)))
    assert np.all(np.abs(m1.mean(axis=0) - theta) < 0.5 * sd), (m1.mean(axis=0), theta, sd)
    # unsupported combinations fail loudly instead of falling back
    with pytest.raises(p.UnsupportedError):
        p.BPS(d, p.LogReg(X, y, s0))
    with pytest.raises(p.UnsupportedError):
        p.ZigZag(d, p.LogReg(X, y, s0), grid_size=0)


@pytest.mark.parametrize("kind", ["zigzag", "bps", "boomerang", "fecmc", "logreg"])
def test_time_horizon_variant_parity(p, kind):
    """sample_skeleton(sampler, T::Float64, ...) (src/sample.jl:323-439) against the oracle's literal restatement:
    same ragged column counts, t[end] == T exactly, event columns and the final flowed point within tolerance."""
    from oracle_cases import logreg_data
    d, nch, T = 6, 7, 9.0
    g = np.random.default_rng(5)
    x0 = 0.3 * g.standard_normal((nch, d))
    if kind == "zigzag":
        s, cfg, v0 = p.ZigZagAD(d, p.GaussStd()), oc.make_cfg(0, 0, d), np.where(g.random((nch, d)) < 0.5, -1.0, 1.0)
    elif kind == "bps":
        s, cfg = p.BPS(d, p.GaussDiag(np.linspace(0.5, 2, d)), refresh_rate=0.3), oc.make_cfg(1, 1, d, np.linspace(0.5, 2, d), tmax=1.0, refresh_rate=0.3)
        v0 = g.standard_normal((nch, d)); v0 /= np.linalg.norm(v0, axis=1, keepdims=True)
    elif kind == "boomerang":
        s, cfg = p.Boomerang(d, p.GaussStd(), refresh_rate=0.4, AD_backend="ForwardDiff"), oc.make_cfg(3, 0, d, tmax=1.0, refresh_rate=0.4)
        v0 = g.standard_normal((nch, d))
    elif kind == "fecmc":
        s, cfg = p.ForwardECMC(d, p.GaussStd()), oc.make_cfg(2, 0, d)
        v0 = g.standard_normal((nch, d)); v0 /= np.linalg.norm(v0, axis=1, keepdims=True)
    else:
        X, y, s0 = logreg_data(60, d)
        s, cfg = p.ZigZagAD(d, p.LogReg(X, y, s0), grid_size=5), oc.make_cfg(0, 5, d, np.concatenate([[60.0, s0], X.ravel(), y]), grid_size=5)
        v0 = np.where(g.random((nch, d)) < 0.5, -1.0, 1.0); T = 1.5
    E = g.standard_exponential((nch, 4000)); U = g.random((nch, 4000)); N = g.standard_normal((nch, 4000 * d))
    r = oc.sample_skeleton_until(cfg, T, 1000, x0, v0, tape=(E, U, N))
    assert (r.status == 0).all() and (r.ncols >= 2).all()
    hs = p.sample_skeleton(s, T, x0, v0, tape=(E, U, N), batch=True)     # float T -> time-horizon method
    assert [len(h) for h in hs] == r.ncols.tolist()
    tol = 1e-9
    for c, h in enumerate(hs):
        n = r.ncols[c]
        assert h.t[-1] == T and h.X.shape == (d, n)
        assert relerr(h.X.T, r.X[c, :n]) < tol and relerr(h.V.T, r.V[c, :n]) < tol and relerr(h.t, r.t[c, :n]) < tol
        assert np.array_equal(h.rejected, r.rejected[c, :n]) and np.array_equal(h.hitting_horizon, r.hitting_horizon[c, :n])
        assert h.ar[-1] == 0 and h.rejected[-1] == 0 and h.hitting_horizon[-1] == 0
    # capacity growth path (reference: _grow_history doubling) and the single-chain return type
    h1 = p.sample_skeleton_until(s, T, x0[0], v0[0], tape=(E[:1], U[:1], N[:1]), init_capacity=2)
    assert len(h1) == r.ncols[0] and h1.t[-1] == T and relerr(h1.X.T, r.X[0, :r.ncols[0]]) < tol
    h0 = p.sample_skeleton(s, 0.0, x0[0], v0[0], seed=1)
    assert len(h0) == 1 and h0.t[0] == 0.0
    with pytest.raises(p.ArgumentError):
        p.sample_skeleton(s, -1.0, x0[0], v0[0], seed=1)
    # sample_from_skeleton on the ragged result uses t[end] == T as its time scale
    xs = p.sample_from_skeleton(s, 50, hs[0])
    assert xs.shape == (d, 50) and np.isfinite(xs).all()


def test_sample_from_skeleton_dt_methods(p):
    """The dt method (src/sample.jl:573-646) and the (N, dt) method (:649-682) against a direct numpy evaluation."""
    d, n_sk = 4, 500
    for s, fk in ((p.ZigZagAD(d, p.GaussStd()), 0), (p.Boomerang(d, p.GaussStd(), refresh_rate=0.5), 1)):
        h = p.sample_skeleton(s, n_sk, np.zeros(d), np.ones(d), seed=4)

        def ref(nuse, dt):
            tt = h.t[:nuse]
            M = int(np.floor(tt[-1] / dt))
            out = np.empty((2 * d + 1, M))
            for j in range(1, M + 1):
                tm = j * dt
                i = np.searchsorted(tt, tm, side="right") - 1
                tau = tm - tt[i]
                if fk:
                    out[:d, j - 1] = h.X[:, i] * np.cos(tau) + h.V[:, i] * np.sin(tau)
                    out[d:2 * d, j - 1] = -h.X[:, i] * np.sin(tau) + h.V[:, i] * np.cos(tau)
                else:
                    out[:d, j - 1] = h.X[:, i] + h.V[:, i] * tau
                    out[d:2 * d, j - 1] = h.V[:, i]
                out[2 * d, j - 1] = tm
            return out
        dt = h.t[-1] / 333.3
        a = p.sample_from_skeleton(s, dt, h)                       # (sampler, dt, history)
        r = ref(n_sk, dt)
        assert a.shape == (d, r.shape[1]) and np.allclose(a, r[:d], rtol=1e-12, atol=1e-13)
        b = p.sample_from_skeleton(s, 200, h, dt, discard_vt=False)  # (sampler, N, dt, history)
        r2 = ref(200, dt)
        assert b.shape == r2.shape and np.allclose(b, r2, rtol=1e-12, atol=1e-13)
    with pytest.raises(p.ArgumentError):
        p.sample_from_skeleton(s, -0.1, h)


@pytest.mark.parametrize("kind", ["zigzag", "zigzag_brent", "bps", "boomerang", "fecmc"])
def test_fused_moments_match_skeleton_integrals(p, kind):
    """In-kernel running integrals of x and x^2 (no stored skeleton needed) equal the closed-form integrals over the
    stored skeleton, also across several advance() calls, with a NULL history and in the time-horizon mode."""
    import torch
    d, nch, n_ev = 12, 40, 300
    g = np.random.default_rng(8)
    x0 = g.standard_normal((nch, d))
    v0 = np.where(g.random((nch, d)) < 0.5, -1.0, 1.0) if kind.startswith("zigzag") else g.standard_normal((nch, d))
    s = {"zigzag": lambda: p.ZigZagAD(d, p.Banana()), "zigzag_brent": lambda: p.ZigZag(d, p.Banana(), grid_size=0),
         "bps": lambda: p.BPS(d, p.GaussEquicorr(0.5), refresh_rate=0.3),
         "boomerang": lambda: p.Boomerang(d, p.GaussDiag(np.linspace(0.5, 2, d)), refresh_rate=0.4),
         "fecmc": lambda: p.ForwardECMC(d, p.GaussStd())}[kind]()
    dev = torch.device("cuda")
    f64 = torch.float64
    ch = p.DeviceChains(s, x0, v0, seed=21)
    ch.enable_moments()
    X = torch.empty((nch, n_ev + 1, d), dtype=f64, device=dev); V = torch.empty_like(X)
    t = torch.empty((nch, n_ev + 1), dtype=f64, device=dev)
    view = p.device_history_view(n_ev + 1, X=X, V=V, t=t)
    ch.record(view, 0)
    ch.advance(100, view, 1)
    ch.advance(n_ev - 100, view, 101)
    torch.cuda.synchronize()
    m1, m2 = ch.moments()
    hb = p.PDMPHistoryBatch(nch, n_ev + 1, d)
    hb.X[:] = X.cpu().numpy(); hb.V[:] = V.cpu().numpy(); hb.t[:] = t.cpu().numpy()
    r1, r2, T = p.skeleton_moments(s, hb)
    assert np.allclose(m1, r1 * T[:, None], rtol=1e-10, atol=1e-11) and np.allclose(m2, r2 * T[:, None], rtol=1e-10, atol=1e-11)
    # no history at all + stop at T: the integrals cover exactly [0, T]
    ch2 = p.DeviceChains(s, x0, v0, seed=21)
    ch2.enable_moments()
    Tstop = float(hb.t[:, 150].min())
    ch2.set_stop_time(Tstop)
    ch2.advance(400)
    a1, a2 = ch2.moments()
    _, _, tt, _ = ch2.get_state()
    assert np.all(tt == Tstop)
    # reference value: integrate the stored skeleton up to Tstop with dense sampling of the exact path
    dense = p.sample_from_skeleton(s, 200000, hb)  # (C, N, d) over [0, t_end]
    for c in range(0, nch, 13):
        n_in = int(np.floor(Tstop / (hb.t[c, -1] / 200000)))
        approx = dense[c, :n_in].mean(axis=0) * Tstop
        assert np.allclose(a1[c], approx, atol=5e-3 * max(1.0, Tstop))


def test_rv_diagnostic_reference_kat_and_errors(p):
    """The reference's own known answer (test/test_diagnostics.jl:100-124) through the C ABI, plus its error paths."""
    X = np.array([[0.0, 0.5, 1.0]]); V = np.ones((1, 3)); t = np.array([0.0, 0.5, 1.0])
    z = np.zeros(3); zi = np.zeros(3, dtype=np.int32)
    h = p.PDMPHistory(X, V, t, z, z, zi, np.zeros((5, 3)), zi, zi)
    U = lambda x: x ** 2 / 2
    expected = sum((U(k / 4) - U((k - 1) / 4)) ** 2 for k in range(1, 5))
    assert p.RV_diagnostic(h, p.GaussStd(), B=4) == pytest.approx(expected, rel=1e-14)
    assert p.RV_diagnostic(h, p.GaussStd(), B=0) > 0.0
    with pytest.raises(p.ArgumentError):
        p.RV_diagnostic(h, p.GaussStd(), B=-1)
    h0 = p.PDMPHistory(X[:, :1], V[:, :1], t[:1], z[:1], z[:1], zi[:1], np.zeros((5, 1)), zi[:1], zi[:1])
    assert p.RV_diagnostic(h0, p.GaussStd(), B=3) == 0.0                    # T == 0
    hneg = p.PDMPHistory(X, V, np.array([0.0, 0.5, np.inf]), z, z, zi, np.zeros((5, 3)), zi, zi)
    with pytest.raises(p.ArgumentError):
        p.RV_diagnostic(hneg, p.GaussStd())


@pytest.mark.parametrize("kind", ["zigzag_banana", "zigzag_readme", "bps_equicorr", "fecmc_std", "boomerang_diag"])
def test_rv_diagnostic_matches_oracle(p, kind):
    """Device RV_diagnostic against the oracle's literal restatement (src/diagnostic.jl:37-75) on sampled skeletons,
    1e-10 relative: batches, B = 0 and explicit, and the offline diagnostic's straight lines even for Boomerang."""
    import pdmp_oracle_np as onp
    d, nch, n_sk = 9, 6, 400
    g = np.random.default_rng(17)
    mk = {"zigzag_banana": (lambda: p.ZigZagAD(d, p.Banana()), onp.Banana()),
          "zigzag_readme": (lambda: p.ZigZag(d, p.GaussStd()), onp.BananaReadmeScalar()),
          "bps_equicorr": (lambda: p.BPS(d, p.GaussEquicorr(0.6), refresh_rate=0.2), onp.GaussEquicorr(d, 0.6)),
          "fecmc_std": (lambda: p.ForwardECMC(d, p.GaussStd()), onp.GaussStd()),
          "boomerang_diag": (lambda: p.Boomerang(d, p.GaussDiag(np.linspace(0.5, 2, d)), refresh_rate=0.3),
                             onp.GaussDiag(np.linspace(0.5, 2, d)))}[kind]
    s, opot = mk[0](), mk[1]
    dev_pot = {"zigzag_readme": p.BananaReadmeScalar()}.get(kind, s.potential)
    x0 = g.standard_normal((nch, d))
    v0 = np.where(g.random((nch, d)) < 0.5, -1.0, 1.0) if kind.startswith("zigzag") else g.standard_normal((nch, d))
    hb = p.sample_skeleton(s, n_sk, x0, v0, seed=5)
    for B in (0, 7, 250):
        rv = p.RV_diagnostic(hb, dev_pot, B=B)
        ref = np.array([onp.rv_diagnostic(hb.X[c].T, hb.V[c].T, hb.t[c], opot.value, B=B) for c in range(nch)])
        assert rv.shape == (nch,) and np.allclose(rv, ref, rtol=1e-10, atol=0), (B, rv, ref)
    one = p.RV_diagnostic(hb.chain(2), dev_pot, B=31)
    assert one == pytest.approx(onp.rv_diagnostic(hb.X[2].T, hb.V[2].T, hb.t[2], opot.value, B=31), rel=1e-10)


def test_sample_skeleton_with_diagnostic_online_equals_offline(p):
    """test/test_diagnostics.jl:126-143: ForwardECMCAD(3, |x|^2/2, grid_size=8, tmax=1, adaptive=false), T = 3, B = 20,
    seed = 42: the online value equals RV_diagnostic(history; B = 20) to rtol 1e-10; ragged batches; the Boomerang
    variant follows its rotation flow (checked against a direct evaluation)."""
    import pdmp_oracle_np as onp
    dim = 3
    s = p.ForwardECMCAD(dim, p.GaussStd(), grid_size=8, tmax=1.0, adaptive=False)
    xinit = np.zeros(dim); vinit = np.ones(dim) / np.sqrt(dim)
    hist, rv_online = p.sample_skeleton_with_diagnostic(s, 3.0, xinit, vinit, B=20, seed=42, verbose=False)
    assert hist.t[-1] == 3.0
    rv_offline = p.RV_diagnostic(hist, p.GaussStd(), B=20)
    assert rv_online == pytest.approx(rv_offline, rel=1e-10, abs=1e-12)
    assert rv_online == pytest.approx(onp.rv_diagnostic(hist.X, hist.V, hist.t, onp.GaussStd().value, B=20), rel=1e-10)
    # ragged batch: every chain ends at T with its own number of events
    g = np.random.default_rng(2)
    hs, rvs = p.sample_skeleton_with_diagnostic(s, 40.0, g.standard_normal((5, dim)), np.tile(vinit, (5, 1)), B=20, seed=7)
    assert len({h.t.shape[0] for h in hs}) > 1 and rvs.shape == (5,)
    for h, r in zip(hs, rvs):
        assert r == pytest.approx(onp.rv_diagnostic(h.X, h.V, h.t, onp.GaussStd().value, B=20), rel=1e-10)
    # Boomerang: online value goes through the rotation flow
    sb = p.Boomerang(dim, p.GaussDiag(np.array([0.5, 1.0, 2.0])), refresh_rate=0.5)
    hbm, rvb = p.sample_skeleton_with_diagnostic(sb, 4.0, np.array([0.3, -0.2, 0.1]), np.array([1.0, 0.5, -0.7]), B=16, seed=3)
    U = onp.GaussDiag(np.array([0.5, 1.0, 2.0])).value
    tb = onp.grid_times(4.0, 17)
    idx = np.searchsorted(hbm.t, tb, side="right") - 1
    tau = tb - hbm.t[idx]
    pos = hbm.X[:, idx] * np.cos(tau) + hbm.V[:, idx] * np.sin(tau)
    vals = np.array([U(pos[:, k]) for k in range(17)])
    vals[0] = U(hbm.X[:, 0])
    assert rvb == pytest.approx(np.sum(np.diff(vals) ** 2) / 4.0, rel=1e-10)
    with pytest.raises(p.ArgumentError):
        p.sample_skeleton_with_diagnostic(s, -1.0, xinit, vinit, B=20)


def test_edge_sizes_match_oracle(p):
    """Smallest and largest shapes the path accepts: n_sk = 1 (the initial column only, src/sample.jl:266-268), d = 1,
    grid_size = 2 (smallest valid; 1 indexes t[2] out of bounds upstream, UpperBound.jl:95,205) and 64 (device maximum),
    a single chain and a chain count that is not a multiple of any team/CTA packing."""
    g = np.random.default_rng(4)
    # n_sk = 1: one column = the initial state, zero statistics, no draws consumed
    s = p.BPS(4, p.GaussStd())
    x0 = g.standard_normal((3, 4)); v0 = g.standard_normal((3, 4))
    h = p.sample_skeleton(s, 1, x0, v0, seed=1)
    assert np.array_equal(h.X[:, 0], x0) and np.array_equal(h.V[:, 0], v0) and np.all(h.t == 0.0)
    assert not h.rejected.any() and not h.hitting_horizon.any() and not h.errored_bound.any()
    # grid sizes 2 and 64, teacher-free short runs against the C oracle with an injected tape
    for (sk, d, G, nch) in ((0, 1, 2, 1), (0, 5, 64, 7), (1, 3, 2, 5), (1, 6, 64, 3), (3, 1, 64, 2), (2, 2, 2, 3)):
        name = "edge_%d_%d_%d" % (sk, d, G)
        xg, vg, tape = case_inputs(name, sk, d, 60, n_chains=nch)
        kw = dict(grid_size=G, **({1: dict(tmax=1.0, refresh_rate=0.1), 3: dict(tmax=1.0, refresh_rate=0.1)}.get(sk, {})))
        r = oc.sample_skeleton(oc.make_cfg(sk, 0, d, np.zeros(0), **kw), 60, xg, vg, tape=tape)
        hg = p.sample_skeleton(make_sampler(p, sk, 0, np.zeros(0), d, kw), 60, xg, vg, tape=tape)
        ok = r.status == 0
        assert ok.any(), name
        assert np.array_equal(hg.status == 0, ok), name
        assert relerr(hg.X[ok], r.X[ok]) < 1e-9 and relerr(hg.t[ok], r.t[ok]) < 1e-9, name
        assert np.array_equal(hg.rejected[ok], r.rejected[ok]) and np.array_equal(hg.hitting_horizon[ok], r.hitting_horizon[ok]), name
    with pytest.raises(p.ArgumentError):
        p.ZigZag(3, p.GaussStd(), grid_size=1)
    with pytest.raises(p.UnsupportedError):
        p.ZigZag(3, p.GaussStd(), grid_size=65)


@pytest.mark.parametrize("d", [20, 36, 60, 70, 90, 128])
def test_logreg_every_mma_work_split(p, d):
    """The logistic-regression kernel is compiled once per (whole m-tiles per warp, split last tile) combination
    (logreg.cu: lr_consume); d = 5, 8, 13, 100 are covered by the cases above, these dimensions reach the other
    variants (d = 128 also runs with the shallower X ring).  Free-running parity against the C oracle."""
    from oracle_cases import logreg_data
    n, n_sk, nch = 150, 40, 3
    X, y, s0 = logreg_data(n, d)
    pp = np.concatenate([[float(n), s0], X.ravel(), y])
    x0, v0, tape = case_inputs("logreg_split%d" % d, 0, d, n_sk, n_chains=nch)
    r = oc.sample_skeleton(oc.make_cfg(0, 5, d, pp, grid_size=5), n_sk, x0, v0, tape=tape)
    h = p.sample_skeleton(p.ZigZagAD(d, p.LogReg(X, y, s0), grid_size=5), n_sk, x0, v0, tape=tape)
    assert (r.status == 0).all()
    assert relerr(h.X, r.X) < 1e-9 and relerr(h.t, r.t) < 1e-9 and np.array_equal(h.V, r.V)
    assert np.array_equal(h.rejected, r.rejected) and np.array_equal(h.hitting_horizon, r.hitting_horizon)


def test_logreg_zw_cache_matches_recompute(p):
    """The cached / incrementally updated (z, w) = (X x, X v) rows (logreg.cu: lr_produce) against recomputing them by
    DMMA in every pass: same skeleton to 1e-10 over several hundred events (long enough to cross the periodic exact
    refresh), identical discrete decisions."""
    from oracle_cases import logreg_data
    n, d, n_sk, nch = 333, 21, 500, 9
    X, y, s0 = logreg_data(n, d)
    g = np.random.default_rng(12)
    x0 = 0.3 * g.standard_normal((nch, d)); v0 = np.where(g.random((nch, d)) < 0.5, -1.0, 1.0)
    outs = []
    for off in ("0", "1"):
        os.environ["PDMPFLUX_LOGREG_NO_ZW_CACHE"] = off
        try:
            s = p.ZigZagAD(d, p.LogReg(X, y, s0), grid_size=7)
            outs.append(p.sample_skeleton(s, n_sk, x0, v0, seed=99))
        finally:
            os.environ.pop("PDMPFLUX_LOGREG_NO_ZW_CACHE")
    a, b = outs
    assert relerr(a.X, b.X) < 1e-10 and relerr(a.t, b.t) < 1e-10 and np.array_equal(a.V, b.V)
    assert np.array_equal(a.rejected, b.rejected) and np.array_equal(a.hitting_horizon, b.hitting_horizon)


@pytest.mark.parametrize("d,nch,n_sk", [(50, 37, 300), (7, 5, 129), (33, 3, 64), (1, 4, 40)])
def test_zigzag_sign_bit_transfer_is_bit_identical(p, d, nch, n_sk):
    """Host-buffer path of Zig-Zag: the V rows cross PCIe as sign bits and are rebuilt by worker threads as
    copysign(|vinit_i|, bit) (api.cu: pack_signs_kernel).  Must give exactly the bytes of the plain copy: arbitrary
    velocity magnitudes, -0.0, odd d (unaligned rows), many small slices, the time-horizon variant."""
    g = np.random.default_rng(d)
    x0 = g.standard_normal((nch, d))
    v0 = g.standard_normal((nch, d)) * np.where(g.random((nch, d)) < 0.2, 3.0, 1.0)
    v0[0, 0] = -0.0 if d > 1 else v0[0, 0]
    s = p.ZigZagAD(d, p.GaussStd())
    outs = []
    for forced in ("1", "0"):
        os.environ["PDMPFLUX_VBITS"] = forced
        os.environ["PDMPFLUX_SLAB_BYTES"] = str(1 << 16)
        os.environ["PDMPFLUX_HOST_THREADS"] = "3"
        try:
            outs.append((p.sample_skeleton(s, n_sk, x0, v0, seed=31), p.sample_skeleton(s, 2.5, x0, v0, seed=31)))
        finally:
            for k in ("PDMPFLUX_VBITS", "PDMPFLUX_SLAB_BYTES", "PDMPFLUX_HOST_THREADS"):
                os.environ.pop(k)
    (a, ta), (b, tb) = outs
    for f in ("horizon", "ar", "error_value_ar", "errored_bound", "rejected", "hitting_horizon"):
        assert getattr(a, f).tobytes() == getattr(b, f).tobytes(), f
    assert a.V.tobytes() == b.V.tobytes() and a.X.tobytes() == b.X.tobytes() and np.array_equal(a.t, b.t)
    assert np.array_equal(np.abs(a.V), np.broadcast_to(np.abs(v0)[:, None, :], a.V.shape))
    for ha, hb in zip(ta, tb):
        assert ha.V.tobytes() == hb.V.tobytes() and np.array_equal(ha.t, hb.t)


def test_zero_slices_of_error_columns_stay_on_device(p):
    """Host-buffer path of Zig-Zag: slices whose errored_bound column is all zero are not copied (their error_value_ar /
    errored_bound rows are zero-filled on the host); slices with a violated bound are.  A coarse 2-node grid on the
    banana violates its bound now and then, so both kinds of slices occur; every column must equal the plain path."""
    d, nch, n_sk = 4, 11, 600
    g = np.random.default_rng(5)
    x0 = g.standard_normal((nch, d)); v0 = np.where(g.random((nch, d)) < 0.5, -1.0, 1.0)
    s = p.ZigZagAD(d, p.Banana(), grid_size=2, tmax=3.0, adaptive=False)
    outs = []
    for forced in ("1", "0"):
        os.environ["PDMPFLUX_VBITS"] = forced
        os.environ["PDMPFLUX_SLAB_BYTES"] = str(1 << 14)
        try:
            outs.append(p.sample_skeleton(s, n_sk, x0, v0, seed=4))
        finally:
            os.environ.pop("PDMPFLUX_VBITS"); os.environ.pop("PDMPFLUX_SLAB_BYTES")
    a, b = outs
    assert a.errored_bound.any() and not a.errored_bound.all()
    cols_with = a.errored_bound.any(axis=0)
    assert cols_with.any() and not cols_with.all()
    for f in ("X", "V", "t", "horizon", "ar", "error_value_ar", "errored_bound", "rejected", "hitting_horizon"):
        assert getattr(a, f).tobytes() == getattr(b, f).tobytes(), f


def test_rv_diagnostic_logistic_regression(p):
    """RV_diagnostic with the logistic-regression U plugin (a pass over X per block boundary) against the oracle."""
    import pdmp_oracle_np as onp
    from oracle_cases import logreg_data
    n, d, nch, n_sk = 157, 9, 4, 200
    X, y, s0 = logreg_data(n, d)
    g = np.random.default_rng(6)
    s = p.ZigZagAD(d, p.LogReg(X, y, s0), grid_size=6)
    hb = p.sample_skeleton(s, n_sk, 0.2 * g.standard_normal((nch, d)), np.where(g.random((nch, d)) < 0.5, -1.0, 1.0), seed=8)
    opot = onp.LogReg(X, y, s0)
    for B in (0, 23):
        rv = p.RV_diagnostic(hb, s.potential, B=B)
        ref = np.array([onp.rv_diagnostic(hb.X[c].T, hb.V[c].T, hb.t[c], opot.value, B=B) for c in range(nch)])
        assert np.allclose(rv, ref, rtol=1e-9, atol=0), (B, rv, ref)


def test_logreg_work_queue_matches_static_assignment(p):
    """With more chains than 4 x SMs the logistic-regression kernel runs persistent CTAs whose warps pull chains from
    a work queue (logreg.cu).  Which warp ran a chain must not matter: a 1500-chain run equals the same chains run in
    shards small enough for the static assignment, bit for bit, including a second launch (resume) and the
    time-horizon variant with its ragged column counts."""
    from oracle_cases import logreg_data
    n, d, nch, n_sk = 96, 5, 1500, 9
    X, y, s0 = logreg_data(n, d)
    g = np.random.default_rng(13)
    x0 = 0.3 * g.standard_normal((nch, d)); v0 = np.where(g.random((nch, d)) < 0.5, -1.0, 1.0)
    s = p.ZigZagAD(d, p.LogReg(X, y, s0), grid_size=4)
    big = p.sample_skeleton(s, n_sk, x0, v0, seed=77)
    for lo in (0, 500, 1000):
        part = p.sample_skeleton(s, n_sk, x0[lo:lo + 500], v0[lo:lo + 500], seed=77, chain_offset=lo)
        for f in ("X", "V", "t", "horizon", "ar", "rejected", "hitting_horizon", "errored_bound"):
            assert np.array_equal(getattr(big, f)[lo:lo + 500], getattr(part, f)), (lo, f)
    assert (big.status == 0).all() and np.all(np.diff(big.t, axis=1) > 0)
    T = float(np.median(big.t[:, -1]))
    hs = p.sample_skeleton(s, T, x0, v0, seed=77)
    hp = p.sample_skeleton(s, T, x0[700:1000], v0[700:1000], seed=77, chain_offset=700)
    assert len({h.t.shape[0] for h in hs}) > 1
    for a, b in zip(hs[700:1000], hp):
        assert a.t.shape == b.t.shape and np.array_equal(a.X, b.X) and a.t[-1] == T
