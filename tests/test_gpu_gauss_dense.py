"""GaussDense on the GPU: injected-draw parity against the C oracle (Zig-Zag grid / Brent, BPS grid / Brent, teams of 8
and 32, ragged ownership), agreement with the structured Gaussians it generalises, bit-exact slicing and sharding, the
time-horizon variant and fused moments, and the sampled mean / covariance of a d = 50 target."""
import os

import numpy as np
import pytest

import oracle_c as oc
from conftest import record_parity_error
from oracle_cases import case_inputs
from test_gauss_dense_cpu import dense_case, oracle_skeleton, oracle_skeleton_until, relerr

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def p():
    import ctypes
    import pdmpflux_b200
    n = ctypes.c_int(0)
    pdmpflux_b200.lib().pdmpflux_device_count(ctypes.byref(n))
    assert n.value > 0, "GPU tests need a CUDA device"
    return pdmpflux_b200


# name, sampler, config kwargs (oracle spelling)
CONFIGS = [
    ("zz_grid", oc.ZIGZAG, dict(grid_size=10)),
    ("zz_brent", oc.ZIGZAG, dict(grid_size=0)),
    ("bps_grid", oc.BPS, dict(tmax=1.0, refresh_rate=0.3)),
    ("bps_brent_gv", oc.BPS, dict(tmax=1.0, refresh_rate=0.3, grid_size=0, gaussian_velocity=True)),
]


def make_sampler(p, sampler, d, P, mu, kw):
    kw = dict(kw)
    pot = p.GaussDense(P, mu)
    if sampler == oc.ZIGZAG:
        return p.ZigZag(d, pot, AD_backend="ForwardDiff", **kw)
    if "gaussian_velocity" in kw:
        kw["Gaussian_velocity"] = kw.pop("gaussian_velocity")
    return p.BPS(d, pot, AD_backend="ForwardDiff", **kw)


def free_running(p, name, sampler, kw, d, n_sk, nch=2, seed=0):
    P, mu = dense_case(d, seed=seed)
    x0, v0, (E, U, N) = case_inputs(f"dense_{name}_{d}", sampler, d, n_sk, n_chains=nch)
    x0 = x0 + mu
    r = oracle_skeleton(sampler, P, mu, kw, n_sk, x0, v0, (E, U, N))
    assert (r.status == 0).all()
    h = p.sample_skeleton(make_sampler(p, sampler, d, P, mu, kw), n_sk, x0, v0, tape=(E, U, N))
    assert (h.status == 0).all()
    ex = max(relerr(h.X[c], r.X[c]) for c in range(nch))
    et = max(relerr(h.t[c], r.t[c]) for c in range(nch))
    ev = max(relerr(h.V[c], r.V[c]) for c in range(nch))
    if sampler == oc.ZIGZAG:
        assert np.array_equal(h.V, r.V)
    else:
        assert np.array_equal(np.sign(h.V), np.sign(r.V))
    assert np.array_equal(h.rejected, r.rejected) and np.array_equal(h.hitting_horizon, r.hitting_horizon)
    assert np.array_equal(h.tape_pos, r.tape_used)
    return ex, et, ev


@pytest.mark.parametrize("d", [5, 33, 100, 300])
@pytest.mark.parametrize("cfg", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_parity_with_oracle(p, cfg, d):
    name, sampler, kw = cfg
    if sampler == oc.BPS and d == 5:
        # In so few dimensions every BPS bounce turns v by a large angle and a free run amplifies rounding about tenfold
        # every ten events (measured on a B200: 1e-15 at event 20, 1e-8 by event 60 on one chain, 4e-3 at 160 on
        # another; alike for teams of 8 and 32 and for d = 6 .. 9).  test_one_step_parity_with_oracle holds every
        # transition of this case to 1e-9.
        pytest.skip("BPS at d = 5 is chaotic: free runs diverge from rounding; covered event by event by the one-step test")
    n_sk = 300 if d <= 100 else 120
    ex, et, ev = free_running(p, name, sampler, kw, d, n_sk)
    record_parity_error(f"gauss_dense/{name}/d{d}", x=ex, t=et, v=ev, events=n_sk - 1, tol=1e-9)
    assert max(ex, et, ev) < 1e-9, dict(x=ex, t=et, v=ev)


@pytest.mark.parametrize("d", [5, 33, 100, 300])
@pytest.mark.parametrize("cfg", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_one_step_parity_with_oracle(p, cfg, d):
    """Teacher-forced: every event k is regenerated on the device from the oracle's state k-1 (g and h recomputed from
    it by chains_create) and its tape cursor."""
    name, sampler, kw = cfg
    n_sk = 200 if d <= 100 else 80
    P, mu = dense_case(d)
    x0, v0, (E, U, N) = case_inputs(f"dense1_{name}_{d}", sampler, d, n_sk)
    x0 = x0 + mu
    r = oracle_skeleton(sampler, P, mu, kw, n_sk, x0, v0, (E, U, N))
    assert r.status[0] == 0
    pos = r.tape_pos[0]
    use = np.diff(pos, axis=0)
    w = [int(use[:, i].max()) + 1 for i in range(3)]
    tapes = [np.concatenate([a[0], np.ones(wi)])[pos[:-1, i][:, None] + np.arange(wi)[None, :]]
             for i, (a, wi) in enumerate(zip((E, U, N), w))]
    h = p.sample_skeleton(make_sampler(p, sampler, d, P, mu, kw), 2, r.X[0, :-1], r.V[0, :-1], tape=tuple(tapes),
                          t0=r.t[0, :-1], horizon0=r.horizon[0, :-1], batch=True)
    ex = (np.abs(h.X[:, 1] - r.X[0, 1:]).max(axis=1) / np.abs(r.X[0, 1:]).max(axis=1)).max()
    ev = (np.abs(h.V[:, 1] - r.V[0, 1:]).max(axis=1) / np.abs(r.V[0, 1:]).max(axis=1)).max()
    dt = r.t[0, 1:] - r.t[0, :-1]
    et = (np.abs((h.t[:, 1] - h.t[:, 0]) - dt) / dt).max()
    record_parity_error(f"gauss_dense_one_step/{name}/d{d}", x=ex, t=et, v=ev, tol=1e-9)
    assert max(ex, et, ev) < 1e-9, dict(x=ex, t=et, v=ev)
    assert np.array_equal(np.sign(h.V[:, 1]), np.sign(r.V[0, 1:]))
    assert np.array_equal(h.rejected[:, 1], r.rejected[0, 1:]) and np.array_equal(h.hitting_horizon[:, 1], r.hitting_horizon[0, 1:])


@pytest.mark.parametrize("cfg", [CONFIGS[0], CONFIGS[2]], ids=["zz_grid", "bps_grid"])
def test_long_run_drift(p, cfg):
    """g = P (x - mu) and h = P v are updated incrementally on the device and recomputed by the oracle: 5000 events bound
    the drift."""
    name, sampler, kw = cfg
    ex, et, ev = free_running(p, name, sampler, kw, 40, 5001, nch=1, seed=7)
    record_parity_error(f"gauss_dense/{name}/d40_long", x=ex, t=et, v=ev, events=5000, tol=1e-8)
    assert max(ex, et, ev) < 1e-8, dict(x=ex, t=et, v=ev)


def test_team_and_generic_requests_fall_back(p):
    """There is no thread-per-chain or generic kernel for the dense Gaussian: PDMPFLUX_TEAM=1 and
    PDMPFLUX_FORCE_GENERIC=1 run the default kernels, bit for bit."""
    d, nch = 12, 20
    P, mu = dense_case(d, seed=2)
    g = np.random.default_rng(1)
    x0 = g.standard_normal((nch, d)); v0 = np.where(g.random((nch, d)) < 0.5, -1.0, 1.0)
    for grid_size in (0, 10):
        s = p.ZigZagAD(d, p.GaussDense(P, mu), grid_size=grid_size)
        h = p.sample_skeleton(s, 200, x0, v0, seed=4)
        os.environ["PDMPFLUX_TEAM"] = "1"; os.environ["PDMPFLUX_FORCE_GENERIC"] = "1"
        try:
            h1 = p.sample_skeleton(s, 200, x0, v0, seed=4)
        finally:
            os.environ.pop("PDMPFLUX_TEAM"); os.environ.pop("PDMPFLUX_FORCE_GENERIC")
        assert np.array_equal(h.X, h1.X) and np.array_equal(h.t, h1.t)


def test_agrees_with_structured_gaussians(p):
    """GaussDense(diag(p)) follows GaussDiag(p), GaussDense of the equicorrelated precision follows GaussEquicorr: the
    same arithmetic up to reassociation, so the paths agree to rounding (not bits)."""
    d, nch, n_sk = 33, 8, 200
    g = np.random.default_rng(9)
    x0 = g.standard_normal((nch, d))
    vz = np.where(g.random((nch, d)) < 0.5, -1.0, 1.0)
    vb = g.standard_normal((nch, d)); vb /= np.linalg.norm(vb, axis=1, keepdims=True)
    prec = np.linspace(0.5, 2.0, d)
    rho = 0.5
    alpha = 1.0 / (1.0 - rho); beta = rho / ((1.0 - rho) * (1.0 - rho + d * rho))
    Peq = alpha * np.eye(d) - beta * np.ones((d, d))
    worst = {}
    for tag, dense, ref in (("diag", p.GaussDense(np.diag(prec)), p.GaussDiag(prec)),
                            ("equicorr", p.GaussDense(Peq), p.GaussEquicorr(rho))):
        for sname, mk, v0 in (("zz_grid", lambda pot: p.ZigZagAD(d, pot), vz),
                              ("zz_brent", lambda pot: p.ZigZag(d, pot, grid_size=0), vz),
                              ("bps", lambda pot: p.BPS(d, pot, refresh_rate=0.3), vb)):
            a = p.sample_skeleton(mk(dense), n_sk, x0, v0, seed=3)
            b = p.sample_skeleton(mk(ref), n_sk, x0, v0, seed=3)
            e = max(relerr(a.X, b.X), relerr(a.t, b.t), relerr(a.V, b.V))
            worst[f"{tag}/{sname}"] = e
            assert np.array_equal(a.rejected, b.rejected) and np.array_equal(np.sign(a.V), np.sign(b.V))
            assert e < 1e-10, (tag, sname, e)
    record_parity_error("gauss_dense/structured", **worst)


def test_slicing_and_sharding_are_bit_identical(p):
    import torch
    d, nch, n_ev = 70, 24, 300
    P, mu = dense_case(d, seed=5)
    g = np.random.default_rng(6)
    x0 = g.standard_normal((nch, d))
    vz = np.where(g.random((nch, d)) < 0.5, -1.0, 1.0)
    vb = g.standard_normal((nch, d)); vb /= np.linalg.norm(vb, axis=1, keepdims=True)
    dev, f64 = torch.device("cuda"), torch.float64
    for s, v0 in ((p.ZigZag(d, p.GaussDense(P, mu), grid_size=0), vz), (p.ZigZagAD(d, p.GaussDense(P, mu)), vz),
                  (p.BPS(d, p.GaussDense(P, mu), refresh_rate=0.4), vb)):
        outs = []
        for cuts in ((n_ev,), (37, 100, 163)):
            ch = p.DeviceChains(s, x0, v0, seed=11)
            X = torch.empty((nch, n_ev + 1, d), dtype=f64, device=dev); V = torch.empty_like(X)
            t = torch.empty((nch, n_ev + 1), dtype=f64, device=dev)
            view = p.device_history_view(n_ev + 1, X=X, V=V, t=t)
            ch.record(view, 0)
            col = 1
            for n in cuts:
                ch.advance(n, view, col)
                col += n
            torch.cuda.synchronize()
            outs.append((X.cpu().numpy(), V.cpu().numpy(), t.cpu().numpy()) + tuple(ch.get_state()))
            ch.close()
        for a, b in zip(*outs):
            assert np.array_equal(a, b)
        # Philox streams keyed by the global chain id: a shard reproduces its chains of the big run
        h = p.sample_skeleton(s, 120, x0, v0, seed=13)
        hs = p.sample_skeleton(s, 120, x0[5:9], v0[5:9], seed=13, chain_offset=5)
        assert np.array_equal(hs.X, h.X[5:9]) and np.array_equal(hs.V, h.V[5:9]) and np.array_equal(hs.t, h.t[5:9])


@pytest.mark.parametrize("sampler", [oc.ZIGZAG, oc.BPS], ids=["zigzag", "bps"])
def test_time_horizon_variant_and_fused_moments(p, sampler):
    import torch
    d, nch, T = 20, 6, 6.0
    P, mu = dense_case(d, seed=8)
    kw = dict(grid_size=10) if sampler == oc.ZIGZAG else dict(tmax=1.0, refresh_rate=0.3)
    g = np.random.default_rng(12)
    x0 = mu + 0.3 * g.standard_normal((nch, d))
    if sampler == oc.ZIGZAG:
        v0 = np.where(g.random((nch, d)) < 0.5, -1.0, 1.0)
    else:
        v0 = g.standard_normal((nch, d)); v0 /= np.linalg.norm(v0, axis=1, keepdims=True)
    s = make_sampler(p, sampler, d, P, mu, kw)
    E = g.standard_exponential((nch, 20000)); U = g.random((nch, 20000)); N = g.standard_normal((nch, 4000 * d))
    r = oracle_skeleton_until(sampler, P, mu, kw, T, 5000, x0, v0, (E, U, N))
    assert (r.status == 0).all() and (r.ncols >= 2).all()
    hs = p.sample_skeleton(s, T, x0, v0, tape=(E, U, N), batch=True)
    assert [len(h) for h in hs] == r.ncols.tolist()
    for c, h in enumerate(hs):
        n = r.ncols[c]
        assert h.t[-1] == T
        assert relerr(h.X.T, r.X[c, :n]) < 1e-9 and relerr(h.t, r.t[c, :n]) < 1e-9 and relerr(h.V.T, r.V[c, :n]) < 1e-9
    xs = p.sample_from_skeleton(s, 50, hs[0])
    assert xs.shape == (d, 50) and np.isfinite(xs).all()
    # fused moments across two advance() calls equal the closed-form integrals over the stored skeleton
    n_ev = 400
    ch = p.DeviceChains(s, x0, v0, seed=21)
    ch.enable_moments()
    dev, f64 = torch.device("cuda"), torch.float64
    X = torch.empty((nch, n_ev + 1, d), dtype=f64, device=dev); V = torch.empty_like(X)
    t = torch.empty((nch, n_ev + 1), dtype=f64, device=dev)
    view = p.device_history_view(n_ev + 1, X=X, V=V, t=t)
    ch.record(view, 0)
    ch.advance(150, view, 1)
    ch.advance(n_ev - 150, view, 151)
    torch.cuda.synchronize()
    m1, m2 = ch.moments()
    hb = p.PDMPHistoryBatch(nch, n_ev + 1, d)
    hb.X[:] = X.cpu().numpy(); hb.V[:] = V.cpu().numpy(); hb.t[:] = t.cpu().numpy()
    r1, r2, TT = p.skeleton_moments(s, hb)
    assert np.allclose(m1, r1 * TT[:, None], rtol=1e-10, atol=1e-10)
    assert np.allclose(m2, r2 * TT[:, None], rtol=1e-10, atol=1e-10)
    ch.close()


@pytest.mark.parametrize("sampler", [oc.ZIGZAG, oc.BPS], ids=["zigzag", "bps"])
def test_statistics_d50(p, sampler):
    """4096 Philox chains started in the target (x0 ~ N(mu, inv(P))): per-chain time averages (fused moments) give the
    pooled mean and marginal variances, 256 chains' skeletons (sample_from_skeleton) three covariances.  Each estimate
    must lie within 6 standard errors of the truth, the standard error taken over the chains' own estimates."""
    d, nch, n_ev = 50, 4096, 3000
    P, mu = dense_case(d, seed=21)
    Sigma = np.linalg.inv(P)
    L = np.linalg.cholesky(Sigma)
    g = np.random.default_rng(31)
    x0 = mu + g.standard_normal((nch, d)) @ L.T
    if sampler == oc.ZIGZAG:
        s = p.ZigZagAD(d, p.GaussDense(P, mu))
        v0 = np.where(g.random((nch, d)) < 0.5, -1.0, 1.0)
    else:
        s = p.BPS(d, p.GaussDense(P, mu), refresh_rate=1.0)
        v0 = g.standard_normal((nch, d)); v0 /= np.linalg.norm(v0, axis=1, keepdims=True)
    ch = p.DeviceChains(s, x0, v0, seed=2024)
    ch.enable_moments()
    ch.advance(n_ev)
    ch.status()
    m1, m2 = ch.moments()
    _, _, T, _ = ch.get_state()
    ch.close()
    mc, sc = m1 / T[:, None], m2 / T[:, None]          # per-chain time averages of x_i and x_i^2
    mean, se_mean = mc.mean(0), mc.std(0, ddof=1) / np.sqrt(nch)
    assert np.all(np.abs(mean - mu) < 6 * se_mean), np.abs(mean - mu) / se_mean
    vc = sc - 2 * mu * mc + mu * mu                     # per-chain averages of (x_i - mu_i)^2
    var, se_var = vc.mean(0), vc.std(0, ddof=1) / np.sqrt(nch)
    assert np.all(np.abs(var - np.diag(Sigma)) < 6 * se_var), np.abs(var - np.diag(Sigma)) / se_var
    # covariances: the most correlated pair and two others, from samples along 256 chains' skeletons
    C = Sigma / np.sqrt(np.outer(np.diag(Sigma), np.diag(Sigma)))
    iu = np.triu_indices(d, 1)
    top = np.argmax(np.abs(C[iu]))
    pairs = [(iu[0][top], iu[1][top]), (0, d - 1), (3, 17)]
    h = p.sample_skeleton(s, 2000, x0[:256], v0[:256], seed=7)
    xs = p.sample_from_skeleton(s, 1000, h) - mu          # (256, 1000, d)
    for i, j in pairs:
        cc = (xs[:, :, i] * xs[:, :, j]).mean(1)
        est, se = cc.mean(), cc.std(ddof=1) / np.sqrt(len(cc))
        assert abs(est - Sigma[i, j]) < 6 * se, (i, j, est, Sigma[i, j], se)
