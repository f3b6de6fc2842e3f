"""Source potentials (CudaPotential) that declare a line model, on the device: restated built-ins reproduce the
built-in fast-path kernels bit for bit (every Zig-Zag x Brent line model, the affine-cell grid bound, the O(1) BPS /
ForwardECMC line sums and the fused split reflection) and the C2 digests; two targets with no built-in match the numpy
oracle event by event and their known law in distribution; Boomerang and PDMPFLUX_FORCE_GENERIC keep the generic
kernel."""
import json
import os
import zlib

import numpy as np
import pytest

import pdmp_oracle_np as onp
from conftest import record_parity_error
from oracle_cases import tier_tolerance
from test_gpu_c2_identity import DIGESTS, _run as c2_run
from test_gpu_source_potential import COLUMNS, equicorr_ab, start
from test_source_line_model_cpu import (BANANA_LM_SRC, BANANA_PREC_SRC, GAUSS_DIAG_SPLIT_SRC, LOWRANK_SRC,
                                        equicorr_split_src, lowrank_params)
from test_source_potential_cpu import BANANA_SRC

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def p():
    import ctypes

    import pdmpflux_b200
    n = ctypes.c_int(0)
    pdmpflux_b200.lib().pdmpflux_device_count(ctypes.byref(n))
    assert n.value > 0, "GPU tests need a CUDA device"
    return pdmpflux_b200


def run(p, s, x0, v0, team, n_sk, generic=False, **kw):
    env = {"PDMPFLUX_TEAM": str(team)} if team else {}
    if generic:
        env["PDMPFLUX_FORCE_GENERIC"] = "1"
    os.environ.update(env)
    try:
        return p.sample_skeleton(s, n_sk, x0, v0, **kw)
    finally:
        for k in env:
            os.environ.pop(k)


def same(a, b):
    for col in COLUMNS:
        ca, cb = getattr(a, col, None), getattr(b, col, None)
        if ca is None and cb is None:
            continue
        assert np.array_equal(ca, cb), col


def pots(p, which, d):
    """(built-in, restated source with its line model)"""
    if which == "banana":
        return p.Banana(), p.CudaPotential(BANANA_LM_SRC)
    if which == "diag":
        prec = np.linspace(0.5, 2.0, d)
        return p.GaussDiag(prec), p.CudaPotential(GAUSS_DIAG_SPLIT_SRC, prec)
    return p.GaussEquicorr(0.4), p.CudaPotential(equicorr_split_src(*equicorr_ab(d, 0.4)))


SAMPLERS = {
    "zz_brent": lambda p, d, pot: p.ZigZag(d, pot, grid_size=0, AD_backend="ForwardDiff"),
    "zz_grid": lambda p, d, pot: p.ZigZag(d, pot, AD_backend="ForwardDiff"),
    "bps": lambda p, d, pot: p.BPS(d, pot, AD_backend="ForwardDiff"),
    "bps_brent": lambda p, d, pot: p.BPS(d, pot, grid_size=0, AD_backend="ForwardDiff"),
    "fecmc": lambda p, d, pot: p.ForwardECMC(d, pot, AD_backend="ForwardDiff"),
    "fecmc_brent": lambda p, d, pot: p.ForwardECMC(d, pot, grid_size=0, AD_backend="ForwardDiff"),
}

# (sampler, potential, d, team): Zig-Zag x Brent on every line model -- thread-per-chain compressed (team 1), the
# transposed team search (8, d <= 64), register (8, d = 100) and shared (8, d = 136: 17 owned coordinates) line
# models, a warp per chain (32) -- the affine-cell grid bound, and the BPS / ForwardECMC line sums, split or not
IDENTITY_CASES = [
    ("zz_brent", "banana", 12, 1), ("zz_brent", "banana", 12, 8), ("zz_brent", "banana", 100, 8),
    ("zz_brent", "banana", 136, 8), ("zz_brent", "banana", 12, 32), ("zz_brent", "banana", 50, 8),
    ("zz_grid", "banana", 12, 1), ("zz_grid", "banana", 12, 8), ("zz_grid", "banana", 40, 32),
    ("bps", "banana", 12, 8), ("bps_brent", "banana", 12, 8), ("bps_brent", "banana", 12, 1), ("fecmc", "banana", 12, 8),
]
for _kind in ("bps", "bps_brent", "fecmc", "fecmc_brent"):
    for _which in ("diag", "equicorr"):
        IDENTITY_CASES += [(_kind, _which, 12, 1), (_kind, _which, 12, 8), (_kind, _which, 40, 32)]


@pytest.mark.parametrize("case", IDENTITY_CASES, ids=[f"{a}-{b}-d{c}-t{t}" for a, b, c, t in IDENTITY_CASES])
def test_bit_identical_to_builtin_fast_path(p, case):
    kind, which, d, team = case
    builtin, source = pots(p, which, d)
    n = 256
    x0, v0 = start(d, n, zlib.crc32(f"{kind}{which}{d}".encode()))
    if not kind.startswith("zz"):
        v0 = np.random.default_rng(3).standard_normal((n, d))
    a = run(p, SAMPLERS[kind](p, d, builtin), x0, v0, team, 300, seed=77)
    b = run(p, SAMPLERS[kind](p, d, source), x0, v0, team, 300, seed=77)
    same(a, b)
    assert (np.diff(a.t, axis=1) > 0).all()


def test_fast_path_is_taken(p):
    """the declared source does not run the generic kernel: its bits differ from the generic run's (reassociated
    sums), and equal the built-in's on its fast path (above)"""
    d = 12
    x0, v0 = start(d, 256, 1)
    s = SAMPLERS["zz_brent"](p, d, p.CudaPotential(BANANA_LM_SRC))
    fast = run(p, s, x0, v0, 8, 300, seed=5)
    generic = run(p, s, x0, v0, 8, 300, seed=5, generic=True)
    assert not np.array_equal(fast.X, generic.X)


def test_c2_digests(p):
    """the bench workload's inputs (tests/test_gpu_c2_identity.py, c2_team8) with the restated banana"""
    with open(DIGESTS) as f:
        want = json.load(f)["c2_team8"]
    g = np.random.default_rng(20261020)
    nch, n_sk, d = 512, 200, 50
    x0 = g.standard_normal((nch, d))
    v0 = np.where(g.random((nch, d)) < 0.5, -1.0, 1.0)
    got = c2_run(p, p.ZigZag(d, p.CudaPotential(BANANA_LM_SRC), grid_size=0), x0, v0, n_sk, 2024, 8)
    for name, digest in want.items():
        assert got[name] == digest, f"c2_team8: {name} differs from the built-in's recorded digest"


# ---- targets with no built-in: the numpy oracle ------------------------------------------------------------------
class BananaPrec:
    """U = x0^2 / 2 + (x1 - x0^2 + 1)^2 / 2 + sum_{i >= 2} p_i x_i^2 / 2"""

    def __init__(self, prec):
        self.p = np.asarray(prec, dtype=np.float64)

    def value(self, x):
        r = x[1] - x[0] ** 2 + 1.0
        return 0.5 * (x[0] ** 2 + r * r + float(np.sum(self.p[2:] * x[2:] ** 2)))

    def grad(self, x):
        g = self.p * x
        r = x[1] - x[0] ** 2 + 1.0
        g[0] = x[0] - 2.0 * x[0] * r
        g[1] = r
        return g

    def hvp(self, x, v):
        h = self.p * v
        r = x[1] - x[0] ** 2 + 1.0
        h[0] = (1.0 - 2.0 * r + 4.0 * x[0] ** 2) * v[0] - 2.0 * x[0] * v[1]
        h[1] = -2.0 * x[0] * v[0] + v[1]
        return h


class LowRank:
    """U = sum_i p_i (x_i - mu_i)^2 / 2 + |U^T x|^2 / 2"""

    def __init__(self, prec, mu, u):
        self.p, self.mu, self.u = prec, mu, u

    def value(self, x):
        return 0.5 * float(np.sum(self.p * (x - self.mu) ** 2)) + 0.5 * float(np.sum((self.u @ x) ** 2))

    def grad(self, x):
        return self.p * (x - self.mu) + self.u.T @ (self.u @ x)

    def hvp(self, x, v):
        return self.p * v + self.u.T @ (self.u @ v)


def target(which, d):
    """(oracle target, source, params)"""
    if which == "banana_prec":
        prec = np.linspace(0.5, 2.0, d)
        return BananaPrec(prec), BANANA_PREC_SRC, prec
    prec, mu, u, params = lowrank_params(d)
    return LowRank(prec, mu, u), LOWRANK_SRC, params


PARITY_KINDS = {  # name: (oracle sampler kind, oracle config, device constructor)
    "zz_brent": (onp.ZIGZAG, dict(grid_size=0), SAMPLERS["zz_brent"]),
    "zz_grid": (onp.ZIGZAG, dict(), SAMPLERS["zz_grid"]),
    "bps": (onp.BPS, dict(tmax=1.0, refresh_rate=0.1, vectorized_bound=False), SAMPLERS["bps"]),
    "bps_brent": (onp.BPS, dict(grid_size=0, tmax=1.0, refresh_rate=0.1, vectorized_bound=False), SAMPLERS["bps_brent"]),
    "fecmc": (onp.FECMC, dict(), SAMPLERS["fecmc"]),
}
PARITY_CASES = [(k, w, d, t) for w in ("banana_prec", "lowrank")
                for k, d, t in (("zz_brent", 12, 1), ("zz_brent", 12, 8), ("zz_brent", 100, 8), ("zz_grid", 12, 8),
                                ("zz_grid", 12, 1), ("bps", 12, 8), ("bps_brent", 12, 8), ("bps_brent", 12, 1),
                                ("fecmc", 12, 8), ("fecmc", 40, 32))]


@pytest.mark.parametrize("case", PARITY_CASES, ids=[f"{w}-{k}-d{d}-t{t}" for k, w, d, t in PARITY_CASES])
def test_one_step_parity(p, case):
    """Teacher-forced: every event of the oracle's skeleton is regenerated on the GPU from the previous state."""
    kind, which, d, team = case
    okind, kw, make = PARITY_KINDS[kind]
    n_sk = 200
    tgt, src, params = target(which, d)
    g = np.random.default_rng(zlib.crc32(f"{kind}{which}{d}{team}".encode()))
    x0 = 0.6 * g.standard_normal(d)
    v0 = np.where(g.random(d) < 0.5, -1.0, 1.0) if okind == onp.ZIGZAG else g.standard_normal(d)
    E = g.standard_exponential(12 * n_sk); U = g.random(12 * n_sk); N = g.standard_normal(4 * d * n_sk + 8)
    so = onp.Sampler(d, tgt, onp.Config(sampler=okind, **kw))
    tape = onp.Tape(E, U, N)
    ch = onp.Chain(so, x0, v0, tape)
    states, cursors, recs = [(x0.copy(), v0.copy(), 0.0, ch.state.horizon)], [list(tape.pos)], []
    for _ in range(1, n_sk):
        st = ch.get_event_state()
        states.append((st.x.copy(), st.v.copy(), float(st.t), float(st.horizon)))
        cursors.append(list(tape.pos))
        recs.append((float(st.ar), int(st.rejected), int(st.hitting_horizon), int(st.errored_bound)))
    pos = np.array(cursors)
    use = np.diff(pos, axis=0)
    wE, wU, wN = (int(use[:, i].max()) + 1 for i in range(3))
    idx = lambda s0, w: s0[:, None] + np.arange(w)[None, :]
    pad = lambda a, w: np.concatenate([a, np.ones(w)])
    tE, tU, tN = pad(E, wE)[idx(pos[:-1, 0], wE)], pad(U, wU)[idx(pos[:-1, 1], wU)], pad(N, wN)[idx(pos[:-1, 2], wN)]
    X = np.array([q[0] for q in states]); V = np.array([q[1] for q in states])
    T = np.array([q[2] for q in states]); H = np.array([q[3] for q in states])
    s = make(p, d, p.CudaPotential(src, params))
    h = run(p, s, X[:-1], V[:-1], team, 2, tape=(tE, tU, tN), t0=T[:-1], horizon0=H[:-1], batch=True)
    ex = (np.abs(h.X[:, 1] - X[1:]).max(axis=1) / np.maximum(np.abs(X[1:]).max(axis=1), 1e-300)).max()
    ev = (np.abs(h.V[:, 1] - V[1:]).max(axis=1) / np.maximum(np.abs(V[1:]).max(axis=1), 1e-300)).max()
    dt_o = T[1:] - T[:-1]
    et = (np.abs((h.t[:, 1] - h.t[:, 0]) - dt_o) / dt_o).max()
    eh = (np.abs(h.horizon[:, 1] - H[1:]) / H[1:]).max()
    ea = np.abs(h.ar[:, 1] - np.array([r[0] for r in recs])).max()
    tol = tier_tolerance(kw)
    record_parity_error(f"source_line_model_one_step/{which}/{kind}/d{d}/t{team}", x=ex, v=ev, t=et, horizon=eh, ar=ea,
                        tol=tol)
    assert max(ex, ev, et, eh, ea) < tol, dict(x=ex, v=ev, t=et, horizon=eh, ar=ea)
    assert np.array_equal(h.rejected[:, 1], [r[1] for r in recs])
    assert np.array_equal(h.hitting_horizon[:, 1], [r[2] for r in recs])
    assert np.array_equal(h.tape_pos, use)


@pytest.mark.parametrize("kind", ["zz_brent", "bps"])
def test_lowrank_known_answer(p, kind):
    """U = sum_i p_i (x_i - mu_i)^2 / 2 + |U^T x|^2 / 2 is N(m, S) with S = (D + U U^T)^-1, m = S D mu"""
    d, n = 10, 4096
    prec, mu, u, params = lowrank_params(d)
    S = np.linalg.inv(np.diag(prec) + u.T @ u)
    m = S @ (prec * mu)
    sampler = SAMPLERS[kind](p, d, p.CudaPotential(LOWRANK_SRC, params))
    g = np.random.default_rng(1)
    x0 = m + g.standard_normal((n, d)) @ np.linalg.cholesky(S).T
    v0 = np.where(g.random((n, d)) < 0.5, -1.0, 1.0) if kind == "zz_brent" else g.standard_normal((n, d))
    ch = p.DeviceChains(sampler, x0, v0, seed=2024)
    ch.advance(200)                      # burn-in
    t0 = ch.get_state()[2]
    ch.enable_moments()
    ch.advance(2000)
    m1, m2 = ch.moments()
    length = ch.get_state()[2] - t0      # each chain's moment window
    ch.close()
    mean_c, sq_c = m1 / length[:, None], m2 / length[:, None]
    for est, want in ((mean_c, m), (sq_c, np.diag(S) + m * m)):
        se = est.std(axis=0, ddof=1) / np.sqrt(n)
        z = np.abs(est.mean(axis=0) - want) / se
        assert (z < 5).all(), (kind, z, est.mean(axis=0), want)


def test_sharding_and_resume_bit_identical(p):
    """on the thread-per-chain compressed Zig-Zag x Brent kernel"""
    d, n, n_sk = 12, 64, 301
    s = SAMPLERS["zz_brent"](p, d, p.CudaPotential(BANANA_PREC_SRC, np.linspace(0.5, 2.0, d)))
    x0, v0 = start(d, n, 11)
    full = run(p, s, x0, v0, 1, n_sk, seed=5)
    part = run(p, s, x0[20:37], v0[20:37], 1, n_sk, seed=5, chain_offset=20)
    for col in ("X", "V", "t", "horizon", "ar"):
        assert np.array_equal(getattr(full, col)[20:37], getattr(part, col)), col
    k = 150
    first = run(p, s, x0, v0, 1, k + 1, seed=5)
    rest = run(p, s, first.X[:, -1], first.V[:, -1], 1, n_sk - k, seed=5, t0=first.t[:, -1],
               horizon0=first.horizon[:, -1], event0=k)
    for col in ("X", "V", "t", "horizon", "ar"):
        assert np.array_equal(getattr(full, col)[:, k + 1:], getattr(rest, col)[:, 1:]), col


@pytest.mark.parametrize("team", [1, 8])
def test_boomerang_stays_generic(p, team):
    """A declared source on Boomerang runs the generic kernel: a Gaussian with a non-zero mean, whose fast path would
    take <grad U(x), x> as <P x, x>, gives the same bits with and without PDMPFLUX_FORCE_GENERIC"""
    d, n = 12, 128
    params = lowrank_params(d)[3]
    s = p.Boomerang(d, p.CudaPotential(LOWRANK_SRC, params), AD_backend="ForwardDiff")
    x0 = np.random.default_rng(2).standard_normal((n, d)); v0 = np.random.default_rng(3).standard_normal((n, d))
    same(run(p, s, x0, v0, team, 300, seed=9), run(p, s, x0, v0, team, 300, seed=9, generic=True))


@pytest.mark.parametrize("kind", ["zz_brent", "bps"])
def test_force_generic_matches_undeclared(p, kind):
    """PDMPFLUX_FORCE_GENERIC puts a declared source on the kernel an undeclared copy of it runs"""
    d, n = 12, 128
    x0, v0 = start(d, n, 21)
    if kind == "bps":
        v0 = np.random.default_rng(4).standard_normal((n, d))
    for team in (1, 8):
        a = run(p, SAMPLERS[kind](p, d, p.CudaPotential(BANANA_LM_SRC)), x0, v0, team, 300, seed=3, generic=True)
        b = run(p, SAMPLERS[kind](p, d, p.CudaPotential(BANANA_SRC)), x0, v0, team, 300, seed=3)
        same(a, b)


def test_params_share_kernels(p):
    """a second sampler that only changes the parameters compiles nothing"""
    count = p.lib().pdmpflux_jit_compile_count
    src = LOWRANK_SRC + "\n// params test\n"
    d = 12
    p.ZigZag(d, p.CudaPotential(src, lowrank_params(d, 1)[3]), grid_size=0)
    n0 = count()
    s = p.ZigZag(d, p.CudaPotential(src, lowrank_params(d, 2)[3]), grid_size=0)
    h = p.sample_skeleton(s, 20, np.zeros((16, d)), np.ones((16, d)), seed=1)
    assert np.isfinite(h.X).all() and count() == n0
