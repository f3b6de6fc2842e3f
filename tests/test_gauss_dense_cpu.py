"""GaussDense (a Gaussian with a dense precision matrix) without a GPU: constructor validation, the sampler / option
restriction to the fast-path kernels, the ABI value of the kind, and the two CPU oracles against each other on a
dense case with a non-zero mean.

The C oracle's dense Gaussian (`P_GAUSS_DENSE`, params = P row-major) has mean zero.  Every sampler's dynamics commute
with a translation of x (the flows are x + t v, and the rates, bounds and jumps see x only through g = P (x - mu)), so
a run with mean mu is the oracle's run of y = x - mu shifted back by mu: `oracle_skeleton` / `oracle_skeleton_until`.
The numpy restatement with the mean is `NpGaussDense` below."""
import os
import re

import numpy as np
import pytest

import oracle_c as oc
import pdmp_oracle_np as onp
import pdmpflux_b200 as p
from oracle_cases import case_inputs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def random_spd(d, cond=100.0, seed=0):
    """Symmetric positive-definite d x d matrix with condition number `cond` (random eigenvectors)."""
    g = np.random.default_rng([seed, d])
    q, _ = np.linalg.qr(g.standard_normal((d, d)))
    ev = np.geomspace(1.0, cond, d) if d > 1 else np.ones(1)
    P = (q * ev) @ q.T
    return 0.5 * (P + P.T)


def dense_case(d, seed=0):
    P = random_spd(d, seed=seed)
    mu = np.random.default_rng([seed, d, 1]).uniform(-1.0, 1.0, d)
    return P, mu


class NpGaussDense:
    """numpy restatement (the interface of oracle/pdmp_oracle_np.py's potentials): U = (x - mu)' P (x - mu) / 2."""
    kind = 6

    def __init__(self, P, mu):
        self.P = np.asarray(P, dtype=np.float64)
        self.mu = np.asarray(mu, dtype=np.float64)

    def value(self, x):
        y = x - self.mu
        return float(y @ self.P @ y) / 2.0

    def grad(self, x):
        return self.P @ (x - self.mu)

    def hvp(self, x, v):
        return self.P @ v


def oracle_skeleton(sampler, P, mu, kw, n_sk, x0, v0, tape):
    """C oracle skeleton of the dense Gaussian with mean mu (rows of x0 / v0 = chains), positions in x."""
    d = P.shape[0]
    r = oc.sample_skeleton(oc.make_cfg(sampler, oc.GAUSS_DENSE, d, P.ravel(), **kw), n_sk, x0 - mu, v0, tape=tape)
    r.X = r.X + mu
    return r


def oracle_skeleton_until(sampler, P, mu, kw, T, cap, x0, v0, tape):
    d = P.shape[0]
    r = oc.sample_skeleton_until(oc.make_cfg(sampler, oc.GAUSS_DENSE, d, P.ravel(), **kw), T, cap, x0 - mu, v0, tape=tape)
    r.X = r.X + mu
    return r


def test_kind_value_is_seven():
    hdr = open(os.path.join(ROOT, "include", "pdmpflux_cuda.h")).read()
    assert re.search(r"PDMPFLUX_GAUSS_DENSE\s*=\s*7\b", hdr)
    assert re.search(r"PDMPFLUX_SOURCE\s*=\s*6\b", hdr)
    assert p.GaussDense(np.eye(2)).kind == 7
    assert oc.GAUSS_DENSE == 6   # the oracle keeps its own numbering


def test_constructor_validation():
    P, mu = dense_case(5)
    with pytest.raises(p.ArgumentError, match="square"):
        p.GaussDense(np.ones((3, 4)))
    with pytest.raises(p.ArgumentError, match="square"):
        p.GaussDense(np.ones(4))
    with pytest.raises(p.DimensionMismatch):
        p.ZigZag(4, p.GaussDense(P, mu), grid_size=0)
    with pytest.raises(p.DimensionMismatch):
        p.ZigZag(5, p.GaussDense(P, mu[:4]), grid_size=0)
    asym = P.copy()
    asym[0, 1] += 1e-6
    with pytest.raises(p.ArgumentError, match="not symmetric"):
        p.ZigZag(5, p.GaussDense(asym, mu), grid_size=0)
    indef = P.copy()
    indef[2, 2] = -1.0
    with pytest.raises(p.ArgumentError, match="not positive definite"):
        p.BPS(5, p.GaussDense(indef, mu))
    with pytest.raises(p.ArgumentError, match="not positive definite"):
        p.BPS(2, p.GaussDense(np.ones((2, 2))))      # singular
    nan = P.copy()
    nan[1, 3] = nan[3, 1] = np.nan
    with pytest.raises(p.ArgumentError, match="finite"):
        p.BPS(5, p.GaussDense(nan, mu))
    with pytest.raises(p.ArgumentError, match="finite"):
        p.BPS(5, p.GaussDense(P, np.where(np.arange(5) == 2, np.inf, mu)))
    # asymmetry within the tolerance is accepted (the library symmetrises)
    near = P.copy()
    near[0, 1] += 1e-14 * np.abs(P).max()
    assert p.BPS(5, p.GaussDense(near, mu))._handle


def test_dimension_limit():
    with pytest.raises(p.UnsupportedError, match="2048"):
        p.BPS(2049, p.GaussDense(np.eye(2049)))


def test_supported_configurations_construct():
    P, mu = dense_case(6)
    pot = p.GaussDense(P, mu)
    for make in (lambda: p.ZigZag(6, pot, grid_size=0), lambda: p.ZigZag(6, pot, grid_size=0, vectorized_bound=False, signed_bound=False),
                 lambda: p.ZigZagAD(6, pot), lambda: p.ZigZagAD(6, pot, grid_size=4, signed_bound=False),
                 lambda: p.BPS(6, pot), lambda: p.BPS(6, pot, AD_backend="FiniteDiff"), lambda: p.BPS(6, pot, grid_size=0),
                 lambda: p.BPS(6, pot, Gaussian_velocity=True)):
        assert make()._handle


@pytest.mark.parametrize("make, what", [
    (lambda pot: p.ForwardECMC(6, pot), "ForwardECMC"),
    (lambda pot: p.Boomerang(6, pot), "Boomerang"),
    (lambda pot: p.StickyZigZag(6, pot, np.full(6, 0.5)), "StickyZigZag"),
    (lambda pot: p.SpeedUpZigZag(6, pot), "SpeedUpZigZag"),
    (lambda pot: p.ZigZagAD(6, pot, vectorized_bound=False, signed_bound=False), "vectorized_bound=false"),
    (lambda pot: p.ZigZag(6, pot, AD_backend="FiniteDiff"), "FiniteDiff"),
], ids=["fecmc", "boomerang", "sticky", "speedup", "zz_scalar_grid", "zz_grid_fd"])
def test_unsupported_samplers_and_options_raise_at_construction(make, what):
    P, mu = dense_case(6)
    with pytest.raises(p.UnsupportedError, match=what):
        make(p.GaussDense(P, mu))


# name, sampler, dim, config kwargs, n_sk
DENSE_CASES = [
    ("zz_dense7", oc.ZIGZAG, 7, dict(grid_size=10), 300),
    ("zz_dense9_brent", oc.ZIGZAG, 9, dict(grid_size=0), 300),
    ("bps_dense8", oc.BPS, 8, dict(tmax=1.0, refresh_rate=0.2), 300),
    ("bps_dense6_brent_gv", oc.BPS, 6, dict(tmax=1.0, refresh_rate=0.3, grid_size=0, gaussian_velocity=True), 300),
]


def relerr(a, b):
    scale = max(np.max(np.abs(a)), np.max(np.abs(b)), 1e-300)
    return float(np.max(np.abs(a - b)) / scale)


@pytest.mark.parametrize("case", DENSE_CASES, ids=[c[0] for c in DENSE_CASES])
def test_numpy_vs_c_oracle_one_step(case):
    """Teacher-forced: every event of the C oracle is regenerated by the numpy restatement from the previous state."""
    name, sampler, d, kw, n_sk = case
    P, mu = dense_case(d, seed=3)
    x0, v0, (E, U, N) = case_inputs(name, sampler, d, n_sk)
    x0 = x0 + mu
    r = oracle_skeleton(sampler, P, mu, kw, n_sk, x0, v0, (E, U, N))
    assert r.status[0] == oc.ST_OK
    s = onp.Sampler(d, NpGaussDense(P, mu), onp.Config(sampler=sampler, **kw))
    tape = onp.Tape(E[0], U[0], N[0])
    ch = onp.Chain(s, x0[0], v0[0], tape)
    for k in range(1, n_sk):
        st = ch.state
        st.x = r.X[0, k - 1].copy(); st.v = r.V[0, k - 1].copy()
        st.t = float(r.t[0, k - 1]); st.horizon = float(r.horizon[0, k - 1])
        tape.pos = [int(a) for a in r.tape_pos[0, k - 1]]
        st = ch.get_event_state()
        e = max(relerr(st.x, r.X[0, k]), relerr(st.v, r.V[0, k]), abs(st.t - r.t[0, k]) / max(abs(st.t), 1e-300),
                abs(st.horizon - r.horizon[0, k]) / st.horizon, abs(st.ar - r.ar[0, k]))
        assert e < 1e-10, (k, e)
        assert (st.rejected, st.hitting_horizon, st.errored_bound) == \
            (r.rejected[0, k], r.hitting_horizon[0, k], r.errored_bound[0, k]), k
        assert tape.pos == [int(a) for a in r.tape_pos[0, k]], k
