"""Source potentials (CudaPotential) on the device: restated built-ins are bit-identical to the built-in plugins on the
generic kernel, a target with no built-in matches the numpy oracle event by event and the hyperbolic-secant law in
distribution, and sharding, resume, the compile cache and multi-GPU behave as for the built-ins."""
import os
import zlib

import numpy as np
import pytest

import pdmp_oracle_np as onp
from conftest import record_parity_error
from oracle_cases import tier_tolerance

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def p():
    import ctypes

    import pdmpflux_b200
    n = ctypes.c_int(0)
    pdmpflux_b200.lib().pdmpflux_device_count(ctypes.byref(n))
    assert n.value > 0, "GPU tests need a CUDA device"
    return pdmpflux_b200


# ---- the built-in plugins of csrc/potentials.cuh, restated as user sources --------------------------------------
BANANA_SRC = r"""
struct UserPotential {
    static constexpr int K = 2;
    __device__ static void accum(const pdmpflux::PotParams&, int i, double xi, double* acc) {
        if (i == 0) acc[0] += xi;
        if (i == 1) acc[1] += xi;
    }
    __device__ static double grad(const pdmpflux::PotParams&, int i, double xi, const double* Lx) {
        if (i >= 2) return xi;
        const double x0 = Lx[0], r = Lx[1] - x0 * x0 + 1.0;
        return i == 0 ? x0 - 2.0 * x0 * r : r;
    }
    __device__ static void eval(const pdmpflux::PotParams&, int i, double xi, double di, const double* Lx,
                                const double* Ld, double& g, double& hd) {
        if (i >= 2) { g = xi; hd = di; return; }
        const double x0 = Lx[0], r = Lx[1] - x0 * x0 + 1.0;
        if (i == 0) {
            g = x0 - 2.0 * x0 * r;
            hd = (1.0 - 2.0 * r + 4.0 * x0 * x0) * Ld[0] - 2.0 * x0 * Ld[1];
        } else {
            g = r;
            hd = -2.0 * x0 * Ld[0] + Ld[1];
        }
    }
};
"""

GAUSS_DIAG_SRC = r"""
struct UserPotential {   // params: the d precisions
    static constexpr int K = 0;
    __device__ static void accum(const pdmpflux::PotParams&, int, double, double*) {}
    __device__ static double grad(const pdmpflux::PotParams& pp, int i, double xi, const double*) {
        return __ldg(pp.vec + i) * xi;
    }
    __device__ static void eval(const pdmpflux::PotParams& pp, int i, double xi, double di, const double*, const double*,
                                double& g, double& hd) {
        const double p = __ldg(pp.vec + i);
        g = p * xi; hd = p * di;
    }
};
"""

GAUSS_EQUICORR_SRC = r"""
struct UserPotential {   // params: alpha, beta of P = alpha I - beta 1 1^T
    static constexpr int K = 1;
    __device__ static void accum(const pdmpflux::PotParams&, int, double xi, double* acc) { acc[0] += xi; }
    __device__ static double grad(const pdmpflux::PotParams& pp, int, double xi, const double* Lx) {
        return pp.vec[0] * xi - pp.vec[1] * Lx[0];
    }
    __device__ static void eval(const pdmpflux::PotParams& pp, int, double xi, double di, const double* Lx,
                                const double* Ld, double& g, double& hd) {
        g = pp.vec[0] * xi - pp.vec[1] * Lx[0];
        hd = pp.vec[0] * di - pp.vec[1] * Ld[0];
    }
};
"""

# U = sum_i log cosh(s_i x_i) + c/2 (sum_i x_i)^2 ; params = s[0..d-1], c   (no built-in equivalent)
LOGCOSH_SRC = r"""
struct UserPotential {
    static constexpr int K = 1;
    __device__ static void accum(const pdmpflux::PotParams&, int i, double xi, double* acc) { acc[0] += xi; }
    __device__ static double grad(const pdmpflux::PotParams& pp, int i, double xi, const double* Lx) {
        const double s = pp.vec[i];
        return s * tanh(s * xi) + pp.vec[pp.n - 1] * Lx[0];
    }
    __device__ static void eval(const pdmpflux::PotParams& pp, int i, double xi, double di, const double* Lx,
                                const double* Ld, double& g, double& hd) {
        const double s = pp.vec[i], th = tanh(s * xi), c = pp.vec[pp.n - 1];
        g = s * th + c * Lx[0];
        hd = s * s * (1.0 - th * th) * di + c * Ld[0];
    }
};
"""


def equicorr_ab(d, rho):
    return [1.0 / (1.0 - rho), rho / ((1.0 - rho) * (1.0 - rho + d * rho))]


def pots(p, which, d):
    """(built-in, restated source) for one of the three restated plugins"""
    if which == "banana":
        return p.Banana(), p.CudaPotential(BANANA_SRC)
    if which == "diag":
        prec = np.linspace(0.5, 2.0, d)
        return p.GaussDiag(prec), p.CudaPotential(GAUSS_DIAG_SRC, prec)
    return p.GaussEquicorr(0.4), p.CudaPotential(GAUSS_EQUICORR_SRC, equicorr_ab(d, 0.4))


SAMPLERS = {
    "zz_jvp": lambda p, d, pot: p.ZigZag(d, pot, AD_backend="ForwardDiff"),
    "zz_fd": lambda p, d, pot: p.ZigZag(d, pot, AD_backend="FiniteDiff"),
    "zz_brent": lambda p, d, pot: p.ZigZag(d, pot, grid_size=0, AD_backend="ForwardDiff"),
    "bps": lambda p, d, pot: p.BPS(d, pot, AD_backend="ForwardDiff"),
    "fecmc": lambda p, d, pot: p.ForwardECMC(d, pot, AD_backend="ForwardDiff"),
    "boomerang": lambda p, d, pot: p.Boomerang(d, pot, AD_backend="ForwardDiff"),
    "sticky": lambda p, d, pot: p.StickyZigZag(d, pot, np.full(d, 0.7), AD_backend="ForwardDiff"),
    "speedup": lambda p, d, pot: p.SpeedUpZigZag(d, pot, AD_backend="ForwardDiff"),
}

# every sampler, every restated plugin, d = 12 (all three team widths) and d = 40 (teams of 8 and 32)
IDENTITY_CASES = [
    ("zz_jvp", "banana", 12), ("zz_fd", "banana", 12), ("zz_brent", "diag", 12), ("bps", "equicorr", 12),
    ("fecmc", "banana", 12), ("boomerang", "diag", 12), ("sticky", "equicorr", 12), ("speedup", "banana", 12),
    ("zz_jvp", "equicorr", 40),
]
COLUMNS = ("X", "V", "t", "horizon", "ar", "error_value_ar", "errored_bound", "rejected", "hitting_horizon", "status",
           "counters", "tape_pos", "is_active")


def run(p, s, x0, v0, team, n_sk, **kw):
    os.environ["PDMPFLUX_TEAM"] = str(team)
    os.environ["PDMPFLUX_FORCE_GENERIC"] = "1"
    try:
        return p.sample_skeleton(s, n_sk, x0, v0, **kw)
    finally:
        os.environ.pop("PDMPFLUX_TEAM")
        os.environ.pop("PDMPFLUX_FORCE_GENERIC")


def start(d, n_chains, seed):
    g = np.random.default_rng(seed)
    return 0.5 * g.standard_normal((n_chains, d)), np.where(g.random((n_chains, d)) < 0.5, -1.0, 1.0)


@pytest.mark.parametrize("team", [1, 8, 32])
@pytest.mark.parametrize("case", IDENTITY_CASES, ids=[f"{a}-{b}-d{c}" for a, b, c in IDENTITY_CASES])
def test_bit_identical_to_builtin(p, case, team):
    kind, which, d = case
    if team == 1 and d > 16:
        pytest.skip("thread-per-chain is for small d")
    builtin, source = pots(p, which, d)
    x0, v0 = start(d, 256, zlib.crc32(f"{kind}{which}".encode()))
    if kind in ("bps", "boomerang", "fecmc"):
        v0 = np.random.default_rng(3).standard_normal((256, d))
    a = run(p, SAMPLERS[kind](p, d, builtin), x0, v0, team, 300, seed=77)
    b = run(p, SAMPLERS[kind](p, d, source), x0, v0, team, 300, seed=77)
    for col in COLUMNS:
        ca, cb = getattr(a, col, None), getattr(b, col, None)
        if ca is None and cb is None:
            continue
        assert np.array_equal(ca, cb), col
    assert (np.diff(a.t, axis=1) > 0).all()


def test_fused_moments_bit_identical(p):
    d, n = 12, 512
    x0, v0 = start(d, n, 5)
    out = []
    for pot in pots(p, "banana", d):
        os.environ["PDMPFLUX_FORCE_GENERIC"] = "1"
        try:
            ch = p.DeviceChains(p.ZigZag(d, pot, AD_backend="ForwardDiff"), x0, v0, seed=9)
            ch.enable_moments()
            ch.advance(200)
            out.append(ch.moments())
            ch.close()
        finally:
            os.environ.pop("PDMPFLUX_FORCE_GENERIC")
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])


# ---- a target with no built-in: the numpy oracle ---------------------------------------------------------------
class LogCosh:
    """U = sum_i log cosh(s_i x_i) + c/2 (sum_i x_i)^2"""

    def __init__(self, s, c):
        self.s, self.c = np.asarray(s, dtype=np.float64), float(c)

    def value(self, x):
        return float(np.sum(np.log(np.cosh(self.s * x)))) + 0.5 * self.c * float(np.sum(x)) ** 2

    def grad(self, x):
        return self.s * np.tanh(self.s * x) + self.c * np.sum(x)

    def hvp(self, x, v):
        th = np.tanh(self.s * x)
        return self.s * self.s * (1.0 - th * th) * v + self.c * np.sum(v)


PARITY_KINDS = {  # name: (oracle sampler kind, config kwargs of the oracle, device constructor)
    "zz_jvp": (onp.ZIGZAG, dict(), lambda p, d, pot: p.ZigZag(d, pot, AD_backend="ForwardDiff")),
    "zz_fd": (onp.ZIGZAG, dict(deriv_mode=onp.DERIV_FD), lambda p, d, pot: p.ZigZag(d, pot, AD_backend="FiniteDiff")),
    "zz_brent": (onp.ZIGZAG, dict(grid_size=0), lambda p, d, pot: p.ZigZag(d, pot, grid_size=0, AD_backend="ForwardDiff")),
    "bps": (onp.BPS, dict(tmax=1.0, refresh_rate=0.1, vectorized_bound=False),
            lambda p, d, pot: p.BPS(d, pot, AD_backend="ForwardDiff")),
    "fecmc": (onp.FECMC, dict(), lambda p, d, pot: p.ForwardECMC(d, pot, AD_backend="ForwardDiff")),
    "boomerang": (onp.BOOMERANG, dict(tmax=1.0, refresh_rate=0.1, vectorized_bound=False),
                  lambda p, d, pot: p.Boomerang(d, pot, AD_backend="ForwardDiff")),
}


@pytest.mark.parametrize("d", [9, 40])
@pytest.mark.parametrize("kind", list(PARITY_KINDS))
def test_logcosh_one_step_parity(p, kind, d):
    """Teacher-forced: every event of the oracle's skeleton is regenerated on the GPU from the previous state."""
    okind, kw, make = PARITY_KINDS[kind]
    n_sk = 200
    s_ = np.linspace(0.5, 2.0, d)
    c = 0.05
    g = np.random.default_rng(zlib.crc32(f"{kind}{d}".encode()))
    x0 = 0.6 * g.standard_normal(d)
    v0 = np.where(g.random(d) < 0.5, -1.0, 1.0) if okind == onp.ZIGZAG else g.standard_normal(d)
    E = g.standard_exponential(12 * n_sk); U = g.random(12 * n_sk); N = g.standard_normal(4 * d * n_sk + 8)
    so = onp.Sampler(d, LogCosh(s_, c), onp.Config(sampler=okind, **kw))
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
    idx = lambda start, w: start[:, None] + np.arange(w)[None, :]
    pad = lambda a, w: np.concatenate([a, np.ones(w)])
    tE, tU, tN = pad(E, wE)[idx(pos[:-1, 0], wE)], pad(U, wU)[idx(pos[:-1, 1], wU)], pad(N, wN)[idx(pos[:-1, 2], wN)]
    X = np.array([q[0] for q in states]); V = np.array([q[1] for q in states])
    T = np.array([q[2] for q in states]); H = np.array([q[3] for q in states])
    s = make(p, d, p.CudaPotential(LOGCOSH_SRC, np.concatenate([s_, [c]])))
    h = p.sample_skeleton(s, 2, X[:-1], V[:-1], tape=(tE, tU, tN), t0=T[:-1], horizon0=H[:-1], batch=True)
    ex = (np.abs(h.X[:, 1] - X[1:]).max(axis=1) / np.maximum(np.abs(X[1:]).max(axis=1), 1e-300)).max()
    ev = (np.abs(h.V[:, 1] - V[1:]).max(axis=1) / np.maximum(np.abs(V[1:]).max(axis=1), 1e-300)).max()
    dt_o = T[1:] - T[:-1]
    et = (np.abs((h.t[:, 1] - h.t[:, 0]) - dt_o) / dt_o).max()
    eh = (np.abs(h.horizon[:, 1] - H[1:]) / H[1:]).max()
    ea = np.abs(h.ar[:, 1] - np.array([r[0] for r in recs])).max()
    tol = tier_tolerance(dict(deriv_mode=kw.get("deriv_mode", 0)))
    record_parity_error(f"source_logcosh_one_step/{kind}/d{d}", x=ex, v=ev, t=et, horizon=eh, ar=ea, tol=tol)
    assert max(ex, ev, et, eh, ea) < tol, dict(x=ex, v=ev, t=et, horizon=eh, ar=ea)
    assert np.array_equal(h.rejected[:, 1], [r[1] for r in recs])
    assert np.array_equal(h.hitting_horizon[:, 1], [r[2] for r in recs])
    assert np.array_equal(h.tape_pos, use)


@pytest.mark.parametrize("kind", ["zz", "bps"])
def test_hyperbolic_secant_known_answer(p, kind):
    """U = sum_i log cosh(s_i x_i): x_i has the hyperbolic-secant law, mean 0 and E[x_i^2] = pi^2 / (4 s_i^2)."""
    d, n = 10, 4096
    s_ = np.linspace(0.5, 2.0, d)
    pot = p.CudaPotential(LOGCOSH_SRC, np.concatenate([s_, [0.0]]))
    sampler = p.ZigZag(d, pot, AD_backend="ForwardDiff") if kind == "zz" else p.BPS(d, pot, AD_backend="ForwardDiff")
    g = np.random.default_rng(1)
    x0 = g.standard_normal((n, d)) / s_
    v0 = np.where(g.random((n, d)) < 0.5, -1.0, 1.0) if kind == "zz" else g.standard_normal((n, d))
    ch = p.DeviceChains(sampler, x0, v0, seed=2024)
    ch.advance(200)                      # burn-in
    t0 = ch.get_state()[2]
    ch.enable_moments()
    ch.advance(2000)
    m1, m2 = ch.moments()
    length = ch.get_state()[2] - t0      # each chain's moment window
    ch.close()
    mean_c, sq_c = m1 / length[:, None], m2 / length[:, None]
    for est, target in ((mean_c, np.zeros(d)), (sq_c, np.pi ** 2 / (4 * s_ ** 2))):
        se = est.std(axis=0, ddof=1) / np.sqrt(n)
        z = np.abs(est.mean(axis=0) - target) / se
        assert (z < 5).all(), (kind, z, est.mean(axis=0), target)


def test_sharding_and_resume_bit_identical(p):
    d, n, n_sk = 9, 64, 301
    pot = p.CudaPotential(LOGCOSH_SRC, np.concatenate([np.linspace(0.5, 2.0, d), [0.05]]))
    s = p.ZigZag(d, pot, AD_backend="ForwardDiff")
    x0, v0 = start(d, n, 11)
    full = p.sample_skeleton(s, n_sk, x0, v0, seed=5)
    part = p.sample_skeleton(s, n_sk, x0[20:37], v0[20:37], seed=5, chain_offset=20)
    for col in ("X", "V", "t", "horizon", "ar"):
        assert np.array_equal(getattr(full, col)[20:37], getattr(part, col)), col
    k = 150
    first = p.sample_skeleton(s, k + 1, x0, v0, seed=5)
    rest = p.sample_skeleton(s, n_sk - k, first.X[:, -1], first.V[:, -1], seed=5, t0=first.t[:, -1],
                             horizon0=first.horizon[:, -1], event0=k)
    for col in ("X", "V", "t", "horizon", "ar"):
        assert np.array_equal(getattr(full, col)[:, k + 1:], getattr(rest, col)[:, 1:]), col


def test_compile_cache_ignores_params(p):
    count = p.lib().pdmpflux_jit_compile_count
    src = LOGCOSH_SRC + "\n// cache test\n"
    p.ZigZag(9, p.CudaPotential(src, np.concatenate([np.ones(9), [0.1]])))
    n0 = count()
    s = p.ZigZag(9, p.CudaPotential(src, np.concatenate([np.full(9, 2.0), [0.3]])))
    assert count() == n0
    h = p.sample_skeleton(s, 20, np.zeros((16, 9)), np.ones((16, 9)), seed=1)
    assert np.isfinite(h.X).all() and count() == n0


def test_rv_diagnostic_is_unsupported(p):
    d = 5
    pot = p.CudaPotential(BANANA_SRC)
    h = p.sample_skeleton(p.ZigZag(d, pot), 50, np.zeros(d), np.ones(d), seed=3)
    with pytest.raises(p.UnsupportedError):
        p.RV_diagnostic(h, pot)


def test_two_devices_same_bits(p):
    import ctypes
    n = ctypes.c_int(0)
    p.lib().pdmpflux_device_count(ctypes.byref(n))
    if n.value < 2:
        pytest.skip("needs two GPUs")
    d = 9
    x0, v0 = start(d, 128, 4)
    out = []
    for dev in (0, 1):
        p.lib().pdmpflux_set_device(dev)
        try:
            s = p.ZigZag(d, p.CudaPotential(LOGCOSH_SRC, np.concatenate([np.linspace(0.5, 2.0, d), [0.05]])))
            out.append(p.sample_skeleton(s, 200, x0, v0, seed=8))
        finally:
            p.lib().pdmpflux_set_device(0)
    assert np.array_equal(out[0].X, out[1].X) and np.array_equal(out[0].t, out[1].t)
