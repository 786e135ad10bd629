"""The one-dimensional model (SURVEY §8f-4) on the CPU: the oracle against the reference's formulas restated
independently, the merge rule as typed, and the DEVICE header (physics1d.h, host build) against the oracle bit for bit."""
import ctypes as C
import math
import os

import mpmath as mp
import numpy as np
import pytest

import host_build
from oracle import oned
from picles_b200._abi import PiclesCounters, PiclesParams
from scenarios_1d import SCENARIOS_1D, compare_models_1d, grid_1d, params_1d, run_pair_1d

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- host build of the device header -----------------------------------------------------------------------
class Shim1D:
    _lib = None

    @classmethod
    def lib(cls):
        if cls._lib is None:
            L = host_build.load("host_shim_1d", src=os.path.join(ROOT, "tests", "host_shim_1d.cpp"))
            vp, d = C.c_void_p, C.c_double
            L.shim1_create.restype = vp
            L.shim1_create.argtypes = [C.c_int, d, d, vp, C.POINTER(PiclesParams)]
            L.shim1_destroy.argtypes = [vp]
            L.shim1_seed.argtypes = [vp, vp]
            L.shim1_step.argtypes = [vp, d, d, vp, vp]
            L.shim1_get_state.argtypes = [vp, vp]
            L.shim1_get_particles.argtypes = [vp, vp, vp, vp, vp, vp]
            L.shim1_get_counters.argtypes = [vp, C.POINTER(PiclesCounters)]
            L.shim1_merge.argtypes = [vp, vp]
            L.shim1_rhs.argtypes = [C.POINTER(PiclesParams), vp, d, vp]
            cls._lib = L
        return cls._lib

    def __init__(self, g, P):
        self.L = self.lib()
        self.Nx = g["Nx"]
        xn = np.ascontiguousarray(g["x"], np.float64)
        self.h = self.L.shim1_create(self.Nx, g["xmin"], g["dx"], xn.ctypes.data_as(C.c_void_p), C.byref(P))

    def seed(self, u0):
        u0 = np.ascontiguousarray(np.broadcast_to(u0, (self.Nx,)), np.float64)
        self.L.shim1_seed(self.h, u0.ctypes.data_as(C.c_void_p))

    def step(self, t, DT, a, b):
        a = np.ascontiguousarray(a, np.float64)
        b = np.ascontiguousarray(b, np.float64)
        self.L.shim1_step(self.h, t, DT, a.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p))

    def state(self):
        S = np.empty((3, self.Nx))
        self.L.shim1_get_state(self.h, S.ctypes.data_as(C.c_void_p))
        return S

    def particles(self):
        z, t, dt = np.empty((3, self.Nx)), np.empty(self.Nx), np.empty(self.Nx)
        fl, st = np.empty(self.Nx, np.uint8), np.empty(self.Nx, np.int32)
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        self.L.shim1_get_particles(self.h, p(z), p(t), p(dt), p(fl), p(st))
        return dict(z=z, t=t, dt=dt, flags=fl, status=st)

    def counters(self):
        c = PiclesCounters()
        self.L.shim1_get_counters(self.h, C.byref(c))
        return {n: getattr(c, n) for n, _ in c._fields_}


def make_oracle_1d(g, P):
    return oned.Oracle1D(g["Nx"], g["xmin"], g["dx"], g["x"], P)


# ---- the reference's formulas, restated a second time in 50-digit arithmetic -----------------------------
def rhs_mp(P, z, u):
    """particle_waves_v5.jl:597-646, from the Julia text"""
    mp.mp.dps = 50
    f = mp.mpf
    lne, cx = f(z[0]), f(z[1])
    r_g, C_a, C_e, p, n, e_T = f(P.r_g), f(P.C_alpha), f(P.C_e), f(P.p), f(P.n), f(P.e_T)
    us = abs(f(u))
    c_gp = abs(cx) / r_g
    kp = f("9.81") / (4 * max(c_gp ** 2, f("1e-2")))
    wp = f("9.81") / (2 * max(abs(c_gp), f("0.1")))
    alpha = min(us / (2 * c_gp), 500)
    Hp = (1 + mp.tanh(p * (alpha - f("0.85")))) / 2
    Dp = 1 - f("1.25") * mp.sech(10 * (alpha - f("0.85"))) ** 2
    It = C_e * Hp * alpha ** 2
    Dt = mp.exp(n * lne) * (kp / e_T) ** (2 * n)
    Scg = C_a * Dp * kp ** 4 * mp.exp(2 * lne)
    return [wp * r_g * Scg + wp * (It - Dt), -cx * wp * r_g * Scg, cx]


def test_rhs_against_the_julia_text_in_exact_arithmetic():
    P = params_1d()
    rng = np.random.default_rng(3)
    for _ in range(200):
        z = [rng.uniform(-12, 1), rng.choice([-1, 1]) * np.exp(rng.uniform(-3, 2.5)), rng.uniform(0, 1e6)]
        u = rng.uniform(-25, 25)
        got = oned.rhs(P, z, u)
        ref = rhs_mp(P, z, u)
        scale = max(abs(float(r)) for r in ref[:2]) + 1e-300
        # Hp = (1 + tanh)/2 and Dp = 1 - 1.25 sech^2 cancel in the reference too: compare on the conditioning-aware scale
        terms = float(abs(ref[0])) + 1e-3 * scale
        assert abs(got[0] - float(ref[0])) <= 1e-12 * max(terms, abs(float(ref[0]))) + 1e-11 * scale
        assert abs(got[1] - float(ref[1])) <= 1e-11 * scale
        assert got[2] == z[1]


def test_windsea_1d_against_the_mirror_formula():
    """get_initial_windsea(U10, T), FetchRelations.jl:254-287"""
    from picles_b200 import FetchRelations as FR
    for U in (15.0, -7.5, 2.0, 31.0):
        for T in (600.0, 1200.0, 43200.0):
            tau = 9.81 * T / abs(U)
            X = FR.X_tilde_from_tau(tau)
            f_m = FR.fₘ_from_X_tilde(abs(U), X)
            E = FR.E_JONSWAP(f_m, FR.alpha_j(abs(U), f_m))
            cg = math.copysign(9.81 * (0.9 / (f_m * 9.81 / abs(U))) / (4 * math.pi), U)
            lne, cgb = oned.windsea(U, T)
            assert abs(lne - math.log(E)) < 1e-12 * abs(math.log(E))
            assert abs(cgb - cg) < 1e-13 * abs(cg)


def test_merge_rule_as_typed():
    """merge!(grid_point, charge), ParticleInCell.jl:228-252: with m_y = 0 the 'cos theta' is the raw product of the
    two momenta, so an occupied node only accepts charges whose momentum product reaches 0.5"""
    assert np.array_equal(oned.merge([0, 0, 0], [2e-3, 1e-4, 0]), [2e-3, 1e-4, 0])           # empty node: add
    assert np.array_equal(oned.merge([2e-3, 1e-4, 0], [1e-3, 2e-4, 0]), [2e-3, 1e-4, 0])     # occupied, small momenta: dropped
    assert np.array_equal(oned.merge([1e-3, 1e-4, 0], [2e-3, 2e-4, 0]), [1e-3, 1e-4, 0])     # ... even when the charge is larger
    assert np.array_equal(oned.merge([1.0, 1.0, 0], [0.5, 0.6, 0]), [1.5, 1.6, 0])           # product 0.6 >= 0.5: add
    assert np.array_equal(oned.merge([1.0, 1.0, 0], [0.5, 0.4, 0]), [1.0, 1.0, 0])           # product 0.4: dropped
    g = oned.merge([1.0, 1.0, 0], [0.5, 0.0, 0])                                             # 0/0 in the formula: NaN, no branch taken
    assert np.array_equal(g, [1.0, 1.0, 0])


@pytest.mark.parametrize("name", sorted(SCENARIOS_1D))
def test_device_header_on_the_host_matches_the_oracle(name):
    g, P, wind, DT, steps = SCENARIOS_1D[name]()
    run_pair_1d(make_oracle_1d(g, P), Shim1D(g, P), g, wind, DT, steps, compare_models_1d)


def test_scenarios_exercise_what_they_claim():
    def run(name):
        g, P, wind, DT, steps = SCENARIOS_1D[name]()
        o = make_oracle_1d(g, P)
        x = g["x"]
        o.seed(wind(x, 0.0))
        t, rows = 0.0, []
        for _ in range(steps):
            o.step(t, DT, wind(x, t), wind(x, t + DT))
            t += DT
            rows.append(o.counters())
        return g, o, rows
    g, o, rows = run("steady_nonperiodic")
    S = o.state()
    assert rows[-1]["n_integrated"] == g["Nx"] - 2 and rows[-1]["n_failed"] == 0          # the two boundary particles never integrate
    assert np.all(np.isfinite(S)) and S[0, 1:-1].min() > 0 and np.all(S[2] == 0.0)
    # the merge rule as typed: once a node holds the ceil-corner share of the upstream particle (a few per cent of its
    # charge), the node's own particle — next in order — is turned away; only the first interior node keeps its own
    assert rows[1]["n_deposited"] == g["Nx"] - 2
    o2 = make_oracle_1d(*SCENARIOS_1D["steady_nonperiodic"]()[:2])
    x = g["x"]
    o2.seed(np.full(g["Nx"], 15.0))
    o2.step(0.0, 600.0, np.full(g["Nx"], 15.0), np.full(g["Nx"], 15.0))
    o2.step(600.0, 600.0, np.full(g["Nx"], 15.0), np.full(g["Nx"], 15.0))
    S2 = o2.state()
    assert S2[0, 2] < 0.05 * S2[0, 1] and np.allclose(S2[0, 3:10], S2[0, 2], rtol=1e-6)
    _, _, rows = run("ramp_winds")
    assert sum(r["n_remesh_D"] for r in rows) > 0 and sum(r["n_remesh_B"] + r["n_reseed_advance"] for r in rows) > 0
    _, _, rows = run("emax_reset")
    assert sum(r["n_fixups"] for r in rows) > 0


def test_staged_winds_against_the_closure():
    """The reference calls winds(x, t) at the particle's position and the stage time; the staged path reads the node
    values of the levels t and t + DT, linear in x between nodes and linear in t.  Identical for a steady wind;
    rounding-level for a wind that is piecewise linear in x and steady in time; for a wind that also varies in time the
    two-level rule is what remains (the 2-D path's B-2 deviation): median |delta lne / lne| 3e-4 for a 12 h modulation
    at DT = 20 min, 6e-3 for a 2 h one."""
    g, P, wind, DT, steps = SCENARIOS_1D["steady_nonperiodic"]()
    L = 600e3
    x0 = 0.2 * L

    def ramp(period):
        def u(x, t):
            r = np.where(np.asarray(x) < x0, 0.02, (np.asarray(x) - x0) / (L - x0))
            out = 12.0 * r * (0.8 + 0.2 * np.sin(2 * np.pi * t / period))
            return out if np.ndim(x) else float(out)
        return u

    def deviation(g, P, w, DT, steps):
        a, b = make_oracle_1d(g, P), make_oracle_1d(g, P)
        b.set_wind_closure(lambda x, t: float(w(np.float64(x), t)))
        x = g["x"]
        a.seed(w(x, 0.0)); b.seed(w(x, 0.0))
        t = 0.0
        for _ in range(steps):
            a.step(t, DT, w(x, t), w(x, t + DT)); b.step(t, DT, w(x, t), w(x, t + DT))
            t += DT
        return a.state(), b.state()

    Sa, Sb = deviation(g, P, wind, DT, steps)
    assert np.array_equal(Sa, Sb)
    g, P, _, DT, steps = SCENARIOS_1D["ramp_winds"]()
    for period, tol in ((1e12, 1e-10), (43200.0, 2e-3), (7200.0, 3e-2)):
        Sa, Sb = deviation(g, P, ramp(period), DT, steps)
        on = (Sa[0] > 0) & (Sb[0] > 0)
        assert on.sum() > 30
        rel = np.abs(np.log(Sa[0][on]) - np.log(Sb[0][on])) / np.abs(np.log(Sb[0][on]))
        assert np.median(rel) < tol, (period, np.median(rel))


@pytest.mark.parametrize("name", ["steady_nonperiodic", "ramp_winds", "fast_periodic"])
def test_golden_fixture_1d(name):
    """frozen oracle outputs (tests/golden/oned.npz, written by the generator in its docstring): guards the oracle,
    pmath.h and — through the host build above — the device header against silent changes

        python - <<'PY'   # regenerate on purpose only
        (see the commit that added tests/golden/oned.npz: the scenario loop of this test, saved with np.savez_compressed)
        PY
    """
    G = np.load(os.path.join(ROOT, "tests", "golden", "oned.npz"))
    g, P, wind, DT, steps = SCENARIOS_1D[name]()
    o = make_oracle_1d(g, P)
    x = g["x"]
    o.seed(wind(x, 0.0))
    t = 0.0
    for _ in range(steps):
        o.step(t, DT, wind(x, t), wind(x, t + DT))
        t += DT
    p, c = o.particles(), o.counters()
    from scenarios_1d import bits_equal
    assert bits_equal(o.state(), G[name + "/state"]) and bits_equal(p["z"], G[name + "/z"])
    assert np.array_equal(p["flags"], G[name + "/flags"]) and bits_equal(p["t"], G[name + "/t"])
    keys = ("n_integrated", "n_substeps", "n_rejects", "n_rhs", "n_remesh_A", "n_remesh_B", "n_remesh_D", "n_deposited")
    assert [c[k] for k in keys] == list(G[name + "/counters"])


def test_integrator_1d_converges_to_an_independent_solver():
    """One DT of the 1-D system under a steady wind, integrated by scipy's DOP853 (rtol 1e-12) on the oracle's right-hand
    side: the oracle's Tsit5 at the reference's tolerances stays within 5e-3 of it and converges as they tighten.
    Uniform periodic chain: every particle is the same, and node 1 keeps the floor-corner share of particle 1 (the
    first charge to arrive there), so State[1, 1] = w_floor * exp(lne(DT))."""
    from scipy.integrate import solve_ivp
    g, P, wind, DT, _ = SCENARIOS_1D["steady_periodic"]()
    U = 10.0

    def first_node_energy(P):
        o = make_oracle_1d(g, P)
        o.seed(np.full(g["Nx"], U))
        z0 = o.particles()["z"][:, 0].copy()
        o.step(0.0, DT, np.full(g["Nx"], U), np.full(g["Nx"], U))
        return z0, o.state()[0, 0]

    z0, e_ref_tol = first_node_energy(P)
    sol = solve_ivp(lambda t, z: oned.rhs(P, z, U), (0.0, DT), z0, method="DOP853", rtol=1e-12, atol=1e-14)
    lne, _, x = sol.y[:, -1]
    xn = (x - g["xmin"]) / g["dx"]
    expect = (1.0 - (xn - math.floor(xn))) * math.exp(lne)
    assert abs(e_ref_tol - expect) < 5e-3 * expect
    P2 = params_1d(600.0, periodic=True)
    P2.abstol, P2.reltol = 1e-11, 1e-10
    _, e_tight = first_node_energy(P2)
    assert abs(e_tight - expect) < 1e-7 * expect


from scenarios_1d import EDGE_1D  # noqa: E402


@pytest.mark.parametrize("name", sorted(EDGE_1D))
def test_device_header_edge_cases_match_the_oracle(name):
    g, P, wind, DT, steps = EDGE_1D[name]()
    a, b = make_oracle_1d(g, P), Shim1D(g, P)
    run_pair_1d(a, b, g, wind, DT, steps, compare_models_1d)
    c = a.counters()
    if name == "calm":
        assert c["n_integrated"] == 0 and c["n_remesh_D"] == g["Nx"]
    if name == "maxiters":
        assert c["n_failed"] > 0 or (a.particles()["status"] & 1).any()
    if name == "dtmin_no_force":
        assert (a.particles()["status"] & 2).any()
    if name == "tiny_periodic_fast":
        assert b.counters()["reach"] * 2 + 1 >= g["Nx"]


def test_device_header_merge_and_rhs_known_answers():
    """the device header's merge rule and right-hand side by themselves against the oracle's, on the branch boundaries the
    scenarios never hit exactly (cos theta == 0.5, dE == 0, an empty charge) and on random states"""
    L = Shim1D.lib()
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    cases = [([0, 0, 0], [2e-3, 1e-4, 0]), ([1.0, 1.0, 0], [0.5, 0.5, 0]), ([1.0, 1.0, 0], [0.5, 0.4999999999999999, 0]),
             ([1.0, 2.0, 0], [1.0, 0.1, 0]), ([1.0, 1.0, 0], [0.5, 0.0, 0]), ([1.0, -1.0, 0], [0.5, -0.7, 0]),
             ([1.0, -1.0, 0], [2.0, 0.7, 0]), ([0.0, 0.0, 0.0], [0.0, 0.0, 0.0]), ([1e-3, 1e-4, 0], [np.nan, 1e-4, 0])]
    for g0, c0 in cases:
        g = np.array(g0, np.float64)
        c = np.array(c0, np.float64)
        L.shim1_merge(p(g), p(c))
        ref = oned.merge(g0, c0)
        assert np.array_equal(g, ref, equal_nan=True), (g0, c0, g, ref)
    assert np.array_equal(oned.merge([1.0, 1.0, 0], [0.5, 0.5, 0]), [1.5, 1.5, 0])   # cos theta == 0.5 exactly: added
    P = params_1d()
    rng = np.random.default_rng(11)
    for _ in range(300):
        z = np.array([rng.uniform(-14, 2), rng.choice([-1, 1]) * np.exp(rng.uniform(-5, 3)), rng.uniform(0, 1e6)])
        u = rng.uniform(-30, 30)
        dz = np.empty(3)
        L.shim1_rhs(C.byref(P), p(z), float(u), p(dz))
        assert np.array_equal(dz.view(np.uint64), oned.rhs(P, z, u).view(np.uint64))


def test_1d_system_is_the_2d_system_on_the_x_axis():
    """Two separately transcribed right-hand sides: with the wind and the group velocity both along +x the 2-D system
    (particle_waves_v5.jl:479-556; alpha_p, S_dir, great-circle term) reduces to the 1-D one (:597-646; alpha) — the same
    tendencies of lne and c̄_x up to rounding, and dx/dt = c̄_x against M = identity."""
    import oracle
    from common import default_params
    P1, P2 = params_1d(), default_params()
    rng = np.random.default_rng(5)
    for _ in range(200):
        lne, cx, u = rng.uniform(-12, 1), np.exp(rng.uniform(-3, 2.5)), rng.uniform(0.5, 25)
        if u / (2 * cx / P1.r_g) > 499.0:
            continue
        d1 = oned.rhs(P1, [lne, cx, 0.0], u)
        d2 = oracle.rhs(P2, [lne, cx, 0.0, 0.0, 0.0], u, 0.0, M=(1.0, 0.0, 0.0, 1.0), pc=0.0)
        scale = max(abs(d2[0]), abs(d2[1]), 1e-300)
        assert abs(d1[0] - d2[0]) <= 1e-12 * max(abs(d2[0]), 1e-2 * scale) + 1e-13 * scale
        assert abs(d1[1] - d2[1]) <= 1e-12 * scale
        assert d2[2] == 0.0 and d1[2] == d2[3] == cx and d2[4] == 0.0


def fuzz_case_1d(seed):
    """a random 1-D configuration: chain length and spacing, grid offset, periodicity, solver, thresholds, source
    terms on or off, a wind that varies along the chain and in time with a weak stretch swelling across the on/off
    thresholds"""
    rng = np.random.default_rng(seed)
    Nx = int(rng.integers(5, 60))
    L = float(rng.choice([20e3, 100e3, 600e3, 1500e3]))
    xmin = float(rng.choice([0.0, 1e3]))
    periodic = bool(rng.random() < 0.5)
    DT = float(rng.choice([600.0, 1200.0, 1800.0]))
    solver = str(rng.choice(["Tsit5", "Tsit5", "DP5"]))
    kw = dict(input=False, dissipation=False, peak_shift=False) if rng.random() < 0.2 else {}
    P = params_1d(DT, solver=solver, periodic=periodic, wind_min_squared=float(rng.choice([2.0, 4.0])),
                  log_energy_maximum=float(rng.choice([math.log(17), -6.0])), **kw)
    g = grid_1d(xmin, xmin + L, Nx)
    a, b, c = rng.uniform(-15, 15), rng.uniform(-10, 10), rng.uniform(0, 6)
    om = 2 * math.pi / float(rng.choice([3600.0, 14400.0, 1e9]))
    calm = rng.uniform(0, 0.5)

    def wind(x, t):
        s = (np.asarray(x, float) - xmin) / L
        w = np.where(s < calm, 1.2 * (1 + 0.9 * np.sin(om * t)), a + b * s + c * np.sin(om * t + 3 * s))
        return w if np.ndim(x) else float(w)
    return g, P, wind, DT


@pytest.mark.parametrize("seed", range(12))
def test_random_configurations_1d(seed):
    """the two transcriptions of the 1-D model (oracle/picles_oracle_1d.c and physics1d.h on the host) on random
    configurations, bit for bit after every step (300 seeds were run once: no difference)"""
    g, P, wind, DT = fuzz_case_1d(seed)
    run_pair_1d(make_oracle_1d(g, P), Shim1D(g, P), g, wind, DT, 5, compare_models_1d)


@pytest.mark.parametrize("flag", [False, True])
def test_nan_error_estimate_switch_1d(flag):
    """picles_params_t::nan_eest_rejects on the 1-D path: DP5 under winds across the 14 m/s band loses a particle to an
    overflowing trial step with the switch off (DtNaN) and none with it on; oracle = device header either way"""
    g = grid_1d(0.0, 200e3, 21)
    P = params_1d(600.0, solver="DP5", nan_eest_rejects=flag)
    wind = lambda x, t: np.linspace(13.6, 14.4, 21) if np.ndim(x) else 14.0
    a, b = make_oracle_1d(g, P), Shim1D(g, P)
    run_pair_1d(a, b, g, wind, 600.0, 3, compare_models_1d)
    dead = int(((a.particles()["status"] & 4) != 0).sum())
    assert dead == (0 if flag else 1)
