"""GPU tests (-m gpu) of ensembles with one wind mesh per member (picles_set_member_wind_meshes): every member's sampled
wind and every step taken with it, against the CPU oracle run with that member's mesh alone and against a single-member
handle given that mesh — bit for bit after every step."""

import numpy as np
import pytest

import oracle
from common import BND_PERIODIC, TALLY_NAMES, bits_equal, cartesian_grid, default_params, make_oracle, tripolar_grid
from test_gpu_ensemble import compare_member, ensemble_engine
from test_wind_levels import mid_times

pytestmark = pytest.mark.gpu

TIMES = (0.0, 100.0, 2500.0, 4321.5, 7000.0, 9000.0, -500.0, -3 * 7000.0 - 17.0, 5 * 7000.0 + 17.0)


def meshes(g, E, seed=0, calm=(), nan=()):
    """E meshes on shared knots that the nodes spill over (periodic wrap), non-uniform in x; members in `calm` have no
    wind, members in `nan` a NaN patch.  Time knots are not multiples of the steps, so kinks fall inside steps."""
    rng = np.random.default_rng(seed)
    x, y = np.asarray(g["x"], np.float64), np.asarray(g["y"], np.float64)
    x0, x1, y0, y1 = x.min(), x.max(), y.min(), y.max()
    Lx, Ly = x1 - x0, y1 - y0
    c = np.concatenate([[0.0], np.cumsum(rng.uniform(0.2, 3.0, 10))])
    xw = x0 + 0.1 * Lx + 0.85 * Lx * c / c[-1]
    yw = np.linspace(y0 - 0.05 * Ly, y1 - 0.1 * Ly, 7)
    tw = np.array([0.0, 1000.0, 2500.0, 4000.0, 7000.0])
    sh = (E, tw.size, yw.size, xw.size)
    sign = np.where(np.arange(E) % 2 == 0, 1.0, -1.0)[:, None, None, None]
    U = sign * (9.0 + 4.0 * rng.random(sh))
    V = 5.0 - 8.0 * rng.random(sh)
    for m in calm:
        U[m] = V[m] = 0.0
    for m in nan:
        U[m, :, 2:4, 3:5] = np.nan
    return xw, yw, tw, U, V


def mesh_engine(g, P, mesh):
    xw, yw, tw, U, V = mesh
    eng = ensemble_engine(g, P, U.shape[0])
    eng.set_member_wind_meshes(xw, yw, tw, U, V, g["x"], g["y"])
    return eng


def oracle_sampler(g, mesh, m):
    xw, yw, tw, U, V = mesh
    return lambda t: oracle.wind_mesh_sample(xw, yw, tw, U[m], V[m], g["x"], g["y"], t)


def check_step(eng, refs, autotsit5):
    out = (eng.state(), eng.particles(), eng.solver_state() if autotsit5 else None)
    for m, r in enumerate(refs):
        compare_member(r, out, m, autotsit5)
    c = eng.counters()
    cr = [r.counters() for r in refs]
    for name in TALLY_NAMES:
        if name in ("reach", "max_attempts"):
            assert c[name] == max(x[name] for x in cr), name
        else:
            assert c[name] == sum(x[name] for x in cr), name


def run_against_oracles(g, P, mesh, DT, nsteps, n_mid=0, autotsit5=False, jump=None):
    """seed_wind_mesh + nsteps of step_wind_mesh on one ensemble handle, and per member the oracle stepped with the
    oracle's interpolation of that member's mesh; compared after every step.  jump = t of one more step that does not
    continue the last, so its t level is sampled again instead of reused."""
    E = mesh[3].shape[0]
    eng = mesh_engine(g, P, mesh)
    refs = [make_oracle(g, P) for _ in range(E)]
    samp = [oracle_sampler(g, mesh, m) for m in range(E)]
    eng.seed_wind_mesh(0.0)
    for r, s in zip(refs, samp):
        r.seed(*s(0.0))
    times = [DT * k for k in range(nsteps)] + ([jump] if jump is not None else [])
    for t in times:
        for r, s in zip(refs, samp):
            if n_mid:
                lv = [s(tm) for tm in mid_times(t, DT, n_mid)]
                r.set_wind_midlevels([a for a, _ in lv], [b for _, b in lv])
            r.step(t, DT, *s(t), *s(t + DT))
        eng.step_wind_mesh(t, DT, n_mid)
        check_step(eng, refs, autotsit5)
    return eng, refs


@pytest.mark.parametrize("E", [3, 13])
def test_member_sampler_matches_the_oracle(gpu_lib, E):
    """13 members: more than one member chunk of k_wind_sample_members, and odd; 57 x 31 nodes, an odd count"""
    g = cartesian_grid(57, 31, dx=1370.0, dy=3110.0)
    mesh = meshes(g, E, seed=E)
    eng = mesh_engine(g, default_params(), mesh)
    for t in TIMES:
        u, v = eng.sample_wind_mesh(t)
        assert u.shape == v.shape == (E, 31, 57)
        for m in range(E):
            uo, vo = oracle_sampler(g, mesh, m)(t)
            assert bits_equal(uo, u[m]) and bits_equal(vo, v[m]), (m, t)
    assert eng.measure_wind_sample(100.0, reps=3) > 0


def test_one_member_is_set_wind_mesh(gpu_lib):
    from test_gpu_parity import engine_for
    g = cartesian_grid(40, 23)
    P = default_params()
    xw, yw, tw, U, V = meshes(g, 1, seed=4)
    a, b = engine_for(g, P), engine_for(g, P)
    a.set_wind_mesh(xw, yw, tw, U[0], V[0], g["x"], g["y"])
    b.set_member_wind_meshes(xw, yw, tw, U, V, g["x"], g["y"])
    for t in TIMES:
        ua, va = a.sample_wind_mesh(t)
        ub, vb = b.sample_wind_mesh(t)
        assert bits_equal(ua, ub) and bits_equal(va, vb)
    for e in (a, b):
        e.seed_wind_mesh(0.0)
        for k in range(3):
            e.step_wind_mesh(600.0 * k, 600.0, 1)
    assert bits_equal(a.state(), b.state())


@pytest.mark.parametrize("n_mid", [0, 1, 2, 3])
def test_steps_match_the_oracle_per_member(gpu_lib, n_mid):
    g = cartesian_grid(44, 30)
    P = default_params(DT=600.0)
    run_against_oracles(g, P, meshes(g, 4, seed=10 + n_mid), 600.0, 5, n_mid=n_mid, jump=5000.0 if n_mid == 1 else None)


def test_autotsit5_members(gpu_lib):
    """fine cells and strong winds: members switch to Rosenbrock23 beside members that do not"""
    g = cartesian_grid(40, 16, dx=300.0, dy=300.0)
    P = default_params(DT=600.0, wind_min_squared=2.0, solver="AutoTsit5")
    mesh = meshes(g, 4, seed=21, calm=(1,))
    mesh[3][0] *= 2.2
    mesh[4][0] *= 2.2
    eng, refs = run_against_oracles(g, P, mesh, 600.0, 5, n_mid=1, autotsit5=True, jump=9000.0)
    # the AutoSwitch state moved in the windy members and not in the calm one
    assert all(np.any(refs[m].solver_state() != 0) for m in (0, 2, 3)) and not np.any(refs[1].solver_state() != 0)


def test_periodic_and_tripolar_grids(gpu_lib):
    g = cartesian_grid(48, 26, bx=BND_PERIODIC, by=BND_PERIODIC)
    run_against_oracles(g, default_params(DT=600.0, periodic_boundary=True), meshes(g, 3, seed=31), 600.0, 4, n_mid=1)
    g = tripolar_grid(48, 36)
    run_against_oracles(g, default_params(DT=1200.0), meshes(g, 3, seed=32), 1200.0, 4, n_mid=2, jump=6100.0)


def test_calm_and_nan_members_leave_the_others_alone(gpu_lib):
    g = cartesian_grid(36, 28, dx=800.0, dy=800.0)
    P = default_params(DT=600.0)
    mesh = meshes(g, 5, seed=41, calm=(1,), nan=(3,))
    eng, refs = run_against_oracles(g, P, mesh, 600.0, 4)
    # the normal members alone, without their calm and NaN neighbours, take the same steps
    keep = [0, 2, 4]
    sub = mesh[:3] + (mesh[3][keep], mesh[4][keep])
    alone = mesh_engine(g, P, sub)
    alone.seed_wind_mesh(0.0)
    for k in range(4):
        alone.step_wind_mesh(600.0 * k, 600.0, 0)
    assert bits_equal(alone.state(), eng.state()[:, keep])
    assert bits_equal(alone.member_energy_sums(), eng.member_energy_sums()[keep])


def test_each_member_equals_a_single_handle_with_its_mesh(gpu_lib):
    from test_gpu_parity import engine_for
    g = tripolar_grid(40, 30)
    P = default_params(DT=1200.0)
    mesh = meshes(g, 4, seed=51)
    xw, yw, tw, U, V = mesh
    eng = mesh_engine(g, P, mesh)
    singles = [engine_for(g, P) for _ in range(4)]
    for m, s in enumerate(singles):
        s.set_wind_mesh(xw, yw, tw, U[m], V[m], g["x"], g["y"])
    for e in [eng] + singles:
        e.seed_wind_mesh(0.0)
    for t in (0.0, 1200.0, 2400.0, 7300.0, 8500.0):
        for e in [eng] + singles:
            e.step_wind_mesh(t, 1200.0, 2)
        S, p = eng.state(), eng.particles()
        for m, s in enumerate(singles):
            assert bits_equal(S[:, m], s.state())
            ps = s.particles()
            for k in ("z", "t", "dt"):
                assert bits_equal(p[k][:, m] if k == "z" else p[k][m], ps[k])
            assert np.array_equal(p["flags"][m], ps["flags"]) and np.array_equal(p["status"][m], ps["status"])
        assert bits_equal(eng.member_energy_sums(), np.array([s.energy_sum() for s in singles]))
        ue, ve = eng.sample_wind_mesh(t)
        for m, s in enumerate(singles):
            us, vs = s.sample_wind_mesh(t)
            assert bits_equal(ue[m], us) and bits_equal(ve[m], vs)


def test_stage_then_step_equals_step_wind_mesh(gpu_lib):
    g = cartesian_grid(30, 22)
    P = default_params(DT=600.0)
    mesh = meshes(g, 3, seed=61)
    a, b = mesh_engine(g, P, mesh), mesh_engine(g, P, mesh)
    for e in (a, b):
        e.seed_wind_mesh(0.0)
    for t, n_mid in ((0.0, 0), (600.0, 2), (1200.0, 1), (4000.0, 3)):
        a.step_wind_mesh(t, 600.0, n_mid)
        b.stage_wind_mesh(t, 600.0, n_mid)
        b.step(t, 600.0)  # picles_step with no host winds: the staged levels
        assert bits_equal(a.state(), b.state())
        pa, pb = a.particles(), b.particles()
        assert bits_equal(pa["z"], pb["z"]) and np.array_equal(pa["flags"], pb["flags"])


def test_launches_per_step_do_not_depend_on_the_member_count(gpu_lib):
    g = cartesian_grid(20, 16)
    P = default_params(DT=600.0)
    counts = []
    for E in (2, 256):
        eng = mesh_engine(g, P, meshes(g, E, seed=71))
        eng.seed_wind_mesh(0.0)
        eng.step_wind_mesh(0.0, 600.0, 1)
        before = eng.launch_count()
        eng.step_wind_mesh(600.0, 600.0, 1)
        counts.append(eng.launch_count() - before)
    assert counts[0] == counts[1], counts


def test_refusals_of_the_new_call_leave_the_device_state_alone(gpu_lib):
    from picles_b200._abi import PiclesError
    g = cartesian_grid(24, 18)
    P = default_params(DT=600.0)
    xw, yw, tw, U, V = mesh = meshes(g, 2, seed=81)
    eng = ensemble_engine(g, P, 2)
    eng.seed(np.stack([np.full((18, 24), 8.0), np.full((18, 24), -6.0)]), 3.0)
    eng.step(0.0, 600.0, None, None, 9.0, 4.0)
    S, p = eng.state(), eng.particles()
    bad = [lambda: eng.set_member_wind_meshes(xw[::-1].copy(), yw, tw, U[:, :, :, ::-1], V, g["x"], g["y"]),
           lambda: eng.set_member_wind_meshes(xw[:1], yw, tw, U[:, :, :, :1], V[:, :, :, :1], g["x"], g["y"])]
    for call in bad:
        with pytest.raises(PiclesError, match="ERR_ARG"):
            call()
    xa, ya, ta = (np.ascontiguousarray(a) for a in (xw, yw, tw))
    rc = gpu_lib.picles_set_member_wind_meshes(eng.h, xw.size, yw.size, tw.size, xa.ctypes.data, ya.ctypes.data,
                                               ta.ctypes.data, None, None, None, None)
    assert rc == -1 and b"null array" in gpu_lib.picles_last_error(eng.h)
    # without member meshes the wind-mesh calls still refuse
    with pytest.raises(PiclesError, match="ERR_ARG.*ensemble"):
        eng.step_wind_mesh(600.0, 600.0)
    assert bits_equal(S, eng.state())
    p2 = eng.particles()
    for k in ("z", "t", "dt"):
        assert bits_equal(p[k], p2[k])
    # a refused call keeps the meshes set before it; one mesh for every member is still refused
    eng.set_member_wind_meshes(*mesh, g["x"], g["y"])
    with pytest.raises(PiclesError, match="ERR_ARG.*strictly increasing"):
        eng.set_member_wind_meshes(xw, yw, tw[::-1].copy(), U, V, g["x"], g["y"])
    with pytest.raises(PiclesError, match="ERR_ARG.*ensemble.*picles_set_member_wind_meshes"):
        eng.set_wind_mesh(xw, yw, tw, U[0], V[0], g["x"], g["y"])
    u, v = eng.sample_wind_mesh(2500.0)
    for m in range(2):
        uo, vo = oracle_sampler(g, mesh, m)(2500.0)
        assert bits_equal(uo, u[m]) and bits_equal(vo, v[m])
    assert bits_equal(S, eng.state())


def test_ensemble_model_with_gridded_winds_through_run(gpu_lib):
    """WaveGrowth2DEnsemble(winds=[GriddedWinds ...]) through run with cash_store: every member and every snapshot
    equals WaveGrowth2D(winds=that GriddedWinds)"""
    from picles_b200.Models import WaveGrowth2D, WaveGrowth2DEnsemble
    from picles_b200.Simulations.run import Simulation, run
    from picles_b200.Utils.WindEmulator import GriddedWinds
    from test_ensemble import ensemble_kwargs
    rng = np.random.default_rng(91)
    xw, yw = np.linspace(-5e3, 55e3, 11), np.linspace(-3e3, 35e3, 8)
    tw = np.array([0.0, 700.0, 1500.0, 2600.0])
    E = 3
    fields = [(rng.normal(8.0, 3.0, (xw.size, yw.size, tw.size)) * (-1) ** m, rng.normal(-2.0, 4.0, (xw.size, yw.size, tw.size)))
              for m in range(E)]
    ens = WaveGrowth2DEnsemble(winds=[GriddedWinds(xw, yw, tw, u, v) for u, v in fields], **ensemble_kwargs())
    sim = Simulation(ens, 600.0, stop_time=3 * 600.0, verbose=False)
    run(sim, cash_store=True)
    for m, (u, v) in enumerate(fields):
        gw = GriddedWinds(xw, yw, tw, u, v)
        single = WaveGrowth2D(winds=gw, **ensemble_kwargs())
        s = Simulation(single, 600.0, stop_time=3 * 600.0, verbose=False)
        run(s, cash_store=True)
        assert bits_equal(ens.State[m], single.State)
        assert len(sim.store.store) == len(s.store.store)
        for a, b in zip(sim.store.store, s.store.store):
            assert bits_equal(a[m], b)
        pe, ps = ens.ParticleCollection, single.ParticleCollection
        assert bits_equal(pe.u[m], ps.u) and bits_equal(pe.t[m], ps.t)
        assert bits_equal(ens.member_energy_sums()[m:m + 1], np.array([single.engine.energy_sum()]))
        # each member's GriddedWinds reads its own planes
        assert bits_equal(ens.winds[m].u(None, None, 950.0), gw.u(None, None, 950.0))
        assert bits_equal(ens.winds[m].v(None, None, 950.0), gw.v(None, None, 950.0))
