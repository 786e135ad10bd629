"""GPU tests (-m gpu) of ensembles (picles_set_members): every member of one handle, stepped together with the
others, against the CPU oracle run with that member's winds — bit for bit after every step."""
import numpy as np
import pytest

from common import TALLY_NAMES, bits_equal, cartesian_grid, default_params, make_oracle
from scenarios import SCENARIOS, _growing

pytestmark = pytest.mark.gpu


def ensemble_engine(grid, P, members):
    from picles_b200.engine import B200Engine
    return B200Engine(grid["Nx"], grid["Ny"], grid["bx"], grid["by"], grid["mask"], P, M=grid["M"],
                      M_const=grid["M_const"], pc=grid["pc"], members=members)


def full(x, g):
    return np.broadcast_to(np.asarray(x, np.float64), (g["Ny"], g["Nx"]))


def stack(winds, g, t):
    w = [wf(t) for wf in winds]
    return np.stack([full(a, g) for a, _ in w]), np.stack([full(b, g) for _, b in w])


def compare_member(ref, eng_out, m, autotsit5):
    S, p, sol = eng_out
    Sr = ref.state()
    assert bits_equal(Sr, S[:, m]), f"member {m}: State differs"
    pr = ref.particles()
    act = (pr["flags"] & 8) != 0
    for k in range(5):
        assert bits_equal(pr["z"][k][act], p["z"][k, m][act]), f"member {m}: particle component {k} differs"
    assert bits_equal(pr["t"][act], p["t"][m][act]), f"member {m}: t differs"
    live = act & ((pr["flags"] & 4) == 0)
    assert bits_equal(pr["dt"][live], p["dt"][m][live]), f"member {m}: dt differs"
    assert np.array_equal(pr["flags"][act], p["flags"][m][act]), f"member {m}: flags differ"
    assert np.array_equal(pr["status"][act], p["status"][m][act]), f"member {m}: status differs"
    if autotsit5:
        assert np.array_equal(ref.solver_state()[act], sol[m][act]), f"member {m}: AutoSwitch state differs"


def run_ensemble(g, P, winds, DT, nsteps, mid_levels=0, accumulate=False, autotsit5=False):
    """seed + nsteps of one ensemble handle and of one oracle per member, compared after every step; returns the
    engine and the oracles"""
    E = len(winds)
    eng = ensemble_engine(g, P, E)
    refs = [make_oracle(g, P) for _ in range(E)]
    u0, v0 = stack(winds, g, 0.0)
    eng.seed(u0, v0)
    for m, r in enumerate(refs):
        r.seed(u0[m], v0[m])
    if accumulate:
        eng.set_accumulate(True)
        for r in refs:
            r.set_accumulate(True)
    t = 0.0
    for _ in range(nsteps):
        if mid_levels:
            lv = [stack(winds, g, t + DT * k / (mid_levels + 1)) for k in range(1, mid_levels + 1)]
            eng.set_wind_midlevels([a for a, _ in lv], [b for _, b in lv])
            for m, r in enumerate(refs):
                r.set_wind_midlevels([a[m] for a, _ in lv], [b[m] for _, b in lv])
        ut, vt = stack(winds, g, t)
        ut1, vt1 = stack(winds, g, t + DT)
        eng.step(t, DT, ut, vt, ut1, vt1)
        for m, r in enumerate(refs):
            r.step(t, DT, ut[m], vt[m], ut1[m], vt1[m])
        t += DT
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
    return eng, refs


def scenario_members(name, variants):
    """the scenario's grid and params, and its wind scaled/rotated per member: variants = [(su, sv, swap)]"""
    g, P, wind, DT, n = SCENARIOS[name]()

    def member(su, sv, swap):
        def w(t):
            u, v = wind(t)
            u, v = (v, u) if swap else (u, v)
            return su * np.asarray(u, np.float64), sv * np.asarray(v, np.float64)
        return w

    return g, P, [member(*v) for v in variants], DT, n


SIGNS = [(1.0, 1.0, False), (-1.0, 1.0, False), (1.0, -1.0, True), (-0.6, -0.8, False)]


@pytest.mark.parametrize("solver", ["Tsit5", "AutoTsit5"])
def test_growing_winds_members_of_different_signs(gpu_lib, solver):
    g = cartesian_grid(66, 21, dx=4000.0, dy=4000.0)
    P = default_params(DT=1200.0, wind_min_squared=2.0, solver=solver)
    if solver == "AutoTsit5":
        # stiff members switch to Rosenbrock23 (a strong wind on fine cells) beside members that never do: the parked
        # particles of several members share one pending list
        g = cartesian_grid(40, 16, dx=300.0, dy=300.0)
        P = default_params(DT=1200.0, wind_min_squared=2.0, solver=solver)
        winds = [lambda t: (24.0, 18.0), lambda t: (0.8, 0.5), _growing(g, -12.0, 4.0), lambda t: (-22.0, 15.0)]
    else:
        winds = [_growing(g, 10.0 * su, 3.0 * sv) for su, sv, _ in SIGNS]
    eng, refs = run_ensemble(g, P, winds, 1200.0, 6, autotsit5=(solver == "AutoTsit5"))
    if solver == "AutoTsit5":
        switched = [r.counters()["n_stiff_switches"] for r in refs]
        triggered = [int(np.any(r.solver_state() != 0)) for r in refs]
        assert any(switched) or any(triggered)


@pytest.mark.parametrize("name", ["tripolar", "periodic_grid", "odd_periodic_strip", "fast_box"])
def test_members_on_every_gather_path(gpu_lib, name):
    g, P, winds, DT, n = scenario_members(name, SIGNS[:3])
    eng, refs = run_ensemble(g, P, winds, DT, n)
    if name == "fast_box":
        assert max(r.counters()["reach"] for r in refs) > 2


def test_members_stay_isolated(gpu_lib):
    """a member whose deposits cross its first and last rows, beside a calm member and one with a NaN wind patch"""
    g = cartesian_grid(24, 20, dx=500.0, dy=500.0)
    P = default_params()
    nan = SCENARIOS["nan_wind"]()[2]
    winds = [lambda t: (0.6, -0.5), lambda t: (3.0, 16.0), nan, lambda t: (-2.0, -15.0), lambda t: (0.6, -0.5)]
    run_ensemble(g, P, winds, 600.0, 4)


def test_mid_levels_and_accumulate(gpu_lib):
    g, P, winds, DT, n = scenario_members("growing_winds", SIGNS[:3])
    run_ensemble(g, P, winds, DT, 4, mid_levels=2)
    run_ensemble(g, P, winds, DT, 3, accumulate=True)


def test_set_members_one_is_the_single_model(gpu_lib):
    g, P, wind, DT, n = SCENARIOS["growing_winds"]()
    outs = []
    for call in (False, True):
        if not call:
            eng = ensemble_engine(g, P, 1)  # B200Engine calls picles_set_members only for E > 1
        else:  # the same handle with picles_set_members(h, 1) called before the grid
            import ctypes as C
            from picles_b200.engine import B200Engine
            eng = B200Engine.__new__(B200Engine)
            eng.lib = gpu_lib
            eng.h = C.c_void_p()
            assert gpu_lib.picles_create(C.byref(eng.h), 0) == 0
            assert gpu_lib.picles_set_members(eng.h, 1) == 0
            eng.Nx, eng.Ny, eng.ny, eng.members, eng._nodes = g["Nx"], g["Ny"], g["Ny"], 1, (g["Ny"], g["Nx"])
            Mc = np.ascontiguousarray(g["M_const"], np.float64)
            mask = np.ascontiguousarray(g["mask"], np.uint8)
            assert gpu_lib.picles_set_grid(eng.h, g["Nx"], g["Ny"], g["bx"], g["by"], 0, g["Ny"], 0,
                                           mask.ctypes.data, None, Mc.ctypes.data, None) == 0
            eng.params = P
            assert gpu_lib.picles_set_params(eng.h, C.byref(P)) == 0
        eng.seed(*wind(0.0))
        before = eng.launch_count()
        t = 0.0
        for _ in range(n):
            eng.step(t, DT, *wind(t), *wind(t + DT))
            t += DT
        launches = eng.launch_count() - before
        outs.append((eng.state(), eng.particles(), launches, eng.energy_sum(), eng.member_energy_sums()))
    (S0, p0, l0, e0, m0), (S1, p1, l1, e1, m1) = outs
    assert bits_equal(S0, S1) and l0 == l1
    for k in ("t", "dt"):
        assert bits_equal(p0[k], p1[k])
    assert np.array_equal(p0["flags"], p1["flags"])
    assert bits_equal(np.array([e0]), m0) and bits_equal(np.array([e1]), m1)


def test_member_energy_sums_equal_single_models(gpu_lib):
    g, P, winds, DT, n = scenario_members("land_block", SIGNS)
    E = len(winds)
    eng = ensemble_engine(g, P, E)
    singles = [ensemble_engine(g, P, 1) for _ in range(E)]
    u0, v0 = stack(winds, g, 0.0)
    eng.seed(u0, v0)
    for m, s in enumerate(singles):
        s.seed(u0[m], v0[m])
    t = 0.0
    for _ in range(3):
        ut, vt = stack(winds, g, t)
        ut1, vt1 = stack(winds, g, t + DT)
        eng.step(t, DT, ut, vt, ut1, vt1)
        for m, s in enumerate(singles):
            s.step(t, DT, ut[m], vt[m], ut1[m], vt1[m])
        t += DT
    sums = eng.member_energy_sums()
    assert bits_equal(sums, np.array([s.energy_sum() for s in singles]))
    rows = eng.row_reach()
    assert rows.shape == (E, g["Ny"])
    for m, s in enumerate(singles):
        assert np.array_equal(rows[m], s.row_reach())
        f, fs = eng.fields(), s.fields()
        for k in ("Hs", "c_x", "c_y"):
            assert bits_equal(f[k][m], fs[k])


def test_refusals_leave_the_device_state_alone(gpu_lib):
    import ctypes as C

    from picles_b200._abi import PiclesError
    from picles_b200.engine import B200Engine
    g, P, winds, DT, n = scenario_members("minimal", SIGNS[:2])
    # grid-time refusals: strip cut, too many particles; set_members after the grid
    for kw in (dict(j0=0, ny_local=g["Ny"] - 1), dict(halo=1)):
        with pytest.raises(PiclesError, match="ERR_ARG.*ensemble"):
            B200Engine(g["Nx"], g["Ny"], g["bx"], g["by"], g["mask"][: kw.get("ny_local", g["Ny"])], P,
                       M_const=g["M_const"], members=2, **kw)
    big = cartesian_grid(1024, 1024)
    with pytest.raises(PiclesError, match="ERR_ARG.*2\\^31"):
        B200Engine(1024, 1024, big["bx"], big["by"], big["mask"], P, M_const=big["M_const"], members=2048)
    eng = ensemble_engine(g, P, 2)
    assert gpu_lib.picles_set_members(eng.h, 3) == -5  # PICLES_ERR_STATE after the grid
    u0, v0 = stack(winds, g, 0.0)
    eng.seed(u0, v0)
    eng.step(0.0, DT, u0, v0, *stack(winds, g, DT))
    S, p = eng.state(), eng.particles()
    calls = [lambda: eng.halo_rows(), lambda: eng.halo_widen(2), lambda: eng.halo_buffers(), lambda: eng.halo_pack(),
             lambda: eng.halo_unpack(), lambda: eng.halo_exchange(), lambda: eng.step_strip(DT, DT),
             lambda: eng.set_wind_mesh([0, 1], [0, 1], [0, 1], np.zeros((2, 2, 2)), np.zeros((2, 2, 2)), 0.0, 0.0),
             lambda: eng.seed_wind_mesh(0.0), lambda: eng.step_wind_mesh(DT, DT), lambda: eng.stage_wind_mesh(DT, DT),
             lambda: eng.sample_wind_mesh(0.0), lambda: eng.checkpoint(), lambda: eng.restore(np.zeros(64, np.uint8))]
    for call in calls:
        with pytest.raises(PiclesError, match="ERR_ARG.*ensemble"):
            call()
    assert gpu_lib.picles_comm_init(eng.h, b"\0" * 128, 0, 1, None) == -1
    assert gpu_lib.picles_comm_destroy(eng.h) == -1
    assert bits_equal(S, eng.state())
    p2 = eng.particles()
    for k in ("z", "t", "dt"):
        assert bits_equal(p[k], p2[k])
    assert np.array_equal(p["flags"], p2["flags"])


def test_ensemble_model_through_run(gpu_lib):
    """WaveGrowth2DEnsemble through init_particles / time_step / Simulations.run with cash_store: every member equals
    the WaveGrowth2D with its winds"""
    from picles_b200.Models import WaveGrowth2D, WaveGrowth2DEnsemble
    from picles_b200.Simulations.run import Simulation, run
    from test_ensemble import WINDS as winds, ensemble_kwargs
    ens = WaveGrowth2DEnsemble(winds=winds, **ensemble_kwargs())
    sim = Simulation(ens, 600.0, stop_time=3 * 600.0, verbose=False)
    run(sim, cash_store=True)
    for m, w in enumerate(winds):
        single = WaveGrowth2D(winds=w, **ensemble_kwargs())
        s = Simulation(single, 600.0, stop_time=3 * 600.0, verbose=False)
        run(s, cash_store=True)
        assert bits_equal(ens.State[m], single.State)
        assert len(sim.store.store) == len(s.store.store)
        for a, b in zip(sim.store.store, s.store.store):
            assert bits_equal(a[m], b)
        pe, ps = ens.ParticleCollection, single.ParticleCollection
        assert bits_equal(pe.u[m], ps.u) and bits_equal(pe.t[m], ps.t)
        assert bits_equal(ens.member_energy_sums()[m:m + 1], np.array([single.engine.energy_sum()]))
