"""GPU tests (-m gpu) of ensembles at the sizes and launch limits they run at: every member against an oracle run with
that member's winds, bit for bit after every step, on handles large enough for the graded wind-upload pipeline of
advance_range (2^20 nodes and more), with block edges inside members, every block of an AutoTsit5 step holding parked
particles, and 65535 members (the largest launch dimension picles_set_members accepts).

Every case first checks its premise: the kernels launched per step are the row blocks of ensemble_scale_cases.
graded_blocks (twice that under AutoTsit5: k_advance and k_advance_resume per block), plus one gather.  The energy sums
are compared with energy_sum_restated, an independent statement of the reduction's order, bit for bit."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle
from common import BND_PERIODIC, TALLY_NAMES, bits_equal, cartesian_grid, compare_models, default_params, make_oracle
from ensemble_scale_cases import energy_sum_restated, graded_blocks, member_winds
from test_gpu_ensemble import ensemble_engine

pytestmark = pytest.mark.gpu

DT = 600.0


def compare_group(ref, out, members, autotsit5, what=""):
    """every member in `members` against the one oracle `ref` (members with the same winds): the checks of
    test_gpu_ensemble.compare_member, over the group at once"""
    S, p, sol = out
    ms = np.asarray(members)
    tag = f"{what}members {ms[:4].tolist()}{'...' if ms.size > 4 else ''}"
    Sr = ref.state()
    assert bits_equal(np.broadcast_to(Sr[:, None], (3, ms.size) + Sr.shape[1:]), S[:, ms]), f"{tag}: State differs"
    pr = ref.particles()
    act = (pr["flags"] & 8) != 0
    live = act & ((pr["flags"] & 4) == 0)
    for k in range(5):
        assert bits_equal(np.broadcast_to(pr["z"][k][act], (ms.size, int(act.sum()))), p["z"][k][ms][:, act]), \
            f"{tag}: particle component {k} differs"
    assert bits_equal(np.broadcast_to(pr["t"][act], (ms.size, int(act.sum()))), p["t"][ms][:, act]), f"{tag}: t differs"
    assert bits_equal(np.broadcast_to(pr["dt"][live], (ms.size, int(live.sum()))), p["dt"][ms][:, live]), \
        f"{tag}: dt differs"
    assert np.array_equal(np.broadcast_to(pr["flags"][act], (ms.size, int(act.sum()))), p["flags"][ms][:, act]), \
        f"{tag}: flags differ"
    assert np.array_equal(np.broadcast_to(pr["status"][act], (ms.size, int(act.sum()))), p["status"][ms][:, act]), \
        f"{tag}: status differs"
    if autotsit5:
        assert np.array_equal(np.broadcast_to(ref.solver_state()[act], (ms.size, int(act.sum()))), sol[ms][:, act]), \
            f"{tag}: AutoSwitch state differs"


def check_counters(eng, refs, owner, what=""):
    """the ensemble's counters: the sums (and maxima) over its members' oracles"""
    c = eng.counters()
    cr = [r.counters() for r in refs]
    used = np.bincount(owner, minlength=len(refs))
    for name in TALLY_NAMES:
        if name in ("reach", "max_attempts"):
            assert c[name] == max(x[name] for x, u in zip(cr, used) if u), f"{what}{name}"
        else:
            assert c[name] == sum(int(u) * x[name] for x, u in zip(cr, used)), f"{what}{name}"


def check_energy(eng, E, g):
    """member_energy_sums and energy_sum against the restatement of the reduction over the downloaded State"""
    e = eng.state()[0].reshape(E, g["Ny"] * g["Nx"])
    assert bits_equal(eng.member_energy_sums(), energy_sum_restated(e)), "member_energy_sums"
    assert bits_equal(np.array([eng.energy_sum()]), np.array([energy_sum_restated(e.ravel())])), "energy_sum"


def run_members(g, P, winds, nsteps, owner, DTs=DT, mid_step=None, t1_only_step=None, split=False, autotsit5=False):
    """seed + nsteps of one ensemble handle (member m has the winds of oracle owner[m]) stepped through picles_step,
    and of one oracle per distinct wind; compared after every step.  winds(t) -> (U, V) of shape (R, Ny, Nx) for the R
    oracles.  mid_step: the step that has two intermediate wind levels; t1_only_step: the step that uploads only the
    t+DT level (the t level is the previous step's t+DT level, swapped in on the device).  split: a second handle
    takes the same steps through upload_winds + step_advance + step_project_remesh (one block) and is held to the same
    oracles.  Returns the graded handle and the oracles."""
    E = owner.size
    R = int(owner.max()) + 1
    engs = {"graded": ensemble_engine(g, P, E)}
    if split:
        engs["split"] = ensemble_engine(g, P, E)
    refs = [make_oracle(g, P) for _ in range(R)]
    groups = [np.flatnonzero(owner == k) for k in range(R)]
    mult = 2 if autotsit5 else 1
    expect = {"graded": len(graded_blocks(g["Ny"] * E, g["Nx"], True)) * mult + 1,
              "split": len(graded_blocks(g["Ny"] * E, g["Nx"], False)) * mult + 1}
    U0, V0 = winds(0.0)
    for eng in engs.values():
        eng.seed(U0[owner], V0[owner])
    for k, r in enumerate(refs):
        r.seed(U0[k], V0[k])
    t = 0.0
    for step in range(nsteps):
        Ut, Vt = winds(t)
        Ut1, Vt1 = winds(t + DTs)
        if step == mid_step:
            lv = [winds(t + DTs * j / 3.0) for j in (1, 2)]
            for eng in engs.values():
                eng.set_wind_midlevels([a[owner] for a, _ in lv], [b[owner] for _, b in lv])
            for k, r in enumerate(refs):
                r.set_wind_midlevels([a[k] for a, _ in lv], [b[k] for _, b in lv])
        up = (None, None) if step == t1_only_step else (Ut[owner], Vt[owner])
        for mode, eng in engs.items():
            before = eng.launch_count()
            if mode == "graded":
                eng.step(t, DTs, *up, Ut1[owner], Vt1[owner])
            else:
                eng.upload_winds(*up, Ut1[owner], Vt1[owner])
                eng.step_advance(t, DTs)
                eng.step_project_remesh(t, DTs)
            launched = eng.launch_count() - before
            assert launched == expect[mode], f"{mode} step {step}: {launched} launches, the premise is {expect[mode]}"
        for k, r in enumerate(refs):
            r.step(t, DTs, Ut[k], Vt[k], Ut1[k], Vt1[k])
        t += DTs
        for mode, eng in engs.items():
            out = (eng.state(), eng.particles(), eng.solver_state() if autotsit5 else None)
            for k, r in enumerate(refs):
                compare_group(r, out, groups[k], autotsit5, f"{mode} step {step}: ")
            check_counters(eng, refs, owner, f"{mode} step {step}: ")
    for eng in engs.values():
        check_energy(eng, E, g)
    return engs["graded"], refs


def random_winds(g, E, seed, lo=6.0, hi=14.0):
    rng = np.random.default_rng(seed)
    return member_winds(g, rng.uniform(lo, hi, E), rng.uniform(0.0, 2 * np.pi, E), rng.uniform(0.0, 2 * np.pi, E))


@pytest.mark.parametrize("E,blocks", [(1023, 1), (1024, 7)])
def test_threshold_of_the_graded_pipeline(gpu_lib, E, blocks):
    """32 x 32 periodic x E: 1 047 552 nodes run as one block, 1 048 576 (= PIPE_MIN_NODES) as seven.  Periodic, so
    the first and last row of every member, where the block edges fall, hold active particles"""
    g = cartesian_grid(32, 32, bx=BND_PERIODIC, by=BND_PERIODIC)
    assert len(graded_blocks(32 * E, 32, True)) == blocks
    run_members(g, default_params(periodic_boundary=True), random_winds(g, E, E), 2, np.arange(E))


def test_eighth_block_takes_the_rest(gpu_lib):
    """16 x 16 periodic x 4500: all eight work-queue slots, the eighth block the last 2048 rows"""
    g = cartesian_grid(16, 16, bx=BND_PERIODIC, by=BND_PERIODIC)
    E = 4500
    b = graded_blocks(16 * E, 16, True)
    assert len(b) == 8 and b[-1][1] - b[-1][0] == 2048
    run_members(g, default_params(periodic_boundary=True), random_winds(g, E, 11), 2, np.arange(E))


def test_bench_shape_blocks_inside_members(gpu_lib):
    """51 x 51 x 512 (C1): every block edge inside a member; a step with two intermediate levels, then a step that
    uploads only the t+DT level; a second handle takes the same steps through the phase-split calls (one block)"""
    g = cartesian_grid(51, 51)
    E = 512
    b = graded_blocks(51 * E, 51, True)
    assert len(b) == 7 and all(a % 51 for a, _, _ in b[1:])
    run_members(g, default_params(), random_winds(g, E, 51), 3, np.arange(E), mid_step=1, t1_only_step=2, split=True)


def test_autotsit5_parks_particles_in_many_blocks(gpu_lib):
    """32 x 32 periodic x 1024 on 300 m cells under AutoTsit5: slow-wind members that switch to Rosenbrock23 in each of
    the seven blocks, interleaved with 16.5-19.5 m/s members that never switch; every k_advance_resume walks the pending
    list of the whole step"""
    g = cartesian_grid(32, 32, dx=300.0, dy=300.0, bx=BND_PERIODIC, by=BND_PERIODIC)
    P = default_params(DT=1200.0, wind_min_squared=2.0, solver="AutoTsit5", periodic_boundary=True)
    E = 1024
    # about three in each block (members 0-1, 2-7, 8-25, 26-79, 80-241, 242-727, 728-1023)
    stiff = np.array([0, 1, 3, 5, 7, 9, 15, 25, 30, 50, 70, 100, 180, 240, 300, 500, 700, 750, 900, 1023])
    rng = np.random.default_rng(3)
    speed = rng.uniform(16.5, 19.5, E)
    speed[stiff] = rng.uniform(1.6, 2.0, stiff.size)
    winds = member_winds(g, speed, rng.uniform(0.0, 2 * np.pi, E), rng.uniform(0.0, 2 * np.pi, E))
    eng, refs = run_members(g, P, winds, 2, np.arange(E), DTs=1200.0, autotsit5=True)
    switched = np.array([r.counters()["n_stiff_switches"] for r in refs])
    blocks = graded_blocks(32 * E, 32, True)
    block_of = lambda m: next(c for a, e, c in blocks if a <= 32 * m < e)
    hit = {block_of(m) for m in np.flatnonzero(switched)}
    assert len(hit) >= 3, f"parked particles only in blocks {sorted(hit)}"
    assert np.count_nonzero(switched == 0) > E // 2


def test_autotsit5_single_model_stiff_band_across_block_edges(gpu_lib):
    """1024 x 1024 (2^20 nodes, four graded blocks) under AutoTsit5: a band of rows 40..299 that switches to
    Rosenbrock23 across the edges at rows 64 and 256, against the threaded oracle"""
    from picles_b200.engine import B200Engine
    Nx = Ny = 1024
    g = cartesian_grid(Nx, Ny, dx=300.0, dy=300.0)
    P = default_params(DT=1200.0, wind_min_squared=2.0, solver="AutoTsit5")
    assert [(a, e) for a, e, _ in graded_blocks(Ny, Nx, True)] == [(0, 64), (64, 256), (256, 832), (832, 1024)]
    base = member_winds(g, [28.0], [0.64], [0.3])
    scale = np.where((np.arange(Ny) >= 40) & (np.arange(Ny) < 300), 10.0 / 28.0, 1.0)[:, None]

    def wind(t):
        u, v = base(t)
        return u[0] * scale, v[0] * scale

    eng = B200Engine(Nx, Ny, g["bx"], g["by"], g["mask"], P, M_const=g["M_const"])
    ref = make_oracle(g, P, variant="omp", threads=os.cpu_count() or 8)
    eng.seed(*wind(0.0))
    ref.seed(*wind(0.0))
    t, rows_switched = 0.0, np.zeros(Ny, bool)
    for step in range(2):
        w = [*wind(t), *wind(t + 1200.0)]
        before = eng.launch_count()
        eng.step(t, 1200.0, *w)
        assert eng.launch_count() - before == 4 * 2 + 1, f"step {step}: premise"
        ref.step(t, 1200.0, *w)
        t += 1200.0
        compare_models(ref, eng, check_aux=False)
        assert np.array_equal(ref.solver_state(), eng.solver_state()), f"step {step}: AutoSwitch state differs"
        rows_switched |= (ref.solver_state() >= 64).any(axis=1)  # Rosenbrock23 current
    r = np.flatnonzero(rows_switched)
    assert ref.counters()["n_stiff_switches"] > 0
    assert r.min() < 64 and np.any((r >= 64) & (r < 256)) and r.max() >= 256, "the band does not cross two block edges"
    assert r.min() >= 40 and r.max() < 320, "stiff rows outside the band"
    assert bits_equal(np.array([eng.energy_sum()]), np.array([energy_sum_restated(eng.state()[0].ravel())]))


def families(g, R=21):
    """R = 7 families (direction, shape of the modulation) x 3 scales of wind: wind k = 3 * family + scale"""
    fam, sc = np.arange(R) // 3, np.arange(R) % 3
    return member_winds(g, 5.0 + 3.5 * sc, 2 * np.pi * fam / 7.0 + 0.2, 0.9 * fam + 0.4 * sc)


def test_65535_members(gpu_lib):
    """4 x 4 periodic x 65535 (1 048 560 nodes, one block): member m has wind m mod 21, so neighbouring members always
    differ and a member offset by anything but a multiple of 21 changes bits.  Then the energy sums, the fields and the
    per-row reach of every member; 65535 member wind meshes (m mod 7) sampled on the device; 65536 and 0 members
    refused"""
    from picles_b200._abi import PiclesError
    from picles_b200.engine import B200Engine
    E = 65535
    g = cartesian_grid(4, 4, dx=20000.0, dy=20000.0, bx=BND_PERIODIC, by=BND_PERIODIC)
    P = default_params(periodic_boundary=True)
    owner = np.arange(E) % 21
    assert graded_blocks(4 * E, 4, True) == [(0, 4 * E, 0)]
    eng, refs = run_members(g, P, families(g), 2, owner)
    # fields: IEEE square root and division, the same bits in numpy
    S = eng.state()
    f = eng.fields()
    e, mx, my = S[0], S[1], S[2]
    amp = np.sqrt(mx * mx + my * my)
    den = 2.0 * (amp * amp)
    assert bits_equal(f["Hs"], 4.0 * np.sqrt(e))
    assert bits_equal(f["c_x"], mx * e / den) and bits_equal(f["c_y"], my * e / den)
    for k, r in enumerate(refs):
        fr = r.fields()
        for name in ("Hs", "c_x", "c_y"):
            assert bits_equal(np.broadcast_to(fr[name], (np.count_nonzero(owner == k),) + fr[name].shape),
                              f[name][owner == k]), name
    rows = eng.row_reach()
    assert rows.shape == (E, 4)
    reach = np.array([r.counters()["reach"] for r in refs])
    assert np.array_equal(rows.max(axis=1), reach[owner])

    # 65535 meshes on shared knots, 7 distinct: the last chunk of 8 members of k_wind_sample_members is partial
    rng = np.random.default_rng(7)
    xw = np.array([-15000.0, 10000.0, 35000.0, 90000.0])
    yw = np.array([-5000.0, 30000.0, 70000.0])
    tw = np.array([0.0, 900.0, 2500.0])
    Uk = 8.0 * rng.random((7, tw.size, yw.size, xw.size)) - 4.0
    Vk = 8.0 * rng.random((7, tw.size, yw.size, xw.size)) - 4.0
    eng.set_member_wind_meshes(xw, yw, tw, Uk[np.arange(E) % 7], Vk[np.arange(E) % 7], g["x"], g["y"])
    for t in (0.0, 450.0, 900.0, 2500.0, 1733.25, 3100.0, -700.0):
        u, v = eng.sample_wind_mesh(t)
        assert u.shape == (E, 4, 4)
        for k in range(7):
            ur, vr = oracle.wind_mesh_sample(xw, yw, tw, Uk[k], Vk[k], g["x"], g["y"], t)
            ms = np.arange(k, E, 7)
            assert bits_equal(u[ms], np.broadcast_to(ur, (ms.size, 4, 4))), f"t = {t}: mesh {k}, u"
            assert bits_equal(v[ms], np.broadcast_to(vr, (ms.size, 4, 4))), f"t = {t}: mesh {k}, v"
    eng.close()

    h = C.c_void_p()
    assert gpu_lib.picles_create(C.byref(h), 0) == 0
    try:
        assert gpu_lib.picles_set_members(h, 65536) == -1
        assert gpu_lib.picles_set_members(h, 0) == -1
        assert gpu_lib.picles_set_members(h, 65535) == 0
    finally:
        gpu_lib.picles_destroy(h)
    with pytest.raises(PiclesError, match="ERR_ARG"):
        B200Engine(4, 4, g["bx"], g["by"], g["mask"], P, M_const=g["M_const"], members=65536)
