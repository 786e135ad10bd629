"""GPU tests (-m gpu): the CUDA path, called through the C ABI, against the CPU oracle.

Bit-exact for everything: pmath.h + explicit fma + --fmad=false make device and oracle
arithmetic identical, so the tolerance the north-star allows for floating point
(<= 1e-6 relative on lne and cg_bar) is checked as well but is never the binding bound."""
import numpy as np
import pytest

from common import BND_NONPERIODIC, cartesian_grid, compare_models, default_params, make_oracle
from scenarios import SCENARIOS, run_pair

pytestmark = pytest.mark.gpu

REL_TOL = 1e-6  # north_star: fields within 1e-6 relative of the Float64 reference run


def engine_for(grid, P, **kw):
    from picles_b200.engine import B200Engine
    return B200Engine(grid["Nx"], grid["Ny"], grid["bx"], grid["by"], grid["mask"], P, M=grid["M"],
                      M_const=grid["M_const"], pc=grid["pc"], **kw)


class StripSet:
    """N strip handles on one GPU with the host-driven halo exchange a multi-GPU host
    performs (here: device-to-device copies through the C ABI)."""

    def __init__(self, grid, P, nstrips, halo, bounds=None):
        """bounds: the (first, end) rows of every strip; default: nstrips strips of nearly equal height"""
        from picles_b200._abi import BND_PERIODIC
        from picles_b200.engine import B200Engine
        self.g, self.ns, self.halo = grid, nstrips, halo
        self.periodic = grid["by"] == BND_PERIODIC
        Nx, Ny = grid["Nx"], grid["Ny"]
        self.Nx, self.Ny = Nx, Ny
        self.bounds = bounds or [(Ny * r // nstrips, Ny * (r + 1) // nstrips) for r in range(nstrips)]
        assert len(self.bounds) == nstrips
        self.e = []
        for a, b in self.bounds:
            M = grid["M"][:, a:b] if grid["M"] is not None else None
            pc = grid["pc"][a:b] if grid["pc"] is not None else None
            self.e.append(B200Engine(Nx, Ny, grid["bx"], grid["by"], grid["mask"][a:b], P, M=M, M_const=grid["M_const"],
                                     pc=pc, j0=a, ny_local=b - a, halo=halo))

    def _full(self, x):
        return np.broadcast_to(np.asarray(x, np.float64), (self.Ny, self.Nx))

    def seed(self, u0, v0):
        u0, v0 = self._full(u0), self._full(v0)
        for (a, b), e in zip(self.bounds, self.e):
            e.seed(u0[a:b], v0[a:b])

    def step(self, t, DT, ut, vt, ut1, vt1):
        w = [self._full(x) for x in (ut, vt, ut1, vt1)]
        for (a, b), e in zip(self.bounds, self.e):
            e.upload_winds(*[x[a:b] for x in w])
            e.step_advance(t, DT)
            e.halo_pack()
        for e in self.e:
            e.synchronize()
        bufs = [e.halo_buffers() for e in self.e]
        ns = self.ns
        for r, e in enumerate(self.e):
            (slo, shi, rlo, rhi), nb = bufs[r]
            lo, hi = r - 1, r + 1
            if self.periodic:
                lo, hi = (lo + ns) % ns, hi % ns
            if 0 <= lo < ns:   # my lower halo <- lower neighbour's last rows (its send_hi)
                e.copy_dev(rlo, bufs[lo][0][1], nb)
            if 0 <= hi < ns:   # my upper halo <- upper neighbour's first rows (its send_lo)
                e.copy_dev(rhi, bufs[hi][0][0], nb)
            e.halo_unpack()
        for e in self.e:
            e.step_project_remesh(t, DT)

    def state(self):
        return np.concatenate([e.state() for e in self.e], axis=1)

    def particles(self):
        ps = [e.particles() for e in self.e]
        return {k: np.concatenate([p[k] for p in ps], axis=(1 if k == "z" else 0)) for k in ps[0]}

    def counters(self):
        cs = [e.counters() for e in self.e]
        out = {k: sum(c[k] for c in cs) for k in cs[0]}
        out["reach"] = max(c["reach"] for c in cs)
        out["max_attempts"] = max(c["max_attempts"] for c in cs)
        return out


def tolerant_compare(ref, dut):
    """north-star tolerance check (<= 1e-6 relative on lne and cg_bar); a strict subset of
    compare_models, kept so the stated tolerance is written in a test."""
    pr, pd = ref.particles(), dut.particles()
    act = (pr["flags"] & 8) != 0
    for k in range(3):
        a, b = pr["z"][k][act], pd["z"][k][act]
        fin = np.isfinite(a) & np.isfinite(b)
        assert np.all(np.abs(a[fin] - b[fin]) <= REL_TOL * np.maximum(np.abs(a[fin]), 1e-300))
        assert np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(a[np.isinf(a)], b[np.isinf(a)])


@pytest.mark.parametrize("name", sorted(SCENARIOS))
def test_gpu_matches_oracle_bit_exact(gpu_lib, name):
    g, P, wind, DT, n = SCENARIOS[name]()

    def both(ref, dut):
        compare_models(ref, dut)
        tolerant_compare(ref, dut)

    run_pair(make_oracle(g, P), engine_for(g, P), wind, DT, n, both)


@pytest.mark.parametrize("name,nstrips,halo", [("minimal", 2, 2), ("periodic_grid", 2, 5), ("tripolar", 3, 6),
                                               ("land_block", 4, 2), ("fast_box", 3, 5), ("periodic_x_only", 2, 3),
                                               ("growing_winds_persist", 2, 2), ("growing_winds", 3, 2),
                                               ("pulse_winds", 2, 2), ("dp5_blowup", 2, 2)])
def test_gpu_strips_match_oracle(gpu_lib, name, nstrips, halo):
    g, P, wind, DT, n = SCENARIOS[name]()
    run_pair(make_oracle(g, P), StripSet(g, P, nstrips, halo), wind, DT, n, compare_models)


def test_gpu_reach_beyond_halo_is_an_error(gpu_lib):
    """host-driven exchange with too few rows: the gather refuses (PICLES_ERR_HALO) and changes nothing"""
    from picles_b200 import PiclesError
    g, P, wind, DT, n = SCENARIOS["periodic_grid"]()
    s = StripSet(g, P, 2, 1)
    u0, v0 = wind(0.0)
    s.seed(u0, v0)
    with pytest.raises(PiclesError, match="ERR_HALO"):
        t = 0.0
        for _ in range(n):
            before = s.state()
            s.step(t, DT, *wind(t), *wind(t + DT))
            t += DT
    assert np.array_equal(s.state().view(np.uint64), before.view(np.uint64))  # State untouched by the refused gather


@pytest.mark.parametrize("name,nstrips", [("fast_box", 3), ("periodic_grid", 2)])
def test_gpu_halo_widens_instead_of_failing(gpu_lib, name, nstrips):
    """SURVEY.md §8e 'falling back to a wider exchange': strips created with a halo of ONE row while the
    particles cross 2-4 cells per step.  The gather refuses, the host widens every strip to the rows the
    error names and repeats exchange + gather (the advance is not repeated): bit-exact against the oracle."""
    from picles_b200 import PiclesError
    g, P, wind, DT, n = SCENARIOS[name]()

    class Widening(StripSet):
        widened = 0

        def finish(self, t, DT):
            for e in self.e:
                e.halo_pack()
            for e in self.e:
                e.synchronize()
            bufs = [e.halo_buffers() for e in self.e]
            ns = self.ns
            for r, e in enumerate(self.e):
                (slo, shi, rlo, rhi), nb = bufs[r]
                lo, hi = r - 1, r + 1
                if self.periodic:
                    lo, hi = (lo + ns) % ns, hi % ns
                if 0 <= lo < ns:
                    e.copy_dev(rlo, bufs[lo][0][1], nb)
                if 0 <= hi < ns:
                    e.copy_dev(rhi, bufs[hi][0][0], nb)
                e.halo_unpack()
            need = 0
            for e in self.e:
                try:
                    e.step_project_remesh(t, DT)
                except PiclesError as ex:
                    assert "ERR_HALO" in str(ex)
                    need = max(need, int(str(ex).split("picles_halo_widen(")[1].split(")")[0]))
            return need

    # all strips see the global reach when the host all-reduces it first (what StripStepper's torch-p2p path does)
    class Validating(Widening):
        def step(self, t, DT, ut, vt, ut1, vt1):
            w = [self._full(x) for x in (ut, vt, ut1, vt1)]
            for (a, b), e in zip(self.bounds, self.e):
                e.upload_winds(*[x[a:b] for x in w])
                e.step_advance(t, DT)
            need = max(e.reach() for e in self.e)
            if need > self.e[0].halo_rows()[0]:
                type(self).widened += 1
                for e in self.e:
                    e.halo_widen(need)
            assert self.finish(t, DT) == 0

    s = Validating(g, P, nstrips, 1)
    assert s.e[0].halo_rows()[0] == 1 and s.e[0].halo_rows()[1] >= 4
    run_pair(make_oracle(g, P), s, wind, DT, n, compare_models)
    assert Validating.widened >= 1 and s.e[0].halo_rows()[0] >= 2

    # ... and the refusal itself: the strips exchange too few rows first, every gather refuses (each was told the
    # global reach), all widen to the rows the error names and repeat exchange + gather — not the advance
    class Refused(Widening):
        def step(self, t, DT, ut, vt, ut1, vt1):
            w = [self._full(x) for x in (ut, vt, ut1, vt1)]
            for (a, b), e in zip(self.bounds, self.e):
                e.upload_winds(*[x[a:b] for x in w])
                e.step_advance(t, DT)
            reach = max(e.reach() for e in self.e)
            for e in self.e:
                e.set_global_reach(reach)
            need = self.finish(t, DT)
            if need:
                assert need == reach
                type(self).widened += 1
                for e in self.e:
                    e.halo_widen(need)
                assert self.finish(t, DT) == 0

    s2 = Refused(g, P, nstrips, 1)
    run_pair(make_oracle(g, P), s2, wind, DT, n, compare_models)
    assert Refused.widened >= 1


def test_gpu_medium_box_against_threaded_oracle(gpu_lib):
    """512x384 homogeneous box, 5 steps: 196k particles, bit-exact against the oracle
    (OpenMP over particles in the ODE phase; deposit in canonical serial order)."""
    g = cartesian_grid(512, 384)
    P = default_params()
    o = make_oracle(g, P, variant="omp", threads=8)
    e = engine_for(g, P)
    run_pair(o, e, lambda t: (10.0, 10.0), 600.0, 5, lambda a, b: compare_models(a, b), every=5)


def test_gpu_headline_box_against_threaded_oracle(gpu_lib):
    """BASELINE.json configs[1] itself — the 4096 x 4096 homogeneous box the bench line is quoted on, 16.76 M
    particles — compared DIRECTLY with the oracle, all of it: State, particle state, flags, status and counters
    bit for bit after every one of three steps (OpenMP over particles in the oracle's ODE phase, its deposit in
    canonical serial order; about a minute of host time), both outflow edges included."""
    import os
    N = 4096
    g = cartesian_grid(N, N)
    P = default_params()
    o = make_oracle(g, P, variant="omp", threads=os.cpu_count() or 8)
    e = engine_for(g, P)
    run_pair(o, e, lambda t: (10.0, 10.0), 600.0, 3, lambda a, b: compare_models(a, b))
    c = e.counters()
    assert c["n_active"] == (N - 2) ** 2 and c["n_failed"] == 0 and c["reach"] == 1


def test_gpu_large_box_properties(gpu_lib):
    """C2-sized run (4096x4096, BASELINE.json configs[1]) checked through size-independent
    properties: every interior node far from the boundary carries the same bits as the
    same node of a small box (translation invariance of the homogeneous problem), total
    deposited energy equals the sum over particles, no failures, reach stays 1."""
    N = 4096
    g = cartesian_grid(N, N)
    P = default_params()
    e = engine_for(g, P)
    small = cartesian_grid(64, 64)
    es = engine_for(small, P)
    e.seed(10.0, 10.0)
    es.seed(10.0, 10.0)
    t = 0.0
    for _ in range(3):
        e.step(t, 600.0, 10.0, 10.0, 10.0, 10.0)
        es.step(t, 600.0, 10.0, 10.0, 10.0, 10.0)
        t += 600.0
    c = e.counters()
    assert c["n_active"] == (N - 2) ** 2 and c["n_failed"] == 0 and c["n_fixups"] == 0
    assert c["n_remesh_A"] == c["n_active"] and c["reach"] == 1
    S, Ss = e.state(), es.state()
    # wind blows towards +x,+y: nodes far downstream of the inflow edges are identical
    # everywhere, and equal to the far-downstream corner region of the small box
    ref = Ss[:, 40, 40]
    blk = S[:, 2000:2100, 3000:3100]
    assert np.array_equal(blk.view(np.uint64), np.broadcast_to(ref[:, None, None], blk.shape).copy().view(np.uint64))
    # upstream corner region matches the small box bit-for-bit (same fetch-limited pattern)
    assert np.array_equal(S[:, :32, :32].view(np.uint64), Ss[:, :32, :32].view(np.uint64))
    # energy sum accessor agrees with a host sum of the downloaded plane
    assert abs(e.energy_sum() - S[0].sum()) <= 1e-9 * S[0].sum()


def test_gpu_pipelined_wind_upload_equals_phase_split(gpu_lib):
    """picles_step on a strip large enough for the chunked upload (host winds copied on a
    second stream while earlier row blocks integrate) against upload_winds + the phase-split
    calls on the same inputs: same bits."""
    Nx, Ny = 1536, 1024
    g = cartesian_grid(Nx, Ny)
    P = default_params()
    a, b = engine_for(g, P), engine_for(g, P)
    x = np.linspace(0.0, 1.0, Nx)[None, :]
    y = np.linspace(0.0, 1.0, Ny)[:, None]

    def wind(t):
        f = 1.0 + 0.3 * np.sin(t / 3000.0)
        return (6.0 + 6.0 * x + 0 * y) * f, (-4.0 + 9.0 * y + 0 * x) * f

    u0, v0 = wind(0.0)
    a.seed(u0, v0)
    b.seed(u0, v0)
    t = 0.0
    for _ in range(3):
        w = [*wind(t), *wind(t + 600.0)]
        a.step(t, 600.0, *w)
        b.upload_winds(*w)
        b.step_advance(t, 600.0)
        b.step_project_remesh(t, 600.0)
        t += 600.0
    assert np.array_equal(a.state().view(np.uint64), b.state().view(np.uint64))
    pa, pb = a.particles(), b.particles()
    assert np.array_equal(pa["z"].view(np.uint64), pb["z"].view(np.uint64))
    assert a.counters()["n_substeps"] == b.counters()["n_substeps"]


def test_gpu_grid_metric_and_masks_bit_exact(gpu_lib):
    """k_grid_metric and k_make_boundaries (the device-side grid lookups) against the oracle:
    per-node projection kernel and great-circle coefficient with the same bits, total masks
    identical (incl. the 21x11 fixture of src/Grids/mask_utils_test.jl: 30 / 60)."""
    import oracle
    from common import BND_PERIODIC, BND_TRIPOLAR_NORTH, tripolar_grid
    rng = np.random.default_rng(7)
    Nx, Ny = 96, 70
    g = tripolar_grid(Nx, Ny)
    dx = rng.uniform(500.0, 120e3, (Ny, Nx))
    dy = rng.uniform(500.0, 120e3, (Ny, Nx))
    ang = rng.uniform(-180.0, 180.0, (Ny, Nx))
    lat = np.linspace(-89.9, 89.9, Ny)[:, None] + 0 * dx
    from picles_b200.engine import B200Engine
    e = B200Engine(Nx, Ny, BND_PERIODIC, BND_TRIPOLAR_NORTH, g["mask"], default_params(),
                   metric=dict(dx=dx, dy=dy, angle_dx=ang, lat=lat))
    M, pc = e.metric()
    Mo, pco = oracle.grid_metric(dx, dy, ang, lat)
    assert np.array_equal(M.view(np.uint64), Mo.view(np.uint64))
    assert np.array_equal(pc.view(np.uint64), pco.view(np.uint64))
    # masks
    ocean = np.ones((11, 21), np.uint8)
    ocean[4:10, 9:20] = 0
    tot = e.make_boundaries(ocean, BND_NONPERIODIC, BND_NONPERIODIC)
    assert np.array_equal(tot, oracle.make_boundaries(ocean, BND_NONPERIODIC, BND_NONPERIODIC))
    assert (tot == 2).sum() == 30 and (tot == 3).sum() == 60 and (tot == 0).sum() == 36 and (tot == 1).sum() == 105
    big = (rng.uniform(size=(301, 517)) > 0.35).astype(np.uint8)
    for bx, by in ((0, 0), (1, 0), (1, 1), (1, 2), (0, 1)):
        assert np.array_equal(e.make_boundaries(big, bx, by), oracle.make_boundaries(big, bx, by))


def test_gpu_tripolar_run_with_device_formed_metric(gpu_lib):
    """the tripolar scenario with its kernel and great-circle term formed on the device from
    (dx, dy, angle_dx, lat), against the oracle fed with oracle.grid_metric of the same planes."""
    import oracle
    from common import tripolar_grid
    Nx, Ny = 48, 36
    ocean = np.ones((Ny, Nx), np.uint8)
    ocean[:2, :] = 0
    ocean[10:16, 8:15] = 0
    g = tripolar_grid(Nx, Ny, ocean=ocean)
    lon = -280.0 + (np.arange(Nx) + 0.5) * 360.0 / Nx
    lat = -70.0 + (np.arange(Ny) + 0.5) * 159.0 / Ny
    LON, LAT = np.meshgrid(lon, lat)
    ang = 40.0 * np.clip((LAT - 60.0) / 30.0, 0.0, 1.0) * np.sin(np.deg2rad(2 * (LON + 280.0)))
    dx = np.maximum(6.371e6 * np.cos(np.deg2rad(LAT)) * np.deg2rad(360.0 / Nx), 2000.0) / 60.0
    dy = np.full_like(dx, 6.371e6 * np.deg2rad(159.0 / Ny)) / 60.0
    M, pc = oracle.grid_metric(dx, dy, ang, LAT)
    g = dict(g, M=M, pc=pc)
    P = default_params(DT=1200.0, periodic_boundary=True)
    from picles_b200.engine import B200Engine
    e = B200Engine(Nx, Ny, g["bx"], g["by"], g["mask"], P, metric=dict(dx=dx, dy=dy, angle_dx=ang, lat=LAT))
    wind = lambda t: (15.0, -10.0 * np.cos(5 * t / (3600 * 2 * np.pi)))
    run_pair(make_oracle(g, P), e, wind, 1200.0, 5, compare_models)
    assert e.counters()["reach"] >= 1


def test_gpu_output_fields_and_async_snapshots(gpu_lib):
    """output path: derived fields (Hs, group velocity) bit-exact against the oracle, and
    asynchronous State snapshots taken while the next steps run equal the synchronous reads."""
    g, P, wind, DT, n = SCENARIOS["land_block"]()
    o, e = make_oracle(g, P), engine_for(g, P)
    u0, v0 = wind(0.0)
    o.seed(u0, v0)
    e.seed(u0, v0)
    stage = e.pinned_state_buffer()
    t = 0.0
    snaps, refs = [], []
    for k in range(4):
        w = [*wind(t), *wind(t + DT)]
        o.step(t, DT, *w)
        e.step(t, DT, *w)
        t += DT
        if k > 0:
            e.snapshot_wait()
            snaps.append(stage.copy())
        e.snapshot_begin(stage)          # returns at once; the next step overwrites State meanwhile
        refs.append(o.state())
        fo, fe = o.fields(), e.fields()
        for key in ("Hs", "c_x", "c_y"):
            assert np.array_equal(np.isnan(fo[key]), np.isnan(fe[key]))
            ok = ~np.isnan(fo[key])
            assert np.array_equal(fo[key][ok].view(np.uint64), fe[key][ok].view(np.uint64)), key
    e.snapshot_wait()
    snaps.append(stage.copy())
    for a, b in zip(refs, snaps):
        assert np.array_equal(a.view(np.uint64), b.view(np.uint64))


@pytest.mark.parametrize("name", ["growing_winds_persist", "tripolar", "maxiters", "pulse_winds", "dp5_blowup"])
def test_gpu_checkpoint_resume_is_bit_identical(gpu_lib, name):
    """run k steps, checkpoint, continue; a fresh handle restored from the blob continues with the
    same bits (particle controller memory, pending dt resets, retcodes and wind level included)."""
    g, P, wind, DT, n = SCENARIOS[name]()
    a = engine_for(g, P)
    a.seed(*wind(0.0))
    t = 0.0
    for _ in range(3):
        a.step(t, DT, *wind(t), *wind(t + DT))
        t += DT
    blob = a.checkpoint()
    b = engine_for(g, P)
    b.restore(blob)
    tb = t
    for _ in range(3):
        a.step(t, DT, None, None, *wind(t + DT))       # only the new level is uploaded, as run! does
        t += DT
    for _ in range(3):
        b.step(tb, DT, None, None, *wind(tb + DT))
        tb += DT
    assert np.array_equal(a.state().view(np.uint64), b.state().view(np.uint64))
    pa, pb = a.particles(), b.particles()
    for k in ("z", "t", "dt"):
        assert np.array_equal(pa[k].view(np.uint64), pb[k].view(np.uint64)), k
    assert np.array_equal(pa["flags"], pb["flags"]) and np.array_equal(pa["status"], pb["status"])
    ca, cb = a.counters(), b.counters()
    assert all(ca[k] == cb[k] for k in ("n_substeps", "n_rhs", "n_rejects", "n_failed", "reach"))
    # a blob of another grid is refused
    other = engine_for(cartesian_grid(9, 7), default_params())
    from picles_b200 import PiclesError
    with pytest.raises(PiclesError, match="ERR_ARG"):
        other.restore(blob)
    # ... and so is one written under other parameters (the restored controller / AutoSwitch state would not match)
    P2 = default_params(DT=DT, dtmin=2e-4)
    with pytest.raises(PiclesError, match="different parameters"):
        engine_for(g, P2).restore(blob)
    # intermediate wind levels staged for the next step are not part of a blob: saving then is refused
    a.set_wind_midlevels([wind(t + DT / 2)[0]], [wind(t + DT / 2)[1]])
    with pytest.raises(PiclesError, match="intermediate wind levels"):
        a.checkpoint()


def test_gpu_attempt_histogram_and_launch_count(gpu_lib):
    """the work per particle-step is data-dependent (SURVEY.md §8d): its distribution is reported per step, and
    the library counts the kernels it launches (bench.py's gpu_launches is this count, not arithmetic)"""
    for name in ("growing_winds", "minimal"):
        g, P, wind, DT, n = SCENARIOS[name]()
        e = engine_for(g, P)
        e.seed(*wind(0.0))
        t = 0.0
        for _ in range(3):
            k0 = e.launch_count()
            e.step(t, DT, *wind(t), *wind(t + DT))
            assert e.launch_count() - k0 == 2          # k_advance + k_project_remesh
            t += DT
            c, h = e.counters(), e.attempt_histogram()
            assert h.sum() == c["n_integrated"]
            assert int(np.nonzero(h)[0].max()) == min(c["max_attempts"], h.size - 1)
            assert int((h * np.arange(h.size)).sum()) == c["n_substeps"] + c["n_rejects"] or c["max_attempts"] >= h.size - 1
        assert e.attempt_histogram(8).sum() == c["n_integrated"]


def test_gpu_state_roundtrip_and_accessors(gpu_lib):
    g = cartesian_grid(33, 17)
    P = default_params()
    e = engine_for(g, P)
    e.seed(10.0, 10.0)
    S = np.random.default_rng(1).standard_normal((3, 17, 33))
    e.set_state(S)
    assert np.array_equal(e.state(), S)
    p = e.particles()
    assert p["z"].shape == (5, 17, 33) and p["flags"].dtype == np.uint8


def test_gpu_call_order_errors(gpu_lib):
    import ctypes as C
    from picles_b200 import PiclesError
    from picles_b200.engine import B200Engine
    g = cartesian_grid(8, 8)
    e = engine_for(g, default_params())
    with pytest.raises(PiclesError, match="ERR_STATE"):
        e.step(0.0, 600.0)
    with pytest.raises(PiclesError):
        B200Engine(8, 8, 0, 0, g["mask"], default_params(), M_const=g["M_const"], device=99)


def test_gpu_fast_division_and_sqrt_equal_ieee(gpu_lib):
    """pm_div_fast / pm_sqrt_fast (the branch-free fast paths used inside the advance kernel)
    must equal the IEEE operators bit-for-bit whenever their validity flag is clear:
    ~3.7e9 random operand pairs over raw bit patterns, physics-range magnitudes and
    special values."""
    g = cartesian_grid(8, 8)
    e = engine_for(g, default_params())
    tot = None
    for seed in (1, 2, 3):
        r = e.selftest_math(seed=seed, iters=4096)
        tot = r if tot is None else {k: tot[k] + r[k] for k in r}
    assert tot["n_div"] > 3e9 and tot["n_sqrt"] > 3e9
    assert tot["mismatch_div"] == 0 and tot["mismatch_sqrt"] == 0, tot
    # the physics-range class must never be flagged: at most the raw/special classes are
    assert tot["flagged_div"] < 0.7 * tot["n_div"], tot
