"""Shared builders for the tests: synthetic configurations (SURVEY.md §8d), the oracle,
the CPU host build of the device physics (tests/host_shim.cpp) and comparison helpers."""
from __future__ import annotations

import ctypes as C
import math
import os

import numpy as np

import host_build
import oracle
from picles_b200 import FetchRelations as FR
from picles_b200._abi import (BND_NONPERIODIC, BND_PERIODIC, BND_TRIPOLAR_NORTH, PiclesCounters,  # noqa: F401
                              PiclesParams)
from picles_b200.ParticleSystems import particle_waves_v5 as PW
from picles_b200.params import make_params

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def default_params(DT=600.0, solver="Tsit5", dt=1e-3, dtmin=1e-4, force_dtmin=True, periodic_boundary=False,
                   on_persist=False, wind_min_squared=4.0, log_energy_maximum=math.log(17), defaults=None, nan_eest_rejects=False,
                   timestep=None, minimal_state=None, C_phi=None, **switches):
    """example_00_minimal.jl:17-67 settings unless overridden."""
    pars, cid, _ = PW.ODEParameters(r_g=0.85)
    if C_phi is not None:
        pars["C_φ"] = C_phi
    ps = PW.particle_equations(None, None, γ=cid.γ, q=cid.q, **switches)
    ts = DT if timestep is None else timestep
    sets = PW.ODESettings(Parameters=pars, log_energy_minimum=FR.MinimalWindsea(10, 10, DT)["lne"], saving_step=DT,
                          timestep=ts, total_time=6 * 86400.0, dt=dt, dtmin=dtmin, force_dtmin=force_dtmin,
                          solver=solver, wind_min_squared=wind_min_squared, log_energy_maximum=log_energy_maximum)
    ms = FR.MinimalState(2, 2, ts) if minimal_state is None else minimal_state
    return make_params(sets, ps, ms, defaults=defaults, periodic_boundary=periodic_boundary, on_persist=on_persist,
                       nan_eest_rejects=nan_eest_rejects)


def cartesian_grid(Nx, Ny, dx=2000.0, dy=2000.0, bx=BND_NONPERIODIC, by=BND_NONPERIODIC, ocean=None):
    """TwoDCartesianGridMesh: x[i]=i*dx, y[j]=j*dy, total mask, uniform kernel diag(1/dx,1/dy)."""
    ocean = np.ones((Ny, Nx), np.uint8) if ocean is None else np.asarray(ocean, np.uint8)
    mask = oracle.make_boundaries(ocean, bx, by)
    x = np.broadcast_to(np.arange(Nx) * dx, (Ny, Nx)).copy()
    y = np.broadcast_to((np.arange(Ny) * dy)[:, None], (Ny, Nx)).copy()
    return dict(Nx=Nx, Ny=Ny, bx=bx, by=by, mask=mask, x=x, y=y, M_const=np.array([1 / dx, 0.0, 0.0, 1 / dy]), M=None,
                pc=None)


def tripolar_grid(Nx, Ny, ocean=None, lat_min=-70.0, lat_max=89.0, R_earth=6.371e6, seed=0):
    """Synthetic tripolar-like mesh: periodic x, tripolar-north y, per-node rotated kernel
    [cos/dx sin/dy; -sin/dx cos/dy] (TripolarGridMOM6.jl:448-459) and great-circle coefficient
    sign(φ)·min(sign(φ)·tand(φ),60)/R (spherical_grid_corrections.jl:13)."""
    lon = -280.0 + (np.arange(Nx) + 0.5) * 360.0 / Nx
    lat = lat_min + (np.arange(Ny) + 0.5) * (lat_max - lat_min) / Ny
    LON, LAT = np.meshgrid(lon, lat)
    cap = np.clip((LAT - 60.0) / 30.0, 0.0, 1.0)
    angle = 40.0 * cap * np.sin(np.deg2rad(2 * (LON + 280.0)))
    dlon, dlat = 360.0 / Nx, (lat_max - lat_min) / Ny
    dx = np.maximum(R_earth * np.cos(np.deg2rad(LAT)) * np.deg2rad(dlon), 2000.0)
    dy = np.full_like(dx, R_earth * np.deg2rad(dlat))
    ca, sa = np.cos(angle * np.pi / 180), np.sin(angle * np.pi / 180)
    M = np.stack([ca / dx, sa / dy, -sa / dx, ca / dy])
    sgn = np.sign(LAT)
    pc = (sgn * np.minimum(sgn * np.tan(np.deg2rad(LAT)), 60.0)) / 6.3710e6
    ocean = np.ones((Ny, Nx), np.uint8) if ocean is None else np.asarray(ocean, np.uint8)
    mask = oracle.make_boundaries(ocean, BND_PERIODIC, BND_TRIPOLAR_NORTH)
    return dict(Nx=Nx, Ny=Ny, bx=BND_PERIODIC, by=BND_TRIPOLAR_NORTH, mask=mask, x=LON, y=LAT, M=M, M_const=None, pc=pc)


def make_oracle(grid, P, variant="default", threads=1):
    return oracle.Oracle(grid["Nx"], grid["Ny"], grid["bx"], grid["by"], grid["mask"], P, M=grid["M"],
                         M_const=grid["M_const"], pc=grid["pc"], variant=variant, threads=threads)


# ---- host build of the device physics ------------------------------------------------

_shim = None


def shim_lib():
    global _shim
    if _shim is None:
        lib = host_build.load("host_shim", src=os.path.join(HERE, "host_shim.cpp"))
        vp, d, i32, i64 = C.c_void_p, C.c_double, C.c_int, C.c_int64
        lib.shim_create.restype = vp
        lib.shim_create.argtypes = [i32, i32, i32, i32, i32, i32, vp, vp, vp, vp, C.POINTER(PiclesParams)]
        lib.shim_destroy.argtypes = [vp]
        lib.shim_set_accumulate.argtypes = [vp, i32]
        lib.shim_set_specialised.argtypes = [i32]
        lib.shim_get_specialised.restype = i32
        lib.shim_advance_template.restype = i32
        lib.shim_advance_template.argtypes = [C.POINTER(PiclesParams), i32]
        lib.shim_set_wind_midlevels.argtypes = [vp, i32, vp, vp, i64]
        lib.shim_wind_mesh_sample.argtypes = [i32, i32, i32, vp, vp, vp, vp, vp, i64, vp, vp, d, vp, vp]
        lib.shim_wind_mesh_sample_members.argtypes = [i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, i64, vp, vp, d, vp,
                                                      vp]
        lib.shim_seed.argtypes = [vp, vp, vp]
        lib.shim_step.argtypes = [vp, d, d, vp, vp, vp, vp]
        lib.shim_get_state.argtypes = [vp, vp]
        lib.shim_set_state.argtypes = [vp, vp]
        lib.shim_get_particles.argtypes = [vp] + [vp] * 7
        lib.shim_get_tally.argtypes = [vp, vp]
        lib.shim_get_solver_state.argtypes = [vp, vp]
        lib.shim_get_solver_state_local.argtypes = [vp, vp]
        lib.shim_corner_target.restype = i64
        lib.shim_corner_target.argtypes = [i32, i32, i32, i32, i64, i64]
        lib.shim_rhs.argtypes = [C.POINTER(PiclesParams), vp, d, d, vp, d, vp]
        lib.shim_pack_roundtrip.argtypes = [i32, i32, i32, vp]
        lib.shim_create_strip.restype = vp
        lib.shim_create_strip.argtypes = [i32, i32, i32, i32, i32, i32, i32, vp, vp, vp, vp, C.POINTER(PiclesParams)]
        lib.shim_strip_seed.argtypes = [vp, vp, vp]
        lib.shim_strip_advance.argtypes = [vp, d, vp, vp, vp, vp]
        lib.shim_strip_halo_bytes.restype = i64
        lib.shim_strip_halo_bytes.argtypes = [vp]
        lib.shim_strip_pack.argtypes = [vp, vp, vp]
        lib.shim_strip_unpack.argtypes = [vp, vp, vp]
        lib.shim_strip_project_remesh.argtypes = [vp, d, vp, vp]
        lib.shim_get_state_local.argtypes = [vp, vp]
        lib.shim_get_particles_local.argtypes = [vp] + [vp] * 7
        _shim = lib
    return _shim


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


TALLY_NAMES = ["n_integrated", "n_substeps", "n_rejects", "n_rhs", "n_reseed_advance", "n_fixups", "n_failed",
               "n_deposited", "n_remesh_A", "n_remesh_B", "n_remesh_C", "n_remesh_D", "reach", "max_attempts",
               "n_stiff_switches", "n_stiff_attempts"]


class HostShim:
    """The device code path (physics.h) executed on the CPU, optionally split in y-strips."""

    def __init__(self, grid, P, nstrips=1, halo=0):
        self.lib = shim_lib()
        self.Nx, self.Ny = grid["Nx"], grid["Ny"]
        m = np.ascontiguousarray(grid["mask"], dtype=np.uint8)
        M = np.ascontiguousarray(grid["M"], dtype=np.float64) if grid["M"] is not None else None
        Mc = np.ascontiguousarray(grid["M_const"], dtype=np.float64) if grid["M_const"] is not None else None
        pc = np.ascontiguousarray(grid["pc"], dtype=np.float64) if grid["pc"] is not None else None
        self._keep = (m, M, Mc, pc)
        self.h = self.lib.shim_create(self.Nx, self.Ny, grid["bx"], grid["by"], nstrips, halo, _p(m), _p(M), _p(Mc),
                                      _p(pc), C.byref(P))

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.shim_destroy(self.h)
            self.h = None

    def _full(self, a):
        return np.ascontiguousarray(np.broadcast_to(np.asarray(a, np.float64), (self.Ny, self.Nx)))

    def set_accumulate(self, on):
        self.lib.shim_set_accumulate(self.h, int(bool(on)))

    def seed(self, u0, v0):
        a, b = self._full(u0), self._full(v0)
        self.lib.shim_seed(self.h, _p(a), _p(b))

    def set_wind_midlevels(self, u_mid, v_mid):
        """intermediate wind levels of the next step: sequences of (Ny, Nx) arrays"""
        n = len(u_mid)
        um = np.ascontiguousarray(np.stack([self._full(x) for x in u_mid])) if n else np.zeros((0, self.Ny, self.Nx))
        vm = np.ascontiguousarray(np.stack([self._full(x) for x in v_mid])) if n else np.zeros((0, self.Ny, self.Nx))
        self.lib.shim_set_wind_midlevels(self.h, n, _p(um), _p(vm), self.Ny * self.Nx)

    def step(self, t, DT, u_t, v_t, u_t1, v_t1):
        a = [self._full(x) for x in (u_t, v_t, u_t1, v_t1)]
        self.lib.shim_step(self.h, float(t), float(DT), *[_p(x) for x in a])

    def state(self):
        S = np.empty((3, self.Ny, self.Nx))
        self.lib.shim_get_state(self.h, _p(S))
        return S

    def set_state(self, S):
        S = np.ascontiguousarray(np.asarray(S, np.float64).reshape(3, self.Ny, self.Nx))
        self.lib.shim_set_state(self.h, _p(S))

    def zero_state(self):
        self.set_state(np.zeros((3, self.Ny, self.Nx)))

    def particles(self):
        sh = (self.Ny, self.Nx)
        z = np.empty((5,) + sh)
        t, dt, qold = np.empty(sh), np.empty(sh), np.empty(sh)
        it = np.empty(sh, np.int32)
        fl = np.empty(sh, np.uint8)
        st = np.empty(sh, np.int32)
        self.lib.shim_get_particles(self.h, _p(z), _p(t), _p(dt), _p(qold), _p(it), _p(fl), _p(st))
        return dict(z=z, t=t, dt=dt, qold=qold, iter=it, flags=fl, status=st)

    def counters(self):
        out = np.empty(16, np.int32)
        self.lib.shim_get_tally(self.h, _p(out))
        return dict(zip(TALLY_NAMES, [int(v) for v in out]))

    def solver_state(self):
        a = np.empty((self.Ny, self.Nx), np.int8)
        self.lib.shim_get_solver_state(self.h, _p(a))
        return a


def bits_equal(a, b):
    """bit-for-bit equality of two float64 arrays; a NaN matches a NaN whatever its sign and
    payload (x86 and sm_100a generate different default NaNs)."""
    a = np.ascontiguousarray(a, np.float64)
    b = np.ascontiguousarray(b, np.float64)
    if a.shape != b.shape:
        return False
    same = a.view(np.uint64) == b.view(np.uint64)
    return bool(np.all(same | (np.isnan(a) & np.isnan(b))))


def compare_models(ref, dut, check_aux=True):
    """Assert that `dut` (HostShim or the B200 engine adaptor) reproduces `ref` (Oracle) exactly."""
    Sr, Sd = ref.state(), dut.state()
    assert bits_equal(Sr, Sd), f"State differs: max abs diff {np.nanmax(np.abs(Sr - Sd))}"
    pr, pd = ref.particles(), dut.particles()
    exists = (pr["flags"] & 8) != 0  # PF_ACTIVE: only iterated particles are meaningful
    for k in range(5):
        assert bits_equal(pr["z"][k][exists], pd["z"][k][exists]), f"particle component {k} differs"
    assert bits_equal(pr["t"][exists], pd["t"][exists])
    assert np.array_equal(pr["flags"][exists], pd["flags"][exists])
    assert np.array_equal(pr["status"][exists], pd["status"][exists])
    # dt is only meaningful while no auto_dt_reset! is pending
    live = exists & ((pr["flags"] & 4) == 0)
    assert bits_equal(pr["dt"][live], pd["dt"][live])
    if check_aux and "qold" in pd:
        ar = ref.aux()
        assert bits_equal(ar["qold"][exists], pd["qold"][exists])
        assert np.array_equal(ar["iter"][exists], pd["iter"][exists].astype(np.int64))
    cr, cd = ref.counters(), dut.counters()
    for name in TALLY_NAMES:
        assert cr[name] == cd[name], f"counter {name}: oracle {cr[name]} vs device path {cd[name]}"


class ShimEngine(HostShim):
    """HostShim behind the B200Engine interface (wind levels kept between steps, `None`
    reuses them) so the host API (WaveGrowth2D / Simulation / run) can be exercised on CPU."""

    def __init__(self, grid, P, **kw):
        super().__init__(grid, P, **kw)
        self.ny = self.Ny
        self._t = None
        self._t1 = None

    def seed(self, u0, v0):
        super().seed(u0, v0)
        self._t = (self._full(u0).copy(), self._full(v0).copy())
        self._t1 = self._t

    def step(self, t, DT, u_t=None, v_t=None, u_t1=None, v_t1=None):
        if u_t is not None:
            self._t = (self._full(u_t).copy(), self._full(v_t).copy())
        elif u_t1 is not None:
            self._t = self._t1
        if u_t1 is not None:
            self._t1 = (self._full(u_t1).copy(), self._full(v_t1).copy())
        super().step(t, DT, self._t[0], self._t[1], self._t1[0], self._t1[1])

    def counters(self):
        c = super().counters()
        c["n_active"] = c["n_remesh_A"] + c["n_remesh_B"] + c["n_remesh_C"] + c["n_remesh_D"]
        return c

    # wind ingestion: the device-side sampler (wind_mesh.h) run on the host
    def set_wind_mesh(self, xw, yw, tw, U, V, node_x, node_y):
        f = lambda a: np.ascontiguousarray(np.asarray(a, np.float64))
        self._mesh = (f(xw), f(yw), f(tw), f(U), f(V), self._full(node_x).copy(), self._full(node_y).copy())

    def sample_wind_mesh(self, t):
        xw, yw, tw, U, V, nx, ny = self._mesh
        u, v = np.empty(nx.shape), np.empty(nx.shape)
        self.lib.shim_wind_mesh_sample(xw.size, yw.size, tw.size, _p(xw), _p(yw), _p(tw), _p(U), _p(V), nx.size, _p(nx),
                                       _p(ny), float(t), _p(u), _p(v))
        return u, v

    def seed_wind_mesh(self, t0=0.0):
        self.seed(*self.sample_wind_mesh(t0))

    def step_wind_mesh(self, t, DT, n_mid=0, lo=-1, hi=-1):
        if n_mid:
            lv = [self.sample_wind_mesh(t + DT * float(k) / float(n_mid + 1)) for k in range(1, n_mid + 1)]
            self.set_wind_midlevels([a for a, _ in lv], [b for _, b in lv])
        self.step(t, DT, *self.sample_wind_mesh(t), *self.sample_wind_mesh(t + DT))


class ShimStripEngine:
    """One y-strip of the host build of the device code behind the phase-split interface of
    B200Engine (upload_winds / step_advance / halo_pack / halo_buffers / halo_unpack /
    step_project_remesh), with host numpy halo buffers: what one rank of the world_size-2
    gloo tests drives through picles_b200.distributed.StripStepper."""

    def __init__(self, grid, P, j0, j1, halo):
        self.lib = shim_lib()
        self.Nx, self.Ny, self.j0, self.ny, self.halo = grid["Nx"], grid["Ny"], j0, j1 - j0, halo
        self.device = -1
        m = np.ascontiguousarray(grid["mask"][j0:j1], dtype=np.uint8)
        M = np.ascontiguousarray(grid["M"][:, j0:j1], dtype=np.float64) if grid["M"] is not None else None
        Mc = np.ascontiguousarray(grid["M_const"], dtype=np.float64) if grid["M_const"] is not None else None
        pc = np.ascontiguousarray(grid["pc"][j0:j1], dtype=np.float64) if grid["pc"] is not None else None
        self.h = self.lib.shim_create_strip(self.Nx, self.Ny, grid["bx"], grid["by"], j0, self.ny, halo, _p(m), _p(M),
                                            _p(Mc), _p(pc), C.byref(P))
        nb = int(self.lib.shim_strip_halo_bytes(self.h))
        self._bufs = [np.zeros(nb, np.uint8), np.zeros(nb, np.uint8), np.full(nb, 0xFF, np.uint8),
                      np.full(nb, 0xFF, np.uint8)]  # send_lo, send_hi, recv_lo, recv_hi
        self._w = [None] * 4

    def __del__(self):
        if getattr(self, "h", None):
            self.lib.shim_destroy(self.h)
            self.h = None

    def _loc(self, a):
        return np.ascontiguousarray(np.broadcast_to(np.asarray(a, np.float64), (self.ny, self.Nx)))

    def seed(self, u0, v0):
        a, b = self._loc(u0), self._loc(v0)
        self.lib.shim_strip_seed(self.h, _p(a), _p(b))
        self._w = [a, b, a, b]

    def upload_winds(self, u_t=None, v_t=None, u_t1=None, v_t1=None):
        if u_t is not None:
            self._w[0], self._w[1] = self._loc(u_t), self._loc(v_t)
        elif u_t1 is not None:
            self._w[0], self._w[1] = self._w[2], self._w[3]
        if u_t1 is not None:
            self._w[2], self._w[3] = self._loc(u_t1), self._loc(v_t1)

    def set_wind_midlevels(self, u_mid=(), v_mid=()):
        n = len(u_mid)
        um = np.ascontiguousarray(np.stack([self._loc(x) for x in u_mid])) if n else np.zeros((0, self.ny, self.Nx))
        vm = np.ascontiguousarray(np.stack([self._loc(x) for x in v_mid])) if n else np.zeros((0, self.ny, self.Nx))
        self.lib.shim_set_wind_midlevels(self.h, n, _p(um), _p(vm), self.ny * self.Nx)

    def set_wind_mesh(self, xw, yw, tw, U, V, node_x, node_y):
        f = lambda a: np.ascontiguousarray(np.asarray(a, np.float64))
        self._mesh = (f(xw), f(yw), f(tw), f(U), f(V), self._loc(node_x).copy(), self._loc(node_y).copy())

    def sample_wind_mesh(self, t):
        xw, yw, tw, U, V, nx, ny = self._mesh
        u, v = np.empty(nx.shape), np.empty(nx.shape)
        self.lib.shim_wind_mesh_sample(xw.size, yw.size, tw.size, _p(xw), _p(yw), _p(tw), _p(U), _p(V), nx.size, _p(nx),
                                       _p(ny), float(t), _p(u), _p(v))
        return u, v

    def seed_wind_mesh(self, t0=0.0):
        self.seed(*self.sample_wind_mesh(t0))

    def step_advance(self, t, DT):
        self.lib.shim_strip_advance(self.h, float(DT), *[_p(x) for x in self._w])

    def halo_buffers(self):
        return self._bufs, self._bufs[0].nbytes

    def halo_pack(self):
        self.lib.shim_strip_pack(self.h, _p(self._bufs[0]), _p(self._bufs[1]))

    def halo_unpack(self):
        self.lib.shim_strip_unpack(self.h, _p(self._bufs[2]), _p(self._bufs[3]))

    def step_project_remesh(self, t, DT):
        self.lib.shim_strip_project_remesh(self.h, float(DT), _p(self._w[0]), _p(self._w[1]))

    def synchronize(self):
        pass

    def state(self):
        S = np.empty((3, self.ny, self.Nx))
        self.lib.shim_get_state_local(self.h, _p(S))
        return S

    def particles(self):
        sh = (self.ny, self.Nx)
        z = np.empty((5,) + sh)
        t, dt, qold = np.empty(sh), np.empty(sh), np.empty(sh)
        it = np.empty(sh, np.int32)
        fl = np.empty(sh, np.uint8)
        st = np.empty(sh, np.int32)
        self.lib.shim_get_particles_local(self.h, _p(z), _p(t), _p(dt), _p(qold), _p(it), _p(fl), _p(st))
        return dict(z=z, t=t, dt=dt, qold=qold, iter=it, flags=fl, status=st)

    def counters(self):
        out = np.empty(16, np.int32)
        self.lib.shim_get_tally(self.h, _p(out))
        return dict(zip(TALLY_NAMES, [int(v) for v in out]))


def grid_dict_from_mesh(grid):
    """tests-side view of a picles_b200 grid object as the dict the oracle builders use."""
    met = grid.device_metric()
    T = lambda a: None if a is None else np.ascontiguousarray(np.asarray(a).T)
    M = None if met["M"] is None else np.stack([T(met["M"][k]) for k in range(4)])
    return dict(Nx=grid.stats.Nx.N, Ny=grid.stats.Ny.N, bx=grid.stats.Nx.code, by=grid.stats.Ny.code,
                mask=T(grid.data.mask).astype(np.uint8), x=T(grid.data.x), y=T(grid.data.y), M=M,
                M_const=met["M_const"], pc=T(met["pc"]))
