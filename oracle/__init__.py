"""ctypes wrapper of the CPU oracle (oracle/picles_oracle.c).

TEST INFRASTRUCTURE ONLY — imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs; never by the product package.  PARITY UNPINNED
(see the header of picles_oracle.c).
"""
from __future__ import annotations

import ctypes as C
import fcntl
import os
import subprocess

import numpy as np

from picles_b200._abi import PiclesCounters, PiclesParams

HERE = os.path.dirname(os.path.abspath(__file__))
BUILD = os.path.join(HERE, "_build")
_VARIANTS = {
    "default": "libpicles_oracle.so",
    "omp": "libpicles_oracle_omp.so",
    "libm": "libpicles_oracle_libm.so",
    "fastpow": "libpicles_oracle_fastpow.so",      # controller powers in Float32 (sensitivity study)
    "fastpow12": "libpicles_oracle_fastpow12.so",  # ... cut to 12 mantissa bits
}
_libs: dict = {}


def make(*targets: str) -> None:
    """Run the committed Makefile (every variant when no target is named) under a lock on the build directory, so that
    processes starting at the same time build each library once and none loads one being written."""
    os.makedirs(BUILD, exist_ok=True)
    fd = os.open(os.path.join(BUILD, ".lock"), os.O_RDONLY | os.O_CREAT, 0o644)
    try:
        fcntl.flock(fd, fcntl.LOCK_EX)
        r = subprocess.run(["make", "-s", "-C", HERE, *targets], capture_output=True, text=True)
    finally:
        os.close(fd)
    if r.returncode != 0:
        raise RuntimeError("oracle build failed:\n" + r.stdout + r.stderr)


def build(force: bool = False) -> None:
    """Compile the oracle variants with the committed Makefile; `force` rebuilds every one."""
    make("-B" if force else "all")


def _dp(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def load(variant: str = "default"):
    if variant in _libs:
        return _libs[variant]
    make("_build/" + _VARIANTS[variant])
    lib = C.CDLL(os.path.join(BUILD, _VARIANTS[variant]))
    vp, d, i64, i32 = C.c_void_p, C.c_double, C.c_int64, C.c_int
    lib.oracle_create.restype = vp
    lib.oracle_create.argtypes = [i32, i32, i32, i32, vp, vp, vp, vp, C.POINTER(PiclesParams)]
    lib.oracle_destroy.argtypes = [vp]
    lib.oracle_set_threads.argtypes = [vp, i32]
    lib.oracle_set_accumulate.argtypes = [vp, i32]
    lib.oracle_set_wind_midlevels.argtypes = [vp, i32, vp, vp]
    lib.oracle_set_wind_closure.argtypes = [vp, vp, vp, vp]
    lib.oracle_wind_mesh_sample.argtypes = [i32, i32, i32, vp, vp, vp, vp, vp, i64, vp, vp, d, vp, vp]
    lib.oracle_seed.argtypes = [vp, vp, vp]
    lib.oracle_step.argtypes = [vp, d, d, vp, vp, vp, vp]
    lib.oracle_get_state.argtypes = [vp, vp]
    lib.oracle_set_state.argtypes = [vp, vp]
    lib.oracle_get_particles.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.oracle_get_aux.argtypes = [vp, vp, vp]
    lib.oracle_get_counters.argtypes = [vp, C.POINTER(PiclesCounters)]
    lib.oracle_get_solver_state.argtypes = [vp, vp]
    lib.oracle_n_ocean.restype = i64
    lib.oracle_n_ocean.argtypes = [vp]
    lib.oracle_fields.argtypes = [vp, vp, vp, vp]
    lib.oracle_stiff_triggers.restype = i64
    lib.oracle_stiff_triggers.argtypes = [vp]
    lib.oracle_get_ocean_points.argtypes = [vp, vp]
    lib.oracle_make_boundaries.argtypes = [vp, i32, i32, i32, i32, vp]
    lib.oracle_rhs.argtypes = [C.POINTER(PiclesParams), vp, d, d, vp, d, vp]
    lib.oracle_windsea.argtypes = [d, d, d, vp, vp, vp]
    lib.oracle_minimal_state.argtypes = [d, d, d, vp, vp]
    lib.oracle_particle_to_charge.argtypes = [vp, vp]
    lib.oracle_vertex_to_particle.argtypes = [vp, vp]
    lib.oracle_weights.argtypes = [d, i64, vp, vp]
    lib.oracle_wrap_index.restype = i64
    lib.oracle_wrap_index.argtypes = [i64, i64]
    lib.oracle_corner_target.restype = i64
    lib.oracle_corner_target.argtypes = [i32, i32, i32, i32, i64, i64]
    lib.oracle_integrate_one.argtypes = [C.POINTER(PiclesParams), vp, d, vp, vp, vp, vp, vp, i32, d, d, d, d, d,
                                         C.POINTER(PiclesCounters), vp]
    lib.oracle_integrate_one_as.argtypes = [C.POINTER(PiclesParams), vp, d, vp, vp, vp, vp, vp, i32, d, d, d, d, d,
                                            C.POINTER(PiclesCounters), vp, vp]
    lib.oracle_rhs_jacobian.argtypes = [C.POINTER(PiclesParams), vp, d, d, d, d, vp, d, vp, vp]
    lib.oracle_grid_metric.argtypes = [i64, vp, vp, vp, vp, d, vp, vp]
    for f in ("exp", "log", "tanh", "sech", "cosh", "eps", "sin", "cos", "sind", "cosd", "tand"):
        getattr(lib, "oracle_pm_" + f).argtypes = [i64, vp, vp]
    lib.oracle_pm_pow.argtypes = [i64, vp, vp, vp]
    lib.oracle_uses_libm.restype = i32
    lib.oracle_max_threads.restype = i32
    _libs[variant] = lib
    return lib


def _f64(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64))


class Oracle:
    """One CPU model instance: oracle_create / seed / step / accessors.

    Arrays are (Ny, Nx) C-ordered numpy arrays == column-major (Nx, Ny) Julia arrays
    (i fastest), State is (3, Ny, Nx).
    """

    def __init__(self, Nx, Ny, bx, by, mask, params: PiclesParams, M=None, M_const=None, pc=None,
                 variant: str = "default", threads: int = 1):
        self.lib = load(variant)
        self.Nx, self.Ny = int(Nx), int(Ny)
        mask = np.ascontiguousarray(np.asarray(mask, dtype=np.uint8).reshape(Ny, Nx))
        self._keep = [mask]
        Mp = _f64(M).reshape(4, Ny, Nx) if M is not None else None
        Mc = _f64(M_const).reshape(4) if M_const is not None else None
        pcp = _f64(pc).reshape(Ny, Nx) if pc is not None else None
        if Mp is None and Mc is None:
            raise ValueError("need M or M_const")
        self.params = params
        self.h = self.lib.oracle_create(self.Nx, self.Ny, int(bx), int(by), _dp(mask), _dp(Mp), _dp(Mc), _dp(pcp),
                                        C.byref(params))
        if threads > 1:
            self.lib.oracle_set_threads(self.h, int(threads))

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.oracle_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def set_accumulate(self, on):
        self.lib.oracle_set_accumulate(self.h, int(bool(on)))

    def seed(self, u0, v0):
        u0 = _f64(np.broadcast_to(u0, (self.Ny, self.Nx)))
        v0 = _f64(np.broadcast_to(v0, (self.Ny, self.Nx)))
        self.lib.oracle_seed(self.h, _dp(u0), _dp(v0))

    def set_wind_midlevels(self, u_mid, v_mid):
        """intermediate wind levels (t + k*DT/(n+1), k = 1..n) of the next step only"""
        sh = (self.Ny, self.Nx)
        n = len(u_mid)
        um = _f64(np.stack([np.broadcast_to(x, sh) for x in u_mid])) if n else None
        vm = _f64(np.stack([np.broadcast_to(x, sh) for x in v_mid])) if n else None
        self.lib.oracle_set_wind_midlevels(self.h, n, _dp(um), _dp(vm))

    def set_wind_closure(self, fn, x, y):
        """reference semantics: fn(x, y, t) -> (u, v) is called at the home node and the stage
        time of every right-hand side (small grids only: a Python callback per evaluation)"""
        if fn is None:
            self._cb = None
            self.lib.oracle_set_wind_closure(self.h, None, None, None)
            return
        CB = C.CFUNCTYPE(None, C.c_double, C.c_double, C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_double))

        def tramp(xx, yy, tt, pu, pv):
            u, v = fn(xx, yy, tt)
            pu[0] = u
            pv[0] = v

        self._cb = CB(tramp)
        sh = (self.Ny, self.Nx)
        xa, ya = _f64(np.broadcast_to(x, sh)), _f64(np.broadcast_to(y, sh))
        self.lib.oracle_set_wind_closure(self.h, C.cast(self._cb, C.c_void_p), _dp(xa), _dp(ya))

    def step(self, t, DT, u_t, v_t, u_t1, v_t1):
        sh = (self.Ny, self.Nx)
        a = [_f64(np.broadcast_to(x, sh)) for x in (u_t, v_t, u_t1, v_t1)]
        self.lib.oracle_step(self.h, float(t), float(DT), *[_dp(x) for x in a])

    def state(self):
        S = np.empty((3, self.Ny, self.Nx))
        self.lib.oracle_get_state(self.h, _dp(S))
        return S

    def set_state(self, S):
        S = _f64(S).reshape(3, self.Ny, self.Nx)
        self.lib.oracle_set_state(self.h, _dp(S))

    def particles(self):
        sh = (self.Ny, self.Nx)
        z = np.empty((5,) + sh)
        t = np.empty(sh)
        dt = np.empty(sh)
        flags = np.empty(sh, dtype=np.uint8)
        status = np.empty(sh, dtype=np.int32)
        self.lib.oracle_get_particles(self.h, _dp(z), _dp(t), _dp(dt), _dp(flags), _dp(status))
        return dict(z=z, t=t, dt=dt, flags=flags, status=status)

    def aux(self):
        sh = (self.Ny, self.Nx)
        qold = np.empty(sh)
        it = np.empty(sh, dtype=np.int64)
        self.lib.oracle_get_aux(self.h, _dp(qold), _dp(it))
        return dict(qold=qold, iter=it)

    def counters(self):
        c = PiclesCounters()
        self.lib.oracle_get_counters(self.h, C.byref(c))
        return c.as_dict()

    def ocean_points(self):
        n = self.lib.oracle_n_ocean(self.h)
        idx = np.empty(n, dtype=np.int64)
        self.lib.oracle_get_ocean_points(self.h, _dp(idx))
        return idx

    def fields(self):
        sh = (self.Ny, self.Nx)
        Hs, cx, cy = np.empty(sh), np.empty(sh), np.empty(sh)
        self.lib.oracle_fields(self.h, _dp(Hs), _dp(cx), _dp(cy))
        return dict(Hs=Hs, c_x=cx, c_y=cy)

    def solver_state(self):
        """AutoSwitch state per particle: run length of the stiffness test, +64 while Rosenbrock23 is current"""
        a = np.empty((self.Ny, self.Nx), dtype=np.int8)
        self.lib.oracle_get_solver_state(self.h, _dp(a))
        return a

    def stiff_triggers(self):
        return int(self.lib.oracle_stiff_triggers(self.h))


# ---- function-level hooks ------------------------------------------------------

def make_boundaries(ocean_mask, bx, by, variant="default"):
    lib = load(variant)
    m = np.ascontiguousarray(np.asarray(ocean_mask, dtype=np.uint8))
    Ny, Nx = m.shape
    out = np.empty_like(m)
    lib.oracle_make_boundaries(_dp(m), Nx, Ny, int(bx), int(by), _dp(out))
    return out


def rhs(params, z, u, v, M=(1.0, 0.0, 0.0, 1.0), pc=0.0, variant="default"):
    lib = load(variant)
    z = _f64(z)
    M = _f64(M)
    dz = np.empty(5)
    lib.oracle_rhs(C.byref(params), _dp(z), float(u), float(v), _dp(M), float(pc), _dp(dz))
    return dz


def windsea(u, v, T, variant="default"):
    lib = load(variant)
    out = np.empty(5)
    E = np.empty(1)
    cg = np.empty(1)
    lib.oracle_windsea(float(u), float(v), float(T), _dp(out), _dp(E), _dp(cg))
    return out, float(E[0]), float(cg[0])


def minimal_state(u, v, T, variant="default"):
    lib = load(variant)
    out = np.empty(2)
    part = np.empty(5)
    lib.oracle_minimal_state(float(u), float(v), float(T), _dp(out), _dp(part))
    return out, part


def particle_to_charge(u5, variant="default"):
    lib = load(variant)
    u5 = _f64(u5)
    ch = np.empty(3)
    lib.oracle_particle_to_charge(_dp(u5), _dp(ch))
    return ch


def vertex_to_particle(s3, variant="default"):
    lib = load(variant)
    s3 = _f64(s3)
    u = np.empty(5)
    lib.oracle_vertex_to_particle(_dp(s3), _dp(u))
    return u


def weights(zp, i_node, variant="default"):
    lib = load(variant)
    idx = np.empty(2, dtype=np.int64)
    w = np.empty(2)
    lib.oracle_weights(float(zp), int(i_node), _dp(idx), _dp(w))
    return idx, w


def corner_target(Nx, Ny, bx, by, i, j, variant="default"):
    return int(load(variant).oracle_corner_target(Nx, Ny, bx, by, int(i), int(j)))


def rhs_jacobian(params, z, u, v, ut=0.0, vt=0.0, M=(1.0, 0.0, 0.0, 1.0), pc=0.0, variant="default"):
    """(J, dT): df/dz (5x5) and df/dt of the right-hand side by forward-mode dual numbers"""
    lib = load(variant)
    z, M = _f64(z), _f64(M)
    J, dT = np.empty((5, 5)), np.empty(5)
    lib.oracle_rhs_jacobian(C.byref(params), _dp(z), float(u), float(v), float(ut), float(vt), _dp(M), float(pc), _dp(J),
                            _dp(dT))
    return J, dT


def integrate_one(params, u5, t=0.0, dt=None, qold=1e-4, it=0, dt_reset=False, wind0=(10.0, 10.0), wind1=None,
                  DT=600.0, M=(1 / 2000.0, 0.0, 0.0, 1 / 2000.0), pc=0.0, status=0, variant="default", as_state=None):
    lib = load(variant)
    u5 = _f64(u5).copy()
    M = _f64(M)
    tt = np.array([t], dtype=np.float64)
    dd = np.array([params.dt if dt is None else dt], dtype=np.float64)
    qq = np.array([qold], dtype=np.float64)
    ii = np.array([it], dtype=np.int64)
    st = np.array([status], dtype=np.int32)
    wind1 = wind0 if wind1 is None else wind1
    c = PiclesCounters()
    as2 = np.array(as_state if as_state is not None else (0, 0), dtype=np.int32)
    lib.oracle_integrate_one_as(C.byref(params), _dp(M), float(pc), _dp(u5), _dp(tt), _dp(dd), _dp(qq), _dp(ii),
                                int(dt_reset), float(wind0[0]), float(wind0[1]), float(wind1[0]), float(wind1[1]),
                                float(DT), C.byref(c), _dp(st), _dp(as2))
    return dict(u=u5, t=float(tt[0]), dt=float(dd[0]), qold=float(qq[0]), iter=int(ii[0]), status=int(st[0]),
                counters=c.as_dict(), as_state=(int(as2[0]), int(as2[1])))


def pm(func, x, y=None, variant="default"):
    lib = load(variant)
    x = _f64(x).ravel()
    out = np.empty_like(x)
    if func == "pow":
        y = _f64(np.broadcast_to(y, x.shape)).ravel()
        lib.oracle_pm_pow(x.size, _dp(x), _dp(y), _dp(out))
    else:
        getattr(lib, "oracle_pm_" + func)(x.size, _dp(x), _dp(out))
    return out


def grid_metric(dx, dy, angle_dx, lat, R_earth=6.3710e6, variant="default"):
    """per-node projection kernel planes (4, ...) and great-circle coefficient"""
    lib = load(variant)
    dx, dy, angle_dx, lat = (_f64(np.broadcast_to(a, np.shape(dx))) for a in (dx, dy, angle_dx, lat))
    M = np.empty((4,) + dx.shape)
    pc = np.empty(dx.shape)
    lib.oracle_grid_metric(dx.size, _dp(dx), _dp(dy), _dp(angle_dx), _dp(lat), float(R_earth), _dp(M), _dp(pc))
    return M, pc


def wind_mesh_sample(xw, yw, tw, U, V, x, y, t, variant="default"):
    """Interpolations.LinearInterpolation((xw, yw, tw), U, extrapolation_bc=Periodic()) at the
    points (x, y) and time t; U, V: (nt, ny, nx) C-ordered == Julia U[ix, iy, it]"""
    lib = load(variant)
    xw, yw, tw, U, V = _f64(xw), _f64(yw), _f64(tw), _f64(U), _f64(V)
    x = _f64(x)
    y = _f64(np.broadcast_to(y, x.shape))
    u, v = np.empty(x.shape), np.empty(x.shape)
    lib.oracle_wind_mesh_sample(xw.size, yw.size, tw.size, _dp(xw), _dp(yw), _dp(tw), _dp(U), _dp(V), x.size, _dp(x),
                                _dp(y), float(t), _dp(u), _dp(v))
    return u, v


def max_threads():
    return int(load("omp").oracle_max_threads())
