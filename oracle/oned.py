"""ctypes front of oracle/picles_oracle_1d.c — the CPU checker of the one-dimensional path.  Test infrastructure."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from oracle import BUILD, make
from picles_b200._abi import PiclesCounters, PiclesParams

_lib = None
WIND_FN = C.CFUNCTYPE(C.c_double, C.c_double, C.c_double)


def lib():
    global _lib
    if _lib is None:
        make("_build/libpicles_oracle_1d.so")
        L = C.CDLL(os.path.join(BUILD, "libpicles_oracle_1d.so"))
        vp, d = C.c_void_p, C.c_double
        L.oracle1d_create.restype = vp
        L.oracle1d_create.argtypes = [C.c_int, d, d, vp, C.POINTER(PiclesParams)]
        L.oracle1d_destroy.argtypes = [vp]
        L.oracle1d_set_wind_closure.argtypes = [vp, WIND_FN]
        L.oracle1d_seed.argtypes = [vp, vp]
        L.oracle1d_step.argtypes = [vp, d, d, vp, vp]
        L.oracle1d_get_state.argtypes = [vp, vp]
        L.oracle1d_get_particles.argtypes = [vp, vp, vp, vp, vp, vp]
        L.oracle1d_get_counters.argtypes = [vp, C.POINTER(PiclesCounters)]
        L.oracle1d_rhs.argtypes = [C.POINTER(PiclesParams), vp, d, vp]
        L.oracle1d_windsea.argtypes = [d, d, vp]
        L.oracle1d_merge.argtypes = [vp, vp]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class Oracle1D:
    def __init__(self, Nx, xmin, dx, x_nodes, params):
        self.L = lib()
        self.Nx = int(Nx)
        xn = np.ascontiguousarray(x_nodes, np.float64)
        self.P = params
        self.h = self.L.oracle1d_create(self.Nx, float(xmin), float(dx), _p(xn), C.byref(params))
        if not self.h:
            raise RuntimeError("oracle1d_create failed")
        self._cb = None

    def set_wind_closure(self, f):
        """reference semantics: winds(x, t) called at the particle's position and the stage time"""
        self._cb = WIND_FN(lambda x, t: float(f(x, t)))
        self.L.oracle1d_set_wind_closure(self.h, self._cb)

    def _plane(self, a):
        return np.ascontiguousarray(np.broadcast_to(np.asarray(a, np.float64), (self.Nx,)))

    def seed(self, u0):
        u0 = self._plane(u0)
        self.L.oracle1d_seed(self.h, _p(u0))

    def step(self, t, DT, u_t, u_t1):
        a, b = self._plane(u_t), self._plane(u_t1)
        self.L.oracle1d_step(self.h, float(t), float(DT), _p(a), _p(b))

    def state(self):
        S = np.empty((3, self.Nx), np.float64)
        self.L.oracle1d_get_state(self.h, _p(S))
        return S

    def particles(self):
        z = np.empty((3, self.Nx), np.float64)
        t = np.empty(self.Nx, np.float64)
        dt = np.empty(self.Nx, np.float64)
        flags = np.empty(self.Nx, np.uint8)
        status = np.empty(self.Nx, np.int32)
        self.L.oracle1d_get_particles(self.h, _p(z), _p(t), _p(dt), _p(flags), _p(status))
        return dict(z=z, t=t, dt=dt, flags=flags, status=status)

    def counters(self):
        c = PiclesCounters()
        self.L.oracle1d_get_counters(self.h, C.byref(c))
        return {name: getattr(c, name) for name, _ in c._fields_}

    def close(self):
        if self.h:
            self.L.oracle1d_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def rhs(params, z, u):
    z = np.ascontiguousarray(z, np.float64)
    dz = np.empty(3)
    lib().oracle1d_rhs(C.byref(params), _p(z), float(u), _p(dz))
    return dz


def windsea(u, T):
    out = np.empty(2)
    lib().oracle1d_windsea(float(u), float(T), _p(out))
    return out


def merge(g, c):
    g = np.array(g, np.float64)
    c = np.ascontiguousarray(c, np.float64)
    lib().oracle1d_merge(_p(g), _p(c))
    return g
