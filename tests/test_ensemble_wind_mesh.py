"""Ensembles with one wind mesh per member, on the CPU: the host build of the member sampler of wind_mesh.h equals the
oracle's interpolation run on each member's mesh alone, bit for bit; the new C ABI call is declared, exported and
mirrored; the model and engine check their arguments."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import oracle
from common import bits_equal

from picles_b200 import _abi

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SRC = os.path.join(HERE, "wind_members_shim.cpp")
SO = os.path.join(HERE, "_build", "libwind_members_shim.so")
CHUNK = 8  # WM_MEMBER_CHUNK of picles_kernels.cu


def shim():
    deps = [SRC] + [os.path.join(ROOT, "picles_b200", "csrc", h) for h in ("wind_mesh.h", "pmath.h")]
    if not (os.path.exists(SO) and all(os.path.getmtime(SO) >= os.path.getmtime(d) for d in deps)):
        os.makedirs(os.path.dirname(SO), exist_ok=True)
        gxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        tmp = SO + ".%d" % os.getpid()
        r = subprocess.run([gxx, "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-mfma", "-shared",
                            "-o", tmp, SRC], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        os.replace(tmp, SO)
    lib = C.CDLL(SO)
    vp, i32 = C.c_void_p, C.c_int
    lib.shim_wind_mesh_sample_members.argtypes = [i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, C.c_int64, vp, vp,
                                                  C.c_double, vp, vp]
    return lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def sample_members(xw, yw, tw, U, V, x, y, t, chunk=CHUNK):
    """U, V: (E, nt, ny, nx); returns (E, n) planes"""
    E = U.shape[0]
    U, V = np.ascontiguousarray(U, np.float64), np.ascontiguousarray(V, np.float64)
    x, y = np.ascontiguousarray(x, np.float64), np.ascontiguousarray(y, np.float64)
    u, v = np.full((E, x.size), np.nan), np.full((E, x.size), np.nan)
    shim().shim_wind_mesh_sample_members(xw.size, yw.size, tw.size, E, chunk, _p(xw), _p(yw), _p(tw), _p(U), _p(V),
                                         x.size, _p(x), _p(y), float(t), _p(u), _p(v))
    return u, v


def member_mesh(E, seed=5):
    """strongly non-uniform x knots (the lookup's walk gives up and bisects), uniform y, uneven t; E random fields"""
    rng = np.random.default_rng(seed)
    xw = np.concatenate([[-3000.0], -3000.0 + 40.0 * np.cumsum(2.0 ** np.arange(12))])
    yw = np.linspace(-1000.0, 30000.0, 9)
    tw = np.array([0.0, 21600.0, 30000.0, 64800.0, 86400.0])
    U = rng.normal(8.0, 4.0, (E, tw.size, yw.size, xw.size))
    V = rng.normal(-3.0, 5.0, (E, tw.size, yw.size, xw.size))
    return xw, yw, tw, U, V


def query_points(xw, yw, seed=0):
    """n = 4 * k + 3 nodes: random points inside and up to three periods outside, every knot, rows of a regular grid"""
    rng = np.random.default_rng(seed)
    Lx, Ly = xw[-1] - xw[0], yw[-1] - yw[0]
    gx, gy = np.meshgrid(np.linspace(xw[0] - 5000.0, xw[-1] + 9000.0, 37), np.linspace(yw[0] - 700.0, yw[-1] + 700.0, 11))
    x = np.concatenate([rng.uniform(xw[0] - 3 * Lx, xw[-1] + 3 * Lx, 2000), xw, [xw[0], xw[-1]], gx.ravel(),
                        rng.uniform(xw[0], xw[0] + 200.0, 50)])
    y = np.concatenate([rng.uniform(yw[0] - 2 * Ly, yw[-1] + 2 * Ly, 2000), np.resize(yw, xw.size), [yw[-1], yw[0]],
                        gy.ravel(), rng.uniform(yw[0], yw[-1], 50)])
    k = x.size - (x.size - 3) % 4
    return x[:k], y[:k]


TIMES = (0.0, 100.0, 21600.0, 50000.5, 86400.0, 90000.0, -500.0, -86400.0 * 2 - 17.0, 3 * 86400.0 + 17.0)


@pytest.mark.parametrize("E", [1, 2, 3, 17])
def test_member_sampler_equals_the_oracle_on_each_members_mesh(E):
    xw, yw, tw, U, V = member_mesh(E)
    x, y = query_points(xw, yw)
    assert x.size % 4 == 3
    for t in TIMES:
        u, v = sample_members(xw, yw, tw, U, V, x, y, t)
        for m in range(E):
            uo, vo = oracle.wind_mesh_sample(xw, yw, tw, U[m], V[m], x, y, t)
            assert bits_equal(uo, u[m]) and bits_equal(vo, v[m]), (E, m, t)


def test_member_sampler_does_not_depend_on_the_member_chunk():
    xw, yw, tw, U, V = member_mesh(17, seed=9)
    x, y = query_points(xw, yw, seed=4)
    for t in (1234.5, -77.0):
        ref = sample_members(xw, yw, tw, U, V, x, y, t, chunk=17)
        for chunk in (1, 3, 8):
            got = sample_members(xw, yw, tw, U, V, x, y, t, chunk=chunk)
            assert bits_equal(ref[0], got[0]) and bits_equal(ref[1], got[1])


def test_the_query_points_reach_the_bisection():
    """the x knots double in spacing, so the equal-spacing guess of wm_locate is four or more knots off for many of
    the query points inside the mesh: its walk gives up and it bisects"""
    xw, yw = member_mesh(1)[:2]
    x = query_points(xw, yw)[0]
    x = x[(x >= xw[0]) & (x <= xw[-1])]
    inv_h = (xw.size - 1) / (xw[-1] - xw[0])
    guess = np.minimum(((x - xw[0]) * inv_h).astype(int), xw.size - 1)
    below = np.searchsorted(xw, x, side="left") - 1
    assert np.count_nonzero(np.abs(guess - below) >= 4) > 100


def test_new_symbol_is_declared_exported_and_mirrored():
    hdr = open(os.path.join(ROOT, "include", "picles_b200.h")).read()
    assert int(re.search(r"#define PICLES_ABI_VERSION (\d+)", hdr).group(1)) == _abi.ABI_VERSION == 3
    name = "picles_set_member_wind_meshes"
    assert re.search(r"\bint %s\(" % name, hdr) and name in _abi.SYMBOLS
    lib = _abi.load_library()
    assert hasattr(lib, name) and lib.picles_abi_version() == 3
    res, args = _abi.SYMBOLS[name]
    assert res is C.c_int and args == _abi.SYMBOLS["picles_set_wind_mesh"][1]
    # no handle: refused before any device work
    assert lib.picles_set_member_wind_meshes(None, 2, 2, 2, None, None, None, None, None, None, None) == -5


def _gridded(E, seed=1, shift_t=False):
    from picles_b200.Utils.WindEmulator import GriddedWinds
    xw, yw, tw, U, V = member_mesh(E, seed)
    out = []
    for m in range(E):
        t = tw + (1.0 if shift_t and m == 2 else 0.0)
        out.append(GriddedWinds(xw, yw, t, U[m].transpose(2, 1, 0), V[m].transpose(2, 1, 0)))
    return out


def test_ensemble_model_takes_gridded_winds_on_shared_knots():
    from picles_b200.Models import WaveGrowth2DEnsemble
    from picles_b200.Models.WaveGrowthModels2DEnsemble import MemberGriddedWinds
    from test_ensemble import WINDS, ensemble_kwargs
    kw = ensemble_kwargs()
    gw = _gridded(3)
    m = WaveGrowth2DEnsemble(winds=gw, **kw)
    assert m.members == 3 and isinstance(m._gridded_winds, MemberGriddedWinds)
    # closures only: no device meshes
    assert WaveGrowth2DEnsemble(winds=WINDS, **kw)._gridded_winds is None
    # a list that mixes closures and GriddedWinds, either way round
    with pytest.raises(ValueError, match="member 1 has GriddedWinds"):
        WaveGrowth2DEnsemble(winds=[WINDS[0], gw[0]], **kw)
    with pytest.raises(ValueError, match="member 0 has GriddedWinds and member 2 has not"):
        WaveGrowth2DEnsemble(winds=[gw[0], gw[1], WINDS[1]], **kw)
    # knots that differ in one member: the first such member is named
    with pytest.raises(ValueError, match="member 2 has GriddedWinds on other knots"):
        WaveGrowth2DEnsemble(winds=_gridded(4, shift_t=True), **kw)
    other = _gridded(2)
    other[1].x = other[1].x.copy()
    other[1].x[3] = np.nextafter(other[1].x[3], np.inf)
    with pytest.raises(ValueError, match="member 1 has GriddedWinds on other knots"):
        WaveGrowth2DEnsemble(winds=other, **kw)


class _FakeEngine:
    """records the mesh call and returns E planes from sample_wind_mesh, as an ensemble engine does"""

    def __init__(self, E, ny, Nx):
        self.E, self.ny, self.Nx = E, ny, Nx

    def set_member_wind_meshes(self, *args):
        self.args = args

    def sample_wind_mesh(self, t):
        m = np.arange(self.E, dtype=np.float64)[:, None, None]
        base = np.arange(self.ny * self.Nx, dtype=np.float64).reshape(self.ny, self.Nx)
        return m * 1000.0 + base + t, -(m * 1000.0 + base + t)


def test_member_meshes_bind_in_one_call_and_each_member_reads_its_planes():
    from picles_b200.Models.WaveGrowthModels2DEnsemble import MemberGriddedWinds
    gw = _gridded(3)
    eng = _FakeEngine(3, 4, 5)
    nx_, ny_ = np.zeros((4, 5)), np.ones((4, 5))
    MemberGriddedWinds(gw).bind(eng, nx_, ny_)
    xw, yw, tw, U, V, a, b = eng.args
    assert U.shape == V.shape == (3, tw.size, yw.size, xw.size)
    for m in range(3):
        assert np.array_equal(U[m], gw[m].U) and np.array_equal(V[m], gw[m].V)
        u = gw[m].u(None, None, 7.0)
        assert u.shape == (5, 4) and np.array_equal(u, eng.sample_wind_mesh(7.0)[0][m].T)
        assert np.array_equal(gw[m].v(None, None, 7.0), eng.sample_wind_mesh(7.0)[1][m].T)


def test_set_member_wind_meshes_checks_the_shapes():
    from picles_b200.engine import B200Engine
    eng = B200Engine.__new__(B200Engine)  # no device: the shape check runs before the library is called
    eng.members, eng.ny, eng.Nx, eng.h = 3, 4, 5, None
    xw, yw, tw, U, V = member_mesh(3)
    with pytest.raises(ValueError, match="shape"):
        eng.set_member_wind_meshes(xw, yw, tw, U[0], V[0], 0.0, 0.0)
    with pytest.raises(ValueError, match="shape"):
        eng.set_member_wind_meshes(xw, yw, tw, U[:2], V[:2], 0.0, 0.0)
    with pytest.raises(ValueError, match="shape"):
        eng.set_member_wind_meshes(xw, yw, tw, U, V[:, :, :, :-1], 0.0, 0.0)
    with pytest.raises(ValueError, match="shape"):
        eng.set_member_wind_meshes(xw[:-1], yw, tw, U, V, 0.0, 0.0)
