"""Ensembles on the CPU: the C ABI additions agree between library, header and ctypes mirror; WaveGrowth2DEnsemble
checks its arguments and refuses what it does not support; the layout between the model's (E, Nx, Ny, 3) State and the
engine's flat planes."""
import os
import re

import numpy as np
import pytest

from picles_b200 import FetchRelations, _abi
from picles_b200.Grids.CartesianGrid import TwoDCartesianGridMesh
from picles_b200.Models import WaveGrowth2D, WaveGrowth2DEnsemble
from picles_b200.Models.WaveGrowthModels2DEnsemble import planes_from_state, state_from_planes
from picles_b200.ParticleSystems import particle_waves_v5 as PW

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def ensemble_kwargs(Nx=30, Ny=20):
    """example_00_minimal.jl settings on a small box, without the winds"""
    DT = 600.0
    grid = TwoDCartesianGridMesh(60e3, Nx, 40e3, Ny)
    pars, cid, _ = PW.ODEParameters(r_g=0.85)
    sets = PW.ODESettings(Parameters=pars, log_energy_minimum=FetchRelations.MinimalWindsea(10, 10, DT)["lne"],
                          saving_step=DT, timestep=DT, total_time=6 * 86400.0, dt=1e-3, dtmin=1e-4, force_dtmin=True)
    return dict(grid=grid, ODEsys=PW.particle_equations(None, None, γ=cid.γ, q=cid.q), ODEsets=sets,
                periodic_boundary=False)


WINDS = [(lambda x, y, t: 10.0 + 0 * x, lambda x, y, t: 6.0 + 0 * x),
         dict(u=lambda x, y, t: -7.0 + 1e-4 * x, v=lambda x, y, t: 3.0 + 0 * y + 1e-3 * t),
         (lambda x, y, t: 0.5, lambda x, y, t: 0.4)]


def test_abi_version_and_ensemble_symbols_agree():
    hdr = open(os.path.join(ROOT, "include", "picles_b200.h")).read()
    assert int(re.search(r"#define PICLES_ABI_VERSION (\d+)", hdr).group(1)) == _abi.ABI_VERSION == 3
    lib = _abi.load_library()
    assert lib.picles_abi_version() == 3
    for name in ("picles_set_members", "picles_member_energy_sums"):
        assert re.search(r"\bint %s\(" % name, hdr) and name in _abi.SYMBOLS and hasattr(lib, name)


def test_set_members_needs_a_handle():
    lib = _abi.load_library()
    assert lib.picles_set_members(None, 4) == -1
    assert lib.picles_member_energy_sums(None, None) == -1


def test_ensemble_argument_checks():
    from picles_b200.Utils.WindEmulator import GriddedWinds
    kw = ensemble_kwargs()
    with pytest.raises(ValueError, match="non-empty list"):
        WaveGrowth2DEnsemble(winds=[], **kw)
    with pytest.raises(ValueError, match="non-empty list"):
        WaveGrowth2DEnsemble(winds=WINDS[1], **kw)
    with pytest.raises(ValueError, match="strip"):
        WaveGrowth2DEnsemble(winds=WINDS, strip=(0, 10, 2), **kw)
    gw = GriddedWinds.__new__(GriddedWinds)
    with pytest.raises(ValueError, match="member 1 has GriddedWinds"):
        WaveGrowth2DEnsemble(winds=[WINDS[0], gw], **kw)
    with pytest.raises(ValueError, match="member 0 needs winds"):
        WaveGrowth2DEnsemble(winds=[(1.0, 2.0)], **kw)
    m = WaveGrowth2DEnsemble(winds=WINDS, **kw)
    assert m.members == 3 and WaveGrowth2D.members == 1
    assert m.params.periodic_boundary == WaveGrowth2D(winds=WINDS[0], **kw).params.periodic_boundary


def test_member_wind_planes_have_one_plane_per_member():
    kw = ensemble_kwargs()
    m = WaveGrowth2DEnsemble(winds=WINDS, **kw)
    m._engine, m._rows = object(), slice(0, m.Ny)  # no device: only the host-side staging is exercised
    u, v = m._wind_planes(600.0)
    assert u.shape == v.shape == (3, m.Ny, m.Nx) and u.flags["C_CONTIGUOUS"]
    for k, w in enumerate(WINDS):
        s = WaveGrowth2D(winds=w, **kw)
        s._engine, s._rows = object(), slice(0, s.Ny)
        us, vs = s._wind_planes(600.0)
        assert np.array_equal(u[k], us) and np.array_equal(v[k], vs)


def test_ensemble_without_a_gpu_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: the failure path is exercised on the CPU box")
    from picles_b200.Simulations.run import init_particles
    m = WaveGrowth2DEnsemble(winds=WINDS, **ensemble_kwargs())
    with pytest.raises(_abi.PiclesError, match="ERR_CUDA"):
        init_particles(m)


def test_state_layout_round_trip():
    E, ny, Nx = 3, 5, 7
    planes = np.random.default_rng(0).standard_normal((3, E, ny, Nx))
    State = state_from_planes(planes)
    assert State.shape == (E, Nx, ny, 3)
    for m in range(E):
        # member m is what a single model makes of its own (3, ny, Nx) planes
        assert np.array_equal(State[m], planes[:, m].transpose(2, 1, 0))
    back = planes_from_state(State)
    assert np.array_equal(back, planes)
    # flat C layout: 3 planes of E*ny*Nx values, member slowest
    flat = np.ascontiguousarray(back).reshape(-1)
    assert np.array_equal(flat[: E * ny * Nx].reshape(E, ny, Nx)[1], planes[0, 1])


def test_cash_store_layout_of_an_ensemble_snapshot():
    """run() turns a (3, E, ny, Nx) snapshot buffer into the (E, Nx, Ny, 3) State the model returns"""
    planes = np.arange(3 * 2 * 4 * 5, dtype=np.float64).reshape(3, 2, 4, 5)
    got = np.moveaxis(planes, 0, -1).swapaxes(-2, -3)
    assert np.array_equal(got, state_from_planes(planes))
    single = planes[:, 0]
    assert np.array_equal(np.moveaxis(single, 0, -1).swapaxes(-2, -3), single.transpose(2, 1, 0))
