"""`WaveGrowth2D` — the model container of `src/Models/WaveGrowthModels2D.jl:42-91,194-345`
with the same keyword constructor, backed by one B200 engine (C ABI handle).

What lives where: the host keeps the grid, the wind closures, the settings and the clock;
particle state and the (Nx,Ny,3) State live in HBM and are fetched on access
(`model.State`, `model.ParticleCollection`).  Wind closures u(x,y,t), v(x,y,t) are
evaluated on the host mesh every step and uploaded (north-star)."""
from __future__ import annotations

from types import SimpleNamespace

import numpy as np

from .. import FetchRelations
from ..Architectures import B200, CPU
from ..Grids.mask_utils import make_boundary_lists
from ..Operators.core_2D import ParticleDefaults
from ..params import make_params


class Clock:
    """Oceananigans.TimeSteppers.Clock: time and iteration, advanced by tick!."""

    def __init__(self, time=0.0):
        self.time = float(time)
        self.iteration = 0

    def tick(self, Δt):
        self.time += Δt
        self.iteration += 1

    def __repr__(self):
        return f"Clock(time={self.time}, iteration={self.iteration})"


def _as_winds(winds):
    if isinstance(winds, dict):
        return SimpleNamespace(u=winds["u"], v=winds["v"])
    if isinstance(winds, (tuple, list)) and len(winds) == 2:
        return SimpleNamespace(u=winds[0], v=winds[1])
    return winds


def eval_wind(f, X, Y, t):
    """Evaluate a wind closure on the mesh: vectorised call first, scalar loop as fallback."""
    try:
        out = f(X, Y, t)
        out = np.asarray(out, dtype=np.float64)
        if out.shape == ():
            return np.full(X.shape, float(out))
        if out.shape == X.shape:
            return out
    except Exception:
        pass
    return np.vectorize(lambda a, b: float(f(a, b, t)), otypes=[np.float64])(X, Y)


class WaveGrowth2D:
    members = 1  # models stepped together on this grid (WaveGrowth2DEnsemble)

    def __init__(self, *, grid, winds, ODEsys, ODEvars=None, layers=1, clock=None, ODEsets=None,
                 ODEinit_type="wind_sea", minimal_particle=None, minimal_state=None, currents=None,
                 periodic_boundary=True, boundary_type="same", CBsets=None, movie=False,
                 architecture=B200(), on_persist=False, strip=None, nan_eest_rejects=False):
        if ODEsets is None:
            raise ValueError("ODEsets is required")
        if layers != 1:
            raise NotImplementedError("layers > 1: the reference's stepping path cannot index a 4-D State (SURVEY B-12)")
        if isinstance(architecture, CPU):
            raise NotImplementedError("CPU architecture: use the Julia reference; picles_b200 has no CPU compute path")
        self.architecture = architecture
        self.grid = grid
        self.layers = layers
        self.clock = clock or Clock(0.0)
        self.dims = 2
        self.winds = _as_winds(winds)
        self.currents = currents
        self.ODEvars = ODEvars
        self.ODEsystem = ODEsys
        self.ODEsettings = ODEsets
        # WaveGrowthModels2D.jl:223-231
        if isinstance(ODEinit_type, ParticleDefaults):
            self.ODEdefaults = ODEinit_type
        elif ODEinit_type == "wind_sea":
            self.ODEdefaults = None
        elif ODEinit_type == "mininmal":
            self.ODEdefaults = ParticleDefaults(-11.0, 1e-3, 0.0)
        else:
            raise ValueError("ODEinit_type must be either 'wind_sea','mininmal', or ParticleDefaults instance ")
        # :234-246
        self.minimal_particle = (FetchRelations.MinimalParticle(2, 2, ODEsets.timestep)
                                 if minimal_particle is None else minimal_particle)
        self.minimal_state = (FetchRelations.MinimalState(2, 2, ODEsets.timestep)
                              if minimal_state is None else minimal_state)
        self.periodic_boundary = bool(periodic_boundary)
        # :256-270
        Glists = make_boundary_lists(grid.data.mask)
        if periodic_boundary:
            self.ocean_points = np.concatenate([Glists["ocean"], Glists["grid_boundary"]])
            self.boundary_points = Glists["land_boundary"]
        else:
            self.ocean_points = Glists["ocean"]
            self.boundary_points = np.concatenate([Glists["land_boundary"], Glists["grid_boundary"]])
        if boundary_type not in ("wind_sea", "mininmal", "same"):
            raise ValueError("boundary_type must be either 'wind_sea','mininmal', or 'same' ")
        self.boundary_type = boundary_type
        self.movie = movie
        self.MovieState = None
        self.FailedCollection = []
        self.on_persist = bool(on_persist)
        self.params = make_params(ODEsets, ODEsys, self.minimal_state,
                                  defaults=None if self.ODEdefaults is None else self.ODEdefaults.as_list(),
                                  periodic_boundary=self.periodic_boundary, on_persist=self.on_persist,
                                  nan_eest_rejects=nan_eest_rejects or getattr(architecture, "nan_eest_rejects", False))
        self.Nx, self.Ny = grid.stats.Nx.N, grid.stats.Ny.N
        self._strip = strip  # (j0, ny_local, halo) when this model is one y-strip of a larger grid
        self._engine = None
        self._wind_level_time = None
        self._seeded = False
        from ..Utils.WindEmulator import GriddedWinds
        self._gridded_winds = self.winds if isinstance(self.winds, GriddedWinds) else None

    # ---- device plumbing ---------------------------------------------------------
    @property
    def engine(self):
        if self._engine is None:
            from ..engine import B200Engine
            g = self.grid
            met = g.device_metric()
            j0, ny, halo = self._strip if self._strip else (0, self.Ny, 0)
            rows = slice(j0, j0 + ny)
            plane = lambda a: np.ascontiguousarray(np.asarray(a)[:, rows].T)  # (Nx,Ny) F-view -> (ny,Nx) C
            raw = met.get("raw")
            if raw is not None:   # per-node metric: formed on the device from the raw mesh planes
                metric = {k: plane(raw[k]) for k in ("dx", "dy", "angle_dx", "lat")}
                metric["R_earth"] = raw["R_earth"]
                M = pc = None
            else:
                metric = None
                M = None if met["M"] is None else np.stack([plane(met["M"][k]) for k in range(4)])
                pc = None if met["pc"] is None else plane(met["pc"])
            self._engine = B200Engine(self.Nx, self.Ny, g.stats.Nx.code, g.stats.Ny.code,
                                      plane(g.data.mask).astype(np.uint8), self.params, M=M, M_const=met["M_const"],
                                      pc=pc, device=self.architecture.devices[0], j0=j0, ny_local=ny, halo=halo,
                                      metric=metric, members=self.members)
            self._rows = rows
            if self._gridded_winds is not None:  # upload the wind mesh once; sampled on the device
                self._gridded_winds.bind(self._engine, plane(g.data.x), plane(g.data.y))
        return self._engine

    def _wind_planes(self, t):
        """(u, v) at time t on this model's rows, as (ny, Nx) C-ordered planes."""
        eng = self.engine
        if self._gridded_winds is not None:
            return eng.sample_wind_mesh(t)
        X = self.grid.data.x[:, self._rows]
        Y = self.grid.data.y[:, self._rows]
        u = eval_wind(self.winds.u, X, Y, t)
        v = eval_wind(self.winds.v, X, Y, t)
        return np.ascontiguousarray(u.T), np.ascontiguousarray(v.T)

    # ---- fields (fetched from HBM on access) -----------------------------------------
    @property
    def State(self):
        """(Nx_local rows of) the (Nx, Ny, 3) node state [e, m_x, m_y], indexed [i, j, k]."""
        return self.engine.state().transpose(2, 1, 0)

    @State.setter
    def State(self, S):
        self.engine.set_state(np.asarray(S, dtype=np.float64).transpose(2, 1, 0))

    @property
    def ParticleCollection(self):
        """StructArray-like view of the particles: fields indexed [i, j]."""
        p = self.engine.particles()
        T = lambda a: a.T
        return SimpleNamespace(u=p["z"].transpose(0, 2, 1), lne=T(p["z"][0]), c̄_x=T(p["z"][1]), c̄_y=T(p["z"][2]),
                               x=T(p["z"][3]), y=T(p["z"][4]), t=T(p["t"]), dt=T(p["dt"]),
                               on=T((p["flags"] & 1) != 0), boundary=T((p["flags"] & 2) != 0),
                               active=T((p["flags"] & 8) != 0), status=T(p["status"]))

    def counters(self):
        return self.engine.counters()


def fields(model):
    """WaveGrowthModels2D.jl `fields(model)`: the prognostic State."""
    return dict(State=model.State)
