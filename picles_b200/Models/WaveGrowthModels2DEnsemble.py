"""`WaveGrowth2DEnsemble` — E `WaveGrowth2D` models on one grid, each with its own winds, stepped
together in one B200 engine (an ensemble handle, picles_set_members).

The reference runs many small configurations one after another (the sweeps over wind sign and
periodicity of T04_2D_reg_test.jl, the (U10, V10) variants of T04_2D_growing_decaying_winds.jl); an
ensemble of wind forcings is also how a wave forecast expresses its uncertainty.  Here the members
share the grid, the mask, the projection kernel and every setting, and each step launches the
kernels one model launches, whatever E is.

Layout: `State` is (E, Nx, Ny, 3) and every field of `ParticleCollection` gains a leading member
axis; member m is exactly the `WaveGrowth2D` with `winds[m]`."""
from __future__ import annotations

from types import SimpleNamespace

import numpy as np

from .WaveGrowthModels2D import WaveGrowth2D, _as_winds, eval_wind


def state_from_planes(S):
    """engine State planes (3, E, ny, Nx) -> model State (E, Nx, Ny, 3)"""
    return np.asarray(S).transpose(1, 3, 2, 0)


def planes_from_state(State):
    """model State (E, Nx, Ny, 3) -> engine State planes (3, E, ny, Nx)"""
    return np.asarray(State, dtype=np.float64).transpose(3, 0, 2, 1)


class WaveGrowth2DEnsemble(WaveGrowth2D):
    def __init__(self, *, winds, strip=None, **kwargs):
        """The keyword constructor of WaveGrowth2D; `winds` is a list of E wind specifications, each what
        WaveGrowth2D accepts except GriddedWinds (member m steps with winds[m])."""
        from ..Utils.WindEmulator import GriddedWinds
        if strip is not None:
            raise ValueError("WaveGrowth2DEnsemble: strip= is not supported; split the members over models instead")
        if not isinstance(winds, (list, tuple)) or len(winds) == 0:
            raise ValueError("WaveGrowth2DEnsemble: winds must be a non-empty list with one wind specification per member")
        members = [_as_winds(w) for w in winds]
        for m, w in enumerate(members):
            if isinstance(w, GriddedWinds):
                raise ValueError(f"WaveGrowth2DEnsemble: member {m} has GriddedWinds; the wind mesh is one per model, "
                                 "give the members wind closures")
            if not (callable(getattr(w, "u", None)) and callable(getattr(w, "v", None))):
                raise ValueError(f"WaveGrowth2DEnsemble: member {m} needs winds u(x, y, t) and v(x, y, t)")
        super().__init__(winds=members[0], strip=None, **kwargs)
        self.winds = members
        self.members = len(members)

    def _wind_planes(self, t):
        """(u, v) at time t of every member, as (E, ny, Nx) C-ordered planes."""
        self.engine  # noqa: B018  (binds self._rows)
        X = self.grid.data.x[:, self._rows]
        Y = self.grid.data.y[:, self._rows]
        u = np.stack([eval_wind(w.u, X, Y, t).T for w in self.winds])
        v = np.stack([eval_wind(w.v, X, Y, t).T for w in self.winds])
        return np.ascontiguousarray(u), np.ascontiguousarray(v)

    @property
    def State(self):
        """the (E, Nx, Ny, 3) node state [e, m_x, m_y] of every member, indexed [m, i, j, k]."""
        return state_from_planes(self.engine.state())

    @State.setter
    def State(self, S):
        S = np.asarray(S, dtype=np.float64)
        if S.shape != (self.members, self.Nx, self.Ny, 3):
            raise ValueError(f"State must have shape {(self.members, self.Nx, self.Ny, 3)}, not {S.shape}")
        self.engine.set_state(planes_from_state(S))

    @property
    def ParticleCollection(self):
        """the particles of every member: fields indexed [m, i, j] (u: [m, component, i, j])."""
        p = self.engine.particles()
        T = lambda a: a.transpose(0, 2, 1)
        z = p["z"]
        return SimpleNamespace(u=z.transpose(1, 0, 3, 2), lne=T(z[0]), c̄_x=T(z[1]), c̄_y=T(z[2]), x=T(z[3]), y=T(z[4]),
                               t=T(p["t"]), dt=T(p["dt"]), on=T((p["flags"] & 1) != 0),
                               boundary=T((p["flags"] & 2) != 0), active=T((p["flags"] & 8) != 0), status=T(p["status"]))

    def member_energy_sums(self):
        """sum of State[m, :, :, 0] per member, each bit for bit what the member alone returns"""
        return self.engine.member_energy_sums()
