"""`WaveGrowth2DEnsemble` — E `WaveGrowth2D` models on one grid, each with its own winds, stepped
together in one B200 engine (an ensemble handle, picles_set_members).

The reference runs many small configurations one after another (the sweeps over wind sign and
periodicity of T04_2D_reg_test.jl, the (U10, V10) variants of T04_2D_growing_decaying_winds.jl); an
ensemble of wind forcings is also how a wave forecast expresses its uncertainty.  Here the members
share the grid, the mask, the projection kernel and every setting, and each step launches the
kernels one model launches, whatever E is.

Layout: `State` is (E, Nx, Ny, 3) and every field of `ParticleCollection` gains a leading member
axis; member m is exactly the `WaveGrowth2D` with `winds[m]`.  Gridded winds (every member a
`GriddedWinds` on the same knots) stay on the device, one mesh per member."""
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


def _same_bits(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


class MemberGriddedWinds:
    """The GriddedWinds of every member, on shared knots, bound to an ensemble engine as one call
    (picles_set_member_wind_meshes): each member's mesh is then sampled on the device every step."""

    def __init__(self, members):
        self.members = list(members)

    def bind(self, engine, node_x, node_y):
        w0 = self.members[0]
        U = np.stack([w.U for w in self.members])
        V = np.stack([w.V for w in self.members])
        engine.set_member_wind_meshes(w0.x, w0.y, w0.t, U, V, node_x, node_y)
        for m, w in enumerate(self.members):
            w._engine, w._member = engine, m


class WaveGrowth2DEnsemble(WaveGrowth2D):
    def __init__(self, *, winds, strip=None, **kwargs):
        """The keyword constructor of WaveGrowth2D; `winds` is a list of E wind specifications, each what
        WaveGrowth2D accepts (member m steps with winds[m]).  GriddedWinds are taken when every member has them,
        on bitwise-identical knots: the E meshes then stay on the device and are sampled there."""
        from ..Utils.WindEmulator import GriddedWinds
        if strip is not None:
            raise ValueError("WaveGrowth2DEnsemble: strip= is not supported; split the members over models instead")
        if not isinstance(winds, (list, tuple)) or len(winds) == 0:
            raise ValueError("WaveGrowth2DEnsemble: winds must be a non-empty list with one wind specification per member")
        members = [_as_winds(w) for w in winds]
        gridded = [isinstance(w, GriddedWinds) for w in members]
        if any(gridded) and not all(gridded):
            if gridded[0]:
                k = gridded.index(False)
                raise ValueError(f"WaveGrowth2DEnsemble: member 0 has GriddedWinds and member {k} has not; the members "
                                 "take GriddedWinds on shared knots or wind closures, not both")
            k = gridded.index(True)
            raise ValueError(f"WaveGrowth2DEnsemble: member {k} has GriddedWinds and member 0 has not; the members "
                             "take GriddedWinds on shared knots or wind closures, not both")
        if all(gridded):
            w0 = members[0]
            for m, w in enumerate(members[1:], 1):
                if not (_same_bits(w.x, w0.x) and _same_bits(w.y, w0.y) and _same_bits(w.t, w0.t)):
                    raise ValueError(f"WaveGrowth2DEnsemble: member {m} has GriddedWinds on other knots than member 0; "
                                     "the members' meshes share x, y and t")
        else:
            for m, w in enumerate(members):
                if not (callable(getattr(w, "u", None)) and callable(getattr(w, "v", None))):
                    raise ValueError(f"WaveGrowth2DEnsemble: member {m} needs winds u(x, y, t) and v(x, y, t)")
        super().__init__(winds=members[0], strip=None, **kwargs)
        self.winds = members
        self.members = len(members)
        self._gridded_winds = MemberGriddedWinds(members) if all(gridded) else None

    def _wind_planes(self, t):
        """(u, v) at time t of every member, as (E, ny, Nx) C-ordered planes."""
        eng = self.engine  # binds self._rows
        if self._gridded_winds is not None:
            return eng.sample_wind_mesh(t)
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
