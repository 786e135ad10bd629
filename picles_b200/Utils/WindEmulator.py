"""Gridded winds — `wind_interpolator` of `src/Utils/WindEmulator.jl:18-43` and the ERA5 loader
pattern of `tests/T03_PIC_tripolar_realistic.jl:61-73`:

    u_grid = LinearInterpolation((x, y, t), U, extrapolation_bc=Periodic())

On the B200 architecture a `GriddedWinds` given as `winds=` of `WaveGrowth2D` is uploaded once
(`picles_set_wind_mesh`) and sampled at the nodes ON THE DEVICE every step (`k_wind_sample`), so a
model step moves no wind data over PCIe.  The object is also callable like the reference's
interpolators, `winds.u(x, y, t)`, for scripts that plot or inspect the forcing: that evaluation
runs on the GPU as well (`picles_sample_wind_mesh`) once the model owns an engine; before that it
raises — there is no CPU evaluation path in this package.
"""
from __future__ import annotations

import numpy as np


class GriddedWinds:
    """wind_grid = (u=U[ix,iy,it], v=V[ix,iy,it], x=xi, y=yi, t=ti)  ->  device-resident mesh."""

    def __init__(self, x, y, t, u, v):
        self.x = np.ascontiguousarray(np.asarray(x, np.float64))
        self.y = np.ascontiguousarray(np.asarray(y, np.float64))
        self.t = np.ascontiguousarray(np.asarray(t, np.float64))
        shape = (self.x.size, self.y.size, self.t.size)
        u, v = np.asarray(u, np.float64), np.asarray(v, np.float64)
        if u.shape != shape or v.shape != shape:
            raise ValueError(f"u and v must be indexed [ix, iy, it] with shape {shape}")
        for k in (self.x, self.y, self.t):
            if k.size < 2 or not np.all(np.diff(k) > 0):
                raise ValueError("knot vectors need at least 2 strictly increasing values")
        # device layout: nt slices of ny*nx, x fastest
        self.U = np.ascontiguousarray(u.transpose(2, 1, 0))
        self.V = np.ascontiguousarray(v.transpose(2, 1, 0))
        self._engine = None
        self._member = None  # the member this mesh drives in an ensemble engine (WaveGrowth2DEnsemble)

    def bind(self, engine, node_x, node_y):
        engine.set_wind_mesh(self.x, self.y, self.t, self.U, self.V, node_x, node_y)
        self._engine, self._member = engine, None

    def _planes(self, t):
        if self._engine is None:
            raise RuntimeError("GriddedWinds is evaluated on the device: attach it to a WaveGrowth2D model first")
        u, v = self._engine.sample_wind_mesh(t)
        if self._member is not None:  # the ensemble engine samples every member: this member's planes
            return u[self._member], v[self._member]
        return u, v

    # the reference's closures, on the model's own nodes
    def u(self, x, y, t):
        return self._planes(t)[0].T

    def v(self, x, y, t):
        return self._planes(t)[1].T


def wind_interpolator(wind_grid):
    """wind_interpolator(wind_grid) for 2-D grids: dict / namespace with u, v, x, y, t."""
    g = wind_grid if isinstance(wind_grid, dict) else vars(wind_grid)
    if "y" not in g or "u" not in g or "v" not in g:
        raise NotImplementedError("only 2-D wind grids with both components (u, v, x, y, t) are supported on this path")
    return GriddedWinds(g["x"], g["y"], g["t"], g["u"], g["v"])
