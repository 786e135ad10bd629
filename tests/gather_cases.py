"""Cases for the projection gather (k_project_remesh), shared by tests/test_gather_geometry_cpu.py (host build of the device
header against the oracle) and tests/test_gpu_gather_geometry.py (the CUDA path against the oracle).

The gather picks its geometry from the reach R of the step's deposits: narrow tiles (64 x 16 targets, 2 halo rows) or
wide ones (64 x 12, 4 halo rows), guessed from the previous step's reach; a per-tile reach Rt from the rows within R of
the tile; the untiled path when Rt exceeds the tile's halo rows; the generic path near a periodic seam or the tripolar
fold.  Every case here fixes the reach of each of its steps, so that these choices are made on purpose:

- Propagation-only particles (source terms off) keep their c̄ from step to step, and a step of length dt moves every
  particle by M c̄ dt cells.  With c̄ set by ParticleDefaults, a step of (r - 1/2) / |M c̄| seconds gives reach r exactly
  (half a cell from either integer).  Without defaults c̄ comes from the wind sea of the local wind, so the reach varies
  with the wind: per member, or per row.
- A few cases run the full physics beside wide windows, so the reseed and switch-off branches of the remesh run there.

`observed(case, reaches, rows)` names the regimes a run of the case went through, from the reach of each step (the
oracle's counter) and, for propagation-only cases, the per-row reach (`row_reach_prediction`, which the GPU test checks
against B200Engine.row_reach).
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from common import (BND_NONPERIODIC, BND_PERIODIC, BND_TRIPOLAR_NORTH, cartesian_grid, default_params,
                    tripolar_grid)

# tile geometry of the gather (picles_b200/csrc/picles_device.h) and the largest reach it supports
TILE_X = 64
TILE_ROWS = 20
HY_NARROW = 2
HY_WIDE = 4
REACH_MAX = 15

SEQUENCES = ((1, 4, 4, 1), (2, 3, 9, 2), (4, 15, 1))


@dataclass
class Case:
    name: str
    grid: dict
    params: object
    winds: list                 # one wind function t -> (u, v) per member (one for a single model)
    dts: list                   # dt_model of every step
    claims: frozenset           # regimes the case is there for (each must be observed)
    propagation: bool = True    # c̄ is constant during a step: the per-row reach can be predicted
    accumulate: bool = False    # bare time_step! (State not zeroed before the gather)
    strips: tuple | None = None  # (nstrips, halo): y-strips with a host-driven exchange

    @property
    def wind(self):
        assert len(self.winds) == 1
        return self.winds[0]


def _const(u, v):
    return lambda t: (u, v)


def prop_params(c=None, DT=600.0, **kw):
    """source terms off; c = (c̄_x, c̄_y) of ParticleDefaults (lne = -3), or None for the wind sea of the local wind"""
    defaults = None if c is None else [-3.0, float(c[0]), float(c[1]), 0.0, 0.0]
    return default_params(DT=DT, defaults=defaults, input=False, dissipation=False, peak_shift=False, direction=False, **kw)


def dts_for(reaches, cells_per_second):
    """steps whose particles all move by (r - 1/2) cells along their fastest axis: reach r"""
    return [(r - 0.5) / cells_per_second for r in reaches]


def _seams(ocean, cols=(), rows=()):
    """land across the tile seams: a short run of land on each side of every given 0-based column / row"""
    Ny, Nx = ocean.shape
    for c in cols:
        if c + 1 < Nx:
            ocean[Ny // 3: Ny // 3 + 3, c:c + 2] = 0
    for r in rows:
        if r + 1 < Ny:
            ocean[r:r + 2, Nx // 4: Nx // 4 + 5] = 0
    return ocean


def _box(Nx, Ny, c, reaches, claims, bx=BND_NONPERIODIC, by=BND_NONPERIODIC, d=2000.0, seams=True, **kw):
    ocean = np.ones((Ny, Nx), np.uint8)
    if seams:
        _seams(ocean, cols=(TILE_X - 1,), rows=(11, 15))
    g = cartesian_grid(Nx, Ny, dx=d, dy=d, bx=bx, by=by, ocean=ocean)
    cps = max(abs(c[0]), abs(c[1])) / d
    P = prop_params(c, **{k: v for k, v in kw.items() if k in ("periodic_boundary",)})
    rest = {k: v for k, v in kw.items() if k not in ("periodic_boundary",)}
    return g, P, [_const(5.0, 5.0)], dts_for(reaches, cps), frozenset(claims), rest


def _case(name, Nx, Ny, c, reaches, claims, **kw):
    g, P, w, dts, cl, rest = _box(Nx, Ny, c, reaches, claims, **kw)
    return Case(name, g, P, w, dts, cl, **rest)


def _tripolar_band():
    """tripolar 64 x 33 (periodic x, fold at the top), per-node kernel whose cells shrink towards the pole: the rows
    next to the fold move several times further than the rest, so tiles far from the pole have a small window"""
    Nx, Ny = 64, 33
    ocean = np.ones((Ny, Nx), np.uint8)
    ocean[Ny - 2:, 20:27] = 0
    ocean[11:13, 40:44] = 0
    g = tripolar_grid(Nx, Ny, ocean=ocean, lat_min=-40.0)
    g["M"] = g["M"] * 40.0
    P = prop_params((2.0, 1.0), DT=1800.0, periodic_boundary=True)
    M = g["M"]
    cps = float(np.max(np.maximum(np.abs(M[0] * 2.0 + M[1] * 1.0), np.abs(M[2] * 2.0 + M[3] * 1.0))))
    return Case("tripolar_fold_band_64x33", g, P, [_const(5.0, 5.0)], dts_for([3, 8, 15, 2], cps),
                frozenset({"tripolar fold at reach > 2", "per-row reach: Rt <= HY < R", "reach 15", "Nx=64", "Ny=33"}))


def _row_band():
    """wind-sea particles on 128 x 33: a light wind below row 24 (reach 1), a strong one above row 27 (reach > 4)"""
    Nx, Ny = 128, 33
    ocean = _seams(np.ones((Ny, Nx), np.uint8), cols=(TILE_X - 1,), rows=(15,))
    g = cartesian_grid(Nx, Ny, dx=100.0, dy=100.0, ocean=ocean)
    rows = np.arange(Ny)[:, None] + np.zeros((1, Nx))
    u = np.where(rows < 24, 3.0, np.where(rows < 28, 8.0, 14.0))
    v = 0.3 * u
    return Case("row_band_128x33", g, prop_params(None), [_const(u, v)], [600.0] * 3,
                frozenset({"per-row reach: Rt <= HY < R", "reach 5-14", "Nx=128", "Ny=33"}))


def _physics_box():
    """full physics on 131 x 24 cells of 500 m: growing winds with a calm inflow strip (particles switched off and
    reseeded) and steps long enough for wide and untiled windows"""
    from scenarios import _growing
    Nx, Ny = 131, 24
    ocean = _seams(np.ones((Ny, Nx), np.uint8), cols=(TILE_X - 1, 2 * TILE_X - 1), rows=(11,))
    g = cartesian_grid(Nx, Ny, dx=500.0, dy=500.0, ocean=ocean)
    P = default_params(DT=1200.0, wind_min_squared=2.0)
    return Case("physics_growing_131x24", g, P, [_growing(g, 14.0, -5.0)], [1200.0, 1800.0, 2400.0, 900.0, 1500.0],
                frozenset({"full physics beside wide windows", "Nx=131", "Ny=24"}), propagation=False)


def _physics_tripolar():
    """full physics on the tripolar grid with the model's periodic flag: reseeds next to the fold at reach > 2"""
    Nx, Ny = 64, 24
    ocean = np.ones((Ny, Nx), np.uint8)
    ocean[:2, :] = 0
    ocean[10:14, 8:15] = 0
    g = tripolar_grid(Nx, Ny, ocean=ocean)
    g["M"] = g["M"] * 60.0
    P = default_params(DT=1200.0, periodic_boundary=True)

    def wind(t):
        return 15.0, -10.0 * np.cos(5 * t / (3600 * 2 * np.pi))

    return Case("physics_tripolar_64x24", g, P, [wind], [1200.0, 2400.0, 1200.0, 3600.0],
                frozenset({"full physics beside wide windows", "tripolar fold at reach > 2"}), propagation=False)


def ensemble_case():
    """three members on 65 x 17 (a partial last tile in x and in y): calm (nothing deposited), reach 1, reach > 6"""
    g = cartesian_grid(65, 17, dx=100.0, dy=100.0)
    return Case("ensemble_calm_1_11_65x17", g, prop_params(None),
                [_const(0.6, -0.5), _const(3.0, 1.0), _const(-20.0, 6.0)], [600.0] * 3,
                frozenset({"ensemble: calm, 1, >= 6", "Nx=65", "Ny=17"}))


def cases():
    out = [
        _case("seq_1441_64x16", 64, 16, (2.0, 0.7), [1, 4, 4, 1],
              {"sequence 1->4->4->1", "reach 1", "reach 3-4 narrow tiles", "reach 3-4 wide tiles", "nonperiodic",
               "Nx=64", "Ny=16"}),
        _case("seq_2392_65x33", 65, 33, (-2.0, 1.2), [2, 3, 9, 2],
              {"sequence 2->3->9->2", "reach 2", "reach 5-14", "guess wide, reach >=5", "land on tile seams", "Nx=65",
               "Ny=33"}),
        _case("seq_4151_131x24", 131, 24, (2.5, -1.5), [4, 15, 1],
              {"sequence 4->15->1", "reach 15", "guess narrow, reach <=2", "Nx=131", "Ny=24"}),
        _case("periodic_x_63x13", 63, 13, (2.0, -1.0), [1, 2, 6, 12, 6],
              {"periodic x", "guess narrow, reach >=5", "Nx=63", "Ny=13"}, bx=BND_PERIODIC),
        _case("periodic_y_128x17", 128, 17, (0.8, -2.0), [3, 3, 2, 5, 4],
              {"periodic y", "guess wide, reach <=2", "guess wide, reach 3-4", "Nx=128", "Ny=17"}, by=BND_PERIODIC),
        _case("periodic_xy_130x12", 130, 12, (2.0, 2.0), [2, 4, 8, 3],
              {"periodic x and y", "periodic y, 2R+1 > Ny", "Nx=130", "Ny=12"}, bx=BND_PERIODIC, by=BND_PERIODIC),
        _case("periodic_x_thin_5x33", 5, 33, (2.0, 0.3), [3, 6, 2],
              {"periodic x, 2R+1 > Nx", "Nx=5", "Ny=33"}, bx=BND_PERIODIC, seams=False),
        _case("periodic_y_thin_65x7", 65, 7, (0.3, -2.0), [4, 7, 1],
              {"periodic y, 2R+1 > Ny", "Nx=65", "Ny=7"}, by=BND_PERIODIC),
        _case("periodic_xy_5x7", 5, 7, (2.0, 1.5), [2, 5, 9],
              {"periodic x and y", "periodic x, 2R+1 > Nx", "periodic y, 2R+1 > Ny", "Nx=5", "Ny=7"},
              bx=BND_PERIODIC, by=BND_PERIODIC, seams=False),
        _case("model_periodic_130x24", 130, 24, (2.0, -0.9), [2, 3, 6, 3],
              {"two deposit classes at reach > 1, several tiles wide", "Nx=130", "Ny=24"}, periodic_boundary=True),
        _case("accumulate_untiled_65x17", 65, 17, (-1.5, -2.0), [1, 6, 3, 4],
              {"accumulate, untiled", "Nx=65", "Ny=17"}, accumulate=True),
        _tripolar_band(),
        _row_band(),
        _physics_box(),
        _physics_tripolar(),
        _case("strips3_halo8_65x33", 65, 33, (1.2, 2.0), [5, 8, 6],
              {"strips, halo = reach 5-8", "Nx=65", "Ny=33"}, strips=(3, 8)),
        _case("strips2_halo7_131x17", 131, 17, (2.0, -1.1), [5, 7],
              {"strips, halo = reach 5-8", "Nx=131", "Ny=17"}, strips=(2, 7)),
    ]
    return out


CASES = {c.name: c for c in cases()}

# every regime the generator has to reach (test_gather_geometry_cpu asserts each is observed in some case)
REQUIRED = frozenset(
    {"reach 1", "reach 2", "reach 3-4 wide tiles", "reach 3-4 narrow tiles", "reach 5-14", "reach 15"}
    | {"sequence " + "->".join(map(str, s)) for s in SEQUENCES}
    | {f"guess {g}, reach {r}" for g in ("narrow", "wide") for r in ("<=2", "3-4", ">=5")}
    | {"nonperiodic", "periodic x", "periodic y", "periodic x and y", "periodic x, 2R+1 > Nx", "periodic y, 2R+1 > Ny",
       "tripolar fold at reach > 2", "per-row reach: Rt <= HY < R", "two deposit classes at reach > 1, several tiles wide",
       "accumulate, untiled", "full physics beside wide windows", "land on tile seams", "strips, halo = reach 5-8",
       "ensemble: calm, 1, >= 6"}
    | {f"Nx={n}" for n in (5, 63, 64, 65, 128, 130, 131)}
    | {f"Ny={n}" for n in (7, 12, 13, 16, 17, 24, 33)})


# ---- what a run went through ------------------------------------------------------------------------------------

def tile_guess(prev_reach):
    """the tile geometry k_project_remesh is launched with, from the previous step's reach (picles_capi.cu wide_tiles)"""
    return "wide" if HY_NARROW < prev_reach <= HY_WIDE else "narrow"


def tile_halo(guess):
    return HY_WIDE if guess == "wide" else HY_NARROW


def row_reach_prediction(grid, particles, dt):
    """per row: the largest reach of the deposits this step's particles will write, for propagation-only particles (c̄
    constant during the step): a particle that is iterated and on moves by M c̄ dt cells from its home node"""
    Ny, Nx = grid["Ny"], grid["Nx"]
    if grid["M"] is not None:
        M = grid["M"]
    else:
        M = np.broadcast_to(np.asarray(grid["M_const"], np.float64)[:, None, None], (4, Ny, Nx))
    fl = particles["flags"]
    deposits = ((fl & 8) != 0) & ((fl & 1) != 0)
    cx, cy = particles["z"][1], particles["z"][2]
    fx = np.floor((M[0] * cx + M[1] * cy) * dt)
    fy = np.floor((M[2] * cx + M[3] * cy) * dt)
    r = np.maximum.reduce([np.abs(fx), np.abs(fx + 1), np.abs(fy), np.abs(fy + 1)])
    r = np.where(deposits, r, 0).astype(np.int64)
    return r.max(axis=1)


def tiles_narrowed(rows, R, guess):
    """tiles of the guessed geometry whose own window Rt (rows within R of their targets) fits the halo rows although R
    does not"""
    HY = tile_halo(guess)
    TY = TILE_ROWS - 2 * HY
    n = 0
    for jr0 in range(0, len(rows), TY):
        lo, hi = max(jr0 - R, 0), min(jr0 + TY + R, len(rows))
        Rt = min(int(rows[lo:hi].max()), R)
        n += Rt <= HY < R
    return n


def observed(case, reaches, rows=None, member_reaches=None):
    """regimes of one run: reaches = the oracle's reach of each step; rows = per step, the per-row reach (or None)"""
    g, out = case.grid, set()
    prev = 0
    for k, r in enumerate(reaches):
        guess = tile_guess(prev)
        if r in (1, 2):
            out.add(f"reach {r}")
        elif r in (3, 4):
            out.add(f"reach 3-4 {guess} tiles")
        elif 5 <= r <= 14:
            out.add("reach 5-14")
        elif r == 15:
            out.add("reach 15")
        cls = "<=2" if r <= 2 else ("3-4" if r <= 4 else ">=5")
        out.add(f"guess {guess}, reach {cls}")
        untiled = r > HY_WIDE or (r > HY_NARROW and guess == "narrow")
        if case.accumulate and untiled:
            out.add("accumulate, untiled")
        if rows is not None and rows[k] is not None and tiles_narrowed(rows[k], r, guess):
            out.add("per-row reach: Rt <= HY < R")
        prev = r
    for s in SEQUENCES:
        if any(tuple(reaches[k:k + len(s)]) == s for k in range(len(reaches))):
            out.add("sequence " + "->".join(map(str, s)))
    R = max(reaches)
    bx, by = g["bx"], g["by"]
    if by == BND_TRIPOLAR_NORTH:
        if g["M"] is not None and R > 2:
            out.add("tripolar fold at reach > 2")
    elif bx == BND_PERIODIC and by == BND_PERIODIC:
        out.add("periodic x and y")
    elif bx == BND_PERIODIC:
        out.add("periodic x")
    elif by == BND_PERIODIC:
        out.add("periodic y")
    else:
        out.add("nonperiodic")
    if bx == BND_PERIODIC and 2 * R + 1 > g["Nx"]:
        out.add("periodic x, 2R+1 > Nx")
    if by == BND_PERIODIC and 2 * R + 1 > g["Ny"]:
        out.add("periodic y, 2R+1 > Ny")
    if case.params.periodic_boundary and by == BND_NONPERIODIC and R > 1 and g["Nx"] > 2 * TILE_X:
        out.add("two deposit classes at reach > 1, several tiles wide")
    if not case.propagation and R > HY_NARROW:
        out.add("full physics beside wide windows")
    land = (g["mask"] == 0) | (g["mask"] == 2)  # total mask: 0 land, 2 coast, 1 ocean, 3 ocean on the grid edge
    seams_x = [c for c in (TILE_X - 1, 2 * TILE_X - 1) if c + 1 < g["Nx"]]
    seams_y = [r for r in (11, 15) if r + 1 < g["Ny"]]
    if any(land[:, c:c + 2].any() for c in seams_x) and any(land[r:r + 2].any() for r in seams_y):
        out.add("land on tile seams")
    if case.strips:
        ns, halo = case.strips
        edges = [g["Ny"] * k // ns for k in range(1, ns)]
        if 5 <= halo <= 8 and halo == R and all(e % 16 and e % 12 for e in edges):
            out.add("strips, halo = reach 5-8")
    if member_reaches is not None and len(member_reaches) == 3:
        if sorted(member_reaches)[0] == 0 and 1 in member_reaches and max(member_reaches) >= 6:
            out.add("ensemble: calm, 1, >= 6")
    out.add(f"Nx={g['Nx']}")
    out.add(f"Ny={g['Ny']}")
    return out


def run_case(ref, dut, case, compare, wind=None, on_step=None):
    """seed + every step of `case` on both models (one wind: `wind`, else the case's), compared after the seed and after
    every step; on_step(k, ref, dut, particles_before) is called after each step's comparison"""
    wind = wind or case.wind
    u0, v0 = wind(0.0)
    ref.seed(u0, v0)
    dut.seed(u0, v0)
    if case.accumulate:
        ref.set_accumulate(True)
        dut.set_accumulate(True)
    compare(ref, dut)
    t = 0.0
    for k, dt in enumerate(case.dts):
        before = ref.particles()
        ut, vt = wind(t)
        ut1, vt1 = wind(t + dt)
        ref.step(t, dt, ut, vt, ut1, vt1)
        dut.step(t, dt, ut, vt, ut1, vt1)
        t += dt
        compare(ref, dut)
        if on_step is not None:
            on_step(k, ref, dut, before)
