"""Ensembles forced by gridded winds, one mesh per member: one JSON line per (grid, members) on stdout.

    python profiles/bench_ensemble_wind.py [--steps 5] [--warmup 2] [--rounds 2] [--out FILE]

Grids as profiles/bench_ensemble.py: C1 (51 x 51) and 512 x 512, members E in {16, 256, 1024}; a size that does not fit in
device memory is reported and skipped.  Every member has its own time-varying mesh on shared knots: 25 km spacing (an
ERA5-like 0.25 degrees) over the domain, 25 hourly time knots; the 600 s steps fall between time knots, so every step
samples new levels.

Timed, alternating in each round (the best round of each is kept):
  (a) the ensemble handle with member meshes (picles_set_member_wind_meshes): picles_step_wind_mesh, device events;
  (b) the same handle with the winds interpolated on the host (numpy, node lookup precomputed once) and uploaded every
      step: the t+dt level of E members per step, the t level reused; a host clock around interpolation + picles_step;
  (c) E single-member handles, each with its own mesh (picles_set_wind_mesh), stepped one after another; a host clock.
      Skipped where E handles do not fit beside the ensemble (the line says so).
Before timing, (a) is checked bit for bit against (c) on every member (or, where (c) is skipped, against single handles
for members 0, E/2 and E-1): State and energy sum.

Also recorded: the time of one wind level of the member sampler (picles_measure_wind_sample: both passes, CUDA events)
against the bytes the two passes must move, the HBM copy bandwidth measured in the same call (picles_measure_hbm_copy),
whether the E-slice scratch fits the 126 MB L2, and the card's name and power limit.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, ".."))
sys.path.insert(0, HERE)

from bench_ensemble import GRIDS, card, grid, params  # noqa: E402
from picles_b200._abi import PiclesError  # noqa: E402
from picles_b200.engine import B200Engine  # noqa: E402

MEMBERS = (16, 256, 1024)
DT = 600.0
L2_BYTES = 126 * 2 ** 20
SINGLES_MAX_NODES = 2 ** 28  # E * Nx * Ny above this: (c) is not run (E more handles of this size beside the ensemble)


def member_meshes(E, Nx, Ny, dx, seed=0):
    """shared knots, member m's fields: a mean wind turning with m plus travelling and random parts"""
    rng = np.random.default_rng(seed)
    Lx, Ly = Nx * dx, Ny * dx
    xw = np.linspace(-dx, Lx + dx, int(np.ceil(Lx / 25e3)) + 3)
    yw = np.linspace(-dx, Ly + dx, int(np.ceil(Ly / 25e3)) + 3)
    tw = 3600.0 * np.arange(25)
    m = np.arange(E)[:, None, None, None]
    T, Y, X = np.meshgrid(tw, yw, xw, indexing="ij")
    speed = 6.0 + 8.0 * ((m * 0.618034) % 1.0)
    ang = 2 * np.pi * m / E + 0.3 * np.sin(2 * np.pi * (X / Lx - T / 86400.0))[None]
    U = speed * np.cos(ang) + rng.normal(0.0, 1.0, (E,) + T.shape)
    V = speed * np.sin(ang) + rng.normal(0.0, 1.0, (E,) + T.shape)
    return xw, yw, tw, np.ascontiguousarray(U), np.ascontiguousarray(V)


class HostSampler:
    """the same interpolation on the host: node lookup once, then per level a time blend and four gathers per member"""

    def __init__(self, xw, yw, tw, U, V, X, Y, chunk=32):
        self.tw, self.U, self.V, self.chunk = tw, U, V, chunk
        ix = np.clip(np.searchsorted(xw, X.ravel(), "left") - 1, 0, xw.size - 2)
        iy = np.clip(np.searchsorted(yw, Y.ravel(), "left") - 1, 0, yw.size - 2)
        self.dx = (X.ravel() - xw[ix]) / (xw[ix + 1] - xw[ix])
        self.dy = (Y.ravel() - yw[iy]) / (yw[iy + 1] - yw[iy])
        self.off, self.row, self.shape = ix + xw.size * iy, xw.size, X.shape

    def __call__(self, t):
        tw = self.tw
        tp = (t - tw[0]) % (tw[-1] - tw[0]) + tw[0]
        it = int(np.clip(np.searchsorted(tw, tp, "left") - 1, 0, tw.size - 2))
        w = (tp - tw[it]) / (tw[it + 1] - tw[it])
        E = self.U.shape[0]
        out = [np.empty((E,) + self.shape) for _ in range(2)]
        o, r, dx, dy = self.off, self.row, self.dx, self.dy
        for A, res in zip((self.U, self.V), out):
            for m0 in range(0, E, self.chunk):
                S = ((1 - w) * A[m0:m0 + self.chunk, it] + w * A[m0:m0 + self.chunk, it + 1]).reshape(-1, A.shape[2] * A.shape[3])
                v = (1 - dx) * ((1 - dy) * S[:, o] + dy * S[:, o + r]) + dx * ((1 - dy) * S[:, o + 1] + dy * S[:, o + r + 1])
                res[m0:m0 + self.chunk] = v.reshape((-1,) + self.shape)
        return out


def same_bits(a, b):
    a, b = np.ascontiguousarray(a, np.float64), np.ascontiguousarray(b, np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def run_line(gname, Nx, Ny, dx, E, P, steps, warmup, rounds):
    mask = grid(Nx, Ny)
    Mc = np.array([1 / dx, 0.0, 0.0, 1 / dx])
    X, Y = np.meshgrid(np.arange(Nx) * dx, np.arange(Ny) * dx)
    xw, yw, tw, U, V = member_meshes(E, Nx, Ny, dx)
    n = Nx * Ny
    line = dict(grid=gname, Nx=Nx, Ny=Ny, members=E, mesh=[int(xw.size), int(yw.size), int(tw.size)], steps=steps,
                warmup=warmup, rounds=rounds)
    run_c = E * n <= SINGLES_MAX_NODES
    check = list(range(E)) if run_c else sorted({0, E // 2, E - 1})
    ens, singles = None, []
    try:
        ens = B200Engine(Nx, Ny, 0, 0, mask, P, M_const=Mc, members=E)
        ens.set_member_wind_meshes(xw, yw, tw, U, V, X, Y)
        for m in check:
            s = B200Engine(Nx, Ny, 0, 0, mask, P, M_const=Mc)
            s.set_wind_mesh(xw, yw, tw, U[m], V[m], X, Y)
            singles.append(s)
    except PiclesError as e:
        line["skipped"] = f"does not fit: {e}"
        for x in [ens] + singles:
            if x is not None:
                x.close()
        return line
    if not run_c:
        line["separate_handles"] = f"not run: {E} handles of {Nx}x{Ny} beside the ensemble; checked members {check}"
    for e in [ens] + singles:
        e.seed_wind_mesh(0.0)
    t = 0.0
    for _ in range(warmup):
        for e in [ens] + singles:
            e.step_wind_mesh(t, DT, 0)
        t += DT
    S = ens.state()
    sums = ens.member_energy_sums()
    for m, s in zip(check, singles):
        if not same_bits(S[:, m], s.state()) or not same_bits(sums[m:m + 1], np.array([s.energy_sum()])):
            raise SystemExit(f"{gname} E={E}: member {m} differs from its single-member handle")
    line["bit_identical_members"] = len(check)
    host = HostSampler(xw, yw, tw, U, V, X, Y)
    best = dict(a=float("inf"), b=float("inf"), c=float("inf"))
    launches = None
    for _ in range(rounds):
        t0s = t
        l0 = ens.launch_count()
        ens.timer_start()
        for _ in range(steps):
            ens.step_wind_mesh(t, DT, 0)
            t += DT
        best["a"] = min(best["a"], ens.timer_stop() / steps)
        launches = (ens.launch_count() - l0) / steps
        # (b): the first step uploads both levels, the others only t+dt (the t level is reused on the device)
        tb = t0s
        c0 = time.perf_counter()
        for k in range(steps):
            u1, v1 = host(tb + DT)
            if k == 0:
                ut, vt = host(tb)
                ens.step(tb, DT, ut, vt, u1, v1)
            else:
                ens.step(tb, DT, None, None, u1, v1)
            tb += DT
        best["b"] = min(best["b"], (time.perf_counter() - c0) * 1e3 / steps)
        if run_c:
            tc = t0s
            c0 = time.perf_counter()
            for _ in range(steps):
                for s in singles:
                    s.step_wind_mesh(tc, DT, 0)
                tc += DT
            best["c"] = min(best["c"], (time.perf_counter() - c0) * 1e3 / steps)
    st = xw.size * yw.size
    ms_level = ens.measure_wind_sample(t + 0.5 * DT, reps=20)
    hbm = ens.measure_hbm_copy()
    bytes_level = 48 * E * st + 16 * n + 16 * E * n
    line.update(ms_per_step_member_meshes=best["a"], ms_per_step_host_winds=best["b"],
                host_upload_bytes_per_step=16 * E * n, launches_per_step_member_meshes=launches,
                ms_per_wind_level=ms_level, bytes_per_wind_level=bytes_level,
                GBps_wind_level=bytes_level / (ms_level * 1e6), hbm_copy_GBps=hbm,
                share_of_copy_bandwidth=bytes_level / (ms_level * 1e6) / hbm if hbm > 0 else None,
                scratch_bytes=16 * E * st, scratch_fits_l2=16 * E * st <= L2_BYTES,
                speedup_vs_host_winds=best["b"] / best["a"],
                particle_steps_per_s_member_meshes=E * n / (best["a"] * 1e-3))
    if run_c:
        line.update(ms_per_step_separate=best["c"], speedup_vs_separate=best["c"] / best["a"])
    for x in [ens] + singles:
        x.close()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--grids", default=",".join(GRIDS))
    ap.add_argument("--members", default=",".join(map(str, MEMBERS)))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    P = params()
    info = card()
    out = open(a.out, "a") if a.out else None
    for gname in a.grids.split(","):
        Nx, Ny, dx = GRIDS[gname]
        for E in map(int, a.members.split(",")):
            line = run_line(gname, Nx, Ny, dx, E, P, a.steps, a.warmup, a.rounds)
            line.update(info)
            s = json.dumps(line)
            print(s, flush=True)
            if out:
                out.write(s + "\n")
                out.flush()


if __name__ == "__main__":
    main()
