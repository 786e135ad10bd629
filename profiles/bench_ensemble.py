"""Ensembles against separate handles: one JSON line per (grid, members) on stdout.

    python profiles/bench_ensemble.py [--steps 10] [--warmup 3] [--rounds 2] [--out FILE]

Grids: C1 (51 x 51, example_00_minimal.jl: the size PiCLES is run at most, where one model is launch-bound) and
512 x 512.  Members E in {1, 16, 256, 1024}; a size that does not fit in device memory is reported and skipped.  Member m
has its own steady wind (speed and direction vary over the members); the winds are staged once at the seed, so the
timed steps upload nothing.

For each line: the ensemble handle is stepped `steps` times (device events around the steps on its stream), then the
same E members as E single-member handles on the same GPU, one after another (a host clock around the steps: every
picles_step ends in a stream synchronise).  The two are alternated `rounds` times and the best round of each is kept.
Before timing, every member's State and energy sum are checked bit for bit against its single-member handle.
The card's name and power limit are read in the same call.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

from picles_b200 import FetchRelations as FR  # noqa: E402
from picles_b200._abi import PiclesError  # noqa: E402
from picles_b200.engine import B200Engine  # noqa: E402
from picles_b200.params import make_params  # noqa: E402
from picles_b200.ParticleSystems import particle_waves_v5 as PW  # noqa: E402

GRIDS = {"C1_51x51": (51, 51, 2000.0), "512x512": (512, 512, 2000.0)}
MEMBERS = (1, 16, 256, 1024)
DT = 600.0


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in out.split(",")]
        return dict(gpu=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # the numbers are still taken; the line says what could not be read
        return dict(gpu=f"unknown ({e})")


def params():
    pars, cid, _ = PW.ODEParameters(r_g=0.85)
    ps = PW.particle_equations(None, None, γ=cid.γ, q=cid.q)
    sets = PW.ODESettings(Parameters=pars, log_energy_minimum=FR.MinimalWindsea(10, 10, DT)["lne"], saving_step=DT,
                          timestep=DT, total_time=6 * 86400.0, dt=1e-3, dtmin=1e-4, force_dtmin=True)
    return make_params(sets, ps, FR.MinimalState(2, 2, DT), periodic_boundary=False)


def grid(Nx, Ny):
    """example_00_minimal.jl: non-periodic box, ocean everywhere, edges are grid boundary (mask 3)"""
    mask = np.ones((Ny, Nx), np.uint8)
    mask[0, :] = mask[-1, :] = 3
    mask[:, 0] = mask[:, -1] = 3
    return mask


def member_winds(E, Nx, Ny):
    """member m: 6-14 m/s, direction turning over the members"""
    m = np.arange(E)
    speed = 6.0 + 8.0 * ((m * 0.618034) % 1.0)
    ang = 2 * np.pi * m / max(E, 1)
    u = np.broadcast_to((speed * np.cos(ang))[:, None, None], (E, Ny, Nx))
    v = np.broadcast_to((speed * np.sin(ang))[:, None, None], (E, Ny, Nx))
    return np.ascontiguousarray(u), np.ascontiguousarray(v)


def run_line(gname, Nx, Ny, dx, E, P, steps, warmup, rounds):
    mask = grid(Nx, Ny)
    Mc = np.array([1 / dx, 0.0, 0.0, 1 / dx])
    u, v = member_winds(E, Nx, Ny)
    line = dict(grid=gname, Nx=Nx, Ny=Ny, members=E, steps=steps, warmup=warmup, rounds=rounds)
    ens = singles = None
    try:
        ens = B200Engine(Nx, Ny, 0, 0, mask, P, M_const=Mc, members=E)
        singles = [B200Engine(Nx, Ny, 0, 0, mask, P, M_const=Mc) for _ in range(E)]
    except PiclesError as e:
        line["skipped"] = f"does not fit: {e}"
        for x in [ens] + (singles or []):
            if x is not None:
                x.close()
        return line
    ens.seed(u if E > 1 else u[0], v if E > 1 else v[0])
    for m, s in enumerate(singles):
        s.seed(u[m], v[m])
    t = 0.0
    for _ in range(warmup):
        ens.step(t, DT)
        for s in singles:
            s.step(t, DT)
        t += DT
    # every member equals its single-member run, bit for bit
    S = ens.state().reshape(3, E, Ny, Nx)
    sums = ens.member_energy_sums()
    for m, s in enumerate(singles):
        Ss = s.state()
        if not np.array_equal(S[:, m].view(np.uint64), Ss.view(np.uint64)) or \
                np.float64(sums[m]).view(np.uint64) != np.float64(s.energy_sum()).view(np.uint64):
            raise SystemExit(f"{gname} E={E}: member {m} differs from its single-member run")
    line["bit_identical_members"] = E
    best_e = best_s = float("inf")
    launches = None
    for _ in range(rounds):
        l0 = ens.launch_count()
        ens.timer_start()
        for _ in range(steps):
            ens.step(t, DT)
            t += DT
        ms = ens.timer_stop() / steps
        launches = (ens.launch_count() - l0) / steps
        best_e = min(best_e, ms)
        t0 = time.perf_counter()
        ts = t - steps * DT
        for _ in range(steps):
            for s in singles:
                s.step(ts, DT)
            ts += DT
        best_s = min(best_s, (time.perf_counter() - t0) * 1e3 / steps)
    c = ens.counters()
    n = E * Nx * Ny
    line.update(ms_per_step_ensemble=best_e, ms_per_step_separate=best_s, speedup=best_s / best_e,
                particle_steps_per_s_ensemble=n / (best_e * 1e-3), particle_steps_per_s_separate=n / (best_s * 1e-3),
                launches_per_step_ensemble=launches, n_integrated_last_step=c["n_integrated"])
    ens.close()
    for s in singles:
        s.close()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
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
