#!/usr/bin/env python
"""bench.py — particle-steps/s of the PiCLES per-timestep particle-in-cell loop on B200.

  python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, through the C ABI)
  python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the oracle port on all host cores
  python bench.py ... --dump-outputs DIR                   # also save what the last timed step computed (dump_outputs)
  (N > 1: launched by torch.distributed.run, one rank per GPU)

Workload (BASELINE.json configs[1]): T04_2D_reg_test_large_grid / bench06 homogeneous box
scaled to 4096x4096 Cartesian, dx=dy=2 km, constant wind u=v=10 m/s, model step 10 min,
example_00_minimal ODE settings (Tsit5 controller, dt=1e-3, dtmin=1e-4, force_dtmin).
A "step" is one model step: State .= 0; advance! (adaptive RK over DT for every particle);
ParticleToNode! projection; remesh!.  With N GPUs every rank owns a 4096x4096 y-strip of a
4096 x (4096*N) box (weak scaling: `value`) and exchanges a halo of particle records per step.
Three more legs run when N > 1, untimed by the headline: `strong` — the FIXED 4096x4096 box cut in N
strips, with the same box on one GPU timed by rank 0 in the same process (BASELINE.md's 85 % target
is on this); `strip_parity` — a small growing-wind box stepped in N strips over NCCL and as one
domain on rank 0, compared bit for bit; and `strong_c5` — BASELINE configs[4], the 4320x3840 tripolar +
land grid cut in N strips by measured cost, against the same grid on one GPU.

One JSON line is printed by rank 0.  See DESIGN.md §measurement for every field.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def ncu_record():
    """What ncu measured, never under the timer: dram__bytes_read.sum + dram__bytes_write.sum per launch and
    sm__pipe_fp64_cycles_active of the kernels of the 4096^2 bench step, read from the tracked summary that
    profiles/ncu_to_json.py writes from the committed `ncu --set full` captures.  The file names the commit
    the captured library was built from; the bench line carries that stamp next to the numbers."""
    p = os.path.join(ROOT, "profiles", "ncu_metrics.json")
    try:
        with open(p) as f:
            return json.load(f)
    except (OSError, ValueError):
        return {"commit": None, "kernels": {}}

METRIC = "particle-steps/s"
UNIT = "particle-steps/s"

# Algorithmic FP64 work (DESIGN.md §advance kernel): source-level operation counts of
# physics.h with fma = 2, add/mul/compare-select = 1, div = sqrt = 8, exp = 30,
# tanh = sech = log = 35, pow = 70 flop.
F_RHS = 329          # one right-hand side (rhs3 + prop + wind interpolation)
F_ATTEMPT = 511      # one RK attempt minus its 6 RHS: stage sums, error norm, PI controller
F_INITDT = 319       # Hairer initial step minus its RHS
F_DEPOSIT = 105      # charge + weights of the deposit record
# Algorithmic HBM bytes per node of the fused gather + remesh kernel (DESIGN.md §4.2): read one
# deposit record (5 f64 + packed cell) and the particle flags; write 3 f64 of State, the
# particle's u[5] and its flags (remesh branch A, the steady state of an all-ocean box)
B_PROJECT_REMESH = 44 + 1 + 24 + 40 + 1


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ---------------------------------------------------------------------------------------
def workload(nx, ny_per_gpu, n_gpus, rank):
    """Global homogeneous box Nx x (ny_per_gpu*n_gpus), both axes non-periodic, all ocean."""
    Ny = ny_per_gpu * n_gpus
    j0 = rank * ny_per_gpu
    mask = np.ones((ny_per_gpu, nx), np.uint8)
    mask[:, 0] = 3
    mask[:, -1] = 3
    if j0 == 0:
        mask[0, :] = 3
    if j0 + ny_per_gpu == Ny:
        mask[-1, :] = 3
    return dict(Nx=nx, Ny=Ny, j0=j0, ny=ny_per_gpu, mask=mask, M_const=np.array([1 / 2000.0, 0.0, 0.0, 1 / 2000.0]))


SOLVER = "Tsit5"


def params(solver=None, DT=600.0, wind_min_squared=4.0, periodic_boundary=False):
    """example_00_minimal.jl:17-67 settings (T04_2D_reg_test uses the same), flattened by the host
    mirror of the reference API — no test or oracle module is involved on the b200 arm."""
    from picles_b200 import FetchRelations as FR
    from picles_b200.ParticleSystems import particle_waves_v5 as PW
    from picles_b200.params import make_params
    pars, cid, _ = PW.ODEParameters(r_g=0.85)
    ps = PW.particle_equations(None, None, γ=cid.γ, q=cid.q)
    sets = PW.ODESettings(Parameters=pars, log_energy_minimum=FR.MinimalWindsea(10, 10, DT)["lne"], saving_step=DT,
                          timestep=DT, total_time=6 * 86400.0, dt=1e-3, dtmin=1e-4, force_dtmin=True,
                          solver=solver or SOLVER, wind_min_squared=wind_min_squared)
    return make_params(sets, ps, FR.MinimalState(2, 2, DT), defaults=None, periodic_boundary=periodic_boundary, on_persist=False)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw = [], [], []
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)),
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (driver-measured copy bandwidth)"
    return 6650.0, "fallback 6.65 TB/s of B200_PROFILING.md (MEASURED_PEAKS.json absent)"


# ---------------------------------------------------------------------------------------
def _cpu_run(sample_n, steps, warmup, threads):
    """seed + warmup + `steps` timed model steps of a sample_n x sample_n homogeneous box on the CPU port"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))  # the CPU legs (and only they) use the tests' oracle builders
    from common import cartesian_grid, make_oracle
    g = cartesian_grid(sample_n, sample_n)
    o = make_oracle(g, params(), variant="omp", threads=threads)
    w = np.full((sample_n, sample_n), 10.0)  # one contiguous plane, passed for all four levels: nothing is copied per step
    o.seed(w, w)
    t = 0.0
    for _ in range(warmup):
        o.step(t, 600.0, w, w, w, w)
        t += 600.0
    t0 = time.perf_counter()
    for _ in range(steps):
        o.step(t, 600.0, w, w, w, w)
        t += 600.0
    dt = time.perf_counter() - t0
    c = o.counters()
    return dt, (sample_n - 2) ** 2, c["n_substeps"] / max(c["n_integrated"], 1)


def cpu_arm(steps, warmup, sample_n=None, threads=None, full_n=4096, budget_s=240.0):
    """The reference arm / cpu_baseline: the oracle port (OpenMP over particles in the ODE phase, serial
    canonical-order deposit) on all host cores.  sample_n = None: the TRUE workload (full_n x full_n, the same
    step indices) when a probe says warmup + steps fit `budget_s` on this host, else the largest power-of-two
    sample that does; the line says which."""
    threads = threads or os.cpu_count() or 1
    chosen = sample_n
    if chosen is None:
        probe_n = 512
        dt, n_act, _ = _cpu_run(probe_n, 1, 1, threads)
        per_particle = dt / n_act
        chosen = full_n
        while chosen > probe_n and per_particle * (chosen - 2) ** 2 * (steps + warmup + 1.5) > budget_s:
            chosen //= 2
    dt, n_active, sub = _cpu_run(chosen, steps, warmup, threads)
    what = "the full workload" if chosen == full_n else "a bounded sample of the workload"
    return dict(value=n_active * steps / dt, unit=UNIT, cores=threads, kind="port", sample_n=chosen, is_full=(chosen == full_n),
                sample=f"{chosen}x{chosen} homogeneous box ({what}; same physics/settings), steps {warmup + 1}..{warmup + steps}, "
                       f"oracle/picles_oracle.c with OpenMP over particles; {dt:.2f} s wall",
                ms_per_step=dt / steps * 1e3, substeps_per_particle_step=sub)


_REAL_STDOUT = None


def bind_rank_to_gpu_cpus(local_rank):
    """N > 1: one process per GPU, each kept on the CPUs next to ITS GPU (the NVML affinity mask of the device), so
    that the pinned staging buffers of the end-to-end leg are first touched on that GPU's NUMA node.  Unbound, half
    of eight ranks stage their 268 MB per step through the other socket (the e2e line of the 8-GPU run of round 2 sat
    at 86 % of the device-timed one, 95 % on one GPU).  Best effort: any failure leaves the process as it was.
    Returns the number of CPUs the process may run on afterwards, or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        try:
            import torch
            pr = torch.cuda.get_device_properties(local_rank)
            bus = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
            h = pynvml.nvmlDeviceGetHandleByPciBusId(bus)
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        before = len(os.sched_getaffinity(0))
        pynvml.nvmlDeviceSetCpuAffinity(h)
        after = len(os.sched_getaffinity(0))
        if after < 4:                       # a mask too small to be a socket: not what this is for
            pynvml.nvmlDeviceClearCpuAffinity(h)
            return None
        return {"cpus_before": before, "cpus_after": after}
    except Exception:
        return None


def claim_stdout():
    """Everything libraries print on fd 1 (NCCL's version banner, …) goes to stderr; the one
    JSON line is written to the real stdout by emit()."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


# At most this many nodes are dumped over all ranks: State (3 f64), particle u[5] (5 f64), the particle's clock t,
# step size dt, flags and status (f64 each) and the node index come to 104 B a node, 55 MB here, under the 64 MB the
# dump may take.
DUMP_NODES = 1 << 19


def dump_outputs(out_dir, eng, counters, max_nodes=DUMP_NODES, suffix=""):
    """--dump-outputs: what the timed path computed in its last step, as float64 .npy files in out_dir, so that two
    builds run with the same arguments (hence the same inputs) can be compared output for output.  State (3, n), the
    particles' u[5] (5, n), t, dt, flags and status (n each) at n nodes: every node of the strip when it has at most
    max_nodes, else a sample of max_nodes drawn with a fixed seed, its flat (row-major) indices in node_index (n).
    counters: the step's integer counters in picles_counters_t order, timings left out."""
    S = eng.state().reshape(3, -1)
    p = eng.particles()
    n = S.shape[1]
    idx = np.arange(n) if n <= max_nodes else np.sort(np.random.default_rng(0).choice(n, max_nodes, replace=False))
    arrays = {"state": S[:, idx], "particles_u": p["z"].reshape(5, -1)[:, idx],
              **{"particles_" + k: p[k].reshape(-1)[idx] for k in ("t", "dt", "flags", "status")},
              "node_index": idx,
              "counters": np.array([v for k, v in counters.items() if not k.startswith("ms_")])}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), np.ascontiguousarray(a, np.float64))


def growing_wind(x_nodes):
    """BASELINE configs[2] shape (tests/T04_2D_growing_decaying_winds.jl:126-132): calm foot, linear ramp in x,
    modulated in time so every step stages two different levels; on/off particle thresholds are in play"""
    Lx = float(x_nodes.max())
    x0 = 50.0 / 260.0 * Lx
    ramp = np.where(x_nodes < x0, 0.01, (x_nodes - x0) / (Lx - x0))
    return lambda t: (10.0 * ramp * (0.6 + 0.4 * np.sin(2 * np.pi * t / 7200.0)), 3.0 * ramp + 0.05)


def strip_parity_leg(dist, rank, world, local_rank, nx=512, rows_per_rank=256, steps=6):
    """N strips over NCCL (picles_step_strip: in-library exchange, reach all-reduce) against ONE domain on
    rank 0's GPU, same box, same winds: State, particle state and flags compared bit for bit after every
    step.  Growing/decaying winds: time-varying levels, particles seeded off, reseeds, both remesh branches."""
    from picles_b200.distributed import StripStepper
    from picles_b200.engine import B200Engine
    DT = 1200.0
    Ny = rows_per_rank * world
    P = params(DT=DT, wind_min_squared=2.0)
    mask = np.ones((Ny, nx), np.uint8)
    mask[:, 0] = mask[:, -1] = 3
    mask[0, :] = mask[-1, :] = 3
    Mc = np.array([1 / 4000.0, 0.0, 0.0, 1 / 4000.0])
    X = np.broadcast_to(np.arange(nx) * 4000.0, (Ny, nx))
    wind = growing_wind(X)
    full = lambda a: np.ascontiguousarray(np.broadcast_to(np.asarray(a, np.float64), (Ny, nx)))
    j0, j1 = rank * rows_per_rank, (rank + 1) * rows_per_rank
    eng = B200Engine(nx, Ny, 0, 0, mask[j0:j1], P, M_const=Mc, device=local_rank, j0=j0, ny_local=j1 - j0, halo=2)
    st = StripStepper(eng, rank, world, periodic_y=False)
    ref = B200Engine(nx, Ny, 0, 0, mask, P, M_const=Mc, device=local_rank) if rank == 0 else None
    u0, v0 = [full(a) for a in wind(0.0)]
    eng.seed(u0[j0:j1], v0[j0:j1])
    if ref is not None:
        ref.seed(u0, v0)
    t, bad, compared = 0.0, [], 0
    for k in range(steps):
        w = [full(a) for a in (*wind(t), *wind(t + DT))]
        st.step(t, DT, winds=[a[j0:j1] for a in w])
        if ref is not None:
            ref.step(t, DT, *w)
        t += DT
        pr = eng.particles()
        parts = [None] * world if rank == 0 else None
        dist.gather_object((eng.state(), pr["z"], pr["flags"], eng.counters()["n_active"]), parts, dst=0)
        if rank == 0:
            S = np.concatenate([q[0] for q in parts], axis=1)
            Z = np.concatenate([q[1] for q in parts], axis=1)
            F = np.concatenate([q[2] for q in parts], axis=0)
            rp = ref.particles()
            act = (rp["flags"] & 8) != 0
            same = lambda a, b: bool(np.all((a.view(np.uint64) == b.view(np.uint64)) | (np.isnan(a) & np.isnan(b))))
            if not same(ref.state(), S):
                bad.append(f"State after step {k + 1}")
            if not all(same(rp["z"][c][act], Z[c][act]) for c in range(5)):
                bad.append(f"particles after step {k + 1}")
            if not np.array_equal(rp["flags"][act], F[act]):
                bad.append(f"flags after step {k + 1}")
            if sum(q[3] for q in parts) != ref.counters()["n_active"]:
                bad.append(f"n_active after step {k + 1}")
            compared += 1
    off = int(((ref.particles()["flags"] & 9) == 8).sum()) if ref is not None else 0
    eng.close()
    if ref is not None:
        ref.close()
        return {"result": "bit-exact" if not bad else "MISMATCH: " + "; ".join(bad[:4]), "strips": world,
                "box": f"{nx}x{Ny} Cartesian, growing/decaying winds (BASELINE configs[2] shape), DT=1200 s, halo 2",
                "steps_compared": compared, "compared": ["State", "particle u[5]", "particle flags", "n_active"],
                "against": "the same box as ONE domain on rank 0's GPU (picles_step)", "transport": "NCCL inside the library (picles_step_strip)",
                "particles_seeded_off": off}
    return None


def strong_leg(dist, rank, world, local_rank, args, barrier_all):
    """BASELINE.md §2 row 3: the FIXED nx x nx box cut in `world` y-strips; the same box on ONE GPU is timed by
    rank 0 in the same process, the same step indices (the work per step falls over the first steps)."""
    import torch
    from picles_b200.distributed import StripStepper, strip_bounds
    from picles_b200.engine import B200Engine
    n = args.nx
    P = params()
    Wf = workload(n, n, 1, 0)
    j0, j1 = strip_bounds(n, world)[rank]
    eng = B200Engine(n, n, 0, 0, Wf["mask"][j0:j1], P, M_const=Wf["M_const"], device=local_rank, j0=j0, ny_local=j1 - j0,
                     halo=args.halo)
    st = StripStepper(eng, rank, world, periodic_y=False)
    eng.seed(10.0, 10.0)
    t = 0.0
    for _ in range(args.warmup):
        st.step(t, 600.0)
        t += 600.0
    barrier_all(eng)
    eng.timer_start()
    n_act, ms_adv = 0, []
    for _ in range(args.steps):
        st.step(t, 600.0)
        t += 600.0
        c = eng.counters()
        n_act += c["n_active"]
        ms_adv.append(c["ms_advance"])
    ms = eng.timer_stop()
    barrier_all(eng)
    tt = torch.tensor([ms, float(np.mean(ms_adv))], dtype=torch.float64, device="cuda")
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ww = torch.tensor([float(n_act)], dtype=torch.float64, device="cuda")
    dist.all_reduce(ww, op=dist.ReduceOp.SUM)
    rows = eng.halo_rows()[0]
    eng.close()
    one = None
    if rank == 0:
        e1 = B200Engine(n, n, 0, 0, Wf["mask"], P, M_const=Wf["M_const"], device=local_rank)
        e1.seed(10.0, 10.0)
        t1 = 0.0
        for _ in range(args.warmup):
            e1.step(t1, 600.0)
            t1 += 600.0
        e1.synchronize()
        e1.timer_start()
        n1 = 0
        for _ in range(args.steps):
            e1.step(t1, 600.0)
            t1 += 600.0
            n1 += e1.counters()["n_active"]
        ms1 = e1.timer_stop()
        e1.close()
        one = n1 / (ms1 * 1e-3)
    barrier_all(None)
    if rank != 0:
        return None
    ms_all, adv_all = tt.tolist()
    v = ww.item() / (ms_all * 1e-3)
    return {"scaling": "strong", "workload": f"the fixed {n}x{n} box of config.workload cut in {world} y-strips of {n // world} rows",
            "value": v, "unit": UNIT, "n_gpus": world, "ms_per_step": ms_all / args.steps, "ms_advance_max_rank": adv_all,
            "halo_rows_exchanged": rows, "value_1gpu_same_run": one, "ms_per_step_1gpu": 1e3 * (n - 2) ** 2 / one,
            "efficiency": v / (world * one), "target": 0.85,
            "timing": "CUDA events around the K steps on every rank, max over ranks; rank 0 then times the same box as one domain"}


def c5_grid(Nx=4320, Ny=3840, lat_min=-70.0, lat_max=89.0, R_earth=6.371e6):
    """BASELINE configs[4] shape: a synthetic tripolar grid (x periodic, y tripolar-north) with a rotated per-node
    projection kernel [cos/dx sin/dy; -sin/dx cos/dy] (TripolarGridMOM6.jl:448-459), the great-circle coefficient
    (spherical_grid_corrections.jl:13), a masked southern cap and four round land masses; masks by the host mirror
    of make_boundaries (mask_utils.jl:38-55).  The same grid as profiles/bench_configs.py "C5" (tests build theirs
    through the oracle's make_boundaries; tests/test_bench_contract.py holds the two bit-equal)."""
    from picles_b200.Architectures import N_Periodic, N_TripolarNorth
    from picles_b200.Grids.mask_utils import make_boundaries
    lon = -280.0 + (np.arange(Nx) + 0.5) * 360.0 / Nx
    lat = lat_min + (np.arange(Ny) + 0.5) * (lat_max - lat_min) / Ny
    LON, LAT = np.meshgrid(lon, lat)
    cap = np.clip((LAT - 60.0) / 30.0, 0.0, 1.0)
    angle = 40.0 * cap * np.sin(np.deg2rad(2 * (LON + 280.0)))
    dlon, dlat = 360.0 / Nx, (lat_max - lat_min) / Ny
    dx = np.maximum(R_earth * np.cos(np.deg2rad(LAT)) * np.deg2rad(dlon), 2000.0)
    dy = np.full_like(dx, R_earth * np.deg2rad(dlat))
    ca, sa = np.cos(angle * np.pi / 180), np.sin(angle * np.pi / 180)
    M = np.stack([ca / dx, sa / dy, -sa / dx, ca / dy]) * 1.2
    sgn = np.sign(LAT)
    pc = (sgn * np.minimum(sgn * np.tan(np.deg2rad(LAT)), 60.0)) / 6.3710e6
    ocean = np.ones((Ny, Nx), np.uint8)
    ocean[: max(2, Ny // 40), :] = 0
    yy, xx = np.mgrid[0:Ny, 0:Nx]
    for cx, cy, r in ((0.2, 0.45, 0.08), (0.55, 0.6, 0.1), (0.8, 0.3, 0.06), (0.5, 0.97, 0.04)):
        ocean[((xx - cx * Nx) / Nx) ** 2 + ((yy - cy * Ny) / Ny) ** 2 < r * r] = 0
    mask = np.ascontiguousarray(make_boundaries(ocean.T, N_Periodic(Nx), N_TripolarNorth(Ny)).T.astype(np.uint8))
    return dict(Nx=Nx, Ny=Ny, bx=1, by=2, mask=mask, M=np.ascontiguousarray(M), pc=np.ascontiguousarray(pc))


def strong_c5_leg(dist, rank, world, local_rank, steps, warmup, halo=6):
    """BASELINE configs[4]: "T03_PIC_tripolar_land with synthetic land mask at high resolution, 8-GPU y-strip
    partition" — ONE 4320x3840 tripolar + land grid cut in `world` y-strips (strong scaling), time-varying winds
    resident before each timed step, halo exchange over NCCL inside the library.  Land and the small cells near
    the pole make rows unequal, so the strips are cut by MEASURED cost: a calibration run on equal strips (per-strip
    kernel times, per-row reach) first.  (A second pass that re-cut by the step times measured on the
    re-cut strips bought nothing — 80.9 % on 8 GPUs either way, 96.5 -> 95.5 % on 2: a strip's step time is mostly the slowest
    strip's advance, DESIGN.md §5 — and was dropped.)  Rank 0 then times the same grid as one domain on its GPU, same steps."""
    import torch
    from picles_b200.distributed import (StripStepper, overlapped_step_estimate, row_cost_measured, strip_bounds,
                                         strip_bounds_overlapped, strip_bounds_weighted)
    from picles_b200.engine import B200Engine
    g = c5_grid()
    Nx, Ny = g["Nx"], g["Ny"]
    DT = 1200.0
    P = params(DT=DT, periodic_boundary=True)
    wind = lambda t: (15.0, -10.0 * np.cos(5 * t / (3600 * 2 * np.pi)))  # tests/T03_PIC_tripolar_aqua.jl:67-68

    def run(bounds, nwarm, nsteps, one_domain=False):
        j0, j1 = (0, Ny) if one_domain else bounds[rank]
        eng = B200Engine(Nx, Ny, g["bx"], g["by"], g["mask"][j0:j1], P, M=g["M"][:, j0:j1], pc=g["pc"][j0:j1], device=local_rank,
                         j0=j0, ny_local=j1 - j0, halo=0 if one_domain else halo)
        st = None if one_domain else StripStepper(eng, rank, world, periodic_y=False)
        loc = lambda x: np.ascontiguousarray(np.broadcast_to(np.asarray(x, np.float64), (j1 - j0, Nx)))
        eng.seed(*[loc(x) for x in wind(0.0)])
        t, rows, ms_total = 0.0, [], 0.0
        for k in range(nwarm + nsteps):
            eng.upload_winds(*[loc(x) for x in (*wind(t), *wind(t + DT))])
            eng.synchronize()
            if not one_domain:
                dist.barrier()
                torch.cuda.synchronize()
            eng.timer_start()
            if one_domain:
                eng.step(t, DT)
            else:
                st.step(t, DT)
            ms = eng.timer_stop()
            t += DT
            if k >= nwarm:
                rows.append(eng.counters())
                ms_total += ms
        out = dict(ms=ms_total, active=sum(r["n_active"] for r in rows), adv=float(np.mean([r["ms_advance"] for r in rows])),
                   prj=float(np.mean([r["ms_project"] for r in rows])), failed=sum(r["n_failed"] for r in rows), rows=j1 - j0,
                   row_reach=eng.row_reach().tolist(), halo_rows=eng.halo_rows()[0])
        eng.close()
        return out

    eq = strip_bounds(Ny, world)
    cal = run(eq, warmup, 2)
    allc = [None] * world
    dist.all_gather_object(allc, cal)
    active_rows = ((g["mask"] == 1) | (g["mask"] == 3)).sum(axis=1)
    reach_rows = np.concatenate([np.asarray(c["row_reach"]) for c in allc])
    adv_cost, gat_cost = row_cost_measured(active_rows, Nx, reach_rows, eq, [c["adv"] for c in allc], [c["prj"] for c in allc],
                                           split=True)
    # the overlapped step of a strip costs the SLOWEST strip's advance plus its own gather (measured on 2 and 8 GPUs,
    # DESIGN.md §5), so the cut evens out the advance rather than the summed cost, unless that piles gather on one strip
    bounds, lam, est = strip_bounds_overlapped(adv_cost, gat_cost, world, min_rows=max(halo, 1))
    est_sum = overlapped_step_estimate(adv_cost, gat_cost, strip_bounds_weighted(adv_cost + gat_cost, world, min_rows=max(halo, 1)))
    mine = run(bounds, warmup, steps)
    parts = [None] * world if rank == 0 else None
    dist.gather_object(mine, parts, dst=0)
    one = run(None, warmup, steps, one_domain=True) if rank == 0 else None
    dist.barrier()
    if rank != 0:
        return None
    ms_max = max(p["ms"] for p in parts)
    v = sum(p["active"] for p in parts) / (ms_max * 1e-3)
    v1 = one["active"] / (one["ms"] * 1e-3)
    return {"scaling": "strong", "workload": f"tripolar + land {Nx}x{Ny} (synthetic; BASELINE configs[4]) cut in {world} y-strips by measured cost, "
                                             f"DT=1200 s, u=15, v=-10 cos(5t/(3600 2pi)), periodic_boundary model, halo {halo} rows",
            "value": v, "unit": UNIT, "n_gpus": world, "steps": steps, "ms_per_step": ms_max / steps,
            "partition": {"objective": "max_r(advance) + max_r(gather) from the calibration run's per-row costs", "blend": lam,
                          "estimate_ms": est, "estimate_ms_if_summed_cost_were_balanced": est_sum},
            "rows_per_rank": [p["rows"] for p in parts], "ms_per_step_per_rank": [p["ms"] / steps for p in parts],
            "ms_advance_per_rank": [p["adv"] for p in parts], "ms_project_remesh_per_rank": [p["prj"] for p in parts],
            "halo_rows_exchanged": max(p["halo_rows"] for p in parts), "failed": sum(p["failed"] for p in parts),
            "value_1gpu_same_run": v1, "ms_per_step_1gpu": one["ms"] / steps, "efficiency": v / (world * v1), "target": 0.85,
            "timing": "CUDA events around every step (winds uploaded before, barrier between steps), summed per rank, max over ranks; "
                      "rank 0 then times the same grid as one domain"}


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--nx", type=int, default=4096)
    ap.add_argument("--ny", type=int, default=4096, help="rows per GPU")
    ap.add_argument("--halo", type=int, default=2)
    ap.add_argument("--cpu-sample", type=int, default=None,
                    help="side of the box the CPU port is timed on (default: the full workload when it fits the time budget, "
                         "else the largest power-of-two sample that does; the cpu_baseline of the b200 arm always samples 1024)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra-legs", action="store_true", help="N > 1: skip the strong-scaling and strip-parity legs")
    ap.add_argument("--solver", default="Tsit5", choices=["Tsit5", "DP5", "AutoTsit5"],
                    help="ODESettings.solver; AutoTsit5 = the reference's default AutoTsit5(Rosenbrock23()): the same "
                         "arithmetic as Tsit5 on this workload (the stiffness monitor never fires) plus the monitor")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed steps computed in their last step to DIR/<name>.npy (see dump_outputs; "
                         "with N > 1 every rank writes its strip as <name>_rank<r>.npy)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the CUDA path: not with --impl reference")
    global SOLVER
    SOLVER = args.solver
    if args.warmup < 3:
        log("warmup raised to 3 (timing rules)")
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    config = {"workload": f"homogeneous box {args.nx}x{args.ny * max(world, 1)} Cartesian (BASELINE configs[1]: "
                          f"T04_2D_reg_test_large_grid/bench06 scaled), dx=dy=2km, u=v=10 m/s, DT=600 s, "
                          f"{args.solver} abstol=1e-4 reltol=1e-3 dt=1e-3 dtmin=1e-4 force_dtmin",
              "nx": args.nx, "ny_per_gpu": args.ny, "parallelism": f"y-strips x{max(world, 1)}",
              "l2_policy": "inputs_exceed_l2 (3.3 GB of per-node planes per GPU >> 126 MB L2)"}

    if args.impl == "reference":
        if rank != 0:
            return 0
        # the reference's CPU path on ONE strip's workload (the per-GPU unit of the weak-scaling arm): nx x ny
        cb = cpu_arm(args.steps, args.warmup, args.cpu_sample, full_n=args.nx)
        if not cb["is_full"]:
            config["workload"] += f" [this arm: timed on a {cb['sample_n']}x{cb['sample_n']} sample of it, see cpu_baseline.sample]"
        line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config, "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0, "sample_is_full_workload": cb["is_full"],
                "note": "Julia is not installed on this image: the reference's CPU path is timed as its C port "
                        "(oracle/), all host threads; BASELINE.md quotes 4-7e4 particle-steps/s for the Julia original. "
                        "One host runs one box whatever --gpus says (the reference has no domain decomposition)"}
        emit(line)
        return 0

    # ---- our arm ------------------------------------------------------------------------------
    # The library build() compiled, unless a source has changed since: then its sources are compiled into a
    # temporary directory and that library is timed, so the numbers are always those of the sources as they stand
    # and the tree (possibly read-only) is left as build() left it.
    import build_lib
    if build_lib.needs_build():
        import tempfile
        from picles_b200 import _abi
        lib_dir = tempfile.TemporaryDirectory(prefix="picles_b200_")  # removed when main() returns
        log(f"libpicles_b200.so is missing or older than its sources: building them into {lib_dir.name}")
        _abi.LIB_PATH = build_lib.build(out=os.path.join(lib_dir.name, "libpicles_b200.so"))
    dist = None
    affinity = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        affinity = bind_rank_to_gpu_cpus(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
    from picles_b200.engine import B200Engine
    W = workload(args.nx, args.ny, world, rank)
    P = params()
    halo = args.halo if world > 1 else 0
    eng = B200Engine(W["Nx"], W["Ny"], 0, 0, W["mask"], P, M_const=W["M_const"], device=local_rank, j0=W["j0"],
                     ny_local=W["ny"], halo=halo)
    n_nodes = W["Nx"] * W["ny"]
    stepper = None
    if world > 1:
        from picles_b200.distributed import StripStepper
        stepper = StripStepper(eng, rank, world, periodic_y=False)

    fp64_peak = eng.measure_fp64_peak()
    hbm_meas = eng.measure_hbm_copy(2048)
    hbm_peak, hbm_src = measured_peaks()

    def do_step(t, host_ptrs=None):
        if stepper is None:
            if host_ptrs is None:
                eng.step(t, 600.0)
            else:
                eng.step_raw(t, 600.0, None, None, host_ptrs[0], host_ptrs[1])
        else:
            stepper.step(t, 600.0, host_ptrs)

    def barrier(e=eng):
        if e is not None:
            e.synchronize()
        if dist is not None:
            dist.barrier()
            import torch
            torch.cuda.synchronize()

    eng.seed(10.0, 10.0)
    t = 0.0
    for _ in range(args.warmup):
        do_step(t)
        t += 600.0

    # ---- timed region A: inputs resident in HBM -----------------------------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    per_step = []
    hist = np.zeros(48, np.int64)
    barrier()
    launches0 = eng.launch_count()
    eng.timer_start()
    for _ in range(args.steps):
        do_step(t)
        t += 600.0
        per_step.append(eng.counters())
    ms_total = eng.timer_stop()
    launches = eng.launch_count() - launches0  # counted by the library where it launches; timer_stop launches nothing
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    hist += eng.attempt_histogram()            # of the last timed step
    n_active = sum(c["n_active"] for c in per_step)  # particle-steps of this rank in the region
    if args.dump_outputs:                      # before the legs below step the same engine further
        dump_outputs(args.dump_outputs, eng, per_step[-1], DUMP_NODES // world, f"_rank{rank}" if world > 1 else "")

    # ---- the reference's default solver on the same workload ---------------------------------
    # ODESettings.solver defaults to AutoTsit5(Rosenbrock23()) (particle_waves_v5.jl:47).  On this
    # workload its stiffness monitor never fires (n_stiff_switches = 0, tested), so its results are
    # the Tsit5 results bit for bit; the monitor-carrying kernel is timed here for the record.
    auto_variant = None
    if world == 1 and args.solver == "Tsit5" and not args.no_e2e:
        eng2 = B200Engine(W["Nx"], W["Ny"], 0, 0, W["mask"], params("AutoTsit5"),
                          M_const=W["M_const"], device=local_rank)
        eng2.seed(10.0, 10.0)
        t2 = 0.0
        for _ in range(args.warmup):
            eng2.step(t2, 600.0)
            t2 += 600.0
        k2 = min(args.steps, 5)
        rows2 = []
        eng2.synchronize()
        eng2.timer_start()
        for _ in range(k2):
            eng2.step(t2, 600.0)
            t2 += 600.0
            rows2.append(eng2.counters())
        ms2 = eng2.timer_stop()
        auto_variant = {"solver": "AutoTsit5(Rosenbrock23())", "steps": k2,
                        "value": sum(r["n_active"] for r in rows2) / (ms2 * 1e-3), "unit": UNIT, "ms_per_step": ms2 / k2,
                        "ms_advance": float(np.mean([r["ms_advance"] for r in rows2])),
                        "n_stiff_switches": int(sum(r["n_stiff_switches"] for r in rows2)),
                        "n_stiff_attempts": int(sum(r["n_stiff_attempts"] for r in rows2))}
        eng2.close()

    # ---- timed region B: end to end through host buffers ----------------------------
    e2e = None
    e2e_store = None
    if not args.no_e2e:
        import torch
        # pinned host staging of the step's inputs: wind at t+DT evaluated on the host mesh
        hu = torch.full((W["ny"], W["Nx"]), 10.0, dtype=torch.float64).pin_memory()
        hv = torch.full((W["ny"], W["Nx"]), 10.0, dtype=torch.float64).pin_memory()
        ptrs = (ctypes.c_void_p(hu.data_ptr()), ctypes.c_void_p(hv.data_ptr()))
        do_step(t, ptrs)
        t += 600.0
        barrier()
        t0 = time.perf_counter()
        eng.timer_start()
        n_e2e = 0
        for _ in range(args.steps):
            do_step(t, ptrs)           # H2D of u,v at t+DT (2 planes), step, D2H of the counters
            t += 600.0
            _ = eng.energy_sum()       # D2H read of the step's result: sum of the energy plane
            n_e2e += eng.counters()["n_active"]
        ms_e2e = eng.timer_stop()
        barrier()
        wall_e2e = (time.perf_counter() - t0) * 1e3
        ms_e2e = max(ms_e2e, wall_e2e)  # host-side work (API, staging) counts end to end
        e2e = dict(ms=ms_e2e, n=n_e2e, h2d=2 * n_nodes * 8, d2h=ctypes.sizeof(ctypes.c_double) * 1024 + 88)

        # ---- the same with the step's full result brought back: run!(...; cash_store=true) pushes State to the
        # host after every step (src/Simulations/run.jl:104-112).  picles_snapshot_begin stages State on the compute
        # stream and copies it to pinned host memory on its own stream while the next step integrates; the copy of
        # the last step is waited for inside the timed region.
        snap = eng.pinned_state_buffer()
        do_step(t, ptrs)
        t += 600.0
        eng.snapshot_begin(snap)
        eng.snapshot_wait()
        barrier()
        t0 = time.perf_counter()
        eng.timer_start()
        n_st = 0
        for _ in range(args.steps):
            do_step(t, ptrs)
            t += 600.0
            eng.snapshot_begin(snap)   # waits for the previous step's copy first: one snapshot in flight
            n_st += eng.counters()["n_active"]
        eng.snapshot_wait()
        ms_st = eng.timer_stop()
        barrier()
        ms_st = max(ms_st, (time.perf_counter() - t0) * 1e3)
        e2e_store = dict(ms=ms_st, n=n_st, checksum=float(snap[0].sum()))

    # ---- timed region C: end to end with a device-resident wind mesh (wind ingestion) ----------
    # Same workload; the wind comes from a gridded field kept on the device (9 x 9 x 3 knots of
    # u = v = 10 m/s, the reference's LinearInterpolation((x,y,t), U, Periodic()) closure) and is
    # sampled at the nodes by k_wind_sample every step: no wind bytes cross PCIe.
    e2e_mesh = None
    if not args.no_e2e:
        xw = np.linspace(-1.0e4, 2000.0 * W["Nx"] + 1.0e4, 9)
        yw = np.linspace(-1.0e4, 2000.0 * W["Ny"] + 1.0e4, 9)
        tw = np.array([0.0, 1.0e6, 2.0e6])
        Uw = np.full((3, 9, 9), 10.0)
        nx_ = np.broadcast_to(np.arange(W["Nx"]) * 2000.0, (W["ny"], W["Nx"]))
        ny_ = np.broadcast_to(((W["j0"] + np.arange(W["ny"])) * 2000.0)[:, None], (W["ny"], W["Nx"]))
        eng.set_wind_mesh(xw, yw, tw, Uw, Uw, nx_, ny_)
        lo, hi = (stepper.lo, stepper.hi) if stepper is not None else (-1, -1)
        eng.step_wind_mesh(t, 600.0, 0, lo, hi)
        t += 600.0
        barrier()
        t0 = time.perf_counter()
        eng.timer_start()
        n_mesh = 0
        for _ in range(args.steps):
            eng.step_wind_mesh(t, 600.0, 0, lo, hi)
            t += 600.0
            _ = eng.energy_sum()
            n_mesh += eng.counters()["n_active"]
        ms_mesh = eng.timer_stop()
        barrier()
        ms_mesh = max(ms_mesh, (time.perf_counter() - t0) * 1e3)
        e2e_mesh = dict(ms=ms_mesh, n=n_mesh, ms_sample=eng.measure_wind_sample(t, 20))

    # ---- reduce over ranks: max time, sum of work ------------------------------------
    if dist is not None:
        import torch
        tt = torch.tensor([ms_total, e2e["ms"] if e2e else 0.0, e2e_mesh["ms"] if e2e_mesh else 0.0,
                           e2e_store["ms"] if e2e_store else 0.0], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ww = torch.tensor([float(n_active), float(e2e["n"]) if e2e else 0.0, float(e2e_mesh["n"]) if e2e_mesh else 0.0,
                           float(e2e_store["n"]) if e2e_store else 0.0, float(launches)], dtype=torch.float64, device="cuda")
        dist.all_reduce(ww, op=dist.ReduceOp.SUM)
        ms_total, ms_e2e_all, ms_mesh_all, ms_store_all = tt.tolist()
        n_active_all, n_e2e_all, n_mesh_all, n_store_all, launches_all = ww.tolist()
    else:
        ms_e2e_all = e2e["ms"] if e2e else 0.0
        ms_mesh_all = e2e_mesh["ms"] if e2e_mesh else 0.0
        ms_store_all = e2e_store["ms"] if e2e_store else 0.0
        n_active_all, n_e2e_all = float(n_active), float(e2e["n"]) if e2e else 0.0
        n_mesh_all = float(e2e_mesh["n"]) if e2e_mesh else 0.0
        n_store_all = float(e2e_store["n"]) if e2e_store else 0.0
        launches_all = float(launches)

    # ---- N > 1: the strong-scaling record and NCCL strip parity (untimed by the headline) ----------
    strong = parity = strong_c5 = None
    if dist is not None and not args.no_extra_legs:
        eng.close()
        eng = None
        strong = strong_leg(dist, rank, world, local_rank, args, barrier)
        parity = strip_parity_leg(dist, rank, world, local_rank)
        strong_c5 = strong_c5_leg(dist, rank, world, local_rank, min(args.steps, 5), args.warmup)
        barrier(None)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    # ---- rooflines from the live CUDA-event times of the timed region ------------------
    ms_adv = float(np.mean([c["ms_advance"] for c in per_step]))
    ms_prj = float(np.mean([c["ms_project"] for c in per_step]))
    ncu = ncu_record()
    std_size = (args.nx, args.ny) == (4096, 4096)  # the size the committed ncu captures were taken at
    nk = ncu.get("kernels", {}) if std_size else {}
    ncu_src = {"file": "profiles/ncu_metrics.json", "library_commit": ncu.get("commit"), "captured_with": ncu.get("command")}
    rhs = float(np.mean([c["n_rhs"] for c in per_step]))
    att = float(np.mean([c["n_substeps"] + c["n_rejects"] for c in per_step]))
    integ = float(np.mean([c["n_integrated"] for c in per_step]))
    dep = float(np.mean([c["n_deposited"] for c in per_step]))
    flops = rhs * F_RHS + att * F_ATTEMPT + integ * F_INITDT + dep * F_DEPOSIT
    adv_tf = flops / (ms_adv * 1e-3) / 1e12
    prj_gbs = n_nodes * B_PROJECT_REMESH / (ms_prj * 1e-3) / 1e9
    roofline = {"kernel": "k_advance", "bound": "fp64", "achieved": adv_tf, "peak": fp64_peak,
                "unit": "TFLOP/s", "frac": adv_tf / fp64_peak, "traffic": nk.get("k_advance", {}).get("dram_bytes"),
                "peak_source": "DFMA-chain microbenchmark run in this process (picles_measure_fp64_peak); "
                               "MEASURED_PEAKS.json has no FP64 entry",
                "flop_model": {"F_RHS": F_RHS, "F_ATTEMPT": F_ATTEMPT, "F_INITDT": F_INITDT, "F_DEPOSIT": F_DEPOSIT,
                               "rhs_per_launch": rhs, "attempts_per_launch": att},
                "ncu_fp64_pipe_active_pct": nk.get("k_advance", {}).get("fp64_pipe_pct"), "ncu_source": ncu_src,
                "ms_per_launch": ms_adv, "share_of_step": ms_adv / (ms_adv + ms_prj)}
    roofline_hbm = [
        {"kernel": "k_project_remesh", "bound": "hbm", "achieved": prj_gbs, "peak": hbm_peak, "unit": "GB/s",
         "frac": prj_gbs / hbm_peak, "traffic": nk.get("k_project_remesh", {}).get("dram_bytes"), "ncu_source": ncu_src,
         "bytes_per_node": B_PROJECT_REMESH, "nodes_per_launch": n_nodes, "ms_per_launch": ms_prj,
         "share_of_step": ms_prj / (ms_adv + ms_prj), "peak_source": hbm_src},
    ]

    value = n_active_all / (ms_total * 1e-3)
    nz = np.nonzero(hist)[0]
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
            "roofline": roofline, "roofline_hbm": roofline_hbm,
            "measured_here": {"fp64_dfma_tflops": fp64_peak, "hbm_copy_gbs": hbm_meas},
            "clocks": clocks,
            # counted by the library at every kernel launch (picles_launch_count), summed over ranks, resident-input region:
            # per step and rank k_advance + k_project_remesh; on strips the advance is three launches (two boundary blocks
            # first, then the interior) plus k_halo_pack and k_halo_unpack (NCCL's own kernels are not ours and not counted)
            "gpu_launches": int(launches_all),
            "substeps_per_particle_step": float(np.mean([c["n_substeps"] / max(c["n_integrated"], 1) for c in per_step])),
            "max_attempts": int(max(c["max_attempts"] for c in per_step)),
            "attempt_histogram_last_step": {str(int(k)): int(hist[k]) for k in nz},
            "rejects": int(sum(c["n_rejects"] for c in per_step)),
            "failed": int(sum(c["n_failed"] for c in per_step))}
    if world > 1:
        line["rank0_cpu_affinity"] = affinity if affinity else "unchanged (NVML affinity not applied)"
    if e2e:
        line["e2e"] = {"value": n_e2e_all / (ms_e2e_all * 1e-3), "unit": UNIT, "h2d_bytes_per_step": e2e["h2d"],
                       "d2h_bytes_per_step": e2e["d2h"], "ms_per_step": ms_e2e_all / args.steps,
                       "api": "picles_step through the C ABI with pinned host wind buffers + picles_state_energy_sum"}
    if e2e_store:
        line["e2e_store"] = {"value": n_store_all / (ms_store_all * 1e-3), "unit": UNIT, "h2d_bytes_per_step": e2e["h2d"],
                             "d2h_bytes_per_step": 3 * n_nodes * 8 + 88, "ms_per_step": ms_store_all / args.steps,
                             "state_checksum": e2e_store["checksum"],
                             "api": "picles_step with pinned host wind buffers + picles_snapshot_begin/wait of the whole State "
                                    "into pinned host memory every step (run!(...; cash_store=true), run.jl:104-112)"}
    if auto_variant:
        line["default_solver_variant"] = auto_variant
    if e2e_mesh:
        # the same metric with the wind ingested on the device; k_wind_sample: 16 B of node
        # coordinates in + 16 B of wind out per node (the mesh itself is L2-resident)
        gbs = n_nodes * 32 / (e2e_mesh["ms_sample"] * 1e-3) / 1e9
        line["e2e_wind_mesh"] = {"value": n_mesh_all / (ms_mesh_all * 1e-3), "unit": UNIT, "h2d_bytes_per_step": 0,
                                 "d2h_bytes_per_step": e2e["d2h"] if e2e else 0, "ms_per_step": ms_mesh_all / args.steps,
                                 "api": "picles_step_wind_mesh (wind sampled on the device from a resident wind mesh) "
                                        "+ picles_state_energy_sum"}
        line["roofline_hbm"].append({"kernel": "k_wind_sample", "note": "k_wind_timeblend (mesh-sized, ~3 us) + k_wind_sample, timed as a pair",
                                     "bound": "hbm", "achieved": gbs, "peak": hbm_peak,
                                     "unit": "GB/s", "frac": gbs / hbm_peak,
                                     "traffic": (nk.get("k_wind_sample_x4") or nk.get("k_wind_sample", {})).get("dram_bytes"), "ncu_source": ncu_src, "bytes_per_node": 32,
                                     "nodes_per_launch": n_nodes, "ms_per_launch": e2e_mesh["ms_sample"],
                                     "share_of_step": e2e_mesh["ms_sample"] / (ms_adv + ms_prj + e2e_mesh["ms_sample"]),
                                     "peak_source": hbm_src})
    if strong:
        line["strong"] = strong
    if parity:
        line["strip_parity"] = parity
    if strong_c5:
        line["strong_c5"] = strong_c5
    if not args.no_cpu_baseline:
        cb = cpu_arm(min(args.steps, 3), args.warmup, 1024 if args.cpu_sample is None else args.cpu_sample)
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
    emit(line)
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
