"""`Simulation`, `run!`, `initialize_simulation!`, `reset_simulation!`, `init_particles!` of
`src/Simulations/{simulation,run}.jl` for models on the B200 architecture.  (Python has no
`!` in identifiers: run! -> run, init_particles! -> init_particles, ...)"""
from __future__ import annotations

import logging
import time
import warnings

import numpy as np

from ..Operators.TimeSteppers import time_step

log = logging.getLogger("picles_b200")


class EmptyStore:
    def __init__(self, iteration=1):
        self.iteration = iteration


class CashStore:
    """storing.jl:15-18 — in-memory list of State copies."""

    def __init__(self, store=None, iteration=1):
        self.store = [] if store is None else store
        self.iteration = iteration


class Simulation:
    """simulation.jl:12-28,52-99."""

    def __init__(self, model, Δt, verbose=True, stop_iteration=float("inf"), stop_time=float("inf"),
                 wall_time_limit=float("inf")):
        if stop_iteration == float("inf") and stop_time == float("inf") and wall_time_limit == float("inf"):
            warnings.warn("This simulation will run forever as stop iteration = stop time = wall time limit = Inf.")
        self.model = model
        self.timestepper = None
        self.Δt = float(Δt)
        self.stop_iteration = float(stop_iteration)
        self.stop_time = float(stop_time)
        self.wall_time_limit = float(wall_time_limit)
        self.diagnostics = {}
        self.output_writers = {}
        self.callbacks = {}
        self.run_wall_time = 0.0
        self.running = False
        self.initialized = False
        self.verbose = verbose
        self.store = EmptyStore(1)
        self.store_itereation = 0


def _is_1d(model):
    return getattr(model, "dims", 2) == 1


def init_particles(model, defaults=None, verbose=False):
    """init_particles!(model; defaults): SeedParticle for every node with the wind at t = 0
    (run.jl:199-247; the Abstract1DModel method: run.jl:268-302) — one picles_seed / picles1d_seed call."""
    if _is_1d(model):
        from ..Models.WaveGrowthModels1D import init_particles_1D
        init_particles_1D(model, defaults=defaults, verbose=verbose)
        return
    if model._gridded_winds is not None:
        model.engine.seed_wind_mesh(0.0)
    else:
        u0, v0 = model._wind_planes(0.0)
        model.engine.seed(u0, v0)
    model._wind_level_time = 0.0
    model._seeded = True


def initialize_simulation(sim):
    """initialize_simulation!, run.jl:130-146."""
    init_particles(sim.model, defaults=sim.model.ODEdefaults, verbose=sim.verbose)
    if sim.model.clock.iteration != 0:
        sim.model.clock.iteration = 0
        sim.model.clock.time = 0.0
    if not _is_1d(sim.model):
        sim.model._wind_level_time = 0.0 if sim.model.clock.time == 0.0 else None
    sim.initialized = True


def reset_simulation(sim):
    """reset_simulation!, run.jl:154-181."""
    sim.running = False
    sim.run_wall_time = 0.0
    sim.model.clock.iteration = 0
    sim.model.clock.time = 0.0
    init_particles(sim.model, defaults=sim.model.ODEdefaults, verbose=sim.verbose)
    if not _is_1d(sim.model):
        sim.model.engine.zero_state()
    sim.initialized = True


def run(sim, store=False, pickup=False, cash_store=False, debug=False):
    """run!(sim; store, cash_store, debug), run.jl:36-122: while stop_time >= clock.time:
    State .= 0; time_step!; optional stores.  ('>=' ⇒ floor(stop/Δt)+1 steps.)"""
    if store:
        raise NotImplementedError("StateStore (HDF5) output is outside the B200 path; use cash_store")
    t0 = time.perf_counter_ns()
    if not sim.initialized:
        initialize_simulation(sim)
    sim.run_wall_time = 0.0
    sim.running = sim.stop_time >= sim.model.clock.time
    if not sim.running:
        log.info("stop_time exceeded, run not executed")
    eng = sim.model.engine
    # CashStore pushes are asynchronous snapshots where the engine offers them (B200Engine):
    # the device-to-host copy of step n overlaps the integration of step n+1
    snap = hasattr(eng, "snapshot_begin") and cash_store
    pending = None

    def collect():
        nonlocal pending
        if pending is not None:
            eng.snapshot_wait()
            # (3, [E,] ny, Nx) -> ([E,] Nx, Ny, 3) like model.State
            sim.store.store.append(np.array(np.moveaxis(pending, 0, -1).swapaxes(-2, -3), copy=True))
            sim.store.iteration += 1
            pending = None

    if cash_store:
        sim.store = CashStore([], 1)
        sim.store.iteration += 1
        sim.store.store.append(np.array(sim.model.State, copy=True))
        if snap:
            stage = eng.pinned_state_buffer()
    while sim.running:
        if _is_1d(sim.model):
            from ..Models.WaveGrowthModels1D import time_step_1D
            time_step_1D(sim.model, sim.Δt, debug=debug)   # State .= 0 is part of picles1d_step
        else:
            time_step(sim.model, sim.Δt, debug=debug, zero_state_first=True)
        if debug and len(sim.model.FailedCollection) > 0:
            log.info("debug mode: found failed particles: %s; break", sim.model.FailedCollection)
            break
        if cash_store:
            if snap:
                collect()
                eng.snapshot_begin(stage)
                pending = stage
            else:
                sim.store.store.append(np.array(sim.model.State, copy=True))
                sim.store.iteration += 1
        sim.running = sim.stop_time >= sim.model.clock.time
        if sim.verbose:
            log.info("%s", sim.model.clock)
    collect()
    sim.run_wall_time += 1e-9 * (time.perf_counter_ns() - t0)
