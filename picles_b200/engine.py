"""B200Engine — thin object wrapper over the C ABI of libpicles_b200.so.

One engine = one `picles_t` handle = one GPU = one y-strip of the global grid.  All
arrays cross the boundary as host numpy buffers (row-major (ny, Nx) == the reference's
column-major (Nx, ny), i fastest); nothing here computes — every method is one or two
C-ABI calls, and every failure of the library raises PiclesError.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from ._abi import ERR_NAMES, PiclesCounters, PiclesError, PiclesParams, load_library


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class B200Engine:
    def __init__(self, Nx, Ny, bx, by, mask, params: PiclesParams, M=None, M_const=None, pc=None, device=0,
                 j0=0, ny_local=None, halo=0, metric=None, members=1):
        """mask/M/pc cover the rows this strip owns: (ny_local, Nx), (4, ny_local, Nx), (ny_local, Nx).
        metric = dict(dx, dy, angle_dx, lat[, R_earth]) of (ny_local, Nx) planes: the per-node
        kernel and great-circle coefficient are then formed on the device (picles_set_grid_metric).
        members = E > 1: an ensemble of E models on this grid (picles_set_members), stepped together.  Every
        per-node array then gains a member axis in front of its node axes: winds (E, ny, Nx), State (3, E, ny, Nx),
        particle planes (5, E, ny, Nx) and (E, ny, Nx); the grid arrays above stay single planes."""
        self.lib = load_library()
        self.Nx, self.Ny = int(Nx), int(Ny)
        self.j0 = int(j0)
        self.ny = int(Ny if ny_local is None else ny_local)
        self.halo = int(halo)
        self.device = int(device)
        self.h = C.c_void_p()
        self._check(self.lib.picles_create(C.byref(self.h), int(device)), None)
        self.members = int(members)
        # node-plane shape of every per-node array: (ny, Nx), or (E, ny, Nx) for an ensemble
        self._nodes = (self.ny, self.Nx) if self.members == 1 else (self.members, self.ny, self.Nx)
        if self.members != 1:
            self._check(self.lib.picles_set_members(self.h, self.members))
        mask = np.ascontiguousarray(np.asarray(mask, np.uint8).reshape(self.ny, self.Nx))
        Mp = np.ascontiguousarray(np.asarray(M, np.float64).reshape(4, self.ny, self.Nx)) if M is not None else None
        Mc = np.ascontiguousarray(np.asarray(M_const, np.float64).reshape(4)) if M_const is not None else None
        pcp = np.ascontiguousarray(np.asarray(pc, np.float64).reshape(self.ny, self.Nx)) if pc is not None else None
        if metric is not None:
            raw = [np.ascontiguousarray(np.asarray(metric[k], np.float64).reshape(self.ny, self.Nx))
                   for k in ("dx", "dy", "angle_dx", "lat")]
            self._check(self.lib.picles_set_grid_metric(self.h, self.Nx, self.Ny, int(bx), int(by), self.j0, self.ny,
                                                        self.halo, _ptr(mask), *[_ptr(a) for a in raw],
                                                        float(metric.get("R_earth", 6.3710e6))))
        else:
            self._check(self.lib.picles_set_grid(self.h, self.Nx, self.Ny, int(bx), int(by), self.j0, self.ny,
                                                 self.halo, _ptr(mask), _ptr(Mp), _ptr(Mc), _ptr(pcp)))
        self.params = params
        self._check(self.lib.picles_set_params(self.h, C.byref(params)))

    # -- plumbing ------------------------------------------------------------------
    def _check(self, rc, h="self"):
        if rc != 0:
            hh = self.h if h == "self" else None
            msg = self.lib.picles_last_error(hh)
            raise PiclesError(f"{ERR_NAMES.get(rc, rc)}: {msg.decode() if msg else ''}")

    def close(self):
        if getattr(self, "h", None) is not None and self.h:
            self.lib.picles_snapshot_wait(self.h)
            self.lib.picles_destroy(self.h)
            self.h = None
            for p in getattr(self, "_pinned", []):
                self.lib.picles_host_free(p)
            self._pinned = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _wind(self, a):
        if a is None:
            return None
        a = np.asarray(a, np.float64)
        if a.shape != self._nodes:
            a = np.broadcast_to(a, self._nodes)
        return np.ascontiguousarray(a)

    # -- the path ------------------------------------------------------------------
    def seed(self, u0, v0):
        a, b = self._wind(u0), self._wind(v0)
        self._check(self.lib.picles_seed(self.h, _ptr(a), _ptr(b)))

    def step(self, t, DT, u_t=None, v_t=None, u_t1=None, v_t1=None):
        """State .= 0; time_step!  —  None reuses the winds already on the device."""
        a = [self._wind(x) for x in (u_t, v_t, u_t1, v_t1)]
        self._check(self.lib.picles_step(self.h, float(t), float(DT), *[_ptr(x) for x in a]))

    def set_wind_midlevels(self, u_mid=(), v_mid=()):
        """intermediate wind levels of the NEXT step at t + k*DT/(n+1), k = 1..n (n <= 3): the wind
        at a stage time is then the polynomial through all n+2 levels instead of the linear rule."""
        n = len(u_mid)
        if n == 0:
            self._check(self.lib.picles_set_wind_midlevels(self.h, 0, None, None))
            return
        um = np.ascontiguousarray(np.stack([self._wind(x) for x in u_mid]))
        vm = np.ascontiguousarray(np.stack([self._wind(x) for x in v_mid]))
        self._check(self.lib.picles_set_wind_midlevels(self.h, n, _ptr(um), _ptr(vm)))

    # wind ingestion: gridded winds resident on the device
    def set_wind_mesh(self, xw, yw, tw, U, V, node_x, node_y):
        """LinearInterpolation((xw, yw, tw), U, extrapolation_bc=Periodic()) kept on the device.
        U, V: (nt, ny_w, nx_w) (== Julia U[ix, iy, it]); node_x, node_y: (ny, Nx) coordinates of
        this strip's nodes (grid.data.x, grid.data.y)."""
        f = lambda a: np.ascontiguousarray(np.asarray(a, np.float64))
        xw, yw, tw, U, V = f(xw), f(yw), f(tw), f(U), f(V)
        if U.shape != (tw.size, yw.size, xw.size) or V.shape != U.shape:
            raise ValueError(f"U, V must have shape (nt, ny, nx) = {(tw.size, yw.size, xw.size)}")
        nx_, ny_ = self._wind(node_x), self._wind(node_y)
        self._check(self.lib.picles_set_wind_mesh(self.h, xw.size, yw.size, tw.size, _ptr(xw), _ptr(yw), _ptr(tw),
                                                  _ptr(U), _ptr(V), _ptr(nx_), _ptr(ny_)))

    def set_member_wind_meshes(self, xw, yw, tw, U, V, node_x, node_y):
        """an ensemble's wind meshes, one per member on shared knots (picles_set_member_wind_meshes).
        U, V: (E, nt, ny_w, nx_w), member m's mesh as set_wind_mesh takes it; node_x, node_y: (ny, Nx), shared by
        the members.  seed/stage/step_wind_mesh and sample_wind_mesh then sample every member on the device."""
        f = lambda a: np.ascontiguousarray(np.asarray(a, np.float64))
        xw, yw, tw, U, V = f(xw), f(yw), f(tw), f(U), f(V)
        shape = (self.members, tw.size, yw.size, xw.size)
        if U.shape != shape or V.shape != shape:
            raise ValueError(f"U, V must have shape (E, nt, ny, nx) = {shape}, not {U.shape} and {V.shape}")
        plane = lambda a: np.ascontiguousarray(np.broadcast_to(np.asarray(a, np.float64), (self.ny, self.Nx)))
        nx_, ny_ = plane(node_x), plane(node_y)
        self._check(self.lib.picles_set_member_wind_meshes(self.h, xw.size, yw.size, tw.size, _ptr(xw), _ptr(yw),
                                                           _ptr(tw), _ptr(U), _ptr(V), _ptr(nx_), _ptr(ny_)))

    def sample_wind_mesh(self, t):
        """(u, v) of the mesh at this strip's nodes at time t: (ny, Nx) each, or (E, ny, Nx) on an ensemble"""
        # an ensemble with member meshes writes E planes: the buffers are sized for them before the call
        u, v = np.empty(self._nodes), np.empty(self._nodes)
        self._check(self.lib.picles_sample_wind_mesh(self.h, float(t), _ptr(u), _ptr(v)))
        return u, v

    def seed_wind_mesh(self, t0=0.0):
        self._check(self.lib.picles_seed_wind_mesh(self.h, float(t0)))

    def step_wind_mesh(self, t, DT, n_mid=0, lo=-1, hi=-1):
        """one model step with every wind level sampled on the device from the resident mesh"""
        self._check(self.lib.picles_step_wind_mesh(self.h, float(t), float(DT), int(n_mid), int(lo), int(hi)))

    def stage_wind_mesh(self, t, DT, n_mid=0):
        """sample every wind level of [t, t+DT] from the resident mesh into the device planes
        (the phase-split calls then run without any wind upload)"""
        self._check(self.lib.picles_stage_wind_mesh(self.h, float(t), float(DT), int(n_mid)))

    def step_raw(self, t, DT, pu_t=None, pv_t=None, pu_t1=None, pv_t1=None):
        """Same as step() with raw host pointers (ints), e.g. of pinned torch tensors."""
        self._check(self.lib.picles_step(self.h, float(t), float(DT), pu_t, pv_t, pu_t1, pv_t1))

    # phase-split form (multi-strip)
    def upload_winds(self, u_t=None, v_t=None, u_t1=None, v_t1=None):
        a = [self._wind(x) for x in (u_t, v_t, u_t1, v_t1)]
        self._check(self.lib.picles_upload_winds(self.h, *[_ptr(x) for x in a]))

    def upload_winds_raw(self, pu_t=None, pv_t=None, pu_t1=None, pv_t1=None):
        self._check(self.lib.picles_upload_winds(self.h, pu_t, pv_t, pu_t1, pv_t1))

    def step_advance(self, t, DT):
        self._check(self.lib.picles_step_advance(self.h, float(t), float(DT)))

    def halo_buffers(self):
        p = [C.c_void_p() for _ in range(4)]
        nb = C.c_int64()
        self._check(self.lib.picles_halo_buffers(self.h, *[C.byref(x) for x in p], C.byref(nb)))
        return [x.value for x in p], nb.value

    def halo_rows(self):
        """(rows exchanged with each y-neighbour, most the strip can exchange)"""
        a, b = C.c_int(), C.c_int()
        self._check(self.lib.picles_halo_rows(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def halo_widen(self, rows):
        """exchange at least `rows` rows from now on (never narrowed)"""
        self._check(self.lib.picles_halo_widen(self.h, int(rows)))

    def set_global_reach(self, reach):
        """the all-reduced reach of this step (host-driven exchange): lets the gather check the halo width exactly"""
        self._check(self.lib.picles_set_global_reach(self.h, int(reach)))

    def halo_pack(self):
        self._check(self.lib.picles_halo_pack(self.h))

    def halo_unpack(self):
        self._check(self.lib.picles_halo_unpack(self.h))

    def step_project_remesh(self, t, DT):
        self._check(self.lib.picles_step_project_remesh(self.h, float(t), float(DT)))

    def halo_exchange(self, lo=-1, hi=-1):
        """pack -> ncclSend/ncclRecv with the ranks owning the rows below/above -> unpack"""
        self._check(self.lib.picles_halo_exchange(self.h, int(lo), int(hi)))

    def step_strip(self, t, DT, u_t=None, v_t=None, u_t1=None, v_t1=None, lo=-1, hi=-1):
        a = [self._wind(x) for x in (u_t, v_t, u_t1, v_t1)]
        self._check(self.lib.picles_step_strip(self.h, float(t), float(DT), *[_ptr(x) for x in a], int(lo), int(hi)))

    def step_strip_raw(self, t, DT, pu_t, pv_t, pu_t1, pv_t1, lo=-1, hi=-1):
        self._check(self.lib.picles_step_strip(self.h, float(t), float(DT), pu_t, pv_t, pu_t1, pv_t1, int(lo), int(hi)))

    def synchronize(self):
        self._check(self.lib.picles_synchronize(self.h))

    def reach(self):
        r = C.c_int32()
        self._check(self.lib.picles_get_reach(self.h, C.byref(r)))
        return r.value

    def row_reach(self):
        """per owned row: the largest reach (cells) of the deposits its particles wrote in the last step"""
        r = np.empty(self._nodes[:-1], np.int32)
        self._check(self.lib.picles_get_row_reach(self.h, _ptr(r)))
        return r

    # -- accessors -----------------------------------------------------------------
    def state(self):
        S = np.empty((3,) + self._nodes)
        self._check(self.lib.picles_get_state(self.h, _ptr(S)))
        return S

    def set_state(self, S):
        S = np.ascontiguousarray(np.asarray(S, np.float64).reshape((3,) + self._nodes))
        self._check(self.lib.picles_set_state(self.h, _ptr(S)))

    def particles(self):
        sh = self._nodes
        z = np.empty((5,) + sh)
        t, dt = np.empty(sh), np.empty(sh)
        flags = np.empty(sh, np.uint8)
        status = np.empty(sh, np.int32)
        self._check(self.lib.picles_get_particles(self.h, _ptr(z), _ptr(t), _ptr(dt), _ptr(flags), _ptr(status)))
        return dict(z=z, t=t, dt=dt, flags=flags, status=status)

    def metric(self):
        """(M, pc) in use: M (4, ny, Nx) planes M11, M12, M21, M22; pc (ny, Nx)."""
        M = np.empty((4, self.ny, self.Nx))
        pc = np.empty((self.ny, self.Nx))
        self._check(self.lib.picles_get_metric(self.h, _ptr(M), _ptr(pc)))
        return M, pc

    def make_boundaries(self, ocean, bx, by):
        """make_boundaries(mask, Nx, Ny) on the device: ocean (Ny, Nx) 0/1 -> total mask 0..3."""
        o = np.ascontiguousarray(np.asarray(ocean, np.uint8))
        out = np.empty_like(o)
        self._check(self.lib.picles_make_boundaries(self.h, o.shape[1], o.shape[0], int(bx), int(by), _ptr(o), _ptr(out)))
        return out

    def fields(self):
        """derived output fields on the device: dict(Hs=4*sqrt(e), c_x, c_y) of (ny, Nx)."""
        out = [np.empty(self._nodes) for _ in range(3)]
        self._check(self.lib.picles_get_fields(self.h, *[_ptr(a) for a in out]))
        return dict(Hs=out[0], c_x=out[1], c_y=out[2])

    def pinned_state_buffer(self):
        """(3, ny, Nx) (an ensemble: (3, E, ny, Nx)) float64 array in pinned host memory (freed with the engine)."""
        size = 3 * int(np.prod(self._nodes))
        nbytes = size * 8
        p = C.c_void_p()
        self._check(self.lib.picles_host_alloc(C.byref(p), nbytes), None)
        self._pinned = getattr(self, "_pinned", []) + [p]
        buf = (C.c_double * size).from_address(p.value)
        return np.frombuffer(buf, dtype=np.float64).reshape((3,) + self._nodes)

    def snapshot_begin(self, S_host):
        """start an asynchronous copy of State into S_host (3, ny, Nx); stepping may continue."""
        assert S_host.dtype == np.float64 and S_host.flags["C_CONTIGUOUS"] and S_host.size == 3 * int(np.prod(self._nodes))
        self._check(self.lib.picles_snapshot_begin(self.h, _ptr(S_host)))

    def snapshot_wait(self):
        self._check(self.lib.picles_snapshot_wait(self.h))

    def checkpoint(self):
        """the complete state of the path as one uint8 array (picles_checkpoint_save)"""
        n = C.c_int64()
        self._check(self.lib.picles_checkpoint_size(self.h, C.byref(n)))
        blob = np.empty(n.value, np.uint8)
        self._check(self.lib.picles_checkpoint_save(self.h, _ptr(blob), n.value))
        return blob

    def restore(self, blob):
        """resume from a checkpoint() of an engine with the same grid and parameters"""
        blob = np.ascontiguousarray(blob, np.uint8)
        self._check(self.lib.picles_checkpoint_load(self.h, _ptr(blob), blob.size))

    def counters(self):
        c = PiclesCounters()
        self._check(self.lib.picles_get_counters(self.h, C.byref(c)))
        return c.as_dict()

    def attempt_histogram(self, nbins=48):
        """particles that integrated in the last step by Runge-Kutta attempts taken (last bin: that many or more)"""
        h = np.zeros(int(nbins), np.int64)
        self._check(self.lib.picles_get_attempt_histogram(self.h, _ptr(h), int(nbins)))
        return h

    def launch_count(self):
        """kernels launched by the library in this process so far"""
        return int(self.lib.picles_launch_count())

    def solver_state(self):
        """AutoSwitch state per particle (AutoTsit5): run length of the stiffness test, +64 while
        Rosenbrock23 is the current algorithm"""
        a = np.empty(self._nodes, np.int8)
        self._check(self.lib.picles_get_solver_state(self.h, _ptr(a)))
        return a

    def set_accumulate(self, on: bool):
        """False: run! semantics (State zeroed before the step); True: bare time_step!."""
        self._check(self.lib.picles_set_option(self.h, 1, int(bool(on))))

    def zero_state(self):
        self._check(self.lib.picles_zero_state(self.h))

    def copy_dev(self, dst, src, nbytes):
        self._check(self.lib.picles_copy_dev(self.h, dst, src, int(nbytes)))

    def timer_start(self):
        self._check(self.lib.picles_timer_start(self.h))

    def timer_stop(self):
        ms = C.c_double()
        self._check(self.lib.picles_timer_stop(self.h, C.byref(ms)))
        return ms.value

    def selftest_math(self, seed=1, iters=4096):
        out = (C.c_int64 * 6)()
        self._check(self.lib.picles_selftest_math(self.h, int(seed), int(iters), out))
        names = ("n_div", "flagged_div", "mismatch_div", "n_sqrt", "flagged_sqrt", "mismatch_sqrt")
        return dict(zip(names, [int(v) for v in out]))

    def measure_fp64_peak(self):
        v = C.c_double()
        self._check(self.lib.picles_measure_fp64_peak(self.h, C.byref(v)))
        return v.value

    def measure_hbm_copy(self, mib=2048):
        v = C.c_double()
        self._check(self.lib.picles_measure_hbm_copy(self.h, int(mib), C.byref(v)))
        return v.value

    def measure_wind_sample(self, t=0.0, reps=20):
        """ms per wind level (time blend + sampler, or their member forms) over this strip (CUDA events)"""
        v = C.c_double()
        self._check(self.lib.picles_measure_wind_sample(self.h, float(t), int(reps), C.byref(v)))
        return v.value

    def energy_sum(self):
        s = C.c_double()
        self._check(self.lib.picles_state_energy_sum(self.h, C.byref(s)))
        return s.value

    def member_energy_sums(self):
        """energy_sum() of every member, (E,): bit for bit what a single-member engine with that member's State returns"""
        s = np.empty(self.members)
        self._check(self.lib.picles_member_energy_sums(self.h, _ptr(s)))
        return s
