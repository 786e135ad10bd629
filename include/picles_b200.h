/*
 * picles_b200.h — C ABI of the B200-native PiCLES per-timestep particle-in-cell path.
 *
 * The reference (mochell/PiCLES, pure Julia) has no FFI; the seam this library cuts
 * is "everything `init_particles!` and `time_step!` do" (SURVEY.md §8b):
 *
 *   picles_seed   replaces  init_particles!          src/Simulations/run.jl:199-247
 *                           SeedParticle             src/Operators/core_2D.jl:434-488
 *   picles_step   replaces  State .= 0               src/Simulations/run.jl:75-79
 *                           time_step!               src/Operators/TimeSteppers.jl:109-166
 *                             advance!               src/Operators/mapping_2D.jl:118-243
 *                             ParticleToNode!        src/Operators/mapping_2D.jl:59-73
 *                             remesh!/NodeToParticle! src/Operators/mapping_2D.jl:250-356
 *   picles_set_grid         grid.data / grid.stats   src/Grids/CartesianGrid.jl:26-136,
 *                                                    src/Grids/TripolarGridMOM6.jl:288-459
 *   picles_set_params       ODESettings/ODEParameters src/ParticleSystems/particle_waves_v5.jl:34-75,184-196
 *                           WaveGrowth2D kwargs      src/Models/WaveGrowthModels2D.jl:194-345
 *
 * Conventions
 *   - all entry points return 0 on success, a negative picles_status_t on failure;
 *     picles_last_error() returns a message for the most recent failure on a handle.
 *   - array arguments are caller-owned HOST pointers (column-major, i fastest,
 *     Float64 / Int32 / UInt8) unless the name ends in `_dev`; they are copied during
 *     the call.  Device memory is owned by the opaque handle.
 *   - one handle = one GPU = one y-strip of the global grid (a single strip for 1 GPU).
 *   - calls are synchronous unless stated, and a handle must be driven by one host
 *     thread at a time.  No callbacks into the host language.
 *   - per-particle integration failures are status codes (picles_get_particles),
 *     not call failures — mirroring the reference's "push to FailedCollection and
 *     carry on" (mapping_2D.jl:151-170).
 *   - there is NO CPU fallback: every entry point that computes fails with
 *     PICLES_ERR_CUDA when no sm_100-class device is usable.
 */
#ifndef PICLES_B200_H
#define PICLES_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PICLES_ABI_VERSION 3

typedef struct picles_handle picles_t;

typedef enum {
    PICLES_OK = 0,
    PICLES_ERR_ARG = -1,      /* bad argument / call order */
    PICLES_ERR_CUDA = -2,     /* CUDA runtime error or no usable device */
    PICLES_ERR_ALLOC = -3,    /* device allocation failed */
    PICLES_ERR_HALO = -4,     /* particle reach exceeded the halo width */
    PICLES_ERR_STATE = -5,    /* grid/params/seed missing */
    PICLES_ERR_COMM = -6      /* NCCL unavailable or a collective failed */
} picles_status_t;

/* axis boundary types: custom_structures.jl:51-61 */
enum { PICLES_BND_NONPERIODIC = 0, PICLES_BND_PERIODIC = 1, PICLES_BND_TRIPOLAR_NORTH = 2 };
/* total mask values: mask_utils.jl:26-30 */
enum { PICLES_MASK_LAND = 0, PICLES_MASK_OCEAN = 1, PICLES_MASK_LAND_BOUNDARY = 2, PICLES_MASK_GRID_BOUNDARY = 3 };
/* solver ids: ODESettings.solver (particle_waves_v5.jl:47) */
enum {
    PICLES_SOLVER_TSIT5 = 0,
    PICLES_SOLVER_DP5 = 1,
    /* AutoTsit5(Rosenbrock23()), the ODESettings default: Tsit5 with OrdinaryDiffEq's AutoSwitch
       stiffness monitor (Hairer II p. 22 eigenvalue estimate, stiff for more than 10 consecutive
       attempts -> Rosenbrock23 with an automatic-differentiation Jacobian, dt doubled; back after
       more than 3 non-stiff attempts, dt halved).  On every configuration where the monitor never
       fires it is Tsit5, bit for bit. */
    PICLES_SOLVER_AUTOTSIT5 = 2
};

/* per-particle status bits (picles_get_particles) */
enum {
    PICLES_PST_OK = 0,
    PICLES_PST_MAXITERS = 1,      /* iter > maxiters: integrator stopped */
    PICLES_PST_DTMIN = 2,         /* dt <= dtmin without force_dtmin */
    PICLES_PST_UNSTABLE = 4,      /* NaN in u during integration */
    PICLES_PST_NAN_RESET = 8,     /* advance!: NaN  -> reseed (mapping_2D.jl:196-209) */
    PICLES_PST_INF_RESET = 16,    /* advance!: Inf  -> reseed (mapping_2D.jl:211-220) */
    PICLES_PST_EMAX_CLAMP = 32    /* advance!: lne > log_energy_maximum (mapping_2D.jl:222-233) */
};

/* particle flag bits (picles_get_particles `flags`) */
enum {
    PICLES_PF_ON = 1,             /* ParticleInstance2D.on */
    PICLES_PF_BOUNDARY = 2,       /* ParticleInstance2D.boundary */
    PICLES_PF_DT_RESET = 4,       /* auto_dt_reset! pending (evaluated lazily at the next advance) */
    PICLES_PF_ACTIVE = 8          /* member of ocean_points (iterated by time_step!) */
};

/*
 * Flattened ODESettings + ODEParameters + WaveGrowth2D keyword arguments.
 * The host language computes the derived constants exactly as the reference does
 * (IDConstants / magic_fractions / e_T_func, particle_waves_v5.jl:87-128,271) and
 * FetchRelations.MinimalState (FetchRelations.jl:412-415); the library never
 * re-derives them, so oracle and device see identical inputs.
 */
typedef struct {
    /* ODEParameters (particle_waves_v5.jl:184-196) */
    double r_g;
    double C_alpha;
    double C_varphi;
    double C_e;
    double g;            /* carried for API parity; the RHS uses the 9.81 default of
                            c_g_conversions_vector (particle_waves_v5.jl:281,504) */
    /* particle_equations constants (particle_waves_v5.jl:393-394) */
    double p;            /* magic_fractions(q)[1] */
    double q;
    double n;            /* magic_fractions(q)[3] */
    double e_T;          /* e_T_func(γ,p,q,n; c_β,c_D,c_e,c_α) */
    /* term switches of particle_equations (particle_waves_v5.jl:382-390) */
    int32_t propagation;
    int32_t input;
    int32_t dissipation;
    int32_t peak_shift;
    int32_t direction;
    /* ODESettings (particle_waves_v5.jl:34-75) */
    int32_t solver;
    double abstol;
    double reltol;
    double dt;           /* initial substep after seeding */
    double dtmin;
    double dtmax;        /* OrdinaryDiffEq default: tspan length = total_time */
    int32_t force_dtmin;
    int32_t adaptive;    /* must be 1 */
    int64_t maxiters;
    double log_energy_minimum;  /* carried; unused by the 2-D path (SURVEY B-7) */
    double log_energy_maximum;
    double wind_min_squared;
    double seed_timescale;      /* ODESettings.timestep: fetch-law time scale at seeding (run.jl:223) */
    /* WaveGrowth2D */
    double minimal_state[2];    /* [E_min, |m|^2_min]  (WaveGrowthModels2D.jl:241-246) */
    int32_t has_defaults;       /* 0: ODEinit_type == "wind_sea" (ODEdefaults === nothing) */
    double defaults[5];         /* ParticleDefaults lne, c̄_x, c̄_y, x, y */
    int32_t periodic_boundary;  /* the MODEL kwarg: selects ocean_points (WaveGrowthModels2D.jl:256-270) */
    /* quirk switches (SURVEY Appendix B) */
    int32_t on_persist;         /* 0: `on` frozen at seed (as the reference runs, B-1); 1: as intended */
    int32_t nan_eest_rejects;   /* a trial step whose stages overflow has EEst = NaN and is rejected; what the reject rule
                                   dt /= min(1/qmin, EEst^beta1/gamma) makes of it depends on OrdinaryDiffEq's (unpinned)
                                   version.  0: exact powers — NaN^beta1 = NaN, Julia's min propagates it, dt = NaN, the
                                   integrator ends with DtNaN (status PICLES_PST_UNSTABLE).  1: `fastpow` / FastPower's
                                   `fastpower` — they read the NaN bit pattern as a large finite number, so the step is
                                   rejected by the full factor 1/qmin and the integration goes on */
} picles_params_t;

/* per-step device counters (summed over this handle's strip) */
typedef struct {
    int64_t n_active;        /* particles iterated (|ocean_points| of this strip) */
    int64_t n_integrated;    /* particles that took the step! branch */
    int64_t n_substeps;      /* accepted RK substeps */
    int64_t n_rejects;       /* rejected RK substeps */
    int64_t n_rhs;           /* RHS evaluations (incl. fsal resets and dt resets) */
    int64_t n_reseed_advance;/* off->on reseeds in advance! */
    int64_t n_fixups;        /* NaN/Inf/e_max fix-ups in advance! */
    int64_t n_failed;        /* maxiters / dtmin / unstable stops */
    int64_t n_deposited;     /* particles projected onto the grid */
    int64_t n_remesh_A;      /* node -> particle (enough energy) */
    int64_t n_remesh_B;      /* wind-sea reseed (interior) */
    int64_t n_remesh_C;      /* wind-sea reseed (boundary) */
    int64_t n_remesh_D;      /* switched off */
    int32_t reach;           /* max |node offset| of any deposit corner, in cells */
    int32_t max_attempts;    /* max RK attempts of any particle this step */
    double ms_advance;       /* CUDA-event times of the three kernels of the last step */
    double ms_project;
    double ms_remesh;
    int64_t n_stiff_switches;/* AutoTsit5: switches Tsit5 -> Rosenbrock23 this step */
    int64_t n_stiff_attempts;/* AutoTsit5: Rosenbrock23 attempts this step (accepted + rejected) */
} picles_counters_t;

/* ---- lifecycle --------------------------------------------------------- */
int picles_abi_version(void);
/* device_id: CUDA ordinal.  Fails with PICLES_ERR_CUDA when no device is usable. */
int picles_create(picles_t** h, int device_id);
int picles_destroy(picles_t* h);
const char* picles_last_error(picles_t* h);

/* ---- ensembles: many members on one grid, stepped together ------------------------------
 * A handle may carry `members` models that share the grid (mask, projection kernel, great-circle
 * coefficient, boundary types) and picles_params_t; each member has its own winds, particles,
 * deposit records and State.  All members step with the same t and dt_model in the same kernel
 * launches: one step launches the kernels one model does, whatever the member count.
 *
 * Layout rule: every per-node plane argument grows from ny_local*Nx to members*ny_local*Nx values,
 * member slowest — a plane of E members is E single-member planes back to back.  This holds for the
 * winds of picles_seed / picles_step / picles_upload_winds / picles_set_wind_midlevels, for
 * picles_get_state / picles_set_state (3 planes of E*ny_local*Nx), picles_get_particles,
 * picles_get_solver_state, picles_get_fields, picles_snapshot_begin, picles_state_dev /
 * picles_wind_dev and picles_get_row_reach (E*ny_local rows).  The grid arguments of
 * picles_set_grid* (mask, M, pc_coef, the raw metric) and picles_get_metric stay single planes.
 * Counters and the attempt histogram are summed over the members; reach and max_attempts are the
 * maximum over the members; picles_state_energy_sum sums every member.
 *
 * With members > 1 these return PICLES_ERR_ARG: a strip cut (j0 != 0, ny_local != Ny or halo != 0),
 * members*ny_local*Nx >= 2^31, picles_comm_init / picles_comm_destroy, picles_halo_*,
 * picles_step_strip, picles_set_wind_mesh (one mesh for every member) and picles_checkpoint_*; and,
 * until picles_set_member_wind_meshes has given every member its mesh, picles_seed_wind_mesh /
 * picles_stage_wind_mesh / picles_step_wind_mesh / picles_sample_wind_mesh /
 * picles_measure_wind_sample.
 */
/* before picles_set_grid* (PICLES_ERR_STATE after it); 1..65535, default 1 */
int picles_set_members(picles_t* h, int members);
/* per member (members values): picles_state_energy_sum of that member's State, by the same two-stage
   reduction, so sums[m] equals what a single-member handle with member m's State returns, bit for bit */
int picles_member_energy_sums(picles_t* h, double* sums);

/* ---- setup ------------------------------------------------------------- */
/*
 * Global grid shape and boundary types plus this handle's y-strip.
 *   Nx, Ny        global node counts            (grid.stats.Nx.N, grid.stats.Ny.N)
 *   bx, by        PICLES_BND_*                  (typeof(grid.stats.Nx / Ny))
 *   j0, ny_local  first global row (0-based) and row count owned by this handle
 *   halo          rows of neighbour particle records kept on each side (0 for 1 strip)
 *   mask          uint8 total mask of rows [j0-halo, j0+ny_local+halo) clipped/wrapped
 *                 by the caller: (ny_local + 2*halo) * Nx values; halo rows outside a
 *                 non-periodic domain are ignored
 *   M             per-node projection kernel, 4 planes (M11,M12,M21,M22) of ny_local*Nx,
 *                 or NULL with M_const != NULL for a uniform kernel (Cartesian)
 *   pc_coef       great-circle coefficient per node (ny_local*Nx) or NULL (=0)
 */
int picles_set_grid(picles_t* h, int Nx, int Ny, int bx, int by,
                    int j0, int ny_local, int halo,
                    const uint8_t* mask, const double* M, const double* M_const,
                    const double* pc_coef);
/*
 * Same as picles_set_grid for grids with a per-node metric (MOM6GridMesh), but the
 * projection kernel and the great-circle coefficient are formed ON THE DEVICE from the raw
 * mesh planes of this strip (ny_local*Nx each, host):
 *   M  = [cos a/dx  sin a/dy; -sin a/dx  cos a/dy],  a = angle_dx*pi/180
 *                                  ProjetionKernel(Gi, stats), TripolarGridMOM6.jl:448-459
 *   pc = sign(lat)*min(sign(lat)*tand(lat), 60)/R_earth
 *                                  SphericalPropagationCorrection, spherical_grid_corrections.jl:13,49-51
 * with the deterministic sin/cos/tand of pmath_trig.h (bit-identical to the CPU oracle).
 */
int picles_set_grid_metric(picles_t* h, int Nx, int Ny, int bx, int by,
                           int j0, int ny_local, int halo, const uint8_t* mask,
                           const double* dx, const double* dy, const double* angle_dx,
                           const double* lat, double R_earth);
/* read back the metric in use: M = 4 planes (M11,M12,M21,M22) of ny_local*Nx, pc = 1 plane */
int picles_get_metric(picles_t* h, double* M, double* pc);
/*
 * make_boundaries(mask, Nx, Ny) (mask_utils.jl:14-22,38-55) on the device for a whole grid:
 * ocean[Nx*Ny] (1 ocean / 0 land) -> total[Nx*Ny] with PICLES_MASK_* values.  bx/by: only
 * PICLES_BND_NONPERIODIC axes get their edges marked 3.  Needs no grid to be set.
 */
int picles_make_boundaries(picles_t* h, int Nx, int Ny, int bx, int by,
                           const uint8_t* ocean, uint8_t* total);
int picles_set_params(picles_t* h, const picles_params_t* p);

/* ---- the path ---------------------------------------------------------- */
/* init_particles!: wind at t = 0 on this strip's nodes (ny_local*Nx each). */
int picles_seed(picles_t* h, const double* u0, const double* v0);

/*
 * One model step on this strip:  State .= 0 ; advance! ; ParticleToNode! ; remesh!.
 * u_t/v_t: wind at the pre-step clock time t, u_t1/v_t1 at t+dt_model (ny_local*Nx
 * each, host).  Any of them may be NULL to reuse what is already on the device
 * (u_t NULL: the previous step's t1 level becomes this step's t level).
 * Single-strip handles run the whole step; multi-strip handles must use the
 * phase-split calls below so the host can exchange halos in between.
 */
int picles_step(picles_t* h, double t, double dt_model,
                const double* u_t, const double* v_t,
                const double* u_t1, const double* v_t1);

/* Phase-split form of picles_step (same arithmetic):                          */
int picles_upload_winds(picles_t* h, const double* u_t, const double* v_t,
                        const double* u_t1, const double* v_t1);
/*
 * Intermediate wind levels of the NEXT step (wind ingestion, SURVEY.md §8f-3).  The reference
 * calls the wind closures u(x,y,t), v(x,y,t) at every Runge-Kutta stage time
 * (particle_waves_v5.jl:489-495); this library integrates against wind levels staged per model
 * step.  With the two levels t, t+dt_model the wind is linear in time over the step (exact for
 * steady winds and for gridded winds that are linear between their time knots,
 * tests/T03_PIC_tripolar_realistic.jl:61-73).  n_mid > 0 adds the levels at
 * t + k*dt_model/(n_mid+1), k = 1..n_mid: the wind at a stage time is then the polynomial of
 * degree n_mid+1 through all levels, which converges to the closure value for smooth winds
 * (measured in tests/test_wind_levels.py).  u_mid / v_mid: n_mid planes of ny_local*Nx each,
 * host.  The levels are consumed by the next picles_step / picles_step_strip /
 * picles_step_advance call; n_mid = 0 clears them.
 */
#define PICLES_WIND_MID_MAX 3
int picles_set_wind_midlevels(picles_t* h, int n_mid, const double* u_mid, const double* v_mid);
int picles_step_advance(picles_t* h, double t, double dt_model);   /* async on the handle's stream */
/* device pointers + byte count of the packed halo rows to send to / receive from the
   lower (j0-1) and upper (j0+ny_local) neighbour; valid after picles_step_advance */
int picles_halo_buffers(picles_t* h, void** send_lo_dev, void** send_hi_dev,
                        void** recv_lo_dev, void** recv_hi_dev, int64_t* nbytes);
int picles_halo_pack(picles_t* h);     /* records -> send buffers (async) */
int picles_halo_unpack(picles_t* h);   /* recv buffers -> halo rows (async) */
int picles_step_project_remesh(picles_t* h, double t, double dt_model);
int picles_synchronize(picles_t* h);
/* reach (cells) of the last advance on this strip; the caller all-reduces(max) it */
int picles_get_reach(picles_t* h, int32_t* reach);
/* the same per owned row (ny_local values): the largest reach of any deposit written by the particles of that row in
   the last step — what sizes the gather's window tile by tile, and a measured input for cutting strips by cost */
int picles_get_row_reach(picles_t* h, int32_t* reach_rows);

/* ---- multi-GPU: y-strips, one handle per GPU/process ------------------------- */
/*
 * The reference has no domain decomposition (SURVEY.md §8e); strips are this library's
 * own.  Between the advance and the gather each strip sends the deposit records of its
 * first / last `halo` rows to its y-neighbours, so every GPU sums its own nodes in the
 * reference's canonical order and the result does not depend on the GPU count.
 *   picles_comm_unique_id   rank 0 creates the NCCL id (128 bytes); the host broadcasts it
 *                           with whatever it has (MPI.jl, Distributed.jl, torch.distributed)
 *   picles_comm_init        every rank joins; nccl_path = libnccl.so.2 to dlopen, NULL =
 *                           the copy already in the process, else the default soname
 *   picles_halo_exchange    pack -> ncclSend/ncclRecv (one group) -> unpack, asynchronous on
 *                           the handle's stream; lo_rank / hi_rank = ranks owning the rows
 *                           below / above this strip, -1 for none (domain edge)
 *   picles_step_strip       picles_step for a strip, exchange included
 */
#define PICLES_COMM_ID_BYTES 128
int picles_comm_unique_id(char* id128, const char* nccl_path);
int picles_comm_init(picles_t* h, const char* id128, int rank, int nranks, const char* nccl_path);
int picles_comm_destroy(picles_t* h);
int picles_halo_exchange(picles_t* h, int lo_rank, int hi_rank);
/*
 * How many rows travel.  The `halo` of picles_set_grid* is the number of rows exchanged to begin with;
 * the record planes of a strip hold room for rows_max = min(15, ny_local), the widest window the gather
 * supports.  The reference enforces no CFL limit (ParticleInCell.jl:58-71), so a step may deposit further
 * than the rows exchanged: the gather then changes nothing and
 *   - picles_step_strip widens the exchange to the all-reduced reach (ncclAllReduce(max), 4 bytes) on every
 *     strip and repeats exchange + gather by itself (the advance is not repeated);
 *   - picles_step_project_remesh (host-driven exchange) returns PICLES_ERR_HALO naming the rows needed:
 *     call picles_halo_widen on every strip, repeat the exchange and the call.  The check sees this strip's own
 *     reach and the reach of the rows it received; give it the all-reduced picles_get_reach of the step
 *     (picles_set_global_reach) and every strip refuses together.  A host that widens from that all-reduced
 *     reach before the exchange never sees the error.
 * The exchange is never narrowed again.  A reach beyond rows_max is a PICLES_ERR_HALO that stands.
 */
int picles_halo_rows(picles_t* h, int* rows_exchanged, int* rows_max);
/* host-driven exchange: the all-reduced (max over strips) picles_get_reach of this step, so that the gather's check
   covers deposits of a neighbour's interior rows too; call between picles_step_advance and picles_step_project_remesh */
int picles_set_global_reach(picles_t* h, int reach);
int picles_halo_widen(picles_t* h, int rows);
int picles_step_strip(picles_t* h, double t, double dt_model,
                      const double* u_t, const double* v_t,
                      const double* u_t1, const double* v_t1,
                      int lo_rank, int hi_rank);

/* ---- wind ingestion: a device-resident wind mesh --------------------------------------- */
/*
 * Gridded winds kept on the device, so a step uploads nothing: the reference builds its wind
 * closures from gridded data as Interpolations.LinearInterpolation((x, y, t), U,
 * extrapolation_bc=Periodic()) (tests/T03_PIC_tripolar_realistic.jl:61-73,
 * src/Utils/WindEmulator.jl:18-43) and calls them at the home node of every particle.
 *   nxw, nyw, ntw   knots per axis (each >= 2); xw, yw, tw strictly increasing knot vectors
 *   U, V            ntw slices of nyw*nxw values, x fastest (Julia: U[ix, iy, it])
 *   node_x, node_y  coordinates of this strip's nodes, ny_local*Nx each (grid.data.x, grid.data.y)
 * Sampling is multilinear in (x, y, t); a coordinate outside its knot range is wrapped with
 * period (last knot - first knot), as extrapolation_bc = Periodic() does.  The mesh stays
 * resident until the next picles_set_wind_mesh / picles_set_grid call (all arrays are copied).
 */
int picles_set_wind_mesh(picles_t* h, int nxw, int nyw, int ntw,
                         const double* xw, const double* yw, const double* tw,
                         const double* U, const double* V,
                         const double* node_x, const double* node_y);
/* an ensemble's wind meshes, one per member on shared knots: xw, yw, tw, node_x and node_y as in
 * picles_set_wind_mesh (node_x, node_y: one plane of ny_local*Nx, shared by the members); U and V
 * hold members*ntw*nyw*nxw values, member slowest, each member's mesh as picles_set_wind_mesh takes
 * it.  Checks, codes and messages as picles_set_wind_mesh, all before an old mesh is freed; the
 * device holds 16*members*ntw*nyw*nxw bytes of mesh plus 16*members*nyw*nxw of scratch
 * (PICLES_ERR_ALLOC names the bytes).  With one member this is picles_set_wind_mesh.  Then
 * picles_seed_wind_mesh, picles_stage_wind_mesh, picles_step_wind_mesh, picles_sample_wind_mesh
 * and picles_measure_wind_sample work on every member: member m's wind, and everything a step does
 * with it, is bit for bit what a single-member handle given member m's mesh computes.  Each level
 * is still two kernel launches, whatever the member count.  Not supported: knot vectors per member,
 * and time slices streamed from the host (the whole time axis is resident). */
int picles_set_member_wind_meshes(picles_t* h, int nxw, int nyw, int ntw,
                                  const double* xw, const double* yw, const double* tw,
                                  const double* U, const double* V,
                                  const double* node_x, const double* node_y);
/* the mesh sampled at this strip's nodes at time t, to host (ny_local*Nx each; an ensemble with
   member meshes: members*ny_local*Nx each, member slowest): the values the closure
   u.(grid.data.x, grid.data.y, t) would return */
int picles_sample_wind_mesh(picles_t* h, double t, double* u_out, double* v_out);
/* picles_seed with the wind of the mesh at time t0 */
int picles_seed_wind_mesh(picles_t* h, double t0);
/* picles_step (single strip) / picles_step_strip (lo_rank, hi_rank as there; pass -1, -1 on a
   single-strip handle) with every wind level sampled on the device from the mesh: levels t and
   t+dt_model plus n_mid intermediate ones (0..PICLES_WIND_MID_MAX).  The previous step's t+dt
   level is reused as this step's t level when the times match. */
int picles_step_wind_mesh(picles_t* h, double t, double dt_model, int n_mid, int lo_rank, int hi_rank);
/* the wind half of picles_step_wind_mesh alone, for hosts that drive the phase-split calls
   (picles_step_advance / halo exchange / picles_step_project_remesh) themselves: every level of the
   step [t, t+dt_model] is sampled into the device planes; nothing is integrated */
int picles_stage_wind_mesh(picles_t* h, double t, double dt_model, int n_mid);

/* ---- state access ------------------------------------------------------ */
int picles_get_state(picles_t* h, double* S /* ny_local*Nx*3: planes e, m_x, m_y */);
int picles_set_state(picles_t* h, const double* S);
int picles_get_particles(picles_t* h, double* z /* 5 planes of ny_local*Nx */,
                         double* t, double* dt, uint8_t* flags, int32_t* status);
int picles_get_counters(picles_t* h, picles_counters_t* c);
/* the particles that integrated in the last step, by the number of Runge-Kutta attempts (accepted + rejected
   substeps, both algorithms under AutoTsit5) they took: hist[a] for a < nbins - 1, the rest in the last bin.
   The work per particle-step is data-dependent (SURVEY.md §8d); this is its distribution. */
int picles_get_attempt_histogram(picles_t* h, int64_t* hist, int nbins);
/* kernels launched by this library in this process so far (every entry point counts the kernels it launches) */
int64_t picles_launch_count(void);
/* AutoSwitch state of every particle (ny_local*Nx): the signed run length of the stiffness test
   (positive: consecutive stiff attempts, negative: non-stiff), +64 when Rosenbrock23 is current */
int picles_get_solver_state(picles_t* h, int8_t* as);
/* sum over this strip of State[:,:,0] (mean_of_state, run.jl:23-25, times n) — a cheap
   per-step scalar read-back */
int picles_state_energy_sum(picles_t* h, double* sum_e);

/* ---- output path (the "next" row after the step itself) ------------------------- */
/* derived fields of the node State, computed on the device, any output may be NULL
   (ny_local*Nx each):  Hs = 4*sqrt(e)                     src/visualization/movie_2D.jl:50
                        c_x, c_y = m*e/(2|m|^2)            GetGroupVelocity, src/Operators/core_2D.jl:138-147 */
int picles_get_fields(picles_t* h, double* Hs, double* c_x, double* c_y);
/* pinned host memory for asynchronous transfers (hosts without their own CUDA binding) */
int picles_host_alloc(void** p, int64_t nbytes);
int picles_host_free(void* p);
/* asynchronous State snapshot for the stores of run! (CashStore / StateStore pushes,
   src/Simulations/run.jl:94-112): returns at once; State is copied device-to-device on the
   compute stream and device-to-host on a second stream while the following steps run.
   S_host (3 planes, pinned for true overlap) is valid after picles_snapshot_wait; one
   snapshot may be in flight per handle (a second begin waits for the first). */
int picles_snapshot_begin(picles_t* h, double* S_host);
int picles_snapshot_wait(picles_t* h);

/* ---- checkpoint / resume --------------------------------------------------------- */
/* The reference cannot resume (run!(…; pickup=false) is unused, src/Simulations/run.jl:36).
   Here the particle planes (the AutoSwitch state of AutoTsit5 included), the node State and the
   pending wind level are the complete state of the path: save writes them into a caller-owned host blob of picles_checkpoint_size
   bytes; load restores them into a handle with the same grid and parameters (set_grid* and
   set_params called, picles_seed not needed).  A resumed run continues bit-identically. */
int picles_checkpoint_size(picles_t* h, int64_t* nbytes);
int picles_checkpoint_save(picles_t* h, void* blob, int64_t nbytes);
int picles_checkpoint_load(picles_t* h, const void* blob, int64_t nbytes);

/* device pointers for zero-copy consumers (torch / CUDA.jl): planes as above */
int picles_state_dev(picles_t* h, double** S_dev /* out: 3 plane pointers e, m_x, m_y */);
int picles_wind_dev(picles_t* h, double** u_t_dev, double** v_t_dev,
                    double** u_t1_dev, double** v_t1_dev);

/* ---- options -------------------------------------------------------------- */
enum {
    /* 0 (default): the step starts from State == 0, as run! does (run.jl:75-79).
       1: a bare time_step! on whatever State holds — deposits are added to the current
          node values in the reference's order (ParticleInCell.jl:372), as the scripts
          that call time_step! directly do (tests/T03_PIC_tripolar_aqua.jl:216-225). */
    PICLES_OPT_ACCUMULATE_STATE = 1
};
int picles_set_option(picles_t* h, int option, int value);
/* State .= 0 */
int picles_zero_state(picles_t* h);

/* ---- utilities for hosts without their own CUDA binding ------------------ */
/* async device-to-device copy on the handle's stream (same GPU or a peer) */
int picles_copy_dev(picles_t* h, void* dst_dev, const void* src_dev, int64_t nbytes);
/* CUDA-event stopwatch on the handle's stream: start; ...calls...; stop -> milliseconds */
int picles_timer_start(picles_t* h);
int picles_timer_stop(picles_t* h, double* ms);
/* measured FP64 FMA throughput of this device (register-resident DFMA chains), the
   roofline denominator of the advance kernel; ~50 ms */
int picles_measure_fp64_peak(picles_t* h, double* tflops);
/* self-test of the device fast-path division / sqrt (pmath.h) against the IEEE operators
   on random operands (raw bit patterns, physics-range magnitudes, special values).
   out6 = {n_div, flagged_div, mismatch_div, n_sqrt, flagged_sqrt, mismatch_sqrt};
   a mismatch is an unflagged result that differs from a/b or sqrt(x): must be 0. */
int picles_selftest_math(picles_t* h, uint64_t seed, int iters, int64_t* out6);
/* CUDA-event time per level of the wind-mesh sampling over this strip — the mesh-sized time blend
   plus the per-node kernel, as one step launches them (mean of `reps` repetitions): 32 algorithmic
   bytes per node (coordinates in, wind out) against the HBM roofline.  With member meshes: the member
   forms of both kernels, 48 bytes per member mesh point in the time blend and 16 per node plus 16 per
   member and node in the sampler */
int picles_measure_wind_sample(picles_t* h, double t, int reps, double* ms_per_launch);
/* measured HBM copy bandwidth (read+write bytes / s) over a buffer of `mib` MiB */
int picles_measure_hbm_copy(picles_t* h, int mib, double* gbs);

/* ---- the ONE-DIMENSIONAL model (WaveGrowth1D; SURVEY §8f-4) ---------------------------------
 * The same seam, one dimension down: everything `init_particles!(::Abstract1DModel)` and
 * `time_step!(::Abstract1DModel, dt)` do.
 *   picles1d_seed  replaces  init_particles!                 src/Simulations/run.jl:268-302
 *                            SeedParticle!                   src/Operators/core_1D.jl:270-330
 *   picles1d_step  replaces  State .= 0                      src/Simulations/run.jl:72-80
 *                            time_step!(::Abstract1DModel)   src/Operators/TimeSteppers.jl:51-92
 *                              advance!                      src/Operators/mapping_1D.jl:84-190
 *                              ParticleToNode! / push_to_grid! + merge!
 *                                                            src/Operators/mapping_1D.jl:41-53, src/ParticleInCell.jl:562-590, 228-252
 *                              remesh! / NodeToParticle!     src/Operators/mapping_1D.jl:197-283
 *   picles1d_set_grid        OneDGrid / OneDGridNotes        src/ParticleMesh.jl:102-134
 * The state vector of a particle is [lne, c̄_x, x] (particle_waves_v5.jl:584-650); State is (Nx, 3) column-major
 * [e, m_x, 0].  picles_params_t is shared with the 2-D path: C_varphi, direction, defaults, on_persist and
 * minimal_state as [E_min, m_x^2_min] — `periodic_boundary` is the model kwarg that wraps deposits and removes the
 * two boundary particles.  Solver ids: Tsit5, DP5; AutoTsit5 runs as Tsit5 (the Rosenbrock23 branch is 2-D only).
 * Winds: node values at t and t + dt_model; the particle reads them at its own position (linear in x between
 * nodes, linear in time).  has_defaults must be 0 (wind-sea seeding).
 */
typedef struct picles1d_handle picles1d_t;
int picles1d_create(picles1d_t** h, int device_id);
int picles1d_destroy(picles1d_t* h);
const char* picles1d_last_error(picles1d_t* h);
/* x_nodes[Nx]: OneDGridNotes.x (the particles' coordinates); xmin, dx: OneDGrid.xmin, .dx (the frame of the
   deposit weights, ParticleInCell.jl:165) */
int picles1d_set_grid(picles1d_t* h, int Nx, double xmin, double dx, const double* x_nodes);
int picles1d_set_params(picles1d_t* h, const picles_params_t* params);
/* u0[Nx]: winds(x_i, 0) */
int picles1d_seed(picles1d_t* h, const double* u0);
/* u_t[Nx], u_t1[Nx]: winds(x_i, t), winds(x_i, t + dt_model) */
int picles1d_step(picles1d_t* h, double t, double dt_model, const double* u_t, const double* u_t1);
int picles1d_get_state(picles1d_t* h, double* S /* Nx*3 */);
/* z[3*Nx] planes lne, c̄_x, x; t, dt, flags, status may be NULL */
int picles1d_get_particles(picles1d_t* h, double* z, double* t, double* dt, uint8_t* flags, int32_t* status);
int picles1d_get_counters(picles1d_t* h, picles_counters_t* out);

#ifdef __cplusplus
}
#endif
#endif /* PICLES_B200_H */
