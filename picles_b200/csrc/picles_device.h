/* picles_device.h — device-side data layout shared by the kernels and the C ABI layer. */
#ifndef PICLES_DEVICE_H
#define PICLES_DEVICE_H

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/picles_b200.h"

/* launch shapes: grids are capped at (SM count x resident blocks) and grid-stride */
#ifndef ADV_THREADS
#define ADV_THREADS 128
#endif
#ifndef ADV_MIN_BLOCKS
#define ADV_MIN_BLOCKS 3
#endif
/* advance launches per step that may be in flight on one DeviceCounters: the pipelined row blocks of an upload
   (slots 0..7) and the two boundary blocks of a strip (8, 9) */
#define ADV_SLOTS 12
#define ADV_SLOT_BOUNDARY 8 /* work queue of the launch that advances a strip's two boundary zones (picles_step_strip) */
#define ADV_HIST_BINS 48
/* projection gather + remesh: one block per tile of PR_TX x TY target nodes; the record tile
   (targets + a halo) is staged in shared memory by TMA.  The TMA box is always PR_BW x PR_BH
   = 72 x 20 elements; it is cut either as 16 target rows + 2 halo rows (reach <= 2, the common
   case) or as 12 target rows + 4 halo rows (reach 3-4: the small cells near a pole), chosen
   per launch from the previous step's reach.  TMA needs the box's first element 16-byte
   aligned in the inner dimension (measured: profiles/micro/tma_probe.cu — a misaligned start
   raises "illegal instruction"), so the int32 cell plane forces the x-halo PR_HX to a
   multiple of 4. */
#define PR_THREADS 256
#define PR_TX 64
#define PR_HX 4
#define PR_BW (PR_TX + 2 * PR_HX)
#define PR_BH 20
#define PR_HY_NARROW 2
#define PR_HY_WIDE 4
#ifndef PR_MIN_BLOCKS
#define PR_MIN_BLOCKS 3
#endif
/* row pitch of the record planes: multiple of 4 elements, so int32 rows are 16-byte
   multiples as TMA tensor maps require */
#define REC_PITCH_ALIGN 4
/* largest particle reach (cells) the projection gather supports; == PH_REACH_MAX */
#define PH_REACH_MAX_ABI 15

namespace picles {

/*
 * All planes are ny*Nx doubles, x fastest, for the rows this strip owns; `rec`/`cell`
 * have (ny + 2*halo) rows of pitch rp >= Nx (neighbour rows below and above).
 */
struct DeviceArrays {
    int Nx, Ny;       /* global shape */
    int bx, by;       /* PICLES_BND_* */
    int j0, ny, halo; /* strip: first global row (0-based), rows owned, halo rows the record planes hold on each side */
    int hx;           /* halo rows exchanged with the y-neighbours this step (<= halo; widened when the reach asks for it) */
    int rp;           /* row pitch (elements) of the record planes rec[] / cell */
    /* ensemble (picles_set_members): `members` models share the grid planes mask, M and pc; every other plane holds
       `members` single-member planes of ny*Nx nodes back to back (member slowest), the record planes and rowreach
       included.  1 for a single model.  Read by k_seed and by the ensemble forms of k_advance, k_advance_resume and
       k_project_remesh, which the launchers pick when it is above 1. */
    int members;
    double* z[5];     /* lne, c̄_x, c̄_y, x, y */
    double *t, *dt, *qold;
    int32_t* iter;
    uint8_t *flags, *status, *mask;
    int8_t* as;                      /* AutoTsit5: AutoSwitch state per particle (run length, +64 = Rosenbrock23 current) */
    int32_t* pending;                /* AutoTsit5: strip-local indices of the particles parked for k_advance_resume */
    double *u_t, *v_t, *u_t1, *v_t1; /* staged winds at t and t+DT */
    double *u_mid[PICLES_WIND_MID_MAX], *v_mid[PICLES_WIND_MID_MAX]; /* intermediate levels (allocated on first use) */
    int n_mid;                       /* intermediate levels staged for the next advance (0: linear in time) */
    double *u_lag, *v_lag;           /* B-1 as run: the wind at integrator time 0 + DT (the first step's t+DT level), read by the
                                        particles that were seeded off and therefore never advance their own clock; nullptr
                                        when there are none, under on_persist, and during the first step (== u_t1 then) */
    double* M[4];                    /* per-node projection kernel planes, or nullptr */
    double Mc[4];                    /* uniform projection kernel */
    double* pc;                      /* great-circle coefficient plane, or nullptr */
    double* rec[5];                  /* deposit records: e, m_x, m_y, w_x(ceil), w_y(ceil) */
    int32_t* cell;                   /* packed floor offsets + class, PH_CELL_INVALID if none */
    int32_t* rowreach;               /* per record row (ny + 2*halo): max reach of its deposits this step */
    double* S[3];                    /* State planes e, m_x, m_y */
};

struct DeviceCounters {
    /* integrated, substeps, rejects, rhs, reseed, fixups, failed, deposited, A, B, C, D, stiff switches, stiff attempts */
    unsigned long long sums[14];
    int32_t reach;        /* max reach of this strip's own deposits */
    int32_t max_attempts;
    int32_t reach_halo;   /* max reach of the records received into the halo rows */
    int32_t class1;       /* a deposit of the second class (a mask-3 particle of a periodic model) exists */
    int32_t n_pending;    /* AutoTsit5: particles parked by k_advance this step (entries of DeviceArrays::pending) */
    int32_t reach_all;    /* strips: 1 + the all-reduced reach that decides whether the hx rows exchanged suffice (the strips' boundary zones
                             under picles_step_strip, whole strips when the host all-reduces picles_get_reach); 0: not set, the gather
                             then judges by what this strip knows itself */
    int32_t halo_short;   /* strips: set by the gather when deposits reach further than the hx rows exchanged — it then changes nothing */
    int32_t n_seed_off;   /* written by k_seed: active particles seeded off (they need the lag wind level under B-1 as run) */
    int32_t reach_bnd;    /* strips: max reach of the deposits of the two boundary zones (the rows within the supported reach of a
                             strip edge: only their particles can land on a neighbour), known as soon as the boundary launch is done */
    /* work queue of the advance launches of one step: launch `slot` hands out its 32-particle chunks from next_chunk[slot] */
    unsigned long long next_chunk[ADV_SLOTS];
    /* particles that integrated this step by the number of Runge-Kutta attempts they took (last bin: >= ADV_HIST_BINS - 1) */
    unsigned long long attempt_hist[ADV_HIST_BINS];
};

void launch_seed(const DeviceArrays& A, const picles_params_t& P, const double* u0, const double* v0, DeviceCounters* dc,
                 int sms, cudaStream_t st);
void launch_advance(const DeviceArrays& A, const picles_params_t& P, double DT, DeviceCounters* dc, int sms,
                    cudaStream_t st, int64_t l_begin, int64_t l_end, int slot);
void launch_advance2(const DeviceArrays& A, const picles_params_t& P, double DT, DeviceCounters* dc, int sms,
                     cudaStream_t st, int64_t l_begin, int64_t l_end, int64_t l2_begin, int64_t l2_end, int slot);
/* *dst = *src + 1 on the stream: the word the strips all-reduce (1 + reach, so that 0 reads as "not set") */
void launch_reach_word(const int32_t* src, int32_t* dst, cudaStream_t st);
/* kernels launched by this library since it was loaded (every launch_* call counts its kernels) */
long long launch_count();
/* TMA tensor maps of the six record planes (box PR_BW x PR_BH x 1 member) */
struct ProjectMaps {
    CUtensorMap rec[5];
    CUtensorMap cell;
};
int project_remesh_smem_bytes();
cudaError_t project_remesh_configure();
void launch_project_remesh(const ProjectMaps& maps, const DeviceArrays& A, const picles_params_t& P, double DT,
                           int n_classes, int accumulate, int wide, DeviceCounters* dc, cudaStream_t st);
/* gridded wind field resident on the device (wind_mesh.h) + the node coordinates it is sampled at */
struct DeviceWindMesh {
    int nx, ny, nt;
    double *xw, *yw, *tw, *U, *V;
    double *node_x, *node_y; /* ny*Nx each */
    double *Ub, *Vb;         /* scratch: the slice blended in time for the level being sampled, nx*ny each (a slice per
                                member with member meshes) */
};
void launch_wind_sample(const DeviceWindMesh& W, int64_t n, double t, double* u_out, double* v_out, int sms, cudaStream_t st);
/* `members` meshes on W's knots (U, V: members meshes back to back; Ub, Vb: members slices), sampled at the n nodes of
   W.node_x/node_y into members planes of n values each, member slowest */
void launch_wind_sample_members(const DeviceWindMesh& W, int members, int64_t n, double t, double* u_out, double* v_out,
                                int sms, cudaStream_t st);
/* nblocks partial sums of each of `members` planes of n values back to back, in one launch: partial[m*nblocks + b] */
void launch_energy(const double* e, int64_t n, int members, double* partial, int nblocks, cudaStream_t st);
void launch_halo_pack(const DeviceArrays& A, char* lo, char* hi, int sms, cudaStream_t st);
void launch_halo_unpack(const DeviceArrays& A, const char* lo, const char* hi, DeviceCounters* dc, int sms, cudaStream_t st);
void launch_grid_metric(int64_t n, const double* dx, const double* dy, const double* angle_dx, const double* lat,
                        double R_earth, double* M11, double* M12, double* M21, double* M22, double* pc, int sms, cudaStream_t st);
void launch_make_boundaries(const uint8_t* ocean, uint8_t* total, int Nx, int Ny, int bx, int by, int sms, cudaStream_t st);
void launch_fields(int64_t n, const double* e, const double* mx, const double* my, double* Hs, double* cx, double* cy,
                   int sms, cudaStream_t st);
void launch_fill_i32(int32_t* p, int64_t n, int32_t v, int sms, cudaStream_t st);
void launch_selftest_math(uint64_t seed, int iters, unsigned long long* out, int sms, cudaStream_t st);
void launch_fp64_peak(double* out, int iters, int sms, cudaStream_t st, int64_t* fmas);
void launch_copy_f64(double* dst, const double* src, int64_t n, int sms, cudaStream_t st);

} /* namespace picles */
#endif
