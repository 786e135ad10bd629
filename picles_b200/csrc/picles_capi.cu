/*
 * picles_capi.cu — the C ABI of include/picles_b200.h: handle, device memory, streams,
 * host<->device staging and kernel orchestration of one model step on one y-strip.
 * No torch types, no CPU fallback.
 */
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stdarg.h>
#include <stddef.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <utility>
#include <vector>

#include "../../include/picles_b200.h"
#include "picles_device.h"

using namespace picles;

#define ENERGY_BLOCKS 1024
/* host winds are uploaded in this many row chunks, each chunk's advance starting as soon as
   its rows have landed (copy stream + events), when the strip is large enough to matter */
#define PIPE_CHUNKS 8
#define PIPE_MIN_NODES (1 << 20)
static_assert(PIPE_CHUNKS + 2 <= ADV_SLOTS, "one work queue per advance launch of a step");
static_assert(PIPE_CHUNKS == ADV_SLOT_BOUNDARY, "the boundary launch takes the queue behind the interior's chunks");
#define PIPE_EVENTS (PIPE_CHUNKS + 6) /* chunk landed x8, boundary blocks x2, boundary advanced, halo exchanged, interior advanced, compute stream idle */

struct picles_handle {
    int device = -1;
    int sms = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;           /* wind upload pipelined against the advance */
    cudaEvent_t pev[PIPE_EVENTS] = {};
    cudaStream_t comm_stream = nullptr;           /* halo exchange overlapped with the interior advance */
    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr}; /* adv0, adv1, prj0, prj1=rms0, rms1 */
    cudaEvent_t tev[2] = {nullptr, nullptr};                           /* user stopwatch */
    bool have_grid = false, have_params = false, seeded = false, winds_loaded = false;
    DeviceArrays A;
    ProjectMaps maps; /* TMA tensor maps of the record planes */
    picles_params_t P;
    DeviceCounters* d_counters = nullptr;
    DeviceCounters* h_counters = nullptr; /* pinned */
    double* d_partial = nullptr;
    double* h_partial = nullptr;          /* pinned */
    char *send_lo = nullptr, *send_hi = nullptr, *recv_lo = nullptr, *recv_hi = nullptr;
    int64_t halo_bytes = 0;                       /* capacity of each halo buffer (A.halo rows) */
    int32_t* reach_send = nullptr;                /* staging word of the reach all-reduce */
    int32_t reach_all_host = 0;                   /* picles_set_global_reach: staging word */
    int n_halo_widened = 0;                       /* steps that repeated exchange + gather with wider rows */
    std::vector<void*> allocs;
    picles_counters_t last;
    int64_t n_active = 0;
    bool timing_valid = false;
    int accumulate = 0; /* PICLES_OPT_ACCUMULATE_STATE */
    int64_t steps_since_seed = 0; /* model steps taken since picles_seed (the integrator clocks started at 0 then) */
    int32_t n_seed_off = 0;       /* active particles seeded off: under B-1 as run they read the lag wind level */
    double *lag_u = nullptr, *lag_v = nullptr; /* storage of DeviceArrays::u_lag / v_lag (allocated on first use) */
    double* snap = nullptr;       /* staging copy of State for asynchronous snapshots (3 planes) */
    cudaStream_t snap_stream = nullptr; /* D2H of snapshots: its own stream, so wind uploads are not queued behind it */
    cudaEvent_t snap_ev[2] = {nullptr, nullptr}; /* staging copy done / D2H done */
    bool snap_pending = false;
    DeviceWindMesh wm = {};        /* resident wind mesh + node coordinates (picles_set_wind_mesh) */
    std::vector<void*> wm_allocs;
    bool have_wind_mesh = false;
    int wm_members = 1;            /* meshes resident in wm: one, or one per member (picles_set_member_wind_meshes) */
    bool wm_t1_valid = false;      /* the t1 wind level was sampled from the mesh at wm_t1_time */
    double wm_t1_time = 0.0;
    int members = 1;               /* picles_set_members: ensemble members stepped together (A.members once a grid is set) */
    double* d_member_partial = nullptr; /* picles_member_energy_sums: ENERGY_BLOCKS partial sums per member */
    double* h_member_partial = nullptr; /* pinned */
    void* comm = nullptr; /* ncclComm_t of the strip communicator */
    int comm_rank = -1, comm_size = 0;
    char err[512];
};

static thread_local char g_err[512] = "";

static int fail(picles_t* h, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h) snprintf(h->err, sizeof h->err, "%s", buf);
    snprintf(g_err, sizeof g_err, "%s", buf);
    return code;
}

#define CK(call)                                                                                        \
    do {                                                                                                \
        cudaError_t e_ = (call);                                                                        \
        if (e_ != cudaSuccess)                                                                          \
            return fail(h, PICLES_ERR_CUDA, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__,        \
                        cudaGetErrorString(e_));                                                        \
    } while (0)

template <class T>
static int dalloc(picles_t* h, T** p, int64_t count) {
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, (size_t)(count > 0 ? count : 1) * sizeof(T));
    if (e != cudaSuccess) return fail(h, PICLES_ERR_ALLOC, "cudaMalloc(%lld bytes): %s", (long long)(count * sizeof(T)), cudaGetErrorString(e));
    h->allocs.push_back(q);
    *p = (T*)q;
    return 0;
}
#define DALLOC(ptr, count)                      \
    do {                                        \
        int rc_ = dalloc(h, &(ptr), (count));   \
        if (rc_) return rc_;                    \
    } while (0)

/* ---- TMA tensor maps of the record planes --------------------------------------------
 * cuTensorMapEncodeTiled is a driver entry point; it is resolved through the runtime so the
 * library does not link libcuda.  Planes are 3-D (Nx, ny + 2*halo, members) with row pitch rp; the box
 * is the projection tile (PR_BW x PR_BH) of one member, so it never reaches into the next member's rows;
 * out-of-bounds elements are zero-filled. */
typedef CUresult (*pk_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                       const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                       CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static int make_project_maps(picles_t* h) {
    static pk_encode_tiled_fn encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        CK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
        if (!fn || q != cudaDriverEntryPointSuccess) return fail(h, PICLES_ERR_CUDA, "cuTensorMapEncodeTiled is not available in this driver");
        encode = (pk_encode_tiled_fn)fn;
    }
    const DeviceArrays& A = h->A;
    cuuint64_t dims[3] = {(cuuint64_t)A.Nx, (cuuint64_t)(A.ny + 2 * A.halo), (cuuint64_t)A.members};
    cuuint32_t box[3] = {PR_BW, PR_BH, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    for (int k = 0; k < 6; k++) {
        bool cell = (k == 5);
        const cuuint64_t row = (cuuint64_t)A.rp * (cell ? 4 : 8);
        cuuint64_t stride[2] = {row, row * (cuuint64_t)(A.ny + 2 * A.halo)};
        CUresult r = encode(cell ? &h->maps.cell : &h->maps.rec[k], cell ? CU_TENSOR_MAP_DATA_TYPE_INT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT64,
                            3, cell ? (void*)A.cell : (void*)A.rec[k], dims, stride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(h, PICLES_ERR_CUDA, "cuTensorMapEncodeTiled(plane %d) failed with CUresult %d", k, (int)r);
    }
    CK(project_remesh_configure());
    return 0;
}

static void free_grid(picles_t* h) {
    if (h->snap_stream) cudaStreamSynchronize(h->snap_stream); /* a snapshot may still read the staging copy */
    for (void* p : h->allocs) cudaFree(p);
    h->allocs.clear();
    for (void* p : h->wm_allocs) cudaFree(p);
    h->wm_allocs.clear();
    h->wm = DeviceWindMesh{};
    h->wm_members = 1;
    h->have_wind_mesh = h->wm_t1_valid = false;
    memset(&h->A, 0, sizeof h->A);
    h->send_lo = h->send_hi = h->recv_lo = h->recv_hi = nullptr;
    h->reach_send = nullptr;
    h->snap = nullptr;
    h->d_member_partial = nullptr;
    if (h->h_member_partial) { cudaFreeHost(h->h_member_partial); h->h_member_partial = nullptr; }
    h->snap_pending = false;
    h->lag_u = h->lag_v = nullptr;
    h->steps_since_seed = 0;
    h->n_seed_off = 0;
    h->have_grid = h->seeded = h->winds_loaded = false;
}

/* ---- NCCL, bound at run time --------------------------------------------------------
 * The strip communicator is the only place the library talks to another GPU.  NCCL is
 * resolved with dlopen so a single-GPU host (or one that exchanges halos itself through
 * picles_halo_buffers) needs no NCCL at all; a host process that already loaded NCCL
 * (torch, NCCL.jl) shares that copy.  Only the types the six entry points need are
 * declared here (nccl.h: ncclUniqueId is 128 opaque bytes, ncclInt8 = 0, ncclInt32 = 2, ncclMax = 2). */
typedef struct { char internal[128]; } pk_nccl_id_t;
typedef int (*pk_nccl_get_id_fn)(pk_nccl_id_t*);
typedef int (*pk_nccl_init_rank_fn)(void**, int, pk_nccl_id_t, int);
typedef int (*pk_nccl_destroy_fn)(void*);
typedef int (*pk_nccl_sendrecv_fn)(void*, size_t, int, int, void*, cudaStream_t);
typedef int (*pk_nccl_allreduce_fn)(const void*, void*, size_t, int, int, void*, cudaStream_t);
typedef int (*pk_nccl_group_fn)(void);
typedef const char* (*pk_nccl_errstr_fn)(int);
static struct {
    void* dl = nullptr;
    pk_nccl_get_id_fn get_id = nullptr;
    pk_nccl_init_rank_fn init_rank = nullptr;
    pk_nccl_destroy_fn destroy = nullptr;
    pk_nccl_sendrecv_fn send = nullptr, recv = nullptr;
    pk_nccl_allreduce_fn all_reduce = nullptr;
    pk_nccl_group_fn group_start = nullptr, group_end = nullptr;
    pk_nccl_errstr_fn errstr = nullptr;
} g_nccl;

static int nccl_load(picles_t* h, const char* path) {
    if (g_nccl.dl) return 0;
    void* dl = nullptr;
    if (path && *path) dl = dlopen(path, RTLD_NOW | RTLD_GLOBAL);
    if (!dl) dl = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL); /* the host's copy */
    if (!dl) dl = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!dl) dl = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!dl) return fail(h, PICLES_ERR_COMM, "cannot load NCCL (%s); pass the path of libnccl.so.2", dlerror());
#define PK_SYM(field, type, name)                                                                \
    g_nccl.field = (type)dlsym(dl, name);                                                        \
    if (!g_nccl.field) return fail(h, PICLES_ERR_COMM, "NCCL symbol %s not found", name);
    PK_SYM(get_id, pk_nccl_get_id_fn, "ncclGetUniqueId")
    PK_SYM(init_rank, pk_nccl_init_rank_fn, "ncclCommInitRank")
    PK_SYM(destroy, pk_nccl_destroy_fn, "ncclCommDestroy")
    PK_SYM(send, pk_nccl_sendrecv_fn, "ncclSend")
    PK_SYM(recv, pk_nccl_sendrecv_fn, "ncclRecv")
    PK_SYM(all_reduce, pk_nccl_allreduce_fn, "ncclAllReduce")
    PK_SYM(group_start, pk_nccl_group_fn, "ncclGroupStart")
    PK_SYM(group_end, pk_nccl_group_fn, "ncclGroupEnd")
    PK_SYM(errstr, pk_nccl_errstr_fn, "ncclGetErrorString")
#undef PK_SYM
    g_nccl.dl = dl;
    return 0;
}
#define NCK(call)                                                                                   \
    do {                                                                                            \
        int r_ = (call);                                                                            \
        if (r_ != 0) return fail(h, PICLES_ERR_COMM, "%s failed: %s", #call, g_nccl.errstr(r_));    \
    } while (0)


extern "C" {

int picles_abi_version(void) { return PICLES_ABI_VERSION; }

const char* picles_last_error(picles_t* h) { return h ? h->err : g_err; }

static int create_resources(picles_t* h) {
    CK(cudaSetDevice(h->device));
    CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&h->snap_stream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&h->comm_stream, cudaStreamNonBlocking));
    for (int k = 0; k < PIPE_EVENTS; k++) CK(cudaEventCreateWithFlags(&h->pev[k], cudaEventDisableTiming));
    for (int k = 0; k < 5; k++) CK(cudaEventCreate(&h->ev[k]));
    for (int k = 0; k < 2; k++) CK(cudaEventCreate(&h->tev[k]));
    for (int k = 0; k < 2; k++) CK(cudaEventCreateWithFlags(&h->snap_ev[k], cudaEventDisableTiming));
    CK(cudaMalloc((void**)&h->d_counters, sizeof(DeviceCounters)));
    CK(cudaMallocHost((void**)&h->h_counters, sizeof(DeviceCounters)));
    CK(cudaMalloc((void**)&h->d_partial, ENERGY_BLOCKS * sizeof(double)));
    CK(cudaMallocHost((void**)&h->h_partial, ENERGY_BLOCKS * sizeof(double)));
    return PICLES_OK;
}

int picles_create(picles_t** out, int device_id) {
    picles_t* h = nullptr;
    if (!out) return fail(nullptr, PICLES_ERR_ARG, "picles_create: null handle pointer");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, PICLES_ERR_CUDA, "no CUDA device available (%s); this library has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    if (device_id < 0 || device_id >= ndev) return fail(nullptr, PICLES_ERR_ARG, "device %d out of range [0,%d)", device_id, ndev);
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device_id);
    if (e != cudaSuccess) return fail(nullptr, PICLES_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    if (prop.major != 10)
        return fail(nullptr, PICLES_ERR_CUDA, "device %d is sm_%d%d; this library ships sm_100a code only", device_id,
                    prop.major, prop.minor);
    h = new picles_handle();
    h->err[0] = 0;
    h->device = device_id;
    h->sms = prop.multiProcessorCount;
    memset(&h->A, 0, sizeof h->A);
    memset(&h->last, 0, sizeof h->last);
    int rc = create_resources(h);
    if (rc) { /* nothing half-built survives a failed create: the caller holds no handle to clean up with */
        snprintf(g_err, sizeof g_err, "%s", h->err);
        picles_destroy(h);
        return rc;
    }
    *out = h;
    return PICLES_OK;
}

int picles_destroy(picles_t* h) {
    if (!h) return PICLES_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->copy_stream) cudaStreamSynchronize(h->copy_stream);
    if (h->snap_stream) cudaStreamSynchronize(h->snap_stream);
    if (h->comm_stream) cudaStreamSynchronize(h->comm_stream);
    if (h->comm && g_nccl.destroy) { g_nccl.destroy(h->comm); h->comm = nullptr; }
    free_grid(h);
    if (h->d_counters) cudaFree(h->d_counters);
    if (h->h_counters) cudaFreeHost(h->h_counters);
    if (h->d_partial) cudaFree(h->d_partial);
    if (h->h_partial) cudaFreeHost(h->h_partial);
    if (h->h_member_partial) cudaFreeHost(h->h_member_partial);
    for (int k = 0; k < 5; k++)
        if (h->ev[k]) cudaEventDestroy(h->ev[k]);
    for (int k = 0; k < 2; k++)
        if (h->tev[k]) cudaEventDestroy(h->tev[k]);
    for (int k = 0; k < 2; k++)
        if (h->snap_ev[k]) cudaEventDestroy(h->snap_ev[k]);
    for (int k = 0; k < PIPE_EVENTS; k++)
        if (h->pev[k]) cudaEventDestroy(h->pev[k]);
    if (h->comm_stream) cudaStreamDestroy(h->comm_stream);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->snap_stream) cudaStreamDestroy(h->snap_stream);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return PICLES_OK;
}

/* refusal of the calls an ensemble does not support (strips, halo exchange, checkpoints) */
static int refuse_members(picles_t* h, const char* what) {
    if (!h) return fail(nullptr, PICLES_ERR_ARG, "null handle");
    if (h->members > 1)
        return fail(h, PICLES_ERR_ARG, "%s is not supported for an ensemble (%d members): %s", what, h->members,
                    "members are stepped in one handle on one GPU and are not checkpointed");
    return PICLES_OK;
}
#define REFUSE_MEMBERS(h, what)                    \
    do {                                           \
        int rm_ = refuse_members((h), (what));     \
        if (rm_) return rm_;                       \
    } while (0)
/* the wind-mesh calls sample every member of an ensemble: each member needs its mesh (picles_set_member_wind_meshes) */
static int refuse_members_without_meshes(picles_t* h, const char* what) {
    if (!h) return fail(nullptr, PICLES_ERR_ARG, "null handle");
    if (h->members > 1 && !(h->have_wind_mesh && h->wm_members == h->members))
        return fail(h, PICLES_ERR_ARG, "%s is not supported for an ensemble (%d members) without member wind meshes: "
                    "set one mesh per member with picles_set_member_wind_meshes", what, h->members);
    return PICLES_OK;
}
#define REFUSE_MEMBERS_WITHOUT_MESHES(h, what)                  \
    do {                                                        \
        int rm_ = refuse_members_without_meshes((h), (what));   \
        if (rm_) return rm_;                                    \
    } while (0)

/* particles of the handle: Nx*ny per member */
static int64_t nodes(const picles_t* h) { return (int64_t)h->A.Nx * h->A.ny * h->A.members; }
/* entries of rowreach: the record rows of every member */
static int64_t record_rows(const picles_t* h) { return (int64_t)(h->A.ny + 2 * h->A.halo) * h->A.members; }

int picles_set_members(picles_t* h, int members) {
    if (!h) return fail(nullptr, PICLES_ERR_ARG, "null handle");
    if (h->have_grid) return fail(h, PICLES_ERR_STATE, "picles_set_members must be called before picles_set_grid*");
    /* members is a launch dimension (grid z of the gather, grid y of the per-member energy sum) */
    if (members < 1 || members > 65535) return fail(h, PICLES_ERR_ARG, "members = %d outside 1..65535", members);
    h->members = members;
    return PICLES_OK;
}

/* raw metric arrays of the strip's nodes (host): what ProjetionKernel(ij_mesh, stats) and
   SphericalPropagationCorrection(ij_mesh, stats) consume */
struct RawMetric {
    const double *dx, *dy, *angle_dx, *lat;
    double R_earth;
};

static int set_grid_impl(picles_t* h, int Nx, int Ny, int bx, int by, int j0, int ny_local, int halo,
                         const uint8_t* mask, const double* M, const double* M_const, const double* pc_coef,
                         const RawMetric* raw) {
    if (!h) return fail(nullptr, PICLES_ERR_ARG, "null handle");
    if (Nx < 1 || Ny < 1 || ny_local < 1 || j0 < 0 || j0 + ny_local > Ny || halo < 0)
        return fail(h, PICLES_ERR_ARG, "bad grid shape Nx=%d Ny=%d j0=%d ny=%d halo=%d", Nx, Ny, j0, ny_local, halo);
    if (bx < 0 || bx > 1 || by < 0 || by > 2) return fail(h, PICLES_ERR_ARG, "bad boundary types bx=%d by=%d", bx, by);
    if (!mask) return fail(h, PICLES_ERR_ARG, "mask is required");
    if (!M && !M_const && !raw) return fail(h, PICLES_ERR_ARG, "one of M / M_const is required");
    if (raw && (!raw->dx || !raw->dy || !raw->angle_dx || !raw->lat || !(raw->R_earth > 0)))
        return fail(h, PICLES_ERR_ARG, "dx, dy, angle_dx, lat and a positive R_earth are required");
    if (halo > PH_REACH_MAX_ABI) return fail(h, PICLES_ERR_ARG, "halo %d exceeds the supported reach %d", halo, PH_REACH_MAX_ABI);
    if (ny_local != Ny && halo > ny_local) return fail(h, PICLES_ERR_ARG, "halo %d wider than the strip (%d rows)", halo, ny_local);
    const int E = h->members;
    if (E > 1 && (j0 != 0 || ny_local != Ny || halo != 0))
        return fail(h, PICLES_ERR_ARG, "an ensemble (%d members) cannot be a strip: j0 = %d, ny_local = %d of %d, halo = %d; "
                    "split the members over handles instead", E, j0, ny_local, Ny, halo);
    if (E > 1 && (int64_t)E * Nx * ny_local >= ((int64_t)1 << 31))
        return fail(h, PICLES_ERR_ARG, "%d members x %d x %d nodes: an ensemble holds fewer than 2^31 particles "
                    "(the AutoTsit5 pending list stores 32-bit particle indices)", E, Nx, ny_local);
    /* `halo` rows are exchanged to begin with; the record planes of a strip hold room for the widest exchange the
       gather supports, so a step whose deposits reach further only repeats exchange + gather with more rows */
    const int halo_x = halo;
    if (ny_local != Ny && halo > 0) halo = (ny_local < PH_REACH_MAX_ABI) ? ny_local : PH_REACH_MAX_ABI;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    free_grid(h);
    DeviceArrays& A = h->A;
    A.Nx = Nx; A.Ny = Ny; A.bx = bx; A.by = by; A.j0 = j0; A.ny = ny_local; A.halo = halo; A.hx = halo_x;
    A.rp = (Nx + REC_PITCH_ALIGN - 1) / REC_PITCH_ALIGN * REC_PITCH_ALIGN;
    A.members = E;
    int64_t n = (int64_t)Nx * ny_local; /* the grid planes */
    const int64_t nE = n * E;           /* the particle-side planes */
    int64_t ne = (int64_t)A.rp * (ny_local + 2 * halo) * E;
    for (int k = 0; k < 5; k++) DALLOC(A.z[k], nE);
    DALLOC(A.t, nE); DALLOC(A.dt, nE); DALLOC(A.qold, nE);
    DALLOC(A.iter, nE);
    DALLOC(A.flags, nE); DALLOC(A.status, nE); DALLOC(A.mask, n);
    DALLOC(A.as, nE);
    CK(cudaMemsetAsync(A.as, 0, (size_t)nE, h->stream));
    DALLOC(A.pending, nE);
    DALLOC(A.u_t, nE); DALLOC(A.v_t, nE); DALLOC(A.u_t1, nE); DALLOC(A.v_t1, nE);
    for (int k = 0; k < 5; k++) DALLOC(A.rec[k], ne);
    DALLOC(A.cell, ne);
    DALLOC(A.rowreach, record_rows(h));
    CK(cudaMemsetAsync(A.rowreach, 0, (size_t)record_rows(h) * 4, h->stream));
    for (int k = 0; k < 3; k++) DALLOC(A.S[k], nE);
    CK(cudaMemcpyAsync(A.mask, mask, (size_t)n, cudaMemcpyHostToDevice, h->stream));
    if (M) {
        for (int k = 0; k < 4; k++) {
            DALLOC(A.M[k], n);
            CK(cudaMemcpyAsync(A.M[k], M + k * n, (size_t)n * 8, cudaMemcpyHostToDevice, h->stream));
        }
    } else if (raw) {
        /* grid-metric lookup on the device: per-node kernel and great-circle coefficient */
        double* tmp = nullptr;
        cudaError_t e = cudaMalloc((void**)&tmp, (size_t)n * 4 * 8);
        if (e != cudaSuccess) return fail(h, PICLES_ERR_ALLOC, "cudaMalloc(metric staging): %s", cudaGetErrorString(e));
        const double* src[4] = {raw->dx, raw->dy, raw->angle_dx, raw->lat};
        for (int k = 0; k < 4; k++) {
            e = cudaMemcpyAsync(tmp + k * n, src[k], (size_t)n * 8, cudaMemcpyHostToDevice, h->stream);
            if (e != cudaSuccess) { cudaFree(tmp); return fail(h, PICLES_ERR_CUDA, "metric upload: %s", cudaGetErrorString(e)); }
        }
        for (int k = 0; k < 4; k++) DALLOC(A.M[k], n);
        DALLOC(A.pc, n);
        launch_grid_metric(n, tmp, tmp + n, tmp + 2 * n, tmp + 3 * n, raw->R_earth, A.M[0], A.M[1], A.M[2], A.M[3], A.pc, h->sms, h->stream);
        e = cudaStreamSynchronize(h->stream);
        cudaFree(tmp);
        if (e != cudaSuccess) return fail(h, PICLES_ERR_CUDA, "k_grid_metric: %s", cudaGetErrorString(e));
    } else {
        for (int k = 0; k < 4; k++) { A.M[k] = nullptr; A.Mc[k] = M_const[k]; }
    }
    if (pc_coef && !raw) {
        DALLOC(A.pc, n);
        CK(cudaMemcpyAsync(A.pc, pc_coef, (size_t)n * 8, cudaMemcpyHostToDevice, h->stream));
    }
    for (int k = 0; k < 5; k++) CK(cudaMemsetAsync(A.rec[k], 0, (size_t)ne * 8, h->stream));
    launch_fill_i32(A.cell, ne, -1, h->sms, h->stream);
    for (int k = 0; k < 3; k++) CK(cudaMemsetAsync(A.S[k], 0, (size_t)nE * 8, h->stream));
    CK(cudaMemsetAsync(A.flags, 0, (size_t)nE, h->stream));
    h->halo_bytes = (int64_t)halo * A.rp * (5 * 8 + 4); /* capacity of each buffer; a message carries hx rows */
    if (halo > 0) {
        DALLOC(h->send_lo, h->halo_bytes); DALLOC(h->send_hi, h->halo_bytes);
        DALLOC(h->recv_lo, h->halo_bytes); DALLOC(h->recv_hi, h->halo_bytes);
        DALLOC(h->reach_send, 1);
        /* until a neighbour delivers rows, received halos are "no deposit" */
        CK(cudaMemsetAsync(h->recv_lo, 0xff, (size_t)h->halo_bytes, h->stream));
        CK(cudaMemsetAsync(h->recv_hi, 0xff, (size_t)h->halo_bytes, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
    int rc_maps = make_project_maps(h);
    if (rc_maps) return rc_maps;
    /* |ocean_points| of this strip */
    h->n_active = -1; /* resolved at seed (depends on the model's periodic_boundary) */
    h->have_grid = true;
    return PICLES_OK;
}

int picles_set_grid(picles_t* h, int Nx, int Ny, int bx, int by, int j0, int ny_local, int halo,
                    const uint8_t* mask, const double* M, const double* M_const, const double* pc_coef) {
    return set_grid_impl(h, Nx, Ny, bx, by, j0, ny_local, halo, mask, M, M_const, pc_coef, nullptr);
}

int picles_set_grid_metric(picles_t* h, int Nx, int Ny, int bx, int by, int j0, int ny_local, int halo,
                           const uint8_t* mask, const double* dx, const double* dy, const double* angle_dx,
                           const double* lat, double R_earth) {
    RawMetric raw = {dx, dy, angle_dx, lat, R_earth};
    return set_grid_impl(h, Nx, Ny, bx, by, j0, ny_local, halo, mask, nullptr, nullptr, nullptr, &raw);
}

int picles_get_metric(picles_t* h, double* M, double* pc) {
    if (!h || !h->have_grid) return fail(h, PICLES_ERR_STATE, "grid not set");
    CK(cudaSetDevice(h->device));
    const DeviceArrays& A = h->A;
    int64_t n = (int64_t)A.Nx * A.ny;
    if (M) {
        if (A.M[0]) {
            for (int k = 0; k < 4; k++) CK(cudaMemcpyAsync(M + k * n, A.M[k], (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
        } else {
            for (int k = 0; k < 4; k++)
                for (int64_t l = 0; l < n; l++) M[k * n + l] = A.Mc[k];
        }
    }
    if (pc) {
        if (A.pc) CK(cudaMemcpyAsync(pc, A.pc, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
        else memset(pc, 0, (size_t)n * 8);
    }
    CK(cudaStreamSynchronize(h->stream));
    return PICLES_OK;
}

/* make_boundaries(mask, Nx, Ny) on the device: ocean (1) / land (0) -> total mask 0..3 */
int picles_make_boundaries(picles_t* h, int Nx, int Ny, int bx, int by, const uint8_t* ocean, uint8_t* total) {
    if (!h || !ocean || !total || Nx < 1 || Ny < 1 || bx < 0 || bx > 1 || by < 0 || by > 2)
        return fail(h, PICLES_ERR_ARG, "picles_make_boundaries: bad argument");
    CK(cudaSetDevice(h->device));
    size_t n = (size_t)Nx * Ny;
    uint8_t* d = nullptr;
    if (cudaMalloc((void**)&d, 2 * n) != cudaSuccess) return fail(h, PICLES_ERR_ALLOC, "cannot allocate %zu bytes", 2 * n);
    cudaError_t e = cudaMemcpyAsync(d, ocean, n, cudaMemcpyHostToDevice, h->stream);
    if (e == cudaSuccess) {
        launch_make_boundaries(d, d + n, Nx, Ny, bx, by, h->sms, h->stream);
        e = cudaMemcpyAsync(total, d + n, n, cudaMemcpyDeviceToHost, h->stream);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    cudaFree(d);
    if (e != cudaSuccess) return fail(h, PICLES_ERR_CUDA, "picles_make_boundaries: %s", cudaGetErrorString(e));
    return PICLES_OK;
}

int picles_set_params(picles_t* h, const picles_params_t* p) {
    if (!h || !p) return fail(h, PICLES_ERR_ARG, "null argument");
    if (p->solver != PICLES_SOLVER_TSIT5 && p->solver != PICLES_SOLVER_DP5 && p->solver != PICLES_SOLVER_AUTOTSIT5)
        return fail(h, PICLES_ERR_ARG, "unknown solver id %d", p->solver);
    if (!p->adaptive) return fail(h, PICLES_ERR_ARG, "adaptive=false is not supported");
    if (!(p->abstol > 0) || !(p->reltol > 0) || !(p->dtmin >= 0) || !(p->dt > 0) || !(p->dtmax > 0) || !(p->r_g > 0) || !(p->e_T > 0))
        return fail(h, PICLES_ERR_ARG, "non-positive tolerance / step / constant in params");
    if (p->maxiters < 1 || p->maxiters > 2000000000LL) return fail(h, PICLES_ERR_ARG, "maxiters out of range");
    h->P = *p;
    h->have_params = true;
    return PICLES_OK;
}

static int need_ready(picles_t* h, bool seeded) {
    if (!h) return fail(nullptr, PICLES_ERR_ARG, "null handle");
    if (!h->have_grid || !h->have_params) return fail(h, PICLES_ERR_STATE, "picles_set_grid and picles_set_params must be called first");
    if (seeded && !h->seeded) return fail(h, PICLES_ERR_STATE, "picles_seed must be called first");
    cudaError_t e = cudaSetDevice(h->device);
    if (e != cudaSuccess) return fail(h, PICLES_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
    return 0;
}

/* the wind level in the t1 slots is also the t level: the first step of a seeded or restored run reads it from both */
static int t_level_from_t1(picles_t* h) {
    const size_t bytes = (size_t)nodes(h) * 8;
    CK(cudaMemcpyAsync(h->A.u_t, h->A.u_t1, bytes, cudaMemcpyDeviceToDevice, h->stream));
    CK(cudaMemcpyAsync(h->A.v_t, h->A.v_t1, bytes, cudaMemcpyDeviceToDevice, h->stream));
    return PICLES_OK;
}

/* SeedParticle from the wind already in the t1 slots (the first step's t level, see picles_step) */
static int seed_from_t1(picles_t* h) {
    DeviceArrays& A = h->A;
    CK(cudaMemsetAsync(h->d_counters, 0, sizeof(DeviceCounters), h->stream));
    launch_seed(A, h->P, A.u_t1, A.v_t1, h->d_counters, h->sms, h->stream);
    CK(cudaGetLastError());
    int rc = t_level_from_t1(h);
    if (rc) return rc;
    CK(cudaMemcpyAsync(&h->h_counters->n_seed_off, &h->d_counters->n_seed_off, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->n_seed_off = h->h_counters->n_seed_off;
    h->steps_since_seed = 0;
    A.u_lag = A.v_lag = nullptr; /* the first step's t+DT level IS the lag level */
    A.n_mid = 0;
    h->seeded = true;
    h->winds_loaded = true;
    memset(&h->last, 0, sizeof h->last);
    return PICLES_OK;
}

int picles_seed(picles_t* h, const double* u0, const double* v0) {
    int rc = need_ready(h, false);
    if (rc) return rc;
    if (!u0 || !v0) return fail(h, PICLES_ERR_ARG, "picles_seed: wind arrays are required");
    DeviceArrays& A = h->A;
    int64_t n = nodes(h);
    /* stage the t=0 wind in the t1 slots: the first step's t level (see picles_step) */
    CK(cudaMemcpyAsync(A.u_t1, u0, (size_t)n * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(A.v_t1, v0, (size_t)n * 8, cudaMemcpyHostToDevice, h->stream));
    h->wm_t1_valid = false;
    return seed_from_t1(h);
}

/* intermediate wind levels of the next step (host planes -> device, consumed by the next advance) */
static int ensure_mid_planes(picles_t* h, int n_mid) {
    DeviceArrays& A = h->A;
    const int64_t n = nodes(h);
    for (int k = 0; k < n_mid; k++) {
        if (!A.u_mid[k]) { DALLOC(A.u_mid[k], n); DALLOC(A.v_mid[k], n); }
    }
    return PICLES_OK;
}
int picles_set_wind_midlevels(picles_t* h, int n_mid, const double* u_mid, const double* v_mid) {
    int rc = need_ready(h, true);
    if (rc) return rc;
    if (n_mid < 0 || n_mid > PICLES_WIND_MID_MAX) return fail(h, PICLES_ERR_ARG, "n_mid = %d outside 0..%d", n_mid, PICLES_WIND_MID_MAX);
    if (n_mid > 0 && (!u_mid || !v_mid)) return fail(h, PICLES_ERR_ARG, "picles_set_wind_midlevels: level arrays are required");
    DeviceArrays& A = h->A;
    rc = ensure_mid_planes(h, n_mid);
    if (rc) return rc;
    const int64_t n = nodes(h);
    /* same stream as the kernels: ordered after the previous step's advance, before the next one */
    for (int k = 0; k < n_mid; k++) {
        CK(cudaMemcpyAsync(A.u_mid[k], u_mid + (int64_t)k * n, (size_t)n * 8, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(A.v_mid[k], v_mid + (int64_t)k * n, (size_t)n * 8, cudaMemcpyHostToDevice, h->stream));
    }
    if (n_mid > 0) CK(cudaStreamSynchronize(h->stream)); /* the host arrays may be reused on return */
    A.n_mid = n_mid;
    return PICLES_OK;
}

/* host wind levels (null: not given) come as (u, v) pairs */
static int check_wind_pairs(picles_t* h, const double* u_t, const double* v_t, const double* u_t1, const double* v_t1) {
    if ((u_t == nullptr) != (v_t == nullptr) || (u_t1 == nullptr) != (v_t1 == nullptr))
        return fail(h, PICLES_ERR_ARG, "wind components must be given in pairs");
    return PICLES_OK;
}

/* the wind slots of the next step, of which the caller writes the t level (new_t) and the t+DT level (new_t1).  A new
   t+DT level without a new t level makes the previous step's t+DT level this step's t level: the slots are swapped,
   nothing is copied.  A written level is no longer the one picles_stage_wind_mesh sampled (wm_t1_valid). */
static void next_wind_levels(picles_t* h, bool new_t, bool new_t1) {
    DeviceArrays& A = h->A;
    if (new_t || new_t1) h->wm_t1_valid = false;
    if (!new_t && new_t1) {
        std::swap(A.u_t, A.u_t1);
        std::swap(A.v_t, A.v_t1);
    }
}

int picles_upload_winds(picles_t* h, const double* u_t, const double* v_t, const double* u_t1, const double* v_t1) {
    int rc = need_ready(h, true);
    if (rc) return rc;
    rc = check_wind_pairs(h, u_t, v_t, u_t1, v_t1);
    if (rc) return rc;
    DeviceArrays& A = h->A;
    size_t bytes = (size_t)nodes(h) * 8;
    next_wind_levels(h, u_t, u_t1);
    if (u_t) {
        CK(cudaMemcpyAsync(A.u_t, u_t, bytes, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(A.v_t, v_t, bytes, cudaMemcpyHostToDevice, h->stream));
    }
    if (u_t1) {
        CK(cudaMemcpyAsync(A.u_t1, u_t1, bytes, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(A.v_t1, v_t1, bytes, cudaMemcpyHostToDevice, h->stream));
    }
    return PICLES_OK;
}

/* B-1 as run (`on` frozen at seed, on_persist == 0): a particle seeded off never integrates, its integrator
   clock stays at 0 and advance! tests the wind at t_end = integ.t + DT = DT on every step
   (mapping_2D.jl:132,172-176).  That level is the first step's t+DT level: kept here, behind the first
   step's advance on the compute stream (by then every upload of the level has landed), and read by
   k_advance from the second step on.  Nothing is kept when every particle was seeded on. */
static int keep_lag_level(picles_t* h) {
    DeviceArrays& A = h->A;
    if (h->steps_since_seed != 0 || h->P.on_persist || h->n_seed_off == 0) return PICLES_OK;
    const int64_t n = nodes(h);
    if (!h->lag_u) { DALLOC(h->lag_u, n); DALLOC(h->lag_v, n); }
    CK(cudaMemcpyAsync(h->lag_u, A.u_t1, (size_t)n * 8, cudaMemcpyDeviceToDevice, h->stream));
    CK(cudaMemcpyAsync(h->lag_v, A.v_t1, (size_t)n * 8, cudaMemcpyDeviceToDevice, h->stream));
    A.u_lag = h->lag_u; A.v_lag = h->lag_v;
    return PICLES_OK;
}

/* ---- upload + advance, pipelined over row blocks -------------------------------------------
 * begin_advance: wind-level bookkeeping (same semantics as picles_upload_winds), counters and
 * per-row reach zeroed, start event.  advance_range: the host winds of each block of rows are copied on
 * the copy stream and the advance of those rows starts as soon as they have landed, so block c
 * integrates while block c+1 is still in flight. */
static int begin_advance(picles_t* h, double dt_model, const double* u_t, const double* v_t, const double* u_t1,
                         const double* v_t1) {
    int rc = check_wind_pairs(h, u_t, v_t, u_t1, v_t1);
    if (rc) return rc;
    if (!(dt_model > 0)) return fail(h, PICLES_ERR_ARG, "dt_model must be positive");
    next_wind_levels(h, u_t, u_t1);
    CK(cudaMemsetAsync(h->d_counters, 0, sizeof(DeviceCounters), h->stream));
    CK(cudaMemsetAsync(h->A.rowreach, 0, (size_t)record_rows(h) * 4, h->stream));
    if (u_t || u_t1) {
        /* the copy stream may only overwrite the wind planes once the compute stream is past
           every earlier kernel that read them */
        CK(cudaEventRecord(h->pev[PIPE_EVENTS - 1], h->stream));
        CK(cudaStreamWaitEvent(h->copy_stream, h->pev[PIPE_EVENTS - 1], 0));
    }
    CK(cudaEventRecord(h->ev[0], h->stream));
    h->timing_valid = false;
    return PICLES_OK;
}
/* host winds of rows [r0, r1) onto the device on the copy stream; `consumer` waits until they have landed */
static int upload_rows(picles_t* h, const double* u_t, const double* v_t, const double* u_t1, const double* v_t1, int r0,
                       int r1, cudaEvent_t landed, cudaStream_t consumer) {
    DeviceArrays& A = h->A;
    if (r0 >= r1 || !(u_t || u_t1)) return PICLES_OK;
    const int64_t off = (int64_t)r0 * A.Nx;
    const size_t bytes = (size_t)(r1 - r0) * A.Nx * 8;
    if (u_t) {
        CK(cudaMemcpyAsync(A.u_t + off, u_t + off, bytes, cudaMemcpyHostToDevice, h->copy_stream));
        CK(cudaMemcpyAsync(A.v_t + off, v_t + off, bytes, cudaMemcpyHostToDevice, h->copy_stream));
    }
    if (u_t1) {
        CK(cudaMemcpyAsync(A.u_t1 + off, u_t1 + off, bytes, cudaMemcpyHostToDevice, h->copy_stream));
        CK(cudaMemcpyAsync(A.v_t1 + off, v_t1 + off, bytes, cudaMemcpyHostToDevice, h->copy_stream));
    }
    CK(cudaEventRecord(landed, h->copy_stream));
    CK(cudaStreamWaitEvent(consumer, landed, 0));
    return PICLES_OK;
}
/* rows [r0, r1), block c on work queue c.  Graded blocks when host winds are uploaded and the range has at least
   PIPE_MIN_NODES nodes, one block otherwise: 64 rows first, each next block three times the one before (an upload
   takes about a third of the advance of the same rows, so it still hides), the last takes the rest.  Only the first
   block's upload is exposed: 0.08 ms instead of the 0.6 ms of eight equal blocks at 4096^2 (end to end 16.39 -> 15.76
   ms per step, profiles/README.md). */
static int advance_range(picles_t* h, double dt_model, const double* u_t, const double* v_t, const double* u_t1,
                         const double* v_t1, int r0, int r1) {
    const DeviceArrays& A = h->A;
    const bool graded = (u_t || u_t1) && (int64_t)(r1 - r0) * A.Nx >= PIPE_MIN_NODES;
    int a = r0, len = 64;
    for (int c = 0; c < PIPE_CHUNKS && a < r1; c++) {
        const int b = (!graded || c == PIPE_CHUNKS - 1 || a + len >= r1) ? r1 : a + len;
        int rc = upload_rows(h, u_t, v_t, u_t1, v_t1, a, b, h->pev[c], h->stream);
        if (rc) return rc;
        const int64_t l_end = (int64_t)b * A.Nx;
        launch_advance(A, h->P, dt_model, h->d_counters, h->sms, h->stream, (int64_t)a * A.Nx, l_end, l_end, l_end, c);
        a = b; len *= 3;
    }
    return PICLES_OK;
}
/* the rows of every member: an ensemble's particle-side planes are one plane of members*ny rows */
static int upload_and_advance(picles_t* h, double dt_model, const double* u_t, const double* v_t, const double* u_t1,
                              const double* v_t1) {
    int rc = begin_advance(h, dt_model, u_t, v_t, u_t1, v_t1);
    if (rc) return rc;
    rc = advance_range(h, dt_model, u_t, v_t, u_t1, v_t1, 0, h->A.ny * h->A.members);
    if (rc) return rc;
    CK(cudaEventRecord(h->ev[1], h->stream));
    CK(cudaGetLastError());
    return keep_lag_level(h);
}

int picles_step_advance(picles_t* h, double t, double dt_model) {
    int rc = need_ready(h, true);
    if (rc) return rc;
    (void)t;
    return upload_and_advance(h, dt_model, nullptr, nullptr, nullptr, nullptr);
}

int picles_get_reach(picles_t* h, int32_t* reach) {
    int rc = need_ready(h, true);
    if (rc) return rc;
    CK(cudaMemcpyAsync(&h->h_counters->reach, &h->d_counters->reach, sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    *reach = h->h_counters->reach;
    return PICLES_OK;
}

/* bytes of one halo message: hx rows of the five record planes and the cell plane */
static int64_t halo_msg_bytes(const picles_t* h) { return (int64_t)h->A.hx * h->A.rp * (5 * 8 + 4); }

int picles_halo_rows(picles_t* h, int* rows_exchanged, int* rows_max) {
    if (!h || !h->have_grid) return fail(h, PICLES_ERR_STATE, "grid not set");
    REFUSE_MEMBERS(h, "picles_halo_rows");
    if (rows_exchanged) *rows_exchanged = h->A.hx;
    if (rows_max) *rows_max = h->A.halo;
    return PICLES_OK;
}

int picles_halo_widen(picles_t* h, int rows) {
    if (!h || !h->have_grid) return fail(h, PICLES_ERR_STATE, "grid not set");
    REFUSE_MEMBERS(h, "picles_halo_widen");
    if (rows <= h->A.hx) return PICLES_OK; /* never narrowed: rows beyond hx would keep stale records */
    if (rows > h->A.halo)
        return fail(h, PICLES_ERR_HALO, "a halo of %d rows is asked for; this strip (%d rows) can exchange at most %d", rows, h->A.ny, h->A.halo);
    h->A.hx = rows;
    return PICLES_OK;
}

int picles_set_global_reach(picles_t* h, int reach) {
    int rc = need_ready(h, true);
    if (rc) return rc;
    if (reach < 0) return fail(h, PICLES_ERR_ARG, "negative reach");
    h->reach_all_host = reach + 1; /* 0 means "not set" to the gather */
    CK(cudaMemcpyAsync(&h->d_counters->reach_all, &h->reach_all_host, sizeof(int32_t), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return PICLES_OK;
}

int picles_get_row_reach(picles_t* h, int32_t* reach_rows) {
    int rc = need_ready(h, true);
    if (rc) return rc;
    if (!reach_rows) return fail(h, PICLES_ERR_ARG, "null output");
    const DeviceArrays& A = h->A;
    /* an ensemble has no halo rows: its members' rows are back to back */
    CK(cudaMemcpyAsync(reach_rows, A.rowreach + A.halo, (size_t)A.ny * A.members * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return PICLES_OK;
}

int picles_halo_buffers(picles_t* h, void** send_lo, void** send_hi, void** recv_lo, void** recv_hi, int64_t* nbytes) {
    if (!h || !h->have_grid) return fail(h, PICLES_ERR_STATE, "grid not set");
    REFUSE_MEMBERS(h, "picles_halo_buffers");
    if (send_lo) *send_lo = h->send_lo;
    if (send_hi) *send_hi = h->send_hi;
    if (recv_lo) *recv_lo = h->recv_lo;
    if (recv_hi) *recv_hi = h->recv_hi;
    if (nbytes) *nbytes = halo_msg_bytes(h);
    return PICLES_OK;
}

int picles_halo_pack(picles_t* h) {
    int rc = need_ready(h, true);
    if (rc) return rc;
    REFUSE_MEMBERS(h, "picles_halo_pack");
    launch_halo_pack(h->A, h->send_lo, h->send_hi, h->sms, h->stream);
    CK(cudaGetLastError());
    return PICLES_OK;
}

int picles_halo_unpack(picles_t* h) {
    int rc = need_ready(h, true);
    if (rc) return rc;
    REFUSE_MEMBERS(h, "picles_halo_unpack");
    launch_halo_unpack(h->A, h->recv_lo, h->recv_hi, h->d_counters, h->sms, h->stream);
    CK(cudaGetLastError());
    return PICLES_OK;
}

static int finish_counters(picles_t* h) {
    CK(cudaMemcpyAsync(h->h_counters, h->d_counters, sizeof(DeviceCounters), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    const DeviceCounters& d = *h->h_counters;
    picles_counters_t& c = h->last;
    c.n_integrated = (int64_t)d.sums[0]; c.n_substeps = (int64_t)d.sums[1]; c.n_rejects = (int64_t)d.sums[2];
    c.n_rhs = (int64_t)d.sums[3]; c.n_reseed_advance = (int64_t)d.sums[4]; c.n_fixups = (int64_t)d.sums[5];
    c.n_failed = (int64_t)d.sums[6]; c.n_deposited = (int64_t)d.sums[7];
    c.n_remesh_A = (int64_t)d.sums[8]; c.n_remesh_B = (int64_t)d.sums[9]; c.n_remesh_C = (int64_t)d.sums[10];
    c.n_remesh_D = (int64_t)d.sums[11];
    c.n_stiff_switches = (int64_t)d.sums[12]; c.n_stiff_attempts = (int64_t)d.sums[13];
    c.n_active = c.n_remesh_A + c.n_remesh_B + c.n_remesh_C + c.n_remesh_D;
    c.reach = d.reach; c.max_attempts = d.max_attempts;
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, h->ev[0], h->ev[1])); c.ms_advance = ms;
    CK(cudaEventElapsedTime(&ms, h->ev[2], h->ev[3])); c.ms_project = ms;
    CK(cudaEventElapsedTime(&ms, h->ev[3], h->ev[4])); c.ms_remesh = ms;
    h->timing_valid = true;
    return PICLES_OK;
}

/* tile geometry of the gather for this step, guessed from the previous step's reach */
static int wide_tiles(const picles_t* h) { return h->last.reach > PR_HY_NARROW && h->last.reach <= PR_HY_WIDE; }

/* gather + remesh, counters read back (the one host synchronisation of a step).  *need = 0, or — on a strip whose
   deposits reach further than the hx rows that were exchanged — the rows needed: the kernel then changed nothing
   (k_project_remesh) and the caller repeats exchange and gather with wider rows, or reports PICLES_ERR_HALO */
static int project_remesh_once(picles_t* h, double dt_model, int* need) {
    *need = 0;
    /* a halo exchange may have run since the advance: ms_project brackets the gather alone */
    CK(cudaEventRecord(h->ev[2], h->stream));
    launch_project_remesh(h->maps, h->A, h->P, dt_model, h->P.periodic_boundary ? 2 : 1, h->accumulate, wide_tiles(h), h->d_counters, h->stream);
    CK(cudaEventRecord(h->ev[3], h->stream));
    CK(cudaEventRecord(h->ev[4], h->stream));
    CK(cudaGetLastError());
    int rc = finish_counters(h);
    if (rc) return rc;
    if (h->A.ny != h->A.Ny && h->h_counters->halo_short > 0) {
        *need = h->h_counters->halo_short;
        CK(cudaMemsetAsync(&h->d_counters->halo_short, 0, sizeof(int32_t), h->stream));
        return PICLES_OK;
    }
    h->A.n_mid = 0; /* intermediate wind levels are consumed by one step */
    h->steps_since_seed++;
    if (h->last.reach > PH_REACH_MAX_ABI)
        return fail(h, PICLES_ERR_HALO, "particle reach %d cells exceeds the supported reach %d", h->last.reach, PH_REACH_MAX_ABI);
    return PICLES_OK;
}

int picles_step_project_remesh(picles_t* h, double t, double dt_model) {
    int rc = need_ready(h, true);
    if (rc) return rc;
    (void)t;
    int need = 0;
    rc = project_remesh_once(h, dt_model, &need);
    if (rc) return rc;
    if (need > 0)
        return fail(h, PICLES_ERR_HALO, "deposits reach %d rows but %d halo rows were exchanged; nothing was changed: "
                    "picles_halo_widen(%d) on every strip, then repeat the exchange and this call", need, h->A.hx, need);
    return PICLES_OK;
}

int picles_step(picles_t* h, double t, double dt_model, const double* u_t, const double* v_t, const double* u_t1,
                const double* v_t1) {
    int rc = need_ready(h, true);
    if (rc) return rc;
    (void)t;
    if (h->A.ny != h->A.Ny)
        return fail(h, PICLES_ERR_STATE, "picles_step needs a single-strip handle; use the phase-split calls for strips");
    rc = upload_and_advance(h, dt_model, u_t, v_t, u_t1, v_t1);
    if (rc) return rc;
    int need = 0;
    return project_remesh_once(h, dt_model, &need);
}

int picles_synchronize(picles_t* h) {
    if (!h) return fail(nullptr, PICLES_ERR_ARG, "null handle");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    return PICLES_OK;
}

int picles_get_state(picles_t* h, double* S) {
    int rc = need_ready(h, false);
    if (rc) return rc;
    if (!S) return fail(h, PICLES_ERR_ARG, "null output");
    int64_t n = nodes(h);
    for (int k = 0; k < 3; k++) CK(cudaMemcpyAsync(S + k * n, h->A.S[k], (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return PICLES_OK;
}

int picles_set_state(picles_t* h, const double* S) {
    int rc = need_ready(h, false);
    if (rc) return rc;
    if (!S) return fail(h, PICLES_ERR_ARG, "null input");
    int64_t n = nodes(h);
    for (int k = 0; k < 3; k++) CK(cudaMemcpyAsync(h->A.S[k], S + k * n, (size_t)n * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return PICLES_OK;
}

int picles_get_particles(picles_t* h, double* z, double* t, double* dt, uint8_t* flags, int32_t* status) {
    int rc = need_ready(h, true);
    if (rc) return rc;
    const DeviceArrays& A = h->A;
    int64_t n = nodes(h);
    if (z) for (int k = 0; k < 5; k++) CK(cudaMemcpyAsync(z + k * n, A.z[k], (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
    if (t) CK(cudaMemcpyAsync(t, A.t, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
    if (dt) CK(cudaMemcpyAsync(dt, A.dt, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
    if (flags) CK(cudaMemcpyAsync(flags, A.flags, (size_t)n, cudaMemcpyDeviceToHost, h->stream));
    std::vector<uint8_t> st8;
    if (status) {
        st8.resize((size_t)n);
        CK(cudaMemcpyAsync(st8.data(), A.status, (size_t)n, cudaMemcpyDeviceToHost, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    if (status) for (int64_t l = 0; l < n; l++) status[l] = st8[(size_t)l];
    return PICLES_OK;
}

int picles_get_solver_state(picles_t* h, int8_t* as) {
    int rc = need_ready(h, false);
    if (rc) return rc;
    if (!as) return fail(h, PICLES_ERR_ARG, "null output");
    CK(cudaMemcpyAsync(as, h->A.as, (size_t)nodes(h), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return PICLES_OK;
}

int picles_get_counters(picles_t* h, picles_counters_t* c) {
    if (!h || !c) return fail(h, PICLES_ERR_ARG, "null argument");
    *c = h->last;
    return PICLES_OK;
}

int picles_get_attempt_histogram(picles_t* h, int64_t* hist, int nbins) {
    if (!h || !hist || nbins < 1) return fail(h, PICLES_ERR_ARG, "picles_get_attempt_histogram: bad argument");
    if (!h->timing_valid) return fail(h, PICLES_ERR_STATE, "no completed step to report");
    for (int k = 0; k < nbins; k++) hist[k] = 0;
    for (int k = 0; k < ADV_HIST_BINS; k++) hist[k < nbins ? k : nbins - 1] += (int64_t)h->h_counters->attempt_hist[k];
    return PICLES_OK;
}

int64_t picles_launch_count(void) { return (int64_t)launch_count(); }

/* the energy sum of each of `groups` planes of n values of State[0], back to back, by a deterministic two-stage
   reduction: ENERGY_BLOCKS partial sums per plane on the device (d_part), added on the host in block order (h_part) */
static int energy_sums(picles_t* h, int64_t n, int groups, double* d_part, double* h_part, double* sums) {
    launch_energy(h->A.S[0], n, groups, d_part, ENERGY_BLOCKS, h->stream);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h_part, d_part, (size_t)groups * ENERGY_BLOCKS * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (int m = 0; m < groups; m++) {
        double s = 0.0;
        for (int k = 0; k < ENERGY_BLOCKS; k++) s += h_part[(int64_t)m * ENERGY_BLOCKS + k];
        sums[m] = s;
    }
    return PICLES_OK;
}

int picles_state_energy_sum(picles_t* h, double* sum_e) {
    int rc = need_ready(h, false);
    if (rc) return rc;
    if (!sum_e) return fail(h, PICLES_ERR_ARG, "null output");
    return energy_sums(h, nodes(h), 1, h->d_partial, h->h_partial, sum_e);
}

int picles_member_energy_sums(picles_t* h, double* sums) {
    int rc = need_ready(h, false);
    if (rc) return rc;
    if (!sums) return fail(h, PICLES_ERR_ARG, "null output");
    /* each member's plane is reduced as picles_state_energy_sum reduces a single model's, so that sums[m] is what a
       single-member handle with member m's State returns */
    const int E = h->A.members;
    if (!h->d_member_partial) DALLOC(h->d_member_partial, (int64_t)E * ENERGY_BLOCKS);
    if (!h->h_member_partial) CK(cudaMallocHost((void**)&h->h_member_partial, (size_t)E * ENERGY_BLOCKS * sizeof(double)));
    return energy_sums(h, (int64_t)h->A.Nx * h->A.ny, E, h->d_member_partial, h->h_member_partial, sums);
}

int picles_state_dev(picles_t* h, double** S_dev) {
    if (!h || !h->have_grid || !S_dev) return fail(h, PICLES_ERR_STATE, "grid not set");
    /* the three State planes are separate allocations: return them as 3 pointers */
    S_dev[0] = h->A.S[0]; S_dev[1] = h->A.S[1]; S_dev[2] = h->A.S[2];
    return PICLES_OK;
}

int picles_wind_dev(picles_t* h, double** u_t, double** v_t, double** u_t1, double** v_t1) {
    if (!h || !h->have_grid) return fail(h, PICLES_ERR_STATE, "grid not set");
    if (u_t) *u_t = h->A.u_t;
    if (v_t) *v_t = h->A.v_t;
    if (u_t1) *u_t1 = h->A.u_t1;
    if (v_t1) *v_t1 = h->A.v_t1;
    return PICLES_OK;
}

int picles_set_option(picles_t* h, int option, int value) {
    if (!h) return fail(nullptr, PICLES_ERR_ARG, "null handle");
    switch (option) {
        case PICLES_OPT_ACCUMULATE_STATE: h->accumulate = value ? 1 : 0; return PICLES_OK;
        default: return fail(h, PICLES_ERR_ARG, "unknown option %d", option);
    }
}

int picles_zero_state(picles_t* h) {
    int rc = need_ready(h, false);
    if (rc) return rc;
    int64_t n = nodes(h);
    for (int k = 0; k < 3; k++) CK(cudaMemsetAsync(h->A.S[k], 0, (size_t)n * 8, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return PICLES_OK;
}

int picles_copy_dev(picles_t* h, void* dst, const void* src, int64_t nbytes) {
    if (!h || !dst || !src || nbytes < 0) return fail(h, PICLES_ERR_ARG, "picles_copy_dev: bad argument");
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpyAsync(dst, src, (size_t)nbytes, cudaMemcpyDefault, h->stream));
    return PICLES_OK;
}

int picles_timer_start(picles_t* h) {
    if (!h) return fail(nullptr, PICLES_ERR_ARG, "null handle");
    CK(cudaSetDevice(h->device));
    CK(cudaEventRecord(h->tev[0], h->stream));
    return PICLES_OK;
}

int picles_timer_stop(picles_t* h, double* ms) {
    if (!h || !ms) return fail(h, PICLES_ERR_ARG, "null argument");
    CK(cudaSetDevice(h->device));
    CK(cudaEventRecord(h->tev[1], h->stream));
    CK(cudaEventSynchronize(h->tev[1]));
    float f = 0.f;
    CK(cudaEventElapsedTime(&f, h->tev[0], h->tev[1]));
    *ms = f;
    return PICLES_OK;
}

int picles_selftest_math(picles_t* h, uint64_t seed, int iters, int64_t* out6) {
    if (!h || !out6 || iters < 1) return fail(h, PICLES_ERR_ARG, "bad argument");
    CK(cudaSetDevice(h->device));
    unsigned long long* d = nullptr;
    CK(cudaMalloc((void**)&d, 6 * sizeof(unsigned long long)));
    CK(cudaMemsetAsync(d, 0, 6 * sizeof(unsigned long long), h->stream));
    launch_selftest_math(seed, iters, d, h->sms, h->stream);
    unsigned long long hbuf[6];
    cudaError_t e = cudaMemcpyAsync(hbuf, d, sizeof hbuf, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    cudaFree(d);
    if (e != cudaSuccess) return fail(h, PICLES_ERR_CUDA, "selftest: %s", cudaGetErrorString(e));
    for (int k = 0; k < 6; k++) out6[k] = (int64_t)hbuf[k];
    return PICLES_OK;
}

int picles_measure_fp64_peak(picles_t* h, double* tflops) {
    if (!h || !tflops) return fail(h, PICLES_ERR_ARG, "null argument");
    CK(cudaSetDevice(h->device));
    int64_t fmas = 0;
    double best = 0.0;
    launch_fp64_peak(h->d_partial, 256, h->sms, h->stream, &fmas); /* warm-up */
    CK(cudaStreamSynchronize(h->stream));
    for (int rep = 0; rep < 5; rep++) {
        CK(cudaEventRecord(h->tev[0], h->stream));
        launch_fp64_peak(h->d_partial, 4096, h->sms, h->stream, &fmas);
        CK(cudaEventRecord(h->tev[1], h->stream));
        CK(cudaEventSynchronize(h->tev[1]));
        CK(cudaGetLastError());
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, h->tev[0], h->tev[1]));
        double tf = 2.0 * (double)fmas / (ms * 1e-3) / 1e12;
        if (tf > best) best = tf;
    }
    *tflops = best;
    return PICLES_OK;
}

int picles_measure_hbm_copy(picles_t* h, int mib, double* gbs) {
    if (!h || !gbs || mib < 1) return fail(h, PICLES_ERR_ARG, "bad argument");
    CK(cudaSetDevice(h->device));
    int64_t n = (int64_t)mib * 1024 * 1024 / 8;
    double *a = nullptr, *b = nullptr;
    if (cudaMalloc((void**)&a, (size_t)n * 8) != cudaSuccess || cudaMalloc((void**)&b, (size_t)n * 8) != cudaSuccess) {
        if (a) cudaFree(a);
        return fail(h, PICLES_ERR_ALLOC, "cannot allocate 2 x %d MiB", mib);
    }
    cudaMemsetAsync(a, 0, (size_t)n * 8, h->stream);
    double best = 0.0;
    for (int rep = 0; rep < 6; rep++) {
        cudaEventRecord(h->tev[0], h->stream);
        launch_copy_f64(b, a, n, h->sms, h->stream);
        cudaEventRecord(h->tev[1], h->stream);
        cudaEventSynchronize(h->tev[1]);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, h->tev[0], h->tev[1]);
        double g = 2.0 * (double)n * 8 / (ms * 1e-3) / 1e9;
        if (rep > 0 && g > best) best = g;
    }
    cudaFree(a);
    cudaFree(b);
    CK(cudaGetLastError());
    *gbs = best;
    return PICLES_OK;
}

/* ---- output path ------------------------------------------------------------------------ */
int picles_get_fields(picles_t* h, double* Hs, double* c_x, double* c_y) {
    int rc = need_ready(h, false);
    if (rc) return rc;
    const DeviceArrays& A = h->A;
    const int64_t n = nodes(h);
    const int nout = (Hs != nullptr) + (c_x != nullptr) + (c_y != nullptr);
    if (nout == 0) return PICLES_OK;
    double* d = nullptr;
    if (cudaMalloc((void**)&d, (size_t)n * 8 * nout) != cudaSuccess) return fail(h, PICLES_ERR_ALLOC, "cannot allocate the field planes");
    double* p = d;
    double* dHs = Hs ? p : nullptr; if (Hs) p += n;
    double* dcx = c_x ? p : nullptr; if (c_x) p += n;
    double* dcy = c_y ? p : nullptr;
    launch_fields(n, A.S[0], A.S[1], A.S[2], dHs, dcx, dcy, h->sms, h->stream);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess && Hs) e = cudaMemcpyAsync(Hs, dHs, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess && c_x) e = cudaMemcpyAsync(c_x, dcx, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess && c_y) e = cudaMemcpyAsync(c_y, dcy, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    cudaFree(d);
    if (e != cudaSuccess) return fail(h, PICLES_ERR_CUDA, "picles_get_fields: %s", cudaGetErrorString(e));
    return PICLES_OK;
}

int picles_host_alloc(void** p, int64_t nbytes) {
    picles_t* h = nullptr;
    if (!p || nbytes < 1) return fail(nullptr, PICLES_ERR_ARG, "picles_host_alloc: bad argument");
    CK(cudaMallocHost(p, (size_t)nbytes));
    return PICLES_OK;
}
int picles_host_free(void* p) {
    picles_t* h = nullptr;
    if (p) CK(cudaFreeHost(p));
    return PICLES_OK;
}

/* State snapshot that does not stall the stepping: a device-to-device copy into a staging
   buffer on the compute stream (ordered before the next step overwrites State), then the
   device-to-host copy on the copy stream while the next steps run. */
int picles_snapshot_begin(picles_t* h, double* S_host) {
    int rc = need_ready(h, false);
    if (rc) return rc;
    if (!S_host) return fail(h, PICLES_ERR_ARG, "null output");
    if (h->snap_pending) {
        rc = picles_snapshot_wait(h);
        if (rc) return rc;
    }
    const int64_t n = nodes(h);
    if (!h->snap) DALLOC(h->snap, 3 * n);
    for (int k = 0; k < 3; k++)
        CK(cudaMemcpyAsync(h->snap + k * n, h->A.S[k], (size_t)n * 8, cudaMemcpyDeviceToDevice, h->stream));
    CK(cudaEventRecord(h->snap_ev[0], h->stream));
    CK(cudaStreamWaitEvent(h->snap_stream, h->snap_ev[0], 0));
    CK(cudaMemcpyAsync(S_host, h->snap, (size_t)n * 8 * 3, cudaMemcpyDeviceToHost, h->snap_stream));
    CK(cudaEventRecord(h->snap_ev[1], h->snap_stream));
    h->snap_pending = true;
    return PICLES_OK;
}
int picles_snapshot_wait(picles_t* h) {
    if (!h) return fail(nullptr, PICLES_ERR_ARG, "null handle");
    if (!h->snap_pending) return PICLES_OK;
    CK(cudaSetDevice(h->device));
    CK(cudaEventSynchronize(h->snap_ev[1]));
    h->snap_pending = false;
    return PICLES_OK;
}

/* ---- checkpoint / resume ------------------------------------------------------------------
 * The particle planes (u[5], t, dt, qold, iter, flags, status), the node State and the wind
 * level that the next step takes as its t level are the complete state of the path (the
 * reference has no checkpointing: run!(…; pickup=false) is unused, run.jl:36).  Layout of the
 * blob: a 64-byte header {magic, version, Nx, ny, j0, Ny, bx, by, halo, n_bytes} then the planes in
 * the order below, each ny*Nx elements. */
struct CkptHeader {
    uint64_t magic;
    int32_t version, Nx, ny, j0, Ny, bx, by, halo;
    int64_t n_bytes;
    uint64_t params_hash; /* FNV-1a of the picles_params_t the run was made with */
    uint64_t clock;       /* bit 0: the lag wind level follows the planes; bits 1..32: particles seeded off; bits 33..: steps since the seed */
};
static_assert(sizeof(CkptHeader) == 64, "checkpoint header layout");
#define CKPT_MAGIC 0x50694342323030ull /* "PiCB200" */

static uint64_t params_hash(const picles_params_t& P) {
    /* the two runs of fields around the padding word behind has_defaults (and the one at the tail) */
    const unsigned char* b = (const unsigned char*)&P;
    const size_t span[2][2] = {{0, offsetof(picles_params_t, has_defaults) + sizeof(int32_t)},
                               {offsetof(picles_params_t, defaults), offsetof(picles_params_t, nan_eest_rejects) + sizeof(int32_t)}};
    uint64_t hsh = 1469598103934665603ull;
    for (int r = 0; r < 2; r++)
        for (size_t k = span[r][0]; k < span[r][1]; k++) { hsh ^= b[k]; hsh *= 1099511628211ull; }
    return hsh;
}
static int64_t ckpt_bytes(const picles_t* h, bool with_lag) {
    const int64_t n = (int64_t)h->A.Nx * h->A.ny;
    return (int64_t)sizeof(CkptHeader) + n * (8 * (5 + 3 + 3 + 2 + (with_lag ? 2 : 0)) + 4 + 1 + 1 + 1);
}
int picles_checkpoint_size(picles_t* h, int64_t* nbytes) {
    if (!h || !h->have_grid || !nbytes) return fail(h, PICLES_ERR_STATE, "grid not set");
    REFUSE_MEMBERS(h, "picles_checkpoint_size");
    *nbytes = ckpt_bytes(h, h->A.u_lag != nullptr);
    return PICLES_OK;
}
/* the planes of a checkpoint, in blob order */
static int ckpt_planes(picles_t* h, bool with_lag, void** ptr, size_t* bytes) {
    DeviceArrays& A = h->A;
    const size_t n = (size_t)A.Nx * A.ny;
    int k = 0;
    for (int c = 0; c < 5; c++) { ptr[k] = A.z[c]; bytes[k++] = n * 8; }
    ptr[k] = A.t; bytes[k++] = n * 8;
    ptr[k] = A.dt; bytes[k++] = n * 8;
    ptr[k] = A.qold; bytes[k++] = n * 8;
    for (int c = 0; c < 3; c++) { ptr[k] = A.S[c]; bytes[k++] = n * 8; }
    ptr[k] = A.u_t1; bytes[k++] = n * 8; /* becomes the t level of the next step */
    ptr[k] = A.v_t1; bytes[k++] = n * 8;
    ptr[k] = A.iter; bytes[k++] = n * 4;
    ptr[k] = A.flags; bytes[k++] = n;
    ptr[k] = A.status; bytes[k++] = n;
    ptr[k] = A.as; bytes[k++] = n;
    if (with_lag) {
        ptr[k] = h->lag_u; bytes[k++] = n * 8;
        ptr[k] = h->lag_v; bytes[k++] = n * 8;
    }
    return k;
}
int picles_checkpoint_save(picles_t* h, void* blob, int64_t nbytes) {
    int rc = need_ready(h, true);
    if (rc) return rc;
    REFUSE_MEMBERS(h, "picles_checkpoint_save");
    const DeviceArrays& A = h->A;
    /* intermediate wind levels staged for the next step are not part of the blob: a run resumed from it
       would integrate that step against two levels only */
    if (A.n_mid > 0) return fail(h, PICLES_ERR_STATE, "%d intermediate wind levels are staged for the next step; checkpoint before picles_set_wind_midlevels or after the step", A.n_mid);
    const bool with_lag = A.u_lag != nullptr;
    if (!blob || nbytes < ckpt_bytes(h, with_lag)) return fail(h, PICLES_ERR_ARG, "checkpoint buffer too small (%lld < %lld bytes)", (long long)nbytes, (long long)ckpt_bytes(h, with_lag));
    CkptHeader hd = {CKPT_MAGIC, PICLES_ABI_VERSION, A.Nx, A.ny, A.j0, A.Ny, A.bx, A.by, A.halo, ckpt_bytes(h, with_lag), params_hash(h->P),
                     (uint64_t)(with_lag ? 1 : 0) | ((uint64_t)(uint32_t)h->n_seed_off << 1) | ((uint64_t)h->steps_since_seed << 33)};
    memcpy(blob, &hd, sizeof hd);
    void* ptr[24];
    size_t bytes[24];
    const int np = ckpt_planes(h, with_lag, ptr, bytes);
    char* out = (char*)blob + sizeof hd;
    for (int k = 0; k < np; k++) {
        CK(cudaMemcpyAsync(out, ptr[k], bytes[k], cudaMemcpyDeviceToHost, h->stream));
        out += bytes[k];
    }
    CK(cudaStreamSynchronize(h->stream));
    return PICLES_OK;
}
/* the handle must have the same grid (picles_set_grid*) and parameters (picles_set_params) as the one that saved:
   both are checked */
int picles_checkpoint_load(picles_t* h, const void* blob, int64_t nbytes) {
    int rc = need_ready(h, false);
    if (rc) return rc;
    REFUSE_MEMBERS(h, "picles_checkpoint_load");
    if (!blob || nbytes < (int64_t)sizeof(CkptHeader)) return fail(h, PICLES_ERR_ARG, "not a checkpoint");
    CkptHeader hd;
    memcpy(&hd, blob, sizeof hd);
    DeviceArrays& A = h->A;
    if (hd.magic != CKPT_MAGIC || hd.version != PICLES_ABI_VERSION) return fail(h, PICLES_ERR_ARG, "not a checkpoint of this library version");
    if (hd.Nx != A.Nx || hd.ny != A.ny || hd.j0 != A.j0 || hd.Ny != A.Ny || hd.bx != A.bx || hd.by != A.by)
        return fail(h, PICLES_ERR_ARG, "checkpoint is for a %dx%d strip at row %d of %d; this handle owns %dx%d at row %d of %d", hd.Nx,
                    hd.ny, hd.j0, hd.Ny, A.Nx, A.ny, A.j0, A.Ny);
    if (hd.params_hash != params_hash(h->P))
        return fail(h, PICLES_ERR_ARG, "checkpoint was written with different parameters (picles_set_params): solver state, tolerances "
                                       "and switches would not match the restored particles");
    const bool with_lag = (hd.clock & 1u) != 0;
    if (nbytes < hd.n_bytes || hd.n_bytes != ckpt_bytes(h, with_lag)) return fail(h, PICLES_ERR_ARG, "truncated checkpoint");
    const int64_t n = (int64_t)A.Nx * A.ny;
    if (with_lag && !h->lag_u) { DALLOC(h->lag_u, n); DALLOC(h->lag_v, n); }
    void* ptr[24];
    size_t bytes[24];
    const int np = ckpt_planes(h, with_lag, ptr, bytes);
    const char* in = (const char*)blob + sizeof hd;
    for (int k = 0; k < np; k++) {
        CK(cudaMemcpyAsync(ptr[k], in, bytes[k], cudaMemcpyHostToDevice, h->stream));
        in += bytes[k];
    }
    /* no deposit records are carried over: every step rewrites them before they are read */
    const int64_t ne = (int64_t)A.rp * (A.ny + 2 * A.halo);
    launch_fill_i32(A.cell, ne, -1, h->sms, h->stream);
    rc = t_level_from_t1(h);
    if (rc) return rc;
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
    A.u_lag = with_lag ? h->lag_u : nullptr;
    A.v_lag = with_lag ? h->lag_v : nullptr;
    h->n_seed_off = (int32_t)((hd.clock >> 1) & 0xffffffffu);
    h->steps_since_seed = (int64_t)(hd.clock >> 33);
    h->seeded = true;
    h->winds_loaded = true;
    h->wm_t1_valid = false;
    h->A.n_mid = 0;
    memset(&h->last, 0, sizeof h->last);
    return PICLES_OK;
}

/* ---- strip communicator: halo exchange over NVLink inside the library ----------------- */
int picles_comm_unique_id(char* id128, const char* nccl_path) {
    picles_t* h = nullptr;
    if (!id128) return fail(nullptr, PICLES_ERR_ARG, "null id buffer");
    int rc = nccl_load(nullptr, nccl_path);
    if (rc) return rc;
    pk_nccl_id_t id;
    NCK(g_nccl.get_id(&id));
    memcpy(id128, id.internal, sizeof id.internal);
    return PICLES_OK;
}

int picles_comm_init(picles_t* h, const char* id128, int rank, int nranks, const char* nccl_path) {
    if (!h || !id128) return fail(h, PICLES_ERR_ARG, "null argument");
    REFUSE_MEMBERS(h, "picles_comm_init");
    if (nranks < 1 || rank < 0 || rank >= nranks) return fail(h, PICLES_ERR_ARG, "bad rank %d of %d", rank, nranks);
    if (h->comm) return fail(h, PICLES_ERR_STATE, "communicator already initialised");
    int rc = nccl_load(h, nccl_path);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    pk_nccl_id_t id;
    memcpy(id.internal, id128, sizeof id.internal);
    NCK(g_nccl.init_rank(&h->comm, nranks, id, rank));
    h->comm_rank = rank;
    h->comm_size = nranks;
    return PICLES_OK;
}

int picles_comm_destroy(picles_t* h) {
    if (!h) return fail(nullptr, PICLES_ERR_ARG, "null handle");
    REFUSE_MEMBERS(h, "picles_comm_destroy");
    if (h->comm) {
        cudaSetDevice(h->device);
        cudaStreamSynchronize(h->stream);
        NCK(g_nccl.destroy(h->comm));
        h->comm = nullptr;
        h->comm_rank = -1;
        h->comm_size = 0;
    }
    return PICLES_OK;
}

/* pack -> grouped ncclSend/ncclRecv with the two y-neighbours -> unpack, all enqueued on the
   handle's stream: no host synchronisation between the advance and the gather */
static int exchange_on(picles_t* h, int lo_rank, int hi_rank, cudaStream_t st) {
    if (h->A.hx == 0) return PICLES_OK;
    if ((lo_rank >= 0 || hi_rank >= 0) && !h->comm)
        return fail(h, PICLES_ERR_STATE, "picles_comm_init must be called before picles_halo_exchange");
    if (lo_rank >= h->comm_size || hi_rank >= h->comm_size || (lo_rank >= 0 && lo_rank == h->comm_rank) ||
        (hi_rank >= 0 && hi_rank == h->comm_rank)) {
        /* a periodic ring of one strip would be its own neighbour: not a strip decomposition */
        return fail(h, PICLES_ERR_ARG, "bad neighbour ranks lo=%d hi=%d (rank %d of %d)", lo_rank, hi_rank, h->comm_rank, h->comm_size);
    }
    launch_halo_pack(h->A, h->send_lo, h->send_hi, h->sms, st);
    CK(cudaGetLastError());
    if (lo_rank >= 0 || hi_rank >= 0) {
        size_t nb = (size_t)halo_msg_bytes(h);
        NCK(g_nccl.group_start());
        /* my first rows -> the lower neighbour's upper halo, my last rows -> the upper
           neighbour's lower halo.  Sends are issued lo,hi and receives hi,lo so that a
           periodic ring of two strips (lo_rank == hi_rank) pairs them up correctly:
           NCCL matches the operations between two ranks in issue order. */
        if (lo_rank >= 0) NCK(g_nccl.send(h->send_lo, nb, 0 /* ncclInt8 */, lo_rank, h->comm, st));
        if (hi_rank >= 0) NCK(g_nccl.send(h->send_hi, nb, 0, hi_rank, h->comm, st));
        if (hi_rank >= 0) NCK(g_nccl.recv(h->recv_hi, nb, 0, hi_rank, h->comm, st));
        if (lo_rank >= 0) NCK(g_nccl.recv(h->recv_lo, nb, 0, lo_rank, h->comm, st));
        NCK(g_nccl.group_end());
    }
    launch_halo_unpack(h->A, h->recv_lo, h->recv_hi, h->d_counters, h->sms, st);
    CK(cudaGetLastError());
    return PICLES_OK;
}

int picles_halo_exchange(picles_t* h, int lo_rank, int hi_rank) {
    int rc = need_ready(h, true);
    if (rc) return rc;
    REFUSE_MEMBERS(h, "picles_halo_exchange");
    return exchange_on(h, lo_rank, hi_rank, h->stream);
}

/* the reach that decides whether enough halo rows were exchanged, the same number on every strip: a 4-byte
   ncclAllReduce(max), every rank of the communicator taking part in every step.  Only particles within the supported
   reach (PH_REACH_MAX_ABI rows) of a strip edge can land on a neighbour, so picles_step_strip advances exactly those
   rows in its boundary launch and all-reduces THEIR reach (boundary_zones) while the interior still integrates: no
   strip waits for another strip's interior.  The serial path all-reduces the whole strip's reach behind its advance. */
static int reach_allreduce(picles_t* h, cudaStream_t st, bool boundary_zones) {
    if (!h->comm || h->comm_size < 2 || !h->reach_send) return PICLES_OK;
    /* 1 + reach: the gather reads 0 as "nobody all-reduced" */
    launch_reach_word(boundary_zones ? &h->d_counters->reach_bnd : &h->d_counters->reach, h->reach_send, st);
    CK(cudaGetLastError());
    NCK(g_nccl.all_reduce(h->reach_send, &h->d_counters->reach_all, 1, 2 /* ncclInt32 */, 2 /* ncclMax */, h->comm, st));
    return PICLES_OK;
}

/* one model step of a strip, exchange included; one host synchronisation at the end (the
   counters).  The first and last hx rows are advanced first; their deposit records travel
   to the neighbours on a second stream (pack, ncclSend/ncclRecv, unpack) while the interior
   rows integrate, so neither the exchange nor a slower neighbour shows up in the step time.
   The reference enforces no CFL limit (ParticleInCell.jl:58-71): when some particle of some strip
   reached further than the hx rows exchanged, the gather refuses (it changes nothing), every strip
   widens hx to the all-reduced reach and exchange + gather are repeated — the advance is not. */
int picles_step_strip(picles_t* h, double t, double dt_model, const double* u_t, const double* v_t, const double* u_t1,
                      const double* v_t1, int lo_rank, int hi_rank) {
    int rc = need_ready(h, true);
    if (rc) return rc;
    REFUSE_MEMBERS(h, "picles_step_strip");
    (void)t;
    const DeviceArrays& A = h->A;
    /* boundary zones: the hb rows next to each strip edge, hb = the widest exchange the strip supports.  A particle
       further inside cannot reach a neighbour (PICLES_ERR_HALO otherwise), so the zones' reach is all the neighbours
       need to know — and it is known early */
    const int hb = A.halo;
    const bool overlap = A.hx > 0 && (lo_rank >= 0 || hi_rank >= 0) && hb >= A.hx && A.ny > 2 * hb;
    if (!overlap) {
        rc = upload_and_advance(h, dt_model, u_t, v_t, u_t1, v_t1);
        if (rc) return rc;
        rc = exchange_on(h, lo_rank, hi_rank, h->stream);
        if (rc) return rc;
        rc = reach_allreduce(h, h->stream, false);
        if (rc) return rc;
    } else {
        rc = begin_advance(h, dt_model, u_t, v_t, u_t1, v_t1);
        if (rc) return rc;
        /* the two boundary zones: ONE launch on the communication stream, submitted first so that its few blocks
           are resident before the interior launch (whose blocks stay until the work queue is empty) fills the SMs.
           Behind each other on the compute stream the two small launches cost their full latency (~0.15 ms each,
           one chunk per warp) with the GPU idle: the fixed cost that capped strong scaling. */
        cudaEvent_t ready = h->pev[PIPE_CHUNKS + 2], exchanged = h->pev[PIPE_CHUNKS + 3];
        CK(cudaEventRecord(ready, h->stream));                     /* counters and per-row reach zeroed */
        CK(cudaStreamWaitEvent(h->comm_stream, ready, 0));
        rc = upload_rows(h, u_t, v_t, u_t1, v_t1, 0, hb, h->pev[PIPE_CHUNKS], h->comm_stream);
        if (rc) return rc;
        rc = upload_rows(h, u_t, v_t, u_t1, v_t1, A.ny - hb, A.ny, h->pev[PIPE_CHUNKS + 1], h->comm_stream);
        if (rc) return rc;
        launch_advance(A, h->P, dt_model, h->d_counters, h->sms, h->comm_stream, 0, (int64_t)hb * A.Nx,
                       (int64_t)(A.ny - hb) * A.Nx, (int64_t)A.ny * A.Nx, ADV_SLOT_BOUNDARY);
        CK(cudaGetLastError());
        if (u_t || u_t1) { /* whole-plane readers on the compute stream (the lag-level copy, the remesh) see the boundary rows too */
            CK(cudaStreamWaitEvent(h->stream, h->pev[PIPE_CHUNKS], 0));
            CK(cudaStreamWaitEvent(h->stream, h->pev[PIPE_CHUNKS + 1], 0));
        }
        /* the interior is enqueued before the exchange: the host side of the NCCL group (tens of microseconds) must not
           sit between the two advance launches */
        rc = advance_range(h, dt_model, u_t, v_t, u_t1, v_t1, hb, A.ny - hb);
        if (rc) return rc;
        rc = exchange_on(h, lo_rank, hi_rank, h->comm_stream);     /* boundary records written: pack, send/recv, unpack */
        if (rc) return rc;
        rc = reach_allreduce(h, h->comm_stream, true);             /* ... and the zones' reach: nothing here waits for an interior */
        if (rc) return rc;
        CK(cudaEventRecord(exchanged, h->comm_stream));            /* halo rows in place, reach of every strip's zones known */
        CK(cudaEventRecord(h->ev[1], h->stream));
        CK(cudaGetLastError());
        rc = keep_lag_level(h);
        if (rc) return rc;
        CK(cudaStreamWaitEvent(h->stream, exchanged, 0));
    }
    for (;;) {
        int need = 0;
        rc = project_remesh_once(h, dt_model, &need);
        if (rc || need == 0) return rc;
        /* every strip reads the same all-reduced reach, so every strip is here with the same `need` */
        if (!h->comm && (lo_rank >= 0 || hi_rank >= 0)) return fail(h, PICLES_ERR_STATE, "no communicator");
        rc = picles_halo_widen(h, need);
        if (rc) return rc;
        h->n_halo_widened++;
        rc = exchange_on(h, lo_rank, hi_rank, h->stream);
        if (rc) return rc;
    }
}

/* ---- wind ingestion: resident wind mesh ---------------------------------------------------- */
static int wm_alloc_copy(picles_t* h, double** dst, const double* src, int64_t count) {
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, (size_t)count * sizeof(double));
    if (e != cudaSuccess) return fail(h, PICLES_ERR_ALLOC, "cudaMalloc(%lld bytes): %s", (long long)(count * sizeof(double)), cudaGetErrorString(e));
    h->wm_allocs.push_back(q);
    e = cudaMemcpyAsync(q, src, (size_t)count * sizeof(double), cudaMemcpyHostToDevice, h->stream);
    if (e != cudaSuccess) return fail(h, PICLES_ERR_CUDA, "wind mesh upload: %s", cudaGetErrorString(e));
    *dst = (double*)q;
    return 0;
}
static bool strictly_increasing(const double* k, int n) {
    for (int i = 0; i < n; i++) {
        if (!(k[i] == k[i]) || (i > 0 && !(k[i] > k[i - 1]))) return false;
    }
    return true;
}
/* `E` meshes on shared knots (E = 1: the single mesh), member slowest in U and V; every check runs before the old
   mesh is freed */
static int set_wind_meshes(picles_t* h, const char* what, int E, int nxw, int nyw, int ntw, const double* xw, const double* yw,
                           const double* tw, const double* U, const double* V, const double* node_x, const double* node_y) {
    if (nxw < 2 || nyw < 2 || ntw < 2) return fail(h, PICLES_ERR_ARG, "wind mesh needs at least 2 knots per axis (%d, %d, %d)", nxw, nyw, ntw);
    if (!xw || !yw || !tw || !U || !V || !node_x || !node_y) return fail(h, PICLES_ERR_ARG, "%s: null array", what);
    if ((int64_t)nxw * nyw >= ((int64_t)1 << 31)) return fail(h, PICLES_ERR_ARG, "wind mesh slices are limited to 2^31 values");
    if (!strictly_increasing(xw, nxw) || !strictly_increasing(yw, nyw) || !strictly_increasing(tw, ntw))
        return fail(h, PICLES_ERR_ARG, "wind mesh knot vectors must be strictly increasing");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    for (void* p : h->wm_allocs) cudaFree(p);
    h->wm_allocs.clear();
    h->have_wind_mesh = h->wm_t1_valid = false;
    h->wm_members = 1;
    DeviceWindMesh& W = h->wm;
    W = DeviceWindMesh{};
    W.nx = nxw; W.ny = nyw; W.nt = ntw;
    const int64_t n = (int64_t)h->A.Nx * h->A.ny, st = (int64_t)nxw * nyw, nm = st * ntw * E;
    int rc;
    if ((rc = wm_alloc_copy(h, &W.xw, xw, nxw)) || (rc = wm_alloc_copy(h, &W.yw, yw, nyw)) ||
        (rc = wm_alloc_copy(h, &W.tw, tw, ntw)) || (rc = wm_alloc_copy(h, &W.U, U, nm)) ||
        (rc = wm_alloc_copy(h, &W.V, V, nm)) || (rc = wm_alloc_copy(h, &W.node_x, node_x, n)) ||
        (rc = wm_alloc_copy(h, &W.node_y, node_y, n)))
        return rc;
    {
        /* scratch of the two-pass sampler: one time-blended slice per component and member */
        void* q = nullptr;
        const size_t nb = (size_t)st * E * 16;
        if (cudaMalloc(&q, nb) != cudaSuccess) return fail(h, PICLES_ERR_ALLOC, "cannot allocate %lld bytes", (long long)nb);
        h->wm_allocs.push_back(q);
        W.Ub = (double*)q; W.Vb = W.Ub + st * E;
    }
    CK(cudaStreamSynchronize(h->stream));
    h->wm_members = E;
    h->have_wind_mesh = true;
    return PICLES_OK;
}
int picles_set_wind_mesh(picles_t* h, int nxw, int nyw, int ntw, const double* xw, const double* yw, const double* tw,
                         const double* U, const double* V, const double* node_x, const double* node_y) {
    if (!h || !h->have_grid) return fail(h, PICLES_ERR_STATE, "picles_set_grid must be called first");
    if (h->members > 1)
        return fail(h, PICLES_ERR_ARG, "picles_set_wind_mesh (one mesh) is not supported for an ensemble (%d members): "
                    "give every member its mesh with picles_set_member_wind_meshes", h->members);
    return set_wind_meshes(h, "picles_set_wind_mesh", 1, nxw, nyw, ntw, xw, yw, tw, U, V, node_x, node_y);
}
int picles_set_member_wind_meshes(picles_t* h, int nxw, int nyw, int ntw, const double* xw, const double* yw,
                                  const double* tw, const double* U, const double* V, const double* node_x,
                                  const double* node_y) {
    if (!h || !h->have_grid) return fail(h, PICLES_ERR_STATE, "picles_set_grid must be called first");
    return set_wind_meshes(h, "picles_set_member_wind_meshes", h->members, nxw, nyw, ntw, xw, yw, tw, U, V, node_x, node_y);
}

/* the wind of every member at time t at the nodes: one plane of Nx*ny values per member, member slowest */
static void wind_sample(picles_t* h, double t, double* u_out, double* v_out) {
    const int64_t n = (int64_t)h->A.Nx * h->A.ny;
    if (h->wm_members > 1) launch_wind_sample_members(h->wm, h->wm_members, n, t, u_out, v_out, h->sms, h->stream);
    else launch_wind_sample(h->wm, n, t, u_out, v_out, h->sms, h->stream);
}

int picles_sample_wind_mesh(picles_t* h, double t, double* u_out, double* v_out) {
    if (h) REFUSE_MEMBERS_WITHOUT_MESHES(h, "picles_sample_wind_mesh (a wind mesh)");
    if (!h || !h->have_wind_mesh) return fail(h, PICLES_ERR_STATE, "picles_set_wind_mesh must be called first");
    if (!u_out || !v_out) return fail(h, PICLES_ERR_ARG, "null output");
    CK(cudaSetDevice(h->device));
    const int64_t n = nodes(h);
    double* tmp = nullptr;
    if (cudaMalloc((void**)&tmp, (size_t)n * 16) != cudaSuccess) return fail(h, PICLES_ERR_ALLOC, "cannot allocate %lld bytes", (long long)n * 16);
    wind_sample(h, t, tmp, tmp + n);
    cudaError_t e = cudaMemcpyAsync(u_out, tmp, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(v_out, tmp + n, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e == cudaSuccess) e = cudaGetLastError();
    cudaFree(tmp);
    if (e != cudaSuccess) return fail(h, PICLES_ERR_CUDA, "k_wind_sample: %s", cudaGetErrorString(e));
    return PICLES_OK;
}

/* CUDA-event time of one wind level over this strip (both passes: k_wind_timeblend + k_wind_sample, or their member
   forms; mean of `reps` launches after one warm-up), written into scratch planes of its own: the roofline of the
   ingestion kernels */
int picles_measure_wind_sample(picles_t* h, double t, int reps, double* ms_per_launch) {
    if (h) REFUSE_MEMBERS_WITHOUT_MESHES(h, "picles_measure_wind_sample (a wind mesh)");
    if (!h || !h->have_wind_mesh) return fail(h, PICLES_ERR_STATE, "picles_set_wind_mesh must be called first");
    if (reps < 1 || !ms_per_launch) return fail(h, PICLES_ERR_ARG, "picles_measure_wind_sample: bad argument");
    CK(cudaSetDevice(h->device));
    const int64_t n = nodes(h);
    /* its own scratch planes: the wind levels staged for the next step are left alone */
    double* tmp = nullptr;
    if (cudaMalloc((void**)&tmp, (size_t)n * 16) != cudaSuccess) return fail(h, PICLES_ERR_ALLOC, "cannot allocate %lld bytes", (long long)n * 16);
    wind_sample(h, t, tmp, tmp + n);
    cudaError_t e = cudaEventRecord(h->tev[0], h->stream);
    for (int r = 0; r < reps; r++) wind_sample(h, t, tmp, tmp + n);
    if (e == cudaSuccess) e = cudaEventRecord(h->tev[1], h->stream);
    if (e == cudaSuccess) e = cudaEventSynchronize(h->tev[1]);
    if (e == cudaSuccess) e = cudaGetLastError();
    float ms = 0.f;
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, h->tev[0], h->tev[1]);
    cudaFree(tmp);
    if (e != cudaSuccess) return fail(h, PICLES_ERR_CUDA, "picles_measure_wind_sample: %s", cudaGetErrorString(e));
    *ms_per_launch = (double)ms / reps;
    return PICLES_OK;
}

int picles_seed_wind_mesh(picles_t* h, double t0) {
    int rc = need_ready(h, false);
    if (rc) return rc;
    REFUSE_MEMBERS_WITHOUT_MESHES(h, "picles_seed_wind_mesh (a wind mesh)");
    if (!h->have_wind_mesh) return fail(h, PICLES_ERR_STATE, "picles_set_wind_mesh must be called first");
    DeviceArrays& A = h->A;
    wind_sample(h, t0, A.u_t1, A.v_t1);
    h->wm_t1_valid = true;
    h->wm_t1_time = t0;
    return seed_from_t1(h);
}

/* every wind level of the step [t, t+dt_model] sampled from the mesh into the device planes: what
   picles_upload_winds + picles_set_wind_midlevels do from host arrays */
int picles_stage_wind_mesh(picles_t* h, double t, double dt_model, int n_mid) {
    int rc = need_ready(h, true);
    if (rc) return rc;
    REFUSE_MEMBERS_WITHOUT_MESHES(h, "picles_stage_wind_mesh (a wind mesh)");
    if (!h->have_wind_mesh) return fail(h, PICLES_ERR_STATE, "picles_set_wind_mesh must be called first");
    if (!(dt_model > 0)) return fail(h, PICLES_ERR_ARG, "dt_model must be positive");
    if (n_mid < 0 || n_mid > PICLES_WIND_MID_MAX) return fail(h, PICLES_ERR_ARG, "n_mid = %d outside 0..%d", n_mid, PICLES_WIND_MID_MAX);
    DeviceArrays& A = h->A;
    rc = ensure_mid_planes(h, n_mid);
    if (rc) return rc;
    /* false: the previous step's t+dt level is this step's t level */
    const bool new_t = !(h->wm_t1_valid && h->wm_t1_time == t);
    next_wind_levels(h, new_t, true);
    if (new_t) wind_sample(h, t, A.u_t, A.v_t);
    const double t1 = t + dt_model;
    wind_sample(h, t1, A.u_t1, A.v_t1);
    for (int k = 1; k <= n_mid; k++)
        wind_sample(h, t + dt_model * (double)k / (double)(n_mid + 1), A.u_mid[k - 1], A.v_mid[k - 1]);
    CK(cudaGetLastError());
    A.n_mid = n_mid;
    h->wm_t1_valid = true;
    h->wm_t1_time = t1;
    return PICLES_OK;
}

int picles_step_wind_mesh(picles_t* h, double t, double dt_model, int n_mid, int lo_rank, int hi_rank) {
    REFUSE_MEMBERS_WITHOUT_MESHES(h, "picles_step_wind_mesh (a wind mesh)");
    int rc = picles_stage_wind_mesh(h, t, dt_model, n_mid);
    if (rc) return rc;
    const DeviceArrays& A = h->A;
    if (A.ny == A.Ny && lo_rank < 0 && hi_rank < 0) return picles_step(h, t, dt_model, nullptr, nullptr, nullptr, nullptr);
    return picles_step_strip(h, t, dt_model, nullptr, nullptr, nullptr, nullptr, lo_rank, hi_rank);
}

} /* extern "C" */
