/*
 * picles_kernels.cu — sm_100a kernels of the PiCLES particle-in-cell step.
 *
 *   k_seed      SeedParticle for every node                      (run.jl:199-247, core_2D.jl:434-488)
 *   k_advance   advance! : adaptive RK over DT + deposit record  (mapping_2D.jl:118-243)  FP64-bound
 *   k_project_remesh  ParticleToNode! as a deterministic gather   (mapping_2D.jl:59-73,
 *                     over TMA-staged record tiles, fused with     ParticleInCell.jl:341-538)
 *                     remesh!/NodeToParticle!                     (mapping_2D.jl:250-356)  HBM-bound
 *   k_energy_members  sum of State[:,:,1], per member            (run.jl:23-25)
 *
 * Layout in HBM (one y-strip per GPU): every per-node quantity is its own plane of
 * ny*Nx doubles with i (x) fastest — the memory order of the reference's column-major
 * (Nx,Ny[,3]) arrays — so a warp touches 32 consecutive doubles (256 B) per plane.
 * Deposit records carry `halo` extra rows on both sides for the neighbour strips and a
 * row pitch rounded up to 4 elements (16-byte rows for the TMA tensor maps).
 *
 * Compiled with --fmad=false: physics.h spells out every fused multiply-add so the
 * results are bit-identical to the CPU oracle.
 */
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>
#include <stdlib.h>

#include <atomic>

#include "stiff.h"
#include "picles_device.h"
#include "pmath_trig.h"
#include "wind_mesh.h"

namespace picles {

static_assert(PH_REACH_MAX == PH_REACH_MAX_ABI, "reach limits out of sync");

/* every kernel this library launches is counted where it is launched (bench.py reports the count of its timed region) */
static std::atomic<long long> g_launches{0};
long long launch_count() { return g_launches.load(); }
#define COUNT_LAUNCH(n) g_launches.fetch_add(n)

/* ---- block-level tally reduction: one atomic set per block ------------------- */
__device__ __forceinline__ int32_t warp_sum(int32_t v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int32_t warp_max(int32_t v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_down_sync(0xffffffffu, v, o));
    return v;
}

#define TALLY_NSUM 14
__device__ __forceinline__ void tally_merge(Tally& a, const Tally& b) {
    a.integrated += b.integrated; a.substeps += b.substeps; a.rejects += b.rejects; a.rhs += b.rhs;
    a.reseed += b.reseed; a.fixups += b.fixups; a.failed += b.failed; a.deposited += b.deposited;
    a.A += b.A; a.B += b.B; a.C += b.C; a.D += b.D;
    a.reach = max(a.reach, b.reach); a.max_attempts = max(a.max_attempts, b.max_attempts);
    a.stiff_switches += b.stiff_switches; a.stiff_attempts += b.stiff_attempts;
}
__device__ void tally_flush(const Tally& c, DeviceCounters* dc, bool boundary_zone = false) {
    __shared__ int32_t s_sum[TALLY_NSUM];
    __shared__ int32_t s_max[2];
    if (threadIdx.x < TALLY_NSUM) s_sum[threadIdx.x] = 0;
    if (threadIdx.x < 2) s_max[threadIdx.x] = 0;
    __syncthreads();
    int32_t v[TALLY_NSUM] = {c.integrated, c.substeps, c.rejects, c.rhs, c.reseed, c.fixups,
                             c.failed, c.deposited, c.A, c.B, c.C, c.D, c.stiff_switches, c.stiff_attempts};
    int lane = threadIdx.x & 31;
#pragma unroll
    for (int k = 0; k < TALLY_NSUM; k++) {
        int32_t s = warp_sum(v[k]);
        if (lane == 0 && s) atomicAdd(&s_sum[k], s);
    }
    int32_t r = warp_max(c.reach), a = warp_max(c.max_attempts);
    if (lane == 0) {
        atomicMax(&s_max[0], r);
        atomicMax(&s_max[1], a);
    }
    __syncthreads();
    if (threadIdx.x < TALLY_NSUM && s_sum[threadIdx.x])
        atomicAdd(&dc->sums[threadIdx.x], (unsigned long long)s_sum[threadIdx.x]);
    if (threadIdx.x == 0) {
        if (s_max[0]) atomicMax(&dc->reach, s_max[0]);
        if (s_max[0] && boundary_zone) atomicMax(&dc->reach_bnd, s_max[0]);
        if (s_max[1]) atomicMax(&dc->max_attempts, s_max[1]);
    }
}

__device__ __forceinline__ void load_particle(const DeviceArrays& A, int64_t l, Particle& p) {
    p.u0 = A.z[0][l]; p.u1 = A.z[1][l]; p.u2 = A.z[2][l]; p.u3 = A.z[3][l]; p.u4 = A.z[4][l];
    p.t = A.t[l]; p.dt = A.dt[l]; p.qold = A.qold[l];
    p.iter = A.iter[l];
    p.flags = A.flags[l];
    p.status = A.status[l];
    p.as = 0; /* the AutoSwitch plane is touched only under PICLES_SOLVER_AUTOTSIT5 (load_as / store_as) */
}
__device__ __forceinline__ void load_as(const DeviceArrays& A, const picles_params_t& P, int64_t l, Particle& p) {
    if (P.solver == PICLES_SOLVER_AUTOTSIT5) p.as = A.as[l];
}
__device__ __forceinline__ void store_as(const DeviceArrays& A, const picles_params_t& P, int64_t l, const Particle& p) {
    if (P.solver == PICLES_SOLVER_AUTOTSIT5) A.as[l] = p.as;
}
__device__ __forceinline__ void store_particle(const DeviceArrays& A, int64_t l, const Particle& p) {
    A.z[0][l] = p.u0; A.z[1][l] = p.u1; A.z[2][l] = p.u2; A.z[3][l] = p.u3; A.z[4][l] = p.u4;
    A.t[l] = p.t; A.dt[l] = p.dt; A.qold[l] = p.qold;
    A.iter[l] = p.iter;
    A.flags[l] = p.flags;
    A.status[l] = p.status;
}
__device__ __forceinline__ void store_record(const DeviceArrays& A, int64_t le, const Record& r) {
    A.rec[0][le] = r.e; A.rec[1][le] = r.mx; A.rec[2][le] = r.my; A.rec[3][le] = r.wxc; A.rec[4][le] = r.wyc;
    A.cell[le] = r.cell;
}

/* index of node l (= jr*Nx + i) in the record planes */
__device__ __forceinline__ int64_t rec_index(const DeviceArrays& A, int64_t l) {
    if (A.rp == A.Nx) return l + (int64_t)A.halo * A.Nx;
    int64_t jr = l / A.Nx;
    return (jr + A.halo) * A.rp + (l - jr * A.Nx);
}

/* node of the shared grid planes (mask, M, pc) that particle l lives on: l within its member under ENS, l itself for
   a single model (strips included).  The record index and the record row stay linear in l (rec_index): members are
   whole blocks of rows, and an ensemble has no halo rows */
template <bool ENS>
__device__ __forceinline__ int64_t grid_node(const DeviceArrays& A, int64_t l) {
    return ENS ? l % ((int64_t)A.Nx * A.ny) : l;
}

/* ---- seed ------------------------------------------------------------------ */
__global__ void __launch_bounds__(256) k_seed(DeviceArrays A, picles_params_t P, const double* __restrict__ u0,
                                              const double* __restrict__ v0, DeviceCounters* dc) {
    int64_t n = (int64_t)A.Nx * A.ny * A.members;
    int32_t n_off = 0; /* iterated particles seeded off */
    for (int64_t l = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; l < n; l += (int64_t)gridDim.x * blockDim.x) {
        Particle p;
        double e, mx, my;
        seed_particle(P, A.mask[grid_node<true>(A, l)], u0[l], v0[l], p, e, mx, my);
        if ((p.flags & PICLES_PF_ACTIVE) && !(p.flags & PICLES_PF_ON)) n_off++;
        store_particle(A, l, p);
        A.as[l] = 0;
        A.S[0][l] = e; A.S[1][l] = mx; A.S[2][l] = my;
        Record r;
        r.e = r.mx = r.my = r.wxc = r.wyc = 0.0;
        r.cell = PH_CELL_INVALID;
        store_record(A, rec_index(A, l), r);
    }
    n_off = warp_sum(n_off);
    if ((threadIdx.x & 31) == 0 && n_off) atomicAdd(&dc->n_seed_off, n_off);
}

/* ---- advance ---------------------------------------------------------------- */
/*
 * One thread per particle.  Work is handed out warp by warp: a warp takes the next chunk of 32
 * consecutive particles of the launch's range from a counter in global memory (one atomic per
 * chunk, i.e. per ~10^6 instructions), integrates it and comes back for more, until the range is
 * exhausted.  Within a chunk the adaptive loop runs in SIMT lock-step (lanes whose particle reached
 * t+DT wait at the loop exit for the slowest lane: neighbouring nodes carry near-identical states,
 * measured 29.0-32.0 active lanes per instruction over the configurations, profiles/README.md);
 * across chunks nobody waits: a warp that drew slow particles (40 attempts against a mean of 6.6 at
 * the calm foot of a wind ramp) simply takes fewer chunks.  The static grid-stride assignment this
 * replaces visited only Nx/32 / gcd(Nx/32, warps in flight) distinct x-positions per warp, so on a
 * field that varies along x whole warps drew nothing but slow chunks and the launch ended on them
 * (growing-wind configuration: 7.3 ms against 4.5 ms for a step with 4 % more instructions).
 */
#ifdef ADV_MAXNREG /* register cap given directly; ADV_MIN_BLOCKS then only sizes the grid */
#define ADV_BOUNDS __maxnreg__(ADV_MAXNREG)
#else
#define ADV_BOUNDS __launch_bounds__(ADV_THREADS, ADV_MIN_BLOCKS)
#endif
template <bool PER_NODE_M, bool AUTOSW, int TSIT5 = 0, bool ENS = false>
__global__ void ADV_BOUNDS
k_advance(DeviceArrays A, picles_params_t P, double DT, DeviceCounters* dc, int64_t l_begin, int64_t l_end, int64_t l2_begin,
          int64_t l2_end, int slot) {
    /* stage derivatives k_j[0:3], j = 1..7: 21 doubles per thread, one column per thread
       (consecutive threads -> consecutive 8-byte words: conflict-free) */
    __shared__ double s_k[KS_SLOTS * ADV_THREADS];
    __shared__ int32_t s_hist[ADV_HIST_BINS];
    KStrided K;
    K.base = &s_k[threadIdx.x];
    K.stride = ADV_THREADS;
    Tally c;
    tally_zero(c);
    if (threadIdx.x < ADV_HIST_BINS) s_hist[threadIdx.x] = 0;
    pm_exptab_shared_init(); /* the exp table of the fast right-hand side (pmath.h) */
    __syncthreads();
    const int lane = threadIdx.x & 31;
    unsigned long long* const queue = &dc->next_chunk[slot];
    /* the launch covers [l_begin, l_end) and then [l2_begin, l2_end) (a strip's two boundary row blocks in one
       launch; empty for everything else) */
    const int64_t n1 = (l_end - l_begin + 31) >> 5;
    for (;;) {
        unsigned long long chunk = 0;
        if (lane == 0) chunk = atomicAdd(queue, 1ull);
        chunk = __shfl_sync(0xffffffffu, chunk, 0);
        const bool second = (int64_t)chunk >= n1;
        const int64_t l0 = second ? l2_begin + ((int64_t)chunk - n1) * 32 : l_begin + (int64_t)chunk * 32;
        const int64_t lim = second ? l2_end : l_end;
        if (l0 >= lim) break; /* uniform over the warp */
        const int64_t l = l0 + lane;
        const uint8_t flags = (l < lim) ? A.flags[l] : (uint8_t)0;
        if (flags & PICLES_PF_ACTIVE) { /* else: the record stays invalid (set at seed) */
            int64_t le = rec_index(A, l);
            const int64_t g = grid_node<ENS>(A, l);
            Particle p;
            load_particle(A, l, p);
            if (AUTOSW) load_as(A, P, l, p);
            double M[4];
            if (PER_NODE_M) { M[0] = A.M[0][g]; M[1] = A.M[1][g]; M[2] = A.M[2][g]; M[3] = A.M[3][g]; }
            else { M[0] = A.Mc[0]; M[1] = A.Mc[1]; M[2] = A.Mc[2]; M[3] = A.Mc[3]; }
            double pc = A.pc ? A.pc[g] : 0.0;
            Record r;
            double um[PH_WIND_SEG_MAX], vm[PH_WIND_SEG_MAX];
#pragma unroll
            for (int k = 0; k < PICLES_WIND_MID_MAX; k++) {
                if (k < A.n_mid) { um[k] = A.u_mid[k][l]; vm[k] = A.v_mid[k][l]; }
                else { um[k] = 0.0; vm[k] = 0.0; }
            }
            um[PH_WIND_SEG_MAX - 1] = 0.0; vm[PH_WIND_SEG_MAX - 1] = 0.0;
            const double t_start = p.t;
            int attempts = -1;
            /* winds(x, y, t_end) with t_end = integ.t + DT (mapping_2D.jl:172-176): a particle that was seeded off under
               B-1 as run never advances its own clock, so its t_end stays at 0 + DT — the level kept from the first step */
            double wu1 = A.u_t1[l], wv1 = A.v_t1[l];
            if (A.u_lag && !(flags & PICLES_PF_ON)) { wu1 = A.u_lag[l]; wv1 = A.v_lag[l]; }
            const bool pending = advance_particle<AUTOSW, TSIT5>(P, p, A.mask[g], DT, A.u_t[l], A.v_t[l], wu1, wv1, A.n_mid, um,
                                                          vm, M, pc, r, c, K, attempts);
            if (AUTOSW && pending) {
                /* AutoSwitch handed the particle to Rosenbrock23: park the state reached so far; the
                   resume kernel that follows finishes the step (the record slot carries what it needs) */
                r.cell = PH_CELL_PENDING;
                r.e = t_start; r.mx = (double)attempts;
                r.my = r.wxc = r.wyc = 0.0;
                A.pending[atomicAdd(&dc->n_pending, 1)] = (int32_t)l;
            } else if (attempts >= 0) {
                atomicAdd(&s_hist[attempts < ADV_HIST_BINS ? attempts : ADV_HIST_BINS - 1], 1);
            }
            store_particle(A, l, p);
            if (AUTOSW) store_as(A, P, l, p);
            store_record(A, le, r);
            if (r.cell != PH_CELL_INVALID && !(AUTOSW && r.cell == PH_CELL_PENDING)) {
                /* per-row reach (lets the gather size its window tile by tile) and class presence */
                const int rr = cell_reach(r.cell);
                int32_t* rslot = &A.rowreach[le / A.rp];
                if (rr > __ldcg(rslot)) atomicMax(rslot, rr);
                if (((uint32_t)r.cell >> 28) & 1u) dc->class1 = 1;
            }
        }
    }
    tally_flush(c, dc, slot == ADV_SLOT_BOUNDARY);
    if (threadIdx.x < ADV_HIST_BINS && s_hist[threadIdx.x])
        atomicAdd(&dc->attempt_hist[threadIdx.x], (unsigned long long)s_hist[threadIdx.x]);
}

/*
 * AutoTsit5 only: the particles k_advance parked (cell == PH_CELL_PENDING) finish their step here —
 * Rosenbrock23 attempts, possibly back to Tsit5 and forth — with the cold code of stiff.h.  A
 * handful of particles per step at most (none on most configurations): k_advance appends their
 * indices to a list, so this kernel costs one launch when the list is empty.  One block per SM,
 * all registers: nothing here is tuned.
 */
template <bool PER_NODE_M, bool ENS = false>
__global__ void __launch_bounds__(ADV_THREADS, 1)
k_advance_resume(DeviceArrays A, picles_params_t P, double DT, DeviceCounters* dc, int64_t l_begin, int64_t l_end) {
    __shared__ double s_k[KS_SLOTS * ADV_THREADS];
    KStrided K;
    K.base = &s_k[threadIdx.x];
    K.stride = ADV_THREADS;
    Tally c;
    tally_zero(c);
    (void)l_begin; (void)l_end;
    pm_exptab_shared_init();
    __syncthreads();
    const int n_pending = dc->n_pending; /* entries parked earlier in the step are skipped by their cell marker */
    for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < n_pending; q += gridDim.x * blockDim.x) {
        const int64_t l = A.pending[q];
        const int64_t le = rec_index(A, l);
        if (A.cell[le] != PH_CELL_PENDING) continue;
        const int64_t g = grid_node<ENS>(A, l);
        Particle p;
        load_particle(A, l, p);
        load_as(A, P, l, p);
        ResumeArgs R;
        R.mask = A.mask[g]; R.nmid = A.n_mid; R.attempts = (int)A.rec[1][le];
        R.DT = DT; R.t_start = A.rec[0][le];
        R.wu0 = A.u_t[l]; R.wv0 = A.v_t[l]; R.wu1 = A.u_t1[l]; R.wv1 = A.v_t1[l];
        for (int k = 0; k < PH_WIND_SEG_MAX; k++) {
            const bool have = k < A.n_mid && k < PICLES_WIND_MID_MAX;
            R.um[k] = have ? A.u_mid[k][l] : 0.0;
            R.vm[k] = have ? A.v_mid[k][l] : 0.0;
        }
        if (PER_NODE_M) { R.M[0] = A.M[0][g]; R.M[1] = A.M[1][g]; R.M[2] = A.M[2][g]; R.M[3] = A.M[3][g]; }
        else { R.M[0] = A.Mc[0]; R.M[1] = A.Mc[1]; R.M[2] = A.Mc[2]; R.M[3] = A.Mc[3]; }
        R.pc = A.pc ? A.pc[g] : 0.0;
        Record r;
        const int32_t max_before = c.max_attempts;
        c.max_attempts = 0;
        advance_resume(&P, &R, &p, &r, &c, K);
        { /* c.max_attempts now holds this particle's attempts */
            const int a = c.max_attempts;
            atomicAdd(&dc->attempt_hist[a < ADV_HIST_BINS ? a : ADV_HIST_BINS - 1], 1ull);
            c.max_attempts = max(max_before, a);
        }
        store_particle(A, l, p);
        store_as(A, P, l, p);
        store_record(A, le, r);
        if (r.cell != PH_CELL_INVALID) {
            const int rr = cell_reach(r.cell);
            int32_t* slot = &A.rowreach[le / A.rp];
            if (rr > __ldcg(slot)) atomicMax(slot, rr);
            if (((uint32_t)r.cell >> 28) & 1u) dc->class1 = 1;
        }
    }
    /* a parked particle may lie in a boundary zone: counted there too (an over-estimate can only widen an exchange) */
    tally_flush(c, dc, true);
}

/* ---- projection gather + remesh ---------------------------------------------------- */
/*
 * One block per tile of PR_TX x TY target nodes (TY = PR_BH - 2*HY).  One thread arms an mbarrier and issues
 * six TMA tile loads (cp.async.bulk.tensor.3d): the five record planes and the cell plane of its member
 * over the targets plus a halo of PR_HX x HY cells.  Boxes that stick out of the planes are
 * zero-filled by the TMA unit; a zero cell decodes to an offset that never matches, i.e.
 * "no deposit", which is exactly what lies beyond a non-periodic edge.  While the tiles are in
 * flight every thread loads the remesh inputs of its 3-4 nodes (flags, wind at
 * t), so the node loop below touches HBM only to store.
 *
 * Per node: sum the window from shared memory (gather_window, compile-time offsets) in the
 * reference's order, store State, and — the node value still being in registers — run
 * NodeToParticle! for the node's particle.  Nodes whose window crosses a periodic seam or the
 * tripolar fold, and tiles whose reach exceeds HY, take gather_node() on the planes in HBM.
 */
/* GetVariablesAtVertex with results in registers (hot: remesh branch A) */
struct Vtx3 { double u0, u1, u2; };
__device__ __noinline__ Vtx3 vertex_values_cold(double e, double mx, double my) {
    Particle p;
    vertex_t<OpsSafe>(e, mx, my, p, (unsigned*)0);
    Vtx3 r = {p.u0, p.u1, p.u2};
    return r;
}
__device__ __forceinline__ void vertex_values(double e, double mx, double my, double& u0, double& u1, double& u2) {
#if defined(__CUDA_ARCH__)
    unsigned bad = 0;
    double m_amp = OpsFast::sqrtz(mx * mx + my * my, &bad);
    double den = 2.0 * (m_amp * m_amp);
    u0 = OpsFast::log_(e, &bad);
    u1 = OpsFast::divz(mx * e, den, &bad);
    u2 = OpsFast::divz(my * e, den, &bad);
    if (bad) {
        Vtx3 r = vertex_values_cold(e, mx, my);
        u0 = r.u0; u1 = r.u1; u2 = r.u2;
    }
#endif
}

struct PRTile {
    double rec[5][PR_BH * PR_BW];
    int32_t cell[PR_BH * PR_BW];
    unsigned long long mbar;
};
static_assert((PR_BH * PR_BW * 8) % 128 == 0 && (PR_BW * 4) % 16 == 0 && PR_HX % 4 == 0 && PR_TX % 4 == 0 &&
              PR_HX >= PR_HY_WIDE && (PR_BH - 2 * PR_HY_WIDE) % (PR_THREADS / PR_TX) == 0 &&
              (PR_BH - 2 * PR_HY_NARROW) % (PR_THREADS / PR_TX) == 0 && (PR_BH - 2 * PR_HY_NARROW) / (PR_THREADS / PR_TX) <= 4,
              "TMA tile alignment / nodes per thread (their flags are packed in 32 bits)");
#define PR_TILE_BYTES (5 * PR_BH * PR_BW * 8 + PR_BH * PR_BW * 4)

/* window of run-time reach R from a staged tile (reach 3-4 of the wide tile geometry) */
template <int NCLS>
__device__ __forceinline__ void gather_window_rt(const PRTile& T, int base, int R, double& s0, double& s1, double& s2) {
    for (int cls = 0; cls < NCLS; cls++)
        for (int dj = -R; dj <= R; dj++)
            for (int di = -R; di <= R; di++) {
                const int le = base + dj * PR_BW + di;
                const uint32_t cell = (uint32_t)T.cell[le];
                const unsigned dx = (unsigned)(PH_CELL_BIAS - di) - (cell & 0x3fffu);
                const unsigned dy = (unsigned)(PH_CELL_BIAS - dj) - ((cell >> 14) & 0x3fffu);
                if (dx > 1u || dy > 1u) continue;
                if (NCLS > 1 && (int)((cell >> 28) & 1u) != cls) continue;
                const double wxc = T.rec[3][le], wyc = T.rec[4][le];
                const double wx = dx ? wxc : 1.0 - wxc;
                const double wy = dy ? wyc : 1.0 - wyc;
                const double w = wx * wy;
                s0 += w * T.rec[0][le];
                s1 += w * T.rec[1][le];
                s2 += w * T.rec[2][le];
            }
}

/*
 * Everything of the node loop that is not "reach-1 window from the tile, then remesh branch A"
 * is deferred to this out-of-line pass, so the hot loop contains no call and keeps its state
 * in registers.  `mask` bit k: node k still needs its gather (window crossing a periodic seam
 * or the tripolar fold, reach > 1, two deposit classes, untiled step); bit 4+k: node k was
 * gathered but its remesh is not branch A (wind-sea reseed or switch-off).  Returns the remesh
 * branch counts (A, B, C, D) of the nodes handled here.
 */
template <int HY>
__device__ __noinline__ int4 cold_nodes(const DeviceArrays* Ap, const picles_params_t* Pp, const PRTile* Tp, uint32_t mask,
                                        uint32_t fl_all, int i, int jr0, int tx, int ty, int R, int Rt, int n_classes,
                                        int accumulate, bool tiled, double DT) {
    const DeviceArrays& A = *Ap;
    const picles_params_t& P = *Pp;
    const PRTile& T = *Tp;
    Tally c;
    tally_zero(c);
    for (int k = 0; k < (PR_BH - 2 * HY) / (PR_THREADS / PR_TX); k++) {
        if (!(mask & (0x11u << k))) continue;
        const int jl = ty + k * (PR_THREADS / PR_TX);
        const int jr = jr0 + jl;
        const int I = i + 1, J = jr + 1 + A.j0;
        const int64_t l = (int64_t)jr * A.Nx + i;
        const uint8_t flags = (uint8_t)(fl_all >> (8 * k));
        double s0, s1, s2;
        if (mask & (1u << k)) {
            s0 = s1 = s2 = 0.0;
            if (accumulate) { s0 = A.S[0][l]; s1 = A.S[1][l]; s2 = A.S[2][l]; }
            const bool fast_x = (A.bx == PICLES_BND_NONPERIODIC) || (I > R && I <= A.Nx - R);
            const bool fast_y = (A.by == PICLES_BND_NONPERIODIC) || (A.by == PICLES_BND_PERIODIC && J > R && J <= A.Ny - R) ||
                                (A.by == PICLES_BND_TRIPOLAR_NORTH && J <= A.Ny - R);
            if (tiled && fast_x && fast_y) {
                const int base = (jl + HY) * PR_BW + (tx + PR_HX);
                if (n_classes == 1) gather_window_rt<1>(T, base, Rt, s0, s1, s2);
                else gather_window_rt<2>(T, base, Rt, s0, s1, s2);
            } else {
                RecView V;
                V.Nx = A.Nx; V.Ny = A.Ny; V.bx = A.bx; V.by = A.by; V.j0 = A.j0; V.ny = A.ny; V.halo = A.halo; V.hx = A.hx; V.pitch = A.rp;
                V.e = A.rec[0]; V.mx = A.rec[1]; V.my = A.rec[2]; V.wx = A.rec[3]; V.wy = A.rec[4];
                V.cell = A.cell;
                gather_node(V, I, J, R, n_classes, s0, s1, s2);
            }
            A.S[0][l] = s0; A.S[1][l] = s1; A.S[2][l] = s2;
        } else {
            s0 = A.S[0][l]; s1 = A.S[1][l]; s2 = A.S[2][l];
        }
        if (!(flags & PICLES_PF_ACTIVE)) continue;
        const double wu = A.u_t[l], wv = A.v_t[l];
        Particle p;
        load_particle(A, l, p);
        load_as(A, P, l, p);
        remesh_particle(P, p, s0, s1, s2, wu, wv, DT, c);
        store_particle(A, l, p);
        store_as(A, P, l, p);
    }
    return make_int4(c.A, c.B, c.C, c.D);
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

/* the planes of ensemble member m, as a single-member DeviceArrays (an ensemble has no halo rows: every member owns
   whole rows; member 0 is the handle's own planes, a strip's halo rows included) */
__device__ __forceinline__ void member_planes(const DeviceArrays& A, int m, DeviceArrays& B) {
    B = A;
    const int64_t o = (int64_t)m * A.Nx * A.ny, orec = (int64_t)m * A.ny * A.rp;
    for (int k = 0; k < 5; k++) { B.z[k] += o; B.rec[k] += orec; }
    B.t += o; B.dt += o; B.qold += o; B.iter += o; B.flags += o; B.status += o; B.as += o;
    B.u_t += o; B.v_t += o; B.u_t1 += o; B.v_t1 += o;
    for (int k = 0; k < PICLES_WIND_MID_MAX; k++)
        if (B.u_mid[k]) { B.u_mid[k] += o; B.v_mid[k] += o; }
    if (B.u_lag) { B.u_lag += o; B.v_lag += o; }
    for (int k = 0; k < 3; k++) B.S[k] += o;
    B.cell += orec;
    B.rowreach += (int64_t)m * A.ny;
    B.members = 1;
}
/* the planes the gather of this block reads and writes: those of its member (blockIdx.z) in an ensemble, placed in
   shared memory once per block.  A single model reads its own from the kernel parameter: the copy in shared memory
   costs it 8-10 % of the gather (measured at 4096^2) */
template <bool ENS>
__device__ __forceinline__ const DeviceArrays& block_planes(const DeviceArrays& A) {
    if constexpr (ENS) {
        __shared__ DeviceArrays s_member;
        if (threadIdx.x == 0) member_planes(A, blockIdx.z, s_member);
        __syncthreads();
        return s_member;
    } else {
        return A;
    }
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, int c0, int c1, int c2, unsigned long long* mbar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 :
                 : "r"(smem_u32(dst)), "l"((unsigned long long)map), "r"(smem_u32(mbar)), "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}

/* blockIdx.z is the ensemble member (0 for a single model).  Its tiles come from 3-D tensor maps (x, row, member), so
   a box that sticks out of the member's rows is zero-filled as it is beyond a single model's edge, and no member reads
   another's records.  ENS: more than one member (block_planes) */
template <int HY, bool ENS = false>
__global__ void __launch_bounds__(PR_THREADS, PR_MIN_BLOCKS)
k_project_remesh(const __grid_constant__ ProjectMaps maps, const __grid_constant__ DeviceArrays A_all,
                 const __grid_constant__ picles_params_t P, double DT, int n_classes,
                 int accumulate, DeviceCounters* dc) {
    const DeviceArrays& A = block_planes<ENS>(A_all);
    extern __shared__ __align__(128) unsigned char pr_smem[];
    /* TMA destinations must be 128-byte aligned whatever static shared memory precedes them */
    PRTile& T = *reinterpret_cast<PRTile*>(pr_smem + ((128u - (smem_u32(pr_smem) & 127u)) & 127u));
    constexpr int TY = PR_BH - 2 * HY;                 /* target rows of a tile */
    constexpr int NPT = TY / (PR_THREADS / PR_TX);     /* nodes per thread */
    const int i0 = blockIdx.x * PR_TX, jr0 = blockIdx.y * TY;
    /* deposits landing on this strip come from its own particles (reach) and from the
       neighbours' rows received into the halo (reach_halo) */
    int R = min(max(dc->reach, dc->reach_halo), PH_REACH_MAX);
    if (A.ny != A.Ny) {
        /* strips: a deposit of a neighbour's particle can land here from as far as the largest reach of the particles
           near a strip edge.  If that is more than the hx rows exchanged, records are missing: touch nothing, say so,
           and let the host repeat exchange and gather with wider rows (picles_step_strip does; the advance is not repeated) */
        /* reach_all - 1: the all-reduced reach, the same number on every strip (so every strip takes this branch together,
           which the repeated exchange relies on); 0: nobody all-reduced, judge by what this strip knows */
        const int ra = dc->reach_all;
        const int need = ra > 0 ? ra - 1 : max(dc->reach, dc->reach_halo);
        if (need > A.hx) {
            if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) dc->halo_short = need;
            return;
        }
    }
    /* two passes over the window are only needed when deposits of both classes exist */
    if (!dc->class1) n_classes = 1;
    /* reach of the records that can land on this tile: rows within R of its targets.  A few
       fast rows (the shrinking cells near a pole) then do not widen every tile's window. */
    __shared__ int s_rt;
    if (R <= 1) { /* nothing to narrow */
        if (threadIdx.x == 0) s_rt = R;
    } else if (threadIdx.x < 32) {
        const int first = jr0 + A.halo - R, count = TY + 2 * R, rows = A.ny + 2 * A.halo;
        int rt = 0;
        for (int q = threadIdx.x; q < count; q += 32) {
            const int row = first + q;
            if (row >= 0 && row < rows) rt = max(rt, A.rowreach[row]);
        }
        rt = warp_max(rt);
        if (threadIdx.x == 0) s_rt = rt;
    }
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&T.mbar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int Rt = min(s_rt, R);       /* window of this tile's fast-zone nodes */
    const bool tiled = (Rt <= HY);
    if (tiled && threadIdx.x == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&T.mbar)), "r"(PR_TILE_BYTES)
                     : "memory");
        const int c0 = i0 - PR_HX, c1 = jr0 + A.halo - HY;
#pragma unroll
        for (int k = 0; k < 5; k++) tma_load_3d(T.rec[k], &maps.rec[k], c0, c1, blockIdx.z, &T.mbar);
        tma_load_3d(T.cell, &maps.cell, c0, c1, blockIdx.z, &T.mbar);
    }
    /* the flags of my nodes, issued while the tiles are in flight (branch A of the remesh
       needs nothing else; the wind is only read on the rare reseed / switch-off branches) */
    const int tx = threadIdx.x & (PR_TX - 1), ty = threadIdx.x / PR_TX;
    const int i = i0 + tx;
    uint32_t fl_all = 0;
#pragma unroll
    for (int k = 0; k < NPT; k++) {
        const int jr = jr0 + ty + k * (PR_THREADS / PR_TX);
        if (i < A.Nx && jr < A.ny) fl_all |= (uint32_t)A.flags[(int64_t)jr * A.Nx + i] << (8 * k);
    }
    if (tiled) {
        uint32_t done = 0;
        while (!done) {
            asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                         : "=r"(done)
                         : "r"(smem_u32(&T.mbar))
                         : "memory");
        }
    }
    int nA = 0; /* remesh branch-A count of this thread */
    uint32_t cold = 0; /* nodes deferred to cold_nodes() */
    const bool hot_window = tiled && (n_classes == 1);
#pragma unroll 1
    for (int k = 0; k < NPT; k++) {
        const int jl = ty + k * (PR_THREADS / PR_TX); /* row inside the tile */
        const int jr = jr0 + jl;
        if (i >= A.Nx || jr >= A.ny) continue;
        const int I = i + 1, J = jr + 1 + A.j0; /* global 1-based node */
        const bool fast_x = (A.bx == PICLES_BND_NONPERIODIC) || (I > R && I <= A.Nx - R);
        const bool fast_y = (A.by == PICLES_BND_NONPERIODIC) || (A.by == PICLES_BND_PERIODIC && J > R && J <= A.Ny - R) ||
                            (A.by == PICLES_BND_TRIPOLAR_NORTH && J <= A.Ny - R);
        if (!(hot_window && fast_x && fast_y)) { cold |= 1u << k; continue; }
        const int64_t l = (int64_t)jr * A.Nx + i;
        double s0 = 0.0, s1 = 0.0, s2 = 0.0;
        if (accumulate) { s0 = A.S[0][l]; s1 = A.S[1][l]; s2 = A.S[2][l]; }
        const int64_t base = (int64_t)(jl + HY) * PR_BW + (tx + PR_HX);
        if (Rt <= 1) gather_window<1, PR_BW, 1>(T.rec[0], T.rec[1], T.rec[2], T.rec[3], T.rec[4], T.cell, PR_BW, base, s0, s1, s2);
        else if (Rt == 2) gather_window<2, PR_BW, 1>(T.rec[0], T.rec[1], T.rec[2], T.rec[3], T.rec[4], T.cell, PR_BW, base, s0, s1, s2);
        else gather_window_rt<1>(T, (int)base, Rt, s0, s1, s2);
        A.S[0][l] = s0;
        A.S[1][l] = s1;
        A.S[2][l] = s2;
        /* ---- remesh! for the particle whose home is this node ---- */
        const uint32_t flags = (fl_all >> (8 * k)) & 0xffu;
        if (!(flags & PICLES_PF_ACTIVE)) continue;
        const bool enough = (s0 >= P.minimal_state[0]) && (s1 * s1 + s2 * s2 >= P.minimal_state[1]);
        if ((flags & PICLES_PF_BOUNDARY) || !enough) { cold |= 16u << k; continue; }
        /* branch A: GetVariablesAtVertex; touches only u and flags */
        double u0, u1, u2;
        vertex_values(s0, s1, s2, u0, u1, u2);
        uint32_t nf = flags | PICLES_PF_DT_RESET;
        if (P.on_persist) nf |= PICLES_PF_ON;
        nA++;
        A.z[0][l] = u0; A.z[1][l] = u1; A.z[2][l] = u2; A.z[3][l] = 0.0; A.z[4][l] = 0.0;
        if (nf != flags) A.flags[l] = (uint8_t)nf;
    }
    int nB = 0, nC = 0, nD = 0;
    if (cold) {
        int4 cc = cold_nodes<HY>(&A, &P, &T, cold, fl_all, i, jr0, tx, ty, R, Rt, n_classes, accumulate, tiled, DT);
        nA += cc.x; nB = cc.y; nC = cc.z; nD = cc.w;
    }
    /* branch counts: one warp reduction each, one global atomic per warp and non-zero count */
    nA = warp_sum(nA); nB = warp_sum(nB); nC = warp_sum(nC); nD = warp_sum(nD);
    if ((threadIdx.x & 31) == 0) {
        if (nA) atomicAdd(&dc->sums[8], (unsigned long long)nA);
        if (nB) atomicAdd(&dc->sums[9], (unsigned long long)nB);
        if (nC) atomicAdd(&dc->sums[10], (unsigned long long)nC);
        if (nD) atomicAdd(&dc->sums[11], (unsigned long long)nD);
    }
}

/* ---- energy sum (deterministic two-stage) ---------------------------------------- */
__device__ __forceinline__ void energy_partial(const double* __restrict__ e, int64_t n, double* __restrict__ partial) {
    __shared__ double sh[256];
    double s = 0.0;
    for (int64_t l = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; l < n; l += (int64_t)gridDim.x * blockDim.x) s += e[l];
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[blockIdx.x] = sh[0];
}
/* blockIdx.y is the member, whose plane of n values is reduced by the same blocks in the same order whatever gridDim.y is */
__global__ void __launch_bounds__(256) k_energy_members(const double* __restrict__ e, int64_t n, double* __restrict__ partial) {
    energy_partial(e + blockIdx.y * n, n, partial + (int64_t)blockIdx.y * gridDim.x);
}

/* ---- halo pack / unpack: H rows of the 5 record planes + cell plane -------------- */
__global__ void k_halo_pack(DeviceArrays A, char* __restrict__ send_lo, char* __restrict__ send_hi) {
    int64_t m = (int64_t)A.hx * A.rp;
    for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < m; q += (int64_t)gridDim.x * blockDim.x) {
        int64_t lo = (int64_t)A.halo * A.rp + q;                 /* first hx owned rows */
        int64_t hi = (int64_t)(A.halo + A.ny - A.hx) * A.rp + q; /* last hx owned rows */
#pragma unroll
        for (int k = 0; k < 5; k++) {
            ((double*)send_lo)[k * m + q] = A.rec[k][lo];
            ((double*)send_hi)[k * m + q] = A.rec[k][hi];
        }
        ((int32_t*)(send_lo + 5 * m * 8))[q] = A.cell[lo];
        ((int32_t*)(send_hi + 5 * m * 8))[q] = A.cell[hi];
    }
}
__global__ void k_halo_unpack(DeviceArrays A, const char* __restrict__ recv_lo, const char* __restrict__ recv_hi,
                              DeviceCounters* dc) {
    int64_t m = (int64_t)A.hx * A.rp;
    int32_t reach = 0;
    for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < m; q += (int64_t)gridDim.x * blockDim.x) {
        int64_t lo = (int64_t)(A.halo - A.hx) * A.rp + q;         /* the hx halo rows next to the first owned row */
        int64_t hi = (int64_t)(A.ny + A.halo) * A.rp + q;         /* the hx halo rows behind the last owned row */
#pragma unroll
        for (int k = 0; k < 5; k++) {
            A.rec[k][lo] = ((const double*)recv_lo)[k * m + q];
            A.rec[k][hi] = ((const double*)recv_hi)[k * m + q];
        }
        int32_t clo = ((const int32_t*)(recv_lo + 5 * m * 8))[q], chi = ((const int32_t*)(recv_hi + 5 * m * 8))[q];
        A.cell[lo] = clo;
        A.cell[hi] = chi;
        const int rlo = cell_reach(clo), rhi = cell_reach(chi);
        const int row = A.halo - A.hx + (int)(q / A.rp);
        if (rlo > 0 && rlo > __ldcg(&A.rowreach[row])) atomicMax(&A.rowreach[row], rlo);
        const int row_hi = A.ny + A.halo + (int)(q / A.rp);
        if (rhi > 0 && rhi > __ldcg(&A.rowreach[row_hi])) atomicMax(&A.rowreach[row_hi], rhi);
        if ((clo != PH_CELL_INVALID && (((uint32_t)clo >> 28) & 1u)) || (chi != PH_CELL_INVALID && (((uint32_t)chi >> 28) & 1u)))
            dc->class1 = 1;
        reach = max(reach, max(rlo, rhi));
    }
    reach = warp_max(reach);
    if ((threadIdx.x & 31) == 0 && reach) atomicMax(&dc->reach_halo, reach);
}
__global__ void k_fill_i32(int32_t* p, int64_t n, int32_t v) {
    for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < n; q += (int64_t)gridDim.x * blockDim.x) p[q] = v;
}

/* ---- grid lookups -------------------------------------------------------------------- */
/* per-node projection kernel M = [cosα/dx sinα/dy; −sinα/dx cosα/dy] and great-circle
   coefficient from the raw metric planes (TripolarGridMOM6.jl:448-459,
   spherical_grid_corrections.jl:13); coalesced plane reads and writes, 72 B/node */
__global__ void __launch_bounds__(256) k_grid_metric(int64_t n, const double* __restrict__ dx, const double* __restrict__ dy,
                                                     const double* __restrict__ angle_dx, const double* __restrict__ lat,
                                                     double R_earth, double* __restrict__ M11, double* __restrict__ M12,
                                                     double* __restrict__ M21, double* __restrict__ M22, double* __restrict__ pc) {
    for (int64_t l = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; l < n; l += (int64_t)gridDim.x * blockDim.x) {
        double a, b, c, d, p;
        pm_grid_metric_node(dx[l], dy[l], angle_dx[l], lat[l], R_earth, &a, &b, &c, &d, &p);
        M11[l] = a; M12[l] = b; M21[l] = c; M22[l] = d; pc[l] = p;
    }
}
/* make_boundaries (mask_utils.jl:14-22,38-55): land nodes with an ocean 4-neighbour (circular
   shifts, as circshift) become 2, edges of non-periodic axes 3.  The +-1 row/column reads
   of neighbouring threads overlap and are served by L1. */
__global__ void __launch_bounds__(256) k_make_boundaries(const uint8_t* __restrict__ ocean, uint8_t* __restrict__ total,
                                                         int Nx, int Ny, int bx, int by) {
    for (int j = blockIdx.y; j < Ny; j += gridDim.y) {
        const int jm = (j == 0) ? Ny - 1 : j - 1, jp = (j == Ny - 1) ? 0 : j + 1;
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < Nx; i += gridDim.x * blockDim.x) {
            const int im = (i == 0) ? Nx - 1 : i - 1, ip = (i == Nx - 1) ? 0 : i + 1;
            const int64_t row = (int64_t)j * Nx;
            int self = ocean[row + i] != 0;
            int b = 0;
            if (!self)
                b = (ocean[row + im] != 0) | (ocean[row + ip] != 0) | (ocean[(int64_t)jm * Nx + i] != 0) |
                    (ocean[(int64_t)jp * Nx + i] != 0);
            int v = self + 2 * b;
            if (bx == PICLES_BND_NONPERIODIC && (i == 0 || i == Nx - 1)) v = 3;
            if (by == PICLES_BND_NONPERIODIC && (j == 0 || j == Ny - 1)) v = 3;
            total[row + i] = (uint8_t)v;
        }
    }
}

/* ---- derived output fields ------------------------------------------------------------ */
/* Hs = 4*sqrt(e) (visualization/movie_2D.jl:50) and the mean group velocity
   c = m*e/(2|m|^2) of GetGroupVelocity (core_2D.jl:138-147); nullptr outputs are skipped.
   IEEE sqrt and division: identical to the host arithmetic. */
__global__ void __launch_bounds__(256) k_fields(int64_t n, const double* __restrict__ e, const double* __restrict__ mx,
                                                const double* __restrict__ my, double* __restrict__ Hs,
                                                double* __restrict__ cx, double* __restrict__ cy) {
    for (int64_t l = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; l < n; l += (int64_t)gridDim.x * blockDim.x) {
        const double ev = e[l];
        if (Hs) Hs[l] = 4.0 * sqrt(ev);
        if (cx || cy) {
            const double a = mx[l], b = my[l];
            const double m_amp = sqrt(a * a + b * b);
            const double den = 2.0 * (m_amp * m_amp);
            if (cx) cx[l] = a * ev / den;
            if (cy) cy[l] = b * ev / den;
        }
    }
}

/* ---- roofline denominators measured in place ------------------------------------ */
/* 8 independent DFMA chains per thread: the FP64 pipe's issue-rate ceiling */
__global__ void __launch_bounds__(256) k_fp64_peak(double* out, int iters) {
    double a0 = threadIdx.x * 1e-3, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m = 0.999999, c = 1e-7;
    for (int k = 0; k < iters; k++) {
#pragma unroll
        for (int r = 0; r < 8; r++) {
            a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
            a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
        }
    }
    double s = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
    if (s == 123.456) out[0] = s; /* keep the chains alive */
}
__global__ void __launch_bounds__(256) k_copy_f64(double2* __restrict__ dst, const double2* __restrict__ src, int64_t n2) {
    for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < n2; q += (int64_t)gridDim.x * blockDim.x) dst[q] = src[q];
}

/* ---- self-test of the fast-path arithmetic (pmath.h) against the IEEE operators ---- */
__device__ __forceinline__ uint64_t st_next(uint64_t& s) {
    s ^= s << 13; s ^= s >> 7; s ^= s << 17;
    return s;
}
/* operand classes: 0 raw bit patterns (every exponent, NaN/Inf/denormals included),
   1 moderate magnitudes 2^[-40,40] (the physics range), 2 one operand from a table of
   special values */
__device__ double st_operand(uint64_t& s, int cls) {
    uint64_t r = st_next(s);
    if (cls == 0) return __longlong_as_double((long long)r);
    if (cls == 1) {
        uint64_t mant = r & 0x000fffffffffffffull;
        uint64_t e = 1023 - 40 + ((r >> 52) % 81);
        uint64_t sign = (r >> 63) << 63;
        return __longlong_as_double((long long)(sign | (e << 52) | mant));
    }
    const double tab[12] = {0.0, -0.0, 1.0, -1.0, 4.9406564584124654e-324, 2.2250738585072014e-308,
                            1.7976931348623157e308, __longlong_as_double(0x7ff0000000000000ll),
                            __longlong_as_double(0x7ff8000000000000ll), 1.9999999999999998, 0.85, 1e-300};
    return tab[(r >> 32) % 12];
}
__global__ void k_selftest_math(uint64_t seed, int iters, unsigned long long* out /* [6] */) {
    uint64_t s = seed ^ (0x9E3779B97F4A7C15ull * (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x + 1));
    unsigned long long n_div = 0, bad_div = 0, mis_div = 0, n_sqrt = 0, bad_sqrt = 0, mis_sqrt = 0;
    for (int it = 0; it < iters; it++) {
        int cls = it % 3;
        double a = st_operand(s, cls == 2 ? (it & 1 ? 2 : 1) : cls);
        double b = st_operand(s, cls == 2 ? (it & 1 ? 1 : 2) : cls);
        unsigned bad = 0;
        double q = (it & 4) ? pm_divz_fast(a, b, &bad) : pm_div_fast(a, b, &bad);
        double qi = a / b;
        n_div++;
        if (bad) bad_div++;
        else if (__double_as_longlong(q) != __double_as_longlong(qi) && !(q != q && qi != qi)) mis_div++;
        double x = fabs(a);
        if (cls == 2 && (it & 2)) x = a;
        bad = 0;
        double r = (it & 4) ? pm_sqrtz_fast(x, &bad) : pm_sqrt_fast(x, &bad);
        double ri = sqrt(x);
        n_sqrt++;
        if (bad) bad_sqrt++;
        else if (__double_as_longlong(r) != __double_as_longlong(ri) && !(r != r && ri != ri)) mis_sqrt++;
    }
    atomicAdd(&out[0], n_div); atomicAdd(&out[1], bad_div); atomicAdd(&out[2], mis_div);
    atomicAdd(&out[3], n_sqrt); atomicAdd(&out[4], bad_sqrt); atomicAdd(&out[5], mis_sqrt);
}

/* ---- wind ingestion: sample the resident wind mesh at the nodes ---------------------------
 * Two passes per level (wind_mesh.h).  The time interval and weight are the same for every node,
 * so the blend in time is done once per mesh point (k_wind_timeblend, mesh-sized); k_wind_sample
 * then runs one thread per node — 16 B of coordinates in, 16 B of wind out (HBM-bound) — on that
 * slice: knots and 2 x 2 corner values per component, served by L1/L2. */
/* pass 1: the mesh slice at time t (nx*ny points, a few microseconds) */
__global__ void __launch_bounds__(256) k_wind_timeblend(DeviceWindMesh D, double t) {
    WindMesh W;
    W.nx = D.nx; W.ny = D.ny; W.nt = D.nt; W.xw = D.xw; W.yw = D.yw; W.tw = D.tw; W.U = D.U; W.V = D.V;
    const WindMeshTime T = wm_time(W, t);
    const int64_t st = (int64_t)D.nx * D.ny;
    for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < st; p += (int64_t)gridDim.x * blockDim.x) {
        D.Ub[p] = wm_timeblend(D.U, st, T.it, T.dt, p);
        D.Vb[p] = wm_timeblend(D.V, st, T.it, T.dt, p);
    }
}
/* pass 2: every node */
__global__ void __launch_bounds__(256) k_wind_sample(DeviceWindMesh D, int64_t n, double* __restrict__ u_out,
                                                     double* __restrict__ v_out) {
    WindMesh W;
    W.nx = D.nx; W.ny = D.ny; W.nt = D.nt; W.xw = D.xw; W.yw = D.yw; W.tw = D.tw; W.U = D.U; W.V = D.V;
    WindMeshTime T;
    T.it = 0; T.dt = 0.0;
    T.x0 = W.xw[0]; T.x1 = W.xw[W.nx - 1]; T.y0 = W.yw[0]; T.y1 = W.yw[W.ny - 1];
    T.inv_hx = wm_inv_h(W.xw, W.nx); T.inv_hy = wm_inv_h(W.yw, W.ny);
    const double* __restrict__ Ub = D.Ub;
    const double* __restrict__ Vb = D.Vb;
    const double* __restrict__ nx = D.node_x;
    const double* __restrict__ ny = D.node_y;
    /* software pipeline: the coordinates of the next node are in flight (HBM latency) while this
       one is located and blended (L1/L2 latency) */
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int64_t l = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    double xn = 0.0, yn = 0.0;
    if (l < n) { xn = __ldcs(nx + l); yn = __ldcs(ny + l); }
    for (; l < n; l += stride) {
        const double x = xn, y = yn;
        const int64_t l2 = l + stride;
        if (l2 < n) { xn = __ldcs(nx + l2); yn = __ldcs(ny + l2); }
        double u, v;
        wm_sample2d(W, T, Ub, Vb, x, y, u, v);
        __stcs(u_out + l, u);
        __stcs(v_out + l, v);
    }
}

/* one thread per four consecutive nodes (wm_sample2d_x4: the y lookup shared along a row), 16-byte loads and
   stores: 0.200 -> 0.163 ms at 4096^2.  The launcher falls back to k_wind_sample when a plane is not 16-byte
   aligned, and a scalar tail takes the last n % 4 nodes */
__global__ void __launch_bounds__(256) k_wind_sample_x4(DeviceWindMesh D, int64_t n, double* __restrict__ u_out,
                                                        double* __restrict__ v_out) {
    WindMesh W;
    W.nx = D.nx; W.ny = D.ny; W.nt = D.nt; W.xw = D.xw; W.yw = D.yw; W.tw = D.tw; W.U = D.U; W.V = D.V;
    WindMeshTime T;
    T.it = 0; T.dt = 0.0;
    T.x0 = W.xw[0]; T.x1 = W.xw[W.nx - 1]; T.y0 = W.yw[0]; T.y1 = W.yw[W.ny - 1];
    T.inv_hx = wm_inv_h(W.xw, W.nx); T.inv_hy = wm_inv_h(W.yw, W.ny);
    const double* __restrict__ Ub = D.Ub;
    const double* __restrict__ Vb = D.Vb;
    const double2* __restrict__ nx2 = (const double2*)D.node_x;
    const double2* __restrict__ ny2 = (const double2*)D.node_y;
    const int64_t n4 = n >> 2;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    double2 xa = {0, 0}, xb = {0, 0}, ya = {0, 0}, yb = {0, 0};
    if (g < n4) { xa = __ldcs(nx2 + 2 * g); xb = __ldcs(nx2 + 2 * g + 1); ya = __ldcs(ny2 + 2 * g); yb = __ldcs(ny2 + 2 * g + 1); }
    for (; g < n4; g += stride) {
        const double x[4] = {xa.x, xa.y, xb.x, xb.y}, y[4] = {ya.x, ya.y, yb.x, yb.y};
        const int64_t g2 = g + stride;
        if (g2 < n4) { xa = __ldcs(nx2 + 2 * g2); xb = __ldcs(nx2 + 2 * g2 + 1); ya = __ldcs(ny2 + 2 * g2); yb = __ldcs(ny2 + 2 * g2 + 1); }
        double u[4], v[4];
        wm_sample2d_x4(W, T, Ub, Vb, x, y, u, v);
        __stcs((double2*)u_out + 2 * g, make_double2(u[0], u[1])); __stcs((double2*)u_out + 2 * g + 1, make_double2(u[2], u[3]));
        __stcs((double2*)v_out + 2 * g, make_double2(v[0], v[1])); __stcs((double2*)v_out + 2 * g + 1, make_double2(v[2], v[3]));
    }
    /* tail */
    const int64_t l = 4 * n4 + blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (l < n) {
        double u, v;
        wm_sample2d(W, T, Ub, Vb, D.node_x[l], D.node_y[l], u, v);
        u_out[l] = u; v_out[l] = v;
    }
}

/* ---- an ensemble's member meshes on shared knots (picles_set_member_wind_meshes) -------------
 * D.U, D.V hold `members` meshes back to back and D.Ub, D.Vb `members` blended slices.  The same two passes as above,
 * each still one launch whatever the number of members. */
/* pass 1: every member's slice at time t, blockIdx.y = member (48 B per member mesh point) */
__global__ void __launch_bounds__(256) k_wind_timeblend_members(DeviceWindMesh D, int members, double t) {
    WindMesh W;
    W.nx = D.nx; W.ny = D.ny; W.nt = D.nt; W.xw = D.xw; W.yw = D.yw; W.tw = D.tw; W.U = D.U; W.V = D.V;
    const WindMeshTime T = wm_time(W, t);
    const int64_t st = (int64_t)D.nx * D.ny;
    for (int m = blockIdx.y; m < members; m += gridDim.y) {
        double* __restrict__ ub = D.Ub + st * m;
        double* __restrict__ vb = D.Vb + st * m;
        for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < st; p += (int64_t)gridDim.x * blockDim.x) {
            ub[p] = wm_timeblend_member(D.U, st, D.nt, T.it, T.dt, m, p);
            vb[p] = wm_timeblend_member(D.V, st, D.nt, T.it, T.dt, m, p);
        }
    }
}
/* pass 2: one thread per node and chunk of WM_MEMBER_CHUNK members (blockIdx.y): the node is located once and blended
   for each member of the chunk, its stores coalesced along the nodes of every member plane.  The member dimension fills
   the SMs when a member has few nodes (2601 at 51 x 51). */
#define WM_MEMBER_CHUNK 8
__global__ void __launch_bounds__(256) k_wind_sample_members(DeviceWindMesh D, int members, int64_t n,
                                                             double* __restrict__ u_out, double* __restrict__ v_out) {
    WindMesh W;
    W.nx = D.nx; W.ny = D.ny; W.nt = D.nt; W.xw = D.xw; W.yw = D.yw; W.tw = D.tw; W.U = D.U; W.V = D.V;
    WindMeshTime T;
    T.it = 0; T.dt = 0.0;
    T.x0 = W.xw[0]; T.x1 = W.xw[W.nx - 1]; T.y0 = W.yw[0]; T.y1 = W.yw[W.ny - 1];
    T.inv_hx = wm_inv_h(W.xw, W.nx); T.inv_hy = wm_inv_h(W.yw, W.ny);
    const int m0 = blockIdx.y * WM_MEMBER_CHUNK;
    const int m1 = (m0 + WM_MEMBER_CHUNK < members) ? m0 + WM_MEMBER_CHUNK : members;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t l = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; l < n; l += stride) {
        const WindMeshNode q = wm_node(W, T, __ldg(D.node_x + l), __ldg(D.node_y + l));
        wm_sample2d_members(W, q, D.Ub, D.Vb, m0, m1, n, l, u_out, v_out);
    }
}

/* ---- launchers ------------------------------------------------------------------ */
static int grid_for(int64_t n, int threads, int sms, int blocks_per_sm) {
    int64_t need = (n + threads - 1) / threads;
    int64_t cap = (int64_t)sms * blocks_per_sm;
    if (need < 1) need = 1;
    return (int)(need < cap ? need : cap);
}

void launch_seed(const DeviceArrays& A, const picles_params_t& P, const double* u0, const double* v0, DeviceCounters* dc,
                 int sms, cudaStream_t st) {
    int64_t n = (int64_t)A.Nx * A.ny * A.members;
    k_seed<<<grid_for(n, 256, sms, 8), 256, 0, st>>>(A, P, u0, v0, dc);
    COUNT_LAUNCH(1);
}

/* launch_advance2 for an ensemble: the same choice of instantiation, each in its ensemble form */
static void launch_advance_members(const DeviceArrays& A, const picles_params_t& P, double DT, DeviceCounters* dc, int sms,
                                   cudaStream_t st, int64_t l_begin, int64_t l_end, int64_t l2_begin, int64_t l2_end,
                                   int slot, int g, bool pn) {
    const int64_t count = (l_end - l_begin) + (l2_end - l2_begin);
    const bool spec = !P.nan_eest_rejects;
#define ADV_ARGS A, P, DT, dc, l_begin, l_end, l2_begin, l2_end, slot
    if (P.solver == PICLES_SOLVER_AUTOTSIT5) {
        const int gr = grid_for(count, ADV_THREADS, sms, 1);
        if (pn) {
            if (P.propagation && spec) k_advance<true, true, 3, true><<<g, ADV_THREADS, 0, st>>>(ADV_ARGS);
            else k_advance<true, true, 0, true><<<g, ADV_THREADS, 0, st>>>(ADV_ARGS);
            k_advance_resume<true, true><<<gr, ADV_THREADS, 0, st>>>(A, P, DT, dc, l_begin, l_end);
        } else {
            if (P.propagation && spec) k_advance<false, true, 3, true><<<g, ADV_THREADS, 0, st>>>(ADV_ARGS);
            else k_advance<false, true, 0, true><<<g, ADV_THREADS, 0, st>>>(ADV_ARGS);
            k_advance_resume<false, true><<<gr, ADV_THREADS, 0, st>>>(A, P, DT, dc, l_begin, l_end);
        }
        COUNT_LAUNCH(2);
    } else {
        const bool ts5 = (P.solver == PICLES_SOLVER_TSIT5) && P.propagation && spec;
        if (pn && ts5) k_advance<true, false, 1, true><<<g, ADV_THREADS, 0, st>>>(ADV_ARGS);
        else if (pn) k_advance<true, false, 0, true><<<g, ADV_THREADS, 0, st>>>(ADV_ARGS);
        else if (ts5) k_advance<false, false, 1, true><<<g, ADV_THREADS, 0, st>>>(ADV_ARGS);
        else if (P.solver == PICLES_SOLVER_DP5 && P.propagation && spec) k_advance<false, false, 2, true><<<g, ADV_THREADS, 0, st>>>(ADV_ARGS);
        else k_advance<false, false, 0, true><<<g, ADV_THREADS, 0, st>>>(ADV_ARGS);
        COUNT_LAUNCH(1);
    }
#undef ADV_ARGS
}

/* particles [l_begin, l_end) and then [l2_begin, l2_end) of the strip (the whole strip: 0, Nx*ny and an empty
   second range); slot: the work queue of this launch (DeviceCounters::next_chunk, zeroed with the counters at the
   start of the step) */
void launch_advance2(const DeviceArrays& A, const picles_params_t& P, double DT, DeviceCounters* dc, int sms,
                     cudaStream_t st, int64_t l_begin, int64_t l_end, int64_t l2_begin, int64_t l2_end, int slot) {
    if (l2_end < l2_begin) l2_end = l2_begin;
    if (l_end < l_begin) l_end = l_begin;
    const int64_t count = (l_end - l_begin) + (l2_end - l2_begin);
    if (count <= 0) return;
    int g = grid_for(count, ADV_THREADS, sms, ADV_MIN_BLOCKS);
    bool pn = (A.M[0] != nullptr);
    if (A.members > 1) {
        launch_advance_members(A, P, DT, dc, sms, st, l_begin, l_end, l2_begin, l2_end, slot, g, pn);
        return;
    }
    /* picles_params_t::nan_eest_rejects (a NaN error estimate rejected by 1/qmin instead of ending the integrator) lives
       in the generic instantiations only: the specialised ones keep the code they were measured with */
    const bool spec = !P.nan_eest_rejects;
#define ADV_ARGS A, P, DT, dc, l_begin, l_end, l2_begin, l2_end, slot
    /* AutoTsit5 runs the instantiation that carries the stiffness monitor and the Rosenbrock23 branch */
    if (P.solver == PICLES_SOLVER_AUTOTSIT5) {
        const int gr = grid_for(count, ADV_THREADS, sms, 1);
        /* (third template argument 3: propagation on, known at compile time, as in the Tsit5 / DP5 instantiations) */
        if (pn) {
            if (P.propagation && spec) k_advance<true, true, 3><<<g, ADV_THREADS, 0, st>>>(ADV_ARGS);
            else k_advance<true, true><<<g, ADV_THREADS, 0, st>>>(ADV_ARGS);
            k_advance_resume<true><<<gr, ADV_THREADS, 0, st>>>(A, P, DT, dc, l_begin, l_end);
        } else {
            if (P.propagation && spec) k_advance<false, true, 3><<<g, ADV_THREADS, 0, st>>>(ADV_ARGS);
            else k_advance<false, true><<<g, ADV_THREADS, 0, st>>>(ADV_ARGS);
            k_advance_resume<false><<<gr, ADV_THREADS, 0, st>>>(A, P, DT, dc, l_begin, l_end);
        }
        COUNT_LAUNCH(2);
    } else {
        /* Tsit5 has its own instantiation (compile-time tableau without zero coefficients) */
        /* (the specialised instantiations take propagation as given: a run without it — the reference's
           propagation = false switch — is served by the generic one) */
        const bool ts5 = (P.solver == PICLES_SOLVER_TSIT5) && P.propagation && spec;
        if (pn && ts5) k_advance<true, false, true><<<g, ADV_THREADS, 0, st>>>(ADV_ARGS);
        else if (pn) k_advance<true, false><<<g, ADV_THREADS, 0, st>>>(ADV_ARGS);
        else if (ts5) k_advance<false, false, true><<<g, ADV_THREADS, 0, st>>>(ADV_ARGS);
        /* ... and so has DP5 on a uniform kernel (the bench06 settings): -1.5 % */
        else if (P.solver == PICLES_SOLVER_DP5 && P.propagation && spec) k_advance<false, false, 2><<<g, ADV_THREADS, 0, st>>>(ADV_ARGS);
        else k_advance<false, false><<<g, ADV_THREADS, 0, st>>>(ADV_ARGS);
        COUNT_LAUNCH(1);
    }
#undef ADV_ARGS
}
void launch_advance(const DeviceArrays& A, const picles_params_t& P, double DT, DeviceCounters* dc, int sms,
                    cudaStream_t st, int64_t l_begin, int64_t l_end, int slot) {
    launch_advance2(A, P, DT, dc, sms, st, l_begin, l_end, l_end, l_end, slot);
}

int project_remesh_smem_bytes() { return (int)sizeof(PRTile) + 128; }
cudaError_t project_remesh_configure() {
    const int b = project_remesh_smem_bytes();
    cudaError_t e = cudaFuncSetAttribute(k_project_remesh<PR_HY_NARROW>, cudaFuncAttributeMaxDynamicSharedMemorySize, b);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_project_remesh<PR_HY_WIDE>, cudaFuncAttributeMaxDynamicSharedMemorySize, b);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_project_remesh<PR_HY_NARROW, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, b);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_project_remesh<PR_HY_WIDE, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, b);
    return e;
}
/* wide: cut the 72 x 20 box as 12 target rows + 4 halo rows (previous step's reach was 3-4)
   instead of 16 + 2; a wrong guess only sends tiles through the generic gather */
void launch_project_remesh(const ProjectMaps& maps, const DeviceArrays& A, const picles_params_t& P, double DT,
                           int n_classes, int accumulate, int wide, DeviceCounters* dc, cudaStream_t st) {
    const int TY = PR_BH - 2 * (wide ? PR_HY_WIDE : PR_HY_NARROW);
    dim3 grid((A.Nx + PR_TX - 1) / PR_TX, (A.ny + TY - 1) / TY, A.members);
    if (A.members > 1) {
        if (wide) k_project_remesh<PR_HY_WIDE, true><<<grid, PR_THREADS, project_remesh_smem_bytes(), st>>>(maps, A, P, DT, n_classes, accumulate, dc);
        else k_project_remesh<PR_HY_NARROW, true><<<grid, PR_THREADS, project_remesh_smem_bytes(), st>>>(maps, A, P, DT, n_classes, accumulate, dc);
    } else if (wide) k_project_remesh<PR_HY_WIDE><<<grid, PR_THREADS, project_remesh_smem_bytes(), st>>>(maps, A, P, DT, n_classes, accumulate, dc);
    else k_project_remesh<PR_HY_NARROW><<<grid, PR_THREADS, project_remesh_smem_bytes(), st>>>(maps, A, P, DT, n_classes, accumulate, dc);
    COUNT_LAUNCH(1);
}

void launch_wind_sample(const DeviceWindMesh& W, int64_t n, double t, double* u_out, double* v_out, int sms, cudaStream_t st) {
    if (n <= 0) return;
    COUNT_LAUNCH(2);
    k_wind_timeblend<<<grid_for((int64_t)W.nx * W.ny, 256, sms, 8), 256, 0, st>>>(W, t);
    if (n >= 4 && (((uintptr_t)W.node_x | (uintptr_t)W.node_y | (uintptr_t)u_out | (uintptr_t)v_out) & 15) == 0) {
        k_wind_sample_x4<<<grid_for(n >> 2, 256, sms, 8), 256, 0, st>>>(W, n, u_out, v_out);
        return;
    }
    k_wind_sample<<<grid_for(n, 256, sms, 8), 256, 0, st>>>(W, n, u_out, v_out);
}
void launch_wind_sample_members(const DeviceWindMesh& W, int members, int64_t n, double t, double* u_out, double* v_out,
                                int sms, cudaStream_t st) {
    if (n <= 0) return;
    COUNT_LAUNCH(2);
    /* about 8 blocks per SM over both grid dimensions, at least one block per member (chunk) */
    const int64_t cap = (int64_t)sms * 8;
    const int64_t st_pts = (int64_t)W.nx * W.ny;
    const int my = members < 65535 ? members : 65535;
    int64_t bx = (cap + my - 1) / my, need = (st_pts + 255) / 256;
    if (bx > need) bx = need;
    k_wind_timeblend_members<<<dim3((unsigned)bx, (unsigned)my), 256, 0, st>>>(W, members, t);
    const int chunks = (members + WM_MEMBER_CHUNK - 1) / WM_MEMBER_CHUNK;
    bx = (cap + chunks - 1) / chunks;
    need = (n + 255) / 256;
    if (bx > need) bx = need;
    k_wind_sample_members<<<dim3((unsigned)bx, (unsigned)chunks), 256, 0, st>>>(W, members, n, u_out, v_out);
}
void launch_energy(const double* e, int64_t n, int members, double* partial, int nblocks, cudaStream_t st) {
    k_energy_members<<<dim3(nblocks, members), 256, 0, st>>>(e, n, partial);
    COUNT_LAUNCH(1);
}

__global__ void k_reach_word(const int32_t* src, int32_t* dst) { *dst = *src + 1; }
void launch_reach_word(const int32_t* src, int32_t* dst, cudaStream_t st) {
    k_reach_word<<<1, 1, 0, st>>>(src, dst);
    COUNT_LAUNCH(1);
}

void launch_halo_pack(const DeviceArrays& A, char* lo, char* hi, int sms, cudaStream_t st) {
    int64_t m = (int64_t)A.hx * A.rp;
    if (m > 0) { k_halo_pack<<<grid_for(m, 256, sms, 4), 256, 0, st>>>(A, lo, hi); COUNT_LAUNCH(1); }
}
void launch_halo_unpack(const DeviceArrays& A, const char* lo, const char* hi, DeviceCounters* dc, int sms, cudaStream_t st) {
    int64_t m = (int64_t)A.hx * A.rp;
    if (m > 0) { k_halo_unpack<<<grid_for(m, 256, sms, 4), 256, 0, st>>>(A, lo, hi, dc); COUNT_LAUNCH(1); }
}
void launch_grid_metric(int64_t n, const double* dx, const double* dy, const double* angle_dx, const double* lat,
                        double R_earth, double* M11, double* M12, double* M21, double* M22, double* pc, int sms, cudaStream_t st) {
    if (n > 0) k_grid_metric<<<grid_for(n, 256, sms, 8), 256, 0, st>>>(n, dx, dy, angle_dx, lat, R_earth, M11, M12, M21, M22, pc);
    COUNT_LAUNCH(1);
}
void launch_make_boundaries(const uint8_t* ocean, uint8_t* total, int Nx, int Ny, int bx, int by, int sms, cudaStream_t st) {
    (void)sms;
    dim3 grid((Nx + 255) / 256, Ny < 65535 ? Ny : 65535);
    k_make_boundaries<<<grid, 256, 0, st>>>(ocean, total, Nx, Ny, bx, by);
    COUNT_LAUNCH(1);
}
void launch_fields(int64_t n, const double* e, const double* mx, const double* my, double* Hs, double* cx, double* cy,
                   int sms, cudaStream_t st) {
    if (n > 0) k_fields<<<grid_for(n, 256, sms, 8), 256, 0, st>>>(n, e, mx, my, Hs, cx, cy);
    COUNT_LAUNCH(1);
}
void launch_fill_i32(int32_t* p, int64_t n, int32_t v, int sms, cudaStream_t st) {
    if (n > 0) k_fill_i32<<<grid_for(n, 256, sms, 4), 256, 0, st>>>(p, n, v);
    COUNT_LAUNCH(1);
}

void launch_selftest_math(uint64_t seed, int iters, unsigned long long* out, int sms, cudaStream_t st) {
    k_selftest_math<<<sms * 8, 256, 0, st>>>(seed, iters, out);
    COUNT_LAUNCH(1);
}
void launch_fp64_peak(double* out, int iters, int sms, cudaStream_t st, int64_t* fmas) {
    int blocks = sms * 8;
    k_fp64_peak<<<blocks, 256, 0, st>>>(out, iters);
    *fmas = (int64_t)blocks * 256 * (int64_t)iters * 64;
    COUNT_LAUNCH(1);
}
void launch_copy_f64(double* dst, const double* src, int64_t n, int sms, cudaStream_t st) {
    k_copy_f64<<<sms * 16, 256, 0, st>>>((double2*)dst, (const double2*)src, n / 2);
    COUNT_LAUNCH(1);
}

} /* namespace picles */
