/*
 * host_shim.cpp — TEST-ONLY host build of picles_b200/csrc/physics.h.
 *
 * Runs the product's per-particle / per-node device functions (advance_particle,
 * gather_node, remesh_particle, seed_particle) on the CPU with the same data layout and
 * strip/halo decomposition the CUDA kernels use, so the bit-exact comparison with the
 * oracle and the multi-strip logic can be checked without a GPU.  This file is not part
 * of the product and is never loaded by it.
 */
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../picles_b200/csrc/stiff.h"
#include "../picles_b200/csrc/wind_mesh.h"

using namespace picles;

struct Strip {
    int j0, ny, halo;
    std::vector<double> z[5], t, dt, qold, ut, vt, ut1, vt1, rec[5], S[3], M[4], pc;
    std::vector<int32_t> iter, cell;
    std::vector<uint8_t> flags, status, mask;
    std::vector<int8_t> as;
    std::vector<double> ulag, vlag; /* the lag wind level as the ABI layer keeps it (picles_capi.cu: keep_lag_level) */
};

struct Shim {
    int Nx, Ny, bx, by, nstrips, halo;
    picles_params_t P;
    double Mc[4];
    bool perM, hasPc;
    std::vector<Strip> s;
    Tally tally;
    int accumulate = 0;
    int reach_halo = 0; /* per-process strips: max reach of the received halo records */
    int n_mid = 0;      /* intermediate wind levels of the next step (global planes, consumed by it) */
    std::vector<double> u_mid, v_mid;
    int64_t steps_since_seed = 0;
};

static void load(const Strip& s, int64_t l, Particle& p) {
    p.u0 = s.z[0][l]; p.u1 = s.z[1][l]; p.u2 = s.z[2][l]; p.u3 = s.z[3][l]; p.u4 = s.z[4][l];
    p.t = s.t[l]; p.dt = s.dt[l]; p.qold = s.qold[l]; p.iter = s.iter[l]; p.flags = s.flags[l]; p.status = s.status[l];
    p.as = s.as[l];
}
static void store(Strip& s, int64_t l, const Particle& p) {
    s.z[0][l] = p.u0; s.z[1][l] = p.u1; s.z[2][l] = p.u2; s.z[3][l] = p.u3; s.z[4][l] = p.u4;
    s.t[l] = p.t; s.dt[l] = p.dt; s.qold[l] = p.qold; s.iter[l] = p.iter; s.flags[l] = p.flags; s.status[l] = p.status;
    s.as[l] = p.as;
}
static void tally_add(Tally& a, const Tally& b) {
    a.integrated += b.integrated; a.substeps += b.substeps; a.rejects += b.rejects; a.rhs += b.rhs;
    a.reseed += b.reseed; a.fixups += b.fixups; a.failed += b.failed; a.deposited += b.deposited;
    a.A += b.A; a.B += b.B; a.C += b.C; a.D += b.D;
    if (b.reach > a.reach) a.reach = b.reach;
    if (b.max_attempts > a.max_attempts) a.max_attempts = b.max_attempts;
    a.stiff_switches += b.stiff_switches; a.stiff_attempts += b.stiff_attempts;
}

extern "C" {

/* the third template argument of the k_advance instantiation the library launches (physics.h: ph_advance_variant),
   which the specialised host build runs the same copy of, for the tests to hold to their mirror */
int shim_advance_template(const picles_params_t* P, int per_node_M) { return ph_advance_variant(*P, per_node_M); }

Shim* shim_create(int Nx, int Ny, int bx, int by, int nstrips, int halo, const uint8_t* mask, const double* M,
                  const double* M_const, const double* pc, const picles_params_t* P) {
    Shim* h = new Shim();
    h->Nx = Nx; h->Ny = Ny; h->bx = bx; h->by = by; h->nstrips = nstrips; h->halo = (nstrips > 1) ? halo : 0;
    h->P = *P;
    h->perM = (M != nullptr);
    h->hasPc = (pc != nullptr);
    if (M_const) memcpy(h->Mc, M_const, sizeof h->Mc);
    h->s.resize(nstrips);
    int64_t plane = (int64_t)Nx * Ny;
    for (int r = 0; r < nstrips; r++) {
        Strip& s = h->s[r];
        s.j0 = (int)((int64_t)Ny * r / nstrips);
        int j1 = (int)((int64_t)Ny * (r + 1) / nstrips);
        s.ny = j1 - s.j0; s.halo = h->halo;
        int64_t n = (int64_t)Nx * s.ny, ne = (int64_t)Nx * (s.ny + 2 * s.halo);
        for (int k = 0; k < 5; k++) { s.z[k].assign(n, 0.0); s.rec[k].assign(ne, 0.0); }
        s.t.assign(n, 0.0); s.dt.assign(n, 0.0); s.qold.assign(n, 0.0);
        s.ut.assign(n, 0.0); s.vt.assign(n, 0.0); s.ut1.assign(n, 0.0); s.vt1.assign(n, 0.0);
        for (int k = 0; k < 3; k++) s.S[k].assign(n, 0.0);
        s.iter.assign(n, 0); s.cell.assign(ne, PH_CELL_INVALID);
        s.flags.assign(n, 0); s.status.assign(n, 0); s.as.assign(n, 0);
        s.mask.assign(mask + (int64_t)s.j0 * Nx, mask + (int64_t)s.j0 * Nx + n);
        if (M) for (int k = 0; k < 4; k++) s.M[k].assign(M + k * plane + (int64_t)s.j0 * Nx, M + k * plane + (int64_t)s.j0 * Nx + n);
        if (pc) s.pc.assign(pc + (int64_t)s.j0 * Nx, pc + (int64_t)s.j0 * Nx + n);
    }
    tally_zero(h->tally);
    return h;
}
void shim_destroy(Shim* h) { delete h; }
void shim_set_accumulate(Shim* h, int on) { h->accumulate = on ? 1 : 0; }
/* process-wide: take the specialised code paths (physics.h: ph_host_specialised) */
void shim_set_specialised(int on) { ph_host_specialised = on ? 1 : 0; }
int shim_get_specialised() { return ph_host_specialised; }
/* n_mid planes with the extent of the wind arrays of the next step call (global for shim_step,
   strip-local for shim_strip_advance) */
void shim_set_wind_midlevels(Shim* h, int n_mid, const double* u_mid, const double* v_mid, int64_t plane) {
    h->n_mid = n_mid;
    h->u_mid.assign(u_mid, u_mid + (size_t)n_mid * plane);
    h->v_mid.assign(v_mid, v_mid + (size_t)n_mid * plane);
}
/* the device-side wind mesh sampler (wind_mesh.h) on the host */
void shim_wind_mesh_sample(int nx, int ny, int nt, const double* xw, const double* yw, const double* tw, const double* U,
                           const double* V, int64_t n, const double* x, const double* y, double t, double* u_out,
                           double* v_out) {
    WindMesh W;
    W.nx = nx; W.ny = ny; W.nt = nt; W.xw = xw; W.yw = yw; W.tw = tw; W.U = U; W.V = V;
    const WindMeshTime T = wm_time(W, t);
    /* the two passes of the device sampler (k_wind_timeblend, k_wind_sample), checked against the
       one-pass form on every node */
    const int64_t st = (int64_t)nx * ny;
    std::vector<double> Ub(st), Vb(st);
    for (int64_t p = 0; p < st; p++) { Ub[p] = wm_timeblend(U, st, T.it, T.dt, p); Vb[p] = wm_timeblend(V, st, T.it, T.dt, p); }
    int rc = 0;
    for (int64_t l = 0; l < n; l++) {
        wm_sample2d(W, T, Ub.data(), Vb.data(), x[l], y[l], u_out[l], v_out[l]);
        double u1, v1;
        wm_sample(W, T, x[l], y[l], u1, v1);
        if (memcmp(&u1, &u_out[l], 8) != 0 || memcmp(&v1, &v_out[l], 8) != 0) rc = 1; /* the two forms must agree bit for bit */
    }
    /* ... and the four-nodes-at-once form (shared y lookup along a row) */
    for (int64_t l = 0; l + 4 <= n; l += 4) {
        double u4[4], v4[4];
        wm_sample2d_x4(W, T, Ub.data(), Vb.data(), x + l, y + l, u4, v4);
        if (memcmp(u4, u_out + l, 32) != 0 || memcmp(v4, v_out + l, 32) != 0) rc = 1;
    }
    if (rc) { for (int64_t l = 0; l < n; l++) u_out[l] = v_out[l] = NAN; }
}

/* the ensemble wind sampler of wind_mesh.h (k_wind_timeblend_members + k_wind_sample_members): E meshes on shared
   knots (U, V: E*nt*ny*nx values, member slowest) sampled at n nodes into E planes of n values; members in chunks of
   `chunk`, as the device's blockIdx.y takes them */
void shim_wind_mesh_sample_members(int nx, int ny, int nt, int E, int chunk, const double* xw, const double* yw,
                                   const double* tw, const double* U, const double* V, int64_t n, const double* x,
                                   const double* y, double t, double* u_out, double* v_out) {
    WindMesh W;
    W.nx = nx; W.ny = ny; W.nt = nt; W.xw = xw; W.yw = yw; W.tw = tw; W.U = U; W.V = V;
    const WindMeshTime T = wm_time(W, t);
    const int64_t st = (int64_t)nx * ny;
    std::vector<double> Ub(st * E), Vb(st * E);
    for (int m = 0; m < E; m++)
        for (int64_t p = 0; p < st; p++) {
            Ub[st * m + p] = wm_timeblend_member(U, st, nt, T.it, T.dt, m, p);
            Vb[st * m + p] = wm_timeblend_member(V, st, nt, T.it, T.dt, m, p);
        }
    for (int m0 = 0; m0 < E; m0 += chunk) {
        const int m1 = m0 + chunk < E ? m0 + chunk : E;
        for (int64_t l = 0; l < n; l++) {
            const WindMeshNode q = wm_node(W, T, x[l], y[l]);
            wm_sample2d_members(W, q, Ub.data(), Vb.data(), m0, m1, n, l, u_out, v_out);
        }
    }
}

void shim_seed(Shim* h, const double* u0, const double* v0) {
    h->steps_since_seed = 0;
    for (auto& s : h->s) {
        s.ulag.clear(); s.vlag.clear();
        int64_t n = (int64_t)h->Nx * s.ny, off = (int64_t)s.j0 * h->Nx;
        for (int64_t l = 0; l < n; l++) {
            Particle p;
            double e, mx, my;
            seed_particle(h->P, s.mask[l], u0[off + l], v0[off + l], p, e, mx, my);
            store(s, l, p);
            s.S[0][l] = e; s.S[1][l] = mx; s.S[2][l] = my;
        }
        std::fill(s.cell.begin(), s.cell.end(), PH_CELL_INVALID);
    }
}

static void shim_advance_all(Shim* h, double DT, const double* u_t, const double* v_t, const double* u_t1,
                             const double* v_t1, Tally& T, bool local_winds) {
    const int Nx = h->Nx;
    for (auto& s : h->s) {
        int64_t n = (int64_t)Nx * s.ny, off = local_winds ? 0 : (int64_t)s.j0 * Nx;
        for (int64_t l = 0; l < n; l++) {
            if (!(s.flags[l] & PICLES_PF_ACTIVE)) continue;
            Particle p;
            load(s, l, p);
            double M[4];
            if (h->perM) { M[0] = s.M[0][l]; M[1] = s.M[1][l]; M[2] = s.M[2][l]; M[3] = s.M[3][l]; }
            else memcpy(M, h->Mc, sizeof M);
            double pc = h->hasPc ? s.pc[l] : 0.0;
            Record r;
            Tally c;
            tally_zero(c);
            KLocal K;
            double um[PH_WIND_SEG_MAX] = {0, 0, 0, 0}, vm[PH_WIND_SEG_MAX] = {0, 0, 0, 0};
            {
                /* mid-level planes have the extent of the wind arrays: global, or strip-local */
                const int64_t plane = local_winds ? n : (int64_t)Nx * h->Ny;
                for (int k = 0; k < h->n_mid; k++) { um[k] = h->u_mid[k * plane + off + l]; vm[k] = h->v_mid[k * plane + off + l]; }
            }
            const double t_start = p.t;
            int attempts = 0;
            /* as k_advance: a particle seeded off under B-1 as run reads the level kept from the first step */
            double wu1 = u_t1[off + l], wv1 = v_t1[off + l];
            if (!s.ulag.empty() && !(p.flags & PICLES_PF_ON)) { wu1 = s.ulag[l]; wv1 = s.vlag[l]; }
            /* as launch_advance picks the kernel.  For 0 the host runs advance_particle<true, 0> whatever the solver,
               where the device's generic Tsit5 / DP5 kernels run advance_particle<false, 0>: on the host the monitor
               is gated on the solver at run time (physics.h integrate), so both compute the same. */
            const int tsit5 = ph_host_specialised ? ph_advance_variant(h->P, h->perM) : 0;
            const bool pending = (tsit5 == 1)
                ? advance_particle<false, 1>(h->P, p, s.mask[l], DT, u_t[off + l], v_t[off + l], wu1,
                                             wv1, h->n_mid, um, vm, M, pc, r, c, K, attempts)
                : (tsit5 == 2)
                ? advance_particle<false, 2>(h->P, p, s.mask[l], DT, u_t[off + l], v_t[off + l], wu1,
                                             wv1, h->n_mid, um, vm, M, pc, r, c, K, attempts)
                : (tsit5 == 3)
                ? advance_particle<true, 3>(h->P, p, s.mask[l], DT, u_t[off + l], v_t[off + l], wu1,
                                            wv1, h->n_mid, um, vm, M, pc, r, c, K, attempts)
                : advance_particle<true>(h->P, p, s.mask[l], DT, u_t[off + l], v_t[off + l], wu1,
                                         wv1, h->n_mid, um, vm, M, pc, r, c, K, attempts);

            if (pending) { /* as the kernel: the stiff part of the step runs through advance_resume */
                ResumeArgs R;
                R.mask = s.mask[l]; R.nmid = h->n_mid; R.attempts = attempts;
                R.DT = DT; R.t_start = t_start;
                R.wu0 = u_t[off + l]; R.wv0 = v_t[off + l]; R.wu1 = u_t1[off + l]; R.wv1 = v_t1[off + l];
                for (int k = 0; k < PH_WIND_SEG_MAX; k++) { R.um[k] = um[k]; R.vm[k] = vm[k]; }
                memcpy(R.M, M, sizeof R.M);
                R.pc = pc;
                Tally c2;
                tally_zero(c2);
                advance_resume(&h->P, &R, &p, &r, &c2, K);
                tally_add(c, c2);
            }
            tally_add(T, c);
            store(s, l, p);
            int64_t le = l + (int64_t)s.halo * Nx;
            s.rec[0][le] = r.e; s.rec[1][le] = r.mx; s.rec[2][le] = r.my; s.rec[3][le] = r.wxc; s.rec[4][le] = r.wyc;
            s.cell[le] = r.cell;
        }
        /* keep_lag_level of the ABI layer: behind the first step's advance, only when a particle was seeded off */
        if (h->steps_since_seed == 0 && !h->P.on_persist) {
            bool any_off = false;
            for (int64_t l = 0; l < n; l++) any_off = any_off || ((s.flags[l] & PICLES_PF_ACTIVE) && !(s.flags[l] & PICLES_PF_ON));
            if (any_off) { s.ulag.assign(u_t1 + off, u_t1 + off + n); s.vlag.assign(v_t1 + off, v_t1 + off + n); }
        }
    }
    h->steps_since_seed++;
}

static void shim_project_remesh_all(Shim* h, double DT, int R, const double* u_t, const double* v_t, Tally& T,
                                    bool local_winds) {
    const int Nx = h->Nx;
    for (auto& s : h->s) {
        RecView V;
        V.Nx = Nx; V.Ny = h->Ny; V.bx = h->bx; V.by = h->by; V.j0 = s.j0; V.ny = s.ny; V.halo = s.halo; V.hx = s.halo; V.pitch = Nx;
        V.e = s.rec[0].data(); V.mx = s.rec[1].data(); V.my = s.rec[2].data(); V.wx = s.rec[3].data(); V.wy = s.rec[4].data();
        V.cell = s.cell.data();
        int64_t n = (int64_t)Nx * s.ny, off = local_winds ? 0 : (int64_t)s.j0 * Nx;
        for (int64_t l = 0; l < n; l++) {
            int I = (int)(l % Nx) + 1, J = (int)(l / Nx) + 1 + s.j0;
            if (!h->accumulate) { s.S[0][l] = 0.0; s.S[1][l] = 0.0; s.S[2][l] = 0.0; }
            gather_node(V, I, J, R, h->P.periodic_boundary ? 2 : 1, s.S[0][l], s.S[1][l], s.S[2][l]);
        }
        for (int64_t l = 0; l < n; l++) {
            if (!(s.flags[l] & PICLES_PF_ACTIVE)) continue;
            Particle p;
            load(s, l, p);
            Tally c;
            tally_zero(c);
            remesh_particle(h->P, p, s.S[0][l], s.S[1][l], s.S[2][l], u_t[off + l], v_t[off + l], DT, c);
            tally_add(T, c);
            store(s, l, p);
        }
    }
}

void shim_step(Shim* h, double t, double DT, const double* u_t, const double* v_t, const double* u_t1, const double* v_t1) {
    (void)t;
    const int Nx = h->Nx;
    Tally T;
    tally_zero(T);
    shim_advance_all(h, DT, u_t, v_t, u_t1, v_t1, T, false);
    h->n_mid = 0;
    /* halo exchange: my first/last H owned rows -> neighbour's upper/lower halo rows */
    int H = h->halo, ns = h->nstrips;
    if (ns > 1 && H > 0) {
        for (int r = 0; r < ns; r++) {
            Strip& s = h->s[r];
            int64_t m = (int64_t)H * Nx;
            int lo = r - 1, hi = r + 1;
            if (h->by == PICLES_BND_PERIODIC) { lo = (lo + ns) % ns; hi = hi % ns; }
            if (lo >= 0) { /* my first H owned rows -> upper halo of the lower neighbour */
                Strip& d = h->s[lo];
                int64_t src = (int64_t)H * Nx, dst = (int64_t)(d.ny + H) * Nx;
                for (int k = 0; k < 5; k++) memcpy(&d.rec[k][dst], &s.rec[k][src], m * 8);
                memcpy(&d.cell[dst], &s.cell[src], m * 4);
            }
            if (hi < ns) { /* my last H owned rows -> lower halo of the upper neighbour */
                Strip& d = h->s[hi];
                int64_t src = (int64_t)s.ny * Nx, dst = 0;
                for (int k = 0; k < 5; k++) memcpy(&d.rec[k][dst], &s.rec[k][src], m * 8);
                memcpy(&d.cell[dst], &s.cell[src], m * 4);
            }
        }
    }
    int R = T.reach < PH_REACH_MAX ? T.reach : PH_REACH_MAX;
    if (ns > 1 && R > H) R = H;
    shim_project_remesh_all(h, DT, R, u_t, v_t, T, false);
    h->tally = T;
}

/* ---- one strip per process: the phase-split interface of the C ABI ---------------- */
Shim* shim_create_strip(int Nx, int Ny, int bx, int by, int j0, int ny, int halo, const uint8_t* mask /* ny*Nx */,
                        const double* M /* 4 planes ny*Nx */, const double* M_const, const double* pc,
                        const picles_params_t* P) {
    Shim* h = new Shim();
    h->Nx = Nx; h->Ny = Ny; h->bx = bx; h->by = by; h->nstrips = (ny == Ny) ? 1 : 2; h->halo = halo;
    h->P = *P;
    h->perM = (M != nullptr);
    h->hasPc = (pc != nullptr);
    if (M_const) memcpy(h->Mc, M_const, sizeof h->Mc);
    h->s.resize(1);
    Strip& s = h->s[0];
    s.j0 = j0; s.ny = ny; s.halo = halo;
    int64_t n = (int64_t)Nx * ny, ne = (int64_t)Nx * (ny + 2 * halo);
    for (int k = 0; k < 5; k++) { s.z[k].assign(n, 0.0); s.rec[k].assign(ne, 0.0); }
    s.t.assign(n, 0.0); s.dt.assign(n, 0.0); s.qold.assign(n, 0.0);
    for (int k = 0; k < 3; k++) s.S[k].assign(n, 0.0);
    s.iter.assign(n, 0); s.cell.assign(ne, PH_CELL_INVALID);
    s.flags.assign(n, 0); s.status.assign(n, 0); s.as.assign(n, 0);
    s.mask.assign(mask, mask + n);
    if (M) for (int k = 0; k < 4; k++) s.M[k].assign(M + k * n, M + (k + 1) * n);
    if (pc) s.pc.assign(pc, pc + n);
    tally_zero(h->tally);
    return h;
}
void shim_strip_seed(Shim* h, const double* u0, const double* v0) {
    Strip& s = h->s[0];
    h->steps_since_seed = 0;
    s.ulag.clear(); s.vlag.clear();
    int64_t n = (int64_t)h->Nx * s.ny;
    for (int64_t l = 0; l < n; l++) {
        Particle p;
        double e, mx, my;
        seed_particle(h->P, s.mask[l], u0[l], v0[l], p, e, mx, my);
        store(s, l, p);
        s.S[0][l] = e; s.S[1][l] = mx; s.S[2][l] = my;
    }
    std::fill(s.cell.begin(), s.cell.end(), PH_CELL_INVALID);
}
void shim_strip_advance(Shim* h, double DT, const double* u_t, const double* v_t, const double* u_t1, const double* v_t1) {
    Tally T;
    tally_zero(T);
    shim_advance_all(h, DT, u_t, v_t, u_t1, v_t1, T, true);
    h->n_mid = 0;
    h->tally = T;
    h->reach_halo = 0;
}
int64_t shim_strip_halo_bytes(const Shim* h) { return (int64_t)h->halo * h->Nx * 44; }
/* same packing as k_halo_pack / k_halo_unpack: 5 planes of doubles then the cell plane */
void shim_strip_pack(const Shim* h, char* lo, char* hi) {
    const Strip& s = h->s[0];
    int64_t m = (int64_t)h->halo * h->Nx;
    for (int k = 0; k < 5; k++) {
        memcpy(lo + k * m * 8, &s.rec[k][(int64_t)s.halo * h->Nx], m * 8);
        memcpy(hi + k * m * 8, &s.rec[k][(int64_t)s.ny * h->Nx], m * 8);
    }
    memcpy(lo + 5 * m * 8, &s.cell[(int64_t)s.halo * h->Nx], m * 4);
    memcpy(hi + 5 * m * 8, &s.cell[(int64_t)s.ny * h->Nx], m * 4);
}
void shim_strip_unpack(Shim* h, const char* lo, const char* hi) {
    Strip& s = h->s[0];
    int64_t m = (int64_t)h->halo * h->Nx;
    for (int k = 0; k < 5; k++) {
        memcpy(&s.rec[k][0], lo + k * m * 8, m * 8);
        memcpy(&s.rec[k][(int64_t)(s.ny + s.halo) * h->Nx], hi + k * m * 8, m * 8);
    }
    memcpy(&s.cell[0], lo + 5 * m * 8, m * 4);
    memcpy(&s.cell[(int64_t)(s.ny + s.halo) * h->Nx], hi + 5 * m * 8, m * 4);
    /* as k_halo_unpack: the gather's window must cover the neighbours' deposits too */
    for (int64_t q = 0; q < m; q++) {
        int r = cell_reach(s.cell[q]);
        if (r > h->reach_halo) h->reach_halo = r;
        r = cell_reach(s.cell[(int64_t)(s.ny + s.halo) * h->Nx + q]);
        if (r > h->reach_halo) h->reach_halo = r;
    }
}
void shim_strip_project_remesh(Shim* h, double DT, const double* u_t, const double* v_t) {
    Tally T = h->tally;
    int R = T.reach > h->reach_halo ? T.reach : h->reach_halo;
    if (R > PH_REACH_MAX) R = PH_REACH_MAX;
    if (h->s[0].ny != h->Ny && R > h->halo) R = h->halo;
    shim_project_remesh_all(h, DT, R, u_t, v_t, T, true);
    h->tally = T;
}

void shim_get_state(const Shim* h, double* S) {
    int64_t plane = (int64_t)h->Nx * h->Ny;
    for (auto& s : h->s) {
        int64_t n = (int64_t)h->Nx * s.ny, off = (int64_t)s.j0 * h->Nx;
        for (int k = 0; k < 3; k++) memcpy(S + k * plane + off, s.S[k].data(), n * 8);
    }
}
void shim_set_state(Shim* h, const double* S) {
    int64_t plane = (int64_t)h->Nx * h->Ny;
    for (auto& s : h->s) {
        int64_t n = (int64_t)h->Nx * s.ny, off = (int64_t)s.j0 * h->Nx;
        for (int k = 0; k < 3; k++) memcpy(s.S[k].data(), S + k * plane + off, n * 8);
    }
}
void shim_get_particles(const Shim* h, double* z, double* t, double* dt, double* qold, int32_t* iter, uint8_t* flags,
                        int32_t* status) {
    int64_t plane = (int64_t)h->Nx * h->Ny;
    for (auto& s : h->s) {
        int64_t n = (int64_t)h->Nx * s.ny, off = (int64_t)s.j0 * h->Nx;
        for (int k = 0; k < 5; k++) memcpy(z + k * plane + off, s.z[k].data(), n * 8);
        memcpy(t + off, s.t.data(), n * 8);
        memcpy(dt + off, s.dt.data(), n * 8);
        memcpy(qold + off, s.qold.data(), n * 8);
        memcpy(iter + off, s.iter.data(), n * 4);
        memcpy(flags + off, s.flags.data(), n);
        for (int64_t l = 0; l < n; l++) status[off + l] = s.status[l];
    }
}
/* strip-local accessors (shim_create_strip handles: one strip, local plane size) */
void shim_get_state_local(const Shim* h, double* S) {
    const Strip& s = h->s[0];
    int64_t n = (int64_t)h->Nx * s.ny;
    for (int k = 0; k < 3; k++) memcpy(S + k * n, s.S[k].data(), n * 8);
}
void shim_get_particles_local(const Shim* h, double* z, double* t, double* dt, double* qold, int32_t* iter,
                              uint8_t* flags, int32_t* status) {
    const Strip& s = h->s[0];
    int64_t n = (int64_t)h->Nx * s.ny;
    for (int k = 0; k < 5; k++) memcpy(z + k * n, s.z[k].data(), n * 8);
    memcpy(t, s.t.data(), n * 8);
    memcpy(dt, s.dt.data(), n * 8);
    memcpy(qold, s.qold.data(), n * 8);
    memcpy(iter, s.iter.data(), n * 4);
    memcpy(flags, s.flags.data(), n);
    for (int64_t l = 0; l < n; l++) status[l] = s.status[l];
}
/* integrated, substeps, rejects, rhs, reseed, fixups, failed, deposited, A, B, C, D, reach, max_attempts,
   stiff_switches, stiff_attempts */
void shim_get_tally(const Shim* h, int32_t* out16) { memcpy(out16, &h->tally, 16 * sizeof(int32_t)); }
void shim_get_solver_state(const Shim* h, int8_t* as) {
    for (auto& s : h->s) memcpy(as + (int64_t)s.j0 * h->Nx, s.as.data(), s.as.size());
}
void shim_get_solver_state_local(const Shim* h, int8_t* as) { memcpy(as, h->s[0].as.data(), h->s[0].as.size()); }

int64_t shim_corner_target(int Nx, int Ny, int bx, int by, int64_t i, int64_t j) {
    int64_t ii, jj;
    if (!corner_target(Nx, Ny, bx, by, i, j, ii, jj)) return -1;
    return (ii - 1) + (jj - 1) * (int64_t)Nx;
}
void shim_rhs(const picles_params_t* P, const double* z, double u, double v, const double* M, double pc, double* dz) {
    Hoist H;
    H.y_rg = 0.0; H.y_eT = 0.0; H.us0 = 0.0; H.steady = false; H.steady_warp = false; H.std_terms = false;
    rhs3<OpsSafe, false>(*P, H, z[0], z[1], z[2], u, v, sqrt(u * u + v * v), pc, dz[0], dz[1], dz[2], (unsigned*)0);
    prop(*P, M, z[1], z[2], dz[3], dz[4]);
}
void shim_pack_roundtrip(int32_t fx, int32_t fy, int cls, int32_t* out3) {
    int32_t c = pack_cell(fx, fy, cls);
    int k;
    unpack_cell(c, out3[0], out3[1], k);
    out3[2] = k;
}
}
