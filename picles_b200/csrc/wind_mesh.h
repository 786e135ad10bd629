/*
 * wind_mesh.h — sampling of a gridded wind field at the model nodes (wind ingestion).
 *
 * The reference builds its wind closures from gridded data with Interpolations.jl,
 *     u_grid = LinearInterpolation((x, y, t), U, extrapolation_bc=Periodic())
 * (tests/T03_PIC_tripolar_realistic.jl:61-73, src/Utils/WindEmulator.jl:18-43) and calls
 * u(x, y, t) = u_grid(x, y, t) with the home-node coordinates of a particle.  Interpolations.jl is
 * a third-party dependency absent from /root/reference (Project.toml, no [compat] bound); the
 * restated rule is its published one:
 *   - Periodic() extrapolation maps every coordinate with  periodic(y, l, u) = mod(y-l, u-l) + l
 *     (l, u = first and last knot; Julia's floating-point mod: the sign follows the divisor);
 *   - Gridded(Linear()): knot interval i = clamp(#{knots < y}, 1, n-1), dx = (y - k_i)/(k_{i+1} - k_i),
 *     weights (1-dx, dx); the value is the nested weighted sum with the first axis outermost.
 *
 * `__host__ __device__` so tests/ can run the same code on the CPU against the CPU checker's own
 * restatement of the rule; the product only calls it from the wind kernels.  Build rules as physics.h (no contraction; nothing here needs an fma).
 */
#ifndef PICLES_WIND_MESH_H
#define PICLES_WIND_MESH_H

#include <math.h>
#include <stdint.h>

#include "pmath.h"

namespace picles {

struct WindMesh {
    int nx, ny, nt;              /* knots per axis */
    const double *xw, *yw, *tw;  /* knot vectors */
    const double *U, *V;         /* nt slices of ny*nx values, x fastest */
};

/* Julia mod(x, y) for Float64 (y > 0 here) */
PM_HD double wm_mod(double x, double y) {
    if (x >= 0.0 && x < y) return x + 0.0; /* fmod(x, y) == x exactly; +0.0: mod(-0.0, y) is +0.0 */
    double r = fmod(x, y);
    if (r == 0.0) return copysign(r, y);
    if ((r > 0.0) != (y > 0.0)) return r + y;
    return r;
}
/* periodic(y, l, u) */
PM_HD double wm_periodic(double y, double l, double u) { return wm_mod(y - l, u - l) + l; }

/* 0-based lower knot of the interval holding y (knots strictly increasing) and the weight of
   the upper knot: idx = clamp(#{knots < y} - 1, 0, n-2).  The count is found from a guess
   (exact for equally spaced knots, inv_h = (n-1)/(k[n-1]-k[0])) corrected by a short walk, with
   a bisection behind it for strongly non-uniform knots: same result as searchsortedfirst. */
PM_HD void wm_locate(const double* __restrict__ k, int n, double y, double inv_h, int& i, double& d) {
    double gf = (y - k[0]) * inv_h;
    int g = (gf >= 0.0) ? ((gf < (double)(n - 1)) ? (int)gf : n - 1) : 0; /* NaN -> 0 */
    int walk = 0;
    /* largest g with k[g] < y, or -1 */
    while (g >= 0 && !(k[g] < y) && walk < 4) { g--; walk++; }
    while (g + 1 < n && k[g + 1] < y && walk < 4) { g++; walk++; }
    if (walk >= 4) { /* bisection over the whole vector */
        int lo = 0, hi = n;
        while (lo < hi) {
            int mid = (lo + hi) >> 1;
            if (k[mid] < y) lo = mid + 1;
            else hi = mid;
        }
        g = lo - 1;
    }
    int idx = g;
    if (idx < 0) idx = 0;
    if (idx > n - 2) idx = n - 2;
    i = idx;
    const double l = k[idx], u = k[idx + 1];
#if defined(__CUDA_ARCH__)
    /* the compiler's own division fast path with its validity tests as a flag (pmath.h): equal
       to the IEEE quotient whenever the flag stays clear */
    unsigned bad = 0;
    const double q = pm_divz_fast(y - l, u - l, &bad);
    d = bad ? (y - l) / (u - l) : q;
#else
    d = (y - l) / (u - l);
#endif
}
PM_HD double wm_inv_h(const double* __restrict__ k, int n) { return (double)(n - 1) / (k[n - 1] - k[0]); }

/* time interval and weight: the same for every node of a level */
struct WindMeshTime {
    int it;
    double dt;
    double x0, x1, y0, y1, inv_hx, inv_hy; /* loop invariants of the spatial lookup */
};
PM_HD WindMeshTime wm_time(const WindMesh& W, double t) {
    WindMeshTime r;
    const double tp = wm_periodic(t, W.tw[0], W.tw[W.nt - 1]);
    wm_locate(W.tw, W.nt, tp, wm_inv_h(W.tw, W.nt), r.it, r.dt);
    r.x0 = W.xw[0]; r.x1 = W.xw[W.nx - 1]; r.y0 = W.yw[0]; r.y1 = W.yw[W.ny - 1];
    r.inv_hx = wm_inv_h(W.xw, W.nx); r.inv_hy = wm_inv_h(W.yw, W.ny);
    return r;
}

/* nested weighted sum over the 2 x 2 x 2 corners: a0/a1 point at the (ix, iy) corner of the
   lower / upper time slice, row = knots per mesh row */
PM_HD double wm_blend(const double* __restrict__ a0, const double* __restrict__ a1, int row, double dx, double dy,
                      double dt) {
    const double wx0 = 1.0 - dx, wy0 = 1.0 - dy, wt0 = 1.0 - dt;
    const double* __restrict__ b0 = a0 + row;
    const double* __restrict__ b1 = a1 + row;
    const double a00 = wt0 * a0[0] + dt * a1[0];
    const double a01 = wt0 * b0[0] + dt * b1[0];
    const double a10 = wt0 * a0[1] + dt * a1[1];
    const double a11 = wt0 * b0[1] + dt * b1[1];
    return wx0 * (wy0 * a00 + dy * a01) + dx * (wy0 * a10 + dy * a11);
}

/* u_grid(x, y, t), v_grid(x, y, t) */
PM_HD void wm_sample(const WindMesh& W, const WindMeshTime& T, double x, double y, double& u, double& v) {
    const double xp = wm_periodic(x, T.x0, T.x1);
    const double yp = wm_periodic(y, T.y0, T.y1);
    int ix, iy;
    double dx, dy;
    wm_locate(W.xw, W.nx, xp, T.inv_hx, ix, dx);
    wm_locate(W.yw, W.ny, yp, T.inv_hy, iy, dy);
    const int64_t st = (int64_t)W.nx * W.ny;
    const int off = ix + W.nx * iy; /* nx*ny < 2^31: checked when the mesh is set */
    const double* __restrict__ u0 = W.U + st * T.it + off;
    const double* __restrict__ v0 = W.V + st * T.it + off;
    u = wm_blend(u0, u0 + st, W.nx, dx, dy, T.dt);
    v = wm_blend(v0, v0 + st, W.nx, dx, dy, T.dt);
}

/* ---- the same sample in two passes --------------------------------------------------------
   The time interval and weight of a level are the same for every node, so the innermost blend of
   wm_blend, wt0*a0[p] + dt*a1[p], depends on the mesh point p only: wm_timeblend evaluates it once
   per mesh point (the same expression, hence the same bits) and wm_sample2d then does the spatial
   part of the nested sum on that slice — 4 gathered values and 9 operations per component and
   node instead of 8 and 21. */
PM_HD double wm_timeblend(const double* __restrict__ A, int64_t st, int it, double dt, int64_t p) {
    const double wt0 = 1.0 - dt;
    return wt0 * A[st * it + p] + dt * A[st * (it + 1) + p];
}
PM_HD double wm_blend2d(const double* __restrict__ a, int row, double dx, double dy) {
    const double wx0 = 1.0 - dx, wy0 = 1.0 - dy;
    const double* __restrict__ b = a + row;
    return wx0 * (wy0 * a[0] + dy * b[0]) + dx * (wy0 * a[1] + dy * b[1]);
}
/* Ub, Vb: the time-blended slices (nx*ny values each) */
PM_HD void wm_sample2d(const WindMesh& W, const WindMeshTime& T, const double* __restrict__ Ub,
                       const double* __restrict__ Vb, double x, double y, double& u, double& v) {
    const double xp = wm_periodic(x, T.x0, T.x1);
    const double yp = wm_periodic(y, T.y0, T.y1);
    int ix, iy;
    double dx, dy;
    wm_locate(W.xw, W.nx, xp, T.inv_hx, ix, dx);
    wm_locate(W.yw, W.ny, yp, T.inv_hy, iy, dy);
    const int off = ix + W.nx * iy;
    u = wm_blend2d(Ub + off, W.nx, dx, dy);
    v = wm_blend2d(Vb + off, W.nx, dx, dy);
}

/* Four consecutive nodes at once (k_wind_sample_x4).  On a regular grid
   the nodes of a row share y, and with it the y interval, its weight and the division behind it: they
   are looked up once per group and again only for a node whose y differs in any bit, so every node
   still gets exactly what wm_sample2d gives it. */
PM_HD void wm_sample2d_x4(const WindMesh& W, const WindMeshTime& T, const double* __restrict__ Ub,
                          const double* __restrict__ Vb, const double* x, const double* y, double* u, double* v) {
    int iy0;
    double dy0;
    wm_locate(W.yw, W.ny, wm_periodic(y[0], T.y0, T.y1), T.inv_hy, iy0, dy0);
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int k = 0; k < 4; k++) {
        int iy = iy0, ix;
        double dy = dy0, dx;
        if (k > 0 && pm_d2i(y[k]) != pm_d2i(y[0])) wm_locate(W.yw, W.ny, wm_periodic(y[k], T.y0, T.y1), T.inv_hy, iy, dy);
        wm_locate(W.xw, W.nx, wm_periodic(x[k], T.x0, T.x1), T.inv_hx, ix, dx);
        const int off = ix + W.nx * iy;
        u[k] = wm_blend2d(Ub + off, W.nx, dx, dy);
        v[k] = wm_blend2d(Vb + off, W.nx, dx, dy);
    }
}

/* ---- E member meshes on shared knots (k_wind_timeblend_members, k_wind_sample_members) -----
   An ensemble's meshes share xw, yw, tw and the node coordinates; U and V hold E meshes back to
   back, member slowest, and the time-blended scratch holds E slices of nx*ny points.  The time
   interval and weight are the same for every member, and a node's (ix, dx, iy, dy) does not depend
   on the member: it is located once and blended for each member with wm_blend2d, the expression
   wm_sample2d uses, so member m gets exactly what a single mesh made of member m's data gives. */
struct WindMeshNode {
    int off; /* ix + nx*iy */
    double dx, dy;
};
PM_HD WindMeshNode wm_node(const WindMesh& W, const WindMeshTime& T, double x, double y) {
    const double xp = wm_periodic(x, T.x0, T.x1);
    const double yp = wm_periodic(y, T.y0, T.y1);
    int ix, iy;
    WindMeshNode q;
    wm_locate(W.xw, W.nx, xp, T.inv_hx, ix, q.dx);
    wm_locate(W.yw, W.ny, yp, T.inv_hy, iy, q.dy);
    q.off = ix + W.nx * iy;
    return q;
}
/* pass 1 of member m at mesh point p (slice = nx*ny): member m's slice of the scratch */
PM_HD double wm_timeblend_member(const double* __restrict__ A, int64_t slice, int nt, int it, double dt, int m, int64_t p) {
    return wm_timeblend(A + (int64_t)m * nt * slice, slice, it, dt, p);
}
/* pass 2 for node l and members [m0, m1): u_out[m*n + l], v_out[m*n + l] (the layout of every
   per-node plane of an ensemble), so the stores of consecutive nodes stay consecutive per member */
PM_HD void wm_sample2d_members(const WindMesh& W, const WindMeshNode& q, const double* __restrict__ Ub,
                               const double* __restrict__ Vb, int m0, int m1, int64_t n, int64_t l,
                               double* __restrict__ u_out, double* __restrict__ v_out) {
    const int64_t slice = (int64_t)W.nx * W.ny;
    for (int m = m0; m < m1; m++) {
        const double u = wm_blend2d(Ub + slice * m + q.off, W.nx, q.dx, q.dy);
        const double v = wm_blend2d(Vb + slice * m + q.off, W.nx, q.dx, q.dy);
#if defined(__CUDA_ARCH__)
        __stcs(u_out + n * m + l, u);
        __stcs(v_out + n * m + l, v);
#else
        u_out[n * m + l] = u;
        v_out[n * m + l] = v;
#endif
    }
}

} /* namespace picles */
#endif
