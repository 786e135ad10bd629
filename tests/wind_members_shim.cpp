/* Host build of the ensemble wind sampler of wind_mesh.h (k_wind_timeblend_members + k_wind_sample_members), for
   tests/test_ensemble_wind_mesh.py.  Built with the flags of tests/host_shim.cpp (no contraction). */
#include <stdint.h>

#include <vector>

#include "../picles_b200/csrc/wind_mesh.h"

using namespace picles;

extern "C" {

/* E meshes on shared knots (U, V: E*nt*ny*nx values, member slowest) sampled at n nodes into E planes of n values;
   members in chunks of `chunk`, as the device's blockIdx.y takes them */
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

} /* extern "C" */
