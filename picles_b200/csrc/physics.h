/*
 * physics.h — per-particle arithmetic of the PiCLES particle-in-cell step, written for
 * the sm_100a kernels (registers only, no arrays of stage derivatives for the
 * propagation components, explicit fused multiply-adds).
 *
 * Every function is `__host__ __device__` so that tests/ can compile this header with
 * g++ and compare it bit-for-bit with the CPU oracle before any GPU time is spent;
 * the product itself only ever calls these from kernels (there is no CPU path).
 *
 * Build rules: device code with --fmad=false, host code with -ffp-contract=off.  All
 * contractions are written out with fma(), all transcendentals come from pmath.h, so
 * host and device agree bit-for-bit and accept/reject decisions of the adaptive
 * controller cannot flip.
 *
 * Reference call sites (paths relative to /root/reference/src):
 *   rhs3 / prop      ParticleSystems/particle_waves_v5.jl:479-556
 *   integrate        Operators/mapping_2D.jl:152  step!(integ, DT, true)  [OrdinaryDiffEq Tsit5/DP5]
 *   initdt           Operators/mapping_2D.jl:95,103,110 auto_dt_reset!     [OrdinaryDiffEq initdt]
 *   windsea          FetchRelations.jl:314-359
 *   charge / vertex  Operators/core_2D.jl:69-78, 121-128
 *   weights_1d       ParticleInCell.jl:58-71
 *   corner_target    ParticleInCell.jl:341-376, 409-428, 444-466
 *   advance_particle Operators/mapping_2D.jl:118-243
 *   remesh_particle  Operators/mapping_2D.jl:250-356
 */
#ifndef PICLES_PHYSICS_H
#define PICLES_PHYSICS_H

#include "../../include/picles_b200.h"
#include "pmath.h"

#if defined(__CUDACC__)
#define PM_HD_NOINLINE_DECL __host__ __device__ __noinline__
#else
#define PM_HD_NOINLINE_DECL static inline
#endif

#if defined(__CUDACC__)
#define PM_HDM __host__ __device__ __forceinline__
#else
#define PM_HDM inline
#endif

#define PH_QOLDINIT 1e-4
#define PH_LOG_QOLDINIT (-0x1.26bb1bbb55515p+3) /* = pm_log(PH_QOLDINIT) */
#define PH_CELL_INVALID ((int32_t)-1)
#define PH_CELL_PENDING ((int32_t)-2) /* AutoTsit5: the particle's step is finished by the resume kernel */
#define PH_CELL_BIAS 8192
#define PH_REACH_MAX 15
#define PH_WIND_SEG_MAX (PICLES_WIND_MID_MAX + 1) /* time segments of the staged wind: levels - 1 */

namespace picles {

#if !defined(__CUDACC__)
/* tests/host_shim.cpp only: run the specialised copies (switch-free right-hand side, Tsit5
   instantiation) on the host where the kernels would pick them, so the CPU suite covers them */
inline int ph_host_specialised = 0;
#endif

/* the advance kernel a step launches (launch_advance, picles_kernels.cu; the specialised host build runs the same
   copy): the TSIT5 template argument of k_advance, whose AUTOSW is solver == AutoTsit5.  1 Tsit5 and 2 DP5 on a
   uniform kernel (their tableaus at compile time), 3 AutoTsit5: each takes propagation as on; 0 the generic one,
   which also serves the reference's propagation = false switch.  nan_eest_rejects lives in the generic one only: the
   specialised ones keep the code they were measured with. */
inline int ph_advance_variant(const picles_params_t& P, bool per_node_M) {
    if (!P.propagation || P.nan_eest_rejects) return 0;
    if (P.solver == PICLES_SOLVER_AUTOTSIT5) return 3;
    if (P.solver == PICLES_SOLVER_TSIT5) return 1;
    if (P.solver == PICLES_SOLVER_DP5 && !per_node_M) return 2; /* -1.5 % on the bench06 settings */
    return 0;
}

/* ---- tableaus (OrdinaryDiffEq Tsit5ConstantCache / DP5ConstantCache) ----- */
/* a[s][j]: weight of k_j in the argument of stage s (s = 2..7, j = 1..s-1; row 7 = b);
   c[s-1]: time fraction of stage s; bt[j]: error weights (btilde). */
struct Tableau {
    double c[8];
    double a[8][8];
    double bt[8];
    double beta1, beta2;
};
#define PH_TABLEAU_INIT                                                                                          \
    {                                                                                                            \
        /* Tsit5 */                                                                                              \
        {{0, 0.161, 0.327, 0.9, 0.9800255409045097, 1.0, 1.0, 0},                                                \
         {{0}, {0},                                                                                              \
          {0, 0.161},                                                                                            \
          {0, -0.008480655492356989, 0.335480655492357},                                                         \
          {0, 2.8971530571054935, -6.359448489975075, 4.3622954328695815},                                       \
          {0, 5.325864828439257, -11.748883564062828, 7.4955393428898365, -0.09249506636175525},                 \
          {0, 5.86145544294642, -12.92096931784711, 8.159367898576159, -0.071584973281401, -0.028269050394068383}, \
          {0, 0.09646076681806523, 0.01, 0.4798896504144996, 1.379008574103742, -3.290069515436081,              \
           2.324710524099774}},                                                                                  \
         {0, -0.00178001105222577714, -0.0008164344596567469, 0.007880878010261995, -0.1447110071732629,         \
          0.5823571654525552, -0.45808210592918697, 0.015151515151515152},                                       \
         0.14, 0.08},                                                                                            \
        /* DP5 */                                                                                                \
        {{0, 0.2, 0.3, 0.8, 8.0 / 9.0, 1.0, 1.0, 0},                                                             \
         {{0}, {0},                                                                                              \
          {0, 0.2},                                                                                              \
          {0, 3.0 / 40.0, 9.0 / 40.0},                                                                           \
          {0, 44.0 / 45.0, -56.0 / 15.0, 32.0 / 9.0},                                                            \
          {0, 19372.0 / 6561.0, -25360.0 / 2187.0, 64448.0 / 6561.0, -212.0 / 729.0},                            \
          {0, 9017.0 / 3168.0, -355.0 / 33.0, 46732.0 / 5247.0, 49.0 / 176.0, -5103.0 / 18656.0},                \
          {0, 35.0 / 384.0, 0.0, 500.0 / 1113.0, 125.0 / 192.0, -2187.0 / 6784.0, 11.0 / 84.0}},                 \
         {0, -71.0 / 57600.0, 0.0, 71.0 / 16695.0, -71.0 / 1920.0, 17253.0 / 339200.0, -22.0 / 525.0,            \
          1.0 / 40.0},                                                                                           \
         0.17, 0.04}                                                                                             \
    }
#if defined(__CUDACC__)
__constant__ Tableau d_tableaus[2] = PH_TABLEAU_INIT;
#endif
static const Tableau h_tableaus[2] = PH_TABLEAU_INIT;

PM_HD const Tableau& tableau(int solver) {
    int k = (solver == PICLES_SOLVER_DP5) ? 1 : 0;
#if defined(__CUDA_ARCH__)
    return d_tableaus[k];
#else
    return h_tableaus[k];
#endif
}

/* per-thread scratch of one integration: the stage derivatives k_j[c] (j = 1..7, c = 0..2) and
   the loop-carried scalars that are touched once per stage or less (slots below).  Shared
   memory on the device, one column per thread (consecutive threads -> consecutive 8-byte
   words: conflict-free), so the registers go to the right-hand side; a local array on the
   host. */
enum {
    KS_U3 = 21, KS_U4, KS_TSTOP, KS_LQ, KS_QOLD, KS_DT0, KS_D1N, KS_DTMIN,
    KS_WT0, KS_WIDT,
    KS_G60, KS_G61, /* AutoTsit5 monitor: argument of stage 6, components 0 and 1 (component 2: KS_DT0, idle during attempts) */
    KS_AS,        /* AutoTsit5: AutoSwitch run length (as a double; +PH_AS_STIFF once switched) */
    KS_WCU,                            /* Newton coefficients c_1..c_4 of the wind's u component in time */
    KS_WCV = KS_WCU + PH_WIND_SEG_MAX, /* ... and of v */
    KS_SLOTS = KS_WCV + PH_WIND_SEG_MAX
};
struct KLocal {
    double k[KS_SLOTS];
    PM_HDM double get(int j, int c) const { return k[(j - 1) * 3 + c]; }
    PM_HDM void set(int j, int c, double v) { k[(j - 1) * 3 + c] = v; }
    PM_HDM double ld(int slot) const { return k[slot]; }
    PM_HDM void st(int slot, double v) { k[slot] = v; }
};
struct KStrided {
    double* base; /* &smem[threadIdx.x] */
    int stride;   /* blockDim.x */
    PM_HDM double get(int j, int c) const { return base[((j - 1) * 3 + c) * stride]; }
    PM_HDM void set(int j, int c, double v) { base[((j - 1) * 3 + c) * stride] = v; }
    PM_HDM double ld(int slot) const { return base[slot * stride]; }
    PM_HDM void st(int slot, double v) { base[slot * stride] = v; }
};

/* per-thread view of one particle (ODEIntegrator fields that survive between steps) */
struct Particle {
    double u0, u1, u2, u3, u4; /* lne, c̄_x, c̄_y, x, y */
    double t, dt, qold;
    int32_t iter;
    uint8_t flags;  /* PICLES_PF_* */
    uint8_t status; /* PICLES_PST_* */
    int8_t as;      /* AutoTsit5: run length of the stiffness test, +64 while Rosenbrock23 is current */
};
#define PH_AS_STIFF 64
#define PH_AS_CLAMP 60

/* wind at the home node: nseg+1 levels equally spaced over [t, t+DT] (lvl[0] = level t,
   lvl[nseg] = level t+DT; nseg = 1 unless intermediate levels were staged) */
struct Wind {
    double ul[PH_WIND_SEG_MAX + 1], vl[PH_WIND_SEG_MAX + 1];
    int nseg;
    double t_start, inv_DT;
};

/* Newton forward-difference coefficients of the interpolant through equally spaced levels:
   w(sigma) = c0 + sigma*(c1 + (sigma-1)*(c2 + (sigma-2)*(c3 + (sigma-3)*c4))), sigma = nseg*(t - t0)/DT,
   c_m = Delta^m w_0 / m!.  Two levels: c1 = w1 - w0, the linear rule.  In place: l[0..nseg] -> c[0..nseg]. */
PM_HD void wind_newton(double* l, int nseg) {
    /* compile-time trip counts, predicated on nseg: every index is an immediate after unrolling,
       so the levels stay in registers on the device */
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int m = 1; m <= PH_WIND_SEG_MAX; m++) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (int k = PH_WIND_SEG_MAX; k >= m; k--)
            if (k <= nseg) l[k] = l[k] - l[k - 1];
    }
    if (nseg >= 2) l[2] = l[2] * 0.5;
    if (nseg >= 3) l[3] = l[3] * (1.0 / 6.0);
    if (nseg >= 4) l[4] = l[4] * (1.0 / 24.0);
}

/* loop invariants of one particle's integration, hoisted out of the stage loop */
struct Hoist {
    double y_rg, y_eT; /* Newton reciprocals of r_g and e_T (fast path only) */
    double us0;        /* sqrt(u0^2+v0^2): the wind speed when the wind does not change over DT */
    bool steady;       /* every time coefficient of the staged wind is zero */
    bool steady_warp;  /* ... for every lane of the warp that was here when the invariants were formed (device) */
    bool std_terms;    /* every source term on and n == 2 (the defaults): the right-hand side instantiated without its term switches */
    int nseg;          /* time segments of the staged wind (levels - 1) */
};

/* per-thread counter deltas */
struct Tally {
    int32_t integrated, substeps, rejects, rhs, reseed, fixups, failed, deposited, A, B, C, D;
    int32_t reach, max_attempts;
    int32_t stiff_switches, stiff_attempts; /* AutoTsit5: Tsit5 -> Rosenbrock23 switches, Rosenbrock23 attempts */
};
PM_HD void tally_zero(Tally& c) {
    c.integrated = c.substeps = c.rejects = c.rhs = c.reseed = c.fixups = c.failed = c.deposited = 0;
    c.A = c.B = c.C = c.D = 0;
    c.reach = 0;
    c.max_attempts = 0;
    c.stiff_switches = c.stiff_attempts = 0;
}

/* deposit record written by the advance kernel and read by the projection gather */
struct Record {
    double e, mx, my; /* GetParticleEnergyMomentum */
    double wxc, wyc;  /* ceil-side weights; floor-side = 1 - w */
    int32_t cell;     /* packed floor offsets + class, or PH_CELL_INVALID */
};

/* ---- FetchRelations.get_initial_windsea(...; particle_state=true) ---------- */
/* cold: reseeds only — kept out of line so the advance kernel's hot loop stays small */
PM_HD_NOINLINE_DECL void windsea(double U10, double V10, double time_scale, double& lne, double& cgx, double& cgy) {
    double U_amp = sqrt(U10 * U10 + V10 * V10);
    U_amp = (U_amp < 0.1) ? 0.1 : U_amp;
    time_scale = fabs(time_scale);
    double tau = 9.81 * time_scale / fabs(U_amp);
    double X_tilde = pm_pow(tau / (22.8013 * 2.4097), 1.0 / (1.0 - 0.2748));
    double f_m = 3.5 * (9.81 / U_amp) * pm_pow(X_tilde, -0.33);
    double a_j = 0.033 * pm_pow(f_m * U_amp / 9.81, 0.67);
    double w = f_m * 2.0 * 3.141592653589793;
    double iw = 1.0 / w;
    double iw2 = iw * iw;
    double E = 0.31 * (9.81 * 9.81) * a_j * (iw2 * iw2);
    double f_peak = f_m * 9.81 / U_amp;
    double T_bar = 0.9 * (1.0 / f_peak);
    double cg_amp = 9.81 * T_bar / (4.0 * 3.141592653589793);
    cgx = cg_amp * U10 / U_amp;
    cgy = cg_amp * V10 / U_amp;
    lne = pm_log(E);
}

/* MinimalParticle(U,V,T): fetch law at unit wind speed, rand_sign() fixed to +1 */
PM_HD void minimal_particle(double U10, double V10, double T, double& lne, double& cgx, double& cgy) {
    if (U10 == 0.0) U10 = 1.0;
    if (V10 == 0.0) V10 = 1.0;
    double Uamp = sqrt(U10 * U10 + V10 * V10);
    double a = 1.0 * U10 / Uamp, b = 1.0 * V10 / Uamp;
    windsea(a, b, T, lne, cgx, cgy);
}

/* ResetParticleValues(defaults, (0,0), wind, DT) */
PM_HD void reset_particle_values(const picles_params_t& P, double wu, double wv, double DT, Particle& p) {
    if (!P.has_defaults) {
        windsea(wu, wv, DT, p.u0, p.u1, p.u2);
    } else {
        p.u0 = P.defaults[0];
        p.u1 = P.defaults[1];
        p.u2 = P.defaults[2];
    }
    p.u3 = 0.0;
    p.u4 = 0.0;
}

/* GetParticleEnergyMomentum */
PM_HD void charge(double lne, double cx, double cy, double& e, double& mx, double& my) {
    e = pm_exp(lne);
    double cs = sqrt(cx * cx + cy * cy);
    mx = cx * e / (cs * cs) / 2.0;
    my = cy * e / (cs * cs) / 2.0;
}

/* ---- arithmetic policies ----------------------------------------------------- */
/* IEEE operators (host, oracle parity, device fallback and cold paths) */
struct OpsSafe {
    static PM_HDM double div(double a, double b, unsigned*) { return a / b; }
    static PM_HDM double divz(double a, double b, unsigned*) { return a / b; }
    static PM_HDM double prep(double) { return 0.0; }
    static PM_HDM double div_pre(double a, double b, double, unsigned*) { return a / b; }
    static PM_HDM double divz_pre(double a, double b, double, unsigned*) { return a / b; }
    static PM_HDM double sqrt_(double x, unsigned*) { return sqrt(x); }
    static PM_HDM double sqrtz(double x, unsigned*) { return sqrt(x); }
    static PM_HDM double div_nc(double a, double b) { return a / b; }
    static PM_HDM double div_pre_nc(double a, double b, double) { return a / b; }
    static PM_HDM double sqrt_r(double x, unsigned*) { return sqrt(x); }
    static PM_HDM double absnn(double x) { return fabs(x); }
    static PM_HDM double tanh_(double x, unsigned*) { return pm_tanh_safe(x); }
    static PM_HDM double sech(double x, unsigned*) { return pm_sech_safe(x); }
    static PM_HDM double exp_(double x, unsigned*) { return pm_exp(x); }
    static PM_HDM double pow_(double x, double y, unsigned*) { return pm_pow_safe(x, y); }
    static PM_HDM double log_(double x, unsigned*) { return pm_log_safe(x); }
    static PM_HDM double log_pos(double x, unsigned*) { return pm_log_safe(x); }
    static PM_HDM double log10_(double x, unsigned*) { return pm_log10_safe(x); }
    /* compares: the FP64 operators */
    static PM_HDM bool above(double x, double c) { return x > c; }
    static PM_HDM bool iszero(double x) { return x == 0.0; }
    static PM_HDM double maxc(double a, double c) { return pm_maxc(a, c); }
    static PM_HDM double minc(double a, double c) { return pm_min(c, a); }
    static PM_HDM double max_mag(double a, double b) { return pm_max(a, b); }
};
#if defined(__CUDA_ARCH__)
/* device fast paths with a deferred validity flag (pmath.h) */
struct OpsFast {
    static __device__ __forceinline__ double div(double a, double b, unsigned* bad) { return pm_div_fast(a, b, bad); }
    static __device__ __forceinline__ double divz(double a, double b, unsigned* bad) { return pm_divz_fast(a, b, bad); }
    static __device__ __forceinline__ double prep(double b) { return pm_rcp_newton(b); }
    static __device__ __forceinline__ double div_pre(double a, double b, double y, unsigned* bad) { return pm_div_pre_fast(a, b, y, bad); }
    static __device__ __forceinline__ double divz_pre(double a, double b, double y, unsigned* bad) { return pm_divz_pre_fast(a, b, y, bad); }
    static __device__ __forceinline__ double sqrt_(double x, unsigned* bad) { return pm_sqrt_fast(x, bad); }
    static __device__ __forceinline__ double sqrtz(double x, unsigned* bad) { return pm_sqrtz_fast(x, bad); }
    /* unchecked divisions and the range-limited root they lean on (pmath.h); |x| of a value known to be >= +0 */
    static __device__ __forceinline__ double div_nc(double a, double b) { return pm_div_nc_fast(a, b); }
    static __device__ __forceinline__ double div_pre_nc(double a, double b, double y) { return pm_div_pre_nc_fast(a, b, y); }
    static __device__ __forceinline__ double sqrt_r(double x, unsigned* bad) { return pm_sqrt_r_fast(x, bad); }
    static __device__ __forceinline__ double absnn(double x) { return x; }
    static __device__ __forceinline__ double tanh_(double x, unsigned* bad) { return pm_tanh_fast(x, bad); }
    static __device__ __forceinline__ double sech(double x, unsigned* bad) { return pm_sech_fast(x, bad); }
    static __device__ __forceinline__ double exp_(double x, unsigned* bad) { return pm_expx_fast(x, bad); }
    static __device__ __forceinline__ double pow_(double x, double y, unsigned* bad) { return pm_pow_fast(x, y, bad); }
    static __device__ __forceinline__ double log_(double x, unsigned* bad) { return pm_log_fast(x, bad); }
    /* log of an operand that is positive and finite whenever the flag is clear: no special-case selects */
    static __device__ __forceinline__ double log_pos(double x, unsigned* bad) { return pm_log_core_fast(x, bad); }
    static __device__ __forceinline__ double log10_(double x, unsigned* bad) { return pm_log10_fast(x, bad); }
    /* compares off the FP64 pipe (pmath.h), each exact for every operand the fast path lets through unflagged:
       above(x, c) is the test of a clamp x > c ? c : x with c's low word zero, where x == c gives c either way, and
       x is never NaN unflagged; maxc / minc take an operand that is NaN only if the flag is raised; max_mag two
       magnitudes */
    static __device__ __forceinline__ bool above(double x, double c) { return pm_ge_hw(x, c); }
    static __device__ __forceinline__ bool iszero(double x) { return pm_iszero(x); }
    static __device__ __forceinline__ double maxc(double a, double c) { return pm_maxc_i(a, c); }
    static __device__ __forceinline__ double minc(double a, double c) { return pm_minc_i(a, c); }
    static __device__ __forceinline__ double max_mag(double a, double b) { return pm_max_mag(a, b); }
};
#endif

/* GetVariablesAtVertex(state, 0, 0) */
template <class O>
PM_HD void vertex_t(double e, double mx, double my, Particle& p, unsigned* bad) {
    double m_amp = O::sqrtz(mx * mx + my * my, bad);
    double den = 2.0 * (m_amp * m_amp);
    p.u0 = O::log_(e, bad);
    p.u1 = O::divz(mx * e, den, bad);
    p.u2 = O::divz(my * e, den, bad);
    p.u3 = 0.0;
    p.u4 = 0.0;
}
PM_HD_NOINLINE_DECL void vertex_cold(double e, double mx, double my, Particle& p) {
    vertex_t<OpsSafe>(e, mx, my, p, (unsigned*)0);
}
PM_HD void vertex(double e, double mx, double my, Particle& p) {
#if defined(__CUDA_ARCH__)
    unsigned bad = 0;
    vertex_t<OpsFast>(e, mx, my, p, &bad);
    if (bad) vertex_cold(e, mx, my, p);
#else
    vertex_cold(e, mx, my, p);
#endif
}

/* ---- right-hand side: components lne, c̄_x, c̄_y --------------------------- */
/* Straight-line: the term switches and guards are selects, so with O = OpsFast the whole
   evaluation is one basic block and its independent chains (tanh, sech, the two exps,
   the k_p / ω_p divisions) overlap in the FP64 pipe. */
template <class O, bool STD>
PM_HD void rhs3(const picles_params_t& P, const Hoist& H, double lne, double cx, double cy, double u, double v,
                double us, double pc, double& d0, double& d1, double& d2, unsigned* bad) {
    /* STD: the caller has checked that all four source terms are on and n == 2 (uniform over the
       launch), so the switches below fold away; same arithmetic either way */
    const bool t_input = STD || P.input, t_diss = STD || P.dissipation, t_peak = STD || P.peak_shift,
               t_dir = STD || P.direction;
    const double P_n = STD ? 2.0 : P.n;
    double r_g = P.r_g;
    /*
     * STD also says r_g, e_T in [2^-64, 2^64] and p finite (make_hoist).  Then four of the divisions below and
     * the one inside sech cannot leave the premises of the fast path and carry no validity test (pmath.h):
     *   cbar   passes sqrt_r only for cx^2+cy^2 in [2^-970, 2^576) -> cbar in [2^-485, 2^288), never NaN;
     *   c_gp   = cbar / r_g in [2^-549, 2^352): dividend >= 2^-485, quotient normal;
     *   kp     = 2.4525 / max(c_gp^2, 1e-2): divisor in [1e-2, 2^704), quotient in (2^-703, 245.25];
     *   wp     = 4.905 / max(c_gp, 0.1): divisor in [0.1, 2^352);
     *   kp/e_T : dividend in (2^-703, 245.25], quotient in (2^-767, 2^72).
     * Whenever sqrt_r raises the flag these hold garbage, and the whole evaluation is repeated with the IEEE
     * operators, as for every other flag.  cbar and c_gp are >= +0, so their fabs() is the identity.
     */
#if defined(PH_CHECK_ALL) /* profiles/: every division with its validity test, to time what leaving them out buys */
    const bool NC = false;
#else
    const bool NC = STD;
#endif
    double cbar = NC ? O::sqrt_r(cx * cx + cy * cy, bad) : O::sqrt_(cx * cx + cy * cy, bad);
    double c_gp = NC ? O::div_pre_nc(O::absnn(cbar), r_g, H.y_rg) : O::div_pre(fabs(cbar), r_g, H.y_rg, bad);
    /* g/(4m) and g/(2m) with the power of two moved into the dividend: the same real quotient,
       hence the same rounded one (neither can leave the normal range), one multiplication less each */
    double kp = NC ? O::div_nc(9.81 / 4.0, O::maxc(c_gp * c_gp, 1e-2)) : O::div(9.81 / 4.0, O::maxc(c_gp * c_gp, 1e-2), bad);
    double wp = NC ? O::div_nc(9.81 / 2.0, O::maxc(O::absnn(c_gp), 0.1)) : O::div(9.81 / 2.0, O::maxc(fabs(c_gp), 0.1), bad);
    double gx = O::divz_pre(cx, r_g, H.y_rg, bad), gy = O::divz_pre(cy, r_g, H.y_rg, bad);
    double a1 = O::div(us, 2.0 * c_gp, bad); /* α_func(us, c_gp) */
    double alpha = O::above(a1, 500.0) ? 500.0 : a1;
    double sg = O::sqrt_(gx * gx + gy * gy, bad);
    double msg = O::maxc(sg, 1e-4);
    double alpha_p = O::div(u * gx + v * gy, 2.0 * (msg * msg), bad);
    /* the fast tanh and sech do not test for NaN: alpha_p is NaN only if its division raised the flag, and with a
       finite p (STD) neither argument can be NaN otherwise */
    const double x_t = P.p * (alpha_p - 0.85);
    if (!STD && bad) *bad |= (x_t != x_t) ? 1u : 0u;
    double Hp = 0.5 * (1.0 + O::tanh_(x_t, bad));
    double sch = O::sech(10.0 * (alpha_p - 0.85), bad);
    double Dp = 1.0 - 1.25 * (sch * sch);
    double It = t_input ? P.C_e * Hp * (alpha * alpha) : 0.0;
    double Dt, Scg;
    {
        double r = NC ? O::div_pre_nc(kp, P.e_T, H.y_eT) : O::div_pre(kp, P.e_T, H.y_eT, bad), pw;
        double twon = 2.0 * P_n;
        double r2 = r * r;
        pw = (twon == 4.0) ? r2 * r2 : r2;
        if (twon != 4.0 && twon != 2.0) pw = O::pow_(r, twon, bad); /* general q: uniform, cold */
        /* n == 2 (q = -1/4): exp(n*lne) and exp(2*lne) are the same evaluation */
        double e2 = O::exp_(2.0 * lne, bad);
        double en = (P_n == 2.0) ? e2 : O::exp_(P_n * lne, bad);
        Dt = t_diss ? en * pw : 0.0;
        double k2 = kp * kp;
        Scg = t_peak ? P.C_alpha * Dp * (k2 * k2) * e2 : 0.0;
    }
    double Sdir;
    {
        double a2r = O::div(us, 2.0 * sg, bad); /* α_func(us, sg) */
        double a2 = O::above(a2r, 500.0) ? 500.0 : a2r;
        double prod = us * sg;
        bool zero = O::iszero(prod);
        double den = zero ? 1.0 : prod * prod;
        double s2 = O::div(2.0, den, bad) *
                    (u * v * (2.0 * (gy * gy) - sg * sg) - gx * gy * (2.0 * (v * v) - us * us));
        s2 = zero ? 0.0 : s2;
        Sdir = t_dir ? a2 * a2 * P.C_varphi * Hp * s2 : 0.0;
    }
    double Ssph = cx * pc;
    d0 = wp * r_g * Scg + wp * (It - Dt);
    d1 = -cx * wp * r_g * Scg + cy * Sdir + cy * Ssph;
    d2 = -cy * wp * r_g * Scg - cx * Sdir - cx * Ssph;
}

/* propagation components: [dz4, dz5] = M * [c̄_x, c̄_y] */
PM_HD void prop(const picles_params_t& P, const double* M, double cx, double cy, double& d3, double& d4) {
    if (P.propagation) {
        d3 = M[0] * cx + M[1] * cy;
        d4 = M[2] * cx + M[3] * cy;
    } else {
        d3 = 0.0;
        d4 = 0.0;
    }
}

/* wind at stage time ts: the polynomial through the staged levels (linear for the two levels
   t, t+DT).  A wind that does not change over DT gives u0, v0 and the hoisted us0 exactly; the
   time coefficients and the time base of an unsteady wind live in the scratch slots. */
template <class KS>
PM_HD void stage_uv(double wu0, double wv0, const Hoist& H, const KS& K, double ts, double& u, double& v) {
    double sg = (ts - K.ld(KS_WT0)) * K.ld(KS_WIDT);
    int m = H.nseg - 1;
    double pu = K.ld(KS_WCU + m), pv = K.ld(KS_WCV + m);
    /* two levels (the default): the loop does not run; more levels are rare enough to stay rolled */
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (; m >= 1; m--) {
        double a = sg - (double)m;
        pu = fma(pu, a, K.ld(KS_WCU + m - 1));
        pv = fma(pv, a, K.ld(KS_WCV + m - 1));
    }
    u = fma(pu, sg, wu0);
    v = fma(pv, sg, wv0);
}
template <class O, class KS>
PM_HD void stage_wind(double wu0, double wv0, const Hoist& H, const KS& K, double ts, double& u, double& v, double& us,
                      unsigned* bad) {
    if (H.steady) {
        u = wu0; v = wv0; us = H.us0;
    } else {
        stage_uv(wu0, wv0, H, K, ts, u, v);
        us = O::sqrtz(u * u + v * v, bad);
    }
}

/* IEEE right-hand side, one shared out-of-line copy: the fallback of the fast path (and the
   only path on the host).  Everything by value: nothing of the caller is forced into local
   memory. */
struct D3 { double d0, d1, d2; };
PM_HD_NOINLINE_DECL D3 f3_cold(const picles_params_t* Pp, double u, double v, double pc, double lne, double cx,
                               double cy) {
    Hoist H;
    H.y_rg = 0.0; H.y_eT = 0.0; H.us0 = 0.0; H.steady = false; H.steady_warp = false; H.std_terms = false; H.nseg = 1;
    double us = sqrt(u * u + v * v);
    D3 r;
    rhs3<OpsSafe, false>(*Pp, H, lne, cx, cy, u, v, us, pc, r.d0, r.d1, r.d2, (unsigned*)0);
    return r;
}

/* loop invariants of the hot right-hand side */
PM_HD void make_hoist(const picles_params_t& P, double wu0, double wv0, bool steady, int nseg, Hoist& H) {
#if defined(__CUDA_ARCH__)
    H.y_rg = pm_rcp_newton(P.r_g);
    H.y_eT = pm_rcp_newton(P.e_T);
#else
    (void)P;
    H.y_rg = 0.0; H.y_eT = 0.0;
#endif
    H.steady = steady;
#if defined(__CUDA_ARCH__)
    /* one vote per particle and model step, here, instead of one per right-hand side: the lanes that reach a
       right-hand side later are a subset of the lanes voting now (lanes only ever leave the integration loop), so
       "all steady" now implies "all steady" there; a warp that says no takes the copy that reads the wind per lane */
    H.steady_warp = __all_sync(__activemask(), steady);
#else
    H.steady_warp = steady;
#endif
    /* ... and parameters in the range the unchecked divisions of the switch-free copy assume (rhs3) */
    const bool sane = (P.r_g >= 0x1p-64) && (P.r_g <= 0x1p64) && (P.e_T >= 0x1p-64) && (P.e_T <= 0x1p64) && (fabs(P.p) <= 0x1p64);
    H.std_terms = P.input && P.dissipation && P.peak_shift && P.direction && (P.n == 2.0) && sane;
    H.nseg = nseg;
    H.us0 = sqrt(wu0 * wu0 + wv0 * wv0);
   
}

/* hot right-hand side of the stage loop */
template <class KS>
PM_HD void f3(const picles_params_t& P, double wu0, double wv0, const Hoist& H, const KS& K, double pc, double lne, double cx,
              double cy, double ts, double& d0, double& d1, double& d2) {
#if defined(__CUDA_ARCH__)
    double u, v, us;
    unsigned bad = 0;
    /* a wind that does not change over DT (the homogeneous-box configurations): its own copy of the
       right-hand side, fed from the hoisted values directly — no wind branch at its head.  Taken
       only when every lane of the warp that is here is steady (a vote, so the choice never splits
       a warp; a lane that votes yes is steady itself): a field that is constant up to rounding noise (a
       constant wind mesh sampled at the nodes) mixes steady and unsteady lanes, and a split warp
       would run both copies */
#if defined(PH_VOTE_PER_RHS) /* profiles/: the vote at the head of every right-hand side, as before */
    if (H.std_terms && __all_sync(__activemask(), H.steady)) {
#else
    if (H.std_terms && H.steady_warp) {
#endif
        u = wu0; v = wv0;
        rhs3<OpsFast, true>(P, H, lne, cx, cy, wu0, wv0, H.us0, pc, d0, d1, d2, &bad);
    } else {
        stage_wind<OpsFast>(wu0, wv0, H, K, ts, u, v, us, &bad);
        if (H.std_terms) rhs3<OpsFast, true>(P, H, lne, cx, cy, u, v, us, pc, d0, d1, d2, &bad);
        else rhs3<OpsFast, false>(P, H, lne, cx, cy, u, v, us, pc, d0, d1, d2, &bad);
    }
    if (bad) { /* rare: denormal/huge/non-finite operands */
        D3 r = f3_cold(&P, u, v, pc, lne, cx, cy);
        d0 = r.d0; d1 = r.d1; d2 = r.d2;
    }
#else
    double u = wu0, v = wv0;
    if (!H.steady) stage_uv(wu0, wv0, H, K, ts, u, v);
#if !defined(__CUDACC__) /* tests/: the host build takes the switch-free copy where the kernels do */
    if (ph_host_specialised && H.std_terms) {
        rhs3<OpsSafe, true>(P, H, lne, cx, cy, u, v, sqrt(u * u + v * v), pc, d0, d1, d2, (unsigned*)0);
        return;
    }
#endif
    D3 r = f3_cold(&P, u, v, pc, lne, cx, cy);
    d0 = r.d0; d1 = r.d1; d2 = r.d2;
#endif
}

template <class O>
PM_HD double rms5(double a, double b, double c, double d, double e, unsigned* bad) {
    double s = 0.0;
    s += a * a;
    s += b * b;
    s += c * c;
    s += d * d;
    s += e * e;
    return O::sqrtz(O::divz(s, 5.0, bad), bad);
}

/* ---- ode_determine_initdt (Hairer), split around its one right-hand side ---------- */
/* part A: from u and f0 = f(u,t) to either a final dt (returns true) or the trial step
   dt0 of the second evaluation f1 = f(u + dt0*f0, t + dt0) (returns false) */
template <class O>
PM_HD bool initdt_a(const picles_params_t& P, double u0, double u1, double u2, double u3, double u4, double k0,
                    double k1, double k2, double k3, double k4, double& dt_out, double& dt0_out, double& d1_out,
                    unsigned* bad) {
    double dtmin = pm_nextfloat_pos(P.dtmin);
    const double smalldt = 1e-6;
    double s0 = fma(fabs(u0), P.reltol, P.abstol);
    double s1 = fma(fabs(u1), P.reltol, P.abstol);
    double s2 = fma(fabs(u2), P.reltol, P.abstol);
    double s3 = fma(fabs(u3), P.reltol, P.abstol);
    double s4 = fma(fabs(u4), P.reltol, P.abstol);
    double d0 = rms5<O>(O::divz(u0, s0, bad), O::divz(u1, s1, bad), O::divz(u2, s2, bad), O::divz(u3, s3, bad),
                        O::divz(u4, s4, bad), bad);
    double d1 = rms5<O>(O::divz(k0, s0, bad), O::divz(k1, s1, bad), O::divz(k2, s2, bad), O::divz(k3, s3, bad),
                        O::divz(k4, s4, bad), bad);
    bool tiny = (d0 < 1e-5) | (d1 < 1e-5);
    double dt0 = tiny ? smalldt : O::div(O::div(d0, tiny ? 1.0 : d1, bad), 100.0, bad);
    dt0 = pm_min(dt0, P.dtmax);
    d1_out = d1;
    dt0_out = dt0;
    if (d1 != d1) { dt_out = dtmin; return true; }
    if (dt0 < 10.0 * 2.220446049250313e-16) { dt_out = pm_max(smalldt, dtmin); return true; }
    return false;
}
/* part B: with f1 in hand */
template <class O>
PM_HD double initdt_b(const picles_params_t& P, double u0, double u1, double u2, double u3, double u4, double k0,
                      double k1, double k2, double k3, double k4, double f0, double f1, double f2, double f3x,
                      double f4x, double dt0, double d1, double order, unsigned* bad) {
    double dtmin = pm_nextfloat_pos(P.dtmin);
    bool same = (k0 == f0) & (k1 == f1) & (k2 == f2) & (k3 == f3x) & (k4 == f4x);
    double s0 = fma(fabs(u0), P.reltol, P.abstol);
    double s1 = fma(fabs(u1), P.reltol, P.abstol);
    double s2 = fma(fabs(u2), P.reltol, P.abstol);
    double s3 = fma(fabs(u3), P.reltol, P.abstol);
    double s4 = fma(fabs(u4), P.reltol, P.abstol);
    double d2 = O::div(rms5<O>(O::divz(f0 - k0, s0, bad), O::divz(f1 - k1, s1, bad), O::divz(f2 - k2, s2, bad),
                               O::divz(f3x - k3, s3, bad), O::divz(f4x - k4, s4, bad), bad),
                       dt0, bad);
    double mx = pm_max(d1, d2);
    bool flat = (mx <= 1e-15);
    double lg = O::log10_(flat ? 1.0 : mx, bad);
    double dt1 = flat ? pm_max(1e-6, dt0 * 1e-3) : pm_exp10(O::div(-(2.0 + lg), order, bad)); /* get_current_alg_order: 5, or 2 under Rosenbrock23 */
    double dt = pm_max(dtmin, pm_min(pm_min(100.0 * dt0, dt1), P.dtmax));
    return same ? pm_max(dtmin, 100.0 * dt0) : dt;
}
/* IEEE fallbacks, out of line */
PM_HD_NOINLINE_DECL bool initdt_a_cold(const picles_params_t& P, double u0, double u1, double u2, double u3, double u4,
                                       double k0, double k1, double k2, double k3, double k4, double& dt_out,
                                       double& dt0_out, double& d1_out) {
    return initdt_a<OpsSafe>(P, u0, u1, u2, u3, u4, k0, k1, k2, k3, k4, dt_out, dt0_out, d1_out, (unsigned*)0);
}
PM_HD_NOINLINE_DECL double initdt_b_cold(const picles_params_t& P, double u0, double u1, double u2, double u3,
                                         double u4, double k0, double k1, double k2, double k3, double k4, double f0,
                                         double f1, double f2, double f3x, double f4x, double dt0, double d1, double order) {
    return initdt_b<OpsSafe>(P, u0, u1, u2, u3, u4, k0, k1, k2, k3, k4, f0, f1, f2, f3x, f4x, dt0, d1, order, (unsigned*)0);
}

/* ---- error estimate + PI controller of one attempt -------------------------------- */
/* utilde = dt*sum(btilde_j k_j); calculate_residuals; RMS norm; stepsize_controller!:
   q = EEst^beta1 / qold^beta2 evaluated as exp(beta1*log(EEst) - beta2*log(qold)) (the
   reference's OrdinaryDiffEq uses an approximate fastpow here; see DESIGN.md).  lq is
   log(qold), carried between attempts; t1 = beta1*log(EEst) feeds the reject branch. */
struct StepCtl {
    double EEst, q, t1, lE;
};
template <class O>
PM_HD void step_control(const picles_params_t& P, const Tableau& T, double dt, double e0, double e1, double e2,
                        double xe, double ye, double u0, double u1, double u2, double u3, double u4, double n0,
                        double n1, double n2, double n3, double n4, double lq, StepCtl& sc, unsigned* bad) {
    const double qmin = 0.2, qmax = 10.0, gamma = 0.9;
    double r0 = O::divz(dt * e0, fma(O::max_mag(fabs(u0), fabs(n0)), P.reltol, P.abstol), bad);
    double r1 = O::divz(dt * e1, fma(O::max_mag(fabs(u1), fabs(n1)), P.reltol, P.abstol), bad);
    double r2 = O::divz(dt * e2, fma(O::max_mag(fabs(u2), fabs(n2)), P.reltol, P.abstol), bad);
    double r3 = O::divz(dt * xe, fma(O::max_mag(fabs(u3), fabs(n3)), P.reltol, P.abstol), bad);
    double r4 = O::divz(dt * ye, fma(O::max_mag(fabs(u4), fabs(n4)), P.reltol, P.abstol), bad);
    double EEst = rms5<O>(r0, r1, r2, r3, r4, bad);
    bool zero = O::iszero(EEst);
    /* EEst = sqrtz(...): with the flag clear it is +0 (replaced by 1) or a positive normal number, so the fast log
       needs none of its special cases; the exponent below is flagged outside [-700, 700] by the fast exp, whose
       in-range value is pm_exp's (pmath.h) */
    double lE = O::log_pos(zero ? 1.0 : EEst, bad);
    double t1 = T.beta1 * lE;
    double q = O::exp_(t1 - T.beta2 * lq, bad);
    q = O::maxc(O::minc(O::div(q, gamma, bad), 1.0 / qmin), 1.0 / qmax);
    sc.EEst = EEst;
    sc.q = zero ? 1.0 / qmax : q;
    sc.t1 = t1;
    sc.lE = lE;
}
PM_HD_NOINLINE_DECL void step_control_cold(const picles_params_t& P, const Tableau& T, double dt, double e0, double e1,
                                           double e2, double xe, double ye, double u0, double u1, double u2, double u3,
                                           double u4, double n0, double n1, double n2, double n3, double n4, double lq,
                                           StepCtl& sc) {
    step_control<OpsSafe>(P, T, dt, e0, e1, e2, xe, ye, u0, u1, u2, u3, u4, n0, n1, n2, n3, n4, lq, sc, (unsigned*)0);
}

/* time coefficients of the staged wind -> scratch slots (two levels: c1 = the increment), and the
   loop invariants of the right-hand side; once per particle and model step */
template <class KS>
PM_HD void wind_to_slots(const picles_params_t& P, const Wind& w, KS& K, Hoist& H) {
    double cu[PH_WIND_SEG_MAX + 1], cv[PH_WIND_SEG_MAX + 1];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int m = 0; m <= PH_WIND_SEG_MAX; m++) { cu[m] = w.ul[m]; cv[m] = w.vl[m]; }
    wind_newton(cu, w.nseg);
    wind_newton(cv, w.nseg);
    bool steady = true;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int m = 1; m <= PH_WIND_SEG_MAX; m++) {
        if (m <= w.nseg) {
            K.st(KS_WCU + m - 1, cu[m]); K.st(KS_WCV + m - 1, cv[m]);
            steady = steady && (cu[m] == 0.0) && (cv[m] == 0.0);
        }
    }
    make_hoist(P, w.ul[0], w.vl[0], steady, w.nseg, H);
    K.st(KS_WT0, w.t_start); K.st(KS_WIDT, (double)w.nseg * w.inv_DT);
}

/* Tsit5 inside a composite algorithm: eigen_est = max_i |k7_i - k6_i| / |g7_i - g6_i| (Hairer II,
   p. 22).  g7 = u_new (n); g6 = the argument of stage 6: its first three components were saved
   when the stage was set up, the propagation part comes from the running sums x6, y6.
   num[i] = k7_i - k6_i, den[i] = g7_i - g6_i.  Once per attempt, AutoTsit5 only. */
template <class KS>
PM_HD void stiffness_terms(const picles_params_t& P, const double* M, const KS& K, double dt, double x6, double y6, double u3,
                           double u4, double n0, double n1, double n2, double n3, double n4, double* num, double* den) {
    const double g60 = K.ld(KS_G60), g61 = K.ld(KS_G61), g62 = K.ld(KS_DT0); /* saved when stage 6 was set up */
    const double g63 = fma(dt, x6, u3), g64 = fma(dt, y6, u4);
    double k6x, k6y, k7x, k7y;
    prop(P, M, g61, g62, k6x, k6y);
    prop(P, M, n1, n2, k7x, k7y);
    num[0] = K.get(7, 0) - K.get(6, 0); den[0] = n0 - g60;
    num[1] = K.get(7, 1) - K.get(6, 1); den[1] = n1 - g61;
    num[2] = K.get(7, 2) - K.get(6, 2); den[2] = n2 - g62;
    num[3] = k7x - k6x; den[3] = n3 - g63;
    num[4] = k7y - k6y; den[4] = n4 - g64;
}
/* the AutoSwitch test as OrdinaryDiffEq evaluates it: |eigen_est * dt / stability_size| > nonstifftol
   with eigen_est = max_i |num_i / den_i| (IEEE divisions), dt the step the controller proposes */
PM_HD_NOINLINE_DECL bool stiffness_test_exact(double a0, double a1, double a2, double a3, double a4, double b0, double b1,
                                              double b2, double b3, double b4, double dt_next) {
    double eig = 0.0;
    eig = pm_max(eig, fabs(a0 / b0));
    eig = pm_max(eig, fabs(a1 / b1));
    eig = pm_max(eig, fabs(a2 / b2));
    eig = pm_max(eig, fabs(a3 / b3));
    eig = pm_max(eig, fabs(a4 / b4));
    return fabs(eig * dt_next / 3.5068) > 0.9;
}
/*
 * The same decision without a division.  With c = 0.9 * 3.5068 and p_i = |num_i| * dt, d_i = |den_i|:
 *   p_i <  c (1 - 1e-13) d_i  for every i  =>  every rounded |num_i/den_i| * dt / 3.5068 ends below 0.9
 *                                              (three roundings of 1.1e-16 each): not stiff;
 *   p_i >  c (1 + 1e-13) d_i  for some i, every other component decided one way or the other
 *                                          =>  that quotient alone carries the maximum above 0.9: stiff.
 * A quotient 0/0 (a component that did not move in the attempt) is NaN, which makes eigen_est NaN
 * and the test false whatever the other components are; x/0 is Inf and makes it true unless a NaN
 * is about: decided as well (both occur in the first, rounding-noise-sized attempts after a reset).  A component is undecided
 * inside the 1e-13 band, when d_i is so small (< 1e-200) that p_i could underflow out of the
 * argument, and whenever a comparison involves NaN or Inf/Inf.  Only
 * undecided attempts take the exact test, out of line: in practice none, so no warp diverges into
 * it.  Bit-identical decisions (tests/test_autotsit5.py compares every attempt's outcome through
 * the switch counts and the State).
 */
PM_HD bool stiffness_test(const double* num, const double* den, double dt_next) {
    const double c_lo = 3.15612 * (1.0 - 1e-13), c_hi = 3.15612 * (1.0 + 1e-13);
    /* level 1 (all most attempts need): every component clearly below the threshold */
    bool all_clear = true;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int i = 0; i < 5; i++) {
        const double di = fabs(den[i]);
        all_clear = all_clear & (di > 1e-200) & (fabs(num[i]) * dt_next < c_lo * di);
    }
    if (all_clear) return false;
    /* level 2: the stiff side and the degenerate quotients */
    bool all_decided = true, any_stiff = false, any_nan = false;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int i = 0; i < 5; i++) {
        const double pi = fabs(num[i]) * dt_next, di = fabs(den[i]);
        const bool ok = di > 1e-200;             /* false for NaN too */
        const bool clear = ok & (pi < c_lo * di);
        const bool stiff = ok & (pi > c_hi * di);
        const bool zz = (num[i] == 0.0) & (den[i] == 0.0); /* 0/0 */
        /* x/0, x finite and non-zero: the quotient is Inf, and Inf * dt / 3.5068 > 0.9 for dt > 0 */
        const bool xz = (den[i] == 0.0) & (fabs(num[i]) > 0.0) & (fabs(num[i]) < 1.7976931348623157e308) & (dt_next > 0.0);
        all_decided = all_decided & (clear | stiff | zz | xz);
        any_stiff = any_stiff | stiff | xz;
        any_nan = any_nan | zz;
    }
    if (all_decided) return any_stiff & !any_nan;
    return stiffness_test_exact(num[0], num[1], num[2], num[3], num[4], den[0], den[1], den[2], den[3], den[4], dt_next);
}

/* ---- step!(integrator, DT, true): advance particle p from p.t to p.t + DT ------------ */
/*
 * Every right-hand side of the integration — the FSAL reset k1 = f(u,t), the second
 * evaluation of the initial-step heuristic, and the six new stages of each attempt —
 * goes through ONE inlined call site, driven by a small phase machine, so the kernel's
 * instruction footprint stays inside the SM's instruction cache:
 *   ph = 1  k1 = f(u, t)                       (then initdt part A when a reset is pending)
 *   ph = 0  f1 = f(u + dt0*k1, t + dt0)         (then initdt part B)
 *   ph = 2..7 stage ph of the current attempt   (after 7: error estimate, controller,
 *                                               accept/reject, header of the next attempt)
 * Stage derivatives of (lne, c̄_x, c̄_y) live in K; the propagation derivatives
 * k_j[3:4] = M*c̄_j are folded into the running sums of stage 7 (x7,y7) and of the error
 * estimate (xe,ye) as each k_j appears — the same fma chain as storing them.
 */
/*
 * AutoTsit5 (P.solver == PICLES_SOLVER_AUTOTSIT5, AUTOSW instantiation): every attempt also leaves
 * OrdinaryDiffEq's stiffness estimate and the AutoSwitch run length (kept in a scratch slot) is
 * updated with |eigen_est * dt / 3.5068| > 9/10; more than ten stiff attempts in a row hand the
 * particle to Rosenbrock23 (stiff.h, out of line): the loop is left with dt doubled and `true` is
 * returned.  A particle whose current algorithm is Rosenbrock23 at the start of a step never
 * enters here (advance_particle).  tstop = p.t + DT of the first entry; attempts accumulates over
 * re-entries.
 */
#define PH_AUTOSW_ROLLED AUTOSW /* unrolled there too: 17.58 -> 17.77 ms (profiles/README.md) */
template <bool AUTOSW, int TSIT5 = 0, class KS>
PM_HD bool integrate(const picles_params_t& P, const double wu0, const double wv0, const Hoist& H, const double* M, double pc,
                     double tstop_in, Particle& p, Tally& c, KS& K, int& as_count, int& attempts_io) {
    if (p.status & (PICLES_PST_MAXITERS | PICLES_PST_DTMIN | PICLES_PST_UNSTABLE)) return false;
    /* compile-time switch: the kernels are instantiated with and without the monitor, so the
       Tsit5 / DP5 loop carries none of it */
#if defined(__CUDA_ARCH__)
    const bool autosw = AUTOSW; /* the monitor-carrying kernels are launched for PICLES_SOLVER_AUTOTSIT5 only */
#else
    const bool autosw = AUTOSW && (P.solver == PICLES_SOLVER_AUTOTSIT5);
#endif
    bool switched = false;
    double x6r = 0.0, y6r = 0.0; /* AutoTsit5: running sums of a6j*k_j[3:4], parked in K before the monitor reads them */
    /* TSIT5: the kernel was launched for a solver whose tableau is Tsit5's (uniform over the launch),
       which has no zero coefficient: the skip tests below fold away and the coefficient addresses
       are compile-time.  Same arithmetic either way. */
#if defined(__CUDA_ARCH__)
    const bool nz = AUTOSW || TSIT5 == 1; /* the monitor-carrying kernels run the Tsit5 tableau too */
#else
    const bool nz = TSIT5 == 1; /* the host build serves every solver from one AUTOSW instantiation; TSIT5 only when asked (tests) */
#endif
    /* TSIT5 == 2: DP5's tableau at compile time; its two zero coefficients,
       a[7][2] and bt[2], are tested where they are and nowhere else */
    const bool dz = !nz && TSIT5 == 2;
    const Tableau& T = nz ? tableau(PICLES_SOLVER_TSIT5) : (dz ? tableau(PICLES_SOLVER_DP5) : tableau(P.solver));
#define PH_COEF_ON(c, can_be_zero) (nz || (dz && !(can_be_zero)) || (c) != 0.0)
    /* prop() in the attempt loop: the Tsit5 / DP5 instantiations are launched with propagation on only
       (ph_advance_variant), so they carry no test per stage; the
       monitor-carrying kernels have a second instantiation for it, TSIT5 == 3 */
#define PH_PROP(cx_, cy_, ox_, oy_)                                                              \
    do {                                                                                         \
        if ((!AUTOSW && TSIT5 != 0) || (AUTOSW && TSIT5 == 3)) { ox_ = M[0] * (cx_) + M[1] * (cy_); oy_ = M[2] * (cx_) + M[3] * (cy_); } \
        else prop(P, M, (cx_), (cy_), ox_, oy_);                                                 \
    } while (0)
    double t = p.t;
    K.st(KS_TSTOP, tstop_in);
    double u0 = p.u0, u1 = p.u1, u2 = p.u2;
    K.st(KS_U3, p.u3); K.st(KS_U4, p.u4);
    double dt = p.dt;
    K.st(KS_QOLD, p.qold);
    K.st(KS_LQ, pm_log(p.qold));
    const double LQ0 = PH_LOG_QOLDINIT; /* pm_log(1e-4), pinned by tests/test_pmath.py */
    int32_t iter = p.iter;
    int32_t nrhs = 0, attempts = attempts_io;
    const double qmin = 0.2, gamma = 0.9;
    const double order = 5.0; /* get_current_alg_order of Tsit5 / DP5 */
    if (autosw) K.st(KS_AS, (double)as_count);
    bool need_reset = (p.flags & PICLES_PF_DT_RESET) != 0;
    p.flags &= (uint8_t)~PICLES_PF_DT_RESET;

    int ph = 1;
    double n0 = u0, n1 = u1, n2 = u2, ts = t; /* argument of the next right-hand side */
    /* running sums of the propagation components of stage 7 and of the error estimate: registers (in scratch
       slots: +1.7 % time, profiles/README.md) */
    double x7s = 0.0, y7s = 0.0, xes = 0.0, yes = 0.0;
    K.st(KS_DT0, 0.0); K.st(KS_D1N, 0.0);
    K.st(KS_DTMIN, pm_max(pm_eps(t), P.dtmin)); /* max(eps(t), dtmin): kept current on every accepted step */
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (;;) {
        double d0, d1, d2;
        f3(P, wu0, wv0, H, K, pc, n0, n1, n2, ts, d0, d1, d2);
        nrhs++;
        if (ph >= 2) {
            K.set(ph, 0, d0); K.set(ph, 1, d1); K.set(ph, 2, d2);
            double kx, ky;
            PH_PROP(n1, n2, kx, ky);
            if (ph < 7) {
                double a7 = T.a[7][ph];
                if (PH_COEF_ON(a7, ph == 2)) { x7s = fma(a7, kx, x7s); y7s = fma(a7, ky, y7s); }
            }
            double bs = T.bt[ph];
            if (PH_COEF_ON(bs, ph == 2)) { xes = fma(bs, kx, xes); yes = fma(bs, ky, yes); }
            if (autosw && ph < 6) {
                double a6 = T.a[6][ph];
                if (PH_COEF_ON(a6, false)) { x6r = fma(a6, kx, x6r); y6r = fma(a6, ky, y6r); }
            }
            if (ph < 7) {
                /* argument of stage s = ph+1 >= 3 */
                int s = ++ph;
                double a1 = T.a[s][1];
                double i0 = a1 * K.get(1, 0), i1 = a1 * K.get(1, 1), i2 = a1 * K.get(1, 2);
                if (PH_AUTOSW_ROLLED) {
                    /* the monitor-carrying loop sits at the edge of the instruction cache (profiles/README.md):
                       the same sums, rolled */
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
                    for (int j = 2; j < s; j++) {
                        double aj = T.a[s][j];
                        if (PH_COEF_ON(aj, s == 7 && j == 2)) {
                            i0 = fma(aj, K.get(j, 0), i0); i1 = fma(aj, K.get(j, 1), i1); i2 = fma(aj, K.get(j, 2), i2);
                        }
                    }
                } else {
                    for (int j = 2; j < s; j++) {
                        double aj = T.a[s][j];
                        if (PH_COEF_ON(aj, s == 7 && j == 2)) {
                            i0 = fma(aj, K.get(j, 0), i0); i1 = fma(aj, K.get(j, 1), i1); i2 = fma(aj, K.get(j, 2), i2);
                        }
                    }
                }
                n0 = fma(dt, i0, u0); n1 = fma(dt, i1, u1); n2 = fma(dt, i2, u2);
                /* c_6 = c_7 = 1 in both tableaus, and fma(1, dt, t) is t + dt: no select needed for the last two stages */
                ts = fma(T.c[s - 1], dt, t);
                if (autosw && s == 6) { K.st(KS_G60, n0); K.st(KS_G61, n1); K.st(KS_DT0, n2); } /* g6 of the monitor */
                continue;
            }
            /* all seven stages done: (n0,n1,n2) is u_new */
            const double u3 = K.ld(KS_U3), u4 = K.ld(KS_U4);
            double n3 = fma(dt, x7s, u3), n4 = fma(dt, y7s, u4);
            double b1 = T.bt[1];
            double e0 = b1 * K.get(1, 0), e1 = b1 * K.get(1, 1), e2 = b1 * K.get(1, 2);
            if (PH_AUTOSW_ROLLED) {
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
                for (int j = 2; j <= 7; j++) {
                    double bj = T.bt[j];
                    if (PH_COEF_ON(bj, j == 2)) { e0 = fma(bj, K.get(j, 0), e0); e1 = fma(bj, K.get(j, 1), e1); e2 = fma(bj, K.get(j, 2), e2); }
                }
            } else {
                for (int j = 2; j <= 7; j++) {
                    double bj = T.bt[j];
                    if (PH_COEF_ON(bj, j == 2)) { e0 = fma(bj, K.get(j, 0), e0); e1 = fma(bj, K.get(j, 1), e1); e2 = fma(bj, K.get(j, 2), e2); }
                }
            }
            StepCtl sc;
            const double xe = xes, ye = yes, lq = K.ld(KS_LQ);
#if defined(__CUDA_ARCH__)
            unsigned bad = 0;
            step_control<OpsFast>(P, T, dt, e0, e1, e2, xe, ye, u0, u1, u2, u3, u4, n0, n1, n2, n3, n4, lq, sc, &bad);
            if (bad) step_control_cold(P, T, dt, e0, e1, e2, xe, ye, u0, u1, u2, u3, u4, n0, n1, n2, n3, n4, lq, sc);
#else
            step_control_cold(P, T, dt, e0, e1, e2, xe, ye, u0, u1, u2, u3, u4, n0, n1, n2, n3, n4, lq, sc);
#endif
            double EEst = sc.EEst;
            /* EEst is a root of a sum of squares: +0 or above, or NaN.  For such operands (and the magnitude |dt|
               against a positive bound) the compares below are integer compares of the bit patterns (pmath.h) */
            const bool accept = pm_le_u(EEst, 1.0) || (P.force_dtmin && pm_le_u(fabs(dt), K.ld(KS_DTMIN)));
            /* the step size the controller proposes (and, accepted, the new time) first: the
               AutoSwitch test below needs it while the state of the attempt is still intact */
            double dt_next, t_next = t, dtmin_next = 0.0;
            if (accept) {
                /* step_accept_controller!, fixed_t_for_floatingpoint_error!, calc_dt_propose! */
                double dtnew = dt / sc.q;
                double ttmp = t + dt;
                const double tstop = K.ld(KS_TSTOP);
                t_next = pm_lt_u(fabs(ttmp - tstop), 100.0 * pm_eps(tstop)) ? tstop : ttmp; /* bound > 0: tstop finite */
                double dtp = pm_min(P.dtmax, dtnew);
                dtmin_next = pm_max(pm_eps(t_next), P.dtmin);
                dt_next = pm_max(dtp, dtmin_next);
            } else {
                /* step_reject_controller!: dt /= min(1/qmin, q11/gamma), q11 = EEst^beta1 */
                double q11 = pm_iszero(EEst) ? 1.0 : pm_exp(sc.t1);
#if defined(__CUDA_ARCH__)
                /* the specialised copies (TSIT5 != 0) are launched only with the switch off (ph_advance_variant): their
                   code is what it was before the switch existed */
                dt_next = dt / pm_reject_factor(TSIT5 == 0 ? P.nan_eest_rejects : 0, q11, qmin, gamma);
#else
                dt_next = dt / pm_reject_factor(P.nan_eest_rejects, q11, qmin, gamma);
#endif
            }
            bool is_stiff = false;
            if (autosw) {
                double num[5], den[5];
                stiffness_terms(P, M, K, dt, x6r, y6r, u3, u4, n0, n1, n2, n3, n4, num, den);
                is_stiff = stiffness_test(num, den, dt_next);
            }
            if (accept) {
                bool big = !pm_le_u(EEst, PH_QOLDINIT); /* EEst > qoldinit or NaN */
                K.st(KS_QOLD, big ? EEst : PH_QOLDINIT); /* max(EEst, qoldinit) */
                K.st(KS_LQ, big ? sc.lE : LQ0);
                t = t_next;
                K.st(KS_DTMIN, dtmin_next); /* the loopheader! of the next attempt reads it */
                u0 = n0; u1 = n1; u2 = n2;
                K.st(KS_U3, n3); K.st(KS_U4, n4);
                K.set(1, 0, K.get(7, 0)); K.set(1, 1, K.get(7, 1)); K.set(1, 2, K.get(7, 2)); /* FSAL */
                c.substeps++;
            } else {
                c.rejects++;
            }
            dt = dt_next;
            if (accept && ((u0 != u0) | (u1 != u1) | (u2 != u2) | (n3 != n3) | (n4 != n4))) {
                p.status |= PICLES_PST_UNSTABLE; c.failed++; break;
            }
            if (autosw) {
                /* AutoSwitch: maxstiffstep 10, nonstifftol 9//10, dtfac 2, stability_size(Tsit5) 3.5068 */
                int cnt = (int)K.ld(KS_AS);
                cnt = is_stiff ? ((cnt < 0) ? 1 : cnt + 1) : ((cnt > 0) ? -1 : cnt - 1);
                cnt = (cnt > PH_AS_CLAMP) ? PH_AS_CLAMP : ((cnt < -PH_AS_CLAMP) ? -PH_AS_CLAMP : cnt);
                K.st(KS_AS, (double)cnt);
                if (cnt > 10) {
                    dt = dt * 2.0;
                    c.stiff_switches++;
                    switched = true;
                    break;
                }
            }
        } else if (ph == 1) {
            K.set(1, 0, d0); K.set(1, 1, d1); K.set(1, 2, d2);
            if (need_reset) {
                need_reset = false;
                double k3, k4, dtr, dt0, d1n;
                prop(P, M, u1, u2, k3, k4);
                const double u3 = K.ld(KS_U3), u4 = K.ld(KS_U4);
                bool final_;
#if defined(__CUDA_ARCH__)
                unsigned bad = 0;
                final_ = initdt_a<OpsFast>(P, u0, u1, u2, u3, u4, d0, d1, d2, k3, k4, dtr, dt0, d1n, &bad);
                if (bad) final_ = initdt_a_cold(P, u0, u1, u2, u3, u4, d0, d1, d2, k3, k4, dtr, dt0, d1n);
#else
                final_ = initdt_a_cold(P, u0, u1, u2, u3, u4, d0, d1, d2, k3, k4, dtr, dt0, d1n);
#endif
                K.st(KS_DT0, dt0); K.st(KS_D1N, d1n);
                if (final_) {
                    dt = dtr;
                } else {
                    n0 = fma(dt0, d0, u0); n1 = fma(dt0, d1, u1); n2 = fma(dt0, d2, u2);
                    ts = t + dt0;
                    ph = 0;
                    continue;
                }
            }
        } else { /* ph == 0: (d0,d1,d2) = f1 of the initial-step heuristic */
            double k3, k4, f3x, f4x;
            prop(P, M, u1, u2, k3, k4);
            prop(P, M, n1, n2, f3x, f4x);
            double k0 = K.get(1, 0), k1 = K.get(1, 1), k2 = K.get(1, 2);
            const double u3 = K.ld(KS_U3), u4 = K.ld(KS_U4), dt0 = K.ld(KS_DT0), d1n = K.ld(KS_D1N);
#if defined(__CUDA_ARCH__)
            unsigned bad = 0;
            dt = initdt_b<OpsFast>(P, u0, u1, u2, u3, u4, k0, k1, k2, k3, k4, d0, d1, d2, f3x, f4x, dt0, d1n, order, &bad);
            if (bad) dt = initdt_b_cold(P, u0, u1, u2, u3, u4, k0, k1, k2, k3, k4, d0, d1, d2, f3x, f4x, dt0, d1n, order);
#else
            dt = initdt_b_cold(P, u0, u1, u2, u3, u4, k0, k1, k2, k3, k4, d0, d1, d2, f3x, f4x, dt0, d1n, order);
#endif
        }
        /* ---- header of the next attempt: loopheader!, check_error! ---- */
        const double tstop = K.ld(KS_TSTOP);
        if (!(t < tstop)) break;
        iter++;
        const double dtmin_t = K.ld(KS_DTMIN); /* = max(eps(t), dtmin) */
        dt = pm_min(P.dtmax, dt);
        dt = pm_max(dt, dtmin_t);
        dt = pm_min(dt, tstop - t);
        if (dt != dt) { p.status |= PICLES_PST_UNSTABLE; c.failed++; break; }
        if ((int64_t)iter > P.maxiters) { p.status |= PICLES_PST_MAXITERS; c.failed++; break; }
        if (!P.force_dtmin && dt <= P.dtmin && (t + dt < tstop)) { p.status |= PICLES_PST_DTMIN; c.failed++; break; }
        attempts++;
        {
            double kx, ky;
            PH_PROP(u1, u2, kx, ky);
            x7s = T.a[7][1] * kx; y7s = T.a[7][1] * ky;
            xes = T.bt[1] * kx; yes = T.bt[1] * ky;
            if (autosw) { x6r = T.a[6][1] * kx; y6r = T.a[6][1] * ky; }
            double a = dt * T.a[2][1];
            n0 = fma(a, K.get(1, 0), u0); n1 = fma(a, K.get(1, 1), u1); n2 = fma(a, K.get(1, 2), u2);
            ts = fma(T.c[1], dt, t);
            ph = 2;
        }
    }
    p.u0 = u0; p.u1 = u1; p.u2 = u2; p.u3 = K.ld(KS_U3); p.u4 = K.ld(KS_U4);
    p.t = t; p.dt = dt; p.qold = K.ld(KS_QOLD); p.iter = iter;
    c.rhs += nrhs;
    attempts_io = attempts;
    if (autosw) as_count = (int)K.ld(KS_AS);
    return switched;
}
#undef PH_COEF_ON
#undef PH_PROP

/* ---- ParticleInCell ------------------------------------------------------- */
/* get_absolute_i_and_w(zp, i_node): floor offset and ceil-side weight */
PM_HD bool weights_1d(double zp, int32_t& f, double& wc) {
    if (!(fabs(zp) < 1.0e9)) return false;
    double base = floor(zp);
    f = (int32_t)base;
    wc = rint((zp - base) * 1e6) / 1e6;
    return true;
}

/* pos % N (C remainder: the sign of pos) without the 64-bit division whenever |pos| < 2N — always, for a corner
   within the supported reach of a node; the division stays behind for anything else, so the value is the same */
PM_HD int64_t rem_near(int64_t pos, int64_t N) {
    if (pos >= 0) {
        if (pos < N) return pos;
        if (pos < 2 * N) return pos - N;
    } else {
        if (pos > -N) return pos;
        if (pos > -2 * N) return pos + N;
    }
    return pos % N;
}
PM_HD int64_t wrap_index(int64_t pos, int64_t N) {
    pos = rem_near(pos, N);
    if (pos < 0) pos += N;
    else if (pos == 0) pos += N;
    return pos;
}

/* push_to_grid! boundary rules for one corner (1-based global i,j):
   returns false if the corner is dropped, else the 1-based target (ii,jj) */
PM_HD bool corner_target(int Nx, int Ny, int bx, int by, int64_t i, int64_t j, int64_t& ii, int64_t& jj) {
    if (((bx == PICLES_BND_NONPERIODIC) && !(i > 0 && i <= Nx)) ||
        ((by == PICLES_BND_NONPERIODIC) && !(j > 0 && j <= Ny)) || ((by == PICLES_BND_TRIPOLAR_NORTH) && (j < 1)))
        return false;
    if ((by == PICLES_BND_TRIPOLAR_NORTH) && (j > Ny)) {
        if (bx != PICLES_BND_PERIODIC) return false;
        if (i < 0) ii = Nx - (Nx + rem_near(i, Nx));
        else ii = Nx - rem_near(i, Nx);
        jj = 2 * (int64_t)Ny - j + 1;
        if (ii < 1 || ii > Nx || jj < 1 || jj > Ny) return false;
    } else {
        ii = wrap_index(i, Nx);
        jj = wrap_index(j, Ny);
    }
    return true;
}

PM_HD int32_t pack_cell(int32_t fx, int32_t fy, int cls) {
    return (int32_t)(((uint32_t)(fx + PH_CELL_BIAS) & 0x3fffu) | (((uint32_t)(fy + PH_CELL_BIAS) & 0x3fffu) << 14) |
                     ((uint32_t)(cls & 1) << 28));
}
PM_HD void unpack_cell(int32_t cell, int32_t& fx, int32_t& fy, int& cls) {
    fx = (int32_t)((uint32_t)cell & 0x3fffu) - PH_CELL_BIAS;
    fy = (int32_t)(((uint32_t)cell >> 14) & 0x3fffu) - PH_CELL_BIAS;
    cls = (int)(((uint32_t)cell >> 28) & 1u);
}
/* reach of one deposit record: max |corner - home| over its four corners (0 if none) */
PM_HD int32_t cell_reach(int32_t cell) {
    if (cell == PH_CELL_INVALID) return 0;
    int32_t fx, fy, d, r = 0;
    int cls;
    unpack_cell(cell, fx, fy, cls);
    d = fx < 0 ? -fx : fx; if (d > r) r = d;
    d = fx + 1 < 0 ? -(fx + 1) : fx + 1; if (d > r) r = d;
    d = fy < 0 ? -fy : fy; if (d > r) r = d;
    d = fy + 1 < 0 ? -(fy + 1) : fy + 1; if (d > r) r = d;
    return r;
}


/* ---- ParticleToNode! as a gather --------------------------------------------- */
/* read-only view of the deposit records of one strip (+ halo rows) */
struct RecView {
    int Nx, Ny, bx, by; /* global shape and boundary types */
    int j0, ny, halo;   /* strip: first owned global row (0-based), rows owned, halo rows the planes hold on each side */
    int hx;             /* ... of which the hx next to the owned rows carry this step's neighbour records */
    int pitch;          /* elements between consecutive rows of the record planes (>= Nx) */
    const double *e, *mx, *my, *wx, *wy;
    const int32_t* cell;
};

/* local extended row of global 1-based row j, or -1 */
PM_HD int ext_row(const RecView& V, int64_t j) {
    /* only the hx halo rows next to the owned ones were exchanged: a row further out is not "that row,
       empty" but a row this strip does not have — on a periodic ring it may still be there as a wrapped row */
    const int64_t lo = V.halo - V.hx, hi = V.ny + V.halo + V.hx;
    int64_t r = j - 1 - V.j0 + V.halo;
    if (r >= lo && r < hi) return (int)r;
    if (V.by == PICLES_BND_PERIODIC) { /* wrapped neighbour rows live in the halo */
        r = j + V.Ny - 1 - V.j0 + V.halo;
        if (r >= lo && r < hi) return (int)r;
        r = j - V.Ny - 1 - V.j0 + V.halo;
        if (r >= lo && r < hi) return (int)r;
    }
    return -1;
}

/* insert v into a sorted list without duplicates */
PM_HD void list_insert(int* lst, int& n, int v) {
    int k = 0;
    while (k < n && lst[k] < v) k++;
    if (k < n && lst[k] == v) return;
    for (int m = n; m > k; m--) lst[m] = lst[m - 1];
    lst[k] = v;
    n++;
}

#define PH_GEN_LIST_MAX (2 * (2 * PH_REACH_MAX + 1) + 2)

/* candidate source indices (1-based, in-domain, ascending) along one axis whose corners
   can reach target T directly (|src - T| <= R, wrapped or clipped) or through the
   tripolar fold (rows: corner row 2N+1-T; columns: corner column ≡ N-T mod N) */
PM_HD void axis_candidates(int* lst, int& n, int64_t T, int R, int N, int bnd, bool fold_x, bool fold_y) {
    n = 0;
    for (int d = -R; d <= R; d++) {
        int64_t s = T + d;
        if (bnd == PICLES_BND_PERIODIC) s = wrap_index(s, N);
        else if (s < 1 || s > N) continue;
        list_insert(lst, n, (int)s);
    }
    if (fold_y) {
        int64_t cj = 2 * (int64_t)N + 1 - T;
        for (int d = -R; d <= R; d++) {
            int64_t s = cj + d;
            if (s < 1 || s > N) continue;
            list_insert(lst, n, (int)s);
        }
    }
    if (fold_x) {
        int64_t ci = (int64_t)N - T;
        for (int d = -R; d <= R; d++) list_insert(lst, n, (int)wrap_index(ci + d, N));
    }
}

/* window fast path with a compile-time reach R (fully unrolled (2R+1)^2 window): every
   candidate row/column is addressable relative to `base`, the element of (I,J) itself, in
   planes of row pitch `pitch` — the record planes in HBM, or a tile of them staged in shared
   memory (PITCH > 0: compile-time pitch, so every offset is an immediate).  Elements that
   hold no deposit (PH_CELL_INVALID, or the zero fill of a TMA box outside the planes)
   never match.  Order: class, then j, then i — the reference's ocean_points order. */
template <int R, int PITCH, int NCLS>
PM_HD void gather_window(const double* __restrict__ pe, const double* __restrict__ pmx, const double* __restrict__ pmy,
                         const double* __restrict__ pwx, const double* __restrict__ pwy,
                         const int32_t* __restrict__ pcell, int pitch_rt, int64_t base, double& s0, double& s1,
                         double& s2) {
    const int pitch = PITCH > 0 ? PITCH : pitch_rt;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int cls = 0; cls < NCLS; cls++) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (int dj = -R; dj <= R; dj++) {
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
            for (int di = -R; di <= R; di++) {
                int64_t le = base + (int64_t)dj * pitch + di;
                uint32_t cell = (uint32_t)pcell[le];
                /* source (I+di, J+dj) reaches (I,J) iff fx in {-di-1,-di} and fy in {-dj-1,-dj};
                   PH_CELL_INVALID (all ones) and a zero-filled cell decode to |offsets| ~ 8191
                   and never match.  With one class every record is class 0. */
                unsigned dx = (unsigned)(PH_CELL_BIAS - di) - (cell & 0x3fffu);
                unsigned dy = (unsigned)(PH_CELL_BIAS - dj) - ((cell >> 14) & 0x3fffu);
                if (dx > 1u || dy > 1u) continue;
                if (NCLS > 1 && (int)((cell >> 28) & 1u) != cls) continue;
                double wxc = pwx[le], wyc = pwy[le];
                double wx = dx ? wxc : 1.0 - wxc;
                double wy = dy ? wyc : 1.0 - wyc;
                double w = wx * wy;
                s0 += w * pe[le];
                s1 += w * pmx[le];
                s2 += w * pmy[le];
            }
        }
    }
}

/*
 * Sum of all deposits landing on global node (I,J) (1-based), accumulated in the
 * reference's single-thread order: ocean_points order (class 0 = mask 1 nodes, then
 * class 1 = mask 3 nodes when the model is periodic; within a class column-major, i
 * fastest), corners (x0,y0),(x1,y0),(x0,y1),(x1,y1) within a particle.  R = reach of
 * this step (max |corner - home| over all deposits).  s0,s1,s2 are in/out: the caller
 * initialises them with 0 (run!: State .= 0 before the step) or with the node's current
 * State (a bare time_step! on a non-zero State accumulates, ParticleInCell.jl:372).
 */
PM_HD void gather_node(const RecView& V, int I, int J, int R, int n_classes, double& s0, double& s1, double& s2) {
    const int Nx = V.Nx, Ny = V.Ny;
    bool fast_x = (V.bx == PICLES_BND_NONPERIODIC) || (I > R && I <= Nx - R);
    bool fast_y = (V.by == PICLES_BND_NONPERIODIC) || (V.by == PICLES_BND_PERIODIC && J > R && J <= Ny - R) ||
                  (V.by == PICLES_BND_TRIPOLAR_NORTH && J <= Ny - R);
    /* deep interior, small reach: unrolled window (same order: class, j, then i) */
    if (R <= 2 && I > R && I <= Nx - R && J > R && J <= Ny - R && fast_x && fast_y) {
        int64_t base = (int64_t)(J - 1 - V.j0 + V.halo) * V.pitch + (I - 1);
        if (n_classes == 1) {
            if (R <= 1) gather_window<1, 0, 1>(V.e, V.mx, V.my, V.wx, V.wy, V.cell, V.pitch, base, s0, s1, s2);
            else gather_window<2, 0, 1>(V.e, V.mx, V.my, V.wx, V.wy, V.cell, V.pitch, base, s0, s1, s2);
        } else {
            if (R <= 1) gather_window<1, 0, 2>(V.e, V.mx, V.my, V.wx, V.wy, V.cell, V.pitch, base, s0, s1, s2);
            else gather_window<2, 0, 2>(V.e, V.mx, V.my, V.wx, V.wy, V.cell, V.pitch, base, s0, s1, s2);
        }
        return;
    }
    if (fast_x && fast_y) {
        /* no wrap, no fold: a source (i,j) reaches (I,J) through exactly one corner,
           dx = I-i-fx in {0,1}, dy = J-j-fy in {0,1} */
        int jlo = (J - R > 1) ? J - R : 1, jhi = (J + R < Ny) ? J + R : Ny;
        int ilo = (I - R > 1) ? I - R : 1, ihi = (I + R < Nx) ? I + R : Nx;
        for (int cls = 0; cls < n_classes; cls++) {
            for (int j = jlo; j <= jhi; j++) {
                int64_t row = (int64_t)(j - 1 - V.j0 + V.halo) * V.pitch;
                for (int i = ilo; i <= ihi; i++) {
                    int64_t le = row + (i - 1);
                    int32_t cell = V.cell[le];
                    if (cell == PH_CELL_INVALID) continue;
                    int32_t fx, fy;
                    int k;
                    unpack_cell(cell, fx, fy, k);
                    int dx = I - i - fx, dy = J - j - fy;
                    if (k != cls || (unsigned)dx > 1u || (unsigned)dy > 1u) continue;
                    double wxc = V.wx[le], wyc = V.wy[le];
                    double wx = dx ? wxc : 1.0 - wxc;
                    double wy = dy ? wyc : 1.0 - wyc;
                    double w = wx * wy;
                    s0 += w * V.e[le];
                    s1 += w * V.mx[le];
                    s2 += w * V.my[le];
                }
            }
        }
        return;
    }
    /* generic path (wrap / fold zones): enumerate candidate sources in canonical order
       and push all four corners through the reference's boundary rules */
    int rows[PH_GEN_LIST_MAX], cols[PH_GEN_LIST_MAX];
    int nr, nc;
    bool tri = (V.by == PICLES_BND_TRIPOLAR_NORTH);
    axis_candidates(rows, nr, J, R, Ny, tri ? PICLES_BND_NONPERIODIC : V.by, false, tri);
    axis_candidates(cols, nc, I, R, Nx, V.bx, tri && V.bx == PICLES_BND_PERIODIC, false);
    const int64_t tgt = (int64_t)(I - 1) + (int64_t)(J - 1) * Nx;
    for (int cls = 0; cls < n_classes; cls++) {
        for (int a = 0; a < nr; a++) {
            int j = rows[a];
            int er = ext_row(V, j);
            if (er < 0) continue;
            for (int b = 0; b < nc; b++) {
                int i = cols[b];
                int64_t le = (int64_t)er * V.pitch + (i - 1);
                int32_t cell = V.cell[le];
                if (cell == PH_CELL_INVALID) continue;
                int32_t fx, fy;
                int k;
                unpack_cell(cell, fx, fy, k);
                if (k != cls) continue;
                if (V.by != PICLES_BND_PERIODIC) {
                    /* rows first (no wrap in y here): a corner row jy lands on row J directly (jy == J <= Ny) or through
                       the fold (2Ny - jy + 1 == J); most candidates of the cross product fail this and need none of the
                       four corner evaluations */
                    const int64_t jy0 = (int64_t)j + fy, jf = 2 * (int64_t)Ny + 1 - J;
                    if (jy0 != J && jy0 + 1 != J && jy0 != jf && jy0 + 1 != jf) continue;
                }
                double wxc = V.wx[le], wyc = V.wy[le];
                double ce = V.e[le], cmx = V.mx[le], cmy = V.my[le];
                for (int q = 0; q < 4; q++) { /* (x0,y0),(x1,y0),(x0,y1),(x1,y1) */
                    int dx = q & 1, dy = q >> 1;
                    int64_t ii, jj;
                    if (!corner_target(Nx, Ny, V.bx, V.by, (int64_t)i + fx + dx, (int64_t)j + fy + dy, ii, jj)) continue;
                    if ((ii - 1) + (jj - 1) * Nx != tgt) continue;
                    double wx = dx ? wxc : 1.0 - wxc;
                    double wy = dy ? wyc : 1.0 - wyc;
                    double w = wx * wy;
                    s0 += w * ce;
                    s1 += w * cmx;
                    s2 += w * cmy;
                }
            }
        }
    }
}

/* levels 0..nseg of one particle's staged wind: t, the intermediate ones, t+DT */
PM_HD void make_wind(Wind& w, int nmid, double wu0, double wv0, double wu1, double wv1, const double* um, const double* vm,
                     double t_start, double DT) {
    w.nseg = nmid + 1;
    w.ul[0] = wu0; w.vl[0] = wv0;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int k = 1; k <= PH_WIND_SEG_MAX; k++) {
        w.ul[k] = (k <= nmid) ? um[k - 1] : ((k == nmid + 1) ? wu1 : 0.0);
        w.vl[k] = (k <= nmid) ? vm[k - 1] : ((k == nmid + 1) ? wv1 : 0.0);
    }
    w.t_start = t_start; w.inv_DT = 1.0 / DT;
}

/* tail of advance!: NaN / Inf / e_max fix-ups (mapping_2D.jl:196-235) and the deposit record that
   replaces ParticleToNode! */
PM_HD void advance_finish(const picles_params_t& P, Particle& p, bool on, int mask, double DT, double wu0, double wv0,
                          double wu1, double wv1, Record& rec, Tally& c) {
    bool anynan = (p.u0 != p.u0) | (p.u1 != p.u1) | (p.u2 != p.u2);
    bool anyinf = pm_isinf(p.u0) | pm_isinf(p.u1) | pm_isinf(p.u2);
    if (anynan) {
        reset_particle_values(P, wu1, wv1, DT, p);
        p.flags |= PICLES_PF_DT_RESET; p.status |= PICLES_PST_NAN_RESET; c.fixups++;
    } else if (anyinf) {
        reset_particle_values(P, wu0, wv0, DT, p);
        p.flags |= PICLES_PF_DT_RESET; p.status |= PICLES_PST_INF_RESET; c.fixups++;
    } else if (p.u0 > P.log_energy_maximum) {
        p.u0 = P.log_energy_maximum;
        p.flags |= PICLES_PF_DT_RESET; p.status |= PICLES_PST_EMAX_CLAMP; c.fixups++;
    }
    if (P.on_persist) p.flags = (uint8_t)(on ? (p.flags | PICLES_PF_ON) : (p.flags & ~PICLES_PF_ON));
    /* ParticleToNode!: weights + charge -> record */
    rec.cell = PH_CELL_INVALID;
    rec.e = rec.mx = rec.my = rec.wxc = rec.wyc = 0.0;
    if (on) {
        int32_t fx, fy;
        double wxc, wyc;
        if (weights_1d(p.u3, fx, wxc) && weights_1d(p.u4, fy, wyc)) {
            int32_t r = 0, d;
            d = fx < 0 ? -fx : fx; if (d > r) r = d;
            d = fx + 1 < 0 ? -(fx + 1) : fx + 1; if (d > r) r = d;
            d = fy < 0 ? -fy : fy; if (d > r) r = d;
            d = fy + 1 < 0 ? -(fy + 1) : fy + 1; if (d > r) r = d;
            if (r > c.reach) c.reach = r;
            if (r < PH_CELL_BIAS - 2) {
                charge(p.u0, p.u1, p.u2, rec.e, rec.mx, rec.my);
                rec.wxc = wxc; rec.wyc = wyc;
                rec.cell = pack_cell(fx, fy, mask == PICLES_MASK_GRID_BOUNDARY);
            }
            c.deposited++;
        }
    }
}

/*
 * advance! of one particle.  um/vm: the nmid intermediate wind levels at t + k*DT/(nmid+1),
 * k = 1..nmid (nmid = 0: none).  Returns true only in the AUTOSW instantiation, when AutoSwitch
 * needs Rosenbrock23 for this particle (it is the current algorithm at the start of the step, or
 * the monitor switched just now): p then holds the state reached so far (t < t_start + DT),
 * attempts_out the attempts made, nothing else has been done, and the caller finishes the step
 * with advance_resume() — out of line, so the hot loop here shares no registers with the cold code.
 */
template <bool AUTOSW, int TSIT5 = 0, class KS>
PM_HD bool advance_particle(const picles_params_t& P, Particle& p, int mask, double DT, double wu0, double wv0,
                            double wu1, double wv1, int nmid, const double* um, const double* vm, const double* M,
                            double pc, Record& rec, Tally& c, KS& K, int& attempts_out) {
    double t_start = p.t;
    bool on = (p.flags & PICLES_PF_ON) != 0;
    if (on) {
        if (!(p.status & (PICLES_PST_MAXITERS | PICLES_PST_DTMIN | PICLES_PST_UNSTABLE))) {
            const bool autosw = AUTOSW && (P.solver == PICLES_SOLVER_AUTOTSIT5);
            const double tstop = t_start + DT;
            int attempts = 0;
            int as_count = 0;
            if (autosw) {
                if (p.as > PH_AS_CLAMP) { attempts_out = 0; return true; } /* Rosenbrock23 is current */
                as_count = (int)p.as;
            }
            Hoist H;
            {
                Wind w;
                make_wind(w, nmid, wu0, wv0, wu1, wv1, um, vm, t_start, DT);
                wind_to_slots(P, w, K, H);
            }
            const bool switched = integrate<AUTOSW, TSIT5>(P, wu0, wv0, H, M, pc, tstop, p, c, K, as_count, attempts);
            if (autosw) {
                p.as = (int8_t)(as_count + (switched ? PH_AS_STIFF : 0));
                if (switched && (p.t < tstop)) { attempts_out = attempts; return true; }
            }
            c.integrated++;
            if (attempts > c.max_attempts) c.max_attempts = attempts;
            attempts_out = attempts;
        }
    } else {
        if (wu1 * wu1 + wv1 * wv1 >= P.wind_min_squared) {
            reset_particle_values(P, wu1, wv1, DT, p);
            p.flags |= PICLES_PF_DT_RESET;
            on = true;
            c.reseed++;
        }
    }
    advance_finish(P, p, on, mask, DT, wu0, wv0, wu1, wv1, rec, c);
    return false;
}

/* the Rosenbrock23 attempts of a particle AutoSwitch has declared stiff (stiff.h, out of line).
   Everything the cold code touches travels in one struct.  true: handed back to Tsit5 with time
   left in the step */
struct WindPoly {
    int nseg;
    double cu[PH_WIND_SEG_MAX + 1], cv[PH_WIND_SEG_MAX + 1]; /* c[0] = the level at t_start */
    double t0, scale;                                         /* sigma = (ts - t0) * scale */
};
struct StiffArgs {
    WindPoly W;
    double M[4];
    Particle p;
    int as_count, as_stiff, attempts;
    Tally c;
};
PM_HD_NOINLINE_DECL bool stiff_phase(const picles_params_t* Pp, StiffArgs* a, double pc, double tstop);

/* wind levels and projection kernel of one particle, by value (cold call) */
struct ResumeArgs {
    int mask, nmid, attempts;
    double DT, t_start, wu0, wv0, wu1, wv1, um[PH_WIND_SEG_MAX], vm[PH_WIND_SEG_MAX], M[4], pc;
};
/*
 * The rest of advance! for a particle advance_particle<true> handed over: alternate between
 * Rosenbrock23 (stiff_phase) and Tsit5 (a second, cold copy of the integration loop) until the step
 * is complete, then the common tail.  tally: a zeroed Tally of the caller, merged afterwards.
 */
template <class KS>
PM_HD_NOINLINE_DECL void advance_resume(const picles_params_t* Pp, const ResumeArgs* Rp, Particle* pp, Record* rec, Tally* cp, KS K) {
    const picles_params_t& P = *Pp;
    const ResumeArgs& R = *Rp;
    Particle& p = *pp;
    Tally& c = *cp;
    const double tstop = R.t_start + R.DT;
    Hoist H;
    {
        Wind w;
        make_wind(w, R.nmid, R.wu0, R.wv0, R.wu1, R.wv1, R.um, R.vm, R.t_start, R.DT);
        wind_to_slots(P, w, K, H);
    }
    int attempts = R.attempts;
    bool as_stiff = p.as > PH_AS_CLAMP;
    int as_count = as_stiff ? (int)p.as - PH_AS_STIFF : (int)p.as;
    bool stiff_now = as_stiff;
    for (;;) {
        if (stiff_now) {
            StiffArgs a; /* the wind polynomial back from the scratch slots */
            a.W.nseg = H.nseg;
            a.W.cu[0] = R.wu0; a.W.cv[0] = R.wv0;
            for (int m = 1; m <= PH_WIND_SEG_MAX; m++) {
                a.W.cu[m] = (m <= H.nseg) ? K.ld(KS_WCU + m - 1) : 0.0;
                a.W.cv[m] = (m <= H.nseg) ? K.ld(KS_WCV + m - 1) : 0.0;
            }
            a.W.t0 = K.ld(KS_WT0); a.W.scale = K.ld(KS_WIDT);
            a.M[0] = R.M[0]; a.M[1] = R.M[1]; a.M[2] = R.M[2]; a.M[3] = R.M[3];
            a.p = p;
            a.as_count = as_count; a.as_stiff = 1; a.attempts = attempts;
            tally_zero(a.c);
            const bool back = stiff_phase(Pp, &a, R.pc, tstop);
            p = a.p;
            as_count = a.as_count; as_stiff = a.as_stiff != 0; attempts = a.attempts;
            c.substeps += a.c.substeps; c.rejects += a.c.rejects; c.rhs += a.c.rhs; c.failed += a.c.failed;
            c.stiff_attempts += a.c.stiff_attempts;
            if (!back) break;
        }
        stiff_now = integrate<true>(P, R.wu0, R.wv0, H, R.M, R.pc, tstop, p, c, K, as_count, attempts);
        if (!stiff_now) break;
        as_stiff = true;
        if (!(p.t < tstop)) break; /* switched on the last attempt of the step */
    }
    p.as = (int8_t)(as_count + (as_stiff ? PH_AS_STIFF : 0));
    c.integrated++;
    if (attempts > c.max_attempts) c.max_attempts = attempts;
    advance_finish(P, p, true, R.mask, R.DT, R.wu0, R.wv0, R.wu1, R.wv1, *rec, c);
}

/* ---- remesh! / NodeToParticle! ---------------------------------------------- */
PM_HD void remesh_particle(const picles_params_t& P, Particle& p, double e, double mx, double my, double wu,
                           double wv, double DT, Tally& c) {
    bool boundary = (p.flags & PICLES_PF_BOUNDARY) != 0;
    bool on;
    if (!boundary && (e >= P.minimal_state[0]) && (mx * mx + my * my >= P.minimal_state[1])) {
        vertex(e, mx, my, p);
        p.flags |= PICLES_PF_DT_RESET;
        on = true;
        c.A++;
    } else if (!boundary && (wu * wu + wv * wv >= P.wind_min_squared)) {
        reset_particle_values(P, wu, wv, DT, p);
        p.qold = PH_QOLDINIT; p.iter = 0; p.status = 0;
        p.as = 0; /* reinit!: a fresh AutoSwitch state */
        p.flags |= PICLES_PF_DT_RESET;
        on = true;
        c.B++;
    } else if (boundary && (wu * wu + wv * wv >= P.wind_min_squared)) {
        reset_particle_values(P, wu, wv, DT, p);
        p.qold = PH_QOLDINIT; p.iter = 0; p.status = 0;
        p.as = 0;
        p.flags |= PICLES_PF_DT_RESET;
        on = true;
        c.C++;
    } else {
        on = false;
        c.D++;
    }
    if (P.on_persist) p.flags = (uint8_t)(on ? (p.flags | PICLES_PF_ON) : (p.flags & ~PICLES_PF_ON));
}

/* ---- SeedParticle -------------------------------------------------------- */
/* returns false for land (mask 0: dummy instance); fills p and the initial node state */
PM_HD bool seed_particle(const picles_params_t& P, int mask, double wu, double wv, Particle& p, double& e,
                         double& mx, double& my) {
    p.u0 = p.u1 = p.u2 = p.u3 = p.u4 = 0.0;
    p.t = 0.0; p.dt = 0.0; p.qold = 0.0; p.iter = 0; p.flags = 0; p.status = 0; p.as = 0;
    e = mx = my = 0.0;
    if (mask == PICLES_MASK_LAND) return false;
    bool on;
    if (!P.has_defaults) {
        if (sqrt(wu * wu + wv * wv) > sqrt(2.0)) {
            windsea(wu, wv, P.seed_timescale, p.u0, p.u1, p.u2);
            on = true;
        } else {
            minimal_particle(wu, wv, P.seed_timescale, p.u0, p.u1, p.u2);
            on = false;
        }
    } else {
        p.u0 = P.defaults[0]; p.u1 = P.defaults[1]; p.u2 = P.defaults[2];
        on = true;
    }
    bool boundary = P.periodic_boundary ? (mask == PICLES_MASK_LAND_BOUNDARY) : (mask >= 2);
    bool active = (mask == PICLES_MASK_OCEAN) || (P.periodic_boundary && mask == PICLES_MASK_GRID_BOUNDARY);
    if (on) charge(p.u0, p.u1, p.u2, e, mx, my);
    p.dt = P.dt; p.qold = PH_QOLDINIT;
    p.flags = (uint8_t)((on ? PICLES_PF_ON : 0) | (boundary ? PICLES_PF_BOUNDARY : 0) | (active ? PICLES_PF_ACTIVE : 0));
    return true;
}

} /* namespace picles */
#endif /* PICLES_PHYSICS_H */
