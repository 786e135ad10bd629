/*
 * pmath_body.h — bodies of the pmath functions that divide or take square roots.
 * Included (twice) by pmath.h with PMV / PM_DIV / PM_DIVZ / PM_SQRT / PM_BADP / PM_BADA
 * set for the IEEE ("_safe") or the device fast-path ("_fast") instantiation; see pmath.h.
 * No include guard on purpose.  Straight-line code only (selects, no early returns).
 */

/* log(x) for x positive and finite (normal or subnormal), fdlibm/musl kernel */
PM_FN double PMV(pm_log_core)(double x PM_BADP) {
    uint64_t ub = (uint64_t)pm_d2i(x);
    int sub = ((ub >> 52) == 0); /* +0 or positive subnormal: scale up by 2^54 */
    double xs = sub ? x * 18014398509481984.0 : x;
    int k = sub ? -54 : 0;
    int64_t b = pm_d2i(xs);
    /* normalise the mantissa to [sqrt(2)/2, sqrt(2)) */
    uint32_t hx = (uint32_t)((uint64_t)b >> 32);
    hx += 0x3ff00000u - 0x3fe6a09eu;
    k += (int)(hx >> 20) - 0x3ff;
    hx = (hx & 0x000fffffu) + 0x3fe6a09eu;
    b = (int64_t)(((uint64_t)hx << 32) | ((uint64_t)b & 0xffffffffu));
    double m = pm_i2d(b);

    double f = m - 1.0;
    double hfsq = 0.5 * f * f;
    double s = PM_DIVZ(f, 2.0 + f);
    double z = s * s;
    double w = z * z;
    double t1 = w * (PMK.Lg[2] + w * (PMK.Lg[4] + w * PMK.Lg[6]));
    double t2 = z * (PMK.Lg[1] + w * (PMK.Lg[3] + w * (PMK.Lg[5] + w * PMK.Lg[7])));
    double R = t2 + t1;
    double dk = (double)k;
    return s * (hfsq + R) + dk * PMK.LN2_LO - hfsq + f + dk * PMK.LN2_HI;
}
/* log(x): x <= 0, inf, NaN handled by the trailing selects */
PM_FN double PMV(pm_log)(double x PM_BADP) {
    double res = PMV(pm_log_core)(x PM_BADA);
    res = pm_isinf(x) ? x : res;
    res = (x == 0.0) ? -pm_inf() : res;
    res = (x < 0.0) ? pm_nan() : res;
    return (x != x) ? x : res;
}

PM_FN double PMV(pm_log10)(double x PM_BADP) {
    /* a plain quotient is enough for the initial-step heuristic this feeds */
    return PM_DIVZ(PMV(pm_log)(x PM_BADA), PMK.LN10);
}

/* x^y for x >= 0 (naive exp(y*log x): controller and fetch-law exponents) */
PM_FN double PMV(pm_pow)(double x, double y PM_BADP) {
    double l = PMV(pm_log)(x PM_BADA);
    double r = pm_exp(y * l);
    r = (x == 0.0) ? ((y > 0.0) ? 0.0 : pm_inf()) : r;
    r = (x < 0.0) ? pm_nan() : r;
    r = (x != x || y != y) ? pm_nan() : r;
    return (y == 0.0) ? 1.0 : r;
}

/* tanh(x) = em1/(em1+2), em1 = expm1(2|x|) */
PM_FN double PMV(pm_tanh)(double x PM_BADP) {
    double ax = fabs(x);
    /* fast instantiation: the clamps below as high-word compares (pm_ge_hw).  At ax == 25 and ax == 22 both sides of
       each select give the same value (2*25; tanh(22) rounds to 1), so `>=` is `>` here */
#ifdef PM_FAST_RANGE
    double y = pm_ge_hw(ax, 25.0) ? 50.0 : 2.0 * ax;
#else
    double y = (ax > 25.0) ? 50.0 : 2.0 * ax;
#endif
#ifndef PM_FAST_RANGE
    y = (x != x) ? 0.0 : y;
#endif
    /* fast instantiation: a NaN argument is the CALLER's to flag (the right-hand side's argument is NaN only
       if the quotient it comes from is, and that division raises the flag); nothing here tests for it */
    double em, sj, sl;
    int k = PM_EXP_REDUCE(y, &em, &sj, &sl); /* 0 <= k <= 72 */
    /* expm1(y) = T (1 + em) - 1 with T = 2^k 2^(j/128) = th + tl: T - 1 is exact for T < 2 (and free of
       cancellation above), and for y below ln2/256 it is em itself (T = 1, tl = 0) */
    double s = pm_pow2i(k);
    double th = sj * s, tl = sl * s;
    double em1 = fma(th, em, (th - 1.0) + tl);
    double t = PM_DIVZ(em1, em1 + 2.0);
#ifdef PM_FAST_RANGE
    t = pm_ge_hw(ax, 22.0) ? 1.0 : t;
#else
    t = (ax > 22.0) ? 1.0 : t;
#endif
    t = copysign(t, x); /* t >= 0: one bit operation instead of compare, negate and select */
#ifdef PM_FAST_RANGE
    return t;
#else
    return (x != x) ? x : t;
#endif
}

/* sech(x) = 2e/(e^2+1), e = exp(min(|x|,350)); only ever used squared inside
   1 - 1.25*sech^2, where anything below 1e-9 vanishes */
PM_FN double PMV(pm_sech)(double x PM_BADP) {
    double ax = fabs(x);
#ifdef PM_FAST_RANGE
    ax = pm_ge_hw(ax, 350.0) ? 350.0 : ax; /* the same clamp: ties give 350 either way */
#else
    ax = (ax > 350.0) ? 350.0 : ax;
#endif
#ifndef PM_FAST_RANGE
    ax = (x != x) ? 0.0 : ax; /* fast instantiation: NaN is the caller's to flag, as in pm_tanh */
#endif
#ifdef PM_FAST_RANGE
    double e = pm_exp_core_inrange(ax); /* 0 <= ax <= 350 */
#else
    double e = pm_exp_core(ax);
#endif
    /* e in [1, 2^505]: dividend 2e in [2, 2^506], divisor e^2 + 1 in [2, 2^1010], quotient in [2^-505, 1] —
       always inside the fast path's premises, so the division carries no validity test */
    double t = PM_DIV_NC(2.0 * e, fma(e, e, 1.0));
#ifdef PM_FAST_RANGE
    return t;
#else
    return (x != x) ? x : t;
#endif
}

/* exp(x): the fast instantiation flags everything outside [-700, 700] (and NaN) */
PM_FN double PMV(pm_expx)(double x PM_BADP) {
#ifdef PM_FAST_RANGE
    *pm_bad |= pm_absge_hw(x, 700.0) ? 1u : 0u; /* also flags |x| == 700, which the IEEE instantiation gives the same bits */
    return pm_exp_core_inrange(x);
#else
    return pm_exp(x);
#endif
}
