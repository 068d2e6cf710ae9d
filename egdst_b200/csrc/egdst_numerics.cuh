// egdst_numerics.cuh -- device numerics shared by the solver and simulator kernels.
//
// Device restatement of the reference's shared numerics (@egdstmodel/egdst_lib.c):
//   bracket search      egdst_lib.c:123-165  (bxsearch / bxsearch_common / optimd)
//   linter              egdst_lib.c:168-176
//   linter_extrap       egdst_lib.c:179-206
//   cdfni (Acklam)      egdst_lib.c:435-519
//   cdfinv/rescale/expectation per DISTRIB   egdst_lib.c:66-101
//   cashinhandinverse   egdst_lib.c:275-296
// All FP64.  Nothing here allocates; tables are read through plain pointers so the same code
// serves global memory, shared memory (TMA-staged) and the host emulator used for debugging.
#pragma once

#include "modelspec_dev.h"

#ifndef EGDST_DEV
#ifdef __CUDACC__
#define EGDST_DEV static __device__ __forceinline__
#else
#define EGDST_DEV static inline
#endif
#endif

// ---------------------------------------------------------------------------------------------
// bracket search: index i of the interval [grid[i], grid[i+1]] used for interpolation.
// Reference semantics (egdst_lib.c:138-165): 0 if x<grid[1]; n-2 if x>=grid[n-2] (type 0) or n-1 if
// x>=grid[n-1] (type 1); otherwise the largest interior i with grid[i]<=x.  For a strictly increasing
// grid that is "largest i with grid[i]<=x, clamped", which is what is computed here (branch-free
// bisection over the same interior range, so the visiting order of the reference is kept).
// ---------------------------------------------------------------------------------------------
EGDST_DEV int egdst_bracket(double x, const double *__restrict__ grid, int n, int type) {
    if (x < grid[1]) return 0;
    if (type == 0 && x >= grid[n - 2]) return n - 2;
    if (type == 1 && x >= grid[n - 1]) return n - 1;
    int lo = 1, hi = n - 2;
    while (hi - lo > 1) {
        int mid = (hi + lo) >> 1;
        if (grid[mid] > x) hi = mid; else lo = mid;
    }
    return lo;
}

// optimal discrete decision from the threshold table (egdst_lib.c:129-132)
EGDST_DEV int egdst_optimd(double m, const double *__restrict__ th, const double *__restrict__ dd, int nth) {
    if (nth <= 1) return (int)dd[0];  // the reference reads grid[1] here (SURVEY 8a quirks); one threshold => one choice
    return (int)dd[egdst_bracket(m, th, nth, 1)];
}
// The decision of policy() for the simulator and call() (egdst_simulator.c:145-199): a linear scan for the last
// threshold <= m (the first decision below every threshold).  The reference's solver uses the bisection of optimd
// instead; the two agree on increasing thresholds but not on others, so each path keeps its reference's rule.
EGDST_DEV int egdst_policy_decision(double m, const double *th, const double *dd, int nth) {
    int ith = 0;
    while (ith < nth && m >= th[ith]) ith++;
    return (int)dd[ith > 0 ? ith - 1 : 0];
}

// linear interpolation / extrapolation on interval i (egdst_lib.c:175)
EGDST_DEV double egdst_lerp(double x, double g0, double g1, double f0, double f1) {
    double w = g1 - g0;
    return f1 * (x - g0) / w + f0 * (g1 - x) / w;
}

// The same quotients a/w, correctly rounded, when several numerators share one denominator (Markstein: with
// y = RN(1/w), q0 = RN(a*y), r = a - w*q0 exactly (fma), RN(q0 + r*y) is the IEEE quotient).  The EGM node divides
// four times by the same interval width; this is bit-identical to four `/` at a third of the instructions.
EGDST_DEV double egdst_div_by(double a, double w, double y) {
    const double q0 = a * y;
    const double r = fma(-w, q0, a);
    return fma(r, y, q0);
}
EGDST_DEV bool egdst_div_safe(double w) { const double aw = fabs(w); return aw > 1e-290 && aw < 1e290; }
EGDST_DEV double egdst_lerp_y(double x, double g0, double g1, double f0, double f1, double w, double y) {
    const double a1 = f1 * (x - g0), a0 = f0 * (g1 - x);
    if (!(fabs(a1) < 1e290 && fabs(a0) < 1e290)) return a1 / w + a0 / w;  // infinite values (V = -inf rows): plain quotients
    return egdst_div_by(a1, w, y) + egdst_div_by(a0, w, y);
}

EGDST_DEV double egdst_linter(double x, int n, const double *__restrict__ grid, const double *__restrict__ fun) {
    int i = egdst_bracket(x, grid, n, 0);
    return egdst_lerp(x, grid[i], grid[i + 1], fun[i], fun[i + 1]);
}

// interpolation with transform-weighted extrapolation outside the grid (egdst_lib.c:179-206)
EGDST_DEV double egdst_linter_extrap_at(const egdst_ctx *cx, const PeriodVars *prd, double x, int i, int n,
                                         const double *__restrict__ grid, const double *__restrict__ fun) {
    double f0 = fun[i], f1 = fun[i + 1];
    if (!isfinite(f0)) return f0;
    if (!isfinite(f1)) return f1;
    double g0 = grid[i], g1 = grid[i + 1];
    if (x > cx->a0 && (x > grid[n - 1] || x < grid[0])) {
        double tx = tr(cx, prd, x - cx->a0), t0 = tr(cx, prd, g0 - cx->a0), t1 = tr(cx, prd, g1 - cx->a0);
        return f1 * (tx - t0) / (t1 - t0) + f0 * (t1 - tx) / (t1 - t0);
    }
    return egdst_lerp(x, g0, g1, f0, f1);
}

// the same on an interval given by value (gfirst, glast = first and last abscissa of the table)
EGDST_DEV double egdst_linter_extrap_iv(const egdst_ctx *cx, const PeriodVars *prd, double x, double g0, double g1, double f0, double f1,
                                         double gfirst, double glast, double w, double y /* RN(1/w) or 0: plain divisions */) {
    if (!isfinite(f0)) return f0;
    if (!isfinite(f1)) return f1;
    if (x > cx->a0 && (x > glast || x < gfirst)) {
        double tx = tr(cx, prd, x - cx->a0), t0 = tr(cx, prd, g0 - cx->a0), t1 = tr(cx, prd, g1 - cx->a0);
        return f1 * (tx - t0) / (t1 - t0) + f0 * (t1 - tx) / (t1 - t0);
    }
    return y != 0.0 ? egdst_lerp_y(x, g0, g1, f0, f1, w, y) : egdst_lerp(x, g0, g1, f0, f1);
}

// ---------------------------------------------------------------------------------------------
// Acklam's rational approximation of the standard normal quantile (egdst_lib.c:435-519).
// Parity at 1e-9 needs this polynomial, not normcdfinv (SURVEY 0, fact 3).
// ---------------------------------------------------------------------------------------------
// The 21 coefficients live in the constant bank: as literals every use costs two uniform moves (UMOV) to
// materialise the 64-bit immediate; as c[bank][offset] they are direct DFMA operands.
#ifdef __CUDACC__
__constant__
#else
static const
#endif
double EGDST_CDFNI_K[21] = {
    -3.969683028665376e+01, 2.209460984245205e+02, -2.759285104469687e+02, 1.383577518672690e+02, -3.066479806614716e+01, 2.506628277459239e+00,  // a0..a5
    -5.447609879822406e+01, 1.615858368580409e+02, -1.556989798598866e+02, 6.680131188771972e+01, -1.328068155288572e+01,                        // b0..b4
    -7.784894002430293e-03, -3.223964580411365e-01, -2.400758277161838e+00, -2.549732539343734e+00, 4.374664141464968e+00, 2.938163982698783e+00,  // c0..c5
    7.784695709041462e-03, 3.224671290700398e-01, 2.445134137142996e+00, 3.754408661907416e+00};                                                // d0..d3

EGDST_DEV double egdst_cdfni(double p) {
    const double *K = EGDST_CDFNI_K;
    if (p < 0 || p > 1) return 0.0;
    if (p == 0) return -EGDST_INF;
    if (p == 1) return EGDST_INF;
    if (p < 0.02425 || p > 0.97575) {
        // both tails share one code path (less divergence): the upper tail is -f(1-p) (egdst_lib.c:506-511)
        const bool upper = p > 0.97575;
        const double q = sqrt(-2 * log(upper ? 1 - p : p));
        const double v = (((((K[11] * q + K[12]) * q + K[13]) * q + K[14]) * q + K[15]) * q + K[16]) /
                         ((((K[17] * q + K[18]) * q + K[19]) * q + K[20]) * q + 1);
        return upper ? -v : v;
    }
    const double q = p - 0.5, r = q * q;
    return (((((K[0] * r + K[1]) * r + K[2]) * r + K[3]) * r + K[4]) * r + K[5]) * q /
           (((((K[6] * r + K[7]) * r + K[8]) * r + K[9]) * r + K[10]) * r + 1);
}

// The simulator's quantile: the same rational functions with fused Horner steps.  The solver transforms its ny
// quadrature abscissas with the separately rounded form above (bit-compatible with the reference build); the
// simulator evaluates one quantile per agent-period, where the contraction changes the shock in its last bits
// (far inside the 1e-9 of the parity protocol) and no discrete branch depends on those bits except at exact ties.
EGDST_DEV double egdst_cdfni_fused(double p) {
    const double *K = EGDST_CDFNI_K;
    if (p < 0 || p > 1) return 0.0;
    if (p == 0) return -EGDST_INF;
    if (p == 1) return EGDST_INF;
    if (p < 0.02425 || p > 0.97575) {
        const bool upper = p > 0.97575;
        const double q = sqrt(-2 * log(upper ? 1 - p : p));
        const double num = fma(fma(fma(fma(fma(K[11], q, K[12]), q, K[13]), q, K[14]), q, K[15]), q, K[16]);
        const double den = fma(fma(fma(fma(K[17], q, K[18]), q, K[19]), q, K[20]), q, 1.0);
        const double v = num / den;
        return upper ? -v : v;
    }
    const double q = p - 0.5, r = q * q;
    const double num = fma(fma(fma(fma(fma(K[0], r, K[1]), r, K[2]), r, K[3]), r, K[4]), r, K[5]) * q;
    const double den = fma(fma(fma(fma(fma(K[6], r, K[7]), r, K[8]), r, K[9]), r, K[10]), r, 1.0);
    return num / den;
}

// shock distribution helpers (egdst_lib.c:66-101); DISTRIB 1 = lognormal, 2 = normal
EGDST_DEV double egdst_cdfinv(double p, double mu, double sigma) {
#if EGDST_DISTRIB == 1
    return exp(sigma * egdst_cdfni_fused(p) + mu);
#else
    return sigma * egdst_cdfni_fused(p) + mu;
#endif
}
EGDST_DEV double egdst_expectation(const egdst_ctx *cx, const PeriodVars *curr, const PeriodVars *next) {
#if EGDST_DISTRIB == 1
    double s = sigma_param(cx, curr, next);
    return exp(mu_param(cx, curr, next) + s * s / 2);
#else
    return mu_param(cx, curr, next);
#endif
}
EGDST_DEV double egdst_rescale(const egdst_ctx *cx, const PeriodVars *curr, const PeriodVars *next, double z) {
#if EGDST_DISTRIB == 1
    return exp(mu_param(cx, curr, next) + z * sigma_param(cx, curr, next));
#else
    return mu_param(cx, curr, next) + z * sigma_param(cx, curr, next);
#endif
}

// Newton inversion of the budget: a such that cashinhand(a)=arg (egdst_lib.c:275-296).
// Returns the number of iterations through *fail (>=100 => EGDST_ERR_CASHINVERSE).
EGDST_DEV double egdst_cashinhandinverse(const egdst_ctx *cx, const PeriodVars *curr, PeriodVars next, double arg, int *fail) {
    int cnt = 0;
    next.savings = arg;
    while (fabs(cashinhand(cx, curr, &next) - arg) > cx->zeroconsumption / 10) {
        next.savings -= (cashinhand(cx, curr, &next) - arg) / cashinhand_marginal(cx, curr, &next);
        if (++cnt >= 100) { *fail = 1; return -1.0; }
    }
    return next.savings;
}

// fill the value-coded parts of a PeriodVars (only read when byval>0, i.e. never in the solver;
// kept so that generated code that references curr->st/dc is always initialised)
EGDST_DEV void egdst_fill_state(const egdst_ctx *cx, PeriodVars *p) {
#pragma unroll
    for (int i = 0; i < EGDST_NNST; i++) p->st[i] = cx->states[i * cx->nst + p->ist];
}
EGDST_DEV void egdst_fill_decision(const egdst_ctx *cx, PeriodVars *p) {
#pragma unroll
    for (int i = 0; i < EGDST_NND; i++) p->dc[i] = cx->decisions[i * cx->nd + p->id];
}
