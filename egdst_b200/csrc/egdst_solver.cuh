// egdst_solver.cuh -- the EGM phases of one backward-induction period (all states, all decisions, all
// parameter vectors of a team at once).
//
// Restates the reference's egmbellman (egdst_solver.c:370-752) in parallel form:
//   egdst_ph_terminal   terminal-period closed-form grid                     egdst_solver.c:452-475
//   egdst_ph_seed       adraw stage 0/1 + ZEROCONSUMPTION feedback            egdst_solver.c:955-1099, 583-627
//   egdst_ph_egm        expectation over (ist1, iy) + Euler inversion         egdst_solver.c:490-665
//                       fused with the adraw stop rule, the drop rules and fold detection
//                                                                            egdst_solver.c:1100-1152, 640-664, 819
//   egdst_ph_resend     a zero-consumption re-send after the seed stage      egdst_solver.c:1080-1099
// The upper envelopes are in egdst_envelope.cuh, the period loop in egdst_period.cuh.
//
// Parallel decomposition (SURVEY 7, hard part 1): the A-grid is sequential in the reference only
// through (i) the stage-0 bisection, whose candidates mmax, (mmax+a0)/2, ... are known in advance and
// are evaluated concurrently, (ii) the a0 point and its re-sends (serial, a handful of evaluations),
// (iii) the stop rule, which is applied after all N-1 closed-form grid points were evaluated, and (iv) a
// re-send requested by a later grid point, after which the REST of the grid is a new closed form: the
// EGM phase keeps the points before it, egdst_ph_resend re-seeds, and the EGM phase runs again from there.
#pragma once

#include "egdst_tables.cuh"

// next-period tables of one state ist1
struct EgdstNext {
    const double *M, *C, *V;  // rows 0..n1 (row 0 = a0 row)
    const double *th, *dd;
    int n1, nth;              // n1 = egdims (rows excluding the a0 row)
    double evf;
    int cell;
    const EgdstRow *ivl;      // row table of the cell (egdst_tables.cuh)
    double M1, Mlast, Clast;  // M[1], M[n1], C[n1]
};

// The tables of a cell with at least two rows after row 0, without thresholds: decision cells of the smoothing mode have
// none (thlen and thTH are sized for the solution cells only).
EGDST_DEV EgdstNext egdst_cell_tables(const EgdstDev &P, int cell) {
    EgdstNext t;
    t.M = egdst_colM(P, cell);
    t.C = egdst_colC(P, cell);
    t.V = egdst_colV(P, cell);
    t.n1 = P.mlen[cell] - 1;
    t.th = 0; t.dd = 0; t.nth = 0;
    t.evf = P.evf[cell];
    t.cell = cell;
    t.ivl = egdst_cell_rows(P, cell);
    t.M1 = t.M[1]; t.Mlast = t.M[t.n1]; t.Clast = t.C[t.n1];
    return t;
}
EGDST_DEV EgdstNext egdst_next_tables(const EgdstDev &P, int ivec, int it1, int ist1) {
    EgdstNext t = egdst_cell_tables(P, egdst_cell(P, ivec, it1, ist1));
    t.th = P.thTH + (size_t)t.cell * P.cx.nthrhmax;
    t.dd = P.thD + (size_t)t.cell * P.cx.nthrhmax;
    t.nth = P.thlen[t.cell];
    return t;
}

// accumulator of one Euler evaluation (possibly a partial one: a strided subset of the nodes)
struct EgdstAcc {
    double rhs, evf, checksum;
    int badq;        // smallest flattened node index ist1*ny+iy that aborted the evaluation, or INT_MAX
    int badtype;     // EGDST_PT_C1NEG or EGDST_PT_EVFINF
    double badcash, badshock;
};
#define EGDST_NOBAD 0x7fffffff

// Quadrature shocks and node probabilities of one (it, ist, id) for every (ist1, iy): shk/shp [nst*ny].
// Valid when the model image says they cannot depend on savings (EGDST_SHOCK_INDEP_A, codegen): computed once
// per work item instead of once per node (one exp per node saved).  shp == 0 marks nodes the reference skips
// (infeasible ist1, zero transition probability, iy >= niy).
EGDST_DEV void egdst_fill_shocktab(const egdst_ctx *cx, const EgdstDev &P, const PeriodVars *curr, double *shk, double *shp, int tid, int nthreads) {
    const int ny = cx->ny, nst = cx->nst;
    for (int q = tid; q < nst * ny; q += nthreads) {
        const int ist1 = q / ny, iy = q - ist1 * ny;
        PeriodVars next;
        next.it = curr->it + 1; next.savings = 0.0; next.id = 0; next.cash = 0.0; next.shock = 0.0; next.ist = ist1;
        double p = 0.0, sh = 0.0;
        if (feasible(cx, &next) == 1) {
            const int niy = (sigma_param(cx, curr, &next) <= 0 || ny == 1) ? 1 : ny;
            if (iy < niy) {
                sh = (niy == 1) ? egdst_expectation(cx, curr, &next) : egdst_rescale(cx, curr, &next, P.qz[iy]);
                next.shock = sh;
                p = trpr(cx, curr, &next, 1);
                if (niy > 1) p *= P.qw[iy];
            }
        }
        shk[q] = sh; shp[q] = p;
    }
}

// One quadrature node of the expectation (egdst_solver.c:547-573), all cases: table-free cells, extrapolation on either
// side of the grid, the credit-constrained branch of the value function, decision-dependent marginal utility, aborts.
// Returns false when the evaluation ends at this node (acc.bad* say why).  The hot loop of egdst_eval_nodes takes the
// common cases through egdst_fast_lookup / egdst_fast_interp and calls this for the rest.
EGDST_DEV bool egdst_eval_node(const egdst_ctx *cx, const EgdstDev &P, const EgdstNext &t, bool tab, const PeriodVars *curr, PeriodVars &next,
                                    int keep, int q, double pr1, EgdstAcc &acc) {
    acc.checksum += pr1;
    next.cash = cashinhand(cx, curr, &next);
    // one bracket lookup serves consumption (rows 0..n1) and value (rows 1..n1): the second bracket of the
    // reference is max(i,1) of the first (same strictly increasing grid); rows i, i+1 come as one record
    EgdstInterval iv;
    const int i = egdst_cell_lookup(P, t.cell, tab, next.cash, t.n1 + 1, iv);
    // the reference's quotients are kept bit for bit (two divisions per interpolation, egdst_lib.c:175): next to its
    // instability boundary (SURVEY 0, fact 7) a plain reciprocal-multiply variant drifted 1e-2 away in C, so the
    // shared-reciprocal form below is the exactly rounded one (egdst_div_by)
    double w = iv.g1 - iv.g0;
    double y = iv.y;  // shared correctly rounded reciprocal RN(1/w), from the table (0: degenerate interval, plain divisions)
    double c1 = y != 0.0 ? egdst_lerp_y(next.cash, iv.g0, iv.g1, iv.c0, iv.c1, w, y) : egdst_lerp(next.cash, iv.g0, iv.g1, iv.c0, iv.c1);
    if (next.cash > t.Mlast) c1 = MAX(c1, t.Clast);  // constant extrapolation guard (egdst_solver.c:554)
    if (c1 <= 0) {
        acc.badq = q; acc.badtype = EGDST_PT_C1NEG; acc.badcash = next.cash; acc.badshock = next.shock;
        return false;
    }
    if (!EGDST_OPT_MUNOD || (!EGDST_OPT_UNOD && keep == 1 && next.cash < t.M1))
        next.id = egdst_optimd(next.cash, t.th, t.dd, t.nth);
    else
        next.id = 0;
    acc.rhs += pr1 * utility_marginal(cx, &next, c1) * cashinhand_marginal(cx, curr, &next);
    if (keep == 1) {
        double v1;
        if (next.cash < t.M1 && t.evf > -EGDST_INF) {
            v1 = utility(cx, &next, next.cash - cx->a0) + discount(cx, &next) * t.evf;  // egdst_solver.c:763
        } else {
            if (i < 1) {  // value table starts at row 1 (row 0 of V is evf(a0), not a value)
                iv = egdst_cell_interval(P, t.cell, tab, 1);
                w = iv.g1 - iv.g0;
                y = iv.y;
            }
            v1 = egdst_linter_extrap_iv(cx, &next, next.cash, iv.g0, iv.g1, iv.v0, iv.v1, t.M1, t.Mlast, w, y);
        }
        const double term = pr1 * v1;
        acc.evf += term;
        if (term == -EGDST_INF) {
            acc.badq = q; acc.badtype = EGDST_PT_EVFINF; acc.badcash = next.cash; acc.badshock = next.shock;
            return false;
        }
    }
    return true;
}

// ---- taste-shock smoothing (opt-in extension, P.sigmaEps > 0; the reference has no such mode) --------------------
// With additive extreme-value taste shocks of scale sigma on the discrete choice (DC-EGM, Iskhakov, Jorgensen, Rust and
// Schjerning 2017), next period's choice is probabilistic: the expectation uses the choice-specific policies c_d(M'),
// v_d(M') -- kept per decision in the decision cells (egdst_ph_dsave) instead of being discarded after the primary
// envelope (egdst_solver.c:720-730) -- through
//     EV(M')  = sigma * log sum_d exp(v_d(M')/sigma)          P_d(M') = exp(v_d/sigma) / sum_d' exp(v_d'/sigma)
//     rhs    += pr * sum_d P_d u'_d(c_d(M')) * dM'/dA          evf += pr * EV(M')
// As sigma -> 0 this is the hard max of the reference.  Each decision's table is read exactly as the reference reads
// the merged cell: bracket + linear interpolation of consumption with the constant-extrapolation guard, the
// credit-constrained branch below the first endogenous point, transformed extrapolation of the value above the grid.
#define EGDST_SMOOTH_MAXND 8
#if EGDST_SMOOTHING
// The choice-specific values at the cash x.cash of cell1 = (x.it, x.ist), by the rules above, with the caller's parameter
// values in cx (the solve's, or a simulation launch's).  Per decision d: c[d], v[d] consumption and value at cash (v[d]
// = -inf: not available, or no finite value), vl[d] the value at the bound of the unified grid.  avail: bit d set when
// decision d is available (its cell has at least 3 rows); above: cash lies above some decision's grid; vmax: max of v.
struct EgdstChoiceVals { double c[EGDST_SMOOTH_MAXND], v[EGDST_SMOOTH_MAXND], vl[EGDST_SMOOTH_MAXND], vmax; unsigned avail; bool above; };
EGDST_DEV void egdst_choice_values(const EgdstDev &P, const egdst_ctx *cx, int cell1, PeriodVars x, EgdstChoiceVals &cv) {
    const double cash = x.cash;
    cv.vmax = -EGDST_INF; cv.avail = 0u; cv.above = false;
    const int nm = P.mlen[cell1];
    const double g0m = nm >= 3 ? egdst_colM(P, cell1)[nm - 2] : -EGDST_INF;  // second-to-last abscissa of the merged cell
    for (int d1 = 0; d1 < cx->nd; d1++) {
        cv.v[d1] = -EGDST_INF; cv.c[d1] = 0.0; cv.vl[d1] = -EGDST_INF;
        const int dcell = egdst_dcell(P, cell1, d1);
        if (P.mlen[dcell] < 3) continue;  // decision not available in (it, ist)
        cv.avail |= 1u << d1;
        const EgdstNext t = egdst_cell_tables(P, dcell);
        cv.vl[d1] = t.V[t.n1];
        cv.above = cv.above || cash > t.Mlast;
        const bool tab = egdst_cell_has_tab(P, t.cell, t.n1 + 1);
        EgdstInterval iv;
        const int i = egdst_cell_lookup(P, t.cell, tab, cash, t.n1 + 1, iv);
        double w = iv.g1 - iv.g0, y = iv.y;
        double c1 = y != 0.0 ? egdst_lerp_y(cash, iv.g0, iv.g1, iv.c0, iv.c1, w, y) : egdst_lerp(cash, iv.g0, iv.g1, iv.c0, iv.c1);
        if (cash > t.Mlast) c1 = MAX(c1, t.Clast);
        cv.c[d1] = c1;
        x.id = d1;
        double v1;
        if (cash < t.M1 && t.evf > -EGDST_INF) {
            v1 = utility(cx, &x, cash - cx->a0) + discount(cx, &x) * t.evf;
        } else {
            if (i < 1) {
                iv = egdst_cell_interval(P, t.cell, tab, 1);
                w = iv.g1 - iv.g0; y = iv.y;
            }
            v1 = egdst_linter_extrap_iv(cx, &x, cash, iv.g0, iv.g1, iv.v0, iv.v1, t.M1, t.Mlast, w, y);
            if (cash > t.Mlast && g0m > t.M1 && g0m < t.Mlast) {
                // above the grid the value is extrapolated in the metric of the transform (egdst_lib.c:179-206), which depends on
                // the chord it continues: the reference continues the last interval of the MERGED cell, so every decision's value
                // is continued from that abscissa (g0m) -- the limit sigma -> 0 is then the reference's extrapolation exactly
                EgdstInterval jv;
                egdst_cell_lookup(P, t.cell, tab, g0m, t.n1 + 1, jv);
                const double vg = egdst_lerp(g0m, jv.g0, jv.g1, jv.v0, jv.v1);
                v1 = egdst_linter_extrap_iv(cx, &x, cash, g0m, t.Mlast, vg, t.V[t.n1], t.M1, t.Mlast, t.Mlast - g0m, 0.0);
            }
        }
        cv.v[d1] = v1;
        if (v1 > cv.vmax) cv.vmax = v1;
    }
}

// The choice probabilities P_d = e_d / ssum of the values cv: f(d, e_d) is called for every decision with a weight, in
// decision order, and ssum is the sum of the weights.  e_d = exp((w_d - wmax) / sigma), w_d = v_d, or above the unified
// grid (all choice-specific tables end at its bound, egdst_ph_dsave) the value at the bound vl_d: the probabilities are
// held at their values at the bound, because the reference holds the argmax of the bound there (it extrapolates the last
// interval of the merged cell), so this is its limit as sigma -> 0; extrapolated choice-specific values are not compared
// with each other.  False: no decision has a finite value, and every available decision weighs 1.
template <class F>
EGDST_DEV bool egdst_choice_weights(int nd, const EgdstChoiceVals &cv, double sig, double &ssum, double &wmax, F &&f) {
    wmax = cv.vmax;
    if (cv.above) { wmax = -EGDST_INF; for (int d1 = 0; d1 < nd; d1++) if (cv.v[d1] > -EGDST_INF && cv.vl[d1] > wmax) wmax = cv.vl[d1]; }
    ssum = 0.0;
    if (wmax > -EGDST_INF) {
        for (int d1 = 0; d1 < nd; d1++) {
            if (!(cv.v[d1] > -EGDST_INF)) continue;
            const double wv = cv.above ? cv.vl[d1] : cv.v[d1];
            if (!(wv > -EGDST_INF)) continue;
            const double e = exp((wv - wmax) / sig);
            ssum += e;
            f(d1, e);
        }
    }
    if (ssum > 0.0) return true;
    for (int d1 = 0; d1 < nd; d1++) if (cv.avail >> d1 & 1u) { ssum += 1.0; f(d1, 1.0); }
    return false;
}

// Out of line, with scalar arguments and the kernel-argument block read from its copy in global memory (P.self): the
// reference-parity kernels must not pay registers, local memory or instruction-cache space for this mode (a by-reference
// call would pin the caller's context structs to local memory).
struct EgdstSmoothOut { double mu, ev; int bad; };  // bad: 0, EGDST_PT_C1NEG or EGDST_PT_EVFINF
EGDST_NOINLINE EgdstSmoothOut egdst_smooth_node(const EgdstDev *Pg, int ivec, int it1, int ist1, double savings, double shock, double cash, int keep) {
    const EgdstDev &P = *Pg;
    EgdstSmoothOut o; o.mu = 0.0; o.ev = 0.0; o.bad = 0;
    egdst_ctx cxs; egdst_load_ctx(P, ivec, cxs);
    const egdst_ctx *cx = &cxs;
    PeriodVars next; next.it = it1; next.ist = ist1; next.id = 0; next.savings = savings; next.shock = shock; next.cash = cash;
    const int nd = cx->nd;
    EgdstChoiceVals cv;
    egdst_choice_values(P, cx, egdst_cell(P, ivec, it1, ist1), next, cv);
    double md[EGDST_SMOOTH_MAXND];
    for (int d1 = 0; d1 < nd; d1++) {
        md[d1] = 0.0;
        if (!(cv.avail >> d1 & 1u)) continue;
        if (cv.c[d1] <= 0) { o.bad = EGDST_PT_C1NEG; return o; }
        next.id = d1;
        md[d1] = utility_marginal(cx, &next, cv.c[d1]);
    }
    if (cv.avail == 0u || (keep == 1 && !(cv.vmax > -EGDST_INF))) { o.bad = EGDST_PT_EVFINF; return o; }  // the reference's evf = -inf abort (egdst_solver.c:596)
    double ssum, wmax, mu = 0.0, dv = 0.0;
    if (!egdst_choice_weights(nd, cv, P.sigmaEps, ssum, wmax, [&](int d1, double e) {
            mu += e * md[d1];
            if (cv.above) dv += e * (cv.v[d1] - cv.vl[d1]);
        })) {  // keep == 0 with every value at -inf
        o.mu = mu / ssum; o.ev = -EGDST_INF;
        return o;
    }
    o.mu = mu / ssum;
    o.ev = wmax + P.sigmaEps * log(ssum) + dv / ssum;
    return o;
}

#endif  // EGDST_SMOOTHING

// The common cases of a node, straight-line.  The cell has tables and either
//   (interior) cash lies inside the value grid [M[1], M[last]] (no extrapolation, no credit-constrained branch), the
//              bucket of the index resolves the bracket by itself, the interval is safely invertible, or
//   (above)    cash lies above the grid: the last interval extrapolates consumption linearly (with the constant guard of
//              egdst_solver.c:554) and the value in the metric of the transform (egdst_lib.c:179-206); everything about
//              that interval, including its image under the transform, comes with the cell (EgdstCellTop) -- no gather.
// Values must be finite.  Two nodes are prepared side by side so that their gathers and their arithmetic overlap;
// `ok` says whether the straight-line result may be used.  The operations and their order are those of the general
// path (egdst_eval_node), so the results are the same bits.
struct EgdstFastNode { double cash, c1, v1; bool ok; };
EGDST_DEV void egdst_fast_lookup(const EgdstDev &P, const EgdstNext &t, const EgdstCellTop &top, double cash, int &i, bool &ok) {
    if (cash > top.g1) { i = -1; ok = top.y != 0.0 && top.yt != 0.0 && cash > P.cx.a0; return; }
    i = egdst_lut_rank(P, t.cell, t.M, cash);
    ok = i >= 1 && i <= t.n1 - 1;  // rows i, i+1 exist and belong to the value grid (no clamp: others take the general path)
}
EGDST_DEV void egdst_fast_interp(const egdst_ctx *cx, const PeriodVars *next, const EgdstNext &t, const EgdstCellTop &top, int i, double cash, EgdstFastNode &f) {
    const double big = 1e290;
    if (i < 0) {  // above the grid
        const double w = top.g1 - top.g0, y = top.y;
        const double ac1 = top.c1 * (cash - top.g0), ac0 = top.c0 * (top.g1 - cash);
        const double tx = tr(cx, next, cash - cx->a0);
        const double wt = top.t1 - top.t0;
        const double av1 = top.v1 * (tx - top.t0), av0 = top.v0 * (top.t1 - tx);
        f.ok = f.ok && fabs(ac1) < big && fabs(ac0) < big && fabs(av1) < big && fabs(av0) < big && fabs(top.v0) < big && fabs(top.v1) < big;
        const double c = egdst_div_by(ac1, w, y) + egdst_div_by(ac0, w, y);
        f.c1 = MAX(c, top.c1);
        f.v1 = egdst_div_by(av1, wt, top.yt) + egdst_div_by(av0, wt, top.yt);
        return;
    }
    const EgdstInterval iv = egdst_load_interval(t.ivl + i);
    const double w = iv.g1 - iv.g0, y = iv.y;
    const double xl = cash - iv.g0, xr = iv.g1 - cash;
    const double ac1 = iv.c1 * xl, ac0 = iv.c0 * xr, av1 = iv.v1 * xl, av0 = iv.v0 * xr;
    f.ok = f.ok && y != 0.0 && cash >= iv.g0 && cash <= iv.g1 && fabs(ac1) < big && fabs(ac0) < big && fabs(av1) < big && fabs(av0) < big;
    f.c1 = egdst_div_by(ac1, w, y) + egdst_div_by(ac0, w, y);
    f.v1 = egdst_div_by(av1, w, y) + egdst_div_by(av0, w, y);
}

// Evaluate nodes iy = part, part+nparts, ... (of every ist1) of the expectation at end-of-period savings A
// (egdst_solver.c:494-574).  keep==0 skips the value function (adraw seed phase).  The optim_* switches are
// constants of the model image (EGDST_OPT_*).  Nodes are taken in ascending order; with a shock table (shk/shp) and
// keep==1 -- the EGM phase -- two nodes at a time go through the straight-line path when both qualify.
EGDST_DEV void egdst_eval_nodes(const egdst_ctx *cx, const EgdstDev &P, int ivec, const PeriodVars *curr, double A, int keep,
                                int part, int nparts, EgdstAcc &acc, const double *shk = 0, const double *shp = 0) {
    const int ny = cx->ny, nst = cx->nst;
    acc.rhs = 0.0; acc.evf = 0.0; acc.checksum = 0.0; acc.badq = EGDST_NOBAD; acc.badtype = 0; acc.badcash = 0.0; acc.badshock = 0.0;
    PeriodVars next;
    next.it = curr->it + 1;
    next.savings = A;
    next.id = 0;
    next.cash = 0.0;
    next.shock = 0.0;
    for (int ist1 = 0; ist1 < nst; ist1++) {
        next.ist = ist1;
        if (feasible(cx, &next) != 1) continue;
        double pr1pre = 0.0;
        int niy = ny;
        if (!shk) {
#if EGDST_OPT_TRPRNOSH
            pr1pre = trpr(cx, curr, &next, 1);
            if (pr1pre == 0.0) continue;
#endif
            niy = (sigma_param(cx, curr, &next) <= 0 || ny == 1) ? 1 : ny;
        }
        const EgdstNext t = egdst_next_tables(P, ivec, next.it, ist1);
        const bool tab = egdst_cell_has_tab(P, t.cell, t.n1 + 1);
        int iy = part;
#if EGDST_OPT_MUNOD
        if (!EGDST_SMOOTHING && shk && tab && keep == 1 && t.n1 >= 3) {
            const EgdstCellTop top = P.tabTop[t.cell];
            for (; iy + nparts < niy; iy += 2 * nparts) {
                const int qa = ist1 * ny + iy, qb = qa + nparts;
                if (qa > acc.badq) break;
                const double pa = shp[qa], pb = shp[qb], sa = shk[qa], sb = shk[qb];
                EgdstFastNode fa, fb;
                next.shock = sa; fa.cash = cashinhand(cx, curr, &next);
                next.shock = sb; fb.cash = cashinhand(cx, curr, &next);
                int ia, ib;
                egdst_fast_lookup(P, t, top, fa.cash, ia, fa.ok);
                egdst_fast_lookup(P, t, top, fb.cash, ib, fb.ok);
                fa.ok = fa.ok && pa != 0.0; fb.ok = fb.ok && pb != 0.0;
                if (fa.ok && fb.ok) {
                    next.id = 0;
                    next.shock = sa; next.cash = fa.cash; egdst_fast_interp(cx, &next, t, top, ia, fa.cash, fa);
                    next.shock = sb; next.cash = fb.cash; egdst_fast_interp(cx, &next, t, top, ib, fb.cash, fb);
                }
                if (fa.ok && fb.ok && fa.c1 > 0 && fb.c1 > 0) {
                    // same operations in the same order as the general path, node qa then node qb
                    next.id = 0;
                    next.shock = sa; next.cash = fa.cash;
                    acc.checksum += pa;
                    acc.rhs += pa * utility_marginal(cx, &next, fa.c1) * cashinhand_marginal(cx, curr, &next);
                    acc.evf += pa * fa.v1;
                    next.shock = sb; next.cash = fb.cash;
                    acc.checksum += pb;
                    acc.rhs += pb * utility_marginal(cx, &next, fb.c1) * cashinhand_marginal(cx, curr, &next);
                    acc.evf += pb * fb.v1;
                    continue;
                }
                // general path, one node after the other
                if (pa != 0.0) { next.shock = sa; if (!egdst_eval_node(cx, P, t, tab, curr, next, keep, qa, pa, acc)) break; }
                if (pb != 0.0) {
                    if (qb > acc.badq) break;
                    next.shock = sb; if (!egdst_eval_node(cx, P, t, tab, curr, next, keep, qb, pb, acc)) break;
                }
            }
            if (acc.badq != EGDST_NOBAD) continue;  // the evaluation ended in (or before) this state: nothing is left for this slice
        }
#endif
        for (; iy < niy; iy += nparts) {
            double pr1;
            if (shk) {
                pr1 = shp[ist1 * ny + iy];
                next.shock = shk[ist1 * ny + iy];
            } else if (niy == 1) {
                next.shock = egdst_expectation(cx, curr, &next);
                pr1 = EGDST_OPT_TRPRNOSH ? pr1pre : trpr(cx, curr, &next, 1);
            } else {
                next.shock = egdst_rescale(cx, curr, &next, P.qz[iy]);
                pr1 = EGDST_OPT_TRPRNOSH ? pr1pre : trpr(cx, curr, &next, 1);
                pr1 *= P.qw[iy];
            }
            if (pr1 == 0.0) continue;
            const int q = ist1 * ny + iy;
            if (q > acc.badq) break;  // the reference would have stopped before this node
#if EGDST_SMOOTHING
            {  // taste-shock smoothing (extension): logsum and choice probabilities over the choice-specific tables
                acc.checksum += pr1;
                next.cash = cashinhand(cx, curr, &next);
                const EgdstSmoothOut o = egdst_smooth_node(P.self, ivec, next.it, ist1, next.savings, next.shock, next.cash, keep);
                if (o.bad) { acc.badq = q; acc.badtype = o.bad; acc.badcash = next.cash; acc.badshock = next.shock; break; }
                acc.rhs += pr1 * o.mu * cashinhand_marginal(cx, curr, &next);
                if (keep == 1) {
                    const double term = pr1 * o.ev;
                    acc.evf += term;
                    if (term == -EGDST_INF) { acc.badq = q; acc.badtype = EGDST_PT_EVFINF; acc.badcash = next.cash; acc.badshock = next.shock; break; }
                }
                continue;
            }
#endif
            if (!egdst_eval_node(cx, P, t, tab, curr, next, keep, q, pr1, acc)) break;
        }
    }
}

// combine partial accumulators across a warp; every lane ends with the full result
EGDST_DEV void egdst_warp_combine(EgdstAcc &a) {
    const int minq = __shfl_sync(EGDST_FULL, egdst_warp_min(a.badq), 0);
    const unsigned owner = __ballot_sync(EGDST_FULL, a.badq == minq && minq != EGDST_NOBAD);
    a.rhs = __shfl_sync(EGDST_FULL, egdst_warp_sum(a.rhs), 0);
    a.evf = __shfl_sync(EGDST_FULL, egdst_warp_sum(a.evf), 0);
    a.checksum = __shfl_sync(EGDST_FULL, egdst_warp_sum(a.checksum), 0);
    if (minq != EGDST_NOBAD) {
        const int src = __ffs(owner) - 1;
        a.badtype = __shfl_sync(EGDST_FULL, a.badtype, src);
        a.badcash = __shfl_sync(EGDST_FULL, a.badcash, src);
        a.badshock = __shfl_sync(EGDST_FULL, a.badshock, src);
    }
    a.badq = minq;
}

// ---------------------------------------------------------------------------------------------
// terminal period: M_i = trinv(m1 + i (m2-m1)/(N-1)), C = M, V = u(C); evfa0 = -inf   (END2, A0T = 0)
// ---------------------------------------------------------------------------------------------
EGDST_DEV void egdst_ph_terminal(const EgdstDev &P, int it, const EgdstTeam &T) {
    const int B = blockDim.x, nxb = (P.N + B - 1) / B, jpv = P.cx.nst * P.cx.nd;
    const int nwork = T.nv * jpv * nxb;
    for (int w = T.rank; w < nwork; w += T.size) {
        int ivec, jy, xb;
        egdst_item(T, w, jpv, ivec, jy, xb);
        const int ist = jy / P.cx.nd, id = jy % P.cx.nd;
        egdst_ctx cx; egdst_load_ctx(P, ivec, cx);
        const int sd = egdst_sd(P, ivec, ist, id);
        PeriodVars curr; curr.it = it; curr.ist = ist; curr.id = id; curr.cash = 0; curr.savings = 0; curr.shock = 0;
        const int act = (feasible(&cx, &curr) == 1) && (inchoiceset(&cx, &curr) == 1);
        const int i = xb * B + threadIdx.x;
        if (i == 0) {
            P.active[sd] = act;
            P.evfa0[sd] = -EGDST_INF;
            P.ptN[sd] = act ? P.N : 0;
            P.nfold[sd] = 0;
            if (act) atomicAdd(P.units + ivec, (unsigned long long)P.N);
        }
        if (!act || i >= P.N) continue;
        const double m1 = tr(&cx, &curr, cx.zeroconsumption - 0.0), m2 = tr(&cx, &curr, cx.mmax - 0.0);
        const double m = trinv(&cx, &curr, m1 + i * (m2 - m1) / (P.N - 1)) + 0.0;
        const double c = m - 0.0;
        P.ptX[(size_t)sd * P.gcap + i] = m;
        P.ptC[(size_t)sd * P.gcap + i] = c;
        P.ptV[(size_t)sd * P.gcap + i] = utility(&cx, &curr, c);
    }
}

// ---------------------------------------------------------------------------------------------
// seed: one CTA per (ist,id,ivec).  Warps evaluate the stage-0 candidates concurrently; the whole CTA
// evaluates A=a0 and any re-sent point; thread 0 runs the adraw state machine.
// ---------------------------------------------------------------------------------------------
struct EgdstSeedShared {
    double candA[EGDST_MAXCAND], candM[EGDST_MAXCAND];
    int candBad[EGDST_MAXCAND];
    double wr[32], we[32], wc[32], wcash[32], wshock[32];
    int wq[32], wt[32];
    double A, rhs, evf, checksum, badcash, badshock;
    int ncand, badq, badtype, go, calls;
};

EGDST_DEV void egdst_block_eval(const egdst_ctx *cx, const EgdstDev &P, int ivec, const PeriodVars *curr, double A, int keep,
                                EgdstSeedShared &S, const double *shk, const double *shp) {
    EgdstAcc a;
#ifdef EGDST_HOSTEMU
    // diagnostic of the host emulator (EGDST_SEED_SERIAL=1): thread 0 sums all nodes in the reference's order.  The
    // partitioned sum below differs from the reference's sequential one in the last bit now and then; on degenerate models
    // that bit decides a run split periods later (DESIGN.md section 5.1).
    static const bool serial = getenv("EGDST_SEED_SERIAL") && atoi(getenv("EGDST_SEED_SERIAL")) != 0;
    if (serial) {
        if (threadIdx.x == 0) egdst_eval_nodes(cx, P, ivec, curr, A, keep, 0, 1, a, shk, shp);
        else { a.rhs = 0; a.evf = 0; a.checksum = 0; a.badq = EGDST_NOBAD; a.badtype = 0; a.badcash = 0; a.badshock = 0; }
    } else
#endif
    egdst_eval_nodes(cx, P, ivec, curr, A, keep, threadIdx.x, blockDim.x, a, shk, shp);
    egdst_warp_combine(a);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    if (lane == 0) { S.wr[w] = a.rhs; S.we[w] = a.evf; S.wc[w] = a.checksum; S.wq[w] = a.badq; S.wt[w] = a.badtype; S.wcash[w] = a.badcash; S.wshock[w] = a.badshock; }
    egdst_cta_sync();
    if (threadIdx.x == 0) {
        double r = 0, e = 0, c = 0; int bq = EGDST_NOBAD, bw = 0;
        for (int k = 0; k < nw; k++) { r += S.wr[k]; e += S.we[k]; c += S.wc[k]; if (S.wq[k] < bq) { bq = S.wq[k]; bw = k; } }
        S.rhs = r; S.evf = e; S.checksum = c; S.badq = bq; S.badtype = S.wt[bw]; S.badcash = S.wcash[bw]; S.badshock = S.wshock[bw];
    }
    egdst_cta_sync();
}

// adraw limits from the line through the base point and (A, M) (egdst_solver.c:1032-1076), or, after a zero-consumption
// re-send, through the base point and (a0, a0) with the re-sent point as the new focal point (:1080-1099)
struct EgdstLims { double lim1, lim2, lim3, lim2p, lim3p, k3; };
EGDST_DEV void egdst_lims_first(const egdst_ctx *cx, const PeriodVars *curr, double aM, double lastA, double baseA, double baseM, int N, EgdstLims &L) {
    const double aa = (aM - baseM) / (lastA - baseA), bb = baseM - aa * baseA;
    L.lim2p = MIN(cx->mmax, (cx->mmax - bb) / aa);
    L.lim3p = -bb / aa;
    if (cx->a0 < 0 && cx->a0 < L.lim3p) L.k3 = MAX(floor(N * (L.lim3p - cx->a0) / (L.lim2p - cx->a0)), 2.0);
    else { L.lim3p = cx->a0; L.k3 = 1.0; }
    L.lim1 = tr(cx, curr, L.lim3p - cx->a0); L.lim2 = tr(cx, curr, L.lim2p - L.lim3p); L.lim3 = tr(cx, curr, 0);
}
EGDST_DEV void egdst_lims_resend(const egdst_ctx *cx, const PeriodVars *curr, double lastA, double baseA, double baseM, EgdstLims &L) {
    const double aa = (cx->a0 - baseM) / (cx->a0 - baseA), bb = baseM - aa * baseA;
    L.lim2p = MIN(cx->mmax, (cx->mmax - bb) / aa);
    L.lim3p = lastA - cx->zeroconsumption;
    L.k3 = 1.0;
    L.lim1 = tr(cx, curr, L.lim3p - cx->a0); L.lim2 = tr(cx, curr, L.lim2p - L.lim3p); L.lim3 = tr(cx, curr, 0);
}
// the savings point that replaces one whose evaluation met c1<=0 at node (ist1, shock) (egdst_solver.c:600-616)
EGDST_DEV double egdst_resend_point(const egdst_ctx *cx, const EgdstDev &P, int ivec, const PeriodVars *curr, int it, double lastA,
                                    int badq, double badshock, double badcash, int *fail) {
    PeriodVars next; next.it = it + 1; next.ist = badq / cx->ny; next.id = 0; next.savings = lastA; next.shock = badshock; next.cash = badcash;
    const EgdstNext t = egdst_next_tables(P, ivec, it + 1, next.ist);
    const double target = (t.evf > -EGDST_INF) ? cx->a0 : t.M[1];
    return egdst_cashinhandinverse(cx, curr, next, target, fail) + cx->zeroconsumption;
}

// publish the state of a (re)seeded savings grid: slot 0 of the job's chained scan holds the inclusive prefix the
// EGM items start from -- points kept so far, and "the grid stopped" (egdst_solver.c:1100)
EGDST_DEV void egdst_seed_publish(const EgdstDev &P, int sd, double *seed, const EgdstLims &L, double lastA, int nfirst, int calls,
                                  double baseA, double baseM, int kept, int stop, int pass) {
    seed[0] = L.lim1; seed[1] = L.lim2; seed[2] = L.lim3; seed[3] = L.lim3p; seed[4] = L.k3; seed[5] = lastA;
    seed[6] = (double)nfirst; seed[7] = (double)calls; seed[8] = baseA; seed[9] = baseM; seed[10] = (double)pass;
    P.scanC[(size_t)sd * P.chC] = EGDST_SCAN_INC | egdst_scan_pack(kept, stop);
}

// The adraw loop from savings point S.A on (egdst_solver.c:1032-1099), serial in A, parallel over nodes: the CTA
// evaluates the point; thread 0 classifies it, replaces a point whose consumption vanished by its zero-consumption re-send
// (egdst_resend_point), stores a point with a finite M as row `slot` of the grid (if slot < P.gcap), and goes on while
// the point asks for a re-send.  On return S.go is 0 (done) or -1 (failed), and thread 0 holds the last point, its M,
// evf(a0) (-inf after an abort) and the limits L of the closed-form grid after it (the first ones when L.k3 == 0).
struct EgdstAdraw { double lastA, aM, evfa0; int stored, storedAny; };  // stored: by the last evaluation / by any
EGDST_DEV EgdstAdraw egdst_adraw(const egdst_ctx *cx, const EgdstDev &P, int it, int ivec, int ist, int id, const PeriodVars *curr, double beta,
                                 int slot, double baseA, double baseM, EgdstLims &L, EgdstSeedShared &S, const double *shk, const double *shp) {
    const size_t row = (size_t)egdst_sd(P, ivec, ist, id) * P.gcap + slot;
    EgdstAdraw r; r.lastA = cx->a0; r.aM = 0; r.evfa0 = 0.0; r.stored = 0; r.storedAny = 0;
    while (true) {
        egdst_block_eval(cx, P, ivec, curr, S.A, 1, S, shk, shp);
        if (threadIdx.x == 0) {
            r.lastA = S.A;
            r.stored = 0;
            int resend = 0, fatal = 0;
            if (S.badq == EGDST_NOBAD && fabs(S.checksum - 1) > cx->tolerance) {
                egdst_fail(P, ivec, EGDST_ERR_CHECKSUM, it, ist, id); fatal = 1;
            } else if (S.badq != EGDST_NOBAD) {
                r.evfa0 = -EGDST_INF;
                r.aM = S.badcash;
                if (S.badtype == EGDST_PT_C1NEG) {
                    r.aM = cx->a0 - 1;
                    int fail = 0;
                    r.lastA = egdst_resend_point(cx, P, ivec, curr, it, r.lastA, S.badq, S.badshock, S.badcash, &fail);
                    if (fail) { egdst_fail(P, ivec, EGDST_ERR_CASHINVERSE, it, ist, id); fatal = 1; }
                }
            } else {
                r.aM = r.lastA + utility_marginal_inverse(cx, curr, beta * S.rhs);
                if (isfinite(r.aM)) {
                    if (fabs(r.lastA - cx->a0) < cx->tolerance && r.evfa0 > -EGDST_INF) r.evfa0 = S.evf;
                    if (slot < P.gcap) {
                        P.ptX[row] = r.aM; P.ptC[row] = r.aM - r.lastA; P.ptV[row] = utility(cx, curr, r.aM - r.lastA) + beta * S.evf;
                        r.stored = 1; r.storedAny = 1;
                    }
                }
            }
            if (!fatal) {
                // adraw, ngenerated==1 branch (egdst_solver.c:1032-1099)
                if (L.k3 == 0) egdst_lims_first(cx, curr, r.aM, r.lastA, baseA, baseM, P.N, L);
                if (r.aM <= cx->a0 - 1 + cx->tolerance) {
                    egdst_lims_resend(cx, curr, r.lastA, baseA, baseM, L);
                    resend = 1;
                    if (++S.calls >= cx->ngridmax) { egdst_fail(P, ivec, EGDST_ERR_ADRAW_LOOP, it, ist, id); resend = 0; fatal = 1; }
                }
            }
            S.A = r.lastA;
            S.go = fatal ? -1 : resend;
        }
        egdst_cta_sync();
        if (S.go != 1) return r;
    }
}

EGDST_DEV void egdst_seed_job(const EgdstDev &P, int it, int ivec, int ist, int id, EgdstSeedShared &S, double *shsm, int useTab) {
    egdst_ctx cx; egdst_load_ctx(P, ivec, cx);
    const int sd = egdst_sd(P, ivec, ist, id);
    PeriodVars curr; curr.it = it; curr.ist = ist; curr.id = id; curr.cash = 0; curr.savings = 0; curr.shock = 0;
    const int act = (feasible(&cx, &curr) == 1) && (inchoiceset(&cx, &curr) == 1);
    double *seed = P.seed + (size_t)sd * EGDST_SEEDW;
    egdst_cta_sync();  // S and the shock table of the previous job are free
    if (threadIdx.x == 0) {
        P.active[sd] = act;
        P.evfa0[sd] = 0.0;
        P.ptN[sd] = 0;
        P.nfold[sd] = 0;
        P.lateN[sd] = 0x7fffffff;
        P.scanC[(size_t)sd * P.chC] = EGDST_SCAN_INC | egdst_scan_pack(0, 1);  // "stopped, no points" unless the seed succeeds
        seed[6] = 1.0; seed[7] = 0.0; seed[10] = 0.0;
        // stage-0 candidates (egdst_solver.c:979-1027): mmax, then halfway to a0 until A-a0<TOLERANCE
        int n = 0; double A = cx.mmax;
        while (n < EGDST_MAXCAND) { S.candA[n++] = A; if (A - cx.a0 < cx.tolerance) break; A = (A + cx.a0) / 2; }
        S.ncand = n;
        S.go = 0;
    }
    egdst_cta_sync();
    if (!act) return;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const double beta = discount(&cx, &curr);
    const double *shk = 0, *shp = 0;
    if (useTab) {  // shocks and node probabilities of this (it, ist, id), once per CTA
        egdst_fill_shocktab(&cx, P, &curr, shsm, shsm + cx.nst * cx.ny, threadIdx.x, blockDim.x);
        shk = shsm; shp = shsm + cx.nst * cx.ny;
        egdst_cta_sync();
    }
    // stage 0 in waves of one candidate per warp: the base point is almost always among the first few
    // candidates (mmax, (mmax+a0)/2, ...), so later waves rarely run
    double baseA = 0, baseM = 0;
    for (int k0 = 0; k0 < S.ncand; k0 += nw) {
        const int kk = k0 + w;
        if (kk < S.ncand) {
            EgdstAcc a;
            egdst_eval_nodes(&cx, P, ivec, &curr, S.candA[kk], 0, lane, 32, a, shk, shp);
            egdst_warp_combine(a);
            if (lane == 0) {
                int bad = 0;
                if (a.badq != EGDST_NOBAD) bad = EGDST_PT_C1NEG;
                else if (fabs(a.checksum - 1) > cx.tolerance) bad = EGDST_PT_CHECKSUM;
                S.candBad[kk] = bad;
                S.candM[kk] = S.candA[kk] + utility_marginal_inverse(&cx, &curr, beta * a.rhs);
            }
        }
        egdst_cta_sync();
        // thread 0: first candidate with M<=mmax is the base point (sequential semantics of adraw stage 0)
        if (threadIdx.x == 0) {
            const int kend = k0 + nw < S.ncand ? k0 + nw : S.ncand;
            for (int k = k0; k < kend; k++) {
                if (S.candBad[k] == EGDST_PT_C1NEG) { egdst_fail(P, ivec, EGDST_ERR_NOSAVINGS, it, ist, id); S.go = -1; break; }
                if (S.candBad[k] == EGDST_PT_CHECKSUM) { egdst_fail(P, ivec, EGDST_ERR_CHECKSUM, it, ist, id); S.go = -1; break; }
                if (S.candM[k] <= cx.mmax) { baseA = S.candA[k]; baseM = S.candM[k]; S.go = 1; S.calls = k + 2; break; }  // adraw calls so far: k+1 guesses + the call that returns a0
                if (S.candA[k] - cx.a0 < cx.tolerance) { egdst_fail(P, ivec, EGDST_ERR_ADRAW_INIT, it, ist, id); S.go = -1; break; }
            }
            if (kend == S.ncand && S.go == 0) { egdst_fail(P, ivec, EGDST_ERR_ADRAW_INIT, it, ist, id); S.go = -1; }
            S.A = cx.a0;
        }
        egdst_cta_sync();
        if (S.go != 0) break;
    }
    if (S.go != 1) return;
    // stage 1 (+ re-sends): the point a0 becomes row 0 of the grid
    EgdstLims L; L.lim1 = 0; L.lim2 = 0; L.lim3 = 0; L.lim2p = 0; L.lim3p = 0; L.k3 = 0;
    const EgdstAdraw r = egdst_adraw(&cx, P, it, ivec, ist, id, &curr, beta, 0, baseA, baseM, L, S, shk, shp);
    if (threadIdx.x == 0) {
        P.evfa0[sd] = r.evfa0;
        if (S.go == 0) {
            egdst_seed_publish(P, sd, seed, L, r.lastA, 1, S.calls, baseA, baseM, r.storedAny, (r.aM < cx.mmax) ? 0 : 1, 0);
            if (r.storedAny) atomicAdd(P.units + ivec, 1ULL);
        }
    }
}

EGDST_DEV int egdst_use_shocktab(const EgdstDev &P) {
    return (EGDST_SHOCK_INDEP_A && (size_t)2 * P.cx.nst * P.cx.ny * sizeof(double) <= EGDST_SHOCKTAB_BYTES) ? 1 : 0;
}

EGDST_DEV void egdst_ph_seed(const EgdstDev &P, int it, const EgdstTeam &T, void *scratch, double *shsm) {
    EgdstSeedShared &S = *reinterpret_cast<EgdstSeedShared *>(scratch);
    const int jpv = P.cx.nst * P.cx.nd, nwork = T.nv * jpv;
    const int useTab = egdst_use_shocktab(P);
    for (int w = T.rank; w < nwork; w += T.size) {
        const int ivec = T.v0 + w / jpv, jy = w % jpv;
        egdst_seed_job(P, it, ivec, jy / P.cx.nd, jy % P.cx.nd, S, shsm, useTab);
    }
}

// closed-form A-grid after the seed (egdst_solver.c:1104-1136); n = nfirst..N-1
EGDST_DEV double egdst_agrid_target(const egdst_ctx *cx, const PeriodVars *curr, const double *seed, int n, int N) {
    const double lim1 = seed[0], lim2 = seed[1], lim3 = seed[2], lim3p = seed[3], k3 = seed[4];
    if (n < (int)k3 - 1) return -trinv(cx, curr, lim3 + (k3 - 1 - n) * (lim1 - lim3) / (k3 - 1)) + lim3p;
    return trinv(cx, curr, lim3 + (n - k3 + 1) * (lim2 - lim3) / (N - k3)) + lim3p;
}
EGDST_DEV double egdst_agrid(const egdst_ctx *cx, const PeriodVars *curr, const double *seed, int n, int N) {
    const double t = egdst_agrid_target(cx, curr, seed, n, N);
    const double prev = (n == (int)seed[6]) ? seed[5] : egdst_agrid_target(cx, curr, seed, n - 1, N);
    return (t - prev < 0) ? prev + 1e-5 : t;  // astep<0 rule (egdst_solver.c:1120-1133)
}

// ---------------------------------------------------------------------------------------------
// EGM step for grid points n = nfirst..N-1 of every (ist, id): expectation, Euler inversion, and -- in the same
// work item -- the stop rule, the drop rules and the compaction into the decision's point list.
//
// A work item is a run of P.egmP consecutive grid points of one (ist, id); thread t handles point t % egmP and the
// quadrature nodes t / egmP, t / egmP + slices, ... (slices = threads / egmP): the threads of a warp are consecutive
// A points (their next-period cash values are neighbours, so the table gathers of a warp stay coherent), the slices
// combine through shared memory in a fixed order.  The host sizes egmP so that the items of one period fill the
// team exactly once (no tail wave).
//
// The reference generates point n only while every earlier returned M was < mmax (egdst_solver.c:1100) and no
// earlier point asked for a zero-consumption re-send (:1080); stored points are those with a finite M and no abort
// (:640-664).  The items of one (ist, id) are chained by a decoupled look-back scan whose state carries (points kept
// so far, "the grid ended here"); slot 0 of the chain is the seed's own contribution.  Folds (M or V decreasing,
// :819) inside an item's output are appended to an unordered list; the last item to finish adds the folds on item
// boundaries, orders the list and publishes the counts.
// ---------------------------------------------------------------------------------------------
template <int BS>
struct EgdstEgmShared {
    double rhs[BS], evf[BS], chk[BS], cash[BS];
    int q[BS], t[BS];
    double kx[BS], kv[BS];  // kept points of the item in output order (fold test between neighbours)
    int sh[40];
    int evmin[2];                              // first point of the item that stops the grid / asks for a re-send
    int last;
    unsigned long long excl;
};

// The runs of the point list of sd (n points, nf folds at the positions in its fold list, unordered): runStart = 0, the
// fold positions in ascending order, n; and the counts.  All threads of the CTA; the list may have been written by other
// CTAs, so it is read past L1.
EGDST_DEV void egdst_fold_runs(const EgdstDev &P, int sd, int nf, int n) {
    const int *foldList = P.foldList + (size_t)sd * (P.gcap + 1);
    int *runStart = P.runStart + (size_t)sd * (P.gcap + 1);
    for (int i = threadIdx.x; i < nf; i += blockDim.x) {  // rank sort (folds are rare)
        const int v = EGDST_LDCG(foldList + i);
        int r = 0;
        for (int j = 0; j < nf; j++) r += EGDST_LDCG(foldList + j) < v ? 1 : 0;
        runStart[r + 1] = v;
    }
    if (threadIdx.x == 0) {
        runStart[0] = 0;
        runStart[nf + 1] = n;
        P.ptN[sd] = n;
        P.nfold[sd] = nf;
    }
}

EGDST_DEV void egdst_egm_epilogue(const EgdstDev &P, int it, int ivec, int ist, int id, int sd, int nitems, int slot) {
    // last item of this (ist,id): folds on item boundaries, ordering of the fold list, counts
    const volatile unsigned long long *st = P.scanC + (size_t)sd * P.chC;
    const double *X = P.ptX + (size_t)sd * P.gcap, *V = P.ptV + (size_t)sd * P.gcap;
    int *foldList = P.foldList + (size_t)sd * (P.gcap + 1);
    const unsigned long long tot = egdst_scan_inclusive(st, nitems);
    const int kept = egdst_scan_lo(tot);
    const int nvd = kept < P.gcap ? kept : P.gcap;
    for (int c = threadIdx.x; c < nitems; c += blockDim.x) {
        const unsigned long long pe = egdst_scan_inclusive(st, c), pi = egdst_scan_inclusive(st, c + 1);  // before / after item c
        const int p = egdst_scan_lo(pe);
        if (!egdst_scan_hi(pe) && egdst_scan_lo(pi) > p && p > 0 && p < nvd)
            if (EGDST_LDCG(X + p - 1) > EGDST_LDCG(X + p) || EGDST_LDCG(V + p - 1) > EGDST_LDCG(V + p)) {
                const int k = atomicAdd(P.foldCnt + sd, 1); if (k <= P.gcap) foldList[k] = p;
            }
    }
    egdst_cta_sync();
    int nf = *((volatile int *)(P.foldCnt + sd));
    if (nf > P.gcap - 1) nf = P.gcap - 1;
    egdst_fold_runs(P, sd, nf, nvd);
    if (threadIdx.x == 0) {
        if (kept >= P.cx.ngridmax) egdst_fail(P, ivec, EGDST_ERR_GRIDSPACE, it, ist, id);
        if (nf > 0) atomicAdd(P.flags + 8 * slot + 3, 1);  // the period needs the secondary envelope
    }
}

template <int BS>
EGDST_DEV void egdst_ph_egm(const EgdstDev &P, int it, const EgdstTeam &T, int pass, void *scratch, double *shsm) {
    EgdstEgmShared<BS> &E = *reinterpret_cast<EgdstEgmShared<BS> *>(scratch);
    const int N = P.N, B = blockDim.x, Pp = P.egmP, nsl = B / Pp;
    const int jpv = P.cx.nst * P.cx.nd;
    const int nitems = (N - 1 + Pp - 1) / Pp;  // items per (ist,id): the grid points 1..N-1 (a re-seeded pass covers fewer)
    const int nwork = T.nv * jpv * nitems;
    const int useTab = egdst_use_shocktab(P);
    const int p = threadIdx.x % Pp, s = threadIdx.x / Pp;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned ltmask = (1u << lane) - 1u;
    int tabsd = -1;  // (ist,id,ivec) whose shock table is in shared memory
    for (int w = T.rank; w < nwork; w += T.size) {
        int ivec, jy, item;
        egdst_item(T, w, jpv, ivec, jy, item);
        const int ist = jy / P.cx.nd, id = jy % P.cx.nd;
        const int sd = egdst_sd(P, ivec, ist, id);
        if (!P.active[sd]) continue;  // uniform per CTA
        const double *seed = P.seed + (size_t)sd * EGDST_SEEDW;
        volatile unsigned long long *st = P.scanC + (size_t)sd * P.chC;
        // a pass after a re-send covers only the grids that were re-seeded for it (the others are complete)
        if ((int)seed[10] != pass) continue;
        const int nfirst = (int)seed[6];
        const int n = nfirst + item * Pp + p;
        if (nfirst + item * Pp >= N || egdst_scan_hi(egdst_scan_inclusive(st, 0))) {
            // nothing to evaluate (the grid ended at its seed, or a re-seeded pass starts beyond this item): the item
            // still takes part in the chain and in the completion count
            egdst_cta_sync();
            if (warp == 0) { int err = 0; egdst_lookback<1>(st, item + 1, egdst_scan_pack(0, 0), &err); }
            __threadfence();
            egdst_cta_sync();
            if (threadIdx.x == 0) E.last = (atomicAdd(P.tickC + 2 * sd + 1, 1) == nitems - 1);
            egdst_cta_sync();
            if (E.last) { __threadfence(); egdst_egm_epilogue(P, it, ivec, ist, id, sd, nitems, T.slot); }
            continue;
        }
        egdst_ctx cx; egdst_load_ctx(P, ivec, cx);
        PeriodVars curr; curr.it = it; curr.ist = ist; curr.id = id; curr.cash = 0; curr.savings = 0; curr.shock = 0;
        const double *shk = 0, *shp = 0;
        egdst_cta_sync();  // the previous item's shared scratch is free
        if (useTab) {  // shocks and node probabilities of this (it, ist, id), once per run of items of the same job
            if (tabsd != sd) {
                egdst_fill_shocktab(&cx, P, &curr, shsm, shsm + cx.nst * cx.ny, threadIdx.x, B);
                tabsd = sd;
            }
            shk = shsm; shp = shsm + cx.nst * cx.ny;
        }
        if (threadIdx.x == 0) { E.evmin[0] = 0x7fffffff; E.evmin[1] = 0x7fffffff; }
        egdst_cta_sync();
        // the loop guard of adraw (egdst_solver.c:963-978): the call that would return point n is call seed[7]+n
        const bool valid = s < nsl && n < N && (int)seed[7] + n < cx.ngridmax;
        double A = 0.0;
        EgdstAcc a; a.rhs = 0; a.evf = 0; a.checksum = 0; a.badq = EGDST_NOBAD; a.badtype = 0; a.badcash = 0; a.badshock = 0;
        if (valid) {
            A = egdst_agrid(&cx, &curr, seed, n, N);
            egdst_eval_nodes(&cx, P, ivec, &curr, A, 1, s, nsl, a, shk, shp);
        }
        E.rhs[threadIdx.x] = a.rhs; E.evf[threadIdx.x] = a.evf; E.chk[threadIdx.x] = a.checksum;
        E.q[threadIdx.x] = a.badq; E.t[threadIdx.x] = a.badtype; E.cash[threadIdx.x] = a.badcash;
        egdst_cta_sync();
        // threads 0..Pp-1 own the points of the item, in order
        int flag = EGDST_PT_NONE;
        double M = 0, c = 0, v = 0;
        if (s == 0 && n < N) {
            if (!valid) {
                flag = EGDST_PT_NONE;
                atomicMin(&E.evmin[0], p);  // the grid ends before this point (loop guard)
                if (n == nfirst || (int)seed[7] + n - 1 < cx.ngridmax) egdst_fail(P, ivec, EGDST_ERR_ADRAW_LOOP, it, ist, id);
            } else {
                double rhs = 0, evf = 0, chk = 0, badcash = 0; int bq = EGDST_NOBAD, bt = 0;
                for (int k = 0; k < nsl; k++) {
                    const int o = k * Pp + p;
                    rhs += E.rhs[o]; evf += E.evf[o]; chk += E.chk[o];
                    if (E.q[o] < bq) { bq = E.q[o]; bt = E.t[o]; badcash = E.cash[o]; }
                }
                double stopv;
                if (bq != EGDST_NOBAD) {
                    flag = bt;
                    stopv = (bt == EGDST_PT_C1NEG) ? cx.a0 - 1 : badcash;
                } else if (fabs(chk - 1) > cx.tolerance) {
                    flag = EGDST_PT_CHECKSUM; stopv = EGDST_INF;
                } else {
                    const double beta = discount(&cx, &curr);
                    M = A + utility_marginal_inverse(&cx, &curr, beta * rhs);
                    stopv = M;
                    if (!isfinite(M)) flag = EGDST_PT_NONFINITE;
                    else { c = M - A; v = utility(&cx, &curr, c) + beta * evf; flag = EGDST_PT_OK; }
                }
                if (flag == EGDST_PT_C1NEG) atomicMin(&E.evmin[1], p);     // asks for a re-send: not kept, ends this pass
                else if (!(stopv < cx.mmax)) atomicMin(&E.evmin[0], p + 1);  // stop rule: this point is the last one generated
            }
        }
        egdst_cta_sync();
        // points of the item that the sequential generator would have produced: p < lim
        const int ls = E.evmin[0], ll = E.evmin[1];
        const int lim = ll < ls ? ll : ls;
        const bool in = s == 0 && n < N && p < lim;
        const bool keep = in && flag == EGDST_PT_OK;
        const unsigned bal = __ballot_sync(EGDST_FULL, keep);
        int total;
        int woff = egdst_block_excl_scan(lane == 0 ? __popc(bal) : 0, E.sh, &total);
        woff = __shfl_sync(EGDST_FULL, woff, 0);
        int err = 0;
        if (warp == 0) {
            const unsigned long long e = egdst_lookback<1>(st, item + 1, egdst_scan_pack(total, lim != 0x7fffffff ? 1 : 0), &err);
            if (lane == 0) E.excl = e;
        }
        egdst_cta_sync();
        const unsigned long long excl = E.excl;
        if (!egdst_scan_hi(excl)) {  // the grid did not end in an earlier item: this item's points count
            if (in && flag == EGDST_PT_CHECKSUM) egdst_fail(P, ivec, EGDST_ERR_CHECKSUM, it, ist, id);
            if (in && flag == EGDST_PT_EVFINF) P.evfa0[sd] = -EGDST_INF;  // egdst_solver.c:596 (the point itself is dropped)
            if (threadIdx.x == 0 && ll < ls) {  // first re-send request of this grid: egdst_ph_resend takes over at that point
                P.lateN[sd] = nfirst + item * Pp + ll;
                atomicAdd(P.flags + 8 * T.slot + (pass % 3), 1);
            }
            const int first = egdst_scan_lo(excl);
            double *X = P.ptX + (size_t)sd * P.gcap, *Cc = P.ptC + (size_t)sd * P.gcap, *V = P.ptV + (size_t)sd * P.gcap;
            if (keep) {
                const int loc = woff + __popc(bal & ltmask);
                const int dst = first + loc;
                if (dst < P.gcap) { X[dst] = M; Cc[dst] = c; V[dst] = v; }
                E.kx[loc] = M; E.kv[loc] = v;
            }
            egdst_cta_sync();
            // folds between neighbours that this item wrote itself (M or V decreasing, egdst_solver.c:819)
            if (threadIdx.x >= 1 && threadIdx.x < total && first + threadIdx.x < P.gcap)
                if (E.kx[threadIdx.x - 1] > E.kx[threadIdx.x] || E.kv[threadIdx.x - 1] > E.kv[threadIdx.x]) {
                    const int k = atomicAdd(P.foldCnt + sd, 1); if (k <= P.gcap) P.foldList[(size_t)sd * (P.gcap + 1) + k] = first + threadIdx.x;
                }
            if (threadIdx.x == 0 && total > 0) atomicAdd(P.units + ivec, (unsigned long long)total);
        }
        if (err) egdst_fail(P, ivec, EGDST_ERR_ENV2SPACE, it, ist, id);
        __threadfence();
        egdst_cta_sync();
        if (threadIdx.x == 0) E.last = (atomicAdd(P.tickC + 2 * sd + 1, 1) == nitems - 1);
        egdst_cta_sync();
        if (E.last) { __threadfence(); egdst_egm_epilogue(P, it, ivec, ist, id, sd, nitems, T.slot); }
    }
}

// ---------------------------------------------------------------------------------------------
// A zero-consumption re-send requested by a grid point after the seed stage (egdst_solver.c:583-627, 1080-1099):
// the reference replaces that point by A = cashinhandinverse(...) + ZEROCONSUMPTION, makes it the new focal point of
// the grid (k3 = 1, limits from the line through the base point and (a0, a0)) and generates the REST of the grid from
// there.  One CTA per (ist,id) that asked: re-evaluate the offending point to learn where consumption vanished,
// re-send (repeatedly if the re-sent point asks again), store the point, publish the new closed form.  The EGM phase
// then runs again for the grid points after it.
// ---------------------------------------------------------------------------------------------
EGDST_DEV void egdst_ph_resend(const EgdstDev &P, int it, const EgdstTeam &T, int pass, void *scratch, double *shsm) {
    EgdstSeedShared &S = *reinterpret_cast<EgdstSeedShared *>(scratch);
    const int jpv = P.cx.nst * P.cx.nd, nwork = T.nv * jpv;
    const int useTab = egdst_use_shocktab(P);
    const int N = P.N;
    if (T.rank == 0 && threadIdx.x == 0) P.flags[8 * T.slot + ((pass + 1) % 3)] = 0;  // the counter of the next pass
    for (int w = T.rank; w < nwork; w += T.size) {
        const int ivec = T.v0 + w / jpv, jy = w % jpv, ist = jy / P.cx.nd, id = jy % P.cx.nd;
        const int sd = egdst_sd(P, ivec, ist, id);
        egdst_cta_sync();
        const int nl = P.lateN[sd];
        if (!P.active[sd] || nl == 0x7fffffff) continue;  // grids that did not ask are complete
        egdst_ctx cx; egdst_load_ctx(P, ivec, cx);
        PeriodVars curr; curr.it = it; curr.ist = ist; curr.id = id; curr.cash = 0; curr.savings = 0; curr.shock = 0;
        double *seed = P.seed + (size_t)sd * EGDST_SEEDW;
        const double *X = P.ptX + (size_t)sd * P.gcap, *V = P.ptV + (size_t)sd * P.gcap;
        const int nitems = (N - 1 + P.egmP - 1) / P.egmP;
        const double beta = discount(&cx, &curr);
        const double *shk = 0, *shp = 0;
        if (useTab) {
            egdst_fill_shocktab(&cx, P, &curr, shsm, shsm + cx.nst * cx.ny, threadIdx.x, blockDim.x);
            shk = shsm; shp = shsm + cx.nst * cx.ny;
        }
        int kept = egdst_scan_lo(egdst_scan_inclusive(P.scanC + (size_t)sd * P.chC, nitems));  // points before the offending one
        if (kept > P.gcap) kept = P.gcap;
        const double baseA = seed[8], baseM = seed[9];
        if (threadIdx.x == 0) { S.A = egdst_agrid(&cx, &curr, seed, nl, N); S.calls = (int)seed[7]; S.go = 1; }
        egdst_cta_sync();
        // the limits of the published seed (k3 >= 1: egdst_adraw does not take the first ones again)
        EgdstLims L; L.lim1 = seed[0]; L.lim2 = seed[1]; L.lim3 = seed[2]; L.lim3p = seed[3]; L.k3 = seed[4]; L.lim2p = 0;
        const EgdstAdraw r = egdst_adraw(&cx, P, it, ivec, ist, id, &curr, beta, kept, baseA, baseM, L, S, shk, shp);
        if (threadIdx.x == 0) {
            P.evfa0[sd] = -EGDST_INF;  // egdst_solver.c:596
            atomicAdd(P.units + P.nvec + ivec, 1ULL);  // diagnostic: re-sends after the seed stage handled in this solve
            if (r.stored) {
                if (kept > 0 && (X[kept - 1] > X[kept] || V[kept - 1] > V[kept])) {
                    const int k = atomicAdd(P.foldCnt + sd, 1); if (k <= P.gcap) P.foldList[(size_t)sd * (P.gcap + 1) + k] = kept;
                }
                kept += 1;
                atomicAdd(P.units + ivec, 1ULL);
            }
            // the grid goes on after the re-sent point (which took the place of point nl) unless it ended there
            const int stop = (S.go == -1 || !(r.aM < cx.mmax)) ? 1 : 0;
            egdst_seed_publish(P, sd, seed, L, r.lastA, nl + 1, S.calls, baseA, baseM, kept, stop, pass + 1);
            for (int c = 1; c < P.chC; c++) P.scanC[(size_t)sd * P.chC + c] = 0ULL;
            P.tickC[2 * sd + 1] = 0;
            P.lateN[sd] = 0x7fffffff;
        }
    }
}
