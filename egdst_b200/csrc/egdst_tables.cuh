// egdst_tables.cuh -- per-cell lookup tables shared by the solver (period t reads the tables of t+1) and the
// simulator.  Built by egdst_k_tab right after a cell's primary envelope is final.
//
// Every table access of the hot loops is a per-thread gather, so the layout is chosen to make one policy/value
// lookup cost four 16-byte loads (neighbouring A points / agents with neighbouring cash hit the same lines):
//   lut [ncell][lutcap+1] EgdstLutEntry  direct index by the leading bits of the IEEE representation of
//        (x - a0 + 1): key = exponent and the top `mbits` mantissa bits, a piecewise-linear log2 -- the endogenous
//        grids are (sym-)log spaced (egdst_solver.c:1104-1136), so buckets are evenly filled.  Entry b (32 bytes)
//        holds l = #rows with key < b, the number of rows in the bucket and the abscissas of its first three rows
//        (+inf where there is none): #rows <= x is l + (m0<=x) + (m1<=x) + (m2<=x) without touching the grid, so the
//        bracket is final after ONE gather; only buckets with more than three rows bisect.
//   row [ncell][tabcap+1] EgdstRow       (M_i, C_i, V_i, RN(1/(M_i+1 - M_i))), 32 bytes = one sector per row: rows i and
//        i+1 -- 64 contiguous bytes -- are everything the interpolations of the EGM step (egdst_solver.c:552-567,
//        755-772) and of policy() (egdst_simulator.c:178-197) need.  The correctly rounded reciprocal of the interval
//        width is a function of the two abscissas only, so it is computed once per row here instead of once per lookup.
// The tables of one cell take 32 B per row plus 32 B per index bucket (about one bucket per row): the working set of
// the simulator -- every period's tables at once -- has to stay L2-resident next to its output stream.
// This replaces the 14-step bisections of bxsearch (egdst_lib.c:138-165), 2 per quadrature node and agent-period.
// Cells with more rows than tabcap+1 (possible only when ngridmax >> 2*ngridm is actually used) keep the bisection.
#pragma once

#include "egdst_common.cuh"

EGDST_DEV int egdst_lut_key(double x, double a0, int mbits) {
    const double y = x - a0 + 1.0;
#ifdef EGDST_HOSTEMU
    long long bits; memcpy(&bits, &y, 8);
    const int hi = (int)(bits >> 32);
#else
    const int hi = __double2hiint(y);
#endif
    return (hi >> (20 - mbits)) - (0x3FF00000 >> (20 - mbits));
}

EGDST_DEV const EgdstRow *egdst_cell_rows(const EgdstDev &P, int cell) { return P.tabRow + (size_t)cell * (P.tabcap + 1); }
EGDST_DEV const EgdstLutEntry *egdst_cell_lut(const EgdstDev &P, int cell) { return P.tabLut + (size_t)cell * (P.lutcap + 1); }
// A cell has usable tables when it fits them and its grid is increasing.  The reference's bisection (bxsearch,
// egdst_lib.c:138-165; restated by egdst_bracket) is defined on ANY array, and degenerate models do produce cells whose
// grid steps back (e.g. a row below a0 after a re-send, examples.deaton_meanstest): there the direct index, which counts
// rows below x, and the bisection, which follows its own path, disagree -- such cells take the bisection.
EGDST_DEV bool egdst_cell_fits_tab(const EgdstDev &P, int n) { return n - 1 <= P.tabcap; }
EGDST_DEV bool egdst_cell_has_tab(const EgdstDev &P, int cell, int n) { return n - 1 <= P.tabcap && P.tabOk[cell] != 0; }

// L2 eviction-priority hints (PTX createpolicy / ld.global.L2::cache_hint): the simulator streams tens of GB of
// output through L2; table lines loaded with evict_last survive that stream, the output is written evict_first.
#ifndef EGDST_HOSTEMU
EGDST_DEV unsigned long long egdst_policy_evict_last() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
EGDST_DEV double2 egdst_ld16_hint(const void *p, unsigned long long pol) {
    double2 v;
    asm volatile("ld.global.L2::cache_hint.v2.f64 {%0, %1}, [%2], %3;" : "=d"(v.x), "=d"(v.y) : "l"(p), "l"(pol));
    return v;
}
#endif

// rows i and i+1 as one interval: four 16-byte loads of 64 contiguous bytes
EGDST_DEV EgdstInterval egdst_load_interval(const EgdstRow *p) {
    EgdstInterval iv;
#ifdef EGDST_HOSTEMU
    iv.g0 = p[0].m; iv.c0 = p[0].c; iv.v0 = p[0].v; iv.y = p[0].y; iv.g1 = p[1].m; iv.c1 = p[1].c; iv.v1 = p[1].v;
#else
    const double2 *q = reinterpret_cast<const double2 *>(p);
    const double2 q0 = q[0], q1 = q[1], q2 = q[2];
    const double v1 = reinterpret_cast<const double *>(p)[6];
    iv.g0 = q0.x; iv.c0 = q0.y; iv.v0 = q1.x; iv.y = q1.y; iv.g1 = q2.x; iv.c1 = q2.y; iv.v1 = v1;
#endif
    iv.pad = 0.0;
    return iv;
}

// Start-of-period housekeeping for parameter vector ivec (all threads of one CTA): reset the chained-scan state of
// its jobs, mark infeasible (it,ist) cells as empty and detect empty choice sets (egdst_solver.c:294-300, 694-702).
EGDST_DEV void egdst_cells_body(const EgdstDev &P, int ivec, int it) {
    const int nsdv = P.cx.nst * P.cx.nd, sd0 = ivec * nsdv;
    for (int i = threadIdx.x; i < nsdv * P.chC; i += blockDim.x) P.scanC[(size_t)sd0 * P.chC + i] = 0ULL;
    for (int i = threadIdx.x; i < nsdv * 2; i += blockDim.x) P.tickC[2 * sd0 + i] = 0;
    for (int i = threadIdx.x; i < nsdv; i += blockDim.x) { P.foldCnt[sd0 + i] = 0; P.lateN[sd0 + i] = 0x7fffffff; }
    for (int i = threadIdx.x; i < nsdv * P.chE; i += blockDim.x) P.scanE[(size_t)sd0 * P.chE + i] = 0ULL;          // secondary slots
    for (int i = threadIdx.x; i < nsdv * 2; i += blockDim.x) P.tickE[2 * sd0 + i] = 0;
    for (int i = threadIdx.x; i < nsdv; i += blockDim.x) P.envNact[sd0 + i] = 0;
    const int ps0 = P.priSync0 + ivec * P.cx.nst;                                                                  // primary jobs
    for (int i = threadIdx.x; i < P.cx.nst * P.chE; i += blockDim.x) P.scanE[(size_t)ps0 * P.chE + i] = 0ULL;
    for (int i = threadIdx.x; i < P.cx.nst * 2; i += blockDim.x) P.tickE[2 * ps0 + i] = 0;
    for (int i = threadIdx.x; i < P.cx.nst; i += blockDim.x) P.envNact[ps0 + i] = 0;
    for (int ist = threadIdx.x; ist < P.cx.nst; ist += blockDim.x) {
        {   // the tables of the period's cells (and, in the smoothing mode, choice-specific cells) are usable unless their build says otherwise
            const int c0 = egdst_cell(P, ivec, it, ist);
            P.tabOk[c0] = 1;
            if (EGDST_SMOOTHING) for (int d_ = 0; d_ < P.cx.nd; d_++) P.tabOk[egdst_dcell(P, c0, d_)] = 1;
        }
        egdst_ctx cx; egdst_load_ctx(P, ivec, cx);
        PeriodVars curr; curr.it = it; curr.ist = ist; curr.id = 0; curr.cash = 0; curr.savings = 0; curr.shock = 0;
        const int cell = egdst_cell(P, ivec, it, ist);
        if (feasible(&cx, &curr) != 1) { P.mlen[cell] = 0; P.thlen[cell] = 0; continue; }
        int any = 0;
        for (curr.id = 0; curr.id < cx.nd; curr.id++) any |= (inchoiceset(&cx, &curr) == 1);
        if (!any) { P.mlen[cell] = 0; P.thlen[cell] = 0; egdst_fail(P, ivec, EGDST_ERR_EMPTYCHOICE, it, ist, -1); }
    }
}
// the same for every vector of a team, plus the team's period flags
EGDST_DEV void egdst_ph_cells(const EgdstDev &P, int it, const EgdstTeam &T) {
    for (int v = T.rank; v < T.nv; v += T.size) egdst_cells_body(P, T.v0 + v, it);
    if (T.rank == 0 && threadIdx.x < 8) P.flags[8 * T.slot + threadIdx.x] = 0;
}

// Build the tables of one cell: the share of virtual block vb of nvb (all threads of the CTA, 1-D blocks).
EGDST_DEV void egdst_tab_cell(const EgdstDev &P, int cell, int vb, int nvb) {
    const int n = P.mlen[cell];
    if (n < 2 || !egdst_cell_fits_tab(P, n)) return;
    const double a0 = P.cx.a0;
    const double *M = egdst_colM(P, cell), *C = egdst_colC(P, cell), *V = egdst_colV(P, cell);
    EgdstRow *r = P.tabRow + (size_t)cell * (P.tabcap + 1);
    const int stride = nvb * blockDim.x, t0 = vb * blockDim.x + threadIdx.x;
    if (t0 == 0) {  // the cell's last interval and its image under the extrapolation transform
        EgdstCellTop T; T.g0 = M[n - 2]; T.g1 = M[n - 1]; T.c0 = C[n - 2]; T.c1 = C[n - 1]; T.v0 = V[n - 2]; T.v1 = V[n - 1];
        const double w = T.g1 - T.g0;
        T.y = egdst_div_safe(w) ? 1.0 / w : 0.0;
        const int mc = cell < P.ncellMain ? cell : (cell - P.ncellMain) / P.cx.nd;  // decision cells (smoothing mode) follow the solution cells
        const int ist = mc % P.cx.nst, it = (mc / P.cx.nst) % P.NT, ivec = mc / (P.cx.nst * P.NT);
        egdst_ctx cx; egdst_load_ctx(P, ivec, cx);
        PeriodVars prd; prd.it = it; prd.ist = ist; prd.id = 0; prd.cash = 0; prd.savings = 0; prd.shock = 0;
        egdst_fill_state(&cx, &prd);
        T.t0 = tr(&cx, &prd, T.g0 - a0); T.t1 = tr(&cx, &prd, T.g1 - a0);
        const double wt = T.t1 - T.t0;
        T.yt = egdst_div_safe(wt) ? 1.0 / wt : 0.0;
        P.tabTop[cell] = T;
    }
    for (int i = t0; i < n; i += stride) {
        EgdstRow v; v.m = M[i]; v.c = C[i]; v.v = V[i]; v.y = 0.0;
        if (i + 1 < n && M[i + 1] < v.m) atomicMin(P.tabOk + cell, 0);  // the grid steps back: no tables for this cell
        if (i + 1 < n) { const double w = M[i + 1] - v.m; v.y = egdst_div_safe(w) ? 1.0 / w : 0.0; }  // shared correctly rounded reciprocal (0: plain divisions)
        r[i] = v;
    }
    // direct index, row-centric (no searches): row r is the first row with key >= b for every bucket b in
    // (key(r-1), key(r)]; the bucket key(r) also gets the number of rows that share the key and their abscissas
    EgdstLutEntry *L = P.tabLut + (size_t)cell * (P.lutcap + 1);
    const int kmax = P.lutcap - 1;
    const int lane = threadIdx.x & 31;
    for (int base = vb * blockDim.x; base < n; base += stride) {  // warp-uniform trip count
        const int r = base + threadIdx.x;
        int gap0 = 0, gap1 = 0;
        EgdstLutEntry e; e.l = r; e.cnt = 0; e.m0 = EGDST_INF; e.m1 = EGDST_INF; e.m2 = EGDST_INF;
        if (r < n) {
            const double m = M[r];
            int kr = egdst_lut_key(m, a0, P.mbits); kr = kr < 0 ? 0 : (kr > kmax ? kmax : kr);
            int kp = -1;
            if (r > 0) { kp = egdst_lut_key(M[r - 1], a0, P.mbits); kp = kp < 0 ? 0 : (kp > kmax ? kmax : kp); }
            if (kr > kp) {
                int cnt = 1;
                EgdstLutEntry f = e;
                f.m0 = m;
                while (r + cnt < n) {
                    const double mn = M[r + cnt];
                    int kn = egdst_lut_key(mn, a0, P.mbits); kn = kn < 0 ? 0 : (kn > kmax ? kmax : kn);
                    if (kn != kr) break;
                    if (cnt == 1) f.m1 = mn; else if (cnt == 2) f.m2 = mn;
                    cnt++;
                }
                f.cnt = cnt;
                L[kr] = f;
                gap0 = kp + 1; gap1 = kr;  // empty buckets [gap0, gap1) point at row r too
            }
        }
        if (gap1 - gap0 <= 8) { for (int bb = gap0; bb < gap1; bb++) L[bb] = e; gap1 = gap0; }
        // long runs of empty buckets (coarse stretches of a sym-log grid) are filled by the whole warp
        unsigned longm = __ballot_sync(EGDST_FULL, gap1 > gap0);
        while (longm) {
            const int src = __ffs(longm) - 1;
            longm &= longm - 1;
            const int b0 = __shfl_sync(EGDST_FULL, gap0, src), b1 = __shfl_sync(EGDST_FULL, gap1, src);
            EgdstLutEntry f; f.l = __shfl_sync(EGDST_FULL, e.l, src); f.cnt = 0; f.m0 = EGDST_INF; f.m1 = EGDST_INF; f.m2 = EGDST_INF;
            for (int bb = b0 + lane; bb < b1; bb += 32) L[bb] = f;
        }
    }
    {   // buckets above the last row's key
        int kl = egdst_lut_key(M[n - 1], a0, P.mbits); kl = kl < 0 ? 0 : (kl > kmax ? kmax : kl);
        EgdstLutEntry e; e.l = n; e.cnt = 0; e.m0 = EGDST_INF; e.m1 = EGDST_INF; e.m2 = EGDST_INF;
        for (int bb = kl + 1 + t0; bb <= P.lutcap; bb += stride) L[bb] = e;
    }
}

// tables of the cells (ivec, it, all ist) of a team: nvb virtual blocks per cell
EGDST_DEV void egdst_ph_tab(const EgdstDev &P, int it, const EgdstTeam &T, int nvb) {
    const int jpv = P.cx.nst, nwork = T.nv * jpv * nvb;
    for (int w = T.rank; w < nwork; w += T.size) {
        const int njobs = T.nv * jpv, vb = w / njobs, j = w - vb * njobs;
        egdst_tab_cell(P, egdst_cell(P, T.v0 + j / jpv, it, j % jpv), vb, nvb);
    }
    if (EGDST_SMOOTHING) {  // smoothing mode: the choice-specific tables of the period
        const int nd = P.cx.nd, jpd = jpv * nd, nworkd = T.nv * jpd * nvb;
        for (int w = T.rank; w < nworkd; w += T.size) {
            const int njobs = T.nv * jpd, vb = w / njobs, j = w - vb * njobs, r = j % jpd;
            egdst_tab_cell(P, egdst_dcell(P, egdst_cell(P, T.v0 + j / jpd, it, r / nd), r % nd), vb, nvb);
        }
    }
}
// smoothing mode: each decision's point list (after its secondary envelope) becomes a cell of its own, in the layout
// of the solution cells (row 0 = a0, 0, a0, evf_d(a0)); an unavailable decision has 0 rows.  Like the reference's
// envelop(), which ends the unified grid at the smallest of the decisions' last abscissae (egdst_solver.c:1266-1271)
// and keeps the interpolated values there, a list that reaches further is cut at that bound: sigma_eps -> 0 then
// reproduces the reference's cells also where next period's cash lands above the unified grid.
EGDST_DEV void egdst_ph_dsave(const EgdstDev &P, int it, const EgdstTeam &T) {
    const int nd = P.cx.nd, jpd = P.cx.nst * nd, nwork = T.nv * jpd;
    for (int w = T.rank; w < nwork; w += T.size) {
        const int ivec = T.v0 + w / jpd, r = w % jpd, ist = r / nd, id = r % nd;
        const int sd = egdst_sd(P, ivec, ist, id), dcell = egdst_dcell(P, egdst_cell(P, ivec, it, ist), id);
        int n = P.active[sd] ? P.ptN[sd] : 0;
        if (n > P.rowcap - 2) n = P.rowcap - 2;
        const double *X = P.ptX + (size_t)sd * P.gcap, *Cc = P.ptC + (size_t)sd * P.gcap, *V = P.ptV + (size_t)sd * P.gcap;
        double grb = EGDST_INF;
        for (int f = 0; f < nd; f++) {
            const int sf = egdst_sd(P, ivec, ist, f), nf = P.active[sf] ? P.ptN[sf] : 0;
            if (nf > 0) { const double xl = P.ptX[(size_t)sf * P.gcap + nf - 1]; if (xl < grb) grb = xl; }
        }
        // rows with x <= grb: the list is sorted, every thread bisects for itself (no exchange needed)
        int keep = 0;
        { int l = 0, h = n; while (l < h) { const int mid = (l + h) >> 1; if (X[mid] <= grb) l = mid + 1; else h = mid; } keep = l; }
        double *oM = egdst_colM(P, dcell), *oC = egdst_colC(P, dcell), *oA = egdst_colA(P, dcell), *oV = egdst_colV(P, dcell);
        for (int i = threadIdx.x; i < keep; i += blockDim.x) { const double x = X[i], c = Cc[i]; oM[1 + i] = x; oC[1 + i] = c; oA[1 + i] = x - c; oV[1 + i] = V[i]; }
        if (threadIdx.x == 0) {
            int rows = keep;
            if (keep > 0 && keep < n && X[keep - 1] < grb) {  // the values at the bound, interpolated on the interval that straddles it
                const double x0 = X[keep - 1], x1 = X[keep];
                const double c = egdst_lerp(grb, x0, x1, Cc[keep - 1], Cc[keep]), v = egdst_lerp(grb, x0, x1, V[keep - 1], V[keep]);
                oM[1 + keep] = grb; oC[1 + keep] = c; oA[1 + keep] = grb - c; oV[1 + keep] = v;
                rows = keep + 1;
            }
            const double e = P.evfa0[sd], a0 = P.cx.a0;
            oM[0] = a0; oC[0] = 0.0; oA[0] = a0; oV[0] = e;
            P.evf[dcell] = e;
            P.mlen[dcell] = rows > 0 ? rows + 1 : 0;
        }
    }
}
// tables of imported cells (egdst_solution_import): grid (nblk, nst, 1)
__global__ void egdst_k_tabonly(EgdstDev P, int it) { egdst_tab_cell(P, egdst_cell(P, blockIdx.z, it, blockIdx.y), blockIdx.x, gridDim.x); }

// the simulator's version: the same loads with the evict_last hint
EGDST_DEV EgdstInterval egdst_load_interval_keep(const EgdstRow *p, unsigned long long pol) {
#ifdef EGDST_HOSTEMU
    return egdst_load_interval(p);
#else
    const double2 q0 = egdst_ld16_hint(p, pol), q1 = egdst_ld16_hint((const double2 *)p + 1, pol), q2 = egdst_ld16_hint((const double2 *)p + 2, pol),
                  q3 = egdst_ld16_hint((const double2 *)p + 3, pol);
    EgdstInterval iv; iv.g0 = q0.x; iv.c0 = q0.y; iv.v0 = q1.x; iv.y = q1.y; iv.g1 = q2.x; iv.c1 = q2.y; iv.v1 = q3.x; iv.pad = 0.0;
    return iv;
#endif
}

// Index entry of x's bucket.  KEEP: load with the evict_last hint `pol`.
template <bool KEEP = false>
EGDST_DEV EgdstLutEntry egdst_lut_entry(const EgdstDev &P, int cell, double x, unsigned long long pol = 0ULL) {
    int b = egdst_lut_key(x, P.cx.a0, P.mbits);
    b = b < 0 ? 0 : (b > P.lutcap - 1 ? P.lutcap - 1 : b);
    const EgdstLutEntry *lut = egdst_cell_lut(P, cell);
#ifdef EGDST_HOSTEMU
    const EgdstLutEntry e = lut[b];
#else
    EgdstLutEntry e;
    if (KEEP) {
        const double2 r0 = egdst_ld16_hint(lut + b, pol), r1 = egdst_ld16_hint((const double2 *)(lut + b) + 1, pol);
        const long long lo = __double_as_longlong(r0.x);
        e.l = (int)(lo & 0xffffffffLL); e.cnt = (int)(lo >> 32); e.m0 = r0.y; e.m1 = r1.x; e.m2 = r1.y;
    } else {
        const int4 r0 = *reinterpret_cast<const int4 *>(lut + b);
        const double2 r1 = *(reinterpret_cast<const double2 *>(lut + b) + 1);
        e.l = r0.x; e.cnt = r0.y; e.m0 = __hiloint2double(r0.w, r0.z); e.m1 = r1.x; e.m2 = r1.y;
    }
#endif
    return e;
}
// The rank the index entry e of x's bucket gives: (#rows <= x) - 1, where crowded buckets (more than three rows: the
// grid is dense around a focal point or holds double points) bisect their remaining rows of M.  Not clamped.
EGDST_DEV int egdst_lut_entry_rank(const EgdstLutEntry &e, const double *M, double x) {
    int i = e.l - 1 + (e.m0 <= x ? 1 : 0) + (e.m1 <= x ? 1 : 0) + (e.m2 <= x ? 1 : 0);
    if (e.cnt > 3 && e.m2 <= x) {
        int l = e.l + 3, h = e.l + e.cnt;
        while (l < h) { const int mid = (l + h) >> 1; if (M[mid] <= x) l = mid + 1; else h = mid; }
        i = l - 1;
    }
    return i;
}
template <bool KEEP = false>
EGDST_DEV int egdst_lut_rank(const EgdstDev &P, int cell, const double *M, double x, unsigned long long pol = 0ULL) {
    return egdst_lut_entry_rank(egdst_lut_entry<KEEP>(P, cell, x, pol), M, x);
}

// The record of rows i and i+1 of a cell: from the row table when the cell's tables may be used (tab,
// egdst_cell_has_tab), otherwise from the columns, with y filled as the table rows fill it (RN(1/w), 0 where the width
// is degenerate: plain divisions).  KEEP: load with the evict_last hint `pol`.
template <bool KEEP = false>
EGDST_DEV EgdstInterval egdst_cell_interval(const EgdstDev &P, int cell, bool tab, int i, unsigned long long pol = 0ULL) {
    if (tab) {
        const EgdstRow *r = egdst_cell_rows(P, cell) + i;
        return KEEP ? egdst_load_interval_keep(r, pol) : egdst_load_interval(r);
    }
    const double *M = egdst_colM(P, cell), *C = egdst_colC(P, cell), *V = egdst_colV(P, cell);
    EgdstInterval iv;
    iv.g0 = M[i]; iv.g1 = M[i + 1]; iv.c0 = C[i]; iv.c1 = C[i + 1]; iv.v0 = V[i]; iv.v1 = V[i + 1];
    iv.y = egdst_div_safe(iv.g1 - iv.g0) ? 1.0 / (iv.g1 - iv.g0) : 0.0;
    iv.pad = 0.0;
    return iv;
}

// Bracket i of x in a cell of n rows and the record of rows i and i+1.  With tables, two dependent gathers (the index
// entry, then 64 contiguous bytes of rows); without, the reference's bisection (egdst_bracket).  On a strictly
// increasing grid both give (#rows <= x) - 1 clamped to [0, n-2].
template <bool KEEP = false>
EGDST_DEV int egdst_cell_lookup(const EgdstDev &P, int cell, bool tab, double x, int n, EgdstInterval &iv, unsigned long long pol = 0ULL) {
    const double *M = egdst_colM(P, cell);
    int i;
    if (tab) {
        i = egdst_lut_rank<KEEP>(P, cell, M, x, pol);
        i = i > n - 2 ? n - 2 : i;
        i = i < 0 ? 0 : i;
    } else {
        i = egdst_bracket(x, M, n, 0);
    }
    iv = egdst_cell_interval<KEEP>(P, cell, tab, i, pol);
    return i;
}

// The second half of egdst_cell_lookup for a cell with tables, from the index entry e of x (egdst_lut_entry<true>):
// the simulator's pipelined period loop issues the entry gather a period ahead of this.  The solver keeps the fused
// egdst_cell_lookup: built on these halves, the grid-scope solve kernel gets a larger stack frame.
EGDST_DEV int egdst_cell_lookup_finish(const EgdstDev &P, int cell, double x, int n, const EgdstLutEntry &e, EgdstInterval &iv,
                                       unsigned long long pol) {
    int i = egdst_lut_entry_rank(e, egdst_colM(P, cell), x);
    i = i > n - 2 ? n - 2 : i;
    i = i < 0 ? 0 : i;
    iv = egdst_cell_interval<true>(P, cell, true, i, pol);
    return i;
}
