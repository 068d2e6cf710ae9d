// egdst_simulator.cuh -- forward Monte-Carlo simulation of agents on a solved model.
//
// Restates the reference's simulator (@egdstmodel/egdst_simulator.c):
//   simulator()   :204-383   one agent's path over it = 0..T-t0 (survival, state transition by inverse-CDF
//                            sampling over trpr, shock = cdfinv(u) or expectation, budget, equations)
//   policy()      :145-199   c = linter(cash; M,C), id by threshold scan, vf exact below M(a0) else linter
//   simsoutput()  :122-143   the nsimout output columns
//   continuous states :310-373 (multilinear mix over the 2^k surrounding grid cells; compiled in when EGDST_NCONT > 0)
// A warp walks a tile of 32 agents through all periods (persistent grid of one resident wave).  The
// [nsimout, nt, nsim] output is written through a per-warp shared-memory tile so that each store instruction
// covers contiguous runs of an agent's record (the per-thread pattern of the reference has stride nsimout*nt).
// Uniforms come either from the reference's randstream layout (parity mode) or from counter-based
// Philox4x32-10 keyed by (seed; global agent id, period).
//
// The kernel is bound by instruction issue and gather latency before it is bound by the output stream, so
// everything the launch knows in advance is a template parameter (source of uniforms, which outputs exist, where
// the moment accumulators and the per-cell headers live) and everything the model image knows in advance is a
// macro of the generated header (EGDST_OPT_TRPRNOSH ...): the period loop carries no run-time mode switches.
#pragma once

#include "egdst_solver.cuh"

#define EGDST_NSIMOUT_MAX (11 + EGDST_NNST + EGDST_NND + EGDST_NREQ)
#ifdef EGDST_HOSTEMU
#define EGDST_SIM_BLOCK 64
#else
#define EGDST_SIM_BLOCK 256
#endif
#ifndef EGDST_SIM_MINBLOCKS
#define EGDST_SIM_MINBLOCKS 4
#endif
// CTA width of the two-periods-per-write variant: two CTAs of 12 warps per SM leave each thread 80 registers, which the
// pipelined period loop needs, and room for the per-CTA moment accumulators next to the staged rows
#ifdef EGDST_HOSTEMU
#define EGDST_SIM_WIDE 128
#else
#define EGDST_SIM_WIDE 384
#endif

// the sims array is written once and never re-read by the kernel: evict-first (st.global.cs) keeps the policy
// tables resident in L2 instead of the output stream
#ifdef EGDST_HOSTEMU
#define EGDST_STREAM_STORE2(ptr, v) (*reinterpret_cast<double2 *>(ptr) = (v))
#else
#define EGDST_STREAM_STORE2(ptr, v) __stcs(reinterpret_cast<double2 *>(ptr), (v))
#endif

// Philox4x32-10 (Salmon et al. 2011); counter = (c0,c1,c2,c3), key = (k0,k1)
EGDST_DEV void egdst_philox4x32(unsigned c0, unsigned c1, unsigned c2, unsigned c3, unsigned k0, unsigned k1,
                                unsigned &o0, unsigned &o1, unsigned &o2, unsigned &o3) {
    for (int r = 0; r < 10; r++) {
        const unsigned long long p0 = (unsigned long long)0xD2511F53u * c0, p1 = (unsigned long long)0xCD9E8D57u * c2;
        const unsigned hi0 = (unsigned)(p0 >> 32), lo0 = (unsigned)p0, hi1 = (unsigned)(p1 >> 32), lo1 = (unsigned)p1;
        const unsigned n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    o0 = c0; o1 = c1; o2 = c2; o3 = c3;
}
EGDST_DEV double egdst_u01(unsigned x) { return ((double)x + 0.5) * (1.0 / 4294967296.0); }

// Per-cell scalars the policy lookup needs every period (rows, thresholds, evf(a0), M[1]).  With ~190 KB of the SM's
// SRAM carved out as shared memory the L1 is a few tens of KB and these 'uniform' global loads would go to L2 every
// agent-period; they travel instead as a by-value kernel argument (constant bank, up to EGDST_SIM_MAXHDR cells).
#define EGDST_SIM_TH8 4
#define EGDST_SIM_MAXHDR 128
#define EGDST_HDR_NOTAB 0x40000000  /* flag in EgdstCellHdr::n */
struct EgdstCellHdr { int n, nth; double evf, M1; double th[EGDST_SIM_TH8], dd[EGDST_SIM_TH8]; };
#define EGDST_SIM_MAXTAB 96
struct EgdstSimHdrs {
    EgdstCellHdr h[EGDST_SIM_MAXHDR];
    // the model's small tables (stm, states, decisions: egdst_lib.c:241-252), when they fit
    double stm[16], states[EGDST_SIM_MAXTAB], decisions[EGDST_SIM_MAXTAB];
    int tabs_ok;
};

// gathers the headers of parameter vector ivec (host copy -> kernel argument of later simulations)
__global__ void egdst_k_simhdr(EgdstDev P, int ivec, EgdstCellHdr *out) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= P.NT * P.cx.nst) return;
    const int cell = egdst_cell(P, ivec, c / P.cx.nst, c % P.cx.nst);
    EgdstCellHdr h;
    h.n = P.mlen[cell]; h.nth = P.thlen[cell]; h.evf = P.evf[cell];
    h.M1 = h.n > 1 ? egdst_colM(P, cell)[1] : 0.0;
    if (P.tabOk[cell] == 0) h.n |= EGDST_HDR_NOTAB;  // the cell's grid steps back: bisection, not the direct index (egdst_cell_has_tab)
    for (int k = 0; k < EGDST_SIM_TH8; k++) {
        h.th[k] = k < h.nth ? P.thTH[(size_t)cell * P.cx.nthrhmax + k] : EGDST_INF;
        h.dd[k] = k < h.nth ? P.thD[(size_t)cell * P.cx.nthrhmax + k] : 0.0;
    }
    out[c] = h;
}

struct EgdstSimArgs {
    const double *init;        // [nsim] 1-based ist0 of the agents of this launch
    const double *init_m0;     // [nsim] m0 (the second column of the reference's init matrix)
    int nsim;
    int ivec;
    const double *randstream;  // reference layout (template PHILOX = false)
    int rndtype;               // 1 = same shocks for all agents
    long long agent0;
    unsigned long long seed;
    double *sims;              // [nsimout, nt, nsim]   (template OUT & 1)
    double *moments;           // [3, nsimout, nt]      (template OUT & 2)
    int nsimout;
    int mom_smem;              // 1: per-CTA moment accumulators for all periods live in shared memory (flushed at the end)
    double param[EGDST_NPARAM_];  // parameter values of the vector (template HDR: single-vector launches)
};

// One cell's policy at `cash` (egdst_simulator.c:145-199): interval record and M[1]; false if the cell holds no solution.
EGDST_DEV bool egdst_sim_interval(const EgdstDev &P, int cell, int nm, bool tabok, double cash, unsigned long long l2keep, EgdstInterval &iv) {
    if (nm < 2) return false;
    if (tabok && egdst_cell_fits_tab(P, nm)) {
        egdst_cell_lookup<true>(P, cell, true, cash, nm, iv, l2keep);
    } else {
        // cells without tables: the same bracket as egdst_cell_lookup, but y = 0 (egdst_sim_weights divides here), because
        // the record's own reciprocal costs a PB == 2 instantiation of egdst_k_simulate spill space
        const double *Mg = egdst_colM(P, cell), *Cg = egdst_colC(P, cell), *Vg = egdst_colV(P, cell);
        const int i = egdst_bracket(cash, Mg, nm, 0);
        iv.g0 = Mg[i]; iv.g1 = Mg[i + 1]; iv.c0 = Cg[i]; iv.c1 = Cg[i + 1]; iv.v0 = Vg[i]; iv.v1 = Vg[i + 1]; iv.y = 0.0;
    }
    return true;
}
// Whether the policy lookup of a cell of nm rows goes through its tables (tabok: egdst_cell_has_tab's flag), as in
// egdst_sim_interval; the pipelined period order then gathers the index entry of cash (egdst_lut_entry) a period ahead.
EGDST_DEV bool egdst_sim_tab(const EgdstDev &P, int nm, bool tabok) { return nm >= 2 && tabok && egdst_cell_fits_tab(P, nm); }
// One division for the weights of both interpolations (the reference divides four times, egdst_lib.c:175): the
// reciprocal comes with the record.  The exactly rounded quotients of the solver (egdst_div_by) are not needed here:
// the difference is in the last bit and no discrete branch of the simulator depends on it.
EGDST_DEV void egdst_sim_weights(const EgdstInterval &iv, double cash, double &wl, double &wr) {
    const double rw = iv.y != 0.0 ? iv.y : 1.0 / (iv.g1 - iv.g0);
    wl = (cash - iv.g0) * rw; wr = (iv.g1 - cash) * rw;
}

#if EGDST_NCONT > 0
// Policy of ONE cell of the solution at `cash`: consumption, discrete decision and value.  Used by the
// continuous-state branch, which mixes the policies of the 2^NCONT grid cells around the agent's exact state.
EGDST_DEV bool egdst_sim_policy_cell(const EgdstDev &P, const egdst_ctx &cx, int cell, PeriodVars &pv, unsigned long long l2keep,
                                     double &c, double &vf) {
    const int nm = P.mlen[cell];
    EgdstInterval iv;
    if (!egdst_sim_interval(P, cell, nm, P.tabOk[cell] != 0, pv.cash, l2keep, iv)) return false;
    const double M1 = egdst_colM(P, cell)[1];
    double wl, wr;
    egdst_sim_weights(iv, pv.cash, wl, wr);
    c = iv.c1 * wl + iv.c0 * wr;
    pv.id = egdst_policy_decision(pv.cash, P.thTH + (size_t)cell * cx.nthrhmax, P.thD + (size_t)cell * cx.nthrhmax, P.thlen[cell]);
    egdst_fill_decision(&cx, &pv);
    const double evf = P.evf[cell];
    if (pv.cash < M1 && evf > -EGDST_INF) vf = utility(&cx, &pv, c) + discount(&cx, &pv) * evf;
    else vf = iv.v1 * wl + iv.v0 * wr;
    return true;
}
#endif

// One step of an agent's path from period cur.it into period `it` (egdst_simulator.c:259-309): survival, the next
// discrete state by inverse-CDF sampling over trpr, shock, cash in hand and the equations of the new period, from the
// uniforms (rrr, rrr1, rrr2) of period `it`.  False: the agent dies (the rest of its record stays NaN).
EGDST_DEV bool egdst_sim_transition(const egdst_ctx &cx, const PeriodVars &cur, PeriodVars &nx, int it, double rrr, double rrr1, double rrr2,
                                    double &mu, double &sigma, double *eqs) {
    if (rrr2 > survival(&cx, &cur)) return false;
    nx = cur;
    nx.it = it;
    nx.savings = cur.savings;
    int chosen = -1, lastfeas = -1;
    for (int ist1 = 0; ist1 < cx.nst; ist1++) {
#if EGDST_NCONT > 0
        {   // continuous states are carried by value: only the cells at their first grid point stand
            // for the discrete part of the state (egdst_simulator.c:268-271)
            bool first = true;
#pragma unroll
            for (int k = 0; k < EGDST_NCONT; k++) {
                const int j0 = egdst_contvar[k];
                if ((ist1 / (int)cx.stm[cx.nnst + j0]) % (int)cx.stm[j0] != 0) first = false;
            }
            if (!first) continue;
        }
#endif
        nx.ist = ist1;
        egdst_fill_state(&cx, &nx);
#if EGDST_NCONT > 0
        trpr_cont(&cx, &cur, &nx);  // exact next-period values of the continuous states
#endif
        if (!feasible(&cx, &nx)) continue;
        lastfeas = ist1;
        double pr;
#if EGDST_OPT_TRPRNOSH
        pr = trpr(&cx, &cur, &nx, 0);
#else
        mu = mu_param(&cx, &cur, &nx); sigma = sigma_param(&cx, &cur, &nx);
        nx.shock = (sigma <= 0) ? egdst_expectation(&cx, &cur, &nx) : egdst_cdfinv(rrr1, mu, sigma);
        pr = trpr(&cx, &cur, &nx, 0);
#endif
        rrr -= pr;
        if (rrr <= 0) { chosen = ist1; break; }
    }
    if (chosen < 0) chosen = lastfeas < 0 ? 0 : lastfeas;  // the reference runs off the end here
    nx.ist = chosen;
    egdst_fill_state(&cx, &nx);
#if EGDST_NCONT > 0
    trpr_cont(&cx, &cur, &nx);
#endif
#if EGDST_OPT_TRPRNOSH
    // shocks for the shock-independent case (egdst_simulator.c:292-298)
    mu = mu_param(&cx, &cur, &nx); sigma = sigma_param(&cx, &cur, &nx);
    nx.shock = (sigma <= 0) ? egdst_expectation(&cx, &cur, &nx) : egdst_cdfinv(rrr1, mu, sigma);
#endif
    nx.cash = cashinhand(&cx, &cur, &nx);
    eqs_sim(&cx, &cur, &nx, eqs);
    return true;
}

// Dynamic shared memory layout of egdst_k_simulate:
//   tile[warps][32*TS]                PB staged records per agent of the warp's tile
//   mom[nt][nso][3] + clean[nt]       (mom_smem) per-CTA moment accumulators, flushed once at the end
// Template parameters:
//   PHILOX  uniforms from Philox4x32-10 (else: the caller's randstream, egdst_simulator.c:259-261)
//   OUT     bit 0: write the sims array; bit 1: accumulate moments; bit 2 (smoothing images): choice draws, each period's
//           decision drawn from the choice probabilities of the solve (egdst_choice_weights) and the record that of the
//           drawn decision's choice cell; PB == 1 and !HDR only
//   HDR     single-vector launch whose per-cell headers and parameter values travel in the kernel arguments
//   PB      periods per write of the sims array:
//     1  one record (8*nso bytes) per agent and store pass; rows padded to an odd stride (conflict-free staging and
//        column walks), 8 warps per CTA, 4 CTAs/SM at 64 registers, the plain period order (below)
//     2  two consecutive periods of an agent are staged side by side and written together (nt even): the output
//        stream is 1.5e5 concurrent per-agent runs, and DRAM takes runs of 16*nso bytes much better than runs of 8*nso
//        (tools/micro/wpat.cu).  Rows are unpadded and column-rotated by (lane/4)%4 instead; 12 warps per CTA, 2
//        CTAs/SM at 80 registers, the software-pipelined period order, moments always in shared memory
// Period order: PB == 2 (NCONT == 0) runs the transition into period it+1 and the index-entry gather of its cell
// during period it, before the value, utility, moments and store pass of period it, so that the gather's latency
// overlaps that work.  PB == 1 and the continuous-state branch keep the plain order (transition into period it, then
// its policy): pipelined, PB == 1 spills at 64 registers, and at 80 registers the occupancy lost costs more than the
// overlap gains.
template <bool PHILOX, int OUT, bool HDR, int PB>
__global__ void __launch_bounds__(PB == 2 ? EGDST_SIM_WIDE : EGDST_SIM_BLOCK, PB == 2 ? 2 : EGDST_SIM_MINBLOCKS)
egdst_k_simulate(EgdstDev P, EgdstSimArgs S, const EGDST_GRID_CONSTANT EgdstSimHdrs H) {
    EGDST_DYN_SMEM(double, egdst_sim_smem);
    constexpr int NSO = EGDST_NSIMOUT_MAX;   // the model image fixes nsimout (checked on the host)
    constexpr int W = PB * NSO;              // doubles per staged row (one agent)
    constexpr bool SWZ = PB == 2;
    constexpr int TS = SWZ ? W : (W | 1);
    constexpr int WPB = (PB == 2 ? EGDST_SIM_WIDE : EGDST_SIM_BLOCK) / 32;
    constexpr bool SIMS = (OUT & 1) != 0, MOM = (OUT & 2) != 0, DRAW = (OUT & 4) != 0;
    constexpr bool PIPE = PB == 2 && EGDST_NCONT == 0;  // pipelined period order
    static_assert(!DRAW || (PB == 1 && !HDR && EGDST_SMOOTHING && EGDST_NCONT == 0), "choice draws: plain period order, choice cells in global memory");
    // position of column j in the row of the agent staged by lane l: rotated rows spread a column over the banks
#define EGDST_TILE_POS(l, j) ((l) * TS + (SWZ ? (((j) + (((l) >> 2) & 3) >= W) ? (j) + (((l) >> 2) & 3) - W : (j) + (((l) >> 2) & 3)) : (j)))
    // blockIdx.y walks the parameter vectors of a batched sweep: same agents and shocks under every vector,
    // per-vector output blocks (sims [nvec][nsimout,nt,nsim], moments [nvec][3,nsimout,nt])
    const int ivec = S.ivec + blockIdx.y;
    egdst_ctx cx; egdst_load_ctx(P, ivec, cx);
    cx.status = 0;
#if EGDST_NCONT > 0
    cx.byval = 1;  // model functions read the exact continuous state from curr->st (egdst_simulator.c:91-92)
#endif
    if (HDR) {
#pragma unroll
        for (int i = 0; i < EGDST_NPARAM; i++) cx.param[i] = S.param[i];
    }
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int nt = P.NT;
    double *sims = SIMS ? S.sims + (size_t)blockIdx.y * NSO * nt * S.nsim : (double *)0;
    double *gmom = MOM ? S.moments + (size_t)blockIdx.y * NSO * nt * 3 : (double *)0;
    double *tile = egdst_sim_smem + (size_t)w * 32 * TS;
    double *smom = egdst_sim_smem + (size_t)WPB * 32 * TS;                    // [nt][NSO][3] when mom_smem
    int *clean_s = reinterpret_cast<int *>(smom + (size_t)nt * NSO * 3);      // [nt] clean tiles per period
    const bool momsm = MOM && S.mom_smem;
    const double NaN = EGDST_NAN;
    const int ntiles = (S.nsim + 31) / 32;
#ifndef EGDST_HOSTEMU
    const unsigned long long l2keep = egdst_policy_evict_last();
#else
    const unsigned long long l2keep = 0ULL;
#endif
    if (H.tabs_ok) { cx.stm = H.stm; cx.states = H.states; cx.decisions = H.decisions; }
    if (momsm) {
        for (int i = threadIdx.x; i < nt * NSO * 3; i += blockDim.x) smom[i] = 0.0;
        for (int i = threadIdx.x; i < nt; i += blockDim.x) clean_s[i] = 0;
        __syncthreads();
    }
    const size_t rowpitch = (size_t)nt * NSO;  // doubles between the records of consecutive agents
    // persistent: every warp strides over tiles of 32 agents and walks each tile through all periods
    for (int tileidx = blockIdx.x * WPB + w; tileidx < ntiles; tileidx += gridDim.x * WPB) {
        const int isim = tileidx * 32 + lane;
        const bool live_lane = isim < S.nsim;
        PeriodVars cur; cur.it = 0; cur.ist = 0; cur.id = 0; cur.cash = 0; cur.savings = 0; cur.shock = NaN;
#pragma unroll
        for (int i = 0; i < EGDST_NNST; i++) cur.st[i] = 0;
#pragma unroll
        for (int i = 0; i < EGDST_NND; i++) cur.dc[i] = 0;
        double mu = NaN, sigma = NaN, c = 0, vf = 0, uu = 0, bb = 0;  // uu, bb: utility and discount factor of the record
        double eqs[EGDST_NREQ > 0 ? EGDST_NREQ : 1];
        int state = live_lane ? 0 : 2;  // 0 alive, 1 dead/skipped (NaN rows), 2 no agent
        if (live_lane) {
            const int ist0 = (int)S.init[isim] - 1;
            const double m0 = S.init_m0[isim];
            if (ist0 < 0 || ist0 >= cx.nst || m0 < cx.a0 || m0 > cx.mmax) state = 1;  // egdst_simulator.c:215-216
            else { cur.ist = ist0; cur.cash = m0; egdst_fill_state(&cx, &cur); if (!feasible(&cx, &cur)) state = 1; }
        }
        // Uniforms are drawn one period ahead of the transition that uses them: the Philox rounds are independent of
        // the agent's state, so their integer pipeline work overlaps the table gathers.  The plain order steps into
        // period it during period it and draws the uniforms of it+1; the pipelined order steps into it+1 and draws it+2.
        unsigned pr0 = 0, pr1 = 0, pr2 = 0, pr3 = 0;
        const unsigned long long gid = (unsigned long long)(S.agent0 + isim);
        if (PHILOX && nt > 1)
            egdst_philox4x32((unsigned)gid, (unsigned)(gid >> 32), 1u, 0u, (unsigned)S.seed, (unsigned)(S.seed >> 32), pr0, pr1, pr2, pr3);
        const double *rs = PHILOX ? (const double *)0 : S.randstream + (S.rndtype == 1 ? 0 : (size_t)4 * nt * isim);
        // DRAW: the choice uniform of period it is word 3 of the Philox block of (gid, it), whose words 0-2 feed the
        // transition into it (period 0: a block of its own), or slot 3*(nt-1)+it of the agent's randstream block
        unsigned pw3 = 0;
        if (DRAW && PHILOX) {
            unsigned q0, q1, q2;
            egdst_philox4x32((unsigned)gid, (unsigned)(gid >> 32), 0u, 0u, (unsigned)S.seed, (unsigned)(S.seed >> 32), q0, q1, q2, pw3);
        }
        // cooperative write of the tile: lane = (agent sub-index, 16-byte piece); running pointer over the periods
        constexpr bool VEC = (W & 1) == 0 && W <= 32;
        constexpr int SL = W / 2 <= 8 ? 8 : 16, APT = 32 / SL;
        const int wk = lane % SL, wa0 = lane / SL;
        const int na = S.nsim - tileidx * 32 < 32 ? S.nsim - tileidx * 32 : 32;
        const bool vecok = VEC && (((size_t)sims & 15) == 0);
        double *wdst = SIMS ? sims + (size_t)tileidx * 32 * rowpitch + (vecok ? (size_t)wa0 * rowpitch + 2 * wk : 0) : (double *)0;
#if EGDST_NCONT == 0
        // PIPE: the index entry of the next record's cell (tabnext: its lookup goes through the tables), gathered one
        // period ahead so that it is in flight while the value, utility, moments and store pass of a period run
        EgdstLutEntry ent;
        bool tabnext = false;
        auto lookup_begin = [&](int p, const PeriodVars &v) {
            const int cell = egdst_cell(P, ivec, p, v.ist);
            const int nmraw = HDR ? H.h[p * cx.nst + v.ist].n : P.mlen[cell];
            const int nm = HDR ? (nmraw & ~EGDST_HDR_NOTAB) : nmraw;
            const bool tabok = HDR ? (nmraw & EGDST_HDR_NOTAB) == 0 : P.tabOk[cell] != 0;
            tabnext = egdst_sim_tab(P, nm, tabok);
            if (tabnext) ent = egdst_lut_entry<true>(P, cell, v.cash, l2keep);
        };
        if (PIPE && state == 0) {  // period 0 has no transition into it
            eqs_sim(&cx, &cur, (const PeriodVars *)0, eqs);
            lookup_begin(0, cur);
        }
#endif
        for (int it = 0; it < nt; it++) {
            const unsigned cr0 = pr0, cr1 = pr1, cr2 = pr2, cr3 = it > 0 ? pr3 : pw3;
            if (PHILOX && (PIPE ? it + 2 < nt : it > 0 && it + 1 < nt))
                egdst_philox4x32((unsigned)gid, (unsigned)(gid >> 32), (unsigned)(it + (PIPE ? 2 : 1)), 0u, (unsigned)S.seed, (unsigned)(S.seed >> 32), pr0, pr1, pr2, pr3);
            // the record of this period is staged in the tile (PB == 2: odd periods go to the second half of the agent's row)
            const int half = (PB == 2) ? (it & 1) : 0;
            const int hoff = half * NSO;
#define EGDST_REC(j) tile[EGDST_TILE_POS(lane, hoff + (j))]
            int rstate;  // state of this period's record; PIPE: `state` moves on to the next period
            if (!PIPE) {
                if (state == 0 && it > 0) {
                    double rrr, rrr1, rrr2;
                    if (!PHILOX) {
                        const double *r3 = rs + (size_t)3 * (it - 1);
                        rrr = r3[0]; rrr1 = r3[1]; rrr2 = r3[2];
                    } else {
                        rrr = egdst_u01(cr0); rrr1 = egdst_u01(cr1); rrr2 = egdst_u01(cr2);
                    }
                    PeriodVars nx;
                    if (!egdst_sim_transition(cx, cur, nx, it, rrr, rrr1, rrr2, mu, sigma, eqs)) state = 1;  // death: the rest of the record stays NaN
                    else cur = nx;
                } else if (state == 0) {
                    eqs_sim(&cx, &cur, (const PeriodVars *)0, eqs);
                }
#if EGDST_NCONT > 0
                if (state == 0) {
                    // Continuous states (egdst_simulator.c:309-365): consumption and value are the multilinear mix of the
                    // policies of the 2^NCONT surrounding grid cells (weights <= 0 are skipped, as there); the recorded
                    // cell and discrete decision are those of the corner at which the cumulated weight passes one half.
                    // The reference never assigns the value column on this branch (policy(...,0) skips it); here it is
                    // the same mix of the corner values.  At it == 0 the cell index of `init` may point at any grid point
                    // of a continuous state: its grid part is removed before the corners are addressed (the reference
                    // adds the corner offset on top of it and leaves the table, egdst_simulator.c:313).
                    int j1[EGDST_NCONT], stride[EGDST_NCONT];
                    double wlo[EGDST_NCONT], whi[EGDST_NCONT];
                    int base = cur.ist;
#pragma unroll
                    for (int k = 0; k < EGDST_NCONT; k++) {
                        const int j0 = egdst_contvar[k], n = (int)cx.stm[j0];
                        const double *g = egdst_contgrid(k);
                        const double x = cur.st[j0];
                        stride[k] = (int)cx.stm[cx.nnst + j0];
                        base -= ((cur.ist / stride[k]) % n) * stride[k];
                        j1[k] = egdst_gridcell(x, g, n);
                        wlo[k] = (g[j1[k] + 1] - x) / (g[j1[k] + 1] - g[j1[k]]);
                        whi[k] = (x - g[j1[k]]) / (g[j1[k] + 1] - g[j1[k]]);
                    }
                    double wc = 0, wvf = 0, rr = .5;
                    int ist1 = -1, id1 = 0, istlast = -1, idlast = 0;
                    bool ok = true;
                    for (int ii = 0; ii < (1 << EGDST_NCONT) && ok; ii++) {
                        double wt = 1;
                        int ist = base;
#pragma unroll
                        for (int k = 0; k < EGDST_NCONT; k++) {
                            const int up = (ii >> k) & 1;
                            wt *= up ? whi[k] : wlo[k];
                            ist += stride[k] * (j1[k] + up);
                        }
                        if (!(wt > 0)) continue;
                        PeriodVars pv = cur;
                        pv.ist = ist;
                        double cc, vv;
                        ok = egdst_sim_policy_cell(P, cx, egdst_cell(P, ivec, it, ist), pv, l2keep, cc, vv);
                        if (!ok) break;
                        wc += cc * wt;
                        wvf += vv * wt;
                        rr -= wt;
                        istlast = ist; idlast = pv.id;
                        if (rr < 0 && ist1 == -1) { ist1 = ist; id1 = pv.id; }
                    }
                    if (!ok || istlast < 0) state = 1;
                    else {
                        if (ist1 < 0) { ist1 = istlast; id1 = idlast; }
                        c = MIN(wc, cur.cash - cx.a0);
                        cur.savings = cur.cash - c;
                        vf = wvf;
                        cur.ist = ist1;
                        cur.id = id1;
                        egdst_fill_decision(&cx, &cur);
                        uu = utility(&cx, &cur, c); bb = discount(&cx, &cur);
                    }
                }
#else
#if EGDST_SMOOTHING
                if (DRAW) {
                    if (state == 0) {
                        // choice draw: P_d(cash) as the solve weighs decision d, d = the first available decision whose
                        // cumulative probability reaches u, and the policy and value of d's choice cell by the rules of
                        // the modal branch below (interpolation, exact value below M[1])
                        const int cell = egdst_cell(P, ivec, it, cur.ist);
                        EgdstChoiceVals cv;
                        egdst_choice_values(P, &cx, cell, cur, cv);
                        double pe[EGDST_SMOOTH_MAXND], ssum, wmax;
                        for (int d = 0; d < cx.nd; d++) pe[d] = 0.0;
                        egdst_choice_weights(cx.nd, cv, P.sigmaEps, ssum, wmax, [&](int d, double e) { pe[d] = e; });
                        const double u = PHILOX ? egdst_u01(cr3) : rs[(size_t)3 * (nt - 1) + it];
                        int dr = -1;
                        double cum = 0.0;
                        for (int d = 0; d < cx.nd; d++) {
                            if (!(cv.avail >> d & 1u)) continue;
                            cum += pe[d] / ssum;
                            dr = d;  // the last available decision if rounding keeps the sum below u
                            if (cum >= u) break;
                        }
                        if (dr < 0) { state = 1; }  // no decision available in (it, ist)
                        else {
                            const int dcell = egdst_dcell(P, cell, dr);
                            EgdstInterval iv;
                            egdst_sim_interval(P, dcell, P.mlen[dcell], P.tabOk[dcell] != 0, cur.cash, l2keep, iv);
                            double wl, wr;
                            egdst_sim_weights(iv, cur.cash, wl, wr);
                            c = iv.c1 * wl + iv.c0 * wr;
                            cur.savings = cur.cash - c;
                            cur.id = dr;
                            egdst_fill_decision(&cx, &cur);
                            const double evf = P.evf[dcell], M1 = egdst_colM(P, dcell)[1];
                            uu = utility(&cx, &cur, c); bb = discount(&cx, &cur);
                            if (cur.cash < M1 && evf > -EGDST_INF) vf = uu + bb * evf;
                            else vf = iv.v1 * wl + iv.v0 * wr;
                        }
                    }
                } else
#endif
                if (state == 0) {
                    // policy (egdst_simulator.c:145-199)
                    const int cell = egdst_cell(P, ivec, it, cur.ist);
                    const EgdstCellHdr *hc = H.h + it * cx.nst + cur.ist;
                    const int nmraw = HDR ? hc->n : P.mlen[cell];
                    const int nm = HDR ? (nmraw & ~EGDST_HDR_NOTAB) : nmraw;
                    const bool tabok = HDR ? (nmraw & EGDST_HDR_NOTAB) == 0 : P.tabOk[cell] != 0;
                    EgdstInterval iv;
                    if (!egdst_sim_interval(P, cell, nm, tabok, cur.cash, l2keep, iv)) { state = 1; }
                    else {
                        double wl, wr;
                        egdst_sim_weights(iv, cur.cash, wl, wr);
                        c = iv.c1 * wl + iv.c0 * wr;
                        cur.savings = cur.cash - c;
                        const int nth = HDR ? hc->nth : P.thlen[cell];
                        if (HDR && nth <= EGDST_SIM_TH8) cur.id = egdst_policy_decision(cur.cash, hc->th, hc->dd, nth);
                        else cur.id = egdst_policy_decision(cur.cash, P.thTH + (size_t)cell * cx.nthrhmax, P.thD + (size_t)cell * cx.nthrhmax, nth);
                        egdst_fill_decision(&cx, &cur);
                        const double evf = HDR ? hc->evf : P.evf[cell];  // == V(row 0)
                        const double M1 = HDR ? hc->M1 : egdst_colM(P, cell)[1];
                        uu = utility(&cx, &cur, c); bb = discount(&cx, &cur);  // output columns 9, 10; shared with the exact value below
                        if (cur.cash < M1 && evf > -EGDST_INF) vf = uu + bb * evf;
                        else vf = iv.v1 * wl + iv.v0 * wr;
                    }
                }
#endif
                if (state == 0) {
                    EGDST_REC(0) = cur.cash; EGDST_REC(1) = c; EGDST_REC(2) = cur.savings; EGDST_REC(3) = vf; EGDST_REC(4) = (double)cur.id; EGDST_REC(5) = (double)cur.ist;
                    EGDST_REC(6) = mu; EGDST_REC(7) = sigma; EGDST_REC(8) = cur.shock; EGDST_REC(9) = uu; EGDST_REC(10) = bb;
#pragma unroll
                    for (int i = 0; i < EGDST_NNST; i++) EGDST_REC(11 + i) = cur.st[i];
#pragma unroll
                    for (int i = 0; i < EGDST_NND; i++) EGDST_REC(11 + EGDST_NNST + i) = cur.dc[i];
#pragma unroll
                    for (int i = 0; i < EGDST_NREQ; i++) EGDST_REC(11 + EGDST_NNST + EGDST_NND + i) = eqs[i];
                } else {
#pragma unroll
                    for (int j = 0; j < NSO; j++) EGDST_REC(j) = NaN;
                }
                rstate = state;
            }
#if EGDST_NCONT == 0
            else {
                // Pipelined order: (1) the policy of period it from the index entry gathered during period it-1, and
                // the record columns that do not wait for the value; (2) the transition into period it+1 and the
                // index-entry gather of its cell; (3) value, utility and discount of period it.  Only independent
                // work moves, every expression is the one of the plain order: the records are the same to the bit.
                double evf = 0.0, vlin = 0.0;
                bool vexact = false;
                if (state == 0) {
                    const int cell = egdst_cell(P, ivec, it, cur.ist);
                    const EgdstCellHdr *hc = H.h + it * cx.nst + cur.ist;
                    const int nm = HDR ? (hc->n & ~EGDST_HDR_NOTAB) : P.mlen[cell];
                    EgdstInterval iv;
                    if (nm < 2) { state = 1; }
                    else {
                        if (tabnext) egdst_cell_lookup_finish(P, cell, cur.cash, nm, ent, iv, l2keep);
                        else egdst_sim_interval(P, cell, nm, false, cur.cash, l2keep, iv);
                        double wl, wr;
                        egdst_sim_weights(iv, cur.cash, wl, wr);
                        c = iv.c1 * wl + iv.c0 * wr;
                        cur.savings = cur.cash - c;
                        const int nth = HDR ? hc->nth : P.thlen[cell];
                        if (HDR && nth <= EGDST_SIM_TH8) cur.id = egdst_policy_decision(cur.cash, hc->th, hc->dd, nth);
                        else cur.id = egdst_policy_decision(cur.cash, P.thTH + (size_t)cell * cx.nthrhmax, P.thD + (size_t)cell * cx.nthrhmax, nth);
                        egdst_fill_decision(&cx, &cur);
                        evf = HDR ? hc->evf : P.evf[cell];  // == V(row 0)
                        const double M1 = HDR ? hc->M1 : egdst_colM(P, cell)[1];
                        vexact = cur.cash < M1 && evf > -EGDST_INF;  // the value is exact below M[1], else interpolated
                        vlin = iv.v1 * wl + iv.v0 * wr;
                    }
                }
                rstate = state;
                if (state == 0) {
                    EGDST_REC(0) = cur.cash; EGDST_REC(1) = c; EGDST_REC(2) = cur.savings; EGDST_REC(4) = (double)cur.id; EGDST_REC(5) = (double)cur.ist;
                    EGDST_REC(6) = mu; EGDST_REC(7) = sigma; EGDST_REC(8) = cur.shock;
#pragma unroll
                    for (int i = 0; i < EGDST_NNST; i++) EGDST_REC(11 + i) = cur.st[i];
#pragma unroll
                    for (int i = 0; i < EGDST_NND; i++) EGDST_REC(11 + EGDST_NNST + i) = cur.dc[i];
#pragma unroll
                    for (int i = 0; i < EGDST_NREQ; i++) EGDST_REC(11 + EGDST_NNST + EGDST_NND + i) = eqs[i];
                } else {
#pragma unroll
                    for (int j = 0; j < NSO; j++) EGDST_REC(j) = NaN;
                }
                PeriodVars nx;
                bool stepped = false;
                if (state == 0 && it + 1 < nt) {
                    double rrr, rrr1, rrr2;
                    if (!PHILOX) {
                        const double *r3 = rs + (size_t)3 * it;
                        rrr = r3[0]; rrr1 = r3[1]; rrr2 = r3[2];
                    } else {
                        rrr = egdst_u01(cr0); rrr1 = egdst_u01(cr1); rrr2 = egdst_u01(cr2);
                    }
                    stepped = egdst_sim_transition(cx, cur, nx, it + 1, rrr, rrr1, rrr2, mu, sigma, eqs);
                    if (!stepped) state = 1;  // death in period it+1; this period's record stands
                    else lookup_begin(it + 1, nx);
                }
                if (rstate == 0) {
                    uu = utility(&cx, &cur, c); bb = discount(&cx, &cur);
                    vf = vexact ? uu + bb * evf : vlin;
                    EGDST_REC(3) = vf; EGDST_REC(9) = uu; EGDST_REC(10) = bb;
                }
                if (stepped) cur = nx;
            }
#endif
#undef EGDST_REC
            const bool clean = MOM && __all_sync(EGDST_FULL, rstate == 0) && it > 0;  // no NaN record in the tile
            __syncwarp();
            if (SIMS && (PB == 1 || half == 1)) {
                if (vecok) {
                    // 16-byte pieces, SL slots per agent (W/2 used): agent = APT*t + lane/SL, piece = lane%SL
                    if (wk < W / 2) {
                        if (na == 32) {
#pragma unroll
                            for (int t = 0; t < 32 / APT; t++) {
                                const int a = APT * t + wa0;
                                EGDST_STREAM_STORE2(wdst + (size_t)t * APT * rowpitch, make_double2(tile[EGDST_TILE_POS(a, 2 * wk)], tile[EGDST_TILE_POS(a, 2 * wk + 1)]));
                            }
                        } else {
                            for (int t = 0; APT * t + wa0 < na; t++) {
                                const int a = APT * t + wa0;
                                EGDST_STREAM_STORE2(wdst + (size_t)t * APT * rowpitch, make_double2(tile[EGDST_TILE_POS(a, 2 * wk)], tile[EGDST_TILE_POS(a, 2 * wk + 1)]));
                            }
                        }
                    }
                } else {
                    for (int e = lane; e < na * W; e += 32) {
                        const int a = e / W, j = e - a * W;
                        wdst[(size_t)a * rowpitch + j] = tile[EGDST_TILE_POS(a, j)];
                    }
                }
                wdst += W;
            }
            if (MOM) {
                // column sums over the tile: lanes split the NSO columns (two half-tiles when 2*NSO <= 32)
                constexpr int HV = (2 * NSO <= 32) ? 2 : 1;
                double s1 = 0, s2 = 0, n = 0;
                if (lane < HV * NSO) {
                    const int j = lane % NSO, h = lane / NSO;
                    const int a_lo = h * (32 / HV), cj = hoff + j;
                    if (clean) {
                        // every agent of the tile is alive: sum without NaN tests (warp-uniform branch); a column that
                        // holds a NaN after all (user equations) shows up as a NaN sum and is redone below
#pragma unroll
                        for (int a = 0; a < 32 / HV; a++) { const double x = tile[EGDST_TILE_POS(a_lo + a, cj)]; s1 += x; s2 = fma(x, x, s2); }
                        n = 32 / HV;
                    }
                    if (!clean || s1 != s1 || s2 != s2) {
                        s1 = 0; s2 = 0; n = 0;
                        for (int a = 0; a < 32 / HV; a++) { const double x = tile[EGDST_TILE_POS(a_lo + a, cj)]; if (x == x) { s1 += x; s2 = fma(x, x, s2); n += 1; } }
                    }
                }
                if (HV == 2) {
                    s1 += __shfl_down_sync(EGDST_FULL, s1, NSO);
                    s2 += __shfl_down_sync(EGDST_FULL, s2, NSO);
                    n += __shfl_down_sync(EGDST_FULL, n, NSO);
                }
                // a clean tile adds 32 to the count of every column: one integer atomic per tile instead of NSO
                // floating-point ones (clean_s[it], folded into the counts at the final flush)
                const bool cntint = momsm && clean && __all_sync(EGDST_FULL, lane >= NSO || n == 32.0);
                if (momsm) {
                    if (cntint && lane == 0) atomicAdd(clean_s + it, 1);
                    if (lane < NSO && n > 0) {
                        double *d = smom + ((size_t)it * NSO + lane) * 3;
                        atomicAdd(d + 0, s1); atomicAdd(d + 1, s2);
                        if (!cntint) atomicAdd(d + 2, n);
                    }
                } else if (lane < NSO && n > 0) {
                    double *d = gmom + ((size_t)it * NSO + lane) * 3;
                    atomicAdd(d + 0, s1); atomicAdd(d + 1, s2); atomicAdd(d + 2, n);
                }
            }
            __syncwarp();
        }
    }
    if (momsm) {
        __syncthreads();
        for (int i = threadIdx.x; i < nt * NSO * 3; i += blockDim.x) {
            double v = smom[i];
            if (i % 3 == 2) v += 32.0 * clean_s[i / (3 * NSO)];
            if (v != 0.0) atomicAdd(gmom + i, v);
        }
    }
}
#undef EGDST_TILE_POS

