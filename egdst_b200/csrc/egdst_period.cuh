// egdst_period.cuh -- the backward induction as ONE kernel: solver() and egmbellman() of the reference
// (egdst_solver.c:258-339, 370-752) with the period loop on the device.
//
//   for it = T-t0 .. 0:                                                      egdst_solver.c:288
//       terminal grid                      | seed -> EGM (+ re-send passes)   :452-475 | :477-665
//       secondary envelope (only if a decision's grid folded back)            :668, 776-913
//       primary envelope over decisions, thresholds, cell header              :720-730, 1165-1550
//       lookup tables of the new cells (read by period it-1 and by the simulator) + housekeeping of period it-1
//
// Scope GRID: a cooperative launch of one resident wave, every CTA takes part in every phase, phases separated by a
// grid barrier (one model or a few vectors).  Scope CTA: every CTA walks its own parameter vector through all periods,
// phases separated by egdst_cta_sync() (sweeps of many small models: no launches and no inter-CTA waits at all).
// Period t reads the cells of t+1 where saveoutput left them (the arena), exactly as the reference does (:931-951).
#pragma once

#include "egdst_envelope.cuh"
#include "egdst_solver.cuh"

// phase boundary: team barrier, and (measurement aid, GRID scope) the device time since the previous boundary
#ifndef EGDST_HOSTEMU
EGDST_DEV unsigned long long egdst_globaltimer() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#else
EGDST_DEV unsigned long long egdst_globaltimer() { return 0ULL; }
#endif
template <bool GRID>
EGDST_DEV bool egdst_phase_end(const EgdstDev &P, const EgdstTeam &T, int phase, unsigned long long &t0) {
    const bool ok = egdst_team_sync<GRID>(P);
    if (P.phase_ns && T.rank == 0 && threadIdx.x == 0 && (GRID || T.v0 == 0)) {  // CTA scope: the CTA of vector 0 reports
        const unsigned long long t = egdst_globaltimer();
        P.phase_ns[phase] += t - t0;
        t0 = t;
    }
    if (!ok && threadIdx.x == 0) egdst_fail(P, T.v0, EGDST_ERR_BARRIER, -1, -1, -1);
    return ok;
}
#define EGDST_PHASE_END(phase) do { if (!egdst_phase_end<GRID>(P, T, phase, t0)) return; } while (0)

#ifdef EGDST_HOSTEMU
// debugging aid of the host emulator: the per-decision point lists of one period, before and after the secondary envelope
static void egdst_debug_dump(const EgdstDev &P, int it, const char *tag) {
    const char *e = getenv("EGDST_DEBUG_DUMP_IT");
    if (!e || atoi(e) != it || threadIdx.x != 0) return;
    for (int sd = 0; sd < P.nvec * P.cx.nst * P.cx.nd; sd++) {
        char name[256];
        snprintf(name, sizeof(name), "/tmp/egdst_pt_%s_sd%d.bin", tag, sd);
        FILE *f = fopen(name, "wb");
        if (!f) continue;
        const int n = P.ptN[sd], nf = P.nfold[sd];
        const double ev = P.evfa0[sd];
        fwrite(&n, sizeof(int), 1, f); fwrite(&nf, sizeof(int), 1, f); fwrite(&ev, sizeof(double), 1, f);
        fwrite(P.ptX + (size_t)sd * P.gcap, sizeof(double), n, f);
        fwrite(P.ptC + (size_t)sd * P.gcap, sizeof(double), n, f);
        fwrite(P.ptV + (size_t)sd * P.gcap, sizeof(double), n, f);
        fwrite(P.runStart + (size_t)sd * (P.gcap + 1), sizeof(int), nf + 2, f);
        fclose(f);
    }
}
#define EGDST_DEBUG_DUMP(tag) egdst_debug_dump(P, it, tag)
#else
#define EGDST_DEBUG_DUMP(tag)
#endif

// Shared memory of the solve kernels (dynamic): one scratch area that the phases use in turn -- they never overlap in
// time within a CTA -- followed by the per-CTA table of quadrature shocks and node probabilities.
template <int BS>
struct EgdstScratch {
    static constexpr size_t a_ = sizeof(EgdstSeedShared) > sizeof(EgdstEgmShared<BS>) ? sizeof(EgdstSeedShared) : sizeof(EgdstEgmShared<BS>);
    static constexpr size_t b_ = sizeof(EgdstEnvShared<BS>) > sizeof(EgdstRankShared<BS>) ? sizeof(EgdstEnvShared<BS>) : sizeof(EgdstRankShared<BS>);
    static constexpr size_t bytes = (((a_ > b_ ? a_ : b_) + 127) / 128) * 128;
};

// LOCK (WARP scope): all groups of the CTA start the phases of a period together; `live` = this group has a vector
// (groups without one only keep the barriers company).  Nothing else differs between the scopes.
#define EGDST_LOCKSTEP(k) do { if (LOCK && ((EGDST_LOCK_MASK >> (k)) & 1)) __syncthreads(); } while (0)
#ifndef EGDST_LOCK_MASK
#define EGDST_LOCK_MASK 0x01 /* measured: the warps of a CTA stay together on their own; one rendezvous per period bounds the drift */
#endif
template <bool GRID, int BS, bool LOCK>
EGDST_DEV void egdst_solve_team(const EgdstDev &P, const EgdstTeam &T, void *scratch, double *shsm, bool live) {
    const int N = P.N, B = blockDim.x, nd = P.cx.nd;
    // virtual blocks per job of the rank step and of the table build: sized for the usual list lengths (a decision
    // keeps at most N points plus the few the secondary envelope inserts); longer lists are covered by stride loops
    const int nptA1 = B / P.envA1parts;
    const int nvbA1 = GRID ? MIN((2 * P.gcap + nptA1 - 1) / nptA1, (N + 64 + nptA1 - 1) / nptA1 + 1) : 1;
    const int nvbA0 = GRID ? MIN((nd * P.gcap + B - 1) / B, (nd * (N + 64) + B - 1) / B + 1) : 1;
    // work items of the merge: enough to take the usual number of chunks at once; they loop over tickets for more
    const int nvbM1 = GRID ? MIN(P.chE, (N + 64 + B - 1) / B + 1) : 1;
    const int nvbM0 = GRID ? MIN(P.chE, (nd * (N + 64) + B - 1) / B + 1) : 1;
    int nvbT = GRID ? (P.lutcap + 1 + B - 1) / B : 1;
    if (GRID && T.nv * P.cx.nst * nvbT > 8 * T.size) nvbT = MAX(1, 8 * T.size / (T.nv * P.cx.nst));
    unsigned long long t0 = 0ULL;
    if (live) egdst_ph_cells(P, P.itStart, T);
    if (!egdst_team_sync<GRID>(P)) return;
    if (P.phase_ns) t0 = egdst_globaltimer();
    for (int it = P.itStart; it >= P.itStop; it--) {
        EGDST_LOCKSTEP(0);
        if (it == P.NT - 1) {
            if (live) egdst_ph_terminal(P, it, T);
            EGDST_PHASE_END(0);
        } else {
            if (live) egdst_ph_seed(P, it, T, scratch, shsm);
            EGDST_PHASE_END(1);
            EGDST_LOCKSTEP(1);
            for (int pass = 0; live; pass++) {
                egdst_ph_egm<BS>(P, it, T, pass, scratch, shsm);
                EGDST_PHASE_END(2);
                if ((GRID ? EGDST_LDCG(P.flags + 8 * T.slot + (pass % 3)) : *((volatile int *)(P.flags + 8 * T.slot + (pass % 3)))) == 0) break;  // no grid asked for a zero-consumption re-send
                egdst_ph_resend(P, it, T, pass, scratch, shsm);
                EGDST_PHASE_END(3);
            }
            EGDST_DEBUG_DUMP("raw");
            EGDST_LOCKSTEP(2);
            if (live && (GRID ? EGDST_LDCG(P.flags + 8 * T.slot + 3) : *((volatile int *)(P.flags + 8 * T.slot + 3))) != 0) {  // some decision's grid folded back: secondary envelope
                egdst_ph_envA<1, BS>(P, it, T, nvbA1, scratch);
                EGDST_PHASE_END(4);
                egdst_ph_envBC<1, BS>(P, it, T, nvbM1, scratch);
                EGDST_PHASE_END(4);
                EGDST_DEBUG_DUMP("env2");
            }
        }
        EGDST_LOCKSTEP(3);
        if (EGDST_SMOOTHING && live) egdst_ph_dsave(P, it, T);  // smoothing mode: keep the choice-specific tables (read by period it-1)
        if (live) egdst_ph_envA<0, BS>(P, it, T, nvbA0, scratch);
        EGDST_PHASE_END(5);
        EGDST_LOCKSTEP(4);
        if (live) egdst_ph_envBC<0, BS>(P, it, T, nvbM0, scratch);
        EGDST_PHASE_END(6);
        EGDST_LOCKSTEP(5);
        if (live) {
            egdst_ph_tab(P, it, T, nvbT);
            if (it > P.itStop) egdst_ph_cells(P, it - 1, T);
        }
        EGDST_PHASE_END(7);
    }
}

// GRID scope: cooperative launch, gridDim.x = one resident wave
__global__ void __launch_bounds__(EGDST_BLOCK, EGDST_SOLVE_MINB) egdst_k_solve_grid(EgdstDev P) {
    EGDST_DYN_SMEM(double, dyn);
    EgdstTeam T; T.rank = blockIdx.x; T.size = gridDim.x; T.v0 = 0; T.nv = P.nvec; T.slot = 0;
    egdst_solve_team<true, EGDST_BLOCK, false>(P, T, dyn, dyn + EgdstScratch<EGDST_BLOCK>::bytes / sizeof(double), true);
}
// CTA scope: CTA b solves vectors b, b + gridDim.x, ...  Narrow CTAs (EGDST_CTA_BLOCK threads): the jobs of a small
// model occupy a few dozen threads, and what hides the latency of its dependent phases is the number of vectors in
// flight per SM.  The small per-job state of a vector -- scan words, tickets, counters, flags, seeds -- is only ever
// touched by the vector's own CTA, so it lives in shared memory (syncOff >= 0: byte offset of that area in the dynamic
// shared memory): the atomics, polls and fences of the chained scans then never leave the SM.
template <class T_>
EGDST_DEV T_ *egdst_carve(unsigned char *&p, size_t n) { T_ *r = reinterpret_cast<T_ *>(p); p += ((n * sizeof(T_) + 15) / 16) * 16; return r; }
// the kernel-argument block with the per-job state of vector v redirected to the shared-memory area at p: index sd
// (and, for the primary jobs, sd0 + nsdv + ist) of the global arrays lands in the area
EGDST_DEV void egdst_redirect_state(EgdstDev &Q, const EgdstDev &P, int v, int slot, unsigned char *p) {
    const int nsdv = P.cx.nst * P.cx.nd, nst = P.cx.nst, sd0 = v * nsdv;
    Q.priSync0 = sd0 + nsdv - v * nst;
    Q.scanC = egdst_carve<unsigned long long>(p, (size_t)nsdv * P.chC) - (size_t)sd0 * P.chC;
    Q.scanE = egdst_carve<unsigned long long>(p, (size_t)(nsdv + nst) * P.chE) - (size_t)sd0 * P.chE;
    Q.seed = egdst_carve<double>(p, (size_t)nsdv * EGDST_SEEDW) - (size_t)sd0 * EGDST_SEEDW;
    Q.evfa0 = egdst_carve<double>(p, nsdv) - sd0;
    Q.tickC = egdst_carve<int>(p, 2 * nsdv) - 2 * sd0;
    Q.tickE = egdst_carve<int>(p, 2 * (nsdv + nst)) - 2 * sd0;
    Q.envNact = egdst_carve<int>(p, nsdv + nst) - sd0;
    Q.foldCnt = egdst_carve<int>(p, nsdv) - sd0;
    Q.lateN = egdst_carve<int>(p, nsdv) - sd0;
    Q.active = egdst_carve<int>(p, nsdv) - sd0;
    Q.ptN = egdst_carve<int>(p, nsdv) - sd0;
    Q.nfold = egdst_carve<int>(p, nsdv) - sd0;
    Q.flags = egdst_carve<int>(p, 8) - 8 * slot;
}
__global__ void __launch_bounds__(EGDST_CTA_BLOCK, EGDST_CTA_MINB) egdst_k_solve_cta(EgdstDev P, int syncOff) {
    EGDST_DYN_SMEM(double, dyn);
    for (int v = blockIdx.x; v < P.nvec; v += gridDim.x) {
        EgdstTeam T; T.rank = 0; T.size = 1; T.v0 = v; T.nv = 1; T.slot = 1 + v;
        EgdstDev Q = P;
        if (syncOff >= 0) egdst_redirect_state(Q, P, v, T.slot, reinterpret_cast<unsigned char *>(dyn) + syncOff);
        egdst_solve_team<false, EGDST_CTA_BLOCK, false>(Q, T, dyn, dyn + EgdstScratch<EGDST_CTA_BLOCK>::bytes / sizeof(double), true);
        egdst_cta_sync();
    }
}
// WARP scope: blockDim = (32, groups); warp y of CTA b solves vectors b*groups + y, (b + gridDim.x)*groups + y, ...
// Each warp has its own slice of the dynamic shared memory (groupBytes: scratch, shock table, per-vector state at
// syncOff).  Why not simply more 32-thread CTAs: the kernel's code is far larger than the SM's instruction cache, and
// independent CTAs drift apart until every warp of the SM fetches a different part of it (measured: instruction
// fetch, not issue or memory, bounds the CTA scope -- profiles/r02_batch_solve.md); here all warps of the SM walk
// through the same phase of the same period at the same time.
#define EGDST_WARP_GROUPS 32
__global__ void __launch_bounds__(32 * EGDST_WARP_GROUPS, 1) egdst_k_solve_warps(EgdstDev P, int syncOff, int groupBytes) {
    EGDST_DYN_SMEM(double, dyn);
    unsigned char *mine = reinterpret_cast<unsigned char *>(dyn) + (size_t)threadIdx.y * groupBytes;
    const int G = blockDim.y;
    for (int v0 = blockIdx.x * G; v0 < P.nvec; v0 += gridDim.x * G) {  // uniform over the CTA
        const int v = v0 + threadIdx.y;
        const bool live = v < P.nvec;
        EgdstTeam T; T.rank = live ? 0 : 1; T.size = 1; T.v0 = live ? v : 0; T.nv = 1; T.slot = 1 + T.v0;  // rank 1 of 1: no work items
        EgdstDev Q = P;
        egdst_redirect_state(Q, P, T.v0, T.slot, mine + syncOff);
        egdst_solve_team<false, 32, true>(Q, T, mine, reinterpret_cast<double *>(mine + EgdstScratch<32>::bytes), live);
        __syncthreads();
    }
}
// bytes of the per-vector state above
static inline size_t egdst_cta_sync_bytes(const EgdstDev &P) {
    const size_t nsdv = (size_t)P.cx.nst * P.cx.nd, nst = P.cx.nst;
    auto r16 = [](size_t b) { return ((b + 15) / 16) * 16; };
    return r16(8 * nsdv * P.chC) + r16(8 * (nsdv + nst) * P.chE) + r16(8 * nsdv * EGDST_SEEDW) + r16(8 * nsdv) + r16(4 * 2 * nsdv) + r16(4 * 2 * (nsdv + nst)) +
           r16(4 * (nsdv + nst)) + 5 * r16(4 * nsdv) + r16(4 * 8);
}

// Diagnostic entry (egdst_test_envelope2): the secondary envelope of given EGM points of decision id of state 0 (of a
// scratch solution object), as the period loop runs it: folds (egdst_solver.c:819) -> runs -> rank -> merge.  One CTA.
__global__ void __launch_bounds__(EGDST_BLOCK, EGDST_SOLVE_MINB) egdst_k_env2_only(EgdstDev P, int it, int n, int id) {
    EgdstTeam T; T.rank = 0; T.size = 1; T.v0 = 0; T.nv = 1; T.slot = 1;
    EGDST_DYN_SMEM(double, dyn);
    __shared__ int s_nf;
    egdst_cells_body(P, 0, it);
    if (threadIdx.x == 0) s_nf = 0;
    egdst_cta_sync();
    const int sd = id;  // ist = 0
    const double *X = P.ptX + (size_t)sd * P.gcap, *V = P.ptV + (size_t)sd * P.gcap;
    int *foldList = P.foldList + (size_t)sd * (P.gcap + 1);
    for (int p = 1 + threadIdx.x; p < n; p += blockDim.x)
        if (X[p - 1] > X[p] || V[p - 1] > V[p]) { const int k = atomicAdd(&s_nf, 1); foldList[k] = p; }
    egdst_cta_sync();
    const int nf = s_nf;
    egdst_fold_runs(P, sd, nf, n);
    if (threadIdx.x == 0) P.active[sd] = 1;
    for (int k = threadIdx.x; k < P.cx.nst * P.cx.nd; k += blockDim.x) if (k != sd) { P.active[k] = 0; P.nfold[k] = 0; P.ptN[k] = 0; }
    egdst_cta_sync();
    if (nf == 0) return;
    egdst_ph_envA<1, EGDST_BLOCK>(P, it, T, 1, dyn);
    egdst_cta_sync();
    egdst_ph_envBC<1, EGDST_BLOCK>(P, it, T, 1, dyn);
}
