// egdst_common.cuh -- device-side problem descriptor, launch macro and block/warp collectives.
#pragma once

#include "egdst_numerics.cuh"

#ifdef EGDST_HOSTEMU
// tools/hostemu: the kernels are compiled by g++ against an emulation of the CUDA execution model so that
// their logic can be debugged without a GPU.  Development aid only -- never loaded by the product.
#include "cuda_emul.h"
#define EGDST_BLOCK 64
#define EGDST_ENVW 64
#else
#include <cuda_runtime.h>
#define EGDST_BLOCK 256
#define EGDST_ENVW 256   /* envelope merge kernels: 8 positions per thread, chained across CTAs */
#define EGDST_LAUNCH(kernel, grid, block, smem, stream, ...) kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__)
#define EGDST_DYN_SMEM(type, name) extern __shared__ __align__(128) type name[]
#define EGDST_LDCG(p) __ldcg(p)
#define EGDST_GRID_CONSTANT __grid_constant__
#endif

#ifdef __CUDACC__
#define EGDST_DEV_M __device__ __forceinline__
#define EGDST_NOINLINE static __device__ __noinline__
#else
#define EGDST_DEV_M inline
#define EGDST_NOINLINE static __attribute__((noinline))
#endif

#define EGDST_FULL 0xffffffffu
#define EGDST_SEEDW 12
#define EGDST_NPHASE 8  /* terminal, seed, egm, resend, envelope2, rank, merge, tables */
#define EGDST_SHOCKTAB_BYTES (40 * 1024)  /* per-CTA table of quadrature shocks and node probabilities (dynamic shared memory) */
#ifdef EGDST_HOSTEMU
#define EGDST_SOLVE_MINB 1
#define EGDST_CTA_BLOCK 32
#define EGDST_CTA_MINB 1
#else
#ifndef EGDST_SOLVE_MINB
#define EGDST_SOLVE_MINB 3   /* CTAs per SM of the solve kernel (register budget 80) */
#endif
#ifndef EGDST_CTA_BLOCK
#define EGDST_CTA_BLOCK 64   /* threads per CTA in the vector-per-CTA scope */
#endif
#ifndef EGDST_CTA_MINB
#define EGDST_CTA_MINB 16
#endif
#endif
// taste-shock smoothing (extension; egdst_solver.cuh): a property of the model image (codegen emits 1 for models with sigma_eps > 0),
// so that the reference-parity images carry none of its code
#ifndef EGDST_SMOOTHING
#define EGDST_SMOOTHING 0
#endif
#define EGDST_MAXCAND 72   /* stage-0 bisection candidates: (mmax-a0)/2^k < TOLERANCE well before 72 halvings */
#define EGDST_ENV_STACK 24 /* crossing-chain stack (thresholds() recursion depth) */
#define EGDST_ENV_MARKW 32 /* 32*32 = 1024 functions (envelope2 runs) can be marked */

// raw-point flags written by the seed/EGM kernels
enum { EGDST_PT_OK = 0, EGDST_PT_C1NEG = 1, EGDST_PT_EVFINF = 2, EGDST_PT_CHECKSUM = 3, EGDST_PT_NONFINITE = 4, EGDST_PT_NONE = 5 };

// lookup tables of a solution cell (egdst_tables.cuh): 32-byte index entries, 64-byte interval records
struct EgdstLutEntry { int l, cnt; double m0, m1, m2; };                 // first row of the bucket, rows in it, their abscissas (+inf: none)
struct EgdstRow { double m, c, v, y; };                                   // row i of (M, C, V); y = RN(1/(M[i+1]-M[i])), 0 when not safely invertible / last row
struct EgdstInterval { double g0, g1, c0, c1, v0, v1, y, pad; };        // rows i, i+1 as the interpolations use them (two consecutive EgdstRow)
// the last interval of a cell and its image under the extrapolation transform tr(x - a0) (egdst_lib.c:179-206): what a
// lookup above the grid needs, without touching the tables; yt = RN(1/(t1-t0)), 0 when not safely invertible
struct EgdstCellTop { double g0, g1, c0, c1, v0, v1, y, t0, t1, yt; };

// Everything a kernel needs.  Leading dimension of every array is the parameter-vector index `ivec`
// (batched solves; nvec=1 for a single model).
struct EgdstDev {
    egdst_ctx cx;
    int NT, nvec, rowcap, gcap, N;  // rowcap = ngridmax+2 rows per arena column; gcap = ngridmax; N = ngridm
    const double *bparams;          // [nvec*NPARAM] or null
    const double *qw, *qz;          // quadrature weights, std-normal abscissas (cdfni applied) [ny]
    // solution arena
    double *arena;                  // [(nvec*NT*nst) * 4 * rowcap]  columns M,C,A,V
    int *mlen;                      // [nvec*NT*nst] rows incl. the a0 row (0 = no solution)
    double *thD, *thTH;             // [nvec*NT*nst * nthrhmax]
    int *thlen;                     // [nvec*NT*nst]
    double *evf;                    // [nvec*NT*nst]
    // per-period workspace, indexed by sd = (ivec*nst+ist)*nd+id
    int *active;                    // 1 if feasible(ist) && inchoiceset(id)
    double *seed;                   // [nsd*EGDST_SEEDW]: lim1,lim2,lim3,lim3p,k3,A(prev),nfirst,ncalls,baseA,baseM (egdst_solver.cuh)
    double *evfa0;                  // [nsd]
    double *ptX, *ptC, *ptV;        // [nsd*gcap] per-id point lists
    int *ptN, *nfold, *runStart;    // [nsd], [nsd], [nsd*(gcap+1)]
    // envelope scratch: secondary jobs use slot sd, primary jobs use slot nsd_total + (ivec*nst+ist)
    double *mgX; int *mgF, *mgK, *mgA;     // merged order, capacity envcap per slot
    double *outX, *outC, *outV;            // per-slot output staging, capacity envcap
    int envcap;
    int *status;                    // [nvec*4]: code, it, ist, id of the first error
    unsigned long long *units;      // [2*nvec] EGM grid points stored over all (it,ist,id): the solve work unit; then: late re-sends handled
    // chained scans across CTAs (decoupled look-back): state words per chunk, [ticket, done] counters per job;
    // zeroed at the start of every period by egdst_k_cells
    unsigned long long *scanC, *scanE;  // [nsd*chC] compaction, [nslot*chE] envelope merge
    int *tickC, *tickE;                 // [nsd*2], [nslot*2]
    int chC, chE;                       // chunks per job
    int envA1parts;                     // threads that share the runs of one point in the rank step of the secondary envelope (1 or 8)
    int *foldList, *foldCnt;            // [nsd*(gcap+1)] unordered fold positions, [nsd]
    int *envNact;                       // [nslot] active prefix length of the merged union (egdst_k_envA)
    int *lateN;                         // [nsd] first grid index whose evaluation asked for a zero-consumption re-send in this pass (INT_MAX: none)
    int *flags;                         // [(1+nvec)*8] per team: [0..2] re-sends pending after EGM pass k%3, [3] folds found in this period
    unsigned *bar;                      // grid barrier word of the cooperative solve kernel
    unsigned long long *phase_ns;       // [EGDST_NPHASE] device time per phase of the solve kernel (measurement aid; null = off)
    const struct EgdstDev *self;        // this block, in global memory (read by out-of-line device functions)
    double sigmaEps;                    // > 0: taste-shock smoothing (extension): scale of the extreme-value choice shocks
    int ncellMain;                      // nvec*NT*nst: the decision cells of the smoothing mode follow the solution cells in every per-cell array
    int priSync0;                       // index of the first primary-envelope job in the synchronisation arrays (scanE, tickE, envNact): nvec*nst*nd
    int itStop;                         // last period to solve (0; higher: test hook)
    int itStart;                        // period the backward induction starts from (NT-1; lower: test hook, cells of later periods are given)
    int egmP;                           // grid points per work item of the EGM phase (<= threads per CTA); slices = threads / egmP
    // per-cell lookup tables (egdst_tables.cuh)
    EgdstRow *tabRow;                   // [ncell*(tabcap+1)]
    EgdstCellTop *tabTop;               // [ncell]
    EgdstLutEntry *tabLut;              // [ncell*(lutcap+1)]
    int tabcap, lutcap, mbits;
    int *tabOk;                         // [ncell] != 0: the cell's grid is increasing, its tables may be used (egdst_tables.cuh)
};

EGDST_DEV int egdst_cell(const EgdstDev &P, int ivec, int it, int ist) { return (ivec * P.NT + it) * P.cx.nst + ist; }
EGDST_DEV int egdst_dcell(const EgdstDev &P, int cell, int id) { return P.ncellMain + cell * P.cx.nd + id; }  // choice-specific tables (smoothing mode)
EGDST_DEV int egdst_sd(const EgdstDev &P, int ivec, int ist, int id) { return (ivec * P.cx.nst + ist) * P.cx.nd + id; }
EGDST_DEV double *egdst_colM(const EgdstDev &P, int cell) { return P.arena + (size_t)cell * 4 * P.rowcap; }
EGDST_DEV double *egdst_colC(const EgdstDev &P, int cell) { return P.arena + ((size_t)cell * 4 + 1) * P.rowcap; }
EGDST_DEV double *egdst_colA(const EgdstDev &P, int cell) { return P.arena + ((size_t)cell * 4 + 2) * P.rowcap; }
EGDST_DEV double *egdst_colV(const EgdstDev &P, int cell) { return P.arena + ((size_t)cell * 4 + 3) * P.rowcap; }

EGDST_DEV void egdst_load_ctx(const EgdstDev &P, int ivec, egdst_ctx &cx) {
    cx = P.cx;
    if (P.bparams) for (int i = 0; i < EGDST_NPARAM; i++) cx.param[i] = P.bparams[(size_t)ivec * EGDST_NPARAM + i];
    cx.status = P.status ? P.status + 4 * ivec : 0;
}

// first error wins (soft errors keep the partial solution, like err[300] in the reference)
EGDST_DEV void egdst_fail(const EgdstDev &P, int ivec, int code, int it, int ist, int id) {
    int *s = P.status + 4 * ivec;
    if (atomicCAS(s, 0, code) == 0) { s[1] = it; s[2] = ist; s[3] = id; }
}

// ---- teams ------------------------------------------------------------------------------------
// The backward induction runs as ONE kernel (egdst_period.cuh).  A team is the set of CTAs that cooperate on the
// periods of a set of parameter vectors [v0, v0+nv):
//   GRID scope  every CTA of a cooperative launch (one resident wave) works on all vectors; the phases of a period
//               are separated by a grid-wide barrier                                  -- one large model, few vectors
//   CTA scope   one CTA owns one vector at a time and walks it through all periods; phases are separated by
//               egdst_cta_sync()                                                        -- sweeps of many small models
//   WARP scope  the CTA scope with a warp in the role of the CTA: the 32-thread "CTAs" of up to 32 vectors form one
//               real CTA (blockDim = (32, groups)) and start every phase together, so that all warps of an SM run
//               the same stretch of code at the same time (instruction-cache locality; egdst_period.cuh)
// Every phase is a loop `for (w = rank; w < nwork; w += size)` over work items, so the same code serves all of them.
struct EgdstTeam { int rank, size, v0, nv, slot; };

// barrier of the threads that work on one item: the CTA, or the warp where blockDim.y > 1 (WARP scope).  The phases
// only ever use threadIdx.x / blockDim.x, which is the thread's rank within that group in either case.
EGDST_DEV void egdst_cta_sync() {
#ifdef EGDST_NO_WARP_SCOPE
    __syncthreads();
#else
    if (blockDim.y == 1) __syncthreads(); else __syncwarp();
#endif
}

// Grid-wide barrier of a cooperative launch (all CTAs resident): CTA barrier, one thread arrives on a global word
// with release/acquire fences around it, CTA barrier (the scheme of cooperative_groups::grid_group::sync; the high
// bit of the word flips once per generation, so the counter never has to be reset).  The acquire side also
// invalidates this SM's L1, which is what lets the phases after the barrier read with plain cached loads the arrays
// that other CTAs rewrote.
// Returns false when the barrier was abandoned: polls are bounded (a protocol bug or a CTA that died must surface as
// an error status, never as a hung device); bar[1] is the abort flag every waiting CTA also watches.
#define EGDST_BARRIER_POLLS (1 << 24)
EGDST_DEV bool egdst_grid_barrier(unsigned *bar) {
    egdst_cta_sync();
#ifndef EGDST_HOSTEMU
    if (gridDim.x > 1) {
        __shared__ int s_ok;
        if (threadIdx.x == 0) {
            const unsigned nb = (blockIdx.x == 0) ? 0x80000000u - (gridDim.x - 1u) : 1u;
            __threadfence();
            const unsigned old = atomicAdd(bar, nb);
            int polls = 0, ok = 1;
            while ((((old ^ *((volatile unsigned *)bar)) & 0x80000000u) == 0u)) {
                if (((++polls) & 1023) == 0 && (polls >= EGDST_BARRIER_POLLS || *((volatile unsigned *)(bar + 1)) != 0u)) { *((volatile unsigned *)(bar + 1)) = 1u; ok = 0; break; }
            }
            __threadfence();
            s_ok = ok;
        }
        egdst_cta_sync();
        return s_ok != 0;
    }
#endif
    return true;
}
// work items of a phase: w = vb * njobs + j with j = (ivec - T.v0) * jobs_per_vector + jy; virtual blocks of a job are
// spread over the CTAs that run at the same time (chained scans wait on lower virtual blocks of the same job only)
EGDST_DEV void egdst_item(const EgdstTeam &T, int w, int jpv, int &ivec, int &jy, int &vb) {
    const int njobs = T.nv * jpv;
    vb = w / njobs;
    const int j = w - vb * njobs;
    ivec = T.v0 + j / jpv;
    jy = j - (j / jpv) * jpv;
}
template <bool GRID>
EGDST_DEV bool egdst_team_sync(const EgdstDev &P) {
    if (GRID) return egdst_grid_barrier(P.bar);
    egdst_cta_sync();
    return true;
}

// ---- warp / block collectives (shuffle based) -------------------------------------------------
EGDST_DEV double egdst_warp_sum(double v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(EGDST_FULL, v, o);
    return v;
}
EGDST_DEV int egdst_warp_min(int v) {
    for (int o = 16; o > 0; o >>= 1) { int w = __shfl_down_sync(EGDST_FULL, v, o); v = w < v ? w : v; }
    return v;
}
EGDST_DEV int egdst_warp_incl_scan(int v, int lane) {
    for (int o = 1; o < 32; o <<= 1) { int w = __shfl_up_sync(EGDST_FULL, v, o); if (lane >= o) v += w; }
    return v;
}
// 64-bit variant (two packed 32-bit counters share one scan): same barriers as egdst_block_excl_scan
EGDST_DEV long long egdst_warp_incl_scan64(long long v, int lane) {
    for (int o = 1; o < 32; o <<= 1) { long long w = __shfl_up_sync(EGDST_FULL, v, o); if (lane >= o) v += w; }
    return v;
}
EGDST_DEV long long egdst_block_excl_scan64(long long v, long long *sh, long long *total) {
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    long long inc = egdst_warp_incl_scan64(v, lane);
    if (lane == 31) sh[w] = inc;
    egdst_cta_sync();
    if (w == 0) {
        long long s = lane < nw ? sh[lane] : 0;
        long long si = egdst_warp_incl_scan64(s, lane);
        if (lane < nw) sh[lane] = si - s;
        if (lane == nw - 1) sh[nw] = si;
    }
    egdst_cta_sync();
    long long res = inc - v + sh[w];
    *total = sh[nw];
    egdst_cta_sync();
    return res;
}
EGDST_DEV int egdst_block_min(int v, int *sh) {  // sh: 32 ints; every thread gets the block minimum
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = egdst_warp_min(v);
    if (lane == 0) sh[w] = v;
    egdst_cta_sync();
    int r = sh[0];
    for (int k = 1; k < nw; k++) r = sh[k] < r ? sh[k] : r;
    egdst_cta_sync();
    return r;
}

// ---------------------------------------------------------------------------------------------
// Chained scan across the CTAs of one job (single-pass prefix sum with decoupled look-back, Merrill & Garland
// 2016).  Chunk ids are handed out by an atomic ticket, so a CTA only ever waits on CTAs that are already running.
// State word: bits 63..62 = 0 empty / 1 aggregate / 2 inclusive prefix; payload = two 31-bit fields (lo, hi).
// KIND 0: both fields add (grid points, thresholds).  KIND 1: lo adds until hi ("the savings grid stopped
// here", egdst_solver.c:1100) is set -- later chunks contribute nothing.  Polls are bounded: a protocol bug
// shows up as an error status, never as a hung device.
// ---------------------------------------------------------------------------------------------
#define EGDST_SCAN_AGG (1ULL << 62)
#define EGDST_SCAN_INC (2ULL << 62)
#define EGDST_SCAN_MASK ((1ULL << 62) - 1ULL)
#define EGDST_SCAN_POLLS (1 << 22)
EGDST_DEV unsigned long long egdst_scan_pack(int lo, int hi) { return (unsigned long long)(unsigned)lo | ((unsigned long long)(unsigned)hi << 31); }
EGDST_DEV int egdst_scan_lo(unsigned long long p) { return (int)(p & 0x7fffffffULL); }
EGDST_DEV int egdst_scan_hi(unsigned long long p) { return (int)((p >> 31) & 0x7fffffffULL); }
template <int KIND>
EGDST_DEV unsigned long long egdst_scan_combine(unsigned long long earlier, unsigned long long later) {
    if (KIND == 1) {
        if (egdst_scan_hi(earlier)) return earlier;
        return egdst_scan_pack(egdst_scan_lo(earlier) + egdst_scan_lo(later), egdst_scan_hi(later));
    }
    return egdst_scan_pack(egdst_scan_lo(earlier) + egdst_scan_lo(later), egdst_scan_hi(earlier) + egdst_scan_hi(later));
}
// Called by all 32 lanes of one warp.  Publishes this chunk's aggregate, returns the exclusive prefix over the
// earlier chunks and publishes the inclusive prefix.  The chunks of a phase finish at about the same time, so a chunk
// usually has to walk back over many aggregates before it meets an inclusive prefix: the state words of the next
// EGDST_SCAN_NW windows of 32 predecessors are requested together (independent loads, one round trip to L2), then
// resolved nearest first.
#define EGDST_SCAN_NW 8
template <int KIND>
EGDST_DEV unsigned long long egdst_lookback(volatile unsigned long long *st, int chunk, unsigned long long agg, int *err) {
    const int lane = threadIdx.x & 31;
    if (lane == 0 && chunk > 0) st[chunk] = EGDST_SCAN_AGG | agg;
    unsigned long long excl = 0ULL;
    bool done = false;
    for (int base = chunk - 1; base >= 0 && !done; base -= 32 * EGDST_SCAN_NW) {
        unsigned long long wv[EGDST_SCAN_NW];
#pragma unroll
        for (int r = 0; r < EGDST_SCAN_NW; r++) {
            const int idx = base - 32 * r - lane;
            wv[r] = idx >= 0 ? st[idx] : EGDST_SCAN_INC;  // positions before chunk 0: inclusive prefix = identity
        }
#pragma unroll
        for (int r = 0; r < EGDST_SCAN_NW; r++) {
            if (done || base - 32 * r < 0) break;  // warp-uniform
            const int idx = base - 32 * r - lane;
            unsigned long long w = wv[r];
            if (idx >= 0 && (w >> 62) == 0ULL) {
                int polls = 0;
                do { w = st[idx]; } while ((w >> 62) == 0ULL && ++polls < EGDST_SCAN_POLLS);
                if ((w >> 62) == 0ULL) { *err = 1; w = EGDST_SCAN_INC; }
            }
            const unsigned incmask = __ballot_sync(EGDST_FULL, (w >> 62) == 2ULL);
            const int cut = incmask ? __ffs(incmask) - 1 : 31;  // nearest predecessor that already knows its prefix
            // ordered reduction over lanes cut..0 (far to near; the combine is associative): lanes beyond `cut` are the identity
            unsigned long long acc = lane <= cut ? (w & EGDST_SCAN_MASK) : 0ULL;
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long far = __shfl_down_sync(EGDST_FULL, acc, o);
                if (lane + o < 32) acc = egdst_scan_combine<KIND>(far, acc);
            }
            acc = __shfl_sync(EGDST_FULL, acc, 0);
            excl = egdst_scan_combine<KIND>(acc, excl);
            if (incmask) done = true;
        }
    }
    if (lane == 0) st[chunk] = EGDST_SCAN_INC | egdst_scan_combine<KIND>(excl, agg);
    return excl;
}
EGDST_DEV unsigned long long egdst_scan_inclusive(const volatile unsigned long long *st, int chunk) { return st[chunk] & EGDST_SCAN_MASK; }

// exclusive block scan of one int per thread; returns the exclusive prefix, *total gets the block sum.
// `sh` must hold blockDim.x/32+1 ints.  Contains two egdst_cta_sync().
EGDST_DEV int egdst_block_excl_scan(int v, int *sh, int *total) {
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    int inc = egdst_warp_incl_scan(v, lane);
    if (lane == 31) sh[w] = inc;
    egdst_cta_sync();
    if (w == 0) {
        int s = lane < nw ? sh[lane] : 0;
        int si = egdst_warp_incl_scan(s, lane);
        if (lane < nw) sh[lane] = si - s;
        if (lane == nw - 1) sh[nw] = si;
    }
    egdst_cta_sync();
    int res = inc - v + sh[w];
    *total = sh[nw];
    egdst_cta_sync();
    return res;
}
