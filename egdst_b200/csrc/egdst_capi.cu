// egdst_capi.cu -- host orchestration and the C ABI (include/egdst_b200.h).
//
// Replaces the reference's MEX gateways and driver loops:
//   mexFunction/solver()      egdst_solver.c:143-339   -> egdst_solve / egdst_resolve (one kernel: the period loop runs on the device)
//   saveoutput/swappointers   egdst_solver.c:917-952,342 -> the device arena (next period reads the cells in place)
//   parseModel/loadparameters egdst_lib.c:34-62          -> egdst_desc
// There is no host arithmetic on the data path: even the cdfni transform of the quadrature abscissas
// (egdst_solver.c:162-164) runs on the device.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "egdst_b200.h"
#ifndef EGDST_HOSTEMU
#include <cuda.h>
#include <cudaTypedefs.h>
#endif
#include "egdst_period.cuh"
#include "egdst_simulator.cuh"
#include "egdst_loglik.cuh"

#ifndef EGDST_MODEL_KEY
#define EGDST_MODEL_KEY "unknown"
#endif

static thread_local std::string g_err;
static thread_local cudaStream_t g_stream = 0;

// ---- launch counter and optional per-kernel-class event timing (bench.py's roofline leg) --------------
enum { KC_SETUP = 0, KC_SOLVE, KC_TAB, KC_SIM, KC_OTHER, KC_COUNT };
static const char *const g_kc_names[KC_COUNT] = {"setup", "solve", "tables", "simulate", "other"};
static std::atomic<long long> g_launches{0};
static bool g_prof_on = false;  // profiling is a single-threaded measurement aid (egdst_profile_enable)
struct ProfRec { int cls; cudaEvent_t a, b; };
static std::vector<ProfRec> g_prof_pending;
static double g_prof_ms[KC_COUNT];
static long long g_prof_n[KC_COUNT];
static void prof_begin(int cls, cudaStream_t st) {
    g_launches++;
    if (!g_prof_on) return;
    ProfRec r; r.cls = cls;
    cudaEventCreate(&r.a); cudaEventCreate(&r.b);
    cudaEventRecord(r.a, st);
    g_prof_pending.push_back(r);
}
static void prof_end(cudaStream_t st) {
    if (!g_prof_on) return;
    cudaEventRecord(g_prof_pending.back().b, st);
}
static void prof_collect() {
    for (ProfRec &r : g_prof_pending) {
        float ms = 0.f;
        cudaEventSynchronize(r.b);
        cudaEventElapsedTime(&ms, r.a, r.b);
        g_prof_ms[r.cls] += ms; g_prof_n[r.cls]++;
        cudaEventDestroy(r.a); cudaEventDestroy(r.b);
    }
    g_prof_pending.clear();
}
#define KLAUNCH(cls, kernel, grid, block, smem, stream, ...) \
    do { prof_begin(cls, stream); EGDST_LAUNCH(kernel, grid, block, smem, stream, __VA_ARGS__); prof_end(stream); } while (0)

static int fail(int code, const std::string &msg) { g_err = msg; return code; }

#define CK(call)                                                                                       \
    do {                                                                                               \
        cudaError_t e_ = (call);                                                                       \
        if (e_ != cudaSuccess) return fail(2, std::string("CUDA error: ") + cudaGetErrorString(e_) + " at " #call); \
    } while (0)
// error-accumulating form (cudaError_t ce in scope): once a call has failed, the following ones are skipped
#define EGDST_TRY(call) do { if (ce == cudaSuccess) ce = (call); } while (0)

// grow-only device buffer of n elements: reallocated, without its contents, when n does not fit
template <class T>
static cudaError_t grow(T **p, size_t *cap, size_t n) {
    if (*p && n <= *cap) return cudaSuccess;
    if (*p) cudaFree(*p);
    *p = 0;
    *cap = 0;
    const cudaError_t e = cudaMalloc((void **)p, (n ? n : 1) * sizeof(T));
    if (e == cudaSuccess) *cap = n;
    return e;
}

static const char *status_text(int code) {
    switch (code) {  // wording of the reference's error() sites
    case EGDST_ERR_CHECKSUM: return "Transition probabilities don't sum up! Check model specification!";
    case EGDST_ERR_NOSAVINGS: return "Failed to find any value of savings to result in positive consumption next period! Increase mmax.";
    case EGDST_ERR_GRIDSPACE: return "Not enough space for endogenous grid. Increase max number of grid points for M!";
    case EGDST_ERR_EMPTYCHOICE: return "Empty choiceset encountered! Check model specifications!";
    case EGDST_ERR_ALLINF: return "All of the choices lead to -inf value functions for all values of money-at-hand!";
    case EGDST_ERR_ENVELOPE: return "Failed to compute upper envelope, most likely individual grids don't overlap!";
    case EGDST_ERR_ADRAW_INIT: return "Could not complete initial stage in adraw()..\nSeems like M(a0)>mmax! Increase mmax!";
    case EGDST_ERR_ADRAW_LOOP: return "Emergiency exit from adraw, possibly infinite loop! Check model specifications!";
    case EGDST_ERR_THRSPACE: return "Not enough space for thresholds. Increase max number of threshold points!";
    case EGDST_ERR_TWO_ANALYTIC: return "Fatal error in threshold module. Two analytical value functions seem to intersect. Utility is not additively separable in consumption and discrete choices.";
    case EGDST_ERR_BRACKET: return "Fatal error in braketing module! Solution is outside of brackets.";
    case EGDST_ERR_CASHINVERSE: return "Did not manage to invert the intertemporal budget (cashinhand) after performing many-many iterations!";
    case EGDST_ERR_INTERP2PT: return "Error: At least two points are required for interpolation!";
    case EGDST_ERR_ENV2SPACE: return "Not enough space for endogenous grid in envelop2()";
    case EGDST_ERR_BARRIER: return "internal error: a phase barrier of the solve kernel timed out";
    case EGDST_ERR_TRPR_INDEX: return "Error in trpr: unknown index of the state variable";
    case EGDST_ERR_TRPR_CASES: return "Error in trpr: unknown combination of current state and decision (the set of cases is not complete)!";
    default: return "unknown error";
    }
}

enum { SCOPE_GRID = 0, SCOPE_CTA, SCOPE_WARP };  // work partitions of the solve kernel (egdst_period.cuh)

// Test hooks, read from the environment when a solution object is created (read_hooks).  None is set in production.
struct EgdstHooks {
    int scope;                  // EGDST_SOLVE_SCOPE: "grid", "warp", any other value CTA; -1: chosen by the shape
    int warpG, warpGSet;        // EGDST_WARP_G: warps per CTA of the WARP scope (when set, no fall-back to the CTA scope)
    int egmP;                   // EGDST_EGM_P: grid points per work item of the EGM phase
    int tabcap;                 // EGDST_TABCAP: lookup-table capacity; cells with more rows take the table-free path
    int solveFrom, solveTo;     // EGDST_SOLVE_FROM/_TO: solve these periods only, the cells of later ones are imported
};

static EgdstHooks read_hooks() {
    auto num = [](const char *v, int unset) { return v ? atoi(v) : unset; };
    const char *scope = getenv("EGDST_SOLVE_SCOPE"), *warpG = getenv("EGDST_WARP_G");
    EgdstHooks h;
    h.scope = !scope ? -1 : strcmp(scope, "grid") == 0 ? SCOPE_GRID : strcmp(scope, "warp") == 0 ? SCOPE_WARP : SCOPE_CTA;
    h.warpG = num(warpG, 0);
    h.warpGSet = warpG != 0;
    h.egmP = num(getenv("EGDST_EGM_P"), 0);
    h.tabcap = num(getenv("EGDST_TABCAP"), 0);
    h.solveFrom = num(getenv("EGDST_SOLVE_FROM"), -1);
    h.solveTo = num(getenv("EGDST_SOLVE_TO"), -1);
    return h;
}

// How the solve kernel is launched for one object (plan_solve)
struct SolvePlan {
    int scope = SCOPE_GRID;
    int ctas = 0, block = 0, warps = 0;  // CTAs (one resident wave), threads per CTA (per warp in the WARP scope), warps per CTA
    size_t smem = 0;                     // dynamic shared memory
    int syncOff = -1, groupBytes = 0;    // per-vector state in shared memory (CTA and WARP scopes), bytes per warp (WARP)
    int egmP = 0, chC = 0, chE = 0;      // grid points per EGM work item; scan windows per job of the EGM phase and of the merge
    int itStart = 0, itStop = 0;         // periods solved
};

struct egdst_solution {
    EgdstDev P{};
    int device = 0;
    int dims[12] = {};    // shape signature for re-use
    double dkey[2] = {};  // mmax, a0: the geometry of the lookup tables (mbits, lutcap) is derived from them at creation
    EgdstHooks hooks{};   // in effect at creation; part of the re-use key, since the plan and tabcap depend on them
    SolvePlan plan;
    int nsd = 0, ncell = 0, nslot = 0;
    int ncell_all = 0;    // ncell, plus the ncell*nd choice-specific cells of the smoothing mode
    size_t bytes = 0;     // device bytes of the allocations made at creation (cache policy)
    double *d_qraw = 0;   // quadrature as passed (weights, abscissas)
    double *d_stm = 0, *d_states = 0, *d_decisions = 0, *d_bparams = 0, *d_q = 0;
    EgdstDev *d_self = 0; // copy of P in global memory (smoothing mode)
    int *d_moff = 0, *d_toff = 0;
    unsigned long long *d_phase = 0;  // per-phase device time of profiled solves
    unsigned char *tab_base = 0;      // lookup tables (one allocation)
    // grow-only buffers (grow)
    double *d_pack = 0; size_t pack_cap = 0;                // export / import staging
    EgdstCellHdr *d_hdr = 0; size_t hdr_cap = 0;            // simulator cell headers
    double *d_llpart = 0; size_t llpart_cap = 0;            // block partials of the choice log-likelihood
    double *d_llrow = 0; size_t llrow_cap = 0;              // row values [nvec][nobs] of the mixture log-likelihood
    double *d_llind = 0; size_t llind_cap = 0;              // per-individual values [nvec][nind] of the same
    double *d_llmix = 0; size_t llmix_cap = 0;              // per-individual mixture values [nmix][nind] of the scores
    // every device allocation, by the field that holds it
    std::vector<void **> owned{(void **)&d_pack, (void **)&d_hdr, (void **)&d_llpart, (void **)&d_llrow, (void **)&d_llind,
                               (void **)&d_llmix};
    // state of the current owner (adopt)
    std::vector<int> h_mlen, h_thlen, h_status;
    bool sizes_valid = false;
    std::vector<double> h_params;  // host copy of the parameter matrix of the last solve (simulator kernel arguments)
    std::vector<EgdstCellHdr> h_hdr; int hdr_ivec = -1;  // simulator cell headers (kernel argument), -1 = stale
    bool choice_cells = false;  // the choice-specific cells hold a solve's result (an import leaves them empty)
    bool choice_draws = false;  // simulations draw each period's decision from the choice probabilities
};

template <class T>
static cudaError_t dalloc(egdst_solution *s, T **p, size_t n) {
    cudaError_t e = cudaMalloc((void **)p, (n ? n : 1) * sizeof(T));
    if (e == cudaSuccess) { s->owned.push_back((void **)p); s->bytes += (n ? n : 1) * sizeof(T); }
    return e;
}

// One released solution object is kept for re-use by the next egdst_solve of the same shape: the MEX gateway
// solves, exports and frees on every call, and ~45 cudaMalloc/cudaFree pairs cost far more than the solve itself.
static std::mutex g_cache_mu;
static egdst_solution *g_cached = 0;
static const size_t EGDST_CACHE_MAX_BYTES = (size_t)2 << 30;
static void destroy_solution(egdst_solution *s) {
    cudaSetDevice(s->device);
    for (void **p : s->owned) if (*p) cudaFree(*p);
    delete s;
}

// quadrature abscissas -> standard normal quantiles (egdst_solver.c:162-164), on the device
__global__ void egdst_k_quadrature(const double *qraw, double *q, int ny) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < ny) { q[i] = qraw[i]; q[ny + i] = egdst_cdfni(qraw[ny + i]); }
}

// the descriptor must describe the model this image was generated from: sizes of the generated structures and the
// optim_* switches, which are functions of the exec strings (compile.m:669-747) and compiled into the kernels
static int check_image(const egdst_desc *d) {
    if (!d) return fail(2, "null descriptor");
    if (d->abi_version != EGDST_ABI_VERSION) return fail(2, "egdst_desc.abi_version mismatch");
    if (d->nparam != EGDST_NPARAM) return fail(2, "number of parameters does not match the compiled model image");
    if (d->nnst > EGDST_NNST || d->nnd > EGDST_NND) return fail(2, "state/decision vector size does not match the compiled model image");
    if ((d->optim_UasD != 0) != (EGDST_OPT_UASD != 0) || (d->optim_MUnoD != 0) != (EGDST_OPT_MUNOD != 0) ||
        (d->optim_UnoD != 0) != (EGDST_OPT_UNOD != 0) || (d->optim_TRPRnoSH != 0) != (EGDST_OPT_TRPRNOSH != 0))
        return fail(2, "optim_* switches of the descriptor do not match the compiled model image");
    if (EGDST_NPARAM > 0 && !d->params) return fail(2, "parameter values missing");
    if ((d->sigma_eps > 0.0) != (EGDST_SMOOTHING != 0))
        return fail(2, "taste-shock smoothing (sigma_eps > 0) is a property of the compiled model image: set it before compiling the model");
    return 0;
}

static int fill_ctx(const egdst_desc *d, egdst_ctx *cx) {
    const int rci = check_image(d);
    if (rci) return rci;
    if (d->ngridm < 2 || d->ngridmax <= d->ngridm || d->T < d->t0 || d->nst < 1 || d->nd < 1 || d->ny < 1 || d->nthrhmax < 2)
        return fail(2, "invalid model dimensions");
    memset(cx, 0, sizeof(*cx));
    cx->t0 = d->t0; cx->T = d->T; cx->ngridm = d->ngridm; cx->ngridmax = d->ngridmax; cx->nthrhmax = d->nthrhmax;
    cx->ny = d->ny; cx->nd = d->nd; cx->nnd = d->nnd; cx->nst = d->nst; cx->nnst = d->nnst;
    cx->optim_UasD = d->optim_UasD; cx->optim_MUnoD = d->optim_MUnoD; cx->optim_UnoD = d->optim_UnoD; cx->optim_TRPRnoSH = d->optim_TRPRnoSH;
    cx->byval = 0;
    cx->mmax = d->mmax; cx->a0 = d->a0;
    cx->tolerance = d->tolerance; cx->zeroconsumption = d->zeroconsumption; cx->doublepoint_delta = d->doublepoint_delta;
    for (int i = 0; i < EGDST_NPARAM; i++) cx->param[i] = d->params[i];
    return 0;
}

static int check_device(int device) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) return fail(2, "no CUDA device: egdst_b200 has no CPU path");
    if (device < 0 || device >= n) return fail(2, "invalid CUDA device ordinal");
    if (cudaSetDevice(device) != cudaSuccess) return fail(2, "cudaSetDevice failed");
    return 0;
}

static inline int imin(int a, int b) { return a < b ? a : b; }

// the model of d (validated by fill_ctx into cx) becomes the model of s
static void set_model(egdst_solution *s, const egdst_desc *d, egdst_ctx cx) {
    cx.stm = s->d_stm; cx.states = s->d_states; cx.decisions = s->d_decisions;
    s->P.cx = cx;
    s->P.sigmaEps = d->sigma_eps;
}

// hand s to a new owner: nothing of a previous owner (sizes, status, parameter values, simulator headers) survives
static void adopt(egdst_solution *s, const egdst_desc *d, const egdst_ctx &cx) {
    set_model(s, d, cx);
    s->P.bparams = 0;
    cudaMemset(s->P.units, 0, sizeof(unsigned long long) * 2 * s->P.nvec);
    s->h_mlen.assign(s->ncell, 0);
    s->h_thlen.assign(s->ncell, 0);
    s->h_status.assign(4 * s->P.nvec, 0);
    s->sizes_valid = false;
    s->h_params.clear();
    s->hdr_ivec = -1;
    s->choice_cells = false;
    s->choice_draws = false;
}

// every device array of a new object of the shape of d with nvec parameter vectors (s->P.cx: the model of d)
static int alloc_solution(egdst_solution *s, const egdst_desc *d, int nvec) {
    EgdstDev &P = s->P;
    P.NT = d->T - d->t0 + 1; P.nvec = nvec; P.rowcap = d->ngridmax + 2; P.gcap = d->ngridmax; P.N = d->ngridm;
    const int nst = d->nst, nd = d->nd;
    s->ncell = nvec * P.NT * nst; s->nsd = nvec * nst * nd; s->nslot = s->nsd + nvec * nst;
    s->ncell_all = d->sigma_eps > 0.0 ? s->ncell * (1 + nd) : s->ncell;
    P.ncellMain = s->ncell;
    P.envcap = (nd > 2 ? nd : 2) * P.gcap + 2;
#define DA(ptr, n) do { cudaError_t e_ = dalloc(s, &(ptr), (size_t)(n)); if (e_ != cudaSuccess) return fail(2, std::string("cudaMalloc failed: ") + cudaGetErrorString(e_)); } while (0)
    DA(s->d_stm, 2 * d->nnst); DA(s->d_states, nst * d->nnst); DA(s->d_decisions, nd * d->nnd);
    DA(s->d_bparams, (size_t)nvec * EGDST_NPARAM_); DA(s->d_qraw, 2 * d->ny); DA(s->d_q, 2 * d->ny);
    DA(P.tabOk, s->ncell_all);
    DA(P.arena, (size_t)s->ncell_all * 4 * P.rowcap); DA(P.mlen, s->ncell_all); DA(P.thlen, s->ncell); DA(P.evf, s->ncell_all);
    DA(P.thD, (size_t)s->ncell * d->nthrhmax); DA(P.thTH, (size_t)s->ncell * d->nthrhmax);
    DA(P.active, s->nsd); DA(P.seed, (size_t)s->nsd * EGDST_SEEDW); DA(P.evfa0, s->nsd);
    DA(P.ptX, (size_t)s->nsd * P.gcap); DA(P.ptC, (size_t)s->nsd * P.gcap); DA(P.ptV, (size_t)s->nsd * P.gcap);
    DA(P.ptN, s->nsd); DA(P.nfold, s->nsd); DA(P.runStart, (size_t)s->nsd * (P.gcap + 1));
    DA(P.mgX, (size_t)s->nslot * P.envcap); DA(P.mgF, (size_t)s->nslot * P.envcap); DA(P.mgK, (size_t)s->nslot * P.envcap); DA(P.mgA, (size_t)s->nslot * P.envcap);
    DA(P.outX, (size_t)s->nsd * P.envcap); DA(P.outC, (size_t)s->nsd * P.envcap); DA(P.outV, (size_t)s->nsd * P.envcap);
    // lookup tables (egdst_tables.cuh): capacity 2*ngridm+64 intervals per cell, about two buckets per grid row
    P.tabcap = P.rowcap - 1 < 2 * P.N + 64 ? P.rowcap - 1 : 2 * P.N + 64;
    if (s->hooks.tabcap >= 1 && s->hooks.tabcap < P.tabcap) P.tabcap = s->hooks.tabcap;
    {
        const double span = 2.0 * (d->mmax - d->a0) + 2.0;
        const double octaves = log2(span > 2.0 ? span : 2.0);
        int mbits = 3;
        // buckets per grid row: an index entry resolves up to three rows of a bucket by itself, so about one bucket
        // per row keeps the index small (the simulator wants every period's tables L2-resident next to its output stream)
        while (mbits < 16 && (double)(1 << mbits) * octaves < (double)(P.N + 1)) mbits++;
        P.mbits = mbits;
        P.lutcap = (int)(octaves * (double)(1 << mbits)) + 2;
    }
    {   // one allocation for both tables: a single L2 access-policy window can then keep them resident (sim_launch)
        const size_t lutbytes = ((sizeof(EgdstLutEntry) * (size_t)s->ncell_all * (P.lutcap + 1) + 255) / 256) * 256;
        const size_t ivlbytes = ((sizeof(EgdstRow) * (size_t)s->ncell_all * (P.tabcap + 1) + 255) / 256) * 256;
        const size_t topbytes = sizeof(EgdstCellTop) * (size_t)s->ncell_all;
        DA(s->tab_base, lutbytes + ivlbytes + topbytes);
        P.tabLut = (EgdstLutEntry *)s->tab_base; P.tabRow = (EgdstRow *)(s->tab_base + lutbytes); P.tabTop = (EgdstCellTop *)(s->tab_base + lutbytes + ivlbytes);
    }
    // chained scans: one state word per work item of a job plus the seed's slot (EGM phase: at least 8 grid points per
    // item), one per chunk of union positions (envelope merge); the allocation serves the narrowest team (a warp),
    // plan_solve sets the values of the scope
    P.chC = (P.N - 1 + 7) / 8 + 2;
    P.chE = (P.envcap + 31) / 32 + 1;
    // a point of the secondary envelope ranks itself against every run (~10^2 in the zig-zag periods of S1): with few
    // jobs, 8 threads share the runs of a point
    P.envA1parts = (nvec * nst * nd < 148) ? 8 : 1;
    DA(P.scanC, (size_t)s->nsd * P.chC); DA(P.tickC, (size_t)2 * s->nsd); DA(P.foldList, (size_t)s->nsd * (P.gcap + 1)); DA(P.foldCnt, s->nsd);
    DA(P.scanE, (size_t)s->nslot * P.chE); DA(P.tickE, (size_t)2 * s->nslot); DA(P.envNact, s->nslot);
    DA(P.lateN, s->nsd); DA(P.flags, (size_t)8 * (nvec + 1)); DA(P.bar, 4); DA(s->d_phase, EGDST_NPHASE);
    cudaMemset(s->d_phase, 0, sizeof(unsigned long long) * EGDST_NPHASE);
    DA(s->d_self, 1); DA(P.status, 4 * nvec); DA(P.units, 2 * nvec); DA(s->d_moff, s->ncell + 1); DA(s->d_toff, s->ncell + 1);
#undef DA
    P.qw = s->d_q; P.qz = s->d_q + d->ny;
    return 0;
}

// The launch of the solve kernel, chosen once per object.  Scope (egdst_period.cuh): sweeps of many small models run
// a CTA (or a warp) per parameter vector, which walks its vector through all periods on its own; everything else is a
// cooperative launch of exactly one resident wave whose CTAs share every phase of every period.
static int plan_solve(egdst_solution *s) {
    const EgdstDev &P = s->P;
    const EgdstHooks &h = s->hooks;
    SolvePlan &pl = s->plan;
    const int nvec = P.nvec, N = P.N;
    int sms = 1;  // the host emulator runs one CTA
#ifndef EGDST_HOSTEMU
    int dev = 0;
    CK(cudaGetDevice(&dev));
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    // small models, many of them: a CTA (or warp) per vector keeps all of a vector's arrays in its SM's L1/L2
    // neighbourhood and needs neither launches nor inter-CTA waits
    if (nvec >= 2 * sms && N <= 4 * EGDST_BLOCK) pl.scope = nvec >= 8 * sms ? SCOPE_WARP : SCOPE_CTA;
#endif
    if (h.scope >= 0) pl.scope = h.scope;
    // per-CTA table of quadrature shocks and node probabilities (models whose shocks cannot depend on savings)
    const size_t shbytes = (size_t)2 * P.cx.nst * P.cx.ny * sizeof(double);
    const size_t shtab = (EGDST_SHOCK_INDEP_A && shbytes <= EGDST_SHOCKTAB_BYTES) ? shbytes : 0;
    // CTA and WARP scopes: a team of B threads takes the whole grid of a decision at a time (few scan windows), and the
    // vector's small state fits shared memory; returns the bytes of that state
    auto team = [&](int B) {
        pl.block = B;
        pl.chE = (P.envcap + B - 1) / B + 1;
        pl.egmP = B < N - 1 ? B : (N - 1 < 8 ? 8 : N - 1);
        if (h.egmP >= 8 && h.egmP <= B) pl.egmP = h.egmP;
        pl.chC = imin(P.chC, (N - 1 + pl.egmP - 1) / pl.egmP + 2);
        EgdstDev Q = P;
        Q.chC = pl.chC;
        Q.chE = pl.chE;
        return egdst_cta_sync_bytes(Q);
    };
    if (pl.scope == SCOPE_WARP) {
        const size_t sb = team(32);
        pl.syncOff = (int)((EgdstScratch<32>::bytes + shtab + 15) / 16 * 16);
        pl.groupBytes = (int)((pl.syncOff + sb + 127) / 128 * 128);
        // as many warps per CTA as shared memory allows, and no more than spreads the vectors over all SMs
        pl.warps = imin(imin((200 * 1024) / pl.groupBytes, EGDST_WARP_GROUPS), (nvec + sms - 1) / sms);
        if (h.warpG >= 1 && h.warpG <= pl.warps) pl.warps = h.warpG;
        pl.smem = (size_t)pl.groupBytes * pl.warps;
        if (pl.warps < 4 && !h.warpGSet) pl.scope = SCOPE_CTA;  // too few warps per SM to hide anything
    }
    if (pl.scope == SCOPE_CTA) {
        const size_t sb = team(EGDST_CTA_BLOCK);
        pl.warps = 0;
        pl.smem = EgdstScratch<EGDST_CTA_BLOCK>::bytes + shtab;
        pl.syncOff = -1;
        if (sb <= 6144) { pl.syncOff = (int)((pl.smem + 15) / 16 * 16); pl.smem = pl.syncOff + sb; }
    }
    if (pl.scope == SCOPE_GRID) {
        pl.block = EGDST_BLOCK;
        pl.chE = (P.envcap + EGDST_BLOCK - 1) / EGDST_BLOCK + 1;
        pl.chC = P.chC;
        pl.smem = EgdstScratch<EGDST_BLOCK>::bytes + shtab;
    }
    int occ = 1;
#ifndef EGDST_HOSTEMU
    const void *kern = pl.scope == SCOPE_WARP ? (const void *)egdst_k_solve_warps
                       : pl.scope == SCOPE_CTA ? (const void *)egdst_k_solve_cta : (const void *)egdst_k_solve_grid;
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
    if (pl.scope != SCOPE_WARP && (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, pl.block, pl.smem) != cudaSuccess || occ < 1)) occ = 1;
#endif
    pl.ctas = sms * occ;
    if (pl.scope != SCOPE_GRID) {
        pl.ctas = imin(pl.ctas, pl.warps ? (nvec + pl.warps - 1) / pl.warps : nvec);  // no more CTAs than vectors to take
    } else {
        // grid points per work item of the EGM phase: the items of one period fill the grid exactly once (no tail wave)
        const long long jobs = (long long)nvec * P.cx.nst * P.cx.nd;
        int egmP = (int)(((long long)(N - 1) * jobs + pl.ctas - 1) / pl.ctas);
        if (egmP < 8) egmP = 8;
        if (egmP > EGDST_BLOCK) egmP = EGDST_BLOCK;
        if (egmP > N - 1 && N - 1 >= 1) egmP = N - 1 < 8 ? 8 : N - 1;
        if (h.egmP >= 8 && h.egmP <= EGDST_BLOCK) egmP = h.egmP;
        pl.egmP = egmP;
    }
    if ((N - 1 + pl.egmP - 1) / pl.egmP + 2 > pl.chC) return fail(2, "internal: scan state too small for the EGM items");
    pl.itStart = h.solveFrom >= 0 && h.solveFrom < P.NT - 1 ? h.solveFrom : P.NT - 1;
    pl.itStop = h.solveTo >= 0 && h.solveTo <= pl.itStart ? h.solveTo : 0;
    return 0;
}

static int create_solution(const egdst_desc *d, int nvec, egdst_solution **out) {
    egdst_ctx cx;
    int rc = fill_ctx(d, &cx);
    if (rc) return rc;
    if ((rc = check_device(d->device))) return rc;
    const bool smooth = d->sigma_eps > 0.0;  // taste-shock smoothing: choice-specific cells next to the solution cells
    if (smooth && d->nd > EGDST_SMOOTH_MAXND) return fail(2, "sigma_eps > 0 supports at most 8 decisions");
    if (d->sigma_eps < 0.0 || d->sigma_eps != d->sigma_eps) return fail(2, "sigma_eps must be >= 0");
    const int dims[12] = {d->device, nvec, d->T - d->t0 + 1, d->nst, d->nd, d->ngridm, d->ngridmax, d->nthrhmax, d->ny, d->nnst, d->nnd, smooth ? 1 : 0};
    const EgdstHooks hooks = read_hooks();
    egdst_solution *s = 0;
    {
        std::lock_guard<std::mutex> lk(g_cache_mu);
        if (g_cached && memcmp(g_cached->dims, dims, sizeof(dims)) == 0 && g_cached->dkey[0] == d->mmax && g_cached->dkey[1] == d->a0 &&
            memcmp(&g_cached->hooks, &hooks, sizeof(hooks)) == 0) {
            s = g_cached;
            g_cached = 0;
        }
    }
    if (!s) {
        s = new egdst_solution();
        s->device = d->device; memcpy(s->dims, dims, sizeof(dims)); s->dkey[0] = d->mmax; s->dkey[1] = d->a0; s->hooks = hooks;
        s->P.cx = cx;
        if ((rc = alloc_solution(s, d, nvec)) || (rc = plan_solve(s))) { destroy_solution(s); return rc; }
    }
    adopt(s, d, cx);
    *out = s;
    return 0;
}

// One backward-induction pass = one kernel on `st`, launched as planned (plan_solve)
static int launch_solve(egdst_solution *s, cudaStream_t st) {
    EgdstDev &P = s->P;
    const SolvePlan &pl = s->plan;
    P.itStart = pl.itStart;
    P.itStop = pl.itStop;
    CK(cudaMemsetAsync(P.status, 0, sizeof(int) * 4 * P.nvec, st));
    CK(cudaMemsetAsync(P.units, 0, sizeof(unsigned long long) * 2 * P.nvec, st));
    CK(cudaMemsetAsync(P.bar, 0, sizeof(unsigned) * 4, st));
    if (P.itStart == P.NT - 1) {
        CK(cudaMemsetAsync(P.mlen, 0, sizeof(int) * s->ncell_all, st));
        CK(cudaMemsetAsync(P.thlen, 0, sizeof(int) * s->ncell, st));
        CK(cudaMemsetAsync(P.tabOk, 1, sizeof(int) * s->ncell_all, st));  // non-zero: usable; cleared by the table build of a cell whose grid steps back
    }
    P.priSync0 = P.nvec * P.cx.nst * P.cx.nd;
    P.egmP = pl.egmP; P.chC = pl.chC; P.chE = pl.chE;
    P.self = s->d_self;
    P.phase_ns = g_prof_on ? s->d_phase : 0;  // measurement aid: in-kernel phase timers while profiling is enabled
    if (EGDST_SMOOTHING) CK(cudaMemcpyAsync(s->d_self, &P, sizeof(EgdstDev), cudaMemcpyHostToDevice, st));  // read by egdst_smooth_node
    switch (pl.scope) {
    case SCOPE_WARP: KLAUNCH(KC_SOLVE, egdst_k_solve_warps, dim3(pl.ctas), dim3(32, pl.warps), pl.smem, st, P, pl.syncOff, pl.groupBytes); break;
    case SCOPE_CTA: KLAUNCH(KC_SOLVE, egdst_k_solve_cta, dim3(pl.ctas), dim3(pl.block), pl.smem, st, P, pl.syncOff); break;
    default: {
#ifndef EGDST_HOSTEMU
        void *args[] = {(void *)&P};
        prof_begin(KC_SOLVE, st);
        CK(cudaLaunchCooperativeKernel((const void *)egdst_k_solve_grid, dim3(pl.ctas), dim3(pl.block), args, pl.smem, st));
        prof_end(st);
#else
        KLAUNCH(KC_SOLVE, egdst_k_solve_grid, dim3(pl.ctas), dim3(pl.block), pl.smem, st, P);
#endif
    }
    }
    CK(cudaGetLastError());
    return 0;
}

// the model tables of d (stm, states, decisions) to the device copies of s
static cudaError_t upload_tables(egdst_solution *s, const egdst_desc *d, cudaStream_t st) {
    cudaError_t ce = cudaSuccess;
    EGDST_TRY(cudaMemcpyAsync(s->d_stm, d->stm, sizeof(double) * 2 * d->nnst, cudaMemcpyHostToDevice, st));
    EGDST_TRY(cudaMemcpyAsync(s->d_states, d->states, sizeof(double) * d->nst * d->nnst, cudaMemcpyHostToDevice, st));
    EGDST_TRY(cudaMemcpyAsync(s->d_decisions, d->decisions, sizeof(double) * d->nd * d->nnd, cudaMemcpyHostToDevice, st));
    return ce;
}

// one backward-induction pass of the model in s->P.cx (d: its descriptor); asynchronous
static int run_solve(egdst_solution *s, const egdst_desc *d, const double *params) {
    EgdstDev &P = s->P;
    if (d->ny > 1 && !d->quadrature) return fail(2, "quadrature missing");
    CK(cudaSetDevice(s->device));
    cudaStream_t st = g_stream;
    CK(upload_tables(s, d, st));
    // parameter values always travel through the device array (one row per vector), never through the kernel
    // arguments: the argument block then depends on the shape only
    if (!params && P.nvec != 1) return fail(2, "egdst_resolve: a batched solution needs the parameter matrix");
    s->h_params.assign(params ? params : d->params, (params ? params : d->params) + (size_t)P.nvec * EGDST_NPARAM);
    if (EGDST_NPARAM > 0) CK(cudaMemcpyAsync(s->d_bparams, params ? params : d->params, sizeof(double) * (size_t)P.nvec * EGDST_NPARAM, cudaMemcpyHostToDevice, st));
    P.bparams = s->d_bparams;
    for (int i = 0; i < EGDST_NPARAM_; i++) P.cx.param[i] = 0.0;
    if (d->ny > 1) {
        CK(cudaMemcpyAsync(s->d_qraw, d->quadrature, sizeof(double) * 2 * d->ny, cudaMemcpyHostToDevice, st));
        KLAUNCH(KC_SETUP, egdst_k_quadrature, dim3((d->ny + 127) / 128), dim3(128), 0, st, s->d_qraw, s->d_q, d->ny);
    }
    int rc = launch_solve(s, st);
    if (rc) return rc;
    s->sizes_valid = false;
    s->hdr_ivec = -1;
    s->choice_cells = s->ncell_all > s->ncell;
    CK(cudaGetLastError());
    return 0;
}

static int fetch_sizes(egdst_solution *s) {
    if (s->sizes_valid) return 0;
    CK(cudaSetDevice(s->device));
    cudaStream_t st = g_stream;
    CK(cudaMemcpyAsync(s->h_mlen.data(), s->P.mlen, sizeof(int) * s->ncell, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(s->h_thlen.data(), s->P.thlen, sizeof(int) * s->ncell, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(s->h_status.data(), s->P.status, sizeof(int) * 4 * s->P.nvec, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    s->sizes_valid = true;
    return 0;
}

static int status_rc(egdst_solution *s) {
    for (int v = 0; v < s->P.nvec; v++) {
        const int code = s->h_status[4 * v];
        if (code) {
            char buf[512];
            snprintf(buf, sizeof(buf), "Error:\n%s\n(vector %d, period it=%d, ist=%d, id=%d)", status_text(code), v, s->h_status[4 * v + 1],
                     s->h_status[4 * v + 2], s->h_status[4 * v + 3]);
            return fail(code >= 100 ? 2 : 1, buf);
        }
    }
    return 0;
}

// gather the ragged cells into the packed export layout
__global__ void egdst_k_pack(EgdstDev P, const int *moff, const int *toff, double *Mbuf, double *Dbuf, int ncell) {
    const int cell = blockIdx.x;
    if (cell >= ncell) return;
    const int n = P.mlen[cell], nth = P.thlen[cell];
    const double *src = P.arena + (size_t)cell * 4 * P.rowcap;
    double *dst = Mbuf + (size_t)4 * moff[cell];
    for (int i = threadIdx.x; i < 4 * n; i += blockDim.x) dst[i] = src[(size_t)(i / n) * P.rowcap + (i % n)];
    double *dd = Dbuf + (size_t)2 * toff[cell];
    for (int i = threadIdx.x; i < nth; i += blockDim.x) {
        dd[i] = P.thD[(size_t)cell * P.cx.nthrhmax + i];
        dd[nth + i] = P.thTH[(size_t)cell * P.cx.nthrhmax + i];
    }
}

// scatter host cells into the arena (egdst_solution_import)
__global__ void egdst_k_unpack(EgdstDev P, const int *moff, const int *toff, const double *Mbuf, const double *Dbuf, int ncell) {
    const int cell = blockIdx.x;
    if (cell >= ncell) return;
    const int n = P.mlen[cell], nth = P.thlen[cell];
    double *dst = P.arena + (size_t)cell * 4 * P.rowcap;
    const double *src = Mbuf + (size_t)4 * moff[cell];
    for (int i = threadIdx.x; i < 4 * n; i += blockDim.x) dst[(size_t)(i / n) * P.rowcap + (i % n)] = src[i];
    const double *dd = Dbuf + (size_t)2 * toff[cell];
    for (int i = threadIdx.x; i < nth; i += blockDim.x) {
        P.thD[(size_t)cell * P.cx.nthrhmax + i] = dd[i];
        P.thTH[(size_t)cell * P.cx.nthrhmax + i] = dd[nth + i];
    }
    if (threadIdx.x == 0 && n > 0) P.evf[cell] = src[3 * n];
}

// offsets of the cells in the packed layout (rows mlen, thresholds thlen) to the device, and a pack buffer that holds
// the layout's nm M values and nd2 D values
static int pack_layout(egdst_solution *s, const int *mlen, const int *thlen, size_t *nm, size_t *nd2) {
    std::vector<int> moff(s->ncell + 1, 0), toff(s->ncell + 1, 0);
    for (int c = 0; c < s->ncell; c++) { moff[c + 1] = moff[c] + mlen[c]; toff[c + 1] = toff[c] + thlen[c]; }
    *nm = (size_t)4 * moff[s->ncell];
    *nd2 = (size_t)2 * toff[s->ncell];
    CK(grow(&s->d_pack, &s->pack_cap, *nm + *nd2));
    CK(cudaMemcpyAsync(s->d_moff, moff.data(), sizeof(int) * (s->ncell + 1), cudaMemcpyHostToDevice, g_stream));
    CK(cudaMemcpyAsync(s->d_toff, toff.data(), sizeof(int) * (s->ncell + 1), cudaMemcpyHostToDevice, g_stream));
    return 0;
}

// sum over the vectors of row `row` of P.units (0: solve work units, 1: re-sends); -1 on error
static long long units_sum(egdst_solution *s, int row) {
    if (!s) return -1;
    if (cudaSetDevice(s->device) != cudaSuccess) return -1;
    std::vector<unsigned long long> u(s->P.nvec, 0ULL);
    if (cudaMemcpyAsync(u.data(), s->P.units + (size_t)row * s->P.nvec, sizeof(unsigned long long) * s->P.nvec, cudaMemcpyDeviceToHost, g_stream) != cudaSuccess) return -1;
    if (cudaStreamSynchronize(g_stream) != cudaSuccess) return -1;
    long long tot = 0;
    for (unsigned long long x : u) tot += (long long)x;
    return tot;
}

// frees a scratch or failed solution object (egdst_free_solution) on every return that does not release it
typedef std::unique_ptr<egdst_solution, void (*)(egdst_solution *)> SolutionGuard;

extern "C" {

int egdst_abi_version(void) { return EGDST_ABI_VERSION; }
const char *egdst_model_key(void) { return EGDST_MODEL_KEY; }
int egdst_model_nparam(void) { return EGDST_NPARAM; }
int egdst_model_neq(void) { return EGDST_NREQ; }
const char *egdst_last_error(void) { return g_err.c_str(); }
void egdst_set_stream(void *cuda_stream) { g_stream = (cudaStream_t)cuda_stream; }
long long egdst_launch_count(void) { return g_launches.load(); }
int egdst_profile_classes(void) { return KC_COUNT; }
const char *egdst_profile_class_name(int cls) { return (cls >= 0 && cls < KC_COUNT) ? g_kc_names[cls] : ""; }
void egdst_profile_enable(int on) {
    prof_collect();
    g_prof_on = on != 0;
    if (on) for (int i = 0; i < KC_COUNT; i++) { g_prof_ms[i] = 0.0; g_prof_n[i] = 0; }
}
int egdst_profile_read(double *ms, long long *count) {
    prof_collect();
    for (int i = 0; i < KC_COUNT; i++) { if (ms) ms[i] = g_prof_ms[i]; if (count) count[i] = g_prof_n[i]; }
    return KC_COUNT;
}

int egdst_solve_batch(const egdst_desc *d, const double *params, int nvec, egdst_solution **out) {
    if (!out || nvec < 1) return fail(2, "invalid arguments");
    *out = 0;
    egdst_solution *s = 0;
    int rc = create_solution(d, nvec, &s);
    if (rc) return rc;
    SolutionGuard guard(s, egdst_free_solution);
    if ((rc = run_solve(s, d, params)) || (rc = fetch_sizes(s))) return rc;
    rc = status_rc(s);
    if (rc != 2) *out = guard.release();
    return rc;
}

int egdst_solve(const egdst_desc *d, egdst_solution **out) { return egdst_solve_batch(d, 0, 1, out); }

int egdst_resolve(egdst_solution *s, const egdst_desc *d, const double *params) {
    if (!s) return fail(2, "null solution");
    egdst_ctx cx;
    int rc = fill_ctx(d, &cx);
    if (rc) return rc;
    const EgdstDev &P = s->P;
    if (d->ngridm != P.N || d->ngridmax != P.gcap || d->T - d->t0 + 1 != P.NT || d->nst != P.cx.nst || d->nd != P.cx.nd ||
        d->ny != P.cx.ny || d->nthrhmax != P.cx.nthrhmax)
        return fail(2, "egdst_resolve: dimensions differ from the solution object");
    if ((d->sigma_eps > 0.0) != (s->ncell_all > s->ncell)) return fail(2, "egdst_resolve: sigma_eps switches the smoothing mode on or off; solve anew");
    set_model(s, d, cx);
    return run_solve(s, d, params);
}

int egdst_solution_sizes(egdst_solution *s, int *mlen, int *thlen) {
    if (!s) return fail(2, "null solution");
    int rc = fetch_sizes(s);
    if (rc) return rc;
    if (mlen) memcpy(mlen, s->h_mlen.data(), sizeof(int) * s->ncell);
    if (thlen) memcpy(thlen, s->h_thlen.data(), sizeof(int) * s->ncell);
    return status_rc(s) == 2 ? 2 : 0;
}

int egdst_solution_export(egdst_solution *s, double *Mbuf, double *Dbuf) {
    if (!s || !Mbuf || !Dbuf) return fail(2, "invalid arguments");
    size_t nm = 0, nd2 = 0;
    int rc = fetch_sizes(s);
    if (rc || (rc = pack_layout(s, s->h_mlen.data(), s->h_thlen.data(), &nm, &nd2))) return rc;
    cudaStream_t st = g_stream;
    KLAUNCH(KC_OTHER, egdst_k_pack, dim3(s->ncell), dim3(EGDST_BLOCK), 0, st, s->P, s->d_moff, s->d_toff, s->d_pack, s->d_pack + nm, s->ncell);
    CK(cudaMemcpyAsync(Mbuf, s->d_pack, sizeof(double) * nm, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(Dbuf, s->d_pack + nm, sizeof(double) * nd2, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return 0;
}

int egdst_solution_choice_cell(egdst_solution *s, int ivec, int it, int ist, int id, double *M, int cap, int *rows) {
    if (!s || !rows) return fail(2, "invalid arguments");
    if (s->ncell_all == s->ncell) return fail(2, "the solution was computed without taste-shock smoothing (sigma_eps = 0): no choice-specific cells");
    const EgdstDev &P = s->P;
    if (ivec < 0 || ivec >= P.nvec || it < 0 || it >= P.NT || ist < 0 || ist >= P.cx.nst || id < 0 || id >= P.cx.nd) return fail(2, "cell index out of range");
    CK(cudaSetDevice(s->device));
    const int dcell = P.ncellMain + ((ivec * P.NT + it) * P.cx.nst + ist) * P.cx.nd + id;
    int n = 0;
    CK(cudaMemcpyAsync(&n, P.mlen + dcell, sizeof(int), cudaMemcpyDeviceToHost, g_stream));
    CK(cudaStreamSynchronize(g_stream));
    *rows = n;
    if (!M || n == 0) return 0;
    if (cap < n) return fail(2, "buffer too small for the cell");
    for (int c = 0; c < 4; c++)
        CK(cudaMemcpyAsync(M + (size_t)c * n, P.arena + ((size_t)dcell * 4 + c) * P.rowcap, sizeof(double) * n, cudaMemcpyDeviceToHost, g_stream));
    CK(cudaStreamSynchronize(g_stream));
    return 0;
}

int egdst_solution_status(egdst_solution *s, int ivec, int *it, int *ist, int *id) {
    if (!s || ivec < 0 || ivec >= s->P.nvec) return -1;
    if (fetch_sizes(s)) return -1;
    if (it) *it = s->h_status[4 * ivec + 1];
    if (ist) *ist = s->h_status[4 * ivec + 2];
    if (id) *id = s->h_status[4 * ivec + 3];
    const int code = s->h_status[4 * ivec];
    if (code) status_rc(s);
    return code;
}

int egdst_solution_nvec(const egdst_solution *s) { return s ? s->P.nvec : 0; }

// the solve work unit (SURVEY 8d): every EGM grid point stored for an (it, ist, id) -- the mgridvecs
// quadruples of egdst_solver.c:646-650, terminal period included; counted on the device by the kernels.
long long egdst_solution_units(egdst_solution *s) { return units_sum(s, 0); }

// diagnostic: zero-consumption re-sends requested by grid points after the seed stage (egdst_solver.c:1080-1099)
// that the last solve handled, over all vectors
long long egdst_solution_resends(egdst_solution *s) { return units_sum(s, 1); }

int egdst_solution_phase_ms(egdst_solution *s, double *ms) {
    // device time per phase of the solve kernel (terminal, seed, egm, resend, envelope2, rank, merge, tables), accumulated over
    // the solves of this object that ran while egdst_profile_enable(1) was in effect; reading resets the counters
    if (!s || !ms) return -1;
    if (cudaSetDevice(s->device) != cudaSuccess) return -1;
    unsigned long long ns[EGDST_NPHASE];
    if (cudaMemcpyAsync(ns, s->d_phase, sizeof(ns), cudaMemcpyDeviceToHost, g_stream) != cudaSuccess) return -1;
    if (cudaMemsetAsync(s->d_phase, 0, sizeof(ns), g_stream) != cudaSuccess) return -1;
    if (cudaStreamSynchronize(g_stream) != cudaSuccess) return -1;
    for (int i = 0; i < EGDST_NPHASE; i++) ms[i] = (double)ns[i] * 1e-6;
    return EGDST_NPHASE;
}

int egdst_test_envelope2(const egdst_desc *d, int it, int ist, int id, const double *X, const double *Cc, const double *V, int n, double evfa0,
                         double *outX, double *outC, double *outV, int *nout) {
    // diagnostic: the secondary upper envelope (envelope2, egdst_solver.c:776-913) of n EGM points of decision id in
    // generation order, run by the same phases as the solve; the counterpart of the reference harness of the tests
    if (!d || !X || !Cc || !V || !outX || !outC || !outV || !nout || n < 1) return fail(2, "invalid arguments");
    if (ist != 0 || id < 0 || id >= d->nd) return fail(2, "egdst_test_envelope2: ist must be 0 and id a decision index");
    if (n >= d->ngridmax) return fail(2, "egdst_test_envelope2: more points than ngridmax");
    egdst_solution *s = 0;
    int rc = create_solution(d, 1, &s);
    if (rc) return rc;
    SolutionGuard scratch(s, egdst_free_solution);
    const EgdstDev &P = s->P;
    cudaStream_t st = g_stream;
    cudaError_t ce = upload_tables(s, d, st);
    // the decision's slot is sd = 0 of the scratch object; its decision index travels in the view (ist = 0 => sd = id):
    // place the points in the slot of (ist 0, id) so that the analytic segment uses the right decision
    const size_t off = (size_t)id * P.gcap;
    EGDST_TRY(cudaMemsetAsync(P.status, 0, sizeof(int) * 4, st));
    EGDST_TRY(cudaMemcpyAsync(P.ptX + off, X, sizeof(double) * n, cudaMemcpyHostToDevice, st));
    EGDST_TRY(cudaMemcpyAsync(P.ptC + off, Cc, sizeof(double) * n, cudaMemcpyHostToDevice, st));
    EGDST_TRY(cudaMemcpyAsync(P.ptV + off, V, sizeof(double) * n, cudaMemcpyHostToDevice, st));
    EGDST_TRY(cudaMemcpyAsync(P.evfa0 + id, &evfa0, sizeof(double), cudaMemcpyHostToDevice, st));
    int nres = 0;
    if (ce == cudaSuccess) {
        KLAUNCH(KC_OTHER, egdst_k_env2_only, dim3(1), dim3(EGDST_BLOCK), EgdstScratch<EGDST_BLOCK>::bytes, st, P, it, n, id);
        EGDST_TRY(cudaGetLastError());
        EGDST_TRY(cudaMemcpyAsync(&nres, P.ptN + id, sizeof(int), cudaMemcpyDeviceToHost, st));
        EGDST_TRY(cudaStreamSynchronize(st));
    }
    if (ce == cudaSuccess && nres > 0) {
        EGDST_TRY(cudaMemcpyAsync(outX, P.ptX + off, sizeof(double) * nres, cudaMemcpyDeviceToHost, st));
        EGDST_TRY(cudaMemcpyAsync(outC, P.ptC + off, sizeof(double) * nres, cudaMemcpyDeviceToHost, st));
        EGDST_TRY(cudaMemcpyAsync(outV, P.ptV + off, sizeof(double) * nres, cudaMemcpyDeviceToHost, st));
        EGDST_TRY(cudaStreamSynchronize(st));
    }
    if (ce != cudaSuccess) return fail(2, std::string("CUDA error in egdst_test_envelope2: ") + cudaGetErrorString(ce));
    *nout = nres;
    return (rc = fetch_sizes(s)) ? rc : status_rc(s);
}

void egdst_free_solution(egdst_solution *s) {
    if (!s) return;
    {
        std::lock_guard<std::mutex> lk(g_cache_mu);
        if (!g_cached && s->bytes <= EGDST_CACHE_MAX_BYTES) { g_cached = s; return; }
    }
    destroy_solution(s);
}


int egdst_solution_import(const egdst_desc *d, const int *mlen, const int *thlen, const double *Mbuf, const double *Dbuf, egdst_solution **out) {
    if (!out || !mlen || !thlen || !Mbuf || !Dbuf) return fail(2, "invalid arguments");
    *out = 0;
    egdst_solution *s = 0;
    int rc = create_solution(d, 1, &s);
    if (rc) return rc;
    SolutionGuard guard(s, egdst_free_solution);
    for (int c = 0; c < s->ncell; c++) {
        if (mlen[c] > s->P.rowcap || thlen[c] > d->nthrhmax) return fail(2, "imported cell exceeds ngridmax/nthrhmax");
        if (mlen[c] < 0 || mlen[c] == 1 || thlen[c] < 0 || (mlen[c] == 0) != (thlen[c] == 0)) return fail(2, "imported cell has an invalid number of rows");
    }
    size_t nm = 0, nd2 = 0;
    if ((rc = pack_layout(s, mlen, thlen, &nm, &nd2))) return rc;
    cudaStream_t st = g_stream;
    cudaError_t ce = upload_tables(s, d, st);
    EGDST_TRY(cudaMemcpyAsync(s->d_pack, Mbuf, sizeof(double) * nm, cudaMemcpyHostToDevice, st));
    EGDST_TRY(cudaMemcpyAsync(s->d_pack + nm, Dbuf, sizeof(double) * nd2, cudaMemcpyHostToDevice, st));
    EGDST_TRY(cudaMemcpyAsync(s->P.mlen, mlen, sizeof(int) * s->ncell, cudaMemcpyHostToDevice, st));
    EGDST_TRY(cudaMemcpyAsync(s->P.thlen, thlen, sizeof(int) * s->ncell, cudaMemcpyHostToDevice, st));
    EGDST_TRY(cudaMemsetAsync(s->P.status, 0, sizeof(int) * 4, st));
    EGDST_TRY(cudaMemsetAsync(s->P.tabOk, 1, sizeof(int) * s->ncell_all, st));  // imported cells: usable unless egdst_k_tabonly finds a grid that steps back
    if (ce == cudaSuccess) {
        KLAUNCH(KC_OTHER, egdst_k_unpack, dim3(s->ncell), dim3(EGDST_BLOCK), 0, st, s->P, s->d_moff, s->d_toff, s->d_pack, s->d_pack + nm, s->ncell);
        const int tb = (s->P.lutcap + 1 + EGDST_BLOCK - 1) / EGDST_BLOCK;
        for (int it = 0; it < s->P.NT; it++) KLAUNCH(KC_TAB, egdst_k_tabonly, dim3(tb, d->nst, 1), dim3(EGDST_BLOCK), 0, st, s->P, it);
        EGDST_TRY(cudaGetLastError());
    }
    EGDST_TRY(cudaStreamSynchronize(st));
    if (ce != cudaSuccess) return fail(2, std::string("CUDA error in import: ") + cudaGetErrorString(ce));
    memcpy(s->h_mlen.data(), mlen, sizeof(int) * s->ncell);
    memcpy(s->h_thlen.data(), thlen, sizeof(int) * s->ncell);
    s->h_params.assign(d->params, d->params + EGDST_NPARAM);  // the imported model's own parameter values
    s->sizes_valid = true;
    *out = guard.release();
    return 0;
}

}  // extern "C"

#include "egdst_capi_sim.inc"
