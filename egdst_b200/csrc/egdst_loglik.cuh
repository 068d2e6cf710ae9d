// egdst_loglik.cuh -- log-likelihood of observed discrete choices (and consumption) under a taste-shock solution
// (opt-in extension of the smoothing mode; the reference has no counterpart).
//
// One thread per (observation, parameter vector); blockIdx.y walks the vectors as in egdst_k_simulate.  A row's
// choice probability is what the draw simulator evaluates at the same (it, ist, cash): egdst_choice_values and
// egdst_choice_weights, so the edge rules (unavailable decisions, held at the bound above the grid, equal weights when
// every value is -inf) have one implementation.  The per-vector total is deterministic: a fixed-order warp and block
// reduction writes one partial per block, and egdst_k_choice_loglik_sum adds the partials of a vector in a fixed
// order.  The block partition depends on nobs only, so the total of the same rows has the same bits for any nvec,
// ivec0 or launch.
//
// Finite mixtures over unobserved types (egdst_mixture_loglik) take three passes: egdst_k_choice_loglik writes the
// row values [nvec][nobs] to a scratch buffer (keeping its (row x vector) parallelism), egdst_k_indiv_loglik adds each
// individual's rows in row order (one thread per (individual, vector)), and egdst_k_mixture_loglik combines the types
// of each mixture per individual (one thread per (individual, mixture), blockIdx.y over the mixtures) and writes one
// fixed-order partial per block, which egdst_k_choice_loglik_sum adds up.  The block partition depends on nind only.
// So an individual's value under a vector does not depend on nvec, ivec0 or the launch, and a mixture's values and
// total have the same bits whether it is evaluated alone or with other mixtures, in any ivec0 window holding its vectors.
//
// Central-difference scores (egdst_mixture_scores) add one pass after those three: egdst_k_mixture_scores takes a fixed
// chunk of EGDST_SC_CHUNK individuals per block (a partition that depends on nind only), computes the chunk's
// s_ip = (mixll[mplus_p][i] - mixll[mminus_p][i]) * hinv_p into shared memory, and then one thread per entry of the
// list grad[0..P-1], opg[p][q] (p <= q) adds the chunk's terms in individual order and writes one partial per
// (entry, block); an off-diagonal partial goes to both opg[p][q] and opg[q][p].  egdst_k_choice_loglik_sum adds each
// entry's partials in a fixed order.  So grad[p], opg[p][q] and the scores depend only on the rows and on the mixtures
// and factors of components p and q: not on npar, the other components or their order, nvec, ivec0 or the launch.
#pragma once

#include "egdst_solver.cuh"

#ifdef EGDST_HOSTEMU
#define EGDST_LL_BLOCK 64
#else
#define EGDST_LL_BLOCK 256
#endif
// minimum resident blocks per SM of egdst_k_choice_loglik: 3 caps it at 80 registers (60 bytes of spill stores) where
// it needs 116 without a bound; 24 instead of 16 resident warps hide more of the table gathers' latency, and the
// kernel ran 1.19-1.29x faster so (tools/loglik_time.py, DESIGN 6b)
#ifndef EGDST_LL_MINBLOCKS
#define EGDST_LL_MINBLOCKS 3
#endif
// egdst_k_mixture_scores: individuals per block (fewer on the emulator, so that its tests cross block boundaries),
// threads per block, and the most score components per launch (shared memory holds [EGDST_SC_MAXPAR][chunk])
#ifdef EGDST_HOSTEMU
#define EGDST_SC_CHUNK 16
#define EGDST_SC_BLOCK 32
#else
#define EGDST_SC_CHUNK 64
#define EGDST_SC_BLOCK 128
#endif
#define EGDST_SC_MAXPAR 32

struct EgdstLlArgs {
    const double *obs;   // [k][nobs]: age, state (1-based), cash, decision (1-based), x_1..x_NCONT[, consumption]
    int nobs, k, ivec0;
    int prm_on;          // 1: the parameter values are param (a single model: this call's); 0: the solve's (P.bparams)
    double sigma_c;      // consumption measurement error (0: no consumption term)
    double param[EGDST_NPARAM_];
    double *rowll;       // [nvec][nobs] or null
    double *part;        // [nvec][gridDim.x] block partials
};

struct EgdstMixArgs {
    const double *indll; // [nvec][nind] per-individual values
    const int *tvec;     // [nmix][ntypes] vector of each type, relative to ivec0
    const double *w;     // [nmix][ntypes] type weights (normalised here)
    int nind, nvec, ntypes;
    double *mixll;       // [nmix][nind] or null
    double *post;        // [nmix][ntypes][nind] or null
    double *part;        // [nmix][gridDim.x] block partials
};

struct EgdstScoreArgs {
    const double *mixll; // [nmix][nind] per-individual mixture values
    const int *mplus;    // [npar] mixture of the upper member of each difference
    const int *mminus;   // [npar] mixture of the lower member
    const double *hinv;  // [npar] 1 / (theta_plus - theta_minus)
    int nind, nmix, npar;
    double *scores;      // [npar][nind] or null
    double *part;        // [npar + npar * npar][gridDim.x] block partials: grad, then opg row-major
};

#if EGDST_SMOOTHING
// log P_d(M) (+ the consumption term) of row i under the parameter values in cx; NaN for a malformed row.  With
// continuous states, P_d is that of the mixed choice values at the row's exact state x_1..x_NCONT (columns 4..) and the
// consumption term is centred on the consumption a choice draw records, min(c_d, M - a0) (egdst_choice_values_cont)
EGDST_DEV double egdst_choice_loglik_row(const EgdstDev &P, const egdst_ctx &cx, int ivec, const EgdstLlArgs &A, int i) {
    const size_t n = (size_t)A.nobs;  // column offsets in size_t: k * nobs exceeds INT_MAX for panels of 430 M rows
    const double age = A.obs[i], sti = A.obs[n + i], cash = A.obs[2 * n + i], dob = A.obs[3 * n + i];
    if (!(age >= cx.t0 && age <= cx.T && age == floor(age)) || !(sti >= 1 && sti <= cx.nst && sti == floor(sti)) ||
        !(dob >= 1 && dob <= cx.nd && dob == floor(dob)) || !(cash >= cx.a0 && cash < EGDST_INF))
        return EGDST_NAN;
    PeriodVars x;
    x.it = (int)age - cx.t0; x.ist = (int)sti - 1; x.id = (int)dob - 1;
    x.cash = cash; x.savings = 0; x.shock = 0;
    egdst_fill_state(&cx, &x);
    egdst_fill_decision(&cx, &x);
    const int id = x.id;
    EgdstChoiceVals cv;
#if EGDST_NCONT > 0
#pragma unroll
    for (int k = 0; k < EGDST_NCONT; k++) {
        const double xk = A.obs[(4 + k) * n + i];
        if (!(fabs(xk) < EGDST_INF)) return EGDST_NAN;
        x.st[egdst_contvar[k]] = xk;
    }
    int istrec;
    if (!egdst_choice_values_cont(P, &cx, ivec, x, cv, istrec)) return EGDST_NAN;
#else
    egdst_choice_values(P, &cx, egdst_cell(P, ivec, x.it, x.ist), x, cv);
#endif
    double ssum, wmax, ed = 0.0;
    egdst_choice_weights(cx.nd, cv, P.sigmaEps, ssum, wmax, [&](int d, double e) { if (d == id) ed = e; });
    // a decision without weight (not available, or exp underflows) has probability 0
    double ll = ed > 0.0 ? log(ed) - log(ssum) : -EGDST_INF;
    if (A.k == 5 + EGDST_NCONT && A.sigma_c > 0.0) {
        const double cobs = A.obs[(4 + EGDST_NCONT) * n + i];
        if (!isnan(cobs)) {
#if EGDST_NCONT > 0
            const double cd = MIN(cv.c[id], cash - cx.a0);  // the consumption a choice draw records
#else
            const double cd = cv.c[id];
#endif
            const double z = (cobs - cd) / A.sigma_c;
            ll += -0.5 * z * z - 0.91893853320467274178 - log(A.sigma_c);  // log phi(z) - log sigma_c
        }
    }
    return ll;
}

__global__ void __launch_bounds__(EGDST_LL_BLOCK, EGDST_LL_MINBLOCKS) egdst_k_choice_loglik(EgdstDev P, EgdstLlArgs A) {
    __shared__ double wsum[EGDST_LL_BLOCK / 32];
    const int i = blockIdx.x * EGDST_LL_BLOCK + threadIdx.x;
    const int v = blockIdx.y, ivec = A.ivec0 + v;
    double ll = 0.0;
    if (i < A.nobs) {
        egdst_ctx cx; egdst_load_ctx(P, ivec, cx);
        cx.status = 0;
#if EGDST_NCONT > 0
        cx.byval = 1;  // model functions read the row's exact continuous state from x.st
#endif
        if (A.prm_on) {
#pragma unroll
            for (int j = 0; j < EGDST_NPARAM; j++) cx.param[j] = A.param[j];
        }
        ll = egdst_choice_loglik_row(P, cx, ivec, A, i);
        if (A.rowll) A.rowll[(size_t)v * A.nobs + i] = ll;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ll += __shfl_down_sync(0xffffffffu, ll, o);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = ll;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int w = 0; w < EGDST_LL_BLOCK / 32; w++) s += wsum[w];
        A.part[(size_t)v * gridDim.x + blockIdx.x] = s;
    }
}

// loglik[v] += the sum of the nblocks partials of vector v (one warp per vector, lanes stride the partials)
__global__ void __launch_bounds__(32) egdst_k_choice_loglik_sum(const double *part, int nblocks, double *loglik) {
    const int v = blockIdx.x, lane = threadIdx.x;
    double s = 0.0;
    for (int b = lane; b < nblocks; b += 32) s += part[(size_t)v * nblocks + b];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if (lane == 0) loglik[v] += s;
}

// indll[v][i] = the rows start[i]..start[i+1]-1 of rowll[v], added in row order (0 for an empty individual; NaN for
// offsets that decrease or leave 0..nobs, which only the _device entry point lets through)
__global__ void __launch_bounds__(EGDST_LL_BLOCK) egdst_k_indiv_loglik(const double *rowll, int nobs, const int *start,
                                                                      int nind, double *indll) {
    const int i = blockIdx.x * EGDST_LL_BLOCK + threadIdx.x, v = blockIdx.y;
    if (i >= nind) return;
    const int lo = start[i], hi = start[i + 1];
    double s = 0.0;
    if (lo < 0 || hi < lo || hi > nobs) {
        s = EGDST_NAN;
    } else {
        const double *r = rowll + (size_t)v * nobs;
        for (int j = lo; j < hi; j++) s += r[j];
    }
    indll[(size_t)v * nind + i] = s;
}

// mixture x = blockIdx.y, individual i: over the types k with w_k > 0 (ascending), a_k = log(w_k / sum w) +
// indll[tvec_k][i], m = max a_k, mixll = m + log sum exp(a_k - m) (-inf when m = -inf), post_k = exp(a_k - m) / sum
// (0 for zero weights, NaN when mixll is -inf or NaN).  A type vector outside 0..nvec-1 (the _device entry point does
// not check them) gives NaN.
__global__ void __launch_bounds__(EGDST_LL_BLOCK) egdst_k_mixture_loglik(EgdstMixArgs A) {
    __shared__ double wsum[EGDST_LL_BLOCK / 32];
    const int i = blockIdx.x * EGDST_LL_BLOCK + threadIdx.x, x = blockIdx.y, nk = A.ntypes;
    const int *tv = A.tvec + (size_t)x * nk;
    const double *w = A.w + (size_t)x * nk;
    double ll = 0.0;
    if (i < A.nind) {
        double wt = 0.0;
        for (int k = 0; k < nk; k++) wt += w[k];
        auto a = [&](int k) {
            const int t = tv[k];
            return t >= 0 && t < A.nvec ? log(w[k] / wt) + A.indll[(size_t)t * A.nind + i] : EGDST_NAN;
        };
        double m = -EGDST_INF;  // NaN-propagating maximum
        for (int k = 0; k < nk; k++) {
            if (!(w[k] > 0.0)) continue;
            const double ak = a(k);
            if (ak > m || isnan(ak)) m = ak;
        }
        double s = 0.0;
        for (int k = 0; k < nk; k++)
            if (w[k] > 0.0) s += exp(a(k) - m);
        const bool none = m == -EGDST_INF;
        ll = none ? -EGDST_INF : m + log(s);
        if (A.mixll) A.mixll[(size_t)x * A.nind + i] = ll;
        if (A.post) {
            double *p = A.post + (size_t)x * nk * A.nind + i;
            for (int k = 0; k < nk; k++)
                p[(size_t)k * A.nind] = !(w[k] > 0.0) ? 0.0 : none ? EGDST_NAN : exp(a(k) - m) / s;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ll += __shfl_down_sync(0xffffffffu, ll, o);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = ll;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int k = 0; k < EGDST_LL_BLOCK / 32; k++) s += wsum[k];
        A.part[(size_t)x * gridDim.x + blockIdx.x] = s;
    }
}

// individuals blockIdx.x * EGDST_SC_CHUNK.. : s_ip = (mixll[mplus_p][i] - mixll[mminus_p][i]) * hinv_p (NaN for a
// mixture index outside 0..nmix-1, which only the _device entry point lets through), then one partial per block of
// each entry: grad[p] = sum s_ip and opg[p][q] = sum s_ip s_iq, added in individual order
__global__ void __launch_bounds__(EGDST_SC_BLOCK) egdst_k_mixture_scores(EgdstScoreArgs A) {
    constexpr int LD = EGDST_SC_CHUNK + 1;  // padded row: the entries' threads read different rows at one column
    __shared__ double sc[EGDST_SC_MAXPAR * LD];
    const int i0 = blockIdx.x * EGDST_SC_CHUNK, np = A.npar;
    const int n = A.nind - i0 < EGDST_SC_CHUNK ? A.nind - i0 : EGDST_SC_CHUNK;
    for (int e = threadIdx.x; e < np * EGDST_SC_CHUNK; e += EGDST_SC_BLOCK) {
        const int p = e / EGDST_SC_CHUNK, j = e % EGDST_SC_CHUNK, i = i0 + j;
        if (j >= n) continue;
        const int a = A.mplus[p], b = A.mminus[p];
        const double s = a >= 0 && a < A.nmix && b >= 0 && b < A.nmix
                             ? (A.mixll[(size_t)a * A.nind + i] - A.mixll[(size_t)b * A.nind + i]) * A.hinv[p]
                             : EGDST_NAN;
        sc[p * LD + j] = s;
        if (A.scores) A.scores[(size_t)p * A.nind + i] = s;
    }
    __syncthreads();
    const size_t nb = gridDim.x;
    for (int e = threadIdx.x; e < np + np * (np + 1) / 2; e += EGDST_SC_BLOCK) {
        if (e < np) {
            const double *x = sc + e * LD;
            double s = 0.0;
            for (int j = 0; j < n; j++) s += x[j];
            A.part[e * nb + blockIdx.x] = s;
        } else {
            int p = 0, r = e - np;  // the upper triangle row by row: (0,0), (0,1), .., (0,P-1), (1,1), ..
            while (r >= np - p) r -= np - p++;
            const int q = p + r;
            const double *x = sc + p * LD, *y = sc + q * LD;
            double s = 0.0;
            for (int j = 0; j < n; j++) s += x[j] * y[j];
            A.part[(np + p * np + q) * nb + blockIdx.x] = s;
            A.part[(np + q * np + p) * nb + blockIdx.x] = s;
        }
    }
}
#endif  // EGDST_SMOOTHING
