/* egdst_b200.h -- C ABI of the B200-native egdst solver / simulator library.
 *
 * One shared library is built per generated model image (libegdst_b200_<key>.so: the user's exec
 * strings compiled into the sm_100a kernels).  Its entry points are what the reference's three MEX
 * gateways bind (INTEGRATION.md shows the MEX stubs):
 *
 *   egdst_solve        replaces  [M,D,dbg] = egdst_solver(model)      @egdstmodel/egdst_solver.c:143-239
 *   egdst_simulate     replaces  sims = egdst_simulator(model,rnd)    @egdstmodel/egdst_simulator.c:47-117
 *   egdst_call         replaces  res  = egdst_call(model,sw,args)     @egdstmodel/egdst_call.c:17-125
 *   egdst_desc         replaces  parseModel()/loadparameters()        @egdstmodel/egdst_lib.c:34-62, compile.m:469-474
 *   egdst_last_error   replaces  err[300] / mexWarnMsgTxt / mexErrMsgTxt  egdst_lib.c:299-302, egdst_solver.c:237
 *
 * plus the multi-GPU / batched entry points the reference does not have (egdst_solve_batch,
 * egdst_sim_moments, Philox-driven simulation).
 *
 * Conventions: plain pointers and sizes, caller owns every input and output buffer, the library owns
 * egdst_solution objects until egdst_free_solution.  Return codes: 0 ok; 1 soft error (partial result
 * kept, message available -- the reference warns and returns partial M,D, egdst_solver.c:237); 2 hard
 * error (mexErrMsgTxt in the reference).  All device work runs on the stream set with egdst_set_stream
 * (default: the legacy default stream).  There is no CPU path: without a CUDA device every compute
 * entry point returns 2 with "no CUDA device".
 */
#ifndef EGDST_B200_H
#define EGDST_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define EGDST_ABI_VERSION 2

/* The model object flattened to a POD: exactly the properties the reference reads across the MEX
 * boundary (egdst_lib.c:37-55, compile.m:472, egdst_solver.c:162) plus the -D flags of compile.m:757-777. */
typedef struct egdst_desc {
    int abi_version;
    int t0, T, ngridm, ngridmax, nthrhmax, ny, nd, nnd, nst, nnst;
    double mmax, a0;
    int optim_UasD, optim_MUnoD, optim_UnoD, optim_TRPRnoSH;
    double tolerance, zeroconsumption, doublepoint_delta; /* cflags TOLERANCE, ZEROCONSUMPTION, DOUBLEPOINT_DELTA */
    const double *stm;        /* [2*nnst]                                       */
    const double *states;     /* [nst*nnst] column-major                        */
    const double *decisions;  /* [nd*nnd]  column-major                         */
    const double *params;     /* [nparam] param(i).value                        */
    int nparam;
    const double *quadrature; /* [2*ny] weights then abscissas in (0,1), as model.quadrature (may be NULL if ny==1) */
    int neq;                  /* numel(model.eq)                                 */
    int device;               /* CUDA device ordinal                             */
    double sigma_eps;         /* EXTENSION (no reference counterpart; 0 = off = the reference's hard max): scale of additive
                               * extreme-value taste shocks on the discrete choice.  > 0: the expectation uses the logsum and the
                               * choice probabilities of the choice-specific value functions (egdst_solution_choice_cell)   */
} egdst_desc;

typedef struct egdst_solution egdst_solution;

/* library / model-image introspection */
int egdst_abi_version(void);
const char *egdst_model_key(void);   /* key of the model image compiled into this library */
int egdst_model_nparam(void);
int egdst_model_neq(void);
const char *egdst_last_error(void);  /* per-thread message of the last non-zero return */
void egdst_set_stream(void *cuda_stream);
/* measurement aids: number of kernels launched by this library so far; optional CUDA-event timing of
 * every launch, accumulated per kernel class (setup, solve, tables, simulate, other).  Profiling adds two event
 * records per launch and switches the solve kernel's phase timers on -- never enable it in a timed region. */
long long egdst_launch_count(void);
int egdst_profile_classes(void);
const char *egdst_profile_class_name(int cls);
void egdst_profile_enable(int on);
int egdst_profile_read(double *ms, long long *count); /* arrays of egdst_profile_classes() entries */

/* ---- solve ------------------------------------------------------------------------------- */
/* Backward induction for one model.  *out receives a new solution object (device resident). */
int egdst_solve(const egdst_desc *d, egdst_solution **out);
/* nvec parameter vectors of the same model solved in one pass (params: [nvec*nparam], row = vector). */
int egdst_solve_batch(const egdst_desc *d, const double *params, int nvec, egdst_solution **out);
/* Re-run the solve into an existing solution object (same dimensions; new parameter values allowed).
 * Asynchronous on the library stream: no host synchronisation, no allocation. */
int egdst_resolve(egdst_solution *s, const egdst_desc *d, const double *params);
/* Rows per cell.  mlen/thlen: [nvec*NT*nst], index (ivec*NT+it)*nst+ist; 0 rows = infeasible (it,ist). */
int egdst_solution_sizes(egdst_solution *s, int *mlen, int *thlen);
/* Packed copy-out in cell order: M cell = mlen x 4 column-major (M,C,A,V; row 0 = a0,0,a0,evf(a0)),
 * D cell = thlen x 2 column-major (decision index, threshold) -- the layouts of saveoutput,
 * egdst_solver.c:917-951.  Mbuf holds 4*sum(mlen) doubles, Dbuf 2*sum(thlen). */
int egdst_solution_export(egdst_solution *s, double *Mbuf, double *Dbuf);
/* EXTENSION, smoothing mode only (desc.sigma_eps > 0): the choice-specific cell of decision id in (it, ist) -- what the
 * reference discards after envelop() (egdst_solver.c:720-730).  rows x 4 column-major (M,C,A,V; row 0 = a0,0,a0,
 * evf_d(a0)); *rows = 0: decision not available.  M may be NULL to query the row count. */
int egdst_solution_choice_cell(egdst_solution *s, int ivec, int it, int ist, int id, double *M, int cap, int *rows);
/* status of the last (re)solve of vector ivec: returns the code, fills it/ist/id of the first failure */
int egdst_solution_status(egdst_solution *s, int ivec, int *it, int *ist, int *id);
int egdst_solution_nvec(const egdst_solution *s);
/* total number of EGM grid points kept over all (it,ist,id) of the last solve (the solve work unit) */
long long egdst_solution_units(egdst_solution *s);
/* diagnostic: how many zero-consumption re-sends requested by grid points AFTER the seed stage of the savings grid
 * (egdst_solver.c:1080-1099) the last solve went through */
long long egdst_solution_resends(egdst_solution *s);
/* measurement aid: device time in ms per phase of the solve kernel -- terminal, seed, egm, resend, envelope2, rank,
 * merge, tables (8 entries) -- accumulated over this object's solves while egdst_profile_enable(1) was in effect;
 * reading resets the counters.  Returns the number of entries. */
int egdst_solution_phase_ms(egdst_solution *s, double *ms);
/* diagnostic: the secondary upper envelope (envelope2, egdst_solver.c:776-913) of n EGM points (M, C, V_d) of decision
 * id (state 0, period it) in generation order, run by the solve kernel's own phases.  out*: room for ngridmax
 * doubles each; *nout receives the number of points kept.  The tests compare it with the reference's envelope2. */
int egdst_test_envelope2(const egdst_desc *d, int it, int ist, int id, const double *X, const double *C, const double *V, int n,
                         double evfa0, double *outX, double *outC, double *outV, int *nout);
void egdst_free_solution(egdst_solution *s);
/* Frees what the library keeps between calls: the one released solution object it caches for re-use by the next
 * solve of the same shape, and the calling thread's simulation workspace.  (The reference leaks on error paths and
 * relies on MATLAB clearing the MEX file, egdst_solver.c:19; a long-lived host calls this when it unloads a model.) */
void egdst_shutdown(void);
/* Build a solution object from host M/D cells (the MEX simulator receives model.M, model.D). */
int egdst_solution_import(const egdst_desc *d, const int *mlen, const int *thlen, const double *Mbuf, const double *Dbuf,
                          egdst_solution **out);

/* ---- simulate ---------------------------------------------------------------------------- */
/* sims: [nsimout, nt, nsim] column-major doubles, nsimout = 11+nnst+nnd+neq, NaN after death
 * (egdst_simulator.c:95-143).  init: [nsim*2] column-major (1-based ist0, m0).  randstream: U(0,1),
 * 4 slots per agent-period; rndtype 0 = own shocks, 1 = same shocks (egdst_simulator.c:71-75,109-114). */
int egdst_simulate(const egdst_desc *d, egdst_solution *s, int ivec, const double *init, int nsim,
                   const double *randstream, long long nrand, int rndtype, double *sims);
/* Same simulation with counter-based Philox4x32-10 uniforms generated on the device (no randstream).
 * agent0 = global index of the first agent (results do not depend on how agents are sharded).
 * sims may be NULL (moments only).  moments: [3, nsimout, nt] = sum x, sum x^2, alive count. */
int egdst_simulate_philox(const egdst_desc *d, egdst_solution *s, int ivec, const double *init, int nsim,
                          long long agent0, unsigned long long seed, double *sims, double *moments);
/* device-resident variants for sharded multi-GPU runs: d_init [nsim*2], d_sims / d_moments device pointers
 * (either may be NULL); asynchronous on the library stream. */
int egdst_simulate_device(const egdst_desc *d, egdst_solution *s, int ivec, const double *d_init, int nsim,
                          long long agent0, unsigned long long seed, const double *d_randstream, int rndtype,
                          double *d_sims, double *d_moments);

/* Estimation sweeps: moments-only simulation of the same agents (and the same Philox shocks) under parameter
 * vectors ivec0..ivec0+nvec-1 of a batched solution, in one launch.  moments: [nvec][3*nsimout*nt].
 * The _device variant takes device pointers, is asynchronous on the library stream and accumulates into
 * d_moments (the caller zeroes it), so a rank can all-reduce the buffer right after. */
int egdst_sim_moments(const egdst_desc *d, egdst_solution *s, int ivec0, int nvec, const double *init, int nsim,
                      long long agent0, unsigned long long seed, double *moments);
int egdst_sim_moments_device(const egdst_desc *d, egdst_solution *s, int ivec0, int nvec, const double *d_init, int nsim,
                             long long agent0, unsigned long long seed, double *d_moments);

/* EXTENSION, smoothing mode only (desc.sigma_eps > 0): choice draws.  on != 0: every later simulation of s (all the
 * simulate and moments entry points above) draws each period's decision d from the choice probabilities the solve
 * weighs the decisions with, P_d(M) = softmax_d(v_d(M)/sigma_eps) over the available decisions (held at their values
 * at the grid's bound above it; equal when every value is -inf): d is the first available decision whose cumulative
 * probability reaches a uniform u.  The record is then that of d's choice cell (egdst_solution_choice_cell):
 * consumption c_d(M), savings M - c, value v_d(M) (without the realised taste shock), decision d, utility and discount
 * of (c, d).  No available decision: the record is NaN from that period on.  on = 0 (the default): the decision of
 * the merged policy's thresholds, the modal choice.  The uniform of period it (0..nt-1):
 *   randstream  slot 3*(nt-1)+it of the agent's 4*nt block (the transitions use slots 0..3*(nt-1)-1), shared by all
 *               agents with rndtype 1 as the other slots are;
 *   Philox      word 3 of the block of counter (agent, it), whose words 0-2 drive the transition into it.
 * Returns 2 when on != 0 for a solution without choice cells (sigma_eps = 0, or imported), or for a model image with
 * continuous states.  The setting belongs to the solution object: egdst_resolve keeps it, a new solve starts with
 * it off. */
int egdst_solution_set_choice_draws(egdst_solution *s, int on);

/* EXTENSION, smoothing images only: log-likelihood of observed choices (and consumption) under the parameter vectors
 * ivec0..ivec0+nvec-1 of s, one launch.  obs: [nobs x k] column-major, k = 4 or 5, rows as in egdst_call:
 *   0 age (t0..T; period it = age - t0), 1 state ist (1-based), 2 cash-in-hand M at the start of the period (the cash
 *   column of a simulation record), 3 observed decision id (1-based), 4 (k = 5) observed consumption c_obs, NaN: not
 *   observed.
 * Per row and vector:  ll = log P_d(M) + [log phi((c_obs - c_d(M)) / sigma_c) - log sigma_c]
 * with the bracket only when k = 5, sigma_c > 0 and c_obs is not NaN; phi is the standard normal density.  P_d(M)
 * and c_d(M) are exactly what the choice draws evaluate (the probability rule of the solve, egdst_solution_set_choice_draws:
 * held at the bound above the grid, equal weights when every value is -inf, the credit-constrained branch below the
 * first grid point), and log P_d = log e_d - log sum_d' e_d' of its weights.  A row contributes -inf when its decision
 * is not available in (it, ist) or its weight underflows (a non-modal choice as sigma_eps -> 0): such a total is -inf.
 * Parameter values: a batched solution uses the vectors it was solved with, a single model those of d (as the
 * simulate entry points do).
 *   loglik  [nvec] per-vector totals (overwritten).  rowll: [nvec][nobs] per-row values, or NULL.
 * The totals are deterministic: the rows are summed in a fixed order over a block partition that depends on nobs only,
 * so the same obs give the same bits whatever nvec, ivec0 or launch.  The host entry point checks every row and
 * returns 2, naming the first malformed row, for an age, state or decision that is not an integer in range, or cash
 * that is not finite or lies below a0.  Returns 2 as well for a solution without choice cells (sigma_eps = 0, or
 * imported), an image with continuous states or without smoothing, k not 4 or 5, sigma_c < 0, or a vector range out of
 * bounds (at most 65535 vectors).  The _device variant takes device pointers, is asynchronous on the library stream,
 * checks no rows (a malformed row gets rowll = NaN, and its vector's total is NaN) and adds each vector's total to
 * d_loglik (the caller zeroes it), so a rank can all-reduce the buffer right after. */
int egdst_choice_loglik(const egdst_desc *d, egdst_solution *s, int ivec0, int nvec, const double *obs, int nobs, int k,
                        double sigma_c, double *loglik, double *rowll);
int egdst_choice_loglik_device(const egdst_desc *d, egdst_solution *s, int ivec0, int nvec, const double *d_obs, int nobs,
                               int k, double sigma_c, double *d_loglik, double *d_rowll);

/* EXTENSION, smoothing images only: finite-mixture log-likelihood over unobserved types (Keane-Wolpin types), for
 * nmix mixtures of ntypes types each, one launch.  obs and its rows are those of egdst_choice_loglik, grouped by
 * individual: individual i owns rows start[i]..start[i+1]-1 (start [nind+1]: start[0] = 0, non-decreasing,
 * start[nind] = nobs; empty individuals are allowed).  tvec [nmix][ntypes]: the vector of each type, relative to ivec0
 * (0..nvec-1; a vector may serve several types and mixtures).  w [nmix][ntypes]: type weights, finite and >= 0 with a
 * positive sum per mixture, normalised here (w~_k = w_k / sum_k w_k), so unnormalised or softmax weights can be passed.
 *   indll [nvec][nind]:  L_i(v) = the sum of individual i's row values under vector v (0 for an empty individual).
 *   mixll [nmix][nind]:  over the types k with w_k > 0 only, a_k = log w~_k + L_i(tvec_k), m = max_k a_k and
 *                        mixll = m + log sum_k exp(a_k - m), summed in ascending k; -inf when m = -inf.
 *   post [nmix][ntypes][nind]: the posterior type probabilities exp(a_k - m) / sum; 0 for zero-weight types, NaN for
 *                        the other types where mixll is -inf (or NaN).
 *   loglik [nmix]:       the sum of mixll over individuals (overwritten by the host entry point).
 * Zero-weight types are skipped entirely: a -inf or NaN under them does not matter.  ntypes = 1 with any positive
 * weight gives mixll == indll bit for bit.  indll, mixll and post are optional (NULL).
 * Determinism: the rows of an individual are added in row order and mixtures are summed over a block partition that
 * depends on nind only.  So an individual's indll under a vector does not depend on nvec, ivec0 or the launch, and a
 * mixture's mixll, post and total have the same bits whether it is evaluated alone or with other mixtures, and in any
 * ivec0 window holding its vectors.
 * Returns 2 under the conditions of egdst_choice_loglik (the host entry point checks every row) and for nind < 0,
 * ntypes < 1, nmix < 1 or nmix > 65535.  The host entry point also returns 2, naming the first offending index, for
 * offsets that do not start at 0, decrease or do not end at nobs, a tvec entry outside 0..nvec-1, a weight that is
 * negative or not finite, and a mixture whose weights sum to 0.  The _device variant takes device pointers (d_start
 * and d_tvec int32), is asynchronous on the library stream, checks no rows, offsets, type vectors or weights (a
 * malformed row makes its individual's indll NaN, and so the mixll and totals of every mixture that gives it positive
 * weight; a malformed offset or type vector gives NaN likewise) and adds each mixture's total to d_loglik (the caller
 * zeroes it).  It keeps the row values [nvec][nobs] (and indll when d_indll is NULL) in grow-only buffers of s. */
int egdst_mixture_loglik(const egdst_desc *d, egdst_solution *s, int ivec0, int nvec, const double *obs, int nobs, int k,
                         double sigma_c, const int *start, int nind, int ntypes, int nmix, const int *tvec, const double *w,
                         double *loglik, double *indll, double *mixll, double *post);
int egdst_mixture_loglik_device(const egdst_desc *d, egdst_solution *s, int ivec0, int nvec, const double *d_obs, int nobs,
                                int k, double sigma_c, const int *d_start, int nind, int ntypes, int nmix, const int *d_tvec,
                                const double *d_w, double *d_loglik, double *d_indll, double *d_mixll, double *d_post);

/* EXTENSION, smoothing images only: central-difference scores of mixture log-likelihoods, with their sum (the
 * gradient) and the outer-product-of-gradients (OPG) matrix, one launch after the passes of egdst_mixture_loglik.  obs,
 * start, tvec and w are those of egdst_mixture_loglik.  A plain one-type likelihood is the mixture with ntypes = 1 and
 * weight 1 (mixll == indll bit for bit).  Component p (npar of them, 1..32) is the pair of mixtures mplus[p], mminus[p]
 * (0..nmix-1) and the factor hinv[p] = 1 / (theta_plus - theta_minus), computed by the caller from the perturbed values
 * actually solved (a forward difference is the pair (perturbed, centre)).  Parameters that enter the solve are
 * perturbed as vectors of the batch, type weights as mixtures over the same vectors.  Per individual i:
 *   s_ip = (mixll[mplus[p]][i] - mixll[mminus[p]][i]) * hinv[p]
 *   grad [npar]:         sum_i s_ip.
 *   opg [npar][npar]:    sum_i s_ip s_iq, both triangles from one sum (opg[q][p] has the bits of opg[p][q]).
 *   loglik [nmix]:       the mixture totals of egdst_mixture_loglik.
 *   scores [npar][nind]: s_ip, or NULL.
 * An individual whose mixll is -inf under both members of a pair gets a NaN score, and that NaN propagates into grad
 * and opg (-inf under one member only gives an infinite score); neither is masked.
 * Determinism: the individuals are summed in index order within blocks of a partition that depends on nind only, and
 * the block partials in a fixed order.  So grad[p], opg[p][q] and the scores of p depend only on the rows and on the
 * mixtures and hinv of components p and q: not on npar, on which other components are requested or in what order, on
 * nvec or ivec0, or on the launch.
 * Returns 2 under the conditions of egdst_mixture_loglik (the host entry point checks every row, offset, type vector
 * and weight) and for npar < 1 or npar > 32.  The host entry point also returns 2, naming the first offending
 * component, for an mplus or mminus entry outside 0..nmix-1 and a hinv that is 0 or not finite; it overwrites loglik,
 * grad and opg.  The _device variant takes device pointers (d_start, d_tvec, d_mplus and d_mminus int32), is
 * asynchronous on the library stream, checks no data (an out-of-range mixture index gives NaN scores, never an
 * out-of-bounds read) and adds into d_loglik, d_grad and d_opg (the caller zeroes them).  It keeps the row, individual
 * and mixture values in grow-only buffers of s. */
int egdst_mixture_scores(const egdst_desc *d, egdst_solution *s, int ivec0, int nvec, const double *obs, int nobs, int k,
                         double sigma_c, const int *start, int nind, int ntypes, int nmix, const int *tvec, const double *w,
                         int npar, const int *mplus, const int *mminus, const double *hinv, double *loglik, double *grad,
                         double *opg, double *scores);
int egdst_mixture_scores_device(const egdst_desc *d, egdst_solution *s, int ivec0, int nvec, const double *d_obs, int nobs,
                                int k, double sigma_c, const int *d_start, int nind, int ntypes, int nmix, const int *d_tvec,
                                const double *d_w, int npar, const int *d_mplus, const int *d_mminus, const double *d_hinv,
                                double *d_loglik, double *d_grad, double *d_opg, double *d_scores);

/* ---- call -------------------------------------------------------------------------------- */
/* sw: 1 utility, 2 marginal utility, 3 discount, 4 budget, 5 marginal budget, 6 value function;
 * args: [narg*k] column-major with k = 4,4,2,6,6,3 (egdst_call.c:45-58); res: [narg]. */
int egdst_call(const egdst_desc *d, egdst_solution *s, int sw, const double *args, int narg, int k, double *res);

#ifdef __cplusplus
}
#endif
#endif
