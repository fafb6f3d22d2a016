/*
 * gpmc.h -- C ABI of libgpmc.so: the B200 (sm_100a) implementation of the GP
 * log-marginal-likelihood hot path of t-kychen/GaussianProcess-MCMC.
 *
 * The reference has no FFI: its boundary is the Python call
 * kcMCMC/sliceSample.py:76  surrogate_slice_sampling(f, x, y, hyp, scale, iter)
 * and, below it, the kcGP primitives imported at sliceSample.py:13.  Each entry
 * point here states the reference lines it replaces.  INTEGRATION.md shows the
 * ctypes binding a reference maintainer would add.
 *
 * Conventions
 *  - plain pointers and sizes only; no torch / C++ types cross this boundary.
 *  - every array is FP64 (IEEE double), C order (row-major), as numpy gives the
 *    reference; `ld` is the leading dimension (elements between row starts).
 *  - pointers named *_dev are DEVICE pointers, *_host are HOST pointers.
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *  - return value: 0 on success, a cudaError_t (>0) on a CUDA failure, or a
 *    negative GPMC_E* code for a bad argument.  gpmc_last_error() gives text.
 *    Nothing is thrown across the ABI.  Numerical status is per item in
 *    info[b]: 0 ok, k>0 = leading minor k not positive definite (LAPACK dpotrf
 *    convention), GPMC_INFO_NOT_PD (-1) = the jitchol ladder gave up (the
 *    reference raises numpy.linalg.LinAlgError there).
 *  - the caller owns every buffer including workspace, sized by
 *    gpmc_workspace_bytes().
 *  - hyper-parameter rows are natural scale, hyp[b] = (ell_1..ell_E, sf, sn)
 *    with E = 1 (GPMC_KIND_SE_ISO, the reference's covK.RBF, and the Matern
 *    kinds) or E = D (GPMC_KIND_SE_ARD); P = E + 2.  Every entry point that
 *    takes `kind` accepts the five kinds below and returns GPMC_EINVAL for any
 *    other value, or for a P that does not fit the kind.
 *  - threading: like the reference (one Python thread, sliceSample.py uses the
 *    global numpy RNG) the library is meant for one host thread per process and
 *    one process per GPU; it keeps per-process state (side streams and events of
 *    the look-ahead schedule, the host-path staging buffers, the pinned status
 *    ring of the resident sampler loop -- one per device --, tuning switches).
 *    Every computing entry point takes a process-wide recursive lock, so calls
 *    from several host threads are SERIALISED, not racing; gpmc_last_error() is
 *    per thread; kernel attributes are set per device, so a thread may drive
 *    several devices in turn.  Calls are asynchronous on `stream` except where a
 *    jitter policy needs info[] on the host (one synchronisation per wave) and
 *    inside gpmc_sds_sweep / gpmc_sds_run, which return when the last chain has
 *    finished (the host polls a status word meanwhile).
 */
#ifndef GPMC_H
#define GPMC_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GPMC_VERSION 100

/* covariance functions (`kind`), with u = x / ell (SE) or u = sqrt(d) x / ell (Matern), s = |u_i - u_j|^2, t = sqrt(s):
 *   SE:          K = sf2 * exp(-0.5 * s)                            (pyGPs 1.3.4 cov.RBF / cov.RBFard)
 *   Matern d:    K = sf2 * (f_d(t) * exp(-t)),  f_1 = 1, f_3 = 1 + t, f_5 = 1 + t * (1 + t / 3)
 *                (pyGPs 1.3.4 cov.Matern(log_ell, d, log_sigma) as restated in oracle/matern_oracle.py; d = 2 nu, isotropic)
 * sf2 = sf^2; K_ii = sf2 for every kind. */
#define GPMC_KIND_SE_ISO 0
#define GPMC_KIND_SE_ARD 1
#define GPMC_KIND_MATERN1 2
#define GPMC_KIND_MATERN3 3
#define GPMC_KIND_MATERN5 4

/* flags of gpmc_cov_assemble */
#define GPMC_ASM_ADD_S      1   /* add S_ii (sliceSample.py:184-190) on the diagonal */
#define GPMC_ASM_LOWER_ONLY 2   /* write only tiles on/below the diagonal (internal fast path) */
#define GPMC_ASM_PRED       4   /* K / sn^2 + I, the matrix inf_mcmc factors (sliceSample.py:256-257) */

/* jitter policies of the Cholesky (kcGP.tools.jitchol semantics) */
#define GPMC_JITTER_NONE    0   /* one dpotrf attempt, asynchronous, info as LAPACK */
#define GPMC_JITTER_PYGPS   1   /* pyGPs 1.3.4 ladder: mean(diag)*1e-6*10^k, k<5 (one host sync) */

#define GPMC_INFO_NOT_PD   (-1)

#define GPMC_EINVAL   (-22)
#define GPMC_ENOMEM   (-12)
#define GPMC_EALIGN   (-14)

/* workspace query ops */
#define GPMC_OP_POTRF   1
#define GPMC_OP_LOGLIK  2
#define GPMC_OP_SDS     3
#define GPMC_OP_LOGLIK_GRAD 4
#define GPMC_OP_MARGINAL 5

int gpmc_version(void);
/* panel width (block-column width) of the blocked Cholesky this build was compiled with: 64 or 128 */
int gpmc_panel_width(void);
const char *gpmc_last_error(void);
/* sm count, compute capability, total HBM bytes of the current device */
int gpmc_device_info(int *sm_count, int *cc_major, int *cc_minor, size_t *hbm_bytes);

size_t gpmc_workspace_bytes(int op, int N, int D, int B);

/*
 * Fused covariance assembly.  Replaces
 *   covK.RBF(np.log(ll), np.log(sf)).getCovMatrix(x, mode='train')   sliceSample.py:104-105,136-137
 *   S build / K+S                                                     sliceSample.py:183-190,207
 * A[b] = sf_b^2 * exp(-0.5 * sum_d ((x_id - x_jd)/ell_bd)^2), or the Matern K of `kind`  (+ S_ii on the diagonal with
 * GPMC_ASM_ADD_S; + jitter_dev[b] when jitter_dev != NULL).  Full symmetric fill unless
 * GPMC_ASM_LOWER_ONLY.  x_dev[N,D]; hyp_dev[B,P]; A_dev[B][N][ld], ld >= N, ld even.
 */
int gpmc_cov_assemble(const double *x_dev, int N, int D, const double *hyp_dev, int B, int P,
                      int kind, int flags, const double *jitter_dev,
                      double *A_dev, int ld, void *stream);

/*
 * Batched lower Cholesky, in place.  Replaces kcGP.tools.jitchol (pyGPs 1.3.4 tools.jitchol ->
 * LAPACK dpotrf(lower=1)) at sliceSample.py:196,205.  On return the lower triangle of A[b]
 * (row-major) holds L with L L^T = A; the strict upper triangle is zeroed when zero_upper != 0
 * (as jitchol returns it), else left untouched.  With GPMC_JITTER_PYGPS the caller must pass a
 * workspace from gpmc_workspace_bytes(GPMC_OP_POTRF, ...) (it keeps a copy for the retries).
 */
int gpmc_potrf_batched(double *A_dev, int N, int ld, int B, int *info_dev, int jitter_policy,
                       int zero_upper, void *ws_dev, size_t ws_bytes, void *stream);

/*
 * The metric's unit, "one GP log-lik eval", for B (theta, g) pairs: assemble K+S, Cholesky,
 * forward substitution, quadratic form and log-determinant, never holding more than one N x N
 * matrix per in-flight item.  Replaces sliceSample.py:136-137 + :183-190 + :196 + :147 (and the
 * same at :104-105,:122):
 *   loglik[b] = -( 0.5 * g_b^T (K_b+S_b)^-1 g_b + sum_i log L_ii + 0.5 * N * log(2 pi) )
 * g_dev[B,N]; hyp_dev[B,P]; loglik_dev[B]; info_dev[B].  A failed item (info != 0 after the
 * ladder) gets loglik = NaN, which the sampler treats as a rejected proposal
 * (sliceSample.py:154).  Items are processed in waves sized to the workspace.
 */
int gpmc_loglik_batched(const double *x_dev, int N, int D, const double *g_dev, const double *hyp_dev,
                        int B, int P, int kind, int jitter_policy,
                        double *loglik_dev, int *info_dev,
                        void *ws_dev, size_t ws_bytes, void *stream);

/*
 * The log-lik unit above and its gradient with respect to the hyper-parameters, for B (theta, g) pairs -- what a type-II
 * maximum-likelihood fit of theta (pyGPs 1.3.4 GPR.optimize, the reference's gpK.GPR at framework.py:158,208 and
 * demoRegression.py:110-115) and any gradient-based sampler need.  With A = K(ell, sf) + sn^2 I (the S_ii of
 * sliceSample.py:184-187 is differentiated as the sn^2 it equals):
 *   loglik(theta)       = -(0.5 g^T A^-1 g + 0.5 log|A| + 0.5 N log 2 pi)      (loglik_dev[b], as gpmc_loglik_batched)
 *   d loglik / d th_p   = 0.5 sum_ij (alpha_i alpha_j - W_ij) dA_ij/d th_p,   alpha = A^-1 g,  W = A^-1
 *     dA_ij / d ell     = K_ij r2_ij / ell^3              (GPMC_KIND_SE_ISO, r2 = |x_i - x_j|^2)
 *     dA_ij / d ell_d   = K_ij (x_id - x_jd)^2 / ell_d^3  (GPMC_KIND_SE_ARD)
 *     dA_ij / d ell     = sf2 g_d(t) exp(-t) / ell       (Matern d, t as above; g_1 = t, g_3 = t^2, g_5 = t^2 (1 + t) / 3)
 *     dA_ij / d sf      = 2 K_ij / sf
 *     dA / d sn         = 2 sn I              ->  sn (alpha.alpha - tr W)
 * grad_dev[B,P] is taken with respect to the NATURAL-scale row hyp[b] = (ell.., sf, sn).  An item the jitter ladder
 * rescued gets loglik and gradient of A + jitter I, the jitter held constant.  An item whose info != 0 after the ladder
 * gets loglik = NaN and a row of NaN; so does the gradient of a row with a parameter that is not a positive finite
 * number.  Arguments are checked as in gpmc_loglik_batched; B = 0 returns 0.  Items are processed in waves sized to the
 * workspace (gpmc_workspace_bytes(GPMC_OP_LOGLIK_GRAD, N, D, B)): per item two N x N matrices (the factor with g as its
 * border row, and W), the saved diagonal-block inverses of the factorisation and a few vectors.
 * Pipeline per wave: assemble and factor (jitter ladder), z = L^-1 g and loglik, U = L^-T, alpha = U z, W = U U^T on the
 * lower tiles that can meet K_ij != 0 (the band of tuning keys 14/15; outside it dA/dtheta is an exact zero), then one
 * pass over those tiles that recomputes K_ij and contracts.  Repeated calls are bitwise identical.
 */
int gpmc_loglik_grad_batched(const double *x_dev, int N, int D, const double *g_dev, const double *hyp_dev,
                             int B, int P, int kind, int jitter_policy,
                             double *loglik_dev, double *grad_dev, int *info_dev,
                             void *ws_dev, size_t ws_bytes, void *stream);

/*
 * Same unit with HOST buffers (what a numpy caller holds): pinned staging, H2D of (x, g, hyp),
 * the device path above, D2H of (loglik, info), all on an internal stream; blocking.
 * This is the call bench.py times for `e2e`.
 */
int gpmc_loglik_host(const double *x_host, int N, int D, const double *g_host, const double *hyp_host,
                     int B, int P, int kind, int jitter_policy, double *loglik_host, int *info_host);

/*
 * One surrogate-data slice-sampling transition for B independent chains, shrink loop on the device.
 * Replaces kcMCMC/sliceSample.py:76-163 (surrogate_slice_sampling) including aux_var_model (:165-207),
 * log_gamma (:209-232) and likK.TruncatedGauss2.evaluate (:117-118,142-143), i.e. the body of the caller
 * loops framework.py:68-75 / demoRegression.py:23-30 for many chains at once.
 *   F_dev[B,N], hyp_dev[B,P]   in: current (f, theta) of every chain; out: the accepted (f', theta')
 *   scale_dev[P]               slice widths (:110-112); prior_k_dev / prior_theta_dev[P] (:124-125)
 *   iter                       MCMC iteration: noise frozen and its prior dropped while iter < 500 (:128,133,151)
 *   my, lower, upper           mean(y), 0 - my, 100 - my (:102,114-115)
 *   randomness                 tape_* != NULL: explicit draws in the reference's order -- z[B,N] (:194),
 *                              v[B,P] (:110), u0[B] (:127), U[B,tape_trips,P] (:132), all U(0,1)/N(0,1);
 *                              else Philox4x32-10 keyed by (seed, chain0 + chain index, iter)
 *   max_trips                  bound on the shrink loop (the reference's `while True`); a chain that uses it
 *                              up keeps its state and gets status 1
 *   ntrips_dev[B], loglik_dev[B] (log N(g;0,K+S) at the returned theta), status_dev[B]  may be NULL
 * Chains are processed in waves sized to the workspace (gpmc_sds_workspace_bytes(N, P, chains_per_wave)).
 */
size_t gpmc_sds_workspace_bytes(int N, int P, int chains_per_wave);
int gpmc_sds_sweep(const double *x_dev, const double *y_dev, int N, int D, double *F_dev, double *hyp_dev, int B, int P,
                   int kind, const double *scale_dev, const double *prior_k_dev, const double *prior_theta_dev, int iter,
                   double my, double lower, double upper, unsigned long long seed, unsigned chain0,
                   const double *tape_z, const double *tape_v, const double *tape_u0, const double *tape_U, int tape_trips,
                   int max_trips, int jitter_policy, int *ntrips_dev, double *loglik_dev, int *status_dev,
                   void *ws_dev, size_t ws_bytes, void *stream);

/*
 * The caller loop of framework.py:68-75 / demoRegression.py:23-30 -- `for i in range(iters): propF, propHyp =
 * surrogate_slice_sampling(propF, x, y, propHyp, scale, iter=i)` -- for B chains in ONE call: every chain runs its
 * transitions iter_begin .. iter_begin + n_iters - 1 back to back inside the resident loop of gpmc_sds_sweep, so no chain
 * waits for the slowest one at an iteration boundary (the workspace slots stay full until the call runs out of work).
 * Randomness: Philox keyed by (seed, chain0 + chain, iteration) -- the results are those of n_iters gpmc_sds_sweep calls
 * bit for bit.  F_dev / hyp_dev: state in, final state out.  History (any pointer may be NULL):
 *   hist_hyp_dev[B, n_iters, P], hist_loglik_dev[B, n_iters] (log N(g; 0, K+S) at the sample), hist_trips_dev[B, n_iters],
 *   hist_f_dev[B, n_keep, N]: f after iterations iter_begin + k * thin, k < n_keep;
 *   n_exhausted_dev[1]: transitions that used up max_trips (their chain kept its state for that iteration).
 */
int gpmc_sds_run(const double *x_dev, const double *y_dev, int N, int D, double *F_dev, double *hyp_dev, int B, int P,
                 int kind, const double *scale_dev, const double *prior_k_dev, const double *prior_theta_dev, int iter_begin,
                 int n_iters, double my, double lower, double upper, unsigned long long seed, unsigned chain0, int max_trips,
                 int jitter_policy, double *hist_hyp_dev, double *hist_loglik_dev, int *hist_trips_dev, double *hist_f_dev,
                 int thin, int n_keep, int *n_exhausted_dev, void *ws_dev, size_t ws_bytes, void *stream);

/*
 * Slice sampling of the hyper-parameters of GP regression with a Gaussian likelihood, the latent f integrated out: B
 * independent chains with target  p(theta | y) ~ N(y - m; 0, K_theta + S_theta) * prod_p prior_p(theta_p),  i.e. the
 * log-likelihood unit of gpmc_loglik_batched (y - m as every item's right-hand side) plus the hyper-priors of
 * gpmc_sds_sweep (log_gamma, sliceSample.py:209-232).  Each transition is the reference's hyper-rectangle slice sampler
 * (sliceSample.py:110-163) without f, g and the truncated-Gaussian term:
 *   bracket (:110-112)   v ~ U(0, scale)^P, hyp_min = max(hyp - v, 0), hyp_max = hyp_min + scale
 *   threshold (:127-129) log u0 + prior[sf] + prior[ell..] + G_cur (+ prior[sn] once iter >= burn_in); G_cur is the
 *                        log-likelihood at the chain's current theta, carried from the accepted proposal (evaluated once per
 *                        call, for every chain, in the first round)
 *   shrink loop (:131-163) theta' = hyp_min + (hyp_max - hyp_min) U; while iter < burn_in theta'_sn = hyp_sn and the sn prior
 *                        is left out of both sides (the reference's rule with burn_in = 500; 0 turns it off); G' =
 *                        loglik(theta'); accept if 0 + priors + G' > threshold and finite, else shrink every dimension
 *                        toward hyp.  A factorisation that fails even with the jitter ladder gives G' = NaN: rejected.
 *   x_dev[N,D], y_dev[N], m    data and the constant mean (the reference's mean(y), :102)
 *   hyp_dev[B,P]               state on entry, final state on return (natural scale, as every other entry point)
 *   scale_dev[P], prior_k_dev[P], prior_theta_dev[P]   as gpmc_sds_sweep
 *   iter_begin, n_iters        every chain runs its transitions iter_begin .. iter_begin + n_iters - 1 back to back
 *   randomness                 Philox4x32-10 keyed by (seed, chain0 + chain, iteration) on the streams of gpmc_sds_run (a
 *                              chain draws the v, u0 and U gpmc_sds_run would), or, with all three tapes given,
 *                              tape_v[B, n_iters, P], tape_u0[B, n_iters], tape_U[B, n_iters, tape_trips, P] (U(0,1));
 *                              the trip budget is then min(max_trips, tape_trips)
 *   max_trips                  a transition that uses it up keeps the chain's state and is counted in exhausted_dev[b]
 *   history (any may be NULL)  hist_hyp_dev[B, n_iters, P], hist_loglik_dev[B, n_iters] (G of the sample),
 *                              hist_trips_dev[B, n_iters]; exhausted_dev[B] (may be NULL): transitions that used up the
 *                              budget, or -1 for a chain whose log-likelihood at its starting state is not finite (it keeps
 *                              that state for the whole call, its history repeats it with 0 trips, and it costs nothing)
 * Every chain stays in flight: a round proposes for every chain still inside a transition, evaluates those proposals in
 * one gpmc_loglik_batched-style call (waves, compact band layout and jitter ladder unchanged), accepts or shrinks, and
 * starts the next transition of every chain that finished one.  The host reads the active count once per round, so launch
 * sizes, and the results, repeat bit for bit.  Returns when every chain has finished; gpmc_loglik_layout then reports the
 * layout of the last round.  Workspace: gpmc_workspace_bytes(GPMC_OP_MARGINAL, N, D, B) (the sampler's O(B P) arrays plus
 * the log-likelihood unit's; a smaller one runs the rounds in more waves).  GPMC_EINVAL for an unknown kind, a P that does
 * not fit it, n_iters < 0, iter_begin < 0, burn_in < 0, max_trips <= 0, an unknown jitter policy, a tape that is not all
 * three arrays with tape_trips >= 1 (or none with tape_trips = 0), and missing inputs; B = 0 or n_iters = 0 return 0.
 */
int gpmc_marginal_run(const double *x_dev, int N, int D, const double *y_dev, double m,
                      double *hyp_dev, int B, int P, int kind,
                      const double *scale_dev, const double *prior_k_dev, const double *prior_theta_dev,
                      int iter_begin, int n_iters, int burn_in, unsigned long long seed, unsigned chain0,
                      const double *tape_v, const double *tape_u0, const double *tape_U, int tape_trips,
                      int max_trips, int jitter_policy,
                      double *hist_hyp_dev, double *hist_loglik_dev, int *hist_trips_dev, int *exhausted_dev,
                      void *ws_dev, size_t ws_bytes, void *stream);
/* Rounds of the last gpmc_marginal_run on this process: returns their number; the first `capacity` of them give the
 * chains evaluated in the round (active_out) and its host wall time in ms, which ends in a synchronisation (ms_out).
 * Either pointer may be NULL. */
int gpmc_marginal_rounds(int capacity, int *active_out, double *ms_out);

/*
 * aux_var_model(f, K, sn, g) for one caller-supplied K (sliceSample.py:165-207).  K_dev[N][ld] (ld % 16 == 0, pad
 * columns zero), S_dev[ld] = diag of S (sliceSample.py:184-190; entries beyond N zero), g_dev[ld].  Outputs
 * L_dev = chol(K+S) (:196), m_dev[ld] = R S^-1 g (:204), C_dev = chol(R + 1e-11 I) (:205), both N x ld lower with
 * zeroed strict upper triangle; info_dev[0/1] = dpotrf status of the two factorisations (no jitter retry here: the
 * Python mirror applies kcGP.tools.jitchol semantics by re-calling with jitter).
 */
size_t gpmc_aux_workspace_bytes(int N);
int gpmc_aux_var_model(const double *K_dev, int N, int ld, const double *S_dev, const double *g_dev, double *L_dev,
                       double *m_dev, double *C_dev, int *info_dev, void *ws_dev, size_t ws_bytes, void *stream);

/*
 * Forward substitution L x = b for B right-hand sides rhs_dev[B][ldv] (strideL = 0: one shared L) -- the triangular
 * solves of tools.solve_chol (sliceSample.py:258) and inf_mcmc (:269).  quad_dev (optional) receives
 * log N(b; 0, L L^T) = -(0.5 x.x + sum log L_ii + 0.5 N log 2 pi).
 */
int gpmc_trsv_lower_batched(const double *L_dev, int N, int ld, long long strideL, const double *rhs_dev, int ldv, int B,
                            double *out_dev, double *quad_dev, void *stream);

/*
 * Rectangular cross-covariance K(x, z) for prediction: covK.RBF.getCovMatrix(x=, z=, mode='cross'), sliceSample.py:263.
 * x_dev[N,D], z_dev[M,D], one hyper-parameter row hyp_dev[P]; out_dev[N][ld], ld >= M.
 */
int gpmc_cov_cross(const double *x_dev, int N, const double *z_dev, int M, int D, const double *hyp_dev, int P, int kind,
                   double *out_dev, int ld, void *stream);

/*
 * likK.TruncatedGauss2.evaluate(y=y-my, mu=mu_b) for B latent vectors (sliceSample.py:50,62,118,143; ASSUMPTION-1):
 * out[b] = sum_i log TN(y_i - my; mu_b[i], sn_b, [lower, upper]).  mu_dev[B][ldmu], sn_dev[B].
 */
int gpmc_tg2_loglik(const double *y_dev, double my, const double *mu_dev, int ldmu, int N, int B, const double *sn_dev,
                    double lower, double upper, double *out_dev, void *stream);

/*
 * inf_mcmc (kcMCMC/sliceSample.py:234-284; callers framework.py:223-243, plotResult.py:121) for S stored MCMC samples at
 * once.  Per sample s with hyper-parameters hyp[s] and centred latent vector fm[s] = f_s - m (the mean function is the
 * caller's): factor K/sn^2 + I (:256-257, jitchol), and return
 *     fmu[s][j] = (Ks^T alpha)_j,  alpha = (K + sn^2 I)^-1 fm        (:258,266; the caller adds ms)
 *     fs2[s][j] = kss_j - sum_i V_ij^2,  V = L^-1 (sW o Ks)          (:262-263,269-270; the caller clamps at 0)
 * for the M test inputs xs[M,D].  The 1 + M right-hand sides ride through the factorisation as border rows.
 * info[s] as in gpmc_potrf_batched; a failed sample gets NaN.
 */
size_t gpmc_predict_workspace_bytes(int N, int M, int S);
int gpmc_predict_batched(const double *x_dev, int N, int D, const double *xs_dev, int M, const double *fm_dev,
                         const double *hyp_dev, int S, int P, int kind, int jitter_policy, double *fmu_dev, double *fs2_dev,
                         int *info_dev, void *ws_dev, size_t ws_bytes, void *stream);

/*
 * elliptical_slice (kcMCMC/sliceSample.py:15-74) for B chains: F_dev[B,N] in/out, hyp_dev[B,P] (ell.., sf, sn).
 *   nu ~ N(0, K): tape_nu[B,N] given -> used as is; else nu = chol(K) z with K = covK.RBF(...).getCovMatrix(x) (:38-39),
 *                 z = tape_z[B,N] or Philox (the reference draws through numpy's SVD route, :41: equal in distribution)
 *   tape_u[B]            U(0,1) for the slice level (:51);  tape_theta[B,tape_trips] U(0,1): the initial angle (:54) and
 *                        one redraw per rejected proposal (:74); NULL -> Philox keyed by (seed, chain0 + chain, iter)
 *   ntrips[B] proposals evaluated; status[B]: 0 accepted, 1 max_trips used up (state kept), 2 chol(K) failed even with
 *   jitter (the reference raises LinAlgError); info[B] = status of the factorisation.
 */
size_t gpmc_ess_workspace_bytes(int N, int B);
int gpmc_ess_sweep(const double *x_dev, const double *y_dev, int N, int D, double *F_dev, const double *hyp_dev, int B, int P,
                   int kind, double my, double lower, double upper, unsigned long long seed, unsigned chain0, int iter,
                   const double *tape_nu, const double *tape_z, const double *tape_u, const double *tape_theta, int tape_trips,
                   int max_trips, int jitter_policy, int *ntrips_dev, int *status_dev, int *info_dev,
                   void *ws_dev, size_t ws_bytes, void *stream);

/* Kernel tuning knobs for experiments.
 * (Environment, read once: GPMC_GEMM_CFG=<key 0 value> preselects the tile kernel variant; GPMC_ENVELOPE=0 presets key 14
 *  to 0; GPMC_DEBUG=1 makes the SDS loops print their round counters to stderr.)
 * key 0: DMMA tile kernel variant (0/1/2 cp.async staged, 3 TMA lock-step, 4 TMA free-running = default, 5 = 4 with
 *        persistent CTAs drawing tiles in order from a global counter: measured slower, kept for A/B).
 * key 1: panel factor kernel (0 = the register-resident kernel potf2_reg.cu (default), 3 = the same fragments as a dataflow
 *        program without block barriers, potf2_flow.cu, 2 = the shared-memory kernel potf2_lite.cu -- all three emit the
 *        8x8 diagonal inverses only --, 1 = always the full-inverse kernel potf2.cu).
 * key 2: look-ahead in the blocked Cholesky (panel kernels overlapped with the update GEMM on side streams):
 *        0 auto (on when at most #SMs/2 matrices are in flight), 1 off, 2 on.
 * key 3: window (columns, multiple of 128) of the windowed schedule used for few large matrices; 0 = default.
 * key 4: panel solve kernel: 0 = 8-column sub-blocks, 2 CTAs/SM (default), 1 = 32-column sub-blocks.
 * key 5: 64-row blocks one CTA of the panel solve takes: 0 = auto (1, 2 or 4 by launch size), else forced.
 * key 6: gpmc_sds_sweep loop: 0 = resident loop (slots refilled on the device, host polls a status word without
 *        synchronising; default), 1 = wave loop (one status read per trip, waves drained to their slowest chain).
 * key 7: rounds the resident loop queues ahead of the last status word it has seen (0 = default: 1, every status word is
 *        read before the next round is sized: launch sizes and results independent of host timing; 2..7: deeper, polled).
 * key 8: form of the posterior covariance inside gpmc_sds_sweep / gpmc_sds_run: 0 = reduced, R = S - S (K+S)^-1 S (4/3 N^3
 *        flop per evaluation; default), 1 = literal, V = solve(L, K), R = K - V^T V, m = (R inv(S)) g exactly as
 *        sliceSample.py:197-198,204 write it (8/3 N^3; twice the workspace per chain -- query gpmc_sds_workspace_bytes
 *        after setting it).  Used for parity with the reference, not for speed.
 * key 9: panel factor + panel solve of a block column in ONE launch (one CTA per matrix): 0 = auto (many small matrices in
 *        flight, and every wave of the compact band layout, key 17), 1 = never, 2 = whenever the default panel kernels are
 *        selected.
 * key 10: in-window update of a look-ahead column: 0 = auto (split in a long and a K = 128 short part when a trailing update
 *        runs beside the window or the launches are small; one launch otherwise), 1 = always split, 2 = one launch in every
 *        window that runs alone.
 * key 11: window (columns, multiple of 128) of the triangular inverse U = L^-T: -1 = auto (windows of 512 / 1024 columns when
 *        few matrices are in flight), 0 = none (one long-K product per block column), else forced.
 * key 13: 1 = the resident SDS loop chooses its factorisation schedules from a constant (min(slots, chains)) instead of the
 *        launch sizes: with a run-ahead deeper than 1 (key 7) those follow polled status words, and this keeps results
 *        repeatable bit for bit beyond N = 512 (1-4 % of the sweep time).  0 = default (not needed at run-ahead 1).
 * key 14: envelope skips in gpmc_loglik_batched / gpmc_loglik_host: 1 = on (default): the assembly records, per 64-row block,
 *        the first column that holds a nonzero, and the update GEMM and the panel solve skip the products it shows to be
 *        exact zeros (K of a stationary kernel underflows to 0 far from the diagonal; results are bit-identical); 0 = dense.
 *        Dense-layout waves factored with fused panel launches (key 9) do not record or use it.
 * key 15: band (with key 14 on): 1 = on (default): a bound from bounding boxes of x / ell gives, per 64-row block, the first
 *        64-column tile that can hold a nonzero; only the band right of it is assembled, and the update GEMM and the panel
 *        solve launch only the rows of the widest band of the wave (bit-identical results); 0 = envelope skips only.
 *        GPMC_BAND=0 presets it to 0.
 *        The band is used only with the envelope-aware kernels (key 0 = 4, key 4 = 0); with the others key 15 acts as 0.
 * key 16: where the band's key 15 stores the +0 left of the band, which nothing on the factorisation path reads: 2 = inline
 *        in the assembly (default), 1 = on a low-priority side stream beside the factorisation (measured slower on the
 *        bench workload: the stores compete with the band's assembly), 0 = not at all (the workspace keeps what it held
 *        there; results are unchanged).  GPMC_BAND_CLEAR=<value> presets it.
 * key 17: compact band storage (with key 15 on): 1 = automatic (default): when the dense layout would need several waves,
 *        the band of every item of the call is bounded first and, if rows of W = 128 + 64 * (widest band) columns need
 *        fewer waves that run the plain left-looking schedule, each row keeps only those W columns (nothing left of the
 *        band is written or cleared; results are bit-identical); 0 = always the dense layout.  GPMC_BAND_COMPACT=0
 *        presets it to 0.  One item with a wide band (non-finite input, a huge length-scale) makes the whole call dense. */
int gpmc_set_tuning(int key, int value);

/* Layout the last gpmc_loglik_batched / gpmc_loglik_host call used: *band_W = 0 for the dense layout, else the row width
 * of the compact band layout (key 17); *waves = the number of waves the call's items were factored in.  After
 * gpmc_marginal_run: the layout of its last round. */
int gpmc_loglik_layout(int *band_W, int *waves);

/* FP64 micro-benchmarks used by bench.py to put a measured peak beside the roofline:
 * register-resident DMMA (mma.sync m8n8k4 f64) and DFMA loops over the whole chip. */
int gpmc_bench_fp64_peak(int which /*0 = DMMA, 1 = DFMA*/, int iters, double *tflops_out, double *ms_out);
/* DMMA issue rate with `nacc` (1,2,4,8,16,32) independent accumulators per warp and `warps_per_sm` warps on every SM:
 * the instruction-level parallelism the FP64 tensor pipe needs (DESIGN.md, tile shapes). */
int gpmc_bench_dmma_ilp(int nacc, int warps_per_sm, int iters, double *tflops_out);

/* Timing hooks: the library records CUDA-event durations of its own kernels per class
 * (0 assemble, 1 Cholesky update GEMM, 2 panel potf2, 3 panel trsm, 4 solve+reduce, 5 triangular inverse,
 *  6 posterior-covariance SYRK (and W = U U^T of gpmc_loglik_grad_batched), 7 vector/control kernels, 8 band clear,
 *  9 gradient contraction of gpmc_loglik_grad_batched)
 * when enabled; used by bench.py for roofline.achieved. */
/* Diagnostics of the last gpmc_sds_sweep on this thread: rounds queued, rounds that found nothing to do (queued past the
 * end), times the host-side jitter ladder had to run. */
int gpmc_sds_loop_stats(long long *rounds, long long *idle_rounds, long long *ladders);
int gpmc_profile_enable(int on);
int gpmc_profile_read(int kernel_class, double *total_ms, long long *launches);
int gpmc_profile_reset(void);
/* Debug: every recorded launch of `kernel_class` as (start, end) pairs in ms, measured from the start of the first
 * recorded launch of `origin_class` (launch order; look-ahead streams overlap in time). */
int gpmc_profile_timeline(int kernel_class, int origin_class, double *start_end_ms, long long capacity, long long *written);

#ifdef __cplusplus
}
#endif
#endif /* GPMC_H */
