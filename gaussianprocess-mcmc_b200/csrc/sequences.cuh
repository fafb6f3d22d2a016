// Host-side sequencing of the batched kernels (definitions in sequences.cu).
#pragma once
#include "common.cuh"

#include <functional>

namespace gpmc {

// Left-looking blocked Cholesky of every item of A (lower, in place).  The inverse of diagonal block j is
// written to W + item*strideW + j*w_step (w_step = 0: one scratch block per item, overwritten every step;
// w_step = NB*NB: all blocks kept, as inverse_sequence needs them).
//
// border_rows > 0: the buffer holds that many extra rows below the matrix (rows n .. n+border_rows-1, right-hand sides
// stored as ROWS).  They ride through the update GEMMs and panel solves like any other row below the diagonal, so on
// return row n holds (L^-1 rhs)^T for every column block but the last (the bordered-matrix form of forward
// substitution: chol([[A, g], [g^T, c]]) has (L^-1 g)^T as its last row); border_finish() completes the last block.
// fuse != 0: panel factor and panel solve of every block column in ONE launch (launch_panel_fused); the border rows are
// then COMPLETE on return, the last block column included (pass the same flag to border_finish).  Callers decide once
// per batch with potrf_fuse_auto() and use the same flag for every call on those buffers (retries of subsets included).
// In the compact band layout (A.W > 0) the fused launches leave the border row's last block to border_finish (solved = 0).
// env: envelope of A as launch_cov_assemble wrote it -- the update GEMMs and the panel solves skip the work it shows to
// be zero (bit-identical results); the fused panel launches use it in the compact band layout only.
int potrf_sequence(BatchView A, int n, int B, int *info, double *W, long long strideW, long long w_step,
                   int zero_upper, cudaStream_t s, int border_rows = 0, int fuse = 0, Envelope env = {});
int potrf_fuse_auto(int n, int B, int border_rows);
// potrf_sequence of B matrices of order n would run the plain left-looking schedule with the kernels that know the compact
// band layout (BatchView::W)
bool potrf_compact_ok(int n, int B);
// the fuse flag of potrf_sequence for the compact band layout (1 unless gpmc_set_tuning(9, 1))
int potrf_fuse_compact();

// One wave of assemble-and-factor with the pyGPs jitter ladder (capi.cu); shared by the log-lik unit, the predictive
// path and the elliptical slice sampler's Cholesky draw.
// env: the envelope `fill` writes for the items it assembles (see potrf_sequence)
// w_step: as potrf_sequence's (0: one scratch block per item; NB*NB: every diagonal-block inverse kept, W holds
// (N+NB-1)/NB blocks per item)
int factor_wave(const std::function<int(BatchView, int, const double *)> &fill, const std::function<double(const double *)> &diag_value,
                BatchView A, int N, int nb, const double *hyp_w, int P, int *info_w, double *W, double *jit_dev, int *map_dev,
                int jitter_policy, int border_rows, cudaStream_t s, int fuse = 0, Envelope env = {}, long long w_step = 0);
// the envelope skips are on unless gpmc_set_tuning(14, 0) or GPMC_ENVELOPE=0 forced the dense path
bool envelope_enabled();
// the band (with the envelope) is on unless gpmc_set_tuning(15, 0) or GPMC_BAND=0, and the selected kernels honour it
bool band_enabled();

// Write rhs[item] (length n, row stride ldv) into border row n of every item (zero padded up to ld).
int border_set(BatchView A, int n, const double *rhs, int ldv, int B, cudaStream_t s);
// Finish z = L^-1 rhs in border row n (solve against the last diagonal block) and, when loglik != nullptr,
// loglik = -(0.5 z.z + sum log L_ii + 0.5 n log 2 pi)  (sliceSample.py:122,147); NaN for items with info != 0.
// solved != 0: the factorisation already solved the last block column of the border row (fused panel launches)
int border_finish(BatchView A, int n, double *loglik, const int *info, int B, cudaStream_t s, int solved = 0);
// Copy the border row out: z[item] (row stride ldv) = row n of the item (NaN for items with info != 0).
int border_get(BatchView A, int n, double *z, int ldv, const int *info, int B, cudaStream_t s);

// In place L (lower) -> U = L^-T (upper triangle incl. diagonal blocks; the strict lower block part keeps L).
// Needs the saved diagonal-block inverses of potrf_sequence (w_step = NB*NB).
int inverse_sequence(BatchView A, int n, int B, const double *W, long long strideW, cudaStream_t s);
// pin the batch size the schedules are CHOSEN from (0 = each launch's own): see sequences.cu
void set_schedule_batch(int B);

// R = S - S (U U^T) S + 1e-11 I, lower tiles only, from U (upper, in A) into Rm.  svec = diag(S) per item.
int r_sequence(BatchView Rm, BatchView U, int n, int B, const double *svec, long long stride_s, cudaStream_t s);

// gpmc_workspace_bytes(GPMC_OP_LOGLIK_GRAD, ...) (loglik_grad.cu)
size_t loglik_grad_workspace_bytes(int N, int D, int B);
// the sampler's own arrays inside a gpmc_marginal_run workspace (marginal.cu); the log-likelihood unit gets the rest
size_t marginal_state_bytes(int N, int P, int B);
// gpmc_loglik_batched with the right-hand side of item b at g_dev + b * ldg (ldg = 0: one row shared by every item) (capi.cu)
int loglik_batched(const double *x_dev, int N, int D, const double *g_dev, int ldg, const double *hyp_dev, int B, int P, int kind,
                   int jitter_policy, double *loglik_dev, int *info_dev, void *ws_dev, size_t ws_bytes, cudaStream_t s);

// small helpers
int fill_int(int *p, int v, int n, cudaStream_t s);
int fill_int_mapped(int *p, int v, const int *map, const int *count, int nmax, cudaStream_t s);
int add_diag(BatchView A, int n, const double *jitter, int B, cudaStream_t s);
int diag_stats(BatchView A, int n, double *mean_out, int *nonpos_out, int B, cudaStream_t s);
int add_diag_vec(BatchView A, int n, const double *v, int ldv, int B, cudaStream_t s);
int zero_upper(BatchView A, int n, int B, cudaStream_t s);
int copy_rows(double *dst, int ldd, const double *src, int lds, int n, int rows, cudaStream_t s);

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
inline int ld_for(int n) { return (n + 15) / 16 * 16; }

}  // namespace gpmc
