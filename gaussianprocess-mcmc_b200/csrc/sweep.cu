// gpmc_sds_sweep: one surrogate-data slice-sampling transition (kcMCMC/sliceSample.py:76-163) for B chains,
// with the hyper-parameter shrink loop resident on the device.
//
// Per evaluation of the auxiliary model at theta (aux_var_model, sliceSample.py:165-207, plus the log-marginal
// :122/:147) the device does, for every active chain at once:
//     K+S (lower)            cov_assemble                                  :136-137,183-190
//     L = chol(K+S)          potrf_sequence (+ pyGPs jitter ladder)        :196
//     z = L^-1 g, log N(g)   g rides through potrf_sequence as a border    :147
//                            row; border_finish (last block, quad form)
//     U = L^-T               inverse_sequence
//     m = g - S (U z)        trmv (upper)        == R S^-1 g               :204
//     R = S - S (U U^T) S    r_sequence          == K - V^T V, V = L^-1 K  :197-198   (+1e-11 I, :205)
//     C = chol(R + 1e-11 I)  potrf_sequence (+ ladder)                     :205
// R is formed in its algebraically reduced form: K - K (K+S)^-1 K = S - S (K+S)^-1 S for diagonal S.  It is the
// same matrix with less cancellation (entries of size S instead of differences of entries of size sf^2) and
// 4/3 N^3 flops per proposal instead of 8/3 N^3 (DESIGN.md, "SDS proposal").
#include "common.cuh"
#include "sequences.cuh"
#include "sds.cuh"
#include "../../include/gpmc.h"

#include <algorithm>
#include <vector>
#include <math.h>
#include <stdlib.h>

namespace gpmc {

struct SweepBuffers {
    int n, ld, ldv, P, nt, cap;                  // cap = chains per wave
    long long mat;                               // doubles per slot of buf2 (and of buf1 in the reduced form): n rows + the border row that carries g
    long long mat1;                              // doubles per slot of buf1: (n + 1) rows, or (2n + 1) in the literal form (K rides below g)
    double *buf1, *buf2, *Wsave, *Wtmp;
    double *Fin, *Fout, *g, *svec, *fprop, *z, *m, *eta;          // [cap, ldv]
    double *theta, *hyp_min, *hyp_max, *hyp_in, *hyp_out;         // [cap, P]
    double *G, *log_u0, *threshold, *cur_llk, *curG, *last_prop, *last_llk, *jit, *mean, *loglik_out;   // [cap]
    int *done, *ntrips, *map, *count, *info1, *info2, *bad, *fmap;   // ints
    int *chain_of, *phase, *parked, *resolved, *map_new, *map_act, *iter_of;   // resident loop (sds.cuh)
    int *count_new, *count_act, *status_word, *next_chain;           // (inside the 256-byte block of `count`)
};

// R = K - V^T V (sliceSample.py:197-198) formed as the reference writes it (gpmc_set_tuning(8, 1)) instead of the reduced form
static int g_sds_pin_schedule = 0;     // tuning key 13
void set_sds_pin_schedule(int v) { g_sds_pin_schedule = v ? 1 : 0; }
static int g_sds_literal = 0;
void set_sds_literal(int v) { g_sds_literal = v ? 1 : 0; }

static char *carve(char *&p, size_t bytes) { char *r = p; p += align_up(bytes, 256); return r; }

// Carve the wave's buffers out of `base` (nullptr: only measure).  Returns the number of bytes used, so the size query
// and the real layout can never disagree.
static size_t layout(SweepBuffers &w, char *base, int n, int P, int cap)
{
    char *p = base;
    w.n = n; w.ld = ld_for(n); w.ldv = w.ld; w.P = P; w.nt = (n + NB - 1) / NB; w.cap = cap;
    w.mat = (long long)(n + 1) * w.ld;
    w.mat1 = g_sds_literal ? (long long)(2 * n + 1) * w.ld : w.mat;
    const size_t mat = (size_t)w.mat * 8;
    w.buf1 = (double *)carve(p, (size_t)w.mat1 * 8 * cap);
    w.buf2 = (double *)carve(p, mat * cap);
    w.Wsave = (double *)carve(p, (size_t)w.nt * NB * NB * 8 * cap);
    w.Wtmp = (double *)carve(p, (size_t)NB * NB * 8 * cap);
    double **vecs[] = {&w.Fin, &w.Fout, &w.g, &w.svec, &w.fprop, &w.z, &w.m, &w.eta};
    for (double **v : vecs) *v = (double *)carve(p, (size_t)w.ldv * 8 * cap);
    double **hyps[] = {&w.theta, &w.hyp_min, &w.hyp_max, &w.hyp_in, &w.hyp_out};
    for (double **v : hyps) *v = (double *)carve(p, (size_t)P * 8 * cap);
    double **scal[] = {&w.G, &w.log_u0, &w.threshold, &w.cur_llk, &w.curG, &w.last_prop, &w.last_llk, &w.jit, &w.mean, &w.loglik_out};
    for (double **v : scal) *v = (double *)carve(p, (size_t)8 * cap);
    int **ints[] = {&w.done, &w.ntrips, &w.map, &w.info1, &w.info2, &w.bad, &w.fmap,
                    &w.chain_of, &w.phase, &w.parked, &w.resolved, &w.map_new, &w.map_act, &w.iter_of};
    for (int **v : ints) *v = (int *)carve(p, (size_t)4 * cap);
    w.count = (int *)carve(p, 256);                  // [0] count, [16] ladder scratch count, then the resident loop's words
    w.count_new = w.count + 24; w.count_act = w.count + 25; w.next_chain = w.count + 26; w.status_word = w.count + 32;
    return (size_t)(p - base);
}

static size_t sweep_bytes(int n, int P, int cap)
{
    SweepBuffers w;
    return layout(w, nullptr, n, P, cap) + 256;
}

// S_ii and diag(K+S) on the host (sliceSample.py:185-190 expression order), used only to size the ladder's jitter
static double host_diag_value(const double *h, int P)
{
    const double sf = h[P - 2], sn = h[P - 1];
    const double sf2 = exp(2.0 * log(sf));
    const double kinv = 1.0 / sf2;
    const double v1 = 1.0 / (sn * sn) + kinv;
    double Sii = 1.0 / (v1 - kinv);
    if (Sii < 0.0) Sii = 0.0;
    return sf2 + Sii;
}

static bool debug_on()
{
    static int v = -1;
    if (v < 0) { const char *e = getenv("GPMC_DEBUG"); v = (e && e[0] == '1') ? 1 : 0; }
    return v == 1;
}

struct AuxCtx {
    const double *x; int N, D, P, kind;
    SweepBuffers *w;
    cudaStream_t s;
    int jitter_policy;
};

// Read info[] of the currently active chains and return the wave-local ids that failed.
static int failed_items(const AuxCtx &c, const int *info_dev, const std::vector<int> &active, std::vector<int> &failed,
                        std::vector<int> &info_host)
{
    info_host.resize(c.w->cap);
    GPMC_CUDA_CHECK(cudaMemcpyAsync(info_host.data(), info_dev, c.w->cap * sizeof(int), cudaMemcpyDeviceToHost, c.s));
    GPMC_CUDA_CHECK(cudaStreamSynchronize(c.s));
    failed.clear();
    for (int id : active) if (info_host[id] != 0) failed.push_back(id);
    return 0;
}

// Mark wave-local chains as "jitchol gave up" (the reference raises LinAlgError; here the proposal is rejected).
static int mark_not_pd(const AuxCtx &c, int *info_dev, const std::vector<int> &ids)
{
    if (ids.empty()) return 0;
    std::vector<int> marks(c.w->cap, 0);
    GPMC_CUDA_CHECK(cudaMemcpyAsync(marks.data(), info_dev, c.w->cap * 4, cudaMemcpyDeviceToHost, c.s));
    GPMC_CUDA_CHECK(cudaStreamSynchronize(c.s));
    for (int id : ids) marks[id] = GPMC_INFO_NOT_PD;
    GPMC_CUDA_CHECK(cudaMemcpyAsync(info_dev, marks.data(), c.w->cap * 4, cudaMemcpyHostToDevice, c.s));
    GPMC_CUDA_CHECK(cudaStreamSynchronize(c.s));
    return 0;
}

// ---- literal form of the posterior covariance (sliceSample.py:197-198,204), for parity with the reference as written:
//   V = solve(L, K)          K rides through the factorisation of K+S as n MORE border rows (rows n+1 .. 2n of the slot,
//                            below g): the update GEMMs and panel solves leave X = K L^-T = V^T there -- a backward
//                            stable triangular solve with n right-hand sides on DMMA, no explicit inverse
//   R = K - V^T V            K assembled again into the second buffer, minus X X^T by the DMMA tile kernel (lower tiles)
//   m = (R inv(S)) g         symmetric matrix-vector product from the lower triangle
//   C = chol(R + 1e-11 I)
// 8/3 N^3 flop per evaluation instead of 4/3 N^3; used for parity (gpmc_set_tuning(8, 1)), not for speed.
__global__ void __launch_bounds__(256)
symv_lower_kernel(BatchView R, int n, const double *__restrict__ g, const double *__restrict__ svec, int ldv, double *__restrict__ out)
{
    // out[i] = sum_j Rsym[i][j] * (g[j] / S[j]) for the 32 rows i = k0 .. k0+31; Rsym from the lower triangle of R
    const int b = blockIdx.y;
    if (R.count && b >= *R.count) return;
    const int m = batch_item(R, b);
    const double *Rb = R.base + (size_t)m * R.stride;
    const double *gv = g + (size_t)m * ldv, *sv = svec + (size_t)m * ldv;
    const int k0 = blockIdx.x * 32;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __shared__ double part_col[8][32], part_row[32];
    // strict-upper part, column-wise: entry (i, j), j > i, is R[j][i]; lane = column i, warps stride the rows j
    double acc = 0.0;
    const int i = k0 + lane;
    for (int j = k0 + warp; j < n; j += 8)
        if (i < n && j > i) acc = fma(Rb[(size_t)j * R.ld + i], (1.0 / sv[j]) * gv[j], acc);
    part_col[warp][lane] = acc;
    // lower part incl. the diagonal, row-wise: warp w takes rows k0 + 4w .. k0 + 4w + 3
    for (int rr = 0; rr < 4; ++rr) {
        const int r = k0 + warp * 4 + rr;
        double a = 0.0;
        if (r < n) {
            const double *row = Rb + (size_t)r * R.ld;
            for (int j = lane; j <= r; j += 32) a = fma(row[j], (1.0 / sv[j]) * gv[j], a);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
        if (lane == 0) part_row[warp * 4 + rr] = a;
    }
    __syncthreads();
    if (threadIdx.x < 32 && k0 + threadIdx.x < n) {
        double v = part_row[threadIdx.x];
        for (int w8 = 0; w8 < 8; ++w8) v += part_col[w8][threadIdx.x];
        out[(size_t)m * ldv + k0 + threadIdx.x] = v;
    }
}

__global__ void add_diag_const_kernel(BatchView A, int n, double v)
{
    const int b = blockIdx.y;
    if (A.count && b >= *A.count) return;
    const int m = batch_item(A, b);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) A.base[(size_t)m * A.stride + (size_t)i * A.ld + i] += v;
}

// Assemble K+S (+ jitter) with its border rows into the slots of V1: g below the matrix, and in the literal form K
// itself below g.
static int aux_fill(const AuxCtx &c, BatchView V1, int nitems, const double *jit)
{
    SweepBuffers &w = *c.w;
    int rc;
    if ((rc = launch_cov_assemble(c.x, c.N, c.D, w.theta, c.P, c.kind, GPMC_ASM_ADD_S | GPMC_ASM_LOWER_ONLY, jit, V1, nitems, c.s))) return rc;
    if ((rc = border_set(V1, w.n, w.g, w.ldv, nitems, c.s))) return rc;
    if (g_sds_literal) {
        BatchView Krows{V1.base + (size_t)(w.n + 1) * w.ld, V1.stride, V1.ld, V1.map, V1.count};
        if ((rc = launch_cov_assemble(c.x, c.N, c.D, w.theta, c.P, c.kind, 0, nullptr, Krows, nitems, c.s))) return rc;     // full K, no S
    }
    return 0;
}
static int aux_border_rows(const SweepBuffers &w) { return g_sds_literal ? 1 + w.n : 1; }

// R (+ 1e-11 I) into V2 from the factored slot V1
static int aux_form_R(const AuxCtx &c, BatchView V1, BatchView V2, int nitems, bool with_m)
{
    SweepBuffers &w = *c.w;
    cudaStream_t s = c.s;
    int rc;
    if (!g_sds_literal) {
        // U = L^-T is already in V1;  R = S - S U U^T S + 1e-11 I (:197-198,205)
        return r_sequence(V2, V1, w.n, nitems, w.svec, w.ldv, s);
    }
    // R = K - X X^T with X = K L^-T in rows n+1 .. 2n of V1 (:197-198)
    if ((rc = launch_cov_assemble(c.x, c.N, c.D, w.theta, c.P, c.kind, GPMC_ASM_LOWER_ONLY, nullptr, V2, nitems, s))) return rc;
    GemmArgs g{};
    g.C = V2;
    g.A = Operand{V1.base + (size_t)(w.n + 1) * w.ld, V1.stride, V1.ld};
    g.B = g.A;
    g.cr0 = 0; g.cc0 = 0; g.rows = w.n; g.cols = w.n;
    g.ar0 = 0; g.br0 = 0; g.k0 = 0; g.bk0 = 0; g.klen = w.n;
    g.lower_only = 1;
    g.epi = EPI_SUB;
    g.skip_upper = 1;
    if ((rc = launch_gemm(g, nitems, KC_SYRK_R, s))) return rc;
    if (with_m) {
        // m = (R inv(S)) g (:204), before the 1e-11 goes onto the diagonal
        prof_begin(KC_VEC, s);
        symv_lower_kernel<<<dim3((w.n + 31) / 32, nitems), 256, 0, s>>>(V2, w.n, w.g, w.svec, w.ldv, w.m);
        prof_end(KC_VEC, s);
        GPMC_LAUNCH_CHECK();
    }
    add_diag_const_kernel<<<dim3((w.n + 255) / 256, nitems), 256, 0, s>>>(V2, w.n, 1e-11);      // :205
    GPMC_LAUNCH_CHECK();
    return 0;
}

// From a factored K+S (V1: L in the lower triangle, z in the border row up to its last block) to C = chol(R + 1e-11 I)
// in V2, for the items of the views:
static int aux_downstream(const AuxCtx &c, BatchView V1, BatchView V2, int nitems, int fuse1)
{
    SweepBuffers &w = *c.w;
    cudaStream_t s = c.s;
    const long long strideW = (long long)w.nt * NB * NB;
    int rc;
    if (g_sds_literal) {
        // several border rows: z = L^-1 g is complete in row n (the last block column was solved with the others)
        if ((rc = launch_quad_logdet(V1, w.n, V1.base + (size_t)w.n * w.ld, (int)V1.stride, w.G, w.info1, nitems, s))) return rc;   // :147
        if ((rc = aux_form_R(c, V1, V2, nitems, true))) return rc;
    } else {
        // ---- z = L^-1 g and the log marginal (:147)
        if ((rc = border_finish(V1, w.n, w.G, w.info1, nitems, s, fuse1))) return rc;
        if ((rc = border_get(V1, w.n, w.z, w.ldv, w.info1, nitems, s))) return rc;
        // ---- U = L^-T, m = g - S U z (:204), R = S - S U U^T S + 1e-11 I (:197-198,205)
        if ((rc = inverse_sequence(V1, w.n, nitems, w.Wsave, strideW, s))) return rc;
        if ((rc = launch_trmv(V1, w.n, 1, 1, w.z, w.g, w.svec, w.ldv, w.m, nitems, s))) return rc;
        if ((rc = aux_form_R(c, V1, V2, nitems, true))) return rc;
    }
    // ---- C = chol(R + 1e-11 I) (jitchol, :205)
    if ((rc = fill_int_mapped(w.info2, 0, V1.map, V1.count, nitems, s))) return rc;
    return potrf_sequence(V2, w.n, nitems, w.info2, w.Wtmp, NB * NB, 0, 0, s, 0, potrf_fuse_auto(w.n, nitems, 0));
}

// Evaluate the auxiliary model at w.theta for the chains listed in `active` (w.map/w.count hold the same list).
// The factorisations are run optimistically: chol(K+S), everything that follows from it, and chol(R + 1e-11 I) are
// queued without looking at info[], then BOTH status vectors are read in one host synchronisation; only when a
// factorisation failed (rare) does the pyGPs jitter ladder run, for the failed chains alone.
// The optimistic pass: chol(K+S), everything that follows from it and chol(R + 1e-11 I) for the slots listed in
// w.map / w.count (at most `na` of them), queued without looking at info[] -- no host synchronisation.
static int aux_queue(const AuxCtx &c, int na)
{
    SweepBuffers &w = *c.w;
    cudaStream_t s = c.s;
    if (na <= 0) return 0;
    BatchView A1{w.buf1, w.mat1, w.ld, w.map, w.count};
    BatchView A2{w.buf2, w.mat, w.ld, w.map, w.count};
    const long long strideW = (long long)w.nt * NB * NB;
    int rc;
    // ---- K+S and its Cholesky factor (jitchol, :196); g rides through the factorisation as a border row:
    //      z = L^-1 g comes out of the update GEMMs and panel solves
    if ((rc = fill_int_mapped(w.info1, 0, w.map, w.count, na, s))) return rc;
    if ((rc = aux_fill(c, A1, na, nullptr))) return rc;
    const int fuse1 = potrf_fuse_auto(w.n, na, aux_border_rows(w));
    if ((rc = potrf_sequence(A1, w.n, na, w.info1, w.Wsave, strideW, NB * NB, 0, s, aux_border_rows(w), fuse1))) return rc;
    return aux_downstream(c, A1, A2, na, fuse1);
}

static int aux_eval(const AuxCtx &c, const std::vector<int> &active)
{
    SweepBuffers &w = *c.w;
    cudaStream_t s = c.s;
    const int na = (int)active.size();
    if (na == 0) return 0;
    const long long mat = w.mat, mat1 = w.mat1;
    const long long strideW = (long long)w.nt * NB * NB;
    int rc;
    if ((rc = aux_queue(c, na))) return rc;
    if (c.jitter_policy != GPMC_JITTER_PYGPS) return 0;
    const int fuse1 = potrf_fuse_auto(w.n, na, aux_border_rows(w));      // what aux_queue used: the retries below must leave the
                                                                         // border row in the same state

    // ---- one synchronisation: status of both factorisations
    std::vector<int> info1(w.cap), info2(w.cap);
    GPMC_CUDA_CHECK(cudaMemcpyAsync(info1.data(), w.info1, w.cap * sizeof(int), cudaMemcpyDeviceToHost, s));
    GPMC_CUDA_CHECK(cudaMemcpyAsync(info2.data(), w.info2, w.cap * sizeof(int), cudaMemcpyDeviceToHost, s));
    GPMC_CUDA_CHECK(cudaStreamSynchronize(s));
    std::vector<int> failed1, failed2;
    for (int id : active) {
        if (info1[id] != 0) failed1.push_back(id);
        else if (info2[id] != 0) failed2.push_back(id);
    }
    if (failed1.empty() && failed2.empty()) return 0;
    int *cnt = w.count + 16;             // scratch count next to the main one (same 256-byte slot)

    if (!failed1.empty()) {
        if (debug_on()) fprintf(stderr, "[gpmc] chol(K+S) failed for %zu of %d chains (first: chain %d, info %d): jitter ladder\n",
                                failed1.size(), na, failed1[0], info1[failed1[0]]);
        std::vector<double> th((size_t)w.cap * c.P), jit(w.cap, 0.0);
        GPMC_CUDA_CHECK(cudaMemcpyAsync(th.data(), w.theta, th.size() * 8, cudaMemcpyDeviceToHost, s));
        GPMC_CUDA_CHECK(cudaStreamSynchronize(s));
        std::vector<int> todo, hopeless, recovered;
        for (int id : failed1) {
            const double dv = host_diag_value(&th[(size_t)id * c.P], c.P);
            if (dv <= 0.0) hopeless.push_back(id);              // any(diag <= 0): LinAlgError
            else { jit[id] = dv * 1e-6; todo.push_back(id); }   // (NaN diag lands here and keeps failing)
        }
        for (int attempt = 0; attempt < 5 && !todo.empty(); ++attempt) {
            const int nf = (int)todo.size();
            GPMC_CUDA_CHECK(cudaMemcpyAsync(w.fmap, todo.data(), nf * 4, cudaMemcpyHostToDevice, s));
            GPMC_CUDA_CHECK(cudaMemcpyAsync(cnt, &nf, 4, cudaMemcpyHostToDevice, s));
            GPMC_CUDA_CHECK(cudaMemcpyAsync(w.jit, jit.data(), w.cap * 8, cudaMemcpyHostToDevice, s));
            BatchView F1{w.buf1, mat1, w.ld, w.fmap, cnt};
            if ((rc = fill_int_mapped(w.info1, 0, w.fmap, cnt, nf, s))) return rc;
            if ((rc = aux_fill(c, F1, nf, w.jit))) return rc;
            if ((rc = potrf_sequence(F1, w.n, nf, w.info1, w.Wsave, strideW, NB * NB, 0, s, aux_border_rows(w), fuse1))) return rc;
            std::vector<int> still, tmp;
            if ((rc = failed_items(c, w.info1, todo, still, tmp))) return rc;
            for (int id : todo) if (tmp[id] == 0) recovered.push_back(id);
            for (int id : still) jit[id] *= 10.0;
            todo.swap(still);
        }
        // "not positive definite, even with jitter"
        hopeless.insert(hopeless.end(), todo.begin(), todo.end());
        if ((rc = mark_not_pd(c, w.info1, hopeless))) return rc;
        // the chains the ladder rescued: everything downstream of chol(K+S) again, for them alone
        if (!recovered.empty()) {
            const int nr = (int)recovered.size();
            GPMC_CUDA_CHECK(cudaMemcpyAsync(w.fmap, recovered.data(), nr * 4, cudaMemcpyHostToDevice, s));
            GPMC_CUDA_CHECK(cudaMemcpyAsync(cnt, &nr, 4, cudaMemcpyHostToDevice, s));
            BatchView F1{w.buf1, mat1, w.ld, w.fmap, cnt};
            BatchView F2{w.buf2, mat, w.ld, w.fmap, cnt};
            if ((rc = aux_downstream(c, F1, F2, nr, fuse1))) return rc;
            std::vector<int> bad2, tmp;
            if ((rc = failed_items(c, w.info2, recovered, bad2, tmp))) return rc;
            failed2.insert(failed2.end(), bad2.begin(), bad2.end());
        }
        // chains whose K+S stayed unfactorable carry NaN everywhere (and a nonzero info2 from the optimistic pass): they
        // are rejected proposals, nothing to retry
    }

    if (!failed2.empty()) {
        std::vector<int> todo = failed2;
        if (debug_on()) fprintf(stderr, "[gpmc] chol(R+1e-11 I) failed for %zu of %d chains (first: chain %d): jitter ladder\n",
                                todo.size(), na, todo[0]);
        std::vector<double> jit(w.cap, 0.0), mean(w.cap, 0.0);
        std::vector<int> bad(w.cap, 0);
        bool first = true;
        for (int attempt = 0; attempt < 5 && !todo.empty(); ++attempt) {
            const int nf = (int)todo.size();
            GPMC_CUDA_CHECK(cudaMemcpyAsync(w.fmap, todo.data(), nf * 4, cudaMemcpyHostToDevice, s));
            GPMC_CUDA_CHECK(cudaMemcpyAsync(cnt, &nf, 4, cudaMemcpyHostToDevice, s));
            BatchView F1{w.buf1, mat1, w.ld, w.fmap, cnt};
            BatchView F2{w.buf2, mat, w.ld, w.fmap, cnt};
            if ((rc = aux_form_R(c, F1, F2, nf, false))) return rc;                   // rebuild R + 1e-11 I
            if (first) {
                if ((rc = diag_stats(F2, w.n, w.mean, w.bad, nf, s))) return rc;
                GPMC_CUDA_CHECK(cudaMemcpyAsync(mean.data(), w.mean, w.cap * 8, cudaMemcpyDeviceToHost, s));
                GPMC_CUDA_CHECK(cudaMemcpyAsync(bad.data(), w.bad, w.cap * 4, cudaMemcpyDeviceToHost, s));
                GPMC_CUDA_CHECK(cudaStreamSynchronize(s));
                std::vector<int> keep;
                for (int id : todo) { if (!bad[id]) { jit[id] = mean[id] * 1e-6; keep.push_back(id); } }
                first = false;
                if (keep.size() != todo.size()) { todo.swap(keep); --attempt; continue; }
            }
            GPMC_CUDA_CHECK(cudaMemcpyAsync(w.jit, jit.data(), w.cap * 8, cudaMemcpyHostToDevice, s));
            if ((rc = add_diag(F2, w.n, w.jit, nf, s))) return rc;
            if ((rc = fill_int_mapped(w.info2, 0, w.fmap, cnt, nf, s))) return rc;
            if ((rc = potrf_sequence(F2, w.n, nf, w.info2, w.Wtmp, NB * NB, 0, 0, s))) return rc;
            std::vector<int> still, tmp;
            if ((rc = failed_items(c, w.info2, todo, still, tmp))) return rc;
            for (int id : still) jit[id] *= 10.0;
            todo.swap(still);
        }
        if ((rc = mark_not_pd(c, w.info2, todo))) return rc;
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// The resident loop (default).  The wave loop further down drains every wave to its slowest chain and reads a status
// vector from the device after every trip; here the workspace is a set of SLOTS instead:
//   * a round = [admit] -> begin (new slots) / propose (slots in their shrink loop) -> auxiliary model for every occupied
//     slot -> whitening + threshold (new slots) / f' + accept-or-shrink (the others);
//   * the admit kernel hands the slots of chains that accepted (or ran out of trips) to the next waiting chains of the
//     call, so the number of matrices per launch stays at capacity until the call runs out of chains;
//   * the host never waits for a round: it enqueues rounds ahead and polls, without blocking, a small status word that
//     every round copies into pinned memory (how many slots are occupied, how many chains are still waiting); launches
//     are sized by the last value seen (an upper bound -- the kernels cut at the device-side counts), and rounds that
//     were queued after the last chain finished find empty lists and exit;
//   * a factorisation that fails parks its slot (no decision is taken for it); when the host sees parked slots in the
//     status word it drains the stream and runs the pyGPs jitter ladder for those slots alone (aux_eval), then resumes.
// Results are those of the wave loop bit for bit: randomness and tapes are keyed by the chain, not by the slot or round.
// gpmc_sds_run: where the history of a multi-iteration call goes (all pointers may be nullptr)
struct RunSpec {
    int n_iters = 1;
    double *hist_hyp = nullptr, *hist_loglik = nullptr, *hist_f = nullptr;
    int *hist_trips = nullptr, *n_exhausted = nullptr;
    int thin = 0, n_keep = 0;
};

struct ResidentHost {
    static constexpr int RING = 8;
    int *pinned = nullptr;                      // RING status words
    cudaEvent_t ev[RING] = {};
    bool ok = false;
};
static ResidentHost *resident_host()
{
    static ResidentHost per_dev[64];
    static bool tried[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    ResidentHost &h = per_dev[dev];
    if (!tried[dev]) {
        tried[dev] = true;
        bool ok = cudaHostAlloc((void **)&h.pinned, ResidentHost::RING * SDS_SW_WORDS * sizeof(int), cudaHostAllocPortable) == cudaSuccess;
        for (int i = 0; ok && i < ResidentHost::RING; ++i) ok = cudaEventCreateWithFlags(&h.ev[i], cudaEventDisableTiming) == cudaSuccess;
        h.ok = ok;
    }
    return h.ok ? &h : nullptr;
}

static int g_sds_mode = 0;            // 0: resident loop, 1: wave loop
static int g_sds_runahead = 0;        // rounds the host may queue ahead of the last status it has seen (0: auto)
void set_sds_mode(int mode) { g_sds_mode = mode; }
void set_sds_runahead(int r) { g_sds_runahead = r; }
static long long g_sds_rounds = 0, g_sds_idle_rounds = 0, g_sds_ladders = 0;   // diagnostics of the last call
void sds_loop_stats(long long *rounds, long long *idle_rounds, long long *ladders)
{
    if (rounds) *rounds = g_sds_rounds;
    if (idle_rounds) *idle_rounds = g_sds_idle_rounds;
    if (ladders) *ladders = g_sds_ladders;
}

static int sds_sweep_resident(const double *x_dev, const double *y_dev, int N, int D, double *F_dev, double *hyp_dev, int B, int P,
                              int kind, const double *scale_dev, const double *prior_k_dev, const double *prior_theta_dev, int iter,
                              double my, double lower, double upper, unsigned long long seed, unsigned chain0,
                              const double *tape_z, const double *tape_v, const double *tape_u0, const double *tape_U, int tape_trips,
                              int max_trips, int jitter_policy, int *ntrips_dev, double *loglik_dev, int *status_dev,
                              SweepBuffers &w, cudaStream_t s, const RunSpec *run = nullptr)
{
    ResidentHost *rh = resident_host();
    if (!rh) { set_error("sds_sweep: cannot allocate the pinned status ring"); return GPMC_ENOMEM; }
    const int cap = w.cap;
    // Launch sizes follow the polled status words in the tail of the call, and the factorisation schedules are chosen from
    // them (few matrices left: look-ahead, windows).  With tuning key 13 the choice is made from this constant instead: the
    // summation order, and so every bit of the result, is then independent of the host's timing, at 1-4 % of the sweep
    // (N=4096 x 256: 2.59 -> 2.69 s).  N <= 512 has a single schedule and repeats exactly either way.
    struct SchedulePin {
        explicit SchedulePin(int B) { set_schedule_batch(B); }
        ~SchedulePin() { set_schedule_batch(0); }
    } pin(g_sds_pin_schedule ? std::min(cap, B) : 0);
    AuxCtx ctx{x_dev, N, D, P, kind, &w, s, jitter_policy};
    int rc;
    // every slot free, nothing admitted yet
    GPMC_CUDA_CHECK(cudaMemsetAsync(w.chain_of, 0xFF, (size_t)cap * 4, s));
    GPMC_CUDA_CHECK(cudaMemsetAsync(w.done, 0, (size_t)cap * 4, s));
    GPMC_CUDA_CHECK(cudaMemsetAsync(w.parked, 0, (size_t)cap * 4, s));
    GPMC_CUDA_CHECK(cudaMemsetAsync(w.resolved, 0, (size_t)cap * 4, s));
    GPMC_CUDA_CHECK(cudaMemsetAsync(w.phase, 0, (size_t)cap * 4, s));
    GPMC_CUDA_CHECK(cudaMemsetAsync(w.count, 0, 256, s));
    if (status_dev) GPMC_CUDA_CHECK(cudaMemsetAsync(status_dev, 0, (size_t)B * 4, s));

    SdsState st{};
    st.n = N; st.P = P; st.ldv = w.ldv; st.iter = iter; st.sweep = (unsigned)iter; st.chain0 = chain0; st.seed = seed;
    st.my = my; st.lower = lower; st.upper = upper;
    st.y = y_dev; st.scale = scale_dev; st.prior_k = prior_k_dev; st.prior_theta = prior_theta_dev;
    st.F = w.Fin; st.hyp = w.hyp_in; st.F_out = w.Fout; st.hyp_out = w.hyp_out; st.loglik_out = w.loglik_out;
    st.g = w.g; st.svec = w.svec; st.fprop = w.fprop; st.theta = w.theta; st.hyp_min = w.hyp_min; st.hyp_max = w.hyp_max;
    st.G = w.G; st.log_u0 = w.log_u0; st.threshold = w.threshold; st.cur_llk = w.cur_llk; st.curG = w.curG;
    st.last_proposal = w.last_prop; st.last_llk = w.last_llk;
    st.done = w.done; st.ntrips = w.ntrips; st.map = w.map; st.count = w.count;
    st.tape_z = tape_z; st.tape_v = tape_v; st.tape_u0 = tape_u0; st.tape_U = tape_U; st.tape_trips = tape_trips;
    st.chain_of = w.chain_of; st.phase = w.phase; st.parked = w.parked; st.resolved = w.resolved;
    st.info1 = w.info1; st.info2 = w.info2;
    st.map_new = w.map_new; st.count_new = w.count_new; st.map_act = w.map_act; st.count_act = w.count_act;
    st.status_word = w.status_word; st.next_chain = w.next_chain;
    st.n_chains = B; st.cap = cap; st.max_trips = tape_U ? std::min(max_trips, tape_trips) : max_trips;
    st.F_glob = F_dev; st.F_glob_out = F_dev; st.hyp_glob = hyp_dev; st.hyp_glob_out = hyp_dev;
    st.ntrips_glob = ntrips_dev; st.status_glob = status_dev; st.loglik_glob = loglik_dev;
    st.hyp_stage = w.hyp_in; st.F_stage = w.Fin;
    if (run) {
        // many iterations per call: `iter` is the first one, every slot carries its chain's own iteration
        st.iter_of = w.iter_of; st.n_iters = run->n_iters;
        st.hist_hyp = run->hist_hyp; st.hist_loglik = run->hist_loglik; st.hist_trips = run->hist_trips;
        st.hist_f = run->hist_f; st.thin = run->thin; st.n_keep = run->n_keep; st.n_exhausted = run->n_exhausted;
        if (run->n_exhausted) GPMC_CUDA_CHECK(cudaMemsetAsync(run->n_exhausted, 0, sizeof(int), s));
    }

    const BatchView C2all{w.buf2, w.mat, w.ld, w.map, w.count};
    const BatchView C2new{w.buf2, w.mat, w.ld, w.map_new, w.count_new};
    const BatchView C2act{w.buf2, w.mat, w.ld, w.map_act, w.count_act};
    (void)C2all;

    // what the host knows (stale, but on the safe side): chains admitted so far (only grows), occupied slots
    int known_next = 0, known_count = cap, known_parked = 0;
    bool finished = false;
    long long round = 0, polled = 0;            // rounds queued / status words consumed
    // Run-ahead: ONE round.  The host sizes round r from the status word of round r-1's admission -- a word that is ready
    // early in round r-1, so the host still queues a whole round ahead of the device -- and it reads EVERY word before it
    // sizes the next round (the blocking wait below), so launch sizes, schedules and results do not depend on its timing.
    // Deeper run-ahead (tuning key 7) sizes rounds from older, larger bounds and queues idle rounds past the end of the
    // call: measured 1.4-4 % slower at N=1024 ... 4096 (and no faster anywhere), and no longer repeatable bit for bit.
    int runahead = g_sds_runahead > 0 ? g_sds_runahead : 1;
    runahead = std::min(runahead, ResidentHost::RING - 1);
    g_sds_rounds = g_sds_idle_rounds = g_sds_ladders = 0;

    auto consume = [&](bool block) -> int {
        // read status words of completed rounds, oldest first
        while (polled < round) {
            const int slot = (int)(polled % ResidentHost::RING);
            cudaError_t q = block ? cudaEventSynchronize(rh->ev[slot]) : cudaEventQuery(rh->ev[slot]);
            if (q == cudaErrorNotReady) { (void)cudaGetLastError(); break; }
            if (q != cudaSuccess) { set_error("sds_sweep: status poll failed: %s", cudaGetErrorString(q)); return (int)q; }
            const int *sw = rh->pinned + slot * SDS_SW_WORDS;
            known_next = sw[SDS_SW_NEXT]; known_count = sw[SDS_SW_COUNT]; known_parked = sw[SDS_SW_PARKED];
            if (known_count == 0 && known_parked == 0 && known_next >= B) finished = true;
            if (known_count == 0) ++g_sds_idle_rounds;
            ++polled;
            block = false;                       // at most one blocking wait per call
        }
        return 0;
    };

    while (true) {
        if ((rc = consume(round - polled >= runahead))) return rc;
        if (finished) break;
        if (known_parked > 0) {
            // ---- rare path: a factorisation failed.  Let everything queued finish, then run the auxiliary model WITH the
            // jitter ladder for the parked slots alone and take their pending decision.
            GPMC_CUDA_CHECK(cudaStreamSynchronize(s));
            if ((rc = consume(false))) return rc;
            std::vector<int> parked(cap), phase(cap);
            GPMC_CUDA_CHECK(cudaMemcpyAsync(parked.data(), w.parked, (size_t)cap * 4, cudaMemcpyDeviceToHost, s));
            GPMC_CUDA_CHECK(cudaMemcpyAsync(phase.data(), w.phase, (size_t)cap * 4, cudaMemcpyDeviceToHost, s));
            GPMC_CUDA_CHECK(cudaStreamSynchronize(s));
            std::vector<int> ids, ids_new, ids_act, ones;
            for (int c = 0; c < cap; ++c) if (parked[c]) { ids.push_back(c); (phase[c] == SDS_PHASE_NEW ? ids_new : ids_act).push_back(c); }
            if (!ids.empty()) {
                ++g_sds_ladders;
                const int np = (int)ids.size(), nn = (int)ids_new.size(), nact = (int)ids_act.size();
                GPMC_CUDA_CHECK(cudaMemcpyAsync(w.map, ids.data(), (size_t)np * 4, cudaMemcpyHostToDevice, s));
                GPMC_CUDA_CHECK(cudaMemcpyAsync(w.count, &np, 4, cudaMemcpyHostToDevice, s));
                if ((rc = aux_eval(ctx, ids))) return rc;                     // optimistic pass + ladder, synchronous
                // decisions may be taken now whatever info[] says (a factorisation the ladder could not rescue is a
                // non-finite, i.e. rejected, proposal -- :154)
                std::vector<int> flags(cap, 0);
                for (int c : ids) flags[c] = 1;
                GPMC_CUDA_CHECK(cudaMemcpyAsync(w.resolved, flags.data(), (size_t)cap * 4, cudaMemcpyHostToDevice, s));
                GPMC_CUDA_CHECK(cudaMemsetAsync(w.parked, 0, (size_t)cap * 4, s));
                if (nn) {
                    GPMC_CUDA_CHECK(cudaMemcpyAsync(w.map_new, ids_new.data(), (size_t)nn * 4, cudaMemcpyHostToDevice, s));
                    GPMC_CUDA_CHECK(cudaMemcpyAsync(w.count_new, &nn, 4, cudaMemcpyHostToDevice, s));
                    if ((rc = launch_solve_reduce(C2new, N, w.Fin, w.m, w.ldv, w.eta, nullptr, w.info2, nn, s))) return rc;
                    if ((rc = launch_sds_threshold(st, nn, s))) return rc;
                }
                if (nact) {
                    GPMC_CUDA_CHECK(cudaMemcpyAsync(w.map_act, ids_act.data(), (size_t)nact * 4, cudaMemcpyHostToDevice, s));
                    GPMC_CUDA_CHECK(cudaMemcpyAsync(w.count_act, &nact, 4, cudaMemcpyHostToDevice, s));
                    if ((rc = launch_trmv(C2act, N, 0, 0, w.eta, w.m, nullptr, w.ldv, w.fprop, nact, s))) return rc;
                    if ((rc = launch_sds_accept(st, nact, s))) return rc;
                }
                GPMC_CUDA_CHECK(cudaStreamSynchronize(s));                    // the host vectors above die here
            }
            known_parked = 0;
            known_count = cap;                   // the parked slots are back in the lists
        }
        // ---- one round, sized by what the host knows
        const int nb_all = known_next < B ? std::min(cap, B) : std::min(cap, known_count);
        // new transitions this round: chains that can still be admitted -- or, with many iterations per call, any slot
        const int nb_new = run ? nb_all : std::min(cap, B - known_next);
        const int nb_act = nb_all;
        if ((rc = launch_sds_admit(st, (int)round, s))) return rc;
        {
            const int slot = (int)(round % ResidentHost::RING);
            GPMC_CUDA_CHECK(cudaMemcpyAsync(rh->pinned + slot * SDS_SW_WORDS, w.status_word, SDS_SW_WORDS * sizeof(int), cudaMemcpyDeviceToHost, s));
            GPMC_CUDA_CHECK(cudaEventRecord(rh->ev[slot], s));
        }
        ++round;
        ++g_sds_rounds;
        if (nb_all <= 0) { if ((rc = consume(true))) return rc; continue; }   // nothing can be running: wait for the word
        if (nb_new > 0 && (rc = launch_sds_begin(st, nb_new, s))) return rc;                                       // :102-112,194
        if ((rc = launch_sds_propose(st, nb_act, 0, s))) return rc;                                                 // :132-134
        if ((rc = aux_queue(ctx, nb_all))) return rc;                                                               // :136-139,147
        if (nb_new > 0) {
            if ((rc = launch_solve_reduce(C2new, N, w.Fin, w.m, w.ldv, w.eta, nullptr, w.info2, nb_new, s))) return rc;   // eta, :108
            if ((rc = launch_sds_threshold(st, nb_new, s))) return rc;                                              // :114-129
        }
        if ((rc = launch_trmv(C2act, N, 0, 0, w.eta, w.m, nullptr, w.ldv, w.fprop, nb_act, s))) return rc;          // f' = C eta + m, :140
        if ((rc = launch_sds_accept(st, nb_act, s))) return rc;                                                     // :142-163
    }
    return 0;
}


}  // namespace gpmc

using namespace gpmc;

extern "C" {

// ---------------------------------------------------------------------------------------------------------
// aux_var_model(f, K, sn, g) for ONE caller-supplied covariance matrix (sliceSample.py:165-207): the caller passes K
// and the diagonal of S (sliceSample.py:184-190, O(N) host arithmetic) and g; returns L = chol(K+S) (:196),
// m = R S^-1 g (:204) and C = chol(R + 1e-11 I) (:205), all N x ld row-major lower triangular with zeroed upper part.
size_t gpmc_aux_workspace_bytes(int N)
{
    if (N <= 0) return 0;
    const size_t nt = (N + NB - 1) / NB;
    return align_up((size_t)N * ld_for(N) * 8, 256) + align_up(nt * NB * NB * 8, 256) + align_up((size_t)NB * NB * 8, 256)
           + 2 * align_up((size_t)ld_for(N) * 8, 256) + 1024;
}

int gpmc_aux_var_model(const double *K_dev, int N, int ld, const double *S_dev, const double *g_dev, double *L_dev,
                       double *m_dev, double *C_dev, int *info_dev /*[2]*/, void *ws_dev, size_t ws_bytes, void *stream)
{
    GPMC_API_LOCK();
    cudaStream_t s = (cudaStream_t)stream;
    if (N <= 0 || ld < N || (ld & 15)) { set_error("aux_var_model: need ld %% 16 == 0 and ld >= N (N=%d ld=%d)", N, ld); return GPMC_EALIGN; }
    if (!ws_dev || ws_bytes < gpmc_aux_workspace_bytes(N)) { set_error("aux_var_model: workspace too small"); return GPMC_ENOMEM; }
    const int nt = (N + NB - 1) / NB;
    char *p = (char *)ws_dev;
    double *U = (double *)p; p += align_up((size_t)N * ld * 8, 256);
    double *Wsave = (double *)p; p += align_up((size_t)nt * NB * NB * 8, 256);
    double *Wtmp = (double *)p; p += align_up((size_t)NB * NB * 8, 256);
    double *z = (double *)p; p += align_up((size_t)ld * 8, 256);
    const long long mat = (long long)N * ld;
    int rc;
    if ((rc = fill_int(info_dev, 0, 2, s))) return rc;
    // K + S -> L (in the caller's L buffer), keeping the block inverses
    GPMC_CUDA_CHECK(cudaMemcpyAsync(L_dev, K_dev, (size_t)mat * 8, cudaMemcpyDeviceToDevice, s));
    BatchView Lv{L_dev, mat, ld, nullptr, nullptr};
    if ((rc = add_diag_vec(Lv, N, S_dev, ld, 1, s))) return rc;
    if ((rc = potrf_sequence(Lv, N, 1, info_dev, Wsave, (long long)nt * NB * NB, NB * NB, 0, s))) return rc;
    if ((rc = launch_solve_reduce(Lv, N, g_dev, nullptr, ld, z, nullptr, info_dev, 1, s))) return rc;
    // U = L^-T on a copy (L itself is an output)
    GPMC_CUDA_CHECK(cudaMemcpyAsync(U, L_dev, (size_t)mat * 8, cudaMemcpyDeviceToDevice, s));
    BatchView Uv{U, mat, ld, nullptr, nullptr};
    if ((rc = inverse_sequence(Uv, N, 1, Wsave, (long long)nt * NB * NB, s))) return rc;
    if ((rc = launch_trmv(Uv, N, 1, 1, z, g_dev, S_dev, ld, m_dev, 1, s))) return rc;
    BatchView Cv{C_dev, mat, ld, nullptr, nullptr};
    if ((rc = r_sequence(Cv, Uv, N, 1, S_dev, ld, s))) return rc;
    if ((rc = potrf_sequence(Cv, N, 1, info_dev + 1, Wtmp, NB * NB, 0, 0, s))) return rc;
    if ((rc = zero_upper(Lv, N, 1, s))) return rc;
    if ((rc = zero_upper(Cv, N, 1, s))) return rc;
    return 0;
}

// Forward substitution  L x = b  for B right-hand sides; strideL = 0 shares one L between all of them.
// (the solve inside tools.solve_chol, sliceSample.py:258, and inside inf_mcmc, :269)
int gpmc_trsv_lower_batched(const double *L_dev, int N, int ld, long long strideL, const double *rhs_dev, int ldv, int B,
                            double *out_dev, double *quad_dev, void *stream)
{
    GPMC_API_LOCK();
    if (N <= 0 || B < 0 || ld < N || (ld & 1) || (ldv & 1) || ldv < N) { set_error("trsv: bad shape N=%d ld=%d ldv=%d B=%d", N, ld, ldv, B); return GPMC_EINVAL; }
    BatchView Lv{const_cast<double *>(L_dev), strideL, ld, nullptr, nullptr};
    // quad_dev (optional) receives -(0.5 x.x + sum log L_ii + 0.5 N log 2pi), i.e. log N(b; 0, L L^T)
    return launch_solve_reduce(Lv, N, rhs_dev, nullptr, ldv, out_dev, quad_dev, nullptr, B, (cudaStream_t)stream);
}

int gpmc_sds_run(const double *x_dev, const double *y_dev, int N, int D, double *F_dev, double *hyp_dev, int B, int P,
                 int kind, const double *scale_dev, const double *prior_k_dev, const double *prior_theta_dev, int iter_begin, int n_iters,
                 double my, double lower, double upper, unsigned long long seed, unsigned chain0, int max_trips, int jitter_policy,
                 double *hist_hyp_dev, double *hist_loglik_dev, int *hist_trips_dev, double *hist_f_dev, int thin, int n_keep,
                 int *n_exhausted_dev, void *ws_dev, size_t ws_bytes, void *stream)
{
    GPMC_API_LOCK();
    cudaStream_t s = (cudaStream_t)stream;
    const int n_ell = kind_n_ell(kind, D);
    if (N <= 0 || D <= 0 || B < 0 || P != n_ell + 2 || kind_cf(kind) < 0 || max_trips <= 0 || n_iters < 0 || (hist_f_dev && (thin <= 0 || n_keep <= 0))) {
        set_error("sds_run: bad shape N=%d D=%d B=%d P=%d kind=%d max_trips=%d n_iters=%d thin=%d n_keep=%d", N, D, B, P, kind, max_trips,
                  n_iters, thin, n_keep);
        return GPMC_EINVAL;
    }
    if (B == 0 || n_iters == 0) return 0;
    int cap = std::min(B, MAX_BATCH_ITEMS);
    while (cap > 1 && sweep_bytes(N, P, cap) > ws_bytes) cap = (cap + 1) / 2;
    if (!ws_dev || sweep_bytes(N, P, cap) > ws_bytes) {
        set_error("sds_run: workspace %zu bytes cannot hold one chain (%zu needed)", ws_bytes, sweep_bytes(N, P, 1));
        return GPMC_ENOMEM;
    }
    SweepBuffers w;
    layout(w, (char *)ws_dev, N, P, cap);
    if (w.ld != N) {
        GPMC_CUDA_CHECK(cudaMemset2DAsync(w.buf1 + N, (size_t)w.ld * 8, 0, (size_t)(w.ld - N) * 8, (size_t)(w.mat1 / w.ld) * cap, s));
        GPMC_CUDA_CHECK(cudaMemset2DAsync(w.buf2 + N, (size_t)w.ld * 8, 0, (size_t)(w.ld - N) * 8, (size_t)(N + 1) * cap, s));
    }
    RunSpec run;
    run.n_iters = n_iters; run.hist_hyp = hist_hyp_dev; run.hist_loglik = hist_loglik_dev; run.hist_trips = hist_trips_dev;
    run.hist_f = hist_f_dev; run.thin = thin; run.n_keep = n_keep; run.n_exhausted = n_exhausted_dev;
    return sds_sweep_resident(x_dev, y_dev, N, D, F_dev, hyp_dev, B, P, kind, scale_dev, prior_k_dev, prior_theta_dev, iter_begin,
                              my, lower, upper, seed, chain0, nullptr, nullptr, nullptr, nullptr, 0, max_trips, jitter_policy,
                              nullptr, nullptr, nullptr, w, s, &run);
}

size_t gpmc_sds_workspace_bytes(int N, int P, int chains_per_wave)
{
    GPMC_API_LOCK();
    if (N <= 0 || P < 3 || chains_per_wave <= 0) return 0;
    return sweep_bytes(N, P, chains_per_wave);
}

int gpmc_sds_sweep(const double *x_dev, const double *y_dev, int N, int D, double *F_dev, double *hyp_dev, int B, int P,
                   int kind, const double *scale_dev, const double *prior_k_dev, const double *prior_theta_dev, int iter,
                   double my, double lower, double upper, unsigned long long seed, unsigned chain0,
                   const double *tape_z, const double *tape_v, const double *tape_u0, const double *tape_U, int tape_trips,
                   int max_trips, int jitter_policy, int *ntrips_dev, double *loglik_dev, int *status_dev,
                   void *ws_dev, size_t ws_bytes, void *stream)
{
    GPMC_API_LOCK();
    cudaStream_t s = (cudaStream_t)stream;
    const int n_ell = kind_n_ell(kind, D);
    if (N <= 0 || D <= 0 || B < 0 || P != n_ell + 2 || kind_cf(kind) < 0 || max_trips <= 0) {
        set_error("sds_sweep: bad shape N=%d D=%d B=%d P=%d kind=%d max_trips=%d", N, D, B, P, kind, max_trips);
        return GPMC_EINVAL;
    }
    if (tape_U && tape_trips < 1) { set_error("sds_sweep: tape_U given with tape_trips=%d", tape_trips); return GPMC_EINVAL; }
    if (B == 0) return 0;
    // chains per wave from the workspace
    int cap = std::min(B, MAX_BATCH_ITEMS);            // chains ride in grid.y
    while (cap > 1 && sweep_bytes(N, P, cap) > ws_bytes) cap = (cap + 1) / 2;
    if (!ws_dev || sweep_bytes(N, P, cap) > ws_bytes) {
        set_error("sds_sweep: workspace %zu bytes cannot hold one chain (%zu needed)", ws_bytes, sweep_bytes(N, P, 1));
        return GPMC_ENOMEM;
    }
    SweepBuffers w;
    layout(w, (char *)ws_dev, N, P, cap);
    // pad columns of the matrices must be zero (the DMMA kernels contract over multiples of 16)
    // (every slot has N + 1 rows -- the border row included -- and the slots are contiguous)
    if (w.ld != N) {
        GPMC_CUDA_CHECK(cudaMemset2DAsync(w.buf1 + N, (size_t)w.ld * 8, 0, (size_t)(w.ld - N) * 8, (size_t)(w.mat1 / w.ld) * cap, s));
        GPMC_CUDA_CHECK(cudaMemset2DAsync(w.buf2 + N, (size_t)w.ld * 8, 0, (size_t)(w.ld - N) * 8, (size_t)(N + 1) * cap, s));
    }
    if (g_sds_mode == 0)
        return sds_sweep_resident(x_dev, y_dev, N, D, F_dev, hyp_dev, B, P, kind, scale_dev, prior_k_dev, prior_theta_dev, iter,
                                  my, lower, upper, seed, chain0, tape_z, tape_v, tape_u0, tape_U, tape_trips, max_trips,
                                  jitter_policy, ntrips_dev, loglik_dev, status_dev, w, s);
    // ---- wave loop (gpmc_set_tuning(6, 1)): kept for A/B and as the reference the resident loop is tested against
    AuxCtx ctx{x_dev, N, D, P, kind, &w, s, jitter_policy};
    std::vector<int> active;
    for (int c0 = 0; c0 < B; c0 += cap) {
        const int nb = std::min(cap, B - c0);
        // stage the wave's state into stride-ldv rows
        int rc;
        if ((rc = copy_rows(w.Fin, w.ldv, F_dev + (size_t)c0 * N, N, N, nb, s))) return rc;
        if ((rc = copy_rows(w.Fout, w.ldv, F_dev + (size_t)c0 * N, N, N, nb, s))) return rc;
        GPMC_CUDA_CHECK(cudaMemcpyAsync(w.hyp_in, hyp_dev + (size_t)c0 * P, (size_t)nb * P * 8, cudaMemcpyDeviceToDevice, s));
        GPMC_CUDA_CHECK(cudaMemcpyAsync(w.hyp_out, hyp_dev + (size_t)c0 * P, (size_t)nb * P * 8, cudaMemcpyDeviceToDevice, s));

        SdsState st{};
        st.n = N; st.P = P; st.ldv = w.ldv; st.iter = iter; st.sweep = (unsigned)iter; st.chain0 = chain0 + (unsigned)c0; st.seed = seed;
        st.my = my; st.lower = lower; st.upper = upper;
        st.y = y_dev; st.scale = scale_dev; st.prior_k = prior_k_dev; st.prior_theta = prior_theta_dev;
        st.F = w.Fin; st.hyp = w.hyp_in; st.F_out = w.Fout; st.hyp_out = w.hyp_out; st.loglik_out = w.loglik_out;
        st.g = w.g; st.svec = w.svec; st.fprop = w.fprop; st.theta = w.theta; st.hyp_min = w.hyp_min; st.hyp_max = w.hyp_max;
        st.G = w.G; st.log_u0 = w.log_u0; st.threshold = w.threshold; st.cur_llk = w.cur_llk; st.curG = w.curG;
        st.last_proposal = w.last_prop; st.last_llk = w.last_llk;
        st.done = w.done; st.ntrips = w.ntrips; st.map = w.map; st.count = w.count;
        st.tape_z = tape_z ? tape_z + (size_t)c0 * N : nullptr;
        st.tape_v = tape_v ? tape_v + (size_t)c0 * P : nullptr;
        st.tape_u0 = tape_u0 ? tape_u0 + c0 : nullptr;
        st.tape_U = tape_U ? tape_U + (size_t)c0 * tape_trips * P : nullptr;
        st.tape_trips = tape_trips;

        // ---- current state: g, bracket, aux model at theta, whitening, threshold (:102-129)
        if ((rc = launch_sds_begin(st, nb, s))) return rc;
        active.resize(nb);
        for (int i = 0; i < nb; ++i) active[i] = i;
        if ((rc = aux_eval(ctx, active))) return rc;
        BatchView C2{w.buf2, w.mat, w.ld, w.map, w.count};
        if ((rc = launch_solve_reduce(C2, N, w.Fin, w.m, w.ldv, w.eta, nullptr, w.info2, nb, s))) return rc;     // eta, :108
        if ((rc = launch_sds_threshold(st, nb, s))) return rc;
        GPMC_CUDA_CHECK(cudaMemcpyAsync(w.loglik_out, w.G, (size_t)nb * 8, cudaMemcpyDeviceToDevice, s));

        // ---- shrink loop (:131-163): device decides, host only learns how many chains remain
        const int trips_allowed = tape_U ? std::min(max_trips, tape_trips) : max_trips;
        std::vector<int> done(nb);
        for (int trip = 0; trip < trips_allowed && !active.empty(); ++trip) {
            const int na = (int)active.size();
            if ((rc = launch_sds_propose(st, na, trip, s))) return rc;
            if ((rc = aux_eval(ctx, active))) return rc;
            if ((rc = launch_trmv(C2, N, 0, 0, w.eta, w.m, nullptr, w.ldv, w.fprop, na, s))) return rc;          // f' = C eta + m, :140
            if ((rc = launch_sds_accept(st, na, s))) return rc;
            if ((rc = launch_sds_compact(st, nb, s))) return rc;
            GPMC_CUDA_CHECK(cudaMemcpyAsync(done.data(), w.done, nb * 4, cudaMemcpyDeviceToHost, s));
            GPMC_CUDA_CHECK(cudaStreamSynchronize(s));
            active.clear();
            for (int i = 0; i < nb; ++i) if (!done[i]) active.push_back(i);
        }
        // ---- results of the wave
        if ((rc = copy_rows(F_dev + (size_t)c0 * N, N, w.Fout, w.ldv, N, nb, s))) return rc;
        GPMC_CUDA_CHECK(cudaMemcpyAsync(hyp_dev + (size_t)c0 * P, w.hyp_out, (size_t)nb * P * 8, cudaMemcpyDeviceToDevice, s));
        if (ntrips_dev) GPMC_CUDA_CHECK(cudaMemcpyAsync(ntrips_dev + c0, w.ntrips, nb * 4, cudaMemcpyDeviceToDevice, s));
        if (loglik_dev) GPMC_CUDA_CHECK(cudaMemcpyAsync(loglik_dev + c0, w.loglik_out, nb * 8, cudaMemcpyDeviceToDevice, s));
        if (status_dev) {
            // 0 = accepted; 1 = the trip budget ran out (state unchanged)
            std::vector<int> st_host(nb, 0);
            for (int id : active) st_host[id] = 1;
            GPMC_CUDA_CHECK(cudaMemcpyAsync(status_dev + c0, st_host.data(), nb * 4, cudaMemcpyHostToDevice, s));
            GPMC_CUDA_CHECK(cudaStreamSynchronize(s));
        }
    }
    return 0;
}

}  // extern "C"
