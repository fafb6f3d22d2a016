// Host-side sequencing of the batched kernels: blocked Cholesky, triangular inverse, posterior covariance.
#include "sequences.cuh"
#include "../../include/gpmc.h"

#include <algorithm>

namespace gpmc {

// ------------------------------------------------------------------------------ small kernels
__global__ void zero_upper_kernel(BatchView A, int n)
{
    const int b = blockIdx.z;
    if (A.count && b >= *A.count) return;
    const int m = batch_item(A, b);
    double *Ab = A.base + (size_t)m * A.stride;
    const int r = blockIdx.y * blockDim.y + threadIdx.y;
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n && c < n && c > r) Ab[(size_t)r * A.ld + c] = 0.0;
}

__global__ void fill_int_kernel(int *p, int v, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}
__global__ void fill_int_mapped_kernel(int *p, int v, const int *map, const int *count)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < *count) p[map[i]] = v;
}

__global__ void add_diag_kernel(BatchView A, int n, const double *jitter)
{
    const int b = blockIdx.y;
    if (A.count && b >= *A.count) return;
    const int m = batch_item(A, b);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) A.base[(size_t)m * A.stride + (size_t)i * A.ld + i] += jitter[m];
}

// mean(diag) and any(diag <= 0) per item -- inputs of the jitchol ladder
__global__ void diag_stats_kernel(BatchView A, int n, double *mean_out, int *nonpos_out)
{
    const int b = blockIdx.x;
    if (A.count && b >= *A.count) return;
    const int m = batch_item(A, b);
    const double *Ab = A.base + (size_t)m * A.stride;
    __shared__ double ssum[256];
    __shared__ int sbad[256];
    double s = 0.0;
    int bad = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double d = Ab[(size_t)i * A.ld + i];
        s += d;
        bad |= (d <= 0.0);
    }
    ssum[threadIdx.x] = s;
    sbad[threadIdx.x] = bad;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) { ssum[threadIdx.x] += ssum[threadIdx.x + o]; sbad[threadIdx.x] |= sbad[threadIdx.x + o]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { mean_out[m] = ssum[0] / n; nonpos_out[m] = sbad[0]; }
}

// U_ii = (L_ii^-1)^T: upper triangular diagonal block with explicit zeros below the diagonal
__global__ void __launch_bounds__(256) write_diag_block_T_kernel(BatchView A, int n, int i0, const double *W, long long strideW)
{
    const int b = blockIdx.x;
    if (A.count && b >= *A.count) return;
    const int m = batch_item(A, b);
    __shared__ double tile[32][33];
    double *Ab = A.base + (size_t)m * A.stride;
    const double *Wb = W + (size_t)m * strideW;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;      // 32 x 8
    for (int br = 0; br < NB; br += 32) {
        for (int bc = 0; bc < NB; bc += 32) {
            // tile of U at (br, bc) = transpose of the tile of W at (bc, br)
            for (int r = ty; r < 32; r += 8) tile[r][tx] = Wb[(bc + r) * NB + br + tx];
            __syncthreads();
            for (int r = ty; r < 32; r += 8) {
                const int gr = i0 + br + r, gc = i0 + bc + tx;
                if (gr < n && gc < n) Ab[(size_t)gr * A.ld + gc] = (bc + tx >= br + r) ? tile[tx][r] : 0.0;
            }
            __syncthreads();
        }
    }
}

// A[i][i] += v[i] (per-item vector); used to form K + S for a caller-supplied K
__global__ void add_diag_vec_kernel(BatchView A, int n, const double *v, int ldv)
{
    const int b = blockIdx.y;
    const int m = batch_item(A, b);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) A.base[(size_t)m * A.stride + (size_t)i * A.ld + i] += v[(size_t)m * ldv + i];
}

__global__ void copy_rows_kernel(double *dst, int ldd, const double *src, int lds, int n)
{
    const int r = blockIdx.y;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        dst[(size_t)r * ldd + i] = src[(size_t)r * lds + i];
}

int fill_int(int *p, int v, int n, cudaStream_t s)
{
    if (n <= 0) return 0;
    fill_int_kernel<<<(n + 255) / 256, 256, 0, s>>>(p, v, n);
    GPMC_LAUNCH_CHECK();
    return 0;
}
int fill_int_mapped(int *p, int v, const int *map, const int *count, int nmax, cudaStream_t s)
{
    if (nmax <= 0) return 0;
    fill_int_mapped_kernel<<<(nmax + 255) / 256, 256, 0, s>>>(p, v, map, count);
    GPMC_LAUNCH_CHECK();
    return 0;
}
int add_diag(BatchView A, int n, const double *jitter, int B, cudaStream_t s)
{
    if (B <= 0) return 0;
    add_diag_kernel<<<dim3((n + 255) / 256, B), 256, 0, s>>>(A, n, jitter);
    GPMC_LAUNCH_CHECK();
    return 0;
}
int diag_stats(BatchView A, int n, double *mean_out, int *nonpos_out, int B, cudaStream_t s)
{
    if (B <= 0) return 0;
    diag_stats_kernel<<<B, 256, 0, s>>>(A, n, mean_out, nonpos_out);
    GPMC_LAUNCH_CHECK();
    return 0;
}
int add_diag_vec(BatchView A, int n, const double *v, int ldv, int B, cudaStream_t s)
{
    if (B <= 0) return 0;
    add_diag_vec_kernel<<<dim3((n + 255) / 256, B), 256, 0, s>>>(A, n, v, ldv);
    GPMC_LAUNCH_CHECK();
    return 0;
}
int zero_upper(BatchView A, int n, int B, cudaStream_t s)
{
    if (B <= 0) return 0;
    dim3 blk(32, 8);
    dim3 grid((n + 31) / 32, (n + 7) / 8, B);
    zero_upper_kernel<<<grid, blk, 0, s>>>(A, n);
    GPMC_LAUNCH_CHECK();
    return 0;
}
int copy_rows(double *dst, int ldd, const double *src, int lds, int n, int rows, cudaStream_t s)
{
    if (rows <= 0) return 0;
    copy_rows_kernel<<<dim3(std::max(1, std::min(8, (n + 255) / 256)), rows), 256, 0, s>>>(dst, ldd, src, lds, n);
    GPMC_LAUNCH_CHECK();
    return 0;
}

// ------------------------------------------------------------------ blocked Cholesky sequencing
// Block columns of NB.  With many matrices per launch the schedule is purely LEFT-LOOKING: update the block column
// with everything to its left (one long-K DMMA GEMM), factor the diagonal block (+ its inverse for
// inverse_sequence), solve the rows below by blocked substitution.  When one launch would not fill the chip (few
// matrices: B * N/128 < 1024, e.g. the single N=16384 matrix of BASELINE config 4) the columns are grouped in WINDOWS:
// left-looking inside a window (contraction limited to the window), then ONE right-looking trailing update
// A22 -= L21 L21^T with thousands of tiles and K = window -- the classic DMMA trailing update.
static int sm_count()
{
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0)
            sms = 148;
    }
    return sms;
}

// The schedules below are chosen from the number of matrices in the launch.  A caller whose launch sizes are only upper
// bounds that move with timing (the resident SDS loop in the tail of a call) pins the number the CHOICE is made from, so that
// the summation order -- and with it every bit of the result -- repeats from run to run.
static int g_schedule_batch = 0;       // 0: choose from the launch's own B
void set_schedule_batch(int B) { g_schedule_batch = B > 0 ? B : 0; }
static int schedule_batch(int B) { return g_schedule_batch > 0 ? g_schedule_batch : B; }

static int g_window_override = 0;
void set_potrf_window(int w) { g_window_override = (w > 0 && w % NB == 0) ? w : 0; }

static int potrf_window_for(int n, int B)
{
    const int nt = (n + 127) / 128;                 // 128-row tiles of a block column
    if (g_window_override) return g_window_override >= n ? 0 : g_window_override;   // experiments: forced (>= n: plain left-looking)
    // plain left-looking once the launches fill the chip several times over -- unless the look-ahead schedule is on anyway
    // (at most #SMs/2 matrices): there windows of 512 measured 3.5 % faster than none at N=2048 x 64 (tools/window_c2.py)
    if ((long long)B * nt >= 1024 && 2 * B > sm_count()) return 0;
    // (N=8192 x 1: 8.58 / 8.65 / 9.00 / 10.4 ms with windows of 256 / 512 / 1024 / 2048 columns; N=16384 x 1 does not care)
    return n >= 12288 ? 1024 : 512;
}

static int g_trsm_mode = 0;
void set_trsm_mode(int mode) { g_trsm_mode = mode; }
bool trsm_honours_envelope() { return g_trsm_mode == 0; }
static int g_potf2_mode = 0;
void set_potf2_mode(int mode) { g_potf2_mode = mode; }
static bool lite_panels() { return g_trsm_mode == 0 && g_potf2_mode != 1; }


// Look-ahead.  With few matrices in flight the panel kernels (one CTA per matrix) leave most of the chip idle, so the
// sequence is spread over up to three streams:
//   * P (high priority): potf2 + panel solve of block column j,
//   * Q: the in-window update of block column j+1, split in a LONG part (contraction over everything left of column j:
//     independent of what P is doing, runs concurrently with it) and a SHORT part (K = the 128 columns P just finished),
//   * G (the caller's stream): the right-looking trailing update after a window, split in the part that touches the
//     NEXT window's columns (everything in that window waits for it) and the rest, which overlaps the next window.
// Dependencies are expressed with events only; the caller's stream joins everything before potrf_sequence returns.
struct LookAhead {
    cudaStream_t panel = nullptr, inwin = nullptr;
    cudaEvent_t ev_q = nullptr, ev_p = nullptr, ev_a = nullptr;
    bool ok = false;
};
static LookAhead *lookahead_ctx()
{
    // streams and events belong to a device: one set per device ordinal
    static LookAhead las[64];
    static bool tried_dev[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    LookAhead &la = las[dev];
    bool &tried = tried_dev[dev];
    if (!tried) {
        tried = true;
        int lo = 0, hi = 0;
        bool ok = cudaDeviceGetStreamPriorityRange(&lo, &hi) == cudaSuccess;
        ok = ok && cudaStreamCreateWithPriority(&la.panel, cudaStreamNonBlocking, hi) == cudaSuccess;
        ok = ok && cudaStreamCreateWithPriority(&la.inwin, cudaStreamNonBlocking, hi) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&la.ev_q, cudaEventDisableTiming) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&la.ev_p, cudaEventDisableTiming) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&la.ev_a, cudaEventDisableTiming) == cudaSuccess;
        la.ok = ok;
    }
    return la.ok ? &la : nullptr;
}
static int g_lookahead_mode = 0;       // 0 auto (B <= #SMs / 2), 1 off, 2 on
void set_lookahead_mode(int mode) { g_lookahead_mode = mode; }

// In-window update of a look-ahead column: split in a long part (runs beside the previous column's panel kernels) and a
// K = 128 short part, or one launch after the previous column's panel solve.  0 auto, 1 always split, 2 never split a
// window that has no trailing update running beside it.
static int g_split_mode = 0;
void set_lookahead_split(int mode) { g_split_mode = mode; }

static int g_panel_fuse = 0;           // 0 auto, 1 never, 2 whenever the default panel kernels are selected
void set_panel_fuse(int mode) { g_panel_fuse = mode; }

// One launch per block column for factor + solve pays when many small matrices are in flight: a CTA then owns a matrix's
// whole block column (35 us of latency-bound factor steps, then 64 rows of solve at a time), and co-resident CTAs drift
// into different phases.  With few or large matrices the solve needs many CTAs per matrix: separate launches.
int potrf_fuse_auto(int n, int B, int border_rows)
{
    B = schedule_batch(B);
    if (!lite_panels() || (g_potf2_mode != 0 && g_potf2_mode != 3) || g_panel_fuse == 1) return 0;
    if (g_panel_fuse == 2) return 1;
    // many small matrices (co-resident CTAs drift into different phases), or any number of very small ones (two launches
    // and the last-block solve of the border row saved per block column: latency of a single small chain)
    if (n + border_rows <= 640) return 1;
    return (B >= 4 * sm_count() && n + border_rows <= 1664) ? 1 : 0;
}

// The compact band layout (BatchView::W) is known to the envelope-aware update tile kernel, the register-resident panel
// factor (alone or fused with the panel solve) and the 8-column panel solve.  The layout is chosen for waves that run the
// plain left-looking schedule; the jitter ladder's retries of a few items may run windows and look-ahead on it (every
// update tile there also starts at the envelope and leaves before touching C when its contraction is empty).
static bool compact_kernels() { return NB == BAND_ROWS && g_trsm_mode == 0 && g_potf2_mode == 0; }
bool potrf_compact_ok(int n, int B)
{
    const int Bs = schedule_batch(B);
    return compact_kernels() && potrf_window_for(n, Bs) == 0 && g_lookahead_mode != 2;
}
// Every block column of a banded matrix has only the band's few rows below its diagonal block, which is what the fused
// panel launches are for: the compact layout fuses them unless gpmc_set_tuning(9, 1) forbids it.
int potrf_fuse_compact() { return g_panel_fuse == 1 ? 0 : 1; }

int potrf_sequence(BatchView A, int n, int B, int *info, double *W, long long strideW, long long w_step,
                   int zero_upper_flag, cudaStream_t s, int border_rows, int fuse, Envelope env)
{
    if (A.W && (border_rows != 1 || w_step || zero_upper_flag || !env.blk || !compact_kernels())) {
        set_error("potrf_sequence: the compact band layout needs the envelope-aware kernels and one border row");
        return GPMC_EINVAL;
    }
    if (fuse && (!lite_panels() || (g_potf2_mode != 0 && g_potf2_mode != 3))) { set_error("potrf_sequence: fused panels need the default panel kernels"); return GPMC_EINVAL; }
    if (border_rows < 0) { set_error("potrf_sequence: border_rows < 0"); return GPMC_EINVAL; }
    const int nr = n + border_rows;                     // rows that take part in the panel solves
    // ONE border row is carried by the idle diagonal warp of the update kernel (border duty); several of them (the
    // right-hand sides of the predictive path) are simply more rows below the matrix for the update GEMM
    const int xrows = border_rows > 1 ? border_rows : 0;
    const int brow = border_rows == 1 ? n : 0;
    // w_step != 0: the caller keeps every diagonal-block inverse for inverse_sequence -> full inverse needed
    // The lite kernel emits the 8x8 diagonal inverses only: enough for trsm_panel8 (not for trsm_panel's 32x32 blocks).
    // Measured: it is the faster of the two at every batch size.  Callers that keep the block inverses (w_step != 0)
    // get them completed by inverse_sequence (launch_inv_blocks8) from those 8x8 blocks.
    const bool lite = lite_panels();
    const int Bs = schedule_batch(B);                   // what the schedule is chosen from (launch sizes keep using B)
    const int window = potrf_window_for(n, Bs);
    const Operand self{A.base, A.stride, A.ld};
    const int wlen = window > 0 ? window : n;
    LookAhead *la = nullptr;
    if (!fuse && n > 2 * NB && (g_lookahead_mode == 2 || (g_lookahead_mode == 0 && 2 * Bs <= sm_count()))) la = lookahead_ctx();
    // streams: trailing updates / in-window updates / panel kernels
    const cudaStream_t sG = s;
    const cudaStream_t sQ = la ? (window > 0 ? la->inwin : s) : s;
    const cudaStream_t sP = la ? la->panel : s;

    auto update = [&](int j0, int width, int k_begin, int k_end, cudaStream_t st) -> int {
        GemmArgs g{};
        g.C = A; g.A = self; g.B = self;
        g.cr0 = j0; g.cc0 = j0; g.rows = n - j0 + xrows; g.cols = width;
        // band: rows more than env.band row blocks below the block column are zero left of it (their tiles would leave at
        // once).  The diagonal tile, which carries the border row, is always launched.  The right-looking trailing updates
        // of the windowed schedule keep their full grids.
        if (env.band >= 0 && xrows == 0) g.rows = std::min(g.rows, NB + env.band * ENV_ROWS);
        g.border_row = brow;
        g.ar0 = j0; g.br0 = j0; g.k0 = k_begin; g.bk0 = k_begin; g.klen = k_end - k_begin;
        g.epi = EPI_SUB;
        g.skip_upper = 1;                               // potf2 reads the lower triangle of the diagonal block only
        g.env = env;
        return launch_gemm(g, B, KC_GEMM, st);
    };

    // several border rows under a SQUARE (lower-only) trailing update: one more, rectangular, launch for those rows
    auto extra_rows_update = [&](int c0, int cols, int k_begin, int klen, cudaStream_t st) -> int {
        if (xrows == 0 || cols <= 0) return 0;
        GemmArgs g{};
        g.C = A; g.A = self; g.B = self;
        g.cr0 = n; g.cc0 = c0; g.rows = xrows; g.cols = cols;
        g.ar0 = n; g.br0 = c0; g.k0 = k_begin; g.bk0 = k_begin; g.klen = klen;
        g.epi = EPI_SUB;
        return launch_gemm(g, B, KC_GEMM, st);
    };

    for (int w0 = 0; w0 < n; w0 += wlen) {
        const int w1 = std::min(n, w0 + wlen);
        if (la && sQ != sG) {                           // this window's columns are final on G up to here
            GPMC_CUDA_CHECK(cudaEventRecord(la->ev_a, sG));
            GPMC_CUDA_CHECK(cudaStreamWaitEvent(sQ, la->ev_a, 0));
            if (w0 > 0 && w1 < n) {
                // the rest of the previous window's trailing update: columns right of this window (overlaps it)
                GemmArgs g{};
                g.C = A; g.A = self; g.B = self;
                g.cr0 = w1; g.cc0 = w1; g.rows = n - w1; g.cols = n - w1;
                g.border_row = brow;
                g.ar0 = w1; g.br0 = w1; g.k0 = w0 - wlen; g.bk0 = w0 - wlen; g.klen = wlen;
                g.lower_only = 1;
                g.epi = EPI_SUB;
                g.skip_upper = 1;
                g.env = env;
                int rc = launch_gemm(g, B, KC_GEMM, sG);
                if (rc) return rc;
                if ((rc = extra_rows_update(w1, n - w1, w0 - wlen, wlen, sG))) return rc;
            }
        }
        // A window with a trailing update running beside it keeps the split (the panel factor kernel is slowed several
        // times by co-resident update CTAs and hides behind the long part).  The first and the last window run alone:
        // when their launches fill the chip several times over anyway, the two K-short launches (23 TFLOP/s at K = 128)
        // cost more than the 35 us of an exposed panel factor kernel (tools/timeline.py).
        const bool paired = w0 > 0 && w1 < n;
        const bool many_ctas = (long long)Bs * ((n - w0 + 127) / 128) * 2 >= 8LL * sm_count();
        const bool split_cols = la && (g_split_mode == 1 || paired || (g_split_mode == 0 && !many_ctas));
        for (int j0 = w0; j0 < w1; j0 += NB) {
            const int width = std::min(NB, n - j0);
            double *Wj = W + (size_t)(j0 / NB) * w_step;
            int rc;
            if (!la) {
                if (j0 > w0 && (rc = update(j0, width, w0, j0, s))) return rc;
            } else if (!split_cols) {
                if (j0 > w0) {
                    GPMC_CUDA_CHECK(cudaStreamWaitEvent(sQ, la->ev_p, 0));                        // column j-1 solved
                    if ((rc = update(j0, width, w0, j0, sQ))) return rc;
                }
                GPMC_CUDA_CHECK(cudaEventRecord(la->ev_q, sQ));
                GPMC_CUDA_CHECK(cudaStreamWaitEvent(sP, la->ev_q, 0));
            } else {
                if (j0 - NB > w0 && (rc = update(j0, width, w0, j0 - NB, sQ))) return rc;         // long part
                if (j0 > w0) {
                    GPMC_CUDA_CHECK(cudaStreamWaitEvent(sQ, la->ev_p, 0));                        // column j-1 solved
                    if ((rc = update(j0, width, j0 - NB, j0, sQ))) return rc;                     // short part
                }
                GPMC_CUDA_CHECK(cudaEventRecord(la->ev_q, sQ));
                GPMC_CUDA_CHECK(cudaStreamWaitEvent(sP, la->ev_q, 0));
            }
            if (fuse) {
                if ((rc = (g_potf2_mode == 3 ? launch_panel_fused_flow(A, n, nr, j0, Wj, strideW, info, zero_upper_flag, B, sP)
                                             : launch_panel_fused(A, n, nr, j0, Wj, strideW, info, zero_upper_flag, B, sP, A.W ? env : Envelope{})))) return rc;
                if (la) GPMC_CUDA_CHECK(cudaEventRecord(la->ev_p, sP));
                continue;
            }
            rc = !lite ? launch_potf2(A, n, j0, Wj, strideW, info, zero_upper_flag, B, sP)
                 : (g_potf2_mode == 2 ? launch_potf2_lite(A, n, j0, Wj, strideW, info, zero_upper_flag, B, sP)
                    : (g_potf2_mode == 3 ? launch_potf2_flow(A, n, j0, Wj, strideW, info, zero_upper_flag, B, sP)
                                         : launch_potf2_reg(A, n, j0, Wj, strideW, info, zero_upper_flag, B, sP)));
            if (rc) return rc;
            if (j0 + NB < n && (rc = (g_trsm_mode == 1 ? launch_trsm_panel(A, nr, j0, Wj, strideW, B, sP)
                                                        : launch_trsm_panel8(A, nr, j0, Wj, strideW, B, sP, -1, -1, env)))) return rc;
            // several border rows: the last block column is solved for them here too (a single border row is finished by
            // border_finish together with the quadratic form)
            if (j0 + NB >= n && xrows > 0 && (rc = launch_trsm_panel8(A, nr, j0, Wj, strideW, B, sP, n, n))) return rc;
            if (la) GPMC_CUDA_CHECK(cudaEventRecord(la->ev_p, sP));
        }
        if (la) GPMC_CUDA_CHECK(cudaStreamWaitEvent(sG, la->ev_p, 0));                            // join
        if (w1 < n) {
            const bool split = la && sQ != sG;
            const int w2 = std::min(n, w1 + wlen);
            GemmArgs g{};
            g.C = A; g.A = self; g.B = self;
            g.cr0 = w1; g.cc0 = w1; g.rows = n - w1 + (split ? xrows : 0); g.cols = split ? w2 - w1 : n - w1;
            g.border_row = brow;
            g.ar0 = w1; g.br0 = w1; g.k0 = w0; g.bk0 = w0; g.klen = w1 - w0;
            g.lower_only = split ? 0 : 1;               // split: the next window's columns first (rectangular, the tiles
            g.epi = EPI_SUB;                            // above the diagonal exit at once), the rest at the top of the loop
            g.skip_upper = 1;
            g.env = env;
            int rc = launch_gemm(g, B, KC_GEMM, sG);
            if (rc) return rc;
            if (!split && (rc = extra_rows_update(w1, n - w1, w0, w1 - w0, sG))) return rc;
        }
    }
    if (zero_upper_flag) return zero_upper(A, n, B, s);
    return 0;
}

// ------------------------------------------------------------------ border row (right-hand side carried as row n)
__global__ void border_set_kernel(BatchView A, int n, const double *__restrict__ rhs, int ldv, int len)
{
    const int b = blockIdx.y;
    if (A.count && b >= *A.count) return;
    const int m = batch_item(A, b);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < len) *view_elem(A, m, n, i) = (i < n) ? rhs[(size_t)m * ldv + i] : 0.0;
}

int border_set(BatchView A, int n, const double *rhs, int ldv, int B, cudaStream_t s)
{
    if (B <= 0) return 0;
    const int len = A.W ? (int)A.border_stride : A.ld;     // the row padded to the dense leading dimension
    prof_begin(KC_VEC, s);
    border_set_kernel<<<dim3((len + 255) / 256, B), 256, 0, s>>>(A, n, rhs, ldv, len);
    prof_end(KC_VEC, s);
    GPMC_LAUNCH_CHECK();
    return 0;
}

__global__ void border_get_kernel(BatchView A, int n, double *__restrict__ z, int ldv, const int *__restrict__ info)
{
    const int b = blockIdx.y;
    if (A.count && b >= *A.count) return;
    const int m = batch_item(A, b);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) z[(size_t)m * ldv + i] = (info && info[m] != 0) ? nan("") : *view_elem(A, m, n, i);
}

int border_get(BatchView A, int n, double *z, int ldv, const int *info, int B, cudaStream_t s)
{
    if (B <= 0) return 0;
    prof_begin(KC_VEC, s);
    border_get_kernel<<<dim3((n + 255) / 256, B), 256, 0, s>>>(A, n, z, ldv, info);
    prof_end(KC_VEC, s);
    GPMC_LAUNCH_CHECK();
    return 0;
}

int border_finish(BatchView A, int n, double *loglik, const int *info, int B, cudaStream_t s, int solved)
{
    if (B <= 0) return 0;
    const long long bstride = view_border_stride(A);
    if (bstride > 0x7fffffffLL) { set_error("border_finish: item stride %lld does not fit the vector stride", bstride); return GPMC_EINVAL; }
    double *row = view_elem(A, 0, n, 0);                // item m's border row = row + m * bstride
    // the fused panel launches solved the border row through the last block column as well
    if (solved) return loglik ? launch_quad_logdet(A, n, row, (int)bstride, loglik, info, B, s) : 0;
    const int j0 = (n - 1) / NB * NB;                   // last block column: its part of the row is updated, not solved
    const int nv = n - j0;
    // the last diagonal block as a dense view (its rows share one row stride in either layout)
    BatchView D{view_elem(A, 0, j0, j0), A.stride, A.ld, A.map, A.count};
    int rc = launch_solve_reduce(D, nv, row + j0, nullptr, (int)bstride, row + j0, nullptr, info, B, s);
    if (rc || !loglik) return rc;
    return launch_quad_logdet(A, n, row, (int)bstride, loglik, info, B, s);
}

// U = L^-T, built block column by block column in the upper triangle of the same buffer:
//   U[0:i0, i] = -(U[0:i0, 0:i0] L[i, 0:i0]^T) (L_ii^-1)^T ,   U[i, i] = (L_ii^-1)^T
// (the k < row part of U is zero, so every tile starts its contraction at its own first row).
// Window of the triangular inverse (0 = none).  The plain sequence computes block column i of U = L^-T as
// Y_i = U[0:i0, 0:i0] L[i, 0:i0]^T (one launch of i0/128 x 2 tiles per matrix, contraction up to i0) and multiplies by
// -W_i^T: with few matrices in flight every one of those launches is a fraction of a wave of long-K tiles (measured: 0.30
// of DGEMM for 2-3 matrices of 8192, profiles/r02r_large_n_sds.json).  Windowed: the strict upper triangle is zeroed and
// serves as the accumulator of Y; inside a window the contraction is limited to the window's own columns, and after a
// window ONE launch adds its contribution to every later block column,  Y[0:w1, w1:n] += U[0:w1, w0:w1] L[w1:n, w0:w1]^T
// -- thousands of tiles with K = window, like the trailing update of the windowed Cholesky.
static int g_inverse_window = -1;      // -1 auto, 0 off, else forced (multiple of 128)
void set_inverse_window(int w) { g_inverse_window = (w >= 0 && w % NB == 0) ? w : -1; }

static int inverse_window_for(int n, int B)
{
    int w = g_inverse_window;
    if (w < 0) {
        const int nt = (n + NB - 1) / NB;
        w = (long long)B * nt >= 1024 ? 0 : (n >= 8192 ? 1024 : 512);
    }
    return (w > 0 && w < n) ? w : 0;
}

static int inverse_sequence_windowed(BatchView A, int n, int B, const double *W, long long strideW, int window, cudaStream_t s)
{
    const Operand self{A.base, A.stride, A.ld};
    int rc = zero_upper(A, n, B, s);                    // Y accumulates in the strict upper triangle
    if (rc) return rc;
    // The product that follows a window is split like the trailing update of the windowed Cholesky: the NEXT window's
    // columns first (its block columns wait for them), the columns beyond on the caller's stream while the next window's
    // chain of small launches runs on the high-priority side stream.  Events only; the caller's stream joins at the end.
    LookAhead *la = lookahead_ctx();
    const cudaStream_t sC = la ? la->panel : s;         // chain: in-window products, panel multiplies, diagonal blocks, near parts
    const cudaStream_t sF = s;                          // far parts
    if (la) {
        GPMC_CUDA_CHECK(cudaEventRecord(la->ev_a, s));
        GPMC_CUDA_CHECK(cudaStreamWaitEvent(sC, la->ev_a, 0));
    }
    bool far_pending = false;
    auto add_product = [&](int rows, int c0, int cols, int k_begin, int k_end, cudaStream_t st) -> int {
        // Y[0:rows, c0:c0+cols] += U[0:rows, k_begin:k_end] L[c0:c0+cols, k_begin:k_end]^T   (U upper triangular: rows below k skip)
        GemmArgs g{};
        g.C = A; g.A = self; g.B = self;
        g.cr0 = 0; g.cc0 = c0; g.rows = rows; g.cols = cols;
        g.ar0 = 0; g.br0 = c0; g.k0 = k_begin; g.bk0 = k_begin; g.klen = k_end - k_begin;
        g.k_follow_row = 1;
        g.epi = EPI_ADD;
        return launch_gemm(g, B, KC_INV, st);
    };
    for (int w0 = 0; w0 < n; w0 += window) {
        const int w1 = std::min(n, w0 + window);
        for (int i0 = w0; i0 < w1; i0 += NB) {
            const int width = std::min(NB, n - i0);
            const double *Wi = W + (size_t)(i0 / NB) * NB * NB;
            if (i0 > 0) {
                if (i0 > w0 && (rc = add_product(i0, i0, width, w0, i0, sC))) return rc;
                // U[0:i0, i] = -(Y W_i^T), in place
                if ((rc = launch_trmm_panel8(A, i0, i0, width, Wi, strideW, B, sC))) return rc;
            }
            prof_begin(KC_INV, sC);
            write_diag_block_T_kernel<<<B, 256, 0, sC>>>(A, n, i0, Wi, strideW);
            prof_end(KC_INV, sC);
            GPMC_LAUNCH_CHECK();
        }
        if (w1 >= n) break;
        const int w2 = std::min(n, w1 + window);
        if (la) GPMC_CUDA_CHECK(cudaEventRecord(la->ev_p, sC));                       // this window's columns of U are final
        if (la && far_pending) GPMC_CUDA_CHECK(cudaStreamWaitEvent(sC, la->ev_q, 0)); // the near part adds on top of the last far part
        if ((rc = add_product(w1, w1, w2 - w1, w0, w1, sC))) return rc;               // near: the next window's columns
        if (w2 < n) {
            if (la) GPMC_CUDA_CHECK(cudaStreamWaitEvent(sF, la->ev_p, 0));
            if ((rc = add_product(w1, w2, n - w2, w0, w1, sF))) return rc;            // far: everything beyond
            if (la) { GPMC_CUDA_CHECK(cudaEventRecord(la->ev_q, sF)); far_pending = true; }
        }
    }
    if (la) {                                           // join
        GPMC_CUDA_CHECK(cudaEventRecord(la->ev_p, sC));
        GPMC_CUDA_CHECK(cudaStreamWaitEvent(s, la->ev_p, 0));
    }
    return 0;
}

int inverse_sequence(BatchView A, int n, int B, const double *W, long long strideW, cudaStream_t s)
{
    const int nt = (n + NB - 1) / NB;
    const Operand self{A.base, A.stride, A.ld};
    if (lite_panels()) {
        // the factorisation left only the 8x8 diagonal inverses in W: complete every W_i = L_ii^-1 in one launch
        int rc = launch_inv_blocks8(A, n, const_cast<double *>(W), strideW, B, s);
        if (rc) return rc;
    }
    if (const int window = inverse_window_for(n, schedule_batch(B))) return inverse_sequence_windowed(A, n, B, W, strideW, window, s);
    for (int i = 0; i < nt; ++i) {
        const int i0 = i * NB;
        const int width = std::min(NB, n - i0);
        const double *Wi = W + (size_t)i * NB * NB;
        if (i > 0) {
            GemmArgs g{};
            g.C = A; g.A = self; g.B = self;
            g.cr0 = 0; g.cc0 = i0; g.rows = i0; g.cols = width;
            g.ar0 = 0; g.br0 = i0; g.k0 = 0; g.bk0 = 0; g.klen = i0;
            g.k_follow_row = 1;
            g.epi = EPI_SET;
            int rc = launch_gemm(g, B, KC_INV, s);
            if (rc) return rc;
            // U[0:i0, i] = -(Y W_i^T), in place (every warp of the panel kernel reads its rows before it writes them)
            rc = launch_trmm_panel8(A, i0, i0, width, Wi, strideW, B, s);
            if (rc) return rc;
        }
        prof_begin(KC_INV, s);
        write_diag_block_T_kernel<<<B, 256, 0, s>>>(A, n, i0, Wi, strideW);
        prof_end(KC_INV, s);
        GPMC_LAUNCH_CHECK();
    }
    return 0;
}

int r_sequence(BatchView Rm, BatchView U, int n, int B, const double *svec, long long stride_s, cudaStream_t s)
{
    GemmArgs g{};
    g.C = Rm; g.A = Operand{U.base, U.stride, U.ld}; g.B = g.A;
    g.cr0 = 0; g.cc0 = 0; g.rows = n; g.cols = n;
    g.ar0 = 0; g.br0 = 0; g.k0 = 0; g.bk0 = 0; g.klen = n;
    g.lower_only = 1; g.k_follow_row = 1;
    g.epi = EPI_R; g.svec = svec; g.stride_s = stride_s;
    g.skip_upper = 1;                                   // only chol(R + 1e-11 I) reads R, and only its lower triangle
    return launch_gemm(g, B, KC_SYRK_R, s);
}

}  // namespace gpmc
