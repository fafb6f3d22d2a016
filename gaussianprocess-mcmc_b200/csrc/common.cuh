// Shared declarations of libgpmc's kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>

namespace gpmc {

#ifndef GPMC_NB
#define GPMC_NB 128
#endif
constexpr int NB = GPMC_NB;        // panel width of the blocked Cholesky (64 or 128)
static_assert(NB == 64 || NB == 128, "panel width must be 64 or 128");
constexpr int MAX_ELL = 8;         // max number of length-scales (ARD input dimension)
constexpr int MAX_BATCH_ITEMS = 32768;   // batch items of one launch ride in grid.y / grid.z (limit 65535)

// kernel classes for the profiling hooks (gpmc_profile_read)
enum KernelClass { KC_ASSEMBLE = 0, KC_GEMM = 1, KC_POTF2 = 2, KC_TRSM = 3, KC_SOLVE = 4, KC_INV = 5, KC_SYRK_R = 6, KC_VEC = 7,
                   KC_CLEAR = 8, KC_GRAD = 9, KC_COUNT = 10 };

void set_error(const char *fmt, ...);
// Every computing entry point of the C ABI takes this (recursive) lock: the library keeps per-process state (side streams,
// staging buffers, tuning switches), so calls from several host threads are SERIALISED rather than racing.
struct ApiLock { ApiLock(); ~ApiLock(); };
#define GPMC_API_LOCK() gpmc::ApiLock _gpmc_api_lock
void prof_begin(int kc, cudaStream_t s);
void prof_end(int kc, cudaStream_t s);

#define GPMC_CUDA_CHECK(expr)                                                                 \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) {                                                              \
            gpmc::set_error("%s failed at %s:%d: %s", #expr, __FILE__, __LINE__,              \
                            cudaGetErrorString(_e));                                          \
            return (int)_e;                                                                   \
        }                                                                                     \
    } while (0)

#define GPMC_LAUNCH_CHECK()                                                                   \
    do {                                                                                      \
        cudaError_t _e = cudaGetLastError();                                                  \
        if (_e != cudaSuccess) {                                                              \
            gpmc::set_error("kernel launch failed at %s:%d: %s", __FILE__, __LINE__,          \
                            cudaGetErrorString(_e));                                          \
            return (int)_e;                                                                   \
        }                                                                                     \
    } while (0)

// Per-device "do this once" latch: function attributes (cudaFuncAttributeMaxDynamicSharedMemorySize) belong to the
// device that was current when they were set, so a process that drives several GPUs must set them once PER DEVICE.
struct DeviceOnce {
    unsigned long long mask[4] = {0, 0, 0, 0};
    bool first()
    {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return true;
        unsigned long long &w = mask[(dev >> 6) & 3];
        const unsigned long long bit = 1ull << (dev & 63);
        if (w & bit) return false;
        w |= bit;
        return true;
    }
};

// ---------------------------------------------------------------------------------------------
// Batched matrix view.  Item b of a launch is matrix `map ? map[b] : b` of the allocation, so a
// compacted list of active chains / failed items can be processed without moving data.
// Compact band layout (W > 0, gpmc_loglik_batched when its band is narrow): row r keeps only the W columns
// band_col0(r, W) .. band_col0(r, W) + W - 1, stored at base + item * stride + r * W.  The shift is constant over each
// 128-row block (the update tile's height and the panel width), so every tile the kernels touch is still a rectangle with
// row stride W, and it ends at the diagonal block.  band_col0 may be negative for the first blocks.  W is a multiple of 16,
// so the 16-column contraction chunks line up with the dense ones.  The border row (row n, the right-hand side carried
// through the factorisation) is dense and lives in its own array.  Nothing outside the band may be read (see Band).
constexpr int BAND_ROWS = 128;
struct BatchView {
    double *base;          // first matrix
    long long stride;      // elements between matrices
    int ld;                // leading dimension (even; multiple of 16 for internal buffers); == W in the compact layout
    const int *map;        // optional indirection (device), may be nullptr
    const int *count;      // optional device-side item count; CTAs with blockIdx.y >= *count exit
    int W = 0;             // 0: dense; > 0: compact band layout of width W
    int n = 0;             // compact layout: order of the matrix; row n is the border row
    double *border = nullptr;        // compact layout: border rows, item m's at border + m * border_stride
    long long border_stride = 0;
};

__device__ __forceinline__ int batch_item(const BatchView &v, int b) { return v.map ? v.map[b] : b; }

__host__ __device__ __forceinline__ int band_col0(int r, int W) { return (r / BAND_ROWS) * BAND_ROWS + BAND_ROWS - W; }

// element (r, c) of item m -- every kernel that may see the compact layout addresses the matrix through this
__host__ __device__ __forceinline__ double *view_elem(const BatchView &v, int m, int r, int c)
{
    if (!v.W) return v.base + (size_t)m * v.stride + (size_t)r * v.ld + c;
    if (r >= v.n) return v.border + (size_t)m * v.border_stride + c;
    return v.base + ((long long)m * v.stride + (long long)r * v.W + (c - band_col0(r, v.W)));
}
// elements between the border rows of consecutive items
__host__ __device__ __forceinline__ long long view_border_stride(const BatchView &v) { return v.W ? v.border_stride : v.stride; }

// ---------------------------------------------------------------------------------------------
// Envelope of an assembled matrix.  blk[item * ld + r] is the smallest column that holds a nonzero in rows
// ENV_ROWS*r .. ENV_ROWS*r+ENV_ROWS-1 of the lower triangle, as the assembly wrote it.  Cholesky keeps the envelope
// (L_ik = 0 exactly for every k left of row i's first nonzero), so a product over k below it adds only zeros and can be
// skipped without changing a bit.  Rows >= n (right-hand sides carried below the matrix) are not covered and count as
// dense; blk == nullptr means dense everywhere.
constexpr int ENV_ROWS = 64;
struct Envelope {
    int *blk = nullptr;
    int ld = 0;            // ints between items
    int n = 0;             // order of the matrix
    int band = -1;         // >= 0: no row block r of any item holds a nonzero left of 64-column tile r - band (so rows more
                           // than `band` blocks below a block column's last tile are zero in it: the update GEMM and the
                           // panel solve launch no CTA for them); -1: unknown
};

// Band of an assembled matrix (gpmc_loglik_batched with the band on).  A conservative bound taken from bounding boxes of
// x / ell gives, per item and 64-row block r, lo[r]: the leftmost 64-column tile that can hold a nonzero.  The assembly
// writes only tiles w[r] .. r of row block r, with
//     w[r] = min(lo[r-1], lo[r], lo[r+1]) rounded down to a multiple of NB / 64.
// Nothing on the factorisation path reads a row left of its w, which is why the stored band may stay unwritten (or be
// cleared off the critical path):
//   * the update GEMM's 128-row A tile (two row blocks) starts at the later envelope of its rows, >= the min of their lo,
//     floor 16; B rows start at their own envelope; its C tile (columns of the block column) is only read by a tile whose
//     contraction is not empty, i.e. when one of its row blocks has a nonzero left of the block column -- so both row
//     blocks have w left of the block column;
//   * the panel factor reads the diagonal NB x NB block (w rounded down to NB / 64 tiles keeps its lower part written);
//   * the panel solve reads a row block's whole NB-wide block column only when the block has a nonzero in it (lo <= the
//     block column's last tile, so the rounded-down w is at or left of its first tile);
//   * the last-block solve, the quadratic form and the log-determinant read the diagonal and the diagonal blocks;
//   * the jitter ladder re-assembles the same band (the bound does not depend on the jitter).
// The compact layout (see BatchView) stores exactly that much: with width = max over items of r - w[r], W >= 128 +
// 64 width puts band_col0 of every 128-row block at or left of 64 w[r] of both its 64-row blocks.
struct Band {
    const int *w = nullptr;  // w[item * ld + r]; nullptr: the whole lower triangle is assembled
    int ld = 0;
    int width = 0;           // max over the wave of r - w[r] (tiles left of the diagonal tile the assembly writes)
    int clear = 0;           // cov_assemble also writes +0 left of w[r] (band clear done inline)
};
__host__ __device__ inline int env_blocks(int n) { return (n + ENV_ROWS - 1) / ENV_ROWS; }

// first column that may hold a nonzero in rows r0 .. r1-1 of item m (0 when any of them is not covered)
__device__ __forceinline__ int env_first_col(const Envelope &e, int m, int r0, int r1)
{
    if (!e.blk || r1 > e.n || r1 <= r0) return 0;
    const int *p = e.blk + (size_t)m * e.ld;
    int k = 0x7fffffff;
    for (int r = r0 / ENV_ROWS; r <= (r1 - 1) / ENV_ROWS; ++r) k = min(k, p[r]);
    return k;
}

// ---------------------------------------------------------------------------------------------
// launchers (definitions in the .cu files)

// cov_assemble.cu
// env.blk != nullptr: also writes the envelope of every assembled item (the items A selects)
// band.w != nullptr: only the tiles of the band (see Band) are written
int launch_cov_assemble(const double *x, int N, int D, const double *hyp, int P, int n_ell, int flags,
                        const double *jitter, BatchView A, int B, cudaStream_t s, Envelope env = {}, Band band = {});
// Band bound of items 0 .. B-1 (hyp rows, as launch_cov_assemble reads them): w[item * ldw + r] (see Band), and
// band_out[0] = max over items and r of r - lo[r], band_out[1] = max of r - w[r] (band_out must start at 0).
// xbox: scratch of 2 * D * env_blocks(N) doubles.
int launch_band_bound(const double *x, int N, int D, const double *hyp, int P, int n_ell, int B, int *w, int ldw,
                      int *band_out, double *xbox, cudaStream_t s);
// +0 into every element of rows 0 .. N-1 of items 0 .. B-1 left of their row block's w (store only, small grid)
int launch_band_clear(BatchView A, int N, Band band, int B, cudaStream_t s);

// grad_contract.cu : the contraction of gpmc_loglik_grad_batched for items 0 .. B-1 (item stride strideW / ldv / ldw):
//   grad[b][p] = 0.5 sum_ij (alpha_i alpha_j - W_ij) dA_ij/dtheta_p  from the lower triangle of W (row stride ldW),
//   K_ij recomputed from x and hyp with cov_assemble's expression.  band_w != nullptr: row block r of item b reads only the
//   64-column tiles from band_w[b * ldw + r] on (left of them K_ij is +0).  partial: scratch of B * env_blocks(N) * P
//   doubles.  Items with info != 0, or a parameter that is not a positive finite number, get a NaN row.
int launch_grad_contract(const double *x, int N, int D, const double *hyp, int P, int n_ell, const double *alpha, int ldv,
                         const double *W, int ldW, long long strideW, const int *band_w, int ldw, const int *info,
                         double *partial, double *grad, int B, cudaStream_t s);

// gemm_dmma.cu :  C[i][j] (op)= sum_k A[i][k] * B[j][k]   ("NT": both operands K-contiguous, row-major)
struct Operand {
    const double *base;    // first matrix
    long long stride;      // elements between matrices of consecutive batch items
    int ld;
};
enum Epilogue {
    EPI_SUB = 0,           // C = C - acc            (Cholesky update)
    EPI_SET = 1,           // C = acc                (panel TRSM via inverse; Y = U L^T)
    EPI_NEGSET = 2,        // C = -acc               (block column of U = L^-T)
    EPI_R = 3,             // C = S - S acc S (+1e-11 on the diagonal), S = diag(svec)   (posterior covariance R)
    EPI_ADD = 4            // C = C + acc            (windowed triangular inverse: Y accumulated window by window)
};
struct GemmArgs {
    BatchView C;           // output matrices; its map/count select the batch items of the launch
    Operand A, B;          // A rows <-> output rows, B rows <-> output cols (indexed by the same mapped item)
    int cr0, cc0;          // output origin (row, col) in C
    int rows, cols;        // output extent
    int ar0, br0;          // operand rows corresponding to cr0 / cc0
    int k0, bk0;           // first contraction column in A / in B
    int klen;              // contraction length (the tail beyond a multiple of 16 must be zero-padded in memory)
    int lower_only;        // enumerate only tiles with tile-row >= tile-col (square output, SYRK use)
    int k_follow_row;      // A (and B) are upper triangular in (row, k): start k at the tile's first A row
    int epi;               // Epilogue
    int skip_upper;        // C's strict upper triangle (global row < global col) is never read by the caller: warps whose
                           // whole sub-tile lies there may skip their contraction and leave C untouched
    int border_row;        // > 0 (EPI_SUB, skip_upper, cr0 == cc0, A == C buffers): global row of a right-hand side carried as a
                           // ROW below the matrix; it receives the same update, C[border_row, cols] -= A[border_row, k] B[cols, k]^T
    const double *svec;    // EPI_R: per-item diagonal of S, [N]
    long long stride_s;
    Envelope env;          // EPI_SUB Cholesky updates with A = B = C: envelope of the matrix (cfg 4 starts each tile's
                           // contraction at it; the other variants ignore it)
};
int launch_gemm(const GemmArgs &a, int B, int kclass, cudaStream_t s);
void set_gemm_config(int cfg);
bool gemm_honours_envelope();      // the selected tile kernel starts its contractions at the envelope (cfg 4)

// potf2.cu : factor the NB x NB diagonal block at (j0, j0) in place, write its inverse to W
int launch_potf2(BatchView A, int n, int j0, double *W, long long strideW, int *info, int zero_upper,
                 int B, cudaStream_t s);
// potf2_lite.cu : same factor, but only the inverses of the sixteen 8x8 diagonal sub-blocks are written to W (all that
// launch_trsm_panel8 reads); 2 CTAs per SM.  Not for callers that go on to inverse_sequence or use launch_trsm_panel.
int launch_potf2_lite(BatchView A, int n, int j0, double *W, long long strideW, int *info, int zero_upper,
                      int B, cudaStream_t s);
// potf2_reg.cu : same contract as launch_potf2_lite; the block lives in registers as DMMA fragments over 8 warps and is
// factored in 16 steps of 8 columns (the default panel factor kernel)
int launch_potf2_reg(BatchView A, int n, int j0, double *W, long long strideW, int *info, int zero_upper,
                     int B, cudaStream_t s);
// potf2_flow.cu : the register-resident panel factor kernel as a dataflow program (flags in shared memory instead of block
// barriers between the 16 steps; measured slower than potf2_reg.cu, kept for A/B: gpmc_set_tuning(1, 3)), and its fused form
int launch_potf2_flow(BatchView A, int n, int j0, double *W, long long strideW, int *info, int zero_upper,
                      int B, cudaStream_t s);
int launch_panel_fused_flow(BatchView A, int n, int n_rows, int j0, double *W, long long strideW, int *info, int zero_upper,
                            int B, cudaStream_t s);
// potf2_reg.cu : panel factor AND panel solve of block column j0 in one launch (n_rows = n + border rows; in the last block
// column the border rows are solved too) -- for many small matrices in flight.  Compact band layout (A.W > 0): one border
// row, env required; only the rows trsm_panel8 would solve for env are solved, and the last block column solves none.
int launch_panel_fused(BatchView A, int n, int n_rows, int j0, double *W, long long strideW, int *info, int zero_upper,
                       int B, cudaStream_t s, Envelope env = {});
void set_lookahead_mode(int mode); // potrf_sequence: 0 auto (few matrices in flight), 1 off, 2 on
void set_potrf_window(int w);      // override the window of the windowed schedule (multiple of NB; 0 = default)
void set_potf2_mode(int mode);     // 0: register-resident kernel (default), 3: the same as a dataflow program (no block barriers),
                                   // 2: the shared-memory lite kernel, 1: always the full-inverse one

// trsm_panel.cu : rows below the factored diagonal block at (j0, j0):  X L11^T = A21  (W = L11^-1 from launch_potf2)
int launch_trsm_panel(BatchView A, int n, int j0, const double *W, long long strideW, int B, cudaStream_t s);
// trsm_panel8.cu : the same solve with 8-column sub-blocks, shuffle-based fragment conversion, 2 CTAs per SM (default)
//   row_start >= 0: solve only rows row_start .. n-1 (border rows of the last block column); n_mat >= 0: order of the matrix
//   (rows / columns of the diagonal block at or beyond it read as identity)
//   env: envelope of A -- a 64-row block whose rows have no nonzero left of j0 + NB is zero and stays so (skipped); with
//   env.band >= 0 and rows below the matrix only the band's row blocks and those rows are launched
int launch_trsm_panel8(BatchView A, int n, int j0, const double *W, long long strideW, int B, cudaStream_t s,
                       int row_start = -1, int n_mat = -1, Envelope env = {});
// trmm_panel8.cu : in place  A[0:rows, c0:c0+width] = -(A[0:rows, c0:c0+128] W^T)  for a lower triangular 128x128 W
//   (the second product of the triangular inverse, inverse_sequence)
int launch_trmm_panel8(BatchView A, int rows, int c0, int width, const double *W, long long strideW, int B, cudaStream_t s);
// W_i = L_ii^-1 for every diagonal block of a factored matrix, from the 8x8 diagonal inverses potf2_lite left in W
//   (W: nt blocks of NB x NB per item, item stride strideW)
int launch_inv_blocks8(BatchView A, int n, double *W, long long strideW, int B, cudaStream_t s);
void set_trsm_mode(int mode);      // 0: trsm_panel8 (default), 1: trsm_panel (32-column sub-blocks)
bool trsm_honours_envelope();      // the selected panel solve skips the row blocks the envelope shows to be zero (mode 0)
void set_trsm_blocks_per_cta(int v);   // 0: auto (1, 2 or 4 by launch size), else forced

// solve_reduce.cu : z = L^-1 (a - b), optional outputs: z, loglik = -(0.5 z.z + sum log L_ii + 0.5 n log 2pi)
//   a, b, zout are per-item vectors with row stride ldv (b, zout, loglik may be nullptr)
int launch_solve_reduce(BatchView L, int n, const double *a, const double *b, int ldv, double *zout,
                        double *loglik, const int *info, int B, cudaStream_t s);
// loglik[m] = -(0.5 z.z + sum_i log L_ii + 0.5 n log 2pi) from a finished z (row stride ldv per item)
int launch_quad_logdet(BatchView L, int n, const double *z, int ldv, double *loglik, const int *info, int B, cudaStream_t s);
// trmv.cu : out = T x (+ add) for a triangular row-major T;  upper=0: lower triangle, upper=1: upper triangle.
//   mode 0: out = T x + add            (f' = C eta + m, sliceSample.py:140)
//   mode 1: out = add - svec * (T x)   (m = g - S (K+S)^-1 g with T = L^-T, x = L^-1 g; sliceSample.py:204)
//   mode 2: out = T x                  (nu = chol(K) z, the draw of elliptical_slice; sliceSample.py:41)
int launch_trmv(BatchView T, int n, int upper, int mode, const double *x, const double *add, const double *svec,
                int ldv, double *out, int B, cudaStream_t s);

// sweep.cu
void set_sds_mode(int mode);       // 0: resident loop (default), 1: wave loop
void set_panel_fuse(int mode);
void set_lookahead_split(int mode);
void set_inverse_window(int w);     // fused panel factor + solve launches: 0 auto (many small matrices), 1 never, 2 whenever possible
void set_sds_literal(int v);       // 1: R = K - V^T V as the reference writes it (parity), 0: reduced form (default)
void set_sds_runahead(int r);      // rounds queued ahead of the last status word seen (0: auto)
void set_sds_pin_schedule(int v);  // 1: factorisation schedules of the resident loop chosen from a constant (bit-reproducible runs)
void sds_loop_stats(long long *rounds, long long *idle_rounds, long long *ladders);

// microbench.cu
int run_fp64_peak(int which, int iters, double *tflops, double *ms);
int run_dmma_ilp(int nacc, int warps_per_sm, int iters, double *tflops);

}  // namespace gpmc
