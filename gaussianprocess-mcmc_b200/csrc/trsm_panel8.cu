// Panel triangular solve, second form:  X L11^T = A21  with 8-column sub-blocks (trsm_panel.cu works on 32).
//
// Same numerics as trsm_panel.cu -- per sub-block an inverse-multiply plus ONE step of iterative refinement against the
// diagonal block itself,  X0 = A W8^T,  r = A - X0 L8^T,  X = X0 + r W8^T  (W8 = the 8x8 diagonal block of L11^-1, which
// is the inverse of the 8x8 diagonal block of L11) -- but with the three small products done on 8x8 blocks the
// triangular waste of the 32-wide products is gone: 336 DMMAs per 8 rows x 128 columns instead of 432, and the part
// that remains is the plain update  acc[:, later] -= X_b L[later, b]^T.
//
// A warp owns 8 rows x 128 columns as DMMA accumulator fragments.  The contraction index of an m8n8k4 DMMA may be
// permuted freely as long as both operands agree, and an 8-wide block is exactly two k-steps of four lanes: with
// step 0 taking k = 2 fk and step 1 taking k = 2 fk + 1, the two doubles a lane holds of an ACCUMULATOR fragment (row fr,
// columns 2 fk and 2 fk + 1) ARE its A-operand fragments for the next product.  So the chain  X0 -> r -> X -> update  needs
// no layout change at all (no shuffles, no shared-memory round trip), and the matching B fragments (W8[c][2fk], W8[c][2fk+1])
// are adjacent in memory: one 16-byte load per pair of DMMAs.  Finished columns go to global memory straight from the
// accumulator registers, so the CTA needs shared memory only for L11 and the sixteen W8 blocks (108 KB): TWO CTAs of
// 64 rows share an SM and one CTA's prologue (loading L11) hides behind the other's DMMA stream.
//
// History (3 bench steps, N=4096 x 1024 chains): trsm_panel.cu (32-column sub-blocks, layout changes through shared
// memory) 221 ms; 8-column sub-blocks with shuffle-based layout changes 184 ms (shared-memory-pipe bound: one 8-byte
// B-fragment load per DMMA plus 504 shuffles per warp); two 8-row fragments per warp 210 ms (too few warps).
#include "common.cuh"
#include "../../include/gpmc.h"

namespace gpmc {

constexpr int T8_ROWS = 64;                   // rows per CTA (8 warps x 8 rows)
constexpr int T8_WARPS = T8_ROWS / 8 + 1;     // + one warp for a border row that follows a full last CTA
constexpr int T8_THREADS = T8_WARPS * 32;
constexpr int T8_B = 40;                      // row stride of a 32x32 L block (8 mod 16: conflict-free 16-byte fragment loads)
constexpr int T8_LBLK = 32 * T8_B;
constexpr int T8_NSB = NB / 32;
constexpr int T8_NLB = T8_NSB * (T8_NSB + 1) / 2;
constexpr int T8_NB8 = NB / 8;                // 8-column sub-blocks
constexpr int T8_WS = 8;                      // row stride of an 8x8 W block (dense: conflict-free 16-byte fragment loads)
constexpr int T8_SMEM = (T8_NLB * T8_LBLK + T8_NB8 * 8 * T8_WS) * (int)sizeof(double);

__device__ __forceinline__ int lblk8_index(int bi, int bj) { return bi * (bi + 1) / 2 + bj; }     // bi >= bj

__device__ __forceinline__ void dmma884_8(double &c0, double &c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

__global__ void __launch_bounds__(T8_THREADS, 2)
trsm_panel8_kernel(BatchView A, int n_rows, int j0, const double *__restrict__ W, long long strideW, int nblk, int row_start, int n_mat,
                   Envelope env, int nband)
{
    extern __shared__ __align__(16) double sm[];
    double *Lb = sm;                              // 10 lower 32x32 blocks of L11
    double *W8 = sm + T8_NLB * T8_LBLK;           // 16 diagonal 8x8 blocks of L11^-1, [blk][8][T8_WS]
    const int b = blockIdx.y;
    if (A.count && b >= *A.count) return;
    const int m = batch_item(A, b);
    // nband >= 0: the launch takes row blocks 0 .. nband-1 (the band) and then the last row block for its border rows only
    // (its matrix rows lie below the band: zero in this block column, and not necessarily written)
    const int nlaunch = nband >= 0 ? nband + 1 : nblk;
    auto blk_of = [&](int i) { return (nband >= 0 && i == nband) ? nblk - 1 : i; };
    // the last row block solves its matrix rows only when the envelope shows a nonzero in them: zero rows stay zero, and
    // left of a band they may not have been written (a failed factorisation would otherwise leave NaN there for good)
    auto border_only = [&](int rb) {
        if (rb != nblk - 1) return false;
        const int row0 = row_start + rb * T8_ROWS;
        return nband >= 0 || (env.blk && row0 < env.n && env_first_col(env, m, row0, env.n) >= j0 + NB);
    };
    // a row block with no nonzero left of column j0 + NB is zero in this block column, and so is its solution: skip it,
    // and leave at once when that holds for every row block of this CTA (border rows are never skipped)
    auto empty_block = [&](int rb) {
        const int row0 = row_start + rb * T8_ROWS;
        const int rows_valid = (rb == nblk - 1) ? min(T8_ROWS + 8, n_rows - row0) : T8_ROWS;
        return env_first_col(env, m, row0, row0 + rows_valid) >= j0 + NB;
    };
    if (env.blk) {
        bool any = false;
        for (int i = blockIdx.x; i < nlaunch && !any; i += gridDim.x) any = !empty_block(blk_of(i));
        if (!any) return;
    }
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int fr = lane >> 2, fk = lane & 3;
    const int ncv = min(NB, n_mat - j0);          // columns of this block column that exist (ragged last block: < NB)
    const double *L11 = view_elem(A, m, j0, j0);  // the diagonal block: one 128-row block, row stride A.ld in either layout

    for (int e = tid; e < T8_NLB * 32 * 16; e += T8_THREADS) {        // 16 16-byte pieces per block row
        const int blk = e / (32 * 16), rem = e - blk * 32 * 16;
        const int r = rem / 16, c2 = (rem - r * 16) * 2;
        int bi = 0;
        while ((bi + 1) * (bi + 2) / 2 <= blk) ++bi;
        const int bj = blk - bi * (bi + 1) / 2;
        double *dstp = &Lb[blk * T8_LBLK + r * T8_B + c2];
        const int gr = j0 + bi * 32 + r, gc = j0 + bj * 32 + c2;
        if (gr < n_mat && gc < n_mat) {
            const unsigned dst = (unsigned)__cvta_generic_to_shared(dstp);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst), "l"(L11 + (size_t)(gr - j0) * A.ld + (gc - j0)));
        } else {                                  // beyond the matrix (ragged last block solved for border rows): identity
            dstp[0] = (gr == gc) ? 1.0 : 0.0;
            dstp[1] = (gr == gc + 1) ? 1.0 : 0.0;
        }
    }
    const double *Wb = W + (size_t)m * strideW;
    for (int e = tid; e < T8_NB8 * 8 * 4; e += T8_THREADS) {          // 4 pieces per row of an 8x8 block
        const int blk = e >> 5, r = (e >> 2) & 7, c2 = (e & 3) * 2;
        const unsigned dst = (unsigned)__cvta_generic_to_shared(&W8[(blk * 8 + r) * T8_WS + c2]);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst), "l"(Wb + (size_t)(blk * 8 + r) * NB + blk * 8 + c2));
    }
    asm volatile("cp.async.commit_group;\n" ::);
    // Row blocks of 64 rows are dealt round-robin to the CTAs of this matrix (blockIdx.x, stride gridDim.x): with many
    // matrices in flight a CTA solves several row blocks against the L11 it staged once (the 108 KB prologue is what
    // kept the DMMA pipe at 75 % when every CTA took a single block).
    // n_rows counts a border row too; the last row block takes every row that is left (at most 64 + 1)
    const int rb_first = blk_of(blockIdx.x);
    const int row0_first = row_start + rb_first * T8_ROWS;
    const int rv_first = (rb_first == nblk - 1) ? min(T8_ROWS + 8, n_rows - row0_first) : T8_ROWS;
    // this warp's 8 rows as accumulator fragments: acc[b8] = row warp*8 + fr, cols b8*8 + 2fk, +1
    double acc[T8_NB8][2];
    const int r_loc = warp * 8 + fr;
    // rows this lane solves in row block rb
    auto row_ok = [&](int rb, int row0, int rows_valid) { return r_loc < rows_valid && (!border_only(rb) || row0 + r_loc >= env.n); };
    {
        const double *grow0 = view_elem(A, m, row0_first + min(r_loc, max(rv_first, 1) - 1), j0 + 2 * fk);
        const bool ok = row_ok(rb_first, row0_first, rv_first);
#pragma unroll
        for (int b8 = 0; b8 < T8_NB8; ++b8) {
            double2 v = make_double2(0.0, 0.0);
            if (ok && b8 * 8 + 2 * fk < ncv) v = *reinterpret_cast<const double2 *>(grow0 + b8 * 8);
            acc[b8][0] = v.x;
            acc[b8][1] = v.y;
        }
    }
    asm volatile("cp.async.wait_group 0;\n" ::);
    __syncthreads();
    // the strict upper triangle of the diagonal blocks is garbage in global memory (L) or must read as zero (W8)
    for (int e = tid; e < T8_NSB * 32 * 32; e += T8_THREADS) {
        const int d = e >> 10, r = (e >> 5) & 31, c = e & 31;
        if (c > r) Lb[lblk8_index(d, d) * T8_LBLK + r * T8_B + c] = 0.0;
    }
    for (int e = tid; e < T8_NB8 * 64; e += T8_THREADS) {
        const int blk = e >> 6, r = (e >> 3) & 7, c = e & 7;
        if (c > r) W8[(blk * 8 + r) * T8_WS + c] = 0.0;
    }
    __syncthreads();

    for (int li = blockIdx.x; li < nlaunch; li += gridDim.x) {
    const int rb = blk_of(li);
    const int row0 = row_start + rb * T8_ROWS;
    const int rows_valid = (rb == nblk - 1) ? min(T8_ROWS + 8, n_rows - row0) : T8_ROWS;
    if (warp * 8 >= rows_valid) continue;         // nothing to solve (no border row, or a ragged last block)
    if (border_only(rb) && row0 + warp * 8 + 7 < env.n) continue;
    if (env.blk && empty_block(rb)) continue;
    const bool ok = row_ok(rb, row0, rows_valid);
    double *grow = view_elem(A, m, row0 + min(r_loc, max(rows_valid, 1) - 1), j0 + 2 * fk);
    if (rb != rb_first) {
#pragma unroll
        for (int b8 = 0; b8 < T8_NB8; ++b8) {
            double2 v = make_double2(0.0, 0.0);
            if (ok && b8 * 8 + 2 * fk < ncv) v = *reinterpret_cast<const double2 *>(grow + b8 * 8);
            acc[b8][0] = v.x;
            acc[b8][1] = v.y;
        }
    }
#pragma unroll
    for (int b8 = 0; b8 < T8_NB8; ++b8) {
        const int sb = b8 >> 2, q = b8 & 3;
        // B fragments of the diagonal 8x8 blocks: lane (c = fr, fk) takes [c][2fk] for k-step 0 and [c][2fk+1] for k-step 1
        const double2 w = *reinterpret_cast<const double2 *>(W8 + (b8 * 8 + fr) * T8_WS + 2 * fk);
        const double2 l = *reinterpret_cast<const double2 *>(Lb + lblk8_index(sb, sb) * T8_LBLK + (q * 8 + fr) * T8_B + q * 8 + 2 * fk);
        // ---- X0 = A W8^T   (the accumulator pair is the A operand of the two k-steps)
        double x0 = 0.0, x1 = 0.0;
        dmma884_8(x0, x1, acc[b8][0], w.x);
        dmma884_8(x0, x1, acc[b8][1], w.y);
        // ---- r = A - X0 L8^T
        double r0 = acc[b8][0], r1 = acc[b8][1];
        dmma884_8(r0, r1, -x0, l.x);
        dmma884_8(r0, r1, -x1, l.y);
        // ---- X = X0 + r W8^T   (one step of iterative refinement)
        dmma884_8(x0, x1, r0, w.x);
        dmma884_8(x0, x1, r1, w.y);
        acc[b8][0] = x0; acc[b8][1] = x1;
        // ---- later columns:  acc[:, b'] -= X L[b', b8]^T   (the next block first: it is the one the chain waits for)
        const double nx0 = -x0, nx1 = -x1;
#pragma unroll
        for (int bp = b8 + 1; bp < T8_NB8; ++bp) {
            const double2 lp = *reinterpret_cast<const double2 *>(Lb + lblk8_index(bp >> 2, sb) * T8_LBLK + ((bp & 3) * 8 + fr) * T8_B + q * 8 + 2 * fk);
            dmma884_8(acc[bp][0], acc[bp][1], nx0, lp.x);
            dmma884_8(acc[bp][0], acc[bp][1], nx1, lp.y);
        }
        // ---- the finished 8 columns leave from the accumulator registers (4 lanes x 16 bytes per row)
        if (ok) {
            const int c = b8 * 8 + 2 * fk;
            if (c + 1 < ncv) *reinterpret_cast<double2 *>(grow + b8 * 8) = make_double2(x0, x1);
            else if (c < ncv) grow[b8 * 8] = x0;
        }
    }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Block inverses for inverse_sequence:  W_i = L_ii^-1 for every 128x128 diagonal block of a factored matrix, from the
// 8x8 diagonal inverses the panel factor kernel left in W.  It is the same solve run on the identity:
// Y L_ii^T = I  gives  Y = L_ii^-T = W_i^T  (one refinement step included), stored transposed.  One launch covers all
// blocks of all matrices (2 CTAs of 64 identity rows per block); the 8x8 diagonal blocks of W are kept as they are, so
// the two CTAs of a block never write what the other one reads.
__global__ void __launch_bounds__(T8_THREADS, 2)
inv_blocks8_kernel(BatchView A, int n, double *__restrict__ W, long long strideW)
{
    extern __shared__ __align__(16) double sm[];
    double *Lb = sm;
    double *W8 = sm + T8_NLB * T8_LBLK;
    const int b = blockIdx.y;
    if (A.count && b >= *A.count) return;
    const int m = batch_item(A, b);
    const int blk_i = blockIdx.x >> 1, half = blockIdx.x & 1;
    const int i0 = blk_i * NB;
    const int nv = min(NB, n - i0);               // rows/cols of this diagonal block that exist
    const double *Ab = A.base + (size_t)m * A.stride;
    const int ld = A.ld;
    double *Wi = W + (size_t)m * strideW + (size_t)blk_i * NB * NB;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int fr = lane >> 2, fk = lane & 3;

    for (int e = tid; e < T8_NLB * 32 * 16; e += T8_THREADS) {
        const int blk = e / (32 * 16), rem = e - blk * 32 * 16;
        const int r = rem / 16, c2 = (rem - r * 16) * 2;
        int bi = 0;
        while ((bi + 1) * (bi + 2) / 2 <= blk) ++bi;
        const int bj = blk - bi * (bi + 1) / 2;
        const int gr = bi * 32 + r, gc = bj * 32 + c2;
        double *dstp = &Lb[blk * T8_LBLK + r * T8_B + c2];
        if (gr < nv && gc < nv) {
            const unsigned dst = (unsigned)__cvta_generic_to_shared(dstp);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst), "l"(Ab + (size_t)(i0 + gr) * ld + i0 + gc));
        } else {                                  // beyond the matrix: identity
            dstp[0] = (gr == gc) ? 1.0 : 0.0;
            dstp[1] = (gr == gc + 1) ? 1.0 : 0.0;
        }
    }
    for (int e = tid; e < T8_NB8 * 8 * 4; e += T8_THREADS) {
        const int blk = e >> 5, r = (e >> 2) & 7, c2 = (e & 3) * 2;
        const unsigned dst = (unsigned)__cvta_generic_to_shared(&W8[(blk * 8 + r) * T8_WS + c2]);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst), "l"(Wi + (size_t)(blk * 8 + r) * NB + blk * 8 + c2));
    }
    asm volatile("cp.async.commit_group;\n" ::);
    asm volatile("cp.async.wait_group 0;\n" ::);
    __syncthreads();
    for (int e = tid; e < T8_NSB * 32 * 32; e += T8_THREADS) {
        const int d = e >> 10, r = (e >> 5) & 31, c = e & 31;
        if (c > r || (d * 32 + c == nv && d * 32 + r < nv)) Lb[lblk8_index(d, d) * T8_LBLK + r * T8_B + c] = 0.0;   // (pair spill-over at nv)
    }
    for (int e = tid; e < T8_NB8 * 64; e += T8_THREADS) {
        const int blk = e >> 6, r = (e >> 3) & 7, c = e & 7;
        if (c > r) W8[(blk * 8 + r) * T8_WS + c] = 0.0;
    }
    __syncthreads();
    if (warp >= T8_ROWS / 8) return;              // (the border warp of the panel solve has no role here)

    const int rb = half * (T8_ROWS / 8) + warp;   // this warp's identity rows 8 rb .. 8 rb + 7
    double acc[T8_NB8][2];
#pragma unroll
    for (int b8 = 0; b8 < T8_NB8; ++b8) {
        acc[b8][0] = (b8 == rb && 2 * fk == fr) ? 1.0 : 0.0;
        acc[b8][1] = (b8 == rb && 2 * fk + 1 == fr) ? 1.0 : 0.0;
    }
#pragma unroll
    for (int b8 = 0; b8 < T8_NB8; ++b8) {
        // W[c][r] = Y[r][c]:  c = 8 b8 + 2 fk (+1),  r = 8 rb + fr
        double *out = Wi + (size_t)(b8 * 8 + 2 * fk) * NB + rb * 8 + fr;
        if (b8 < rb) { out[0] = 0.0; out[NB] = 0.0; continue; }      // Y is upper triangular: W has zeros above its diagonal
        const int sb = b8 >> 2, q = b8 & 3;
        const double2 w = *reinterpret_cast<const double2 *>(W8 + (b8 * 8 + fr) * T8_WS + 2 * fk);
        const double2 l = *reinterpret_cast<const double2 *>(Lb + lblk8_index(sb, sb) * T8_LBLK + (q * 8 + fr) * T8_B + q * 8 + 2 * fk);
        double x0 = 0.0, x1 = 0.0;
        dmma884_8(x0, x1, acc[b8][0], w.x);
        dmma884_8(x0, x1, acc[b8][1], w.y);
        double r0 = acc[b8][0], r1 = acc[b8][1];
        dmma884_8(r0, r1, -x0, l.x);
        dmma884_8(r0, r1, -x1, l.y);
        dmma884_8(x0, x1, r0, w.x);
        dmma884_8(x0, x1, r1, w.y);
        const double nx0 = -x0, nx1 = -x1;
#pragma unroll
        for (int bp = b8 + 1; bp < T8_NB8; ++bp) {
            const double2 lp = *reinterpret_cast<const double2 *>(Lb + lblk8_index(bp >> 2, sb) * T8_LBLK + ((bp & 3) * 8 + fr) * T8_B + q * 8 + 2 * fk);
            dmma884_8(acc[bp][0], acc[bp][1], nx0, lp.x);
            dmma884_8(acc[bp][0], acc[bp][1], nx1, lp.y);
        }
        if (b8 > rb) { out[0] = x0; out[NB] = x1; }                  // the diagonal 8x8 blocks stay as the factor kernel wrote them
    }
}

int launch_inv_blocks8(BatchView A, int n, double *W, long long strideW, int B, cudaStream_t s)
{
    if (B <= 0 || n <= 0) return 0;
    if (A.ld & 1) { set_error("inv_blocks: ld=%d must be even", A.ld); return GPMC_EALIGN; }
    static DeviceOnce attr_set;
    if (attr_set.first()) {
        GPMC_CUDA_CHECK(cudaFuncSetAttribute(inv_blocks8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, T8_SMEM));
    }
    const int nt = (n + NB - 1) / NB;
    dim3 grid(2 * nt, B);
    prof_begin(KC_INV, s);
    inv_blocks8_kernel<<<grid, T8_THREADS, T8_SMEM, s>>>(A, n, W, strideW);
    prof_end(KC_INV, s);
    GPMC_LAUNCH_CHECK();
    return 0;
}

static int g_trsm_blocks_per_cta = 0;
void set_trsm_blocks_per_cta(int v) { g_trsm_blocks_per_cta = v; }

int launch_trsm_panel8(BatchView A, int n_rows, int j0, const double *W, long long strideW, int B, cudaStream_t s, int row_start, int n_mat,
                       Envelope env)
{
    // default: every row below the diagonal block; row_start / n_mat: only the rows from row_start on (the border rows
    // of the LAST block column, whose diagonal block may be ragged: L11 rows / columns >= n_mat read as identity)
    if (row_start < 0) row_start = j0 + NB;
    if (n_mat < 0) n_mat = 0x7fffffff;
    int rows = n_rows - row_start;
    if (B <= 0 || rows <= 0) return 0;
    if ((A.ld & 1) || (j0 & 1)) { set_error("trsm_panel: ld=%d j0=%d must be even", A.ld, j0); return GPMC_EALIGN; }
    if (rows > 1 && rows % T8_ROWS == 1) rows -= 1;         // 64 k + 1: the extra row rides in the last CTA
    static DeviceOnce attr_set;
    if (attr_set.first()) {
        GPMC_CUDA_CHECK(cudaFuncSetAttribute(trsm_panel8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, T8_SMEM));
    }
    const int nblk = (rows + T8_ROWS - 1) / T8_ROWS;
    // band (env.band >= 0, rows below the matrix present): the row blocks that can hold a nonzero left of j0 + NB are the
    // first env.band ones; the others would leave at once -- launch those and the last block (its border rows)
    int nband = -1;
    if (env.blk && env.band >= 0 && n_rows > env.n && row_start == j0 + NB && env.band < nblk - 1) nband = env.band;
    const int nlaunch = nband >= 0 ? nband + 1 : nblk;
    // CTAs per matrix: one per row block while the launch would not fill the chip several times over, else up to
    // four row blocks per CTA (g_trsm_blocks_per_cta overrides: experiments)
    int per_cta = g_trsm_blocks_per_cta;
    if (per_cta <= 0) {
        const long long ctas = (long long)nlaunch * B;
        per_cta = ctas >= 16 * 296 ? 4 : (ctas >= 8 * 296 ? 2 : 1);
    }
    dim3 grid((nlaunch + per_cta - 1) / per_cta, B);
    prof_begin(KC_TRSM, s);
    trsm_panel8_kernel<<<grid, T8_THREADS, T8_SMEM, s>>>(A, n_rows, j0, W, strideW, nblk, row_start, n_mat, env, nband);
    prof_end(KC_TRSM, s);
    GPMC_LAUNCH_CHECK();
    return 0;
}

}  // namespace gpmc
