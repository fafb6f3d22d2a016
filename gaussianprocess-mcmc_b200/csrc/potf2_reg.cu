// Panel factor kernel, third form: the 128x128 diagonal block lives in REGISTERS as 8x8 DMMA accumulator fragments
// spread over 8 warps, and is factored right-looking in 16 steps of 8 columns.  Used wherever potf2_lite.cu was
// (kcGP.tools.jitchol call sites sliceSample.py:196,205): same inputs, same outputs (L11 in place, the sixteen 8x8
// diagonal inverses in W, LAPACK-style info).
//
// Why: potf2_lite spends 42 % of its time in ONE warp that walks the 32 columns of a 32x32 sub-block with a row per
// lane (ncu stall sampling, round 1) while the other warps wait, and stages the block through 90 KB of shared memory.
// Here the sequential part shrinks to an 8x8 factorisation per step, and everything else is DMMA work on
// register-resident fragments:
//
//   step b = 0..15  (block column b of 8x8 fragments)
//     A  the warp that owns fragment (b,b) factors it together with its inverse: the 8 rows of the fragment and the 8
//        rows of an identity ride in lanes 0-7 and 8-15 of ONE instruction stream (the elimination applies the same
//        row operation to both), the next pivot is computed and broadcast before anything else (it is the critical
//        path of the whole kernel) and its reciprocal square root is MUFU.RSQ64H + two Newton steps
//     B  owners of fragments (r,b), r > b:  X = A W8^T, r = A - X L8^T, X += r W8^T  (inverse-multiply + one step of
//        iterative refinement, the scheme of trsm_panel8.cu) -> global memory and the shared panel buffer
//     C  every fragment (r,c), c > b:  acc -= X_r X_c^T   (2 DMMAs; X_r is the owner's own register pair -- with the
//        contraction index of m8n8k4 permuted (k-step 0: k = 2 fk, k-step 1: k = 2 fk + 1) an accumulator pair IS the
//        A-operand pair -- and X_c is one 16-byte shared-memory load)
//   two block barriers per step; the owner of (b+1,b+1) updates that fragment first and starts factoring while the
//   others finish their updates.
//
// Ownership: warp w holds block rows w and 15-w = 17 fragments = 34 doubles per lane, in slots with COMPILE-TIME
// register indices, ordered by block column (slot 2c / 2c+1 = column c of row w / row 15-w while c <= w, then the
// remaining columns of row 15-w).  With that order the fragments still alive at step b (column > b) are a SUFFIX of
// the slot list, so phase C is one computed jump into a straight-line sequence of 17 slot updates -- no per-slot
// predicates (the first version walked all 17 slots with warp-uniform tests in phases B and C: 3400 warp instructions
// per step, ncu r02c) -- and phase B picks its (at most two) fragments with a 17-way switch.
// Shared memory: 10 KB; registers bound the occupancy at two CTAs (two matrices) per SM, which hides one CTA's
// single-warp phase A behind the other's DMMA phases.
#include "common.cuh"
#include "../../include/gpmc.h"

namespace gpmc {

static_assert(NB == 128, "potf2_reg is written for a panel width of 128 (16 x 16 fragments, 8 warps)");
constexpr int PR_NF = NB / 8;                 // 8x8 fragments per block row / column (16)
constexpr int PR_WARPS = PR_NF / 2;           // 8 warps: warp w owns block rows w and PR_NF-1-w
constexpr int PR_THREADS = PR_WARPS * 32;
constexpr int PR_SLOTS = PR_NF + 1;           // (w + 1) + (PR_NF - w) fragments per warp

__device__ __forceinline__ void dmma884_r(double &c0, double &c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// 1/sqrt(a) for the pivot chain: the hardware approximation (MUFU.RSQ64H, ~2^-22) plus two Newton steps,
// y <- y + y (1/2 - (a/2) y^2): 6 dependent FP64 operations instead of the ~25 instructions (special-case handling
// included) of the library rsqrt(), which sat on the critical path of every one of the 128 pivots.  Result within 1-2 ulp;
// a <= 0 or NaN gives NaN / inf, which is what a failed pivot is allowed to produce (info is set by the caller).
__device__ __forceinline__ double pivot_rsqrt(double a)
{
    // one third-order step from the hardware approximation (MUFU.RSQ64H, ~2^-22):  e = 1/2 - (a/2) y^2,
    // y <- y + y e (1 + 3/2 e)  (error ~ e^3): 4 dependent FP64 operations
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(a));
    const double h = 0.5 * a;
    const double e = fma(-(h * y), y, 0.5);
    return fma(y * e, fma(1.5, e, 1.0), y);
}
// 1/a for the pivot CHAIN (the next pivot is a_{c+1,c+1} - a_{c+1,c}^2 / a_cc and must not wait for the square root):
// MUFU.RCP64H + one third-order step,  e = 1 - a y,  y <- y + y (e + e^2): 3 dependent FP64 operations
__device__ __forceinline__ double pivot_rcp(double a)
{
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(a));
    const double e = fma(-a, y, 1.0);
    return fma(y, fma(e, e, e), y);
}

// slot -> (block row, block column) of warp w (see the header comment)
__device__ __forceinline__ void slot_rc(int s, int w, int &R, int &C, bool &isA)
{
    if (s < 2 * (w + 1)) { C = s >> 1; isA = (s & 1) == 0; }
    else { C = s - w - 1; isA = false; }
    R = isA ? w : PR_NF - 1 - w;
}

// phase C for one slot: acc -= X_R X_C^T
template <int S>
__device__ __forceinline__ void slot_update(double (&acc)[PR_SLOTS][2], int w, double xa0, double xa1, double xb0, double xb1,
                                            const double (*sX)[64], int frag_off)
{
    int R, C; bool isA;
    slot_rc(S, w, R, C, isA);
    const double n0 = isA ? -xa0 : -xb0, n1 = isA ? -xa1 : -xb1;
    double2 xc;
    if (C == R) xc = make_double2(-n0, -n1);                              // diagonal fragment: X_C is this warp's own pair
    else xc = *reinterpret_cast<const double2 *>(&sX[C][frag_off]);
    dmma884_r(acc[S][0], acc[S][1], n0, xc.x);
    dmma884_r(acc[S][0], acc[S][1], n1, xc.y);
}

#define PR_CASE(S) case S: slot_update<S>(acc, w, xa0, xa1, xb0, xb1, sX, frag_off);
#define PR_PICK(S) case S: p0 = acc[S][0]; p1 = acc[S][1]; break;
#define PR_PICK_ALL PR_PICK(0) PR_PICK(1) PR_PICK(2) PR_PICK(3) PR_PICK(4) PR_PICK(5) PR_PICK(6) PR_PICK(7) PR_PICK(8) \
    PR_PICK(9) PR_PICK(10) PR_PICK(11) PR_PICK(12) PR_PICK(13) PR_PICK(14) PR_PICK(15) PR_PICK(16)

__device__ __forceinline__ void pick_slot(const double (&acc)[PR_SLOTS][2], int slot, double &p0, double &p1)
{
    p0 = p1 = 0.0;
    switch (slot) { PR_PICK_ALL default: break; }
}

// FUSED = true: the panel SOLVE of the block column happens in the same launch (n_rows > n: border rows included; in the
// last block column only the border rows are left to solve).  The factor's fragments and the 8x8 diagonal inverses are
// kept in 76 KB of shared memory as dense 8x8 blocks (a lane's 16-byte B-operand loads of a block are 512 contiguous
// bytes per warp: conflict free), and after the 16 factor steps every warp takes 8 rows at a time through the same
// inverse-multiply + refinement chain as trsm_panel8.cu.  With one CTA per matrix and two CTAs per SM, one matrix's
// latency-bound factor steps overlap the other's DMMA-bound solve -- which separate launches cannot do: every CTA of a
// launch is in the same phase.  Used when many small matrices are in flight (potrf_sequence decides), and for the compact
// band layout, where every block column has only the band's few rows below its diagonal block.
constexpr int PF_LC_ELEMS = (PR_NF * (PR_NF + 1) / 2) * 64;      // lower 8x8 blocks of L11: block (R, C) at R (R + 1) / 2 + C
constexpr int PF_SMEM = (PF_LC_ELEMS + PR_NF * 64) * (int)sizeof(double);

// Panel solve of one warp's 8 rows,  X L11^T = A21,  from L11 (Lc) and the 8x8 diagonal inverses (W8c) in shared memory:
// the lane's row starts at grow (column j0 + 2 fk; rv: the row exists, else nothing is read or written), nv columns exist.
// Sub-blocks b8 < b8s (warp-uniform) hold exact +0: their X is +0 and their updates of later sub-blocks add +-0, so the
// chain starts at b8s and leaves them as stored.
__device__ __forceinline__ void fused_solve8(double *grow, bool rv, int nv, int b8s, const double *Lc, const double *W8c,
                                             int frag_off, int fk)
{
    double t[PR_NF][2];
#pragma unroll
    for (int b8 = 0; b8 < PR_NF; ++b8) {
        double2 v = make_double2(0.0, 0.0);
        if (rv && b8 >= b8s && b8 * 8 + 2 * fk < nv) v = *reinterpret_cast<const double2 *>(grow + b8 * 8);
        t[b8][0] = v.x;
        t[b8][1] = v.y;
    }
#pragma unroll
    for (int b8 = 0; b8 < PR_NF; ++b8) {
        if (b8 < b8s) continue;
        const double2 wv = *reinterpret_cast<const double2 *>(&W8c[b8 * 64 + frag_off]);
        const double2 lv = *reinterpret_cast<const double2 *>(&Lc[(b8 * (b8 + 1) / 2 + b8) * 64 + frag_off]);
        double x0 = 0.0, x1 = 0.0;
        dmma884_r(x0, x1, t[b8][0], wv.x);                                  // X0 = A W8^T
        dmma884_r(x0, x1, t[b8][1], wv.y);
        double r0 = t[b8][0], r1 = t[b8][1];
        dmma884_r(r0, r1, -x0, lv.x);                                       // r = A - X0 L8^T
        dmma884_r(r0, r1, -x1, lv.y);
        dmma884_r(x0, x1, r0, wv.x);                                        // X = X0 + r W8^T
        dmma884_r(x0, x1, r1, wv.y);
        const double nx0 = -x0, nx1 = -x1;
#pragma unroll
        for (int bp = b8 + 1; bp < PR_NF; ++bp) {
            const double2 lp = *reinterpret_cast<const double2 *>(&Lc[(bp * (bp + 1) / 2 + b8) * 64 + frag_off]);
            dmma884_r(t[bp][0], t[bp][1], nx0, lp.x);
            dmma884_r(t[bp][0], t[bp][1], nx1, lp.y);
        }
        if (rv) {
            const int c = b8 * 8 + 2 * fk;
            if (c + 1 < nv) *reinterpret_cast<double2 *>(grow + b8 * 8) = make_double2(x0, x1);
            else if (c < nv) grow[b8 * 8] = x0;
        }
    }
}

template <bool FUSED>
__global__ void __launch_bounds__(PR_THREADS, 2)
potf2_reg_kernel(BatchView A, int n, int j0, double *__restrict__ W, long long strideW, int *__restrict__ info, int zero_upper, int n_rows,
                 Envelope env)
{
    extern __shared__ __align__(16) double pf_dyn[];
    double *Lc = pf_dyn;                                 // FUSED only
    double *W8c = pf_dyn + PF_LC_ELEMS;
    __shared__ __align__(16) double sD[64];              // diagonal fragment on its way to the row-per-lane layout
    __shared__ __align__(16) double sL8[64], sW8[64];    // factor of the current diagonal fragment and its inverse (zeros above)
    __shared__ __align__(16) double sX[PR_NF][64];       // solved fragments X[block row][8][8] of the current block column
    __shared__ int s_fail;
    const int item = blockIdx.x;
    if (A.count && item >= *A.count) return;
    const int m = batch_item(A, item);
    double *Ab = view_elem(A, m, j0, j0);        // the diagonal block: one 128-row block, row stride A.ld in either layout
    double *Wb = W + (size_t)m * strideW;
    const int ld = A.ld;
    const int nv = min(NB, n - j0);
    const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
    const int fr = lane >> 2, fk = lane & 3;
    const int frag_off = fr * 8 + 2 * fk;
    const int rowA = w, rowB = PR_NF - 1 - w;

    if (tid == 0) s_fail = 0;
    // ---- the block's lower fragments straight into registers (rows / columns beyond the matrix: identity)
    double acc[PR_SLOTS][2];
#pragma unroll
    for (int s = 0; s < PR_SLOTS; ++s) {
        int R, C; bool isA;
        slot_rc(s, w, R, C, isA);
        const int gr = R * 8 + fr, gc = C * 8 + 2 * fk;
        double2 v = make_double2(0.0, 0.0);
        if (gr < nv && gc < nv) v = *reinterpret_cast<const double2 *>(Ab + (size_t)gr * ld + gc);
        if (gr >= nv || gc >= nv) v.x = (gr == gc) ? 1.0 : 0.0;
        if (gr >= nv || gc + 1 >= nv) v.y = (gr == gc + 1) ? 1.0 : 0.0;
        acc[s][0] = v.x;
        acc[s][1] = v.y;
    }
    double xa0 = 0.0, xa1 = 0.0, xb0 = 0.0, xb1 = 0.0;   // solved fragments of rows rowA / rowB in the current block column
    __syncthreads();

#pragma unroll 1
    for (int b = 0; b < PR_NF; ++b) {
        // ------------------------------------------------------------------ A: 8x8 diagonal fragment, one warp
        const bool own_diag = (b < PR_WARPS) ? (w == b) : (w == PR_NF - 1 - b);
        if (own_diag) {
            double d0, d1;
            pick_slot(acc, (b < PR_WARPS) ? 2 * b : PR_SLOTS - 1, d0, d1);
            *reinterpret_cast<double2 *>(&sD[frag_off]) = make_double2(d0, d1);
            __syncwarp();
            // lanes 0-7: row (lane) of the fragment; lanes 8-15: row (lane - 8) of an identity -- eliminating [A; I] gives
            // [L; W^T] column by column: lane 8 + k ends with column k of W8 = L8^-1.  Lanes 16-31 repeat lanes 0-15.
            const int l16 = lane & 15, r8 = lane & 7;
            double v[8];
#pragma unroll
            for (int c = 0; c < 8; c += 2) {
                const double2 t = *reinterpret_cast<const double2 *>(&sD[r8 * 8 + c]);
                v[c] = (l16 < 8) ? ((c <= r8) ? t.x : 0.0) : ((c == r8) ? 1.0 : 0.0);
                v[c + 1] = (l16 < 8) ? ((c + 1 <= r8) ? t.y : 0.0) : ((c + 1 == r8) ? 1.0 : 0.0);
            }
            int fail = 0;
            double piv = __shfl_sync(0xffffffffu, v[0], 0);
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                if (!(piv > 0.0) && fail == 0) fail = j0 + b * 8 + c + 1;           // dpotf2: ajj <= 0 or NaN
                // the next pivot first (it is the critical path of the whole kernel): row c+1 holds its diagonal entry and
                // its own unscaled multiplier a_{c+1,c}, so  a_{c+1,c+1} - a_{c+1,c}^2 / a_cc  needs the reciprocal of the pivot
                // only -- the reciprocal square root (one dependent operation longer) is off the chain
                const double pr = pivot_rcp(piv);
                const double rinv = pivot_rsqrt(piv);
                const double pnext = (c < 7) ? __shfl_sync(0xffffffffu, fma(-(v[c] * v[c]), pr, v[c + 1]), c + 1) : 0.0;
                v[c] = (l16 == c) ? piv * rinv : v[c] * rinv;                       // the pivot row: sqrt(piv) from the pivot the chain used
#pragma unroll
                for (int j = c + 1; j < 8; ++j) {
                    const double ljc = __shfl_sync(0xffffffffu, v[c], j);           // l_{j,c} from row j of the fragment
                    v[j] = fma(-v[c], ljc, v[j]);
                }
                piv = pnext;
            }
            if (lane < 8) {
                const int gr = b * 8 + r8;
#pragma unroll
                for (int c = 0; c < 8; c += 2) {
                    const double2 lrow = make_double2((c <= r8) ? v[c] : 0.0, (c + 1 <= r8) ? v[c + 1] : 0.0);
                    *reinterpret_cast<double2 *>(&sL8[r8 * 8 + c]) = lrow;
                    if (FUSED) *reinterpret_cast<double2 *>(&Lc[(b * (b + 1) / 2 + b) * 64 + r8 * 8 + c]) = lrow;
                }
#pragma unroll
                for (int c = 0; c < 8; ++c)
                    if (c <= r8 && gr < nv) Ab[(size_t)gr * ld + b * 8 + c] = v[c];
                if (fail != 0 && lane == 0 && s_fail == 0) s_fail = fail;           // the FIRST failing pivot (later ones are NaN)
            } else if (lane < 16) {
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    sW8[c * 8 + r8] = v[c];                                         // W8[c][k = r8]; zero for c < k
                    if (FUSED) W8c[b * 64 + c * 8 + r8] = v[c];
                    Wb[(size_t)(b * 8 + c) * NB + b * 8 + r8] = v[c];
                }
            }
        }
        __syncthreads();
        // ------------------------------------------------------------------ B: fragments (r, b), r > b (at most two per warp)
        {
            // slot of (rowA, b): 2b while b < w;  slot of (rowB, b): 2b+1 while b <= w, then w+1+b while b < rowB
            const int slotA = (b < w) ? 2 * b : -1;
            const int slotB = (b <= w) ? 2 * b + 1 : ((b < rowB) ? w + 1 + b : -1);
            if (slotB >= 0) {
                const double2 wv = *reinterpret_cast<const double2 *>(&sW8[frag_off]);
                const double2 lv = *reinterpret_cast<const double2 *>(&sL8[frag_off]);
                double a0, a1, b0, b1;
                pick_slot(acc, slotA, a0, a1);                                      // zeros when the warp has no row-A fragment here
                pick_slot(acc, slotB, b0, b1);
                double x0 = 0.0, x1 = 0.0, y0 = 0.0, y1 = 0.0;
                dmma884_r(x0, x1, a0, wv.x);                                        // X0 = A W8^T   (two independent chains)
                dmma884_r(y0, y1, b0, wv.x);
                dmma884_r(x0, x1, a1, wv.y);
                dmma884_r(y0, y1, b1, wv.y);
                double r0 = a0, r1 = a1, q0 = b0, q1 = b1;
                dmma884_r(r0, r1, -x0, lv.x);                                       // r = A - X0 L8^T
                dmma884_r(q0, q1, -y0, lv.x);
                dmma884_r(r0, r1, -x1, lv.y);
                dmma884_r(q0, q1, -y1, lv.y);
                dmma884_r(x0, x1, r0, wv.x);                                        // X = X0 + r W8^T
                dmma884_r(y0, y1, q0, wv.x);
                dmma884_r(x0, x1, r1, wv.y);
                dmma884_r(y0, y1, q1, wv.y);
                xb0 = y0; xb1 = y1;
                *reinterpret_cast<double2 *>(&sX[rowB][frag_off]) = make_double2(y0, y1);
                if (FUSED) *reinterpret_cast<double2 *>(&Lc[(rowB * (rowB + 1) / 2 + b) * 64 + frag_off]) = make_double2(y0, y1);
                {
                    const int gr = rowB * 8 + fr, gc = b * 8 + 2 * fk;
                    if (gr < nv) {
                        if (gc + 1 < nv) *reinterpret_cast<double2 *>(Ab + (size_t)gr * ld + gc) = make_double2(y0, y1);
                        else if (gc < nv) Ab[(size_t)gr * ld + gc] = y0;
                    }
                }
                if (slotA >= 0) {
                    xa0 = x0; xa1 = x1;
                    *reinterpret_cast<double2 *>(&sX[rowA][frag_off]) = make_double2(x0, x1);
                    if (FUSED) *reinterpret_cast<double2 *>(&Lc[(rowA * (rowA + 1) / 2 + b) * 64 + frag_off]) = make_double2(x0, x1);
                    const int gr = rowA * 8 + fr, gc = b * 8 + 2 * fk;
                    if (gr < nv) {
                        if (gc + 1 < nv) *reinterpret_cast<double2 *>(Ab + (size_t)gr * ld + gc) = make_double2(x0, x1);
                        else if (gc < nv) Ab[(size_t)gr * ld + gc] = x0;
                    }
                }
            }
        }
        __syncthreads();
        // ------------------------------------------------------------------ C: fragments (r, c), c > b: a suffix of the slots
        {
            const int start = (b + 1 <= w) ? 2 * (b + 1) : w + b + 2;
            // (walking the suffix twice, k-step 0 of every slot first, and picking phase B's fragments before the barrier were
            //  both measured: 34.8 -> 36.2 us per block -- not kept)
            switch (start) {
                PR_CASE(0) PR_CASE(1) PR_CASE(2) PR_CASE(3) PR_CASE(4) PR_CASE(5) PR_CASE(6) PR_CASE(7) PR_CASE(8)
                PR_CASE(9) PR_CASE(10) PR_CASE(11) PR_CASE(12) PR_CASE(13) PR_CASE(14) PR_CASE(15) PR_CASE(16)
                default: break;
            }
        }
    }

    __syncthreads();
    if (tid == 0 && s_fail != 0) {
        if (info[m] == 0) info[m] = s_fail;
    }
    if (FUSED && !A.W) {
        // ---------------------------------------------------------------- panel solve: X L11^T = A21 for the rows below
        // (trsm_panel8.cu's chain; a warp owns 8 rows x 128 columns as accumulator fragments, 64 rows per pass of the CTA)
        const int row_start = (j0 + NB < n) ? NB : n - j0;            // relative to the block's first row; last column: border rows only
        const int rows_end = n_rows - j0;
#pragma unroll 1
        for (int row0 = row_start; row0 < rows_end; row0 += 8 * PR_WARPS) {
            if (row0 + w * 8 >= rows_end) continue;                     // warp-uniform
            const int r = row0 + w * 8 + fr;
            fused_solve8(Ab + (size_t)min(r, rows_end - 1) * ld + 2 * fk, r < rows_end, nv, 0, Lc, W8c, frag_off, fk);
        }
    }
    if (FUSED && A.W && j0 + NB < n) {
        // ---------------------------------------------------------------- the same solve in the compact band layout
        // Exactly the rows trsm_panel8 solves for this envelope: the band's 64-row blocks below the diagonal block (all of
        // them when the band reaches the last one) that hold a nonzero left of j0 + NB, then the border row (row n) alone.
        // Other rows are not stored.  The last block column solves nothing: border_finish solves the border row's last
        // block, as after separate launches, so the result is the same to the bit.
        const int r_first = j0 + NB;
        const int nmb = (n - r_first + 63) / 64;
        const int nbl = (env.band >= 0 && env.band < nmb - 1) ? env.band : nmb;
#pragma unroll 1
        for (int rb = 0; rb <= nbl; ++rb) {
            const int row0 = r_first + rb * 64;
            if (rb < nbl) {
                const int e = env_first_col(env, m, row0, min(row0 + 64, n));
                if (e >= j0 + NB || row0 + w * 8 >= n) continue;        // block- / warp-uniform
                const int r = min(row0 + w * 8 + fr, n - 1);
                fused_solve8(view_elem(A, m, r, j0 + 2 * fk), row0 + w * 8 + fr < n, nv, max(e - j0, 0) / 8, Lc, W8c, frag_off, fk);
            } else if (w == 0) {
                fused_solve8(view_elem(A, m, n, j0 + 2 * fk), fr == 0, nv, 0, Lc, W8c, frag_off, fk);
            }
        }
    }
    if (zero_upper) {
        for (int e = tid; e < nv * nv; e += PR_THREADS) {
            const int r = e / nv, c = e - r * nv;
            if (c > r) Ab[(size_t)r * ld + c] = 0.0;
        }
    }
}

int launch_potf2_reg(BatchView A, int n, int j0, double *W, long long strideW, int *info, int zero_upper, int B, cudaStream_t s)
{
    if (B <= 0) return 0;
    if ((A.ld & 1) || (j0 & 1)) { set_error("potf2: ld=%d j0=%d must be even", A.ld, j0); return GPMC_EALIGN; }
    prof_begin(KC_POTF2, s);
    potf2_reg_kernel<false><<<B, PR_THREADS, 0, s>>>(A, n, j0, W, strideW, info, zero_upper, n, Envelope{});
    prof_end(KC_POTF2, s);
    GPMC_LAUNCH_CHECK();
    return 0;
}

// panel factor + panel solve of block column j0 in one launch; n_rows = n + border rows
int launch_panel_fused(BatchView A, int n, int n_rows, int j0, double *W, long long strideW, int *info, int zero_upper, int B, cudaStream_t s,
                       Envelope env)
{
    if (B <= 0) return 0;
    if ((A.ld & 1) || (j0 & 1)) { set_error("panel: ld=%d j0=%d must be even", A.ld, j0); return GPMC_EALIGN; }
    if (A.W && (!env.blk || n_rows != n + 1)) { set_error("panel: the compact band layout needs its envelope and one border row"); return GPMC_EINVAL; }
    static DeviceOnce attr_set;
    if (attr_set.first()) GPMC_CUDA_CHECK(cudaFuncSetAttribute(potf2_reg_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, PF_SMEM));
    prof_begin(KC_POTF2, s);
    potf2_reg_kernel<true><<<B, PR_THREADS, PF_SMEM, s>>>(A, n, j0, W, strideW, info, zero_upper, n_rows, env);
    prof_end(KC_POTF2, s);
    GPMC_LAUNCH_CHECK();
    return 0;
}

}  // namespace gpmc
