// The contraction of the log-likelihood gradient (gpmc_loglik_grad_batched, include/gpmc.h):
//     d loglik / d theta_p = 0.5 sum_ij (alpha_i alpha_j - W_ij) dA_ij/d theta_p,   alpha = A^-1 g,  W = A^-1,
// from the lower triangle of W, one pass over it.  dA_ij/d theta is proportional to K_ij off the diagonal, so K_ij is
// recomputed here from x and theta with cov_assemble_kernel's expression (same operation order, no FMA in the distance):
// its zeros are the assembly's zeros, and the tiles the band bound skipped (K_ij = +0 there) would only add exact zeros.
//     ell (iso):   K_ij s_ij / ell,  s = |x_i - x_j|^2 / ell^2      ell_d (ARD): K_ij (u_id - u_jd)^2 / ell_d,  u = x / ell
//     sf:          2 K_ij / sf                                   sn:          2 sn on the diagonal
// Layout: one CTA per (64-row block r, item), 8 warps x 8 rows, a lane owns two adjacent columns of every 64-column tile
// (W rows are read with 16-byte loads).  Each thread sums its elements tile by tile in column order; the CTA reduces its
// P partials in a fixed tree and writes them out, and a second kernel sums the row blocks of an item in order -- no
// atomics, so repeated calls are bitwise identical, and skipping a tile of exact zeros changes no bit (an accumulator
// that starts at +0 never becomes -0, so adding a +-0 term leaves it as it is).  FP64 throughout; bound by the exp()
// and the W reads (O(N w P) per item for a band of width w).
#include "common.cuh"
#include "../../include/gpmc.h"

namespace gpmc {

constexpr int GT = ENV_ROWS;        // tile edge: one envelope / band row block
constexpr int GC_THREADS = 256;

// E: partials of the length-scales (1 for iso, D for ARD); ISO: one ell for every input dimension
template <int E, bool ISO>
__global__ void __launch_bounds__(GC_THREADS)
grad_contract_kernel(const double *__restrict__ x, int N, int Drt, const double *__restrict__ hyp, int P, int n_ell,
                     const double *__restrict__ alpha, int ldv, const double *__restrict__ W, int ldW, long long strideW,
                     const int *__restrict__ band_w, int ldw, double *__restrict__ partial)
{
    constexpr int NP = E + 2;                       // ell.., sf, sn
    const int D = ISO ? Drt : E;
    const int r = blockIdx.x, b = blockIdx.y, nblk = gridDim.x;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, cl = 2 * lane;
    __shared__ double s_ell[MAX_ELL];
    __shared__ double s_ui[MAX_ELL][GT], s_uj[MAX_ELL][GT];
    __shared__ double s_ai[GT], s_aj[GT];
    __shared__ double s_sf2;
    __shared__ double s_red[GC_THREADS / 32][NP];
    const double *h = hyp + (size_t)b * P;
    if (tid < n_ell) s_ell[tid] = exp(log(h[tid]));             // as cov_assemble_kernel forms them
    if (tid == 32) s_sf2 = exp(2.0 * log(h[n_ell]));
    __syncthreads();
    const int i0 = r * GT;
    const double *ab = alpha + (size_t)b * ldv;
    for (int e = tid; e < GT * D; e += GC_THREADS) {
        const int i = e / D, d = e - i * D;
        s_ui[d][i] = (i0 + i < N) ? x[(size_t)(i0 + i) * D + d] / s_ell[ISO ? 0 : d] : 0.0;
    }
    if (tid < GT) s_ai[tid] = (i0 + tid < N) ? ab[i0 + tid] : 0.0;
    const double sf2 = s_sf2;
    const double *Wb = W + (size_t)b * strideW;

    double acc[NP];
#pragma unroll
    for (int p = 0; p < NP; ++p) acc[p] = 0.0;
    const int c_first = band_w ? band_w[(size_t)b * ldw + r] : 0;
    for (int c = c_first; c <= r; ++c) {
        const int j0 = c * GT;
        __syncthreads();                            // the previous tile's column data has been read
        for (int e = tid; e < GT * D; e += GC_THREADS) {
            const int j = e / D, d = e - j * D;
            s_uj[d][j] = (j0 + j < N) ? x[(size_t)(j0 + j) * D + d] / s_ell[ISO ? 0 : d] : 0.0;
        }
        if (tid < GT) s_aj[tid] = (j0 + tid < N) ? ab[j0 + tid] : 0.0;
        __syncthreads();
        const int gj = j0 + cl;
        for (int rr = 0; rr < 8; ++rr) {
            const int rl = warp * 8 + rr, gi = i0 + rl;
            if (gi >= N) break;                     // rows beyond the matrix
            if (gj > gi) continue;                  // the pair lies above the diagonal (a later row may not)
            const double *wrow = Wb + (size_t)gi * ldW + gj;
            double w0, w1 = 0.0;
            if (gj + 1 < N) { const double2 t = *reinterpret_cast<const double2 *>(wrow); w0 = t.x; w1 = t.y; }
            else w0 = wrow[0];
            const double ai = s_ai[rl];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int jl = cl + q, gjq = gj + q;
                if (gjq > gi || gjq >= N) continue;
                const double wij = q ? w1 : w0;
                double sq[E], s = 0.0;
                if (ISO) {
                    for (int d = 0; d < D; ++d) {
                        const double du = s_ui[d][rl] - s_uj[d][jl];
                        s = __dadd_rn(s, __dmul_rn(du, du));          // cdist 'sqeuclidean' order, as the assembly
                    }
                } else {
#pragma unroll
                    for (int d = 0; d < E; ++d) {
                        const double du = s_ui[d][rl] - s_uj[d][jl];
                        sq[d] = __dmul_rn(du, du);
                        s = __dadd_rn(s, sq[d]);
                    }
                }
                const double k = sf2 * exp(-0.5 * s);
                if (gjq == gi) acc[E + 1] += ai * ai - wij;           // sn: alpha.alpha - tr W
                if (k != 0.0) {
                    double cf = (ai * s_aj[jl] - wij) * k;
                    if (gjq < gi) cf = cf + cf;                       // (i, j) and (j, i)
                    acc[E] += cf;
                    if (ISO) acc[0] += cf * s;
                    else {
#pragma unroll
                        for (int d = 0; d < E; ++d) acc[d] += cf * sq[d];
                    }
                }
            }
        }
    }
#pragma unroll
    for (int p = 0; p < NP; ++p) {
        double v = acc[p];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) s_red[warp][p] = v;
    }
    __syncthreads();
    if (tid < NP) {
        double v = 0.0;
        for (int w8 = 0; w8 < GC_THREADS / 32; ++w8) v += s_red[w8][tid];
        partial[((size_t)b * nblk + r) * NP + tid] = v;
    }
}

// Sum the row blocks of an item in order and scale to the natural-scale gradient.
__global__ void grad_finish_kernel(const double *__restrict__ hyp, int P, int n_ell, const int *__restrict__ info, int nblk,
                                   const double *__restrict__ partial, double *__restrict__ grad)
{
    const int b = blockIdx.x, p = threadIdx.x;
    if (p >= P) return;
    const double *h = hyp + (size_t)b * P;
    double a = 0.0;
    for (int r = 0; r < nblk; ++r) a += partial[((size_t)b * nblk + r) * P + p];
    bool ok = info[b] == 0;
    for (int q = 0; q < P; ++q) ok = ok && isfinite(h[q]) && h[q] > 0.0;
    double g;
    if (p < n_ell) g = 0.5 * a / exp(log(h[p]));    // the ell the assembly used
    else if (p == n_ell) g = a / h[n_ell];
    else g = h[n_ell + 1] * a;
    grad[(size_t)b * P + p] = ok ? g : nan("");
}

int launch_grad_contract(const double *x, int N, int D, const double *hyp, int P, int n_ell, const double *alpha, int ldv,
                         const double *W, int ldW, long long strideW, const int *band_w, int ldw, const int *info,
                         double *partial, double *grad, int B, cudaStream_t s)
{
    if (B <= 0) return 0;
    if (D > MAX_ELL || n_ell > MAX_ELL || P != n_ell + 2 || (n_ell != 1 && n_ell != D)) {
        set_error("grad contraction: D=%d n_ell=%d P=%d", D, n_ell, P);
        return GPMC_EINVAL;
    }
    if ((ldW & 1) || (strideW & 1)) { set_error("grad contraction: W row stride %d must be even", ldW); return GPMC_EALIGN; }
    const int nblk = env_blocks(N);
    dim3 grid(nblk, B);
    prof_begin(KC_GRAD, s);
#define GPMC_GC_LAUNCH(E_, ISO_) \
    grad_contract_kernel<E_, ISO_><<<grid, GC_THREADS, 0, s>>>(x, N, D, hyp, P, n_ell, alpha, ldv, W, ldW, strideW, band_w, ldw, partial)
    switch (n_ell) {
        case 1: GPMC_GC_LAUNCH(1, true); break;
        case 2: GPMC_GC_LAUNCH(2, false); break;
        case 3: GPMC_GC_LAUNCH(3, false); break;
        case 4: GPMC_GC_LAUNCH(4, false); break;
        case 5: GPMC_GC_LAUNCH(5, false); break;
        case 6: GPMC_GC_LAUNCH(6, false); break;
        case 7: GPMC_GC_LAUNCH(7, false); break;
        default: GPMC_GC_LAUNCH(8, false); break;
    }
#undef GPMC_GC_LAUNCH
    grad_finish_kernel<<<B, 32, 0, s>>>(hyp, P, n_ell, info, nblk, partial, grad);
    prof_end(KC_GRAD, s);
    GPMC_LAUNCH_CHECK();
    return 0;
}

}  // namespace gpmc
