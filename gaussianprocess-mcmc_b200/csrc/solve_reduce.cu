// Fused forward substitution + quadratic form + log-determinant:
//   z = L^-1 (a - b) ;  loglik = -( 0.5 * z.z + sum_i log L_ii + 0.5 * n * log(2 pi) )
// (also used for the whitening eta = C^-1 (f - m), sliceSample.py:108, with loglik = nullptr)
//
// Replaces the reference's log-marginal term (sliceSample.py:122,147; Cholesky/alpha form :120-121,145-146):
//   -(g^T inv(K_S) g / 2 + log(diag(L_ks^T)).sum() + n*log(2*pi)/2)
// g^T (L L^T)^-1 g = |L^-1 g|^2, so one triangular solve replaces the dense inverse (or the two
// solves of solve_chol) and L is read exactly once: 8*n*(n+1)/2 bytes per item, HBM-read bound.
//
// One CTA per batch item.  z lives in shared memory; the matrix is walked in block rows of 64:
// a coalesced GEMV (w = g_R - L[R, :k] z[:k], double2 row reads) followed by a 64x64 triangular
// solve done by one warp with register-resident w and shuffle broadcasts.
#include "common.cuh"
#include "../../include/gpmc.h"

namespace gpmc {

constexpr int SB = 64;                 // block-row height
constexpr int SBP = SB + 1;            // padded stride of the staged diagonal block
constexpr int SOLVE_THREADS = 256;
constexpr int SOLVE_MAX_N = 16384;

__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__global__ void __launch_bounds__(SOLVE_THREADS, 1)
solve_reduce_kernel(BatchView L, int n, const double *va, const double *__restrict__ vb, int ldv,
                    double *zout, double *__restrict__ loglik, const int *__restrict__ info)     // zout may alias va (in place)
{
    extern __shared__ __align__(16) double sm[];
    const int npad = (n + SB - 1) / SB * SB;
    double *z = sm;                        // [npad]
    double *D = sm + npad;                 // [SB][SBP] diagonal block
    double *red = D + SB * SBP;            // [16] reduction scratch
    const int b = blockIdx.x;
    if (L.count && b >= *L.count) return;
    const int m = batch_item(L, b);
    const double *Lb = L.base + (size_t)m * L.stride;
    const int ld = L.ld;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (info && info[m] != 0) {
        if (tid == 0 && loglik) loglik[m] = nan("");
        if (zout) for (int i = tid; i < n; i += SOLVE_THREADS) zout[(size_t)m * ldv + i] = nan("");
        return;
    }
    for (int i = tid; i < npad; i += SOLVE_THREADS) {
        double v = 0.0;
        if (i < n) { v = va[(size_t)m * ldv + i]; if (vb) v -= vb[(size_t)m * ldv + i]; }
        z[i] = v;
    }
    __syncthreads();

    double logdet = 0.0;                   // accumulated by warp 0 lanes
    const int nblk = npad / SB;
    for (int jb = 0; jb < nblk; ++jb) {
        const int r0 = jb * SB;
        const int kmax = r0;               // columns [0, kmax) are solved
        // stage the diagonal block (rows r0.., cols r0..); rows beyond n -> identity
        for (int e = tid; e < SB * SB; e += SOLVE_THREADS) {
            const int r = e / SB, c = e - r * SB;
            double v = 0.0;
            if (r0 + r < n) { if (c <= r) v = Lb[(size_t)(r0 + r) * ld + r0 + c]; }
            else if (c == r) v = 1.0;
            D[r * SBP + c] = v;
        }
        // GEMV: each warp owns 8 rows, 4 at a time
        for (int rr = 0; rr < 8; rr += 4) {
            double acc[4] = {0.0, 0.0, 0.0, 0.0};
            const double *rowp[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int r = r0 + warp * 8 + rr + q;
                rowp[q] = Lb + (size_t)min(r, n - 1) * ld;
            }
#pragma unroll 4
            for (int k = 2 * lane; k < kmax; k += 64) {
                const double2 zz = *reinterpret_cast<const double2 *>(z + k);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const double2 l = *reinterpret_cast<const double2 *>(rowp[q] + k);
                    acc[q] = fma(l.x, zz.x, acc[q]);
                    acc[q] = fma(l.y, zz.y, acc[q]);
                }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const double s = warp_sum(acc[q]);
                const int r = r0 + warp * 8 + rr + q;
                if (lane == 0 && r < n) z[r] -= s;
            }
        }
        __syncthreads();
        // 64x64 triangular solve by warp 0; lane holds rows lane and lane+32
        if (warp == 0) {
            double w0 = z[r0 + lane], w1 = z[r0 + lane + 32];
            const double d0 = D[lane * SBP + lane], d1 = D[(lane + 32) * SBP + lane + 32];
            const double i0 = 1.0 / d0, i1 = 1.0 / d1;
            if (r0 + lane < n) logdet += log(d0);
            if (r0 + lane + 32 < n) logdet += log(d1);
            for (int c = 0; c < 32; ++c) {
                const double zc = __shfl_sync(0xffffffffu, w0 * i0, c);
                if (lane == c) w0 = zc;
                if (lane > c) w0 = fma(-D[lane * SBP + c], zc, w0);
                w1 = fma(-D[(lane + 32) * SBP + c], zc, w1);
            }
            for (int c = 0; c < 32; ++c) {
                const double zc = __shfl_sync(0xffffffffu, w1 * i1, c);
                if (lane == c) w1 = zc;
                if (lane > c) w1 = fma(-D[(lane + 32) * SBP + 32 + c], zc, w1);
            }
            z[r0 + lane] = w0;
            z[r0 + lane + 32] = w1;
        }
        __syncthreads();
    }
    if (zout) for (int i = tid; i < n; i += SOLVE_THREADS) zout[(size_t)m * ldv + i] = z[i];
    if (!loglik) return;
    // quadratic form
    double q = 0.0;
    for (int i = tid; i < n; i += SOLVE_THREADS) q = fma(z[i], z[i], q);
    q = warp_sum(q);
    if (lane == 0) red[warp] = q;
    if (warp == 0) { logdet = warp_sum(logdet); if (lane == 0) red[8] = logdet; }
    __syncthreads();
    if (tid == 0) {
        double qs = 0.0;
        for (int w = 0; w < SOLVE_THREADS / 32; ++w) qs += red[w];
        const double log2pi = 1.8378770664093453;      // log(2*pi)
        loglik[m] = -(qs / 2.0 + red[8] + n * log2pi / 2.0);
    }
}

// ---- few matrices (B < 32): the one-CTA-per-matrix walk above would leave the chip idle (N=16384: 1 GiB read by one
// SM), so the same substitution is run RIGHT-LOOKING in launches: solve the 128x128 diagonal block (the kernel above
// on a sub-view), then every row below subtracts its 128-column contribution in parallel over the whole chip.
__global__ void __launch_bounds__(256)
gemv_sub_kernel(BatchView L, int n, int j0, const double *z, double *w, int ldv, const int *__restrict__ info)   // w aliases z (other rows)
{
    const int b = blockIdx.y;
    if (L.count && b >= *L.count) return;
    const int m = batch_item(L, b);
    if (info && info[m] != 0) return;
    const double *Lb = L.base + (size_t)m * L.stride;
    const double *zv = z + (size_t)m * ldv + j0;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double2 zc[NB / 64];
#pragma unroll
    for (int q = 0; q < NB / 64; ++q) zc[q] = *reinterpret_cast<const double2 *>(zv + q * 64 + 2 * lane);
#pragma unroll
    for (int rr = 0; rr < 4; ++rr) {
        const int r = j0 + NB + blockIdx.x * 32 + warp * 4 + rr;
        if (r >= n) break;
        const double *row = Lb + (size_t)r * L.ld + j0;
        double acc = 0.0;
#pragma unroll
        for (int q = 0; q < NB / 64; ++q) {
            const double2 l = *reinterpret_cast<const double2 *>(row + q * 64 + 2 * lane);
            acc = fma(l.x, zc[q].x, fma(l.y, zc[q].y, acc));
        }
        acc = warp_sum(acc);
        if (lane == 0) w[(size_t)m * ldv + r] -= acc;
    }
}

// w[m] = a[m] for the (possibly mapped) items of the launch
__global__ void copy_vec_mapped_kernel(BatchView L, int n, const double *__restrict__ a, double *__restrict__ w, int ldv)
{
    const int b = blockIdx.y;
    if (L.count && b >= *L.count) return;
    const int m = batch_item(L, b);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) w[(size_t)m * ldv + i] = a[(size_t)m * ldv + i];
}

__global__ void __launch_bounds__(256)
quad_logdet_kernel(BatchView L, int n, const double *__restrict__ z, int ldv, double *__restrict__ loglik, const int *__restrict__ info)
{
    const int b = blockIdx.x;
    if (L.count && b >= *L.count) return;
    const int m = batch_item(L, b);
    __shared__ double rq[8], rl[8];
    if (info && info[m] != 0) { if (threadIdx.x == 0) loglik[m] = nan(""); return; }
    double q = 0.0, ld = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double zi = z[(size_t)m * ldv + i];
        q = fma(zi, zi, q);
        ld += log(*view_elem(L, m, i, i));
    }
    q = warp_sum(q); ld = warp_sum(ld);
    if ((threadIdx.x & 31) == 0) { rq[threadIdx.x >> 5] = q; rl[threadIdx.x >> 5] = ld; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double qs = 0.0, ls = 0.0;
        for (int w = 0; w < 8; ++w) { qs += rq[w]; ls += rl[w]; }
        loglik[m] = -(qs / 2.0 + ls + n * 1.8378770664093453 / 2.0);
    }
}

int launch_quad_logdet(BatchView L, int n, const double *z, int ldv, double *loglik, const int *info, int B, cudaStream_t s)
{
    if (B <= 0) return 0;
    prof_begin(KC_SOLVE, s);
    quad_logdet_kernel<<<B, 256, 0, s>>>(L, n, z, ldv, loglik, info);
    prof_end(KC_SOLVE, s);
    GPMC_LAUNCH_CHECK();
    return 0;
}

int launch_solve_reduce(BatchView L, int n, const double *a, const double *b, int ldv, double *zout,
                        double *loglik, const int *info, int B, cudaStream_t s)
{
    if (B <= 0) return 0;
    if (n > SOLVE_MAX_N) { set_error("solve_reduce: n=%d exceeds %d", n, SOLVE_MAX_N); return GPMC_EINVAL; }
    static DeviceOnce attr_set;
    if (attr_set.first()) GPMC_CUDA_CHECK(cudaFuncSetAttribute(solve_reduce_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    if (B < 32 && n >= 1024 && zout && !b && (n % NB) == 0 && (ldv & 1) == 0) {
        // right-looking in launches; zout doubles as the working right-hand side
        copy_vec_mapped_kernel<<<dim3((n + 255) / 256, B), 256, 0, s>>>(L, n, a, zout, ldv);   // items may be mapped slots
        const int smem128 = (NB + SB * SBP + 16) * (int)sizeof(double);
        prof_begin(KC_SOLVE, s);
        for (int j0 = 0; j0 < n; j0 += NB) {
            BatchView D{L.base + (size_t)j0 * L.ld + j0, L.stride, L.ld, L.map, L.count};
            solve_reduce_kernel<<<B, SOLVE_THREADS, smem128, s>>>(D, NB, zout + j0, nullptr, ldv, zout + j0, nullptr, info);
            if (j0 + NB < n)
                gemv_sub_kernel<<<dim3((n - j0 - NB + 31) / 32, B), 256, 0, s>>>(L, n, j0, zout, zout, ldv, info);
        }
        if (loglik) quad_logdet_kernel<<<B, 256, 0, s>>>(L, n, zout, ldv, loglik, info);
        prof_end(KC_SOLVE, s);
        GPMC_LAUNCH_CHECK();
        return 0;
    }
    const int npad = (n + SB - 1) / SB * SB;
    const int smem = (npad + SB * SBP + 16) * (int)sizeof(double);
    prof_begin(KC_SOLVE, s);
    solve_reduce_kernel<<<B, SOLVE_THREADS, smem, s>>>(L, n, a, b, ldv, zout, loglik, info);
    prof_end(KC_SOLVE, s);
    GPMC_LAUNCH_CHECK();
    return 0;
}

}  // namespace gpmc
