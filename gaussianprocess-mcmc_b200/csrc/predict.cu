// The two samplers' "next" rows as device paths (SURVEY 8f):
//
//  gpmc_predict_batched   inf_mcmc (kcMCMC/sliceSample.py:234-284; callers framework.py:223-243, plotResult.py:121) for
//                         S stored MCMC samples (f_s, theta_s) AT ONCE: per sample assemble K/sn^2 + I (:256-257), factor
//                         it (jitchol), and carry 1 + ns right-hand sides -- f_s - m and the ns columns of sW o Ks
//                         (:258,263,269) -- through the factorisation as border ROWS below the matrix: the update GEMM and
//                         the panel solve treat them like any other rows under the diagonal, so
//                             z0 = L^-1 (f - m),   V = L^-1 (sW o Ks)
//                         come out of the Cholesky launches on DMMA with no separate triangular solve, and
//                             Fmu - ms = Ks^T alpha = V^T z0 * sW        (alpha = (K + sn^2 I)^-1 (f - m), :258,266)
//                             fs2      = kss - sum_i V_i^2               (:270)
//                         are two dot products per test point.
//
//  gpmc_ess_sweep         elliptical_slice (sliceSample.py:15-74) for B chains: nu = chol(K) z on the device (the
//                         reference draws nu ~ N(0, K) through numpy's SVD route, :41 -- equal in distribution), then the
//                         whole bracket-shrinking loop on the ellipse (:58-74) in ONE kernel per chain; randomness from
//                         an explicit tape in the reference's draw order (:51,54,74) or Philox.
#include "common.cuh"
#include "sequences.cuh"
#include "tg2.cuh"
#include "../../include/gpmc.h"

#include <algorithm>
#include <vector>

namespace gpmc {

// ------------------------------------------------------------------------------------ predictive path
// Border rows of sample `item`:  row n = fm (= f - m),  row n + 1 + j = sW * K(x, xs_j)   (sW = 1 / sqrt(sn2))
template <int CF>
__global__ void __launch_bounds__(256)
pred_border_kernel(BatchView A, int n, int D, int M, const double *__restrict__ x, const double *__restrict__ xs,
                   const double *__restrict__ hyp, int P, int n_ell, const double *__restrict__ fm)
{
    const int b = blockIdx.z;
    if (A.count && b >= *A.count) return;
    const int m = batch_item(A, b);
    const int row = blockIdx.y;                       // 0: f - m, 1 + j: test point j
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= A.ld) return;
    double *dst = A.base + (size_t)m * A.stride + (size_t)(n + row) * A.ld;
    if (i >= n) { dst[i] = 0.0; return; }
    if (row == 0) { dst[i] = fm[(size_t)m * n + i]; return; }
    const double *h = hyp + (size_t)m * P;
    const int j = row - 1;
    double s = 0.0;
    for (int d = 0; d < D; ++d) {
        const double ell = exp(log(h[n_ell == 1 ? 0 : d]));
        const double df = cov_u<CF>(x[(size_t)i * D + d], ell) - cov_u<CF>(xs[(size_t)j * D + d], ell);
        s = __dadd_rn(s, __dmul_rn(df, df));
    }
    const double sf2 = exp(2.0 * log(h[n_ell]));
    const double snl = exp(log(h[n_ell + 1]));
    const double sW = 1.0 / sqrt(snl * snl);          // sliceSample.py:259
    dst[i] = sW * cov_k<CF>(sf2, s);              // np.tile(sW, (1, ns)) * Ks, :269
}

// fmu[item][j] = sW * (V_j . z0),  fs2[item][j] = kss - V_j . V_j   (rows n and n + 1 + j of the factored slot)
__global__ void __launch_bounds__(128)
pred_reduce_kernel(BatchView A, int n, int M, const double *__restrict__ hyp, int P, int n_ell, const int *__restrict__ info,
                   double *__restrict__ fmu, double *__restrict__ fs2)
{
    const int b = blockIdx.y;
    if (A.count && b >= *A.count) return;
    const int m = batch_item(A, b);
    const int j = blockIdx.x;
    __shared__ double r0[4], r1[4];
    if (info && info[m] != 0) {
        if (threadIdx.x == 0) { fmu[(size_t)m * M + j] = nan(""); fs2[(size_t)m * M + j] = nan(""); }
        return;
    }
    const double *z0 = A.base + (size_t)m * A.stride + (size_t)n * A.ld;
    const double *v = z0 + (size_t)(1 + j) * A.ld;
    double a = 0.0, q = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double vi = v[i];
        a = fma(vi, z0[i], a);
        q = fma(vi, vi, q);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); q += __shfl_xor_sync(0xffffffffu, q, o); }
    if ((threadIdx.x & 31) == 0) { r0[threadIdx.x >> 5] = a; r1[threadIdx.x >> 5] = q; }
    __syncthreads();
    if (threadIdx.x == 0) {
        const double *h = hyp + (size_t)m * P;
        const double sf2 = exp(2.0 * log(h[n_ell]));                  // kss: getCovMatrix(z=xs, mode='self_test'), :262
        const double snl = exp(log(h[n_ell + 1]));
        const double sW = 1.0 / sqrt(snl * snl);
        fmu[(size_t)m * M + j] = sW * (r0[0] + r0[1] + r0[2] + r0[3]);
        fs2[(size_t)m * M + j] = sf2 - (r1[0] + r1[1] + r1[2] + r1[3]);
    }
}

struct PredLayout { int ld; size_t mat_elems, per_item_bytes, fixed_bytes; };
static PredLayout pred_layout(int N, int M, int B)
{
    PredLayout l;
    l.ld = ld_for(N);
    l.mat_elems = (size_t)(N + 1 + M) * l.ld;
    l.per_item_bytes = l.mat_elems * sizeof(double) + (size_t)NB * NB * sizeof(double);
    l.fixed_bytes = align_up((size_t)B * sizeof(double), 256) + align_up((size_t)B * sizeof(int), 256) + 256;
    return l;
}

// ------------------------------------------------------------------------------------ elliptical slice sampling
__device__ __forceinline__ void ess_philox(unsigned long long seed, unsigned c0, unsigned c1, unsigned c2, unsigned c3, double &u0, double &u1)
{
    // Philox4x32-10 (same generator as sds.cu; its own stream ids)
    unsigned k0 = (unsigned)seed, k1 = (unsigned)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned long long p0 = 0xD2511F53ull * c0, p1 = 0xCD9E8D57ull * c2;
        const unsigned h0 = (unsigned)(p0 >> 32), l0 = (unsigned)p0, h1 = (unsigned)(p1 >> 32), l1 = (unsigned)p1;
        c0 = h1 ^ c1 ^ k0; c1 = l1; c2 = h0 ^ c3 ^ k1; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    const unsigned long long a = ((unsigned long long)c0 << 32 | c1) >> 11, b = ((unsigned long long)c2 << 32 | c3) >> 11;
    u0 = ((double)a + 0.5) * (1.0 / 9007199254740992.0);
    u1 = ((double)b + 0.5) * (1.0 / 9007199254740992.0);
}
enum { ESS_STREAM_Z = 8, ESS_STREAM_U = 9 };

// z for the draw nu = chol(K) z  (tape or Philox Box-Muller), written with row stride ldv
__global__ void __launch_bounds__(256)
ess_z_kernel(int n, int ldv, const double *__restrict__ tape_z, unsigned long long seed, unsigned chain0, unsigned sweep, double *__restrict__ z)
{
    const int c = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ldv) return;
    double v = 0.0;
    if (i < n) {
        if (tape_z) v = tape_z[(size_t)c * n + i];
        else {
            double u0, u1;
            ess_philox(seed, chain0 + c, sweep, ESS_STREAM_Z, i >> 1, u0, u1);
            const double rad = sqrt(-2.0 * log(u0));
            v = (i & 1) ? rad * sin(6.283185307179586 * u1) : rad * cos(6.283185307179586 * u1);
        }
    }
    z[(size_t)c * ldv + i] = v;
}

// The slice loop of one chain (sliceSample.py:50-74), one CTA:
//   cur = llk(f) + log(u)                                   :50-51
//   theta = 2 pi u';  [theta_min, theta_max] = [theta - 2 pi, theta]   :54-56
//   loop: f' = f cos(theta) + nu sin(theta); accept if llk(f') > cur and finite; else shrink towards 0 and redraw  :59-74
__global__ void __launch_bounds__(256)
ess_loop_kernel(int n, int ldnu, const double *__restrict__ y, double my, double lower, double upper, double *__restrict__ F,
                const double *__restrict__ nu, const double *__restrict__ hyp, int P, const int *__restrict__ info,
                const double *__restrict__ tape_u, const double *__restrict__ tape_theta, int tape_trips, int max_trips,
                unsigned long long seed, unsigned chain0, unsigned sweep, int *__restrict__ ntrips, int *__restrict__ status)
{
    const int c = blockIdx.x;
    extern __shared__ double sm[];
    double *sf = sm, *snu = sm + n, *sp = sm + 2 * n;     // f, nu, f'
    __shared__ double red[8];
    const double sn = exp(log(hyp[(size_t)c * P + P - 1]));                // TruncatedGauss2(log_sigma=np.log(hyp[2])), :47
    double *f = F + (size_t)c * n;
    if (info && info[c] != 0) {                         // chol(K) failed even with jitter: the reference raises LinAlgError
        if (threadIdx.x == 0) { if (ntrips) ntrips[c] = 0; if (status) status[c] = 2; }
        return;
    }
    for (int i = threadIdx.x; i < n; i += blockDim.x) { sf[i] = f[i]; snu[i] = nu[(size_t)c * ldnu + i]; }
    __syncthreads();
    double u, theta_u, dummy;
    if (tape_u) u = tape_u[c]; else ess_philox(seed, chain0 + c, sweep, ESS_STREAM_U, 0, u, dummy);
    if (tape_theta) theta_u = tape_theta[(size_t)c * tape_trips]; else ess_philox(seed, chain0 + c, sweep, ESS_STREAM_U, 1, theta_u, dummy);
    const double cur = tg2_loglik_block(y, my, sf, n, sn, lower, upper, red) + log(u);        // :50-51
    double theta = 0.0 + (2.0 * 3.141592653589793 - 0.0) * theta_u;                           // np.random.uniform(high=2*pi), :54
    double theta_min = theta - 2.0 * 3.141592653589793, theta_max = theta;                    // :55-56
    const int budget = tape_theta ? min(max_trips, tape_trips) : max_trips;
    for (int trip = 1; trip <= budget; ++trip) {
        const double ct = cos(theta), st = sin(theta);
        for (int i = threadIdx.x; i < n; i += blockDim.x) sp[i] = sf[i] * ct + snu[i] * st;    // :60
        __syncthreads();
        const double llk = tg2_loglik_block(y, my, sp, n, sn, lower, upper, red);              // :62
        if (llk > cur && isfinite(llk)) {                                                      // :64
            for (int i = threadIdx.x; i < n; i += blockDim.x) f[i] = sp[i];
            if (threadIdx.x == 0) { if (ntrips) ntrips[c] = trip; if (status) status[c] = 0; }
            return;
        }
        if (theta >= 0.0) theta_max = theta; else theta_min = theta;                           // :69-72
        if (trip == budget) break;
        double t;
        if (tape_theta) t = tape_theta[(size_t)c * tape_trips + trip]; else ess_philox(seed, chain0 + c, sweep, ESS_STREAM_U, 1 + trip, t, dummy);
        theta = theta_min + (theta_max - theta_min) * t;                                       // :74
        __syncthreads();
    }
    if (threadIdx.x == 0) { if (ntrips) ntrips[c] = budget; if (status) status[c] = 1; }       // budget used up: state kept
}

}  // namespace gpmc

using namespace gpmc;

extern "C" {

size_t gpmc_predict_workspace_bytes(int N, int M, int S)
{
    if (N <= 0 || M <= 0 || S <= 0) return 0;
    const PredLayout l = pred_layout(N, M, S);
    return l.fixed_bytes + (size_t)S * l.per_item_bytes;
}

int gpmc_predict_batched(const double *x_dev, int N, int D, const double *xs_dev, int M, const double *fm_dev, const double *hyp_dev,
                         int S, int P, int kind, int jitter_policy, double *fmu_dev, double *fs2_dev, int *info_dev,
                         void *ws_dev, size_t ws_bytes, void *stream)
{
    GPMC_API_LOCK();
    cudaStream_t s = (cudaStream_t)stream;
    const int n_ell = kind_n_ell(kind, D);
    if (N <= 0 || D <= 0 || D > MAX_ELL || M <= 0 || S < 0 || P != n_ell + 2 || kind_cf(kind) < 0) {
        set_error("predict: bad shape N=%d D=%d M=%d S=%d P=%d kind=%d", N, D, M, S, P, kind);
        return GPMC_EINVAL;
    }
    if (S == 0) return 0;
    if (M + 1 > 65535) { set_error("predict: at most 65534 test points per call"); return GPMC_EINVAL; }
    const PredLayout l = pred_layout(N, M, S);
    if (!ws_dev || ws_bytes < l.fixed_bytes + l.per_item_bytes) {
        set_error("predict: workspace %zu bytes cannot hold one sample (%zu needed)", ws_bytes, l.fixed_bytes + l.per_item_bytes);
        return GPMC_ENOMEM;
    }
    char *wp = (char *)ws_dev;
    double *jit_dev = (double *)wp; wp += align_up((size_t)S * sizeof(double), 256);
    int *map_dev = (int *)wp; wp += align_up((size_t)S * sizeof(int), 256);
    wp += 256;
    const int wave = (int)std::min<size_t>(std::min<size_t>((ws_bytes - l.fixed_bytes) / l.per_item_bytes, (size_t)MAX_BATCH_ITEMS), (size_t)S);
    double *mats = (double *)wp;
    double *W = (double *)(wp + (size_t)wave * l.mat_elems * sizeof(double));
    int rc;
    if ((rc = fill_int(info_dev, 0, S, s))) return rc;
    for (int s0 = 0; s0 < S; s0 += wave) {
        const int nb = std::min(wave, S - s0);
        const double *hyp_w = hyp_dev + (size_t)s0 * P;
        const double *fm_w = fm_dev + (size_t)s0 * N;
        int *info_w = info_dev + s0;
        BatchView A{mats, (long long)l.mat_elems, l.ld, nullptr, nullptr};
        auto fill = [&](BatchView V, int nitems, const double *jit) -> int {
            int r = launch_cov_assemble(x_dev, N, D, hyp_w, P, kind, GPMC_ASM_PRED | GPMC_ASM_LOWER_ONLY, jit, V, nitems, s);
            if (r) return r;
            prof_begin(KC_VEC, s);
            const dim3 grid((l.ld + 255) / 256, 1 + M, nitems);
            switch (kind_cf(kind)) {
                case 1: pred_border_kernel<1><<<grid, 256, 0, s>>>(V, N, D, M, x_dev, xs_dev, hyp_w, P, n_ell, fm_w); break;
                case 3: pred_border_kernel<3><<<grid, 256, 0, s>>>(V, N, D, M, x_dev, xs_dev, hyp_w, P, n_ell, fm_w); break;
                case 5: pred_border_kernel<5><<<grid, 256, 0, s>>>(V, N, D, M, x_dev, xs_dev, hyp_w, P, n_ell, fm_w); break;
                default: pred_border_kernel<0><<<grid, 256, 0, s>>>(V, N, D, M, x_dev, xs_dev, hyp_w, P, n_ell, fm_w); break;
            }
            prof_end(KC_VEC, s);
            GPMC_LAUNCH_CHECK();
            return 0;
        };
        auto diag = [&](const double *h) {            // diag(K / sn2 + I) = sf2 / sn2 + 1
            const double sf2 = exp(2.0 * log(h[n_ell])), snl = exp(log(h[n_ell + 1]));
            return sf2 / (snl * snl) + 1.0;
        };
        if ((rc = factor_wave(fill, diag, A, N, nb, hyp_w, P, info_w, W, jit_dev, map_dev, jitter_policy, 1 + M, s))) return rc;
        prof_begin(KC_SOLVE, s);
        pred_reduce_kernel<<<dim3(M, nb), 128, 0, s>>>(A, N, M, hyp_w, P, n_ell, info_w, fmu_dev + (size_t)s0 * M, fs2_dev + (size_t)s0 * M);
        prof_end(KC_SOLVE, s);
        GPMC_LAUNCH_CHECK();
    }
    return 0;
}

size_t gpmc_ess_workspace_bytes(int N, int B)
{
    if (N <= 0 || B <= 0) return 0;
    const size_t ld = ld_for(N);
    return align_up((size_t)B * sizeof(double), 256) + align_up((size_t)B * sizeof(int), 256) + 256
           + (size_t)B * ((size_t)N * ld * 8 + (size_t)NB * NB * 8 + 2 * ld * 8 + 256);
}

int gpmc_ess_sweep(const double *x_dev, const double *y_dev, int N, int D, double *F_dev, const double *hyp_dev, int B, int P, int kind,
                   double my, double lower, double upper, unsigned long long seed, unsigned chain0, int iter,
                   const double *tape_nu, const double *tape_z, const double *tape_u, const double *tape_theta, int tape_trips,
                   int max_trips, int jitter_policy, int *ntrips_dev, int *status_dev, int *info_dev,
                   void *ws_dev, size_t ws_bytes, void *stream)
{
    GPMC_API_LOCK();
    cudaStream_t s = (cudaStream_t)stream;
    const int n_ell = kind_n_ell(kind, D);
    if (N <= 0 || D <= 0 || D > MAX_ELL || B < 0 || P != n_ell + 2 || kind_cf(kind) < 0 || max_trips <= 0 || (tape_theta && tape_trips < 1)) {
        set_error("ess_sweep: bad shape N=%d D=%d B=%d P=%d kind=%d max_trips=%d", N, D, B, P, kind, max_trips);
        return GPMC_EINVAL;
    }
    if (B == 0) return 0;
    if (B > MAX_BATCH_ITEMS) { set_error("ess_sweep: B=%d exceeds %d chains per call", B, MAX_BATCH_ITEMS); return GPMC_EINVAL; }
    if ((size_t)3 * N * 8 > 200 * 1024) { set_error("ess_sweep: N=%d too large for the one-CTA slice loop", N); return GPMC_EINVAL; }
    const int ld = ld_for(N);
    int rc;
    if ((rc = fill_int(info_dev, 0, B, s))) return rc;
    const double *nu = tape_nu;
    int ldnu = N;
    if (!tape_nu) {
        if (!ws_dev || ws_bytes < gpmc_ess_workspace_bytes(N, B)) { set_error("ess_sweep: workspace too small"); return GPMC_ENOMEM; }
        char *wp = (char *)ws_dev;
        double *jit_dev = (double *)wp; wp += align_up((size_t)B * sizeof(double), 256);
        int *map_dev = (int *)wp; wp += align_up((size_t)B * sizeof(int), 256);
        wp += 256;
        double *mats = (double *)wp; wp += (size_t)B * N * ld * 8;
        double *W = (double *)wp; wp += (size_t)B * NB * NB * 8;
        double *z = (double *)wp; wp += (size_t)B * ld * 8;
        double *nuv = (double *)wp;
        BatchView A{mats, (long long)N * ld, ld, nullptr, nullptr};
        if (ld != N) GPMC_CUDA_CHECK(cudaMemset2DAsync(mats + N, (size_t)ld * 8, 0, (size_t)(ld - N) * 8, (size_t)N * B, s));
        // K = covK.RBF(...).getCovMatrix(x, 'train') (:38-39), L = jitchol(K), nu = L z
        auto fill = [&](BatchView V, int nitems, const double *jit) -> int {
            return launch_cov_assemble(x_dev, N, D, hyp_dev, P, kind, GPMC_ASM_LOWER_ONLY, jit, V, nitems, s);
        };
        auto diag = [&](const double *h) { return exp(2.0 * log(h[n_ell])); };
        if ((rc = factor_wave(fill, diag, A, N, B, hyp_dev, P, info_dev, W, jit_dev, map_dev, jitter_policy, 0, s))) return rc;
        ess_z_kernel<<<dim3((ld + 255) / 256, B), 256, 0, s>>>(N, ld, tape_z, seed, chain0, (unsigned)iter, z);
        GPMC_LAUNCH_CHECK();
        if ((rc = launch_trmv(A, N, 0, 2, z, nullptr, nullptr, ld, nuv, B, s))) return rc;
        nu = nuv;
        ldnu = ld;
    }
    static DeviceOnce attr_set;
    if (attr_set.first()) GPMC_CUDA_CHECK(cudaFuncSetAttribute(ess_loop_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    prof_begin(KC_VEC, s);
    ess_loop_kernel<<<B, 256, (size_t)3 * N * 8, s>>>(N, ldnu, y_dev, my, lower, upper, F_dev, nu, hyp_dev, P, info_dev, tape_u, tape_theta,
                                                       tape_trips, max_trips, seed, chain0, (unsigned)iter, ntrips_dev, status_dev);
    prof_end(KC_VEC, s);
    GPMC_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"
