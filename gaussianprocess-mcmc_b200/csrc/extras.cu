// Kernels of the "next" rows around the hot path (SURVEY 8f): rectangular cross-covariance for prediction
// (covK.RBF.getCovMatrix(x=, z=, mode='cross'), sliceSample.py:263) and the stand-alone truncated-Gaussian
// log-likelihood (likK.TruncatedGauss2.evaluate(y=, mu=), sliceSample.py:50,62,118,143).
#include "common.cuh"
#include "tg2.cuh"
#include "../../include/gpmc.h"

namespace gpmc {

// K[i][j] = cov_k(sf2, sum_d (u(x_id) - u(z_jd))^2) (SE: sf2 * exp(-0.5 * sum_d ((x_id - z_jd)/ell_d)^2)), x[N,D], z[M,D],
// out[N][ld]; one hyper-parameter row.
template <int CF>
__global__ void __launch_bounds__(256)
cov_cross_kernel(const double *__restrict__ x, const double *__restrict__ z, int N, int M, int D,
                 const double *__restrict__ hyp, int n_ell, double *__restrict__ out, int ld)
{
    __shared__ double s_ell[MAX_ELL];
    __shared__ double s_sf2;
    if (threadIdx.x < n_ell) s_ell[threadIdx.x] = exp(log(hyp[threadIdx.x]));
    if (threadIdx.x == 32) s_sf2 = exp(2.0 * log(hyp[n_ell]));
    __syncthreads();
    const int i = blockIdx.y;
    const double sf2 = s_sf2;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < M; j += gridDim.x * blockDim.x) {
        double s = 0.0;
        for (int d = 0; d < D; ++d) {
            const double ell = s_ell[n_ell == 1 ? 0 : d];
            const double df = cov_u<CF>(x[(size_t)i * D + d], ell) - cov_u<CF>(z[(size_t)j * D + d], ell);
            s = __dadd_rn(s, __dmul_rn(df, df));
        }
        out[(size_t)i * ld + j] = cov_k<CF>(sf2, s);
    }
}

__global__ void __launch_bounds__(256)
tg2_loglik_kernel(const double *__restrict__ y, double my, const double *__restrict__ mu, int ldmu, int n,
                  const double *__restrict__ sn, double lower, double upper, double *__restrict__ out)
{
    __shared__ double red[8];
    const int b = blockIdx.x;
    const double v = tg2_loglik_block(y, my, mu + (size_t)b * ldmu, n, sn[b], lower, upper, red);
    if (threadIdx.x == 0) out[b] = v;
}

}  // namespace gpmc

using namespace gpmc;

extern "C" {

int gpmc_cov_cross(const double *x_dev, int N, const double *z_dev, int M, int D, const double *hyp_dev, int P, int kind,
                   double *out_dev, int ld, void *stream)
{
    GPMC_API_LOCK();
    const int n_ell = kind_n_ell(kind, D);
    if (N <= 0 || M <= 0 || D <= 0 || D > MAX_ELL || P != n_ell + 2 || kind_cf(kind) < 0 || ld < M) {
        set_error("cov_cross: bad shape N=%d M=%d D=%d P=%d kind=%d ld=%d", N, M, D, P, kind, ld);
        return GPMC_EINVAL;
    }
    dim3 grid((M + 255) / 256 > 64 ? 64 : (M + 255) / 256, N);
    cudaStream_t s = (cudaStream_t)stream;
    switch (kind_cf(kind)) {
        case 1: cov_cross_kernel<1><<<grid, 256, 0, s>>>(x_dev, z_dev, N, M, D, hyp_dev, n_ell, out_dev, ld); break;
        case 3: cov_cross_kernel<3><<<grid, 256, 0, s>>>(x_dev, z_dev, N, M, D, hyp_dev, n_ell, out_dev, ld); break;
        case 5: cov_cross_kernel<5><<<grid, 256, 0, s>>>(x_dev, z_dev, N, M, D, hyp_dev, n_ell, out_dev, ld); break;
        default: cov_cross_kernel<0><<<grid, 256, 0, s>>>(x_dev, z_dev, N, M, D, hyp_dev, n_ell, out_dev, ld); break;
    }
    GPMC_LAUNCH_CHECK();
    return 0;
}

int gpmc_tg2_loglik(const double *y_dev, double my, const double *mu_dev, int ldmu, int N, int B, const double *sn_dev,
                    double lower, double upper, double *out_dev, void *stream)
{
    GPMC_API_LOCK();
    if (N <= 0 || B < 0 || ldmu < N) { set_error("tg2_loglik: bad shape N=%d B=%d ldmu=%d", N, B, ldmu); return GPMC_EINVAL; }
    if (B == 0) return 0;
    tg2_loglik_kernel<<<B, 256, 0, (cudaStream_t)stream>>>(y_dev, my, mu_dev, ldmu, N, sn_dev, lower, upper, out_dev);
    GPMC_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"
