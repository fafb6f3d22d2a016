// Device helpers shared by the two hyper-parameter slice samplers (sds.cu, marginal.cu): the Philox stream both key by
// (seed, global chain id, iteration), the hyper-priors of sliceSample.py:209-232 and the density sum of :127-129,150-152.
#pragma once
#include "common.cuh"

namespace gpmc {

// ------------------------------------------------------------------------------------- Philox4x32-10
static __device__ __forceinline__ void philox_round(unsigned &c0, unsigned &c1, unsigned &c2, unsigned &c3, unsigned k0, unsigned k1)
{
    const unsigned long long p0 = 0xD2511F53ull * c0, p1 = 0xCD9E8D57ull * c2;
    const unsigned h0 = (unsigned)(p0 >> 32), l0 = (unsigned)p0, h1 = (unsigned)(p1 >> 32), l1 = (unsigned)p1;
    c0 = h1 ^ c1 ^ k0; c1 = l1; c2 = h0 ^ c3 ^ k1; c3 = l0;
}
static __device__ void philox4x32(unsigned long long seed, unsigned c0, unsigned c1, unsigned c2, unsigned c3, unsigned out[4])
{
    unsigned k0 = (unsigned)seed, k1 = (unsigned)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        philox_round(c0, c1, c2, c3, k0, k1);
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
// two uniforms on (0,1) with 53 random bits each, from one Philox block
static __device__ __forceinline__ void philox_uniform2(unsigned long long seed, unsigned chain, unsigned sweep, unsigned stream,
                                                       unsigned idx, double &u0, double &u1)
{
    unsigned o[4];
    philox4x32(seed, chain, sweep, stream, idx, o);
    const unsigned long long a = ((unsigned long long)o[0] << 32 | o[1]) >> 11;
    const unsigned long long b = ((unsigned long long)o[2] << 32 | o[3]) >> 11;
    u0 = ((double)a + 0.5) * (1.0 / 9007199254740992.0);
    u1 = ((double)b + 0.5) * (1.0 / 9007199254740992.0);
}
enum { STREAM_Z = 0, STREAM_BRACKET = 1, STREAM_TRIP = 2 };

// --------------------------------------------------------------------------------- scalar formulas
// log_gamma (sliceSample.py:209-232): Gamma log-pdf for every entry, inverse-Gamma for the last (noise).
static __device__ double log_prior_entry(double x, double k, double theta, bool inverse_gamma)
{
    if (!inverse_gamma) return (k - 1.0) * log(x) - x / theta - k * log(theta) - log(tgamma(k));       // :224
    return log(pow(theta, k)) - log(tgamma(k)) + (-k - 1.0) * log(x) + (-theta / x);                   // :229
}

// head + prior[sf] + prior[ell_0..] + G (+ prior[sn] once iter >= burn_in): the summation order of :127-129,150-152.
// The surrogate-data sampler passes the reference's burn_in = 500.
static __device__ double density_sum(double head, const double *hyp, const double *pk, const double *pth, int P, double G, int iter,
                                     int burn_in)
{
    const int n_ell = P - 2;
    double acc = head + log_prior_entry(hyp[n_ell], pk[n_ell], pth[n_ell], false);
    for (int d = 0; d < n_ell; ++d) acc = acc + log_prior_entry(hyp[d], pk[d], pth[d], false);
    acc = acc + G;
    if (iter >= burn_in) acc += log_prior_entry(hyp[P - 1], pk[P - 1], pth[P - 1], true);
    return acc;
}

}  // namespace gpmc
