// gpmc_loglik_grad_batched: the log-lik unit and its gradient with respect to the hyper-parameters (include/gpmc.h).
//
// Per wave of items:
//     K+S (lower), g as border row N    cov_assemble (+ band bound)                      as gpmc_loglik_batched's dense path
//     L = chol(K+S), z = L^-1 g          factor_wave (jitter ladder), every diagonal-block inverse kept
//     loglik                             border_finish
//     U = L^-T                           inverse_sequence
//     alpha = U z = A^-1 g               trmv (upper)
//     W = U U^T = A^-1, lower tiles      DMMA tile kernel, EPI_SET; with the band only the tiles that can meet K_ij != 0
//     grad                               grad_contract.cu (one pass over those tiles of W, K_ij recomputed)
// The factor is held densely (no compact band layout): U = L^-T fills the upper triangle.  Cost per item: N^3/3 flop for
// the inverse, about N^2 w / 2 for the banded W (w = band width), the banded Cholesky and an O(N w P) contraction.
#include "common.cuh"
#include "sequences.cuh"
#include "../../include/gpmc.h"

#include <algorithm>
#include <vector>

namespace gpmc {

struct GradLayout {
    int ld, nt, nblk;
    size_t mat_elems;        // per item: N + 1 rows (the border row carries g)
    size_t fixed_bytes;      // per call
    size_t per_item_bytes;   // factor + W + saved inverses + z, alpha + envelope, band + partials
};
static GradLayout grad_layout(int N, int P, int B)
{
    GradLayout l;
    l.ld = ld_for(N);
    l.nt = (N + NB - 1) / NB;
    l.nblk = env_blocks(N);
    l.mat_elems = (size_t)(N + 1) * l.ld;
    l.per_item_bytes = (l.mat_elems + (size_t)N * l.ld + (size_t)l.nt * NB * NB + 2 * (size_t)l.ld) * sizeof(double)
                       + align_up(2 * (size_t)l.nblk * sizeof(int), 8) + (size_t)l.nblk * P * sizeof(double);
    l.fixed_bytes = align_up((size_t)B * sizeof(double), 256)      // jitter
                    + align_up((size_t)B * sizeof(int), 256)       // map
                    + 256                                          // band bound maxima
                    + align_up((size_t)32 * l.ld * sizeof(double), 256)   // boxes of x for the band bound
                    + 8 * 256;                                     // alignment of the per-wave arrays
    return l;
}

size_t loglik_grad_workspace_bytes(int N, int D, int B)
{
    const GradLayout l = grad_layout(N, D + 2, B);
    // as GPMC_OP_LOGLIK: as many items per wave as fit in 48 GiB, at most 8192
    const size_t cap = (size_t)48 << 30;
    const size_t wave = std::min<size_t>(std::min<size_t>(B, 8192), std::max<size_t>(1, cap / l.per_item_bytes));
    return l.fixed_bytes + wave * l.per_item_bytes;
}

// diag(K+S) of an item from its hyper-parameter row (sliceSample.py:185-190 expression order), to size the ladder's jitter
static double diag_value(const double *h, int n_ell)
{
    const double sf = h[n_ell], sn = h[n_ell + 1];
    const double sf2 = exp(2.0 * log(sf));
    const double kinv = 1.0 / sf2;
    double Sii = 1.0 / ((1.0 / (sn * sn) + kinv) - kinv);
    if (Sii < 0.0) Sii = 0.0;
    return sf2 + Sii;
}

// W = U U^T into Wm, lower tiles.  width >= 0: the band bound's widest band of the wave, in 64-column tiles: each 128-row
// block row R launches only the columns from 64 max(0, 2R - width) on.  Every tile is computed exactly as in the full
// lower-triangle launch (same contraction start, k = its first row, same order), so the two agree bit for bit.
static int w_sequence(BatchView Wm, BatchView U, int n, int B, int width, cudaStream_t s)
{
    GemmArgs g{};
    g.C = Wm; g.A = Operand{U.base, U.stride, U.ld}; g.B = g.A;
    g.k0 = 0; g.bk0 = 0; g.klen = n;
    g.k_follow_row = 1;                                 // U is upper triangular: row i is zero left of column i
    g.epi = EPI_SET;
    g.skip_upper = 1;                                   // the contraction reads the lower triangle only
    const int nrb = (n + NB - 1) / NB;
    if (width < 0 || 2 * (nrb - 1) - width <= 0) {
        g.cr0 = 0; g.cc0 = 0; g.rows = n; g.cols = n;
        g.ar0 = 0; g.br0 = 0;
        g.lower_only = 1;
        return launch_gemm(g, B, KC_SYRK_R, s);
    }
    for (int R = 0; R < nrb; ++R) {
        const int r0 = R * NB, c0 = std::max(0, 2 * R - width) * ENV_ROWS;
        g.cr0 = r0; g.ar0 = r0; g.rows = std::min(NB, n - r0);
        g.cc0 = c0; g.br0 = c0; g.cols = std::min(n, r0 + NB) - c0;
        int rc = launch_gemm(g, B, KC_SYRK_R, s);
        if (rc) return rc;
    }
    return 0;
}

}  // namespace gpmc

using namespace gpmc;

extern "C" int gpmc_loglik_grad_batched(const double *x_dev, int N, int D, const double *g_dev, const double *hyp_dev, int B,
                                        int P, int kind, int jitter_policy, double *loglik_dev, double *grad_dev, int *info_dev,
                                        void *ws_dev, size_t ws_bytes, void *stream)
{
    GPMC_API_LOCK();
    cudaStream_t s = (cudaStream_t)stream;
    const int n_ell = (kind == GPMC_KIND_SE_ARD) ? D : 1;
    if (N <= 0 || D <= 0 || B < 0 || (kind != GPMC_KIND_SE_ISO && kind != GPMC_KIND_SE_ARD) || P != n_ell + 2) {
        set_error("loglik_grad: bad shape N=%d D=%d B=%d P=%d kind=%d", N, D, B, P, kind);
        return GPMC_EINVAL;
    }
    if (D > MAX_ELL) { set_error("loglik_grad: D=%d exceeds MAX_ELL=%d", D, MAX_ELL); return GPMC_EINVAL; }
    if (B == 0) return 0;
    if (!x_dev || !g_dev || !hyp_dev || !loglik_dev || !grad_dev || !info_dev) { set_error("loglik_grad: null buffer"); return GPMC_EINVAL; }
    const GradLayout l = grad_layout(N, P, B);
    if (!ws_dev || ws_bytes < l.fixed_bytes + l.per_item_bytes) {
        set_error("loglik_grad: workspace %zu bytes cannot hold one item (%zu needed)", ws_bytes, l.fixed_bytes + l.per_item_bytes);
        return GPMC_ENOMEM;
    }
    const int wave = (int)std::min<size_t>(std::min<size_t>((ws_bytes - l.fixed_bytes) / l.per_item_bytes, (size_t)MAX_BATCH_ITEMS), (size_t)B);
    char *wp = (char *)ws_dev;
    auto carve = [&](size_t bytes) { char *r = wp; wp += align_up(bytes, 256); return r; };
    double *jit_dev = (double *)carve((size_t)B * sizeof(double));
    int *map_dev = (int *)carve((size_t)B * sizeof(int));
    int *band_dev = (int *)carve(2 * sizeof(int));
    double *xbox = (double *)carve((size_t)32 * l.ld * sizeof(double));
    double *mats = (double *)carve((size_t)wave * l.mat_elems * sizeof(double));
    double *Wm = (double *)carve((size_t)wave * N * l.ld * sizeof(double));
    double *Wsave = (double *)carve((size_t)wave * l.nt * NB * NB * sizeof(double));
    double *zv = (double *)carve((size_t)wave * l.ld * sizeof(double));
    double *av = (double *)carve((size_t)wave * l.ld * sizeof(double));
    double *partial = (double *)carve((size_t)wave * l.nblk * P * sizeof(double));
    int *env_blk = (int *)carve((size_t)wave * l.nblk * sizeof(int));
    int *band_w = (int *)wp;                            // wave * nblk ints: the last array, inside the per-item bytes
    const long long strideWsave = (long long)l.nt * NB * NB;

    { int rc0 = fill_int(info_dev, 0, B, s); if (rc0) return rc0; }
    // pad columns of the factor are contracted over by the DMMA kernels (multiples of 16 columns): zero once per call
    if (l.ld != N) GPMC_CUDA_CHECK(cudaMemset2DAsync(mats + N, (size_t)l.ld * 8, 0, (size_t)(l.ld - N) * 8, (size_t)(N + 1) * wave, s));

    const bool band_on = envelope_enabled() && band_enabled();
    for (int s0 = 0; s0 < B; s0 += wave) {
        const int nb = std::min(wave, B - s0);
        const double *hyp_w = hyp_dev + (size_t)s0 * P;
        const double *g_w = g_dev + (size_t)s0 * N;
        int *info_w = info_dev + s0;
        BatchView A{mats, (long long)l.mat_elems, l.ld, nullptr, nullptr};
        const int fuse = potrf_fuse_auto(N, nb, 1);
        // the dense path of gpmc_loglik_batched: envelope skips unless the fused panel launches run; with the band, only
        // the band is assembled and +0 is stored left of it in the same launch (inverse_sequence reads those zeros)
        Envelope env = (envelope_enabled() && !fuse) ? Envelope{env_blk, l.nblk, N} : Envelope{};
        Band band{};
        int width = -1;
        if (band_on) {
            GPMC_CUDA_CHECK(cudaMemsetAsync(band_dev, 0, 2 * sizeof(int), s));
            int rc = launch_band_bound(x_dev, N, D, hyp_w, P, n_ell, nb, band_w, l.nblk, band_dev, xbox, s);
            if (rc) return rc;
            int bh[2] = {0, 0};
            GPMC_CUDA_CHECK(cudaMemcpyAsync(bh, band_dev, sizeof(bh), cudaMemcpyDeviceToHost, s));
            GPMC_CUDA_CHECK(cudaStreamSynchronize(s));
            width = bh[1];
            if (env.blk) {
                env.band = bh[0];
                band = Band{band_w, l.nblk, bh[1], 1};
            }
        }
        auto fill = [&](BatchView V, int nitems, const double *jit) -> int {
            int rc = launch_cov_assemble(x_dev, N, D, hyp_w, P, n_ell, GPMC_ASM_ADD_S | GPMC_ASM_LOWER_ONLY, jit, V, nitems, s, env, band);
            if (rc) return rc;
            return border_set(V, N, g_w, N, nitems, s);
        };
        auto diag = [&](const double *h) { return diag_value(h, n_ell); };
        int rc = factor_wave(fill, diag, A, N, nb, hyp_w, P, info_w, Wsave, jit_dev, map_dev, jitter_policy, 1, s, fuse, env, NB * NB);
        if (rc) return rc;
        if ((rc = border_finish(A, N, loglik_dev + s0, info_w, nb, s, fuse))) return rc;
        if ((rc = border_get(A, N, zv, l.ld, info_w, nb, s))) return rc;
        if ((rc = inverse_sequence(A, N, nb, Wsave, strideWsave, s))) return rc;
        if ((rc = launch_trmv(A, N, 1, 2, zv, nullptr, nullptr, l.ld, av, nb, s))) return rc;
        BatchView Wv{Wm, (long long)N * l.ld, l.ld, nullptr, nullptr};
        if ((rc = w_sequence(Wv, A, N, nb, width, s))) return rc;
        if ((rc = launch_grad_contract(x_dev, N, D, hyp_w, P, n_ell, av, l.ld, Wm, l.ld, (long long)N * l.ld,
                                       band_on ? band_w : nullptr, l.nblk, info_w, partial, grad_dev + (size_t)s0 * P, nb, s)))
            return rc;
    }
    return 0;
}
