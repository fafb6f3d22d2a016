// Fused covariance assembly: SE (iso / ARD) kernel + S diagonal + jitter + symmetric fill.
//
// Replaces, per batch item, the reference's
//   Kc = covK.RBF(np.log(hyp[0]), np.log(hyp[1])); K = Kc.getCovMatrix(x=x, mode='train')   sliceSample.py:104-105,136-137
//   S_ii = 1/((1/sn^2 + 1/K_ii) - 1/K_ii); S = max(S, 0); K+S                               sliceSample.py:183-190,196
// (pyGPs 1.3.4 cov.RBF: K = sf2 * exp(-0.5 * cdist(x/ell, x/ell, 'sqeuclidean')), ell = exp(log_ell),
//  sf2 = exp(2 log_sigma)); the operation order of those expressions is kept so the matrix matches
//  numpy's to the last bits of exp().
//
// Layout: one CTA = one 64x64 tile on or below the diagonal.  Each lane owns two adjacent columns
// (double2, 16 B stores; a warp writes 512 contiguous bytes of one row), the tile is mirrored
// through shared memory so the transposed tile is written with the same coalesced double2 stores
// and every exp() is evaluated once.  HBM-write bound: 8*N^2 bytes per matrix (8*N*(N+64)/2 with
// GPMC_ASM_LOWER_ONLY).
#include "common.cuh"
#include "../../include/gpmc.h"

#include <algorithm>

namespace gpmc {

constexpr int AT = 64;          // tile edge
constexpr int AT_PAD = 66;      // smem row stride (doubles): keeps double2 stores 16 B aligned
constexpr int ASM_TPC = 1;      // tiles per CTA (4 was measured: N=4096 x 256 4.17 -> 4.69 ms, slower -- the per-CTA scalar prologue is not the limiter)

// lower-triangle tile t -> (tm >= tn), row-major
__device__ __forceinline__ void tile_decode(int t, int &tm, int &tn)
{
    tm = (int)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
    while ((tm + 1) * (tm + 2) / 2 <= t) ++tm;
    while (tm * (tm + 1) / 2 > t) --tm;
    tn = t - tm * (tm + 1) / 2;
}

// DT > 0: input dimension known at compile time (the distance loop unrolls and the column values live in registers);
// DT == 0: generic D.  The kernel is instruction-issue bound (ncu: 79 % issue slots, FP64 pipe 47 %, DRAM 33 %), so the
// fast path strips everything that is not the exp itself: no bounds tests on interior tiles, no diagonal tests off
// the diagonal.
// PRED: the K / sn^2 + I variant of inf_mcmc (GPMC_ASM_PRED) -- a template parameter, not a run-time test: a uniform
// `if (pred)` in the fast path cost the hot (non-PRED) instantiation 20 % (3.5 vs 4.2 TB/s at N=4096, round 2).
template <int DT, bool PRED>
__global__ void __launch_bounds__(256)
cov_assemble_kernel(const double *__restrict__ x, int N, int Drt, const double *__restrict__ hyp, int P, int n_ell,
                    int flags, const double *__restrict__ jitter, BatchView A, Envelope env, Band band)
{
    const int D = DT > 0 ? DT : Drt;
    const int b = blockIdx.y;
    if (A.count && b >= *A.count) return;
    const int m = batch_item(A, b);
    const int nt1 = (N + AT - 1) / AT;
    if (band.w) {
        // band grid: CTA (row block r, slot k) takes tile (r, r - k) and leaves at once when that lies left of the band;
        // inline clear: the triangular grid, tiles left of the band get +0
        static_assert(ASM_TPC == 1, "the band grid maps one tile to a CTA");
        int tm, tn;
        if (band.clear) {
            tile_decode(blockIdx.x, tm, tn);
        } else {
            tm = blockIdx.x / (band.width + 1);
            tn = tm - (blockIdx.x - tm * (band.width + 1));
            if (tn < 0) return;
        }
        if (tn < band.w[(size_t)m * band.ld + tm]) {
            if (!band.clear) return;
            const int cl = 2 * (threadIdx.x & 31);
            const int gc = tn * AT + cl;
            double *dst = A.base + (size_t)m * A.stride + (size_t)(tm * AT + (threadIdx.x >> 5) * 8) * A.ld + gc;
            for (int rr = 0; rr < 8; ++rr) {
                if (tm * AT + (threadIdx.x >> 5) * 8 + rr >= N) break;
                if (gc + 1 < N) *reinterpret_cast<double2 *>(dst + (size_t)rr * A.ld) = make_double2(0.0, 0.0);
                else if (gc < N) dst[(size_t)rr * A.ld] = 0.0;
            }
            return;
        }
    }

    __shared__ double s_ell[MAX_ELL];
    __shared__ double s_ui[MAX_ELL][AT];
    __shared__ double s_uj[MAX_ELL][AT];
    __shared__ __align__(16) double s_tile[AT][AT_PAD];
    __shared__ double s_scal[4];       // sf2, Sii (or 1 with GPMC_ASM_PRED), jitter, sn2 (GPMC_ASM_PRED)

    const double *h = hyp + (size_t)m * P;
    const int tid = threadIdx.x;
    if (tid < n_ell) {
        // covK.RBF(np.log(ll), ...): ell = exp(log(ll))   (log/exp round trip kept)
        s_ell[tid] = exp(log(h[tid]));
    }
    if (tid == 32) {
        const double sf = h[n_ell], sn = h[n_ell + 1];
        const double sf2 = exp(2.0 * log(sf));                 // sf2 = exp(2*log_sigma)
        const double Kii = sf2;                                // sf2 * exp(-0.5*0) == sf2
        // sliceSample.py:185-187,190
        const double K_ii_inv = 1.0 / Kii;
        const double v_1 = 1.0 / (sn * sn) + K_ii_inv;
        double Sii = 1.0 / (v_1 - K_ii_inv);
        Sii = (Sii < 0.0) ? 0.0 : Sii;                         // np.maximum(S, 0) (NaN propagates)
        s_scal[0] = sf2;
        s_scal[1] = (flags & GPMC_ASM_ADD_S) ? Sii : 0.0;
        s_scal[2] = jitter ? jitter[m] : 0.0;
        if (PRED) {
            // inf_mcmc (sliceSample.py:256-257): sn2 = likfunc.sn**2 with likfunc.sn = exp(log_sigma); K/sn2 + eye(n)
            const double snl = exp(log(sn));
            s_scal[3] = snl * snl;
            s_scal[1] = 1.0;
        } else s_scal[3] = 1.0;
    }
    __syncthreads();
    const int warp = tid >> 5, lane = tid & 31;
    const double sf2 = s_scal[0];
    const double diag_add = s_scal[1], jit = s_scal[2], sn2 = s_scal[3];
    constexpr bool pred = PRED;
    const bool has_jit = (jitter != nullptr);
    const int cl = 2 * lane;
    const int ntiles = band.w && !band.clear ? nt1 * (band.width + 1) : nt1 * (nt1 + 1) / 2;
    // A CTA takes ASM_TPC consecutive tiles of its matrix (experiment: amortise the per-item scalars above -- two
    // exp(log(.)) round trips and the S_ii expression on one or two threads while the rest of the CTA waits; ncu r02f shows
    // barrier stalls of 2.6 per issue -- over several tiles.  Measured slower with 4, so the default is 1.)
    for (int tt = 0; tt < ASM_TPC; ++tt) {
    const int t = blockIdx.x * ASM_TPC + tt;
    if (t >= ntiles) break;
    int tm, tn;
    if (band.w && !band.clear) { tm = t / (band.width + 1); tn = tm - (t - tm * (band.width + 1)); }
    else tile_decode(t, tm, tn);
    const int r0 = tm * AT, c0 = tn * AT;
    if (tt > 0) __syncthreads();                 // the previous tile's u vectors / mirrored tile are still being read
    // u = x / ell for the tile's rows and columns
    for (int e = tid; e < 2 * AT * D; e += 256) {
        const int which = e / (AT * D);
        const int rem = e - which * AT * D;
        const int i = rem / D, d = rem - i * D;
        const int gi = (which ? c0 : r0) + i;
        const double ell = s_ell[n_ell == 1 ? 0 : d];
        const double v = (gi < N) ? x[(size_t)gi * D + d] / ell : 0.0;
        if (which) s_uj[d][i] = v; else s_ui[d][i] = v;
    }
    __syncthreads();

    const int gc = c0 + cl;
    // envelope: this thread's first column holding a nonzero in the tile's lower-triangle rows (NaN counts as nonzero)
    bool nz0 = false, nz1 = false;
    const bool mirror = (tm != tn) && !(flags & GPMC_ASM_LOWER_ONLY);

    const bool interior = (r0 + AT <= N) && (c0 + AT <= N) && (tm != tn);
    if (DT > 0 && interior) {
        // fast path: full tile strictly below the diagonal
        double uj0[DT > 0 ? DT : 1], uj1[DT > 0 ? DT : 1];
#pragma unroll
        for (int d = 0; d < DT; ++d) { uj0[d] = s_uj[d][cl]; uj1[d] = s_uj[d][cl + 1]; }
        double *dst = view_elem(A, m, r0 + warp * 8, gc);     // 8 rows of one 64-row block: row stride A.ld
#pragma unroll
        for (int rr = 0; rr < 8; ++rr) {
            const int rl = warp * 8 + rr;
            double s0 = 0.0, s1 = 0.0;
#pragma unroll
            for (int d = 0; d < DT; ++d) {
                const double ui = s_ui[d][rl];
                const double d0 = ui - uj0[d], d1 = ui - uj1[d];
                s0 = __dadd_rn(s0, __dmul_rn(d0, d0));
                s1 = __dadd_rn(s1, __dmul_rn(d1, d1));
            }
            double k0 = sf2 * exp(-0.5 * s0);
            double k1 = sf2 * exp(-0.5 * s1);
            if (pred) { k0 = k0 / sn2; k1 = k1 / sn2; }
            if (mirror) *reinterpret_cast<double2 *>(&s_tile[rl][cl]) = make_double2(k0, k1);
            *reinterpret_cast<double2 *>(dst + (size_t)rr * A.ld) = make_double2(k0, k1);
            nz0 |= (k0 != 0.0);
            nz1 |= (k1 != 0.0);
        }
    } else {
#pragma unroll
    for (int rr = 0; rr < 8; ++rr) {
        const int rl = warp * 8 + rr;
        const int gr = r0 + rl;
        double s0 = 0.0, s1 = 0.0;
        for (int d = 0; d < D; ++d) {
            const double ui = s_ui[d][rl];
            const double d0 = ui - s_uj[d][cl];
            const double d1 = ui - s_uj[d][cl + 1];
            s0 = __dadd_rn(s0, __dmul_rn(d0, d0));            // cdist 'sqeuclidean': s += d*d, no FMA
            s1 = __dadd_rn(s1, __dmul_rn(d1, d1));
        }
        double k0 = sf2 * exp(-0.5 * s0);
        double k1 = sf2 * exp(-0.5 * s1);
        if (pred) { k0 = k0 / sn2; k1 = k1 / sn2; }
        if (gr == gc)     { k0 = k0 + diag_add; if (has_jit) k0 = k0 + jit; }
        if (gr == gc + 1) { k1 = k1 + diag_add; if (has_jit) k1 = k1 + jit; }
        if (mirror) *reinterpret_cast<double2 *>(&s_tile[rl][cl]) = make_double2(k0, k1);
        if (gr < N) {
            double *dst = view_elem(A, m, gr, gc);
            if (gc + 1 < N)      *reinterpret_cast<double2 *>(dst) = make_double2(k0, k1);
            else if (gc < N)     dst[0] = k0;
            nz0 |= (k0 != 0.0 && gc < N && gc <= gr);
            nz1 |= (k1 != 0.0 && gc + 1 < N && gc + 1 <= gr);
        }
    }
    }
    if (env.blk) {
        __shared__ int s_env;
        if (tid == 0) s_env = 0x7fffffff;
        __syncthreads();
        const int first = __reduce_min_sync(0xffffffffu, nz0 ? gc : (nz1 ? gc + 1 : 0x7fffffff));
        if (lane == 0 && first != 0x7fffffff) atomicMin(&s_env, first);
        __syncthreads();
        if (tid == 0 && s_env != 0x7fffffff) atomicMin(env.blk + (size_t)m * env.ld + tm, s_env);
    }
    if (!mirror) continue;
    __syncthreads();
    // mirrored tile: rows c0.., cols r0..
#pragma unroll
    for (int rr = 0; rr < 8; ++rr) {
        const int cm = warp * 8 + rr;            // row of the mirrored tile (a column of this tile)
        const int gr = c0 + cm;
        const int gcol = r0 + cl;
        const double k0 = s_tile[cl][cm];
        const double k1 = s_tile[cl + 1][cm];
        if (gr < N) {
            double *dst = view_elem(A, m, gr, gcol);
            if (gcol + 1 < N)    *reinterpret_cast<double2 *>(dst) = make_double2(k0, k1);
            else if (gcol < N)   dst[0] = k0;
        }
    }
    }
}

// every envelope entry of the items A selects starts as "no nonzero"; the assembly lowers it
__global__ void env_init_kernel(BatchView A, Envelope env)
{
    const int b = blockIdx.x;
    if (A.count && b >= *A.count) return;
    const int m = batch_item(A, b);
    for (int r = threadIdx.x; r < env_blocks(env.n); r += blockDim.x) env.blk[(size_t)m * env.ld + r] = 0x7fffffff;
}

// ---------------------------------------------------------------------------------------------------------- band bound
// Per 64-row block r and input dimension d: min and max of x[rows of r][d] (NaN when one of them is not finite).  Division
// by a positive ell is monotone under round-to-nearest, so min(x) / ell is exactly the min of the x / ell the assembly forms.
__global__ void band_xbox_kernel(const double *__restrict__ x, int N, int D, double *__restrict__ xbox)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= env_blocks(N) * D) return;
    const int r = e / D, d = e - r * D;
    double lo = INFINITY, hi = -INFINITY;
    bool finite = true;
    for (int i = r * AT; i < min(N, r * AT + AT); ++i) {
        const double v = x[(size_t)i * D + d];
        finite = finite && isfinite(v);
        lo = fmin(lo, v);
        hi = fmax(hi, v);
    }
    xbox[2 * e] = finite ? lo : NAN;
    xbox[2 * e + 1] = finite ? hi : NAN;
}

// One CTA per item.  Tile (r, c) is certainly +0 when the squared distance of the two boxes of x / ell, s, satisfies
// 0.5 s > 760 + max(0, ln sf2) (with relative slack): every element's distance is at least s (each difference, square and
// sum rounds monotonically), and exp underflows to +0 below -745.2, so sf2 * exp(-0.5 s) is +0 for all of them.
__global__ void band_bound_kernel(const double *__restrict__ hyp, int P, int n_ell, int N, int D, const double *__restrict__ xbox,
                                  int *__restrict__ w, int ldw, int *__restrict__ band_out)
{
    extern __shared__ int s_lo[];
    __shared__ double s_ell[MAX_ELL];
    __shared__ double s_thr;
    __shared__ int s_max[2];
    const int m = blockIdx.x, tid = threadIdx.x;
    const int nt1 = env_blocks(N);
    const double *h = hyp + (size_t)m * P;
    if (tid < n_ell) s_ell[tid] = exp(log(h[tid]));           // as cov_assemble_kernel forms them
    if (tid == 0) {
        const double sf2 = exp(2.0 * log(h[n_ell]));
        s_thr = (isfinite(sf2) && sf2 > 0.0) ? 760.0 + fmax(0.0, log(sf2)) : NAN;
        s_max[0] = s_max[1] = 0;
    }
    __syncthreads();
    bool dense = !(s_thr == s_thr);
    for (int d = 0; d < n_ell; ++d) dense = dense || !(isfinite(s_ell[d]) && s_ell[d] > 0.0);
    for (int e = tid; e < nt1 * D; e += blockDim.x) dense = dense || !(xbox[2 * e] == xbox[2 * e]);
    dense = __syncthreads_or(dense);
    const double thr = s_thr;
    // a warp per row block, its lanes over 32 column tiles at a time: lo[r] is the first tile that may hold a nonzero
    const int lane = tid & 31, nwarps = blockDim.x >> 5;
    for (int r = tid >> 5; r < nt1; r += nwarps) {
        int lo = r;
        if (dense) lo = 0;
        else
            for (int c0 = 0; c0 < r; c0 += 32) {
                const int c = c0 + lane;
                bool maybe = false;
                if (c < r) {
                    double s = 0.0;
                    for (int d = 0; d < D; ++d) {
                        const double ell = s_ell[n_ell == 1 ? 0 : d];
                        const double rlo = xbox[2 * (r * D + d)] / ell, rhi = xbox[2 * (r * D + d) + 1] / ell;
                        const double clo = xbox[2 * (c * D + d)] / ell, chi = xbox[2 * (c * D + d) + 1] / ell;
                        double g = 0.0;
                        if (rlo - chi > g) g = rlo - chi;
                        if (clo - rhi > g) g = clo - rhi;
                        s = __dadd_rn(s, __dmul_rn(g, g));
                    }
                    maybe = !(0.5 * s * (1.0 - 1e-9) > thr);
                }
                const unsigned hit = __ballot_sync(0xffffffffu, maybe);
                if (hit) { lo = c0 + __ffs(hit) - 1; break; }
            }
        if (lane == 0) s_lo[r] = lo;
    }
    __syncthreads();
    constexpr int WALIGN = NB / ENV_ROWS;
    int mlo = 0, mw = 0;
    for (int r = tid; r < nt1; r += blockDim.x) {
        int v = s_lo[r];
        if (r > 0) v = min(v, s_lo[r - 1]);
        if (r + 1 < nt1) v = min(v, s_lo[r + 1]);
        v = v / WALIGN * WALIGN;
        w[(size_t)m * ldw + r] = v;
        mlo = max(mlo, r - s_lo[r]);
        mw = max(mw, r - v);
    }
    atomicMax(&s_max[0], mlo);
    atomicMax(&s_max[1], mw);
    __syncthreads();
    if (tid == 0) { atomicMax(band_out, s_max[0]); atomicMax(band_out + 1, s_max[1]); }
}

int launch_band_bound(const double *x, int N, int D, const double *hyp, int P, int n_ell, int B, int *w, int ldw,
                      int *band_out, double *xbox, cudaStream_t s)
{
    if (D > MAX_ELL || n_ell > MAX_ELL) { set_error("D=%d exceeds MAX_ELL=%d", D, MAX_ELL); return GPMC_EINVAL; }
    if (B <= 0) return 0;
    const int nt1 = env_blocks(N);
    if ((size_t)nt1 * sizeof(int) > 48 * 1024) { set_error("band bound: N=%d has too many row blocks", N); return GPMC_EINVAL; }
    prof_begin(KC_ASSEMBLE, s);
    band_xbox_kernel<<<(nt1 * D + 127) / 128, 128, 0, s>>>(x, N, D, xbox);
    band_bound_kernel<<<B, 256, nt1 * sizeof(int), s>>>(hyp, P, n_ell, N, D, xbox, w, ldw, band_out);
    prof_end(KC_ASSEMBLE, s);
    GPMC_LAUNCH_CHECK();
    return 0;
}

// One warp per row: +0 into columns 0 .. 64 w[r] - 1.  A few CTAs walk over all rows, so that the stores run beside the
// factorisation without taking many of its SM slots.
__global__ void __launch_bounds__(256) band_clear_kernel(BatchView A, int N, Band band, int B)
{
    const int lane = threadIdx.x & 31;
    const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long gw = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); gw < (long long)B * N; gw += nwarps) {
        const int b = (int)(gw / N), i = (int)(gw - (long long)b * N);
        const int m = batch_item(A, b);
        const int cols = band.w[(size_t)m * band.ld + i / AT] * AT;       // <= 64 (i / 64) <= i < N
        double *row = A.base + (size_t)m * A.stride + (size_t)i * A.ld;
        for (int c = 2 * lane; c < cols; c += 64) *reinterpret_cast<double2 *>(row + c) = make_double2(0.0, 0.0);
    }
}

int launch_band_clear(BatchView A, int N, Band band, int B, cudaStream_t s)
{
    if (B <= 0 || !band.w) return 0;
    if (A.W) { set_error("band clear: the compact layout has no storage left of the band"); return GPMC_EINVAL; }
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
    }
    prof_begin(KC_CLEAR, s);
    band_clear_kernel<<<sms, 256, 0, s>>>(A, N, band, B);
    prof_end(KC_CLEAR, s);
    GPMC_LAUNCH_CHECK();
    return 0;
}

int launch_cov_assemble(const double *x, int N, int D, const double *hyp, int P, int n_ell, int flags,
                        const double *jitter, BatchView A, int B, cudaStream_t s, Envelope env, Band band)
{
    if (D > MAX_ELL || n_ell > MAX_ELL) { set_error("D=%d exceeds MAX_ELL=%d", D, MAX_ELL); return GPMC_EINVAL; }
    if (B <= 0) return 0;
    static_assert(AT == ENV_ROWS, "one tile row block is one envelope block");
    if (env.blk && (env.n != N || env.ld < env_blocks(N))) { set_error("cov_assemble: envelope n=%d ld=%d for N=%d", env.n, env.ld, N); return GPMC_EINVAL; }
    if (band.w && (!(flags & GPMC_ASM_LOWER_ONLY) || band.width < 0)) { set_error("cov_assemble: band needs the lower-only assembly"); return GPMC_EINVAL; }
    // the compact layout stores the band only: its tiles are all the assembly may write
    if (A.W && (!band.w || band.clear || A.n != N)) { set_error("cov_assemble: the compact layout needs the band grid without a clear"); return GPMC_EINVAL; }
    const int nt = (N + AT - 1) / AT;
    dim3 grid(band.w && !band.clear ? nt * (std::min(band.width, nt - 1) + 1) : (nt * (nt + 1) / 2 + ASM_TPC - 1) / ASM_TPC, B);
    prof_begin(KC_ASSEMBLE, s);
    if (env.blk) env_init_kernel<<<B, 128, 0, s>>>(A, env);
    if (band.w) band.width = std::min(band.width, nt - 1);
#define GPMC_ASM_LAUNCH(DT_)                                                                                                     \
    do {                                                                                                                          \
        if (flags & GPMC_ASM_PRED) cov_assemble_kernel<DT_, true><<<grid, 256, 0, s>>>(x, N, D, hyp, P, n_ell, flags, jitter, A, env, band);  \
        else cov_assemble_kernel<DT_, false><<<grid, 256, 0, s>>>(x, N, D, hyp, P, n_ell, flags, jitter, A, env, band);                       \
    } while (0)
    switch (D) {
        case 1: GPMC_ASM_LAUNCH(1); break;
        case 2: GPMC_ASM_LAUNCH(2); break;
        case 3: GPMC_ASM_LAUNCH(3); break;
        case 4: GPMC_ASM_LAUNCH(4); break;
        default: GPMC_ASM_LAUNCH(0); break;
    }
#undef GPMC_ASM_LAUNCH
    prof_end(KC_ASSEMBLE, s);
    GPMC_LAUNCH_CHECK();
    return 0;
}

}  // namespace gpmc
