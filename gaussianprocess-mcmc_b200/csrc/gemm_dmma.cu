// FP64 tensor-core (DMMA) tile kernel, cp.async-staged variants: every dense contraction of the hot path is an "NT"
// product
//     C[i][j]  (op)=  sum_k  A[i][k] * B[j][k]
// of two row-major operands whose contraction index is contiguous in memory:
//   * Cholesky block-column / trailing update   C -= L[i,:k] L[j,:k]^T          (kcGP.tools.jitchol -> dpotrf,
//                                                                                 sliceSample.py:196,205)
//   * triangular inverse U = L^-T, block column  Y  = U[:i,:i] L[i,:i]^T, then  U[:i,i] = -Y (L_ii^-1)^T
//   * posterior covariance                      R  = S - S (U U^T) S (+1e-11 I)  (sliceSample.py:197-198,205 in the
//                                                                                 algebraically reduced form, DESIGN.md)
// sm_100a has no FP64 kind in tcgen05; FP64 tensor cores are reached with mma.sync.m8n8k4.f64 (SASS DMMA.8x8x4).
// The DEFAULT kernel is the TMA-staged one in gemm_dmma_tma.cu; the variants here (128x128 with 8 or 16 warps,
// 128x64 with two CTAs per SM) stage operands with 16-byte cp.async into a ring of K=16 chunks whose rows are padded
// to 20 doubles, so the 8-byte fragment loads of a half-warp (4 rows x 4 k) hit 16 distinct bank pairs (ncu: 0 shared
// bank conflicts); rows beyond the matrix are zero-filled by cp.async's src-size operand.  They are kept for A/B
// measurements (GPMC_GEMM_CFG / gpmc_set_tuning) and as the fallback when an operand cannot be described by a
// tensor map.  launch_gemm() below dispatches.
#include "common.cuh"
#include "gemm_common.cuh"
#include "../../include/gpmc.h"
#include <stdlib.h>

namespace gpmc {

constexpr int BM = 128, BK = 16;
constexpr int SROW = BK + 4;                    // padded smem row (doubles)
constexpr int gemm_smem_bytes(int bn, int stages) { return stages * (BM + bn) * SROW * (int)sizeof(double); }

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem, int src_bytes)
{
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(src_bytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// Stage one K=16 chunk of a ROWS-row operand: ROWS rows x 8 16-byte pieces.
template <int THREADS, int ROWS>
__device__ __forceinline__ void load_operand(double *sdst, const double *gsrc, int ld, int rows_valid, int tid)
{
#pragma unroll
    for (int i = 0; i < ROWS * 8 / THREADS; ++i) {
        const int piece = tid + i * THREADS;
        const int row = piece >> 3, kc = piece & 7;
        const bool ok = row < rows_valid;
        const double *src = gsrc + (size_t)(ok ? row : 0) * ld + kc * 2;
        cp_async16(sdst + row * SROW + kc * 2, src, ok ? 16 : 0);
    }
}

// CTA tile 128 x BN; WARPS_M x WARPS_N warps, each owning (128/WARPS_M) x (BN/WARPS_N) as 8x8 DMMA fragments;
// STAGES-deep cp.async ring; CTAS_PER_SM resident CTAs (2 lets one CTA's barrier / prologue / epilogue hide behind
// the other's DMMA stream).
template <int WARPS_M, int WARPS_N, int BN, int STAGES, int CTAS_PER_SM>
__global__ void __launch_bounds__(WARPS_M * WARPS_N * 32, CTAS_PER_SM)
gemm_dmma_kernel(GemmArgs p)
{
    constexpr int THREADS = WARPS_M * WARPS_N * 32;
    constexpr int FM = BM / WARPS_M / 8;        // fragments per warp along M
    constexpr int FN = BN / WARPS_N / 8;
    constexpr int A_ELEMS = BM * SROW, STAGE_ELEMS = (BM + BN) * SROW;
    extern __shared__ __align__(16) double smem[];
    const int b = blockIdx.y;
    if (p.C.count && b >= *p.C.count) return;
    const int m = batch_item(p.C, b);

    int tm, tn;
    gemm_tile_decode<BM, BN>(p, blockIdx.x, tm, tn);
    const int rows_valid = min(BM, p.rows - tm * BM);
    const int cols_valid = min(BN, p.cols - tn * BN);

    // contraction range of this tile (triangular operands skip their zero part)
    int koff = 0;
    if (p.k_follow_row) koff = max(0, (p.ar0 + tm * BM) - p.k0) & ~(BK - 1);
    const int klen = p.klen - koff;
    const int nk = klen > 0 ? (klen + BK - 1) / BK : 0;

    const double *gA = p.A.base + (size_t)m * p.A.stride + (size_t)(p.ar0 + tm * BM) * p.A.ld + p.k0 + koff;
    const double *gB = p.B.base + (size_t)m * p.B.stride + (size_t)(p.br0 + tn * BN) * p.B.ld + p.bk0 + koff;
    const int lda = p.A.ld, ldb = p.B.ld;
    const int tid = threadIdx.x;

    auto stage_a = [&](int s) { return smem + (size_t)s * STAGE_ELEMS; };
    auto stage_b = [&](int s) { return smem + (size_t)s * STAGE_ELEMS + A_ELEMS; };

#pragma unroll
    for (int s = 0; s < STAGES - 1; ++s) {
        if (s < nk) {
            load_operand<THREADS, BM>(stage_a(s), gA + s * BK, lda, rows_valid, tid);
            load_operand<THREADS, BN>(stage_b(s), gB + s * BK, ldb, cols_valid, tid);
        }
        cp_async_commit();
    }

    const int warp = tid >> 5, lane = tid & 31;
    const int wm = warp / WARPS_N, wn = warp % WARPS_N;
    const int frow = lane >> 2, fk = lane & 3;      // fragment coordinates

    double acc[FM][FN][2];
#pragma unroll
    for (int i = 0; i < FM; ++i)
#pragma unroll
        for (int j = 0; j < FN; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    for (int kc = 0; kc < nk; ++kc) {
        cp_async_wait<STAGES - 2>();
        __syncthreads();
        {   // refill the stage consumed in the previous iteration
            const int nxt = kc + STAGES - 1;
            if (nxt < nk) {
                const int s = nxt % STAGES;
                load_operand<THREADS, BM>(stage_a(s), gA + nxt * BK, lda, rows_valid, tid);
                load_operand<THREADS, BN>(stage_b(s), gB + nxt * BK, ldb, cols_valid, tid);
            }
            cp_async_commit();
        }
        const double *sa = stage_a(kc % STAGES) + (wm * FM * 8 + frow) * SROW + fk;
        const double *sb = stage_b(kc % STAGES) + (wn * FN * 8 + frow) * SROW + fk;
#pragma unroll
        for (int ks = 0; ks < BK / 4; ++ks) {
            double af[FM], bf[FN];
#pragma unroll
            for (int i = 0; i < FM; ++i) af[i] = sa[i * 8 * SROW + ks * 4];
#pragma unroll
            for (int j = 0; j < FN; ++j) bf[j] = sb[j * 8 * SROW + ks * 4];
#pragma unroll
            for (int i = 0; i < FM; ++i)
#pragma unroll
                for (int j = 0; j < FN; ++j) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
        }
    }
    cp_async_wait<0>();

    gemm_epilogue<FM, FN, BM, BN>(p, m, tm, tn, wm, wn, frow, fk, rows_valid, cols_valid, acc);
}

bool gemm_tma_supported(const GemmArgs &a);
int launch_gemm_tma(const GemmArgs &a, int B, int kclass, bool free_running, cudaStream_t s, bool persistent = false);

// 0: 8 warps 128x128; 1: 16 warps 128x128; 2: 8 warps 128x64, two CTAs per SM (cp.async); 3: as 2, TMA-staged;
// 4: TMA-staged with full/empty mbarrier pairs (no block barrier in the main loop); 5: as 4, persistent CTAs that fetch
// the next tile's first chunks during the current tile's tail (used for short contractions when 4 is selected: see below)
static int g_gemm_cfg = 4;
void set_gemm_config(int cfg) { g_gemm_cfg = cfg; }
static void read_gemm_env()
{
    static bool env_read = false;
    if (!env_read) {            // GPMC_GEMM_CFG=0..3 selects the tile-kernel variant (experiments / A-B tests)
        const char *e = getenv("GPMC_GEMM_CFG");
        if (e && e[0] >= '0' && e[0] <= '5') g_gemm_cfg = e[0] - '0';
        env_read = true;
    }
}
bool gemm_honours_envelope()
{
    read_gemm_env();
    return g_gemm_cfg == 4;
}

template <typename K>
static int launch_variant(K kernel, const GemmArgs &a, int B, int bn, int threads, int smem, int kclass, cudaStream_t s, DeviceOnce &attr_set)
{
    if (attr_set.first()) GPMC_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const int tiles_m = (a.rows + BM - 1) / BM;
    const int tiles_n = (a.cols + bn - 1) / bn;
    const int tiles = a.lower_only ? (BM / bn) * tiles_m * (tiles_m + 1) / 2 : tiles_m * tiles_n;
    dim3 grid(tiles, B);
    prof_begin(kclass, s);
    kernel<<<grid, threads, smem, s>>>(a);
    prof_end(kclass, s);
    GPMC_LAUNCH_CHECK();
    return 0;
}

int launch_gemm(const GemmArgs &a, int B, int kclass, cudaStream_t s)
{
    if (B <= 0 || a.rows <= 0 || a.cols <= 0) return 0;
    if ((a.A.ld & 1) || (a.B.ld & 1) || (a.C.ld & 1) || (a.k0 & 1) || (a.bk0 & 1) || (a.cc0 & 1)) {
        set_error("gemm: k0=%d bk0=%d cc0=%d lda=%d ldb=%d ldc=%d violate the 16-byte staging alignment",
                  a.k0, a.bk0, a.cc0, a.A.ld, a.B.ld, a.C.ld);
        return GPMC_EALIGN;
    }
    static DeviceOnce set0, set1, set2;
    read_gemm_env();
    const bool border_fusable = a.border_row == 0 || (a.skip_upper && a.epi == EPI_SUB && a.cr0 == a.cc0 && a.A.base == a.C.base);
    // persistent form: every tile needs at least one chunk, and the tile count must fit the scheduler's 32-bit words
    const bool persist_ok = !a.k_follow_row && a.klen >= 1 &&
                            (long long)((a.rows + 127) / 128 + 1) * ((a.cols + 63) / 64 + 1) * B < 0x70000000LL;
    if (g_gemm_cfg == 5 && persist_ok && gemm_tma_supported(a) && border_fusable) return launch_gemm_tma(a, B, kclass, true, s, true);
    if (g_gemm_cfg == 4 && gemm_tma_supported(a) && border_fusable) return launch_gemm_tma(a, B, kclass, true, s);   // border row fused in-kernel
    // a band (env.band >= 0) leaves the matrix unwritten left of it: only the kernel above keeps its reads inside
    if (a.env.band >= 0) { set_error("gemm: a banded update needs the envelope-aware TMA tile kernel (tuning key 0 = 4)"); return GPMC_EINVAL; }
    if (a.border_row > 0) {
        // the other variants have no border duty: take the row along as one more output row (it follows the matrix)
        if (a.cr0 + a.rows != a.border_row || a.ar0 != a.cr0) { set_error("gemm: border row %d is not adjacent to the output rows", a.border_row); return GPMC_EINVAL; }
        GemmArgs b = a;
        b.rows += 1;
        b.border_row = 0;
        return launch_gemm(b, B, kclass, s);
    }
    if (g_gemm_cfg == 3 && gemm_tma_supported(a)) return launch_gemm_tma(a, B, kclass, false, s);
    if (g_gemm_cfg == 0) return launch_variant(gemm_dmma_kernel<2, 4, 128, 4, 1>, a, B, 128, 256, gemm_smem_bytes(128, 4), kclass, s, set0);
    if (g_gemm_cfg >= 2) return launch_variant(gemm_dmma_kernel<4, 2, 64, 3, 2>, a, B, 64, 256, gemm_smem_bytes(64, 3), kclass, s, set2);
    return launch_variant(gemm_dmma_kernel<4, 4, 128, 4, 1>, a, B, 128, 512, gemm_smem_bytes(128, 4), kclass, s, set1);
}

}  // namespace gpmc
