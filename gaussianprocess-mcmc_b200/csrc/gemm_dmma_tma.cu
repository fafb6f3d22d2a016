// TMA-staged variant of the FP64 DMMA tile kernel (same contraction and epilogues as gemm_dmma.cu).
//
// Operand tiles are fetched by the Tensor Memory Accelerator: one elected thread issues
// cp.async.bulk.tensor.3d (box = 16 doubles x {128|64} rows x 1 matrix) per operand and stage, completion is
// signalled on an mbarrier (expect_tx / complete_tx), the 256 consumer threads wait on the barrier's phase bit.
// Rows beyond the operand's extent are zero-filled by the TMA unit itself (tensor-map bounds), so there is no
// per-thread predication, address arithmetic or cp.async issue slot in the main loop.
//
// Shared-memory layout: dense 128-byte rows (16 doubles) with the hardware 128B swizzle: the 16-byte piece p of
// row r lands at piece p ^ (r & 7).  A DMMA m8n8k4 fragment wants, per half-warp, 4 rows x 4 k: to keep that
// conflict-free under the swizzle the kernel permutes the contraction index inside a K=16 chunk (legal: both
// operands use the same permutation): step s of a chunk uses k in {2s, 2s+1, 8+2s, 9+2s}, lane (row, fk) reads
// piece ((fk>>1)*4 + s) ^ row, half (fk & 1) -> the 16 lanes of a half-warp touch 16 distinct 8-byte slots.
#include "common.cuh"
#include "gemm_common.cuh"
#include "../../include/gpmc.h"

#include <cuda.h>
#include <algorithm>
#include <type_traits>
#include <cudaTypedefs.h>

namespace gpmc {

constexpr int TBM = 128, TBN = 64, TBK = 16;
constexpr int TSTAGES = 4;
constexpr int TTHREADS = 256;
constexpr int A_BYTES = TBM * TBK * 8;                 // 16 KiB
constexpr int B_BYTES = TBN * TBK * 8;                 //  8 KiB
constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int TMA_SMEM = TSTAGES * STAGE_BYTES + 1024 + 128 + 64;  // + alignment slack + barriers (+ the producer's tile records)

__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes));
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, unsigned parity)
{
    unsigned ok;
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                 : "=r"(ok) : "r"((unsigned)__cvta_generic_to_shared(bar)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity)
{
    // bounded: a TMA that never completes (bad descriptor) must not hang the GPU
    for (unsigned it = 0; it < (1u << 26); ++it)
        if (mbar_try_wait(bar, parity)) return;
    __trap();
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void *smem, const CUtensorMap *map, uint64_t *bar, int c0, int c1, int c2)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];\n"
                 ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(map), "r"((unsigned)__cvta_generic_to_shared(bar)),
                   "r"(c0), "r"(c1), "r"(c2) : "memory");
}

// FREE_RUNNING = false: one __syncthreads per K chunk recycles the stages (all warps in lock step).
// FREE_RUNNING = true : full/empty mbarrier pairs per stage -- every warp arrives on empty[s] when it has read stage s,
//                       the producer thread refills a stage once its empty barrier completed, and no block barrier
//                       is left in the main loop, so the eight warps drift apart instead of stalling together.
template <bool FREE_RUNNING>
__global__ void __launch_bounds__(TTHREADS, 2)
gemm_dmma_tma_kernel(GemmArgs p, const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB)
{
    constexpr int WARPS_N = 2, FM = 4, FN = 4;          // 4 x 2 warps, warp tile 32 x 32
    extern __shared__ __align__(16) unsigned char smem_raw[];
    unsigned char *smem = (unsigned char *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);   // swizzle atoms: 1024 B
    uint64_t *full = (uint64_t *)(smem + TSTAGES * STAGE_BYTES);
    uint64_t *empty = full + TSTAGES;
    const int b = blockIdx.y;
    if (p.C.count && b >= *p.C.count) return;
    const int m = batch_item(p.C, b);
    int tm, tn;
    gemm_tile_decode<TBM, TBN>(p, blockIdx.x, tm, tn);
    if (p.skip_upper && p.cr0 + tm * TBM + TBM - 1 < p.cc0 + tn * TBN) return;     // whole tile above the diagonal
    const int rows_valid = min(TBM, p.rows - tm * TBM);
    const int cols_valid = min(TBN, p.cols - tn * TBN);
    int koff = 0;
    if (p.k_follow_row) koff = max(0, (p.ar0 + tm * TBM) - p.k0) & ~(TBK - 1);
    if (p.env.blk) {
        // L[r, k] = 0 for k left of row r's envelope: chunks below the later envelope of the A-tile rows and the B-tile
        // rows add exact zeros (+0 accumulators stay +0, the rest is summed in the same order) -- start after them.  The
        // border-row warp of a diagonal tile contracts against the B tile, so it may start there too.
        const int ra = p.ar0 + tm * TBM, rb = p.br0 + tn * TBN;
        const int kenv = max(env_first_col(p.env, m, ra, ra + rows_valid), env_first_col(p.env, m, rb, rb + cols_valid));
        koff = max(koff, (kenv & ~(TBK - 1)) - p.k0);
        if (koff >= p.klen) return;                   // every product of the tile is zero: C stays as it is
    }
    const int klen = p.klen - koff;
    const int nk = klen > 0 ? (klen + TBK - 1) / TBK : 0;
    const int tid = threadIdx.x;

    if (tid == 0) {
        asm volatile("prefetch.tensormap [%0];\n" ::"l"(&tmA));
        asm volatile("prefetch.tensormap [%0];\n" ::"l"(&tmB));
        for (int s = 0; s < TSTAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], TTHREADS / 32); }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::);
    }
    __syncthreads();

    const int arow = p.ar0 + tm * TBM, brow = p.br0 + tn * TBN;
    const int ak = p.k0 + koff, bk = p.bk0 + koff;
    // compact layout (A = B = C): a box's rows lie in one 128-row block, its column coordinate is relative to that block's
    // first stored column
    const int acol = p.C.W ? ak - band_col0(arow, p.C.W) : ak, bcol = p.C.W ? bk - band_col0(brow, p.C.W) : bk;
    auto issue = [&](int chunk) {
        const int s = chunk % TSTAGES;
        unsigned char *st = smem + s * STAGE_BYTES;
        mbar_expect_tx(&full[s], STAGE_BYTES);
        tma_load_3d(st, &tmA, &full[s], acol + chunk * TBK, arow, m);
        tma_load_3d(st + A_BYTES, &tmB, &full[s], bcol + chunk * TBK, brow, m);
    };
    if (tid == 0)      // lock step: one stage stays free for the refill; free running: all stages start full
        for (int s = 0; s < (FREE_RUNNING ? TSTAGES : TSTAGES - 1) && s < nk; ++s) issue(s);

    // the epilogue subtracts from the C tile: ask L2 for its 512 lines now (two per thread), so that the loads at the
    // end of the K loop do not wait for HBM -- matters for the short contractions only (K = 128 parts of the look-ahead,
    // N = 512 matrices: +1 ... 1.5 %; long contractions hide the epilogue behind the co-resident CTA anyway)
    if ((p.epi == EPI_SUB || p.epi == EPI_ADD) && klen <= 512) {
        const double *Cb = view_elem(p.C, m, p.cr0 + tm * TBM, p.cc0 + tn * TBN);
#pragma unroll
        for (int e = tid; e < TBM * (TBN / 16); e += TTHREADS) {
            const int r = e / (TBN / 16), c = (e % (TBN / 16)) * 16;
            if (r < rows_valid && c < cols_valid) asm volatile("prefetch.global.L2 [%0];\n" ::"l"(Cb + (size_t)r * p.C.ld + c));
        }
    }

    const int warp = tid >> 5, lane = tid & 31;
    const int wm = warp / WARPS_N, wn = warp % WARPS_N;
    const int frow = lane >> 2, fk = lane & 3;
    // swizzled fragment offsets (bytes) inside a tile row: piece ((fk>>1)*4 + s) ^ frow, half (fk & 1)
    int foff[4];
#pragma unroll
    for (int s = 0; s < 4; ++s) foff[s] = ((((fk >> 1) * 4 + s) ^ frow) << 4) + ((fk & 1) << 3);

    double acc[FM][FN][2];
#pragma unroll
    for (int i = 0; i < FM; ++i)
#pragma unroll
        for (int j = 0; j < FN; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    // diagonal tiles of a symmetric update: a warp whose 32x32 sub-tile is strictly above the diagonal has nothing to
    // contribute (6 of the 16 sub-tiles of a 128x128 diagonal block) -- it only keeps the stage hand-shake going and
    // leaves its DMMA issue slots to the other resident warps
    // ... and so has a warp whose rows all lie beyond the output (ragged last row tile, e.g. a single border row)
    const bool skip = (wm * FM * 8 >= rows_valid) ||
                      (p.skip_upper && (p.cr0 + tm * TBM + (wm + 1) * FM * 8 - 1 < p.cc0 + tn * TBN + wn * FN * 8));
    const bool on_diag = p.skip_upper && (p.cr0 + tm * TBM + wm * FM * 8 == p.cc0 + tn * TBN + wn * FN * 8);
    if (FREE_RUNNING && skip) {
        // Border duty: in a tile on the diagonal the warp (wm, wn) = (0, 1) is always one of the skippers.  It carries
        // the right-hand side stored as row p.border_row through the same update for the tile's 64 columns:
        // one real row in the 8-row A fragment (read straight from global memory, one chunk ahead), B fragments
        // from the staged tile -- 8 DMMAs per k step instead of none.
        const bool duty = p.border_row > 0 && wm == 0 && wn == 1 && (p.cr0 + tm * TBM == p.cc0 + (tn * TBN) / TBM * TBM);
        const double *zrow = view_elem(p.C, m, p.border_row, ak);      // (A == C: the launcher checks)
        const int kq = (fk >> 1) * 8 + (fk & 1);        // this lane's k inside a chunk at step ks: kq + 2 ks (the permuted order)
        double bacc[8][2];
#pragma unroll
        for (int j = 0; j < 8; ++j) bacc[j][0] = bacc[j][1] = 0.0;
        double zn[4] = {0.0, 0.0, 0.0, 0.0};
        auto zload = [&](int chunk) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
                const int k = chunk * TBK + kq + 2 * ks;
                zn[ks] = (frow == 0 && k < klen) ? zrow[k] : 0.0;
            }
        };
        if (duty && nk > 0) zload(0);
        for (int kc = 0; kc < nk; ++kc) {
            const int s = kc % TSTAGES;
            double zc[4];
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) zc[ks] = zn[ks];
            if (duty && kc + 1 < nk) zload(kc + 1);
            mbar_wait(&full[s], (kc / TSTAGES) & 1);
            if (duty) {
                const unsigned char *sb = smem + s * STAGE_BYTES + A_BYTES + frow * 128;
#pragma unroll
                for (int ks = 0; ks < 4; ++ks)
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        dmma884(bacc[j][0], bacc[j][1], zc[ks], *reinterpret_cast<const double *>(sb + j * 8 * 128 + foff[ks]));
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[s]);
            if (tid == 0 && kc >= 1 && kc + TSTAGES - 1 < nk) {
                const int prev = kc - 1;
                mbar_wait(&empty[prev % TSTAGES], (prev / TSTAGES) & 1);
                asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
                issue(kc + TSTAGES - 1);
            }
        }
        if (duty && frow == 0) {
            double *crow = view_elem(p.C, m, p.border_row, p.cc0 + tn * TBN);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int cl = j * 8 + fk * 2;
                if (cl >= cols_valid) continue;
                if (cl + 1 < cols_valid) {
                    double2 c = *reinterpret_cast<const double2 *>(crow + cl);
                    c.x -= bacc[j][0]; c.y -= bacc[j][1];
                    *reinterpret_cast<double2 *>(crow + cl) = c;
                } else crow[cl] -= bacc[j][0];
            }
        }
        return;
    }

    // the K loop, in two compiled shapes: every 8x8 block of the warp's sub-tile, or (sub-tile ON the diagonal of a
    // skip_upper update) only the blocks with j <= i -- chosen once per warp, outside the loop
    auto main_loop = [&](auto diag_tag) {
        constexpr bool DIAG = decltype(diag_tag)::value;
        for (int kc = 0; kc < nk; ++kc) {
            const int s = kc % TSTAGES;
            mbar_wait(&full[s], (kc / TSTAGES) & 1);
            if (!FREE_RUNNING) {
                __syncthreads();                              // everyone is done with the stage refilled below
                if (tid == 0 && kc + TSTAGES - 1 < nk) {
                    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
                    issue(kc + TSTAGES - 1);
                }
            }
            const unsigned char *sa = smem + s * STAGE_BYTES + (wm * FM * 8 + frow) * 128;
            const unsigned char *sb = smem + s * STAGE_BYTES + A_BYTES + (wn * FN * 8 + frow) * 128;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
                double af[FM], bf[FN];
#pragma unroll
                for (int i = 0; i < FM; ++i) af[i] = *reinterpret_cast<const double *>(sa + i * 8 * 128 + foff[ks]);
#pragma unroll
                for (int j = 0; j < FN; ++j) bf[j] = *reinterpret_cast<const double *>(sb + j * 8 * 128 + foff[ks]);
                if (FREE_RUNNING && ks == 3) {
                    // the fragments of this stage are in registers: release it, and let the producer refill the stage
                    // that every warp released one chunk ago
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&empty[s]);
                    if (tid == 0 && kc >= 1 && kc + TSTAGES - 1 < nk) {
                        const int prev = kc - 1;
                        mbar_wait(&empty[prev % TSTAGES], (prev / TSTAGES) & 1);
                        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
                        issue(kc + TSTAGES - 1);
                    }
                }
#pragma unroll
                for (int i = 0; i < FM; ++i)
#pragma unroll
                    for (int j = 0; j < FN; ++j)
                        if (!DIAG || j <= i) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
            }
        }
    };
    // lock step keeps every warp on one path (block barriers inside the loop)
    if (FREE_RUNNING && on_diag) main_loop(std::true_type{});
    else main_loop(std::false_type{});
    gemm_epilogue<FM, FN, TBM, TBN>(p, m, tm, tn, wm, wn, frow, fk, rows_valid, cols_valid, acc);
}

// ------------------------------------------------------------------------------------------ persistent form
// One CTA per resident slot (2 per SM) walks over the launch's tiles (item-major: consecutive CTAs take consecutive tiles
// of one matrix).  The stage ring and its mbarrier phases run on across tiles -- chunks are numbered globally per CTA -- so
// the producer thread fetches the first chunks of the NEXT tile while the warps are still in the tail and the epilogue of
// the current one.  What it buys is the per-tile prologue (barrier setup, first TMA round trip: ~2 us), which the
// one-tile-per-CTA kernel only hides while the two co-resident CTAs happen to be out of phase; it matters for the short
// contractions (K = 128 ... 512: 8 ... 32 chunks per tile).
// Tiles are handed out IN ORDER from a global counter (sched[0]; thread 0 draws the next tile at the start of the current
// one and publishes it to the other warps through a sequence-tagged slot in shared memory): like the hardware's own CTA
// dispatch this keeps the ~300 tiles in flight on a handful of matrices, whose operands the L2 then serves.  Static
// striding (tile = blockIdx.x + i * gridDim.x) lets the CTAs drift apart and was measured 9 % (N=4096) to 25 % (N=512)
// SLOWER than one tile per CTA: L2 hit rate 13-40 % instead of 42-51 % (profiles/r02p_ncu_gemm_persistent.txt).
// The last CTA to leave resets the counters (sched[1] counts finished CTAs), so a slot of the launcher's ring is clean
// again when its turn comes round.  Every tile must have at least one chunk (the launcher checks): the stage ring then
// bounds how far thread 0 can run ahead of the slowest warp (5 tiles), and the 8 published slots are never overwritten
// before they were read.
struct TileCtx {
    int m, tm, tn, rows_valid, cols_valid, arow, brow, ak, bk, nk, klen;
};

__device__ __forceinline__ bool decode_work(const GemmArgs &p, long long w, int tiles, TileCtx &t)
{
    const int b = (int)(w / tiles);
    const int ti = (int)(w - (long long)b * tiles);
    gemm_tile_decode<TBM, TBN>(p, ti, t.tm, t.tn);
    if (p.skip_upper && p.cr0 + t.tm * TBM + TBM - 1 < p.cc0 + t.tn * TBN) return false;      // whole tile above the diagonal
    t.m = batch_item(p.C, b);
    t.rows_valid = min(TBM, p.rows - t.tm * TBM);
    t.cols_valid = min(TBN, p.cols - t.tn * TBN);
    int koff = 0;
    if (p.k_follow_row) koff = max(0, (p.ar0 + t.tm * TBM) - p.k0) & ~(TBK - 1);
    t.klen = p.klen - koff;
    t.nk = t.klen > 0 ? (t.klen + TBK - 1) / TBK : 0;
    t.arow = p.ar0 + t.tm * TBM;
    t.brow = p.br0 + t.tn * TBN;
    t.ak = p.k0 + koff;
    t.bk = p.bk0 + koff;
    return true;
}

__global__ void __launch_bounds__(TTHREADS, 2)
gemm_dmma_tma_persistent_kernel(GemmArgs p, const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                                int tiles, int n_items_max, int *sched)
{
    constexpr int W_NONE = 0x7fffffff;
    constexpr int WARPS_N = 2, FM = 4, FN = 4;          // 4 x 2 warps, warp tile 32 x 32
    extern __shared__ __align__(16) unsigned char smem_raw[];
    unsigned char *smem = (unsigned char *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t *full = (uint64_t *)(smem + TSTAGES * STAGE_BYTES);
    uint64_t *empty = full + TSTAGES;
    const int tid = threadIdx.x;
    const int n_items = p.C.count ? min(*p.C.count, n_items_max) : n_items_max;
    const int total = tiles * n_items;              // (the launcher keeps this below 2^31)
    int *pctx = reinterpret_cast<int *>(empty + TSTAGES);                              // producer's tile records, 16 ints
    volatile long long *slots = reinterpret_cast<volatile long long *>(pctx + 16);     // published tiles: (sequence << 32) | tile
    // draw tiles from the global counter until one has work (tiles wholly above the diagonal have none)
    auto draw = [&](TileCtx &t) -> int {
        while (true) {
            const int w = atomicAdd(sched, 1) + (int)gridDim.x;
            if (w >= total) return W_NONE;
            if (decode_work(p, w, tiles, t)) return w;
        }
    };

    if (tid == 0) {
        asm volatile("prefetch.tensormap [%0];\n" ::"l"(&tmA));
        asm volatile("prefetch.tensormap [%0];\n" ::"l"(&tmB));
        for (int s = 0; s < TSTAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], TTHREADS / 32); }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::);
        TileCtx t;
        int w = blockIdx.x;                          // the first gridDim.x tiles are dealt by position
        if (w >= total) w = W_NONE;
        else if (!decode_work(p, w, tiles, t)) w = draw(t);
        for (int i = 1; i < 8; ++i) slots[i] = -1;
        slots[0] = (long long)(unsigned)w;           // sequence 0
    }
    __syncthreads();

    const int warp = tid >> 5, lane = tid & 31;
    const int wm = warp / WARPS_N, wn = warp % WARPS_N;
    const int frow = lane >> 2, fk = lane & 3;
    int foff[4];
#pragma unroll
    for (int s = 0; s < 4; ++s) foff[s] = ((((fk >> 1) * 4 + s) ^ frow) << 4) + ((fk & 1) << 3);

    // what the producer thread needs of the current and of the next tile lives in shared memory (it alone reads and
    // writes it): {m, arow, brow, ak, bk, nk}; nk = 0 for "no next tile"
    TileCtx cur;
    int wc = (int)slots[0];
    if (wc != W_NONE) decode_work(p, wc, tiles, cur);
    int seq = 0;                        // tiles this CTA has started
    unsigned gbase = 0;                 // global number (per CTA) of the current tile's first chunk
    unsigned g_next = 0;                // next chunk to fetch (thread 0)

    // chunk g (global) goes into stage g % TSTAGES once every warp has released chunk g - TSTAGES
    auto fetch = [&](unsigned g, const volatile int *t, int local) {
        const int s = g % TSTAGES;
        if (g >= (unsigned)TSTAGES) {
            mbar_wait(&empty[s], ((g / TSTAGES) - 1) & 1);
            asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
        }
        unsigned char *st = smem + s * STAGE_BYTES;
        mbar_expect_tx(&full[s], STAGE_BYTES);
        tma_load_3d(st, &tmA, &full[s], t[3] + local * TBK, t[1], t[0]);
        tma_load_3d(st + A_BYTES, &tmB, &full[s], t[4] + local * TBK, t[2], t[0]);
    };
    auto pump = [&](unsigned upto) {          // thread 0: fetch every chunk up to global number `upto` that exists
        const volatile int *c0 = pctx, *c1 = pctx + 8;
        while (g_next <= upto) {
            const unsigned off = g_next - gbase, nk0 = (unsigned)c0[5];
            if (off < nk0) fetch(g_next, c0, (int)off);
            else if (off - nk0 < (unsigned)c1[5]) fetch(g_next, c1, (int)(off - nk0));
            else break;
            ++g_next;
        }
    };

    while (wc != W_NONE) {
        // the tile after this one: thread 0 draws it now, publishes it, and fetches its first chunks before this one is finished
        if (tid == 0) {
            TileCtx nx;
            nx.m = nx.arow = nx.brow = nx.ak = nx.bk = nx.nk = 0;
            const int wnext = draw(nx);
            pctx[0] = cur.m; pctx[1] = cur.arow; pctx[2] = cur.brow; pctx[3] = cur.ak; pctx[4] = cur.bk; pctx[5] = cur.nk;
            pctx[8] = nx.m; pctx[9] = nx.arow; pctx[10] = nx.brow; pctx[11] = nx.ak; pctx[12] = nx.bk; pctx[13] = wnext != W_NONE ? nx.nk : 0;
            slots[(seq + 1) & 7] = ((long long)(seq + 1) << 32) | (long long)(unsigned)wnext;
            pump(gbase + TSTAGES - 1 - (gbase ? 1 : 0));      // (first tile: all stages; later: as in the K loop)
        }

        const int m = cur.m, tm = cur.tm, tn = cur.tn, rows_valid = cur.rows_valid, cols_valid = cur.cols_valid, nk = cur.nk;
        if ((p.epi == EPI_SUB || p.epi == EPI_ADD) && cur.klen <= 512) {
            const double *Cb = p.C.base + (size_t)m * p.C.stride + (size_t)(p.cr0 + tm * TBM) * p.C.ld + p.cc0 + tn * TBN;
#pragma unroll
            for (int e = tid; e < TBM * (TBN / 16); e += TTHREADS) {
                const int r = e / (TBN / 16), c = (e % (TBN / 16)) * 16;
                if (r < rows_valid && c < cols_valid) asm volatile("prefetch.global.L2 [%0];\n" ::"l"(Cb + (size_t)r * p.C.ld + c));
            }
        }

        const bool skip = (wm * FM * 8 >= rows_valid) ||
                          (p.skip_upper && (p.cr0 + tm * TBM + (wm + 1) * FM * 8 - 1 < p.cc0 + tn * TBN + wn * FN * 8));
        const bool on_diag = p.skip_upper && (p.cr0 + tm * TBM + wm * FM * 8 == p.cc0 + tn * TBN + wn * FN * 8);
        if (skip) {
            // (border duty as in the one-tile kernel: see there)
            const bool duty = p.border_row > 0 && wm == 0 && wn == 1 && (p.cr0 + tm * TBM == p.cc0 + (tn * TBN) / TBM * TBM);
            const double *zrow = p.A.base + (size_t)m * p.A.stride + (size_t)p.border_row * p.A.ld + cur.ak;
            const int kq = (fk >> 1) * 8 + (fk & 1);
            double bacc[8][2];
#pragma unroll
            for (int j = 0; j < 8; ++j) bacc[j][0] = bacc[j][1] = 0.0;
            double zn[4] = {0.0, 0.0, 0.0, 0.0};
            auto zload = [&](int chunk) {
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {
                    const int k = chunk * TBK + kq + 2 * ks;
                    zn[ks] = (frow == 0 && k < cur.klen) ? zrow[k] : 0.0;
                }
            };
            if (duty && nk > 0) zload(0);
            for (int kc = 0; kc < nk; ++kc) {
                const unsigned g = gbase + kc;
                const int s = g % TSTAGES;
                double zc[4];
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) zc[ks] = zn[ks];
                if (duty && kc + 1 < nk) zload(kc + 1);
                mbar_wait(&full[s], (g / TSTAGES) & 1);
                if (duty) {
                    const unsigned char *sb = smem + s * STAGE_BYTES + A_BYTES + frow * 128;
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks)
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            dmma884(bacc[j][0], bacc[j][1], zc[ks], *reinterpret_cast<const double *>(sb + j * 8 * 128 + foff[ks]));
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[s]);
                if (tid == 0) pump(g + TSTAGES - 1);
            }
            if (duty && frow == 0) {
                double *crow = p.C.base + (size_t)m * p.C.stride + (size_t)p.border_row * p.C.ld + p.cc0 + tn * TBN;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int cl = j * 8 + fk * 2;
                    if (cl >= cols_valid) continue;
                    if (cl + 1 < cols_valid) {
                        double2 c = *reinterpret_cast<const double2 *>(crow + cl);
                        c.x -= bacc[j][0]; c.y -= bacc[j][1];
                        *reinterpret_cast<double2 *>(crow + cl) = c;
                    } else crow[cl] -= bacc[j][0];
                }
            }
        } else {
            double acc[FM][FN][2];
#pragma unroll
            for (int i = 0; i < FM; ++i)
#pragma unroll
                for (int j = 0; j < FN; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
            auto main_loop = [&](auto diag_tag) {
                constexpr bool DIAG = decltype(diag_tag)::value;
                for (int kc = 0; kc < nk; ++kc) {
                    const unsigned g = gbase + kc;
                    const int s = g % TSTAGES;
                    mbar_wait(&full[s], (g / TSTAGES) & 1);
                    const unsigned char *sa = smem + s * STAGE_BYTES + (wm * FM * 8 + frow) * 128;
                    const unsigned char *sb = smem + s * STAGE_BYTES + A_BYTES + (wn * FN * 8 + frow) * 128;
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {
                        double af[FM], bf[FN];
#pragma unroll
                        for (int i = 0; i < FM; ++i) af[i] = *reinterpret_cast<const double *>(sa + i * 8 * 128 + foff[ks]);
#pragma unroll
                        for (int j = 0; j < FN; ++j) bf[j] = *reinterpret_cast<const double *>(sb + j * 8 * 128 + foff[ks]);
                        if (ks == 3) {
                            __syncwarp();
                            if (lane == 0) mbar_arrive(&empty[s]);
                            if (tid == 0) pump(g + TSTAGES - 1);
                        }
#pragma unroll
                        for (int i = 0; i < FM; ++i)
#pragma unroll
                            for (int j = 0; j < FN; ++j)
                                if (!DIAG || j <= i) dmma884(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
                    }
                }
            };
            if (on_diag) main_loop(std::true_type{});
            else main_loop(std::false_type{});
            gemm_epilogue<FM, FN, TBM, TBN>(p, m, tm, tn, wm, wn, frow, fk, rows_valid, cols_valid, acc);
        }
        gbase += (unsigned)nk;
        ++seq;
        {
            // the tile thread 0 published for this position (written at the start of the tile just finished)
            long long v = slots[seq & 7];
            for (unsigned it = 0; (int)(v >> 32) != seq; ++it) {
                if (it > (1u << 26)) __trap();
                v = slots[seq & 7];
            }
            wc = (int)(unsigned)(v & 0xffffffffLL);
        }
        if (wc != W_NONE) decode_work(p, wc, tiles, cur);
    }
    if (tid == 0) {
        // last CTA out resets the scheduler words for the launch that gets this ring slot next
        __threadfence();
        if (atomicAdd(sched + 1, 1) == (int)gridDim.x - 1) { sched[0] = 0; sched[1] = 0; __threadfence(); }
    }
}

// ------------------------------------------------------------------------------------------ host side
static PFN_cuTensorMapEncodeTiled_v12000 g_encode = nullptr;

static int get_encoder()
{
    if (g_encode) return 0;
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
        set_error("cuTensorMapEncodeTiled is not available from the driver (%s)", cudaGetErrorString(e));
        return GPMC_EINVAL;
    }
    g_encode = (PFN_cuTensorMapEncodeTiled_v12000)fn;
    return 0;
}

// 3-D map over matrices stored as [batch][row][ld]: dims (inner -> outer) = {ld, rows_extent, nbatch}
static int make_map(CUtensorMap *map, const Operand &op, int rows_extent, int box_rows)
{
    const cuuint64_t dims[3] = {(cuuint64_t)op.ld, (cuuint64_t)rows_extent, (cuuint64_t)1 << 20};
    const cuuint64_t strides[2] = {(cuuint64_t)op.ld * 8, (cuuint64_t)op.stride * 8};
    const cuuint32_t box[3] = {(cuuint32_t)TBK, (cuuint32_t)box_rows, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = g_encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, (void *)op.base, dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed (%d): base=%p ld=%d stride=%lld rows=%d", (int)r, (const void *)op.base, op.ld,
                  op.stride, rows_extent);
        return GPMC_EINVAL;
    }
    return 0;
}

bool gemm_tma_supported(const GemmArgs &a)
{
    // TMA needs 16-byte aligned bases and strides; a zero batch stride (shared operand) is not mapped
    return a.A.stride > 0 && a.B.stride > 0 && ((uintptr_t)a.A.base % 16 == 0) && ((uintptr_t)a.B.base % 16 == 0) &&
           (a.A.ld % 2 == 0) && (a.B.ld % 2 == 0) && (a.A.stride % 2 == 0) && (a.B.stride % 2 == 0) &&
           a.A.ld >= TBK && a.B.ld >= TBK;
}

int launch_gemm_tma(const GemmArgs &a, int B, int kclass, bool free_running, cudaStream_t s, bool persistent)
{
    int rc = get_encoder();
    if (rc) return rc;
    static DeviceOnce attr_set;
    if (attr_set.first()) {
        GPMC_CUDA_CHECK(cudaFuncSetAttribute(gemm_dmma_tma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TMA_SMEM));
        GPMC_CUDA_CHECK(cudaFuncSetAttribute(gemm_dmma_tma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TMA_SMEM));
        GPMC_CUDA_CHECK(cudaFuncSetAttribute(gemm_dmma_tma_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TMA_SMEM));
    }
    CUtensorMap tmA, tmB;
    // rows at or beyond (origin + extent) are out of bounds for the TMA unit -> zero fill
    if (a.C.W) {
        // compact layout: only the one-tile kernel of the Cholesky updates knows it (A = B = C, envelope exits before any
        // access outside the band, boxes and C tiles inside one 128-row block)
        if (persistent || !free_running || a.A.base != a.C.base || a.B.base != a.C.base || !a.env.blk ||
            a.k_follow_row || a.epi != EPI_SUB || a.A.ld != a.C.W || a.B.ld != a.C.W || a.ar0 % BAND_ROWS || a.br0 % BAND_ROWS ||
            a.cr0 % BAND_ROWS) {
            set_error("gemm: the compact band layout is supported by the Cholesky updates of the one-tile kernel only");
            return GPMC_EINVAL;
        }
    }
    if ((rc = make_map(&tmA, a.A, a.ar0 + a.rows, TBM))) return rc;
    if ((rc = make_map(&tmB, a.B, a.br0 + a.cols, TBN))) return rc;
    const int tiles_m = (a.rows + TBM - 1) / TBM;
    const int tiles_n = (a.cols + TBN - 1) / TBN;
    const int tiles = a.lower_only ? (TBM / TBN) * tiles_m * (tiles_m + 1) / 2 : tiles_m * tiles_n;
    if (persistent) {
        static int slots = 0;                      // resident CTAs of this kernel on the whole chip (2 per SM)
        if (slots == 0) {
            int dev = 0, sms = 0;
            if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
            slots = 2 * sms;
        }
        const long long total = (long long)tiles * B;
        // scheduler words: a ring of (next tile, finished CTAs) pairs per device, every launch takes the next pair; the
        // kernel leaves its pair zeroed.  (Far more pairs than launches can be in flight at once.)
        constexpr int RING = 8192;
        static int *ring[64] = {};
        static unsigned ring_pos[64] = {};
        int dev = 0;
        GPMC_CUDA_CHECK(cudaGetDevice(&dev));
        if (dev < 0 || dev >= 64) { set_error("gemm: device ordinal %d out of range", dev); return GPMC_EINVAL; }
        if (!ring[dev]) {
            GPMC_CUDA_CHECK(cudaMalloc(&ring[dev], (size_t)RING * 2 * sizeof(int)));
            GPMC_CUDA_CHECK(cudaMemset(ring[dev], 0, (size_t)RING * 2 * sizeof(int)));
        }
        int *sched = ring[dev] + 2 * (ring_pos[dev]++ % RING);
        prof_begin(kclass, s);
        gemm_dmma_tma_persistent_kernel<<<(unsigned)std::min<long long>(total, slots), TTHREADS, TMA_SMEM, s>>>(a, tmA, tmB, tiles, B, sched);
        prof_end(kclass, s);
        GPMC_LAUNCH_CHECK();
        return 0;
    }
    dim3 grid(tiles, B);
    prof_begin(kclass, s);
    if (free_running) gemm_dmma_tma_kernel<true><<<grid, TTHREADS, TMA_SMEM, s>>>(a, tmA, tmB);
    else gemm_dmma_tma_kernel<false><<<grid, TTHREADS, TMA_SMEM, s>>>(a, tmA, tmB);
    prof_end(kclass, s);
    GPMC_LAUNCH_CHECK();
    return 0;
}

}  // namespace gpmc
