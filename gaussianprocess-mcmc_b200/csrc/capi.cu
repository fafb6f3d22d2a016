// C ABI of libgpmc.so (declared in include/gpmc.h) and the host-side drivers that sequence the kernels.
#include "common.cuh"
#include "sequences.cuh"
#include "../../include/gpmc.h"

#include <stdarg.h>
#include <string.h>
#include <mutex>
#include <algorithm>
#include <vector>

namespace gpmc {

// ------------------------------------------------------------------------------------ error text
static thread_local char g_err[1024] = "";          // the text belongs to the thread whose call failed
static std::recursive_mutex g_api_mutex;
ApiLock::ApiLock() { g_api_mutex.lock(); }
ApiLock::~ApiLock() { g_api_mutex.unlock(); }
void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

// ------------------------------------------------------------------------------ profiling hooks
struct EventPair { cudaEvent_t a, b; };
static bool g_prof_on = false;
static std::vector<EventPair> g_pool[KC_COUNT];
static size_t g_used[KC_COUNT] = {};

void prof_begin(int kc, cudaStream_t s)
{
    if (!g_prof_on) return;
    if (g_used[kc] == g_pool[kc].size()) {
        EventPair p;
        cudaEventCreate(&p.a);
        cudaEventCreate(&p.b);
        g_pool[kc].push_back(p);
    }
    cudaEventRecord(g_pool[kc][g_used[kc]].a, s);
}
void prof_end(int kc, cudaStream_t s)
{
    if (!g_prof_on) return;
    cudaEventRecord(g_pool[kc][g_used[kc]].b, s);
    ++g_used[kc];
}

// ------------------------------------------------------------------------------ small kernels
// restore item map[b] from the backup copy and add jitter[map[b]] to its diagonal
__global__ void restore_jitter_kernel(BatchView A, const double *backup, int n, const double *jitter)
{
    const int b = blockIdx.y;
    const int m = batch_item(A, b);
    double *Ab = A.base + (size_t)m * A.stride;
    const double *Bb = backup + (size_t)m * A.stride;
    const size_t total = (size_t)n * A.ld;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(e / A.ld), c = (int)(e - (size_t)r * A.ld);
        double v = Bb[e];
        if (r == c) v = v + jitter[m];
        Ab[e] = v;
    }
}


// S_ii and K_ii + S_ii on the host (same expression order as the kernel / sliceSample.py:185-190),
// used only to size the jitter of the ladder.
static double host_diag_value(const double *h, int n_ell)
{
    const double sf = h[n_ell], sn = h[n_ell + 1];
    const double sf2 = exp(2.0 * log(sf));
    const double kinv = 1.0 / sf2;
    const double v1 = 1.0 / (sn * sn) + kinv;
    double Sii = 1.0 / (v1 - kinv);
    if (Sii < 0.0) Sii = 0.0;
    return sf2 + Sii;
}

struct LoglikLayout {
    int ld;
    size_t mat_elems;        // per item
    size_t fixed_bytes;      // per-call scratch independent of the wave
    size_t per_item_bytes;   // matrix + W + envelope + band
};
static LoglikLayout loglik_layout(int N, int B)
{
    LoglikLayout l;
    l.ld = ld_for(N);
    l.mat_elems = (size_t)(N + 1) * l.ld;            // + the border row that carries g through the factorisation
    l.per_item_bytes = l.mat_elems * sizeof(double) + (size_t)NB * NB * sizeof(double) + 2 * (size_t)env_blocks(N) * sizeof(int);
    l.fixed_bytes = align_up((size_t)B * sizeof(double), 256)      // jitter
                    + align_up((size_t)B * sizeof(int), 256)       // map
                    + 256                                          // count
                    + align_up((size_t)32 * l.ld * sizeof(double), 256);   // z scratch of the small-batch solve
    return l;
}

// Envelope skips (gpmc_set_tuning(14, .)): -1 until set, then the GPMC_ENVELOPE environment variable decides once
static int g_envelope = -1;
bool envelope_enabled()
{
    if (g_envelope < 0) {
        const char *e = getenv("GPMC_ENVELOPE");
        g_envelope = (e && e[0] == '0') ? 0 : 1;
    }
    return g_envelope != 0;
}

// Band-only assembly and launches (gpmc_set_tuning(15, .), GPMC_BAND), and where the region left of the band is cleared
// (gpmc_set_tuning(16, .), GPMC_BAND_CLEAR): 2 = inline in the assembly (default: measured faster on the bench workload,
// profiles/r03b_band_ab.json), 1 = side stream, 0 = not at all
static int g_band = -1, g_band_clear = -1, g_band_compact = -1;
bool band_enabled()
{
    if (g_band < 0) {
        const char *e = getenv("GPMC_BAND");
        g_band = (e && e[0] == '0') ? 0 : 1;
    }
    // a band leaves the matrix unwritten left of it: only the update and solve kernels that start at the envelope keep
    // their reads inside it (the other tile-kernel variants and the 32-column panel solve read whole rows)
    return g_band != 0 && gemm_honours_envelope() && trsm_honours_envelope();
}
// Compact band storage (gpmc_set_tuning(17, .), GPMC_BAND_COMPACT): 1 = automatic (default), 0 = always the dense layout
static bool band_compact_allowed()
{
    if (g_band_compact < 0) {
        const char *e = getenv("GPMC_BAND_COMPACT");
        g_band_compact = (e && e[0] == '0') ? 0 : 1;
    }
    return g_band_compact != 0;
}
// layout of the last gpmc_loglik_batched call (gpmc_loglik_layout)
static int g_last_W = 0, g_last_waves = 0;

static int band_clear_mode()
{
    if (g_band_clear < 0) {
        const char *e = getenv("GPMC_BAND_CLEAR");
        g_band_clear = (e && e[0] >= '0' && e[0] <= '2') ? e[0] - '0' : 2;
    }
    return g_band_clear;
}

// The band clear runs on a low-priority side stream per device: it starts after the band bound of its wave and the
// caller's stream waits for it before the next wave's bound and before gpmc_loglik_batched returns.
struct ClearStream {
    cudaStream_t s = nullptr;
    cudaEvent_t start = nullptr, done = nullptr;
    bool ok = false;
};
static ClearStream *clear_stream()
{
    static ClearStream cs[64];
    static bool tried[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    if (!tried[dev]) {
        tried[dev] = true;
        int lo = 0, hi = 0;
        ClearStream &c = cs[dev];
        bool ok = cudaDeviceGetStreamPriorityRange(&lo, &hi) == cudaSuccess;
        ok = ok && cudaStreamCreateWithPriority(&c.s, cudaStreamNonBlocking, lo) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&c.start, cudaEventDisableTiming) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&c.done, cudaEventDisableTiming) == cudaSuccess;
        c.ok = ok;
    }
    return cs[dev].ok ? &cs[dev] : nullptr;
}
// the caller's stream waits for an issued clear on every way out of gpmc_loglik_batched (errors included)
struct ClearJoin {
    cudaStream_t s;
    ClearStream *cs = nullptr;
    bool pending = false;
    ~ClearJoin() { if (pending) cudaStreamWaitEvent(s, cs->done, 0); }
};

// Assemble-and-factor one wave with kcGP.tools.jitchol semantics (pyGPs 1.3.4): one plain attempt for every item, then --
// for the items that failed only -- any(diag <= 0) -> GPMC_INFO_NOT_PD, else the ladder mean(diag) * 1e-6 * 10^k, k < 5,
// re-assembling the item with the jitter on its diagonal.  `fill` assembles the listed items INCLUDING their border
// rows; `diag_value` is the (constant) diagonal of an item's matrix from its hyper-parameter row.
int factor_wave(const std::function<int(BatchView, int, const double *)> &fill, const std::function<double(const double *)> &diag_value,
                BatchView A, int N, int nb, const double *hyp_w, int P, int *info_w, double *W, double *jit_dev, int *map_dev,
                int jitter_policy, int border_rows, cudaStream_t s, int fuse, Envelope env, long long w_step)
{
    // w_step = NB*NB keeps every diagonal-block inverse (item stride: all block columns' worth), as inverse_sequence needs
    const long long strideW = w_step ? (long long)((N + NB - 1) / NB) * w_step : NB * NB;
    int rc = fill(A, nb, nullptr);
    if (rc) return rc;
    if ((rc = potrf_sequence(A, N, nb, info_w, W, strideW, w_step, 0, s, border_rows, fuse, env))) return rc;
    if (jitter_policy != GPMC_JITTER_PYGPS) return 0;
    std::vector<int> info(nb);
    GPMC_CUDA_CHECK(cudaMemcpyAsync(info.data(), info_w, nb * sizeof(int), cudaMemcpyDeviceToHost, s));
    GPMC_CUDA_CHECK(cudaStreamSynchronize(s));
    std::vector<int> todo;
    for (int i = 0; i < nb; ++i) if (info[i] != 0) todo.push_back(i);
    if (todo.empty()) return 0;
    std::vector<double> hyp_host((size_t)nb * P);
    GPMC_CUDA_CHECK(cudaMemcpyAsync(hyp_host.data(), hyp_w, (size_t)nb * P * sizeof(double), cudaMemcpyDeviceToHost, s));
    GPMC_CUDA_CHECK(cudaStreamSynchronize(s));
    std::vector<double> jit(nb, 0.0);
    std::vector<int> keep;
    for (int i : todo) {
        const double dv = diag_value(&hyp_host[(size_t)i * P]);
        if (dv <= 0.0) info[i] = GPMC_INFO_NOT_PD;       // any(diag <= 0): LinAlgError
        else { jit[i] = dv * 1e-6; keep.push_back(i); }   // NaN diag also lands here and keeps failing
    }
    todo.swap(keep);
    for (int attempt = 0; attempt < 5 && !todo.empty(); ++attempt) {
        const int nf = (int)todo.size();
        GPMC_CUDA_CHECK(cudaMemcpyAsync(map_dev, todo.data(), nf * sizeof(int), cudaMemcpyHostToDevice, s));
        GPMC_CUDA_CHECK(cudaMemcpyAsync(jit_dev, jit.data(), nb * sizeof(double), cudaMemcpyHostToDevice, s));
        for (int i : todo) info[i] = 0;
        GPMC_CUDA_CHECK(cudaMemcpyAsync(info_w, info.data(), nb * sizeof(int), cudaMemcpyHostToDevice, s));
        BatchView Am = A;                               // the failed items, re-assembled in place
        Am.map = map_dev;
        Am.count = nullptr;
        if ((rc = fill(Am, nf, jit_dev))) return rc;
        if ((rc = potrf_sequence(Am, N, nf, info_w, W, strideW, w_step, 0, s, border_rows, fuse, env))) return rc;
        GPMC_CUDA_CHECK(cudaMemcpyAsync(info.data(), info_w, nb * sizeof(int), cudaMemcpyDeviceToHost, s));
        GPMC_CUDA_CHECK(cudaStreamSynchronize(s));
        std::vector<int> still;
        for (int i : todo) if (info[i] != 0) { still.push_back(i); jit[i] *= 10.0; }
        todo.swap(still);
    }
    for (int i : todo) info[i] = GPMC_INFO_NOT_PD;
    GPMC_CUDA_CHECK(cudaMemcpyAsync(info_w, info.data(), nb * sizeof(int), cudaMemcpyHostToDevice, s));
    GPMC_CUDA_CHECK(cudaStreamSynchronize(s));
    return 0;
}

}  // namespace gpmc

using namespace gpmc;

extern "C" {

int gpmc_version(void) { return GPMC_VERSION; }
int gpmc_panel_width(void) { return NB; }
const char *gpmc_last_error(void) { return g_err; }

int gpmc_device_info(int *sm_count, int *cc_major, int *cc_minor, size_t *hbm_bytes)
{
    int dev = 0;
    GPMC_CUDA_CHECK(cudaGetDevice(&dev));
    cudaDeviceProp p;
    GPMC_CUDA_CHECK(cudaGetDeviceProperties(&p, dev));
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (cc_major) *cc_major = p.major;
    if (cc_minor) *cc_minor = p.minor;
    if (hbm_bytes) *hbm_bytes = p.totalGlobalMem;
    return 0;
}

size_t gpmc_workspace_bytes(int op, int N, int D, int B)
{
    if (N <= 0 || B <= 0) return 0;
    const size_t w = (size_t)NB * NB * sizeof(double);
    if (op == GPMC_OP_POTRF) {
        // W per item + (for the jitter ladder) a backup of every matrix + ladder scratch
        // (sized for a caller ld <= N rounded up to 16)
        return (size_t)B * w + (size_t)B * (size_t)N * (size_t)ld_for(N) * sizeof(double)
               + 4 * align_up((size_t)B * sizeof(double), 256) + 256;
    }
    if (op == GPMC_OP_LOGLIK) {
        const LoglikLayout l = loglik_layout(N, B);
        // recommended wave: as many items as fit in 48 GiB (large waves amortise the panel kernels' latency and the
        // per-wave host synchronisation of the jitter check), at most 8192
        const size_t cap = (size_t)48 << 30;
        size_t wave = std::min<size_t>(std::min<size_t>(B, 8192), std::max<size_t>(1, cap / l.per_item_bytes));
        return l.fixed_bytes + wave * l.per_item_bytes;
    }
    if (op == GPMC_OP_LOGLIK_GRAD) return loglik_grad_workspace_bytes(N, D, B);
    return 0;
}

int gpmc_cov_assemble(const double *x_dev, int N, int D, const double *hyp_dev, int B, int P, int kind, int flags,
                      const double *jitter_dev, double *A_dev, int ld, void *stream)
{
    GPMC_API_LOCK();
    const int n_ell = (kind == GPMC_KIND_SE_ARD) ? D : 1;
    if (N <= 0 || D <= 0 || B < 0 || P != n_ell + 2) { set_error("cov_assemble: bad shape N=%d D=%d B=%d P=%d kind=%d", N, D, B, P, kind); return GPMC_EINVAL; }
    if (ld < N || (ld & 1)) { set_error("cov_assemble: ld=%d must be even and >= N=%d", ld, N); return GPMC_EALIGN; }
    BatchView A{A_dev, (long long)N * ld, ld, nullptr, nullptr};
    return launch_cov_assemble(x_dev, N, D, hyp_dev, P, n_ell, flags, jitter_dev, A, B, (cudaStream_t)stream);
}

int gpmc_potrf_batched(double *A_dev, int N, int ld, int B, int *info_dev, int jitter_policy, int zero_upper,
                       void *ws_dev, size_t ws_bytes, void *stream)
{
    GPMC_API_LOCK();
    cudaStream_t s = (cudaStream_t)stream;
    if (N <= 0 || B < 0) { set_error("potrf: bad shape N=%d B=%d", N, B); return GPMC_EINVAL; }
    if (B == 0) return 0;
    if (ld < N || (ld & 1)) { set_error("potrf: ld=%d must be even and >= N=%d (pad the matrix)", ld, N); return GPMC_EALIGN; }
    const size_t wbytes = (size_t)B * NB * NB * sizeof(double);
    const size_t mat_bytes = (size_t)B * N * ld * sizeof(double);
    if (B > MAX_BATCH_ITEMS) { set_error("potrf: B=%d exceeds %d items per call (grid.y limit); split the batch", B, MAX_BATCH_ITEMS); return GPMC_EINVAL; }
    const size_t need = wbytes + (jitter_policy == GPMC_JITTER_PYGPS ? mat_bytes + 4 * align_up((size_t)B * sizeof(double), 256) + 256 : 0);
    if (!ws_dev || ws_bytes < need) { set_error("potrf: workspace %zu < %zu bytes", ws_bytes, need); return GPMC_ENOMEM; }
    char *wp = (char *)ws_dev;
    double *W = (double *)wp; wp += wbytes;
    BatchView A{A_dev, (long long)N * ld, ld, nullptr, nullptr};
    { int rc0 = fill_int(info_dev, 0, B, s); if (rc0) return rc0; }

    const int fuse = potrf_fuse_auto(N, B, 0);
    if (jitter_policy != GPMC_JITTER_PYGPS) return potrf_sequence(A, N, B, info_dev, W, NB * NB, 0, zero_upper, s, 0, fuse);

    // pyGPs jitchol: keep a copy, try once, then the jitter ladder on the items that failed.
    double *backup = (double *)wp; wp += mat_bytes;
    double *mean_dev = (double *)wp; wp += align_up((size_t)B * sizeof(double), 256);
    double *jit_dev = (double *)wp; wp += align_up((size_t)B * sizeof(double), 256);
    int *map_dev = (int *)wp; wp += align_up((size_t)B * sizeof(int), 256);
    int *bad_dev = (int *)wp;
    GPMC_CUDA_CHECK(cudaMemcpyAsync(backup, A_dev, mat_bytes, cudaMemcpyDeviceToDevice, s));
    int rc = potrf_sequence(A, N, B, info_dev, W, NB * NB, 0, zero_upper, s, 0, fuse);
    if (rc) return rc;
    std::vector<int> info(B);
    GPMC_CUDA_CHECK(cudaMemcpyAsync(info.data(), info_dev, B * sizeof(int), cudaMemcpyDeviceToHost, s));
    GPMC_CUDA_CHECK(cudaStreamSynchronize(s));
    std::vector<int> failed;
    for (int i = 0; i < B; ++i) if (info[i] != 0) failed.push_back(i);
    if (failed.empty()) return 0;

    // diag statistics of the ORIGINAL matrices
    BatchView Bk{backup, (long long)N * ld, ld, nullptr, nullptr};
    { int rc0 = diag_stats(Bk, N, mean_dev, bad_dev, B, s); if (rc0) return rc0; }
    std::vector<double> mean(B);
    std::vector<int> bad(B);
    GPMC_CUDA_CHECK(cudaMemcpyAsync(mean.data(), mean_dev, B * sizeof(double), cudaMemcpyDeviceToHost, s));
    GPMC_CUDA_CHECK(cudaMemcpyAsync(bad.data(), bad_dev, B * sizeof(int), cudaMemcpyDeviceToHost, s));
    GPMC_CUDA_CHECK(cudaStreamSynchronize(s));
    std::vector<double> jit(B, 0.0);
    std::vector<int> todo;
    for (int i : failed) {
        if (bad[i]) info[i] = GPMC_INFO_NOT_PD;          // "not pd: non-positive diagonal elements"
        else { jit[i] = mean[i] * 1e-6; todo.push_back(i); }
    }
    for (int attempt = 0; attempt < 5 && !todo.empty(); ++attempt) {
        const int nf = (int)todo.size();
        GPMC_CUDA_CHECK(cudaMemcpyAsync(map_dev, todo.data(), nf * sizeof(int), cudaMemcpyHostToDevice, s));
        GPMC_CUDA_CHECK(cudaMemcpyAsync(jit_dev, jit.data(), B * sizeof(double), cudaMemcpyHostToDevice, s));
        BatchView Am{A_dev, (long long)N * ld, ld, map_dev, nullptr};
        restore_jitter_kernel<<<dim3(64, nf), 256, 0, s>>>(Am, backup, N, jit_dev);
        GPMC_LAUNCH_CHECK();
        for (int i : todo) info[i] = 0;
        GPMC_CUDA_CHECK(cudaMemcpyAsync(info_dev, info.data(), B * sizeof(int), cudaMemcpyHostToDevice, s));
        rc = potrf_sequence(Am, N, nf, info_dev, W, NB * NB, 0, zero_upper, s);
        if (rc) return rc;
        GPMC_CUDA_CHECK(cudaMemcpyAsync(info.data(), info_dev, B * sizeof(int), cudaMemcpyDeviceToHost, s));
        GPMC_CUDA_CHECK(cudaStreamSynchronize(s));
        std::vector<int> still;
        for (int i : todo) if (info[i] != 0) { still.push_back(i); jit[i] *= 10.0; }
        todo.swap(still);
    }
    for (int i : todo) info[i] = GPMC_INFO_NOT_PD;        // "not positive definite, even with jitter."
    GPMC_CUDA_CHECK(cudaMemcpyAsync(info_dev, info.data(), B * sizeof(int), cudaMemcpyHostToDevice, s));
    GPMC_CUDA_CHECK(cudaStreamSynchronize(s));
    return 0;
}

int gpmc_loglik_batched(const double *x_dev, int N, int D, const double *g_dev, const double *hyp_dev, int B, int P,
                        int kind, int jitter_policy, double *loglik_dev, int *info_dev, void *ws_dev, size_t ws_bytes,
                        void *stream)
{
    GPMC_API_LOCK();
    cudaStream_t s = (cudaStream_t)stream;
    const int n_ell = (kind == GPMC_KIND_SE_ARD) ? D : 1;
    if (N <= 0 || D <= 0 || B < 0 || P != n_ell + 2) { set_error("loglik: bad shape N=%d D=%d B=%d P=%d kind=%d", N, D, B, P, kind); return GPMC_EINVAL; }
    if (B == 0) return 0;
    const LoglikLayout l = loglik_layout(N, B);
    if (!ws_dev || ws_bytes < l.fixed_bytes + l.per_item_bytes) {
        set_error("loglik: workspace %zu bytes cannot hold one item (%zu needed)", ws_bytes, l.fixed_bytes + l.per_item_bytes);
        return GPMC_ENOMEM;
    }
    char *wp = (char *)ws_dev;
    double *jit_dev = (double *)wp; wp += align_up((size_t)B * sizeof(double), 256);
    int *map_dev = (int *)wp; wp += align_up((size_t)B * sizeof(int), 256);
    int *band_dev = (int *)wp; wp += 256;                          // band bound: max r - lo[r], max r - w[r]
    double *xbox = (double *)wp;                                    // band bound: boxes of x (2 D env_blocks(N) <= 32 ld doubles)
    wp += align_up((size_t)32 * l.ld * sizeof(double), 256);
    const size_t wave_cap = std::min<size_t>((ws_bytes - l.fixed_bytes) / l.per_item_bytes, (size_t)MAX_BATCH_ITEMS);   // items ride in grid.y
    const int wave = (int)std::min<size_t>(wave_cap, (size_t)B);
    g_last_W = 0;
    g_last_waves = (B + wave - 1) / wave;
    { int rc0 = fill_int(info_dev, 0, B, s); if (rc0) return rc0; }

    // Compact band layout: when the dense layout needs several waves, bound the band of every item of the call first.
    // Rows W = 128 + 64 * (widest band) columns wide hold every element the factorisation reads (see BatchView, Band); it
    // is used when it needs fewer waves and those waves run the plain left-looking schedule (the kernels that know it).
    if (wave < B && band_compact_allowed() && envelope_enabled() && band_enabled()) {
        const int nblk = env_blocks(N);
        const size_t wenv = align_up((size_t)B * nblk * sizeof(int), 256);
        char *cp = wp;
        int *w_all = (int *)cp; cp += wenv;              // band starts of every item of the call
        int *env_all = (int *)cp; cp += wenv;            // envelopes of every item of the call
        const size_t room = ws_bytes - l.fixed_bytes;
        if (2 * wenv + 256 < room) {
            GPMC_CUDA_CHECK(cudaMemsetAsync(band_dev, 0, 2 * sizeof(int), s));
            int rc = launch_band_bound(x_dev, N, D, hyp_dev, P, n_ell, B, w_all, nblk, band_dev, xbox, s);
            if (rc) return rc;
            int bh[2] = {0, 0};
            GPMC_CUDA_CHECK(cudaMemcpyAsync(bh, band_dev, sizeof(bh), cudaMemcpyDeviceToHost, s));
            GPMC_CUDA_CHECK(cudaStreamSynchronize(s));
            const int Wc = (int)align_up((size_t)BAND_ROWS + (size_t)ENV_ROWS * bh[1], 16);
            // per item: the rows, the border row and the panel factor's scratch
            const size_t per_item = (size_t)N * Wc * sizeof(double) + (size_t)l.ld * sizeof(double) + (size_t)NB * NB * sizeof(double);
            const size_t wave_c = std::min<size_t>((room - 2 * wenv - 256) / per_item, (size_t)MAX_BATCH_ITEMS);   // 256: the border rows' alignment
            const int waves_c = wave_c > 0 ? (int)((B + wave_c - 1) / wave_c) : 0;
            // equal waves (sizes differ by one at most), so that every wave runs the same schedule
            const int nb_lo = waves_c > 0 ? B / waves_c : 0, nb_hi = waves_c > 0 ? (B + waves_c - 1) / waves_c : 0;
            if (Wc < l.ld && waves_c > 0 && waves_c < g_last_waves && potrf_compact_ok(N, nb_lo) && potrf_compact_ok(N, nb_hi)) {
                double *border = (double *)cp; cp += align_up((size_t)nb_hi * l.ld * sizeof(double), 256);
                double *Wsc = (double *)cp; cp += (size_t)nb_hi * NB * NB * sizeof(double);
                double *mats_c = (double *)cp;
                g_last_W = Wc;
                g_last_waves = waves_c;
                for (int wi = 0, s0 = 0; wi < waves_c; ++wi) {
                    const int nb = nb_lo + (wi < B % waves_c ? 1 : 0);
                    BatchView A{mats_c, (long long)N * Wc, Wc, nullptr, nullptr, Wc, N, border, l.ld};
                    const Envelope env{env_all + (size_t)s0 * nblk, nblk, N, bh[0]};
                    const Band band{w_all + (size_t)s0 * nblk, nblk, bh[1], 0};
                    const double *hyp_w = hyp_dev + (size_t)s0 * P;
                    const double *g_w = g_dev + (size_t)s0 * N;
                    int *info_w = info_dev + s0;
                    auto fill = [&](BatchView V, int nitems, const double *jit) -> int {
                        int rc = launch_cov_assemble(x_dev, N, D, hyp_w, P, n_ell, GPMC_ASM_ADD_S | GPMC_ASM_LOWER_ONLY, jit, V, nitems, s, env, band);
                        if (rc) return rc;
                        return border_set(V, N, g_w, N, nitems, s);
                    };
                    auto diag = [&](const double *h) { return host_diag_value(h, n_ell); };
                    rc = factor_wave(fill, diag, A, N, nb, hyp_w, P, info_w, Wsc, jit_dev, map_dev, jitter_policy, 1, s, potrf_fuse_compact(), env);
                    if (rc) return rc;
                    if ((rc = border_finish(A, N, loglik_dev + s0, info_w, nb, s, 0))) return rc;
                    s0 += nb;
                }
                return 0;
            }
        }
    }

    double *mats = (double *)wp;
    double *W = (double *)(wp + (size_t)wave * l.mat_elems * sizeof(double));
    const Envelope env_ws{(int *)(W + (size_t)wave * NB * NB), env_blocks(N), N};
    int *band_w = env_ws.blk + (size_t)wave * env_blocks(N);
    ClearJoin clear{s};

    for (int s0 = 0; s0 < B; s0 += wave) {
        const int nb = std::min(wave, B - s0);
        const double *hyp_w = hyp_dev + (size_t)s0 * P;
        const double *g_w = g_dev + (size_t)s0 * N;
        int *info_w = info_dev + s0;
        BatchView A{mats, (long long)l.mat_elems, l.ld, nullptr, nullptr};
        const int fuse = potrf_fuse_auto(N, nb, 1);
        // The fused panel launches (many small matrices) ignore the envelope, and the few short update contractions of
        // those matrices save less than recording and reading it costs (N=512 x 4096, ARD: 1 % slower): dense there.
        Envelope env = (envelope_enabled() && !fuse) ? env_ws : Envelope{};
        // Band: a bound taken before the assembly says which tiles can hold a nonzero; only those (widened, see Band) are
        // assembled, and the update GEMM and the panel solve launch only the rows of the widest band of the wave.  The
        // zeros left of the band are stored by a clear that nothing on the factorisation path waits for.
        Band band{};
        int rc = 0;
        if (env.blk && band_enabled()) {
            const int mode = band_clear_mode();
            if (clear.pending) {                        // the previous wave's clear still writes these buffers
                GPMC_CUDA_CHECK(cudaStreamWaitEvent(s, clear.cs->done, 0));
                clear.pending = false;
            }
            GPMC_CUDA_CHECK(cudaMemsetAsync(band_dev, 0, 2 * sizeof(int), s));
            rc = launch_band_bound(x_dev, N, D, hyp_w, P, n_ell, nb, band_w, env_blocks(N), band_dev, xbox, s);
            if (rc) return rc;
            // The launch sizes need the band on the host: one synchronisation.  The inline clear's assembly grid does not,
            // and with few matrices in flight the update and solve launches are small anyway (N=16384 x 1 measured 0.3 %
            // slower with the read-back), so such waves keep full launch grids.
            int bh[2] = {-1, 0};
            if (mode != 2 || (long long)nb * ((N + NB - 1) / NB) >= 1024) {
                GPMC_CUDA_CHECK(cudaMemcpyAsync(bh, band_dev, sizeof(bh), cudaMemcpyDeviceToHost, s));
                GPMC_CUDA_CHECK(cudaStreamSynchronize(s));
            }
            env.band = bh[0];
            band = Band{band_w, env_blocks(N), bh[1], mode == 2};
            if (mode == 1) {
                ClearStream *cs = clear.cs ? clear.cs : (clear.cs = clear_stream());
                if (!cs) { set_error("loglik: the band clear stream could not be created"); return GPMC_EINVAL; }
                GPMC_CUDA_CHECK(cudaEventRecord(cs->start, s));
                GPMC_CUDA_CHECK(cudaStreamWaitEvent(cs->s, cs->start, 0));
                BatchView Aw{mats, (long long)l.mat_elems, l.ld, nullptr, nullptr};
                if ((rc = launch_band_clear(Aw, N, band, nb, cs->s))) return rc;
                GPMC_CUDA_CHECK(cudaEventRecord(cs->done, cs->s));
                clear.pending = true;
            }
        }
        auto fill = [&](BatchView V, int nitems, const double *jit) -> int {
            int rc = launch_cov_assemble(x_dev, N, D, hyp_w, P, n_ell, GPMC_ASM_ADD_S | GPMC_ASM_LOWER_ONLY, jit, V, nitems, s, env, band);
            if (rc) return rc;
            return border_set(V, N, g_w, N, nitems, s);
        };
        auto diag = [&](const double *h) { return host_diag_value(h, n_ell); };
        rc = factor_wave(fill, diag, A, N, nb, hyp_w, P, info_w, W, jit_dev, map_dev, jitter_policy, 1, s, fuse, env);
        if (rc) return rc;
        // z = L^-1 g sits in the border row except for the last column block: finish it, then quad form + log det
        rc = border_finish(A, N, loglik_dev + s0, info_w, nb, s, fuse);
        if (rc) return rc;
    }
    return 0;
}

// ------------------------------------------------------------------------------ host-buffer path
struct HostPath {
    cudaStream_t stream = nullptr;
    void *dev = nullptr;  size_t dev_bytes = 0;     // x, g, hyp, loglik, info
    void *ws = nullptr;   size_t ws_bytes = 0;
    void *pin = nullptr;  size_t pin_bytes = 0;
};
static HostPath g_hp;

static int ensure(void **p, size_t *have, size_t need, bool pinned)
{
    if (*have >= need) return 0;
    if (*p) { if (pinned) cudaFreeHost(*p); else cudaFree(*p); *p = nullptr; *have = 0; }
    cudaError_t e = pinned ? cudaMallocHost(p, need) : cudaMalloc(p, need);
    if (e != cudaSuccess) { set_error("allocation of %zu bytes failed: %s", need, cudaGetErrorString(e)); return (int)e; }
    *have = need;
    return 0;
}

int gpmc_loglik_host(const double *x_host, int N, int D, const double *g_host, const double *hyp_host, int B, int P,
                     int kind, int jitter_policy, double *loglik_host, int *info_host)
{
    GPMC_API_LOCK();
    if (N <= 0 || D <= 0 || B <= 0) { set_error("loglik_host: bad shape"); return GPMC_EINVAL; }
    if (!g_hp.stream) GPMC_CUDA_CHECK(cudaStreamCreateWithFlags(&g_hp.stream, cudaStreamNonBlocking));
    cudaStream_t s = g_hp.stream;
    const size_t bx = align_up((size_t)N * D * 8, 256), bg = align_up((size_t)B * N * 8, 256), bh = align_up((size_t)B * P * 8, 256);
    const size_t bl = align_up((size_t)B * 8, 256), bi = align_up((size_t)B * 4, 256);
    const size_t io = bx + bg + bh + bl + bi;
    int rc = ensure(&g_hp.dev, &g_hp.dev_bytes, io, false);
    if (rc) return rc;
    rc = ensure(&g_hp.pin, &g_hp.pin_bytes, io, true);
    if (rc) return rc;
    // workspace: as many items per wave as half of the free memory allows
    size_t want = gpmc_workspace_bytes(GPMC_OP_LOGLIK, N, D, B);
    if (g_hp.ws_bytes < want) {
        size_t free_b = 0, total_b = 0;
        GPMC_CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
        free_b += g_hp.ws_bytes;
        const LoglikLayout l = loglik_layout(N, B);
        const size_t floor_b = l.fixed_bytes + l.per_item_bytes;
        size_t take = std::min(want, free_b / 2);
        if (take < floor_b) take = floor_b;
        rc = ensure(&g_hp.ws, &g_hp.ws_bytes, take, false);
        if (rc) return rc;
    }
    char *pin = (char *)g_hp.pin, *dev = (char *)g_hp.dev;
    memcpy(pin, x_host, (size_t)N * D * 8);
    memcpy(pin + bx, g_host, (size_t)B * N * 8);
    memcpy(pin + bx + bg, hyp_host, (size_t)B * P * 8);
    GPMC_CUDA_CHECK(cudaMemcpyAsync(dev, pin, bx + bg + bh, cudaMemcpyHostToDevice, s));
    rc = gpmc_loglik_batched((const double *)dev, N, D, (const double *)(dev + bx), (const double *)(dev + bx + bg), B, P, kind,
                             jitter_policy, (double *)(dev + bx + bg + bh), (int *)(dev + bx + bg + bh + bl), g_hp.ws,
                             g_hp.ws_bytes, s);
    if (rc) return rc;
    GPMC_CUDA_CHECK(cudaMemcpyAsync(pin + bx + bg + bh, dev + bx + bg + bh, bl + bi, cudaMemcpyDeviceToHost, s));
    GPMC_CUDA_CHECK(cudaStreamSynchronize(s));
    memcpy(loglik_host, pin + bx + bg + bh, (size_t)B * 8);
    if (info_host) memcpy(info_host, pin + bx + bg + bh + bl, (size_t)B * 4);
    return 0;
}

int gpmc_bench_fp64_peak(int which, int iters, double *tflops_out, double *ms_out)
{
    GPMC_API_LOCK();
    double tf = 0.0, ms = 0.0;
    const int rc = run_fp64_peak(which, iters, &tf, &ms);
    if (tflops_out) *tflops_out = tf;
    if (ms_out) *ms_out = ms;
    return rc;
}

int gpmc_bench_dmma_ilp(int nacc, int warps_per_sm, int iters, double *tflops_out)
{
    GPMC_API_LOCK();
    double tf = 0.0;
    const int rc = run_dmma_ilp(nacc, warps_per_sm, iters, &tf);
    if (tflops_out) *tflops_out = tf;
    return rc;
}

int gpmc_set_tuning(int key, int value)
{
    GPMC_API_LOCK();
    if (key == 0) { set_gemm_config(value); return 0; }
    if (key == 1) { set_potf2_mode(value); return 0; }
    if (key == 2) { set_lookahead_mode(value); return 0; }
    if (key == 3) { set_potrf_window(value); return 0; }
    if (key == 4) { set_trsm_mode(value); return 0; }
    if (key == 5) { set_trsm_blocks_per_cta(value); return 0; }
    if (key == 6) { set_sds_mode(value); return 0; }
    if (key == 7) { set_sds_runahead(value); return 0; }
    if (key == 8) { set_sds_literal(value); return 0; }
    if (key == 9) { set_panel_fuse(value); return 0; }
    if (key == 10) { set_lookahead_split(value); return 0; }
    if (key == 11) { set_inverse_window(value); return 0; }
    if (key == 13) { set_sds_pin_schedule(value); return 0; }
    if (key == 14) { g_envelope = value != 0; return 0; }
    if (key == 15) { g_band = value != 0; return 0; }
    if (key == 16) { if (value < 0 || value > 2) return GPMC_EINVAL; g_band_clear = value; return 0; }
    if (key == 17) { g_band_compact = value != 0; return 0; }
    return GPMC_EINVAL;
}

int gpmc_loglik_layout(int *band_W, int *waves)
{
    GPMC_API_LOCK();
    if (band_W) *band_W = g_last_W;
    if (waves) *waves = g_last_waves;
    return 0;
}

int gpmc_sds_loop_stats(long long *rounds, long long *idle_rounds, long long *ladders)
{
    GPMC_API_LOCK();
    sds_loop_stats(rounds, idle_rounds, ladders);
    return 0;
}

int gpmc_profile_enable(int on) { GPMC_API_LOCK(); g_prof_on = (on != 0); return 0; }

int gpmc_profile_reset(void)
{
    GPMC_API_LOCK();
    for (int k = 0; k < KC_COUNT; ++k) g_used[k] = 0;
    return 0;
}

int gpmc_profile_read(int kernel_class, double *total_ms, long long *launches)
{
    GPMC_API_LOCK();
    if (kernel_class < 0 || kernel_class >= KC_COUNT) return GPMC_EINVAL;
    GPMC_CUDA_CHECK(cudaDeviceSynchronize());
    double tot = 0.0;
    for (size_t i = 0; i < g_used[kernel_class]; ++i) {
        float ms = 0.f;
        GPMC_CUDA_CHECK(cudaEventElapsedTime(&ms, g_pool[kernel_class][i].a, g_pool[kernel_class][i].b));
        tot += ms;
    }
    if (total_ms) *total_ms = tot;
    if (launches) *launches = (long long)g_used[kernel_class];
    return 0;
}

// every recorded launch of one class as (start, end) in ms after `origin_class`'s first launch began (its order in the
// returned list is the order of the launches); returns the number of intervals written
int gpmc_profile_timeline(int kernel_class, int origin_class, double *start_end_ms, long long capacity, long long *written)
{
    GPMC_API_LOCK();
    if (kernel_class < 0 || kernel_class >= KC_COUNT || origin_class < 0 || origin_class >= KC_COUNT || !start_end_ms || !written)
        return GPMC_EINVAL;
    if (g_used[origin_class] == 0) { set_error("gpmc_profile_timeline: no launch of the origin class recorded"); return GPMC_EINVAL; }
    GPMC_CUDA_CHECK(cudaDeviceSynchronize());
    const cudaEvent_t t0 = g_pool[origin_class][0].a;
    long long w = 0;
    for (size_t i = 0; i < g_used[kernel_class] && w < capacity; ++i, ++w) {
        float a = 0.f, b = 0.f;
        GPMC_CUDA_CHECK(cudaEventElapsedTime(&a, t0, g_pool[kernel_class][i].a));
        GPMC_CUDA_CHECK(cudaEventElapsedTime(&b, t0, g_pool[kernel_class][i].b));
        start_end_ms[2 * w] = a;
        start_end_ms[2 * w + 1] = b;
    }
    *written = w;
    return 0;
}

}  // extern "C"
