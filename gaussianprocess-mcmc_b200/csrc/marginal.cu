// gpmc_marginal_run: slice sampling of the GP hyper-parameters with the latent f integrated out (Gaussian likelihood).
// The target is p(theta | y) ~ N(y - m; 0, K_theta + S_theta) * prod_p prior_p(theta_p): the log-likelihood unit of
// gpmc_loglik_batched plus the hyper-priors of sliceSample.py:209-232.  The transition is the reference's hyper-rectangle
// slice sampler (kcMCMC/sliceSample.py:110-163) without f, g and the truncated-Gaussian term:
//
//   marginal_begin    :110-112  bracket [hyp_min, hyp_max];  :127-129 threshold log u0 + priors + G_cur
//   marginal_propose  :132-134  theta' ~ U(hyp_min, hyp_max), noise frozen while iter < burn_in
//   loglik_batched              G' = log N(y - m; 0, K + S) at every active chain's theta' (y - m shared by all items)
//   marginal_accept   :149-163  priors + G', accept / shrink; a finished transition starts the chain's next one in place
//   marginal_compact            order-preserving list of the chains still inside a transition
//
// A chain's state is O(P) (theta, bracket, threshold, the G of its current theta, iteration, trips), so every chain of the
// call stays in flight and goes through its transitions on its own; each round evaluates one proposal per active chain.
// G_cur is carried from the accepted proposal: the log-likelihood at the current theta is evaluated once per call.
// Randomness is keyed by (seed, chain0 + chain, iteration) on the streams of the surrogate-data sampler (sds.cu), so a
// chain draws the v, u0 and U that gpmc_sds_run would draw for it, or comes from explicit tapes.
#include "common.cuh"
#include "sequences.cuh"
#include "slice_common.cuh"
#include "../../include/gpmc.h"

#include <algorithm>
#include <chrono>
#include <vector>

namespace gpmc {

struct MarginalState {
    int P, B, n_iters, iter_begin, burn_in, max_trips;
    unsigned long long seed;
    unsigned chain0;
    const double *scale, *prior_k, *prior_theta;   // [P]
    double *hyp;                   // [B, P] the caller's state (in / out)
    double *hyp_min, *hyp_max;     // [B, P]
    double *prop;                  // [B, P] proposals of the round, in active-list order
    double *ll;                    // [B]    log-likelihood of the round, in active-list order
    double *curG, *threshold;      // [B]
    int *k, *trips, *done, *exhausted;   // [B]
    int *info;                     // [B]    status of the round's factorisations (not read: a failed item has G = NaN)
    int *map, *count;              // active list
    double *hist_hyp, *hist_loglik;      // [B, n_iters, P], [B, n_iters] (may be nullptr)
    int *hist_trips;               // [B, n_iters] (may be nullptr)
    const double *tape_v, *tape_u0, *tape_U;   // [B, n_iters, P], [B, n_iters], [B, n_iters, T, P] (all nullptr: Philox)
    int tape_trips;
};

__global__ void marginal_center_kernel(const double *__restrict__ y, double m, int n, double *__restrict__ out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = y[i] - m;
}

// New transition of chain c at MCMC iteration iter_begin + k[c]: bracket (:110-112) and threshold (:127-129) from the
// carried G of the chain's current theta.
__device__ void marginal_begin(const MarginalState &st, int c)
{
    const int P = st.P, k = st.k[c], it = st.iter_begin + k;
    const double *hyp = st.hyp + (size_t)c * P;
    const size_t t = (size_t)c * st.n_iters + k;
    for (int p = 0; p < P; ++p) {
        double u, u1;
        if (st.tape_v) u = st.tape_v[t * P + p];
        else philox_uniform2(st.seed, st.chain0 + c, (unsigned)it, STREAM_BRACKET, p, u, u1);
        const double v = 0.0 + (st.scale[p] - 0.0) * u;
        const double lo = fmax(hyp[p] - v, 0.0);
        st.hyp_min[(size_t)c * P + p] = lo;
        st.hyp_max[(size_t)c * P + p] = lo + st.scale[p];
    }
    double u0, u1;
    if (st.tape_u0) u0 = st.tape_u0[t];
    else philox_uniform2(st.seed, st.chain0 + c, (unsigned)it, STREAM_BRACKET, 1000, u0, u1);
    st.threshold[c] = density_sum(log(u0), hyp, st.prior_k, st.prior_theta, P, st.curG[c], it, st.burn_in);
    st.trips[c] = 0;
}

// After the first round (the log-likelihood at every chain's starting theta, in chain order in ll): start the first
// transition, or retire a chain whose starting state cannot define a slice.
__global__ void marginal_start_kernel(MarginalState st)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= st.B) return;
    const double G = st.ll[c];
    st.curG[c] = G;
    st.k[c] = 0;
    if (isfinite(G)) {
        st.exhausted[c] = 0;
        st.done[c] = 0;
        marginal_begin(st, c);
        return;
    }
    // the state is kept for the whole call, its history repeats it with 0 trips, and no evaluation is spent on it
    st.exhausted[c] = -1;
    st.done[c] = 1;
    const int P = st.P;
    for (int k = 0; k < st.n_iters; ++k) {
        const size_t t = (size_t)c * st.n_iters + k;
        if (st.hist_hyp) for (int p = 0; p < P; ++p) st.hist_hyp[t * P + p] = st.hyp[(size_t)c * P + p];
        if (st.hist_loglik) st.hist_loglik[t] = G;
        if (st.hist_trips) st.hist_trips[t] = 0;
    }
}

// theta' of every active chain (:132-134), written to prop in active-list order.  One thread per chain: the work is O(P).
__global__ void marginal_propose_kernel(MarginalState st)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= *st.count) return;
    const int c = st.map[i], P = st.P, k = st.k[c], it = st.iter_begin + k, trip = st.trips[c];
    const size_t t = (size_t)c * st.n_iters + k;
    double *th = st.prop + (size_t)i * P;
    for (int p = 0; p < P; ++p) {
        double u, u1;
        if (st.tape_U) u = st.tape_U[(t * st.tape_trips + trip) * P + p];
        else philox_uniform2(st.seed, st.chain0 + c, (unsigned)it, STREAM_TRIP, trip * 64 + p, u, u1);
        const double lo = st.hyp_min[(size_t)c * P + p], hi = st.hyp_max[(size_t)c * P + p];
        th[p] = __dadd_rn(lo, __dmul_rn(hi - lo, u));          // :132, rounded as written (no contraction)
    }
    if (it < st.burn_in) th[P - 1] = st.hyp[(size_t)c * P + P - 1];                  // :133-134
}

// Accept or shrink (:149-163); a finished transition is recorded and the chain's next one starts in place.
__global__ void marginal_accept_kernel(MarginalState st)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= *st.count) return;
    const int c = st.map[i], P = st.P, k = st.k[c], it = st.iter_begin + k;
    const double *th = st.prop + (size_t)i * P;
    double *h = st.hyp + (size_t)c * P;
    const double G = st.ll[i];
    const double proposal = density_sum(0.0, th, st.prior_k, st.prior_theta, P, G, it, st.burn_in);   // :149-152
    const bool ok = (proposal > st.threshold[c]) && isfinite(proposal);                                // :154
    const int trips = st.trips[c] + 1;
    st.trips[c] = trips;
    bool finished = ok;
    if (ok) {
        for (int p = 0; p < P; ++p) h[p] = th[p];                                                       // :156
        st.curG[c] = G;
    } else {
        for (int p = 0; p < P; ++p) {                                                                   // :159-163
            if (th[p] < h[p]) st.hyp_min[(size_t)c * P + p] = th[p];
            else st.hyp_max[(size_t)c * P + p] = th[p];
        }
        if (trips >= st.max_trips) {          // the budget ran out (the reference's `while True` would go on): state kept
            finished = true;
            st.exhausted[c] += 1;
        }
    }
    if (!finished) return;
    const size_t t = (size_t)c * st.n_iters + k;
    if (st.hist_hyp) for (int p = 0; p < P; ++p) st.hist_hyp[t * P + p] = h[p];
    if (st.hist_loglik) st.hist_loglik[t] = st.curG[c];
    if (st.hist_trips) st.hist_trips[t] = trips;
    if (k + 1 < st.n_iters) {
        st.k[c] = k + 1;
        marginal_begin(st, c);
    } else {
        st.done[c] = 1;
    }
}

// One CTA: order-preserving list of the chains that are not done (ballot + prefix in chunks of blockDim.x).
__global__ void __launch_bounds__(1024) marginal_compact_kernel(MarginalState st)
{
    __shared__ int warp_cnt[32];
    __shared__ int s_count;
    if (threadIdx.x == 0) s_count = 0;
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int base = 0; base < st.B; base += blockDim.x) {
        const int c = base + threadIdx.x;
        const int alive = (c < st.B) && st.done[c] == 0;
        const unsigned bal = __ballot_sync(0xffffffffu, alive);
        if (lane == 0) warp_cnt[warp] = __popc(bal);
        __syncthreads();
        int off = s_count, tot = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { if (w < warp) off += warp_cnt[w]; tot += warp_cnt[w]; }
        if (alive) st.map[off + __popc(bal & ((1u << lane) - 1))] = c;
        __syncthreads();
        if (threadIdx.x == 0) s_count += tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) *st.count = s_count;
}

static char *carve(char *&p, size_t bytes) { char *r = p; p += align_up(bytes, 256); return r; }

// the sampler's own arrays; the rest of the workspace goes to the log-likelihood unit
static size_t marginal_layout(MarginalState *st, double **ycen, char *base, int N, int P, int B)
{
    MarginalState tmp{};
    MarginalState &s = st ? *st : tmp;
    double *yc = nullptr;
    char *p = base;
    double **mats[] = {&s.hyp_min, &s.hyp_max, &s.prop};
    for (double **v : mats) *v = (double *)carve(p, (size_t)B * P * 8);
    double **vecs[] = {&s.ll, &s.curG, &s.threshold};
    for (double **v : vecs) *v = (double *)carve(p, (size_t)B * 8);
    int **ints[] = {&s.k, &s.trips, &s.done, &s.exhausted, &s.info, &s.map};
    for (int **v : ints) *v = (int *)carve(p, (size_t)B * 4);
    s.count = (int *)carve(p, 256);
    yc = (double *)carve(p, (size_t)N * 8);
    if (ycen) *ycen = yc;
    return (size_t)(p - base);
}

size_t marginal_state_bytes(int N, int P, int B) { return marginal_layout(nullptr, nullptr, nullptr, N, P, B); }

// rounds of the last call: active chains and host wall time (ms, the round ends in a synchronisation)
static std::vector<int> g_round_active;
static std::vector<double> g_round_ms;

}  // namespace gpmc

using namespace gpmc;

extern "C" {

int gpmc_marginal_run(const double *x_dev, int N, int D, const double *y_dev, double m, double *hyp_dev, int B, int P, int kind,
                      const double *scale_dev, const double *prior_k_dev, const double *prior_theta_dev, int iter_begin, int n_iters,
                      int burn_in, unsigned long long seed, unsigned chain0, const double *tape_v, const double *tape_u0,
                      const double *tape_U, int tape_trips, int max_trips, int jitter_policy, double *hist_hyp_dev,
                      double *hist_loglik_dev, int *hist_trips_dev, int *exhausted_dev, void *ws_dev, size_t ws_bytes, void *stream)
{
    GPMC_API_LOCK();
    cudaStream_t s = (cudaStream_t)stream;
    const int n_ell = kind_n_ell(kind, D);
    if (N <= 0 || D <= 0 || B < 0 || kind_cf(kind) < 0 || P != n_ell + 2 || n_iters < 0 || iter_begin < 0 || burn_in < 0 ||
        max_trips <= 0 || (jitter_policy != GPMC_JITTER_NONE && jitter_policy != GPMC_JITTER_PYGPS)) {
        set_error("marginal_run: bad arguments N=%d D=%d B=%d P=%d kind=%d n_iters=%d iter_begin=%d burn_in=%d max_trips=%d "
                  "jitter_policy=%d", N, D, B, P, kind, n_iters, iter_begin, burn_in, max_trips, jitter_policy);
        return GPMC_EINVAL;
    }
    const int n_tape = (tape_v != nullptr) + (tape_u0 != nullptr) + (tape_U != nullptr);
    if ((n_tape != 0 && n_tape != 3) || (n_tape == 3 && tape_trips < 1) || (n_tape == 0 && tape_trips != 0)) {
        set_error("marginal_run: the tape is tape_v, tape_u0 and tape_U together with tape_trips >= 1, or none of them "
                  "with tape_trips = 0 (got %d of 3, tape_trips=%d)", n_tape, tape_trips);
        return GPMC_EINVAL;
    }
    if (B == 0 || n_iters == 0) return 0;
    if (!x_dev || !y_dev || !hyp_dev || !scale_dev || !prior_k_dev || !prior_theta_dev) {
        set_error("marginal_run: x, y, hyp, scale and the prior constants are required");
        return GPMC_EINVAL;
    }
    const size_t own = marginal_state_bytes(N, P, B);
    if (!ws_dev || ws_bytes <= own) {
        set_error("marginal_run: workspace %zu bytes cannot hold the sampler's state (%zu bytes) and one log-likelihood item",
                  ws_bytes, own);
        return GPMC_ENOMEM;
    }
    MarginalState st{};
    double *ycen = nullptr;
    marginal_layout(&st, &ycen, (char *)ws_dev, N, P, B);
    char *ws_ll = (char *)ws_dev + own;
    const size_t ws_ll_bytes = ws_bytes - own;
    st.P = P; st.B = B; st.n_iters = n_iters; st.iter_begin = iter_begin; st.burn_in = burn_in;
    st.max_trips = tape_U ? std::min(max_trips, tape_trips) : max_trips;
    st.seed = seed; st.chain0 = chain0;
    st.scale = scale_dev; st.prior_k = prior_k_dev; st.prior_theta = prior_theta_dev;
    st.hyp = hyp_dev;
    st.hist_hyp = hist_hyp_dev; st.hist_loglik = hist_loglik_dev; st.hist_trips = hist_trips_dev;
    st.tape_v = tape_v; st.tape_u0 = tape_u0; st.tape_U = tape_U; st.tape_trips = tape_trips;
    g_round_active.clear();
    g_round_ms.clear();
    auto t0 = std::chrono::steady_clock::now();
    auto end_round = [&](int active) {
        const auto t1 = std::chrono::steady_clock::now();
        g_round_active.push_back(active);
        g_round_ms.push_back(std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    };
    int rc;
    const int tpb = 128, grid_b = (B + tpb - 1) / tpb;

    // ---- first round: G at every chain's current theta (:122), then the first transition's bracket and threshold
    marginal_center_kernel<<<(N + 255) / 256, 256, 0, s>>>(y_dev, m, N, ycen);
    GPMC_LAUNCH_CHECK();
    if ((rc = loglik_batched(x_dev, N, D, ycen, 0, hyp_dev, B, P, kind, jitter_policy, st.ll, st.info, ws_ll, ws_ll_bytes, s))) return rc;
    marginal_start_kernel<<<grid_b, tpb, 0, s>>>(st);
    GPMC_LAUNCH_CHECK();
    int active = 0;
    marginal_compact_kernel<<<1, 1024, 0, s>>>(st);
    GPMC_LAUNCH_CHECK();
    GPMC_CUDA_CHECK(cudaMemcpyAsync(&active, st.count, sizeof(int), cudaMemcpyDeviceToHost, s));
    GPMC_CUDA_CHECK(cudaStreamSynchronize(s));
    end_round(B);

    // ---- shrink rounds (:131-163): one proposal per active chain; launch sizes are the device count read at the end of
    // the previous round, so a call repeats bit for bit
    while (active > 0) {
        const int grid_a = (active + tpb - 1) / tpb;
        marginal_propose_kernel<<<grid_a, tpb, 0, s>>>(st);
        GPMC_LAUNCH_CHECK();
        if ((rc = loglik_batched(x_dev, N, D, ycen, 0, st.prop, active, P, kind, jitter_policy, st.ll, st.info, ws_ll, ws_ll_bytes, s))) return rc;
        marginal_accept_kernel<<<grid_a, tpb, 0, s>>>(st);
        GPMC_LAUNCH_CHECK();
        marginal_compact_kernel<<<1, 1024, 0, s>>>(st);
        GPMC_LAUNCH_CHECK();
        const int was = active;
        GPMC_CUDA_CHECK(cudaMemcpyAsync(&active, st.count, sizeof(int), cudaMemcpyDeviceToHost, s));
        GPMC_CUDA_CHECK(cudaStreamSynchronize(s));
        end_round(was);
    }
    if (exhausted_dev) GPMC_CUDA_CHECK(cudaMemcpyAsync(exhausted_dev, st.exhausted, (size_t)B * sizeof(int), cudaMemcpyDeviceToDevice, s));
    return 0;
}

int gpmc_marginal_rounds(int capacity, int *active_out, double *ms_out)
{
    GPMC_API_LOCK();
    const int n = (int)g_round_active.size();
    for (int r = 0; r < std::min(n, capacity); ++r) {
        if (active_out) active_out[r] = g_round_active[r];
        if (ms_out) ms_out[r] = g_round_ms[r];
    }
    return n;
}

}  // extern "C"
