// Device-resident control of the surrogate-data slice-sampling transition (kcMCMC/sliceSample.py:76-163):
// the bracket, threshold, proposal draw, accept test and per-dimension shrink of every chain are decided on
// the GPU; only "how many chains are still active" travels to the host between trips.
//
//   sds_begin      :102-112  S_ii, surrogate draw g = f + sqrt(S_ii) z (:194), bracket [hyp_min, hyp_max]
//   sds_threshold  :114-129  truncated-Gaussian likelihood of f, hyper-priors (log_gamma, :209-232), threshold
//   sds_propose    :132-134  theta' ~ U(hyp_min, hyp_max), noise frozen while iter < 500
//   sds_accept     :142-163  likelihood of f', priors, accept / shrink
//   sds_compact             active-chain list for the next trip (replaces the reference's per-chain `while True`)
// Randomness is either an explicit tape (parity tests; the reference's own draw order) or Philox4x32-10
// keyed by (seed, global chain id), so results do not depend on how chains are sharded over GPUs.
#include "common.cuh"
#include "sds.cuh"
#include "slice_common.cuh"
#include "tg2.cuh"
#include "../../include/gpmc.h"

namespace gpmc {

// --------------------------------------------------------------------------------- scalar formulas
// S_ii of aux_var_model (sliceSample.py:184-190) for the SE kernel, whose diagonal is sf2 everywhere.
__device__ __forceinline__ double s_diag_value(double sf, double sn)
{
    const double sf2 = exp(2.0 * log(sf));
    const double K_ii_inv = 1.0 / sf2;
    const double v_1 = 1.0 / (sn * sn) + K_ii_inv;
    double Sii = 1.0 / (v_1 - K_ii_inv);
    return (Sii < 0.0) ? 0.0 : Sii;
}

// ------------------------------------------------------------------------------------------ kernels
__global__ void __launch_bounds__(256) sds_begin_kernel(SdsState st)
{
    // wave path: every chain of the wave (slot == chain of the wave); resident loop: the slots admitted this round
    int c = blockIdx.x, gid = blockIdx.x;
    if (st.chain_of) {
        if (blockIdx.x >= *st.count_new) return;
        c = st.map_new[blockIdx.x];
        gid = st.chain_of[c];
    }
    const int P = st.P, n = st.n;
    const unsigned sweep = st.iter_of ? (unsigned)st.iter_of[c] : st.sweep;
    __shared__ double s_S;
    if (st.chain_of) {
        // the chain's current state comes straight from the caller's arrays into the slot rows
        for (int p = threadIdx.x; p < P; p += blockDim.x) st.hyp_stage[(size_t)c * P + p] = st.hyp_glob[(size_t)gid * P + p];
        for (int i = threadIdx.x; i < st.ldv; i += blockDim.x) st.F_stage[(size_t)c * st.ldv + i] = (i < n) ? st.F_glob[(size_t)gid * n + i] : 0.0;
        __syncthreads();
    }
    const double *hyp = st.hyp + (size_t)c * P;
    if (threadIdx.x == 0) {
        s_S = s_diag_value(hyp[P - 2], hyp[P - 1]);
        // bracket (:110-112): v ~ U(0, scale); hyp_min = max(hyp - v, 0); hyp_max = hyp_min + scale
        for (int p = 0; p < P; ++p) {
            double u;
            if (st.tape_v) u = st.tape_v[(size_t)gid * P + p];
            else { double u1; philox_uniform2(st.seed, st.chain0 + gid, sweep, STREAM_BRACKET, p, u, u1); }
            const double v = 0.0 + (st.scale[p] - 0.0) * u;
            const double lo = fmax(hyp[p] - v, 0.0);
            st.hyp_min[(size_t)c * P + p] = lo;
            st.hyp_max[(size_t)c * P + p] = lo + st.scale[p];
            st.theta[(size_t)c * P + p] = hyp[p];      // the aux model is first evaluated at the current theta
        }
        double u0;
        if (st.tape_u0) u0 = st.tape_u0[gid];
        else { double u1; philox_uniform2(st.seed, st.chain0 + gid, sweep, STREAM_BRACKET, 1000, u0, u1); }
        st.log_u0[c] = log(u0);
        st.done[c] = 0;
        st.ntrips[c] = 0;
        if (st.chain_of) { st.parked[c] = 0; st.resolved[c] = 0; }
        else {
            st.map[c] = c;
            if (c == 0) *st.count = gridDim.x;
        }
    }
    __syncthreads();
    const double S = s_S, sd = sqrt(S);
    const double *f = st.F + (size_t)c * st.ldv;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        double z;
        if (st.tape_z) z = st.tape_z[(size_t)gid * n + i];
        else {
            double u0, u1;
            philox_uniform2(st.seed, st.chain0 + gid, sweep, STREAM_Z, i >> 1, u0, u1);
            const double rad = sqrt(-2.0 * log(u0));
            z = (i & 1) ? rad * sin(6.283185307179586 * u1) : rad * cos(6.283185307179586 * u1);
        }
        st.g[(size_t)c * st.ldv + i] = f[i] + sd * z;                                   // :194
        st.svec[(size_t)c * st.ldv + i] = S;
    }
}

__global__ void __launch_bounds__(256) sds_threshold_kernel(SdsState st)
{
    int c = blockIdx.x, gid = blockIdx.x;
    if (st.chain_of) {
        if (blockIdx.x >= *st.count_new) return;
        c = st.map_new[blockIdx.x];
        gid = st.chain_of[c];
        // a factorisation of this evaluation failed and the jitter ladder (host side) has not run yet: wait for it
        if ((st.info1[c] != 0 || st.info2[c] != 0) && !st.resolved[c]) { if (threadIdx.x == 0) st.parked[c] = 1; return; }
    }
    __shared__ double red[8];
    const int P = st.P;
    const double *hyp = st.hyp + (size_t)c * P;
    const double sn0 = exp(log(hyp[P - 1]));           // likK.TruncatedGauss2(log_sigma=np.log(hyp[2])), :117
    const double llk = tg2_loglik_block(st.y, st.my, st.F + (size_t)c * st.ldv, st.n, sn0, st.lower, st.upper, red);   // :118
    if (threadIdx.x == 0) {
        st.cur_llk[c] = llk;
        const int it = st.iter_of ? st.iter_of[c] : st.iter;
        st.threshold[c] = density_sum(st.log_u0[c] + llk, hyp, st.prior_k, st.prior_theta, P, st.G[c], it, 500);            // :127-129
        st.curG[c] = st.G[c];
        if (st.chain_of) {
            st.phase[c] = SDS_PHASE_ACTIVE;
            if (st.loglik_glob && !st.iter_of) st.loglik_glob[gid] = st.G[c];     // what a chain that never accepts reports
        }
    }
}

__global__ void __launch_bounds__(256) sds_propose_kernel(SdsState st, int trip)
{
    int c, gid;
    if (st.chain_of) {
        if (blockIdx.x >= *st.count_act) return;
        c = st.map_act[blockIdx.x];
        gid = st.chain_of[c];
        trip = st.ntrips[c];                           // chains of one round are at different trips
    } else {
        if (blockIdx.x >= *st.count) return;
        c = st.map[blockIdx.x];
        gid = c;
    }
    const int P = st.P;
    const int it = st.iter_of ? st.iter_of[c] : st.iter;
    __shared__ double s_S;
    if (threadIdx.x == 0) {
        double *th = st.theta + (size_t)c * P;
        for (int p = 0; p < P; ++p) {
            double u;
            if (st.tape_U) u = st.tape_U[((size_t)gid * st.tape_trips + trip) * P + p];
            else { double u1; philox_uniform2(st.seed, st.chain0 + gid, (unsigned)it, STREAM_TRIP, trip * 64 + p, u, u1); }
            const double lo = st.hyp_min[(size_t)c * P + p], hi = st.hyp_max[(size_t)c * P + p];
            th[p] = lo + (hi - lo) * u;                                                 // :132
        }
        if (it < 500) th[P - 1] = st.hyp[(size_t)c * P + P - 1];                       // :133-134
        s_S = s_diag_value(th[P - 2], th[P - 1]);
        if (st.chain_of) st.resolved[c] = 0;
    }
    __syncthreads();
    const double S = s_S;
    for (int i = threadIdx.x; i < st.n; i += blockDim.x) st.svec[(size_t)c * st.ldv + i] = S;
}

__global__ void __launch_bounds__(256) sds_accept_kernel(SdsState st)
{
    int c, gid;
    if (st.chain_of) {
        if (blockIdx.x >= *st.count_act) return;
        c = st.map_act[blockIdx.x];
        gid = st.chain_of[c];
        if ((st.info1[c] != 0 || st.info2[c] != 0) && !st.resolved[c]) { if (threadIdx.x == 0) st.parked[c] = 1; return; }
    } else {
        if (blockIdx.x >= *st.count) return;
        c = st.map[blockIdx.x];
        gid = c;
    }
    __shared__ double red[8];
    __shared__ int s_accept, s_finished;
    const int P = st.P;
    const double *th = st.theta + (size_t)c * P;
    const double *fp = st.fprop + (size_t)c * st.ldv;
    const int it = st.iter_of ? st.iter_of[c] : st.iter;          // (read before the block barriers inside tg2_loglik_block:
    const double llk = tg2_loglik_block(st.y, st.my, fp, st.n, th[P - 1], st.lower, st.upper, red);   // thread 0 advances it below)  :142-143
    if (threadIdx.x == 0) {
        const double proposal = density_sum(llk, th, st.prior_k, st.prior_theta, P, st.G[c], it, 500);                     // :149-152
        const bool ok = (proposal > st.threshold[c]) && isfinite(proposal);                                         // :154
        st.ntrips[c] += 1;
        st.last_proposal[c] = proposal;
        st.last_llk[c] = llk;
        bool finished = ok;                                // this transition is over (accepted, or out of trips)
        if (ok) {
            if (st.chain_of) {
                for (int p = 0; p < P; ++p) st.hyp_glob_out[(size_t)gid * P + p] = th[p];
                if (st.loglik_glob) st.loglik_glob[gid] = st.G[c];
                if (st.ntrips_glob) st.ntrips_glob[gid] = st.ntrips[c];
                if (st.status_glob && !st.iter_of) st.status_glob[gid] = 0;
            } else {
                for (int p = 0; p < P; ++p) st.hyp_out[(size_t)c * P + p] = th[p];
                st.loglik_out[c] = st.G[c];
            }
        } else {
            const double *h = st.hyp + (size_t)c * P;
            for (int p = 0; p < P; ++p) {                                                                           // :159-163
                if (th[p] < h[p]) st.hyp_min[(size_t)c * P + p] = th[p];
                else st.hyp_max[(size_t)c * P + p] = th[p];
            }
            if (st.chain_of && st.ntrips[c] >= st.max_trips) {
                // the trip budget ran out (the reference's `while True` would go on): the chain keeps its state
                finished = true;
                if (st.ntrips_glob) st.ntrips_glob[gid] = st.ntrips[c];
                if (st.status_glob) st.status_glob[gid] = 1;
                if (st.n_exhausted) atomicAdd(st.n_exhausted, 1);
            }
        }
        if (finished) {
            if (st.iter_of) {
                // many iterations per call: record the sample, then either start the chain's next transition in this slot
                // (the state it reads back is the one just written) or free the slot
                const int k = it - st.iter;
                const double *hrec = ok ? th : st.hyp + (size_t)c * P;
                if (st.hist_hyp) for (int p = 0; p < P; ++p) st.hist_hyp[((size_t)gid * st.n_iters + k) * P + p] = hrec[p];
                if (st.hist_loglik) st.hist_loglik[(size_t)gid * st.n_iters + k] = ok ? st.G[c] : st.curG[c];
                if (st.hist_trips) st.hist_trips[(size_t)gid * st.n_iters + k] = st.ntrips[c];
                if (k + 1 < st.n_iters) { st.iter_of[c] = it + 1; st.phase[c] = SDS_PHASE_NEW; }
                else st.done[c] = 1;
            } else st.done[c] = 1;
        }
        s_accept = ok ? 1 : 0;
        s_finished = finished ? 1 : 0;
    }
    __syncthreads();
    if (s_accept) {
        if (st.chain_of) {
            double *fo = st.F_glob_out + (size_t)gid * st.n;
            for (int i = threadIdx.x; i < st.n; i += blockDim.x) fo[i] = fp[i];                                     // :156
        } else {
            double *fo = st.F_out + (size_t)c * st.ldv;
            for (int i = threadIdx.x; i < st.n; i += blockDim.x) fo[i] = fp[i];                                     // :156
        }
    }
    if (s_finished && st.iter_of && st.hist_f) {
        const int k = it - st.iter;
        if (st.thin > 0 && (k % st.thin) == 0 && k / st.thin < st.n_keep) {
            const double *src = s_accept ? fp : st.F + (size_t)c * st.ldv;        // accepted f', or the unchanged f
            double *dst = st.hist_f + ((size_t)gid * st.n_keep + k / st.thin) * st.n;
            for (int i = threadIdx.x; i < st.n; i += blockDim.x) dst[i] = src[i];
        }
    }
}

// One CTA: rebuild the list of chains that have not accepted yet.
__global__ void __launch_bounds__(1024) sds_compact_kernel(SdsState st, int nchains)
{
    __shared__ int s_count;
    if (threadIdx.x == 0) s_count = 0;
    __syncthreads();
    // order-preserving compaction in chunks of blockDim.x (ballot + prefix within the block)
    for (int base = 0; base < nchains; base += blockDim.x) {
        const int c = base + threadIdx.x;
        const int alive = (c < nchains) && (st.done[c] == 0);
        const unsigned bal = __ballot_sync(0xffffffffu, alive);
        __shared__ int warp_cnt[32];
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
        if (lane == 0) warp_cnt[warp] = __popc(bal);
        __syncthreads();
        int off = s_count;
        for (int w = 0; w < warp; ++w) off += warp_cnt[w];
        if (alive) st.map[off + __popc(bal & ((1u << lane) - 1))] = c;
        __syncthreads();
        if (threadIdx.x == 0) { int t = 0; for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += warp_cnt[w]; s_count += t; }
        __syncthreads();
    }
    if (threadIdx.x == 0) *st.count = s_count;
}

// Resident loop, once per round (one CTA): slots whose chain finished (or that never held one) take the next waiting
// chains of the call, then the three slot lists of the round are rebuilt in slot order:
//   map / count          every occupied slot that is not parked      (the auxiliary model is evaluated for these)
//   map_new / count_new  slots admitted now                          (evaluate at the current theta: :104-129)
//   map_act / count_act  slots inside their shrink loop              (propose, evaluate, accept / shrink: :131-163)
// and the status word the host polls (without synchronising) is published.
__device__ __forceinline__ int block_excl_rank(int flag, int *warp_cnt, int &total)
{
    const unsigned bal = __ballot_sync(0xffffffffu, flag);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncthreads();                                   // warp_cnt is reused from the previous call
    if (lane == 0) warp_cnt[warp] = __popc(bal);
    __syncthreads();
    int off = 0, tot = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { if (w < warp) off += warp_cnt[w]; tot += warp_cnt[w]; }
    total = tot;
    return off + __popc(bal & ((1u << lane) - 1));
}

__global__ void __launch_bounds__(1024) sds_admit_kernel(SdsState st, int round)
{
    __shared__ int warp_cnt[32];
    __shared__ int s_next, s_all, s_new, s_act, s_parked;
    if (threadIdx.x == 0) { s_next = *st.next_chain; s_all = s_new = s_act = s_parked = 0; }
    __syncthreads();
    for (int base = 0; base < st.cap; base += blockDim.x) {
        const int c = base + threadIdx.x;
        const int is_free = (c < st.cap) && (st.chain_of[c] < 0 || st.done[c] != 0);
        int total;
        const int rank = block_excl_rank(is_free, warp_cnt, total);
        const int next = s_next;
        if (is_free) {
            const int id = next + rank;
            if (id < st.n_chains) {
                st.chain_of[c] = id; st.phase[c] = SDS_PHASE_NEW; st.parked[c] = 0; st.resolved[c] = 0; st.ntrips[c] = 0;
                if (st.iter_of) st.iter_of[c] = st.iter;
            }
            else { st.chain_of[c] = -1; st.phase[c] = SDS_PHASE_FREE; }
            st.done[c] = 0;
        }
        __syncthreads();
        if (threadIdx.x == 0) s_next = min(st.n_chains, next + total);
        __syncthreads();
    }
    for (int base = 0; base < st.cap; base += blockDim.x) {
        const int c = base + threadIdx.x;
        const bool occ = (c < st.cap) && st.chain_of[c] >= 0;
        const bool pk = occ && st.parked[c] != 0;
        const int ph = occ ? st.phase[c] : SDS_PHASE_FREE;
        const int f_all = occ && !pk, f_new = f_all && ph == SDS_PHASE_NEW, f_act = f_all && ph == SDS_PHASE_ACTIVE;
        int t_all, t_new, t_act, t_pk;
        const int r_all = block_excl_rank(f_all, warp_cnt, t_all);
        const int r_new = block_excl_rank(f_new, warp_cnt, t_new);
        const int r_act = block_excl_rank(f_act, warp_cnt, t_act);
        (void)block_excl_rank(pk ? 1 : 0, warp_cnt, t_pk);
        if (f_all) st.map[s_all + r_all] = c;
        if (f_new) st.map_new[s_new + r_new] = c;
        if (f_act) st.map_act[s_act + r_act] = c;
        __syncthreads();
        if (threadIdx.x == 0) { s_all += t_all; s_new += t_new; s_act += t_act; s_parked += t_pk; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        *st.next_chain = s_next;
        *st.count = s_all; *st.count_new = s_new; *st.count_act = s_act;
        st.status_word[SDS_SW_COUNT] = s_all; st.status_word[SDS_SW_NEW] = s_new; st.status_word[SDS_SW_ACT] = s_act;
        st.status_word[SDS_SW_PARKED] = s_parked; st.status_word[SDS_SW_NEXT] = s_next; st.status_word[SDS_SW_ROUND] = round;
    }
}

int launch_sds_admit(const SdsState &st, int round, cudaStream_t s)
{
    sds_admit_kernel<<<1, 1024, 0, s>>>(st, round);
    GPMC_LAUNCH_CHECK();
    return 0;
}

int launch_sds_begin(const SdsState &st, int nchains, cudaStream_t s)
{
    prof_begin(KC_VEC, s);
    sds_begin_kernel<<<nchains, 256, 0, s>>>(st);
    prof_end(KC_VEC, s);
    GPMC_LAUNCH_CHECK();
    return 0;
}
int launch_sds_threshold(const SdsState &st, int nchains, cudaStream_t s)
{
    prof_begin(KC_VEC, s);
    sds_threshold_kernel<<<nchains, 256, 0, s>>>(st);
    prof_end(KC_VEC, s);
    GPMC_LAUNCH_CHECK();
    return 0;
}
int launch_sds_propose(const SdsState &st, int nactive, int trip, cudaStream_t s)
{
    prof_begin(KC_VEC, s);
    sds_propose_kernel<<<nactive, 256, 0, s>>>(st, trip);
    prof_end(KC_VEC, s);
    GPMC_LAUNCH_CHECK();
    return 0;
}
int launch_sds_accept(const SdsState &st, int nactive, cudaStream_t s)
{
    prof_begin(KC_VEC, s);
    sds_accept_kernel<<<nactive, 256, 0, s>>>(st);
    prof_end(KC_VEC, s);
    GPMC_LAUNCH_CHECK();
    return 0;
}
int launch_sds_compact(const SdsState &st, int nchains, cudaStream_t s)
{
    sds_compact_kernel<<<1, 1024, 0, s>>>(st, nchains);
    GPMC_LAUNCH_CHECK();
    return 0;
}

}  // namespace gpmc
