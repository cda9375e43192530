// mbp.cu -- MBP-IBIS layer on the device (SURVEY.md row a12): one trajectory with its full event list per theta-particle.
//
// Replaces, for ALL theta-particles of a rank in one launch each:
//   iterate_particle!             src/hmm_sim.jl:6-25      -> mbp_iterate_kernel
//   partial_model_based_proposal  src/hmm_mbp.jl:83-108    -> mbp_propose_kernel  (iterate_mbp! :7-44,
//                                                             initialise_trajectory! :47-80 inlined)
//   ptcls2[p] = deepcopy(ptcls[nidx[p]]) (src/hmm_ibis.jl:196-199), ptcls[p] = xf (:214) -> mbp_copy_kernel
//
// Trajectory store in HBM: per particle `cap` events as f64 time + u8 type (1-based), int32 length, int32 final state,
// f64 log_like[2].  One thread per trajectory (the Gillespie / MBP walks are sequential per trajectory; the work is
// ~300 events per trajectory, tiny next to the particle filter), f64 arithmetic with the reference's expressions, never
// contracted, so the walks are draw-for-draw comparable with the oracle.  `cap` plays the role of MAX_TRAJ
// (src/DiscretePOMP.jl:40): a trajectory that would exceed it gets log_like = -Inf.
#include <math.h>
#include <string.h>

#include <new>
#include <string>
#include <vector>

#include <chrono>
#include <stdlib.h>

#include "dpomp_dev.cuh"
#include "dpomp_internal.cuh"
#include "dpomp_models.cuh"
#include "obs_count.cuh"
#include "mbp_walk.cuh"

namespace dpomp {

// ---- event-list access policies -------------------------------------------------------------------------------------
// The walks below are written once against an IO policy, so the thread-per-trajectory and the warp-per-trajectory kernels
// execute literally the same arithmetic in the same order (bit-identical trajectories).
//   ThreadIO: one thread per trajectory, event lists read / written in HBM directly (many trajectories: throughput).
//   WarpIO:   one WARP per trajectory; every lane executes the (warp-uniform) walk redundantly, the old event list is
//             prefetched into shared memory in windows of kMbpWin events with coalesced loads, new events are staged in
//             shared memory and flushed with coalesced stores (few trajectories: latency -- no divergence between
//             trajectories, no dependent trip to HBM per event).
constexpr int kMbpWin = 256;
constexpr int kMbpWarpsPerCta = 4;
// trajectories per launch up to which the warp-per-trajectory kernels are used (B200, SIS / pooley.csv, propose call,
// warp vs thread per trajectory: 16 trajectories 1.04 vs 1.43 ms, 1024: 1.37 vs 1.96 ms, 4096: 2.53 vs 2.21 ms, 16384: 7.1 vs 2.9 ms)
constexpr int kMbpWarpThreshold = 2048;
// Growable trajectory store: the stores reserve `cap` (the current stride) events per trajectory, far fewer than the hard
// limit cap_max (the reference's MAX_TRAJ = 196000, src/DiscretePOMP.jl:40).  A walk that reaches the stride before cap_max
// does not commit its particle (no state, length or log-likelihood is written) and raises need_grow; the host doubles the
// stride and re-launches the same kernel with the same key for the particles that have not committed (`done[p] != call_id`),
// so the result is exactly that of a store with cap_max events per trajectory.  Reaching cap_max itself is the
// reference's overflow: log-likelihood -Inf (src/hmm_sim.jl:17-20, src/hmm_mbp.jl:98-101).
constexpr int kMbpInitialStride = 1024;
struct MbpGrow {
    int cap_max;
    int call_id;
    int* done;       // [n] id of the last call that committed the particle
    int* need_grow;  // [1]
};

struct ThreadIO {
    const double* it; const unsigned char* iy; int ilen;   // old trajectory (unused by the simulator)
    double* ft; unsigned char* fy;                          // new trajectory
    __device__ __forceinline__ double in_time(int e) { return it[e]; }
    __device__ __forceinline__ int in_type(int e) { return iy[e]; }
    __device__ __forceinline__ void push(int pos, double t, int type1) { ft[pos] = t; fy[pos] = (unsigned char)type1; }
    __device__ __forceinline__ void finish(int) {}
};
struct WarpIO {
    const double* it; const unsigned char* iy; int ilen;
    double* ft; unsigned char* fy;
    double* s_it; unsigned char* s_iy;   // [kMbpWin] window of the old list: events [ibase, ibase + kMbpWin)
    double* s_ft; unsigned char* s_fy;   // [kMbpWin] staged new events [fbase, fbase + kMbpWin)
    int ibase, fbase;
    int capc;  // trajectory capacity (bounds-checked debug build)
    __device__ __forceinline__ void load(int start) {
        const int lane = threadIdx.x & 31;
        __syncwarp();
        ibase = start;
        for (int i = lane; i < kMbpWin && start + i < ilen; i += 32) { s_it[i] = it[start + i]; s_iy[i] = iy[start + i]; }
        __syncwarp();
    }
    __device__ __forceinline__ double in_time(int e) {
        if (e >= ibase + kMbpWin) load(e);
        DPOMP_CHECK_IDX(e - ibase, kMbpWin);
        DPOMP_CHECK_IDX(e, ilen);
        return s_it[e - ibase];
    }
    __device__ __forceinline__ int in_type(int e) {
        if (e >= ibase + kMbpWin) load(e);
        DPOMP_CHECK_IDX(e - ibase, kMbpWin);
        DPOMP_CHECK_IDX(e, ilen);
        return s_iy[e - ibase];
    }
    __device__ __forceinline__ void flush(int upto) {
        const int lane = threadIdx.x & 31;
        __syncwarp();
        for (int i = lane; fbase + i < upto; i += 32) {
            DPOMP_CHECK_IDX(i, kMbpWin);
#ifdef DPOMP_BOUNDS_CHECK
            DPOMP_CHECK_IDX(fbase + i, capc);
#endif
            ft[fbase + i] = s_ft[i]; fy[fbase + i] = s_fy[i];
        }
        __syncwarp();
        fbase = upto;
    }
    __device__ __forceinline__ void push(int pos, double t, int type1) {
        if (pos - fbase >= kMbpWin) flush(pos);
        DPOMP_CHECK_IDX(pos - fbase, kMbpWin);
        if ((threadIdx.x & 31) == 0) { s_ft[pos - fbase] = t; s_fy[pos - fbase] = (unsigned char)type1; }
    }
    __device__ __forceinline__ void finish(int flen) { flush(flen); }
};
struct WarpShared {  // per warp
    double it[kMbpWin], ft[kMbpWin];
    unsigned char iy[kMbpWin], fy[kMbpWin];
};

// iterate_particle! (src/hmm_sim.jl:6-25) of particle p; `writer`: this thread stores the particle's scalars
template <int MODEL, class IO>
__device__ __forceinline__ void mbp_iterate_body(const MbpModel& m, MbpStore& st, IO& io, int p, bool writer, const double* theta,
                                                 const double* obs_time, const double* obs_ysum, int cap, int t, int fresh, int has_lik,
                                                 uint64_t key, uint32_t id0, double* out_logg, const MbpGrow& g, const CountObs& co) {
    using R = MbpRates<MODEL>;
    const int nc = mbp_nc<R>(m), ne = mbp_ne<R>(m);
    const double* thp = theta + (size_t)p * m.n_params;
    double th[R::PMAX];
    R::load_params(m, thp, th);
    int x[R::CMAX];
#pragma unroll
    for (int c = 0; c < R::CMAX; ++c) x[c] = (c < nc) ? st.fc[(size_t)p * nc + c] : 0;
    int len = st.len[p];
    double time = fresh ? (m.t0_index > 0 ? thp[m.t0_index - 1] : 0.0) : obs_time[t - 1];
    const double t_obs = obs_time[t];
    MbpStream rs = mbp_stream_init(key, id0 + (uint32_t)p, (uint32_t)t, 0u);
    double cum[R::EMAX];
    bool overflow = false;
    for (;;) {
        R::rates(m, th, x, cum);
        mbp_cumsum<R>(m, cum);
        const double tot = R::pick(cum, ne - 1);
        if (!(tot > 0.0)) break;
        const uint2 w = mbp_draw(rs);
        time = time - log(u32_open_f64(w.x)) / tot;
        if (time > t_obs) break;
        const int e = mbp_choose<R>(m, cum, u32_open_f64(w.y));
        R::apply(m, e, x);
        if (len >= cap) { overflow = true; break; }
        io.push(len, time, e + 1);
        ++len;
    }
    io.finish(len);
    const double out = overflow ? -INFINITY : mbp_obs_ll<MODEL>(m, co, th, t, obs_ysum[t], x);
    if (!writer) return;
    if (overflow && cap < g.cap_max) {  // the stride, not MAX_TRAJ: nothing is committed, the host grows the store and re-launches
        *g.need_grow = 1;
        return;
    }
#pragma unroll
    for (int c = 0; c < R::CMAX; ++c)
        if (c < nc) st.fc[(size_t)p * nc + c] = x[c];
    st.len[p] = len;
    if (overflow) st.ll[2 * (size_t)p] = -INFINITY;
    else if (has_lik) st.ll[2 * (size_t)p] += out;
    out_logg[p] = out;
    g.done[p] = g.call_id;
}

// WARP: one warp per trajectory (WarpIO), else one thread per trajectory (ThreadIO); 128 threads per CTA either way
template <int MODEL, bool WARP>
__global__ void __launch_bounds__(32 * kMbpWarpsPerCta) mbp_iterate_kernel(const __grid_constant__ MbpModel m, MbpStore st,
                                                           const double* theta, const double* obs_time, const double* obs_ysum, int n,
                                                           int cap, int t, int fresh, int has_lik, uint64_t key, uint32_t id0,
                                                           double* out_logg, MbpGrow g, const __grid_constant__ CountObs co) {
    if constexpr (WARP) {
        __shared__ WarpShared sh[kMbpWarpsPerCta];
        const int warp = threadIdx.x >> 5, p = blockIdx.x * kMbpWarpsPerCta + warp;
        if (p >= n || g.done[p] == g.call_id) return;
        WarpShared& w = sh[warp];
        const int len0 = st.len[p];
        WarpIO io{nullptr, nullptr, 0, st.ev_time + (size_t)p * cap, st.ev_type + (size_t)p * cap, w.it, w.iy, w.ft, w.fy, 0, len0, cap};
        mbp_iterate_body<MODEL>(m, st, io, p, (threadIdx.x & 31) == 0, theta, obs_time, obs_ysum, cap, t, fresh, has_lik, key, id0,
                                out_logg, g, co);
    } else {
        const int p = blockIdx.x * blockDim.x + threadIdx.x;
        if (p >= n || g.done[p] == g.call_id) return;
        ThreadIO io{nullptr, nullptr, 0, st.ev_time + (size_t)p * cap, st.ev_type + (size_t)p * cap};
        mbp_iterate_body<MODEL>(m, st, io, p, true, theta, obs_time, obs_ysum, cap, t, fresh, has_lik, key, id0, out_logg, g, co);
    }
}

// partial_model_based_proposal (src/hmm_mbp.jl:83-108): xi = current store (through io), xf = proposal store
template <int MODEL, class IO>
__device__ __forceinline__ void mbp_propose_body(const MbpModel& m, MbpStore& xf, IO& io, int p, bool writer, bool is_valid,
                                                 const double* theta_i, const double* theta_f, const double* obs_time,
                                                 const double* obs_ysum, const int* obs_haslik, int cap, int ymax, uint64_t key,
                                                 uint32_t id0, double* out_ll, const MbpGrow& g, const CountObs& co) {
    using R = MbpRates<MODEL>;
    const int nc = mbp_nc<R>(m), ne = mbp_ne<R>(m);
    double ll0 = 0.0, ll1 = 0.0;
    int flen = 0;
    int xfc[R::CMAX], pop_i[R::CMAX];
#pragma unroll
    for (int c = 0; c < R::CMAX; ++c) xfc[c] = pop_i[c] = (c < nc) ? m.ic[c] : 0;
    if (!is_valid) {
        ll0 = ll1 = -INFINITY;
    } else {
        double thi[R::PMAX], thf[R::PMAX];
        R::load_params(m, theta_i + (size_t)p * m.n_params, thi);
        R::load_params(m, theta_f + (size_t)p * m.n_params, thf);
        const int ilen = io.ilen;
        MbpStream rs = mbp_stream_init(key, id0 + (uint32_t)p, 0u, 1u);
        double lf[R::EMAX], li[R::EMAX], ld[R::EMAX];
        int evt = 0;
        double time = 0.0;
        bool overflow = false;
        if (m.t0_index > 0) {  // initialise_trajectory! (:47-80)
            const double t0f = theta_f[(size_t)p * m.n_params + m.t0_index - 1], t0i = theta_i[(size_t)p * m.n_params + m.t0_index - 1];
            if (t0f < t0i) {
                double t = t0f;
                for (;;) {
                    R::rates(m, thf, xfc, lf);
                    mbp_cumsum<R>(m, lf);
                    const double tot = R::pick(lf, ne - 1);
                    if (!(tot > 0.0)) break;
                    const uint2 w = mbp_draw(rs);
                    t = t - log(u32_open_f64(w.x)) / tot;
                    if (t > t0i) break;
                    const int e = mbp_choose<R>(m, lf, u32_open_f64(w.y));
                    if (flen >= cap) { overflow = true; break; }
                    io.push(flen, t, e + 1); ++flen;
                    R::apply(m, e, xfc);
                }
            } else {
                while (evt < ilen && !(io.in_time(evt) > t0f)) {
                    R::apply(m, io.in_type(evt) - 1, pop_i);
                    ++evt;
                }
            }
            time = t0f > t0i ? t0f : t0i;
        }
        for (int oi = 0; oi < ymax && !overflow; ++oi) {
            const double t_obs = obs_time[oi];
            for (;;) {  // iterate_mbp! (:14-42)
                const double t_next = (evt >= ilen) ? INFINITY : io.in_time(evt);
                const double tmax = (evt >= ilen) ? t_obs : (t_obs < t_next ? t_obs : t_next);
                R::rates(m, thi, pop_i, li);
                for (;;) {
                    R::rates(m, thf, xfc, lf);
#pragma unroll
                    for (int e = 0; e < R::EMAX; ++e) {
                        if (e < ne) {
                            const double dlt = __dsub_rn(lf[e], li[e]);
                            ld[e] = dlt > 0.0 ? dlt : 0.0;
                        }
                    }
                    mbp_cumsum<R>(m, ld);
                    const double tot = R::pick(ld, ne - 1);
                    if (!(tot > 0.0)) break;
                    const uint2 w = mbp_draw(rs);
                    time = time - log(u32_open_f64(w.x)) / tot;
                    if (time > tmax) break;
                    const int e = mbp_choose<R>(m, ld, u32_open_f64(w.y));
                    R::apply(m, e, xfc);
                    if (flen >= cap) { overflow = true; break; }
                    io.push(flen, time, e + 1); ++flen;
                }
                if (overflow) break;
                if (evt >= ilen) break;
                if (t_next > t_obs) break;
                const int e = io.in_type(evt) - 1;
                time = t_next;
                const double prob_keep = __ddiv_rn(R::pick(lf, e), R::pick(li, e));
                bool keep = prob_keep > 1.0;
                if (!keep) {
                    const uint2 w = mbp_draw(rs);
                    keep = prob_keep > u53(w.x, w.y);
                }
                if (keep) {
                    if (flen >= cap) { overflow = true; break; }
                    io.push(flen, time, e + 1); ++flen;
                    R::apply(m, e, xfc);
                }
                R::apply(m, e, pop_i);
                ++evt;
            }
            if (overflow) break;
            time = t_obs;
            ll1 = mbp_obs_ll<MODEL>(m, co, thf, oi, obs_ysum[oi], xfc);
            if (obs_haslik[oi]) ll0 += ll1;
        }
        if (overflow) ll0 = -INFINITY;
    }
    io.finish(flen);
    if (!writer) return;
    if (flen >= cap && cap < g.cap_max && ll0 == -INFINITY && is_valid) {  // stopped at the stride, not at MAX_TRAJ: see MbpGrow
        *g.need_grow = 1;
        return;
    }
#pragma unroll
    for (int c = 0; c < R::CMAX; ++c)
        if (c < nc) xf.fc[(size_t)p * nc + c] = xfc[c];
    xf.len[p] = flen;
    xf.ll[2 * (size_t)p] = ll0;
    xf.ll[2 * (size_t)p + 1] = ll1;
    out_ll[2 * (size_t)p] = ll0;
    out_ll[2 * (size_t)p + 1] = ll1;
    g.done[p] = g.call_id;
}

template <int MODEL, bool WARP>
__global__ void __launch_bounds__(32 * kMbpWarpsPerCta) mbp_propose_kernel(const __grid_constant__ MbpModel m, MbpStore xi,
                                                           MbpStore xf, const double* theta_i, const double* theta_f,
                                                           const unsigned char* valid, const double* obs_time, const double* obs_ysum,
                                                           const int* obs_haslik, int n, int cap, int ymax, uint64_t key, uint32_t id0,
                                                           double* out_ll, MbpGrow g, const __grid_constant__ CountObs co) {
    if constexpr (WARP) {
        __shared__ WarpShared sh[kMbpWarpsPerCta];
        const int warp = threadIdx.x >> 5, p = blockIdx.x * kMbpWarpsPerCta + warp;
        if (p >= n || g.done[p] == g.call_id) return;
        WarpShared& w = sh[warp];
        WarpIO io{xi.ev_time + (size_t)p * cap, xi.ev_type + (size_t)p * cap, xi.len[p], xf.ev_time + (size_t)p * cap,
                  xf.ev_type + (size_t)p * cap, w.it, w.iy, w.ft, w.fy, 0, 0, cap};
        const bool is_valid = valid[p] != 0;
        if (is_valid) io.load(0);
        mbp_propose_body<MODEL>(m, xf, io, p, (threadIdx.x & 31) == 0, is_valid, theta_i, theta_f, obs_time, obs_ysum, obs_haslik, cap,
                                ymax, key, id0, out_ll, g, co);
    } else {
        const int p = blockIdx.x * blockDim.x + threadIdx.x;
        if (p >= n || g.done[p] == g.call_id) return;
        ThreadIO io{xi.ev_time + (size_t)p * cap, xi.ev_type + (size_t)p * cap, xi.len[p], xf.ev_time + (size_t)p * cap,
                    xf.ev_type + (size_t)p * cap};
        mbp_propose_body<MODEL>(m, xf, io, p, true, valid[p] != 0, theta_i, theta_f, obs_time, obs_ysum, obs_haslik, cap, ymax, key,
                                id0, out_ll, g, co);
    }
}

// dst[dst_slot[k]] <- src[src_slot[k]] : one CTA per particle, only the live part of the trajectory moves
__global__ void __launch_bounds__(128) mbp_copy_kernel(MbpStore dst, MbpStore src, const int64_t* dst_slots, const int64_t* src_slots,
                                                        int cap, int n_comp) {
    const int k = blockIdx.x;
    const long long d = dst_slots ? dst_slots[k] - 1 : k, s = src_slots ? src_slots[k] - 1 : k;
    const int len = src.len[s];
    const double* st = src.ev_time + (size_t)s * cap;
    double* dt = dst.ev_time + (size_t)d * cap;
    const unsigned char* sy = src.ev_type + (size_t)s * cap;
    unsigned char* dy = dst.ev_type + (size_t)d * cap;
    for (int i = threadIdx.x; i < len; i += blockDim.x) {
        dt[i] = st[i];
        dy[i] = sy[i];
    }
    if (threadIdx.x < n_comp) dst.fc[(size_t)d * n_comp + threadIdx.x] = src.fc[(size_t)s * n_comp + threadIdx.x];
    if (threadIdx.x == 32) dst.len[d] = len;
    if (threadIdx.x == 64) { dst.ll[2 * d] = src.ll[2 * s]; dst.ll[2 * d + 1] = src.ll[2 * s + 1]; }
}

// growth of the stride: the live prefix of every trajectory moves to its place in the wider arrays
__global__ void __launch_bounds__(128) mbp_restride_kernel(double* dt, unsigned char* dy, const double* st, const unsigned char* sy,
                                                            const int* len, int old_cap, int new_cap) {
    const size_t p = blockIdx.x;
    const int l = min(max(len[p], 0), old_cap);
    for (int i = threadIdx.x; i < l; i += blockDim.x) {
        dt[p * new_cap + i] = st[p * old_cap + i];
        dy[p * new_cap + i] = sy[p * old_cap + i];
    }
}

// migration: pack / unpack whole particles.  fixed record = 16 int32 words: [0] length, [1..8] final state, [10..13] log_like[2]
constexpr int kMbpFixedWords = 16;
__global__ void __launch_bounds__(128) mbp_pack_kernel(MbpStore st, const int64_t* slots, const int64_t* offsets, int* fixed,
                                                        double* times, unsigned char* types, int cap, int n_comp, int unpack) {
    const int k = blockIdx.x;
    const long long p = slots[k] - 1;
    int* fx = fixed + (size_t)k * kMbpFixedWords;
    double* et = st.ev_time + (size_t)p * cap;
    unsigned char* ey = st.ev_type + (size_t)p * cap;
    const long long off = offsets[k];
    if (!unpack) {
        const int len = st.len[p];
        for (int i = threadIdx.x; i < len; i += blockDim.x) { times[off + i] = et[i]; types[off + i] = ey[i]; }
        if (threadIdx.x == 0) fx[0] = len;
        if (threadIdx.x < n_comp) fx[1 + threadIdx.x] = st.fc[(size_t)p * n_comp + threadIdx.x];
        if (threadIdx.x == 32) { double* l = reinterpret_cast<double*>(fx + 10); l[0] = st.ll[2 * p]; l[1] = st.ll[2 * p + 1]; }
    } else {
        const int len = min(fx[0], cap);  // never past the stride: importers widen it first (dpomp_mbp_reserve / resample_migrate)
        for (int i = threadIdx.x; i < len; i += blockDim.x) { et[i] = times[off + i]; ey[i] = types[off + i]; }
        if (threadIdx.x == 0) st.len[p] = len;
        if (threadIdx.x < n_comp) st.fc[(size_t)p * n_comp + threadIdx.x] = fx[1 + threadIdx.x];
        if (threadIdx.x == 32) { const double* l = reinterpret_cast<const double*>(fx + 10); st.ll[2 * p] = l[0]; st.ll[2 * p + 1] = l[1]; }
    }
}

__global__ void mbp_reset_kernel(const __grid_constant__ MbpModel m, MbpStore st, int n) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    for (int c = 0; c < m.n_comp; ++c) st.fc[(size_t)p * m.n_comp + c] = m.ic[c];
    st.len[p] = 0;
    st.ll[2 * (size_t)p] = st.ll[2 * (size_t)p + 1] = 0.0;
}

// ------------------------------------------------------------------------------------------------------------
// Device-resident outer layer of MBP-IBIS (run_mbp_ibis src/hmm_ibis.jl:140-244): theta, prior, log-likelihood, weights and
// the marginal increments of ALL n_total theta-particles live on the device, REPLICATED on every rank; the replicated
// kernels below are O(n_total) and deterministic (fixed reduction trees over the global arrays), so every rank takes
// identical decisions and results do not depend on the number of ranks.  Only the trajectory kernels (iterate / propose /
// accept copy) are sharded.  Proposal and accept draws: Philox4x32-10 keyed by the GLOBAL particle id.
// ------------------------------------------------------------------------------------------------------------
constexpr uint32_t kTagOuter = 3u;
constexpr int kOuterThreads = 1024;

// deterministic sum of k values per thread over a single CTA of kOuterThreads threads: thread-serial over its strided
// elements, then a shared-memory tree
template <int K>
__device__ __forceinline__ void outer_block_sum(double (&v)[K], double* out /*[K] global*/) {
    __shared__ double red[kOuterThreads];
    const int tid = threadIdx.x;
#pragma unroll 1
    for (int k = 0; k < K; ++k) {  // one tree per value, the 8 KB buffer reused
        double mine = v[0];
#pragma unroll
        for (int j = 1; j < K; ++j) mine = (k == j) ? v[j] : mine;  // (registers: no dynamic indexing)
        red[tid] = mine;
        __syncthreads();
        for (int s = kOuterThreads / 2; s > 0; s >>= 1) {
            if (tid < s) red[tid] = __dadd_rn(red[tid], red[tid + s]);
            __syncthreads();
        }
        if (tid == 0) out[k] = red[0];
        __syncthreads();
    }
}

// logpdf(Product(Uniform.(lo, hi)), theta) for every particle (src/hmm_ibis.jl:153); w = 1, log_like = 0
__global__ void outer_init_kernel(const double* theta, const double* lo, const double* hi, int d, long long n, double* prior,
                                  double* w, double* log_like) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    double lp = 0.0;
    bool inside = true;
    for (int k = 0; k < d; ++k) {
        const double v = theta[p * d + k];
        inside = inside && v >= lo[k] && v <= hi[k];
        lp -= log(hi[k] - lo[k]);
    }
    prior[p] = inside ? lp : -INFINITY;
    w[p] = 1.0;
    log_like[p] = 0.0;
}

// :181-185  gx = exp(lg); S0 = sum w, S1 = sum w gx; w *= gx; S2 = sum w, S3 = sum w^2; log_like += lg.  One CTA.
__global__ void __launch_bounds__(kOuterThreads) outer_reweight_kernel(const double* lg, double* w, double* gx, double* log_like,
                                                                        long long n, int has_lik, double* out5) {
    double v[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (long long p = threadIdx.x; p < n; p += kOuterThreads) {
        if (!has_lik) continue;
        const double g = exp(lg[p]);
        const double w0 = w[p], w1 = w0 * g;
        gx[p] = g;
        log_like[p] += lg[p];  // -Inf propagates for overflowed trajectories (src/hmm_sim.jl:17-20)
        w[p] = w1;
        v[0] = __dadd_rn(v[0], w0);
        v[1] = __dadd_rn(v[1], w0 * g);
        v[2] = __dadd_rn(v[2], w1);
        v[3] = __dadd_rn(v[3], w1 * w1);
        v[4] = __dadd_rn(v[4], w1 * g);  // (:231 uses the already updated w, as written in the reference)
    }
    outer_block_sum<5>(v, out5);
}

// compute_is_mu_covar! (src/cmn.jl:91-99), pass 1: sum w and sum w theta_k; pass 2: sum w (theta_i - mu_i)(theta_j - mu_j)
template <int DMAX>
__global__ void __launch_bounds__(kOuterThreads) outer_moment1_kernel(const double* theta, const double* w, int d, long long n,
                                                                       double* out /*[1 + DMAX]*/) {
    double v[1 + DMAX];
#pragma unroll
    for (int k = 0; k < 1 + DMAX; ++k) v[k] = 0.0;
    for (long long p = threadIdx.x; p < n; p += kOuterThreads) {
        const double wp = w[p];
        v[0] = __dadd_rn(v[0], wp);
#pragma unroll
        for (int k = 0; k < DMAX; ++k)
            if (k < d) v[1 + k] = __dadd_rn(v[1 + k], wp * theta[p * d + k]);
    }
    outer_block_sum<1 + DMAX>(v, out);
}
template <int DMAX>
__global__ void __launch_bounds__(kOuterThreads) outer_moment2_kernel(const double* theta, const double* w, const double* mu, int d,
                                                                       long long n, double* out /*[DMAX * (DMAX + 1) / 2]*/) {
    constexpr int NT = DMAX * (DMAX + 1) / 2;
    double v[NT];
#pragma unroll
    for (int k = 0; k < NT; ++k) v[k] = 0.0;
    for (long long p = threadIdx.x; p < n; p += kOuterThreads) {
        const double wp = w[p];
        int t = 0;
#pragma unroll
        for (int i = 0; i < DMAX; ++i)
#pragma unroll
            for (int j = 0; j <= i; ++j, ++t)
                if (i < d) v[t] = __dadd_rn(v[t], wp * (theta[p * d + i] - mu[i]) * (theta[p * d + j] - mu[j]));
    }
    outer_block_sum<NT>(v, out);
}

// resample gather (:196-201 for the host-side fields): new[p] = old[nidx[p] - 1]
__global__ void outer_gather_kernel(const int64_t* nidx, int d, long long n, const double* theta, const double* prior, const double* log_like,
                                    const double* gx, double* theta2, double* prior2, double* log_like2, double* mtd_gx, double* w) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const long long s = nidx[p] - 1;
    for (int k = 0; k < d; ++k) theta2[p * d + k] = theta[s * d + k];
    prior2[p] = prior[s];
    log_like2[p] = log_like[s];
    mtd_gx[p] = gx[s];
    w[p] = 1.0;  // :227
}
__global__ void __launch_bounds__(kOuterThreads) outer_sum_kernel(const double* x, long long n, double* out1) {
    double v[1] = {0.0};
    for (long long p = threadIdx.x; p < n; p += kOuterThreads) v[0] = __dadd_rn(v[0], x[p]);
    outer_block_sum<1>(v, out1);
}

__device__ __forceinline__ double outer_u53_open(uint32_t hi, uint32_t lo) {  // (0, 1]
    return 1.0 - u53(hi, lo);
}
// get_mv_param (src/hmm_cmn.jl:13-18) for every particle: theta_f = base + scale * (L z), z ~ N(0, I) by Box-Muller on
// Philox draws keyed by the global particle id; base = mu (ind_prop) or the particle's theta; prior_f and valid (:204-206)
template <int DMAX>
__global__ void outer_propose_kernel(const double* theta, const double* mu, const double* chol /*[d][d] row-major lower*/, double scale,
                                     int ind_prop, const double* lo, const double* hi, int d, long long n, uint64_t key,
                                     double* theta_f, double* prior_f, unsigned char* valid) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    double z[DMAX];
#pragma unroll
    for (int j = 0; j < DMAX; j += 2) {
        if (j < d) {
            const Philox4 q = stream_draw(key, (uint32_t)p, (uint32_t)(j >> 1), 0u, kTagOuter, 0u);
            const double r = sqrt(-2.0 * log(outer_u53_open(q.w0, q.w1)));
            double sn, cs;
            sincospi(2.0 * u53(q.w2, q.w3), &sn, &cs);
            z[j] = r * cs;
            if (j + 1 < DMAX) z[j + 1] = r * sn;
        }
    }
    double lp = 0.0;
    bool inside = true;
#pragma unroll
    for (int i = 0; i < DMAX; ++i) {
        if (i < d) {
            double acc = 0.0;
#pragma unroll
            for (int j = 0; j <= i; ++j) acc += chol[i * d + j] * z[j];
            const double v = (ind_prop ? mu[i] : theta[p * d + i]) + scale * acc;
            theta_f[p * d + i] = v;
            inside = inside && v >= lo[i] && v <= hi[i];
            lp -= log(hi[i] - lo[i]);
        }
    }
    prior_f[p] = inside ? lp : -INFINITY;
    valid[p] = inside ? 1 : 0;
}

// :212-218 for every particle: accept iff exp(prior_f - prior) * exp(ll_f[0] - log_like) > rand()
__global__ void outer_accept_kernel(const double* llf /*[n][2]*/, const double* theta_f, const double* prior_f, int d, long long n,
                                    uint64_t key, double* theta, double* prior, double* log_like, double* mtd_gx, unsigned char* acc) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const Philox4 q = stream_draw(key, (uint32_t)p, 0xffffu, 0u, kTagOuter, 1u);
    const double u = u53(q.w0, q.w1);
    const double ratio = exp(prior_f[p] - prior[p]) * exp(llf[2 * p] - log_like[p]);
    const bool a = ratio > u;  // NaN compares false, as in the reference
    acc[p] = a ? 1 : 0;
    if (a) {
        for (int k = 0; k < d; ++k) theta[p * d + k] = theta_f[p * d + k];
        prior[p] = prior_f[p];
        log_like[p] = llf[2 * p];
        mtd_gx[p] = exp(llf[2 * p + 1]);
    }
}
__global__ void __launch_bounds__(kOuterThreads) outer_count_kernel(const unsigned char* acc, long long n, double* out1) {
    double v[1] = {0.0};
    for (long long p = threadIdx.x; p < n; p += kOuterThreads) v[0] += acc[p] ? 1.0 : 0.0;
    outer_block_sum<1>(v, out1);
}
// ptcls[p] = xf for the accepted particles of this rank's block (:214): dst = current store, src = proposal store
__global__ void __launch_bounds__(128) mbp_copy_flagged_kernel(MbpStore dst, MbpStore src, const unsigned char* acc, int cap, int n_comp) {
    const int p = blockIdx.x;
    if (!acc[p]) return;
    const int len = src.len[p];
    const double* st = src.ev_time + (size_t)p * cap;
    double* dt = dst.ev_time + (size_t)p * cap;
    const unsigned char* sy = src.ev_type + (size_t)p * cap;
    unsigned char* dy = dst.ev_type + (size_t)p * cap;
    for (int i = threadIdx.x; i < len; i += blockDim.x) { dt[i] = st[i]; dy[i] = sy[i]; }
    if (threadIdx.x < n_comp) dst.fc[(size_t)p * n_comp + threadIdx.x] = src.fc[(size_t)p * n_comp + threadIdx.x];
    if (threadIdx.x == 32) dst.len[p] = len;
    if (threadIdx.x == 64) { dst.ll[2 * p] = src.ll[2 * p]; dst.ll[2 * p + 1] = src.ll[2 * p + 1]; }
}

}  // namespace dpomp

// ------------------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------------------
using namespace dpomp;

// struct dpomp_model and dpomp_set_error: dpomp_internal.cuh; MCK: mbp_walk.cuh

// replicated device state of the outer layer (all n_total theta-particles; see the kernels above)
struct MbpOuter {
    dpomp_comm* comm = nullptr;
    long long n_total = 0, lo = 0, hi = 0;
    int d = 0;
    double *theta = nullptr, *theta2 = nullptr, *theta_f = nullptr, *prior = nullptr, *prior2 = nullptr, *prior_f = nullptr;
    double *log_like = nullptr, *log_like2 = nullptr, *w = nullptr, *gx = nullptr, *mtd_gx = nullptr, *lg_all = nullptr, *llf_all = nullptr;
    double *box = nullptr;      // [2][d] prior bounds
    double *par = nullptr;      // [d + d*d] mu, chol of the current sweep
    double *red = nullptr;      // [64] reduction results
    double *cw = nullptr, *u = nullptr;  // [n_total] cumulative weights / resampling draws
    int64_t* nidx = nullptr;    // [n_total]
    unsigned char *valid = nullptr, *acc = nullptr;
    double* h_red = nullptr;    // pinned [64]
    std::vector<double> h_w;    // host copies for the sequential cumsum
    std::vector<int64_t> h_nidx;
    uint64_t sweep = 0;
};


static uint64_t mbp_splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
uint64_t mbp_next_key(dpomp_mbp* h) {
    const uint64_t k = h->key_forced ? h->forced_key : mbp_splitmix64(h->seed ^ mbp_splitmix64(0x4D4250ull + h->call_index));
    h->key_forced = false;
    h->call_index += 1;
    return k;
}
// one warp per trajectory while the warps of a launch fit on the device a few times over, else one thread per trajectory
static bool mbp_use_warps(const dpomp_mbp* h, int n) { return h->mode == 2 || (h->mode == 0 && n <= kMbpWarpThreshold); }
static void mbp_outer_free(dpomp_mbp* h) {
    MbpOuter* o = h->outer;
    if (!o) return;
    cudaFree(o->theta); cudaFree(o->theta2); cudaFree(o->theta_f); cudaFree(o->prior); cudaFree(o->prior2); cudaFree(o->prior_f);
    cudaFree(o->log_like); cudaFree(o->log_like2); cudaFree(o->w); cudaFree(o->gx); cudaFree(o->mtd_gx); cudaFree(o->lg_all);
    cudaFree(o->llf_all); cudaFree(o->box); cudaFree(o->par); cudaFree(o->red); cudaFree(o->cw); cudaFree(o->u); cudaFree(o->nidx);
    cudaFree(o->valid); cudaFree(o->acc); cudaFreeHost(o->h_red);
    delete o;
    h->outer = nullptr;
}
static void mbp_free(dpomp_mbp* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    mbp_outer_free(h);
    for (int s = 0; s < 3; ++s) {
        cudaFree(h->store[s].ev_time); cudaFree(h->store[s].ev_type); cudaFree(h->store[s].len);
        cudaFree(h->store[s].fc); cudaFree(h->store[s].ll);
    }
    cudaFree(h->theta_i); cudaFree(h->theta_f); cudaFree(h->out); cudaFree(h->obs_time); cudaFree(h->obs_ysum);
    cudaFree(h->obs_haslik); cudaFree(h->obs_lgy); cudaFree(h->obs_lgk); cudaFree(h->valid); cudaFree(h->slots); cudaFree(h->done); cudaFree(h->need_grow); cudaFree(h->da_work);
    cudaFreeHost(h->h_need_grow);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

// widen the stride of all three stores to new_cap (<= cap_max); the live prefixes are copied on the store's stream
int mbp_grow(dpomp_mbp* h, int new_cap) {
    if (new_cap > h->cap_max) new_cap = h->cap_max;
    if (new_cap <= h->cap) return DPOMP_OK;
    const size_t N = (size_t)h->n;
    for (int s = 0; s < 3; ++s) {
        double* nt = nullptr;
        unsigned char* ny = nullptr;
        if (cudaMalloc((void**)&nt, N * (size_t)new_cap * sizeof(double)) != cudaSuccess ||
            cudaMalloc((void**)&ny, N * (size_t)new_cap) != cudaSuccess) {
            cudaFree(nt);
            return dpomp_set_error(DPOMP_ERR_CUDA, std::string("growing the trajectory store: ") + cudaGetErrorString(cudaGetLastError()));
        }
        mbp_restride_kernel<<<(unsigned)h->n, 128, 0, h->stream>>>(nt, ny, h->store[s].ev_time, h->store[s].ev_type, h->store[s].len,
                                                                   h->cap, new_cap);
        MCK(cudaGetLastError());
        MCK(cudaStreamSynchronize(h->stream));
        cudaFree(h->store[s].ev_time);
        cudaFree(h->store[s].ev_type);
        h->store[s].ev_time = nt;
        h->store[s].ev_type = ny;
    }
    h->cap = new_cap;
    return DPOMP_OK;
}

// launch() until every particle has committed: a walk that reaches the stride commits nothing and raises need_grow, the host
// widens the stride and launches the same kernel again with the same key for the particles left (see MbpGrow); synchronises
template <class Launch>
static int mbp_launch_until_committed(dpomp_mbp* h, Launch&& launch) {
    for (;;) {
        MCK(cudaMemsetAsync(h->need_grow, 0, sizeof(int), h->stream));
        launch();
        MCK(cudaGetLastError());
        MCK(cudaMemcpyAsync(h->h_need_grow, h->need_grow, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        MCK(cudaStreamSynchronize(h->stream));
        if (!*h->h_need_grow) return DPOMP_OK;
        const int rc = mbp_grow(h, h->cap > h->cap_max / 2 ? h->cap_max : 2 * h->cap);
        if (rc) return rc;
    }
}
// CTAs of a walk launch over n trajectories: 128 threads per CTA, one trajectory per thread or per warp
static unsigned mbp_walk_grid(bool warps, int n) {
    return warps ? (unsigned)((n + kMbpWarpsPerCta - 1) / kMbpWarpsPerCta) : (unsigned)((n + 127) / 128);
}

// iterate_particle! for particles 1..n of this store, theta / outputs on the DEVICE (theta_dev [n][d], h->out [n])
static int mbp_launch_iterate(dpomp_mbp* h, const double* theta_dev, int n, int obs_i, int fresh, uint64_t key) {
    const bool warps = mbp_use_warps(h, n);
    const int has_lik = h->model->h.obs_id[obs_i - 1] > 0;
    const MbpGrow g{h->cap_max, ++h->call_id, h->done, h->need_grow};
    return mbp_launch_until_committed(h, [&] {
        with_walk_model(h->model_id, [&](auto model) {
            constexpr int MODEL = decltype(model)::value;
            const auto kern = warps ? mbp_iterate_kernel<MODEL, true> : mbp_iterate_kernel<MODEL, false>;
            kern<<<mbp_walk_grid(warps, n), 32 * kMbpWarpsPerCta, 0, h->stream>>>(
                h->dm, h->store[h->cur], theta_dev, h->obs_time, h->obs_ysum, n, h->cap, obs_i - 1, fresh ? 1 : 0, has_lik, key,
                (uint32_t)h->batch_offset, h->out, g, h->cobs);
        });
    });
}

// partial_model_based_proposal for particles 1..n, all arguments on the DEVICE; result in h->out [n][2]
static int mbp_launch_propose(dpomp_mbp* h, const double* theta_i_dev, const double* theta_f_dev, const unsigned char* valid_dev, int n,
                              int ymax, uint64_t key) {
    const bool warps = mbp_use_warps(h, n);
    const MbpGrow g{h->cap_max, ++h->call_id, h->done, h->need_grow};
    return mbp_launch_until_committed(h, [&] {
        with_walk_model(h->model_id, [&](auto model) {
            constexpr int MODEL = decltype(model)::value;
            const auto kern = warps ? mbp_propose_kernel<MODEL, true> : mbp_propose_kernel<MODEL, false>;
            kern<<<mbp_walk_grid(warps, n), 32 * kMbpWarpsPerCta, 0, h->stream>>>(
                h->dm, h->store[h->cur], h->store[2], theta_i_dev, theta_f_dev, valid_dev, h->obs_time, h->obs_ysum, h->obs_haslik, n,
                h->cap, ymax, key, (uint32_t)h->batch_offset, h->out, g, h->cobs);
        });
    });
}

extern "C" {

int dpomp_mbp_create(const dpomp_model* model, int32_t n_particles, int32_t max_traj, uint64_t seed, int32_t device,
                     dpomp_mbp** out) {
    if (!model || !out) return dpomp_set_error(DPOMP_ERR_ARG, "null argument");
    if (n_particles < 1 || max_traj < 1) return dpomp_set_error(DPOMP_ERR_ARG, "n_particles and max_traj must be positive");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev < 1)
        return dpomp_set_error(DPOMP_ERR_CUDA, std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e));
    if (device < 0) MCK(cudaGetDevice(&device));
    if (device >= ndev) return dpomp_set_error(DPOMP_ERR_ARG, "device index out of range");
    MCK(cudaSetDevice(device));
    dpomp_mbp* h = new (std::nothrow) dpomp_mbp();
    if (!h) return dpomp_set_error(DPOMP_ERR_ARG, "out of host memory");
    const dpomp_model_desc& d = model->h.desc;
    h->model = model; h->device = device; h->n = n_particles; h->seed = seed;
    h->cap_max = max_traj;
    h->cap = max_traj < kMbpInitialStride ? max_traj : kMbpInitialStride;
    MbpModel& m = h->dm;
    m.n_comp = d.n_compartments; m.n_events = d.n_events; m.n_params = d.n_params; m.t0_index = d.t0_index;
    h->model_id = kernel_model_id(model->h);
    for (int ev = 0; ev < DPOMP_MAX_EVENTS; ++ev) {
        m.par[ev] = d.rate_par[ev]; m.k1[ev] = d.rate_k1[ev]; m.k2[ev] = d.rate_k2[ev]; m.kd[ev] = d.rate_kd[ev];
        m.has_den[ev] = d.rate_has_den[ev];
        for (int c = 0; c < DPOMP_MAX_COMPARTMENTS; ++c) {
            m.f1[ev][c] = d.rate_f1[ev][c]; m.f2[ev][c] = d.rate_f2[ev][c]; m.dn[ev][c] = d.rate_dn[ev][c];
            m.trans[ev][c] = d.trans[ev][c];
        }
    }
    for (int c = 0; c < DPOMP_MAX_COMPARTMENTS; ++c) { m.xmask[c] = d.obs_xmask[c]; m.ic[c] = (int)d.initial_condition[c]; }
    m.obs_tmp1 = log(1.0 / (sqrt(2.0 * 3.14159265358979323846) * d.obs_sigma));
    m.obs_tmp2 = 2.0 * d.obs_sigma * d.obs_sigma;
    const size_t N = (size_t)n_particles, CAP = (size_t)h->cap;
    bool ok = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) == cudaSuccess;
    for (int s = 0; s < 3 && ok; ++s) {
        ok = cudaMalloc((void**)&h->store[s].ev_time, N * CAP * sizeof(double)) == cudaSuccess &&
             cudaMalloc((void**)&h->store[s].ev_type, N * CAP) == cudaSuccess &&
             cudaMalloc((void**)&h->store[s].len, N * sizeof(int)) == cudaSuccess &&
             cudaMalloc((void**)&h->store[s].fc, N * m.n_comp * sizeof(int)) == cudaSuccess &&
             cudaMalloc((void**)&h->store[s].ll, N * 2 * sizeof(double)) == cudaSuccess;
    }
    std::vector<int> haslik(d.n_obs);
    for (int t = 0; t < d.n_obs; ++t) haslik[t] = model->h.obs_id[t] > 0;
    ok = ok && cudaMalloc((void**)&h->theta_i, N * m.n_params * sizeof(double)) == cudaSuccess &&
         cudaMalloc((void**)&h->theta_f, N * m.n_params * sizeof(double)) == cudaSuccess &&
         cudaMalloc((void**)&h->out, N * 2 * sizeof(double)) == cudaSuccess &&
         cudaMalloc((void**)&h->obs_time, d.n_obs * sizeof(double)) == cudaSuccess &&
         cudaMalloc((void**)&h->obs_ysum, d.n_obs * sizeof(double)) == cudaSuccess &&
         cudaMalloc((void**)&h->obs_haslik, d.n_obs * sizeof(int)) == cudaSuccess &&
         cudaMalloc((void**)&h->valid, N) == cudaSuccess && cudaMalloc((void**)&h->slots, 2 * N * sizeof(int64_t)) == cudaSuccess &&
         cudaMalloc((void**)&h->done, N * sizeof(int)) == cudaSuccess && cudaMalloc((void**)&h->need_grow, sizeof(int)) == cudaSuccess &&
         cudaMallocHost((void**)&h->h_need_grow, sizeof(int)) == cudaSuccess &&
         cudaMemset(h->done, 0, N * sizeof(int)) == cudaSuccess &&
         cudaMemcpy(h->obs_time, model->h.obs_time.data(), d.n_obs * sizeof(double), cudaMemcpyHostToDevice) == cudaSuccess &&
         cudaMemcpy(h->obs_ysum, model->h.obs_ysum.data(), d.n_obs * sizeof(double), cudaMemcpyHostToDevice) == cudaSuccess &&
         cudaMemcpy(h->obs_haslik, haslik.data(), d.n_obs * sizeof(int), cudaMemcpyHostToDevice) == cudaSuccess;
    if (ok && model->h.obs_family != DPOMP_OBS_GAUSSIAN) {
        ok = cudaMalloc((void**)&h->obs_lgy, d.n_obs * sizeof(double)) == cudaSuccess &&
             cudaMalloc((void**)&h->obs_lgk, d.n_obs * sizeof(double)) == cudaSuccess &&
             cudaMemcpy(h->obs_lgy, model->h.obs_lgy.data(), d.n_obs * sizeof(double), cudaMemcpyHostToDevice) == cudaSuccess &&
             cudaMemcpy(h->obs_lgk, model->h.obs_lgk.data(), d.n_obs * sizeof(double), cudaMemcpyHostToDevice) == cudaSuccess;
        h->cobs = count_obs_of(model->h, h->obs_lgy, h->obs_lgk);
    }
    if (!ok) {
        std::string msg = std::string("dpomp_mbp_create: ") + cudaGetErrorString(cudaGetLastError());
        mbp_free(h);
        return dpomp_set_error(DPOMP_ERR_CUDA, msg);
    }
    mbp_reset_kernel<<<(n_particles + 127) / 128, 128, 0, h->stream>>>(h->dm, h->store[0], n_particles);
    MCK(cudaGetLastError());
    MCK(cudaStreamSynchronize(h->stream));
    model->frozen.store(true);
    *out = h;
    return DPOMP_OK;
}

int dpomp_mbp_destroy(dpomp_mbp* h) { mbp_free(h); return DPOMP_OK; }

int dpomp_mbp_set_batch_offset(dpomp_mbp* h, int64_t off) {
    if (!h || off < 0 || off + h->n > 0xffffffffll) return dpomp_set_error(DPOMP_ERR_ARG, "batch_offset out of range");
    h->batch_offset = off;
    return DPOMP_OK;
}
int dpomp_mbp_set_mode(dpomp_mbp* h, int32_t mode) {
    if (!h || mode < 0 || mode > 2) return dpomp_set_error(DPOMP_ERR_ARG, "mode must be 0 (automatic), 1 (thread) or 2 (warp per trajectory)");
    h->mode = mode;
    return DPOMP_OK;
}
int dpomp_mbp_set_stream_key(dpomp_mbp* h, uint64_t key) {
    if (!h) return dpomp_set_error(DPOMP_ERR_ARG, "null handle");
    h->forced_key = key; h->key_forced = true;
    return DPOMP_OK;
}
int dpomp_mbp_reset(dpomp_mbp* h) {
    if (!h) return dpomp_set_error(DPOMP_ERR_ARG, "null handle");
    MCK(cudaSetDevice(h->device));
    mbp_reset_kernel<<<(h->n + 127) / 128, 128, 0, h->stream>>>(h->dm, h->store[h->cur], h->n);
    MCK(cudaGetLastError());
    MCK(cudaStreamSynchronize(h->stream));
    return DPOMP_OK;
}

int dpomp_mbp_iterate(dpomp_mbp* h, const double* theta, int32_t n, int32_t obs_i, int32_t fresh, double* out_logg) {
    if (!h || !theta || !out_logg) return dpomp_set_error(DPOMP_ERR_ARG, "null argument");
    const dpomp_model_desc& d = h->model->h.desc;
    if (n < 1 || n > h->n || obs_i < 1 || obs_i > d.n_obs) return dpomp_set_error(DPOMP_ERR_ARG, "argument out of range");
    MCK(cudaSetDevice(h->device));
    const uint64_t key = mbp_next_key(h);
    MCK(cudaMemcpyAsync(h->theta_i, theta, (size_t)n * d.n_params * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    const int rc = mbp_launch_iterate(h, h->theta_i, n, obs_i, fresh, key);
    if (rc) return rc;
    MCK(cudaMemcpyAsync(out_logg, h->out, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    MCK(cudaStreamSynchronize(h->stream));
    return DPOMP_OK;
}

int dpomp_mbp_propose(dpomp_mbp* h, const double* theta_i, const double* theta_f, const uint8_t* valid, int32_t n, int32_t ymax,
                      double* out_loglike) {
    if (!h || !theta_i || !theta_f || !valid || !out_loglike) return dpomp_set_error(DPOMP_ERR_ARG, "null argument");
    const dpomp_model_desc& d = h->model->h.desc;
    if (n < 1 || n > h->n || ymax < 1 || ymax > d.n_obs) return dpomp_set_error(DPOMP_ERR_ARG, "argument out of range");
    MCK(cudaSetDevice(h->device));
    const uint64_t key = mbp_next_key(h);
    const size_t tb = (size_t)n * d.n_params * sizeof(double);
    MCK(cudaMemcpyAsync(h->theta_i, theta_i, tb, cudaMemcpyHostToDevice, h->stream));
    MCK(cudaMemcpyAsync(h->theta_f, theta_f, tb, cudaMemcpyHostToDevice, h->stream));
    MCK(cudaMemcpyAsync(h->valid, valid, (size_t)n, cudaMemcpyHostToDevice, h->stream));
    const int rc = mbp_launch_propose(h, h->theta_i, h->theta_f, h->valid, n, ymax, key);
    if (rc) return rc;
    MCK(cudaMemcpyAsync(out_loglike, h->out, (size_t)n * 2 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    MCK(cudaStreamSynchronize(h->stream));
    return DPOMP_OK;
}

static int mbp_copy(dpomp_mbp* h, int dst_store, int src_store, const int64_t* dst_slots, const int64_t* src_slots, int n) {
    if (n == 0) return DPOMP_OK;
    for (int i = 0; i < n; ++i) {
        if (dst_slots && (dst_slots[i] < 1 || dst_slots[i] > h->n)) return dpomp_set_error(DPOMP_ERR_ARG, "particle index out of range");
        if (src_slots && (src_slots[i] < 1 || src_slots[i] > h->n)) return dpomp_set_error(DPOMP_ERR_ARG, "particle index out of range");
    }
    if (dst_slots) MCK(cudaMemcpyAsync(h->slots, dst_slots, (size_t)n * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
    if (src_slots) MCK(cudaMemcpyAsync(h->slots + h->n, src_slots, (size_t)n * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
    mbp_copy_kernel<<<n, 128, 0, h->stream>>>(h->store[dst_store], h->store[src_store], dst_slots ? h->slots : nullptr,
                                              src_slots ? h->slots + h->n : nullptr, h->cap, h->dm.n_comp);
    MCK(cudaGetLastError());
    MCK(cudaStreamSynchronize(h->stream));
    return DPOMP_OK;
}

int dpomp_mbp_accept(dpomp_mbp* h, const int64_t* slots, int32_t n) {
    if (!h || (!slots && n > 0)) return dpomp_set_error(DPOMP_ERR_ARG, "null argument");
    if (n < 0 || n > h->n) return dpomp_set_error(DPOMP_ERR_ARG, "n out of range");
    MCK(cudaSetDevice(h->device));
    return mbp_copy(h, h->cur, 2, slots, slots, n);
}

int dpomp_mbp_permute(dpomp_mbp* h, const int64_t* nidx, int32_t n) {
    if (!h || !nidx) return dpomp_set_error(DPOMP_ERR_ARG, "null argument");
    if (n != h->n) return dpomp_set_error(DPOMP_ERR_ARG, "permute needs one index per particle");
    for (int i = 0; i < n; ++i)
        if (nidx[i] < 1 || nidx[i] > h->n) return dpomp_set_error(DPOMP_ERR_ARG, "particle index out of range");
    MCK(cudaSetDevice(h->device));
    int rc = mbp_copy(h, h->cur ^ 1, h->cur, nullptr, nidx, n);
    if (rc) return rc;
    h->cur ^= 1;
    return DPOMP_OK;
}

int dpomp_mbp_get_lengths(dpomp_mbp* h, const int64_t* slots, int32_t n, int32_t* out_len) {
    if (!h || !slots || !out_len) return dpomp_set_error(DPOMP_ERR_ARG, "null argument");
    if (n < 0 || n > h->n) return dpomp_set_error(DPOMP_ERR_ARG, "n out of range");
    MCK(cudaSetDevice(h->device));
    std::vector<int> all((size_t)h->n);
    MCK(cudaMemcpy(all.data(), h->store[h->cur].len, (size_t)h->n * sizeof(int), cudaMemcpyDeviceToHost));
    for (int i = 0; i < n; ++i) {
        if (slots[i] < 1 || slots[i] > h->n) return dpomp_set_error(DPOMP_ERR_ARG, "particle index out of range");
        out_len[i] = all[(size_t)slots[i] - 1];
    }
    return DPOMP_OK;
}

static int mbp_pack(dpomp_mbp* h, const int64_t* slots, const int64_t* offsets, int n, void* fixed, void* times, void* types, int unpack) {
    if (!h || (n > 0 && (!slots || !offsets || !fixed))) return dpomp_set_error(DPOMP_ERR_ARG, "null argument");
    if (n == 0) return DPOMP_OK;
    if (n < 0 || n > h->n) return dpomp_set_error(DPOMP_ERR_ARG, "n out of range");
    for (int i = 0; i < n; ++i)
        if (slots[i] < 1 || slots[i] > h->n) return dpomp_set_error(DPOMP_ERR_ARG, "particle index out of range");
    MCK(cudaSetDevice(h->device));
    MCK(cudaMemcpyAsync(h->slots, slots, (size_t)n * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
    MCK(cudaMemcpyAsync(h->slots + h->n, offsets, (size_t)n * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
    mbp_pack_kernel<<<n, 128, 0, h->stream>>>(h->store[h->cur], h->slots, h->slots + h->n, (int*)fixed, (double*)times,
                                              (unsigned char*)types, h->cap, h->dm.n_comp, unpack);
    MCK(cudaGetLastError());
    MCK(cudaStreamSynchronize(h->stream));
    return DPOMP_OK;
}
int dpomp_mbp_export(dpomp_mbp* h, const int64_t* slots, const int64_t* offsets, int32_t n, void* dev_fixed, void* dev_times,
                     void* dev_types) {
    return mbp_pack(h, slots, offsets, n, dev_fixed, dev_times, dev_types, 0);
}
int dpomp_mbp_import(dpomp_mbp* h, const int64_t* slots, const int64_t* offsets, int32_t n, const void* dev_fixed,
                     const void* dev_times, const void* dev_types) {
    return mbp_pack(h, slots, offsets, n, const_cast<void*>(dev_fixed), const_cast<void*>(dev_times), const_cast<void*>(dev_types), 1);
}

// ptcls2[p] = deepcopy(ptcls[nidx[p]]) (src/hmm_ibis.jl:196-199) across ranks: nidx is the GLOBAL 1-based ancestor vector of
// all n_total theta-particles.  Two-phase exchange over NCCL on the store's stream: event counts first, then the packed
// fixed records (64 B per particle), event times (f64) and event types (u8); local ancestors are copied on the device.
int dpomp_mbp_resample_migrate(dpomp_mbp* h, dpomp_comm* c, const int64_t* nidx, int64_t n_total) {
    if (!h || !c || !nidx) return dpomp_set_error(DPOMP_ERR_ARG, "null argument");
    static const bool trace = getenv("DPOMP_TRACE_MIGRATE") != nullptr;  // per-segment host times on stderr (diagnostics)
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto t_seg = now();
    auto seg = [&](const char* name) {
        if (!trace) return;
        const auto t1 = now();
        fprintf(stderr, "[mbp_migrate] %-12s %8.1f us\n", name, std::chrono::duration<double, std::micro>(t1 - t_seg).count());
        t_seg = t1;
    };
    const int world = comm_world(c), rank = comm_rank(c);
    for (int64_t p = 0; p < n_total; ++p)
        if (nidx[p] < 1 || nidx[p] > n_total) return dpomp_set_error(DPOMP_ERR_ARG, "ancestor index out of range");
    if (world == 1) return dpomp_mbp_permute(h, nidx, (int32_t)n_total);
    MCK(cudaSetDevice(h->device));
    MigrationPlan pl;
    migration_plan(nidx, n_total, world, rank, pl);
    const size_t n_send = pl.send_slots.size(), n_recv = pl.recv_slots.size(), n_loc = pl.local_src.size();
    if ((int)n_loc > h->n) return dpomp_set_error(DPOMP_ERR_ARG, "this rank's block exceeds the store");
    cudaStream_t st = h->stream;
    seg("plan");
    // phase 1: event counts
    std::vector<int> all_len((size_t)h->n);
    MCK(cudaMemcpyAsync(all_len.data(), h->store[h->cur].len, (size_t)h->n * sizeof(int), cudaMemcpyDeviceToHost, st));
    MCK(cudaStreamSynchronize(st));
    CommScratch sc;
    int rc = comm_scratch(c, 0, 0, 0, n_send + n_recv, &sc);
    if (rc) return rc;
    std::vector<size_t> sb((size_t)world), rb((size_t)world);
    for (size_t k = 0; k < n_send; ++k) sc.h_int[k] = all_len[(size_t)pl.send_slots[k] - 1];
    for (int r = 0; r < world; ++r) {
        sb[(size_t)r] = (size_t)pl.send_counts[(size_t)r] * sizeof(int);
        rb[(size_t)r] = (size_t)pl.recv_counts[(size_t)r] * sizeof(int);
    }
    MCK(cudaMemcpyAsync(sc.d_int, sc.h_int, n_send * sizeof(int), cudaMemcpyHostToDevice, st));
    rc = comm_alltoallv_bytes(c, sc.d_int, sb.data(), sc.d_int + n_send, rb.data(), st);
    if (rc) return rc;
    MCK(cudaMemcpyAsync(sc.h_int + n_send, sc.d_int + n_send, n_recv * sizeof(int), cudaMemcpyDeviceToHost, st));
    MCK(cudaStreamSynchronize(st));
    seg("lengths");
    // phase 2: payload.  packed layout per direction: [fixed: n x 64 B][times: events x 8 B][types: events x 1 B]
    std::vector<int64_t> off_s(n_send + 1, 0), off_r(n_recv + 1, 0);
    int max_recv = 0;
    for (size_t k = 0; k < n_send; ++k) off_s[k + 1] = off_s[k] + sc.h_int[k];
    for (size_t k = 0; k < n_recv; ++k) {
        if (sc.h_int[n_send + k] < 0 || sc.h_int[n_send + k] > h->cap_max) return dpomp_set_error(DPOMP_ERR_COMM, "received trajectory length out of range");
        off_r[k + 1] = off_r[k] + sc.h_int[n_send + k];
        max_recv = sc.h_int[n_send + k] > max_recv ? sc.h_int[n_send + k] : max_recv;
    }
    while (max_recv > h->cap) {  // a trajectory grown on another rank: widen the local stride before it arrives
        rc = mbp_grow(h, h->cap > h->cap_max / 2 ? h->cap_max : 2 * h->cap);
        if (rc) return rc;
    }
    const size_t ev_s = (size_t)off_s[n_send], ev_r = (size_t)off_r[n_recv];
    const size_t fixed_b = (size_t)kMbpFixedWords * sizeof(int);
    const size_t n_slots = 2 * n_send + n_loc + 2 * n_recv;
    rc = comm_scratch(c, n_slots, n_send * fixed_b + ev_s * 9 + 64, n_recv * fixed_b + ev_r * 9 + 64, n_send + n_recv, &sc);
    if (rc) return rc;
    int64_t* hs = sc.h_slots;
    for (size_t k = 0; k < n_send; ++k) { hs[k] = pl.send_slots[k]; hs[n_send + k] = off_s[k]; }
    for (size_t k = 0; k < n_loc; ++k) hs[2 * n_send + k] = pl.local_src[k];
    for (size_t k = 0; k < n_recv; ++k) { hs[2 * n_send + n_loc + k] = pl.recv_slots[k]; hs[2 * n_send + n_loc + n_recv + k] = off_r[k]; }
    MCK(cudaMemcpyAsync(sc.d_slots, hs, n_slots * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    seg("scratch");
    int* fx_s = (int*)sc.d_send; double* tm_s = (double*)(sc.d_send + n_send * fixed_b); unsigned char* ty_s = sc.d_send + n_send * fixed_b + ev_s * 8;
    int* fx_r = (int*)sc.d_recv; double* tm_r = (double*)(sc.d_recv + n_recv * fixed_b); unsigned char* ty_r = sc.d_recv + n_recv * fixed_b + ev_r * 8;
    if (n_send) {
        mbp_pack_kernel<<<(unsigned)n_send, 128, 0, st>>>(h->store[h->cur], sc.d_slots, sc.d_slots + n_send, fx_s, tm_s, ty_s, h->cap, h->dm.n_comp, 0);
        MCK(cudaGetLastError());
    }
    std::vector<size_t> es((size_t)world, 0), er((size_t)world, 0);  // events per peer
    {
        size_t ks = 0, kr = 0;
        for (int r = 0; r < world; ++r) {
            for (int j = 0; j < pl.send_counts[(size_t)r]; ++j, ++ks) es[(size_t)r] += (size_t)(off_s[ks + 1] - off_s[ks]);
            for (int j = 0; j < pl.recv_counts[(size_t)r]; ++j, ++kr) er[(size_t)r] += (size_t)(off_r[kr + 1] - off_r[kr]);
        }
    }
    for (int part = 0; part < 3; ++part) {
        for (int r = 0; r < world; ++r) {
            sb[(size_t)r] = part == 0 ? (size_t)pl.send_counts[(size_t)r] * fixed_b : es[(size_t)r] * (part == 1 ? 8 : 1);
            rb[(size_t)r] = part == 0 ? (size_t)pl.recv_counts[(size_t)r] * fixed_b : er[(size_t)r] * (part == 1 ? 8 : 1);
        }
        const void* sp = part == 0 ? (const void*)fx_s : part == 1 ? (const void*)tm_s : (const void*)ty_s;
        void* rp = part == 0 ? (void*)fx_r : part == 1 ? (void*)tm_r : (void*)ty_r;
        rc = comm_alltoallv_bytes(c, sp, sb.data(), rp, rb.data(), st);
        if (rc) return rc;
    }
    if (trace) { MCK(cudaStreamSynchronize(st)); seg("pack+nccl"); }
    if (n_loc) {
        mbp_copy_kernel<<<(unsigned)n_loc, 128, 0, st>>>(h->store[h->cur ^ 1], h->store[h->cur], nullptr, sc.d_slots + 2 * n_send, h->cap, h->dm.n_comp);
        MCK(cudaGetLastError());
        h->cur ^= 1;
    }
    if (n_recv) {
        mbp_pack_kernel<<<(unsigned)n_recv, 128, 0, st>>>(h->store[h->cur], sc.d_slots + 2 * n_send + n_loc, sc.d_slots + 2 * n_send + n_loc + n_recv,
                                                          fx_r, tm_r, ty_r, h->cap, h->dm.n_comp, 1);
        MCK(cudaGetLastError());
    }
    MCK(cudaStreamSynchronize(st));
    seg("copy+unpack");
    return DPOMP_OK;
}

// ---- device-resident outer layer (see the kernels "Device-resident outer layer of MBP-IBIS") -----------------------------
#define OUTER_OR_FAIL(h)                                                                                   \
    if (!(h) || !(h)->outer) return dpomp_set_error(DPOMP_ERR_STATE, "dpomp_mbp_outer_begin has not been called"); \
    MbpOuter* o = (h)->outer;                                                                              \
    MCK(cudaSetDevice((h)->device));                                                                       \
    cudaStream_t st = (h)->stream

int dpomp_mbp_outer_begin(dpomp_mbp* h, dpomp_comm* c, int64_t n_total, const double* theta_all, const double* prior_lo,
                          const double* prior_hi) {
    if (!h || !c || !theta_all || !prior_lo || !prior_hi) return dpomp_set_error(DPOMP_ERR_ARG, "null argument");
    const int d = h->dm.n_params;
    if (d > 8) return dpomp_set_error(DPOMP_ERR_ARG, "the device-resident outer layer supports up to 8 parameters");
    long long lo, hi;
    comm_bounds(c, n_total, &lo, &hi);
    if (hi - lo > h->n) return dpomp_set_error(DPOMP_ERR_ARG, "this rank's block exceeds the store");
    MCK(cudaSetDevice(h->device));
    mbp_outer_free(h);
    MbpOuter* o = new (std::nothrow) MbpOuter();
    if (!o) return dpomp_set_error(DPOMP_ERR_ARG, "out of host memory");
    h->outer = o;
    o->comm = c; o->n_total = n_total; o->lo = lo; o->hi = hi; o->d = d;
    const size_t N = (size_t)n_total, D = (size_t)d;
    bool ok = true;
#define OA(ptr, count, T) ok = ok && cudaMalloc((void**)&o->ptr, (count) * sizeof(T)) == cudaSuccess
    OA(theta, N * D, double); OA(theta2, N * D, double); OA(theta_f, N * D, double);
    OA(prior, N, double); OA(prior2, N, double); OA(prior_f, N, double);
    OA(log_like, N, double); OA(log_like2, N, double); OA(w, N, double); OA(gx, N, double); OA(mtd_gx, N, double);
    OA(lg_all, N, double); OA(llf_all, 2 * N, double); OA(box, 2 * D, double); OA(par, D + D * D, double); OA(red, 64, double);
    OA(cw, N, double); OA(u, N, double); OA(nidx, N, int64_t); OA(valid, N, unsigned char); OA(acc, N, unsigned char);
#undef OA
    ok = ok && cudaMallocHost((void**)&o->h_red, 64 * sizeof(double)) == cudaSuccess;
    if (!ok) {
        mbp_outer_free(h);
        return dpomp_set_error(DPOMP_ERR_CUDA, std::string("dpomp_mbp_outer_begin: ") + cudaGetErrorString(cudaGetLastError()));
    }
    o->h_w.resize(N); o->h_nidx.resize(N);
    cudaStream_t st = h->stream;
    MCK(cudaMemcpyAsync(o->theta, theta_all, N * D * sizeof(double), cudaMemcpyHostToDevice, st));
    MCK(cudaMemcpyAsync(o->box, prior_lo, D * sizeof(double), cudaMemcpyHostToDevice, st));
    MCK(cudaMemcpyAsync(o->box + D, prior_hi, D * sizeof(double), cudaMemcpyHostToDevice, st));
    MCK(cudaMemsetAsync(o->gx, 0, N * sizeof(double), st));
    outer_init_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(o->theta, o->box, o->box + D, d, n_total, o->prior, o->w, o->log_like);
    MCK(cudaGetLastError());
    h->batch_offset = lo;
    MCK(cudaStreamSynchronize(st));
    return dpomp_mbp_reset(h);
}

// iterate_particle! for this rank's block (:176-179), all-gather of log g, then (if the observation carries a likelihood)
// gx = exp(log g), w *= gx (:181-185).  out5 = { sum w_old, sum w_old gx, sum w_new, sum w_new^2, sum w_new gx } for lml, the
// ESS and the non-resampling evidence update (:231).
int dpomp_mbp_outer_iterate(dpomp_mbp* h, int32_t obs_i, int32_t fresh, double* out5) {
    OUTER_OR_FAIL(h);
    if (!out5 || obs_i < 1 || obs_i > h->model->h.desc.n_obs) return dpomp_set_error(DPOMP_ERR_ARG, "argument out of range");
    const int n_loc = (int)(o->hi - o->lo);
    const uint64_t key = mbp_next_key(h);
    if (n_loc) {
        const int rc = mbp_launch_iterate(h, o->theta + (size_t)o->lo * o->d, n_loc, obs_i, fresh, key);
        if (rc) return rc;
    }
    int rc = comm_allgather_rows_device(o->comm, h->out, o->n_total, 1, o->lg_all, st);
    if (rc) return rc;
    const int has_lik = h->model->h.obs_id[obs_i - 1] > 0;
    outer_reweight_kernel<<<1, kOuterThreads, 0, st>>>(o->lg_all, o->w, o->gx, o->log_like, o->n_total, has_lik, o->red);
    MCK(cudaGetLastError());
    MCK(cudaMemcpyAsync(o->h_red, o->red, 5 * sizeof(double), cudaMemcpyDeviceToHost, st));
    MCK(cudaStreamSynchronize(st));
    memcpy(out5, o->h_red, 5 * sizeof(double));
    return DPOMP_OK;
}

// compute_is_mu_covar! (src/cmn.jl:91-99) on the device state: mu[d], cv[d][d]
int dpomp_mbp_outer_moments(dpomp_mbp* h, double* out_mu, double* out_cv) {
    OUTER_OR_FAIL(h);
    if (!out_mu || !out_cv) return dpomp_set_error(DPOMP_ERR_ARG, "null argument");
    const int d = o->d;
    outer_moment1_kernel<8><<<1, kOuterThreads, 0, st>>>(o->theta, o->w, d, o->n_total, o->red);
    MCK(cudaGetLastError());
    MCK(cudaMemcpyAsync(o->h_red, o->red, 9 * sizeof(double), cudaMemcpyDeviceToHost, st));
    MCK(cudaStreamSynchronize(st));
    const double sw = o->h_red[0];
    double mu[8];
    for (int k = 0; k < d; ++k) { mu[k] = o->h_red[1 + k] / sw; out_mu[k] = mu[k]; }
    MCK(cudaMemcpyAsync(o->par, mu, (size_t)d * sizeof(double), cudaMemcpyHostToDevice, st));
    outer_moment2_kernel<8><<<1, kOuterThreads, 0, st>>>(o->theta, o->w, o->par, d, o->n_total, o->red);
    MCK(cudaGetLastError());
    MCK(cudaMemcpyAsync(o->h_red, o->red, 36 * sizeof(double), cudaMemcpyDeviceToHost, st));
    MCK(cudaStreamSynchronize(st));
    int t = 0;
    for (int i = 0; i < 8; ++i)
        for (int j = 0; j <= i; ++j, ++t)
            if (i < d) out_cv[i * d + j] = out_cv[j * d + i] = o->h_red[t] / sw;
    return DPOMP_OK;
}

// outer resample (:194-201): nidx = rs_systematic / rs_stratified (w) with the given rand() draws (cumsum sequential on the
// host like the reference's, search on the device), gather of the replicated fields, migration of the trajectories, w = 1.
// out2 = { mean(gx[nidx]), unused }
int dpomp_mbp_outer_resample(dpomp_mbp* h, int32_t rs_type, const double* u, int64_t n_u, double* out2) {
    OUTER_OR_FAIL(h);
    if (!u || !out2 || (rs_type != DPOMP_RS_SYSTEMATIC && rs_type != DPOMP_RS_STRATIFIED)) return dpomp_set_error(DPOMP_ERR_ARG, "bad argument");
    const long long n = o->n_total;
    const int64_t need_u = rs_type == DPOMP_RS_SYSTEMATIC ? 1 : n;
    if (n_u < need_u) return dpomp_set_error(DPOMP_ERR_ARG, "not enough uniforms");
    MCK(cudaMemcpyAsync(o->h_w.data(), o->w, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, st));
    MCK(cudaStreamSynchronize(st));
    for (long long i = 1; i < n; ++i) o->h_w[(size_t)i] = o->h_w[(size_t)i - 1] + o->h_w[(size_t)i];  // cumsum (src/hmm_resample.jl:45,67)
    MCK(cudaMemcpyAsync(o->cw, o->h_w.data(), (size_t)n * sizeof(double), cudaMemcpyHostToDevice, st));
    MCK(cudaMemcpyAsync(o->u, u, (size_t)need_u * sizeof(double), cudaMemcpyHostToDevice, st));
    MCK(launch_search_hook(rs_type, o->cw, n, o->u, n, o->nidx, st));
    MCK(cudaMemcpyAsync(o->h_nidx.data(), o->nidx, (size_t)n * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    outer_gather_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(o->nidx, o->d, n, o->theta, o->prior, o->log_like, o->gx, o->theta2,
                                                                    o->prior2, o->log_like2, o->mtd_gx, o->w);
    MCK(cudaGetLastError());
    std::swap(o->theta, o->theta2); std::swap(o->prior, o->prior2); std::swap(o->log_like, o->log_like2);
    outer_sum_kernel<<<1, kOuterThreads, 0, st>>>(o->mtd_gx, n, o->red);
    MCK(cudaGetLastError());
    MCK(cudaMemcpyAsync(o->h_red, o->red, sizeof(double), cudaMemcpyDeviceToHost, st));
    MCK(cudaStreamSynchronize(st));
    out2[0] = o->h_red[0] / (double)n;
    out2[1] = 0.0;
    return dpomp_mbp_resample_migrate(h, o->comm, o->h_nidx.data(), n);
}

// one mutation sweep over all particles (:203-219).  out2 = { accepted proposals, mean(mtd_gx) after the sweep }
int dpomp_mbp_outer_sweep(dpomp_mbp* h, const double* mu, const double* chol, double scale, int32_t ind_prop, int32_t obs_i, double* out2) {
    OUTER_OR_FAIL(h);
    if (!mu || !chol || !out2 || obs_i < 1 || obs_i > h->model->h.desc.n_obs) return dpomp_set_error(DPOMP_ERR_ARG, "bad argument");
    const int d = o->d;
    const long long n = o->n_total;
    const int n_loc = (int)(o->hi - o->lo);
    const uint64_t key = mbp_next_key(h);
    double par[8 + 64];
    memcpy(par, mu, (size_t)d * sizeof(double));
    memcpy(par + d, chol, (size_t)d * d * sizeof(double));
    // (a pageable source is staged by the runtime before cudaMemcpyAsync returns)
    MCK(cudaMemcpyAsync(o->par, par, (size_t)(d + d * d) * sizeof(double), cudaMemcpyHostToDevice, st));
    const unsigned grid = (unsigned)((n + 255) / 256);
    outer_propose_kernel<8><<<grid, 256, 0, st>>>(o->theta, o->par, o->par + d, scale, ind_prop, o->box, o->box + d, d, n,
                                                 key ^ 0x9E3779B97F4A7C15ull, o->theta_f, o->prior_f, o->valid);
    MCK(cudaGetLastError());
    if (n_loc) {
        const int rc = mbp_launch_propose(h, o->theta + (size_t)o->lo * d, o->theta_f + (size_t)o->lo * d, o->valid + o->lo, n_loc, obs_i, key);
        if (rc) return rc;
    }
    int rc = comm_allgather_rows_device(o->comm, h->out, n, 2, o->llf_all, st);
    if (rc) return rc;
    outer_accept_kernel<<<grid, 256, 0, st>>>(o->llf_all, o->theta_f, o->prior_f, d, n, key ^ 0xD1B54A32D192ED03ull, o->theta, o->prior,
                                              o->log_like, o->mtd_gx, o->acc);
    MCK(cudaGetLastError());
    if (n_loc) {
        mbp_copy_flagged_kernel<<<(unsigned)n_loc, 128, 0, st>>>(h->store[h->cur], h->store[2], o->acc + o->lo, h->cap, h->dm.n_comp);
        MCK(cudaGetLastError());
    }
    outer_count_kernel<<<1, kOuterThreads, 0, st>>>(o->acc, n, o->red);
    outer_sum_kernel<<<1, kOuterThreads, 0, st>>>(o->mtd_gx, n, o->red + 1);
    MCK(cudaGetLastError());
    MCK(cudaMemcpyAsync(o->h_red, o->red, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
    MCK(cudaStreamSynchronize(st));
    out2[0] = o->h_red[0];
    out2[1] = o->h_red[1] / (double)n;
    return DPOMP_OK;
}

// theta [n_total][d] and w [n_total] of all particles
int dpomp_mbp_outer_get(dpomp_mbp* h, double* out_theta, double* out_w) {
    OUTER_OR_FAIL(h);
    if (out_theta) MCK(cudaMemcpyAsync(out_theta, o->theta, (size_t)o->n_total * o->d * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (out_w) MCK(cudaMemcpyAsync(out_w, o->w, (size_t)o->n_total * sizeof(double), cudaMemcpyDeviceToHost, st));
    MCK(cudaStreamSynchronize(st));
    return DPOMP_OK;
}
int dpomp_mbp_outer_end(dpomp_mbp* h) {
    if (!h) return dpomp_set_error(DPOMP_ERR_ARG, "null handle");
    MCK(cudaSetDevice(h->device));
    mbp_outer_free(h);
    return DPOMP_OK;
}

int dpomp_mbp_capacity(dpomp_mbp* h, int32_t* out_stride, int32_t* out_max_traj) {
    if (!h) return dpomp_set_error(DPOMP_ERR_ARG, "null handle");
    if (out_stride) *out_stride = h->cap;
    if (out_max_traj) *out_max_traj = h->cap_max;
    return DPOMP_OK;
}
int dpomp_mbp_reserve(dpomp_mbp* h, int32_t stride) {
    if (!h || stride < 1) return dpomp_set_error(DPOMP_ERR_ARG, "bad argument");
    MCK(cudaSetDevice(h->device));
    return mbp_grow(h, stride);
}

int dpomp_mbp_get_states(dpomp_mbp* h, int32_t n, int64_t* out) {
    if (!h || !out) return dpomp_set_error(DPOMP_ERR_ARG, "null argument");
    if (n < 1 || n > h->n) return dpomp_set_error(DPOMP_ERR_ARG, "n out of range");
    MCK(cudaSetDevice(h->device));
    std::vector<int> tmp((size_t)n * h->dm.n_comp);
    MCK(cudaMemcpy(tmp.data(), h->store[h->cur].fc, tmp.size() * sizeof(int), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < tmp.size(); ++i) out[i] = tmp[i];
    return DPOMP_OK;
}

int dpomp_mbp_get_particle(dpomp_mbp* h, int32_t p, int32_t which, int64_t* fc, int64_t* len, double* times, int32_t* types,
                           int64_t cap_out, double* loglike2) {
    if (!h || !fc || !len || !loglike2) return dpomp_set_error(DPOMP_ERR_ARG, "null argument");
    if (p < 1 || p > h->n) return dpomp_set_error(DPOMP_ERR_ARG, "particle index out of range");
    MCK(cudaSetDevice(h->device));
    const MbpStore& s = h->store[which ? 2 : h->cur];
    int l = 0;
    int fci[DPOMP_MAX_COMPARTMENTS];
    MCK(cudaMemcpy(&l, s.len + (p - 1), sizeof(int), cudaMemcpyDeviceToHost));
    MCK(cudaMemcpy(fci, s.fc + (size_t)(p - 1) * h->dm.n_comp, h->dm.n_comp * sizeof(int), cudaMemcpyDeviceToHost));
    MCK(cudaMemcpy(loglike2, s.ll + 2 * (size_t)(p - 1), 2 * sizeof(double), cudaMemcpyDeviceToHost));
    for (int c = 0; c < h->dm.n_comp; ++c) fc[c] = fci[c];
    *len = l;
    const int ncopy = l < cap_out ? l : (int)cap_out;
    if (times && types && ncopy > 0) {
        std::vector<unsigned char> ty((size_t)ncopy);
        MCK(cudaMemcpy(times, s.ev_time + (size_t)(p - 1) * h->cap, (size_t)ncopy * sizeof(double), cudaMemcpyDeviceToHost));
        MCK(cudaMemcpy(ty.data(), s.ev_type + (size_t)(p - 1) * h->cap, (size_t)ncopy, cudaMemcpyDeviceToHost));
        for (int i = 0; i < ncopy; ++i) types[i] = ty[(size_t)i];
    }
    return DPOMP_OK;
}

}  // extern "C"
