// pf_sim.cuh -- kernel 1 of the particle filter: per-particle Gillespie simulation between two observation times,
// observation log-weight, and the per-tile / per-filter log-sum-exp partials.
//
// Replaces iterate_particles! (src/hmm_particle_filter.jl:9-33) with choose_event (src/hmm_cmn.jl:4-10), the rate
// closures (src/hmm_examples.jl:103-168) and the Gaussian observation model (src/hmm_examples.jl:59-67) of the
// reference, plus the `log(cum_weight[end]/N)` accumulation of partial_log_likelihood! (src/hmm_particle_filter.jl:60).
//
// Mapping: one CTA of kBlockThreads (128) threads per (filter, tile of kBlockThreads * ITEMS particles).  The tile's int32
// states are staged in shared memory; each warp then drains its chunk of 32 * ITEMS particles through a ballot-based work
// queue: one loop iteration is ONE event attempt for every lane (branch free in the f32 loop), and a lane whose particle
// reached the observation time parks it and pulls the next unassigned particle of the chunk, so all lanes stay busy until
// the chunk is empty (no atomics: the queue head is warp-uniform).  Compartment counts live in registers as Real during the
// loop.  One Philox2x32-10 call per attempt yields the waiting-time and event-type uniforms.  The observation log-weights
// are formed afterwards in a convergent pass in the integer domain (tile maximum by integer min, exp from a per-CTA table)
// together with the coalesced write-back, the tile scan and the two-level ticket combine.
#pragma once
#include <type_traits>

#include "dpomp_dev.cuh"
#include "dpomp_internal.cuh"
#include "dpomp_models.cuh"
#include "obs_count.cuh"
#include "pf_resample.cuh"

namespace dpomp {

template <typename Real> struct Arith;
template <> struct Arith<float> {
    static __device__ __forceinline__ float mul(float a, float b) { return a * b; }
    static __device__ __forceinline__ float add(float a, float b) { return a + b; }
    static __device__ __forceinline__ float div(float a, float b) { return __fdividef(a, b); }
};
template <> struct Arith<double> {  // round-to-nearest, never contracted: the reference's f64 expressions bit for bit
    static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
    static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
    static __device__ __forceinline__ double div(double a, double b) { return __ddiv_rn(a, b); }
};

// resident CTAs per SM the register allocation is tuned for (the f64 parity loop is not tuned)
// particles a lane of the f32 event loop works on at once (2 measured on B200: C2 3.76 vs 3.66 ms, SEIR batch 15.0 vs 14.6 ms,
// LOTKA batch 76.1 vs 77.6 ms -- the second slot costs more in the refill path than it hides in the dependency chains)
#ifndef DPOMP_SIM_ILP
#define DPOMP_SIM_ILP 1
#endif
#ifndef DPOMP_SIM_PIPE
#define DPOMP_SIM_PIPE 1
#endif
// 256-thread CTAs: 4 resident (64 registers, no spills) beat 5 / 6 (48 / 40 registers) on B200; 128-thread CTAs: 7 resident
#ifndef DPOMP_SIM_MINB
#define DPOMP_SIM_MINB (DPOMP_BLOCK_THREADS == 128 ? 7 : 4)
#endif
template <typename Real, int C, int E>
constexpr int sim_min_blocks() { return sizeof(Real) == 4 ? DPOMP_SIM_MINB : 1; }

template <int N>
struct alignas(4 * N) IntVec { int v[N]; };

// rate_function + cumsum! (src/hmm_particle_filter.jl:20-21): cumulative event rates of state x
template <typename Real, int C, int E, int MODEL>
__device__ __forceinline__ void cum_rates(const DevModel<Real, C, E>& m, const Real (&par)[E], const Real (&x)[C], Real (&cum)[E]) {
    if constexpr (MODEL != kModelGeneric) {
        using BM = Builtin<MODEL>;
#pragma unroll
        for (int e = 0; e < E; ++e) {
            Real rate = Arith<Real>::mul(par[e], x[BM::A(e)]);
            if (BM::B(e) >= 0) rate = Arith<Real>::mul(rate, x[BM::B(e) >= 0 ? BM::B(e) : 0]);
            cum[e] = (e == 0) ? rate : Arith<Real>::add(cum[e - 1], rate);
        }
    } else {
#pragma unroll
        for (int e = 0; e < E; ++e) {
            Real l1 = m.k1[e], l2 = m.k2[e];
#pragma unroll
            for (int c = 0; c < C; ++c) {
                l1 += m.f1[e][c] * x[c];
                l2 += m.f2[e][c] * x[c];
            }
            Real rate = Arith<Real>::mul(Arith<Real>::mul(par[e], l1), l2);
            if (m.any_den && m.has_den[e]) {
                Real dn = m.kd[e];
#pragma unroll
                for (int c = 0; c < C; ++c) dn += m.dn[e][c] * x[c];
                rate = (dn == (Real)0) ? (Real)0 : Arith<Real>::div(rate, dn);
            }
            cum[e] = (e == 0) ? rate : Arith<Real>::add(cum[e - 1], rate);
        }
    }
}

// choose_event (src/hmm_cmn.jl:4-10): transition row of the first event i < E with cum[i] > etc, else of event E
template <typename Real, int C, int E, int MODEL>
__device__ __forceinline__ void chosen_transition(const DevModel<Real, C, E>& m, const Real (&cum)[E], Real etc, Real (&dx)[C]) {
    if constexpr (MODEL != kModelGeneric) {
        using BM = Builtin<MODEL>;
#pragma unroll
        for (int c = 0; c < C; ++c) dx[c] = (Real)BM::T(E - 1, c);
#pragma unroll
        for (int i = E - 2; i >= 0; --i) {
            const bool hit = cum[i] > etc;
#pragma unroll
            for (int c = 0; c < C; ++c) dx[c] = hit ? (Real)BM::T(i, c) : dx[c];
        }
    } else {
#pragma unroll
        for (int c = 0; c < C; ++c) dx[c] = m.trans[E - 1][c];
#pragma unroll
        for (int i = E - 2; i >= 0; --i) {
            const bool hit = cum[i] > etc;
#pragma unroll
            for (int c = 0; c < C; ++c) dx[c] = hit ? m.trans[i][c] : dx[c];
        }
    }
}

// FUSED: the same CTA also resamples its tile after the filter's combine (one launch per observation).  The CTA takes
// its logical index from an arrival-order ticket, so every resident CTA has a lower index than any CTA not yet started;
// the host only selects this variant when all tiles of a filter fit on the device at once, hence waiting for the
// combine of the CTA's own filter cannot deadlock.  The tile's states and its scan stay in shared memory / registers
// between the two phases: neither the states nor the scans of a resampling step go through HBM.
//
// PERSIST (MODE 2): ONE cooperative launch runs the observations a.t .. a.t_last.  CTA (filter, tile) keeps its tile for
// the whole call; there is no kernel boundary and no grid-wide barrier besides the combine itself:
//   wait until every row of my tile has been written by the resample phase of the previous observation
//   (rows_done[filter][tile], a counter the producers add their row counts to) -> stage -> event loop -> weights ->
//   ticket combine (the last tile publishes the filter's generation flag, replicated per group of tiles so that only
//   kGroupTiles CTAs poll one address) -> wait for the flag -> resample my tile from shared memory, scatter the
//   offspring rows, add my row counts to the counters of the destination tiles -> next observation.
// A tile starts observation t+1 as soon as ITS rows are there (dataflow), not when the whole grid has finished t.
// The host launches it cooperatively (all CTAs co-resident or the launch fails), so the waits cannot deadlock.
constexpr int kModePlain = 0, kModeFused = 1, kModePersist = 2;
__device__ __forceinline__ unsigned int ld_acquire_u32(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// MODEL = kModelCountObs: the generic rate table with a count observation family (obs_count.cuh, a.cobs) in the weight pass
constexpr int kModelCountObs = -1;
template <typename Real, int C, int E, int ITEMS, int MODEL = kModelGeneric, int MODE = kModePlain, int ILP = DPOMP_SIM_ILP>
__global__ void __launch_bounds__(kBlockThreads, sim_min_blocks<Real, C, E>())
pf_sim_weight_kernel(const __grid_constant__ DevModel<Real, C, E> m, const __grid_constant__ SimLaunch a) {
    constexpr bool COUNT = MODEL == kModelCountObs;
    constexpr int RMODEL = COUNT ? kModelGeneric : MODEL;  // rate table of the event loop
    constexpr int TILE = kBlockThreads * ITEMS;
    constexpr int CHUNK = 32 * ITEMS;  // particles owned by one warp
    constexpr bool kF32 = sizeof(Real) == 4;
    constexpr unsigned FULL = 0xffffffffu;
    constexpr bool FUSED = MODE == kModeFused, PERSIST = MODE == kModePersist;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // staged compartment counts: f32 loop keeps them as floats (no conversions in the divergent refill path; exact
    // below 2^24), the f64 parity loop as int32
    using SState = typename std::conditional<kF32, float, int>::type;
    int* ovf_s = reinterpret_cast<int*>(smem_raw);        // [TILE] parked particle: events | (hit the event cap) << 31
    SState* st_s = reinterpret_cast<SState*>(ovf_s + TILE);  // [C][TILE]
    __shared__ double warp_scratch[kBlockThreads / 32];
    __shared__ unsigned warp_min_s[kBlockThreads / 32];
    __shared__ double wtab_s[kBlockThreads];  // exp(logw(d_min + j) - m_b), j = 0..kBlockThreads-1
    __shared__ uint32_t stream_s[3];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    unsigned int logical = blockIdx.x;
    if constexpr (FUSED) {
        __shared__ unsigned int logical_s;
        // (work_counter == nullptr: every CTA of the launch is co-resident, the launch order does not matter)
        if (a.work_counter) {
            if (tid == 0) logical_s = (unsigned int)(atomicAdd(a.work_counter, 1ull) - a.work_base);
            __syncthreads();
            logical = logical_s;
        }
    }
    const int tile = logical % a.ntiles;
    const int b = logical / a.ntiles;
    const long long base_n = (long long)tile * TILE;
    const uint32_t gfilter = a.filter_ids ? a.filter_ids[b] : a.filter0 + (uint32_t)b;
    const double* th = a.theta + (size_t)b * m.n_params;

    Real par[E];
#pragma unroll
    for (int e = 0; e < E; ++e) par[e] = m.par[e] >= 0 ? (Real)th[m.par[e]] : (Real)1;
    const uint32_t max_ev = (uint32_t)a.max_events;
    // PERSIST: the loop over the observations of the call; the other modes run its body once (t_end == a.t)
    const int t_end = PERSIST ? a.t_last : a.t;
    int flip = 0;              // PERSIST: resampling steps done so far (ping-pong of the population buffers)
    bool staged = false;       // PERSIST: the tile's states are still in shared memory from the previous observation
    bool wait_rows = false;    // PERSIST: the previous observation resampled, my rows come from other CTAs
    __shared__ int warp_max_s[kBlockThreads / 32];
    __shared__ long long lohi_s[2];
    int t = a.t;
#pragma unroll 1
    do {  // (a do-while with a compile-time false condition outside PERSIST: the other modes carry no loop at all)
    const bool fresh = a.fresh && t == a.t;
    const int has_lik = PERSIST ? (a.obs_haslik[t] > 0) : a.has_lik;
    const bool do_rs = PERSIST ? (has_lik && t + 1 < a.n_obs_total) : (a.do_resample != 0);
    const bool resample_here = (FUSED || PERSIST) && do_rs;
    const double t_obs = a.obs_time[t];
    const double t_prev = fresh ? (m.t0_index > 0 ? th[m.t0_index - 1] : 0.0) : a.obs_time[t - 1];
    const double ysum = a.obs_ysum[t];
    int32_t* pop_b = ((PERSIST && (flip & 1)) ? a.pop_dst : a.pop) + (size_t)b * a.n_comp * a.n_pad;
    int32_t* pop_other = ((PERSIST && (flip & 1)) ? a.pop : a.pop_dst);
    const unsigned int gen_t = a.gen + (unsigned int)(t - a.t);

    DPOMP_STAMP(0, 0);
    DPOMP_STAMP_NEXT(0, 7);
    if (tid == 0) {  // independent of the predecessor kernel: overlaps its tail
        const SimStream s0 = sim_stream_init(a.key, gfilter, (uint32_t)t);
        stream_s[0] = s0.k; stream_s[1] = s0.a; stream_s[2] = s0.b;
    }
    if constexpr (PERSIST) {
        if (wait_rows) {  // every row of my tile must have been written by the resample phase of observation t - 1
            if (tid == 0) {
                const long long rem_rows = a.n - base_n;
                const unsigned int want = (unsigned int)(rem_rows < TILE ? (rem_rows > 0 ? rem_rows : 0) : TILE);
                unsigned int* cnt = a.rows_done + (size_t)b * a.ntiles + tile;
                while (ld_acquire_u32(cnt) < want) __nanosleep(40);
                *cnt = 0u;  // the next producers of this tile only run after my ticket of this observation
            }
        }
        __syncthreads();  // also: the previous iteration is done with ovf_s (offspring windows) and st_s
    } else {
        pdl_wait();  // everything below reads or writes buffers shared with the predecessor kernel
    }
    DPOMP_STAMP(0, 1);
    // stage the tile: each thread moves ITEMS consecutive particles per compartment with one vector access
    using Vec = IntVec<ITEMS>;
    {
        Vec z;
#pragma unroll
        for (int kk = 0; kk < ITEMS; ++kk) z.v[kk] = 0;
        *reinterpret_cast<Vec*>(ovf_s + tid * ITEMS) = z;
    }
    // compartments present: a compile-time constant for the predefined models
    const int n_comp = (RMODEL != kModelGeneric) ? C : a.n_comp;
    if (PERSIST && staged) {
        // no resampling at the previous observation: the tile's states are still in shared memory
    } else if (!fresh) {
#pragma unroll
        for (int c = 0; c < C; ++c)
            if (c < n_comp)
            {
                DPOMP_CHECK_IDX(base_n + tid * ITEMS + ITEMS - 1, a.n_pad);
                const int32_t* src = pop_b + (size_t)c * a.n_pad + base_n + tid * ITEMS;
                Vec v;
                if constexpr (PERSIST) {  // rows written by other SMs during this launch: bypass the (incoherent) L1
#pragma unroll
                    for (int kk = 0; kk < ITEMS; kk += (ITEMS % 4 == 0 ? 4 : 1)) {
                        if constexpr (ITEMS % 4 == 0) {
                            const int4 w4 = __ldcg(reinterpret_cast<const int4*>(src + kk));
                            v.v[kk] = w4.x; v.v[kk + 1] = w4.y; v.v[kk + 2] = w4.z; v.v[kk + 3] = w4.w;
                        } else {
                            v.v[kk] = __ldcg(src + kk);
                        }
                    }
                } else {
                    v = *reinterpret_cast<const Vec*>(src);
                }
#pragma unroll
                for (int kk = 0; kk < ITEMS; ++kk) st_s[c * TILE + tid * ITEMS + kk] = (SState)v.v[kk];
            }
    } else {  // fn_initial_condition() rows (src/hmm_particle_filter.jl:44-46): the work queue always refills from shared memory
#pragma unroll
        for (int c = 0; c < C; ++c)
            if (c < n_comp) {
#pragma unroll
                for (int kk = 0; kk < ITEMS; ++kk) st_s[c * TILE + tid * ITEMS + kk] = (SState)m.ic[c];
            }
    }
    __syncthreads();
    DPOMP_STAMP(0, 2);
    const SimStream ss{stream_s[0], stream_s[1], stream_s[2]};

    // ---- event loop: each warp drains its chunk of CHUNK particles through a ballot-based work queue ----------
    // A lane can work on S particles at once (template parameter ILP): independent instruction streams per lane.  Measured on
    // B200: in the throughput regime S = 2 loses (C2 3.76 vs 3.66 ms; 4000 x 200 SIS 3.60 vs 3.17 ms: the loop is pipe bound),
    // in the latency regime of a few small filters it wins (1 and 64 x 200 SIS: 0.350 / 0.370 vs 0.427 / 0.451 ms), so the
    // 256-particle-tile kernels of the predefined models are instantiated for both and the host picks by the size of the grid.
    constexpr int S = (kF32 && C <= 4 && E <= 3) ? ILP : 1;  // the wide generic shapes would spill
    const int chunk0 = warp * CHUNK;
    const long long left = a.n - (base_n + chunk0);
    const int chunk_valid = left < CHUNK ? (left > 0 ? (int)left : 0) : CHUNK;
    const unsigned lt_mask = (1u << lane) - 1u;
    // Warp-uniform queue head: tile index of the next unassigned slot of the chunk.  Every slot handed out after the first
    // 32 * S replaces a parked particle, so head - chunk0 - 32 * S particles are done.  A lane's particle is its tile index q;
    // slots at or past chunk_valid are idle, so `q < qend` is the lane's active flag.
    int head = chunk0 + 32 * S;
    const int qend = chunk0 + chunk_valid;
    const uint32_t g_tile = (uint32_t)base_n;  // global index of the tile's first particle (mod 2^32)
    int q[S];
    Real x[S][C];
    Real tm[S];
    const Real tm0 = kF32 ? (Real)(t_obs - t_prev) : (Real)t_prev;  // f32: remaining time; f64: absolute time
    uint32_t k[S];
    uint32_t pc[S];  // first Philox counter word of the lane's particle: (global particle index) ^ A, fixed until the refill
    // Latency regime (the two-particles-per-lane instantiation the host picks for a few small filters): the Philox words of
    // attempt k + 1 depend on nothing the attempt k computes (an attempt either goes on to counter k + 1 or ends the
    // particle), so they are drawn one attempt AHEAD and the loop-carried chain of an iteration is the float chain alone
    // (rates -> rcp / lg2 -> compare -> state) instead of Philox (20 dependent integer operations) + float chain.  Same
    // counters, same draws.  Not used in the throughput regime: the refill path would pay a second Philox call per particle
    // and the loop is issue bound there.
    constexpr bool PIPE = DPOMP_SIM_PIPE && kF32 && S == 2;
    uint2 wn[S];
#pragma unroll
    for (int s = 0; s < S; ++s) {
        const int slot = lane + 32 * s;
        const int q0 = chunk0 + (slot < CHUNK ? slot : lane);
        q[s] = chunk0 + slot;
        tm[s] = tm0;
        k[s] = 0;
        pc[s] = (uint32_t)(base_n + q0) ^ ss.a;
        if constexpr (PIPE) wn[s] = philox2x32_10(pc[s], 0u ^ ss.b, ss.k);
#pragma unroll
        for (int c = 0; c < C; ++c) x[s][c] = (c < n_comp) ? (Real)st_s[c * TILE + q0] : (Real)0;  // idle lanes: harmless values
    }

    const int head_end = qend + 32 * S;  // head once every particle of the chunk is parked
    while (head < head_end) {
        bool fin[S], ovf[S];
#pragma unroll
        for (int s = 0; s < S; ++s) {
            fin[s] = false;
            ovf[s] = false;
            if constexpr (kF32) {
                // One attempt for every lane, branch free: an absorbed state (`cum_rates[end] == 0.0 && break`, :22) makes
                // the waiting time -inf / NaN, so `tmn >= 0` is false; the event cap is folded into the same predicate.
                Real cum[E];
                cum_rates<Real, C, E, RMODEL>(m, par, x[s], cum);
                const Real rtot = cum[E - 1];
                uint2 w;
                if constexpr (PIPE) {
                    w = wn[s];
                    wn[s] = philox2x32_10(pc[s], (k[s] + 1u) ^ ss.b, ss.k);  // the draws of the next attempt of this particle
                } else {
                    w = philox2x32_10(pc[s], k[s] ^ ss.b, ss.k);
                }
                // time -= log(rand()) / R  (:23) as remaining time; lg2.approx + rcp.approx on the XU pipe
                const Real tmn = fmaf(lg2_ftz(u32_wait_f32(w.x)), rcp_ftz(rtot) * 0.693147180559945f, tm[s]);
                const bool capped = k[s] >= max_ev;  // event cap: documented divergence, the reference loop is unbounded
                const bool go = (rtot > (Real)0) && !capped && (tmn >= (Real)0);  // `time > tmax && break` (:24)
                Real dx[C];
                chosen_transition<Real, C, E, RMODEL>(m, cum, u32_event_f32(w.y) * rtot, dx);  // choose_event + fn_transition (:25-26)
                if (go) {
#pragma unroll
                    for (int c = 0; c < C; ++c) x[s][c] += dx[c];
                    ++k[s];
                }
                tm[s] = tmn;  // a failed attempt ends the particle, whose remaining time is never read again
                fin[s] = q[s] < qend && !go;
                ovf[s] = capped && (rtot > (Real)0);
            } else {
                if (q[s] < qend) {
                    Real cum[E];
                    cum_rates<Real, C, E, RMODEL>(m, par, x[s], cum);
                    const Real rtot = cum[E - 1];
                    fin[s] = !(rtot > (Real)0);  // `cum_rates[end] == 0.0 && break` (:22)
                    if (!fin[s]) {
                        if (k[s] >= max_ev) {  // event cap: documented divergence, the reference loop is unbounded
                            fin[s] = true;
                            ovf[s] = true;
                        } else {
                            const uint2 w = philox2x32_10(pc[s], k[s] ^ ss.b, ss.k);
                            tm[s] = tm[s] - log(u32_open_f64(w.x)) / rtot;  // time -= log(rand()) / R (:23)
                            fin[s] = tm[s] > t_obs;                           // `time > tmax && break` (:24)
                            if (!fin[s]) {
                                Real dx[C];
                                chosen_transition<Real, C, E, RMODEL>(m, cum, __dmul_rn(u32_open_f64(w.y), rtot), dx);
#pragma unroll
                                for (int c = 0; c < C; ++c) x[s][c] += dx[c];
                                ++k[s];
                            }
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int s = 0; s < S; ++s) {
            const unsigned fmask = __ballot_sync(FULL, fin[s]);
            if (fmask) {  // warp-uniform: finished lanes park their particle and pull the next slot of the chunk
                // Park (finished lanes) and refill (finished lanes that get a slot of the chunk) as flat predicated blocks: no
                // divergent region to reconverge.  Park stores the particle's event count and cap flag as k | ovf << 31
                // (k <= max_ev < 2^31), summed in the weight pass; the flag needs no `fin` guard, since an active lane with
                // ovf always parks and an idle lane's k is never stored.
                if (ovf[s]) k[s] |= 0x80000000u;
                if (fin[s]) {
                    DPOMP_CHECK_IDX(q[s], TILE);
#pragma unroll
                    for (int c = 0; c < C; ++c)
                        if (c < n_comp) st_s[c * TILE + q[s]] = (SState)x[s][c];
                    ovf_s[q[s]] = (int)k[s];
                }
                const int qn = head + __popc(fmask & lt_mask);
                if (fin[s]) q[s] = qn;
                if (fin[s] && qn < qend) {
                    DPOMP_CHECK_IDX(qn, TILE);
                    DPOMP_CHECK_IDX(qn - chunk0, CHUNK);
                    DPOMP_CHECK_IDX(base_n + qn, a.n);
                    pc[s] = (g_tile + (uint32_t)qn) ^ ss.a;
#pragma unroll
                    for (int c = 0; c < C; ++c) x[s][c] = (c < n_comp) ? (Real)st_s[c * TILE + qn] : (Real)0;
                    tm[s] = tm0;
                    k[s] = 0;
                    if constexpr (PIPE) wn[s] = philox2x32_10(pc[s], 0u ^ ss.b, ss.k);
                }
                head += __popc(fmask);
            }
        }
    }
    // every thread's ITEMS particles of the blocked pass below lie in its own warp's chunk
    __syncwarp();
    DPOMP_STAMP(0, 3);

    pdl_trigger();
    // ---- convergent pass (blocked: thread owns ITEMS consecutive particles): observation log-weight
    // (src/hmm_examples.jl:63-65, exp deferred) and vectorised write-back of states and log weights
    // The log-weight depends on the particle only through the integer |sum(y) - sum(x)| =: d (Int64 observations and
    // counts), and it is non-increasing in d, so: the tile maximum m_b is the log-weight of the smallest d (an integer
    // min-reduction), and exp(logw - m_b) comes from a per-CTA table indexed by d - d_min, each entry evaluated with
    // exactly the per-particle f64 expression (bit-identical to the direct evaluation, one exp per thread instead of
    // ITEMS).  Offsets beyond the table and non-integer / huge sum(y) take the direct expression.
    double av[ITEMS], incl[ITEMS], excl[ITEMS];
    auto logw_of = [&](double d) -> double {  // tmp1 - (y - x)^2 / tmp2 (src/hmm_examples.jl:63-65)
        const double dd = __dmul_rn(d, d);
        const double quot = m.obs_tmp2_pow2 ? __dmul_rn(dd, m.obs_inv_tmp2) : __ddiv_rn(dd, m.obs_tmp2);
        return m.obs_tmp1 - quot;
    };
    constexpr unsigned kExcluded = 0xffffffffu;  // padding slot or particle that hit the event cap: weight 0
    const bool int_obs = fabs(ysum) < 1073741824.0 && ysum == rint(ysum);  // CTA-uniform
    double m_b;
    {
        int xs[ITEMS];
#pragma unroll
        for (int kk = 0; kk < ITEMS; ++kk) xs[kk] = 0;
#pragma unroll
        for (int c = 0; c < C; ++c)
            if (c < n_comp) {
                Vec v;
#pragma unroll
                for (int kk = 0; kk < ITEMS; ++kk) v.v[kk] = (int)st_s[c * TILE + tid * ITEMS + kk];
#pragma unroll
                for (int kk = 0; kk < ITEMS; ++kk) xs[kk] += m.xmask_i[c] * v.v[kk];
                if (!resample_here)  // (fused + resampling: the pre-resampling states are never read from HBM again)
                    *reinterpret_cast<Vec*>(pop_b + (size_t)c * a.n_pad + base_n + tid * ITEMS) = v;  // padding slots included
            }
        const Vec of = *reinterpret_cast<const Vec*>(ovf_s + tid * ITEMS);
        bool excluded[ITEMS];
#pragma unroll
        for (int kk = 0; kk < ITEMS; ++kk) excluded[kk] = !(base_n + tid * ITEMS + kk < a.n) || of.v[kk] < 0;

        // event statistics (padding slots are never parked and stay 0): one RED per warp, spread over one counter per
        // (filter, group of tiles) -- round 1 put all 4096 REDs of a C2 launch on ONE address (0.8 us per observation),
        // summing along the combine tree instead lengthened the serial tail by more than that; the counters are summed by a
        // tiny kernel at the end of the call (capi.cu).  Issued by lane 1: thread 0 takes the tickets below, and its
        // __threadfence would wait for its own RED
        unsigned long long ev_w = 0, ovf_w = 0;
#pragma unroll
        for (int kk = 0; kk < ITEMS; ++kk) {
            ev_w += (uint32_t)of.v[kk] & 0x7fffffffu;
            ovf_w += of.v[kk] < 0;
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            ev_w += __shfl_xor_sync(0xffffffffu, ev_w, d);
            ovf_w += __shfl_xor_sync(0xffffffffu, ovf_w, d);
        }
        if (lane == 1 && ev_w) atomicAdd(a.grp_ev + (size_t)b * a.ngroups + tile / kGroupTiles, ev_w);
        if (lane == 1 && ovf_w) atomicAdd(a.ovf_count, ovf_w);

        if constexpr (COUNT) {
            // Count families: the log pmf is not monotone in |Y - X|, so there is no integer min-reduction or exp table; every
            // particle takes the direct path.  The (filter, observation) constants are CTA-uniform and formed once.
            const CountObsConst cc = count_obs_const(a.cobs, th, t, ysum);
            double it[ITEMS], mloc = -INFINITY;
#pragma unroll
            for (int kk = 0; kk < ITEMS; ++kk) {
                it[kk] = excluded[kk] ? -INFINITY : count_obs_logpmf(cc, ysum, (double)xs[kk]);
                mloc = fmax(mloc, it[kk]);
            }
            if (a.record_logw) {
                double* lw_b = a.logw + (size_t)b * a.n_pad + base_n + (size_t)tid * ITEMS;
#pragma unroll
                for (int kk = 0; kk < ITEMS; ++kk) lw_b[kk] = it[kk];
            }
            m_b = block_max(mloc, warp_scratch);
            const double ref = (m_b == -INFINITY) ? 0.0 : m_b;
#pragma unroll
            for (int kk = 0; kk < ITEMS; ++kk) av[kk] = (it[kk] == -INFINITY) ? 0.0 : exp(it[kk] - ref);
        } else if (int_obs) {
            const int ys = (int)ysum;
            unsigned du[ITEMS], dloc = kExcluded;
#pragma unroll
            for (int kk = 0; kk < ITEMS; ++kk) {
                const long long df = (long long)ys - (long long)xs[kk];
                du[kk] = excluded[kk] ? kExcluded : (unsigned)(df < 0 ? -df : df);  // < 2^32 - 1
                dloc = min(dloc, du[kk]);
            }
            dloc = __reduce_min_sync(0xffffffffu, dloc);
            if (lane == 0) warp_min_s[warp] = dloc;
            __syncthreads();
            unsigned dmin = warp_min_s[0];
#pragma unroll
            for (int w = 1; w < kBlockThreads / 32; ++w) dmin = min(dmin, warp_min_s[w]);
            if (dmin == kExcluded) {  // no particle with a weight in this tile
                m_b = -INFINITY;
#pragma unroll
                for (int kk = 0; kk < ITEMS; ++kk) av[kk] = 0.0;
            } else {
                m_b = logw_of((double)dmin);
                wtab_s[tid] = exp(logw_of((double)dmin + (double)tid) - m_b);
                __syncthreads();
#pragma unroll
                for (int kk = 0; kk < ITEMS; ++kk) {
                    const unsigned off = du[kk] - dmin;
                    av[kk] = du[kk] == kExcluded ? 0.0
                           : (off < (unsigned)kBlockThreads ? wtab_s[off] : exp(logw_of((double)du[kk]) - m_b));
                    DPOMP_CHECK_IDX(du[kk] == kExcluded ? 0u : (off < (unsigned)kBlockThreads ? off : 0u), kBlockThreads);
                }
            }
            if (a.record_logw) {
                double* lw_b = a.logw + (size_t)b * a.n_pad + base_n + (size_t)tid * ITEMS;
#pragma unroll
                for (int kk = 0; kk < ITEMS; ++kk) lw_b[kk] = du[kk] == kExcluded ? -INFINITY : logw_of((double)du[kk]);
            }
        } else {
            double it[ITEMS], mloc = -INFINITY;
#pragma unroll
            for (int kk = 0; kk < ITEMS; ++kk) {
                it[kk] = excluded[kk] ? -INFINITY : logw_of(ysum - (double)xs[kk]);
                mloc = fmax(mloc, it[kk]);
            }
            if (a.record_logw) {
                double* lw_b = a.logw + (size_t)b * a.n_pad + base_n + (size_t)tid * ITEMS;
#pragma unroll
                for (int kk = 0; kk < ITEMS; ++kk) lw_b[kk] = it[kk];
            }
            m_b = block_max(mloc, warp_scratch);
            const double ref = (m_b == -INFINITY) ? 0.0 : m_b;
#pragma unroll
            for (int kk = 0; kk < ITEMS; ++kk) av[kk] = (it[kk] == -INFINITY) ? 0.0 : exp(it[kk] - ref);
        }
    }
    DPOMP_STAMP(0, 4);
    // tile partials (m_b, s_b) in the blocked item order of the scan tree
    const double s_b = tile_scan<ITEMS, false>(av, incl, excl, warp_scratch);
    // ---- two-level combine of the tile partials, each level done by whoever finishes last (tickets) -----------------
    // level 1: the kGroupTiles tiles of a group, level 2: the groups of the filter.  Both levels are one warp with the
    // same tree (one value per lane, Kogge-Stone over the lanes, chunks of 32 chained sequentially): no block barriers on
    // the serial tail of the kernel.
    DPOMP_STAMP(0, 5);
    const int grp = tile / kGroupTiles;
    const int grp_tiles = min(kGroupTiles, a.ntiles - grp * kGroupTiles);
    // Only warp 0 stays for the tickets; in the two-kernel path the other warps are done (no block barrier on the tail).
    int grp_last = 0;
    if (tid == 0) {
        a.tile_m[(size_t)b * a.ntiles + tile] = m_b;
        a.tile_s[(size_t)b * a.ntiles + tile] = s_b;
        __threadfence();
        const unsigned int ticket = atomicAdd(&a.grp_counter[(size_t)b * a.ngroups + grp], 1u);
        grp_last = (ticket == (unsigned int)(grp_tiles - 1));
    }
    // the scan goes out AFTER thread 0 took its ticket: its consumer is the next kernel, and the fence above then has no
    // bulk stores of this thread to wait for
    if (!resample_here) {  // the tile-local inclusive scan of exp(logw - m_b) is all the resample kernel needs
        double* wt_b = a.wtile + (size_t)b * a.n_pad + base_n + (size_t)tid * ITEMS;
        if constexpr (ITEMS % 2 == 0) {
#pragma unroll
            for (int kk = 0; kk < ITEMS; kk += 2) *reinterpret_cast<double2*>(wt_b + kk) = make_double2(incl[kk], incl[kk + 1]);
        } else {
#pragma unroll
            for (int kk = 0; kk < ITEMS; ++kk) wt_b[kk] = incl[kk];
        }
    }
    if (tid < 32) grp_last = __shfl_sync(0xffffffffu, grp_last, 0);
    if (grp_last && tid < 32) {
    // level 1: tiles of this group -> f_{b|g}, o_{b|g}, (m_g, s_g)
    int last_group = 0;
    {
        const int i = grp * kGroupTiles + tid;
        const bool have = i < a.ntiles;
        const double mb = have ? __ldcg(a.tile_m + (size_t)b * a.ntiles + i) : -INFINITY;
        const double sb = have ? __ldcg(a.tile_s + (size_t)b * a.ntiles + i) : 0.0;
        double mg = mb;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) mg = fmax(mg, __shfl_xor_sync(0xffffffffu, mg, d));
        const double f = (mb == -INFINITY) ? 0.0 : exp(mb - mg);
        double inc = __dmul_rn(f, sb);
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const double y = __shfl_up_sync(0xffffffffu, inc, d);
            if (tid >= d) inc = __dadd_rn(y, inc);
        }
        double prev = __shfl_up_sync(0xffffffffu, inc, 1);
        if (tid == 0) prev = 0.0;
        if (have) {
            a.tile_f[(size_t)b * a.ntiles + i] = f;
            a.tile_off[(size_t)b * a.ntiles + i] = prev;
        }
        if (tid == 31) {
            a.grp_m[(size_t)b * a.ngroups + grp] = mg;
            a.grp_s[(size_t)b * a.ngroups + grp] = inc;
            a.grp_counter[(size_t)b * a.ngroups + grp] = 0u;
            // Plain kernel with the resample kernel behind it: the kernel boundary publishes the group partials and every
            // resample CTA runs level 2 (<= 64 values) itself while its tile loads are in flight -- the second ticket level
            // (fence, atomic, dependent load, combine: ~2.5 us on the serial tail of the last tile) is gone.
            if (!(MODE == kModePlain && a.defer_l2)) {
                __threadfence();
                const unsigned int ticket = atomicAdd(&a.tile_counter[b], 1u);
                last_group = (ticket == (unsigned int)(a.ngroups - 1));
            }
        }
        last_group = __shfl_sync(0xffffffffu, last_group, 31);
    }
    if (last_group) {
    // level 2: groups of the filter -> M, F_g = exp(m_g - M), O_g, S and the log-likelihood increment
    const Level2 l2 = combine_level2(a.grp_m + (size_t)b * a.ngroups, a.grp_s + (size_t)b * a.ngroups, a.ngroups,
                                     a.grp_f + (size_t)b * a.ngroups, a.grp_off + (size_t)b * a.ngroups);
    if (tid == 0) {
        a.filt_s[b] = l2.big_s;
        a.filt_m[b] = l2.big_m;
        // log(cum_weight[end] / N) (:60) as log-sum-exp; one add per kernel and filter, so the RED is deterministic
        if (has_lik) atomicAdd(&a.ll_acc[b], l2.big_m + log(l2.big_s / (double)a.n));
        a.tile_counter[b] = 0u;
    }
    if constexpr (FUSED) {  // publish the combine to the CTAs of this filter that wait below: one flag per group of tiles
        __syncwarp();       // (own 128-byte line: kGroupTiles pollers per address instead of every tile of the filter on one)
        __threadfence();
        for (int g = tid; g < a.ngroups; g += 32)
            *reinterpret_cast<volatile unsigned int*>(a.gen_flags + ((size_t)b * a.ngroups + g) * 32) = a.gen;
    }
    if constexpr (PERSIST) {  // one flag per group of tiles (own 128-byte line): kGroupTiles pollers per address, not ntiles
        __syncwarp();
        __threadfence();
        for (int g = tid; g < a.ngroups; g += 32)
            *reinterpret_cast<volatile unsigned int*>(a.gen_flags + ((size_t)b * a.ngroups + g) * 32) = gen_t;
    }
    }  // last_group
    }  // group-last warp
    DPOMP_STAMP(0, 6);

    if constexpr (FUSED) {
        if (!do_rs) return;
        // ---- wait for this filter's combine, then resample the tile from shared memory ---------------------------------
        if (tid == 0) {
            const unsigned int* flag = a.gen_flags + ((size_t)b * a.ngroups + grp) * 32;
            while (ld_acquire_u32(flag) != a.gen) __nanosleep(32);
        }
        __syncthreads();
        DPOMP_STAMP(1, 1);
        const RsArgs ra{a.tile_f, a.tile_off, a.grp_f, a.grp_off, a.filt_s, nullptr, nullptr, nullptr, a.pop_dst, a.anc, a.n, a.n_pad,
                        a.ntiles, a.ngroups, a.n_comp, t, a.rs_type, a.key, a.perm};
        // ovf_s (TILE ints) is free after the weight pass: it becomes the per-warp offspring windows
        resample_tile<ITEMS, SState, true, 0, true, (RMODEL != kModelGeneric ? C : 0)>(ra, b, tile, gfilter, incl, st_s, TILE, ovf_s,
                                                                                      warp_max_s, lohi_s);
        DPOMP_STAMP(1, 4);
    }
    if constexpr (PERSIST) {
        // ---- wait for this filter's combine (also when this observation does not resample: the ticket counters are only
        // reusable after it) ------------------------------------------------------------------------------------------------
        if (tid == 0) {
            const unsigned int* flag = a.gen_flags + ((size_t)b * a.ngroups + grp) * 32;
            while (ld_acquire_u32(flag) != gen_t) __nanosleep(40);
        }
        __syncthreads();
        if (do_rs) {
            const RsArgs ra{a.tile_f, a.tile_off, a.grp_f, a.grp_off, a.filt_s, nullptr, nullptr, nullptr, pop_other, a.anc, a.n, a.n_pad,
                            a.ntiles, a.ngroups, a.n_comp, t, a.rs_type, a.key, a.perm};
            resample_tile<ITEMS, SState, true, 0, false>(ra, b, tile, gfilter, incl, st_s, TILE, ovf_s, warp_max_s, lohi_s);
            // every offspring row of this tile is written: add the row counts to the counters of the destination tiles
            __threadfence();
            __syncthreads();
            const long long lo = lohi_s[0], hi = lohi_s[1];
            if (hi > lo) {
                const int d0 = (int)(lo / TILE), d1 = (int)((hi - 1) / TILE);
                for (int d = d0 + tid; d <= d1; d += kBlockThreads) {
                    const long long from = max(lo, (long long)d * TILE), to = min(hi, (long long)(d + 1) * TILE);
                    atomicAdd(a.rows_done + (size_t)b * a.ntiles + d, (unsigned int)(to - from));
                }
            }
            ++flip;
            wait_rows = true;
            staged = false;
        } else {
            wait_rows = false;
            staged = true;
        }
    }
    } while (PERSIST && ++t <= t_end);  // observations
}

// ---- host-side model padding and dispatch ---------------------------------------------------------------------
template <typename Real, int C, int E>
static DevModel<Real, C, E> make_dev_model(const ModelHost& mh) {
    const dpomp_model_desc& d = mh.desc;
    DevModel<Real, C, E> m{};
    const int e_real = d.n_events;
    m.any_den = 0;
    for (int e = 0; e < E; ++e) {
        const int src = e < e_real ? e : e_real - 1;  // padded events: zero rate, transition row of the last real event
        const bool pad = e >= e_real;
        m.par[e] = pad ? -1 : d.rate_par[src];
        m.k1[e] = pad ? (Real)0 : (Real)d.rate_k1[src];
        m.k2[e] = pad ? (Real)0 : (Real)d.rate_k2[src];
        m.kd[e] = pad ? (Real)1 : (Real)d.rate_kd[src];
        m.has_den[e] = pad ? 0 : d.rate_has_den[src];
        m.any_den |= m.has_den[e];
        for (int c = 0; c < C; ++c) {
            const bool cpad = c >= d.n_compartments;
            m.f1[e][c] = (pad || cpad) ? (Real)0 : (Real)d.rate_f1[src][c];
            m.f2[e][c] = (pad || cpad) ? (Real)0 : (Real)d.rate_f2[src][c];
            m.dn[e][c] = (pad || cpad) ? (Real)0 : (Real)d.rate_dn[src][c];
            m.trans[e][c] = cpad ? (Real)0 : (Real)d.trans[src][c];
        }
    }
    for (int c = 0; c < C; ++c) {
        const bool cpad = c >= d.n_compartments;
        m.xmask_i[c] = cpad ? 0 : (int)d.obs_xmask[c];
        m.ic[c] = cpad ? 0 : (int)d.initial_condition[c];
    }
    m.obs_tmp1 = log(1.0 / (sqrt(2.0 * 3.14159265358979323846) * d.obs_sigma));
    m.obs_tmp2 = 2.0 * d.obs_sigma * d.obs_sigma;
    {
        int ex = 0;
        m.obs_tmp2_pow2 = frexp(m.obs_tmp2, &ex) == 0.5 ? 1 : 0;  // then x / tmp2 == x * (1 / tmp2) bit for bit
        m.obs_inv_tmp2 = 1.0 / m.obs_tmp2;
    }
    m.t0_index = d.t0_index;
    m.n_params = d.n_params;
    return m;
}

// mode 0: launch the plain kernel, 1: launch the fused kernel, 2: return the fused kernel's co-resident CTA capacity,
// 3: launch the persistent kernel cooperatively (all observations of the call in one launch), 4: its co-resident capacity
template <typename Real, int C, int E, int ITEMS, int MODEL = kModelGeneric, int ILP = DPOMP_SIM_ILP>
static int sim_inst(const ModelHost& mh, const SimLaunch& a, cudaStream_t stream, int mode) {
    constexpr int TILE = kBlockThreads * ITEMS;
    const size_t smem = (size_t)TILE * (1 + C) * sizeof(int);
    auto kern = pf_sim_weight_kernel<Real, C, E, ITEMS, MODEL, kModePlain, ILP>;
    auto kern_fused = pf_sim_weight_kernel<Real, C, E, ITEMS, MODEL, kModeFused, ILP>;
    static bool configured = false;
    if (!configured) {
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        cudaFuncSetAttribute(kern_fused, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(kern_fused, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        configured = true;
    }
    if (mode == 2) {
        int per_sm = 0, dev = 0, sms = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern_fused, kBlockThreads, smem) != cudaSuccess) return 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        return per_sm * sms;
    }
    if constexpr (sizeof(Real) == 4 && MODEL > kModelGeneric) {
        // the persistent kernel is instantiated for the f32 loop of the predefined models
        auto kern_p = pf_sim_weight_kernel<Real, C, E, ITEMS, MODEL, kModePersist, ILP>;
        static bool configured_p = false;
        if (!configured_p) {
            cudaFuncSetAttribute(kern_p, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            cudaFuncSetAttribute(kern_p, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            configured_p = true;
        }
        if (mode == 4) {
            int per_sm = 0, dev = 0, sms = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern_p, kBlockThreads, smem) != cudaSuccess) return 0;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
            return per_sm * sms;
        }
        if (mode == 3) {
            const DevModel<Real, C, E> m = make_dev_model<Real, C, E>(mh);
            cudaLaunchConfig_t cfg{};
            cfg.gridDim = dim3((unsigned)(a.n_filters * a.ntiles));
            cfg.blockDim = dim3(kBlockThreads);
            cfg.dynamicSmemBytes = smem;
            cfg.stream = stream;
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeCooperative;  // all CTAs co-resident, or the launch fails
            attr[0].val.cooperative = 1;
            cfg.attrs = attr;
            cfg.numAttrs = 1;
            return (int)cudaLaunchKernelEx(&cfg, kern_p, m, a);
        }
    }
    if (mode == 4) return 0;
    if (mode == 3) return (int)cudaErrorInvalidValue;
    const DevModel<Real, C, E> m = make_dev_model<Real, C, E>(mh);
    const unsigned grid = (unsigned)(a.n_filters * a.ntiles);
    return (int)(mode == 1 ? launch_pdl(kern_fused, grid, kBlockThreads, smem, stream, m, a)
                           : launch_pdl(kern, grid, kBlockThreads, smem, stream, m, a));
}

// Plain kernel of a predefined model on 1024-particle tiles with TWO particles per lane and the Philox words drawn one attempt
// ahead (the loop of the latency regime): for event-heavy models (>= ~16 events per particle and interval: rare refills) in
// launches that under-fill the device it is the faster loop -- 64 x 4096 LOTKA 9.24 -> 7.20 ms -- and the slower one for every
// ~2-events-per-interval model and for full launches (profiles/r2_experiments.md 15, 16); the host selects it per call from
// the event intensity of the handle's previous call (SimLaunch::two_per_lane).  Same counters, same draws: bit-identical.
template <typename Real, int C, int E, int ITEMS, int MODEL>
static int sim_plain_two_per_lane(const ModelHost& mh, const SimLaunch& a, cudaStream_t stream) {
    constexpr int TILE = kBlockThreads * ITEMS;
    const size_t smem = (size_t)TILE * (1 + C) * sizeof(int);
    auto kern = pf_sim_weight_kernel<Real, C, E, ITEMS, MODEL, kModePlain, 2>;
    static bool configured = false;
    if (!configured) {
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        configured = true;
    }
    const DevModel<Real, C, E> m = make_dev_model<Real, C, E>(mh);
    return (int)launch_pdl(kern, (unsigned)(a.n_filters * a.ntiles), kBlockThreads, smem, stream, m, a);
}

constexpr int kLatencyRegimeCtas = 296;  // 2 CTAs per SM
// the instantiated generic (C, E) shapes; a model runs on the smallest shape that covers it
#define DPOMP_SIM_SHAPES(X) X(2, 1) X(2, 2) X(2, 3) X(3, 2) X(3, 3) X(4, 3) X(4, 6) X(8, 8)
#define DPOMP_SIM_BUILTINS(X) X(kModelSI) X(kModelSIR) X(kModelSIS) X(kModelSEI) X(kModelSEIR) X(kModelSEIS) X(kModelLOTKA)

template <typename Real>
static int sim_typed(const ModelHost& mh, int items, const SimLaunch& a, cudaStream_t stream, int mode) {
    const int c = mh.desc.n_compartments, e = mh.desc.n_events;
    const int model_id = builtin_model_id(mh.desc);
    // latency regime: a few small filters (the reference's default 200 particles) leave most of the device idle, and a lane
    // that interleaves its two particles halves the dependent chain of a step
    const bool latency = sizeof(Real) == 4 && items == kItemsSmall && a.n_filters > 0 &&
                         (long long)a.n_filters * a.ntiles <= kLatencyRegimeCtas;
#define X(ID)                                                                                                             \
    if (model_id == ID) {                                                                                                 \
        if (items == kItemsSmall)                                                                                         \
            return latency ? sim_inst<Real, Builtin<ID>::C, Builtin<ID>::E, kItemsSmall, ID, 2>(mh, a, stream, mode)      \
                           : sim_inst<Real, Builtin<ID>::C, Builtin<ID>::E, kItemsSmall, ID, 1>(mh, a, stream, mode);     \
        if constexpr (sizeof(Real) == 4 && DPOMP_SIM_ILP == 1) {                                                          \
            if (mode == 0 && a.two_per_lane)                                                                              \
                return sim_plain_two_per_lane<Real, Builtin<ID>::C, Builtin<ID>::E, kItemsLarge, ID>(mh, a, stream);      \
        }                                                                                                                 \
        return sim_inst<Real, Builtin<ID>::C, Builtin<ID>::E, kItemsLarge, ID>(mh, a, stream, mode);                      \
    }
    DPOMP_SIM_BUILTINS(X)
#undef X
#define X(CC, EE)                                                                                      \
    if (c <= CC && e <= EE) {                                                                          \
        return items == kItemsSmall ? sim_inst<Real, CC, EE, kItemsSmall>(mh, a, stream, mode)         \
                                    : sim_inst<Real, CC, EE, kItemsLarge>(mh, a, stream, mode);        \
    }
    DPOMP_SIM_SHAPES(X)
#undef X
    return (mode == 2 || mode == 4) ? 0 : (int)cudaErrorInvalidValue;
}

// count observation families: the generic (C, E) shapes only -- never the predefined-model, persistent or two-per-lane kernels
template <typename Real>
static int sim_count_typed(const ModelHost& mh, int items, const SimLaunch& a, cudaStream_t stream, int mode) {
    if (mode == 3 || mode == 4) return mode == 4 ? 0 : (int)cudaErrorInvalidValue;
    const int c = mh.desc.n_compartments, e = mh.desc.n_events;
#define X(CC, EE)                                                                                                \
    if (c <= CC && e <= EE) {                                                                                    \
        return items == kItemsSmall ? sim_inst<Real, CC, EE, kItemsSmall, kModelCountObs>(mh, a, stream, mode) \
                                    : sim_inst<Real, CC, EE, kItemsLarge, kModelCountObs>(mh, a, stream, mode); \
    }
    DPOMP_SIM_SHAPES(X)
#undef X
    return mode == 2 ? 0 : (int)cudaErrorInvalidValue;
}

}  // namespace dpomp
