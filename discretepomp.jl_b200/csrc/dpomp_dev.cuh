// dpomp_dev.cuh -- device-side building blocks shared by the particle-filter kernels (sm_100a).
//   * Philox4x32-10 counter-based RNG and the stream layout of DESIGN.md ("random streams")
//   * the deterministic block scan tree (DESIGN.md "deterministic scan tree")
//   * the counting form of the systematic / stratified search with the reference's exact f64 expressions
//     (src/hmm_pf_resample.jl:24-42, src/hmm_resample.jl:66-83 of the reference)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/dpomp.h"

namespace dpomp {

// CTA geometry of the particle-filter kernels.  128 threads x 8 particles per thread (1024-particle tiles) lets 7-8 CTAs
// share an SM, so the 1024 tiles of a 2^20-particle filter are all resident at once (148 x 7 = 1036 slots): no second
// wave, and 8 particles per lane keep the warp work queues full longer.  Filters of <= 256 particles use 2 per thread.
#ifndef DPOMP_BLOCK_THREADS
#define DPOMP_BLOCK_THREADS 128
#endif
#ifndef DPOMP_ITEMS_LARGE
#define DPOMP_ITEMS_LARGE 8
#endif
#ifndef DPOMP_ITEMS_SMALL
#define DPOMP_ITEMS_SMALL 2
#endif
// Debug build only (-DDPOMP_PHASE_TIMERS, scripts/phase_probe.py): thread 0 of every CTA stamps %globaltimer at phase
// boundaries of the launches of observation index DPOMP_PHASE_OBS into a device array read back by dpomp_debug_phases.
#ifdef DPOMP_PHASE_TIMERS
#ifndef DPOMP_PHASE_OBS
#define DPOMP_PHASE_OBS 50
#endif
static __device__ unsigned long long g_dpomp_phase[2][4096][8];  // one copy per translation unit (no -rdc)
__device__ __forceinline__ unsigned long long dpomp_gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define DPOMP_STAMP(K, P)                                                                                   \
    do {                                                                                                    \
        if (threadIdx.x == 0 && a.t == DPOMP_PHASE_OBS && blockIdx.x < 4096) g_dpomp_phase[K][blockIdx.x][P] = dpomp_gtime(); \
    } while (0)
// slot P of the simulate kernel of the FOLLOWING observation (the resample -> simulate boundary of the timeline)
#define DPOMP_STAMP_NEXT(K, P)                                                                              \
    do {                                                                                                    \
        if (threadIdx.x == 0 && a.t == DPOMP_PHASE_OBS + 1 && blockIdx.x < 4096) g_dpomp_phase[K][blockIdx.x][P] = dpomp_gtime(); \
    } while (0)
#else
#define DPOMP_STAMP(K, P) do { } while (0)
#define DPOMP_STAMP_NEXT(K, P) do { } while (0)
#endif
// Debug build only (-DDPOMP_BOUNDS_CHECK, lib/variants/libdpomp_bounds.so, tests/test_gpu_bounds.py): every shared / global
// index of the resample phase, the warp work queue and the MBP windows is checked against its buffer and traps (the pool's
// compute-sanitizer is closed, SURVEY.md 5).  The release build compiles the checks away.
#ifdef DPOMP_BOUNDS_CHECK
#define DPOMP_CHECK_IDX(i, n)                                                                                          \
    do {                                                                                                               \
        if (!((long long)(i) >= 0 && (long long)(i) < (long long)(n))) {                                               \
            printf("dpomp bounds: %s:%d: index %lld outside [0, %lld)\n", __FILE__, __LINE__, (long long)(i), (long long)(n)); \
            __trap();                                                                                                  \
        }                                                                                                              \
    } while (0)
#else
#define DPOMP_CHECK_IDX(i, n) do { } while (0)
#endif
constexpr int kBlockThreads = DPOMP_BLOCK_THREADS;
constexpr int kItemsLarge = DPOMP_ITEMS_LARGE, kItemsSmall = DPOMP_ITEMS_SMALL;

// Programmatic dependent launch: consecutive kernels of one filter pass are launched with the
// programmatic-stream-serialization attribute, so the launch latency and block scheduling of kernel k+1 overlap the
// tail of kernel k; every kernel calls pdl_wait() before it touches memory written by its predecessor.
__device__ __forceinline__ void pdl_wait() {
#if __CUDA_ARCH__ >= 900
    cudaGridDependencySynchronize();
#endif
}
__device__ __forceinline__ void pdl_trigger() {
#if __CUDA_ARCH__ >= 900 && defined(DPOMP_PDL_TRIGGER)
    cudaTriggerProgrammaticLaunchCompletion();
#endif
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t stream, Args... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, args...);
}
// Two-level combination of the tile partials (DESIGN.md "deterministic scan tree"): kGroupTiles consecutive tiles form a
// group that is combined by the last of its tiles to finish (one warp), the groups by the last group to finish.
//   cw_q = O_g + F_g * (o_{b|g} + f_{b|g} * incl_q)
constexpr int kGroupTiles = 32;
// filters of at most this many groups (2^21 particles) leave level 2 of the combine to the resample kernel (pf_kernels.cu)
constexpr int kDeferGroups = 64;
__device__ __forceinline__ double tile_cw(double grp_off, double grp_f, double tile_o, double tile_f, double incl) {
    return __dadd_rn(grp_off, __dmul_rn(grp_f, __dadd_rn(tile_o, __dmul_rn(tile_f, incl))));
}
// ------------------------------------------------------------------------------------------------------------
// Level 2 of the combine (DESIGN.md "deterministic scan tree"), executed by ONE warp: the groups of a filter ->
// M = max m_g, F_g = exp(m_g - M), O_g = exclusive offsets (Kogge-Stone over the 32 lanes of a chunk, chunks chained
// sequentially), S = total.
// ------------------------------------------------------------------------------------------------------------
struct Level2 {
    double big_m, big_s;
};
// CG: the group partials were written by other SMs during this launch (read from L2); otherwise plain loads (written
// before the launch)
template <bool CG = true>
__device__ __forceinline__ Level2 combine_level2(const double* gm_b, const double* gs_b, int ngroups, double* grp_f_out,
                                                 double* grp_off_out) {
    auto ld = [](const double* p) -> double {
        if constexpr (CG) return __ldcg(p); else return *p;
    };
    const int lane = threadIdx.x & 31;
    double big_m = -INFINITY;
    for (int i = lane; i < ngroups; i += 32) big_m = fmax(big_m, ld(gm_b + i));
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) big_m = fmax(big_m, __shfl_xor_sync(0xffffffffu, big_m, d));
    double carry = 0.0;
    for (int c0 = 0; c0 < ngroups; c0 += 32) {
        const int i = c0 + lane;
        const bool have = i < ngroups;
        const double mg = have ? ld(gm_b + i) : -INFINITY;
        const double f = (mg == -INFINITY) ? 0.0 : exp(mg - big_m);
        double inc = have ? __dmul_rn(f, ld(gs_b + i)) : 0.0;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const double y = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc = __dadd_rn(y, inc);
        }
        double prev = __shfl_up_sync(0xffffffffu, inc, 1);
        if (lane == 0) prev = 0.0;
        if (have) {
            grp_f_out[i] = f;
            grp_off_out[i] = __dadd_rn(carry, prev);
        }
        carry = __dadd_rn(carry, __shfl_sync(0xffffffffu, inc, 31));
    }
    return Level2{big_m, carry};
}
// ------------------------------------------------------------------------------------------------------------
// Offspring placement (dpomp_pf_set_scatter).  The reference writes offspring i to row i (src/hmm_pf_resample.jl:38), so
// after systematic resampling neighbouring rows share their lineage and the work of the next simulation step clusters
// in a few tiles.  With the interleaved placement the 32-offspring chunk k goes to chunk position sigma(k), where sigma
// orders the full chunks by (k mod M, k div M) with M = number of tiles: consecutive chunks land in consecutive tiles and
// every tile receives a uniform sample of the lineages.  sigma is a bijection on the ncf = floor(N / 32) full chunks
// (ncf = q * M + r); the trailing partial chunk stays in place; ncf = 0 means identity (the reference's order).
// Particle order is arbitrary in a bootstrap filter; ancestors given (cw, u) are unchanged, only their rows move.
// ------------------------------------------------------------------------------------------------------------
struct ChunkPerm {
    int ncf, m, q, r;
};
__host__ __device__ __forceinline__ int chunk_sigma(const ChunkPerm& p, int rr, int qq) {  // < n_pad / 32
    return rr * p.q + (rr < p.r ? rr : p.r) + qq;
}
__host__ __device__ __forceinline__ long long perm_pos(const ChunkPerm& p, long long i) {
    const int k = (int)(i >> 5);
    if (k >= p.ncf) return i;
    return ((long long)chunk_sigma(p, k % p.m, k / p.m) << 5) | (i & 31);
}
inline ChunkPerm make_chunk_perm(int scatter_mode, long long n, int ntiles) {
    ChunkPerm p{0, 1, 0, 0};
    if (scatter_mode != 0 && ntiles > 1) {
        p.ncf = (int)(n >> 5);
        p.m = ntiles;
        p.q = p.ncf / ntiles;
        p.r = p.ncf % ntiles;
    }
    return p;
}

constexpr uint32_t kTagSim = 0u;
constexpr uint32_t kTagResample = 1u;

// ------------------------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011).  ctr = (particle, filter, observation, tag<<30 | block), key = 64-bit call key.
// ------------------------------------------------------------------------------------------------------------
struct Philox4 {
    uint32_t w0, w1, w2, w3;
};

__device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                                 uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return Philox4{c0, c1, c2, c3};
}

__device__ __forceinline__ Philox4 stream_draw(uint64_t key, uint32_t particle, uint32_t filter, uint32_t obs,
                                               uint32_t tag, uint32_t block) {
    return philox4x32_10(particle, filter, obs, (tag << 30) | block, (uint32_t)key, (uint32_t)(key >> 32));
}

// Philox2x32-10: 64-bit counter, 32-bit key.  One call = the two uniforms of one event attempt.
__device__ __forceinline__ uint2 philox2x32_10(uint32_t c0, uint32_t c1, uint32_t key) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi = __umulhi(0xD256D193u, c0), lo = 0xD256D193u * c0;
        c0 = hi ^ key ^ c1;
        c1 = lo;
        key += 0x9E3779B9u;
    }
    return make_uint2(c0, c1);
}

// Event-loop stream of one (call key, filter, observation): Philox2x32 key K and counter masks A, B, hashed once with
// Philox4x32-10 (DESIGN.md "random streams").  Attempt k of particle n draws philox2x32_10(n ^ A, k ^ B, K).
struct SimStream {
    uint32_t k, a, b;
};
__device__ __forceinline__ SimStream sim_stream_init(uint64_t key, uint32_t filter, uint32_t obs) {
    const Philox4 p = stream_draw(key, 0u, filter, obs, kTagSim, 0u);
    return SimStream{p.w0, p.w1, p.w2};
}

// (0,1) with 32-bit resolution; the f64 value is exact
__device__ __forceinline__ double u32_open_f64(uint32_t w) { return ((double)w + 0.5) * 0x1.0p-32; }
// f32 uniforms of the event loop (24-bit resolution after rounding):
//   waiting time: (0, 1] -- never 0 (log stays finite); the top 128 words round to exactly 1.0f, i.e. a zero waiting time
//                 with probability 3e-8 per draw (harmless: the reference's rand() is [0,1), -log(1-u) has the same law)
//   event choice: [0, 1) like the reference's rand() (src/hmm_cmn.jl:5) -- round toward zero, so the largest value is
//                 1 - 2^-24 and fl(u * R) < R for every R > 0: `cum[i] > etc` always holds for some event with a positive
//                 rate and choose_event can never fall through to a zero-rate last event
__device__ __forceinline__ float u32_wait_f32(uint32_t w) { return fmaf(__uint2float_rn(w), 0x1.0p-32f, 0x1.0p-33f); }
__device__ __forceinline__ float u32_event_f32(uint32_t w) { return __uint2float_rz(w) * 0x1.0p-32f; }
// The two XU operations of the f32 waiting time, pinned to their flush-to-zero forms whatever -ftz the translation unit is
// built with (the non-ftz forms add a denormal scaling and, for the quotient, a range fix-up around the MUFU):
//   lg2_ftz: the argument is u32_wait_f32(w) >= 2^-33, never subnormal, so the ftz form returns the same value;
//   rcp_ftz: for every normal total rate the same value as the non-ftz reciprocal.  A subnormal rate (flushed to 0) gives
//            +inf instead of ~1e38, so the new remaining time is -inf or NaN rather than a huge negative number: the attempt
//            fails `t_new >= 0` either way.
__device__ __forceinline__ float lg2_ftz(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_ftz(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// [0,1) with 53-bit resolution (Julia's rand() range) for the resampling draws
__device__ __forceinline__ double u53(uint32_t hi, uint32_t lo) {
    return (double)(((uint64_t)hi << 21) | (uint64_t)(lo >> 11)) * 0x1.0p-53;
}

// ------------------------------------------------------------------------------------------------------------
// Deterministic tile scan.  Thread `tid` (lane l of warp w) owns ITEMS consecutive values a[0..ITEMS).
//   r_k   = a_0 + ... + a_k          (left to right)
//   I_l   = Kogge-Stone inclusive scan over lanes of r_{ITEMS-1}
//   P_w   = W_0 + ... + W_{w-1}      (left to right over warps, W_w = I_31 of warp w)
//   incl_k = (P_w + I_{l-1}) + r_k ,  excl_k = (P_w + I_{l-1}) + r_{k-1}
// Returns the tile total P_{nw-1} + W_{nw-1}.  All adds are round-to-nearest f64, never contracted.
// `warp_tot` is shared scratch of kBlockThreads/32 doubles.  Contains two __syncthreads(); the trailing one (TAIL_SYNC)
// only protects `warp_tot` against reuse and may be dropped when nothing writes the scratch afterwards.
// ------------------------------------------------------------------------------------------------------------
template <int ITEMS, bool TAIL_SYNC = true>
__device__ __forceinline__ double tile_scan(const double (&a)[ITEMS], double (&incl)[ITEMS], double (&excl)[ITEMS],
                                            double* warp_tot) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double r[ITEMS];
    r[0] = a[0];
#pragma unroll
    for (int k = 1; k < ITEMS; ++k) r[k] = __dadd_rn(r[k - 1], a[k]);
    double inc = r[ITEMS - 1];
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const double y = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc = __dadd_rn(y, inc);
    }
    double prev = __shfl_up_sync(0xffffffffu, inc, 1);
    if (lane == 0) prev = 0.0;
    if (lane == 31) warp_tot[warp] = inc;
    __syncthreads();
    double prefix = 0.0, total = 0.0;
#pragma unroll
    for (int w = 0; w < kBlockThreads / 32; ++w) {
        if (w == warp) prefix = total;
        total = __dadd_rn(total, warp_tot[w]);
    }
    const double base = __dadd_rn(prefix, prev);
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        incl[k] = __dadd_rn(base, r[k]);
        excl[k] = __dadd_rn(base, k > 0 ? r[k - 1] : 0.0);
    }
    if constexpr (TAIL_SYNC) __syncthreads();
    return total;
}

__device__ __forceinline__ double block_max(double v, double* warp_scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, d));
    if (lane == 0) warp_scratch[warp] = v;
    __syncthreads();
    double m = warp_scratch[0];
#pragma unroll
    for (int w = 1; w < kBlockThreads / 32; ++w) m = fmax(m, warp_scratch[w]);
    __syncthreads();
    return m;
}

// ------------------------------------------------------------------------------------------------------------
// Resampling uniforms in the reference's expression order and the counting form of the search.
//   systematic: u_i = ((r/N) + ((i-1)/N)) * S          (src/hmm_pf_resample.jl:27-32)
//   stratified: u_i = ((r_i/N) + ((i-1)/N)) * S        (src/hmm_resample.jl:69-73)
//   E(v) = #{ i in 1..N : u_i <= v }   -- u_i is non-decreasing in i, so ancestor(i) = first j with E(cw_j) >= i,
//   which is exactly the walk `while u[i] > cw[j]; j += 1`.
// ------------------------------------------------------------------------------------------------------------
struct ResampleCtx {
    int rs_type;
    long long n;
    double dn;        // (double) n
    double inv_n;     // exact iff n is a power of two
    bool pow2;
    double s;         // cw[end]
    double inv_s;     // only used for the (inexact) initial guess
    double r1_over_n; // systematic: r / N
    uint64_t key;
    uint32_t filter, obs;
};

__device__ __forceinline__ double div_by_n(const ResampleCtx& c, double v) {
    return c.pow2 ? v * c.inv_n : __ddiv_rn(v, c.dn);
}

// RS: compile-time resampler (DPOMP_RS_SYSTEMATIC / DPOMP_RS_STRATIFIED) or 0 = take c.rs_type at run time.  The
// systematic instantiation contains no Philox code: the stand-alone resample kernel shrinks from 5176 to a fraction of
// the SASS instructions (round 1: stalled_no_instruction 1.84 per issue from instruction-cache misses).
template <int RS = 0>
__device__ __forceinline__ double resample_u(const ResampleCtx& c, int i /*1-based, n < 2^31*/) {
    const double q = div_by_n(c, (double)(i - 1));
    double r = c.r1_over_n;
    if ((RS ? RS : c.rs_type) == DPOMP_RS_STRATIFIED) {
        const Philox4 p = stream_draw(c.key, (uint32_t)(i - 1), c.filter, c.obs, kTagResample, 1u);
        r = div_by_n(c, u53(p.w0, p.w1));
    }
    return __dmul_rn(__dadd_rn(r, q), c.s);
}

// The count in two steps: a closed-form guess (`exact` = it needs no verification) and the exact correction by
// comparisons with u_i.  Callers with many values per thread take the guess for all of them first and run ONE copy of
// the correction code for the few that need it (resample_tile), instead of one inlined copy per value.
template <int RS = 0>
__device__ __forceinline__ int resample_ecount_guess(const ResampleCtx& c, double v, bool& exact) {
    const int n = (int)c.n;
    exact = true;
    if (!(c.s > 0.0)) return n;
    double g;
    if ((RS ? RS : c.rs_type) == DPOMP_RS_STRATIFIED) {
        g = floor(v * c.inv_s * c.dn);
    } else {
        // u_i <= v  <=>  i <= t + 1 with t = v N / S - r in exact arithmetic.  The f64 evaluation of t and the rounding of
        // the reference's expression for u_i are both off by < 2^-20 index units for N < 2^31, so unless t lies within
        // 2^-12 of an integer (or outside (0, N - 1)) the count is floor(t) + 1 and needs no verification.
        const double t = (v * c.inv_s - c.r1_over_n) * c.dn;
        const double fl = floor(t);
        const double frac = t - fl;
#ifndef DPOMP_NO_ECOUNT_FAST
        if (frac > 0x1.0p-12 && frac < 1.0 - 0x1.0p-12 && t > 0.0 && t < c.dn - 1.0) return (int)fl + 1;
#endif
        g = fl + 1.0;
    }
    exact = false;
    return (int)fmin(fmax(g, 0.0), c.dn);
}
template <int RS = 0>
__device__ __forceinline__ int resample_ecount_correct(const ResampleCtx& c, double v, int e) {
    const int n = (int)c.n;
    while (e < n && resample_u<RS>(c, e + 1) <= v) ++e;
    while (e > 0 && resample_u<RS>(c, e) > v) --e;
    return e;
}
template <int RS = 0>
__device__ __forceinline__ long long resample_ecount(const ResampleCtx& c, double v) {
    bool exact;
    const int e = resample_ecount_guess<RS>(c, v, exact);
    return exact ? e : resample_ecount_correct<RS>(c, v, e);
}

__device__ __forceinline__ ResampleCtx make_resample_ctx(int rs_type, long long n, double s, uint64_t key,
                                                         uint32_t filter, uint32_t obs, double r_systematic) {
    ResampleCtx c;
    c.rs_type = rs_type;
    c.n = n;
    c.dn = (double)n;
    c.pow2 = (n & (n - 1)) == 0;
    c.inv_n = 1.0 / c.dn;
    c.s = s;
    c.inv_s = (s > 0.0) ? 1.0 / s : 0.0;
    c.key = key;
    c.filter = filter;
    c.obs = obs;
    c.r1_over_n = div_by_n(c, r_systematic);
    return c;
}

}  // namespace dpomp
