// pf_history.cu -- the hidden-state history of the particle filter (dpomp_pf_set_history): the per-observation record
// kernel that runs between the simulate and the resample kernel, the moments combine and the path sampler.
//
// partial_log_likelihood! (src/hmm_particle_filter.jl:39-76) holds weighted particles at every observation and drops them
// at the next one.  The record kernel keeps, for observation t, what the filter already computed: the simulated states
// (before resampling) and tile partials of their weighted moments; the resample kernel writes its ancestors into slice t of
// the ancestor history.  Nothing here is read by the filter itself.
#include "dpomp_dev.cuh"
#include "dpomp_internal.cuh"

namespace dpomp {

// Deterministic sum of one value per thread over the CTA, in a fixed association: xor butterfly inside each warp, then the
// warp totals in warp order (by the caller, after a barrier).  Lane 0 of every warp stores its warp's total at red[warp].
__device__ __forceinline__ void warp_total_to(double v, double* red) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, d));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
}

// One CTA per (filter, tile), on the filter's tile geometry.  Reads the tile's int32 states and f64 log weights once
// (about 4 C + 8 bytes per particle), writes the states into the state history (4 C bytes per particle) and one row of
// tile partials:  m = max logw, sum w, sum w^2, sum w d_c, sum w d_c^2 with w = exp(logw - m), d_c = x_c - x0_c, and x0_c.
// Without a likelihood at t every particle weighs 1.  Sums are run-to-run identical whatever the scheduling.
template <int ITEMS>
__global__ void __launch_bounds__(kBlockThreads) pf_history_kernel(const __grid_constant__ HistoryLaunch a) {
    constexpr int TILE = kBlockThreads * ITEMS;
    constexpr int NW = kBlockThreads / 32;
    constexpr int kMaxSlots = 3 + 2 * DPOMP_MAX_COMPARTMENTS;
    __shared__ double red_s[kMaxSlots][NW];
    __shared__ double scratch_s[NW];
    const int tid = threadIdx.x, warp = tid >> 5;
    const int tile = blockIdx.x % a.ntiles;
    const int b = blockIdx.x / a.ntiles;
    const long long base_n = (long long)tile * TILE;
    const int32_t* pop_b = a.pop + (size_t)b * a.n_comp * a.n_pad;

    pdl_wait();  // the states and log weights are written by the simulate kernel of this observation
    if (a.states) {  // 128-bit coalesced copy of the tile, padding included (n_pad is a multiple of the tile)
        int32_t* dst_b = a.states + (size_t)b * a.n_comp * a.n_pad;
        for (int c = 0; c < a.n_comp; ++c) {
            const int4* src = reinterpret_cast<const int4*>(pop_b + (size_t)c * a.n_pad + base_n);
            int4* dst = reinterpret_cast<int4*>(dst_b + (size_t)c * a.n_pad + base_n);
            for (int v = tid; v < TILE / 4; v += kBlockThreads) {
                DPOMP_CHECK_IDX(base_n + 4 * v + 3, a.n_pad);
                dst[v] = src[v];
            }
        }
    }
    if (!a.part) return;

    // blocked ownership: thread tid holds particles base_n + tid * ITEMS + k
    const long long p0 = base_n + (long long)tid * ITEMS;
    double lw[ITEMS], mloc = -INFINITY;
    const double* lw_b = a.logw + (size_t)b * a.n_pad + p0;
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        DPOMP_CHECK_IDX(p0 + k, a.n_pad);
        const bool valid = p0 + k < a.n;
        lw[k] = !valid ? -INFINITY : (a.has_lik ? lw_b[k] : 0.0);
        mloc = fmax(mloc, lw[k]);
    }
    const double m = block_max(mloc, scratch_s);
    double w[ITEMS], s = 0.0, s2 = 0.0;
#pragma unroll
    for (int k = 0; k < ITEMS; ++k) {
        w[k] = lw[k] == -INFINITY ? 0.0 : exp(lw[k] - m);
        s = __dadd_rn(s, w[k]);
        s2 = __dadd_rn(s2, __dmul_rn(w[k], w[k]));
    }
    warp_total_to(s, red_s[1]);
    warp_total_to(s2, red_s[2]);
    for (int c = 0; c < a.n_comp; ++c) {
        const double x0 = (double)pop_b[(size_t)c * a.n_pad];
        const int32_t* x_c = pop_b + (size_t)c * a.n_pad + p0;
        double sx = 0.0, sxx = 0.0;
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            const double d = (double)x_c[k] - x0;
            const double wd = __dmul_rn(w[k], d);
            sx = __dadd_rn(sx, wd);
            sxx = __dadd_rn(sxx, __dmul_rn(wd, d));
        }
        warp_total_to(sx, red_s[3 + c]);
        warp_total_to(sxx, red_s[3 + a.n_comp + c]);
    }
    __syncthreads();
    const int K = history_partials_stride(a.n_comp);
    double* out = a.part + ((size_t)b * a.ntiles + tile) * K;
    if (tid == 0) out[0] = m;
    if (tid >= 1 && tid < 3 + 2 * a.n_comp) {
        DPOMP_CHECK_IDX(tid, kMaxSlots);
        double v = 0.0;
#pragma unroll
        for (int i = 0; i < NW; ++i) v = __dadd_rn(v, red_s[tid][i]);
        out[tid] = v;
    }
    if (tid < a.n_comp) out[3 + 2 * a.n_comp + tid] = (double)pop_b[(size_t)tid * a.n_pad];
}

cudaError_t launch_history(int items, const HistoryLaunch& a, cudaStream_t stream) {
    const unsigned grid = (unsigned)(a.n_filters * a.ntiles);
    // programmatic dependent launch like the rest of the chain: the resample kernel behind it waits for this kernel, which
    // itself waits for the simulate kernel, so the resample kernel still sees every write of the simulate kernel
    return items == kItemsSmall ? launch_pdl(pf_history_kernel<kItemsSmall>, grid, kBlockThreads, 0, stream, a)
                                : launch_pdl(pf_history_kernel<kItemsLarge>, grid, kBlockThreads, 0, stream, a);
}

// One warp per (filter, observation): the tile partials combined with a fixed tree (lane-strided over the tiles, xor
// butterfly over the lanes) into mean_c, var_c and ESS = (sum w)^2 / sum w^2.
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, d));
    return v;
}
__global__ void __launch_bounds__(128) history_moments_kernel(const double* part, int t_last, int n_batch, int nb, int ntiles,
                                                              int n_comp, double* out) {
    const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (gw >= (long long)nb * t_last) return;  // warp-uniform
    const int b = (int)(gw / t_last), t = (int)(gw % t_last);
    const int K = history_partials_stride(n_comp);
    const double* P = part + ((size_t)t * n_batch + b) * ntiles * K;
    double big_m = -INFINITY;
    for (int i = lane; i < ntiles; i += 32) big_m = fmax(big_m, P[(size_t)i * K]);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) big_m = fmax(big_m, __shfl_xor_sync(0xffffffffu, big_m, d));
    auto scale = [&](int i) -> double {
        const double mi = P[(size_t)i * K];
        return mi == -INFINITY ? 0.0 : exp(mi - big_m);
    };
    double s = 0.0, s2 = 0.0;
    for (int i = lane; i < ntiles; i += 32) {
        DPOMP_CHECK_IDX(((size_t)t * n_batch + b) * ntiles + i, (size_t)t_last * n_batch * ntiles);
        const double f = scale(i);
        s = __dadd_rn(s, __dmul_rn(f, P[(size_t)i * K + 1]));
        s2 = __dadd_rn(s2, __dmul_rn(__dmul_rn(f, f), P[(size_t)i * K + 2]));
    }
    s = warp_sum(s);
    s2 = warp_sum(s2);
    double* o = out + ((size_t)b * t_last + t) * (2 * n_comp + 1);
    for (int c = 0; c < n_comp; ++c) {
        double sx = 0.0, sxx = 0.0;
        for (int i = lane; i < ntiles; i += 32) {
            const double f = scale(i);
            sx = __dadd_rn(sx, __dmul_rn(f, P[(size_t)i * K + 3 + c]));
            sxx = __dadd_rn(sxx, __dmul_rn(f, P[(size_t)i * K + 3 + n_comp + c]));
        }
        sx = warp_sum(sx);
        sxx = warp_sum(sxx);
        if (lane == 0) {
            const double md = sx / s;
            o[c] = P[3 + 2 * n_comp + c] + md;
            o[n_comp + c] = fmax(sxx / s - md * md, 0.0);
        }
    }
    if (lane == 0) o[2 * n_comp] = s * s / s2;
}

cudaError_t launch_history_moments(const double* part, int t_last, int n_batch, int nb, int ntiles, int n_comp, double* out,
                                   cudaStream_t stream) {
    const long long threads = (long long)nb * t_last * 32;
    history_moments_kernel<<<(unsigned)((threads + 127) / 128), 128, 0, stream>>>(part, t_last, n_batch, nb, ntiles, n_comp, out);
    return cudaGetLastError();
}

// One thread per (filter, path).  The lineage end is the multinomial draw of pf_multinomial_gather_kernel (pf_kernels.cu) on
// the same cumulative weights cw_q = tile_cw(O_g, F_g, o_b, f_b, incl_q) -- evaluated where they are searched, never
// materialised -- then the genealogy is traced back: t_last dependent ancestor loads and C state loads per observation.
__global__ void __launch_bounds__(128) history_paths_kernel(const __grid_constant__ PathLaunch a) {
    const long long gi = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (gi >= (long long)a.nb * a.n_paths) return;
    const int b = (int)(gi / a.n_paths), path = (int)(gi % a.n_paths);
    const uint32_t gfilter = a.filter_ids ? a.filter_ids[b] : a.filter0 + (uint32_t)b;
    const Philox4 p = stream_draw(a.key, (uint32_t)path, gfilter, (uint32_t)(a.t_last - 1), kTagResample, 2u);
    const double u = u53(p.w0, p.w1);
    long long k;
    if (!a.haslik[a.t_last - 1]) {
        k = min((long long)(u * (double)a.n), a.n - 1);
    } else {
        const double big_s = a.filt_s[b];
        const double chs = __dmul_rn(u, big_s);
        auto cw_at = [&](long long q) -> double {
            const int t = (int)(q / a.tile), g = t / kGroupTiles;
            DPOMP_CHECK_IDX(q, a.n_pad);
            DPOMP_CHECK_IDX(g, a.ngroups);
            return tile_cw(a.grp_off[(size_t)b * a.ngroups + g], a.grp_f[(size_t)b * a.ngroups + g],
                           a.tile_off[(size_t)b * a.ntiles + t], a.tile_f[(size_t)b * a.ntiles + t], a.wtile[(size_t)b * a.n_pad + q]);
        };
        auto tile_end = [&](int t) -> double {  // offset of tile t + 1; the filter total after the last tile
            if (t + 1 >= a.ntiles) return big_s;
            const int g2 = (t + 1) / kGroupTiles;
            DPOMP_CHECK_IDX(g2, a.ngroups);
            return tile_cw(a.grp_off[(size_t)b * a.ngroups + g2], a.grp_f[(size_t)b * a.ngroups + g2],
                           a.tile_off[(size_t)b * a.ntiles + t + 1], 1.0, 0.0);
        };
        int lt = 0, ht = a.ntiles;
        while (lt < ht) {
            const int mid = (lt + ht) >> 1;
            if (chs < tile_end(mid)) ht = mid; else lt = mid + 1;
        }
        k = a.n - 1;
        if (lt < a.ntiles) {
            const long long base = (long long)lt * a.tile;
            const long long rem = a.n - base;
            const int nvalid = rem < a.tile ? (int)rem : a.tile;
            int lq = 0, hq = nvalid;
            while (lq < hq) {
                const int mid = (lq + hq) >> 1;
                if (chs < cw_at(base + mid)) hq = mid; else lq = mid + 1;
            }
            k = base + lq;
            if (lq >= nvalid) {  // rounding seam between the tile's last cw and tile_end (see pf_multinomial_gather_kernel)
                k = a.n - 1;
                for (long long q2 = base + nvalid; q2 < a.n; ++q2)
                    if (chs < cw_at(q2)) { k = q2; break; }
            }
        }
    }
    const size_t st_slice = (size_t)a.n_batch * a.n_comp * a.n_pad, anc_slice = (size_t)a.n_batch * a.n_pad;
    int64_t* o = a.out + ((size_t)b * a.n_paths + path) * a.t_last * a.n_comp;
    for (int t = a.t_last; t >= 1; --t) {
        DPOMP_CHECK_IDX(k, a.n);
        const int32_t* st = a.states + (size_t)(t - 1) * st_slice + (size_t)b * a.n_comp * a.n_pad;
        for (int c = 0; c < a.n_comp; ++c) o[(size_t)(t - 1) * a.n_comp + c] = st[(size_t)c * a.n_pad + k];
        // observation t - 1 resampled iff it has a likelihood (it is not the last observation)
        if (t > 1 && a.haslik[t - 2]) k = a.anc[(size_t)(t - 2) * anc_slice + (size_t)b * a.n_pad + k];
    }
}

cudaError_t launch_paths(const PathLaunch& a, cudaStream_t stream) {
    const long long threads = (long long)a.nb * a.n_paths;
    history_paths_kernel<<<(unsigned)((threads + 127) / 128), 128, 0, stream>>>(a);
    return cudaGetLastError();
}

}  // namespace dpomp
