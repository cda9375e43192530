// pf_kernels.cu -- kernel 2 of the particle filter (scan + search + gather fused), the multinomial variant, the
// outer-layer filter gather / pack kernels and the bit-exactness hook for the resampling searches.
//
// Replaces rsp_systematic (src/hmm_pf_resample.jl:24-42), the intended rsp_stratified / rsp_multinomial (:46-63, :5-20,
// broken in the reference, specified by rs_stratified / rs_multinomial src/hmm_resample.jl:66-83, 4-20), the
// `old_p .= pop` copy of partial_log_likelihood! (src/hmm_particle_filter.jl:66) and the population gathers of
// run_pibis (src/hmm_ibis.jl:71-79, 105-108).
#include "dpomp_dev.cuh"
#include "dpomp_internal.cuh"
#include "pf_resample.cuh"

namespace dpomp {

int sim_f32(const ModelHost& m, int items, const SimLaunch& a, cudaStream_t stream, int mode);
int sim_f64(const ModelHost& m, int items, const SimLaunch& a, cudaStream_t stream, int mode);
// count observation families: generic-table kernels only (pf_sim_count_f32.cu / pf_sim_count_f64.cu)
int sim_count_f32(const ModelHost& m, int items, const SimLaunch& a, cudaStream_t stream, int mode);
int sim_count_f64(const ModelHost& m, int items, const SimLaunch& a, cudaStream_t stream, int mode);

static int sim_dispatch(const ModelHost& m, int sim_precision, int items, const SimLaunch& a, cudaStream_t stream, int mode) {
    if (m.obs_family != DPOMP_OBS_GAUSSIAN)
        return sim_precision == DPOMP_SIM_F64 ? sim_count_f64(m, items, a, stream, mode) : sim_count_f32(m, items, a, stream, mode);
    return sim_precision == DPOMP_SIM_F64 ? sim_f64(m, items, a, stream, mode) : sim_f32(m, items, a, stream, mode);
}

cudaError_t launch_sim_weight(const ModelHost& m, int sim_precision, int items, int fused, const SimLaunch& a, cudaStream_t stream) {
    const int mode = fused;  // 0 plain, 1 fused step, 3 persistent
    return (cudaError_t)sim_dispatch(m, sim_precision, items, a, stream, mode);
}
int sim_fused_capacity(const ModelHost& m, int sim_precision, int items) {
    SimLaunch dummy{};
    return sim_dispatch(m, sim_precision, items, dummy, nullptr, 2);
}

int sim_persist_capacity(const ModelHost& m, int sim_precision, int items) {
    SimLaunch dummy{};
    return sim_precision == DPOMP_SIM_F64 ? 0 : sim_dispatch(m, sim_precision, items, dummy, nullptr, 4);
}

CountObs count_obs_of(const ModelHost& m, const double* lgy_dev, const double* lgk_dev) {
    CountObs c{};
    c.family = m.obs_family;
    for (int i = 0; i < 2; ++i) {
        c.par_index[i] = m.obs_par_index[i];
        c.par_value[i] = m.obs_par_value[i];
    }
    c.lgy = lgy_dev;
    c.lgk = lgk_dev;
    return c;
}

// does the rate table equal one of the hand-specialised predefined models (pf_sim.cuh Builtin<>)?
namespace {
struct BuiltinSpec { int id, C, E; int A[3], B[3]; int T[3][4]; };
const BuiltinSpec kSpecs[] = {
    {1, 2, 1, {0}, {1}, {{-1, 1}}},
    {2, 3, 2, {0, 1}, {1, -1}, {{-1, 1, 0}, {0, -1, 1}}},
    {3, 2, 2, {0, 1}, {1, -1}, {{-1, 1}, {1, -1}}},
    {4, 3, 2, {0, 1}, {2, -1}, {{-1, 1, 0}, {0, -1, 1}}},
    {5, 4, 3, {0, 1, 2}, {2, -1, -1}, {{-1, 1, 0, 0}, {0, -1, 1, 0}, {0, 0, -1, 1}}},
    {6, 3, 3, {0, 1, 2}, {2, -1, -1}, {{-1, 1, 0}, {0, -1, 1}, {1, 0, -1}}},
    {7, 2, 3, {1, 0, 0}, {-1, 1, -1}, {{0, 1}, {1, -1}, {-1, 0}}},
};
}  // namespace
int builtin_model_id(const dpomp_model_desc& d) {
    for (const BuiltinSpec& s : kSpecs) {
        if (d.n_compartments != s.C || d.n_events != s.E) continue;
        bool ok = true;
        for (int e = 0; e < s.E && ok; ++e) {
            ok = d.rate_par[e] == e && d.rate_has_den[e] == 0 && d.rate_k1[e] == 0 && d.rate_k2[e] == (s.B[e] >= 0 ? 0 : 1);
            for (int c = 0; c < s.C && ok; ++c)
                ok = d.rate_f1[e][c] == (c == s.A[e] ? 1 : 0) && d.rate_f2[e][c] == (c == s.B[e] ? 1 : 0) && d.trans[e][c] == s.T[e][c];
        }
        if (ok) return s.id;
    }
    return 0;
}

int sim_kernel_supported(int n_comp, int n_events) {
    return n_comp >= 1 && n_comp <= 8 && n_events >= 1 && n_events <= 8;
}

// ------------------------------------------------------------------------------------------------------------
// Kernel 2: one CTA per (filter, ancestor tile), one block barrier in total.
//   cw_q = off_b + f_b * incl_q                 (incl_q: tile-local scan stored by kernel 1, deterministic tree)
//   e_q  = E(cw_q) = #{ i : u_i <= cw_q }       (counting form of `while u[i] > cw[j]`, src/hmm_pf_resample.jl:34-40)
//   offspring (lo_b, hi_b] belong to this tile; offspring i takes the first q with e_q >= i, i.e. ancestor q owns
//   (max_{q'<q} e_q', max_{q'<=q} e_q'].
// After the barrier that publishes (lo_b, hi_b) and the per-warp maxima, every warp works alone on the 32*ITEMS
// ancestors it owns: the offspring -> ancestor map of a window of 32*ITEMS offspring is built in the warp's slice of
// shared memory by a scatter of the range starts followed by an inclusive max-scan (no per-offspring search); state
// rows are then copied with coalesced 128-byte writes over i and near-sorted reads over q.
// ------------------------------------------------------------------------------------------------------------
#ifndef DPOMP_RS_MINB
#define DPOMP_RS_MINB (DPOMP_BLOCK_THREADS == 128 ? 7 : 4)
#endif
template <int ITEMS, int RS, bool PERM, int NC>
__global__ void __launch_bounds__(kBlockThreads, DPOMP_RS_MINB) pf_resample_kernel(const __grid_constant__ ResampleLaunch a) {
    constexpr int TILE = kBlockThreads * ITEMS;
    constexpr int CHUNK = 32 * ITEMS;
    constexpr int NW = kBlockThreads / 32;
    constexpr unsigned FULL = 0xffffffffu;
    __shared__ int am_s[NW][CHUNK];  // per warp: offspring window -> ancestor index within the warp's chunk
    extern __shared__ __align__(16) int st_dyn[];  // [n_comp][TILE] states of the tile's ancestors (gather source)
    __shared__ int warp_max_s[NW];
    __shared__ long long lohi_s[2];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tile = blockIdx.x % a.ntiles;
    const int b = blockIdx.x / a.ntiles;
    const long long base_n = (long long)tile * TILE;
    const uint32_t gfilter = a.filter_ids ? a.filter_ids[b] : a.filter0 + (uint32_t)b;

    DPOMP_STAMP(1, 0);
    pdl_wait();
    DPOMP_STAMP(1, 1);
    const int grp = tile / kGroupTiles;
    // stage the states of this warp's CHUNK ancestors (coalesced, independent of everything below): the gather then reads
    // shared memory instead of paying a second dependent trip to L2
    {
        const int32_t* src_w = a.pop_src + (size_t)b * a.n_comp * a.n_pad + base_n + warp * CHUNK + lane * ITEMS;
        for (int c = 0; c < a.n_comp; ++c) {
            if constexpr (ITEMS % 4 == 0) {  // 16-byte asynchronous copies global -> shared (no registers, waited for below)
#pragma unroll
                for (int k = 0; k < ITEMS; k += 4) {
                    const unsigned dst = (unsigned)__cvta_generic_to_shared(st_dyn + c * TILE + tid * ITEMS + k);
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src_w + (size_t)c * a.n_pad + k) : "memory");
                }
            } else {
#pragma unroll
                for (int k = 0; k < ITEMS; ++k) st_dyn[c * TILE + tid * ITEMS + k] = src_w[(size_t)c * a.n_pad + k];
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    }
    double incl[ITEMS];
    const double* wt = a.wtile + (size_t)b * a.n_pad + base_n + (size_t)tid * ITEMS;
    if constexpr (ITEMS % 2 == 0) {  // 128-bit loads
#pragma unroll
        for (int k = 0; k < ITEMS; k += 2) {
            const double2 v = *reinterpret_cast<const double2*>(wt + k);
            incl[k] = v.x;
            incl[k + 1] = v.y;
        }
    } else {
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) incl[k] = wt[k];
    }

    // Deferred level 2 of the combine (the simulate kernel stopped after the group level): warp 0 combines the <= 64 group
    // partials of the filter while the tile loads above are in flight -- M, F_g = exp(m_g - M), O_g, S with exactly the tree
    // of combine_level2 -- into shared memory (a prefetch of the partials at the top of the kernel made it 2 us SLOWER); the
    // tile-0 CTA of the filter also stores them for later consumers and adds the log-likelihood increment
    // log(cum_weight[end] / N) (src/hmm_particle_filter.jl:60) as M + log(S / N).
    __shared__ double l2f_s[kDeferGroups], l2off_s[kDeferGroups];
    __shared__ double l2s_s;
    if (a.defer_l2) {
        if (warp == 0) {
            const Level2 l2 = combine_level2<false>(a.grp_m + (size_t)b * a.ngroups, a.grp_s + (size_t)b * a.ngroups, a.ngroups, l2f_s, l2off_s);
            if (lane == 0) l2s_s = l2.big_s;
            if (tile == 0) {
                __syncwarp();
                for (int g = lane; g < a.ngroups; g += 32) {
                    a.grp_f_w[(size_t)b * a.ngroups + g] = l2f_s[g];
                    a.grp_off_w[(size_t)b * a.ngroups + g] = l2off_s[g];
                }
                if (lane == 0) {
                    a.filt_s_w[b] = l2.big_s;
                    a.filt_m_w[b] = l2.big_m;
                    if (a.has_lik) atomicAdd(&a.ll_acc[b], l2.big_m + log(l2.big_s / (double)a.n));
                }
            }
        }
        __syncthreads();
    }
    const double* l2_f = a.defer_l2 ? l2f_s : nullptr;
    const double* l2_off = a.defer_l2 ? l2off_s : nullptr;
    const double* l2_s = a.defer_l2 ? &l2s_s : nullptr;
    if (a.rs_type == DPOMP_RS_MULTINOMIAL) {  // materialise cw; the per-offspring search is a second kernel 
        const double g_off = l2_off ? l2_off[grp] : a.grp_off[(size_t)b * a.ngroups + grp], g_f = l2_f ? l2_f[grp] : a.grp_f[(size_t)b * a.ngroups + grp];
        const double t_off = a.tile_off[(size_t)b * a.ntiles + tile], t_f = a.tile_f[(size_t)b * a.ntiles + tile];
        double* cw = a.cw + (size_t)b * a.n_pad + base_n + (size_t)tid * ITEMS;
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) cw[k] = tile_cw(g_off, g_f, t_off, t_f, incl[k]);
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        return;
    }
    const RsArgs ra{a.tile_f, a.tile_off, a.grp_f, a.grp_off, a.filt_s, l2_f, l2_off, l2_s, a.pop_dst, a.anc, a.n, a.n_pad,
                    a.ntiles, a.ngroups, a.n_comp, a.t, a.rs_type, a.key, a.perm};
    DPOMP_STAMP(1, 2);
    resample_tile<ITEMS, int, false, RS, PERM, NC>(ra, b, tile, gfilter, incl, st_dyn, TILE, &am_s[0][0], warp_max_s, lohi_s);
    DPOMP_STAMP(1, 4);
}

// multinomial: offspring i draws chs = r_i * S; ancestor = first p2 < N with chs < cw[p2], else N (src/hmm_resample.jl:9-16)
__global__ void __launch_bounds__(kBlockThreads) pf_multinomial_gather_kernel(const __grid_constant__ ResampleLaunch a, int tile_size) {
    pdl_wait();
    const long long gi = (long long)blockIdx.x * kBlockThreads + threadIdx.x;
    const int b = (int)(gi / a.n_pad);
    const long long i = gi % a.n_pad;
    if (b >= a.n_filters || i >= a.n) return;
    const uint32_t gfilter = a.filter_ids ? a.filter_ids[b] : a.filter0 + (uint32_t)b;
    const double big_s = a.filt_s[b];
    const Philox4 p = stream_draw(a.key, (uint32_t)i, gfilter, (uint32_t)a.t, kTagResample, 1u);
    const double chs = __dmul_rn(u53(p.w0, p.w1), big_s);
    auto tile_end = [&](int t) -> double {  // offset of tile t + 1 (= end of tile t); the filter total after the last tile
        if (t + 1 >= a.ntiles) return big_s;
        const int g2 = (t + 1) / kGroupTiles;
        return tile_cw(a.grp_off[(size_t)b * a.ngroups + g2], a.grp_f[(size_t)b * a.ngroups + g2],
                       a.tile_off[(size_t)b * a.ntiles + t + 1], 1.0, 0.0);
    };
    int lt = 0, ht = a.ntiles;  // first tile with chs < end(tile)
    while (lt < ht) {
        const int mid = (lt + ht) >> 1;
        if (chs < tile_end(mid)) ht = mid; else lt = mid + 1;
    }
    long long res = a.n - 1;
    if (lt < a.ntiles) {
        const long long base = (long long)lt * tile_size;
        const long long rem = a.n - base;
        const int nvalid = rem < tile_size ? (int)rem : tile_size;
        const double* cw = a.cw + (size_t)b * a.n_pad + base;
        int lq = 0, hq = nvalid;
        while (lq < hq) {
            const int mid = (lq + hq) >> 1;
            if (chs < cw[mid]) hq = mid; else lq = mid + 1;
        }
        // cw of the tile's last particle and tile_end(lt) are rounded differently: a draw with cw_last <= chs < tile_end(lt)
        // belongs to the first particle of the following tile whose cw exceeds it (src/hmm_resample.jl:9-16), not to this tile
        res = base + lq;
        if (lq >= nvalid) {
            res = a.n - 1;
            for (long long q2 = base + nvalid; q2 < a.n; ++q2) {  // cw is non-decreasing: ends after a step or two
                if (chs < a.cw[(size_t)b * a.n_pad + q2]) { res = q2; break; }
            }
        }
    }
    const int32_t* src_b = a.pop_src + (size_t)b * a.n_comp * a.n_pad;
    int32_t* dst_b = a.pop_dst + (size_t)b * a.n_comp * a.n_pad;
    const long long row = perm_pos(a.perm, i);
    for (int c = 0; c < a.n_comp; ++c) dst_b[(size_t)c * a.n_pad + row] = src_b[(size_t)c * a.n_pad + res];
    if (a.anc) a.anc[(size_t)b * a.n_pad + row] = (int32_t)res;
}

// sum of the per-(filter, group) event counters of a call into the call's counter
__global__ void __launch_bounds__(256) sum_events_kernel(const unsigned long long* grp_ev, long long n, unsigned long long* out) {
    __shared__ unsigned long long red[256];
    unsigned long long v = 0;
    for (long long i = threadIdx.x; i < n; i += 256) v += grp_ev[i];
    red[threadIdx.x] = v;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = red[0];
}
cudaError_t launch_sum_events(const unsigned long long* grp_ev_dev, long long n, unsigned long long* out_dev, cudaStream_t stream) {
    sum_events_kernel<<<1, 256, 0, stream>>>(grp_ev_dev, n, out_dev);
    return cudaGetLastError();
}

cudaError_t launch_resample(int items, const ResampleLaunch& a, cudaStream_t stream) {
    const unsigned grid = (unsigned)(a.n_filters * a.ntiles);
    const size_t smem = (size_t)kBlockThreads * items * a.n_comp * sizeof(int);  // staged ancestor states
    // one instantiation per resampler: the systematic one carries no stratified (Philox) code (multinomial only uses the
    // cw materialisation at the top of the kernel)
    const bool strat = a.rs_type == DPOMP_RS_STRATIFIED, perm = a.perm.ncf > 0;
    cudaError_t err;
    // the identity placement (the reference's row order) is instantiated per compartment count of the predefined models
#define DPOMP_RS_LAUNCH(IT, RS, PM, NC) launch_pdl(pf_resample_kernel<IT, RS, PM, NC>, grid, kBlockThreads, smem, stream, a)
#define DPOMP_RS_NC(IT, RS)                                                                      \
    (a.n_comp == 2 ? DPOMP_RS_LAUNCH(IT, RS, false, 2) : a.n_comp == 3 ? DPOMP_RS_LAUNCH(IT, RS, false, 3) \
     : a.n_comp == 4 ? DPOMP_RS_LAUNCH(IT, RS, false, 4) : DPOMP_RS_LAUNCH(IT, RS, false, 0))
#define DPOMP_RS_PICK(IT)                                                                                  \
    (strat ? (perm ? DPOMP_RS_LAUNCH(IT, DPOMP_RS_STRATIFIED, true, 0) : DPOMP_RS_NC(IT, DPOMP_RS_STRATIFIED))   \
           : (perm ? DPOMP_RS_LAUNCH(IT, DPOMP_RS_SYSTEMATIC, true, 0) : DPOMP_RS_NC(IT, DPOMP_RS_SYSTEMATIC)))
    err = items == kItemsSmall ? DPOMP_RS_PICK(kItemsSmall) : DPOMP_RS_PICK(kItemsLarge);
#undef DPOMP_RS_PICK
#undef DPOMP_RS_NC
#undef DPOMP_RS_LAUNCH
    if (err != cudaSuccess) return err;
    if (a.rs_type == DPOMP_RS_MULTINOMIAL) {
        const long long total = (long long)a.n_filters * a.n_pad;
        pf_multinomial_gather_kernel<<<(unsigned)((total + kBlockThreads - 1) / kBlockThreads), kBlockThreads, 0, stream>>>(
            a, kBlockThreads * items);
        err = cudaGetLastError();
    }
    return err;
}

// ------------------------------------------------------------------------------------------------------------
// Whole-filter copies for the outer layer: dst filter dst_slots[k] <- src filter src_slots[k] (1-based slots).
// 128-bit vectorised; filter_stride_words = C * n_pad is a multiple of 256.
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlockThreads) gather_filters_kernel(int32_t* dst, const int32_t* src, const int64_t* dst_slots,
                                                                        const int64_t* src_slots, long long stride_words) {
    const int k = blockIdx.y;
    const long long d = dst_slots ? dst_slots[k] - 1 : k;
    const long long s = src_slots ? src_slots[k] - 1 : k;
    const int4* sp = reinterpret_cast<const int4*>(src + s * stride_words);
    int4* dp = reinterpret_cast<int4*>(dst + d * stride_words);
    const long long nvec = stride_words / 4;
    for (long long v = (long long)blockIdx.x * kBlockThreads + threadIdx.x; v < nvec; v += (long long)gridDim.x * kBlockThreads)
        dp[v] = sp[v];
}

cudaError_t launch_gather_filters(int32_t* dst, const int32_t* src, const int64_t* dst_slots_dev, const int64_t* src_slots_dev,
                                  int n, long long filter_stride_words, cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    const long long nvec = filter_stride_words / 4;
    long long bx = (nvec + kBlockThreads - 1) / kBlockThreads;
    if (bx > 64) bx = 64;
    if (bx < 1) bx = 1;
    for (int k0 = 0; k0 < n; k0 += 65535) {  // gridDim.y limit
        const int cnt = (n - k0) < 65535 ? (n - k0) : 65535;
        gather_filters_kernel<<<dim3((unsigned)bx, (unsigned)cnt), kBlockThreads, 0, stream>>>(
            dst, src, dst_slots_dev ? dst_slots_dev + k0 : nullptr, src_slots_dev ? src_slots_dev + k0 : nullptr,
            filter_stride_words);
        if (!dst_slots_dev || !src_slots_dev) {
            // identity side: offset the dense buffer by k0 filters
            if (!dst_slots_dev) dst += (long long)cnt * filter_stride_words;
            if (!src_slots_dev) src += (long long)cnt * filter_stride_words;
        }
    }
    return cudaGetLastError();
}

cudaError_t launch_pack_filters(int32_t* packed, const int32_t* pop, const int64_t* slots_dev, int n,
                                long long filter_stride_words, int unpack, cudaStream_t stream) {
    if (unpack) return launch_gather_filters(const_cast<int32_t*>(pop), packed, slots_dev, nullptr, n, filter_stride_words, stream);
    return launch_gather_filters(packed, pop, nullptr, slots_dev, n, filter_stride_words, stream);
}

// ------------------------------------------------------------------------------------------------------------
// Bit-exactness hook: literal searches on a given cumulative-weight array (1-based output).
//   systematic / stratified: first j with NOT (u_i > cw_j)   (walk of src/hmm_pf_resample.jl:34-40 as a lower bound;
//                            u_i is non-decreasing so the walk and the bound agree)
//   multinomial:             first p2 < n with chs < cw[p2], else n  (src/hmm_resample.jl:9-16)
// ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlockThreads) search_hook_kernel(int rs_type, const double* cw, long long n, const double* u,
                                                                     long long n_out, int64_t* out) {
    const long long i = (long long)blockIdx.x * kBlockThreads + threadIdx.x;
    if (i >= n_out) return;
    const double s = cw[n - 1];
    const double dn = (double)n;
    long long lo = 0, hi = n - 1;  // answer in [0, n-1]
    if (rs_type == DPOMP_RS_MULTINOMIAL) {
        const double chs = __dmul_rn(u[i], s);
        while (lo < hi) {
            const long long mid = (lo + hi) >> 1;
            if (chs < cw[mid]) hi = mid; else lo = mid + 1;
        }
    } else {
        const double r = (rs_type == DPOMP_RS_STRATIFIED) ? u[i] : u[0];
        const double ui = __dmul_rn(__dadd_rn(__ddiv_rn(r, dn), __ddiv_rn((double)i, dn)), s);
        while (lo < hi) {
            const long long mid = (lo + hi) >> 1;
            if (!(ui > cw[mid])) hi = mid; else lo = mid + 1;
        }
    }
    out[i] = lo + 1;
}

cudaError_t launch_search_hook(int rs_type, const double* cw_dev, long long n, const double* u_dev, long long n_out,
                               int64_t* out_dev, cudaStream_t stream) {
    search_hook_kernel<<<(unsigned)((n_out + kBlockThreads - 1) / kBlockThreads), kBlockThreads, 0, stream>>>(
        rs_type, cw_dev, n, u_dev, n_out, out_dev);
    return cudaGetLastError();
}

__global__ void debug_uniforms_kernel(const uint32_t* w, int n, float* wait, float* evt) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        wait[i] = u32_wait_f32(w[i]);
        evt[i] = u32_event_f32(w[i]);
    }
}

}  // namespace dpomp

// diagnostics: the two f32 uniform conversions of the event loop evaluated on the device for the given Philox words
extern "C" int dpomp_debug_uniforms_f32(const uint32_t* words, int32_t n, float* out_wait, float* out_event) {
    if (!words || !out_wait || !out_event || n < 1) return DPOMP_ERR_ARG;
    uint32_t* w = nullptr;
    float* o = nullptr;
    if (cudaMalloc((void**)&w, (size_t)n * 4) != cudaSuccess || cudaMalloc((void**)&o, (size_t)n * 8) != cudaSuccess) {
        cudaFree(w);
        return DPOMP_ERR_CUDA;
    }
    cudaMemcpy(w, words, (size_t)n * 4, cudaMemcpyHostToDevice);
    dpomp::debug_uniforms_kernel<<<(n + 127) / 128, 128>>>(w, n, o, o + n);
    cudaError_t e = cudaMemcpy(out_wait, o, (size_t)n * 4, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(out_event, o + n, (size_t)n * 4, cudaMemcpyDeviceToHost);
    cudaFree(w);
    cudaFree(o);
    return e == cudaSuccess ? DPOMP_OK : DPOMP_ERR_CUDA;
}

#ifdef DPOMP_BOUNDS_CHECK
// bounds-checked debug build only: proves that the checker is live (a deliberately out-of-range index must trap)
namespace dpomp {
__global__ void bounds_selftest_kernel(int i, int n) { DPOMP_CHECK_IDX(i, n); }
}  // namespace dpomp
extern "C" int dpomp_debug_bounds_selftest(int i, int n) {
    dpomp::bounds_selftest_kernel<<<1, 1>>>(i, n);
    return cudaDeviceSynchronize() == cudaSuccess ? 0 : -2;
}
#endif

#ifdef DPOMP_PHASE_TIMERS
extern "C" int dpomp_debug_phases_rs(unsigned long long* out /* [2][4096][8] */) {
    return (int)cudaMemcpyFromSymbol(out, dpomp::g_dpomp_phase, sizeof(unsigned long long) * 2 * 4096 * 8);
}
#endif
