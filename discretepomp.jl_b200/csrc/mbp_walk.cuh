// mbp_walk.cuh -- what the trajectory walks of mbp.cu (MBP-IBIS, MBP-MCMC) and da.cu (data-augmented MCMC) share: the
// trajectory store, the rate policies MbpRates<MODEL>, the observation log-likelihood, and the host handle dpomp_mbp with
// the helpers that key its calls, widen its stride and pick the walk instantiation of its model.
#pragma once
#include <math.h>
#include <stdint.h>

#include <string>
#include <type_traits>

#include "dpomp_dev.cuh"
#include "dpomp_internal.cuh"
#include "dpomp_models.cuh"
#include "obs_count.cuh"

namespace dpomp {

constexpr uint32_t kTagMbp = 2u;

struct MbpModel {  // integer rate table + f64 observation constants, runtime C / E
    int n_comp, n_events, n_params, t0_index;
    int par[DPOMP_MAX_EVENTS];
    int f1[DPOMP_MAX_EVENTS][DPOMP_MAX_COMPARTMENTS], k1[DPOMP_MAX_EVENTS];
    int f2[DPOMP_MAX_EVENTS][DPOMP_MAX_COMPARTMENTS], k2[DPOMP_MAX_EVENTS];
    int dn[DPOMP_MAX_EVENTS][DPOMP_MAX_COMPARTMENTS], kd[DPOMP_MAX_EVENTS], has_den[DPOMP_MAX_EVENTS];
    int trans[DPOMP_MAX_EVENTS][DPOMP_MAX_COMPARTMENTS];
    int xmask[DPOMP_MAX_COMPARTMENTS], ic[DPOMP_MAX_COMPARTMENTS];
    double obs_tmp1, obs_tmp2;
};

struct MbpStore {
    double* ev_time;      // [n][cap]
    unsigned char* ev_type;  // [n][cap]
    int* len;             // [n]
    int* fc;              // [n][C]
    double* ll;           // [n][2]
};

struct MbpStream {
    uint32_t k, a, b, id, j;
};
__device__ __forceinline__ MbpStream mbp_stream_init(uint64_t key, uint32_t id, uint32_t obs, uint32_t which) {
    const Philox4 p = stream_draw(key, 0u, id, obs, kTagMbp, which);
    return MbpStream{p.w0, p.w1, p.w2, id, 0u};
}
__device__ __forceinline__ uint2 mbp_draw(MbpStream& s) {
    const uint2 w = philox2x32_10(s.id ^ s.a, s.j ^ s.b, s.k);
    s.j += 1;
    return w;
}

// ---- rate policies ----------------------------------------------------------------------------------------------------
// MbpRates<kModelGeneric>: the integer rate table with run-time C / E (any model the table compiler accepts); also the rate
// table of MbpRates<kModelCountObs>, whose walks differ only in mbp_obs_ll.
// MbpRates<ID>: a predefined model with compile-time structure -- loops unroll, states and rates stay in registers, and
// rate[e] = (theta[e] * x_a) * x_b is the same f64 expression the table evaluates (l1 = x_a, l2 = x_b or 1 exactly), so both
// give bit-identical walks; a walk is one dependent instruction chain, so its length is what the kernels' time is made of.
template <int MODEL>
struct MbpRates {
    using BM = Builtin<MODEL>;
    static constexpr int C = BM::C, E = BM::E, CMAX = BM::C, EMAX = BM::E, PMAX = BM::E;  // parameter e drives event e
    static __device__ __forceinline__ void load_params(const MbpModel&, const double* src, double (&th)[PMAX]) {
#pragma unroll
        for (int i = 0; i < PMAX; ++i) th[i] = src[i];
    }
    static __device__ __forceinline__ void rates(const MbpModel&, const double (&th)[PMAX], const int (&x)[CMAX], double (&out)[EMAX]) {
#pragma unroll
        for (int e = 0; e < E; ++e) {
            double r = __dmul_rn(th[e], (double)x[BM::A(e)]);
            r = __dmul_rn(r, BM::B(e) >= 0 ? (double)x[BM::B(e) >= 0 ? BM::B(e) : 0] : 1.0);
            out[e] = r;
        }
    }
    static __device__ __forceinline__ void apply(const MbpModel&, int e, int (&x)[CMAX]) {
#pragma unroll
        for (int i = 0; i < E; ++i)
#pragma unroll
            for (int c = 0; c < C; ++c) x[c] += (e == i) ? BM::T(i, c) : 0;
    }
    static __device__ __forceinline__ double pick(const double (&v)[EMAX], int e) {
        double r = v[0];
#pragma unroll
        for (int i = 1; i < E; ++i) r = (e == i) ? v[i] : r;
        return r;
    }
};
template <>
struct MbpRates<kModelGeneric> {
    static constexpr int C = 0, E = 0, CMAX = DPOMP_MAX_COMPARTMENTS, EMAX = DPOMP_MAX_EVENTS, PMAX = DPOMP_MAX_PARAMS;
    static __device__ __forceinline__ void load_params(const MbpModel& m, const double* src, double (&th)[PMAX]) {
        for (int i = 0; i < m.n_params; ++i) th[i] = src[i];
    }
    static __device__ __forceinline__ void rates(const MbpModel& m, const double (&th)[PMAX], const int (&x)[CMAX], double (&out)[EMAX]) {
        for (int e = 0; e < m.n_events; ++e) {
            long long l1 = m.k1[e], l2 = m.k2[e], dn = m.kd[e];
            for (int c = 0; c < m.n_comp; ++c) {
                l1 += (long long)m.f1[e][c] * x[c];
                l2 += (long long)m.f2[e][c] * x[c];
                dn += (long long)m.dn[e][c] * x[c];
            }
            const double p = m.par[e] >= 0 ? th[m.par[e]] : 1.0;
            double r = __dmul_rn(__dmul_rn(p, (double)l1), (double)l2);
            if (m.has_den[e]) r = (dn == 0) ? 0.0 : __ddiv_rn(r, (double)dn);
            out[e] = r;
        }
    }
    static __device__ __forceinline__ void apply(const MbpModel& m, int e, int (&x)[CMAX]) {
        for (int c = 0; c < m.n_comp; ++c) x[c] += m.trans[e][c];
    }
    static __device__ __forceinline__ double pick(const double (&v)[EMAX], int e) { return v[e]; }
};
template <>
struct MbpRates<kModelCountObs> : MbpRates<kModelGeneric> {};
template <class R> __device__ __forceinline__ int mbp_nc(const MbpModel& m) { if constexpr (R::C > 0) return R::C; else return m.n_comp; }
template <class R> __device__ __forceinline__ int mbp_ne(const MbpModel& m) { if constexpr (R::E > 0) return R::E; else return m.n_events; }

template <class R>
__device__ __forceinline__ void mbp_cumsum(const MbpModel& m, double (&v)[R::EMAX]) {
    const int n = mbp_ne<R>(m);
#pragma unroll
    for (int i = 1; i < n; ++i) v[i] = __dadd_rn(v[i - 1], v[i]);
}
// choose_event (src/hmm_cmn.jl:4-10): first i < E - 1 with cum[i] > etc, else the last event (0-based)
template <class R>
__device__ __forceinline__ int mbp_choose(const MbpModel& m, const double (&cum)[R::EMAX], double u) {
    const int n = mbp_ne<R>(m);
    const double etc = __dmul_rn(u, R::pick(cum, n - 1));
    int e = n - 1;
#pragma unroll
    for (int i = R::EMAX - 2; i >= 0; --i)
        if (i < n - 1 && cum[i] > etc) e = i;
    return e;
}
// log g of observation t: the Gaussian, or for kModelCountObs the model's count observation family (obs_count.cuh) with its
// theta-indexed parameters taken from th (the walk's theta)
template <int MODEL>
__device__ __forceinline__ double mbp_obs_ll(const MbpModel& m, const CountObs& co, const double* th, int t, double ysum,
                                             const int (&x)[MbpRates<MODEL>::CMAX]) {
    using R = MbpRates<MODEL>;
    long long xs = 0;
    if constexpr (MODEL == kModelCountObs) {
        for (int c = 0; c < m.n_comp; ++c) xs += (long long)m.xmask[c] * x[c];
        return count_obs_logpmf(count_obs_const(co, th, t, ysum), ysum, (double)xs);
    } else {
        const int nc = mbp_nc<R>(m);
#pragma unroll
        for (int c = 0; c < R::CMAX; ++c)
            if (c < nc) xs += (long long)m.xmask[c] * x[c];
        const double d = ysum - (double)xs;
        return m.obs_tmp1 - __ddiv_rn(__dmul_rn(d, d), m.obs_tmp2);
    }
}

}  // namespace dpomp

using dpomp::CountObs;
using dpomp::MbpModel;
using dpomp::MbpStore;
struct MbpOuter;  // replicated device state of the MBP-IBIS outer layer (mbp.cu)

struct dpomp_mbp {
    MbpOuter* outer = nullptr;
    const dpomp_model* model = nullptr;
    int device = 0, n = 0;
    int cap = 0;       // current stride of the stores (events reserved per trajectory); grows on demand up to cap_max
    int cap_max = 0;   // MAX_TRAJ (src/DiscretePOMP.jl:40): the reference's hard limit, beyond which log-likelihood = -Inf
    int call_id = 0;   // id of the current iterate / propose call (MbpGrow)
    int* done = nullptr;       // [n]
    int* need_grow = nullptr;  // [1] device
    int* h_need_grow = nullptr;  // pinned
    cudaStream_t stream = nullptr;
    MbpModel dm{};
    MbpStore store[3]{};   // [cur], [cur ^ 1] (resample workspace), [2] proposal
    int cur = 0;
    int mode = 0;          // 0 automatic, 1 one thread per trajectory, 2 one warp per trajectory
    int model_id = 0;      // kernel_model_id of the model: the walk instantiation its launches run
    uint64_t seed = 0, call_index = 0, forced_key = 0;
    bool key_forced = false;
    long long batch_offset = 0;
    double *theta_i = nullptr, *theta_f = nullptr, *out = nullptr, *obs_time = nullptr, *obs_ysum = nullptr;
    int* obs_haslik = nullptr;
    double *obs_lgy = nullptr, *obs_lgk = nullptr;  // count observation constants [T] (count families only)
    CountObs cobs{};                                // count observation family (read only by the kModelCountObs walks)
    unsigned char* valid = nullptr;
    int64_t* slots = nullptr;  // 2 * n
    int* da_work = nullptr;    // [3 n + 1] data-augmented MCMC (da.cu): accept counts per chain, longest trajectory
};

// Philox key of the handle's next call (the forced key of dpomp_mbp_set_stream_key, else one derived from the seed)
uint64_t mbp_next_key(dpomp_mbp* h);
// widen the stride of all three stores to new_cap (<= cap_max), keeping every trajectory
int mbp_grow(dpomp_mbp* h, int new_cap);

namespace dpomp {

// launch(std::integral_constant<int, MODEL>{}) with the walk instantiation MODEL of model_id (kernel_model_id): a predefined
// model, kModelCountObs or kModelGeneric
template <class Launch>
void with_walk_model(int model_id, Launch&& launch) {
    switch (model_id) {
#define X(ID) case ID: return launch(std::integral_constant<int, ID>{});
        DPOMP_BUILTIN_MODELS(X)
#undef X
        case kModelCountObs: return launch(std::integral_constant<int, kModelCountObs>{});
        default: return launch(std::integral_constant<int, kModelGeneric>{});
    }
}

}  // namespace dpomp

// return the CUDA error of expr from a C-ABI entry point
#define MCK(expr)                                                                                         \
    do {                                                                                                  \
        cudaError_t _e = (expr);                                                                          \
        if (_e != cudaSuccess) return dpomp_set_error(DPOMP_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
    } while (0)
