// da.cu -- data-augmented MCMC on the device (run_std_mcmc, src/hmm_mcmc.jl): the complete-data log-likelihood of a stored
// trajectory (compute_full_log_like! :78) and the Gibbs step of gibbs_mh_alg! (:138) with the insert / delete / move proposals
// of src/hmm_std.jl, over the trajectory store of the MBP layer (mbp_walk.cuh).
//
// One thread per chain.  A proposal is evaluated by walking the current event list with the edit applied virtually (the
// deleted index is skipped, the inserted event is merged at its time); nothing is written unless the proposal is accepted,
// and an accepted edit shifts the affected range of that chain's events by one slot.  The host widens the stride to the
// longest trajectory + traj_props before the launch, so no edit can run out of room.  f64 arithmetic with the reference's
// expressions, never contracted, so the walks and the edits are draw-for-draw comparable with oracle/dpomp_oracle_da.c.
#include <math.h>
#include <string.h>

#include <new>
#include <string>
#include <vector>

#include "mbp_walk.cuh"

namespace dpomp {

// Random streams of dpomp_da_step: proposal j (0-based) of the chain with global id g draws, with the call key K,
//   P = Philox4x32-10(ctr = (g, j, 0, kTagDa << 30 | 2), K)   the proposal
//   A = Philox4x32-10(ctr = (g, j, 0, kTagDa << 30 | 3), K)   the accept uniform u53(A.w0, A.w1) in [0, 1)
// kind = 1 + floor(P.w0 * mvp / 2^32); type = floor(P.w1 * E / 2^32) (insert) or index = floor(P.w1 * n / 2^32) (delete, move);
// time = t0 + (1 - u53(P.w2, P.w3)) * (T - t0) in (t0, T] (insert, move).  The tag is the outer layer's; its blocks are 0 and 1.
constexpr uint32_t kTagDa = 3u;
constexpr uint32_t kDaBlockProposal = 2u, kDaBlockAccept = 3u;

__device__ __forceinline__ int da_uniform_int(uint32_t w, int n) { return (int)(((uint64_t)w * (uint64_t)n) >> 32); }

// compute_full_log_like! of the event list (et, ey)[0, n) with index `del` skipped (-1: none) and the event (tins, eins)
// merged after the events at times <= tins (eins < 0: none).  Returns the full log-likelihood; llo = its observation part,
// x = the final state, q = position of the inserted event in the edited list.  -Inf (both parts): a zero rate for an event,
// a negative compartment, an event at or before t0, or an event after the last observation.
template <int MODEL>
__device__ __forceinline__ double da_walk(const MbpModel& m, const CountObs& co, const double (&th)[MbpRates<MODEL>::PMAX], double t0,
                                          const double* et, const unsigned char* ey, int n, int del, double tins, int eins,
                                          const double* obs_time, const double* obs_ysum, const int* obs_haslik, int n_obs,
                                          int (&x)[MbpRates<MODEL>::CMAX], double& llo, int& q) {
    using R = MbpRates<MODEL>;
    const int nc = mbp_nc<R>(m), ne = mbp_ne<R>(m);
#pragma unroll
    for (int c = 0; c < R::CMAX; ++c) x[c] = (c < nc) ? m.ic[c] : 0;
    double t = t0, ll = 0.0, lam[R::EMAX];
    bool ins = eins >= 0;
    int k = 0;
    llo = 0.0;
    q = 0;
    for (int oi = 0; oi < n_obs; ++oi) {
        const double t_obs = obs_time[oi];
        for (;;) {
            if (k == del) ++k;
            const double tk = k < n ? et[k] : INFINITY;
            const bool take_ins = ins && !(tk <= tins);
            if (!take_ins && k >= n) break;
            const double te = take_ins ? tins : tk;
            if (te > t_obs) break;
            const int e = take_ins ? eins : ey[k] - 1;
            if (!(te > t0)) { llo = -INFINITY; return -INFINITY; }
            R::rates(m, th, x, lam);
            const double le = R::pick(lam, e);
            mbp_cumsum<R>(m, lam);
            const double tot = R::pick(lam, ne - 1);
            if (!(le > 0.0)) { llo = -INFINITY; return -INFINITY; }
            ll = __dadd_rn(ll, __dsub_rn(log(le), __dmul_rn(tot, __dsub_rn(te, t))));
            R::apply(m, e, x);
            bool neg = false;
#pragma unroll
            for (int c = 0; c < R::CMAX; ++c) neg = neg || (c < nc && x[c] < 0);
            if (neg) { llo = -INFINITY; return -INFINITY; }
            t = te;
            if (take_ins) {
                ins = false;
                q = k - ((del >= 0 && del < k) ? 1 : 0);
            } else {
                ++k;
            }
        }
        R::rates(m, th, x, lam);
        mbp_cumsum<R>(m, lam);
        ll = __dsub_rn(ll, __dmul_rn(R::pick(lam, ne - 1), __dsub_rn(t_obs, t)));
        t = t_obs;
        if (obs_haslik[oi]) {
            const double g = mbp_obs_ll<MODEL>(m, co, th, oi, obs_ysum[oi], x);
            ll = __dadd_rn(ll, g);
            llo = __dadd_rn(llo, g);
        }
    }
    if (k == del) ++k;
    if (ins || k < n) { llo = -INFINITY; return -INFINITY; }
    return ll;
}

// kind == nullptr (dpomp_da_loglike): every chain evaluates its trajectory under theta_f.  Otherwise per chain: 0 evaluates under
// theta_f, 1 runs traj_props proposals under theta_cur and commits the accepted ones, 2 does nothing.
template <int MODEL>
__global__ void __launch_bounds__(128) da_step_kernel(const __grid_constant__ MbpModel m, MbpStore st, const double* theta_cur,
                                                       const double* theta_f, const unsigned char* kind, int n, int cap, int cap_max,
                                                       int traj_props, int mvp, const double* obs_time, const double* obs_ysum,
                                                       const int* obs_haslik, int n_obs, uint64_t key, uint32_t id0, double* out_ll,
                                                       int* out_acc, const __grid_constant__ CountObs co) {
    using R = MbpRates<MODEL>;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const int kd = kind ? kind[p] : 0;
    if (out_acc) out_acc[3 * p] = out_acc[3 * p + 1] = out_acc[3 * p + 2] = 0;
    if (kd == 2) {
        out_ll[2 * (size_t)p] = out_ll[2 * (size_t)p + 1] = -INFINITY;
        return;
    }
    double* et = st.ev_time + (size_t)p * cap;
    unsigned char* ey = st.ev_type + (size_t)p * cap;
    int len = st.len[p];
    const double* thp = (kd == 0 ? theta_f : theta_cur) + (size_t)p * m.n_params;
    double th[R::PMAX];
    R::load_params(m, thp, th);
    const double t0 = m.t0_index > 0 ? thp[m.t0_index - 1] : 0.0;
    int x[R::CMAX], q;
    double llo;
    double ll = da_walk<MODEL>(m, co, th, t0, et, ey, len, -1, 0.0, -1, obs_time, obs_ysum, obs_haslik, n_obs, x, llo, q);
    if (kd == 1) {
        const int ne = mbp_ne<R>(m), nc = mbp_nc<R>(m);
        const double span = __dsub_rn(obs_time[n_obs - 1], t0);
        const uint32_t gid = id0 + (uint32_t)p;
        int acc[3] = {0, 0, 0};
        for (int j = 0; j < traj_props; ++j) {
            const Philox4 w = stream_draw(key, gid, (uint32_t)j, 0u, kTagDa, kDaBlockProposal);
            const int mk = 1 + da_uniform_int(w.w0, mvp);
            const double tnew = __dadd_rn(t0, __dmul_rn(__dsub_rn(1.0, u53(w.w2, w.w3)), span));
            int del = -1, eins = -1;
            double r;
            if (mk == 1) {  // insert
                if (len >= cap_max) continue;
                eins = da_uniform_int(w.w1, ne);
                r = __ddiv_rn(__dmul_rn((double)ne, span), (double)(len + 1));
            } else {        // delete, move
                if (len == 0) continue;
                del = da_uniform_int(w.w1, len);
                if (mk == 2) {
                    r = __ddiv_rn((double)len, __dmul_rn((double)ne, span));
                } else {
                    eins = ey[del] - 1;
                    r = 1.0;
                }
            }
            int xf[R::CMAX], qf;
            double llof;
            const double llf = da_walk<MODEL>(m, co, th, t0, et, ey, len, del, tnew, eins, obs_time, obs_ysum, obs_haslik, n_obs, xf,
                                              llof, qf);
            const Philox4 a = stream_draw(key, gid, (uint32_t)j, 0u, kTagDa, kDaBlockAccept);
            if (!(__dmul_rn(r, exp(__dsub_rn(llf, ll))) > u53(a.w0, a.w1))) continue;  // NaN compares false
            // apply the edit in place: one slot shift of the range between the removed and the inserted position
            if (del < 0) {
                for (int i = len - 1; i >= qf; --i) { et[i + 1] = et[i]; ey[i + 1] = ey[i]; }
                ++len;
            } else if (eins < 0) {
                for (int i = del; i < len - 1; ++i) { et[i] = et[i + 1]; ey[i] = ey[i + 1]; }
                --len;
            } else if (qf < del) {
                for (int i = del - 1; i >= qf; --i) { et[i + 1] = et[i]; ey[i + 1] = ey[i]; }
            } else {
                for (int i = del; i < qf; ++i) { et[i] = et[i + 1]; ey[i] = ey[i + 1]; }
            }
            if (eins >= 0) { et[qf] = tnew; ey[qf] = (unsigned char)(eins + 1); }
            ll = llf;
            llo = llof;
#pragma unroll
            for (int c = 0; c < R::CMAX; ++c) x[c] = xf[c];
            acc[mk < 3 ? mk - 1 : 2] += 1;
        }
#pragma unroll
        for (int c = 0; c < R::CMAX; ++c)
            if (c < nc) st.fc[(size_t)p * nc + c] = x[c];
        st.len[p] = len;
        st.ll[2 * (size_t)p] = ll;
        st.ll[2 * (size_t)p + 1] = llo;
        out_acc[3 * p] = acc[0]; out_acc[3 * p + 1] = acc[1]; out_acc[3 * p + 2] = acc[2];
    }
    out_ll[2 * (size_t)p] = ll;
    out_ll[2 * (size_t)p + 1] = llo;
}

__global__ void da_max_len_kernel(const int* len, int n, int* out) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n) atomicMax(out, len[p]);
}

}  // namespace dpomp

using namespace dpomp;

// one launch over chains 1..n; theta_cur / theta_f / kind already on the device (h->theta_i, h->theta_f, h->valid)
static int da_launch(dpomp_mbp* h, const unsigned char* kind_dev, int n, int traj_props, int mvp, double* out_ll_host,
                     int32_t* out_acc_host) {
    const dpomp_model_desc& d = h->model->h.desc;
    const uint64_t key = mbp_next_key(h);
    int* acc = kind_dev ? h->da_work : nullptr;
    const unsigned grid = (unsigned)((n + 127) / 128);
    with_walk_model(h->model_id, [&](auto model) {
        da_step_kernel<decltype(model)::value><<<grid, 128, 0, h->stream>>>(
            h->dm, h->store[h->cur], h->theta_i, h->theta_f, kind_dev, n, h->cap, h->cap_max, traj_props, mvp, h->obs_time, h->obs_ysum,
            h->obs_haslik, d.n_obs, key, (uint32_t)h->batch_offset, h->out, acc, h->cobs);
    });
    MCK(cudaGetLastError());
    MCK(cudaMemcpyAsync(out_ll_host, h->out, (size_t)n * 2 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (out_acc_host) MCK(cudaMemcpyAsync(out_acc_host, acc, (size_t)n * 3 * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    MCK(cudaStreamSynchronize(h->stream));
    return DPOMP_OK;
}

extern "C" {

int dpomp_da_loglike(dpomp_mbp* h, const double* theta, int32_t n, double* out_ll2) {
    if (!h || !theta || !out_ll2) return dpomp_set_error(DPOMP_ERR_ARG, "null argument");
    if (n < 1 || n > h->n) return dpomp_set_error(DPOMP_ERR_ARG, "n out of range");
    MCK(cudaSetDevice(h->device));
    MCK(cudaMemcpyAsync(h->theta_f, theta, (size_t)n * h->dm.n_params * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    return da_launch(h, nullptr, n, 0, 1, out_ll2, nullptr);
}

int dpomp_da_step(dpomp_mbp* h, const double* theta_cur, const double* theta_f, const uint8_t* kind, int32_t n, int32_t traj_props,
                  int32_t mvp, double* out_ll2, int32_t* out_acc) {
    if (!h || !theta_cur || !theta_f || !kind || !out_ll2 || !out_acc) return dpomp_set_error(DPOMP_ERR_ARG, "null argument");
    if (n < 1 || n > h->n) return dpomp_set_error(DPOMP_ERR_ARG, "n out of range");
    if (traj_props < 0 || traj_props > (1 << 20)) return dpomp_set_error(DPOMP_ERR_ARG, "traj_props must be in 0..2^20");
    if (mvp < 1) return dpomp_set_error(DPOMP_ERR_ARG, "mvp must be positive");
    for (int p = 0; p < n; ++p)
        if (kind[p] > 2) return dpomp_set_error(DPOMP_ERR_ARG, "kind must be 0 (theta), 1 (trajectory) or 2 (skip)");
    MCK(cudaSetDevice(h->device));
    if (!h->da_work) MCK(cudaMalloc((void**)&h->da_work, (3 * (size_t)h->n + 1) * sizeof(int)));
    // room for traj_props inserts on the longest trajectory (inserts beyond max_traj are rejected)
    int* d_max = h->da_work + 3 * (size_t)h->n;
    MCK(cudaMemsetAsync(d_max, 0, sizeof(int), h->stream));
    da_max_len_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(h->store[h->cur].len, n, d_max);
    MCK(cudaGetLastError());
    MCK(cudaMemcpyAsync(h->h_need_grow, d_max, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    MCK(cudaStreamSynchronize(h->stream));
    const long long need0 = (long long)*h->h_need_grow + traj_props;
    const int need = need0 < h->cap_max ? (int)need0 : h->cap_max;
    if (need > h->cap) {
        const int rc = mbp_grow(h, need > 2 * (long long)h->cap ? need : (h->cap > h->cap_max / 2 ? h->cap_max : 2 * h->cap));
        if (rc) return rc;
    }
    const size_t tb = (size_t)n * h->dm.n_params * sizeof(double);
    MCK(cudaMemcpyAsync(h->theta_i, theta_cur, tb, cudaMemcpyHostToDevice, h->stream));
    MCK(cudaMemcpyAsync(h->theta_f, theta_f, tb, cudaMemcpyHostToDevice, h->stream));
    MCK(cudaMemcpyAsync(h->valid, kind, (size_t)n, cudaMemcpyHostToDevice, h->stream));
    return da_launch(h, h->valid, n, traj_props, mvp, out_ll2, out_acc);
}

}  // extern "C"
