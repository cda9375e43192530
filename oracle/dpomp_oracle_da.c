/*
 * dpomp_oracle_da.c -- CPU restatement of data-augmented MCMC (TEST INFRASTRUCTURE ONLY, see dpomp_oracle.c):
 *   compute_full_log_like!   src/hmm_mcmc.jl:78    -> orc_da_loglike
 *   gibbs_mh_alg!            src/hmm_mcmc.jl:138   -> orc_da_props (the trajectory branch; the theta branch is the host's)
 *   add_event! / proposals   src/hmm_std.jl:4, :18
 * The law is the one stated in include/dpomp.h (dpomp_da_loglike / dpomp_da_step); the draws are those of
 * discretepomp.jl_b200/csrc/da.cu: proposal j of chain `id` takes P = Philox4x32-10((id, j, 0, 3<<30 | 2), key) and the accept
 * uniform from A = Philox4x32-10((id, j, 0, 3<<30 | 3), key).  oracle/da_oracle.py links this file with the count-family
 * oracle, so orcc_family() / orcc_obs() select the observation law of the compiled model.
 */
#include <math.h>
#include <stdint.h>
#include <string.h>
#include "../include/dpomp.h"

void orc_philox4x32_10(const uint32_t ctr_in[4], const uint32_t key_in[2], uint32_t out[4]);
int orcc_family(void);
double orcc_obs(const dpomp_model_desc* m, const double* th, int t, const int64_t* x);

#define TAG_DA 3u
static void da_draw(uint64_t key, uint32_t id, uint32_t j, uint32_t block, uint32_t w[4]) {
    uint32_t ctr[4] = {id, j, 0u, (TAG_DA << 30) | block}, k[2] = {(uint32_t)key, (uint32_t)(key >> 32)};
    orc_philox4x32_10(ctr, k, w);
}
static inline double u53(uint32_t hi, uint32_t lo) { return (double)(((uint64_t)hi << 21) | (uint64_t)(lo >> 11)) * 0x1.0p-53; }
static inline int uint_below(uint32_t w, int n) { return (int)(((uint64_t)w * (uint64_t)n) >> 32); }

static void rates(const dpomp_model_desc* m, const double* th, const int64_t* x, double* out) {
    for (int e = 0; e < m->n_events; ++e) {
        int64_t l1 = m->rate_k1[e], l2 = m->rate_k2[e], dn = m->rate_kd[e];
        for (int c = 0; c < m->n_compartments; ++c) {
            l1 += (int64_t)m->rate_f1[e][c] * x[c];
            l2 += (int64_t)m->rate_f2[e][c] * x[c];
            dn += (int64_t)m->rate_dn[e][c] * x[c];
        }
        double p = m->rate_par[e] >= 0 ? th[m->rate_par[e]] : 1.0;
        double r = (p * (double)l1) * (double)l2;
        if (m->rate_has_den[e]) r = (dn == 0) ? 0.0 : r / (double)dn;
        out[e] = r;
    }
}
static double rate_sum(const double* r, int n) { double s = r[0]; for (int i = 1; i < n; ++i) s = s + r[i]; return s; }
static double obs_ll(const dpomp_model_desc* m, const double* th, int t, const int64_t* x) {
    if (orcc_family()) return orcc_obs(m, th, t, x);
    double tmp1 = log(1.0 / (sqrt(2.0 * M_PI) * m->obs_sigma)), tmp2 = 2.0 * m->obs_sigma * m->obs_sigma;
    int64_t ys = 0, xs = 0;
    for (int v = 0; v < m->n_obs_vals; ++v) ys += (int64_t)m->obs_ymask[v] * m->obs_val[(int64_t)t * m->n_obs_vals + v];
    for (int c = 0; c < m->n_compartments; ++c) xs += (int64_t)m->obs_xmask[c] * x[c];
    int64_t d = ys - xs;
    return tmp1 - ((double)(d * d) / tmp2);
}

/* full log-likelihood of (times, types)[0, n) (types 1-based) with index del skipped (-1: none) and the event (tins, eins)
 * (eins 0-based, -1: none) merged after the events at times <= tins.  ll2 = {full, observation part}; x = final state;
 * *q = position of the inserted event in the edited list. */
static void walk(const dpomp_model_desc* m, const double* th, const double* times, const int32_t* types, int64_t n, int64_t del,
                 double tins, int eins, int64_t* x, double* ll2, int64_t* q) {
    const int C = m->n_compartments, E = m->n_events;
    const double t0 = m->t0_index > 0 ? th[m->t0_index - 1] : 0.0;
    double lam[DPOMP_MAX_EVENTS], t = t0, ll = 0.0, llo = 0.0;
    int ins = eins >= 0;
    int64_t k = 0;
    for (int c = 0; c < C; ++c) x[c] = m->initial_condition[c];
    *q = 0;
    for (int oi = 0; oi < m->n_obs; ++oi) {
        const double t_obs = m->obs_time[oi];
        for (;;) {
            if (k == del) ++k;
            const double tk = k < n ? times[k] : INFINITY;
            const int take_ins = ins && !(tk <= tins);
            if (!take_ins && k >= n) break;
            const double te = take_ins ? tins : tk;
            if (te > t_obs) break;
            const int e = take_ins ? eins : types[k] - 1;
            if (!(te > t0)) goto invalid;
            rates(m, th, x, lam);
            if (!(lam[e] > 0.0)) goto invalid;
            ll += log(lam[e]) - rate_sum(lam, E) * (te - t);
            for (int c = 0; c < C; ++c) { x[c] += m->trans[e][c]; if (x[c] < 0) goto invalid; }
            t = te;
            if (take_ins) { ins = 0; *q = k - ((del >= 0 && del < k) ? 1 : 0); }
            else ++k;
        }
        rates(m, th, x, lam);
        ll -= rate_sum(lam, E) * (t_obs - t);
        t = t_obs;
        if (m->obs_id[oi] > 0) { const double g = obs_ll(m, th, oi, x); ll += g; llo += g; }
    }
    if (k == del) ++k;
    if (ins || k < n) goto invalid;
    ll2[0] = ll; ll2[1] = llo;
    return;
invalid:
    ll2[0] = ll2[1] = -INFINITY;
}

void orc_da_loglike(const dpomp_model_desc* m, const double* theta, const double* times, const int32_t* types, int64_t n,
                    int64_t* fc, double* ll2) {
    int64_t q;
    walk(m, theta, times, types, n, -1, 0.0, -1, fc, ll2, &q);
}

/* traj_props trajectory proposals of chain `id` under theta, applied in place to (times, types)[0, *len) (room for
 * *len + traj_props events); fc, ll2 = final state and {full, observation} log-likelihood of the result; acc[3] = accepted
 * inserts, deletes, moves.  max_traj: an insert into a trajectory of max_traj events is rejected. */
void orc_da_props(const dpomp_model_desc* m, const double* theta, double* times, int32_t* types, int64_t* len, int64_t max_traj,
                  int traj_props, int mvp, uint64_t key, uint32_t id, int64_t* fc, double* ll2, int64_t* acc) {
    const int C = m->n_compartments, E = m->n_events;
    const double t0 = m->t0_index > 0 ? theta[m->t0_index - 1] : 0.0, span = m->obs_time[m->n_obs - 1] - t0;
    int64_t q, xf[DPOMP_MAX_COMPARTMENTS];
    double llf[2];
    walk(m, theta, times, types, *len, -1, 0.0, -1, fc, ll2, &q);
    acc[0] = acc[1] = acc[2] = 0;
    for (int j = 0; j < traj_props; ++j) {
        uint32_t w[4], a[4];
        da_draw(key, id, (uint32_t)j, 2u, w);
        const int mk = 1 + uint_below(w[0], mvp);
        const double tnew = t0 + (1.0 - u53(w[2], w[3])) * span;
        const int64_t n = *len;
        int64_t del = -1;
        int eins = -1;
        double r;
        if (mk == 1) {
            if (n >= max_traj) continue;
            eins = uint_below(w[1], E);
            r = ((double)E * span) / (double)(n + 1);
        } else {
            if (n == 0) continue;
            del = uint_below(w[1], (int)n);
            if (mk == 2) r = (double)n / ((double)E * span);
            else { eins = types[del] - 1; r = 1.0; }
        }
        walk(m, theta, times, types, n, del, tnew, eins, xf, llf, &q);
        da_draw(key, id, (uint32_t)j, 3u, a);
        if (!(r * exp(llf[0] - ll2[0]) > u53(a[0], a[1]))) continue;
        /* the edited list: (times without del) with tnew inserted at q */
        if (del >= 0) {
            memmove(times + del, times + del + 1, sizeof(double) * (size_t)(n - del - 1));
            memmove(types + del, types + del + 1, sizeof(int32_t) * (size_t)(n - del - 1));
        }
        const int64_t n1 = del >= 0 ? n - 1 : n;
        if (eins >= 0) {
            memmove(times + q + 1, times + q, sizeof(double) * (size_t)(n1 - q));
            memmove(types + q + 1, types + q, sizeof(int32_t) * (size_t)(n1 - q));
            times[q] = tnew; types[q] = eins + 1;
        }
        *len = eins >= 0 ? n1 + 1 : n1;
        ll2[0] = llf[0]; ll2[1] = llf[1];
        for (int c = 0; c < C; ++c) fc[c] = xf[c];
        acc[mk < 3 ? mk - 1 : 2] += 1;
    }
}
