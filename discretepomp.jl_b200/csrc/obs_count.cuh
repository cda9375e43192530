// obs_count.cuh -- the count observation families of dpomp_model_set_obs_model (include/dpomp.h): Poisson, binomial and
// negative-binomial log pmfs of Y = ymask.y given X = xmask.x, in f64, shared by the filter's weight pass (pf_sim.cuh) and the
// MBP walks (mbp.cu).
//
// Everything that depends only on (filter or trajectory, observation) is formed once in count_obs_const: log rho, log p,
// log1p(-p), k, the host constant lgamma(Y+1) and lgamma(Y+k) - lgamma(k) (host value when k is fixed, device lgamma when it
// is theta-indexed).  Per particle the Poisson law then costs one log, the binomial two lgamma, the negative binomial two
// log.  The association of every expression is the one of oracle/dpomp_oracle_count.c (explicitly rounded: no contraction), so
// with fixed parameters the log weights differ from the oracle's only by CUDA log / lgamma against glibc.
#pragma once
#include <math.h>
#include <stdint.h>

#include "../../include/dpomp.h"

namespace dpomp {

// the model's count observation law as the kernels receive it (by value; the pointers are device arrays [T])
struct CountObs {
    int family;             // DPOMP_OBS_POISSON / _BINOMIAL / _NEGBIN
    int par_index[2];       // 0-based theta index, or -1: par_value
    double par_value[2];
    const double* lgy;      // [T] lgamma(Y+1)
    const double* lgk;      // [T] lgamma(Y+k) - lgamma(k) for a fixed k (negative binomial), else unused
};

// per (filter, observation) constants; CTA-uniform in the filter's weight pass
struct CountObsConst {
    int family;
    bool bad;      // parameter out of range or Y < 0: every log g is -Inf
    double a;      // rho (Poisson, negative binomial) or p (binomial)
    double k;      // size (negative binomial)
    double la;     // log rho or log p
    double lb;     // log1p(-p)
    double lgy;    // lgamma(Y+1)
    double lgk;    // lgamma(Y+k) - lgamma(k)
};

__device__ __forceinline__ double count_obs_par(const CountObs& co, const double* th, int i) {
    return co.par_index[i] >= 0 ? th[co.par_index[i]] : co.par_value[i];
}

__device__ __forceinline__ CountObsConst count_obs_const(const CountObs& co, const double* th, int t, double y) {
    CountObsConst c{};
    c.family = co.family;
    c.a = count_obs_par(co, th, 0);
    c.bad = !(y >= 0.0);
    c.lgy = co.lgy[t];
    if (co.family == DPOMP_OBS_BINOMIAL) {
        c.bad = c.bad || !(c.a >= 0.0 && c.a <= 1.0);
        c.la = log(c.a);
        c.lb = log1p(-c.a);
    } else {
        c.bad = c.bad || !(c.a > 0.0 && c.a < INFINITY);
        c.la = log(c.a);
        if (co.family == DPOMP_OBS_NEGBIN) {
            c.k = count_obs_par(co, th, 1);
            c.bad = c.bad || !(c.k > 0.0 && c.k < INFINITY);
            c.lgk = co.par_index[1] >= 0 ? __dsub_rn(lgamma(__dadd_rn(y, c.k)), lgamma(c.k)) : co.lgk[t];
        }
    }
    return c;
}

// log g(Y | X) of the model's family; x >= 0 (0/1 masks)
__device__ __forceinline__ double count_obs_logpmf(const CountObsConst& c, double y, double x) {
    if (c.bad) return -INFINITY;
    switch (c.family) {
        case DPOMP_OBS_POISSON: {
            if (x == 0.0) return y == 0.0 ? 0.0 : -INFINITY;
            const double ylog = y == 0.0 ? 0.0 : __dmul_rn(y, __dadd_rn(c.la, log(x)));
            return __dsub_rn(__dsub_rn(ylog, __dmul_rn(c.a, x)), c.lgy);
        }
        case DPOMP_OBS_BINOMIAL: {
            if (y > x) return -INFINITY;
            if (c.a == 0.0) return y == 0.0 ? 0.0 : -INFINITY;
            if (c.a == 1.0) return y == x ? 0.0 : -INFINITY;
            const double nx = __dsub_rn(x, y);
            double r = __dsub_rn(__dsub_rn(lgamma(__dadd_rn(x, 1.0)), c.lgy), lgamma(__dadd_rn(nx, 1.0)));
            r = __dadd_rn(r, __dmul_rn(y, c.la));
            return __dadd_rn(r, __dmul_rn(nx, c.lb));
        }
        default: {  // DPOMP_OBS_NEGBIN
            if (x == 0.0) return y == 0.0 ? 0.0 : -INFINITY;
            const double mu = __dmul_rn(c.a, x);
            const double km = __dadd_rn(c.k, mu);
            double r = __dadd_rn(__dsub_rn(c.lgk, c.lgy), __dmul_rn(c.k, log(__ddiv_rn(c.k, km))));
            return y == 0.0 ? r : __dadd_rn(r, __dmul_rn(y, log(__ddiv_rn(mu, km))));
        }
    }
}

}  // namespace dpomp
