/*
 * dpomp_oracle_count.c -- count observation families of the CPU oracle (TEST INFRASTRUCTURE ONLY).
 *
 * The laws of dpomp_model_set_obs_model (include/dpomp.h): Poisson(rho X), Binomial(X, p) and the negative binomial of mean
 * rho X and size k, as log pmfs of Y = ymask.y given X = xmask.x, in plain C with glibc lgamma / log / log1p and the
 * association of the device code (discretepomp.jl_b200/csrc/obs_count.cuh).  oracle/count_oracle.py links this file with the
 * oracle's filter and MBP sources, whose observation calls it redirects here when a count family is selected; the reference
 * oracle (liboracle.so) is built from the unchanged sources and keeps the Gaussian only.
 */
#include <math.h>
#include <stdint.h>

#include "../include/dpomp.h"

double orc_count_logpmf(int family, int64_t yi, int64_t xi, double a, double k) {
    const double y = (double)yi, x = (double)xi;
    if (yi < 0) return -INFINITY;
    if (family == DPOMP_OBS_POISSON) {
        if (!(a > 0.0 && a < INFINITY)) return -INFINITY;
        if (xi == 0) return yi == 0 ? 0.0 : -INFINITY;
        const double ylog = yi == 0 ? 0.0 : y * (log(a) + log(x));
        return (ylog - a * x) - lgamma(y + 1.0);
    }
    if (family == DPOMP_OBS_BINOMIAL) {
        if (!(a >= 0.0 && a <= 1.0)) return -INFINITY;
        if (yi > xi) return -INFINITY;
        if (a == 0.0) return yi == 0 ? 0.0 : -INFINITY;
        if (a == 1.0) return yi == xi ? 0.0 : -INFINITY;
        const double nx = x - y;
        double r = (lgamma(x + 1.0) - lgamma(y + 1.0)) - lgamma(nx + 1.0);
        r = r + y * log(a);
        return r + nx * log1p(-a);
    }
    if (family == DPOMP_OBS_NEGBIN) {
        if (!(a > 0.0 && a < INFINITY) || !(k > 0.0 && k < INFINITY)) return -INFINITY;
        if (xi == 0) return yi == 0 ? 0.0 : -INFINITY;
        const double mu = a * x, km = k + mu;
        const double r = ((lgamma(y + k) - lgamma(k)) - lgamma(y + 1.0)) + k * log(k / km);
        return yi == 0 ? r : r + y * log(mu / km);
    }
    return NAN;
}

/* the family of the next calls (count_oracle.py sets it from the compiled model before every call); 0 = Gaussian */
static int g_family = DPOMP_OBS_GAUSSIAN;
static int32_t g_index[2] = {-1, -1};
static double g_value[2] = {0.0, 0.0};
void orc_set_obs_model(int family, const int32_t* par_index, const double* par_value) {
    g_family = family;
    for (int i = 0; i < 2; ++i) {
        g_index[i] = par_index ? par_index[i] : -1;
        g_value[i] = par_value ? par_value[i] : 0.0;
    }
}
int orcc_family(void) { return g_family; }

/* log g of observation t (0-based) at state x, theta-indexed parameters from th */
double orcc_obs(const dpomp_model_desc* m, const double* th, int t, const int64_t* x) {
    int64_t ys = 0, xs = 0;
    for (int v = 0; v < m->n_obs_vals; ++v) ys += (int64_t)m->obs_ymask[v] * m->obs_val[(int64_t)t * m->n_obs_vals + v];
    for (int c = 0; c < m->n_compartments; ++c) xs += (int64_t)m->obs_xmask[c] * x[c];
    const double a = g_index[0] >= 0 ? th[g_index[0]] : g_value[0];
    const double k = g_index[1] >= 0 ? th[g_index[1]] : g_value[1];
    return orc_count_logpmf(g_family, ys, xs, a, k);
}
