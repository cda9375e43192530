"""CPU tests of the count observation families (Poisson, binomial, negative binomial; include/dpomp.h DPOMP_OBS_*): the
constructors and the oracle against scipy.stats, the closure probe of rate_table.compile_obs_table, argument validation of
dpomp_model_set_obs_model, and the oracle's filter against the exact forward algorithm of a pure-death chain."""
import ctypes as C
import math

import numpy as np
import pytest
from scipy import stats

POISSON, BINOMIAL, NEGBIN = 1, 2, 3


@pytest.fixture(scope="module")
def corc():
    """the CPU oracle with the count observation families (oracle/count_oracle.py)"""
    from oracle import count_oracle

    count_oracle.build()
    return count_oracle


def scipy_logpmf(family, y, x, a, k=0.0):
    if family == POISSON:
        return stats.poisson.logpmf(y, a * x)
    if family == BINOMIAL:
        return stats.binom.logpmf(y, x, a)
    return stats.nbinom.logpmf(y, k, k / (k + a * x))


def close(got, want, rtol=1e-12):
    if math.isinf(want) or math.isinf(got):
        return got == want
    return abs(got - want) <= rtol * max(1.0, abs(want))


CASES = [(POISSON, 0.7, 0.0), (BINOMIAL, 0.35, 0.0), (NEGBIN, 0.6, 3.5)]


@pytest.mark.parametrize("family,a,k", CASES)
def test_constructors_match_scipy(dp, family, a, k):
    ctor = {POISSON: lambda: dp.partial_poisson_obs_model(a), BINOMIAL: lambda: dp.partial_binomial_obs_model(a),
            NEGBIN: lambda: dp.partial_negbin_obs_model(a, k)}[family]
    om = ctor()
    rng = np.random.default_rng(family)
    for _ in range(300):
        x = int(rng.integers(0, 200)); y = int(rng.integers(0, 220))
        got = om(dp.Observation(1.0, 1, 1.0, [0, y]), np.array([5, x]), np.zeros(2))
        assert close(got, scipy_logpmf(family, y, x, a, k)), (family, y, x, got)
    tab = om.obs_table(2, 2)
    assert tab.family == family and tab.xmask.tolist() == [0, 1] and tab.ymask.tolist() == [0, 1]


def test_boundary_cases(dp):
    cl = dp.rate_table.count_logpmf
    for fam in (POISSON, NEGBIN):  # zero mean: 0 for Y = 0, -inf otherwise
        assert cl(fam, 0, 0, 0.5, 2.0) == 0.0 and cl(fam, 1, 0, 0.5, 2.0) == -math.inf
    assert cl(BINOMIAL, 5, 4, 0.5) == -math.inf                              # Y > X
    assert cl(BINOMIAL, 0, 7, 0.0) == 0.0 and cl(BINOMIAL, 1, 7, 0.0) == -math.inf  # p = 0 exact
    assert cl(BINOMIAL, 7, 7, 1.0) == 0.0 and cl(BINOMIAL, 6, 7, 1.0) == -math.inf  # p = 1 exact
    assert cl(BINOMIAL, 0, 0, 0.3) == 0.0                                    # 0 log 0 = 0
    assert cl(POISSON, 0, 9, 0.5) == pytest.approx(-4.5, rel=1e-15)          # 0 log(rho X) = 0
    for bad in ((BINOMIAL, 1.2, 0.0), (BINOMIAL, -0.1, 0.0), (POISSON, 0.0, 0.0), (NEGBIN, 0.5, 0.0), (NEGBIN, -1.0, 2.0)):
        assert cl(bad[0], 3, 10, bad[1], bad[2]) == -math.inf                # theta-indexed value out of range
    assert cl(POISSON, -1, 10, 0.5) == -math.inf


@pytest.mark.parametrize("family,a,k", CASES)
def test_oracle_families_match_scipy(corc, family, a, k):
    rng = np.random.default_rng(10 + family)
    for _ in range(300):
        x = int(rng.integers(0, 200)); y = int(rng.integers(0, 220))
        assert close(corc.count_logpmf(family, y, x, a, k), scipy_logpmf(family, y, x, a, k)), (family, y, x)
    assert corc.count_logpmf(BINOMIAL, 0, 0, 0.3) == 0.0 and corc.count_logpmf(BINOMIAL, 4, 3, 0.3) == -math.inf
    assert corc.count_logpmf(POISSON, 1, 0, 0.3) == -math.inf and corc.count_logpmf(NEGBIN, 0, 0, 0.3, 2.0) == 0.0
    assert corc.count_logpmf(BINOMIAL, 3, 3, 1.0) == 0.0 and corc.count_logpmf(BINOMIAL, 2, 3, 1.5) == -math.inf


def _compile(dp, om, n_comp=3, n_vals=3, n_params=3):
    return dp.compile_obs_table(om, n_comp, n_vals, n_params)


def test_probe_compiles_scipy_and_lgamma_closures(dp):
    def pois(y, pop, th):  # logpdf(Poisson(0.4 * pop[2]), y.val[2])
        return stats.poisson.logpmf(y.val[1], 0.4 * pop[1])

    def pois_theta(y, pop, th):  # logpdf(Poisson(theta[3] * pop[2]), y.val[2])
        return stats.poisson.logpmf(y.val[1], th[2] * pop[1])

    def binom_lgamma(y, pop, th):  # hand-written with math.lgamma, detection probability 0.25, two observed compartments
        n, k, p = int(pop[1] + pop[2]), int(y.val[2]), 0.25
        if k > n:
            return -math.inf
        return math.lgamma(n + 1) - math.lgamma(k + 1) - math.lgamma(n - k + 1) + k * math.log(p) + (n - k) * math.log1p(-p)

    def nb_theta(y, pop, th):  # mean theta[1] * I, size 4
        mu = th[0] * pop[1]
        return stats.nbinom.logpmf(y.val[1], 4.0, 4.0 / (4.0 + mu))

    t = _compile(dp, pois)
    assert (t.family, t.par_index[0], t.par_value[0]) == (POISSON, -1, 0.4)
    assert t.xmask.tolist() == [0, 1, 0] and t.ymask.tolist() == [0, 1, 0]
    t = _compile(dp, pois_theta)
    assert (t.family, t.par_index[0]) == (POISSON, 2)
    t = _compile(dp, binom_lgamma)
    assert (t.family, t.par_index[0], t.par_value[0]) == (BINOMIAL, -1, 0.25)
    assert t.xmask.tolist() == [0, 1, 1] and t.ymask.tolist() == [0, 0, 1]
    t = _compile(dp, nb_theta)
    assert (t.family, t.par_index, t.par_value[1]) == (NEGBIN, (0, -1), 4.0)


def test_probe_keeps_gaussian_and_rejects_other_laws(dp):
    t = _compile(dp, dp.partial_gaussian_obs_model(2.0), 3, 3)  # carries its table
    assert t.family == 0

    def gauss(y, pop, th):
        return math.log(1 / (math.sqrt(2 * math.pi) * 3.0)) - (y.val[1] - pop[1]) ** 2 / 18.0

    t = _compile(dp, gauss)
    assert t.family == 0 and t.sigma == pytest.approx(3.0) and t.xmask.tolist() == [0, 1, 0]

    def laplace(y, pop, th):
        return -abs(y.val[1] - pop[1]) - math.log(2.0)

    with pytest.raises(dp.ModelCompileError):
        _compile(dp, laplace)

    def pois_of_square(y, pop, th):
        return stats.poisson.logpmf(y.val[1], 0.1 * pop[1] ** 2)

    with pytest.raises(dp.ModelCompileError):
        _compile(dp, pois_of_square)


def _desc(dp, om=None):
    model = dp.generate_custom_model("SIS", lambda o, p, x: (o.__setitem__(0, p[0] * x[0] * x[1]), o.__setitem__(1, p[1] * x[1])),
                                     [100, 1], [[-1, 1], [1, -1]], obs_model=om)
    y = [dp.Observation(1.0, 1, 1.0, [0, 3]), dp.Observation(2.0, 1, 1.0, [0, 5])]
    return dp.compile_model(model, y)


def test_set_obs_model_validates_its_arguments(built_lib, dp):
    assert built_lib.dpomp_version() == 102
    cm = _desc(dp)
    h = C.c_void_p()
    assert built_lib.dpomp_model_create(C.byref(cm.desc), C.byref(h)) == 0
    idx = np.array([-1, -1], dtype=np.int32)
    val = np.array([0.5, 2.0])

    def call(family, i0=-1, v0=0.5, i1=-1, v1=2.0):
        idx[:] = (i0, i1); val[:] = (v0, v1)
        return built_lib.dpomp_model_set_obs_model(h, family, idx.ctypes.data, val.ctypes.data)

    try:
        assert call(7) == -1 and b"unknown" in built_lib.dpomp_last_error()
        assert call(-1) == -1
        assert built_lib.dpomp_model_set_obs_model(h, 1, None, val.ctypes.data) == -1
        assert call(POISSON, i0=2) == -3           # n_params = 2
        assert call(NEGBIN, i1=5) == -3
        assert call(BINOMIAL, v0=1.5) == -3        # fixed p out of range
        assert call(POISSON, v0=0.0) == -3
        assert call(NEGBIN, v1=-1.0) == -3
        assert call(POISSON) == 0 and call(BINOMIAL, i0=1) == 0 and call(NEGBIN, i0=0, i1=1) == 0
        assert call(0) == 0                        # back to the Gaussian
    finally:
        built_lib.dpomp_model_destroy(h)
    # count families need 0/1 masks
    bad = dp._capi.ModelDesc.from_buffer_copy(bytes(cm.desc))
    bad.obs_xmask[1] = 2
    h = C.c_void_p()
    assert built_lib.dpomp_model_create(C.byref(bad), C.byref(h)) == 0
    try:
        assert call(POISSON) == -3 and b"0/1" in built_lib.dpomp_last_error()
        assert call(0) == 0
    finally:
        built_lib.dpomp_model_destroy(h)


def test_device_model_carries_the_count_family(built_lib, dp):
    cm = _desc(dp, dp.partial_negbin_obs_model(0.5, 3.0, rho_index=1))
    assert cm.obs.family == NEGBIN and cm.desc.obs_spec == (NEGBIN, (1, -1), (0.5, 3.0))
    dm = dp.DeviceModel(cm)  # dpomp_model_create + dpomp_model_set_obs_model, no device needed
    assert dm.handle


# ---- the oracle's filter against the exact forward algorithm --------------------------------------------------------------
YS_COUNT = [38, 30, 23, 17, 14]


def count_death_case(dp, om, family, a, k=0.0):
    """Pure-death chain of conftest.pure_death_case (I0 = 60, death rate 0.05, five observations 5 apart) observed through a
    count family; returns (compiled model, theta, exact log-likelihood by the forward recursion over the 61 states)."""
    model = dp.generate_custom_model("SIS", lambda o, p, x: (o.__setitem__(0, p[0] * x[0] * x[1]), o.__setitem__(1, p[1] * x[1])),
                                     [40, 60], [[-1, 1], [1, -1]], obs_model=om)
    y = [dp.Observation(5.0 * (i + 1), 1, 1.0, [0, v]) for i, v in enumerate(YS_COUNT)]
    gam = 0.05
    states = np.arange(61)
    trans = stats.binom.pmf(states[None, :], states[:, None], np.exp(-gam * 5.0))
    alpha = np.zeros(61); alpha[60] = 1.0
    ll = 0.0
    for v in YS_COUNT:
        em = np.exp([scipy_logpmf(family, v, s, a, k) for s in states])
        alpha = (alpha @ trans) * em
        ll += np.log(alpha.sum())
        alpha /= alpha.sum()
    return dp.compile_model(model, y), np.array([0.0, gam]), float(ll)


@pytest.mark.parametrize("family,a,k", [(POISSON, 0.8, 0.0), (BINOMIAL, 0.8, 0.0), (NEGBIN, 0.8, 5.0)])
def test_oracle_filter_matches_exact_forward_algorithm(dp, corc, family, a, k):
    om = {POISSON: lambda: dp.partial_poisson_obs_model(a), BINOMIAL: lambda: dp.partial_binomial_obs_model(a),
          NEGBIN: lambda: dp.partial_negbin_obs_model(a, k)}[family]()
    cm, theta, exact = count_death_case(dp, om, family, a, k)
    est = [corc.pf_loglik(cm.desc, theta, 4000, key=s, threads=corc.max_threads())[0] for s in range(8)]
    # the likelihood estimate is unbiased; its log is biased low by about var / 2 (tiny at 4000 particles)
    assert abs(np.log(np.mean(np.exp(np.array(est) - exact)))) < 0.05, (est, exact)
    # the oracle's per-particle log weights at the last observation (which does not resample) are the family's log pmf
    ll, lw, anc, ev, ovf, pop = corc.pf_partial(cm.desc, theta, 64, None, 1, 5, key=3)
    for p in range(64):
        assert close(lw[p], scipy_logpmf(family, YS_COUNT[-1], int(pop[p, 1]), a, k), 1e-11)
