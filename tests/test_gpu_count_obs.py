"""GPU tests of the count observation families (Poisson, binomial, negative binomial; dpomp_model_set_obs_model): the f64
event loop draw for draw against the oracle, the f32 loop by z-test, the likelihood estimate against the exact forward
algorithm, theta-indexed parameters in a batch, the MBP walks against the oracle, and the posterior of the samplers."""
import ctypes as C
import math
import os

import numpy as np
import pytest
from scipy import stats

from conftest import GOLDEN

pytestmark = pytest.mark.gpu

POISSON, BINOMIAL, NEGBIN = 1, 2, 3


@pytest.fixture(scope="module")
def corc():
    """the CPU oracle with the count observation families (oracle/count_oracle.py)"""
    from oracle import count_oracle

    count_oracle.build()
    return count_oracle


FAMILIES = [(POISSON, 0.6, 0.0), (BINOMIAL, 0.6, 0.0), (NEGBIN, 0.6, 4.0)]


def obs_model(dp, family, a, k=0.0, a_index=None, k_index=None, seq=(2,)):
    if family == POISSON:
        return dp.partial_poisson_obs_model(a, rho_index=a_index, seq=seq)
    if family == BINOMIAL:
        return dp.partial_binomial_obs_model(a, p_index=a_index, seq=seq)
    return dp.partial_negbin_obs_model(a, k, rho_index=a_index, k_index=k_index, seq=seq)


def count_case(dp, shape, om, prior=None):
    """SIS on pooley.csv (2 compartments) or SEIR on seir_c3.csv (4 compartments, I observed) with the observed counts scaled
    by 0.6 (reported fraction), observed through the count model `om`."""
    if shape == "sis":
        rf = lambda o, p, x: (o.__setitem__(0, p[0] * x[0] * x[1]), o.__setitem__(1, p[1] * x[1]))
        model = dp.generate_custom_model("SIS", rf, [100, 1], [[-1, 1], [1, -1]], obs_model=om, prior=prior)
        y = dp.get_observations(os.path.join(GOLDEN, "pooley.csv"))
        theta = np.array([0.003, 0.1])
    else:
        def rf(o, p, x):
            o[0] = p[0] * x[0] * x[2]; o[1] = p[1] * x[1]; o[2] = p[2] * x[2]
        model = dp.generate_custom_model("SEIR", rf, [100, 0, 1, 0], [[-1, 1, 0, 0], [0, -1, 1, 0], [0, 0, -1, 1]], obs_model=om,
                                         prior=prior)
        y = dp.get_observations(os.path.join(GOLDEN, "seir_c3.csv"))
        theta = np.array([0.005, 0.2, 0.1])
    y = [dp.Observation(o.time, o.obs_id, o.prop, np.floor(0.6 * np.asarray(o.val)).astype(np.int64)) for o in y]
    if prior is not None and len(prior) > len(theta):
        theta = np.concatenate([theta, 0.5 * (prior.lower + prior.upper)[len(theta):]])
    return model, y, dp.get_private_model(model, y), theta


def _pf(dp, hmm, n, nb=1, rs=1, seed=1, f64=True):
    pf = dp.ParticleFilter(dp.device_model(hmm), n, nb, rs, seed=seed, sim_precision=dp._capi.SIM_F64 if f64 else dp._capi.SIM_F32)
    pf.set_record_ancestors(True)
    return pf


def rel_close(got, want, rtol):
    got, want = np.asarray(got), np.asarray(want)
    fin = np.isfinite(want)
    if not np.array_equal(fin, np.isfinite(got)) or not np.array_equal(got[~fin], want[~fin]):
        return False
    return bool(np.all(np.abs(got[fin] - want[fin]) <= rtol * np.maximum(np.abs(want[fin]), 1.0)))


@pytest.mark.parametrize("family,a,k", FAMILIES)
@pytest.mark.parametrize("shape", ["sis", "seir"])
def test_f64_loop_matches_oracle(dp, corc, family, a, k, shape):
    model, y, hmm, theta = count_case(dp, shape, obs_model(dp, family, a, k, seq=(2,) if shape == "sis" else (3,)))
    ymax = min(len(y), 4)
    for rs_type in (1, 2, 3):
        for n in (200, 1024, 3000, 4133):  # one 256-particle tile (fused kernel), one 1024 tile, ragged multi-tile chains
            pf = _pf(dp, hmm, n, rs=rs_type)
            tile, items = pf.geometry()
            key = 0xC0DE00 + n + 7 * rs_type + family
            pf.set_stream_key(key)
            ll = pf.partial(theta, 1, ymax)[0]
            o_ll, o_lw, o_anc, o_ev, o_ovf, o_pop = corc.pf_partial(pf.dmodel.compiled.desc, theta, n, None, 1, ymax, rs_type, key, 0,
                                                                   corc.MODE_DEVICE, tile, items)
            ctx = (family, shape, rs_type, n)
            assert pf.last_event_count() == o_ev, ctx
            assert np.array_equal(pf.get_pop(1), o_pop), ctx
            assert rel_close(pf.last_logw(), o_lw, 1e-13), ctx  # CUDA log / lgamma against glibc
            if ymax < len(y):
                assert np.array_equal(pf.last_ancestors(), o_anc), ctx
            assert abs(ll - o_ll) <= 1e-12 * max(1.0, abs(o_ll)), (ctx, ll, o_ll)


@pytest.mark.parametrize("family,a,k", FAMILIES)
def test_f32_loglik_z_test_against_oracle(dp, corc, family, a, k):
    model, y, hmm, theta = count_case(dp, "sis", obs_model(dp, family, a, k))
    n, reps = 1024, 128
    pf = _pf(dp, hmm, n, reps, seed=99, f64=False)
    gpu = pf.loglik(np.tile(theta[:, None], (1, reps)))
    ref, _ = corc.pf_partial_batch(pf.dmodel.compiled.desc, np.tile(theta[:, None], (1, reps)), n, 1, len(y), 1, key=20261021,
                                  threads=corc.max_threads())
    assert np.all(np.isfinite(gpu)) and np.all(np.isfinite(ref))
    z = (gpu.mean() - ref.mean()) / np.sqrt(gpu.var(ddof=1) / reps + ref.var(ddof=1) / reps)
    assert abs(z) < 4.5, (family, gpu.mean(), ref.mean(), z)
    assert 0.5 < gpu.std() / ref.std() < 2.0


YS_DEATH = [38, 30, 23, 17, 14]


def death_case(dp, family, a, k=0.0, a_index=None, prior=None):
    """Pure-death chain (I0 = 60, rate 0.05 per infective, observations 5 apart) observed through a count family, and its exact
    log-likelihood by the forward recursion over the 61 states."""
    rf = lambda o, p, x: (o.__setitem__(0, p[0] * x[0] * x[1]), o.__setitem__(1, p[1] * x[1]))
    om = obs_model(dp, family, a, k, a_index=a_index)
    model = dp.generate_custom_model("SIS", rf, [40, 60], [[-1, 1], [1, -1]], obs_model=om, prior=prior)
    y = [dp.Observation(5.0 * (i + 1), 1, 1.0, [0, v]) for i, v in enumerate(YS_DEATH)]
    states = np.arange(61)
    trans = stats.binom.pmf(states[None, :], states[:, None], np.exp(-0.05 * 5.0))
    alpha = np.zeros(61); alpha[60] = 1.0
    ll = 0.0
    for v in YS_DEATH:
        lp = {POISSON: lambda: stats.poisson.logpmf(v, a * states), BINOMIAL: lambda: stats.binom.logpmf(v, states, a),
              NEGBIN: lambda: stats.nbinom.logpmf(v, k, k / (k + a * states))}[family]()
        alpha = (alpha @ trans) * np.exp(lp)
        ll += np.log(alpha.sum())
        alpha /= alpha.sum()
    return model, y, dp.get_private_model(model, y), float(ll)


@pytest.mark.parametrize("family,a,k", [(POISSON, 0.8, 0.0), (BINOMIAL, 0.8, 0.0), (NEGBIN, 0.8, 5.0)])
@pytest.mark.parametrize("f64", [True, False])
def test_loglik_against_exact_forward_algorithm(dp, family, a, k, f64):
    model, y, hmm, exact = death_case(dp, family, a, k)
    nb = 64
    lls = _pf(dp, hmm, 4000, nb, seed=3, f64=f64).loglik(np.tile(np.array([[0.0], [0.05]]), (1, nb)))
    # the likelihood estimate is unbiased: the mean of exp(ll - exact) is 1 within its Monte-Carlo error
    r = np.exp(lls - exact)
    assert abs(r.mean() - 1.0) < 4.5 * r.std(ddof=1) / np.sqrt(nb) + 1e-3, (family, f64, lls.mean(), exact)


@pytest.mark.parametrize("family,lo,hi", [(POISSON, 0.3, 0.9), (BINOMIAL, 0.3, 0.9), (NEGBIN, 0.3, 0.9)])
def test_theta_indexed_parameter_in_a_batch(dp, family, lo, hi):
    prior = dp.UniformProduct([0.0, 0.0, lo], [0.01, 0.5, hi])
    model, y, hmm, theta = count_case(dp, "sis", obs_model(dp, family, 0.5, 4.0, a_index=2), prior=prior)
    assert dp.device_model(hmm).compiled.obs.par_index[0] == 2
    n, nb = 1500, 6
    thetas = np.tile(theta[:, None], (1, nb))
    thetas[2] = np.linspace(lo, hi, nb)
    thetas[2, 4] = 1.5 if family == BINOMIAL else -0.5  # outside the parameter's range: -Inf for filter 4 only
    pf = _pf(dp, hmm, n, nb)
    pf.set_stream_key(4242)
    lls = pf.partial(thetas, 1, 5)
    assert np.isneginf(lls[4]) and np.all(np.isfinite(np.delete(lls, 4))), lls
    for b in (0, 3, 5):
        single = _pf(dp, hmm, n, 1)
        single.set_batch_offset(b)
        single.set_stream_key(4242)
        assert single.partial(thetas[:, b], 1, 5)[0] == lls[b]
        assert np.array_equal(single.get_pop(1), pf.get_pop(b + 1))
    # the reporting rate moves the likelihood
    assert len(set(np.round(np.delete(lls, 4), 6))) == nb - 1


def test_theta_indexed_size_matches_oracle(dp, corc):
    prior = dp.UniformProduct([0.0, 0.0, 0.1, 1.0], [0.01, 0.5, 1.0, 10.0])
    model, y, hmm, theta = count_case(dp, "sis", obs_model(dp, NEGBIN, 0.5, 3.0, a_index=2, k_index=3), prior=prior)
    pf = _pf(dp, hmm, 3000)
    tile, items = pf.geometry()
    pf.set_stream_key(99)
    ll = pf.partial(theta, 1, 3)[0]
    o = corc.pf_partial(pf.dmodel.compiled.desc, theta, 3000, None, 1, 3, 1, 99, 0, corc.MODE_DEVICE, tile, items)
    assert np.array_equal(pf.get_pop(1), o[5]) and rel_close(pf.last_logw(), o[1], 1e-13) and abs(ll - o[0]) <= 1e-12 * abs(o[0])


def test_obs_id_zero_is_skipped(dp, corc):
    model, y, hmm, theta = count_case(dp, "sis", obs_model(dp, POISSON, 0.6))
    y2 = [dp.Observation(o.time, 0 if i == 1 else 1, 1.0, o.val) for i, o in enumerate(y)]
    hmm2 = dp.get_private_model(model, y2)
    pf = _pf(dp, hmm2, 1024)
    tile, items = pf.geometry()
    pf.set_stream_key(55)
    ll = pf.loglik(theta)[0]
    o = corc.pf_partial(pf.dmodel.compiled.desc, theta, 1024, None, 1, 5, 1, 55, 0, corc.MODE_DEVICE, tile, items)
    assert abs(ll - o[0]) <= 1e-12 * abs(o[0]) and np.array_equal(pf.get_pop(1), o[5])
    pf.set_stream_key(55)
    assert pf.loglik(theta)[0] == ll
    full = _pf(dp, hmm, 1024)
    full.set_stream_key(55)
    assert full.loglik(theta)[0] != ll  # the skipped observation contributes nothing


def test_set_obs_model_after_a_filter_handle_is_refused(dp):
    model, y, hmm, theta = count_case(dp, "sis", obs_model(dp, POISSON, 0.6))
    dm = dp.DeviceModel(dp.compile_model(model, y))
    idx = np.array([-1, -1], dtype=np.int32); val = np.array([0.5, 0.0])
    lib = dp._capi.lib()
    assert lib.dpomp_model_set_obs_model(dm.handle, BINOMIAL, idx.ctypes.data, val.ctypes.data) == 0
    pf = dp.ParticleFilter(dm, 256)
    assert lib.dpomp_model_set_obs_model(dm.handle, POISSON, idx.ctypes.data, val.ctypes.data) == -4
    assert pf.loglik(theta)[0] <= 0.0


@pytest.mark.parametrize("family,a,k", FAMILIES)
@pytest.mark.parametrize("mode", [1, 2])  # one thread / one warp per trajectory
def test_mbp_iterate_and_propose_match_oracle(dp, corc, family, a, k, mode):
    prior = dp.UniformProduct([0.0, 0.0, 0.3], [0.01, 0.5, 0.9])
    model, y, hmm, theta = count_case(dp, "sis", obs_model(dp, family, a, k, a_index=2), prior=prior)
    dm = dp.device_model(hmm)
    desc = dm.compiled.desc
    n, cap = 48, 4096
    rng = np.random.default_rng(3)
    thetas = theta[:, None] * rng.uniform(0.8, 1.25, size=(3, n))
    pt = dp.MbpParticles(dm, n, cap, seed=5)
    pt.set_mode(mode)
    n_obs = 4
    o_fc = np.tile(np.asarray(model.initial_condition, dtype=np.int64), (n, 1))
    o_t = np.zeros((n, cap)); o_y = np.zeros((n, cap), dtype=np.int32); o_len = np.zeros(n, dtype=np.int64); o_ll = np.zeros((n, 2))
    for obs_i in range(1, n_obs + 1):
        key = 9100 + obs_i
        pt.set_stream_key(key)
        lg = pt.iterate(thetas, obs_i, fresh=(obs_i == 1))
        for p in range(n):
            t_start = 0.0 if obs_i == 1 else y[obs_i - 2].time
            g, o_len[p] = corc.mbp_iterate(desc, thetas[:, p], o_fc[p], o_t[p], o_y[p], o_len[p], o_ll[p], t_start, obs_i, key, p)
            assert rel_close([lg[p]], [g], 1e-12), (p, obs_i, lg[p], g)
    theta_f = thetas * rng.uniform(0.85, 1.2, size=thetas.shape)
    valid = np.ones(n, dtype=bool); valid[3] = False
    pt.set_stream_key(777)
    ll_f = pt.propose(thetas, theta_f, valid, n_obs)
    assert np.all(np.isneginf(ll_f[3]))
    for p in (0, 1, 7, 20, n - 1):
        times, types, fc, ll, rc = corc.mbp_propose(desc, thetas[:, p], theta_f[:, p], o_t[p], o_y[p], o_len[p], cap, n_obs, 777, p)
        g_fc, g_times, g_types, g_ll = pt.get_particle(p + 1, proposal=True)
        assert rc == 0 and np.array_equal(g_fc, fc) and np.array_equal(g_types, types)
        assert rel_close(g_ll, ll, 1e-12) and rel_close(ll_f[p], ll, 1e-12)


def _death_posterior(dp, nodes=1201):
    """One-parameter pure-death model (rate theta * I, prior U(0, 0.2)) with Poisson(0.8 I) observations of YS_DEATH, the
    exact likelihood on a grid and the posterior mean by quadrature."""
    def rf(out, p, x):
        out[0] = p[0] * x[1]
    model = dp.generate_custom_model("DEATH", rf, [40, 60], [[1, -1]], obs_model=dp.partial_poisson_obs_model(0.8),
                                     prior=dp.UniformProduct([0.0], [0.2]))
    y = [dp.Observation(5.0 * (i + 1), 1, 1.0, [0, v]) for i, v in enumerate(YS_DEATH)]
    states = np.arange(61)

    def exact_ll(gam):
        trans = stats.binom.pmf(states[None, :], states[:, None], np.exp(-gam * 5.0))
        alpha = np.zeros(61); alpha[60] = 1.0
        ll = 0.0
        for v in YS_DEATH:
            alpha = (alpha @ trans) * stats.poisson.pmf(v, 0.8 * states)
            ll += np.log(alpha.sum())
            alpha /= alpha.sum()
        return ll
    g = np.linspace(0.0, 0.2, nodes)
    lik = np.exp(np.array([exact_ll(v) for v in g]))
    z = np.trapezoid(lik, g)
    mean = np.trapezoid(lik * g, g) / z
    sd = np.sqrt(np.trapezoid(lik * (g - mean) ** 2, g) / z)
    return model, y, float(mean), float(sd)


def test_mbp_mcmc_and_pmcmc_posterior_against_quadrature(dp):
    model, y, mean, sd = _death_posterior(dp)
    th0 = np.random.default_rng(8).uniform(0.03, 0.07, size=(1, 8))
    r = dp.run_mcmc_analysis(model, y, n_chains=8, initial_parameters=th0, steps=4000, adapt_period=800, seed=5, verbose=False)
    post = r.samples.theta[0, 800:, :].ravel()
    assert abs(post.mean() - mean) < 0.25 * sd, (post.mean(), mean, sd)
    hmm = dp.get_private_model(model, y)
    res = dp.run_pmcmc(hmm, th0, steps=3000, adapt_period=600, p=256, seed=11, verbose=False)
    post = res.samples.theta[0, 600:, :].ravel()
    assert abs(post.mean() - mean) < 0.25 * sd, (post.mean(), mean, sd)


def test_smc2_theta_indexed_reporting_rate_against_oracle(dp, corc):
    prior = dp.UniformProduct([0.0, 0.0, 0.2], [0.01, 0.5, 1.0])
    model, y, hmm, theta = count_case(dp, "sis", obs_model(dp, POISSON, 0.5, a_index=2), prior=prior)
    cm = dp.compile_model(model, y)
    reps, n_outer, npf = 4, 1000, 200
    ours, ref = [], []
    for s in range(reps):
        r = dp.run_ibis_analysis(model, y, np=n_outer, npf=npf, seed=40 + s, verbose=False)
        ours.append(r.bme[0])
        th0 = prior.rand(n_outer, np.random.default_rng(70 + s))
        ref.append(corc.run_pibis(cm.desc, th0, prior.lower, prior.upper, npf=npf, seed=90 + s, threads=corc.max_threads())["bme"][0])
    ours, ref = np.array(ours), np.array(ref)
    assert np.all(np.isfinite(ours)) and np.all(np.isfinite(ref))
    z = (ours.mean() - ref.mean()) / np.sqrt(ours.var(ddof=1) / reps + ref.var(ddof=1) / reps + 1e-6)
    assert abs(z) < 4.5, (ours, ref)


def test_user_written_poisson_closure_runs_end_to_end(dp):
    """A closure with the reference's signature, logpdf(Poisson(theta[3] * pop[2]), y.val[2]), compiles to the device table
    and runs through the filter, MBP-MCMC and SMC^2."""
    def obs(y, pop, th):
        return stats.poisson.logpmf(y.val[1], th[2] * pop[1])

    prior = dp.UniformProduct([0.0, 0.0, 0.2], [0.01, 0.5, 1.0])
    rf = lambda o, p, x: (o.__setitem__(0, p[0] * x[0] * x[1]), o.__setitem__(1, p[1] * x[1]))
    model = dp.generate_custom_model("SIS", rf, [100, 1], [[-1, 1], [1, -1]], obs_model=obs, prior=prior)
    y = count_case(dp, "sis", dp.partial_poisson_obs_model(0.6))[1]
    cm = dp.compile_model(model, y)
    assert (cm.obs.family, cm.obs.par_index[0]) == (POISSON, 2)
    f = dp.get_particle_filter_lpdf(model, y, np=2000)
    assert np.isfinite(f(np.array([0.003, 0.1, 0.6])))
    r = dp.run_mcmc_analysis(model, y, n_chains=2, steps=200, seed=3, verbose=False)
    assert np.all(np.isfinite(r.samples.theta))
    s = dp.run_ibis_analysis(model, y, np=200, npf=100, seed=2, verbose=False)
    assert np.all(np.isfinite(s.mu))
