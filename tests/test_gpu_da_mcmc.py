"""GPU tests of data-augmented MCMC (dpomp_da_loglike, dpomp_da_step, run_std_mcmc): the full log-likelihood and the
insert / delete / move step against the oracle on identical Philox draws, the host driver on the device store against the
oracle-backed store, posteriors, and the growth of the store under inserts."""
import os
import sys

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, load_case

sys.path.insert(0, os.path.join(ROOT, "tests"))
pytestmark = pytest.mark.gpu

POISSON, BINOMIAL, NEGBIN = 1, 2, 3


@pytest.fixture(scope="module")
def dao():
    from oracle import da_oracle

    da_oracle.build()
    return da_oracle


def _case(dp, name):
    """(model, y, hmm, theta) of the cases the walks are checked on"""
    if name in ("sis_pooley", "seir_c3"):
        return load_case(dp, name)
    y = dp.get_observations(os.path.join(GOLDEN, "pooley.csv"))
    if name == "sis_freq":  # denominators: the generic rate-table kernel
        model = dp.generate_model("SIS", [100, 1], freq_dep=True)
        return model, y, dp.get_private_model(model, y), np.array([0.3, 0.1])
    rf = lambda o, p, x: (o.__setitem__(0, p[0] * x[0] * x[1]), o.__setitem__(1, p[1] * x[1]))
    if name == "sis_t0":
        model = dp.generate_custom_model("SIS", rf, [100, 1], [[-1, 1], [1, -1]], prior=dp.generate_weak_prior(3), t0_index=3)
        return model, y, dp.get_private_model(model, y), np.array([0.003, 0.1, 4.0])
    family = {"poisson": POISSON, "binomial": BINOMIAL, "negbin": NEGBIN}[name]
    om = {POISSON: lambda: dp.partial_poisson_obs_model(0.6, rho_index=2),
          BINOMIAL: lambda: dp.partial_binomial_obs_model(0.6, p_index=2),
          NEGBIN: lambda: dp.partial_negbin_obs_model(0.6, 4.0, rho_index=2)}[family]()
    prior = dp.UniformProduct([0.0, 0.0, 0.3], [0.01, 0.5, 0.9])
    model = dp.generate_custom_model("SIS", rf, [100, 1], [[-1, 1], [1, -1]], obs_model=om, prior=prior)
    y = [dp.Observation(o.time, o.obs_id, o.prop, np.floor(0.6 * np.asarray(o.val)).astype(np.int64)) for o in y]
    return model, y, dp.get_private_model(model, y), np.array([0.003, 0.1, 0.6])


CASES = ["sis_pooley", "seir_c3", "sis_freq", "sis_t0", "poisson", "binomial", "negbin"]


def rel_close(got, want, rtol=1e-12):
    got, want = np.asarray(got, dtype=float), np.asarray(want, dtype=float)
    fin = np.isfinite(want)
    if not np.array_equal(fin, np.isfinite(got)) or not np.array_equal(got[~fin], want[~fin]):
        return False
    return bool(np.all(np.abs(got[fin] - want[fin]) <= rtol * np.maximum(np.abs(want[fin]), 1.0)))


def _thetas(theta, n, rng, t0):
    th = theta[:, None] * rng.uniform(0.8, 1.25, size=(len(theta), n))
    if t0:
        th[2] = rng.uniform(1.0, 8.0, n)
    return th


def _generate(dp, hmm, n, thetas, max_traj=196000, key0=9000):
    pt = dp.MbpParticles(dp.device_model(hmm), n, max_traj, seed=5)
    for obs_i in range(1, len(hmm.obs_data) + 1):
        pt.set_stream_key(key0 + obs_i)
        pt.iterate(thetas, obs_i, fresh=(obs_i == 1))
    return pt


def _oracle_state(pt, n, cap):
    st = [pt.get_particle(p + 1) for p in range(n)]
    t = np.zeros((n, cap)); y = np.zeros((n, cap), dtype=np.int32); ln = np.zeros(n, dtype=np.int64)
    for p, (fc, times, types, ll) in enumerate(st):
        ln[p] = len(times); t[p, : ln[p]] = times; y[p, : ln[p]] = types
    return t, y, ln


@pytest.mark.parametrize("case", CASES)
def test_loglike_matches_oracle(dp, dao, case):
    model, y, hmm, theta = _case(dp, case)
    dm = dp.device_model(hmm)
    desc = dm.compiled.desc
    n = 48
    rng = np.random.default_rng(11)
    thetas = _thetas(theta, n, rng, case == "sis_t0")
    pt = _generate(dp, hmm, n, thetas)
    t, ty, ln = _oracle_state(pt, n, 8192)
    for th in (thetas, thetas * rng.uniform(0.9, 1.1, size=thetas.shape)):
        got = pt.da_loglike(th)
        for p in range(n):
            want, _ = dao.da_loglike(desc, th[:, p], t[p, : ln[p]], ty[p, : ln[p]])
            assert rel_close(got[p], want), (case, p, got[p], want)
        assert np.isfinite(got[:, 0]).any()
    # the store is not written
    assert all(len(pt.get_particle(p + 1)[1]) == ln[p] for p in (0, n - 1))


def _step_against_oracle(dp, dao, pt, desc, n, theta_cur, theta_f, kind, traj_props, mvp, key, max_traj=196000, offset=0):
    t, ty, ln = _oracle_state(pt, n, 8192)
    pt.set_stream_key(key)
    ll2, acc = pt.da_step(theta_cur, theta_f, kind, traj_props, mvp)
    for p in range(n):
        fc, times, types, ll = pt.get_particle(p + 1)
        if kind[p] == 1:
            o_len, o_fc, o_ll, o_acc = dao.da_props(desc, theta_cur[:, p], t[p], ty[p], ln[p], max_traj, traj_props, mvp, key, offset + p)
            assert len(times) == o_len and np.array_equal(types, ty[p, :o_len]) and np.array_equal(times, t[p, :o_len]), p
            assert np.array_equal(fc, o_fc) and np.array_equal(acc[p], o_acc), (p, acc[p], o_acc)
            assert rel_close(ll2[p], o_ll) and rel_close(ll, o_ll), (p, ll2[p], o_ll)
        else:
            assert len(times) == ln[p] and np.array_equal(times, t[p, : ln[p]]) and not acc[p].any()
            if kind[p] == 0:
                assert rel_close(ll2[p], dao.da_loglike(desc, theta_f[:, p], t[p, : ln[p]], ty[p, : ln[p]])[0])
            else:
                assert np.all(np.isneginf(ll2[p]))
    return acc


@pytest.mark.parametrize("case", CASES)
def test_step_matches_oracle(dp, dao, case):
    model, y, hmm, theta = _case(dp, case)
    dm = dp.device_model(hmm)
    desc = dm.compiled.desc
    n = 64
    rng = np.random.default_rng(12)
    thetas = _thetas(theta, n, rng, case == "sis_t0")
    pt = _generate(dp, hmm, n, thetas)
    pt.set_batch_offset(100)
    total = np.zeros(3, dtype=np.int64)
    for s, (traj_props, mvp) in enumerate(((1, 3), (8, 3), (6, 1), (6, 2), (5, 4))):
        kind = rng.choice([0, 1, 1, 2], size=n).astype(np.uint8)
        theta_f = thetas * rng.uniform(0.95, 1.05, size=thetas.shape)
        total += _step_against_oracle(dp, dao, pt, desc, n, thetas, theta_f, kind, traj_props, mvp, 4000 + s, offset=100).sum(axis=0)
    assert np.all(total > 0), total  # inserts, deletes and moves were accepted


def test_driver_matches_oracle_store(dp, dao):
    from fake_da import OracleDa
    for case, prior_hi in (("sis_pooley", [0.01, 0.5]), ("sis_t0", [0.01, 0.5, 10.0]), ("poisson", [0.01, 0.5, 0.9])):
        model, y, hmm, theta = _case(dp, case)
        y = y[:12]
        model.prior = dp.UniformProduct([0.0, 0.0] + ([0.3] if case == "poisson" else [0.0] * (len(prior_hi) - 2)), prior_hi)
        hmm = dp.get_private_model(model, y)
        cm = dp.compile_model(model, y)
        mk = lambda n, sd: OracleDa(cm.desc, [o.time for o in y], hmm.t0_index, n, 4096, sd)
        th0 = theta[:, None] * np.random.default_rng(2).uniform(0.9, 1.1, size=(len(theta), 4))
        a = dp.run_std_mcmc(hmm, th0, 200, 60, traj_props=4, seed=31, verbose=False)
        b = dp.run_std_mcmc(hmm, th0, 200, 60, traj_props=4, seed=31, particles_factory=mk, verbose=False)
        assert np.allclose(a.samples.theta, b.samples.theta, rtol=1e-9, atol=0), case
        assert np.array_equal(a.a_cnt, b.a_cnt) and np.array_equal(a.traj_acc, b.traj_acc), case
        assert a.a_cnt[:, 1].sum() > 0 and a.traj_acc.sum() > 0


YS_DEATH = [38, 30, 23, 17, 14]


def _death_posterior(dp, nodes=1201):
    """One-parameter pure-death model (rate theta * I, prior U(0, 0.2)) with Poisson(0.8 I) observations of YS_DEATH, the
    exact likelihood on a grid and the posterior mean by quadrature."""
    from scipy import stats

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


def test_death_posterior_against_quadrature(dp):
    model, y, mean, sd = _death_posterior(dp)
    hmm = dp.get_private_model(model, y)
    th0 = np.random.default_rng(8).uniform(0.03, 0.07, size=(1, 64))
    r = dp.run_std_mcmc(hmm, th0, 4000, 1000, traj_props=8, seed=5, verbose=False)
    post = r.samples.theta[0, 1000:, :].ravel()
    assert abs(post.mean() - mean) < 0.25 * sd, (post.mean(), mean, sd)


def test_sir_posterior_agrees_with_mbp_mcmc(dp):
    """A small two-parameter SIR (30 individuals, Poisson reports): DA-MCMC and MBP-MCMC posterior means agree within their
    Monte Carlo error (chains are independent, so the error is the spread of the per-chain means)."""
    rf = lambda o, p, x: (o.__setitem__(0, p[0] * x[0] * x[1]), o.__setitem__(1, p[1] * x[1]))
    model = dp.generate_custom_model("SIR", rf, [29, 1, 0], [[-1, 1, 0], [0, -1, 1]], obs_model=dp.partial_poisson_obs_model(0.7, seq=(2,)),
                                     prior=dp.UniformProduct([0.0, 0.0], [0.1, 1.0]))
    ys = [1, 3, 5, 6, 5, 3, 2, 1]
    y = [dp.Observation(2.0 * (i + 1), 1, 1.0, [0, v, 0]) for i, v in enumerate(ys)]
    hmm = dp.get_private_model(model, y)
    th0 = np.array([0.03, 0.3])[:, None] * np.random.default_rng(3).uniform(0.8, 1.2, size=(2, 64))
    da = dp.run_std_mcmc(hmm, th0, 4000, 1000, traj_props=8, seed=7, verbose=False)
    mb = dp.run_mbp_mcmc(hmm, th0, 4000, 1000, seed=9, verbose=False)
    for j in range(2):
        a = da.samples.theta[j, 1000:, :].mean(axis=0)
        b = mb.samples.theta[j, 1000:, :].mean(axis=0)
        z = (a.mean() - b.mean()) / np.sqrt(a.var(ddof=1) / len(a) + b.var(ddof=1) / len(b))
        assert abs(z) < 4.5, (j, a.mean(), b.mean(), z)


def test_inserts_across_the_stride_match_a_reserved_store(dp, dao):
    """dpomp_da_step widens the stride to the longest trajectory + traj_props before its launch: from trajectories of a few
    hundred events, 512 proposals per chain take the store past the initial stride of 1024 events, and every trajectory,
    state, log-likelihood and accept count equals that of a store that reserved 8192 events from the start."""
    model, y, hmm, theta = load_case(dp, "lotka_c4")
    y = y[:3]
    hmm = dp.get_private_model(model, y)
    n = 32
    th = np.tile(theta[:, None], (1, n)) * np.linspace(0.95, 1.05, n)[None, :]
    res = []
    for reserve in (None, 8192):
        pt = _generate(dp, hmm, n, th)
        if reserve:
            pt.reserve(reserve)
        lens0 = [len(pt.get_particle(p + 1)[1]) for p in range(n)]
        lls, accs = [], []
        for s in range(3):
            pt.set_stream_key(50 + s)
            ll2, acc = pt.da_step(th, th, np.ones(n, dtype=np.uint8), 512, 3 if s else 1)
            lls.append(ll2); accs.append(acc)
        res.append((lens0, [pt.get_particle(p + 1) for p in range(n)], np.array(accs), np.array(lls), pt.capacity()[0]))
    a, b = res
    assert max(a[0]) < 1024 < a[4] and b[4] == 8192, (max(a[0]), a[4])  # the stride grew in dpomp_da_step
    assert np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3]) and a[2].sum() > 0
    for u, v in zip(a[1], b[1]):
        assert all(np.array_equal(x, z) for x, z in zip(u, v))


def test_insert_at_max_traj_is_rejected(dp, dao):
    """max_traj is the hard limit of the store: an insert into a trajectory of max_traj events is rejected, on the device as in
    the oracle (trajectories that reached it while being generated have log-likelihood -Inf and stay at max_traj)."""
    model, y, hmm, theta = load_case(dp, "sis_pooley")
    y = y[:4]
    hmm = dp.get_private_model(model, y)
    desc = dp.device_model(hmm).compiled.desc
    n, max_traj = 48, 64
    th = theta[:, None] * np.random.default_rng(4).uniform(0.8, 1.2, size=(2, n))
    pt = _generate(dp, hmm, n, th, max_traj=max_traj)
    for s in range(20):
        _step_against_oracle(dp, dao, pt, desc, n, th, th, np.ones(n, dtype=np.uint8), 16, 1 if s % 2 else 3, 700 + s,
                             max_traj=max_traj)
    lens = np.array([len(pt.get_particle(p + 1)[1]) for p in range(n)])
    assert lens.max() == max_traj and np.all(lens <= max_traj), lens
