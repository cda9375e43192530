"""CPU tests of data-augmented MCMC (run_std_mcmc, dpomp_da_loglike / dpomp_da_step): the oracle's full log-likelihood against
an independent numpy restatement, the oracle's insert / delete / move chain against an exact posterior, and the host driver
on the oracle-backed store (tests/fake_da.py) sharded over two gloo ranks."""
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp
from scipy import stats

from conftest import GOLDEN, ROOT


@pytest.fixture(scope="module")
def dao():
    from oracle import da_oracle

    da_oracle.build()
    return da_oracle


def full_loglike(rates, trans, ic, theta, t0, obs, log_g, times, types):
    """compute_full_log_like! restated from the law in include/dpomp.h; obs = [(time, obs_id)], log_g(i, x)."""
    x = np.array(ic, dtype=np.int64)
    t, ll, llo, k = t0, 0.0, 0.0, 0
    if any(tk <= t0 for tk in times):
        return -math.inf, -math.inf, x
    for i, (t_obs, oid) in enumerate(obs):
        while k < len(times) and times[k] <= t_obs:
            lam = rates(theta, x)
            e = types[k] - 1
            if lam[e] <= 0.0:
                return -math.inf, -math.inf, x
            tot = 0.0
            for v in lam:
                tot += v
            ll += math.log(lam[e]) - tot * (times[k] - t)
            x = x + trans[e]
            if (x < 0).any():
                return -math.inf, -math.inf, x
            t = times[k]
            k += 1
        tot = 0.0
        for v in rates(theta, x):
            tot += v
        ll -= tot * (t_obs - t)
        t = t_obs
        if oid > 0:
            g = log_g(i, x)
            ll += g
            llo += g
    if k < len(times):
        return -math.inf, -math.inf, x
    return ll, llo, x


def _gauss(desc, y):
    sigma = desc.obs_sigma
    xm = np.array([desc.obs_xmask[c] for c in range(desc.n_compartments)])
    ym = np.array([desc.obs_ymask[v] for v in range(desc.n_obs_vals)])

    def g(i, x):
        d = int(ym @ np.asarray(y[i].val, dtype=np.int64)) - int(xm @ x)
        return math.log(1.0 / (math.sqrt(2.0 * math.pi) * sigma)) - (d * d) / (2.0 * sigma * sigma)
    return g


def _sim(rates, trans, ic, theta, t0, t_end, rng):
    x, t, times, types = np.array(ic, dtype=np.int64), t0, [], []
    while True:
        lam = np.asarray(rates(theta, x))
        if lam.sum() <= 0:
            return times, types
        t += rng.exponential(1.0 / lam.sum())
        if t > t_end:
            return times, types
        e = rng.choice(len(lam), p=lam / lam.sum())
        x = x + trans[e]
        times.append(t); types.append(e + 1)


def _check(dao, desc, rates, trans, ic, theta, t0, obs, log_g, times, types, rtol=1e-12):
    ll2, fc = dao.da_loglike(desc, theta, np.asarray(times, dtype=np.float64), np.asarray(types, dtype=np.int32))
    want = full_loglike(rates, trans, ic, theta, t0, obs, log_g, list(times), list(types))
    if math.isinf(want[0]):
        assert np.isneginf(ll2[0]) and np.isneginf(ll2[1]), (ll2, want)
        return False
    assert abs(ll2[0] - want[0]) <= rtol * max(1.0, abs(want[0])), (ll2, want)
    assert abs(ll2[1] - want[1]) <= rtol * max(1.0, abs(want[1])), (ll2, want)
    assert np.array_equal(fc, want[2])
    return True


def test_full_loglike_matches_numpy_sis(dp, dao):
    model = dp.generate_model("SIS", [100, 1])
    y = dp.get_observations(os.path.join(GOLDEN, "pooley.csv"))
    y = [dp.Observation(o.time, 0 if i in (2, 5) else o.obs_id, o.prop, o.val) for i, o in enumerate(y)]  # obs_id <= 0
    cm = dp.compile_model(model, y)  # owns the observation arrays the descriptor points to
    desc = cm.desc
    trans = np.array(model.m_transition, dtype=np.int64)
    rates = lambda th, x: [th[0] * x[0] * x[1], th[1] * x[1]]
    obs = [(o.time, o.obs_id) for o in y]
    g = _gauss(desc, y)
    rng = np.random.default_rng(1)
    finite = 0
    for r in range(40):
        theta = np.array([0.003, 0.1]) * rng.uniform(0.7, 1.3, 2)
        times, types = _sim(rates, trans, [100, 1], theta, 0.0, y[-1].time, rng)
        if r % 4 == 1 and times:  # an event exactly at an observation time: it belongs to the interval ending there
            j = int(np.searchsorted(times, y[1].time))
            if 0 < j < len(times):
                times[j - 1] = y[1].time
        if r % 4 == 2:  # random edits: zero-rate events, negative compartments, events after T
            for _ in range(3):
                pos = int(rng.integers(0, len(times) + 1))
                times.insert(pos, float(rng.uniform(0, y[-1].time + 5.0)))
                types.insert(pos, int(rng.integers(1, 3)))
            order = np.argsort(times, kind="stable")
            times, types = [times[i] for i in order], [types[i] for i in order]
        finite += _check(dao, desc, rates, trans, [100, 1], theta, 0.0, obs, g, times, types)
    assert finite >= 25
    # a recovery of the only infective, then an infection: the infection has rate 0
    assert not _check(dao, desc, rates, trans, [100, 1], np.array([0.003, 0.1]), 0.0, obs, g, [1.0, 2.0], [2, 1])
    assert _check(dao, desc, rates, trans, [100, 1], np.array([0.003, 0.1]), 0.0, obs, g, [], [])


def test_full_loglike_negative_compartment_and_t0(dp, dao):
    # event 1 is driven by S but removes an I: with I = 0 its rate is positive and the state goes negative
    rf = lambda o, p, x: (o.__setitem__(0, p[0] * x[0]), o.__setitem__(1, p[1] * x[1]), o.__setitem__(2, p[2] * x[1]))
    model = dp.generate_custom_model("X", rf, [5, 1], [[0, -1], [1, -1], [-1, 1]], prior=dp.generate_weak_prior(4), t0_index=4)
    y = [dp.Observation(4.0 * (i + 1), 1, 1.0, [0, v]) for i, v in enumerate([1, 2, 1, 0])]
    cm = dp.compile_model(model, y)  # owns the observation arrays the descriptor points to
    desc = cm.desc
    trans = np.array(model.m_transition, dtype=np.int64)
    rates = lambda th, x: [th[0] * x[0], th[1] * x[1], th[2] * x[1]]
    obs = [(o.time, o.obs_id) for o in y]
    g = _gauss(desc, y)
    theta = np.array([0.05, 0.3, 0.2, 1.0])  # t0 = theta[4] = 1.0
    assert _check(dao, desc, rates, trans, [5, 1], theta, 1.0, obs, g, [1.5, 3.0], [3, 2])
    assert not _check(dao, desc, rates, trans, [5, 1], theta, 1.0, obs, g, [1.5, 3.0], [2, 1])  # I = -1 after event 1
    assert not _check(dao, desc, rates, trans, [5, 1], theta, 1.0, obs, g, [0.5, 3.0], [3, 2])  # before t0
    assert not _check(dao, desc, rates, trans, [5, 1], theta, 1.0, obs, g, [1.0, 3.0], [3, 2])  # at t0
    th2 = theta.copy(); th2[3] = 0.25
    assert _check(dao, desc, rates, trans, [5, 1], th2, 0.25, obs, g, [0.5, 3.0], [3, 2])
    rng = np.random.default_rng(5)
    finite = 0
    for _ in range(30):
        th = theta * rng.uniform(0.7, 1.3, 4)
        times, types = _sim(rates, trans, [5, 1], th, th[3], y[-1].time, rng)
        finite += _check(dao, desc, rates, trans, [5, 1], th, th[3], obs, g, times, types)
    assert finite > 0


def test_full_loglike_poisson_observations(dp, dao):
    rf = lambda o, p, x: (o.__setitem__(0, p[0] * x[0] * x[1]), o.__setitem__(1, p[1] * x[1]))
    model = dp.generate_custom_model("SIS", rf, [100, 1], [[-1, 1], [1, -1]], obs_model=dp.partial_poisson_obs_model(0.6))
    y = dp.get_observations(os.path.join(GOLDEN, "pooley.csv"))
    y = [dp.Observation(o.time, o.obs_id, o.prop, np.floor(0.6 * np.asarray(o.val)).astype(np.int64)) for o in y]
    cm = dp.compile_model(model, y)  # owns the observation arrays the descriptor points to
    desc = cm.desc
    trans = np.array(model.m_transition, dtype=np.int64)
    rates = lambda th, x: [th[0] * x[0] * x[1], th[1] * x[1]]
    g = lambda i, x: float(stats.poisson.logpmf(int(y[i].val[1]), 0.6 * x[1]))
    rng = np.random.default_rng(2)
    for _ in range(10):
        th = np.array([0.003, 0.1]) * rng.uniform(0.8, 1.2, 2)
        times, types = _sim(rates, trans, [100, 1], th, 0.0, y[-1].time, rng)
        _check(dao, desc, rates, trans, [100, 1], th, 0.0, [(o.time, o.obs_id) for o in y], g, times, types, rtol=1e-11)


YS_DEATH = [38, 30, 23, 17, 14]


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


def _oracle_store(dp, model, y, cap=4096, max_traj=196000):
    from fake_da import OracleDa

    hmm = dp.get_private_model(model, y)
    cm = dp.compile_model(model, y)
    return hmm, lambda n, sd: OracleDa(cm.desc, [o.time for o in y], hmm.t0_index, n, cap, sd, max_traj)


def test_oracle_da_chain_matches_quadrature_posterior(dp, dao):
    model, y, mean, sd = _death_posterior(dp)
    hmm, mk = _oracle_store(dp, model, y)
    th0 = np.random.default_rng(8).uniform(0.03, 0.07, size=(1, 4))
    r = dp.run_std_mcmc(hmm, th0, 6000, 1000, seed=5, traj_props=8, particles_factory=mk, verbose=False)
    post = r.samples.theta[0, 1000:, :].ravel()
    assert abs(post.mean() - mean) < 0.25 * sd, (post.mean(), mean, sd)
    assert np.all(r.traj_acc > 0) and np.all(r.a_cnt[:, 1] > 0)


def test_insert_at_max_traj_is_rejected(dp, dao):
    model, y, mean, sd = _death_posterior(dp)
    cm = dp.compile_model(model, y)  # owns the observation arrays the descriptor points to
    desc = cm.desc
    theta = np.array([0.06])
    t = np.zeros(80); ty = np.zeros(80, dtype=np.int32)
    t[:3] = [1.0, 2.0, 3.0]; ty[:3] = 1
    for key in range(40):  # mvp = 1: every proposal is an insert
        n, fc, ll, acc = dao.da_props(desc, theta, t.copy(), ty.copy(), 3, 3, 4, 1, key, 0)
        assert n == 3 and acc.sum() == 0
    grown = sum(dao.da_props(desc, theta, t.copy(), ty.copy(), 3, 4, 4, 1, key, 0)[3][0] for key in range(40))
    assert grown > 0


def _da_worker(rank, world, port, out_path):
    import sys
    sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
    import dpomp_b200 as dp
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    comm = None
    if world > 1:
        torch.distributed.init_process_group("gloo", rank=rank, world_size=world)
        comm = dp.Comm()
    model = dp.generate_model("SIS", [100, 1])
    model.prior = dp.UniformProduct([0, 0], [0.01, 0.5])
    y = dp.get_observations(os.path.join(ROOT, "tests", "golden", "pooley.csv"))[:6]
    hmm, mk = _oracle_store(dp, model, y)
    theta0 = model.prior.rand(5, np.random.default_rng(4)) * 0.5 + np.array([[0.002], [0.05]])
    res = dp.run_std_mcmc(hmm, theta0, 80, 30, seed=8, traj_props=3, comm=comm, particles_factory=mk, verbose=False)
    if rank == 0:
        np.savez(out_path, theta=res.samples.theta, acc=res.a_cnt, tacc=res.traj_acc)
    if world > 1:
        torch.distributed.destroy_process_group()


def test_world_size_2_gloo_matches_single_process(tmp_path):
    one = str(tmp_path / "one.npz"); two = str(tmp_path / "two.npz")
    _da_worker(0, 1, 0, one)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]
    mp.spawn(_da_worker, args=(2, port, two), nprocs=2, join=True)
    a, b = np.load(one), np.load(two)
    for k in a.files:
        assert np.array_equal(a[k], b[k]), k
    assert a["tacc"].sum() > 0


def test_run_mcmc_analysis_without_mbp_still_raises(dp):
    model = dp.generate_model("SIS", [100, 1])
    y = dp.get_observations(os.path.join(GOLDEN, "pooley.csv"))
    with pytest.raises(NotImplementedError, match="run_std_mcmc"):
        dp.run_mcmc_analysis(model, y, mbp=False)
