"""GPU tests of the hidden-state history (dpomp_pf_set_history, dpomp_pf_get_filtered_moments, dpomp_pf_sample_paths,
get_filtered_states, run_pmcmc(state_interval=k)): the filter's results do not change with the history on, the history
equals the oracle's draw for draw, split calls and the invalidating operations behave as documented, and the moments and
paths agree with the exact filtering and smoothing distributions of the pure-death model."""
import numpy as np
import pytest

from conftest import death_rate_case, load_case, pure_death_case
from test_pf_history_cpu import exact_filtering

pytestmark = pytest.mark.gpu

F32, F64 = 0, 1
KEY = 0x5EED_1234_ABCD


def _pf(dp, hmm, n, nb, rs=1, f64=True, seed=3):
    pf = dp.ParticleFilter(dp.device_model(hmm), n, nb, rs, seed=seed, sim_precision=dp._capi.SIM_F64 if f64 else dp._capi.SIM_F32)
    pf.set_record_ancestors(True)
    return pf


def _theta_cols(theta, nb):
    return np.tile(np.asarray(theta, dtype=np.float64)[:, None], (1, nb))


def _death_case_with_skip(dp):
    """pure_death_case with observation 3 carrying obs_id 0 (no likelihood, no resampling)"""
    model, y, _, theta, _ = pure_death_case(dp)
    y = [dp.Observation(o.time, 0 if k == 2 else o.obs_id, o.prop, o.val) for k, o in enumerate(y)]
    return model, y, dp.get_private_model(model, y), theta


def _count_case(dp):
    model = dp.generate_custom_model("SIS", lambda o, p, x: (o.__setitem__(0, p[0] * x[0] * x[1]), o.__setitem__(1, p[1] * x[1])),
                                     [100, 1], [[-1, 1], [1, -1]], obs_model=dp.partial_poisson_obs_model(0.6, seq=(2,)))
    _, y, _, theta = load_case(dp, "sis_pooley")
    y = [dp.Observation(o.time, o.obs_id, o.prop, np.floor(0.6 * np.asarray(o.val)).astype(np.int64)) for o in y]
    return model, y, dp.get_private_model(model, y), theta


# (case, n, nb, rs, f64, scatter, handle option)
IDENTITY_CASES = [
    ("sir_c2", 5000, 3, 1, False, 0, None),
    ("sir_c2", 5000, 3, 2, True, 0, None),
    ("sir_c2", 5000, 3, 3, False, 0, None),
    ("sir_c2", 40000, 2, 1, False, 1, None),
    ("sir_c2", 40000, 2, 2, False, 0, None),
    ("sir_c2", 40000, 2, 3, True, 1, None),
    ("seir_c3", 1000, 4, 1, False, 0, "fused"),
    ("seir_c3", 3000, 4, 1, False, 0, "fused2"),
    ("sir_c2", 3000, 4, 2, False, 0, "persistent"),
    ("sis_pooley", 200, 8, 1, False, 0, "persistent"),
    ("skip", 3000, 3, 1, True, 0, None),
    ("skip", 3000, 3, 3, False, 0, None),
    ("count", 5000, 3, 1, False, 0, None),
    ("count", 5000, 3, 2, True, 0, None),
]


def _case(dp, name):
    if name == "skip":
        return _death_case_with_skip(dp)
    if name == "count":
        return _count_case(dp)
    model, y, hmm, theta = load_case(dp, name)
    return model, y, hmm, theta


@pytest.mark.parametrize("name,n,nb,rs,f64,scatter,opt", IDENTITY_CASES)
def test_results_do_not_change_with_history_on(dp, name, n, nb, rs, f64, scatter, opt):
    _, _, hmm, theta = _case(dp, name)
    th = _theta_cols(theta, nb) * np.linspace(0.9, 1.1, nb)[None, :]
    outs = []
    for flags in (0, 1, 3):
        pf = _pf(dp, hmm, n, nb, rs, f64)
        pf.set_scatter(scatter)
        if opt == "fused":
            pf.set_fused(1)
        elif opt == "fused2":
            pf.set_fused(2)
        elif opt == "persistent":
            pf.set_persistent(2)
        if flags:
            pf.set_history(moments=bool(flags & 1), paths=bool(flags & 2))
        pf.set_stream_key(KEY)
        ll = pf.loglik(th)
        res = dict(ll=ll, ev=pf.last_event_count(), pops=[pf.get_pop(b) for b in range(1, nb + 1)],
                   lw=[pf.last_logw(b) for b in range(1, nb + 1)])
        # a split call: the ancestors of the resampling after observation 1 (every case resamples there unless skipped)
        pf.set_stream_key(KEY)
        pf.partial(th, 1, 1)
        res["anc"] = [pf.last_ancestors(b) for b in range(1, nb + 1)]
        outs.append(res)
    for res in outs[1:]:
        assert np.array_equal(res["ll"], outs[0]["ll"])
        assert res["ev"] == outs[0]["ev"]
        for b in range(nb):
            assert np.array_equal(res["pops"][b], outs[0]["pops"][b])
            assert np.array_equal(res["lw"][b], outs[0]["lw"][b])
            assert np.array_equal(res["anc"][b], outs[0]["anc"][b])


@pytest.mark.parametrize("rs,scatter", [(1, 0), (2, 0), (3, 0), (1, 1)])
def test_history_matches_oracle(dp, orc, rs, scatter):
    """f64 loop, device mode: paths equal a numpy backtrace of the oracle history with the documented draws, moments agree
    with numpy moments of the oracle history to 1e-12 relative"""
    from oracle import history_oracle as ho

    model, y, hmm, theta = load_case(dp, "sir_c2")
    cm = dp.compile_model(model, y)  # owns the observation arrays desc points to
    desc = cm.desc
    n, nb, T, n_paths = 3000, 2, 30, 2000
    pf = _pf(dp, hmm, n, nb, rs, True)
    pf.set_scatter(scatter)
    pf.set_history(moments=True, paths=True)
    pf.set_filter_ids([11, 4])
    tile, items = pf.geometry()
    th = _theta_cols(theta, nb)
    pf.set_stream_key(KEY)
    ll = pf.partial(th, 1, T)
    mean, var, ess = pf.filtered_moments(nb, T)
    paths = pf.sample_paths(n_paths, 0xABC, nb, T)
    mode = orc.MODE_DEVICE_INTERLEAVED if scatter else orc.MODE_DEVICE
    for b, fid in enumerate([11, 4]):
        h = ho.pf_history(desc, theta, n, 1, T, rs_type=rs, key=KEY, filter_id=fid, mode=mode, tile=tile, items=items)
        assert abs(h["loglik"] - ll[b]) <= 1e-9 * abs(ll[b])
        for t in range(1, T + 1):
            m, v, e = ho.moments(h, desc, t)
            np.testing.assert_allclose(mean[b, t - 1], m, rtol=1e-12)
            np.testing.assert_allclose(var[b, t - 1], v, rtol=1e-10, atol=1e-12 * np.abs(m).max() ** 2)
            assert ess[b, t - 1] == pytest.approx(e, rel=1e-12)
        ends = ho.lineage_ends(h, desc, T, ho.path_uniforms(0xABC, fid, T, n_paths))
        want = ho.backtrace(h, desc, T, ends)
        assert np.array_equal(paths[b], want)


def test_split_calls_invalidation_and_arguments(dp):
    _, _, hmm, theta = load_case(dp, "sir_c2")
    n, nb, T = 5000, 2, 40
    th = _theta_cols(theta, nb)
    res = []
    for split in (False, True):
        pf = _pf(dp, hmm, n, nb, 2, False)
        pf.set_history(moments=True, paths=True)
        pf.set_stream_key(KEY)
        if split:
            pf.partial(th, 1, 17)
            with pytest.raises(dp._capi.DpompError) as e:
                pf.filtered_moments(nb, 18)
            assert e.value.code == -4
            pf.set_stream_key(KEY)
            pf.partial(th, 18, T)
        else:
            pf.partial(th, 1, T)
        res.append((pf.filtered_moments(nb, T), pf.sample_paths(64, 9, nb, T)))
    for a, b in zip(res[0][0], res[1][0]):
        assert np.array_equal(a, b)
    assert np.array_equal(res[0][1], res[1][1])

    def err(fn):
        with pytest.raises(dp._capi.DpompError) as e:
            fn()
        return e.value.code

    pf = _pf(dp, hmm, n, nb, 1, False)
    assert err(lambda: pf.filtered_moments(nb, 1)) == -4  # history off
    with pytest.raises(dp._capi.DpompError):
        dp._capi.check(dp._capi.lib().dpomp_pf_set_history(pf._h, 4))
    pf.set_history(moments=True, paths=True)
    assert err(lambda: pf.filtered_moments(nb, 1)) == -4  # nothing recorded yet
    pf.partial(th, 1, 10)
    assert err(lambda: pf.filtered_moments(0, 5)) == -1
    assert err(lambda: pf.filtered_moments(nb + 1, 5)) == -1
    assert err(lambda: pf.filtered_moments(nb, 0)) == -1
    assert err(lambda: pf.filtered_moments(nb, pf.n_obs + 1)) == -1
    assert err(lambda: pf.filtered_moments(nb, 11)) == -4
    assert err(lambda: pf.sample_paths(0, 1, nb, 10)) == -1
    assert err(lambda: pf.sample_paths(4, 1, nb, 9)) == -4  # the weights of 9 are gone
    pf.filtered_moments(nb, 9)
    pf.sample_paths(4, 1, nb, 10)
    pf.partial(th[:, :1], 11, 12)  # one filter only: the history of filter 2 stops at 10
    assert err(lambda: pf.filtered_moments(nb, 12)) == -4
    pf.filtered_moments(1, 12)
    pf.sample_paths(4, 1, 1, 12)

    other = _pf(dp, hmm, n, nb, 1, False)
    other.partial(th, 1, 3)
    ops = {
        "permute": lambda p: p.permute(np.array([2, 1])),
        "copy_filters": lambda p: p.copy_from(other, [1], [2]),
        "set_pop": lambda p: p.set_pop(1, p.get_pop(1)),
        "import": lambda p: p.import_tensor([1], p.export_tensor([2])),
    }
    for name, op in ops.items():
        pf.partial(th, 1, 10)
        pf.filtered_moments(nb, 10)
        op(pf)
        assert err(lambda: pf.filtered_moments(1, 10)) == -4, name
        assert err(lambda: pf.sample_paths(1, 1, 1, 10)) == -4, name


@pytest.mark.parametrize("f64", [False, True])
def test_filtered_means_match_exact_pure_death(dp, f64):
    """32 filters x 2^16 particles: the mean over filters of the filtered mean of I against the exact p(I_t | y_1..t)
    mean, z-test with the standard error estimated from the spread over the filters"""
    model, y, hmm, theta, _ = pure_death_case(dp)
    nb = 32
    fs = dp.get_filtered_states(model, y, _theta_cols(theta, nb), np=1 << 16, seed=11,
                                sim_precision=dp._capi.SIM_F64 if f64 else dp._capi.SIM_F32)
    assert fs.mean.shape == (nb, 5, 2) and fs.var.shape == (nb, 5, 2) and fs.ess.shape == (nb, 5)
    assert fs.paths.shape == (nb, 0, 5, 2) and np.array_equal(fs.time, [5.0, 10.0, 15.0, 20.0, 25.0])
    states, filt, _ = exact_filtering([47, 36, 29, 22, 18])
    est = fs.mean[:, :, 1]
    z = (est.mean(axis=0) - filt @ states) / (est.std(axis=0, ddof=1) / np.sqrt(nb))
    assert np.all(np.abs(z) < 4.5), z
    assert np.allclose(fs.mean.sum(axis=2), 100.0)
    ex_var = filt @ states ** 2 - (filt @ states) ** 2
    assert np.all(np.abs(fs.var[:, :, 1].mean(axis=0) / ex_var - 1) < 0.05)
    assert np.all((fs.ess > 1) & (fs.ess <= 1 << 16))


def test_paths_match_exact_smoothing_pure_death(dp):
    """one path from each of 512 filters: per-observation means of I against the exact p(I_t | y_1..T) means"""
    model, y, hmm, theta, _ = pure_death_case(dp)
    nb = 512
    fs = dp.get_filtered_states(model, y, _theta_cols(theta, nb), np=4096, n_paths=1, seed=5)
    paths = fs.paths[:, 0]
    assert paths.shape == (nb, 5, 2)
    assert np.all(np.diff(paths[:, :, 1], axis=1) <= 0)
    assert np.all(paths.sum(axis=2) == 100)
    states, _, smooth = exact_filtering([47, 36, 29, 22, 18])
    sm_mean = smooth @ states
    sm_sd = np.sqrt(smooth @ states ** 2 - sm_mean ** 2)
    z = (paths[:, :, 1].mean(axis=0) - sm_mean) / (sm_sd / np.sqrt(nb))
    assert np.all(np.abs(z) < 4.5), z
    one = dp.get_filtered_states(model, y, theta, np=1000, n_paths=3, seed=5)  # 1-D theta drops the batch axis
    assert one.mean.shape == (5, 2) and one.paths.shape == (3, 5, 2) and isinstance(one.loglik, float)


def test_pmcmc_states_against_quadrature(dp):
    """death_rate_case: the posterior mean of I_t from MCMCSample.states against quadrature over the grid of the exact
    smoothing means (batch means over the chains); the theta chains are bit-identical with and without states"""
    from scipy import stats

    c = death_rate_case(dp)
    n_chains, steps, adapt = 16, 1500, 300
    init = np.linspace(0.03, 0.08, n_chains)[None, :]
    kw = dict(steps=steps, adapt_period=adapt, p=1000, seed=21, verbose=False)
    plain = dp.run_pmcmc(c["hmm"], init, **kw)
    res = dp.run_pmcmc(c["hmm"], init, state_interval=5, **kw)
    assert np.array_equal(plain.samples.theta, res.samples.theta)
    assert not hasattr(plain, "states")
    n_kept = len(range(adapt, steps, 5))
    assert res.states.shape == (n_chains, n_kept, 5, 2)
    assert np.all(np.diff(res.states[:, :, :, 1], axis=2) <= 0) and np.all(res.states.sum(axis=3) == 100)
    # exact E[I_t | y] = int p(theta | y) E[I_t | theta, y] dtheta on the grid of death_rate_case
    states = np.arange(61)
    ys, sigma = [47, 36, 29, 22, 18], 2.0

    def smooth_mean(gam):
        trans = stats.binom.pmf(states[None, :], states[:, None], np.exp(-gam * 5.0))
        g = [np.exp(-(v - states) ** 2 / (2 * sigma * sigma)) for v in ys]
        alpha, filt = np.zeros(61), []
        alpha[60] = 1.0
        for gt in g:
            alpha = (alpha @ trans) * gt
            alpha /= alpha.sum()
            filt.append(alpha)
        beta, out = np.ones(61), np.zeros(5)
        for t in range(4, -1, -1):
            s = filt[t] * beta
            out[t] = (s / s.sum()) @ states
            beta = trans @ (g[t] * beta)
            beta /= beta.sum()
        return out

    g = c["g"][::10]
    lik = c["lik"][::10]
    sm = np.array([smooth_mean(v) for v in g])
    want = np.trapezoid(lik[:, None] * sm, g, axis=0) / np.trapezoid(lik, g)
    chain_means = res.states[:, :, :, 1].mean(axis=1)  # (chains, T)
    z = (chain_means.mean(axis=0) - want) / (chain_means.std(axis=0, ddof=1) / np.sqrt(n_chains))
    assert np.all(np.abs(z) < 4.5), (z, want, chain_means.mean(axis=0))
