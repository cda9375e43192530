"""GPU tests of every compiled model instantiation against the oracle.

The filter's event loop, the MBP walks and the DA walks are compiled once per model structure: the seven predefined
density-dependent models (dpomp_models.cuh Builtin<ID>, recognised by kernel_model_id in pf_kernels.cu) and the generic
rate table on each (compartments, events) shape of DPOMP_SIM_SHAPES (pf_sim.cuh).  Each instantiation is a kernel of its own
that can be wrong on its own, and the oracle only evaluates the run-time table, so every one of them is put next to the oracle
here on identical Philox draws.

The case lists below are module constants (importing this file needs no GPU): tests/test_model_matrix_cpu.py parses the
instantiation lists of csrc/ and fails when an instantiation has no case here, and checks that every generic case lands on
the shape it is meant for.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

POISSON, BINOMIAL, NEGBIN = 1, 2, 3
BUILTIN_IDS = {"SI": 1, "SIR": 2, "SIS": 3, "SEI": 4, "SEIR": 5, "SEIS": 6, "LOTKA": 7}
OBS_TIMES = (1.0, 2.0, 3.5, 5.0)

# predefined models (generate_model, density dependent): initial condition, theta, Gaussian observations of the compartment
# generate_model observes (I; the prey of LOTKA), taken from one oracle trajectory so that the weights are not degenerate
PREDEFINED = {
    "SI": ([50, 1], [0.02], (4, 8, 20, 38)),
    "SIR": ([100, 3, 0], [0.004, 0.2], (9, 7, 12, 12)),
    "SIS": ([100, 2], [0.004, 0.15], (7, 4, 7, 8)),
    "SEI": ([80, 0, 2], [0.01, 0.4], (3, 6, 12, 22)),
    "SEIR": ([100, 0, 2, 0], [0.006, 0.5, 0.2], (2, 1, 2, 3)),
    "SEIS": ([60, 0, 3], [0.01, 0.5, 0.3], (6, 3, 3, 4)),
    "LOTKA": ([70, 70], [0.5, 0.0025, 0.3], (114, 142, 237, 320)),
}


# ---- custom models of the generic rate-table kernels, one (or more) per instantiated shape ------------------------------
def _rf_2x1(o, p, x):  # infection with a background source: L2 = x_I + 1 (k2 = 1)
    o[0] = p[0] * x[0] * (x[1] + 1)


def _rf_2x2(o, p, x):  # SIS whose recovery rate is 20 theta_1: one parameter drives both events, f1 coefficient 20
    o[0] = p[0] * x[0] * x[1]
    o[1] = 20 * p[0] * x[1]


def _rf_2x3(o, p, x):  # predator-prey with prey immigration: L1 = x_prey + 1 (k1 = 1)
    o[0] = p[0] * (x[1] + 1)
    o[1] = p[1] * x[0] * x[1]
    o[2] = p[2] * x[0]


def _rf_3x1(o, p, x):  # SI with a cumulative-incidence counter: one event, padded onto (3, 2)
    o[0] = p[0] * x[0] * x[1]


def _rf_3x2(o, p, x):  # S -> E with pressure from I plus 2 (k2 = 2), E -> I: SEI's structure with a constant
    o[0] = p[0] * x[0] * (x[2] + 2)
    o[1] = p[1] * x[1]


def _rf_3x3(o, p, x):  # SIRS with S -> I at theta_1 S / (I + R): the denominator is 0 (rate 0) once I = R = 0 with S > 0
    o[0] = p[0] * x[0] / (x[1] + x[2])
    o[1] = p[1] * x[1]
    o[2] = p[2] * x[2]


def _rf_4x3(o, p, x):  # SEIR whose E -> I and I -> R share theta_2
    o[0] = p[0] * x[0] * x[2]
    o[1] = p[1] * x[1]
    o[2] = p[1] * x[2]


def _rf_4x5(o, p, x):  # SEIRS with vaccination S -> R: five events, padded onto (4, 6)
    o[0] = p[0] * x[0] * x[2]
    o[1] = p[1] * x[1]
    o[2] = p[2] * x[2]
    o[3] = p[3] * x[3]
    o[4] = p[4] * x[0]


def _rf_5x5(o, p, x):  # two strains and a cumulative-incidence counter: padded onto (8, 8)
    o[0] = p[0] * x[0] * x[1]
    o[1] = p[1] * x[0] * x[2]
    o[2] = p[2] * x[1]
    o[3] = p[2] * x[2]
    o[4] = p[3] * x[3]


def _rf_8x8(o, p, x):  # S E1 E2 I1 I2 R V D: Erlang latency, two infectious stages, waning, vaccination, death
    o[0] = p[0] * x[0] * (x[3] + x[4])
    o[1] = p[1] * x[1]
    o[2] = p[1] * x[2]
    o[3] = p[2] * x[3]
    o[4] = p[3] * x[4]
    o[5] = p[4] * x[5]
    o[6] = p[5] * x[0] * (x[6] + 1)
    o[7] = p[6] * x[3]


def _rows(c, moves):
    """transition rows from (from, to) compartment pairs; -1 = none, extra = further +1 entries"""
    out = []
    for mv in moves:
        r = [0] * c
        src, dst = mv[0], mv[1]
        if src >= 0:
            r[src] -= 1
        if dst >= 0:
            r[dst] += 1
        for extra in mv[2:]:
            r[extra] += 1
        out.append(r)
    return out


# name: (rate function, transition rows, initial condition, theta, observed compartment (1-based), observed values, the
# (compartments, events) shape of DPOMP_SIM_SHAPES the model runs on: the first with c <= CC and e <= EE)
GENERIC = {
    "gen_2x1": (_rf_2x1, _rows(2, [(0, 1)]), [40, 0], [0.01], 2, (2, 4, 6, 11), (2, 1)),
    "gen_2x2": (_rf_2x2, _rows(2, [(0, 1), (1, 0)]), [100, 2], [0.005], 2, (7, 7, 13, 22), (2, 2)),
    "gen_2x3": (_rf_2x3, _rows(2, [(-1, 1), (1, 0), (0, -1)]), [30, 40], [0.4, 0.004, 0.3], 2, (69, 82, 136, 173), (2, 3)),
    "gen_3x1_pad": (_rf_3x1, _rows(3, [(0, 1, 2)]), [30, 1, 0], [0.03], 3, (3, 6, 13, 22), (3, 2)),
    "gen_3x2": (_rf_3x2, _rows(3, [(0, 1), (1, 2)]), [40, 0, 0], [0.01, 0.5], 3, (1, 4, 4, 8), (3, 2)),
    "gen_3x3": (_rf_3x3, _rows(3, [(0, 1), (1, 2), (2, 0)]), [30, 1, 0], [0.05, 0.6, 0.5], 2, (2, 2, 2, 1), (3, 3)),
    "gen_4x3": (_rf_4x3, _rows(4, [(0, 1), (1, 2), (2, 3)]), [100, 0, 2, 0], [0.006, 0.3], 3, (2, 1, 2, 3), (4, 3)),
    "gen_4x5_pad": (_rf_4x5, _rows(4, [(0, 1), (1, 2), (2, 3), (3, 0), (0, 3)]), [80, 0, 3, 0], [0.01, 0.5, 0.3, 0.2, 0.05], 3,
                    (4, 3, 3, 3), (4, 6)),
    "gen_5x5_pad": (_rf_5x5, _rows(5, [(0, 1, 4), (0, 2, 4), (1, 3), (2, 3), (3, 0)]), [50, 1, 1, 0, 0], [0.01, 0.008, 0.3, 0.1],
                    5, (7, 7, 13, 18), (8, 8)),
    "gen_8x8": (_rf_8x8, _rows(8, [(0, 1), (1, 2), (2, 3), (3, 4), (4, 5), (5, 0), (0, 6), (3, 7)]), [60, 0, 0, 3, 0, 0, 0, 0],
                [0.01, 0.8, 0.5, 0.3, 0.2, 0.002, 0.05], 4, (3, 2, 4, 3), (8, 8)),
}

CASES = list(PREDEFINED) + list(GENERIC)
# the predefined models the filter variants are checked on, and the generic cases (plain and fused kernels only)
FILTER_VARIANT_MODELS = list(PREDEFINED)
# count families: Poisson on every generic case (every shape), binomial and negative binomial on (3, 3) and (8, 8)
COUNT_CASES = ([(g, POISSON) for g in GENERIC] + [(g, f) for g in ("gen_3x3", "gen_8x8") for f in (BINOMIAL, NEGBIN)])
# the trajectory walks: every predefined-model instantiation and the generic one on the (3, 3) and (8, 8) models
MBP_MODELS = list(PREDEFINED) + ["gen_3x3", "gen_8x8"]
DA_MODELS = list(PREDEFINED) + ["gen_3x3", "gen_8x8"]


def build_case(dp, name, family=0):
    """(model, observations, theta) of a case; family > 0 observes the same compartment through a count family (reported
    fraction 0.7, negative-binomial size 4) with the observed values scaled by 0.7."""
    if name in PREDEFINED:
        ic, theta, vals = PREDEFINED[name]
        model = dp.generate_model(name, ic)
        obs_c = 3 if name in ("SEI", "SEIR", "SEIS") else 2
        n_c = len(ic)
    else:
        rf, rows, ic, theta, obs_c, vals, _ = GENERIC[name]
        n_c = len(ic)
        om = None if family else dp.partial_gaussian_obs_model(2.0, seq=(obs_c,))
        if family == POISSON:
            om = dp.partial_poisson_obs_model(0.7, seq=(obs_c,))
        elif family == BINOMIAL:
            om = dp.partial_binomial_obs_model(0.7, seq=(obs_c,))
        elif family == NEGBIN:
            om = dp.partial_negbin_obs_model(0.7, 4.0, seq=(obs_c,))
        model = dp.generate_custom_model(name.upper(), rf, ic, rows, obs_model=om, prior=dp.generate_weak_prior(len(theta)))
    if family:
        vals = [int(np.floor(0.7 * v)) for v in vals]
    y = []
    for t, v in zip(OBS_TIMES, vals):
        val = [0] * n_c
        val[obs_c - 1] = v
        y.append(dp.Observation(t, 1, 1.0, val))
    return model, y, np.asarray(theta, dtype=np.float64)


def builtin_id(dp, dm):
    import ctypes as C

    out = C.c_int32(-1)
    dp._capi.check(dp._capi.lib().dpomp_model_builtin_id(dm.handle, C.byref(out)))
    return int(out.value)


def _device_model(dp, name, family=0):
    """the device model of a case, after asserting which instantiation it runs on"""
    model, y, theta = build_case(dp, name, family)
    dm = dp.device_model(dp.get_private_model(model, y))
    want = BUILTIN_IDS.get(name, 0) if not family else 0
    assert builtin_id(dp, dm) == want, (name, family)
    if name in GENERIC:
        d = dm.compiled.desc
        assert (d.n_compartments, d.n_events) == (len(GENERIC[name][2]), len(GENERIC[name][1]))
    return model, y, dm, theta


@pytest.fixture(scope="module")
def corc():
    from oracle import count_oracle

    count_oracle.build()
    return count_oracle


@pytest.fixture(scope="module")
def dao():
    from oracle import da_oracle

    da_oracle.build()
    return da_oracle


def _pf(dp, dm, n, nb=1, rs=1, seed=1, f64=False):
    pf = dp.ParticleFilter(dm, n, nb, rs, seed=seed, sim_precision=dp._capi.SIM_F64 if f64 else dp._capi.SIM_F32)
    pf.set_record_ancestors(True)
    return pf


def rel_close(got, want, rtol):
    got, want = np.asarray(got, dtype=float), np.asarray(want, dtype=float)
    fin = np.isfinite(want)
    if not np.array_equal(fin, np.isfinite(got)) or not np.array_equal(got[~fin], want[~fin]):
        return False
    return bool(np.all(np.abs(got[fin] - want[fin]) <= rtol * np.maximum(np.abs(want[fin]), 1.0)))


# ---- 1. f64 event loop, draw for draw ---------------------------------------------------------------------------------
@pytest.mark.parametrize("rs_type", [1, 2])
@pytest.mark.parametrize("case", CASES)
def test_f64_loop_is_bit_exact_against_oracle(dp, orc, case, rs_type):
    """n = 200 (one 256-particle tile) and 3000 (ragged 1024-particle tiles); observations 1..3 of 4, so that the last one
    evaluated resamples and its ancestors are defined."""
    model, y, dm, theta = _device_model(dp, case)
    ymax = len(y) - 1
    for n in (200, 3000):
        pf = _pf(dp, dm, n, rs=rs_type, f64=True)
        tile, items = pf.geometry()
        key = 0x3A7000 + n + 17 * rs_type
        pf.set_stream_key(key)
        ll = pf.partial(theta, 1, ymax)[0]
        o_ll, o_lw, o_anc, o_ev, o_ovf, o_pop = orc.pf_partial(dm.compiled.desc, theta, n, None, 1, ymax, rs_type, key, 0,
                                                               orc.MODE_DEVICE, tile, items)
        ctx = (case, rs_type, n)
        assert o_ev > 0 and o_ovf == 0, ctx
        assert pf.last_event_count() == o_ev, ctx
        assert np.array_equal(pf.last_logw(), o_lw), ctx
        assert np.array_equal(pf.last_ancestors(), o_anc), ctx
        assert np.array_equal(pf.get_pop(1), o_pop), ctx
        assert abs(ll - o_ll) <= 1e-12 * max(1.0, abs(o_ll)), (ctx, ll, o_ll)
        assert np.isfinite(o_ll) and len(np.unique(o_anc)) > n // 20, ctx  # the weights are not degenerate


# ---- 2. f32 event loop, per trajectory --------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES)
def test_f32_loop_trajectories_match_oracle(dp, orc, case):
    """Same Philox draws, f32 event loop against the f64 literal oracle over the first observation interval, 2 stream keys x
    4096 trajectories.  A trajectory whose f32 waiting times and event choices never cross a decision boundary of the f64 walk
    ends in the identical state, and its log-weight (f64 from integers) is then identical.

    Threshold: a trajectory of k events takes k event choices and k waiting times in f32.  Each choice is off by a few f32 ulps
    (~1e-7 relative) against gaps of order one, so it flips with probability ~1e-6 per event; the accumulated time is off by
    ~1e-7 k^0.5 of the interval, which moves the last event across the observation time with probability ~1e-7 k^1.5.  At
    k <= 200 both stay below 5e-4; the bar 1 - (1e-3 + 1e-5 k) leaves an order of magnitude for the sample of 8192, and a
    wrong rate, transition row or state in one kernel moves almost every trajectory with an event, far past it."""
    model, y, dm, theta = _device_model(dp, case)
    n, keys = 4096, (51001, 51002)
    f64 = _pf(dp, dm, n, f64=True)
    f64.set_stream_key(keys[0])
    f64.partial(theta, 1, 1)
    k = f64.last_event_count() / n  # events per trajectory in the interval
    assert k > 0.3, (case, k)
    min_same = 1.0 - (1e-3 + 1e-5 * k)
    same_all, lw_all, ref_all = [], [], []
    for key in keys:
        pf = _pf(dp, dm, n)
        pf.set_stream_key(key)
        pf.partial(theta, 1, 1)
        o = orc.pf_partial(dm.compiled.desc, theta, n, None, 1, 1, 1, key, 0, orc.MODE_LITERAL)
        lw = pf.last_logw()
        same_all.append(lw == o[1]); lw_all.append(lw); ref_all.append(o[1])
    same, lw, ref = np.concatenate(same_all), np.concatenate(lw_all), np.concatenate(ref_all)
    print(f"{case}: {k:.1f} events per trajectory, {same.mean():.5f} of {same.size} f32 trajectories identical to the oracle")
    assert same.mean() > min_same, (case, k, same.mean(), min_same)
    fin = same & np.isfinite(ref)
    assert np.all(np.abs(lw[fin] - ref[fin]) <= 1e-6 * np.abs(ref[fin]))
    both = np.isfinite(lw) & np.isfinite(ref)
    assert both.mean() > 0.999
    w_gpu, w_ref = np.exp(lw[both] - ref[both].max()), np.exp(ref[both] - ref[both].max())
    assert abs(np.log(w_gpu.mean()) - np.log(w_ref.mean())) < 5.0 / np.sqrt(both.sum())


# ---- 3. variants of the predefined-model kernels: bit-identical to the plain chain --------------------------------------
def _run(pf, thetas, nb, ymax, key=555):
    pf.set_stream_key(key)
    ll = pf.partial(thetas, 1, ymax)
    return ll, [pf.get_pop(b + 1) for b in range(nb)], pf.last_ancestors(nb), pf.last_event_count(), pf.last_timing()[1]


def _same(a, b):
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[2], b[2]) and a[3] == b[3]
    assert all(np.array_equal(u, v) for u, v in zip(a[1], b[1]))


@pytest.mark.parametrize("case", FILTER_VARIANT_MODELS)
def test_two_per_lane_large_tiles_equal_one_per_lane(dp, case, monkeypatch):
    model, y, dm, theta = _device_model(dp, case)
    nb, n = 3, 3000
    thetas = theta[:, None] * np.linspace(0.95, 1.05, nb)[None, :]
    out = []
    for knob in ("1", "0"):
        monkeypatch.setenv("DPOMP_TWO_PER_LANE", knob)  # read when the handle is created
        pf = _pf(dp, dm, n, nb, seed=8)
        pf.set_fused(0)
        out.append(_run(pf, thetas, nb, len(y) - 1))
    _same(*out)


@pytest.mark.parametrize("case", FILTER_VARIANT_MODELS)
def test_latency_small_tiles_equal_throughput_small_tiles(dp, case):
    """200-particle filters: two particles per lane at once in a small launch (the latency regime), one at a time in a batch of
    400 filters; the streams are keyed by (filter, particle, event), so the results are identical."""
    model, y, dm, theta = _device_model(dp, case)
    nb_big = 400
    thetas = theta[:, None] * np.linspace(0.8, 1.2, nb_big)[None, :]
    big = _pf(dp, dm, 200, nb_big, seed=3)
    big.set_stream_key(4242)
    ll_big = big.loglik(thetas)
    ids = np.array([10, 11, 12, 399])
    small = _pf(dp, dm, 200, len(ids), seed=3)
    small.set_filter_ids(ids)
    small.set_stream_key(4242)
    ll_small = small.loglik(thetas[:, ids])
    assert np.all(np.isfinite(ll_big))
    assert np.array_equal(ll_small, ll_big[ids])
    for j, b in enumerate(ids):
        assert np.array_equal(small.get_pop(j + 1), big.get_pop(int(b) + 1))


@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("case", CASES)
def test_fused_step_equals_two_kernel_path(dp, case, f64):
    model, y, dm, theta = _device_model(dp, case)
    nb, n = 3, 3000
    thetas = theta[:, None] * np.linspace(0.9, 1.1, nb)[None, :]
    out = []
    for fused in (2, 0):
        pf = _pf(dp, dm, n, nb, seed=4, f64=f64)
        pf.set_fused(fused)
        out.append(_run(pf, thetas, nb, len(y) - 1))
    _same(*out)
    assert out[0][4] < out[1][4]  # one launch per resampling observation instead of two


@pytest.mark.parametrize("case", FILTER_VARIANT_MODELS)
def test_persistent_kernel_equals_launch_chain(dp, case):
    model, y, dm, theta = _device_model(dp, case)
    nb, n = 3, 3000
    thetas = theta[:, None] * np.linspace(0.9, 1.1, nb)[None, :]
    out = []
    for mode in (2, 0):
        pf = _pf(dp, dm, n, nb, seed=4)
        pf.set_persistent(mode)
        pf.set_fused(0)
        out.append(_run(pf, thetas, nb, len(y) - 1))
        assert pf.overflow_count() == 0
    _same(*out)
    assert out[0][4] == 1 and out[1][4] > 1  # one launch for the whole call


# ---- 4. count observation families on every generic shape ---------------------------------------------------------------
@pytest.mark.parametrize("case,family", COUNT_CASES)
def test_count_family_f64_loop_matches_oracle(dp, corc, case, family):
    model, y, dm, theta = _device_model(dp, case, family)
    ymax = len(y) - 1
    for n in (200, 3000):
        pf = _pf(dp, dm, n, f64=True)
        tile, items = pf.geometry()
        key = 0xC0C0 + n + family
        pf.set_stream_key(key)
        ll = pf.partial(theta, 1, ymax)[0]
        o_ll, o_lw, o_anc, o_ev, o_ovf, o_pop = corc.pf_partial(dm.compiled.desc, theta, n, None, 1, ymax, 1, key, 0,
                                                                corc.MODE_DEVICE, tile, items)
        ctx = (case, family, n)
        assert pf.last_event_count() == o_ev and o_ev > 0, ctx
        assert np.array_equal(pf.get_pop(1), o_pop), ctx
        assert rel_close(pf.last_logw(), o_lw, 1e-13), ctx  # CUDA log / lgamma against glibc
        assert np.array_equal(pf.last_ancestors(), o_anc), ctx
        assert np.isfinite(o_ll) and abs(ll - o_ll) <= 1e-12 * max(1.0, abs(o_ll)), (ctx, ll, o_ll)


# ---- 5. MBP walks --------------------------------------------------------------------------------------------------------
def _thetas(theta, n, rng):
    return theta[:, None] * rng.uniform(0.8, 1.25, size=(len(theta), n))


@pytest.mark.parametrize("mode", [1, 2])  # one thread / one warp per trajectory
@pytest.mark.parametrize("case", MBP_MODELS)
def test_mbp_iterate_and_propose_match_oracle(dp, orc, case, mode):
    """Every particle: event types exact, event times, final states and log-likelihoods to 1e-12."""
    model, y, dm, theta = _device_model(dp, case)
    desc = dm.compiled.desc
    n, cap = 48, 4096
    rng = np.random.default_rng(3)
    thetas = _thetas(theta, n, rng)
    pt = dp.MbpParticles(dm, n, cap, seed=5)
    pt.set_mode(mode)
    o_fc = np.tile(np.asarray(model.initial_condition, dtype=np.int64), (n, 1))
    o_t = np.zeros((n, cap)); o_y = np.zeros((n, cap), dtype=np.int32); o_len = np.zeros(n, dtype=np.int64); o_ll = np.zeros((n, 2))
    for obs_i in range(1, len(y) + 1):
        key = 9300 + obs_i
        pt.set_stream_key(key)
        lg = pt.iterate(thetas, obs_i, fresh=(obs_i == 1))
        for p in range(n):
            t_start = 0.0 if obs_i == 1 else y[obs_i - 2].time
            g, o_len[p] = orc.mbp_iterate(desc, thetas[:, p], o_fc[p], o_t[p], o_y[p], o_len[p], o_ll[p], t_start, obs_i, key, p)
            assert rel_close([lg[p]], [g], 1e-12), (case, p, obs_i, lg[p], g)
    assert o_len.sum() > n and np.isfinite(o_ll[:, 0]).any()
    for p in range(n):
        fc, times, types, ll = pt.get_particle(p + 1)
        assert np.array_equal(fc, o_fc[p]) and len(times) == o_len[p], (case, p)
        assert np.array_equal(types, o_y[p, : o_len[p]]) and rel_close(times, o_t[p, : o_len[p]], 1e-12), (case, p)
        assert rel_close(ll[:1], o_ll[p, :1], 1e-12), (case, p)
    theta_f = thetas * rng.uniform(0.85, 1.2, size=thetas.shape)
    valid = np.ones(n, dtype=bool); valid[3] = False
    pt.set_stream_key(777)
    ll_f = pt.propose(thetas, theta_f, valid, len(y))
    assert np.all(np.isneginf(ll_f[3]))
    for p in np.flatnonzero(valid):
        times, types, fc, ll, rc = orc.mbp_propose(desc, thetas[:, p], theta_f[:, p], o_t[p], o_y[p], o_len[p], cap, len(y), 777, p)
        g_fc, g_times, g_types, g_ll = pt.get_particle(p + 1, proposal=True)
        assert rc == 0 and np.array_equal(g_fc, fc) and np.array_equal(g_types, types), (case, p)
        assert rel_close(g_times, times, 1e-12) and rel_close(g_ll, ll, 1e-12) and rel_close(ll_f[p], ll, 1e-12), (case, p)


# ---- 6. DA walks ---------------------------------------------------------------------------------------------------------
def _generate(dp, dm, n, thetas, n_obs, key0=9000):
    pt = dp.MbpParticles(dm, n, 196000, seed=5)
    for obs_i in range(1, n_obs + 1):
        pt.set_stream_key(key0 + obs_i)
        pt.iterate(thetas, obs_i, fresh=(obs_i == 1))
    return pt


def _oracle_state(pt, n, cap):
    t = np.zeros((n, cap)); ty = np.zeros((n, cap), dtype=np.int32); ln = np.zeros(n, dtype=np.int64)
    for p in range(n):
        fc, times, types, ll = pt.get_particle(p + 1)
        ln[p] = len(times); t[p, : ln[p]] = times; ty[p, : ln[p]] = types
    return t, ty, ln


def _step_against_oracle(dao, pt, desc, n, theta_cur, theta_f, kind, traj_props, mvp, key, offset, max_traj=196000):
    t, ty, ln = _oracle_state(pt, n, 8192)
    pt.set_stream_key(key)
    ll2, acc = pt.da_step(theta_cur, theta_f, kind, traj_props, mvp)
    for p in range(n):
        fc, times, types, ll = pt.get_particle(p + 1)
        if kind[p] == 1:
            o_len, o_fc, o_ll, o_acc = dao.da_props(desc, theta_cur[:, p], t[p], ty[p], ln[p], max_traj, traj_props, mvp, key, offset + p)
            assert len(times) == o_len and np.array_equal(types, ty[p, :o_len]) and np.array_equal(times, t[p, :o_len]), p
            assert np.array_equal(fc, o_fc) and np.array_equal(acc[p], o_acc), (p, acc[p], o_acc)
            assert rel_close(ll2[p], o_ll, 1e-12) and rel_close(ll, o_ll, 1e-12), (p, ll2[p], o_ll)
        else:
            assert len(times) == ln[p] and np.array_equal(times, t[p, : ln[p]]) and not acc[p].any()
            if kind[p] == 0:
                assert rel_close(ll2[p], dao.da_loglike(desc, theta_f[:, p], t[p, : ln[p]], ty[p, : ln[p]])[0], 1e-12)
            else:
                assert np.all(np.isneginf(ll2[p]))
    return acc


@pytest.mark.parametrize("case", DA_MODELS)
def test_da_loglike_and_step_match_oracle(dp, dao, case):
    model, y, dm, theta = _device_model(dp, case)
    desc = dm.compiled.desc
    n = 48
    rng = np.random.default_rng(12)
    thetas = _thetas(theta, n, rng)
    pt = _generate(dp, dm, n, thetas, len(y))
    t, ty, ln = _oracle_state(pt, n, 8192)
    for th in (thetas, thetas * rng.uniform(0.9, 1.1, size=thetas.shape)):
        got = pt.da_loglike(th)
        for p in range(n):
            want, _ = dao.da_loglike(desc, th[:, p], t[p, : ln[p]], ty[p, : ln[p]])
            assert rel_close(got[p], want, 1e-12), (case, p, got[p], want)
        assert np.isfinite(got[:, 0]).any()
    pt.set_batch_offset(100)
    total = np.zeros(3, dtype=np.int64)
    for s, (traj_props, mvp) in enumerate(((1, 3), (8, 3), (6, 1), (6, 2), (5, 4), (12, 3))):
        kind = rng.choice([0, 1, 1, 1, 2], size=n).astype(np.uint8)
        theta_f = thetas * rng.uniform(0.95, 1.05, size=thetas.shape)
        total += _step_against_oracle(dao, pt, desc, n, thetas, theta_f, kind, traj_props, mvp, 4100 + s, 100).sum(axis=0)
    assert np.all(total > 0), (case, total)  # inserts, deletes and moves were accepted
