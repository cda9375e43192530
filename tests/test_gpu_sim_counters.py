"""Event and event-cap counts of the simulate kernel.

The event loop records each parked particle's event count and cap flag in one shared-memory word, and the weight pass sums
those words in 64 bits.  These tests pin the counts at a lowered cap, where many particles are capped, and at the largest
cap the API accepts (2^31 - 1), where an event count fills all 31 bits below the flag:
  * f64 loop: event and overflow counts equal the oracle's, draw for draw;
  * f32 loop: on a pure-death model observed once (no resampling, so the final population is the simulated one), every
    event moves one individual, so the event count is sum(I_0 - I_end) and a particle is capped exactly when I_0 - I_end
    equals the cap.
"""
import numpy as np
import pytest

from conftest import load_case

pytestmark = pytest.mark.gpu

CAP_MAX = (1 << 31) - 1


@pytest.mark.parametrize("cap", [10, CAP_MAX])
@pytest.mark.parametrize("n", [1024, 3000])
def test_f64_loop_counts_match_oracle(dp, orc, cap, n):
    model, y, hmm, theta = load_case(dp, "sis_pooley")  # ~200 events per particle and interval
    pf = dp.ParticleFilter(dp.device_model(hmm), n, 1, 1, seed=3, sim_precision=dp._capi.SIM_F64, max_events=cap)
    tile, items = pf.geometry()
    key = 0x5EED + n + cap
    pf.set_stream_key(key)
    pf.partial(theta, 1, 4)
    o = orc.pf_partial(pf.dmodel.compiled.desc, theta, n, None, 1, 4, 1, key, 0, orc.MODE_DEVICE, tile, items,
                       max_events=cap)
    o_ev, o_ovf = o[3], o[4]
    assert pf.last_event_count() == o_ev
    assert pf.overflow_count() == o_ovf
    assert (o_ovf > 0) == (cap == 10)


def _pure_death_once(dp):
    # SIS with infection rate 0: only deaths I -> S, rate gamma * I; one observation, so the filter never resamples
    model = dp.generate_model("SIS", [40, 60])
    y = [dp.Observation(5.0, 1, 1.0, [0, 47])]
    return dp.get_private_model(model, y), np.array([0.0, 0.05])


@pytest.mark.parametrize("cap", [10, CAP_MAX])
@pytest.mark.parametrize("n", [200, 5000])  # a 256-particle tile; ragged 1024-particle tiles with padding slots
def test_f32_loop_counts_are_the_population_change(dp, cap, n):
    hmm, theta = _pure_death_once(dp)
    pf = dp.ParticleFilter(dp.device_model(hmm), n, 1, 1, seed=11, max_events=cap)
    pf.set_record_ancestors(True)
    pf.partial(theta, 1, 1)
    pop = pf.get_pop(1)
    deaths = 60 - pop[:, 1]
    assert np.all(pop[:, 0] + pop[:, 1] == 100) and np.all(deaths >= 0) and np.all(deaths <= min(cap, 60))
    assert pf.last_event_count() == int(deaths.sum())
    capped = int((deaths == cap).sum())  # 5 time units at rate 0.05 * 60: about 13 deaths expected, most reach 10
    assert pf.overflow_count() == capped
    assert (capped > n // 2) == (cap == 10)
    assert np.isneginf(pf.last_logw()).sum() == capped
