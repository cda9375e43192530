"""CPU tests of the hidden-state history (dpomp_pf_set_history): the C ABI is declared and bound, and the oracle-side
history (oracle/history_oracle.py) that the GPU tests compare against gives the exact filtering means of the pure-death
model and paths that respect its dynamics."""
import os
import re

import numpy as np
import pytest
from scipy import stats

from conftest import ROOT, pure_death_case

NEW_SYMBOLS = ("dpomp_pf_set_history", "dpomp_pf_get_filtered_moments", "dpomp_pf_sample_paths")


def exact_filtering(ys, sigma=2.0, gam=0.05, i0=60, dt=5.0):
    """p(I_t | y_1..t) and p(I_t | y_1..T) of pure_death_case: forward recursion over the 61 states, one backward pass"""
    states = np.arange(i0 + 1)
    trans = np.array([stats.binom.pmf(states, k, np.exp(-gam * dt)) for k in states])
    g = [np.exp(-(v - states) ** 2 / (2 * sigma * sigma)) for v in ys]
    alpha, filt = np.zeros(i0 + 1), []
    alpha[i0] = 1.0
    for gt in g:
        alpha = (alpha @ trans) * gt
        alpha /= alpha.sum()
        filt.append(alpha)
    beta, smooth = np.ones(i0 + 1), [None] * len(ys)
    for t in range(len(ys) - 1, -1, -1):
        s = filt[t] * beta
        smooth[t] = s / s.sum()
        beta = trans @ (g[t] * beta)
        beta /= beta.sum()
    return states, np.array(filt), np.array(smooth)


def test_history_entry_points_are_declared_and_bound(dp):
    header = open(os.path.join(ROOT, "include", "dpomp.h")).read()
    for name in NEW_SYMBOLS:
        assert re.search(r"\bint " + name + r"\(", header), name
        assert name in dp._capi.EXPORTED_SYMBOLS
    assert "#define DPOMP_HISTORY_MOMENTS 1" in header and "#define DPOMP_HISTORY_PATHS 2" in header
    assert (dp._capi.HISTORY_MOMENTS, dp._capi.HISTORY_PATHS) == (1, 2)
    assert callable(dp.get_filtered_states)


def test_history_symbols_are_exported(built_lib):
    for name in NEW_SYMBOLS:
        assert hasattr(built_lib, name)
    assert built_lib.dpomp_version() == 102


def test_exact_smoothing_reference_is_consistent():
    """the backward pass of exact_filtering: the last smoothing marginal equals the last filtering one, and every
    smoothing marginal integrates the one-step transition of the next"""
    _, filt, smooth = exact_filtering([47, 36, 29, 22, 18])
    assert np.allclose(filt[-1], smooth[-1], atol=1e-15)
    assert np.allclose(smooth.sum(axis=1), 1.0)
    assert np.all(np.diff(smooth @ np.arange(61)) < 0)  # the expected population only dies


def test_oracle_filtering_means_match_exact(dp, orc):
    """oracle history of one 40000-particle filter (literal mode): weighted means of I at every observation against the
    exact p(I_t | y_1..t) means, z-test with the ESS-based standard error inflated by 2 for resampling"""
    from oracle import history_oracle as ho

    model, y, hmm, theta, _ = pure_death_case(dp)
    cm = dp.compile_model(model, y)  # owns the observation arrays desc points to
    desc = cm.desc
    n = 40000
    h = ho.pf_history(desc, theta, n, rs_type=1, key=0xC0FFEE)
    states, filt, _ = exact_filtering([47, 36, 29, 22, 18])
    for t in range(1, 6):
        mean, var, ess = ho.moments(h, desc, t)
        ex_mean = filt[t - 1] @ states
        ex_var = filt[t - 1] @ (states - ex_mean) ** 2
        z = (mean[1] - ex_mean) / np.sqrt(2.0 * ex_var / ess)
        assert abs(z) < 4.5, (t, mean[1], ex_mean, z)
        assert mean[0] + mean[1] == pytest.approx(100.0, abs=1e-9)


def test_oracle_paths_follow_the_dynamics(dp, orc):
    """backtraced oracle paths: I never increases, S + I stays 100, and the lineage ends follow the weights"""
    from oracle import history_oracle as ho

    model, y, hmm, theta, _ = pure_death_case(dp)
    cm = dp.compile_model(model, y)  # owns the observation arrays desc points to
    desc = cm.desc
    h = ho.pf_history(desc, theta, 2000, rs_type=2, key=7)
    u = ho.path_uniforms(0x1234, 0, 5, 300)
    assert np.all((u >= 0) & (u < 1))
    ends = ho.lineage_ends(h, desc, 5, u)
    paths = ho.backtrace(h, desc, 5, ends)
    assert paths.shape == (300, 5, 2)
    assert np.all(np.diff(paths[:, :, 1], axis=1) <= 0)
    assert np.all(paths.sum(axis=2) == 100)
    for p, k in enumerate(ends):
        assert np.array_equal(paths[p, -1], h["states"][-1][k])
