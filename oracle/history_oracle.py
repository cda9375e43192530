"""Per-observation history of the CPU oracle's particle filter.  TEST INFRASTRUCTURE ONLY (the reference for
dpomp_pf_set_history / dpomp_pf_get_filtered_moments / dpomp_pf_sample_paths).

pf_history runs orc_pf_partial (oracle/dpomp_oracle.c) one observation at a time.  Observation t is run twice from the same
input population with the same draws: once on a copy of the model whose last observation is t (so nothing resamples and the
returned population is the simulated states before resampling), and once on the full model (the ancestors and the
population the next observation starts from).  Moments and path backtraces are computed from these outputs in numpy."""
from __future__ import annotations

import numpy as np

from . import oracle as orc


def pf_history(desc, theta, n: int, ymin: int = 1, ymax=None, pop=None, rs_type: int = 1, key: int = 0, filter_id: int = 0,
               mode: int = orc.MODE_LITERAL, tile: int = 1024, items: int = 4, max_events: int = 1 << 20):
    """Observations ymin..ymax (1-based) of one filter.  pop: (n, C) int64 input state for ymin > 1 (updated in place).
    Returns dict(loglik, states[t] (n, C) before resampling, logw[t] (n,), anc[t] (n,) 0-based or None, pop (n, C) after)."""
    ymax = desc.n_obs if ymax is None else ymax
    cur = np.zeros((n, desc.n_compartments), dtype=np.int64) if pop is None else np.asarray(pop, dtype=np.int64).copy()
    last = type(desc).from_buffer_copy(desc)  # same observation arrays, n_obs set per call below
    ll, states, logw, anc = 0.0, [], [], []
    for oi in range(ymin, ymax + 1):
        last.n_obs = oi
        pre = cur.copy()
        _, lw, _, _, _, _ = orc.pf_partial(last, theta, n, pre, oi, oi, rs_type, key, filter_id, mode, tile, items, max_events)
        inc, lw2, a, _, _, _ = orc.pf_partial(desc, theta, n, cur, oi, oi, rs_type, key, filter_id, mode, tile, items, max_events)
        assert np.array_equal(lw, lw2)
        ll += inc
        states.append(pre)
        logw.append(lw)
        resampled = desc.obs_id[oi - 1] > 0 and oi < desc.n_obs
        anc.append(a - 1 if resampled else None)
    if pop is not None:
        pop[...] = cur
    return dict(loglik=ll, states=states, logw=logw, anc=anc, pop=cur)


def weights(h, desc, t: int) -> np.ndarray:
    """normalised weights of observation t (1-based); equal weights without a likelihood"""
    lw = h["logw"][t - 1]
    if desc.obs_id[t - 1] <= 0:
        return np.full(len(lw), 1.0 / len(lw))
    w = np.exp(lw - lw.max())
    return w / w.sum()


def moments(h, desc, t: int):
    """(mean[C], var[C], ess) of observation t: weighted mean, biased second central moment, (sum w)^2 / sum w^2"""
    w = weights(h, desc, t)
    x = h["states"][t - 1].astype(np.float64)
    mean = w @ x
    var = w @ (x - mean) ** 2
    return mean, var, 1.0 / np.sum(w * w)


def path_uniforms(key: int, filter_id: int, t_last: int, n_paths: int) -> np.ndarray:
    """u53 of Philox(key; path, filter, t_last - 1, resample tag 1, block 2) for every path"""
    out = np.empty(n_paths)
    for p in range(n_paths):
        w = orc.philox([p, filter_id, t_last - 1, (1 << 30) | 2], [key & 0xFFFFFFFF, key >> 32])
        out[p] = float(((int(w[0]) << 21) | (int(w[1]) >> 11)) * 2.0 ** -53)
    return out


def backtrace(h, desc, t_last: int, ends) -> np.ndarray:
    """paths [len(ends), t_last, C] from lineage ends (0-based particles of observation t_last)"""
    out = np.empty((len(ends), t_last, desc.n_compartments), dtype=np.int64)
    for p, k in enumerate(ends):
        for t in range(t_last, 0, -1):
            out[p, t - 1] = h["states"][t - 1][k]
            if t > 1 and h["anc"][t - 2] is not None:
                k = h["anc"][t - 2][k]
    return out


def lineage_ends(h, desc, t_last: int, u: np.ndarray) -> np.ndarray:
    """first q with u S < cw_q over the cumulative weights of t_last (floor(u n) without a likelihood).  cw is a sequential
    sum here; the device sums in its scan tree, which differs in the last bits only, so an end differs only for a draw
    within rounding distance of a boundary."""
    lw = h["logw"][t_last - 1]
    n = len(lw)
    if desc.obs_id[t_last - 1] <= 0:
        return np.minimum(np.floor(u * n).astype(np.int64), n - 1)
    w = np.where(np.isneginf(lw), 0.0, np.exp(lw - lw.max()))
    cw = np.cumsum(w)
    return np.minimum(np.searchsorted(cw, u * cw[-1], side="right"), n - 1)
