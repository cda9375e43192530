"""Particle MCMC -- the caller of the particle filter specified by run_pmcmc (src/hmm_mcmc.jl:349-365) and the
commented generic_mcmc! (src/hmm_mcmc.jl:166-211) of the reference (dead code there, F7; built here from that
specification because BASELINE config C3 needs it).

Adaptive random-walk Metropolis on theta with target log prior + PF log-likelihood estimate (estimate_likelihood with
systematic resampling).  All chains advance in lock step: one BATCHED dpomp_pf_loglik call evaluates the proposals of
every chain of this rank per MCMC step.  Chains are independent, so they shard over ranks with no communication until
the final gather of the samples.
"""
from __future__ import annotations

import math
import time
from typing import Callable, Optional

import numpy as np

from .distributed import Comm
from .ibis import _M64, splitmix64
from .particle_filter import ParticleFilter, device_model, get_private_model
from .structs import DPOMPModel, HiddenMarkovModel, MCMCSample, RejectionSample

C_INITIAL = 0.1  # proposal scalar (src/hmm_mcmc.jl:7)
C_DF_MCMC_STEPS = 50000  # src/DiscretePOMP.jl:41-42
C_DF_MCMC_ADAPT = 0.2


def handle_rej_samples(theta: np.ndarray, ap: int = 0) -> RejectionSample:
    """handle_rej_samples (src/cmn.jl:8-17): mean and covariance of theta[:, ap+1:end, :] pooled over chains."""
    d = theta.shape[0]
    kept = theta[:, ap:, :].reshape(d, -1)
    mu = kept.mean(axis=1)
    cv = np.atleast_2d(np.cov(kept)) if kept.shape[1] > 1 else np.zeros((d, d))
    return RejectionSample(theta, mu, cv)


def gelman_diagnostic_sre(samples: np.ndarray, discard: int) -> np.ndarray:
    """Point estimate of the scale reduction factor per parameter (the central column of gelman_diagnostic's `sre`,
    src/cmn.jl:20-88, without the F-quantile bounds): sqrt(((n-1)/n W + (1 + 1/m) B/n) / W)."""
    x = samples[:, discard:, :]
    d, n, m = x.shape
    sre = np.full((d, 3), np.nan)
    if m < 2 or n < 2:
        return sre
    means = x.mean(axis=1)
    b = n * means.var(axis=1, ddof=1)
    w = x.var(axis=1, ddof=1).mean(axis=1)
    with np.errstate(divide="ignore", invalid="ignore"):
        sre[:, 1] = np.sqrt(((n - 1) / n * w + (1 + 1 / m) * b / n) / w)
    return sre


def run_pmcmc(model: HiddenMarkovModel, theta_init: np.ndarray, steps: int = 50000, adapt_period: int = 10000,
              p: int = 200, seed: int = 1, comm: Optional[Comm] = None, pf_factory: Optional[Callable] = None,
              verbose: bool = True, state_interval: int = 0) -> MCMCSample:
    """run_pmcmc(model, theta_init, steps = 50000, adapt_period = 10000, p = 200) (src/hmm_mcmc.jl:349-365);
    theta_init is (n_theta, n_chains).  Returns MCMCSample with samples.theta of shape (n_theta, steps, n_chains).

    state_interval = k > 0 also samples the hidden states (particle marginal Metropolis-Hastings, Andrieu, Doucet &
    Holenstein 2010): every filter call draws one state path per chain from its particle genealogy, an accepted chain takes
    its proposal's path, and after the adaptation period the current path of every k-th step is kept in
    MCMCSample.states, shape (n_chains, n_kept, T, C)."""
    comm = comm or Comm(None)
    start_time = time.time_ns()
    theta_init = np.asarray(theta_init, dtype=np.float64)
    d, n_chains = theta_init.shape
    lo, hi = comm.bounds(n_chains)
    n_loc = hi - lo
    if verbose and comm.rank == 0:
        print(f"Running PMCMC analysis: {n_chains} x {steps} samples")
    make = pf_factory or (lambda nb, sd: ParticleFilter(device_model(model), p, nb, 1, seed=sd))
    pf = make(max(n_loc, 1), seed)
    if state_interval > 0:
        pf.set_history(moments=False, paths=True)
        n_obs, n_comp = pf.n_obs, pf.n_comp
        paths = np.zeros((n_loc, n_obs, n_comp), dtype=np.int64)  # path of the last evaluation of every chain slot
        kept = []
    adapt_interval = adapt_period / 10  # ADAPT_INTERVAL = adapt_period / 10 is a Float64 in the reference (:168)
    chains = np.zeros((n_loc, steps, d))
    chol = np.zeros((n_loc, d, d))
    t0s = theta_init[:, lo:hi].T
    chol[:, np.arange(d), np.arange(d)] = np.sqrt(0.1 * np.where(t0s == 0.0, 1.0, t0s * t0s))  # covar[i,i] = 0.1 * theta0[i]^2 (:171-174)
    c = np.full(n_loc, C_INITIAL)
    accepted_total = np.zeros(n_loc, dtype=np.int64)

    from .ibis import prior_logpdf_columns

    timers = {"filter_calls_wall": 0.0, "filter_device_ms": 0.0}  # seconds in the batched C-ABI call / its CUDA-event time
    last_ids = [None]

    def target(thetas: np.ndarray, step: int) -> np.ndarray:
        """model prior + estimate_likelihood(model, theta, p, ps, rsp_systematic) for each local chain (:356-358)."""
        lp = prior_logpdf_columns(model.prior, thetas.T)
        valid = np.nonzero(lp != -np.inf)[0]
        out = np.full(n_loc, -np.inf)
        if len(valid):
            if last_ids[0] is None or not np.array_equal(last_ids[0], valid):  # filter slot j simulates chain lo + valid[j]
                pf.set_filter_ids(lo + valid)
                last_ids[0] = valid
            key = splitmix64((seed & _M64) ^ splitmix64(step + 1))
            pf.set_stream_key(key)
            t0 = time.perf_counter()
            out[valid] = lp[valid] + pf.loglik(np.ascontiguousarray(thetas[valid].T))
            timers["filter_calls_wall"] += time.perf_counter() - t0
            if hasattr(pf, "last_timing"):
                timers["filter_device_ms"] += pf.last_timing()[0]
            if state_interval > 0:  # the lineage ends use a stream block the filter itself never draws from
                paths[valid] = pf.sample_paths(1, key, nb=len(valid))[:, 0]
        return out

    chains[:, 0, :] = t0s
    ll_i = target(chains[:, 0, :], 0)
    if state_interval > 0:
        cur_paths = paths.copy()
    # running sums of every chain's samples, SHIFTED by the chain's starting point (no cancellation for tightly
    # concentrated chains): the covariance of the adaptation step without a pass over the history
    shift = chains[:, 0, :].copy()
    sum_x = np.zeros((n_loc, d))
    sum_xx = np.zeros((n_loc, d, d))
    for i in range(1, steps):
        # host draws of step i for ALL chains from one stream keyed by (seed, i); a rank uses the rows of its chains, so the
        # chains do not depend on the number of ranks.  get_mv_param(propd, c, theta[mc, i-1, :]) (:181)
        g = np.random.default_rng([seed & 0xFFFFFFFF, 0x504D, i])
        z = g.standard_normal((n_chains, d))[lo:hi]
        u = g.random(n_chains)[lo:hi]
        prop = chains[:, i - 1, :] + c[:, None] * np.einsum("kij,kj->ki", chol, z)
        ll_f = target(prop, i)
        with np.errstate(over="ignore", invalid="ignore"):
            mh = np.exp(np.minimum(ll_f - ll_i, 700.0))
        ok = (ll_f != -np.inf) & ((mh > 1) | (mh > u))  # :189-190
        ll_i = np.where(ok, ll_f, ll_i)
        chains[:, i, :] = np.where(ok[:, None], prop, chains[:, i - 1, :])
        if state_interval > 0:
            cur_paths[ok] = paths[ok]
            if i >= adapt_period and (i - adapt_period) % state_interval == 0:
                kept.append(cur_paths.copy())
        accepted_total += ok
        dx = chains[:, i, :] - shift
        sum_x += dx
        sum_xx += np.einsum("ki,kj->kij", dx, dx)
        if i + 1 < adapt_period:  # Julia's 1-based step index is i + 1 (:198)
            c *= np.where(ok, 1.002, 0.999)
            if adapt_interval > 0 and math.fmod(i + 1, adapt_interval) == 0:  # i % ADAPT_INTERVAL == 0 (:200)
                n_s = i + 1
                mean = sum_x / n_s
                covar = (sum_xx - n_s * np.einsum("ki,kj->kij", mean, mean)) / (n_s - 1)
                flat_chain = covar.reshape(n_loc, -1).sum(axis=1) == 0
                if verbose and flat_chain.any():
                    print("warning: low acceptance rate detected in adaptation period")
                for k in np.nonzero(~flat_chain)[0]:
                    try:
                        chol[k] = np.linalg.cholesky(covar[k])
                    except np.linalg.LinAlgError:
                        pass
    flat = comm.allgather_f64(chains.reshape(n_loc, steps * d), n_chains)
    theta = np.ascontiguousarray(flat.reshape(n_chains, steps, d).transpose(2, 1, 0))
    rs = handle_rej_samples(theta, adapt_period)
    out = MCMCSample(rs, adapt_period, gelman_diagnostic_sre(theta, adapt_period), time.time_ns() - start_time)
    out.accepted = comm.allgather_f64(accepted_total.astype(np.float64), n_chains).astype(np.int64)
    timers["total_wall"] = (time.time_ns() - start_time) * 1e-9
    out.timers = timers
    if state_interval > 0:
        n_kept = len(kept)
        loc = np.stack(kept, axis=1) if n_kept else np.zeros((n_loc, 0, n_obs, n_comp), dtype=np.int64)
        flat = comm.allgather_f64(loc.reshape(n_loc, -1).astype(np.float64), n_chains)  # counts < 2^31: exact in f64
        out.states = flat.reshape(n_chains, n_kept, n_obs, n_comp).astype(np.int64)
    return out


def run_pmcmc_analysis(model: DPOMPModel, obs_data, n_chains: int = 3, initial_parameters: Optional[np.ndarray] = None,
                       steps: int = C_DF_MCMC_STEPS, adapt_period: Optional[int] = None, np_: int = 200, seed: int = 1,
                       comm: Optional[Comm] = None, state_interval: int = 0, **kw) -> MCMCSample:
    """Public-model wrapper in the style of run_mcmc_analysis (src/DiscretePOMP.jl:185-193): chains start from draws of
    the prior unless `initial_parameters` (n_theta, n_chains) is given.  state_interval: see run_pmcmc."""
    mdl = get_private_model(model, obs_data)
    if adapt_period is None:
        adapt_period = int(np.floor(steps * C_DF_MCMC_ADAPT))
    if initial_parameters is None:
        initial_parameters = mdl.prior.rand(n_chains, np.random.default_rng(seed))
    return run_pmcmc(mdl, initial_parameters, steps, adapt_period, np_, seed=seed, comm=comm, state_interval=state_interval, **kw)
