"""MBP-MCMC -- host-side mirror of run_mbp_mcmc (src/hmm_mcmc.jl:330-345) with met_hastings_alg! (:123-141), the
default algorithm of run_mcmc_analysis (src/DiscretePOMP.jl:185-193).

Every chain is one trajectory of the device trajectory store (dpomp_mbp handle, the `Particle` of
src/hmm_structs.jl:51-58).  The reference runs its chains one after the other; here all chains advance in lock step and
the per-chain calls of the reference become one C-ABI call per step over all chains of this rank:
    generate_x0 -> gillespie_sim (src/hmm_sim.jl:160-168, 85-102)    -> dpomp_mbp_iterate over obs 1..T
    model_based_proposal(model, theta_f, xi) (src/hmm_mbp.jl:147-150)  -> dpomp_mbp_propose(ymax = T)
    xi = xf for accepted proposals (@mcmc_handle_mh_step, :66-73)      -> dpomp_mbp_accept
The adaptive random walk (@initialise_mcmc :10-25, @met_hastings_adapt :44-52, @mcmc_adapt_period :28-41), the prior
and the accept/reject decisions stay host code, as in the reference.  Chains are independent, so they shard over ranks
with no communication until the final gather of the samples (every chain has its own host random stream and its device
draws are keyed by the global chain index: results do not depend on the number of ranks).
"""
from __future__ import annotations

import math
import time
from typing import Callable, Optional

import numpy as np

from .distributed import Comm
from .ibis import _M64, get_prop_density, ProposalDensity, prior_logpdf_columns, splitmix64
from .mbp_ibis import MbpParticles
from .mcmc import C_DF_MCMC_ADAPT, C_DF_MCMC_STEPS, C_INITIAL, gelman_diagnostic_sre, handle_rej_samples
from .particle_filter import device_model, get_private_model
from .structs import DPOMPModel, HiddenMarkovModel, MCMCSample

C_MCMC_ADAPT_INTERVALS = 10  # src/DiscretePOMP.jl:45


def generate_x0(model: HiddenMarkovModel, ptcls: MbpParticles, theta: np.ndarray, next_key: Callable[[], int],
                ntries: int = 10000) -> np.ndarray:
    """generate_x0 (src/hmm_sim.jl:160-168) for every chain of the handle: simulate a trajectory over all observations
    and return its log-likelihood log_like[1]; retried while any trajectory is invalid (-Inf: event capacity exceeded).
    `theta` is (n_theta, n)."""
    n = theta.shape[1]
    ll = np.full(n, -np.inf)
    for attempt in range(ntries):
        if attempt and hasattr(ptcls, "reset"):  # the device store keeps its events across calls: retries start afresh
            ptcls.reset()
        ll = np.zeros(n)
        for obs_i in range(1, len(model.obs_data) + 1):
            ptcls.set_stream_key(next_key())
            lg = ptcls.iterate(theta, obs_i, fresh=(obs_i == 1))
            if model.obs_data[obs_i - 1].obs_id > 0:  # y.obs_id > 0 && (p.log_like[1] += output) (src/hmm_sim.jl:23)
                ll = ll + lg
            else:
                ll = np.where(np.isneginf(lg), -np.inf, ll)
        if not np.any(np.isneginf(ll)):
            return ll
    print("WARNING: having an issue generating a valid trajectory")
    return ll


class AdaptiveRandomWalk:
    """The adaptive random walk on theta of the reference's MCMC samplers, for every chain of this rank: @initialise_mcmc
    (src/hmm_mcmc.jl:10-25), get_mv_param (src/hmm_cmn.jl:13-18), @met_hastings_adapt (:44-52) and @mcmc_adapt_period
    (:28-41).  theta is (n_theta, n_chains)."""

    def __init__(self, theta: np.ndarray, adapt_period: int):
        d, n = theta.shape
        # @initialise_mcmc: covar[i,i] = theta[i] == 0 ? 1 : theta[i]^2; propd = MvNormal(covar); c = C_INITIAL
        self.chol = np.zeros((n, d, d))  # Cholesky factor of every chain's proposal covariance
        self.chol[:, np.arange(d), np.arange(d)] = np.where(theta.T == 0.0, 1.0, np.abs(theta.T))
        self.c = np.full(n, C_INITIAL)
        self.sum_x = theta.T.copy()                                   # running sums of the samples of every chain: the
        self.sum_xx = np.einsum("ki,kj->kij", theta.T, theta.T)       # covariance of @mcmc_adapt_period without a pass over them
        self.adapt_interval = adapt_period / C_MCMC_ADAPT_INTERVALS  # Float64, like the reference

    def propose(self, theta: np.ndarray, z: np.ndarray) -> np.ndarray:
        """theta + c L z for standard normal z (n_chains, n_theta)"""
        return theta + (self.c[:, None] * np.einsum("kij,kj->ki", self.chol, z)).T

    def record(self, theta: np.ndarray) -> None:
        """the samples of the current step enter the running sums"""
        self.sum_x += theta.T
        self.sum_xx += np.einsum("ki,kj->kij", theta.T, theta.T)

    def scale(self, accepted: np.ndarray, on: Optional[np.ndarray] = None) -> None:
        """c *= 1.002 after an accepted, 0.999 after a rejected proposal; `on` restricts the update to those chains"""
        f = np.where(accepted, 1.002, 0.999)
        if on is None:
            self.c *= f
        else:
            self.c[on] *= f[on]

    def adapt_period(self, i: int) -> None:
        """@mcmc_adapt_period at step i (1-based): every adapt_period / 10 steps the proposal covariance becomes that of the
        samples 1..i"""
        if self.adapt_interval > 0 and math.fmod(i, self.adapt_interval) == 0:
            # covar = cov(transpose(theta[:, 1:i, mc])); propd = get_prop_density(covar, propd): kept when the
            # covariance is not positive definite (src/hmm_cmn.jl:33-42)
            mean = self.sum_x / i
            covar = (self.sum_xx - i * np.einsum("ki,kj->kij", mean, mean)) / (i - 1)
            sym = np.triu(covar) + np.transpose(np.triu(covar, 1), (0, 2, 1))  # Hermitian(): the upper triangle
            ok = np.linalg.eigvalsh(sym).min(axis=1) > 0
            if ok.any():
                try:
                    self.chol[ok] = np.linalg.cholesky(sym[ok])
                except np.linalg.LinAlgError:  # borderline matrices: decide chain by chain
                    for k in np.nonzero(ok)[0]:
                        self.chol[k] = get_prop_density(sym[k], ProposalDensity(self.chol[k])).chol


def run_mbp_mcmc(model: HiddenMarkovModel, theta_init: np.ndarray, steps: int, adapt_period: int, fin_adapt: bool = False,
                 seed: int = 1, comm: Optional[Comm] = None, max_traj: int = 196000,
                 particles_factory: Optional[Callable] = None, verbose: bool = True) -> MCMCSample:
    """run_mbp_mcmc(model, theta_init, steps, adapt_period, fin_adapt) (src/hmm_mcmc.jl:330-345); theta_init is
    (n_theta, n_chains).  Returns MCMCSample with samples.theta of shape (n_theta, steps, n_chains)."""
    comm = comm or Comm(None)
    start_time = time.time_ns()
    theta_init = np.asarray(theta_init, dtype=np.float64)
    d, n_chains = theta_init.shape
    lo, hi = comm.bounds(n_chains)
    n_loc = hi - lo
    if verbose and comm.rank == 0:
        print(f"Running: {n_chains}-chain {steps}-sample {'finite-' if fin_adapt else ''}adaptive MBP-MCMC analysis "
              f"(model: {model.model_name})")
    make = particles_factory or (lambda n, sd: MbpParticles(device_model(model), n, max_traj, sd))
    ptcls = make(max(n_loc, 1), seed)
    ptcls.set_batch_offset(lo)
    call = 0

    def next_key() -> int:
        nonlocal call
        call += 1
        return splitmix64((seed & _M64) ^ splitmix64(0x4D43 + call))

    chains = np.zeros((n_loc, steps, d))
    theta = np.array(theta_init[:, lo:hi], dtype=np.float64, order="C")  # own copy (d, n_loc): current theta of every local chain
    a_cnt = np.zeros((n_loc, 2), dtype=np.int64)
    if n_loc:
        log_like = generate_x0(model, ptcls, theta, next_key)  # x0.log_like[1]
        prior = prior_logpdf_columns(model.prior, theta)       # x0.prior
        rw = AdaptiveRandomWalk(theta, adapt_period)
        chains[:, 0, :] = theta.T
        a_cnt[:, 0] = 1
        n_obs = len(model.obs_data)
        for i in range(2, steps + 1):  # Julia's 1-based step index
            # host draws of step i for ALL chains from one stream keyed by (seed, i); a rank uses the rows of its chains, so
            # the chains do not depend on the number of ranks
            g = np.random.default_rng([seed & 0xFFFFFFFF, 0x4D43, i])
            z = g.standard_normal((n_chains, d))[lo:hi]
            u = g.random(n_chains)[lo:hi]
            theta_f = rw.propose(theta, z)  # get_mv_param(propd, c, theta[:, i-1, mc]) (:126)
            prior_f = prior_logpdf_columns(model.prior, theta_f)
            valid = prior_f != -np.inf
            ptcls.set_stream_key(next_key())
            ll_f = ptcls.propose(theta, theta_f, valid, n_obs)[:, 0]  # xf.log_like[1]
            with np.errstate(over="ignore", invalid="ignore"):
                mh_prob = np.exp(prior_f - prior) * np.exp(ll_f - log_like)  # :131
            accepted = valid & (ll_f != -np.inf) & ((mh_prob > 1) | (mh_prob > u))  # :127-133, NaN compares false
            ptcls.accept(np.nonzero(accepted)[0] + 1)  # xi = xf
            theta[:, accepted] = theta_f[:, accepted]
            prior[accepted] = prior_f[accepted]
            log_like[accepted] = ll_f[accepted]
            a_cnt[accepted, 1 if i > adapt_period else 0] += 1
            chains[:, i - 1, :] = theta.T
            rw.record(theta)
            if (not fin_adapt) or i < adapt_period:  # @met_hastings_adapt
                rw.scale(accepted)
                rw.adapt_period(i)
    flat = comm.allgather_f64(chains.reshape(n_loc, steps * d), n_chains)
    samples = np.ascontiguousarray(flat.reshape(n_chains, steps, d).transpose(2, 1, 0))
    rejs = handle_rej_samples(samples, adapt_period)
    out = MCMCSample(rejs, adapt_period, gelman_diagnostic_sre(samples, adapt_period), time.time_ns() - start_time)
    out.a_cnt = comm.allgather_f64(a_cnt.astype(np.float64), n_chains).astype(np.int64)
    out.particles = ptcls
    if verbose and comm.rank == 0:
        aar = 100.0 * out.a_cnt[:, 1] / max(steps - adapt_period, 1)
        print(f"- finished in {out.run_time / 1e9:.1f} seconds. E(x) := {rejs.mu} (AAR := {np.round(aar, 1)}%)")
    return out


def run_mcmc_analysis(model: DPOMPModel, obs_data, n_chains: int = 3, initial_parameters: Optional[np.ndarray] = None,
                      steps: int = C_DF_MCMC_STEPS, adapt_period: Optional[int] = None, fin_adapt: bool = False,
                      mbp: bool = True, ppp: float = 0.3, mvp: int = 3, seed: int = 1, comm: Optional[Comm] = None,
                      **kw) -> MCMCSample:
    """run_mcmc_analysis(model, obs_data; n_chains = 3, initial_parameters = rand(model.prior, n_chains), steps,
    adapt_period, fin_adapt = false, mbp = true, ppp, mvp) (src/DiscretePOMP.jl:185-193).  Only the MBP-MCMC default is on
    the accelerated path; `mbp = false` (the standard data-augmented Gibbs sampler, run_std_mcmc) is out of scope."""
    if not mbp:
        raise NotImplementedError("run_mcmc_analysis(mbp = false) is not provided; call run_std_mcmc for the data-augmented "
                                  "sampler, or use mbp = True")
    mdl = get_private_model(model, obs_data)
    if adapt_period is None:
        adapt_period = int(math.floor(steps * C_DF_MCMC_ADAPT))
    if initial_parameters is None:
        initial_parameters = mdl.prior.rand(n_chains, np.random.default_rng(seed))
    return run_mbp_mcmc(mdl, np.asarray(initial_parameters, dtype=np.float64), steps, adapt_period, fin_adapt, seed=seed,
                        comm=comm, **kw)
