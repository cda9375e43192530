"""Data-augmented MCMC -- host-side mirror of run_std_mcmc with gibbs_mh_alg! (src/hmm_mcmc.jl:138) and the trajectory
proposals of src/hmm_std.jl, the sampler of run_mcmc_analysis(...; mbp = false) in the reference.

Every chain is one trajectory of the device trajectory store (dpomp_mbp handle).  All chains advance in lock step, one
C-ABI call per step over all chains of this rank:
    generate_x0 (src/hmm_sim.jl:160-168)          -> dpomp_mbp_iterate over obs 1..T, then dpomp_da_loglike
    theta proposal: compute_full_log_like!(xf)     -> dpomp_da_step, kind 0 (the host takes the MH decision)
    trajectory proposals (insert / delete / move)  -> dpomp_da_step, kind 1 (drawn, decided and applied on the device)
Each step a chain makes a theta proposal with probability ppp, else traj_props trajectory proposals.  The adaptive random
walk on theta is the one of run_mbp_mcmc; its scale adapts on theta steps only.  Chains shard over ranks with no
communication until the final gather (host draws from one stream per step, device draws keyed by the global chain index:
results do not depend on the number of ranks).
"""
from __future__ import annotations

import time
from typing import Callable, Optional

import numpy as np

from .distributed import Comm
from .ibis import _M64, prior_logpdf_columns, splitmix64
from .mbp_ibis import MbpParticles
from .mbp_mcmc import AdaptiveRandomWalk, generate_x0
from .mcmc import gelman_diagnostic_sre, handle_rej_samples
from .particle_filter import device_model
from .structs import HiddenMarkovModel, MCMCSample

KIND_THETA, KIND_TRAJECTORY, KIND_SKIP = 0, 1, 2


def run_std_mcmc(model: HiddenMarkovModel, theta_init: np.ndarray, steps: int, adapt_period: int, fin_adapt: bool = False,
                 ppp: float = 0.3, mvp: int = 3, traj_props: int = 1, seed: int = 1, comm: Optional[Comm] = None,
                 max_traj: int = 196000, particles_factory: Optional[Callable] = None, verbose: bool = True) -> MCMCSample:
    """run_std_mcmc(model, theta_init, steps, adapt_period, fin_adapt, ppp, mvp) (src/hmm_mcmc.jl); theta_init is
    (n_theta, n_chains).  Returns MCMCSample with samples.theta of shape (n_theta, steps, n_chains); `a_cnt` counts the
    accepted theta proposals (before / after adapt_period) and `traj_acc` (n_chains, 3) the accepted inserts, deletes and
    moves."""
    if not 0.0 <= ppp <= 1.0 or mvp < 1 or traj_props < 0:
        raise ValueError("need 0 <= ppp <= 1, mvp >= 1 and traj_props >= 0")
    comm = comm or Comm(None)
    start_time = time.time_ns()
    theta_init = np.asarray(theta_init, dtype=np.float64)
    d, n_chains = theta_init.shape
    lo, hi = comm.bounds(n_chains)
    n_loc = hi - lo
    if verbose and comm.rank == 0:
        print(f"Running: {n_chains}-chain {steps}-sample {'finite-' if fin_adapt else ''}adaptive DA-MCMC analysis "
              f"(model: {model.model_name})")
    make = particles_factory or (lambda n, sd: MbpParticles(device_model(model), n, max_traj, sd))
    ptcls = make(max(n_loc, 1), seed)
    ptcls.set_batch_offset(lo)
    call = 0

    def next_key() -> int:
        nonlocal call
        call += 1
        return splitmix64((seed & _M64) ^ splitmix64(0x4441 + call))

    chains = np.zeros((n_loc, steps, d))
    theta = np.array(theta_init[:, lo:hi], dtype=np.float64, order="C")
    a_cnt = np.zeros((n_loc, 2), dtype=np.int64)
    t_acc = np.zeros((n_loc, 3), dtype=np.int64)
    if n_loc:
        generate_x0(model, ptcls, theta, next_key)
        log_like = ptcls.da_loglike(theta)[:, 0]  # compute_full_log_like!(x0)
        prior = prior_logpdf_columns(model.prior, theta)
        rw = AdaptiveRandomWalk(theta, adapt_period)
        chains[:, 0, :] = theta.T
        a_cnt[:, 0] = 1
        for i in range(2, steps + 1):
            # host draws of step i for ALL chains from one stream keyed by (seed, i); a rank uses the rows of its chains
            g = np.random.default_rng([seed & 0xFFFFFFFF, 0x4441, i])
            z = g.standard_normal((n_chains, d))[lo:hi]
            u = g.random(n_chains)[lo:hi]
            on_theta = g.random(n_chains)[lo:hi] < ppp
            theta_f = rw.propose(theta, z)
            prior_f = prior_logpdf_columns(model.prior, theta_f)
            valid = prior_f != -np.inf
            kind = np.where(on_theta, np.where(valid, KIND_THETA, KIND_SKIP), KIND_TRAJECTORY).astype(np.uint8)
            ptcls.set_stream_key(next_key())
            ll2, acc = ptcls.da_step(theta, theta_f, kind, traj_props, mvp)
            traj = kind == KIND_TRAJECTORY
            log_like[traj] = ll2[traj, 0]
            t_acc += acc
            ll_f = ll2[:, 0]
            with np.errstate(over="ignore", invalid="ignore"):
                mh_prob = np.exp(prior_f - prior) * np.exp(ll_f - log_like)
            accepted = (kind == KIND_THETA) & (ll_f != -np.inf) & ((mh_prob > 1) | (mh_prob > u))  # NaN compares false
            theta[:, accepted] = theta_f[:, accepted]
            prior[accepted] = prior_f[accepted]
            log_like[accepted] = ll_f[accepted]
            a_cnt[accepted, 1 if i > adapt_period else 0] += 1
            chains[:, i - 1, :] = theta.T
            rw.record(theta)
            if (not fin_adapt) or i < adapt_period:
                rw.scale(accepted, on=on_theta)
                rw.adapt_period(i)
    flat = comm.allgather_f64(chains.reshape(n_loc, steps * d), n_chains)
    samples = np.ascontiguousarray(flat.reshape(n_chains, steps, d).transpose(2, 1, 0))
    rejs = handle_rej_samples(samples, adapt_period)
    out = MCMCSample(rejs, adapt_period, gelman_diagnostic_sre(samples, adapt_period), time.time_ns() - start_time)
    out.a_cnt = comm.allgather_f64(a_cnt.astype(np.float64), n_chains).astype(np.int64)
    out.traj_acc = comm.allgather_f64(t_acc.astype(np.float64), n_chains).astype(np.int64)
    out.particles = ptcls
    if verbose and comm.rank == 0:
        print(f"- finished in {out.run_time / 1e9:.1f} seconds. E(x) := {rejs.mu} "
              f"(accepted trajectory proposals: {out.traj_acc.sum(axis=0).tolist()} inserts / deletes / moves)")
    return out
