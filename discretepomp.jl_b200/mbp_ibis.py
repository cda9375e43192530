"""MBP-IBIS -- host-side mirror of run_mbp_ibis (src/hmm_ibis.jl:140-244).

Each theta-particle is ONE trajectory with its event list (struct Particle, src/hmm_structs.jl:51-58), kept in HBM by
the dpomp_mbp handle.  The per-particle loops of the reference become one C-ABI call each:
    iterate_particle! over all particles        (:176-179)  -> dpomp_mbp_iterate
    ptcls2[p] = deepcopy(ptcls[nidx[p]])        (:196-199)  -> dpomp_mbp_permute
    partial_model_based_proposal over particles (:207)      -> dpomp_mbp_propose
    ptcls[p] = xf for accepted proposals        (:214)      -> dpomp_mbp_accept
Priors, MvNormal proposals, accept/reject and the evidence bookkeeping stay host code, as in the reference.

Stated departures: (1) a mutation sweep proposes for all particles at once, so the random-walk scale `tj`
(ind_prop = false, the MBP-IBIS default) is frozen within a sweep and updated afterwards with the same factors
(SURVEY.md 7); (2) `outer_rs` may be rs_stratified (BASELINE config C5) where the reference hard-codes rs_systematic
(:194).  `max_traj` is the reference's MAX_TRAJ = 196000 (src/DiscretePOMP.jl:40): the device store reserves a small stride
per trajectory and grows on demand, so the limit costs no memory (include/dpomp.h).
"""
from __future__ import annotations

import ctypes as C
import time
from typing import Callable, Optional

import numpy as np

from . import _capi
from .distributed import Comm
from .ibis import (_M64, ProposalDensity, compute_is_mu_covar, get_mv_param, get_prop_density, prior_logpdf_columns,
                   splitmix64)
from .particle_filter import compute_ess, device_model
from .resample import rs_systematic
from .structs import HiddenMarkovModel, ImportanceSample


MAX_TRAJ = 196000  # src/DiscretePOMP.jl:40


class MbpParticles:
    """dpomp_mbp handle: the trajectories of this process's theta-particles."""

    def __init__(self, dmodel, n_particles: int, max_traj: int = MAX_TRAJ, seed: int = 1, device: int = -1):
        self.dmodel, self.n, self.cap = dmodel, int(n_particles), int(max_traj)
        self.n_params = int(dmodel.compiled.desc.n_params)
        self.n_comp = int(dmodel.compiled.desc.n_compartments)
        self._h = C.c_void_p()
        _capi.check(_capi.lib().dpomp_mbp_create(dmodel.handle, self.n, self.cap, C.c_uint64(seed & _M64), device,
                                                 C.byref(self._h)))

    def __del__(self):
        try:
            if self._h:
                _capi.lib().dpomp_mbp_destroy(self._h)
                self._h = C.c_void_p()
        except Exception:
            pass

    def set_stream_key(self, key: int) -> None:
        _capi.check(_capi.lib().dpomp_mbp_set_stream_key(self._h, C.c_uint64(key)))

    def set_batch_offset(self, off: int) -> None:
        _capi.check(_capi.lib().dpomp_mbp_set_batch_offset(self._h, int(off)))

    def set_mode(self, mode: int) -> None:
        """Trajectory walks: 0 automatic, 1 one thread per trajectory, 2 one warp per trajectory (identical results)."""
        _capi.check(_capi.lib().dpomp_mbp_set_mode(self._h, int(mode)))

    def reset(self) -> None:
        _capi.check(_capi.lib().dpomp_mbp_reset(self._h))

    def capacity(self):
        """(current stride of the device store, hard limit max_traj) in events per trajectory."""
        a, b = C.c_int32(), C.c_int32()
        _capi.check(_capi.lib().dpomp_mbp_capacity(self._h, C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def reserve(self, stride: int) -> None:
        _capi.check(_capi.lib().dpomp_mbp_reserve(self._h, int(stride)))

    def _cols(self, theta) -> np.ndarray:
        return np.ascontiguousarray(np.asarray(theta, dtype=np.float64).T)  # (n, n_theta) == Julia column-major

    def iterate(self, theta, obs_i: int, fresh: bool) -> np.ndarray:
        th = self._cols(theta)
        out = np.empty(th.shape[0])
        _capi.check(_capi.lib().dpomp_mbp_iterate(self._h, _capi.ptr(th), th.shape[0], int(obs_i), 1 if fresh else 0,
                                                  _capi.ptr(out)))
        return out

    def propose(self, theta_i, theta_f, valid, ymax: int) -> np.ndarray:
        ti, tf = self._cols(theta_i), self._cols(theta_f)
        v = np.ascontiguousarray(valid, dtype=np.uint8)
        out = np.empty((ti.shape[0], 2))
        _capi.check(_capi.lib().dpomp_mbp_propose(self._h, _capi.ptr(ti), _capi.ptr(tf), _capi.ptr(v), ti.shape[0], int(ymax),
                                                  _capi.ptr(out)))
        return out

    def da_loglike(self, theta) -> np.ndarray:
        """dpomp_da_loglike: full log-likelihood {full, observation} (n, 2) of trajectories 1..n under theta (n_theta, n)."""
        th = self._cols(theta)
        out = np.empty((th.shape[0], 2))
        _capi.check(_capi.lib().dpomp_da_loglike(self._h, _capi.ptr(th), th.shape[0], _capi.ptr(out)))
        return out

    def da_step(self, theta_cur, theta_f, kind, traj_props: int, mvp: int):
        """dpomp_da_step: one data-augmented Gibbs step of chains 1..n (kind 0 theta, 1 trajectory, 2 nothing).  Returns
        ({full, observation} log-likelihoods (n, 2), accepted inserts / deletes / moves (n, 3))."""
        tc, tf = self._cols(theta_cur), self._cols(theta_f)
        k = np.ascontiguousarray(kind, dtype=np.uint8)
        out = np.empty((tc.shape[0], 2))
        acc = np.empty((tc.shape[0], 3), dtype=np.int32)
        _capi.check(_capi.lib().dpomp_da_step(self._h, _capi.ptr(tc), _capi.ptr(tf), _capi.ptr(k), tc.shape[0], int(traj_props),
                                              int(mvp), _capi.ptr(out), _capi.ptr(acc)))
        return out, acc.astype(np.int64)

    def accept(self, slots) -> None:
        s = _capi.as_i64(slots)
        if len(s):
            _capi.check(_capi.lib().dpomp_mbp_accept(self._h, _capi.ptr(s), len(s)))

    def permute(self, nidx) -> None:
        s = _capi.as_i64(nidx)
        _capi.check(_capi.lib().dpomp_mbp_permute(self._h, _capi.ptr(s), len(s)))

    def resample_migrate(self, comm, nidx, n_total: int) -> None:
        """dpomp_mbp_resample_migrate: particle p <- particle nidx[p] (1-based GLOBAL indices) across the ranks of `comm`."""
        s = _capi.as_i64(nidx)
        _capi.check(_capi.lib().dpomp_mbp_resample_migrate(self._h, comm.handle, _capi.ptr(s), int(n_total)))

    # -- migration between ranks (lengths first, then one packed payload) -------------------------------------
    FIXED_WORDS = 16

    def lengths(self, slots) -> np.ndarray:
        s = _capi.as_i64(slots)
        out = np.zeros(len(s), dtype=np.int32)
        if len(s):
            _capi.check(_capi.lib().dpomp_mbp_get_lengths(self._h, _capi.ptr(s), len(s), _capi.ptr(out)))
        return out

    def export_particles(self, slots, lens):
        """Pack the listed particles (1-based) into CUDA tensors (fixed int32 records, f64 times, u8 types)."""
        import torch

        s = _capi.as_i64(slots)
        off = np.concatenate(([0], np.cumsum(lens, dtype=np.int64)))
        fixed = torch.zeros(len(s) * self.FIXED_WORDS, dtype=torch.int32, device="cuda")
        times = torch.empty(int(off[-1]), dtype=torch.float64, device="cuda")
        types = torch.empty(int(off[-1]), dtype=torch.uint8, device="cuda")
        if len(s):
            o = _capi.as_i64(off[:-1])
            _capi.check(_capi.lib().dpomp_mbp_export(self._h, _capi.ptr(s), _capi.ptr(o), len(s), C.c_void_p(fixed.data_ptr()),
                                                     C.c_void_p(times.data_ptr()), C.c_void_p(types.data_ptr())))
        return fixed, times, types

    def import_particles(self, slots, lens, fixed, times, types) -> None:
        s = _capi.as_i64(slots)
        if len(s):
            self.reserve(int(np.max(lens)) if len(lens) else 1)  # trajectories that grew on another rank
            o = _capi.as_i64(np.concatenate(([0], np.cumsum(lens, dtype=np.int64)))[:-1])
            _capi.check(_capi.lib().dpomp_mbp_import(self._h, _capi.ptr(s), _capi.ptr(o), len(s), C.c_void_p(fixed.data_ptr()),
                                                     C.c_void_p(times.data_ptr()), C.c_void_p(types.data_ptr())))

    # -- device-resident outer layer (dpomp_mbp_outer_*): theta, weights, priors of ALL particles on the device -------------
    def outer_begin(self, comm_handle, theta: np.ndarray, prior_lo, prior_hi) -> None:
        th = self._cols(theta)
        lo, hi = _capi.as_f64(prior_lo), _capi.as_f64(prior_hi)
        _capi.check(_capi.lib().dpomp_mbp_outer_begin(self._h, comm_handle, th.shape[0], _capi.ptr(th), _capi.ptr(lo), _capi.ptr(hi)))

    def outer_iterate(self, obs_i: int, fresh: bool) -> np.ndarray:
        out = np.empty(5)
        _capi.check(_capi.lib().dpomp_mbp_outer_iterate(self._h, int(obs_i), 1 if fresh else 0, _capi.ptr(out)))
        return out

    def outer_moments(self):
        mu = np.empty(self.n_params); cv = np.empty((self.n_params, self.n_params))
        _capi.check(_capi.lib().dpomp_mbp_outer_moments(self._h, _capi.ptr(mu), _capi.ptr(cv)))
        return mu, cv

    def outer_resample(self, rs_type: int, u) -> float:
        uu = _capi.as_f64(np.atleast_1d(u)); out = np.empty(2)
        _capi.check(_capi.lib().dpomp_mbp_outer_resample(self._h, int(rs_type), _capi.ptr(uu), len(uu), _capi.ptr(out)))
        return float(out[0])

    def outer_sweep(self, mu, chol, scale: float, ind_prop: bool, obs_i: int):
        m, l = _capi.as_f64(mu), _capi.as_f64(chol); out = np.empty(2)
        _capi.check(_capi.lib().dpomp_mbp_outer_sweep(self._h, _capi.ptr(m), _capi.ptr(l), C.c_double(scale), 1 if ind_prop else 0,
                                                      int(obs_i), _capi.ptr(out)))
        return int(round(out[0])), float(out[1])

    def outer_get(self, n_total: int):
        th = np.empty((n_total, self.n_params)); w = np.empty(n_total)
        _capi.check(_capi.lib().dpomp_mbp_outer_get(self._h, _capi.ptr(th), _capi.ptr(w)))
        return np.ascontiguousarray(th.T), w

    def outer_end(self) -> None:
        _capi.check(_capi.lib().dpomp_mbp_outer_end(self._h))

    def final_conditions(self) -> np.ndarray:
        """(n, C) final states of all particles."""
        out = np.zeros((self.n, self.n_comp), dtype=np.int64)
        _capi.check(_capi.lib().dpomp_mbp_get_states(self._h, self.n, _capi.ptr(out)))
        return out

    def get_particle(self, p: int, proposal: bool = False):
        """(final_condition, times, types(1-based), log_like[2]) of particle p (1-based)."""
        fc = np.zeros(self.n_comp, dtype=np.int64); ln = C.c_int64()
        cap = self.capacity()[0]
        times = np.zeros(cap); types = np.zeros(cap, dtype=np.int32); ll = np.zeros(2)
        _capi.check(_capi.lib().dpomp_mbp_get_particle(self._h, int(p), 1 if proposal else 0, _capi.ptr(fc), C.byref(ln),
                                                       _capi.ptr(times), _capi.ptr(types), cap, _capi.ptr(ll)))
        return fc, times[: ln.value].copy(), types[: ln.value].copy(), ll


def _run_mbp_ibis_device(model, theta, ess_rs_crit, n_props, ind_prop, alpha, rng, seed, comm, ptcls, rs_type, verbose):
    """run_mbp_ibis with the outer layer resident on the device (dpomp_mbp_outer_*): the host keeps scalars only."""
    d, outer_p = theta.shape
    start_time = time.time_ns()
    ess_crit = ess_rs_crit * outer_p
    timers = {}

    def tick(name: str, t0: float) -> float:
        t1 = time.perf_counter()
        timers[name] = timers.get(name, 0.0) + (t1 - t0)
        return t1

    call = 0

    def next_key() -> int:
        nonlocal call
        call += 1
        return splitmix64((seed & _M64) ^ splitmix64(0x4D42 + call))

    t_ph = time.perf_counter()
    ptcls.outer_begin(comm.library_handle(), theta, model.prior.lower, model.prior.upper)
    t_ph = tick("begin", t_ph)
    propd = ProposalDensity.identity(d)
    tj = 0.2
    k_log = np.zeros(2, dtype=np.int64)
    bme = np.zeros(2)
    for obs_i in range(1, len(model.obs_data) + 1):
        ptcls.set_stream_key(next_key())
        t_ph = time.perf_counter()
        s0, s1, s2, s3, s4 = ptcls.outer_iterate(obs_i, fresh=(obs_i == 1))  # :176-185 on the device
        t_ph = tick("iterate", t_ph)
        if model.obs_data[obs_i - 1].obs_id > 0:
            with np.errstate(divide="ignore", invalid="ignore"):
                lml = np.log(s1 / s0)
                ess = s2 * s2 / s3
            bme[0] += lml
            if ess < ess_crit:
                mu, cv = ptcls.outer_moments()
                propd = get_prop_density(cv, propd)
                u = rng.random() if rs_type == 1 else rng.random(outer_p)
                t_ph = time.perf_counter()
                mean_gx = ptcls.outer_resample(rs_type, u)  # :194-201
                t_ph = tick("resample_migrate", t_ph)
                mlr = mean_gx * np.exp(lml)
                mean_mtd = mean_gx
                k_log[0] += outer_p * n_props
                for _ in range(n_props):  # :203-219
                    ptcls.set_stream_key(next_key())
                    n_acc, mean_mtd = ptcls.outer_sweep(mu, propd.chol, 1.0 if ind_prop else tj, ind_prop, obs_i)
                    k_log[1] += n_acc
                    tj *= alpha ** n_acc * 0.999 ** (outer_p - n_acc)
                tick("sweeps", t_ph)
                bme[1] += np.log(mlr / mean_mtd)
            else:
                bme[1] += np.log(s4 / s2)  # :231, with the already updated w as written
    mu, cv = ptcls.outer_moments()
    theta_out, w = ptcls.outer_get(outer_p)
    output = ImportanceSample(mu, cv, theta_out, w, time.time_ns() - start_time, -bme)
    if verbose and comm.rank == 0:
        ar = 100.0 * k_log[1] / k_log[0] if k_log[0] else float("nan")
        print(f"- finished in {output.run_time / 1e9:.1f} seconds (AR := {ar:.3g}%)")
    output.k_log = k_log
    output.timers = timers
    output.particles = ptcls
    return output


def run_mbp_ibis(model: HiddenMarkovModel, theta: np.ndarray, ess_rs_crit: float, n_props: int, ind_prop: bool,
                 alpha: float, msgs: bool = True, rng: Optional[np.random.Generator] = None, seed: int = 1,
                 comm: Optional[Comm] = None, max_traj: int = MAX_TRAJ, outer_rs: Callable = rs_systematic,
                 particles_factory: Optional[Callable] = None, verbose: bool = True,
                 device_outer: Optional[bool] = None) -> ImportanceSample:
    """run_mbp_ibis(model, theta, ess_rs_crit, n_props, ind_prop, alpha, msgs = true) (src/hmm_ibis.jl:140-244).
    `theta` is (n_theta, outer_p).  With `comm`, theta-particles (and their trajectories) are partitioned over the ranks;
    theta, weights and every host decision are replicated (same host RNG), trajectories migrate after the outer resample
    with a two-phase all-to-all (lengths, then the packed events)."""
    comm = comm or Comm(None)
    rng = rng or np.random.default_rng(seed)
    theta = np.array(theta, dtype=np.float64, order="C")
    d, outer_p = theta.shape
    if verbose and comm.rank == 0:
        print(f"Running: {outer_p}-particle MBP-IBIS analysis (model: {model.model_name})")
    lo, hi = comm.bounds(outer_p)
    n_loc = hi - lo
    start_time = time.time_ns()
    ess_crit = ess_rs_crit * outer_p
    make = particles_factory or (lambda n, sd: MbpParticles(device_model(model), n, max_traj, sd))
    ptcls = make(max(n_loc, 1), seed)
    if particles_factory is not None and hasattr(ptcls, "reset"):
        ptcls.reset()  # a caller-provided (pre-allocated, possibly used) store starts from the initial condition
    ptcls.set_batch_offset(lo)
    # Outer layer on the device (theta, weights, proposals, accept test as replicated kernels; the host keeps scalars) when
    # the prior is a product of uniforms and the exchanges go through the C ABI; `device_outer=False` forces the host-driven
    # loop below (same algorithm; host numpy draws instead of Philox streams for the proposals).
    from .examples import UniformProduct
    from .resample import rs_stratified as _rs_strat

    can_device = (isinstance(model.prior, UniformProduct) and hasattr(ptcls, "outer_begin") and d <= 8
                  and outer_rs in (rs_systematic, _rs_strat) and comm.library_handle() is not None)
    if device_outer is None:
        device_outer = can_device
    if device_outer:
        if not can_device:
            raise ValueError("device_outer needs a UniformProduct prior, systematic / stratified outer resampling and the C-ABI communicator")
        return _run_mbp_ibis_device(model, theta, ess_rs_crit, n_props, ind_prop, alpha, rng, seed, comm, ptcls,
                                    2 if outer_rs is _rs_strat else 1, verbose)

    timers = {}  # seconds per phase on this rank

    def tick(name: str, t0: float) -> float:
        t1 = time.perf_counter()
        timers[name] = timers.get(name, 0.0) + (t1 - t0)
        return t1

    def gather(local: np.ndarray) -> np.ndarray:
        t0 = time.perf_counter()
        out = comm.allgather_f64(local, outer_p)
        tick("allgather", t0)
        return out

    def migrate(nidx: np.ndarray) -> None:
        """ptcls2[p] = deepcopy(ptcls[nidx[p]]) (:196-199) across ranks."""
        if comm.world == 1:
            ptcls.permute(nidx)
            return
        if comm.handle is not None and hasattr(ptcls, "resample_migrate"):  # C ABI: NCCL inside the library
            ptcls.resample_migrate(comm, nidx, outer_p)
            return
        import torch
        from .distributed import migration_plan

        local_src, send_slots, send_counts, recv_slots, recv_counts = migration_plan(nidx - 1, outer_p, comm.world, comm.rank)
        send_lens = ptcls.lengths(send_slots + 1)
        lens_t = torch.from_numpy(send_lens.astype(np.int32)).to("cuda")
        recv_lens = comm.all_to_all_v(lens_t, send_counts, recv_counts).cpu().numpy()
        fixed, times, types = ptcls.export_particles(send_slots + 1, send_lens)
        ev_send = [int(send_lens[sum(send_counts[:r]):sum(send_counts[:r + 1])].sum()) for r in range(comm.world)]
        ev_recv = [int(recv_lens[sum(recv_counts[:r]):sum(recv_counts[:r + 1])].sum()) for r in range(comm.world)]
        fw = MbpParticles.FIXED_WORDS
        r_fixed = comm.all_to_all_v(fixed, [c * fw for c in send_counts], [c * fw for c in recv_counts])
        r_times = comm.all_to_all_v(times, ev_send, ev_recv)
        r_types = comm.all_to_all_v(types, ev_send, ev_recv)
        if n_loc:
            ptcls.permute(local_src + 1)
        ptcls.import_particles(recv_slots + 1, recv_lens, r_fixed, r_times, r_types)
    prior = prior_logpdf_columns(model.prior, theta)  # Particle.prior (:153)
    log_like = np.zeros(outer_p)  # Particle.log_like[1], mirrored on the host for the acceptance ratio
    propd = ProposalDensity.identity(d)
    tj = 0.2
    w = np.ones(outer_p)
    k_log = np.zeros(2, dtype=np.int64)
    bme = np.zeros(2)
    call = 0

    def next_key() -> int:
        nonlocal call
        call += 1
        return splitmix64((seed & _M64) ^ splitmix64(0x4D42 + call))

    mu, cv = compute_is_mu_covar(theta, w)
    for obs_i in range(1, len(model.obs_data) + 1):
        ptcls.set_stream_key(next_key())
        t_ph = time.perf_counter()
        lg_loc = ptcls.iterate(theta[:, lo:hi], obs_i, fresh=(obs_i == 1)) if n_loc else np.zeros(0)  # :176-179
        tick("iterate", t_ph)
        lg = gather(lg_loc)
        if model.obs_data[obs_i - 1].obs_id > 0:
            log_like = log_like + lg  # -Inf propagates for overflowed trajectories (src/hmm_sim.jl:17-20)
            gx = np.exp(lg)
            lml = np.log(np.sum(w * gx) / np.sum(w))
            bme[0] += lml
            w = w * gx
            if compute_ess(w) < ess_crit:
                mu, cv = compute_is_mu_covar(theta, w)  # evaluated where it is consumed (the reference: at every observation)
                propd = get_prop_density(cv, propd)
                nidx = outer_rs(w.copy(), rng)
                mtd_gx = gx[nidx - 1].copy()
                t_ph = time.perf_counter()
                migrate(nidx)
                tick("resample_migrate", t_ph)
                theta, prior, log_like = theta[:, nidx - 1], prior[nidx - 1], log_like[nidx - 1]
                mlr = np.mean(gx[nidx - 1]) * np.exp(lml)
                k_log[0] += outer_p * n_props
                for _ in range(n_props):  # :203-219, one sweep over all particles
                    theta_f = (mu[:, None] + propd.rand(rng, outer_p)) if ind_prop else get_mv_param(propd, tj, theta, rng)
                    prior_f = prior_logpdf_columns(model.prior, theta_f)
                    valid = prior_f != -np.inf
                    ptcls.set_stream_key(next_key())
                    t_ph = time.perf_counter()
                    ll_loc = (ptcls.propose(theta[:, lo:hi], theta_f[:, lo:hi], valid[lo:hi], obs_i)
                              if n_loc else np.zeros((0, 2)))
                    tick("propose", t_ph)
                    ll_f = gather(ll_loc)  # (outer_p, 2)
                    u = rng.random(outer_p)
                    with np.errstate(over="ignore", invalid="ignore"):
                        ratio = np.exp(prior_f - prior) * np.exp(ll_f[:, 0] - log_like)  # :212
                    accepted = ratio > u  # NaN compares false, as in the reference
                    t_ph = time.perf_counter()
                    ptcls.accept(np.nonzero(accepted[lo:hi])[0] + 1)
                    tick("accept_copy", t_ph)
                    mtd_gx[accepted] = np.exp(ll_f[accepted, 1])
                    theta[:, accepted] = theta_f[:, accepted]
                    prior[accepted] = prior_f[accepted]
                    log_like[accepted] = ll_f[accepted, 0]
                    n_acc = int(accepted.sum())
                    k_log[1] += n_acc
                    tj *= alpha ** n_acc * 0.999 ** (outer_p - n_acc)
                bme[1] += np.log(mlr / np.mean(mtd_gx))
                w = np.ones(outer_p)
            else:
                bme[1] += np.log(np.sum(w * gx) / np.sum(w))
    mu, cv = compute_is_mu_covar(theta, w)
    output = ImportanceSample(mu, cv, theta, w, time.time_ns() - start_time, -bme)
    if verbose and comm.rank == 0:
        ar = 100.0 * k_log[1] / k_log[0] if k_log[0] else float("nan")
        print(f"- finished in {output.run_time / 1e9:.1f} seconds (AR := {ar:.3g}%)")
    output.k_log = k_log
    output.timers = timers
    output.particles = ptcls
    return output
