"""Bootstrap particle filter entry points -- host-side mirror of src/hmm_particle_filter.jl, src/DiscretePOMP.jl:96-99
and src/hmm_utils.jl:281-284 of the reference.  All numerics run in libdpomp.so (CUDA, sm_100a) through the C ABI.

Reference call stack (SURVEY.md 3A):
    get_particle_filter_lpdf(model, y; np, rs_type)   -> closure f(theta)::Float64
      get_private_model -> get_log_pdf_fn -> estimate_likelihood -> partial_log_likelihood!
Here the closure holds a device handle (`ParticleFilter`) and every f(theta) is one dpomp_pf_loglik call.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, List, Optional, Sequence

import numpy as np

from . import _capi
from .examples import generate_trans_fn
from .rate_table import CompiledModel, build_model_desc, compile_obs_table, compile_rate_table
from .structs import DPOMPModel, HiddenMarkovModel, Observation

C_DF_PF_P = 200  # src/DiscretePOMP.jl:48
C_DF_ESS_CRIT = 0.3  # src/DiscretePOMP.jl:49


def compute_ess(w: np.ndarray) -> float:
    """compute_ess (src/hmm_particle_filter.jl:4-6)"""
    w = np.asarray(w, dtype=np.float64)
    return float(np.sum(w) ** 2 / np.sum(w * w))


class DeviceModel:
    """dpomp_model handle: the compiled rate / observation table plus the observations."""

    def __init__(self, compiled: CompiledModel):
        self.compiled = compiled
        self._h = C.c_void_p()
        _capi.check(_capi.lib().dpomp_model_create(C.byref(compiled.desc), C.byref(self._h)))
        obs = compiled.obs
        if obs is not None and obs.family != _capi.OBS_GAUSSIAN:
            idx = np.ascontiguousarray(obs.par_index, dtype=np.int32)
            val = np.ascontiguousarray(obs.par_value, dtype=np.float64)
            _capi.check(_capi.lib().dpomp_model_set_obs_model(self._h, int(obs.family), _capi.ptr(idx), _capi.ptr(val)))

    @property
    def handle(self) -> C.c_void_p:
        return self._h

    def __del__(self):
        try:
            if self._h:
                _capi.lib().dpomp_model_destroy(self._h)
                self._h = C.c_void_p()
        except Exception:
            pass


def compile_model(model: DPOMPModel, obs_data: Sequence[Observation]) -> CompiledModel:
    n_events, n_comp = model.m_transition.shape
    n_params = len(model.prior) if hasattr(model.prior, "__len__") else n_events
    rate = compile_rate_table(model.rate_function, n_events, n_params, n_comp)
    n_vals = len(obs_data[0].val) if len(obs_data) else n_comp
    obs = compile_obs_table(model.obs_model, n_comp, n_vals, n_params)
    return build_model_desc(rate, obs, model.m_transition, model.initial_condition, model.t0_index, obs_data)


def get_private_model(m: DPOMPModel, y: Sequence[Observation]) -> HiddenMarkovModel:
    """get_private_model (src/DiscretePOMP.jl:96-99)"""

    def fnic():
        return m.initial_condition

    hmm = HiddenMarkovModel(m.model_name, m.m_transition.shape[0], m.rate_function, fnic,
                            generate_trans_fn(m.m_transition), m.obs_function, m.obs_model, list(y), m.prior,
                            m.t0_index)
    hmm._public = m
    return hmm


def device_model(mdl: HiddenMarkovModel) -> DeviceModel:
    if mdl._device_model is None:
        public = mdl._public
        if public is None:
            public = DPOMPModel(mdl.model_name, mdl.rate_function, np.asarray(mdl.fn_initial_condition()),
                                np.stack([mdl.fn_transition(e + 1) for e in range(mdl.n_events)]), mdl.obs_function,
                                mdl.obs_model, mdl.prior, mdl.t0_index)
        mdl._device_model = DeviceModel(compile_model(public, mdl.obs_data))
    return mdl._device_model


class ParticleFilter:
    """dpomp_pf handle: `n_batch` independent filters of `n_particles` with device-resident populations."""

    def __init__(self, dmodel: DeviceModel, n_particles: int, n_batch: int = 1, rs_type: int = 1, seed: int = 1,
                 device: int = -1, sim_precision: int = _capi.SIM_F32, max_events: Optional[int] = None):
        self.dmodel = dmodel
        self.n_particles, self.n_batch, self.rs_type = int(n_particles), int(n_batch), int(rs_type)
        self.n_params = int(dmodel.compiled.desc.n_params)
        self.n_comp = int(dmodel.compiled.desc.n_compartments)
        self.n_obs = int(dmodel.compiled.desc.n_obs)
        self._h = C.c_void_p()
        lib = _capi.lib()
        _capi.check(lib.dpomp_pf_create(dmodel.handle, self.n_particles, self.n_batch, self.rs_type,
                                        C.c_uint64(seed & 0xFFFFFFFFFFFFFFFF), device, C.byref(self._h)))
        if sim_precision != _capi.SIM_F32:
            _capi.check(lib.dpomp_pf_set_sim_precision(self._h, sim_precision))
        if max_events is not None:
            _capi.check(lib.dpomp_pf_set_max_events(self._h, int(max_events)))

    def __del__(self):
        try:
            if self._h:
                _capi.lib().dpomp_pf_destroy(self._h)
                self._h = C.c_void_p()
        except Exception:
            pass

    # -- options -----------------------------------------------------------------------------------------------
    def set_batch_offset(self, off: int) -> None:
        _capi.check(_capi.lib().dpomp_pf_set_batch_offset(self._h, int(off)))

    def set_fused(self, mode) -> None:
        """Fused simulate+resample launch per observation: 0/False never, 1 (default) for one-tile filters, 2/True
        whenever all tiles of a filter fit on the device at once."""
        mode = 2 if mode is True else int(mode)
        _capi.check(_capi.lib().dpomp_pf_set_fused(self._h, mode))

    def set_persistent(self, mode: int) -> None:
        """One cooperative launch per call (all observations): 0 never, 1 for calls over several observations, 2 always."""
        _capi.check(_capi.lib().dpomp_pf_set_persistent(self._h, int(mode)))

    def set_scatter(self, mode: int) -> None:
        """Row order of the offspring: 0 the reference's (offspring i in row i), 1 chunk-interleaved over the tiles."""
        _capi.check(_capi.lib().dpomp_pf_set_scatter(self._h, int(mode)))

    def set_filter_ids(self, ids) -> None:
        """Explicit 0-based GLOBAL ids of the first len(ids) filters (random-stream keying); None resets."""
        if ids is None:
            _capi.check(_capi.lib().dpomp_pf_set_filter_ids(self._h, None, 0))
        else:
            a = _capi.as_i64(ids)
            _capi.check(_capi.lib().dpomp_pf_set_filter_ids(self._h, _capi.ptr(a), len(a)))

    def set_stream_key(self, key: int) -> None:
        _capi.check(_capi.lib().dpomp_pf_set_stream_key(self._h, C.c_uint64(key)))

    def next_stream_key(self) -> int:
        k = C.c_uint64()
        _capi.check(_capi.lib().dpomp_pf_get_stream_key(self._h, C.byref(k)))
        return int(k.value)

    def geometry(self):
        t, i = C.c_int32(), C.c_int32()
        _capi.check(_capi.lib().dpomp_pf_geometry(self._h, C.byref(t), C.byref(i)))
        return int(t.value), int(i.value)

    def set_record_ancestors(self, on: bool) -> None:
        _capi.check(_capi.lib().dpomp_pf_set_record_ancestors(self._h, 1 if on else 0))

    # -- the path ----------------------------------------------------------------------------------------------
    def _theta(self, theta) -> np.ndarray:
        th = _capi.as_f64(theta)
        if th.ndim == 1:
            th = th.reshape(self.n_params, 1)
        if th.shape[0] != self.n_params:
            raise ValueError(f"theta must be ({self.n_params}, n_batch)")
        # Julia layout (n_theta, B) column-major == C layout (B, n_theta)
        return np.ascontiguousarray(th.T)

    def loglik(self, theta) -> np.ndarray:
        """estimate_likelihood (src/hmm_particle_filter.jl:79-84) for each column of theta."""
        th = self._theta(theta)
        out = np.empty(th.shape[0], dtype=np.float64)
        _capi.check(_capi.lib().dpomp_pf_loglik(self._h, _capi.ptr(th), th.shape[0], _capi.ptr(out)))
        return out

    def partial(self, theta, ymin: int, ymax: int) -> np.ndarray:
        """partial_log_likelihood! (src/hmm_particle_filter.jl:39-76) for each column of theta; 1-based ymin..ymax."""
        th = self._theta(theta)
        out = np.empty(th.shape[0], dtype=np.float64)
        _capi.check(_capi.lib().dpomp_pf_partial(self._h, _capi.ptr(th), th.shape[0], int(ymin), int(ymax),
                                                 _capi.ptr(out)))
        return out

    def partial_allgather(self, comm, theta_local, ymin: int, ymax: int, n_total: int) -> np.ndarray:
        """dpomp_pf_partial_allgather: partial() for this rank's block of the n_total filters, then the increments of ALL
        ranks (one stream-ordered sequence inside the library: kernels -> ncclAllGather -> one copy to the host)."""
        th = self._theta(theta_local) if np.size(theta_local) else np.zeros((0, self.n_params))
        out = np.empty(int(n_total), dtype=np.float64)
        _capi.check(_capi.lib().dpomp_pf_partial_allgather(self._h, comm.handle, _capi.ptr(th) if th.size else None, th.shape[0],
                                                           int(ymin), int(ymax), int(n_total), _capi.ptr(out)))
        return out

    def resample_migrate(self, comm, nidx, n_total: int) -> None:
        """dpomp_pf_resample_migrate: filter p <- filter nidx[p] (1-based GLOBAL indices) across the ranks of `comm`."""
        idx = _capi.as_i64(nidx)
        _capi.check(_capi.lib().dpomp_pf_resample_migrate(self._h, comm.handle, _capi.ptr(idx), int(n_total)))

    def permute(self, nidx: np.ndarray) -> None:
        idx = _capi.as_i64(nidx)
        _capi.check(_capi.lib().dpomp_pf_permute(self._h, _capi.ptr(idx), len(idx)))

    def copy_from(self, src: "ParticleFilter", dst_slots, src_slots) -> None:
        d, s = _capi.as_i64(dst_slots), _capi.as_i64(src_slots)
        if len(d):
            _capi.check(_capi.lib().dpomp_pf_copy_filters(self._h, src._h, _capi.ptr(d), _capi.ptr(s), len(d)))

    def get_pop(self, b: int = 1) -> np.ndarray:
        """Population of filter b (1-based) as the reference's Matrix{Int64}: shape (n_particles, C)."""
        out = np.empty((self.n_comp, self.n_particles), dtype=np.int64)
        _capi.check(_capi.lib().dpomp_pf_get_pop(self._h, int(b), _capi.ptr(out)))
        return out.T

    def set_pop(self, b: int, pop: np.ndarray) -> None:
        arr = np.ascontiguousarray(np.asarray(pop, dtype=np.int64).T)
        _capi.check(_capi.lib().dpomp_pf_set_pop(self._h, int(b), _capi.ptr(arr)))

    def last_logw(self, b: int = 1) -> np.ndarray:
        out = np.empty(self.n_particles, dtype=np.float64)
        _capi.check(_capi.lib().dpomp_pf_get_last_logw(self._h, int(b), _capi.ptr(out)))
        return out

    def last_ancestors(self, b: int = 1) -> np.ndarray:
        out = np.empty(self.n_particles, dtype=np.int64)
        _capi.check(_capi.lib().dpomp_pf_get_last_ancestors(self._h, int(b), _capi.ptr(out)))
        return out

    def overflow_count(self) -> int:
        v = C.c_int64()
        _capi.check(_capi.lib().dpomp_pf_overflow_count(self._h, C.byref(v)))
        return int(v.value)

    def last_event_count(self) -> int:
        v = C.c_int64()
        _capi.check(_capi.lib().dpomp_pf_last_event_count(self._h, C.byref(v)))
        return int(v.value)

    def last_timing(self):
        ms, n = C.c_float(), C.c_int32()
        _capi.check(_capi.lib().dpomp_pf_last_timing(self._h, C.byref(ms), C.byref(n)))
        return float(ms.value), int(n.value)

    def set_kernel_timing(self, on: bool) -> None:
        _capi.check(_capi.lib().dpomp_pf_set_kernel_timing(self._h, 1 if on else 0))

    def last_kernel_timing(self):
        """((ms_sim, ms_resample), (launches_sim, launches_resample)) of the last call (kernel timing on)."""
        ms = (C.c_float * 2)(); n = (C.c_int32 * 2)()
        _capi.check(_capi.lib().dpomp_pf_last_kernel_timing(self._h, ms, n))
        return (float(ms[0]), float(ms[1])), (int(n[0]), int(n[1]))

    def loglik_device(self, theta_dev_ptr: int, n_batch_used: int, out_dev_ptr: int) -> None:
        _capi.check(_capi.lib().dpomp_pf_loglik_device(self._h, C.c_void_p(theta_dev_ptr), int(n_batch_used),
                                                       C.c_void_p(out_dev_ptr)))

    @property
    def filter_words(self) -> int:
        """int32 words of one packed filter: n_compartments * padded particle count."""
        tile, _ = self.geometry()
        return self.n_comp * (-(-self.n_particles // tile) * tile)

    def export_tensor(self, slots):
        """Pack the listed filters (1-based) into a new torch int32 CUDA tensor (migration send buffer)."""
        import torch

        s = _capi.as_i64(slots)
        buf = torch.empty(len(s) * self.filter_words, dtype=torch.int32, device="cuda")
        if len(s):
            self.export_filters(s, buf.data_ptr())
        return buf

    def import_tensor(self, slots, buf) -> None:
        s = _capi.as_i64(slots)
        if len(s):
            self.import_filters(s, buf.data_ptr())

    def export_filters(self, slots, device_dst_ptr: int) -> None:
        s = _capi.as_i64(slots)
        _capi.check(_capi.lib().dpomp_pf_export_filters(self._h, _capi.ptr(s), len(s), C.c_void_p(device_dst_ptr)))

    def import_filters(self, slots, device_src_ptr: int) -> None:
        s = _capi.as_i64(slots)
        _capi.check(_capi.lib().dpomp_pf_import_filters(self._h, _capi.ptr(s), len(s), C.c_void_p(device_src_ptr)))


def estimate_likelihood(model: HiddenMarkovModel, parameters, particles: int, rs_type: int = 1, seed: int = 1,
                        **kw) -> float:
    """estimate_likelihood (src/hmm_particle_filter.jl:79-84): one fresh filter over all observations."""
    pf = ParticleFilter(device_model(model), particles, 1, rs_type, seed, **kw)
    return float(pf.loglik(np.asarray(parameters, dtype=np.float64))[0])


def get_log_pdf_fn(mdl: HiddenMarkovModel, p: int = C_DF_PF_P, rs_type: int = 1, essc: float = C_DF_ESS_CRIT,
                   seed: int = 1, n_batch: int = 1, **kw) -> Callable:
    """get_log_pdf_fn (src/hmm_particle_filter.jl:87-101).  `essc` is accepted and unused, as in the reference (F5).
    The returned closure accepts a parameter vector (-> float) or an (n_theta, B<=n_batch) matrix (-> array)."""
    pf = ParticleFilter(device_model(mdl), p, n_batch, rs_type if rs_type in (2, 3) else 1, seed, **kw)

    def comp_log_pdf(parameters):
        th = np.asarray(parameters, dtype=np.float64)
        res = pf.loglik(th)
        return float(res[0]) if th.ndim == 1 else res

    comp_log_pdf.particle_filter = pf  # keep the handle reachable for diagnostics
    return comp_log_pdf


def get_particle_filter_lpdf(model: DPOMPModel, obs_data: List[Observation], np: int = C_DF_PF_P, rs_type: int = 1,
                             essc: float = C_DF_ESS_CRIT, **kw) -> Callable:
    """get_particle_filter_lpdf(model, obs_data; np, rs_type, essc) (src/hmm_utils.jl:281-284)"""
    mdl = get_private_model(model, obs_data)
    return get_log_pdf_fn(mdl, np, rs_type, essc=essc, **kw)
