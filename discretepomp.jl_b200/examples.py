"""Predefined models, the Gaussian observation model and priors -- mirror of src/hmm_examples.jl.

`generate_model` (src/hmm_examples.jl:99-211) returns a DPOMPModel whose rate function is an ordinary host closure
with the reference's signature `rate_function(output, parameters, population)`; `get_private_model` compiles it to the
device rate table by probing (rate_table.py).  Model names are exactly those the reference's code accepts (:171-204).
"""
from __future__ import annotations

from typing import Callable, Optional, Sequence

import numpy as np

from . import _capi
from .rate_table import ObsTable, count_logpmf
from .structs import DPOMPModel, Observation


def dmy_obs_fn(y: Observation, population: np.ndarray, parameters: np.ndarray) -> None:
    """dmy_obs_fn (src/hmm_examples.jl:6-8): y.val .= population"""
    y.val[:] = population


def generate_trans_fn(tm: np.ndarray) -> Callable[[int], np.ndarray]:
    """generate_trans_fn (src/hmm_examples.jl:11-16); `et` is 1-based like the reference."""
    tm = np.atleast_2d(np.asarray(tm, dtype=np.int64))

    def fnt(et: int) -> np.ndarray:
        return tm[et - 1, :]

    return fnt


class UniformProduct:
    """Distributions.Product(Distributions.Uniform.(lower, upper)) as used by generate_weak_prior
    (src/hmm_examples.jl:33-35) and the reference's tests (test/runtests.jl:29)."""

    def __init__(self, lower: Sequence[float], upper: Sequence[float]):
        self.lower = np.asarray(lower, dtype=np.float64)
        self.upper = np.asarray(upper, dtype=np.float64)

    def __len__(self) -> int:
        return len(self.lower)

    def logpdf(self, theta: np.ndarray) -> float:
        theta = np.asarray(theta, dtype=np.float64)
        if np.any(theta < self.lower) or np.any(theta > self.upper):
            return -np.inf
        return float(-np.sum(np.log(self.upper - self.lower)))

    def logpdf_batch(self, theta: np.ndarray) -> np.ndarray:
        """logpdf of every column of an (n_theta, n) matrix (vectorised; same values as logpdf)."""
        theta = np.asarray(theta, dtype=np.float64)
        inside = np.ones(theta.shape[1], dtype=bool)
        for k in range(theta.shape[0]):  # one pass per parameter: fast for either memory layout of the (n_theta, n) matrix
            row = theta[k]
            inside &= (row >= self.lower[k]) & (row <= self.upper[k])
        return np.where(inside, float(-np.sum(np.log(self.upper - self.lower))), -np.inf)

    def rand(self, n: int = 1, rng: Optional[np.random.Generator] = None) -> np.ndarray:
        """rand(prior, n) -> (n_theta, n) like Julia."""
        rng = rng or np.random.default_rng()
        return self.lower[:, None] + (self.upper - self.lower)[:, None] * rng.random((len(self.lower), n))


def generate_weak_prior(n: int, b: float = 1.0) -> UniformProduct:
    """generate_weak_prior (src/hmm_examples.jl:33-35)"""
    return UniformProduct(np.zeros(n), np.full(n, b))


class GaussianObsModel:
    """Closure `gom2` of partial_gaussian_obs_model (src/hmm_examples.jl:59-67); seq / y_seq are 1-based index lists."""

    def __init__(self, sigma: float = 2.0, seq=(2,), y_seq=None):
        self.sigma = float(sigma)
        self.seq = tuple(int(s) for s in (seq if np.iterable(seq) else (seq,)))
        ys = self.seq if y_seq is None else y_seq
        self.y_seq = tuple(int(s) for s in (ys if np.iterable(ys) else (ys,)))
        self._tmp1 = np.log(1.0 / (np.sqrt(2.0 * np.pi) * self.sigma))
        self._tmp2 = 2.0 * self.sigma * self.sigma

    def __call__(self, y: Observation, population: np.ndarray, theta: np.ndarray) -> float:
        ys = int(sum(int(y.val[i - 1]) for i in self.y_seq))
        xs = int(sum(int(population[i - 1]) for i in self.seq))
        return float(self._tmp1 - ((ys - xs) ** 2) / self._tmp2)

    def obs_table(self, n_compartments: int, n_obs_vals: int) -> ObsTable:
        xm = np.zeros(n_compartments, dtype=np.int64)
        ym = np.zeros(n_obs_vals, dtype=np.int64)
        for i in self.seq:
            xm[i - 1] += 1
        for i in self.y_seq:
            ym[i - 1] += 1
        return ObsTable(self.sigma, xm, ym)


def partial_gaussian_obs_model(sigma: float = 2.0, seq=(2,), y_seq=None) -> GaussianObsModel:
    """partial_gaussian_obs_model(σ = 2.0; seq = 2:2, y_seq = seq) (src/hmm_examples.jl:59-67)"""
    return GaussianObsModel(sigma, seq, y_seq)


class CountObsModel:
    """Count observation model: Y = sum(y.val[y_seq]) given X = sum(population[seq]) (1-based index lists, like
    GaussianObsModel) follows a Poisson, binomial or negative-binomial law (include/dpomp.h DPOMP_OBS_*).  A parameter is a
    fixed value or, with its *_index (0-based), the theta component of each filter / trajectory, so that pMCMC, SMC^2 and ARQ
    infer it.  Calls return the log pmf, like the reference's obs_model closures; `obs_table` is what the device evaluates."""

    def __init__(self, family: int, values, indices, seq=(2,), y_seq=None):
        self.family = int(family)
        self.par_value = tuple(float(v) for v in values)
        self.par_index = tuple(-1 if i is None else int(i) for i in indices)
        self.seq = tuple(int(s) for s in (seq if np.iterable(seq) else (seq,)))
        ys = self.seq if y_seq is None else y_seq
        self.y_seq = tuple(int(s) for s in (ys if np.iterable(ys) else (ys,)))
        if any(i < -1 for i in self.par_index):
            raise ValueError("parameter indices are 0-based theta components")
        ok = {_capi.OBS_POISSON: lambda a, k: a > 0.0, _capi.OBS_BINOMIAL: lambda a, k: 0.0 <= a <= 1.0,
              _capi.OBS_NEGBIN: lambda a, k: a > 0.0 and k > 0.0}[self.family]
        a, k = (v if i < 0 else 0.5 for v, i in zip(self.par_value, self.par_index))
        if not ok(a, k) or not all(np.isfinite(self.par_value)):
            raise ValueError(f"fixed observation parameters {self.par_value} outside their range")

    def __call__(self, y: Observation, population: np.ndarray, theta: np.ndarray) -> float:
        ys = int(sum(int(y.val[i - 1]) for i in self.y_seq))
        xs = int(sum(int(population[i - 1]) for i in self.seq))
        a, k = self.obs_table(len(population), len(y.val)).count_params(theta)
        return count_logpmf(self.family, ys, xs, a, k)

    def obs_table(self, n_compartments: int, n_obs_vals: int) -> ObsTable:
        xm = np.zeros(n_compartments, dtype=np.int64)
        ym = np.zeros(n_obs_vals, dtype=np.int64)
        for i in self.seq:
            xm[i - 1] = 1
        for i in self.y_seq:
            ym[i - 1] = 1
        return ObsTable(1.0, xm, ym, self.family, self.par_index, self.par_value)


def partial_poisson_obs_model(rho: float = 1.0, rho_index: Optional[int] = None, seq=(2,), y_seq=None) -> CountObsModel:
    """Cases reported at rate rho: Y ~ Poisson(rho * X), e.g. `logpdf(Poisson(theta[3] * pop[2]), y.val[2])` with
    rho_index = 2 (0-based)."""
    return CountObsModel(_capi.OBS_POISSON, (rho, 0.0), (rho_index, None), seq, y_seq)


def partial_binomial_obs_model(p: float = 1.0, p_index: Optional[int] = None, seq=(2,), y_seq=None) -> CountObsModel:
    """Each counted individual detected with probability p: Y ~ Binomial(X, p)."""
    return CountObsModel(_capi.OBS_BINOMIAL, (p, 0.0), (p_index, None), seq, y_seq)


def partial_negbin_obs_model(rho: float = 1.0, k: float = 1.0, rho_index: Optional[int] = None, k_index: Optional[int] = None,
                             seq=(2,), y_seq=None) -> CountObsModel:
    """Over-dispersed reporting: Y negative binomial with mean rho * X and size k (variance mu + mu^2 / k)."""
    return CountObsModel(_capi.OBS_NEGBIN, (rho, k), (rho_index, k_index), seq, y_seq)


def generate_model(model_name: str, initial_condition: Sequence[int], freq_dep: bool = False,
                   obs_error: float = 2.0) -> Optional[DPOMPModel]:
    """generate_model(model_name, initial_condition; freq_dep = false, obs_error = 2.0) (src/hmm_examples.jl:99-211)"""

    # density dependent (src/hmm_examples.jl:103-121)
    def si_rf(output, parameters, population):
        output[0] = parameters[0] * population[0] * population[1]

    def sir_rf(output, parameters, population):
        output[0] = parameters[0] * population[0] * population[1]
        output[1] = parameters[1] * population[1]

    def sei_rf(output, parameters, population):
        output[0] = parameters[0] * population[0] * population[2]
        output[1] = parameters[1] * population[1]

    def seir_rf(output, parameters, population):
        output[0] = parameters[0] * population[0] * population[2]
        output[1] = parameters[1] * population[1]
        output[2] = parameters[2] * population[2]

    # frequency dependent (src/hmm_examples.jl:126-144)
    def si_rf_fd(output, parameters, population):
        output[0] = parameters[0] * population[0] * population[1] / np.sum(population)

    def sir_rf_fd(output, parameters, population):
        output[0] = parameters[0] * population[0] * population[1] / np.sum(population)
        output[1] = parameters[1] * population[1]

    def sei_rf_fd(output, parameters, population):
        output[0] = parameters[0] * population[0] * population[2] / np.sum(population)
        output[1] = parameters[1] * population[1]

    def seir_rf_fd(output, parameters, population):
        output[0] = parameters[0] * population[0] * population[2] / np.sum(population)
        output[1] = parameters[1] * population[1]
        output[2] = parameters[2] * population[2]

    # Lotka-Volterra (src/hmm_examples.jl:149-154): state = (predator, prey)
    def lotka_rf(output, parameters, population):
        output[0] = parameters[0] * population[1]
        output[1] = parameters[1] * population[0] * population[1]
        output[2] = parameters[2] * population[0]

    # Ross-MacDonald (src/hmm_examples.jl:159-168)
    def rossmac_rf(output, parameters, population):
        output[0] = parameters[0] * (population[2] + population[3])
        output[1] = parameters[0] * population[2]
        output[2] = parameters[0] * population[3]
        output[3] = parameters[1] * (population[0] * population[3] / (population[0] + population[1]))
        output[4] = parameters[2] * (population[1] * population[2] / (population[2] + population[3]))
        output[5] = parameters[3] * population[1]

    if model_name == "SI":
        rate_fn = si_rf_fd if freq_dep else si_rf
        m_transition = [[-1, 1]]
        obs_model = partial_gaussian_obs_model(obs_error)
    elif model_name == "SIR":
        rate_fn = sir_rf_fd if freq_dep else sir_rf
        m_transition = [[-1, 1, 0], [0, -1, 1]]
        obs_model = partial_gaussian_obs_model(obs_error)
    elif model_name == "SIS":
        rate_fn = sir_rf_fd if freq_dep else sir_rf
        m_transition = [[-1, 1], [1, -1]]
        obs_model = partial_gaussian_obs_model(obs_error)
    elif model_name == "SEI":
        rate_fn = sei_rf_fd if freq_dep else sei_rf
        m_transition = [[-1, 1, 0], [0, -1, 1]]
        obs_model = partial_gaussian_obs_model(obs_error, seq=(3,))
    elif model_name == "SEIR":
        rate_fn = seir_rf_fd if freq_dep else seir_rf
        m_transition = [[-1, 1, 0, 0], [0, -1, 1, 0], [0, 0, -1, 1]]
        obs_model = partial_gaussian_obs_model(obs_error, seq=(3,))
    elif model_name == "SEIS":
        rate_fn = seir_rf_fd if freq_dep else seir_rf
        m_transition = [[-1, 1, 0], [0, -1, 1], [1, 0, -1]]
        obs_model = partial_gaussian_obs_model(obs_error, seq=(3,))
    elif model_name == "LOTKA":
        model_name = "PN"
        rate_fn = lotka_rf
        m_transition = [[0, 1], [1, -1], [-1, 0]]
        obs_model = partial_gaussian_obs_model(obs_error)
    elif model_name == "ROSSMAC":
        model_name = "SIAB"
        rate_fn = rossmac_rf
        m_transition = [[0, 0, 1, 0], [0, 0, -1, 0], [0, 0, 0, -1], [-1, 1, 0, 0], [0, 0, -1, 1], [1, -1, 0, 0]]
        obs_model = partial_gaussian_obs_model(obs_error)
    else:
        print(f" - SORRY: model name '{model_name}' not recognised.")  # src/hmm_examples.jl:205-207
        return None
    m_transition = np.asarray(m_transition, dtype=np.int64)
    prior = generate_weak_prior(m_transition.shape[0])
    return DPOMPModel(model_name, rate_fn, np.asarray(initial_condition, dtype=np.int64), m_transition, dmy_obs_fn,
                      obs_model, prior, 0)


def generate_custom_model(model_name: str, rate_function: Callable, initial_condition: Sequence[int],
                          m_transition: np.ndarray, obs_function: Callable = dmy_obs_fn, obs_error: float = 2.0,
                          obs_model: Optional[Callable] = None, prior=None, t0_index: int = 0) -> DPOMPModel:
    """generate_custom_model (src/hmm_examples.jl:237-239).  The reference's default `obs_model` passes a nonexistent
    `n=` keyword (SURVEY 8f); here the default is the plain partial_gaussian_obs_model(obs_error)."""
    m_transition = np.atleast_2d(np.asarray(m_transition, dtype=np.int64))
    if obs_model is None:
        obs_model = partial_gaussian_obs_model(obs_error)
    if prior is None:
        prior = generate_weak_prior(m_transition.shape[0])
    return DPOMPModel(model_name, rate_function, np.asarray(initial_condition, dtype=np.int64), m_transition,
                      obs_function, obs_model, prior, t0_index)
