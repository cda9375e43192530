"""Compile the user-supplied model closures to the device rate table (struct dpomp_model_desc, include/dpomp.h).

The reference evaluates `rate_function(out, theta, x)`, `fn_transition(et)` and `obs_model(y, x, theta)` as Julia
closures inside the event loop (src/hmm_particle_filter.jl:20-29).  Closures cannot run on the device, so the host
PROBES them and fits the table

    rate[e] = theta[p_e] * (k1 + f1.x) * (k2 + f2.x) / (kd + dn.x)          (integer forms)
    log g   = log(1/(sqrt(2 pi) sigma)) - (ymask.y - xmask.x)^2 / (2 sigma^2)
          or  a Poisson / binomial / negative-binomial log pmf of Y = ymask.y given X = xmask.x (0/1 masks)

which covers every predefined model (src/hmm_examples.jl:103-168, incl. freq_dep and ROSSMAC) and the custom models of
the reference's tests (test/runtests.jl:74-100).  The fit is verified on random states; a closure that does not fit
raises ModelCompileError -- there is no CPU fallback.
"""
from __future__ import annotations

import itertools
from dataclasses import dataclass, field
from typing import Callable, List, Optional, Sequence

import numpy as np

import math

from . import _capi
from .structs import Observation


class ModelCompileError(ValueError):
    pass


@dataclass
class RateTable:
    n_compartments: int
    n_events: int
    n_params: int
    par: np.ndarray  # (E,) 0-based parameter index or -1
    f1: np.ndarray  # (E, C)
    k1: np.ndarray
    f2: np.ndarray
    k2: np.ndarray
    has_den: np.ndarray
    dn: np.ndarray
    kd: np.ndarray

    def evaluate(self, theta: np.ndarray, x: np.ndarray) -> np.ndarray:
        """Reference-order evaluation of the table (used only to verify the fit)."""
        out = np.zeros(self.n_events)
        for e in range(self.n_events):
            p = theta[self.par[e]] if self.par[e] >= 0 else 1.0
            l1 = float(self.k1[e] + int(self.f1[e] @ x))
            l2 = float(self.k2[e] + int(self.f2[e] @ x))
            r = (p * l1) * l2
            if self.has_den[e]:
                d = self.kd[e] + int(self.dn[e] @ x)
                r = 0.0 if d == 0 else r / float(d)
            out[e] = r
        return out


@dataclass
class ObsTable:
    sigma: float
    xmask: np.ndarray  # (C,)
    ymask: np.ndarray  # (V,)
    # observation family (include/dpomp.h DPOMP_OBS_*); count families: parameter i is theta[par_index[i]] (0-based) or,
    # for par_index[i] = -1, the fixed par_value[i]; Poisson (rho, -), binomial (p, -), negative binomial (rho, k)
    family: int = _capi.OBS_GAUSSIAN
    par_index: tuple = (-1, -1)
    par_value: tuple = (0.0, 0.0)

    def count_params(self, theta) -> tuple:
        """(a, k) of a count family at theta: a = rho or p, k = negative-binomial size."""
        return tuple(float(theta[i]) if i >= 0 else float(v) for i, v in zip(self.par_index, self.par_value))


def count_logpmf(family: int, y: int, x: int, a: float, k: float = 0.0) -> float:
    """log g(Y = y | X = x) of a count family with the boundary cases of include/dpomp.h: 0 log 0 = 0, a zero mean gives 0 for
    y = 0 and -inf otherwise, y > x in the binomial gives -inf, p = 0 / 1 are exact, a parameter out of range gives -inf.  Same
    association as the device code and the oracle."""
    y, x = int(y), int(x)
    if y < 0:
        return -math.inf
    yf, xf = float(y), float(x)
    if family == _capi.OBS_POISSON:
        if not (0.0 < a < math.inf):
            return -math.inf
        if x == 0:
            return 0.0 if y == 0 else -math.inf
        ylog = 0.0 if y == 0 else yf * (math.log(a) + math.log(xf))
        return (ylog - a * xf) - math.lgamma(yf + 1.0)
    if family == _capi.OBS_BINOMIAL:
        if not (0.0 <= a <= 1.0) or y > x:
            return -math.inf
        if a == 0.0:
            return 0.0 if y == 0 else -math.inf
        if a == 1.0:
            return 0.0 if y == x else -math.inf
        nx = xf - yf
        r = (math.lgamma(xf + 1.0) - math.lgamma(yf + 1.0)) - math.lgamma(nx + 1.0)
        return (r + yf * math.log(a)) + nx * math.log1p(-a)
    if family == _capi.OBS_NEGBIN:
        if not (0.0 < a < math.inf) or not (0.0 < k < math.inf):
            return -math.inf
        if x == 0:
            return 0.0 if y == 0 else -math.inf
        mu = a * xf
        km = k + mu
        r = ((math.lgamma(yf + k) - math.lgamma(k)) - math.lgamma(yf + 1.0)) + k * math.log(k / km)
        return r if y == 0 else r + yf * math.log(mu / km)
    raise ValueError(f"unknown count family {family}")


def _call_rates(fn: Callable, n_events: int, theta: np.ndarray, x: np.ndarray) -> np.ndarray:
    out = np.zeros(n_events, dtype=np.float64)
    fn(out, np.asarray(theta, dtype=np.float64), np.asarray(x, dtype=np.int64))
    return out


def _monomials(x: np.ndarray) -> np.ndarray:
    c = len(x)
    quad = [x[a] * x[b] for a in range(c) for b in range(a, c)]
    return np.concatenate(([1.0], x.astype(np.float64), np.asarray(quad, dtype=np.float64)))


def _fit_quadratic(points: np.ndarray, vals: np.ndarray, n_c: int, tol: float = 1e-7) -> Optional[np.ndarray]:
    """Least-squares fit of an integer-coefficient quadratic polynomial; None if it does not fit."""
    a = np.stack([_monomials(p) for p in points])
    coef, *_ = np.linalg.lstsq(a, vals, rcond=None)
    rounded = np.round(coef)
    if np.max(np.abs(coef - rounded)) > tol:
        return None
    if np.max(np.abs(a @ rounded - vals)) > tol * max(1.0, np.max(np.abs(vals))):
        return None
    return rounded.astype(np.int64)


def _poly_of_forms(k1, f1, k2, f2) -> np.ndarray:
    c = len(f1)
    const = k1 * k2
    lin = [k1 * f2[a] + k2 * f1[a] for a in range(c)]
    quad = []
    for a in range(c):
        for b in range(a, c):
            quad.append(f1[a] * f2[a] if a == b else f1[a] * f2[b] + f1[b] * f2[a])
    return np.asarray([const] + lin + quad, dtype=np.int64)


def _factor_quadratic(poly: np.ndarray, n_c: int):
    """Write an integer quadratic polynomial as (k1 + f1.x)(k2 + f2.x); L1 has 0/1 coefficients."""
    lin = poly[1 : 1 + n_c]
    quad = poly[1 + n_c :]
    if not np.any(quad):  # affine: L2 = 1
        return int(poly[0]), lin.copy(), 1, np.zeros(n_c, dtype=np.int64)
    # candidate L1 with 0/1 coefficients (sums of compartments, optional +1); L2 by matching coefficients
    qmat = np.zeros((n_c, n_c), dtype=np.int64)
    it = iter(quad)
    for a in range(n_c):
        for b in range(a, n_c):
            qmat[a, b] = next(it)
    for bits in itertools.product((0, 1), repeat=n_c + 1):
        k1, f1 = bits[0], np.asarray(bits[1:], dtype=np.int64)
        if not np.any(f1):
            continue
        a0 = int(np.argmax(f1))  # first compartment in L1: x_a0^2 coefficient gives f2[a0]
        f2 = np.zeros(n_c, dtype=np.int64)
        f2[a0] = qmat[a0, a0]
        ok = True
        for b in range(n_c):
            if b == a0:
                continue
            lo, hi = min(a0, b), max(a0, b)
            # coefficient of x_a0 x_b = f1[a0] f2[b] + f1[b] f2[a0]
            f2[b] = qmat[lo, hi] - f1[b] * f2[a0]
        # k2 from the linear coefficient of x_a0: k1 f2[a0] + k2 f1[a0]
        k2 = int(lin[a0] - k1 * f2[a0])
        if np.array_equal(_poly_of_forms(k1, f1, k2, f2), poly) and ok:
            # canonical order: the factor whose leading compartment has the lower index comes first, which is how the
            # reference writes its mass-action products (theta * x_a * x_b with a < b, src/hmm_examples.jl:107-154)
            if np.any(f2) and int(np.argmax(f2 != 0)) < int(np.argmax(f1 != 0)):
                return int(k2), f2, int(k1), f1
            return int(k1), f1, int(k2), f2
    return None


def compile_rate_table(rate_function: Callable, n_events: int, n_params: int, n_compartments: int,
                       rng: Optional[np.random.Generator] = None) -> RateTable:
    rng = rng or np.random.default_rng(20261018)
    c, e_n = n_compartments, n_events
    if not (1 <= c <= _capi.MAX_COMPARTMENTS and 1 <= e_n <= _capi.MAX_EVENTS and 1 <= n_params <= _capi.MAX_PARAMS):
        raise ModelCompileError(f"model size (C={c}, E={e_n}, n_theta={n_params}) exceeds the device table limits")
    tab = RateTable(c, e_n, n_params, -np.ones(e_n, dtype=np.int64), np.zeros((e_n, c), dtype=np.int64),
                    np.zeros(e_n, dtype=np.int64), np.zeros((e_n, c), dtype=np.int64), np.ones(e_n, dtype=np.int64),
                    np.zeros(e_n, dtype=np.int64), np.zeros((e_n, c), dtype=np.int64), np.zeros(e_n, dtype=np.int64))
    theta0 = rng.uniform(0.5, 1.5, size=n_params)
    x0 = rng.integers(3, 20, size=c)
    r0 = _call_rates(rate_function, e_n, theta0, x0)
    # 1. which parameter multiplies each rate
    for e in range(e_n):
        if r0[e] == 0.0:
            raise ModelCompileError(f"event {e + 1}: rate is zero at a strictly positive state; cannot probe")
        hits = []
        for p in range(n_params):
            th = theta0.copy()
            th[p] *= 2.0
            ratio = _call_rates(rate_function, e_n, th, x0)[e] / r0[e]
            if abs(ratio - 2.0) < 1e-9:
                hits.append(p)
            elif abs(ratio - 1.0) > 1e-9:
                raise ModelCompileError(f"event {e + 1}: rate is not linear in theta[{p + 1}]")
        if len(hits) > 1:
            raise ModelCompileError(f"event {e + 1}: rate depends on more than one parameter {hits}")
        tab.par[e] = hits[0] if hits else -1
    # 2. state dependence with the parameter set to one
    ones = np.ones(n_params)
    n_mono = 1 + c + c * (c + 1) // 2
    pts = rng.integers(1, 12, size=(3 * n_mono + 8, c))
    vals = np.stack([_call_rates(rate_function, e_n, ones, p) for p in pts])  # (npts, E)
    den_candidates: List[Optional[np.ndarray]] = [None]
    for k in range(c, 1, -1):
        for idx in itertools.combinations(range(c), k):
            d = np.zeros(c, dtype=np.int64)
            d[list(idx)] = 1
            den_candidates.append(d)
    for e in range(e_n):
        done = False
        for dn in den_candidates:
            scaled = vals[:, e] if dn is None else vals[:, e] * (pts @ dn)
            poly = _fit_quadratic(pts, scaled, c)
            if poly is None:
                continue
            fac = _factor_quadratic(poly, c)
            if fac is None:
                continue
            tab.k1[e], tab.f1[e], tab.k2[e], tab.f2[e] = fac
            if dn is not None:
                tab.has_den[e], tab.dn[e] = 1, dn
            done = True
            break
        if not done:
            raise ModelCompileError(
                f"event {e + 1}: rate is not of the form theta_p * L1(x) * L2(x) / D(x) with small integer forms")
    # 3. verify on fresh random points (values of the closure vs the table)
    for _ in range(64):
        th = rng.uniform(0.01, 2.0, size=n_params)
        x = rng.integers(1, 200, size=c)
        want = _call_rates(rate_function, e_n, th, x)
        got = tab.evaluate(th, x)
        if not np.allclose(got, want, rtol=1e-12, atol=0.0):
            raise ModelCompileError(f"rate table verification failed at theta={th}, x={x}: {got} vs {want}")
    return tab


def compile_obs_table(obs_model: Callable, n_compartments: int, n_obs_vals: int, n_params: int) -> ObsTable:
    """Fit the observation table: the Gaussian first, then the count families.  Objects produced by
    partial_gaussian_obs_model and the partial_*_obs_model count constructors carry it directly."""
    direct = getattr(obs_model, "obs_table", None)
    if direct is not None:
        return direct(n_compartments, n_obs_vals)
    try:
        tab = _fit_gaussian_obs(obs_model, n_compartments, n_obs_vals, n_params)
    except (ArithmeticError, ValueError):  # a count law: -inf / degenerate values at the Gaussian probe points
        tab = None
    if tab is None:
        tab = _fit_count_obs(obs_model, n_compartments, n_obs_vals, n_params)
    if tab is None:
        raise ModelCompileError("obs_model is not a Gaussian in integer masks of (y, x), nor a Poisson, binomial or negative-binomial "
                                "law of 0/1 masks; no device table")
    return tab


def _fit_gaussian_obs(obs_model: Callable, n_compartments: int, n_obs_vals: int, n_params: int) -> Optional[ObsTable]:
    c, v = n_compartments, n_obs_vals
    theta = np.ones(n_params)

    def g(yv, xv):
        return float(obs_model(Observation(0.0, 1, 1.0, np.asarray(yv, dtype=np.int64)),
                               np.asarray(xv, dtype=np.int64), theta))

    zero_y, zero_x = np.zeros(v, dtype=np.int64), np.zeros(c, dtype=np.int64)
    a = g(zero_y, zero_x)
    sigma = float(np.exp(-a) / np.sqrt(2.0 * np.pi))
    b = 2.0 * sigma * sigma
    xm, ym = np.zeros(c, dtype=np.int64), np.zeros(v, dtype=np.int64)
    for i in range(c):
        x = zero_x.copy(); x[i] = 1
        xm[i] = int(round(np.sqrt(max(0.0, (a - g(zero_y, x)) * b))))
    for j in range(v):
        y = zero_y.copy(); y[j] = 1
        ym[j] = int(round(np.sqrt(max(0.0, (a - g(y, zero_x)) * b))))
    # relative signs within x (and within y) from pairwise probes: (m_i + s m_j)^2
    def _signs(mask, probe):
        nz = [i for i in range(len(mask)) if mask[i] != 0]
        for i in nz[1:]:
            z = np.zeros(len(mask), dtype=np.int64); z[nz[0]] = 1; z[i] = 1
            if abs((a - probe(z)) * b - (mask[nz[0]] + mask[i]) ** 2) > 1e-6:
                mask[i] = -mask[i]
    _signs(xm, lambda z: g(zero_y, z))
    _signs(ym, lambda z: g(z, zero_x))
    tab = ObsTable(sigma, xm, ym)
    rng = np.random.default_rng(7)
    tmp1, tmp2 = np.log(1.0 / (np.sqrt(2.0 * np.pi) * sigma)), 2.0 * sigma * sigma
    for _ in range(64):
        y = rng.integers(0, 50, size=v); x = rng.integers(0, 50, size=c)
        want = g(y, x)
        d = int(ym @ y) - int(xm @ x)
        if not np.isclose(tmp1 - d * d / tmp2, want, rtol=1e-10, atol=1e-12):
            return None
    return tab


def _snap(v: float) -> float:
    """a probed parameter read back through exp / log: the nearby 12-digit decimal when it is that value up to rounding"""
    s = float(f"{v:.12g}")
    return s if abs(s - v) <= 1e-12 * abs(v) else v


def _fit_count_obs(obs_model: Callable, n_compartments: int, n_obs_vals: int, n_params: int) -> Optional[ObsTable]:
    """Probe a closure for a count law: 0/1 masks from the components that move its value, the parameters from a few probe
    points (g(0, X) = -rho X for the Poisson, g(1, 1) = log p for the binomial, g(1, X) - g(0, X) = log(k mu / (k + mu)) at
    X = 1, 2 for the negative binomial), theta-indexing by perturbing each theta component, then 64 random verification points."""
    c, v = n_compartments, n_obs_vals
    rng = np.random.default_rng(11)
    theta0 = rng.uniform(0.2, 0.8, size=n_params)

    def g(yv, xv, th):
        with np.errstate(all="ignore"):
            return float(obs_model(Observation(0.0, 1, 1.0, np.asarray(yv, dtype=np.int64)), np.asarray(xv, dtype=np.int64),
                                   np.asarray(th, dtype=np.float64)))

    try:
        # 1. masks: components whose unit change moves the value at an interior point (Y well below X)
        x0, y0 = np.full(c, 50, dtype=np.int64), np.ones(v, dtype=np.int64)
        base = g(y0, x0, theta0)
        if not math.isfinite(base):
            return None
        xm = np.zeros(c, dtype=np.int64)
        ym = np.zeros(v, dtype=np.int64)
        for i in range(c):
            x = x0.copy(); x[i] += 1
            xm[i] = int(g(y0, x, theta0) != base)
        for j in range(v):
            y = y0.copy(); y[j] += 1
            ym[j] = int(g(y, x0, theta0) != base)
        if not xm.any() or not ym.any():
            return None
        ix, iy = int(np.argmax(xm)), int(np.argmax(ym))

        def G(yy, xx, th):  # Y in the first y component of the mask, X in the first x component, the rest zero
            y = np.zeros(v, dtype=np.int64); y[iy] = yy
            x = np.zeros(c, dtype=np.int64); x[ix] = xx
            return g(y, x, th)

        # 2. parameters of each family at theta, None if the probe values are not those of the family
        def fit(family, th):
            if family == _capi.OBS_POISSON:
                return (-G(0, 1, th), 0.0)
            if family == _capi.OBS_BINOMIAL:
                return (math.exp(G(1, 1, th)), 0.0)
            e1 = math.exp(-(G(1, 1, th) - G(0, 1, th)))
            e2 = math.exp(-(G(1, 2, th) - G(0, 2, th)))
            inv_rho, inv_k = 2.0 * (e1 - e2), 2.0 * e2 - e1
            return (1.0 / inv_rho, 1.0 / inv_k)

        for family in (_capi.OBS_POISSON, _capi.OBS_BINOMIAL, _capi.OBS_NEGBIN):
            n_par = 2 if family == _capi.OBS_NEGBIN else 1
            try:
                vals = fit(family, theta0)
            except (ArithmeticError, ValueError):
                continue
            if not all(math.isfinite(vals[i]) for i in range(n_par)):
                continue
            # 3. theta-indexing: a parameter equal to theta[j] that follows a perturbation of theta[j]
            idx, fixed = [-1, -1], [0.0, 0.0]
            for i in range(n_par):
                for jth in range(n_params):
                    if not math.isclose(vals[i], theta0[jth], rel_tol=1e-9):
                        continue
                    th = theta0.copy(); th[jth] *= 0.9
                    try:
                        moved = fit(family, th)[i]
                    except (ArithmeticError, ValueError):
                        continue
                    if math.isclose(moved, th[jth], rel_tol=1e-9):
                        idx[i] = jth
                        break
                if idx[i] < 0:
                    fixed[i] = _snap(vals[i])
            tab = ObsTable(1.0, xm, ym, family, tuple(idx), tuple(fixed))
            # 4. verification on random points (scipy / lgamma closures agree with the table to rounding)
            ok = True
            vrng = np.random.default_rng(7)
            for _ in range(64):
                y = vrng.integers(0, 20, size=v); x = vrng.integers(0, 60, size=c)
                th = vrng.uniform(0.2, 0.8, size=n_params)
                want = g(y, x, th)
                got = count_logpmf(family, int(ym @ y), int(xm @ x), *tab.count_params(th))
                if not (got == want or np.isclose(got, want, rtol=1e-9, atol=1e-9)):
                    ok = False
                    break
            if ok:
                return tab
    except (ArithmeticError, ValueError, TypeError, IndexError):
        return None
    return None


@dataclass
class CompiledModel:
    """dpomp_model_desc plus the numpy buffers its pointers refer to (kept alive here)."""

    desc: "_capi.ModelDesc"
    obs_time: np.ndarray
    obs_id: np.ndarray
    obs_val: np.ndarray
    rate: RateTable = field(repr=False, default=None)
    obs: ObsTable = field(repr=False, default=None)


def build_model_desc(rate: RateTable, obs: ObsTable, m_transition: np.ndarray, initial_condition: Sequence[int],
                     t0_index: int, obs_data: Sequence[Observation]) -> CompiledModel:
    import ctypes as C

    c, e_n = rate.n_compartments, rate.n_events
    trans = np.atleast_2d(np.asarray(m_transition, dtype=np.int64))
    if trans.shape != (e_n, c):
        raise ModelCompileError(f"m_transition has shape {trans.shape}, expected ({e_n}, {c})")
    d = _capi.ModelDesc()
    d.n_compartments, d.n_events, d.n_params, d.t0_index = c, e_n, rate.n_params, int(t0_index)
    for e in range(e_n):
        d.rate_par[e] = int(rate.par[e])
        d.rate_k1[e], d.rate_k2[e] = int(rate.k1[e]), int(rate.k2[e])
        d.rate_has_den[e], d.rate_kd[e] = int(rate.has_den[e]), int(rate.kd[e])
        for k in range(c):
            d.rate_f1[e][k], d.rate_f2[e][k] = int(rate.f1[e, k]), int(rate.f2[e, k])
            d.rate_dn[e][k] = int(rate.dn[e, k])
            d.trans[e][k] = int(trans[e, k])
    for e in range(e_n, _capi.MAX_EVENTS):
        d.rate_par[e] = -1
    for k in range(c):
        d.initial_condition[k] = int(initial_condition[k])
        d.obs_xmask[k] = int(obs.xmask[k])
    d.obs_sigma = float(obs.sigma)
    # the count-family oracle (oracle/count_oracle.py) reads the observation family from here; the device model gets it through
    # dpomp_model_set_obs_model (particle_filter.DeviceModel)
    d.obs_spec = (int(obs.family), tuple(int(i) for i in obs.par_index), tuple(float(p) for p in obs.par_value))
    n_t = len(obs_data)
    v = len(obs_data[0].val) if n_t else 1
    if not (1 <= v <= _capi.MAX_OBS_VALS):
        raise ModelCompileError(f"observation vectors of length {v} exceed the device table limit")
    d.n_obs_vals = v
    for j in range(v):
        d.obs_ymask[j] = int(obs.ymask[j]) if j < len(obs.ymask) else 0
    times = np.ascontiguousarray([o.time for o in obs_data], dtype=np.float64)
    ids = np.ascontiguousarray([o.obs_id for o in obs_data], dtype=np.int32)
    vals = np.ascontiguousarray(np.stack([o.val for o in obs_data]) if n_t else np.zeros((0, v)), dtype=np.int64)
    d.n_obs = n_t
    d.obs_time = times.ctypes.data_as(C.POINTER(C.c_double))
    d.obs_id = ids.ctypes.data_as(C.POINTER(C.c_int32))
    d.obs_val = vals.ctypes.data_as(C.POINTER(C.c_int64))
    return CompiledModel(d, times, ids, vals, rate, obs)
