"""The CPU oracle with the count observation families (dpomp_model_set_obs_model).  TEST INFRASTRUCTURE ONLY.

The reference oracle (oracle.py / liboracle.so) evaluates the Gaussian observation model only.  This module builds a second
library from the SAME oracle sources plus dpomp_oracle_count.c: the three observation calls of the oracle (the filter's log
weight in orc_pf_partial and the MBP iterate / propose log-likelihoods) are redirected, when a count family is selected, to
orcc_obs with the call's theta; every other line of the oracle is compiled unchanged.  The library is built in a temporary
directory keyed by the sources (the tree may be read-only) and the wrappers of oracle.py are reused against it: every wrapper
below first selects the family of the compiled model (`desc.obs_spec`, set by rate_table.build_model_desc; a descriptor
without it is Gaussian), so the selection never leaks from one call to the next.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import importlib.util
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_CFLAGS = ["-O3", "-std=gnu11", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math"]  # those of oracle/Makefile
_PROTO = ('#include "../include/dpomp.h"\n'
          "int orcc_family(void);\n"
          "double orcc_obs(const dpomp_model_desc* m, const double* th, int t, const int64_t* x);\n")
# (file, original text, redirected text): each original must occur exactly once, so a change of the oracle fails loudly here
_EDITS = [
    ("dpomp_oracle.c", "lw[p] = ovf ? -INFINITY : obs_model(m, t, x);",
     "lw[p] = ovf ? -INFINITY : (orcc_family() ? orcc_obs(m, theta, t, x) : obs_model(m, t, x));"),
    ("dpomp_oracle_mbp.c", "double out = obs_ll(m, t, fc);",
     "double out = orcc_family() ? orcc_obs(m, theta, t, fc) : obs_ll(m, t, fc);"),
    ("dpomp_oracle_mbp.c", "xf_loglike[1] = obs_ll(m, oi - 1, xf_fc);",
     "xf_loglike[1] = orcc_family() ? orcc_obs(m, theta_f, oi - 1, xf_fc) : obs_ll(m, oi - 1, xf_fc);"),
]
_SOURCES = ["dpomp_oracle.c", "dpomp_oracle_ibis.c", "dpomp_oracle_mbp.c", "dpomp_oracle_count.c"]
_lib = None
_base = None


def build() -> str:
    texts = {f: open(os.path.join(_HERE, f)).read() for f in _SOURCES}
    header = open(os.path.join(_HERE, "..", "include", "dpomp.h")).read()
    for f, old, new in _EDITS:
        if texts[f].count(old) != 1:
            raise RuntimeError(f"oracle/{f}: the observation call `{old}` is not there exactly once")
        texts[f] = _PROTO + texts[f].replace(old, new)
    h = hashlib.sha256((header + "".join(texts[f] for f in _SOURCES) + " ".join(_CFLAGS)).encode()).hexdigest()[:16]
    out_dir = os.path.join(tempfile.gettempdir(), f"dpomp_oracle_count_{h}")
    so = os.path.join(out_dir, "liboracle_count.so")
    if os.path.exists(so):
        return so
    os.makedirs(out_dir, exist_ok=True)
    paths = []
    for f in _SOURCES:
        p = os.path.join(out_dir, f)
        with open(p, "w") as fh:
            fh.write(texts[f])
        paths.append(p)
    cc = "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else "gcc"
    tmp = so + f".{os.getpid()}.tmp"
    # the sources include "../include/dpomp.h": resolved against -I oracle/ of the tree
    subprocess.run([cc, *_CFLAGS, "-I", _HERE, "-shared", "-o", tmp, *paths, "-lm"], check=True, capture_output=True)
    os.replace(tmp, so)
    return so


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.orc_compute_ess.restype = C.c_double
        _lib.orc_count_logpmf.restype = C.c_double
        _lib.orc_count_logpmf.argtypes = [C.c_int, C.c_int64, C.c_int64, C.c_double, C.c_double]
    return _lib


def _wrappers():
    """oracle.py loaded a second time, bound to the count library"""
    global _base
    if _base is None:
        spec = importlib.util.spec_from_file_location("_dpomp_oracle_count_wrappers", os.path.join(_HERE, "oracle.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod._lib = lib()
        _base = mod
    return _base


def _select(desc) -> None:
    family, idx, val = getattr(desc, "obs_spec", (0, (-1, -1), (0.0, 0.0)))
    i = np.ascontiguousarray(idx, dtype=np.int32)
    v = np.ascontiguousarray(val, dtype=np.float64)
    lib().orc_set_obs_model(int(family), i.ctypes.data_as(C.c_void_p), v.ctypes.data_as(C.c_void_p))


def count_logpmf(family: int, y: int, x: int, a: float, k: float = 0.0) -> float:
    """log pmf of a count family (include/dpomp.h DPOMP_OBS_*) in the oracle's C"""
    return float(lib().orc_count_logpmf(int(family), int(y), int(x), float(a), float(k)))


def max_threads() -> int:
    return _wrappers().max_threads()


def _with_family(name):
    def call(desc, *args, **kw):
        _select(desc)
        return getattr(_wrappers(), name)(desc, *args, **kw)
    call.__name__ = name
    call.__doc__ = f"oracle.{name} with the observation family of the compiled model"
    return call


pf_partial = _with_family("pf_partial")
pf_loglik = _with_family("pf_loglik")
pf_partial_batch = _with_family("pf_partial_batch")
run_pibis = _with_family("run_pibis")
run_pmcmc = _with_family("run_pmcmc")
mbp_iterate = _with_family("mbp_iterate")
mbp_propose = _with_family("mbp_propose")
run_mbp_ibis = _with_family("run_mbp_ibis")
MODE_LITERAL, MODE_DEVICE, MODE_DEVICE_INTERLEAVED = 0, 1, 2
