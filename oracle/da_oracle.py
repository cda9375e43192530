"""The CPU oracle of data-augmented MCMC (dpomp_da_loglike / dpomp_da_step).  TEST INFRASTRUCTURE ONLY.

Builds one more library, in a temporary directory keyed by the sources (the tree may be read-only): the sources of the
count-family oracle (count_oracle.py: the unchanged oracle sources with their observation calls redirected, plus
dpomp_oracle_count.c) and dpomp_oracle_da.c.  So the MBP walks that generate the starting trajectories and the full
log-likelihood of the data-augmented sampler use the observation law of the compiled model, Gaussian or count.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import importlib.util
import os
import subprocess
import tempfile

import numpy as np

from . import count_oracle as _co

_HERE = os.path.dirname(os.path.abspath(__file__))
_DA = "dpomp_oracle_da.c"
_lib = None
_base = None


def build() -> str:
    texts = {f: open(os.path.join(_HERE, f)).read() for f in _co._SOURCES + [_DA]}
    header = open(os.path.join(_HERE, "..", "include", "dpomp.h")).read()
    for f, old, new in _co._EDITS:
        if texts[f].count(old) != 1:
            raise RuntimeError(f"oracle/{f}: the observation call `{old}` is not there exactly once")
        texts[f] = _co._PROTO + texts[f].replace(old, new)
    names = _co._SOURCES + [_DA]
    h = hashlib.sha256((header + "".join(texts[f] for f in names) + " ".join(_co._CFLAGS)).encode()).hexdigest()[:16]
    out_dir = os.path.join(tempfile.gettempdir(), f"dpomp_oracle_da_{h}")
    so = os.path.join(out_dir, "liboracle_da.so")
    if os.path.exists(so):
        return so
    os.makedirs(out_dir, exist_ok=True)
    paths = []
    for f in names:
        p = os.path.join(out_dir, f)
        with open(p, "w") as fh:
            fh.write(texts[f])
        paths.append(p)
    cc = "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else "gcc"
    tmp = so + f".{os.getpid()}.tmp"
    subprocess.run([cc, *_co._CFLAGS, "-I", _HERE, "-shared", "-o", tmp, *paths, "-lm"], check=True, capture_output=True)
    os.replace(tmp, so)
    return so


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.orc_compute_ess.restype = C.c_double
    return _lib


def _wrappers():
    """oracle.py loaded once more, bound to this library"""
    global _base
    if _base is None:
        spec = importlib.util.spec_from_file_location("_dpomp_oracle_da_wrappers", os.path.join(_HERE, "oracle.py"))
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


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def mbp_iterate(desc, *args, **kw):
    """oracle.mbp_iterate with the observation family of the compiled model"""
    _select(desc)
    return _wrappers().mbp_iterate(desc, *args, **kw)


def da_loglike(desc, theta, times, types):
    """full log-likelihood of one trajectory (types 1-based).  Returns ({full, observation}, final state)."""
    _select(desc)
    th = np.ascontiguousarray(theta, dtype=np.float64)
    t = np.ascontiguousarray(times, dtype=np.float64); y = np.ascontiguousarray(types, dtype=np.int32)
    fc = np.zeros(desc.n_compartments, dtype=np.int64); ll = np.zeros(2)
    lib().orc_da_loglike(C.byref(desc), _p(th), _p(t), _p(y), C.c_int64(len(t)), _p(fc), _p(ll))
    return ll, fc


def da_props(desc, theta, times, types, length, max_traj, traj_props, mvp, key, cid):
    """traj_props trajectory proposals of chain `cid` (global id) with call key `key`, applied in place to the flat arrays
    times / types (f64 / int32, room for length + traj_props events).  Returns (new length, final state, {full, observation},
    accepted [inserts, deletes, moves])."""
    _select(desc)
    th = np.ascontiguousarray(theta, dtype=np.float64)
    assert times.dtype == np.float64 and types.dtype == np.int32 and len(times) >= length + traj_props
    ln = C.c_int64(int(length))
    fc = np.zeros(desc.n_compartments, dtype=np.int64); ll = np.zeros(2); acc = np.zeros(3, dtype=np.int64)
    lib().orc_da_props(C.byref(desc), _p(th), _p(times), _p(types), C.byref(ln), C.c_int64(int(max_traj)), int(traj_props),
                       int(mvp), C.c_uint64(int(key)), C.c_uint32(int(cid)), _p(fc), _p(ll), _p(acc))
    return ln.value, fc, ll, acc
