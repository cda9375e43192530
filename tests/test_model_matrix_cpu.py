"""CPU tests of the instantiation matrix: which kernel a model gets (dpomp_model_builtin_id), and a guard that every compiled
instantiation of csrc/ has a case in tests/test_gpu_model_matrix.py, landing on the shape it is meant for."""
import ctypes as C
import os
import re
import sys

import numpy as np
import pytest

import test_gpu_model_matrix as gm
from conftest import ROOT

CSRC = os.path.join(ROOT, "discretepomp.jl_b200", "csrc")
IDS = gm.BUILTIN_IDS


def _xmacro(fname, macro):
    """the entries of the one-line X-macro list `#define macro(X) X(...) X(...)` as tuples of strings"""
    src = open(os.path.join(CSRC, fname)).read()
    m = re.search(r"^#define %s\(X\)((?:\s*X\([^)]*\))+)\s*$" % macro, src, flags=re.M)
    assert m, f"{macro} not found in {fname}"
    return [tuple(a.strip() for a in e.split(",")) for e in re.findall(r"X\(([^)]*)\)", m.group(1))]


def sim_shapes():
    return [(int(c), int(e)) for c, e in _xmacro("pf_sim.cuh", "DPOMP_SIM_SHAPES")]


def shape_of(shapes, c, e):
    """the dispatch rule of sim_shaped: the first listed shape that covers (c, e)"""
    return next(((cc, ee) for cc, ee in shapes if c <= cc and e <= ee), None)


def _model_id(dp, model, y=None):
    y = y or [dp.Observation(1.0, 1, 1.0, [0] * len(model.initial_condition))]
    dm = dp.device_model(dp.get_private_model(model, y))
    return gm.builtin_id(dp, dm), dm


# ---- which kernel a model gets ------------------------------------------------------------------------------------------
PREDEF_IC = {"SI": [10, 1], "SIR": [100, 1, 0], "SIS": [100, 1], "SEI": [10, 1, 1], "SEIR": [100, 0, 1, 0], "SEIS": [10, 1, 1],
             "LOTKA": [70, 70]}


@pytest.mark.parametrize("name", list(PREDEF_IC))
def test_predefined_models_are_recognised(built_lib, dp, name):
    assert _model_id(dp, dp.generate_model(name, PREDEF_IC[name]))[0] == IDS[name]


@pytest.mark.parametrize("name", ["SI", "SIR", "SIS", "SEI", "SEIR", "SEIS"])
def test_frequency_dependent_variants_run_the_generic_table(built_lib, dp, name):
    assert _model_id(dp, dp.generate_model(name, PREDEF_IC[name], freq_dep=True))[0] == 0


def test_rossmac_runs_the_generic_table(built_lib, dp):
    assert _model_id(dp, dp.generate_model("ROSSMAC", [10, 1, 10, 1]))[0] == 0


# closures that restate each predefined model, and the permutation of their parameters that must not be taken for it
CLOSURES = {
    "SI": (lambda o, p, x: o.__setitem__(0, p[0] * x[0] * x[1]), [[-1, 1]], None),
    "SIR": (lambda o, p, x: (o.__setitem__(0, p[0] * x[0] * x[1]), o.__setitem__(1, p[1] * x[1])), [[-1, 1, 0], [0, -1, 1]], (1, 0)),
    "SIS": (lambda o, p, x: (o.__setitem__(0, p[0] * x[0] * x[1]), o.__setitem__(1, p[1] * x[1])), [[-1, 1], [1, -1]], (1, 0)),
    "SEI": (lambda o, p, x: (o.__setitem__(0, p[0] * x[0] * x[2]), o.__setitem__(1, p[1] * x[1])), [[-1, 1, 0], [0, -1, 1]], (1, 0)),
    "SEIR": (lambda o, p, x: (o.__setitem__(0, p[0] * x[0] * x[2]), o.__setitem__(1, p[1] * x[1]), o.__setitem__(2, p[2] * x[2])),
             [[-1, 1, 0, 0], [0, -1, 1, 0], [0, 0, -1, 1]], (2, 0, 1)),
    "SEIS": (lambda o, p, x: (o.__setitem__(0, p[0] * x[0] * x[2]), o.__setitem__(1, p[1] * x[1]), o.__setitem__(2, p[2] * x[2])),
             [[-1, 1, 0], [0, -1, 1], [1, 0, -1]], (1, 2, 0)),
    "LOTKA": (lambda o, p, x: (o.__setitem__(0, p[0] * x[1]), o.__setitem__(1, p[1] * x[0] * x[1]), o.__setitem__(2, p[2] * x[0])),
              [[0, 1], [1, -1], [-1, 0]], (0, 2, 1)),
}


@pytest.mark.parametrize("name", list(CLOSURES))
def test_custom_closures_of_a_predefined_model(built_lib, dp, name):
    """A user-written closure that is algebraically the predefined model, with the same parameter order, gets the predefined
    kernels; the same closure reading its parameters in another order does not.  With a count observation family every
    model runs the generic table."""
    rf, rows, perm = CLOSURES[name]
    ic = PREDEF_IC[name]
    n_par = len(rows)
    model = dp.generate_custom_model(name, rf, ic, rows, prior=dp.generate_weak_prior(n_par))
    assert _model_id(dp, model)[0] == IDS[name]
    if perm is not None:
        permuted = lambda o, p, x: rf(o, np.asarray(p)[list(perm)], x)
        assert _model_id(dp, dp.generate_custom_model(name, permuted, ic, rows, prior=dp.generate_weak_prior(n_par)))[0] == 0
    counted = dp.generate_custom_model(name, rf, ic, rows, obs_model=dp.partial_poisson_obs_model(0.5), prior=dp.generate_weak_prior(n_par))
    ident, dm = _model_id(dp, counted)
    assert dm.compiled.obs.family == gm.POISSON and ident == 0


def test_builtin_id_rejects_null_arguments(built_lib, dp):
    out = C.c_int32()
    assert built_lib.dpomp_model_builtin_id(None, C.byref(out)) == -1
    dm = _model_id(dp, dp.generate_model("SIR", [100, 1, 0]))[1]
    assert built_lib.dpomp_model_builtin_id(dm.handle, None) == -1


# ---- every instantiation has a case -----------------------------------------------------------------------------------------
def _model_names(entries):
    """kModelSI -> SI, kModelGeneric -> None"""
    out = []
    for (e,) in entries:
        assert e.startswith("kModel"), e
        out.append(None if e == "kModelGeneric" else e[len("kModel"):])
    return out


def builtin_models():
    """DPOMP_BUILTIN_MODELS (dpomp_models.cuh): the filter, the MBP walks and the DA walks are instantiated for each entry"""
    return _model_names(_xmacro("dpomp_models.cuh", "DPOMP_BUILTIN_MODELS"))


def _generic_shape(name):
    return shape_of(sim_shapes(), len(gm.GENERIC[name][2]), len(gm.GENERIC[name][1]))


def test_every_builtin_model_has_a_filter_case():
    names = builtin_models()
    assert None not in names and sorted(names) == sorted(IDS)
    for nm in names:
        assert nm in gm.CASES and nm in gm.FILTER_VARIANT_MODELS, nm


def test_every_generic_shape_has_a_gaussian_and_a_count_case():
    shapes = sim_shapes()
    assert len(shapes) == len(set(shapes)) and shapes
    gaussian = {_generic_shape(g) for g in gm.GENERIC if g in gm.CASES}
    poisson = {_generic_shape(g) for g, f in gm.COUNT_CASES if f == gm.POISSON}
    for s in shapes:
        assert s in gaussian, f"shape {s} of DPOMP_SIM_SHAPES has no Gaussian case in test_gpu_model_matrix.py"
        assert s in poisson, f"shape {s} of DPOMP_SIM_SHAPES has no Poisson case in test_gpu_model_matrix.py"


@pytest.mark.parametrize("walk,cases", [("mbp", gm.MBP_MODELS), ("da", gm.DA_MODELS)], ids=["mbp", "da"])
def test_every_walk_instantiation_has_a_case(walk, cases):
    """the walks are instantiated for every predefined model and for the generic rate table (with_walk_model, mbp_walk.cuh)"""
    for nm in builtin_models():
        assert nm in IDS and nm in cases, (walk, nm)
    assert any(c in gm.GENERIC for c in cases), walk


def test_guard_fails_for_an_instantiation_without_a_case(tmp_path, monkeypatch):
    """the guard itself: a shape added to the list is reported, and a predefined model added to the list is reported for the
    filter and for both walks"""
    src = open(os.path.join(CSRC, "pf_sim.cuh")).read()
    added = re.sub(r"(#define DPOMP_SIM_SHAPES\(X\)[^\n]*)", r"\1 X(6, 4)", src, count=1)
    (tmp_path / "pf_sim.cuh").write_text(added)
    models = open(os.path.join(CSRC, "dpomp_models.cuh")).read()
    (tmp_path / "dpomp_models.cuh").write_text(re.sub(r"(#define DPOMP_BUILTIN_MODELS\(X\)[^\n]*)", r"\1 X(kModelSIRS)", models, count=1))
    monkeypatch.setattr(sys.modules[__name__], "CSRC", str(tmp_path))
    assert (6, 4) in sim_shapes() and "SIRS" in builtin_models()
    with pytest.raises(AssertionError, match=r"\(6, 4\)"):
        test_every_generic_shape_has_a_gaussian_and_a_count_case()
    with pytest.raises(AssertionError):
        test_every_builtin_model_has_a_filter_case()
    for walk, cases in (("mbp", gm.MBP_MODELS), ("da", gm.DA_MODELS)):
        with pytest.raises(AssertionError, match="SIRS"):
            test_every_walk_instantiation_has_a_case(walk, cases)


# ---- the shape each generic case runs on --------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(gm.GENERIC))
def test_generic_case_lands_on_its_shape(built_lib, dp, name):
    """The compiled table has the case's (compartments, events), the library reports the generic kernels, and the dispatch
    rule -- the first shape of DPOMP_SIM_SHAPES, in order, with c <= CC and e <= EE -- picks the intended shape."""
    model, y, theta = gm.build_case(dp, name)
    dm = dp.device_model(dp.get_private_model(model, y))
    d = dm.compiled.desc
    assert gm.builtin_id(dp, dm) == 0
    assert (d.n_compartments, d.n_events) == (len(gm.GENERIC[name][2]), len(gm.GENERIC[name][1]))
    assert shape_of(sim_shapes(), d.n_compartments, d.n_events) == gm.GENERIC[name][6]
    for family in (gm.POISSON, gm.BINOMIAL, gm.NEGBIN):
        model_c, y_c, _ = gm.build_case(dp, name, family)
        assert gm.builtin_id(dp, dp.device_model(dp.get_private_model(model_c, y_c))) == 0


def test_padded_cases_and_table_features_are_covered(dp):
    """At least two cases sit strictly inside their shape (padded events or compartments), among them one event on (3, 2)
    and a model on (8, 8) smaller than it; one is the full 8 x 8; and the tables have the features the generic kernels
    treat specially: constants k1 / k2, a denominator, a parameter that drives two events."""
    shapes = sim_shapes()
    padded, k1, k2, den, shared = [], False, False, False, False
    for name in gm.GENERIC:
        model, y, theta = gm.build_case(dp, name)
        rate = dp.compile_model(model, y).rate
        c, e = rate.n_compartments, rate.n_events
        cc, ee = shape_of(shapes, c, e)
        if (c, e) != (cc, ee):
            padded.append((name, c, e, cc, ee))
        k1 |= bool(np.any(rate.k1 != 0))
        k2 |= bool(np.any((rate.k2 != 0) & np.any(rate.f2 != 0, axis=1)))
        den |= bool(np.any(rate.has_den))
        shared |= len(set(rate.par.tolist())) < e
    assert len(padded) >= 2, padded
    assert any((c, e, cc, ee) == (3, 1, 3, 2) for _, c, e, cc, ee in padded), padded
    assert any((cc, ee) == (8, 8) and c < 8 and e < 8 for _, c, e, cc, ee in padded), padded
    assert any(len(v[2]) == 8 and len(v[1]) == 8 for v in gm.GENERIC.values())
    assert k1 and k2 and den and shared


def test_denominator_case_reaches_a_zero_denominator(dp):
    """gen_3x3: S -> I at theta_1 S / (I + R); the oracle's trajectories reach I = R = 0 with S > 0, where the table's rate is 0"""
    from oracle import oracle as orc

    model, y, theta = gm.build_case(dp, "gen_3x3")
    cm = dp.compile_model(model, y)
    assert cm.rate.has_den[0] == 1 and cm.rate.dn[0].tolist() == [0, 1, 1]
    assert orc.cum_rates(cm.desc, theta, [31, 0, 0])[0] == 0.0
    ends = [orc.gillespie_sim(cm.desc, theta, key=k)[0][-1] for k in range(40)]
    assert any(s[0] > 0 and s[1] == 0 and s[2] == 0 for s in ends)
