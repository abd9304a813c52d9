"""CPU: the host side of candidate assessment (fot_assess_candidates): the declaration, every argument the C call
refuses before it touches the device, and the Python plumbing while the planner has no engine."""
import ctypes
import os
import re

import numpy as np
import pytest

from tests import scenarios

import integrated_path_planning_b200 as ipp
from integrated_path_planning_b200 import _lib
from integrated_path_planning_b200.engine import ASSESS_FIELDS, SweepResult

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = open(os.path.join(ROOT, "include", "fot.h")).read()
NAMES = tuple(f[0] for f in ASSESS_FIELDS) + ("keep",)


def test_declaration_and_symbol_match_header():
    decl = re.search(r"int fot_assess_candidates\((.*?)\);", HEADER, re.S).group(1)
    params = [p.strip() for p in " ".join(decl.split()).split(",")]
    assert params == ["fot_handle_t* h", "const fot_batch_t* queries", "const fot_batch_t* field", "int cand_stride",
                      "const fot_assessed_t* out", "int32_t* keep", "void* stream"]
    entry = {s[0]: s for s in _lib.SYMBOLS}["fot_assess_candidates"]
    assert len(entry[2]) == len(params)
    assert _lib.FOT_ABI_MINOR == int(re.search(r"#define FOT_ABI_MINOR (\d+)", HEADER).group(1)) == 1


def _lib_or_skip():
    try:
        return _lib.load()
    except _lib.FotError as e:
        pytest.skip(str(e))


def _valid():
    """(queries, field, stride, out) that pass every check the C call makes before it reads the handle."""
    fake = 0x1000
    b = _lib.FotBatch(n_q=2, n_v_max=3, frenet=fake, target_speed=fake, v_grid=fake, n_v=fake)
    f = _lib.FotBatch(n_q=2)
    stride = 40
    a = _lib.FotAssessed(m=stride, n_t=0, n_r=2, r2=fake)
    for name, _ in _lib.FotAssessed._fields_[6:]:
        setattr(a, name, fake)
    return b, f, stride, a


CASES = {
    "series": ("series and len must be null", lambda b, f, a: setattr(a, "series", 0x1000)),
    "len": ("series and len must be null", lambda b, f, a: setattr(a, "len", 0x1000)),
    "m_small": ("m must equal cand_stride", lambda b, f, a: setattr(a, "m", 39)),
    "m_large": ("m must equal cand_stride", lambda b, f, a: setattr(a, "m", 41)),
    "nr0": ("n_r must be", lambda b, f, a: setattr(a, "n_r", 0)),
    "nr17": ("n_r must be", lambda b, f, a: setattr(a, "n_r", 17)),
    "r2": ("null r2", lambda b, f, a: setattr(a, "r2", None)),
    **{"out_" + n: ("null output array", (lambda n: lambda b, f, a: setattr(a, n, None))(n))
       for n, _ in _lib.FotAssessed._fields_[6:]},
    "nq0": ("n_q and n_v_max must be", lambda b, f, a: setattr(b, "n_q", 0)),
    "nq_neg": ("n_q and n_v_max must be", lambda b, f, a: setattr(b, "n_q", -3)),
    "nv0": ("n_q and n_v_max must be", lambda b, f, a: setattr(b, "n_v_max", 0)),
    "frenet": ("null query array", lambda b, f, a: setattr(b, "frenet", None)),
    "n_v": ("null query array", lambda b, f, a: setattr(b, "n_v", None)),
    "S": ("negative obstacle shape", lambda b, f, a: setattr(f, "S", -1)),
    "M": ("negative obstacle shape", lambda b, f, a: setattr(f, "n_static", -1)),
    "static": ("static obstacles missing", lambda b, f, a: setattr(f, "n_static", 4)),
    "dyn": ("dynamic obstacles missing",
            lambda b, f, a: (setattr(f, "dyn_mode", 2), setattr(f, "S", 2), setattr(f, "P", 3), setattr(f, "T_obs", 5))),
    "mode": ("bad dyn_mode", lambda b, f, a: setattr(f, "dyn_mode", 5)),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_every_rejected_argument_fails_before_the_device(case):
    """The checks read only the structs: a handle that is never dereferenced shows that each rejection comes before
    the handle or the device is touched, and fot_last_error names the problem."""
    lib = _lib_or_skip()
    b, f, stride, a = _valid()
    message, edit = CASES[case]
    edit(b, f, a)
    rc = lib.fot_assess_candidates(ctypes.c_void_p(0x10), ctypes.byref(b), ctypes.byref(f), stride, ctypes.byref(a),
                                   None, None)
    assert rc == -1
    assert message in lib.fot_last_error().decode()


def test_null_arguments_are_rejected():
    lib = _lib_or_skip()
    b, f, stride, a = _valid()
    for args in ((None, ctypes.byref(b), ctypes.byref(f)), (ctypes.c_void_p(0x10), None, ctypes.byref(f)),
                 (ctypes.c_void_p(0x10), ctypes.byref(b), None)):
        assert lib.fot_assess_candidates(*args, stride, ctypes.byref(a), None, None) == -1
        assert "null argument" in lib.fot_last_error().decode()
    assert lib.fot_assess_candidates(ctypes.c_void_p(0x10), ctypes.byref(b), ctypes.byref(f), stride, None, None, None) == -1


# ---- Python plumbing, with no engine --------------------------------------------------------------------------------
def _planner():
    return ipp.BatchFrenetPlanner(ipp.CubicSpline2D(*scenarios.STRAIGHT_60), **scenarios.S1_KNOBS)


def test_python_checks_raise_before_the_device():
    pl = _planner()
    frenet = np.zeros((3, 6))
    frenet[:, 1] = 2.0
    for bad in (np.zeros((17, 2)), np.zeros((2, 3)), [1.0, 2.0, 3.0]):
        with pytest.raises(ValueError, match="r2 must be"):
            pl.plan_batch(frenet, 6.0, assess_candidates=True, assess_r2=bad)
        with pytest.raises(ValueError, match="r2 must be"):
            pl.candidate_assessment(None, None, r2=bad)
    with pytest.raises(ValueError, match="assess_obstacles must be"):
        pl.plan_batch(frenet, 6.0, assess_candidates=True, assess_obstacles=np.zeros((2, 1, 3, 4, 2)))
    with pytest.raises(ValueError, match="assess_obstacles must be"):
        pl.candidate_assessment(None, None, assess_obstacles=np.zeros((3, 4, 2)))
    with pytest.raises(ValueError, match="route ids"):
        pl.plan_batch_from_ego(np.zeros((3, 5)), 6.0, assess_candidates=True, route=[0, 1, 0])
    assert pl._engine is None                                           # nothing reached the device


def _result(n_q=3, stride=7, n_r=2):
    res = SweepResult(best_idx=np.zeros(n_q, np.int32), best_cost=np.zeros(n_q), stats=np.zeros((n_q, 8), np.int32),
                      winner_len=np.ones(n_q, np.int32), winner=np.zeros((n_q, 15, 4)))
    res.n_cand = np.array([7, 5, 6])
    res.cand_assessed = {"dyn_min": np.ones((n_q, stride)), "static_min": np.ones((n_q, stride)),
                         "dyn_at": np.zeros((n_q, stride, 4), np.int32), "static_at": np.zeros((n_q, stride, 3), np.int32),
                         **{k: np.ones((n_q, stride, n_r), np.int32) for k in ("dyn_hits", "first_hit", "static_hit")},
                         "keep": np.full((n_q, stride), 26, np.int32)}
    return res


def test_candidate_assessment_accessor_trims_and_copies():
    res = _result()
    a = res.candidate_assessment(1)
    assert set(a) == set(NAMES)
    assert a["dyn_min"].shape == (5,) and a["dyn_at"].shape == (5, 4) and a["dyn_hits"].shape == (5, 2)
    a["dyn_min"][0] = 9.0
    assert res.cand_assessed["dyn_min"][1, 0] == 1.0                     # a copy
    res.cand_cat = np.arange(21, dtype=np.uint8).reshape(3, 7)
    res.cand_cost = np.arange(21.0).reshape(3, 7)
    a = res.candidate_assessment(2)
    assert a["cand_cat"].tolist() == list(range(14, 20)) and a["cand_cost"].shape == (6,)
    plain = _result()
    plain.cand_assessed = None
    with pytest.raises(ValueError, match="assess_candidates=True"):
        plain.candidate_assessment(0)
    assert SweepResult.cand_assessed is None                             # a plain attribute, not a dataclass field


def test_blank_blanks_candidate_rows():
    res = _result()
    res.assessed = {"dyn_min": np.ones((3, 1)), "static_min": np.ones((3, 1)), "dyn_at": np.zeros((3, 1, 4), np.int32),
                    "static_at": np.zeros((3, 1, 3), np.int32),
                    **{k: np.ones((3, 1, 2), np.int32) for k in ("dyn_hits", "first_hit", "static_hit")}}
    res.blank(np.array([False, True, False]))
    c = res.cand_assessed
    assert np.all(np.isposinf(c["dyn_min"][1])) and np.all(np.isposinf(c["static_min"][1]))
    assert np.all(c["dyn_at"][1] == -1) and np.all(c["static_at"][1] == -1) and np.all(c["first_hit"][1] == -1)
    assert np.all(c["dyn_hits"][1] == 0) and np.all(c["static_hit"][1] == 0) and np.all(c["keep"][1] == 0)
    assert np.all(c["dyn_min"][[0, 2]] == 1.0) and np.all(c["keep"][[0, 2]] == 26)
    assert np.all(np.isposinf(res.assessed["dyn_min"][1])) and "keep" not in res.assessed
