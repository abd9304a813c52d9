"""CPU: the host side of trajectory assessment (fot_assessed_t, fot_assess_trajectories) and its NumPy restatement."""
import ctypes
import os
import re
from types import SimpleNamespace

import numpy as np
import pytest

from tests import assess_oracle as AO
from tests import scenarios

import integrated_path_planning_b200 as ipp
from integrated_path_planning_b200 import _lib
from integrated_path_planning_b200.batch import _assess_field
from integrated_path_planning_b200.engine import ASSESS_FIELDS, SweepResult, assess_radii, pack_paths
from integrated_path_planning_b200.types import SERIES

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = open(os.path.join(ROOT, "include", "fot.h")).read()


def _define(name):
    return int(re.search(r"#define %s (\d+)" % name, HEADER).group(1))


def test_assessed_struct_layout_limits_and_symbol_match_header():
    body = re.search(r"typedef struct fot_assessed \{(.*?)\} fot_assessed_t;", HEADER, re.S).group(1)
    fields = re.findall(r"\*?\s*(\w+);", re.sub(r"/\*.*?\*/", "", body, flags=re.S))
    assert fields == [name for name, _ in _lib.FotAssessed._fields_]
    assert ctypes.sizeof(_lib.FotAssessed) == 3 * 4 + 4 + 10 * 8       # three int32 (padded to 16) + ten pointers
    assert _lib.FotAssessed.series.offset == 16
    assert _define("FOT_MAX_ASSESSED") == _lib.FOT_MAX_ASSESSED == 256
    assert _define("FOT_MAX_RADII") == _lib.FOT_MAX_RADII == 16
    assert _define("FOT_MAX_ASSESS_NT") == _lib.FOT_MAX_ASSESS_NT == 320
    assert _define("FOT_ABI_VERSION") == _lib.FOT_ABI_VERSION == 8
    assert _define("FOT_ABI_MINOR") == _lib.FOT_ABI_MINOR
    assert "int fot_assess_trajectories(fot_handle_t* h, const fot_batch_t* obstacles, const fot_assessed_t* a," in HEADER
    assert "fot_assess_trajectories" in [s[0] for s in _lib.SYMBOLS]
    assert [f[0] for f in ASSESS_FIELDS] == [n for n, _ in _lib.FotAssessed._fields_[6:]]


def _lib_or_skip():
    try:
        return _lib.load()
    except _lib.FotError as e:
        pytest.skip(str(e))


def _valid():
    """A fot_batch_t / fot_assessed_t pair that passes every argument check (pointers are never dereferenced by them)."""
    fake = 0x1000
    b = _lib.FotBatch(n_q=2)
    a = _lib.FotAssessed(m=3, n_t=26, n_r=2, series=fake, len=fake, r2=fake)
    for name, _ in _lib.FotAssessed._fields_[6:]:
        setattr(a, name, fake)
    return b, a


@pytest.mark.parametrize("case, message", [
    ("m0", "m must be"), ("m257", "m must be"), ("nr0", "n_r must be"), ("nr17", "n_r must be"),
    ("nt0", "n_t must be"), ("nt321", "n_t must be"), ("series", "null series or len"), ("len", "null series or len"),
    ("r2", "null r2"), ("out", "null output"), ("nq0", "n_q must be"), ("S", "negative obstacle shape"),
    ("P", "negative obstacle shape"), ("T", "negative obstacle shape"), ("M", "negative obstacle shape"),
    ("static", "static obstacles missing"), ("dyn", "dynamic obstacles missing"), ("mode", "bad dyn_mode"),
])
def test_every_rejected_argument_fails_before_the_device(case, message):
    """The C checks read only the two structs: a handle that is never dereferenced shows that each rejection happens
    before the device (or the handle) is touched, and fot_last_error names the problem."""
    lib = _lib_or_skip()
    b, a = _valid()
    edit = {"m0": lambda: setattr(a, "m", 0), "m257": lambda: setattr(a, "m", 257), "nr0": lambda: setattr(a, "n_r", 0),
            "nr17": lambda: setattr(a, "n_r", 17), "nt0": lambda: setattr(a, "n_t", 0),
            "nt321": lambda: setattr(a, "n_t", 321), "series": lambda: setattr(a, "series", None),
            "len": lambda: setattr(a, "len", None), "r2": lambda: setattr(a, "r2", None),
            "out": lambda: setattr(a, "first_hit", None), "nq0": lambda: setattr(b, "n_q", 0),
            "S": lambda: setattr(b, "S", -1), "P": lambda: setattr(b, "P", -1), "T": lambda: setattr(b, "T_obs", -1),
            "M": lambda: setattr(b, "n_static", -1), "static": lambda: setattr(b, "n_static", 4),
            "dyn": lambda: (setattr(b, "dyn_mode", 2), setattr(b, "S", 2), setattr(b, "P", 3), setattr(b, "T_obs", 5)),
            "mode": lambda: setattr(b, "dyn_mode", 7)}
    edit[case]()
    handle = ctypes.c_void_p(0x10)                                   # never dereferenced by a rejected call
    rc = lib.fot_assess_trajectories(handle, ctypes.byref(b), ctypes.byref(a), None)
    assert rc == -1
    assert message in lib.fot_last_error().decode()


def test_null_handle_is_rejected():
    lib = _lib_or_skip()
    b, a = _valid()
    assert lib.fot_assess_trajectories(None, ctypes.byref(b), ctypes.byref(a), None) == -1
    assert "null argument" in lib.fot_last_error().decode()


def test_python_checks_raise_before_the_device():
    pl = ipp.FrenetPlanner(ipp.CubicSpline2D(*scenarios.STRAIGHT_60), **scenarios.S1_KNOBS)
    path = SimpleNamespace(t=[0.0, 0.2], x=[0.0, 1.0], y=[0.0, 0.0], yaw=[0.0, 0.0])
    with pytest.raises(ValueError, match="1 to 256 paths"):
        pl.assess([], None)
    with pytest.raises(ValueError, match="1 to 256 paths"):
        pl.assess([path] * 257, None)
    long = SimpleNamespace(t=np.arange(321) * 0.2, x=np.arange(321.0), y=np.zeros(321), yaw=np.zeros(321))
    with pytest.raises(ValueError, match="up to 320 samples"):
        pl.assess([long], None)
    for bad in ([1.0, 2.0, 3.0], np.zeros((17, 2)), np.zeros((0, 2)), np.zeros((2, 3))):
        with pytest.raises(ValueError, match="r2 must be"):
            pl.assess([path], None, r2=bad)
    assert pl._engine is None                                         # nothing reached the device
    with pytest.raises(ValueError, match="assess_obstacles must be"):
        _assess_field(np.zeros((3, 2, 4, 2)), 3)
    with pytest.raises(ValueError, match="assess_obstacles must be"):
        _assess_field(np.zeros((2, 2, 3, 4, 2)), 3)
    with pytest.raises(ValueError, match="assess_obstacles must be"):
        _assess_field(np.zeros((3, 0, 3, 4, 2)), 3)
    assert assess_radii((4.0, 5.0)).shape == (1, 2)
    assert assess_radii(np.ones((16, 2))).flags.c_contiguous


def test_pack_paths_series_layout():
    rng = np.random.default_rng(0)
    paths = []
    for n in (5, 1, 9):
        p = SimpleNamespace(**{name: rng.normal(size=n) for name in SERIES})
        p.x, p.yaw = p.x.tolist(), p.yaw.tolist()                        # FrenetPath keeps x..a as lists
        paths.append(p)
    series, lens = pack_paths(paths)
    assert series.shape == (3, 15, 9) and series.dtype == np.float64 and lens.dtype == np.int32
    assert lens.tolist() == [5, 1, 9]
    for j, p in enumerate(paths):
        n = lens[j]
        for r, name in enumerate(SERIES):
            assert np.array_equal(series[j, r, :n], np.asarray(getattr(p, name), dtype=float))
            assert np.all(np.isnan(series[j, r, n:]))
    series, lens = pack_paths(paths[:1], n_t=26)                        # the row length of the library's blocks
    assert series.shape == (1, 15, 26)
    empty = SimpleNamespace(t=[], x=[], y=[], yaw=[])                  # an empty path is a blank slot
    series, lens = pack_paths([empty, paths[0]])
    assert lens.tolist() == [0, 5]


def test_assessment_accessor_and_blank():
    n_q, m, n_r = 2, 3, 2
    res = SweepResult(best_idx=np.zeros(n_q, np.int32), best_cost=np.zeros(n_q), stats=np.zeros((n_q, 8), np.int32),
                      winner_len=np.ones(n_q, np.int32), winner=np.zeros((n_q, 15, 4)))
    with pytest.raises(ValueError, match="assess=True"):
        res.assessment(0)
    res.assessed = {"dyn_min": np.ones((n_q, m)), "static_min": np.ones((n_q, m)),
                    "dyn_at": np.zeros((n_q, m, 4), np.int32), "static_at": np.zeros((n_q, m, 3), np.int32),
                    **{k: np.ones((n_q, m, n_r), np.int32) for k in ("dyn_hits", "first_hit", "static_hit")}}
    a = res.assessment(1)
    assert set(a) == {f[0] for f in ASSESS_FIELDS} and a["dyn_hits"].shape == (m, n_r)
    a["dyn_min"][0] = 5.0
    assert res.assessed["dyn_min"][1, 0] == 1.0                                  # a copy
    res.blank([0])
    a = res.assessed
    assert np.all(np.isposinf(a["dyn_min"][0])) and np.all(a["dyn_at"][0] == -1) and np.all(a["dyn_hits"][0] == 0)
    assert np.all(a["first_hit"][0] == -1) and np.all(a["static_hit"][0] == 0) and np.all(a["static_at"][0] == -1)
    assert np.all(a["dyn_min"][1] == 1.0) and np.all(a["dyn_hits"][1] == 1)
    assert SweepResult.assessed is None                               # a plain attribute, not a dataclass field


# ---- the NumPy restatement on hand-built cases ----------------------------------------------------------------------
def test_oracle_argmin_and_ties_on_hand_built_cases():
    t = np.array([0.0, 0.2, 0.4])
    x, y, yaw = np.array([0.0, 1.0, 2.0]), np.zeros(3), np.zeros(3)
    dyn = np.full((2, 3, 3, 2), 100.0)                                 # S=2, P=3, T=3, far away
    dyn[1, 2, 1] = (1.0, 3.0)                                          # sample n=1 at distance 3 (s=1, p=2)
    dyn[0, 1, 2] = (2.0, -3.0)                                         # n=2 at distance 3 as well: (n=1) comes first
    a = AO.assess_trajectory(t, x, y, yaw, 0.2, dyn=dyn, r2=[(9.0, 0.0), (8.99, 0.0)])
    assert a["dyn_min"] == 3.0 and a["dyn_at"].tolist() == [1, 0, 1, 2]
    assert a["dyn_hits"].tolist() == [2, 0] and a["first_hit"].tolist() == [1, -1]
    # a NaN anywhere drops that pedestrian, even at a step no sample reads
    dyn[1, 2, 0] = (np.nan, 0.0)
    a = AO.assess_trajectory(t, x, y, yaw, 0.2, dyn=dyn, r2=[(9.0, 0.0)])
    assert a["dyn_at"].tolist() == [2, 0, 0, 1] and a["dyn_hits"].tolist() == [1] and a["first_hit"].tolist() == [2]
    # the time index is clip(round(t / dt)): past T_obs the last step
    a = AO.assess_trajectory(np.array([0.0, 0.9, 5.0]), x, y, yaw, 0.2, dyn=dyn, r2=[(9.0, 0.0)])
    assert a["dyn_at"].tolist() == [2, 0, 0, 1]
    # inf positions are entries (inf), never hits; all-inf: the first entry, as np.argmin picks
    far = np.full((1, 2, 3, 2), np.inf)
    a = AO.assess_trajectory(t, x, y, yaw, 0.2, dyn=far, r2=[(1e300, 0.0)])
    assert a["dyn_min"] == np.inf and a["dyn_at"].tolist() == [0, 0, 0, 0] and a["dyn_hits"].tolist() == [0]
    # static points, with two footprint circles: (n, circle, point) order
    static = np.array([[5.0, 0.0], [0.5, 0.0]])
    a = AO.assess_trajectory(t, x, y, yaw, 0.2, static=static, r2=[(0.0, 0.25), (0.0, 0.2)], offsets=[-0.5, 0.5])
    assert a["static_min"] == 0.0 and a["static_at"].tolist() == [0, 1, 1]
    assert a["static_hit"].tolist() == [1, 1] and a["first_hit"].tolist() == [0, 0]
    # no field, empty trajectory: blank
    a = AO.assess_trajectory(t[:0], x[:0], y[:0], yaw[:0], 0.2, static=static, dyn=dyn)
    assert a["dyn_min"] == np.inf and a["dyn_at"].tolist() == [-1] * 4 and a["static_at"].tolist() == [-1] * 3
    a = AO.assess_trajectory(t, x, y, yaw, 0.2)
    assert a["dyn_min"] == np.inf and a["static_min"] == np.inf and a["first_hit"].tolist() == [-1]
    assert AO.verdict(a, 0.0, 1, False)
