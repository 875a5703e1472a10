"""Host-side checks of the single-track rollout ABI (f1l_vehicle, f1l_rollout_st_dev): the ctypes
struct follows include/f1l.h, the defaults are f1tenth_gym's, and a null handle or vehicle is
rejected before any device is touched."""
import ctypes

import pytest

from tests.test_rollout_abi import CTYPES, _header_struct

DEFAULTS = dict(mu=1.0489, C_Sf=4.718, C_Sr=5.4562, lf=0.15875, lr=0.17145, h=0.074, m=3.74, I=0.04712,
                max_steer_vel=3.2, v_switch=7.319, v_kin=0.5)


def test_vehicle_struct_matches_header():
    from f1tenth_planning_b200 import _lib
    hdr = _header_struct("f1l_vehicle")
    assert [f for f, _ in hdr] == [f for f, _ in _lib.Vehicle._fields_] == list(DEFAULTS)
    for (f, ctype), (_, pytype) in zip(hdr, _lib.Vehicle._fields_):
        assert ctypes.sizeof(CTYPES[ctype]) == ctypes.sizeof(pytype), f
        assert getattr(_lib.Vehicle, f).offset % ctypes.sizeof(pytype) == 0, f
    assert ctypes.sizeof(_lib.Vehicle) == 11 * 8


def test_default_vehicle_and_rejections_without_device():
    from f1tenth_planning_b200 import _lib, rollout
    L = _lib.lib()
    v = _lib.Vehicle()
    assert L.f1l_default_vehicle(ctypes.byref(v)) == 0
    assert {f: getattr(v, f) for f, _ in v._fields_} == DEFAULTS
    assert rollout.Vehicle()._asdict() == DEFAULTS
    assert L.f1l_default_vehicle(None) == -1
    rc = _lib.RolloutConfig()
    assert L.f1l_default_rollout_config(ctypes.byref(rc)) == 0
    fl = _lib.FleetBuffers(*([8] * 7))   # never dereferenced
    dyn = ctypes.c_void_p(8)
    assert L.f1l_rollout_st_dev(None, ctypes.byref(rc), ctypes.byref(v), ctypes.byref(fl), dyn, None, 4, 1,
                                None, None, None) == -1
    assert L.f1l_rollout_st_dev(None, ctypes.byref(rc), None, ctypes.byref(fl), dyn, None, 4, 1,
                                None, None, None) == -1


@pytest.mark.parametrize("field", list(DEFAULTS))
def test_python_vehicle_values_are_checked(field):
    from f1tenth_planning_b200 import rollout
    bad = [float("nan"), -1.0] + ([] if field == "h" else [0.0])
    for val in bad:
        with pytest.raises(ValueError):
            rollout._vehicle_struct(rollout.Vehicle(**{field: val}))
    ok = rollout._vehicle_struct(rollout.Vehicle(**{field: 0.0 if field == "h" else 2.0}))
    assert getattr(ok, field) == (0.0 if field == "h" else 2.0)
