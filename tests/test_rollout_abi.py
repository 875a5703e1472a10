"""Host-side checks of the rollout ABI (f1l_rollout_dev): the ctypes structs follow include/f1l.h,
the defaults are the documented ones, and a null handle is rejected before any device is touched."""
import ctypes
import math
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CTYPES = {"double": ctypes.c_double, "int32_t": ctypes.c_int32, "double*": ctypes.c_void_p,
          "float*": ctypes.c_void_p, "uint8_t*": ctypes.c_void_p, "int32_t*": ctypes.c_void_p}


def _header_struct(name):
    """[(field, C type)] of `typedef struct { ... } name;` in include/f1l.h"""
    src = open(os.path.join(ROOT, "include", "f1l.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    body = re.search(r"typedef struct \{([^}]*)\}\s*" + name + r"\s*;", src).group(1)
    fields = []
    for decl in body.split(";"):
        m = re.match(r"\s*([a-z0-9_]+)\s*(\*?)\s*(.+)", decl.strip()) if decl.strip() else None
        if m:
            for v in m.group(3).split(","):
                v = v.strip()
                fields.append((v.lstrip("*"), m.group(1) + ("*" if m.group(2) or v.startswith("*") else "")))
    return fields


def test_rollout_structs_match_header():
    from f1tenth_planning_b200 import _lib
    for cname, cls in (("f1l_rollout_config", _lib.RolloutConfig), ("f1l_fleet", _lib.FleetBuffers),
                       ("f1l_rollout_trace", _lib.RolloutTraceBuffers)):
        hdr = _header_struct(cname)
        assert [f for f, _ in hdr] == [f for f, _ in cls._fields_], cname
        for (f, ctype), (_, pytype) in zip(hdr, cls._fields_):
            assert ctypes.sizeof(CTYPES[ctype]) == ctypes.sizeof(pytype), (cname, f)
            assert getattr(cls, f).offset % ctypes.sizeof(pytype) == 0, (cname, f)
    assert ctypes.sizeof(_lib.RolloutConfig) == 40
    assert ctypes.sizeof(_lib.FleetBuffers) == 7 * 8
    assert ctypes.sizeof(_lib.RolloutTraceBuffers) == 5 * 8


def test_rollout_defaults_and_null_handle_without_device():
    from f1tenth_planning_b200 import _lib
    L = _lib.lib()
    rc = _lib.RolloutConfig()
    assert L.f1l_default_rollout_config(ctypes.byref(rc)) == 0
    assert (rc.dt, rc.substeps, rc.group, rc.max_steer, rc.max_accel) == (0.01, 1, 1, 0.4189, 9.51)
    assert rc.v_max == math.inf
    assert L.f1l_default_rollout_config(None) == -1
    fl = _lib.FleetBuffers(*([8] * 7))   # never dereferenced
    assert L.f1l_rollout_dev(None, ctypes.byref(rc), ctypes.byref(fl), 4, 1, None, None) == -1
