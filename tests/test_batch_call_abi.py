"""Host-side checks of the batch-call ABI (f1l_plan_batch_call / _dev, f1l_rollout_weights_dev): the
ctypes struct follows include/f1l.h field for field, and a null handle or call struct is rejected
before any device is touched."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CTYPES = {"int32_t": ctypes.c_int32, "double*": ctypes.c_void_p, "float*": ctypes.c_void_p,
          "uint8_t*": ctypes.c_void_p, "int32_t*": ctypes.c_void_p}


def _header_struct(name):
    """[(field, C type)] of `typedef struct { ... } name;` in include/f1l.h (const dropped)"""
    src = open(os.path.join(ROOT, "include", "f1l.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    body = re.search(r"typedef struct \{([^}]*)\}\s*" + name + r"\s*;", src).group(1)
    fields = []
    for decl in body.split(";"):
        decl = re.sub(r"\bconst\b", "", decl).strip()
        m = re.match(r"([a-z0-9_]+)\s*(\*?)\s*(.+)", decl) if decl else None
        if m:
            for v in m.group(3).split(","):
                v = v.strip()
                fields.append((v.lstrip("*"), m.group(1) + ("*" if m.group(2) or v.startswith("*") else "")))
    return fields


def test_batch_call_struct_matches_header():
    from f1tenth_planning_b200 import _lib
    hdr = _header_struct("f1l_batch_call")
    assert [f for f, _ in hdr] == [f for f, _ in _lib.BatchCall._fields_]
    for (f, ctype), (_, pytype) in zip(hdr, _lib.BatchCall._fields_):
        assert ctypes.sizeof(CTYPES[ctype]) == ctypes.sizeof(pytype), f
        assert getattr(_lib.BatchCall, f).offset % ctypes.sizeof(pytype) == 0, f
    assert ctypes.sizeof(_lib.BatchCall) == 13 * 8 + 4 * 4


def test_null_handle_or_call_without_device():
    from f1tenth_planning_b200 import _lib
    L = _lib.lib()
    b = _lib.BatchCall(poses=8, n_scenarios=4)   # never dereferenced
    assert L.f1l_plan_batch_call_dev(None, ctypes.byref(b), None) == -1
    assert L.f1l_plan_batch_call(None, ctypes.byref(b)) == -1
    assert L.f1l_plan_batch_call_dev(None, None, None) == -1
    assert L.f1l_plan_batch_call(None, None) == -1
    rc = _lib.RolloutConfig()
    assert L.f1l_default_rollout_config(ctypes.byref(rc)) == 0
    fl = _lib.FleetBuffers(*([8] * 7))
    assert L.f1l_rollout_weights_dev(None, ctypes.byref(rc), ctypes.byref(fl), None, 4, 1, None, None) == -1
