"""The field tables of the arrays the library uses in place (_lib.BATCH_FIELDS, FLEET_FIELDS,
PP_FIELDS), the one array check and the one BatchCall builder, called without an Engine: an array
passes only with its row's exact dtype, shape and layout (and on the host, writeable where the
library writes it), and a valid call carries every array's own address."""
import os
import re

import numpy as np
import pytest

from f1tenth_planning_b200 import _lib
from tests.test_batch_call_abi import ROOT, _header_struct

DIMS = dict(S=3, K=2, C=5, M=7, B=4)
HOST_ROWS = [(t, n) for t, table in (("batch", _lib.BATCH_FIELDS), ("pp", _lib.PP_FIELDS)) for n in table]
DEVICE_ROWS = [(t, n) for t, table in (("batch", _lib.BATCH_FIELDS), ("fleet", _lib.FLEET_FIELDS)) for n in table]
TABLES = {"batch": _lib.BATCH_FIELDS, "fleet": _lib.FLEET_FIELDS, "pp": _lib.PP_FIELDS}
C_DTYPE = {"double*": "float64", "float*": "float32", "int32_t*": "int32", "uint8_t*": "uint8"}


def _valid(table):
    return {n: np.zeros(_lib.shape_of(row, DIMS), row[0][0]) for n, row in TABLES[table].items()}


def _bad(a, dtypes):
    """the same array with a wrong dtype, two wrong shapes, a strided layout, and as a list"""
    wrong = next(d for d in ("float64", "float32", "int32", "int64") if d not in dtypes)
    strided = np.zeros(a.shape[:-1] + (2 * a.shape[-1],), a.dtype)[..., ::2]
    return [a.astype(wrong), np.zeros((a.shape[0] + 1,) + a.shape[1:], a.dtype), a[None], strided,
            a.tolist()]


def test_every_pointer_field_has_one_row():
    for cname, table in (("f1l_batch_call", "batch"), ("f1l_fleet", "fleet")):
        ptrs = [(f, t) for f, t in _header_struct(cname) if t.endswith("*")]
        assert sorted(f for f, _ in ptrs) == sorted(TABLES[table]), cname
        for f, ctype in ptrs:
            dtypes = TABLES[table][f][0]
            assert dtypes[0] == C_DTYPE[ctype], (cname, f)
            assert all(np.dtype(d).itemsize == np.dtype(dtypes[0]).itemsize for d in dtypes), (cname, f)
    src = open(os.path.join(ROOT, "include", "f1l.h")).read()
    args = re.search(r"int f1l_pure_pursuit_batch\(([^)]*)\)", src).group(1)
    outs = [a.split("*")[1].strip() for a in args.split(",") if "*" in a][1:]   # after poses
    assert outs == list(_lib.PP_FIELDS)


def test_valid_host_arrays_give_their_addresses():
    a = _valid("batch")
    for update_prev in (False, True):
        b = _lib.batch_call(a, "host", DIMS, update_prev)
        for n, arr in a.items():
            assert getattr(b, n) == arr.ctypes.data, n
        assert (b.n_scenarios, b.max_opp, b.update_prev, b.reserved) == (3, 2, int(update_prev), 0)
    a["has_prev"] = np.zeros(3, bool)
    b = _lib.batch_call(dict(poses=a["poses"], prev_theta=a["prev_theta"], has_prev=a["has_prev"]),
                        "host", DIMS, True)
    assert b.has_prev == a["has_prev"].ctypes.data and b.best_idx is None and b.opp is None


def test_has_prev_or_update_prev_need_prev_theta():
    a = _valid("batch")
    del a["prev_theta"]
    with pytest.raises(ValueError):
        _lib.batch_call(a, "host", DIMS, False)
    del a["has_prev"]
    with pytest.raises(ValueError):
        _lib.batch_call(a, "host", DIMS, True)
    _lib.batch_call(a, "host", DIMS, False)


@pytest.mark.parametrize("table,name", HOST_ROWS)
def test_host_row_rejects_bad_arrays(table, name):
    dtypes, _, direction = TABLES[table][name]
    a = _valid(table)
    shape = _lib.shape_of(TABLES[table][name], DIMS)

    def call(arr, update_prev):
        if table == "batch":
            _lib.batch_call(dict(a, **{name: arr}), "host", DIMS, update_prev)
        else:   # the pure-pursuit outputs are always written
            _lib.check_array(name, arr, shape, dtypes, "host", writes=True)

    ro = a[name].copy()
    ro.flags.writeable = False
    for update_prev in (False, True):
        for bad in _bad(a[name], dtypes):
            with pytest.raises(ValueError):
                call(bad, update_prev)
        if direction == _lib.OUT or (direction == _lib.INOUT and update_prev):
            with pytest.raises(ValueError):
                call(ro, update_prev)
        else:
            call(ro, update_prev)


@pytest.mark.parametrize("table,name", DEVICE_ROWS)
def test_device_row_rejects_host_memory(table, name):
    torch = pytest.importorskip("torch")
    row = TABLES[table][name]
    host = _valid(table)[name]
    for bad in (torch.from_numpy(host), host):
        with pytest.raises(ValueError):
            _lib.check_array(name, bad, host.shape, row[0], 0)


@pytest.mark.gpu
@pytest.mark.parametrize("table,name", DEVICE_ROWS)
def test_device_row_rejects_bad_tensors(table, name):
    """rejected by the check alone: nothing here reaches the library"""
    import torch
    dev = torch.device("cuda", 0)
    row = TABLES[table][name]
    a = {n: torch.from_numpy(v).to(dev) for n, v in _valid(table).items()}
    t = a[name]

    def call(arr):
        if table == "batch":
            return _lib.batch_call(dict(a, **{name: arr}), 0, DIMS, True)
        _lib.check_array(name, arr, tuple(t.shape), row[0], 0)

    b = call(t)
    if table == "batch":
        assert getattr(b, name) == t.data_ptr()
    for bad in [torch.from_numpy(x).to(dev) for x in _bad(t.cpu().numpy(), row[0])[:3]] + [
            torch.zeros(t.shape[:-1] + (2 * t.shape[-1],), dtype=t.dtype, device=dev)[..., ::2], t.cpu()]:
        with pytest.raises(ValueError):
            call(bad)


@pytest.mark.gpu
def test_engine_rejects_arrays_the_library_would_overrun(ellipse, corridor):
    """arrays of the wrong size or type for what the library writes or reads are rejected before
    any call reaches it"""
    import torch
    from f1tenth_planning_b200 import synth
    from tests.test_gpu_batch_prev import _pair
    eng, _, _ = _pair(ellipse, corridor)
    S, C, M = 8, eng.n_candidates, eng.n_samples
    poses, opp, n_opp = synth.scenario_batch(ellipse, S, 2, 1201)
    dev = torch.device("cuda", eng.device)
    tX, to, tn = (torch.from_numpy(x).to(dev) for x in (poses, opp, n_opp))
    for kw in (dict(steer_speed=torch.zeros(S, 2, device=dev)),
               dict(best_traj=torch.zeros(S, C, device=dev)),
               dict(best_idx=torch.zeros(S, dtype=torch.int64, device=dev)),
               dict(costs=torch.zeros(S, C - 1, device=dev))):
        with pytest.raises(ValueError):
            eng.plan_batch_dev(tX, to, tn, **kw)
    for args in ((tX, to[:, 0]), (tX.float(), to), (tX, to, tn.long()), (tX[:, :3], to)):
        with pytest.raises(ValueError):
            eng.plan_batch_dev(*args)
    for out in (dict(best_idx=np.zeros(S, np.int16)), dict(steer_speed=np.zeros((S, 2), np.float32)),
                dict(best_traj=np.zeros((S, M), np.float32)), dict(costs=np.zeros((S - 1, C), np.float32))):
        with pytest.raises(ValueError):
            eng.plan_batch(poses, opp, n_opp, out=out)
    with pytest.raises(ValueError):
        eng.plan_batch(poses, opp[:, 0], n_opp)
    with pytest.raises(ValueError):
        eng.pure_pursuit_batch(poses[:, :3], 0.8, out=dict(nearest=np.zeros((S, 2))))
    with pytest.raises(ValueError):
        eng.pure_pursuit_batch(poses[:, :3], 0.8, out=dict(status=np.zeros(S, np.int64)))
    with pytest.raises(ValueError):
        eng.intersect_point_batch(poses[:, :2], np.zeros(S - 1), 0.8, True)
    torch.cuda.synchronize(dev)
