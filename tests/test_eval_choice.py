"""The eval_kernel instance choice of the library (no GPU), through f1l_debug_eval_choice /
f1l_debug_eval_builds: every choice over the sample-count bucket edges, candidate counts 1 ...
65 536, scenario counts 1 ... 10^5, both generators, lone queries and batches, with and without
per-scenario weights lands on a built instance, and every built instance is chosen somewhere --
a build the launch policy cannot reach fails here."""
import ctypes as C
import functools

import pytest

from f1tenth_planning_b200 import _lib

SM = 148   # B200

# the edges of every bucket of the instance table (largest M 32, 64, 104, 128, 208, 256), the
# smallest M the ABI accepts, and the odd-row edges of the S = 13 shapes (M = 97, 101, 105; 193,
# 201, 209)
M_EDGES = [2, 3, 31, 32, 33, 63, 64, 65, 96, 97, 100, 101, 104, 105, 127, 128, 129, 192, 193, 200,
           201, 208, 209, 255, 256]
CANDS = [1, 2, 3, 4, 7, 8, 13, 15, 16, 25, 28, 29, 30, 31, 32, 56, 64, 100, 255, 256, 257, 1000, 1024, 4096,
         8192, 16384, 32768, 65536]
SCENARIOS = [1, 2, 4, 5, 31, 32, 64, 100, 384, 1000, 4095, 4735, 4736, 5000, 8287, 8288, 10000, 20000,
             100000]

KEYS = ("nw", "chunk", "ctas_per_scenario", "item", "m_max", "ipl", "s", "sg", "minb", "wide",
        "persistent", "pw", "max_window")


@functools.lru_cache(maxsize=None)
def eval_choice(n_cand, S, M, generator=0, lone=False, weights=False, sm=SM):
    """What a pipeline launch of S scenarios x n_cand candidates at M samples runs: the instance
    (bucket row, nw, minb, wide, pw), its CTA plan and the largest window its shared memory holds"""
    out = (C.c_int32 * 13)()
    flags = (_lib.EVAL_LONE if lone else 0) | (_lib.EVAL_WEIGHTS if weights else 0)
    rc = _lib.lib().f1l_debug_eval_choice(n_cand, S, M, sm, generator, flags, out, 13)
    assert rc == 0, rc
    return dict(zip(KEYS, (int(v) for v in out)))


def eval_builds():
    """rows of the instance table: dicts with m_max, ipl, s, sg and minb of nw 4, 7, 8 and wide"""
    out = (C.c_int32 * 256)()
    n = _lib.lib().f1l_debug_eval_builds(out, 256)
    assert n > 0, n
    keys = ("m_max", "ipl", "s", "sg", "nw4", "nw7", "nw8", "wide")
    return [dict(zip(keys, out[8 * r:8 * r + 8])) for r in range(n)]


def built_instances(rows=None):
    """{(m_max, nw, minb, wide, pw)} of every compiled eval_kernel; the wide build has no PW twin"""
    got = set()
    for r in rows or eval_builds():
        for nw in (4, 7, 8):
            if r["nw%d" % nw]:
                got |= {(r["m_max"], nw, r["nw%d" % nw], 0, pw) for pw in (0, 1)}
        if r["wide"]:
            got.add((r["m_max"], 8, r["wide"], 1, 0))
    return got


def instance(c):
    return (c["m_max"], c["nw"], c["minb"], c["wide"], c["pw"])


def regime(c):
    """what a workload exercises beyond its instance: persistent grid and candidates per pull"""
    return instance(c) + (c["persistent"], c["item"])


def workloads(M):
    """every (n_cand, S, generator, lone, weights) of the sweep at M"""
    for n in CANDS:
        for S in SCENARIOS:
            for gen in (0, 1):
                for lone in ((False, True) if S == 1 else (False,)):
                    for w in (False, True):
                        yield n, S, gen, lone, w


def reachable(M, sm=SM):
    """{regime: the workload with the least work that reaches it} at M"""
    best = {}
    for n, S, gen, lone, w in workloads(M):
        key = regime(eval_choice(n, S, M, gen, lone, w, sm)) + (gen,)
        if key not in best or n * S < best[key][0] * best[key][1]:
            best[key] = (n, S, gen, lone, w)
    return best


def test_table_rows():
    rows = eval_builds()
    assert [r["m_max"] for r in rows] == [32, 64, 104, 128, 208, 256]
    for r in rows:
        assert r["s"] * r["sg"] >= r["m_max"]              # the sample slab holds every sample
        assert r["sg"] in (8, 16) and 32 % r["sg"] == 0
        assert r["nw8"] > 0                                # the fall-back warp count is always built
        # the M > 128 shapes: 8 warps only (their 72-register builds spill); the wide build serves
        # their dense lone queries
        if r["m_max"] > 128:
            assert r["nw4"] == 0 and r["nw7"] == 0 and r["wide"] == 2, r
        else:
            assert r["nw4"] > 0 and r["nw7"] > 0 and r["wide"] == 0, r
    out = (C.c_int32 * 8)()
    assert _lib.lib().f1l_debug_eval_builds(out, 8) < 0
    assert _lib.lib().f1l_debug_eval_builds(None, 256) < 0


@pytest.mark.parametrize("M", M_EDGES)
def test_every_choice_is_built(M):
    rows = eval_builds()
    row = next(r for r in rows if M <= r["m_max"])
    built = built_instances(rows)
    for n, S, gen, lone, w in workloads(M):
        c = eval_choice(n, S, M, gen, lone, w)
        where = (n, S, M, gen, lone, w, c)
        assert instance(c) in built, where
        assert (c["m_max"], c["ipl"], c["s"], c["sg"]) == (row["m_max"], row["ipl"], row["s"], row["sg"]), where
        assert c["pw"] == int(w), where
        assert c["nw"] in (4, 7, 8) and c["chunk"] % c["nw"] == 0 and c["chunk"] >= c["nw"], where
        resident = c["minb"] * SM
        if c["persistent"]:
            # a lone query with more CTAs than one wave: one wave of CTAs pulling candidates
            assert lone and c["nw"] != 4, where
            assert c["ctas_per_scenario"] == resident, where
            assert c["item"] == (4 if gen == 0 and n >= 16 * resident * c["nw"] else 1), where
        else:
            # the chunks cover every candidate, and no CTA is empty
            assert c["ctas_per_scenario"] * c["chunk"] >= n, where
            assert (c["ctas_per_scenario"] - 1) * c["chunk"] < n, where
            # the shared Newton solve needs the cubic generator and four candidates per warp
            assert c["item"] == (4 if gen == 0 and c["chunk"] >= 4 * c["nw"] else 1), where
        if c["wide"]:
            assert c["persistent"] and c["nw"] == 8 and not w and n >= 4 * 3 * SM * 8, where
        # the same call without the weights runs the same plan on the PW = false twin
        if w and not c["wide"]:
            d = eval_choice(n, S, M, gen, lone, False)
            if not d["wide"]:
                assert {k: v for k, v in d.items() if k != "pw"} == {k: v for k, v in c.items() if k != "pw"}
        assert c["max_window"] >= 4096 and c["max_window"] % 32 == 0, where
        # the first four entries are what an n = 4 caller gets
        out = (C.c_int32 * 4)()
        flags = (_lib.EVAL_LONE if lone else 0) | (_lib.EVAL_WEIGHTS if w else 0)
        assert _lib.lib().f1l_debug_eval_choice(n, S, M, SM, gen, flags, out, 4) == 0
        assert list(out) == [c["nw"], c["chunk"], c["ctas_per_scenario"], c["item"]], where
        # ... and, for a batch without weights, what f1l_debug_eval_plan gives
        if not lone and not w:
            assert _lib.lib().f1l_debug_eval_plan(n, S, M, SM, gen, out, 4) == 0
            assert list(out) == [c["nw"], c["chunk"], c["ctas_per_scenario"], c["item"]], where


def test_every_build_is_reached():
    reached = set()
    for M in M_EDGES:
        for n, S, gen, lone, w in workloads(M):
            reached.add(instance(eval_choice(n, S, M, gen, lone, w)))
    built = built_instances()
    assert reached == built, (sorted(built - reached), sorted(reached - built))


def test_regimes_of_each_bucket():
    """regimes the GPU instance tests run: in every M <= 128 bucket the throughput 4-warp build
    with four candidates per pull, 7- and 8-warp CTAs and the persistent grid of lone dense
    queries; in the M > 128 buckets 8-warp CTAs, static or persistent, and the wide build with
    one and four candidates per pull"""
    union = set()
    for M in (32, 64, 104, 128):
        r = reachable(M)
        have = {(k[1], k[5], k[6]) for k in r}   # (nw, persistent, item)
        assert {(4, 0, 4), (7, 0, 1), (7, 0, 4), (8, 0, 1), (7, 1, 1)} <= have, (M, have)
        assert all(k[1] != 4 or not k[5] for k in r)          # 4-warp CTAs never run persistent
        union |= have
    assert {(4, 0, 1), (8, 0, 4)} <= union, union
    for M in (208, 256):
        r = reachable(M)
        have = {(k[1], k[3], k[5], k[6]) for k in r}   # (nw, wide, persistent, item)
        assert {(8, 0, 0, 1), (8, 0, 0, 4), (8, 0, 1, 1), (8, 1, 1, 1), (8, 1, 1, 4)} <= have, (M, have)
        assert all(k[1] == 8 for k in r)


def test_lone_dense_queries_and_weights():
    # config 5: 65 536 candidates at M = 200 -> persistent grid on the wide build, four per pull
    c = eval_choice(65536, 1, 200, lone=True)
    assert (c["nw"], c["minb"], c["wide"], c["persistent"], c["item"], c["pw"]) == (8, 2, 1, 1, 4, 0), c
    # the same candidates as a batch row never run persistent or wide
    c = eval_choice(65536, 1, 200)
    assert not c["persistent"] and not c["wide"], c
    # with per-scenario weights the 8-warp static build's PW twin (the wide build has none)
    c = eval_choice(65536, 1, 200, lone=True, weights=True)
    assert (c["nw"], c["minb"], c["wide"], c["pw"]) == (8, 3, 0, 1), c
    # C3: 4096 candidates at M = 100 -> 7-warp CTAs, about one wave: static
    c = eval_choice(4096, 1, 100, lone=True)
    assert c["nw"] == 7 and not c["persistent"], c
    # the bench batch: 4-warp CTAs, items of four, on the PW twin when weighted
    c = eval_choice(28, 100000, 100, weights=True)
    assert (c["nw"], c["minb"], c["item"], c["pw"]) == (4, 4, 4, 1), c


def test_debug_eval_choice_rejects_bad_flags():
    out = (C.c_int32 * 13)()
    L = _lib.lib()
    assert L.f1l_debug_eval_choice(28, 2, 100, SM, 0, _lib.EVAL_LONE, out, 13) < 0   # lone needs S = 1
    assert L.f1l_debug_eval_choice(28, 1, 100, SM, 0, 4, out, 13) < 0                # unknown flag
    assert L.f1l_debug_eval_choice(28, 1, 257, SM, 0, 0, out, 13) < 0
