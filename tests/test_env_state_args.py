"""CPU: the state-record layout (ge_state_record_bytes) and the argument checks of ge_state_save / ge_state_load /
ge_gather_instances and of BatchedGraphEnv.save_states / load_states / gather_instances, none of which needs a device."""
import ctypes as C

import numpy as np
import pytest
import torch

from graphenvs_b200 import _native
from graphenvs_b200.batch import STATE_ALL, STATE_CLOCK, STATE_DYNAMIC, STATE_STATS, BatchedGraphEnv, EnvStates

# (name, element bytes, elements per env) in record order; include/graphenvs_b200.h, GE_STATE_*
STATE = [("head", 4, lambda d: 1), ("node_bits", 4, lambda d: d.NW), ("node_bits2", 4, lambda d: d.NW),
         ("edge_bits", 4, lambda d: d.MW), ("dist32", 4, lambda d: d.N), ("bestkey", 8, lambda d: d.N), ("cost", 8, lambda d: 1),
         ("counters", 4, lambda d: 4), ("done", 1, lambda d: 1), ("mask_bits", 4, lambda d: d.AW), ("mask_cnt", 4, lambda d: 8),
         ("env_steps", 4, lambda d: 1), ("acc", 8, lambda d: 4), ("traj", 8, lambda d: 1)]


def layout_bytes(d, present):
    """The layout rule restated: sections of <= 64 bytes per env first at natural alignment, then, from a 16-byte boundary,
    the larger ones at 16-byte offsets; the record is rounded up to 16 bytes."""
    al = lambda x, a: (x + a - 1) // a * a  # noqa: E731
    off = 0
    for name, esz, n in STATE:
        if name in present and esz * n(d) <= 64:
            off = al(off, esz) + esz * n(d)
    off = al(off, 16)
    for name, esz, n in STATE:
        if name in present and esz * n(d) > 64:
            off = al(off, 16) + esz * n(d)
    return al(off, 16)


def desc(kind, B, N, M, present=(), **fields):
    d = _native.GeBatch()
    d.kind, d.B, d.N, d.M = kind, B, N, M
    for k, v in fields.items():
        setattr(d, k, v)
    assert _native.lib().ge_fill_layout(C.byref(d)) == 0
    for i, name in enumerate(present):
        setattr(d, name, 0x100000 * (i + 1))    # dummy, 16-byte aligned, never dereferenced
    return d


BASE = ("head", "node_bits", "cost", "counters", "done", "mask_bits", "acc", "traj")
KINDS = [   # (kind, N, M, extra state arrays): every kind, with the arrays BatchedGraphEnv gives it
    (0, 10, 30, ()), (0, 300, 1400, ()), (1, 50, 400, ("env_steps",)), (2, 100, 1000, ("mask_cnt",)), (3, 200, 39800, ()),
    (4, 50, 200, ()), (5, 80, 400, ("node_bits2",)), (6, 500, 8000, ("edge_bits", "dist32", "bestkey", "mask_cnt", "env_steps")),
    (6, 120, 1200, ("edge_bits", "dist32")), (7, 500, 8000, ("node_bits2",)), (8, 40, 200, ()),
]


@pytest.mark.parametrize("kind, N, M, extra", KINDS, ids=["k%d-N%d" % (k[0], k[1]) for k in KINDS])
def test_record_bytes_follow_the_layout_rule(kind, N, M, extra):
    present = BASE + extra
    d = desc(kind, 1000, N, M, present)
    got = _native.lib().ge_state_record_bytes(C.byref(d))
    assert got == layout_bytes(d, present)
    assert got % 16 == 0
    # an absent array has no section
    d2 = desc(kind, 1000, N, M, tuple(p for p in present if p != "traj"))
    assert _native.lib().ge_state_record_bytes(C.byref(d2)) == layout_bytes(d2, tuple(p for p in present if p != "traj"))


def test_record_sizes_quoted_in_the_docs():
    d = desc(1, 65536, 50, 400, BASE)                   # cfg2 LongestPath: about 100 bytes
    assert layout_bytes(d, BASE) == 96 == _native.lib().ge_state_record_bytes(C.byref(d))
    mc = BASE + ("edge_bits", "dist32", "bestkey", "mask_cnt")
    d = desc(6, 131072, 500, 8000, mc, parenting=4)   # cfg5 Multicast: about 8.3 KB
    assert 8000 < _native.lib().ge_state_record_bytes(C.byref(d)) == layout_bytes(d, mc) < 8400


def _err():
    return _native.lib().ge_last_error().decode()


def test_save_and_load_reject_bad_arguments():
    L = _native.lib()
    d = desc(1, 64, 50, 400, BASE)
    x = C.c_void_p(0x200000)
    assert L.ge_state_record_bytes(None) == -1
    assert L.ge_state_save(None, None, 4, x, None) == -1 and "null batch" in _err()
    assert L.ge_state_save(C.byref(d), None, 65, x, None) == -1 and "count 65" in _err()
    assert L.ge_state_save(C.byref(d), None, -1, x, None) == -1
    assert L.ge_state_save(C.byref(d), None, 4, None, None) == -1 and "records" in _err()
    assert L.ge_state_save(C.byref(d), None, 4, C.c_void_p(0x200004), None) == -1 and "16-byte aligned" in _err()
    assert L.ge_state_load(C.byref(d), x, 64, None, STATE_CLOCK, None) == -1 and "GE_STATE_DYNAMIC" in _err()
    assert L.ge_state_load(C.byref(d), x, 64, None, STATE_STATS | STATE_CLOCK, None) == -1
    assert L.ge_state_load(C.byref(d), x, 64, None, STATE_ALL | 8, None) == -1
    assert L.ge_state_load(C.byref(d), x, 63, None, STATE_ALL, None) == -1 and "n_records 63 < B 64" in _err()
    assert L.ge_state_load(C.byref(d), x, -1, x, STATE_ALL, None) == -1
    assert L.ge_state_load(C.byref(d), None, 64, None, STATE_ALL, None) == -1 and "records" in _err()
    raw = _native.GeBatch()                         # layout never filled
    raw.kind, raw.B, raw.N, raw.M = 1, 64, 50, 400
    assert L.ge_state_record_bytes(C.byref(raw)) == -1 and "ge_fill_layout" in _err()
    # nothing to do: no device work, success
    assert L.ge_state_save(C.byref(d), None, 0, None, None) == 0
    assert L.ge_state_load(C.byref(d), None, 0, x, STATE_DYNAMIC, None) == 0


STATIC = ("row_ptr", "col", "w64", "adj_bits", "wsort", "src", "dest", "heuristic")


def _pair(**dst_fields):
    """Two ShortestPath N=300 descriptors whose static arrays live at disjoint dummy addresses."""
    dst = desc(0, 64, 300, 1400)
    src = desc(0, 128, 300, 1400)
    for i, name in enumerate(STATIC):
        setattr(dst, name, 0x10000000 * (i + 1))
        setattr(src, name, 0x10000000 * (i + 1) + 0x8000000)
    for k, v in dst_fields.items():
        setattr(dst, k, v)
    return dst, src


@pytest.mark.parametrize("field, value, match", [
    ("N", 301, "not shaped like"), ("M", 1402, "not shaped like"), ("kind", 1, "not shaped like"),
    ("parenting", 3, "not shaped like"), ("n_dests", 2, "not shaped like"), ("n_choices", 5, "not shaped like"),
    ("n_targets", 7, "not shaped like"), ("max_distance", 0.5, "not shaped like"), ("flags", 8, "not shaped like"),
    ("dfa_bytes", 40, "dfa_bytes"),
])
def test_gather_rejects_mismatched_batches(field, value, match):
    dst, src = _pair()
    if field in ("N", "M", "kind"):
        setattr(dst, field, value)
        _native.lib().ge_fill_layout(C.byref(dst))
    else:
        setattr(dst, field, value)
    assert _native.lib().ge_gather_instances(C.byref(dst), C.byref(src), None, None) == -1
    assert match in _err()


def test_gather_rejects_missing_arrays_overlap_and_short_sources():
    L = _native.lib()
    idx = C.c_void_p(0x300000)
    dst, src = _pair(wmat=0x7f0000000)                   # dst carries an array src lacks
    assert L.ge_gather_instances(C.byref(dst), C.byref(src), idx, None) == -1 and "lacks" in _err()
    dst, src = _pair()
    src.col = dst.col + 64 * dst.MP * 4 - 4              # src's col starts inside dst's last col row
    assert L.ge_gather_instances(C.byref(dst), C.byref(src), idx, None) == -1 and "overlap" in _err()
    dst, src = _pair()
    src.heuristic = dst.row_ptr                          # different arrays may not overlap either
    assert L.ge_gather_instances(C.byref(dst), C.byref(src), idx, None) == -1 and "overlap" in _err()
    assert L.ge_gather_instances(C.byref(src), C.byref(src), idx, None) == -1 and "overlap" in _err()
    dst, src = _pair()
    dst.B, src.B = 128, 64                               # without an index every dst env needs its own src env
    src.acc_stride = dst.acc_stride = 128
    assert L.ge_gather_instances(C.byref(dst), C.byref(src), None, None) == -1 and "src B 64 < dst B 128" in _err()
    assert L.ge_gather_instances(None, C.byref(src), idx, None) == -1


# ------------------------------------------------------------------ the Python layer: checks before any native call
class _NoNative:
    def __getattr__(self, name):
        raise AssertionError("native library reached (%s)" % name)


def bare_env(env_id="LongestPath-v0", B=8, N=50, M=400, kind=1, parenting=2, clock=False, dfa=None):
    """A BatchedGraphEnv shell on the CPU: descriptor and state dict only; any native call fails the test."""
    env = BatchedGraphEnv.__new__(BatchedGraphEnv)
    env.lib = _NoNative()
    env.env_id, env.B, env.N, env.M = env_id, B, N, M
    env.device = torch.device("cpu")
    d = _native.GeBatch()
    d.kind, d.B, d.N, d.M, d.parenting = kind, B, N, M, parenting
    env.desc = d
    env.t = {k: torch.zeros(1) for k in BASE}
    if dfa is not None:
        env.t["dfa"] = dfa
    env.env_steps = torch.zeros(B, dtype=torch.int32) if clock else None
    env._loaded = True
    return env


def _states(env, n, sig=None):
    return EnvStates(torch.zeros((n, 96), dtype=torch.uint8), sig if sig is not None else env.state_signature())


@pytest.mark.parametrize("case, err, match", [
    (lambda e: e.load_states(_states(e, 8, bare_env(parenting=3).state_signature())), ValueError, "signature"),
    (lambda e: e.load_states(_states(e, 8, bare_env(clock=True).state_signature())), ValueError, "signature"),
    (lambda e: e.load_states(_states(e, 8, bare_env("ShortestPath-v0", kind=0).state_signature())), ValueError, "signature"),
    (lambda e: e.load_states(torch.zeros((8, 96), dtype=torch.uint8)), TypeError, "EnvStates"),
    (lambda e: e.load_states(_states(e, 4)), ValueError, "4 records for 8 envs"),
    (lambda e: e.load_states(_states(e, 4), [0, 1, 2, 3, 4, 0, 1, 2]), ValueError, r"\[-1, 4\)"),
    (lambda e: e.load_states(_states(e, 4), [0, 1, 2, 3, -2, 0, 1, 2]), ValueError, r"\[-1, 4\)"),
    (lambda e: e.load_states(_states(e, 4), np.zeros(7, np.int64)), ValueError, "8 entries"),
    (lambda e: e.load_states(_states(e, 4), np.zeros(8, np.float32)), ValueError, "integer"),
    (lambda e: e.load_states(_states(e, 8), torch.full((8,), 8)), ValueError, r"\[-1, 8\)"),
    (lambda e: e.save_states([0, 8]), ValueError, r"\[0, 8\)"),
    (lambda e: e.save_states([-1]), ValueError, r"\[0, 8\)"),
    (lambda e: e.save_states(list(range(8)) * 2), ValueError, "<= 8"),
    (lambda e: e.gather_instances(bare_env(B=4), [0, 1, 2, 3, 4, 0, 0, 0]), ValueError, r"\[-1, 4\)"),
    (lambda e: e.gather_instances(bare_env(B=4)), ValueError, "pass an index"),
    (lambda e: e.gather_instances(bare_env("ShortestPath-v0", kind=0)), ValueError, "loaded LongestPath"),
    (lambda e: e.gather_instances(e), ValueError, "another batch"),
    (lambda e: e.gather_instances(object()), TypeError, "BatchedGraphEnv"),
])
def test_python_checks_raise_before_any_native_call(case, err, match):
    with pytest.raises(err, match=match):
        case(bare_env())


def test_python_gather_checks_the_distance_automaton_first():
    a, b = torch.tensor([3, 2, 1], dtype=torch.uint8), torch.tensor([3, 2, 2], dtype=torch.uint8)
    dc = dict(env_id="DistributionCenter-v0", kind=7, N=120, M=1000)
    with pytest.raises(ValueError, match="different distance automata"):
        bare_env(**dc, dfa=a).gather_instances(bare_env(**dc, dfa=b))
    with pytest.raises(ValueError, match="covers every env"):     # dst without an automaton, partial gather
        bare_env(**dc).gather_instances(bare_env(**dc, dfa=a), [0, 1, 2, -1, 0, 1, 2, 3])
    with pytest.raises(ValueError, match="covers every env"):     # dst with one, src without
        bare_env(**dc, dfa=a).gather_instances(bare_env(**dc))
