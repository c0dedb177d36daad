"""CPU: the C layout of ge_gumbel_params against its ctypes mirror, the argument checks of ge_gumbel_root / ge_gumbel_select /
ge_gumbel_result and of ge_mcts_select on a log-prior tree (dummy descriptors, never dereferenced), the host table of considered
visits against mctx's sequence function, and the checks of graphenvs_b200.GumbelMCTS that need no device."""
import ctypes as C
import math
import os
import subprocess
import tempfile

import pytest

import graphenvs_b200
from graphenvs_b200 import _native
from graphenvs_b200.mcts import GumbelMCTS, MCTS, considered_visits_table
from test_mcts_args import _err, _unloaded, tree

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOG_PRIOR = 32


def test_exported():
    assert {"ge_gumbel_root", "ge_gumbel_select", "ge_gumbel_result"} <= set(_native.EXPORTS)
    assert graphenvs_b200.GumbelMCTS is GumbelMCTS and issubclass(GumbelMCTS, MCTS)


def test_params_struct_matches_c_layout():
    fields = [f[0] for f in _native.GumbelParams._fields_]
    prog = ("#include <stdio.h>\n#include <stddef.h>\n#include \"graphenvs_b200.h\"\n"
            "int main(){printf(\"%zu %d\\n\", sizeof(ge_gumbel_params), GE_MCTS_LOG_PRIOR);\n")
    for f in fields:
        prog += "printf(\"%%zu\\n\", offsetof(ge_gumbel_params, %s));\n" % f
    prog += "return 0;}\n"
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "t.c")
        open(src, "w").write(prog)
        exe = os.path.join(td, "t")
        subprocess.check_call(["/usr/bin/gcc", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        out = subprocess.check_output([exe]).decode().split()
    assert int(out[0]) == C.sizeof(_native.GumbelParams)
    assert int(out[1]) == LOG_PRIOR
    for f, off in zip(fields, out[2:]):
        assert getattr(_native.GumbelParams, f).offset == int(off), f


def params(**fields):
    p = _native.GumbelParams()
    p.m, p.value_scale, p.maxvisit_init, p.table, p.noise = 16, 0.1, 50.0, 0x600000, 0x700000
    for k, v in fields.items():
        setattr(p, k, v)
    return p


def gtree(**fields):
    fields.setdefault("flags", LOG_PRIOR)
    return tree(**fields)


A_, P_, Q_ = C.c_void_p(0x800000), C.c_void_p(0x900000), C.c_void_p(0xA00000)


def _byref(x):
    return None if x is None else C.byref(x)


def root(t, p, k=None):
    return _native.lib().ge_gumbel_root(_byref(t), _byref(p), 7, 0, 0, None)


def select(t, p, k=1):
    return _native.lib().ge_gumbel_select(_byref(t), _byref(p), k, None)


def result(t, p, k=None, action=A_, policy=P_, cq=Q_):
    return _native.lib().ge_gumbel_result(_byref(t), _byref(p), action, policy, cq, None)


_CASES = [
    (lambda f: f(None, params()), "null tree"),
    (lambda f: f(gtree(G=0), params()), "bad tree shape"),
    (lambda f: f(gtree(AW=1), params()), "bad tree shape"),
    (lambda f: f(gtree(c_puct=float("nan")), params()), "c_puct"),
    (lambda f: f(gtree(flags=0), params()), "GE_MCTS_LOG_PRIOR"),
    (lambda f: f(gtree(flags=16), params()), "GE_MCTS_LOG_PRIOR"),
    (lambda f: f(gtree(), None), "null params"),
    (lambda f: f(gtree(), params(m=0)), "m = 0"),
    (lambda f: f(gtree(), params(m=-3)), "m = -3"),
    (lambda f: f(gtree(), params(value_scale=-0.1)), "value_scale"),
    (lambda f: f(gtree(), params(value_scale=float("nan"))), "value_scale"),
    (lambda f: f(gtree(), params(value_scale=float("inf"))), "value_scale"),
    (lambda f: f(gtree(), params(maxvisit_init=-1.0)), "maxvisit_init"),
    (lambda f: f(gtree(), params(maxvisit_init=float("nan"))), "maxvisit_init"),
    (lambda f: f(gtree(), params(maxvisit_init=float("inf"))), "maxvisit_init"),
    (lambda f: f(gtree(), params(table=None)), "null table"),
    (lambda f: f(gtree(), params(noise=None)), "null table / noise"),
] + [(lambda f, a=a: f(gtree(**{a: None}), params()), "null tree array") for a in ("child", "prior", "mask", "visits", "sel_node")]


@pytest.mark.parametrize("entry", [root, select, result], ids=["root", "select", "result"])
@pytest.mark.parametrize("case, match", _CASES)
def test_rejects_bad_arguments(entry, case, match):
    assert case(entry) == -1
    assert match in _err()


@pytest.mark.parametrize("k", [0, -1, 9])
def test_select_rejects_k_out_of_range(k):
    assert select(gtree(), params(), k) == -1 and ("k = %d" % k) in _err()


@pytest.mark.parametrize("kw, match", [(dict(action=None), "null action"), (dict(policy=None), "null action"),
                                       (dict(cq=None), "completed_q")])
def test_result_rejects_null_outputs(kw, match):
    assert result(gtree(), params(), **kw) == -1
    assert match in _err()


def test_puct_select_refuses_a_log_prior_tree():
    assert _native.lib().ge_mcts_select(C.byref(gtree()), 1, None) == -1
    assert "GE_MCTS_LOG_PRIOR" in _err()
    assert _native.lib().ge_mcts_select(C.byref(gtree(flags=LOG_PRIOR | 16)), 1, None) == -1


# ------------------------------------------------------------------ the table of considered visits
def mctx_sequence(m, S):
    """mctx/_src/seq_halving.py: get_sequence_of_considered_visits, restated."""
    if m <= 1:
        return tuple(range(S))
    log2max = int(math.ceil(math.log2(m)))
    sequence, visits, num_considered = [], [0] * m, m
    while len(sequence) < S:
        num_extra_visits = max(1, int(S / (log2max * num_considered)))
        for _ in range(num_extra_visits):
            sequence.extend(visits[:num_considered])
            for i in range(num_considered):
                visits[i] += 1
        num_considered = max(2, num_considered // 2)
    return tuple(sequence[:S])


@pytest.mark.parametrize("m, S, row", [
    (1, 4, [0, 1, 2, 3]),
    (2, 6, [0, 0, 1, 1, 2, 2]),
    (3, 7, [0, 0, 0, 1, 1, 2, 2]),
    (4, 8, [0, 0, 0, 0, 1, 1, 2, 2]),
    (4, 16, [0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5]),
    (16, 16, [0] * 16),
])
def test_table_reference_rows(m, S, row):
    tab = considered_visits_table(m, S)
    assert len(tab) == m + 1 and all(len(r) == S for r in tab)
    assert tab[m] == row


def test_table_equals_mctx_up_to_32_and_256():
    for S in list(range(1, 65)) + [96, 100, 128, 200, 255, 256]:
        tab = considered_visits_table(32, S)
        for m in range(33):
            assert tuple(tab[m]) == mctx_sequence(m, S), (m, S)
            assert tab[m] == considered_visits_table(m, S)[m]


# ------------------------------------------------------------------ the Python layer
@pytest.mark.parametrize("kw, match", [
    (dict(max_considered=0), "max_considered"), (dict(max_considered=2.0), "max_considered"),
    (dict(max_considered=True), "max_considered"), (dict(max_considered=None), "max_considered"),
    (dict(value_scale=-0.1), "value_scale"), (dict(value_scale=float("nan")), "value_scale"),
    (dict(value_scale=float("inf")), "value_scale"), (dict(value_scale="0.1"), "value_scale"),
    (dict(maxvisit_init=-1), "maxvisit_init"), (dict(maxvisit_init=float("inf")), "maxvisit_init"),
    (dict(maxvisit_init=None), "maxvisit_init"),
    (dict(seed=-1), "seed"), (dict(seed=1 << 64), "seed"), (dict(seed=1.5), "seed"), (dict(seed=True), "seed"),
])
def test_rejects_bad_arguments_without_a_device(kw, match):
    with pytest.raises(ValueError, match=match):
        GumbelMCTS(_unloaded(), 8, **kw)


def test_inherits_the_base_checks():
    with pytest.raises(ValueError, match="num_simulations"):
        GumbelMCTS(_unloaded(), 0)
    with pytest.raises(ValueError, match="no instances"):
        GumbelMCTS(_unloaded(False), 8)
    with pytest.raises(TypeError, match="BatchedGraphEnv"):
        GumbelMCTS(object(), 8)
