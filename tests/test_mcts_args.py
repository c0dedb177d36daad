"""CPU: the C layout of ge_mcts_tree against its ctypes mirror, the argument checks of ge_mcts_select / ge_mcts_expand
(dummy descriptors, never dereferenced) and the checks of graphenvs_b200.MCTS that need no device."""
import ctypes as C
import os
import subprocess
import tempfile

import pytest
import torch

import graphenvs_b200
from graphenvs_b200 import _native
from graphenvs_b200.mcts import MCTS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _err():
    return _native.lib().ge_last_error().decode()


def test_exported():
    assert {"ge_mcts_select", "ge_mcts_expand"} <= set(_native.EXPORTS)
    assert graphenvs_b200.MCTS is MCTS


def test_tree_struct_matches_c_layout():
    fields = [f[0] for f in _native.MctsTree._fields_]
    prog = "#include <stdio.h>\n#include <stddef.h>\n#include \"graphenvs_b200.h\"\nint main(){printf(\"%zu\\n\", sizeof(ge_mcts_tree));\n"
    for f in fields:
        prog += "printf(\"%%zu\\n\", offsetof(ge_mcts_tree, %s));\n" % f
    prog += "return 0;}\n"
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "t.c")
        open(src, "w").write(prog)
        exe = os.path.join(td, "t")
        subprocess.check_call(["/usr/bin/gcc", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        out = subprocess.check_output([exe]).decode().split()
    assert int(out[0]) == C.sizeof(_native.MctsTree)
    for f, off in zip(fields, out[1:]):
        assert getattr(_native.MctsTree, f).offset == int(off), f


ARRAYS = ("parent", "action", "visits", "wsum", "reward", "value", "terminal", "child", "prior", "mask", "qmin", "qmax",
          "sel_node", "sel_action", "load_index", "depth")


def tree(G=16, S=8, A=50, **fields):
    t = _native.MctsTree()
    t.G, t.S, t.A, t.AW, t.c_puct = G, S, A, (A + 31) // 32, 1.25
    for i, f in enumerate(ARRAYS):
        setattr(t, f, 0x1000000 + 0x100000 * i)
    for k, v in fields.items():
        setattr(t, k, v)
    return t


def leaf(B=16, N=50, M=400, kind=1, **fields):
    d = _native.GeBatch()
    d.kind, d.B, d.N, d.M = kind, B, N, M
    assert _native.lib().ge_fill_layout(C.byref(d)) == 0
    d.mask_bits, d.done = 0x100000, 0x200000
    for k, v in fields.items():
        setattr(d, k, v)
    return d


X, R, V = C.c_void_p(0x300000), C.c_void_p(0x400000), C.c_void_p(0x500000)


def select(t, k=1):
    return _native.lib().ge_mcts_select(None if t is None else C.byref(t), k, None)


def expand(t, k=1, d="default", reward=R, logits=X, dtype=0, value=V):
    d = leaf() if d == "default" else d
    return _native.lib().ge_mcts_expand(None if t is None else C.byref(t), k, None if d is None else C.byref(d), reward, logits,
                                        dtype, value, None)


_TREE_CASES = [
    (lambda t: t(), "null tree"),
    (lambda t: t(tree(G=0)), "bad tree shape"),
    (lambda t: t(tree(S=0)), "bad tree shape"),
    (lambda t: t(tree(A=0)), "bad tree shape"),
    (lambda t: t(tree(AW=1)), "bad tree shape"),
    (lambda t: t(tree(c_puct=-0.5)), "c_puct"),
    (lambda t: t(tree(c_puct=float("nan"))), "c_puct"),
    (lambda t: t(tree(c_puct=float("inf"))), "c_puct"),
    (lambda t: t(tree(), k=9), "k = 9"),
    (lambda t: t(tree(), k=-1), "k = -1"),
] + [(lambda t, f=f: t(tree(**{f: None})), "null tree array") for f in ARRAYS]


@pytest.mark.parametrize("case, match", _TREE_CASES)
def test_select_rejects_bad_arguments(case, match):
    assert case(lambda t=None, k=1: select(t, k)) == -1
    assert match in _err()


def test_select_rejects_k_zero():
    assert select(tree(), 0) == -1 and "k = 0" in _err()


@pytest.mark.parametrize("case, match", _TREE_CASES)
def test_expand_rejects_bad_tree(case, match):
    assert case(lambda t=None, k=1: expand(t, k)) == -1
    assert match in _err()


@pytest.mark.parametrize("case, match", [
    (lambda: expand(tree(), d=None), "null leaf"),
    (lambda: expand(tree(), dtype=2), "dtype 2"),
    (lambda: expand(tree(), dtype=-1), "dtype -1"),
    (lambda: expand(tree(), d=leaf(B=15)), "leaf batch B=15"),
    (lambda: expand(tree(), d=leaf(N=51)), "A=51"),
    (lambda: expand(tree(), reward=None), "null reward"),
    (lambda: expand(tree(), logits=None), "null reward"),
    (lambda: expand(tree(), value=None), "null reward"),
    (lambda: expand(tree(), d=leaf(mask_bits=None)), "mask_bits"),
    (lambda: expand(tree(), d=leaf(done=None)), "done"),
])
def test_expand_rejects_bad_arguments(case, match):
    assert case() == -1
    assert match in _err()


# ------------------------------------------------------------------ the Python layer
def _unloaded(loaded=True):
    from graphenvs_b200.batch import BatchedGraphEnv
    env = BatchedGraphEnv.__new__(BatchedGraphEnv)
    env._loaded = loaded
    return env


@pytest.mark.parametrize("n", [0, -3, 2.0, True, "8", None])
def test_rejects_bad_num_simulations(n):
    with pytest.raises(ValueError, match="num_simulations"):
        MCTS(_unloaded(), n)


@pytest.mark.parametrize("c", [-1.0, float("nan"), float("inf"), "1", True, None])
def test_rejects_bad_c_puct(c):
    with pytest.raises(ValueError, match="c_puct"):
        MCTS(_unloaded(), 8, c)


def test_needs_a_loaded_batch():
    with pytest.raises(ValueError, match="no instances"):
        MCTS(_unloaded(False), 8)
    with pytest.raises(TypeError, match="BatchedGraphEnv"):
        MCTS(object(), 8)


def _shell(G=8, A=40):
    m = MCTS.__new__(MCTS)
    m.G, m.A = G, A
    m.leaf = type("Leaf", (), {})()
    m.leaf.device = torch.device("cpu")
    return m


@pytest.mark.parametrize("out, err, match", [
    ((torch.zeros((8, 40), dtype=torch.float64), torch.zeros(8)), TypeError, "float32 or bfloat16"),
    ((torch.zeros((8, 40)), torch.zeros(8, dtype=torch.float64)), TypeError, "value must be float32"),
    ((torch.zeros((8, 40)), torch.zeros(8, dtype=torch.bfloat16)), TypeError, "value must be float32"),
    ((torch.zeros((8, 41)), torch.zeros(8)), ValueError, "logits shape"),
    ((torch.zeros((4, 40)), torch.zeros(8)), ValueError, "logits shape"),
    ((torch.zeros((8, 40)), torch.zeros(7)), ValueError, "value shape"),
    ((torch.zeros((8, 40)), torch.zeros((8, 1))), ValueError, "value shape"),
    ((torch.zeros((8, 40)).numpy(), torch.zeros(8)), ValueError, "tensor"),
    ((torch.zeros((8, 40)), torch.zeros(8, device="meta")), ValueError, "tensor on cpu"),
    (torch.zeros((8, 40)), TypeError, "return \\(logits, value\\)"),
    ((torch.zeros((8, 40)),), TypeError, "return \\(logits, value\\)"),
])
def test_checks_policy_output(out, err, match):
    with pytest.raises(err, match=match):
        _shell()._policy_out(out)


def test_accepts_a_good_policy_output():
    lg, v = _shell()._policy_out((torch.zeros((8, 40), dtype=torch.bfloat16), torch.zeros(8)))
    assert lg.dtype == torch.bfloat16 and v.shape == (8,)
