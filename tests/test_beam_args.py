"""CPU: argument checks of ge_beam_expand and of BeamSearch that need no device (dummy descriptors, never dereferenced)."""
import ctypes as C

import pytest
import torch

import graphenvs_b200
from graphenvs_b200 import _native
from graphenvs_b200.beam import BeamSearch


def _err():
    return _native.lib().ge_last_error().decode()


def desc(B=64, N=50, M=400, kind=1, **fields):
    d = _native.GeBatch()
    d.kind, d.B, d.N, d.M = kind, B, N, M
    assert _native.lib().ge_fill_layout(C.byref(d)) == 0
    d.mask_bits, d.done = 0x100000, 0x200000
    for k, v in fields.items():
        setattr(d, k, v)
    return d


X = C.c_void_p(0x300000)
SCORE, OUT, PAR, ACT, LOAD = (C.c_void_p(0x400000 + 0x10000 * i) for i in range(5))


def expand(d, W=8, logits=X, dtype=0, score=SCORE, out=OUT, parent=PAR, action=ACT, load=LOAD):
    return _native.lib().ge_beam_expand(None if d is None else C.byref(d), W, logits, dtype, score, out, parent, action, load, None)


def test_exported():
    assert "ge_beam_expand" in _native.EXPORTS
    assert graphenvs_b200.BeamSearch is BeamSearch


@pytest.mark.parametrize("case, match", [
    (lambda: expand(None), "null batch"),
    (lambda: expand(desc(), dtype=2), "dtype 2"),
    (lambda: expand(desc(), dtype=-1), "dtype -1"),
    (lambda: expand(desc(), W=0), "W = 0"),
    (lambda: expand(desc(), W=33), "W = 33"),
    (lambda: expand(desc(), W=-4), "W = -4"),
    (lambda: expand(desc(B=60), W=8), "not a multiple"),
    (lambda: expand(desc(B=64), W=5), "not a multiple"),
    (lambda: expand(desc(B=0), W=1), "bad shape"),
    (lambda: expand(desc(AW=3)), "bad shape"),
    (lambda: expand(desc(), logits=None), "null"),
    (lambda: expand(desc(), score=None), "null"),
    (lambda: expand(desc(), out=None), "null"),
    (lambda: expand(desc(), parent=None), "null"),
    (lambda: expand(desc(), action=None), "null"),
    (lambda: expand(desc(), load=None), "null"),
    (lambda: expand(desc(mask_bits=None)), "mask_bits"),
    (lambda: expand(desc(done=None)), "done"),
    (lambda: expand(desc(), out=SCORE), "overlap"),                                # score_out aliases score
    (lambda: expand(desc(), out=C.c_void_p(0x400000 + 4 * 63)), "overlap"),       # ... or overlaps it
    (lambda: expand(desc(), parent=ACT), "overlap"),
    (lambda: expand(desc(), load=C.c_void_p(0x400000 + 0x10000 * 3 - 8)), "overlap"),
])
def test_expand_rejects_bad_arguments(case, match):
    assert case() == -1
    assert match in _err()


class _Loaded:
    pass


@pytest.mark.parametrize("width", [0, 33, -1, 2.0, True, "8"])
def test_beam_search_rejects_bad_width(width):
    from graphenvs_b200.batch import BatchedGraphEnv
    env = BatchedGraphEnv.__new__(BatchedGraphEnv)
    env._loaded = True
    with pytest.raises(ValueError, match="width"):
        BeamSearch(env, width=width)


def test_beam_search_needs_a_loaded_batch():
    from graphenvs_b200.batch import BatchedGraphEnv
    env = BatchedGraphEnv.__new__(BatchedGraphEnv)
    env._loaded = False
    with pytest.raises(ValueError, match="no instances"):
        BeamSearch(env, width=4)
    with pytest.raises(TypeError, match="BatchedGraphEnv"):
        BeamSearch(object(), width=4)


def _shell(B=8, A=40):
    bs = BeamSearch.__new__(BeamSearch)
    bs.B = B
    bs.wide = _Loaded()
    bs.wide.device = torch.device("cpu")
    bs.wide.desc = _native.GeBatch()
    bs.wide.desc.A = A
    return bs


@pytest.mark.parametrize("bad, err, match", [
    (torch.zeros((8, 40), dtype=torch.float64), TypeError, "float32 or bfloat16"),
    (torch.zeros((8, 41)), ValueError, "shape"),
    (torch.zeros((4, 40)), ValueError, "shape"),
    (torch.zeros((8, 40)).numpy(), ValueError, "tensor"),
])
def test_beam_search_checks_logits(bad, err, match):
    with pytest.raises(err, match=match):
        _shell()._check_logits(bad)
