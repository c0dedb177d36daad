"""CPU: argument checks of ge_beam_expand_sampled and of StochasticBeamSearch that need no device (dummy descriptors, never
dereferenced), and the host-side root keys."""
import ctypes as C
import itertools

import numpy as np
import pytest

import graphenvs_b200
from graphenvs_b200 import _native
from graphenvs_b200.beam import StochasticBeamSearch, root_gumbel, root_key


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
NAMES = ["logp", "key", "node_key", "logp_out", "key_out", "node_key_out", "parent", "action", "load_index", "threshold"]
BASE = {n: 0x400000 + 0x10000 * i for i, n in enumerate(NAMES)}     # 64 KB apart: no overlap at B = 64
SIZE = {n: (8 if n.startswith("node_key") else 4) for n in NAMES}      # bytes per env (threshold: per group)


def expand(d, W=8, logits=X, dtype=0, **ptrs):
    p = {n: C.c_void_p(BASE[n]) for n in NAMES}
    p.update({n: (None if v is None else C.c_void_p(v)) for n, v in ptrs.items()})
    return _native.lib().ge_beam_expand_sampled(None if d is None else C.byref(d), W, logits, dtype, *[p[n] for n in NAMES], None)


def test_exported():
    assert "ge_beam_expand_sampled" in _native.EXPORTS
    assert hasattr(_native.lib(), "ge_beam_expand_sampled")
    assert graphenvs_b200.StochasticBeamSearch is StochasticBeamSearch


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
    (lambda: expand(desc(mask_bits=None)), "mask_bits"),
    (lambda: expand(desc(done=None)), "done"),
] + [(lambda n=n: expand(desc(), **{n: None}), "null") for n in NAMES[:-1]])
def test_expand_rejects_bad_arguments(case, match):
    assert case() == -1
    assert match in _err()


@pytest.mark.parametrize("a, b", list(itertools.combinations(NAMES, 2)))
def test_expand_rejects_each_overlapping_pair(a, b):
    B, W = 64, 8
    n_a = SIZE[a] * (B // W if a == "threshold" else B)
    assert expand(desc(B=B), W=W, **{b: BASE[a]}) == -1                  # b aliases a
    assert "overlap" in _err()
    assert expand(desc(B=B), W=W, **{b: BASE[a] + n_a - 4}) == -1         # b starts on a's last element
    assert "overlap" in _err()
    n_b = SIZE[b] * (B // W if b == "threshold" else B)
    assert expand(desc(B=B), W=W, **{a: BASE[b] + n_b - 4}) == -1         # a starts on b's last element
    assert "overlap" in _err()


def test_adjacent_arrays_and_null_threshold_pass_the_checks():
    """Arrays that touch without overlapping, and threshold = NULL, pass every argument check.  Without a device the call then
    fails at the launch (GE_ERR_CUDA), which shows the checks let it through; with one, the dummy pointers must not reach a
    kernel, and test_cuda_stochastic_beam covers threshold = NULL on real buffers."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device would run the kernel on dummy pointers")
    d = desc(B=64)
    touching = {n: 0x400000 + 512 * i for i, n in enumerate(NAMES)}     # back to back: 512 bytes = 8 bytes x 64 envs
    for ptrs in (touching, dict(touching, threshold=None), {"threshold": None}):
        assert expand(d, **ptrs) == -2
        assert "launch" in _err()


# ------------------------------------------------------------------ the decoder's own checks
class _Loaded:
    pass


def _env(loaded=True):
    from graphenvs_b200.batch import BatchedGraphEnv
    env = BatchedGraphEnv.__new__(BatchedGraphEnv)
    env._loaded = loaded
    return env


@pytest.mark.parametrize("width", [0, 33, -1, 2.0, True, "8"])
def test_rejects_bad_width(width):
    with pytest.raises(ValueError, match="width"):
        StochasticBeamSearch(_env(), width=width, seed=0)


@pytest.mark.parametrize("seed", [1.0, "3", None, True, np.float32(2)])
def test_rejects_a_seed_that_is_not_an_int(seed):
    with pytest.raises(TypeError, match="seed"):
        StochasticBeamSearch(_env(), width=4, seed=seed)


@pytest.mark.parametrize("seed", [-1, 1 << 64])
def test_rejects_a_seed_out_of_range(seed):
    with pytest.raises(ValueError, match="seed"):
        StochasticBeamSearch(_env(), width=4, seed=seed)


def test_needs_a_loaded_batch():
    with pytest.raises(ValueError, match="no instances"):
        StochasticBeamSearch(_env(loaded=False), width=4, seed=0)
    with pytest.raises(TypeError, match="BatchedGraphEnv"):
        StochasticBeamSearch(object(), width=4, seed=0)


# ------------------------------------------------------------------ root keys (restated from include/graphenvs_b200.h)
def _mix32(seed, env, t):
    M = (1 << 64) - 1
    z = (seed + 0x9E3779B97F4A7C15 * (env * 0x100000001 + ((t << 32) | 0x5bd1e995))) & M
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M
    return (z ^ (z >> 31)) >> 32


def test_root_keys_follow_the_documented_formula():
    for seed in (0, 1, 12345, (1 << 64) - 1):
        ids = np.array([0, 1, 7, 1 << 20, (1 << 32) - 1], dtype=np.uint64)
        got = root_key(seed, ids)
        for i, k in zip(ids.tolist(), got.tolist()):
            assert k == (_mix32(seed, i, 0x52DCE729) << 32) | _mix32(seed ^ 0xD1B54A32D192ED03, i, 0x52DCE729)
            h = _mix32(k, 0xFFFFFFFF, 0x85EBCA6B)
            u = ((h >> 8) + 0.5) / 2.0 ** 24
            assert root_gumbel(np.uint64(k)) == -np.log(-np.log(u))
