"""CPU: the C-ABI library loads and exports every symbol include/graphenvs_b200.h declares, the
ctypes mirror of `ge_batch` matches the C layout, host-side helpers behave, and the product
package never touches oracle/."""
import ctypes as C
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from graphenvs_b200 import _native, spec, utils

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "graphenvs_b200.h")


def _declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ge_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_the_declared_symbols_and_abi_version():
    path = _native.build()
    lib = C.CDLL(path)
    syms = _declared_symbols()
    assert len(syms) >= 15
    for s in syms:
        assert hasattr(lib, s), "missing export %s" % s
    assert sorted(_native.EXPORTS) == syms
    lib.ge_abi_version.restype = C.c_int
    assert lib.ge_abi_version() == 4


def test_ctypes_struct_matches_c_layout():
    """sizeof/offsetof of ge_batch as the C compiler sees it == the ctypes mirror."""
    fields = [f[0] for f in _native.GeBatch._fields_]
    prog = "#include <stdio.h>\n#include <stddef.h>\n#include \"graphenvs_b200.h\"\nint main(){printf(\"%zu\\n\", sizeof(ge_batch));\n"
    for f in fields:
        prog += "printf(\"%%zu\\n\", offsetof(ge_batch, %s));\n" % f
    prog += "printf(\"%zu %zu\\n\", sizeof(ge_step_flags), sizeof(ge_step_out)); return 0;}\n"
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "l.c")
        open(src, "w").write(prog)
        exe = os.path.join(td, "l")
        subprocess.check_call(["/usr/bin/gcc", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        out = subprocess.check_output([exe]).decode().split()
    assert int(out[0]) == C.sizeof(_native.GeBatch)
    for f, off in zip(fields, out[1:1 + len(fields)]):
        assert getattr(_native.GeBatch, f).offset == int(off), f
    assert int(out[-2]) == C.sizeof(_native.StepFlags) == 4
    assert int(out[-1]) == C.sizeof(_native.StepOut)


def test_fill_layout_and_arg_errors_without_gpu():
    L = _native.lib()
    d = _native.GeBatch()
    d.kind, d.B, d.N, d.M = 6, 4, 500, 8000
    assert L.ge_fill_layout(C.byref(d)) == 0
    assert (d.NW, d.MW, d.A, d.AW, d.AP) == (16, 250, 8000, 250, 8000)
    assert d.RP % 4 == 0 and d.MP % 4 == 0 and d.ADJS % 4 == 0
    d2 = _native.GeBatch()
    d2.kind, d2.B, d2.N, d2.M = 99, 1, 10, 40
    L.ge_fill_layout(C.byref(d2))
    assert L.ge_reset(C.byref(d2), None, None) == -1       # GE_ERR_ARG, no CUDA call made
    assert b"unknown kind" in L.ge_last_error()


def test_engine_refuses_to_run_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from graphenvs_b200 import BatchedGraphEnv
    with pytest.raises(_native.NativeError):
        BatchedGraphEnv("ShortestPath-v0", 4, 10, 20)


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "graphenvs_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f
                assert "libgraphenvs_oracle" not in txt, f


def test_env_info_table_and_vectorize_roundtrip():
    exp = {"ShortestPath-v0": (7, 1, "node"), "SteinerTree-v0": (7, 2, "edge"), "MaxIndependentSet-v0": (7, 1, "node"),
           "TSP-v0": (9, 1, "node"), "DistributionCenter-v0": (10, 1, "node"), "MulticastRouting-v0": (9, 2, "edge"),
           "LongestPath-v0": (7, 1, "node"), "DensestSubgraph-v0": (6, 1, "node")}
    for k, v in exp.items():
        assert spec.get_env_info(k) == v                    # graph_envs/utils.py:32-73
    with pytest.raises(AssertionError):
        spec.get_env_info("Nope-v0")
    rng = np.random.default_rng(0)
    N, E = 6, 9
    g = utils.GraphInstance(rng.random((N, 9), dtype=np.float32), rng.random((2 * E, 2), dtype=np.float32),
                            rng.integers(0, N, (2 * E, 2)).astype(np.int64))
    v = utils.vectorize_graph(g)
    assert v.dtype == np.float32 and v.shape == (N * 9 + 2 * E * 2 + 4 * E,)
    x, ef, ei = utils.devectorize_graph(v[None, :], "MulticastRouting-v0", n_nodes=N, n_edges=E)
    np.testing.assert_array_equal(x[0], g.nodes)
    np.testing.assert_array_equal(ef[0], g.edges)
    np.testing.assert_array_equal(ei[0], g.edge_links)   # reference test_max_independent_set.py:26-31 round trip


def test_registry_ids():
    from graphenvs_b200 import registration
    assert sorted(registration.registry) == sorted(spec.ENV_SPECS)
    assert "PerishableProductDelivery-v0" in registration.registry      # round 2: the ninth reference id
    with pytest.raises(KeyError):
        registration.make("NoSuchEnv-v0", n_nodes=5, n_edges=6)
    with pytest.raises(AssertionError):                                   # perishable_product_delivery.py:29
        spec.check_ctor_args("PerishableProductDelivery-v0", 10, 20, {"parenting": 2})


def test_flags8_decoding_matches_the_header_macros():
    """BatchedGraphEnv.unpack_flags8 (compact host results, ge_step_host_compact) = GE_FLAGS8_* of include/graphenvs_b200.h."""
    import numpy as np
    from graphenvs_b200.batch import BatchedGraphEnv
    cases = [(d, s, st, h) for d in (0, 1) for s in (-1, 0, 1) for st in (0, 1, 2) for h in (0, 1)]
    f8 = np.array([d | (s + 1) << 1 | st << 3 | h << 5 for d, s, st, h in cases], dtype=np.uint8)
    done, solved, status, has_mask = BatchedGraphEnv.unpack_flags8(f8)
    for i, (d, s, st, h) in enumerate(cases):
        assert (int(done[i]), int(solved[i]), int(status[i]), int(has_mask[i])) == (d, s, st, h)
    hdr = open(os.path.join(ROOT, "include", "graphenvs_b200.h")).read()
    for macro in ("GE_FLAGS8_DONE(f) ((f) & 1)", "GE_FLAGS8_SOLVED(f) ((int)(((f) >> 1) & 3) - 1)", "GE_FLAGS8_STATUS(f) (((f) >> 3) & 3)",
                  "GE_FLAGS8_HAS_MASK(f) (((f) >> 5) & 1)"):
        assert macro in hdr
