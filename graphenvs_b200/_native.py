"""ctypes binding of libgraphenvs_b200.so (include/graphenvs_b200.h).

There is NO fallback: if the CUDA library is missing or fails to load, importing the engine
raises.  `build()` compiles it in-tree with nvcc for sm_100a (works without a GPU).
"""
import ctypes as C
import glob
import os
import shutil
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)
LIB_PATH = os.path.join(_PKG, "libgraphenvs_b200.so")
_SOURCES = sorted(glob.glob(os.path.join(_PKG, "csrc", "*.cu")))
_HEADERS = sorted(glob.glob(os.path.join(_PKG, "csrc", "*.cuh"))) + [os.path.join(_ROOT, "include", "graphenvs_b200.h")]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "--expt-extended-lambda", "-Xcompiler", "-fPIC", "-shared"]


def _stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(p) > t for p in _SOURCES + _HEADERS if os.path.exists(p))


def build(force=False, verbose=False):
    """nvcc -> graphenvs_b200/libgraphenvs_b200.so (sm_100a, -lineinfo).  Every .cu is compiled to an object
    in graphenvs_b200/_build/ (in parallel, only when stale), then linked."""
    if not force and not _stale():
        return LIB_PATH
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: cannot build libgraphenvs_b200.so")
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    bdir = os.path.join(_PKG, "_build")
    os.makedirs(bdir, exist_ok=True)
    flags = [f for f in NVCC_FLAGS if f != "-shared"]
    extra = ["-Xptxas=-v"] if verbose else []
    tag = os.path.join(bdir, "flags.txt")
    flag_sig = " ".join(flags + extra)
    same_flags = os.path.exists(tag) and open(tag).read() == flag_sig
    hdr_time = max(os.path.getmtime(p) for p in _HEADERS if os.path.exists(p))
    jobs, objs = [], []
    for src in _SOURCES:
        obj = os.path.join(bdir, os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        fresh = (not force and same_flags and os.path.exists(obj)
                 and os.path.getmtime(obj) > max(os.path.getmtime(src), hdr_time))
        if not fresh:
            cmd = [nvcc] + flags + extra + ["-I", os.path.join(_ROOT, "include"), "-I", os.path.join(_PKG, "csrc"), "-c", src, "-o", obj]
            jobs.append((src, subprocess.Popen(cmd, env=env)))
    failed = [src for src, p in jobs if p.wait() != 0]
    if failed:
        raise RuntimeError("nvcc failed for %s" % ", ".join(os.path.basename(f) for f in failed))
    open(tag, "w").write(flag_sig)
    subprocess.check_call([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB_PATH] + objs + ["-ldl"], env=env)
    return LIB_PATH


class StepFlags(C.Structure):
    _fields_ = [("done", C.c_uint8), ("solved", C.c_int8), ("status", C.c_uint8), ("has_mask", C.c_uint8)]


_P = C.c_void_p


class GeBatch(C.Structure):
    """Mirror of `struct ge_batch` (include/graphenvs_b200.h) -- keep field order in sync."""
    _fields_ = [
        ("kind", C.c_int32), ("B", C.c_int32), ("N", C.c_int32), ("M", C.c_int32),
        ("parenting", C.c_int32), ("n_dests", C.c_int32), ("n_choices", C.c_int32), ("n_targets", C.c_int32),
        ("flags", C.c_uint32), ("env_id0", C.c_int32),
        ("NW", C.c_int32), ("MW", C.c_int32), ("A", C.c_int32), ("AW", C.c_int32), ("AP", C.c_int32),
        ("RP", C.c_int32), ("MP", C.c_int32), ("ADJS", C.c_int32), ("acc_stride", C.c_int32), ("dfa_bytes", C.c_int32),
        ("max_distance", C.c_double),
        ("row_ptr", _P), ("col", _P), ("w32", _P), ("w64", _P), ("adj_bits", _P), ("rev", _P), ("esrc", _P), ("wsort", _P), ("wcode", _P), ("dfa", _P), ("dc_edges", _P), ("wmin", _P), ("wmat", _P),
        ("src", _P), ("dest", _P), ("target_bits", _P), ("node_cost", _P), ("node_xy", _P),
        ("max_dist32", _P), ("targets", _P), ("in_range", _P), ("heuristic", _P), ("heuristic_alt", _P), ("features", _P),
        ("head", _P), ("node_bits", _P), ("node_bits2", _P), ("edge_bits", _P), ("dist32", _P), ("bestkey", _P),
        ("cost", _P), ("counters", _P), ("done", _P), ("mask_bits", _P), ("mask_cnt", _P), ("mask_bytes", _P), ("mask0_bits", _P), ("acc", _P), ("traj", _P), ("env_steps", _P), ("obs_x", _P), ("dc_rows", _P), ("progress", _P),
    ]


class StepOut(C.Structure):
    _fields_ = [("reward", _P), ("flags", _P), ("solution_cost", _P)]


class MctsTree(C.Structure):
    """Mirror of `struct ge_mcts_tree` (include/graphenvs_b200.h) -- keep field order in sync."""
    _fields_ = [
        ("G", C.c_int32), ("S", C.c_int32), ("A", C.c_int32), ("AW", C.c_int32), ("flags", C.c_uint32), ("c_puct", C.c_double),
        ("parent", _P), ("action", _P), ("visits", _P), ("wsum", _P), ("reward", _P), ("value", _P), ("terminal", _P),
        ("child", _P), ("prior", _P), ("mask", _P), ("qmin", _P), ("qmax", _P),
        ("sel_node", _P), ("sel_action", _P), ("load_index", _P), ("depth", _P),
    ]


class GumbelParams(C.Structure):
    """Mirror of `struct ge_gumbel_params` (include/graphenvs_b200.h) -- keep field order in sync."""
    _fields_ = [("m", C.c_int32), ("value_scale", C.c_double), ("maxvisit_init", C.c_double), ("table", _P), ("noise", _P)]


EXPORTS = ["ge_abi_version", "ge_last_error", "ge_fill_layout", "ge_step_smem_bytes", "ge_build_adjacency",
           "ge_prepare", "ge_features", "ge_generate", "ge_generate_fallbacks", "ge_pool_refill", "ge_reset", "ge_step", "ge_step_sampled", "ge_sample_actions", "ge_obs_len",
           "ge_obs_flat", "ge_obs_graph", "ge_obs_nodes", "ge_step_kernel_name", "ge_batch_slice", "ge_step_host", "ge_step_host_pipelined", "ge_step_host_compact", "ge_progress_supported",
           "ge_step_host_release", "ge_mask_bytes_current", "ge_mask_bytes", "ge_stats",
           "ge_sample_logits", "ge_masked_log_prob", "ge_masked_log_prob_backward", "ge_beam_expand", "ge_beam_expand_sampled",
           "ge_mcts_select", "ge_mcts_expand", "ge_gumbel_root", "ge_gumbel_select", "ge_gumbel_result",
           "ge_state_record_bytes", "ge_state_save", "ge_state_load", "ge_gather_instances"]

LOGITS_F32, LOGITS_BF16 = 0, 1   # GE_LOGITS_*
STATE_DYNAMIC, STATE_CLOCK, STATE_STATS, STATE_ALL = 1, 2, 4, 7   # GE_STATE_*

_lib = None


class NativeError(RuntimeError):
    pass


def lib():
    """Loads the CUDA library; raises (never falls back) when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError(
            "graphenvs_b200: %s is missing. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    L.ge_last_error.restype = C.c_char_p
    BP = C.POINTER(GeBatch)
    L.ge_fill_layout.argtypes = [BP]
    L.ge_step_smem_bytes.argtypes = [BP]
    L.ge_build_adjacency.argtypes = [BP, _P]
    L.ge_prepare.argtypes = [BP, C.c_int, _P, _P]
    L.ge_features.argtypes = [BP, _P]
    L.ge_generate.argtypes = [BP, C.c_uint64, _P, _P, _P, _P, _P]
    L.ge_generate_fallbacks.argtypes = [_P]
    L.ge_pool_refill.argtypes = [BP, BP, C.c_int, _P, C.c_int, _P, _P, _P]
    L.ge_reset.argtypes = [BP, _P, _P]
    L.ge_step.argtypes = [BP, _P, C.POINTER(StepOut), _P]
    L.ge_sample_actions.argtypes = [BP, C.c_uint64, C.c_uint32, _P, _P]
    L.ge_step_sampled.argtypes = [BP, C.c_uint64, C.c_uint32, _P, C.POINTER(StepOut), _P]
    L.ge_obs_len.argtypes = [BP]
    L.ge_obs_flat.argtypes = [BP, C.c_int, C.c_int, _P, _P]
    L.ge_obs_graph.argtypes = [BP, C.c_int, C.c_int, _P, _P, _P, _P]
    L.ge_step_host.argtypes = [BP, _P, _P, C.POINTER(StepOut), _P, _P, _P, _P, _P, _P]
    L.ge_step_host_pipelined.argtypes = [BP, _P, C.POINTER(StepOut), _P, _P, _P, _P, C.c_int, _P]
    L.ge_step_host_compact.argtypes = [BP, _P, C.POINTER(StepOut), _P, _P, _P, _P, C.c_int, _P]
    L.ge_step_host_release.argtypes = [BP]
    L.ge_obs_nodes.argtypes = [BP, C.c_int, C.c_int, _P, _P]
    L.ge_step_kernel_name.argtypes = [BP, C.c_int]
    L.ge_step_kernel_name.restype = C.c_char_p
    L.ge_batch_slice.argtypes = [BP, C.c_int, C.c_int, BP]
    L.ge_stats.argtypes = [BP, _P, _P]
    L.ge_mask_bytes_current.argtypes = [BP]
    L.ge_mask_bytes.argtypes = [BP, C.c_int, C.c_int, _P]
    L.ge_sample_logits.argtypes = [BP, _P, C.c_int, C.c_int, C.c_uint64, C.c_uint32, _P, _P, _P, _P]
    L.ge_masked_log_prob.argtypes = [_P, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P]
    L.ge_masked_log_prob_backward.argtypes = [_P, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P, _P, _P]
    L.ge_beam_expand.argtypes = [BP, C.c_int, _P, C.c_int, _P, _P, _P, _P, _P, _P]
    L.ge_beam_expand_sampled.argtypes = [BP, C.c_int, _P, C.c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]
    TP = C.POINTER(MctsTree)
    L.ge_mcts_select.argtypes = [TP, C.c_int, _P]
    L.ge_mcts_expand.argtypes = [TP, C.c_int, BP, _P, _P, C.c_int, _P, _P]
    GP = C.POINTER(GumbelParams)
    L.ge_gumbel_root.argtypes = [TP, GP, C.c_uint64, C.c_uint32, C.c_int32, _P]
    L.ge_gumbel_select.argtypes = [TP, GP, C.c_int, _P]
    L.ge_gumbel_result.argtypes = [TP, GP, _P, _P, _P, _P]
    L.ge_state_record_bytes.argtypes = [BP]
    L.ge_state_save.argtypes = [BP, _P, C.c_int, _P, _P]
    L.ge_state_load.argtypes = [BP, _P, C.c_int, _P, C.c_uint, _P]
    L.ge_gather_instances.argtypes = [BP, BP, _P, _P]
    if L.ge_abi_version() != 4:
        raise NativeError("ABI version mismatch")
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise NativeError("graphenvs_b200 native call failed (%d): %s" % (rc, lib().ge_last_error().decode()))
