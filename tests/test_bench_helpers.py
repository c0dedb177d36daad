"""CPU: the parts of bench.py that do not need a GPU -- workload table, compulsory-bytes model, clock-sample
parsing, the host policy, and the reference arm's JSON contract (run for real on a tiny budget)."""
import ctypes as C
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from graphenvs_b200 import _native  # noqa: E402
from graphenvs_b200.spec import ENV_SPECS  # noqa: E402


def _fake_env(wl):
    env_id, N, E, kw, B, survey, desc = bench.WORKLOADS[wl]
    d = _native.GeBatch()
    d.kind, d.B, d.N, d.M = ENV_SPECS[env_id].kind, 4, N, 2 * E
    d.parenting = kw.get("parenting", -1)
    d.n_targets = kw.get("target_count", 0)
    d.n_dests = kw.get("n_dests", kw.get("n_products", 0))
    _native.lib().ge_fill_layout(C.byref(d))
    return types.SimpleNamespace(desc=d, N=N, M=2 * E, env_id=env_id, t={"mask_bytes": 1})


def test_workloads_cover_every_baseline_config_and_env():
    ids = {w[0] for w in bench.WORKLOADS.values()}
    assert ids == set(ENV_SPECS), "every env of north_star has a bench workload"
    assert bench.DEFAULT_WORKLOAD == "cfg2_longest_path"
    env_id, N, E, kw, B, _, _ = bench.WORKLOADS[bench.DEFAULT_WORKLOAD]
    assert (env_id, N, E, kw["parenting"], B) == ("LongestPath-v0", 50, 200, 2, 65536)   # BASELINE.json configs[1]


def test_compulsory_bytes_model_is_positive_and_below_the_survey_figure_for_incremental_kernels():
    for wl, spec in bench.WORKLOADS.items():
        b = bench.layout_bytes_per_step(_fake_env(wl))
        assert b > 50, wl
        if wl in ("cfg3_mst", "cfg5_multicast", "cfg4_tsp_p2", "cfg2_longest_path"):
            assert b < spec[5], (wl, b, spec[5])


def test_clock_sampler_parses_nvidia_smi_rows():
    s = bench.ClockSampler(0)
    s.proc = types.SimpleNamespace(terminate=lambda: None)
    rows = ["0, 1965, 1965, 380.5, 0x0000000000000000, Not Active, Not Active, Not Active, Not Active",
            "0, 1950, 1965, 401.0, 0x0000000000000004, Not Active, Not Active, Not Active, Active",
            "garbage"]
    s.rows = [(100.0 + i, r) for i, r in enumerate(rows)]
    out = s.stop(99.0, 110.0)
    assert out["sm_mhz"] == 1957.5 and out["sm_max_mhz"] == 1965.0 and out["reasons"] == ["sw_power_cap"] and out["samples"] == 2


def test_host_policy_picks_valid_actions():
    rng = np.random.default_rng(0)
    mask = rng.random((500, 37)) < 0.2
    mask[:, 5] = True
    a = bench.host_policy(rng, mask)
    assert a.dtype == np.int32 and mask[np.arange(500), a].all()
    assert len(np.unique(a)) > 5


def _fake_stepped_env(B, A, seed=0):
    rng = np.random.default_rng(seed)
    mask = rng.random((B, A)) < 0.3
    AW = (A + 31) // 32
    bits = np.packbits(np.pad(mask, ((0, 0), (0, 32 * AW - A))), axis=1, bitorder="little").view(np.int32)
    flags = np.stack([rng.integers(0, 2, B), rng.integers(-1, 2, B) & 0xFF, rng.integers(0, 2, B), rng.integers(0, 2, B)], 1)
    env = types.SimpleNamespace(B=B, desc=types.SimpleNamespace(A=A), t={"mask_bits": torch.from_numpy(bits)},
                                flags=torch.from_numpy(flags.astype(np.uint8)), reward=torch.from_numpy(rng.random(B, dtype=np.float32)),
                                solution_cost=torch.from_numpy(rng.random(B)), actions_dev=torch.from_numpy(rng.integers(0, A, B, dtype=np.int32)))
    return env, mask, flags


def test_step_outputs_are_float_arrays_of_what_the_caller_receives():
    env, mask, flags = _fake_stepped_env(100, 40)
    out = bench.step_outputs(env)
    assert all(a.dtype in (np.float32, np.float64) and a.shape[0] == 100 for a in out.values())
    np.testing.assert_array_equal(out["mask"], mask)
    np.testing.assert_array_equal(out["solved"], flags[:, 1].astype(np.uint8).view(np.int8))
    np.testing.assert_array_equal(out["action"], env.actions_dev.numpy())
    np.testing.assert_array_equal(out["solution_cost"], env.solution_cost.numpy())
    np.testing.assert_array_equal(out["env_index"], np.arange(100))


def test_step_outputs_of_a_large_batch_are_a_fixed_sample_within_the_budget():
    env, mask, _ = _fake_stepped_env(5000, 300)
    full = bench.step_outputs(env)
    budget = 200_000
    out = bench.step_outputs(env, budget=budget)
    assert 0 < sum(a.nbytes for a in out.values()) <= budget
    idx = out["env_index"].astype(np.int64)
    assert len(idx) < 5000 and np.all(np.diff(idx) > 0)
    for name, a in out.items():
        np.testing.assert_array_equal(a, full[name][idx])
    again = bench.step_outputs(env, budget=budget)
    for name, a in out.items():
        np.testing.assert_array_equal(a, again[name])


@pytest.mark.gpu
def test_dump_outputs_are_identical_from_run_to_run(tmp_path):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--only-headline", "--steps", "7", "--warmup", "3", "--no-cpu",
           "--e2e-steps", "3", "--no-e2e-obs"]
    runs = []
    for name in ("a", "b"):
        out = subprocess.check_output(cmd + ["--dump-outputs", str(tmp_path / name)]).decode().strip().splitlines()[-1]
        assert json.loads(out)["steps"] == 7
        runs.append({f[:-len(".npy")]: np.load(tmp_path / name / f) for f in os.listdir(tmp_path / name)})
    a, b = runs
    assert sorted(a) == sorted(("env_index", "action", "reward", "done", "solved", "status", "has_mask", "solution_cost", "mask"))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64_000_000
    for f in a:
        assert a[f].dtype in (np.float32, np.float64)
        np.testing.assert_array_equal(a[f], b[f], err_msg=f)
    assert a["done"].any() and a["mask"].any()


def test_reference_arm_prints_the_contract_line():
    env = dict(os.environ, OMP_NUM_THREADS="1", RANK="0", WORLD_SIZE="1")
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "5", "--warmup", "3",
                                   "--workload", "cfg1_shortest_path"], env=env).decode().strip().splitlines()[-1]
    d = json.loads(out)
    assert d["impl"] == "reference" and d["metric"] == bench.METRIC and d["unit"] == bench.UNIT and d["higher_is_better"] is True
    assert d["steps"] == 5 and d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # ranks other than 0 stay silent
    env["RANK"] = "1"
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "3"], env=env)
    assert out.decode().strip() == ""
