"""Stochastic beam search (ge_beam_expand_sampled, graphenvs_b200.StochasticBeamSearch) against the deterministic expand and
the i.i.d. alternative, on the shapes of profiles/beam_search.py.

For every workload (bench.WORKLOADS shapes; G = the bench's env count / 16 instances x W = 16 beams) and for float32 and
bfloat16 logits, real masks of a sampled decode a few steps in, times in us per call, the variants alternating in the same run
and every timed window starting from the same state:
  sampled_expand  ge_beam_expand_sampled over the wide batch (with the group thresholds)
  expand          ge_beam_expand on the same masks and logits (scores = the sampled decode's log-probs)
  decode_step     StochasticBeamSearch.advance: sampled expand + fork + step_async, one whole decode step
  iid_step        sample_logits + step_async over the same wide batch: the i.i.d. rollouts a user draws without it
                  (these two: one call per event pair, each from the saved state, so no call meets a batch of finished beams)
Logits rotate over enough tensors to exceed 3 x the 126 MB L2.  One JSON line per (workload, dtype), then, at cfg2, one line
counting the duplicate rate of K = 16 i.i.d. rollouts per instance (a fixed state-dependent table policy, every rollout to its
end) against the stochastic beam of the same width (distinct by construction, counted all the same).

    python profiles/stochastic_beam.py --out profiles/r06_stochastic_beam.jsonl [--workloads cfg2_longest_path,...]
"""
import argparse
import ctypes as C
import json
import math
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from beam_search import gpu_identity  # noqa: E402

DEFAULT = "cfg2_longest_path,cfg3_mst,cfg5_multicast,cfg5_distcenter"
L2 = 126 << 20
W = 16


def distinct_per_group(seqs, G, K):
    """seqs int32 [G * K, T] (-1 padded): the number of distinct sequences in each group of K rows."""
    import torch
    s = seqs.view(G, K, -1)
    eq = (s[:, :, None, :] == s[:, None, :, :]).all(-1)                # [G, K, K] row j equals row i
    first = ~torch.tril(eq, diagonal=-1).any(-1)                       # no earlier row equals it
    return first.sum(-1)


def duplicates(wl, K, seed_env, seed_pol):
    """Duplicate rate of K i.i.d. rollouts per instance, and of the width-K stochastic beam, under one table policy."""
    import torch
    import bench
    import graphenvs_b200 as ge
    from graphenvs_b200 import BatchedGraphEnv
    env_id, N, E, kw, Bb, _, _ = bench.WORKLOADS[wl]
    G = Bb // K
    venv = BatchedGraphEnv(env_id, G, N, E, **dict(kw))
    venv.generate(seed=seed_env)
    A = venv.desc.A
    gen = torch.Generator(device="cuda").manual_seed(seed_pol)
    tab = torch.randn((G, N, A), generator=gen, device="cuda")

    def policy(env):
        return tab[torch.arange(env.B, device="cuda") // K, env.t["head"].long().clamp(0, N - 1)]

    wide = venv.like(G * K, auto_reset=False)
    wide.gather_instances(venv, torch.arange(G, dtype=torch.int32, device="cuda").repeat_interleave(K))
    wide.reset()
    acts = []
    for t in range(4 * N):
        if bool((wide.t["done"] != 0).all()):
            break
        a = wide.sample_logits(policy(wide), 2024, t)[0]
        a = torch.where(wide.t["done"] != 0, torch.full_like(a, -1), a)
        acts.append(a.clone())
        wide.step_async(a)
    iid = torch.stack(acts, 1)
    finished = bool((wide.t["done"] != 0).all())
    d_iid = distinct_per_group(iid, G, K).double()
    res = ge.StochasticBeamSearch(venv, width=K, seed=2024).run(policy)
    sbs = res.beams.actions.reshape(G * K, -1)
    d_sbs = distinct_per_group(sbs, G, K).double()
    return {
        "workload": wl, "env_id": env_id, "what": "duplicates", "G": G, "K": K, "A": A, "policy": "randn table [G, N, A] by head",
        "iid_all_finished": finished, "iid_steps": len(acts),
        "iid_duplicate_rate": round(1 - float(d_iid.mean()) / K, 4), "iid_mean_distinct": round(float(d_iid.mean()), 3),
        "iid_groups_with_a_duplicate": round(float((d_iid < K).double().mean()), 4),
        "sbs_duplicate_rate": round(1 - float(d_sbs.mean()) / K, 4), "sbs_steps": res.steps,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--workloads", default=DEFAULT)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warm-steps", type=int, default=3)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("stochastic_beam.py measures on a CUDA device; none found")
    import bench
    import graphenvs_b200 as ge
    from graphenvs_b200 import BatchedGraphEnv
    from graphenvs_b200.beam import _ptr
    from graphenvs_b200.policy import _DTYPES

    ident = gpu_identity()
    dev_name = torch.cuda.get_device_name(0)
    out = open(args.out, "w")

    def emit(line):
        line.update({"gpu": dev_name, "nvidia_smi": ident, "time": time.strftime("%Y-%m-%dT%H:%M:%S")})
        print(json.dumps(line), flush=True)
        out.write(json.dumps(line) + "\n")
        out.flush()

    def timed(fn, n, restore=None):
        if restore is not None:
            restore()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(n):
            fn(i)
        e.record()
        e.synchronize()
        return s.elapsed_time(e) * 1e3 / n

    for wl in args.workloads.split(","):
        env_id, N, E, kw, Bb, _, _ = bench.WORKLOADS[wl]
        G = Bb // W
        venv = BatchedGraphEnv(env_id, G, N, E, **dict(kw))
        venv.generate(seed=bench.SEED)
        sbs = ge.StochasticBeamSearch(venv, width=W, seed=7)
        wide = sbs.wide
        B, A, AW = wide.B, wide.desc.A, wide.desc.AW
        gen = torch.Generator(device="cuda").manual_seed(3)
        sbs.start()
        for _ in range(args.warm_steps):
            sbs.advance(torch.randn((B, A), generator=gen, device="cuda"))
        torch.cuda.synchronize()
        bits = wide.t["mask_bits"].view(torch.uint8)
        valid = sum(int(((bits >> k) & 1).sum()) for k in range(8))
        sd0, t0 = wide.state_dict(), sbs.t
        saved = [x.clone() for x in (sbs.score, sbs.key, sbs.node_key)]
        n_done, n_dead = int((wide.t["done"] != 0).sum()), int((saved[1] == float("-inf")).sum())

        def restore():
            wide.load_state_dict(sd0)
            for x, y in zip((sbs.score, sbs.key, sbs.node_key), saved):
                x.copy_(y)
            sbs.t = t0

        for dtype in (torch.float32, torch.bfloat16):
            esz = 2 if dtype == torch.bfloat16 else 4
            nrot = max(1, min(64, math.ceil(3 * L2 / (B * A * esz))))
            Ls = [torch.randn((B, A), generator=gen, device="cuda").to(dtype) for _ in range(nrot)]
            n = max(10, min(200, int(4e9 / (B * A * 4))))
            n_step = min(n, 20)
            sbs.reserve(t0 + n + 4)
            lp_in, key_in, nk_in = (x.clone() for x in saved)
            lp_out, key_out, thr = torch.empty(B, device="cuda"), torch.empty(B, device="cuda"), torch.empty(G, device="cuda")
            nk_out = torch.empty(B, dtype=torch.int64, device="cuda")
            par, act, load = (torch.empty(B, dtype=torch.int32, device="cuda") for _ in range(3))

            def f_sampled(i):
                x = Ls[i % nrot]
                ge._native.check(wide.lib.ge_beam_expand_sampled(
                    C.byref(wide.desc), W, _ptr(x), _DTYPES[dtype], _ptr(lp_in), _ptr(key_in), _ptr(nk_in), _ptr(lp_out),
                    _ptr(key_out), _ptr(nk_out), _ptr(par), _ptr(act), _ptr(load), _ptr(thr), wide._stream()))

            def f_expand(i):
                x = Ls[i % nrot]
                ge._native.check(wide.lib.ge_beam_expand(C.byref(wide.desc), W, _ptr(x), _DTYPES[dtype], _ptr(lp_in), _ptr(lp_out),
                                                         _ptr(par), _ptr(act), _ptr(load), wide._stream()))

            def f_decode(i):
                sbs.advance(Ls[i % nrot])

            def f_iid(i):
                a = wide.sample_logits(Ls[i % nrot], 5, i)[0]
                wide.step_async(a)

            fns = [("sampled_expand", f_sampled), ("expand", f_expand), ("decode_step", f_decode), ("iid_step", f_iid)]
            for _, f in fns:   # warm-up of every shape the timed windows use
                timed(f, 2, restore)
            res = {k: [] for k, _ in fns}
            for r in range(args.reps):
                for k, f in fns:
                    if k in ("decode_step", "iid_step"):
                        res[k].append(sum(timed(lambda _: f(i), 1, restore) for i in range(n_step)) / n_step)
                    else:
                        res[k].append(timed(f, n, restore))
            restore()
            med = {k: sorted(v)[len(v) // 2] for k, v in res.items()}
            emit({
                "workload": wl, "env_id": env_id, "dtype": "bf16" if esz == 2 else "f32", "G": G, "W": W, "B": B, "A": A, "AW": AW,
                "decode_steps_before": t0, "done_beams": n_done, "dead_beams": n_dead, "valid_actions_per_env": valid / B,
                "logits_rotation": nrot, "calls_per_window": n, "step_calls_each_from_saved_state": n_step, "reps": args.reps,
                "us": {k: round(v, 2) for k, v in med.items()},
                "us_all": {k: [round(x, 2) for x in v] for k, v in res.items()},
                "sampled_over_deterministic_expand": round(med["sampled_expand"] / med["expand"], 2),
                "sampled_expand_share_of_decode_step": round(med["sampled_expand"] / med["decode_step"], 2),
                "decode_step_over_iid_step": round(med["decode_step"] / med["iid_step"], 2),
            })
            del Ls
            torch.cuda.empty_cache()
        del sbs, wide, venv, sd0
        torch.cuda.empty_cache()
    if "cfg2_longest_path" in args.workloads.split(","):
        emit(duplicates("cfg2_longest_path", W, bench.SEED, 11))


if __name__ == "__main__":
    main()
