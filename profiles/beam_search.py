"""Beam search (ge_beam_expand, graphenvs_b200.BeamSearch) against the torch path a user writes without it.

For every workload (bench.WORKLOADS shapes; G = the bench's env count / 16 instances x W = 16 beams, so the wide batch has as
many envs as the bench's) and for float32 and bfloat16 logits, real masks of a beam decode a few steps in, times in us per call,
the variants alternating in the same run and every timed window starting from the same state:
  (a) expand        ge_beam_expand over the wide batch
      torch_expand  masked_fill, log_softmax, + beam score, a stay column for finished beams, view [G, W * (A + 1)], topk(W),
                    // and % (A + 1): the same selection, checked here (scores by rank to 1e-5; log_softmax rounds differently
                    from fl32(l - lse), so candidates an ulp apart may swap ranks: their count is reported)
  (b) fork          save_states + load_states with the expand's load_index (every env saved, the moved ones loaded)
      decode_step   BeamSearch.advance: expand + fork + step_async, one whole decode step
      sample_step   sample_logits + step_async over the same wide batch, a policy-driven step without search
                    (these two: one call per event pair, each from the saved state, so no call meets a batch of finished beams)
  (c) bytes         `dense` = logits + mask words + done + scores + outputs; `sector` = the 32-byte logits sectors holding a valid
                    action + the same small arrays, the least a kernel that reads only valid logits must move.
Logits rotate over enough tensors to exceed 3 x the 126 MB L2.  Writes one JSON line per (workload, dtype).

    python profiles/beam_search.py --out profiles/r05_beam_search.jsonl [--workloads cfg2_longest_path,...]
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

DEFAULT = "cfg2_longest_path,cfg3_mst,cfg5_multicast,cfg5_distcenter"
L2 = 126 << 20
W = 16


def gpu_identity():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:  # the device name from torch is still recorded
        return "nvidia-smi unavailable (%s)" % e


def torch_expand(x, mask, done, score, G, W):
    """The torch path: every logit read, a topk over G x W x (A + 1) candidates."""
    B, A = x.shape
    lp = torch.log_softmax(x.float().masked_fill(~mask, float("-inf")), -1)
    cand = score[:, None] + lp
    cand = torch.where(done[:, None], torch.full_like(cand, float("-inf")), cand)
    stay = torch.where(done, score, torch.full_like(score, float("-inf")))
    cand = torch.cat([stay[:, None], cand], 1).view(G, W * (A + 1))
    val, idx = cand.topk(W, dim=1)
    base = torch.arange(G, device=x.device)[:, None] * W
    parent = torch.where(val > float("-inf"), idx // (A + 1) + base, torch.full_like(idx, -1))
    action = torch.where(val > float("-inf"), idx % (A + 1) - 1, torch.full_like(idx, -1))
    return val.flatten(), parent.flatten(), action.flatten()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--workloads", default=DEFAULT)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warm-steps", type=int, default=3)
    args = ap.parse_args()

    global torch
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("beam_search.py measures on a CUDA device; none found")
    import bench
    import graphenvs_b200 as ge
    from graphenvs_b200 import BatchedGraphEnv

    ident = gpu_identity()
    dev_name = torch.cuda.get_device_name(0)
    out = open(args.out, "w")

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
        bs = ge.BeamSearch(venv, width=W)
        wide = bs.wide
        B, A, AW = wide.B, wide.desc.A, wide.desc.AW
        gen = torch.Generator(device="cuda").manual_seed(3)
        bs.start()
        for _ in range(args.warm_steps):
            bs.advance(torch.randn((B, A), generator=gen, device="cuda"))
        torch.cuda.synchronize()
        mb = wide.t["mask_bits"]
        bits = mb.view(torch.uint8)
        valid = sum(int(((bits >> k) & 1).sum()) for k in range(8))
        sect = {torch.float32: int((bits != 0).sum()), torch.bfloat16: int((mb.view(torch.int16) != 0).sum())}
        mask = wide.mask.clone()
        done = wide.t["done"] != 0
        sd0, score0, t0 = wide.state_dict(), bs.score.clone(), bs.t
        n_done, n_dead = int(done.sum()), int((score0 == float("-inf")).sum())

        def restore():
            wide.load_state_dict(sd0)
            bs.score.copy_(score0)
            bs.t = t0

        for dtype in (torch.float32, torch.bfloat16):
            esz = 2 if dtype == torch.bfloat16 else 4
            logit_bytes = B * A * esz
            nrot = max(1, min(64, math.ceil(3 * L2 / logit_bytes)))
            Ls = [torch.randn((B, A), generator=gen, device="cuda").to(dtype) for _ in range(nrot)]
            n = max(10, min(200, int(4e9 / (B * A * 4))))
            n_step = min(n, 20)
            bs.reserve(t0 + n + 4)
            small = B * AW * 4 + B * 1 + B * 4 + B * 16
            dense, sector = logit_bytes + small, sect[dtype] * 32 + small
            s_in = score0.clone()
            s_out, par, act, load = (torch.empty(B, device="cuda"),) + tuple(torch.empty(B, dtype=torch.int32, device="cuda") for _ in range(3))
            from graphenvs_b200.beam import _ptr
            from graphenvs_b200.policy import _DTYPES
            import ctypes as C

            def f_expand(i):
                x = Ls[i % nrot]
                ge._native.check(wide.lib.ge_beam_expand(C.byref(wide.desc), W, _ptr(x), _DTYPES[dtype], _ptr(s_in), _ptr(s_out),
                                                         _ptr(par), _ptr(act), _ptr(load), wide._stream()))

            def f_torch(i):
                return torch_expand(Ls[i % nrot], mask, done, s_in, G, W)

            # correctness of the comparison: the same selection
            f_expand(0)
            tv, tp, ta = f_torch(0)
            torch.cuda.synchronize()
            # log_softmax rounds differently from fl32(l - lse): candidates within an ulp or two may swap ranks, nothing else
            swapped = (par != tp.int()) | (act != ta.int())
            assert torch.allclose(s_out, tv, rtol=1e-5, atol=1e-5), "torch path and ge_beam_expand disagree"
            n_swapped = int(swapped.sum())
            load_fixed = load.clone()

            def f_fork(i):
                wide.save_states(out=bs.records)
                wide.load_states(bs.records, load_fixed)

            def f_decode(i):
                bs.advance(Ls[i % nrot])

            def f_sample_step(i):
                a = wide.sample_logits(Ls[i % nrot], 5, i)[0]
                wide.step_async(a)

            fns = [("expand", f_expand), ("torch_expand", f_torch), ("fork", f_fork), ("decode_step", f_decode), ("sample_step", f_sample_step)]
            for _, f in fns:   # warm-up of every shape the timed windows use
                timed(f, 2, restore)
            res = {k: [] for k, _ in fns}
            for r in range(args.reps):
                for k, f in fns:
                    if k in ("decode_step", "sample_step"):   # one step from the saved state per event pair: no window of finished beams
                        res[k].append(sum(timed(lambda _: f(i), 1, restore) for i in range(n_step)) / n_step)
                    else:
                        res[k].append(timed(f, n, restore))
            restore()
            med = {k: sorted(v)[len(v) // 2] for k, v in res.items()}
            line = {
                "workload": wl, "env_id": env_id, "dtype": "bf16" if esz == 2 else "f32", "G": G, "W": W, "B": B, "A": A, "AW": AW,
                "decode_steps_before": t0, "torch_near_tie_rank_swaps": n_swapped, "done_beams": n_done, "dead_beams": n_dead,
                "valid_actions_per_env": valid / B, "valid_frac": valid / (B * A),
                "record_bytes": wide.record_bytes(),
                "bytes_dense": dense, "bytes_sector_bound": sector, "logits_rotation": nrot, "calls_per_window": n, "step_calls_each_from_saved_state": n_step, "reps": args.reps,
                "us": {k: round(v, 2) for k, v in med.items()},
                "us_all": {k: [round(x, 2) for x in v] for k, v in res.items()},
                "speedup_expand_vs_torch": round(med["torch_expand"] / med["expand"], 2),
                "step_in_decode_us": round(med["decode_step"] - med["expand"] - med["fork"], 2),
                "decode_step_over_sample_step": round(med["decode_step"] / med["sample_step"], 2),
                "expand_GBps_of_sector_bound": round(sector / (med["expand"] * 1e3), 1),
                "expand_GBps_dense_equiv": round(dense / (med["expand"] * 1e3), 1),
                "gpu": dev_name, "nvidia_smi": ident, "time": time.strftime("%Y-%m-%dT%H:%M:%S"),
            }
            print(json.dumps(line), flush=True)
            out.write(json.dumps(line) + "\n")
            out.flush()
            del Ls
            torch.cuda.empty_cache()
        del bs, wide, venv, sd0, mask
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
