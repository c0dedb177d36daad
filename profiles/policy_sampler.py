"""Masked categorical over policy logits (csrc/ge_policy.cu) against the torch path a user writes without it.

For every workload (bench.WORKLOADS shapes, real masks of generated, reset envs after a few sampled steps) and for float32
and bfloat16 logits, times in us per call, the fused and the torch variant alternating in the same run:
  (a) sample        BatchedGraphEnv.sample_logits
      torch_sample  venv.mask (with the ge_mask_bytes expansion where the kind needs it), masked_fill, log_softmax,
                    Gumbel-max draw, gather, entropy
  (c) fwdbwd        policy.masked_log_prob forward + backward (dense grad_logits)
      torch_fwdbwd  the same values and gradient through torch autograd (bool masks from a rollout buffer, not timed)
  (d) sample_step   sample_logits + step_async, one policy-driven step
      step_sampled  the uniform random step (one launch), the cost of a policy-driven step over a random one
Every timed window starts from the same env state (the masks counted below).  Inputs are kept cold: the logits rotate over enough tensors to exceed 3 x the 126 MB L2.  Bytes are counted from shapes
and masks: `dense` = logits + mask words + outputs; `sector` = the 32-byte logits sectors (aligned groups of 8 fp32 /
16 bf16 actions of a row) holding at least one valid action + mask words + outputs, the least a kernel that reads only
valid logits must move.  Writes one JSON line per (workload, dtype).

    python profiles/policy_sampler.py --out profiles/r03_policy_sampler.jsonl [--workloads cfg2_longest_path,...]
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

DEFAULT = "cfg2_longest_path,cfg3_mst,cfg4_tsp_p1,cfg5_multicast,cfg5_distcenter"
L2 = 126 << 20


def gpu_identity():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:  # the device name from torch is still recorded
        return "nvidia-smi unavailable (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--workloads", default=DEFAULT)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warm-steps", type=int, default=4)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("policy_sampler.py measures on a CUDA device; none found")
    import bench
    from graphenvs_b200 import BatchedGraphEnv, masked_log_prob

    ident = gpu_identity()
    dev_name = torch.cuda.get_device_name(0)
    out = open(args.out, "w")

    def timed(fn, n, env=None, sd=None):
        if sd is not None:
            env.load_state_dict(sd)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(n):
            fn(i)
        e.record()
        e.synchronize()
        return s.elapsed_time(e) * 1e3 / n

    for wl in args.workloads.split(","):
        env_id, N, E, kw, B, _, _ = bench.WORKLOADS[wl]
        kw = dict(kw)
        env = BatchedGraphEnv(env_id, B, N, E, auto_reset=True, **kw)
        env.generate(seed=bench.SEED)
        env.reset()
        for t in range(args.warm_steps):
            env.step_sampled(1, t)
        torch.cuda.synchronize()
        A, AW = env.desc.A, env.desc.AW
        mb = env.t["mask_bits"]
        bits = mb.view(torch.uint8)                                    # one byte = 8 actions, two = 16
        valid = sum(int(((bits >> k) & 1).sum()) for k in range(8))
        sect = {torch.float32: int((bits != 0).sum()), torch.bfloat16: int((mb.view(torch.int16) != 0).sum())}
        bool_mask = env.mask.clone()                                   # rollout-buffer masks for (c)'s torch path
        sd0 = env.state_dict()                                         # every timed window starts from these masks
        for dtype in (torch.float32, torch.bfloat16):
            esz = 2 if dtype == torch.bfloat16 else 4
            logit_bytes = B * A * esz
            nrot = max(1, min(64, math.ceil(3 * L2 / logit_bytes)))
            gen = torch.Generator(device="cuda").manual_seed(7)
            L = [(torch.randn((B, A), generator=gen, device="cuda") * 2).to(dtype) for _ in range(nrot)]
            n = max(10, min(200, int(4e9 / (B * A * 4))))
            aux = B * AW * 4 + B * 12
            dense = logit_bytes + aux
            sector = sect[dtype] * 32 + aux
            res = {k: [] for k in ("sample", "torch_sample", "fwdbwd", "torch_fwdbwd", "sample_step", "step_sampled")}

            def f_sample(i):
                env.sample_logits(L[i % nrot], 3, i)

            def f_torch_sample(i):
                x = L[i % nrot]
                m = env.mask
                lp_all = torch.log_softmax(x.masked_fill(~m, float("-inf")), -1, dtype=torch.float32)
                g = -torch.log(-torch.log(torch.rand(lp_all.shape, device="cuda")))
                a = (lp_all + g).argmax(-1, keepdim=True)
                lp = lp_all.gather(-1, a)
                ent = -torch.where(m, lp_all.exp() * lp_all, torch.zeros((), device="cuda")).sum(-1)
                return a, lp, ent

            acts = env.sample_logits(L[0], 3, 0)[0].clone()
            mb0 = mb.clone()                                           # the masks the actions were drawn under
            g1 = torch.randn(B, device="cuda")
            g2 = torch.randn(B, device="cuda") * 0.01

            def f_fwdbwd(i):
                x = L[i % nrot].requires_grad_(True)
                lp, H = masked_log_prob(x, mb0, acts)
                torch.autograd.grad((lp, H), x, (g1, g2))
                x.requires_grad_(False)

            def f_torch_fwdbwd(i):
                x = L[i % nrot].requires_grad_(True)
                lp_all = torch.log_softmax(x.masked_fill(~bool_mask, float("-inf")), -1, dtype=torch.float32)
                lp = lp_all.gather(-1, acts.long()[:, None])[:, 0]
                ent = -torch.where(bool_mask, lp_all.exp() * lp_all, torch.zeros((), device="cuda")).sum(-1)
                torch.autograd.grad((lp, ent), x, (g1, g2))
                x.requires_grad_(False)

            def f_sample_step(i):
                a = env.sample_logits(L[i % nrot], 5, i)[0]
                env.step_async(a)

            def f_step_sampled(i):
                env.step_sampled(5, i)

            pairs = [("sample", f_sample, "torch_sample", f_torch_sample), ("fwdbwd", f_fwdbwd, "torch_fwdbwd", f_torch_fwdbwd),
                     ("sample_step", f_sample_step, "step_sampled", f_step_sampled)]
            for _, fa, _, fb in pairs:   # warm-up of every shape the timed windows use
                timed(fa, 2)
                timed(fb, 2)
            for r in range(args.reps):
                for ka, fa, kb, fb in pairs:
                    res[ka].append(timed(fa, n, env, sd0))
                    res[kb].append(timed(fb, n, env, sd0))
            med = {k: sorted(v)[len(v) // 2] for k, v in res.items()}
            line = {
                "workload": wl, "env_id": env_id, "dtype": "bf16" if esz == 2 else "f32", "B": B, "A": A, "AW": AW,
                "valid_actions_per_env": valid / B, "valid_frac": valid / (B * A),
                "bytes_dense": dense, "bytes_sector_bound": sector, "logits_rotation": nrot, "calls_per_window": n, "reps": args.reps,
                "us": {k: round(v, 2) for k, v in med.items()},
                "us_all": {k: [round(x, 2) for x in v] for k, v in res.items()},
                "speedup_sample_vs_torch": round(med["torch_sample"] / med["sample"], 2),
                "speedup_fwdbwd_vs_torch": round(med["torch_fwdbwd"] / med["fwdbwd"], 2),
                "policy_step_over_uniform_step": round(med["sample_step"] / med["step_sampled"], 2),
                "sample_GBps_of_sector_bound": round(sector / (med["sample"] * 1e3), 1),
                "sample_GBps_dense_equiv": round(dense / (med["sample"] * 1e3), 1),
                "fwdbwd_bytes": 2 * sector + logit_bytes,
                "fwdbwd_GBps": round((2 * sector + logit_bytes) / (med["fwdbwd"] * 1e3), 1),
                "gpu": dev_name, "nvidia_smi": ident, "time": time.strftime("%Y-%m-%dT%H:%M:%S"),
            }
            print(json.dumps(line), flush=True)
            out.write(json.dumps(line) + "\n")
            out.flush()
            del L
            torch.cuda.empty_cache()
        del env, bool_mask, sd0
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
