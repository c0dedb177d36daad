"""GPU: the masked categorical over policy logits (csrc/ge_policy.cu) -- BatchedGraphEnv.sample_logits and
policy.masked_log_prob against a float64 reference over the valid entries, a numpy restatement of the sampler's noise,
the C oracle under policy-driven rollouts, and slice / CUDA-graph / PDL scheduling."""
import ctypes as C
import random

import numpy as np
import pytest
import torch

import cuda_util as cu
from graphenvs_b200 import BatchedGraphEnv, _native, masked_log_prob, policy
from graphenvs_b200.instances import generate_instance
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

DTYPES = [torch.float32, torch.bfloat16]
M64 = (1 << 64) - 1


# ------------------------------------------------------------------ helpers
def pack(mask):
    """bool [..., A] -> int32 [..., ceil(A/32)] packed words (bit i of word w = action 32 w + i)."""
    m = np.asarray(mask, dtype=bool)
    A = m.shape[-1]
    AW = (A + 31) // 32
    pad = np.zeros(m.shape[:-1] + (AW * 32,), dtype=bool)
    pad[..., :A] = m
    return np.packbits(pad, axis=-1, bitorder="little").view(np.uint32).view(np.int32).reshape(m.shape[:-1] + (AW,))


def unpack(words, A):
    return np.unpackbits(np.ascontiguousarray(words).view(np.uint8), bitorder="little")[:A].astype(bool)


def make_masks(R, A, rng, stray=True):
    """Row kinds in turn: dense, sparse (5 %), one bit, empty, half.  Stray bits >= A in the last word when requested."""
    m = np.zeros((R, A), dtype=bool)
    for r in range(R):
        k = r % 5
        if k == 0:
            m[r] = rng.random(A) < 0.9
        elif k == 1:
            m[r] = rng.random(A) < 0.05
        elif k == 2:
            m[r, rng.integers(A)] = True
        elif k == 4:
            m[r] = rng.random(A) < 0.5
    bits = pack(m)
    if stray and A % 32:
        bits[:, -1] |= np.int32(np.uint32(~((1 << (A % 32)) - 1) & 0xFFFFFFFF).view(np.int32))
    return m, bits


def random_valid_actions(m, rng):
    a = np.full(m.shape[0], -1, dtype=np.int32)
    for r in range(m.shape[0]):
        idx = np.flatnonzero(m[r])
        if idx.size:
            a[r] = rng.choice(idx)
    return a


def reference(x, valid, actions):
    """float64 masked log-softmax over the valid entries only (torch.where, no -inf fill): (log_prob, entropy, lse)."""
    neg = torch.tensor(-np.inf, dtype=x.dtype, device=x.device)
    any_ = valid.any(-1)
    m = torch.where(valid, x, neg).amax(-1).detach()
    m = torch.where(any_, m, torch.zeros_like(m))
    xs = torch.where(valid, x, m[..., None])                          # invalid entries never reach exp / the products
    e = torch.where(valid, torch.exp(xs - m[..., None]), torch.zeros_like(xs))
    se = e.sum(-1)
    se1 = torch.where(any_, se, torch.ones_like(se))
    lse = m + torch.log(se1)
    p = e / se1[..., None]
    H = torch.where(any_, lse - torch.where(valid, p * xs, torch.zeros_like(xs)).sum(-1), torch.zeros_like(lse))
    A = x.shape[-1]
    ac = actions.long().clamp(0, A - 1)
    ok = (actions >= 0) & (actions < A) & valid.gather(-1, ac[..., None])[..., 0]
    la = xs.gather(-1, ac[..., None])[..., 0]
    lp = torch.where(ok, la - lse, torch.full_like(lse, -np.inf))
    lp = torch.where(any_, lp, torch.zeros_like(lp))
    lse = torch.where(any_, lse, torch.full_like(lse, -np.inf))
    return lp, H, lse, ok


def close(got, ref, what):
    got = got.double()
    fin = torch.isfinite(ref)
    assert torch.equal(torch.isfinite(got), fin), what + ": infinities differ"
    assert torch.equal(got[~fin], ref[~fin]), what + ": infinities differ"
    err = (got[fin] - ref[fin]).abs()
    tol = 1e-5 + 1e-5 * ref[fin].abs()
    assert bool((err <= tol).all()), "%s: max err %.3g" % (what, float((err - tol).max()))


def sampler_env(B, A, **kw):
    """A batch used only as the holder of B packed masks of A actions (node-action kind with N = A)."""
    return BatchedGraphEnv("ShortestPath-v0", B, A, 2 * A, byte_mask=False, **kw)


def np_mix32(seed, env, t):
    """ge_common.cuh:mix32 in numpy uint64 arithmetic (wrapping); arguments broadcast."""
    with np.errstate(over="ignore"):
        seed, env, t = np.uint64(seed), np.asarray(env, dtype=np.uint64), np.asarray(t, dtype=np.uint64)
        z = seed + np.uint64(0x9E3779B97F4A7C15) * (env * np.uint64(0x100000001) + ((t << np.uint64(32)) | np.uint64(0x5bd1e995)))
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
        return z >> np.uint64(32)


def np_gumbel(seed, e, t, A):
    """The sampler's noise (include/graphenvs_b200.h, ge_sample_logits) for actions 0..A-1, in float64."""
    key = (int(np_mix32(seed, e, t)) << 32) | int(np_mix32(seed ^ 0xD1B54A32D192ED03, e, t))
    h = np_mix32(key, np.arange(A, dtype=np.uint64), 0x85EBCA6B)
    u = ((h >> np.uint64(8)).astype(np.float64) + 0.5) / 2.0 ** 24
    return -np.log(-np.log(u))


# ------------------------------------------------------------------ 1. forward values
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
@pytest.mark.parametrize("A", [1, 31, 32, 33, 50, 1000, 8000])
def test_forward_matches_float64_reference(A, dtype):
    rng = np.random.default_rng(A)
    R = 40
    m, bits = make_masks(R, A, rng)
    acts = random_valid_actions(m, rng)
    logits = (torch.from_numpy(rng.standard_normal((R, A)).astype(np.float32)) * 3).to(dtype).cuda()
    mb, at = torch.from_numpy(bits).cuda(), torch.from_numpy(acts).cuda()
    lp, H = masked_log_prob(logits, mb, at)
    rlp, rH, rlse, _ = reference(logits.double(), torch.from_numpy(m).cuda(), at)
    close(lp, rlp, "log_prob")
    close(H, rH, "entropy")
    # lse, through the C entry point
    lse, lp2, H2 = (torch.empty(R, device="cuda") for _ in range(3))
    _native.check(_native.lib().ge_masked_log_prob(C.c_void_p(logits.data_ptr()), policy._DTYPES[dtype], R, A, C.c_void_p(mb.data_ptr()),
                                                   C.c_void_p(at.data_ptr()), C.c_void_p(lp2.data_ptr()), C.c_void_p(H2.data_ptr()),
                                                   C.c_void_p(lse.data_ptr()), None))
    torch.cuda.synchronize()
    close(lse, rlse, "lse")
    assert torch.equal(lp2, lp) and torch.equal(H2, H)
    empty = ~m.any(-1)
    assert empty.any()
    assert bool((lp[torch.from_numpy(empty).cuda()] == 0).all()) and bool((H[torch.from_numpy(empty).cuda()] == 0).all())
    # stray bits >= A change nothing
    clean = torch.from_numpy(pack(m)).cuda()
    lp3, H3 = masked_log_prob(logits, clean, at)
    assert torch.equal(lp3, lp) and torch.equal(H3, H)
    # NaN / inf in invalid entries change nothing (they are never read)
    dirty = logits.clone()
    inv = torch.from_numpy(~m).cuda()
    fill = torch.tensor([np.nan, np.inf, -np.inf], dtype=dtype, device="cuda")[torch.arange(A, device="cuda") % 3]
    dirty = torch.where(inv, fill.expand(R, A), dirty)
    lp4, H4 = masked_log_prob(dirty, mb, at)
    assert torch.equal(lp4, lp) and torch.equal(H4, H)
    # leading dims [T, B, .]
    lp5, H5 = masked_log_prob(logits.view(4, R // 4, A), mb.view(4, R // 4, -1), at.view(4, R // 4))
    assert torch.equal(lp5.reshape(-1), lp) and torch.equal(H5.reshape(-1), H)


def test_forward_is_deterministic_and_int64_actions_agree():
    rng = np.random.default_rng(5)
    R, A = 300, 1000
    m, bits = make_masks(R, A, rng)
    acts = random_valid_actions(m, rng)
    logits = torch.from_numpy(rng.standard_normal((R, A)).astype(np.float32)).cuda()
    mb, at = torch.from_numpy(bits).cuda(), torch.from_numpy(acts).cuda()
    a, b = masked_log_prob(logits, mb, at), masked_log_prob(logits, mb, at.long())
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    c = masked_log_prob(logits, mb, at)
    assert torch.equal(a[0], c[0]) and torch.equal(a[1], c[1])


# ------------------------------------------------------------------ 2. backward
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
@pytest.mark.parametrize("A", [1, 33, 50, 1000, 8000])
def test_backward_matches_autograd(A, dtype):
    rng = np.random.default_rng(100 + A)
    R = 40
    m, bits = make_masks(R, A, rng)
    acts = random_valid_actions(m, rng)
    bad = [r for r in range(R) if m[r].any()][:3]           # out-of-mask actions: -inf and no log_prob gradient
    acts[bad[0]] = A
    acts[bad[1]] = -5
    if not m[bad[2]].all():
        acts[bad[2]] = int(np.flatnonzero(~m[bad[2]])[0])
    logits = torch.from_numpy(rng.standard_normal((R, A)).astype(np.float32) * 2).to(dtype).cuda()
    mb, at = torch.from_numpy(bits).cuda(), torch.from_numpy(acts).cuda()
    g_lp = torch.from_numpy(rng.standard_normal(R).astype(np.float32)).cuda()
    g_H = torch.from_numpy(rng.standard_normal(R).astype(np.float32)).cuda()
    x = logits.clone().requires_grad_(True)
    lp, H = masked_log_prob(x, mb, at)
    for r in bad[:2]:
        assert lp[r].item() == -np.inf
    (gx,) = torch.autograd.grad((lp, H), x, (g_lp, g_H))
    assert gx.dtype == dtype and gx.shape == logits.shape
    valid = torch.from_numpy(m).cuda()
    x64 = logits.double().requires_grad_(True)
    rlp, rH, _, ok = reference(x64, valid, at)
    (rg,) = torch.autograd.grad((rlp, rH), x64, (torch.where(ok, g_lp.double(), torch.zeros_like(rlp)), g_H.double()))
    assert bool((gx[~valid] == 0).all()), "gradient on invalid entries"
    empty = torch.from_numpy(~m.any(-1)).cuda()
    assert bool((gx[empty] == 0).all()), "gradient on empty rows"
    if dtype == torch.float32:
        close(gx[valid], rg[valid], "grad_logits")
    else:   # the gradient is stored in bfloat16: within its rounding of the float64 value
        err = (gx[valid].double() - rg[valid]).abs()
        assert bool((err <= 1e-5 + 2.0 ** -8 * rg[valid].abs()).all()), float(err.max())
    # only one of the two outputs used
    (g1,) = torch.autograd.grad(masked_log_prob(x, mb, at)[1].sum(), x)
    (r1,) = torch.autograd.grad(reference(x64, valid, at)[1].sum(), x64)
    if dtype == torch.float32:
        close(g1[valid], r1[valid], "grad_logits (entropy only)")


# ------------------------------------------------------------------ 3. greedy
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
@pytest.mark.parametrize("A", [31, 50, 1000, 8000])
def test_greedy_equals_masked_argmax(A, dtype):
    rng = np.random.default_rng(7 + A)
    B = 64
    m, bits = make_masks(B, A, rng)
    env = sampler_env(B, A)
    env.t["mask_bits"].copy_(torch.from_numpy(bits))
    x = rng.standard_normal((B, A)).astype(np.float32)
    x[::3] = np.round(x[::3])            # deliberate ties: integer logits in every third row
    x[1::7] = 0.5                        # and rows of all-equal logits
    logits = torch.from_numpy(x).to(dtype).cuda()
    acts, lp, H = env.sample_logits(logits, 0, 0, greedy=True)
    valid = torch.from_numpy(m).cuda()
    x64 = logits.double()
    ref = torch.where(valid, x64, torch.full_like(x64, -np.inf)).argmax(-1)
    any_ = valid.any(-1)
    exp = torch.where(any_, ref, torch.full_like(ref, -1)).int()
    assert torch.equal(acts, exp)
    assert bool((lp[~any_] == 0).all()) and bool((H[~any_] == 0).all())


# ------------------------------------------------------------------ 4. stochastic draw, exact
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
@pytest.mark.parametrize("A", [33, 50, 1000, 8000])
def test_gumbel_draw_matches_numpy_restatement(A, dtype):
    rng = np.random.default_rng(11 + A)
    B, seed, t, env_id0 = 96, 1234567, 17, 4096
    m, bits = make_masks(B, A, rng)
    env = sampler_env(B, A, env_id0=env_id0)
    env.t["mask_bits"].copy_(torch.from_numpy(bits))
    clock = env.enable_env_clock()
    clock.copy_(torch.arange(B, dtype=torch.int32) * 3)
    logits = torch.from_numpy(rng.standard_normal((B, A)).astype(np.float32)).to(dtype).cuda()
    acts = env.sample_logits(logits, seed, t)[0].cpu().numpy()
    x = logits.double().cpu().numpy()
    near = 0
    for b in range(B):
        if not m[b].any():
            assert acts[b] == -1
            continue
        g = np_gumbel(seed, env_id0 + b, t + 3 * b, A)
        score = np.where(m[b], x[b] + g, -np.inf)
        best = int(np.argmax(score))
        a = int(acts[b])
        assert 0 <= a < A and m[b, a], "row %d drew an invalid action %d" % (b, a)
        if a != best:
            assert score[best] - score[a] <= 1e-4, "row %d: %d (%.7f) vs %d (%.7f)" % (b, a, score[a], best, score[best])
            near += 1
    assert near <= 2, "%d rows needed the near-tie tolerance" % near


# ------------------------------------------------------------------ 5. stochastic draw, distribution
def test_gumbel_draw_distribution_chi_square():
    from scipy.stats import chisquare
    B, A = 1 << 18, 50
    rng = np.random.default_rng(3)
    valid = rng.random(A) < 0.8
    valid[:2] = True
    row = np.linspace(-3.0, 2.0, A).astype(np.float32)
    env = sampler_env(B, A)
    env.t["mask_bits"].copy_(torch.from_numpy(pack(np.broadcast_to(valid, (B, A)))))
    logits = torch.from_numpy(row).cuda().expand(B, A)
    acts = env.sample_logits(logits, 99, 5)[0].cpu().numpy()
    counts = np.bincount(acts, minlength=A)
    assert counts[~valid].sum() == 0
    p = np.exp(row.astype(np.float64) - row[valid].max()) * valid
    p /= p.sum()
    res = chisquare(counts[valid], p[valid] * B)
    assert res.pvalue > 1e-6, res


# ------------------------------------------------------------------ 6. sampler == forward, bit for bit
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "bf16"])
@pytest.mark.parametrize("greedy", [False, True])
@pytest.mark.parametrize("A", [31, 1000, 8000])
def test_sampler_log_prob_equals_forward_bitwise(A, greedy, dtype):
    rng = np.random.default_rng(21 + A)
    B = 200
    m, bits = make_masks(B, A, rng)
    env = sampler_env(B, A)
    env.t["mask_bits"].copy_(torch.from_numpy(bits))
    logits = (torch.from_numpy(rng.standard_normal((B, A)).astype(np.float32)) * 4).to(dtype).cuda()
    acts, lp, H = env.sample_logits(logits, 8, 2, greedy=greedy)
    flp, fH = masked_log_prob(logits, env.t["mask_bits"], acts)
    assert torch.equal(lp, flp) and torch.equal(H, fH)
    assert bool(torch.exp(flp - lp)[acts >= 0].eq(1).all()), "PPO ratio"


# ------------------------------------------------------------------ 7. policy-driven rollouts vs the C oracle
ROLLOUTS = [
    ("LongestPath-v0", 50, 200, {"parenting": 2}, False),                      # lane-per-env
    ("ShortestPath-v0", 300, 700, {}, False),                                  # group-per-env
    ("SteinerTree-v0", 100, 500, {"n_dests": 99}, False),                      # incremental mask
    ("MulticastRouting-v0", 120, 600, {"parenting": 4, "n_dests": 5}, False),  # incremental mask
    ("DistributionCenter-v0", 120, 500, {"parenting": 2}, False),              # dc family
    ("PerishableProductDelivery-v0", 40, 100, {"n_products": 3, "parenting": 1}, False),
    ("LongestPath-v0", 50, 200, {"parenting": 2}, True),                       # warp-per-env
]


def _traj(cs, a, o):
    cs = ((cs << 7) | (cs >> 57)) & M64
    return cs ^ (a & 0xFFFFFFFF) ^ (int(o["done"]) << 40) ^ ((o["solved"] & 3) << 44) ^ (o["status"] << 48)


@pytest.mark.parametrize("cfg", ROLLOUTS, ids=["%s-N%d%s" % (c[0][:-3], c[1], "-warp" if c[4] else "") for c in ROLLOUTS])
def test_policy_rollout_matches_oracle(cfg):
    env_id, N, E, kw, warp = cfg
    B, T, seed = 150, 40, 13
    env = BatchedGraphEnv(env_id, B, N, E, auto_reset=True, force_warp=warp, **kw)
    p = env.params
    inst = []
    for b in range(B):
        random.seed(2000 + b)
        np.random.seed(2000 + b)
        inst.append(generate_instance(env_id, p))
    env.load_instances(inst)
    if env_id == "MulticastRouting-v0":
        env.finalize_graphs(u01=torch.tensor([i.u01 for i in inst], dtype=torch.float64, device="cuda"))
        md = env.t["max_dist32"].cpu().numpy()
        for b, i in enumerate(inst):
            i.max_distance = float(md[b])
    oenvs = [cu.oracle_from_instance(env_id, i, p) for i in inst]
    env.reset()
    masks = [oe.mask(reset_patch=True) for oe in oenvs]
    A = env.desc.A
    gen = torch.Generator(device="cuda")
    cs = [0] * B
    for t in range(T):
        gen.manual_seed(t)
        logits = torch.randn((B, A), generator=gen, device="cuda") * 2
        acts, lp, H = env.sample_logits(logits, seed, t)
        a = acts.cpu().numpy()
        for b in range(B):
            assert 0 <= a[b] < A and masks[b][a[b]], "%s env %d step %d: action %d not valid" % (env_id, b, t, a[b])
        reward, done, info = env.step(acts)
        torch.cuda.synchronize()
        status = info["status"].cpu().numpy()
        gmask = env.t["mask_bits"].cpu().numpy()
        for b, oe in enumerate(oenvs):
            o = oe.step(int(a[b]))
            tag = "%s env %d step %d" % (env_id, b, t)
            assert o["status"] == 0 and status[b] == 0, tag
            cs[b] = _traj(cs[b], int(a[b]), o)
            if o["done"]:
                oe.reset_state()
                masks[b] = oe.mask(reset_patch=True)
            elif o["has_mask"]:
                masks[b] = o["mask"]
            np.testing.assert_array_equal(unpack(gmask[b], A), masks[b], err_msg="mask " + tag)
    traj = env.t["traj"].cpu().numpy().view(np.uint64)
    assert [int(x) for x in traj] == cs


# ------------------------------------------------------------------ 8. scheduling equivalence
def _rollout_env(**kw):
    e = BatchedGraphEnv("LongestPath-v0", 256, 50, 200, parenting=2, auto_reset=True, **kw)
    e.generate(seed=31)
    e.reset()
    return e


def test_slice_sampler_uses_global_env_ids():
    e = _rollout_env()
    lo, n = 64, 128
    logits = torch.randn((e.B, e.desc.A), device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
    acts, lp, H = e.sample_logits(logits, 77, 3)
    sd = e.slice_desc(lo, n)
    sa = torch.empty(n, dtype=torch.int32, device="cuda")
    slp, sH = torch.empty(n, device="cuda"), torch.empty(n, device="cuda")
    part = logits[lo:lo + n].contiguous()
    _native.check(e.lib.ge_sample_logits(C.byref(sd), C.c_void_p(part.data_ptr()), 0, 0, 77, 3, C.c_void_p(sa.data_ptr()),
                                         C.c_void_p(slp.data_ptr()), C.c_void_p(sH.data_ptr()), e._stream()))
    assert torch.equal(sa, acts[lo:lo + n]) and torch.equal(slp, lp[lo:lo + n]) and torch.equal(sH, H[lo:lo + n])


def test_graph_replay_and_pdl_equal_eager():
    K, seed = 30, 5
    logits = torch.randn((256, 50), device="cuda", generator=torch.Generator(device="cuda").manual_seed(2))
    runs = {}
    for mode in ("eager", "graph", "pdl"):
        e = _rollout_env()
        e.enable_env_clock()
        if mode == "pdl":
            e.enable_pdl()
        lp = torch.empty(e.B, device="cuda")
        H = torch.empty(e.B, device="cuda")
        out = (e.actions_dev, lp, H)
        log = []
        if mode == "graph":
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                e.sample_logits(logits, seed, 0, out=out)
                e.step_async(e.actions_dev)
            for _ in range(K):
                g.replay()
                log.append((e.actions_dev.clone(), lp.clone()))
        else:
            for _ in range(K):
                e.sample_logits(logits, seed, 0, out=out)
                e.step_async(e.actions_dev)
                log.append((e.actions_dev.clone(), lp.clone()))
        torch.cuda.synchronize()
        runs[mode] = (e, log)
    e0, l0 = runs["eager"]
    assert len(torch.unique(torch.stack([a for a, _ in l0])[:, 0])) > 1, "the env clock must vary the draws"
    for mode in ("graph", "pdl"):
        e1, l1 = runs[mode]
        for (a0, p0), (a1, p1) in zip(l0, l1):
            assert torch.equal(a0, a1) and torch.equal(p0, p1), mode
        for name in ("traj", "acc", "mask_bits", "head"):
            assert torch.equal(e0.t[name], e1.t[name]), (mode, name)
