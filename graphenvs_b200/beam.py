"""Beam search and multi-start decoding on the device (ge_beam_expand in csrc/ge_policy.cu, forks through csrc/ge_state.cu).

    bs = BeamSearch(venv, width=16)      # a wide batch of G * W envs: W beams per instance of venv
    res = bs.run(policy)                 # policy(wide_env) -> logits [G * W, A] float32 / bfloat16
    res.actions, res.ret, res.solution_cost, res.solved, res.log_prob, res.found, res.beams

Beam j of instance g lives in env g * W + j of the wide batch.  A decode step asks the policy for logits, keeps the W best
continuations of every group (ge_beam_expand: score = sum of masked log-probs, exact total order), forks each slot from
the beam it continues (save every env, load by index), and steps every slot with its action.  A finished beam stays a
candidate with its score and is stepped with -1 (GE_STEP_AFTER_DONE: state and statistics unchanged), so each env's `acc`
column -- zeroed at the start and forked with its beam -- is that branch's own return, final cost and solved flag.  The
initial scores [0, -inf, ..., -inf] make the first expansion pick W distinct first actions: multi-start decoding is the
same loop.

    sbs = StochasticBeamSearch(venv, width=16, seed=0)   # 16 distinct sequences per instance, sampled without replacement
    res = sbs.run(policy)                                # as above, plus res.kappa and res.beams.log_prob / key / weight

StochasticBeamSearch is the same loop with ge_beam_expand_sampled: candidates ranked by Gumbel-perturbed log-probs conditioned
on their parent's (Kool, van Hoof, Welling 2019), with noise keyed by (seed, global instance id, action prefix).
"""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import torch

from . import _native
from .policy import _DTYPES

MAX_WIDTH = 32


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class BeamSearch:
    """Beam search of width `width` (1 <= width <= 32) over every instance of the loaded batch `venv`.

    The wide batch (`self.wide`, venv.like(G * width, auto_reset=False)), its record buffer and the per-step history are
    allocated here and reused by every run(); the history grows (by doubling) when a run needs more steps than it holds."""

    def __init__(self, venv, width=16):
        from .batch import BatchedGraphEnv, EnvStates
        if not isinstance(venv, BatchedGraphEnv):
            raise TypeError("BeamSearch: venv must be a BatchedGraphEnv")
        if isinstance(width, bool) or not isinstance(width, int) or not 1 <= width <= MAX_WIDTH:
            raise ValueError("BeamSearch: width must be an integer in [1, %d], got %r" % (MAX_WIDTH, width))
        if not venv._loaded:
            raise ValueError("BeamSearch: venv has no instances (load_instances() or generate() first)")
        self.venv, self.W, self.G = venv, width, venv.B
        self.B = self.G * width
        self.wide = venv.like(self.B, auto_reset=False)
        if venv.env_steps is not None:       # same state arrays as venv, so from_current can load its records
            self.wide.enable_env_clock()
        dev = self.wide.device
        self.src_index = torch.arange(self.G, dtype=torch.int32, device=dev).repeat_interleave(width)
        self.records = EnvStates(torch.empty((self.B, self.wide.record_bytes()), dtype=torch.uint8, device=dev),
                                 self.wide.state_signature())
        self.score = torch.empty(self.B, dtype=torch.float32, device=dev)
        self._score_next = torch.empty(self.B, dtype=torch.float32, device=dev)
        self.load_index = torch.empty(self.B, dtype=torch.int32, device=dev)
        self._parents = torch.empty((0, self.B), dtype=torch.int32, device=dev)    # history: parent env / action of every slot
        self._actions = torch.empty((0, self.B), dtype=torch.int32, device=dev)
        self.t = 0

    # ------------------------------------------------------------------ the loop, piece by piece
    def reserve(self, steps):
        """Room for `steps` decode steps in the history (before capturing a decode in a CUDA graph)."""
        cap = self._parents.shape[0]
        if steps <= cap:
            return
        new = max(int(steps), 2 * cap, 16)
        p = torch.empty((new, self.B), dtype=torch.int32, device=self.wide.device)
        a = torch.empty_like(p)
        p[:self.t].copy_(self._parents[:self.t])
        a[:self.t].copy_(self._actions[:self.t])
        self._parents, self._actions = p, a

    def start(self, from_current=False):
        """Every slot of group g <- instance g of venv, from reset() or (from_current=True) from venv's current state; acc is
        zeroed and the scores are [0, -inf, ..., -inf] per group."""
        wide = self.wide
        wide.gather_instances(self.venv, self.src_index)
        if from_current:
            wide.load_states(self.venv.save_states(), self.src_index)
        else:
            wide.reset()
        wide.t["acc"].zero_()
        self.score.fill_(float("-inf"))
        self.score.view(self.G, self.W)[:, 0] = 0.0
        self.t = 0

    def _check_logits(self, logits):
        A = self.wide.desc.A
        if not isinstance(logits, torch.Tensor) or logits.device != self.wide.device:
            raise ValueError("BeamSearch: logits must be a tensor on %s" % self.wide.device)
        if logits.dtype not in _DTYPES:
            raise TypeError("BeamSearch: logits must be float32 or bfloat16, got %s" % logits.dtype)
        if tuple(logits.shape) != (self.B, A):
            raise ValueError("BeamSearch: logits shape %s, expected (%d, %d)" % (tuple(logits.shape), self.B, A))
        return logits.detach().contiguous()

    def expand(self, logits, parent=None, action=None):
        """One ge_beam_expand over the wide batch's current masks: the W best continuations of every group.  Replaces
        self.score with the new scores and returns (parent, action, load_index) int32 [G * W] (include/graphenvs_b200.h).
        The caller then forks and steps: wide.save_states(out=bs.records); wide.load_states(bs.records, load_index);
        wide.step_async(action)."""
        x = self._check_logits(logits)
        if parent is None:
            parent = torch.empty(self.B, dtype=torch.int32, device=self.wide.device)
        if action is None:
            action = torch.empty(self.B, dtype=torch.int32, device=self.wide.device)
        wide = self.wide
        _native.check(wide.lib.ge_beam_expand(C.byref(wide.desc), self.W, _ptr(x), _DTYPES[x.dtype], _ptr(self.score),
                                              _ptr(self._score_next), _ptr(parent), _ptr(action), _ptr(self.load_index),
                                              wide._stream()))
        self.score, self._score_next = self._score_next, self.score
        return parent, action, self.load_index

    def advance(self, logits):
        """One decode step: expand into the history, fork every slot from its parent, step every slot with its action."""
        self.reserve(self.t + 1)
        parent, action, load_index = self.expand(logits, self._parents[self.t], self._actions[self.t])
        wide = self.wide
        wide.save_states(out=self.records)
        wide.load_states(self.records, load_index)
        wide.step_async(action)
        self.t += 1

    def live(self):
        """True while some slot holds a beam (score > -inf) whose episode has not ended (one device sync)."""
        return bool(((self.score > float("-inf")) & (self.wide.t["done"] == 0)).any())

    def result(self):
        """The decode so far: per group the best finished beam (highest return, ties to the lowest slot), and every beam."""
        G, W, T, dev = self.G, self.W, self.t, self.wide.device
        acc = self.wide.t["acc"]
        done = self.wide.t["done"] != 0
        alive = self.score > float("-inf")
        # backtrack every slot through the history; an empty slot (score -inf) has no sequence
        seq = torch.full((self.B, T), -1, dtype=torch.int32, device=dev)
        cur = torch.arange(self.B, dtype=torch.int64, device=dev)
        for t in range(T - 1, -1, -1):
            c = cur.clamp(min=0)
            seq[:, t] = self._actions[t][c]
            cur = self._parents[t][c].long()
        seq[~alive] = -1
        ret = acc[2].clone()
        finished = alive & done
        key = torch.where(finished, ret, torch.full_like(ret, float("-inf"))).view(G, W)
        best = key.argmax(dim=1)                                   # first maximum: the lowest slot on ties
        found = finished.view(G, W).any(dim=1)
        rows = torch.arange(G, device=dev) * W + best
        nan = torch.full((G,), float("nan"), dtype=torch.float64, device=dev)
        beams = SimpleNamespace(actions=seq.view(G, W, T), ret=ret.view(G, W), score=self.score.clone().view(G, W),
                                done=done.view(G, W), solution_cost=acc[3].clone().view(G, W), solved=(acc[1] > 0).view(G, W))
        return SimpleNamespace(
            actions=torch.where(found[:, None], seq[rows], torch.full_like(seq[rows], -1)),
            ret=torch.where(found, ret[rows], nan),
            solution_cost=torch.where(found, acc[3][rows], nan),
            solved=found & (acc[1][rows] > 0),
            log_prob=torch.where(found, self.score[rows], torch.full_like(self.score[rows], float("-inf"))),
            found=found, steps=T, beams=beams)

    # ------------------------------------------------------------------ the whole decode
    def run(self, policy, max_steps=None, from_current=False, check_every=8):
        """Decodes every instance of venv: start(from_current), then advance(policy(self.wide)) until every beam has finished
        (checked on the host every `check_every` steps) or after max_steps steps (default 4 * N).  Returns result():
          actions        int32 [G, T] the best finished beam of each instance, -1 padded (T = steps run)
          ret            float64 [G] its return (sum of rewards), NaN when no beam finished
          solution_cost  float64 [G] its final solution_cost (0 when the last step reported none), NaN when no beam finished
          solved         bool [G] info['solved'] of its last step
          log_prob       float32 [G] its score, the sum of its masked log-probs
          found          bool [G] some beam of the instance finished within max_steps
          beams          every slot: actions [G, W, T], ret, solution_cost, solved, score [G, W] and done [G, W]
        A beam's score ties with others' only through equal log-probs; among finished beams the return decides."""
        if max_steps is None:
            max_steps = 4 * self.wide.N
        self.start(from_current)
        self.reserve(max_steps)
        check_every = max(1, int(check_every))
        while self.t < max_steps:
            if self.t % check_every == 0 and not self.live():
                break
            self.advance(policy(self.wide))
        return self.result()


# ---------------------------------------------------------------------- stochastic beam search
_M64 = (1 << 64) - 1
ROOT_T = 0x52DCE729          # the counter of the root node keys (include/graphenvs_b200.h, ge_beam_expand_sampled)


def _mix32(seed, env, t):
    """csrc/ge_common.cuh:mix32 in numpy uint64 arithmetic (wrapping); seed / env broadcast."""
    with np.errstate(over="ignore"):
        seed, env, t = np.asarray(seed, dtype=np.uint64), np.asarray(env, dtype=np.uint64), np.uint64(t)
        z = seed + np.uint64(0x9E3779B97F4A7C15) * (env * np.uint64(0x100000001) + ((t << np.uint64(32)) | np.uint64(0x5bd1e995)))
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
        return z >> np.uint64(32)


def root_key(seed, instance):
    """Node key of the root of global instance id(s) `instance` (numpy uint64):
    (uint64) mix32(seed, i, 0x52DCE729) << 32 | mix32(seed ^ 0xD1B54A32D192ED03, i, 0x52DCE729)."""
    i = np.asarray(instance, dtype=np.uint64)
    return (_mix32(np.uint64(seed), i, ROOT_T) << np.uint64(32)) | _mix32(np.uint64(seed ^ 0xD1B54A32D192ED03), i, ROOT_T)


def root_gumbel(node_key):
    """The Gumbel(0) key of a root: the noise of ge_sample_logits' formula at action 0xFFFFFFFF of the root's node key, in
    float64 (the caller rounds it to float32)."""
    h = _mix32(np.asarray(node_key, dtype=np.uint64), 0xFFFFFFFF, 0x85EBCA6B)
    u = ((h >> np.uint64(8)).astype(np.float64) + 0.5) / 2.0 ** 24
    return -np.log(-np.log(u))


class StochasticBeamSearch(BeamSearch):
    """Stochastic beam search (Kool, van Hoof, Welling 2019): per instance of `venv`, `width` distinct sequences drawn without
    replacement from the policy's sequence distribution, with ge_beam_expand_sampled as the expand step.

    It is BeamSearch's loop (wide batch, forks, steps, history, backtracking) with three ping-pong arrays per slot instead of
    the score: the log-prob phi (kept in `score`, so an empty slot is still score -inf), the perturbed log-prob `key` and the
    tree-node key `node_key` that keys the Gumbel noise.  The noise of a node depends only on (seed, global instance id,
    action prefix), so a wider search extends a narrower one (its first W slots are the width-W search), a rank slice of the
    instances (venv.desc.env_id0 > 0) draws what the full batch draws for them, and width 1 is ancestral sampling."""

    def __init__(self, venv, width=16, seed=0):
        if isinstance(seed, bool) or not isinstance(seed, int):
            raise TypeError("StochasticBeamSearch: seed must be an int, got %r" % (seed,))
        if not 0 <= seed <= _M64:
            raise ValueError("StochasticBeamSearch: seed must be in [0, 2^64), got %d" % seed)
        super().__init__(venv, width)
        self.seed = seed
        dev = self.wide.device
        rk = root_key(seed, int(venv.desc.env_id0) + np.arange(self.G, dtype=np.uint64))
        self._root_key = torch.from_numpy(rk.view(np.int64).copy()).to(dev)
        self._root_gumbel = torch.from_numpy(root_gumbel(rk).astype(np.float32)).to(dev)
        self.key = torch.empty(self.B, dtype=torch.float32, device=dev)
        self._key_next = torch.empty_like(self.key)
        self.node_key = torch.empty(self.B, dtype=torch.int64, device=dev)       # uint64 bit patterns
        self._node_key_next = torch.empty_like(self.node_key)
        self._thresholds = torch.empty((0, self.G), dtype=torch.float32, device=dev)

    def reserve(self, steps):
        super().reserve(steps)
        cap = self._parents.shape[0]
        if self._thresholds.shape[0] < cap:
            th = torch.empty((cap, self.G), dtype=torch.float32, device=self.wide.device)
            th[:self.t].copy_(self._thresholds[:self.t])
            self._thresholds = th

    def start(self, from_current=False):
        """BeamSearch.start, then slot 0 of group g becomes the root: logp 0, key G_root(g), node key root_key(seed,
        venv.desc.env_id0 + g); the other slots are dead (key -inf)."""
        super().start(from_current)
        self.key.fill_(float("-inf"))
        self.key.view(self.G, self.W)[:, 0] = self._root_gumbel
        self.node_key.zero_()
        self.node_key.view(self.G, self.W)[:, 0] = self._root_key

    def expand(self, logits, parent=None, action=None):
        """One ge_beam_expand_sampled over the wide batch's current masks: per group the W children of largest conditioned
        key.  Replaces score (phi), key and node_key, records the group thresholds at history row t (reserve(t + 1) first) and
        returns (parent, action, load_index) as BeamSearch.expand does."""
        x = self._check_logits(logits)
        dev = self.wide.device
        if parent is None:
            parent = torch.empty(self.B, dtype=torch.int32, device=dev)
        if action is None:
            action = torch.empty(self.B, dtype=torch.int32, device=dev)
        self.reserve(self.t + 1)
        wide = self.wide
        _native.check(wide.lib.ge_beam_expand_sampled(
            C.byref(wide.desc), self.W, _ptr(x), _DTYPES[x.dtype], _ptr(self.score), _ptr(self.key), _ptr(self.node_key),
            _ptr(self._score_next), _ptr(self._key_next), _ptr(self._node_key_next), _ptr(parent), _ptr(action),
            _ptr(self.load_index), _ptr(self._thresholds[self.t]), wide._stream()))
        self.score, self._score_next = self._score_next, self.score
        self.key, self._key_next = self._key_next, self.key
        self.node_key, self._node_key_next = self._node_key_next, self.node_key
        return parent, action, self.load_index

    def result(self):
        """BeamSearch.result() (the best finished return per group, every slot), plus:
          beams.log_prob  float32 [G, W] phi, the sum of each sequence's masked log-probs (= beams.score)
          beams.key       float32 [G, W] its perturbed log-prob G; slots come in descending key order, so slot 0 is an exact
                          draw from the policy's sequence distribution
          kappa           float32 [G] the largest group threshold over the steps: the (W+1)-th largest leaf key, -inf when
                          the search enumerated every sequence
          beams.weight    float64 [G, W] exp(phi) / q, q = -expm1(-exp(phi - kappa)) the inclusion probability (q = 1 when
                          kappa = -inf); 0 for an empty slot, NaN for every slot of a group with a live unfinished beam.
        sum_j weight[g, j] f(y_j) is an unbiased estimate of E_y[f(y)] (priority sampling)."""
        res = super().result()
        G, W, T = self.G, self.W, self.t
        neg = float("-inf")
        if T:
            kappa = self._thresholds[:T].amax(dim=0)
        else:
            kappa = torch.full((G,), neg, dtype=torch.float32, device=self.wide.device)
        phi = self.score.view(G, W).double()
        k = kappa.double()[:, None]
        q = torch.where(k == neg, torch.ones_like(phi), -torch.expm1(-torch.exp(phi - k)))
        alive = phi > neg
        weight = torch.where(alive, torch.exp(phi) / q, torch.zeros_like(phi))
        unfinished = (alive & ~res.beams.done).any(dim=1, keepdim=True)
        weight = torch.where(unfinished, torch.full_like(weight, float("nan")), weight)
        res.beams.log_prob = res.beams.score
        res.beams.key = self.key.clone().view(G, W)
        res.beams.weight = weight
        res.kappa = kappa
        return res
