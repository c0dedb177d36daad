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
"""
import ctypes as C
from types import SimpleNamespace

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
