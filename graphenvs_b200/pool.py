"""Instance turnover for BatchedGraphEnv: every reference reset() builds a NEW graph (e.g. shortest_path.py:47-98); here a
resident pool of G fully prepared banks feeds the envs whose episodes end, and a background stream keeps regenerating
banks (SURVEY.md 8(f1), csrc/ge_pool.cu).

    pool = InstancePool(env, banks=4, seed=1)        # env: BatchedGraphEnv(auto_reset=False)
    ...
    env.step_sampled(seed, t)                          # or env.step(actions)
    pool.turn_over()                                   # done envs get their next instance + reset(); others untouched
"""
import ctypes as C

import torch

from . import _native
from .batch import _ptr


class InstancePool:
    def __init__(self, env, banks=4, seed=0, background=True):
        assert not (env.desc.flags & 1), "the live batch must run with auto_reset=False: the pool performs the resets"
        assert 2 <= banks <= 8
        self.env, self.G, self.seed = env, int(banks), int(seed)
        self.banks = []
        for k in range(self.G):
            # banks keep their float64 weights: a generate() without them synchronises, and banks regenerate in the background
            b = env.like(env.B, byte_mask=False, keep_w64=True)
            b.generate(seed=self._next_seed(), check=False)
            if "mask0_bits" in b.t:
                b.reset()                       # fills mask0_bits (the first mask depends only on the instance)
            self.banks.append(b)
        if "dfa" in env.t:
            for b in self.banks:
                assert torch.equal(b.t["dfa"], env.t["dfa"]), "banks must share the live batch's distance automaton"
        self._descs = (_native.GeBatch * self.G)(*[b.desc for b in self.banks])
        dev = env.device
        self.background = bool(background)
        self.n_active = self.G - 1 if self.background else self.G
        self.order = torch.arange(self.n_active, dtype=torch.int32, device=dev)
        self._host_order = list(range(self.n_active))
        self.episode = torch.zeros(env.B, dtype=torch.int32, device=dev)
        self.select = torch.zeros(env.B, dtype=torch.uint8, device=dev)
        self.refills = 0
        self.regenerated = 0
        self._side = torch.cuda.Stream(device=dev) if self.background else None
        self._spare = self.G - 1                  # the bank that is not in `order` and may be rewritten
        self._gen_done = None
        if self.background:
            self._start_regeneration()

    def _next_seed(self):
        self.seed += 1
        return 0x5EED0000 + self.seed

    def _start_regeneration(self):
        """Rewrites the spare bank on the side stream.  Nothing on the main stream reads it (it is not in `order`)."""
        bank = self.banks[self._spare]
        self._side.wait_stream(torch.cuda.current_stream(self.env.device))   # the swap that retired this bank has been enqueued
        with torch.cuda.stream(self._side):
            bank.generate(seed=self._next_seed(), check=False)
            if "mask0_bits" in bank.t:
                bank.reset()
            self._gen_done = torch.cuda.Event()
            self._gen_done.record(self._side)

    def _maybe_swap(self):
        """When the spare bank is ready: it replaces the OLDEST active bank (on the main stream, so every refill already
        enqueued still sees the old order), and the retired bank becomes the next one to regenerate."""
        if not self.background or self._gen_done is None or not self._gen_done.query():
            return
        main = torch.cuda.current_stream(self.env.device)
        main.wait_event(self._gen_done)
        pos = self.regenerated % self.n_active
        retired = self._host_order[pos]            # the order is mirrored on the host: no device read-back
        self._host_order[pos] = self._spare
        self.order[pos:pos + 1].fill_(self._spare)
        self._spare = retired
        self.regenerated += 1
        self._start_regeneration()

    def turn_over(self):
        """Gives every finished env its next instance and resets it (two launches on the current stream)."""
        env = self.env
        self._maybe_swap()
        _native.check(env.lib.ge_pool_refill(C.byref(env.desc), self._descs, self.G, _ptr(self.order), self.n_active,
                                             _ptr(self.episode), _ptr(self.select), env._stream()))
        _native.check(env.lib.ge_reset(C.byref(env.desc), _ptr(self.select), env._stream()))
        self.refills += 1

    def close(self):
        if self._side is not None:
            self._side.synchronize()
