"""Monte Carlo tree search with PUCT selection on the device (ge_mcts_select / ge_mcts_expand in csrc/ge_policy.cu, forks
through csrc/ge_state.cu).

    mcts = MCTS(venv, num_simulations=64, c_puct=1.25)
    out = mcts.search(policy)     # policy(leaf_env) -> (logits [G, A] float32 / bfloat16, value [G] float32)
    out.visits, out.q, out.value, out.action
    res = mcts.run(policy)        # whole episodes: one search per move, then the most-visited action is stepped
    res.actions, res.ret, res.solution_cost, res.solved, res.found, res.steps, res.root_value

Every instance g of venv is searched in parallel with num_simulations simulations, AlphaZero / MuZero style (the semantics,
bit for bit, are in include/graphenvs_b200.h).  Node k of every instance is created in simulation k, so the env state
records are laid out [S + 1, G, R] and a simulation round is: select; load every instance's parent node record into the
leaf batch (G envs); step it with the selected actions; ask the policy; save the leaf batch as the node-k records; expand
and back up.  The leaf batch is stepped only through these forks, so the searched env itself is never touched.
"""
import ctypes as C
from types import SimpleNamespace

import torch

from . import _native
from .policy import _DTYPES

_PDL = 16   # GE_FLAG_PDL


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def unpack_mask(bits, A):
    """Packed masks int32 [..., AW] -> bool [..., A]."""
    shifts = torch.arange(32, device=bits.device, dtype=torch.int32)
    b = (bits.unsqueeze(-1) >> shifts) & 1
    return b.flatten(-2)[..., :A].bool()


class MCTS:
    """Monte Carlo tree search over every instance of the loaded batch `venv`: `num_simulations` (>= 1) simulations per
    search, PUCT exploration constant `c_puct` (finite, >= 0).

    The tree tensors (node-major, [S + 1, G] and [S + 1, G, A]; include/graphenvs_b200.h, ge_mcts_tree), the record buffer
    `records` ([S + 1, G, R]) and the leaf batch `leaf` (venv.like(G, auto_reset=False), with the env clock when venv has
    one) are allocated here and reused by every search.  `sel_action` and `depth` (int32 [G]) hold the current simulation's
    selection -- the action that led to the leaf and the leaf's depth -- for policies keyed on them (-1 and 0 while the
    roots are evaluated)."""

    def __init__(self, venv, num_simulations, c_puct=1.25):
        from .batch import BatchedGraphEnv, EnvStates
        if not isinstance(venv, BatchedGraphEnv):
            raise TypeError("MCTS: venv must be a BatchedGraphEnv")
        if isinstance(num_simulations, bool) or not isinstance(num_simulations, int) or num_simulations < 1:
            raise ValueError("MCTS: num_simulations must be an integer >= 1, got %r" % (num_simulations,))
        if isinstance(c_puct, bool) or not isinstance(c_puct, (int, float)) or not 0.0 <= float(c_puct) < float("inf"):
            raise ValueError("MCTS: c_puct must be a finite number >= 0, got %r" % (c_puct,))
        if not venv._loaded:
            raise ValueError("MCTS: venv has no instances (load_instances() or generate() first)")
        self.venv, self.G, self.S, self.c_puct = venv, venv.B, num_simulations, float(c_puct)
        self.leaf = venv.like(self.G, auto_reset=False)
        if venv.env_steps is not None:       # same state arrays as venv, so its records load into the leaf batch
            self.leaf.enable_env_clock()
        G, S, dev = self.G, self.S, self.leaf.device
        A, AW = self.leaf.desc.A, self.leaf.desc.AW
        self.A = A
        i32 = dict(dtype=torch.int32, device=dev)
        self.parent = torch.full((S + 1, G), -1, **i32)
        self.action = torch.full((S + 1, G), -1, **i32)
        self.visits = torch.zeros((S + 1, G), **i32)
        self.wsum = torch.zeros((S + 1, G), dtype=torch.float64, device=dev)
        self.reward = torch.zeros((S + 1, G), dtype=torch.float32, device=dev)
        self.value = torch.zeros((S + 1, G), dtype=torch.float32, device=dev)
        self.terminal = torch.zeros((S + 1, G), dtype=torch.uint8, device=dev)
        self.child = torch.empty((S + 1, G, A), **i32)                       # read only where the node's mask is set
        self.prior = torch.empty((S + 1, G, A), dtype=torch.float32, device=dev)
        self.mask = torch.zeros((S + 1, G, AW), **i32)
        self.qmin = torch.empty(G, dtype=torch.float64, device=dev)
        self.qmax = torch.empty(G, dtype=torch.float64, device=dev)
        self.sel_node = torch.zeros(G, **i32)
        self.sel_action = torch.full((G,), -1, **i32)
        self.load_index = torch.full((G,), -1, **i32)
        self.depth = torch.zeros(G, **i32)
        sig = self.leaf.state_signature()
        self.records = EnvStates(torch.empty(((S + 1) * G, self.leaf.record_bytes()), dtype=torch.uint8, device=dev), sig)
        self._node_records = [EnvStates(self.records.data[k * G:(k + 1) * G], sig) for k in range(S + 1)]
        t = _native.MctsTree()
        t.G, t.S, t.A, t.AW, t.c_puct = G, S, A, AW, self.c_puct
        for f in ("parent", "action", "visits", "wsum", "reward", "value", "terminal", "child", "prior", "mask", "qmin", "qmax",
                  "sel_node", "sel_action", "load_index", "depth"):
            setattr(t, f, getattr(self, f).data_ptr())
        self.tree = t
        self.k = -1              # the last simulation run (0: the roots are expanded)
        self._game = None

    def memory_bytes(self):
        """Device bytes of the tree, the record buffer and the leaf batch: per node about R + 8 A + 4 AW + 29."""
        ts = (self.parent, self.action, self.visits, self.wsum, self.reward, self.value, self.terminal, self.child, self.prior,
              self.mask, self.qmin, self.qmax, self.sel_node, self.sel_action, self.load_index, self.depth, self.records.data)
        return sum(x.numel() * x.element_size() for x in ts) + self.leaf.memory_bytes()

    # ------------------------------------------------------------------ the search, piece by piece
    def _policy_out(self, out):
        """Checks policy(leaf) -> (logits [G, A] float32 / bfloat16, value [G] float32) on the leaf batch's device."""
        dev, G, A = self.leaf.device, self.G, self.A
        if not isinstance(out, (tuple, list)) or len(out) != 2:
            raise TypeError("MCTS: the policy must return (logits, value)")
        logits, value = out
        for name, x in (("logits", logits), ("value", value)):
            if not isinstance(x, torch.Tensor) or x.device != dev:
                raise ValueError("MCTS: policy %s must be a tensor on %s" % (name, dev))
        if logits.dtype not in _DTYPES:
            raise TypeError("MCTS: policy logits must be float32 or bfloat16, got %s" % logits.dtype)
        if value.dtype != torch.float32:
            raise TypeError("MCTS: policy value must be float32, got %s" % value.dtype)
        if tuple(logits.shape) != (G, A):
            raise ValueError("MCTS: policy logits shape %s, expected (%d, %d)" % (tuple(logits.shape), G, A))
        if tuple(value.shape) != (G,):
            raise ValueError("MCTS: policy value shape %s, expected (%d,)" % (tuple(value.shape), G))
        return logits.detach().contiguous(), value.detach().contiguous()

    def _expand(self, policy, k):
        leaf = self.leaf
        logits, value = self._policy_out(policy(leaf))
        _native.check(leaf.lib.ge_mcts_expand(C.byref(self.tree), k, C.byref(leaf.desc), _ptr(leaf.reward), _ptr(logits),
                                              _DTYPES[logits.dtype], _ptr(value), leaf._stream()))

    def start(self, policy, env=None):
        """Simulation 0: the leaf batch <- the instances and current states of `env` (default venv; G envs of venv's
        signature, left untouched), saved as the root records; the policy evaluates the roots, which become node 0."""
        from .batch import BatchedGraphEnv
        env = self.venv if env is None else env
        if not isinstance(env, BatchedGraphEnv) or env.B != self.G:
            raise ValueError("MCTS: env must be a BatchedGraphEnv of %d envs" % self.G)
        leaf = self.leaf
        leaf.gather_instances(env)
        env.save_states(out=self._node_records[0])
        leaf.load_states(self._node_records[0])
        self.sel_action.fill_(-1)
        self.depth.zero_()
        self._expand(policy, 0)
        self.k = 0

    def simulate(self, policy):
        """Simulation k = self.k + 1: select, fork the leaf batch from the parent nodes, step, ask the policy, save the node-k
        records, expand and back up.  No host synchronisation: a sequence of simulate() calls can be captured in a CUDA graph."""
        k = self.k + 1
        if not 1 <= k <= self.S:
            raise RuntimeError("MCTS: simulate() needs start() first and runs at most %d simulations" % self.S)
        leaf = self.leaf
        self.tree.flags = leaf.desc.flags & _PDL
        _native.check(leaf.lib.ge_mcts_select(C.byref(self.tree), k, leaf._stream()))
        leaf.load_states(self.records, self.load_index)
        leaf.step_async(self.sel_action)
        logits, value = self._policy_out(policy(leaf))
        leaf.save_states(out=self._node_records[k])
        _native.check(leaf.lib.ge_mcts_expand(C.byref(self.tree), k, C.byref(leaf.desc), _ptr(leaf.reward), _ptr(logits),
                                              _DTYPES[logits.dtype], _ptr(value), leaf._stream()))
        self.k = k

    def result(self):
        """The roots' statistics after the simulations so far:
          visits  int32 [G, A]    visit counts of the root's children (0 for unexpanded and invalid actions)
          q       float64 [G, A]  Q(root, a) = r(c) + Wsum(c) / N(c), NaN where unvisited
          value   float64 [G]     Wsum / N of the root
          action  int32 [G]       the most-visited action, ties to the lowest; -1 for a done root or one without valid actions"""
        G, A = self.G, self.A
        valid = unpack_mask(self.mask[0], A)
        ch = self.child[0]
        has = valid & (ch >= 0)
        idx = torch.where(has, ch, 0).long()
        g = torch.arange(G, device=idx.device)[:, None]
        n = torch.where(has, self.visits[idx, g], 0)
        q = torch.where(has, self.reward[idx, g].double() + self.wsum[idx, g] / n.clamp(min=1), float("nan"))
        action = torch.where((self.terminal[0] == 0) & has.any(dim=1), n.argmax(dim=1), -1)
        return SimpleNamespace(visits=n.int(), q=q, value=self.wsum[0] / self.visits[0], action=action.int())

    def search(self, policy, env=None):
        """start(policy, env), then num_simulations simulate(policy); returns result()."""
        self.start(policy, env)
        for _ in range(self.S):
            self.simulate(policy)
        return self.result()

    # ------------------------------------------------------------------ whole episodes
    def run(self, policy, max_steps=None, from_current=False):
        """Decodes every instance of venv on a copy (a G-env batch, auto-reset off): from reset() or (from_current=True) from
        venv's current state, one search per move, then the most-visited action is stepped, until every episode has ended
        (checked on the host after every move) or after max_steps moves (default 4 * N).  venv is left untouched.  Returns
          actions        int32 [G, T] the moves, -1 after the episode ended (T = moves made)
          ret            float64 [G] the return (sum of rewards), NaN when the episode did not end
          solution_cost  float64 [G] the final solution_cost (0 when the last step reported none), NaN when it did not end
          solved         bool [G] info['solved'] of the last step
          found          bool [G] the episode ended within max_steps
          steps          T
          root_value     float64 [G, T] Wsum / N of the root of each move's search, NaN after the episode ended"""
        venv = self.venv
        if max_steps is None:
            max_steps = 4 * venv.N
        if self._game is None:
            self._game = venv.like(self.G, auto_reset=False)
            if venv.env_steps is not None:
                self._game.enable_env_clock()
        game = self._game
        game.gather_instances(venv)
        if from_current:
            game.load_states(venv.save_states())
        else:
            game.reset()
        game.t["acc"].zero_()
        dev = game.device
        actions = torch.full((self.G, max_steps), -1, dtype=torch.int32, device=dev)
        root_value = torch.full((self.G, max_steps), float("nan"), dtype=torch.float64, device=dev)
        t = 0
        while t < max_steps:
            live = game.t["done"] == 0
            if not bool(live.any()):
                break
            out = self.search(policy, game)
            actions[:, t] = torch.where(live, out.action, -1)
            root_value[:, t] = torch.where(live, out.value, float("nan"))
            game.step_async(out.action)       # a done env gets -1: GE_STEP_AFTER_DONE, state and statistics unchanged
            t += 1
        acc = game.t["acc"]
        found = game.t["done"] != 0
        nan = torch.full((self.G,), float("nan"), dtype=torch.float64, device=dev)
        return SimpleNamespace(actions=actions[:, :t].clone(), ret=torch.where(found, acc[2], nan),
                               solution_cost=torch.where(found, acc[3], nan), solved=found & (acc[1] > 0), found=found,
                               steps=t, root_value=root_value[:, :t].clone())
