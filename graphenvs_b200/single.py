"""Gymnasium-shaped single environment over the CUDA engine (B = 1 batch).

Keeps the reference surface: ids and constructor kwargs (graph_envs/__init__.py:9-56 and the
constructors listed in spec.py), `reset(seed=None, options={}) -> (obs, info)`,
`step(action) -> (obs, reward, done, False, info)`, info['mask' / 'solved' / 'solution_cost' /
'heuristic_solution'], `AssertionError` for the actions the reference rejects.

reset(seed) reseeds the process-global `random` / `numpy.random` exactly like the reference
(shortest_path.py:49-52) and regenerates the same instance (instances.py); state, masks,
transitions, structural features and the tie-independent heuristics are computed on the GPU.
"""
import copy
import random
import warnings

import numpy as np
import torch

from .batch import STATE_ALL, BatchedGraphEnv
from .instances import generate_instance
from .utils import graph_from_obs

try:  # optional: the real gymnasium base class / spaces when they are installed
    import gymnasium as _gym
    _Base = _gym.Env
except Exception:  # pragma: no cover - gymnasium is absent in the build image
    _gym = None

    class _Base:  # minimal stand-in with the attributes user loops touch
        metadata = {}

        def close(self):
            pass


class _Discrete:
    def __init__(self, n):
        self.n = int(n)

    def contains(self, x):
        return 0 <= int(x) < self.n

    def sample(self):
        return int(np.random.randint(self.n))


class _Box:
    def __init__(self, low, high, shape):
        self.low, self.high, self.shape = low, high, tuple(shape)


_EVERY_STEP_HEURISTIC = ("LongestPath-v0", "DensestSubgraph-v0", "MulticastRouting-v0", "PerishableProductDelivery-v0")


class GraphEnv(_Base):
    def __init__(self, env_id, n_nodes, n_edges=-1, device=None, **kwargs):
        self.env_id = env_id
        self._ctor = (n_nodes, n_edges, device, dict(kwargs))
        self.core = BatchedGraphEnv(env_id, 1, n_nodes, n_edges, device=device, structural_features=True, **kwargs)
        c, P = self.core, self.core.params
        self.params = P
        self.n_nodes, self.n_edges = c.N, c.E
        self.is_eval_env = c.is_eval_env
        self.return_graph_obs = bool(P.get("return_graph_obs", False))
        # reference: Discrete(n_nodes) / Discrete(n_edges) (steiner_tree.py:43 -- E although actions range over 2E)
        n_act = c.E if c.spec.action_type == "edge" else c.N
        obs_shape = (c.obs_len,)
        if _gym is not None:
            self.action_space = _gym.spaces.Discrete(n_act)
            self.observation_space = _gym.spaces.Box(low=0, high=1000, shape=obs_shape)
        else:
            self.action_space = _Discrete(n_act)
            self.observation_space = _Box(0, 1000, obs_shape)
        self._heur_on_device = c.spec.heuristic_on_device(P)
        self._warned = False
        self.instance = None
        self._track = None

    def __deepcopy__(self, memo):
        """Branch this env: a new env with its own engine batch holding the same instance (ge_gather_instances) and the same
        state, env clock and statistics (ge_state_save / ge_state_load), plus deep copies of the host-side attributes.  The
        copy and the original then evolve independently."""
        new = type(self).__new__(type(self))
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            if k != "core":
                setattr(new, k, copy.deepcopy(v, memo))
        n_nodes, n_edges, device, kwargs = self._ctor
        new.core = BatchedGraphEnv(self.env_id, 1, n_nodes, n_edges, device=device, structural_features=True, **kwargs)
        if self.core.env_steps is not None:
            new.core.enable_env_clock()
        if self.core._loaded:
            new.core.gather_instances(self.core)
            new.core.load_states(self.core.save_states(), what=STATE_ALL)
        return new

    # ------------------------------------------------------------------ helpers
    def _obs(self):
        return self.core.obs_flat(0, 1)[0].cpu().numpy()

    def _mask(self):
        return self.core.mask[0].cpu().numpy().copy()

    def _heuristic(self):
        kind = self.env_id
        if kind == "DistributionCenter-v0":
            return -1                                              # distribution_center.py:91
        if not self.is_eval_env:
            return 0
        if kind == "DensestSubgraph-v0":
            return -1                                              # densest_subgraph.py:88
        if kind == "MaxIndependentSet-v0" and self.params["weighted"]:
            return -1                                              # max_independent_set.py:66-67
        if self._heur_on_device or self.instance.heuristic is not None:
            return float(self.core.t["heuristic"][0].item())   # device value, or a host value loaded with the instance
        if not self._warned:
            warnings.warn("%s: the reference's eval heuristic here (Kou / Christofides / Ramsey) is defined by networkx's set "
                          "iteration order and is not reproduced: heuristic_solution = nan; info['heuristic_device'] carries "
                          "the device-computed %s" % (kind, self.core.heuristic_device_name))
            self._warned = True
        return float("nan")

    # ------------------------------------------------------------------ gym API
    def reset(self, seed=None, options={}):
        if seed is not None:
            if _gym is not None:
                super().reset(seed=seed)
            random.seed(seed)
            np.random.seed(seed)
        c = self.core
        ins = generate_instance(self.env_id, self.params)
        self.instance = ins
        c.load_instances([ins], prepare=True)
        c.reset()
        self.src, self.dest, self.dests = ins.src, ins.dest, ins.dests
        self.start = 0
        self._track = [] if self.env_id in ("LongestPath-v0", "PerishableProductDelivery-v0") else set()
        self._head = ins.src
        info = {"mask": self._mask()}
        if self.env_id == "PerishableProductDelivery-v0":          # perishable_product_delivery.py:158-160
            P = self.params["n_products"]
            self.pickups, self.dropoffs = [int(x) for x in ins.dests[:P]], [int(x) for x in ins.dests[P:]]
            info["pickups"], info["dropoffs"], info["time_left"] = self.pickups, self.dropoffs, ins.max_distance
            self._head = 0
        obs = self._obs()
        if self.return_graph_obs:
            info["graph_obs"] = graph_from_obs(obs, self.env_id, c.N, c.E)
        return obs, info

    def step(self, action):
        c = self.core
        a = int(action)
        acts = torch.tensor([a], dtype=torch.int32, device=c.device)
        reward, done, binfo = c.step(acts)
        flags = c.flags[0].cpu().numpy()
        done_b, solved, status, has_mask = bool(flags[0]), int(np.int8(flags[1])), int(flags[2]), bool(flags[3])
        if status == 1:
            raise AssertionError("Action %d is not valid in the current state (mask is False / out of bounds)!" % a)
        if status == 2:
            raise AssertionError("step() called on a finished episode; call reset()")
        r = float(reward[0].item())
        sol = float(c.solution_cost[0].item())
        info = {}
        if has_mask:
            info["mask"] = self._mask()
        if solved >= 0:
            info["solved"] = bool(solved)
        if sol == sol:
            info["solution_cost"] = sol
        if done_b or self.env_id in _EVERY_STEP_HEURISTIC:
            info["heuristic_solution"] = self._heuristic()
            if self.is_eval_env and c.heuristic_device_name and not (self.env_id == "MaxIndependentSet-v0" and self.params["weighted"]):
                info["heuristic_device"] = float(c.t["heuristic_alt"][0].item())
                info["heuristic_device_name"] = c.heuristic_device_name
        if self.env_id == "LongestPath-v0":                        # longest_path.py:160,166
            self._track.append((self._head, a))
            info["edges_taken"] = self._track
            if has_mask:
                self._head = a
        elif self.env_id == "PerishableProductDelivery-v0":        # perishable_product_delivery.py:212,220,226
            info["edges_taken"] = self._track
            if has_mask or done_b:
                self._track.append((self._head, a))
                self._head = a
        elif self.env_id == "DensestSubgraph-v0":                  # densest_subgraph.py:151,193
            if a != c.N - 1:
                self._track.add(a)
            if done_b:
                info["nodes_taken"] = self._track
        obs = self._obs()
        if self.return_graph_obs:
            info["graph_obs"] = graph_from_obs(obs, self.env_id, c.N, c.E)
        return obs, r, done_b, False, info
