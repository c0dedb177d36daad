"""BatchedGraphEnv -- the batched vector-env entry point over the CUDA engine.

Per-env semantics are those of the reference's single-instance gymnasium envs
(graph_envs/<env>.py, see include/graphenvs_b200.h for the line map); B instances of one env
kind with uniform (n_nodes, n_edges) live on one GPU as CSR + SoA weights + packed bitsets.
All state tensors are torch tensors on the device and are exposed as zero-copy views.
"""
import ctypes as C
import math

import numpy as np
import torch

from . import _native
from .spec import ENV_SPECS, check_ctor_args

PREP_HEURISTIC, PREP_MAXDIST, PREP_INRANGE, PREP_ALT_HEURISTIC, PREP_DC_EDGES = 1, 2, 4, 8, 16
STATE_DYNAMIC, STATE_CLOCK, STATE_STATS, STATE_ALL = (_native.STATE_DYNAMIC, _native.STATE_CLOCK, _native.STATE_STATS,
                                                      _native.STATE_ALL)
# the state arrays of a record (include/graphenvs_b200.h, GE_STATE_*): dynamic, clock, stats
_STATE_ARRAYS = ("head", "node_bits", "node_bits2", "edge_bits", "dist32", "bestkey", "cost", "counters", "done", "mask_bits",
                 "mask_cnt", "env_steps", "acc", "traj")


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class EnvStates:
    """Saved per-env states (BatchedGraphEnv.save_states): `data` is a uint8 [n, record_bytes] device tensor of opaque records
    (ge_state_save), `signature` the env id, shape and set of state arrays a batch must have to load them."""

    def __init__(self, data, signature):
        self.data, self.signature = data, signature

    def __len__(self):
        return self.data.shape[0]


class BatchedGraphEnv:
    def __init__(self, env_id, num_envs, n_nodes, n_edges=-1, *, device=None, byte_mask=True, auto_reset=False,
                 structural_features=False, env_id0=0, keep_w64=True, force_warp=False, **kwargs):
        self.lib = _native.lib()  # raises when the CUDA library is absent -- no fallback
        if not torch.cuda.is_available():
            raise _native.NativeError("graphenvs_b200 needs a CUDA device (sm_100a); there is no CPU path")
        self.spec = ENV_SPECS[env_id]
        self.env_id = env_id
        self.params = check_ctor_args(env_id, n_nodes, n_edges, kwargs)  # reference ctor rules
        P = self.params
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self.B, self.N, self.E = int(num_envs), int(P["n_nodes"]), int(P["n_edges"])
        self.M = 2 * self.E
        self.is_eval_env = bool(P.get("is_eval_env", False))
        self.structural_features = bool(structural_features)
        d = _native.GeBatch()
        d.kind, d.B, d.N, d.M = self.spec.kind, self.B, self.N, self.M
        d.parenting = int(P.get("parenting", -1))
        d.n_dests = int(P.get("n_dests", P.get("n_products", 0)))     # PerishableProductDelivery: products
        d.n_choices = int(P.get("n_choices", 0))
        d.n_targets = int(P.get("target_count", 0)) if env_id != "PerishableProductDelivery-v0" else 2 * int(P["n_products"])
        d.flags = ((1 if auto_reset else 0) | (2 if env_id == "TSP-v0" else 0) | (0 if P.get("weighted", True) else 4)
                   | (8 if force_warp else 0))
        d.env_id0 = int(env_id0)
        d.max_distance = float(P.get("max_distance", 0.0)) if env_id == "DistributionCenter-v0" else 0.0
        _native.check(self.lib.ge_fill_layout(C.byref(d)))
        self.desc = d
        self.F = self.spec.node_f + 5
        self.Fe = self.spec.edge_f
        self.obs_len = self.N * self.F + self.M * self.Fe + 2 * self.M

        dev, B, N = self.device, self.B, self.N
        z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)  # noqa: E731
        self.t = {}
        T = self.t
        T["row_ptr"] = z((B, d.RP), torch.int32)
        T["col"] = z((B, d.MP), torch.int32)
        if self.spec.step_w == "f32":
            T["w32"] = z((B, d.MP), torch.float32)
        if self.spec.step_w == "f64" or (keep_w64 and self.spec.step_w == "f32"):
            T["w64"] = z((B, d.MP), torch.float64)
        if self.spec.uses_adj:
            B32 = (B + 31) // 32 * 32                             # whole tiles of 32 envs for the N <= 64 layout
            self._adj_store = z((B32 * d.ADJS,), torch.int32)
            T["adj_bits"] = self._adj_store
            if env_id == "PerishableProductDelivery-v0" and (N > 64 or force_warp):
                pass                                                  # warp-per-env kernel: looks its one edge weight up in the CSR row
            elif N <= 64 and self.spec.step_w == "f64":
                T["wmat"] = z((B, N, N), torch.float64)              # dense fp64 weights for the lane-per-env kernels
            elif self.spec.step_w == "f64":
                T["wsort"] = z((B, d.MP), torch.float64)             # destination-sorted weights: O(1) adj[u, v] by bit rank
        par = int(P.get("parenting", -1))
        if not force_warp:   # derived / state arrays of the incremental-mask kernels (csrc/ge_incr.cu)
            if env_id == "SteinerTree-v0" or (env_id == "MulticastRouting-v0" and par == 2):
                T["rev"] = z((B, d.MP), torch.int32)
            if env_id == "MulticastRouting-v0" and par == 2:
                T["esrc"] = z((B, d.MP), torch.int32)
            if env_id == "MulticastRouting-v0" and par >= 3:
                T["bestkey"] = z((B, N), torch.int64)
            if (env_id == "SteinerTree-v0" or (env_id == "MulticastRouting-v0" and par >= 2)) and d.AW > 64 and d.NW > 8:
                T["mask_cnt"] = z((B, 8), torch.int32)                 # chunk popcounts of the packed mask for the in-kernel sampler
        if env_id == "DistributionCenter-v0":
            T["wmin"] = z((B,), torch.float64)
        T["src"] = z((B,), torch.int32)
        T["dest"] = z((B,), torch.int32)
        if self.spec.has_targets:
            T["target_bits"] = z((B, d.NW), torch.int32)
        if self.spec.has_node_cost:
            T["node_cost"] = z((B, N), torch.float32)
        if P.get("spatial"):
            T["node_xy"] = z((B, N, 2), torch.float32)
        if env_id == "MulticastRouting-v0":
            T["max_dist32"] = z((B,), torch.float32)
            T["edge_bits"] = z((B, d.MW), torch.int32)
            T["dist32"] = z((B, N), torch.float32)
        if env_id == "PerishableProductDelivery-v0":
            T["max_dist32"] = z((B,), torch.float32)                 # delivery time (the TIME_LEFT columns)
            T["targets"] = z((B, d.n_targets), torch.int32)           # pickups, then dropoffs
        if env_id == "DistributionCenter-v0":
            T["targets"] = z((B, max(d.n_targets, 1)), torch.int32)
            T["in_range"] = z((B, max(d.n_targets, 1), d.NW), torch.int32)
        T["heuristic"] = z((B,), torch.float64)
        self.heuristic_device_name = None
        if self.is_eval_env:
            self.heuristic_device_name = self.spec.heuristic_alternative(P)
            if self.heuristic_device_name:
                T["heuristic_alt"] = z((B,), torch.float64)
        if self.structural_features:
            T["features"] = z((B, N, 5), torch.float32)
        T["head"] = z((B,), torch.int32)
        T["node_bits"] = z((B, d.NW), torch.int32)
        if env_id in ("DistributionCenter-v0", "DensestSubgraph-v0"):
            T["node_bits2"] = z((B, d.NW), torch.int32)
        T["cost"] = z((B,), torch.float64)
        T["counters"] = z((B, 4), torch.int32)
        T["done"] = z((B,), torch.uint8)
        # step outputs + packed mask live back to back in one block => one D2H copy in ge_step_host
        Bp = (B + 3) & ~3                                     # every section of the block starts 16-byte aligned (128-bit copies)
        self._io = z((16 * Bp + 4 * B * d.AW,), torch.uint8)
        self._io_layout = (Bp, 16 * Bp + 4 * B * d.AW)
        T["mask_bits"] = self._io[16 * Bp:].view(torch.int32).view(B, d.AW)
        if byte_mask:
            T["mask_bytes"] = z((B, d.AP), torch.uint8)
        if auto_reset and self.spec.action_type == "node":
            T["mask0_bits"] = z((B, d.AW), torch.int32)     # reset-time mask, reused by auto-reset (lane / group kernels)
        T["acc"] = z((4, B), torch.float64)                      # component-major: one stream per statistic
        T["traj"] = z((B,), torch.int64)
        self.env_steps = None   # enable_env_clock(): per-env step counts feeding the samplers (CUDA-graph replays)
        # step outputs
        self.reward = self._io[:4 * B].view(torch.float32)
        self.flags = self._io[4 * Bp:4 * Bp + 4 * B].view(B, 4)
        self.solution_cost = self._io[8 * Bp:8 * Bp + 8 * B].view(torch.float64)
        self.actions_dev = z((B,), torch.int32)
        self._stats = z((4,), torch.float64)
        self._sync_desc()
        self._out = _native.StepOut(_ptr(self.reward), _ptr(self.flags), _ptr(self.solution_cost))
        self._loaded = False

    def like(self, num_envs, **overrides):
        """A new batch of `num_envs` envs, nothing loaded yet, with this batch's env id, parameters and engine options (device,
        byte_mask, auto_reset, structural_features, env_id0, keep_w64, force_warp); `overrides` replace
        any of them.  Fill it with gather_instances(), e.g. the wide batch of a multi-start decoder."""
        P = {k: v for k, v in self.params.items() if k in dict(self.spec.defaults)}   # ctor kwargs only, not derived values
        P.pop("structural_features", None)          # ShortestPath's ignored ctor kwarg (shortest_path.py:23) vs the engine's own flag
        n_nodes, n_edges = self.params["n_nodes"], self.params["n_edges"]
        d = self.desc
        opts = dict(device=self.device, byte_mask="mask_bytes" in self.t, auto_reset=bool(d.flags & 1),
                    structural_features=self.structural_features, env_id0=d.env_id0, keep_w64="w64" in self.t,
                    force_warp=bool(d.flags & 8))
        opts.update(P)
        opts.update(overrides)
        return BatchedGraphEnv(self.env_id, num_envs, n_nodes, n_edges, **opts)

    # ------------------------------------------------------------------ plumbing
    def _sync_desc(self):
        for name in ("row_ptr", "col", "w32", "w64", "adj_bits", "rev", "esrc", "bestkey", "wsort", "wcode", "dfa", "dc_edges", "dc_rows", "wmin", "wmat", "src", "dest", "target_bits", "node_cost", "node_xy",
                     "max_dist32", "targets", "in_range", "heuristic", "heuristic_alt", "features", "head", "node_bits", "node_bits2",
                     "edge_bits", "dist32", "cost", "counters", "done", "mask_bits", "mask_cnt", "mask_bytes", "mask0_bits", "acc", "traj"):
            t = self.t.get(name)
            setattr(self.desc, name, t.data_ptr() if t is not None else None)

    def enable_env_clock(self):
        """Per-env step counters: ge_step increments them and the samplers add them to `t`, so a
        captured CUDA graph (frozen kernel arguments) draws fresh actions on every replay."""
        if self.env_steps is None:
            self.env_steps = torch.zeros((self.B,), dtype=torch.int32, device=self.device)
            self.desc.env_steps = self.env_steps.data_ptr()
        return self.env_steps

    def enable_pdl(self, on=True):
        """GE_FLAG_PDL (include/graphenvs_b200.h): step launches may start under the tail of the previous launch of the stream
        and prefetch static instance data; valid while the preceding work in the stream is another step or a save_states() /
        load_states() (not generate() / finalize_graphs() / gather_instances() / an InstancePool refill, which rewrite static
        arrays)."""
        self.desc.flags = (self.desc.flags | 16) if on else (self.desc.flags & ~16)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def memory_bytes(self):
        return sum(t.numel() * t.element_size() for t in self.t.values())

    def release_w64(self):
        """Drop the float64 weights of kinds that step in float32 (after prepare)."""
        if self.spec.step_w == "f32" and "w64" in self.t:
            del self.t["w64"]
            self._sync_desc()

    # ------------------------------------------------------------------ instance loading
    def load_instances(self, instances, prepare=True):
        """instances: list of B `Instance`s (graphenvs_b200.instances) -- host data, reference edge order."""
        assert len(instances) == self.B, "need exactly num_envs instances"
        d, B, N, M = self.desc, self.B, self.N, self.M
        row_ptr = np.zeros((B, d.RP), np.int32)
        col = np.zeros((B, d.MP), np.int32)
        w64 = np.zeros((B, d.MP), np.float64)
        src = np.zeros(B, np.int32)
        dest = np.zeros(B, np.int32)
        tbits = np.zeros((B, d.NW), np.uint32)
        ncost = np.zeros((B, N), np.float32)
        nxy = np.zeros((B, N, 2), np.float32)
        maxd = np.zeros(B, np.float32)
        targets = np.zeros((B, max(d.n_targets, 1)), np.int32)
        heur = np.zeros(B, np.float64)
        have_heur = True
        for b, ins in enumerate(instances):
            links = np.asarray(ins.links, dtype=np.int64).reshape(-1, 2)
            assert ins.n_nodes == N and links.shape[0] == M, "instance shape mismatch"
            s = links[:, 0]
            assert np.all(s[1:] >= s[:-1]), "edge_links must be source-sorted (reference order)"
            row_ptr[b, 1:N + 1] = np.cumsum(np.bincount(s, minlength=N))
            if self.spec.action_type == "edge":
                assert np.all(np.diff(row_ptr[b, :N + 1]) > 0), "edge-action envs need every node to have degree >= 1"
            col[b, :M] = links[:, 1]
            w64[b, :M] = ins.w64
            src[b], dest[b] = ins.src, ins.dest
            if self.spec.has_targets and ins.dests is not None:
                for t in np.asarray(ins.dests).ravel():
                    tbits[b, t >> 5] |= np.uint32(1 << (int(t) & 31))
                if self.env_id == "DistributionCenter-v0":
                    tl = np.asarray(ins.dests, dtype=np.int32).ravel()
                    assert tl.shape[0] == d.n_targets
                    targets[b, :d.n_targets] = tl
            if self.env_id == "PerishableProductDelivery-v0":
                tl = np.asarray(ins.dests, dtype=np.int32).ravel()
                assert tl.shape[0] == d.n_targets
                targets[b, :d.n_targets] = tl
            if ins.node_cost is not None:
                ncost[b] = np.asarray(ins.node_cost, dtype=np.float64).astype(np.float32)
            if ins.node_xy is not None:
                nxy[b] = np.asarray(ins.node_xy, dtype=np.float64).astype(np.float32)
            if ins.max_distance is not None:
                maxd[b] = np.float32(ins.max_distance)
            if ins.heuristic is None:
                have_heur = False
            else:
                heur[b] = ins.heuristic
        T, dev = self.t, self.device
        up = lambda a: torch.from_numpy(a).to(dev)  # noqa: E731
        T["row_ptr"].copy_(up(row_ptr))
        T["col"].copy_(up(col))
        if "w64" in T:
            T["w64"].copy_(up(w64))
        if "w32" in T:
            T["w32"].copy_(up(w64.astype(np.float32)))
        T["src"].copy_(up(src))
        T["dest"].copy_(up(dest))
        if "target_bits" in T:
            T["target_bits"].copy_(up(tbits.view(np.int32)))
        if "node_cost" in T:
            T["node_cost"].copy_(up(ncost))
        if "node_xy" in T:
            T["node_xy"].copy_(up(nxy))
        if "max_dist32" in T:
            T["max_dist32"].copy_(up(maxd))
        if "targets" in T:
            T["targets"].copy_(up(targets))
        if have_heur:
            T["heuristic"].copy_(up(heur))
        feats = [ins.features for ins in instances]
        if self.structural_features and all(f is not None for f in feats):
            T["features"].copy_(up(np.stack([np.asarray(f, dtype=np.float32) for f in feats])))
            self._features_loaded = True
        else:
            self._features_loaded = False
        u01 = None
        if self.env_id == "MulticastRouting-v0" and all(i.max_distance is None and i.u01 is not None for i in instances):
            u01 = up(np.array([i.u01 for i in instances], dtype=np.float64))  # multicast_routing.py:103 draw
        self.finalize_graphs(prepare=prepare, heuristics=self.is_eval_env and not have_heur, u01=u01)

    def finalize_graphs(self, prepare=True, heuristics=False, u01=None, features=None, maxdist_from_generator=False):
        """Derived static data after the CSR arrays are in place (load_instances / generate)."""
        L, d = self.lib, self.desc
        if self.spec.uses_adj or "rev" in self.t or "esrc" in self.t or "wmin" in self.t:
            _native.check(L.ge_build_adjacency(C.byref(d), self._stream()))
        if self.env_id == "DistributionCenter-v0" and not (d.flags & 8):
            self._build_distance_automaton()
        what = 0
        if prepare and self.env_id == "DistributionCenter-v0" and d.parenting == 2:
            what |= PREP_INRANGE
        if "dc_edges" in self.t:
            what |= PREP_DC_EDGES
        if heuristics and self.spec.heuristic_on_device(self.params):
            what |= PREP_HEURISTIC
        if self.is_eval_env and "heuristic_alt" in self.t and ("w64" in self.t or self.env_id == "MaxIndependentSet-v0"):
            what |= PREP_ALT_HEURISTIC
        if (u01 is not None or maxdist_from_generator) and self.env_id == "MulticastRouting-v0":
            what |= PREP_MAXDIST
        if what:
            _native.check(L.ge_prepare(C.byref(d), what, _ptr(u01), self._stream()))
        if features is None:
            features = self.structural_features and not getattr(self, "_features_loaded", False)
        if features:
            _native.check(L.ge_features(C.byref(d), self._stream()))
        self._loaded = True

    def _build_distance_automaton(self):
        """Exact fp64 distance automaton for the cutoff SSSP (include/graphenvs_b200.h: ge_batch.dfa).  Applies when
        every edge weight of the batch is one of <= 15 distinct doubles (k/10 in the reference) and the closure of
        left-fold sums within the cutoff has < 255 values; otherwise the fp64 search stays in charge."""
        T, d, B, M = self.t, self.desc, self.B, self.M
        for k in ("wcode", "dfa", "dc_edges", "dc_rows"):
            T.pop(k, None)
        self._sync_desc()
        self.desc.dfa_bytes = 0
        w = T.get("w64")
        if w is None or M == 0:
            return False
        ws_t = torch.unique(w[:min(B, 1024), :M])                     # ascending; verified against every edge below
        if ws_t.numel() == 0 or ws_t.numel() > 15:
            return False
        ws = [float(x) for x in ws_t.cpu().numpy()]                    # python floats = IEEE doubles, same adds as DADD
        cutoff = float(d.max_distance)
        states, frontier = {0.0}, [0.0]
        while frontier:
            s = frontier.pop()
            for x in ws:
                t = s + x
                if t <= cutoff and t not in states:
                    states.add(t)
                    frontier.append(t)
                    if len(states) > 254:
                        return False
        st = sorted(states)
        idx = {v: i for i, v in enumerate(st)}
        S, W = len(st), len(ws)
        tab = np.full((S, W), 255, dtype=np.uint8)
        for i, s in enumerate(st):
            for j, x in enumerate(ws):
                if s + x <= cutoff:
                    tab[i, j] = idx[s + x]
        expand = np.array([1 if s + ws[0] <= cutoff else 0 for s in st], dtype=np.uint8)
        cmax = np.array([max([j for j in range(W) if tab[i, j] != 255], default=255) for i in range(S)], dtype=np.uint8)
        for i in range(S):          # fl(value + weight) is monotone in the weight: the usable codes of a state are a prefix
            assert all(tab[i, j] != 255 for j in range(0 if cmax[i] == 255 else cmax[i] + 1))
        code = torch.zeros((B, d.MP), dtype=torch.uint8, device=self.device)
        step = max(1, (64 << 20) // max(M, 1))
        for lo in range(0, B, step):
            seg = w[lo:lo + step, :M]
            c = torch.searchsorted(ws_t, seg).clamp_(max=W - 1)
            if not bool((ws_t[c] == seg).all()):
                return False                                           # a weight outside the sampled set: keep fp64
            code[lo:lo + step, :M] = c.to(torch.uint8)
        T["wcode"] = code
        T["dfa"] = torch.from_numpy(np.concatenate([np.array([S, W], dtype=np.uint8), tab.ravel(), expand, cmax])).to(self.device)
        if self.N <= 1024 and self.N < 65536:
            T["dc_edges"] = torch.zeros((B, d.MP), dtype=torch.int32, device=self.device)   # weight-sorted rows for csrc/ge_dc.cu
            T["dc_rows"] = torch.zeros((B, self.N, 32), dtype=torch.int32, device=self.device)  # their first 32 entries at a fixed 128-byte stride (64 KB per env at N=500)
        self._sync_desc()
        self.desc.dfa_bytes = int(T["dfa"].numel())
        return True

    def export_instances(self, env_lo=0, count=None):
        """Host copies of `count` resident instances as `Instance`s (reference edge-order contract)."""
        from .instances import Instance
        count = self.B - env_lo if count is None else count
        sl = slice(env_lo, env_lo + count)
        T, N, M, d = self.t, self.N, self.M, self.desc
        g = lambda k: T[k][sl].cpu().numpy() if k in T else None  # noqa: E731
        rp, col = g("row_ptr"), g("col")
        w = g("w64") if "w64" in T else (g("w32").astype(np.float64) if "w32" in T else np.ones((count, d.MP)))
        src, dest, heur = g("src"), g("dest"), g("heuristic")
        tb, nc, xy, md, tg = g("target_bits"), g("node_cost"), g("node_xy"), g("max_dist32"), g("targets")
        out = []
        for i in range(count):
            deg = np.diff(rp[i, :N + 1])
            links = np.stack([np.repeat(np.arange(N, dtype=np.int32), deg), col[i, :M]], axis=1).astype(np.int32)
            ins = Instance(n_nodes=N, links=links, w64=w[i, :M].astype(np.float64), src=int(src[i]), dest=int(dest[i]),
                           heuristic=float(heur[i]))
            if self.env_id in ("DistributionCenter-v0", "PerishableProductDelivery-v0"):
                ins.dests = tg[i, :d.n_targets].astype(np.int32)
            elif tb is not None:
                bits = np.unpackbits(tb[i].view(np.uint8), bitorder="little")[:N]
                ins.dests = np.flatnonzero(bits).astype(np.int32)
            if nc is not None:
                ins.node_cost = nc[i].astype(np.float64)
            if xy is not None:
                ins.node_xy = xy[i].astype(np.float64)
            if md is not None:
                ins.max_distance = float(md[i])
            out.append(ins)
        return out

    def adjacency_rows(self):
        """uint32-as-int32 [B, N, NW] view/copy of the adjacency bit-matrix in env-major order, whatever the
        device layout (include/graphenvs_b200.h: tiles of 32 envs for the lane-per-env family)."""
        d, B, N = self.desc, self.B, self.N
        a = self.t["adj_bits"]
        tiled = N <= 64 and self.env_id in ("ShortestPath-v0", "LongestPath-v0", "TSP-v0", "MaxIndependentSet-v0",
                                            "DensestSubgraph-v0") and not (d.flags & 8)
        if tiled:
            nt = (B + 31) // 32
            return a[:nt * N * 32 * d.NW].view(nt, N, 32, d.NW).permute(0, 2, 1, 3).reshape(nt * 32, N, d.NW)[:B]
        return a[:B * d.ADJS].view(B, d.ADJS)[:, :N * d.NW].view(B, N, d.NW)

    def generate(self, seed=0, check=True):
        """Device-side instance generation (distribution parity with the reference's reset()).  check=True reads back how
        many envs needed the connected-by-construction fallback (one stream sync) into self.generate_fallbacks."""
        L, d, T = self.lib, self.desc, self.t
        w64 = T.get("w64")
        tmp64 = None
        if w64 is None:
            tmp64 = torch.zeros((self.B, d.MP), dtype=torch.float64, device=self.device)
            w64 = tmp64
            d.w64 = w64.data_ptr()
        _native.check(L.ge_generate(C.byref(d), int(seed), _ptr(T["row_ptr"]), _ptr(T["col"]), _ptr(w64),
                                    _ptr(T.get("w32")), self._stream()))
        # Multicast: the max_distance uniform (multicast_routing.py:103) is drawn by the generator per GLOBAL env id, so a
        # rank-sliced batch gets the same distances as the single-GPU batch (ge_prepare reads it from max_dist32)
        self.finalize_graphs(prepare=True, heuristics=self.is_eval_env, maxdist_from_generator=self.env_id == "MulticastRouting-v0")
        if tmp64 is not None:
            torch.cuda.current_stream(self.device).synchronize()
            self._sync_desc()
        if check:
            n = int(L.ge_generate_fallbacks(self._stream()))
            if n < 0:
                _native.check(n)
            self.generate_fallbacks = n
            if n:
                import warnings
                warnings.warn("ge_generate: %d of %d envs found no connected G(n=%d, m=%d) in 4096 draws and were emitted "
                              "connected-by-construction (random tree / ring + random edges)" % (n, self.B, self.N, self.E))

    # ------------------------------------------------------------------ hot path
    def reset(self, select=None):
        """State init + first mask for all envs (or those with select[b] != 0)."""
        assert self._loaded, "load_instances() or generate() first"
        sel = None
        if select is not None:
            sel = select.to(device=self.device, dtype=torch.uint8).contiguous()
        _native.check(self.lib.ge_reset(C.byref(self.desc), _ptr(sel), self._stream()))
        return self.info()

    def step(self, actions):
        """actions: int32[B] on the device.  Returns (reward f32[B], done bool[B], info)."""
        if actions.dtype != torch.int32 or actions.device != self.device or not actions.is_contiguous():
            actions = actions.to(device=self.device, dtype=torch.int32).contiguous()
        _native.check(self.lib.ge_step(C.byref(self.desc), _ptr(actions), C.byref(self._out), self._stream()))
        return self.reward, self.flags[:, 0].bool(), self.info(step=True)

    def step_async(self, actions):
        """Same as step() without building the info dict (bench / rollout loops)."""
        _native.check(self.lib.ge_step(C.byref(self.desc), _ptr(actions), C.byref(self._out), self._stream()))

    def step_sampled(self, seed, t, out=None):
        """Random-rollout step: uniform valid action drawn in-kernel + step, one launch.  Results as step_async."""
        out = self.actions_dev if out is None else out
        _native.check(self.lib.ge_step_sampled(C.byref(self.desc), int(seed), int(t), _ptr(out), C.byref(self._out),
                                               self._stream()))
        return out

    def sample_actions(self, seed, t, out=None):
        out = self.actions_dev if out is None else out
        _native.check(self.lib.ge_sample_actions(C.byref(self.desc), int(seed), int(t), _ptr(out), self._stream()))
        return out

    def sample_logits(self, logits, seed, t, greedy=False, out=None):
        """Policy-driven action draw (ge_sample_logits): a categorical over the valid actions of the current packed mask.

        logits: CUDA [B, A] float32 / bfloat16 on this batch's device (made contiguous).  greedy=False draws by Gumbel-max with
        counter-based noise of (seed, global env id, t + env clock, action); greedy=True takes the argmax (lowest index on
        ties).  Returns (actions int32[B], log_prob f32[B], entropy f32[B]); actions default to self.actions_dev, `out` =
        (actions, log_prob, entropy) preallocated tensors.  Follow with step(actions) / step_async(actions).  Empty mask rows
        give (-1, 0, 0).  The log_prob / entropy equal policy.masked_log_prob's on the same inputs bit for bit."""
        from .policy import _DTYPES
        if not isinstance(logits, torch.Tensor) or logits.device != self.device:
            raise ValueError("sample_logits: logits must be a tensor on %s" % self.device)
        if logits.dtype not in _DTYPES:
            raise TypeError("sample_logits: logits must be float32 or bfloat16, got %s" % logits.dtype)
        if tuple(logits.shape) != (self.B, self.desc.A):
            raise ValueError("sample_logits: logits shape %s, expected (%d, %d)" % (tuple(logits.shape), self.B, self.desc.A))
        logits = logits.detach().contiguous()
        if out is None:
            acts = self.actions_dev
            lp = torch.empty((self.B,), dtype=torch.float32, device=self.device)
            ent = torch.empty((self.B,), dtype=torch.float32, device=self.device)
        else:
            acts, lp, ent = out
        _native.check(self.lib.ge_sample_logits(C.byref(self.desc), _ptr(logits), _DTYPES[logits.dtype], int(bool(greedy)), int(seed),
                                                int(t), _ptr(acts), _ptr(lp), _ptr(ent), self._stream()))
        return acts, lp, ent

    def host_io(self):
        """Pinned host mirror of the device output block: (block, reward, flags, solution_cost, mask_bits) views."""
        Bp, nbytes = self._io_layout
        B, AW = self.B, self.desc.AW
        blk = torch.zeros((nbytes,), dtype=torch.uint8).pin_memory()
        return (blk, blk[:4 * B].view(torch.float32), blk[4 * Bp:4 * Bp + 4 * B].view(B, 4),
                blk[8 * Bp:8 * Bp + 8 * B].view(torch.float64), blk[16 * Bp:].view(torch.int32).view(B, AW))

    def host_io_compact(self):
        """Pinned host buffers of the COMPACT result format (ge_step_host_compact): reward f32[B], flags8 u8[B], solution_cost f32[B],
        mask_bits i32[B, AW].  unpack_flags8() decodes the flag byte."""
        B, AW = self.B, self.desc.AW
        return (torch.zeros(B, dtype=torch.float32).pin_memory(), torch.zeros(B, dtype=torch.uint8).pin_memory(),
                torch.zeros(B, dtype=torch.float32).pin_memory(), torch.zeros((B, AW), dtype=torch.int32).pin_memory())

    @staticmethod
    def unpack_flags8(f8):
        """flags8 -> (done bool, solved int8 in {-1, 0, 1}, status uint8, has_mask bool); include/graphenvs_b200.h: GE_FLAGS8_*."""
        f = f8.numpy() if isinstance(f8, torch.Tensor) else np.asarray(f8)
        return (f & 1).astype(bool), (((f >> 1) & 3).astype(np.int8) - 1), ((f >> 3) & 3).astype(np.uint8), ((f >> 5) & 1).astype(bool)

    def host_stepper(self, h_actions, h_reward, h_flags, h_cost, h_mask=None, h_mask_bits=None, stream=None, pipelined=False,
                     chunks=4, obs_x=None, compact=False):
        """Zero-argument callable = step_host on FIXED pinned buffers, arguments marshalled once.  On a
        non-default stream the C side replays the whole copy-in / step / copy-out sequence as one CUDA graph.
        pipelined=True: ge_step_host_pipelined -- the batch is stepped in `chunks` slices on parallel graph branches,
        slice i's results cross PCIe while slice i+1 steps (needs a created stream; the byte mask is not returned).  chunks=0: ONE step
        kernel + a concurrent write-back kernel fed by per-1024-env progress counters (multi-wave batches: 387 vs 486 us per host step at
        1M cfg2 envs; no gain for one-wave batches); chunks=None picks between the two."""
        st = stream if stream is not None else torch.cuda.current_stream(self.device)
        if chunks is None:   # auto: batches of several waves whose kernel signals progress stream their results (chunks = 0), the rest use two slices
            wave = 148 * 16 * 32 if self.N <= 64 else 148 * 6 * 8          # envs resident at once: lane-per-env tiles / DistributionCenter warps
            chunks = 0 if (self.B >= 4 * wave and self.lib.ge_progress_supported(C.byref(self.desc))) else 2
        # obs_x: float32[B, N, F] on the device -- the pipelined step also rewrites the observation's node columns, slice by
        # slice on its write-back lane (ge_batch.obs_x); None switches that off again
        assert obs_x is None or (pipelined and obs_x.is_cuda and obs_x.dtype == torch.float32 and obs_x.is_contiguous()
                                 and obs_x.numel() == self.B * self.N * self.F)
        self.desc.obs_x = obs_x.data_ptr() if obs_x is not None else None
        if compact:   # flags as one byte per env, solution_cost as float32 (host_io_compact() buffers)
            assert pipelined and st.cuda_stream != 0 and h_mask is None and h_flags.dtype == torch.uint8 and h_cost.dtype == torch.float32
        if pipelined and st.cuda_stream != 0 and h_mask is None:
            args = (C.byref(self.desc), _ptr(h_actions), C.byref(self._out), _ptr(h_reward), _ptr(h_flags),
                    _ptr(h_cost), _ptr(h_mask_bits), int(chunks), C.c_void_p(st.cuda_stream))
            fn = self.lib.ge_step_host_compact if compact else self.lib.ge_step_host_pipelined
        else:
            args = (C.byref(self.desc), _ptr(h_actions), _ptr(self.actions_dev), C.byref(self._out), _ptr(h_reward), _ptr(h_flags),
                    _ptr(h_cost), _ptr(h_mask), _ptr(h_mask_bits), C.c_void_p(st.cuda_stream))
            fn = self.lib.ge_step_host
        check = _native.check
        keep = (h_actions, h_reward, h_flags, h_cost, h_mask, h_mask_bits, st, obs_x)

        def call():
            check(fn(*args))
        call._keep = keep
        call.chunks = int(chunks)
        return call

    def step_host(self, h_actions, h_reward, h_flags, h_cost, h_mask=None, h_mask_bits=None):
        """End-to-end C-ABI call with HOST (pinned) buffers: H2D actions, step, D2H results, sync."""
        _native.check(self.lib.ge_step_host(C.byref(self.desc), _ptr(h_actions), _ptr(self.actions_dev),
                                            C.byref(self._out), _ptr(h_reward), _ptr(h_flags), _ptr(h_cost),
                                            _ptr(h_mask), _ptr(h_mask_bits), self._stream()))

    def step_kernel_name(self, sampled=False):
        """Name of the CUDA kernel ge_step (ge_step_sampled) dispatches this batch to."""
        return self.lib.ge_step_kernel_name(C.byref(self.desc), int(bool(sampled))).decode()

    def slice_desc(self, lo, count):
        """C descriptor of the sub-batch [lo, lo+count) (ge_batch_slice): same memory, steppable on its own."""
        out = _native.GeBatch()
        _native.check(self.lib.ge_batch_slice(C.byref(self.desc), int(lo), int(count), C.byref(out)))
        return out

    def __del__(self):
        try:
            self.lib.ge_step_host_release(C.byref(self.desc))   # cached CUDA graphs reference this batch's memory
        except Exception:
            pass

    def info(self, step=False):
        d = {"mask": self.mask, "mask_bits": self.t["mask_bits"], "heuristic_solution": self.t["heuristic"]}
        if self.heuristic_device_name:      # labelled alternative (Kou / Christofides / Ramsey are defined by networkx's iteration order)
            d["heuristic_device"] = self.t["heuristic_alt"]
            d["heuristic_device_name"] = self.heuristic_device_name
        if step:
            f = self.flags
            d.update(solved=f[:, 1].view(torch.int8), status=f[:, 2], has_mask=f[:, 3].bool(),
                     solution_cost=self.solution_cost)
        return d

    @property
    def mask(self):
        """bool[B, A] view of the current valid-action masks (None when byte_mask=False).  For the lane-per-env kinds
        (N <= 64: ShortestPath, LongestPath, TSP, MaxIndependentSet, DensestSubgraph) and the incremental-mask kinds
        (SteinerTree, Multicast parenting >= 2, MaxIndependentSet N > 64) the step kernels keep only the packed mask
        current and this property expands it into the byte view first (ge_mask_bytes, one coalesced pass)."""
        mb = self.t.get("mask_bytes")
        if mb is None:
            return None
        if not self.lib.ge_mask_bytes_current(C.byref(self.desc)):
            _native.check(self.lib.ge_mask_bytes(C.byref(self.desc), 0, self.B, self._stream()))
        return mb[:, :self.desc.A].view(torch.bool)

    def obs_flat(self, env_lo=0, count=None):
        """Reference wire format (utils.vectorize_graph): float32[count, obs_len]."""
        count = self.B - env_lo if count is None else count
        out = torch.empty((count, self.obs_len), dtype=torch.float32, device=self.device)
        _native.check(self.lib.ge_obs_flat(C.byref(self.desc), int(env_lo), int(count), _ptr(out), self._stream()))
        return out

    def obs_graph(self, env_lo=0, count=None):
        """(x [count,N,F] f32, edge_features [count,2E,Fe] f32, edge_index [count,2E,2] int64) on the device:
        utils.devectorize_graph of the flat observation without materialising it (GNN / PyG consumers)."""
        count = self.B - env_lo if count is None else count
        x = torch.empty((count, self.N, self.F), dtype=torch.float32, device=self.device)
        ea = torch.empty((count, self.M, self.Fe), dtype=torch.float32, device=self.device)
        ei = torch.empty((count, self.M, 2), dtype=torch.int64, device=self.device)
        _native.check(self.lib.ge_obs_graph(C.byref(self.desc), int(env_lo), int(count), _ptr(x), _ptr(ea), _ptr(ei), self._stream()))
        return x, ea, ei

    def obs_nodes(self, env_lo=0, count=None, out=None):
        """x float32[count, N, F] only: the node columns are the part of the observation a step changes."""
        count = self.B - env_lo if count is None else count
        if out is None:
            out = torch.empty((count, self.N, self.F), dtype=torch.float32, device=self.device)
        _native.check(self.lib.ge_obs_nodes(C.byref(self.desc), int(env_lo), int(count), _ptr(out), self._stream()))
        return out

    def compute_features(self):
        if "features" not in self.t:
            self.t["features"] = torch.zeros((self.B, self.N, 5), dtype=torch.float32, device=self.device)
            self.structural_features = True
            self._sync_desc()
        _native.check(self.lib.ge_features(C.byref(self.desc), self._stream()))
        return self.t["features"]

    def stats(self):
        """Device-side reduction of the per-env accumulators: episodes, solved, sum reward, sum final cost."""
        _native.check(self.lib.ge_stats(C.byref(self.desc), _ptr(self._stats), self._stream()))
        return self._stats

    def state_dict(self):
        return {k: v.clone() for k, v in self.t.items()}

    # ------------------------------------------------------------------ branching (csrc/ge_state.cu)
    def state_signature(self):
        """What a batch must share with the one a record was saved from: env id, shape parameters and the set of state arrays."""
        d = self.desc
        present = tuple(k for k in _STATE_ARRAYS if (self.env_steps is not None if k == "env_steps" else k in self.t))
        return (self.env_id, d.kind, d.N, d.M, d.parenting, d.n_dests, d.n_choices, d.n_targets, present)

    def record_bytes(self):
        """Bytes of one env's state record (ge_state_record_bytes)."""
        n = self.lib.ge_state_record_bytes(C.byref(self.desc))
        if n < 0:
            _native.check(n)
        return n

    def _index(self, index, n, lo, hi, who):
        """An env / record index as int32 on the device.  A device tensor is trusted (out-of-range entries are skipped by the
        kernels); host data must have n entries (any number up to self.B when n is None), all in [lo, hi)."""
        if isinstance(index, torch.Tensor) and index.is_cuda:
            if index.device != self.device or index.dim() != 1 or (n is not None and index.numel() != n):
                raise ValueError("%s: index must be a 1-D tensor of %s entries on %s" % (who, n if n is not None else "<= B", self.device))
            return index.to(torch.int32).contiguous()
        a = np.asarray(index.numpy() if isinstance(index, torch.Tensor) else index)
        if a.ndim != 1 or (a.size and a.dtype.kind not in "iu") or (n is not None and a.shape[0] != n) or (n is None and a.shape[0] > self.B):
            raise ValueError("%s: index must be a 1-D integer sequence of %s entries" % (who, n if n is not None else "<= %d" % self.B))
        if a.size and (int(a.min()) < lo or int(a.max()) >= hi):
            raise ValueError("%s: index entries must lie in [%d, %d)" % (who, lo, hi))
        return torch.from_numpy(a.astype(np.int32)).to(self.device)

    def save_states(self, index=None, out=None):
        """EnvStates of envs `index` (all envs when None), one record each, every state array included (ge_state_save).
        out: an EnvStates of this batch's signature with as many records, to write into."""
        idx = None if index is None else self._index(index, None, 0, self.B, "save_states")
        n = self.B if idx is None else idx.numel()
        sig = self.state_signature()
        if out is None:
            out = EnvStates(torch.empty((n, self.record_bytes()), dtype=torch.uint8, device=self.device), sig)
        elif not isinstance(out, EnvStates) or out.signature != sig or tuple(out.data.shape) != (n, self.record_bytes()):
            raise ValueError("save_states: out must be EnvStates of this batch's signature with %d records" % n)
        _native.check(self.lib.ge_state_save(C.byref(self.desc), _ptr(idx), n, _ptr(out.data), self._stream()))
        return out

    def load_states(self, states, index=None, what=STATE_ALL):
        """Env b <- record index[b] of `states` (record b when index is None) -- ge_state_load.  what: STATE_DYNAMIC, plus
        STATE_CLOCK (env_steps) and / or STATE_STATS (acc, traj).  A host index is validated (-1 = leave env b as it is); a
        device index is trusted and its out-of-range entries leave their envs untouched.  An in-place fork within one batch is
        env.load_states(env.save_states(), parents)."""
        if not isinstance(states, EnvStates):
            raise TypeError("load_states: states must be EnvStates (from save_states)")
        if states.signature != self.state_signature():
            raise ValueError("load_states: records saved from a batch of signature %s cannot be loaded into one of %s"
                             % (states.signature, self.state_signature()))
        data = states.data
        if data.device != self.device or data.dtype != torch.uint8 or data.dim() != 2 or not data.is_contiguous():
            raise ValueError("load_states: records must be a contiguous uint8 [n, record_bytes] tensor on %s" % self.device)
        n = data.shape[0]
        if index is None and n < self.B:
            raise ValueError("load_states: %d records for %d envs (pass an index)" % (n, self.B))
        idx = None if index is None else self._index(index, self.B, -1, n, "load_states")
        if data.shape[1] != self.record_bytes():
            raise ValueError("load_states: records of %d bytes, this batch's are %d" % (data.shape[1], self.record_bytes()))
        _native.check(self.lib.ge_state_load(C.byref(self.desc), _ptr(data), n, _ptr(idx), int(what), self._stream()))

    def gather_instances(self, src, index=None):
        """Env b <- the instance (every static array) of src env index[b] (src env b when None) -- ge_gather_instances.
        src: a loaded BatchedGraphEnv of the same env id and shape (e.g. this batch's like()).  A host index is validated
        (-1 = leave env b as it is); a device index is trusted.  Writes no state: follow with reset() or load_states().
        DistributionCenter: the batches must share the distance automaton; a batch without one takes src's when the gather
        covers every env."""
        if not isinstance(src, BatchedGraphEnv):
            raise TypeError("gather_instances: src must be a BatchedGraphEnv")
        if src is self:
            raise ValueError("gather_instances: src must be another batch (no in-place gather)")
        if src.env_id != self.env_id or not src._loaded:
            raise ValueError("gather_instances: src must be a loaded %s batch" % self.env_id)
        if index is None and src.B < self.B:
            raise ValueError("gather_instances: src has %d envs, this batch %d (pass an index)" % (src.B, self.B))
        idx = None if index is None else self._index(index, self.B, -1, src.B, "gather_instances")
        if "dfa" in self.t or "dfa" in src.t:
            if "dfa" in self.t and "dfa" in src.t:
                if not torch.equal(self.t["dfa"], src.t["dfa"]):
                    raise ValueError("gather_instances: the batches have different distance automata")
            elif "dfa" in src.t and (idx is None or bool(((idx >= 0) & (idx < src.B)).all())):
                self._take_automaton(src)
            else:
                raise ValueError("gather_instances: the distance automaton of src (%s) and of this batch (%s) differ; a batch "
                                 "takes src's only when the gather covers every env" % ("dfa" in src.t, "dfa" in self.t))
        _native.check(self.lib.ge_gather_instances(C.byref(self.desc), C.byref(src.desc), _ptr(idx), self._stream()))
        self._loaded = True
        self._features_loaded = "features" in self.t

    def _take_automaton(self, src):
        """DistributionCenter: src's distance automaton and room for the arrays derived from it (filled by the gather)."""
        T, B, MP = self.t, self.B, self.desc.MP
        T["dfa"] = src.t["dfa"].clone()
        T["wcode"] = torch.zeros((B, MP), dtype=torch.uint8, device=self.device)
        if "dc_edges" in src.t:
            T["dc_edges"] = torch.zeros((B, MP), dtype=torch.int32, device=self.device)
            T["dc_rows"] = torch.zeros((B, self.N, 32), dtype=torch.int32, device=self.device)
        self._sync_desc()
        self.desc.dfa_bytes = src.desc.dfa_bytes

    def load_state_dict(self, sd):
        for k, v in sd.items():
            self.t[k].copy_(v)


class SliceStreams:
    """C sub-batches of ONE resident batch, each advanced on its own CUDA stream.

    Envs are independent, so step t+1 of an env only has to follow step t of the SAME env: slice c's launches form a chain
    on stream c, and the chains are not ordered against each other.  A launch over a whole small-graph batch is one wave
    of the machine that alternates between an all-memory phase (state + adjacency tiles in) and an all-compute phase (the
    mask searches); C free-running chains de-phase, so one slice's searches run under another slice's loads.

        ss = SliceStreams(env, 4)
        ss.fork()                       # the slice streams wait for what is on the current stream
        for t in range(T): ss.step_sampled(seed, t)
        ss.join()                       # the current stream waits for every slice
    Works under CUDA-graph capture (fork / join become the graph's fork / join edges)."""

    def __init__(self, env, chunks, streams=None):
        self.env = env                                          # (descriptor is read NOW: enable_env_clock() / enable_pdl() first)
        B, C_ = env.B, int(chunks)
        per = ((B + C_ - 1) // C_ + 31) // 32 * 32             # slice starts are multiples of 32 envs (tiled adjacency)
        self.bounds = [(lo, min(per, B - lo)) for lo in range(0, B, per)]
        self.descs = [env.slice_desc(lo, n) for lo, n in self.bounds]
        self.outs = [_native.StepOut(_ptr(env.reward[lo:]), _ptr(env.flags[lo:]), _ptr(env.solution_cost[lo:])) for lo, _ in self.bounds]
        self.acts = [_ptr(env.actions_dev[lo:]) for lo, _ in self.bounds]
        self.streams = streams if streams is not None else [torch.cuda.Stream(device=env.device) for _ in self.bounds]
        assert len(self.streams) >= len(self.bounds)

    def fork(self):
        cur = torch.cuda.current_stream(self.env.device)
        for s in self.streams:
            s.wait_stream(cur)

    def join(self):
        cur = torch.cuda.current_stream(self.env.device)
        for s in self.streams:
            cur.wait_stream(s)

    def step_sampled(self, seed, t):
        L = self.env.lib
        for d, o, a, s in zip(self.descs, self.outs, self.acts, self.streams):
            _native.check(L.ge_step_sampled(C.byref(d), int(seed), int(t), a, C.byref(o), C.c_void_p(s.cuda_stream)))

    def step(self, actions):
        L = self.env.lib
        for (lo, _), d, o, s in zip(self.bounds, self.descs, self.outs, self.streams):
            _native.check(L.ge_step(C.byref(d), _ptr(actions[lo:]), C.byref(o), C.c_void_p(s.cuda_stream)))
