// ge_common.cuh -- shared device helpers of the graphenvs_b200 engine (sm_100a).
//
// Four kernel families share these helpers (DESIGN.md section 4):
//   general   ge_envs.cuh + ge_api.cu   one WARP per env, sets staged in a per-warp shared-memory slice
//   lane      ge_lane.cu                one LANE per env for N <= 64 (sets are 64-bit registers)
//   group     ge_group.cu               8/16/32 lanes per env for 64 < N <= 1024 (one set word per lane)
//   incr      ge_incr.cu                incremental masks for the tree-growing kinds and MaxIndependentSet
// Node/edge sets are packed bitsets everywhere; warp / group votes and REDUX do the set algebra.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "graphenvs_b200.h"

#ifndef __CUDA_ARCH__
#include <nvtx3/nvToolsExt.h>
// NVTX range around a C-ABI entry point (SURVEY section 5 "tracing / profiling"): visible in Nsight Systems timelines,
// a few nanoseconds when no tool is attached.
struct GeNvtxRange {
    explicit GeNvtxRange(const char *name) { nvtxRangePushA(name); }
    ~GeNvtxRange() { nvtxRangePop(); }
};
#define GE_NVTX(name) GeNvtxRange _ge_nvtx_range(name)
#else
#define GE_NVTX(name)
#endif

#define GE_FULL 0xffffffffu
#define GE_WPB 8  // warps (= environments) per thread block

// Step-kernel launch.  With GE_FLAG_PDL in the descriptor the launch carries the programmatic-stream-serialization
// attribute: the kernel may become resident while the previous launch of the stream is still running; its pdl_wait()
// (below) is then what orders it behind that launch (include/graphenvs_b200.h: GE_FLAG_PDL).
template <class... KArgs, class... Args>
inline cudaError_t ge_launch_step(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, const ge_batch &d, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = (d.flags & GE_FLAG_PDL) ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, d, args...);   // a failure is also left for cudaGetLastError() (the callers' *_launched() checks)
}

namespace ge {

typedef unsigned long long u64;

// ge_batch.progress: the threads of a warp that have finished their envs (one env per thread, same 1024-env chunk: chunks are
// tile-aligned) publish them together -- group barrier, then ONE release (fence + atomic) by the group's first thread, which by
// cumulativity covers the stores of the whole group.  Whatever subset of the warp arrives here together forms a group.
#define GE_PROGRESS_SHIFT 10
__device__ __forceinline__ void signal_progress(const ge_batch &d, int b) {
    const unsigned m = __activemask();
    __syncwarp(m);
    if ((threadIdx.x & 31) == (unsigned)(__ffs(m) - 1)) {
        __threadfence();
        atomicAdd(d.progress + (b >> GE_PROGRESS_SHIFT), (unsigned)__popc(m));
    }
}

// griddepcontrol (sm_90+): no-ops when the kernel was not launched as a programmatic dependent.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// Per-warp shared-memory scratch.
struct Scr {
    u64 *q;         // [N]  fp64 distances as ordered bit patterns / (dist32,edge) keys
    uint32_t *vis;  // [NW] HAS_MSG / TAKEN
    uint32_t *aux;  // [NW] second node set (covered, neighbour-union, residual ...)
    uint32_t *t0, *t1, *t2, *t3;  // [NW] temporaries (frontier / next / reach / candidates)
    uint32_t *msk;  // [AW] mask under construction
    uint16_t *lst;  // [2N] two frontier node lists of the cutoff SSSP (DistributionCenter only)
};

__host__ __device__ inline int dist_words(const ge_batch &d) {  // per-node distance scratch: fp64 bit patterns, or
    return (d.kind == GE_DISTRIBUTION_CENTER && d.wcode && d.dfa) ? d.N : 2 * d.N;  // 32-bit automaton states
}
__host__ __device__ inline int scratch_words(const ge_batch &d) {
    int w = ((dist_words(d) + 1) & ~1) + 6 * d.NW + d.AW;
    if (d.kind == GE_DISTRIBUTION_CENTER) w += d.N;  // two uint16 node lists
    return (w + 3) & ~3;  // keep every warp slice 16-byte aligned
}

__device__ inline Scr carve(uint32_t *base, const ge_batch &d) {
    Scr s;
    s.q = reinterpret_cast<u64 *>(base);
    uint32_t *p = base + ((dist_words(d) + 1) & ~1);
    s.vis = p; p += d.NW;
    s.aux = p; p += d.NW;
    s.t0 = p; p += d.NW;
    s.t1 = p; p += d.NW;
    s.t2 = p; p += d.NW;
    s.t3 = p; p += d.NW;
    s.msk = p; p += d.AW;
    s.lst = reinterpret_cast<uint16_t *>(p);
    return s;
}

// Kinds the lane-per-env family (ge_lane.cu, N <= 64) steps.
__host__ __device__ inline bool lane_kind(int kind) {
    return kind == GE_SHORTEST_PATH || kind == GE_LONGEST_PATH || kind == GE_TSP || kind == GE_MAX_INDEPENDENT_SET ||
           kind == GE_DENSEST_SUBGRAPH;
}
// Layout of adj_bits.  Default: env-major, [B, ADJS] = N rows of NW words per env.  For the lane-per-env family
// (N <= 64) the matrix is stored in TILES of 32 envs, [ceil(B/32)][N rows][32 envs] of NW-word elements: lane l of a
// warp reads row r_l of ITS env at element (r_l * 32 + l), so whatever rows the 32 lanes pick, their shared-memory
// accesses fall on 32 different banks (env-major rows collided on 55 % of the wavefronts,
// profiles/r01_lane_step_kernel_cfg2_v4_fused.md), and a block's tiles are still one contiguous bulk copy.
__host__ __device__ inline bool adj_tiled(const ge_batch &d) {
    return d.N <= 64 && lane_kind(d.kind) && !(d.flags & GE_FLAG_FORCE_WARP);
}
__host__ __device__ inline size_t adj_word_index(const ge_batch &d, int b, int row, int w) {
    if (adj_tiled(d)) return ((((size_t)(b >> 5) * d.N + row) << 5) + (b & 31)) * d.NW + w;
    return (size_t)b * d.ADJS + (size_t)row * d.NW + w;
}

__device__ inline bool tbit(const uint32_t *w, int i) { return (w[i >> 5] >> (i & 31)) & 1u; }
__device__ inline uint32_t tail_mask(int n, int w) {  // valid-bit mask of word w of an n-bit set
    int rem = n - (w << 5);
    return rem >= 32 ? 0xffffffffu : (rem <= 0 ? 0u : ((1u << rem) - 1u));
}
__device__ inline uint32_t expand4(uint32_t b) {  // 4 mask bits -> 4 bytes of 0/1
    return ((b & 0xfu) * 0x00204081u) & 0x01010101u;
}

// Position of the n-th (0-based) set bit of a word that has more than n bits set: five popcount halvings
// (the __fns intrinsic is a software loop over the bits).
__device__ __forceinline__ int nth_set_bit(uint32_t w, int n) {
    int pos = 0;
#pragma unroll
    for (int s = 16; s; s >>= 1) {
        const int c = __popc(w & ((1u << s) - 1u));
        if (n >= c) { n -= c; w >>= s; pos += s; }
    }
    return pos;
}

// Counter-based RNG shared bit-for-bit with oracle/graphenvs_oracle.c (ge_mix).
__host__ __device__ inline uint32_t mix32(uint64_t seed, uint32_t env, uint32_t t) {
    uint64_t z = seed + 0x9E3779B97F4A7C15ull * ((uint64_t)env * 0x100000001ull + (((uint64_t)t) << 32 | 0x5bd1e995u));
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z = z ^ (z >> 31);
    return (uint32_t)(z >> 32);
}

// Uniform choice among the valid bits of a packed mask (README.md:54-68 loop): the r-th set bit,
// r = mix32(seed, env, t) * popcount >> 32.  Warp-cooperative; result is warp-uniform, -1 if empty.
// `known_total` >= 0: the caller already tracks the mask's popcount (incremental kernels) -- skips a full pass.
__device__ inline int warp_sample(const uint32_t *mb, int AW, int lane, uint64_t seed, uint32_t env, uint32_t t,
                                  int known_total = -1) {
    int total = known_total;
    if (total < 0) {
        total = 0;
        for (int w = lane; w < AW; w += 32) total += __popc(mb[w]);
        total = __reduce_add_sync(GE_FULL, total);
    }
    if (total <= 0) return -1;
    uint32_t r = (uint32_t)(((uint64_t)mix32(seed, env, t) * (uint64_t)total) >> 32);
    int before = 0, action = -1;
    for (int w0 = 0; w0 < AW; w0 += 32) {
        int w = w0 + lane;
        uint32_t word = w < AW ? mb[w] : 0u;
        int c = __popc(word), inc = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int x = __shfl_up_sync(GE_FULL, inc, o);
            if (lane >= o) inc += x;
        }
        int chunk = __shfl_sync(GE_FULL, inc, 31);
        if ((int)r < before + chunk) {
            unsigned hit = __ballot_sync(GE_FULL, (int)r < before + inc);
            int src_lane = __ffs(hit) - 1;
            int excl = before + inc - c;
            int pos = (lane == src_lane) ? nth_set_bit(word, (int)r - excl) : 0;
            pos = __shfl_sync(GE_FULL, pos, src_lane);
            action = ((w0 + src_lane) << 5) + pos;
            break;
        }
        before += chunk;
    }
    return action;
}

// A GROUP of G lanes (G = 8, 16 or 32, aligned inside its warp) works on one env.  These kernels are chains of
// dependent memory rounds -- throughput is (envs in flight) / (chain latency) -- and a CSR row here is 10-20
// edges, so narrower groups keep 2-4x more envs in flight per resident warp at the same lane utilisation.
template <int G>
struct Grp {
    int gl;         // lane inside the group
    unsigned mask;  // participation mask of the group inside its warp
    int base;       // first warp lane of the group
    __device__ __forceinline__ Grp() {
        const int lane = threadIdx.x & 31;
        gl = lane & (G - 1);
        base = lane & ~(G - 1);
        mask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << base);
    }
    __device__ __forceinline__ unsigned ballot(bool p) const { return (__ballot_sync(mask, p) >> base) & ((G == 32) ? 0xffffffffu : ((1u << G) - 1u)); }
    template <class T> __device__ __forceinline__ T shfl(T v, int src) const { return __shfl_sync(mask, v, src, G); }
    __device__ __forceinline__ int sum(int v) const { return __reduce_add_sync(mask, v); }
    __device__ __forceinline__ void sync() const { __syncwarp(mask); }
};

// Group version of ge_common.cuh:warp_sample (same draw): r-th set bit of the packed mask, popcount known.
template <int G>
__device__ __forceinline__ int group_sample(const Grp<G> &g, const uint32_t *mb, int AW, uint64_t seed, uint32_t env, uint32_t t, int total) {
    if (total <= 0) return -1;
    uint32_t r = (uint32_t)(((uint64_t)mix32(seed, env, t) * (uint64_t)total) >> 32);
    int before = 0, action = -1;
    for (int w0 = 0; w0 < AW; w0 += G) {
        int w = w0 + g.gl;
        uint32_t word = w < AW ? mb[w] : 0u;
        int c = __popc(word), inc = c;
#pragma unroll
        for (int o = 1; o < G; o <<= 1) {
            int x = __shfl_up_sync(g.mask, inc, o, G);
            if (g.gl >= o) inc += x;
        }
        int chunk = g.shfl(inc, G - 1);
        if ((int)r < before + chunk) {
            unsigned hit = g.ballot((int)r < before + inc);
            int src_lane = __ffs(hit) - 1;
            int excl = before + inc - c;
            int pos = (g.gl == src_lane) ? nth_set_bit(word, (int)r - excl) : 0;
            pos = g.shfl(pos, src_lane);
            action = ((w0 + src_lane) << 5) + pos;
            break;
        }
        before += chunk;
    }
    return action;
}

// The same draw with the whole mask in REGISTERS: lane l of the group loads WPL consecutive words (AW <= G * WPL) up front --
// independent loads, one memory round -- instead of walking the mask G words at a time with an early exit that makes every
// trip wait for its own load (ncu r02: the walk was ~30 % of the instructions and 18 % of the stall samples of the Multicast
// step, whose mask is 250 words).  `total` must be the mask's popcount (the incremental kernels track it).
template <int G, int WPL>
__device__ __forceinline__ int group_sample_regs(const Grp<G> &g, const uint32_t *mb, int AW, uint64_t seed, uint32_t env, uint32_t t, int total) {
    if (total <= 0) return -1;
    const uint32_t r = (uint32_t)(((uint64_t)mix32(seed, env, t) * (uint64_t)total) >> 32);
    uint32_t w[WPL];
    const int base = g.gl * WPL;
#pragma unroll
    for (int k = 0; k < WPL; ++k) w[k] = (base + k < AW) ? mb[base + k] : 0u;
    int cnt = 0;
#pragma unroll
    for (int k = 0; k < WPL; ++k) cnt += __popc(w[k]);
    int inc = cnt;
#pragma unroll
    for (int o = 1; o < G; o <<= 1) {
        const int x = __shfl_up_sync(g.mask, inc, o, G);
        if (g.gl >= o) inc += x;
    }
    const int excl = inc - cnt;
    const bool mine = (int)r >= excl && (int)r < inc;
    int rr = (int)r - excl, kk = 0;
    uint32_t word = 0;
    bool found = false;
#pragma unroll
    for (int k = 0; k < WPL; ++k) {
        const int c = __popc(w[k]);
        if (!found) {
            if (rr < c) { found = true; word = w[k]; kk = k; }
            else rr -= c;
        }
    }
    int a = (mine && found) ? (((base + kk) << 5) + nth_set_bit(word, rr)) : -1;
    const unsigned hit = g.ballot(mine && found);
    if (!hit) return -1;
    return g.shfl(a, __ffs(hit) - 1);
}

// Publishes the mask built in shared memory: packed words, optional byte mask; returns popcount.
__device__ inline int emit_mask(const ge_batch &d, int b, int lane, uint32_t *msk) {
    int cnt = 0;
    for (int w = lane; w < d.AW; w += 32) {
        uint32_t m = msk[w] & tail_mask(d.A, w);
        msk[w] = m;
        cnt += __popc(m);
        d.mask_bits[(size_t)b * d.AW + w] = m;
    }
    cnt = __reduce_add_sync(GE_FULL, cnt);
    if (d.mask_bytes) {
        __syncwarp();
        uint4 *mb = reinterpret_cast<uint4 *>(d.mask_bytes + (size_t)b * d.AP);
        for (int c = lane; c < (d.AP >> 4); c += 32) {  // 16 mask entries -> one 128-bit store
            uint32_t bits = (msk[c >> 1] >> ((c & 1) * 16)) & 0xffffu;
            uint4 v;
            v.x = expand4(bits);
            v.y = expand4(bits >> 4);
            v.z = expand4(bits >> 8);
            v.w = expand4(bits >> 12);
            mb[c] = v;
        }
    }
    __syncwarp();
    return cnt;
}

// Index of edge u->v in row u (warp scan of the row), -1 if absent.  Result is warp-uniform.
__device__ inline int find_edge(const int32_t *rp, const int32_t *col, int u, int v, int lane) {
    int lo = rp[u], hi = rp[u + 1];
    for (int base = lo; base < hi; base += 32) {
        int e = base + lane;
        bool hit = e < hi && col[e] == v;
        unsigned bal = __ballot_sync(GE_FULL, hit);
        if (bal) return base + __ffs(bal) - 1;
    }
    return -1;
}

// adj[u, v] of the reference's dense float64 matrix (0 when there is no edge) without scanning the CSR
// row: the rank of v among the set bits of u's adjacency bit-row indexes the destination-sorted weights.
// Warp-cooperative (lane w counts word w); result is warp-uniform.
__device__ inline double edge_weight_ranked(const ge_batch &d, int b, const uint32_t *adj, int u, int v, int lane) {
    const uint32_t *row = adj + (size_t)u * d.NW;
    const int vw = v >> 5;
    int rank = 0;
    bool present = false;
    for (int w = lane; w <= vw; w += 32) {
        uint32_t bits = row[w];
        if (w == vw) { present = (bits >> (v & 31)) & 1u; bits &= (1u << (v & 31)) - 1u; }
        rank += __popc(bits);
    }
    rank = __reduce_add_sync(GE_FULL, rank);
    if (!__any_sync(GE_FULL, present)) return 0.0;
    return d.wsort[(size_t)b * d.MP + d.row_ptr[(size_t)b * d.RP + u] + rank];
}

// Source node of directed edge e (binary search over row_ptr; warp-uniform when e is).
__device__ inline int edge_src(const int32_t *rp, int N, int e) {
    int lo = 0, hi = N;  // invariant: rp[lo] <= e < rp[hi]
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (rp[mid] <= e) lo = mid; else hi = mid;
    }
    return lo;
}

// Load-balanced warp expansion of the CSR rows of a node set.
// For every node u in `set` (NW words, in shared memory) and every edge e of row u, calls
//     f(owner_lane, e, active)
// from ALL 32 lanes (so f may shuffle); `owner_lane` is the lane that holds the per-node payload
// the caller loaded in `load(u)`; `active` is false for padding lanes.  The 32 nodes of one set
// word are handled together: lane l owns node 32w+l (row bounds = two coalesced 128-byte loads),
// an inclusive scan of the row lengths lays the edges of all member rows out on one line, and each
// group of 32 consecutive edge slots finds its owning row with a 5-step shuffle binary search.
// Edges are walked in row order => coalesced segments, up to 32 rows in flight, no per-row serial
// latency chain, and no find-nth-set-bit (ncu: __fns was 25-30 % of the instructions of the first
// version, profiles/r01_step_kernel_cfg5_distcenter_warp_v1.md).
template <class Load, class Visit>
__device__ inline void expand_set(const int32_t *rp, const uint32_t *set, int NW, int lane, Load load, Visit f) {
    for (int w = 0; w < NW; ++w) {
        const uint32_t bits = set[w];  // warp-uniform (broadcast read)
        if (!bits) continue;
        const bool member = (bits >> lane) & 1u;
        const int u = (w << 5) + lane;
        int lo = 0, len = 0;
        if (member) { lo = rp[u]; len = rp[u + 1] - lo; }
        load(member ? u : -1);  // caller captures payload for node u in registers of this lane
        int incl = len;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int t = __shfl_up_sync(GE_FULL, incl, o);
            if (lane >= o) incl += t;
        }
        const int total = __shfl_sync(GE_FULL, incl, 31);
        const int base = lo - (incl - len);  // edge id = base + slot for the slots of this lane's row
        for (int t0 = 0; t0 < total; t0 += 32) {
            const int t = t0 + lane;
            int owner = 0;  // first lane whose inclusive prefix exceeds t
#pragma unroll
            for (int step = 16; step; step >>= 1) {
                int v = __shfl_sync(GE_FULL, incl, owner + step - 1);
                if (v <= t) owner += step;
            }
            owner &= 31;
            const int ob = __shfl_sync(GE_FULL, base, owner);
            f(owner, ob + t, t < total);
        }
    }
}

// fp64 SSSP with optional cutoff, value semantics of nx _dijkstra_multisource
// (nx:algorithms/shortest_paths/weighted.py:853-881): distances are left-fold fp64 path sums,
// relaxations with dist+w > cutoff are skipped.  Frontier Bellman-Ford to the fixed point gives
// the same values because fp64 add is monotone.  Result: s.q[v] = bit pattern of dist (+inf if
// unreached).  Uses s.t0 / s.t1 as frontier / next.
__device__ inline void sssp_warp(const ge_batch &d, int b, int lane, Scr &s, int source, double cutoff, bool use_cutoff) {
    const int32_t *rp = d.row_ptr + (size_t)b * d.RP;
    const int32_t *col = d.col + (size_t)b * d.MP;
    const double *w64 = d.w64 + (size_t)b * d.MP;
    const u64 INF = 0x7ff0000000000000ull;
    // A node whose distance plus the instance's SMALLEST weight already exceeds the cutoff cannot relax
    // anything (fp64 add is monotone in the weight), so it never enters the frontier: with cutoff 1.0
    // and weights k/10 >= 0.3 only nodes within 0.7 are expanded.  Exact, not a heuristic.
    const double wmin = (use_cutoff && d.wmin) ? d.wmin[b] : 0.0;
    for (int v = lane; v < d.N; v += 32) s.q[v] = INF;
    for (int w = lane; w < d.NW; w += 32) { s.t0[w] = 0; s.t1[w] = 0; }
    __syncwarp();
    if (lane == 0) { s.q[source] = 0ull; s.t0[source >> 5] = 1u << (source & 31); }
    __syncwarp();
    for (int round = 0; round < 4 * d.N + 4; ++round) {
        double du = 0.0;
        expand_set(
            rp, s.t0, d.NW, lane, [&](int u) { du = u >= 0 ? __longlong_as_double((long long)s.q[u]) : 0.0; },
            [&](int owner, int e, bool active) {
                double dsrc = __shfl_sync(GE_FULL, du, owner);
                if (active) {
                    int v = col[e];
                    double nd = dsrc + w64[e];
                    if (!use_cutoff || nd <= cutoff) {
                        u64 nb = (u64)__double_as_longlong(nd);
                        u64 old = atomicMin(&s.q[v], nb);
                        if (nb < old && (!use_cutoff || nd + wmin <= cutoff)) atomicOr(&s.t1[v >> 5], 1u << (v & 31));
                    }
                }
            });
        __syncwarp();
        uint32_t any = 0;
        for (int w = lane; w < d.NW; w += 32) { uint32_t n = s.t1[w]; s.t0[w] = n; s.t1[w] = 0; any |= n; }
        __syncwarp();
        if (!__any_sync(GE_FULL, any != 0)) break;
    }
}

// Cutoff SSSP from one node (find_nodes_in_range, distribution_center.py:25-26 =
// nx.single_source_dijkstra_path_length(cutoff=...), nx:algorithms/shortest_paths/weighted.py:853-881):
// leaves in s.t2 the set of nodes whose fp64 left-fold distance is <= cutoff.  Label-correcting rounds
// over a compact LIST of frontier nodes (a ball of radius 1.0 under weights >= 0.3 has a few dozen
// expandable nodes scattered over all 16 set words -- a bitset frontier would walk 16 mostly empty words
// per round).  Up to 32 frontier rows are laid out on one line by an inclusive scan and consumed 32
// edges at a time (shuffle binary search for the owning row).  64-bit shared-memory atomicMin is a CAS
// spin on this hardware (SASS ATOMS.CAST.SPIN.64), so a plain read filters the relaxations that cannot
// improve anything before the atomic.  Uses s.q (distances), s.t0 (queued-for-next-round), s.t1[0]
// (next-round count), s.lst.
__device__ inline void sssp_cutoff_warp(const ge_batch &d, int b, int lane, Scr &s, int source, double cutoff) {
    const int32_t *rp = d.row_ptr + (size_t)b * d.RP;
    const int32_t *col = d.col + (size_t)b * d.MP;
    const double *w64 = d.w64 + (size_t)b * d.MP;
    const u64 INF = 0x7ff0000000000000ull;
    const double wmin = d.wmin ? d.wmin[b] : 0.0;  // see sssp_warp: exact pruning of nodes that cannot relax anything
    const int N = d.N;
    uint16_t *cur = s.lst, *nxt = s.lst + N;
    int *cnt = reinterpret_cast<int *>(s.t1);
    for (int v = lane; v < N; v += 32) s.q[v] = INF;
    for (int w = lane; w < d.NW; w += 32) { s.t0[w] = 0; s.t2[w] = 0; }
    __syncwarp();
    if (lane == 0) { s.q[source] = 0ull; s.t2[source >> 5] = 1u << (source & 31); cur[0] = (uint16_t)source; *cnt = 0; }
    __syncwarp();
    int ncur = (0.0 + wmin <= cutoff) ? 1 : 0;
    while (ncur > 0) {
        for (int base0 = 0; base0 < ncur; base0 += 32) {
            const int i = base0 + lane;
            int lo = 0, len = 0;
            double du = 0.0;
            if (i < ncur) {
                int u = cur[i];
                lo = rp[u];
                len = rp[u + 1] - lo;
                du = __longlong_as_double((long long)s.q[u]);
            }
            int incl = len;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int t = __shfl_up_sync(GE_FULL, incl, o);
                if (lane >= o) incl += t;
            }
            const int total = __shfl_sync(GE_FULL, incl, 31);
            const int rbase = lo - (incl - len);
            // Software-pipelined over 32-edge slot groups: the loads of group i+1 (destination + weight) are in
            // flight while group i is relaxed, so a round costs about one memory latency instead of one per group.
            auto fetch = [&](int t0, int &v, double &wt, double &dsrc, bool &active) {
                const int t = t0 + lane;
                int owner = 0;
#pragma unroll
                for (int step = 16; step; step >>= 1) {
                    int x = __shfl_sync(GE_FULL, incl, owner + step - 1);
                    if (x <= t) owner += step;
                }
                owner &= 31;
                const int e = __shfl_sync(GE_FULL, rbase, owner) + t;
                dsrc = __shfl_sync(GE_FULL, du, owner);
                active = t < total;
                v = active ? col[e] : 0;
                wt = active ? w64[e] : 0.0;
            };
            int v0 = 0, v1 = 0;
            double w0 = 0.0, w1 = 0.0, d0 = 0.0, d1 = 0.0;
            bool a0 = false, a1 = false;
            if (total > 0) fetch(0, v0, w0, d0, a0);
            for (int t0 = 0; t0 < total; t0 += 32) {
                const bool more = t0 + 32 < total;
                if (more) fetch(t0 + 32, v1, w1, d1, a1);
                if (a0) {
                    const int v = v0;
                    const double nd = d0 + w0;
                    if (nd <= cutoff) {                                     // nx: skip when dist + w > cutoff
                        const u64 nb = (u64)__double_as_longlong(nd);
                        if (nb < s.q[v]) {
                            const u64 old = atomicMin(&s.q[v], nb);
                            if (nb < old) {
                                if (old == INF) atomicOr(&s.t2[v >> 5], 1u << (v & 31));
                                if (nd + wmin <= cutoff) {
                                    const uint32_t bit = 1u << (v & 31);
                                    if (!(atomicOr(&s.t0[v >> 5], bit) & bit)) {
                                        nxt[atomicAdd(cnt, 1)] = (uint16_t)v;
                                        asm volatile("prefetch.global.L2 [%0];" ::"l"(rp + v));  // next round's row bounds
                                    }
                                }
                            }
                        }
                    }
                }
                v0 = v1; w0 = w1; d0 = d1; a0 = more && a1;
            }
        }
        __syncwarp();
        ncur = *cnt;
        __syncwarp();
        if (lane == 0) *cnt = 0;
        for (int w = lane; w < d.NW; w += 32) s.t0[w] = 0;
        uint16_t *tmp = cur; cur = nxt; nxt = tmp;
        __syncwarp();
    }
}

// The same search on the exact distance AUTOMATON (ge_batch.dfa): when the batch's edge weights come from a
// small set (k/10 in the reference), every fp64 left-fold sum that stays within the cutoff is one of a few
// dozen values, enumerated on the host with the same IEEE additions and sorted -- a distance is a state id
// (order-preserving), dist + w is a table lookup, the 64-bit CAS-spin min becomes a native 32-bit shared
// atomicMin, and an edge weight is a one-byte code instead of eight bytes.  Bit-identical sets, by
// construction; tests run both searches against the oracle.
__device__ inline void sssp_cutoff_dfa(const ge_batch &d, int b, int lane, Scr &s, int source) {
    const int32_t *rp = d.row_ptr + (size_t)b * d.RP;
    const int32_t *col = d.col + (size_t)b * d.MP;
    const uint8_t *wc = d.wcode + (size_t)b * d.MP;
    const int W = d.dfa[1];
    const uint8_t *tab = d.dfa + 2, *expand = tab + (int)d.dfa[0] * W;
    const int N = d.N;
    uint32_t *q = reinterpret_cast<uint32_t *>(s.q);
    uint16_t *cur = s.lst, *nxt = s.lst + N;
    int *cnt = reinterpret_cast<int *>(s.t1);
    for (int v = lane; v < N; v += 32) q[v] = 255u;
    for (int w = lane; w < d.NW; w += 32) { s.t0[w] = 0; s.t2[w] = 0; }
    __syncwarp();
    if (lane == 0) { q[source] = 0u; s.t2[source >> 5] = 1u << (source & 31); cur[0] = (uint16_t)source; *cnt = 0; }
    __syncwarp();
    int ncur = __ldg(expand) ? 1 : 0;
    while (ncur > 0) {
        for (int base0 = 0; base0 < ncur; base0 += 32) {
            const int i = base0 + lane;
            int lo = 0, len = 0, du = 0;
            if (i < ncur) {
                int u = cur[i];
                lo = rp[u];
                len = rp[u + 1] - lo;
                du = (int)q[u];
            }
            int incl = len;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int t = __shfl_up_sync(GE_FULL, incl, o);
                if (lane >= o) incl += t;
            }
            const int total = __shfl_sync(GE_FULL, incl, 31);
            const int rbase = lo - (incl - len);
            auto fetch = [&](int t0, int &v, int &code, int &dsrc, bool &active) {
                const int t = t0 + lane;
                int owner = 0;
#pragma unroll
                for (int step = 16; step; step >>= 1) {
                    int x = __shfl_sync(GE_FULL, incl, owner + step - 1);
                    if (x <= t) owner += step;
                }
                owner &= 31;
                const int e = __shfl_sync(GE_FULL, rbase, owner) + t;
                dsrc = __shfl_sync(GE_FULL, du, owner);
                active = t < total;
                v = active ? col[e] : 0;
                code = active ? (int)wc[e] : 0;
            };
            int v0 = 0, v1 = 0, c0 = 0, c1 = 0, d0 = 0, d1 = 0;
            bool a0 = false, a1 = false;
            if (total > 0) fetch(0, v0, c0, d0, a0);
            for (int t0 = 0; t0 < total; t0 += 32) {
                const bool more = t0 + 32 < total;
                if (more) fetch(t0 + 32, v1, c1, d1, a1);
                if (a0) {
                    const uint32_t nid = __ldg(tab + d0 * W + c0);          // state of fl(dist + w), 255 = beyond the cutoff
                    if (nid != 255u && nid < q[v0]) {
                        const uint32_t old = atomicMin(&q[v0], nid);
                        if (nid < old) {
                            if (old == 255u) atomicOr(&s.t2[v0 >> 5], 1u << (v0 & 31));
                            if (__ldg(expand + nid)) {
                                const uint32_t bit = 1u << (v0 & 31);
                                if (!(atomicOr(&s.t0[v0 >> 5], bit) & bit)) {
                                    nxt[atomicAdd(cnt, 1)] = (uint16_t)v0;
                                    asm volatile("prefetch.global.L2 [%0];" ::"l"(rp + v0));
                                }
                            }
                        }
                    }
                }
                v0 = v1; c0 = c1; d0 = d1; a0 = more && a1;
            }
        }
        __syncwarp();
        ncur = *cnt;
        __syncwarp();
        if (lane == 0) *cnt = 0;
        for (int w = lane; w < d.NW; w += 32) s.t0[w] = 0;
        uint16_t *tmp = cur; cur = nxt; nxt = tmp;
        __syncwarp();
    }
}

// find_nodes_in_range: exact automaton when the batch has one, fp64 search otherwise.  Result set in s.t2.
__device__ inline void cutoff_reach(const ge_batch &d, int b, int lane, Scr &s, int source) {
    if (d.wcode && d.dfa) sssp_cutoff_dfa(d, b, lane, s, source);
    else sssp_cutoff_warp(d, b, lane, s, source, d.max_distance);
}

// Reachability over the adjacency bit-matrix inside `allowed`, seeded with the bits already in
// `reach`.  frontier/next are NW-word temporaries.  Lane w owns word w (+32k) of every set.
// With stop_at >= 0 the search ends as soon as |reach| == stop_at (connectivity tests: everything
// allowed has been reached, expanding the last level cannot add anything).
__device__ inline void bfs_bits(const uint32_t *adj, int NW, int lane, const uint32_t *allowed, uint32_t *reach,
                                uint32_t *frontier, uint32_t *next, int stop_at = -1) {
    for (int w = lane; w < NW; w += 32) frontier[w] = reach[w];
    __syncwarp();
    for (;;) {
        for (int w = lane; w < NW; w += 32) next[w] = 0;
        for (int fw = 0; fw < NW; ++fw) {
            uint32_t bits = frontier[fw];
            while (bits) {
                int v = (fw << 5) + __ffs(bits) - 1;
                bits &= bits - 1;
                for (int w = lane; w < NW; w += 32) next[w] |= __ldg(&adj[(size_t)v * NW + w]);
            }
        }
        __syncwarp();
        uint32_t any = 0;
        int cnt = 0;
        for (int w = lane; w < NW; w += 32) {
            uint32_t n = next[w] & allowed[w] & ~reach[w];
            uint32_t r = reach[w] | n;
            reach[w] = r;
            frontier[w] = n;
            any |= n;
            cnt += __popc(r);
        }
        __syncwarp();
        if (!__any_sync(GE_FULL, any != 0)) break;
        if (stop_at >= 0 && __reduce_add_sync(GE_FULL, cnt) == stop_at) break;
    }
}

}  // namespace ge
