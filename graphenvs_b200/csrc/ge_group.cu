// ge_group.cu -- GROUP-PER-ENV kernels for the node-action kinds (ShortestPath, LongestPath, TSP,
// DensestSubgraph) with 64 < N <= 1024: the mask is one adjacency row, optionally pruned by reachability
// (LongestPath parenting >= 2) or by cut-vertex tests (TSP parenting 2) on the adjacency bit-matrix.
//
// Why: ncu on the general warp-per-env kernel showed these steps ISSUE-bound at ~1,000 warp-instructions
// per env-step (profiles/r01_step_kernel_cfg4_tsp_p1_warp_v2.md: 60 % issue utilisation, 5 % of HBM peak):
// shared-memory staging, generic dispatch and a 32-lane warp for a 7-word bitset.  Here a GROUP of G = 8,
// 16 or 32 lanes owns one env, every lane keeps ONE 32-bit word of each node set in a register, set algebra
// is one instruction per word, cross-word facts (popcounts, the rank of the chosen node in its adjacency
// row) are group reductions, and a warp advances 32/G envs.  Same rules as ge_envs.cuh / ge_lane.cu
// (same reference line map); tests run every eligible case through both families.
#include "ge_common.cuh"

using namespace ge;

extern "C" int ge_set_error(int code, const char *fmt, ...);

namespace {

__host__ __device__ inline bool group_kind(const ge_batch &d) {
    return d.kind == GE_SHORTEST_PATH || d.kind == GE_LONGEST_PATH || d.kind == GE_TSP || d.kind == GE_DENSEST_SUBGRAPH;
}

constexpr int NO_NODE = 0x7fffffff;

template <int G>
__device__ __forceinline__ int lowest_node(const Grp<G> &g, uint32_t w) {  // lowest set node id of a distributed set
    return __reduce_min_sync(g.mask, w ? (g.gl << 5) + __ffs(w) - 1 : NO_NODE);
}

// Worklist reachability inside `allowed` (one word per lane) from node `seed`; stops once `stop_count` nodes
// are reached (everything allowed) or the frontier is empty.  Returns the number of reached nodes; leaves
// the reached set in reach_w and, when `internal` is given, the nodes whose expansion discovered something
// (the internal nodes of a spanning tree).  Two frontier rows are fetched per trip (independent loads).
template <int G>
__device__ __forceinline__ int group_reach(const Grp<G> &g, const uint32_t *adj, int NW, uint32_t allowed, int seed, int stop_count,
                                           uint32_t &reach_w, uint32_t *internal) {
    const int lane = g.gl;
    const bool W = lane < NW;
    uint32_t reach = (lane == (seed >> 5)) ? (1u << (seed & 31)) : 0u, frontier = reach, inner = 0;
    int reached = 1;
    while (reached < stop_count) {
        const int r1 = lowest_node(g, frontier);
        if (r1 == NO_NODE) break;
        if (lane == (r1 >> 5)) frontier &= ~(1u << (r1 & 31));
        const int r2 = lowest_node(g, frontier);
        if (r2 != NO_NODE && lane == (r2 >> 5)) frontier &= ~(1u << (r2 & 31));
        const uint32_t row1 = W ? __ldg(adj + (size_t)r1 * NW + lane) : 0u;
        const uint32_t row2 = (W && r2 != NO_NODE) ? __ldg(adj + (size_t)r2 * NW + lane) : 0u;
        uint32_t nx = row1 & allowed & ~reach;
        int added = g.sum(__popc(nx));
        if (added && lane == (r1 >> 5)) inner |= 1u << (r1 & 31);
        reach |= nx; frontier |= nx; reached += added;
        if (r2 != NO_NODE) {
            nx = row2 & allowed & ~reach;
            added = g.sum(__popc(nx));
            if (added && lane == (r2 >> 5)) inner |= 1u << (r2 & 31);
            reach |= nx; frontier |= nx; reached += added;
        }
    }
    reach_w = reach;
    if (internal) *internal = inner;
    return reached;
}

// LongestPath parenting >= 2 (longest_path.py:133-143): keep the candidates that still reach dest in the
// graph induced on unvisited nodes (symmetric => one search from dest).
template <int G>
__device__ __forceinline__ uint32_t group_prune_longest_path(const ge_batch &d, const Grp<G> &g, const uint32_t *adj, uint32_t m,
                                                             uint32_t visw, uint32_t tail, int dest) {
    if ((g.shfl(visw, dest >> 5) >> (dest & 31)) & 1u) return m;                  // dest not in alt_G (:135-136)
    const uint32_t allowed = ~visw & tail;
    const int n_alt = g.sum(__popc(allowed));
    uint32_t reach;
    group_reach(g, adj, d.NW, allowed, dest, n_alt, reach, nullptr);
    m &= reach;
    if (d.parenting == 3 && n_alt <= d.N / 3) m |= allowed;                        // :141-143
    return m;
}

// TSP parenting 2 (tsp.py:181-194): drop the candidates whose removal disconnects alt_G = all - start - taken.
// One spanning search first: only the INTERNAL nodes of a spanning tree can be cut vertices, the literal
// "remove v, test connectivity" runs for those alone (ascending candidate order like the reference).
template <int G>
__device__ __forceinline__ uint32_t group_prune_tsp(const ge_batch &d, const Grp<G> &g, const uint32_t *adj, uint32_t m, uint32_t visw,
                                                    uint32_t tail) {
    const int lane = g.gl;
    uint32_t res = ~visw & tail;
    if (lane == 0) res &= ~1u;
    const int n_res = g.sum(__popc(res));
    uint32_t cand = m;
    if (n_res >= 2) {
        uint32_t reach, inner;
        const int seed = lowest_node(g, res);
        if (group_reach(g, adj, d.NW, res, seed, n_res, reach, &inner) == n_res) cand &= inner | (lane == 0 ? 1u : 0u);
    }
    for (;;) {
        const int v = lowest_node(g, cand);
        if (v == NO_NODE) break;
        if (lane == (v >> 5)) cand &= ~(1u << (v & 31));
        if (v == 0) continue;
        if (n_res - 1 == 0) break;                                                 // :191-192
        uint32_t gw = res;
        if (lane == (v >> 5)) gw &= ~(1u << (v & 31));
        uint32_t reach;
        const int seed = lowest_node(g, gw);
        if (group_reach(g, adj, d.NW, gw, seed, n_res - 1, reach, nullptr) != n_res - 1 && lane == (v >> 5))
            m &= ~(1u << (v & 31));                                               // :193-194
    }
    return m;
}

// the lane's word of the mask for the CURRENT state (ge_envs.cuh: mask_head_row / mask_tsp / mask_densest)
template <int G>
__device__ __forceinline__ uint32_t group_mask_word(const ge_batch &d, const Grp<G> &g, const uint32_t *adj, int dest, uint32_t roww,
                                                    uint32_t visw, uint32_t auxw, uint32_t tail, int k_taken) {
    switch (d.kind) {
    case GE_SHORTEST_PATH: return roww & ~visw;                              // shortest_path.py:105-109
    case GE_LONGEST_PATH: {                                                   // longest_path.py:125-145
        if (d.parenting == 0) return tail;
        uint32_t m = roww & ~visw;
        if (d.parenting >= 2) m = group_prune_longest_path(d, g, adj, m, visw, tail, dest);
        return m; }
    case GE_TSP: {                                                            // tsp.py:174-199
        uint32_t m = roww & ~visw;
        int taken = g.sum(__popc(visw));
        if (taken < d.N - 1 && g.gl == 0) m &= ~1u;
        if (d.parenting >= 2) m = group_prune_tsp(d, g, adj, m, visw, tail);
        return m; }
    case GE_DENSEST_SUBGRAPH:                                                 // densest_subgraph.py:105-129
        if (k_taken == 0) return tail;
        return (d.parenting == 0 ? ~visw : (auxw & ~visw)) & tail;
    }
    return 0;
}

template <int G>
__device__ __forceinline__ void store_mask_word(const ge_batch &d, int b, int lane, uint32_t m) {
    if (lane >= d.AW) return;
    d.mask_bits[(size_t)b * d.AW + lane] = m;
    if (d.mask_bytes) {  // the lane's 32 mask entries = two 128-bit stores
        uint4 *mb = reinterpret_cast<uint4 *>(d.mask_bytes + (size_t)b * d.AP);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            int c = 2 * lane + h;
            if (c < (d.AP >> 4)) {
                uint32_t bits = (m >> (16 * h)) & 0xffffu;
                mb[c] = make_uint4(expand4(bits), expand4(bits >> 4), expand4(bits >> 8), expand4(bits >> 12));
            }
        }
    }
}

template <bool SAMPLED, int G>
__global__ void __launch_bounds__(256, 8) group_step_kernel(ge_batch d, int32_t *__restrict__ actions, ge_step_out out, uint64_t seed,
                                                          uint32_t t) {
    const Grp<G> g;
    const int lane = g.gl;
    const int b = blockIdx.x * (256 / G) + (int)threadIdx.x / G;
    pdl_launch_dependents();   // programmatic dependent launch (ge_common.cuh): no-ops on a plain launch
    pdl_wait();
    if (b >= d.B) return;
    const int N = d.N, NW = d.NW, kind = d.kind;
    const bool W = lane < NW;
    const uint32_t tail = W ? tail_mask(N, lane) : 0u;
    const uint32_t *adj = d.adj_bits + (size_t)b * d.ADJS;
    // ---- round 1: everything that does not depend on the action
    uint32_t visw = W ? d.node_bits[(size_t)b * NW + lane] : 0u;
    uint32_t auxw = (W && d.node_bits2) ? d.node_bits2[(size_t)b * NW + lane] : 0u;
    const uint32_t oldm = W ? d.mask_bits[(size_t)b * d.AW + lane] : 0u;
    const uint32_t m0 = (W && d.mask0_bits) ? d.mask0_bits[(size_t)b * d.AW + lane] : 0u;
    int head = d.head[b];
    double cost = d.cost[b];
    const bool was_done = d.done[b] != 0;
    const uint32_t nsteps = d.env_steps ? d.env_steps[b] : 0u;
    const bool seeded = kind == GE_SHORTEST_PATH || kind == GE_LONGEST_PATH;
    const int dest = seeded ? d.dest[b] : 0, src = seeded ? d.src[b] : 0;
    int4 c = make_int4(0, 0, 0, 0);
    if (kind == GE_DENSEST_SUBGRAPH) c = *reinterpret_cast<const int4 *>(d.counters + (size_t)b * 4);
    const uint32_t rowh = (W && kind != GE_DENSEST_SUBGRAPH) ? adj[(size_t)head * NW + lane] : 0u;  // N(head): weight rank, nb test
    const int rp_head = kind != GE_DENSEST_SUBGRAPH ? d.row_ptr[(size_t)b * d.RP + head] : 0;
    // ---- action
    int a;
    if (SAMPLED) {  // r-th set bit of the mask, same draw as warp_sample
        const int pc = __popc(oldm);
        int inc = pc;
#pragma unroll
        for (int o = 1; o < G; o <<= 1) {
            int x = __shfl_up_sync(g.mask, inc, o, G);
            if (lane >= o) inc += x;
        }
        const int total = g.shfl(inc, G - 1);
        a = -1;
        if (total > 0) {
            const uint32_t r = (uint32_t)(((uint64_t)mix32(seed, (uint32_t)(d.env_id0 + b), t + nsteps) * (uint64_t)total) >> 32);
            const unsigned hit = g.ballot((int)r < inc);
            const int sl = __ffs(hit) - 1;
            int pos = (lane == sl) ? nth_set_bit(oldm, (int)r - (inc - pc)) : 0;
            a = (sl << 5) + g.shfl(pos, sl);
        }
        if (lane == 0) actions[b] = a;
    } else {
        a = actions[b];
    }
    double reward = 0.0, sol = __longlong_as_double(0x7ff8000000000000ll);
    int done = 0, solved = -1, has_mask = 1, status = GE_STEP_OK;
    uint32_t maskw = oldm;
    bool write_state = false;
    const bool a_ok = a >= 0 && a < N;
    const uint32_t oldm_a = g.shfl(oldm, a_ok ? (a >> 5) : 0);
    if (was_done) {
        has_mask = 0; status = GE_STEP_AFTER_DONE;
    } else if (kind == GE_TSP && a == 0 && head == 0) {                          // tsp.py:203-211
        done = 1; reward = -(double)N; solved = 0; sol = -1.0;
        maskw = group_mask_word(d, g, adj, dest, rowh, visw, auxw, tail, 0);
        write_state = true;
    } else if (!(a_ok && ((oldm_a >> (a & 31)) & 1u))) {
        status = GE_STEP_INVALID; has_mask = 0;
    } else {
        write_state = true;
        const int aw = a >> 5;
        const uint32_t abit = 1u << (a & 31);
        const uint32_t rowa = W ? adj[(size_t)a * NW + lane] : 0u;                // N(a): the next mask / Densest's new edges
        double w = 0.0;
        bool nb = true;
        if (kind != GE_DENSEST_SUBGRAPH) {  // adj[head, a] by bit rank (ge_common.cuh:edge_weight_ranked)
            nb = (g.shfl(rowh, aw) >> (a & 31)) & 1u;
            uint32_t below = lane < aw ? rowh : (lane == aw ? (rowh & (abit - 1u)) : 0u);
            int rank = g.sum(__popc(below));
            if (nb) w = d.wsort[(size_t)b * d.MP + rp_head + rank];
        }
        const bool visa = (g.shfl(visw, aw) >> (a & 31)) & 1u;
        switch (kind) {
        case GE_SHORTEST_PATH: {                                                  // shortest_path.py:111-141
            reward = -w; cost += w;
            if (a == dest) { done = 1; solved = 1; }
            if (lane == aw) visw |= abit;
            head = a;
            maskw = group_mask_word(d, g, adj, dest, rowa, visw, auxw, tail, 0);
            if (!done && g.sum(__popc(maskw)) == 0) { done = 1; reward = -(double)N; solved = 0; }
            if (done) sol = cost;
            break; }
        case GE_LONGEST_PATH: {                                                   // longest_path.py:147-196
            if (d.parenting >= 1 && (!nb || visa)) { status = GE_STEP_INVALID; has_mask = 0; write_state = false; break; }
            reward = w; cost -= w; sol = cost;
            if (!nb || visa) { done = 1; solved = 0; reward = -2.0 * N; has_mask = 0; break; }   // :169-173 (parenting 0)
            head = a;
            if (lane == aw) visw |= abit;
            if (a == dest) { done = 1; solved = 1; }
            maskw = group_mask_word(d, g, adj, dest, rowa, visw, auxw, tail, 0);
            if (!done && g.sum(__popc(maskw)) == 0) { done = 1; reward = -2.0 * N; solved = 0; }
            break; }
        case GE_TSP: {                                                            // tsp.py:213-258
            reward = 0.0 - w; cost += w;
            if (lane == aw) visw |= abit;
            head = a;
            const int taken = g.sum(__popc(visw));
            if (taken == N && a == 0) { done = 1; solved = 1; }
            maskw = rowa & ~visw;
            if (taken < N - 1 && lane == 0) maskw &= ~1u;
            if (d.parenting >= 2) maskw = group_prune_tsp(d, g, adj, maskw, visw, tail);
            if (!done && g.sum(__popc(maskw)) == 0) { done = 1; reward -= 2.0 * N; solved = 0; }
            if (done) sol = cost;
            break; }
        case GE_DENSEST_SUBGRAPH: {                                               // densest_subgraph.py:135-196
            solved = 1;
            if (a == N - 1) { reward = 0.0; done = 1; sol = cost; break; }       // stop action: state and mask unchanged
            const int ne = g.sum(__popc(rowa & visw));
            auxw |= rowa;
            if (c.x == 0) reward = 0.0;
            else reward = ((double)(c.y + ne) / (double)(c.x + 1)) - ((double)c.y / (double)c.x);
            c.y += ne; c.x += 1;
            if (lane == aw) visw |= abit;
            cost = (double)c.y / (double)c.x;
            maskw = group_mask_word(d, g, adj, dest, rowa, visw, auxw, tail, c.x);
            if (c.x == d.n_choices) { done = 1; sol = cost; }
            break; }
        }
    }
    if (lane == 0) {
        out.reward[b] = (float)reward;
        ge_step_flags f;
        f.done = (uint8_t)done; f.solved = (int8_t)solved; f.status = (uint8_t)status; f.has_mask = (uint8_t)has_mask;
        out.flags[b] = f;
        out.solution_cost[b] = sol;
        if (d.traj) {
            u64 cs = d.traj[b];
            d.traj[b] = ((cs << 7) | (cs >> 57)) ^ (u64)(uint32_t)a ^ ((u64)done << 40) ^ ((u64)(solved & 3) << 44) ^ ((u64)status << 48);
        }
        if (status == GE_STEP_OK) {
            if (d.env_steps) d.env_steps[b] = nsteps + 1u;
            d.acc[2 * (size_t)d.acc_stride + b] += reward;
            if (done) {
                d.acc[b] += 1.0;
                if (solved == 1) d.acc[(size_t)d.acc_stride + b] += 1.0;
                if (sol == sol) d.acc[3 * (size_t)d.acc_stride + b] += sol;
            }
        }
    }
    const bool auto_reset = done && (d.flags & GE_FLAG_AUTO_RESET);
    if (auto_reset) {                                                            // tail of reset(): state init + cached first mask
        visw = (seeded && lane == (src >> 5)) ? (1u << (src & 31)) : 0u;
        auxw = 0;
        head = src;
        cost = 0.0;
        c = make_int4(0, 0, 0, 0);
        maskw = m0;
    } else if (!write_state) {
        return;
    }
    if (W) {
        d.node_bits[(size_t)b * NW + lane] = visw;
        if (d.node_bits2) d.node_bits2[(size_t)b * NW + lane] = auxw;
    }
    store_mask_word<G>(d, b, lane, maskw);
    if (lane == 0) {
        d.head[b] = head;
        d.cost[b] = cost;
        if (kind == GE_DENSEST_SUBGRAPH) *reinterpret_cast<int4 *>(d.counters + (size_t)b * 4) = c;
        if (done && !auto_reset) d.done[b] = 1;
    }
}

// reset(): state init + first mask, also recorded in mask0_bits for the auto-reset of the step kernel.
template <int G>
__global__ void __launch_bounds__(256) group_reset_kernel(ge_batch d, const uint8_t *__restrict__ select) {
    const Grp<G> g;
    const int lane = g.gl;
    const int b = blockIdx.x * (256 / G) + (int)threadIdx.x / G;
    if (b >= d.B) return;
    if (select && !select[b]) return;
    const int N = d.N, NW = d.NW, kind = d.kind;
    const bool W = lane < NW;
    const uint32_t tail = W ? tail_mask(N, lane) : 0u;
    const bool seeded = kind == GE_SHORTEST_PATH || kind == GE_LONGEST_PATH;
    const int src = seeded ? d.src[b] : 0;
    const uint32_t visw = (seeded && lane == (src >> 5)) ? (1u << (src & 31)) : 0u;
    const uint32_t roww = (W && kind != GE_DENSEST_SUBGRAPH) ? d.adj_bits[(size_t)b * d.ADJS + (size_t)src * NW + lane] : 0u;
    const int dest = seeded ? d.dest[b] : 0;
    uint32_t m = group_mask_word(d, g, d.adj_bits + (size_t)b * d.ADJS, dest, roww, visw, 0u, tail, 0);
    if (kind == GE_TSP && g.sum(__popc(m)) == 0 && lane == 0) m |= 1u;          // tsp.py:154-155
    if (W) {
        d.node_bits[(size_t)b * NW + lane] = visw;
        if (d.node_bits2) d.node_bits2[(size_t)b * NW + lane] = 0;
        if (d.mask0_bits) d.mask0_bits[(size_t)b * d.AW + lane] = m;
    }
    store_mask_word<G>(d, b, lane, m);
    if (lane == 0) {
        d.head[b] = src;
        d.cost[b] = 0.0;
        d.done[b] = 0;
        *reinterpret_cast<int4 *>(d.counters + (size_t)b * 4) = make_int4(0, 0, 0, 0);
    }
}

}  // namespace

// ------------------------------------------------------------------ host launchers (called from ge_api.cu)
bool ge_group_eligible(const ge_batch *d) {
    if (d->flags & GE_FLAG_FORCE_WARP) return false;
    if (!group_kind(*d) || d->N <= 64 || d->NW > 32 || !d->adj_bits) return false;
    if ((d->flags & GE_FLAG_AUTO_RESET) && !d->mask0_bits) return false;
    return d->kind == GE_DENSEST_SUBGRAPH || d->wsort != nullptr;
}

static int group_lanes(const ge_batch *d) { return d->NW <= 8 ? 8 : d->NW <= 16 ? 16 : 32; }

static int group_launched(const char *what) {
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? GE_OK : ge_set_error(GE_ERR_CUDA, "%s launch: %s", what, cudaGetErrorString(e));
}

int ge_group_step(const ge_batch *d, int32_t *actions, const ge_step_out *out, bool sampled, uint64_t seed, uint32_t t, cudaStream_t st) {
    const int G = group_lanes(d), per_block = 256 / G, blocks = (d->B + per_block - 1) / per_block;
    auto kernel = G == 8 ? (sampled ? group_step_kernel<true, 8> : group_step_kernel<false, 8>)
                : G == 16 ? (sampled ? group_step_kernel<true, 16> : group_step_kernel<false, 16>)
                          : (sampled ? group_step_kernel<true, 32> : group_step_kernel<false, 32>);
    ge_launch_step(kernel, dim3(blocks), dim3(256), 0, st, *d, actions, *out, seed, t);
    return group_launched("group_step_kernel");
}

int ge_group_reset(const ge_batch *d, const uint8_t *select, cudaStream_t st) {
    const int G = group_lanes(d), per_block = 256 / G, blocks = (d->B + per_block - 1) / per_block;
    auto kernel = G == 8 ? group_reset_kernel<8> : G == 16 ? group_reset_kernel<16> : group_reset_kernel<32>;
    kernel<<<blocks, 256, 0, st>>>(*d, select);
    return group_launched("group_reset_kernel");
}
