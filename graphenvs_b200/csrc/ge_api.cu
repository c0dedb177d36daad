// ge_api.cu -- kernels + extern "C" entry points of libgraphenvs_b200.so (sm_100a).
// See include/graphenvs_b200.h for the ABI and the reference interfaces each call replaces.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>

#include "ge_envs.cuh"

using namespace ge;

static thread_local char g_err[512] = "";

static int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

// shared with the other translation units of the library (ge_features.cu, ge_generate.cu)
extern "C" int ge_set_error(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define GE_CUDA_OK(expr)                                                                         \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess) return fail(GE_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(_e)); \
    } while (0)

__host__ __device__ static inline bool is_edge_kind(int kind) { return kind == GE_STEINER_TREE || kind == GE_MULTICAST_ROUTING; }
static bool uses_adj(int kind) {
    return kind == GE_SHORTEST_PATH || kind == GE_LONGEST_PATH || kind == GE_TSP || kind == GE_DENSEST_SUBGRAPH ||
           kind == GE_PERISHABLE_DELIVERY;
}

// ------------------------------------------------------------------ kernels
namespace {

// SAMPLED: draw the action from the current mask inside the kernel (ge_step_sampled) and publish it.
// MINB = resident blocks per SM the instantiation is compiled for (register cap 64 / 40 / 32).  The kernels
// are chains of dependent memory rounds, so occupancy buys throughput until spills cost more: measured
// per kind (TSP best at 8, DensestSubgraph at 6, DistributionCenter -- shared-memory limited -- at 4).
template <bool SAMPLED, int MINB>
__global__ void __launch_bounds__(GE_WPB * 32, MINB) step_kernel(ge_batch d, int32_t *__restrict__ actions, ge_step_out out,
                                                         int words_per_warp, uint64_t seed, uint32_t t) {
    extern __shared__ __align__(16) uint32_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * GE_WPB + warp;
    pdl_launch_dependents();   // programmatic dependent launch (ge_common.cuh): no-ops on a plain launch
    pdl_wait();
    if (b >= d.B) return;
    Scr s = carve(smem + (size_t)warp * words_per_warp, d);
    EnvPtrs p = env_ptrs(d, b);
    StepRes r;
    const uint32_t nsteps = d.env_steps ? d.env_steps[b] : 0u;
    int a;
    if (SAMPLED) {
        a = warp_sample(d.mask_bits + (size_t)b * d.AW, d.AW, lane, seed, (uint32_t)(d.env_id0 + b), t + nsteps);
        if (lane == 0) actions[b] = a;
    } else {
        a = actions[b];
    }
    if (d.done[b]) {  // only reachable with auto-reset off
        r.reward = 0.0; r.sol = __longlong_as_double(0x7ff8000000000000ll);
        r.done = 0; r.solved = -1; r.has_mask = 0; r.status = GE_STEP_AFTER_DONE;
    } else {
        step_env(d, p, s, lane, b, a, r);
    }
    if (lane == 0) {
        out.reward[b] = (float)r.reward;
        ge_step_flags f;
        f.done = (uint8_t)r.done; f.solved = (int8_t)r.solved; f.status = (uint8_t)r.status; f.has_mask = (uint8_t)r.has_mask;
        out.flags[b] = f;
        out.solution_cost[b] = r.sol;
        if (d.traj) {
            uint64_t cs = d.traj[b];
            cs = ((cs << 7) | (cs >> 57)) ^ (uint64_t)(uint32_t)a ^ ((uint64_t)r.done << 40) ^ ((uint64_t)(r.solved & 3) << 44) ^
                 ((uint64_t)r.status << 48);
            d.traj[b] = cs;
        }
        if (r.status == GE_STEP_OK) {
            if (d.env_steps) d.env_steps[b] = nsteps + 1u;
            d.acc[2 * (size_t)d.acc_stride + b] += r.reward;  // [4, B]: the per-step stream is one component wide
            if (r.done) {
                d.acc[b] += 1.0;
                if (r.solved == 1) d.acc[(size_t)d.acc_stride + b] += 1.0;
                if (r.sol == r.sol) d.acc[3 * (size_t)d.acc_stride + b] += r.sol;
            }
        }
    }
    if (r.done && (d.flags & GE_FLAG_AUTO_RESET)) {
        __syncwarp();
        reset_env(d, p, s, lane, b);
    }
}

__global__ void __launch_bounds__(GE_WPB * 32) reset_kernel(ge_batch d, const uint8_t *__restrict__ select, int words_per_warp) {
    extern __shared__ __align__(16) uint32_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * GE_WPB + warp;
    if (b >= d.B) return;
    if (select && !select[b]) return;
    Scr s = carve(smem + (size_t)warp * words_per_warp, d);
    EnvPtrs p = env_ptrs(d, b);
    reset_env(d, p, s, lane, b);
}

// Uniform choice among the valid mask bits (README.md:54-68 loop), counter-based RNG.
__global__ void __launch_bounds__(GE_WPB * 32) sample_kernel(ge_batch d, uint64_t seed, uint32_t t, int32_t *__restrict__ actions) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * GE_WPB + warp;
    if (b >= d.B) return;
    if (d.env_steps) t += d.env_steps[b];
    int action = warp_sample(d.mask_bits + (size_t)b * d.AW, d.AW, lane, seed, (uint32_t)(d.env_id0 + b), t);
    if (lane == 0) actions[b] = action;
}

// adjacency bit-matrix from CSR (load time).
__global__ void __launch_bounds__(GE_WPB * 32) adjacency_kernel(ge_batch d) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * GE_WPB + warp;
    if (b >= d.B) return;
    const int32_t *rp = d.row_ptr + (size_t)b * d.RP;
    const int32_t *col = d.col + (size_t)b * d.MP;
    if (d.esrc || d.rev) {  // edge-indexed derived arrays of the incremental kernels (ge_incr.cu)
        int32_t *esrc = d.esrc ? d.esrc + (size_t)b * d.MP : nullptr;
        int32_t *rev = d.rev ? d.rev + (size_t)b * d.MP : nullptr;
        for (int u = lane; u < d.N; u += 32)
            for (int e = rp[u]; e < rp[u + 1]; ++e) {
                if (esrc) esrc[e] = u;
                if (rev) {
                    int v = col[e], r = -1;
                    for (int k = rp[v]; k < rp[v + 1]; ++k)
                        if (col[k] == u) { r = k; break; }
                    rev[e] = r;
                }
            }
    }
    if (d.wmin && d.w64) {
        const double *w64 = d.w64 + (size_t)b * d.MP;
        double m = __longlong_as_double(0x7ff0000000000000ll);
        for (int e = lane; e < d.M; e += 32) m = fmin(m, w64[e]);
        for (int o = 16; o > 0; o >>= 1) m = fmin(m, __shfl_xor_sync(GE_FULL, m, o));
        if (lane == 0) d.wmin[b] = m;
    }
    if (!d.adj_bits) return;
    if (adj_tiled(d)) {  // lane-per-env family: tiles of 32 envs (ge_common.cuh:adj_tiled); lane u owns row u (+32)
        for (int u = lane; u < d.N; u += 32) {
            uint32_t lo = 0, hi = 0;
            for (int e = rp[u]; e < rp[u + 1]; ++e) {
                int c = col[e];
                if (c < 32) lo |= 1u << c; else hi |= 1u << (c - 32);
            }
            d.adj_bits[adj_word_index(d, b, u, 0)] = lo;
            if (d.NW > 1) d.adj_bits[adj_word_index(d, b, u, 1)] = hi;
        }
    } else {
    uint32_t *adj = d.adj_bits + (size_t)b * d.ADJS;
    for (int i = lane; i < d.ADJS; i += 32) adj[i] = 0;
    __syncwarp();
    __threadfence_block();
    for (int u = lane; u < d.N; u += 32)
        for (int e = rp[u]; e < rp[u + 1]; ++e) {
            int c = col[e];
            atomicOr(&adj[(size_t)u * d.NW + (c >> 5)], 1u << (c & 31));
        }
    }
    if (d.wsort && d.w64 && !adj_tiled(d)) {  // weights in ascending-destination order per row: O(1) adj[u, v] lookup by bit rank
        __syncwarp();
        __threadfence_block();
        const double *w64 = d.w64 + (size_t)b * d.MP;
        double *ws = d.wsort + (size_t)b * d.MP;
        const uint32_t *adj = d.adj_bits + (size_t)b * d.ADJS;
        for (int u = 0; u < d.N; ++u) {
            const int lo = rp[u], hi = rp[u + 1];
            const uint32_t *row = adj + (size_t)u * d.NW;
            for (int e = lo + lane; e < hi; e += 32) {
                const int v = col[e];
                int rank = __popc(row[v >> 5] & ((1u << (v & 31)) - 1u));
                for (int w = 0; w < (v >> 5); ++w) rank += __popc(row[w]);
                ws[lo + rank] = w64[e];
            }
        }
    }
    if (d.wmat && d.w64) {  // dense float64 weights (the reference's self.adj, shortest_path.py:82)
        double *wm = d.wmat + (size_t)b * d.N * d.N;
        const double *w64 = d.w64 + (size_t)b * d.MP;
        for (int i = lane; i < d.N * d.N; i += 32) wm[i] = 0.0;
        __syncwarp();
        __threadfence_block();
        for (int u = lane; u < d.N; u += 32)
            for (int e = rp[u]; e < rp[u + 1]; ++e) wm[(size_t)u * d.N + col[e]] = w64[e];
    }
}

// Reference wire format (utils.py:87-88): [nodes.ravel | edges.ravel | edge_links.ravel] float32.
// MODE 0 writes that flat vector; MODE 1 writes the three sections to separate tensors -- x float32[count, N, F],
// edge_attr float32[count, M, Fe], edge_index int64[count, M, 2] -- i.e. what utils.devectorize_graph
// (utils.py:14-23) would slice out of the flat vector, without the float32 round trip of the indices; MODE 2
// writes x only (the node columns are the part of the observation a step changes; edge tensors are static or,
// for Multicast's IS_TAKEN column, one bit per step).  One CTA per env.  No per-element integer division and
// no per-endpoint binary search: the (node, column) pair of a thread advances by a fixed stride, the edge
// sections walk the CSR rows (warp per row), so the source of an edge is the row being walked.
__device__ __forceinline__ float node_value(const ge_batch &d, int b, int v, int c, int dyn, const uint32_t *vis, const uint32_t *aux,
                                            const uint32_t *tgt, int src, int dest, float maxd) {
    const int N = d.N;
    if (c >= dyn) return d.features ? d.features[((size_t)b * N + v) * 5 + (c - dyn)] : 0.f;
    const bool bit = (vis[v >> 5] >> (v & 31)) & 1u;
    switch (d.kind) {
    case GE_SHORTEST_PATH: return c == 0 ? (float)bit : (float)(v == dest);
    case GE_LONGEST_PATH:
        if (c == 0) return (float)bit;
        return (v == dest) ? 1.f : ((d.parenting == 0 && v == src) ? 2.f : 0.f);
    case GE_STEINER_TREE: return c == 0 ? (float)bit : (float)((tgt[v >> 5] >> (v & 31)) & 1u);
    case GE_TSP:
        if (c == 0) return (float)bit;
        if (c == 1) return (float)(v == 0);
        return d.node_xy ? d.node_xy[((size_t)b * N + v) * 2 + (c - 2)] : 0.f;
    case GE_MAX_INDEPENDENT_SET: return c == 0 ? d.node_cost[(size_t)b * N + v] : (float)bit;
    case GE_DENSEST_SUBGRAPH: return (float)bit;
    case GE_MULTICAST_ROUTING:
        if (c == 0) return (float)bit;
        if (c == 1) return (float)((tgt[v >> 5] >> (v & 31)) & 1u);
        if (c == 2) return maxd;
        return d.dist32[(size_t)b * N + v];
    case GE_DISTRIBUTION_CENTER:
        if (c == 0) return d.node_cost[(size_t)b * N + v];
        if (c == 1) return (float)bit;
        if (c == 2) return (float)((tgt[v >> 5] >> (v & 31)) & 1u);
        if (c == 3) return (float)((aux[v >> 5] >> (v & 31)) & 1u);
        return (float)d.max_distance;
    case GE_PERISHABLE_DELIVERY: {   // perishable_product_delivery.py:38-41: IS_HEAD | HAS_P[5] | NEEDS_P[5] | TIME_LEFT[5]
        if (c == 0) return (float)(v == d.head[b]);
        const int i = (c - 1) % 5, grp = (c - 1) / 5, P = d.n_dests;
        if (i >= P) return 0.f;
        const int st = (d.counters[(size_t)b * 4] >> (2 * i)) & 3;
        const int32_t *tg = d.targets + (size_t)b * d.n_targets;
        if (grp == 0) return st == 0 ? (float)(v == tg[i]) : (st == 1 ? -1.f : 0.f);
        if (grp == 1) return st == 2 ? 0.f : (float)(v == tg[P + i]);
        return st == 2 ? 0.f : maxd; }
    }
    return 0.f;
}

template <int MODE>
__global__ void __launch_bounds__(256) obs_kernel(ge_batch d, int env_lo, int count, float *__restrict__ out, int L, float *__restrict__ out_e,
                                                long long *__restrict__ out_i, int warp_per_env) {
    // One CTA per env, or -- small graphs, where a CTA per env is ~1 KB of output behind a block launch (65,536 blocks of two
    // trips each at config 2: 138 us for 92 MB) -- one WARP per env, eight envs per CTA.  (gt, gn) = this thread's index in / the
    // size of the group that writes one env.
    const int gn = warp_per_env ? 32 : (int)blockDim.x, gt = warp_per_env ? ((int)threadIdx.x & 31) : (int)threadIdx.x;
    const int slot = warp_per_env ? (int)blockIdx.x * ((int)blockDim.x >> 5) + ((int)threadIdx.x >> 5) : (int)blockIdx.x;
    if (slot >= count) return;
    const int b = env_lo + slot;
    const int N = d.N, M = d.M, kind = d.kind;
    int dyn;
    switch (kind) {
    case GE_TSP: case GE_MULTICAST_ROUTING: dyn = 4; break;
    case GE_DENSEST_SUBGRAPH: dyn = 1; break;
    case GE_DISTRIBUTION_CENTER: dyn = 5; break;
    case GE_PERISHABLE_DELIVERY: dyn = 16; break;
    default: dyn = 2;
    }
    const int F = dyn + 5, Fe = is_edge_kind(kind) ? 2 : 1;
    const int NF = N * F, MF = M * Fe;
    float *o = out + (size_t)slot * (MODE == 0 ? (size_t)L : (size_t)NF);  // the flat vector, or the node section
    const uint32_t *vis = d.node_bits + (size_t)b * d.NW;
    const uint32_t *aux = d.node_bits2 ? d.node_bits2 + (size_t)b * d.NW : nullptr;
    const uint32_t *tgt = d.target_bits ? d.target_bits + (size_t)b * d.NW : nullptr;
    const bool seeded = kind == GE_SHORTEST_PATH || kind == GE_LONGEST_PATH;
    const int src = seeded ? d.src[b] : 0, dest = seeded ? d.dest[b] : 0;
    const float maxd = (kind == GE_MULTICAST_ROUTING || kind == GE_PERISHABLE_DELIVERY) ? d.max_dist32[b] : 0.f;
    if (!warp_per_env) {
        // CTA per env (large graphs): one THREAD per node evaluates the node's F columns once -- the membership bits and the kind
        // dispatch are per node, not per element (the per-element form was instruction-bound: 2.1 ms for DistributionCenter's
        // 2.6 GB of x at config 5) -- into a shared tile, which the block then streams out coalesced.
        __shared__ __align__(16) float tile[256 * 21];
        for (int v0 = 0; v0 < N; v0 += 256) {
            const int v = v0 + (int)threadIdx.x;
            if (v < N) {
                float *t = tile + (int)threadIdx.x * F;
                const bool bit = (vis[v >> 5] >> (v & 31)) & 1u;
                const bool tb = tgt ? ((tgt[v >> 5] >> (v & 31)) & 1u) : false;
                switch (kind) {
                case GE_SHORTEST_PATH: t[0] = (float)bit; t[1] = (float)(v == dest); break;
                case GE_LONGEST_PATH: t[0] = (float)bit; t[1] = (v == dest) ? 1.f : ((d.parenting == 0 && v == src) ? 2.f : 0.f); break;
                case GE_STEINER_TREE: t[0] = (float)bit; t[1] = (float)tb; break;
                case GE_TSP:
                    t[0] = (float)bit; t[1] = (float)(v == 0);
                    t[2] = d.node_xy ? d.node_xy[((size_t)b * N + v) * 2] : 0.f;
                    t[3] = d.node_xy ? d.node_xy[((size_t)b * N + v) * 2 + 1] : 0.f;
                    break;
                case GE_MAX_INDEPENDENT_SET: t[0] = d.node_cost[(size_t)b * N + v]; t[1] = (float)bit; break;
                case GE_DENSEST_SUBGRAPH: t[0] = (float)bit; break;
                case GE_MULTICAST_ROUTING: t[0] = (float)bit; t[1] = (float)tb; t[2] = maxd; t[3] = d.dist32[(size_t)b * N + v]; break;
                case GE_DISTRIBUTION_CENTER:
                    t[0] = d.node_cost[(size_t)b * N + v]; t[1] = (float)bit; t[2] = (float)tb;
                    t[3] = (float)((aux[v >> 5] >> (v & 31)) & 1u); t[4] = (float)d.max_distance;
                    break;
                default:   // PerishableProductDelivery: 16 columns through the per-element rule
                    for (int c = 0; c < dyn; ++c) t[c] = node_value(d, b, v, c, dyn, vis, aux, tgt, src, dest, maxd);
                }
                const float *f5 = d.features ? d.features + ((size_t)b * N + v) * 5 : nullptr;
#pragma unroll
                for (int c = 0; c < 5; ++c) t[dyn + c] = f5 ? f5[c] : 0.f;
            }
            __syncthreads();
            const int nvals = min(256, N - v0) * F;
            float *ov = o + (size_t)v0 * F;
            if (((reinterpret_cast<size_t>(ov) | (size_t)nvals * 4) & 15) == 0) {   // 128-bit stores (the copy-out was 39 % of the instructions)
                const float4 *t4 = reinterpret_cast<const float4 *>(tile);
                float4 *o4 = reinterpret_cast<float4 *>(ov);
                for (int i = threadIdx.x; i < (nvals >> 2); i += 256) o4[i] = t4[i];
            } else {
                for (int i = threadIdx.x; i < nvals; i += 256) ov[i] = tile[i];
            }
            __syncthreads();
        }
    } else {   // node section, warp per env: element i = (v, c) with v = i / F; the pair advances by (32 / F, 32 % F) per trip
        int v = gt / F, c = gt - v * F;
        const int dv = gn / F, dc = gn - dv * F;
        for (int i = gt; i < NF; i += gn) {
            o[i] = node_value(d, b, v, c, dyn, vis, aux, tgt, src, dest, maxd);
            v += dv; c += dc;
            if (c >= F) { c -= F; ++v; }
        }
    }
    if (MODE == 2) return;
    float *oe = MODE == 0 ? o + NF : out_e + (size_t)slot * MF;
    {   // edge feature section: column 0 = weight (1 for the unweighted kinds), column 1 = IS_TAKEN (Multicast) / zeros
        const bool unit = kind == GE_MAX_INDEPENDENT_SET || kind == GE_DENSEST_SUBGRAPH;
        const float *w32 = d.w32 ? d.w32 + (size_t)b * d.MP : nullptr;
        const double *w64 = d.w64 ? d.w64 + (size_t)b * d.MP : nullptr;
        const uint32_t *eb = kind == GE_MULTICAST_ROUTING ? d.edge_bits + (size_t)b * d.MW : nullptr;
        for (int e = gt; e < M; e += gn) {
            const float w = unit ? 1.f : (w32 ? w32[e] : (float)w64[e]);
            if (Fe == 1) oe[e] = w;
            else {
                const float tk = eb ? (float)((eb[e >> 5] >> (e & 31)) & 1u) : 0.f;
                if (MODE == 1) reinterpret_cast<float2 *>(oe)[e] = make_float2(w, tk);   // own tensor: 8-byte aligned
                else { oe[2 * e] = w; oe[2 * e + 1] = tk; }                             // flat vector: any float offset
            }
        }
    }
    {   // edge_links section: (source, destination) per directed edge, CSR order; one warp per row
        const int32_t *rp = d.row_ptr + (size_t)b * d.RP;
        const int32_t *col = d.col + (size_t)b * d.MP;
        const int warp = warp_per_env ? 0 : (int)threadIdx.x >> 5, lane = threadIdx.x & 31, nw = gn >> 5;
        float *ol = o + NF + MF;
        long long *oi = out_i + (size_t)slot * 2 * M;
        for (int u = warp; u < N; u += nw) {
            const int lo = rp[u], hi = rp[u + 1];
            for (int e = lo + lane; e < hi; e += 32) {
                const int v = col[e];
                if (MODE == 1) reinterpret_cast<longlong2 *>(oi)[e] = make_longlong2(u, v);
                else { ol[2 * e] = (float)u; ol[2 * e + 1] = (float)v; }
            }
        }
    }
}

// ---- reset-time derived data ---------------------------------------------------------------
// SSSP from src: heuristics (shortest_path.py:90, longest_path.py:105, steiner_tree.py:79) and the
// Multicast max_distance draw (multicast_routing.py:98-103) given the reference's U(0,1) sample.
__global__ void __launch_bounds__(GE_WPB * 32) prep_sssp_kernel(ge_batch d, int what, const double *__restrict__ u01, int words_per_warp) {
    extern __shared__ __align__(16) uint32_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * GE_WPB + warp;
    if (b >= d.B) return;
    Scr s = carve(smem + (size_t)warp * words_per_warp, d);
    int src = (d.kind == GE_MULTICAST_ROUTING) ? 0 : d.src[b];
    sssp_warp(d, b, lane, s, src, 0.0, false);
    __syncwarp();
    if (d.kind == GE_SHORTEST_PATH || d.kind == GE_LONGEST_PATH) {
        if (lane == 0 && (what & 1)) {
            double v = __longlong_as_double((long long)s.q[d.dest[b]]);
            d.heuristic[b] = d.kind == GE_LONGEST_PATH ? -v : v;
        }
    } else if (d.kind == GE_STEINER_TREE) {  // n_dests == 1: the single target
        if (what & 1) {
            const uint32_t *tg = d.target_bits + (size_t)b * d.NW;
            int first = 0x7fffffff;
            for (int w = lane; w < d.NW; w += 32)
                if (tg[w]) first = min(first, (w << 5) + __ffs(tg[w]) - 1);
            first = __reduce_min_sync(GE_FULL, first);
            if (lane == 0) d.heuristic[b] = __longlong_as_double((long long)s.q[first]);
        }
    } else if (d.kind == GE_MULTICAST_ROUTING) {
        if (what & 2) {
            const uint32_t *tg = d.target_bits + (size_t)b * d.NW;
            double far_node = 0.0, far_tgt = 0.0;
            for (int v = lane; v < d.N; v += 32) {
                double dv = __longlong_as_double((long long)s.q[v]);
                far_node = fmax(far_node, dv);
                if ((tg[v >> 5] >> (v & 31)) & 1u) far_tgt = fmax(far_tgt, dv);
            }
            for (int o = 16; o > 0; o >>= 1) {
                far_node = fmax(far_node, __shfl_xor_sync(GE_FULL, far_node, o));
                far_tgt = fmax(far_tgt, __shfl_xor_sync(GE_FULL, far_tgt, o));
            }
            if (lane == 0) {
                const double u = u01 ? u01[b] : (double)d.max_dist32[b];   // NULL: the draw ge_generate parked in max_dist32
                double md = __dadd_rn(__dmul_rn(u, __dsub_rn(far_node, far_tgt)), far_tgt);
                d.max_dist32[b] = (float)md;
            }
        }
    }
}

// PerishableProductDelivery eval heuristic (perishable_product_delivery.py:147-153): for every product, Dijkstra distance
// head(0) -> pickup plus pickup -> dropoff (curr_node is never advanced in the reference), summed in product order.
__global__ void __launch_bounds__(GE_WPB * 32) prep_ppd_kernel(ge_batch d, int words_per_warp) {
    extern __shared__ __align__(16) uint32_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * GE_WPB + warp;
    if (b >= d.B) return;
    Scr s = carve(smem + (size_t)warp * words_per_warp, d);
    const int P = d.n_dests;
    const int32_t *tg = d.targets + (size_t)b * d.n_targets;
    double from_head[5];
    sssp_warp(d, b, lane, s, 0, 0.0, false);
    __syncwarp();
    for (int i = 0; i < P; ++i) from_head[i] = __longlong_as_double((long long)s.q[tg[i]]);
    __syncwarp();
    double total = 0.0;
    for (int i = 0; i < P; ++i) {
        sssp_warp(d, b, lane, s, tg[i], 0.0, false);
        __syncwarp();
        total += from_head[i];
        total += __longlong_as_double((long long)s.q[tg[P + i]]);
        __syncwarp();
    }
    if (lane == 0) d.heuristic[b] = total;
}

// MST total weight (steiner_tree.py:81): Prim in fp64; the multiset of MST weights is
// tie-independent, the sum is compared within 1e-5 (summation order differs from Kruskal's).
__global__ void __launch_bounds__(GE_WPB * 32) prep_mst_kernel(ge_batch d, int words_per_warp) {
    extern __shared__ __align__(16) uint32_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * GE_WPB + warp;
    if (b >= d.B) return;
    Scr s = carve(smem + (size_t)warp * words_per_warp, d);
    EnvPtrs p = env_ptrs(d, b);
    const u64 INF = 0x7ff0000000000000ull;
    for (int v = lane; v < d.N; v += 32) s.q[v] = INF;
    for (int w = lane; w < d.NW; w += 32) s.t0[w] = 0;  // in-tree set
    __syncwarp();
    if (lane == 0) s.q[0] = 0ull;
    __syncwarp();
    double total = 0.0;
    for (int it = 0; it < d.N; ++it) {
        u64 best = ~0ull;  // (key bits, node) packed: keys are non-negative doubles -> order preserving
        int bestv = -1;
        for (int v = lane; v < d.N; v += 32)
            if (!tbit(s.t0, v) && s.q[v] < best) { best = s.q[v]; bestv = v; }
        for (int o = 16; o > 0; o >>= 1) {
            u64 ob = __shfl_xor_sync(GE_FULL, best, o);
            int ov = __shfl_xor_sync(GE_FULL, bestv, o);
            if (ob < best || (ob == best && ov >= 0 && (bestv < 0 || ov < bestv))) { best = ob; bestv = ov; }
        }
        if (bestv < 0 || best == INF) break;  // disconnected remainder
        total += __longlong_as_double((long long)best);
        if (lane == 0) s.t0[bestv >> 5] |= 1u << (bestv & 31);
        __syncwarp();
        int lo = p.rp[bestv], hi = p.rp[bestv + 1];
        for (int e = lo + lane; e < hi; e += 32) {
            int v = p.col[e];
            if (!tbit(s.t0, v)) atomicMin(&s.q[v], (u64)__double_as_longlong(p.w64[e]));
        }
        __syncwarp();
    }
    if (lane == 0) d.heuristic[b] = total;
}

// DistributionCenter in-range tables (distribution_center.py:113-116): one warp per (env, target).
__global__ void __launch_bounds__(GE_WPB * 32) prep_inrange_kernel(ge_batch d, int words_per_warp) {
    extern __shared__ __align__(16) uint32_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long job = (long long)blockIdx.x * GE_WPB + warp;
    if (job >= (long long)d.B * d.n_targets) return;
    const int b = (int)(job / d.n_targets), t = (int)(job % d.n_targets);
    Scr s = carve(smem + (size_t)warp * words_per_warp, d);
    int node = d.targets[(size_t)b * d.n_targets + t];
    cutoff_reach(d, b, lane, s, node);
    __syncwarp();
    uint32_t *row = d.in_range + ((size_t)b * d.n_targets + t) * d.NW;
    for (int w = lane; w < d.NW; w += 32) row[w] = s.t2[w];
}

// Packed mask -> byte view (torch.bool [B, AP]) for envs [env_lo, env_lo + count): 16 mask entries per 128-bit store.
__global__ void __launch_bounds__(256) mask_bytes_kernel(ge_batch d, int env_lo, long long total16) {
    const int per_env = d.AP >> 4;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total16; i += (long long)gridDim.x * blockDim.x) {
        const int b = env_lo + (int)(i / per_env), c = (int)(i % per_env);
        const uint32_t word = c < 2 * d.AW ? d.mask_bits[(size_t)b * d.AW + (c >> 1)] : 0u;
        const uint32_t bits = (word >> ((c & 1) * 16)) & 0xffffu;
        reinterpret_cast<uint4 *>(d.mask_bytes + (size_t)b * d.AP)[c] =
            make_uint4(expand4(bits), expand4(bits >> 4), expand4(bits >> 8), expand4(bits >> 12));
    }
}

__global__ void stats_kernel(ge_batch d, double *out4) {
    __shared__ double sh[4][32];
    double a[4] = {0, 0, 0, 0};
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < d.B; b += gridDim.x * blockDim.x)
        for (int k = 0; k < 4; ++k) a[k] += d.acc[(size_t)k * d.acc_stride + b];
    for (int k = 0; k < 4; ++k)
        for (int o = 16; o > 0; o >>= 1) a[k] += __shfl_xor_sync(GE_FULL, a[k], o);
    int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) for (int k = 0; k < 4; ++k) sh[k][warp] = a[k];
    __syncthreads();
    if (warp == 0) {
        for (int k = 0; k < 4; ++k) {
            double v = lane < (int)(blockDim.x >> 5) ? sh[k][lane] : 0.0;
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(GE_FULL, v, o);
            if (lane == 0) atomicAdd(&out4[k], v);
        }
    }
}

}  // namespace

// lane-per-env kernels for N <= 64 (ge_lane.cu)
bool ge_lane_eligible(const ge_batch *d);
int ge_lane_step(const ge_batch *d, int32_t *actions, const ge_step_out *out, bool sampled, uint64_t seed, uint32_t t, cudaStream_t st);
int ge_lane_reset(const ge_batch *d, const uint8_t *select, cudaStream_t st);
int ge_lane_sample(const ge_batch *d, uint64_t seed, uint32_t t, int32_t *actions, cudaStream_t st);
// group-per-env row-mask kernels for 64 < N <= 1024 (ge_group.cu)
bool ge_group_eligible(const ge_batch *d);
int ge_group_step(const ge_batch *d, int32_t *actions, const ge_step_out *out, bool sampled, uint64_t seed, uint32_t t, cudaStream_t st);
int ge_group_reset(const ge_batch *d, const uint8_t *select, cudaStream_t st);
// incremental-mask kernels (ge_incr.cu)
bool ge_incr_eligible(const ge_batch *d);
int ge_incr_step(const ge_batch *d, int32_t *actions, const ge_step_out *out, bool sampled, uint64_t seed, uint32_t t, cudaStream_t st);
int ge_incr_reset(const ge_batch *d, const uint8_t *select, cudaStream_t st);

// dedicated DistributionCenter kernels (ge_dc.cu)
bool ge_dc_eligible(const ge_batch *d);
int ge_dc_step(const ge_batch *d, int32_t *actions, const ge_step_out *out, bool sampled, uint64_t seed, uint32_t t, cudaStream_t st);
int ge_dc_reset(const ge_batch *d, const uint8_t *select, cudaStream_t st);
int ge_dc_build_edges(const ge_batch *d, cudaStream_t st);
// PerishableProductDelivery (ge_ppd.cu)
int ge_ppd_step(const ge_batch *d, int32_t *actions, const ge_step_out *out, bool sampled, uint64_t seed, uint32_t t, cudaStream_t st);
int ge_ppd_reset(const ge_batch *d, const uint8_t *select, cudaStream_t st);
bool ge_ppd_lane(const ge_batch *d);
// eval heuristic kernels (ge_heuristics.cu)
int ge_heuristics_launch(const ge_batch *d, int what, cudaStream_t st);

// ------------------------------------------------------------------ host side
static int check_batch(const ge_batch *d) {
    if (!d) return fail(GE_ERR_ARG, "null batch");
    if (d->kind < 0 || d->kind > 8) return fail(GE_ERR_ARG, "unknown kind %d", d->kind);
    if (d->B <= 0 || d->N < 2 || d->M < 0) return fail(GE_ERR_ARG, "bad shape B=%d N=%d M=%d", d->B, d->N, d->M);
    if (d->N > 4096) return fail(GE_ERR_UNSUPPORTED, "N=%d > 4096 not supported", d->N);
    if (d->NW != (d->N + 31) / 32 || d->MW != (d->M + 31) / 32) return fail(GE_ERR_ARG, "layout not filled (call ge_fill_layout)");
    if (d->acc_stride < d->B) return fail(GE_ERR_ARG, "acc_stride %d < B %d (call ge_fill_layout)", d->acc_stride, d->B);
    return GE_OK;
}

static int launch_cfg(const ge_batch *d, int jobs, int *blocks, int *wpw, size_t *smem) {
    *wpw = scratch_words(*d);
    *smem = (size_t)(*wpw) * GE_WPB * sizeof(uint32_t);
    *blocks = (jobs + GE_WPB - 1) / GE_WPB;
    if (*smem > 227 * 1024) return fail(GE_ERR_UNSUPPORTED, "graph too large for per-warp shared scratch (%zu bytes)", *smem);
    return GE_OK;
}

// Opt-in dynamic shared memory above 48 KB, remembered per kernel so that repeated (and captured)
// launches make no attribute call.  Shared with ge_lane.cu.
int ge_grant_smem(const void *kernel, size_t smem) {
    static struct { const void *k; size_t granted; } table[32];
    static int n = 0;
    static std::mutex mu;
    if (smem <= 48 * 1024) return GE_OK;
    std::lock_guard<std::mutex> lock(mu);
    int i = 0;
    for (; i < n; ++i) if (table[i].k == kernel) break;
    if (i == n) {
        if (n == 32) return fail(GE_ERR_ARG, "kernel table full");
        table[n].k = kernel; table[n].granted = 48 * 1024; ++n;
    }
    if (smem > table[i].granted) {
        GE_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        table[i].granted = smem;
    }
    return GE_OK;
}
template <class K>
static int set_smem(K kernel, size_t smem) { return ge_grant_smem((const void *)kernel, smem); }

extern "C" {

int ge_abi_version(void) { return GE_ABI_VERSION; }
const char *ge_last_error(void) { return g_err; }

int ge_fill_layout(ge_batch *d) {
    if (!d) return fail(GE_ERR_ARG, "null batch");
    d->NW = (d->N + 31) / 32;
    d->MW = (d->M + 31) / 32;
    d->acc_stride = d->B;
    d->A = is_edge_kind(d->kind) ? d->M : d->N;
    d->AW = (d->A + 31) / 32;
    d->AP = (d->A + 15) & ~15;
    d->RP = (d->N + 1 + 3) & ~3;
    d->MP = (d->M + 3) & ~3;
    if (d->MP == 0) d->MP = 4;
    // adjacency bit-matrix stride (words per env).  N <= 64 keeps the odd / 2 x odd stride of the first layout;
    // the lane-per-env family stores those matrices in tiles of 32 envs (ge_common.cuh:adj_tiled), for which
    // B rounded up to 32 envs of ADJS words is enough room.  Larger graphs keep 16-byte alignment.
    if (d->NW == 1) d->ADJS = d->N | 1;
    else if (d->NW == 2) d->ADJS = 2 * (d->N | 1);
    else d->ADJS = (d->N * d->NW + 3) & ~3;
    return GE_OK;
}

int ge_step_smem_bytes(const ge_batch *d) { return scratch_words(*d) * GE_WPB * (int)sizeof(uint32_t); }

int ge_build_adjacency(const ge_batch *d, void *stream) {
    GE_NVTX("ge_build_adjacency");
    int rc = check_batch(d);
    if (rc) return rc;
    if (!d->adj_bits && !d->rev && !d->esrc && !d->wmin) return fail(GE_ERR_ARG, "no derived array requested (adj_bits / rev / esrc / wmin are null)");
    adjacency_kernel<<<(d->B + GE_WPB - 1) / GE_WPB, GE_WPB * 32, 0, (cudaStream_t)stream>>>(*d);
    GE_CUDA_OK(cudaGetLastError());
    return GE_OK;
}

int ge_prepare(const ge_batch *d, int what, const double *u01, void *stream) {
    GE_NVTX("ge_prepare");
    int rc = check_batch(d);
    if (rc) return rc;
    int blocks, wpw;
    size_t smem;
    cudaStream_t st = (cudaStream_t)stream;
    if ((what & 3) && !d->w64) return fail(GE_ERR_ARG, "ge_prepare needs w64");
    if ((what & 8) && !d->w64 && d->kind != GE_MAX_INDEPENDENT_SET) return fail(GE_ERR_ARG, "ge_prepare needs w64");
    if (what & 1) {
        bool sssp = d->kind == GE_SHORTEST_PATH || d->kind == GE_LONGEST_PATH || (d->kind == GE_STEINER_TREE && d->n_dests == 1);
        bool mst = d->kind == GE_STEINER_TREE && d->n_dests == d->N - 1;
        if (sssp) {
            if ((rc = launch_cfg(d, d->B, &blocks, &wpw, &smem))) return rc;
            if ((rc = set_smem(prep_sssp_kernel, smem))) return rc;
            prep_sssp_kernel<<<blocks, GE_WPB * 32, smem, st>>>(*d, 1, nullptr, wpw);
        } else if (mst) {
            if ((rc = launch_cfg(d, d->B, &blocks, &wpw, &smem))) return rc;
            if ((rc = set_smem(prep_mst_kernel, smem))) return rc;
            prep_mst_kernel<<<blocks, GE_WPB * 32, smem, st>>>(*d, wpw);
        } else if (d->kind == GE_PERISHABLE_DELIVERY) {
            if ((rc = launch_cfg(d, d->B, &blocks, &wpw, &smem))) return rc;
            if ((rc = set_smem(prep_ppd_kernel, smem))) return rc;
            prep_ppd_kernel<<<blocks, GE_WPB * 32, smem, st>>>(*d, wpw);
        } else if (d->kind == GE_MULTICAST_ROUTING) {
            if ((rc = ge_heuristics_launch(d, 1, st))) return rc;
        } else if (d->kind == GE_STEINER_TREE || d->kind == GE_TSP) {
            return fail(GE_ERR_UNSUPPORTED, "the reference's Kou / Christofides value is defined by networkx iteration order and is not "
                                            "provided; ask for the labelled alternative (what bit 3 -> heuristic_alt)");
        }
        GE_CUDA_OK(cudaGetLastError());
    }
    if ((what & 8) && (d->kind == GE_STEINER_TREE || d->kind == GE_TSP || d->kind == GE_MAX_INDEPENDENT_SET)) {
        if ((rc = ge_heuristics_launch(d, 8, st))) return rc;
    }
    if ((what & 2) && d->kind == GE_MULTICAST_ROUTING) {
        if ((rc = launch_cfg(d, d->B, &blocks, &wpw, &smem))) return rc;
        if ((rc = set_smem(prep_sssp_kernel, smem))) return rc;
        prep_sssp_kernel<<<blocks, GE_WPB * 32, smem, st>>>(*d, 2, u01, wpw);
        GE_CUDA_OK(cudaGetLastError());
    }
    if ((what & 16) && d->kind == GE_DISTRIBUTION_CENTER) {
        if ((rc = ge_dc_build_edges(d, st))) return rc;
    }
    if ((what & 4) && d->kind == GE_DISTRIBUTION_CENTER && d->n_targets > 0) {
        if (!d->w64) return fail(GE_ERR_ARG, "in-range tables need w64");
        long long jobs = (long long)d->B * d->n_targets;
        if (jobs > 0x7fffffffLL * GE_WPB) return fail(GE_ERR_UNSUPPORTED, "too many (env,target) jobs");
        wpw = scratch_words(*d);
        smem = (size_t)wpw * GE_WPB * sizeof(uint32_t);
        if ((rc = set_smem(prep_inrange_kernel, smem))) return rc;
        prep_inrange_kernel<<<(unsigned)((jobs + GE_WPB - 1) / GE_WPB), GE_WPB * 32, smem, st>>>(*d, wpw);
        GE_CUDA_OK(cudaGetLastError());
    }
    return GE_OK;
}

int ge_reset(const ge_batch *d, const uint8_t *select, void *stream) {
    GE_NVTX("ge_reset");
    int rc = check_batch(d);
    if (rc) return rc;
    if (uses_adj(d->kind) && !d->adj_bits) return fail(GE_ERR_ARG, "kind %d needs adj_bits (ge_build_adjacency)", d->kind);
    if (d->kind == GE_PERISHABLE_DELIVERY) return ge_ppd_reset(d, select, (cudaStream_t)stream);
    if (ge_lane_eligible(d)) return ge_lane_reset(d, select, (cudaStream_t)stream);
    if (ge_group_eligible(d)) return ge_group_reset(d, select, (cudaStream_t)stream);
    if (ge_incr_eligible(d)) return ge_incr_reset(d, select, (cudaStream_t)stream);
    if (ge_dc_eligible(d)) return ge_dc_reset(d, select, (cudaStream_t)stream);
    int blocks, wpw;
    size_t smem;
    if ((rc = launch_cfg(d, d->B, &blocks, &wpw, &smem))) return rc;
    if ((rc = set_smem(reset_kernel, smem))) return rc;
    reset_kernel<<<blocks, GE_WPB * 32, smem, (cudaStream_t)stream>>>(*d, select, wpw);
    GE_CUDA_OK(cudaGetLastError());
    return GE_OK;
}

static int step_impl(const ge_batch *d, int32_t *actions, const ge_step_out *out, bool sampled, uint64_t seed, uint32_t t,
                     void *stream) {
    int rc = check_batch(d);
    if (rc) return rc;
    if (!actions || !out || !out->reward || !out->flags || !out->solution_cost) return fail(GE_ERR_ARG, "null step buffers");
    if (d->kind == GE_PERISHABLE_DELIVERY) return ge_ppd_step(d, actions, out, sampled, seed, t, (cudaStream_t)stream);
    if (ge_lane_eligible(d)) return ge_lane_step(d, actions, out, sampled, seed, t, (cudaStream_t)stream);
    if (ge_group_eligible(d)) return ge_group_step(d, actions, out, sampled, seed, t, (cudaStream_t)stream);
    if (ge_incr_eligible(d)) return ge_incr_step(d, actions, out, sampled, seed, t, (cudaStream_t)stream);
    if (ge_dc_eligible(d)) return ge_dc_step(d, actions, out, sampled, seed, t, (cudaStream_t)stream);
    int blocks, wpw;
    size_t smem;
    if ((rc = launch_cfg(d, d->B, &blocks, &wpw, &smem))) return rc;
    // (TSP / DensestSubgraph ran best at 8 / 6 blocks per SM, but they now live in the group family for N <= 1024;
    //  what is left here -- DistributionCenter, Multicast p=1, N > 1024 -- is shared-memory limited at 4.)
    // DistributionCenter on the distance automaton needs half the scratch: 6 blocks per SM fit.
    const bool six = d->kind == GE_DISTRIBUTION_CENTER && d->wcode && d->dfa;
    auto kernel = sampled ? (six ? step_kernel<true, 6> : step_kernel<true, 4>) : (six ? step_kernel<false, 6> : step_kernel<false, 4>);
    if ((rc = set_smem(kernel, smem))) return rc;
    {
        cudaError_t e = ge_launch_step(kernel, dim3(blocks), dim3(GE_WPB * 32), smem, (cudaStream_t)stream, *d, actions, *out, wpw, seed, t);
        if (e != cudaSuccess) (void)cudaGetLastError();
        GE_CUDA_OK(e);
    }
    return GE_OK;
}

int ge_step(const ge_batch *d, const int32_t *actions, const ge_step_out *out, void *stream) {
    GE_NVTX("ge_step");
    return step_impl(d, const_cast<int32_t *>(actions), out, false, 0, 0, stream);  // not written when !sampled
}

int ge_step_sampled(const ge_batch *d, uint64_t seed, uint32_t t, int32_t *actions, const ge_step_out *out, void *stream) {
    GE_NVTX("ge_step_sampled");
    return step_impl(d, actions, out, true, seed, t, stream);
}

int ge_sample_actions(const ge_batch *d, uint64_t seed, uint32_t t, int32_t *actions, void *stream) {
    GE_NVTX("ge_sample_actions");
    int rc = check_batch(d);
    if (rc) return rc;
    if (d->AW <= 2) return ge_lane_sample(d, seed, t, actions, (cudaStream_t)stream);
    sample_kernel<<<(d->B + GE_WPB - 1) / GE_WPB, GE_WPB * 32, 0, (cudaStream_t)stream>>>(*d, seed, t, actions);
    GE_CUDA_OK(cudaGetLastError());
    return GE_OK;
}

int ge_obs_len(const ge_batch *d) {
    int dyn = (d->kind == GE_TSP || d->kind == GE_MULTICAST_ROUTING) ? 4 : d->kind == GE_DENSEST_SUBGRAPH ? 1 : d->kind == GE_DISTRIBUTION_CENTER ? 5
              : d->kind == GE_PERISHABLE_DELIVERY ? 16 : 2;
    int Fe = is_edge_kind(d->kind) ? 2 : 1;
    return d->N * (dyn + 5) + d->M * Fe + 2 * d->M;
}

// obs_kernel launch shape: elements one env's group writes (mode 2: the node section only) decide between a warp and a CTA per env
static int obs_warp_per_env(const ge_batch *d, int mode) {
    const int nf = ge_obs_len(d) - (is_edge_kind(d->kind) ? 4 : 3) * d->M;
    return (mode == 2 ? nf : ge_obs_len(d)) <= 2048 ? 1 : 0;
}
static int obs_blocks(const ge_batch *d, int count, int mode) { return obs_warp_per_env(d, mode) ? (count + 7) / 8 : count; }

int ge_obs_flat(const ge_batch *d, int env_lo, int count, float *out, void *stream) {
    GE_NVTX("ge_obs_flat");
    int rc = check_batch(d);
    if (rc) return rc;
    if (env_lo < 0 || count <= 0 || env_lo + count > d->B) return fail(GE_ERR_ARG, "bad env range");
    obs_kernel<0><<<obs_blocks(d, count, 0), 256, 0, (cudaStream_t)stream>>>(*d, env_lo, count, out, ge_obs_len(d), nullptr, nullptr, obs_warp_per_env(d, 0));
    GE_CUDA_OK(cudaGetLastError());
    return GE_OK;
}

int ge_obs_graph(const ge_batch *d, int env_lo, int count, float *x, float *edge_attr, int64_t *edge_index, void *stream) {
    GE_NVTX("ge_obs_graph");
    int rc = check_batch(d);
    if (rc) return rc;
    if (env_lo < 0 || count <= 0 || env_lo + count > d->B) return fail(GE_ERR_ARG, "bad env range");
    if (!x || !edge_attr || !edge_index) return fail(GE_ERR_ARG, "null output buffers");
    obs_kernel<1><<<obs_blocks(d, count, 1), 256, 0, (cudaStream_t)stream>>>(*d, env_lo, count, x, ge_obs_len(d), edge_attr, (long long *)edge_index, obs_warp_per_env(d, 1));
    GE_CUDA_OK(cudaGetLastError());
    return GE_OK;
}

int ge_obs_nodes(const ge_batch *d, int env_lo, int count, float *x, void *stream) {
    GE_NVTX("ge_obs_nodes");
    int rc = check_batch(d);
    if (rc) return rc;
    if (env_lo < 0 || count <= 0 || env_lo + count > d->B) return fail(GE_ERR_ARG, "bad env range");
    if (!x) return fail(GE_ERR_ARG, "null output buffer");
    obs_kernel<2><<<obs_blocks(d, count, 2), 256, 0, (cudaStream_t)stream>>>(*d, env_lo, count, x, ge_obs_len(d), nullptr, nullptr, obs_warp_per_env(d, 2));
    GE_CUDA_OK(cudaGetLastError());
    return GE_OK;
}

int ge_progress_supported(const ge_batch *d) {
    if (!d || d->kind == GE_PERISHABLE_DELIVERY) return 0;
    return ge_lane_eligible(d) || ge_dc_eligible(d);
}

// The incremental-mask and lane-per-env families keep only the packed mask current.
int ge_mask_bytes_current(const ge_batch *d) { return d && d->mask_bytes && !ge_incr_eligible(d) && !ge_lane_eligible(d); }

int ge_mask_bytes(const ge_batch *d, int env_lo, int count, void *stream) {
    GE_NVTX("ge_mask_bytes");
    int rc = check_batch(d);
    if (rc) return rc;
    if (!d->mask_bytes) return fail(GE_ERR_ARG, "byte mask not enabled");
    if (env_lo < 0 || count <= 0 || env_lo + count > d->B) return fail(GE_ERR_ARG, "bad env range");
    const long long total16 = (long long)count * (d->AP >> 4);
    long long blocks = (total16 + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    mask_bytes_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(*d, env_lo, total16);
    GE_CUDA_OK(cudaGetLastError());
    return GE_OK;
}

const char *ge_step_kernel_name(const ge_batch *d, int sampled) {
    static thread_local char name[96];
    if (!d) return "";
    const char *fam;
    char shape[48] = "";
    if (d->kind == GE_PERISHABLE_DELIVERY) { fam = ge_ppd_lane(d) ? "ppd_lane_step_kernel" : "ppd_step_kernel"; snprintf(shape, sizeof(shape), "SAMPLED=%d", sampled); }
    else if (ge_lane_eligible(d)) { fam = "lane_step_kernel"; snprintf(shape, sizeof(shape), "STAGED=%d,SAMPLED=%d", (d->kind == GE_LONGEST_PATH || d->kind == GE_TSP) && d->parenting >= 2, sampled); }
    else if (ge_group_eligible(d)) { fam = "group_step_kernel"; snprintf(shape, sizeof(shape), "SAMPLED=%d,G=%d", sampled, d->NW <= 8 ? 8 : d->NW <= 16 ? 16 : 32); }
    else if (ge_incr_eligible(d)) {
        if (d->kind == GE_MAX_INDEPENDENT_SET) { fam = "incr_mis_step_kernel"; snprintf(shape, sizeof(shape), "SAMPLED=%d", sampled); }
        else { fam = "incr_tree_step_kernel"; snprintf(shape, sizeof(shape), "SAMPLED=%d,G=%d", sampled, d->NW <= 8 ? 8 : d->NW <= 16 ? 16 : 32); }
    } else if (ge_dc_eligible(d)) { fam = "dc_step_kernel"; snprintf(shape, sizeof(shape), "SAMPLED=%d", sampled);
    } else { fam = "step_kernel"; snprintf(shape, sizeof(shape), "SAMPLED=%d,MINB=%d", sampled, (d->kind == GE_DISTRIBUTION_CENTER && d->wcode && d->dfa) ? 6 : 4); }
    snprintf(name, sizeof(name), "%s<%s>", fam, shape);
    return name;
}

// The copy-mode body of ge_step_host: H2D actions, step, D2H results (enqueue only, no sync).
static int step_host_enqueue(const ge_batch *d, const int32_t *h_actions, int32_t *d_actions, const ge_step_out *out, float *h_reward,
                             ge_step_flags *h_flags, double *h_solution_cost, uint8_t *h_mask, uint32_t *h_mask_bits, cudaStream_t st) {
    const size_t B = (size_t)d->B;
    GE_CUDA_OK(cudaMemcpyAsync(d_actions, h_actions, sizeof(int32_t) * B, cudaMemcpyHostToDevice, st));
    int rc = ge_step(d, d_actions, out, (void *)st);
    if (rc) return rc;
    // When the caller laid reward | flags | solution_cost | mask_bits out back to back on BOTH sides
    // (BatchedGraphEnv does), the results come back with ONE copy instead of four.
    const char *dr = (const char *)out->reward, *hr = (const char *)h_reward;
    bool packed = h_solution_cost && h_mask_bits && (const char *)out->flags == dr + 4 * B &&
                  (const char *)out->solution_cost == dr + 8 * B && (const char *)d->mask_bits == dr + 16 * B &&
                  (const char *)h_flags == hr + 4 * B && (const char *)h_solution_cost == hr + 8 * B &&
                  (const char *)h_mask_bits == hr + 16 * B;
    if (packed) {
        GE_CUDA_OK(cudaMemcpyAsync(h_reward, out->reward, 16 * B + sizeof(uint32_t) * B * d->AW, cudaMemcpyDeviceToHost, st));
    } else {
        GE_CUDA_OK(cudaMemcpyAsync(h_reward, out->reward, sizeof(float) * B, cudaMemcpyDeviceToHost, st));
        GE_CUDA_OK(cudaMemcpyAsync(h_flags, out->flags, sizeof(ge_step_flags) * B, cudaMemcpyDeviceToHost, st));
        if (h_solution_cost)
            GE_CUDA_OK(cudaMemcpyAsync(h_solution_cost, out->solution_cost, sizeof(double) * B, cudaMemcpyDeviceToHost, st));
        if (h_mask_bits)
            GE_CUDA_OK(cudaMemcpyAsync(h_mask_bits, d->mask_bits, sizeof(uint32_t) * B * d->AW, cudaMemcpyDeviceToHost, st));
    }
    if (h_mask) {
        if (!d->mask_bytes) return fail(GE_ERR_ARG, "byte mask not enabled");
        if (!ge_mask_bytes_current(d) && (rc = ge_mask_bytes(d, 0, d->B, (void *)st))) return rc;
        GE_CUDA_OK(cudaMemcpyAsync(h_mask, d->mask_bytes, B * d->AP, cudaMemcpyDeviceToHost, st));
    }
    return GE_OK;
}

// ge_step_host / ge_step_host_pipelined are fixed sequences over fixed buffers, called once per env step: they are
// captured into a CUDA graph on first use and replayed with ONE launch call afterwards.  The cache key is the whole
// descriptor plus every buffer pointer, the stream and the chunk count; anything else re-captures.  The cache is
// process-wide and mutex-guarded; ge_step_host_release drops a batch's entries.  Capture is impossible on the legacy
// default stream: direct path there.
namespace {
constexpr int HSG_SLOTS = 8, HSG_MAX_CHUNKS = 8;
struct HostStepGraph {
    ge_batch d;
    const void *p[10];
    cudaStream_t st;
    int chunks;
    cudaGraphExec_t exec;
    bool valid;
    uint32_t *progress;      // streamed write-back (chunks code 0x200): device counters, one per 1024 envs ...
    uint32_t *err;           // ... and the writer's give-up flag in mapped host memory
};
HostStepGraph g_hsg[HSG_SLOTS];
bool g_streamed_off = false;                             // set when a streamed write-back ever timed out: sliced path from then on
int g_hsg_next = 0;
std::mutex g_hsg_mu;
cudaStream_t g_side;                                     // write-back lane (the kernels stay on the caller's stream)
cudaEvent_t g_fork, g_stepped[HSG_MAX_CHUNKS], g_join;
bool g_side_ready = false;

void hsg_drop(HostStepGraph &g) {
    if (!g.valid) return;
    cudaGraphExecDestroy(g.exec);
    if (g.progress) cudaFree(g.progress);
    if (g.err) cudaFreeHost(g.err);
    g.progress = g.err = nullptr;
    g.valid = false;
}
HostStepGraph *hsg_entry(const ge_batch *d, const void *const *key, cudaStream_t st, int chunks) {
    for (HostStepGraph &g : g_hsg)
        if (g.valid && g.st == st && g.chunks == chunks && memcmp(&g.d, d, sizeof(ge_batch)) == 0 && memcmp(g.p, key, sizeof(g.p)) == 0)
            return &g;
    return nullptr;
}
void hsg_insert(const ge_batch *d, const void *const *key, cudaStream_t st, int chunks, cudaGraphExec_t exec, uint32_t *progress = nullptr,
                uint32_t *err = nullptr) {
    HostStepGraph &g = g_hsg[g_hsg_next];
    g_hsg_next = (g_hsg_next + 1) % HSG_SLOTS;
    hsg_drop(g);
    memcpy(&g.d, d, sizeof(ge_batch));
    memcpy(g.p, key, sizeof(g.p));
    g.st = st; g.chunks = chunks; g.exec = exec; g.valid = true; g.progress = progress; g.err = err;
}

// Waits for the stream by polling: a blocking synchronize parks the thread and pays the wake-up latency of an
// interrupt (~10 us against a 40 us step); the results are needed by this very thread, so it spins.
cudaError_t spin_until_done(cudaStream_t st) {
    cudaError_t e;
    while ((e = cudaStreamQuery(st)) == cudaErrorNotReady) {
#if defined(__x86_64__) || defined(__i386__)
        __builtin_ia32_pause();
#endif
    }
    return e;
}

// Write-back of one slice's results into the caller's pinned host arrays (UVA-mapped): every thread moves 16-byte
// pieces, consecutive threads consecutive pieces => full 128-byte PCIe write transactions, all four arrays in one launch.
__device__ __forceinline__ void copy_out(void *dst, const void *src, size_t bytes, int tid, int nthreads) {
    const size_t n16 = bytes >> 4;
    const uint4 *s4 = reinterpret_cast<const uint4 *>(src);
    uint4 *d4 = reinterpret_cast<uint4 *>(dst);
    for (size_t i = tid; i < n16; i += nthreads) d4[i] = s4[i];
    const size_t done = n16 << 4;
    for (size_t i = done + tid; i < bytes; i += nthreads) reinterpret_cast<unsigned char *>(dst)[i] = reinterpret_cast<const unsigned char *>(src)[i];
}
__global__ void __launch_bounds__(256) writeback_kernel(const float *reward, const ge_step_flags *flags, const double *cost, const uint32_t *mask_bits,
                                                      float *h_reward, ge_step_flags *h_flags, double *h_cost, uint32_t *h_mask_bits, int n, int AW) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
    copy_out(h_reward, reward, (size_t)n * 4, tid, nt);
    copy_out(h_flags, flags, (size_t)n * 4, tid, nt);
    if (h_cost) copy_out(h_cost, cost, (size_t)n * 8, tid, nt);
    if (h_mask_bits) copy_out(h_mask_bits, mask_bits, (size_t)n * AW * 4, tid, nt);
}
// Compact variant (ge_step_host_compact): flags as ONE byte per env (GE_FLAGS8_*), solution_cost as float32 -- 9 instead of 16
// bytes per env next to the packed mask.  A thread packs 16 envs' flags into one 16-byte store, 4 envs' costs into another.
__device__ __forceinline__ uint32_t flags8(const ge_step_flags &f) {
    return (uint32_t)(f.done & 1u) | ((uint32_t)(f.solved + 1) & 3u) << 1 | ((uint32_t)f.status & 3u) << 3 | ((uint32_t)f.has_mask & 1u) << 5;
}
__global__ void __launch_bounds__(256) writeback_compact_kernel(const float *reward, const ge_step_flags *flags, const double *cost,
                                                              const uint32_t *mask_bits, float *h_reward, uint8_t *h_flags8, float *h_cost32,
                                                              uint32_t *h_mask_bits, int n, int AW) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
    copy_out(h_reward, reward, (size_t)n * 4, tid, nt);
    for (int g = tid; g < (n >> 4); g += nt) {                       // 16 envs -> 16 bytes
        uint32_t w[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const uint4 f4 = reinterpret_cast<const uint4 *>(flags)[4 * g + q];     // four ge_step_flags
            const ge_step_flags *f = reinterpret_cast<const ge_step_flags *>(&f4);
            w[q] = flags8(f[0]) | flags8(f[1]) << 8 | flags8(f[2]) << 16 | flags8(f[3]) << 24;
        }
        reinterpret_cast<uint4 *>(h_flags8)[g] = make_uint4(w[0], w[1], w[2], w[3]);
    }
    for (int b = (n & ~15) + tid; b < n; b += nt) h_flags8[b] = (uint8_t)flags8(flags[b]);
    if (h_cost32) {
        for (int g = tid; g < (n >> 2); g += nt) {                   // 4 envs -> 16 bytes
            const double2 a = reinterpret_cast<const double2 *>(cost)[2 * g], c = reinterpret_cast<const double2 *>(cost)[2 * g + 1];
            reinterpret_cast<float4 *>(h_cost32)[g] = make_float4((float)a.x, (float)a.y, (float)c.x, (float)c.y);
        }
        for (int b = (n & ~3) + tid; b < n; b += nt) h_cost32[b] = (float)cost[b];
    }
    if (h_mask_bits) copy_out(h_mask_bits, mask_bits, (size_t)n * AW * 4, tid, nt);
}

// Streamed write-back (ge_step_host_pipelined, chunks = 0): runs CONCURRENTLY with the one step kernel of the call.  Block j
// waits for chunk c = j, j + gridDim, ... of 1024 envs to be complete (ge_batch.progress, written by the step kernel with
// release semantics), then moves that chunk's results into the pinned host arrays: results cross PCIe while later chunks are
// still being stepped, and the call ends one chunk's transfer after the step kernel instead of a whole slice's.  The wait is
// BOUNDED (it gives up and raises *err; the host then falls back to the sliced path), so a scheduler that serialised the two
// kernels the wrong way round cannot hang the GPU.  Loads bypass L1 (the data was written by other SMs during this kernel).
__device__ __forceinline__ void copy_out_cg(void *dst, const void *src, size_t bytes, int tid, int nthreads) {
    const size_t n16 = bytes >> 4;
    const uint4 *s4 = reinterpret_cast<const uint4 *>(src);
    uint4 *d4 = reinterpret_cast<uint4 *>(dst);
    for (size_t i = tid; i < n16; i += nthreads) d4[i] = __ldcg(s4 + i);
    for (size_t i = (n16 << 4) + tid; i < bytes; i += nthreads) reinterpret_cast<unsigned char *>(dst)[i] = __ldcg(reinterpret_cast<const unsigned char *>(src) + i);
}
__global__ void __launch_bounds__(256) writeback_stream_kernel(uint32_t *progress, int n_chunks, int B, const float *reward, const ge_step_flags *flags,
                                                             const double *cost, const uint32_t *mask_bits, float *h_reward, void *h_flags, void *h_cost,
                                                             uint32_t *h_mask_bits, int AW, int compact, volatile uint32_t *err) {
    __shared__ int ok;
    const int tid = threadIdx.x, nt = blockDim.x;
    for (int c = blockIdx.x; c < n_chunks; c += gridDim.x) {
        const int lo = c << GE_PROGRESS_SHIFT, n = min(1 << GE_PROGRESS_SHIFT, B - lo);
        if (tid == 0) {
            unsigned spins = 0, seen;
            ok = 1;
            for (;;) {
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(progress + c) : "memory");
                if (seen >= (unsigned)n) break;
                if (++spins > (1u << 21)) { ok = 0; break; }          // ~0.2 s: give up, never hang
                __nanosleep(100);
            }
        }
        __syncthreads();
        if (!ok) { if (tid == 0) *err = 1u; return; }
        copy_out_cg(h_reward + lo, reward + lo, (size_t)n * 4, tid, nt);
        if (compact) {
            uint8_t *hf = reinterpret_cast<uint8_t *>(h_flags) + lo;
            for (int g = tid; g < (n >> 4); g += nt) {
                uint32_t w[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const uint4 f4 = __ldcg(reinterpret_cast<const uint4 *>(flags + lo) + 4 * g + q);
                    const ge_step_flags *f = reinterpret_cast<const ge_step_flags *>(&f4);
                    w[q] = flags8(f[0]) | flags8(f[1]) << 8 | flags8(f[2]) << 16 | flags8(f[3]) << 24;
                }
                reinterpret_cast<uint4 *>(hf)[g] = make_uint4(w[0], w[1], w[2], w[3]);
            }
            for (int b = (n & ~15) + tid; b < n; b += nt) { const uint32_t f1 = __ldcg(reinterpret_cast<const uint32_t *>(flags + lo) + b); hf[b] = (uint8_t)flags8(*reinterpret_cast<const ge_step_flags *>(&f1)); }
            if (h_cost) {
                float *hc = reinterpret_cast<float *>(h_cost) + lo;
                for (int g = tid; g < (n >> 2); g += nt) {
                    const double2 a = __ldcg(reinterpret_cast<const double2 *>(cost + lo) + 2 * g), cc = __ldcg(reinterpret_cast<const double2 *>(cost + lo) + 2 * g + 1);
                    reinterpret_cast<float4 *>(hc)[g] = make_float4((float)a.x, (float)a.y, (float)cc.x, (float)cc.y);
                }
                for (int b = (n & ~3) + tid; b < n; b += nt) hc[b] = (float)__ldcg(cost + lo + b);
            }
        } else {
            copy_out_cg(reinterpret_cast<ge_step_flags *>(h_flags) + lo, flags + lo, (size_t)n * 4, tid, nt);
            if (h_cost) copy_out_cg(reinterpret_cast<double *>(h_cost) + lo, cost + lo, (size_t)n * 8, tid, nt);
        }
        if (h_mask_bits) copy_out_cg(h_mask_bits + (size_t)lo * AW, mask_bits + (size_t)lo * AW, (size_t)n * AW * 4, tid, nt);
        __syncthreads();
        if (tid == 0) progress[c] = 0;                                 // consumed: re-armed for the next replay
    }
}
}  // namespace

int ge_batch_slice(const ge_batch *d, int lo, int count, ge_batch *o) {
    if (!d || !o) return fail(GE_ERR_ARG, "null batch");
    if (lo < 0 || count <= 0 || lo + count > d->B || (lo & 31)) return fail(GE_ERR_ARG, "bad slice [%d, %d) of %d envs (lo must be a multiple of 32)", lo, lo + count, d->B);
    *o = *d;
    o->B = count;
    o->env_id0 = d->env_id0 + lo;
    const size_t b = (size_t)lo;
#define ADV(field, per_env) if (d->field) o->field = d->field + b * (size_t)(per_env)
    ADV(row_ptr, d->RP); ADV(col, d->MP); ADV(w32, d->MP); ADV(w64, d->MP);
    if (d->adj_bits) o->adj_bits = d->adj_bits + (adj_tiled(*d) ? (b >> 5) * (size_t)d->N * 32 * d->NW : b * (size_t)d->ADJS);
    ADV(rev, d->MP); ADV(esrc, d->MP); ADV(wsort, d->MP); ADV(wcode, d->MP); ADV(dc_edges, d->MP); ADV(wmin, 1); ADV(wmat, (size_t)d->N * d->N);
    ADV(src, 1); ADV(dest, 1); ADV(target_bits, d->NW); ADV(node_cost, d->N); ADV(node_xy, 2 * d->N); ADV(max_dist32, 1);
    ADV(targets, d->n_targets); ADV(in_range, (size_t)d->n_targets * d->NW); ADV(heuristic, 1); ADV(heuristic_alt, 1); ADV(features, 5 * d->N);
    ADV(head, 1); ADV(node_bits, d->NW); ADV(node_bits2, d->NW); ADV(edge_bits, d->MW); ADV(dist32, d->N); ADV(bestkey, d->N);
    ADV(cost, 1); ADV(counters, 4); ADV(done, 1); ADV(mask_bits, d->AW); ADV(mask_cnt, 8); ADV(mask_bytes, d->AP);
    ADV(mask0_bits, d->AW); ADV(acc, 1); ADV(traj, 1); ADV(env_steps, 1);
    ADV(dc_rows, (size_t)d->N * 32);
    ADV(obs_x, ge_obs_len(d) - (size_t)(is_edge_kind(d->kind) ? 4 : 3) * d->M);   // N * F floats per env
#undef ADV
    return GE_OK;   // dfa is shared by the whole batch; acc keeps the parent's component stride
}

int ge_step_host_release(const ge_batch *d) {
    if (!d) return GE_OK;
    std::lock_guard<std::mutex> lock(g_hsg_mu);
    for (HostStepGraph &g : g_hsg)
        if (g.valid && g.d.mask_bits == d->mask_bits) hsg_drop(g);
    return GE_OK;
}

int ge_step_host(const ge_batch *d, const int32_t *h_actions, int32_t *d_actions, const ge_step_out *out, float *h_reward,
                 ge_step_flags *h_flags, double *h_solution_cost, uint8_t *h_mask, uint32_t *h_mask_bits, void *stream) {
    GE_NVTX("ge_step_host");
    cudaStream_t st = (cudaStream_t)stream;
    if (!d) return fail(GE_ERR_ARG, "null batch");
    if (!d_actions || !out) return fail(GE_ERR_ARG, "null step buffers");
    const void *key[10] = {h_actions, d_actions, out->reward, out->flags, out->solution_cost, h_reward, h_flags, h_solution_cost, h_mask,
                           h_mask_bits};
    const bool capturable = st != nullptr && st != cudaStreamLegacy && st != cudaStreamPerThread;
    if (capturable) {
        cudaGraphExec_t exec = nullptr;
        {
            std::lock_guard<std::mutex> lock(g_hsg_mu);
            if (HostStepGraph *g = hsg_entry(d, key, st, 0)) exec = g->exec;
        }
        if (exec) {
            GE_CUDA_OK(cudaGraphLaunch(exec, st));
            GE_CUDA_OK(cudaStreamSynchronize(st));
            return GE_OK;
        }
        // first call for this (descriptor, buffers, stream): run once directly (also sets kernel attributes), then capture
        int rc = step_host_enqueue(d, h_actions, d_actions, out, h_reward, h_flags, h_solution_cost, h_mask, h_mask_bits, st);
        if (rc) return rc;
        GE_CUDA_OK(cudaStreamSynchronize(st));
        // NOTE: the capture below does not execute anything; the call above already did this step.
        std::lock_guard<std::mutex> lock(g_hsg_mu);
        cudaGraph_t graph = nullptr;
        if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
            int rc2 = step_host_enqueue(d, h_actions, d_actions, out, h_reward, h_flags, h_solution_cost, h_mask, h_mask_bits, st);
            cudaError_t e = cudaStreamEndCapture(st, &graph);
            if (rc2 == GE_OK && e == cudaSuccess && graph) {
                cudaGraphExec_t ex = nullptr;
                if (cudaGraphInstantiate(&ex, graph, 0) == cudaSuccess) hsg_insert(d, key, st, 0, ex);
            }
            if (graph) cudaGraphDestroy(graph);
            (void)cudaGetLastError();
        } else {
            (void)cudaGetLastError();
        }
        return GE_OK;
    }
    int rc = step_host_enqueue(d, h_actions, d_actions, out, h_reward, h_flags, h_solution_cost, h_mask, h_mask_bits, st);
    if (rc) return rc;
    GE_CUDA_OK(cudaStreamSynchronize(st));
    return GE_OK;
}

// The two stages of one slice of the pipelined step (enqueue only).  The step kernels read the actions straight from the
// caller's pinned host buffer (coalesced PCIe reads): measured 59.2 -> 53.0 us per 65,536-env step at two slices against
// H2D copies on a lane of their own (profiles/r02_e2e_breakdown.jsonl).
static int pipelined_step(const ge_batch *d, int lo, int n, const int32_t *h_actions, const ge_step_out *out, cudaStream_t s) {
    ge_batch sl;
    int rc = ge_batch_slice(d, lo, n, &sl);
    if (rc) return rc;
    // slices after the first follow another slice's step kernel on this stream (different envs): programmatic dependent launch
    // lets them become resident under its tail
    if (lo > 0) sl.flags |= GE_FLAG_PDL;
    ge_step_out so = {out->reward + lo, out->flags + lo, out->solution_cost + lo};
    return ge_step(&sl, h_actions + lo, &so, (void *)s);
}
static int pipelined_write_back(const ge_batch *d, int lo, int n, const ge_step_out *out, float *h_reward, void *h_flags,
                                void *h_solution_cost, uint32_t *h_mask_bits, bool compact, cudaStream_t s) {
    const size_t bytes = (size_t)n * (16 + 4 * (size_t)d->AW);
    int blocks = (int)((bytes / 16 + 255) / 256);
    if (blocks > 32) blocks = 32;     // a handful of CTAs saturate PCIe; the rest of the GPU keeps stepping the next slice
    if (blocks < 1) blocks = 1;
    if (compact)
        writeback_compact_kernel<<<blocks, 256, 0, s>>>(out->reward + lo, out->flags + lo, out->solution_cost + lo, d->mask_bits + (size_t)lo * d->AW,
                                                        h_reward + lo, (uint8_t *)h_flags + lo, h_solution_cost ? (float *)h_solution_cost + lo : nullptr,
                                                        h_mask_bits ? h_mask_bits + (size_t)lo * d->AW : nullptr, n, d->AW);
    else
        writeback_kernel<<<blocks, 256, 0, s>>>(out->reward + lo, out->flags + lo, out->solution_cost + lo, d->mask_bits + (size_t)lo * d->AW,
                                                h_reward + lo, (ge_step_flags *)h_flags + lo, h_solution_cost ? (double *)h_solution_cost + lo : nullptr,
                                                h_mask_bits ? h_mask_bits + (size_t)lo * d->AW : nullptr, n, d->AW);
    GE_CUDA_OK(cudaGetLastError());
    if (d->obs_x) {   // node columns of the slice's observation, on the same lane (runs while the next slice steps)
        int rc = ge_obs_nodes(d, lo, n, d->obs_x + (size_t)lo * (ge_obs_len(d) - (size_t)(is_edge_kind(d->kind) ? 4 : 3) * d->M), (void *)s);
        if (rc) return rc;
    }
    return GE_OK;
}

static int step_host_pipelined_impl(const ge_batch *d, const int32_t *h_actions, const ge_step_out *out, float *h_reward,
                                    void *h_flags, void *h_solution_cost, uint32_t *h_mask_bits, int chunks, bool compact, void *stream);

int ge_step_host_pipelined(const ge_batch *d, const int32_t *h_actions, const ge_step_out *out, float *h_reward,
                           ge_step_flags *h_flags, double *h_solution_cost, uint32_t *h_mask_bits, int chunks, void *stream) {
    GE_NVTX("ge_step_host_pipelined");
    return step_host_pipelined_impl(d, h_actions, out, h_reward, h_flags, h_solution_cost, h_mask_bits, chunks, false, stream);
}

int ge_step_host_compact(const ge_batch *d, const int32_t *h_actions, const ge_step_out *out, float *h_reward,
                         uint8_t *h_flags8, float *h_solution_cost32, uint32_t *h_mask_bits, int chunks, void *stream) {
    GE_NVTX("ge_step_host_compact");
    return step_host_pipelined_impl(d, h_actions, out, h_reward, h_flags8, h_solution_cost32, h_mask_bits, chunks, true, stream);
}

static int ensure_side_streams() {   // (g_hsg_mu held)
    if (g_side_ready) return GE_OK;
    GE_CUDA_OK(cudaStreamCreateWithFlags(&g_side, cudaStreamNonBlocking));
    for (int i = 0; i < HSG_MAX_CHUNKS; ++i) GE_CUDA_OK(cudaEventCreateWithFlags(&g_stepped[i], cudaEventDisableTiming));
    GE_CUDA_OK(cudaEventCreateWithFlags(&g_fork, cudaEventDisableTiming));
    GE_CUDA_OK(cudaEventCreateWithFlags(&g_join, cudaEventDisableTiming));
    g_side_ready = true;
    return GE_OK;
}

// chunks = 0: one full-batch step kernel that signals ge_batch.progress + the concurrent writer.
static int step_host_streamed(const ge_batch *d, const void *const *key, const int32_t *h_actions, const ge_step_out *out, float *h_reward,
                              void *h_flags, void *h_solution_cost, uint32_t *h_mask_bits, bool compact, cudaStream_t st) {
    const int code = 0x200 | (compact ? 0x100 : 0);
    const int n_chunks = (d->B + (1 << GE_PROGRESS_SHIFT) - 1) >> GE_PROGRESS_SHIFT;
    cudaGraphExec_t exec = nullptr;
    uint32_t *progress = nullptr, *err = nullptr;
    {
        std::lock_guard<std::mutex> lock(g_hsg_mu);
        if (HostStepGraph *g = hsg_entry(d, key, st, code)) { exec = g->exec; progress = g->progress; err = g->err; }
    }
    int rc;
    if (exec) {
        GE_CUDA_OK(cudaGraphLaunch(exec, st));
        GE_CUDA_OK(spin_until_done(st));
        if (*reinterpret_cast<volatile uint32_t *>(err)) {
            // the writer gave up (the two kernels did not run concurrently): the step itself is done; deliver its results with a
            // plain write-back, re-arm the counters and use the sliced path from now on
            *err = 0;
            g_streamed_off = true;
            GE_CUDA_OK(cudaMemsetAsync(progress, 0, sizeof(uint32_t) * n_chunks, st));
            if ((rc = pipelined_write_back(d, 0, d->B, out, h_reward, h_flags, h_solution_cost, h_mask_bits, compact, st))) return rc;
            GE_CUDA_OK(cudaStreamSynchronize(st));
        }
        return GE_OK;
    }
    // first call: this step through one plain pass, then capture the two-branch graph for the following calls
    if ((rc = pipelined_step(d, 0, d->B, h_actions, out, st))) return rc;
    if ((rc = pipelined_write_back(d, 0, d->B, out, h_reward, h_flags, h_solution_cost, h_mask_bits, compact, st))) return rc;
    GE_CUDA_OK(cudaStreamSynchronize(st));
    std::lock_guard<std::mutex> lock(g_hsg_mu);
    if ((rc = ensure_side_streams())) return rc;
    if (cudaMalloc(&progress, sizeof(uint32_t) * n_chunks) != cudaSuccess || cudaMemset(progress, 0, sizeof(uint32_t) * n_chunks) != cudaSuccess ||
        cudaHostAlloc(&err, sizeof(uint32_t), cudaHostAllocMapped) != cudaSuccess) {
        if (progress) cudaFree(progress);
        (void)cudaGetLastError();
        g_streamed_off = true;           // this step is done; later calls take the sliced path
        return GE_OK;
    }
    *err = 0;
    cudaGraph_t graph = nullptr;
    bool inserted = false;
    if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
        cudaStream_t s_out = g_side;
        bool ok = cudaEventRecord(g_fork, st) == cudaSuccess && cudaStreamWaitEvent(s_out, g_fork, 0) == cudaSuccess;
        int nb = n_chunks < 32 ? n_chunks : 32;
        writeback_stream_kernel<<<nb, 256, 0, s_out>>>(progress, n_chunks, d->B, out->reward, out->flags, out->solution_cost, d->mask_bits, h_reward,
                                                       h_flags, h_solution_cost, h_mask_bits, d->AW, compact ? 1 : 0, err);
        ok = ok && cudaGetLastError() == cudaSuccess;
        ge_batch dd = *d;
        dd.progress = progress;
        int rc2 = ge_step(&dd, h_actions, out, (void *)st);
        if (rc2 == GE_OK && d->obs_x) rc2 = ge_obs_nodes(d, 0, d->B, d->obs_x, (void *)st);
        ok = ok && cudaEventRecord(g_join, s_out) == cudaSuccess && cudaStreamWaitEvent(st, g_join, 0) == cudaSuccess;
        cudaError_t e = cudaStreamEndCapture(st, &graph);
        if (ok && rc2 == GE_OK && e == cudaSuccess && graph) {
            cudaGraphExec_t ex = nullptr;
            if (cudaGraphInstantiate(&ex, graph, 0) == cudaSuccess) { hsg_insert(d, key, st, code, ex, progress, err); inserted = true; }
        }
        if (graph) cudaGraphDestroy(graph);
    }
    (void)cudaGetLastError();
    if (!inserted) { cudaFree(progress); cudaFreeHost(err); g_streamed_off = true; }
    return GE_OK;
}

static int step_host_pipelined_impl(const ge_batch *d, const int32_t *h_actions, const ge_step_out *out, float *h_reward,
                                    void *h_flags, void *h_solution_cost, uint32_t *h_mask_bits, int chunks, bool compact, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    int rc = check_batch(d);
    if (rc) return rc;
    if (!h_actions || !out || !h_reward || !h_flags) return fail(GE_ERR_ARG, "null step buffers");
    if (st == nullptr || st == cudaStreamLegacy || st == cudaStreamPerThread) return fail(GE_ERR_ARG, "ge_step_host_pipelined needs a created (capturable) stream");
    const void *key[10] = {h_actions, out->reward, out->flags, out->solution_cost, h_reward, h_flags, h_solution_cost, h_mask_bits};
    if (chunks <= 0) {   // streamed write-back: ONE step kernel + a concurrent writer fed by ge_batch.progress (see writeback_stream_kernel)
        if (!g_streamed_off && ge_progress_supported(d))
            return step_host_streamed(d, key, h_actions, out, h_reward, h_flags, h_solution_cost, h_mask_bits, compact, st);
        chunks = 2;      // kernel family without progress counters: two slices
    }
    if (chunks > HSG_MAX_CHUNKS) chunks = HSG_MAX_CHUNKS;
    int per = ((d->B + chunks - 1) / chunks + 127) & ~127;    // slice starts are multiples of 128 envs (tiles, vector alignment)
    chunks = (d->B + per - 1) / per;
    cudaGraphExec_t exec = nullptr;
    {
        std::lock_guard<std::mutex> lock(g_hsg_mu);
        if (HostStepGraph *g = hsg_entry(d, key, st, chunks | (compact ? 0x100 : 0))) exec = g->exec;
    }
    if (!exec) {
        // first call: one direct pass on the caller's stream (sets kernel attributes, does THIS step), then capture the
        // two-lane sequence for the following calls
        // (Step kernels storing reward / flags / solution_cost / packed mask straight into the pinned host arrays -- no write-back
        //  kernels -- measured 99-111 us per 65,536-env step against 55-59 us: 4-8 byte stores per lane reach PCIe as 32-byte
        //  sectors, the write-back kernel's 16 bytes per lane as full lines.  profiles/r02_e2e_direct_writes.jsonl)
        for (int i = 0; i < chunks; ++i) {
            const int lo = i * per, n = (lo + per <= d->B) ? per : d->B - lo;
            if ((rc = pipelined_step(d, lo, n, h_actions, out, st))) return rc;
            if ((rc = pipelined_write_back(d, lo, n, out, h_reward, h_flags, h_solution_cost, h_mask_bits, compact, st))) return rc;
        }
        GE_CUDA_OK(cudaStreamSynchronize(st));
        std::lock_guard<std::mutex> lock(g_hsg_mu);
        if ((rc = ensure_side_streams())) return rc;
        // Two lanes: step-kernel chain (caller's stream) -> write-back chain (g_side).
        // The kernels of the slices run ONE AFTER THE OTHER: launched side by side they would share the GPU, finish
        // together, and every write-back would start as late as after a single big kernel (measured: no gain).  Chained,
        // slice i's results cross PCIe while slice i+1 steps.
        cudaGraph_t graph = nullptr;
        if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
            int rc2 = GE_OK;
            cudaStream_t s_out = g_side;
            bool ok = cudaEventRecord(g_fork, st) == cudaSuccess && cudaStreamWaitEvent(s_out, g_fork, 0) == cudaSuccess;
            for (int i = 0; ok && i < chunks && rc2 == GE_OK; ++i) {
                const int lo = i * per, n = (lo + per <= d->B) ? per : d->B - lo;
                rc2 = pipelined_step(d, lo, n, h_actions, out, st);
                ok = ok && cudaEventRecord(g_stepped[i], st) == cudaSuccess && cudaStreamWaitEvent(s_out, g_stepped[i], 0) == cudaSuccess;
                if (rc2 == GE_OK) rc2 = pipelined_write_back(d, lo, n, out, h_reward, h_flags, h_solution_cost, h_mask_bits, compact, s_out);
            }
            ok = ok && cudaEventRecord(g_join, s_out) == cudaSuccess && cudaStreamWaitEvent(st, g_join, 0) == cudaSuccess;
            cudaError_t e = cudaStreamEndCapture(st, &graph);
            if (ok && rc2 == GE_OK && e == cudaSuccess && graph) {
                cudaGraphExec_t ex = nullptr;
                if (cudaGraphInstantiate(&ex, graph, 0) == cudaSuccess) hsg_insert(d, key, st, chunks | (compact ? 0x100 : 0), ex);
            }
            if (graph) cudaGraphDestroy(graph);
            (void)cudaGetLastError();
        } else {
            (void)cudaGetLastError();
        }
        return GE_OK;
    }
    GE_CUDA_OK(cudaGraphLaunch(exec, st));
    GE_CUDA_OK(spin_until_done(st));
    return GE_OK;
}

int ge_stats(const ge_batch *d, double *out4, void *stream) {
    GE_NVTX("ge_stats");
    int rc = check_batch(d);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    GE_CUDA_OK(cudaMemsetAsync(out4, 0, sizeof(double) * 4, st));
    int blocks = (d->B + 255) / 256;
    if (blocks > 592) blocks = 592;
    stats_kernel<<<blocks, 256, 0, st>>>(*d, out4);
    GE_CUDA_OK(cudaGetLastError());
    return GE_OK;
}

}  // extern "C"
