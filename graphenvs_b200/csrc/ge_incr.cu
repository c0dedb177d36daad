// ge_incr.cu -- INCREMENTAL-MASK step kernels: SteinerTree/MST, MulticastRouting (parenting >= 2),
// MaxIndependentSet.
//
// The reference recomputes the whole valid-action mask from scratch in every step (twice).  For
// these envs one step changes the state by ONE node, and the new mask differs from the old one
// only around that node's CSR row:
//   * tree-growing envs (steiner_tree.py:116-120, multicast_routing.py:162-164): when v joins the
//     tree, every edge INTO v stops being valid and every edge v->x with x outside the tree becomes
//     valid  =>  touch row(v) and its reverse edges (rev[]), nothing else;
//   * Multicast parenting >= 3 (multicast_routing.py:166-186): per frontier vertex x the mask keeps
//     argmin_e { dist[src e] + delay[e] } over tree->x edges, lowest edge index on ties.  The tree
//     only grows and distances of tree nodes never change, so the argmin is a running minimum:
//     keep best[x] = (float32 bits << 32 | edge id) per node and fold in the edges of row(v);
//   * MaxIndependentSet (max_independent_set.py:92-100): the mask loses exactly bit `a`.
// Same booleans as the full recompute (ge_envs.cuh, still reachable with GE_FLAG_FORCE_WARP and
// compared bit for bit in the tests), but a step reads ~1 KB instead of up to 77 KB and executes
// ~100 instead of ~4000 warp instructions: ncu on the recompute kernels showed them issue-bound
// on the row-set expansion (profiles/r01_step_kernel_cfg5_multicast_warp_v1.md).
//
// One warp per env (a CSR row is 10-20 edges: one warp iteration); MaxIndependentSet one lane per env.
#include "ge_common.cuh"

using namespace ge;

extern "C" int ge_set_error(int code, const char *fmt, ...);

namespace {

constexpr u64 KEY_NONE = ~0ull;
#define GE_INCR_MINB 8  // resident blocks per SM the tree step kernel is compiled for: 32 registers => 64 warps/SM.
                        // The kernel is a chain of ~5 dependent memory rounds per env, i.e. latency-bound: measured
                        // 0.70 / 0.84 / 0.96 G env-steps/s at cfg3 for 4 / 6 / 8 blocks per SM.

// The incremental kernels keep only the PACKED mask current.  Writing the byte view as well meant one scattered 1-byte
// store per changed edge, each a 32-byte sector read-modify-write in HBM: 2.3 KB of the 4.7 KB a Multicast step moved
// (profiles/r01_final_step_kernel_cfg5_multicast.md, 2.55x the useful bytes).  The byte view (torch.bool for a policy)
// is expanded on demand by ge_mask_bytes (ge_api.cu) in one coalesced pass.
// Large masks additionally keep 16 CHUNK COUNTS (ge_batch.mask_cnt: popcount of every 1/16th of the mask, 16-bit counters,
// one 32-byte sector per env): the in-kernel sampler then finds the chunk that holds the r-th valid action from that one
// sector and reads just that chunk, two memory rounds and ~100 bytes instead of walking up to 1 KB of mask through
// dependent loads (the walk was ~30 % of the instructions and 18 % of the stall samples of the Multicast step at config 5).
__device__ __forceinline__ int mask_chunk_words(const ge_batch &d) { return (d.AW + 15) >> 4; }
__device__ __forceinline__ void mask_count(const ge_batch &d, int b, int e, int delta) {
    const int chunk = (e >> 5) / mask_chunk_words(d);
    atomicAdd(&d.mask_cnt[(size_t)b * 8 + (chunk >> 1)], (uint32_t)delta << (16 * (chunk & 1)));   // counters never underflow: only set bits are cleared
}
__device__ __forceinline__ void mask_set(const ge_batch &d, int b, int e) {
    atomicOr(&d.mask_bits[(size_t)b * d.AW + (e >> 5)], 1u << (e & 31));
    if (d.mask_cnt) mask_count(d, b, e, 1);
}
__device__ __forceinline__ void mask_clear(const ge_batch &d, int b, int e) {
    atomicAnd(&d.mask_bits[(size_t)b * d.AW + (e >> 5)], ~(1u << (e & 31)));
    if (d.mask_cnt) mask_count(d, b, e, -1);
}

// Group-wide zero fill of an env's packed mask.
template <int G>
__device__ __forceinline__ void mask_zero(const ge_batch &d, int b, int lane) {
    uint32_t *mb = d.mask_bits + (size_t)b * d.AW;
    for (int w = lane; w < d.AW; w += G) mb[w] = 0;
    if (d.mask_cnt && lane < 8) d.mask_cnt[(size_t)b * 8 + lane] = 0;
}

// r-th valid action through the chunk counts (same draw as group_sample: r-th set bit of the packed mask).
template <int G>
__device__ __forceinline__ int group_sample_chunks(const Grp<G> &g, const ge_batch &d, int b, uint64_t seed, uint32_t env, uint32_t t, int total) {
    if (total <= 0) return -1;
    const uint32_t r = (uint32_t)(((uint64_t)mix32(seed, env, t) * (uint64_t)total) >> 32);
    const int CW = mask_chunk_words(d);
    // stage 1: lanes 0..15 hold one chunk count each
    int cnt = 0;
    if (g.gl < 16) cnt = (int)((d.mask_cnt[(size_t)b * 8 + (g.gl >> 1)] >> (16 * (g.gl & 1))) & 0xffffu);
    int inc = cnt;
#pragma unroll
    for (int o = 1; o < G; o <<= 1) {
        const int x = __shfl_up_sync(g.mask, inc, o, G);
        if (g.gl >= o) inc += x;
    }
    const unsigned hit = g.ballot((int)r < inc);
    if (!hit) return -1;
    const int chunk = __ffs(hit) - 1;
    int rr = (int)r - (g.shfl(inc, chunk) - g.shfl(cnt, chunk));
    // stage 2: the chunk's CW words, G at a time
    const uint32_t *mb = d.mask_bits + (size_t)b * d.AW;
    for (int w0 = chunk * CW; w0 < (chunk + 1) * CW; w0 += G) {
        const int w = w0 + g.gl;
        const uint32_t word = (w < d.AW && w < (chunk + 1) * CW) ? mb[w] : 0u;
        const int c = __popc(word);
        int in2 = c;
#pragma unroll
        for (int o = 1; o < G; o <<= 1) {
            const int x = __shfl_up_sync(g.mask, in2, o, G);
            if (g.gl >= o) in2 += x;
        }
        const int tot = g.shfl(in2, G - 1);
        if (rr < tot) {
            const unsigned h2 = g.ballot(rr < in2);
            const int sl = __ffs(h2) - 1;
            int pos = (g.gl == sl) ? nth_set_bit(word, rr - (in2 - c)) : 0;
            pos = g.shfl(pos, sl);
            return ((w0 + sl) << 5) + pos;
        }
        rr -= tot;
    }
    return -1;
}

// State init + first mask (tail of reset()) for the tree-growing kinds.  Returns nothing; all lanes.
template <int G>
__device__ __forceinline__ void incr_reset_tree(const ge_batch &d, int b, const Grp<G> &g) {
    const int lane = g.gl;
    const bool mc = d.kind == GE_MULTICAST_ROUTING;
    const int src = mc ? 0 : d.src[b];
    const int32_t *rp = d.row_ptr + (size_t)b * d.RP;
    const int32_t *col = d.col + (size_t)b * d.MP;
    for (int w = lane; w < d.NW; w += G) d.node_bits[(size_t)b * d.NW + w] = (w == (src >> 5)) ? (1u << (src & 31)) : 0u;
    mask_zero<G>(d, b, lane);
    if (mc) {
        for (int w = lane; w < d.MW; w += G) d.edge_bits[(size_t)b * d.MW + w] = 0;
        for (int v = lane; v < d.N; v += G) d.dist32[(size_t)b * d.N + v] = (v == 0) ? 0.f : -1.f;
        if (d.bestkey)
            for (int v = lane; v < d.N; v += G) d.bestkey[(size_t)b * d.N + v] = KEY_NONE;
    }
    g.sync();
    __threadfence_block();
    const int lo = rp[src], hi = rp[src + 1];
    for (int e = lo + lane; e < hi; e += G) {  // every edge out of the root is valid (and is the best edge of its head)
        mask_set(d, b, e);
        if (mc && d.bestkey) {
            float c = __fadd_rn(0.f, d.w32[(size_t)b * d.MP + e]);
            d.bestkey[(size_t)b * d.N + col[e]] = ((u64)__float_as_uint(c) << 32) | (uint32_t)e;
        }
    }
    if (lane == 0) {
        d.head[b] = src;
        d.cost[b] = 0.0;
        d.done[b] = 0;
        // counters: [0] targets in the tree, [1] popcount of the mask, [2] constraints satisfied, [3] unused
        *reinterpret_cast<int4 *>(d.counters + (size_t)b * 4) = make_int4(0, hi - lo, 0, 0);
    }
}

struct Out {
    double reward, sol;
    int done, solved, has_mask, status;
};

__device__ __forceinline__ void publish(const ge_batch &d, const ge_step_out &out, int b, int a, const Out &r, uint32_t nsteps) {
    out.reward[b] = (float)r.reward;
    ge_step_flags f;
    f.done = (uint8_t)r.done; f.solved = (int8_t)r.solved; f.status = (uint8_t)r.status; f.has_mask = (uint8_t)r.has_mask;
    out.flags[b] = f;
    out.solution_cost[b] = r.sol;
    if (d.traj) {
        u64 cs = d.traj[b];
        d.traj[b] = ((cs << 7) | (cs >> 57)) ^ (u64)(uint32_t)a ^ ((u64)r.done << 40) ^ ((u64)(r.solved & 3) << 44) ^ ((u64)r.status << 48);
    }
    if (r.status == GE_STEP_OK) {
        if (d.env_steps) d.env_steps[b] = nsteps + 1u;
        d.acc[2 * (size_t)d.acc_stride + b] += r.reward;
        if (r.done) {
            d.acc[b] += 1.0;
            if (r.solved == 1) d.acc[(size_t)d.acc_stride + b] += 1.0;
            if (r.sol == r.sol) d.acc[3 * (size_t)d.acc_stride + b] += r.sol;
        }
    }
}

template <bool SAMPLED, int G>
__global__ void __launch_bounds__(GE_WPB * 32, GE_INCR_MINB) incr_tree_step_kernel(ge_batch d, int32_t *__restrict__ actions, ge_step_out out,
                                                                   uint64_t seed, uint32_t t) {
    const Grp<G> g;
    const int lane = g.gl;  // lane inside the env's group
    const int b = blockIdx.x * (GE_WPB * 32 / G) + (int)threadIdx.x / G;
    pdl_launch_dependents();   // programmatic dependent launch (ge_common.cuh): no-ops on a plain launch
    pdl_wait();
    if (b >= d.B) return;
    const bool mc = d.kind == GE_MULTICAST_ROUTING;
    const int N = d.N;
    const uint32_t nsteps = d.env_steps ? d.env_steps[b] : 0u;
    int4 c = *reinterpret_cast<const int4 *>(d.counters + (size_t)b * 4);  // [1] = popcount of the mask
    uint32_t *nb = d.node_bits + (size_t)b * d.NW;
    const uint32_t *tg = d.target_bits + (size_t)b * d.NW;
    // tree / target bitsets live in registers (lane w holds word w) when they fit: membership tests of the
    // row's endpoints become shuffles instead of a dependent round trip to memory
    const bool regs = d.NW <= G;
    const uint32_t nbw = (regs && lane < d.NW) ? nb[lane] : 0u;
    const uint32_t tgw = (regs && lane < d.NW) ? tg[lane] : 0u;
    int a;
    if (SAMPLED) {
        const uint32_t *mbits = d.mask_bits + (size_t)b * d.AW;
        // small masks (<= 4 words per lane, e.g. config 3's 32 words): the whole mask in registers, one memory round
        // (cfg3: 20.5 -> 18.8 us per step).  Larger masks keep the walk: 16 words per lane spill at this kernel's 32-register
        // budget and measured slower at config 5 (162 vs 155 us).
        if (d.AW <= 4 * G) a = group_sample_regs<G, 4>(g, mbits, d.AW, seed, (uint32_t)(d.env_id0 + b), t + nsteps, c.y);
        else if (d.mask_cnt && G >= 16) a = group_sample_chunks<G>(g, d, b, seed, (uint32_t)(d.env_id0 + b), t + nsteps, c.y);
        else a = group_sample<G>(g, mbits, d.AW, seed, (uint32_t)(d.env_id0 + b), t + nsteps, c.y);
        if (lane == 0) actions[b] = a;
    } else {
        a = actions[b];
    }
    Out r;
    r.reward = 0.0; r.sol = __longlong_as_double(0x7ff8000000000000ll); r.done = 0; r.solved = -1; r.has_mask = 1; r.status = GE_STEP_OK;
    if (d.done[b]) {
        r.has_mask = 0; r.status = GE_STEP_AFTER_DONE;
        if (lane == 0) publish(d, out, b, a, r, nsteps);
        return;
    }
    // one lane reads the validity bit and broadcasts it: the mask words are mutated further down by other lanes of the
    // group, and every lane must take the same branch here
    uint32_t okw = 0;
    if (lane == 0 && a >= 0 && a < d.A) okw = (d.mask_bits[(size_t)b * d.AW + (a >> 5)] >> (a & 31)) & 1u;
    const bool ok = g.shfl(okw, 0) != 0u;
    if (!ok) {
        r.status = GE_STEP_INVALID; r.has_mask = 0;
        if (lane == 0) publish(d, out, b, a, r, nsteps);
        return;
    }
    const int32_t *rp = d.row_ptr + (size_t)b * d.RP;
    const int32_t *col = d.col + (size_t)b * d.MP;
    const float *w32 = d.w32 + (size_t)b * d.MP;
    const int v = col[a];
    const float w = w32[a];
    const float cost32 = __fadd_rn((float)d.cost[b], w);
    const uint32_t tgv = regs ? g.shfl(tgw, v >> 5) : tg[v >> 5];
    const bool v_is_target = (tgv >> (v & 31)) & 1u;
    const int lo = rp[v], hi = rp[v + 1];
    float dv = 0.f;
    bool violated = false;
    float rew = -w;
    if (mc) {                                                               // multicast_routing.py:191-266
        if (d.parenting >= 3) {
            // `a` is valid => it IS the running-argmin edge of v, whose key holds float32(dist[src a] + delay[a]) in its
            // high word: the very value of :228, computed with the same float32 add when the edge was folded in.
            // No esrc[a] / dist[u] round trip (two scattered sectors).
            uint32_t hi32 = 0;                                              // lane 0 reads (it rewrites best[v] below), the group shares it
            if (lane == 0) hi32 = (uint32_t)(reinterpret_cast<const u64 *>(d.bestkey)[(size_t)b * N + v] >> 32);
            dv = __uint_as_float(g.shfl(hi32, 0));
        } else {
            const int u = d.esrc[(size_t)b * d.MP + a];
            dv = __fadd_rn(d.dist32[(size_t)b * N + u], w);                 // float32 add (:228)
        }
        r.sol = -1.0;
        if (v_is_target) {
            float lim = __fadd_rn(d.max_dist32[b], 1e-4f);                  // float32 compare under numpy 2 (:232)
            if (dv > lim) violated = true;
            else { rew = __fadd_rn(rew, 1.0f); c.z += 1; }
        }
    }
    c.x += v_is_target ? 1 : 0;
    // ---- mask delta around row(v).  node_bits of the neighbours are read before v's bit is published;
    //      v itself is never its own neighbour.
    int gained = 0, lost = 0;
    if (mc && d.parenting >= 3) {
        u64 *best = reinterpret_cast<u64 *>(d.bestkey) + (size_t)b * N;
        if (lane == 0) { mask_clear(d, b, a); best[v] = KEY_NONE; }         // a IS the best edge of v under parenting >= 3
        lost = 1;
        for (int e0 = lo; e0 < hi; e0 += G) {
            const int e = e0 + lane;
            const int x = e < hi ? col[e] : 0;
            const uint32_t xw = regs ? g.shfl(nbw, x >> 5) : nb[x >> 5];
            if (e < hi && !((xw >> (x & 31)) & 1u)) {
                u64 key = ((u64)__float_as_uint(__fadd_rn(dv, w32[e])) << 32) | (uint32_t)e;
                u64 old = best[x];
                if (key < old) {                                            // np.argmin: lowest edge index on ties (:179-185)
                    best[x] = key;
                    if (old != KEY_NONE) mask_clear(d, b, (int)(uint32_t)old); else gained++;
                    mask_set(d, b, e);
                }
            }
        }
    } else {
        const int32_t *rev = d.rev + (size_t)b * d.MP;
        for (int e0 = lo; e0 < hi; e0 += G) {
            const int e = e0 + lane;
            const int x = e < hi ? col[e] : 0;
            const uint32_t xw = regs ? g.shfl(nbw, x >> 5) : nb[x >> 5];
            if (e < hi) {
                if ((xw >> (x & 31)) & 1u) { mask_clear(d, b, rev[e]); lost++; }   // x->v was valid, is not any more
                else { mask_set(d, b, e); gained++; }                                 // v->x becomes valid
            }
        }
    }
    gained = g.sum(gained);
    lost = g.sum(lost);
    if (mc && d.parenting >= 3) lost = 1;
    c.y += gained - lost;
    g.sync();
    if (lane == 0) {
        nb[v >> 5] |= 1u << (v & 31);
        if (mc) {
            d.dist32[(size_t)b * N + v] = dv;
            d.edge_bits[(size_t)b * d.MW + (a >> 5)] |= 1u << (a & 31);
        }
    }
    // ---- outcome
    if (mc) {
        const float penalty = (float)(-2 * N * d.n_dests);
        if (violated) { r.reward = penalty; r.done = 1; r.solved = 0; }      // :231-237
        else {
            r.reward = rew;
            if (c.x == d.n_dests) { r.done = 1; r.solved = 1; r.sol = (double)cost32; }
            else if (c.y == 0) { r.reward = penalty; r.done = 1; r.solved = 0; }   // :254-258
        }
    } else {                                                                 // steiner_tree.py:123-157
        r.reward = -(double)w;
        if (c.x == d.n_dests) { r.done = 1; r.solved = 1; r.sol = (double)cost32; }
    }
    if (lane == 0) {
        publish(d, out, b, a, r, nsteps);
        d.cost[b] = (double)cost32;
        *reinterpret_cast<int4 *>(d.counters + (size_t)b * 4) = c;
        if (r.done) d.done[b] = 1;
    }
    if (r.done && (d.flags & GE_FLAG_AUTO_RESET)) {
        g.sync();
        __threadfence_block();
        incr_reset_tree<G>(d, b, g);
    }
}

__global__ void __launch_bounds__(GE_WPB * 32) incr_tree_reset_kernel(ge_batch d, const uint8_t *__restrict__ select) {
    const Grp<32> g;
    const int b = blockIdx.x * GE_WPB + ((int)threadIdx.x >> 5);
    if (b >= d.B) return;
    if (select && !select[b]) return;
    incr_reset_tree<32>(d, b, g);
}

// ---- MaxIndependentSet, one lane per env (any N): the mask loses bit `a`; episode ends after N picks.
template <bool SAMPLED>
__global__ void __launch_bounds__(256) incr_mis_step_kernel(ge_batch d, int32_t *__restrict__ actions, ge_step_out out, uint64_t seed,
                                                          uint32_t t) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    pdl_launch_dependents();   // programmatic dependent launch (ge_common.cuh): no-ops on a plain launch
    pdl_wait();
    if (b >= d.B) return;
    const int N = d.N;
    const uint32_t nsteps = d.env_steps ? d.env_steps[b] : 0u;
    uint32_t *mb = d.mask_bits + (size_t)b * d.AW;
    int4 c = *reinterpret_cast<const int4 *>(d.counters + (size_t)b * 4);  // [0] = nodes taken
    int a;
    if (SAMPLED) {  // r-th set bit of the packed mask; popcount = N - taken
        int total = N - c.x;
        a = -1;
        if (total > 0) {
            uint32_t r = (uint32_t)(((uint64_t)mix32(seed, (uint32_t)(d.env_id0 + b), t + nsteps) * (uint64_t)total) >> 32);
            for (int w = 0; w < d.AW; ++w) {
                uint32_t word = mb[w];
                int pc = __popc(word);
                if ((int)r < pc) { a = (w << 5) + nth_set_bit(word, (int)r); break; }
                r -= pc;
            }
        }
        actions[b] = a;
    } else {
        a = actions[b];
    }
    Out r;
    r.reward = 0.0; r.sol = __longlong_as_double(0x7ff8000000000000ll); r.done = 0; r.solved = -1; r.has_mask = 1; r.status = GE_STEP_OK;
    if (d.done[b]) { r.has_mask = 0; r.status = GE_STEP_AFTER_DONE; publish(d, out, b, a, r, nsteps); return; }
    if (!(a >= 0 && a < N && ((mb[a >> 5] >> (a & 31)) & 1u))) { r.status = GE_STEP_INVALID; r.has_mask = 0; publish(d, out, b, a, r, nsteps); return; }
    const float w = d.node_cost[(size_t)b * N + a];                        // max_independent_set.py:102-124
    const float cost32 = __fadd_rn((float)d.cost[b], w);
    r.reward = -(double)w;
    c.x += 1;
    if (c.x == N) { r.done = 1; r.solved = 1; r.sol = (double)cost32; }   // mask empty <=> all N nodes taken
    publish(d, out, b, a, r, nsteps);
    if (r.done && (d.flags & GE_FLAG_AUTO_RESET)) {
        for (int wi = 0; wi < d.NW; ++wi) { d.node_bits[(size_t)b * d.NW + wi] = 0; mb[wi] = tail_mask(N, wi); }
        d.cost[b] = 0.0;
        d.head[b] = 0;
        *reinterpret_cast<int4 *>(d.counters + (size_t)b * 4) = make_int4(0, 0, 0, 0);
        return;
    }
    d.node_bits[(size_t)b * d.NW + (a >> 5)] |= 1u << (a & 31);
    mb[a >> 5] &= ~(1u << (a & 31));
    d.cost[b] = (double)cost32;
    *reinterpret_cast<int4 *>(d.counters + (size_t)b * 4) = c;
    if (r.done) d.done[b] = 1;
}

__global__ void __launch_bounds__(256) incr_mis_reset_kernel(ge_batch d, const uint8_t *__restrict__ select) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= d.B) return;
    if (select && !select[b]) return;
    const int N = d.N;
    for (int wi = 0; wi < d.NW; ++wi) { d.node_bits[(size_t)b * d.NW + wi] = 0; d.mask_bits[(size_t)b * d.AW + wi] = tail_mask(N, wi); }
    d.cost[b] = 0.0;
    d.head[b] = 0;
    d.done[b] = 0;
    *reinterpret_cast<int4 *>(d.counters + (size_t)b * 4) = make_int4(0, 0, 0, 0);
}

}  // namespace

// ------------------------------------------------------------------ host launchers (called from ge_api.cu)
bool ge_incr_eligible(const ge_batch *d) {
    if (d->flags & GE_FLAG_FORCE_WARP) return false;
    if (d->kind == GE_STEINER_TREE) return d->rev != nullptr;
    if (d->kind == GE_MULTICAST_ROUTING)
        return d->parenting >= 3 ? d->bestkey != nullptr : (d->parenting == 2 && d->esrc != nullptr && d->rev != nullptr);
    if (d->kind == GE_MAX_INDEPENDENT_SET) return d->N > 64;  // N <= 64 is the lane-per-env family's
    return false;
}

static int launched(const char *what) {
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? GE_OK : ge_set_error(GE_ERR_CUDA, "%s launch: %s", what, cudaGetErrorString(e));
}

int ge_incr_step(const ge_batch *d, int32_t *actions, const ge_step_out *out, bool sampled, uint64_t seed, uint32_t t, cudaStream_t st) {
    if (d->kind == GE_MAX_INDEPENDENT_SET) {
        ge_launch_step(sampled ? incr_mis_step_kernel<true> : incr_mis_step_kernel<false>, dim3((d->B + 255) / 256), dim3(256), 0, st, *d, actions, *out, seed, t);
        return launched("incr_mis_step_kernel");
    }
    // lanes per env: wide enough to hold the node bitsets in registers (NW <= G) and a typical row in one pass
    const int G = d->NW <= 8 ? 8 : d->NW <= 16 ? 16 : 32;
    const int per_block = GE_WPB * 32 / G;
    const int blocks = (d->B + per_block - 1) / per_block;
    auto kernel = G == 8 ? (sampled ? incr_tree_step_kernel<true, 8> : incr_tree_step_kernel<false, 8>)
                : G == 16 ? (sampled ? incr_tree_step_kernel<true, 16> : incr_tree_step_kernel<false, 16>)
                          : (sampled ? incr_tree_step_kernel<true, 32> : incr_tree_step_kernel<false, 32>);
    ge_launch_step(kernel, dim3(blocks), dim3(GE_WPB * 32), 0, st, *d, actions, *out, seed, t);
    return launched("incr_tree_step_kernel");
}

int ge_incr_reset(const ge_batch *d, const uint8_t *select, cudaStream_t st) {
    if (d->kind == GE_MAX_INDEPENDENT_SET) {
        incr_mis_reset_kernel<<<(d->B + 255) / 256, 256, 0, st>>>(*d, select);
        return launched("incr_mis_reset_kernel");
    }
    incr_tree_reset_kernel<<<(d->B + GE_WPB - 1) / GE_WPB, GE_WPB * 32, 0, st>>>(*d, select);
    return launched("incr_tree_reset_kernel");
}
