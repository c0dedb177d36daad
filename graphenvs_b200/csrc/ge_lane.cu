// ge_lane.cu -- ONE LANE PER ENVIRONMENT kernels for small graphs (N <= 64, node-action kinds).
//
// Why: ncu on the warp-per-env step kernel at BASELINE config 2 (LongestPath N=50, B=65536) showed
// 817 warp-instructions per env-step at 45 % issue utilisation and 6.6 % of HBM peak
// (profiles/r01_step_kernel_cfg2_warp_per_env.md): with a 50-node graph every scalar instruction
// of a warp is 32-wide redundant.  Here an env's node sets are single 64-bit registers of ONE
// thread, a warp advances 32 envs, and the only graph data a step needs -- the N x NW adjacency
// bit-matrix -- is staged for the whole block with ONE bulk asynchronous copy (cp.async.bulk,
// SASS UBLKCP) into shared memory while the threads load their scalar state.  The matrix is stored in
// tiles of 32 envs ([tile][row][env], ge_common.cuh:adj_tiled) so that the lane-private row reads of a
// warp never collide on a shared-memory bank, whichever rows the 32 searches are at.
//
// Semantics are those of ge_envs.cuh (same reference line map); tests run every N <= 64 case
// through both paths (GE_FLAG_FORCE_WARP).
#include "ge_common.cuh"

using namespace ge;

extern "C" int ge_set_error(int code, const char *fmt, ...);

// Envs (= threads) per block: one tile.  Small blocks spread the arrival times of the staged copies, so the searches of
// early blocks overlap the transfers of late ones (single-wave launches otherwise alternate between an
// all-memory and an all-compute phase): 9.96 vs 10.17 us per cfg2 step under the streaming protocol; no
// difference when a step runs alone.
constexpr int LANE_T = 32;
// __launch_bounds__ of the lane kernels.  It sets their register budget: with a bound of 32 the compiler gives the
// step kernels 63 instead of 56 registers, a build nobody has measured.
constexpr int LANE_BOUND = 128;
// Minimum resident blocks of LANE_BOUND threads the step kernels declare: a cap of 65,536 / (128 x 8) = 64 registers.  The
// unstaged step kernels run 32 one-warp blocks per SM at 64; left to itself ptxas gives them 56 and spills 12 bytes.
constexpr int LANE_STEP_MIN_BLOCKS = 8;

namespace {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(ok)
                     : "r"(smem_u32(bar)), "r"(parity)
                     : "memory");
    } while (!ok);
}

// kinds/modes whose mask needs reachability over the residual graph => whole bit-matrix staged
__host__ __device__ inline bool lane_stages(const ge_batch &d) {
    return (d.kind == GE_LONGEST_PATH || d.kind == GE_TSP) && d.parenting >= 2;
}

template <bool STAGED>
struct Rows {  // adjacency rows of one env in the TILED layout (ge_common.cuh:adj_tiled): shared-memory copy (STAGED, explicit LDS) or global
    const uint32_t *p;  // element (row 0, this env)
    uint32_t sp;        // shared-window address of the same element when STAGED
    int NW;
    __device__ __forceinline__ u64 row(int r) const {
        if (STAGED) {   // rows of one tile are 32 elements apart: any 32 rows picked by the 32 lanes hit 32 different banks
            if (NW == 1) {
                uint32_t v;
                asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(sp + 128u * (uint32_t)r));
                return (u64)v;
            }
            u64 v;
            asm volatile("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(sp + 256u * (uint32_t)r));
            return v;
        }
        if (NW == 1) return (u64)__ldg(p + 32 * r);
        uint2 t = __ldg(reinterpret_cast<const uint2 *>(p + 64 * r));
        return (u64)t.x | ((u64)t.y << 32);
    }
};

// Worklist reachability from `seed` inside `allowed` (seed subset of allowed, one bit); stops early
// once everything in `allowed` is reached.  Each trip pops up to EIGHT frontier nodes -- four from
// each 32-bit half, the find-first-set chains of the two halves are independent -- and ORs their rows:
// the shared-memory loads are in flight together and the dependent chain of a search is
// ~|reach|/8 trips instead of |reach| (measured: 1 -> 4 pops per trip 8.4 -> 4.9 us of search per 65,536-env
// step, 4 -> 8 pops another 3 % of the step) (the lane-per-env kernels run at ~4 warps per scheduler,
// so per-warp latency, not issue rate, is what a step waits for).  An empty slot re-expands the
// seed, which is harmless.
template <bool STAGED>
__device__ __forceinline__ u64 reach_within(const Rows<STAGED> &R, u64 seed, u64 allowed, u64 need) {
    // `need` (subset of allowed): the search may stop as soon as all of it is reached -- LongestPath only asks
    // about the handful of candidates next to the head, which a well-connected residual graph reaches in one
    // or two trips (reaching the LAST of ~45 allowed nodes took |allowed| / 8 trips).  need == allowed is the
    // plain "everything reached" test.  On an empty frontier the returned set is the full component.
    const int sidx = __ffsll((long long)seed) - 1;
    u64 reach = seed, frontier = seed;
    while (frontier) {
        uint32_t lo = (uint32_t)frontier, hi = (uint32_t)(frontier >> 32);
        uint32_t lo2 = lo & (lo - 1u), lo3 = lo2 & (lo2 - 1u), lo4 = lo3 & (lo3 - 1u);
        uint32_t hi2 = hi & (hi - 1u), hi3 = hi2 & (hi2 - 1u), hi4 = hi3 & (hi3 - 1u);
        u64 a = R.row(lo ? __ffs((int)lo) - 1 : sidx) | R.row(lo2 ? __ffs((int)lo2) - 1 : sidx) |
                R.row(lo3 ? __ffs((int)lo3) - 1 : sidx) | R.row(lo4 ? __ffs((int)lo4) - 1 : sidx);
        if (R.NW > 1)
            a |= R.row(hi ? 31 + __ffs((int)hi) : sidx) | R.row(hi2 ? 31 + __ffs((int)hi2) : sidx) |
                 R.row(hi3 ? 31 + __ffs((int)hi3) : sidx) | R.row(hi4 ? 31 + __ffs((int)hi4) : sidx);
        u64 rest = (u64)(lo4 & (lo4 - 1u)) | ((u64)(hi4 & (hi4 - 1u)) << 32);
        u64 nx = a & allowed & ~reach;
        reach |= nx;
        frontier = rest | nx;
        if (!(need & ~reach)) break;
    }
    return reach;
}

struct LState {
    u64 vis, aux;
    int head, k, ecnt;
    double cost;
};

// ---- masks (ge_envs.cuh: mask_head_row / mask_longest_path / mask_tsp / mask_densest)
template <bool STAGED>
__device__ __forceinline__ u64 lane_mask(const ge_batch &d, const Rows<STAGED> &R, const LState &s, int dest, u64 full) {
    const int N = d.N;
    switch (d.kind) {
    case GE_SHORTEST_PATH: return R.row(s.head) & ~s.vis;                    // shortest_path.py:105-109
    case GE_LONGEST_PATH: {                                                    // longest_path.py:125-145
        if (d.parenting == 0) return full;
        u64 m = R.row(s.head) & ~s.vis;
        if (d.parenting < 2) return m;
        if ((s.vis >> dest) & 1ull) return m;                                  // dest not in alt_G (:135-136)
        u64 allowed = ~s.vis & full;
        if (m) m &= reach_within(R, 1ull << dest, allowed, m);               // has_path(k, dest) for the candidates k (:137-140)
        if (d.parenting == 3 && __popcll(allowed) <= N / 3) m |= allowed;     // :141-143
        return m; }
    case GE_TSP: {                                                             // tsp.py:174-199
        u64 m = R.row(s.head) & ~s.vis;
        if (__popcll(s.vis) < N - 1) m &= ~1ull;                               // :178-179
        if (d.parenting < 2) return m;
        u64 res = ~s.vis & full & ~1ull;                                       // alt_G = all - start - taken
        int n_res = __popcll(res);
        u64 cand = m;
        // One spanning search of alt_G first: a node whose expansion discovered nothing is a LEAF of
        // a spanning tree, and removing a leaf cannot disconnect the graph -- only the tree's
        // internal nodes still need the literal "remove v, test connectivity" of tsp.py:186-194.
        if (n_res >= 2) {
            u64 seed = res & (~res + 1ull), reach = seed, frontier = seed, internal = 0;
            while (frontier && reach != res) {
                int r = __ffsll((long long)frontier) - 1;
                frontier &= frontier - 1;
                u64 nx = R.row(r) & res & ~reach;
                if (nx) internal |= 1ull << r;
                reach |= nx;
                frontier |= nx;
            }
            if (reach == res) cand &= internal | 1ull;   // (bit 0 = start is skipped below anyway)
        }
        while (cand) {
            int v = __ffsll((long long)cand) - 1;
            cand &= cand - 1;
            if (v == 0) continue;
            if (n_res - 1 == 0) break;                                         // :191-192
            u64 g = res & ~(1ull << v);
            u64 seed = g & (~g + 1ull);                                        // lowest node of G_copy
            if (reach_within(R, seed, g, g) != g) m &= ~(1ull << v);           // :193-194
        }
        return m; }
    case GE_MAX_INDEPENDENT_SET: return ~s.vis & full;                         // max_independent_set.py:92-100
    case GE_DENSEST_SUBGRAPH:                                                  // densest_subgraph.py:105-129
        if (s.k == 0) return full;
        if (d.parenting == 0) return ~s.vis & full;
        return s.aux & ~s.vis & full;
    }
    return 0;
}

__device__ __forceinline__ void lane_init_state(const ge_batch &d, int src, LState &s) {  // src = 0 for unseeded kinds
    bool seeded = d.kind == GE_SHORTEST_PATH || d.kind == GE_LONGEST_PATH;
    s.vis = seeded ? (1ull << src) : 0ull;
    s.aux = 0;
    s.head = src;
    s.k = 0;
    s.ecnt = 0;
    s.cost = 0.0;
}

__device__ __forceinline__ void lane_store_state(const ge_batch &d, int b, const LState &s, u64 mask, bool counters) {
    if (d.NW == 1) {
        d.node_bits[b] = (uint32_t)s.vis;
        if (d.node_bits2) d.node_bits2[b] = (uint32_t)s.aux;
    } else {
        reinterpret_cast<uint2 *>(d.node_bits)[b] = make_uint2((uint32_t)s.vis, (uint32_t)(s.vis >> 32));
        if (d.node_bits2) reinterpret_cast<uint2 *>(d.node_bits2)[b] = make_uint2((uint32_t)s.aux, (uint32_t)(s.aux >> 32));
    }
    d.head[b] = s.head;
    d.cost[b] = s.cost;
    if (counters) *reinterpret_cast<int4 *>(d.counters + (size_t)b * 4) = make_int4(s.k, s.ecnt, 0, 0);
    // mask: the packed words only.  The byte view (mask_bytes) is expanded on demand by ge_mask_bytes
    // (ge_mask_bytes_current() == 0 for this family): keeping it current costs AP bytes per env and ~16 % of the
    // step's warp instructions, for a view the samplers and the packed host results do not read.
    if (d.AW == 1) d.mask_bits[b] = (uint32_t)mask;
    else reinterpret_cast<uint2 *>(d.mask_bits)[b] = make_uint2((uint32_t)mask, (uint32_t)(mask >> 32));
}

// adj[u, v] of the reference's dense float64 matrix (shortest_path.py:82); 0 when there is no edge.
// One dependent load from the resident N x N matrix instead of a CSR row scan.
__device__ __forceinline__ double lane_edge_weight(const ge_batch &d, int b, int u, int v) {
    return __ldg(d.wmat + ((size_t)b * d.N + u) * d.N + v);
}

__device__ __forceinline__ u64 load_bits64(const uint32_t *base, int b, int NW) {
    if (NW == 1) return (u64)base[b];
    uint2 t = reinterpret_cast<const uint2 *>(base)[b];
    return (u64)t.x | ((u64)t.y << 32);
}

// Before pdl_wait() the previous launch may still be writing the dynamic state.  These two touch it without being able to
// hand a stale value to the loads after the wait: an L2 prefetch moves no data into the SM, and an L2 load (ld.global.cg, no
// L1 allocation) returns a value that only steers such a prefetch.  L2 is the point of coherence, so the loads after the
// wait see the previous launch's writes either way.
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ uint32_t load_l2(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.global.cg.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ u64 load_l2_bits64(const uint32_t *base, int b, int NW) {
    if (NW == 1) return (u64)load_l2(base + b);
    u64 v;
    asm volatile("ld.global.cg.u64 %0, [%1];" : "=l"(v) : "l"(base + 2 * (size_t)b));
    return v;
}

// Stages the adjacency tiles of the block's envs (blockDim.x / 32 tiles of 32 envs, contiguous) with one bulk
// copy; returns this env's rows.
template <bool STAGED>
__device__ __forceinline__ Rows<STAGED> stage_rows(const ge_batch &d, int b0, uint32_t *smem, uint64_t *bar) {
    Rows<STAGED> R;
    R.NW = d.NW;
    R.sp = 0;
    const int b = min(b0 + (int)threadIdx.x, d.B - 1);
    const size_t tile_words = (size_t)d.N * 32 * d.NW;
    R.p = d.adj_bits + (size_t)(b >> 5) * tile_words + (size_t)(b & 31) * d.NW;
    if (!STAGED) return R;
    if (threadIdx.x == 0) mbar_init(bar, 1);
    __syncthreads();
    if (threadIdx.x == 0) {
        const int ntiles = (min((int)blockDim.x, d.B - b0) + 31) >> 5;     // adj_bits holds whole tiles (B rounded up to 32 envs)
        const uint32_t bytes = (uint32_t)(ntiles * tile_words * 4);        // a multiple of 128
        mbar_expect_tx(bar, bytes);
        bulk_g2s(smem, d.adj_bits + (size_t)(b0 >> 5) * tile_words, bytes, bar);
    }
    R.sp = smem_u32(smem + (size_t)(threadIdx.x >> 5) * tile_words + (size_t)(threadIdx.x & 31) * d.NW);
    return R;
}

// *p += v as a fire-and-forget reduction (SASS REDG.E.ADD.F64.RN): the SM neither loads the statistics rows nor waits for
// them.  Every element has one writer per launch and launches are ordered by grid completion, and the fp64 reduction rounds
// to nearest even like the `*p + v` of a load-add-store, so the rows are bit-identical to one.  Explicit PTX because ptxas
// keeps an atomicAdd whose result is unused an ATOMG (which returns) when a fence may follow, as signal_progress's does.
__device__ __forceinline__ void red_add(double *p, double v) {
    asm volatile("red.relaxed.gpu.global.add.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}

// r-th set bit of a 64-bit mask, r uniform from the counter RNG (same draw as ge_common.cuh:warp_sample).
__device__ __forceinline__ int lane_sample(u64 m, uint64_t seed, uint32_t env, uint32_t t) {
    int total = __popcll(m);
    if (total <= 0) return -1;
    uint32_t r = (uint32_t)(((uint64_t)mix32(seed, env, t) * (uint64_t)total) >> 32);
    uint32_t lo = (uint32_t)m, hi = (uint32_t)(m >> 32);
    int clo = __popc(lo);
    return (int)r < clo ? nth_set_bit(lo, (int)r) : 32 + nth_set_bit(hi, (int)r - clo);
}

template <bool STAGED, bool SAMPLED>
__global__ void __launch_bounds__(LANE_BOUND, LANE_STEP_MIN_BLOCKS) lane_step_kernel(ge_batch d, int32_t *__restrict__ actions, ge_step_out out,
                                                            uint64_t seed, uint32_t t) {
    extern __shared__ __align__(128) uint32_t smem[];
    __shared__ __align__(8) uint64_t bar;
    const int b0 = blockIdx.x * blockDim.x, b = b0 + threadIdx.x;
    // Programmatic dependent launch (ge_common.cuh:pdl_*; no-ops on a plain launch): the next launch in the stream may
    // become resident now, and everything up to pdl_wait() reads only STATIC instance data (the adjacency tiles, dest, src,
    // the reset-time mask) or reaches the dynamic state through L2 alone (prefetch_l2 / load_l2), so it runs under the tail
    // of the previous launch.  A stream that steps other batches in between (sub-batch chains rotating over batches) leaves
    // this batch's state final while the block waits, and the block's loads after the wait hit L2.
    pdl_launch_dependents();
    Rows<STAGED> R = stage_rows<STAGED>(d, b0, smem, &bar);
    const bool live = b < d.B;
    const int N = d.N, kind = d.kind;
    const u64 full = N == 64 ? ~0ull : ((1ull << N) - 1ull);
    const bool needs_w = kind == GE_SHORTEST_PATH || kind == GE_LONGEST_PATH || kind == GE_TSP;
    int dest = 0, src = 0;
    u64 mask0 = 0;
    if (live) {
        if (kind == GE_SHORTEST_PATH || kind == GE_LONGEST_PATH) { dest = d.dest[b]; src = d.src[b]; }
        if (d.mask0_bits && (d.flags & GE_FLAG_AUTO_RESET)) mask0 = load_bits64(d.mask0_bits, b, d.AW);
        prefetch_l2(d.node_bits + (size_t)b * d.NW);
        if (d.node_bits2) prefetch_l2(d.node_bits2 + (size_t)b * d.NW);
        prefetch_l2(d.cost + b);
        prefetch_l2(d.done + b);
        if (d.traj) prefetch_l2(d.traj + b);
        if (kind == GE_DENSEST_SUBGRAPH) prefetch_l2(d.counters + (size_t)b * 4);
        if (!SAMPLED) prefetch_l2(actions + b);
        if (SAMPLED && needs_w) {
            // Guess this step's draw from the state as it is now and prefetch its edge weight, the step's one dependent
            // load.  Right whenever the previous launch did not step this batch; a wrong guess costs one wasted line.
            const u64 m = load_l2_bits64(d.mask_bits, b, d.AW);
            const uint32_t ns = d.env_steps ? load_l2(d.env_steps + b) : 0u;
            const int h = min(max((int)load_l2(reinterpret_cast<const uint32_t *>(d.head) + b), 0), N - 1);
            const int ga = min(max(lane_sample(m, seed, (uint32_t)(d.env_id0 + b), t + ns), 0), N - 1);
            prefetch_l2(d.wmat + ((size_t)b * N + h) * N + ga);
        } else {
            prefetch_l2(d.head + b);
            prefetch_l2(d.mask_bits + (size_t)b * d.AW);
            if (d.env_steps) prefetch_l2(d.env_steps + b);
        }
    }
    pdl_wait();
    // scalar state (coalesced SoA streams) while the bulk copy is in flight
    LState s;
    int a = -1;
    u64 oldmask = 0, cs = 0;
    double w_edge = 0.0;
    float w_node = 0.f;
    bool was_done = false;
    uint32_t nsteps = 0;
    if (live) {
        if (!SAMPLED) a = actions[b];
        if (d.env_steps) nsteps = d.env_steps[b];
        s.vis = load_bits64(d.node_bits, b, d.NW);
        s.aux = d.node_bits2 ? load_bits64(d.node_bits2, b, d.NW) : 0ull;
        s.head = d.head[b];
        s.cost = d.cost[b];
        s.k = 0; s.ecnt = 0;
        if (kind == GE_DENSEST_SUBGRAPH) { int4 c = *reinterpret_cast<const int4 *>(d.counters + (size_t)b * 4); s.k = c.x; s.ecnt = c.y; }
        oldmask = load_bits64(d.mask_bits, b, d.AW);
        if (SAMPLED) {
            a = lane_sample(oldmask, seed, (uint32_t)(d.env_id0 + b), t + nsteps);
            actions[b] = a;
        }
        was_done = d.done[b] != 0;
        if (d.traj) cs = d.traj[b];
        // the one dependent load of the step, issued before waiting for the staged rows
        if (needs_w && a >= 0 && a < N) w_edge = lane_edge_weight(d, b, s.head, a);
        if (kind == GE_MAX_INDEPENDENT_SET && a >= 0 && a < N) w_node = d.node_cost[(size_t)b * N + a];
    }
    if (STAGED) mbar_wait(&bar, 0);
    if (!live) return;

    double reward = 0.0, sol = __longlong_as_double(0x7ff8000000000000ll);
    int done = 0, solved = -1, has_mask = 1, status = GE_STEP_OK;
    u64 mask = oldmask;
    bool write_state = false;

    if (was_done) {
        has_mask = 0; status = GE_STEP_AFTER_DONE;
    } else if (kind == GE_TSP && a == 0 && s.head == 0) {                       // tsp.py:203-211
        done = 1; reward = -(double)N; solved = 0; sol = -1.0;
        mask = lane_mask(d, R, s, dest, full);
        write_state = true;
    } else if (!(a >= 0 && a < N && ((oldmask >> a) & 1ull))) {
        status = GE_STEP_INVALID; has_mask = 0;
    } else {
        write_state = true;
        const u64 abit = 1ull << a;
        switch (kind) {
        case GE_SHORTEST_PATH: {                                                // shortest_path.py:111-141
            s.vis |= abit; s.head = a;
            mask = lane_mask(d, R, s, dest, full);
            double w = w_edge;
            reward = -w;
            s.cost += w;
            if (a == dest) { done = 1; solved = 1; }
            if (!done && mask == 0) { done = 1; reward = -(double)N; solved = 0; }
            if (done) sol = s.cost;
            break; }
        case GE_LONGEST_PATH: {                                                 // longest_path.py:147-196
            bool nb = (R.row(s.head) >> a) & 1ull, vis = (s.vis >> a) & 1ull;
            if (d.parenting >= 1 && (!nb || vis)) { status = GE_STEP_INVALID; has_mask = 0; write_state = false; break; }
            if (nb && !vis) {                                                   // the search first: the weight
                s.head = a; s.vis |= abit;                                      // load stays in flight behind it
                mask = lane_mask(d, R, s, dest, full);
            }
            double w = nb ? w_edge : 0.0;
            reward = w;
            s.cost -= w;
            sol = s.cost;                                                       // every step (:163-165)
            if (!nb || vis) { done = 1; solved = 0; reward = -2.0 * N; has_mask = 0; break; }  // :169-173
            if (a == dest) { done = 1; solved = 1; }
            if (!done && mask == 0) { done = 1; reward = -2.0 * N; solved = 0; }
            break; }
        case GE_TSP: {                                                          // tsp.py:213-258
            s.vis |= abit; s.head = a;
            mask = lane_mask(d, R, s, dest, full);
            double w = w_edge;
            reward = 0.0 - w;
            s.cost += w;
            if (__popcll(s.vis) == N && a == 0) { done = 1; solved = 1; }
            if (!done && mask == 0) { done = 1; reward -= 2.0 * N; solved = 0; }
            if (done) sol = s.cost;
            break; }
        case GE_MAX_INDEPENDENT_SET: {                                          // max_independent_set.py:102-124
            float w = w_node;
            s.cost = (double)__fadd_rn((float)s.cost, w);
            reward = -(double)w;
            s.vis |= abit;
            mask = ~s.vis & full;
            if (mask == 0) { done = 1; solved = 1; sol = s.cost; }
            break; }
        case GE_DENSEST_SUBGRAPH: {                                             // densest_subgraph.py:135-196
            solved = 1;
            if (a == N - 1) { reward = 0.0; done = 1; sol = s.cost; break; }   // stop action (:148-154)
            u64 row = R.row(a);
            int ne = __popcll(row & s.vis);
            s.aux |= row;
            if (s.k == 0) reward = 0.0;
            else reward = ((double)(s.ecnt + ne) / (double)(s.k + 1)) - ((double)s.ecnt / (double)s.k);
            s.ecnt += ne; s.k += 1;
            s.vis |= abit;
            s.cost = (double)s.ecnt / (double)s.k;
            mask = lane_mask(d, R, s, dest, full);
            if (s.k == d.n_choices) { done = 1; sol = s.cost; }
            break; }
        }
    }

    out.reward[b] = (float)reward;
    ge_step_flags f;
    f.done = (uint8_t)done; f.solved = (int8_t)solved; f.status = (uint8_t)status; f.has_mask = (uint8_t)has_mask;
    out.flags[b] = f;
    out.solution_cost[b] = sol;
    if (d.traj)
        d.traj[b] = ((cs << 7) | (cs >> 57)) ^ (u64)(uint32_t)a ^ ((u64)done << 40) ^ ((u64)(solved & 3) << 44) ^ ((u64)status << 48);
    if (status == GE_STEP_OK) {
        if (d.env_steps) d.env_steps[b] = nsteps + 1u;
        const size_t st = (size_t)d.acc_stride;
        red_add(d.acc + 2 * st + b, reward);
        if (done) {
            red_add(d.acc + b, 1.0);
            if (solved == 1) red_add(d.acc + st + b, 1.0);
            if (sol == sol) red_add(d.acc + 3 * st + b, sol);
        }
    }
    if (done && (d.flags & GE_FLAG_AUTO_RESET)) {                               // tail of reset()
        lane_init_state(d, src, s);
        if (d.mask0_bits) mask = mask0;                                         // reset-time mask of this instance (ge_reset)
        else {
            mask = lane_mask(d, R, s, dest, full);
            if (kind == GE_TSP && mask == 0) mask = 1ull;                       // tsp.py:154-155
        }
        lane_store_state(d, b, s, mask, kind == GE_DENSEST_SUBGRAPH);
    } else if (write_state) {
        if (done) d.done[b] = 1;
        lane_store_state(d, b, s, mask, kind == GE_DENSEST_SUBGRAPH);
    }
    if (d.progress) signal_progress(d, b);   // streamed host step: this env's results may cross PCIe now
}

template <bool STAGED>
__global__ void __launch_bounds__(LANE_BOUND) lane_reset_kernel(ge_batch d, const uint8_t *__restrict__ select) {
    extern __shared__ __align__(128) uint32_t smem[];
    __shared__ __align__(8) uint64_t bar;
    const int b0 = blockIdx.x * blockDim.x, b = b0 + threadIdx.x;
    Rows<STAGED> R = stage_rows<STAGED>(d, b0, smem, &bar);
    const bool live = b < d.B && (!select || select[b]);
    int dest = 0, src = 0;
    if (live && (d.kind == GE_SHORTEST_PATH || d.kind == GE_LONGEST_PATH)) { dest = d.dest[b]; src = d.src[b]; }
    if (STAGED) mbar_wait(&bar, 0);
    if (!live) return;
    const u64 full = d.N == 64 ? ~0ull : ((1ull << d.N) - 1ull);
    LState s;
    lane_init_state(d, src, s);
    u64 mask = lane_mask(d, R, s, dest, full);
    if (d.kind == GE_TSP && mask == 0) mask = 1ull;
    d.done[b] = 0;
    *reinterpret_cast<int4 *>(d.counters + (size_t)b * 4) = make_int4(0, 0, 0, 0);
    if (d.mask0_bits) {
        if (d.AW == 1) d.mask0_bits[b] = (uint32_t)mask;
        else reinterpret_cast<uint2 *>(d.mask0_bits)[b] = make_uint2((uint32_t)mask, (uint32_t)(mask >> 32));
    }
    lane_store_state(d, b, s, mask, false);
}

// Uniform choice among the valid mask bits, one lane per env (A <= 64); same draw as sample_kernel.
__global__ void __launch_bounds__(256) lane_sample_kernel(ge_batch d, uint64_t seed, uint32_t t, int32_t *__restrict__ actions) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= d.B) return;
    u64 m = load_bits64(d.mask_bits, b, d.AW);
    if (d.env_steps) t += d.env_steps[b];
    actions[b] = lane_sample(m, seed, (uint32_t)(d.env_id0 + b), t);
}

}  // namespace

// ------------------------------------------------------------------ host launchers (called from ge_api.cu)
bool ge_lane_eligible(const ge_batch *d) {
    return d->N <= 64 && lane_kind(d->kind) && !(d->flags & GE_FLAG_FORCE_WARP) &&
           (d->adj_bits != nullptr || d->kind == GE_MAX_INDEPENDENT_SET);
}

static size_t lane_smem(const ge_batch *d) { return lane_stages(*d) ? (size_t)LANE_T * d->N * d->NW * 4 : 0; }

int ge_grant_smem(const void *kernel, size_t smem);  // ge_api.cu
template <class K>
static int lane_prepare(K kernel, size_t smem) { return ge_grant_smem((const void *)kernel, smem); }

int ge_lane_step(const ge_batch *d, int32_t *actions, const ge_step_out *out, bool sampled, uint64_t seed, uint32_t t, cudaStream_t st) {
    const size_t smem = lane_smem(d);
    const bool needs_w = d->kind == GE_SHORTEST_PATH || d->kind == GE_LONGEST_PATH || d->kind == GE_TSP;
    if (needs_w && !d->wmat) return ge_set_error(GE_ERR_ARG, "kind %d with N <= 64 needs wmat (ge_build_adjacency fills it)", d->kind);
    auto kernel = lane_stages(*d) ? (sampled ? lane_step_kernel<true, true> : lane_step_kernel<true, false>)
                                  : (sampled ? lane_step_kernel<false, true> : lane_step_kernel<false, false>);
    int rc = lane_prepare(kernel, smem);
    if (rc) return rc;
    cudaError_t e = ge_launch_step(kernel, dim3((d->B + LANE_T - 1) / LANE_T), dim3(LANE_T), smem, st, *d, actions, *out, seed, t);
    if (e != cudaSuccess) (void)cudaGetLastError();
    return e == cudaSuccess ? GE_OK : ge_set_error(GE_ERR_CUDA, "lane_step_kernel launch: %s", cudaGetErrorString(e));
}

int ge_lane_reset(const ge_batch *d, const uint8_t *select, cudaStream_t st) {
    const size_t smem = lane_smem(d);
    auto kernel = lane_stages(*d) ? lane_reset_kernel<true> : lane_reset_kernel<false>;
    int rc = lane_prepare(kernel, smem);
    if (rc) return rc;
    kernel<<<(d->B + LANE_T - 1) / LANE_T, LANE_T, smem, st>>>(*d, select);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? GE_OK : ge_set_error(GE_ERR_CUDA, "lane_reset_kernel launch: %s", cudaGetErrorString(e));
}

int ge_lane_sample(const ge_batch *d, uint64_t seed, uint32_t t, int32_t *actions, cudaStream_t st) {
    lane_sample_kernel<<<(d->B + 255) / 256, 256, 0, st>>>(*d, seed, t, actions);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? GE_OK : ge_set_error(GE_ERR_CUDA, "lane_sample_kernel launch: %s", cudaGetErrorString(e));
}
