// ge_ppd.cu -- PerishableProductDelivery-v0 (perishable_product_delivery.py:175-271), SURVEY 8(f4).  One warp per env.
//
// State the reference keeps as 16 node columns, kept here as what determines them:
//   head                      column 0 (IS_HEAD)
//   status of product i       0 = waiting at its pickup (HAS_P[i] = 1 there), 1 = in transit (the whole HAS_P[i] column is -1),
//                             2 = delivered (HAS_P[i], NEEDS_P[i], TIME_LEFT[i] columns all 0)      -> counters[b].x, 2 bits each
//   moves made                len(edges_taken)                                                       -> counters[b].y
//   solution_cost             fp64                                                                   -> cost[b]
// Static: pickups / dropoffs = targets[b, 0:P] / targets[b, P:2P] (P = n_dests = n_products), delivery_time (float32, the
// TIME_LEFT columns) = max_dist32[b].  The reference's clock never runs: it subtracts adj[head, action] AFTER head = action
// (:225,:234), i.e. adj[a, a] = 0, so TIME_LEFT stays at delivery_time until the product is delivered; restated literally.
// info['solution_cost'] is the value BEFORE the move (:211), info['heuristic_solution'] comes with every step.
#include "ge_common.cuh"

using namespace ge;

extern "C" int ge_set_error(int code, const char *fmt, ...);

namespace {

constexpr int PPD_MAXP = 5;

__device__ __forceinline__ void ppd_store_mask(const ge_batch &d, int b, int lane, const uint32_t *adj, int head, bool waiting) {
    uint32_t *mb = d.mask_bits + (size_t)b * d.AW;
    for (int w = lane; w < d.AW; w += 32) {                                    // :175-183 neighbours of the head (+ the head itself
        uint32_t m = adj[(size_t)head * d.NW + w] & tail_mask(d.N, w);        //  when a product waits there: "pick up")
        if (waiting && w == (head >> 5)) m |= 1u << (head & 31);
        mb[w] = m;
    }
    if (d.mask_bytes) {
        __syncwarp();
        __threadfence_block();
        uint4 *out = reinterpret_cast<uint4 *>(d.mask_bytes + (size_t)b * d.AP);
        for (int c = lane; c < (d.AP >> 4); c += 32) {
            const uint32_t word = (c >> 1) < d.AW ? mb[c >> 1] : 0u;
            const uint32_t bits = (word >> ((c & 1) * 16)) & 0xffffu;
            out[c] = make_uint4(expand4(bits), expand4(bits >> 4), expand4(bits >> 8), expand4(bits >> 12));
        }
    }
}

__device__ __forceinline__ bool ppd_waiting_at(const ge_batch &d, int b, int status, int node) {
    const int P = d.n_dests;
    const int32_t *tg = d.targets + (size_t)b * d.n_targets;
    bool w = false;
    for (int i = 0; i < P; ++i) w |= ((status >> (2 * i)) & 3) == 0 && tg[i] == node;
    return w;
}

template <bool SAMPLED>
__global__ void __launch_bounds__(GE_WPB * 32) ppd_step_kernel(ge_batch d, int32_t *__restrict__ actions, ge_step_out out, uint64_t seed, uint32_t t) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * GE_WPB + warp;
    pdl_launch_dependents();   // programmatic dependent launch (ge_common.cuh): no-ops on a plain launch
    pdl_wait();
    if (b >= d.B) return;
    const int N = d.N, P = d.n_dests;
    const uint32_t *adj = d.adj_bits + (size_t)b * d.ADJS;
    const int32_t *tg = d.targets + (size_t)b * d.n_targets;
    const uint32_t nsteps = d.env_steps ? d.env_steps[b] : 0u;
    int4 c = *reinterpret_cast<const int4 *>(d.counters + (size_t)b * 4);
    int head = d.head[b];
    double cost = d.cost[b];
    int a;
    if (SAMPLED) {
        a = warp_sample(d.mask_bits + (size_t)b * d.AW, d.AW, lane, seed, (uint32_t)(d.env_id0 + b), t + nsteps);
        if (lane == 0) actions[b] = a;
    } else {
        a = actions[b];
    }
    double reward = 0.0, sol = __longlong_as_double(0x7ff8000000000000ll);
    int done = 0, solved = -1, has_mask = 1, status = GE_STEP_OK;
    bool write_state = false;
    const bool ok = a >= 0 && a < N && ((d.mask_bits[(size_t)b * d.AW + (a >> 5)] >> (a & 31)) & 1u);
    __syncwarp();
    if (d.done[b]) {
        has_mask = 0; status = GE_STEP_AFTER_DONE;
    } else if (!ok) {
        status = GE_STEP_INVALID; has_mask = 0;
    } else {
        write_state = true;
        sol = cost;                                                           // :211 the value before this move
        if (a == head) {                                                      // :214-221 pick up the product waiting here
            for (int i = 0; i < P; ++i)
                if (((c.x >> (2 * i)) & 3) == 0 && tg[i] == head) { c.x |= 1 << (2 * i); break; }
            reward = 2.0;
            c.y += 1;
        } else {                                                              // :223-249 move
            const int e = find_edge(d.row_ptr + (size_t)b * d.RP, d.col + (size_t)b * d.MP, head, a, lane);
            const double w = e >= 0 ? d.w64[(size_t)b * d.MP + e] : 0.0;
            reward = -w;
            cost = cost - reward;
            c.y += 1;
            head = a;
            const float tl = d.max_dist32[b];
            for (int i = 0; i < P; ++i) {
                if (((c.x >> (2 * i)) & 3) != 1) continue;                    // only products in transit
                // TIME_LEFT[i] -= adj[a, a] (= 0); the column's sum (N copies of the delivery time) below zero ends the episode
                if ((float)N * tl < 0.f - 1e-6f) {                            // :236-241 early return without info['mask']
                    done = 1; reward = -2.0 * N * P; solved = 0; has_mask = 0;
                    break;
                }
                if (tg[P + i] == head) { reward += 2.0; c.x = (c.x & ~(3 << (2 * i))) | (2 << (2 * i)); }   // :243-249 delivered
            }
        }
        if (has_mask) {
            bool all = true;
            for (int i = 0; i < P; ++i) all &= ((c.x >> (2 * i)) & 3) == 2;
            if (all) { done = 1; solved = 1; reward += 2.0 * N; }                                             // :252-255
            else if (c.y >= N * P * 50) { done = 1; solved = 0; reward = -2.0 * N * P; }                      // :256-259
        }
    }
    if (lane == 0) {
        out.reward[b] = (float)reward;
        ge_step_flags f;
        f.done = (uint8_t)done; f.solved = (int8_t)solved; f.status = (uint8_t)status; f.has_mask = (uint8_t)has_mask;
        out.flags[b] = f;
        out.solution_cost[b] = sol;
        if (d.traj) {
            const u64 cs = d.traj[b];
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
    if (!write_state) return;
    const bool auto_reset = done && (d.flags & GE_FLAG_AUTO_RESET);
    if (auto_reset) { head = 0; cost = 0.0; c = make_int4(0, 0, 0, 0); }
    if (has_mask || auto_reset) ppd_store_mask(d, b, lane, adj, head, ppd_waiting_at(d, b, c.x, head));
    if (lane == 0) {
        d.head[b] = head;
        d.cost[b] = cost;
        *reinterpret_cast<int4 *>(d.counters + (size_t)b * 4) = c;
        if (done && !auto_reset) d.done[b] = 1;
    }
}

// N <= 64: one LANE per env (like ge_lane.cu): the mask is one 64-bit register, the edge weight one load from the dense
// wmat, the next mask one adjacency row.  A warp per env spent a whole warp on a 50-node graph (75 us per 65,536-env step).
template <bool SAMPLED>
__global__ void __launch_bounds__(128) ppd_lane_step_kernel(ge_batch d, int32_t *__restrict__ actions, ge_step_out out, uint64_t seed, uint32_t t) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    pdl_launch_dependents();   // programmatic dependent launch (ge_common.cuh): no-ops on a plain launch
    pdl_wait();
    if (b >= d.B) return;
    const int N = d.N, P = d.n_dests, NW = d.NW;
    const int32_t *tg = d.targets + (size_t)b * d.n_targets;
    const uint32_t nsteps = d.env_steps ? d.env_steps[b] : 0u;
    int4 c = *reinterpret_cast<const int4 *>(d.counters + (size_t)b * 4);
    int head = d.head[b];
    double cost = d.cost[b];
    const bool was_done = d.done[b] != 0;
    u64 oldm = NW == 1 ? (u64)d.mask_bits[b] : ((u64)d.mask_bits[2 * (size_t)b] | ((u64)d.mask_bits[2 * (size_t)b + 1] << 32));
    int pk[PPD_MAXP], dr[PPD_MAXP];
#pragma unroll
    for (int i = 0; i < PPD_MAXP; ++i) { pk[i] = i < P ? tg[i] : -1; dr[i] = i < P ? tg[P + i] : -1; }
    int a;
    if (SAMPLED) {
        const int total = __popcll(oldm);
        a = -1;
        if (total > 0) {
            const uint32_t r = (uint32_t)(((uint64_t)mix32(seed, (uint32_t)(d.env_id0 + b), t + nsteps) * (uint64_t)total) >> 32);
            const uint32_t lo = (uint32_t)oldm, hi = (uint32_t)(oldm >> 32);
            const int clo = __popc(lo);
            a = (int)r < clo ? nth_set_bit(lo, (int)r) : 32 + nth_set_bit(hi, (int)r - clo);
        }
        actions[b] = a;
    } else {
        a = actions[b];
    }
    double reward = 0.0, sol = __longlong_as_double(0x7ff8000000000000ll);
    int done = 0, solved = -1, has_mask = 1, status = GE_STEP_OK;
    bool write_state = false;
    if (was_done) {
        has_mask = 0; status = GE_STEP_AFTER_DONE;
    } else if (!(a >= 0 && a < N && ((oldm >> a) & 1ull))) {
        status = GE_STEP_INVALID; has_mask = 0;
    } else {
        write_state = true;
        sol = cost;
        if (a == head) {
#pragma unroll
            for (int i = 0; i < PPD_MAXP; ++i)
                if (i < P && ((c.x >> (2 * i)) & 3) == 0 && pk[i] == head) { c.x |= 1 << (2 * i); break; }
            reward = 2.0;
            c.y += 1;
        } else {
            const double w = __ldg(d.wmat + ((size_t)b * N + head) * N + a);
            reward = -w;
            cost = cost - reward;
            c.y += 1;
            head = a;
            const float tl = d.max_dist32[b];
#pragma unroll
            for (int i = 0; i < PPD_MAXP; ++i) {
                if (i >= P || ((c.x >> (2 * i)) & 3) != 1) continue;
                if ((float)N * tl < 0.f - 1e-6f) { done = 1; reward = -2.0 * N * P; solved = 0; has_mask = 0; break; }
                if (dr[i] == head) { reward += 2.0; c.x = (c.x & ~(3 << (2 * i))) | (2 << (2 * i)); }
            }
        }
        if (has_mask) {
            bool all = true;
#pragma unroll
            for (int i = 0; i < PPD_MAXP; ++i) all &= i >= P || ((c.x >> (2 * i)) & 3) == 2;
            if (all) { done = 1; solved = 1; reward += 2.0 * N; }
            else if (c.y >= N * P * 50) { done = 1; solved = 0; reward = -2.0 * N * P; }
        }
    }
    out.reward[b] = (float)reward;
    ge_step_flags f;
    f.done = (uint8_t)done; f.solved = (int8_t)solved; f.status = (uint8_t)status; f.has_mask = (uint8_t)has_mask;
    out.flags[b] = f;
    out.solution_cost[b] = sol;
    if (d.traj) {
        const u64 cs = d.traj[b];
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
    if (!write_state) return;
    const bool auto_reset = done && (d.flags & GE_FLAG_AUTO_RESET);
    if (auto_reset) { head = 0; cost = 0.0; c = make_int4(0, 0, 0, 0); }
    if (has_mask || auto_reset) {
        const uint32_t *row = d.adj_bits + (size_t)b * d.ADJS + (size_t)head * NW;
        u64 m = NW == 1 ? (u64)row[0] : ((u64)row[0] | ((u64)row[1] << 32));
        bool waiting = false;
#pragma unroll
        for (int i = 0; i < PPD_MAXP; ++i) waiting |= i < P && ((c.x >> (2 * i)) & 3) == 0 && pk[i] == head;
        if (waiting) m |= 1ull << head;
        if (NW == 1) d.mask_bits[b] = (uint32_t)m;
        else { d.mask_bits[2 * (size_t)b] = (uint32_t)m; d.mask_bits[2 * (size_t)b + 1] = (uint32_t)(m >> 32); }
        if (d.mask_bytes) {
            uint4 *mb = reinterpret_cast<uint4 *>(d.mask_bytes + (size_t)b * d.AP);
            for (int k = 0; k < (d.AP >> 4); ++k) {
                const uint32_t bits = (uint32_t)(m >> (16 * k)) & 0xffffu;
                mb[k] = make_uint4(expand4(bits), expand4(bits >> 4), expand4(bits >> 8), expand4(bits >> 12));
            }
        }
    }
    d.head[b] = head;
    d.cost[b] = cost;
    *reinterpret_cast<int4 *>(d.counters + (size_t)b * 4) = c;
    if (done && !auto_reset) d.done[b] = 1;
}

__global__ void __launch_bounds__(GE_WPB * 32) ppd_reset_kernel(ge_batch d, const uint8_t *__restrict__ select) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * GE_WPB + warp;
    if (b >= d.B) return;
    if (select && !select[b]) return;
    ppd_store_mask(d, b, lane, d.adj_bits + (size_t)b * d.ADJS, 0, ppd_waiting_at(d, b, 0, 0));
    if (lane == 0) {
        d.head[b] = 0;                                                        // :133 head = 0
        d.cost[b] = 0.0;
        d.done[b] = 0;
        *reinterpret_cast<int4 *>(d.counters + (size_t)b * 4) = make_int4(0, 0, 0, 0);
    }
}

}  // namespace

static int ppd_launched(const char *what) {
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? GE_OK : ge_set_error(GE_ERR_CUDA, "%s launch: %s", what, cudaGetErrorString(e));
}

int ge_ppd_check(const ge_batch *d) {
    if (d->n_dests < 1 || d->n_dests > PPD_MAXP || d->n_targets != 2 * d->n_dests) return ge_set_error(GE_ERR_ARG, "PerishableProductDelivery: n_dests = n_products in 1..5, n_targets = 2 * n_products");
    if (!d->targets || !d->max_dist32 || !d->adj_bits || !d->w64) return ge_set_error(GE_ERR_ARG, "PerishableProductDelivery needs targets, max_dist32, adj_bits, w64");
    return GE_OK;
}

bool ge_ppd_lane(const ge_batch *d) { return d->N <= 64 && d->wmat != nullptr && !(d->flags & GE_FLAG_FORCE_WARP); }

int ge_ppd_step(const ge_batch *d, int32_t *actions, const ge_step_out *out, bool sampled, uint64_t seed, uint32_t t, cudaStream_t st) {
    int rc = ge_ppd_check(d);
    if (rc) return rc;
    if (ge_ppd_lane(d)) {
        const int T = 128, blocks = (d->B + T - 1) / T;
        ge_launch_step(sampled ? ppd_lane_step_kernel<true> : ppd_lane_step_kernel<false>, dim3(blocks), dim3(T), 0, st, *d, actions, *out, seed, t);
        return ppd_launched("ppd_lane_step_kernel");
    }
    const int blocks = (d->B + GE_WPB - 1) / GE_WPB;
    ge_launch_step(sampled ? ppd_step_kernel<true> : ppd_step_kernel<false>, dim3(blocks), dim3(GE_WPB * 32), 0, st, *d, actions, *out, seed, t);
    return ppd_launched("ppd_step_kernel");
}

int ge_ppd_reset(const ge_batch *d, const uint8_t *select, cudaStream_t st) {
    int rc = ge_ppd_check(d);
    if (rc) return rc;
    ppd_reset_kernel<<<(d->B + GE_WPB - 1) / GE_WPB, GE_WPB * 32, 0, st>>>(*d, select);
    return ppd_launched("ppd_reset_kernel");
}
