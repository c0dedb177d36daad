// ge_dc.cu -- dedicated DistributionCenter kernels (distribution_center.py:25-26,129-174), N <= 1024, exact distance
// automaton available (ge_batch.dfa / wcode).
//
// Why: DistributionCenter bounds BASELINE config 5 (0.116 G env-steps/s, 6x slower than any other env).  ncu on the
// general warp-per-env kernel (profiles/r01_final_step_kernel_cfg5_distcenter.md): 4,190 warp-instructions per
// env-step at 58 % issue utilisation -- issue-bound, not memory-bound -- of which the cutoff search's row-set
// expansion (inclusive scan + 5-step shuffle binary search per 32-edge slot group), generic shared-memory set
// handling and dispatch are the bulk.  Same rules here, restructured:
//   * node sets (taken, covered, targets, mask) live in REGISTERS, lane w owns word w; set algebra is one instruction,
//     membership of an arbitrary node is one shuffle;
//   * the cutoff search (find_nodes_in_range = nx single_source_dijkstra_path_length(cutoff), label-correcting on the
//     exact automaton, see ge_common.cuh:sssp_cutoff_dfa) walks the frontier LIST with a group of 8 lanes per row, four
//     rows per trip, over WEIGHT-SORTED rows of which only the prefix that can stay within the cutoff is visited: no
//     scan, no owner search; the next rows' first pass is loaded one trip ahead; the automaton's tables sit in shared
//     memory (one copy per block);
//   * distances are automaton state ids in a per-warp shared array (native 32-bit atomicMin);
//   * the mask is the OR of the in-range rows of the still uncovered targets, rows fetched 32/L at a time by groups
//     of L >= NW lanes, four passes in flight.
// Bit-identical to the general family (tests run both and the oracle).
#include "ge_common.cuh"

using namespace ge;

extern "C" int ge_set_error(int code, const char *fmt, ...);
int ge_grant_smem(const void *kernel, size_t smem);  // ge_api.cu

namespace {

__host__ __device__ inline int dc_dfa_words(const ge_batch &d, int S, int W) { return ((2 + S * W + 2 * S + 15) & ~15) >> 2; }
__host__ __device__ inline int dc_warp_words(const ge_batch &d) { return ((d.N + d.N + 2 * d.NW + 4) + 3) & ~3; }  // q[N] | two u16 lists | reach, queued | counter

struct DcScr {
    uint32_t *q;        // [N] automaton state of every node, 255 = unreached
    uint16_t *cur, *nxt;
    uint32_t *reach, *queued;
    int *cnt;
};

__device__ __forceinline__ DcScr dc_carve(uint32_t *base, const ge_batch &d) {
    DcScr s;
    s.q = base;
    s.cur = reinterpret_cast<uint16_t *>(base + d.N);
    s.nxt = s.cur + d.N;
    s.reach = base + 2 * d.N;
    s.queued = s.reach + d.NW;
    s.cnt = reinterpret_cast<int *>(s.queued + d.NW);
    return s;
}

// find_nodes_in_range(a): returns the reached set in registers, lane w = word w.
//
// A node at automaton state du can only relax edges whose weight keeps the sum within the cutoff, and those form a PREFIX
// of its WEIGHT-sorted row (code ascending; cmax[du] = the largest such code; fl(dist + w) is monotone in w): with cutoff
// 1.0 and weights 0.3..0.9 a node at distance 0.6 uses 2/7 of its edges.  Skipping the rest is exact -- they would have
// been looked up as "beyond the cutoff" and dropped.  Eight lanes per row, four rows per trip; a row continues with
// another pass of eight while its last lane was still inside the prefix.  (The first version walked whole rows, 16 lanes
// per row: 430 edge visits per step where ~175 can matter; profiles/r02_dc_step_kernel_v1.md.)
//
// The rows are read from ge_batch.dc_rows: the first DC_ROW entries of every weight-sorted row (entry = col | code << 16)
// at a fixed stride (128 bytes, 0xffffffff-padded, code 0xffff is beyond every prefix).  No row_ptr lookup -- the row
// address follows from the node id, one dependent memory round less per level -- sector-aligned rows, and the row's first
// sector is prefetched into L2 when its node is queued.  The first pass of the NEXT four rows is loaded while the current
// four are relaxed.  A prefix longer than DC_ROW entries (a node of degree > 32 whose whole row is within the cutoff)
// continues in ge_batch.dc_edges, where the same rows sit at their CSR offsets (rp).
#define DC_ROW 32
__device__ __forceinline__ uint32_t dc_cutoff_search_rows(const ge_batch &d, const int32_t *__restrict__ rp, const uint32_t *__restrict__ edges,
                                                      const uint32_t *__restrict__ rows, const uint8_t *tab, const uint8_t *expand,
                                                      const uint8_t *cmax, int W, DcScr &s, int lane, int source) {
    const int N = d.N, NW = d.NW;
    {   // q[v] = 255
        uint4 *q4 = reinterpret_cast<uint4 *>(s.q);
        const uint4 f = make_uint4(255u, 255u, 255u, 255u);
        for (int i = lane; i < (N + 3) >> 2; i += 32) q4[i] = f;      // the slice is padded to whole quads
        if (lane < NW) { s.reach[lane] = 0; s.queued[lane] = 0; }
    }
    __syncwarp();
    if (lane == 0) { s.q[source] = 0u; s.reach[source >> 5] = 1u << (source & 31); s.cur[0] = (uint16_t)source; *s.cnt = 0; }
    __syncwarp();
    int ncur = expand[0] ? 1 : 0;
    const int grp = lane >> 3, gl = lane & 7;
    uint16_t *cur = s.cur, *nxt = s.nxt;
    // one edge entry against the automaton: returns whether it was inside the prefix of its row
    auto relax = [&](uint32_t pk, uint32_t cm, const uint8_t *trow) -> bool {
        const uint32_t code = pk >> 16;
        const bool act = code <= cm;                                             // padding has code 0xffff; cm = 0xfffe0000 >> 16 never
        if (act) {
            const int v = (int)(pk & 0xffffu);
            const uint32_t nid = trow[code];                                     // state of fl(dist + w); inside the prefix => never 255
            if (nid < s.q[v]) {
                const uint32_t old = atomicMin(&s.q[v], nid);
                if (nid < old) {
                    const uint32_t bit = 1u << (v & 31);
                    if (expand[nid] && !(atomicOr(&s.queued[v >> 5], bit) & bit)) {
                        nxt[atomicAdd(s.cnt, 1)] = (uint16_t)v;
                        asm volatile("prefetch.global.L2 [%0];" ::"l"(rows + (size_t)v * DC_ROW));   // next round's row
                    }
                }
            }
        }
        return act;
    };
    while (ncur > 0) {
        int u = grp < ncur ? (int)cur[grp] : -1;
        uint32_t pk = u >= 0 ? rows[(size_t)u * DC_ROW + gl] : 0xffffffffu;      // first pass of the first four rows
        for (int i0 = 0; i0 < ncur; i0 += 4) {
            const int u_n = i0 + 4 + grp < ncur ? (int)cur[i0 + 4 + grp] : -1;   // next four rows: first pass in flight now
            const uint32_t pk_n = u_n >= 0 ? rows[(size_t)u_n * DC_ROW + gl] : 0xffffffffu;
            const int du = u >= 0 ? (int)s.q[u] : 0;
            const uint8_t *trow = tab + du * W;
            uint32_t cm = u >= 0 ? (uint32_t)cmax[du] : 255u;
            if (cm == 255u) { cm = 0u; pk = 0xffffffffu; }                       // 255 = nothing within the cutoff: an all-padding row
            const uint32_t *row = rows + (size_t)(u >= 0 ? u : 0) * DC_ROW + gl;
            unsigned cont = 0;
#pragma unroll
            for (int pass = 0; pass < DC_ROW / 8; ++pass) {
                const bool act = relax(pk, cm, trow);
                cont = __ballot_sync(GE_FULL, act && gl == 7);                   // bit 8g + 7: row g filled its whole pass => it continues
                if (!cont) break;                                                // every prefix is exhausted
                pk = 0xffffffffu;
                if (pass + 1 < DC_ROW / 8 && ((cont >> ((lane & ~7) | 7)) & 1u)) pk = row[8 * (pass + 1)];
            }
            if (cont) {   // rare: a prefix longer than DC_ROW entries continues in the CSR copy
                for (int k = DC_ROW + gl;; k += 8) {
                    pk = 0xffffffffu;
                    if ((cont >> ((lane & ~7) | 7)) & 1u) { const int e = rp[u] + k; if (e < rp[u + 1]) pk = edges[e]; }
                    const bool act = relax(pk, cm, trow);
                    cont = __ballot_sync(GE_FULL, act && gl == 7);
                    if (!cont) break;
                }
            }
            u = u_n; pk = pk_n;
        }
        __syncwarp();
        ncur = *s.cnt;
        __syncwarp();
        if (lane == 0) *s.cnt = 0;
        if (lane < NW) s.queued[lane] = 0;
        uint16_t *tmp = cur; cur = nxt; nxt = tmp;
        __syncwarp();
    }
    // reached = every node that got a state (q != 255): one ballot per word instead of
    // an atomic per first visit.  Returned in registers, lane w = word w.
    uint32_t mine = 0;
    for (int w = 0; w < NW; ++w) {
        const int v = (w << 5) + lane;
        const unsigned bits = __ballot_sync(GE_FULL, v < N && s.q[v] != 255u);
        if (lane == w) mine = bits;
    }
    return mine;
}

// OR of the in-range rows of the targets that are not covered yet (distribution_center.py:129-141, parenting 2).
// covw = the lane's word of the covered set.  Returns the lane's word of the union (lanes >= NW: 0).
__device__ __forceinline__ uint32_t dc_union_in_range(const ge_batch &d, int b, int lane, uint32_t covw, uint16_t *live /* >= n_targets */) {
    const int NW = d.NW, NT = d.n_targets;
    const int32_t *tg = d.targets + (size_t)b * NT;
    const uint32_t *ir = d.in_range + (size_t)b * NT * NW;
    int nlive = 0;
    for (int t0 = 0; t0 < NT; t0 += 32) {
        const int t = t0 + lane;
        bool unc = false;
        int node = 0;
        if (t < NT) node = tg[t];
        const uint32_t cw = __shfl_sync(GE_FULL, covw, (node >> 5) & 31);
        if (t < NT) unc = !((cw >> (node & 31)) & 1u);
        const unsigned bal = __ballot_sync(GE_FULL, unc);
        if (unc) live[nlive + __popc(bal & ((1u << lane) - 1u))] = (uint16_t)t;
        nlive += __popc(bal);
    }
    __syncwarp();
    const int L = NW <= 1 ? 1 : NW <= 2 ? 2 : NW <= 4 ? 4 : NW <= 8 ? 8 : NW <= 16 ? 16 : 32;
    const int rpp = 32 / L, grp = lane / L, wl = lane % L;
    uint32_t acc = 0;
    const bool W = wl < NW;
    for (int i0 = 0; i0 < nlive; i0 += 4 * rpp) {
        uint32_t r[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int idx = i0 + j * rpp + grp;
            r[j] = (W && idx < nlive) ? __ldg(ir + (size_t)live[idx] * NW + wl) : 0u;
        }
        acc |= (r[0] | r[1]) | (r[2] | r[3]);
    }
    for (int o = L; o < 32; o <<= 1) acc |= __shfl_xor_sync(GE_FULL, acc, o);
    __syncwarp();
    return (lane < NW) ? acc : 0u;
}

__device__ __forceinline__ void dc_store_mask(const ge_batch &d, int b, int lane, uint32_t m) {
    if (lane >= d.AW) return;
    d.mask_bits[(size_t)b * d.AW + lane] = m;
    if (d.mask_bytes) {  // the lane's 32 mask entries = two 128-bit stores
        uint4 *mb = reinterpret_cast<uint4 *>(d.mask_bytes + (size_t)b * d.AP);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int c = 2 * lane + h;
            if (c < (d.AP >> 4)) {
                const uint32_t bits = (m >> (16 * h)) & 0xffffu;
                mb[c] = make_uint4(expand4(bits), expand4(bits >> 4), expand4(bits >> 8), expand4(bits >> 12));
            }
        }
    }
}

// mask right after reset(): nothing taken, nothing covered
__device__ __forceinline__ uint32_t dc_reset_mask(const ge_batch &d, int b, int lane, uint32_t tail, uint16_t *live) {
    if (d.parenting != 2) return tail;
    return dc_union_in_range(d, b, lane, 0u, live) & tail;
}

template <bool SAMPLED>
__global__ void __launch_bounds__(GE_WPB * 32, 6) dc_step_kernel(ge_batch d, int32_t *__restrict__ actions, ge_step_out out, uint64_t seed,
                                                                uint32_t t, int dfa_words, int warp_words) {
    extern __shared__ __align__(16) uint32_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * GE_WPB + warp;
    pdl_launch_dependents();   // programmatic dependent launch (ge_common.cuh): the automaton (static) is staged before pdl_wait()
    const int S = d.dfa[0], W = d.dfa[1];
    {   // automaton tables: one copy per block
        uint8_t *dst = reinterpret_cast<uint8_t *>(smem);
        const int nbytes = 2 + S * W + 2 * S;
        for (int i = threadIdx.x; i < nbytes; i += blockDim.x) dst[i] = d.dfa[i];
    }
    __syncthreads();
    pdl_wait();
    if (b >= d.B) return;
    const uint8_t *tab = reinterpret_cast<const uint8_t *>(smem) + 2, *expand = tab + S * W, *cmax = expand + S;
    DcScr s = dc_carve(smem + dfa_words + (size_t)warp * warp_words, d);
    const int N = d.N, NW = d.NW;
    const bool WL = lane < NW;
    const uint32_t tail = WL ? tail_mask(N, lane) : 0u;
    // ---- state: one word of every set per lane
    uint32_t takenw = WL ? d.node_bits[(size_t)b * NW + lane] : 0u;
    uint32_t covw = WL ? d.node_bits2[(size_t)b * NW + lane] : 0u;
    const uint32_t tgtw = WL ? d.target_bits[(size_t)b * NW + lane] : 0u;
    const uint32_t oldm = WL ? d.mask_bits[(size_t)b * d.AW + lane] : 0u;
    const uint32_t m0 = (WL && d.mask0_bits) ? d.mask0_bits[(size_t)b * d.AW + lane] : 0u;
    double cost = d.cost[b];
    const bool was_done = d.done[b] != 0;
    const uint32_t nsteps = d.env_steps ? d.env_steps[b] : 0u;
    int a;
    if (SAMPLED) {  // r-th set bit of the mask, same draw as ge_common.cuh:warp_sample
        const int pc = __popc(oldm);
        int inc = pc;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int x = __shfl_up_sync(GE_FULL, inc, o);
            if (lane >= o) inc += x;
        }
        const int total = __shfl_sync(GE_FULL, inc, 31);
        a = -1;
        if (total > 0) {
            const uint32_t r = (uint32_t)(((uint64_t)mix32(seed, (uint32_t)(d.env_id0 + b), t + nsteps) * (uint64_t)total) >> 32);
            const unsigned hit = __ballot_sync(GE_FULL, (int)r < inc);
            const int sl = __ffs(hit) - 1;
            const int pos = (lane == sl) ? nth_set_bit(oldm, (int)r - (inc - pc)) : 0;
            a = (sl << 5) + __shfl_sync(GE_FULL, pos, sl);
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
    const uint32_t oldm_a = __shfl_sync(GE_FULL, oldm, a_ok ? (a >> 5) : 0);
    if (was_done) {
        has_mask = 0; status = GE_STEP_AFTER_DONE;
    } else if (!(a_ok && ((oldm_a >> (a & 31)) & 1u))) {
        status = GE_STEP_INVALID; has_mask = 0;
    } else {                                                                     // distribution_center.py:144-174
        write_state = true;
        const float w = d.node_cost[(size_t)b * N + a];
        cost = (double)__fadd_rn((float)cost, w);
        float rew = -w;
        if (lane == (a >> 5)) takenw |= 1u << (a & 31);
        const uint32_t reachw =                                                   // find_nodes_in_range (:25-26,155)
            dc_cutoff_search_rows(d, d.row_ptr + (size_t)b * d.RP, d.dc_edges + (size_t)b * d.MP, d.dc_rows + (size_t)b * N * DC_ROW, tab, expand, cmax, W, s, lane, a);
        const int gained = __reduce_add_sync(GE_FULL, __popc(reachw & ~covw & tgtw));
        covw |= reachw;
        rew += (float)gained;
        reward = (double)rew;
        __syncwarp();
        if (d.parenting == 2)
            maskw = dc_union_in_range(d, b, lane, covw, s.cur /* free again */) & ~takenw & tail;
        else maskw = ~takenw & tail;
        if (!__any_sync(GE_FULL, (tgtw & ~covw) != 0u)) { done = 1; solved = 1; sol = cost; }
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
    const bool auto_reset = done && (d.flags & GE_FLAG_AUTO_RESET);
    if (auto_reset) {                                                            // tail of reset()
        takenw = 0; covw = 0; cost = 0.0;
        maskw = d.mask0_bits ? m0 : dc_reset_mask(d, b, lane, tail, s.cur);
    }
    if (auto_reset || write_state) {
        if (WL) {
            d.node_bits[(size_t)b * NW + lane] = takenw;
            d.node_bits2[(size_t)b * NW + lane] = covw;
        }
        dc_store_mask(d, b, lane, maskw);
        if (lane == 0) {
            d.cost[b] = cost;
            if (done && !auto_reset) d.done[b] = 1;
        }
    }
    if (d.progress) {   // streamed host step: the whole warp's stores of this env are ordered before one release by lane 0
        __syncwarp();
        if (lane == 0) { __threadfence(); atomicAdd(d.progress + (b >> GE_PROGRESS_SHIFT), 1u); }
    }
}

__global__ void __launch_bounds__(GE_WPB * 32) dc_reset_kernel(ge_batch d, const uint8_t *__restrict__ select) {
    __shared__ uint16_t live_all[GE_WPB][1024];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * GE_WPB + warp;
    if (b >= d.B) return;
    if (select && !select[b]) return;
    const int N = d.N, NW = d.NW;
    const bool WL = lane < NW;
    const uint32_t tail = WL ? tail_mask(N, lane) : 0u;
    const uint32_t m = dc_reset_mask(d, b, lane, tail, live_all[warp]);
    if (WL) {
        d.node_bits[(size_t)b * NW + lane] = 0;
        d.node_bits2[(size_t)b * NW + lane] = 0;
        if (d.mask0_bits) d.mask0_bits[(size_t)b * d.AW + lane] = m;
    }
    dc_store_mask(d, b, lane, m);
    if (lane == 0) {
        d.head[b] = 0;
        d.cost[b] = 0.0;
        d.done[b] = 0;
        *reinterpret_cast<int4 *>(d.counters + (size_t)b * 4) = make_int4(0, 0, 0, 0);
    }
}

// dc_edges: every CSR row re-ordered by weight code (stable), entry = col | code << 16.  One lane per row (rows are short;
// reset-time code): count per code, then place.
__global__ void __launch_bounds__(256) dc_edges_kernel(ge_batch d) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)d.B * d.N) return;
    const int b = (int)(i / d.N), u = (int)(i % d.N);
    const int32_t *rp = d.row_ptr + (size_t)b * d.RP;
    const int32_t *col = d.col + (size_t)b * d.MP;
    const uint8_t *wc = d.wcode + (size_t)b * d.MP;
    uint32_t *out = d.dc_edges + (size_t)b * d.MP;
    const int lo = rp[u], hi = rp[u + 1];
    int pos = lo;
    for (int c = 0; c < 16 && pos < hi; ++c)                       // at most 15 distinct weights (batch.py:_build_distance_automaton)
        for (int e = lo; e < hi; ++e)
            if (wc[e] == c) out[pos++] = (uint32_t)col[e] | ((uint32_t)c << 16);
    if (d.dc_rows) {                                               // the same row at a fixed stride, padded
        uint32_t *row = d.dc_rows + ((size_t)b * d.N + u) * 32;
        for (int k = 0; k < 32; ++k) row[k] = (lo + k < hi) ? out[lo + k] : 0xffffffffu;
    }
}

}  // namespace

int ge_dc_build_edges(const ge_batch *d, cudaStream_t st) {
    if (!d->dc_edges || !d->wcode) return GE_OK;
    const long long rows = (long long)d->B * d->N;
    dc_edges_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(*d);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? GE_OK : ge_set_error(GE_ERR_CUDA, "dc_edges_kernel launch: %s", cudaGetErrorString(e));
}

// ------------------------------------------------------------------ host launchers (called from ge_api.cu)
bool ge_dc_eligible(const ge_batch *d) {
    if (d->flags & GE_FLAG_FORCE_WARP) return false;
    if (d->kind != GE_DISTRIBUTION_CENTER || d->N > 1024 || !d->wcode || !d->dfa || !d->dc_edges || !d->dc_rows) return false;
    if (d->parenting == 2 && (!d->in_range || !d->targets || d->n_targets > 1024 || d->n_targets > d->N)) return false;
    return d->node_bits2 != nullptr && d->target_bits != nullptr;
}

static int dc_launched(const char *what) {
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? GE_OK : ge_set_error(GE_ERR_CUDA, "%s launch: %s", what, cudaGetErrorString(e));
}

int ge_dc_step(const ge_batch *d, int32_t *actions, const ge_step_out *out, bool sampled, uint64_t seed, uint32_t t, cudaStream_t st) {
    // automaton size in bytes (ge_batch.dfa_bytes); unknown => its largest possible table (254 states x 15 weights, 4 KB)
    const int dfa_words = d->dfa_bytes > 0 ? (((d->dfa_bytes + 15) & ~15) >> 2) : dc_dfa_words(*d, 254, 15);
    const int ww = dc_warp_words(*d);
    const size_t smem = ((size_t)dfa_words + (size_t)ww * GE_WPB) * 4;
    auto kernel = sampled ? dc_step_kernel<true> : dc_step_kernel<false>;
    int rc = ge_grant_smem((const void *)kernel, smem);
    if (rc) return rc;
    ge_launch_step(kernel, dim3((d->B + GE_WPB - 1) / GE_WPB), dim3(GE_WPB * 32), smem, st, *d, actions, *out, seed, t, dfa_words, ww);
    return dc_launched("dc_step_kernel");
}

int ge_dc_reset(const ge_batch *d, const uint8_t *select, cudaStream_t st) {
    dc_reset_kernel<<<(d->B + GE_WPB - 1) / GE_WPB, GE_WPB * 32, 0, st>>>(*d, select);
    return dc_launched("dc_reset_kernel");
}
