// ge_policy.cu -- masked categorical over policy logits (sm_100a): ge_sample_logits, ge_masked_log_prob and its backward, and the
// search kernels built on it (beam search, stochastic beam search, Monte Carlo tree search with PUCT and with Gumbel MuZero selection).
//
// One device routine, masked_row(), is the whole reduction: for one row of logits it walks the packed valid-action mask
// and reads ONLY the logits of set bits.  Lane l of the warp owns actions 32w + l; per nonzero mask word it loads its
// logit iff its bit is set, so the warp's loads are coalesced and a 32-byte sector without a valid action is never
// fetched (the frontier masks of Multicast / SteinerTree are sparse).  Mask words are read 32 at a time (one coalesced
// 128-byte load, then broadcast by shuffle) and zero words are skipped warp-uniformly; U nonzero words are loaded before
// any of them is accumulated, so their loads overlap.  Per lane it keeps online accumulators over the valid actions:
//   mx = max l,  se = sum exp(l - mx),  st = sum exp(l - mx) * (l - mx),  and the best (score, index, l),
// merged across the warp by a shuffle butterfly in a fixed order.  Then lse = mx + log(se) and H = log(se) - st / se
// (= lse - sum p l without the cancellation of two large terms).  Every kernel calls the same routine with the same
// arithmetic, so the sampler's log_prob / entropy equal the forward kernel's bit for bit; there are no atomics.
#include <cfloat>
#include <climits>
#include <cstdio>
#include <cuda_bf16.h>

#include "ge_common.cuh"

extern "C" int ge_set_error(int code, const char *fmt, ...);

using namespace ge;

namespace {

constexpr int POL_WPB = 8;  // warps (= rows) per block
constexpr int POL_U = 4;    // nonzero mask words whose logits are loaded together

enum { MODE_STATS = 0, MODE_GREEDY = 1, MODE_GUMBEL = 2, MODE_NODE_GUMBEL = 3 };

template <int DT>
__device__ __forceinline__ float load_logit(const void *row, size_t i) {
    if (DT == GE_LOGITS_BF16) {
        const unsigned short u = __ldg(reinterpret_cast<const unsigned short *>(row) + i);
        return __uint_as_float((uint32_t)u << 16);
    }
    return __ldg(reinterpret_cast<const float *>(row) + i);
}
template <int DT>
__device__ __forceinline__ void store_grad(void *row, size_t i, float g) {
    if (DT == GE_LOGITS_BF16) reinterpret_cast<__nv_bfloat16 *>(row)[i] = __float2bfloat16_rn(g);
    else reinterpret_cast<float *>(row)[i] = g;
}

// Gumbel noise of action a (include/graphenvs_b200.h, ge_sample_logits): key = per-row 64-bit key.
__device__ __forceinline__ float gumbel(uint64_t key, int a) {
    const uint32_t h = mix32(key, (uint32_t)a, 0x85EBCA6Bu);
    const float u = __fmul_rn((float)(h >> 8) + 0.5f, 5.9604644775390625e-8f);  // ((h >> 8) + 1/2) / 2^24, exact, in (0, 1)
    return -logf(-logf(u));
}
// The noise of ge_beam_expand_sampled: gumbel() with u kept below 1.  (h >> 8) + 0.5 rounds to even in float32 once h >> 8 >= 2^23,
// so h >> 8 = 2^24 - 1 gives u = 1 and g = +inf there; here u is clamped to 1 - 2^-24, and every key is finite.
__device__ __forceinline__ float node_gumbel(uint64_t key, int a) {
    const uint32_t h = mix32(key, (uint32_t)a, 0x85EBCA6Bu);
    const float u = fminf(__fmul_rn((float)(h >> 8) + 0.5f, 5.9604644775390625e-8f), 0.99999994f);
    return -logf(-logf(u));
}
__device__ __forceinline__ uint64_t row_key(uint64_t seed, uint32_t env, uint32_t t) {
    return ((uint64_t)mix32(seed, env, t) << 32) | (uint64_t)mix32(seed ^ 0xD1B54A32D192ED03ull, env, t);
}

struct RowStats {
    float mx, se, st;  // max valid logit, sum exp(l - mx), sum exp(l - mx) * (l - mx); se == 0 <=> no valid action
    float bs, bl;      // best score and its logit
    int bi;            // its action (INT_MAX = none)
};

__device__ __forceinline__ void acc_one(RowStats &r, float l) {
    if (l > r.mx) {
        if (r.se > 0.f) {
            const float dm = __fsub_rn(r.mx, l);  // < 0
            const float sc = expf(dm);
            r.st = __fmul_rn(sc, __fmaf_rn(dm, r.se, r.st));
            r.se = __fmaf_rn(r.se, sc, 1.f);
        } else {
            r.se = 1.f; r.st = 0.f;
        }
        r.mx = l;
    } else {
        const float dl = __fsub_rn(l, r.mx);
        const float e = expf(dl);
        r.se = __fadd_rn(r.se, e);
        r.st = __fmaf_rn(e, dl, r.st);
    }
}

__device__ __forceinline__ void merge(RowStats &r, const RowStats &o) {
    if (o.se > 0.f) {
        if (r.se > 0.f) {
            const float M = fmaxf(r.mx, o.mx);
            const float d1 = __fsub_rn(r.mx, M), d2 = __fsub_rn(o.mx, M);
            const float a1 = expf(d1), a2 = expf(d2);
            r.st = __fadd_rn(__fmul_rn(a1, __fmaf_rn(d1, r.se, r.st)), __fmul_rn(a2, __fmaf_rn(d2, o.se, o.st)));
            r.se = __fadd_rn(__fmul_rn(r.se, a1), __fmul_rn(o.se, a2));
            r.mx = M;
        } else {
            r.mx = o.mx; r.se = o.se; r.st = o.st;
        }
    }
    if (o.bs > r.bs || (o.bs == r.bs && o.bi < r.bi)) { r.bs = o.bs; r.bi = o.bi; r.bl = o.bl; }
}

// The shared reduction over one row (see the file comment).  Warp-cooperative; the result is warp-uniform.
template <int DT, int MODE>
__device__ __forceinline__ RowStats masked_row(const void *row, const uint32_t *__restrict__ mrow, int A, int AW, uint64_t key, int lane) {
    RowStats r;
    r.mx = -INFINITY; r.se = 0.f; r.st = 0.f; r.bs = -INFINITY; r.bl = 0.f; r.bi = INT_MAX;
    for (int w0 = 0; w0 < AW; w0 += 32) {
        const int wl = w0 + lane;
        const uint32_t mw = wl < AW ? (__ldg(mrow + wl) & tail_mask(A, wl)) : 0u;   // bits >= A are ignored
        unsigned nz = __ballot_sync(GE_FULL, mw != 0u);
        while (nz) {
            float v[POL_U];
            int idx[POL_U];
            bool has[POL_U];
#pragma unroll
            for (int k = 0; k < POL_U; ++k) {
                const int src = nz ? __ffs((int)nz) - 1 : 0;
                const bool any = nz != 0u;
                nz &= nz - 1u;
                const uint32_t word = __shfl_sync(GE_FULL, mw, src);
                idx[k] = ((w0 + src) << 5) + lane;
                has[k] = any && ((word >> lane) & 1u);
                v[k] = has[k] ? load_logit<DT>(row, (size_t)idx[k]) : 0.f;
            }
#pragma unroll
            for (int k = 0; k < POL_U; ++k) {
                if (!has[k]) continue;
                acc_one(r, v[k]);
                if (MODE != MODE_STATS) {
                    const float s = MODE == MODE_GUMBEL ? __fadd_rn(v[k], gumbel(key, idx[k]))
                                  : MODE == MODE_NODE_GUMBEL ? __fadd_rn(v[k], node_gumbel(key, idx[k])) : v[k];
                    if (s > r.bs) { r.bs = s; r.bi = idx[k]; r.bl = v[k]; }   // strictly greater: a lane visits its actions in order
                }
            }
        }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        RowStats q;
        q.mx = __shfl_xor_sync(GE_FULL, r.mx, o);
        q.se = __shfl_xor_sync(GE_FULL, r.se, o);
        q.st = __shfl_xor_sync(GE_FULL, r.st, o);
        q.bs = __shfl_xor_sync(GE_FULL, r.bs, o);
        q.bl = __shfl_xor_sync(GE_FULL, r.bl, o);
        q.bi = __shfl_xor_sync(GE_FULL, r.bi, o);
        if (lane & o) { RowStats t = q; merge(t, r); r = t; }   // lower lanes first: the same order on both sides
        else merge(r, q);
    }
    r.mx = __shfl_sync(GE_FULL, r.mx, 0);
    r.se = __shfl_sync(GE_FULL, r.se, 0);
    r.st = __shfl_sync(GE_FULL, r.st, 0);
    r.bl = __shfl_sync(GE_FULL, r.bl, 0);
    r.bi = __shfl_sync(GE_FULL, r.bi, 0);
    return r;
}

__device__ __forceinline__ float row_lse(const RowStats &r) { return r.se > 0.f ? __fadd_rn(r.mx, logf(r.se)) : -INFINITY; }
__device__ __forceinline__ float row_entropy(const RowStats &r) { return r.se > 0.f ? __fsub_rn(logf(r.se), __fdiv_rn(r.st, r.se)) : 0.f; }

template <int DT, int MODE>
__global__ void __launch_bounds__(POL_WPB * 32) policy_sample_kernel(ge_batch d, const void *__restrict__ logits, uint64_t seed, uint32_t t,
                                                                      int32_t *__restrict__ actions, float *__restrict__ log_prob,
                                                                      float *__restrict__ entropy) {
    pdl_launch_dependents();   // programmatic dependent launch (ge_common.cuh): nothing is touched before pdl_wait()
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * POL_WPB + (threadIdx.x >> 5);
    if (b >= d.B) return;
    const size_t esz = DT == GE_LOGITS_BF16 ? 2 : 4;
    const void *row = reinterpret_cast<const char *>(logits) + (size_t)b * d.A * esz;
    uint64_t key = 0;
    if (MODE == MODE_GUMBEL) key = row_key(seed, (uint32_t)(d.env_id0 + b), t + (d.env_steps ? d.env_steps[b] : 0u));
    const RowStats r = masked_row<DT, MODE>(row, d.mask_bits + (size_t)b * d.AW, d.A, d.AW, key, lane);
    if (lane == 0) {
        const bool any = r.se > 0.f;
        actions[b] = any ? r.bi : -1;
        if (log_prob) log_prob[b] = any ? __fsub_rn(r.bl, row_lse(r)) : 0.f;
        if (entropy) entropy[b] = row_entropy(r);
    }
}

__device__ __forceinline__ bool valid_action(const uint32_t *mrow, int A, int a) {
    return a >= 0 && a < A && ((__ldg(mrow + (a >> 5)) >> (a & 31)) & 1u);
}

template <int DT>
__global__ void __launch_bounds__(POL_WPB * 32) policy_logprob_kernel(const void *__restrict__ logits, int B, int A, const uint32_t *__restrict__ mask_bits,
                                                                       const int32_t *__restrict__ actions, float *__restrict__ log_prob,
                                                                       float *__restrict__ entropy, float *__restrict__ lse) {
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * POL_WPB + (threadIdx.x >> 5);
    if (b >= B) return;
    const int AW = (A + 31) >> 5;
    const size_t esz = DT == GE_LOGITS_BF16 ? 2 : 4;
    const void *row = reinterpret_cast<const char *>(logits) + (size_t)b * A * esz;
    const uint32_t *mrow = mask_bits + (size_t)b * AW;
    const RowStats r = masked_row<DT, MODE_STATS>(row, mrow, A, AW, 0, lane);
    if (lane == 0) {
        const int a = actions[b];
        const float L = row_lse(r);
        float lp = 0.f;
        if (r.se > 0.f) lp = valid_action(mrow, A, a) ? __fsub_rn(load_logit<DT>(row, (size_t)a), L) : -INFINITY;
        log_prob[b] = lp;
        entropy[b] = row_entropy(r);
        lse[b] = L;
    }
}

// grad_logits[b, i] = g_lp (1[i = a] - p_i) - g_H p_i (log p_i + H) for valid i, 0 elsewhere; p_i = exp(l_i - lse).
template <int DT>
__global__ void __launch_bounds__(POL_WPB * 32) policy_logprob_bwd_kernel(const void *__restrict__ logits, int B, int A, const uint32_t *__restrict__ mask_bits,
                                                                           const int32_t *__restrict__ actions, const float *__restrict__ lse,
                                                                           const float *__restrict__ entropy, const float *__restrict__ g_lp,
                                                                           const float *__restrict__ g_h, void *__restrict__ grad) {
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * POL_WPB + (threadIdx.x >> 5);
    if (b >= B) return;
    const int AW = (A + 31) >> 5;
    const size_t esz = DT == GE_LOGITS_BF16 ? 2 : 4;
    const void *row = reinterpret_cast<const char *>(logits) + (size_t)b * A * esz;
    void *grow = reinterpret_cast<char *>(grad) + (size_t)b * A * esz;
    const uint32_t *mrow = mask_bits + (size_t)b * AW;
    const int a0 = actions[b];
    const int a = valid_action(mrow, A, a0) ? a0 : -1;   // an invalid action contributes no log_prob gradient
    const float glp = (g_lp && a >= 0) ? g_lp[b] : 0.f;
    const float gh = g_h ? g_h[b] : 0.f;
    const float L = lse[b], H = entropy[b];
    for (int w0 = 0; w0 < AW; w0 += 32) {
        const int wl = w0 + lane;
        const uint32_t mw = wl < AW ? (__ldg(mrow + wl) & tail_mask(A, wl)) : 0u;
        const int nw = min(32, AW - w0);
#pragma unroll 4
        for (int k = 0; k < nw; ++k) {
            const uint32_t word = __shfl_sync(GE_FULL, mw, k);
            const int i = ((w0 + k) << 5) + lane;
            if (i >= A) continue;
            float g = 0.f;
            if ((word >> lane) & 1u) {
                const float lp = __fsub_rn(load_logit<DT>(row, (size_t)i), L);
                const float p = expf(lp);
                g = __fsub_rn(__fmul_rn(glp, __fsub_rn(i == a ? 1.f : 0.f, p)), __fmul_rn(__fmul_rn(gh, p), __fadd_rn(lp, H)));
            }
            store_grad<DT>(grow, (size_t)i, g);
        }
    }
}

// ---- beam search (ge_beam_expand): one CTA per group of W beams, one warp per beam (BEAM_WARPS warps take turns past 8) ----
constexpr int BEAM_MAXW = 32;
constexpr int BEAM_WARPS = 8;

// THE candidate order of ge_beam_expand: score descending, then parent slot ascending, then action ascending.  Stage 1 ranks one
// beam's candidates with it (equal parents), stage 2 merges the beams' lists with it; it is a total order, so every reduction
// below gives the same winner whatever order it visits the candidates in.
__device__ __forceinline__ bool beam_before(float s1, int p1, int a1, float s2, int p2, int a2) {
    return s1 > s2 || (s1 == s2 && (p1 < p2 || (p1 == p2 && a1 < a2)));
}

// Per-candidate scores of the two expand kernels: what beam_next ranks by.
struct LogProbScore {     // ge_beam_expand: the beam's score after action a, fl32(base + fl32(l_a - lse))
    float base, lse;
    __device__ __forceinline__ float operator()(float l, int) const { return __fadd_rn(base, __fsub_rn(l, lse)); }
};
struct PerturbedScore {   // ge_beam_expand_sampled: the Gumbel-max score keyed by the beam's node key, fl32(l_a + g_a)
    uint64_t key;
    __device__ __forceinline__ float operator()(float l, int a) const { return __fadd_rn(l, node_gumbel(key, a)); }
};

// The best candidate of one live beam that comes after (ps, pa) in the order (the best overall when `first`), over its valid
// actions, ranked by score(l_a, a).  Walks the row as masked_row does (zero words skipped warp-uniformly, only logits of set
// bits read); after the first walk the mask and the valid logits are L1-resident.  Warp-uniform result; ba = INT_MAX when no
// candidate is left.
template <int DT, class Score>
__device__ __forceinline__ void beam_next(const void *row, const uint32_t *__restrict__ mrow, int A, int AW, Score score,
                                          bool first, float ps, int pa, int lane, float &bs, int &ba) {
    float s_best = -INFINITY;
    int a_best = INT_MAX;
    for (int w0 = 0; w0 < AW; w0 += 32) {
        const int wl = w0 + lane;
        const uint32_t mw = wl < AW ? (__ldg(mrow + wl) & tail_mask(A, wl)) : 0u;
        unsigned nz = __ballot_sync(GE_FULL, mw != 0u);
        while (nz) {
            float v[POL_U];
            int idx[POL_U];
            bool has[POL_U];
#pragma unroll
            for (int k = 0; k < POL_U; ++k) {
                const int src = nz ? __ffs((int)nz) - 1 : 0;
                const bool any = nz != 0u;
                nz &= nz - 1u;
                const uint32_t word = __shfl_sync(GE_FULL, mw, src);
                idx[k] = ((w0 + src) << 5) + lane;
                has[k] = any && ((word >> lane) & 1u);
                v[k] = has[k] ? load_logit<DT>(row, (size_t)idx[k]) : 0.f;
            }
#pragma unroll
            for (int k = 0; k < POL_U; ++k) {
                if (!has[k]) continue;
                const float s = score(v[k], idx[k]);
                if ((first || beam_before(ps, 0, pa, s, 0, idx[k])) && beam_before(s, 0, idx[k], s_best, 0, a_best)) { s_best = s; a_best = idx[k]; }
            }
        }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const float s = __shfl_xor_sync(GE_FULL, s_best, o);
        const int a = __shfl_xor_sync(GE_FULL, a_best, o);
        if (beam_before(s, 0, a, s_best, 0, a_best)) { s_best = s; a_best = a; }
    }
    bs = s_best; ba = a_best;
}

template <int DT>
__global__ void __launch_bounds__(BEAM_WARPS * 32) beam_expand_kernel(ge_batch d, int W, const void *__restrict__ logits,
                                                                       const float *__restrict__ score, float *__restrict__ score_out,
                                                                       int32_t *__restrict__ parent, int32_t *__restrict__ action,
                                                                       int32_t *__restrict__ load_index) {
    __shared__ float l_s[BEAM_MAXW][BEAM_MAXW];   // per beam: its best min(W, candidates) candidates, in the order
    __shared__ int l_a[BEAM_MAXW][BEAM_MAXW];
    __shared__ int l_n[BEAM_MAXW];
    pdl_launch_dependents();   // as the sampler: nothing is touched before pdl_wait()
    pdl_wait();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int g0 = blockIdx.x * W;   // env index of the group's slot 0
    const size_t esz = DT == GE_LOGITS_BF16 ? 2 : 4;
    // Stage 1: every beam's own sorted candidate list
    for (int p = warp; p < W; p += nwarps) {
        const int b = g0 + p;
        const float base = score[b];
        int n = 0;
        if (base == -INFINITY) {
            n = 0;                                             // dead
        } else if (d.done[b]) {
            if (lane == 0) { l_s[p][0] = base; l_a[p][0] = -1; }   // stay
            n = 1;
        } else {
            const void *row = reinterpret_cast<const char *>(logits) + (size_t)b * d.A * esz;
            const uint32_t *mrow = d.mask_bits + (size_t)b * d.AW;
            const RowStats r = masked_row<DT, MODE_STATS>(row, mrow, d.A, d.AW, 0, lane);
            if (r.se > 0.f) {
                const float lse = row_lse(r);
                float ps = 0.f;
                int pa = 0;
                for (; n < W; ++n) {
                    beam_next<DT>(row, mrow, d.A, d.AW, LogProbScore{base, lse}, n == 0, ps, pa, lane, ps, pa);
                    if (pa == INT_MAX) break;
                    if (lane == 0) { l_s[p][n] = ps; l_a[p][n] = pa; }
                }
            }
        }
        if (lane == 0) l_n[p] = n;
    }
    __syncthreads();
    if (warp != 0) return;
    // Stage 2: lane p holds the head of list p; W rounds of a warp arg-max in the order produce the W winners
    int head = 0;
    const int len = lane < W ? l_n[lane] : 0;
    float my_s = -INFINITY;
    int my_p = -1, my_a = -1;
    for (int j = 0; j < W; ++j) {
        float s = -INFINITY;
        int p = INT_MAX, a = INT_MAX;                          // no candidate: after every real one
        if (head < len) { s = l_s[lane][head]; p = lane; a = l_a[lane][head]; }
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            const float s2 = __shfl_xor_sync(GE_FULL, s, o);
            const int p2 = __shfl_xor_sync(GE_FULL, p, o);
            const int a2 = __shfl_xor_sync(GE_FULL, a, o);
            if (beam_before(s2, p2, a2, s, p, a)) { s = s2; p = p2; a = a2; }
        }
        if (p == INT_MAX) break;                               // the group has fewer than W candidates: the rest stay empty
        if (lane == p) ++head;
        if (lane == j) { my_s = s; my_p = p; my_a = a; }
    }
    if (lane < W) {
        const int b = g0 + lane;
        const int par = my_p < 0 ? -1 : g0 + my_p;
        score_out[b] = my_s;
        parent[b] = par;
        action[b] = my_a;
        load_index[b] = par == b ? -1 : par;
    }
}

// ---- stochastic beam search (ge_beam_expand_sampled): beam_expand_kernel's layout, ranked by conditioned Gumbel keys ----
// log(1 - e^x) for x <= 0, accurate on both sides of -ln 2 (log1mexp(0) = -inf).
__device__ __forceinline__ float log1mexp(float x) {
    return x > -0.6931472f ? logf(-expm1f(x)) : log1pf(-expf(x));
}
// The key of the child whose perturbed score lies x = fl32(s_a - S_b) <= 0 below the beam's best, given the beam's key T and
// D = T - (its children's unconditioned maximum): T - softplus(v), v = (D - x) + log1mexp(x).  x = 0 gives T exactly.
__device__ __forceinline__ float conditioned_key(float T, float D, float x) {
    const float v = __fadd_rn(__fsub_rn(D, x), log1mexp(x));
    return __fsub_rn(T, __fadd_rn(fmaxf(v, 0.f), log1pf(expf(-fabsf(v)))));
}
// The node key of the child of node h by action a (include/graphenvs_b200.h, ge_beam_expand_sampled).
__device__ __forceinline__ uint64_t child_key(uint64_t h, int a) {
    return ((uint64_t)mix32(h, (uint32_t)a, 0x2545F491u) << 32) | (uint64_t)mix32(h ^ 0x9E3779B97F4A7C15ull, (uint32_t)a, 0x6C8E9CF5u);
}

template <int DT>
__global__ void __launch_bounds__(BEAM_WARPS * 32) beam_expand_sampled_kernel(ge_batch d, int W, const void *__restrict__ logits,
                                                                               const float *__restrict__ logp, const float *__restrict__ key,
                                                                               const uint64_t *__restrict__ node_key, float *__restrict__ logp_out,
                                                                               float *__restrict__ key_out, uint64_t *__restrict__ node_key_out,
                                                                               int32_t *__restrict__ parent, int32_t *__restrict__ action,
                                                                               int32_t *__restrict__ load_index, float *__restrict__ threshold) {
    __shared__ float l_g[BEAM_MAXW][BEAM_MAXW + 1];   // per beam: its best min(W + 1, candidates) candidates and their keys
    __shared__ int l_a[BEAM_MAXW][BEAM_MAXW + 1];
    __shared__ int l_n[BEAM_MAXW];
    __shared__ float l_lse[BEAM_MAXW];
    pdl_launch_dependents();   // as the sampler: nothing is touched before pdl_wait()
    pdl_wait();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int g0 = blockIdx.x * W;
    const size_t esz = DT == GE_LOGITS_BF16 ? 2 : 4;
    // Stage 1: every beam's W + 1 best candidates in the order (s_a desc, a asc), and their conditioned keys
    for (int p = warp; p < W; p += nwarps) {
        const int b = g0 + p;
        const float T = key[b];
        int n = 0;
        if (T == -INFINITY) {
            n = 0;                                                 // dead
        } else if (d.done[b]) {
            if (lane == 0) { l_g[p][0] = T; l_a[p][0] = -1; }    // stay
            n = 1;
        } else {
            const void *row = reinterpret_cast<const char *>(logits) + (size_t)b * d.A * esz;
            const uint32_t *mrow = d.mask_bits + (size_t)b * d.AW;
            const uint64_t nk = node_key[b];
            const RowStats r = masked_row<DT, MODE_NODE_GUMBEL>(row, mrow, d.A, d.AW, nk, lane);   // lse and the best (S_b, a)
            if (r.se > 0.f) {
                const float lse = row_lse(r), S = r.bs;
                const float D = __fsub_rn(T, __fadd_rn(logp[b], __fsub_rn(S, lse)));
                if (lane == 0) l_lse[p] = lse;
                float ps = S;
                int pa = r.bi;
                for (;;) {
                    if (lane == 0) { l_g[p][n] = conditioned_key(T, D, __fsub_rn(ps, S)); l_a[p][n] = pa; }
                    if (++n == W + 1) break;
                    beam_next<DT>(row, mrow, d.A, d.AW, PerturbedScore{nk}, false, ps, pa, lane, ps, pa);
                    if (pa == INT_MAX) break;
                }
            }
        }
        if (lane == 0) l_n[p] = n;
    }
    __syncthreads();
    if (warp != 0) return;
    // Lane p puts list p in the merge order (G desc, a asc): the keys follow s_a only up to rounding, so the list is nearly sorted
    const int len = lane < W ? l_n[lane] : 0;
    for (int i = 1; i < len; ++i) {
        const float g = l_g[lane][i];
        const int a = l_a[lane][i];
        int k = i;
        for (; k > 0 && beam_before(g, 0, a, l_g[lane][k - 1], 0, l_a[lane][k - 1]); --k) {
            l_g[lane][k] = l_g[lane][k - 1];
            l_a[lane][k] = l_a[lane][k - 1];
        }
        l_g[lane][k] = g;
        l_a[lane][k] = a;
    }
    // Stage 2: beam_expand_kernel's warp arg-max merge in the order (G desc, parent slot asc, action asc); round W is the threshold
    const int rounds = threshold ? W + 1 : W;
    int head = 0;
    float my_g = -INFINITY, thr = -INFINITY;
    int my_p = -1, my_a = -1;
    for (int j = 0; j < rounds; ++j) {
        float s = -INFINITY;
        int p = INT_MAX, a = INT_MAX;
        if (head < len) { s = l_g[lane][head]; p = lane; a = l_a[lane][head]; }
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            const float s2 = __shfl_xor_sync(GE_FULL, s, o);
            const int p2 = __shfl_xor_sync(GE_FULL, p, o);
            const int a2 = __shfl_xor_sync(GE_FULL, a, o);
            if (beam_before(s2, p2, a2, s, p, a)) { s = s2; p = p2; a = a2; }
        }
        if (p == INT_MAX) break;
        if (j == W) { thr = s; break; }
        if (lane == p) ++head;
        if (lane == j) { my_g = s; my_p = p; my_a = a; }
    }
    if (threshold && lane == 0) threshold[blockIdx.x] = thr;
    if (lane < W) {
        const int b = g0 + lane;
        const int par = my_p < 0 ? -1 : g0 + my_p;
        float lp = -INFINITY;
        uint64_t nk = 0;
        if (par >= 0) {
            lp = logp[par];
            nk = node_key[par];
            if (my_a >= 0) {   // a valid action of a live beam: its logit is read again, for the log-prob of ge_beam_expand
                const void *row = reinterpret_cast<const char *>(logits) + (size_t)par * d.A * esz;
                lp = __fadd_rn(lp, __fsub_rn(load_logit<DT>(row, (size_t)my_a), l_lse[my_p]));
                nk = child_key(nk, my_a);
            }
        }
        logp_out[b] = lp;
        key_out[b] = my_g;
        node_key_out[b] = nk;
        parent[b] = par;
        action[b] = my_a;
        load_index[b] = par == b ? -1 : par;
    }
}

// ---- Monte Carlo tree search (ge_mcts_select / ge_mcts_expand): one warp per instance; the tree arithmetic is float64 with
// every operation explicitly rounded (include/graphenvs_b200.h), so a float64 restatement reproduces it exactly ----
constexpr int MCTS_WPB = 8;   // warps (= instances) per block

__global__ void __launch_bounds__(MCTS_WPB * 32) mcts_select_kernel(ge_mcts_tree t, int k) {
    pdl_launch_dependents();   // as the sampler: nothing is touched before pdl_wait()
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int g = blockIdx.x * MCTS_WPB + (threadIdx.x >> 5);
    if (g >= t.G) return;
    const int G = t.G, A = t.A, AW = t.AW;
    const double qmin = t.qmin[g], qmax = t.qmax[g];
    const bool norm = qmax > qmin;
    const double qden = norm ? __dsub_rn(qmax, qmin) : 1.0;
    int s = 0, depth = 0, load = -1, act = -1;
    while (!t.terminal[(size_t)s * G + g]) {   // a terminal node is revisited
        const size_t row = (size_t)s * G + g;
        const double sq = __dsqrt_rn((double)t.visits[row]);
        const uint32_t *mrow = t.mask + row * AW;
        const float *prow = t.prior + row * A;
        const int32_t *crow = t.child + row * A;
        double best = -INFINITY;
        int ba = INT_MAX, bc = -1;
        // the valid actions of s, walked as masked_row walks a mask row: lane l owns action 32 w + l of every nonzero word w
        for (int w0 = 0; w0 < AW; w0 += 32) {
            const int wl = w0 + lane;
            const uint32_t mw = wl < AW ? (mrow[wl] & tail_mask(A, wl)) : 0u;
            unsigned nz = __ballot_sync(GE_FULL, mw != 0u);
            while (nz) {
                const int src = __ffs((int)nz) - 1;
                nz &= nz - 1u;
                const uint32_t word = __shfl_sync(GE_FULL, mw, src);
                if (!((word >> lane) & 1u)) continue;
                const int a = ((w0 + src) << 5) + lane;
                const int c = crow[a];
                double q = 0.0;
                int n = 0;
                if (c >= 0) {
                    const size_t rc = (size_t)c * G + g;
                    n = t.visits[rc];
                    if (norm) {
                        const double Q = __dadd_rn((double)t.reward[rc], __ddiv_rn(t.wsum[rc], (double)n));
                        q = __ddiv_rn(__dsub_rn(Q, qmin), qden);
                    }
                }
                const double u = __dadd_rn(q, __ddiv_rn(__dmul_rn(__dmul_rn(t.c_puct, (double)prow[a]), sq), (double)(1 + n)));
                if (u > best) { best = u; ba = a; bc = c; }   // strictly greater: a lane visits its actions in order
            }
        }
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            const double u2 = __shfl_xor_sync(GE_FULL, best, o);
            const int a2 = __shfl_xor_sync(GE_FULL, ba, o);
            const int c2 = __shfl_xor_sync(GE_FULL, bc, o);
            if (u2 > best || (u2 == best && a2 < ba)) { best = u2; ba = a2; bc = c2; }
        }
        if (ba == INT_MAX) break;                          // a dead end: revisit s
        ++depth;
        if (bc < 0) { load = (int)row; act = ba; break; }  // an unexpanded edge: expand s by ba
        s = bc;
    }
    if (lane == 0) {
        t.sel_node[g] = s;
        t.sel_action[g] = act;
        t.load_index[g] = load;
        t.depth[g] = depth;
    }
}

template <int DT, bool LOG_PRIOR>
__global__ void __launch_bounds__(MCTS_WPB * 32) mcts_expand_kernel(ge_batch d, ge_mcts_tree t, int k, const float *__restrict__ reward,
                                                                     const void *__restrict__ logits, const float *__restrict__ value) {
    pdl_launch_dependents();   // as the sampler: nothing is touched before pdl_wait()
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int g = blockIdx.x * MCTS_WPB + (threadIdx.x >> 5);
    if (g >= t.G) return;
    const int G = t.G, A = t.A, AW = t.AW;
    const size_t rk = (size_t)k * G + g;
    const int a = k ? t.sel_action[g] : -1;
    const int par = k ? t.sel_node[g] : -1;
    int leaf = par;                                        // a revisit backs up from the selected node
    if (k == 0 || a >= 0) {                                // node k: its mask, and over its valid actions its priors and no child
        const size_t esz = DT == GE_LOGITS_BF16 ? 2 : 4;
        const void *row = reinterpret_cast<const char *>(logits) + (size_t)g * A * esz;
        const uint32_t *lm = d.mask_bits + (size_t)g * d.AW;
        const float lse = row_lse(masked_row<DT, MODE_STATS>(row, lm, A, AW, 0, lane));
        uint32_t *nm = t.mask + rk * AW;
        float *prow = t.prior + rk * A;
        int32_t *crow = t.child + rk * A;
        for (int w0 = 0; w0 < AW; w0 += 32) {
            const int wl = w0 + lane;
            const uint32_t mw = wl < AW ? (__ldg(lm + wl) & tail_mask(A, wl)) : 0u;
            if (wl < AW) nm[wl] = mw;
            unsigned nz = __ballot_sync(GE_FULL, mw != 0u);
            while (nz) {
                const int src = __ffs((int)nz) - 1;
                nz &= nz - 1u;
                const uint32_t word = __shfl_sync(GE_FULL, mw, src);
                if ((word >> lane) & 1u) {
                    const int i = ((w0 + src) << 5) + lane;
                    const float lp = __fsub_rn(load_logit<DT>(row, (size_t)i), lse);
                    prow[i] = LOG_PRIOR ? lp : expf(lp);   // GE_MCTS_LOG_PRIOR: the log-prior of the Gumbel search
                    crow[i] = -1;
                }
            }
        }
        if (lane == 0) {
            const bool term = d.done[g] != 0;
            t.parent[rk] = par;
            t.action[rk] = a;
            t.reward[rk] = k ? reward[g] : 0.f;
            t.terminal[rk] = term;
            t.value[rk] = term ? 0.f : value[g];
            t.visits[rk] = 0;
            t.wsum[rk] = 0.0;
            if (k) t.child[((size_t)par * G + g) * A + a] = k;
            else { t.qmin[g] = INFINITY; t.qmax[g] = -INFINITY; }
        }
        leaf = k;
    } else if (lane == 0) {                                // slot k stays unused
        t.parent[rk] = -1;
        t.action[rk] = -1;
        t.visits[rk] = 0;
    }
    if (lane != 0) return;
    // backup (MuZero's order): from the leaf up to and including the root
    double ret = (double)t.value[(size_t)leaf * G + g];
    double qmin = t.qmin[g], qmax = t.qmax[g];
    for (int c = leaf;;) {
        const size_t rc = (size_t)c * G + g;
        const int n = t.visits[rc] + 1;
        const double w = __dadd_rn(t.wsum[rc], ret);
        t.visits[rc] = n;
        t.wsum[rc] = w;
        if (c == 0) break;
        const double r = (double)t.reward[rc];
        const double Q = __dadd_rn(r, __ddiv_rn(w, (double)n));
        qmin = fmin(qmin, Q);
        qmax = fmax(qmax, Q);
        ret = __dadd_rn(r, ret);
        c = t.parent[rc];
    }
    t.qmin[g] = qmin;
    t.qmax[g] = qmax;
}

// ---- Gumbel MuZero search (ge_gumbel_root / ge_gumbel_select / ge_gumbel_result): one warp per instance over a GE_MCTS_LOG_PRIOR
// tree, with the arithmetic of include/graphenvs_b200.h (float64, every operation explicitly rounded, fixed reduction order) ----

// f(a) for every valid action a of a node, walked as mcts_select_kernel walks it: lane l takes the actions a = l mod 32, ascending.
// f runs on the lanes that own a valid action only, so it must not use warp collectives.
template <class F>
__device__ __forceinline__ void for_valid(const uint32_t *mrow, int A, int AW, int lane, F f) {
    for (int w0 = 0; w0 < AW; w0 += 32) {
        const int wl = w0 + lane;
        const uint32_t mw = wl < AW ? (mrow[wl] & tail_mask(A, wl)) : 0u;
        unsigned nz = __ballot_sync(GE_FULL, mw != 0u);
        while (nz) {
            const int src = __ffs((int)nz) - 1;
            nz &= nz - 1u;
            const uint32_t word = __shfl_sync(GE_FULL, mw, src);
            if ((word >> lane) & 1u) f(((w0 + src) << 5) + lane);
        }
    }
}

// Node s of instance g with the statistics of its completed Q (warp-uniform).
struct GNode {
    const uint32_t *mrow;
    const float *lrow;     // log-priors l(s, a)
    const int32_t *crow;
    double vmix, lo, den, cs;   // q~ = (q^ - lo) / den, sigma = cs * q~
    int M, maxn, nvalid;
};

// N(s, a) of the edge (c = its child, -1 when unexpanded) and q^(a), which is Q(s, a) when N > 0 and vmix otherwise.
__device__ __forceinline__ double edge_q(const ge_mcts_tree &t, const int32_t *crow, int a, int g, double vmix, int &n, int &c) {
    c = crow[a];
    n = 0;
    if (c >= 0) {
        const size_t rc = (size_t)c * t.G + g;
        n = t.visits[rc];
        if (n > 0) return __dadd_rn((double)t.reward[rc], __ddiv_rn(t.wsum[rc], (double)n));
    }
    return vmix;
}

__device__ __forceinline__ double gnode_sigma(const GNode &nd, double qh) {
    return __dmul_rn(nd.cs, __ddiv_rn(__dsub_rn(qh, nd.lo), nd.den));
}

// Pass 1 over the node's valid actions: M, max N, the mixed value and the range of q^.
__device__ __forceinline__ GNode gumbel_node(const ge_mcts_tree &t, const ge_gumbel_params &p, int s, int g, int lane) {
    const size_t row = (size_t)s * t.G + g;
    GNode nd;
    nd.mrow = t.mask + row * t.AW;
    nd.lrow = t.prior + row * t.A;
    nd.crow = t.child + row * t.A;
    double sp = 0.0, spq = 0.0, qlo = INFINITY, qhi = -INFINITY;
    int M = 0, maxn = 0, nvalid = 0;
    bool unvisited = false;
    for_valid(nd.mrow, t.A, t.AW, lane, [&](int a) {
        int n, c;
        const double Q = edge_q(t, nd.crow, a, g, 0.0, n, c);
        ++nvalid;
        if (n > 0) {
            const double P = fmax(exp((double)nd.lrow[a]), DBL_MIN);
            sp = __dadd_rn(sp, P);
            spq = __dadd_rn(spq, __dmul_rn(P, Q));
            qlo = fmin(qlo, Q);
            qhi = fmax(qhi, Q);
            M += n;
            maxn = max(maxn, n);
        } else {
            unvisited = true;
        }
    });
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        sp = __dadd_rn(sp, __shfl_xor_sync(GE_FULL, sp, o));
        spq = __dadd_rn(spq, __shfl_xor_sync(GE_FULL, spq, o));
        qlo = fmin(qlo, __shfl_xor_sync(GE_FULL, qlo, o));
        qhi = fmax(qhi, __shfl_xor_sync(GE_FULL, qhi, o));
        M += __shfl_xor_sync(GE_FULL, M, o);
        maxn = max(maxn, __shfl_xor_sync(GE_FULL, maxn, o));
        nvalid += __shfl_xor_sync(GE_FULL, nvalid, o);
    }
    unvisited = __any_sync(GE_FULL, unvisited);
    const double v = (double)t.value[row];
    nd.vmix = M ? __ddiv_rn(__dadd_rn(v, __dmul_rn((double)M, __ddiv_rn(spq, sp))), (double)(M + 1)) : v;
    if (unvisited) { qlo = fmin(qlo, nd.vmix); qhi = fmax(qhi, nd.vmix); }
    nd.lo = qlo;
    nd.den = fmax(__dsub_rn(qhi, qlo), 1e-8);
    nd.cs = __dmul_rn(__dadd_rn(p.maxvisit_init, (double)maxn), p.value_scale);
    nd.M = M; nd.maxn = maxn; nd.nvalid = nvalid;
    return nd;
}

// Pass 2: the softmax normaliser of z = l + sigma over the valid actions, online per lane, merged in the butterfly order.
__device__ __forceinline__ void gumbel_norm(const ge_mcts_tree &t, const GNode &nd, int g, int lane, double &zm, double &zs) {
    zm = -INFINITY; zs = 0.0;
    for_valid(nd.mrow, t.A, t.AW, lane, [&](int a) {
        int n, c;
        const double z = __dadd_rn((double)nd.lrow[a], gnode_sigma(nd, edge_q(t, nd.crow, a, g, nd.vmix, n, c)));
        if (z > zm) { zs = __dadd_rn(__dmul_rn(zs, exp(__dsub_rn(zm, z))), 1.0); zm = z; }
        else zs = __dadd_rn(zs, exp(__dsub_rn(z, zm)));
    });
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const double zm2 = __shfl_xor_sync(GE_FULL, zm, o), zs2 = __shfl_xor_sync(GE_FULL, zs, o);
        const double mx = fmax(zm, zm2);
        zs = __dadd_rn(zs > 0.0 ? __dmul_rn(zs, exp(__dsub_rn(zm, mx))) : 0.0, zs2 > 0.0 ? __dmul_rn(zs2, exp(__dsub_rn(zm2, mx))) : 0.0);
        zm = mx;
    }
}

// The warp's largest score, ties to the lowest action (ba = INT_MAX when no lane has a candidate).
__device__ __forceinline__ void warp_best(double &best, int &ba, int &bc) {
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const double u2 = __shfl_xor_sync(GE_FULL, best, o);
        const int a2 = __shfl_xor_sync(GE_FULL, ba, o);
        const int c2 = __shfl_xor_sync(GE_FULL, bc, o);
        if (u2 > best || (u2 == best && a2 < ba)) { best = u2; ba = a2; bc = c2; }
    }
}

// The root's score (g + l) + sigma over its valid actions with N = vstar: the best one (pass 2 at the root, and the readout).
__device__ __forceinline__ void gumbel_root_best(const ge_mcts_tree &t, const ge_gumbel_params &p, const GNode &nd, int g, int lane,
                                                 int vstar, int &ba, int &bc) {
    const float *nrow = p.noise + (size_t)g * t.A;
    double best = -INFINITY;
    ba = INT_MAX; bc = -1;
    for_valid(nd.mrow, t.A, t.AW, lane, [&](int a) {
        int n, c;
        const double qh = edge_q(t, nd.crow, a, g, nd.vmix, n, c);
        if (n != vstar) return;
        const double u = __dadd_rn(__dadd_rn((double)nrow[a], (double)nd.lrow[a]), gnode_sigma(nd, qh));
        if (u > best) { best = u; ba = a; bc = c; }   // strictly greater: a lane visits its actions in order
    });
    warp_best(best, ba, bc);
}

__global__ void __launch_bounds__(MCTS_WPB * 32) gumbel_root_kernel(ge_mcts_tree t, ge_gumbel_params p, uint64_t seed, uint32_t step,
                                                                     int env_id0) {
    pdl_launch_dependents();   // as the sampler: nothing is touched before pdl_wait()
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int g = blockIdx.x * MCTS_WPB + (threadIdx.x >> 5);
    if (g >= t.G) return;
    const uint64_t key = row_key(seed, (uint32_t)(env_id0 + g), step);
    float *nrow = p.noise + (size_t)g * t.A;
    for_valid(t.mask + (size_t)g * t.AW, t.A, t.AW, lane, [&](int a) { nrow[a] = node_gumbel(key, a); });
}

__global__ void __launch_bounds__(MCTS_WPB * 32) gumbel_select_kernel(ge_mcts_tree t, ge_gumbel_params p, int k) {
    pdl_launch_dependents();   // as the sampler: nothing is touched before pdl_wait()
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int g = blockIdx.x * MCTS_WPB + (threadIdx.x >> 5);
    if (g >= t.G) return;
    const int G = t.G;
    int s = 0, depth = 0, load = -1, act = -1;
    while (!t.terminal[(size_t)s * G + g]) {   // a terminal node is revisited
        const size_t row = (size_t)s * G + g;
        const GNode nd = gumbel_node(t, p, s, g, lane);
        if (nd.nvalid == 0) break;                         // a dead end: revisit s
        int ba, bc;
        if (s == 0) {                                      // sequential halving over the considered actions
            const int vstar = p.table[(size_t)min(p.m, nd.nvalid) * t.S + min(nd.M, t.S - 1)];
            gumbel_root_best(t, p, nd, g, lane, vstar, ba, bc);
        } else {                                           // pi'(a) - N(s, a) / (1 + M)
            double zm, zs;
            gumbel_norm(t, nd, g, lane, zm, zs);
            const double vden = (double)(1 + nd.M);
            double best = -INFINITY;
            ba = INT_MAX; bc = -1;
            for_valid(nd.mrow, t.A, t.AW, lane, [&](int a) {
                int n, c;
                const double z = __dadd_rn((double)nd.lrow[a], gnode_sigma(nd, edge_q(t, nd.crow, a, g, nd.vmix, n, c)));
                const double u = __dsub_rn(__ddiv_rn(exp(__dsub_rn(z, zm)), zs), __ddiv_rn((double)n, vden));
                if (u > best) { best = u; ba = a; bc = c; }
            });
            warp_best(best, ba, bc);
        }
        if (ba == INT_MAX) break;                          // no considered action: revisit s
        ++depth;
        if (bc < 0) { load = (int)row; act = ba; break; }  // an unexpanded edge: expand s by ba
        s = bc;
    }
    if (lane == 0) {
        t.sel_node[g] = s;
        t.sel_action[g] = act;
        t.load_index[g] = load;
        t.depth[g] = depth;
    }
}

__global__ void __launch_bounds__(MCTS_WPB * 32) gumbel_result_kernel(ge_mcts_tree t, ge_gumbel_params p, int32_t *__restrict__ action,
                                                                       float *__restrict__ policy, double *__restrict__ completed_q) {
    pdl_launch_dependents();   // as the sampler: nothing is touched before pdl_wait()
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const int g = blockIdx.x * MCTS_WPB + (threadIdx.x >> 5);
    if (g >= t.G) return;
    const int A = t.A;
    const GNode nd = gumbel_node(t, p, 0, g, lane);
    double zm, zs;
    gumbel_norm(t, nd, g, lane, zm, zs);
    int ba, bc;
    gumbel_root_best(t, p, nd, g, lane, nd.maxn, ba, bc);
    float *prow = policy + (size_t)g * A;
    double *qrow = completed_q + (size_t)g * A;
    for (int a = lane; a < A; a += 32) {
        float pa = 0.f;
        double q = NAN;
        if ((nd.mrow[a >> 5] >> (a & 31)) & 1u) {
            int n, c;
            q = edge_q(t, nd.crow, a, g, nd.vmix, n, c);
            pa = __double2float_rn(__ddiv_rn(exp(__dsub_rn(__dadd_rn((double)nd.lrow[a], gnode_sigma(nd, q)), zm)), zs));
        }
        prow[a] = pa;
        qrow[a] = q;
    }
    if (lane == 0) action[g] = (t.terminal[g] || ba == INT_MAX) ? -1 : ba;
}

int check_tree(const char *fn, const ge_mcts_tree *t, int k, int kmin) {
    if (!t) return ge_set_error(GE_ERR_ARG, "%s: null tree", fn);
    if (t->G < 1 || t->S < 1 || t->A < 1 || t->AW != (t->A + 31) / 32)
        return ge_set_error(GE_ERR_ARG, "%s: bad tree shape G=%d S=%d A=%d AW=%d", fn, t->G, t->S, t->A, t->AW);
    if (!isfinite(t->c_puct) || t->c_puct < 0.0) return ge_set_error(GE_ERR_ARG, "%s: c_puct = %g must be finite and >= 0", fn, t->c_puct);
    if (k < kmin || k > t->S) return ge_set_error(GE_ERR_ARG, "%s: k = %d not in [%d, %d]", fn, k, kmin, t->S);
    if (!t->parent || !t->action || !t->visits || !t->wsum || !t->reward || !t->value || !t->terminal || !t->child || !t->prior ||
        !t->mask || !t->qmin || !t->qmax || !t->sel_node || !t->sel_action || !t->load_index || !t->depth)
        return ge_set_error(GE_ERR_ARG, "%s: null tree array", fn);
    return GE_OK;
}

int check_gumbel(const char *fn, const ge_mcts_tree *t, const ge_gumbel_params *p, int k, int kmin) {
    const int rc = check_tree(fn, t, k, kmin);
    if (rc) return rc;
    if (!(t->flags & GE_MCTS_LOG_PRIOR)) return ge_set_error(GE_ERR_ARG, "%s: the tree lacks GE_MCTS_LOG_PRIOR", fn);
    if (!p) return ge_set_error(GE_ERR_ARG, "%s: null params", fn);
    if (p->m < 1) return ge_set_error(GE_ERR_ARG, "%s: m = %d must be >= 1", fn, p->m);
    if (!isfinite(p->value_scale) || p->value_scale < 0.0)
        return ge_set_error(GE_ERR_ARG, "%s: value_scale = %g must be finite and >= 0", fn, p->value_scale);
    if (!isfinite(p->maxvisit_init) || p->maxvisit_init < 0.0)
        return ge_set_error(GE_ERR_ARG, "%s: maxvisit_init = %g must be finite and >= 0", fn, p->maxvisit_init);
    if (!p->table || !p->noise) return ge_set_error(GE_ERR_ARG, "%s: null table / noise", fn);
    return GE_OK;
}

// A warp-per-instance tree kernel, launched with programmatic stream serialization when the tree's flags have GE_FLAG_PDL.
template <class... KArgs, class... Args>
int launch_tree(const char *what, void (*kernel)(KArgs...), const ge_mcts_tree *tree, void *stream, Args... args) {
    cudaLaunchConfig_t cfg = {};   // ge_launch_step's launch, with the PDL flag of the tree
    cfg.gridDim = dim3((unsigned)((tree->G + MCTS_WPB - 1) / MCTS_WPB));
    cfg.blockDim = dim3(MCTS_WPB * 32);
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = (tree->flags & GE_FLAG_PDL) ? 1 : 0;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, args...);
    if (e != cudaSuccess) { (void)cudaGetLastError(); return ge_set_error(GE_ERR_CUDA, "%s launch: %s", what, cudaGetErrorString(e)); }
    return GE_OK;
}

int launched(const char *what) {
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? GE_OK : ge_set_error(GE_ERR_CUDA, "%s launch: %s", what, cudaGetErrorString(e));
}

int check_rows(const char *fn, const void *logits, int dtype, int B, int A, const uint32_t *mask_bits, const int32_t *actions) {
    if (dtype != GE_LOGITS_F32 && dtype != GE_LOGITS_BF16) return ge_set_error(GE_ERR_ARG, "%s: unknown logits dtype %d", fn, dtype);
    if (B <= 0 || A <= 0) return ge_set_error(GE_ERR_ARG, "%s: bad shape B=%d A=%d", fn, B, A);
    if (!logits || !mask_bits || !actions) return ge_set_error(GE_ERR_ARG, "%s: null logits / mask_bits / actions", fn);
    return GE_OK;
}

}  // namespace

extern "C" {

int ge_sample_logits(const ge_batch *d, const void *logits, int dtype, int greedy, uint64_t seed, uint32_t t, int32_t *actions,
                     float *log_prob, float *entropy, void *stream) {
    GE_NVTX("ge_sample_logits");
    if (!d) return ge_set_error(GE_ERR_ARG, "ge_sample_logits: null batch");
    if (dtype != GE_LOGITS_F32 && dtype != GE_LOGITS_BF16) return ge_set_error(GE_ERR_ARG, "ge_sample_logits: unknown logits dtype %d", dtype);
    if (d->B <= 0 || d->A <= 0 || d->AW != (d->A + 31) / 32) return ge_set_error(GE_ERR_ARG, "ge_sample_logits: bad shape B=%d A=%d AW=%d (call ge_fill_layout)", d->B, d->A, d->AW);
    if (!logits || !actions || !d->mask_bits) return ge_set_error(GE_ERR_ARG, "ge_sample_logits: null logits / actions / mask_bits");
    const dim3 grid((d->B + POL_WPB - 1) / POL_WPB), block(POL_WPB * 32);
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e;
    if (dtype == GE_LOGITS_BF16)
        e = greedy ? ge_launch_step(policy_sample_kernel<GE_LOGITS_BF16, MODE_GREEDY>, grid, block, 0, st, *d, logits, seed, t, actions, log_prob, entropy)
                   : ge_launch_step(policy_sample_kernel<GE_LOGITS_BF16, MODE_GUMBEL>, grid, block, 0, st, *d, logits, seed, t, actions, log_prob, entropy);
    else
        e = greedy ? ge_launch_step(policy_sample_kernel<GE_LOGITS_F32, MODE_GREEDY>, grid, block, 0, st, *d, logits, seed, t, actions, log_prob, entropy)
                   : ge_launch_step(policy_sample_kernel<GE_LOGITS_F32, MODE_GUMBEL>, grid, block, 0, st, *d, logits, seed, t, actions, log_prob, entropy);
    if (e != cudaSuccess) { (void)cudaGetLastError(); return ge_set_error(GE_ERR_CUDA, "policy_sample_kernel launch: %s", cudaGetErrorString(e)); }
    return GE_OK;
}

int ge_masked_log_prob(const void *logits, int dtype, int B, int A, const uint32_t *mask_bits, const int32_t *actions, float *log_prob,
                       float *entropy, float *lse, void *stream) {
    GE_NVTX("ge_masked_log_prob");
    int rc = check_rows("ge_masked_log_prob", logits, dtype, B, A, mask_bits, actions);
    if (rc) return rc;
    if (!log_prob || !entropy || !lse) return ge_set_error(GE_ERR_ARG, "ge_masked_log_prob: null log_prob / entropy / lse");
    const unsigned grid = (unsigned)((B + POL_WPB - 1) / POL_WPB);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == GE_LOGITS_BF16) policy_logprob_kernel<GE_LOGITS_BF16><<<grid, POL_WPB * 32, 0, st>>>(logits, B, A, mask_bits, actions, log_prob, entropy, lse);
    else policy_logprob_kernel<GE_LOGITS_F32><<<grid, POL_WPB * 32, 0, st>>>(logits, B, A, mask_bits, actions, log_prob, entropy, lse);
    return launched("policy_logprob_kernel");
}

int ge_masked_log_prob_backward(const void *logits, int dtype, int B, int A, const uint32_t *mask_bits, const int32_t *actions,
                                const float *lse, const float *entropy, const float *grad_log_prob, const float *grad_entropy,
                                void *grad_logits, void *stream) {
    GE_NVTX("ge_masked_log_prob_backward");
    int rc = check_rows("ge_masked_log_prob_backward", logits, dtype, B, A, mask_bits, actions);
    if (rc) return rc;
    if (!lse || !entropy || !grad_logits) return ge_set_error(GE_ERR_ARG, "ge_masked_log_prob_backward: null lse / entropy / grad_logits");
    const unsigned grid = (unsigned)((B + POL_WPB - 1) / POL_WPB);
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == GE_LOGITS_BF16)
        policy_logprob_bwd_kernel<GE_LOGITS_BF16><<<grid, POL_WPB * 32, 0, st>>>(logits, B, A, mask_bits, actions, lse, entropy, grad_log_prob, grad_entropy, grad_logits);
    else
        policy_logprob_bwd_kernel<GE_LOGITS_F32><<<grid, POL_WPB * 32, 0, st>>>(logits, B, A, mask_bits, actions, lse, entropy, grad_log_prob, grad_entropy, grad_logits);
    return launched("policy_logprob_bwd_kernel");
}

int ge_beam_expand(const ge_batch *d, int W, const void *logits, int dtype, const float *score, float *score_out, int32_t *parent,
                   int32_t *action, int32_t *load_index, void *stream) {
    GE_NVTX("ge_beam_expand");
    if (!d) return ge_set_error(GE_ERR_ARG, "ge_beam_expand: null batch");
    if (dtype != GE_LOGITS_F32 && dtype != GE_LOGITS_BF16) return ge_set_error(GE_ERR_ARG, "ge_beam_expand: unknown logits dtype %d", dtype);
    if (W < 1 || W > BEAM_MAXW) return ge_set_error(GE_ERR_ARG, "ge_beam_expand: width W = %d not in [1, %d]", W, BEAM_MAXW);
    if (d->B <= 0 || d->A <= 0 || d->AW != (d->A + 31) / 32) return ge_set_error(GE_ERR_ARG, "ge_beam_expand: bad shape B=%d A=%d AW=%d (call ge_fill_layout)", d->B, d->A, d->AW);
    if (d->B % W) return ge_set_error(GE_ERR_ARG, "ge_beam_expand: B = %d is not a multiple of W = %d", d->B, W);
    if (!logits || !score || !score_out || !parent || !action || !load_index)
        return ge_set_error(GE_ERR_ARG, "ge_beam_expand: null logits / score / score_out / parent / action / load_index");
    if (!d->mask_bits || !d->done) return ge_set_error(GE_ERR_ARG, "ge_beam_expand: null mask_bits / done in the batch");
    {   // no two of score, score_out, parent, action, load_index (B 4-byte elements each) may overlap
        const uintptr_t p[5] = {(uintptr_t)score, (uintptr_t)score_out, (uintptr_t)parent, (uintptr_t)action, (uintptr_t)load_index};
        const uintptr_t n = (uintptr_t)d->B * 4u;
        for (int i = 0; i < 5; ++i)
            for (int j = i + 1; j < 5; ++j)
                if (p[i] < p[j] + n && p[j] < p[i] + n)
                    return ge_set_error(GE_ERR_ARG, "ge_beam_expand: score, score_out, parent, action and load_index must not overlap");
    }
    const int warps = W < BEAM_WARPS ? W : BEAM_WARPS;
    const dim3 grid((unsigned)(d->B / W)), block(warps * 32);
    cudaStream_t st = (cudaStream_t)stream;
    const cudaError_t e = dtype == GE_LOGITS_BF16
        ? ge_launch_step(beam_expand_kernel<GE_LOGITS_BF16>, grid, block, 0, st, *d, W, logits, score, score_out, parent, action, load_index)
        : ge_launch_step(beam_expand_kernel<GE_LOGITS_F32>, grid, block, 0, st, *d, W, logits, score, score_out, parent, action, load_index);
    if (e != cudaSuccess) { (void)cudaGetLastError(); return ge_set_error(GE_ERR_CUDA, "beam_expand_kernel launch: %s", cudaGetErrorString(e)); }
    return GE_OK;
}

int ge_beam_expand_sampled(const ge_batch *d, int W, const void *logits, int dtype, const float *logp, const float *key,
                           const uint64_t *node_key, float *logp_out, float *key_out, uint64_t *node_key_out, int32_t *parent,
                           int32_t *action, int32_t *load_index, float *threshold, void *stream) {
    GE_NVTX("ge_beam_expand_sampled");
    const char *fn = "ge_beam_expand_sampled";
    if (!d) return ge_set_error(GE_ERR_ARG, "%s: null batch", fn);
    if (dtype != GE_LOGITS_F32 && dtype != GE_LOGITS_BF16) return ge_set_error(GE_ERR_ARG, "%s: unknown logits dtype %d", fn, dtype);
    if (W < 1 || W > BEAM_MAXW) return ge_set_error(GE_ERR_ARG, "%s: width W = %d not in [1, %d]", fn, W, BEAM_MAXW);
    if (d->B <= 0 || d->A <= 0 || d->AW != (d->A + 31) / 32) return ge_set_error(GE_ERR_ARG, "%s: bad shape B=%d A=%d AW=%d (call ge_fill_layout)", fn, d->B, d->A, d->AW);
    if (d->B % W) return ge_set_error(GE_ERR_ARG, "%s: B = %d is not a multiple of W = %d", fn, d->B, W);
    if (!logits || !logp || !key || !node_key || !logp_out || !key_out || !node_key_out || !parent || !action || !load_index)
        return ge_set_error(GE_ERR_ARG, "%s: null logits / logp / key / node_key / logp_out / key_out / node_key_out / parent / action / load_index", fn);
    if (!d->mask_bits || !d->done) return ge_set_error(GE_ERR_ARG, "%s: null mask_bits / done in the batch", fn);
    {   // no two of the arrays may overlap: B elements of 4 bytes each (8 for the node keys), B / W floats of threshold
        const uintptr_t B = (uintptr_t)d->B;
        const uintptr_t p[10] = {(uintptr_t)logp, (uintptr_t)key, (uintptr_t)node_key, (uintptr_t)logp_out, (uintptr_t)key_out,
                                 (uintptr_t)node_key_out, (uintptr_t)parent, (uintptr_t)action, (uintptr_t)load_index, (uintptr_t)threshold};
        const uintptr_t n[10] = {4 * B, 4 * B, 8 * B, 4 * B, 4 * B, 8 * B, 4 * B, 4 * B, 4 * B, threshold ? 4 * (B / W) : 0};
        for (int i = 0; i < 10; ++i)
            for (int j = i + 1; j < 10; ++j)
                if (n[i] && n[j] && p[i] < p[j] + n[j] && p[j] < p[i] + n[i])
                    return ge_set_error(GE_ERR_ARG, "%s: logp, key, node_key, logp_out, key_out, node_key_out, parent, action, load_index "
                                                    "and threshold must not overlap", fn);
    }
    const int warps = W < BEAM_WARPS ? W : BEAM_WARPS;
    const dim3 grid((unsigned)(d->B / W)), block(warps * 32);
    cudaStream_t st = (cudaStream_t)stream;
    const cudaError_t e = dtype == GE_LOGITS_BF16
        ? ge_launch_step(beam_expand_sampled_kernel<GE_LOGITS_BF16>, grid, block, 0, st, *d, W, logits, logp, key, node_key, logp_out,
                         key_out, node_key_out, parent, action, load_index, threshold)
        : ge_launch_step(beam_expand_sampled_kernel<GE_LOGITS_F32>, grid, block, 0, st, *d, W, logits, logp, key, node_key, logp_out,
                         key_out, node_key_out, parent, action, load_index, threshold);
    if (e != cudaSuccess) { (void)cudaGetLastError(); return ge_set_error(GE_ERR_CUDA, "beam_expand_sampled_kernel launch: %s", cudaGetErrorString(e)); }
    return GE_OK;
}

int ge_mcts_select(const ge_mcts_tree *tree, int k, void *stream) {
    GE_NVTX("ge_mcts_select");
    const int rc = check_tree("ge_mcts_select", tree, k, 1);
    if (rc) return rc;
    if (tree->flags & GE_MCTS_LOG_PRIOR)
        return ge_set_error(GE_ERR_ARG, "ge_mcts_select: the tree has GE_MCTS_LOG_PRIOR (log-priors: use ge_gumbel_select)");
    return launch_tree("mcts_select_kernel", mcts_select_kernel, tree, stream, *tree, k);
}

int ge_mcts_expand(const ge_mcts_tree *tree, int k, const ge_batch *leaf, const float *reward, const void *logits, int dtype,
                   const float *value, void *stream) {
    GE_NVTX("ge_mcts_expand");
    const char *fn = "ge_mcts_expand";
    const int rc = check_tree(fn, tree, k, 0);
    if (rc) return rc;
    if (!leaf) return ge_set_error(GE_ERR_ARG, "%s: null leaf batch", fn);
    if (dtype != GE_LOGITS_F32 && dtype != GE_LOGITS_BF16) return ge_set_error(GE_ERR_ARG, "%s: unknown logits dtype %d", fn, dtype);
    if (leaf->B != tree->G || leaf->A != tree->A || leaf->AW != tree->AW)
        return ge_set_error(GE_ERR_ARG, "%s: leaf batch B=%d A=%d AW=%d, tree G=%d A=%d AW=%d", fn, leaf->B, leaf->A, leaf->AW, tree->G, tree->A, tree->AW);
    if (!reward || !logits || !value) return ge_set_error(GE_ERR_ARG, "%s: null reward / logits / value", fn);
    if (!leaf->mask_bits || !leaf->done) return ge_set_error(GE_ERR_ARG, "%s: null mask_bits / done in the leaf batch", fn);
    const dim3 grid((unsigned)((tree->G + MCTS_WPB - 1) / MCTS_WPB)), block(MCTS_WPB * 32);
    cudaStream_t st = (cudaStream_t)stream;
    const bool lp = (tree->flags & GE_MCTS_LOG_PRIOR) != 0;
    const cudaError_t e = dtype == GE_LOGITS_BF16
        ? (lp ? ge_launch_step(mcts_expand_kernel<GE_LOGITS_BF16, true>, grid, block, 0, st, *leaf, *tree, k, reward, logits, value)
              : ge_launch_step(mcts_expand_kernel<GE_LOGITS_BF16, false>, grid, block, 0, st, *leaf, *tree, k, reward, logits, value))
        : (lp ? ge_launch_step(mcts_expand_kernel<GE_LOGITS_F32, true>, grid, block, 0, st, *leaf, *tree, k, reward, logits, value)
              : ge_launch_step(mcts_expand_kernel<GE_LOGITS_F32, false>, grid, block, 0, st, *leaf, *tree, k, reward, logits, value));
    if (e != cudaSuccess) { (void)cudaGetLastError(); return ge_set_error(GE_ERR_CUDA, "mcts_expand_kernel launch: %s", cudaGetErrorString(e)); }
    return GE_OK;
}

int ge_gumbel_root(const ge_mcts_tree *tree, const ge_gumbel_params *params, uint64_t seed, uint32_t t, int32_t env_id0, void *stream) {
    GE_NVTX("ge_gumbel_root");
    const int rc = check_gumbel("ge_gumbel_root", tree, params, 0, 0);
    if (rc) return rc;
    return launch_tree("gumbel_root_kernel", gumbel_root_kernel, tree, stream, *tree, *params, seed, t, (int)env_id0);
}

int ge_gumbel_select(const ge_mcts_tree *tree, const ge_gumbel_params *params, int k, void *stream) {
    GE_NVTX("ge_gumbel_select");
    const int rc = check_gumbel("ge_gumbel_select", tree, params, k, 1);
    if (rc) return rc;
    return launch_tree("gumbel_select_kernel", gumbel_select_kernel, tree, stream, *tree, *params, k);
}

int ge_gumbel_result(const ge_mcts_tree *tree, const ge_gumbel_params *params, int32_t *action, float *policy, double *completed_q,
                     void *stream) {
    GE_NVTX("ge_gumbel_result");
    const char *fn = "ge_gumbel_result";
    const int rc = check_gumbel(fn, tree, params, 0, 0);
    if (rc) return rc;
    if (!action || !policy || !completed_q) return ge_set_error(GE_ERR_ARG, "%s: null action / policy / completed_q", fn);
    return launch_tree("gumbel_result_kernel", gumbel_result_kernel, tree, stream, *tree, *params, action, policy, completed_q);
}

}  // extern "C"
