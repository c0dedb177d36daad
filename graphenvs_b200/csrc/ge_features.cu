// ge_features.cu -- feature_extraction.generate_features (feature_extraction.py:6-37) on the GPU.
// Per node, in the reference's column order: G.degree (in+out of the directed symmetric graph),
// betweenness (Brandes, nx:centrality/betweenness.py), closeness (Wasserman-Faust,
// nx:centrality/closeness.py), pagerank (scipy power iteration, nx:link_analysis/pagerank_alg.py,
// alpha .85, tol 1e-6, <= 100 it., same stopping rule), clustering (directed Fagiolo form,
// nx:algorithms/cluster.py).  All arithmetic in fp64, rounded to float32 at the end exactly like
// `torch.tensor(sf)` (feature_extraction.py:36).
//
// Round-2 design (features_cta_kernel, N <= 1024): ONE CTA PER ENV, ONE WARP PER BFS SOURCE.
//   * the env's adjacency lives in shared memory as an N x NWP bit-matrix built once from the CSR
//     (row stride NWP words = an odd number of 16-byte quads => lane-private rows are read with
//     conflict-free 128-bit loads);
//   * Brandes runs in PULL form on that matrix, without a single atomic: an unvisited node w joins
//     level k iff row(w) & L_{k-1} != 0, and sigma[w] is the sum of sigma over exactly those bits;
//     the backward sweep is delta[v] = sum over row(v) & L_{k} of sigma[v] * (1 + delta[w]) / sigma[w].
//     Each lane owns the nodes lane, lane+32, ... and walks ITS unvisited ones, so a level costs
//     (unvisited / 32) row scans restricted to the non-empty quads of the previous level set;
//   * sources are independent: warp i takes sources i, i+W, ...; betweenness partials stay in
//     registers (one per owned node) until the end; closeness falls out of the same search;
//   * pagerank is a CTA-wide CSR mat-vec per iteration (G lanes per row), clustering is
//     popcount(row_i & row_j) over the bit-matrix (the first version expanded N x M edges).
// The first version (one warp per env, N serial sources, CSR expansion with shared fp64 atomics:
// 190 us/env at TSP N=200 dense, 73 us/env at N=500) is kept as features_warp_kernel for N > 1024.
// Sums are reassociated relative to networkx (sigma sums are exact while path counts stay below 2^53; delta
// and pagerank differ by fp64 rounding, ~1e-15 relative => within 1 float32 ulp; the other columns are exact).
#include "ge_common.cuh"

using namespace ge;

extern "C" int ge_set_error(int code, const char *fmt, ...);
int ge_grant_smem(const void *kernel, size_t smem);  // ge_api.cu

namespace {

// ============================================================================================
// CTA per env
// ============================================================================================
constexpr uint16_t UNVIS = 0xffffu;

__host__ __device__ inline int feat_nwp(int NW) {  // row stride in words: whole quads, odd quad count
    int q = (NW + 3) >> 2;
    if (!(q & 1)) q += 1;
    return q << 2;
}
__host__ __device__ inline int feat_warp_bytes(int N, int NWP) {  // sigma[N] f64 | delta[N] f64 | lv[NWP] u32 | D[N] u16
    return (16 * N + 4 * NWP + 2 * N + 15) & ~15;
}

__device__ __forceinline__ double block_sum(double v, double *red, int W) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(GE_FULL, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = 0.0;
    for (int w = 0; w < W; ++w) t += red[w];
    __syncthreads();
    return t;
}

// sum of tab[u] over the neighbours u of row [lo, hi) whose level is `want`: four neighbours per trip so that the
// level and value loads of a trip are independent (the plain loop was a chain of three dependent shared-memory loads
// per neighbour at four warps per scheduler)
__device__ __forceinline__ double csr_gather(const uint16_t *col16, const uint16_t *D, const double *tab, int lo, int hi, uint16_t want) {
    double a0 = 0.0, a1 = 0.0;
    int e = lo;
    for (; e + 4 <= hi; e += 4) {
        const int u0 = col16[e], u1 = col16[e + 1], u2 = col16[e + 2], u3 = col16[e + 3];
        const bool p0 = D[u0] == want, p1 = D[u1] == want, p2 = D[u2] == want, p3 = D[u3] == want;
        const double s0 = p0 ? tab[u0] : 0.0, s1 = p1 ? tab[u1] : 0.0, s2 = p2 ? tab[u2] : 0.0, s3 = p3 ? tab[u3] : 0.0;
        a0 += s0 + s2;
        a1 += s1 + s3;
    }
    for (; e < hi; ++e) {
        const int u = col16[e];
        if (D[u] == want) a0 += tab[u];
    }
    return a0 + a1;
}

// sum of tab[base + i] over the set bits i of x
__device__ __forceinline__ void gather_add(const double *tab, int base, uint32_t x, double &acc) {
    while (x) {
        acc += tab[base + __ffs(x) - 1];
        x &= x - 1;
    }
}

// CSRP: sparse graphs (average degree <= 32, M < 65536) gather a node's predecessors / successors by walking its CSR
// row from a 16-bit shared-memory copy and testing the neighbour's level -- ~6 instructions per neighbour with all
// lanes busy -- instead of looping over the set bits of (row & level set) word by word, where a warp-divergent loop per
// 32-bit word served one or two lanes at a time (ncu r02 first capture at N=500: 55 % of all instructions, 15 of 32
// threads active).  The bit-matrix test stays as the cheap "does this node join the level at all" filter.  Dense graphs
// keep the word loops (a complete graph has one level).
template <int NWMAX, bool CSRP>
__global__ void __launch_bounds__(512, 1) features_cta_kernel(ge_batch d, int NWP, int warp_bytes, int G, int csr_bytes) {
    extern __shared__ __align__(16) uint32_t smem[];
    const int b = blockIdx.x;
    const int N = d.N, NW = d.NW;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, W = blockDim.x >> 5, tid = threadIdx.x, NT = blockDim.x;
    const int QN = NWP >> 2;
    uint32_t *mat = smem;
    uint16_t *rp16 = reinterpret_cast<uint16_t *>(mat + (size_t)N * NWP);   // [N + 1] row offsets, [M] neighbour ids (CSRP)
    uint16_t *col16 = rp16 + N + 1;
    char *wbase = reinterpret_cast<char *>(mat + (size_t)N * NWP) + csr_bytes;
    double *sigma = reinterpret_cast<double *>(wbase + (size_t)warp * warp_bytes);
    double *delta = sigma + N;
    uint32_t *lv = reinterpret_cast<uint32_t *>(delta + N);
    uint16_t *D = reinterpret_cast<uint16_t *>(lv + NWP);
    const int32_t *rp = d.row_ptr + (size_t)b * d.RP;
    const int32_t *col = d.col + (size_t)b * d.MP;
    float *out = d.features + (size_t)b * N * 5;

    // ---------------- adjacency bit-matrix from the CSR
    for (int i = tid; i < N * NWP; i += NT) mat[i] = 0;
    for (int i = lane; i < NWP; i += 32) lv[i] = 0;
    __syncthreads();
    for (int u = warp; u < N; u += W) {
        const int lo = rp[u], hi = rp[u + 1];
        for (int e = lo + lane; e < hi; e += 32) {
            const int c = col[e];
            atomicOr(&mat[(size_t)u * NWP + (c >> 5)], 1u << (c & 31));
            if (CSRP) col16[e] = (uint16_t)c;
        }
    }
    if (CSRP)
        for (int i = tid; i <= N; i += NT) rp16[i] = (uint16_t)rp[i];
    __syncthreads();

    // ---------------- betweenness + closeness: one search per source, one warp per source
    double bt[NWMAX];
#pragma unroll
    for (int j = 0; j < NWMAX; ++j) bt[j] = 0.0;

    for (int s = warp; s < N; s += W) {
        uint32_t unv = 0;  // bit j: node lane + 32 j exists and is unvisited
        for (int j = 0; j < NW; ++j) {
            const int v = lane + (j << 5);
            if (v < N) { D[v] = UNVIS; unv |= 1u << j; }
        }
        if (lane < NW) lv[lane] = (lane == (s >> 5)) ? (1u << (s & 31)) : 0u;
        __syncwarp();
        if (lane == (s & 31)) { sigma[s] = 1.0; delta[s] = 0.0; D[s] = 0; unv &= ~(1u << (s >> 5)); }
        uint32_t quads = 1u << (s >> 7);  // non-empty 128-bit groups of the previous level set
        __syncwarp();
        int level = 0, reached = 1;
        long long totsp = 0;
        {   // level 1 is N(s) itself, every node with exactly one shortest path: no scan of the ~N unvisited nodes for it
            const uint32_t *rs = mat + (size_t)s * NWP;
            uint32_t newbits = 0;
            for (int j = 0; j < NW; ++j)
                if ((rs[j] >> lane) & 1u) {
                    const int v = lane + (j << 5);
                    sigma[v] = 1.0; delta[v] = 0.0; D[v] = 1;
                    newbits |= 1u << j;
                }
            const uint32_t myword = lane < NW ? rs[lane] : 0u;
            const uint32_t nz = __ballot_sync(GE_FULL, myword != 0u);
            if (nz) {
                unv &= ~newbits;
                if (lane < NW) lv[lane] = myword;
                quads = 0;
#pragma unroll
                for (int qi = 0; qi < 8; ++qi)
                    if ((nz >> (4 * qi)) & 0xfu) quads |= 1u << qi;
                const int cnt = __reduce_add_sync(GE_FULL, __popc(myword));
                level = 1;
                reached += cnt;
                totsp += cnt;
            }
            __syncwarp();
        }
        while (reached < N) {  // forward sweep (_single_source_shortest_path_basic), pull form
            ++level;
            uint32_t newbits = 0, rem = unv;
            while (rem) {
                const int j = __ffs(rem) - 1;
                rem &= rem - 1;
                const int v = lane + (j << 5);
                const uint4 *row = reinterpret_cast<const uint4 *>(mat + (size_t)v * NWP);
                double sg = 0.0;
                uint32_t q = quads;
                if (CSRP) {
                    uint32_t any = 0;
                    while (q) {
                        const int qi = __ffs(q) - 1;
                        q &= q - 1;
                        const uint4 r = row[qi];
                        const uint4 l = reinterpret_cast<const uint4 *>(lv)[qi];
                        any |= (r.x & l.x) | (r.y & l.y) | (r.z & l.z) | (r.w & l.w);
                    }
                    if (any) sg = csr_gather(col16, D, sigma, rp16[v], rp16[v + 1], (uint16_t)(level - 1));
                } else
                while (q) {
                    const int qi = __ffs(q) - 1;
                    q &= q - 1;
                    const uint4 r = row[qi];
                    const uint4 l = reinterpret_cast<const uint4 *>(lv)[qi];
                    const int base = qi << 7;
                    gather_add(sigma, base, r.x & l.x, sg);
                    gather_add(sigma, base + 32, r.y & l.y, sg);
                    gather_add(sigma, base + 64, r.z & l.z, sg);
                    gather_add(sigma, base + 96, r.w & l.w, sg);
                }
                if (sg > 0.0) { sigma[v] = sg; delta[v] = 0.0; D[v] = (uint16_t)level; newbits |= 1u << j; }
            }
            __syncwarp();
            unv &= ~newbits;
            uint32_t myword = 0;  // lane j keeps word j of the new level set
            for (int j = 0; j < NW; ++j) {
                const uint32_t wd = __ballot_sync(GE_FULL, (newbits >> j) & 1u);
                if (lane == j) myword = wd;
            }
            const uint32_t nz = __ballot_sync(GE_FULL, myword != 0u);
            if (!nz) { --level; break; }
            if (lane < NW) lv[lane] = myword;
            quads = 0;
#pragma unroll
            for (int qi = 0; qi < 8; ++qi)
                if ((nz >> (4 * qi)) & 0xfu) quads |= 1u << qi;
            const int cnt = __reduce_add_sync(GE_FULL, __popc(myword));
            reached += cnt;
            totsp += (long long)cnt * level;
            __syncwarp();
        }
        if (lane == 0) {  // closeness: ((r-1)/totsp) * ((r-1)/(N-1)), 0 when totsp == 0
            double cc = 0.0;
            if (totsp > 0 && N > 1) {
                cc = ((double)reached - 1.0) / (double)totsp;
                cc *= ((double)reached - 1.0) / (double)(N - 1);
            }
            out[s * 5 + 2] = (float)cc;
        }
        // backward sweep (_accumulate_basic), pull form.  coeff[w] = (1 + delta[w]) / sigma[w] overwrites sigma[w]
        // (sigma of level k is dead once its coefficients exist); delta[v] of level k-1 is the sum over its
        // successors.  Level 1 only feeds delta[source], which betweenness never uses.
        for (int k = level; k >= 2; --k) {
            uint32_t myword = 0, prev = 0;
            for (int j = 0; j < NW; ++j) {
                const int v = lane + (j << 5);
                const int dv = v < N ? (int)D[v] : -1;
                const bool in = dv == k;
                if (in) sigma[v] = (1.0 + delta[v]) / sigma[v];
                if (dv == k - 1) prev |= 1u << j;
                if (!CSRP) {
                    const uint32_t wd = __ballot_sync(GE_FULL, in);
                    if (lane == j) myword = wd;
                }
            }
            uint32_t qd = 0;
            if (!CSRP) {
                const uint32_t nz = __ballot_sync(GE_FULL, myword != 0u);
                if (lane < NW) lv[lane] = myword;
#pragma unroll
                for (int qi = 0; qi < 8; ++qi)
                    if ((nz >> (4 * qi)) & 0xfu) qd |= 1u << qi;
            }
            __syncwarp();
            while (prev) {
                const int j = __ffs(prev) - 1;
                prev &= prev - 1;
                const int v = lane + (j << 5);
                const uint4 *row = reinterpret_cast<const uint4 *>(mat + (size_t)v * NWP);
                double acc = 0.0;
                if (CSRP) acc = csr_gather(col16, D, sigma, rp16[v], rp16[v + 1], (uint16_t)k);   // coefficients of the successors
                uint32_t q = CSRP ? 0u : qd;
                while (q) {
                    const int qi = __ffs(q) - 1;
                    q &= q - 1;
                    const uint4 r = row[qi];
                    const uint4 l = reinterpret_cast<const uint4 *>(lv)[qi];
                    const int base = qi << 7;
                    gather_add(sigma, base, r.x & l.x, acc);
                    gather_add(sigma, base + 32, r.y & l.y, acc);
                    gather_add(sigma, base + 64, r.z & l.z, acc);
                    gather_add(sigma, base + 96, r.w & l.w, acc);
                }
                delta[v] = sigma[v] * acc;
            }
            __syncwarp();
        }
#pragma unroll
        for (int j = 0; j < NWMAX; ++j) {
            const int v = lane + (j << 5);
            if (j < NW && v < N && v != s && D[v] != UNVIS) bt[j] += delta[v];
        }
        __syncwarp();
    }
    // betweenness: per-warp partials -> sum; degree column
#pragma unroll
    for (int j = 0; j < NWMAX; ++j) {
        const int v = lane + (j << 5);
        if (j < NW && v < N) sigma[v] = bt[j];
    }
    __syncthreads();
    {
        const double scale = (N - 1 >= 2) ? 1.0 / ((double)(N - 1) * (double)(N - 2)) : 1.0;  // _rescale, directed, normalized
        for (int v = tid; v < N; v += NT) {
            double t = 0.0;
            for (int w = 0; w < W; ++w) t += reinterpret_cast<const double *>(wbase + (size_t)w * warp_bytes)[v];
            out[v * 5 + 1] = (float)(t * scale);
            out[v * 5 + 0] = (float)(2 * (rp[v + 1] - rp[v]));
        }
    }
    __syncthreads();

    // ---------------- pagerank (power iteration, scipy formulation); x / y / invS / red overlay the search scratch
    {
        double *x = reinterpret_cast<double *>(wbase), *y = x + N, *invS = y + N, *red = invS + N;
        const bool weighted = (d.flags & GE_FLAG_WEIGHTED_PR) && d.w64;
        const double *w64 = d.w64 ? d.w64 + (size_t)b * d.MP : nullptr;
        const double p = 1.0 / (double)N, alpha = 0.85;
        const int grp = tid / G, gl = tid % G, ngrp = NT / G;
        int dangling = 0;
        for (int v0 = 0; v0 < N; v0 += ngrp) {  // warp-uniform trip count: the group reductions below use the full mask
            const int v = v0 + grp;
            const bool live = v < N;
            double S = 0.0;
            if (live)
                for (int e = rp[v] + gl; e < rp[v + 1]; e += G) S += weighted ? w64[e] : 1.0;
            for (int o = G >> 1; o > 0; o >>= 1) S += __shfl_xor_sync(GE_FULL, S, o);
            if (live && gl == 0) { invS[v] = S != 0.0 ? 1.0 / S : 0.0; x[v] = p; }
            if (live && S == 0.0) dangling = 1;
        }
        dangling = __syncthreads_or(dangling);
        for (int it = 0; it < 100; ++it) {
            double dsum = 0.0;
            if (dangling) {
                for (int v = tid; v < N; v += NT)
                    if (invS[v] == 0.0) dsum += x[v];
                dsum = block_sum(dsum, red, W);
            }
            double err = 0.0;
            for (int v0 = 0; v0 < N; v0 += ngrp) {
                const int v = v0 + grp;
                const bool live = v < N;
                double acc = 0.0;  // (x @ A)[v] = sum_u x[u] * (invS[u] * w(u,v)); symmetric => in-neighbours = row v
                if (live)
                    for (int e = rp[v] + gl; e < rp[v + 1]; e += G) {
                        const int u = col[e];
                        const double a = invS[u] * (weighted ? w64[e] : 1.0);
                        acc += a * x[u];
                    }
                for (int o = G >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(GE_FULL, acc, o);
                if (live && gl == 0) {
                    const double nx = alpha * (acc + dsum * p) + (1.0 - alpha) * p;
                    err += fabs(nx - x[v]);
                    y[v] = nx;
                }
            }
            err = block_sum(err, red, W);
            double *t = x; x = y; y = t;
            if (err < (double)N * 1.0e-6) break;
        }
        for (int v = tid; v < N; v += NT) out[v * 5 + 3] = (float)x[v];
    }

    // ---------------- clustering: S_i = sum_{j in N(i)} |N(i) & N(j)|, c = S / (d (d-1)); the matrix is still intact
    for (int i = warp; i < N; i += W) {
        const int lo = rp[i], hi = rp[i + 1];
        const uint4 *ri = reinterpret_cast<const uint4 *>(mat + (size_t)i * NWP);
        int cnt = 0;
        for (int e = lo + lane; e < hi; e += 32) {
            const uint4 *rj = reinterpret_cast<const uint4 *>(mat + (size_t)col[e] * NWP);
            for (int q = 0; q < QN; ++q) {
                const uint4 a = ri[q], c = rj[q];
                cnt += __popc(a.x & c.x) + __popc(a.y & c.y) + __popc(a.z & c.z) + __popc(a.w & c.w);
            }
        }
        cnt = __reduce_add_sync(GE_FULL, cnt);
        if (lane == 0) {
            const long long dg = hi - lo;
            const long long t = 8ll * cnt, dt = 2 * dg, db = dg;
            out[i * 5 + 4] = (t == 0) ? 0.f : (float)((double)t / (double)((dt * (dt - 1) - 2 * db) * 2));
        }
    }
}

// ============================================================================================
// One warp per env (round 1), kept for N > 1024 where the bit-matrix does not fit one CTA's shared memory
// ============================================================================================
struct FScr {
    double *sigma, *delta, *bt;  // [N] each
    int *D;                      // [N]
    uint32_t *f0, *f1, *lvl;     // [NW] each
};

__host__ __device__ inline int feat_words(int N, int NW) { return ((6 * N + N + 3 * NW) + 3) & ~3; }

__device__ inline FScr fcarve(uint32_t *base, int N, int NW) {
    FScr s;
    s.sigma = reinterpret_cast<double *>(base);
    s.delta = s.sigma + N;
    s.bt = s.delta + N;
    s.D = reinterpret_cast<int *>(s.bt + N);
    s.f0 = reinterpret_cast<uint32_t *>(s.D + N);
    s.f1 = s.f0 + NW;
    s.lvl = s.f1 + NW;
    return s;
}

__global__ void __launch_bounds__(GE_WPB * 32) features_warp_kernel(ge_batch d, int words_per_warp, int wpb) {
    extern __shared__ __align__(16) uint32_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * wpb + warp;
    if (b >= d.B) return;
    const int N = d.N, NW = d.NW;
    FScr s = fcarve(smem + (size_t)warp * words_per_warp, N, NW);
    const int32_t *rp = d.row_ptr + (size_t)b * d.RP;
    const int32_t *col = d.col + (size_t)b * d.MP;
    float *out = d.features + (size_t)b * N * 5;

    for (int v = lane; v < N; v += 32) s.bt[v] = 0.0;
    __syncwarp();

    for (int src = 0; src < N; ++src) {
        for (int v = lane; v < N; v += 32) { s.D[v] = -1; s.sigma[v] = 0.0; s.delta[v] = 0.0; }
        for (int w = lane; w < NW; w += 32) { s.f0[w] = 0; s.f1[w] = 0; }
        __syncwarp();
        if (lane == 0) { s.D[src] = 0; s.sigma[src] = 1.0; s.f0[src >> 5] = 1u << (src & 31); }
        __syncwarp();
        int level = 0;
        long long totsp = 0;
        int reached = 1;
        for (;;) {
            double sg = 0.0;
            expand_set(
                rp, s.f0, NW, lane, [&](int u) { sg = u >= 0 ? s.sigma[u] : 0.0; },
                [&](int owner, int e, bool active) {
                    double su = __shfl_sync(GE_FULL, sg, owner);
                    if (active) {
                        int w = col[e];
                        int old = atomicCAS(&s.D[w], -1, level + 1);
                        if (old == -1 || old == level + 1) {
                            atomicAdd(&s.sigma[w], su);
                            if (old == -1) atomicOr(&s.f1[w >> 5], 1u << (w & 31));
                        }
                    }
                });
            __syncwarp();
            int cnt = 0;
            uint32_t any = 0;
            for (int w = lane; w < NW; w += 32) { uint32_t n = s.f1[w]; s.f0[w] = n; s.f1[w] = 0; any |= n; cnt += __popc(n); }
            cnt = __reduce_add_sync(GE_FULL, cnt);
            __syncwarp();
            if (!__any_sync(GE_FULL, any != 0)) break;
            ++level;
            reached += cnt;
            totsp += (long long)cnt * level;
        }
        if (lane == 0) {
            double cc = 0.0;
            if (totsp > 0 && N > 1) {
                cc = ((double)reached - 1.0) / (double)totsp;
                cc *= ((double)reached - 1.0) / (double)(N - 1);
            }
            out[src * 5 + 2] = (float)cc;
        }
        for (int L = level; L >= 1; --L) {
            for (int w = lane; w < NW; w += 32) {
                uint32_t bits = 0;
                for (int j = 0; j < 32; ++j) {
                    int v = (w << 5) + j;
                    if (v < N && s.D[v] == L) bits |= 1u << j;
                }
                s.lvl[w] = bits;
            }
            __syncwarp();
            double coeff = 0.0;
            expand_set(
                rp, s.lvl, NW, lane,
                [&](int w) {
                    if (w >= 0) {
                        coeff = (1.0 + s.delta[w]) / s.sigma[w];
                        s.bt[w] += s.delta[w];
                    } else coeff = 0.0;
                },
                [&](int owner, int e, bool active) {
                    double c = __shfl_sync(GE_FULL, coeff, owner);
                    if (active) {
                        int v = col[e];
                        if (s.D[v] == L - 1) atomicAdd(&s.delta[v], s.sigma[v] * c);
                    }
                });
            __syncwarp();
        }
    }
    {
        double scale = (N - 1 >= 2) ? 1.0 / ((double)(N - 1) * (double)(N - 2)) : 1.0;
        for (int v = lane; v < N; v += 32) {
            out[v * 5 + 1] = (float)(s.bt[v] * scale);
            out[v * 5 + 0] = (float)(2 * (rp[v + 1] - rp[v]));
        }
    }
    __syncwarp();
    {
        double *x = s.sigma, *y = s.delta, *invS = s.bt;
        const bool weighted = (d.flags & GE_FLAG_WEIGHTED_PR) && d.w64;
        const double *w64 = d.w64 ? d.w64 + (size_t)b * d.MP : nullptr;
        const double p = 1.0 / (double)N, alpha = 0.85;
        for (int v = lane; v < N; v += 32) {
            double S = 0.0;
            for (int e = rp[v]; e < rp[v + 1]; ++e) S += weighted ? w64[e] : 1.0;
            invS[v] = S != 0.0 ? 1.0 / S : 0.0;
            x[v] = p;
        }
        __syncwarp();
        for (int it = 0; it < 100; ++it) {
            double dsum = 0.0;
            for (int v = lane; v < N; v += 32) if (invS[v] == 0.0) dsum += x[v];
            for (int o = 16; o > 0; o >>= 1) dsum += __shfl_xor_sync(GE_FULL, dsum, o);
            double err = 0.0;
            for (int v = lane; v < N; v += 32) {
                double acc = 0.0;
                for (int e = rp[v]; e < rp[v + 1]; ++e) {
                    int u = col[e];
                    double a = invS[u] * (weighted ? w64[e] : 1.0);
                    acc += a * x[u];
                }
                double nx = alpha * (acc + dsum * p) + (1.0 - alpha) * p;
                err += fabs(nx - x[v]);
                y[v] = nx;
            }
            for (int o = 16; o > 0; o >>= 1) err += __shfl_xor_sync(GE_FULL, err, o);
            __syncwarp();
            double *t = x; x = y; y = t;
            if (err < (double)N * 1.0e-6) break;
        }
        for (int v = lane; v < N; v += 32) out[v * 5 + 3] = (float)x[v];
        __syncwarp();
    }
    for (int i = 0; i < N; ++i) {
        int lo = rp[i], hi = rp[i + 1];
        for (int w = lane; w < NW; w += 32) s.lvl[w] = 0;
        __syncwarp();
        for (int e = lo + lane; e < hi; e += 32) { int j = col[e]; atomicOr(&s.lvl[j >> 5], 1u << (j & 31)); }
        __syncwarp();
        long long cnt = 0;
        expand_set(
            rp, s.lvl, NW, lane, [](int) {},
            [&](int, int e, bool active) {
                if (active) cnt += tbit(s.lvl, col[e]);
            });
        for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(GE_FULL, cnt, o);
        if (lane == 0) {
            long long dg = hi - lo;
            long long t = 8 * cnt, dt = 2 * dg, db = dg;
            out[i * 5 + 4] = (t == 0) ? 0.f : (float)((double)t / (double)((dt * (dt - 1) - 2 * db) * 2));
        }
        __syncwarp();
    }
}

static int launch_warp_family(const ge_batch *d, cudaStream_t st) {
    int wpw = feat_words(d->N, d->NW);
    size_t per_warp = (size_t)wpw * sizeof(uint32_t);
    int wpb = (int)((200 * 1024) / per_warp);
    if (wpb < 1) return ge_set_error(GE_ERR_UNSUPPORTED, "ge_features: N=%d too large for shared scratch", d->N);
    if (wpb > GE_WPB) wpb = GE_WPB;
    size_t smem = per_warp * wpb;
    int rc = ge_grant_smem((const void *)features_warp_kernel, smem);
    if (rc) return rc;
    features_warp_kernel<<<(d->B + wpb - 1) / wpb, wpb * 32, smem, st>>>(*d, wpw, wpb);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return ge_set_error(GE_ERR_CUDA, "features_warp_kernel launch: %s", cudaGetErrorString(e));
    return GE_OK;
}

}  // namespace

extern "C" int ge_features(const ge_batch *d, void *stream) {
    GE_NVTX("ge_features");
    if (!d || !d->features) return ge_set_error(GE_ERR_ARG, "ge_features: features buffer is null");
    cudaStream_t st = (cudaStream_t)stream;
    const int N = d->N, NW = d->NW;
    if (N > 1024 || (d->flags & GE_FLAG_FORCE_WARP)) return launch_warp_family(d, st);
    const int NWP = feat_nwp(NW), wb = feat_warp_bytes(N, NWP);
    const size_t mat_bytes = (size_t)N * NWP * 4;
    const size_t budget = 227 * 1024;
    const int avg = N > 0 ? d->M / N : 1;
    // sparse graphs: 16-bit CSR copy in shared memory for the predecessor / successor gathers
    bool csrp = avg <= 32 && d->M < 65536;
    size_t csr_bytes = csrp ? (((size_t)2 * (N + 1) + (size_t)2 * d->M + 15) & ~(size_t)15) : 0;
    if (csrp && mat_bytes + csr_bytes + 4 * (size_t)wb + 128 > budget) { csrp = false; csr_bytes = 0; }
    int W = (N + 7) / 8;                         // sources per warp >= 8 where there are that many
    if (W < 2) W = 2;                            // the pagerank overlay needs two warps' scratch
    if (W > 16) W = 16;
    while (W > 2 && mat_bytes + csr_bytes + (size_t)W * wb + 8 * 16 > budget) --W;
    const size_t need = (size_t)W * wb + 8 * 16;
    const size_t overlay = 3 * (size_t)N * 8 + 8 * 16;           // x, y, invS, red[W]
    size_t smem = mat_bytes + csr_bytes + (need > overlay ? need : overlay);
    if (smem > budget) return launch_warp_family(d, st);
    int G = 1;
    while (G < 32 && 2 * G <= avg / 2) G <<= 1;                   // lanes per CSR row in the pagerank mat-vec
    const void *kernel;
    if (csrp) {
        if (NW <= 2) kernel = (const void *)features_cta_kernel<2, true>;
        else if (NW <= 4) kernel = (const void *)features_cta_kernel<4, true>;
        else if (NW <= 8) kernel = (const void *)features_cta_kernel<8, true>;
        else if (NW <= 16) kernel = (const void *)features_cta_kernel<16, true>;
        else kernel = (const void *)features_cta_kernel<32, true>;
    } else {
        if (NW <= 2) kernel = (const void *)features_cta_kernel<2, false>;
        else if (NW <= 4) kernel = (const void *)features_cta_kernel<4, false>;
        else if (NW <= 8) kernel = (const void *)features_cta_kernel<8, false>;
        else if (NW <= 16) kernel = (const void *)features_cta_kernel<16, false>;
        else kernel = (const void *)features_cta_kernel<32, false>;
    }
    int rc = ge_grant_smem(kernel, smem);
    if (rc) return rc;
    ge_batch dd = *d;
    int nwp = NWP, wbytes = wb, g = G, cb = (int)csr_bytes;
    void *args[] = {&dd, &nwp, &wbytes, &g, &cb};
    cudaError_t e = cudaLaunchKernel(kernel, dim3((unsigned)d->B), dim3((unsigned)(W * 32)), args, smem, st);
    if (e != cudaSuccess) return ge_set_error(GE_ERR_CUDA, "features_cta_kernel launch: %s", cudaGetErrorString(e));
    return GE_OK;
}
