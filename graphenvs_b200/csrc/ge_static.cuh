// ge_static.cuh -- the static per-env arrays of an instance and the warp copy of one env's instance between batches.
//
// Shared by ge_pool_refill (ge_pool.cu: bank env b -> live env b) and ge_gather_instances (ge_state.cu: src env s -> dst
// env b).  "Static" = everything an instance carries that no step writes: the graph store, the derived arrays, the
// instance parameters, features, heuristics and the reset-time mask.  The dynamic state has its own list (ge_state.cu).
#pragma once
#include <cstddef>

#include "ge_common.cuh"

extern "C" int ge_set_error(int code, const char *fmt, ...);

namespace ge {

constexpr int STATIC_MAX_SRC = 8, STATIC_MAX_ARRAYS = 24;

struct StaticArr {
    const char *src[STATIC_MAX_SRC];  // one base per source descriptor
    char *dst;
    uint32_t bytes;  // per env
    uint32_t tiled;  // adjacency tiles of 32 envs (ge_common.cuh:adj_tiled): element = NW words, N rows at a pitch of 32 elements
};
struct StaticTab {
    int n;
    StaticArr a[STATIC_MAX_ARRAYS];
};

// Every static array `d` carries, with its sources in srcs[0 .. n_src): GE_ERR_ARG when a source lacks one of them.
inline int static_table(const ge_batch &d, const ge_batch *srcs, int n_src, StaticTab &tab, const char *who) {
    tab.n = 0;
    auto add = [&](const void *dst, size_t offset_in_struct, size_t bytes, bool tiled) -> int {
        if (!dst || bytes == 0) return GE_OK;  // the destination does not carry this array
        if (tab.n == STATIC_MAX_ARRAYS) return ge_set_error(GE_ERR_ARG, "%s: array table full", who);
        StaticArr &A = tab.a[tab.n];
        for (int k = 0; k < n_src; ++k) {
            const void *src = *reinterpret_cast<void *const *>(reinterpret_cast<const char *>(&srcs[k]) + offset_in_struct);
            if (!src) return ge_set_error(GE_ERR_ARG, "%s: source %d lacks an array the destination has (struct offset %zu)", who, k, offset_in_struct);
            A.src[k] = reinterpret_cast<const char *>(src);
        }
        A.dst = reinterpret_cast<char *>(const_cast<void *>(dst));
        A.bytes = (uint32_t)bytes;
        A.tiled = tiled ? 1u : 0u;
        ++tab.n;
        return GE_OK;
    };
    int rc = GE_OK;
#define STATIC_ADD(field, bytes) if (rc == GE_OK) rc = add(d.field, offsetof(ge_batch, field), (size_t)(bytes), false)
    STATIC_ADD(row_ptr, d.RP * 4); STATIC_ADD(col, d.MP * 4); STATIC_ADD(w32, d.MP * 4); STATIC_ADD(w64, d.MP * 8);
    if (rc == GE_OK) rc = add(d.adj_bits, offsetof(ge_batch, adj_bits), adj_tiled(d) ? 4 : (size_t)d.ADJS * 4, adj_tiled(d));
    STATIC_ADD(rev, d.MP * 4); STATIC_ADD(esrc, d.MP * 4); STATIC_ADD(wsort, d.MP * 8); STATIC_ADD(wcode, d.MP); STATIC_ADD(dc_edges, d.MP * 4); STATIC_ADD(dc_rows, (size_t)d.N * 128); STATIC_ADD(wmin, 8);
    STATIC_ADD(wmat, (size_t)d.N * d.N * 8); STATIC_ADD(src, 4); STATIC_ADD(dest, 4); STATIC_ADD(target_bits, d.NW * 4);
    STATIC_ADD(node_cost, d.N * 4); STATIC_ADD(node_xy, d.N * 8); STATIC_ADD(max_dist32, 4); STATIC_ADD(targets, d.n_targets * 4);
    STATIC_ADD(in_range, (size_t)d.n_targets * d.NW * 4); STATIC_ADD(heuristic, 8); STATIC_ADD(heuristic_alt, 8);
    STATIC_ADD(features, d.N * 20); STATIC_ADD(mask0_bits, d.AW * 4);
#undef STATIC_ADD
    return rc;
}

// Bytes array A spans in a batch of B envs (for overlap checks).
inline size_t static_span(const ge_batch &d, const StaticArr &A, int B) {
    if (A.tiled) return (size_t)((B + 31) / 32) * d.N * 32 * d.NW * 4;
    return (size_t)B * A.bytes;
}

// One warp copies source k's env `bs` over the destination's env `bt`, array by array.  The tiled adjacency layout is
// addressed per env on both sides, so bs and bt may sit at different positions of their tiles.
__device__ inline void copy_static_env(const ge_batch &d, const StaticTab &tab, int k, size_t bs, size_t bt, int lane) {
    for (int i = 0; i < tab.n; ++i) {
        const StaticArr &A = tab.a[i];
        if (A.tiled) {
            const size_t el = (size_t)d.NW * 4, tile = (size_t)d.N * 32 * el;
            const char *s = A.src[k] + (bs >> 5) * tile + (bs & 31) * el;
            char *t = A.dst + (bt >> 5) * tile + (bt & 31) * el;
            for (int r = lane; r < d.N; r += 32) {
                if (d.NW == 1) *reinterpret_cast<uint32_t *>(t + (size_t)r * 32 * el) = *reinterpret_cast<const uint32_t *>(s + (size_t)r * 32 * el);
                else *reinterpret_cast<uint2 *>(t + (size_t)r * 32 * el) = *reinterpret_cast<const uint2 *>(s + (size_t)r * 32 * el);
            }
            continue;
        }
        const char *s = A.src[k] + bs * A.bytes;
        char *t = A.dst + bt * A.bytes;
        if ((A.bytes & 15u) == 0) {
            const uint4 *s4 = reinterpret_cast<const uint4 *>(s);
            uint4 *t4 = reinterpret_cast<uint4 *>(t);
            for (uint32_t j = lane; j < (A.bytes >> 4); j += 32) t4[j] = s4[j];
        } else {
            const uint32_t *s1 = reinterpret_cast<const uint32_t *>(s);
            uint32_t *t1 = reinterpret_cast<uint32_t *>(t);
            for (uint32_t j = lane; j < (A.bytes >> 2); j += 32) t1[j] = s1[j];
        }
    }
}

}  // namespace ge
