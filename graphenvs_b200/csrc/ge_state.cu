// ge_state.cu -- per-env state records (ge_state_save / ge_state_load) and instance replication (ge_gather_instances):
// the branching primitives of search decoders (multi-start, beam search, lookahead), include/graphenvs_b200.h.
//
// A record is one env's state, laid out by build_layout() from the three lists below.  Sections of at most SMALL_MAX bytes
// per env form the record's HEADER (natural alignment, rounded up to 16 bytes); larger sections follow it in the BODY, each
// at a 16-byte offset.  One block handles a tile of up to TILE envs (load) or records (save):
//   - the headers of the tile's records move between global memory and shared memory as 16-byte vectors (coalesced within
//     and across records), and the header sections move between shared memory and the SoA arrays one ELEMENT per thread,
//     consecutive threads on consecutive elements: a 4-byte `head` or a 1-byte `done` costs a few bytes of a coalesced
//     access, not a warp per env;
//   - every body section (Multicast edge_bits / dist32 / bestkey / mask_bits: hundreds of bytes per env) is copied by one
//     warp per env with the widest vector both sides allow.
// The packed mask's byte view is rebuilt from the loaded mask in the same launch.  Nothing here touches a
// static array, so a load may precede a GE_FLAG_PDL step.
#include "ge_static.cuh"

using namespace ge;

namespace {

constexpr int ST_MAX = 14;           // state arrays in the three lists
constexpr uint32_t SMALL_MAX = 64;   // a section of at most this many bytes per env goes in the header
constexpr int TILE = 64, THREADS = 256, WARPS = THREADS / 32;
constexpr int SMEM_MAX = 32 * 1024;  // header tile in shared memory (TILE halves until it fits; no opt-in above 48 KB needed)

struct Sec {
    char *soa;         // device SoA array
    uint32_t esz, n;   // element bytes (1, 4 or 8), elements per env
    uint32_t cstride;  // 0: env-major [B, n]; else element j of env b sits at j * cstride + b (acc, [4, acc_stride])
    uint32_t off;      // byte offset in the record
    uint32_t vec;      // body sections: bytes per vector of the warp copy (4, 8 or 16)
    uint32_t what;     // GE_STATE_DYNAMIC / _CLOCK / _STATS
};
struct Layout {
    int n, n_head;        // sections [0, n_head) are the header, [n_head, n) the body
    int mask;             // index of the mask_bits section, or -1
    uint32_t head, bytes; // header bytes (multiple of 16), record bytes (multiple of 16)
    Sec s[ST_MAX];
};

inline uint32_t align_up(uint32_t x, uint32_t a) { return (x + a - 1) / a * a; }

// What counts as state.  The step outputs (reward, flags, solution_cost), obs_x and the byte mask are not state; every other
// array of ge_batch is static (ge_static.cuh).  The list order is the section order within the header and within the body.
void build_layout(const ge_batch &d, Layout &L) {
    struct Item { void *p; uint32_t esz, n, cstride, what; };
    const Item items[ST_MAX] = {
        // DYNAMIC: what ge_step reads and writes besides its outputs
        {d.head, 4, 1, 0, GE_STATE_DYNAMIC}, {d.node_bits, 4, (uint32_t)d.NW, 0, GE_STATE_DYNAMIC},
        {d.node_bits2, 4, (uint32_t)d.NW, 0, GE_STATE_DYNAMIC}, {d.edge_bits, 4, (uint32_t)d.MW, 0, GE_STATE_DYNAMIC},
        {d.dist32, 4, (uint32_t)d.N, 0, GE_STATE_DYNAMIC}, {d.bestkey, 8, (uint32_t)d.N, 0, GE_STATE_DYNAMIC},
        {d.cost, 8, 1, 0, GE_STATE_DYNAMIC}, {d.counters, 4, 4, 0, GE_STATE_DYNAMIC}, {d.done, 1, 1, 0, GE_STATE_DYNAMIC},
        {d.mask_bits, 4, (uint32_t)d.AW, 0, GE_STATE_DYNAMIC}, {d.mask_cnt, 4, 8, 0, GE_STATE_DYNAMIC},
        // CLOCK
        {d.env_steps, 4, 1, 0, GE_STATE_CLOCK},
        // STATS
        {d.acc, 8, 4, (uint32_t)d.acc_stride, GE_STATE_STATS}, {d.traj, 8, 1, 0, GE_STATE_STATS},
    };
    L.n = 0;
    L.mask = -1;
    uint32_t off = 0;
    for (int pass = 0; pass < 2; ++pass) {   // 0: header sections, 1: body sections
        if (pass == 1) { off = align_up(off, 16); L.head = off; L.n_head = L.n; }
        for (const Item &it : items) {
            const uint32_t bytes = it.esz * it.n;
            if (!it.p || bytes == 0 || (bytes > SMALL_MAX) != (pass == 1)) continue;
            Sec &S = L.s[L.n];
            off = align_up(off, pass ? 16u : it.esz);
            S.soa = reinterpret_cast<char *>(it.p);
            S.esz = it.esz; S.n = it.n; S.cstride = it.cstride; S.off = off; S.what = it.what;
            const uintptr_t a = reinterpret_cast<uintptr_t>(it.p) | bytes;   // alignment of every env's row on the SoA side
            S.vec = (a & 15u) == 0 ? 16u : (a & 7u) == 0 ? 8u : 4u;
            if (it.p == d.mask_bits) L.mask = L.n;
            off += bytes;
            ++L.n;
        }
    }
    L.bytes = align_up(off, 16);
}

// Tile size whose headers fit SMEM_MAX.
int tile_for(const Layout &L) {
    int te = TILE;
    while (te > 1 && (size_t)te * L.head > (size_t)SMEM_MAX) te >>= 1;
    return te;
}

__device__ __forceinline__ void copy_elem(char *t, const char *s, uint32_t esz) {
    if (esz == 8) *reinterpret_cast<uint2 *>(t) = *reinterpret_cast<const uint2 *>(s);
    else if (esz == 4) *reinterpret_cast<uint32_t *>(t) = *reinterpret_cast<const uint32_t *>(s);
    else *t = *s;
}

// Address of element k of a header section within a tile of te envs, and the env it belongs to.  Component-major sections
// (acc) enumerate component by component so that consecutive k are consecutive SoA addresses.
__device__ __forceinline__ void tile_elem(const Sec &S, uint32_t k, int te, int &e, uint32_t &j) {
    if (S.cstride) { j = k / te; e = (int)(k % te); }
    else { e = (int)(k / S.n); j = k % S.n; }
}
__device__ __forceinline__ size_t soa_index(const Sec &S, size_t b, uint32_t j) {
    return S.cstride ? (size_t)j * S.cstride + b : b * S.n + j;
}

template <typename T>
__device__ __forceinline__ void warp_copy_t(char *__restrict__ dst, const char *__restrict__ src, uint32_t n, int lane) {
    const T *s = reinterpret_cast<const T *>(src);
    T *t = reinterpret_cast<T *>(dst);
    uint32_t j = lane;
    for (; j + 96 < n; j += 128) {   // four vectors in flight per lane
        const T a = s[j], b = s[j + 32], c = s[j + 64], e = s[j + 96];
        t[j] = a; t[j + 32] = b; t[j + 64] = c; t[j + 96] = e;
    }
    for (; j < n; j += 32) t[j] = s[j];
}
__device__ __forceinline__ void warp_copy(char *dst, const char *src, uint32_t bytes, uint32_t vec, int lane) {
    if (vec == 16) warp_copy_t<uint4>(dst, src, bytes >> 4, lane);
    else if (vec == 8) warp_copy_t<uint2>(dst, src, bytes >> 3, lane);
    else warp_copy_t<uint32_t>(dst, src, bytes >> 2, lane);
}

// Record i <- env env_index[i] (i, when env_index is NULL); an env index outside [0, B) leaves record i untouched.
__global__ void __launch_bounds__(THREADS) state_save_kernel(ge_batch d, Layout L, int te_max, char *__restrict__ rec, int count,
                                                             const int32_t *__restrict__ env_index) {
    extern __shared__ uint4 sh4[];
    char *sh = reinterpret_cast<char *>(sh4);
    __shared__ int env[TILE];
    const int i0 = blockIdx.x * te_max, te = min(te_max, count - i0), tid = threadIdx.x;
    const uint32_t hv = L.head >> 4;
    for (int e = tid; e < te; e += THREADS) {
        const int b = env_index ? env_index[i0 + e] : i0 + e;
        env[e] = (b >= 0 && b < d.B) ? b : -1;
    }
    for (uint32_t c = tid; c < (uint32_t)te * hv; c += THREADS) sh4[c] = make_uint4(0, 0, 0, 0);   // padding bytes are zero
    __syncthreads();
    for (int s = 0; s < L.n_head; ++s) {
        const Sec &S = L.s[s];
        for (uint32_t k = tid; k < (uint32_t)te * S.n; k += THREADS) {
            int e; uint32_t j;
            tile_elem(S, k, te, e, j);
            if (env[e] < 0) continue;
            copy_elem(sh + (size_t)e * L.head + S.off + (size_t)j * S.esz, S.soa + soa_index(S, (size_t)env[e], j) * S.esz, S.esz);
        }
    }
    __syncthreads();
    for (uint32_t c = tid; c < (uint32_t)te * hv; c += THREADS) {
        const int e = (int)(c / hv);
        if (env[e] >= 0) reinterpret_cast<uint4 *>(rec + (size_t)(i0 + e) * L.bytes)[c % hv] = sh4[c];
    }
    const int warp = tid >> 5, lane = tid & 31;
    for (int e = warp; e < te; e += WARPS) {
        if (env[e] < 0) continue;
        char *r = rec + (size_t)(i0 + e) * L.bytes;
        for (int s = L.n_head; s < L.n; ++s) {
            const Sec &S = L.s[s];
            const uint32_t bytes = S.esz * S.n, end = s + 1 < L.n ? L.s[s + 1].off : L.bytes;
            warp_copy(r + S.off, S.soa + (size_t)env[e] * bytes, bytes, S.vec, lane);
            if (lane < (int)(end - S.off - bytes)) r[S.off + bytes + lane] = 0;   // alignment gap after the section (< 16 bytes)
        }
    }
}

// Env b <- record record_index[b] (b, when record_index is NULL); an index outside [0, n_records) leaves env b untouched.
// Only the sections in `what` are written.  mask_bytes: rebuild the byte view.
__global__ void __launch_bounds__(THREADS) state_load_kernel(ge_batch d, Layout L, int te_max, const char *__restrict__ rec, int n_records,
                                                             const int32_t *__restrict__ record_index, unsigned what, int mask_bytes) {
    extern __shared__ uint4 sh4[];
    const char *sh = reinterpret_cast<const char *>(sh4);
    __shared__ int rsel[TILE];
    const int b0 = blockIdx.x * te_max, te = min(te_max, d.B - b0), tid = threadIdx.x;
    const uint32_t hv = L.head >> 4;
    for (int e = tid; e < te; e += THREADS) {
        const int r = record_index ? record_index[b0 + e] : b0 + e;
        rsel[e] = (r >= 0 && r < n_records) ? r : -1;
    }
    __syncthreads();
    for (uint32_t c = tid; c < (uint32_t)te * hv; c += THREADS) {
        const int e = (int)(c / hv);
        if (rsel[e] >= 0) sh4[c] = reinterpret_cast<const uint4 *>(rec + (size_t)rsel[e] * L.bytes)[c % hv];
    }
    __syncthreads();
    for (int s = 0; s < L.n_head; ++s) {
        const Sec &S = L.s[s];
        if (!(S.what & what)) continue;
        for (uint32_t k = tid; k < (uint32_t)te * S.n; k += THREADS) {
            int e; uint32_t j;
            tile_elem(S, k, te, e, j);
            if (rsel[e] < 0) continue;
            copy_elem(S.soa + soa_index(S, (size_t)(b0 + e), j) * S.esz, sh + (size_t)e * L.head + S.off + (size_t)j * S.esz, S.esz);
        }
    }
    const int warp = tid >> 5, lane = tid & 31;
    for (int e = warp; e < te; e += WARPS) {
        if (rsel[e] < 0) continue;
        const char *r = rec + (size_t)rsel[e] * L.bytes;
        for (int s = L.n_head; s < L.n; ++s) {
            const Sec &S = L.s[s];
            if (!(S.what & what)) continue;
            const uint32_t bytes = S.esz * S.n;
            warp_copy(S.soa + (size_t)(b0 + e) * bytes, r + S.off, bytes, S.vec, lane);
        }
    }
    if (!mask_bytes || L.mask < 0) return;
    // the byte view of the loaded packed mask, read from the header tile or the record itself
    const Sec &Mk = L.s[L.mask];
    auto word = [&](int e, int w) -> uint32_t {
        const char *base = L.mask < L.n_head ? sh + (size_t)e * L.head : rec + (size_t)rsel[e] * L.bytes;
        return reinterpret_cast<const uint32_t *>(base + Mk.off)[w];
    };
    const int per = d.AP >> 4;   // 16 mask entries per 128-bit store (ge_api.cu:mask_bytes_kernel)
    for (uint32_t k = tid; k < (uint32_t)te * per; k += THREADS) {
        const int e = (int)(k / per), c = (int)(k % per);
        if (rsel[e] < 0) continue;
        const uint32_t bits = c < 2 * d.AW ? (word(e, c >> 1) >> ((c & 1) * 16)) & 0xffffu : 0u;
        reinterpret_cast<uint4 *>(d.mask_bytes + (size_t)(b0 + e) * d.AP)[c] =
            make_uint4(expand4(bits), expand4(bits >> 4), expand4(bits >> 8), expand4(bits >> 12));
    }
}

// dst env b <- the static arrays of src env src_index[b] (b, when src_index is NULL); out of range: env b untouched.
__global__ void __launch_bounds__(256) gather_instances_kernel(ge_batch d, StaticTab tab, const int32_t *__restrict__ src_index, int src_B) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * 8 + warp;
    if (b >= d.B) return;
    const int s = src_index ? src_index[b] : b;
    if (s < 0 || s >= src_B) return;
    copy_static_env(d, tab, 0, (size_t)s, (size_t)b, lane);
}

int check_desc(const ge_batch *d, const char *who) {
    if (!d) return ge_set_error(GE_ERR_ARG, "%s: null batch", who);
    if (d->kind < 0 || d->kind > GE_PERISHABLE_DELIVERY) return ge_set_error(GE_ERR_ARG, "%s: unknown kind %d", who, d->kind);
    if (d->B <= 0 || d->N < 2 || d->M < 0) return ge_set_error(GE_ERR_ARG, "%s: bad shape B=%d N=%d M=%d", who, d->B, d->N, d->M);
    if (d->NW != (d->N + 31) / 32 || d->MW != (d->M + 31) / 32 || d->AW != (d->A + 31) / 32)
        return ge_set_error(GE_ERR_ARG, "%s: layout not filled (call ge_fill_layout)", who);
    if (d->acc && d->acc_stride < d->B) return ge_set_error(GE_ERR_ARG, "%s: acc_stride %d < B %d", who, d->acc_stride, d->B);
    return GE_OK;
}

int launched(const char *what) {
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? GE_OK : ge_set_error(GE_ERR_CUDA, "%s launch: %s", what, cudaGetErrorString(e));
}

}  // namespace

extern "C" int ge_state_record_bytes(const ge_batch *batch) {
    int rc = check_desc(batch, "ge_state_record_bytes");
    if (rc) return rc;
    Layout L;
    build_layout(*batch, L);
    return (int)L.bytes;
}

extern "C" int ge_state_save(const ge_batch *batch, const int32_t *env_index, int count, void *records, void *stream) {
    GE_NVTX("ge_state_save");
    int rc = check_desc(batch, "ge_state_save");
    if (rc) return rc;
    if (count < 0 || count > batch->B) return ge_set_error(GE_ERR_ARG, "ge_state_save: count %d not in [0, B = %d]", count, batch->B);
    if (count == 0) return GE_OK;
    if (!records || (reinterpret_cast<uintptr_t>(records) & 15u)) return ge_set_error(GE_ERR_ARG, "ge_state_save: records must be a 16-byte aligned device pointer");
    Layout L;
    build_layout(*batch, L);
    const int te = tile_for(L);
    state_save_kernel<<<(count + te - 1) / te, THREADS, (size_t)te * L.head, (cudaStream_t)stream>>>(
        *batch, L, te, reinterpret_cast<char *>(records), count, env_index);
    return launched("state_save_kernel");
}

extern "C" int ge_state_load(const ge_batch *batch, const void *records, int n_records, const int32_t *record_index, unsigned what,
                             void *stream) {
    GE_NVTX("ge_state_load");
    int rc = check_desc(batch, "ge_state_load");
    if (rc) return rc;
    if (!(what & GE_STATE_DYNAMIC) || (what & ~GE_STATE_ALL))
        return ge_set_error(GE_ERR_ARG, "ge_state_load: what = %u must include GE_STATE_DYNAMIC and lie within GE_STATE_ALL", what);
    if (n_records < 0) return ge_set_error(GE_ERR_ARG, "ge_state_load: n_records %d < 0", n_records);
    if (!record_index && n_records < batch->B)
        return ge_set_error(GE_ERR_ARG, "ge_state_load: without record_index every env b loads record b: n_records %d < B %d", n_records, batch->B);
    if (n_records == 0) return GE_OK;   // (every index is out of range)
    if (!records || (reinterpret_cast<uintptr_t>(records) & 15u)) return ge_set_error(GE_ERR_ARG, "ge_state_load: records must be a 16-byte aligned device pointer");
    Layout L;
    build_layout(*batch, L);
    const int te = tile_for(L);
    const int mb = ge_mask_bytes_current(batch) ? 1 : 0;
    state_load_kernel<<<(batch->B + te - 1) / te, THREADS, (size_t)te * L.head, (cudaStream_t)stream>>>(
        *batch, L, te, reinterpret_cast<const char *>(records), n_records, record_index, what, mb);
    return launched("state_load_kernel");
}

extern "C" int ge_gather_instances(const ge_batch *dst, const ge_batch *src, const int32_t *src_index, void *stream) {
    GE_NVTX("ge_gather_instances");
    int rc = check_desc(dst, "ge_gather_instances (dst)");
    if (!rc) rc = check_desc(src, "ge_gather_instances (src)");
    if (rc) return rc;
    const ge_batch &d = *dst, &s = *src;
    if (d.kind != s.kind || d.N != s.N || d.M != s.M || d.parenting != s.parenting || d.n_dests != s.n_dests ||
        d.n_choices != s.n_choices || d.n_targets != s.n_targets || d.max_distance != s.max_distance ||
        ((d.flags ^ s.flags) & GE_FLAG_FORCE_WARP))
        return ge_set_error(GE_ERR_ARG, "ge_gather_instances: src is not shaped like dst (kind, N, M, parenting, n_dests, n_choices, "
                                        "n_targets, max_distance and GE_FLAG_FORCE_WARP must agree)");
    if (d.dfa_bytes != s.dfa_bytes)
        return ge_set_error(GE_ERR_ARG, "ge_gather_instances: dfa_bytes differ (%d vs %d): the batches need the same distance automaton",
                            d.dfa_bytes, s.dfa_bytes);
    if (!src_index && s.B < d.B)
        return ge_set_error(GE_ERR_ARG, "ge_gather_instances: without src_index dst env b takes src env b: src B %d < dst B %d", s.B, d.B);
    StaticTab tab;
    if ((rc = static_table(d, src, 1, tab, "ge_gather_instances"))) return rc;
    for (int i = 0; i < tab.n; ++i) {
        const uintptr_t t0 = reinterpret_cast<uintptr_t>(tab.a[i].dst), t1 = t0 + static_span(d, tab.a[i], d.B);
        for (int j = 0; j < tab.n; ++j) {
            const uintptr_t s0 = reinterpret_cast<uintptr_t>(tab.a[j].src[0]), s1 = s0 + static_span(s, tab.a[j], s.B);
            if (t0 < s1 && s0 < t1)
                return ge_set_error(GE_ERR_ARG, "ge_gather_instances: dst and src static arrays overlap (no in-place gather)");
        }
    }
    gather_instances_kernel<<<(d.B + 7) / 8, 256, 0, (cudaStream_t)stream>>>(d, tab, src_index, s.B);
    return launched("gather_instances_kernel");
}
