// ge_pool.cu -- per-env instance turnover ("regenerate on done", SURVEY 8(f1); reset() of every reference env, e.g.
// shortest_path.py:47-98, builds a NEW graph per episode).
//
// A pool of G banks, each a fully prepared batch of B instances (graph store + derived arrays + features + heuristics +
// in-range tables), sits next to the live batch.  After a step, ge_pool_refill gives every env whose episode just ended
// the next instance of ITS slot (bank order[episode[b] % n_active], episode[b]++): one warp copies that instance's static
// arrays over the env's own and flags the env in `select`; ge_reset(select) then re-initialises state and mask.  Copying
// (instead of an indirection in every kernel) keeps the hot step kernels and their tiled / bulk-staged layouts unchanged;
// the copy costs the instance's bytes once per episode.  Banks are regenerated in the background by the host side
// (graphenvs_b200/pool.py) on another stream; a bank being regenerated is simply absent from `order`.
#include "ge_static.cuh"

using namespace ge;

namespace {

__global__ void __launch_bounds__(256) pool_refill_kernel(ge_batch d, StaticTab tab, const int32_t *__restrict__ order, int n_active,
                                                        uint32_t *__restrict__ episode, uint8_t *__restrict__ select) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * 8 + warp;
    if (b >= d.B) return;
    const bool fin = d.done[b] != 0;
    if (lane == 0) select[b] = fin ? 1 : 0;
    if (!fin) return;
    const uint32_t ep = episode[b];
    const int k = order[ep % (uint32_t)n_active];
    __syncwarp();
    if (lane == 0) episode[b] = ep + 1u;
    copy_static_env(d, tab, k, (size_t)b, (size_t)b, lane);
}

}  // namespace

// banks: HOST array of n_banks descriptors shaped like `live`.  order: DEVICE int32[n_active] = the banks that may be read
// now.  episode: DEVICE uint32[B] per-env episode counter.  select: DEVICE uint8[B], written for every env (1 = refilled).
extern "C" int ge_pool_refill(const ge_batch *live, const ge_batch *banks, int n_banks, const int32_t *order, int n_active,
                              uint32_t *episode, uint8_t *select, void *stream) {
    GE_NVTX("ge_pool_refill");
    if (!live || !banks || !order || !episode || !select) return ge_set_error(GE_ERR_ARG, "ge_pool_refill: null argument");
    if (n_banks < 1 || n_banks > STATIC_MAX_SRC || n_active < 1 || n_active > n_banks) return ge_set_error(GE_ERR_ARG, "ge_pool_refill: 1 <= n_active <= n_banks <= %d", STATIC_MAX_SRC);
    for (int k = 0; k < n_banks; ++k)
        if (banks[k].kind != live->kind || banks[k].N != live->N || banks[k].M != live->M || banks[k].B < live->B ||
            ((banks[k].flags ^ live->flags) & GE_FLAG_FORCE_WARP))
            return ge_set_error(GE_ERR_ARG, "ge_pool_refill: bank %d is not shaped like the live batch", k);
    const ge_batch &d = *live;
    StaticTab tab;
    int rc = static_table(d, banks, n_banks, tab, "ge_pool_refill");
    if (rc) return rc;
    pool_refill_kernel<<<(d.B + 7) / 8, 256, 0, (cudaStream_t)stream>>>(d, tab, order, n_active, episode, select);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? GE_OK : ge_set_error(GE_ERR_CUDA, "pool_refill_kernel launch: %s", cudaGetErrorString(e));
}
