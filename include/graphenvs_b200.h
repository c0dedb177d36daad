/* graphenvs_b200.h -- C ABI of the B200-native batched GraphEnvs engine.
 *
 * One `ge_batch` describes B independent environment instances of ONE env kind with uniform
 * (N nodes, M = 2*n_edges directed edges).  Every pointer in it is a DEVICE pointer owned by the
 * caller (the Python host allocates them as torch tensors, a C host with cudaMalloc); the
 * library allocates nothing and keeps no state between calls, so a descriptor can be copied,
 * sliced per rank, or rebuilt freely.  All calls enqueue work on `stream` (a cudaStream_t passed
 * as void*), return 0 on success / a negative ge_status on error (text via ge_last_error()),
 * never throw, and are not thread-safe per descriptor (two host threads may work on DIFFERENT descriptors
 * concurrently: the library's only process-wide state, its kernel-attribute table and its CUDA-graph cache,
 * is mutex-guarded).  No torch types appear here.
 *
 * What each entry point replaces in the reference (paths relative to graph_envs/):
 *   ge_reset          tail of every Env.reset(): state init + first info['mask']
 *                     (shortest_path.py:74-98, longest_path.py:82-122, steiner_tree.py:89-112,
 *                      tsp.py:119-162, max_independent_set.py:70-89, densest_subgraph.py:68-101,
 *                      multicast_routing.py:118-152, distribution_center.py:94-127)
 *   ge_step           Env.step() + Env._get_mask() for the 8 envs
 *                     (shortest_path.py:105-141, longest_path.py:125-196, steiner_tree.py:116-157,
 *                      tsp.py:174-258, max_independent_set.py:92-124, densest_subgraph.py:105-196,
 *                      multicast_routing.py:155-266, distribution_center.py:129-174,
 *                      perishable_product_delivery.py:175-271)
 *   ge_obs_flat       utils.vectorize_graph (utils.py:87-88), layout of utils.devectorize_graph
 *   ge_obs_graph      utils.devectorize_graph (utils.py:14-23) applied on the device: (x, edge_features, edge_index)
 *   ge_features       feature_extraction.generate_features (feature_extraction.py:6-37)
 *   ge_prepare        reset-time derived data: eval heuristics (shortest_path.py:88-90,
 *                     longest_path.py:103-106, steiner_tree.py:77-85, multicast_routing.py:107-115), Multicast max_distance
 *                     (multicast_routing.py:98-103), DistributionCenter in-range tables
 *                     (distribution_center.py:25-26,113-116)
 *   ge_generate       instance generation of reset() (shortest_path.py:54-75 and peers) --
 *                     distribution parity only (device RNG), see DESIGN.md
 *   ge_sample_actions README.md:54-68 "random valid action" loop (policy stand-in for benches)
 *   ge_step_sampled   the same loop body fused: action draw + Env.step() in one launch
 *   ge_sample_logits  the policy side of a training loop: a masked categorical over policy logits (Gumbel-max / greedy),
 *   ge_masked_log_prob (+ _backward)  its differentiable log-prob and entropy for the update (ge_policy.cu)
 *   ge_beam_expand    one beam-search step: every beam's valid continuations scored and the W best per instance kept (ge_policy.cu)
 *   ge_beam_expand_sampled  one stochastic-beam-search step: W distinct sequences per instance sampled without replacement
 *   ge_mcts_select / ge_mcts_expand  Monte Carlo tree search (PUCT): one simulation round's selection and its expansion + backup
 *   ge_state_save / ge_state_load / ge_gather_instances  branching an env, i.e. copy.deepcopy(env) of a gym env: per-env state
 *                     records and instance replication for search decoders (multi-start, beam search, lookahead; ge_state.cu)
 */
#ifndef GRAPHENVS_B200_H
#define GRAPHENVS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GE_ABI_VERSION 4

typedef enum {
    GE_SHORTEST_PATH = 0,      /* ShortestPath-v0        shortest_path.py        node actions */
    GE_LONGEST_PATH = 1,       /* LongestPath-v0         longest_path.py         node actions */
    GE_STEINER_TREE = 2,       /* SteinerTree-v0 / MST   steiner_tree.py         edge actions */
    GE_TSP = 3,                /* TSP-v0                 tsp.py                  node actions */
    GE_MAX_INDEPENDENT_SET = 4,/* MaxIndependentSet-v0   max_independent_set.py  node actions */
    GE_DENSEST_SUBGRAPH = 5,   /* DensestSubgraph-v0     densest_subgraph.py     node actions */
    GE_MULTICAST_ROUTING = 6,  /* MulticastRouting-v0    multicast_routing.py    edge actions */
    GE_DISTRIBUTION_CENTER = 7,/* DistributionCenter-v0  distribution_center.py  node actions */
    GE_PERISHABLE_DELIVERY = 8 /* PerishableProductDelivery-v0  perishable_product_delivery.py  node actions (action == head: pick up).
                                  n_dests = n_products (<= 5), targets = [B, 2 * n_products] pickups then dropoffs,
                                  max_dist32 = delivery time; counters[b] = {2-bit status per product, moves made} */
} ge_kind;

typedef enum {
    GE_OK = 0,
    GE_ERR_ARG = -1,      /* bad descriptor / unsupported size */
    GE_ERR_CUDA = -2,     /* CUDA runtime error, see ge_last_error() */
    GE_ERR_UNSUPPORTED = -3
} ge_status;

/* ge_batch.flags */
#define GE_FLAG_AUTO_RESET 1u   /* on done: re-init the env's state on its own graph inside ge_step */
#define GE_FLAG_WEIGHTED_PR 2u  /* pagerank uses edge weights (TSP stores them as 'weight', tsp.py:90) */
#define GE_FLAG_UNWEIGHTED 4u   /* ge_generate: weighted=False (all edge weights / MIS costs 1.0) */
#define GE_FLAG_FORCE_WARP 8u   /* testing: use the warp-per-env kernels even where the lane-per-env ones apply */
#define GE_FLAG_PDL 16u         /* ge_step / ge_step_sampled launch with programmatic stream serialization: the step kernel may become
                                   resident -- and read STATIC instance data (adjacency tiles, automaton tables, src / dest, the
                                   reset-time mask) -- while the previous launch of the stream is still running; it waits for that launch
                                   (griddepcontrol.wait) before it uses any env state.  Before the wait it may only prefetch env state
                                   into L2, or read it through L2 to pick what to prefetch (the lane-per-env step guesses its draw that
                                   way); such reads are never used as results, and L2 is coherent, so the loads after the wait see the
                                   previous launch's writes.  The caller promises that the preceding work in the stream does not write
                                   this batch's static arrays (i.e. it is another step or a state save / load, not ge_generate /
                                   ge_build_adjacency / ge_pool_refill / ge_gather_instances). */

/* per-env status written by ge_step into flags[b].status */
#define GE_STEP_OK 0
#define GE_STEP_INVALID 1     /* the reference would raise AssertionError; state unchanged */
#define GE_STEP_AFTER_DONE 2  /* env already done and auto-reset off; state unchanged */

/* One 4-byte record per env per step (written with a single 32-bit store). */
typedef struct {
    uint8_t done;     /* 1 if this step ended the episode */
    int8_t solved;    /* -1 = key absent from info, 0 / 1 = info['solved'] */
    uint8_t status;   /* GE_STEP_* */
    uint8_t has_mask; /* 0 only for LongestPath's invalid-move early return (longest_path.py:169-173) */
} ge_step_flags;

typedef struct ge_batch {
    /* ---- shape / parameters ---- */
    int32_t kind, B, N, M;        /* M = 2 * n_edges directed edges */
    int32_t parenting;            /* per-env rules of SURVEY 8(b) are enforced by the host */
    int32_t n_dests;              /* SteinerTree / MulticastRouting */
    int32_t n_choices;            /* DensestSubgraph (already floor(N/e) when defaulted) */
    int32_t n_targets;            /* DistributionCenter target_count (row count of in_range) */
    uint32_t flags;
    int32_t env_id0;              /* global id of env 0 of this slice (rank offset; feeds the action sampler) */
    int32_t NW, MW;               /* ceil(N/32), ceil(M/32) */
    int32_t A, AW, AP;            /* mask length (N or M), its words, byte stride (A rounded up to 16) */
    int32_t RP, MP, ADJS;         /* strides: row_ptr (ints), col/w (elements), adj_bits (words) per env */
    int32_t acc_stride;           /* elements between the 4 components of `acc` (= B of the batch the array was allocated for;
                                     ge_fill_layout sets it to B, ge_batch_slice keeps the parent's) */
    int32_t dfa_bytes;            /* size of the `dfa` array in bytes (0 = unknown) */
    double max_distance;          /* DistributionCenter cutoff */

    /* ---- graph store (static per instance) ---- */
    const int32_t *row_ptr;       /* [B, RP]   CSR offsets, reference edge order (source-sorted) */
    const int32_t *col;           /* [B, MP]   destination of every directed edge */
    const float *w32;             /* [B, MP]   edge feature column 0 (float32), kinds stepping in fp32 */
    const double *w64;            /* [B, MP]   float64 edge attribute, kinds stepping in fp64 / prepare */
    uint32_t *adj_bits;           /* [B, ADJS] N rows of NW words: adjacency bit-matrix (derived by ge_build_adjacency).
                                              For N <= 64 node-action kinds without GE_FLAG_FORCE_WARP the library stores it in
                                              tiles of 32 envs, [ceil(B/32)][N][32 envs] of NW words (bank-conflict-free for the
                                              lane-per-env kernels): allocate (B rounded up to 32) * ADJS words */
    int32_t *rev;                 /* [B, MP]   index of the reverse edge (v->u) of every edge (u->v) (derived), or NULL */
    int32_t *esrc;                /* [B, MP]   source node of every edge (derived), or NULL */
    double *wsort;                /* [B, MP]   w64 permuted so that every row is in ascending destination order (derived), or
                                              NULL: adj[u, v] = wsort[row_ptr[u] + rank of v in the adjacency bit-row of u] */
    const uint8_t *wcode;         /* [B, MP]   index of every edge weight in the batch's small set of distinct weights, or NULL */
    const uint8_t *dfa;           /* exact fp64 distance automaton for the cutoff SSSP, or NULL: [S, W, T[S*W], expand[S], cmax[S]]
                                              (cmax[i] = largest weight code j with T[i*W+j] != 255, or 255).
                                              State i = the i-th smallest value reachable as a left-fold fp64 sum of the W
                                              distinct weights without exceeding max_distance; T[i*W+j] = state of
                                              fl(value_i + weight_j) or 255 when it exceeds the cutoff; expand[i] = value_i +
                                              smallest weight <= cutoff.  Built on the host with the same IEEE additions,
                                              so state order == distance order and every comparison is exact. */
    uint32_t *dc_edges;           /* [B, MP]   DistributionCenter with an automaton: every CSR row re-ordered by weight code,
                                              entry = col | code << 16 (derived by ge_prepare bit 4), or NULL: the cutoff search then
                                              visits only the row prefix that can stay within the cutoff (csrc/ge_dc.cu) */
    double *wmin;                 /* [B]       smallest edge weight of the instance (derived), or NULL: lets the cutoff
                                              SSSP skip nodes that cannot relax anything within the cutoff */
    double *wmat;                 /* [B, N, N] dense float64 weight matrix = the reference's self.adj (derived by
                                              ge_build_adjacency), used when N <= 64 by the kinds stepping in fp64; or NULL */

    /* ---- instance parameters (static) ---- */
    int32_t *src, *dest;          /* [B] */
    uint32_t *target_bits;        /* [B, NW]  IS_TARGET column as a bitset */
    float *node_cost;             /* [B, N]   MIS weight / DistCenter cost column */
    float *node_xy;               /* [B, N, 2] TSP spatial coordinates or NULL */
    float *max_dist32;            /* [B]      Multicast MAX_DISTANCE column value */
    int32_t *targets;             /* [B, n_targets] DistributionCenter target node ids */
    uint32_t *in_range;           /* [B, n_targets, NW] nodes within max_distance of each target */
    double *heuristic;            /* [B]      info['heuristic_solution'] */
    double *heuristic_alt;        /* [B]      info['heuristic_device']: labelled alternative where the reference's value is defined by
                                              networkx iteration order (Steiner shortest-path heuristic, TSP nearest neighbour, greedy
                                              MIS; csrc/ge_heuristics.cu), or NULL */
    float *features;              /* [B, N, 5] structural features or NULL (zeros in obs) */

    /* ---- dynamic state ---- */
    int32_t *head;                /* [B] */
    uint32_t *node_bits;          /* [B, NW]  HAS_MSG / TAKEN column as a bitset */
    uint32_t *node_bits2;         /* [B, NW]  DistCenter IS_COVERED; Densest neighbour-union */
    uint32_t *edge_bits;          /* [B, MW]  Multicast EDGE_IS_TAKEN */
    float *dist32;                /* [B, N]   Multicast DISTANCE_FROM_SOURCE column */
    uint64_t *bestkey;            /* [B, N]   Multicast parenting >= 3: running argmin per frontier vertex,
                                              (float32 bits of dist[src e] + delay[e]) << 32 | e, ~0 = none; or NULL */
    double *cost;                 /* [B]      running solution_cost (fp32 kinds keep a float value in it) */
    int32_t *counters;            /* [B, 4]   Densest: k_taken, edge_cnt.  Incremental kernels (ge_incr.cu): targets in the
                                              tree / nodes taken, popcount of the mask, constraints satisfied */
    uint8_t *done;                /* [B] */
    uint32_t *mask_bits;          /* [B, AW]  current valid-action mask, packed */
    uint32_t *mask_cnt;           /* [B, 8]   incremental-mask kernels with large masks: popcounts of the 16 chunks of ceil(AW/16) words
                                              of the packed mask, 16 bits each (state, maintained with the mask), or NULL */
    uint8_t *mask_bytes;          /* [B, AP]  same mask as bytes (torch.bool view) or NULL.  Kept current by the group,
                                              DistributionCenter, PerishableProductDelivery and general kernels; the LANE-PER-ENV
                                              kernels (N <= 64: ShortestPath, LongestPath, TSP, MaxIndependentSet, DensestSubgraph) and
                                              the INCREMENTAL-mask kernels (SteinerTree, Multicast p >= 2, MaxIndependentSet N > 64)
                                              update only the packed mask (ge_mask_bytes_current() == 0) and the byte view is produced
                                              on demand by ge_mask_bytes */
    uint32_t *mask0_bits;         /* [B, AW]  mask right after reset(), written by ge_reset, or NULL.  It depends only on the
                                              instance, so auto-reset inside ge_step copies it instead of recomputing it */
    double *acc;                  /* [4, acc_stride] per-env statistics: episodes, solved, sum reward, sum final cost */
    uint64_t *traj;               /* [B]      rolling checksum of (action, done, solved, status) per env, or NULL;
                                              same recurrence as oracle/graphenvs_oracle.c oenv_rollout */
    uint32_t *env_steps;          /* [B]      per-env count of accepted steps, or NULL.  ge_step increments it and the
                                              samplers add it to `t`, so a captured CUDA graph (frozen kernel
                                              arguments) draws fresh actions on every replay */
    float *obs_x;                 /* [B, N, F] optional DEVICE buffer, or NULL: ge_step_host_pipelined rewrites the node columns of the
                                              observation (ge_obs_nodes; utils.py:14-23 `x`) of every slice on its write-back lane, while
                                              the next slice steps -- the dynamic part of the observation for a device-resident consumer */
    uint32_t *dc_rows;            /* [B, N, 32] DistributionCenter with an automaton (derived by ge_prepare bit 4 next to dc_edges; the
                                              dedicated kernel needs both, without them the batch steps in the general family): the first
                                              32 entries of every weight-sorted row at a FIXED stride of 128 bytes, padded with 0xffffffff.
                                              The cutoff search then needs no row_ptr lookup (one dependent memory round less per search
                                              level), reads sector-aligned rows, and prefetches a row when its node is queued; a prefix
                                              longer than 32 entries continues in dc_edges */
    uint32_t *progress;           /* [ceil(B / 1024)] optional DEVICE counters, or NULL: a step kernel that supports it (ge_progress_supported)
                                              adds the number of envs it has finished -- every store of those envs made visible first -- to
                                              progress[env >> 10].  ge_step_host_pipelined with chunks = 0 uses it to stream results to the host
                                              from a concurrent write-back kernel while the step kernel is still running */
} ge_batch;

/* step outputs (device pointers) */
typedef struct {
    float *reward;            /* [B] */
    ge_step_flags *flags;     /* [B] */
    double *solution_cost;    /* [B] info['solution_cost'] (NaN = key absent) */
} ge_step_out;

int ge_abi_version(void);
const char *ge_last_error(void);

/* Fills the derived size fields (NW, MW, A, AW, AP, RP, MP, ADJS) from kind/N/M. */
int ge_fill_layout(ge_batch *batch);
/* Descriptor of the sub-batch [lo, lo + count) of `batch`: every per-env pointer advanced, B = count, env_id0 += lo.
 * All arrays are SoA with fixed per-env strides, so a slice is a contiguous range of each of them; it can be stepped,
 * reset and observed on its own (other streams, other host threads).  `lo` must be a multiple of 32. */
int ge_batch_slice(const ge_batch *batch, int lo, int count, ge_batch *out);
/* Bytes of dynamic shared memory one step launch uses (for diagnostics / occupancy reports). */
int ge_step_smem_bytes(const ge_batch *batch);

/* Fills every DERIVED graph array whose pointer is set: adj_bits, wmat, wsort, rev, esrc, wmin. */
int ge_build_adjacency(const ge_batch *batch, void *stream);
/* what: bit0 heuristics with the reference's value: SSSP / MST (tie-independent) and Multicast's union of first-found
 *            shortest paths (networkx's pop order restated on the device),
 *       bit3 labelled alternative heuristics -> heuristic_alt (SteinerTree 1 < n_dests < N-1, TSP, MaxIndependentSet),
 *       bit1 Multicast max_distance from u01[B] (the reference's np.random.rand() draw); u01 == NULL takes the draw
 *            ge_generate left in max_dist32 (a pure function of seed and global env id),
 *       bit2 DistributionCenter in-range tables,
 *       bit4 DistributionCenter weight-sorted edge list dc_edges (needs wcode). */
int ge_prepare(const ge_batch *batch, int what, const double *u01, void *stream);
int ge_features(const ge_batch *batch, void *stream);
int ge_generate(const ge_batch *batch, uint64_t seed, int32_t *row_ptr, int32_t *col, double *w64, float *w32,
                void *stream);

/* Envs of the most recent ge_generate on `stream` whose rejection loop (4096 draws) found no valid graph and that were
 * emitted connected-by-construction instead; synchronises the stream.  Negative = error. */
int ge_generate_fallbacks(void *stream);

/* Instance turnover (every reference reset() builds a new graph): gives each env whose episode has ended (done[b] != 0) the
 * next instance of its slot from a pool of `n_banks` prepared batches -- bank order[episode[b] % n_active], episode[b]++ --
 * by copying that instance's static arrays over the env's own, and writes select[b] = 1 for those envs (0 for the others);
 * follow with ge_reset(batch, select).  banks: HOST array of descriptors shaped like `batch`; order (int32[n_active]),
 * episode (uint32[B]), select (uint8[B]): device arrays.  A bank that is being regenerated is left out of `order`. */
int ge_pool_refill(const ge_batch *batch, const ge_batch *banks, int n_banks, const int32_t *order, int n_active,
                   uint32_t *episode, uint8_t *select, void *stream);

/* select: device uint8[B] (1 = reset this env) or NULL for all. */
int ge_reset(const ge_batch *batch, const uint8_t *select, void *stream);
int ge_step(const ge_batch *batch, const int32_t *actions, const ge_step_out *out, void *stream);
int ge_sample_actions(const ge_batch *batch, uint64_t seed, uint32_t t, int32_t *actions, void *stream);
/* ge_sample_actions + ge_step in ONE launch (random-rollout mode: at these batch sizes a launch costs
 * as much as the work).  The chosen actions are written to `actions` (may not be NULL). */
int ge_step_sampled(const ge_batch *batch, uint64_t seed, uint32_t t, int32_t *actions, const ge_step_out *out, void *stream);

/* Reference wire format (utils.py:87-88): out is float32[count, N*F + M*Fe + 2*M]. */
int ge_obs_len(const ge_batch *batch);
int ge_obs_flat(const ge_batch *batch, int env_lo, int count, float *out, void *stream);
/* The same observation as three tensors (what utils.devectorize_graph, utils.py:14-23, slices out of the flat vector):
 * x float32[count, N, F], edge_attr float32[count, M, Fe], edge_index int64[count, M, 2] -- no float round trip of indices. */
int ge_obs_graph(const ge_batch *batch, int env_lo, int count, float *x, float *edge_attr, int64_t *edge_index, void *stream);
/* x only: the node columns are the part of the observation a step changes (utils.py:14-23 `x`). */
int ge_obs_nodes(const ge_batch *batch, int env_lo, int count, float *x, void *stream);
/* Name of the CUDA kernel ge_step / ge_step_sampled dispatches this descriptor to (reports, profiles). */
const char *ge_step_kernel_name(const ge_batch *batch, int sampled);

/* 1 when every ge_step / ge_reset leaves mask_bytes equal to the packed mask; 0 when the byte view must be refreshed with
 * ge_mask_bytes before it is read: the incremental-mask kernels (a scattered byte store per changed edge was 2.3 KB of HBM
 * traffic per Multicast step against 1.8 KB of useful bytes) and the lane-per-env kernels (AP bytes per env and about 16 %
 * of the step's instructions for a view that the samplers and the packed host results do not read). */
int ge_mask_bytes_current(const ge_batch *batch);
/* Expands the packed mask of envs [env_lo, env_lo + count) into mask_bytes (one coalesced pass). */
int ge_mask_bytes(const ge_batch *batch, int env_lo, int count, void *stream);
/* End-to-end entry with HOST buffers: copies actions H2D, steps, copies reward / flags /
 * solution_cost (and the byte mask [B, AP] when h_mask != NULL, the packed mask [B, AW] when
 * h_mask_bits != NULL) D2H, and synchronises the stream.  If reward | flags | solution_cost |
 * mask_bits are laid out back to back in that order on the device AND on the host (B even), the
 * results come back in one copy.
 * d_actions / out are device staging buffers owned by the caller (GE_ERR_ARG when NULL). */
int ge_step_host(const ge_batch *batch, const int32_t *h_actions, int32_t *d_actions, const ge_step_out *out,
                 float *h_reward, ge_step_flags *h_flags, double *h_solution_cost, uint8_t *h_mask,
                 uint32_t *h_mask_bits, void *stream);

/* PIPELINED end-to-end step with pinned (device-mapped) HOST buffers.  The batch is cut into `chunks` slices; each slice
 * runs step kernel -> write-back on its own branch of ONE CUDA graph, so slice i's results cross PCIe while slice i+1 is
 * stepping.  The step kernels read the actions straight from h_actions (zero-copy), and results are written back by a small
 * copy kernel straight into the caller's four host arrays (coalesced 128-byte PCIe writes; no staging layout imposed on the
 * host side).  Blocks until the results are visible to the host (spin on stream completion).  h_solution_cost / h_mask_bits
 * may be NULL. */
int ge_step_host_pipelined(const ge_batch *batch, const int32_t *h_actions, const ge_step_out *out,
                           float *h_reward, ge_step_flags *h_flags, double *h_solution_cost, uint32_t *h_mask_bits,
                           int chunks, void *stream);
/* ge_step_host_pipelined with COMPACT host results: 9 instead of 16 bytes per env next to the packed mask (PCIe write time is what a
 * host step waits for).  h_flags8[b] = done | (solved + 1) << 1 | status << 3 | has_mask << 5 (GE_FLAGS8_* below); h_solution_cost32 =
 * (float) solution_cost, NaN = key absent (within the 1e-5 relative tolerance of the parity contract; costs of the fp32 kinds are
 * float values already).  Same slices, lanes and completion rule. */
#define GE_FLAGS8_DONE(f) ((f) & 1)
#define GE_FLAGS8_SOLVED(f) ((int)(((f) >> 1) & 3) - 1)
#define GE_FLAGS8_STATUS(f) (((f) >> 3) & 3)
#define GE_FLAGS8_HAS_MASK(f) (((f) >> 5) & 1)
int ge_step_host_compact(const ge_batch *batch, const int32_t *h_actions, const ge_step_out *out,
                         float *h_reward, uint8_t *h_flags8, float *h_solution_cost32, uint32_t *h_mask_bits, int chunks, void *stream);
/* 1 when the step kernel this batch dispatches to signals ge_batch.progress (the lane-per-env families, DistributionCenter). */
int ge_progress_supported(const ge_batch *batch);
/* Drops the cached CUDA graphs ge_step_host / ge_step_host_pipelined built for this batch (call before freeing its memory). */
int ge_step_host_release(const ge_batch *batch);

/* Reduces acc[4,B] to out[4] (device double[4]): episodes, solved, sum reward, sum final cost. */
int ge_stats(const ge_batch *batch, double *out4, void *stream);

/* ---- Rollout helpers: a categorical policy over the valid actions (csrc/ge_policy.cu) ----
 *
 * Logits are row-major [rows, A] on the device, float32 (GE_LOGITS_F32) or bfloat16 (GE_LOGITS_BF16, upcast to float32);
 * all arithmetic is float32.  The mask of row b is the packed bitset of ceil(A/32) words at mask_bits + b * ceil(A/32)
 * (the layout of ge_batch.mask_bits).  Per row, over the VALID actions V only:
 *   lse = log sum_{i in V} exp(l_i),  p_i = exp(l_i - lse),  H = lse - sum_{i in V} p_i l_i  (entropy in nats).
 * Edge semantics (all three calls):
 *   - empty mask row: action -1, log_prob 0, entropy 0, lse -inf, zero gradient (ge_sample_actions also returns -1);
 *   - mask bits at positions >= A are ignored, and no logit at index >= A is ever read;
 *   - logits of invalid actions are never read (NaN / inf there change nothing); logits of valid actions must be finite;
 *   - ge_masked_log_prob with an action outside [0, A) or on a clear bit (non-empty row): log_prob = -inf, the entropy is still
 *     computed, and the backward pass gets no gradient from that row's log_prob term;
 *   - deterministic: no atomics and a fixed reduction order, the same inputs give bit-identical outputs; for the same logits,
 *     mask and action, ge_sample_logits' log_prob / entropy equal ge_masked_log_prob's bit for bit (PPO ratio exactly 1);
 *   - rows are addressed with size_t offsets (rows * A may exceed 2^31 elements).
 * Bad arguments (unknown dtype, rows or A <= 0, a NULL required pointer) return GE_ERR_ARG. */
#define GE_LOGITS_F32 0
#define GE_LOGITS_BF16 1
/* Draws actions[b] for every env of `batch` from its current packed mask (batch->mask_bits) and the logits [B, A]:
 * greedy != 0: argmax of l over the valid actions; otherwise Gumbel-max, argmax of l_a + g_a.  Ties go to the lowest action
 * index (greedy equals torch.argmax of the masked logits).  log_prob / entropy [B] (float32, may be NULL) of the chosen action.
 * Noise: a pure counter-based function of (seed, e, t', a), e = env_id0 + b (global env id), t' = t + env_steps[b] when
 * env_steps is set (uint32 arithmetic), with mix32 = the splitmix of ge_sample_actions (csrc/ge_common.cuh):
 *   key = (uint64) mix32(seed, e, t') << 32 | mix32(seed ^ 0xD1B54A32D192ED03, e, t')
 *   h   = mix32(key, a, 0x85EBCA6B),   u = ((h >> 8) + 0.5) / 2^24  (exact in float32, in (0, 1))
 *   g_a = -logf(-logf(u)),   score_a = l_a + g_a  (float32)
 * So a rank slice draws what the single-GPU batch draws, and a captured CUDA graph with the env clock draws fresh actions on
 * every replay.  With all logits equal the draw is uniform but NOT the action ge_sample_actions picks (different noise).
 * Under GE_FLAG_PDL the launch may start under the previous step's tail; it touches nothing before that step completes, and
 * every step kernel reads actions[b] only after its own wait, so sample -> step -> sample chains are safe. */
int ge_sample_logits(const ge_batch *batch, const void *logits, int dtype, int greedy, uint64_t seed, uint32_t t,
                     int32_t *actions, float *log_prob, float *entropy, void *stream);
/* log_prob, entropy, lse [rows] of actions[rows] under the masked categorical (no ge_batch: masks from a rollout buffer). */
int ge_masked_log_prob(const void *logits, int dtype, int rows, int A, const uint32_t *mask_bits, const int32_t *actions,
                       float *log_prob, float *entropy, float *lse, void *stream);
/* Dense grad_logits [rows, A] in the logits' dtype from lse / entropy of ge_masked_log_prob (no second reduction):
 *   g_lp (1[i = a] - p_i) - g_H p_i (log p_i + H) for valid i, 0 elsewhere.  grad_log_prob / grad_entropy may be NULL (= 0). */
int ge_masked_log_prob_backward(const void *logits, int dtype, int rows, int A, const uint32_t *mask_bits, const int32_t *actions,
                                const float *lse, const float *entropy, const float *grad_log_prob, const float *grad_entropy,
                                void *grad_logits, void *stream);
/* One beam-search step over a batch of B = G * W envs: group g is envs [g*W, g*W + W), 1 <= W <= 32 (W beams of one instance).
 * Reads batch->mask_bits, batch->done, logits [B, A] (layout and dtype of ge_sample_logits) and score [B], the running beam
 * scores (float32 sums of log-probs).  Beam b of group g contributes:
 *   - nothing when score[b] == -inf (a DEAD beam);
 *   - when done[b]: one STAY candidate (b, action -1) of score score[b];
 *   - otherwise one candidate (b, a) per valid action a, of score fl32(score[b] + fl32(l_a - lse_b)), lse_b the masked log-sum-exp
 *     of ge_masked_log_prob (so the log-prob term equals ge_masked_log_prob's bit for bit); a live beam with an empty mask none.
 * Within each group, output slot j (env g*W + j) gets the j-th best candidate of the group in the total order: score descending,
 * then parent slot ascending, then action ascending -- a stable sort of all the group's candidates, exact:
 *   parent[j]     env index (in [0, B) of this descriptor) of the candidate's beam, -1 when the group has fewer than W candidates;
 *   action[j]     the candidate's action, -1 for a stay or an empty slot;
 *   score_out[j]  its score, -inf for an empty slot (which is then dead in the next step);
 *   load_index[j] parent[j], except -1 where parent[j] == g*W + j or the slot is empty: the record_index of ge_state_load after
 *                 ge_state_save of every env, so a slot that continues its own beam is not copied.
 * A decode step is then: save every env, load with load_index, ge_step with action (a stay slot's -1 meets a done env and gets
 * GE_STEP_AFTER_DONE with state and acc unchanged; an empty slot's gets GE_STEP_INVALID).  Deterministic (no atomics); logits of
 * invalid actions are never read and rows are addressed with size_t.  Launched like ge_sample_logits: under GE_FLAG_PDL it may
 * start under the previous step's tail and touches nothing before that step completes.  No synchronisation or allocation: it can
 * be captured in a CUDA graph.  GE_ERR_ARG, before any CUDA call, for an unknown dtype, W outside [1, 32], B % W != 0, a NULL
 * pointer (batch->mask_bits and batch->done included), or overlapping score / score_out / parent / action / load_index. */
int ge_beam_expand(const ge_batch *batch, int W, const void *logits, int dtype, const float *score, float *score_out,
                   int32_t *parent, int32_t *action, int32_t *load_index, void *stream);
/* One step of STOCHASTIC beam search (Kool, van Hoof, Welling 2019): the W beams of a group become W sequences drawn without
 * replacement from the policy's sequence distribution.  Groups, batch fields, logits, parent, action, load_index, the empty-slot
 * conventions, determinism, PDL and graph capture are those of ge_beam_expand.  Per beam b the inputs are
 *   logp[b]      phi_b, the float32 sum of its masked log-probs (ge_beam_expand's score);
 *   key[b]       T_b, its perturbed log-prob (conditioned Gumbel value); -inf marks a DEAD beam;
 *   node_key[b]  a 64-bit key of the beam's tree node (its action prefix).
 * Beam b contributes nothing when dead; when done[b], one STAY candidate (b, -1) carrying logp[b], key[b] and node_key[b]; otherwise
 * one candidate per valid action a, with lse_b the masked log-sum-exp of ge_masked_log_prob and, all in float32:
 *   g_a  = the Gumbel noise of ge_sample_logits with the row key replaced by node_key[b]:
 *          h = mix32(node_key[b], a, 0x85EBCA6B), u = min(fl32((h >> 8) + 0.5) / 2^24, 1 - 2^-24), g_a = -logf(-logf(u))
 *          (the float32 sum rounds to even once h >> 8 >= 2^23, as in ge_sample_logits; the clamp keeps the one u it rounds to 1,
 *          where ge_sample_logits' g is +inf, below 1, so every key is finite)
 *   s_a  = l_a + g_a (ge_sample_logits' score),  S_b = max_a s_a
 *   phi  = logp[b] + (l_a - lse_b)                                   (bit-identical to ge_beam_expand's score)
 *   x_a  = s_a - S_b <= 0,   D_b = T_b - (logp[b] + (S_b - lse_b))
 *   v_a  = (D_b - x_a) + log1mexp(x_a),   log1mexp(x) = log(-expm1(x)) for x > -ln 2, log1p(-exp(x)) otherwise
 *   G_a  = T_b - (max(v_a, 0) + log1p(exp(-|v_a|)))
 * G_a is the stable form of -log(e^-T - e^-Z + e^-(Z + x_a)), Z = logp[b] + S_b - lse_b the largest unconditioned perturbed child:
 * the children's keys conditioned on their maximum being T_b.  log1mexp(0) = -inf, so the best child inherits G = T_b exactly.
 * The child's node key is (uint64) mix32(h, a, 0x2545F491) << 32 | mix32(h ^ 0x9E3779B97F4A7C15, a, 0x6C8E9CF5), h = node_key[b].
 * graphenvs_b200.StochasticBeamSearch(venv, width, seed) starts group g (global instance i = env_id0 + g) from the root node key
 * (uint64) mix32(seed, i, 0x52DCE729) << 32 | mix32(seed ^ 0xD1B54A32D192ED03, i, 0x52DCE729) and the root key G_root = -log(-log(u)),
 * u = ((mix32(root node key, 0xFFFFFFFF, 0x85EBCA6B) >> 8) + 0.5) / 2^24, computed in float64 on the host and rounded to float32.
 * Selection: stage 1 keeps each beam's W + 1 best candidates in the order (s_a desc, a asc) (in exact arithmetic the order of G_a);
 * stage 2 fills output slot j of the group with the j-th of those lists' union in the order (G desc, parent slot asc, action asc),
 * writing parent / action / load_index as ge_beam_expand does and logp_out = phi, key_out = G, node_key_out = the child's node key
 * (-inf, -inf and 0 for an empty slot).  threshold [B / W] (may be NULL): per group the G of the (W+1)-th candidate of that order,
 * -inf when the group has at most W candidates.  Starting from one root per group (logp 0, key a Gumbel(0) draw, the other slots
 * dead), the final keys are the W largest perturbed log-probs of the complete sequences, and the largest threshold over the steps
 * is the (W+1)-th (the kappa of the inclusion probabilities q(y) = 1 - exp(-exp(phi_y - kappa))).  GE_ERR_ARG, before any CUDA
 * call, for an unknown dtype, W outside [1, 32], B % W != 0, a NULL pointer (threshold excepted), or any two overlapping arrays
 * among the ten (node_key and node_key_out hold 8 bytes per env, threshold 4 bytes per group). */
int ge_beam_expand_sampled(const ge_batch *batch, int W, const void *logits, int dtype, const float *logp, const float *key,
                           const uint64_t *node_key, float *logp_out, float *key_out, uint64_t *node_key_out, int32_t *parent,
                           int32_t *action, int32_t *load_index, float *threshold, void *stream);

/* ---- Monte Carlo tree search with PUCT selection (AlphaZero / MuZero style; csrc/ge_policy.cu) ----
 *
 * G instances are searched in parallel, each with S simulations run one after another.  Node 0 of every instance is its root;
 * simulation k (1 <= k <= S) creates at most node k of every instance, so a tree has S + 1 node slots and node n of instance g
 * sits at row n * G + g of every per-node array.  The caller keeps one env state record per node, [S + 1, G, R] (ge_state_save),
 * and a leaf batch of G envs, and runs one simulation round as
 *   ge_mcts_select(tree, k)                                   -> load_index, sel_action, depth
 *   ge_state_load(leaf, records, (S + 1) * G, load_index)     the parent node's state (a revisit loads nothing)
 *   ge_step(leaf, sel_action)                                 -1 for a revisit: GE_STEP_INVALID / AFTER_DONE, state unchanged
 *   policy(leaf) -> logits [G, A], value [G]
 *   ge_state_save(leaf, NULL, G, records + k * G * R)
 *   ge_mcts_expand(tree, k, leaf, step reward, logits, value)
 * and starts a search with ge_mcts_expand(tree, 0, ...) on the leaf batch holding the root states (and their records in row 0).
 *
 * Per node n: parent, action (of the edge into n; -1 at the root), r (float32 step reward on that edge, 0 at the root),
 * terminal (the leaf's done after that step), v (float32 policy value at expansion, 0 when terminal), N (visits) and Wsum
 * (float64 sum of backed-up returns), and over the node's VALID actions only -- its packed mask, copied from the leaf's
 * mask_bits -- the prior P(n, a) = expf(fl32(l_a - lse)) (lse the masked log-sum-exp of ge_masked_log_prob, bit for bit) and
 * child(n, a) (-1 = unexpanded).  Entries of invalid actions are never written or read.  A node slot k that round k did not
 * create (the round revisited a node) gets N = 0, parent = action = -1; every created node has N >= 1.
 * value[g] estimates the undiscounted sum of future rewards from the leaf (discount 1: episodes are finite).
 *
 * Arithmetic: float64 with explicitly rounded operations (no FMA contraction), so a plain float64 restatement is exact:
 *   Q(s, a) = r(c) + Wsum(c) / N(c)                                         for the child c of s by a
 *   qbar    = (Q - qmin) / (qmax - qmin) when qmax > qmin, else 0;  0 for an unexpanded edge      (MuZero min-max normalization)
 *   u(s, a) = qbar + ((c_puct * P(s, a)) * sqrt(N(s))) / (1 + N(s, a)),  N(s, a) = N(c), 0 when unexpanded
 * qmin / qmax (per instance, +inf / -inf at the start) run over every Q computed in a backup.
 * Select (k >= 1), one warp per instance from the root: at a node s that is terminal, or that has no valid action (a dead end),
 * stop and REVISIT s; otherwise take the valid action of largest u (ties to the lowest action); an unexpanded edge stops there
 * (EXPAND s by a), an edge into a terminal child stops there (revisit the child), any other edge descends.  A terminal or done
 * root is revisited on every simulation.  Outputs per instance: load_index = s * G + g and sel_action = a for an expansion,
 * -1 and -1 for a revisit; depth = the depth of the new or revisited node (root 0); sel_node = s or the revisited node.
 * Expand and backup (k >= 0): k = 0 makes node 0 from the leaf's current state (r = 0, terminal = done, v), resets qmin / qmax;
 * k >= 1 with sel_action[g] = a >= 0 makes node k with parent sel_node[g], action a, r = reward[g], terminal = done[g], v, and
 * sets child(s, a) = k.  Then from the new (or revisited) node with ret = its v, for each node c up to and including the root:
 *   N(c) += 1;  Wsum(c) += ret;  if c is not the root: qmin / qmax absorb r(c) + Wsum(c) / N(c), and ret = r(c) + ret.
 * So the root's expansion is its first visit (N = 1, Wsum = v) and after S simulations N(root) = S + 1.
 * No atomics and no noise: results depend only on the inputs.  Both kernels touch nothing before pdl_wait(): select launches
 * with programmatic stream serialization when tree->flags has GE_FLAG_PDL, expand when leaf->flags has it.  No allocation or
 * synchronisation: a whole search can be captured in a CUDA graph.  GE_ERR_ARG, before any CUDA call, for a NULL pointer,
 * G < 1, S < 1, A < 1, AW != ceil(A / 32), a non-finite or negative c_puct, k outside [1, S] (select) / [0, S] (expand), an
 * unknown dtype, leaf->B != G, leaf->A != A, or a NULL leaf->mask_bits / leaf->done.
 * Memory per node: R + 8 A + 4 AW + 29 bytes (record, child + prior, mask, the scalars), plus 32 bytes per instance. */
typedef struct ge_mcts_tree {
    int32_t G, S, A, AW;          /* instances, simulations, mask length and its words */
    uint32_t flags;               /* GE_FLAG_PDL: ge_mcts_select launches with programmatic stream serialization */
    double c_puct;                /* >= 0, finite */
    int32_t *parent;              /* [S + 1, G]     parent node, -1 at the root and in an unused slot */
    int32_t *action;              /* [S + 1, G]     action of the edge into the node, -1 at the root and in an unused slot */
    int32_t *visits;              /* [S + 1, G]     N */
    double *wsum;                 /* [S + 1, G]     Wsum */
    float *reward;                /* [S + 1, G]     r */
    float *value;                 /* [S + 1, G]     v */
    uint8_t *terminal;            /* [S + 1, G] */
    int32_t *child;               /* [S + 1, G, A]  valid actions only */
    float *prior;                 /* [S + 1, G, A]  valid actions only */
    uint32_t *mask;               /* [S + 1, G, AW] packed valid-action mask of the node */
    double *qmin, *qmax;          /* [G] */
    int32_t *sel_node;            /* [G] the current simulation's selection (select writes it, expand reads it) */
    int32_t *sel_action;          /* [G] */
    int32_t *load_index;          /* [G] */
    int32_t *depth;               /* [G] */
} ge_mcts_tree;
/* Selection of simulation k (1 <= k <= S): writes sel_node, sel_action, load_index and depth of every instance. */
int ge_mcts_select(const ge_mcts_tree *tree, int k, void *stream);
/* Expansion and backup of simulation k (0 <= k <= S) from the leaf batch (G envs: leaf->done, leaf->mask_bits), the step's
 * reward [G] (read for k >= 1 only, but required), the policy's logits [G, A] (layout and dtype of ge_sample_logits) and
 * value [G] float32. */
int ge_mcts_expand(const ge_mcts_tree *tree, int k, const ge_batch *leaf, const float *reward, const void *logits, int dtype,
                   const float *value, void *stream);

/* ---- Branching: per-env state records and instance replication (csrc/ge_state.cu) ----
 *
 * A RECORD is one env's state: opaque, ge_state_record_bytes(batch) bytes long (a multiple of 16).  What counts as state:
 *   GE_STATE_DYNAMIC  every non-NULL array among head, node_bits, node_bits2, edge_bits, dist32, bestkey, cost, counters, done,
 *                     mask_bits, mask_cnt (what ge_step reads and writes besides its outputs);
 *   GE_STATE_CLOCK    env_steps;
 *   GE_STATE_STATS    the env's acc column (4 doubles at stride acc_stride) and traj.
 * The step outputs, obs_x and mask_bytes are not state.  Sections come in the order of these lists; those of at most 64 bytes per
 * env first, each at its element's natural alignment, then (from a 16-byte boundary) the larger ones, each at a 16-byte offset; an
 * absent array has no section, and the record is rounded up to 16 bytes.
 * A record can be loaded only into a batch with the same kind, N, M, parenting, n_dests, n_choices and n_targets and the same set of
 * non-NULL state arrays, and it only makes sense in an env that holds the same instance it was saved from: the library checks
 * neither (the Python layer checks the first).  Record buffers are 16-byte aligned device memory; offsets are size_t (a buffer may
 * pass 2^31 bytes).  Save and load never read or write a static array, so a GE_FLAG_PDL step may follow either.  No call here
 * synchronises or allocates: they can be captured in a CUDA graph.  Arguments are checked before any CUDA call. */
#define GE_STATE_DYNAMIC 1u   /* required: what ge_step reads and writes besides its outputs */
#define GE_STATE_CLOCK 2u     /* env_steps */
#define GE_STATE_STATS 4u     /* the env's acc column (4 doubles at stride acc_stride) and traj */
#define GE_STATE_ALL 7u
/* Bytes of one record of this batch (> 0), or a negative ge_status. */
int ge_state_record_bytes(const ge_batch *batch);
/* Record i <- env env_index[i] for i in [0, count) (env i when env_index is NULL); count <= B.  Every section is written; an env
 * index outside [0, B) leaves record i untouched.  records: device [count, ge_state_record_bytes]. */
int ge_state_save(const ge_batch *batch, const int32_t *env_index, int count, void *records, void *stream);
/* For each b in [0, B): env b <- record record_index[b] (record b when record_index is NULL, which requires n_records >= B).  An
 * index < 0 or >= n_records leaves env b untouched, byte for byte.  Only the sections named in `what` are written, and `what` must
 * include GE_STATE_DYNAMIC.  A loaded env's mask_bytes is rebuilt when ge_mask_bytes_current(batch).  records must not overlap
 * the batch's arrays: an in-place fork is a save to a separate buffer followed by a load. */
int ge_state_load(const ge_batch *batch, const void *records, int n_records, const int32_t *record_index, unsigned what,
                  void *stream);
/* For each b in [0, dst->B): dst env b <- the static arrays of src env src_index[b] (src env b when src_index is NULL, which requires
 * src->B >= dst->B); an index < 0 or >= src->B leaves env b untouched.  The arrays copied are those ge_pool_refill copies, every
 * one dst carries.  dst and src may differ in B and either may be a ge_batch_slice.  GE_ERR_ARG when kind, N, M, parenting,
 * n_dests, n_choices, n_targets, max_distance or GE_FLAG_FORCE_WARP differ, when dst carries an array src lacks, when dfa_bytes
 * differ (the shared `dfa` itself is the caller's to copy) or when static ranges of dst and src overlap (no in-place gather).
 * Writes no state: follow it with ge_reset(select) or ge_state_load.  It writes static arrays, so the step after it must not be
 * launched with GE_FLAG_PDL. */
int ge_gather_instances(const ge_batch *dst, const ge_batch *src, const int32_t *src_index, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* GRAPHENVS_B200_H */
