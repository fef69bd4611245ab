/*
 * zebra_b200.h -- C ABI of the B200-native replacement for Zebra's query hot path.
 *
 * The reference (emmyoh/zebra) has no FFI today: its operator interface is the Rust type
 * `LSHIndex<N>` (src/database/index/lsh.rs:145-566) driven by `Database<N, Met, Mod>`
 * (src/database/core.rs:205-213, :245-254, :290-313) and the metric structs of src/distance.rs.
 * Each entry point below names the reference item it replaces; INTEGRATION.md shows the Rust
 * `extern "C"` block and the changed method bodies a maintainer would add.
 *
 * Conventions
 *   - every function returns 0 (ZB_OK) or a negative zb_status; zb_last_error() gives the message of the
 *     calling thread's last failure.  There is NO CPU fallback: without a usable sm_100 device (or without the
 *     CUDA kernels in this library) zb_index_create fails with ZB_ERR_NO_DEVICE.
 *   - the caller owns every buffer; pointers named h_* / plain are HOST memory, d_* are DEVICE memory on
 *     the index's device.  No torch (or other framework) types cross this boundary.
 *   - vectors are `dim` contiguous f32 (Embedding<N>, src/lib.rs:16-48); ids are 16 bytes (uuid::Uuid,
 *     big-endian byte order = Ord); every row also has a u64 ORDINAL (its global insertion index), which is
 *     what ties are broken by and what the *_ordinals outputs carry.  Library-minted ids are UUIDv7 whose
 *     byte order equals ordinal order.
 *   - distances are DistanceUnit = u64 = IEEE bit patterns (src/distance.rs:13; f64 bits for cosine / L2 / L2 squared,
 *     zero-extended f32 bits for the scalar metrics), sorted as unsigned integers exactly like lsh.rs:318 / :561, ties
 *     by id ascending.
 *   - a handle is internally serialised (one mutex): calls from any thread are safe; batch for throughput.
 */
#ifndef ZEBRA_B200_H
#define ZEBRA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ZB_ABI_VERSION 2

typedef struct zb_index zb_index;

typedef enum zb_status {
    ZB_OK = 0,
    ZB_ERR_INVALID = -1,   /* bad argument */
    ZB_ERR_CUDA = -2,      /* CUDA runtime / kernel failure */
    ZB_ERR_NO_DEVICE = -3, /* no CUDA device of compute capability 10.x */
    ZB_ERR_OOM = -4,       /* host or device allocation failed */
    ZB_ERR_STATE = -5,     /* call not valid in this state (e.g. hash before any tree exists) */
    ZB_ERR_COMM = -6       /* NCCL / sharding failure */
} zb_status;

/* Metrics.  0..2 are the north-star path: src/distance.rs:17-32 (Cosine, literal Q4 semantics:
 * (1 - simsimd cosine distance).to_bits()), :36-49 (L2Squared), :101-114 (L2); DistanceUnit = f64 bits.
 * 3..11 are the reference's scalar metrics (the `distances` crate, one f32 fold per pair in element order;
 * DistanceUnit = f32 bits zero-extended, NaN = 0xFFC00000): :51-61 Chebyshev, :63-73 Canberra, :75-85 Bray-Curtis,
 * :87-97 Manhattan, :116-126 L3, :128-138 L4, :140-157 Hamming (popcount over the low byte of every element's
 * bits; DistanceUnit = the count), :159-173 Minkowski and :175-190 p-norm (power in zb_options.metric_power,
 * 0..64; MinkowskiDistance::default() has power 0).  They are served by the gather path of the scan (one thread per
 * pair); the fused leaf-tile kernel covers 0..2. */
typedef enum zb_metric {
    ZB_METRIC_COSINE = 0, ZB_METRIC_L2SQ = 1, ZB_METRIC_L2 = 2,
    ZB_METRIC_CHEBYSHEV = 3, ZB_METRIC_CANBERRA = 4, ZB_METRIC_BRAY_CURTIS = 5, ZB_METRIC_MANHATTAN = 6,
    ZB_METRIC_L3 = 7, ZB_METRIC_L4 = 8, ZB_METRIC_HAMMING = 9, ZB_METRIC_MINKOWSKI = 10, ZB_METRIC_PNORM = 11
} zb_metric;
#define ZB_METRIC_COUNT 12
#define ZB_METRIC_MAX_POWER 64

/* LSHIndexOptions (lsh.rs:124-138) plus device placement.  Zero-initialise, then set fields. */
typedef struct zb_options {
    uint32_t dim;           /* N */
    uint32_t metric;        /* zb_metric */
    uint64_t max_node_size; /* lsh.rs:126, default 5 */
    uint32_t num_trees;     /* lsh.rs:128, default 15 */
    int32_t device;         /* CUDA device ordinal */
    uint64_t seed;          /* seed of the hyperplane sampling stream (reference: unseeded rand::rng()) */
    uint32_t shard_rank;    /* this process's shard; rows with ordinal % shard_count == shard_rank live here */
    uint32_t shard_count;   /* 0 or 1 = unsharded */
    int32_t metric_power;   /* MinkowskiDistance / PNormDistance `power` (distance.rs:164, :181); ignored otherwise */
    uint32_t reserved[3];
} zb_options;

typedef struct zb_stats {
    uint64_t rows;          /* rows stored on this shard, including tombstoned ones */
    uint64_t live_rows;     /* rows on this shard not tombstoned */
    uint64_t total_rows;    /* ordinals handed out so far (all shards) */
    uint64_t nodes, planes, leaves;
    uint64_t device_bytes;  /* HBM held by this index */
    /* last zb_index_search_batch* call */
    uint64_t last_queries, last_visits, last_pairs;   /* pairs = scored (query, row) pairs on this shard */
    uint64_t last_tile_visits, last_tile_pairs;       /* part handled by the fused leaf-tile scan kernel */
    uint64_t last_moved_bytes;                        /* HBM bytes the scan asks for by design (rows, per tile) */
    float last_ms_plan, last_ms_scan, last_ms_select, last_ms_merge, last_ms_total;
    uint32_t last_scan_launches, last_total_launches;
    float last_ms_tile_kernel;    /* the fused leaf-tile scan kernel alone (CUDA events around its launch) */
    uint32_t last_tiles;          /* (leaf, query tile) tiles it processed */
    uint32_t last_filter_flagged; /* L2 dot-product filter: visits of the last batch whose leaf the second pass rescanned exactly */
    uint64_t last_unique_bytes;   /* floor of the scan's HBM traffic: row bytes of the DISTINCT leaves the tile kernel visited */
    uint32_t last_filter_rows;    /* L2 dot-product filter: rows whose exact distance the second pass evaluated */
    float last_ms_refine;         /* ... and the duration of that pass (refine_visits_kernel) */
    uint32_t last_filter_used;    /* 1: the last batch's L2 / L2 squared visits went through the filter */
} zb_stats;

const char* zb_last_error(void);
int zb_abi_version(void);
int zb_device_count(int* out_count);

/* LSHIndex::new (lsh.rs:162-167).  Creates an empty index on options->device. */
int zb_index_create(const zb_options* options, zb_index** out_index);
int zb_index_destroy(zb_index* index);
/* The options the index was created with. */
int zb_index_options(zb_index* index, zb_options* out);

/* LSHIndex::add (lsh.rs:440-466; build_index :411-429 when no tree exists yet, insert :350-382 otherwise).
 * rows: n*dim f32.  ids16: n*16 bytes or NULL (library mints UUIDv7).  out_ids16 / out_ordinals: optional.
 * Sharded index: every rank passes the SAME n rows; each keeps the rows it owns. */
int zb_index_add(zb_index* index, uint64_t n, const float* rows, const uint8_t* ids16, uint8_t* out_ids16,
                 uint64_t* out_ordinals);
/* Same, rows already resident in HBM (d_rows: n*dim f32 on the index's device). */
int zb_index_add_device(zb_index* index, uint64_t n, const float* d_rows, const uint8_t* ids16, uint8_t* out_ids16,
                        uint64_t* out_ordinals);
/* Sharded bulk load without replication: this rank passes only the rows it owns plus their global ordinals
 * (each ordinal % shard_count == shard_rank, ascending); total_n = rows in the batch over all ranks. */
int zb_index_add_owned_device(zb_index* index, uint64_t n_local, const float* d_rows, const uint64_t* ordinals,
                              uint64_t total_n);

/* LSHIndex::remove (lsh.rs:473-503) with the tombstone semantics of DESIGN.md D1.
 * out_removed[i] = 1 if ids[i] was live (on any shard) and is now removed. */
int zb_index_remove(zb_index* index, uint64_t n, const uint8_t* ids16, uint8_t* out_removed);
int zb_index_remove_ordinals(zb_index* index, uint64_t n, const uint64_t* ordinals, uint8_t* out_removed);

/* LSHIndex::deduplicate (lsh.rs:270-288): removes every row whose f32 bit patterns equal those of a row that comes
 * earlier in id order (the reference walks its key-value store in key order and keeps the first of each pattern).
 * *out_count = rows removed; the first min(count, cap) of them (ordinals ascending) are written to out_ordinals /
 * out_ids16 when those are not NULL.  Sharded index: collective, rows are matched by a 128-bit hash of their bits. */
int zb_index_deduplicate(zb_index* index, uint64_t* out_count, uint64_t* out_ordinals, uint8_t* out_ids16, uint64_t cap);

/* LSHIndex::clear (lsh.rs:506-529), without quirk Q12: drops rows AND trees. */
int zb_index_clear(zb_index* index);

/* LSHIndex::no_vectors / no_trees / is_empty (lsh.rs:389-409). */
int zb_index_no_vectors(zb_index* index, int* out);
int zb_index_no_trees(zb_index* index, int* out);

/* LSHIndex::search (lsh.rs:544-565) for a whole batch -- replaces the par_iter at core.rs:299-303.
 * queries: nq*dim f32.  Outputs are [nq][top_k]; unused tail slots are filled with 0xFF bytes;
 * out_counts[q] = number of results of query q.  Any of out_ids16 / out_ordinals may be NULL. */
int zb_index_search_batch(zb_index* index, uint64_t nq, const float* queries, uint64_t top_k, uint8_t* out_ids16,
                          uint64_t* out_ordinals, uint64_t* out_dist_bits, uint32_t* out_counts);
/* Same with queries and outputs resident in HBM (the device-side leg the bench reports as `value`). */
int zb_index_search_batch_device(zb_index* index, uint64_t nq, const float* d_queries, uint64_t top_k,
                                 uint64_t* d_out_ordinals, uint64_t* d_out_dist_bits, uint32_t* d_out_counts);
/* The same call in its scalable form for a sharded index (shard_count = G > 1; collective, every rank calls it with the
 * same nq_total and top_k): the batch of nq_total queries is cut into G contiguous slices of nqp = ceil(nq_total / G)
 * queries, rank r fronts slice r = queries [r * nqp, min(nq_total, (r + 1) * nqp)).  `queries` holds ONLY that slice and
 * the outputs receive ONLY its results ([slice][top_k]), so the host<->device traffic of a rank is 1/G of the batch: the
 * slices are exchanged between the GPUs (ncclAllGather over NVLink), every rank scores the visits of the leaves it owns,
 * and the per-query local lists travel to the rank that fronts the query.  Replaces the same par_iter (core.rs:299-303),
 * one slice of `vectors` per process.  On an unsharded index it is zb_index_search_batch. */
int zb_index_search_slice(zb_index* index, uint64_t nq_total, const float* slice_queries, uint64_t top_k, uint8_t* out_ids16,
                          uint64_t* out_ordinals, uint64_t* out_dist_bits, uint32_t* out_counts);
int zb_index_search_slice_device(zb_index* index, uint64_t nq_total, const float* d_slice_queries, uint64_t top_k,
                                 uint64_t* d_out_ordinals, uint64_t* d_out_dist_bits, uint32_t* d_out_counts);
/* Double buffering for a caller that streams batches (a server looping over Database::query_vectors, core.rs:290-313):
 * starts the host-to-device copy of the `n` query rows at `queries` on the index's copy stream and returns at once.  The next
 * zb_index_search_batch / zb_index_search_slice call that is handed the SAME pointer (and at most `n` rows) finds its queries
 * in HBM, so the upload of batch i + 1 overlaps the scan of batch i.  Two uploads may be pending; the buffer must stay
 * unchanged (and, for the copy to be asynchronous, pinned) until that search call returns.  Purely an optimisation: a search
 * call whose pointer was not announced uploads its queries itself, and results never depend on it. */
int zb_index_search_prefetch(zb_index* index, uint64_t n, const float* queries);

/* Exact (brute-force) search: for each query the top_k smallest (DistanceUnit bits, ordinal) pairs over EVERY live (not
 * removed) row of the index, in the order LSHIndex::search sorts its candidates (lsh.rs:557-564), literal cosine of quirk
 * Q4 included -- the ground truth the LSH search's recall is measured against.  Output layout, 0xFF tail fill, out_counts
 * and the NULL-able outputs are those of zb_index_search_batch / zb_index_search_batch_device; top_k = 0 gives counts 0.
 * Distances are bit-identical to Metric::distance of the pair, so a row both searches return carries the same bits.  The
 * forest is not used: the scan reads the stored rows, ordinals and tombstones; an index without live rows gives counts 0.
 * Served for metrics 0..2 with 1 <= top_k <= 128 and rows of at most 4672 padded dimensions (top_k <= 32) or 4384
 * (top_k 33..128), the shapes of the fused leaf-tile kernel (227 KB of shared memory per block); anything else -- a scalar
 * metric, top_k > 128, a longer row -- returns ZB_ERR_INVALID.  Queries are processed in chunks whose workspace (visit
 * arrays, lists, the dot-product filter's candidates, a sharded call's gathered lists) stays within 256 MiB (knob
 * "exact_budget_mb"), whatever nq is.  It leaves zb_stats alone: zb_index_stats still describes the last LSH batch.
 * Sharded index: collective; every rank passes the same nq queries and receives the full results. */
int zb_index_search_exact(zb_index* index, uint64_t nq, const float* queries, uint64_t top_k, uint8_t* out_ids16,
                          uint64_t* out_ordinals, uint64_t* out_dist_bits, uint32_t* out_counts);
int zb_index_search_exact_device(zb_index* index, uint64_t nq, const float* d_queries, uint64_t top_k,
                                 uint64_t* d_out_ordinals, uint64_t* d_out_dist_bits, uint32_t* d_out_counts);

/* Multi-probe search (this project's extension, DESIGN.md 3.9): raises recall without more trees by also visiting, in every
 * tree, the leaves just across the query's closest hyperplanes.  probes = P, 0 <= P <= ZB_MAX_PROBES; P = 0 is exactly the
 * plain call.  For P > 0, per query and tree:
 *   1. tree_result runs unchanged (count cascade Q1, per-visit n' of Q2); its candidates are kept.
 *   2. On the main path (the walk's first root-to-leaf descent) every inner node gets the margin key |v| / sqrt(n2), in f64
 *      with IEEE round-to-nearest: v = (f64)dot(coef, q) + (f64)constant (the value point_is_above tests), n2 = (f64)
 *      dot(coef, coef), both canonical f32 dots; key = +inf if v is NaN or n2 is 0 or not finite.
 *   3. The min(P, path length) nodes with the smallest (key, depth) -- the shallower node first on equal keys -- are flipped:
 *      from each one's other child the walk descends greedily (no further flips) to one probe leaf.  The probe leaves are
 *      distinct from each other and from the main leaf.
 *   4. A probe leaf with live rows contributes its min(live, top_k) nearest live rows, like a visit with n' = top_k; an empty
 *      one contributes nothing and is not replaced.
 *   5. The result is the top_k of the deduplicated union, in LSHIndex::search's order.
 * The candidates of P + 1 include those of P, so recall never falls as P grows.  Every metric and scan path takes probes.
 * zb_stats describes a probe batch like any other (last_visits / last_pairs include the probe visits).  Layout, 0xFF tail
 * fill, NULL-able outputs, prefetch and sharding are those of the plain calls; on a sharded index every rank passes the same
 * probes, as it passes the same top_k.  probes > ZB_MAX_PROBES returns ZB_ERR_INVALID. */
#define ZB_MAX_PROBES 32
int zb_index_search_probe(zb_index* index, uint64_t nq, const float* queries, uint64_t top_k, uint32_t probes, uint8_t* out_ids16,
                          uint64_t* out_ordinals, uint64_t* out_dist_bits, uint32_t* out_counts);
int zb_index_search_probe_device(zb_index* index, uint64_t nq, const float* d_queries, uint64_t top_k, uint32_t probes,
                                 uint64_t* d_out_ordinals, uint64_t* d_out_dist_bits, uint32_t* d_out_counts);
/* zb_index_search_slice / zb_index_search_slice_device with probes (collective on a sharded index). */
int zb_index_search_slice_probe(zb_index* index, uint64_t nq_total, const float* slice_queries, uint64_t top_k, uint32_t probes,
                                uint8_t* out_ids16, uint64_t* out_ordinals, uint64_t* out_dist_bits, uint32_t* out_counts);
int zb_index_search_slice_probe_device(zb_index* index, uint64_t nq_total, const float* d_slice_queries, uint64_t top_k,
                                       uint32_t probes, uint64_t* d_out_ordinals, uint64_t* d_out_dist_bits,
                                       uint32_t* d_out_counts);

/* Restricted search (DESIGN.md 3.10): run a search over a caller-given set of rows, as if every other row had been removed
 * -- one tenant's documents, the rows a permission check allows, everything but what a user has already seen -- without
 * changing the index for any other caller.
 *   - A rowset is a fixed set of ordinals, fixed when it is made from a list of ordinals or ids: the listed rows, or with
 *     ZB_ROWSET_EXCLUDE every ordinal < total_rows at creation except the listed ones.  Duplicate list entries are allowed;
 *     rows added later are never in a rowset.  *out_count (NULL-able) receives the number of ordinals in the set.
 *   - An ordinal >= total_rows returns ZB_ERR_INVALID (the _device form checks on the device); from ids, an unknown id sets
 *     out_found[i] = 0 (NULL-able) and is ignored.  Any flag bit other than ZB_ROWSET_EXCLUDE returns ZB_ERR_INVALID.
 *   - Restricted search with rowset R is the plain search on the index's current state with every live row outside R treated
 *     as removed (D1): leaves count only the live rows of R (cascade Q1, per-visit n' of Q2, the probe rule of 3.9 over the
 *     same counts), only those rows become candidates, in zb_index_search_batch's order (literal cosine Q4).  This holds for
 *     every metric and scan path, probes 0..ZB_MAX_PROBES, the whole-batch and sliced forms, and the exact search (which
 *     returns the exact top_k over the live rows of R).
 *   - Coverage is taken at call time: rows removed after the rowset was made are excluded; inserts (and the leaf splits they
 *     cause) and zb_index_deduplicate are taken into account.  zb_index_clear, zb_index_load_forest, zb_index_load_flat and
 *     zb_index_import_store reuse ordinals: afterwards a rowset made earlier returns ZB_ERR_STATE.  A rowset of another index
 *     returns ZB_ERR_INVALID; rowset = NULL is the unrestricted call.
 *   - A rowset belongs to its index and holds device memory (a bit per ordinal, and what the first restricted call derives
 *     from it; counted in zb_stats.device_bytes): destroy it before the index.
 *   - Sharded index: every rank makes the rowset from the same list, as with zb_index_add; restricted searches are collective
 *     like the plain ones.
 *   - zb_stats describes a restricted LSH batch like any other; the restricted exact search leaves zb_stats alone.  The first
 *     restricted batch after the index changed (or the first one of a rowset) derives the rowset's masks and leaf counts inside
 *     its timed window: that work is part of its last_ms_plan and last_ms_total.
 * Layout, 0xFF tail fill, NULL-able outputs and the limits on top_k / probes are those of the plain calls. */
typedef struct zb_rowset zb_rowset;
#define ZB_ROWSET_EXCLUDE 1u
int zb_index_rowset_from_ordinals(zb_index* index, uint64_t n, const uint64_t* ordinals, uint32_t flags, uint64_t* out_count,
                                  zb_rowset** out_rowset);
int zb_index_rowset_from_ordinals_device(zb_index* index, uint64_t n, const uint64_t* d_ordinals, uint32_t flags,
                                         uint64_t* out_count, zb_rowset** out_rowset);
int zb_index_rowset_from_ids(zb_index* index, uint64_t n, const uint8_t* ids16, uint32_t flags, uint8_t* out_found,
                             uint64_t* out_count, zb_rowset** out_rowset);
int zb_rowset_destroy(zb_rowset* rowset);
int zb_index_search_rowset(zb_index* index, uint64_t nq, const float* queries, uint64_t top_k, uint32_t probes, zb_rowset* rowset,
                           uint8_t* out_ids16, uint64_t* out_ordinals, uint64_t* out_dist_bits, uint32_t* out_counts);
int zb_index_search_rowset_device(zb_index* index, uint64_t nq, const float* d_queries, uint64_t top_k, uint32_t probes,
                                  zb_rowset* rowset, uint64_t* d_out_ordinals, uint64_t* d_out_dist_bits, uint32_t* d_out_counts);
int zb_index_search_slice_rowset(zb_index* index, uint64_t nq_total, const float* slice_queries, uint64_t top_k, uint32_t probes,
                                 zb_rowset* rowset, uint8_t* out_ids16, uint64_t* out_ordinals, uint64_t* out_dist_bits,
                                 uint32_t* out_counts);
int zb_index_search_slice_rowset_device(zb_index* index, uint64_t nq_total, const float* d_slice_queries, uint64_t top_k,
                                        uint32_t probes, zb_rowset* rowset, uint64_t* d_out_ordinals, uint64_t* d_out_dist_bits,
                                        uint32_t* d_out_counts);
int zb_index_search_exact_rowset(zb_index* index, uint64_t nq, const float* queries, uint64_t top_k, zb_rowset* rowset,
                                 uint8_t* out_ids16, uint64_t* out_ordinals, uint64_t* out_dist_bits, uint32_t* out_counts);
int zb_index_search_exact_rowset_device(zb_index* index, uint64_t nq, const float* d_queries, uint64_t top_k, zb_rowset* rowset,
                                        uint64_t* d_out_ordinals, uint64_t* d_out_dist_bits, uint32_t* d_out_counts);

/* Bucket keys: the root-to-leaf sign path of Hyperplane::point_is_above decisions (lsh.rs:39-43 along
 * :350-366), MSB = root, 1 = above/right, for every (row, tree): out_keys/out_depths/out_leaves are
 * [n][num_trees] (a path longer than 64 keeps its last 64 bits; out_leaves is the leaf number of
 * zb_index_export_forest's numbering and is the full bucket identity). */
int zb_index_hash(zb_index* index, uint64_t n, const float* rows, uint64_t* out_keys, uint32_t* out_depths,
                  int32_t* out_leaves);
int zb_index_hash_device(zb_index* index, uint64_t n, const float* d_rows, uint64_t* d_out_keys,
                         uint32_t* d_out_depths, int32_t* d_out_leaves);

/* Forest interchange (hyperplanes as input: the reference's sampling is unseeded, survey quirk Q8).
 * nodes: n_nodes * {plane, left(below), right(above), leaf} int32 (inner: leaf = -1; leaf: plane = -1);
 * roots: num_trees node numbers; coef: n_planes*dim f32; cst: n_planes f32; leaf_off: n_leaves+1 CSR offsets
 * into members; members: row ordinals.  sizes4 = {n_nodes, n_planes, n_leaves, n_members}. */
int zb_index_forest_sizes(zb_index* index, int64_t* sizes4);
int zb_index_export_forest(zb_index* index, int32_t* nodes, int32_t* roots, float* coef, float* cst,
                           int64_t* leaf_off, uint64_t* members);
/* Replaces the index content with n rows (ordinals 0..n-1; ids16 may be NULL) and the given forest. */
int zb_index_load_forest(zb_index* index, uint64_t n, const float* rows, const uint8_t* ids16,
                         const int64_t* sizes4, const int32_t* nodes, const int32_t* roots, const float* coef,
                         const float* cst, const int64_t* leaf_off, const uint64_t* members);

/* ---------------------------------------------------------------------------------------------------------------
 * Interchange with the reference's stored values (SURVEY.md 8f row 4).  The reference keeps two fjall partitions
 * (lsh.rs:63-85): `embeddings` (key = 16 id bytes, value = bincode(legacy) of Embedding<N> = dim raw LE f32, lsh.rs:91-97)
 * and `trees` (key = 16 tree-id bytes, value = bincode(legacy) of Node<N>, lsh.rs:45-60 and :99-105), plus the `.zebra`
 * file = bincode(legacy) of DatabaseInner (core.rs:19-29, :183-190).  The host reads / writes the key-value engine (it
 * owns the fjall crate); these entry points take and produce the VALUES, so no bincode runs on the host side.
 *   Node::Inner = u32 0 | dim f32 coefficients | f32 constant | left (below) | right (above)
 *   Node::Leaf  = u32 1 | u64 count | count x (u64 16 | 16 id bytes)
 * ------------------------------------------------------------------------------------------------------------- */
/* Pure codecs (no device needed).  Flat form: nodes = n_nodes x {plane, left, right, leaf} as in
 * zb_index_export_forest, numbered in preorder (node, left subtree, right subtree); leaf_off = n_leaves + 1 offsets
 * into member_ids16 (16 bytes per member); sizes4 = {n_nodes, n_planes, n_leaves, n_members}.
 * zb_tree_blob_decode: call once with the output arrays NULL to get sizes4, then again to fill them.  Malformed,
 * truncated or over-long input returns ZB_ERR_INVALID. */
int zb_tree_blob_decode(uint32_t dim, const uint8_t* blob, uint64_t bytes, int64_t* sizes4, int32_t* nodes, float* coef,
                        float* cst, int64_t* leaf_off, uint8_t* member_ids16);
/* Encodes the subtree under `root` of a flat forest (plane / leaf numbers index coef, cst, leaf_off as given).
 * out may be NULL (size query); *out_bytes = blob size. */
int zb_tree_blob_encode(uint32_t dim, int64_t n_nodes, const int32_t* nodes, int32_t root, const float* coef,
                        const float* cst, const int64_t* leaf_off, const uint8_t* member_ids16, uint8_t* out,
                        uint64_t cap, uint64_t* out_bytes);
/* `.zebra` file: uuid (u64 16 | 16 bytes) | model (unit struct, 0 bytes) | metric (0 bytes; Minkowski / p-norm: i32
 * power) | max_node_size u64 | num_trees u64.  metric = the zb_metric the Database type was instantiated with. */
int zb_zebra_file_encode(const uint8_t* uuid16, uint32_t metric, int32_t power, uint64_t max_node_size,
                         uint64_t num_trees, uint8_t* out, uint64_t cap, uint64_t* out_bytes);
int zb_zebra_file_decode(const uint8_t* data, uint64_t bytes, uint32_t metric, uint8_t* out_uuid16, int32_t* out_power,
                         uint64_t* out_max_node_size, uint64_t* out_num_trees);

typedef struct zb_import_report {
    uint64_t rows_loaded;   /* rows now in the index (ordinals 0.. in id order) */
    uint64_t missing_ids;   /* leaf entries whose id has no embedding: vectors the reference removed (quirk Q5); skipped */
    uint64_t orphan_rows;   /* embeddings that some tree does not hold (lost updates of lsh.rs:445-462, Q11); NOT loaded:
                               re-insert them with zb_index_add so that every tree gets them */
    uint64_t nodes, planes, leaves;
    uint32_t max_depth;
    uint32_t reserved[3];
} zb_import_report;
/* A whole store -> the flat forest zb_index_load_forest takes (pure: no device).  Ordinal o is input row
 * row_order[o]; ordinals follow id order (the key order of the reference's store, so ties keep breaking by id); rows
 * some tree does not hold are left out and listed in orphan_rows (input row indices); leaf entries without an
 * embedding are dropped and counted.  zb_flat_store_view lends pointers that live until zb_flat_store_free:
 * sizes4 = {n_nodes, n_planes, n_leaves, n_members}; row_order has report.rows_loaded entries, orphan_rows
 * report.orphan_rows. */
typedef struct zb_flat_store zb_flat_store;
int zb_store_flatten(uint32_t dim, uint64_t n, const uint8_t* ids16, uint32_t n_trees, const uint8_t* const* tree_blobs,
                     const uint64_t* tree_blob_bytes, zb_flat_store** out, zb_import_report* report);
int zb_flat_store_view(const zb_flat_store* store, int64_t* sizes4, const int32_t** nodes, const int32_t** roots,
                       const float** coef, const float** cst, const int64_t** leaf_off, const uint64_t** members,
                       const uint32_t** row_order, const uint32_t** orphan_rows);
int zb_flat_store_free(zb_flat_store* store);
/* Replaces the index content with a reference store: n (id, embedding) pairs and the values of the `trees`
 * partition (n_trees must equal the index's num_trees).  Ordinals are assigned in id order (the key order of the
 * reference's store), so ties keep breaking by id.  out_orphan_ids16 (optional) receives the first orphan_cap orphan
 * ids.  Sharded index: every rank passes the same data. */
int zb_index_import_store(zb_index* index, uint64_t n, const uint8_t* ids16, const float* rows, uint32_t n_trees,
                          const uint8_t* const* tree_blobs, const uint64_t* tree_blob_bytes, zb_import_report* report,
                          uint8_t* out_orphan_ids16, uint64_t orphan_cap);
/* The store back out (unsharded index).  Rows [first_ordinal, first_ordinal + n): embedding value, id, live flag
 * (0 = removed: the reference would have deleted the key). */
int zb_index_export_rows(zb_index* index, uint64_t first_ordinal, uint64_t n, float* out_rows, uint8_t* out_ids16,
                         uint8_t* out_live);
/* Tree `tree` as the reference's blob; removed rows are left out of the leaves (DESIGN.md D1).  out may be NULL. */
int zb_index_export_tree_blob(zb_index* index, uint32_t tree, uint8_t* out, uint64_t cap, uint64_t* out_bytes);
/* All trees with ONE export of the forest: the blobs back to back in out (NULL: size query), out_blob_bytes[t] = size of
 * tree t (num_trees entries), *out_total = their sum. */
int zb_index_export_tree_blobs(zb_index* index, uint8_t* out, uint64_t cap, uint64_t* out_blob_bytes, uint64_t* out_total);

/* FLAT tables: the special case of the reference's tree (lsh.rs:46-60) in which every node at depth d of tree t shares
 * one hyperplane -- the K-bit LSH table of north_star (a).  coef = num_trees * bits planes of dim f32 (table t, bit d
 * at index t * bits + d; bit 0 is the root decision = the key's MSB), cst = their constants; 1 <= bits <= 16.  Replaces
 * the index content with n rows (ordinals 0..n-1) bucketed by the dense projection: one [rows x dim] . [dim x
 * num_trees * bits] pass of Hyperplane::point_is_above (lsh.rs:39-43) in the canonical accumulation order, sign bits
 * packed into the bucket keys with __ballot_sync.  The index then holds the equivalent forest (complete trees of depth
 * `bits`), so search / remove / export behave as for any forest; zb_index_hash* keeps using the dense projection until
 * an insert splits a leaf. */
int zb_index_load_flat(zb_index* index, uint64_t n, const float* rows, const uint8_t* ids16, uint32_t bits,
                       const float* coef, const float* cst);

int zb_index_stats(zb_index* index, zb_stats* out);
/* The CUDA stream (cudaStream_t) every kernel of this index is launched on -- for callers that time the
 * device work with their own events. */
int zb_index_stream(zb_index* index, void** out_stream);
/* Tuning knobs (tests and ablations; results never depend on them): key in {"tile_min_rows", "tile_queries", "use_tile_scan",
 * "scan_gen", "visit_slots", "seq_tile", "seq_prefetch", "hash_variant", "classify_variant", "flat_project", "quad_tile",
 * "select_variant", "bm_stage_mb", "single_exchange", "p2p_queries",
 * "l2_filter" (L2 / L2 squared with top_k <= 16 scored through the dot product + exact second pass: 0 off, 1 adaptive = default,
 *              2 always), "long_list_warps" (math warps per team of the fused scan for top_k > 32: 8 = default, 4),
 * "plan_tail" (count-cascade walkers re-walked by the latency-optimised tail kernel: 1 = default, 0),
 * "exact_budget_mb" (workspace of one query chunk of zb_index_search_exact*, MiB: 256 = default)}. */
int zb_index_set_param(zb_index* index, const char* key, int64_t value);

/* Sharding over the GPUs of one box: one process per GPU, each with its own index
 * (options.shard_rank / shard_count).  The library runs NCCL itself (allreduce of per-leaf live counts and of
 * build statistics, allgather of per-visit local top-n' lists); the host only has to carry the 128-byte
 * unique id from rank 0 to the other ranks. */
int zb_comm_unique_id(uint8_t* out_id128);
int zb_index_comm_init(zb_index* index, const uint8_t* id128);

/* The metric trait and the sign test for n independent pairs (host buffers): Metric::distance of
 * src/distance.rs (every impl, :19-190) with arguments (a = stored row, b = query), and
 * Hyperplane::point_is_above of lsh.rs:39-43.  Used by the host mirror's Metric::distance and by parity tests.
 * power: Minkowski / p-norm only. */
int zb_metric_distance_batch(int device, uint32_t metric, int32_t power, uint64_t n, uint32_t dim, const float* a,
                             const float* b, uint64_t* out_bits);
int zb_point_is_above_batch(int device, uint64_t n, uint32_t dim, const float* coef, const float* cst, const float* x,
                            uint8_t* out);

/* Synthetic data of BASELINE.md (counter-based, identical on any shard): fills d_out[n][dim] with
 * row r = first_row + i.  kind 0: uniform in [-1, 1); kind 1: clustered (centre[r % 4096] + 0.25 * noise). */
int zb_synth_fill_device(int device, float* d_out, uint64_t first_row, uint64_t row_stride, uint64_t n, uint32_t dim,
                         uint64_t seed, uint32_t kind);

#ifdef __cplusplus
}
#endif
#endif /* ZEBRA_B200_H */
