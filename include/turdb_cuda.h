/*
 * turdb_cuda.h — C ABI of libturdb_cuda.so: the B200 (sm_100a) implementation of TurDB's HNSW
 * vector-search hot path.  This is the drop-in boundary: exactly what a `turdb-cuda` Rust crate
 * binds with `extern "C"` (see INTEGRATION.md).  Plain pointers and sizes only; no exceptions or
 * aborts cross it; every entry returns an int32 status (0 = ok) and leaves a message readable
 * through turdb_cuda_last_error() (thread-local).
 *
 * Citations are into kahflane/TurDB (/root/reference).  The reference has no plugin/FFI interface
 * for this path; each entry names the Rust call site it stands behind.
 *
 * Conventions
 *   - node id  = dense u32, the i-th node allocated by allocate_node (src/hnsw/mod.rs:883-904);
 *                the host keeps the NodeId(page_no, slot) <-> dense id map.
 *   - metric   = DistanceFunction discriminant (src/hnsw/mod.rs:129-137): 0 L2, 1 Cosine, 2 IP.
 *                Distances follow select_squared_distance_fn (src/hnsw/distance.rs:438-444):
 *                L2 -> squared L2, Cosine -> 1 - cos (1.0 on a zero norm), IP -> -dot, computed in
 *                the lane order of the reference's AVX2 kernels (distance.rs:105-161,210-285) so
 *                results are bit-identical to the reference on an AVX2+FMA host.
 *   - "host"   entries take host pointers and do their own H2D/D2H copies;
 *     "_device" entries take device pointers on the index's device and enqueue on `stream`
 *                (a cudaStream_t passed as void*; NULL = the legacy default stream).
 */
#ifndef TURDB_CUDA_H
#define TURDB_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TURDB_CUDA_ABI_VERSION 2u

#define TURDB_MAX_L0_NEIGHBORS 32u    /* src/hnsw/mod.rs:126 */
#define TURDB_MAX_LEVEL_NEIGHBORS 16u /* src/hnsw/mod.rs:127 */
#define TURDB_INVALID_NODE 0xFFFFFFFFu /* NodeId::none(), src/hnsw/mod.rs:161-166 */
#define TURDB_INVALID_ROW 0xFFFFFFFFFFFFFFFFull
#define TURDB_SQL_MAX_LIMIT_PLUS_OFFSET 512u /* turdb_cuda_sql_topk_batch: limit + offset */
#define TURDB_EXACT_MAX_K 1024u              /* turdb_cuda_bruteforce_topk: k */

enum turdb_metric { TURDB_METRIC_L2 = 0, TURDB_METRIC_COSINE = 1, TURDB_METRIC_IP = 2 };

enum turdb_status {
  TURDB_OK = 0,
  TURDB_ERR_INVALID_ARGUMENT = 1,
  TURDB_ERR_DIMENSION_MISMATCH = 2, /* "query dimension {} does not match index dimension {}", mod.rs:1099-1104 */
  TURDB_ERR_CUDA = 3,
  TURDB_ERR_OUT_OF_MEMORY = 4,
  TURDB_ERR_UNSUPPORTED = 5,
  TURDB_ERR_NO_DEVICE = 6
};

typedef struct turdb_cuda_index turdb_cuda_index; /* opaque; owns the device arena + adjacency */

/*
 * The flattened graph the host uploads once.  Replaces the per-evaluation read_node() /
 * get_vector() closures of PersistentHnswIndex::search (src/hnsw/mod.rs:1111-1127): node records
 * (HnswNode, mod.rs:228-234) become fixed-stride adjacency rows, vectors a contiguous arena.
 */
typedef struct {
  uint32_t dim;            /* HnswIndex::dimensions, mod.rs:615 */
  uint32_t max_level;      /* HnswIndex::max_level, mod.rs:624 */
  uint64_t n;              /* nodes (node_count, mod.rs:625); may be 0 (empty index) */
  uint32_t entry;          /* dense id of HnswIndex::entry_point, TURDB_INVALID_NODE if None */
  uint32_t reserved;
  const float* vectors;    /* [n][dim] row-major; row i = vector of node i */
  const uint64_t* row_ids; /* [n]  HnswNode::row_id */
  const uint8_t* levels;   /* [n]  HnswNode::max_level */
  const uint32_t* l0_adj;  /* [n][32] level-0 neighbours in stored order (l0_neighbors) */
  const uint8_t* l0_cnt;   /* [n]  l0_count */
  const uint32_t* up_base; /* [n]  first upper slot of node i (slot of level l = up_base[i]+l-1), or INVALID */
  const uint32_t* up_adj;  /* [n_up_slots][16] higher_levels[l-1] in stored order */
  const uint8_t* up_cnt;   /* [n_up_slots] */
  uint64_t n_up_slots;     /* sum over nodes of levels[i] */
} turdb_cuda_graph;

/* per-query traversal counters; feed the bytes-gathered roofline (DESIGN.md §4) */
typedef struct {
  uint32_t n_dist;       /* all distance evaluations */
  uint32_t n_dist_upper; /* entry + greedy upper-level evaluations */
  uint32_t n_expanded;   /* level-0 adjacency rows read */
  uint32_t n_upper_hops; /* upper-level adjacency rows read */
} turdb_cuda_search_stats;

/* ---- library ------------------------------------------------------------------------------ */
uint32_t turdb_cuda_abi_version(void);
const char* turdb_cuda_last_error(void);
int32_t turdb_cuda_device_count(int32_t* out_count);

/* ---- index lifetime: replaces PersistentHnswIndex::open's in-memory state (mod.rs:810-859) --- */
int32_t turdb_cuda_index_create(const turdb_cuda_graph* graph, int32_t device, turdb_cuda_index** out);
int32_t turdb_cuda_index_destroy(turdb_cuda_index* idx);
int32_t turdb_cuda_index_info(const turdb_cuda_index* idx, uint64_t* n, uint32_t* dim,
                              uint32_t* max_level, uint32_t* entry, uint64_t* device_bytes);

/*
 * ---- graph construction: PersistentHnswIndex::insert_with_callback (mod.rs:999-1084) on the device -------------
 * Builds the index from `n` vectors by the reference's insert path: level = select_level(random_values[i], M)
 * (operations.rs:76-83), greedy descent over the levels above it (operations.rs:111-133), one ef_construction beam per
 * level target..0 seeded with the same, never refined entry (operations.rs:135-171), the beam's nearest 2M (level 0) /
 * M results selected, the new node keeps the first 32 / 16 and every selected neighbour that has the level gets a
 * back-link: appended while its list has room (mod.rs:275-301); when full, mode 0 (verbatim) drops it and mode 1
 * (reference-intent) re-selects the list with select_neighbors_heuristic (operations.rs:181-233).  Distances are squared
 * L2 whatever the metric (mod.rs:1031,1046).  Nodes are inserted in id order in steps of up to max_batch nodes (never
 * more than 1/8 of the graph built so far) that search the same snapshot of the graph; max_batch == 1 is the reference's
 * sequential procedure exactly (same graph as the CPU oracle, bit for bit), larger steps are the batched construction.
 * Dense node id = position in `vectors`.
 */
typedef struct {
  uint32_t dim;
  uint32_t m;               /* HnswIndex::m (2..32); m0 = 2 m (mod.rs:628-641) */
  uint32_t ef_construction; /* mod.rs:644 default 100 */
  uint32_t mode;            /* 0 verbatim, 1 reference-intent */
  uint32_t max_batch;       /* 1 .. 16384 */
  uint32_t reserved;
} turdb_cuda_build_params;

int32_t turdb_cuda_index_build(const turdb_cuda_build_params* params, uint64_t n, const float* vectors,
                               const uint64_t* row_ids, const double* random_values, int32_t device,
                               turdb_cuda_index** out);

/*
 * Appends n nodes to idx by the same insert path and parameters as turdb_cuda_index_build: the call is
 * insert_with_callback (mod.rs:999-1084) applied to each new row in order.  New dense ids are idx.n .. idx.n + n - 1;
 * steps continue the build's schedule from the current node count, and entry / max_level advance in id order.  On an
 * index without an entry the first new node only becomes it (mod.rs:1020-1023).  Appending to a graph built with the
 * same params gives the graph one build over all rows gives when the split falls on a step boundary (always with
 * max_batch == 1).  Works on built, uploaded (index_create, hnsw_file_upload) and empty indexes.
 *   - params->dim must equal the index dimension (TURDB_ERR_DIMENSION_MISMATCH); m, ef_construction and max_batch are
 *     checked as by build; idx.n + n must stay below 2^31 - 1 (TURDB_ERR_UNSUPPORTED); n == 0 is a no-op.
 *   - Device arrays grow by at least 1.5x when full, so a stream of small inserts does not copy the index every call;
 *     turdb_cuda_index_info's device_bytes reports what is allocated.  Norms and (after enable_sq8) SQ8 rows are computed
 *     for the new rows; the exact path's 16-bit copies are dropped and rebuilt by the next exact / SQL call.
 *   - Failure: validation, level and slot computation, every allocation and the upload of the new rows happen before the
 *     index changes; if any fails the index is exactly as before.  A CUDA error once the steps have started is reported
 *     as TURDB_ERR_CUDA and leaves the index unusable: destroy it.
 *   - Concurrency: a WRITER call.  The caller excludes every other call on the same index while it runs (the reference's
 *     RwLock write guard); search calls on an index are re-entrant among themselves, not with insert.  The device is
 *     synchronised before replaced buffers are freed, so work enqueued earlier on any stream finishes first.
 */
int32_t turdb_cuda_index_insert(turdb_cuda_index* idx, const turdb_cuda_build_params* params, uint64_t n,
                                const float* vectors, const uint64_t* row_ids, const double* random_values);

/*
 * Deletes nodes from idx: node_ids[0 .. n) (host array of dense node ids, the ids the visibility bitmap uses) become rows
 * the table no longer holds.  Node ids, rows and graph links stay as they are (no compaction, no repair).
 *   - Deleting a deleted node does nothing; duplicates are allowed; n == 0 only reports the count.  *out_n_deleted
 *     (nullable) receives the number of deleted nodes in the index after the call.
 *   - An id >= idx.n, or node_ids null with n > 0, is TURDB_ERR_INVALID_ARGUMENT, checked before anything changes.  The
 *     first delete allocates a bitmap of one bit per node capacity; if that fails (TURDB_ERR_OUT_OF_MEMORY) the index
 *     is unchanged.
 *   - Every read path treats a deleted row as absent from the table.  Traversals (search_batch[_device],
 *     search_batch_sq8_device, shards_search_batch) are search_filtered (search.rs:352-398) with visibility `live`, or
 *     `visible AND live` when the caller passes a bitmap: deleted nodes are traversed, never returned.  sql_topk_batch,
 *     sql_range_batch, sql_range_topk_batch and bruteforce_topk return what the same call returns on an index holding
 *     only the live rows (row ids, keys, values and counts; bruteforce's node ids stay this index's ids); sql_topk's
 *     use_index form is TopK over the rows the filtered traversal returns.
 *   - turdb_cuda_index_insert ignores deletions (the reference's insert path reads no visibility): deleted nodes stay
 *     waypoints and may receive back-links; appended rows are live.  hnsw_file_upload tombstones and export_graph are
 *     unaffected.  An index without a delete runs exactly the launches it ran before this call existed.
 *   - Concurrency: a WRITER call, like insert.  Work enqueued earlier on any stream answers as before the call (the
 *     device is synchronised before bits change in place).
 */
int32_t turdb_cuda_index_delete(turdb_cuda_index* idx, uint64_t n, const uint32_t* node_ids, uint64_t* out_n_deleted);

/* The index's graph as flat host arrays (the turdb_cuda_graph layout; counts = valid ids per row); every pointer is
 * nullable.  up_adj / up_cnt hold *n_up_slots rows (call once with only n_up_slots to size them). */
int32_t turdb_cuda_index_export_graph(turdb_cuda_index* idx, float* vectors, uint64_t* row_ids, uint8_t* levels,
                                      uint32_t* l0_adj, uint8_t* l0_cnt, uint32_t* up_base, uint32_t* up_adj,
                                      uint8_t* up_cnt, uint32_t* entry, uint32_t* max_level, uint64_t* n_up_slots);

/*
 * ---- search: PersistentHnswIndex::search (mod.rs:1092-1174) for a batch of queries ----------
 * For each query: greedy descent over levels max_level..1 (search.rs:283-309), level-0 beam search
 * with ef (search.rs:311-350), truncate to k (search.rs:245-252).  `ef` plays
 * HnswSearchContext::ef_search (search.rs:202-225).  visible == NULL -> search(); otherwise
 * search_filtered (mod.rs:1176-1273, search.rs:352-398) with one bit per NODE id
 * (bit i of word i/64 = is_visible(row_id of node i); the array holds ceil(n / 64) words).
 *
 * Outputs are [nq][k]; out_counts[q] results are valid (<= min(k, ef)), the rest are filled with
 * TURDB_INVALID_ROW / TURDB_INVALID_NODE / +inf.  Results ascend by distance.  out_node_ids,
 * out_stats may be NULL.  Empty index -> counts 0, status OK (mod.rs:1106-1109).
 * query_dim != index dim -> TURDB_ERR_DIMENSION_MISMATCH.  ef == 0 is rejected with
 * TURDB_ERR_INVALID_ARGUMENT (the reference would traverse the whole component and return
 * nothing; documented deviation).  k == 0 returns counts 0.
 */
int32_t turdb_cuda_search_batch(turdb_cuda_index* idx, const float* queries, uint32_t query_dim,
                                uint32_t nq, uint32_t k, uint32_t ef, uint8_t metric,
                                const uint64_t* visible, uint64_t* out_row_ids,
                                uint32_t* out_node_ids, float* out_dist, uint32_t* out_counts,
                                turdb_cuda_search_stats* out_stats);

int32_t turdb_cuda_search_batch_device(turdb_cuda_index* idx, const float* d_queries,
                                       uint32_t query_dim, uint32_t nq, uint32_t k, uint32_t ef,
                                       uint8_t metric, const uint64_t* d_visible,
                                       uint64_t* d_out_row_ids, uint32_t* d_out_node_ids,
                                       float* d_out_dist, uint32_t* d_out_counts,
                                       turdb_cuda_search_stats* d_out_stats, void* stream);

/*
 * ---- SQ8 arena (SURVEY.md §8f rank 4; QuantizationType::SQ8, header byte 43 = 1) ---------------------
 * enable_sq8 encodes every arena row as SQ8Vector::from_f32 does (src/hnsw/quantization.rs:68-95: per-row
 * min, scale = (max - min) / 255, code = round((v - min) / scale)) into rows of `dim` codes | pad to 4 | min f32 |
 * scale f32, row_bytes apart (a multiple of 16), on the device; out_rows (nullable, out_capacity bytes) receives
 * a copy.  search_batch_sq8_device is search_batch_device over that arena: every element is decoded as
 * SQ8Vector::decode does (min + q * scale, :108-113) and fed to the same distance chains, so its results equal
 * the FP32 search over the decoded vectors bit for bit while it gathers dim + 8 instead of 4 dim bytes per
 * distance.  The reference declares SQ8 but never wires it into the index (SURVEY §0), so that equality is
 * the parity contract.  Distances returned are distances to the DECODED vectors.  d_visible (nullable) as in
 * search_batch_device: search_filtered over the code arena.
 */
int32_t turdb_cuda_index_enable_sq8(turdb_cuda_index* idx, uint8_t* out_rows, uint64_t out_capacity,
                                    uint32_t* out_row_bytes);
int32_t turdb_cuda_search_batch_sq8_device(turdb_cuda_index* idx, const float* d_queries,
                                           uint32_t query_dim, uint32_t nq, uint32_t k, uint32_t ef,
                                           uint8_t metric, const uint64_t* d_visible,
                                           uint64_t* d_out_row_ids,
                                           uint32_t* d_out_node_ids, float* d_out_dist,
                                           uint32_t* d_out_counts,
                                           turdb_cuda_search_stats* d_out_stats, void* stream);

/* Tunables of the traversal kernel (0 = automatic).  warps_per_cta (1..4) warps cooperate on one
 * query, staging_slots (8..32) neighbour vectors are in flight per query, hash_bits sizes the
 * shared-memory visited table, segments = pieces a vector is streamed in through its staging slot. */
int32_t turdb_cuda_index_set_tuning(turdb_cuda_index* idx, uint32_t warps_per_cta,
                                    uint32_t staging_slots, uint32_t hash_bits, uint32_t segments);

/* Form of the traversal kernel: 0 automatic (by row length), 1 staged (a team of 2-4 warps per query, rows through
 * shared-memory staging by TMA bulk copies — long rows), 2 direct (one warp per query, rows gathered straight into
 * registers — short rows; FP32 arena only).  Results are identical in every form. */
int32_t turdb_cuda_index_set_traversal_form(turdb_cuda_index* idx, uint32_t form);

/*
 * ---- measurement: per-launch device times of the traversal kernel --------------------------
 * profile_begin arms a ring of `capacity` CUDA-event pairs; every later search_batch_device call on
 * this index brackets its traversal kernel (and the overflow pass) with events on the caller's stream.
 * profile_read (after the caller synchronised the stream) returns up to `cap` per-launch durations in
 * ms, oldest first, and disarms.  Used by bench.py for the roofline's kernel time.
 */
int32_t turdb_cuda_index_profile_begin(turdb_cuda_index* idx, uint32_t capacity);
int32_t turdb_cuda_index_profile_read(turdb_cuda_index* idx, float* main_ms, float* overflow_ms,
                                      uint32_t cap, uint32_t* out_n);

/* Diagnostics: enable != 0 arms 16 per-phase cycle counters inside the traversal kernel (a few
 * clock reads per hop); out16 (nullable) receives the counters accumulated since they were armed. */
int32_t turdb_cuda_index_debug_counters(turdb_cuda_index* idx, int32_t enable, uint64_t* out16);

/* Diagnostics: ceiling of the traversal's access pattern.  Launches ctas_per_sm x SMs CTAs (capped by what
 * cta_smem_bytes of shared memory per CTA lets an SM hold) that gather uniformly random whole arena rows
 * with cp.async.bulk into staging_slots slots each, `rounds` copies per slot, no dependencies and no
 * arithmetic.  out_bytes / out_ms is the random-row gather bandwidth the device sustains at that footprint. */
int32_t turdb_cuda_index_gather_probe(turdb_cuda_index* idx, uint32_t ctas_per_sm, uint32_t staging_slots,
                                      uint32_t cta_smem_bytes, uint32_t rounds, float* out_ms,
                                      uint64_t* out_bytes);

/*
 * ---- exact path: the SQL `ORDER BY vec <op> q LIMIT k` scan (TopKExec, ---------------------
 * src/sql/executor.rs:2239-2392 with the distance of :169-212) over the index's arena.
 * Tensor-core (BF16) dot-product pass used as a CERTIFIED filter, then an FP32 rerank in the reference's lane
 * order: a row is dropped only when its score lies below the (rerank_factor*k)-th best score so far by more than
 * twice a bound on the BF16 score error (from the operands' actual rounding-error norms), so no row of the exact
 * FP32 top-k can be lost; a query whose candidate buffer overflows is redone by a plain FP32 scan kernel.
 * Result = top-k by (FP32 distance, node id).  Distances follow the HNSW metric contract above (squared L2 /
 * 1-cos / -dot), NOT the SQL sqrt form.  k <= TURDB_EXACT_MAX_K; rerank_factor 0 = 1 (the band already certifies
 * k' = k; a larger factor only widens the working set — 6.5 ms against 7.4 ms per 10k queries x 1M x 384 at factor 4);
 * k*rerank_factor is clamped to 2048.  dim <= 2048 (L2: <= 2045, its 16-bit copy carries three extra columns).  Absent
 * vectors (+inf rows) evaluate to +inf.
 * The filter kernel has a one-CTA (tcgen05 cta_group::1) and a two-CTA (cta_group::2, clusters of 2) form; the library
 * picks by dimension (two-CTA above 64 dims, one-CTA when no cluster fits).  Results do not depend on the form.
 * Measurement switches (environment, read per call; never needed in production): TURDB_EXACT_PAIR=0/1 forces a form,
 * TURDB_EXACT_GROWTH=g sets the slice growth factor, TURDB_EXACT_TILE_N=128 runs 128-vector tiles over four accumulators, TURDB_EXACT_FORCE_BF16=1 (read when an index's 16-bit copy is built) forbids FP16 operands,
 * TURDB_EXACT_VERBOSE=1 prints the chosen form to stderr; TURDB_EXACT_SLACK_SCALE and TURDB_EXACT_DIAG make the filter
 * UNCERTIFIED / wrong on purpose and exist only to time its parts.
 */
int32_t turdb_cuda_bruteforce_topk(turdb_cuda_index* idx, const float* queries, uint32_t query_dim,
                                   uint32_t nq, uint32_t k, uint8_t metric, uint32_t rerank_factor,
                                   uint64_t* out_row_ids, uint32_t* out_node_ids, float* out_dist,
                                   uint32_t* out_counts);

int32_t turdb_cuda_bruteforce_topk_device(turdb_cuda_index* idx, const float* d_queries,
                                          uint32_t query_dim, uint32_t nq, uint32_t k,
                                          uint8_t metric, uint32_t rerank_factor,
                                          uint64_t* d_out_row_ids, uint32_t* d_out_node_ids,
                                          float* d_out_dist, uint32_t* d_out_counts, void* stream);

/*
 * ---- the SQL vector-scan operator: ORDER BY vec <op> '[...]' LIMIT limit OFFSET offset, batched -------
 * Replaces PhysicalOperator::TopKExec over a full scan (src/sql/planner/physical.rs:229, executor
 * src/sql/executor.rs:2239-2392) when order_by[0] is Column <op> literal: one call = nq statements against
 * the same table.  op 0 = `<->` (key sqrt(sum_f64((a-b)_f32^2))), 1 = `<=>` (key 1 - dot/(|a||b|) in f64, NULL
 * when a norm is zero): executor.rs:169-212.  `<#>` is rejected with TURDB_ERR_UNSUPPORTED — the reference
 * evaluates it to NULL for every row there (executor.rs:241).
 *
 * Result = the reference's, row for row: its heap procedure (first limit+offset rows pushed and stably sorted worst
 * first, a later row replaces the root iff STRICTLY smaller, left child preferred in the sift-down, final stable
 * ascending sort, :2248-2378) is replayed over a superset of the rows it would ever have pushed, in primary-key
 * (= dense node id) order, with keys in its f64 arithmetic and summation order — so equal keys come back in the
 * order the reference leaves them in.  The superset comes from the certified tensor-core filter (exact scan:
 * BF16 scores, threshold widened by a bound on the score error; a statement whose candidate buffers overflow — e.g.
 * thousands of rows tying with the limit-th key — is redone by a kernel that runs the reference's loop over every
 * row) or, use_index != 0, from the HNSW traversal's ef (>= limit+offset, <= 2048) best rows.  Order among NULL
 * keys is unspecified.  limit + offset <= TURDB_SQL_MAX_LIMIT_PLUS_OFFSET.
 *
 * out_* are [nq][limit]; out_counts[q] = rows returned; the rest is TURDB_INVALID_ROW / NaN.  out_proj (nullable)
 * receives the value `SELECT vec <proj_op> '[...]'` projects for each returned row (src/sql/predicate.rs:1634-1688:
 * f32, sequential; 0 `<->` sqrt(sum (a-b)^2), 1 `<=>` 1 - dot/(|a||b|) or NULL (NaN) on a zero norm, 2 `<#>` +dot),
 * widened to f64 as Value::Float holds it.
 */
int32_t turdb_cuda_sql_topk_batch(turdb_cuda_index* idx, const float* queries, uint32_t query_dim,
                                  uint32_t nq, uint32_t limit, uint32_t offset, uint8_t op, uint8_t proj_op,
                                  int32_t use_index, uint32_t ef, uint64_t* out_row_ids,
                                  double* out_keys, double* out_proj, uint32_t* out_counts);
int32_t turdb_cuda_sql_topk_batch_device(turdb_cuda_index* idx, const float* d_queries,
                                         uint32_t query_dim, uint32_t nq, uint32_t limit,
                                         uint32_t offset, uint8_t op, uint8_t proj_op,
                                         int32_t use_index, uint32_t ef, uint64_t* d_out_row_ids,
                                         double* d_out_keys, double* d_out_proj,
                                         uint32_t* d_out_counts, void* stream);

/*
 * ---- the SQL distance-range scan: WHERE vec <op> '[...]' <cmp> radius LIMIT limit OFFSET offset, batched ---------
 * Replaces a Filter over a full scan when the predicate is Column <op> literal <cmp> constant: one call = nq
 * statements against the same table, statement q with literal queries[q] and constant radius[q] (f64).  op: 0 `<->`,
 * 1 `<=>`, 2 `<#>` — the projected value of src/sql/predicate.rs:1634-1688 (f32, sequential: sqrt L2, 1 - cos with
 * NULL on a zero norm, +dot), widened to f64.  cmp: 0 `<`, 1 `<=`, 2 `>`, 3 `>=`.  Only the near direction is
 * supported (`<`/`<=` with `<->` and `<=>`, `>`/`>=` with `<#>`); any other pair is TURDB_ERR_UNSUPPORTED.
 *
 * Row i qualifies iff its value compares true against radius[q] in f64; a NULL value and an absent vector (a +inf row)
 * never do.  out_counts[q] = the number of qualifying rows; rows [offset, offset + limit) of them, in scan order
 * (= dense node id order), are written to out_row_ids [nq][limit] and their values to out_vals (nullable); unused
 * slots are TURDB_INVALID_ROW / NaN.  limit = 0 is a COUNT (out_row_ids may then be NULL).
 *
 * The certified tensor-core filter of the exact path runs one pass with a per-statement threshold derived from the
 * radius (widened by its score-error bound and a bound on the f32 evaluation error of the value), so no qualifying row
 * is dropped; its survivors are decided by the exact value.  A statement with more survivors than the candidate buffer
 * holds (DESIGN §4.6) is redone by a kernel that runs the reference's loop over every row.  Dimension limits as for
 * turdb_cuda_sql_topk_batch.
 */
int32_t turdb_cuda_sql_range_batch(turdb_cuda_index* idx, const float* queries, uint32_t query_dim, uint32_t nq,
                                   uint8_t op, uint8_t cmp, const double* radius, uint32_t limit, uint32_t offset,
                                   uint64_t* out_row_ids, double* out_vals, uint32_t* out_counts);
int32_t turdb_cuda_sql_range_batch_device(turdb_cuda_index* idx, const float* d_queries, uint32_t query_dim,
                                          uint32_t nq, uint8_t op, uint8_t cmp, const double* d_radius,
                                          uint32_t limit, uint32_t offset, uint64_t* d_out_row_ids,
                                          double* d_out_vals, uint32_t* d_out_counts, void* stream);

/*
 * ---- the nearest rows within a radius: WHERE vec <where_op> '[...]' <cmp> radius ORDER BY vec <order_op> '[...]'
 *      LIMIT limit OFFSET offset, batched (both clauses with the same literal) ------------------------------------------
 * The reference plans TopK(Filter(Scan)): its heap sees the rows that pass the Filter, in primary-key order.  One call =
 * nq such statements against the same table, statement q with literal queries[q] and constant radius[q] (f64).
 *   Filter: exactly turdb_cuda_sql_range_batch's predicate (where_op 0 `<->`, 1 `<=>`, 2 `<#>`; cmp 0 `<`, 1 `<=`,
 *           2 `>`, 3 `>=`; near direction only, other pairs TURDB_ERR_UNSUPPORTED; NULL values and absent vectors never
 *           qualify).
 *   TopK:   exactly turdb_cuda_sql_topk_batch's result over the qualifying rows, row for row, order among equal keys
 *           included: order_op 0 `<->` or 1 `<=>` (`<#>` is TURDB_ERR_UNSUPPORTED), f64 keys, out_row_ids / out_keys
 *           [nq][limit], out_proj (nullable) the value of `SELECT vec <proj_op> '[...]'`, out_counts[q] = rows returned,
 *           unused slots TURDB_INVALID_ROW / NaN, limit + offset <= TURDB_SQL_MAX_LIMIT_PLUS_OFFSET.  Order among NULL
 *           keys (e.g. WHERE `<->`, ORDER BY `<=>` on a zero-norm row) is unspecified.
 * Operators and limit + offset are checked before the index.  The range scan's single filter pass finds the candidates;
 * each statement's survivors go through the exact predicate in scan order and the replayed heap.  A statement with
 * more survivors than the candidate buffer holds is redone by the reference's loop over every row (DESIGN §4.6).
 */
int32_t turdb_cuda_sql_range_topk_batch(turdb_cuda_index* idx, const float* queries, uint32_t query_dim, uint32_t nq,
                                        uint8_t where_op, uint8_t cmp, const double* radius, uint8_t order_op,
                                        uint8_t proj_op, uint32_t limit, uint32_t offset, uint64_t* out_row_ids,
                                        double* out_keys, double* out_proj, uint32_t* out_counts);
int32_t turdb_cuda_sql_range_topk_batch_device(turdb_cuda_index* idx, const float* d_queries, uint32_t query_dim,
                                               uint32_t nq, uint8_t where_op, uint8_t cmp, const double* d_radius,
                                               uint8_t order_op, uint8_t proj_op, uint32_t limit, uint32_t offset,
                                               uint64_t* d_out_row_ids, double* d_out_keys, double* d_out_proj,
                                               uint32_t* d_out_counts, void* stream);

/*
 * ---- multi-GPU: merge of per-shard top-k after the all-gather (one sub-index per GPU) --------
 * gathered_* are [n_shards][nq][k] device arrays (the NCCL all-gather output); ties order by
 * (distance, row_id).  Output [nq][k].
 */
/* Single-process form of the same path: `shards` are sub-indexes (usually one per GPU; several on one device
 * are allowed), `queries` one host batch replicated to all of them; per-shard lists are copied device to device
 * into shard 0's gather buffer and merged there.  Results equal the multi-process (NCCL) path's. */
int32_t turdb_cuda_shards_search_batch(turdb_cuda_index* const* shards, uint32_t n_shards,
                                       const float* queries, uint32_t query_dim, uint32_t nq, uint32_t k,
                                       uint32_t ef, uint8_t metric, uint64_t* out_row_ids,
                                       float* out_dist, uint32_t* out_counts);

/* The same merge over ONE packed block per shard — row ids [nq][k] u64 | distances [nq][k] f32 | counts [nq] u32 —,
 * blocks shard_stride_bytes apart (a multiple of 8): the output of a single all-gather of every rank's block. */
int32_t turdb_cuda_merge_topk_packed_device(int32_t device, const void* d_gathered,
                                            uint64_t shard_stride_bytes, uint32_t n_shards, uint32_t nq,
                                            uint32_t k, uint64_t* d_out_row_ids, float* d_out_dist,
                                            uint32_t* d_out_counts, void* stream);

int32_t turdb_cuda_merge_topk_device(int32_t device, const uint64_t* d_gathered_row_ids,
                                     const float* d_gathered_dist, const uint32_t* d_gathered_counts,
                                     uint32_t n_shards, uint32_t nq, uint32_t k,
                                     uint64_t* d_out_row_ids, float* d_out_dist,
                                     uint32_t* d_out_counts, void* stream);

/*
 * ---- the reference's on-disk index (`.hnsw`) -> device index (SURVEY.md §8f rank 1) -----------
 * Replaces, for a GPU-served index, PersistentHnswIndex::open + rebuild_row_id_map + per-access read_node
 * (src/hnsw/mod.rs:811-859, 906-911; file layout src/hnsw/storage.rs:98-119, 322-383, 485-546; node
 * records src/hnsw/mod.rs:333-421).  Parsing is host-only (no GPU needed); `upload` calls
 * turdb_cuda_index_create.  Vectors are NOT in the file (the table owns them, mod.rs:1097): the caller
 * supplies them per dense id, or through a callback shaped like the reference's `get_vector` closure.
 *
 * Dense ids: readable active slots in (page, slot) order, then "tombstones" — NodeIds that are referenced
 * but unreadable (deleted / missing / damaged); they keep the reference's behaviour for such nodes
 * (distance +inf whatever the metric, no neighbours, row_id 0; mod.rs:1111-1127, 1159-1171): an absent vector is
 * uploaded as a row of +inf, and every kernel evaluates a row whose first element is +inf to distance +inf.
 */
typedef struct turdb_cuda_hnsw_file turdb_cuda_hnsw_file; /* opaque, host memory only */

enum turdb_hnsw_file_flags {
  TURDB_HNSW_FILE_SUSPECT_PAGES = 1u,      /* overlapping records: the 13-bit slot offset of storage.rs:338-344 */
  TURDB_HNSW_FILE_TOMBSTONES = 2u,          /* dangling NodeIds were mapped to tombstones */
  TURDB_HNSW_FILE_NODE_COUNT_MISMATCH = 4u, /* header.node_count != readable active slots */
  TURDB_HNSW_FILE_MAX_LEVEL_CLAMPED = 8u,   /* header.max_level > level of the entry node */
  TURDB_HNSW_FILE_TRAILING_BYTES = 16u      /* file length is not a multiple of the 16 KiB page */
};

typedef struct {
  uint64_t index_id, table_id;           /* storage.rs:100-101 */
  uint32_t dimensions, m, m0, ef_construction, ef_search;
  uint8_t distance_fn;                   /* 0 L2, 1 cosine, 2 inner product (storage.rs:227-233) */
  uint8_t quantization;                  /* 0 none, 1 SQ8, 2 PQ — recorded only; records are never quantised */
  uint8_t header_max_level, max_level;   /* as stored / as uploaded (clamped to the entry node's level) */
  uint8_t has_entry, reserved[3];
  uint32_t entry;                        /* dense id, TURDB_INVALID_NODE when the header has no entry point */
  uint32_t flags;                        /* turdb_hnsw_file_flags */
  uint32_t n_pages, n_foreign_pages, n_suspect_pages;
  uint64_t header_node_count, header_vector_count;
  uint64_t n_nodes, n_tombstones, n_up_slots;
  uint64_t n_deleted_slots, n_unreadable_slots;
} turdb_cuda_hnsw_file_info;

/* get_vector(row_id) -> Option<Vec<f32>> (mod.rs:1097): write `dim` floats to out and return 1, or return 0. */
typedef int32_t (*turdb_cuda_get_vector_fn)(void* user, uint64_t row_id, float* out);

int32_t turdb_cuda_hnsw_file_open(const char* path, turdb_cuda_hnsw_file** out);
int32_t turdb_cuda_hnsw_file_open_memory(const uint8_t* bytes, uint64_t len, turdb_cuda_hnsw_file** out);
int32_t turdb_cuda_hnsw_file_close(turdb_cuda_hnsw_file* file);
int32_t turdb_cuda_hnsw_file_get_info(const turdb_cuda_hnsw_file* file, turdb_cuda_hnsw_file_info* out);
/* per dense id (n_nodes + n_tombstones entries, each pointer nullable): row id, NodeId page, NodeId slot */
int32_t turdb_cuda_hnsw_file_nodes(const turdb_cuda_hnsw_file* file, uint64_t* out_row_ids,
                                   uint32_t* out_pages, uint16_t* out_slots);
/* a turdb_cuda_graph view over the file's arrays (valid until close); `vectors` is stored as given */
int32_t turdb_cuda_hnsw_file_graph(const turdb_cuda_hnsw_file* file, const float* vectors,
                                   turdb_cuda_graph* out);
/* vectors [n_nodes][dim] in dense-id order and/or get_vector; present (nullable, [n_nodes]) marks rows
 * the table still holds.  Absent vectors and tombstones are uploaded as +inf rows. */
int32_t turdb_cuda_hnsw_file_upload(const turdb_cuda_hnsw_file* file, const float* vectors,
                                    const uint8_t* present, turdb_cuda_get_vector_fn get_vector,
                                    void* user, int32_t device, turdb_cuda_index** out);

#ifdef __cplusplus
}
#endif
#endif /* TURDB_CUDA_H */
