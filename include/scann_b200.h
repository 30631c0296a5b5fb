/*
 * scann_b200.h — C ABI of libscann_b200.so: the B200-native (sm_100a) batched-search hot path of
 * sunbains/scann-rust.  This header is the drop-in boundary (SURVEY.md §8b): every entry point is
 * what a thin `extern "C"` FFI layer in the reference crate would bind for the cited Rust method.
 * Plain pointers and sizes only — no torch, no C++ types.
 *
 * Conventions
 *  - Status codes are the ordinals of the reference's `ErrorCode` (src/error.rs:10-45).
 *  - `scann_last_error()` returns a thread-local message for the last non-OK status.
 *  - Every `*_create` copies the caller's index arrays to the GPU; the caller keeps ownership of
 *    what it passed.  Every `*_search` writes caller-allocated outputs.
 *  - `memspace` says where the caller's query/result buffers live: SCANN_HOST (plain or pinned host
 *    memory; the library does the H2D/D2H copies on its stream and synchronises before returning)
 *    or SCANN_DEVICE (device pointers on the handle's device; work is enqueued on `stream` and NOT
 *    synchronised — the caller orders it, e.g. with torch's current stream).
 *  - `stream` is a cudaStream_t passed as void* (NULL = the library's own per-handle stream for
 *    SCANN_HOST calls, the legacy default stream for SCANN_DEVICE calls).
 *  - Result layout for all searchers: ids[nq*k] (u32, 0xFFFFFFFF padding), dists[nq*k] (f32, +inf
 *    padding), counts[nq] = number of valid results of each query (min(k, available)).
 *  - Handles are safe for concurrent `search` calls from several threads (tests/stress_tests.rs:256-297): calls on one
 *    handle serialise on an internal mutex while they enqueue, and their DEVICE work is ordered across streams by an
 *    event each call records and the next one waits on — a SCANN_DEVICE call returns with its kernels only enqueued
 *    and the handle's workspace is shared, so a following call on another stream starts after them.  For concurrency
 *    between searches use one handle per stream (index arrays can be shared through SCANN_TREEAH_BORROW_RAW).
 *  - There is no CPU fallback: every entry point that computes needs a CUDA device and returns
 *    SCANN_UNAVAILABLE when none is usable.
 */
#ifndef SCANN_B200_H_
#define SCANN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef int32_t scann_status;

/* src/error.rs:10-45 ErrorCode ordinals */
enum {
  SCANN_OK = 0,
  SCANN_CANCELLED = 1,
  SCANN_UNKNOWN = 2,
  SCANN_INVALID_ARGUMENT = 3,
  SCANN_DEADLINE_EXCEEDED = 4,
  SCANN_NOT_FOUND = 5,
  SCANN_ALREADY_EXISTS = 6,
  SCANN_PERMISSION_DENIED = 7,
  SCANN_RESOURCE_EXHAUSTED = 8,
  SCANN_FAILED_PRECONDITION = 9,
  SCANN_ABORTED = 10,
  SCANN_OUT_OF_RANGE = 11,
  SCANN_UNIMPLEMENTED = 12,
  SCANN_INTERNAL = 13,
  SCANN_UNAVAILABLE = 14,
  SCANN_DATA_LOSS = 15,
  SCANN_UNAUTHENTICATED = 16
};

/* src/distance_measures/mod.rs:32-66 — the three measures the hot path dispatches to SIMD kernels */
enum { SCANN_SQL2 = 0, SCANN_L2 = 1, SCANN_DOT = 2 };

enum { SCANN_HOST = 0, SCANN_DEVICE = 1 };

typedef struct scann_bf scann_bf;         /* BruteForceSearcher<f32>                     */
typedef struct scann_sq8 scann_sq8;       /* ScalarQuantizedBruteForceSearcher           */
typedef struct scann_part scann_part;     /* TreePartitioner (query side)                */
typedef struct scann_treeah scann_treeah; /* TreeXHybridSearcher / AsymmetricHasher LUT16 */
typedef struct scann_ivf scann_ivf;       /* Scann façade tree modes: Partitioned, TreeAH variant B */

const char* scann_last_error(void);
int scann_version(void);
scann_status scann_device_count(int* count);

/* ---------------------------------------------------------------------------------------------
 * BruteForceSearcher<f32>  (src/brute_force/searcher.rs:34-208)
 *   scann_bf_create  ← BruteForceSearcher::new / with_shared_dataset (:34-55); `db` is
 *                      DenseDataset::raw_data() with its row stride (data_format/dataset.rs:90-96).
 *                      n == 0 is legal (search then returns counts = 0, searcher.rs:78-80).
 *   scann_bf_search  ← search_batched (:170-208) / search (:77-93): k clamped to n; qdim != dim →
 *                      SCANN_INVALID_ARGUMENT (:83-89); nq == 0 → OK.  Dot distances are negated,
 *                      L2 is sqrt(SqL2) (:119-130).
 * ------------------------------------------------------------------------------------------- */
scann_status scann_bf_create(const float* db, size_t n, size_t dim, size_t stride, int measure, int device,
                             int memspace, scann_bf** out);
scann_status scann_bf_search(scann_bf* h, const float* queries, size_t nq, size_t qdim, size_t k, uint32_t* ids,
                             float* dists, uint32_t* counts, int memspace, void* stream);
/*   scann_bf_search_radius ← search_radius (:142-167) for a batch: every row with distance <= radius, ascending
 *                      (distance, id); ids/dists are [nq*max_results], counts[q] = rows written.  When more than
 *                      max_results rows qualify for some query the nearest max_results are written and the call
 *                      returns SCANN_RESOURCE_EXHAUSTED.  max_results < 4096; needs dim <= 256. */
scann_status scann_bf_search_radius(scann_bf* h, const float* queries, size_t nq, size_t qdim, float radius,
                                    size_t max_results, uint32_t* ids, float* dists, uint32_t* counts, int memspace,
                                    void* stream);
void scann_bf_destroy(scann_bf* h);
/* introspection: query chunks answered by the tensor-core ranking path (csrc/tc_gemm.cu + exact re-score)
 * and by the CUDA-core path (dim > 256, list overflow) since the handle was created */
scann_status scann_bf_path_stats(scann_bf* h, uint64_t* tc_chunks, uint64_t* legacy_chunks);

/* ---------------------------------------------------------------------------------------------
 * ScalarQuantizedBruteForceSearcher  (src/brute_force/scalar_quantized.rs:99-326)
 *   scann_sq8_quantize ← QuantizedDataset::from_dataset (src/quantization/scalar.rs:195-226) with
 *                        QuantizationStats::from_dataset (quantization/mod.rs:77-110) and
 *                        ScalarQuantizer::calibrate (scalar.rs:103-130): writes codes[n*dim] (i8,
 *                        levels 0..255 stored wrapped) and cal4 = {min, max, scale, inv_scale}.
 *   scann_sq8_create   ← ScalarQuantizedBruteForceSearcher::from_quantized (:116-129)
 *   scann_sq8_search   ← search_batched (:288-326): distances are q·((i8)x·scale), sign-extended,
 *                        no offset — the reference's behaviour (SURVEY §3.2), reproduced as is.
 * ------------------------------------------------------------------------------------------- */
scann_status scann_sq8_quantize(const float* db, size_t n, size_t dim, size_t stride, int8_t* codes, float* cal4,
                                int device, int memspace);
scann_status scann_sq8_create(const int8_t* codes, size_t n, size_t dim, float scale, int measure, int device,
                              int memspace, scann_sq8** out);
scann_status scann_sq8_search(scann_sq8* h, const float* queries, size_t nq, size_t qdim, size_t k, uint32_t* ids,
                              float* dists, uint32_t* counts, int memspace, void* stream);
void scann_sq8_destroy(scann_sq8* h);
scann_status scann_sq8_path_stats(scann_sq8* h, uint64_t* tc_chunks, uint64_t* legacy_chunks);

/* ---------------------------------------------------------------------------------------------
 * TreePartitioner, query side  (src/partitioning/tree_partitioner.rs:175-229)
 *   scann_part_create ← the `centers` a built TreePartitioner holds (:148-150), row-major [K*dim]
 *   scann_part_select ← Partitioner::partition (:196-229): squared-L2 to all K centres in the
 *                       reference's sequential non-fused f32 order, stable order (dist, centre id),
 *                       first L tokens + distances.  L > K pads with 0xFFFFFFFF / +inf.
 * ------------------------------------------------------------------------------------------- */
scann_status scann_part_create(const float* centers, size_t K, size_t dim, int device, int memspace,
                               scann_part** out);
scann_status scann_part_select(scann_part* h, const float* queries, size_t nq, size_t qdim, size_t L,
                               uint32_t* tokens, float* dists, int memspace, void* stream);
/* replaces the centres of an existing partitioner (same K and dim) without reallocating — the k-means trainer's
 * per-iteration refresh (csrc/build_index.cu); the caller must not run scann_part_select concurrently. */
scann_status scann_part_update(scann_part* h, const float* centers, int memspace);
void scann_part_destroy(scann_part* h);

/* ---------------------------------------------------------------------------------------------
 * Tree-AH / Tree-X-Hybrid with the LUT16 path  (src/tree_x_hybrid/mod.rs:131-364 composed with
 * src/hashes/lut16.rs:43-61,151-173 and src/hashes/lut16_simd.rs:39-141, SURVEY §3.3/§3.5)
 *   scann_treeah_create ← the arrays TreeXHybridSearcher::build leaves behind (:131-209):
 *       centers[K*dim]; codebook[S*16*ds] (ds = dim/S); packed[n*ceil(S/2)] = PackedCodes4Bit rows
 *       (low nibble = even subspace) GROUPED BY PARTITION; ids[n] = datapoint index of each row;
 *       part_offsets[K+1] row offsets; raw[N*stride] = DenseDataset::raw_data() or NULL (no
 *       reorder; results then carry the approximate LUT16 distances); num_raw = N.
 *       K == 1 with use_residuals = 0 is the flat AsymmetricHasher (src/hashes/hasher.rs:162-229).
 *   scann_treeah_search ← TreeXHybridSearcher::search (:240-294) / trait search_batched (:399-409):
 *       partition → per-leaf residual LUT16 → integer scan → top-R by approximate distance
 *       (R = pre_reorder_k) → exact `reorder_measure` distance of the R rows → top-k.
 *       cand_ids/cand_dists (optional, [nq*R]) receive the R approximate candidates in order
 *       (parity tap; pass NULL otherwise), cand_counts[nq] their number.
 *   Limits: 1 <= S <= 256, dim % S == 0, L <= 1024, R <= 2048, leaf size < 2^(32-bits(255*S)).
 * ------------------------------------------------------------------------------------------- */
scann_status scann_treeah_create(const float* centers, size_t K, size_t dim, const float* codebook, size_t S,
                                 const uint8_t* packed, const uint32_t* ids, const uint64_t* part_offsets,
                                 size_t n, const float* raw, size_t num_raw, size_t stride, int use_residuals,
                                 int reorder_measure, int device, int memspace, scann_treeah** out);
/* scann_treeah_create with layout flags (sharded / very large indexes):
 *   SCANN_TREEAH_RAW_BY_POSITION  raw holds one row per INDEX ROW in the order of packed/ids (row = part_offsets[leaf] +
 *                                 position) instead of being indexed by datapoint id — a shard keeps only its own rows
 *                                 while ids stay global (num_raw must equal n);
 *   SCANN_TREEAH_BORROW_RAW       device arrays only: raw is not copied, the caller keeps it alive until destroy. */
enum { SCANN_TREEAH_RAW_BY_POSITION = 1, SCANN_TREEAH_BORROW_RAW = 2 };
scann_status scann_treeah_create_ex(const float* centers, size_t K, size_t dim, const float* codebook, size_t S,
                                    const uint8_t* packed, const uint32_t* ids, const uint64_t* part_offsets,
                                    size_t n, const float* raw, size_t num_raw, size_t stride, int use_residuals,
                                    int reorder_measure, uint32_t flags, int device, int memspace,
                                    scann_treeah** out);
scann_status scann_treeah_search(scann_treeah* h, const float* queries, size_t nq, size_t qdim, size_t L, size_t R,
                                 size_t k, uint32_t* ids, float* dists, uint32_t* counts, uint32_t* cand_ids,
                                 float* cand_dists, uint32_t* cand_counts, int memspace, void* stream);
void scann_treeah_destroy(scann_treeah* h);
/* Restrict filter ← TreeXHybridSearcher::search_with_filter (tree_x_hybrid/mod.rs:245-250): RestrictFilter::is_allowed
 * (restricts/mod.rs:17-31) as a bitmap over datapoint ids — bit i of byte i/8 (LSB first) set = datapoint i may be
 * returned; ids >= num_ids are not allowed.  Applies to every following search on the handle (plain and split) until
 * cleared with allow_by_id = NULL.  Filtered-out points are skipped inside the LUT16 scan exactly where the reference
 * skips them (before the per-leaf top-R), so a leaf contributes its R best ALLOWED points.  Setting or clearing
 * synchronises the device; filters that belong to one call (one per query, safe across threads) are
 * scann_treeah_search_filtered's. */
scann_status scann_treeah_set_filter(scann_treeah* h, const uint8_t* allow_by_id, size_t num_ids, int memspace);
/* Per-query restrict filters of ONE call ← search_with_filter with the filter as an argument of the call: nothing is
 * stored on the handle, so concurrent calls with different filters are safe, and queries with different filters share
 * one batch.  allow = [num_filters][ceil(num_ids/8)] bytes, each row a bitmap in the convention of
 * scann_treeah_set_filter (ids >= num_ids are not allowed); query q uses row filter_of_query[q].  allow and
 * filter_of_query live in `memspace`, like the queries.  Everything else (limits, chunking, outputs, R == 0) is
 * scann_treeah_search.  Errors: INVALID_ARGUMENT for num_filters == 0, a NULL allow / filter_of_query, or (SCANN_HOST)
 * a row index >= num_filters; FAILED_PRECONDITION while a handle-wide filter is set or a split search is in flight.
 * SCANN_DEVICE does not synchronise to check the rows: a query whose row is >= num_filters is allowed nothing and
 * returns count 0. */
scann_status scann_treeah_search_filtered(scann_treeah* h, const float* queries, size_t nq, size_t qdim, size_t L,
                                          size_t R, size_t k, const uint8_t* allow, size_t num_filters, size_t num_ids,
                                          const uint32_t* filter_of_query, uint32_t* ids, float* dists,
                                          uint32_t* counts, uint32_t* cand_ids, float* cand_dists,
                                          uint32_t* cand_counts, int memspace, void* stream);
/* Per-query parameters of ONE call ← Searcher::search_batched_with_params (src/searcher.rs:164-169): query q searches
 * L_of_query[q] partitions, keeps R_of_query[q] candidates before the reorder and returns k_of_query[q] neighbours, and
 * queries with different parameters share one batch.  L, R and k are the batch maxima: they are the row strides of the
 * outputs (ids/dists [nq*k], cand_ids/cand_dists [nq*R]), size the work, and obey the limits of scann_treeah_search.
 * Each array is optional (NULL = every query uses the scalar) and lives in `memspace`, like the queries.  Row q is bit
 * for bit what scann_treeah_search returns for query q alone with (L_q, R_q, k_q), padded beyond counts[q] up to k
 * (0xFFFFFFFF / +inf) and beyond cand_counts[q] up to R; L_q > K clamps to K, and R_q == 0 gives the empty row of a
 * search with R == 0 (its distances are padded with 0x7F7F7F7F).  Nothing is stored on the handle; the handle-wide filter and scann_treeah_set_reorder apply as for
 * scann_treeah_search.  Errors: INVALID_ARGUMENT (SCANN_HOST) for an L_q outside 1..L, an R_q > R or a k_q outside
 * 1..k; FAILED_PRECONDITION while a split search is in flight.  SCANN_DEVICE does not synchronise to check the values:
 * a query with one out of range returns count 0 and cand_count 0, and the other queries are unaffected. */
scann_status scann_treeah_search_with_params(scann_treeah* h, const float* queries, size_t nq, size_t qdim, size_t L,
                                             size_t R, size_t k, const uint32_t* L_of_query, const uint32_t* R_of_query,
                                             const uint32_t* k_of_query, uint32_t* ids, float* dists, uint32_t* counts,
                                             uint32_t* cand_ids, float* cand_dists, uint32_t* cand_counts, int memspace,
                                             void* stream);
/* AsymmetricHasher::search vs ::search_with_reordering (src/hashes/hasher.rs:162-229) on one handle: enable = 0 makes the
 * following searches return the R best approximate (LUT16) distances without the exact re-score even though the handle
 * holds raw rows; enable = 1 (default) restores the re-score.  Handle-wide state, like the filter. */
scann_status scann_treeah_set_reorder(scann_treeah* h, int enable);
/* Split search for a SHARDED index (SURVEY §8e; one process per GPU, every shard sees the whole query batch).
 *   scann_treeah_search_begin: partition -> worklist -> LUT16 probe of every query's CLOSEST leaf when this shard
 *       owns it (its first 4096 points: any R points prove a bound, and a bounded probe keeps this phase short).
 *       tau_out[q] (device, nq floats) receives the R-th smallest approximate distance among them (+inf when the
 *       leaf lives on another shard or the probe saw fewer than R points).
 *   the caller min-reduces tau over the shards (e.g. ncclAllReduce MIN, 4 B per query);
 *   scann_treeah_search_end: scans all probed leaves under tau_in (device, nq floats, or NULL) — a point above
 *       tau_in[q] cannot be among the global top-R of query q because R points at or below it exist — then merges
 *       and re-scores exactly as scann_treeah_search does.
 * The bounds are data-defined (not timing-defined), so results are deterministic and every shard's list is a
 * superset of the global top-R restricted to the shard.  Device pointers only.  Between begin and end the handle is
 * BUSY, not locked: every other entry point answers SCANN_FAILED_PRECONDITION; a caller that cannot reach _end (e.g. its
 * reduction failed) calls scann_treeah_search_abort.  The batch must fit one chunk (nq*L*R*8 <= 2 GiB). */
/* `tokens` (device, nq*L u32, or NULL): the partition stage's output when the caller ran it — e.g. each shard
 * partitions nq/world queries with scann_treeah_partition and the shards all-gather the tokens, so the stage is
 * not repeated on every GPU.  The array must stay valid until scann_treeah_search_end returns.  L must be <= K. */
scann_status scann_treeah_partition(scann_treeah* h, const float* queries, size_t nq, size_t qdim, size_t L,
                                    uint32_t* tokens, void* stream);
scann_status scann_treeah_search_begin(scann_treeah* h, const float* queries, size_t nq, size_t qdim, size_t L,
                                       size_t R, size_t k, const uint32_t* tokens, float* tau_out, void* stream);
scann_status scann_treeah_search_end(scann_treeah* h, const float* tau_in, uint32_t* ids, float* dists,
                                     uint32_t* counts, void* stream);
scann_status scann_treeah_search_abort(scann_treeah* h);
/* introspection used by bench.py for the roofline arithmetic: algorithmic code bytes scanned by the
 * last scann_treeah_search call (Σ over (query, leaf) pairs of leaf_size * ceil(S/2)); host sync. */
scann_status scann_treeah_last_scan_bytes(scann_treeah* h, uint64_t* bytes, uint64_t* pairs);
/* which scan kernel served the query chunks of this handle so far: the tensor-core LUT16 scan (tcgen05.mma kind::i8 over
 * one-hot expanded codes, csrc/tcscan.cu; used when the index supports it — S a multiple of 16, S <= 64 — and a leaf is
 * probed by >= 12 queries of the batch on average; SCANN_SCAN_TC=0/1 overrides) or the register-LUT kernel.  Both
 * compute the same u32 sums and return identical results. */
scann_status scann_treeah_path_stats(scann_treeah* h, uint64_t* tc_chunks, uint64_t* lut_chunks);
/* tensor-core scan share of the profile (valid while profiling is enabled, call BEFORE scann_treeah_get_profile, which
 * resets the accumulators): milliseconds of the LUT-tile build kernel and of the tcgen05 scan kernel summed over their
 * launches, the number of launches, and the algorithmic (query, point) pairs of the LAST search's tensor-core part
 * (Σ over its (query, leaf) pairs of the leaf size; x S*16 x 2 = integer operations of the one-hot contraction). */
scann_status scann_treeah_tc_profile(scann_treeah* h, double* lut_ms, double* scan_ms, uint64_t* launches,
                                     uint64_t* pair_points);
/* live per-stage device timing for the roofline (CUDA events recorded on the search stream around each
 * stage; no host synchronisation while enabled).  get_profile synchronises, returns the milliseconds
 * accumulated since set_profiling(h, 1) / the previous get_profile as ms4 = {partition, worklist,
 * lut16 scan, merge+reorder} and the number of kernel launches, and resets the accumulators. */
scann_status scann_treeah_set_profiling(scann_treeah* h, int enable);
scann_status scann_treeah_get_profile(scann_treeah* h, double* ms4, uint64_t* kernel_launches);

/* ---------------------------------------------------------------------------------------------
 * The Scann façade's tree modes that score EVERY member of the probed leaves (src/scann.rs:175-294)
 *   scann_ivf_create ← what Scann::with_config leaves behind for SearchMode::Partitioned / TreeAH (:70-137):
 *       centers[K*dim]; ids[n] = TreePartitioner::partition_indices concatenated; part_offsets[K+1];
 *       raw[num_raw*stride] (DenseDataset::raw_data, may be NULL for TreeAH without reorder);
 *       codebook[S*C*ds] + codes_by_id[num_raw*S] = AsymmetricHasher's global (non-residual) codebook and
 *       encoded_database (hashes/hasher.rs:109-160), C <= 256 codes per block, or both NULL.
 *   scann_ivf_search, mode 0 ← Scann::search_partitioned (:215-253): partition → exact `measure` distance of every
 *       member of the L leaves (single-pair AVX2 order, bit-identical) → stable sort → first k.
 *   scann_ivf_search, mode 1 ← Scann::search_tree_ah (:256-294): partition → one f32 LookupTable of the query
 *       (hashes/lut.rs:47-82) → sequential f32 sum per member → stable sort → first k.  K = 1, L = 1 is the scoring
 *       of AsymmetricHasher::search (hashes/hasher.rs:162-185).
 *   reorder_measure >= 0 ← ReorderingHelper::reorder (utils/reordering.rs:23-54) of the k results as
 *       Scann::search_impl applies it (:198-209); -1 = off.
 * ------------------------------------------------------------------------------------------- */
scann_status scann_ivf_create(const float* centers, size_t K, size_t dim, const uint32_t* ids,
                              const uint64_t* part_offsets, size_t n, const float* raw, size_t num_raw, size_t stride,
                              const float* codebook, size_t S, size_t C, const uint8_t* codes_by_id, int device,
                              int memspace, scann_ivf** out);
scann_status scann_ivf_search(scann_ivf* h, int mode, const float* queries, size_t nq, size_t qdim, size_t L, size_t k,
                              int measure, int reorder_measure, uint32_t* ids, float* dists, uint32_t* counts,
                              int memspace, void* stream);
void scann_ivf_destroy(scann_ivf* h);

/* ---------------------------------------------------------------------------------------------
 * Parity taps for the LUT16 pieces (bit-exact targets of BASELINE.json)
 *   scann_lut16_build ← Lut16LookupTables::from_query (hashes/lut16.rs:151-173) →
 *       Lut16SimdTables::from_float_tables (hashes/lut16_simd.rs:39-90): for each query (optionally
 *       minus centroids[leaf_of_query[i]]) the u8 table lut8[nq*S*16] and {bias, multiplier}.
 *   scann_lut16_scan  ← lut16_distances_batch (src/simd/dispatch.rs:246-295): u32 sums[n] of one
 *       u8 table over PackedCodes4Bit rows.
 * ------------------------------------------------------------------------------------------- */
scann_status scann_lut16_build(const float* codebook, size_t S, size_t ds, const float* queries, size_t nq,
                               const float* centroids /* [nq*dim] or NULL */, uint8_t* lut8, float* bias,
                               float* mult, int device, int memspace);
scann_status scann_lut16_scan(const uint8_t* packed, size_t n, size_t S, const uint8_t* lut8, uint32_t* sums,
                              int device, int memspace);

/* ---------------------------------------------------------------------------------------------
 * Parity tap for the tensor-core ranking contraction (csrc/tc_gemm.cu; tcgen05 + TMEM + TMA) that stands in
 * for the inner loops of BruteForceSearcher::compute_distances (src/brute_force/searcher.rs:113-139),
 * ScalarQuantizedBruteForceSearcher::compute_distances (src/brute_force/scalar_quantized.rs:204-246) and
 * TreePartitioner::compute_center_distances (src/partitioning/tree_partitioner.rs:175-194) as a RANKING
 * device: v[q][r] = hx[r] - bf16(q * qscale) . bf16(x_r) with f32 accumulation; hx = |x_r|^2 / 2 (of
 * (i8)x * scale for rows_i8) when want_norm, else 0; qscale = scale for i8 rows, 1 otherwise.
 *   thr == NULL: dense[nq*n] receives every score.
 *   thr != NULL: the rows with v <= thr[q] are appended to cand[q*cap ...] as (ordered_key(v) << 32 | row) in
 *                arbitrary order; cand_cnt[q] counts them (values above cap mean overflow: only cap were stored).
 * Host buffers only.  No value this tap returns is ever a search result: the searchers re-score the survivors
 * exactly in the reference's summation order.
 * ------------------------------------------------------------------------------------------- */
scann_status scann_tc_scores(const float* queries, size_t nq, size_t dim, const void* rows, int rows_i8, size_t n,
                             size_t stride, float scale, int want_norm, const float* thr, float* dense,
                             uint64_t* cand, size_t cap, uint32_t* cand_cnt, int device);

/* ---------------------------------------------------------------------------------------------
 * Index-build helpers with the reference's exact semantics (SURVEY §8f-1, needed to build the
 * 10M-row bench index on the GPU)
 *   scann_pq_encode ← Codebook::encode (hashes/codebook.rs:82-95,205-215) of x - centers[assign]
 *       (tree_x_hybrid/mod.rs:177-189; assign NULL → no residual) followed by
 *       PackedCodes4Bit::from_codes (hashes/lut16.rs:43-61): packed[n*ceil(S/2)].
 * ------------------------------------------------------------------------------------------- */
scann_status scann_pq_encode(const float* codebook, size_t S, size_t ds, const float* x, size_t n, size_t stride,
                             const float* centers, const uint32_t* assign, uint8_t* packed, int device,
                             int memspace);

/* ---------------------------------------------------------------------------------------------
 * Index build inside the library (SURVEY §8f-1; csrc/build_index.cu) — the training side of the searchers.
 * The reference seeds its k-means++ from an unpinned rand::StdRng (src/utils/random.rs:20-46), so centroids are
 * not reproducible by anybody; what HAS reference semantics (assignment = TreePartitioner::partition(x, 1), residual
 * encode = Codebook::encode, packing = PackedCodes4Bit::from_codes) runs through the exact kernels of the search path.
 *   scann_kmeans_fit   <- KMeans::fit (src/trees/kmeans.rs:166-432): Lloyd's algorithm from K distinct pseudo-random rows,
 *       exact nearest-centre assignment (ties -> lower id), f64 cluster sums, empty clusters re-seeded; centers[K*dim].
 *       balance_ratio > 1: BALANCED training — Lloyd places K - K/8 centres, then the heaviest cluster is bisected
 *       (2-means on its own rows) until K centres exist.  High-dimensional data has hub clusters that Lloyd never
 *       leaves; bisection keeps every leaf within a few times the mean (and within the LUT16 scan's in-leaf position
 *       limit) and evens the probe load.  <= 1 = plain Lloyd (what Codebook::train uses).
 *   scann_pq_train     <- Codebook::train (src/hashes/codebook.rs:146-202): one 16-code k-means per subspace (seed + s)
 *       over x, or over x - centers[assign] when centers/assign are given (tree_x_hybrid/mod.rs:177-189);
 *       codebook[S*16*(dim/S)].  dim % S != 0 -> SCANN_INVALID_ARGUMENT (codebook.rs:154-159).
 *   scann_treeah_build <- TreeXHybridSearcher::build (src/tree_x_hybrid/mod.rs:131-209) / AsymmetricHasher::build
 *       (src/hashes/hasher.rs:109-159, K = 1 and use_residuals = 0): train on `train_rows` distinct rows (0 = all),
 *       assign + encode + pack every row, group rows by partition in ascending id, return a ready searcher;
 *       keep_raw != 0 keeps the rows for the exact reorder.
 *   scann_ivf_build    <- Scann::init_partitioning (src/scann.rs:140-152): centres + partition_indices -> the searcher of
 *       Scann::search_partitioned (scann_ivf_search mode 0).
 * x is host or device memory per `memspace`; everything is computed on `device`.
 * ------------------------------------------------------------------------------------------- */
scann_status scann_kmeans_fit(const float* x, size_t n, size_t dim, size_t stride, size_t K, int iters, uint64_t seed,
                              float balance_ratio, float* centers, int device, int memspace);
scann_status scann_pq_train(const float* x, size_t n, size_t dim, size_t stride, const float* centers,
                            const uint32_t* assign, size_t num_centers, size_t S, int iters, uint64_t seed,
                            float* codebook, int device, int memspace);
scann_status scann_treeah_build(const float* x, size_t n, size_t dim, size_t stride, size_t K, size_t S,
                                size_t train_rows, int kmeans_iters, uint64_t seed, int use_residuals,
                                int reorder_measure, int keep_raw, int device, int memspace, scann_treeah** out);
scann_status scann_ivf_build(const float* x, size_t n, size_t dim, size_t stride, size_t K, int kmeans_iters,
                             uint64_t seed, int device, int memspace, scann_ivf** out);

/* ---------------------------------------------------------------------------------------------
 * KMeansTree  (src/trees/kmeans_tree.rs) — hierarchical k-means partitioning (SURVEY §8 a7)
 *   The tree is flattened in PREORDER: node i has centers[i*dim..], depth[i]; its children are the node ids
 *   children[child_begin[i] .. child_begin[i] + child_count[i]) in stored order (child_count 0 = leaf).
 *   scann_kmtree_create        <- a tree built elsewhere (e.g. by the reference's KMeansTree::build, :179-280)
 *   scann_kmtree_build         <- KMeansTree::build with KMeansTreeConfig{num_children, max_depth, min_leaf_size,
 *                                 kmeans_max_iterations, seed} (:17-41): the reference's recursion and leaf rules, node
 *                                 centres = f64 mean of the node's points in index order; the k-means is the library's
 *                                 (the reference's k-means++ RNG stream is unpinned).  "Cannot build tree from empty dataset".
 *   scann_kmtree_search_leaves <- KMeansTree::search_leaves (:302-355) for a batch: depth-first walk, children by ascending
 *                                 (distance, stored index), stop at 2k collected leaves, stable sort by distance, first k.
 *                                 leaf_nodes[nq*k] = node ids (0xFFFFFFFF padding), dists / depths optional, counts[nq].
 *   scann_kmtree_info / _export: sizes, then the arrays (any pointer may be NULL); leaf_begin/leaf_count[num_nodes] and
 *                                 leaf_points[num_points] give KMeansTreeNode::datapoint_indices of the leaves (built trees).
 * ------------------------------------------------------------------------------------------- */
typedef struct scann_kmtree scann_kmtree;
scann_status scann_kmtree_create(const float* centers, const uint32_t* depth, const uint32_t* child_begin,
                                 const uint32_t* child_count, const uint32_t* children, size_t num_nodes,
                                 size_t num_child_entries, size_t dim, int device, scann_kmtree** out);
scann_status scann_kmtree_build(const float* x, size_t n, size_t dim, size_t stride, size_t num_children,
                                size_t max_depth, size_t min_leaf_size, int kmeans_iters, uint64_t seed, int device,
                                int memspace, scann_kmtree** out);
scann_status scann_kmtree_info(scann_kmtree* h, size_t* num_nodes, size_t* num_leaves, size_t* num_child_entries,
                               size_t* num_points, size_t* dim);
scann_status scann_kmtree_export(scann_kmtree* h, float* centers, uint32_t* depth, uint32_t* child_begin,
                                 uint32_t* child_count, uint32_t* children, uint32_t* leaf_begin, uint32_t* leaf_count,
                                 uint32_t* leaf_points);
scann_status scann_kmtree_search_leaves(scann_kmtree* h, const float* queries, size_t nq, size_t qdim, size_t k,
                                        uint32_t* leaf_nodes, float* dists, uint32_t* depths, uint32_t* counts,
                                        int memspace, void* stream);
void scann_kmtree_destroy(scann_kmtree* h);

/* ---------------------------------------------------------------------------------------------
 * Multi-GPU merge (SURVEY §8e): k-way merge of `parts` per-shard result lists laid out
 * [parts][nq][k] (as produced by an all-gather of each rank's ids/dists) into [nq][k], ordered by
 * (distance, id); padding entries (id 0xFFFFFFFF) are ignored.
 * ------------------------------------------------------------------------------------------- */
scann_status scann_merge_topk(const uint32_t* ids_in, const float* dists_in, size_t parts, size_t nq, size_t k,
                              uint32_t* ids_out, float* dists_out, uint32_t* counts_out, int device, int memspace,
                              void* stream);
/* The same merge over ONE gathered device buffer laid out [parts][2][nq][k] (32-bit words): each part is a rank's
 * ids block followed by its distances block, i.e. the result of a single all-gather of a packed per-rank buffer. */
scann_status scann_merge_topk_packed(const uint32_t* packed, size_t parts, size_t nq, size_t k, uint32_t* ids_out,
                                     float* dists_out, uint32_t* counts_out, int device, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SCANN_B200_H_ */
