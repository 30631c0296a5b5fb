// scann_b200.hpp — header-only C++ mirror of the reference crate's searcher API over the C ABI
// (scann_b200.h).  The reference is compiled Rust and there is no Rust toolchain in this image, so this is
// the compiled-language host side above the ABI: same type and method names, same argument meaning and
// error behaviour as the Rust types (citations relative to /root/reference):
//
//   scann::BruteForceSearcher                 src/brute_force/searcher.rs:18-209
//   scann::ScalarQuantizedBruteForceSearcher  src/brute_force/scalar_quantized.rs:82-348
//   scann::TreePartitioner                    src/partitioning/tree_partitioner.rs:18-250
//   scann::TreeXHybridSearcher (+Config)      src/tree_x_hybrid/mod.rs:23-380
//   scann::LeafScanSearcher                   src/scann.rs:215-294 (Scann::search_partitioned / search_tree_ah)
//   scann::Result<T> / ScannError / ErrorCode src/error.rs:10-147
//
// `Result<T>` carries {code, message} like `Result<T, ScannError>`; nothing throws across the ABI.
#pragma once

#include <algorithm>
#include <cstdint>
#include <limits>
#include <string>
#include <utility>
#include <vector>

#include "scann_b200.h"

namespace scann {

enum class ErrorCode : int32_t {
  Ok = 0, Cancelled, Unknown, InvalidArgument, DeadlineExceeded, NotFound, AlreadyExists, PermissionDenied,
  ResourceExhausted, FailedPrecondition, Aborted, OutOfRange, Unimplemented, Internal, Unavailable, DataLoss,
  Unauthenticated
};

struct ScannError {
  ErrorCode code = ErrorCode::Ok;
  std::string message;
};

template <class T>
struct Result {
  T value{};
  ScannError error;
  bool ok() const { return error.code == ErrorCode::Ok; }
};

inline ScannError make_error(scann_status st) {
  ScannError e;
  e.code = static_cast<ErrorCode>(st);
  if (st != SCANN_OK) e.message = scann_last_error();
  return e;
}

enum class DistanceMeasure : int { SquaredL2 = SCANN_SQL2, L2 = SCANN_L2, DotProduct = SCANN_DOT };

using DatapointIndex = uint32_t;                                    // src/types.rs:10
using NNResultsVector = std::vector<std::pair<DatapointIndex, float>>;  // src/types.rs:20

namespace detail {
inline std::vector<NNResultsVector> unflatten(const std::vector<uint32_t>& ids, const std::vector<float>& dists,
                                              const std::vector<uint32_t>& counts, size_t k) {
  std::vector<NNResultsVector> out(counts.size());
  for (size_t q = 0; q < counts.size(); ++q) {
    out[q].reserve(counts[q]);
    for (uint32_t j = 0; j < counts[q]; ++j) out[q].emplace_back(ids[q * k + j], dists[q * k + j]);
  }
  return out;
}
// &[Vec<f32>] → contiguous [nq*dim]; ragged batches are an InvalidArgument like a per-query dim mismatch
inline bool flatten(const std::vector<std::vector<float>>& queries, std::vector<float>* flat, size_t* dim) {
  *dim = queries.empty() ? 0 : queries[0].size();
  flat->clear();
  flat->reserve(queries.size() * *dim);
  for (const auto& q : queries) {
    if (q.size() != *dim) return false;
    flat->insert(flat->end(), q.begin(), q.end());
  }
  return true;
}
}  // namespace detail

// ------------------------------------------------------------------------------------------------
class BruteForceSearcher {
 public:
  // BruteForceSearcher::new(dataset, distance_measure); `data` is DenseDataset::raw_data() with `stride`
  static Result<BruteForceSearcher> create(const float* data, size_t n, size_t dim, size_t stride,
                                           DistanceMeasure measure, int device = 0) {
    Result<BruteForceSearcher> r;
    r.error = make_error(scann_bf_create(data, n, dim, stride, static_cast<int>(measure), device, SCANN_HOST, &r.value.h_));
    return r;
  }
  BruteForceSearcher() = default;
  BruteForceSearcher(BruteForceSearcher&& o) noexcept : h_(o.h_) { o.h_ = nullptr; }
  BruteForceSearcher& operator=(BruteForceSearcher&& o) noexcept {
    if (this != &o) { scann_bf_destroy(h_); h_ = o.h_; o.h_ = nullptr; }
    return *this;
  }
  BruteForceSearcher(const BruteForceSearcher&) = delete;
  ~BruteForceSearcher() { scann_bf_destroy(h_); }

  // search_batched(&[Vec<f32>], k) (searcher.rs:170-208)
  Result<std::vector<NNResultsVector>> search_batched(const std::vector<std::vector<float>>& queries, size_t k) const {
    Result<std::vector<NNResultsVector>> r;
    if (queries.empty()) return r;  // Ok(vec![])
    std::vector<float> flat;
    size_t dim;
    if (!detail::flatten(queries, &flat, &dim)) {
      r.error = {ErrorCode::InvalidArgument, "Query dimensionality does not match dataset dimensionality"};
      return r;
    }
    size_t nq = queries.size();
    std::vector<uint32_t> ids(nq * k), counts(nq);
    std::vector<float> dists(nq * k);
    r.error = make_error(scann_bf_search(h_, flat.data(), nq, dim, k, ids.data(), dists.data(), counts.data(),
                                         SCANN_HOST, nullptr));
    if (r.ok()) r.value = detail::unflatten(ids, dists, counts, k);
    return r;
  }
  // search(&[f32], k) (searcher.rs:77-93)
  Result<NNResultsVector> search(const std::vector<float>& query, size_t k) const {
    auto b = search_batched({query}, k);
    Result<NNResultsVector> r;
    r.error = b.error;
    if (b.ok() && !b.value.empty()) r.value = std::move(b.value[0]);
    return r;
  }
  // search_radius(&[T], radius) (searcher.rs:142-167): every row with distance <= radius, ascending.  max_results
  // bounds the output (ResourceExhausted when more rows qualify).
  Result<NNResultsVector> search_radius(const std::vector<float>& query, float radius, size_t max_results = 1024) const {
    Result<NNResultsVector> r;
    std::vector<uint32_t> ids(max_results), counts(1);
    std::vector<float> dists(max_results);
    r.error = make_error(scann_bf_search_radius(h_, query.data(), 1, query.size(), radius, max_results, ids.data(),
                                                dists.data(), counts.data(), SCANN_HOST, nullptr));
    if (r.ok()) r.value = detail::unflatten(ids, dists, counts, max_results)[0];
    return r;
  }

 private:
  scann_bf* h_ = nullptr;
};

// ------------------------------------------------------------------------------------------------
class ScalarQuantizedBruteForceSearcher {
 public:
  // ScalarQuantizedBruteForceSearcher::new(&dataset, config): quantise (QuantizedDataset::from_dataset) + build
  static Result<ScalarQuantizedBruteForceSearcher> create(const float* data, size_t n, size_t dim, size_t stride,
                                                          DistanceMeasure measure, int device = 0) {
    Result<ScalarQuantizedBruteForceSearcher> r;
    std::vector<int8_t> codes(n * dim);
    float cal[4];
    r.error = make_error(scann_sq8_quantize(data, n, dim, stride, codes.data(), cal, device, SCANN_HOST));
    if (!r.ok()) return r;
    r.value.scale_ = cal[2];
    r.error = make_error(scann_sq8_create(codes.data(), n, dim, cal[2], static_cast<int>(measure), device, SCANN_HOST,
                                          &r.value.h_));
    return r;
  }
  // from_quantized(quantized_dataset, distance_measure)
  static Result<ScalarQuantizedBruteForceSearcher> from_quantized(const int8_t* codes, size_t n, size_t dim, float scale,
                                                                  DistanceMeasure measure, int device = 0) {
    Result<ScalarQuantizedBruteForceSearcher> r;
    r.value.scale_ = scale;
    r.error = make_error(scann_sq8_create(codes, n, dim, scale, static_cast<int>(measure), device, SCANN_HOST, &r.value.h_));
    return r;
  }
  ScalarQuantizedBruteForceSearcher() = default;
  ScalarQuantizedBruteForceSearcher(ScalarQuantizedBruteForceSearcher&& o) noexcept : h_(o.h_), scale_(o.scale_) { o.h_ = nullptr; }
  ScalarQuantizedBruteForceSearcher& operator=(ScalarQuantizedBruteForceSearcher&& o) noexcept {
    if (this != &o) { scann_sq8_destroy(h_); h_ = o.h_; scale_ = o.scale_; o.h_ = nullptr; }
    return *this;
  }
  ScalarQuantizedBruteForceSearcher(const ScalarQuantizedBruteForceSearcher&) = delete;
  ~ScalarQuantizedBruteForceSearcher() { scann_sq8_destroy(h_); }

  Result<std::vector<NNResultsVector>> search_batched(const std::vector<std::vector<float>>& queries, size_t k) const {
    Result<std::vector<NNResultsVector>> r;
    if (queries.empty()) return r;
    std::vector<float> flat;
    size_t dim;
    if (!detail::flatten(queries, &flat, &dim)) {
      r.error = {ErrorCode::InvalidArgument, "Query dimensionality does not match dataset dimensionality"};
      return r;
    }
    size_t nq = queries.size();
    std::vector<uint32_t> ids(nq * k), counts(nq);
    std::vector<float> dists(nq * k);
    r.error = make_error(scann_sq8_search(h_, flat.data(), nq, dim, k, ids.data(), dists.data(), counts.data(),
                                          SCANN_HOST, nullptr));
    if (r.ok()) r.value = detail::unflatten(ids, dists, counts, k);
    return r;
  }
  float scale() const { return scale_; }

 private:
  scann_sq8* h_ = nullptr;
  float scale_ = 1.0f;
};

// ------------------------------------------------------------------------------------------------
struct PartitionResult {  // src/partitioning/partitioner.rs:12-21
  std::vector<uint32_t> tokens;
  std::vector<float> distances;
};

class TreePartitioner {
 public:
  static Result<TreePartitioner> from_centers(const float* centers, size_t K, size_t dim, int device = 0) {
    Result<TreePartitioner> r;
    r.value.dim_ = dim;
    r.error = make_error(scann_part_create(centers, K, dim, device, SCANN_HOST, &r.value.h_));
    return r;
  }
  TreePartitioner() = default;
  TreePartitioner(TreePartitioner&& o) noexcept : h_(o.h_), dim_(o.dim_) { o.h_ = nullptr; }
  TreePartitioner& operator=(TreePartitioner&& o) noexcept {
    if (this != &o) { scann_part_destroy(h_); h_ = o.h_; dim_ = o.dim_; o.h_ = nullptr; }
    return *this;
  }
  TreePartitioner(const TreePartitioner&) = delete;
  ~TreePartitioner() { scann_part_destroy(h_); }

  // Partitioner::partition(query, num_partitions) (tree_partitioner.rs:196-229)
  Result<PartitionResult> partition(const std::vector<float>& query, size_t num_partitions) const {
    Result<PartitionResult> r;
    if (!h_) {
      r.error = {ErrorCode::FailedPrecondition, "Partitioner not built"};
      return r;
    }
    r.value.tokens.resize(num_partitions);
    r.value.distances.resize(num_partitions);
    r.error = make_error(scann_part_select(h_, query.data(), 1, query.size(), num_partitions, r.value.tokens.data(),
                                           r.value.distances.data(), SCANN_HOST, nullptr));
    if (r.ok()) {  // drop the padding when num_partitions > K
      size_t m = 0;
      while (m < num_partitions && r.value.tokens[m] != 0xFFFFFFFFu) ++m;
      r.value.tokens.resize(m);
      r.value.distances.resize(m);
    }
    return r;
  }

 private:
  scann_part* h_ = nullptr;
  size_t dim_ = 0;
};

// ------------------------------------------------------------------------------------------------
struct SearchParameters {  // src/searcher.rs:23-77, the fields the GPU path reads (0 = not set)
  size_t num_neighbors = 0;
  size_t pre_reordering_num_neighbors = 0;
  SearchParameters& with_num_neighbors(size_t k) {
    num_neighbors = k;
    return *this;
  }
  SearchParameters& with_pre_reordering_neighbors(size_t n) {
    pre_reordering_num_neighbors = n;
    return *this;
  }
};

struct TreeXHybridConfig {  // src/tree_x_hybrid/mod.rs:23-78
  size_t num_partitions = 100;
  size_t partitions_to_search = 10;
  size_t num_subspaces = 8;       // hash_config.num_subspaces (num_codes is 16 on the LUT16 path)
  bool use_residuals = true;
  float pre_reorder_multiplier = 3.0f;
  DistanceMeasure distance_measure = DistanceMeasure::SquaredL2;  // reorder measure (hard-wired SqL2 in the reference, :124)
  size_t pre_reorder_k(size_t k) const {  // (k as f32 * multiplier) as usize (:263)
    float v = static_cast<float>(k) * pre_reorder_multiplier;
    return v <= 0.0f ? 0 : static_cast<size_t>(v);
  }
};

class TreeXHybridSearcher {
 public:
  explicit TreeXHybridSearcher(TreeXHybridConfig cfg = {}) : cfg_(cfg) {}
  TreeXHybridSearcher(TreeXHybridSearcher&& o) noexcept : cfg_(o.cfg_), h_(o.h_) { o.h_ = nullptr; }
  TreeXHybridSearcher(const TreeXHybridSearcher&) = delete;
  ~TreeXHybridSearcher() { scann_treeah_destroy(h_); }

  // the arrays TreeXHybridSearcher::build leaves behind (:131-209)
  ScannError build_from_index(const float* centers, size_t K, size_t dim, const float* codebook, size_t S,
                              const uint8_t* packed, const uint32_t* ids, const uint64_t* part_offsets, size_t n,
                              const float* raw, size_t num_raw, size_t stride, int device = 0) {
    scann_treeah_destroy(h_);
    h_ = nullptr;
    return make_error(scann_treeah_create(centers, K, dim, codebook, S, packed, ids, part_offsets, n, raw, num_raw, stride,
                                          cfg_.use_residuals ? 1 : 0, static_cast<int>(cfg_.distance_measure), device,
                                          SCANN_HOST, &h_));
  }

  Result<std::vector<NNResultsVector>> search_batched(const std::vector<std::vector<float>>& queries, size_t k) const {
    return search_impl(queries, k, cfg_.pre_reorder_k(k));
  }
  // search(&[f32], k) (:240-242)
  Result<NNResultsVector> search(const std::vector<float>& query, size_t k) const {
    auto b = search_batched({query}, k);
    Result<NNResultsVector> r;
    r.error = b.error;
    if (b.ok() && !b.value.empty()) r.value = std::move(b.value[0]);
    return r;
  }
  // search_with_filter(&[f32], k, Some(filter)) (:245-250): `allowed[i]` = RestrictFilter::is_allowed(i).  The filter
  // belongs to this call only (scann_treeah_search_filtered), so concurrent calls with different filters are safe.
  Result<NNResultsVector> search_with_filter(const std::vector<float>& query, size_t k,
                                             const std::vector<bool>& allowed) const {
    auto b = search_batched_with_filter({query}, k, {allowed}, {0u});
    Result<NNResultsVector> r;
    r.error = b.error;
    if (b.ok() && !b.value.empty()) r.value = std::move(b.value[0]);
    return r;
  }
  // One batch, one filter per query: query q may only return datapoints i with filters[filter_of_query[q]][i] true.
  // filter_of_query[q] >= filters.size() -> InvalidArgument.  Filters shorter than the dataset do not allow the ids
  // beyond their end.
  Result<std::vector<NNResultsVector>> search_batched_with_filter(const std::vector<std::vector<float>>& queries,
                                                                  size_t k,
                                                                  const std::vector<std::vector<bool>>& filters,
                                                                  const std::vector<uint32_t>& filter_of_query) const {
    Result<std::vector<NNResultsVector>> r;
    if (filter_of_query.size() != queries.size()) {
      r.error = {ErrorCode::InvalidArgument, "filter_of_query must hold one filter index per query"};
      return r;
    }
    if (queries.empty()) return r;
    std::vector<float> flat;
    size_t dim;
    if (!detail::flatten(queries, &flat, &dim)) {
      r.error = {ErrorCode::InvalidArgument, "Query dimensionality mismatch"};
      return r;
    }
    size_t num_ids = 0;
    for (const auto& f : filters) num_ids = std::max(num_ids, f.size());
    const size_t row = (num_ids + 7) / 8;
    std::vector<uint8_t> bits(std::max<size_t>(1, filters.size() * row), 0);  // never NULL: empty filters allow nothing
    for (size_t f = 0; f < filters.size(); ++f)
      for (size_t i = 0; i < filters[f].size(); ++i)
        if (filters[f][i]) bits[f * row + (i >> 3)] |= static_cast<uint8_t>(1u << (i & 7));
    const size_t nq = queries.size(), R = cfg_.pre_reorder_k(k);
    std::vector<uint32_t> ids(nq * k), counts(nq);
    std::vector<float> dists(nq * k);
    r.error = make_error(scann_treeah_search_filtered(h_, flat.data(), nq, dim, cfg_.partitions_to_search, R, k,
                                                      bits.data(), filters.size(), num_ids, filter_of_query.data(),
                                                      ids.data(), dists.data(), counts.data(), nullptr, nullptr,
                                                      nullptr, SCANN_HOST, nullptr));
    if (r.ok()) r.value = detail::unflatten(ids, dists, counts, k);
    return r;
  }
  // build(dataset) (:131-209) on the GPU: k-means partition centres, residual PQ codebook (16 codes), exact assignment
  // and encode, all inside the library (scann_treeah_build)
  ScannError build(const float* data, size_t n, size_t dim, size_t stride, size_t train_rows = 1000000,
                   int kmeans_iters = 20, uint64_t seed = 7, int device = 0) {
    scann_treeah_destroy(h_);
    h_ = nullptr;
    return make_error(scann_treeah_build(data, n, dim, stride, cfg_.num_partitions, cfg_.num_subspaces, train_rows,
                                         kmeans_iters, seed, cfg_.use_residuals ? 1 : 0,
                                         static_cast<int>(cfg_.distance_measure), 1, device, SCANN_HOST, &h_));
  }
  // Searcher::search_batched_with_params (src/searcher.rs:164-169): one SearchParameters per query, the whole batch in
  // one call (scann_treeah_search_with_params); k_q = num_neighbors (10 when unset), R_q = pre_reordering_num_neighbors
  // (pre_reorder_k(k_q) when unset); queries.len() != params.len() -> InvalidArgument (searcher.rs:233-237).  An
  // error aborts the whole batch (searcher.rs:192-208).
  Result<std::vector<NNResultsVector>> search_batched_with_params(const std::vector<std::vector<float>>& queries,
                                                                  const std::vector<SearchParameters>& params) const {
    Result<std::vector<NNResultsVector>> r;
    if (queries.size() != params.size()) {
      r.error = {ErrorCode::InvalidArgument, "Number of queries must match number of parameter sets"};
      return r;
    }
    if (queries.empty()) return r;
    std::vector<float> flat;
    size_t dim;
    if (!detail::flatten(queries, &flat, &dim)) {
      r.error = {ErrorCode::InvalidArgument, "Query dimensionality mismatch"};
      return r;
    }
    const size_t nq = queries.size();
    std::vector<uint32_t> kq(nq), rq(nq);
    size_t k = 0, R = 0;
    for (size_t q = 0; q < nq; ++q) {
      const size_t kv = params[q].num_neighbors ? params[q].num_neighbors : 10;
      const size_t rv = params[q].pre_reordering_num_neighbors ? params[q].pre_reordering_num_neighbors
                                                               : cfg_.pre_reorder_k(kv);
      if (kv > 0xFFFFFFFFu || rv > 0xFFFFFFFFu) {
        r.error = {ErrorCode::InvalidArgument, "num_neighbors or pre_reordering_num_neighbors does not fit 32 bits"};
        return r;
      }
      kq[q] = static_cast<uint32_t>(kv);
      rq[q] = static_cast<uint32_t>(rv);
      k = std::max(k, kv);
      R = std::max(R, rv);
    }
    std::vector<uint32_t> ids(nq * k), counts(nq);
    std::vector<float> dists(nq * k);
    r.error = make_error(scann_treeah_search_with_params(h_, flat.data(), nq, dim, cfg_.partitions_to_search, R, k,
                                                         nullptr, rq.data(), kq.data(), ids.data(), dists.data(),
                                                         counts.data(), nullptr, nullptr, nullptr, SCANN_HOST,
                                                         nullptr));
    if (r.ok()) r.value = detail::unflatten(ids, dists, counts, k);
    return r;
  }
  const TreeXHybridConfig& config() const { return cfg_; }
  TreeXHybridConfig& config() { return cfg_; }
  scann_treeah* handle() const { return h_; }

 private:
  Result<std::vector<NNResultsVector>> search_impl(const std::vector<std::vector<float>>& queries, size_t k,
                                                   size_t pre_reorder_k) const {
    Result<std::vector<NNResultsVector>> r;
    if (queries.empty()) return r;
    std::vector<float> flat;
    size_t dim;
    if (!detail::flatten(queries, &flat, &dim)) {
      r.error = {ErrorCode::InvalidArgument, "Query dimensionality mismatch"};
      return r;
    }
    size_t nq = queries.size();
    std::vector<uint32_t> ids(nq * k), counts(nq);
    std::vector<float> dists(nq * k);
    r.error = make_error(scann_treeah_search(h_, flat.data(), nq, dim, cfg_.partitions_to_search, pre_reorder_k, k,
                                             ids.data(), dists.data(), counts.data(), nullptr, nullptr, nullptr,
                                             SCANN_HOST, nullptr));
    if (r.ok()) r.value = detail::unflatten(ids, dists, counts, k);
    return r;
  }
  TreeXHybridConfig cfg_;
  scann_treeah* h_ = nullptr;
};

// ------------------------------------------------------------------------------------------------
// AsymmetricHasher on the LUT16 path (src/hashes/hasher.rs:75-259): one partition holding every point, no residuals.
struct AsymmetricHasherConfig {  // hasher.rs:19-69 (num_codes is 16 on the GPU path)
  size_t num_subspaces = 8;
  uint64_t seed = 42;
  int kmeans_iters = 20;
};

class AsymmetricHasher {
 public:
  explicit AsymmetricHasher(AsymmetricHasherConfig cfg = {}) : cfg_(cfg) {}
  AsymmetricHasher(AsymmetricHasher&& o) noexcept : cfg_(o.cfg_), h_(o.h_) { o.h_ = nullptr; }
  AsymmetricHasher(const AsymmetricHasher&) = delete;
  ~AsymmetricHasher() { scann_treeah_destroy(h_); }

  // build(dataset) (:109-159): Codebook::train on the dataset + encode; "Cannot build from empty dataset" (:110-112)
  ScannError build(const float* data, size_t n, size_t dim, size_t stride, int device = 0) {
    scann_treeah_destroy(h_);
    h_ = nullptr;
    return make_error(scann_treeah_build(data, n, dim, stride, 1, cfg_.num_subspaces, 0, cfg_.kmeans_iters, cfg_.seed, 0,
                                         SCANN_SQL2, 1, device, SCANN_HOST, &h_));
  }
  // search (:162-185): approximate (LUT16) distances, no re-ranking
  Result<NNResultsVector> search(const std::vector<float>& query, size_t k) const { return one(query, k, k, false); }
  // search_with_reordering (:188-229): pre_reorder_k best by the LUT, exact SquaredL2 (hard-wired, :208), first k
  Result<NNResultsVector> search_with_reordering(const std::vector<float>& query, size_t k, size_t pre_reorder_k) const {
    return one(query, k, pre_reorder_k, true);
  }
  // search_batched(&[&[f32]], k) (:232-238)
  Result<std::vector<NNResultsVector>> search_batched(const std::vector<std::vector<float>>& queries, size_t k) const {
    return run(queries, k, k, false);
  }

 private:
  Result<std::vector<NNResultsVector>> run(const std::vector<std::vector<float>>& queries, size_t k, size_t pre,
                                           bool reorder) const {
    Result<std::vector<NNResultsVector>> r;
    if (queries.empty()) return r;
    if (h_ == nullptr) return r;  // empty / unbuilt hasher -> Ok(vec![]) (:163-165)
    std::vector<float> flat;
    size_t dim;
    if (!detail::flatten(queries, &flat, &dim)) {
      r.error = {ErrorCode::InvalidArgument, "Query dimensionality mismatch"};
      return r;
    }
    size_t nq = queries.size();
    std::vector<uint32_t> ids(nq * k), counts(nq);
    std::vector<float> dists(nq * k);
    r.error = make_error(scann_treeah_set_reorder(h_, reorder ? 1 : 0));
    if (!r.ok()) return r;
    r.error = make_error(scann_treeah_search(h_, flat.data(), nq, dim, 1, pre, k, ids.data(), dists.data(), counts.data(),
                                             nullptr, nullptr, nullptr, SCANN_HOST, nullptr));
    if (r.ok()) r.value = detail::unflatten(ids, dists, counts, k);
    return r;
  }
  Result<NNResultsVector> one(const std::vector<float>& query, size_t k, size_t pre, bool reorder) const {
    auto b = run({query}, k, pre, reorder);
    Result<NNResultsVector> r;
    r.error = b.error;
    if (b.ok() && !b.value.empty()) r.value = std::move(b.value[0]);
    return r;
  }
  AsymmetricHasherConfig cfg_;
  scann_treeah* h_ = nullptr;
};

// The Scann facade's tree modes that score every member of the probed leaves (src/scann.rs:215-294):
//   search_partitioned <- Scann::search_partitioned (exact distances inside the L closest leaves)
//   search_tree_ah     <- Scann::search_tree_ah ("variant B": one f32 LookupTable of the query over byte codes)
class LeafScanSearcher {
 public:
  LeafScanSearcher() = default;
  LeafScanSearcher(LeafScanSearcher&& o) noexcept : h_(o.h_) { o.h_ = nullptr; }
  LeafScanSearcher(const LeafScanSearcher&) = delete;
  ~LeafScanSearcher() { scann_ivf_destroy(h_); }

  // centers [K*dim]; ids [n] grouped by partition; part_offsets [K+1]; raw [num_raw*stride] or null;
  // codebook [S*C*ds] + codes_by_id [num_raw*S] or both null
  ScannError build_from_index(const float* centers, size_t K, size_t dim, const uint32_t* ids,
                              const uint64_t* part_offsets, size_t n, const float* raw, size_t num_raw, size_t stride,
                              const float* codebook = nullptr, size_t S = 0, size_t C = 0,
                              const uint8_t* codes_by_id = nullptr, int device = 0) {
    scann_ivf_destroy(h_);
    h_ = nullptr;
    return make_error(scann_ivf_create(centers, K, dim, ids, part_offsets, n, raw, num_raw, stride, codebook, S, C,
                                       codes_by_id, device, SCANN_HOST, &h_));
  }
  Result<std::vector<NNResultsVector>> search_partitioned(const std::vector<std::vector<float>>& queries, size_t k,
                                                          size_t partitions_to_search,
                                                          DistanceMeasure m = DistanceMeasure::SquaredL2) const {
    return run(0, queries, k, partitions_to_search, m, -1);
  }
  // reorder >= 0: ReorderingHelper::reorder of the k results with that measure (scann.rs:198-209)
  Result<std::vector<NNResultsVector>> search_tree_ah(const std::vector<std::vector<float>>& queries, size_t k,
                                                      size_t partitions_to_search, int reorder = -1) const {
    return run(1, queries, k, partitions_to_search, DistanceMeasure::SquaredL2, reorder);
  }

 private:
  Result<std::vector<NNResultsVector>> run(int mode, const std::vector<std::vector<float>>& queries, size_t k, size_t L,
                                           DistanceMeasure m, int reorder) const {
    Result<std::vector<NNResultsVector>> r;
    if (queries.empty()) return r;
    std::vector<float> flat;
    size_t dim;
    if (!detail::flatten(queries, &flat, &dim)) {
      r.error = {ErrorCode::InvalidArgument, "Query dimensionality mismatch"};
      return r;
    }
    size_t nq = queries.size();
    std::vector<uint32_t> ids(nq * k), counts(nq);
    std::vector<float> dists(nq * k);
    r.error = make_error(scann_ivf_search(h_, mode, flat.data(), nq, dim, L, k, static_cast<int>(m), reorder, ids.data(),
                                          dists.data(), counts.data(), SCANN_HOST, nullptr));
    if (r.ok()) r.value = detail::unflatten(ids, dists, counts, k);
    return r;
  }
  scann_ivf* h_ = nullptr;
};

// ------------------------------------------------------------------------------------------------
// Scann / ScannBuilder facade (src/scann.rs:35-432).  Mode selection follows Scann::with_config (:88-100):
// brute_force -> BruteForce; tree + hash -> TreeAH; tree only -> Partitioned; hash only -> Hashed.
//   BruteForce  -> scann_bf_*            exact
//   TreeAH      -> scann_treeah_build    residual LUT16 scan + exact reorder (the north-star path)
//   Hashed      -> scann_treeah_build    one partition, no residuals (flat AsymmetricHasher)
//   Partitioned -> scann_ivf_build       exact distances inside the L closest leaves (:215-253)
enum class SearchMode { BruteForce, Partitioned, Hashed, TreeAH };

struct ScannConfig {  // src/config.rs:11-29, the fields the hot path reads (0 = not configured)
  size_t num_neighbors = 10;
  DistanceMeasure distance_measure = DistanceMeasure::SquaredL2;
  bool brute_force = false;
  size_t num_partitions = 0, num_partitions_to_search = 10;
  size_t hash_num_blocks = 0;
  size_t reorder_num_candidates = 0;
};

class Scann {
 public:
  Scann() = default;
  Scann(Scann&& o) noexcept : cfg_(o.cfg_), mode_(o.mode_), bf_(o.bf_), tree_(o.tree_), leaf_(o.leaf_), pre_(o.pre_) {
    o.bf_ = nullptr;
    o.tree_ = nullptr;
    o.leaf_ = nullptr;
  }
  Scann(const Scann&) = delete;
  ~Scann() {
    scann_bf_destroy(bf_);
    scann_treeah_destroy(tree_);
    scann_ivf_destroy(leaf_);
  }

  // with_config (:64-103); "Dataset cannot be empty" (:66-68)
  static Result<Scann> with_config(const float* data, size_t n, size_t dim, size_t stride, const ScannConfig& cfg,
                                   int device = 0) {
    Result<Scann> r;
    if (n == 0 || data == nullptr) {
      r.error = {ErrorCode::InvalidArgument, "Dataset cannot be empty"};
      return r;
    }
    Scann& s = r.value;
    s.cfg_ = cfg;
    if (cfg.brute_force) s.mode_ = SearchMode::BruteForce;
    else if (cfg.num_partitions && cfg.hash_num_blocks) s.mode_ = SearchMode::TreeAH;
    else if (cfg.num_partitions) s.mode_ = SearchMode::Partitioned;
    else if (cfg.hash_num_blocks) s.mode_ = SearchMode::Hashed;
    else s.mode_ = SearchMode::BruteForce;
    const int measure = static_cast<int>(cfg.distance_measure);
    if (s.mode_ == SearchMode::BruteForce) {
      r.error = make_error(scann_bf_create(data, n, dim, stride, measure, device, SCANN_HOST, &s.bf_));
    } else if (s.mode_ == SearchMode::Partitioned) {
      r.error = make_error(scann_ivf_build(data, n, dim, stride, cfg.num_partitions, 20, 7, device, SCANN_HOST, &s.leaf_));
    } else {
      const bool flat = s.mode_ == SearchMode::Hashed;
      r.error = make_error(scann_treeah_build(data, n, dim, stride, flat ? 1 : cfg.num_partitions, cfg.hash_num_blocks,
                                              1000000, 20, 7, flat ? 0 : 1, measure, cfg.reorder_num_candidates ? 1 : 0,
                                              device, SCANN_HOST, &s.tree_));
      s.pre_ = cfg.reorder_num_candidates ? cfg.reorder_num_candidates : cfg.num_neighbors;
    }
    return r;
  }
  static Result<Scann> brute_force(const float* data, size_t n, size_t dim, size_t stride, int device = 0) {  // :106-109
    ScannConfig c;
    c.brute_force = true;
    return with_config(data, n, dim, stride, c, device);
  }
  static Result<Scann> partitioned(const float* data, size_t n, size_t dim, size_t stride, size_t num_partitions,
                                   size_t partitions_to_search, int device = 0) {  // :112-124
    ScannConfig c;
    c.num_partitions = num_partitions;
    c.num_partitions_to_search = partitions_to_search;
    return with_config(data, n, dim, stride, c, device);
  }
  static Result<Scann> hashed(const float* data, size_t n, size_t dim, size_t stride, size_t num_blocks,
                              int device = 0) {  // :127-137
    ScannConfig c;
    c.hash_num_blocks = num_blocks;
    return with_config(data, n, dim, stride, c, device);
  }

  // search_batched (:297-303); k = 0 -> config.num_neighbors
  Result<std::vector<NNResultsVector>> search_batched(const std::vector<std::vector<float>>& queries, size_t k = 0) const {
    Result<std::vector<NNResultsVector>> r;
    if (queries.empty()) return r;
    if (k == 0) k = cfg_.num_neighbors;
    std::vector<float> flat;
    size_t dim;
    if (!detail::flatten(queries, &flat, &dim)) {
      r.error = {ErrorCode::InvalidArgument, "Query dimensionality mismatch"};
      return r;
    }
    const size_t nq = queries.size();
    std::vector<uint32_t> ids(nq * k), counts(nq);
    std::vector<float> dists(nq * k);
    if (mode_ == SearchMode::BruteForce) {
      r.error = make_error(scann_bf_search(bf_, flat.data(), nq, dim, k, ids.data(), dists.data(), counts.data(),
                                           SCANN_HOST, nullptr));
    } else if (mode_ == SearchMode::Partitioned) {
      r.error = make_error(scann_ivf_search(leaf_, 0, flat.data(), nq, dim, cfg_.num_partitions_to_search, k,
                                            static_cast<int>(cfg_.distance_measure), -1, ids.data(), dists.data(),
                                            counts.data(), SCANN_HOST, nullptr));
    } else {
      const size_t L = mode_ == SearchMode::Hashed ? 1 : cfg_.num_partitions_to_search;
      r.error = make_error(scann_treeah_search(tree_, flat.data(), nq, dim, L, pre_ > k ? pre_ : k, k, ids.data(),
                                               dists.data(), counts.data(), nullptr, nullptr, nullptr, SCANN_HOST,
                                               nullptr));
    }
    if (r.ok()) r.value = detail::unflatten(ids, dists, counts, k);
    return r;
  }
  Result<NNResultsVector> search(const std::vector<float>& query, size_t k = 0) const {  // :175-178
    auto b = search_batched({query}, k);
    Result<NNResultsVector> r;
    r.error = b.error;
    if (b.ok() && !b.value.empty()) r.value = std::move(b.value[0]);
    return r;
  }
  SearchMode search_mode() const { return mode_; }
  const ScannConfig& config() const { return cfg_; }

 private:
  ScannConfig cfg_;
  SearchMode mode_ = SearchMode::BruteForce;
  scann_bf* bf_ = nullptr;
  scann_treeah* tree_ = nullptr;
  scann_ivf* leaf_ = nullptr;
  size_t pre_ = 0;
};

class ScannBuilder {  // src/scann.rs:364-432
 public:
  ScannBuilder& num_neighbors(size_t k) {
    cfg_.num_neighbors = k;
    return *this;
  }
  ScannBuilder& distance_measure(DistanceMeasure m) {
    cfg_.distance_measure = m;
    return *this;
  }
  ScannBuilder& brute_force() {
    cfg_.brute_force = true;
    return *this;
  }
  ScannBuilder& tree(size_t num_partitions, size_t partitions_to_search) {  // .partitioned() in the README spelling
    cfg_.num_partitions = num_partitions;
    cfg_.num_partitions_to_search = partitions_to_search;
    return *this;
  }
  ScannBuilder& partitioned(size_t num_partitions, size_t partitions_to_search) {
    return tree(num_partitions, partitions_to_search);
  }
  ScannBuilder& hash(size_t num_blocks) {  // .hashed() in the README spelling
    cfg_.hash_num_blocks = num_blocks;
    return *this;
  }
  ScannBuilder& hashed(size_t num_blocks) { return hash(num_blocks); }
  ScannBuilder& reorder(size_t num_candidates) {
    cfg_.reorder_num_candidates = num_candidates;
    return *this;
  }
  Result<Scann> build(const float* data, size_t n, size_t dim, size_t stride, int device = 0) const {
    return Scann::with_config(data, n, dim, stride, cfg_, device);
  }

 private:
  ScannConfig cfg_;
};

// ------------------------------------------------------------------------------------------------
// KMeansTree (src/trees/kmeans_tree.rs:154-395): hierarchical k-means partitioning; nodes are numbered in preorder.
struct KMeansTreeConfig {  // :17-56
  size_t num_children = 100;
  size_t max_depth = 1;
  size_t min_leaf_size = 1;
  int kmeans_max_iterations = 20;
  uint64_t seed = 42;
};

struct LeafHit {  // one element of search_leaves' Vec<(depth, distance, &node)> (:302-319)
  uint32_t depth;
  float distance;
  uint32_t node;  // preorder node id of the leaf
};

class KMeansTree {
 public:
  explicit KMeansTree(KMeansTreeConfig cfg = {}) : cfg_(cfg) {}
  KMeansTree(KMeansTree&& o) noexcept : cfg_(o.cfg_), h_(o.h_) { o.h_ = nullptr; }
  KMeansTree(const KMeansTree&) = delete;
  ~KMeansTree() { scann_kmtree_destroy(h_); }

  // build(dataset) (:179-200); "Cannot build tree from empty dataset"
  ScannError build(const float* data, size_t n, size_t dim, size_t stride, int device = 0) {
    scann_kmtree_destroy(h_);
    h_ = nullptr;
    return make_error(scann_kmtree_build(data, n, dim, stride, cfg_.num_children, cfg_.max_depth, cfg_.min_leaf_size,
                                         cfg_.kmeans_max_iterations, cfg_.seed, device, SCANN_HOST, &h_));
  }
  size_t num_leaves() const { return info(1); }  // :293-295
  size_t size() const { return info(3); }        // :298-300
  // search_leaves(query, k) (:302-319)
  Result<std::vector<LeafHit>> search_leaves(const std::vector<float>& query, size_t k) const {
    Result<std::vector<LeafHit>> r;
    if (h_ == nullptr) return r;  // no root -> empty (:311-313)
    std::vector<uint32_t> nodes(k ? k : 1), depths(k ? k : 1);
    std::vector<float> dists(k ? k : 1);
    uint32_t count = 0;
    r.error = make_error(scann_kmtree_search_leaves(h_, query.data(), 1, query.size(), k, nodes.data(), dists.data(),
                                                    depths.data(), &count, SCANN_HOST, nullptr));
    if (r.ok())
      for (uint32_t j = 0; j < count; ++j) r.value.push_back({depths[j], dists[j], nodes[j]});
    return r;
  }
  scann_kmtree* handle() const { return h_; }

 private:
  size_t info(int which) const {
    size_t v[5] = {0, 0, 0, 0, 0};
    if (h_) scann_kmtree_info(h_, &v[0], &v[1], &v[2], &v[3], &v[4]);
    return v[which];
  }
  KMeansTreeConfig cfg_;
  scann_kmtree* h_ = nullptr;
};

}  // namespace scann
