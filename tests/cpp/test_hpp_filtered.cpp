// Per-query restrict filters through the C++ host mirror (include/scann_b200.hpp): search_batched_with_filter gives
// every query its own filter in one batch, search_with_filter is the one-query case of it.
// Built and run by tests/test_gpu_filtered_batch.py with g++ against libscann_b200.so on a GPU box.
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "scann_b200.hpp"

#define CHECK(cond)                                                                 \
  do {                                                                              \
    if (!(cond)) {                                                                  \
      std::fprintf(stderr, "CHECK failed %s:%d: %s\n", __FILE__, __LINE__, #cond); \
      return 1;                                                                     \
    }                                                                               \
  } while (0)

int main() {
  using namespace scann;
  const size_t n = 4000, dim = 16, nq = 6, k = 5;
  std::vector<float> data(n * dim);
  unsigned s = 12345u;
  for (float& v : data) {
    s = s * 1664525u + 1013904223u;
    v = static_cast<float>((s >> 8) & 0xFFFF) / 65536.0f;
  }
  TreeXHybridConfig cfg;
  cfg.num_partitions = 8;
  cfg.partitions_to_search = 8;
  TreeXHybridSearcher t(cfg);
  CHECK(t.build(data.data(), n, dim, dim, n, 4, 7).code == ErrorCode::Ok);

  std::vector<std::vector<bool>> filters(3, std::vector<bool>(n, false));
  for (size_t i = 0; i < n; ++i) {
    filters[0][i] = i % 2 == 0;  // even ids
    filters[1][i] = i < 100;     // a small prefix
  }                              // filters[2]: nothing allowed
  std::vector<std::vector<float>> queries;
  for (size_t q = 0; q < nq; ++q) queries.emplace_back(data.begin() + q * 97 * dim, data.begin() + (q * 97 + 1) * dim);
  const std::vector<uint32_t> fq = {0, 1, 2, 0, 1, 0};

  auto b = t.search_batched_with_filter(queries, k, filters, fq);
  CHECK(b.ok() && b.value.size() == nq);
  for (size_t q = 0; q < nq; ++q) {
    for (auto& r : b.value[q]) CHECK(filters[fq[q]][r.first]);
    CHECK(fq[q] == 2 ? b.value[q].empty() : b.value[q].size() == k);
    // the one-query call answers the same as the query's row of the batch
    auto one = t.search_with_filter(queries[q], k, filters[fq[q]]);
    CHECK(one.ok() && one.value == b.value[q]);
  }
  // an allow-everything filter is the plain search
  auto plain = t.search_batched(queries, k);
  auto all = t.search_batched_with_filter(queries, k, {std::vector<bool>(n, true)}, std::vector<uint32_t>(nq, 0u));
  CHECK(plain.ok() && all.ok() && plain.value == all.value);

  auto bad_row = t.search_batched_with_filter(queries, k, filters, {0, 1, 3, 0, 1, 0});
  CHECK(!bad_row.ok() && bad_row.error.code == ErrorCode::InvalidArgument);
  auto bad_len = t.search_batched_with_filter(queries, k, filters, {0, 1});
  CHECK(!bad_len.ok() && bad_len.error.code == ErrorCode::InvalidArgument);
  auto none = t.search_batched_with_filter(queries, k, {}, fq);
  CHECK(!none.ok() && none.error.code == ErrorCode::InvalidArgument);
  // the handle stays usable
  auto again = t.search_batched_with_filter(queries, k, filters, fq);
  CHECK(again.ok() && again.value == b.value);
  std::printf("hpp filtered ok\n");
  return 0;
}
