// Per-query parameters through the C++ host mirror (include/scann_b200.hpp): search_batched_with_params sends the whole
// batch in one scann_treeah_search_with_params call, and every query's result is that of its own parameters alone.
// Built and run by tests/test_gpu_treeah_params.py with g++ against libscann_b200.so on a GPU box.
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
  const size_t n = 4000, dim = 16, nq = 8;
  std::vector<float> data(n * dim);
  unsigned s = 12345u;
  for (float& v : data) {
    s = s * 1664525u + 1013904223u;
    v = static_cast<float>((s >> 8) & 0xFFFF) / 65536.0f;
  }
  TreeXHybridConfig cfg;
  cfg.num_partitions = 8;
  cfg.partitions_to_search = 4;
  TreeXHybridSearcher t(cfg);
  CHECK(t.build(data.data(), n, dim, dim, n, 4, 7).code == ErrorCode::Ok);

  std::vector<std::vector<float>> queries;
  for (size_t q = 0; q < nq; ++q) queries.emplace_back(data.begin() + q * 97 * dim, data.begin() + (q * 97 + 1) * dim);
  // (num_neighbors, pre_reordering_num_neighbors); 0 = not set: k = 10, R = pre_reorder_k(k)
  const size_t kr[nq][2] = {{1, 0}, {5, 0}, {0, 0}, {20, 0}, {5, 3}, {10, 200}, {3, 1}, {30, 50}};
  std::vector<SearchParameters> params(nq);
  for (size_t q = 0; q < nq; ++q) params[q].with_num_neighbors(kr[q][0]).with_pre_reordering_neighbors(kr[q][1]);

  auto b = t.search_batched_with_params(queries, params);
  CHECK(b.ok() && b.value.size() == nq);
  for (size_t q = 0; q < nq; ++q) {
    // the query alone with its own k and R, through the plain entry point
    const size_t k = kr[q][0] ? kr[q][0] : 10, R = kr[q][1] ? kr[q][1] : cfg.pre_reorder_k(k);
    std::vector<uint32_t> ids(k), counts(1);
    std::vector<float> dists(k);
    CHECK(scann_treeah_search(t.handle(), queries[q].data(), 1, dim, cfg.partitions_to_search, R, k, ids.data(),
                              dists.data(), counts.data(), nullptr, nullptr, nullptr, SCANN_HOST, nullptr) == SCANN_OK);
    CHECK(b.value[q].size() == counts[0] && counts[0] == (k < R ? k : R));
    for (size_t j = 0; j < counts[0]; ++j) CHECK(b.value[q][j].first == ids[j] && b.value[q][j].second == dists[j]);
  }
  // parameters shared by every query are the plain search
  std::vector<SearchParameters> same(nq);
  for (auto& p : same) p.with_num_neighbors(7);
  auto one = t.search_batched_with_params(queries, same);
  auto plain = t.search_batched(queries, 7);
  CHECK(one.ok() && plain.ok() && one.value == plain.value);

  auto bad_len = t.search_batched_with_params(queries, {params[0]});
  CHECK(!bad_len.ok() && bad_len.error.code == ErrorCode::InvalidArgument);
  auto big = params;
  big[3].with_pre_reordering_neighbors(4096);  // above the 2048 limit of pre_reorder_k
  auto bad_r = t.search_batched_with_params(queries, big);
  CHECK(!bad_r.ok() && bad_r.error.code == ErrorCode::InvalidArgument && bad_r.value.empty());
  // the handle stays usable
  auto again = t.search_batched_with_params(queries, params);
  CHECK(again.ok() && again.value == b.value);
  std::printf("hpp params ok\n");
  return 0;
}
