// Byte codes with the f32 LookupTable through the C++ host mirror (include/scann_b200.hpp): build_from_byte_codes,
// search_batched and search_batched_with_filter on a 4 x 4 grid whose neighbours are known by hand.
// Built and run by tests/test_gpu_treeah_f32lut.py with g++ against libscann_b200.so on a GPU box.
#include <cstdio>
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
  // point i = (i % 4, i / 4); one subspace per coordinate, code c = coordinate c, so the approximate distance of a
  // point is its exact squared distance; one partition, no residuals (the flat AsymmetricHasher)
  const size_t n = 16, dim = 2, S = 2, C = 4;
  std::vector<float> raw(n * dim), codebook(S * C), centers(dim, 0.0f);
  std::vector<uint8_t> codes(n * S);
  std::vector<uint32_t> ids(n);
  for (size_t i = 0; i < n; ++i) {
    raw[i * 2] = static_cast<float>(i % 4);
    raw[i * 2 + 1] = static_cast<float>(i / 4);
    codes[i * 2] = static_cast<uint8_t>(i % 4);
    codes[i * 2 + 1] = static_cast<uint8_t>(i / 4);
    ids[i] = static_cast<uint32_t>(i);
  }
  for (size_t s = 0; s < S; ++s)
    for (size_t c = 0; c < C; ++c) codebook[s * C + c] = static_cast<float>(c);
  const uint64_t offsets[2] = {0, n};
  TreeXHybridConfig cfg;
  cfg.num_partitions = 1;
  cfg.partitions_to_search = 1;
  cfg.use_residuals = false;
  TreeXHybridSearcher t(cfg);
  CHECK(t.build_from_byte_codes(centers.data(), 1, dim, codebook.data(), S, C, codes.data(), ids.data(), offsets, n,
                                raw.data(), n, dim)
            .code == ErrorCode::Ok);

  const std::vector<std::vector<float>> queries = {{0.1f, 0.2f}, {2.9f, 2.8f}};
  auto r = t.search_batched(queries, 3);
  CHECK(r.ok() && r.value.size() == 2);
  const uint32_t want[2][3] = {{0, 4, 1}, {15, 11, 14}};  // (x, y) = (0,0) (0,1) (1,0) and (3,3) (3,2) (2,3)
  for (size_t q = 0; q < 2; ++q) {
    CHECK(r.value[q].size() == 3);
    for (size_t j = 0; j < 3; ++j) CHECK(r.value[q][j].first == want[q][j]);
  }
  // only odd ids for query 0, everything for query 1
  std::vector<bool> odd(n), all(n, true);
  for (size_t i = 0; i < n; ++i) odd[i] = (i & 1) != 0;
  auto f = t.search_batched_with_filter(queries, 3, {odd, all}, {0u, 1u});
  CHECK(f.ok() && f.value.size() == 2 && f.value[0].size() == 3);
  const uint32_t want_odd[3] = {1, 5, 9};  // (1,0) (1,1) (1,2)
  for (size_t j = 0; j < 3; ++j) CHECK(f.value[0][j].first == want_odd[j] && f.value[1][j].first == want[1][j]);

  TreeXHybridSearcher bad(cfg);
  codes[5] = 4;  // a code outside the table row
  CHECK(bad.build_from_byte_codes(centers.data(), 1, dim, codebook.data(), S, C, codes.data(), ids.data(), offsets, n,
                                  raw.data(), n, dim)
            .code == ErrorCode::InvalidArgument);
  std::printf("hpp f32lut ok\n");
  return 0;
}
