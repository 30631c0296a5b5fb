// KMeansTree (src/trees/kmeans_tree.rs): hierarchical k-means partitioning — build (:179-280) and search_leaves
// (:302-355) for a batch of queries.
//
// Layout.  The tree is flattened in PREORDER: node i has centre[i][dim], depth[i], and its children are the node ids
// children[child_begin[i] .. child_begin[i] + child_count[i]) in the reference's stored order (child_count = 0 <=> leaf).
// Leaves own the datapoint indices leaf_points[leaf_begin[i] .. + leaf_count[i]).
//
// search_leaves.  The reference walks the tree depth-first, children in ascending (distance to the child's centre,
// stored index) order (a stable sort, :337-340), pushes every leaf it reaches with the distance to the leaf's centre,
// and stops the whole walk as soon as 2k leaves are collected (the `results.len() >= k * 2` test after every child
// unwinds through all levels, :346-349); the collected leaves are then stable-sorted by distance and cut to k
// (:316-318).  One warp per query does exactly that walk:
//   * distances: squared L2 in the reference's order — sequential over dimensions, d = q - c, sum += d*d, unfused;
//   * per level, the sorted child list ((f32 key of the distance) << 32 | stored index, bitonic sort in shared memory)
//     is parked in a per-query global scratch row, so returning to a parent costs nothing;
//   * collected leaves carry (distance key << 32 | visit sequence): the final sort is the reference's stable sort.
// NaN distances compare "Equal" in the reference (partial_cmp(..).unwrap_or(Equal)), which makes its order depend on
// the sort implementation; here NaN sorts last.
//
// build.  The recursion and every rule of build_node are the reference's (leaf when depth >= max_depth, n <=
// min_leaf_size or n <= num_children; k-means with seed + depth on the node's rows; empty clusters dropped; a single
// surviving cluster makes a leaf; the node centre is the f64 mean of ITS points in index order, computed by one thread
// per dimension so the summation order is the reference's).  The k-means itself is the library's (build_index.cu): the
// reference's k-means++ draws from an unpinned rand::StdRng, so its trees are not reproducible by anybody.
#include <algorithm>
#include <vector>

#include "kernels.h"

namespace scann {

namespace {

constexpr int kMaxTreeDepth = 32;
constexpr int kMaxChildren = 1024;

__device__ __forceinline__ float tree_sqdist(const float* __restrict__ q, const float* __restrict__ c, int dim) {
  float acc = 0.0f;
  for (int d = 0; d < dim; ++d) {
    const float df = __fsub_rn(q[d], __ldg(c + d));
    acc = __fadd_rn(acc, __fmul_rn(df, df));
  }
  return acc;
}

__device__ __forceinline__ void warp_bitonic_u64(unsigned long long* keys, int p2, int lane) {
  for (int kk = 2; kk <= p2; kk <<= 1) {
    for (int j = kk >> 1; j > 0; j >>= 1) {
      for (int i = lane; i < p2; i += 32) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const bool asc = (i & kk) == 0;
          const unsigned long long x = keys[i], y = keys[ixj];
          if ((x > y) == asc) {
            keys[i] = y;
            keys[ixj] = x;
          }
        }
      }
      __syncwarp();
    }
  }
}

struct TreeArgs {
  const float* centers;
  const uint32_t* depth;
  const uint32_t* child_begin;
  const uint32_t* child_count;
  const uint32_t* children;
  int dim, max_children, levels;
};

// one warp (= one CTA) per query
__global__ void __launch_bounds__(32) kmtree_search_kernel(TreeArgs t, const float* __restrict__ queries, int nq, int k,
                                                          unsigned long long* __restrict__ scratch,
                                                          uint32_t* __restrict__ out_nodes, float* __restrict__ out_dists,
                                                          uint32_t* __restrict__ out_depths, uint32_t* __restrict__ out_counts) {
  extern __shared__ __align__(16) uint8_t sm[];
  const int q = blockIdx.x, lane = threadIdx.x;
  if (q >= nq) return;
  int mc2 = 1;
  while (mc2 < t.max_children) mc2 <<= 1;
  const int cap = max(2 * k, 1);
  int cap2 = 1;
  while (cap2 < cap) cap2 <<= 1;
  unsigned long long* sortbuf = reinterpret_cast<unsigned long long*>(sm);       // [mc2]
  unsigned long long* res = sortbuf + mc2;                                       // [cap2] (dist key << 32 | visit seq)
  uint32_t* res_node = reinterpret_cast<uint32_t*>(res + cap2);                  // [cap]
  float* qs = reinterpret_cast<float*>(res_node + cap);                          // [dim]
  __shared__ uint32_t lvl_next[kMaxTreeDepth + 1], lvl_cnt[kMaxTreeDepth + 1], lvl_node[kMaxTreeDepth + 1];
  for (int d = lane; d < t.dim; d += 32) qs[d] = queries[static_cast<size_t>(q) * t.dim + d];
  for (int i = lane; i < cap2; i += 32) res[i] = ~0ull;
  __syncwarp();
  unsigned long long* my = scratch + static_cast<size_t>(q) * t.levels * t.max_children;
  int len = 0;

  // sorted child list of `node` into level `lv`
  auto expand = [&](uint32_t node, int lv) {
    const uint32_t cb = t.child_begin[node], cc = t.child_count[node];
    int p2 = 1;
    while (p2 < static_cast<int>(cc)) p2 <<= 1;
    for (int i = lane; i < p2; i += 32) {
      unsigned long long key = ~0ull;
      if (i < static_cast<int>(cc)) {
        const uint32_t child = t.children[cb + i];
        const float d = tree_sqdist(qs, t.centers + static_cast<size_t>(child) * t.dim, t.dim);
        key = (static_cast<unsigned long long>(f32_key(d)) << 32) | static_cast<uint32_t>(i);
      }
      sortbuf[i] = key;
    }
    __syncwarp();
    warp_bitonic_u64(sortbuf, p2, lane);
    unsigned long long* dst = my + static_cast<size_t>(lv) * t.max_children;
    for (int i = lane; i < static_cast<int>(cc); i += 32) dst[i] = sortbuf[i];
    __syncwarp();
    if (lane == 0) {
      lvl_node[lv] = node;
      lvl_next[lv] = 0;
      lvl_cnt[lv] = cc;
    }
    __syncwarp();
  };
  auto record = [&](uint32_t node, uint32_t dkey) {
    if (lane == 0 && len < cap) {
      res[len] = (static_cast<unsigned long long>(dkey) << 32) | static_cast<uint32_t>(len);
      res_node[len] = node;
    }
    ++len;
    __syncwarp();
  };

  if (t.child_count[0] == 0) {  // the root is a leaf
    float d = 0.0f;
    if (lane == 0) d = tree_sqdist(qs, t.centers, t.dim);
    d = __shfl_sync(0xFFFFFFFFu, d, 0);
    record(0u, f32_key(d));
  } else {
    int lv = 0;
    expand(0u, 0);
    while (lv >= 0 && len < cap) {
      const uint32_t nx = lvl_next[lv];
      if (nx >= lvl_cnt[lv]) {  // this node's children are done: back to the parent
        --lv;
        continue;
      }
      const unsigned long long key = my[static_cast<size_t>(lv) * t.max_children + nx];
      __syncwarp();
      if (lane == 0) lvl_next[lv] = nx + 1;
      __syncwarp();
      const uint32_t child = t.children[t.child_begin[lvl_node[lv]] + static_cast<uint32_t>(key & 0xFFFFFFFFu)];
      if (t.child_count[child] == 0) {
        record(child, static_cast<uint32_t>(key >> 32));
      } else {
        ++lv;
        expand(child, lv);
      }
    }
  }
  // stable sort by distance, first k
  const int have = min(len, cap);
  int p2 = 1;
  while (p2 < have) p2 <<= 1;
  __syncwarp();
  warp_bitonic_u64(res, p2, lane);
  const int outn = min(have, k);
  for (int j = lane; j < k; j += 32) {
    const bool ok = j < outn;
    const unsigned long long key = ok ? res[j] : ~0ull;
    const uint32_t node = ok ? res_node[static_cast<uint32_t>(key & 0xFFFFFFFFu)] : 0xFFFFFFFFu;
    out_nodes[static_cast<size_t>(q) * k + j] = node;
    if (out_dists) out_dists[static_cast<size_t>(q) * k + j] = ok ? key_f32(static_cast<uint32_t>(key >> 32)) : __int_as_float(0x7F800000);
    if (out_depths) out_depths[static_cast<size_t>(q) * k + j] = ok ? t.depth[node] : 0u;
  }
  if (lane == 0) out_counts[q] = static_cast<uint32_t>(outn);
}

// centre of a node = f64 mean of its points in index order (compute_center, kmeans_tree.rs:283-298): thread d sums
// dimension d sequentially
__global__ void node_center_kernel(const float* __restrict__ x, size_t dim, const uint32_t* __restrict__ idx, size_t m,
                                   float* __restrict__ center) {
  const size_t d = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (d >= dim) return;
  double s = 0.0;
  for (size_t i = 0; i < m; ++i) s += static_cast<double>(x[static_cast<size_t>(idx[i]) * dim + d]);
  center[d] = m ? static_cast<float>(s / static_cast<double>(m)) : 0.0f;
}

__global__ void gather_idx_rows_kernel(const float* __restrict__ x, size_t dim, const uint32_t* __restrict__ idx, size_t m,
                                       float* __restrict__ dst) {
  const size_t t = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= m * dim) return;
  const size_t i = t / dim, d = t - i * dim;
  dst[t] = x[static_cast<size_t>(idx[i]) * dim + d];
}

}  // namespace

}  // namespace scann

struct scann_kmtree {
  int device = 0;
  size_t dim = 0, num_nodes = 0, num_leaves = 0, num_points = 0;
  int max_children = 1, levels = 1;
  scann::DevBuf<float> centers;
  scann::DevBuf<uint32_t> depth, child_begin, child_count, children;
  // host copies for export / leaf membership
  std::vector<float> h_centers;
  std::vector<uint32_t> h_depth, h_child_begin, h_child_count, h_children, h_leaf_begin, h_leaf_count, h_leaf_points;
  scann::Workspace ws;
  std::mutex mu;
  scann::StreamOrder order;
  cudaStream_t stream = nullptr;
  ~scann_kmtree() {
    if (stream) cudaStreamDestroy(stream);
  }
};

namespace scann {
namespace {

scann_status finish_tree(scann_kmtree* h) {
  const size_t nn = h->num_nodes;
  int maxc = 1, maxd = 0;
  size_t leaves = 0, pts = 0;
  for (size_t i = 0; i < nn; ++i) {
    maxc = std::max<int>(maxc, static_cast<int>(h->h_child_count[i]));
    maxd = std::max<int>(maxd, static_cast<int>(h->h_depth[i]));
    if (h->h_child_count[i] == 0) {
      ++leaves;
      pts += h->h_leaf_count.empty() ? 0 : h->h_leaf_count[i];
    }
  }
  SCANN_REQUIRE(maxc <= kMaxChildren, SCANN_INVALID_ARGUMENT, "a node has %d children (limit %d)", maxc, kMaxChildren);
  SCANN_REQUIRE(maxd < kMaxTreeDepth, SCANN_INVALID_ARGUMENT, "tree depth %d exceeds the limit %d", maxd, kMaxTreeDepth);
  h->max_children = maxc;
  h->levels = maxd + 1;
  h->num_leaves = leaves;
  h->num_points = pts;
  SCANN_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  SCANN_TRY(h->centers.upload(h->h_centers.data(), nn * h->dim, SCANN_HOST, h->stream));
  SCANN_TRY(h->depth.upload(h->h_depth.data(), nn, SCANN_HOST, h->stream));
  SCANN_TRY(h->child_begin.upload(h->h_child_begin.data(), nn, SCANN_HOST, h->stream));
  SCANN_TRY(h->child_count.upload(h->h_child_count.data(), nn, SCANN_HOST, h->stream));
  SCANN_TRY(h->children.upload(h->h_children.data(), std::max<size_t>(1, h->h_children.size()), SCANN_HOST, h->stream));
  SCANN_CUDA(cudaStreamSynchronize(h->stream));
  return SCANN_OK;
}

struct TreeBuilder {
  scann_kmtree* h;
  const float* rows;  // device [n][dim]
  size_t dim;
  size_t num_children, max_depth, min_leaf_size;
  int iters;
  uint64_t seed;
  int device;
  DevBuf<uint32_t> d_idx, d_assign;
  DevBuf<float> d_sub, d_centers, d_center1;

  scann_status node_center(const std::vector<uint32_t>& idx, float* out_host) {
    SCANN_CUDA(cudaMemcpy(d_idx.p, idx.data(), idx.size() * 4, cudaMemcpyHostToDevice));
    node_center_kernel<<<static_cast<unsigned>((dim + 63) / 64), 64>>>(rows, dim, d_idx.p, idx.size(), d_center1.p);
    SCANN_CUDA(cudaGetLastError());
    SCANN_CUDA(cudaMemcpy(out_host, d_center1.p, dim * 4, cudaMemcpyDeviceToHost));
    return SCANN_OK;
  }

  // build_node (kmeans_tree.rs:203-280); returns the node id
  scann_status build(const std::vector<uint32_t>& idx, size_t depth, uint32_t* node_out) {
    const size_t n = idx.size();
    const uint32_t me = static_cast<uint32_t>(h->h_depth.size());
    *node_out = me;
    h->h_depth.push_back(static_cast<uint32_t>(depth));
    h->h_child_begin.push_back(0);
    h->h_child_count.push_back(0);
    h->h_leaf_begin.push_back(0);
    h->h_leaf_count.push_back(0);
    h->h_centers.resize(h->h_centers.size() + dim);
    SCANN_TRY(node_center(idx, h->h_centers.data() + static_cast<size_t>(me) * dim));
    auto make_leaf = [&]() {
      h->h_leaf_begin[me] = static_cast<uint32_t>(h->h_leaf_points.size());
      h->h_leaf_count[me] = static_cast<uint32_t>(n);
      h->h_leaf_points.insert(h->h_leaf_points.end(), idx.begin(), idx.end());
      return SCANN_OK;
    };
    if (depth >= max_depth || n <= min_leaf_size || n <= num_children) return make_leaf();
    const size_t K = std::min(num_children, n);
    gather_idx_rows_kernel<<<static_cast<unsigned>((n * dim + 255) / 256), 256>>>(rows, dim, d_idx.p, n, d_sub.p);
    SCANN_CUDA(cudaGetLastError());
    SCANN_TRY(kmeans_rows_device(d_sub.p, n, dim, K, iters, seed + depth, 0.0f, d_centers.p, d_assign.p, device));
    std::vector<uint32_t> assign(n);
    SCANN_CUDA(cudaMemcpy(assign.data(), d_assign.p, n * 4, cudaMemcpyDeviceToHost));
    std::vector<std::vector<uint32_t>> clusters(K);
    for (size_t i = 0; i < n; ++i)
      if (assign[i] < K) clusters[assign[i]].push_back(idx[i]);
    size_t non_empty = 0;
    for (auto& c : clusters) non_empty += !c.empty();
    if (non_empty <= 1) return make_leaf();  // "All points in one cluster - make leaf" (:262-265)
    std::vector<uint32_t> kids;
    for (auto& c : clusters) {
      if (c.empty()) continue;
      uint32_t child = 0;
      SCANN_TRY(build(c, depth + 1, &child));
      kids.push_back(child);
    }
    h->h_child_begin[me] = static_cast<uint32_t>(h->h_children.size());
    h->h_child_count[me] = static_cast<uint32_t>(kids.size());
    h->h_children.insert(h->h_children.end(), kids.begin(), kids.end());
    return SCANN_OK;
  }
};

}  // namespace
}  // namespace scann

extern "C" {

scann_status scann_kmtree_create(const float* centers, const uint32_t* depth, const uint32_t* child_begin,
                                 const uint32_t* child_count, const uint32_t* children, size_t num_nodes,
                                 size_t num_child_entries, size_t dim, int device, scann_kmtree** out) {
  using namespace scann;
  SCANN_REQUIRE(out != nullptr, SCANN_INVALID_ARGUMENT, "out is NULL");
  *out = nullptr;
  SCANN_REQUIRE(centers && depth && child_begin && child_count && num_nodes > 0 && dim > 0, SCANN_INVALID_ARGUMENT,
                "Cannot build tree from empty dataset");
  SCANN_REQUIRE(children != nullptr || num_child_entries == 0, SCANN_INVALID_ARGUMENT, "children is NULL");
  for (size_t i = 0; i < num_nodes; ++i) {
    SCANN_REQUIRE(static_cast<size_t>(child_begin[i]) + child_count[i] <= num_child_entries, SCANN_INVALID_ARGUMENT,
                  "node %zu: child range outside the children array", i);
    for (uint32_t c = 0; c < child_count[i]; ++c) {
      const uint32_t ch = children[child_begin[i] + c];
      SCANN_REQUIRE(ch > i && ch < num_nodes, SCANN_INVALID_ARGUMENT, "node %zu: child id %u is not a later node (preorder)",
                    i, ch);
    }
  }
  SCANN_TRY(check_device(device));
  DeviceGuard g(device);
  scann_kmtree* h = new scann_kmtree();
  h->device = device;
  h->dim = dim;
  h->num_nodes = num_nodes;
  h->h_centers.assign(centers, centers + num_nodes * dim);
  h->h_depth.assign(depth, depth + num_nodes);
  h->h_child_begin.assign(child_begin, child_begin + num_nodes);
  h->h_child_count.assign(child_count, child_count + num_nodes);
  if (num_child_entries) h->h_children.assign(children, children + num_child_entries);
  scann_status st = finish_tree(h);
  if (st != SCANN_OK) {
    scann_kmtree_destroy(h);
    return st;
  }
  *out = h;
  return SCANN_OK;
}

scann_status scann_kmtree_build(const float* x, size_t n, size_t dim, size_t stride, size_t num_children, size_t max_depth,
                                size_t min_leaf_size, int kmeans_iters, uint64_t seed, int device, int memspace,
                                scann_kmtree** out) {
  using namespace scann;
  SCANN_REQUIRE(out != nullptr, SCANN_INVALID_ARGUMENT, "out is NULL");
  *out = nullptr;
  SCANN_REQUIRE(x != nullptr && n > 0 && dim > 0 && stride >= dim, SCANN_INVALID_ARGUMENT,
                "Cannot build tree from empty dataset");  // kmeans_tree.rs:180-182
  SCANN_REQUIRE(num_children >= 1 && num_children <= static_cast<size_t>(kMaxChildren), SCANN_INVALID_ARGUMENT,
                "num_children %zu outside 1..%d", num_children, kMaxChildren);
  SCANN_REQUIRE(max_depth < static_cast<size_t>(kMaxTreeDepth), SCANN_INVALID_ARGUMENT, "max_depth %zu too large", max_depth);
  SCANN_REQUIRE(n < 0xFFFFFFFFull, SCANN_INVALID_ARGUMENT, "dataset too large for u32 ids");
  SCANN_TRY(check_device(device));
  DeviceGuard g(device);
  DevBuf<float> own;
  const float* rows = x;
  if (!(memspace == SCANN_DEVICE && stride == dim)) {
    SCANN_TRY(own.alloc(n * dim));
    SCANN_CUDA(cudaMemcpy2D(own.p, dim * sizeof(float), x, stride * sizeof(float), dim * sizeof(float), n,
                            memspace == SCANN_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice));
    rows = own.p;
  }
  scann_kmtree* h = new scann_kmtree();
  h->device = device;
  h->dim = dim;
  TreeBuilder b;
  b.h = h;
  b.rows = rows;
  b.dim = dim;
  b.num_children = num_children;
  b.max_depth = max_depth;
  b.min_leaf_size = min_leaf_size;
  b.iters = kmeans_iters;
  b.seed = seed;
  b.device = device;
  scann_status st = SCANN_OK;
  do {
    if ((st = b.d_idx.alloc(n)) != SCANN_OK) break;
    if ((st = b.d_assign.alloc(n)) != SCANN_OK) break;
    if ((st = b.d_sub.alloc(n * dim)) != SCANN_OK) break;
    if ((st = b.d_centers.alloc(num_children * dim)) != SCANN_OK) break;
    if ((st = b.d_center1.alloc(dim)) != SCANN_OK) break;
    std::vector<uint32_t> all(n);
    for (size_t i = 0; i < n; ++i) all[i] = static_cast<uint32_t>(i);
    uint32_t root = 0;
    if ((st = b.build(all, 0, &root)) != SCANN_OK) break;
    h->num_nodes = h->h_depth.size();
    st = finish_tree(h);
  } while (0);
  if (st != SCANN_OK) {
    scann_kmtree_destroy(h);
    return st;
  }
  *out = h;
  return SCANN_OK;
}

scann_status scann_kmtree_info(scann_kmtree* h, size_t* num_nodes, size_t* num_leaves, size_t* num_child_entries,
                               size_t* num_points, size_t* dim) {
  SCANN_REQUIRE(h != nullptr, SCANN_INVALID_ARGUMENT, "NULL handle");
  if (num_nodes) *num_nodes = h->num_nodes;
  if (num_leaves) *num_leaves = h->num_leaves;
  if (num_child_entries) *num_child_entries = h->h_children.size();
  if (num_points) *num_points = h->num_points;
  if (dim) *dim = h->dim;
  return SCANN_OK;
}

scann_status scann_kmtree_export(scann_kmtree* h, float* centers, uint32_t* depth, uint32_t* child_begin,
                                 uint32_t* child_count, uint32_t* children, uint32_t* leaf_begin, uint32_t* leaf_count,
                                 uint32_t* leaf_points) {
  SCANN_REQUIRE(h != nullptr, SCANN_INVALID_ARGUMENT, "NULL handle");
  auto put = [](auto* dst, const auto& v) {
    if (dst && !v.empty()) std::copy(v.begin(), v.end(), dst);
  };
  put(centers, h->h_centers);
  put(depth, h->h_depth);
  put(child_begin, h->h_child_begin);
  put(child_count, h->h_child_count);
  put(children, h->h_children);
  put(leaf_begin, h->h_leaf_begin);
  put(leaf_count, h->h_leaf_count);
  put(leaf_points, h->h_leaf_points);
  return SCANN_OK;
}

scann_status scann_kmtree_search_leaves(scann_kmtree* h, const float* queries, size_t nq, size_t qdim, size_t k,
                                        uint32_t* leaf_nodes, float* dists, uint32_t* depths, uint32_t* counts,
                                        int memspace, void* stream) {
  using namespace scann;
  SCANN_REQUIRE(h != nullptr, SCANN_FAILED_PRECONDITION, "Tree not built");
  if (nq == 0) return SCANN_OK;
  SCANN_REQUIRE(queries && counts && (k == 0 || leaf_nodes), SCANN_INVALID_ARGUMENT, "NULL buffer");
  SCANN_REQUIRE(qdim == h->dim, SCANN_INVALID_ARGUMENT, "Query dimensionality %zu does not match dataset dimensionality %zu",
                qdim, h->dim);
  SCANN_REQUIRE(k <= 1024, SCANN_INVALID_ARGUMENT, "k %zu > 1024 unsupported", k);
  std::lock_guard<std::mutex> lock(h->mu);
  CallScope call(h->device, h->order, memspace, stream, h->stream);
  const size_t per_q = static_cast<size_t>(h->levels) * h->max_children * 8;
  size_t chunk = std::min(nq, std::max<size_t>(1, (size_t(256) << 20) / per_q));
  const QueryOut outs[] = {{leaf_nodes, k * 4}, {dists, k * 4}, {depths, k * 4}, {counts, 4}};
  SCANN_TRY(h->ws.reserve(Workspace::padded(chunk * per_q) + staging_bytes(memspace, chunk, h->dim, outs)));
  TreeArgs t{h->centers.p, h->depth.p, h->child_begin.p, h->child_count.p, h->children.p, static_cast<int>(h->dim),
             h->max_children, h->levels};
  int mc2 = 1;
  while (mc2 < h->max_children) mc2 <<= 1;
  const int cap = std::max<int>(2 * static_cast<int>(k), 1);
  int cap2 = 1;
  while (cap2 < cap) cap2 <<= 1;
  const size_t smem = static_cast<size_t>(mc2) * 8 + static_cast<size_t>(cap2) * 8 + static_cast<size_t>(cap) * 4 +
                      ((h->dim + 3) & ~size_t(3)) * 4;
  if (smem > 48 * 1024)
    SCANN_CUDA(cudaFuncSetAttribute(kmtree_search_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  return run_query_chunks(h->ws, memspace, call.s, queries, nq, h->dim, chunk, outs,
                          [&](const float* q, size_t, size_t nqc, void* const* o) -> scann_status {
                            unsigned long long* scratch = h->ws.take<unsigned long long>(chunk * per_q / 8);
                            kmtree_search_kernel<<<static_cast<unsigned>(nqc), 32, smem, call.s>>>(
                                t, q, static_cast<int>(nqc), static_cast<int>(k), scratch, static_cast<uint32_t*>(o[0]),
                                static_cast<float*>(o[1]), static_cast<uint32_t*>(o[2]), static_cast<uint32_t*>(o[3]));
                            SCANN_CUDA(cudaGetLastError());
                            return SCANN_OK;
                          });
}

void scann_kmtree_destroy(scann_kmtree* h) {
  if (!h) return;
  scann::DeviceGuard g(h->device);
  cudaDeviceSynchronize();
  delete h;
}

}  // extern "C"
