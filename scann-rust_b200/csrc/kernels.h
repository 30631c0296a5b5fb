// Host-side launchers shared between translation units (all take device pointers, enqueue on `s`).
#pragma once

#include "common.cuh"

namespace scann {

// partition.cu — the partition stage: exact squared-L2 centroid scoring + top-L (src/partitioning/tree_partitioner.rs:
// 175-229).  The centres are scored on the tensor cores (tc_gemm.cu scores + exact re-score of the survivors) when the
// shape allows it, else on the CUDA cores; tokens and distances are identical either way.
struct PartTc {
  DevBuf<uint16_t> cbf;  // centres as bf16 [tc_rows_pad(K)][tc_kpad(dim)]
  DevBuf<float> hx;      // |c|^2 / 2
  DevBuf<float> small;
  float cmax2 = 0.0f;    // max |c|^2
  bool ready = false;
};
class CentreScorer {
 public:
  // (re)loads the centres [K][dim] and derives the scoring operands; synchronises s
  scann_status set(const float* centers, size_t K, size_t dim, int memspace, cudaStream_t s);
  // device scratch select() needs for a batch of nq queries
  size_t scratch_bytes(size_t nq) const;
  // tokens [nq][L] (0xFFFFFFFF past min(L, K)), dists [nq][L] or null; all device pointers
  scann_status select(const float* queries, size_t nq, size_t L, uint32_t* tokens, float* dists, void* scratch,
                      cudaStream_t s) const;
  const float* centers() const { return centers_.p; }  // device [K][dim] f32
  int launches() const { return tc_.ready ? 3 : 2; }    // kernels one select() enqueues

 private:
  size_t K_ = 0, dim_ = 0;
  DevBuf<float> centers_, centersT_;  // centersT_: [dim][K]
  PartTc tc_;
  int sms_ = 148;
};

// select.cu — final exact re-score + (dist, id) order, and the multi-GPU merge
//   cand: [nq][kc] candidate row ids (0xFFFFFFFF = empty); writes ids/dists [nq][k], counts [nq]
scann_status launch_rescore_topk(const RescoreParams& rp, const uint32_t* cand, size_t nq, size_t kc, size_t k,
                                 uint32_t* ids, float* dists, uint32_t* counts, cudaStream_t s);
//   lists: [nq][cap] (score key << 32 | row), cnt [nq] entries appended (clamped to cap); rows >= n_rows ignored.
//   qn != nullptr: two-level certification — only the entries within 2*eps of the list's k-th smallest score are
//   re-scored (qn = |q|^2 per query, xmax2 = max |x|^2; see brute_force.cu)
scann_status launch_rescore_lists(const RescoreParams& rp, const unsigned long long* lists, const uint32_t* cnt,
                                  size_t nq, size_t cap, size_t k, size_t n_rows, uint32_t* ids, float* dists,
                                  uint32_t* counts, cudaStream_t s, float radius = __builtin_huge_valf(),
                                  uint32_t* flag = nullptr, const float* qn = nullptr, float xmax2 = 0.0f);  // radius: keep d <= radius; flag |= 2 when > k qualify
//   part_stride: elements between two parts' blocks (0 = nq * k, the dense [parts][nq][k] layout)
scann_status launch_merge_topk(const uint32_t* ids_in, const float* dists_in, size_t parts, size_t nq, size_t k,
                               uint32_t* ids_out, float* dists_out, uint32_t* counts_out, cudaStream_t s,
                               size_t part_stride = 0);

// tc_gemm.cu — tcgen05/TMEM/TMA ranking contraction (bf16 operands, f32 accumulation).  See the file header.
struct TcScoreParams {
  const void* q_bf16;        // [tc_queries_pad(nq, dim)][tc_kpad(dim)] from tc_prepare_queries
  size_t nq, dim;
  const void* rows_bf16;     // [rows_pad_total][tc_kpad(dim)] from tc_prepare_rows
  size_t rows_pad_total;
  const float* hx;           // [rows_pad_total]
  size_t row0, nrows;        // rows [row0, row0 + nrows) of this launch; row0 % 128 == 0
  size_t tile_stride = 1;    // > 1: a sample — the t-th 128-row tile starts at row0 + t * tile_stride * 128
  bool filter;               // false: dense scores, true: threshold filter into candidate lists
  bool hx_is_zero = false;   // hx == 0 for every real row (Dot): the FILTER epilogue skips the hx loads
  float* dense;              // [nq][ld], column = t * 128 + (row inside tile t); whole tiles are written
  size_t ld;
  const float* thr;          // [nq]
  unsigned long long* cand;  // [nq][cap] (ordered score key << 32 | row), arbitrary order
  size_t cap;
  uint32_t* cand_cnt;        // [nq]
  int sms;
};
size_t tc_kpad(size_t dim);
bool tc_supported(size_t dim);                      // dim <= 256
size_t tc_rows_pad(size_t n);                       // multiple of 128
size_t tc_queries_pad(size_t nq, size_t dim);       // multiple of 128 or 256
scann_status tc_prepare_rows(const void* rows, bool i8, size_t n, size_t dim, size_t stride, float scale,
                             bool want_norm, void* dst_bf16, float* hx, float* norm_max, cudaStream_t s);
scann_status tc_prepare_queries(const float* q, size_t nq, size_t dim, float scale, void* dst_bf16, float* qn,
                                cudaStream_t s);
scann_status launch_tc_scores(const TcScoreParams& p, cudaStream_t s);

// build_index.cu — Lloyd's k-means on contiguous device rows (see scann_kmeans_fit); assign_out: final nearest centre
scann_status kmeans_rows_device(const float* x, size_t n, size_t dim, size_t K, int iters, uint64_t seed,
                                float balance_ratio, float* centers, uint32_t* assign_out, int device);

// runtime.cu — accumulation mode of the LUT16 scan for a table of S subspaces (lut16_device.cuh scan_block):
// default 3 (IDP.2A, needs S <= 128) else 2; SCANN_ACC_MODE=0|1|2|3 overrides (tuning / parity tests)
int scan_acc_mode(int S);

}  // namespace scann
