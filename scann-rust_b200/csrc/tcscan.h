// Tensor-core LUT16 scan (tcscan.cu): host-side interface used by treeah.cu.
#pragma once

#include "common.cuh"

namespace scann {

constexpr int kTcsTile = 128;       // points per tile = TMEM lanes (MMA M)
constexpr int kTcsGroup = 128;      // pairs (queries) per group = accumulator columns (MMA N <= 128)
constexpr int kTcsItemTiles = 32;   // point tiles per work item

struct TcScanParams {
  const uint32_t* tokens;    // [nq][L] partition tokens (0xFFFFFFFF / leaves without rows here are skipped)
  size_t nq, L, K, dim, S;
  size_t T;                  // pairs of rank < T are skipped (already scanned by the register-LUT kernel)
  const uint64_t* pt_off;    // [K + 1]
  const uint32_t* leaf_perm; // leaves by descending size
  const uint8_t* codes_rm;   // [n][S / 2] PackedCodes4Bit rows in leaf order
  const float* queries;      // [nq][dim]
  const float* centers;      // [K][dim]
  const float* codebook;     // [S][16][dim / S]
  const uint32_t* qthr;      // [nq] f32 key of the bound tau_q proved by the probe (0xFFFFFFFF = none)
  int use_residuals;
  size_t max_leaf;
  size_t qcap;               // candidate list capacity per query
  int sms;
  cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};  // optional: recorded before the LUT kernel, before and after the scan
  unsigned long long* pair_points = nullptr;        // optional: += Σ over scanned (pair, leaf) of leaf size
  // optional: the per-leaf lists of the pairs of rank >= T that the caller's own worklist has already built
  // (treeah.cu build_worklist counts and scatters them as class B): saves this scan its count + scatter passes
  const uint32_t* wl_cnt = nullptr;          // [K] pairs of rank >= T per leaf
  const uint32_t* wl_pair_start = nullptr;   // [K] first entry of the leaf's list in wl_sorted_pairs
  const uint32_t* wl_sorted_pairs = nullptr; // pair indices (q * L + rank), grouped by leaf
  // optional restrict filters (ScanArgs::allow of lut16_scan_kernel.cuh): a survivor its query's filter row does not
  // allow is dropped before it takes a list slot
  const uint8_t* allow = nullptr;            // [num_filters][allow_stride] one byte per (256-point block, lane)
  size_t allow_stride = 0;
  const uint32_t* qfilt = nullptr;           // [nq] filter row of every query; nullptr = row 0
  uint32_t num_filters = 0;                  // a query whose row is >= num_filters is allowed nothing
  const uint32_t* blk_off = nullptr;         // [K + 1] first 256-point block of every leaf
};

struct TcScanOut {
  const unsigned long long* qcand;  // [nq][qcap] (approx distance key << 32 | leaf rank << 22 | position), unordered
  const uint32_t* qcnt;             // [nq] appended (may exceed qcap)
  const uint32_t* qflag;            // [nq] 1 = no bound or overflow: the register-LUT kernel re-does the query
  const uint32_t* fb_tokens;        // [nq][L] tokens of the flagged queries, 0xFFFFFFFF elsewhere
  int launches;
};

bool tc_scan_supported(size_t S, size_t dim);
size_t tc_scan_workspace_bytes(size_t nq, size_t L, size_t K, size_t S, size_t max_leaf, size_t qcap);
scann_status launch_tc_scan(const TcScanParams& p, Workspace& ws, TcScanOut* out, cudaStream_t s);
scann_status tc_make_map_u8(void* map, const void* base, size_t rows, size_t row_bytes);  // tc_gemm.cu

}  // namespace scann
