// Internal (C++) interface of the Hamming-distance-weights stage; see hdw.cu.
#pragma once
#include <functional>

#include "host_util.h"

namespace ldw {

// codes: device [n x S] uint8.  table: device int32 [n x 5] class counts; mask: observed-allele bitmask; r: popcount.
int snp_allele_stats(cudaStream_t st, const uint8_t* d_codes, int64_t n, int64_t S, int32_t* d_table, uint8_t* d_mask,
                     uint8_t* d_r);
// Largest byte of the device buffer d[0..n) (0 when n <= 0) into the host *out; synchronises st.  Validates a class matrix
// (every class 0..4) in ldw_hdw and ldw_group_load_codes.
int max_byte_device(cudaStream_t st, const uint8_t* d, int64_t n, uint32_t* out);
int exclusive_scan_i32(cudaStream_t st, const int32_t* d_in, int64_t n, int32_t* d_out, int32_t* d_total);
// Multi-GPU share of the distance GEMM (see hdw_device): rank `part` of `n_parts`; `allreduce` sums int32[S] in place
// across the ranks on the given stream; `force` shards even when the problem is small (tests).
struct HdwShard {
  int n_parts = 1, part = 0;
  bool force = false;
  std::function<int(int32_t* d_counts, int64_t S, cudaStream_t st)> allreduce;
  int* sharded_out = nullptr;  // receives 1 when the tiles were dealt across ranks, 0 when every rank computed all
};
// d_neigh: int32[S] neighbour counts (incl. self); d_hdw: double[S]; d_dist: optional int32 [S x S] (column-major).
int hdw_device(cudaStream_t st, const uint8_t* d_codes, int64_t n, int64_t S, int32_t thresh, int32_t* d_neigh,
               double* d_hdw, int32_t* d_dist, int num_sms, const HdwShard* shard = nullptr);

}  // namespace ldw
