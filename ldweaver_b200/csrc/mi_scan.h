// Internal (C++) interface of the MI scan driver (mi_scan.cu) used by the device-group layer (group.cu).
#pragma once
#include <vector>

#include "ctx.h"

namespace ldw {

struct BlockSizes {
  int64_t n_pairs, n_sr, n_lr;
  int err;  // 0 ok, 1 empty block
};

// Several plans (one per device) scanning parts of ONE job into one host table.
struct ScanShared {
  std::vector<BlockSizes> sizes;   // per make_blocks index, all blocks of the job
  std::vector<int64_t> sr_hbase;   // first short-range row of each block in the job's table (make_blocks order)
  int64_t total_sr = 0;
  HostLinks* h_sr = nullptr;       // portable pinned columns sized total_sr; every device copies its rows in place
};

// codes: host matrix (validated + uploaded) or NULL with codes_dev = the matrix already resident on ctx's device
// (borrowed: it must outlive the plan).
int mi_plan_create_impl(ldw_ctx* ctx, const uint8_t* codes, const uint8_t* codes_dev, int64_t n_snp, int64_t nseq,
                        const double* hdw, const int32_t* pos, const int32_t* paint, int64_t blk, ldw_mi_plan** out);
// LDW_ERR_ARG for a combination of LDW_SCAN_* flags that asks for nothing (host only: callable before any device work)
int validate_scan_flags(int flags);
int mi_block_sizes(const ldw_mi_plan* P, double g, double sr_dist, int flags, std::vector<BlockSizes>& out);
int64_t mi_plan_nblocks(const ldw_mi_plan* P);
// owner[b] = part that scans make_blocks block b when the job is split n_parts ways (cost-based dealing)
void mi_block_owners(const ldw_mi_plan* P, int n_parts, std::vector<int>& owner);
// ldw_mi_scan with an optional shared layout: short-range rows land in shared->h_sr at shared->sr_hbase[block] (sr_out then
// only carries the row count of this part); long-range / borderline rows stay in the plan's context.
int mi_scan_impl(ldw_mi_plan* P, double g, double sr_dist, double lr_retain_links, double lr_links_approx, int flags,
                 int n_parts, int part, const ScanShared* shared, ldw_links* sr_out, ldw_links* lr_out,
                 ldw_links* borderline_out, double* thr_out, double* prob_out, ldw_scan_stats* stats_out);

}  // namespace ldw
