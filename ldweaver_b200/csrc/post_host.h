// Pieces of mergeNsort_sr_links (R/computePairwiseMI.R:400-495) shared by the host implementation (post_host.cpp:
// ldw_sr_postprocess) and the device one (post_dev.cu: ldw_sr_postprocess_dev): everything that is O(groups) or
// O(links above the fit) stays on the host in both -- decay fits, beta fit, the de-duplication of cross-cluster links,
// the error checks, publishing the result.  The per-link rules both evaluate are in sr_stats.cuh.
#pragma once
#include <stdint.h>

#include <memory>
#include <vector>

#include "../../include/ldw.h"
#include "ctx.h"

namespace ldwpost {

// Plain host memory for LinkCols (the device path's df rows).
struct HostBuf {
  std::unique_ptr<char[]> p;
  int ensure(size_t n) { p.reset(new char[n]); return 0; }
  template <class T> T* as() const { return reinterpret_cast<T*>(p.get()); }
};
using HostCols = LinkCols<HostBuf>;

struct SrPostPriv {
  std::vector<int32_t> clust_c;
  std::vector<int64_t> row;
  std::vector<double> srp;
  std::vector<int64_t> red, chk;
  std::vector<int64_t> fit_off;
  std::vector<int32_t> fit_len;
  std::vector<double> fit_q95, fit_val, coef, shape, start;
  std::vector<int64_t> n_pos;
  std::vector<int32_t> nm_evals, nm_fail;
  HostCols df;  // device path: link columns of the df rows (the full table never reaches the host)
};

// glist: non-empty groups (cluster-major, ascending length; group id = (c - 1) * nl + len), gq: their 95th percentiles
int decay_fits(SrPostPriv& S, int32_t nclust, int64_t nl, const std::vector<int64_t>& glist, const std::vector<double>& gq);
int beta_fit(SrPostPriv& S, int32_t c, int64_t npos, double s1, double s2, double mean, double v, double par[2]);
// Entry k is row at[k] of L with srp_max srp[k]; returns the k that stay, in the order of their link's first appearance.
std::vector<int64_t> dedup(const ldw_links& L, const std::vector<int64_t>& at, const std::vector<double>& srp);
void publish(SrPostPriv& S, int32_t nclust, ldw_sr_post* out);

// The reference's failures (0 if none): a cluster without member links (goff: offsets of the (cluster, length) groups),
// a residual above 1 in cluster bad_c (0: none), fewer than two links above cluster c's fitted decay.
int check_groups(const std::vector<int64_t>& goff, int32_t nclust, int64_t nl);
int check_residuals(int bad_c);
int check_npos(int32_t c, int64_t npos);

}  // namespace ldwpost
