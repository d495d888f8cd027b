// Per-link rules of mergeNsort_sr_links (R/computePairwiseMI.R:400-495), compiled into the host implementation
// (post_host.cpp, built as CUDA source) and the device one (post_dev.cu) alike, so that the two cannot drift apart.
#pragma once
#include <math.h>
#include <stdint.h>

#include <algorithm>

#include "../../include/ldw.h"

namespace ldwpost {

// Filters of :417-419 and the clusters link i is listed under (:372-376): clust1 and, if different, clust2 (0 = none);
// only 0 < len < sr_dist.
__host__ __device__ __forceinline__ bool member(const ldw_links& T, int64_t i, double sr_dist, int nclust, int& ca, int& cb, int& l) {
  l = T.len[i];
  if (!(l > 0 && (double)l < sr_dist)) return false;
  ca = T.clust1[i]; cb = T.clust2[i];
  if (ca < 1 || ca > nclust) ca = 0;
  if (cb < 1 || cb > nclust || cb == ca) cb = 0;
  return (ca | cb) != 0;
}

// Fitted decay of cluster c (values val[off[c - 1] ..] of its groups) that the reference pairs with a link of length l:
// `mean_dist[sr_links_t$len]` (:448) subscripts the fitted values with the VALUE of len (position in maxvls), which is
// the group of that length only when no shorter length is missing.  Reproduced as is.
template <class Off>
__host__ __device__ __forceinline__ double fit_at(const double* val, const Off& off, int c, int64_t l) { return val[off[c - 1] + l - 1]; }

// Residual d = MI - fit above the fit (:448-450).  A length beyond the number of groups gives NA in R, and the link drops
// out of which(diff > 0).
template <class Off>
__host__ __device__ __forceinline__ bool residual(const double* val, const Off& off, int c, int64_t l, double mi, double& d) {
  if (l > off[c] - off[c - 1]) return false;
  d = mi - fit_at(val, off, c, l);
  return d > 0;
}

// ---- log of the regularised incomplete beta function, continued fraction evaluated with the modified Lentz scheme ----
// log I_x(a, b) given log(x) and log(1 - x); converges fast for x < (a + 1) / (a + b + 2).
__host__ __device__ inline double log_ibeta_cf(double a, double b, double x, double logx, double log1mx, double lbeta) {
  const double tiny = 1e-300, eps = 1e-16;
  const double qab = a + b, qap = a + 1.0, qam = a - 1.0;
  double c = 1.0, d = 1.0 - qab * x / qap;
  if (fabs(d) < tiny) d = tiny;
  d = 1.0 / d;
  double h = d;
  for (int m = 1; m <= 10000; m++) {
    const double m2 = 2.0 * m;
    double aa = m * (b - m) * x / ((qam + m2) * (a + m2));
    d = 1.0 + aa * d; if (fabs(d) < tiny) d = tiny;
    c = 1.0 + aa / c; if (fabs(c) < tiny) c = tiny;
    d = 1.0 / d;
    h *= d * c;
    aa = -(a + m) * (qab + m) * x / ((a + m2) * (qap + m2));
    d = 1.0 + aa * d; if (fabs(d) < tiny) d = tiny;
    c = 1.0 + aa / c; if (fabs(c) < tiny) c = tiny;
    d = 1.0 / d;
    const double del = d * c;
    h *= del;
    if (fabs(del - 1.0) < eps) break;
  }
  return a * logx + b * log1mx - lbeta - log(a) + log(h);
}

// -pbeta(x, a, b, lower.tail = FALSE, log.p = TRUE), 0 < x < 1 (:453)
__host__ __device__ inline double neg_log_upper_beta(double x, double a, double b, double lbeta) {
  const double logx = log(x), log1mx = log1p(-x);
  const double y = 1.0 - x;
  if (y < (b + 1.0) / (a + b + 2.0)) return -log_ibeta_cf(b, a, y, log1mx, logx, lbeta);  // upper tail directly: I_{1-x}(b, a)
  const double lp = log_ibeta_cf(a, b, x, logx, log1mx, lbeta);                              // lower tail, then complement
  return -log1p(-exp(lp));
}

// log B(a, b) (host: the beta fit and the shapes the srp_max passes take)
inline double lbeta_fn(double a, double b) {
  int sg;
  return lgamma_r(a, &sg) + lgamma_r(b, &sg) - lgamma_r(a + b, &sg);
}

// Longest length a member link can have, which sizes the (cluster, length) groups: len < sr_dist bounds it unless
// sr_dist is huge; then -1, and the caller takes the longest length present (one pass over the links).
inline int32_t max_len_bound(double sr_dist) {
  return sr_dist <= (double)(1 << 18) ? (int32_t)std::max(0.0, ceil(sr_dist) - 1.0) : -1;
}

}  // namespace ldwpost
