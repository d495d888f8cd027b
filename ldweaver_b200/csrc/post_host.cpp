// Host side of what follows the scan inside perform_MI_computation (SURVEY.md section 8f, rows 1 and 3):
//   ldw_sr_postprocess  = mergeNsort_sr_links   (R/computePairwiseMI.R:400-495)
//   ldw_run_aracne      = runARACNE             (R/io_functions.R:101-164; .compareToRow / .vecPosMatch / .compareTriplet
//                                                src/computeMI.cpp:25-79, .fast_intersect src/fintersect.cpp:6-33)
// These steps consume every short-range link the device produced (9e7 rows at 616 x 100k).  The reference walks them as
// R data.frames: dplyr group_by + quantile per length, a dbeta() over all positive residuals for each of the ~60-100
// objective evaluations of optim(), and for ARACNE a full scan of the link table per checked link.  Here:
//   * lengths are small integers, so the grouping is a counting sort and the 95th percentiles are nth_element calls on
//     contiguous slices, spread over host threads;
//   * the beta log-likelihood only depends on the data through n, sum(log x) and sum(log(1-x)), so each Nelder-Mead
//     evaluation is O(1) after one pass; the simplex iteration itself follows stats::optim's nmmin step by step;
//   * -log of the upper beta tail is evaluated per link in log space (continued fraction), threads over links;
//   * ARACNE uses a position -> (partner, MI, row) adjacency built once; the triangle test per checked link is a merge of
//     two sorted neighbour lists, first-row-wins on duplicates exactly as .vecPosMatch picks them.
// Pure host code: nothing here needs a device (the link columns are already in host memory when R would see them).
#include <math.h>
#include <stdint.h>
#include <string.h>
#include <stdio.h>
#include <stdlib.h>
#include <sys/mman.h>

#include <algorithm>
#include <atomic>
#include <exception>
#include <new>
#include <chrono>
#include <memory>
#include <mutex>
#include <numeric>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "host_util.h"
#include "post_host.h"
#include "sr_stats.cuh"
#include "../../include/ldw.h"

using ldwpost::SrPostPriv;

namespace {

int host_threads() {  // LDW_HOST_THREADS=<n> overrides (results never depend on it: every pass works on fixed pieces)
  if (const char* e = getenv("LDW_HOST_THREADS")) {
    const int v = atoi(e);
    if (v >= 1) return std::min(v, 256);
  }
  unsigned h = std::thread::hardware_concurrency();
  if (h == 0) h = 4;
  return (int)std::min<unsigned>(h, 32);
}

// fn(chunk_index) over [0, n) with dynamic scheduling (chunks have uneven cost: groups of different sizes).
template <class F>
void parallel_dynamic(int64_t n, F fn) {
  const int nt = (int)std::min<int64_t>(host_threads(), n);
  if (nt <= 1) { for (int64_t i = 0; i < n; i++) fn(i); return; }
  std::atomic<int64_t> next(0);
  std::exception_ptr err;  // first exception of a worker (std::bad_alloc of a growing vector), rethrown on the caller
  std::mutex err_mu;
  std::vector<std::thread> th;
  th.reserve(nt);
  for (int t = 0; t < nt; t++)
    th.emplace_back([&]() {
      try {
        for (;;) { const int64_t i = next.fetch_add(1); if (i >= n) break; fn(i); }
      } catch (...) {
        std::lock_guard<std::mutex> g(err_mu);
        if (!err) err = std::current_exception();
        next.store(n);
      }
    });
  for (auto& x : th) x.join();
  if (err) std::rethrow_exception(err);
}

using ldw::guarded;

struct PhaseTimer {  // LDW_DBG_TIMING=1: phase times on stderr (never stdout)
  bool on;
  std::chrono::steady_clock::time_point t;
  PhaseTimer() : on(getenv("LDW_DBG_TIMING") != nullptr), t(std::chrono::steady_clock::now()) {}
  void lap(const char* what, int c) {
    if (!on) return;
    const auto n = std::chrono::steady_clock::now();
    fprintf(stderr, "[ldw_sr_postprocess] cluster %d %-28s %8.2f ms\n", c, what, std::chrono::duration<double, std::milli>(n - t).count());
    t = n;
  }
};

// Large scratch array, 2 MB-aligned.  LDW_THP=1 asks for transparent huge pages (madvise); off by default: the grouping
// below is organised so that it does not need them, and huge-page faults can stall on compaction.
template <class T>
struct HugeArray {
  T* p = nullptr;
  size_t n = 0;
  explicit HugeArray(size_t count) : n(count) {
    const size_t bytes = std::max<size_t>(sizeof(T) * count, 1), two_mb = size_t(2) << 20;
    void* q = nullptr;
    if (posix_memalign(&q, two_mb, (bytes + two_mb - 1) / two_mb * two_mb) != 0) q = nullptr;
    if (q && getenv("LDW_THP")) madvise(q, (bytes + two_mb - 1) / two_mb * two_mb, MADV_HUGEPAGE);
    p = (T*)q;
  }
  ~HugeArray() { free(p); }
  HugeArray(const HugeArray&) = delete;
  HugeArray& operator=(const HugeArray&) = delete;
  T* data() { return p; }
  T& operator[](size_t i) { return p[i]; }
};

constexpr int64_t kChunk = 1 << 16;  // fixed, so that chunked sums do not depend on the number of threads

// stats::quantile.default(type = 7) of one probability; reorders x.
double quantile7(double* x, int64_t n, double prob) {
  const double index = 1.0 + (double)std::max<int64_t>(n - 1, 0) * prob;
  const int64_t lo = (int64_t)floor(index), hi = (int64_t)ceil(index);
  std::nth_element(x, x + (lo - 1), x + n);
  double qs = x[lo - 1];
  if (hi > lo) {
    const double xhi = *std::min_element(x + lo, x + n);
    if (index > (double)lo && xhi != qs) {
      const double h = index - (double)lo;
      qs = (1.0 - h) * qs + h * xhi;
    }
  }
  return qs;
}

// Least squares of y on [x, 1] through Householder QR (what LAPACK dgels does for arma::solve on a tall matrix).
void ols2(const std::vector<double>& x, const std::vector<double>& y, double coef[2]) {
  const size_t n = x.size();
  std::vector<double> a0(x), a1(n, 1.0), b(y);
  auto house = [&](std::vector<double>& col, size_t k, std::vector<double>* other) {
    double nrm = 0;
    for (size_t i = k; i < n; i++) nrm += col[i] * col[i];
    nrm = sqrt(nrm);
    if (nrm == 0) return;
    const double alpha = col[k] > 0 ? -nrm : nrm;
    std::vector<double> v(n - k);
    for (size_t i = k; i < n; i++) v[i - k] = col[i];
    v[0] -= alpha;
    double vv = 0;
    for (double t : v) vv += t * t;
    if (vv == 0) return;
    auto apply = [&](std::vector<double>& z) {
      double d = 0;
      for (size_t i = k; i < n; i++) d += v[i - k] * z[i];
      d = 2 * d / vv;
      for (size_t i = k; i < n; i++) z[i] -= d * v[i - k];
    };
    if (other) apply(*other);
    apply(b);
    col[k] = alpha;
    for (size_t i = k + 1; i < n; i++) col[i] = 0;
  };
  house(a0, 0, &a1);
  house(a1, 1, nullptr);
  // R = [[a0[0], a1[0]], [0, a1[1]]]
  coef[1] = b[1] / a1[1];
  coef[0] = (b[0] - a1[0] * coef[1]) / a0[0];
}

// ---- stats::optim(method = "Nelder-Mead"): R's nmmin (src/appl/optim.c), two parameters, optim's default controls ----
struct BetaNll {
  double n, s1, s2;  // count, sum(log x), sum(log(1 - x))
  double operator()(const double* p) const {
    const double a = p[0], b = p[1];
    if (!(a > 0 && b > 0)) return NAN;  // dbeta gives NaN there; nmmin replaces a non-finite value by `big`
    return -((a - 1) * s1 + (b - 1) * s2 - n * ldwpost::lbeta_fn(a, b));
  }
};

template <class Fn>
int nmmin2(const Fn& fn, const double start[2], double xout[2], double* fmin, int* fncount) {
  const int n = 2, n1 = 3, C = 4;
  const double big = 1.0e35, alpha = 1.0, bet = 0.5, gamm = 2.0, abstol = -INFINITY, intol = sqrt(2.220446049250313e-16);
  const int maxit = 500;
  double P[3][4] = {{0}};
  double B[2] = {start[0], start[1]};
  int fail = 0;
  double f = fn(B);
  if (!std::isfinite(f)) return -1;
  int funcount = 1;
  const double convtol = intol * (fabs(f) + intol);
  P[n1 - 1][0] = f;
  for (int i = 0; i < n; i++) P[i][0] = B[i];
  int L = 1;
  double size = 0.0, step = 0.0;
  for (int i = 0; i < n; i++) if (0.1 * fabs(B[i]) > step) step = 0.1 * fabs(B[i]);
  if (step == 0.0) step = 0.1;
  for (int j = 2; j <= n1; j++) {
    for (int i = 0; i < n; i++) P[i][j - 1] = B[i];
    double trystep = step;
    while (P[j - 2][j - 1] == B[j - 2]) { P[j - 2][j - 1] = B[j - 2] + trystep; trystep *= 10; }
    size += trystep;
  }
  double oldsize = size;
  bool calcvert = true;
  do {
    if (calcvert) {
      for (int j = 0; j < n1; j++)
        if (j + 1 != L) {
          for (int i = 0; i < n; i++) B[i] = P[i][j];
          f = fn(B);
          if (!std::isfinite(f)) f = big;
          funcount++;
          P[n1 - 1][j] = f;
        }
      calcvert = false;
    }
    double VL = P[n1 - 1][L - 1], VH = VL;
    int H = L;
    for (int j = 1; j <= n1; j++)
      if (j != L) {
        f = P[n1 - 1][j - 1];
        if (f < VL) { L = j; VL = f; }
        if (f > VH) { H = j; VH = f; }
      }
    if (VH <= VL + convtol || VL <= abstol) break;
    for (int i = 0; i < n; i++) {
      double temp = -P[i][H - 1];
      for (int j = 0; j < n1; j++) temp += P[i][j];
      P[i][C - 1] = temp / n;
    }
    for (int i = 0; i < n; i++) B[i] = (1.0 + alpha) * P[i][C - 1] - alpha * P[i][H - 1];
    f = fn(B);
    if (!std::isfinite(f)) f = big;
    funcount++;
    const double VR = f;
    if (VR < VL) {
      P[n1 - 1][C - 1] = f;
      for (int i = 0; i < n; i++) {
        f = gamm * B[i] + (1 - gamm) * P[i][C - 1];
        P[i][C - 1] = B[i];
        B[i] = f;
      }
      f = fn(B);
      if (!std::isfinite(f)) f = big;
      funcount++;
      if (f < VR) {
        for (int i = 0; i < n; i++) P[i][H - 1] = B[i];
        P[n1 - 1][H - 1] = f;
      } else {
        for (int i = 0; i < n; i++) P[i][H - 1] = P[i][C - 1];
        P[n1 - 1][H - 1] = VR;
      }
    } else {
      if (VR < VH) {
        for (int i = 0; i < n; i++) P[i][H - 1] = B[i];
        P[n1 - 1][H - 1] = VR;
      }
      for (int i = 0; i < n; i++) B[i] = (1 - bet) * P[i][H - 1] + bet * P[i][C - 1];
      f = fn(B);
      if (!std::isfinite(f)) f = big;
      funcount++;
      if (f < P[n1 - 1][H - 1]) {
        for (int i = 0; i < n; i++) P[i][H - 1] = B[i];
        P[n1 - 1][H - 1] = f;
      } else if (VR >= VH) {
        calcvert = true;
        size = 0.0;
        for (int j = 0; j < n1; j++)
          if (j + 1 != L)
            for (int i = 0; i < n; i++) {
              P[i][j] = bet * (P[i][j] - P[i][L - 1]) + P[i][L - 1];
              size += fabs(P[i][j] - P[i][L - 1]);
            }
        if (size < oldsize) oldsize = size;
        else { fail = 10; break; }
      }
    }
  } while (funcount <= maxit);
  if (funcount > maxit) fail = 1;
  *fmin = P[n1 - 1][L - 1];
  for (int i = 0; i < n; i++) xout[i] = P[i][L - 1];
  *fncount = funcount;
  return fail;
}

struct KeyHash {
  size_t operator()(const std::pair<int64_t, int64_t>& k) const {
    uint64_t h = (uint64_t)k.first * 0x9E3779B97F4A7C15ull ^ ((uint64_t)k.second + 0x7F4A7C15ull + ((uint64_t)k.first << 6));
    h ^= h >> 29; h *= 0xBF58476D1CE4E5B9ull; h ^= h >> 32;
    return (size_t)h;
  }
};

// sr_links_red = srp_max > srp_cutoff; sr_links_ARACNE_check = MI >= min(sr_links_red$MI)  (:494-495), over the df rows
// of S, whose MI are MI[S.row[i]].
void select_red_chk(SrPostPriv& S, const double* MI, double srp_cutoff) {
  const int64_t ndf = (int64_t)S.row.size();
  double min_mi = INFINITY;
  for (int64_t i = 0; i < ndf; i++)
    if (S.srp[i] > srp_cutoff) { S.red.push_back(i); min_mi = std::min(min_mi, MI[S.row[i]]); }
  for (int64_t i = 0; i < ndf; i++)
    if (MI[S.row[i]] >= min_mi) S.chk.push_back(i);
}

}  // namespace

namespace ldwpost {

int decay_fits(SrPostPriv& S, int32_t nclust, int64_t nl, const std::vector<int64_t>& glist, const std::vector<double>& gq) {
  size_t t = 0;
  for (int32_t c = 1; c <= nclust; c++) {
    std::vector<double> lx, ly;
    const size_t base = S.fit_len.size();
    for (; t < glist.size() && glist[t] < (int64_t)c * nl; t++) {
      const int32_t l = (int32_t)(glist[t] - (int64_t)(c - 1) * nl);
      S.fit_len.push_back(l);
      S.fit_q95.push_back(gq[t]);
      lx.push_back(log((double)l));
      ly.push_back(log(gq[t]));
    }
    const int64_t ng = (int64_t)lx.size();
    if (ng < 2) return ldw::set_error(LDW_ERR_ARG, "ldw_sr_postprocess: cluster %d has fewer than two distinct link lengths", (int)c);
    double coef[2];
    ols2(lx, ly, coef);
    S.fit_val.resize(base + ng);
    for (int64_t gi = 0; gi < ng; gi++) S.fit_val[base + gi] = exp(lx[gi] * coef[0] + coef[1]);
    S.fit_off.push_back((int64_t)(base + ng));
    S.coef.push_back(coef[0]);
    S.coef.push_back(coef[1]);
  }
  return 0;
}

// fitdist(x, "beta") (:452) from the sufficient statistics: moment start values (v = biased variance), then optim's
// Nelder-Mead on the negative log-likelihood n lbeta(a, b) - (a - 1) sum(log x) - (b - 1) sum(log(1 - x)).
int beta_fit(SrPostPriv& S, int32_t c, int64_t npos, double s1, double s2, double mean, double v, double par[2]) {
  const double aux = mean * (1 - mean) / v - 1;
  const double start[2] = {mean * aux, (1 - mean) * aux};
  BetaNll nll{(double)npos, s1, s2};
  double fmin;
  int evals = 0;
  const int fail = nmmin2(nll, start, par, &fmin, &evals);
  if (fail < 0) return ldw::set_error(LDW_ERR_ARG, "ldw_sr_postprocess: cluster %d: the beta likelihood cannot be evaluated at the initial parameters (%g, %g)", (int)c, start[0], start[1]);
  S.shape.push_back(par[0]); S.shape.push_back(par[1]);
  S.start.push_back(start[0]); S.start.push_back(start[1]);
  S.n_pos.push_back(npos);
  S.nm_evals.push_back(evals);
  S.nm_fail.push_back(fail);
  return 0;
}

// Links seen from two clusters: one row per distinct link, the one with the larger srp_max; groups in order of first
// appearance, first maximum wins (:474-483, data.table `.I[which.max(srp_max)], by = keys`).
std::vector<int64_t> dedup(const ldw_links& L, const std::vector<int64_t>& at, const std::vector<double>& srp) {
  struct Grp { int64_t first, best; };
  std::unordered_map<std::pair<int64_t, int64_t>, std::vector<int64_t>, KeyHash> index;  // (pos1, pos2) -> groups
  index.reserve(at.size());
  std::vector<Grp> groups;
  groups.reserve(at.size());
  auto same = [&](int64_t a, int64_t b) {
    return L.pos1[a] == L.pos1[b] && L.pos2[a] == L.pos2[b] && L.clust1[a] == L.clust1[b] && L.clust2[a] == L.clust2[b] &&
           L.len[a] == L.len[b] && L.MI[a] == L.MI[b];
  };
  for (int64_t k = 0; k < (int64_t)at.size(); k++) {
    const int64_t r = at[k];
    auto& lst = index[{(int64_t)L.pos1[r], (int64_t)L.pos2[r]}];
    int64_t g = -1;
    for (int64_t gi : lst) if (same(at[groups[gi].first], r)) { g = gi; break; }
    if (g < 0) { lst.push_back((int64_t)groups.size()); groups.push_back({k, k}); }
    else if (srp[k] > srp[groups[g].best]) groups[g].best = k;
  }
  std::vector<int64_t> win;
  win.reserve(groups.size());
  for (const Grp& g : groups) win.push_back(g.best);
  return win;
}

void publish(SrPostPriv& S, int32_t nclust, ldw_sr_post* out) {
  out->n_df = (int64_t)S.row.size();
  out->clust_c = S.clust_c.data(); out->row = S.row.data(); out->srp_max = S.srp.data();
  out->n_red = (int64_t)S.red.size(); out->red = S.red.data();
  out->n_chk = (int64_t)S.chk.size(); out->chk = S.chk.data();
  out->nclust = nclust;
  out->fit_off = S.fit_off.data(); out->fit_len = S.fit_len.data(); out->fit_q95 = S.fit_q95.data(); out->fit_val = S.fit_val.data();
  out->coef = S.coef.data(); out->shape = S.shape.data(); out->start = S.start.data();
  out->n_pos = S.n_pos.data(); out->nm_evals = S.nm_evals.data(); out->nm_fail = S.nm_fail.data();
}

int check_groups(const std::vector<int64_t>& goff, int32_t nclust, int64_t nl) {
  for (int32_t c = 1; c <= nclust; c++)
    if (goff[(int64_t)c * nl] == goff[(int64_t)(c - 1) * nl])
      return ldw::set_error(LDW_ERR_ARG, "ldw_sr_postprocess: cluster %d holds no short-range link with 0 < len < sr_dist", (int)c);
  return 0;
}

int check_residuals(int bad_c) {
  if (bad_c) return ldw::set_error(LDW_ERR_ARG, "ldw_sr_postprocess: cluster %d: values must be in [0-1] to fit a beta distribution", bad_c);
  return 0;
}

int check_npos(int32_t c, int64_t npos) {
  if (npos < 2) return ldw::set_error(LDW_ERR_ARG, "ldw_sr_postprocess: cluster %d has fewer than two links above the fitted decay", (int)c);
  return 0;
}

}  // namespace ldwpost

extern "C" void ldw_sr_post_free(ldw_sr_post* p) {
  if (!p) return;
  delete (SrPostPriv*)p->priv;
  memset(p, 0, sizeof(*p));
}

extern "C" int ldw_sr_postprocess(const ldw_links* sr, int32_t nclust, double sr_dist, double srp_cutoff, ldw_sr_post* out) {
  return guarded("ldw_sr_postprocess", [&]() -> int {
  if (!sr || !out) return ldw::set_error(LDW_ERR_ARG, "ldw_sr_postprocess: null argument");
  memset(out, 0, sizeof(*out));
  if (nclust < 1) return ldw::set_error(LDW_ERR_ARG, "ldw_sr_postprocess: nclust must be >= 1");
  const int64_t N = sr->n;
  if (N > 0 && (!sr->pos1 || !sr->pos2 || !sr->clust1 || !sr->clust2 || !sr->len || !sr->MI))
    return ldw::set_error(LDW_ERR_ARG, "ldw_sr_postprocess: null link column");
  std::unique_ptr<SrPostPriv> S(new SrPostPriv());
  S->fit_off.assign(1, 0);
  std::vector<int64_t> dup_row;
  std::vector<int32_t> dup_c;
  std::vector<double> dup_srp;
  // Every pass below walks the link table ONCE for all clusters (a link belongs to clust1 and, if different, clust2;
  // R/computePairwiseMI.R:372-376), in a fixed number of contiguous pieces so that the results do not depend on the
  // number of host threads.
  PhaseTimer tm;
  // ---- longest length present (sizes the histograms) ----
  int32_t maxlen = ldwpost::max_len_bound(sr_dist);
  if (maxlen < 0) {
    maxlen = 0;
    const int64_t P0 = 256, p0sz = (N + P0 - 1) / P0;
    std::vector<int32_t> mx0(P0, 0);
    parallel_dynamic(P0, [&](int64_t k) {
      int32_t ml = 0;
      for (int64_t i = k * p0sz; i < std::min(N, (k + 1) * p0sz); i++) {
        int32_t ca, cb, l;
        if (ldwpost::member(*sr, i, sr_dist, nclust, ca, cb, l)) ml = std::max(ml, l);
      }
      mx0[k] = ml;
    });
    for (int64_t k = 0; k < P0; k++) maxlen = std::max(maxlen, mx0[k]);
    tm.lap("longest length", 0);
  }

  // ---- group_by(len) %>% summarise(quantile(MI, 0.95))  (:422): counting sort by (cluster, length) -- per-piece
  //      histograms turned into write cursors, so the scatter is parallel and deterministic -- then one selection per group ----
  const int64_t nl = (int64_t)maxlen + 1;
  const int64_t G = (int64_t)nclust * nl;                       // group id = (c - 1) * nl + len
  int64_t B = std::min<int64_t>(64, std::max<int64_t>(1, (int64_t)(128ll << 20) / (G * 4)));  // histogram memory <= 128 MB
  B = std::max<int64_t>(1, std::min<int64_t>(B, (N + kChunk - 1) / kChunk));
  const int64_t bsz = (N + B - 1) / B;
  std::vector<std::vector<int32_t>> hist(B);
  parallel_dynamic(B, [&](int64_t k) {
    std::vector<int32_t>& h = hist[k];
    h.assign((size_t)G, 0);
    for (int64_t i = k * bsz; i < std::min(N, (k + 1) * bsz); i++) {
      int32_t ca, cb, l;
      if (!ldwpost::member(*sr, i, sr_dist, nclust, ca, cb, l)) continue;
      if (ca) h[(ca - 1) * nl + l]++;
      if (cb) h[(cb - 1) * nl + l]++;
    }
  });
  std::vector<int64_t> gcount((size_t)G, 0), goff((size_t)G + 1, 0);
  for (int64_t k = 0; k < B; k++) for (int64_t g = 0; g < G; g++) gcount[g] += hist[k][g];
  for (int64_t g = 0; g < G; g++) goff[g + 1] = goff[g] + gcount[g];
  LDW_TRY(ldwpost::check_groups(goff, nclust, nl));
  std::vector<int64_t> glist;                                   // non-empty groups, cluster-major, ascending length
  for (int64_t g = 0; g < G; g++) if (gcount[g] > 0) glist.push_back(g);
  std::vector<double> gq((size_t)glist.size());
  {
    // Two levels, so that no pass writes through more than a few hundred cursors (with ~6 x 10^4 groups a direct scatter
    // costs a TLB miss per element): first into <= 512 buckets of consecutive groups -- each bucket's slice of the array is
    // where its groups will finally live --, then bucket by bucket (a few MB each, one thread per bucket) into a local
    // scratch ordered by group, from which the bucket's percentiles are taken.
    int sh = 0;
    while (((G - 1) >> sh) + 1 > 512) sh++;
    const int64_t NB = ((G - 1) >> sh) + 1;
    const int64_t E = goff[G];
    HugeArray<double> tmp_mi((size_t)E);
    HugeArray<uint32_t> tmp_g((size_t)E);
    if (!tmp_mi.data() || !tmp_g.data()) return ldw::set_error(LDW_ERR_NOMEM, "ldw_sr_postprocess: out of memory (%lld values)", (long long)E);
    std::vector<int64_t> bcur((size_t)B * NB);
    {
      std::vector<int64_t> run((size_t)NB);
      for (int64_t b = 0; b < NB; b++) run[b] = goff[b << sh];
      for (int64_t k = 0; k < B; k++) {
        for (int64_t b = 0; b < NB; b++) {
          bcur[(size_t)k * NB + b] = run[b];
          int64_t c = 0;
          for (int64_t g = b << sh; g < std::min(G, (b + 1) << sh); g++) c += hist[k][g];
          run[b] += c;
        }
        std::vector<int32_t>().swap(hist[k]);
      }
    }
    parallel_dynamic(B, [&](int64_t k) {
      int64_t* cu = bcur.data() + (size_t)k * NB;
      for (int64_t i = k * bsz; i < std::min(N, (k + 1) * bsz); i++) {
        int32_t cc[2], l;
        if (!ldwpost::member(*sr, i, sr_dist, nclust, cc[0], cc[1], l)) continue;
        const double v = sr->MI[i];
        for (int q = 0; q < 2; q++) {
          if (!cc[q]) continue;
          const int64_t g = (int64_t)(cc[q] - 1) * nl + l, b = g >> sh, at = cu[b]++;
          tmp_mi[(size_t)at] = v;
          tmp_g[(size_t)at] = (uint32_t)(g - (b << sh));
        }
      }
    });
    tm.lap("scatter into buckets", 0);
    std::vector<double> gq_by_group((size_t)G, 0.0);
    parallel_dynamic(NB, [&](int64_t b) {
      const int64_t g0 = b << sh, g1 = std::min(G, (b + 1) << sh), lo = goff[g0], hi = goff[g1];
      if (hi == lo) return;
      std::vector<double> sc((size_t)(hi - lo));
      std::vector<int64_t> cur((size_t)(g1 - g0));
      for (int64_t g = g0; g < g1; g++) cur[g - g0] = goff[g] - lo;
      for (int64_t e = lo; e < hi; e++) sc[(size_t)cur[tmp_g[(size_t)e]]++] = tmp_mi[(size_t)e];
      for (int64_t g = g0; g < g1; g++)
        if (gcount[g] > 0) gq_by_group[g] = quantile7(sc.data() + (goff[g] - lo), gcount[g], 0.95);
    });
    for (size_t t = 0; t < glist.size(); t++) gq[t] = gq_by_group[glist[t]];
    tm.lap("group + quantiles", 0);
  }
  // ---- fastLm(cbind(log(len), 1), log(max)); fit = exp(fitted)  (:428-429), per cluster ----
  if (int rc = ldwpost::decay_fits(*S, nclust, nl, glist, gq)) return rc;
  tm.lap("decay fits", 0);

  // ---- residuals above the fit (:448-450), the fitted values subscripted by the value of len (sr_stats.cuh) ----
  const int64_t R = std::max<int64_t>(1, std::min<int64_t>(256, (N + kChunk - 1) / kChunk));
  const int64_t rsz = (N + R - 1) / R;
  const int C1 = nclust + 1;
  std::vector<int64_t> pcnt((size_t)(R + 1) * C1, 0);
  std::vector<double> cs1((size_t)R * C1, 0), cs2((size_t)R * C1, 0), csum((size_t)R * C1, 0);
  std::vector<std::vector<int64_t>> lrow((size_t)R * C1);      // per piece and cluster: links above the fit, in scan order
  std::vector<std::vector<double>> lx((size_t)R * C1);
  std::atomic<int> bad(0);
  parallel_dynamic(R, [&](int64_t k) {
    for (int64_t i = k * rsz; i < std::min(N, (k + 1) * rsz); i++) {
      int32_t cc[2], l;
      if (!ldwpost::member(*sr, i, sr_dist, nclust, cc[0], cc[1], l)) continue;
      for (int q = 0; q < 2; q++) {
        double d;
        if (!cc[q] || !ldwpost::residual(S->fit_val.data(), S->fit_off.data(), cc[q], l, sr->MI[i], d)) continue;
        if (d > 1) bad.store(cc[q]);
        const size_t o = (size_t)k * C1 + cc[q];
        lrow[o].push_back(i); lx[o].push_back(d);
        cs1[o] += log(d); cs2[o] += log1p(-d); csum[o] += d;
      }
    }
    for (int c = 1; c <= nclust; c++) pcnt[(size_t)(k + 1) * C1 + c] = (int64_t)lrow[(size_t)k * C1 + c].size();
  });
  LDW_TRY(ldwpost::check_residuals(bad.load()));
  for (int64_t k = 0; k < R; k++) for (int c = 1; c <= nclust; c++) pcnt[(size_t)(k + 1) * C1 + c] += pcnt[(size_t)k * C1 + c];
  std::vector<std::vector<int64_t>> prow(C1);
  std::vector<std::vector<double>> px(C1);
  for (int32_t c = 1; c <= nclust; c++) {
    const int64_t npos = pcnt[(size_t)R * C1 + c];
    LDW_TRY(ldwpost::check_npos(c, npos));
    prow[c].resize((size_t)npos);
    px[c].resize((size_t)npos);
  }
  parallel_dynamic(R, [&](int64_t k) {
    for (int c = 1; c <= nclust; c++) {
      const size_t o = (size_t)k * C1 + c;
      std::copy(lrow[o].begin(), lrow[o].end(), prow[c].begin() + pcnt[o]);
      std::copy(lx[o].begin(), lx[o].end(), px[c].begin() + pcnt[o]);
      std::vector<int64_t>().swap(lrow[o]);
      std::vector<double>().swap(lx[o]);
    }
  });
  tm.lap("residuals", 0);

  for (int32_t c = 1; c <= nclust; c++) {
    const int64_t npos = (int64_t)px[c].size();
    const std::vector<double>& x = px[c];
    // ---- fitdist(x, "beta") (:452): moment start values, then optim's Nelder-Mead on the negative log-likelihood ----
    long double s1 = 0, s2 = 0, sm = 0;
    for (int64_t k = 0; k < R; k++) { s1 += cs1[(size_t)k * C1 + c]; s2 += cs2[(size_t)k * C1 + c]; sm += csum[(size_t)k * C1 + c]; }
    const double mean = (double)(sm / (long double)npos);
    const int64_t pchunks = (npos + kChunk - 1) / kChunk;
    std::vector<double> cvar(pchunks, 0);
    parallel_dynamic(pchunks, [&](int64_t k) {
      const int64_t lo = k * kChunk, hi = std::min(npos, lo + kChunk);
      double s = 0;
      for (int64_t i = lo; i < hi; i++) { const double t = x[i] - mean; s += t * t; }
      cvar[k] = s;
    });
    long double ss = 0;
    for (double v : cvar) ss += v;
    const double var_unbiased = (double)(ss / (long double)(npos - 1));
    const double v = (double)(npos - 1) / (double)npos * var_unbiased;
    double par[2];
    if (int rc = ldwpost::beta_fit(*S, c, npos, (double)s1, (double)s2, mean, v, par)) return rc;
    tm.lap("beta fit", c);
    // ---- srp = -pbeta(x, shape1, shape2, lower.tail = F, log.p = T)  (:453) ----
    const double lbeta = ldwpost::lbeta_fn(par[0], par[1]);
    std::vector<double> psrp(npos);
    parallel_dynamic(pchunks, [&](int64_t k) {
      const int64_t lo = k * kChunk, hi = std::min(npos, lo + kChunk);
      for (int64_t i = lo; i < hi; i++) psrp[i] = x[i] < 1.0 ? ldwpost::neg_log_upper_beta(x[i], par[0], par[1], lbeta) : INFINITY;
    });
    tm.lap("srp", c);
    // ---- same-cluster links go to sr_links_df, links between clusters to duplink_df (:460-468) ----
    S->row.reserve(S->row.size() + (size_t)npos); S->clust_c.reserve(S->clust_c.size() + (size_t)npos); S->srp.reserve(S->srp.size() + (size_t)npos);
    for (int64_t i = 0; i < npos; i++) {
      const int64_t r = prow[c][i];
      if (std::isnan(psrp[i])) continue;  // :458
      if (sr->clust1[r] != sr->clust2[r]) { dup_row.push_back(r); dup_c.push_back(c); dup_srp.push_back(psrp[i]); }
      else { S->row.push_back(r); S->clust_c.push_back(c); S->srp.push_back(psrp[i]); }
    }
    std::vector<int64_t>().swap(prow[c]);
    std::vector<double>().swap(px[c]);
  }
  tm.lap("(last cluster's append)", nclust);
  for (int64_t k : ldwpost::dedup(*sr, dup_row, dup_srp)) { S->row.push_back(dup_row[k]); S->clust_c.push_back(dup_c[k]); S->srp.push_back(dup_srp[k]); }
  select_red_chk(*S, sr->MI, srp_cutoff);

  tm.lap("dedup + red/chk", 0);
  ldwpost::publish(*S, nclust, out);
  out->priv = S.release();
  return 0;
  });
}

// Building blocks exposed for the parity tests: the Nelder-Mead iteration on Rosenbrock's function (the example of R's
// ?optim, whose printed result pins the restatement: par 1.000260 1.000506, value 8.825241e-08, 195 evaluations) and the
// log upper beta tail.
extern "C" int ldw_nm_rosenbrock(const double* start, double* par_out, double* value_out, int* count_out) {
  return guarded("ldw_nm_rosenbrock", [&]() -> int {
  if (!start || !par_out || !value_out || !count_out) return ldw::set_error(LDW_ERR_ARG, "ldw_nm_rosenbrock: null argument");
  struct Fr { double operator()(const double* x) const { const double t = x[1] - x[0] * x[0], u = 1 - x[0]; return 100 * t * t + u * u; } };
  const int fail = nmmin2(Fr(), start, par_out, value_out, count_out);
  if (fail < 0) return ldw::set_error(LDW_ERR_ARG, "ldw_nm_rosenbrock: function cannot be evaluated at initial parameters");
  return 0;
  });
}

extern "C" int ldw_neg_log_pbeta_upper(const double* x, int64_t n, double shape1, double shape2, double* out) {
  return guarded("ldw_neg_log_pbeta_upper", [&]() -> int {
  if (n < 0 || (n > 0 && (!x || !out))) return ldw::set_error(LDW_ERR_ARG, "ldw_neg_log_pbeta_upper: bad argument");
  if (!(shape1 > 0 && shape2 > 0)) return ldw::set_error(LDW_ERR_ARG, "ldw_neg_log_pbeta_upper: shapes must be positive");
  const double lbeta = ldwpost::lbeta_fn(shape1, shape2);
  parallel_dynamic((n + kChunk - 1) / kChunk, [&](int64_t k) {
    for (int64_t i = k * kChunk; i < std::min(n, (k + 1) * kChunk); i++)
      out[i] = x[i] <= 0 ? 0.0 : x[i] >= 1 ? INFINITY : ldwpost::neg_log_upper_beta(x[i], shape1, shape2, lbeta);
  });
  return 0;
  });
}

// ---------------------------------------------------------------------------------------------------------------------
// runARACNE
// ---------------------------------------------------------------------------------------------------------------------
extern "C" int ldw_run_aracne(int64_t n_chk, const double* chk_pos1, const double* chk_pos2, const double* chk_MI, int64_t n_full,
                              const double* full_pos1, const double* full_pos2, const double* full_MI, uint8_t* aracne_out) {
  return guarded("ldw_run_aracne", [&]() -> int {
  if (n_chk < 0 || n_full < 0) return ldw::set_error(LDW_ERR_ARG, "ldw_run_aracne: negative size");
  if ((n_chk > 0 && (!chk_pos1 || !chk_pos2 || !chk_MI || !aracne_out)) || (n_full > 0 && (!full_pos1 || !full_pos2 || !full_MI)))
    return ldw::set_error(LDW_ERR_ARG, "ldw_run_aracne: null argument");
  // positions -> dense ids
  std::unordered_map<int64_t, int32_t> id;
  id.reserve((size_t)n_full * 2);
  auto key = [](double p) { int64_t k; memcpy(&k, &p, 8); return k; };  // matches `==` on doubles except -0 / NaN (not positions)
  for (int64_t i = 0; i < n_full; i++) {
    id.emplace(key(full_pos1[i]), (int32_t)id.size());
    id.emplace(key(full_pos2[i]), (int32_t)id.size());
  }
  const int64_t nv = (int64_t)id.size();
  // adjacency in CSR form; a row with pos1 == pos2 == p contributes no neighbour to p (matX[matX != pX], R/io_functions.R:125)
  struct Nb { int32_t other; int64_t row; };
  std::vector<int64_t> off(nv + 1, 0);
  std::vector<int32_t> a(n_full), b(n_full);
  for (int64_t i = 0; i < n_full; i++) {
    a[i] = id[key(full_pos1[i])]; b[i] = id[key(full_pos2[i])];
    if (a[i] != b[i]) { off[a[i] + 1]++; off[b[i] + 1]++; }
  }
  for (int64_t v = 0; v < nv; v++) off[v + 1] += off[v];
  std::vector<Nb> adj(off[nv]);
  {
    std::vector<int64_t> cur(off.begin(), off.end() - 1);
    for (int64_t i = 0; i < n_full; i++)
      if (a[i] != b[i]) { adj[cur[a[i]]++] = {b[i], i}; adj[cur[b[i]]++] = {a[i], i}; }
  }
  // per vertex: neighbours sorted by id, first row first (.vecPosMatch takes the first row holding the neighbour)
  parallel_dynamic((nv + 1023) / 1024, [&](int64_t k) {
    for (int64_t v = k * 1024; v < std::min(nv, (k + 1) * 1024); v++)
      std::sort(adj.begin() + off[v], adj.begin() + off[v + 1],
                [](const Nb& x, const Nb& y) { return x.other != y.other ? x.other < y.other : x.row < y.row; });
  });
  parallel_dynamic((n_chk + 4095) / 4096, [&](int64_t k) {
    for (int64_t i = k * 4096; i < std::min(n_chk, (k + 1) * 4096); i++) {
      uint8_t keep = 1;  // links that cannot be checked stay TRUE (R/io_functions.R:112)
      auto ix = id.find(key(chk_pos1[i])), iz = id.find(key(chk_pos2[i]));
      if (ix != id.end() && iz != id.end()) {
        const int32_t X = ix->second, Z = iz->second;
        int64_t p = off[X], q = off[Z];
        const int64_t pe = off[X + 1], qe = off[Z + 1];
        const double mi0 = chk_MI[i];
        while (p < pe && q < qe) {
          const int32_t u = adj[p].other, w = adj[q].other;
          if (u < w) p++;
          else if (u > w) q++;
          else {
            // common neighbour (neither X nor Z itself can be one: X is not in its own list, and if u == Z then Z would
            // have to be in Z's list).  .fast_intersect pairs duplicates off one to one, and every copy is looked up by
            // .vecPosMatch to the FIRST row, so only the first rows matter.
            if (mi0 < full_MI[adj[p].row] && mi0 < full_MI[adj[q].row]) { keep = 0; break; }  // .compareTriplet
            while (p < pe && adj[p].other == u) p++;
            while (q < qe && adj[q].other == u) q++;
          }
        }
      }
      aracne_out[i] = keep;
    }
  });
  return 0;
  });
}

// ---------------------------------------------------------------------------------------------------------------------
// Link -> cell of its block's MI matrix (for the fp64 recomputation of short-range MI, ldw_mi_pairs_exact): pos2 is the
// row ("from") SNP and pos1 the column ("to") SNP on diagonal and off-diagonal blocks alike (R/computePairwiseMI.R:
// 319-323, quirk Q5); `block` is the make_blocks index the scan reported.  Binary searches over POS on host threads.
// ---------------------------------------------------------------------------------------------------------------------
extern "C" int ldw_links_to_cells(const int32_t* pos, int64_t n_snp, int64_t blk, const ldw_links* links, int32_t* from_local,
                                  int32_t* to_local) {
  return guarded("ldw_links_to_cells", [&]() -> int {
  if (!pos || !links || n_snp < 1 || blk < 1) return ldw::set_error(LDW_ERR_ARG, "ldw_links_to_cells: bad argument");
  const int64_t n = links->n;
  if (n > 0 && (!links->pos1 || !links->pos2 || !links->block || !from_local || !to_local))
    return ldw::set_error(LDW_ERR_ARG, "ldw_links_to_cells: null column");
  for (int64_t i = 1; i < n_snp; i++)
    if (pos[i] <= pos[i - 1]) return ldw::set_error(LDW_ERR_ARG, "ldw_links_to_cells: POS must be strictly increasing to map links back to SNPs");
  const int64_t nr = (n_snp + blk - 1) / blk;
  std::vector<int32_t> bf(nr * (nr + 1) / 2), bt(nr * (nr + 1) / 2);  // make_blocks order: (i, j >= i) row-major
  {
    int64_t k = 0;
    for (int64_t i = 0; i < nr; i++) for (int64_t j = i; j < nr; j++) { bf[k] = (int32_t)(i * blk); bt[k] = (int32_t)(j * blk); k++; }
  }
  const int64_t nblocks = (int64_t)bf.size();
  std::atomic<int64_t> bad(-1);
  parallel_dynamic((n + kChunk - 1) / kChunk, [&](int64_t c) {
    // the scan lists a block's links column by column (R/computePairwiseMI.R:309): the column SNP repeats and the row SNP
    // advances by one, so the previous answers (or their successors) are right almost every time
    int64_t ha = 0, hb = 0;
    auto find = [&](int32_t q, int64_t& hint) -> const int32_t* {
      if (pos[hint] == q) return pos + hint;
      if (hint + 1 < n_snp && pos[hint + 1] == q) return pos + (++hint);
      const int32_t* r = std::lower_bound(pos, pos + n_snp, q);
      if (r != pos + n_snp) hint = r - pos;
      return r;
    };
    for (int64_t i = c * kChunk; i < std::min(n, (c + 1) * kChunk); i++) {
      const int32_t* a = find(links->pos2[i], ha);
      const int32_t* b = find(links->pos1[i], hb);
      const int64_t k = links->block[i];
      if (a == pos + n_snp || *a != links->pos2[i] || b == pos + n_snp || *b != links->pos1[i] || k < 0 || k >= nblocks) { bad.store(i); continue; }
      const int64_t fl = (a - pos) - bf[k], tl = (b - pos) - bt[k];
      if (fl < 0 || fl >= blk || tl < 0 || tl >= blk) { bad.store(i); continue; }
      from_local[i] = (int32_t)fl;
      to_local[i] = (int32_t)tl;
    }
  });
  if (bad.load() >= 0) return ldw::set_error(LDW_ERR_ARG, "ldw_links_to_cells: link %lld does not belong to the block it names", (long long)bad.load());
  return 0;
  });
}

// ---------------------------------------------------------------------------------------------------------------------
// Copy of a library-owned link table into caller-allocated columns (R vectors, NumPy arrays) on host threads: 2.9 GB at
// 616 x 100k, which one thread moves at memcpy speed minus the page faults of a fresh destination.
// Any destination pointer may be NULL (column skipped).
// ---------------------------------------------------------------------------------------------------------------------
extern "C" int ldw_links_copy(const ldw_links* src, int32_t* pos1, int32_t* pos2, int32_t* clust1, int32_t* clust2, int32_t* len,
                              double* MI, int32_t* block) {
  return guarded("ldw_links_copy", [&]() -> int {
  if (!src) return ldw::set_error(LDW_ERR_ARG, "ldw_links_copy: null table");
  const int64_t n = src->n;
  if (n <= 0) return 0;
  const int32_t* si[6] = {src->pos1, src->pos2, src->clust1, src->clust2, src->len, src->block};
  int32_t* di[6] = {pos1, pos2, clust1, clust2, len, block};
  for (int k = 0; k < 6; k++)
    if (di[k] && !si[k]) return ldw::set_error(LDW_ERR_ARG, "ldw_links_copy: the table has no such column (materialised without host copies?)");
  if (MI && !src->MI) return ldw::set_error(LDW_ERR_ARG, "ldw_links_copy: the table has no MI column");
  const int64_t piece = 1 << 20;
  parallel_dynamic((n + piece - 1) / piece, [&](int64_t c) {
    const int64_t lo = c * piece, m = std::min(n, lo + piece) - lo;
    for (int k = 0; k < 6; k++)
      if (di[k]) memcpy(di[k] + lo, si[k] + lo, sizeof(int32_t) * (size_t)m);
    if (MI) memcpy(MI + lo, src->MI + lo, sizeof(double) * (size_t)m);
  });
  return 0;
  });
}
