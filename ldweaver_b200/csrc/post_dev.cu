// mergeNsort_sr_links (R/computePairwiseMI.R:400-495) on the DEVICE-RESIDENT short-range table of the last scan.
//
// The reference walks all ~10^8 short-range links as R data.frames (group_by(len) + quantile, fitdist, pbeta).  The host
// implementation (post_host.cpp) needs the 2.9 GB of link columns in host memory first; here the table never leaves HBM:
// every pass over the N links is an HBM-bound kernel (or a CUB primitive used for ordering / compaction only), and only
// what is O(groups) or O(links above the fit) crosses PCIe:
//   1. sr_group_count_kernel   membership (0 < len < sr_dist, clusters clust1 / clust2, :372-376, :417-419) + histogram
//                              of the (cluster, length) groups                                       [20 B/link read]
//   2. cub::DeviceScan         group offsets
//   3. sr_group_scatter_kernel MI of every membership into its group's slice                         [+8 B/entry written]
//   4. cub::DeviceSegmentedSort per-group order (library call, ordering step only)
//   5. sr_group_q95_kernel     type-7 95th percentile per group from the sorted slice (:422) -- order statistics, so the
//                              atomics-based scatter order does not matter and the result is bit-identical to the host's
//      host: log-log decay fit per cluster (fastLm, :428-429; shared code, post_host.cpp)
//   6. sr_residual_kernel      d = MI - fit[len], subscripted by the VALUE of len as the reference does (:448); flags of
//                              the links above the fit per cluster, and fixed-order block partials of n, sum log d,
//                              sum log(1-d), sum d, sum d^2
//      host: beta fit from those sufficient statistics (moment start + Nelder-Mead, :452; shared code)
//   7. cub::DeviceSelect::Flagged per cluster: the links above the fit in scan order (the reference's row order)
//   8. sr_srp_kernel           srp_max = -pbeta(d, a, b, lower = F, log = T) in fp64 (continued fraction, :453), and the smallest
//                              MI among the same-cluster links with srp_max > cutoff
//   9. select on the dup flags: row ids, srp_max and the compared columns of the (few) cross-cluster links come to the
//                              host, which keeps them once each (:474-483; shared code)
//  10. sr_keep_kernel + select: row ids and srp_max of ONLY the same-cluster rows sr_links_red (srp_max > cutoff, :494) and
//                              sr_links_ARACNE_check (MI >= min(sr_links_red$MI), :495) need -- a few 10^5 of the 4.5 x 10^6
//                              links above the fit at 616 x 100k
//  11. gather_kernel per column: the link columns of those df rows, by row id, in df order
// The membership filter, the residual lookup and the beta tail are the host implementation's own (sr_stats.cuh).
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>

#include <chrono>
#include <cmath>
#include <memory>
#include <numeric>

#include "../../include/ldw.h"
#include "ctx.h"
#include "post_host.h"
#include "sr_stats.cuh"

using namespace ldw;

namespace {

constexpr int MAXC = 64;  // clusters handled on the device path (cds_var$nclust is 2-3 in practice)

__global__ void sr_group_count_kernel(ldw_links T, double sr_dist, int nclust, int64_t nl, uint32_t* gcount) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < T.n; i += (int64_t)gridDim.x * blockDim.x) {
    int ca, cb, l;
    if (!ldwpost::member(T, i, sr_dist, nclust, ca, cb, l)) continue;
    if (ca) atomicAdd(&gcount[(int64_t)(ca - 1) * nl + l], 1u);
    if (cb) atomicAdd(&gcount[(int64_t)(cb - 1) * nl + l], 1u);
  }
}

__global__ void u32_to_i64_kernel(const uint32_t* in, int64_t n, int64_t* out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = in[i];
}

__global__ void sr_group_scatter_kernel(ldw_links T, double sr_dist, int nclust, int64_t nl, const int64_t* goff, unsigned long long* cursor,
                                        double* keys) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < T.n; i += (int64_t)gridDim.x * blockDim.x) {
    int ca, cb, l;
    if (!ldwpost::member(T, i, sr_dist, nclust, ca, cb, l)) continue;
    const double v = T.MI[i];
    if (ca) { const int64_t g = (int64_t)(ca - 1) * nl + l; keys[goff[g] + (int64_t)atomicAdd(&cursor[g], 1ull)] = v; }
    if (cb) { const int64_t g = (int64_t)(cb - 1) * nl + l; keys[goff[g] + (int64_t)atomicAdd(&cursor[g], 1ull)] = v; }
  }
}

// stats::quantile.default(type = 7), prob 0.95, from an ascending slice (post_host.cpp:quantile7 on unsorted data)
__global__ void sr_group_q95_kernel(const double* sorted, const int64_t* goff, int64_t G, double* gq) {
  int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  const int64_t n = goff[g + 1] - goff[g];
  if (n <= 0) { gq[g] = 0.0; return; }
  const double* x = sorted + goff[g];
  // every product and sum rounded on its own (no FMA contraction): the host evaluates the same expression that way
  const double index = __dadd_rn(1.0, __dmul_rn((double)(n - 1), 0.95));
  const int64_t lo = (int64_t)floor(index), hi = (int64_t)ceil(index);
  double qs = x[lo - 1];
  if (hi > lo) {
    const double xhi = x[lo];  // smallest of the values above position lo
    if (index > (double)lo && xhi != qs) {
      const double h = index - (double)lo;
      qs = __dadd_rn(__dmul_rn(1.0 - h, qs), __dmul_rn(h, xhi));
    }
  }
  gq[g] = qs;
}

struct FitTab {           // fitted decay per cluster as the reference subscripts it: fit[c][len - 1], len <= ng[c]
  const double* val;      // concatenated, cluster c at off[c - 1]
  int64_t off[MAXC + 1];
  int nclust;
};

constexpr int RES_THREADS = 256;
// Each block owns one contiguous piece of the table; its partial sums are reduced in a fixed order (strided per-thread
// accumulation, then a shared-memory tree), so the totals do not depend on scheduling.
__global__ void __launch_bounds__(RES_THREADS) sr_residual_kernel(ldw_links T, double sr_dist, FitTab F, int64_t piece, uint8_t* flags /*[nclust][N]*/,
                                                                  double* part /*[blocks][nclust][5]*/, uint32_t* bad) {
  __shared__ double sh[RES_THREADS];
  const int64_t lo = (int64_t)blockIdx.x * piece, hi = min(T.n, lo + piece);
  for (int c = 1; c <= F.nclust; c++) {
    double acc[5] = {0, 0, 0, 0, 0};
    for (int64_t i = lo + threadIdx.x; i < hi; i += RES_THREADS) {
      int ca, cb, l;
      uint8_t f = 0;
      if (ldwpost::member(T, i, sr_dist, F.nclust, ca, cb, l) && (ca == c || cb == c)) {
        double d;
        if (ldwpost::residual(F.val, F.off, c, l, T.MI[i], d)) {
          f = 1;
          if (d > 1) atomicMax(bad, (uint32_t)c);
          acc[0] += 1.0; acc[1] += log(d); acc[2] += log1p(-d); acc[3] += d; acc[4] += d * d;
        }
      }
      flags[(int64_t)(c - 1) * T.n + i] = f;
    }
    for (int k = 0; k < 5; k++) {
      sh[threadIdx.x] = acc[k];
      __syncthreads();
      for (int o = RES_THREADS / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
      }
      if (threadIdx.x == 0) part[((int64_t)blockIdx.x * F.nclust + (c - 1)) * 5 + k] = sh[0];
      __syncthreads();
    }
  }
}

// order-preserving 64-bit key of a double (for atomicMin on MI values, which may be negative)
__device__ __forceinline__ unsigned long long dbl_key(double v) {
  unsigned long long b = (unsigned long long)__double_as_longlong(v);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

// srp_max of the links above the fit of cluster c (rows[k]); dup[k] = the link joins two clusters (it is listed under both
// and de-duplicated on the host); *min_red_key = smallest MI among the same-cluster links that pass the cut-off.
__global__ void sr_srp_kernel(ldw_links T, FitTab F, int c, double a, double b, double lbeta, double cutoff, const int64_t* rows, int64_t n,
                              double* srp, uint8_t* dup, unsigned long long* min_red_key) {
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t i = rows[k];
  const double mi = T.MI[i];
  const double d = mi - ldwpost::fit_at(F.val, F.off, c, T.len[i]);
  const double v = d < 1.0 ? ldwpost::neg_log_upper_beta(d, a, b, lbeta) : INFINITY;
  srp[k] = v;
  const bool is_dup = T.clust1[i] != T.clust2[i];
  dup[k] = is_dup ? 1 : 0;
  if (!is_dup && v > cutoff) atomicMin(min_red_key, dbl_key(mi));  // NaN compares false: dropped as in :458
}

// which same-cluster rows of the cluster's list travel to the host: those in sr_links_red (srp_max > cutoff) or in
// sr_links_ARACNE_check (MI >= min_mi)
__global__ void sr_keep_kernel(ldw_links T, const int64_t* rows, const double* srp, const uint8_t* dup, int64_t n, double cutoff, double min_mi,
                               uint8_t* keep) {
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const double v = srp[k];
  keep[k] = (!dup[k] && !isnan(v) && (v > cutoff || T.MI[rows[k]] >= min_mi)) ? 1 : 0;
}

template <class T>
__global__ void gather_kernel(const T* src, const int64_t* idx, int64_t n, T* dst) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) dst[t] = src[idx[t]];
}

// dst[t] = src[idx[t]], t < n, elements of el (4 or 8) bytes
void gather(const void* src, size_t el, const int64_t* idx, int64_t n, void* dst, cudaStream_t st) {
  const unsigned nb = (unsigned)((n + 255) / 256);
  if (el == 8) gather_kernel<<<nb, 256, 0, st>>>(static_cast<const uint64_t*>(src), idx, n, static_cast<uint64_t*>(dst));
  else gather_kernel<<<nb, 256, 0, st>>>(static_cast<const uint32_t*>(src), idx, n, static_cast<uint32_t*>(dst));
}

__global__ void max_len_kernel(ldw_links T, double sr_dist, int nclust, int* out) {
  int m = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < T.n; i += (int64_t)gridDim.x * blockDim.x) {
    int ca, cb, l;
    if (ldwpost::member(T, i, sr_dist, nclust, ca, cb, l)) m = max(m, l);
  }
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}

}  // namespace

extern "C" int ldw_sr_postprocess_dev(ldw_ctx* ctx, int32_t nclust, double sr_dist, double srp_cutoff, ldw_sr_post* out, ldw_links* df_rows_out) {
  return ldw::guarded("ldw_sr_postprocess_dev", [&]() -> int {
    if (!ctx || !out) return set_error(LDW_ERR_ARG, "ldw_sr_postprocess_dev: null argument");
    memset(out, 0, sizeof(*out));
    if (df_rows_out) memset(df_rows_out, 0, sizeof(*df_rows_out));
    LDW_TRY(ctx_bind(ctx));
    if (nclust < 1 || nclust > MAXC) return set_error(LDW_ERR_UNSUPPORTED, "ldw_sr_postprocess_dev: nclust must be in 1..%d", MAXC);
    const ldw_links& T = ctx->dev_sr;
    if (T.n < 0) return set_error(LDW_ERR_ARG, "ldw_sr_postprocess_dev: no short-range table on the device (run ldw_mi_scan over the whole job, "
                                                "n_parts = 1, without LDW_SCAN_NO_LINKS / LDW_SCAN_LR_ONLY, first)");
    const int64_t N = T.n;
    if (N > 0x7fffffffLL) return set_error(LDW_ERR_UNSUPPORTED, "ldw_sr_postprocess_dev: more than 2^31 short-range links");
    cudaStream_t st = ctx->stream;
    std::unique_ptr<ldwpost::SrPostPriv> S(new ldwpost::SrPostPriv());
    S->fit_off.assign(1, 0);
    const int nb_stream = ctx->num_sms * 8;
    const bool dbg_t = getenv("LDW_DBG_TIMING") != nullptr;  // phase times on stderr (never stdout)
    auto t_last = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {
      if (!dbg_t) return;
      cudaStreamSynchronize(st);
      const auto t = std::chrono::steady_clock::now();
      fprintf(stderr, "[ldw_sr_postprocess_dev] %-34s %8.2f ms\n", what, std::chrono::duration<double, std::milli>(t - t_last).count());
      t_last = t;
    };

    // ---- groups: (cluster, length) ----
    int32_t maxlen = ldwpost::max_len_bound(sr_dist);
    if (maxlen < 0) {
      maxlen = 0;
      DevBuf d_m;
      LDW_TRY(d_m.alloc(4));
      LDW_CUDA(cudaMemsetAsync(d_m.p, 0, 4, st));
      if (N > 0) max_len_kernel<<<nb_stream, 256, 0, st>>>(T, sr_dist, nclust, d_m.as<int>());
      LDW_CUDA(cudaMemcpyAsync(&maxlen, d_m.p, 4, cudaMemcpyDeviceToHost, st));
      LDW_CUDA(cudaStreamSynchronize(st));
    }
    const int64_t nl = (int64_t)maxlen + 1, G = (int64_t)nclust * nl;
    if (G > ((int64_t)1 << 27)) return set_error(LDW_ERR_UNSUPPORTED, "ldw_sr_postprocess_dev: %lld (cluster, length) groups", (long long)G);
    DevBuf d_gcount, d_gcnt64, d_goff, d_cursor, d_gq;
    LDW_TRY(d_gcount.alloc((size_t)G * 4));
    LDW_TRY(d_gcnt64.alloc((size_t)(G + 1) * 8));
    LDW_TRY(d_goff.alloc((size_t)(G + 1) * 8));
    LDW_TRY(d_cursor.alloc((size_t)G * 8));
    LDW_TRY(d_gq.alloc((size_t)G * 8));
    LDW_CUDA(cudaMemsetAsync(d_gcount.p, 0, (size_t)G * 4, st));
    LDW_CUDA(cudaMemsetAsync(d_cursor.p, 0, (size_t)G * 8, st));
    LDW_CUDA(cudaMemsetAsync(d_gcnt64.p, 0, (size_t)(G + 1) * 8, st));
    if (N > 0) sr_group_count_kernel<<<nb_stream, 256, 0, st>>>(T, sr_dist, nclust, nl, d_gcount.as<uint32_t>());
    u32_to_i64_kernel<<<(unsigned)((G + 255) / 256), 256, 0, st>>>(d_gcount.as<uint32_t>(), G, d_gcnt64.as<int64_t>());
    LDW_CUDA(cudaGetLastError());
    {
      size_t tb = 0;
      cub::DeviceScan::ExclusiveSum(nullptr, tb, d_gcnt64.as<int64_t>(), d_goff.as<int64_t>(), (int)(G + 1), st);
      DevBuf tmp;
      LDW_TRY(tmp.alloc(tb));
      LDW_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tb, d_gcnt64.as<int64_t>(), d_goff.as<int64_t>(), (int)(G + 1), st));
      LDW_CUDA(cudaStreamSynchronize(st));
    }
    std::vector<int64_t> goff((size_t)G + 1);
    LDW_CUDA(cudaMemcpyAsync(goff.data(), d_goff.p, (size_t)(G + 1) * 8, cudaMemcpyDeviceToHost, st));
    LDW_CUDA(cudaStreamSynchronize(st));
    const int64_t E = goff[G];
    lap("group histogram + offsets");
    LDW_TRY(ldwpost::check_groups(goff, nclust, nl));
    // ---- per-group 95th percentiles ----
    std::vector<double> gq_all((size_t)G);
    {
      DevBuf d_keys, d_sorted, tmp;
      LDW_TRY(d_keys.alloc((size_t)std::max<int64_t>(E, 1) * 8));
      LDW_TRY(d_sorted.alloc((size_t)std::max<int64_t>(E, 1) * 8));
      sr_group_scatter_kernel<<<nb_stream, 256, 0, st>>>(T, sr_dist, nclust, nl, d_goff.as<int64_t>(), d_cursor.as<unsigned long long>(), d_keys.as<double>());
      LDW_CUDA(cudaGetLastError());
      if (E > 0x7fffffffLL) return set_error(LDW_ERR_UNSUPPORTED, "ldw_sr_postprocess_dev: more than 2^31 (link, cluster) entries");
      size_t tb = 0;
      cub::DeviceSegmentedSort::SortKeys(nullptr, tb, d_keys.as<double>(), d_sorted.as<double>(), (int)E, (int)G, d_goff.as<int64_t>(),
                                         d_goff.as<int64_t>() + 1, st);
      LDW_TRY(tmp.alloc(tb));
      LDW_CUDA(cub::DeviceSegmentedSort::SortKeys(tmp.p, tb, d_keys.as<double>(), d_sorted.as<double>(), (int)E, (int)G,
                                                  d_goff.as<int64_t>(), d_goff.as<int64_t>() + 1, st));
      lap("scatter + segmented sort");
      sr_group_q95_kernel<<<(unsigned)((G + 255) / 256), 256, 0, st>>>(d_sorted.as<double>(), d_goff.as<int64_t>(), G, d_gq.as<double>());
      LDW_CUDA(cudaGetLastError());
      LDW_CUDA(cudaMemcpyAsync(gq_all.data(), d_gq.p, (size_t)G * 8, cudaMemcpyDeviceToHost, st));
      LDW_CUDA(cudaStreamSynchronize(st));
    }
    std::vector<int64_t> glist;
    std::vector<double> gq;
    for (int64_t g = 0; g < G; g++)
      if (goff[g + 1] > goff[g]) { glist.push_back(g); gq.push_back(gq_all[g]); }
    lap("percentiles to host");
    // ---- decay fits (host) ----
    LDW_TRY(ldwpost::decay_fits(*S, nclust, nl, glist, gq));
    lap("decay fits (host)");
    // ---- residuals: flags + sufficient statistics ----
    FitTab F;
    memset(&F, 0, sizeof(F));
    F.nclust = nclust;
    DevBuf d_fit;
    LDW_TRY(d_fit.alloc(std::max<size_t>(S->fit_val.size(), 1) * 8));
    LDW_CUDA(cudaMemcpyAsync(d_fit.p, S->fit_val.data(), S->fit_val.size() * 8, cudaMemcpyHostToDevice, st));
    F.val = d_fit.as<double>();
    for (int c = 0; c <= nclust; c++) F.off[c] = S->fit_off[c];
    const int64_t piece = 1 << 16;  // fixed piece size: the partial sums, hence the fit, do not depend on the device
    const int64_t nblocks = std::max<int64_t>(1, (N + piece - 1) / piece);
    DevBuf d_flags, d_part, d_bad;
    LDW_TRY(d_flags.alloc((size_t)nclust * (size_t)std::max<int64_t>(N, 1)));
    LDW_TRY(d_part.alloc((size_t)nblocks * nclust * 5 * 8));
    LDW_TRY(d_bad.alloc(4));
    LDW_CUDA(cudaMemsetAsync(d_bad.p, 0, 4, st));
    sr_residual_kernel<<<(unsigned)nblocks, RES_THREADS, 0, st>>>(T, sr_dist, F, piece, d_flags.as<uint8_t>(), d_part.as<double>(), d_bad.as<uint32_t>());
    LDW_CUDA(cudaGetLastError());
    std::vector<double> part((size_t)nblocks * nclust * 5);
    uint32_t bad = 0;
    LDW_CUDA(cudaMemcpyAsync(part.data(), d_part.p, part.size() * 8, cudaMemcpyDeviceToHost, st));
    LDW_CUDA(cudaMemcpyAsync(&bad, d_bad.p, 4, cudaMemcpyDeviceToHost, st));
    LDW_CUDA(cudaStreamSynchronize(st));
    LDW_TRY(ldwpost::check_residuals((int)bad));
    lap("residual flags + sums");

    // Per cluster: the links above the fit in scan order, their srp_max, the smallest MI of those that pass the cut-off.
    struct PerC { DevBuf rows, srp, dup; int64_t npos = 0; };
    std::vector<PerC> pc((size_t)nclust + 1);
    DevBuf d_tmp, d_nsel, d_minkey, d_keep, d_pick, d_row, d_col;
    LDW_TRY(d_nsel.alloc(8));
    LDW_TRY(d_minkey.alloc(8));
    LDW_CUDA(cudaMemsetAsync(d_minkey.p, 0xFF, 8, st));
    // out[0 .. m) = the positions of the set flags among n, in order
    auto select_flagged = [&](const uint8_t* flags, int64_t n, int64_t* out, int64_t& m) -> int {
      thrust::counting_iterator<int64_t> it(0);
      size_t tb = 0;
      cub::DeviceSelect::Flagged(nullptr, tb, it, flags, out, d_nsel.as<int64_t>(), (int)n, st);
      LDW_TRY(d_tmp.ensure(tb));
      LDW_CUDA(cub::DeviceSelect::Flagged(d_tmp.p, tb, it, flags, out, d_nsel.as<int64_t>(), (int)n, st));
      LDW_CUDA(cudaMemcpyAsync(&m, d_nsel.p, 8, cudaMemcpyDeviceToHost, st));
      LDW_CUDA(cudaStreamSynchronize(st));
      return 0;
    };
    for (int32_t c = 1; c <= nclust; c++) {
      long double cnt = 0, s1 = 0, s2 = 0, sm = 0, sq = 0;
      for (int64_t k = 0; k < nblocks; k++) {
        const double* p = &part[((size_t)k * nclust + (c - 1)) * 5];
        cnt += p[0]; s1 += p[1]; s2 += p[2]; sm += p[3]; sq += p[4];
      }
      const int64_t npos = (int64_t)llroundl(cnt);
      LDW_TRY(ldwpost::check_npos(c, npos));
      const double mean = (double)(sm / (long double)npos);
      const double v = (double)((sq - (long double)npos * (long double)mean * (long double)mean) / (long double)npos);  // biased variance
      double par[2];
      LDW_TRY(ldwpost::beta_fit(*S, c, npos, (double)s1, (double)s2, mean, v, par));
      const double lbeta = ldwpost::lbeta_fn(par[0], par[1]);
      PerC& P = pc[c];
      P.npos = npos;
      LDW_TRY(P.rows.alloc((size_t)npos * 8));
      LDW_TRY(P.srp.alloc((size_t)npos * 8));
      LDW_TRY(P.dup.alloc((size_t)npos));
      int64_t nsel = 0;
      LDW_TRY(select_flagged(d_flags.as<uint8_t>() + (size_t)(c - 1) * N, N, P.rows.as<int64_t>(), nsel));
      if (nsel != npos) return set_error(LDW_ERR_INTERNAL, "ldw_sr_postprocess_dev: %lld flagged links but %lld counted", (long long)nsel, (long long)npos);
      sr_srp_kernel<<<(unsigned)((npos + 127) / 128), 128, 0, st>>>(T, F, c, par[0], par[1], lbeta, srp_cutoff, P.rows.as<int64_t>(), npos,
                                                                   P.srp.as<double>(), P.dup.as<uint8_t>(), d_minkey.as<unsigned long long>());
      LDW_CUDA(cudaGetLastError());
    }
    lap("select + srp_max (all clusters)");
    // Only what sr_links_red / sr_links_ARACNE_check need comes to the host (sr_links_df itself -- every link above the fit,
    // 4.5e6 rows at 616 x 100k -- stays on the device): first the cross-cluster links, whose de-duplication decides which of
    // them are in sr_links_red and therefore min(sr_links_red$MI); then the same-cluster rows of the two sets.
    // pick: rows and srp_max of the entries of cluster c's list whose flag is set, in scan order.
    auto pick = [&](int32_t c, const uint8_t* flags, std::vector<int64_t>& row, std::vector<double>& srp) -> int {
      PerC& P = pc[c];
      int64_t m = 0;
      LDW_TRY(d_pick.ensure((size_t)P.npos * 8));
      LDW_TRY(select_flagged(flags, P.npos, d_pick.as<int64_t>(), m));
      row.resize((size_t)m);
      srp.resize((size_t)m);
      if (m == 0) return 0;
      LDW_TRY(d_row.ensure((size_t)m * 8));
      LDW_TRY(d_col.ensure((size_t)m * 8));
      gather(P.rows.p, 8, d_pick.as<int64_t>(), m, d_row.p, st);
      gather(P.srp.p, 8, d_pick.as<int64_t>(), m, d_col.p, st);
      LDW_CUDA(cudaGetLastError());
      LDW_CUDA(cudaMemcpyAsync(row.data(), d_row.p, (size_t)m * 8, cudaMemcpyDeviceToHost, st));
      LDW_CUDA(cudaMemcpyAsync(srp.data(), d_col.p, (size_t)m * 8, cudaMemcpyDeviceToHost, st));
      LDW_CUDA(cudaStreamSynchronize(st));
      return 0;
    };
    // fetch: the link columns of table rows `row` into o, in that order (all, or only those the de-duplication compares).
    auto fetch = [&](const std::vector<int64_t>& row, ldwpost::HostCols& o, bool all) -> int {
      const int64_t m = (int64_t)row.size();
      LDW_TRY(o.ensure(m));
      o.n = m;
      if (m == 0) return 0;
      LDW_TRY(d_row.ensure((size_t)m * 8));
      LDW_TRY(d_col.ensure((size_t)m * 8));
      LDW_CUDA(cudaMemcpyAsync(d_row.p, row.data(), (size_t)m * 8, cudaMemcpyHostToDevice, st));
      for (int k = 0; k < ldwpost::HostCols::NCOL; k++) {
        if (!all && &o.col(k) == &o.blk) continue;
        const size_t el = ldwpost::HostCols::elem(k);
        gather(ldwpost::HostCols::abi_col(T, k), el, d_row.as<int64_t>(), m, d_col.p, st);
        LDW_CUDA(cudaGetLastError());
        LDW_CUDA(cudaMemcpyAsync(o.col(k).p.get(), d_col.p, (size_t)m * el, cudaMemcpyDeviceToHost, st));
      }
      LDW_CUDA(cudaStreamSynchronize(st));
      return 0;
    };
    // ---- phase 0: cross-cluster links -> de-duplicated (:474-483) ----
    std::vector<int64_t> dup_row;
    std::vector<int32_t> dup_c;
    std::vector<double> dup_srp;
    for (int32_t c = 1; c <= nclust; c++) {
      std::vector<int64_t> row;
      std::vector<double> srp;
      LDW_TRY(pick(c, pc[c].dup.as<uint8_t>(), row, srp));
      for (size_t t = 0; t < row.size(); t++) {
        if (std::isnan(srp[t])) continue;  // :458
        dup_row.push_back(row[t]); dup_c.push_back(c); dup_srp.push_back(srp[t]);
      }
    }
    ldwpost::HostCols dup_cols;
    LDW_TRY(fetch(dup_row, dup_cols, false));
    ldw_links dup_tab;
    dup_cols.fill(&dup_tab);
    std::vector<int64_t> dup_at(dup_row.size());
    std::iota(dup_at.begin(), dup_at.end(), 0);
    const std::vector<int64_t> win = ldwpost::dedup(dup_tab, dup_at, dup_srp);
    unsigned long long minkey = ~0ull;
    LDW_CUDA(cudaMemcpyAsync(&minkey, d_minkey.p, 8, cudaMemcpyDeviceToHost, st));
    LDW_CUDA(cudaStreamSynchronize(st));
    double min_mi = INFINITY;  // min(sr_links_red$MI), :495
    if (minkey != ~0ull) {
      const unsigned long long bts = (minkey >> 63) ? (minkey & 0x7FFFFFFFFFFFFFFFull) : ~minkey;
      memcpy(&min_mi, &bts, 8);
    }
    for (int64_t k : win)
      if (dup_srp[k] > srp_cutoff) min_mi = std::min(min_mi, dup_tab.MI[k]);
    lap("cross-cluster links + min MI");
    // ---- phase 1: same-cluster rows of sr_links_red / sr_links_ARACNE_check, cluster by cluster in scan order ----
    for (int32_t c = 1; c <= nclust; c++) {
      PerC& P = pc[c];
      LDW_TRY(d_keep.ensure((size_t)P.npos));
      sr_keep_kernel<<<(unsigned)((P.npos + 255) / 256), 256, 0, st>>>(T, P.rows.as<int64_t>(), P.srp.as<double>(), P.dup.as<uint8_t>(), P.npos,
                                                                       srp_cutoff, min_mi, d_keep.as<uint8_t>());
      LDW_CUDA(cudaGetLastError());
      std::vector<int64_t> row;
      std::vector<double> srp;
      LDW_TRY(pick(c, d_keep.as<uint8_t>(), row, srp));
      S->row.insert(S->row.end(), row.begin(), row.end());
      S->clust_c.insert(S->clust_c.end(), row.size(), c);
      S->srp.insert(S->srp.end(), srp.begin(), srp.end());
    }
    for (int64_t k : win) {  // the de-duplicated cross-cluster links follow (:483), those in either set
      if (!(dup_srp[k] > srp_cutoff || dup_tab.MI[k] >= min_mi)) continue;
      S->row.push_back(dup_row[k]); S->clust_c.push_back(dup_c[k]); S->srp.push_back(dup_srp[k]);
    }
    LDW_TRY(fetch(S->row, S->df, true));
    lap("rows of red / check sets");
    const int64_t ndf = (int64_t)S->row.size();
    const double* df_mi = S->df.mi.as<double>();
    for (int64_t i = 0; i < ndf; i++) {
      if (S->srp[(size_t)i] > srp_cutoff) S->red.push_back(i);
      if (df_mi[i] >= min_mi) S->chk.push_back(i);
    }
    lap("red / chk + reorder (host)");
    ldwpost::publish(*S, nclust, out);
    S->df.fill(df_rows_out);
    out->priv = S.release();
    return 0;
  });
}
