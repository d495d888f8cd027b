// Device groups: the multi-GPU form of the hot path (SURVEY.md section 8e), behind the same C ABI.
//
// Reference loop being replaced: the serial `for each block` of perform_MI_computation (R/computePairwiseMI.R:103-116)
// and the five crossprods of estimate_Hamming_distance_weights (R/performPopulationStuctureCorrection.R:49-76) -- the
// reference has no multi-device code; its blocks are independent, which is what makes the split exact.
//
// One member = one device = one ldw_ctx + one NCCL communicator.  A group either holds ALL ranks of the job in this
// process (ldw_group_create: the form R and Python use; ncclCommInitAll, one host thread per device while an operation
// runs) or ONE rank of a multi-process job (ldw_group_create_rank: the torchrun form bench.py is launched in;
// ncclCommInitRank with an id made by rank 0).  Every operation is collective over the whole job.
//
//   ldw_group_load_codes  rank 0 uploads the class matrix once, ncclBroadcast puts it on every device (row e3)
//   ldw_group_hdw         upper-triangle tiles of the distance GEMM dealt across ranks, ncclAllReduce of the partial
//                         neighbour counts, every rank forms hdw (row e2: doubles as the weight broadcast)
//   ldw_group_mi_scan     each rank packs its operands from the resident matrix and scans its cost-dealt share of the
//                         make_blocks blocks; short-range rows are copied by every device straight to their final
//                         rows of ONE pinned host table (each GPU over its own PCIe link, no merge pass), long-range
//                         and borderline rows are merged into make_blocks order on the host (row e1)
// No collective sits on the scan's data path.
#include <dlfcn.h>
#include <nccl.h>  // types and enums only: the library is bound at run time (see nccl_api below)

#include <chrono>
#include <cmath>
#include <mutex>
#include <string>
#include <thread>

#include "../../include/ldw.h"
#include "ctx.h"
#include "hdw.h"
#include "mi_scan.h"

using namespace ldw;

struct ldw_group {
  struct Member {
    ldw_ctx* ctx = nullptr;
    ncclComm_t comm = nullptr;
    int rank = 0;
    DevBuf d_codes;
    Member() {}
    Member(Member&& o) noexcept : ctx(o.ctx), comm(o.comm), rank(o.rank) {
      d_codes.p = o.d_codes.p; d_codes.bytes = o.d_codes.bytes;
      o.d_codes.p = nullptr; o.d_codes.bytes = 0; o.ctx = nullptr; o.comm = nullptr;
    }
  };
  int world = 1;
  std::vector<Member> m;
  int64_t n_snp = 0, nseq = 0;  // the resident class matrix
  HostLinks h_sr, h_lr, h_border;
};

namespace {

// NCCL is bound at run time, on first use by a group of more than one device: libldwgpu.so itself has no link-time
// dependency on it, so single-GPU users need no NCCL at all and a host process that brings its own libnccl.so.2 (an R
// session with none, a Python process where torch has already loaded its bundled, newer one) keeps exactly one copy --
// dlopen returns the copy that is already loaded under that soname.  LDW_NCCL_LIB names another file.
struct NcclApi {
  decltype(&::ncclGetErrorString) GetErrorString = nullptr;
  decltype(&::ncclGetUniqueId) GetUniqueId = nullptr;
  decltype(&::ncclCommInitAll) CommInitAll = nullptr;
  decltype(&::ncclCommInitRank) CommInitRank = nullptr;
  decltype(&::ncclCommDestroy) CommDestroy = nullptr;
  decltype(&::ncclBroadcast) Broadcast = nullptr;
  decltype(&::ncclAllReduce) AllReduce = nullptr;
};

int nccl_api(const NcclApi** out) {
  static NcclApi api;
  static int state = 0;  // 0 not tried, 1 ok, -1 failed
  static std::string why;
  static std::mutex mu;
  std::lock_guard<std::mutex> lk(mu);
  if (state == 0) {
    const char* names[] = {getenv("LDW_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    void* h = nullptr;
    for (const char* nm : names) {
      if (!nm || !*nm) continue;
      h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
      if (h) break;
      why = dlerror();
    }
    if (h) {
      bool ok = true;
      auto sym = [&](const char* nm) { void* p = dlsym(h, nm); if (!p) { ok = false; why = std::string("missing symbol ") + nm; } return p; };
      api.GetErrorString = (decltype(api.GetErrorString))sym("ncclGetErrorString");
      api.GetUniqueId = (decltype(api.GetUniqueId))sym("ncclGetUniqueId");
      api.CommInitAll = (decltype(api.CommInitAll))sym("ncclCommInitAll");
      api.CommInitRank = (decltype(api.CommInitRank))sym("ncclCommInitRank");
      api.CommDestroy = (decltype(api.CommDestroy))sym("ncclCommDestroy");
      api.Broadcast = (decltype(api.Broadcast))sym("ncclBroadcast");
      api.AllReduce = (decltype(api.AllReduce))sym("ncclAllReduce");
      state = ok ? 1 : -1;
    } else {
      state = -1;
    }
  }
  if (state != 1) return set_error(LDW_ERR_UNSUPPORTED, "multi-GPU groups need NCCL (libnccl.so.2): %s", why.c_str());
  *out = &api;
  return 0;
}

#define LDW_NCCL(call)                                                                                               \
  do {                                                                                                               \
    ncclResult_t r__ = (call);                                                                                       \
    if (r__ != ncclSuccess)                                                                                          \
      return ldw::set_error(LDW_ERR_CUDA, "%s failed: %s (%s:%d)", #call, nccl->GetErrorString(r__), __FILE__, __LINE__); \
  } while (0)

// fn(k) for every local member on its own host thread, bound to the member's device.  The first failure's code and
// message (thread-local in the library) are re-raised on the calling thread.
template <class F>
int for_members(ldw_group* G, F fn) {
  const int n = (int)G->m.size();
  std::vector<int> rc(n, 0);
  std::vector<std::string> msg(n);
  auto body = [&](int k) {
    rc[k] = ldw::guarded("ldw_group", [&]() -> int {
      LDW_TRY(ctx_bind(G->m[k].ctx));
      return fn(k);
    });
    if (rc[k] != 0) msg[k] = last_error_ref();
  };
  if (n == 1) {
    body(0);
  } else {
    std::vector<std::thread> th;
    for (int k = 0; k < n; k++) th.emplace_back(body, k);
    for (auto& t : th) t.join();
  }
  for (int k = 0; k < n; k++)
    if (rc[k] != 0) return set_error(rc[k], "device %d (rank %d): %s", G->m[k].ctx->device, G->m[k].rank, msg[k].c_str());
  return 0;
}

void free_members(ldw_group* G) {
  for (auto& mb : G->m) {
    if (mb.ctx) cudaSetDevice(mb.ctx->device);
    mb.d_codes.release();
    if (mb.comm) {
      const NcclApi* nccl = nullptr;
      if (nccl_api(&nccl) == 0) nccl->CommDestroy(mb.comm);
    }
    if (mb.ctx) ldw_destroy(mb.ctx);
  }
  G->m.clear();
}

}  // namespace

extern "C" {

int ldw_group_create(const int* devices, int n_devices, ldw_group** out) {
  return ldw::guarded("ldw_group_create", [&]() -> int {
    if (!out) return set_error(LDW_ERR_ARG, "ldw_group_create: null out");
    *out = nullptr;
    if (!devices || n_devices < 1) return set_error(LDW_ERR_ARG, "ldw_group_create: need at least one device");
    for (int a = 0; a < n_devices; a++)
      for (int b = a + 1; b < n_devices; b++)
        if (devices[a] == devices[b]) return set_error(LDW_ERR_ARG, "ldw_group_create: device %d listed twice", devices[a]);
    ldw_group* G = new ldw_group();
    G->world = n_devices;
    G->m.resize(n_devices);
    for (int k = 0; k < n_devices; k++) {
      G->m[k].rank = k;
      int rc = ldw_create(devices[k], &G->m[k].ctx);
      if (rc != 0) { free_members(G); delete G; return rc; }
    }
    if (n_devices > 1) {
      const NcclApi* nccl = nullptr;
      if (int e = nccl_api(&nccl)) { free_members(G); delete G; return e; }
      std::vector<ncclComm_t> comms(n_devices);
      ncclResult_t r = nccl->CommInitAll(comms.data(), n_devices, devices);
      if (r != ncclSuccess) {
        free_members(G);
        delete G;
        return set_error(LDW_ERR_CUDA, "ncclCommInitAll over %d devices failed: %s", n_devices, nccl->GetErrorString(r));
      }
      for (int k = 0; k < n_devices; k++) G->m[k].comm = comms[k];
    }
    *out = G;
    return 0;
  });
}

int ldw_group_unique_id(char* id_out) {
  if (!id_out) return set_error(LDW_ERR_ARG, "ldw_group_unique_id: null argument");
  static_assert(sizeof(ncclUniqueId) == LDW_GROUP_ID_BYTES, "ncclUniqueId size");
  const NcclApi* nccl = nullptr;
  LDW_TRY(nccl_api(&nccl));
  ncclUniqueId id;
  LDW_NCCL(nccl->GetUniqueId(&id));
  memcpy(id_out, &id, sizeof(id));
  return 0;
}

int ldw_group_create_rank(int device, int rank, int world, const char* id_bytes, ldw_group** out) {
  return ldw::guarded("ldw_group_create_rank", [&]() -> int {
    if (!out) return set_error(LDW_ERR_ARG, "ldw_group_create_rank: null out");
    *out = nullptr;
    if (world < 1 || rank < 0 || rank >= world) return set_error(LDW_ERR_ARG, "ldw_group_create_rank: bad rank %d of %d", rank, world);
    if (world > 1 && !id_bytes) return set_error(LDW_ERR_ARG, "ldw_group_create_rank: null id");
    ldw_group* G = new ldw_group();
    G->world = world;
    G->m.resize(1);
    G->m[0].rank = rank;
    int rc = ldw_create(device, &G->m[0].ctx);
    if (rc != 0) { delete G; return rc; }
    if (world > 1) {
      const NcclApi* nccl = nullptr;
      if (int e = nccl_api(&nccl)) { free_members(G); delete G; return e; }
      ncclUniqueId id;
      memcpy(&id, id_bytes, sizeof(id));
      cudaSetDevice(device);
      ncclResult_t r = nccl->CommInitRank(&G->m[0].comm, world, id, rank);
      if (r != ncclSuccess) {
        free_members(G);
        delete G;
        return set_error(LDW_ERR_CUDA, "ncclCommInitRank(rank %d of %d) failed: %s", rank, world, nccl->GetErrorString(r));
      }
    }
    *out = G;
    return 0;
  });
}

void ldw_group_destroy(ldw_group* G) {
  if (!G) return;
  free_members(G);
  delete G;
}

int ldw_group_info(const ldw_group* G, int* world_out, int* n_local_out, int* first_rank_out) {
  if (!G) return set_error(LDW_ERR_ARG, "null group");
  if (world_out) *world_out = G->world;
  if (n_local_out) *n_local_out = (int)G->m.size();
  if (first_rank_out) *first_rank_out = G->m.empty() ? 0 : G->m[0].rank;
  return 0;
}

ldw_ctx* ldw_group_ctx(ldw_group* G, int local_index) {
  if (!G || local_index < 0 || local_index >= (int)G->m.size()) return nullptr;
  return G->m[local_index].ctx;
}

int ldw_group_load_codes(ldw_group* G, const uint8_t* codes, int64_t n_snp, int64_t nseq) {
  if (!G) return set_error(LDW_ERR_ARG, "null group");
  if (n_snp <= 0 || nseq <= 0) return set_error(LDW_ERR_ARG, "ldw_group_load_codes: empty matrix");
  bool have_root = false;
  for (auto& mb : G->m) have_root |= (mb.rank == 0);
  if (have_root && !codes) return set_error(LDW_ERR_ARG, "ldw_group_load_codes: the process that holds rank 0 must pass the matrix");
  G->n_snp = n_snp;
  G->nseq = nseq;
  const size_t bytes = (size_t)n_snp * (size_t)nseq;
  const NcclApi* nccl = nullptr;
  if (G->world > 1) LDW_TRY(nccl_api(&nccl));
  int bad_code = 0;
  int rc_all = for_members(G, [&](int k) -> int {
    ldw_group::Member& mb = G->m[k];
    cudaStream_t st = mb.ctx->stream;
    LDW_TRY(mb.d_codes.ensure(bytes));
    if (mb.rank == 0) {
      LDW_CUDA(cudaMemcpyAsync(mb.d_codes.p, codes, bytes, cudaMemcpyHostToDevice, st));
      // every class must be 0..4 (as ldw_mi_plan_create checks on the host): one pass at HBM speed on the device
      uint32_t mx = 0;
      LDW_TRY(max_byte_device(st, mb.d_codes.as<uint8_t>(), (int64_t)bytes, &mx));
      if (mx > 4) bad_code = (int)mx;  // reported after the collective below, so that no rank is left waiting in it
    }
    if (G->world > 1) LDW_NCCL(nccl->Broadcast(mb.d_codes.p, mb.d_codes.p, bytes, ncclUint8, 0, mb.comm, st));
    LDW_CUDA(cudaStreamSynchronize(st));
    return 0;
  });
  if (rc_all != 0) return rc_all;
  if (bad_code) {
    G->n_snp = G->nseq = 0;
    return set_error(LDW_ERR_ARG, "ldw_group_load_codes: the matrix holds a class %d outside 0..4", bad_code);
  }
  return 0;
}

int ldw_group_hdw(ldw_group* G, double threshold, int flags, int32_t* cnt_out, double* hdw_out, int* sharded_out) {
  if (!G) return set_error(LDW_ERR_ARG, "null group");
  if (!hdw_out) return set_error(LDW_ERR_ARG, "ldw_group_hdw: null argument");
  if (G->n_snp <= 0) return set_error(LDW_ERR_ARG, "ldw_group_hdw: call ldw_group_load_codes first");
  const int64_t n = G->n_snp, S = G->nseq;
  if (S > 0x7fffffffLL / 4) return set_error(LDW_ERR_UNSUPPORTED, "ldw_group_hdw: too many sequences");
  const int thresh = (int)((double)n * threshold);  // as.integer(nsnp*threshold): truncation (:23)
  std::vector<int> sharded(G->m.size(), 0);
  const NcclApi* nccl = nullptr;
  if (G->world > 1) LDW_TRY(nccl_api(&nccl));
  int rc = for_members(G, [&](int k) -> int {
    ldw_group::Member& mb = G->m[k];
    cudaStream_t st = mb.ctx->stream;
    DevBuf d_neigh, d_w;
    LDW_TRY(d_neigh.alloc((size_t)S * 4));
    LDW_TRY(d_w.alloc((size_t)S * 8));
    HdwShard sh;
    sh.n_parts = G->world;
    sh.part = mb.rank;
    sh.force = (flags & LDW_HDW_FORCE_SHARD) != 0;
    sh.sharded_out = &sharded[k];
    sh.allreduce = [&mb, nccl](int32_t* d, int64_t cnt, cudaStream_t s) -> int {
      LDW_NCCL(nccl->AllReduce(d, d, (size_t)cnt, ncclInt32, ncclSum, mb.comm, s));
      return 0;
    };
    LDW_TRY(hdw_device(st, mb.d_codes.as<uint8_t>(), n, S, thresh, d_neigh.as<int32_t>(), d_w.as<double>(), nullptr,
                       mb.ctx->num_sms, G->world > 1 ? &sh : nullptr));
    if (k == 0) {  // every rank holds the same counts and weights after the reduction
      if (cnt_out) LDW_CUDA(cudaMemcpyAsync(cnt_out, d_neigh.p, (size_t)S * 4, cudaMemcpyDeviceToHost, st));
      LDW_CUDA(cudaMemcpyAsync(hdw_out, d_w.p, (size_t)S * 8, cudaMemcpyDeviceToHost, st));
      LDW_CUDA(cudaStreamSynchronize(st));
    }
    return 0;
  });
  if (rc == 0 && sharded_out) *sharded_out = sharded[0];
  return rc;
}

int ldw_group_mi_scan(ldw_group* G, const double* hdw, const int32_t* pos, const int32_t* paint, int64_t blk, double g,
                      double sr_dist, double lr_retain_links, double lr_links_approx, int flags, ldw_links* sr_out,
                      ldw_links* lr_out, ldw_links* borderline_out, double* thr_out, double* prob_out,
                      ldw_scan_stats* stats_out, double* t_plan_ms_out) {
  if (!G) return set_error(LDW_ERR_ARG, "null group");
  if (G->n_snp <= 0) return set_error(LDW_ERR_ARG, "ldw_group_mi_scan: call ldw_group_load_codes first");
  if (!hdw || !pos || !paint) return set_error(LDW_ERR_ARG, "ldw_group_mi_scan: null argument");
  return ldw::guarded("ldw_group_mi_scan", [&]() -> int {
    const int nl = (int)G->m.size();
    // ---- every member packs its operands from the resident matrix (no host -> device copy of the matrix here)
    std::vector<ldw_mi_plan*> plans(nl, nullptr);
    auto destroy_plans = [&]() {
      for (int k = 0; k < nl; k++)
        if (plans[k]) { ldw_mi_plan_destroy(plans[k]); plans[k] = nullptr; }
    };
    const auto tp0 = std::chrono::steady_clock::now();
    int rc = for_members(G, [&](int k) -> int {
      return mi_plan_create_impl(G->m[k].ctx, nullptr, G->m[k].d_codes.as<uint8_t>(), G->n_snp, G->nseq, hdw, pos, paint, blk, &plans[k]);
    });
    if (rc != 0) { destroy_plans(); return rc; }
    if (t_plan_ms_out) *t_plan_ms_out = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tp0).count();
    if (nl == 1) {  // one local member (a single device, or one rank of a multi-process job): exactly ldw_mi_scan over this rank's
                    // share -- its own sizing pass over its own blocks, its own tables, nothing to merge
      ldw_scan_stats st1;
      rc = mi_scan_impl(plans[0], g, sr_dist, lr_retain_links, lr_links_approx, flags, G->world, G->m[0].rank, nullptr, sr_out, lr_out,
                        borderline_out, thr_out, prob_out, &st1);
      if (rc != 0) { std::string keep = last_error_ref(); destroy_plans(); return set_error(rc, "%s", keep.c_str()); }
      destroy_plans();
      if (stats_out) stats_out[0] = st1;
      return 0;
    }
    // ---- one layout for the job's short-range table: block sizes once, rows of the blocks this process scans
    ScanShared sh;
    rc = mi_block_sizes(plans[0], g, sr_dist, flags, sh.sizes);
    if (rc != 0) { destroy_plans(); return rc; }
    const int64_t nblk = mi_plan_nblocks(plans[0]);
    std::vector<int> owner;
    mi_block_owners(plans[0], G->world, owner);
    std::vector<char> local_rank(G->world, 0);
    for (auto& mb : G->m) local_rank[mb.rank] = 1;
    sh.sr_hbase.assign(nblk, 0);
    int64_t total_sr = 0;
    for (int64_t b = 0; b < nblk; b++) {
      sh.sr_hbase[b] = total_sr;
      if (local_rank[owner[b]] && sh.sizes[b].err == 0) total_sr += sh.sizes[b].n_sr;
    }
    sh.total_sr = total_sr;
    sh.h_sr = &G->h_sr;
    const bool want_host = !(flags & (LDW_SCAN_NO_LINKS | LDW_SCAN_NO_D2H));
    G->h_sr.n = 0; G->h_lr.n = 0; G->h_border.n = 0;
    const bool sr_rows = !(flags & (LDW_SCAN_NO_LINKS | LDW_SCAN_LR_ONLY));
    if (!sr_rows) total_sr = 0;
    if (want_host) {
      rc = G->h_sr.ensure(total_sr);
      if (rc != 0) { destroy_plans(); return rc; }
    }
    // ---- scan: one host thread per local device
    std::vector<ldw_links> lr(nl), bd(nl), srn(nl);
    std::vector<std::vector<double>> thr(nl, std::vector<double>(nblk, NAN)), prob(nl, std::vector<double>(nblk, NAN));
    std::vector<ldw_scan_stats> stats(nl);
    rc = for_members(G, [&](int k) -> int {
      return mi_scan_impl(plans[k], g, sr_dist, lr_retain_links, lr_links_approx, flags, G->world, G->m[k].rank, &sh, &srn[k],
                          &lr[k], &bd[k], thr[k].data(), prob[k].data(), &stats[k]);
    });
    destroy_plans();
    if (rc != 0) return rc;
    // ---- merge
    if (thr_out) for (int64_t b = 0; b < nblk; b++) thr_out[b] = NAN;
    if (prob_out) for (int64_t b = 0; b < nblk; b++) prob_out[b] = NAN;
    for (int k = 0; k < nl; k++)
      for (int64_t b = 0; b < nblk; b++)
        if (owner[b] == G->m[k].rank) {
          if (thr_out) thr_out[b] = thr[k][b];
          if (prob_out) prob_out[b] = prob[k][b];
        }
    if (stats_out) for (int k = 0; k < nl; k++) stats_out[k] = stats[k];
    if (!want_host) {
      int64_t nsr = 0, nlr = 0;
      for (int k = 0; k < nl; k++) { nsr += srn[k].n; nlr += lr[k].n; }
      if (sr_out) { memset(sr_out, 0, sizeof(*sr_out)); sr_out->n = nsr; }
      if (lr_out) { memset(lr_out, 0, sizeof(*lr_out)); lr_out->n = nlr; }
      if (borderline_out) memset(borderline_out, 0, sizeof(*borderline_out));
      return 0;
    }
    G->h_sr.n = total_sr;
    // long-range and borderline rows: every member's table is in make_blocks order and a block belongs to one member,
    // so the job's table is the members' runs of equal block id, taken in block order
    auto merge = [&](std::vector<ldw_links>& parts, HostLinks& dst) -> int {
      struct Run { int32_t block; int k; int64_t lo, n; };
      std::vector<Run> runs;
      int64_t total = 0;
      for (int k = 0; k < nl; k++) {
        const ldw_links& L = parts[k];
        for (int64_t i = 0; i < L.n;) {
          int64_t j = i;
          while (j < L.n && L.block[j] == L.block[i]) j++;
          runs.push_back({L.block[i], k, i, j - i});
          i = j;
        }
        total += L.n;
      }
      std::stable_sort(runs.begin(), runs.end(), [](const Run& a, const Run& b) { return a.block < b.block; });
      LDW_TRY(dst.ensure(total));
      dst.n = total;
      int64_t o = 0;
      for (const Run& r : runs) {
        const ldw_links& L = parts[r.k];
        memcpy(dst.pos1.as<int32_t>() + o, L.pos1 + r.lo, (size_t)r.n * 4);
        memcpy(dst.pos2.as<int32_t>() + o, L.pos2 + r.lo, (size_t)r.n * 4);
        memcpy(dst.c1.as<int32_t>() + o, L.clust1 + r.lo, (size_t)r.n * 4);
        memcpy(dst.c2.as<int32_t>() + o, L.clust2 + r.lo, (size_t)r.n * 4);
        memcpy(dst.len.as<int32_t>() + o, L.len + r.lo, (size_t)r.n * 4);
        memcpy(dst.blk.as<int32_t>() + o, L.block + r.lo, (size_t)r.n * 4);
        memcpy(dst.mi.as<double>() + o, L.MI + r.lo, (size_t)r.n * 8);
        o += r.n;
      }
      return 0;
    };
    LDW_TRY(merge(lr, G->h_lr));
    LDW_TRY(merge(bd, G->h_border));
    G->h_sr.fill(sr_out);
    G->h_lr.fill(lr_out);
    G->h_border.fill(borderline_out);
    return 0;
  });
}

}  // extern "C"
