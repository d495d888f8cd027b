// The context behind the opaque ldw_ctx handle.
#pragma once
#include "host_util.h"

// The seven link columns pos1 pos2 c1 c2 len blk mi (int32 but mi, which is double) over one kind of buffer: pinned host
// memory (HostLinks) or device memory (the scan's workspace).  col(k) and elem(k), k < NCOL, are column k and the
// size of its element.
template <class Buf>
struct LinkCols {
  static constexpr int NCOL = 7;
  Buf pos1, pos2, c1, c2, len, blk, mi;
  int64_t n = 0;
  static size_t elem(int k) { return k == 6 ? 8 : 4; }
  Buf& col(int k) {
    Buf* c[NCOL] = {&pos1, &pos2, &c1, &c2, &len, &blk, &mi};
    return *c[k];
  }
  int ensure(int64_t m) {
    for (int k = 0; k < NCOL; k++) LDW_TRY(col(k).ensure((size_t)(m > 0 ? m : 1) * elem(k)));
    return 0;
  }
  void fill(ldw_links* o) const {
    if (!o) return;
    o->n = n;
    o->pos1 = pos1.template as<int32_t>(); o->pos2 = pos2.template as<int32_t>();
    o->clust1 = c1.template as<int32_t>(); o->clust2 = c2.template as<int32_t>();
    o->len = len.template as<int32_t>(); o->MI = mi.template as<double>(); o->block = blk.template as<int32_t>();
  }
  // column k of a table handed out through the ABI (the counterpart of fill)
  static const char* abi_col(const ldw_links& L, int k) {
    const void* c[NCOL] = {L.pos1, L.pos2, L.clust1, L.clust2, L.len, L.block, L.MI};
    return static_cast<const char*>(c[k]);
  }
};

// Link columns in pinned host memory (what ldw_links points into).  Owned by the context and reused by every
// scan on it: allocating gigabytes of pinned memory costs far more than the scan itself.
using HostLinks = LinkCols<ldw::PinnedBuf>;

struct ldw_ctx {
  int device = 0;
  int num_sms = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;  // device -> host copies of finished link columns overlap the scan
  cudaStream_t upload_stream = nullptr;  // per-block tables host -> device, ahead of the block's scan
  cudaStream_t select_stream = nullptr;  // fp64 refinement + long-range selection of block b overlap the scan of block b+1
  HostLinks h_sr, h_lr, h_border;
  // scan workspace (device scratch, per-block ring, link columns): allocated on first use by mi_scan.cu, reused by
  // every plan on this context, released by ldw_destroy
  void* scan_ws = nullptr;
  void (*scan_ws_free)(void*) = nullptr;
  // The short-range table the last scan on this context left in device memory (columns inside scan_ws; valid until the
  // next scan): what ldw_sr_postprocess_dev works on.  n < 0: none (no scan yet, a partial scan, or no rows materialised).
  ldw_links dev_sr = {-1};
};

namespace ldw {
// Binds the calling thread to the context's device.
int ctx_bind(ldw_ctx* ctx);
}  // namespace ldw
