// C-ABI entry points for context management, encoding and Hamming-distance weights.
// (The MI-scan entry points live in mi_scan.cu.)
#include "../../include/ldw.h"

#include "ctx.h"
#include "encode.h"
#include "hdw.h"

#include <stdlib.h>

using namespace ldw;

namespace ldw {
int ctx_bind(ldw_ctx* ctx) {
  if (!ctx) return set_error(LDW_ERR_ARG, "null context");
  LDW_CUDA(cudaSetDevice(ctx->device));
  return 0;
}
}  // namespace ldw

extern "C" {

int ldw_abi_version(void) { return LDW_ABI_VERSION; }

const char* ldw_last_error(void) { return last_error_ref().c_str(); }

int ldw_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int ldw_create(int device, ldw_ctx** out) {
  if (!out) return set_error(LDW_ERR_ARG, "ldw_create: null out");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    cudaGetLastError();
    return set_error(LDW_ERR_CUDA, "ldw_create: no CUDA device available (%s); this library has no CPU fallback",
                     e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
  }
  if (device < 0 || device >= n) return set_error(LDW_ERR_ARG, "ldw_create: device %d out of range [0,%d)", device, n);
  LDW_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  LDW_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return set_error(LDW_ERR_UNSUPPORTED, "ldw_create: device %d is sm_%d%d; this build targets sm_100a (B200) only", device,
                     prop.major, prop.minor);
  ldw_ctx* c = new ldw_ctx();
  c->device = device;
  c->num_sms = prop.multiProcessorCount;
  e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) {
    delete c;
    return set_error(LDW_ERR_CUDA, "cudaStreamCreate failed: %s", cudaGetErrorString(e));
  }
  e = cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->select_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->upload_stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) {
    cudaStreamDestroy(c->stream);
    delete c;
    return set_error(LDW_ERR_CUDA, "cudaStreamCreate failed: %s", cudaGetErrorString(e));
  }
  *out = c;
  return 0;
}

void ldw_destroy(ldw_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->scan_ws && ctx->scan_ws_free) ctx->scan_ws_free(ctx->scan_ws);
  cudaDeviceSynchronize();
  ldw::dev_cache_trim();
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  if (ctx->select_stream) cudaStreamDestroy(ctx->select_stream);
  if (ctx->upload_stream) cudaStreamDestroy(ctx->upload_stream);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

}  // extern "C"

namespace {

// The alignment travels to the device in row chunks of at most `budget` bytes, rows padded to a multiple of 16 bytes
// (aligned 128-bit loads in column_count_kernel).  One chunk in the common case; a 100 GB alignment the reference would
// stream record by record (src/getACGTNsites.cpp:49-85) is processed chunk after chunk with O(chunk) device memory.
// LDW_ENCODE_CHUNK_BYTES overrides the 8 GiB default (tests use a few kilobytes to exercise the multi-chunk path).
struct AlnChunks {
  int64_t nseq, slen, pitch, rows_per_chunk, n_chunks;
  DevBuf d;
  int init(int64_t nseq_, int64_t slen_) {
    nseq = nseq_; slen = slen_;
    pitch = round_up(slen, 16);
    int64_t budget = (int64_t)8 << 30;
    if (const char* e = getenv("LDW_ENCODE_CHUNK_BYTES")) { long long v = atoll(e); if (v > 0) budget = v; }
    rows_per_chunk = std::max<int64_t>(1, std::min<int64_t>(nseq, budget / pitch));
    n_chunks = (nseq + rows_per_chunk - 1) / rows_per_chunk;
    return d.alloc((size_t)rows_per_chunk * (size_t)pitch);
  }
  int64_t rows(int64_t c) const { return std::min<int64_t>(rows_per_chunk, nseq - c * rows_per_chunk); }
  int upload(cudaStream_t st, const uint8_t* aln, int64_t c) {
    const int64_t r0 = c * rows_per_chunk;
    LDW_CUDA(cudaMemcpy2DAsync(d.p, (size_t)pitch, aln + r0 * slen, (size_t)slen, (size_t)slen, (size_t)rows(c), cudaMemcpyHostToDevice, st));
    return 0;
  }
};

int check_aln_args(const char* who, const uint8_t* aln, int64_t nseq, int64_t seq_len) {
  if (!aln) return set_error(LDW_ERR_ARG, "%s: null argument", who);
  if (nseq <= 0 || seq_len <= 0) return set_error(LDW_ERR_ARG, "%s: empty alignment (%lld x %lld)", who, (long long)nseq, (long long)seq_len);
  if (nseq > 0x7fffffffLL || seq_len > 0x7fffffffLL) return set_error(LDW_ERR_UNSUPPORTED, "%s: dimensions exceed int32", who);
  return 0;
}

// counts over all chunks, filter, POS to the host.  Leaves the LAST chunk resident in A.d.
int count_and_filter(ldw_ctx* ctx, AlnChunks& A, const uint8_t* aln, int filter, double gap_thresh, double maf_thresh, DevBuf& d_counts,
                     DevBuf& d_pos, int32_t* pos_out, int64_t* n_out) {
  cudaStream_t st = ctx->stream;
  LDW_TRY(d_counts.alloc((size_t)A.slen * 5 * 4));
  LDW_TRY(d_pos.alloc((size_t)A.slen * 4));
  for (int64_t c = 0; c < A.n_chunks; c++) {
    LDW_TRY(A.upload(st, aln, c));
    LDW_TRY(column_counts_device(st, A.d.as<uint8_t>(), A.rows(c), A.slen, A.pitch, d_counts.as<int32_t>(), c > 0));
  }
  int64_t n = 0;
  LDW_TRY(site_filter_device(st, d_counts.as<int32_t>(), A.slen, (int)A.nseq, filter, gap_thresh, maf_thresh, d_pos.as<int32_t>(), &n));
  *n_out = n;
  if (n > 0 && pos_out) LDW_CUDA(cudaMemcpyAsync(pos_out, d_pos.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
  return 0;
}

// class matrix + ACGTN table from the chunks; `resident` = index of the chunk already in A.d (-1: none)
int gather_codes(ldw_ctx* ctx, AlnChunks& A, const uint8_t* aln, int64_t resident, const int32_t* d_pos, int64_t n_snp, DevBuf& d_codes,
                 uint8_t* codes_out, double* table_out) {
  cudaStream_t st = ctx->stream;
  LDW_TRY(d_codes.alloc((size_t)n_snp * A.nseq));
  for (int64_t k = 0; k < A.n_chunks; k++) {
    const int64_t c = (resident >= 0) ? (resident + k) % A.n_chunks : k;  // start with the chunk that is already there
    if (!(resident >= 0 && k == 0)) LDW_TRY(A.upload(st, aln, c));
    LDW_TRY(extract_codes_device(st, A.d.as<uint8_t>(), A.rows(c), A.slen, A.pitch, d_pos, n_snp, d_codes.as<uint8_t>(),
                                 c * A.rows_per_chunk, A.nseq));
  }
  LDW_CUDA(cudaMemcpyAsync(codes_out, d_codes.p, (size_t)n_snp * A.nseq, cudaMemcpyDeviceToHost, st));
  if (table_out) {
    DevBuf d_table, d_mask, d_r, d_dbl;
    LDW_TRY(d_table.alloc((size_t)n_snp * 5 * 4));
    LDW_TRY(d_mask.alloc((size_t)n_snp));
    LDW_TRY(d_r.alloc((size_t)n_snp));
    LDW_TRY(d_dbl.alloc((size_t)n_snp * 5 * 8));
    LDW_TRY(snp_allele_stats(st, d_codes.as<uint8_t>(), n_snp, A.nseq, d_table.as<int32_t>(), d_mask.as<uint8_t>(), d_r.as<uint8_t>()));
    LDW_TRY(counts_to_double_device(st, d_table.as<int32_t>(), n_snp * 5, d_dbl.as<double>()));
    LDW_CUDA(cudaMemcpyAsync(table_out, d_dbl.p, (size_t)n_snp * 5 * 8, cudaMemcpyDeviceToHost, st));
    LDW_CUDA(cudaStreamSynchronize(st));  // the temporaries go out of scope
  }
  LDW_CUDA(cudaStreamSynchronize(st));
  return 0;
}

}  // namespace

extern "C" {

int ldw_aln_param(ldw_ctx* ctx, const uint8_t* aln, int64_t nseq, int64_t seq_len, int filter, double gap_thresh,
                  double maf_thresh, int32_t* pos_out, int64_t* n_snp_out, double* counts_out) {
  LDW_TRY(ctx_bind(ctx));
  LDW_TRY(check_aln_args("ldw_aln_param", aln, nseq, seq_len));
  if (!pos_out || !n_snp_out) return set_error(LDW_ERR_ARG, "ldw_aln_param: null argument");
  if (filter != 0 && filter != 1) return set_error(LDW_ERR_ARG, "ldw_aln_param: filter must be 0 (default) or 1 (relaxed)");
  cudaStream_t st = ctx->stream;
  AlnChunks A;
  LDW_TRY(A.init(nseq, seq_len));
  DevBuf d_counts, d_pos, d_dbl;
  LDW_TRY(count_and_filter(ctx, A, aln, filter, gap_thresh, maf_thresh, d_counts, d_pos, pos_out, n_snp_out));
  if (counts_out) {
    LDW_TRY(d_dbl.alloc((size_t)seq_len * 5 * 8));
    LDW_TRY(counts_to_double_device(st, d_counts.as<int32_t>(), seq_len * 5, d_dbl.as<double>()));
    LDW_CUDA(cudaMemcpyAsync(counts_out, d_dbl.p, (size_t)seq_len * 5 * 8, cudaMemcpyDeviceToHost, st));
  }
  LDW_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int ldw_extract_snps(ldw_ctx* ctx, const uint8_t* aln, int64_t nseq, int64_t seq_len, const int32_t* pos, int64_t n_snp,
                     uint8_t* codes_out, double* table_out) {
  LDW_TRY(ctx_bind(ctx));
  LDW_TRY(check_aln_args("ldw_extract_snps", aln, nseq, seq_len));
  if (!pos || !codes_out) return set_error(LDW_ERR_ARG, "ldw_extract_snps: null argument");
  if (n_snp <= 0) return set_error(LDW_ERR_ARG, "ldw_extract_snps: empty input");
  for (int64_t k = 0; k < n_snp; k++)
    if (pos[k] < 1 || pos[k] > seq_len) return set_error(LDW_ERR_ARG, "ldw_extract_snps: POS[%lld]=%d outside 1..%lld", (long long)k, pos[k], (long long)seq_len);
  cudaStream_t st = ctx->stream;
  AlnChunks A;
  LDW_TRY(A.init(nseq, seq_len));
  DevBuf d_pos, d_codes;
  LDW_TRY(d_pos.alloc((size_t)n_snp * 4));
  LDW_CUDA(cudaMemcpyAsync(d_pos.p, pos, (size_t)n_snp * 4, cudaMemcpyHostToDevice, st));
  return gather_codes(ctx, A, aln, -1, d_pos.as<int32_t>(), n_snp, d_codes, codes_out, table_out);
}

// ldw_aln_param + ldw_extract_snps in one call: the alignment crosses PCIe ONCE when it fits one chunk (the reference
// reads its file three times, src/getACGTNsites.cpp:33,44,212); larger inputs stream through in row chunks, twice.
int ldw_encode_alignment(ldw_ctx* ctx, const uint8_t* aln, int64_t nseq, int64_t seq_len, int filter, double gap_thresh,
                         double maf_thresh, int64_t* n_snp_out, int32_t** pos_out, uint8_t** codes_out, double** table_out) {
  LDW_TRY(ctx_bind(ctx));
  LDW_TRY(check_aln_args("ldw_encode_alignment", aln, nseq, seq_len));
  if (!n_snp_out || !pos_out || !codes_out || !table_out) return set_error(LDW_ERR_ARG, "ldw_encode_alignment: null argument");
  if (filter != 0 && filter != 1) return set_error(LDW_ERR_ARG, "ldw_encode_alignment: filter must be 0 (default) or 1 (relaxed)");
  *n_snp_out = 0; *pos_out = nullptr; *codes_out = nullptr; *table_out = nullptr;
  cudaStream_t st = ctx->stream;
  AlnChunks A;
  LDW_TRY(A.init(nseq, seq_len));
  DevBuf d_counts, d_pos, d_codes;
  int64_t n = 0;
  LDW_TRY(count_and_filter(ctx, A, aln, filter, gap_thresh, maf_thresh, d_counts, d_pos, nullptr, &n));
  *n_snp_out = n;
  if (n == 0) return 0;
  int32_t* pos = (int32_t*)malloc((size_t)n * 4);
  uint8_t* codes = (uint8_t*)malloc((size_t)n * (size_t)nseq);
  double* table = (double*)malloc((size_t)n * 5 * 8);
  int rc = (pos && codes && table) ? 0 : set_error(LDW_ERR_NOMEM, "ldw_encode_alignment: out of host memory");
  if (rc == 0) {
    cudaError_t e = cudaMemcpyAsync(pos, d_pos.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st);
    if (e != cudaSuccess) rc = set_error(LDW_ERR_CUDA, "cudaMemcpyAsync failed: %s", cudaGetErrorString(e));
  }
  if (rc == 0) rc = gather_codes(ctx, A, aln, A.n_chunks - 1, d_pos.as<int32_t>(), n, d_codes, codes, table);
  if (rc != 0) { free(pos); free(codes); free(table); return rc; }
  *pos_out = pos; *codes_out = codes; *table_out = table;
  return 0;
}

int ldw_acgtn2num(ldw_ctx* ctx, double* nv, const char* ref, int64_t n) {
  LDW_TRY(ctx_bind(ctx));
  if (n == 0) return 0;
  if (!nv || !ref || n < 0) return set_error(LDW_ERR_ARG, "ldw_acgtn2num: bad argument");
  cudaStream_t st = ctx->stream;
  DevBuf d_nv, d_ref;
  LDW_TRY(d_nv.alloc((size_t)n * 5 * 8));
  LDW_TRY(d_ref.alloc((size_t)n));
  LDW_CUDA(cudaMemcpyAsync(d_nv.p, nv, (size_t)n * 5 * 8, cudaMemcpyHostToDevice, st));
  LDW_CUDA(cudaMemcpyAsync(d_ref.p, ref, (size_t)n, cudaMemcpyHostToDevice, st));
  LDW_TRY(acgtn2num_device(st, d_nv.as<double>(), d_ref.as<char>(), n));
  LDW_CUDA(cudaMemcpyAsync(nv, d_nv.p, (size_t)n * 5 * 8, cudaMemcpyDeviceToHost, st));
  LDW_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int ldw_hdw(ldw_ctx* ctx, const uint8_t* codes, int64_t n_snp, int64_t nseq, double threshold, int32_t* cnt_out,
            double* hdw_out, int32_t* dist_out) {
  LDW_TRY(ctx_bind(ctx));
  if (!codes || !hdw_out) return set_error(LDW_ERR_ARG, "ldw_hdw: null argument");
  if (n_snp <= 0 || nseq <= 0) return set_error(LDW_ERR_ARG, "ldw_hdw: empty input");
  if (nseq > 0x7fffffffLL / 4) return set_error(LDW_ERR_UNSUPPORTED, "ldw_hdw: too many sequences");
  cudaStream_t st = ctx->stream;
  int thresh = (int)((double)n_snp * threshold);  // as.integer(nsnp*threshold): truncation (:23)
  DevBuf d_codes, d_neigh, d_w, d_dist;
  LDW_TRY(d_codes.alloc((size_t)n_snp * nseq));
  LDW_TRY(d_neigh.alloc((size_t)nseq * 4));
  LDW_TRY(d_w.alloc((size_t)nseq * 8));
  if (dist_out) LDW_TRY(d_dist.alloc((size_t)nseq * nseq * 4));
  LDW_CUDA(cudaMemcpyAsync(d_codes.p, codes, (size_t)n_snp * nseq, cudaMemcpyHostToDevice, st));
  // every class must be 0..4 (as ldw_group_load_codes and ldw_mi_plan_create check): the plane packing compares a code
  // with the allele index, so a byte above 4 would give distances that are neither the reference's nor an error
  uint32_t mx = 0;
  LDW_TRY(max_byte_device(st, d_codes.as<uint8_t>(), n_snp * nseq, &mx));
  if (mx > 4) return set_error(LDW_ERR_ARG, "ldw_hdw: the matrix holds a class %u outside 0..4", mx);
  LDW_TRY(hdw_device(st, d_codes.as<uint8_t>(), n_snp, nseq, thresh, d_neigh.as<int32_t>(), d_w.as<double>(),
                     dist_out ? d_dist.as<int32_t>() : nullptr, ctx->num_sms));
  if (cnt_out) LDW_CUDA(cudaMemcpyAsync(cnt_out, d_neigh.p, (size_t)nseq * 4, cudaMemcpyDeviceToHost, st));
  LDW_CUDA(cudaMemcpyAsync(hdw_out, d_w.p, (size_t)nseq * 8, cudaMemcpyDeviceToHost, st));
  if (dist_out) LDW_CUDA(cudaMemcpyAsync(dist_out, d_dist.p, (size_t)nseq * nseq * 4, cudaMemcpyDeviceToHost, st));
  LDW_CUDA(cudaStreamSynchronize(st));
  return 0;
}

}  // extern "C"
