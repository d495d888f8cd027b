// Auxiliary kernels of the MI scan: operand packing, per-SNP records, exact (fp64) refinement of long-range
// candidates, exact type-7 quantile selection, link materialisation.  All HBM-/latency-bound helpers; the hot
// kernel is mi_kernel.cuh.
#pragma once
#include "mi_types.h"

namespace ldw {

// ------------------------------------------------------------------------------------------------
// Per-slot records.  One warp per slot: class-wise exact fp64 marginals p^a = sum_s w_s [code = a] (kept per SNP for
// the fp64 refinement) and the fixed-point marginals in the SAME digits the GEMM uses, so that
// sum_b C^ab == P^a holds exactly in integers.  T carries the pseudocounts of its row of the joint table (see M below).
__global__ void mi_build_rec_kernel(const uint8_t* __restrict__ codes, int64_t S, const int32_t* __restrict__ slot_snp,
                                    int64_t nslots, const uint8_t* __restrict__ mask, const double* __restrict__ w,
                                    const int32_t* __restrict__ wH, const int32_t* __restrict__ wL, Rec* rec,
                                    int64_t vstride, double* p64 /*[n][5]*/, uint32_t sa, uint32_t sb, uint32_t M) {
  int64_t slot = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (slot >= nslots) return;
  int32_t snp = slot_snp[slot];
  if (snp < 0) {
    if (lane < 4) {
      Rec z;
      for (int q = 0; q < 4; q++) { z.T[q] = 0; z.rp[q] = 0.f; z.q[q] = 1.f; }
      z.T4 = 0; z.rp4 = 0.f; z.q4 = 1.f; z.pad = 0;
      rec[lane * vstride + slot] = z;
    }
    return;
  }
  const uint8_t* row = codes + (int64_t)snp * S;
  double p[5] = {0, 0, 0, 0, 0};
  int h[5] = {0, 0, 0, 0, 0}, l[5] = {0, 0, 0, 0, 0};
  for (int64_t s = lane; s < S; s += 32) {
    int c = row[s];
    double ws = w[s];
    int hs = wH[s], ls = wL[s];
#pragma unroll
    for (int a = 0; a < 5; a++) {
      bool m = (c == a);
      p[a] += m ? ws : 0.0;
      h[a] += m ? hs : 0;
      l[a] += m ? ls : 0;
    }
  }
#pragma unroll
  for (int a = 0; a < 5; a++)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      p[a] += __shfl_xor_sync(0xffffffffu, p[a], o);
      h[a] += __shfl_xor_sync(0xffffffffu, h[a], o);
      l[a] += __shfl_xor_sync(0xffffffffu, l[a], o);
    }
  if (lane == 0)
    for (int a = 0; a < 5; a++) p64[(int64_t)snp * 5 + a] = p[a];
  if (lane < 4) {
    // variant `lane`: partner SNP has r' = lane + 2 observed alleles
    int m = mask[snp];
    uint32_t qt[5] = {0, 0, 0, 0, 0};
    float qr[5] = {0.f, 0.f, 0.f, 0.f, 0.f}, qq[5] = {1.f, 1.f, 1.f, 1.f, 1.f};
    int q = 0;
    for (int a = 0; a < 5; a++) {
      if (m & (1 << a)) {
        // the pseudocount 0.5 is M count units; a row of the joint table holds r' cells, so the marginal carries r' * M
        qt[q] = ((uint32_t)h[a] << sa) + ((uint32_t)l[a] >> sb) + M * (uint32_t)(lane + 2);
        const double v = p[a] + 0.5 * (double)(lane + 2);
        qr[q] = (float)(1.0 / v);
        qq[q] = (float)v;
        q++;
      }
    }
    Rec z;
    for (int t = 0; t < 4; t++) { z.T[t] = qt[t]; z.rp[t] = qr[t]; z.q[t] = qq[t]; }
    z.T4 = qt[4]; z.rp4 = qr[4]; z.q4 = qq[4]; z.pad = 0;
    rec[lane * vstride + slot] = z;
  }
}

// Operand rows.  row_info[R] = snp | allele << 28, or 0xFFFFFFFF for padding rows.  Each thread writes one 16-byte
// chunk (16 sequences) of the one-hot plane matrix X [rows][Kpad]; a match is stored as 0xFF (+255 unsigned /
// -1 signed, see the weight digits in build_plan).
__global__ void mi_pack_operands_kernel(const uint8_t* __restrict__ codes, int64_t S, int64_t Kpad,
                                        const uint32_t* __restrict__ row_info, int64_t nrows, uint8_t* X) {
  int64_t chunks = Kpad / 16;
  int64_t id = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= nrows * chunks) return;
  int64_t R = id / chunks, ch = id % chunks;
  uint32_t info = row_info[R];
  uint32_t x1[4] = {0, 0, 0, 0};
  if (info != 0xFFFFFFFFu) {
    const uint8_t* row = codes + (int64_t)(info & 0x0FFFFFFF) * S;
    int al = info >> 28;
    int64_t s0 = ch * 16;
#pragma unroll
    for (int k = 0; k < 16; k++) {
      int64_t s = s0 + k;
      uint32_t bit = (s < S && row[s] == al) ? 0xFFu : 0u;
      x1[k >> 2] |= bit << (8 * (k & 3));
    }
  }
  *reinterpret_cast<uint4*>(X + R * Kpad + ch * 16) = make_uint4(x1[0], x1[1], x1[2], x1[3]);
}

// ------------------------------------------------------------------------------------------------
// Exact fp64 MI of explicit pairs, following the reference arithmetic literally
// (R/computePairwiseMI.R:260-263, :391-395 and src/computeMI.cpp:19), including quirk Q1.
struct RefineParams {
  const uint8_t* codes;
  int64_t S;
  const double* w;
  const double* p64;      // [n][5]
  const uint8_t* r;       // per SNP
  const uint8_t* mask;    // per SNP
  const int32_t* from_idx;  // local -> global SNP
  const int32_t* to_idx;
  const uint8_t* rfl_arr;   // r of from-list by local index
  const uint8_t* rtl_arr;
  int32_t nf, nt;
  int32_t ideal_q;
  double neff;
};

// One warp per pair.  The joint table is built from the sequences that carry a NON-base class at BOTH sites (base class =
// the heaviest class of a site, typically 5-10 % of the sequences); the cells of the base row / column follow from the
// exact fp64 marginals p64 (sum_b c^ab = p_i^a), the corner from p_i^base.  Against summing all 25 cells directly this
// moves the counts by a few ulp (both forms are fp64 sums of the same weights in a different association; the reference's
// own order is that of a sparse matrix product), far inside the 1e-12 the fp64 paths are held to, and touches a
// sixteenth of the (sequence, cell) updates.
// `acc` is this warp's scratch in shared memory: 32 lanes x 25 cells (doubles, lane-major with a stride of 25 so lanes hit
// different banks), ALL ZERO on entry and on return.  Each lane adds the weights of its sequences into its own row and
// remembers which cells it touched; every touched cell is then reduced over the lanes by a fixed butterfly (deterministic).
constexpr int REFINE_WARPS = 6;
__device__ __forceinline__ int heaviest_class(const double (&p)[5]) {
  int b = 0;
#pragma unroll
  for (int a = 1; a < 5; a++) b = p[a] > p[b] ? a : b;
  return b;
}
__device__ __forceinline__ void refine_scratch_clear(double* acc, int lane) {  // once per kernel, before the first pair
#pragma unroll
  for (int k = 0; k < 25; k++) acc[lane * 25 + k] = 0.0;
}
__device__ __forceinline__ double refine_pair(const RefineParams& P, int il, int jl, int lane, double* acc) {
  const int gi = P.from_idx[il], gj = P.to_idx[jl];
  const uint8_t* ci = P.codes + (int64_t)gi * P.S;
  const uint8_t* cj = P.codes + (int64_t)gj * P.S;
  double pi[5], pj[5];
#pragma unroll
  for (int a = 0; a < 5; a++) { pi[a] = P.p64[(int64_t)gi * 5 + a]; pj[a] = P.p64[(int64_t)gj * 5 + a]; }
  const int bi = heaviest_class(pi), bj = heaviest_class(pj);
  double* mine = acc + lane * 25;
  uint32_t touched = 0;
  if ((P.S & 3) == 0) {
    // rows are 4-byte aligned (S % 4 == 0, cudaMalloc base): four sequences per load, most words hold no such sequence
    const uint32_t* wi = reinterpret_cast<const uint32_t*>(ci);
    const uint32_t* wj = reinterpret_cast<const uint32_t*>(cj);
    const uint32_t vbi = 0x01010101u * (uint32_t)bi, vbj = 0x01010101u * (uint32_t)bj;
    const int nw = (int)(P.S >> 2);
    for (int q = lane; q < nw; q += 32) {
      const uint32_t a4 = __ldg(wi + q), b4 = __ldg(wj + q);
      uint32_t m = __vcmpne4(a4, vbi) & __vcmpne4(b4, vbj);  // 0xFF per byte where both classes differ from their base
      while (m) {
        const int k = (__ffs(m) - 1) >> 3;
        m &= ~(0xFFu << (8 * k));
        const int idx = (int)((a4 >> (8 * k)) & 0xFF) * 5 + (int)((b4 >> (8 * k)) & 0xFF);
        mine[idx] += P.w[4 * q + k];
        touched |= 1u << idx;
      }
    }
  } else {
    for (int64_t s = lane; s < P.S; s += 32) {
      const int a = ci[s], b = cj[s];
      if (a != bi && b != bj) {
        mine[a * 5 + b] += P.w[s];
        touched |= 1u << (a * 5 + b);
      }
    }
  }
  const uint32_t any = __reduce_or_sync(0xffffffffu, touched);
  // lane k < 25 ends up holding the reduced cell k of the non-base block (zero elsewhere)
  double cell = 0.0;
  for (uint32_t m = any; m; m &= m - 1) {
    const int k = __ffs(m) - 1;
    double v = mine[k];
    if ((touched >> k) & 1) mine[k] = 0.0;  // leave the scratch clean for the next pair
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == k) cell = v;
  }
  // row / column sums of the non-base block, then the base row, base column and corner from the marginals
  const int a = lane < 25 ? lane / 5 : 0, b = lane < 25 ? lane % 5 : 0;
  double rs = 0.0, cs = 0.0;
#pragma unroll
  for (int t = 0; t < 5; t++) {
    rs += __shfl_sync(0xffffffffu, cell, a * 5 + t);
    cs += __shfl_sync(0xffffffffu, cell, t * 5 + b);
  }
  double tot = 0.0;
#pragma unroll
  for (int t = 0; t < 5; t++) tot += __shfl_sync(0xffffffffu, rs, t * 5);
  if (lane < 25) {
    if (a == bi && b == bj) {
      double o = 0.0;
#pragma unroll
      for (int t = 0; t < 5; t++) o += (t != bj) ? pj[t] : 0.0;
      cell = pi[bi] - o + tot;
    } else if (a == bi) {
      cell = pj[b] - cs;
    } else if (b == bj) {
      cell = pi[a] - rs;
    }
  }
  const double ri = (double)P.r[gi], rj = (double)P.r[gj];
  const int mi_ = P.mask[gi], mj_ = P.mask[gj];
  const double den = P.neff + ri * rj * 0.5;
  double Q;
  if (P.ideal_q) {
    Q = ri * rj * 0.25;
  } else {
    // quirk Q1: linear index il + jl * nf of the nf x nt matrix, read as (index / nt, index % nt); square blocks: (jl, il)
    uint32_t cdiv = (uint32_t)jl, cmod = (uint32_t)il;
    if (P.nf != P.nt) {
      uint64_t lin = (uint64_t)il + (uint64_t)jl * (uint64_t)P.nf;
      cdiv = (uint32_t)(lin / (uint32_t)P.nt); cmod = (uint32_t)(lin % (uint32_t)P.nt);
    }
    Q = (double)P.rfl_arr[cdiv] * (double)P.rtl_arr[cmod] * 0.25;
  }
  // lane k < 25 owns term (a, b) = (k / 5, k % 5); the 25 terms are summed by a fixed butterfly over the warp
  double term = 0.0;
  if (lane < 25) {
    if (((mi_ >> a) & 1) && ((mj_ >> b) & 1)) {
      double pxy = cell + 0.5;
      double pa = pi[a], pb = pj[b];
      double dsum = pa * pb + Q + pa * (0.5 * ri) + pb * (0.5 * rj);
      term = pxy / den * log(pxy / dsum * den);
    }
  }
  double mi = term;  // lanes 25..31 hold 0
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mi += __shfl_xor_sync(0xffffffffu, mi, o);
  return mi;
}

// ------------------------------------------------------------------------------------------------
// Pre-selection on the fp32 values the scan kernel produced.  The exact (fp64) K-th largest MI of a block lies within
// eps (the fp32 epilogue's error, < 5e-7 measured) of the K-th largest fp32 value v32, and every candidate whose exact
// value reaches it has an fp32 value >= v32 - 2 eps.  So only the candidates with mi32 >= v32 - delta (delta = 4e-6)
// have to be refined and ranked exactly: about K of them instead of every collected candidate (4-30 x K).  Candidates
// below the FINAL candidate threshold are an incomplete sample of their MI range (the threshold rose while they were
// being collected) and never take part.  Single CTA; MSB-first radix select on order-preserving 32-bit keys.
__device__ __forceinline__ uint32_t fkey(float v) {
  uint32_t b = __float_as_uint(v);
  return (b >> 31) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float fkey_inv(uint32_t k) {
  return __uint_as_float((k >> 31) ? (k & 0x7FFFFFFFu) : ~k);
}

// k-th largest (1-based) fp32 MI among the candidates with mi >= tc.  Whole CTA (any block size), MSB-first radix select
// on order-preserving keys; hist: 256 words, bc: 2 words of shared memory.  Four loads in flight per thread: these
// single-CTA passes are latency-bound.
__device__ float kth_largest_f32(const Cand* __restrict__ cand, uint32_t n, float tc, uint32_t kth, uint32_t* hist, uint32_t* bc) {
  uint32_t prefix = 0, mask = 0, remaining = kth;
  for (int byte = 3; byte >= 0; byte--) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < n; i += 4 * blockDim.x) {
      float v[4];
#pragma unroll
      for (int u = 0; u < 4; u++) { const uint32_t j = i + u * blockDim.x; v[u] = j < n ? cand[j].mi : -3.0e38f; }
#pragma unroll
      for (int u = 0; u < 4; u++) {
        if (i + u * blockDim.x < n && v[u] >= tc) {
          const uint32_t k = fkey(v[u]);
          if ((k & mask) == prefix) atomicAdd(&hist[(k >> (8 * byte)) & 255], 1u);
        }
      }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t cum = 0;
      int d = 255;
      for (; d > 0; d--) {
        if (cum + hist[d] >= remaining) break;
        cum += hist[d];
      }
      bc[0] = (uint32_t)d;
      bc[1] = remaining - cum;
    }
    __syncthreads();
    prefix |= bc[0] << (8 * byte);
    mask |= 0xFFu << (8 * byte);
    remaining = bc[1];
    __syncthreads();
  }
  return fkey_inv(prefix);
}

// Pilot seed for the first block of a scan call.  A few dozen tiles spread over the block were scanned with every
// long-range pair collected; the rank K of the block scales to K * (pairs collected / long-range pairs of the block)
// in that sample, and 0.85 x the sample's value at that rank seeds the block's candidate threshold (the MI tail is
// steep: a 15 % error in the rank moves the value by ~2 %).  Without it every CTA's first tile is collected whole
// (~6 x 10^5 candidates per block).  Only steers how much is collected; the selection stays exact and self-checking.
__global__ void __launch_bounds__(1024) mi_pilot_seed_kernel(const Cand* __restrict__ cand, const uint32_t* __restrict__ count,
                                                             uint32_t cap, unsigned long long k_lo, double n_lr, uint32_t* chain_bits) {
  __shared__ uint32_t hist[256];
  __shared__ uint32_t bc[2];
  const uint32_t n = *count < cap ? *count : cap;
  const double ks = (double)k_lo * (double)n / n_lr;
  if (!(ks >= 16.0) || n < 1024) return;  // too small a sample: start from zero as before
  const float v = kth_largest_f32(cand, n, -3.0e38f, (uint32_t)ks, hist, bc);
  if (threadIdx.x == 0 && v > 0.f) *chain_bits = __float_as_uint(0.85f * v);
}

__global__ void __launch_bounds__(1024) mi_presel_kernel(const Cand* __restrict__ cand, const uint32_t* __restrict__ count,
                                                         uint32_t cap, const uint32_t* __restrict__ tcand_bits, int emit_all,
                                                         unsigned long long k_lo, float delta, Cand* vcand, uint32_t* vcount) {
  __shared__ uint32_t hist[256];
  __shared__ uint32_t bc[2];
  __shared__ uint32_t s_nvalid;
  const uint32_t n = *count < cap ? *count : cap;
  const float tc = emit_all ? -3.0e38f : __uint_as_float(*tcand_bits);
  if (threadIdx.x == 0) s_nvalid = 0;
  __syncthreads();
  {
    uint32_t c = 0;
    // four independent loads in flight per thread: these single-CTA passes are latency-bound
    for (uint32_t i = threadIdx.x; i < n; i += 4 * blockDim.x) {
      float v[4];
#pragma unroll
      for (int u = 0; u < 4; u++) { const uint32_t j = i + u * blockDim.x; v[u] = j < n ? cand[j].mi : -3.0e38f; }
#pragma unroll
      for (int u = 0; u < 4; u++) c += (i + u * blockDim.x < n && v[u] >= tc) ? 1u : 0u;
    }
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(&s_nvalid, c);
  }
  __syncthreads();
  float lim = tc;  // fewer valid candidates than the rank asked for: pass them all on, the selection reports it
  if ((unsigned long long)s_nvalid >= k_lo && k_lo >= 1) {
    const float v32 = kth_largest_f32(cand, n, tc, (uint32_t)k_lo, hist, bc);
    lim = fmaxf(tc, v32 - delta);
  }
  const int lane = threadIdx.x & 31;
  for (uint32_t i0 = 0; i0 < n; i0 += blockDim.x) {
    const uint32_t i = i0 + threadIdx.x;
    Cand c;
    bool take = false;
    if (i < n) { c = cand[i]; take = (c.mi >= lim) && (c.mi >= tc); }
    const unsigned bal = __ballot_sync(0xffffffffu, take);
    if (bal) {
      uint32_t base = 0;
      if (lane == __ffs(bal) - 1) base = atomicAdd(vcount, (uint32_t)__popc(bal));
      base = __shfl_sync(0xffffffffu, base, __ffs(bal) - 1);
      if (take) vcand[base + (uint32_t)__popc(bal & ((1u << lane) - 1))] = c;
    }
  }
}

// fp64 refinement of a compact candidate list (one warp per pair).
__global__ void mi_refine_list_kernel(RefineParams P, const Cand* __restrict__ list, const uint32_t* __restrict__ n_ptr, double* vmi) {
  __shared__ double acc_s[REFINE_WARPS][32 * 25];
  const uint32_t n = *n_ptr;
  const int lane = threadIdx.x & 31;
  double* acc = acc_s[threadIdx.x >> 5];
  refine_scratch_clear(acc, threadIdx.x & 31);
  for (uint32_t i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n; i += gridDim.x * (blockDim.x >> 5)) {
    const Cand c = list[i];
    const double v = refine_pair(P, c.il, c.jl, lane, acc);
    if (lane == 0) vmi[i] = v;
  }
}

// Start of a block's long-range collection: counters cleared, histogram cleared, candidate threshold seeded from
// the chained estimate of the previous block (or 0 = collect until the histogram can place a threshold).
__global__ void mi_block_begin_kernel(uint32_t* state /*count, tcand, overflow, -, -, vcount*/, uint32_t* hist,
                                      const uint32_t* chain_bits, int use_chain) {
  for (int i = threadIdx.x; i < MI_HIST_BINS; i += blockDim.x) hist[i] = 0;
  if (threadIdx.x == 0) {
    state[0] = 0;
    state[1] = use_chain ? *chain_bits : 0u;
    state[2] = 0;
    state[5] = 0;
  }
}

__global__ void mi_refine_pairs_kernel(RefineParams P, const int32_t* __restrict__ il, const int32_t* __restrict__ jl,
                                       int64_t n, double* out) {
  __shared__ double acc_s[REFINE_WARPS][32 * 25];
  int lane = threadIdx.x & 31;
  double* acc = acc_s[threadIdx.x >> 5];
  refine_scratch_clear(acc, threadIdx.x & 31);
  for (int64_t i = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n;
       i += (int64_t)gridDim.x * (blockDim.x >> 5)) {
    double v = refine_pair(P, il[i], jl[i], lane, acc);
    if (lane == 0) out[i] = v;
  }
}

// ------------------------------------------------------------------------------------------------
// Exact per-block long-range selection: type-7 quantile over the block's long-range MI values from the
// K largest refined candidates, then `MI >= thr` (R/computePairwiseMI.R:352-358, stats::quantile type 7).
struct BlockResult {
  double thr;
  double v_lo;
  uint32_t n_cand;
  uint32_t n_kept;
  uint32_t n_border;
  uint32_t bad;  // 1: candidate buffer overflowed; 2: fewer candidates than needed; 4: threshold guess not provably safe;
                 // 8: the fp32 epilogue's error observed on this block's refined candidates is too large for the margins used
  float eps_obs; // max |fp32 MI - fp64 MI| over the refined candidates
  uint32_t pad;
};

struct SelectParams {
  const Cand* cand;       // compact: refined candidates only
  const double* mi64;
  const uint32_t* vcount; // number of refined candidates
  const uint32_t* count;  // raw number collected by the scan kernel
  uint32_t cap;
  const uint32_t* overflow;
  const uint32_t* tcand_bits;
  int32_t emit_all;
  uint64_t k_lo, k_hi;  // ranks from the top (1-based) of x[lo], x[hi]
  double h;             // interpolation weight (index - lo)
  int32_t interpolate;  // index > lo
  double tol_safe;      // margin between v_lo and the candidate threshold that proves the candidate set is complete
  double tol_border;
  const int32_t* from_idx;
  const int32_t* to_idx;
  int32_t nf, nt, diag;
  int32_t block;
  // outputs (global, appended)
  uint64_t* kept_key;
  int32_t* kept_gi;
  int32_t* kept_gj;
  double* kept_mi;
  unsigned long long* kept_count;
  uint64_t kept_cap;
  uint32_t* kept_overflow;
  uint32_t* chain_bits;  // seed of the next block's candidate threshold
  BlockResult* result;
};

__device__ __forceinline__ uint64_t dkey(double v) {
  uint64_t b = (uint64_t)__double_as_longlong(v);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double dkey_inv(uint64_t k) {
  uint64_t b = (k >> 63) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k;
  return __longlong_as_double((long long)b);
}

// K-th largest (1-based) of n doubles by MSB-first radix select.  Whole CTA; returns the key to all threads.
__device__ uint64_t select_kth_largest(const double* v, uint32_t n, uint64_t K, uint32_t* hist /*256 smem*/,
                                       uint64_t* bcast /*smem*/) {
  uint64_t prefix = 0, mask = 0, remaining = K;
  for (int byte = 7; byte >= 0; byte--) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < n; i += 4 * blockDim.x) {
      double x[4];
#pragma unroll
      for (int u = 0; u < 4; u++) { const uint32_t j = i + u * blockDim.x; x[u] = j < n ? v[j] : 0.0; }
#pragma unroll
      for (int u = 0; u < 4; u++) {
        if (i + u * blockDim.x < n) {
          const uint64_t k = dkey(x[u]);
          if ((k & mask) == prefix) atomicAdd(&hist[(k >> (8 * byte)) & 255], 1u);
        }
      }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      uint64_t cum = 0;
      int d = 255;
      for (; d > 0; d--) {
        if (cum + hist[d] >= remaining) break;
        cum += hist[d];
      }
      bcast[0] = (uint64_t)d;
      bcast[1] = remaining - cum;
    }
    __syncthreads();
    prefix |= bcast[0] << (8 * byte);
    mask |= 0xFFull << (8 * byte);
    remaining = bcast[1];
    __syncthreads();
  }
  return prefix;
}

// rank of pair (il, jl) in the reference's row order of a block (R/computePairwiseMI.R:306-310)
__device__ __forceinline__ uint64_t pair_rank(int64_t il, int64_t jl, int64_t nf, int64_t nt, int diag) {
  if (diag) {  // lower.tri(t(MI)): column-major over row > col
    int64_t m = jl < nf ? jl : nf;
    return (uint64_t)(m * (nf - 1) - m * (m - 1) / 2 + (il - jl - 1));
  }
  if (il < jl) {  // upper part first
    int64_t U = jl <= nf ? jl * (jl - 1) / 2 : nf * (nf - 1) / 2 + (jl - nf) * nf;
    return (uint64_t)(U + il);
  }
  int64_t n_upper = nt <= nf ? nt * (nt - 1) / 2 : nf * (nf - 1) / 2 + (nt - nf) * nf;
  int64_t m = jl < nf ? jl : nf;
  return (uint64_t)(n_upper + m * (nf - 1) - m * (m - 1) / 2 + (il - jl - 1));
}

__global__ void __launch_bounds__(1024) mi_select_kernel(SelectParams P) {
  __shared__ uint32_t hist[256];
  __shared__ uint64_t bcast[2];
  __shared__ uint32_t s_kept, s_border;
  const uint32_t raw = *P.count;
  const uint32_t n = *P.vcount;
  uint32_t bad = 0;
  if (*P.overflow || raw > P.cap) bad |= 1;
  if ((uint64_t)n < P.k_lo) bad |= 2;
  double thr = 0.0, v_lo = 0.0;
  if (!(bad & 2) && n > 0) {
    v_lo = dkey_inv(select_kth_largest(P.mi64, n, P.k_lo, hist, bcast));
    thr = v_lo;
    if (P.interpolate && P.k_hi >= 1 && P.k_hi != P.k_lo) {
      // x[hi] is the next order statistic above x[lo]: if exactly k_lo - 1 values are strictly greater it is the
      // smallest of them, otherwise (ties at x[lo]) it equals x[lo]
      __shared__ unsigned long long s_min_above;
      __shared__ uint32_t s_above;
      if (threadIdx.x == 0) { s_min_above = ~0ull; s_above = 0; }
      __syncthreads();
      uint32_t cnt = 0;
      unsigned long long mn = ~0ull;
      for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
        double v = P.mi64[i];
        if (v > v_lo) { cnt++; unsigned long long kx = dkey(v); mn = kx < mn ? kx : mn; }
      }
      atomicAdd(&s_above, cnt);
      atomicMin(&s_min_above, mn);
      __syncthreads();
      if ((uint64_t)s_above == P.k_lo - 1 && s_above > 0) {
        double v_hi = dkey_inv((uint64_t)s_min_above);
        if (v_hi != v_lo) thr = (1.0 - P.h) * v_lo + P.h * v_hi;  // stats::quantile type 7
      }
    }
    if (!P.emit_all) {
      double tc = (double)__uint_as_float(*P.tcand_bits);
      if (!(v_lo >= tc + P.tol_safe)) bad |= 4;
    }
  }
  // The pre-selection kept the candidates with fp32 MI >= v32 - tol_safe and the completeness test above uses the same
  // margin; both are sound when the epilogue's error eps satisfies 2 eps <= tol_safe.  That error depends on the input
  // (fixed-point weight rounding adds up coherently inside large clusters of equal weights), so it is MEASURED here on
  // the refined candidates -- the pairs around the threshold, where it matters -- and the block is sent back for a
  // re-run with wider margins unless there is a factor 2 of head room (4 eps_obs <= tol_safe).
  __shared__ float s_eps;
  if (threadIdx.x == 0) s_eps = 0.f;
  __syncthreads();
  {
    float e = 0.f;
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) e = fmaxf(e, (float)fabs((double)P.cand[i].mi - P.mi64[i]));
    for (int o = 16; o > 0; o >>= 1) e = fmaxf(e, __shfl_xor_sync(0xffffffffu, e, o));
    if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<uint32_t*>(&s_eps), __float_as_uint(e));  // e >= 0: bit order == value order
  }
  __syncthreads();
  const float eps_obs = s_eps;
  if (4.0 * (double)eps_obs > P.tol_safe) bad |= 8;
  if (threadIdx.x == 0) { s_kept = 0; s_border = 0; }
  __syncthreads();
  if (!bad) {
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
      double v = P.mi64[i];
      if (fabs(v - thr) <= P.tol_border) atomicAdd(&s_border, 1u);
      if (v >= thr) {
        unsigned long long o = atomicAdd(P.kept_count, 1ull);
        atomicAdd(&s_kept, 1u);
        if (o < P.kept_cap) {
          int il = P.cand[i].il, jl = P.cand[i].jl;
          P.kept_key[o] = ((uint64_t)P.block << 36) | pair_rank(il, jl, P.nf, P.nt, P.diag);
          P.kept_gi[o] = P.from_idx[il];
          P.kept_gj[o] = P.to_idx[jl];
          P.kept_mi[o] = v;
        } else {
          *P.kept_overflow = 1;
        }
      }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    // chain: a later block starts collecting at 0.9 x this block's threshold; after a failure fall back hard
    if (!P.emit_all) {
      float tc = __uint_as_float(*P.tcand_bits);
      float nxt = bad ? 0.25f * tc : 0.9f * (float)v_lo;
      if (!(nxt > 0.f)) nxt = 0.f;
      *P.chain_bits = __float_as_uint(nxt);
    }
    BlockResult r;
    r.thr = thr; r.v_lo = v_lo; r.n_cand = raw; r.n_kept = s_kept; r.n_border = s_border; r.bad = bad;
    r.eps_obs = eps_obs; r.pad = 0;
    *P.result = r;
  }
}

// ------------------------------------------------------------------------------------------------
// Link materialisation.
struct ColInfo {  // per local column jl
  int32_t a0, a1, b0, b1;
  uint32_t baseU, baseL;
};

__device__ __forceinline__ int32_t circ_len_i32(int32_t p1, int32_t p2, int64_t g) {
  int64_t d = (int64_t)p1 - (int64_t)p2;
  if (d < 0) d = -d;
  d %= g;
  int64_t e = g - d;
  return (int32_t)(d < e ? d : e);
}

struct SrMatParams {
  const ColInfo* col;
  const int32_t* from_idx;
  const int32_t* to_idx;
  const int32_t* pos;
  const int32_t* paint;
  const float* sr_mi;  // block's slots
  int32_t nf, nt, diag, block;
  int64_t g;
  int32_t *o_pos1, *o_pos2, *o_c1, *o_c2, *o_len, *o_blk;  // already offset to the block's base
  double* o_mi;
};

__global__ void mi_sr_materialize_kernel(SrMatParams P) {
  int jl = blockIdx.x;
  if (jl >= P.nt) return;
  ColInfo c = P.col[jl];
  int gj = P.to_idx[jl];
  int32_t p1 = P.pos[gj], c1 = P.paint[gj];
  // walk the column's short-range rows in ascending order: interval A then interval B, skipping il == jl,
  // rows < jl go to the upper part (off-diagonal blocks only), rows > jl to the lower part
  int la = c.a1 - c.a0, lb = c.b1 - c.b0;
  int bj = min(max(jl + 1 - c.a0, 0), la) + min(max(jl + 1 - c.b0, 0), lb);  // SR rows <= jl
  int bjm = min(max(jl - c.a0, 0), la) + min(max(jl - c.b0, 0), lb);          // SR rows < jl
  for (int k = threadIdx.x; k < la + lb; k += blockDim.x) {
    int il = k < la ? c.a0 + k : c.b0 + (k - la);
    if (il == jl) continue;
    int64_t slot;
    if (il < jl) {
      if (P.diag) continue;
      slot = (int64_t)c.baseU + k;
    } else {
      slot = (int64_t)c.baseL + (k - bj);
    }
    (void)bjm;
    int gi = P.from_idx[il];
    int32_t p2 = P.pos[gi];
    P.o_pos1[slot] = p1;
    P.o_pos2[slot] = p2;
    P.o_c1[slot] = c1;
    P.o_c2[slot] = P.paint[gi];
    P.o_len[slot] = circ_len_i32(p1, p2, P.g);
    P.o_mi[slot] = (double)P.sr_mi[slot];
    P.o_blk[slot] = P.block;
  }
}

// LDW_SCAN_SR_EXACT: fp64 MI, in the reference's own arithmetic (refine_pair), of every short-range link of a block,
// written over the fp32-derived values mi_sr_materialize_kernel left in the link column.  Same walk over a column's
// short-range rows as that kernel (one CTA per column), one warp per link.
__global__ void __launch_bounds__(32 * REFINE_WARPS) mi_sr_exact_kernel(SrMatParams P, RefineParams R) {
  __shared__ double acc_s[REFINE_WARPS][32 * 25];
  const int jl = blockIdx.x;
  if (jl >= P.nt) return;
  const ColInfo c = P.col[jl];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double* acc = acc_s[warp];
  refine_scratch_clear(acc, lane);
  const int la = c.a1 - c.a0, lb = c.b1 - c.b0;
  const int bj = min(max(jl + 1 - c.a0, 0), la) + min(max(jl + 1 - c.b0, 0), lb);  // SR rows <= jl
  for (int k = warp; k < la + lb; k += REFINE_WARPS) {  // k is warp-uniform: refine_pair synchronises the warp
    const int il = k < la ? c.a0 + k : c.b0 + (k - la);
    if (il == jl) continue;
    int64_t slot;
    if (il < jl) {
      if (P.diag) continue;
      slot = (int64_t)c.baseU + k;
    } else {
      slot = (int64_t)c.baseL + (k - bj);
    }
    const double v = refine_pair(R, il, jl, lane, acc);
    if (lane == 0) P.o_mi[slot] = v;
  }
}

__global__ void mi_lr_materialize_kernel(const uint32_t* __restrict__ order, const uint64_t* __restrict__ keys_sorted,
                                         const int32_t* __restrict__ gi, const int32_t* __restrict__ gj,
                                         const double* __restrict__ mi, const int32_t* __restrict__ pos,
                                         const int32_t* __restrict__ paint, int64_t n, int64_t g, int32_t* o_pos1,
                                         int32_t* o_pos2, int32_t* o_c1, int32_t* o_c2, int32_t* o_len, double* o_mi,
                                         int32_t* o_blk) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t src = order[i];
  int a = gi[src], b = gj[src];
  int32_t p2 = pos[a], p1 = pos[b];
  o_pos1[i] = p1;
  o_pos2[i] = p2;
  o_c1[i] = paint[b];
  o_c2[i] = paint[a];
  o_len[i] = circ_len_i32(p1, p2, g);
  o_mi[i] = mi[src];
  o_blk[i] = (int32_t)(keys_sorted[i] >> 36);
}

// counters the host needs after the last block -> pinned host memory
__global__ void publish_kernel(const unsigned long long* kept_count, const uint32_t* state, unsigned long long* out) {
  out[0] = *kept_count;
  out[1] = state[3];
}

__global__ void iota_u32_kernel(uint32_t* p, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = (uint32_t)i;
}

__global__ void f32_to_f64_kernel(const float* __restrict__ in, int64_t n, double* out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (double)in[i];
}

}  // namespace ldw
