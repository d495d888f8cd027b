// Hamming-distance population-structure weights on sm_100a.
//
// Replaces the body of estimate_Hamming_distance_weights (reference
// R/performPopulationStuctureCorrection.R:20-81): shared = sum_a crossprod(M_a) over the five one-hot allele
// matrices (:49-74), hdw = 1/(colSums((nsnp - shared) < thresh) + 1) (:76).
//
// Formulation (exact integers).  Per site let the observed alleles be a_0 < ... < a_{r-1}.  Because every
// (site, sequence) cell is in exactly one class, the one-hot rows of a site sum to 1 and the match indicator is
//     [code_s == code_t] = sum_{q<r-1} x_q(s) x_q(t) + (1 - z_s)(1 - z_t),   z = [code != a_{r-1}] = sum_{q<r-1} x_q
// so with cnt_s = sum_sites z_s:   dist(s,t) = nsnp - shared(s,t) = cnt_s + cnt_t - G(s,t),
//     G = sum over "planes" A[s,p] * B[t,p],   biallelic site: one plane (A = z, B = 2z);
//                                              r >= 3: planes x_0..x_{r-2} and z (A = B).
// That is an int8 GEMM with K ~= 1.3 nsnp instead of the 5 nsnp one-hot columns, bit-exact in int32.
// G runs on tcgen05 (kind::i8, TMEM accumulators, TMA-fed, 128B-swizzled K-major operands); the epilogue
// applies the strict `< thresh` test and counts neighbours per sequence straight out of TMEM.
#include "hdw.h"

#include "umma.cuh"

#include <vector>

namespace ldw {

// ------------------------------------------------------------------------------------------------
// Per-SNP allele statistics: class counts over sequences -> 5 x n table, observed-allele mask, r.
// One warp per SNP; HBM-bound (n*S bytes read once).
__global__ void snp_allele_stats_kernel(const uint8_t* __restrict__ codes, int64_t n, int64_t S, int32_t* table /*n x 5*/,
                                        uint8_t* mask, uint8_t* r) {
  int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (warp >= n) return;
  const uint8_t* row = codes + warp * S;
  int c0 = 0, c1 = 0, c2 = 0, c3 = 0, c4 = 0;
  for (int64_t s = lane; s < S; s += 32) {
    int v = row[s];
    c0 += (v == 0); c1 += (v == 1); c2 += (v == 2); c3 += (v == 3); c4 += (v >= 4);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    c0 += __shfl_xor_sync(0xffffffffu, c0, o);
    c1 += __shfl_xor_sync(0xffffffffu, c1, o);
    c2 += __shfl_xor_sync(0xffffffffu, c2, o);
    c3 += __shfl_xor_sync(0xffffffffu, c3, o);
    c4 += __shfl_xor_sync(0xffffffffu, c4, o);
  }
  if (lane == 0) {
    int32_t* t = table + warp * 5;
    t[0] = c0; t[1] = c1; t[2] = c2; t[3] = c3; t[4] = c4;
    int m = (c0 > 0) | ((c1 > 0) << 1) | ((c2 > 0) << 2) | ((c3 > 0) << 3) | ((c4 > 0) << 4);
    mask[warp] = (uint8_t)m;
    r[warp] = (uint8_t)__popc(m);
  }
}

// Single-block exclusive scan of small integer counts (n up to a few million; setup path only).
__global__ void exclusive_scan_kernel(const int32_t* __restrict__ in, int64_t n, int32_t* out, int32_t* total) {
  __shared__ int32_t part[1024];
  int t = threadIdx.x;
  int64_t chunk = (n + blockDim.x - 1) / blockDim.x;
  int64_t b = t * chunk, e = b + chunk < n ? b + chunk : n;
  int32_t s = 0;
  for (int64_t i = b; i < e; i++) s += in[i];
  part[t] = s;
  __syncthreads();
  for (int o = 1; o < (int)blockDim.x; o <<= 1) {
    int32_t v = (t >= o) ? part[t - o] : 0;
    __syncthreads();
    part[t] += v;
    __syncthreads();
  }
  int32_t run = part[t] - s;
  for (int64_t i = b; i < e; i++) {
    int32_t v = in[i];
    out[i] = run;
    run += v;
  }
  if (t == (int)blockDim.x - 1 && total) *total = part[t];
}

__global__ void hdw_plane_count_kernel(const uint8_t* __restrict__ r, int64_t n, int32_t* nplanes) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    int ri = r[i];
    nplanes[i] = ri <= 1 ? 0 : (ri == 2 ? 1 : ri);
  }
}

// plane descriptor: snp | allele<<24 | mode<<27 (0: code == allele, 1: code != allele) | w2<<28 | isz<<29
__global__ void hdw_plane_desc_kernel(const uint8_t* __restrict__ mask, const uint8_t* __restrict__ r,
                                      const int32_t* __restrict__ poff, int64_t n, uint32_t* desc) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int ri = r[i], m = mask[i];
  if (ri <= 1) return;
  int al[5], k = 0;
  for (int a = 0; a < 5; a++)
    if (m & (1 << a)) al[k++] = a;
  uint32_t base = (uint32_t)i;
  int32_t o = poff[i];
  if (ri == 2) {
    desc[o] = base | (al[0] << 24) | (0u << 27) | (1u << 28) | (1u << 29);
  } else {
    for (int q = 0; q < ri - 1; q++) desc[o + q] = base | (al[q] << 24);
    desc[o + ri - 1] = base | (al[ri - 1] << 24) | (1u << 27) | (1u << 29);
  }
}

// Pack A (0/1) and B (0/1/2) operands [S_pad x Kh] (plane index contiguous) and accumulate cnt_s.
// Block: 64 sequences x 64 planes; codes tile staged through shared memory so that both the reads
// (sequence-contiguous) and the 16-byte writes (plane-contiguous) are coalesced.
__global__ void __launch_bounds__(256) hdw_pack_kernel(const uint8_t* __restrict__ codes, int64_t n, int64_t S,
                                                       const uint32_t* __restrict__ desc, int32_t kh_real, int64_t Kh,
                                                       uint8_t* A, uint8_t* B, int32_t* cnt) {
  __shared__ uint8_t tile[64][64 + 4];  // [snp - snp_lo][seq - s0]
  __shared__ uint32_t sdesc[64];
  int64_t p0 = (int64_t)blockIdx.x * 64, s0 = (int64_t)blockIdx.y * 64;
  int t = threadIdx.x;
  if (t < 64) sdesc[t] = (p0 + t < kh_real) ? desc[p0 + t] : 0xFFFFFFFFu;
  __syncthreads();
  uint32_t snp_lo = sdesc[0] & 0xFFFFFF;
  // planes are ordered by SNP; the tile normally touches fewer than 64 SNPs (monomorphic sites own no plane
  // and could stretch the range, in which case the codes are read straight from global memory)
  uint32_t last = 0xFFFFFFFFu;
  for (int q = 63; q >= 0; q--)
    if (sdesc[q] != 0xFFFFFFFFu) { last = sdesc[q] & 0xFFFFFF; break; }
  const bool use_tile = sdesc[0] != 0xFFFFFFFFu && (last - snp_lo) < 64;
  if (use_tile) {
    for (int e = t; e < 64 * 64; e += 256) {
      int k = e >> 6, s = e & 63;
      int64_t snp = (int64_t)snp_lo + k, ss = s0 + s;
      tile[k][s] = (snp < n && ss < S) ? codes[snp * S + ss] : (uint8_t)255;
    }
  }
  __syncthreads();
  int s = t >> 2, grp = t & 3;  // 16 planes per thread
  int64_t ss = s0 + s;
  uint32_t a4[4] = {0, 0, 0, 0}, b4[4] = {0, 0, 0, 0};
  int zc = 0;
#pragma unroll
  for (int q = 0; q < 16; q++) {
    uint32_t d = sdesc[grp * 16 + q];
    uint32_t bit = 0, w = 0;
    if (d != 0xFFFFFFFFu && ss < S) {
      int c = use_tile ? tile[(d & 0xFFFFFF) - snp_lo][s] : codes[(int64_t)(d & 0xFFFFFF) * S + ss];
      int al = (d >> 24) & 7;
      bit = ((d >> 27) & 1) ? (c != al) : (c == al);
      w = bit << ((d >> 28) & 1);
      zc += bit & ((d >> 29) & 1);
    }
    a4[q >> 2] |= bit << (8 * (q & 3));
    b4[q >> 2] |= w << (8 * (q & 3));
  }
  int64_t off = ss * Kh + p0 + grp * 16;
  // rows beyond S (padding up to S_pad) are written as zeros
  *reinterpret_cast<uint4*>(A + off) = make_uint4(a4[0], a4[1], a4[2], a4[3]);
  *reinterpret_cast<uint4*>(B + off) = make_uint4(b4[0], b4[1], b4[2], b4[3]);
  // reduce zc over the 4 threads of a sequence, one atomic per (block, sequence)
  zc += __shfl_xor_sync(0xffffffffu, zc, 1);
  zc += __shfl_xor_sync(0xffffffffu, zc, 2);
  if (grp == 0 && ss < S && zc) atomicAdd(&cnt[ss], zc);
}

// ------------------------------------------------------------------------------------------------
// The GEMM.  Persistent, warp-specialised: warp 0 = TMA producer, warp 1 = MMA issuer (+TMEM owner),
// warps 2..5 = epilogue (TMEM lane quarter = warp_idx % 4).
constexpr int HDW_BM = 128, HDW_BN = 256, HDW_BK = 128;  // BK in bytes == int8 elements
constexpr int HDW_STAGES = 4;
constexpr int HDW_THREADS = 192;
constexpr uint32_t HDW_STAGE_A = HDW_BM * HDW_BK, HDW_STAGE_B = HDW_BN * HDW_BK;
constexpr uint32_t HDW_SMEM = HDW_STAGES * (HDW_STAGE_A + HDW_STAGE_B) + 1024 /*align*/ + 256 /*barriers*/ + 2 * HDW_BN * 4;

struct HdwGemmParams {
  int32_t S;         // real sequences
  int32_t tiles_m, tiles_n, ksplit, nkb;  // nkb = Kh / 128
  int32_t thresh;
  int32_t fused;     // 1: count in the epilogue; 0: accumulate G^T into g (ld = ldg)
  int32_t ldg;
  const int32_t* cnt_z;  // per-sequence z counts
  int32_t* neigh;        // per-sequence neighbour counts (fused mode)
  int32_t* g;            // [t * ldg + s] partial G (non-fused mode)
  // G is symmetric: only tiles that hold at least one pair s <= t are computed (the upper triangle of the tile grid),
  // and in multi-GPU runs each rank takes every n_parts-th of them.  tile_list[k] = (tm, tn) of this launch's tiles.
  const int2* tile_list;
  int32_t n_tiles;
};

__global__ void __launch_bounds__(HDW_THREADS, 1)
hdw_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, HdwGemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = smem;
  uint8_t* sB = smem + HDW_STAGES * HDW_STAGE_A;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + HDW_STAGES * (HDW_STAGE_A + HDW_STAGE_B));
  uint64_t* full = bars;
  uint64_t* empty = bars + HDW_STAGES;
  uint64_t* tfull = bars + 2 * HDW_STAGES;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  int32_t* s_cnt = reinterpret_cast<int32_t*>(bars + 32);  // z counts of the tile's column sequences, reloaded per tile
  int32_t* s_col = s_cnt + HDW_BN;                         // neighbours found for the column sequences (pairs s < t)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int i = 0; i < HDW_STAGES; i++) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < 2; i++) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 128); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int total_work = p.n_tiles * p.ksplit;
  const int kb_per = (p.nkb + p.ksplit - 1) / p.ksplit;

  if (warp == 0) {
    if (lane == 0) {
      int st = 0; uint32_t ph = 0;
      for (int w = blockIdx.x; w < total_work; w += gridDim.x) {
        int ks = w % p.ksplit;
        const int2 tl = p.tile_list[w / p.ksplit];
        int tm = tl.x, tn = tl.y;
        int kb0 = ks * kb_per, kb1 = min(p.nkb, kb0 + kb_per);
        for (int kb = kb0; kb < kb1; kb++) {
          mbar_wait(&empty[st], ph ^ 1, 1);
          mbar_arrive_expect_tx(&full[st], HDW_STAGE_A + HDW_STAGE_B);
          tma_load_2d(sA + st * HDW_STAGE_A, &tmA, &full[st], kb * HDW_BK, tm * HDW_BM);
          tma_load_2d(sB + st * HDW_STAGE_B, &tmB, &full[st], kb * HDW_BK, tn * HDW_BN);
          if (++st == HDW_STAGES) { st = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = make_idesc_u8(HDW_BM, HDW_BN);
      int st = 0; uint32_t ph = 0; int as = 0; uint32_t aph = 0;
      for (int w = blockIdx.x; w < total_work; w += gridDim.x) {
        int ks = w % p.ksplit;
        int kb0 = ks * kb_per, kb1 = min(p.nkb, kb0 + kb_per);
        mbar_wait(&tempty[as], aph ^ 1, 2);
        tc_fence_after();
        uint32_t d = tmem_base + as * HDW_BN;
        for (int kb = kb0; kb < kb1; kb++) {
          mbar_wait(&full[st], ph, 3);
          tc_fence_after();
          uint64_t da = make_smem_desc_sw128(smem_u32(sA + st * HDW_STAGE_A));
          uint64_t db = make_smem_desc_sw128(smem_u32(sB + st * HDW_STAGE_B));
#pragma unroll
          for (int k = 0; k < HDW_BK / 32; k++)
            umma_i8(d, da + 2 * k, db + 2 * k, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          umma_commit(&empty[st]);
          if (++st == HDW_STAGES) { st = 0; ph ^= 1; }
        }
        umma_commit(&tfull[as]);
        if (++as == 2) { as = 0; aph ^= 1; }
      }
    }
  } else {
    const int q = warp & 3;            // TMEM lane quarter this warp may read
    const int et = (warp - 2) * 32 + lane;  // 0..127 linear epilogue thread id
    int as = 0; uint32_t aph = 0;
    for (int w = blockIdx.x; w < total_work; w += gridDim.x) {
      int ks = w % p.ksplit;
      const int2 tl = p.tile_list[w / p.ksplit];
      int tm = tl.x, tn = tl.y;
      int kb0 = ks * kb_per;
      bool has_k = kb0 < p.nkb;
      // stage the column sequences' z counts
      asm volatile("bar.sync 1, 128;");
      for (int c = et; c < HDW_BN; c += 128) {
        int t = tn * HDW_BN + c;
        s_cnt[c] = (t < p.S) ? p.cnt_z[t] : 0;
        s_col[c] = 0;
      }
      asm volatile("bar.sync 1, 128;");
      mbar_wait(&tfull[as], aph, 4);
      tc_fence_after();
      const int s = tm * HDW_BM + q * 32 + lane;
      const int cs = (s < p.S) ? p.cnt_z[s] : 0;
      int local = 0;
      const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16) + as * HDW_BN;
#pragma unroll 1
      for (int c0 = 0; c0 < HDW_BN; c0 += 32) {
        uint32_t v[32];
        tmem_ld16(trow + c0, v);
        tmem_ld16(trow + c0 + 16, v + 16);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; j++) {
          int t = tn * HDW_BN + c0 + j;
          int gval = has_k ? (int)v[j] : 0;
          if (p.fused) {
            // dist(s,t) == dist(t,s): a pair s < t counts for both sequences, the diagonal once, s > t is the mirror
            // image of a pair another (or this) tile counts
            int dist = cs + s_cnt[c0 + j] - gval;
            const bool near = (t < p.S && s < p.S && dist < p.thresh);
            local += (near && s <= t) ? 1 : 0;
            const unsigned m = __ballot_sync(0xffffffffu, near && s < t);
            if (m && lane == 0) atomicAdd(&s_col[c0 + j], __popc(m));
          } else if (s < p.S && t < p.S && gval != 0) {
            atomicAdd(&p.g[(int64_t)t * p.ldg + s], gval);
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&tempty[as]);
      if (p.fused) {
        if (s < p.S && local) atomicAdd(&p.neigh[s], local);
        asm volatile("bar.sync 1, 128;");
        for (int c = et; c < HDW_BN; c += 128) {
          const int t = tn * HDW_BN + c, v = s_col[c];
          if (v && t < p.S) atomicAdd(&p.neigh[t], v);
        }
      }
      if (++as == 2) { as = 0; aph ^= 1; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// Non-fused finish: neighbour counts from G^T.
__global__ void hdw_finish_kernel(const int32_t* __restrict__ g, int32_t ldg, const int32_t* __restrict__ cnt_z, int32_t S,
                                  int32_t thresh, int32_t* neigh, int32_t* dist_out /*S x S col-major or null*/) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  int cs = cnt_z[s], c = 0;
  for (int t = 0; t < S; t++) {
    // only tiles of the upper triangle were accumulated: G(s,t) for s <= t sits at [t][s], else at [s][t]
    int d = cs + cnt_z[t] - (s <= t ? g[(int64_t)t * ldg + s] : g[(int64_t)s * ldg + t]);
    c += d < thresh;
    if (dist_out) dist_out[(int64_t)t * S + s] = d;
  }
  neigh[s] = c;
}

__global__ void hdw_weights_kernel(const int32_t* __restrict__ neigh, int32_t S, double* w) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s < S) w[s] = 1.0 / (double)(neigh[s] + 1);
}

// Largest byte of a buffer (input validation of a device-resident class matrix), atomicMax into *out.
__global__ void max_byte_kernel(const uint8_t* __restrict__ p, int64_t n, uint32_t* out) {
  uint32_t m = 0;
  const int64_t n16 = n / 16;
  const uint4* q = reinterpret_cast<const uint4*>(p);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (int64_t)gridDim.x * blockDim.x) {
    const uint4 v = __ldg(q + i);
    m = __vmaxu4(m, __vmaxu4(__vmaxu4(v.x, v.y), __vmaxu4(v.z, v.w)));
  }
  for (int64_t i = n16 * 16 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) m = __vmaxu4(m, (uint32_t)p[i]);
  m = max(max(m & 0xFFu, (m >> 8) & 0xFFu), max((m >> 16) & 0xFFu, m >> 24));
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}

int max_byte_device(cudaStream_t st, const uint8_t* d, int64_t n, uint32_t* out) {
  *out = 0;
  if (n <= 0) return 0;
  DevBuf d_max;
  LDW_TRY(d_max.alloc(4));
  LDW_CUDA(cudaMemsetAsync(d_max.p, 0, 4, st));
  max_byte_kernel<<<148 * 8, 256, 0, st>>>(d, n, d_max.as<uint32_t>());
  LDW_CUDA(cudaGetLastError());
  LDW_CUDA(cudaMemcpyAsync(out, d_max.p, 4, cudaMemcpyDeviceToHost, st));
  LDW_CUDA(cudaStreamSynchronize(st));
  return 0;
}

// ------------------------------------------------------------------------------------------------
int snp_allele_stats(cudaStream_t st, const uint8_t* d_codes, int64_t n, int64_t S, int32_t* d_table, uint8_t* d_mask,
                     uint8_t* d_r) {
  if (n == 0) return 0;
  int wpb = 8;
  snp_allele_stats_kernel<<<(unsigned)((n + wpb - 1) / wpb), wpb * 32, 0, st>>>(d_codes, n, S, d_table, d_mask, d_r);
  LDW_CUDA(cudaGetLastError());
  return 0;
}

int exclusive_scan_i32(cudaStream_t st, const int32_t* d_in, int64_t n, int32_t* d_out, int32_t* d_total) {
  exclusive_scan_kernel<<<1, 1024, 0, st>>>(d_in, n, d_out, d_total);
  LDW_CUDA(cudaGetLastError());
  return 0;
}

int hdw_device(cudaStream_t st, const uint8_t* d_codes, int64_t n, int64_t S, int32_t thresh, int32_t* d_neigh,
               double* d_hdw, int32_t* d_dist, int num_sms, const HdwShard* shard) {
  if (S <= 0 || n <= 0) return set_error(LDW_ERR_ARG, "hdw: empty input (nsnp=%lld nseq=%lld)", (long long)n, (long long)S);
  if (n >= (1 << 24)) return set_error(LDW_ERR_UNSUPPORTED, "hdw: nsnp >= 2^24 not supported");
  DevBuf table, mask, r, npl, poff, total, desc, A, B, cntz, g, tiles_dev;
  LDW_TRY(table.alloc(n * 5 * 4));
  LDW_TRY(mask.alloc(n));
  LDW_TRY(r.alloc(n));
  LDW_TRY(npl.alloc(n * 4));
  LDW_TRY(poff.alloc(n * 4));
  LDW_TRY(total.alloc(4));
  LDW_TRY(snp_allele_stats(st, d_codes, n, S, table.as<int32_t>(), mask.as<uint8_t>(), r.as<uint8_t>()));
  hdw_plane_count_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(r.as<uint8_t>(), n, npl.as<int32_t>());
  LDW_TRY(exclusive_scan_i32(st, npl.as<int32_t>(), n, poff.as<int32_t>(), total.as<int32_t>()));
  int32_t kh_real = 0;
  LDW_CUDA(cudaMemcpyAsync(&kh_real, total.p, 4, cudaMemcpyDeviceToHost, st));
  LDW_CUDA(cudaStreamSynchronize(st));
  int64_t Kh = round_up(kh_real > 0 ? kh_real : 1, HDW_BK);
  int64_t S_pad = round_up(S, HDW_BN);
  LDW_TRY(desc.alloc((size_t)Kh * 4));
  LDW_TRY(A.alloc((size_t)S_pad * Kh));
  LDW_TRY(B.alloc((size_t)S_pad * Kh));
  LDW_TRY(cntz.alloc((size_t)S_pad * 4));
  LDW_CUDA(cudaMemsetAsync(cntz.p, 0, (size_t)S_pad * 4, st));
  LDW_CUDA(cudaMemsetAsync(d_neigh, 0, (size_t)S * 4, st));
  hdw_plane_desc_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(mask.as<uint8_t>(), r.as<uint8_t>(), poff.as<int32_t>(), n,
                                                                     desc.as<uint32_t>());
  {
    dim3 grid((unsigned)(Kh / 64), (unsigned)(S_pad / 64));
    hdw_pack_kernel<<<grid, 256, 0, st>>>(d_codes, n, S, desc.as<uint32_t>(), kh_real, Kh, A.as<uint8_t>(), B.as<uint8_t>(),
                                          cntz.as<int32_t>());
  }
  LDW_CUDA(cudaGetLastError());

  CUtensorMap tmA, tmB;
  LDW_TRY(make_tmap_u8_sw128(&tmA, A.p, (uint64_t)S_pad, (uint64_t)Kh, HDW_BM));
  LDW_TRY(make_tmap_u8_sw128(&tmB, B.p, (uint64_t)S_pad, (uint64_t)Kh, HDW_BN));

  HdwGemmParams p;
  memset(&p, 0, sizeof(p));
  p.S = (int32_t)S;
  p.tiles_m = (int32_t)((S + HDW_BM - 1) / HDW_BM);
  p.tiles_n = (int32_t)((S + HDW_BN - 1) / HDW_BN);
  p.nkb = (int32_t)(Kh / HDW_BK);
  // Upper triangle of the tile grid: tile (tm, tn) holds a pair s <= t iff its first row does not lie below its last column.
  // Listed supertile by supertile (16 row tiles x 8 column tiles = 2048 x 2048 sequences, about one wave of CTAs): the
  // CTAs that run at the same time then share 16 A tiles and 8 B tiles through L2 instead of streaming ~80 different A
  // tiles (every tile re-reads its operands over the whole K: the kernel is HBM-bound without that reuse).
  std::vector<int2> tri;
  constexpr int SUP_M = 16, SUP_N = 8;
  for (int sn = 0; sn < p.tiles_n; sn += SUP_N)
    for (int sm = 0; sm < p.tiles_m; sm += SUP_M)
      for (int tn = sn; tn < std::min(sn + SUP_N, p.tiles_n); tn++)
        for (int tm = sm; tm < std::min(sm + SUP_M, p.tiles_m); tm++)
          if ((int64_t)tm * HDW_BM <= (int64_t)tn * HDW_BN + HDW_BN - 1) tri.push_back(make_int2(tm, tn));
  // Multi-GPU (SURVEY 8e row 2): when every rank still gets at least a wave of whole-K tiles, the triangle's tiles are
  // dealt round-robin, each rank counts the neighbours its tiles reveal and the partial counts are summed across ranks
  // (the `allreduce` callback: ncclAllReduce).  Smaller problems are computed whole on every rank -- identical results,
  // no collective -- because split-K (which they need to fill the SMs) leaves no per-rank share to count from.
  // The decision depends on S, the rank count and the SM count only, so all ranks of a homogeneous box agree.
  int n_parts = 1, part = 0;
  if (shard && shard->n_parts > 1 && d_dist == nullptr &&
      (shard->force || (int64_t)tri.size() >= (int64_t)shard->n_parts * num_sms)) {
    n_parts = shard->n_parts;
    part = shard->part;
  }
  std::vector<int2> mine;
  for (size_t k = 0; k < tri.size(); k++)
    if ((int)(k % (size_t)n_parts) == part) mine.push_back(tri[k]);
  const int tiles = (int)mine.size();
  int ks = tiles > 0 ? (2 * num_sms) / tiles : 1;
  if (n_parts > 1) ks = 1;
  if (ks < 1) ks = 1;
  if (ks > p.nkb) ks = p.nkb;
  // every split must own at least one k-block
  while (ks > 1 && (int64_t)(ks - 1) * ((p.nkb + ks - 1) / ks) >= p.nkb) ks--;
  p.ksplit = ks;
  p.thresh = thresh;
  p.fused = (ks == 1 && d_dist == nullptr) ? 1 : 0;
  p.ldg = (int32_t)S_pad;
  p.cnt_z = cntz.as<int32_t>();
  p.neigh = d_neigh;
  p.g = nullptr;
  p.n_tiles = tiles;
  LDW_TRY(tiles_dev.alloc(std::max<size_t>(mine.size(), 1) * sizeof(int2)));
  if (tiles) LDW_CUDA(cudaMemcpyAsync(tiles_dev.p, mine.data(), mine.size() * sizeof(int2), cudaMemcpyHostToDevice, st));
  p.tile_list = tiles_dev.as<int2>();
  if (!p.fused) {
    LDW_TRY(g.alloc((size_t)S_pad * S_pad * 4));
    LDW_CUDA(cudaMemsetAsync(g.p, 0, (size_t)S_pad * S_pad * 4, st));
    p.g = g.as<int32_t>();
  }
  LDW_CUDA(cudaFuncSetAttribute(hdw_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, HDW_SMEM));
  if (tiles > 0) {
    int grid = tiles * ks < num_sms ? tiles * ks : num_sms;
    hdw_gemm_kernel<<<grid, HDW_THREADS, HDW_SMEM, st>>>(tmA, tmB, p);
    LDW_CUDA(cudaGetLastError());
  }
  if (!p.fused) {
    hdw_finish_kernel<<<(unsigned)((S + 127) / 128), 128, 0, st>>>(g.as<int32_t>(), p.ldg, cntz.as<int32_t>(), (int32_t)S, thresh,
                                                                   d_neigh, d_dist);
    LDW_CUDA(cudaGetLastError());
  }
  if (n_parts > 1) {
    if (!shard->allreduce) return set_error(LDW_ERR_INTERNAL, "hdw: sharded run without a reduction");
    LDW_TRY(shard->allreduce(d_neigh, S, st));  // sum of the ranks' partial neighbour counts, in place, on every rank
  }
  if (shard && shard->sharded_out) *shard->sharded_out = n_parts > 1 ? 1 : 0;
  hdw_weights_kernel<<<(unsigned)((S + 127) / 128), 128, 0, st>>>(d_neigh, (int32_t)S, d_hdw);
  LDW_CUDA(cudaGetLastError());
  LDW_CUDA(cudaStreamSynchronize(st));
  return 0;
}

}  // namespace ldw
