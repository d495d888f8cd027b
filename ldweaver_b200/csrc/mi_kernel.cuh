// The weighted pairwise-MI scan kernel (sm_100a).
//
// What it replaces (reference, per make_blocks block): the ten sqrt(w)-weighted dense allele sub-matrices
// (R/computePairwiseMI.R:238-256), the 25 calls of computeMI_Sprase (:270-298, :390-396: one dense x sparse product
// and five rank-1 nf x nt temporaries each) with their .fastHadamard loop (src/computeMI.cpp:11-21), and the pair
// enumeration / len / sr-lr split (:306-344).
//
// How.  The weighted joint allele counts  c_ij^ab = sum_s w_s [code(i,s)=a][code(j,s)=b]  are an integer GEMM:
// weights are fixed-point (28 bits below the largest weight) split into two 14-bit halves h = 255 a - b with byte
// digits a, b; each half is accumulated exactly in an int32 TMEM accumulator by two K-passes of kind::i8 UMMA over
// the SAME one-hot operand (bytes 0xFF): an unsigned pass (x255, digit a) and a signed pass (x-1, digit b).  Only the r-1 non-complement allele planes of a site enter the GEMM; the remaining
// counts follow from the exact integer marginals (sum_b c^ab = p^a).  SNPs are grouped by plane count so a tile is
// 2 x 128 row SNPs x NJ column SNPs with uniform (PA, PB), computed by a PAIR of CTAs with cta_group::2 MMAs (M = 256: each
// CTA stages its 128 rows and half of the columns and owns the accumulators of its rows).  Per CTA, sixteen epilogue warps
// (4 column groups x 4 TMEM lane quarters)
// read the accumulators straight out of TMEM (thread = row SNP), rebuild the (PA+1)x(PB+1) table, evaluate
//     MI = sum_ab x/den * ln(x den / D),  x = c + 0.5,  D = (p_i^a + r_j/2)(p_j^b + r_i/2) + dQ   (dQ: quirk Q1)
// in fp32 with one MUFU.LG2 per term (two with the Q1 correction), and emit: short-range links to their final,
// position-determined output slot; long-range candidates above a monotonically rising candidate threshold.
// Only the raw one-hot planes travel from L2 to shared memory (the SM's inbound bandwidth, ~30 B/clk, is the scarce
// resource): the expander warps build the four digit-weighted copies of the column tile in place, inside the stage,
// before the MMA warp consumes it.
// Warp roles: 0 = TMA producer, 1 = MMA issuer (leader CTA of the pair only), 2..7 = expanders (2 also owns TMEM),
// 8..23 = epilogue.
#pragma once
#include "mi_types.h"
#include "umma.cuh"

namespace ldw {

constexpr int MI_EXP_WARPS = 6;
constexpr int MI_EXP_THREADS = 32 * MI_EXP_WARPS;
constexpr int MI_EPI_WARP0 = 8;
constexpr int MI_EPI_GROUPS = 4;                          // column groups; each is 4 warps (one per TMEM lane quarter)
constexpr int MI_EPI_WARPS = 4 * MI_EPI_GROUPS;
constexpr int MI_EPI_THREADS = 32 * MI_EPI_WARPS;
constexpr int MI_THREADS = 32 * (MI_EPI_WARP0 + MI_EPI_WARPS);
#define LDW_STR2(x) #x
#define LDW_STR(x) LDW_STR2(x)
// register budget (65536 per SM): control warps shrink, epilogue warps grow
#define MI_REGS_CTRL 48
#define MI_REGS_EPI 96
// the CTA's pool is what the launch allocated: MI_THREADS x (65536 / MI_THREADS rounded down to a multiple of 8)
static_assert(MI_EPI_WARP0 * 32 * MI_REGS_CTRL + MI_EPI_THREADS * MI_REGS_EPI <= MI_THREADS * ((65536 / MI_THREADS) & ~7), "register budget");
constexpr int MI_MAX_STAGES = 4;
constexpr uint32_t MI_ARR_BYTES = 128 * 128;              // one operand array slice: 128 rows x 128 K-bytes
// CTA pairs (cta_group::2): a tile is 256 row SNPs (128 per CTA of the pair) x NJ column SNPs; each CTA stages its own row
// planes and HALF of the column tile (NJ/2 columns, expanded into the four digit copies), and the pair's MMA reads the B
// operand from both shared memories -- per SM that is 3/4 of the operand reads and half of the expansion traffic of a
// one-CTA tile of the same size, which is what the kernel is bound by (shared-memory bandwidth).
// The stage region is cut per tile kind: four 48 KB stages when the kind's planes fit (PA row planes + the 4 digit
// copies of this CTA's half of the PB column planes), else three 64 KB stages, else two 96 KB stages.
constexpr uint32_t MI_STAGE_REGION = 12 * MI_ARR_BYTES;
__host__ __device__ constexpr uint32_t mi_stage_need(int pa, int pb, int njlog2) {
  return (uint32_t)pa * MI_ARR_BYTES + 4u * (uint32_t)pb * (64u << njlog2);
}
__host__ __device__ constexpr int mi_stage_geo(int pa, int pb, int njlog2) {  // 0: 4 x 48 KB, 1: 3 x 64 KB, 2: 2 x 96 KB
  return mi_stage_need(pa, pb, njlog2) <= 3 * MI_ARR_BYTES ? 0 : mi_stage_need(pa, pb, njlog2) <= 4 * MI_ARR_BYTES ? 1 : 2;
}
__host__ __device__ constexpr int mi_geo_stages(int geo) { return 4 - geo; }
__host__ __device__ constexpr uint32_t mi_geo_bytes(int geo) { return geo == 0 ? 3 * MI_ARR_BYTES : geo == 1 ? 4 * MI_ARR_BYTES : 6 * MI_ARR_BYTES; }
constexpr uint32_t MI_JREC_BYTES = 128 * sizeof(Rec);     // per j-buffer
constexpr uint32_t MI_JDYN_BYTES = 128 * sizeof(ColDyn);
// Row-side records of the tile the epilogue is about to start (Rec + RowDyn of this CTA's 128 row SNPs): ONE buffer, filled
// by the producer warp with bulk copies and released by the epilogue as soon as its warps hold their row constants in
// registers -- i.e. at the top of the tile, so the refill for the next tile runs under this tile's batches.  With the tile
// header the producer leaves beside the barriers, the epilogue never waits for global memory at the top of a tile.
constexpr uint32_t MI_IREC_BYTES = 128 * sizeof(Rec);
constexpr uint32_t MI_IDYN_BYTES = 128 * sizeof(RowDyn);
constexpr uint32_t MI_BAR_BYTES = 512;                    // mbarriers, TMEM slot, tile headers, per-warp scratch words
constexpr uint32_t MI_SMEM_BYTES = MI_STAGE_REGION + 2 * (MI_JREC_BYTES + MI_JDYN_BYTES) + MI_IREC_BYTES + MI_IDYN_BYTES + MI_BAR_BYTES + 1024;
static_assert(MI_SMEM_BYTES <= 232448, "shared memory budget (227 KB opt-in)");

__device__ __forceinline__ float lg2_fast(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t ld_volatile_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}

// columns handled per TMEM read batch: keeps the unrolled body near 32-64 MI terms (instruction cache) and the
// accumulator registers at <= 32
__host__ __device__ constexpr int mi_jc(int pa, int pb) {
  return (pa + 1) * (pb + 1) <= 4 ? 8 : (pa + 1) * (pb + 1) <= 9 ? 4 : (pa + 1) * (pb + 1) <= 12 ? 2 : 1;
}
__host__ __device__ constexpr int mi_njlog2(int pa, int pb) {
  return pa * pb == 1 ? 7 : pa * pb == 2 ? 6 : pa * pb <= 4 ? 5 : 4;
}

// Raise the long-range candidate threshold to the lower edge of the histogram bin above which at least
// `kprime` already-emitted candidates lie.  Whole warp.  The threshold only ever rises, and every pair whose
// MI was >= the threshold at the time it was evaluated has been emitted, so all pairs >= the final threshold
// are in the candidate buffer.
__device__ __noinline__ void lr_raise_threshold(const ScanParams& p, int lane) {
  constexpr int PER = MI_HIST_BINS / 32;
  uint32_t s = 0;
  for (int k = 0; k < PER; k++) s += ld_volatile_u32(p.hist + lane * PER + k);
  uint32_t suf = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t v = __shfl_down_sync(0xffffffffu, suf, o);
    if (lane + o < 32) suf += v;
  }
  unsigned m = __ballot_sync(0xffffffffu, suf >= p.kprime);
  if (m == 0) return;
  int sel = 31 - __clz(m);
  if (lane == sel) {
    uint32_t run = suf - s;
    for (int k = PER - 1; k >= 0; k--) {
      run += ld_volatile_u32(p.hist + lane * PER + k);
      if (run >= p.kprime) {
        atomicMax(p.tcand_bits, (uint32_t)(lane * PER + k) << 19);
        break;
      }
    }
  }
}

template <bool DBG>
__device__ __forceinline__ void timed_wait(uint64_t* bar, uint32_t parity, int tag, long long& acc) {
  if constexpr (DBG) {
    long long c0 = clock64();
    mbar_wait(bar, parity, tag);
    acc += clock64() - c0;
  } else {
    mbar_wait(bar, parity, tag);
  }
}

struct EpiCtx {
  int q, cg, lane, rank;
  uint32_t tflags;      // this CTA's half of the tile (TileDesc::flags / flags1)
  uint32_t tmem_base;   // lane-quarter offset already applied, column of this tile's accumulators
  uint32_t jrec_saddr;  // shared-memory byte addresses of this tile's column records
  uint32_t jdyn_saddr;
  uint32_t irec_saddr, idyn_saddr;  // ... of its row records (single buffer, see MI_IREC_BYTES)
  uint32_t rempty_saddr;            // barrier the warp arrives on once its lanes HOLD their row constants
  uint32_t scr_saddr;               // this warp's scratch word (see epi_tile)
};

__device__ __forceinline__ uint4 lds128(uint32_t saddr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(saddr));
  return v;
}

__device__ __forceinline__ uint2 lds64(uint32_t saddr) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(saddr));
  return v;
}

__device__ __forceinline__ void sts128(uint32_t saddr, uint4 v) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

__device__ __forceinline__ float rcp_fast(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// One term of the MI sum.  t: joint count PLUS the pseudocount in the fixed-point unit (x = c + 1/2 = t * kT); the
// factor kT is folded into the per-tile constants and into the final scale, so a term is I2FP + the ratio + LG2 + FMA.
//   QC = false: ra = kT den / (p_i^a + r_j/2), rb = 1 / (p_j^b + r_i/2)              -> ratio = t * ra * rb
//   QC = true : ra = (p_i^a + r_j/2) / (kT den), rb = p_j^b + r_i/2, dq = dQ / (kT den) -> ratio = t / (ra * rb + dq)
// (quirk Q1: dQ is what the reference's transposed rft adds to the denominator on off-diagonal blocks)
template <bool QC>
__device__ __forceinline__ float mi_term(float acc, uint32_t t, float ra, float rb, float dq) {
  const float x = __uint2float_rn(t);
  const float ratio = QC ? x * rcp_fast(fmaf(ra, rb, dq)) : x * (ra * rb);
  return fmaf(x, lg2_fast(ratio), acc);
}

// One row of the joint table (NB cells sharing the row constant ra).  In the Q1 form the reciprocals of the NB
// denominators are taken two at a time -- 1/d0 = d1 / (d0 d1), 1/d1 = d0 / (d0 d1) -- which trades every second
// MUFU.RCP for three FMULs: the MUFU pipe, not the issue slots, is what the epilogue waits for.
template <bool QC, int NB>
__device__ __forceinline__ float mi_row(float acc, const uint32_t (&t)[NB], float ra, const float (&rb)[NB], float dq) {
  if constexpr (!QC) {
#pragma unroll
    for (int b = 0; b < NB; b++) acc = mi_term<false>(acc, t[b], ra, rb[b], dq);
    return acc;
  } else {
    float d[NB], inv[NB];
#pragma unroll
    for (int b = 0; b < NB; b++) d[b] = fmaf(ra, rb[b], dq);
#pragma unroll
    for (int b = 0; b + 1 < NB; b += 2) {
      const float r = rcp_fast(d[b] * d[b + 1]);
      inv[b] = r * d[b + 1];
      inv[b + 1] = r * d[b];
    }
    if (NB & 1) inv[NB - 1] = rcp_fast(d[NB - 1]);
#pragma unroll
    for (int b = 0; b < NB; b++) {
      const float x = __uint2float_rn(t[b]);
      acc = fmaf(x, lg2_fast(x * inv[b]), acc);
    }
    return acc;
  }
}

// Rare path (a long-range candidate somewhere in the warp): reads its parameters straight from the kernel parameters.
__device__ __noinline__ void lr_emit(const ScanParams& p, bool em, int il, int jl, float mi, int lane) {
  const unsigned bal = __ballot_sync(0xffffffffu, em);
  if (bal == 0) return;
  const int leader = __ffs(bal) - 1;
  uint32_t base = 0;
  const uint32_t n_new = (uint32_t)__popc(bal);
  if (lane == leader) base = atomicAdd(p.cand_count, n_new);
  base = __shfl_sync(0xffffffffu, base, leader);
  if (em) {
    uint32_t idx = base + (uint32_t)__popc(bal & ((1u << lane) - 1));
    if (idx < p.cand_cap) {
      Cand cc;
      cc.il = il; cc.jl = jl; cc.mi = mi;
      p.cand[idx] = cc;
    } else {
      *p.overflow = 1;
    }
    uint32_t bits = __float_as_uint(mi);
    atomicAdd(p.hist + ((bits & 0x80000000u) ? 0u : (bits >> 19)), 1u);
  }
  if (!p.emit_all && (base / p.delta) != ((base + n_new) / p.delta)) {
    __threadfence();
    lr_raise_threshold(p, lane);
  }
}

// Short-range link: store MI at the link's final, position-determined slot of the block's output.
__device__ __noinline__ void sr_store(float* sr_out, uint4 d0, uint4 d1, int il, int jl, float mi) {
  const int a0 = (int)d0.z, a1 = (int)d0.w, b0 = (int)d1.x, b1 = (int)d1.y;
  const int la = a1 - a0, lb = b1 - b0;
  int below = min(max(il - a0, 0), la) + min(max(il - b0, 0), lb);  // short-range rows of this column before `il`
  uint32_t slot;
  if (il < jl) {
    slot = d1.z + (uint32_t)below;
  } else {
    int bj = min(max(jl + 1 - a0, 0), la) + min(max(jl + 1 - b0, 0), lb);
    slot = d1.w + (uint32_t)(below - bj);
  }
  sr_out[slot] = mi;
}

// Per-tile constants of the pair loop, all in registers (passed by value into the batch routine).
template <int RA>
struct TileRegs {
  uint32_t Ti[RA];
  float rpad[RA];
  float scale, q0, qod, rtlq, tcand;  // q0, qod, rtlq carry 1 / kT
  uint32_t mul_a, sb, jl_lim, M;
  int il, nf, nt;
  bool ragged, dense, do_lr, has_sr;
  float* sr_out;
};

// Accumulator columns of row plane a (2 PB NJ of them): [columns staged by CTA 0 | columns staged by CTA 1], each half
// [H of plane 0 .. PB-1 | L of plane 0 .. PB-1] with NJ/2 columns per plane -- the order of the B rows in the two CTAs.
template <int PA, int PB, int JC>
__device__ __forceinline__ void epi_load(uint32_t tmem_base, int NJ, int j0, uint32_t (&H)[PA][PB][JC],
                                         uint32_t (&L)[PA][PB][JC]) {
  const int NJh = NJ >> 1;
  const int half = j0 >= NJh ? 1 : 0;
  const uint32_t base = tmem_base + (uint32_t)(half * PB * NJ + (j0 - half * NJh));
#pragma unroll
  for (int a = 0; a < PA; a++)
#pragma unroll
    for (int b = 0; b < PB; b++) {
      tmem_ldn<JC>(base + (uint32_t)(a * 2 * PB * NJ + b * NJh), H[a][b]);
      tmem_ldn<JC>(base + (uint32_t)(a * 2 * PB * NJ + (PB + b) * NJh), L[a][b]);
    }
}

// The PA x PB accumulator cells of a batch as counts in the count unit, pseudocount included.
template <int PA, int PB, int JC>
__device__ __forceinline__ void epi_counts(const uint32_t (&H)[PA][PB][JC], const uint32_t (&L)[PA][PB][JC], uint32_t mul_a,
                                           uint32_t sb, uint32_t M, uint32_t (&T)[PA][PB][JC]) {
#pragma unroll
  for (int a = 0; a < PA; a++)
#pragma unroll
    for (int b = 0; b < PB; b++)
#pragma unroll
      for (int jj = 0; jj < JC; jj++) T[a][b][jj] = H[a][b][jj] * mul_a + ((L[a][b][jj] >> sb) + M);
}

// JC pairs (this thread's row SNP x JC column SNPs), evaluated in lock step: term loop outside, pair loop inside, so
// JC independent dependency chains overlap each other's MUFU / conversion latency.  T: the batch's counts (epi_counts).
template <int PA, int PB, int JC, bool QC, bool RG>
__device__ __forceinline__ void epi_batch(const ScanParams& p, const EpiCtx& c, const TileRegs<PA + 1>& k, int j0,
                                          const uint32_t (&T)[PA][PB][JC]) {
  constexpr int RB = PB + 1;
  uint32_t rpj[JC][RB];
  int jl[JC];
  float dq[JC];
#pragma unroll
  for (int jj = 0; jj < JC; jj++) {
    const uint32_t ra_ = c.jrec_saddr + (uint32_t)(j0 + jj) * (uint32_t)sizeof(Rec);
    const uint4 w1 = lds128(ra_ + (QC ? 32 : 16));  // q (Q1 form) or rp (plain form); the totals T at the last row
    uint32_t w4 = 0;                                 // q4 / rp4
    if (RB == 5) asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w4) : "r"(ra_ + (QC ? 56 : 52)));
    const uint32_t tr[5] = {w1.x, w1.y, w1.z, w1.w, w4};
#pragma unroll
    for (int b = 0; b < RB; b++) rpj[jj][b] = tr[b];
    // only .x (jl) and .y (the Q1 factor) are needed here; the short-range bounds in .z / .w are reloaded at emission
    const uint2 d0 = lds64(c.jdyn_saddr + (uint32_t)(j0 + jj) * (uint32_t)sizeof(ColDyn));
    jl[jj] = (int)d0.x;
    dq[jj] = 0.f;
    if (QC) {
      if (RG) {
        // quirk Q1, general form: rft (nt x nf) is read by the linear index of the nf x nt matrix
        float v = k.q0;
        if (k.il >= 0 && jl[jj] >= 0) {
          uint64_t lin = (uint64_t)k.il + (uint64_t)jl[jj] * (uint64_t)k.nf;
          uint32_t cdiv = (uint32_t)(lin / (uint32_t)k.nt), cmod = (uint32_t)(lin % (uint32_t)k.nt);
          v = (float)p.rfl_arr[cdiv] * (float)p.rtl_arr[cmod] * k.qod;
        }
        dq[jj] = v - k.q0;
      } else {
        dq[jj] = fmaf(k.rtlq, __uint_as_float(d0.y), -k.q0);
      }
    }
  }
  // (PA+1) x (PB+1) joint table: PA x PB cells from the accumulators, the rest by complement in the count unit
  // (floor semantics keep every row / column complement non-negative; only the corner needs a clamp).  Every cell
  // is carried as count + M (M = the pseudocount 1/2 in count units); the marginals in Rec hold their row's M's.
  float acc[JC];
  uint32_t col[JC][PB], tot[JC];
#pragma unroll
  for (int jj = 0; jj < JC; jj++) {
    acc[jj] = 0.f; tot[jj] = 0;
#pragma unroll
    for (int b = 0; b < PB; b++) col[jj][b] = 0;
  }
#pragma unroll
  for (int a = 0; a < PA; a++) {
    uint32_t row[JC][RB];
#pragma unroll
    for (int jj = 0; jj < JC; jj++) {
      uint32_t rsum = 0;
#pragma unroll
      for (int b = 0; b < PB; b++) {
        const uint32_t t = T[a][b][jj];
        rsum += t;
        col[jj][b] += t;
        row[jj][b] = t;
      }
      row[jj][PB] = k.Ti[a] - rsum;
      tot[jj] += rsum;
    }
#pragma unroll
    for (int jj = 0; jj < JC; jj++) {
      float rbv[RB];
#pragma unroll
      for (int b = 0; b < RB; b++) rbv[b] = __uint_as_float(rpj[jj][b]);
      acc[jj] = mi_row<QC, RB>(acc[jj], row[jj], k.rpad[a], rbv, dq[jj]);
    }
  }
#pragma unroll
  for (int jj = 0; jj < JC; jj++) {
    const uint4 w0 = lds128(c.jrec_saddr + (uint32_t)(j0 + jj) * (uint32_t)sizeof(Rec));  // the column totals T
    const uint32_t tj[4] = {w0.x, w0.y, w0.z, w0.w};
    uint32_t row[RB], sj = 0;
    float rbv[RB];
#pragma unroll
    for (int b = 0; b < PB; b++) { row[b] = tj[b] - col[jj][b]; sj += tj[b]; }
#pragma unroll
    for (int b = 0; b < RB; b++) rbv[b] = __uint_as_float(rpj[jj][b]);
    // every marginal carries the pseudocounts of its row / column, so the corner comes out as count + M; the count
    // itself can be slightly negative (floor semantics of the other cells): clamp it at zero.  Unsigned throughout: the
    // corner can hold up to the whole table, i.e. 2^31 count units and more (the unit is sized so that a table fits
    // 32 bits, not 31).  rest = sum_b (cell(PA, b) + M) >= 0: each of its terms is a complement, non-negative under
    // floor semantics.
    const uint32_t rest = sj - tot[jj];
    row[PB] = k.Ti[PA] >= rest ? max(k.Ti[PA] - rest, k.M) : k.M;
    acc[jj] = mi_row<QC, RB>(acc[jj], row, k.rpad[PA], rbv, dq[jj]);
  }
  // ---- classification and emission: tile-uniform branches only; the per-lane work is predicated
  float mi[JC];
#pragma unroll
  for (int jj = 0; jj < JC; jj++) mi[jj] = acc[jj] * k.scale;
  if (k.dense) {
#pragma unroll
    for (int jj = 0; jj < JC; jj++)
      if (k.il >= 0 && jl[jj] >= 0) p.dense_out[(size_t)k.il + (size_t)jl[jj] * (size_t)k.nf] = mi[jj];
    return;
  }
  bool live[JC];  // a wanted pair that is not (yet) classified short-range
#pragma unroll
  for (int jj = 0; jj < JC; jj++) live[jj] = ((uint32_t)jl[jj] < k.jl_lim) && (jl[jj] != k.il);
  if (k.has_sr) {
#pragma unroll
    for (int jj = 0; jj < JC; jj++) {
      const uint4 d0 = lds128(c.jdyn_saddr + (uint32_t)(j0 + jj) * (uint32_t)sizeof(ColDyn));
      const uint4 d1 = lds128(c.jdyn_saddr + (uint32_t)(j0 + jj) * (uint32_t)sizeof(ColDyn) + 16);
      const uint32_t la = d0.w - d0.z, lb = d1.y - d1.x;
      const bool sr = live[jj] && (((uint32_t)k.il - d0.z < la) || ((uint32_t)k.il - d1.x < lb));
      if (sr) sr_store(k.sr_out, d0, d1, k.il, jl[jj], mi[jj]);
      live[jj] = live[jj] && !sr;
    }
  }
  if (k.do_lr) {
    bool any = false;
#pragma unroll
    for (int jj = 0; jj < JC; jj++) {
      live[jj] = live[jj] && (mi[jj] >= k.tcand);
      any = any || live[jj];
    }
    if (__any_sync(0xffffffffu, any)) {
#pragma unroll
      for (int jj = 0; jj < JC; jj++) lr_emit(p, live[jj], k.il, jl[jj], mi[jj], c.lane);
    }
  }
}

// release_acc: hands the tile's accumulators back to the MMA issuer; called as soon as the last batch is in registers.
template <int PA, int PB, bool QC, bool RG, class Rel>
__device__ __forceinline__ void epi_tile(const ScanParams& p, const EpiCtx& c, Rel&& release_acc) {
  constexpr int RA = PA + 1, RB = PB + 1;
  constexpr int JC = mi_jc(PA, PB);
  constexpr int NJ = 1 << mi_njlog2(PA, PB);
  constexpr int NB = (NJ / MI_EPI_GROUPS) / JC;  // batches per warp
  static_assert(NB >= 1 && NB * JC * MI_EPI_GROUPS == NJ, "column split must be exact");
  const int row = c.q * 32 + c.lane;  // within this CTA's half of the pair's 256 row SNPs
  TileRegs<RA> k;
  k.scale = p.scale[RA - 2][RB - 2]; k.q0 = p.q0s[RA - 2][RB - 2];
  k.qod = p.qod[RA - 2][RB - 2];
  k.M = p.M;
  k.nf = p.nf; k.nt = p.nt;
  k.mul_a = 1u << p.sa; k.sb = p.sb;
  k.ragged = p.ragged != 0; k.dense = p.dense != 0;
  k.do_lr = !p.sr_only && !p.dense;
  k.has_sr = (c.tflags & TILE_HAS_SR) != 0;
  k.sr_out = p.sr_out;
  k.tcand = (k.do_lr && !p.emit_all) ? __uint_as_float(ld_volatile_u32(p.tcand_bits)) : -3.0e38f;
  uint32_t r0, r1;
  {
    const uint32_t rv = c.irec_saddr + (uint32_t)row * (uint32_t)sizeof(Rec);
    const uint4 v0 = lds128(rv), v1 = lds128(rv + (QC ? 32 : 16));
    uint4 v3 = make_uint4(0, 0, 0, 0);
    if (RA == 5) v3 = lds128(rv + 48);
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(c.idyn_saddr + (uint32_t)row * (uint32_t)sizeof(RowDyn)));
    // Release the row buffer.  The arrive must not overtake the loads above: an mbarrier arrive issued right behind
    // shared-memory loads whose results nobody has consumed yet can be performed before them, and the producer's next bulk
    // copy (async proxy) then lands under the loads -- measured: one scan in four lost long-range candidates on multi-kind
    // blocks.  So every lane first STORES a word made of what it loaded (the store cannot issue before the loads have
    // returned), the warp synchronises, and lane 0 arrives (release: ordered after the stores).
    {
      const uint32_t dep = (v0.x ^ v0.y ^ v0.z ^ v0.w ^ v1.x ^ v1.y ^ v1.z ^ v1.w ^ v3.x ^ v3.y ^ v3.z ^ r0 ^ r1);
      asm volatile("st.volatile.shared.u32 [%0], %1;" ::"r"(c.scr_saddr), "r"(dep) : "memory");
      __syncwarp();
      if (c.lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(c.rempty_saddr) : "memory");
    }
    const uint32_t tt[5] = {v0.x, v0.y, v0.z, v0.w, v3.x}, tr[5] = {v1.x, v1.y, v1.z, v1.w, QC ? v3.z : v3.y};
    const float rf = QC ? p.rp_qc[RA - 2][RB - 2] : p.rp_plain[RA - 2][RB - 2];
#pragma unroll
    for (int a = 0; a < RA; a++) {
      k.Ti[a] = tt[a];
      // Q1 form: (p + r'/2) / (kT den); plain form: kT den / (p + r'/2)
      k.rpad[a] = __uint_as_float(tr[a]) * rf;
    }
  }
  k.il = (int)r0;
  k.rtlq = __uint_as_float(r1) * k.qod;
  // validity of a pair: diagonal block -> 0 <= jl < il; otherwise 0 <= jl < nt, jl != il (quirk Q2); il must exist
  k.jl_lim = k.il < 0 ? 0u : (p.diag ? (uint32_t)k.il : (uint32_t)p.nt);

  // ---- batches of JC columns, evaluated in lock step
  const int jbeg = c.cg * (NJ / MI_EPI_GROUPS);
  uint32_t H[PA][PB][JC], L[PA][PB][JC];
#pragma unroll 1
  for (int bi = 0; bi < NB; bi++) {
    const int j0 = jbeg + bi * JC;
    epi_load<PA, PB, JC>(c.tmem_base, NJ, j0, H, L);
    tmem_ld_wait();
    if (bi + 1 == NB) release_acc();
    uint32_t T[PA][PB][JC];
    epi_counts<PA, PB, JC>(H, L, k.mul_a, k.sb, k.M, T);
    epi_batch<PA, PB, JC, QC, RG>(p, c, k, j0, T);
  }
}

template <bool QC, bool RG, class Rel>
__device__ __forceinline__ void epi_dispatch(const ScanParams& p, int pa, int pb, const EpiCtx& c, Rel&& rel) {
  switch (pa * 4 + pb - 5) {
    case 0: epi_tile<1, 1, QC, RG>(p, c, rel); break;
    case 1: epi_tile<1, 2, QC, RG>(p, c, rel); break;
    case 2: epi_tile<1, 3, QC, RG>(p, c, rel); break;
    case 3: epi_tile<1, 4, QC, RG>(p, c, rel); break;
    case 4: epi_tile<2, 1, QC, RG>(p, c, rel); break;
    case 5: epi_tile<2, 2, QC, RG>(p, c, rel); break;
    case 6: epi_tile<2, 3, QC, RG>(p, c, rel); break;
    case 7: epi_tile<2, 4, QC, RG>(p, c, rel); break;
    case 8: epi_tile<3, 1, QC, RG>(p, c, rel); break;
    case 9: epi_tile<3, 2, QC, RG>(p, c, rel); break;
    case 10: epi_tile<3, 3, QC, RG>(p, c, rel); break;
    case 11: epi_tile<3, 4, QC, RG>(p, c, rel); break;
    case 12: epi_tile<4, 1, QC, RG>(p, c, rel); break;
    case 13: epi_tile<4, 2, QC, RG>(p, c, rel); break;
    case 14: epi_tile<4, 3, QC, RG>(p, c, rel); break;
    case 15: epi_tile<4, 4, QC, RG>(p, c, rel); break;
    default: break;
  }
}

template <bool DBG>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(MI_THREADS, 1)
mi_scan_kernel(const __grid_constant__ TmapSet tm, const __grid_constant__ ScanParams p) {
  extern __shared__ uint8_t smem_raw[];
  // (the dynamic shared-memory window starts at the same offset in both CTAs of the pair, so the aligned layout is identical)
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* stage_base = smem;
  Rec* jrec = reinterpret_cast<Rec*>(smem + MI_STAGE_REGION);
  ColDyn* jdyn = reinterpret_cast<ColDyn*>(smem + MI_STAGE_REGION + 2 * MI_JREC_BYTES);
  Rec* irec = reinterpret_cast<Rec*>(smem + MI_STAGE_REGION + 2 * (MI_JREC_BYTES + MI_JDYN_BYTES));
  RowDyn* idyn = reinterpret_cast<RowDyn*>(smem + MI_STAGE_REGION + 2 * (MI_JREC_BYTES + MI_JDYN_BYTES) + MI_IREC_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + MI_STAGE_REGION + 2 * (MI_JREC_BYTES + MI_JDYN_BYTES) + MI_IREC_BYTES + MI_IDYN_BYTES);
  uint64_t* full = bars;            // [MI_MAX_STAGES]  raw planes landed (TMA), per CTA
  uint64_t* empty = bars + 4;       // [MI_MAX_STAGES]  MMAs that read the stage have completed (pair commit, both CTAs)
  uint64_t* ready = bars + 8;       // [MI_MAX_STAGES]  LEADER's copy counts the expander warps of both CTAs
  uint64_t* tfull = bars + 12;      // [2]  accumulators complete (pair commit, both CTAs)
  uint64_t* tempty = bars + 14;     // [2]  LEADER's copy counts the epilogue warps of both CTAs
  uint64_t* jfull = bars + 16;      // [2]
  uint64_t* jempty = bars + 18;     // [2]
  uint64_t* drained = bars + 20;    // all MMAs of the tiles issued so far have completed (stage-geometry switch; both CTAs)
  uint64_t* rfull = bars + 21;      // row records of the next non-null tile landed
  uint64_t* rempty = bars + 22;     // every epilogue warp holds its row constants
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 23);
  // per j-buffer tile header {PA | PB << 8 | njlog2 << 16 | this CTA's flags << 24}: written by the producer before it arms
  // jfull, so the epilogue never touches the tile list in global memory; bars + 32 ..: one scratch word per epilogue warp
  uint32_t* thdr = reinterpret_cast<uint32_t*>(bars + 24);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();  // 0 = leader: issues the pair's MMAs
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm.a);
    for (int i = 0; i < MI_MAX_STAGES; i++) {
      mbar_init(&full[i], 1); mbar_init(&empty[i], 1); mbar_init(&ready[i], 2 * MI_EXP_WARPS);
    }
    mbar_init(drained, 1);
    mbar_init(rfull, 1); mbar_init(rempty, MI_EPI_WARPS);
    for (int i = 0; i < 2; i++) {
      mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 2 * MI_EPI_WARPS);
      mbar_init(&jfull[i], 1); mbar_init(&jempty[i], MI_EPI_WARPS);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc_pair(tmem_slot, 512);
  tc_fence_before();
  cluster_sync_all();  // barriers of both CTAs initialised before any remote arrive / pair commit; also a CTA barrier
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // register budget: the control warps (0-7) give registers to the epilogue warps; setmaxnreg sits at the top of
  // each role's own branch so that ptxas allocates every role against its own budget
  const int tile0 = (int)(blockIdx.x >> 1), tstep = (int)(gridDim.x >> 1);  // one tile per CTA pair

  if (warp < MI_EPI_WARP0) {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 " LDW_STR(MI_REGS_CTRL) ";");
  if (warp == 0) {
    // ===================================================================== TMA producer (each CTA: its rows, its half of the columns)
    // Whole warp runs the loop (uniform registers), one elected lane issues the copies.
    // Stage ring: `st` walks the stages of the current geometry, bit i of `phb` is the parity of stage i's barriers
    // (every role of both CTAs walks the same sequence, so the bits agree without communication).
    int st = 0; uint32_t phb = 0; int geo = -1; uint32_t dph = 0;
    int it = 0, rit = 0;  // tiles; tiles whose half of the rows is not null (phases of the row-record buffer)
    long long w_jempty = 0, w_empty = 0, t_begin = DBG ? clock64() : 0;
    for (int t = tile0; t < p.n_tiles; t += tstep, it++) {
      const TileDesc td = p.tiles[t];
      const int PA = td.PA, PB = td.PB, NJ = 1 << td.njlog2, NJh = NJ >> 1;
      const int njidx = 7 - td.njlog2;  // NJ 128,64,32,16 -> tm.b[0..3] (boxes of NJ/2 rows)
      const int g = mi_stage_geo(PA, PB, td.njlog2);
      const int nst = mi_geo_stages(g);
      const uint32_t sbytes = mi_geo_bytes(g);
      if (g != geo) {
        // the stage region is re-cut: every stage of the old geometry must have been consumed
        if (geo >= 0) { mbar_wait(drained, dph, 12); dph ^= 1; }
        geo = g; st = 0;
      }
      // per stage: the raw planes of this CTA's PA row-tile planes and of its half of all PB column planes (the latter
      // into the first digit slot, expanded in place by the expander warps)
      {
        const uint32_t stage_tx = (uint32_t)PA * MI_ARR_BYTES + (uint32_t)(PB * NJh * 128);
        const int a_row = td.a_row0 + (int)rank * 128, b_row = td.b_row0 + (int)rank * NJh;
        for (int kb = 0; kb < p.nkb; kb++) {
          timed_wait<DBG>(&empty[st], ((phb >> st) & 1) ^ 1, 11, w_empty);
          if (elect_one()) {
            uint8_t* sb = stage_base + st * sbytes;
            mbar_arrive_expect_tx(&full[st], stage_tx);
            for (int a = 0; a < PA; a++)
              tma_load_2d(sb + a * MI_ARR_BYTES, &tm.a, &full[st], kb * 128, a_row + a * td.a_pstride);
            uint8_t* sbB = sb + PA * MI_ARR_BYTES;
            for (int b = 0; b < PB; b++)
              tma_load_2d(sbB + b * NJh * 128, &tm.b[njidx], &full[st], kb * 128, b_row + b * td.b_pstride);
          }
          __syncwarp();
          phb ^= 1u << st;
          if (++st == nst) st = 0;
        }
      }
      // column records last: only the epilogue reads them, and waiting for their buffer here (instead of before the
      // operand loads) lets the operands of this tile stream in while the epilogue is still two tiles behind
      const int jb = it & 1;
      timed_wait<DBG>(&jempty[jb], ((it >> 1) & 1) ^ 1, 10, w_jempty);
      if (elect_one()) {
        thdr[jb] = (uint32_t)PA | ((uint32_t)PB << 8) | ((uint32_t)td.njlog2 << 16) | ((uint32_t)(rank ? td.flags1 : td.flags) << 24);
        mbar_arrive_expect_tx(&jfull[jb], (uint32_t)NJ * (uint32_t)(sizeof(Rec) + sizeof(ColDyn)));
        bulk_load_1d(jrec + jb * 128, p.rec + (int64_t)(PA + 1 - 2) * p.rec_vstride + td.j_slot0, NJ * sizeof(Rec), &jfull[jb]);
        bulk_load_1d(jdyn + jb * 128, p.coldyn + td.j_dyn0, NJ * sizeof(ColDyn), &jfull[jb]);
      }
      __syncwarp();
      // row records (single buffer): free as soon as the epilogue has started the previous non-null tile.  A null half has
      // none (its slots may lie beyond the group, even beyond the arrays).
      if (!((rank ? td.flags1 : td.flags) & TILE_NULL)) {
        timed_wait<DBG>(rempty, (uint32_t)(rit & 1) ^ 1, 13, w_jempty);
        if (elect_one()) {
          mbar_arrive_expect_tx(rfull, MI_IREC_BYTES + MI_IDYN_BYTES);
          bulk_load_1d(irec, p.rec + (int64_t)(PB + 1 - 2) * p.rec_vstride + td.i_slot0 + (int)rank * 128, MI_IREC_BYTES, rfull);
          bulk_load_1d(idyn, p.rowdyn + td.i_dyn0 + (int)rank * 128, MI_IDYN_BYTES, rfull);
        }
        __syncwarp();
        rit++;
      }
    }
    if (DBG && p.dbg && lane == 0) {
      p.dbg[blockIdx.x * 16 + 0] = (unsigned long long)(clock64() - t_begin);
      p.dbg[blockIdx.x * 16 + 1] = (unsigned long long)w_jempty;
      p.dbg[blockIdx.x * 16 + 2] = (unsigned long long)w_empty;
    }
  } else if (warp == 1) {
    // ===================================================================== MMA issuer (leader CTA only)
    // The whole warp runs the loop (so addresses and descriptors live in uniform registers); one elected lane
    // issues the tcgen05 instructions for the pair.
    if (rank == 0) {
    int st = 0; uint32_t phb = 0; int geo = -1; int as = 0; uint32_t aph = 0;
    long long w_tempty = 0, w_ready = 0, t_begin = DBG ? clock64() : 0;
    const uint32_t desc_hi = (uint32_t)(make_smem_desc_sw128(0) >> 32);
    for (int t = tile0; t < p.n_tiles; t += tstep) {
      const TileDesc td = p.tiles[t];
      const int PA = td.PA, PB = td.PB, NJ = 1 << td.njlog2;
      const int g = mi_stage_geo(PA, PB, td.njlog2);
      const int nst = mi_geo_stages(g);
      const uint32_t sbytes = mi_geo_bytes(g);
      if (g != geo) { geo = g; st = 0; }
      // does this pair's next tile use another stage geometry?  Then the producers wait for `drained`.
      bool sw = false;
      if (t + tstep < p.n_tiles) {
        const TileDesc tn = p.tiles[t + tstep];
        sw = mi_stage_geo(tn.PA, tn.PB, tn.njlog2) != g;
      }
      const bool big = 2 * PA * PB * NJ > 256;
      const uint32_t ncols = (uint32_t)(2 * PB * NJ);  // [H | L] halves of all PB column planes in one MMA, NJ/2 columns from each CTA
      const uint32_t idesc_u = make_idesc_u8(256, ncols);     // A bytes 0xFF read as +255
      const uint32_t idesc_s = make_idesc_s8u8(256, ncols);   // A bytes 0xFF read as -1
      uint32_t dbase;
      if (big) {
        for (int s2 = 0; s2 < 2; s2++) {
          timed_wait<DBG>(&tempty[as], aph ^ 1, 20, w_tempty);
          if (++as == 2) { as = 0; aph ^= 1; }
        }
        dbase = tmem_base;
      } else {
        timed_wait<DBG>(&tempty[as], aph ^ 1, 21, w_tempty);
        dbase = tmem_base + as * 256;
      }
      tc_fence_after();
      {
        const uint32_t boff = (uint32_t)PA * MI_ARR_BYTES;               // B region follows the A planes
        const uint32_t b2off = boff + (uint32_t)(PB * NJ * 128);         // bH | bL follow aH | aL (2 PB NJ/2 rows of 128 B)
        for (int kb = 0; kb < p.nkb; kb++) {
          timed_wait<DBG>(&ready[st], (phb >> st) & 1, 22, w_ready);
          tc_fence_after();
          // low descriptor word of the stage base: address >> 4 | LBO (1 << 16)
          const uint32_t lo = ((smem_u32(stage_base + st * sbytes) & 0x3FFFFu) >> 4) | (1u << 16);
          if (elect_one()) {
            const uint64_t dBa = ((uint64_t)desc_hi << 32) | (lo + (boff >> 4));
            const uint64_t dBb = ((uint64_t)desc_hi << 32) | (lo + (b2off >> 4));
            const uint32_t acc0 = kb > 0 ? 1u : 0u;
            for (int a = 0; a < PA; a++) {
              const uint64_t dx = ((uint64_t)desc_hi << 32) | (lo + (uint32_t)((a * MI_ARR_BYTES) >> 4));
              const uint32_t dHL = dbase + (uint32_t)(a * 2 * PB * NJ);
              umma_i8_pair(dHL, dx, dBa, idesc_u, acc0);
              umma_i8_pair(dHL, dx, dBb, idesc_s, 1u);
#pragma unroll
              for (int kk = 1; kk < 4; kk++) {
                umma_i8_pair(dHL, dx + 2 * kk, dBa + 2 * kk, idesc_u, 1u);
                umma_i8_pair(dHL, dx + 2 * kk, dBb + 2 * kk, idesc_s, 1u);
              }
            }
            umma_commit_pair(&empty[st]);
          }
          __syncwarp();
          phb ^= 1u << st;
          if (++st == nst) st = 0;
        }
      }
      if (elect_one()) {
        if (sw) umma_commit_pair(drained);
        if (big) {
          umma_commit_pair(&tfull[0]);
          umma_commit_pair(&tfull[1]);
        } else {
          umma_commit_pair(&tfull[as]);
        }
      }
      __syncwarp();
      if (!big) {
        if (++as == 2) { as = 0; aph ^= 1; }
      }
    }
    if (DBG && p.dbg && lane == 0) {
      p.dbg[blockIdx.x * 16 + 3] = (unsigned long long)(clock64() - t_begin);
      p.dbg[blockIdx.x * 16 + 4] = (unsigned long long)w_tempty;
      p.dbg[blockIdx.x * 16 + 5] = (unsigned long long)w_ready;
    }
    }
  } else {
    // ===================================================================== operand expanders (each CTA: its half of the columns)
    // stage layout: PA row planes (raw, used as they are), then aH | aL | bH | bL digit copies of this CTA's NJ/2 columns
    // of all PB column planes (the raw one-hot Y lands in the aH slot; aL, bH, bL are written, aH = Y & digit is formed
    // in place).  Elementwise on the swizzled image; only the digit lookup needs the logical K position, i.e. the 16-byte
    // chunk index XOR (row & 7).
    const int h = (warp - 2) * 32 + lane;  // 0..191
    int st = 0; uint32_t phb = 0; int geo = -1;
    long long w_full = 0, t_begin = DBG ? clock64() : 0;
    for (int t = tile0; t < p.n_tiles; t += tstep) {
      const TileDesc td = p.tiles[t];
      const int PA = td.PA, PB = td.PB, NJh = (1 << td.njlog2) >> 1;
      const int brows = PB * NJh;
      const int g = mi_stage_geo(PA, PB, td.njlog2);
      const int nst = mi_geo_stages(g);
      const uint32_t sbytes = mi_geo_bytes(g);
      if (g != geo) { geo = g; st = 0; }
      for (int kb = 0; kb < p.nkb; kb++) {
        // this thread's digit chunks: logical chunk cl of K block kb
        const int cl = h & 7;
        const uint8_t* dg = p.dig + (int64_t)kb * 128 + cl * 16;
        const uint4 g0 = __ldg(reinterpret_cast<const uint4*>(dg));                 // aH
        const uint4 g1 = __ldg(reinterpret_cast<const uint4*>(dg + p.kpad));        // aL
        const uint4 g2 = __ldg(reinterpret_cast<const uint4*>(dg + 2 * p.kpad));    // bH
        const uint4 g3 = __ldg(reinterpret_cast<const uint4*>(dg + 3 * p.kpad));    // bL
        timed_wait<DBG>(&full[st], (phb >> st) & 1, 40, w_full);
        const uint32_t yb = smem_u32(stage_base + st * sbytes) + (uint32_t)PA * MI_ARR_BYTES;
        const uint32_t slot = (uint32_t)brows * 128u;
        for (int r = h >> 3; r < brows; r += MI_EXP_THREADS / 8) {
          const uint32_t addr = yb + (uint32_t)r * 128u + (uint32_t)((cl ^ (r & 7)) * 16);
          const uint4 y = lds128(addr);  // bytes 0x00 / 0xFF: the one-hot plane is its own select mask
          sts128(addr + slot, make_uint4(y.x & g1.x, y.y & g1.y, y.z & g1.z, y.w & g1.w));          // aL
          sts128(addr + 2 * slot, make_uint4(y.x & g2.x, y.y & g2.y, y.z & g2.z, y.w & g2.w));      // bH
          sts128(addr + 3 * slot, make_uint4(y.x & g3.x, y.y & g3.y, y.z & g3.z, y.w & g3.w));      // bL
          sts128(addr, make_uint4(y.x & g0.x, y.y & g0.y, y.z & g0.z, y.w & g0.w));                 // aH in place
        }
        fence_proxy_async_smem();  // generic-proxy writes -> visible to the tensor core (async proxy)
        __syncwarp();
        // one arrival per warp on the LEADER's barrier: the pair's MMA needs the stage of both CTAs (this CTA's row planes
        // landed with the same `full` phase as its column planes)
        if (lane == 0) mbar_arrive_cluster(&ready[st], 0);
        phb ^= 1u << st;
        if (++st == nst) st = 0;
      }
    }
    if (DBG && p.dbg && h == 0) {
      p.dbg[blockIdx.x * 16 + 12] = (unsigned long long)(clock64() - t_begin);
      p.dbg[blockIdx.x * 16 + 13] = (unsigned long long)w_full;
    }
  }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 " LDW_STR(MI_REGS_EPI) ";");
    // ===================================================================== epilogue (each CTA: its 128 rows x all NJ columns)
    EpiCtx c;
    c.q = warp & 3;
    c.cg = (warp - MI_EPI_WARP0) >> 2;
    c.lane = lane;
    c.rank = (int)rank;
    int as = 0; uint32_t aph = 0;
    int it = 0, rit = 0;
    long long w_jfull = 0, w_tfull = 0, t_begin = DBG ? clock64() : 0;
    c.irec_saddr = smem_u32(irec);
    c.idyn_saddr = smem_u32(idyn);
    c.rempty_saddr = smem_u32(rempty);
    c.scr_saddr = smem_u32(bars + 32) + (uint32_t)(warp - MI_EPI_WARP0) * 4u;
    for (int t = tile0; t < p.n_tiles; t += tstep, it++) {
      const int jb = it & 1;
      timed_wait<DBG>(&jfull[jb], (it >> 1) & 1, 30, w_jfull);
      uint32_t hdr;  // tile header from shared memory (the tile list in global memory is read by the control warps only)
      asm volatile("ld.shared.u32 %0, [%1];" : "=r"(hdr) : "r"(smem_u32(&thdr[jb])));
      const int tPA = (int)(hdr & 0xFF), tPB = (int)((hdr >> 8) & 0xFF);
      c.tflags = hdr >> 24;
      const int NJ = 1 << ((hdr >> 16) & 0xFF);
      const bool big = 2 * tPA * tPB * NJ > 256;
      if (!(c.tflags & TILE_NULL)) { timed_wait<DBG>(rfull, (uint32_t)(rit & 1), 34, w_jfull); rit++; }
      long long c1 = DBG ? clock64() : 0;
      c.jrec_saddr = smem_u32(jrec + jb * 128);
      c.jdyn_saddr = smem_u32(jdyn + jb * 128);
      if (big) {
        // both accumulator halves: wait for the two ring slots in order
        uint32_t ph0 = aph;
        mbar_wait(&tfull[as], ph0, 31);
        int as1 = as ^ 1;
        uint32_t ph1 = (as == 1) ? (aph ^ 1) : aph;
        mbar_wait(&tfull[as1], ph1, 32);
        c.tmem_base = tmem_base + ((uint32_t)(c.q * 32) << 16);
      } else {
        mbar_wait(&tfull[as], aph, 33);
        c.tmem_base = tmem_base + ((uint32_t)(c.q * 32) << 16) + as * 256;
      }
      if constexpr (DBG) w_tfull += clock64() - c1;
      tc_fence_after();
      // The accumulators belong to the pair: release them on the leader's barrier as soon as this warp holds the
      // tile's last batch in registers (its tcgen05.wait::ld has returned; the fence orders the reads before the
      // arrive), not after that batch's arithmetic -- the MMAs of the tile after next can start meanwhile.
      bool released = false;
      auto release_acc = [&]() {
        tc_fence_before();
        __syncwarp();
        if (big) {
          if (lane == 0) { mbar_arrive_cluster(&tempty[0], 0); mbar_arrive_cluster(&tempty[1], 0); }
          aph ^= 1;  // two ring slots consumed: phase flips once
        } else {
          if (lane == 0) mbar_arrive_cluster(&tempty[as], 0);
          if (++as == 2) { as = 0; aph ^= 1; }
        }
        released = true;
      };
      if (!(c.tflags & TILE_NULL)) {
        if (!p.qcorr) epi_dispatch<false, false>(p, tPA, tPB, c, release_acc);
        else if (p.ragged) epi_dispatch<true, true>(p, tPA, tPB, c, release_acc);
        else epi_dispatch<true, false>(p, tPA, tPB, c, release_acc);
      }
      if (!released) release_acc();
      __syncwarp();
      if (lane == 0) mbar_arrive(&jempty[jb]);
    }
    if (DBG && p.dbg && lane == 0 && (warp == MI_EPI_WARP0 || warp == MI_EPI_WARP0 + MI_EPI_WARPS - 1)) {
      int o = warp == MI_EPI_WARP0 ? 6 : 9;
      p.dbg[blockIdx.x * 16 + o] = (unsigned long long)(clock64() - t_begin);
      p.dbg[blockIdx.x * 16 + o + 1] = (unsigned long long)w_jfull;
      p.dbg[blockIdx.x * 16 + o + 2] = (unsigned long long)w_tfull;
    }
  }
  tc_fence_before();
  cluster_sync_all();  // neither CTA may exit (or free tensor memory) while its peer can still address it
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, 512);
  }
}

}  // namespace ldw
