// score_topk_f16.cu — full-ranking top-k: fp16-accumulator tcgen05 FILTER + exact fp32 re-score.
//
// north_star (3): getUsersRating (abstract at LightGCN_SPEX/code/utility1/model.py:14-15; the only
// user x all-items matmul of the reference is NGCF_SPEX/code/utility/batch_test.py:158) followed
// by top-k.  Round 1's kernel (score_topk_tc.cu: bf16 operands, fp32 accumulators) is bound by the
// TMEM -> register drain, not by the MMA pipe: with K = 64 every accumulator element is read after
// 64 MACs and a tcgen05.ld.32x32b.x32 (32 fp32 columns) costs ~190 cycles under MMA load.
// Measured for this round (profiles/microbench/f16acc.cu): the same instruction with .pack::16b
// delivers 64 fp16-accumulator columns in ~200 cycles and x64.pack::16b a whole 128-column tile
// row quarter in ~300 cycles, i.e. 2.3 cycles per column instead of 5.8.  So:
//
//   * operands are fp16 (RN of x * 2^s, s a per-table power of two chosen by spex_pack_f16 so that
//     every row norm is below 2^7: no overflow, |score| < 2^14), same UMMA no-swizzle K-major
//     canonical layout as before (8-row x 16-byte core matrices, one bulk copy per tile);
//   * the tensor core accumulates in fp16 (tcgen05.mma.kind::f16, c_format = F16).  That result
//     `a` is only a FILTER: |a - s| <= eps_u = (DK/16) 2^-11 |u| Vmax + 2^-10 for the exact score s
//     of the same fp16 operands.  Each of the DK/16 K=16 MMAs of a tile reads the fp16 accumulator
//     and writes it back rounded to fp16; the partial sum it rounds is bounded by sum|u_d v_d| <=
//     |u||v|, so with round-to-nearest (unit roundoff 2^-11) each step adds at most 2^-11 |u||v|:
//     2^-9 at D = 64 (4 steps), 2^-8 at D = 128 (8 steps); 2^-10 covers fp16 subnormals.  The bound
//     is nearly reached: tests/test_gpu_ranking_edges.py builds items that lose (DK/16 - 0.6) 2^-11
//     |u| Vmax (a margin of 2^-9 dropped them at D = 128).  Truncation would need twice the margin.
//     One random tile shows ~2^-14 |u||v| (profiles/microbench/f16acc_b200.txt);
//   * an epilogue thread owns one user row: ONE tcgen05.ld.x64.pack::16b brings the 128 scores of
//     its row into 64 registers, the accumulator buffer is handed back to the MMA warp at once,
//     63 HMNMX2 + one compare + one vote reject the tile against the row's threshold thr.
//     (Two software-pipelined variants - two 64-register sets, and three 32-register sets rotating
//     over half tiles - were built and measured: 1322 / 1282 TF for the filter alone against 1430
//     for this one; the TMEM read is throughput-, not latency-bound with 8 epilogue warps per SM);
//   * survivors (a >= thr; ~k ln(m/k) (1 + some %) per row over the whole sweep) pass the merge-
//     cursor test against the user's training items and are appended, with their filter score and
//     a flag, to the row's candidate buffer in shared memory (two stores: the survivor path does no
//     global load).  A full buffer is compacted by the warp WITHOUT leaving the SM: with A = the
//     k-th largest value held, everything below A - 2 eps is provably outside the top-k and thr
//     becomes A - 2 eps.  Only when near-ties crowd the buffer, and once at the end, the flagged
//     entries are re-scored EXACTLY, 32 in parallel (fp32 FMA chain over the fp16 operands: user row
//     from the resident A tile, item row from the packed table in L2), ties by ascending item id.
//     History (profiles/r02_tf_scorer.md): re-scoring every survivor at once cost 46 % of the
//     kernel (770 TF), re-scoring at every compaction 32 % (941 TF), compaction on filter values
//     966 TF; the filter alone runs at 1430 TF, the MMA side alone at 1560.
//     The filter can only let extra items through, never drop one, so the output is the exact
//     top-k of the fp32 scores of the fp16 operands (tests/test_gpu_f16_scorer.py);
//   * D = 64 (4 MMAs per tile, two CTAs per SM) and D = 128 (8 MMAs, NGCF's concatenated layer
//     outputs, NGCF_SPEX/code/main_rec.py:85; one CTA per SM).
//   * warp roles as in round 1: warp 0 bulk-copy producer, warp 1 TMEM allocator + MMA issuer
//     (elect.sync, back-to-back polls), warps 2-5 epilogue (TMEM lane quarter = warp % 4).
#include "tcgen05.cuh"
#include <cuda_fp16.h>
#include <stdlib.h>

namespace spex {
namespace tf {

using namespace tcgen05;

// filter margin per unit |u| Vmax: one fp16 rounding (2^-11) per K=16 step, see the header comment
template <int DK>
constexpr float kEpsRel = (DK / 16) * (1.0f / 2048.0f);   // D = 64: 2^-9, D = 128: 2^-8
constexpr float kEpsAbs = 1.0f / 1024.0f;   // subnormal flush of tiny operands (bound 2^-11)

// tcgen05.ld 32 lanes x 128 columns of 16-bit accumulators packed two per register (column 2i in
// the low half of register i), without waiting
#define SPEX_O32(r, o)                                                                              \
  "=r"(r[o + 0]), "=r"(r[o + 1]), "=r"(r[o + 2]), "=r"(r[o + 3]), "=r"(r[o + 4]), "=r"(r[o + 5]),    \
      "=r"(r[o + 6]), "=r"(r[o + 7]), "=r"(r[o + 8]), "=r"(r[o + 9]), "=r"(r[o + 10]),              \
      "=r"(r[o + 11]), "=r"(r[o + 12]), "=r"(r[o + 13]), "=r"(r[o + 14]), "=r"(r[o + 15]),          \
      "=r"(r[o + 16]), "=r"(r[o + 17]), "=r"(r[o + 18]), "=r"(r[o + 19]), "=r"(r[o + 20]),          \
      "=r"(r[o + 21]), "=r"(r[o + 22]), "=r"(r[o + 23]), "=r"(r[o + 24]), "=r"(r[o + 25]),          \
      "=r"(r[o + 26]), "=r"(r[o + 27]), "=r"(r[o + 28]), "=r"(r[o + 29]), "=r"(r[o + 30]),          \
      "=r"(r[o + 31])
#define SPEX_IO32(r, o)                                                                             \
  "+r"(r[o + 0]), "+r"(r[o + 1]), "+r"(r[o + 2]), "+r"(r[o + 3]), "+r"(r[o + 4]), "+r"(r[o + 5]),    \
      "+r"(r[o + 6]), "+r"(r[o + 7]), "+r"(r[o + 8]), "+r"(r[o + 9]), "+r"(r[o + 10]),              \
      "+r"(r[o + 11]), "+r"(r[o + 12]), "+r"(r[o + 13]), "+r"(r[o + 14]), "+r"(r[o + 15]),          \
      "+r"(r[o + 16]), "+r"(r[o + 17]), "+r"(r[o + 18]), "+r"(r[o + 19]), "+r"(r[o + 20]),          \
      "+r"(r[o + 21]), "+r"(r[o + 22]), "+r"(r[o + 23]), "+r"(r[o + 24]), "+r"(r[o + 25]),          \
      "+r"(r[o + 26]), "+r"(r[o + 27]), "+r"(r[o + 28]), "+r"(r[o + 29]), "+r"(r[o + 30]),          \
      "+r"(r[o + 31])
// tcgen05.ld of 32 lanes x 128 columns of fp16 accumulators into 64 registers (column 2i in the low
// half of register i), without waiting
__device__ __forceinline__ void tmem_ld128h_issue(uint32_t taddr, uint32_t (&r)[64]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x64.pack::16b.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,"
      "%26,%27,%28,%29,%30,%31,%32,%33,%34,%35,%36,%37,%38,%39,%40,%41,%42,%43,%44,%45,%46,%47,%48,%49,"
      "%50,%51,%52,%53,%54,%55,%56,%57,%58,%59,%60,%61,%62,%63}, [%64];"
      : SPEX_O32(r, 0), SPEX_O32(r, 32)
      : "r"(taddr)
      : "memory");
}
// wait for the outstanding tcgen05.ld of this thread; the "+r" operands tie the loaded registers
// to the wait so that no consumer can be scheduled above it
__device__ __forceinline__ void tmem_wait64(uint32_t (&r)[64]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;" : SPEX_IO32(r, 0), SPEX_IO32(r, 32) : : "memory");
}
__device__ __forceinline__ uint32_t hmax2(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("max.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));   // HMNMX2
  return d;
}
__device__ __forceinline__ __half lo_half(uint32_t x) { return __ushort_as_half((unsigned short)(x & 0xffffu)); }
__device__ __forceinline__ __half hi_half(uint32_t x) { return __ushort_as_half((unsigned short)(x >> 16)); }

// Per-row mask cursor (shared memory; only the survivor path touches it).  Items are offered to a
// row in strictly ascending id order and the row's training items (CSR row of R) are ascending
// too, so the mask test is a merge: the cursor only moves forward.
struct MaskCursor {
  const int32_t* cur[BM];
  const int32_t* end[BM];
};

// exact score of (this row, item id): fp32 FMA chain over the fp16 operands, d = 0 .. DK-1
template <int DK>
__device__ __forceinline__ float exact_score(const uint8_t* a_row, const uint8_t* Ib, int id) {
  const uint8_t* b_row = Ib + (size_t)(id >> 3) * (16 * DK) + (size_t)(id & 7) * 16;
  float s = 0.f;
#pragma unroll
  for (int kc = 0; kc < DK / 8; ++kc) {
    const uint4 a = *reinterpret_cast<const uint4*>(a_row + kc * 128);
    const uint4 b = __ldg(reinterpret_cast<const uint4*>(b_row + kc * 128));
    const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, bw[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float2 fa = __half22float2(*reinterpret_cast<const __half2*>(&aw[q]));
      const float2 fb = __half22float2(*reinterpret_cast<const __half2*>(&bw[q]));
      s = fmaf(fa.x, fb.x, s);
      s = fmaf(fa.y, fb.y, s);
    }
  }
  return s;
}

constexpr int kApprox = (int)0x80000000;   // flag in a candidate's id: its score is still the fp16 filter value

// rank of every entry of a row's buffer under (score desc, id asc): entries travel by warp shuffle,
// every lane counts the entries that beat its own (a strict total order, so ranks are a permutation)
template <int EPL>
__device__ __forceinline__ void rank_entries(const float (&ev)[EPL], const int (&ei)[EPL], int (&rank)[EPL]) {
#pragma unroll
  for (int e = 0; e < EPL; ++e) rank[e] = 0;
#pragma unroll
  for (int e2 = 0; e2 < EPL; ++e2) {
#pragma unroll 4
    for (int jj = 0; jj < 32; ++jj) {   // kept rolled: cold code must stay small (i-cache)
      const float vj = __shfl_sync(kFull, ev[e2], jj);
      const int ij = __shfl_sync(kFull, ei[e2], jj);
#pragma unroll
      for (int e = 0; e < EPL; ++e) rank[e] += beats(vj, ij, ev[e], ei[e]) ? 1 : 0;
    }
  }
}

// The same ranks when the first `nso` entries of the buffer are already in rank order among themselves (the
// prefix a previous compaction left: entry p < nso is beaten by exactly p prefix entries): only the entries
// appended since travel by shuffle.  An old entry's rank is its position plus the new entries that beat it;
// a new entry's rank is the number of entries (old or new) that beat it, counted by one vote per slot.
template <int EPL>
__device__ __forceinline__ void rank_entries_partial(const float (&ev)[EPL], const int (&ei)[EPL], int (&rank)[EPL],
                                                     int ns, int nso, int lane) {
#pragma unroll
  for (int e = 0; e < EPL; ++e) rank[e] = (lane + 32 * e < nso) ? lane + 32 * e : 0;
#pragma unroll 1
  for (int j = nso; j < ns; ++j) {
    float sv = ev[0];
    int si = ei[0];
#pragma unroll
    for (int e = 1; e < EPL; ++e) {
      sv = ((j >> 5) == e) ? ev[e] : sv;
      si = ((j >> 5) == e) ? ei[e] : si;
    }
    const float vj = __shfl_sync(kFull, sv, j & 31);
    const int ij = __shfl_sync(kFull, si, j & 31);
    int cnt = 0;
#pragma unroll
    for (int e = 0; e < EPL; ++e) {
      const int p = lane + 32 * e;
      const bool mb = p < ns && beats(ev[e], ei[e], vj, ij);       // my entry beats entry j
      cnt += __popc(__ballot_sync(kFull, mb));
      if (p < nso && !mb) ++rank[e];                               // entry j beats my (old) entry
    }
#pragma unroll
    for (int e = 0; e < EPL; ++e)
      if (lane + 32 * e == j) rank[e] = cnt;
  }
}

// Compaction of the candidate buffers of the rows in `need` (one bit per lane = row of this warp's
// TMEM lane quarter), by the whole warp, out of line (cold code must not bloat the hot loop).
//
// Fast form (no global load): with A = the k-th largest VALUE in the buffer (filter values have
// |a - s| <= eps, exact ones 0), every entry below A - 2 eps is provably outside the top-k (k entries
// have exact scores >= A - eps, the entry's is < A - eps), so the entries with value >= A - 2 eps
// are kept as they are and the row's filter threshold becomes A - 2 eps.
// Exact form (taken when the fast form would leave fewer than 4 free slots - many near-ties - and
// in the final pass): the flagged entries are RE-SCORED EXACTLY, 32 in parallel (fp32 FMA chain over
// the fp16 operands: user row from the resident A tile, item row from the packed table in L2), the
// exact top-k is kept in sorted order and the threshold becomes (exact k-th best) - eps.
// Both thresholds only ever drop items whose exact score is strictly below k exact scores already
// held, so the final exact pass returns the exact top-k.
// Returns this lane's (n, filter threshold as fp32).  `force` = final pass (exact form).
template <int DK, int EPL>
__device__ __noinline__ unsigned long long tf_compact(unsigned need, int n, int nsort, float thrf, float eps, int k,
                                                      int lane, int row0, const uint8_t* sA,
                                                      const uint8_t* Ib, float* cv_warp, int* ci_warp,
                                                      bool force, unsigned long long* stats) {
  constexpr int CAP = 32 * EPL;
  while (need) {
    const long long c0 = stats ? clock64() : 0;
    const int src = __ffs(need) - 1;
    need &= need - 1;
    const int ns = __shfl_sync(kFull, n, src);
    const int nso = __shfl_sync(kFull, nsort, src);
    const float eps_s = __shfl_sync(kFull, eps, src);
    float* cvr = cv_warp + src * CAP;
    int* cir = ci_warp + src * CAP;
    float ev[EPL];
    int ei[EPL], ef[EPL], rank[EPL];
#pragma unroll
    for (int e = 0; e < EPL; ++e) {
      const int p = lane + 32 * e;
      const bool ok = p < ns;
      ev[e] = ok ? cvr[p] : -INFINITY;
      const int raw = ok ? cir[p] : 0x7fffffff;
      ef[e] = raw & kApprox;                     // still a filter value?
      ei[e] = raw & 0x7fffffff;
    }
    rank_entries_partial<EPL>(ev, ei, rank, ns, nso, lane);
    bool exact = force || ns < k;
    float new_thr = -INFINITY;
    int new_n = ns;
    if (!exact) {
      float A = 0.f;                             // k-th largest value
#pragma unroll
      for (int e = 0; e < EPL; ++e) {
        const unsigned b = __ballot_sync(kFull, rank[e] == k - 1);
        if (b) A = __shfl_sync(kFull, ev[e], __ffs(b) - 1);
      }
      const float keep = A - 2.f * eps_s;
      int c_keep = 0;
#pragma unroll
      for (int e = 0; e < EPL; ++e) c_keep += __popc(__ballot_sync(kFull, ev[e] >= keep));
      if (c_keep <= CAP - 4) {
        __syncwarp();
#pragma unroll
        for (int e = 0; e < EPL; ++e) {
          if (rank[e] < c_keep) {                // the kept entries are exactly the c_keep best-ranked
            cvr[rank[e]] = ev[e];
            cir[rank[e]] = ei[e] | ef[e];
          }
        }
        new_n = c_keep;
        new_thr = keep;
      } else {
        exact = true;                            // too many near-ties: settle them exactly
      }
    }
    if (exact) {
      const int rr = row0 + src;
      const uint8_t* a_row = sA + (size_t)(rr >> 3) * (16 * DK) + (size_t)(rr & 7) * 16;
#pragma unroll
      for (int e = 0; e < EPL; ++e) {
        if (ef[e] && lane + 32 * e < ns) ev[e] = exact_score<DK>(a_row, Ib, ei[e]);
      }
      rank_entries<EPL>(ev, ei, rank);
      __syncwarp();
#pragma unroll
      for (int e = 0; e < EPL; ++e) {
        if (lane + 32 * e < ns && rank[e] < k) {
          cvr[rank[e]] = ev[e];
          cir[rank[e]] = ei[e];
        }
      }
      __syncwarp();
      new_n = ns < k ? ns : k;
      new_thr = (ns >= k) ? cvr[k - 1] - eps_s : -INFINITY;
    }
    __syncwarp();
    if (lane == src) {
      n = new_n;
      nsort = new_n;                             // what is left is in rank order
      thrf = fmaxf(thrf, new_thr);               // thresholds never move down
    }
    if (stats && lane == 0) {
      atomicAdd(stats + 3, 1ull);
      if (exact) atomicAdd(stats + 4, 1ull);
      atomicAdd(stats + 5, (unsigned long long)(clock64() - c0));
    }
  }
  return pack_state(n | (nsort << 16), thrf);
}

template <int DK, int EPL>
__global__ void __launch_bounds__(kThreads, DK == 64 ? 2 : 1)
score_topk_f16_kernel(const uint8_t* __restrict__ Uh, const uint8_t* __restrict__ Ih, int64_t B,
                      int m_items, int n_item_tiles, const float* __restrict__ u_meta,
                      const float* __restrict__ i_meta, const int64_t* __restrict__ user_ids,
                      const int64_t* __restrict__ mask_rowptr, const int32_t* __restrict__ mask_col,
                      int k, int32_t* __restrict__ out_idx, float* __restrict__ out_val, int stages,
                      unsigned long long* __restrict__ stats, int dbg) {
  // dbg (bring-up, SPEX_TF_DBG): bit 0 = nothing survives the filter (cost of the survivor path by
  // difference), bit 1 = the epilogue only hands the accumulator back (MMA side alone)
  constexpr int CAP = 32 * EPL;
  constexpr int A_BYTES = BM * DK * 2, B_BYTES = BN * DK * 2;
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bar_full[kMaxStages];
  __shared__ __align__(8) uint64_t bar_empty[kMaxStages];
  __shared__ __align__(8) uint64_t bar_tfull[2];
  __shared__ __align__(8) uint64_t bar_tempty[2];
  __shared__ __align__(8) uint64_t bar_a;
  __shared__ uint32_t tmem_slot;
  __shared__ MaskCursor mc;

  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 127) &
                                             ~(uintptr_t)127);
  uint8_t* sA = smem;                                                    // [128 users][DK] fp16
  uint8_t* sB = smem + A_BYTES;                                          // stages x [128 items][DK]
  float* cv = reinterpret_cast<float*>(sB + (size_t)stages * B_BYTES);   // [BM][CAP]
  int* ci = reinterpret_cast<int*>(cv + (size_t)CAP * BM);               // [BM][CAP]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t tile_m = blockIdx.x;

  const uint32_t tmem_base =
      pipeline_init(warp, stages, bar_full, bar_empty, bar_tfull, bar_tempty, &bar_a, &tmem_slot);

  if (warp == 0) {
    producer_role<DK>(Uh, Ih, tile_m, n_item_tiles, stages, sA, sB, bar_full, bar_empty, &bar_a);
  } else if (warp == 1) {
    // instruction descriptor: c = f16 (0 at [4,6)), a = b = f16 (0 at [7,10), [10,13)), K-major
    // A and B, N>>3 at [17,23), M>>4 at [24,29)
    constexpr uint32_t idesc = ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
    mma_role<DK>(idesc, sA, sB, tmem_base, n_item_tiles, stages, bar_full, bar_empty, bar_tfull,
                 bar_tempty, &bar_a);
  } else {
    // ===== epilogue: thread owns one user row; warp = TMEM lane quarter =====
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int64_t grow = tile_m * BM + row;
    float* cv_warp = cv + q * 32 * CAP;   // + lane * CAP = this thread's row
    int* ci_warp = ci + q * 32 * CAP;
    int n = 0, nsort = 0;   // entries in the row's buffer; leading entries already in rank order
    // filter threshold of this row (fp32, scaled units) and the largest fp16 below it: an item is
    // offered to the row iff its fp16-accumulated score is >= thr
    float thrf = (grow < B) ? -INFINITY : INFINITY;   // +inf: padded row, nothing survives
    if (dbg & 1) thrf = INFINITY;
    // merge cursor over the row's training items (ascending CSR row of R): the next training item id
    // lives in a register, the cursor itself in shared memory (only touched when it advances)
    // (and the one after it in mnext2: when the cursor advances the load of the following id is issued but
    // not waited for - a single-step advance, the common case, costs no global-memory round trip)
    int mnext = 0x7fffffff, mnext2 = 0x7fffffff;
    {
      const int32_t* c = mask_col;
      const int32_t* e = mask_col;
      if (grow < B && mask_rowptr) {
        const int64_t uid = user_ids ? user_ids[grow] : grow;
        c = mask_col + mask_rowptr[uid];
        e = mask_col + mask_rowptr[uid + 1];
        if (c < e) mnext = __ldg(c);
        if (c + 1 < e) mnext2 = __ldg(c + 1);
      }
      mc.cur[row] = c;
      mc.end[row] = e;
    }
    // the row's norm (scaled units) from the resident A tile -> filter margin
    mbar_wait(&bar_a, 0);
    const uint8_t* a_row = sA + (size_t)(row >> 3) * (16 * DK) + (size_t)(row & 7) * 16;
    float un2 = 0.f;
#pragma unroll
    for (int kc = 0; kc < DK / 8; ++kc) {
      const uint4 a = *reinterpret_cast<const uint4*>(a_row + kc * 128);
      const uint32_t aw[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&aw[j]));
        un2 = fmaf(f.x, f.x, un2);
        un2 = fmaf(f.y, f.y, un2);
      }
    }
    const float vmax = i_meta[2];                       // max scaled item-row norm
    const float eps = kEpsRel<DK> * sqrtf(un2) * vmax * 1.0001f + kEpsAbs;
    float* cv_row = cv_warp + lane * CAP;
    int* ci_row = ci_warp + lane * CAP;
    __half thr = __float2half_rd(thrf);                 // -inf (or +inf for padded rows)
    unsigned long long n_hits = 0, n_tiles_slow = 0, c_slow = 0;
    const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16);
    uint32_t r[64];
    for (int t = 0; t < n_item_tiles; ++t) {
      const int buf = t & 1;
      mbar_wait(&bar_tfull[buf], (uint32_t)(t >> 1) & 1u);
      tc_fence_after();
      if (dbg & 2) {   // bring-up: MMA side alone
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar_tempty[buf]);
        continue;
      }
      tmem_ld128h_issue(tq + (uint32_t)(buf * BN), r);
      tmem_wait64(r);
      // the whole quarter tile is in registers: hand the TMEM buffer back at once
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_tempty[buf]);
      // fast reject: eight independent max chains over blocks of 8 registers (16 columns each),
      // 63 HMNMX2 in all, one compare, one vote
      uint32_t m[8];
#pragma unroll
      for (int b = 0; b < 8; ++b) {
        m[b] = r[8 * b];
#pragma unroll
        for (int i = 1; i < 8; ++i) m[b] = hmax2(m[b], r[8 * b + i]);
      }
      const uint32_t mm = hmax2(hmax2(hmax2(m[0], m[1]), hmax2(m[2], m[3])),
                                hmax2(hmax2(m[4], m[5]), hmax2(m[6], m[7])));
      if (__any_sync(kFull, __hge(__hmax(lo_half(mm), hi_half(mm)), thr))) {
        // slow path: which 16-column blocks hold a hit in any lane
        const long long c0 = stats ? clock64() : 0;
        unsigned bm = 0;
#pragma unroll
        for (int b = 0; b < 8; ++b) bm |= __hge(__hmax(lo_half(m[b]), hi_half(m[b])), thr) ? (1u << b) : 0u;
        unsigned blocks = __reduce_or_sync(kFull, bm);
        ++n_tiles_slow;
#pragma unroll 1
        while (blocks) {
          const int bi = __ffs(blocks) - 1;
          blocks &= blocks - 1;
          // warp-uniform pick of the block's eight packed registers (named scalars: an array written in
          // a switch is placed in local memory by the compiler)
          uint32_t p0, p1, p2, p3, p4, p5, p6, p7;
#define SPEX_PICK(b)                                                                                   \
  case b:                                                                                              \
    p0 = r[8 * b]; p1 = r[8 * b + 1]; p2 = r[8 * b + 2]; p3 = r[8 * b + 3];                             \
    p4 = r[8 * b + 4]; p5 = r[8 * b + 5]; p6 = r[8 * b + 6]; p7 = r[8 * b + 7];                         \
    break;
          switch (bi) {
            SPEX_PICK(0) SPEX_PICK(1) SPEX_PICK(2) SPEX_PICK(3) SPEX_PICK(4) SPEX_PICK(5) SPEX_PICK(6)
            default: SPEX_PICK(7)
          }
#undef SPEX_PICK
          const uint32_t p[8] = {p0, p1, p2, p3, p4, p5, p6, p7};
          // this lane's hits among the block's 16 columns, and the columns that hold a hit in any lane
          const int id0 = t * BN + bi * 16;
          unsigned mine = 0;
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const __half a = (j & 1) ? hi_half(p[j >> 1]) : lo_half(p[j >> 1]);
            mine |= __hge(a, thr) ? (1u << j) : 0u;
          }
          if (id0 + 16 > m_items) mine &= (id0 < m_items) ? ((1u << (m_items - id0)) - 1u) : 0u;   // tile padding
          ++n_hits;
          // one lane-local append of a hit (filter score a, item id): merge cursor, two stores
          auto offer = [&](__half a, int id) {
            if (mnext < id) {                          // advance the merge cursor past id
              const int32_t* c = mc.cur[row];
              const int32_t* e = mc.end[row];
              do {
                ++c;
                mnext = mnext2;
                mnext2 = (c + 1 < e) ? __ldg(c + 1) : 0x7fffffff;
              } while (mnext < id);
              mc.cur[row] = c;
            }
            if (mnext != id) {                         // == id: training item of this user, excluded
              cv_row[n] = __half2float(a);
              ci_row[n] = id | kApprox;
              ++n;
            }
          };
          auto compact = [&](unsigned need) {
            const unsigned long long st = tf_compact<DK, EPL>(need, n, nsort, thrf, eps, k, lane, q * 32, sA, Ih,
                                                             cv_warp, ci_warp, false, stats);
            thrf = __uint_as_float((unsigned)(st & 0xffffffffull));
            thr = __float2half_rd(thrf);
            n = (int)(st >> 32) & 0xffff;
            nsort = (int)(st >> 48);
          };
          if (!__any_sync(kFull, (mine & (mine - 1)) != 0)) {
            // common case (all but the first few tiles): no lane has more than one hit in this block.
            // Rows without room are compacted first, then every hit lane appends on its own.
            const unsigned need = __ballot_sync(kFull, mine != 0 && n == CAP);
            if (need) compact(need);
            if (mine) {
              const int j = __ffs(mine) - 1;
              const uint32_t w = p[j >> 1];
              const __half a = (j & 1) ? hi_half(w) : lo_half(w);
              if (__hge(a, thr)) offer(a, id0 + j);    // thr may have risen in the compaction
            }
          } else {
            // general case: visit, warp-uniformly, every column that holds a hit in some lane
            unsigned cols = __reduce_or_sync(kFull, mine);
#pragma unroll 1
            while (cols) {
              const int j = __ffs(cols) - 1;
              cols &= cols - 1;
              const unsigned need = __ballot_sync(kFull, ((mine >> j) & 1u) && n == CAP);
              if (need) compact(need);
              if ((mine >> j) & 1u) {
                const uint32_t w = p[j >> 1];
                const __half a = (j & 1) ? hi_half(w) : lo_half(w);
                if (__hge(a, thr)) offer(a, id0 + j);
              }
            }
          }
        }
        if (stats) c_slow += (unsigned long long)(clock64() - c0);
      }
    }
    // final compaction of every row (sorted best-first), then each thread writes its own row
    n = (int)(tf_compact<DK, EPL>(kFull, n, nsort, thrf, eps, k, lane, q * 32, sA, Ih, cv_warp, ci_warp, true, nullptr) >> 32) & 0xffff;
    if (grow < B) {
      const float inv = u_meta[1] * i_meta[1];   // 2^-(s_u + s_i): exact
      for (int p = 0; p < k; ++p) {
        const bool ok = p < n;
        out_idx[grow * k + p] = ok ? ci_warp[lane * CAP + p] : -1;
        out_val[grow * k + p] = ok ? cv_warp[lane * CAP + p] * inv : -INFINITY;
      }
    }
    if (stats && lane == 0) {   // bring-up statistics, summed over epilogue warps: slow-path tiles, block
      atomicAdd(stats, n_tiles_slow);      // calls, cycles in the slow path; tf_compact adds [3] compactions,
      atomicAdd(stats + 1, n_hits);        // [4] exact compactions, [5] cycles in compactions
      atomicAdd(stats + 2, c_slow);
    }
  }
  pipeline_teardown(warp, tmem_base);
}

// ---- operand packing ---------------------------------------------------------------------------
// meta[0] = scale 2^s, meta[1] = 2^-s, meta[2] = max scaled row norm, meta[3] = max row norm^2 as
// raw bits (atomicMax on non-negative floats is order-independent: deterministic)
__global__ void __launch_bounds__(256)
rownorm_max_kernel(const float* __restrict__ src, const int64_t* __restrict__ rows, int64_t n, int D,
                   unsigned int* __restrict__ meta_bits) {
  const int lane = threadIdx.x & 31;
  int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t stride = ((int64_t)gridDim.x * blockDim.x) >> 5;
  float best = 0.f;
  for (; w < n; w += stride) {
    const int64_t sr = rows ? rows[w] : w;
    float s = 0.f;
    for (int d = lane * 4; d < D; d += 128) {
      const float4 x = *reinterpret_cast<const float4*>(src + sr * D + d);
      s = fmaf(x.x, x.x, s);
      s = fmaf(x.y, x.y, s);
      s = fmaf(x.z, x.z, s);
      s = fmaf(x.w, x.w, s);
    }
    s = warp_sum(s);
    best = fmaxf(best, s);
  }
  if (lane == 0 && best > 0.f) atomicMax(meta_bits + 3, __float_as_uint(best));
}

// scale = 2^(7 - p) with max_norm = f * 2^p, f in [0.5, 1): every scaled row norm is < 2^7
__device__ __forceinline__ float scale_from_maxnorm2(float n2) {
  if (!(n2 > 0.f) || !isfinite(n2)) return 1.f;
  int p;
  frexpf(sqrtf(n2) * 1.0001f, &p);
  int e = 7 - p;
  e = e > 100 ? 100 : (e < -100 ? -100 : e);
  return ldexpf(1.f, e);
}

__global__ void finish_meta_kernel(float* __restrict__ meta) {
  const float n2 = meta[3];
  const float sc = scale_from_maxnorm2(n2);
  meta[0] = sc;
  meta[1] = 1.f / sc;
  meta[2] = sqrtf(n2) * sc * 1.0001f;
}

// fp32 [rows, D] -> fp16(x * scale) in the layout of pack_rows, scale = meta[0]
__global__ void __launch_bounds__(256)
pack_f16_kernel(const float* __restrict__ src, const int64_t* __restrict__ rows, int64_t n,
                int64_t n_pad, int D, const float* __restrict__ meta, uint8_t* __restrict__ dst) {
  const float sc = meta[0];
  pack_rows(src, rows, n, n_pad, D, dst, [sc](float x, float y) -> uint32_t {
    const __half2 h = __floats2half2_rn(x * sc, y * sc);
    return *reinterpret_cast<const uint32_t*>(&h);
  });
}

static unsigned long long* g_stats = nullptr;

template <int DK, int EPL>
static int launch(const void* Uh, const void* Ih, int64_t B, int64_t B_pad, int64_t m_items,
                  int64_t m_pad, const float* u_meta, const float* i_meta, const int64_t* user_ids,
                  const int64_t* mask_rowptr, const int32_t* mask_col, int32_t k, int32_t* out_idx,
                  float* out_val, cudaStream_t st) {
  // D = 64: two CTAs per SM need <= ~113 KB each (228 KB per SM, 1 KB reserved per CTA, static
  // shared memory ~7 KB); D = 128: one CTA per SM, up to 227 KB
  int stages = choose_stages(DK, 32 * EPL, (DK == 64) ? 115712 - 7600 : 227 * 1024 - 7600);
  if (const char* e = getenv("SPEX_TF_STAGES")) stages = atoi(e);   // bring-up experiment
  SPEX_RETURN_IF(stages < 2 || stages > kMaxStages, SPEX_E_BADARG);
  const size_t smem = smem_bytes(DK, 32 * EPL, stages);
  SPEX_RETURN_IF(smem > 227 * 1024 - 7600, SPEX_E_TOOBIG);
  cudaError_t e = cudaFuncSetAttribute(score_topk_f16_kernel<DK, EPL>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  const int64_t grid = B_pad / BM;
  SPEX_RETURN_IF(grid > 0x7fffffffLL, SPEX_E_TOOBIG);
  int dbg = 0;
  if (const char* e = getenv("SPEX_TF_DBG")) dbg = atoi(e);   // bring-up experiment
  score_topk_f16_kernel<DK, EPL><<<(unsigned)grid, kThreads, smem, st>>>(
      (const uint8_t*)Uh, (const uint8_t*)Ih, B, (int)m_items, (int)(m_pad / BN), u_meta, i_meta,
      user_ids, mask_rowptr, mask_col, k, out_idx, out_val, stages, g_stats, dbg);
  count_launch();
  return check_last();
}

template <int DK>
static int launch_k(const void* Uh, const void* Ih, int64_t B, int64_t B_pad, int64_t m_items,
                    int64_t m_pad, const float* u_meta, const float* i_meta, const int64_t* user_ids,
                    const int64_t* mask_rowptr, const int32_t* mask_col, int32_t k, int32_t* out_idx,
                    float* out_val, cudaStream_t st) {
  // candidate buffer capacity CAP = 32*EPL must hold the k kept entries + room to append
  int epl_min = 1;
  if (const char* e = getenv("SPEX_TF_EPL")) epl_min = atoi(e);   // bring-up experiment
  if (k <= 24 && epl_min <= 1)
    return launch<DK, 1>(Uh, Ih, B, B_pad, m_items, m_pad, u_meta, i_meta, user_ids, mask_rowptr, mask_col, k, out_idx, out_val, st);
  if (k <= 56 && epl_min <= 2)
    return launch<DK, 2>(Uh, Ih, B, B_pad, m_items, m_pad, u_meta, i_meta, user_ids, mask_rowptr, mask_col, k, out_idx, out_val, st);
  return launch<DK, 3>(Uh, Ih, B, B_pad, m_items, m_pad, u_meta, i_meta, user_ids, mask_rowptr, mask_col, k, out_idx, out_val, st);
}

}  // namespace tf
}  // namespace spex

using namespace spex;

extern "C" int spex_pack_f16(const float* src, const int64_t* rows, int64_t n, int64_t n_pad,
                             int32_t D, void* dst_f16, float* meta4, void* stream) {
  SPEX_RETURN_IF(!src || !dst_f16 || !meta4 || n < 0 || n_pad < n || (n_pad & 7), SPEX_E_BADARG);
  SPEX_RETURN_IF(D <= 0 || (D & 7) || D > 512, SPEX_E_BADDIM);
  SPEX_RETURN_IF(!aligned16(src) || !aligned16(dst_f16) || !aligned16(meta4), SPEX_E_ALIGN);
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(meta4, 0, 16, st);
  if (e != cudaSuccess) return (int)e;
  if (n > 0) {
    int64_t blocks = (n * 32 + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    tf::rownorm_max_kernel<<<(unsigned)blocks, 256, 0, st>>>(src, rows, n, D, (unsigned int*)meta4);
    count_launch();
  }
  tf::finish_meta_kernel<<<1, 1, 0, st>>>(meta4);
  count_launch();
  if (n_pad > 0) {
    int64_t blocks = (n_pad * (D / 8) + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    tf::pack_f16_kernel<<<(unsigned)blocks, 256, 0, st>>>(src, rows, n, n_pad, D, meta4, (uint8_t*)dst_f16);
    count_launch();
  }
  return check_last();
}

// bring-up only (not part of the declared ABI): device buffer of 2 uint64 counters
extern "C" void spex_debug_tf_stats(void* dev_buf) { tf::g_stats = (unsigned long long*)dev_buf; }

extern "C" int spex_score_topk_f16(const void* Uh, const void* Ih, int32_t D, int64_t B, int64_t B_pad,
                                   int64_t m_items, int64_t m_pad, const float* u_meta,
                                   const float* i_meta, const int64_t* user_ids,
                                   const int64_t* mask_rowptr, const int32_t* mask_col, int32_t k,
                                   int32_t* out_idx, float* out_val, void* stream) {
  SPEX_RETURN_IF(!Uh || !Ih || !u_meta || !i_meta || !out_idx || !out_val || B < 0 || B_pad < B ||
                     m_items < 0 || m_pad < m_items,
                 SPEX_E_BADARG);
  SPEX_RETURN_IF((mask_rowptr == nullptr) != (mask_col == nullptr), SPEX_E_BADARG);
  SPEX_RETURN_IF((B_pad % tf::BM) || (m_pad % tf::BN), SPEX_E_BADARG);
  SPEX_RETURN_IF(D != 64 && D != 128, SPEX_E_BADDIM);
  SPEX_RETURN_IF(k < 1 || k > tf::KMAX_TC || m_pad > 0x7fffffffLL, SPEX_E_TOOBIG);
  SPEX_RETURN_IF(!aligned16(Uh) || !aligned16(Ih), SPEX_E_ALIGN);
  if (B == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (D == 64)
    return tf::launch_k<64>(Uh, Ih, B, B_pad, m_items, m_pad, u_meta, i_meta, user_ids, mask_rowptr, mask_col, k, out_idx, out_val, st);
  return tf::launch_k<128>(Uh, Ih, B, B_pad, m_items, m_pad, u_meta, i_meta, user_ids, mask_rowptr, mask_col, k, out_idx, out_val, st);
}
