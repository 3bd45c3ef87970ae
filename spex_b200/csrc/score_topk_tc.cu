// score_topk_tc.cu — full-ranking top-k on the 5th-generation tensor cores (tcgen05 / TMEM).
//
// north_star (3): getUsersRating (abstract at LightGCN_SPEX/code/utility1/model.py:14-15; the only
// user x all-items matmul in the reference is NGCF_SPEX/code/utility/batch_test.py:158) followed by
// top-k, is a dense [users,64] x [64,items] contraction, so it goes on the tensor cores:
//
//   * operands: bf16, K-major, pre-packed by spex_pack_bf16 into the UMMA "no-swizzle" canonical
//     layout (8-row x 16-byte core matrices; one 8-row group = 1 KB contiguous).  A tile of any
//     multiple of 8 rows is therefore ONE contiguous block of global memory and is staged by a
//     single 1-D bulk async copy (cp.async.bulk -> UBLKCP) that completes on an mbarrier; no
//     tensor map, no swizzle bookkeeping;
//   * tile: one CTA owns 128 users (UMMA M=128) and streams the item table in tiles of N=128
//     through a multi-stage smem ring.  Per tile: 4 tcgen05.mma.cta_group::1.kind::f16 (K = 4 x 16)
//     issued by one thread; fp32 accumulators in TMEM, double buffered (2 x 128 columns).  A
//     4-MMA chain has ~400 cycles of fixed issue->commit->wake latency on B200 (measured,
//     profiles/microbench/mma_lat.cu), far more than its 256 cycles of math, so TWO CTAs are
//     resident per SM (256 TMEM columns each): four tiles are in flight per SM and the tensor
//     pipe of one CTA works while the other CTA's chain drains;
//   * epilogue (4 warps, thread = user row): with K = 64 every accumulator element is read after
//     only 64 MACs, so the TMEM -> register read (tcgen05.ld, ~170 B/cycle/SM while the MMA pipe
//     is busy) is the co-bottleneck of the MMA pipe.  Loads are software-pipelined (chunk c+1 in
//     flight while chunk c is reduced); a 32-score chunk is rejected with a 3-input-max tree
//     (FMNMX3) and ONE compare against the row's threshold tau;
//   * survivors (about k*ln(m/k) per row over the whole sweep) must not stall the pipeline: a
//     survivor is only APPENDED to the row's unsorted candidate buffer in shared memory after a
//     merge-cursor test against the user's training items (CSR row of R; item ids arrive in
//     ascending order, so the cursor only moves forward: no binary search, no dependent global
//     loads).  When a buffer cannot take the next group of survivors the whole warp compacts it:
//     rank-by-counting over the <= CAP entries (exchanged by warp shuffles), the best k are
//     rewritten in sorted order and tau becomes the k-th best.
//     Scores never touch HBM;
//   * warp roles: warp 0 = bulk-copy producer, warp 1 = TMEM allocator + MMA issuer, warps 2-5 =
//     epilogue (TMEM lane quarter = warp % 4).  The two single-thread roles are entered through
//     elect.sync (straight-line UTCHMMA/UTCBAR/UBLKCP instead of one ELECT + BRA.U.ANY loop per
//     instruction) and the MMA thread issues its two mbarrier polls of a tile back to back:
//     together 1134 -> 1699 TFLOP/s for the MMA side alone, 895 -> 935 with the epilogue.
#include "tcgen05.cuh"
#include <cuda_bf16.h>

namespace spex {
namespace tc {

using namespace tcgen05;

constexpr int DK = 64;             // embedding dim  (4 x UMMA K)
constexpr int A_BYTES = BM * DK * 2;
constexpr int B_BYTES = BN * DK * 2;
constexpr int kGroup = 8;          // appends are capacity-checked every 8 scores

// tcgen05.ld 32 lanes x 32 columns (one 32-bit word per lane per column) WITHOUT waiting: the
// registers are only valid after tmem_wait32() on the same array.
#define SPEX_R32(r)                                                                            \
  r[0], r[1], r[2], r[3], r[4], r[5], r[6], r[7], r[8], r[9], r[10], r[11], r[12], r[13], r[14], \
      r[15], r[16], r[17], r[18], r[19], r[20], r[21], r[22], r[23], r[24], r[25], r[26], r[27], \
      r[28], r[29], r[30], r[31]
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
        "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// wait for every outstanding tcgen05.ld of this thread; the "+r" operands tie the loaded
// registers to the wait so that no consumer can be scheduled above it.
__device__ __forceinline__ void tmem_wait32(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]),
                 "+r"(r[7]), "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]),
                 "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]),
                 "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]),
                 "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]),
                 "+r"(r[31])
               :
               : "memory");
}
__device__ __forceinline__ float max3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));  // FMNMX3
  return d;
}
// max of 32 scores in 16 FMNMX3
__device__ __forceinline__ float max32(const uint32_t (&r)[32]) {
#define F(i) __uint_as_float(r[i])
  const float a0 = max3(F(0), F(1), F(2)), a1 = max3(F(3), F(4), F(5)), a2 = max3(F(6), F(7), F(8));
  const float a3 = max3(F(9), F(10), F(11)), a4 = max3(F(12), F(13), F(14));
  const float a5 = max3(F(15), F(16), F(17)), a6 = max3(F(18), F(19), F(20));
  const float a7 = max3(F(21), F(22), F(23)), a8 = max3(F(24), F(25), F(26));
  const float a9 = max3(F(27), F(28), F(29));
  const float b0 = max3(a0, a1, a2), b1 = max3(a3, a4, a5), b2 = max3(a6, a7, a8);
  const float b3 = max3(a9, F(30), F(31));
  return fmaxf(max3(b0, b1, b2), b3);
#undef F
}

// Per-row mask cursor, kept in shared memory because only the rare survivor path touches it.
// Items are offered to a row in strictly ascending id order (tile, chunk, column) and the row's
// training items (CSR row of R) are ascending too, so the mask test is a merge: the cursor only
// moves forward and a row performs at most |train(u)| sequential mask loads over the whole sweep.
struct MaskCursor {
  const int32_t* cur[BM];
  const int32_t* end[BM];
  int next[BM];                // smallest training item id not yet passed (INT_MAX: none left)
};

// One column of a chunk has at least one survivor in this warp (lanes in `b`).  Called by the
// whole warp (convergent), out of line.  Each surviving lane runs the mask cursor and appends
// (v, id) to its row's candidate buffer (row-major in shared memory: entry p of row r at
// cv[r * CAP + p]); rows whose buffer became full are compacted cooperatively: every lane takes
// EPL entries into registers, ranks them by counting the entries that beat them (entries travel
// by warp shuffle; (score desc, id asc) is a strict total order, so ranks are a permutation), the
// best k are written back in sorted order and the row's threshold becomes its k-th best score.
// Returns this lane's (n, tau).  `force` compacts the rows in `b` without appending (final pass).
template <int EPL>
__device__ __noinline__ unsigned long long tc_column(unsigned b, float v, int id, int n, float tau,
                                                     int k, int m_items, int lane, int row, float* cv_warp,
                                                     int* ci_warp, MaskCursor* mc, bool force) {
  constexpr int CAP = 32 * EPL;
  unsigned need = b;
  if (!force) {
    if (((b >> lane) & 1u) && id < m_items) {   // id >= m_items: zero padding of the last tile
      int mnext = mc->next[row];
      if (mnext < id) {
        const int32_t* c = mc->cur[row];
        const int32_t* e = mc->end[row];
        do {
          ++c;
          mnext = (c < e) ? __ldg(c) : 0x7fffffff;
        } while (mnext < id);
        mc->cur[row] = c;
        mc->next[row] = mnext;
      }
      if (mnext != id) {                        // == id: training item of this user, excluded
        cv_warp[lane * CAP + n] = v;
        ci_warp[lane * CAP + n] = id;
        ++n;
      }
    }
    need = __ballot_sync(kFull, n == CAP);
  }
  while (need) {
    const int src = __ffs(need) - 1;
    need &= need - 1;
    const int ns = __shfl_sync(kFull, n, src);
    float* cvr = cv_warp + src * CAP;
    int* cir = ci_warp + src * CAP;
    float ev[EPL];
    int ei[EPL], rank[EPL];
#pragma unroll
    for (int e = 0; e < EPL; ++e) {
      const int p = lane + 32 * e;
      const bool ok = p < ns;
      ev[e] = ok ? cvr[p] : -INFINITY;
      ei[e] = ok ? cir[p] : 0x7fffffff;
      rank[e] = 0;
    }
#pragma unroll
    for (int e2 = 0; e2 < EPL; ++e2) {
#pragma unroll 4
      for (int j = 0; j < 32; ++j) {   // kept rolled: cold code must stay small (i-cache)
        const float vj = __shfl_sync(kFull, ev[e2], j);
        const int ij = __shfl_sync(kFull, ei[e2], j);
#pragma unroll
        for (int e = 0; e < EPL; ++e) rank[e] += beats(vj, ij, ev[e], ei[e]) ? 1 : 0;
      }
    }
    __syncwarp();
#pragma unroll
    for (int e = 0; e < EPL; ++e) {
      if (lane + 32 * e < ns && rank[e] < k) {
        cvr[rank[e]] = ev[e];
        cir[rank[e]] = ei[e];
      }
    }
    __syncwarp();
    const float tau_new = (ns >= k) ? cvr[k - 1] : -INFINITY;
    if (lane == src) {
      n = ns < k ? ns : k;
      tau = tau_new;
    }
  }
  return pack_state(n, tau);
}

__device__ __forceinline__ float tmem_ld1(uint32_t taddr) {
  uint32_t x;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(x) : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" : "+r"(x) : : "memory");
  return __uint_as_float(x);
}

// reduce one 32-score chunk against the row's threshold.  Fast path: 16 FMNMX3 + one compare +
// one warp vote.  The kernel is instruction-fetch sensitive (the hot loop must stay resident in
// the SM's instruction cache while two CTAs and three warp roles share it), so the survivor path
// is written as LOOPS, not unrolled code: each lane builds a 32-bit mask of its surviving
// columns, the warp ORs the masks (REDUX) and visits only the columns that have a survivor,
// re-reading that column from TMEM (the accumulator buffer is still owned by the epilogue).
template <int EPL>
__device__ __forceinline__ void consume_chunk(const uint32_t (&r)[32], uint32_t taddr, int item0, int& n,
                                              float& tau, int k, int m_items, int lane, int row,
                                              float* cv_warp, int* ci_warp, MaskCursor* mc) {
  if (__any_sync(kFull, max32(r) > tau)) {
    unsigned mine = 0;
#pragma unroll
    for (int i = 0; i < 32; ++i) mine |= (__uint_as_float(r[i]) > tau) ? (1u << i) : 0u;
    unsigned cols = __reduce_or_sync(kFull, mine);
#pragma unroll 1
    while (cols) {
      const int i = __ffs(cols) - 1;
      cols &= cols - 1;
      const float v = tmem_ld1(taddr + i);
      const unsigned b = __ballot_sync(kFull, v > tau);   // tau may have risen since the mask was built
      if (b) {
        const unsigned long long st = tc_column<EPL>(b, v, item0 + i, n, tau, k, m_items, lane, row,
                                                     cv_warp, ci_warp, mc, false);
        tau = __uint_as_float((unsigned)(st & 0xffffffffull));
        n = (int)(st >> 32);
      }
    }
  }
}

template <int EPL>
__global__ void __launch_bounds__(kThreads, 2)
score_topk_tc_kernel(const uint8_t* __restrict__ Ub, const uint8_t* __restrict__ Ib, int64_t B,
                     int m_items, int n_item_tiles, const int64_t* __restrict__ user_ids,
                     const int64_t* __restrict__ mask_rowptr, const int32_t* __restrict__ mask_col,
                     int k, int32_t* __restrict__ out_idx, float* __restrict__ out_val, int stages) {
  constexpr int CAP = 32 * EPL;
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
  uint8_t* sA = smem;                                                    // [128 users][64] bf16
  uint8_t* sB = smem + A_BYTES;                                          // stages x [128 items][64]
  float* cv = reinterpret_cast<float*>(sB + (size_t)stages * B_BYTES);   // [BM][CAP]
  int* ci = reinterpret_cast<int*>(cv + (size_t)CAP * BM);               // [BM][CAP]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t tile_m = blockIdx.x;

  const uint32_t tmem_base =
      pipeline_init(warp, stages, bar_full, bar_empty, bar_tfull, bar_tempty, &bar_a, &tmem_slot);

  if (warp == 0) {
    producer_role<DK>(Ub, Ib, tile_m, n_item_tiles, stages, sA, sB, bar_full, bar_empty, &bar_a);
  } else if (warp == 1) {
    // instruction descriptor: c=f32 (1<<4), a=bf16 (1<<7), b=bf16 (1<<10), K-major A and B,
    // N>>3 at [17,23), M>>4 at [24,29)
    constexpr uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) |
                               ((uint32_t)(BM >> 4) << 24);
    mma_role<DK>(idesc, sA, sB, tmem_base, n_item_tiles, stages, bar_full, bar_empty, bar_tfull,
                 bar_tempty, &bar_a);
  } else {
    // ===== epilogue: thread owns one user row; warp = TMEM lane quarter =====
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int64_t grow = tile_m * BM + row;
    float* cv_warp = cv + q * 32 * CAP;   // + lane * CAP = this thread's row
    int* ci_warp = ci + q * 32 * CAP;
    int n = 0;
    float tau = (grow < B) ? -INFINITY : INFINITY;   // +inf: padded row, nothing survives
    {
      const int32_t* c = mask_col;
      const int32_t* e = mask_col;
      int mnext = 0x7fffffff;
      if (grow < B && mask_rowptr) {
        const int64_t uid = user_ids ? user_ids[grow] : grow;
        c = mask_col + mask_rowptr[uid];
        e = mask_col + mask_rowptr[uid + 1];
        if (c < e) mnext = __ldg(c);
      }
      mc.cur[row] = c;
      mc.end[row] = e;
      mc.next[row] = mnext;
    }
    uint32_t ra[32], rb[32], rc[32];
    for (int t = 0; t < n_item_tiles; ++t) {
      const int buf = t & 1;
      const uint32_t use = (uint32_t)(t >> 1) & 1u;
      mbar_wait(&bar_tfull[buf], use);
      tc_fence_after();
      const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BN);
      const int item0 = t * BN;
      // software pipeline over the four 32-column chunks with three register buffers: two
      // tcgen05.ld are in flight while a chunk is reduced (TMEM read latency is ~190 cycles per
      // 4 KB while the MMA pipe is busy, so the read rate scales with the loads in flight)
      tmem_ld32_issue(tbase, ra);
      tmem_ld32_issue(tbase + 32, rb);
      tmem_wait32(ra);
      tmem_wait32(rb);
      tmem_ld32_issue(tbase + 64, rc);
      consume_chunk<EPL>(ra, tbase, item0, n, tau, k, m_items, lane, row, cv_warp, ci_warp, &mc);
      tmem_ld32_issue(tbase + 96, ra);
      consume_chunk<EPL>(rb, tbase + 32, item0 + 32, n, tau, k, m_items, lane, row, cv_warp, ci_warp, &mc);
      tmem_wait32(rc);
      tmem_wait32(ra);
      consume_chunk<EPL>(rc, tbase + 64, item0 + 64, n, tau, k, m_items, lane, row, cv_warp, ci_warp, &mc);
      consume_chunk<EPL>(ra, tbase + 96, item0 + 96, n, tau, k, m_items, lane, row, cv_warp, ci_warp, &mc);
      // every column of this accumulator has been reduced: hand the TMEM buffer back
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_tempty[buf]);
    }
    // final compaction of every row (sorted best-first), then each thread writes its own row
    n = (int)(tc_column<EPL>(kFull, 0.f, 0, n, tau, k, m_items, lane, row, cv_warp, ci_warp, &mc, true) >> 32);
    if (grow < B) {
      for (int p = 0; p < k; ++p) {
        const bool ok = p < n;
        out_idx[grow * k + p] = ok ? ci_warp[lane * CAP + p] : -1;
        out_val[grow * k + p] = ok ? cv_warp[lane * CAP + p] : -INFINITY;
      }
    }
  }
  pipeline_teardown(warp, tmem_base);
}

// fp32 [rows, D] -> bf16 in the layout of pack_rows
__global__ void __launch_bounds__(256)
pack_bf16_kernel(const float* __restrict__ src, const int64_t* __restrict__ rows, int64_t n,
                 int64_t n_pad, int D, uint8_t* __restrict__ dst) {
  pack_rows(src, rows, n, n_pad, D, dst, [](float x, float y) -> uint32_t {
    return (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(x)) |
           ((uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(y)) << 16);
  });
}

}  // namespace tc
}  // namespace spex

using namespace spex;

extern "C" int spex_pack_bf16(const float* src, const int64_t* rows, int64_t n, int64_t n_pad,
                              int32_t D, void* dst_bf16, void* stream) {
  SPEX_RETURN_IF(!src || !dst_bf16 || n < 0 || n_pad < n || (n_pad & 7), SPEX_E_BADARG);
  SPEX_RETURN_IF(D <= 0 || (D & 7) || D > 512, SPEX_E_BADDIM);
  SPEX_RETURN_IF(!aligned16(src) || !aligned16(dst_bf16), SPEX_E_ALIGN);
  if (n_pad == 0) return 0;
  int64_t blocks = (n_pad * (D / 8) + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  tc::pack_bf16_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
      src, rows, n, n_pad, D, (uint8_t*)dst_bf16);
  count_launch();
  return check_last();
}

template <int EPL>
static int tc_launch(const void* Ub, const void* Ib, int64_t B, int64_t B_pad, int64_t m_items,
                     int64_t m_pad, const int64_t* user_ids, const int64_t* mask_rowptr,
                     const int32_t* mask_col, int32_t k, int32_t* out_idx, float* out_val,
                     cudaStream_t st) {
  // two CTAs per SM need <= ~113 KB each (228 KB per SM, 1 KB reserved per CTA, static smem)
  const int stages = tcgen05::choose_stages(tc::DK, 32 * EPL, 115712 - 2800);
  const size_t smem = tcgen05::smem_bytes(tc::DK, 32 * EPL, stages);
  SPEX_RETURN_IF(smem > 226 * 1024, SPEX_E_TOOBIG);
  // per device and per function, and the size depends on `stages`: set on every launch (cheap)
  {
    cudaError_t e = cudaFuncSetAttribute(tc::score_topk_tc_kernel<EPL>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
  }
  const int64_t grid = B_pad / tc::BM;
  SPEX_RETURN_IF(grid > 0x7fffffffLL, SPEX_E_TOOBIG);
  tc::score_topk_tc_kernel<EPL><<<(unsigned)grid, tc::kThreads, smem, st>>>(
      (const uint8_t*)Ub, (const uint8_t*)Ib, B, (int)m_items, (int)(m_pad / tc::BN), user_ids,
      mask_rowptr, mask_col, k, out_idx, out_val, stages);
  count_launch();
  return check_last();
}

extern "C" int spex_score_topk_bf16(const void* Ub, const void* Ib, int64_t B, int64_t B_pad,
                                    int64_t m_items, int64_t m_pad, const int64_t* user_ids,
                                    const int64_t* mask_rowptr, const int32_t* mask_col, int32_t k,
                                    int32_t* out_idx, float* out_val, void* stream) {
  SPEX_RETURN_IF(!Ub || !Ib || !out_idx || !out_val || B < 0 || B_pad < B || m_items < 0 ||
                     m_pad < m_items,
                 SPEX_E_BADARG);
  SPEX_RETURN_IF((mask_rowptr == nullptr) != (mask_col == nullptr), SPEX_E_BADARG);
  SPEX_RETURN_IF((B_pad % tc::BM) || (m_pad % tc::BN), SPEX_E_BADARG);
  SPEX_RETURN_IF(k < 1 || k > tc::KMAX_TC || m_pad > 0x7fffffffLL, SPEX_E_TOOBIG);
  SPEX_RETURN_IF(!aligned16(Ub) || !aligned16(Ib), SPEX_E_ALIGN);
  if (B == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  // candidate buffer capacity CAP = 32*EPL must hold k kept entries + one group of appends
  if (k <= 32 - tc::kGroup)
    return tc_launch<1>(Ub, Ib, B, B_pad, m_items, m_pad, user_ids, mask_rowptr, mask_col, k, out_idx, out_val, st);
  if (k <= 64 - tc::kGroup)
    return tc_launch<2>(Ub, Ib, B, B_pad, m_items, m_pad, user_ids, mask_rowptr, mask_col, k, out_idx, out_val, st);
  return tc_launch<3>(Ub, Ib, B, B_pad, m_items, m_pad, user_ids, mask_rowptr, mask_col, k, out_idx, out_val, st);
}
