// tcgen05.cuh — the tcgen05 pipeline shared by the two tensor-core scorers (score_topk_tc.cu: bf16
// operands, fp32 accumulators; score_topk_f16.cu: fp16 operands, fp16-accumulator filter).
//
// One CTA owns BM = 128 users (UMMA M) and streams the item table in tiles of BN = 128 items (UMMA N)
// through a ring of `stages` shared-memory buffers.  Operands are K-major in the UMMA "no-swizzle"
// canonical layout (8-row x 16-byte core matrices, one 8-row group = 16*DK bytes contiguous), written
// by pack_rows, so a tile is ONE contiguous block staged by a single 1-D bulk async copy.
//   warp 0     producer_role: one thread copies the user tile once, then every item tile;
//   warp 1     TMEM allocator (pipeline_init / pipeline_teardown) and mma_role: one thread issues
//              the DK/16 MMAs of a tile into one of two 128-column accumulator buffers;
//   warps 2-5  the scorer's own epilogue: TMEM lane quarter = warp % 4, one thread per user row.
// Barriers: full[s] / empty[s] per ring stage, tfull[b] / tempty[b] per accumulator buffer (tempty
// takes one arrive per epilogue warp), a = user tile landed.
#pragma once
#include "topk.cuh"

namespace spex {
namespace tcgen05 {

constexpr int BM = 128;            // users per CTA  (UMMA M)
constexpr int BN = 128;            // items per tile (UMMA N)
constexpr int UMMA_K = 16;
constexpr int kThreads = 32 * 6;
constexpr int kMaxStages = 4;
constexpr int kTmemCols = 256;     // 2 accumulator buffers x 128 columns (fp16 accumulators still
                                   // occupy one 32-bit cell each); two CTAs share an SM at D = 64
constexpr int KMAX_TC = 64;
constexpr uint32_t kSpinLimit = 1u << 26;   // bounded waits: trap instead of hanging the GPU

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > kSpinLimit) __trap();
  }
}
// 1-D bulk async copy global -> shared, completion counted in bytes on `bar`
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
// Elect one thread of a converged warp.  With elect.sync the compiler knows that exactly one thread
// runs the guarded block and issues tcgen05.mma / tcgen05.commit / cp.async.bulk straight from
// uniform registers; with `lane == 0` it wraps every such instruction in an ELECT + BRA.U.ANY
// loop with R2UR moves (~61 cycles per MMA issue, measured: profiles/microbench/mma_pipe.cu).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "elect.sync _|P1, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P1;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T; operand and accumulator types come from the instruction
// descriptor (bf16 -> fp32 or fp16 -> fp16)
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc,
                                       uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// UMMA shared-memory descriptor, SWIZZLE_NONE, K-major canonical layout
//   bits [0,14) start>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version=1 | [61,64) layout=0
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}

__device__ __forceinline__ unsigned long long pack_state(int n, float tau) {
  return ((unsigned long long)(unsigned)n << 32) | (unsigned long long)__float_as_uint(tau);
}

// Prologue: thread 0 initialises the barriers, warp 1 allocates the TMEM accumulators.  Called by
// every thread; returns the TMEM base address.
__device__ __forceinline__ uint32_t pipeline_init(int warp, int stages, uint64_t* bar_full,
                                                  uint64_t* bar_empty, uint64_t* bar_tfull,
                                                  uint64_t* bar_tempty, uint64_t* bar_a,
                                                  uint32_t* tmem_slot) {
  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; ++s) {
      mbar_init(&bar_full[s], 1);
      mbar_init(&bar_empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&bar_tfull[b], 1);
      mbar_init(&bar_tempty[b], 4);   // one arrive per epilogue warp
    }
    mbar_init(bar_a, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(tmem_slot)),
                 "r"((uint32_t)kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  return *tmem_slot;
}

// Producer (warp 0): one thread streams the user tile `tile_m` once, then every item tile.
template <int DK>
__device__ __forceinline__ void producer_role(const uint8_t* Ug, const uint8_t* Ig, int64_t tile_m,
                                              int n_item_tiles, int stages, uint8_t* sA, uint8_t* sB,
                                              uint64_t* bar_full, uint64_t* bar_empty, uint64_t* bar_a) {
  constexpr int A_BYTES = BM * DK * 2, B_BYTES = BN * DK * 2;
  if (elect_one()) {
    mbar_arrive_expect_tx(bar_a, A_BYTES);
    bulk_g2s(sA, Ug + tile_m * A_BYTES, A_BYTES, bar_a);
    int t = 0;
    uint32_t ph = 0;
    int s = 0;
    for (; t < n_item_tiles; ++t) {
      mbar_wait(&bar_empty[s], ph ^ 1u);
      mbar_arrive_expect_tx(&bar_full[s], B_BYTES);
      bulk_g2s(sB + (size_t)s * B_BYTES, Ig + (size_t)t * B_BYTES, B_BYTES, &bar_full[s]);
      if (++s == stages) {
        s = 0;
        ph ^= 1u;
      }
    }
  }
}

// MMA issuer (warp 1): one thread drives the tensor core.  Tile t goes to accumulator buffer t & 1;
// its commits free the ring stage and hand the buffer to the epilogue.
template <int DK>
__device__ __forceinline__ void mma_role(uint32_t idesc, uint8_t* sA, uint8_t* sB, uint32_t tmem_base,
                                         int n_item_tiles, int stages, uint64_t* bar_full,
                                         uint64_t* bar_empty, uint64_t* bar_tfull,
                                         uint64_t* bar_tempty, uint64_t* bar_a) {
  constexpr int B_BYTES = BN * DK * 2;
  constexpr uint32_t lbo = 128, sbo = 16 * DK;   // layout written by pack_rows
  if (elect_one()) {
    const uint32_t a_addr = smem_u32(sA);
    constexpr uint32_t kstep = 2 * lbo;  // 16 elements along K = two 8-element core matrices
    mbar_wait(bar_a, 0);
    int s = 0;
    uint32_t ph = 0;
    for (int t = 0; t < n_item_tiles; ++t) {
      const int buf = t & 1;
      const uint32_t use = (uint32_t)(t >> 1) & 1u;
      // While the tensor pipe is busy a poll of an mbarrier takes ~200 cycles even when its
      // phase is long complete (profiles/microbench/mma_pipe.cu), so the two polls of a tile
      // (operands landed, accumulator drained) are issued back to back and overlap.
      bool have_b = mbar_try_wait(&bar_full[s], ph);
      bool have_d = mbar_try_wait(&bar_tempty[buf], use ^ 1u);
      uint32_t spins = 0;
      while (!have_b) {
        have_b = mbar_try_wait(&bar_full[s], ph);
        if (++spins > kSpinLimit) __trap();
      }
      while (!have_d) {
        have_d = mbar_try_wait(&bar_tempty[buf], use ^ 1u);
        if (++spins > kSpinLimit) __trap();
      }
      tc_fence_after();
      const uint32_t b_addr = smem_u32(sB + (size_t)s * B_BYTES);
#pragma unroll
      for (int kk = 0; kk < DK / UMMA_K; ++kk) {
        tc_mma(tmem_base + (uint32_t)(buf * BN), make_desc(a_addr + kk * kstep, lbo, sbo),
               make_desc(b_addr + kk * kstep, lbo, sbo), idesc, kk > 0 ? 1u : 0u);
      }
      tc_commit(&bar_empty[s]);     // smem stage reusable once these MMAs have read it
      tc_commit(&bar_tfull[buf]);   // accumulator ready for the epilogue
      if (++s == stages) {
        s = 0;
        ph ^= 1u;
      }
    }
  }
}

// Teardown: after every role is done, warp 1 frees the TMEM accumulators.  Called by every thread.
__device__ __forceinline__ void pipeline_teardown(int warp, uint32_t tmem_base) {
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"((uint32_t)kTmemCols)
                 : "memory");
  }
}

// fp32 [rows, D] -> 16-bit core-matrix-tiled layout:
//   byte offset of (r, k) = (r/8) * (16*D) + (k/8) * 128 + (r%8) * 16 + (k%8) * 2
// optional row gather; rows in [n, n_pad) are zero.  Thread per (row, 8-element chunk);
// cvt(x, y) converts two elements into one 32-bit word (x in the low half).  No __restrict__ here:
// the calling kernels' restrict parameters already put the row-index loads on the read-only path,
// and restrict on this inlined helper takes them off it (LDG.CONSTANT -> LDG).
template <class Cvt>
__device__ __forceinline__ void pack_rows(const float* src, const int64_t* rows,
                                          int64_t n, int64_t n_pad, int D, uint8_t* dst,
                                          Cvt cvt) {
  const int D8 = D >> 3;
  const int64_t total = n_pad * D8;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < total; i += stride) {
    const int64_t r = i / D8;
    const int kc = (int)(i - r * D8);
    float4 a = f4_zero(), b = f4_zero();
    if (r < n) {
      const int64_t sr = rows ? rows[r] : r;
      a = *reinterpret_cast<const float4*>(src + sr * D + kc * 8);
      b = *reinterpret_cast<const float4*>(src + sr * D + kc * 8 + 4);
    }
    uint4 pk;
    pk.x = cvt(a.x, a.y);
    pk.y = cvt(a.z, a.w);
    pk.z = cvt(b.x, b.y);
    pk.w = cvt(b.z, b.w);
    const int64_t off = (r >> 3) * (16 * (int64_t)D) + (int64_t)kc * 128 + (r & 7) * 16;
    *reinterpret_cast<uint4*>(dst + off) = pk;
  }
}

// ---- host side -----------------------------------------------------------------------------------
// dynamic shared memory of a CTA: 128 B of alignment slack, the user tile, `stages` item tiles and
// the [BM][cap] candidate buffers (fp32 score + int32 id)
static inline size_t smem_bytes(int DK, int cap, int stages) {
  return 128 + (size_t)BM * DK * 2 + (size_t)stages * BN * DK * 2 + (size_t)cap * BM * 8;
}

// the deepest ring (at least 2 stages) whose dynamic shared memory fits `budget` bytes
static inline int choose_stages(int DK, int cap, size_t budget) {
  int stages = kMaxStages;
  while (stages > 2 && smem_bytes(DK, cap, stages) > budget) --stages;
  return stages;
}

}  // namespace tcgen05
}  // namespace spex
