// spmm.cu — deterministic CSR row-per-warp SpMM for the LightGCN propagation (sm_100a).
//
// Replaces torch.sparse.mm(g_droped, all_emb)      LightGCN_SPEX/code/utility1/model.py:91
// and, through the fused epilogue, stack+mean       model.py:94-95
// and the autograd of both                          main_rec.py:35
//
// Design (0.48 flop/B: an HBM / L2-slice bandwidth kernel - no tensor cores on purpose):
//   * one warp owns one output row, one warp per CTA (the block scheduler backfills a warp slot as soon as a
//     row is done); the row's (col,val) run is read coalesced, 32 edges at a time, with streaming hints, one
//     batch ahead of the gathers;
//   * shipped gather loop (warp_row_accumulate8, 32-byte aligned tables): LDG.256 - 8 lanes x 32 B cover a
//     256-byte row (D=64), one warp instruction fetches 4 neighbour rows, 4 in flight per lane before the first
//     FMA; the batch's edges are dealt to the lane groups in consecutive runs so that a segmented shuffle with
//     an immediate lane delivers them; hot columns (bit 31 of col) load with L2::evict_last, the rest with
//     evict_first (static qualifiers, 256-bit loads only).  4.2 instructions per edge.
//     Fallback for tables that are only 16-byte aligned: the 128-bit loop of round 1
//     (warp_row_accumulate: 16 lanes per row, policy descriptors);
//   * lane groups accumulate disjoint edge runs in edge order and are combined by a fixed xor-shuffle tree: the
//     summation order is a pure function of the row => bit-reproducible, no atomics;
//   * rows longer than plan->seg_len are skipped here and reduced by two extra launches over the plan's segment
//     list (warp per run of segments -> partial rows -> warp per long row): hub rows cut at column-block
//     boundaries and listed block-major so that the table window they gather from stays in L2, the other long
//     rows cut every seg_len edges;
//   * epilogue: Y = acc (next layer's input) and/or Z = (addend*a + acc)*b (running layer mean forward,
//     g + A^T G backward) plus, on flagged rows, an added gradient (the BPR L2 term of the last backward layer),
//     optionally stored into every peer's table (P2P or one NVLS multicast store), with the
//     next call's table or a dense Adam step riding on the last layer (row-partitioned modes);
//   * a layer can be restricted to a ROW LIST (RowSubset: the receptive field of a mini-batch) and can be told
//     which rows of X may be non-zero (x_nonzero: the sparse gradient tables of the training backward); both
//     keep every computed row bit-identical to the full dense layer.
#include "common.cuh"
#include <math.h>

namespace spex {

int64_t g_launches = 0;

template <int D>
struct RowShape {
  static_assert(D == 32 || D == 64 || D == 128, "vector path supports D in {32,64,128}");
  static constexpr int LPR = D / 4;    // lanes that cover one row with float4
  static constexpr int G = 32 / LPR;   // neighbour rows gathered per LDG.128 warp instruction
};

// Sum over edges e in [start,end) of val[e] * X[col[e], :], returned in every lane for the
// float4 slot `lane % LPR`.  kList: col[e] lists partial rows of X and val[e] = 1 (val is not read).
// kHot: bit 31 of a column index flags a hot table row (spex_long_plan.flags & SPEX_PLAN_COL_HOTBIT):
// hot rows are gathered with the L2 evict_last policy, the rest with evict_first.
template <int D, int U, bool kList, bool kHot = false>
__device__ __forceinline__ float4 warp_row_accumulate(const int32_t* __restrict__ col,
                                                      const float* __restrict__ val,
                                                      const float* __restrict__ X, int64_t start,
                                                      int64_t end, int lane) {
  constexpr int LPR = RowShape<D>::LPR, G = RowShape<D>::G;
  const int grp = lane / LPR, sub = lane % LPR;
  const float* Xs = X + sub * 4;
  float4 acc = f4_zero();
  uint64_t pol_last = 0, pol_first = 0;
  if (kHot) {
    pol_last = l2_policy_evict_last();
    pol_first = l2_policy_evict_first();
  }
  for (int64_t base = start; base < end; base += 32) {
    const int64_t e = base + lane;
    int c = 0;
    float v = 0.f;
    if (e < end) {
      c = ld_stream_s32(col + e);
      v = kList ? 1.f : ld_stream_f32(val + e);
    }
    const int n = (int)((end - base) < 32 ? (end - base) : 32);
#pragma unroll 1
    for (int j = 0; j < n; j += G * U) {
      float4 x[U];
      float vv[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int idx = j + u * G + grp;
        const int cc = __shfl_sync(kFull, c, idx & 31);
        vv[u] = __shfl_sync(kFull, v, idx & 31);
        if (idx < n) {
          if (kHot)
            x[u] = ld_gather_f4_hint(Xs + (int64_t)(cc & 0x7fffffff) * D, cc < 0 ? pol_last : pol_first);
          else
            x[u] = ld_gather_f4(Xs + (int64_t)cc * D);
        } else {
          x[u] = f4_zero();
          vv[u] = 0.f;
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) f4_fma(acc, vv[u], x[u]);
    }
  }
#pragma unroll
  for (int m = LPR; m < 32; m <<= 1) f4_add(acc, f4_shfl_xor(acc, m));
  return acc;
}

// ---- 256-bit gathers (the shipped path for 32-byte aligned tables) --------------------------------
// Blackwell's LDG.256: a lane fetches 32 B, so LPR8 = D/8 lanes cover a row and one warp instruction gathers
// G8 = 32/LPR8 neighbour rows (4 at D=64) - half the load instructions, shuffles and address arithmetic per
// edge of the 128-bit version above.  The warp's 32-edge batch is dealt to the lane groups in CONSECUTIVE
// runs (group g owns batch edges [g*LPR8, (g+1)*LPR8)), so that a segmented shuffle of width LPR8 with an
// IMMEDIATE source lane hands every group its own edge: no per-lane index arithmetic.  Full batches take a
// branch-free unrolled path, the row's last partial batch a predicated loop.  The (col, val) pair of the
// next batch is loaded before the current batch's gathers are issued, so a row's dependent-latency chain is
// rowptr -> col/val -> gathers, gathers, ... instead of alternating col/val and gather round trips.
// The static L2 eviction priorities exist only on 256-bit loads (ptxas: "requires .v8.b32/.v4.b64 type with
// .L2::evict_last"): a hot column (bit 31, kHot) selects between two predicated LDG.256 - no cache-policy
// descriptor, no uniform-register traffic.  Summation order: fixed per row (group-local edge order, then
// the xor tree), i.e. bit-reproducible, but different from the 128-bit kernel's.
struct f8 {
  float4 a, b;
};
__device__ __forceinline__ f8 ld_gather_f8(const float* p) {
  f8 v;
  asm("ld.global.nc.L1::no_allocate.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
      : "=f"(v.a.x), "=f"(v.a.y), "=f"(v.a.z), "=f"(v.a.w), "=f"(v.b.x), "=f"(v.b.y), "=f"(v.b.z), "=f"(v.b.w)
      : "l"(p));
  return v;
}
__device__ __forceinline__ f8 ld_gather_f8_last(const float* p) {
  f8 v;
  asm("ld.global.nc.L1::no_allocate.L2::evict_last.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
      : "=f"(v.a.x), "=f"(v.a.y), "=f"(v.a.z), "=f"(v.a.w), "=f"(v.b.x), "=f"(v.b.y), "=f"(v.b.z), "=f"(v.b.w)
      : "l"(p));
  return v;
}
__device__ __forceinline__ f8 ld_gather_f8_first(const float* p) {
  f8 v;
  asm("ld.global.nc.L1::no_allocate.L2::evict_first.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
      : "=f"(v.a.x), "=f"(v.a.y), "=f"(v.a.z), "=f"(v.a.w), "=f"(v.b.x), "=f"(v.b.y), "=f"(v.b.z), "=f"(v.b.w)
      : "l"(p));
  return v;
}
// kCold: the L2 priority of a column without the hot bit - evict_first (kCold) or the default one.  Hot columns
// (kHot and bit 31 set) always load with evict_last.
template <int D, bool kHot, bool kCold = kHot>
__device__ __forceinline__ f8 gather_row8(const float* Xs, int cc) {
  // one IMAD.WIDE.U32 (left to itself the compiler builds the 64-bit product from two shifts, two masks and
  // a carry chain: 6 instructions per gather)
  const float* p;
  asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(p) : "r"(kHot ? (uint32_t)cc & 0x7fffffffu : (uint32_t)cc), "n"(D * 4), "l"(Xs));
  if (kHot) return cc < 0 ? ld_gather_f8_last(p) : (kCold ? ld_gather_f8_first(p) : ld_gather_f8(p));
  return kCold ? ld_gather_f8_first(p) : ld_gather_f8(p);
}
__device__ __forceinline__ void f8_fma(f8& acc, float s, const f8& x) {
  f4_fma(acc.a, s, x.a);
  f4_fma(acc.b, s, x.b);
}

// One 32-edge batch of a row or segment: rem (> 0) = edges left from the batch's first edge on, (c, v) = this
// lane's edge of the batch.  Group g adds batch edges [g*LPR8, (g+1)*LPR8) to acc in edge order.
template <int D, int U, bool kHot, bool kCold = kHot>
__device__ __forceinline__ void batch_accumulate8(f8& acc, const float* Xs, int c, float v, int rem, int grp) {
  constexpr int LPR8 = D / 8;          // lanes per row = edges per group per batch = shuffle width
  static_assert(LPR8 % U == 0, "U must divide the group's share of a batch");
  if (rem >= 32) {
#pragma unroll
    for (int k0 = 0; k0 < LPR8; k0 += U) {
      f8 x[U];
      float vv[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int cc = __shfl_sync(kFull, c, k0 + u, LPR8);
        vv[u] = __shfl_sync(kFull, v, k0 + u, LPR8);
        x[u] = gather_row8<D, kHot, kCold>(Xs, cc);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) f8_fma(acc, vv[u], x[u]);
    }
  } else {
    const int ng = rem - grp * LPR8;              // edges of this group (<= 0: none)
    const int nmax = rem < LPR8 ? rem : LPR8;     // group 0 holds the most
#pragma unroll 1
    for (int k0 = 0; k0 < nmax; k0 += U) {
      f8 x[U];
      float vv[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int cc = __shfl_sync(kFull, c, k0 + u, LPR8);
        vv[u] = __shfl_sync(kFull, v, k0 + u, LPR8);
        if (k0 + u < ng) {
          x[u] = gather_row8<D, kHot, kCold>(Xs, cc);
        } else {
          x[u].a = f4_zero();
          x[u].b = f4_zero();
          vv[u] = 0.f;
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) f8_fma(acc, vv[u], x[u]);
    }
  }
}

// the fixed xor tree over the lane groups: afterwards every group holds the whole row
template <int D>
__device__ __forceinline__ void groups_reduce8(f8& acc) {
#pragma unroll
  for (int m = D / 8; m < 32; m <<= 1) {
    f4_add(acc.a, f4_shfl_xor(acc.a, m));
    f4_add(acc.b, f4_shfl_xor(acc.b, m));
  }
}

// Sum over CSR edges [start, end) of val[e] * X[col[e], :]; returns, in the 128-bit kernels' layout (lane l <
// D/4 holds floats [4l, 4l+4)), the finished row.  U = gathers in flight per lane before the first FMA.
template <int D, int U, bool kHot>
__device__ __forceinline__ float4 warp_row_accumulate8(const int32_t* __restrict__ col,
                                                       const float* __restrict__ val,
                                                       const float* __restrict__ X, int64_t start,
                                                       int64_t end, int lane) {
  constexpr int LPR8 = D / 8;
  const int grp = lane / LPR8, sub = lane % LPR8;
  const float* Xs = X + sub * 8;
  f8 acc;
  acc.a = f4_zero();
  acc.b = f4_zero();
  int rem = (int)(end - start);        // a row has < 2^31 edges (columns are int32 and unique)
  const int32_t* cp = col + start + lane;
  const float* vp = val + start + lane;
  int c = 0;
  float v = 0.f;
  if (lane < rem) {
    c = ld_stream_s32(cp);
    v = ld_stream_f32(vp);
  }
  while (rem > 0) {
    int cn = 0;
    float vn = 0.f;
    if (lane + 32 < rem) {             // next batch's (col, val): in flight during this batch's gathers
      cn = ld_stream_s32(cp + 32);
      vn = ld_stream_f32(vp + 32);
    }
    batch_accumulate8<D, U, kHot>(acc, Xs, c, v, rem, grp);
    c = cn;
    v = vn;
    cp += 32;
    vp += 32;
    rem -= 32;
  }
  groups_reduce8<D>(acc);
  // lane l of the 128-bit layout takes half (l & 1) of lane l / 2
  const int src = (lane >> 1) & (LPR8 - 1);
  float4 lo, hi;
  lo.x = __shfl_sync(kFull, acc.a.x, src);
  lo.y = __shfl_sync(kFull, acc.a.y, src);
  lo.z = __shfl_sync(kFull, acc.a.z, src);
  lo.w = __shfl_sync(kFull, acc.a.w, src);
  hi.x = __shfl_sync(kFull, acc.b.x, src);
  hi.y = __shfl_sync(kFull, acc.b.y, src);
  hi.z = __shfl_sync(kFull, acc.b.z, src);
  hi.w = __shfl_sync(kFull, acc.b.w, src);
  return (lane & 1) ? hi : lo;
}

// 256-bit gathers in flight per lane before the first FMA (x 32 B x 32 lanes = bytes in flight per warp) and
// the CTAs-per-SM floor that fixes the register budget (32 -> 64 registers).  Tuning builds: -DSPEX_V8_U=8
// -DSPEX_V8_MINB=20 (8 KB in flight per warp, 20 warps per SM).
#ifndef SPEX_V8_U
#define SPEX_V8_U 4
#endif
#ifndef SPEX_MASK_U
#define SPEX_MASK_U 2
#endif
#ifndef SPEX_V8_MINB
#define SPEX_V8_MINB 32
#endif
// The same sum when most rows of X are known to be ZERO (nz[c] != 0 marks the rows that may be non-zero): the
// second layer of the training backward reads H_1 = g + A^T g, which is non-zero only on the batch's rows and
// their neighbours (~8 % of the edges on the bench graph).  Every lane looks up the byte of its own edge, one
// ballot gives the batch's active edges, and every lane group walks the active edges AMONG ITS OWN eight in
// ascending order - the edges the dense kernel would give it, in the same order, minus terms val * (+0) that
// cannot change a sum (values and zero rows are non-negative zeros) - so the result is bit-identical to the
// dense kernel's.  (col, val) run two batches ahead and the mask byte one batch ahead, so a batch still exposes
// a single dependent latency (its gathers).
template <int D, bool kHot>
__device__ __forceinline__ float4 warp_row_accumulate8_masked(const int32_t* __restrict__ col,
                                                              const float* __restrict__ val,
                                                              const float* __restrict__ X,
                                                              const uint8_t* __restrict__ nz, int64_t start,
                                                              int64_t end, int lane) {
  constexpr int LPR8 = D / 8;
  // active edges taken per lane group and loop trip: with ~8 % of the edges active a group of 8 holds 0-2 of
  // them, and every slot of a trip costs its shuffles and predicates whether it is used or not (ncu: U = 4 left
  // the kernel instruction-bound at 7.4 warp instructions per edge)
  constexpr int U = SPEX_MASK_U;
  const int grp = lane / LPR8, sub = lane % LPR8;
  const float* Xs = X + sub * 8;
  f8 acc;
  acc.a = f4_zero();
  acc.b = f4_zero();
  int rem = (int)(end - start);
  const int32_t* cp = col + start + lane;
  const float* vp = val + start + lane;
  constexpr uint32_t kIdMask = kHot ? 0x7fffffffu : 0xffffffffu;
  int c = 0, cn = 0;
  float v = 0.f, vn = 0.f;
  bool on = false;
  if (lane < rem) {
    c = ld_stream_s32(cp);
    v = ld_stream_f32(vp);
  }
  if (lane + 32 < rem) {
    cn = ld_stream_s32(cp + 32);
    vn = ld_stream_f32(vp + 32);
  }
  if (lane < rem) on = nz[(uint32_t)c & kIdMask] != 0;
  while (rem > 0) {
    int c2 = 0;
    float v2 = 0.f;
    if (lane + 64 < rem) {
      c2 = ld_stream_s32(cp + 64);
      v2 = ld_stream_f32(vp + 64);
    }
    bool onn = false;
    if (lane + 32 < rem) onn = nz[(uint32_t)cn & kIdMask] != 0;
    const unsigned act = __ballot_sync(kFull, on);
    unsigned mine = (act >> (grp * LPR8)) & (LPR8 == 32 ? 0xffffffffu : ((1u << LPR8) - 1u));
#pragma unroll 1
    while (__any_sync(kFull, mine != 0)) {
      f8 x[U];
      float vv[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const bool has = mine != 0;
        const int src = grp * LPR8 + (has ? __ffs(mine) - 1 : 0);
        mine &= mine - 1;
        const int cc = __shfl_sync(kFull, c, src);
        vv[u] = __shfl_sync(kFull, v, src);
        if (has) {
          x[u] = gather_row8<D, kHot>(Xs, cc);
        } else {
          x[u].a = f4_zero();
          x[u].b = f4_zero();
          vv[u] = 0.f;
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) f8_fma(acc, vv[u], x[u]);
    }
    c = cn;
    v = vn;
    on = onn;
    cn = c2;
    vn = v2;
    cp += 32;
    vp += 32;
    rem -= 32;
  }
#pragma unroll
  for (int m = LPR8; m < 32; m <<= 1) {
    f4_add(acc.a, f4_shfl_xor(acc.a, m));
    f4_add(acc.b, f4_shfl_xor(acc.b, m));
  }
  const int src = (lane >> 1) & (LPR8 - 1);
  float4 lo, hi;
  lo.x = __shfl_sync(kFull, acc.a.x, src);
  lo.y = __shfl_sync(kFull, acc.a.y, src);
  lo.z = __shfl_sync(kFull, acc.a.z, src);
  lo.w = __shfl_sync(kFull, acc.a.w, src);
  hi.x = __shfl_sync(kFull, acc.b.x, src);
  hi.y = __shfl_sync(kFull, acc.b.y, src);
  hi.z = __shfl_sync(kFull, acc.b.z, src);
  hi.w = __shfl_sync(kFull, acc.b.w, src);
  return (lane & 1) ? hi : lo;
}

// kV8: 256-bit gathers (table 32-byte aligned), else the 128-bit version; kMask (with kV8): X is zero outside nz
template <int D, int U, bool kHot, bool kV8, bool kMask = false>
__device__ __forceinline__ float4 row_sum(const int32_t* __restrict__ col, const float* __restrict__ val,
                                          const float* __restrict__ X, int64_t start, int64_t end, int lane,
                                          const uint8_t* __restrict__ nz = nullptr) {
  if (kV8 && kMask) return warp_row_accumulate8_masked<D, kHot>(col, val, X, nz, start, end, lane);
  if (kV8) return warp_row_accumulate8<D, (D >= 64 ? SPEX_V8_U : D / 8), kHot>(col, val, X, start, end, lane);
  return warp_row_accumulate<D, U, false, kHot>(col, val, X, start, end, lane);
}

struct Epilogue {
  float* Y;
  const float* addend;
  float addend_scale;
  float* Z;
  float z_scale;
  // optional peer tables (fused all-gather: the Y row is also stored into every peer's copy)
  float* peer[8];
  int n_peers;
  int64_t peer_row_offset;
  // or ONE store to an NVSwitch multicast mapping of the peers' tables (NVLS): the switch
  // replicates it into every GPU's copy, so the row leaves this GPU once instead of P-1 times
  float* mcast;
  // piggy-backed publish (row partition, last layer): the warp that finishes output row r also copies
  // row r of `pub_src` (this rank's slice of the NEXT call's table) into every rank's table - one
  // multimem.st to `pub_mcast`, or P2P stores to `pub_peer[]` - so the E^(0) exchange of the next
  // propagation rides on the last layer's epilogue exactly like the Y rows of the other layers
  const float* pub_src;
  float* pub_mcast;
  float* pub_peer[8];
  int n_pub_peers;
  // fused optimiser (row partition, last layer of the BACKWARD propagation): Z of this row is the row's
  // gradient; the same warp applies dense Adam to the row of (adam_p, adam_m, adam_v) - torch.optim.Adam
  // arithmetic, identical to spex_adam_f32 - and publishes the UPDATED parameter row instead of pub_src
  float* adam_p;
  float* adam_m;
  float* adam_v;
  float adam_b1, adam_b2, adam_eps, adam_step_size, adam_bc2_sqrt;
  // added gradient (spex_spmm_layer_zadd_f32): rows with z_add_rows[i] != 0 get z += z_add[i, :] after the scale,
  // one fp32 add that Z and the fused Adam both see; the other rows never read z_add
  const float* z_add;
  const uint8_t* z_add_rows;
};

// z += row `row` of z_add (flagged rows only); __fadd_rn: an add of its own, never contracted into the scale's FMA
__device__ __forceinline__ void add_z_row(const Epilogue& ep, float4& z, int64_t row, int64_t off) {
  if (ep.z_add && ep.z_add_rows[row]) {
    const float4 g = ld_f4(ep.z_add + off);
    z.x = __fadd_rn(z.x, g.x);
    z.y = __fadd_rn(z.y, g.y);
    z.z = __fadd_rn(z.z, g.z);
    z.w = __fadd_rn(z.w, g.w);
  }
}

__device__ __forceinline__ void adam_update(float& pp, float gg, float& mm, float& vv, const Epilogue& ep) {
  mm = mm + (gg - mm) * (1.f - ep.adam_b1);               // exp_avg.lerp_(grad, 1-beta1)
  vv = vv * ep.adam_b2 + (1.f - ep.adam_b2) * gg * gg;    // exp_avg_sq.mul_(b2).addcmul_(g, g, 1-b2)
  const float denom = sqrtf(vv) / ep.adam_bc2_sqrt + ep.adam_eps;
  pp = pp - ep.adam_step_size * (mm / denom);             // param.addcdiv_(exp_avg, denom, -step_size)
}

template <int D>
__device__ __forceinline__ void row_epilogue(const Epilogue& ep, float4 acc, int64_t row, int lane) {
  constexpr int LPR = RowShape<D>::LPR;
  if (lane < LPR) {
    const int64_t off = row * D + lane * 4;
    if (ep.Y) *reinterpret_cast<float4*>(ep.Y + off) = acc;
    if (ep.mcast) {
      st_multimem_f4(ep.mcast + (row + ep.peer_row_offset) * D + lane * 4, acc);
    } else if (ep.n_peers > 0) {
      const int64_t poff = (row + ep.peer_row_offset) * D + lane * 4;
#pragma unroll
      for (int p = 0; p < 8; ++p)
        if (p < ep.n_peers) *reinterpret_cast<float4*>(ep.peer[p] + poff) = acc;
    }
    float4 z = acc;
    if (ep.Z || ep.adam_p) {
      float4 a = f4_zero();
      if (ep.addend) a = ld_f4(ep.addend + off);
      z.x = (a.x * ep.addend_scale + acc.x) * ep.z_scale;
      z.y = (a.y * ep.addend_scale + acc.y) * ep.z_scale;
      z.z = (a.z * ep.addend_scale + acc.z) * ep.z_scale;
      z.w = (a.w * ep.addend_scale + acc.w) * ep.z_scale;
      add_z_row(ep, z, row, off);
      if (ep.Z) *reinterpret_cast<float4*>(ep.Z + off) = z;
    }
    float4 pnew = f4_zero();
    if (ep.adam_p) {
      pnew = ld_f4(ep.adam_p + off);
      float4 mm = ld_f4(ep.adam_m + off), vv = ld_f4(ep.adam_v + off);
      adam_update(pnew.x, z.x, mm.x, vv.x, ep);
      adam_update(pnew.y, z.y, mm.y, vv.y, ep);
      adam_update(pnew.z, z.z, mm.z, vv.z, ep);
      adam_update(pnew.w, z.w, mm.w, vv.w, ep);
      *reinterpret_cast<float4*>(ep.adam_p + off) = pnew;
      *reinterpret_cast<float4*>(ep.adam_m + off) = mm;
      *reinterpret_cast<float4*>(ep.adam_v + off) = vv;
    }
    if (ep.pub_src || (ep.adam_p && (ep.pub_mcast || ep.n_pub_peers > 0))) {
      const float4 v = ep.adam_p ? pnew : ld_stream_f4(ep.pub_src + off);
      const int64_t poff = (row + ep.peer_row_offset) * D + lane * 4;
      if (ep.pub_mcast) {
        st_multimem_f4(ep.pub_mcast + poff, v);
      } else {
#pragma unroll
        for (int p = 0; p < 8; ++p)
          if (p < ep.n_pub_peers) *reinterpret_cast<float4*>(ep.pub_peer[p] + poff) = v;
      }
    }
  }
}

#ifndef SPEX_ROWS_PER_CTA
#define SPEX_ROWS_PER_CTA 1
#endif
#ifndef SPEX_U64
#define SPEX_U64 8
#endif
// One warp per CTA: measured on the 1B-interaction graph (K=3 step, ms): 8 warps/CTA 230.5, 4: 224.7,
// 2: 221.6, 1: 186.9 (U=8).  A CTA retires only when its slowest row is done, so with degrees from 1
// to 1024 multi-warp CTAs strand resident-warp slots; single-warp CTAs let the block scheduler
// backfill every slot (32 CTAs = 32 warps per SM at 63 registers).
constexpr int kRowsPerCta = SPEX_ROWS_PER_CTA;  // warps (= rows) per CTA

template <int D, int U, bool kHot, bool kV8, bool kMask>
__global__ void __launch_bounds__(kRowsPerCta * 32, SPEX_V8_MINB / kRowsPerCta)
spmm_rows_kernel(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                 const float* __restrict__ val, const float* __restrict__ X, int64_t n_rows,
                 int32_t skip_longer_than, Epilogue ep, const int32_t* __restrict__ row_sel,
                 const uint8_t* __restrict__ nz) {
  const int lane = threadIdx.x & 31;
  int64_t row = (int64_t)blockIdx.x * kRowsPerCta + (threadIdx.x >> 5);
  if (row >= n_rows) return;
  if (row_sel) row = row_sel[row];   // row subset (spex_spmm_layer_f32): n_rows = length of the list
  const int64_t start = rowptr[row], end = rowptr[row + 1];
  if (skip_longer_than > 0 && end > start + skip_longer_than) return;  // long-row path
  // sparse-input layers are bound by the per-row latency chain (rowptr -> col/val -> mask -> gathers -> addend):
  // ask L2 for the epilogue's addend row now (in the dense layers, which are throughput-bound, the same prefetch
  // measured no gain: profiles/r02_spmm_ldg256.md)
  if (kMask && ep.addend && lane < RowShape<D>::LPR && (lane & 7) == 0)
    asm volatile("prefetch.global.L2 [%0];" ::"l"(ep.addend + row * D + lane * 4));
  const float4 acc = row_sum<D, U, kHot, kV8, kMask>(col, val, X, start, end, lane, nz);
  row_epilogue<D>(ep, acc, row, lane);
}

// ---- long rows: the segment list of spex_long_plan ----------------------------------------------
// Hub rows (thousands of edges, columns spread over the whole table) are cut at fixed COLUMN-block
// boundaries, and these cells are listed in block-major order: at any moment the resident warps gather
// from one ~32 MB window of the table, which the 126 MB L2 keeps resident, so each table row of the
// window comes from HBM once instead of once per edge.  The other long rows (mid rows) are cut every
// seg_len edges.  warp per segment -> partial[seg, :]
template <int D, int U, bool kHot, bool kV8, bool kMask>
__global__ void __launch_bounds__(kRowsPerCta * 32, SPEX_V8_MINB / kRowsPerCta)
spmm_seg_list_kernel(const int32_t* __restrict__ col, const float* __restrict__ val,
                     const float* __restrict__ X, const int64_t* __restrict__ seg_start,
                     const int32_t* __restrict__ seg_count, int32_t n_seg, float* __restrict__ partial,
                     const int32_t* __restrict__ seg_sel, const uint8_t* __restrict__ nz) {
  constexpr int LPR = RowShape<D>::LPR;
  const int lane = threadIdx.x & 31;
  int seg = blockIdx.x * kRowsPerCta + (threadIdx.x >> 5);
  if (seg >= n_seg) return;
  if (seg_sel) seg = seg_sel[seg];   // subset: n_seg = length of the list
  const int64_t start = seg_start[seg];
  const float4 acc = row_sum<D, U, kHot, kV8, kMask>(col, val, X, start, start + seg_count[seg], lane, nz);
  if (lane < LPR) *reinterpret_cast<float4*>(partial + (int64_t)seg * D + lane * 4) = acc;
}

// Segments of the list per warp: a run of kHubRun consecutive hub cells (segments
// [0, n_hub_seg), block-major, so a run gathers from one window), or of kMidRun mid-row segments.  A hub cell
// has a median of ~31 edges: as a CTA of its own it was one partial batch, the tree and a store with nothing
// else in flight (and a CTA launch per cell).  Here the run's (start, count) pairs are loaded once, and the
// last batch of a cell loads the next cell's first (col, val) batch, so it is in flight during the current
// gathers, tree and store.
#ifndef SPEX_SEG_HUB_RUN
#define SPEX_SEG_HUB_RUN 8
#endif
#ifndef SPEX_SEG_MID_RUN
#define SPEX_SEG_MID_RUN 2
#endif
constexpr int kHubRun = SPEX_SEG_HUB_RUN, kMidRun = SPEX_SEG_MID_RUN;
static_assert(kHubRun <= 32 && kMidRun <= 32, "a run's segment extents are held one per lane");

// Segments [first, first + n) into their partial rows, each summed exactly as warp_row_accumulate8 sums it.
// kCold: L2 priority of the gathers (evict_first for mid rows, which have no reuse; the default priority for
// hub cells, whose window the block-major order exists to keep in L2).
template <int D, bool kHot, bool kCold>
__device__ __forceinline__ void seg_run8(const int32_t* __restrict__ col, const float* __restrict__ val,
                                         const float* __restrict__ X, const int64_t* __restrict__ seg_start,
                                         const int32_t* __restrict__ seg_count, int first, int n,
                                         float* __restrict__ partial, int lane) {
  constexpr int LPR8 = D / 8, U = D >= 64 ? SPEX_V8_U : D / 8;
  const int grp = lane / LPR8, sub = lane % LPR8;
  const float* Xs = X + sub * 8;
  int64_t my_start = 0;      // lane k < n: extent of segment first + k
  int my_cnt = 0;
  if (lane < n) {
    my_start = seg_start[first + lane];
    my_cnt = seg_count[first + lane];
  }
  int64_t start = __shfl_sync(kFull, my_start, 0);
  int rem = __shfl_sync(kFull, my_cnt, 0);
  int c = 0;
  float v = 0.f;
  if (lane < rem) {
    c = ld_stream_s32(col + start + lane);
    v = ld_stream_f32(val + start + lane);
  }
#pragma unroll 1
  for (int k = 0; k < n; ++k) {
    const int64_t nstart = __shfl_sync(kFull, my_start, (k + 1) & 31);
    const int ncnt = k + 1 < n ? __shfl_sync(kFull, my_cnt, (k + 1) & 31) : 0;
    f8 acc;
    acc.a = f4_zero();
    acc.b = f4_zero();
    int64_t e = start + lane;
#pragma unroll 1
    while (rem > 0) {
      int cn = 0;
      float vn = 0.f;
      if (rem > 32) {                  // next batch of this segment
        if (lane + 32 < rem) {
          cn = ld_stream_s32(col + e + 32);
          vn = ld_stream_f32(val + e + 32);
        }
      } else if (lane < ncnt) {        // first batch of the next segment
        cn = ld_stream_s32(col + nstart + lane);
        vn = ld_stream_f32(val + nstart + lane);
      }
      batch_accumulate8<D, U, kHot, kCold>(acc, Xs, c, v, rem, grp);
      c = cn;
      v = vn;
      e += 32;
      rem -= 32;
    }
    groups_reduce8<D>(acc);
    // group 0 stores the row (lane l: floats [8l, 8l+8)), streaming: the partials are read once by the fix-up
    // and must not push the window out of L2
    if (lane < LPR8) {
      float* p = partial + (int64_t)(first + k) * D + lane * 8;
      st_stream_f4(p, acc.a);
      st_stream_f4(p + 4, acc.b);
    }
    start = nstart;
    rem = ncnt;
  }
}

template <int D, bool kHot>
__global__ void __launch_bounds__(32, SPEX_V8_MINB)
spmm_seg_runs_kernel(const int32_t* __restrict__ col, const float* __restrict__ val, const float* __restrict__ X,
                     const int64_t* __restrict__ seg_start, const int32_t* __restrict__ seg_count, int32_t n_seg,
                     int32_t n_hub_seg, float* __restrict__ partial) {
  const int lane = threadIdx.x;
  const int hub_warps = (n_hub_seg + kHubRun - 1) / kHubRun;
  const int w = blockIdx.x;
  if (w < hub_warps) {
    const int first = w * kHubRun;
    const int n = min(kHubRun, n_hub_seg - first);
    seg_run8<D, kHot, false>(col, val, X, seg_start, seg_count, first, n, partial, lane);
  } else {
    const int first = n_hub_seg + (w - hub_warps) * kMidRun;
    if (first >= n_seg) return;
    const int n = min(kMidRun, n_seg - first);
    seg_run8<D, kHot, kHot>(col, val, X, seg_start, seg_count, first, n, partial, lane);
  }
}

// warp per long row: sum its partial rows in edge order (row_seg: a fixed order), then the epilogue
template <int D, int U>
__global__ void __launch_bounds__(kRowsPerCta * 32)
spmm_long_fix_list_kernel(const int32_t* __restrict__ long_rows,
                          const int32_t* __restrict__ long_segptr, const int32_t* __restrict__ row_seg,
                          int32_t n_long, const float* __restrict__ partial, Epilogue ep,
                          const int32_t* __restrict__ slot_sel) {
  const int lane = threadIdx.x & 31;
  int r = blockIdx.x * kRowsPerCta + (threadIdx.x >> 5);
  if (r >= n_long) return;
  if (slot_sel) r = slot_sel[r];     // subset: n_long = length of the list
  const float4 acc = warp_row_accumulate<D, U, true>(row_seg, nullptr, partial, long_segptr[r],
                                                     long_segptr[r + 1], lane);
  row_epilogue<D>(ep, acc, (int64_t)long_rows[r], lane);
}

// ---- generic D (multiple of 4, <= 512): one edge per step, lane owns float4 slots lane+32*v ----
template <int NV>
__global__ void __launch_bounds__(kRowsPerCta * 32)
spmm_rows_generic_kernel(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                         const float* __restrict__ val, const float* __restrict__ X,
                         int64_t n_rows, int32_t D, Epilogue ep) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * kRowsPerCta + (threadIdx.x >> 5);
  if (row >= n_rows) return;
  const int64_t start = rowptr[row], end = rowptr[row + 1];
  float4 acc[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) acc[v] = f4_zero();
  for (int64_t base = start; base < end; base += 32) {
    const int64_t e = base + lane;
    int c = 0;
    float w = 0.f;
    if (e < end) {
      c = ld_stream_s32(col + e);
      w = ld_stream_f32(val + e);
    }
    const int n = (int)((end - base) < 32 ? (end - base) : 32);
    for (int j = 0; j < n; ++j) {
      const int cc = __shfl_sync(kFull, c, j);
      const float ww = __shfl_sync(kFull, w, j);
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        const int d = (lane + 32 * v) * 4;
        if (d < D) f4_fma(acc[v], ww, ld_gather_f4(X + (int64_t)cc * D + d));
      }
    }
  }
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const int d = (lane + 32 * v) * 4;
    if (d < D) {
      const int64_t off = row * D + d;
      if (ep.Y) *reinterpret_cast<float4*>(ep.Y + off) = acc[v];
      if (ep.mcast) {
        st_multimem_f4(ep.mcast + (row + ep.peer_row_offset) * D + d, acc[v]);
      } else {
        for (int p = 0; p < ep.n_peers; ++p)
          *reinterpret_cast<float4*>(ep.peer[p] + (row + ep.peer_row_offset) * D + d) = acc[v];
      }
      if (ep.Z) {
        float4 a = f4_zero();
        if (ep.addend) a = ld_f4(ep.addend + off);
        float4 z;
        z.x = (a.x * ep.addend_scale + acc[v].x) * ep.z_scale;
        z.y = (a.y * ep.addend_scale + acc[v].y) * ep.z_scale;
        z.z = (a.z * ep.addend_scale + acc[v].z) * ep.z_scale;
        z.w = (a.w * ep.addend_scale + acc[v].w) * ep.z_scale;
        add_z_row(ep, z, row, off);
        *reinterpret_cast<float4*>(ep.Z + off) = z;
      }
    }
  }
}

static bool g_rows_only = false;   // spex_debug_spmm_rows: launch the short-row kernel alone

// Row subset of one layer (spex_spmm_layer_f32): only the listed rows are computed.  `rows` lists them all
// (the rows kernel skips the long ones exactly as in a full layer); the listed rows that take the long-row path
// are given again as slots into plan->long_rows, together with the ids of their segments, so that they run
// through the SAME segment -> partial -> fix-up sequence as in a full layer: a row's result does not depend on
// whether the layer was restricted.
struct RowSubset {
  const int32_t* rows;
  int64_t n_rows;
  const int32_t* long_slots;
  int32_t n_long;
  const int32_t* seg_ids;
  int32_t n_seg;
};

template <int D, int U, bool kHot, bool kV8, bool kMask>
static int launch_vec_h(const int64_t* rowptr, const int32_t* col, const float* val, const float* X,
                        int64_t n_rows, const Epilogue& ep, const spex_long_plan* plan,
                        cudaStream_t st, const RowSubset* sub, const uint8_t* nz) {
  const bool rows_only = g_rows_only;
  const bool has_long = plan && plan->n_long > 0;
  const int64_t n_work = sub ? sub->n_rows : n_rows;
  const int64_t grid = (n_work + kRowsPerCta - 1) / kRowsPerCta;
  if (grid > 0x7fffffffLL) return SPEX_E_TOOBIG;
  if (grid > 0) {
    spmm_rows_kernel<D, U, kHot, kV8, kMask><<<(unsigned)grid, kRowsPerCta * 32, 0, st>>>(
        rowptr, col, val, X, n_work, has_long ? plan->seg_len : 0, ep, sub ? sub->rows : nullptr, nz);
    count_launch();
  }
  if (rows_only) return check_last();
  if (has_long) {
    const int32_t n_seg = sub ? sub->n_seg : plan->n_seg;
    const int32_t n_long = sub ? sub->n_long : plan->n_long;
    const int32_t* seg_sel = sub ? sub->seg_ids : nullptr;
    const int32_t* slot_sel = sub ? sub->long_slots : nullptr;
    if (n_long == 0) return check_last();
    const int gs = (n_seg + kRowsPerCta - 1) / kRowsPerCta;
    const int gf = (n_long + kRowsPerCta - 1) / kRowsPerCta;
    // Runs of segments per warp pay off on a list with hub cells (a table larger than L2: millions of segments,
    // throughput-bound).  A list of mid-row segments only (a table that fits in L2) is short and on the layer's
    // critical path, so each of its segments gets a warp of its own (same bits either way).
    if (kV8 && !kMask && !sub && plan->n_hub_seg > 0) {
      const int n_mid = n_seg - plan->n_hub_seg;
      const int gr = (plan->n_hub_seg + kHubRun - 1) / kHubRun + (n_mid + kMidRun - 1) / kMidRun;
      spmm_seg_runs_kernel<D, kHot><<<gr, 32, 0, st>>>(col, val, X, plan->seg_start, plan->seg_count, n_seg,
                                                       plan->n_hub_seg, plan->partial);
    } else {
      spmm_seg_list_kernel<D, U, kHot, kV8, kMask><<<gs, kRowsPerCta * 32, 0, st>>>(
          col, val, X, plan->seg_start, plan->seg_count, n_seg, plan->partial, seg_sel, nz);
    }
    spmm_long_fix_list_kernel<D, U><<<gf, kRowsPerCta * 32, 0, st>>>(
        plan->long_rows, plan->long_segptr, plan->row_seg, n_long, plan->partial, ep, slot_sel);
    count_launch(2);
  }
  return check_last();
}

template <int D, int U>
static int launch_vec(const int64_t* rowptr, const int32_t* col, const float* val, const float* X,
                      int64_t n_rows, const Epilogue& ep, const spex_long_plan* plan,
                      cudaStream_t st, const RowSubset* sub, const uint8_t* nz) {
  // 256-bit gathers need a 32-byte aligned table (row pitch D*4 is a multiple of 32 for these D)
  const bool v8 = (reinterpret_cast<uintptr_t>(X) & 31u) == 0;
  const bool hot = plan && (plan->flags & SPEX_PLAN_COL_HOTBIT);
  if (nz && v8) {   // sparse-input variant (only with the 256-bit kernels; otherwise the mask is simply not used)
    if (hot) return launch_vec_h<D, U, true, true, true>(rowptr, col, val, X, n_rows, ep, plan, st, sub, nz);
    return launch_vec_h<D, U, false, true, true>(rowptr, col, val, X, n_rows, ep, plan, st, sub, nz);
  }
  if (hot) {
    if (v8) return launch_vec_h<D, U, true, true, false>(rowptr, col, val, X, n_rows, ep, plan, st, sub, nullptr);
    return launch_vec_h<D, U, true, false, false>(rowptr, col, val, X, n_rows, ep, plan, st, sub, nullptr);
  }
  if (v8) return launch_vec_h<D, U, false, true, false>(rowptr, col, val, X, n_rows, ep, plan, st, sub, nullptr);
  return launch_vec_h<D, U, false, false, false>(rowptr, col, val, X, n_rows, ep, plan, st, sub, nullptr);
}

int spmm_launch(const int64_t* rowptr, const int32_t* col, const float* val, const float* X,
                int64_t n_rows, int32_t D, const Epilogue& ep, const spex_long_plan* plan,
                cudaStream_t st, const RowSubset* sub = nullptr, const uint8_t* nz = nullptr) {
  SPEX_RETURN_IF(!rowptr || !X || n_rows < 0, SPEX_E_BADARG);
  SPEX_RETURN_IF(n_rows > 0 && (!col || !val), SPEX_E_BADARG);
  SPEX_RETURN_IF(D <= 0 || (D & 3) || D > 512, SPEX_E_BADDIM);
  SPEX_RETURN_IF(!aligned16(X) || !aligned16(ep.Y) || !aligned16(ep.Z) || !aligned16(ep.addend),
                 SPEX_E_ALIGN);
  SPEX_RETURN_IF(plan && (plan->flags & ~SPEX_PLAN_COL_HOTBIT), SPEX_E_BADARG);
  if (plan && plan->n_long > 0) {
    SPEX_RETURN_IF(plan->seg_len < 32 || !plan->long_rows || !plan->long_segptr ||
                       !plan->partial || plan->n_seg < plan->n_long,
                   SPEX_E_BADARG);
    SPEX_RETURN_IF(!plan->seg_start || !plan->seg_count || !plan->row_seg, SPEX_E_BADARG);
    SPEX_RETURN_IF(plan->n_hub_seg < 0 || plan->n_hub_seg > plan->n_seg, SPEX_E_BADARG);
    SPEX_RETURN_IF(!aligned16(plan->partial), SPEX_E_ALIGN);
  }
  if (n_rows == 0) return 0;
  switch (D) {
    case 32: return launch_vec<32, 4>(rowptr, col, val, X, n_rows, ep, plan, st, sub, nz);
    case 64: return launch_vec<64, SPEX_U64>(rowptr, col, val, X, n_rows, ep, plan, st, sub, nz);
    case 128: return launch_vec<128, 8>(rowptr, col, val, X, n_rows, ep, plan, st, sub, nz);
    default: break;
  }
  SPEX_RETURN_IF(sub != nullptr, SPEX_E_BADDIM);   // row subsets: D in {32, 64, 128} only (a mask is just ignored)
  SPEX_RETURN_IF(plan && (plan->flags & SPEX_PLAN_COL_HOTBIT), SPEX_E_BADDIM);  // D in {32,64,128} only
  SPEX_RETURN_IF(ep.pub_src != nullptr || ep.adam_p != nullptr, SPEX_E_BADDIM);  // same
  // generic path handles long rows serially (no plan needed; still deterministic)
  const int64_t grid = (n_rows + kRowsPerCta - 1) / kRowsPerCta;
  if (grid > 0x7fffffffLL) return SPEX_E_TOOBIG;
  const int nv = (D + 127) / 128;
  switch (nv) {
    case 1: spmm_rows_generic_kernel<1><<<(unsigned)grid, kRowsPerCta * 32, 0, st>>>(rowptr, col, val, X, n_rows, D, ep); break;
    case 2: spmm_rows_generic_kernel<2><<<(unsigned)grid, kRowsPerCta * 32, 0, st>>>(rowptr, col, val, X, n_rows, D, ep); break;
    case 3: spmm_rows_generic_kernel<3><<<(unsigned)grid, kRowsPerCta * 32, 0, st>>>(rowptr, col, val, X, n_rows, D, ep); break;
    default: spmm_rows_generic_kernel<4><<<(unsigned)grid, kRowsPerCta * 32, 0, st>>>(rowptr, col, val, X, n_rows, D, ep); break;
  }
  count_launch();
  return check_last();
}

// scale-copy used for K == 0 (out = E0) and the K == 0 backward (dE0 = g)
__global__ void copy_f4_kernel(const float4* __restrict__ src, float4* __restrict__ dst, int64_t n4) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < n4; i += stride) dst[i] = src[i];
}

// all-gather of one rank's row slice by P2P stores: every 16-byte element is read once and stored
// into each peer's table (the own table is just one more destination).  Peer p of block b is
// visited starting at (b + p) so that the ranks' stores spread over the NVSwitch ports.
struct PeerTables {
  float* peer[8];
  int n_peers;
};
__global__ void __launch_bounds__(256)
push_rows_kernel(const float4* __restrict__ src, int64_t n4, int64_t dst_off4, PeerTables pt) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int rot = blockIdx.x % pt.n_peers;
  for (; i < n4; i += stride) {
    const float4 v = ld_stream_f4(reinterpret_cast<const float*>(src + i));
#pragma unroll
    for (int p = 0; p < 8; ++p) {
      if (p < pt.n_peers) {
        int q = p + rot;
        if (q >= pt.n_peers) q -= pt.n_peers;
        reinterpret_cast<float4*>(pt.peer[q])[dst_off4 + i] = v;
      }
    }
  }
}

// the same all-gather with ONE multicast store per element (NVLS)
__global__ void __launch_bounds__(256)
mcast_rows_kernel(const float4* __restrict__ src, int64_t n4, float* __restrict__ mcast_dst) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < n4; i += stride)
    st_multimem_f4(mcast_dst + 4 * i, ld_stream_f4(reinterpret_cast<const float*>(src + i)));
}

__global__ void gather_scale_kernel(const float* __restrict__ src, const int64_t* __restrict__ idx,
                                    const float* __restrict__ scale, float divisor,
                                    float* __restrict__ out, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    float v = idx ? src[idx[i]] : src[i];
    if (scale) v *= scale[i];
    if (divisor != 1.f) v = v / divisor;  // IEEE fp32 division, as torch's values / keep_prob
    out[i] = v;
  }
}

// The 24-bit draw (h >> 40) of edge (r, c) of the counter-based dropout mask (spex_edge_dropout_f32).
__device__ __forceinline__ uint32_t edge_draw(uint64_t seed, uint32_t r, uint32_t c) {
  return (uint32_t)(splitmix64(seed ^ (((uint64_t)r << 32) | c)) >> 40);
}

constexpr int kDropChunk = 1024;   // contiguous edges per warp and chunk: one row search per chunk
constexpr int kDropUnroll = 4;     // edges per lane in flight

// val_out / valT_out of the edge-dropped graph in one pass.  A warp takes a chunk of kDropChunk edges, finds the
// row of its first edge by binary search and walks forward from there: each lane advances its row over the row
// ends it passes, so an empty row costs one step and a hub row none.  col, val, tpos and both outputs are read
// and written coalesced, 32 consecutive edges per warp instruction.
template <bool kT, bool kTpos>
__global__ void __launch_bounds__(256)
edge_dropout_kernel(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                    const float* __restrict__ val, const int64_t* __restrict__ tpos, int64_t n_rows,
                    int64_t row_offset, uint64_t seed, float keep_prob, float* __restrict__ val_out,
                    float* __restrict__ valT_out) {
  // keep = int(RN(u + keep_prob)) != 0 with u = draw * 2^-24 is nondecreasing in the draw, so it is the test
  // draw >= k_min; k_min (2^24: nothing kept) is found by bisection with the same fp32 operations.
  uint32_t k_min = 0, k_hi = 1u << 24;
  while (k_min < k_hi) {
    const uint32_t mid = (k_min + k_hi) >> 1;
    if (__float2int_rz(__fadd_rn(__uint2float_rn(mid) * 0x1p-24f, keep_prob)) != 0) k_hi = mid; else k_min = mid + 1;
  }
  // (v * keep) / keep_prob is v / keep_prob for a kept edge and v * 0 (the same signed zero) for a dropped one
  const bool divide = keep_prob != 1.f;
  const int lane = threadIdx.x & (kWarp - 1);
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x / kWarp);
  const int64_t e_end = __ldg(rowptr + n_rows);
  for (int64_t c0 = __ldg(rowptr) + ((int64_t)blockIdx.x * (blockDim.x / kWarp) + threadIdx.x / kWarp) * kDropChunk;
       c0 < e_end; c0 += warps * kDropChunk) {
    int64_t lo = 0, hi = n_rows;   // rowptr[lo] <= c0 < rowptr[hi]: lo ends at the last row starting at or before c0
    while (hi - lo > 1) {
      const int64_t mid = (lo + hi) >> 1;
      if (__ldg(rowptr + mid) <= c0) lo = mid; else hi = mid;
    }
    int64_t row = lo;
    int32_t row_end = (int32_t)(__ldg(rowptr + row + 1) - c0);   // chunk-relative from here on
    const int n = (int)min((int64_t)kDropChunk, e_end - c0);
    const int32_t* cc = col + c0;
    const float* vc = val + c0;
    float* oc = val_out + c0;
    float* ot = kT ? valT_out + c0 : nullptr;
    for (int i0 = lane; i0 < n; i0 += kDropUnroll * kWarp) {
      uint32_t cv[kDropUnroll];   // the loads of kDropUnroll edges are issued before any of them is used
      float v[kDropUnroll], vt[kDropUnroll];
#pragma unroll
      for (int k = 0; k < kDropUnroll; ++k) {
        const int i = i0 + k * kWarp;
        if (i < n) {
          cv[k] = (uint32_t)ld_stream_s32(cc + i) & 0x7fffffffu;
          v[k] = ld_stream_f32(vc + i);
          if (kT && kTpos) vt[k] = __ldg(val + __ldcs(tpos + c0 + i));
        }
      }
#pragma unroll
      for (int k = 0; k < kDropUnroll; ++k) {
        const int i = i0 + k * kWarp;
        if (i >= n) break;
        while (row_end <= i) row_end = (int32_t)(__ldg(rowptr + (++row) + 1) - c0);
        const uint32_t r = (uint32_t)(row + row_offset);
        const float q = divide ? v[k] / keep_prob : v[k];   // IEEE fp32 division, as gather_scale_kernel
        __stcs(oc + i, edge_draw(seed, r, cv[k]) >= k_min ? q : v[k] * 0.f);
        if (kT) {
          const float w = kTpos ? vt[k] : v[k];
          const float qt = !kTpos ? q : divide ? w / keep_prob : w;
          __stcs(ot + i, edge_draw(seed, cv[k], r) >= k_min ? qt : w * 0.f);
        }
      }
    }
  }
}

}  // namespace spex

using namespace spex;

extern "C" int spex_spmm_csr_f32(const int64_t* rowptr, const int32_t* col, const float* val,
                                 const float* X, int64_t n_rows, int32_t D, float* Y,
                                 const float* addend, float addend_scale, float* Z, float z_scale,
                                 const spex_long_plan* plan, void* stream) {
  Epilogue ep{};
  ep.Y = Y;
  ep.addend = addend;
  ep.addend_scale = addend_scale;
  ep.Z = Z;
  ep.z_scale = z_scale;
  ep.n_peers = 0;
  ep.peer_row_offset = 0;
  return spmm_launch(rowptr, col, val, X, n_rows, D, ep, plan, (cudaStream_t)stream);
}

// Translates a spex_spmm_epilogue into the kernels' Epilogue: the only check of epilogue arguments.
static int make_epilogue(const spex_spmm_epilogue* d, Epilogue& ep) {
  SPEX_RETURN_IF(!d || d->out_row_offset < 0, SPEX_E_BADARG);
  // Y exchange: at most one of a multicast table and up to 8 peer tables
  SPEX_RETURN_IF(d->y_mcast && d->n_y_peers > 0, SPEX_E_BADARG);
  SPEX_RETURN_IF(d->n_y_peers < 0 || d->n_y_peers > 8 || (d->n_y_peers > 0 && !d->y_peers_host), SPEX_E_BADARG);
  // publish: the rows of pub_src or the rows Adam updates, to exactly one destination
  const bool adam = d->adam_p || d->adam_m || d->adam_v;
  const bool pub_dst = d->pub_mcast || d->n_pub_peers > 0;
  SPEX_RETURN_IF(d->n_pub_peers < 0 || d->n_pub_peers > 8 || (d->n_pub_peers > 0 && !d->pub_peers_host),
                 SPEX_E_BADARG);
  SPEX_RETURN_IF(d->pub_mcast && d->n_pub_peers > 0, SPEX_E_BADARG);
  SPEX_RETURN_IF(d->pub_src && (adam || !pub_dst), SPEX_E_BADARG);
  SPEX_RETURN_IF(pub_dst && !d->pub_src && !adam, SPEX_E_BADARG);
  SPEX_RETURN_IF(adam && (!d->adam_p || !d->adam_m || !d->adam_v || d->step < 1), SPEX_E_BADARG);
  for (int p = 0; p < d->n_y_peers; ++p) SPEX_RETURN_IF(!d->y_peers_host[p], SPEX_E_BADARG);
  for (int p = 0; p < d->n_pub_peers; ++p) SPEX_RETURN_IF(!d->pub_peers_host[p], SPEX_E_BADARG);
  SPEX_RETURN_IF(!aligned16(d->Y) || !aligned16(d->addend) || !aligned16(d->Z) || !aligned16(d->y_mcast) ||
                     !aligned16(d->pub_src) || !aligned16(d->pub_mcast) || !aligned16(d->adam_p) ||
                     !aligned16(d->adam_m) || !aligned16(d->adam_v),
                 SPEX_E_ALIGN);
  for (int p = 0; p < d->n_y_peers; ++p) SPEX_RETURN_IF(!aligned16(d->y_peers_host[p]), SPEX_E_ALIGN);
  for (int p = 0; p < d->n_pub_peers; ++p) SPEX_RETURN_IF(!aligned16(d->pub_peers_host[p]), SPEX_E_ALIGN);
  ep.Y = d->Y;
  ep.addend = d->addend;
  ep.addend_scale = d->addend_scale;
  ep.Z = d->Z;
  ep.z_scale = d->z_scale;
  ep.peer_row_offset = d->out_row_offset;
  ep.mcast = d->y_mcast;
  ep.n_peers = d->n_y_peers;
  for (int p = 0; p < d->n_y_peers; ++p) ep.peer[p] = d->y_peers_host[p];
  ep.pub_src = d->pub_src;
  ep.pub_mcast = d->pub_mcast;
  ep.n_pub_peers = d->n_pub_peers;
  for (int p = 0; p < d->n_pub_peers; ++p) ep.pub_peer[p] = d->pub_peers_host[p];
  if (adam) {
    ep.adam_p = d->adam_p;
    ep.adam_m = d->adam_m;
    ep.adam_v = d->adam_v;
    const double bc1 = 1.0 - pow((double)d->beta1, (double)d->step);
    const double bc2 = 1.0 - pow((double)d->beta2, (double)d->step);
    ep.adam_b1 = d->beta1;
    ep.adam_b2 = d->beta2;
    ep.adam_eps = d->eps;
    ep.adam_step_size = (float)((double)d->lr / bc1);
    ep.adam_bc2_sqrt = (float)sqrt(bc2);
  }
  return 0;
}

// One layer, optionally restricted to a row subset (the receptive field of a mini-batch: main_rec.py:34 calls
// computer() - all N rows of all K layers - for a batch of 256 users; the loss reads ~1.8 k rows of the result,
// which need E^(K-1) only on their neighbours, and so on).  rows: int32 [n_sel] row ids, any order, no
// duplicates; rows with degree > plan->seg_len are skipped by the rows kernel and must be given again as
// long_slots (their positions in plan->long_rows) with seg_ids = the ids of all their segments.  Every listed
// row gets exactly the value the full layer would give it; the other rows of the outputs are not touched.
extern "C" int spex_spmm_layer_zadd_f32(const int64_t* rowptr, const int32_t* col, const float* val, const float* X,
                                        int64_t n_rows, int32_t D, const int32_t* rows, int64_t n_sel,
                                        const int32_t* long_slots, int32_t n_long_sel, const int32_t* seg_ids,
                                        int32_t n_seg_sel, const uint8_t* x_nonzero,
                                        const spex_spmm_epilogue* epilogue, const float* z_add,
                                        const uint8_t* z_add_rows, const spex_long_plan* plan, void* stream) {
  SPEX_RETURN_IF(n_long_sel < 0 || n_seg_sel < 0 || (n_sel > 0 && !rows), SPEX_E_BADARG);
  SPEX_RETURN_IF(n_long_sel > 0 && (!long_slots || !seg_ids || !plan || n_seg_sel < n_long_sel), SPEX_E_BADARG);
  Epilogue ep{};
  const int rc = make_epilogue(epilogue, ep);
  if (rc) return rc;
  // the added gradient needs its row flags and a row it is added to (Z or the fused Adam's gradient)
  SPEX_RETURN_IF(!z_add != !z_add_rows || (z_add && !ep.Z && !ep.adam_p), SPEX_E_BADARG);
  SPEX_RETURN_IF(!aligned16(z_add), SPEX_E_ALIGN);
  ep.z_add = z_add;
  ep.z_add_rows = z_add_rows;
  if (n_sel == 0) return 0;
  RowSubset sub{rows, n_sel, long_slots, n_long_sel, seg_ids, n_seg_sel};
  return spmm_launch(rowptr, col, val, X, n_rows, D, ep, plan, (cudaStream_t)stream, n_sel < 0 ? nullptr : &sub,
                     x_nonzero);
}

extern "C" int spex_spmm_layer_f32(const int64_t* rowptr, const int32_t* col, const float* val, const float* X,
                                   int64_t n_rows, int32_t D, const int32_t* rows, int64_t n_sel,
                                   const int32_t* long_slots, int32_t n_long_sel, const int32_t* seg_ids,
                                   int32_t n_seg_sel, const uint8_t* x_nonzero, const spex_spmm_epilogue* epilogue,
                                   const spex_long_plan* plan, void* stream) {
  return spex_spmm_layer_zadd_f32(rowptr, col, val, X, n_rows, D, rows, n_sel, long_slots, n_long_sel, seg_ids,
                                  n_seg_sel, x_nonzero, epilogue, nullptr, nullptr, plan, stream);
}

// n_ctas == 0: the full-speed grid (8 CTAs per SM); > 0: a small grid for a BACKGROUND exchange that
// runs next to a layer kernel on a high-priority stream (the ingress of 7/8 of the table over
// NVLink, not this kernel's issue rate, bounds the exchange: 148 CTAs sustain ~600 GB/s of stores)
extern "C" int spex_mcast_rows_f32_ex(const float* src, int64_t n_rows, int32_t D, int64_t out_row_offset,
                                      float* mcast_Y, int32_t n_ctas, void* stream) {
  SPEX_RETURN_IF(!src || !mcast_Y || n_rows < 0 || out_row_offset < 0 || n_ctas < 0, SPEX_E_BADARG);
  SPEX_RETURN_IF(D <= 0 || (D & 3), SPEX_E_BADDIM);
  SPEX_RETURN_IF(!aligned16(src) || !aligned16(mcast_Y), SPEX_E_ALIGN);
  if (n_rows == 0) return 0;
  const unsigned grid = n_ctas > 0 ? (unsigned)n_ctas : 148u * 8u;
  mcast_rows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const float4*)src, n_rows * D / 4,
                                                            mcast_Y + out_row_offset * D);
  count_launch();
  return check_last();
}

extern "C" int spex_push_rows_f32_ex(const float* src, int64_t n_rows, int32_t D, int64_t out_row_offset,
                                     float* const* peer_Y_host, int32_t n_peers, int32_t n_ctas,
                                     void* stream) {
  SPEX_RETURN_IF(!src || n_rows < 0 || out_row_offset < 0 || !peer_Y_host || n_ctas < 0, SPEX_E_BADARG);
  SPEX_RETURN_IF(n_peers < 1 || n_peers > 8, SPEX_E_BADARG);
  SPEX_RETURN_IF(D <= 0 || (D & 3), SPEX_E_BADDIM);
  SPEX_RETURN_IF(!aligned16(src), SPEX_E_ALIGN);
  PeerTables pt{};
  pt.n_peers = n_peers;
  for (int p = 0; p < n_peers; ++p) {
    SPEX_RETURN_IF(!peer_Y_host[p] || !aligned16(peer_Y_host[p]), SPEX_E_BADARG);
    pt.peer[p] = peer_Y_host[p];
  }
  if (n_rows == 0) return 0;
  const int64_t n4 = n_rows * D / 4;
  const unsigned grid = n_ctas > 0 ? (unsigned)n_ctas : 148u * 8u;
  push_rows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const float4*)src, n4, out_row_offset * D / 4, pt);
  count_launch();
  return check_last();
}

extern "C" int spex_propagate_mean_f32(const int64_t* rowptr, const int32_t* col, const float* val,
                                       const float* E0, int64_t N, int32_t D, int32_t K, float* out,
                                       float* tmp0, float* tmp1, const spex_long_plan* plan,
                                       void* stream) {
  SPEX_RETURN_IF(!E0 || !out || N < 0 || K < 0, SPEX_E_BADARG);
  SPEX_RETURN_IF(D <= 0 || (D & 3) || D > 512, SPEX_E_BADDIM);
  SPEX_RETURN_IF((K >= 2 && !tmp0) || (K >= 3 && !tmp1), SPEX_E_BADARG);
  cudaStream_t st = (cudaStream_t)stream;
  if (N == 0) return 0;
  if (K == 0) {
    SPEX_RETURN_IF(!aligned16(E0) || !aligned16(out), SPEX_E_ALIGN);
    copy_f4_kernel<<<1184, 256, 0, st>>>((const float4*)E0, (float4*)out, N * D / 4);
    count_launch();
    return check_last();
  }
  const float inv = 1.0f / (float)(K + 1);
  float* tmp[2] = {tmp0, tmp1};
  const float* X = E0;
  for (int k = 0; k < K; ++k) {
    const bool last = (k == K - 1);
    Epilogue ep{};
    ep.Y = last ? nullptr : tmp[k & 1];
    ep.addend = (k == 0) ? E0 : out;
    ep.addend_scale = 1.f;
    ep.Z = out;
    ep.z_scale = last ? inv : 1.f;
    int rc = spmm_launch(rowptr, col, val, X, N, D, ep, plan, st);
    if (rc) return rc;
    X = tmp[k & 1];
  }
  return 0;
}

extern "C" int spex_propagate_mean_bwd_f32(const int64_t* rowptr, const int32_t* col,
                                           const float* valT, const float* g, int64_t N, int32_t D,
                                           int32_t K, float* dE0, float* tmp0, float* tmp1,
                                           const spex_long_plan* plan, void* stream) {
  SPEX_RETURN_IF(!g || !dE0 || N < 0 || K < 0, SPEX_E_BADARG);
  SPEX_RETURN_IF(D <= 0 || (D & 3) || D > 512, SPEX_E_BADDIM);
  SPEX_RETURN_IF((K >= 2 && !tmp0) || (K >= 3 && !tmp1), SPEX_E_BADARG);
  cudaStream_t st = (cudaStream_t)stream;
  if (N == 0) return 0;
  if (K == 0) {
    SPEX_RETURN_IF(!aligned16(g) || !aligned16(dE0), SPEX_E_ALIGN);
    copy_f4_kernel<<<1184, 256, 0, st>>>((const float4*)g, (float4*)dE0, N * D / 4);
    count_launch();
    return check_last();
  }
  // H_K = g; H_k = g + A^T H_{k+1}; dE0 = H_0 / (K+1)
  const float inv = 1.0f / (float)(K + 1);
  float* tmp[2] = {tmp0, tmp1};
  const float* X = g;
  for (int j = 1; j <= K; ++j) {
    const bool last = (j == K);
    Epilogue ep{};
    ep.Y = nullptr;
    ep.addend = g;
    ep.addend_scale = 1.f;
    ep.Z = last ? dE0 : tmp[(j - 1) & 1];
    ep.z_scale = last ? inv : 1.f;
    int rc = spmm_launch(rowptr, col, valT, X, N, D, ep, plan, st);
    if (rc) return rc;
    X = tmp[(j - 1) & 1];
  }
  return 0;
}

extern "C" int spex_gather_f32(const float* src, const int64_t* idx, const float* scale,
                               float divisor, float* out, int64_t n, void* stream) {
  SPEX_RETURN_IF(!src || !out || n < 0 || divisor == 0.f, SPEX_E_BADARG);
  if (n == 0) return 0;
  int64_t blocks = (n + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  gather_scale_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(src, idx, scale, divisor, out, n);
  count_launch();
  return check_last();
}

extern "C" int spex_edge_dropout_f32(const int64_t* rowptr, const int32_t* col, const float* val, const int64_t* tpos,
                                     int64_t n_rows, int64_t row_offset, uint64_t seed, float keep_prob,
                                     float* val_out, float* valT_out, void* stream) {
  SPEX_RETURN_IF(!rowptr || !col || !val || !val_out || n_rows < 0 || row_offset < 0 ||
                     !(keep_prob > 0.f && keep_prob <= 1.f),
                 SPEX_E_BADARG);
  if (n_rows == 0) return 0;
  // the edge count lives on the device (rowptr[n_rows]): one resident wave of CTAs strides over the chunks
  auto kernel = !valT_out ? edge_dropout_kernel<false, false>
                : tpos    ? edge_dropout_kernel<true, true> : edge_dropout_kernel<true, false>;
  int ctas_per_sm = 0;
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, kernel, 256, 0);
  if (e != cudaSuccess) return (int)e;
  kernel<<<148 * ctas_per_sm, 256, 0, (cudaStream_t)stream>>>(rowptr, col, val, tpos, n_rows, row_offset, seed,
                                                             keep_prob, val_out, valT_out);
  count_launch();
  return check_last();
}

// ---- bring-up only (not part of the declared ABI) ------------------------------------------------
// short-row kernel alone over rows [row_begin, row_end) of the graph (the long-row passes are not
// launched; rows longer than plan->seg_len are still skipped): times the user-row and the item-row
// phases of a layer separately (profiles/microbench/spmm_phases.py)
extern "C" int spex_debug_spmm_rows(const int64_t* rowptr, const int32_t* col, const float* val,
                                    const float* X, int64_t row_begin, int64_t row_end, int32_t D,
                                    float* Y, const spex_long_plan* plan, void* stream) {
  Epilogue ep{};
  ep.Y = Y + row_begin * D;
  g_rows_only = true;
  const int rc = spmm_launch(rowptr + row_begin, col, val, X, row_end - row_begin, D, ep, plan,
                             (cudaStream_t)stream);
  g_rows_only = false;
  return rc;
}
