// score_topk_simt.cu — exact fp32 full-ranking top-k (CUDA-core path).
//
// north_star (3) / SURVEY §8 a5: getUsersRating (abstract at LightGCN_SPEX/code/utility1/model.py:
// 14-15) followed by top-k, with the user's training items excluded.  This is the bit-exact fp32
// companion of the tcgen05 bf16 scorer (score_topk_tc.cu): same ordering contract, same outputs;
// it serves small evaluations (epinion2: 3 185 x 12 407) and is the on-GPU cross-check of the
// tensor-core kernel.  Scores are never written to memory.
//
// CTA = 128 threads, TU users resident in shared memory, items streamed 128 per tile (one item
// row per thread, fp32 FMA against the broadcast user rows).  A score enters the candidate buffer
// only if it beats the user's current k-th score and is not a training item (binary search in the
// CSR row of R); buffers are merged into the per-user sorted list once per tile by a warp.
#include "topk.cuh"

namespace spex {

constexpr int TU = 8;        // users per CTA
constexpr int TILE = 128;    // items per tile == threads per CTA
constexpr int KMAX = 128;

// su[u][d] = U[rows[r0 + u]][d] for u < nu, zeros for the rows past nu: the CTA's user rows in shared memory
__device__ __forceinline__ void stage_user_rows(float* su, const float* U, int D, const int64_t* rows, int64_t r0,
                                                int nu, int tid) {
  for (int i = tid; i < TU * D; i += TILE) {
    const int u = i / D, d = i - u * D;
    su[i] = (u < nu) ? U[rows[r0 + u] * D + d] : 0.f;
  }
}

// acc[u] += <item_row, su + u * D> over D4 float4s, for the NU staged user rows (the callers start from zero): the
// one fp32 FMA chain of every score of this file (item element times user element, d ascending), so the top-k,
// rating and rank kernels agree bit for bit
template <int NU>
__device__ __forceinline__ void dot_rows(const float* item_row, const float* su, int D, int D4,
                                         float (&acc)[NU]) {
  const float4* row = reinterpret_cast<const float4*>(item_row);
#pragma unroll 4
  for (int d4 = 0; d4 < D4; ++d4) {
    const float4 x = __ldg(row + d4);
#pragma unroll
    for (int u = 0; u < NU; ++u) {
      const float4 w = *reinterpret_cast<const float4*>(su + u * D + d4 * 4);
      acc[u] = fmaf(x.x, w.x, acc[u]);
      acc[u] = fmaf(x.y, w.y, acc[u]);
      acc[u] = fmaf(x.z, w.z, acc[u]);
      acc[u] = fmaf(x.w, w.w, acc[u]);
    }
  }
}

// the score of one item row against one staged user row (one row: no row stride)
__device__ __forceinline__ float dot_f32(const float* item_row, const float* su_row, int D4) {
  float acc[1] = {0.f};
  dot_rows(item_row, su_row, 0, D4, acc);
  return acc[0];
}

__global__ void __launch_bounds__(TILE)
score_topk_simt_kernel(const float* __restrict__ U, const float* __restrict__ I, int D,
                       const int64_t* __restrict__ users, int64_t B, int64_t m_items,
                       const int64_t* __restrict__ mask_rowptr, const int32_t* __restrict__ mask_col,
                       int k, int32_t* __restrict__ out_idx, float* __restrict__ out_val) {
  extern __shared__ __align__(16) float smem[];
  float* su = smem;                                   // [TU][D]
  float* lv = su + TU * D;                            // [TU][KMAX]
  int* li = reinterpret_cast<int*>(lv + TU * KMAX);   // [TU][KMAX]
  float* cv = reinterpret_cast<float*>(li + TU * KMAX);  // [TU][TILE]
  int* ci = reinterpret_cast<int*>(cv + TU * TILE);      // [TU][TILE]
  __shared__ int cnt[TU];
  __shared__ int ln[TU];
  __shared__ float tau[TU];
  __shared__ int64_t mlo[TU], mhi[TU];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t u0 = (int64_t)blockIdx.x * TU;
  const int nu = (int)((B - u0) < TU ? (B - u0) : TU);

  stage_user_rows(su, U, D, users, u0, nu, tid);
  if (tid < TU) {
    cnt[tid] = 0;
    ln[tid] = 0;
    tau[tid] = -INFINITY;
    int64_t lo = 0, hi = 0;
    if (tid < nu && mask_rowptr) {
      const int64_t uid = users[u0 + tid];
      lo = mask_rowptr[uid];
      hi = mask_rowptr[uid + 1];
    }
    mlo[tid] = lo;
    mhi[tid] = hi;
  }
  __syncthreads();

  const int D4 = D >> 2;
  for (int64_t j0 = 0; j0 < m_items; j0 += TILE) {
    const int64_t j = j0 + tid;
    if (j < m_items) {
      float acc[TU];
#pragma unroll
      for (int u = 0; u < TU; ++u) acc[u] = 0.f;
      dot_rows(I + j * D, su, D, D4, acc);
#pragma unroll
      for (int u = 0; u < TU; ++u) {
        if (u < nu && (acc[u] > tau[u] || ln[u] < k)) {
          if (!mask_contains(mask_col, mlo[u], mhi[u], (int)j)) {
            const int slot = atomicAdd(&cnt[u], 1);  // integer smem atomic: order-free by contract
            cv[u * TILE + slot] = acc[u];
            ci[u * TILE + slot] = (int)j;
          }
        }
      }
    }
    __syncthreads();
    for (int u = warp; u < nu; u += TILE / 32) {
      const int c = cnt[u];
      if (c == 0) continue;
      int n = ln[u];
      for (int q = 0; q < c; ++q)
        warp_list_insert(lv + u * KMAX, li + u * KMAX, n, k, cv[u * TILE + q], ci[u * TILE + q], lane);
      if (lane == 0) {
        ln[u] = n;
        cnt[u] = 0;
        if (n == k) tau[u] = lv[u * KMAX + k - 1];
      }
    }
    __syncthreads();
  }

  for (int i = tid; i < nu * k; i += TILE) {
    const int u = i / k, p = i - u * k;
    const bool ok = p < ln[u];
    out_idx[(u0 + u) * k + p] = ok ? li[u * KMAX + p] : -1;
    out_val[(u0 + u) * k + p] = ok ? lv[u * KMAX + p] : -INFINITY;
  }
}


// Dense rating block  out[b, j] = f(<U[users[b]], I[j]>), f = sigmoid or identity: the API form of
// getUsersRating ([B, m_items] materialised).  Same tiling as the top-k kernel; stores are
// coalesced along items.
__global__ void __launch_bounds__(TILE)
rating_dense_kernel(const float* __restrict__ U, const float* __restrict__ I, int D,
                    const int64_t* __restrict__ users, int64_t B, int64_t m_items, int apply_sigmoid,
                    float* __restrict__ out) {
  extern __shared__ __align__(16) float smem[];
  float* su = smem;  // [TU][D]
  const int tid = threadIdx.x;
  const int64_t u0 = (int64_t)blockIdx.y * TU;
  const int nu = (int)((B - u0) < TU ? (B - u0) : TU);
  stage_user_rows(su, U, D, users, u0, nu, tid);
  __syncthreads();
  const int D4 = D >> 2;
  for (int64_t j = (int64_t)blockIdx.x * TILE + tid; j < m_items; j += (int64_t)gridDim.x * TILE) {
    float acc[TU];
#pragma unroll
    for (int u = 0; u < TU; ++u) acc[u] = 0.f;
    dot_rows(I + j * D, su, D, D4, acc);
#pragma unroll
    for (int u = 0; u < TU; ++u)
      if (u < nu) out[(u0 + u) * m_items + j] = apply_sigmoid ? 1.f / (1.f + expf(-acc[u])) : acc[u];
  }
}

// Rank of held-out pairs, exact fp32: CTA = TU pairs, items streamed through the threads as in the top-k kernel
// above.  Every score is dot_rows' FMA chain, as in the top-k kernel, so a pair's rank is the position of its
// item in the fp32 top-k list bit for bit.  Each thread counts, per pair, the items it scored that beat the
// held-out item t (score desc, id asc; t itself excluded) and un-counts the masked items of the user that beat
// it; the counts are reduced per pair in a fixed order (integers: order-free anyway).
__global__ void __launch_bounds__(TILE)
rank_pairs_f32_kernel(const float* __restrict__ U, const float* __restrict__ I, int D,
                      const int64_t* __restrict__ users, const int32_t* __restrict__ items, int64_t P,
                      int64_t m_items, const int64_t* __restrict__ mask_rowptr, const int32_t* __restrict__ mask_col,
                      int32_t* __restrict__ out_rank) {
  extern __shared__ __align__(16) float smem[];
  float* su = smem;                                   // [TU][D]
  __shared__ float s_st[TU];
  __shared__ int s_t[TU];
  __shared__ int part[TILE / 32][TU];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t p0 = (int64_t)blockIdx.x * TU;
  const int np = (int)((P - p0) < TU ? (P - p0) : TU);
  stage_user_rows(su, U, D, users, p0, np, tid);
  __syncthreads();
  const int D4 = D >> 2;
  if (tid < TU) {
    const int t = tid < np ? items[p0 + tid] : -1;
    s_t[tid] = t;
    s_st[tid] = t >= 0 ? dot_f32(I + (int64_t)t * D, su + tid * D, D4) : INFINITY;
  }
  __syncthreads();
  float st[TU];
  int tt[TU], cnt[TU];
#pragma unroll
  for (int u = 0; u < TU; ++u) {
    st[u] = s_st[u];
    tt[u] = s_t[u];
    cnt[u] = 0;
  }
  for (int64_t j = tid; j < m_items; j += TILE) {
    float acc[TU];
#pragma unroll
    for (int u = 0; u < TU; ++u) acc[u] = 0.f;
    dot_rows(I + j * D, su, D, D4, acc);
#pragma unroll
    for (int u = 0; u < TU; ++u) cnt[u] += ((int)j != tt[u] && beats(acc[u], (int)j, st[u], tt[u])) ? 1 : 0;
  }
#pragma unroll
  for (int u = 0; u < TU; ++u) {
    const int c = (int)__reduce_add_sync(kFull, (unsigned)cnt[u]);
    if (lane == 0) part[warp][u] = c;
  }
  if (mask_rowptr) {
    for (int u = 0; u < np; ++u) {
      const int64_t uid = users[p0 + u];
      const int64_t e = mask_rowptr[uid + 1];
      const int t = s_t[u];
      const float s = s_st[u];
      int c = 0;
      const int64_t b = mask_rowptr[uid];
      for (int64_t k = b + tid; k < e; k += TILE) {
        const int id = __ldg(mask_col + k);
        const bool first = k == b || __ldg(mask_col + k - 1) != id;   // a repeated mask id is subtracted once
        if (first && id != t && id >= 0 && id < m_items &&
            beats(dot_f32(I + (int64_t)id * D, su + u * D, D4), id, s, t))
          ++c;
      }
      c = (int)__reduce_add_sync(kFull, (unsigned)c);
      if (lane == 0) part[warp][u] -= c;
    }
  }
  __syncthreads();
  if (tid < np) {
    int c = 0;
#pragma unroll
    for (int w = 0; w < TILE / 32; ++w) c += part[w][tid];
    out_rank[p0 + tid] = c;
  }
}

}  // namespace spex

using namespace spex;

extern "C" int spex_rank_pairs_f32(const float* U, const float* I, int32_t D, const int64_t* users,
                                   const int32_t* items, int64_t P, int64_t m_items, const int64_t* mask_rowptr,
                                   const int32_t* mask_col, int32_t* out_rank, void* stream) {
  SPEX_RETURN_IF(D <= 0 || (D & 3) || D > 512, SPEX_E_BADDIM);
  SPEX_RETURN_IF(!U || !I || !users || !items || !out_rank || P < 0 || m_items < 0 || (P > 0 && m_items == 0),
                 SPEX_E_BADARG);
  SPEX_RETURN_IF((mask_rowptr == nullptr) != (mask_col == nullptr), SPEX_E_BADARG);
  SPEX_RETURN_IF(m_items > 0x7fffffffLL, SPEX_E_TOOBIG);
  SPEX_RETURN_IF(!aligned16(U) || !aligned16(I), SPEX_E_ALIGN);
  if (P == 0) return 0;
  const int64_t grid = (P + TU - 1) / TU;
  SPEX_RETURN_IF(grid > 0x7fffffffLL, SPEX_E_TOOBIG);
  rank_pairs_f32_kernel<<<(unsigned)grid, TILE, (size_t)TU * D * 4, (cudaStream_t)stream>>>(
      U, I, D, users, items, P, m_items, mask_rowptr, mask_col, out_rank);
  count_launch();
  return check_last();
}

extern "C" int spex_score_topk_f32(const float* U, const float* I, int32_t D, const int64_t* users,
                                   int64_t B, int64_t m_items, const int64_t* mask_rowptr,
                                   const int32_t* mask_col, int32_t k, int32_t* out_idx,
                                   float* out_val, void* stream) {
  SPEX_RETURN_IF(!U || !I || !users || !out_idx || !out_val || B < 0 || m_items < 0, SPEX_E_BADARG);
  SPEX_RETURN_IF((mask_rowptr == nullptr) != (mask_col == nullptr), SPEX_E_BADARG);
  SPEX_RETURN_IF(D <= 0 || (D & 3) || D > 512, SPEX_E_BADDIM);
  SPEX_RETURN_IF(k < 1 || k > KMAX || m_items > 0x7fffffffLL, SPEX_E_TOOBIG);
  SPEX_RETURN_IF(!aligned16(U) || !aligned16(I), SPEX_E_ALIGN);
  if (B == 0) return 0;
  const size_t smem = (size_t)TU * D * 4 + (size_t)TU * KMAX * 8 + (size_t)TU * TILE * 8;
  cudaStream_t st = (cudaStream_t)stream;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(score_topk_simt_kernel,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
  }
  const int64_t grid = (B + TU - 1) / TU;
  SPEX_RETURN_IF(grid > 0x7fffffffLL, SPEX_E_TOOBIG);
  score_topk_simt_kernel<<<(unsigned)grid, TILE, smem, st>>>(U, I, D, users, B, m_items, mask_rowptr,
                                                            mask_col, k, out_idx, out_val);
  count_launch();
  return check_last();
}

extern "C" int spex_rating_f32(const float* U, const float* I, int32_t D, const int64_t* users,
                               int64_t B, int64_t m_items, int32_t apply_sigmoid, float* out,
                               void* stream) {
  SPEX_RETURN_IF(!U || !I || !users || !out || B < 0 || m_items < 0, SPEX_E_BADARG);
  SPEX_RETURN_IF(D <= 0 || (D & 3) || D > 512, SPEX_E_BADDIM);
  SPEX_RETURN_IF(!aligned16(U) || !aligned16(I), SPEX_E_ALIGN);
  if (B == 0 || m_items == 0) return 0;
  const size_t smem = (size_t)TU * D * 4;
  int64_t gx = (m_items + TILE - 1) / TILE;
  if (gx > 148 * 8) gx = 148 * 8;
  const int64_t gy = (B + TU - 1) / TU;
  SPEX_RETURN_IF(gy > 65535, SPEX_E_TOOBIG);
  rating_dense_kernel<<<dim3((unsigned)gx, (unsigned)gy), TILE, smem, (cudaStream_t)stream>>>(
      U, I, D, users, B, m_items, apply_sigmoid, out);
  count_launch();
  return check_last();
}
