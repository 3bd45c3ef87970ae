// metrics.cu — full-ranking Recall / Precision / NDCG / hit rate at up to eight cutoffs, from a top-k block
// that stays on the device.
//
// One warp per user: lane l tests ranks l, l + 32, ... of the user's top-k row against the user's held-out
// items (a binary search in the sorted truth row), and a ballot per 32 ranks gives the hit ranks.  Every
// lane then walks the hit ranks in ascending order (uniform control flow), summing disc[i] into the DCG and
// counting hits; at each cutoff boundary the lane that owns that cutoff keeps the running pair.  Lane
// l < 4 n_cut owns metric l & 3 (recall, precision, ndcg, hit) of cutoff l >> 2, writes it to per_user and
// adds it to its chunk sum: n_cut <= 8 cutoffs x 4 metrics fill one warp exactly.
//
// Determinism without atomics: a block owns one chunk of SPEX_METRICS_CHUNK consecutive users; warp w sums
// users [w * 64, w * 64 + 64) of the chunk in ascending order, and thread l sums the warps' partials in
// ascending warp order.  The chunk sums are therefore a function of the chunk's per-user values alone, which
// makes the totals independent of how a caller splits its users into blocks (at chunk boundaries).
#include "common.cuh"

namespace spex {

constexpr int kMetricsWarps = 16;
constexpr int kUsersPerWarp = SPEX_METRICS_CHUNK / kMetricsWarps;
constexpr int kMaxK = 512;
constexpr int kMaxWords = kMaxK / kWarp;
static_assert(SPEX_METRICS_MAX_CUTOFFS * 4 == kWarp, "one lane per (cutoff, metric)");

struct MetricsCutoffs {
  int32_t c[SPEX_METRICS_MAX_CUTOFFS];
};

// is `target` in the ascending (duplicates allowed) row [lo, hi) of the truth columns?
__device__ __forceinline__ bool truth_has(const int32_t* __restrict__ col, int64_t lo, int64_t hi, int32_t target) {
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    const int32_t c = __ldg(col + mid);
    if (c == target) return true;
    if (c < target) lo = mid + 1; else hi = mid;
  }
  return false;
}

// metric my_m (recall, precision, ndcg, hit) at cutoff my_K of a user with T held-out items, my_h of them in the
// top my_K with DCG my_dcg
__device__ __forceinline__ double metric_value(int my_m, int my_h, double my_dcg, int my_K, int64_t T,
                                               const double* idcg) {
  double v;
  if (my_m == 0) {
    v = T > 0 ? (double)my_h / (double)T : 0.0;
  } else if (my_m == 1) {
    v = (double)my_h / (double)my_K;
  } else if (my_m == 2) {
    const double id = __ldg(idcg + (T < my_K ? T : (int64_t)my_K));
    v = id > 0.0 ? my_dcg / id : 0.0;
  } else {
    v = my_h > 0 ? 1.0 : 0.0;
  }
  return v;
}

// The walk of a user's hit ranks in ascending order reaches rank i with h hits and DCG acc before it: every cutoff
// c <= i is passed (c advances), and the lane that owns cutoff my_c keeps (h, acc) as its (my_h, my_dcg).
// i = INT_MAX passes the cutoffs left after the last hit.
__device__ __forceinline__ void pass_cutoffs(int i, int& c, int n_cut, const int32_t* s_cut, int my_c, int h,
                                             double acc, int& my_h, double& my_dcg) {
  for (; c < n_cut && i >= s_cut[c]; ++c)
    if (c == my_c) my_h = h, my_dcg = acc;
}

__global__ void __launch_bounds__(kMetricsWarps * kWarp)
fullrank_metrics_kernel(const int32_t* __restrict__ topk, int64_t B, int32_t k,
                        const int64_t* __restrict__ rowptr, const int32_t* __restrict__ tcol,
                        MetricsCutoffs cuts, int32_t n_cut, const double* __restrict__ disc,
                        const double* __restrict__ idcg, double* __restrict__ per_user,
                        double* __restrict__ chunk_sums) {
  __shared__ int32_t s_cut[SPEX_METRICS_MAX_CUTOFFS];
  __shared__ double s_part[kMetricsWarps][kWarp];
  if (threadIdx.x < SPEX_METRICS_MAX_CUTOFFS) s_cut[threadIdx.x] = cuts.c[threadIdx.x];
  __syncthreads();
  const int lane = threadIdx.x & (kWarp - 1);
  const int warp = threadIdx.x >> 5;
  const int nv = n_cut * 4;
  const int my_c = lane >> 2, my_m = lane & 3;
  const int my_K = s_cut[my_c < n_cut ? my_c : 0];
  const int nw = (k + kWarp - 1) / kWarp;
  const int64_t u0 = (int64_t)blockIdx.x * SPEX_METRICS_CHUNK + warp * kUsersPerWarp;
  double sum = 0.0;
  for (int t = 0; t < kUsersPerWarp; ++t) {
    const int64_t u = u0 + t;
    if (u >= B) break;
    const int64_t lo = __ldg(rowptr + u), hi = __ldg(rowptr + u + 1);
    const int32_t* row = topk + u * k;
    int32_t ids[kMaxWords];
#pragma unroll
    for (int j = 0; j < kMaxWords; ++j)
      ids[j] = (j < nw && j * kWarp + lane < k) ? __ldcs(row + j * kWarp + lane) : -1;
    double acc = 0.0, my_dcg = 0.0;
    int h = 0, c = 0, my_h = 0;
#pragma unroll
    for (int j = 0; j < kMaxWords; ++j) {
      if (j >= nw) break;
      const bool hit = j * kWarp + lane < k && truth_has(tcol, lo, hi, ids[j]);
      unsigned m = __ballot_sync(kFull, hit);
      while (m) {
        const int i = j * kWarp + __ffs(m) - 1;
        pass_cutoffs(i, c, n_cut, s_cut, my_c, h, acc, my_h, my_dcg);
        acc += __ldg(disc + i);
        ++h;
        m &= m - 1;
      }
    }
    pass_cutoffs(INT_MAX, c, n_cut, s_cut, my_c, h, acc, my_h, my_dcg);
    if (lane < nv) {
      const double v = metric_value(my_m, my_h, my_dcg, my_K, hi - lo, idcg);
      if (per_user) per_user[u * nv + lane] = v;
      sum += v;
    }
  }
  s_part[warp][lane] = sum;
  __syncthreads();
  if (threadIdx.x < nv) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kMetricsWarps; ++w) s += s_part[w][threadIdx.x];
    chunk_sums[(int64_t)blockIdx.x * nv + threadIdx.x] = s;
  }
}

// sums[l] = chunk_sums[0][l] + chunk_sums[1][l] + ...  in ascending chunk order
__global__ void __launch_bounds__(kWarp)
fullrank_metrics_reduce_kernel(const double* __restrict__ chunk_sums, int64_t n_chunks, int32_t nv,
                               double* __restrict__ sums) {
  const int l = threadIdx.x;
  if (l >= nv) return;
  double s = 0.0;
  for (int64_t c = 0; c < n_chunks; ++c) s += __ldg(chunk_sums + c * nv + l);
  sums[l] = s;
}

// Metrics from the ranks of the held-out items (spex_rank_pairs_*), one warp per user, chunks and summation order
// as fullrank_metrics_kernel: the hit ranks are walked in ascending order by a warp minimum per step, so the DCG
// is summed in the order the top-k path sums it.  A held-out item in the user's mask, or a repeat of the previous
// item of its truth row, is never a hit (its effective rank is INT_MAX).  Lanes 0 and 1 of each warp also sum MRR
// and AUC, into chunk_extra (mrr, auc, 0, 0) per chunk.
__global__ void __launch_bounds__(kMetricsWarps * kWarp)
rank_metrics_kernel(const int32_t* __restrict__ ranks, int64_t B, const int64_t* __restrict__ rowptr,
                    const int32_t* __restrict__ tcol, const int64_t* __restrict__ users,
                    const int64_t* __restrict__ mask_rowptr, const int32_t* __restrict__ mask_col, int64_t m_items,
                    MetricsCutoffs cuts, int32_t n_cut, const double* __restrict__ disc,
                    const double* __restrict__ idcg, double* __restrict__ chunk_sums,
                    double* __restrict__ chunk_extra) {
  __shared__ int32_t s_cut[SPEX_METRICS_MAX_CUTOFFS];
  __shared__ double s_part[kMetricsWarps][kWarp];
  __shared__ double s_extra[kMetricsWarps][2];
  if (threadIdx.x < SPEX_METRICS_MAX_CUTOFFS) s_cut[threadIdx.x] = cuts.c[threadIdx.x];
  __syncthreads();
  const int lane = threadIdx.x & (kWarp - 1);
  const int warp = threadIdx.x >> 5;
  const int nv = n_cut * 4;
  const int my_c = lane >> 2, my_m = lane & 3;
  const int my_K = s_cut[my_c < n_cut ? my_c : 0];
  const int Kmax = s_cut[n_cut - 1];
  const int64_t u0 = (int64_t)blockIdx.x * SPEX_METRICS_CHUNK + warp * kUsersPerWarp;
  double sum = 0.0, extra = 0.0;
  for (int t = 0; t < kUsersPerWarp; ++t) {
    const int64_t u = u0 + t;
    if (u >= B) break;
    const int64_t lo = __ldg(rowptr + u), hi = __ldg(rowptr + u + 1);
    int64_t mlo = 0, mhi = 0;
    if (mask_rowptr) {
      const int64_t uid = users[u];
      mlo = __ldg(mask_rowptr + uid);
      mhi = __ldg(mask_rowptr + uid + 1);
    }
    auto masked = [&](int64_t j) { return mask_rowptr && truth_has(mask_col, mlo, mhi, __ldg(tcol + j)); };
    // effective rank: INT_MAX for a masked item or a repeat
    auto eff = [&](int64_t j) {
      const bool rep = j > lo && __ldg(tcol + j) == __ldg(tcol + j - 1);
      return (rep || masked(j)) ? INT_MAX : __ldg(ranks + j);
    };
    int e_min = INT_MAX, n_live = 0;
    for (int64_t j = lo + lane; j < hi; j += kWarp) {
      const int e = eff(j);
      e_min = min(e_min, e);
      n_live += e != INT_MAX ? 1 : 0;
    }
    e_min = __reduce_min_sync(kFull, e_min);
    n_live = (int)__reduce_add_sync(kFull, (unsigned)n_live);
    double acc = 0.0, my_dcg = 0.0;
    int h = 0, c = 0, my_h = 0, prev = -1, next = e_min;
    while (next < Kmax) {
      pass_cutoffs(next, c, n_cut, s_cut, my_c, h, acc, my_h, my_dcg);
      acc += __ldg(disc + next);
      ++h;
      prev = next;
      int nx = INT_MAX;
      for (int64_t j = lo + lane; j < hi; j += kWarp) {
        const int e = eff(j);
        if (e > prev && e < nx) nx = e;
      }
      next = __reduce_min_sync(kFull, nx);
    }
    pass_cutoffs(INT_MAX, c, n_cut, s_cut, my_c, h, acc, my_h, my_dcg);
    const int64_t T = hi - lo;
    if (lane < nv) sum += metric_value(my_m, my_h, my_dcg, my_K, T, idcg);
    // AUC of each held-out item: 1 - (negatives above it) / n_neg, negatives = items outside mask and truth
    int n_mask = 0;                                     // distinct mask ids in [0, m_items): a repeat counts once
    for (int64_t k = mlo + lane; k < mhi; k += kWarp) {
      const int32_t id = __ldg(mask_col + k);
      n_mask += (id >= 0 && id < m_items && (k == mlo || __ldg(mask_col + k - 1) != id)) ? 1 : 0;
    }
    n_mask = (int)__reduce_add_sync(kFull, (unsigned)n_mask);
    const int64_t n_neg = m_items - n_mask - n_live;
    double auc = 0.0;
    for (int64_t j = lo + lane; j < hi; j += kWarp) {
      if (masked(j)) continue;
      const int r = __ldg(ranks + j);
      int above = 0;
      for (int64_t j2 = lo; j2 < hi; ++j2) above += eff(j2) < r ? 1 : 0;
      auc += n_neg > 0 ? 1.0 - (double)(r - above) / (double)n_neg : 1.0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) auc += __shfl_xor_sync(kFull, auc, o);
    if (lane == 0) extra += e_min != INT_MAX ? 1.0 / (1.0 + (double)e_min) : 0.0;
    if (lane == 1) extra += T > 0 ? auc / (double)T : 0.0;
  }
  s_part[warp][lane] = sum;
  if (lane < 2) s_extra[warp][lane] = extra;
  __syncthreads();
  if (threadIdx.x < nv) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kMetricsWarps; ++w) s += s_part[w][threadIdx.x];
    chunk_sums[(int64_t)blockIdx.x * nv + threadIdx.x] = s;
  }
  if (threadIdx.x < 4) {
    double s = 0.0;
    if (threadIdx.x < 2)
      for (int w = 0; w < kMetricsWarps; ++w) s += s_extra[w][threadIdx.x];
    chunk_extra[(int64_t)blockIdx.x * 4 + threadIdx.x] = s;
  }
}

}  // namespace spex

using namespace spex;

// the n_cut host cutoffs into `cuts`: SPEX_E_BADARG unless they are strictly ascending in [1, bound]
static int read_cutoffs(const int32_t* cutoffs_host, int32_t n_cut, int64_t bound, MetricsCutoffs* cuts) {
  *cuts = {};
  for (int i = 0; i < n_cut; ++i) {
    const int32_t K = cutoffs_host[i];
    SPEX_RETURN_IF(K < 1 || K > bound || (i > 0 && K <= cutoffs_host[i - 1]), SPEX_E_BADARG);
    cuts->c[i] = K;
  }
  return 0;
}

extern "C" int spex_rank_metrics(const int32_t* ranks, int64_t B, const int64_t* truth_rowptr,
                                 const int32_t* truth_col, const int64_t* users, const int64_t* mask_rowptr,
                                 const int32_t* mask_col, int64_t m_items, const int32_t* cutoffs_host, int32_t n_cut,
                                 const double* disc, const double* idcg, double* chunk_sums, double* chunk_extra,
                                 void* stream) {
  SPEX_RETURN_IF(n_cut > SPEX_METRICS_MAX_CUTOFFS || m_items > 0x7fffffffLL, SPEX_E_TOOBIG);
  SPEX_RETURN_IF(B < 0 || m_items < 1 || n_cut < 1 || !cutoffs_host || !disc || !idcg, SPEX_E_BADARG);
  SPEX_RETURN_IF((mask_rowptr == nullptr) != (mask_col == nullptr), SPEX_E_BADARG);
  MetricsCutoffs cuts;
  if (const int rc = read_cutoffs(cutoffs_host, n_cut, m_items, &cuts)) return rc;
  if (B == 0) return 0;
  SPEX_RETURN_IF(!ranks || !truth_rowptr || !truth_col || !chunk_sums || !chunk_extra ||
                     (mask_rowptr && !users),
                 SPEX_E_BADARG);
  const int64_t n_chunks = (B + SPEX_METRICS_CHUNK - 1) / SPEX_METRICS_CHUNK;
  rank_metrics_kernel<<<(unsigned)n_chunks, kMetricsWarps * kWarp, 0, (cudaStream_t)stream>>>(
      ranks, B, truth_rowptr, truth_col, users, mask_rowptr, mask_col, m_items, cuts, n_cut, disc, idcg, chunk_sums,
      chunk_extra);
  count_launch();
  return check_last();
}

extern "C" int spex_fullrank_metrics(const int32_t* topk_idx, int64_t B, int32_t k, const int64_t* truth_rowptr,
                                     const int32_t* truth_col, const int32_t* cutoffs_host, int32_t n_cut,
                                     const double* disc, const double* idcg, double* per_user, double* chunk_sums,
                                     void* stream) {
  SPEX_RETURN_IF(k > kMaxK || n_cut > SPEX_METRICS_MAX_CUTOFFS, SPEX_E_TOOBIG);
  SPEX_RETURN_IF(B < 0 || k < 1 || n_cut < 1 || !cutoffs_host || !disc || !idcg, SPEX_E_BADARG);
  MetricsCutoffs cuts;
  if (const int rc = read_cutoffs(cutoffs_host, n_cut, k, &cuts)) return rc;
  if (B == 0) return 0;
  SPEX_RETURN_IF(!topk_idx || !truth_rowptr || !truth_col || !chunk_sums, SPEX_E_BADARG);
  const int64_t n_chunks = (B + SPEX_METRICS_CHUNK - 1) / SPEX_METRICS_CHUNK;
  fullrank_metrics_kernel<<<(unsigned)n_chunks, kMetricsWarps * kWarp, 0, (cudaStream_t)stream>>>(
      topk_idx, B, k, truth_rowptr, truth_col, cuts, n_cut, disc, idcg, per_user, chunk_sums);
  count_launch();
  return check_last();
}

extern "C" int spex_fullrank_metrics_reduce(const double* chunk_sums, int64_t n_chunks, int32_t n_cut, double* sums,
                                            void* stream) {
  SPEX_RETURN_IF(n_cut > SPEX_METRICS_MAX_CUTOFFS, SPEX_E_TOOBIG);
  SPEX_RETURN_IF(n_chunks < 0 || n_cut < 1 || !sums || (n_chunks > 0 && !chunk_sums), SPEX_E_BADARG);
  fullrank_metrics_reduce_kernel<<<1, kWarp, 0, (cudaStream_t)stream>>>(chunk_sums, n_chunks, n_cut * 4, sums);
  count_launch();
  return check_last();
}
