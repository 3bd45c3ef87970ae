// sampler.cu — device-side negative / BPR-triple samplers (SURVEY §8f rank 3).
//
// Replaces the per-epoch host loop of LightTrainData.ng_sample
// (LightGCN_SPEX/code/utility1/dataloader.py:250-265: for every positive (u, i) draw 5 items
// j ~ U[0, m) and re-draw while (u, j) is a training interaction, dok lookup) and provides the
// (user, positive, negative) triples bpr_loss needs (upstream LightGCN UniformSample_original
// semantics: user uniform, positive uniform among the user's items, negative by rejection).
//
// The membership test is a binary search in the user's row of the adjacency CSR (columns ascending,
// item j stored as n_user_rows + j; bit 31 = hot flag, masked).  Randomness is counter-based
// (SplitMix64 of (seed, sample, slot, attempt)): the draw of a slot does not depend on thread
// scheduling, so a seed reproduces the same negatives on every launch and every GPU.
// The CPU sampler (spex_b200/dataloader.py, bit-exact np.random stream of the reference) stays the
// parity oracle of the reference's negatives; this one has the same DISTRIBUTION (uniform over the
// user's non-interacted items), checked by tests/test_gpu_sampler.py.
#include "common.cuh"

namespace spex {

// unbiased enough for m << 2^32: high 32 bits of a 64-bit hash, multiply-shift into [0, m)
__device__ __forceinline__ int32_t draw_below(uint64_t h, int32_t m) {
  return (int32_t)(((h >> 32) * (uint64_t)(uint32_t)m) >> 32);
}
// is item j in row [lo, hi) of the adjacency (columns ascending, stored as off + item)?
__device__ __forceinline__ bool row_has(const int32_t* __restrict__ col, int64_t lo, int64_t hi, int32_t target) {
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    const int32_t c = __ldg(col + mid) & 0x7fffffff;
    if (c == target) return true;
    if (c < target) lo = mid + 1; else hi = mid;
  }
  return false;
}
__device__ __forceinline__ int32_t draw_negative(const int32_t* __restrict__ col, int64_t lo, int64_t hi,
                                                 int32_t off, int32_t m, uint64_t key) {
  int32_t j = 0;
  for (int attempt = 0; attempt < 64; ++attempt) {
    j = draw_below(splitmix64(key + (uint64_t)attempt * 0xD1B54A32D192ED03ull), m);
    if (!row_has(col, lo, hi, off + j)) return j;
  }
  // a user who interacted with almost every item: walk forward from the last draw (<= degree + 1 steps)
  for (int64_t s = 0; s <= hi - lo; ++s) {
    j = (j + 1 == m) ? 0 : j + 1;
    if (!row_has(col, lo, hi, off + j)) return j;
  }
  return -1;   // the user has interacted with every item
}

// out[s, q] = q-th negative of sample s (user users[s])
__global__ void __launch_bounds__(256)
sample_negatives_kernel(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col, int32_t off,
                        int32_t m, const int64_t* __restrict__ users, int64_t n, int32_t n_neg, uint64_t seed,
                        int64_t* __restrict__ out) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; t < n * n_neg; t += stride) {
    const int64_t s = t / n_neg;
    const int64_t u = users[s];
    out[t] = draw_negative(col, rowptr[u], rowptr[u + 1], off, m, splitmix64(seed ^ (uint64_t)t * 0x9E3779B97F4A7C15ull));
  }
}

// (user, pos, neg): user uniform in [0, n_users) re-drawn while its row is empty, pos uniform in the row
__global__ void __launch_bounds__(256)
sample_bpr_kernel(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col, int32_t off, int32_t m,
                  int64_t n_users, int64_t n, uint64_t seed, int64_t* __restrict__ users,
                  int64_t* __restrict__ pos, int64_t* __restrict__ neg) {
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; t < n; t += stride) {
    const uint64_t key = splitmix64(seed ^ (uint64_t)t * 0x9E3779B97F4A7C15ull);
    int64_t u = 0, lo = 0, hi = 0;
    for (int attempt = 0; attempt < 256; ++attempt) {
      u = (int64_t)(((splitmix64(key + attempt) >> 11) * (1.0 / 9007199254740992.0)) * (double)n_users);
      u = u < n_users ? u : n_users - 1;
      lo = rowptr[u];
      hi = rowptr[u + 1];
      if (hi > lo) break;
    }
    users[t] = u;
    if (hi <= lo) {   // no user with interactions found (degenerate graph)
      pos[t] = -1;
      neg[t] = -1;
      continue;
    }
    const int64_t e = lo + (int64_t)(((splitmix64(key ^ 0xA5A5A5A5A5A5A5A5ull) >> 11) * (1.0 / 9007199254740992.0)) *
                                     (double)(hi - lo));
    pos[t] = (int64_t)((__ldg(col + (e < hi ? e : hi - 1)) & 0x7fffffff) - off);
    neg[t] = draw_negative(col, lo, hi, off, m, key ^ 0x5DEECE66Dull);
  }
}

}  // namespace spex

using namespace spex;

extern "C" int spex_sample_negatives(const int64_t* rowptr, const int32_t* col, int32_t item_col_offset,
                                     int32_t m_items, const int64_t* users, int64_t n, int32_t n_neg,
                                     uint64_t seed, int64_t* out, void* stream) {
  SPEX_RETURN_IF(!rowptr || !col || !users || !out || n < 0 || n_neg < 1 || m_items < 1 || item_col_offset < 0,
                 SPEX_E_BADARG);
  if (n == 0) return 0;
  int64_t blocks = (n * n_neg + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  sample_negatives_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(rowptr, col, item_col_offset, m_items,
                                                                              users, n, n_neg, seed, out);
  count_launch();
  return check_last();
}

extern "C" int spex_sample_bpr(const int64_t* rowptr, const int32_t* col, int32_t item_col_offset,
                               int32_t m_items, int64_t n_users, int64_t n, uint64_t seed, int64_t* users,
                               int64_t* pos, int64_t* neg, void* stream) {
  SPEX_RETURN_IF(!rowptr || !col || !users || !pos || !neg || n < 0 || n_users < 1 || m_items < 1 ||
                     item_col_offset < 0,
                 SPEX_E_BADARG);
  if (n == 0) return 0;
  int64_t blocks = (n + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  sample_bpr_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(rowptr, col, item_col_offset, m_items, n_users,
                                                                        n, seed, users, pos, neg);
  count_launch();
  return check_last();
}
