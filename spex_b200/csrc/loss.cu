// loss.cu — fused gather -> dot -> loss kernels and their deterministic backward (sm_100a).
//
// Replaces, in the reference:
//   all_users[users], all_items[items], mul, sum      LightGCN_SPEX/code/utility1/model.py:115-118
//   nn.BCEWithLogitsLoss                              model.py:23,120
//   index backward = index_put_(accumulate=True)      autograd, main_rec.py:35   (atomics there)
//   torch.optim.Adam.step                             main_rec.py:23,37
//   expert gating                                     model_expert_s.py:154-161
//   per-user candidate scoring of Test()              utility1/batch_test.py:28-40
// and adds bpr_loss (north_star; upstream LightGCN semantics, SURVEY §8 a5).
//
// All kernels are HBM/L2-latency bound gathers of 256-byte rows: warp per sample, 128-bit lanes.
// The backward scatter is a segmented reduction in batch order (first occurrence of a row id owns
// the output row and sums every duplicate in ascending batch position): no atomics, so gradients
// are bit-reproducible.
#include "common.cuh"
#include <math.h>
#include <cub/device/device_radix_sort.cuh>

namespace spex {

constexpr int kWarpsPerCta = 8;

template <int NV>
__device__ __forceinline__ void load_row(const float* __restrict__ base, int64_t row, int D, int lane,
                                         float4 (&r)[NV]) {
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const int d = (lane + 32 * v) * 4;
    r[v] = (d < D) ? *reinterpret_cast<const float4*>(base + row * D + d) : f4_zero();
  }
}
template <int NV>
__device__ __forceinline__ float dot_rows(const float4 (&a)[NV], const float4 (&b)[NV]) {
  float s = 0.f;
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    s = fmaf(a[v].x, b[v].x, s);
    s = fmaf(a[v].y, b[v].y, s);
    s = fmaf(a[v].z, b[v].z, s);
    s = fmaf(a[v].w, b[v].w, s);
  }
  return s;
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }
// softplus(x) = max(x,0) + log1p(exp(-|x|))
__device__ __forceinline__ float softplusf_(float x) { return fmaxf(x, 0.f) + log1pf(expf(-fabsf(x))); }

// ------------------------------------------------------------------------------------------------
template <int NV>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
bce_fwd_kernel(const float* __restrict__ U, const float* __restrict__ I, int D,
               const int64_t* __restrict__ users, const int64_t* __restrict__ items,
               const float* __restrict__ labels, int64_t B, float* __restrict__ gamma,
               float* __restrict__ dgamma) {
  const int lane = threadIdx.x & 31;
  const int64_t b = (int64_t)blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
  if (b >= B) return;
  float4 u[NV], it[NV];
  load_row<NV>(U, users[b], D, lane, u);
  load_row<NV>(I, items[b], D, lane, it);
  const float g = warp_sum(dot_rows<NV>(u, it));
  if (lane == 0) {
    gamma[b] = g;
    if (dgamma) dgamma[b] = (sigmoidf_(g) - labels[b]) / (float)B;
  }
}

// single CTA, fixed-order tree: loss = mean_b [(1-y)x + max(-x,0) + log1p(exp(-|x|))]
__global__ void __launch_bounds__(1024)
bce_loss_reduce_kernel(const float* __restrict__ gamma, const float* __restrict__ labels, int64_t B,
                       float* __restrict__ loss) {
  __shared__ float sh[1024];
  float s = 0.f;
  for (int64_t b = threadIdx.x; b < B; b += 1024) {
    const float x = gamma[b], y = labels[b];
    s += (1.f - y) * x + fmaxf(-x, 0.f) + log1pf(expf(-fabsf(x)));
  }
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) loss[0] = sh[0] / (float)B;
}

// ------------------------------------------------------------------------------------------------
// Deterministic scatter:  out[idx(t), :] = sum over t' with idx(t') == idx(t), ascending t', of
//                         w(t') * src[srcidx(t'), :]
// The logical list has nseg*B entries; entry t = (seg = t / B, b = t % B).
struct ScatterList {
  const int64_t* idx[2];
  const int64_t* src_idx[2];
  float sign[2];
  int nseg;
  int64_t B;
  const float* coef;     // per-sample [B] or NULL (=1)
  const float* gscalar;  // device scalar or NULL (=1)
  float cconst;
  // optional row window (row partition across GPUs): only destination rows in [row_lo, row_hi) are
  // written, at out[(row - row_lo), :]; row_hi == 0 means "all rows"
  int64_t row_lo, row_hi;
};
__device__ __forceinline__ bool in_window(const ScatterList& L, int64_t row) {
  return L.row_hi == 0 || (row >= L.row_lo && row < L.row_hi);
}

template <int NV>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
scatter_rows_kernel(ScatterList L, const float* __restrict__ src, float* __restrict__ out, int D) {
  const int lane = threadIdx.x & 31;
  const int64_t total = (int64_t)L.nseg * L.B;
  const int64_t t = (int64_t)blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
  if (t >= total) return;
  const int myseg = (int)(t / L.B);
  const int64_t my = L.idx[myseg][t - (int64_t)myseg * L.B];
  if (!in_window(L, my)) return;
  const float gs = (L.gscalar ? L.gscalar[0] : 1.f) * L.cconst;
  float4 acc[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) acc[v] = f4_zero();
  for (int64_t base = 0; base < total; base += 32) {
    const int64_t tt = base + lane;
    bool match = false;
    if (tt < total) {
      const int sg = (int)(tt / L.B);
      match = (L.idx[sg][tt - (int64_t)sg * L.B] == my);
    }
    unsigned m = __ballot_sync(kFull, match);
    if (base + 32 <= t) {
      if (m) return;  // an earlier entry owns this row
    } else if (base <= t) {
      const unsigned before = (1u << (int)(t - base)) - 1u;
      if (m & before) return;
    }
    while (m) {
      const int bit = __ffs(m) - 1;
      m &= m - 1;
      const int64_t t2 = base + bit;
      const int sg = (int)(t2 / L.B);
      const int64_t b2 = t2 - (int64_t)sg * L.B;
      const float w = L.sign[sg] * (L.coef ? L.coef[b2] : 1.f) * gs;
      float4 r[NV];
      load_row<NV>(src, L.src_idx[sg][b2], D, lane, r);
#pragma unroll
      for (int v = 0; v < NV; ++v) f4_fma(acc[v], w, r[v]);
    }
  }
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const int d = (lane + 32 * v) * 4;
    if (d < D) *reinterpret_cast<float4*>(out + (my - L.row_lo) * D + d) = acc[v];
  }
}

// ---- sorted form (large batches) -------------------------------------------------------------------
// The scan above costs O(total^2 / 32); from a few thousand entries on the list is instead SORTED by
// destination row (stable LSB radix sort of (row, t) pairs: entries of a row stay in ascending t) and
// the warp that owns the FIRST entry of a row's run sums the run in order.  Same summation order as
// the scan (ascending t), so both forms give bit-identical gradients.
__global__ void __launch_bounds__(256)
scatter_keys_kernel(ScatterList L, uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
  const int64_t total = (int64_t)L.nseg * L.B;
  int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; t < total; t += stride) {
    const int sg = (int)(t / L.B);
    keys[t] = (uint32_t)L.idx[sg][t - (int64_t)sg * L.B];
    vals[t] = (uint32_t)t;
  }
}

template <int NV>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
scatter_sorted_kernel(ScatterList L, const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals,
                      const float* __restrict__ src, float* __restrict__ out, int D) {
  const int lane = threadIdx.x & 31;
  const int64_t total = (int64_t)L.nseg * L.B;
  const int64_t p = (int64_t)blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
  if (p >= total) return;
  const uint32_t my = keys[p];
  if (p > 0 && keys[p - 1] == my) return;   // not the head of its row's run
  if (!in_window(L, (int64_t)my)) return;
  const float gs = (L.gscalar ? L.gscalar[0] : 1.f) * L.cconst;
  float4 acc[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) acc[v] = f4_zero();
  for (int64_t e = p; e < total && keys[e] == my; ++e) {
    const int64_t t2 = vals[e];
    const int sg = (int)(t2 / L.B);
    const int64_t b2 = t2 - (int64_t)sg * L.B;
    const float w = L.sign[sg] * (L.coef ? L.coef[b2] : 1.f) * gs;
    float4 r[NV];
    load_row<NV>(src, L.src_idx[sg][b2], D, lane, r);
#pragma unroll
    for (int v = 0; v < NV; ++v) f4_fma(acc[v], w, r[v]);
  }
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const int d = (lane + 32 * v) * 4;
    if (d < D) *reinterpret_cast<float4*>(out + ((int64_t)my - L.row_lo) * D + d) = acc[v];
  }
}

constexpr int64_t kScanLimit = 2048;       // above: sorted form (needs a workspace)
constexpr int64_t kScatterMax = 1ll << 31;  // entries (positions travel as uint32)

static size_t scatter_cub_bytes(int64_t total) {
  size_t tmp = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, tmp, (const uint32_t*)nullptr, (uint32_t*)nullptr,
                                  (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)total);
  return tmp;
}
static int64_t scatter_ws_bytes(int64_t total) {
  if (total <= kScanLimit) return 0;
  const int64_t arr = ((total * 4 + 255) / 256) * 256;
  return 4 * arr + (int64_t)((scatter_cub_bytes(total) + 255) / 256 * 256);
}

static int launch_scatter(const ScatterList& L, const float* src, float* out, int D, void* work,
                          int64_t work_bytes, cudaStream_t st) {
  const int64_t total = (int64_t)L.nseg * L.B;
  if (total == 0) return 0;
  if (total > kScanLimit && work) {
    SPEX_RETURN_IF(total >= kScatterMax, SPEX_E_TOOBIG);
    SPEX_RETURN_IF(work_bytes < scatter_ws_bytes(total) || !aligned16(work), SPEX_E_WORKSPACE);
    const int64_t arr = ((total * 4 + 255) / 256) * 256;
    uint8_t* w8 = (uint8_t*)work;
    uint32_t* k_in = (uint32_t*)w8;
    uint32_t* k_out = (uint32_t*)(w8 + arr);
    uint32_t* v_in = (uint32_t*)(w8 + 2 * arr);
    uint32_t* v_out = (uint32_t*)(w8 + 3 * arr);
    void* tmp = w8 + 4 * arr;
    size_t tmp_bytes = scatter_cub_bytes(total);
    int64_t blocks = (total + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    scatter_keys_kernel<<<(unsigned)blocks, 256, 0, st>>>(L, k_in, v_in);
    cudaError_t e = cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, k_in, k_out, v_in, v_out, (int)total, 0, 32, st);
    if (e != cudaSuccess) return (int)e;
    const unsigned grid = (unsigned)((total + kWarpsPerCta - 1) / kWarpsPerCta);
    if (D <= 128)
      scatter_sorted_kernel<1><<<grid, kWarpsPerCta * 32, 0, st>>>(L, k_out, v_out, src, out, D);
    else
      scatter_sorted_kernel<4><<<grid, kWarpsPerCta * 32, 0, st>>>(L, k_out, v_out, src, out, D);
    count_launch(2);
    return check_last();
  }
  if (total > (1 << 18)) return SPEX_E_WORKSPACE;  // O(total^2/32) duplicate scan: pass a workspace
  const unsigned grid = (unsigned)((total + kWarpsPerCta - 1) / kWarpsPerCta);
  if (D <= 128)
    scatter_rows_kernel<1><<<grid, kWarpsPerCta * 32, 0, st>>>(L, src, out, D);
  else
    scatter_rows_kernel<4><<<grid, kWarpsPerCta * 32, 0, st>>>(L, src, out, D);
  count_launch();
  return check_last();
}

// R[i, :] = table_local[rows[i] - row_lo, :] if rows[i] in [row_lo, row_hi) else 0  (thread per float4)
__global__ void __launch_bounds__(256)
gather_owned_rows_kernel(const float* __restrict__ table_local, const int64_t* __restrict__ rows, int64_t n,
                         int D4, int64_t row_lo, int64_t row_hi, float* __restrict__ R) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < n * D4; i += stride) {
    const int64_t r = rows[i / D4];
    float4 v = f4_zero();
    if (r >= row_lo && r < row_hi) v = reinterpret_cast<const float4*>(table_local)[(r - row_lo) * D4 + (i % D4)];
    reinterpret_cast<float4*>(R)[i] = v;
  }
}

// out[rows[i], :] = 0  (thread per float4; duplicate rows are harmless)
__global__ void __launch_bounds__(256)
clear_rows_kernel(float* __restrict__ table, const int64_t* __restrict__ rows, int64_t n, int D4) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < n * D4; i += stride) {
    const int64_t r = rows[i / D4];
    reinterpret_cast<float4*>(table)[r * D4 + (i % D4)] = f4_zero();
  }
}

// ------------------------------------------------------------------------------------------------
template <int NV>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
bpr_fwd_kernel(const float* __restrict__ U, const float* __restrict__ I, const float* __restrict__ U0,
               const float* __restrict__ I0, int D, const int64_t* __restrict__ users,
               const int64_t* __restrict__ pos, const int64_t* __restrict__ neg, int64_t B,
               float* __restrict__ dscore, float* __restrict__ work) {
  const int lane = threadIdx.x & 31;
  const int64_t b = (int64_t)blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
  if (b >= B) return;
  const int64_t u = users[b], p = pos[b], n = neg[b];
  float4 ru[NV], rp[NV], rn[NV];
  load_row<NV>(U, u, D, lane, ru);
  load_row<NV>(I, p, D, lane, rp);
  load_row<NV>(I, n, D, lane, rn);
  const float ps = warp_sum(dot_rows<NV>(ru, rp));
  const float ns = warp_sum(dot_rows<NV>(ru, rn));
  load_row<NV>(U0, u, D, lane, ru);
  load_row<NV>(I0, p, D, lane, rp);
  load_row<NV>(I0, n, D, lane, rn);
  const float rg = warp_sum(dot_rows<NV>(ru, ru) + dot_rows<NV>(rp, rp) + dot_rows<NV>(rn, rn));
  if (lane == 0) {
    const float x = ns - ps;
    work[b] = softplusf_(x);
    work[B + b] = 0.5f * rg;
    if (dscore) dscore[b] = sigmoidf_(x) / (float)B;
  }
}

// out2 = { mean(work[0:B]), sum(work[B:2B]) / B }, fixed-order tree
__global__ void __launch_bounds__(1024)
pair_mean_reduce_kernel(const float* __restrict__ work, int64_t B, float* __restrict__ out2) {
  __shared__ float sh0[1024];
  __shared__ float sh1[1024];
  float s0 = 0.f, s1 = 0.f;
  for (int64_t b = threadIdx.x; b < B; b += 1024) {
    s0 += work[b];
    s1 += work[B + b];
  }
  sh0[threadIdx.x] = s0;
  sh1[threadIdx.x] = s1;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) {
      sh0[threadIdx.x] += sh0[threadIdx.x + o];
      sh1[threadIdx.x] += sh1[threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    out2[0] = sh0[0] / (float)B;
    out2[1] = sh1[0] / (float)B;
  }
}

// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
adam_kernel(float4* __restrict__ p, const float4* __restrict__ g, float4* __restrict__ m,
            float4* __restrict__ v, int64_t n4, float beta1, float beta2, float eps, float step_size,
            float bc2_sqrt, float* __restrict__ ptail, const float* __restrict__ gtail,
            float* __restrict__ mtail, float* __restrict__ vtail, int ntail) {
  const float omb1 = 1.f - beta1, omb2 = 1.f - beta2;
  auto upd = [&](float& pp, float gg, float& mm, float& vv) {
    mm = mm + (gg - mm) * omb1;                 // exp_avg.lerp_(grad, 1-beta1)
    vv = vv * beta2 + omb2 * gg * gg;           // exp_avg_sq.mul_(b2).addcmul_(g, g, 1-b2)
    const float denom = sqrtf(vv) / bc2_sqrt + eps;
    pp = pp - step_size * (mm / denom);         // param.addcdiv_(exp_avg, denom, -step_size)
  };
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < n4; i += stride) {
    float4 pp = p[i], mm = m[i], vv = v[i];
    const float4 gg = __ldcs(g + i);
    upd(pp.x, gg.x, mm.x, vv.x);
    upd(pp.y, gg.y, mm.y, vv.y);
    upd(pp.z, gg.z, mm.z, vv.z);
    upd(pp.w, gg.w, mm.w, vv.w);
    p[i] = pp;
    m[i] = mm;
    v[i] = vv;
  }
  if (blockIdx.x == 0 && (int)threadIdx.x < ntail) {
    const int t = threadIdx.x;
    upd(ptail[t], gtail[t], mtail[t], vtail[t]);
  }
}

// ------------------------------------------------------------------------------------------------
// expert gating (model_expert_s.py:154-161): warp per row
template <int NV>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
expert_gate_kernel(const float* __restrict__ E0, const float* __restrict__ Eout,
                   const float* __restrict__ W, int64_t n, int D, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
  if (row >= n) return;
  float4 a[NV], b[NV];
  load_row<NV>(E0, row, D, lane, a);
  load_row<NV>(Eout, row, D, lane, b);
  float l0 = 0.f, l1 = 0.f;
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const int d = (lane + 32 * v) * 4;
    if (d < D) {
      const float av[4] = {a[v].x, a[v].y, a[v].z, a[v].w};
      const float bv[4] = {b[v].x, b[v].y, b[v].z, b[v].w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float2 wa = *reinterpret_cast<const float2*>(W + 2 * (d + q));
        const float2 wb = *reinterpret_cast<const float2*>(W + 2 * (D + d + q));
        l0 = fmaf(av[q], wa.x, l0);
        l1 = fmaf(av[q], wa.y, l1);
        l0 = fmaf(bv[q], wb.x, l0);
        l1 = fmaf(bv[q], wb.y, l1);
      }
    }
  }
  l0 = warp_sum(l0);
  l1 = warp_sum(l1);
  const float mx = fmaxf(l0, l1);
  const float e0 = expf(l0 - mx), e1 = expf(l1 - mx);
  const float a0 = e0 / (e0 + e1), a1 = e1 / (e0 + e1);
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const int d = (lane + 32 * v) * 4;
    if (d < D) {
      float4 o;
      o.x = a[v].x * a0 + b[v].x * a1;
      o.y = a[v].y * a0 + b[v].y * a1;
      o.z = a[v].z * a0 + b[v].z * a1;
      o.w = a[v].w * a0 + b[v].w * a1;
      *reinterpret_cast<float4*>(out + row * D + d) = o;
    }
  }
}


// ------------------------------------------------------------------------------------------------
// expert gating backward (autograd of model_expert_s.py:154-161; the gate weights att_exp1/2 are
// trained in main_11.py:69).  Per row: z = [e0|e1].W, a = softmax(z), out = a0 e0 + a1 e1.
//   da_j = <g, e_j>;  dz_j = a_j (da_j - sum_k a_k da_k)
//   de0 = a0 g + W[0:D,:] dz;  de1 = a1 g + W[D:2D,:] dz;  dW[d, j] = sum_rows e[d] dz_j
// dW is reduced without atomics: every warp owns a fixed strided set of rows and keeps its 16
// partial sums in registers; the warps of a CTA are added in warp order, the CTAs in CTA order.
constexpr int kGateBlocks = SPEX_GATE_BWD_BLOCKS;

__global__ void __launch_bounds__(kWarpsPerCta * 32)
expert_gate_bwd_kernel(const float* __restrict__ E0, const float* __restrict__ E1,
                       const float* __restrict__ W, const float* __restrict__ G, int64_t n, int D,
                       float* __restrict__ dE0, float* __restrict__ dE1, float* __restrict__ work) {
  __shared__ float sh[kWarpsPerCta][16 * 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int d = lane * 4;
  const bool act = d < D;
  float2 wa[4], wb[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    wa[q] = act ? *reinterpret_cast<const float2*>(W + 2 * (d + q)) : make_float2(0.f, 0.f);
    wb[q] = act ? *reinterpret_cast<const float2*>(W + 2 * (D + d + q)) : make_float2(0.f, 0.f);
  }
  float acc[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) acc[i] = 0.f;
  for (int64_t row = (int64_t)blockIdx.x * kWarpsPerCta + warp; row < n;
       row += (int64_t)gridDim.x * kWarpsPerCta) {
    float4 a4 = f4_zero(), b4 = f4_zero(), g4 = f4_zero();
    if (act) {
      a4 = *reinterpret_cast<const float4*>(E0 + row * D + d);
      b4 = *reinterpret_cast<const float4*>(E1 + row * D + d);
      g4 = *reinterpret_cast<const float4*>(G + row * D + d);
    }
    const float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
    const float g[4] = {g4.x, g4.y, g4.z, g4.w};
    float l0 = 0.f, l1 = 0.f, da0 = 0.f, da1 = 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      l0 = fmaf(a[q], wa[q].x, l0);
      l1 = fmaf(a[q], wa[q].y, l1);
      l0 = fmaf(b[q], wb[q].x, l0);
      l1 = fmaf(b[q], wb[q].y, l1);
      da0 = fmaf(g[q], a[q], da0);
      da1 = fmaf(g[q], b[q], da1);
    }
    l0 = warp_sum(l0);
    l1 = warp_sum(l1);
    da0 = warp_sum(da0);
    da1 = warp_sum(da1);
    const float mx = fmaxf(l0, l1);
    const float x0 = expf(l0 - mx), x1 = expf(l1 - mx);
    const float p0 = x0 / (x0 + x1), p1 = x1 / (x0 + x1);
    const float sdot = p0 * da0 + p1 * da1;
    const float dz0 = p0 * (da0 - sdot), dz1 = p1 * (da1 - sdot);
    if (act) {
      float o0[4], o1[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        o0[q] = p0 * g[q] + wa[q].x * dz0 + wa[q].y * dz1;
        o1[q] = p1 * g[q] + wb[q].x * dz0 + wb[q].y * dz1;
        acc[4 * q + 0] = fmaf(a[q], dz0, acc[4 * q + 0]);
        acc[4 * q + 1] = fmaf(a[q], dz1, acc[4 * q + 1]);
        acc[4 * q + 2] = fmaf(b[q], dz0, acc[4 * q + 2]);
        acc[4 * q + 3] = fmaf(b[q], dz1, acc[4 * q + 3]);
      }
      *reinterpret_cast<float4*>(dE0 + row * D + d) = make_float4(o0[0], o0[1], o0[2], o0[3]);
      *reinterpret_cast<float4*>(dE1 + row * D + d) = make_float4(o1[0], o1[1], o1[2], o1[3]);
    }
  }
#pragma unroll
  for (int i = 0; i < 16; ++i) sh[warp][i * 32 + lane] = acc[i];
  __syncthreads();
  // CTA partial in warp order; layout of work: [block][i = 4*q + {a.z0,a.z1,b.z0,b.z1}][lane]
  for (int i = threadIdx.x; i < 16 * 32; i += kWarpsPerCta * 32) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kWarpsPerCta; ++w) t += sh[w][i];
    work[(size_t)blockIdx.x * 512 + i] = t;
  }
}

// dW[2D, 2]: sum the CTA partials in CTA order (one thread per output element)
__global__ void __launch_bounds__(256)
expert_gate_dw_kernel(const float* __restrict__ work, int n_blocks, int D, float* __restrict__ dW) {
  const int o = blockIdx.x * blockDim.x + threadIdx.x;   // o = 2 * row + j, row in [0, 2D)
  if (o >= 4 * D) return;
  const int j = o & 1, r = o >> 1;
  const int tab = r >= D ? 1 : 0, dd = r - tab * D;
  const int lane = dd >> 2, q = dd & 3;
  const int i = 4 * q + 2 * tab + j;
  float t = 0.f;
  for (int b = 0; b < n_blocks; ++b) t += work[(size_t)b * 512 + i * 32 + lane];
  dW[o] = t;
}

// ------------------------------------------------------------------------------------------------
// score[u,c] = <U[users[u]], I[cand[u,c]]>: warp per (u,c)
template <int NV>
__global__ void __launch_bounds__(kWarpsPerCta * 32)
score_candidates_kernel(const float* __restrict__ U, const float* __restrict__ I, int D,
                        const int64_t* __restrict__ users, const int32_t* __restrict__ cand,
                        int64_t n_u, int n_c, float* __restrict__ score) {
  const int lane = threadIdx.x & 31;
  const int64_t w = (int64_t)blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5);
  if (w >= n_u * n_c) return;
  const int64_t u = w / n_c;
  float4 a[NV], b[NV];
  load_row<NV>(U, users[u], D, lane, a);
  load_row<NV>(I, (int64_t)cand[w], D, lane, b);
  const float s = warp_sum(dot_rows<NV>(a, b));
  if (lane == 0) score[w] = s;
}

static inline unsigned warp_grid(int64_t n) { return (unsigned)((n + kWarpsPerCta - 1) / kWarpsPerCta); }

}  // namespace spex

using namespace spex;

#define SPEX_CHECK_TABLE(D)                                        \
  SPEX_RETURN_IF((D) <= 0 || ((D)&3) || (D) > 512, SPEX_E_BADDIM)

extern "C" int spex_bce_fwd_f32(const float* U, const float* I, int32_t D, const int64_t* users,
                                const int64_t* items, const float* labels, int64_t B, float* gamma,
                                float* loss, float* dgamma, void* stream) {
  SPEX_RETURN_IF(!U || !I || B < 0, SPEX_E_BADARG);
  SPEX_RETURN_IF(B > 0 && (!users || !items || !gamma || ((loss || dgamma) && !labels)), SPEX_E_BADARG);
  SPEX_CHECK_TABLE(D);
  SPEX_RETURN_IF(!aligned16(U) || !aligned16(I), SPEX_E_ALIGN);
  SPEX_RETURN_IF(B > 0x7fffffffLL, SPEX_E_TOOBIG);
  cudaStream_t st = (cudaStream_t)stream;
  // an empty batch still runs the reduce: the mean of no terms is 0/0 = NaN, as in BCEWithLogitsLoss
  if (B > 0) {
    if (D <= 128)
      bce_fwd_kernel<1><<<warp_grid(B), kWarpsPerCta * 32, 0, st>>>(U, I, D, users, items, labels, B, gamma, dgamma);
    else
      bce_fwd_kernel<4><<<warp_grid(B), kWarpsPerCta * 32, 0, st>>>(U, I, D, users, items, labels, B, gamma, dgamma);
    count_launch();
  }
  if (loss) {
    bce_loss_reduce_kernel<<<1, 1024, 0, st>>>(gamma, labels, B, loss);
    count_launch();
  }
  return check_last();
}

extern "C" int64_t spex_scatter_workspace_bytes(int64_t total_entries) {
  return total_entries < 0 ? 0 : scatter_ws_bytes(total_entries);
}

extern "C" int spex_clear_rows_f32(float* table, const int64_t* rows, int64_t n, int32_t D, void* stream) {
  SPEX_RETURN_IF(!table || (n > 0 && !rows) || n < 0, SPEX_E_BADARG);
  SPEX_CHECK_TABLE(D);
  SPEX_RETURN_IF(!aligned16(table), SPEX_E_ALIGN);
  if (n == 0) return 0;
  int64_t blocks = (n * (D / 4) + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  clear_rows_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(table, rows, n, D / 4);
  count_launch();
  return check_last();
}

extern "C" int spex_gather_owned_rows_f32(const float* table_local, const int64_t* rows, int64_t n, int32_t D,
                                          int64_t row_lo, int64_t row_hi, float* R, void* stream) {
  SPEX_RETURN_IF(!table_local || !R || (n > 0 && !rows) || n < 0 || row_lo < 0 || row_hi < row_lo, SPEX_E_BADARG);
  SPEX_CHECK_TABLE(D);
  SPEX_RETURN_IF(!aligned16(table_local) || !aligned16(R), SPEX_E_ALIGN);
  if (n == 0) return 0;
  int64_t blocks = (n * (D / 4) + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  gather_owned_rows_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(table_local, rows, n, D / 4, row_lo,
                                                                               row_hi, R);
  count_launch();
  return check_last();
}

extern "C" int spex_scatter_rows_f32(const int64_t* dst_rows, const int64_t* src_rows, const float* coef,
                                     const float* gscalar, float cconst, int64_t B, const float* src, int32_t D,
                                     float* out, int64_t row_lo, int64_t row_hi, void* work, int64_t work_bytes,
                                     void* stream) {
  SPEX_RETURN_IF(!src || !out || B < 0 || row_lo < 0 || (row_hi != 0 && row_hi < row_lo), SPEX_E_BADARG);
  SPEX_RETURN_IF(B > 0 && (!dst_rows || !src_rows), SPEX_E_BADARG);
  SPEX_CHECK_TABLE(D);
  SPEX_RETURN_IF(!aligned16(src) || !aligned16(out), SPEX_E_ALIGN);
  ScatterList L{};
  L.nseg = 1;
  L.B = B;
  L.idx[0] = dst_rows;
  L.src_idx[0] = src_rows;
  L.sign[0] = 1.f;
  L.coef = coef;
  L.gscalar = gscalar;
  L.cconst = cconst;
  L.row_lo = row_lo;
  L.row_hi = row_hi;
  return launch_scatter(L, src, out, D, work, work_bytes, (cudaStream_t)stream);
}

extern "C" int spex_bce_bwd_ws_f32(const float* U, const float* I, int32_t D, const int64_t* users,
                                   const int64_t* items, const float* dgamma, const float* grad_loss,
                                   int64_t B, float* gU, float* gI, void* work, int64_t work_bytes,
                                   void* stream) {
  SPEX_RETURN_IF(!U || !I || !gU || !gI || B < 0, SPEX_E_BADARG);
  SPEX_RETURN_IF(B > 0 && (!users || !items || !dgamma), SPEX_E_BADARG);
  SPEX_CHECK_TABLE(D);
  SPEX_RETURN_IF(!aligned16(U) || !aligned16(I) || !aligned16(gU) || !aligned16(gI), SPEX_E_ALIGN);
  cudaStream_t st = (cudaStream_t)stream;
  ScatterList L{};
  L.nseg = 1;
  L.B = B;
  L.coef = dgamma;
  L.gscalar = grad_loss;
  L.cconst = 1.f;
  L.sign[0] = 1.f;
  // gU[users] += dgamma * I[items]
  L.idx[0] = users;
  L.src_idx[0] = items;
  int rc = launch_scatter(L, I, gU, D, work, work_bytes, st);
  if (rc) return rc;
  // gI[items] += dgamma * U[users]
  L.idx[0] = items;
  L.src_idx[0] = users;
  return launch_scatter(L, U, gI, D, work, work_bytes, st);
}

extern "C" int spex_bpr_fwd_f32(const float* U, const float* I, const float* U0, const float* I0,
                                int32_t D, const int64_t* users, const int64_t* pos,
                                const int64_t* neg, int64_t B, float* out2, float* dscore,
                                float* work2B, void* stream) {
  SPEX_RETURN_IF(!U || !I || !U0 || !I0 || !out2 || B < 0, SPEX_E_BADARG);
  SPEX_RETURN_IF(B > 0 && (!users || !pos || !neg || !work2B), SPEX_E_BADARG);
  SPEX_CHECK_TABLE(D);
  SPEX_RETURN_IF(!aligned16(U) || !aligned16(I) || !aligned16(U0) || !aligned16(I0), SPEX_E_ALIGN);
  SPEX_RETURN_IF(B > 0x7fffffffLL, SPEX_E_TOOBIG);
  cudaStream_t st = (cudaStream_t)stream;
  // an empty batch still runs the reduce: both means of no terms are 0/0 = NaN
  if (B > 0) {
    if (D <= 128)
      bpr_fwd_kernel<1><<<warp_grid(B), kWarpsPerCta * 32, 0, st>>>(U, I, U0, I0, D, users, pos, neg, B, dscore, work2B);
    else
      bpr_fwd_kernel<4><<<warp_grid(B), kWarpsPerCta * 32, 0, st>>>(U, I, U0, I0, D, users, pos, neg, B, dscore, work2B);
    count_launch();
  }
  pair_mean_reduce_kernel<<<1, 1024, 0, st>>>(work2B, B, out2);
  count_launch();
  return check_last();
}

extern "C" int spex_bpr_bwd_ws_f32(const float* U, const float* I, const float* U0, const float* I0,
                                   int32_t D, const int64_t* users, const int64_t* pos,
                                   const int64_t* neg, const float* dscore, const float* grad2,
                                   int64_t B, float* gU, float* gI, float* gU0, float* gI0, void* work,
                                   int64_t work_bytes, void* stream) {
  SPEX_RETURN_IF(!U || !I || !U0 || !I0 || B < 0, SPEX_E_BADARG);
  SPEX_RETURN_IF(B > 0 && (!users || !pos || !neg || !dscore), SPEX_E_BADARG);
  SPEX_RETURN_IF(!gU || !gI || !gU0 || !gI0, SPEX_E_BADARG);
  SPEX_CHECK_TABLE(D);
  SPEX_RETURN_IF(!aligned16(U) || !aligned16(I) || !aligned16(U0) || !aligned16(I0), SPEX_E_ALIGN);
  SPEX_RETURN_IF(!aligned16(gU) || !aligned16(gI) || !aligned16(gU0) || !aligned16(gI0), SPEX_E_ALIGN);
  cudaStream_t st = (cudaStream_t)stream;
  int rc;
  ScatterList L{};
  L.B = B;
  L.cconst = 1.f;
  // propagated tables: upstream dL/dloss = grad2[0]
  L.coef = dscore;
  L.gscalar = grad2;
  // gU[u] = sum d * (I[neg] - I[pos])   (pos terms first, then neg: fixed order)
  L.nseg = 2;
  L.idx[0] = users; L.src_idx[0] = pos; L.sign[0] = -1.f;
  L.idx[1] = users; L.src_idx[1] = neg; L.sign[1] = 1.f;
  if ((rc = launch_scatter(L, I, gU, D, work, work_bytes, st))) return rc;
  // gI[pos] -= d*U[u];  gI[neg] += d*U[u]
  L.idx[0] = pos; L.src_idx[0] = users; L.sign[0] = -1.f;
  L.idx[1] = neg; L.src_idx[1] = users; L.sign[1] = 1.f;
  if ((rc = launch_scatter(L, U, gI, D, work, work_bytes, st))) return rc;
  // ego tables: reg = 0.5*sum|.|^2 / B  ->  d/dx = x / B, times upstream grad2[1]
  L.coef = nullptr;
  L.gscalar = grad2 ? grad2 + 1 : nullptr;
  L.cconst = 1.f / (float)(B > 0 ? B : 1);
  L.nseg = 1;
  L.idx[0] = users; L.src_idx[0] = users; L.sign[0] = 1.f;
  if ((rc = launch_scatter(L, U0, gU0, D, work, work_bytes, st))) return rc;
  L.nseg = 2;
  L.idx[0] = pos; L.src_idx[0] = pos; L.sign[0] = 1.f;
  L.idx[1] = neg; L.src_idx[1] = neg; L.sign[1] = 1.f;
  return launch_scatter(L, I0, gI0, D, work, work_bytes, st);
}

extern "C" int spex_adam_f32(float* p, const float* g, float* m, float* v, int64_t n, float lr,
                             float beta1, float beta2, float eps, int32_t step, void* stream) {
  SPEX_RETURN_IF(!p || !g || !m || !v || n < 0 || step < 1, SPEX_E_BADARG);
  SPEX_RETURN_IF(!aligned16(p) || !aligned16(g) || !aligned16(m) || !aligned16(v), SPEX_E_ALIGN);
  if (n == 0) return 0;
  const double bc1 = 1.0 - pow((double)beta1, (double)step);
  const double bc2 = 1.0 - pow((double)beta2, (double)step);
  const float step_size = (float)((double)lr / bc1);
  const float bc2_sqrt = (float)sqrt(bc2);
  const int64_t n4 = n / 4;
  const int ntail = (int)(n - n4 * 4);
  int64_t blocks = (n4 + 255) / 256;
  if (blocks < 1) blocks = 1;
  if (blocks > 148 * 8) blocks = 148 * 8;
  adam_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
      (float4*)p, (const float4*)g, (float4*)m, (float4*)v, n4, beta1, beta2, eps, step_size,
      bc2_sqrt, p + n4 * 4, g + n4 * 4, m + n4 * 4, v + n4 * 4, ntail);
  count_launch();
  return check_last();
}

extern "C" int spex_expert_gate_f32(const float* E0, const float* Eout, const float* W, int64_t n,
                                    int32_t D, float* out, void* stream) {
  SPEX_RETURN_IF(!E0 || !Eout || !W || !out || n < 0, SPEX_E_BADARG);
  SPEX_CHECK_TABLE(D);
  SPEX_RETURN_IF(!aligned16(E0) || !aligned16(Eout) || !aligned16(out) || ((uintptr_t)W & 7), SPEX_E_ALIGN);
  if (n == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (D <= 128)
    expert_gate_kernel<1><<<warp_grid(n), kWarpsPerCta * 32, 0, st>>>(E0, Eout, W, n, D, out);
  else
    expert_gate_kernel<4><<<warp_grid(n), kWarpsPerCta * 32, 0, st>>>(E0, Eout, W, n, D, out);
  count_launch();
  return check_last();
}

extern "C" int spex_score_candidates_f32(const float* U, const float* I, int32_t D,
                                         const int64_t* users, const int32_t* cand, int64_t n_u,
                                         int32_t n_c, float* score, void* stream) {
  SPEX_RETURN_IF(!U || !I || !users || !cand || !score || n_u < 0 || n_c < 0, SPEX_E_BADARG);
  SPEX_CHECK_TABLE(D);
  SPEX_RETURN_IF(!aligned16(U) || !aligned16(I), SPEX_E_ALIGN);
  const int64_t total = n_u * (int64_t)n_c;
  if (total == 0) return 0;
  SPEX_RETURN_IF(total > 0x7fffffffLL * kWarpsPerCta, SPEX_E_TOOBIG);
  cudaStream_t st = (cudaStream_t)stream;
  if (D <= 128)
    score_candidates_kernel<1><<<warp_grid(total), kWarpsPerCta * 32, 0, st>>>(U, I, D, users, cand, n_u, n_c, score);
  else
    score_candidates_kernel<4><<<warp_grid(total), kWarpsPerCta * 32, 0, st>>>(U, I, D, users, cand, n_u, n_c, score);
  count_launch();
  return check_last();
}

extern "C" int spex_expert_gate_bwd_f32(const float* E0, const float* Eout, const float* W,
                                        const float* g, int64_t n, int32_t D, float* dE0,
                                        float* dEout, float* dW, float* work, void* stream) {
  SPEX_RETURN_IF(!E0 || !Eout || !W || !g || !dE0 || !dEout || !dW || !work || n < 0, SPEX_E_BADARG);
  SPEX_RETURN_IF(D <= 0 || (D & 3) || D > 128, SPEX_E_BADDIM);
  SPEX_RETURN_IF(!aligned16(E0) || !aligned16(Eout) || !aligned16(g) || !aligned16(dE0) ||
                     !aligned16(dEout) || ((uintptr_t)W & 7),
                 SPEX_E_ALIGN);
  cudaStream_t st = (cudaStream_t)stream;
  int64_t blocks = (n + kWarpsPerCta - 1) / kWarpsPerCta;
  if (blocks > kGateBlocks) blocks = kGateBlocks;
  if (blocks < 1) blocks = 1;
  expert_gate_bwd_kernel<<<(unsigned)blocks, kWarpsPerCta * 32, 0, st>>>(E0, Eout, W, g, n, D, dE0, dEout, work);
  expert_gate_dw_kernel<<<(4 * D + 255) / 256, 256, 0, st>>>(work, (int)blocks, D, dW);
  count_launch(2);
  return check_last();
}
