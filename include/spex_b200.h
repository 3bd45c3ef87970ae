/*
 * spex_b200.h — C-ABI of libspex_b200.so, the sm_100a hot path behind SPEX's LightGCN_SPEX.
 *
 * The reference (XMUDM/SPEX) is pure Python: it has no FFI of its own.  Every entry point below
 * therefore replaces a *PyTorch library call site* of the reference; the site is cited per
 * function as <file>:<line> relative to /root/reference/.  The binding a maintainer of the
 * reference would add is a ctypes stub (see INTEGRATION.md) — no torch types cross this boundary.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - every function enqueues work on `stream` (a cudaStream_t passed as void*) and returns
 *     without synchronising; 0 = ok, >0 = cudaError_t, <0 = SPEX_E_* argument error;
 *   - the library never allocates device memory that outlives a call; workspaces are passed in;
 *   - embedding tables are row-major fp32 [rows, D], rows 16-byte aligned (D % 4 == 0);
 *   - CSR adjacency: rowptr int64 [n_rows+1], col int32 [nnz] ascending per row, val fp32 [nnz];
 *   - results are deterministic: no floating-point atomics anywhere (north_star (1),(2)).
 */
#ifndef SPEX_B200_H
#define SPEX_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPEX_ABI_VERSION 3

/* argument errors (negative; positive values are cudaError_t) */
#define SPEX_E_BADARG   (-1)  /* null pointer / negative size */
#define SPEX_E_BADDIM   (-2)  /* D unsupported (must be a multiple of 4, <= 512) */
#define SPEX_E_ALIGN    (-3)  /* pointer not 16-byte aligned */
#define SPEX_E_ARCH     (-4)  /* device is not sm_100 (no fallback path exists) */
#define SPEX_E_TOOBIG   (-5)  /* k / batch exceeds a compiled-in limit */
#define SPEX_E_WORKSPACE (-6) /* workspace too small */

int spex_abi_version(void);
/* human-readable name of a code returned by any function below (static storage). */
const char* spex_error_string(int code);
/* fills sm_count / compute capability of the current device; SPEX_E_ARCH if cc != 10.x */
int spex_device_check(int* sm_count, int* cc_major, int* cc_minor);
/* number of kernels this library has launched since load (bench.py's gpu_launches) */
int64_t spex_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * Long-row plan.  Rows with more than `seg_len` non-zeros are cut into segments of at most seg_len
 * edges; each segment is reduced by one warp into a partial row and the partials of a row are
 * summed in a fixed order (deterministic two-pass — no atomics).  The segments form one list:
 *   [0, n_hub_seg)     hub-row cells: a hub row is cut at column-block boundaries (and a cell longer
 *                      than seg_len every seg_len edges), and the cells are listed BLOCK-MAJOR so that
 *                      concurrently running warps gather from one L2-sized window of the table;
 *   [n_hub_seg, n_seg) mid-row segments: every other long row is cut every seg_len edges from its
 *                      first edge, listed in ascending row order.
 * A table that fits in L2 has no hub rows (n_hub_seg == 0).  row_seg lists each long row's segments
 * in edge order: long row r owns row_seg[long_segptr[r] .. long_segptr[r+1]), and its partials are
 * summed in that order.
 * The plan is built once per graph by the host (spex_b200/ops.py: DeviceGraph) and passed to every
 * SpMM as a HOST struct holding device pointers; NULL (or n_long == 0) means "no long rows".
 * ------------------------------------------------------------------------------------------ */
/* flags: bit 31 of every col[] entry marks a HOT table row (one that is gathered so often that it
 * should stay in L2): the kernels strip the bit and gather hot rows with the L2 evict_last policy,
 * all others with evict_first.  A plan with n_long == 0 may still carry this flag.  No other flag
 * bit is defined: a plan that sets one is rejected with SPEX_E_BADARG. */
#define SPEX_PLAN_COL_HOTBIT 1

typedef struct spex_long_plan {
  int32_t seg_len;            /* rows with degree > seg_len take the long-row path (>= 32)    */
  int32_t n_long;             /* number of such rows                                          */
  int32_t n_seg;              /* total number of segments                                     */
  int32_t flags;              /* SPEX_PLAN_* bits                                             */
  const int32_t* long_rows;   /* int32 [n_long]    row ids, ascending                         */
  const int32_t* long_segptr; /* int32 [n_long+1]  exclusive scan of segments per long row    */
  float* partial;             /* fp32  [n_seg, D]  workspace                                  */
  const int64_t* seg_start;   /* int64 [n_seg]  first edge of each segment                    */
  const int32_t* seg_count;   /* int32 [n_seg]  edges in each segment                         */
  const int32_t* row_seg;     /* int32 [n_seg]  segment ids grouped by long row, edge order   */
  int32_t n_hub_seg;          /* segments [0, n_hub_seg) are hub-row cells, gathered with the default L2
                                 priority so that their window stays resident; the rest are mid-row
                                 segments (no reuse: evict_first under COL_HOTBIT)                   */
} spex_long_plan;

/*
 * One propagation layer  Y = A·X  with a fused two-output epilogue
 *      Y[i,:] = acc                                   (skipped if Y == NULL)
 *      Z[i,:] = (addend[i,:] * addend_scale + acc) * z_scale   (skipped if Z == NULL;
 *                                                      addend == NULL means 0)
 * Replaces torch.sparse.mm(g_droped, all_emb)  LightGCN_SPEX/code/utility1/model.py:91
 * (same call: model_expert_s.py:120) and, through Z, the stack+mean of model.py:94-95 and the
 * autograd of both (main_rec.py:35).  The CSR may be a row block of the full matrix (row partition across GPUs,
 * SURVEY §8e): X is always the full [n_cols, D] table, Y/Z/addend are [n_rows, D] (local rows).
 */
int spex_spmm_csr_f32(const int64_t* rowptr, const int32_t* col, const float* val,
                      const float* X, int64_t n_rows, int32_t D,
                      float* Y, const float* addend, float addend_scale,
                      float* Z, float z_scale,
                      const spex_long_plan* plan, void* stream);

/*
 * Epilogue of one propagation layer (spex_spmm_layer_f32): what the warp that finishes output row i does with
 * acc = (A·X)[i,:].  A HOST struct holding device pointers; the *_host members are host arrays of device
 * pointers.  Zero-initialise it and set what the layer needs: every feature is off when its fields are NULL / 0.
 * Tables are fp32 [rows, D], 16-byte aligned (SPEX_E_ALIGN otherwise).
 */
typedef struct spex_spmm_epilogue {
  float* Y;                     /* [n_rows, D]: Y[i,:] = acc (NULL: not written) */
  const float* addend;          /* [n_rows, D]: addend of Z (NULL: 0) */
  float addend_scale;
  float* Z;                     /* [n_rows, D]: Z[i,:] = (addend[i,:] * addend_scale + acc) * z_scale (NULL: none) */
  float z_scale;
  int64_t out_row_offset;       /* >= 0: row i goes to row out_row_offset + i of the exchange / publish tables */
  /* Y exchange (at most one of the two ways): acc is also stored into every GPU's next-layer table, by ONE
   * multimem.st to the NVSwitch multicast mapping y_mcast (cuMulticast*, e.g. torch symmetric memory's
   * multicast_ptr; NVLS), or by P2P stores to the n_y_peers (0..8) tables of y_peers_host (own table included). */
  float* y_mcast;
  float* const* y_peers_host;
  int32_t n_y_peers;
  /* publish: row i of pub_src [n_rows, D] (this rank's slice of the NEXT call's table) is stored into every
   * GPU's table through exactly one of pub_mcast / the n_pub_peers (0..8) tables of pub_peers_host: the E^(0)
   * exchange of the next propagation rides on this layer's epilogue.  Not with Adam. */
  const float* pub_src;
  float* pub_mcast;
  float* const* pub_peers_host;
  int32_t n_pub_peers;
  /* fused dense Adam (adam_p, adam_m, adam_v all set or all NULL; step >= 1): the Z row is the gradient of row
   * i of adam_p [n_rows, D]; the warp applies torch.optim.Adam's arithmetic (that of spex_adam_f32) to the rows
   * of (p, m, v) and, if a publish destination is set, publishes the UPDATED p row.  Z may be NULL. */
  float* adam_p;
  float* adam_m;
  float* adam_v;
  float lr;
  float beta1;
  float beta2;
  float eps;
  int32_t step;
} spex_spmm_epilogue;

/*
 * One propagation layer with any epilogue, optionally restricted to a ROW SUBSET: only the listed rows are
 * computed and written, each with exactly the value the full layer gives it (same kernels, same summation
 * order).  The CSR may be a row block of the full matrix: X is the full [n_cols, D] table, the rows are LOCAL.
 * The subset replaces nothing literal in the reference - it removes work the reference does: main_rec.py:34
 * calls computer() (model.py:66-97: all N rows of all K layers) for a mini-batch whose loss (model.py:115-120)
 * reads only the batch's ~1.8 k rows of the result; layer K is needed on those rows only, layer K-1 on their
 * neighbours, ... (the receptive field), and the backward pass has the mirrored sparsity.
 *   rows        int32 [n_sel]       row ids (no duplicates, any order)
 *   long_slots  int32 [n_long_sel]  for the listed rows of degree > plan->seg_len: their positions in
 *                                   plan->long_rows; seg_ids int32 [n_seg_sel]: the ids of all their segments
 *   n_sel < 0                       all rows (rows / long_slots / seg_ids unused)
 *   x_nonzero   uint8 [n_cols]      optional: X is known to be ZERO (+0.0 in every element) on the rows c with
 *                                   x_nonzero[c] == 0 - the second layer of the training backward reads
 *                                   H_1 = g + A^T g, non-zero only on the batch's rows and their neighbours.  Those
 *                                   gathers are skipped; the result is bit-identical to the dense layer (the
 *                                   skipped terms are val * (+0)).  Used with 32-byte aligned tables, else ignored.
 * Subsets, publish and Adam need D in {32, 64, 128}.  Uses of the row partition (spex_b200/dist.py):
 *   Y exchange   layers 1..K-1 of a propagation: SpMM and all-gather of the next layer's table in one kernel
 *   publish      the last layer of a propagation whose next call's E^(0) is already known
 *   Adam         the last backward layer: main_rec.py:35-37's backward tail, the optimiser and the next
 *                forward's E^(0) all-gather in one kernel
 * The descriptor is checked in full (SPEX_E_BADARG / SPEX_E_ALIGN) before anything else, n_sel == 0 included.
 */
int spex_spmm_layer_f32(const int64_t* rowptr, const int32_t* col, const float* val,
                        const float* X, int64_t n_rows, int32_t D,
                        const int32_t* rows, int64_t n_sel,
                        const int32_t* long_slots, int32_t n_long_sel,
                        const int32_t* seg_ids, int32_t n_seg_sel,
                        const uint8_t* x_nonzero,
                        const spex_spmm_epilogue* ep, const spex_long_plan* plan, void* stream);

/*
 * spex_spmm_layer_f32 with an ADDED GRADIENT in the epilogue: for every computed row i with z_add_rows[i] != 0
 *      z[i,:] = (addend[i,:] * addend_scale + acc) * z_scale + z_add[i,:]
 * (one fp32 add after the scale), and both Z and the fused Adam see that sum; rows whose flag is 0 never read
 * z_add.  Replaces the autograd sum dE0 = dE0_propagated + d(reg)/dE0 of a BPR step (main_rec.py:35 with upstream
 * LightGCN's L2 term): the last backward layer of a row-partitioned step takes the ego rows' L2 gradient.
 *   z_add       fp32 [n_rows, D], 16-byte aligned (SPEX_E_ALIGN)
 *   z_add_rows  uint8 [n_rows]
 * z_add and z_add_rows are both NULL (spex_spmm_layer_f32) or both set, and then the descriptor sets Z or Adam
 * (SPEX_E_BADARG otherwise); everything is checked before anything runs.
 */
int spex_spmm_layer_zadd_f32(const int64_t* rowptr, const int32_t* col, const float* val,
                             const float* X, int64_t n_rows, int32_t D,
                             const int32_t* rows, int64_t n_sel,
                             const int32_t* long_slots, int32_t n_long_sel,
                             const int32_t* seg_ids, int32_t n_seg_sel,
                             const uint8_t* x_nonzero,
                             const spex_spmm_epilogue* ep, const float* z_add, const uint8_t* z_add_rows,
                             const spex_long_plan* plan, void* stream);

/*
 * K-layer propagation + layer mean:  out = (E0 + A·E0 + ... + A^K·E0) / (K+1)
 * E0 [N,D] is the concatenated user+item table (model.py:72); tmp0/tmp1 are [N,D] ping-pong
 * workspaces (K>=2 needs tmp0, K>=3 needs both).  The mean is accumulated in `out` by every
 * layer's epilogue; the last layer never writes its E^(K) to memory.
 * Replaces LightGCN.computer()  model.py:66-97 (K1+K2+K3 of SURVEY §2.1).
 */
int spex_propagate_mean_f32(const int64_t* rowptr, const int32_t* col, const float* val,
                            const float* E0, int64_t N, int32_t D, int32_t K,
                            float* out, float* tmp0, float* tmp1,
                            const spex_long_plan* plan, void* stream);

/*
 * Backward of spex_propagate_mean_f32 w.r.t. E0, given g = dL/d(out):
 *      G_K = g/(K+1);  G_k = g/(K+1) + A^T·G_{k+1};  dE0 = G_0
 * (rowptr,col,val) must describe A^T (for the symmetric normalised adjacency it is A itself;
 * with edge dropout pass the transposed values, see spex_gather_f32).
 * Replaces autograd through model.py:83-95 (K6 of SURVEY §2.1).
 */
int spex_propagate_mean_bwd_f32(const int64_t* rowptr, const int32_t* col, const float* valT,
                                const float* g, int64_t N, int32_t D, int32_t K,
                                float* dE0, float* tmp0, float* tmp1,
                                const spex_long_plan* plan, void* stream);

/* out[i] = (src[idx[i]] * scale[i]) / divisor   (idx NULL = identity, scale NULL = 1).
 * Used for the dropout graph (model.py:46-55: scale = 0/1 keep mask, divisor = keep_prob, an
 * IEEE fp32 division exactly like `values[random_index] / keep_prob`) and for A^T values. */
int spex_gather_f32(const float* src, const int64_t* idx, const float* scale, float divisor,
                    float* out, int64_t n, void* stream);

/*
 * Edge dropout with a counter-based mask generated on the device: the values of A_drop and A_drop^T in one
 * pass, with no host random numbers and no mask to copy.  The mask is a pure function of (seed, global row,
 * global column); for the edge at global row r = row_offset + local row and column c (bit 31 of col stripped):
 *      key  = ((uint64)r << 32) | (uint32)c
 *      h    = splitmix64(seed ^ key)            (SplitMix64 finaliser, including its += 0x9E3779B97F4A7C15)
 *      u    = (float)(h >> 40) * 0x1p-24f       (exact: 24 bits, in [0, 1))
 *      keep = (int)(u + keep_prob) != 0         (fp32 add, round to nearest: (torch.rand(n) + keep_prob).int())
 *      val_out[e]  = (val[e] * (keep(r, c) ? 1 : 0)) / keep_prob
 *      valT_out[e] = (vt     * (keep(c, r) ? 1 : 0)) / keep_prob,   vt = tpos ? val[tpos[e]] : val[e]
 * (no division when keep_prob == 1): the operations of spex_gather_f32 in the same order, so the same mask fed
 * through it gives the same bits.  The two directions of an interaction are independent draws, as in the
 * reference (model.py:46-55 draws every stored entry on its own) - but from a different generator: the
 * reference's torch.rand stream is replaced, so other edges are dropped, with the same distribution.
 *   rowptr/col/val  a CSR or a row block of one (rows r of the block are global rows row_offset + r)
 *   tpos            int64 [nnz] positions of the transposed entries in this CSR; NULL = the values are
 *                   symmetric bit for bit (val of (c, r) == val of (r, c))
 *   valT_out        NULL: only val_out is written
 * keep_prob must be in (0, 1]; n_rows == 0 is a no-op.
 */
int spex_edge_dropout_f32(const int64_t* rowptr, const int32_t* col, const float* val, const int64_t* tpos,
                          int64_t n_rows, int64_t row_offset, uint64_t seed, float keep_prob,
                          float* val_out, float* valT_out, void* stream);

/*
 * BCE step (reference loss): gamma[b] = <U[users[b]], I[items[b]]>  (model.py:115-118),
 * loss = mean BCEWithLogits(gamma, labels) (model.py:23,120).
 *   U, I      propagated user / item tables (views of `out` above), row stride D
 *   gamma     fp32 [B]   (always written; flag=1 of forward() returns it)
 *   loss      fp32 [1]   (NULL to skip: then labels may be NULL too)
 *   dgamma    fp32 [B]   dloss/dgamma = (sigmoid(gamma)-label)/B   (NULL to skip)
 * B == 0: loss = NaN (the mean of no terms, as BCEWithLogitsLoss gives), nothing else is written, and the
 * per-sample arrays (users, items, labels, gamma, dgamma) may be NULL.
 */
int spex_bce_fwd_f32(const float* U, const float* I, int32_t D,
                     const int64_t* users, const int64_t* items, const float* labels,
                     int64_t B, float* gamma, float* loss, float* dgamma, void* stream);

/*
 * Backward of the gather-dot: scatter dgamma[b]*I[items[b]] into gU[users[b]] and
 * dgamma[b]*U[users[b]] into gI[items[b]], times upstream scalar *grad_loss (device fp32[1],
 * NULL = 1).  Duplicate indices are reduced in batch order — no atomics (replaces
 * index_put_(accumulate=True), K6).  gU/gI must be zero-filled by the caller for rows not touched;
 * touched rows are overwritten.
 * work NULL: a segmented duplicate scan (O(B^2/32), <= 2^18 entries).  Otherwise (device, 16-byte
 * aligned, >= spex_scatter_workspace_bytes(max list length) bytes; list length: B for BCE, 2B for
 * BPR): a stable radix sort of (row, position) pairs + one warp per run, which pays from a few
 * thousand samples on - same summation order (ascending batch position), bit-identical gradients.
 * B == 0 writes nothing; the per-sample arrays may then be NULL (also in spex_scatter_rows_f32 and
 * spex_bpr_bwd_ws_f32).
 */
int64_t spex_scatter_workspace_bytes(int64_t total_entries);
int spex_bce_bwd_ws_f32(const float* U, const float* I, int32_t D,
                        const int64_t* users, const int64_t* items, const float* dgamma,
                        const float* grad_loss, int64_t B, float* gU, float* gI,
                        void* work, int64_t work_bytes, void* stream);
/* table[rows[i], :] = 0 for i < n: re-zeroes the rows a backward scatter touched, so that the dense
 * gradient buffer of the propagated table (N x D, 3.84 GB on the 1B-edge graph) is zero-filled
 * once, not every step (replaces the zeros_like of autograd's index backward, main_rec.py:35). */
int spex_clear_rows_f32(float* table, const int64_t* rows, int64_t n, int32_t D, void* stream);
/*
 * Row-partitioned training (SURVEY §8e rows 2-3; spex_b200/dist.py: PartitionedTrainer).
 *   spex_gather_owned_rows_f32: R[i, :] = table_local[rows[i] - row_lo, :] if row_lo <= rows[i] < row_hi,
 *       else 0 - every rank fills the rows of the batch it owns, a sum all-reduce of R then gives every
 *       rank all of them (one non-zero term per row: exact).  Replaces all_users[users] / all_items[items]
 *       (model.py:115-116) when the table is partitioned.
 *   spex_scatter_rows_f32: out[dst_rows[b] - row_lo, :] = sum over b' with the same destination, ascending
 *       b', of coef[b'] * (*gscalar) * cconst * src[src_rows[b'], :], only for destinations inside
 *       [row_lo, row_hi) (row_hi == 0: all rows): the index backward of autograd (main_rec.py:35) restricted
 *       to the rows a rank owns.  Same deterministic segmented reduction (and workspace) as spex_bce_bwd_ws_f32.
 */
int spex_gather_owned_rows_f32(const float* table_local, const int64_t* rows, int64_t n, int32_t D,
                               int64_t row_lo, int64_t row_hi, float* R, void* stream);
int spex_scatter_rows_f32(const int64_t* dst_rows, const int64_t* src_rows, const float* coef,
                          const float* gscalar, float cconst, int64_t B, const float* src, int32_t D,
                          float* out, int64_t row_lo, int64_t row_hi, void* work, int64_t work_bytes,
                          void* stream);

/*
 * BPR step (north_star addition, SURVEY §8 a5; semantics of upstream LightGCN bpr_loss):
 *   loss = mean softplus(<u,n> - <u,p>),  reg = 0.5*(|U0[u]|^2+|I0[p]|^2+|I0[n]|^2)/B
 *   out2 fp32 [2] = {loss, reg};  dscore fp32 [B] = sigmoid(<u,n>-<u,p>)/B  (NULL to skip)
 *   work2B fp32 [2*B] workspace (per-sample terms, reduced in a fixed order)
 * B == 0: out2 = {NaN, NaN} (means of no terms); users, pos, neg, dscore and work2B may be NULL.
 */
int spex_bpr_fwd_f32(const float* U, const float* I, const float* U0, const float* I0, int32_t D,
                     const int64_t* users, const int64_t* pos, const int64_t* neg, int64_t B,
                     float* out2, float* dscore, float* work2B, void* stream);

/*
 * BPR backward.  grad2 (device fp32[2]) = upstream {dL/dloss, dL/dreg}.
 *   gU[u] += gl*dscore*(n-p); gI[p] += -gl*dscore*u; gI[n] += gl*dscore*u   (propagated tables)
 *   gU0[u] += gr*U0[u]/B; gI0[p] += gr*I0[p]/B; gI0[n] += gr*I0[n]/B        (ego tables)
 * Same deterministic reduction and workspace as spex_bce_bwd_ws_f32; touched rows are overwritten,
 * untouched rows must have been zero-filled by the caller.
 */
int spex_bpr_bwd_ws_f32(const float* U, const float* I, const float* U0, const float* I0, int32_t D,
                        const int64_t* users, const int64_t* pos, const int64_t* neg,
                        const float* dscore, const float* grad2, int64_t B,
                        float* gU, float* gI, float* gU0, float* gI0,
                        void* work, int64_t work_bytes, void* stream);

/*
 * Dense Adam over one table (torch.optim.Adam semantics, main_rec.py:23,37; K7):
 *   m = b1*m+(1-b1)*g; v = b2*v+(1-b2)*g*g;
 *   p -= lr/(1-b1^t) * m / (sqrt(v)/sqrt(1-b2^t) + eps)
 */
int spex_adam_f32(float* p, const float* g, float* m, float* v, int64_t n,
                  float lr, float beta1, float beta2, float eps, int32_t step, void* stream);

/*
 * Device-side samplers (replace the host loop of LightTrainData.ng_sample,
 * LightGCN_SPEX/code/utility1/dataloader.py:250-265, and give bpr_loss its triples).
 * (rowptr, col) = the adjacency CSR: the row of user u lists its training items as
 * item_col_offset + item (ascending; bit 31 may carry the hot flag).  Counter-based randomness:
 * the same seed gives the same samples on every launch.
 *   spex_sample_negatives: out int64 [n, n_neg], out[s, q] uniform over the items user users[s]
 *                          has NOT interacted with (-1 only if it interacted with every item);
 *   spex_sample_bpr:       users/pos/neg int64 [n]: user uniform over users with >= 1 interaction,
 *                          pos uniform over its items, neg as above.
 */
int spex_sample_negatives(const int64_t* rowptr, const int32_t* col, int32_t item_col_offset,
                          int32_t m_items, const int64_t* users, int64_t n, int32_t n_neg,
                          uint64_t seed, int64_t* out, void* stream);
int spex_sample_bpr(const int64_t* rowptr, const int32_t* col, int32_t item_col_offset, int32_t m_items,
                    int64_t n_users, int64_t n, uint64_t seed, int64_t* users, int64_t* pos,
                    int64_t* neg, void* stream);

/*
 * Expert gating epilogue (configs[1], model_expert_s.py:154-161):
 *   att = softmax([E0 | Eout] · W[2D,2]);  out = E0*att0 + Eout*att1     per row
 */
int spex_expert_gate_f32(const float* E0, const float* Eout, const float* W, int64_t n,
                         int32_t D, float* out, void* stream);

/*
 * Backward of spex_expert_gate_f32 (the gate weights att_exp1/att_exp2 are trained,
 * main_11.py:62-71): given g = dL/dout, writes dE0, dEout [n, D] and dW [2D, 2].  dW is reduced
 * in a fixed order without atomics through `work` (fp32 [SPEX_GATE_BWD_BLOCKS * 512]).  D <= 128.
 */
#define SPEX_GATE_BWD_BLOCKS 1184
int spex_expert_gate_bwd_f32(const float* E0, const float* Eout, const float* W, const float* g,
                             int64_t n, int32_t D, float* dE0, float* dEout, float* dW, float* work,
                             void* stream);

/*
 * Full-ranking top-k, exact fp32 SIMT path:  for each of B users, the k best items of
 * <U[users[b]], I[j]>, j in [0, m_items), excluding the user's training items
 * (mask_rowptr int64 [n_mask_rows+1], mask_col int32 ascending per row: CSR of R; NULL = none).
 * Ordering: score descending, ties by ascending item id.  Slots beyond the number of
 * unmasked items get idx = -1, val = -inf.
 *   out_idx int32 [B,k], out_val fp32 [B,k];  k <= 128
 * Replaces getUsersRating (abstract at model.py:14-15) + torch.topk; this is the bit-exact
 * companion of the tensor-core path below (SURVEY §8 a5).
 */
int spex_score_topk_f32(const float* U, const float* I, int32_t D,
                        const int64_t* users, int64_t B, int64_t m_items,
                        const int64_t* mask_rowptr, const int32_t* mask_col,
                        int32_t k, int32_t* out_idx, float* out_val, void* stream);

/*
 * Dense rating block (API form of getUsersRating, abstract at utility1/model.py:14-15; the only
 * user x all-items product in the reference is NGCF_SPEX/code/utility/batch_test.py:158):
 *   out[b, j] = f(<U[users[b]], I[j]>),  f = sigmoid if apply_sigmoid else identity
 *   out fp32 [B, m_items] row-major;  B <= 8*65535 per call.
 */
int spex_rating_f32(const float* U, const float* I, int32_t D, const int64_t* users, int64_t B,
                    int64_t m_items, int32_t apply_sigmoid, float* out, void* stream);

/*
 * fp32 [rows, D] -> bf16 (round-to-nearest-even) in the UMMA K-major "no-swizzle" canonical
 * layout: byte offset of element (r, k) = (r/8)*(16*D) + (k/8)*128 + (r%8)*16 + (k%8)*2, i.e.
 * 8-row x 16-byte core matrices, one 8-row group contiguous.  Optional row gather
 * (rows == NULL: identity); rows [n, n_pad) are zero; n_pad % 8 == 0, D % 8 == 0.
 * dst holds n_pad*D bf16.  Feeds spex_score_topk_bf16.
 */
int spex_pack_bf16(const float* src, const int64_t* rows, int64_t n, int64_t n_pad, int32_t D,
                   void* dst_bf16, void* stream);

/*
 * Full-ranking top-k on the 5th-gen tensor cores (tcgen05.mma kind::f16, bf16 in / fp32 TMEM
 * accumulators), D == 64.  Ub [B_pad,64] / Ib [m_pad,64] are packed tables from spex_pack_bf16
 * (B_pad % 128 == 0, m_pad % 128 == 0).  Scores never reach HBM: the epilogue streams TMEM,
 * rejects below the per-row running k-th score, applies the training-item mask to survivors
 * and keeps a per-row top-k.  `user_ids` int64 [B] gives the mask row of each scored row
 * (NULL: row b uses mask row b).  Same ordering / output contract as spex_score_topk_f32;
 * k <= 64.  No workspace.
 */
int spex_score_topk_bf16(const void* Ub, const void* Ib, int64_t B, int64_t B_pad,
                         int64_t m_items, int64_t m_pad, const int64_t* user_ids,
                         const int64_t* mask_rowptr, const int32_t* mask_col,
                         int32_t k, int32_t* out_idx, float* out_val, void* stream);

/*
 * fp32 [rows, D] -> fp16( x * 2^s ) in the same UMMA K-major no-swizzle layout as spex_pack_bf16.
 * s is chosen on the device so that every scaled row norm is < 2^7 (no fp16 overflow anywhere in
 * a score, |score| < 2^14):  meta4 (device fp32 [4], 16-byte aligned) receives
 *   meta4[0] = 2^s, meta4[1] = 2^-s, meta4[2] = max scaled row norm, meta4[3] = max row norm^2.
 * Feeds spex_score_topk_f16 (operands of NGCF_SPEX/code/utility/batch_test.py:158's matmul).
 */
int spex_pack_f16(const float* src, const int64_t* rows, int64_t n, int64_t n_pad, int32_t D,
                  void* dst_f16, float* meta4, void* stream);

/*
 * Full-ranking top-k, fp16-accumulator tensor-core filter + exact fp32 re-score (D == 64 or 128).
 * Uh [B_pad, D] / Ih [m_pad, D] and u_meta / i_meta come from spex_pack_f16.  The tensor core
 * (tcgen05.mma kind::f16, fp16 accumulators: half the TMEM -> register drain of the bf16/fp32
 * kernel) only FILTERS against  tau - eps;  every survivor is re-scored in fp32 from the fp16
 * operands, so the result is the exact top-k of  <fp16(U 2^su), fp16(I 2^si)> 2^-(su+si)
 * (score descending, ties by ascending item id; values in the original units).  Mask, user_ids,
 * outputs and k <= 64 as spex_score_topk_bf16.  No workspace.
 * Replaces torch.matmul(u_g_embeddings, i_g_embeddings^T) + the ranking that follows it
 * (NGCF_SPEX/code/utility/batch_test.py:158) and serves LightGCN.getUsersRating + top-k
 * (abstract at LightGCN_SPEX/code/utility1/model.py:14-15).
 */
int spex_score_topk_f16(const void* Uh, const void* Ih, int32_t D, int64_t B, int64_t B_pad,
                        int64_t m_items, int64_t m_pad, const float* u_meta, const float* i_meta,
                        const int64_t* user_ids, const int64_t* mask_rowptr,
                        const int32_t* mask_col, int32_t k, int32_t* out_idx, float* out_val,
                        void* stream);

/*
 * The same scorer for 1 <= k <= 512: same operands, filter, mask, user_ids and output contract as
 * spex_score_topk_f16 (exact top-k of the fp32 scores of the fp16 operands, score descending, ties
 * by ascending item id, -1 / -inf past the user's unmasked items).  Each user row's candidate
 * buffer lives in the caller's workspace instead of shared memory: work (device, 16-byte aligned)
 * of at least spex_score_topk_f16_wide_workspace_bytes(B_pad, k) bytes, B_pad * cap(k) entries of
 * 8 bytes with cap(k) = 2k + 64 rounded up to 32; its contents on entry do not matter.  Serves
 * the k above 64 that spex_score_topk_f16 rejects (and above 128, where spex_score_topk_f32 stops).
 * Errors, before anything is launched: SPEX_E_TOOBIG for k outside [1, 512] or m_pad >= 2^31;
 * SPEX_E_WORKSPACE for work NULL or smaller than the query; SPEX_E_ALIGN for Uh, Ih or work
 * misaligned; SPEX_E_BADARG for B_pad or m_pad not a multiple of 128, half a mask, NULL operands
 * or outputs; SPEX_E_BADDIM for D not 64 or 128.
 * spex_score_topk_f16_wide_workspace_bytes returns 0 for B_pad < 0 or k outside [1, 512].
 */
int64_t spex_score_topk_f16_wide_workspace_bytes(int64_t B_pad, int32_t k);
int spex_score_topk_f16_wide(const void* Uh, const void* Ih, int32_t D, int64_t B, int64_t B_pad,
                             int64_t m_items, int64_t m_pad, const float* u_meta, const float* i_meta,
                             const int64_t* user_ids, const int64_t* mask_rowptr,
                             const int32_t* mask_col, int32_t k, int32_t* out_idx, float* out_val,
                             void* work, int64_t work_bytes, void* stream);

/*
 * Full-ranking rank of held-out pairs.  Pair p = (user u_p, item t_p); its rank is
 *   r_p = #{ i in [0, m_items) : i not in mask row of u_p, i != t_p, s(u_p, i) > s(u_p, t_p)
 *                                or (s(u_p, i) == s(u_p, t_p) and i < t_p) }
 * with s the exact score of the precision: the position of t_p in that precision's top-k list when it is there,
 * >= k otherwise; t_p may be masked (its rank is still defined).  A mask row may repeat an id (it is
 * excluded once).  out_rank int32 [P], in pair order; one store per
 * pair, no atomics: the same inputs give the same bits.  Item ids must lie in [0, m_items) (not checked here).
 *
 * spex_rank_pairs_f16 (D == 64 or 128): s = the fp32 FMA chain over the fp16 operands of spex_score_topk_f16.  Uh is
 * a table packed by spex_pack_f16 (the users' rows, any order), a_rows int64 [P] the row of Uh of each pair (NULL:
 * row p); Ih / i_meta the packed item table; user_ids int64 [P] the mask row of each pair (NULL: row p); mask as
 * spex_score_topk_f16.  P_pad >= P and m_pad are multiples of 128.  The tensor core computes the fp16 filter
 * value of every (pair, item); only items within the filter's error bound of s(u_p, t_p) are re-scored exactly.
 * Errors, before anything is launched: SPEX_E_BADDIM for D not 64 or 128; SPEX_E_BADARG for P_pad or m_pad not a
 * multiple of 128, half a mask, NULL operands, items or out_rank, m_items == 0 with P > 0; SPEX_E_TOOBIG for
 * m_pad >= 2^31; SPEX_E_ALIGN for Uh or Ih misaligned.
 *
 * spex_rank_pairs_f32 (D a multiple of 4, <= 512): s = the dot product of spex_score_topk_f32 in its accumulation
 * order, over U [.., D] / I [m_items, D] fp32; users int64 [P] are the rows of U and the mask rows.
 * Errors, before anything is launched: SPEX_E_BADDIM for D; SPEX_E_BADARG for half a mask, NULL operands, users,
 * items or out_rank, m_items == 0 with P > 0; SPEX_E_TOOBIG for m_items >= 2^31; SPEX_E_ALIGN for U or I.
 */
int spex_rank_pairs_f16(const void* Uh, const void* Ih, int32_t D, const int64_t* a_rows,
                        const int64_t* user_ids, const int32_t* items, int64_t P, int64_t P_pad,
                        int64_t m_items, int64_t m_pad, const float* i_meta, const int64_t* mask_rowptr,
                        const int32_t* mask_col, int32_t* out_rank, void* stream);
int spex_rank_pairs_f32(const float* U, const float* I, int32_t D, const int64_t* users,
                        const int32_t* items, int64_t P, int64_t m_items, const int64_t* mask_rowptr,
                        const int32_t* mask_col, int32_t* out_rank, void* stream);

/*
 * Sampled-candidate scoring for the reference Test() (batch_test.py:28-40, hoisted):
 *   score[u,c] = <U[users[u]], I[cand[u,c]]>,  cand int32 [n_u, n_c]  ->  score fp32 [n_u, n_c]
 */
int spex_score_candidates_f32(const float* U, const float* I, int32_t D,
                              const int64_t* users, const int32_t* cand, int64_t n_u,
                              int32_t n_c, float* score, void* stream);

/*
 * Full-ranking metrics of one block of top-k lists, at up to SPEX_METRICS_MAX_CUTOFFS cutoffs, with the
 * definitions of spex_b200/metrics.py: fullrank_recall_ndcg (upstream LightGCN).  For user u and cutoff K:
 *   hits      = number of topk_idx[u, :K] entries found in the user's truth row (np.isin semantics)
 *   recall    = hits / |truth| (0 for an empty row)    precision = hits / K    hit = (hits > 0)
 *   ndcg      = DCG / idcg[min(|truth|, K)] (0 where that is 0), DCG = sum of disc[i] over the hit ranks i < K,
 *               summed in ascending i
 *   topk_idx     int32 [B, k], best first, -1 padding (the output of any scorer above); 1 <= k <= 512
 *   truth_rowptr int64 [B + 1], truth_col int32: the held-out items of the users as a CSR over their POSITIONS in
 *                this block, each row ascending (duplicates allowed); the positions are absolute in truth_col, so a
 *                caller ranking users [s, s + b) of a longer list passes truth_rowptr + s
 *   cutoffs_host n_cut (1..8) cutoffs, strictly ascending, each in [1, k]
 *   disc         fp64 [k]: 1 / log2(i + 2);  idcg fp64 [k + 1]: 0 followed by the running sums of disc (both
 *                computed by the caller, so the device never evaluates a logarithm)
 *   per_user     fp64 [B, n_cut, 4] (recall, precision, ndcg, hit) per user and cutoff; NULL: not written
 *   chunk_sums   fp64 [ceil(B / SPEX_METRICS_CHUNK), n_cut, 4]: the sums over each chunk of SPEX_METRICS_CHUNK
 *                consecutive users, in a fixed order that depends only on that chunk's per-user values
 * spex_fullrank_metrics_reduce sums n_chunks chunk sums in ascending chunk order into sums fp64 [n_cut, 4]
 * (n_chunks == 0 writes zeros).  No atomics: the same inputs give the same bits on every run.
 * Errors, before anything is launched: SPEX_E_TOOBIG for k > 512 or n_cut > 8; SPEX_E_BADARG for k < 1, n_cut < 1,
 * B < 0, cutoffs not strictly ascending or outside [1, k], NULL cutoffs, disc or idcg, and (B > 0) NULL topk_idx,
 * truth or chunk_sums.  B == 0 reads and writes nothing.
 * Replaces the per-user np.isin loop over a [B, k] id matrix copied to the host (metrics.py: fullrank_recall_ndcg,
 * called by batch_test.test_fullrank).
 */
#define SPEX_METRICS_MAX_CUTOFFS 8
#define SPEX_METRICS_CHUNK 1024
int spex_fullrank_metrics(const int32_t* topk_idx, int64_t B, int32_t k,
                          const int64_t* truth_rowptr, const int32_t* truth_col,
                          const int32_t* cutoffs_host, int32_t n_cut,
                          const double* disc, const double* idcg,
                          double* per_user, double* chunk_sums, void* stream);
int spex_fullrank_metrics_reduce(const double* chunk_sums, int64_t n_chunks, int32_t n_cut,
                                 double* sums, void* stream);

/*
 * The same metrics from the ranks of the held-out items (spex_rank_pairs_*) instead of top-k lists, at cutoffs up
 * to m_items, plus MRR and AUC.  ranks int32 is aligned with truth_col: ranks[j] is the rank of truth_col[j] for
 * its user.  A held-out item in the user's mask row, or a repeat of the item before it in its truth row, is never a
 * hit, as in spex_fullrank_metrics, where it cannot appear in a list.  For user u with truth row T:
 *   hits, recall, precision, hit, ndcg as spex_fullrank_metrics with "rank < K" for "in topk[:K]"; the DCG sums
 *               disc[r] over the hit ranks in ascending r (the same bits as the top-k path);
 *               disc fp64 [max cutoff], idcg fp64 [max cutoff + 1] as there
 *   mrr       = 1 / (1 + min r) over the hits at any rank (0 when there is none)
 *   auc       = mean over the entries t of T of 1 - (r_t - #{live t' : r_t' < r_t}) / n_neg, n_neg = m_items -
 *               #{distinct ids of the mask row in [0, m_items)} - #{live t'}; a masked entry contributes 0;
 *               n_neg == 0 gives 1 (no negative outranks t)
 * (live = not masked and not a repeat; an empty truth row contributes zeros).  users int64 [B] gives each
 * position's mask row (needed only with a mask).  chunk_sums fp64 [n_chunks, n_cut, 4] as spex_fullrank_metrics,
 * chunk_extra fp64 [n_chunks, 4] = (mrr, auc, 0, 0) sums per chunk: both go through spex_fullrank_metrics_reduce
 * (chunk_extra with n_cut = 1).  No atomics.  One warp per user; a user with T held-out items costs O(T^2 / 32)
 * steps (each entry is compared with every other, and the hit walk scans the row once per hit), which suits
 * leave-one-out and short truth rows, not rows of thousands of items.
 * Errors, before anything is launched: SPEX_E_TOOBIG for n_cut > 8 or m_items >= 2^31; SPEX_E_BADARG for B < 0,
 * m_items < 1, n_cut < 1, cutoffs not strictly ascending or outside [1, m_items], half a mask, NULL cutoffs, disc or
 * idcg and (B > 0) NULL ranks, truth, sums or (with a mask) users.
 */
int spex_rank_metrics(const int32_t* ranks, int64_t B, const int64_t* truth_rowptr,
                      const int32_t* truth_col, const int64_t* users, const int64_t* mask_rowptr,
                      const int32_t* mask_col, int64_t m_items, const int32_t* cutoffs_host,
                      int32_t n_cut, const double* disc, const double* idcg, double* chunk_sums,
                      double* chunk_extra, void* stream);

/*
 * NGCF layer epilogue (configs[2], NGCF_SPEX/code/main_rec.py:76-85), D == 64:
 *   out = lrelu(side·W1^T + b1) + lrelu((ego*side)·W2^T + b2);  norm = out / max(|out|_2, 1e-12)
 * side = A·ego comes from spex_spmm_csr_f32.  W row-major [64,64] (nn.Linear.weight layout).
 * `out` is the next layer's ego (pre-normalisation, dropout applied by the caller in training),
 * `norm` is written with row stride norm_stride floats (the concat buffer of main_rec.py:85).
 */
int spex_ngcf_epilogue_f32(const float* ego, const float* side, const float* W1, const float* b1,
                           const float* W2, const float* b2, int64_t n, int32_t D,
                           float negative_slope, float* out, float* norm, int64_t norm_stride,
                           void* stream);

/*
 * NGCF layer for TRAINING (NGCF_SPEX/code/main_rec.py:76-82 and its autograd), D == 64.
 *   fwd: hd = (lrelu(side W1^T + b1) + lrelu((ego*side) W2^T + b2)) * mask   (mask NULL = 1: the 0 / 1/(1-p)
 *        pattern of nn.Dropout, main_rec.py:81, drawn by the caller with the reference's RNG call);
 *        norm = hd / max(|hd|, 1e-12) written with row stride norm_stride (concat buffer, main_rec.py:82-85).
 *   bwd: d_hd_next = dL/d(hd) from the next layer (NULL for the last), d_norm = dL/d(norm) with its row
 *        stride; writes d_ego, d_side [n, 64] and the weight / bias gradients.  The weight gradients are
 *        reduced deterministically (fixed tile order per CTA, CTA partials summed in CTA order):
 *        work = fp32 [SPEX_NGCF_BWD_BLOCKS * SPEX_NGCF_BWD_WORK_PER_BLOCK] workspace.
 */
#define SPEX_NGCF_BWD_BLOCKS 296
#define SPEX_NGCF_BWD_WORK_PER_BLOCK 8320
int spex_ngcf_layer_fwd_f32(const float* ego, const float* side, const float* W1, const float* b1,
                            const float* W2, const float* b2, const float* mask, int64_t n, int32_t D,
                            float negative_slope, float* hd, float* norm, int64_t norm_stride,
                            void* stream);
int spex_ngcf_layer_bwd_f32(const float* ego, const float* side, const float* W1, const float* b1,
                            const float* W2, const float* b2, const float* mask, const float* d_hd_next,
                            const float* d_norm, int64_t d_norm_stride, int64_t n, int32_t D,
                            float negative_slope, float* d_ego, float* d_side, float* dW1, float* db1,
                            float* dW2, float* db2, float* work, void* stream);

/*
 * CUDA-IPC helpers for the row-partitioned multi-GPU path (SURVEY §8e): each rank allocates its
 * exchange buffer with spex_ipc_alloc, publishes the 64-byte handle, and opens its peers'.  The layer
 * kernel stores into the mapped tables through spex_spmm_epilogue's Y exchange and publish.
 */
int spex_ipc_alloc(int64_t bytes, void** dev_ptr, void* handle64_host);
int spex_ipc_open(const void* handle64_host, void** dev_ptr);
int spex_ipc_close(void* dev_ptr);
int spex_ipc_free(void* dev_ptr);
/* all-gather of this rank's E^(0) rows: src fp32 [n_rows, D] is stored at rows
 * [out_row_offset, out_row_offset + n_rows) of each of the n_peers (<= 8) tables (own included) by P2P
 * stores, or of every GPU's table by ONE multimem.st per element to the multicast mapping mcast_Y.
 * n_ctas == 0 is the full-speed grid; a small n_ctas (e.g. the SM count) makes it a BACKGROUND exchange
 * that can run next to a layer kernel on a high-priority stream (spex_b200/dist.py: the next call's
 * E^(0) is published while the last layer runs). */
int spex_push_rows_f32_ex(const float* src, int64_t n_rows, int32_t D, int64_t out_row_offset,
                          float* const* peer_Y_host, int32_t n_peers, int32_t n_ctas, void* stream);
int spex_mcast_rows_f32_ex(const float* src, int64_t n_rows, int32_t D, int64_t out_row_offset,
                           float* mcast_Y, int32_t n_ctas, void* stream);
/* cudaMemcpyAsync(DeviceToDevice) on `stream`: a copy-engine transfer into an IPC-mapped peer
 * table (dst may be peer memory), used for the E^(0) all-gather so that no SM is involved. */
int spex_memcpy_peer_async(void* dst, const void* src, int64_t bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SPEX_B200_H */
